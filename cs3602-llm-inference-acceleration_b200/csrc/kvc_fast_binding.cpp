// kvc_fast_binding.cpp — compiled host binding for the per-step call of the compress functions.
//
// The reference's decode loop calls compress_fn(kv_list, ...) once per generated token (evaluate.py:154-166), and at
// batch 1 — the only regime the reference published — a call is ~60 us of GPU work.  The ctypes binding
// (kvcompress/_engine.py: run_plans) walks the layers in Python: per layer two tensors are validated, their strides
// and pointers read, a 128-byte record packed; ~160 us per call.  This module does the same walk in C++ on
// at::Tensor directly: one call per compress function, the same `kvc_compress_layers_ws` entry point of
// libkvc_sm100a.so behind it (its address is handed over by the ctypes loader, so there is nothing to link).
//
// It covers the common case only — CUDA tensors, rows the kernels can read in place, one (B, H, D, dtype, device) group,
// no caller-supplied rows/scores, no index output.  Anything else makes run() return None and the Python path, which
// also owns every error message, takes the call.
#include <c10/cuda/CUDAStream.h>
#include <torch/extension.h>

#include <array>
#include <cstdint>
#include <map>
#include <tuple>
#include <vector>

#include "kvc.h"

namespace {

using CompressFn = int (*)(const kvc_shape*, int32_t, const kvc_layer_plan*, const kvc_layer_io*, void*, int64_t, void*);
using WorkspaceFn = int64_t (*)(const kvc_shape*, int32_t, const kvc_layer_plan*);
using AppendFn = int (*)(const kvc_shape*, int32_t, const kvc_slab_layer*, const kvc_slab_new_rows*, void*);

inline void* current_stream(const c10::Device& dev) {
    return reinterpret_cast<void*>(c10::cuda::getCurrentCUDAStream(dev.index()).stream());
}

enum Kind { KEEP = 0, VIEW = 1, GATHER = 2 };

inline int dtype_code(at::ScalarType t) {
    switch (t) {
        case at::kFloat: return KVC_DTYPE_F32;
        case at::kHalf: return KVC_DTYPE_F16;
        case at::kBFloat16: return KVC_DTYPE_BF16;
        default: return -1;
    }
}

inline bool rows_ok(const at::Tensor& t, int64_t e) {
    const auto st = t.strides();
    return (st[3] == 1 || t.size(3) == 1) && (st[0] * e) % 16 == 0 && (st[1] * e) % 16 == 0 && (st[2] * e) % 16 == 0 &&
           reinterpret_cast<uintptr_t>(t.data_ptr()) % 16 == 0;
}

class FastPlans {
public:
    // recs[i] = {kind, seq_len, sink, sel_lo, sel_hi, k_sel, tail, score, pool_kernel}
    FastPlans(const std::vector<std::array<int64_t, 9>>& recs, uintptr_t fn_compress, uintptr_t fn_workspace)
        : compress_(reinterpret_cast<CompressFn>(fn_compress)), workspace_(reinterpret_cast<WorkspaceFn>(fn_workspace)) {
        for (size_t i = 0; i < recs.size(); ++i) {
            const auto& r = recs[i];
            kinds_.push_back((int)r[0]);
            kvc_layer_plan p;
            p.seq_len = (int32_t)r[1];
            p.sink = (int32_t)r[2];
            p.sel_lo = (int32_t)r[3];
            p.sel_hi = (int32_t)r[4];
            p.k_sel = (int32_t)r[5];
            p.tail = (int32_t)r[6];
            p.score = (int32_t)r[7];
            p.pool_kernel = (int32_t)r[8];
            all_plans_.push_back(p);
            if (r[0] == GATHER) {
                gather_.push_back((int)i);
                plans_.push_back(p);
                // caller-supplied rows / scores need tensors this path does not take
                if (p.k_sel > 0 && (p.score == KVC_SCORE_GIVEN_INDEX || p.score == KVC_SCORE_GIVEN_SCORE ||
                                    p.score == KVC_SCORE_GIVEN_SCORE_SHARED))
                    simple_ = false;
            } else if (r[0] == VIEW) {
                simple_ = false;  // views are pure Python slicing: nothing to speed up
            }
        }
        uniform_ = true;
        for (size_t m = 1; m < plans_.size(); ++m)
            uniform_ = uniform_ && out_len(plans_[m]) == out_len(plans_[0]);
    }

    py::object run(py::list kv, py::object norms) {
        const size_t L = kinds_.size();
        if (!simple_ || (size_t)py::len(kv) != L) return py::none();
        // a real shallow copy (py::list(kv) would alias the caller's list): untouched layers stay the caller's own objects
        py::list out = py::reinterpret_steal<py::list>(PyList_GetSlice(kv.ptr(), 0, (Py_ssize_t)L));
        const size_t n = gather_.size();
        if (n == 0) return std::move(out);

        std::vector<at::Tensor> ks(n), vs(n), ns;
        const bool have_norms = !norms.is_none();
        py::sequence norm_seq;
        if (have_norms) {
            norm_seq = norms.cast<py::sequence>();
            if ((size_t)py::len(norm_seq) != L) return py::none();
            ns.resize(n);
        }
        int64_t B = 0, H = 0, D = 0, e = 0;
        int dt = -1;
        c10::Device dev(c10::kCPU);
        for (size_t m = 0; m < n; ++m) {
            py::handle item = kv[gather_[m]];
            if (!py::isinstance<py::tuple>(item) && !py::isinstance<py::list>(item)) return py::none();
            py::sequence pair = py::reinterpret_borrow<py::sequence>(item);
            if (py::len(pair) < 2) return py::none();
            py::object ko = pair[0], vo = pair[1];
            if (!THPVariable_Check(ko.ptr()) || !THPVariable_Check(vo.ptr())) return py::none();
            const at::Tensor& k = THPVariable_Unpack(ko.ptr());
            const at::Tensor& v = THPVariable_Unpack(vo.ptr());
            if (!k.is_cuda() || !v.is_cuda() || k.dim() != 4 || v.dim() != 4) return py::none();
            if (m == 0) {
                dt = dtype_code(k.scalar_type());
                if (dt < 0) return py::none();
                B = k.size(0), H = k.size(1), D = k.size(3), e = (int64_t)k.element_size();
                dev = k.device();
                if ((D * e) % 16 != 0) return py::none();
            }
            if (k.scalar_type() != v.scalar_type() || dtype_code(k.scalar_type()) != dt || k.device() != dev ||
                v.device() != dev || k.size(0) != B || k.size(1) != H || k.size(3) != D || !k.sizes().equals(v.sizes()) ||
                k.size(2) != plans_[m].seq_len || !rows_ok(k, e) || !rows_ok(v, e))
                return py::none();
            ks[m] = k;
            vs[m] = v;
            if (have_norms) {
                py::object no = norm_seq[gather_[m]];
                const kvc_layer_plan& p = plans_[m];
                const bool ranked = p.k_sel > 0 && (p.score == KVC_SCORE_L2_LOW || p.score == KVC_SCORE_L2_HIGH ||
                                                    p.score == KVC_SCORE_SNAPKV_POOL);
                if (!no.is_none() && ranked) {
                    if (!THPVariable_Check(no.ptr())) return py::none();
                    const at::Tensor& t = THPVariable_Unpack(no.ptr());
                    if (t.scalar_type() != k.scalar_type() || t.dim() != 3 || t.size(0) != B || t.size(1) != H ||
                        t.size(2) < p.seq_len || t.stride(2) != 1 || t.device() != dev)
                        return py::none();
                    ns[m] = t;
                }
            }
        }

        // one allocation for every output of the call; per-layer tensors are views of it
        std::vector<at::Tensor> k_out(n), v_out(n);
        const auto opts = ks[0].options();
        if (uniform_) {
            const int64_t C = out_len(plans_[0]);
            at::Tensor big = at::empty({(int64_t)(2 * n), B, H, C, D}, opts);
            for (size_t m = 0; m < n; ++m) {
                k_out[m] = big.select(0, (int64_t)(2 * m));
                v_out[m] = big.select(0, (int64_t)(2 * m + 1));
            }
        } else {
            int64_t total = 0;
            for (size_t m = 0; m < n; ++m) total += 2 * B * H * out_len(plans_[m]) * D;
            at::Tensor flat = at::empty({total}, opts);
            int64_t off = 0;
            for (size_t m = 0; m < n; ++m) {
                const int64_t C = out_len(plans_[m]), sz = B * H * C * D;
                // one view op per tensor (narrow + view would be two): per-layer budgets make 2 x layers of them per call
                k_out[m] = flat.as_strided({B, H, C, D}, {H * C * D, C * D, D, 1}, off);
                v_out[m] = flat.as_strided({B, H, C, D}, {H * C * D, C * D, D, 1}, off + sz);
                off += 2 * sz;
            }
        }

        std::vector<kvc_layer_io> io(n);
        for (size_t m = 0; m < n; ++m) {
            kvc_layer_io& x = io[m];
            x.k_in = ks[m].data_ptr();
            x.v_in = vs[m].data_ptr();
            x.k_out = k_out[m].data_ptr();
            x.v_out = v_out[m].data_ptr();
            x.k_stride_b = ks[m].stride(0), x.k_stride_h = ks[m].stride(1), x.k_stride_s = ks[m].stride(2);
            x.v_stride_b = vs[m].stride(0), x.v_stride_h = vs[m].stride(1), x.v_stride_s = vs[m].stride(2);
            x.idx_out = nullptr;
            x.idx_in = nullptr;
            x.score_in = nullptr;
            x.norms_in = nullptr;
            x.n_stride_b = x.n_stride_h = 0;
            if (have_norms && ns[m].defined()) {
                x.norms_in = ns[m].data_ptr();
                x.n_stride_b = ns[m].stride(0);
                x.n_stride_h = ns[m].stride(1);
            }
        }
        kvc_shape shape;
        shape.batch = (int32_t)B;
        shape.heads = (int32_t)H;
        shape.head_dim = (int32_t)D;
        shape.dtype = dt;
        shape.device = (int32_t)dev.index();

        // selections larger than shared memory need a device workspace: pure host arithmetic, cached per shape
        const auto key = std::make_tuple(B, H, D, dt);
        auto it = ws_need_.find(key);
        if (it == ws_need_.end()) it = ws_need_.emplace(key, workspace_(&shape, (int32_t)n, plans_.data())).first;
        at::Tensor ws;
        void* ws_ptr = nullptr;
        if (it->second > 0) {
            ws = at::empty({it->second}, opts.dtype(at::kByte));
            ws_ptr = ws.data_ptr();
        }
        const int status = compress_(&shape, (int32_t)n, plans_.data(), io.data(), ws_ptr, it->second, current_stream(dev));
        if (status != KVC_OK) return py::none();  // the Python path repeats the call and raises the library's message
        for (size_t m = 0; m < n; ++m) out[gather_[m]] = py::make_tuple(k_out[m], v_out[m]);
        return std::move(out);
    }

private:
    static int64_t out_len(const kvc_layer_plan& p) { return (int64_t)p.sink + p.k_sel + p.tail; }

    CompressFn compress_;
    WorkspaceFn workspace_;
    std::vector<int> kinds_, gather_;
    std::vector<kvc_layer_plan> all_plans_, plans_;
    std::map<std::tuple<int64_t, int64_t, int64_t, int>, int64_t> ws_need_;
    bool simple_ = true, uniform_ = true;
};

// The per-layer `update` of a decode loop on a device-resident KVSlabCache (HF Cache.update contract: append
// [B, H, T, D] rows to one layer, return that layer's (K, V) views): one kvc_slab_append call, no Python packing.
class SlabFast {
public:
    SlabFast(std::vector<at::Tensor> k_layers, std::vector<at::Tensor> v_layers, std::vector<at::Tensor> n_layers,
             uintptr_t fn_append)
        : k_(std::move(k_layers)), v_(std::move(v_layers)), n_(std::move(n_layers)),
          append_(reinterpret_cast<AppendFn>(fn_append)) {
        const at::Tensor& k0 = k_.at(0);
        B_ = k0.size(0), H_ = k0.size(1), cap_ = k0.size(2), D_ = k0.size(3);
        e_ = (int64_t)k0.element_size();
        shape_.batch = (int32_t)B_;
        shape_.heads = (int32_t)H_;
        shape_.head_dim = (int32_t)D_;
        shape_.dtype = dtype_code(k0.scalar_type());
        shape_.device = (int32_t)k0.device().index();
        for (size_t l = 0; l < k_.size(); ++l) {
            kvc_slab_layer s;
            s.k = k_[l].data_ptr();
            s.v = v_[l].data_ptr();
            s.norms = n_[l].data_ptr();
            s.k_stride_b = k_[l].stride(0), s.k_stride_h = k_[l].stride(1);
            s.v_stride_b = v_[l].stride(0), s.v_stride_h = v_[l].stride(1);
            s.n_stride_b = n_[l].stride(0), s.n_stride_h = n_[l].stride(1);
            slabs_.push_back(s);
        }
    }

    // Returns (K view, V view) of rows [0, cur_len + T), or None when the Python path (which owns the diagnostics)
    // should take the call.
    py::object update(const at::Tensor& k_in, const at::Tensor& v_in, int64_t layer, int64_t cur_len) {
        if (layer < 0 || layer >= (int64_t)k_.size()) return py::none();
        const at::Tensor& ks = k_[layer];
        if (!k_in.is_cuda() || k_in.dim() != 4 || k_in.scalar_type() != ks.scalar_type() ||
            v_in.scalar_type() != ks.scalar_type() || k_in.device() != ks.device() || v_in.device() != ks.device() ||
            !k_in.sizes().equals(v_in.sizes()) || k_in.size(0) != B_ || k_in.size(1) != H_ || k_in.size(3) != D_)
            return py::none();
        const int64_t T = k_in.size(2);
        if (T <= 0 || cur_len < 0 || cur_len + T > cap_) return py::none();
        const at::Tensor k = rows_ok(k_in, e_) ? k_in : k_in.contiguous();
        const at::Tensor v = rows_ok(v_in, e_) ? v_in : v_in.contiguous();
        kvc_slab_new_rows r;
        r.k_new = k.data_ptr();
        r.v_new = v.data_ptr();
        r.k_stride_b = k.stride(0), r.k_stride_h = k.stride(1), r.k_stride_s = k.stride(2);
        r.v_stride_b = v.stride(0), r.v_stride_h = v.stride(1), r.v_stride_s = v.stride(2);
        r.cur_len = (int32_t)cur_len;
        r.n_new = (int32_t)T;
        if (append_(&shape_, 1, &slabs_[layer], &r, current_stream(ks.device())) != KVC_OK) return py::none();
        return py::make_tuple(ks.narrow(2, 0, cur_len + T), v_[layer].narrow(2, 0, cur_len + T));
    }

private:
    std::vector<at::Tensor> k_, v_, n_;
    std::vector<kvc_slab_layer> slabs_;
    AppendFn append_;
    kvc_shape shape_;
    int64_t B_ = 0, H_ = 0, cap_ = 0, D_ = 0, e_ = 0;
};

// seq_lens of a list of (K, V) pairs without a Python-level loop
std::vector<int64_t> seq_lens(py::list kv) {
    std::vector<int64_t> out;
    out.reserve(py::len(kv));
    for (py::handle item : kv) {
        py::sequence pair = py::reinterpret_borrow<py::sequence>(item);
        py::object ko = pair[0];
        if (!THPVariable_Check(ko.ptr())) throw py::type_error("layer keys must be tensors");
        out.push_back(THPVariable_Unpack(ko.ptr()).size(2));
    }
    return out;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    m.doc() = "compiled per-call binding of kvcompress-b200 (host-side pointer walk; kernels live in libkvc_sm100a.so)";
    py::class_<FastPlans>(m, "FastPlans")
        .def(py::init<const std::vector<std::array<int64_t, 9>>&, uintptr_t, uintptr_t>())
        .def("run", &FastPlans::run, py::arg("kv"), py::arg("norms"));
    py::class_<SlabFast>(m, "SlabFast")
        .def(py::init<std::vector<at::Tensor>, std::vector<at::Tensor>, std::vector<at::Tensor>, uintptr_t>())
        .def("update", &SlabFast::update, py::arg("key_states"), py::arg("value_states"), py::arg("layer_idx"),
             py::arg("cur_len"));
    m.def("seq_lens", &seq_lens);
    m.attr("KVC_ABI_VERSION") = KVC_ABI_VERSION;
}
