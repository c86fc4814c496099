// quant_cuda_pybind.cpp - the Python module `quant_cuda`: same 12 function names, positional
// signatures and accumulate-into-`mul` semantics as the reference's pybind module
// (squeezellm/quant_cuda.cpp:112-270), implemented as a thin torch::Tensor -> C ABI adapter over
// libsqllm_b200.so (include/sqllm_b200.h).  No kernels live here.
//
// Deliberate differences from the reference wrapper (all "more defined", none changes results):
//   * arguments are validated (device, dtype, contiguity, shapes) and violations raise RuntimeError;
//     the reference has no checks (SURVEY.md section 8(b));
//   * kernels are launched on PyTorch's CURRENT stream (the reference uses the legacy default
//     stream, quant_cuda_kernel.cu:147,172,...), so the calls are CUDA-graph capturable;
//   * `*_balanced_*` is not exported, exactly as in the reference (quant.py:238,282 reference a
//     symbol that quant_cuda.cpp never defines).
// Extra, not in the reference: `lutgemv_fused`, `unpack_indices`, `abi_version`.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <cuda_runtime.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "sqllm_b200.h"

namespace {

void check_status(int rc, const char *what) { TORCH_CHECK(rc == SQLLM_OK, what, ": ", sqllm_last_error()); }

void need(const torch::Tensor &t, const char *name, c10::ScalarType dt, const torch::Tensor &like) {
    TORCH_CHECK(t.defined(), name, " is undefined");
    TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
    TORCH_CHECK(t.device() == like.device(), name, " is on ", t.device(), " but vec is on ", like.device());
    TORCH_CHECK(t.scalar_type() == dt, name, " must have dtype ", dt, " (got ", t.scalar_type(), ")");
    TORCH_CHECK(t.is_contiguous(), name, " must be contiguous");
}

void *cur_stream() { return static_cast<void *>(at::cuda::getCurrentCUDAStream().stream()); }

struct Dense {
    const float *vec;
    const int32_t *mat;
    float *mul;
    const float *lut;
    int height, width, batch, vec_height;
};

Dense check_dense(int bits, const torch::Tensor &vec, const torch::Tensor &mat, const torch::Tensor &mul,
                  const torch::Tensor &lut, bool batched) {
    need(vec, "vec", torch::kFloat32, vec);
    need(mat, "mat", torch::kInt32, vec);
    need(mul, "mul", torch::kFloat32, vec);
    need(lut, "lookup_table", torch::kFloat32, vec);
    TORCH_CHECK(mat.dim() == 2, "mat must be 2-D [in/32*bits, out]");
    Dense d;
    d.height = (int)mat.size(0);
    d.width = (int)mat.size(1);
    TORCH_CHECK(d.height % bits == 0, "mat has ", d.height, " rows, not a multiple of bits=", bits);
    const int64_t K = (int64_t)d.height / bits * 32;
    if (batched) {
        TORCH_CHECK(vec.dim() == 2, "batched vec must be 2-D [batch, in]");
        d.batch = (int)vec.size(0);
        d.vec_height = (int)vec.size(1);
        TORCH_CHECK(mul.numel() == (int64_t)d.batch * d.width, "mul must have batch*out = ", (int64_t)d.batch * d.width, " elements");
    } else {
        d.batch = 1;
        d.vec_height = (int)vec.numel();
        TORCH_CHECK(mul.numel() == d.width, "mul must have out = ", d.width, " elements (got ", mul.numel(), ")");
    }
    TORCH_CHECK(d.vec_height == K, "vec has ", d.vec_height, " features but mat implies ", K);
    TORCH_CHECK(lut.numel() == (int64_t)d.width * (1 << bits), "lookup_table must be [out, 2^bits]");
    d.vec = vec.data_ptr<float>();
    d.mat = mat.data_ptr<int32_t>();
    d.mul = mul.data_ptr<float>();
    d.lut = lut.data_ptr<float>();
    return d;
}

void check_csr(const torch::Tensor &rows, const torch::Tensor &cols, const torch::Tensor &vals, const torch::Tensor &vec,
               int num_rows, int width) {
    need(rows, "rows", torch::kInt32, vec);
    need(cols, "cols", torch::kInt32, vec);
    need(vals, "mat (CSR values)", torch::kFloat32, vec);
    TORCH_CHECK(num_rows == width, "num_rows=", num_rows, " must equal the packed matrix width ", width);
    TORCH_CHECK(rows.numel() == (int64_t)num_rows + 1, "rows must have num_rows+1 entries");
    TORCH_CHECK(cols.numel() == vals.numel(), "cols and vals differ in length");
}

void check_full(const torch::Tensor &full_rows, const torch::Tensor &fri, const torch::Tensor &vec, int64_t K) {
    need(full_rows, "full_rows", torch::kFloat32, vec);
    need(fri, "full_row_indices", torch::kInt32, vec);
    TORCH_CHECK(full_rows.dim() == 2 && full_rows.size(0) == K, "full_rows must be [in, topX]");
    TORCH_CHECK(fri.numel() == full_rows.size(1), "full_row_indices must have topX entries");
}

// ---- dense ------------------------------------------------------------------------------------
template <int BITS, bool BATCHED>
void dense(torch::Tensor vec, torch::Tensor mat, torch::Tensor mul, torch::Tensor lookup_table) {
    const at::cuda::OptionalCUDAGuard guard(device_of(vec));
    const Dense d = check_dense(BITS, vec, mat, mul, lookup_table, BATCHED);
    int rc;
    if (BITS == 3) rc = BATCHED ? sqllm_vecquant3matmul_nuq_perchannel_batched(d.vec, d.mat, d.mul, d.lut, d.height, d.width, d.batch, d.vec_height, cur_stream())
                                : sqllm_vecquant3matmul_nuq_perchannel(d.vec, d.mat, d.mul, d.lut, d.height, d.width, cur_stream());
    else rc = BATCHED ? sqllm_vecquant4matmul_nuq_perchannel_batched(d.vec, d.mat, d.mul, d.lut, d.height, d.width, d.batch, d.vec_height, cur_stream())
                      : sqllm_vecquant4matmul_nuq_perchannel(d.vec, d.mat, d.mul, d.lut, d.height, d.width, cur_stream());
    check_status(rc, "quant_cuda dense LUT matmul");
}

// ---- dense + CSR ------------------------------------------------------------------------------
template <int BITS, bool BATCHED>
void spmv(torch::Tensor rows, torch::Tensor cols, torch::Tensor mat, torch::Tensor vec, torch::Tensor mul, int num_rows,
          torch::Tensor matq, torch::Tensor lookup_table) {
    const at::cuda::OptionalCUDAGuard guard(device_of(vec));
    const Dense d = check_dense(BITS, vec, matq, mul, lookup_table, BATCHED);
    check_csr(rows, cols, mat, vec, num_rows, d.width);
    const int32_t *r = rows.data_ptr<int32_t>(), *c = cols.data_ptr<int32_t>();
    const float *v = mat.data_ptr<float>();
    int rc;
    if (BITS == 3) rc = BATCHED ? sqllm_vecquant3matmul_spmv_nuq_perchannel_batched(r, c, v, d.vec, d.mul, num_rows, d.mat, d.lut, d.height, d.width, d.batch, d.vec_height, cur_stream())
                                : sqllm_vecquant3matmul_spmv_nuq_perchannel(r, c, v, d.vec, d.mul, num_rows, d.mat, d.lut, d.height, d.width, cur_stream());
    else rc = BATCHED ? sqllm_vecquant4matmul_spmv_nuq_perchannel_batched(r, c, v, d.vec, d.mul, num_rows, d.mat, d.lut, d.height, d.width, d.batch, d.vec_height, cur_stream())
                      : sqllm_vecquant4matmul_spmv_nuq_perchannel(r, c, v, d.vec, d.mul, num_rows, d.mat, d.lut, d.height, d.width, cur_stream());
    check_status(rc, "quant_cuda LUT matmul + spmv");
}

// ---- dense + CSR + topX dense rows ------------------------------------------------------------
template <int BITS, bool BATCHED>
void hybrid(torch::Tensor rows, torch::Tensor cols, torch::Tensor mat, torch::Tensor vec, torch::Tensor full_rows,
            torch::Tensor full_row_indices, torch::Tensor mul, int num_rows, torch::Tensor matq, torch::Tensor lookup_table) {
    const at::cuda::OptionalCUDAGuard guard(device_of(vec));
    const Dense d = check_dense(BITS, vec, matq, mul, lookup_table, BATCHED);
    check_csr(rows, cols, mat, vec, num_rows, d.width);
    check_full(full_rows, full_row_indices, vec, d.vec_height);
    const int32_t *r = rows.data_ptr<int32_t>(), *c = cols.data_ptr<int32_t>(), *fi = full_row_indices.data_ptr<int32_t>();
    const float *v = mat.data_ptr<float>(), *fr = full_rows.data_ptr<float>();
    const int frh = (int)full_rows.size(0), frw = (int)full_rows.size(1);
    int rc;
    if (BITS == 3) rc = BATCHED ? sqllm_vecquant3matmul_spmv_hybrid_nuq_perchannel_batched(r, c, v, d.vec, fr, fi, d.mul, num_rows, d.mat, d.lut, d.height, d.width, frh, frw, d.batch, d.vec_height, cur_stream())
                                : sqllm_vecquant3matmul_spmv_hybrid_nuq_perchannel(r, c, v, d.vec, fr, fi, d.mul, num_rows, d.mat, d.lut, d.height, d.width, frh, frw, cur_stream());
    else rc = BATCHED ? sqllm_vecquant4matmul_spmv_hybrid_nuq_perchannel_batched(r, c, v, d.vec, fr, fi, d.mul, num_rows, d.mat, d.lut, d.height, d.width, frh, frw, d.batch, d.vec_height, cur_stream())
                      : sqllm_vecquant4matmul_spmv_hybrid_nuq_perchannel(r, c, v, d.vec, fr, fi, d.mul, num_rows, d.mat, d.lut, d.height, d.width, frh, frw, cur_stream());
    check_status(rc, "quant_cuda LUT matmul + spmv + dense rows");
}

// ---- fused module path ------------------------------------------------------------------------
// Workspace of the fused path: one per (device, stream), allocated on first use (so: before any graph capture on that stream -
// GraphedDecodeStep warms up for exactly this reason), at least 8 MB - every supported shape fits, it is never regrown in
// practice; if it ever is, the old one is kept alive for graphs that captured its address.  A workspace serialises the launches
// that use it: graphs captured on the SAME stream must not be replayed concurrently on different streams (they share it);
// capture them on different streams if they have to overlap.
std::mutex g_ws_mutex;
std::map<std::pair<int, void *>, torch::Tensor> g_ws;  // (device, stream) -> zero-initialised workspace
std::vector<torch::Tensor> g_ws_retired;               // outgrown workspaces: never freed, a captured CUDA graph may still point at them

torch::Tensor workspace_for(const torch::Tensor &like, size_t bytes) {
    std::lock_guard<std::mutex> lock(g_ws_mutex);
    const auto key = std::make_pair((int)like.get_device(), cur_stream());
    auto it = g_ws.find(key);
    if (it == g_ws.end() || (size_t)it->second.numel() < bytes) {
        // grow generously so that the allocation happens once (and never during graph capture of a later call)
        const size_t cap = std::max<size_t>(bytes, 8u << 20);
        torch::Tensor ws = torch::zeros({(int64_t)cap}, torch::TensorOptions().dtype(torch::kUInt8).device(like.device()));
        if (it != g_ws.end()) g_ws_retired.push_back(it->second);
        g_ws[key] = ws;
        return ws;
    }
    return it->second;
}

// shared argument checking / descriptor filling of the two fused entry points
void fill_fused_args(sqllm_lutgemv_args &a, const float *&bias_p, const torch::Tensor &x, const torch::Tensor &qweight,
                     const torch::Tensor &lookup_table, int bits, const c10::optional<torch::Tensor> &bias,
                     const c10::optional<torch::Tensor> &rows, const c10::optional<torch::Tensor> &cols,
                     const c10::optional<torch::Tensor> &vals, const c10::optional<torch::Tensor> &full_rows,
                     const c10::optional<torch::Tensor> &full_row_indices) {
    TORCH_CHECK(x.is_cuda() && x.is_contiguous(), "x must be a contiguous CUDA tensor");
    TORCH_CHECK(x.scalar_type() == torch::kFloat16 || x.scalar_type() == torch::kFloat32, "x must be fp16 or fp32");
    TORCH_CHECK(bits == 3 || bits == 4, "bits must be 3 or 4");
    need(qweight, "qweight", torch::kInt32, x);
    need(lookup_table, "lookup_table", torch::kFloat32, x);
    TORCH_CHECK(qweight.dim() == 2 && qweight.size(0) % bits == 0, "qweight must be [in/32*bits, out]");
    memset(&a, 0, sizeof(a));
    a.bits = bits;
    a.in_features = (int)(qweight.size(0) / bits * 32);
    a.out_features = (int)qweight.size(1);
    a.batch = 1;
    TORCH_CHECK(x.numel() == a.in_features, "x has ", x.numel(), " elements, expected in_features=", a.in_features);
    TORCH_CHECK(lookup_table.numel() == (int64_t)a.out_features * (1 << bits), "lookup_table must be [out, 2^bits]");
    a.qweight = qweight.data_ptr<int32_t>();
    a.lookup_table = lookup_table.data_ptr<float>();
    bias_p = nullptr;
    if (bias.has_value() && bias->defined()) {
        need(*bias, "bias", torch::kFloat32, x);
        TORCH_CHECK(bias->numel() == a.out_features, "bias must have out_features elements");
        bias_p = bias->data_ptr<float>();
    }
    if (rows.has_value() && rows->defined()) {
        TORCH_CHECK(cols.has_value() && vals.has_value(), "rows given without cols / vals");
        check_csr(*rows, *cols, *vals, x, a.out_features, a.out_features);
        a.rows = rows->data_ptr<int32_t>();
        a.cols = cols->data_ptr<int32_t>();
        a.vals = vals->data_ptr<float>();
    }
    if (full_rows.has_value() && full_rows->defined() && full_rows->numel() > 0) {
        TORCH_CHECK(full_row_indices.has_value(), "full_rows given without full_row_indices");
        check_full(*full_rows, *full_row_indices, x, a.in_features);
        a.full_rows = full_rows->data_ptr<float>();
        a.full_row_indices = full_row_indices->data_ptr<int32_t>();
        a.topX = (int)full_rows->size(1);
    }
}

// y = bias + LUT-GEMV(x) [+ CSR] [+ dense rows]; x fp16/fp32 with numel == in; returns [out] in x's dtype
// (QuantLinearLUT.forward's matvec branch, squeezellm/quant.py:212-312, in one launch).
torch::Tensor lutgemv_fused(torch::Tensor x, torch::Tensor qweight, torch::Tensor lookup_table, int bits,
                            c10::optional<torch::Tensor> bias, c10::optional<torch::Tensor> rows,
                            c10::optional<torch::Tensor> cols, c10::optional<torch::Tensor> vals,
                            c10::optional<torch::Tensor> full_rows, c10::optional<torch::Tensor> full_row_indices) {
    const at::cuda::OptionalCUDAGuard guard(device_of(x));
    sqllm_lutgemv_args a;
    const float *bias_p;
    fill_fused_args(a, bias_p, x, qweight, lookup_table, bits, bias, rows, cols, vals, full_rows, full_row_indices);
    const size_t need_ws = sqllm_workspace_bytes(bits, a.in_features, a.out_features, a.topX);
    TORCH_CHECK(need_ws > 0, "sqllm_workspace_bytes failed: ", sqllm_last_error());
    torch::Tensor ws = workspace_for(x, need_ws);
    torch::Tensor y = torch::empty({(int64_t)a.out_features}, x.options());
    const int half = x.scalar_type() == torch::kFloat16;
    const int rc = sqllm_lutgemv_fused(&a, x.data_ptr(), half, y.data_ptr(), half, bias_p, ws.data_ptr(), (size_t)ws.numel(), cur_stream());
    check_status(rc, "quant_cuda.lutgemv_fused");
    return y;
}

// Column shard with the exchange built in (include/sqllm_b200.h, sqllm_lutgemv_fused_exchange): the result is written into every
// rank's symmetric arena; nothing is returned.  peer_base: address of the device array of arena base addresses.
void lutgemv_fused_exchange(torch::Tensor x, torch::Tensor qweight, torch::Tensor lookup_table, int bits,
                            c10::optional<torch::Tensor> bias, c10::optional<torch::Tensor> rows,
                            c10::optional<torch::Tensor> cols, c10::optional<torch::Tensor> vals,
                            c10::optional<torch::Tensor> full_rows, c10::optional<torch::Tensor> full_row_indices,
                            int64_t peer_base, int64_t out_offset, int64_t flag_offset, int64_t state_offset, int64_t error_offset,
                            int world, int rank, int members, int out_features_full) {
    const at::cuda::OptionalCUDAGuard guard(device_of(x));
    sqllm_lutgemv_args a;
    const float *bias_p;
    fill_fused_args(a, bias_p, x, qweight, lookup_table, bits, bias, rows, cols, vals, full_rows, full_row_indices);
    const size_t need_ws = sqllm_workspace_bytes(bits, a.in_features, a.out_features, a.topX);
    TORCH_CHECK(need_ws > 0, "sqllm_workspace_bytes failed: ", sqllm_last_error());
    torch::Tensor ws = workspace_for(x, need_ws);
    sqllm_exchange xc;
    memset(&xc, 0, sizeof(xc));
    xc.world = world; xc.rank = rank; xc.members = members; xc.out_features_full = out_features_full;
    xc.peer_base = reinterpret_cast<const uint64_t *>(peer_base);
    xc.out_offset = (size_t)out_offset; xc.flag_offset = (size_t)flag_offset; xc.state_offset = (size_t)state_offset; xc.error_offset = (size_t)error_offset;
    const int half = x.scalar_type() == torch::kFloat16;
    const int rc = sqllm_lutgemv_fused_exchange(&a, x.data_ptr(), half, half, bias_p, ws.data_ptr(), (size_t)ws.numel(), &xc, cur_stream());
    check_status(rc, "quant_cuda.lutgemv_fused_exchange");
}


// ---- sequences (include/sqllm_b200.h, sqllm_sequence_*): one persistent launch for a list of dependent fused matvecs -----------
// items: list of tuples (qweight, lookup_table, bits, bias|None, rows|None, cols|None, vals|None, full_rows|None, full_row_indices|None,
//                        x_from, x_offset, x_ext|None, members, out_features_full)
// exports: list of (item index, fp16 destination tensor of the item's full output length).  The caller keeps every tensor alive for the
// life of the handle (squeezellm_b200.runtime.DecodeSequence does).  peer_base / arena: several GPUs only (0 / None otherwise).
int64_t sequence_create(py::list items, py::list exports, const std::string &lut_mode, int world, int rank,
                        c10::optional<torch::Tensor> arena, int64_t peer_base) {
    TORCH_CHECK(lut_mode == "exact" || lut_mode == "fp16", "lut mode must be 'exact' or 'fp16'");
    const int n = (int)items.size();
    TORCH_CHECK(n > 0, "sequence_create: no items");
    std::vector<sqllm_seq_item> its(n);
    c10::optional<torch::Tensor> first;
    for (int i = 0; i < n; ++i) {
        py::tuple t = items[i].cast<py::tuple>();
        TORCH_CHECK(t.size() == 14, "sequence item ", i, ": expected a 14-tuple");
        auto opt = [&](int k) -> c10::optional<torch::Tensor> {
            if (t[k].is_none()) return c10::nullopt;
            return t[k].cast<torch::Tensor>();
        };
        torch::Tensor qweight = t[0].cast<torch::Tensor>(), lut = t[1].cast<torch::Tensor>();
        const int bits = t[2].cast<int>();
        sqllm_seq_item &it = its[i];
        memset(&it, 0, sizeof(it));
        it.x_from = t[9].cast<int>();
        it.x_offset = t[10].cast<int>();
        it.members = t[12].cast<int>();
        it.out_features_full = t[13].cast<int>();
        TORCH_CHECK(qweight.is_cuda() && qweight.dim() == 2 && (bits == 3 || bits == 4), "sequence item ", i, ": qweight must be a packed CUDA matrix");
        const int K = (int)(qweight.size(0) / bits * 32);
        torch::Tensor xs;  // what the shared checks look at (device, dtype, numel): the external input, or a stand-in of the right length
        if (it.x_from < 0) {
            TORCH_CHECK(!t[11].is_none(), "sequence item ", i, ": x_from = -1 needs x_ext");
            xs = t[11].cast<torch::Tensor>();
            TORCH_CHECK(xs.scalar_type() == torch::kFloat16, "sequence item ", i, ": x_ext must be fp16");
        } else {
            xs = torch::empty({(int64_t)K}, torch::TensorOptions().dtype(torch::kFloat16).device(qweight.device()));
        }
        const float *bias_p = nullptr;
        fill_fused_args(it.a, bias_p, xs, qweight, lut, bits, opt(3), opt(4), opt(5), opt(6), opt(7), opt(8));
        if (it.x_from < 0) it.x_ext = xs.data_ptr();
        it.bias = bias_p;
        if (!first.has_value()) first = qweight;
    }
    const at::cuda::OptionalCUDAGuard guard(device_of(*first));
    const int ne = (int)exports.size();
    std::vector<int> ex_items(std::max(1, ne));
    std::vector<void *> ex_dst(std::max(1, ne));
    for (int e = 0; e < ne; ++e) {
        py::tuple t = exports[e].cast<py::tuple>();
        ex_items[e] = t[0].cast<int>();
        torch::Tensor d = t[1].cast<torch::Tensor>();
        TORCH_CHECK(d.is_cuda() && d.is_contiguous() && d.scalar_type() == torch::kFloat16, "export ", e, ": destination must be a contiguous fp16 CUDA tensor");
        TORCH_CHECK(ex_items[e] >= 0 && ex_items[e] < n, "export ", e, ": bad item index");
        const sqllm_seq_item &it = its[ex_items[e]];
        const int64_t len = (int64_t)(it.members > 0 ? it.members : 1) * (it.out_features_full > 0 ? it.out_features_full : it.a.out_features / std::max(1, it.members));
        TORCH_CHECK(d.numel() == len, "export ", e, ": destination has ", d.numel(), " elements, the item's output has ", len);
        ex_dst[e] = d.data_ptr();
    }
    sqllm_seq_options o;
    memset(&o, 0, sizeof(o));
    o.lut_mode = lut_mode == "fp16" ? SQLLM_LUT_FP16_PAIR : SQLLM_LUT_EXACT;
    o.world = world; o.rank = rank;
    if (arena.has_value() && arena->defined()) {
        o.arena = arena->data_ptr();
        o.arena_bytes = (size_t)arena->numel() * arena->element_size();
    }
    o.peer_base = reinterpret_cast<const uint64_t *>(peer_base);
    o.n_export = ne; o.export_items = ex_items.data(); o.export_dst = ex_dst.data();
    sqllm_sequence *h = nullptr;
    check_status(sqllm_sequence_create(its.data(), n, &o, &h), "quant_cuda.sequence_create");
    return reinterpret_cast<int64_t>(h);
}

torch::Tensor unpack_indices(torch::Tensor qweight, int bits) {
    const at::cuda::OptionalCUDAGuard guard(device_of(qweight));
    need(qweight, "qweight", torch::kInt32, qweight);
    TORCH_CHECK(bits == 3 || bits == 4, "bits must be 3 or 4");
    TORCH_CHECK(qweight.dim() == 2 && qweight.size(0) % bits == 0, "qweight must be [in/32*bits, out]");
    const int K = (int)(qweight.size(0) / bits * 32), N = (int)qweight.size(1);
    torch::Tensor idx = torch::empty({K, N}, torch::TensorOptions().dtype(torch::kUInt8).device(qweight.device()));
    check_status(sqllm_unpack_indices(bits, qweight.data_ptr<int32_t>(), K, N, idx.data_ptr<uint8_t>(), cur_stream()), "unpack_indices");
    return idx;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    m.doc() = "B200-native drop-in for SqueezeLLM's quant_cuda extension";
    // the reference's 12 symbols (squeezellm/quant_cuda.cpp:258-269), same names and positional order
    m.def("vecquant3matmul_nuq_perchannel", &dense<3, false>, "3-bit per-channel LUT matvec (accumulates into mul)");
    m.def("vecquant4matmul_nuq_perchannel", &dense<4, false>, "4-bit per-channel LUT matvec (accumulates into mul)");
    m.def("vecquant3matmul_nuq_perchannel_batched", &dense<3, true>, "3-bit per-channel LUT matmul, batched");
    m.def("vecquant4matmul_nuq_perchannel_batched", &dense<4, true>, "4-bit per-channel LUT matmul, batched");
    m.def("vecquant3matmul_spmv_nuq_perchannel", &spmv<3, false>, "3-bit LUT matvec + CSR outliers");
    m.def("vecquant4matmul_spmv_nuq_perchannel", &spmv<4, false>, "4-bit LUT matvec + CSR outliers");
    m.def("vecquant3matmul_spmv_nuq_perchannel_batched", &spmv<3, true>, "3-bit LUT matmul + CSR outliers, batched");
    m.def("vecquant4matmul_spmv_nuq_perchannel_batched", &spmv<4, true>, "4-bit LUT matmul + CSR outliers, batched");
    m.def("vecquant3matmul_spmv_hybrid_nuq_perchannel", &hybrid<3, false>, "3-bit LUT matvec + CSR + dense rows");
    m.def("vecquant4matmul_spmv_hybrid_nuq_perchannel", &hybrid<4, false>, "4-bit LUT matvec + CSR + dense rows");
    m.def("vecquant3matmul_spmv_hybrid_nuq_perchannel_batched", &hybrid<3, true>, "3-bit LUT matmul + CSR + dense rows, batched");
    m.def("vecquant4matmul_spmv_hybrid_nuq_perchannel_batched", &hybrid<4, true>, "4-bit LUT matmul + CSR + dense rows, batched");
    // additions
    m.def("lutgemv_fused", &lutgemv_fused, "fused QuantLinearLUT matvec: fp16/fp32 x -> y (bias, CSR, dense rows), one launch",
          py::arg("x"), py::arg("qweight"), py::arg("lookup_table"), py::arg("bits"), py::arg("bias") = py::none(),
          py::arg("rows") = py::none(), py::arg("cols") = py::none(), py::arg("vals") = py::none(),
          py::arg("full_rows") = py::none(), py::arg("full_row_indices") = py::none());
    m.def("lutgemv_fused_exchange", &lutgemv_fused_exchange,
          "fused matvec of a column shard that stores its result into every rank's symmetric arena (NVLink peer memory) and waits for the peers'",
          py::arg("x"), py::arg("qweight"), py::arg("lookup_table"), py::arg("bits"), py::arg("bias"), py::arg("rows"), py::arg("cols"),
          py::arg("vals"), py::arg("full_rows"), py::arg("full_row_indices"), py::arg("peer_base"), py::arg("out_offset"),
          py::arg("flag_offset"), py::arg("state_offset"), py::arg("error_offset"), py::arg("world"), py::arg("rank"), py::arg("members"),
          py::arg("out_features_full"));
    m.def("sequence_create", &sequence_create, "one persistent launch for a list of dependent fused matvecs (see squeezellm_b200.runtime.DecodeSequence)",
          py::arg("items"), py::arg("exports"), py::arg("lut_mode") = "exact", py::arg("world") = 1, py::arg("rank") = 0,
          py::arg("arena") = py::none(), py::arg("peer_base") = 0);
    m.def("sequence_arena_bytes", [](py::list lens) {
              size_t off = 0;
              for (auto l : lens) off += ((size_t)l.cast<int64_t>() * 4 + 127) / 128 * 128;
              return (int64_t)off;
          }, "arena bytes for items with these full output lengths");
    m.def("sequence_run", [](int64_t h) { check_status(sqllm_sequence_run(reinterpret_cast<sqllm_sequence *>(h), cur_stream()), "quant_cuda.sequence_run"); },
          "run the sequence on the current stream (capturable)");
    m.def("sequence_error", [](int64_t h) {
              const int rc = sqllm_sequence_error(reinterpret_cast<sqllm_sequence *>(h), cur_stream());
              TORCH_CHECK(rc >= 0, "sequence_error: ", sqllm_last_error());
              return rc == 1;
          }, "True if a bounded in-kernel wait of the sequence ever timed out (synchronises the current stream)");
    m.def("sequence_reset_error", [](int64_t h) { check_status(sqllm_sequence_reset_error(reinterpret_cast<sqllm_sequence *>(h), cur_stream()), "quant_cuda.sequence_reset_error"); },
          "clear the sequence's error word on the current stream");
    m.def("sequence_destroy", [](int64_t h) { sqllm_sequence_destroy(reinterpret_cast<sqllm_sequence *>(h)); });
    m.def("unpack_indices", &unpack_indices, "GPU unpack of the packed indices -> uint8 [in, out] (test hook)");
    m.def("abi_version", []() { return sqllm_abi_version(); });
    m.def("set_deterministic", [](bool on) { sqllm_set_deterministic(on ? 1 : 0); },
          "fused path: True = bit-reproducible fixed-order reduction, False (default) = red.add accumulation");
    m.def("set_lut_mode", [](const std::string &mode) {
              TORCH_CHECK(mode == "exact" || mode == "fp16", "lut mode must be 'exact' or 'fp16' (got '", mode, "')");
              sqllm_set_lut_mode(mode == "fp16" ? SQLLM_LUT_FP16_PAIR : SQLLM_LUT_EXACT);
          },
          "fused path: 'exact' (default) = fp32 codebook as stored; 'fp16' = centroids rounded to fp16, pair tables + fp16 x fp16 -> fp32 FMAs "
          "(only taken for fp16 x)");
    m.def("get_lut_mode", []() { return std::string(sqllm_get_lut_mode() == SQLLM_LUT_FP16_PAIR ? "fp16" : "exact"); });
    m.def("workspace_error", []() {
              // error word of the current stream's fused-path workspace on the current device (synchronises the stream)
              int dev = 0;
              C10_CUDA_CHECK(cudaGetDevice(&dev));
              torch::Tensor ws;
              {
                  std::lock_guard<std::mutex> lock(g_ws_mutex);
                  auto it = g_ws.find(std::make_pair(dev, cur_stream()));
                  if (it == g_ws.end()) return false;
                  ws = it->second;
              }
              const int rc = sqllm_workspace_error(ws.data_ptr(), cur_stream());
              TORCH_CHECK(rc >= 0, "workspace_error: ", sqllm_last_error());
              return rc == 1;
          },
          "True if a bounded in-kernel wait of the fused path ever timed out on this stream's workspace (results are then incomplete)");
    m.def("sm_count", []() { return sqllm_device_sm_count(); });
    // limits of lutgemv_fused, lutgemv_fused_exchange and sequence_create (the 12 accumulate symbols have neither)
    m.attr("MAX_TOPX_FUSED") = SQLLM_MAX_TOPX_FUSED;
    m.attr("MAX_N_FUSED") = SQLLM_MAX_N_FUSED;
}
