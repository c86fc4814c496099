// lutgemm_batched.cuh - the six *_batched symbols done properly (SURVEY.md 8(f) row 3).  Included by lutgemv_kernels.cu inside its
// anonymous namespace.
//
// Reference: VecQuant{3,4}MatMulKernelNUQPerChannelBatched (squeezellm/quant_cuda_kernel.cu:884-1038) loops `for b` INSIDE every
// thread, one look-up and one FMA per (weight, batch row) with the weight word re-read from memory each time; SPMV_ATOMIC_BATCHED
// (:1061-1089) and DenseMatVecKernelBatched (:1127-1164) are further launches.  Round 1 of this repo launched the batch-1 kernel once
// per row.  Here:
//   * lutgemm_batched_kernel: a CTA owns a (64 columns x K-slab) weight tile and BT = 8 batch rows.  Every lane decodes its 4 columns
//     x 8 inputs ONCE per position (same PRMT-built shared-memory look-ups as the batch-1 kernel, exact fp32 table) and then runs the
//     32 decoded weights against its 8 batch rows: 256 FFMA per 32 look-ups, the look-up cost is amortised 8x and the kernel is
//     FP32-FMA bound.  x rows of the tile sit in shared memory (fp32), accumulators in registers, slab partial sums go out with one
//     red.add per (batch row, column) and CTA.  Larger batches are further CTAs (grid.z) re-reading the tile from L2.
//   * csr_batched_kernel / dense_rows_batched_kernel: the outlier terms, one thread per (batch row, output channel | dense row column).
// Results accumulate into `mul` (the reference's contract: the caller pre-fills zeros or bias, quant.py:316-318).
#pragma once

namespace batched {

constexpr int BT = 8;          // batch rows per CTA tile
constexpr int BW = 8;          // warps per CTA
constexpr int BTHREADS = BW * 32;

template <int BITS>
struct CB {
    static constexpr int L = 1 << BITS;
    static constexpr int TAB = L * STRIP * 4;      // 4 KB / 2 KB, aligned to its size
    static constexpr int ROWS = BITS == 4 ? 1 : 3;
    static constexpr int XU = BITS == 4 ? 8 : 32;  // inputs per unit
};

struct PB {
    const uint32_t *qw;
    const float *lut;
    const float *x;   // [B][K]
    float *mul;       // [B][N]
    int K, N, B, R;   // R = units per strip
    int ks;           // units per K-slab (even)
};

// 3-bit: value of input J (0..31) of a group from its three words; J is a compile-time constant, so every shift is an immediate
template <int J>
__device__ __forceinline__ float lut3_value(const uint32_t w0, const uint32_t w1, const uint32_t w2, const uint32_t lsv) {
    uint32_t f;
    if constexpr (J < 10) f = fld<3 * J>(w0);
    else if constexpr (J == 10) f = __funnelshift_r(w0, w1, 22);
    else if constexpr (J < 21) f = fld<1 + 3 * (J - 11)>(w1);
    else if constexpr (J == 21) f = __funnelshift_r(w1, w2, 23);
    else f = fld<2 + 3 * (J - 22)>(w2);
    return lds_f32((f & 0x700u) | lsv);
}

template <int J0, int U>
struct Dec3 {
    __device__ __forceinline__ static void run(float (&wv)[8], const uint32_t w0, const uint32_t w1, const uint32_t w2, const uint32_t lsv) {
        wv[U] = lut3_value<J0 + U>(w0, w1, w2, lsv);
        if constexpr (U + 1 < 8) Dec3<J0, U + 1>::run(wv, w0, w1, w2, lsv);
    }
};

// acc[b][t] += sum_k wv[t][k] * x_b[k] for the BT batch rows; x rows are BT consecutive rows of `xs` (row pitch xpitch bytes)
__device__ __forceinline__ void fma_rows(float (&acc)[BT][4], const float (&wv)[4][8], const uint32_t xaddr, const uint32_t xpitch) {
#pragma unroll
    for (int b = 0; b < BT; ++b) {
        const float4 xa = lds_v4(xaddr + b * xpitch), xb = lds_v4(xaddr + b * xpitch + 16);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            // the 8 products of this position first, then ONE add into the running sum: the running sum sees K/8/BW additions instead of
            // K/BW dependent FMAs, which keeps the batched results as close to the fp64 oracle as the batch-1 kernel's
            float d = wv[t][0] * xa.x;
            d = fmaf(wv[t][1], xa.y, d); d = fmaf(wv[t][2], xa.z, d); d = fmaf(wv[t][3], xa.w, d);
            d = fmaf(wv[t][4], xb.x, d); d = fmaf(wv[t][5], xb.y, d); d = fmaf(wv[t][6], xb.z, d); d = fmaf(wv[t][7], xb.w, d);
            acc[b][t] += d;
        }
    }
}

template <int BITS>
__global__ void __launch_bounds__(BTHREADS) lutgemm_batched_kernel(const PB p) {
    using C = CB<BITS>;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t tab = (raw + (uint32_t)C::TAB - 1u) & ~((uint32_t)C::TAB - 1u);
    unsigned char *sm = smem_raw + (tab - raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, i16 = lane & 15, jsel = lane >> 4;
    const int strip = blockIdx.x, u_lo = blockIdx.y * p.ks, u_hi = min(p.R, u_lo + p.ks), b0 = blockIdx.z * BT;
    const int nu = u_hi - u_lo, kslab = nu * C::XU;
    const uint32_t xpitch = (uint32_t)(kslab * 4 + 16);  // +16 bytes: the BT rows a lane reads start in different banks
    const uint32_t xs = tab + C::TAB;
    float *part = reinterpret_cast<float *>(sm + C::TAB + BT * xpitch);  // [BW][BT][STRIP]

    // ---- table (exact fp32, [value][slot], slot ((c & 3) << 4) | (c >> 2)) and the x rows of this tile ----
    for (int it = tid; it < STRIP * C::L / 4; it += BTHREADS) {
        const int c = it / (C::L / 4), q = it % (C::L / 4);
        const int col = strip * STRIP + c;
        const float4 v = col < p.N ? __ldg(reinterpret_cast<const float4 *>(p.lut + (size_t)col * C::L) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        const int slot = ((c & 3) << 4) | (c >> 2);
        const uint32_t a = tab + ((4 * q) * STRIP + slot) * 4;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v.x) : "memory");
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(a + STRIP * 4), "f"(v.y) : "memory");
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(a + 2 * STRIP * 4), "f"(v.z) : "memory");
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(a + 3 * STRIP * 4), "f"(v.w) : "memory");
    }
    {
        const int n16 = kslab / 4;  // 16-byte pieces per row
        for (int e = tid; e < BT * n16; e += BTHREADS) {
            const int b = e / n16, q = e - b * n16;
            const bool ok = b0 + b < p.B;
            cp_async16_clip(xs + b * xpitch + 16 * q, p.x + (ok ? (size_t)(b0 + b) * p.K + (size_t)u_lo * C::XU + 4 * q : 0), ok ? 16 : 0);
        }
        cp_async_commit();
        cp_async_wait_all();
    }
    __syncthreads();

    float acc[BT][4];
#pragma unroll
    for (int b = 0; b < BT; ++b)
#pragma unroll
        for (int t = 0; t < 4; ++t) acc[b][t] = 0.f;
    uint32_t l[4];
    const uint32_t tb_hi = BITS == 4 ? (tab & 0xFFFF0000u) : tab;
#pragma unroll
    for (int t = 0; t < 4; ++t) l[t] = tb_hi | (uint32_t)((((t ^ jsel) << 4) | i16) << 2);
    const uint32_t segc = ((tab >> 8) & 0xF0u) * 0x01010101u;
    const int col0 = strip * STRIP + 4 * i16;
    const bool cvalid = col0 < p.N;

    // positions: warp w takes unit pairs u_lo + 2w + jsel, step 2*BW; words are prefetched one position ahead
    int u = 2 * warp + jsel;
    auto load_unit = [&](int uu, uint4 (&w)[C::ROWS]) {
        const uint32_t *src = p.qw + (size_t)((u_lo + uu) * C::ROWS) * p.N + col0;
#pragma unroll
        for (int r = 0; r < C::ROWS; ++r) w[r] = (uu < nu && cvalid) ? ldg_stream(src + (size_t)r * p.N) : make_uint4(0u, 0u, 0u, 0u);
    };
    uint4 cur[C::ROWS], nxt[C::ROWS];
    load_unit(u, cur);
    for (; u - jsel < nu; u += 2 * BW) {   // warp-uniform bound (nu is even: a pair never straddles the end)
        load_unit(u + 2 * BW, nxt);
        const uint32_t xaddr = xs + (uint32_t)(u * C::XU * 4);
        if constexpr (BITS == 4) {
            const uint4 q = cur[0];
            const uint32_t w[4] = {jsel ? q.y : q.x, jsel ? q.x : q.y, jsel ? q.w : q.z, jsel ? q.z : q.w};
            float wv[4][8];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const uint32_t E = (w[t] & 0x0F0F0F0Fu) | segc;
                const uint32_t O = ((w[t] >> 4) & 0x0F0F0F0Fu) | segc;
                wv[t][0] = lds_f32(__byte_perm(E, l[t], 0x7604)); wv[t][1] = lds_f32(__byte_perm(O, l[t], 0x7604));
                wv[t][2] = lds_f32(__byte_perm(E, l[t], 0x7614)); wv[t][3] = lds_f32(__byte_perm(O, l[t], 0x7614));
                wv[t][4] = lds_f32(__byte_perm(E, l[t], 0x7624)); wv[t][5] = lds_f32(__byte_perm(O, l[t], 0x7624));
                wv[t][6] = lds_f32(__byte_perm(E, l[t], 0x7634)); wv[t][7] = lds_f32(__byte_perm(O, l[t], 0x7634));
            }
            fma_rows(acc, wv, xaddr, xpitch);
        } else {
            const uint32_t a[4] = {jsel ? cur[0].y : cur[0].x, jsel ? cur[0].x : cur[0].y, jsel ? cur[0].w : cur[0].z, jsel ? cur[0].z : cur[0].w};
            const uint32_t b[4] = {jsel ? cur[1].y : cur[1].x, jsel ? cur[1].x : cur[1].y, jsel ? cur[1].w : cur[1].z, jsel ? cur[1].z : cur[1].w};
            const uint32_t c[4] = {jsel ? cur[2].y : cur[2].x, jsel ? cur[2].x : cur[2].y, jsel ? cur[2].w : cur[2].z, jsel ? cur[2].z : cur[2].w};
            float wv[4][8];
#pragma unroll
            for (int t = 0; t < 4; ++t) Dec3<0, 0>::run(wv[t], a[t], b[t], c[t], l[t]);
            fma_rows(acc, wv, xaddr, xpitch);
#pragma unroll
            for (int t = 0; t < 4; ++t) Dec3<8, 0>::run(wv[t], a[t], b[t], c[t], l[t]);
            fma_rows(acc, wv, xaddr + 32, xpitch);
#pragma unroll
            for (int t = 0; t < 4; ++t) Dec3<16, 0>::run(wv[t], a[t], b[t], c[t], l[t]);
            fma_rows(acc, wv, xaddr + 64, xpitch);
#pragma unroll
            for (int t = 0; t < 4; ++t) Dec3<24, 0>::run(wv[t], a[t], b[t], c[t], l[t]);
            fma_rows(acc, wv, xaddr + 96, xpitch);
        }
#pragma unroll
        for (int r = 0; r < C::ROWS; ++r) cur[r] = nxt[r];
    }

    // ---- slab sums: fold the two half-warps (lane (i, j=1) holds column t^1 in slot t), one partial row per warp, then one red.add per (b, column)
#pragma unroll
    for (int b = 0; b < BT; ++b) {
        const float v0 = __shfl_xor_sync(0xffffffffu, acc[b][1], 16), v1 = __shfl_xor_sync(0xffffffffu, acc[b][0], 16);
        const float v2 = __shfl_xor_sync(0xffffffffu, acc[b][3], 16), v3 = __shfl_xor_sync(0xffffffffu, acc[b][2], 16);
        if (jsel == 0)
            *reinterpret_cast<float4 *>(part + ((warp * BT + b) * STRIP + 4 * i16)) = make_float4(acc[b][0] + v0, acc[b][1] + v1, acc[b][2] + v2, acc[b][3] + v3);
    }
    __syncthreads();
    for (int e = tid; e < BT * STRIP; e += BTHREADS) {
        const int b = e / STRIP, c = e - b * STRIP;
        float tot = 0.f;
#pragma unroll
        for (int w = 0; w < BW; ++w) tot += part[(w * BT + b) * STRIP + c];
        const int col = strip * STRIP + c;
        if (b0 + b < p.B && col < p.N) atomicAdd(p.mul + (size_t)(b0 + b) * p.N + col, tot);
    }
}

// CSR outliers for a batch: thread = (output channel, batch row); the row's (col, val) pairs are read by all threads of the block
// row at once (broadcast), x is gathered per batch row.  nnz * B FMAs in total - 0.45 % of the dense work.
__global__ void csr_batched_kernel(const int *__restrict__ rows, const int *__restrict__ cols, const float *__restrict__ vals,
                                   const float *__restrict__ x, float *__restrict__ mul, int K, int N, int B) {
    const int row = blockIdx.x * blockDim.y + threadIdx.y;
    if (row >= N) return;
    const int e0 = __ldg(rows + row), e1 = __ldg(rows + row + 1);
    for (int b = blockIdx.y * blockDim.x + threadIdx.x; b < B; b += gridDim.y * blockDim.x) {
        const float *xb = x + (size_t)b * K;
        float a = 0.f;
        for (int e = e0; e < e1; ++e) a += __ldg(vals + e) * __ldg(xb + __ldg(cols + e));  // storage order, like the oracle
        if (e1 > e0) atomicAdd(mul + (size_t)b * N + row, a);
    }
}

// topX dense rows for a batch: mul[b][fri[j]] += sum_k full_rows[k][j] * x[b][k].  One CTA per batch row; thread = (k-slice, dense row j):
// 256 / w slices of K walk their part with four independent fp32 chains, the slices' sums are added in fixed order through shared
// memory (deterministic), one atomicAdd per (b, j).  (First build: one thread per (b, j) walking all K terms in fp64 - 0.37 ms of pure
// latency whatever the batch, 3x SLOWER than the reference's kernels at batch 16: profiles/r02_batched_vs_reference_kernel.jsonl.)
// Rows go in blocks of w <= 64 (grid.y = ceil(topX / w)), so every row has at least 256 / 64 = 4 k-slices: a layer with hundreds of dense
// rows keeps its fp32 chains K / 16 long instead of K / 4.  The rows of the last block past topX idle.
__global__ void dense_rows_batched_kernel(const float *__restrict__ full_rows, const int *__restrict__ fri, int topX, int w,
                                          const float *__restrict__ x, float *__restrict__ mul, int K, int N, int B) {
    __shared__ float part[256];
    const int b = blockIdx.x, nsl = blockDim.x / w;
    const int jl = threadIdx.x % w, j = blockIdx.y * w + jl, sl = threadIdx.x / w;
    const float *xb = x + (size_t)b * K;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    const int per = (K + nsl - 1) / nsl, k0 = sl * per, k1 = j < topX ? min(K, k0 + per) : k0;
    int k = k0;
    for (; k + 3 < k1; k += 4) {
        a0 = fmaf(__ldg(full_rows + (size_t)k * topX + j), __ldg(xb + k), a0);
        a1 = fmaf(__ldg(full_rows + (size_t)(k + 1) * topX + j), __ldg(xb + k + 1), a1);
        a2 = fmaf(__ldg(full_rows + (size_t)(k + 2) * topX + j), __ldg(xb + k + 2), a2);
        a3 = fmaf(__ldg(full_rows + (size_t)(k + 3) * topX + j), __ldg(xb + k + 3), a3);
    }
    for (; k < k1; ++k) a0 = fmaf(__ldg(full_rows + (size_t)k * topX + j), __ldg(xb + k), a0);
    part[threadIdx.x] = (a0 + a1) + (a2 + a3);
    __syncthreads();
    if (sl == 0 && j < topX) {
        float t = 0.f;
        for (int i = 0; i < nsl; ++i) t += part[i * w + jl];
        const int c = __ldg(fri + j);
        if (c >= 0 && c < N) atomicAdd(mul + (size_t)b * N + c, t);
    }
}

}  // namespace batched
