// lutgemv_kernels.cu - B200 (sm_100a) dense-and-sparse LUT GEMV, written from scratch.
//
// Replaces (behaviour, not code) squeezellm/quant_cuda_kernel.cu of SqueezeAILab/SqueezeLLM:
//   VecQuant{3,4}MatMulKernelNUQPerChannel[Batched]  (:741-1038)   LUT GEMV
//   SPMV_ATOMIC[_BATCHED]                            (:1040-1089)  CSR outliers
//   DenseMatVecKernel[Batched]                       (:1092-1164)  topX dense rows
// and the 12 host launchers (:132-738), behind the C ABI of include/sqllm_b200.h.
//
// Design (DESIGN.md has the full story and the measurements):
//   * ONE launch per GEMV.  The [units x strips] iteration space (unit = one packed row for 4-bit,
//     one 3-row / 32-input group for 3-bit; strip = 64 output columns) is flattened strip-major and
//     cut into equal contiguous chunks, one per CTA (stream-K): every SM gets the same number of
//     bytes whatever the shape.  A CTA touches at most MAXSEG strips.
//   * Warp roles (default build, SQLLM_LDG=2): 8 consumer warps + 1 sparse warp, 72 registers, 3 CTAs per SM.
//       - consumers: each lane streams its own 16 bytes per unit row with cp.async into a private ring in shared memory,
//         PF positions ahead (the first PF before the programmatic dependency on the previous kernel resolves - PDL - so
//         the weight traffic of GEMV n+1 overlaps the tail of GEMV n), pulls the word-quad into registers and turns every
//         4-bit index into an LDS address with a single PRMT (the per-strip LUT is staged transposed
//         [value][column-slot] in a 4 KB aligned table so that every lane owns one shared-memory bank: conflict-free
//         gathers); products go into packed fma.rn.f32x2 accumulators.  No tensor cores: this is a gather-bound GEMV.
//         (SQLLM_LDG=1: register ring fed by LDG.128; SQLLM_LDG=0: TMA producer warp + mbarrier ring - measured, not faster.)
//       - sparse warp: CSR rows spread evenly over all CTAs, staged with 16-byte cp.async, x gathered in batches,
//         per-row sums in storage order; plus a k-slice of the topX dense rows.
//   * Only the slice of x a CTA needs is staged (fp32, converted from fp16 on the way in).
//   * Flush: accumulate mode (the reference's 12 symbols; `mul` pre-filled by the caller) issues one red.add.f32 per
//     (CTA, column).  Fused mode (QuantLinearLUT.forward): fast (default) = red.add into a workspace accumulator, a
//     release counter, and the last CTAs of the grid convert / store y (optionally into every rank's peer-mapped arena:
//     the multi-GPU exchange); deterministic = per-strip partials + tickets, fixed summation order.
#include <cuda.h>  // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint, no -lcuda)
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "sqllm_b200.h"

namespace {

#ifndef SQLLM_NW
#define SQLLM_NW 8
#endif
#ifndef SQLLM_LDG
#define SQLLM_LDG 2   // 2: per-thread private cp.async ring in shared memory (default); 1: LDG.128 register ring; 0: TMA producer warp + mbarrier ring
#endif
#ifndef SQLLM_MINB4
#define SQLLM_MINB4 3   // resident CTAs per SM the register budget must allow (shared memory admits 3; at 4 the 56-register
                        // cap makes the compiler rematerialise table addresses inside the loop: 6-13 % slower, profiles/r01)
#endif
#ifndef SQLLM_MINB3
#define SQLLM_MINB3 3
#endif
#ifndef SQLLM_PF4
#define SQLLM_PF4 8   // 128-bit loads in flight per lane, 4-bit path (LDG / cp.async modes)
#endif
#ifndef SQLLM_PF3
#define SQLLM_PF3 3   // 3-row groups in flight per lane, 3-bit path (LDG / cp.async modes)
#endif
constexpr bool LDG_MODE = SQLLM_LDG != 0;   // no producer warp
constexpr bool CPA_MODE = SQLLM_LDG == 2;   // weights staged by each consumer thread into its own cp.async ring
constexpr int NW = SQLLM_NW;              // consumer warps per CTA (multiple of 8)
constexpr int WARP_PRODUCER = LDG_MODE ? -1 : NW;            // warp index of the TMA producer (TMA mode only)
constexpr int WARP_SPARSE = LDG_MODE ? NW : NW + 1;          // warp index of the CSR / dense-row warp
constexpr int THREADS = (NW + (LDG_MODE ? 1 : 2)) * 32;
constexpr int MAXSEG = 4;                 // strips a CTA may touch
constexpr int STRIP = 64;                 // output columns per strip (16 lanes x 4 columns)
constexpr int SU = 2 * NW;                // units per pipeline stage (one pair per consumer warp)
constexpr int CSR_CH = 1024;              // CSR elements staged per chunk
constexpr int SROWS_LD = 68;              // padded row-pointer slice per segment (65 used)
constexpr int MAX_TOPX_FUSED = SQLLM_MAX_TOPX_FUSED;
constexpr int HYB_R = 11;                 // dense rows: k-rows per lane slot requested before the dependency wait
constexpr int MAX_STRIPS = 16320;         // per-strip tickets in the workspace header (out_features <= 1,044,480)
constexpr int MAX_N_FUSED = SQLLM_MAX_N_FUSED;  // fused path: the scratch accumulator lives at a fixed place in the workspace
constexpr size_t WS_ACC_OFF = 65536;       // [64 KB, 64 KB + 4*MAX_N_FUSED): fp32 accumulator (zero between launches)
constexpr int MAX_GRID_V2 = 256;           // v2 runs one CTA per SM
constexpr size_t WS_HBOX_OFF = WS_ACC_OFF + (size_t)MAX_N_FUSED * 4;       // v2 mailboxes: [MAX_GRID_V2][64] x 8 bytes (partial strip sums)
constexpr size_t WS_CBOX_OFF = WS_HBOX_OFF + (size_t)MAX_GRID_V2 * 64 * 8;  // ... and [MAX_N_FUSED] x 8 bytes (outlier row sums); zero between launches
constexpr size_t WS_DBOX_OFF = WS_CBOX_OFF + (size_t)MAX_N_FUSED * 8;          // ... and [MAX_TOPX_FUSED][MAX_GRID_V2] x 8 bytes (dense-row parts, one per contributing CTA)
constexpr size_t WS_HEADER = WS_DBOX_OFF + (size_t)MAX_TOPX_FUSED * MAX_GRID_V2 * 8;  // tickets + accumulator + mailboxes: never shared with data of any shape
constexpr int MAX_NSTAGE = 16;            // weight stages per CTA (runtime count, fills the shared-memory budget)

struct Params {
    const uint32_t *qw;
    const float *lut;
    const void *x;      // fp32 or fp16 [K]
    void *out;          // accumulate mode: float* mul ; fused: fp32/fp16 y
    const float *bias;  // fused only, may be null
    const int *rows, *cols;
    const float *vals;
    const float *full_rows;
    const int *fri;
    int topX;
    int K, N;
    int R;        // units per strip
    int strips;
    int T;        // strips * R
    int chunk;    // units per CTA (even)
    int maxseg;   // strips a CTA of this launch can touch (sizes the LUT tables)
    int nstage;   // weight stages in the TMA ring
    int tma2d;    // 1: stages are fetched with 2-D tensor-map TMA boxes, 0: row-by-row bulk copies (odd shapes)
    int x_direct; // 1: x staged at its natural index (CTA covers whole strips), 0: compact, indexed by unit offset
    int xfloats;  // floats in the x staging buffer
    int hc;       // CTAs that take a slice of the dense rows
    int hrows;    // k-rows per such CTA
    int x_is_half, y_is_half;
    int maxc;     // max dense contributors per strip (fused)
    float *ws_part;   // [strips][maxc+1][64]
    int *ws_cnt;      // [strips]
    float *ws_hyb;    // [hc][topX]
    int *ws_hyb_cnt;  // [1]
    int has_csr;
    int has_stage;   // bytes of the shared-memory staging buffer: 0, CSR_CH*8 (CSR cols+vals) or CSR_CH*16 (+ dense-row partials, deterministic mode)
    int csr_al16;    // cols / vals are 16-byte aligned: stage them with 16-byte cp.async
    int csr_rpc;     // CSR rows (output channels) handled per CTA: rows are spread evenly over all CTAs
    float *ws_csr;   // [N] CSR row sums (deterministic fused mode)
    float *ws_acc;   // [N] fp32 accumulator, zero between launches (fast fused mode)
    // optional exchange (column-sharded layers): finishers store their slice into every rank's arena over NVLink
    int xw_world, xw_rank, xw_members, xw_nfull;   // xw_world == 0: no exchange
    const unsigned long long *xw_base;             // device array [world]: base address of every rank's symmetric arena
    unsigned long long xw_out_off, xw_flag_off, xw_state_off, xw_err_off;
    int nfin;        // fast fused mode: CTAs (the last ones of the grid) that share the final conversion
    int det;         // fused mode: 1 = deterministic per-strip tickets, 0 = red.add into ws_acc + one global ticket per CTA
    int dbg;                    // debug: 1 = skip the gather/FMA math, 2 = no work at all, 4 = skip LUT staging (SQLLM_DEBUG_FLAGS)
    unsigned long long *trace;  // debug timeline (only written when built with -DSQLLM_TRACE and non-null)
};

// ---- per-bit-width constants and the shared memory carve-up (offsets from a 4 KB aligned base) ---
template <int BITS>
struct Cfg {
    static constexpr int L = 1 << BITS;
    static constexpr int TAB = L * STRIP * 4;              // 4096 (w4) / 2048 (w3) bytes per strip table
    static constexpr int ROWS_PER_UNIT = BITS == 4 ? 1 : 3;
    static constexpr int XU = BITS == 4 ? 8 : 32;          // inputs per unit
    static constexpr int UNIT_BYTES = ROWS_PER_UNIT * STRIP * 4;
    static constexpr int STAGE_BYTES = SU * UNIT_BYTES;    // 4 KB (w4) / 12 KB (w3)
    // 2-D TMA box: BU units tall (w4: a whole stage of 16 rows; w3: 4 groups = 12 rows), 64 columns wide.
    // in_features % 128 == 0 (the reference's own precondition) makes every box lie inside one strip.
    static constexpr int BU = BITS == 4 ? SU : 4;
    static constexpr int BOX_ROWS = BU * ROWS_PER_UNIT;
    static constexpr int BOX_BYTES = BOX_ROWS * STRIP * 4;
    // cp.async mode: every consumer thread owns PF slots of POS_BYTES (its 4 columns of one unit), laid out [slot][row-in-unit][thread]
    static constexpr int PF = BITS == 4 ? SQLLM_PF4 : SQLLM_PF3;
    static constexpr int POS_BYTES = ROWS_PER_UNIT * 16;
    static constexpr int RING_BYTES = PF * NW * 32 * POS_BYTES;
    // layout: [tables maxseg*TAB][part maxseg][misc][x][csr stage][weight stages ...]
    __host__ __device__ static int off_part(int maxseg) { return maxseg * TAB; }
    __host__ __device__ static int off_misc(int maxseg) { return off_part(maxseg) + maxseg * NW * STRIP * 4; }
    // misc: 2 x MAX_NSTAGE mbarriers (256 B) + 16 ints (64 B) + dense-row totals float[maxseg + 1][MAX_TOPX_FUSED]
    __host__ __device__ static int off_x(int maxseg) { return off_misc(maxseg) + 256 + 64 + (maxseg + 1) * MAX_TOPX_FUSED * 4; }
    __host__ __device__ static int off_cstage(int maxseg, int xfloats) { return off_x(maxseg) + ((xfloats * 4 + 15) & ~15); }
    __host__ __device__ static int off_stage(int maxseg, int xfloats, int csr) {  // csr: bytes of staging (CSR 8 KB [+ dense-row partials 8 KB])
        return (off_cstage(maxseg, xfloats) + csr + 127) & ~127;
    }
    __host__ __device__ static int total(int maxseg, int xfloats, int csr, int nstage) {
        return 4096 + off_stage(maxseg, xfloats, csr) + (CPA_MODE ? RING_BYTES : nstage * STAGE_BYTES);
    }
};

// ---- small PTX helpers -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float lds_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ float4 lds_v4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint4 lds_u4(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint4 ldg_stream(const void *p) {  // read-once weights: no L1 allocation
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16_clip(uint32_t dst, const void *src, int src_bytes) {  // reads src_bytes (<= 16), zero-fills the rest
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_pending() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void ffma2(uint64_t &acc, uint64_t a, uint64_t b) {  // Blackwell packed fp32 FMA
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
__device__ __forceinline__ float sum2(uint64_t v) {
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
    return lo + hi;
}
__device__ __forceinline__ float warp_sum(float v) {  // fixed xor tree -> deterministic
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}
__device__ __forceinline__ float ldcg_f32(const float *p) { return __ldcg(p); }
// Ticket: one gpu-scope acq_rel atomic.  The release half publishes everything the calling thread wrote - and, by
// cumulativity, what the threads it synchronised with (bar.sync / __syncwarp) wrote before that barrier; the acquire half makes
// the other contributors' published partials visible to whoever draws the last ticket (and, through the next barrier, to its
// whole group).  This replaces the fence / atomic / fence triple (~1 us per fence on a busy B200).
__device__ __forceinline__ int ticket_take(int *counter) {
    int old;
    asm volatile("atom.acq_rel.gpu.global.add.s32 %0, [%1], 1;" : "=r"(old) : "l"(counter) : "memory");
    return old;
}
#if defined(SQLLM_TRACE) || defined(SQLLM_DEBUG)
#define DBG(p) ((p).dbg)
#else
#define DBG(p) 0
#endif
#ifdef SQLLM_TRACE
__device__ __forceinline__ void trace_mark(unsigned long long *trace, int slot) {
    if (trace) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        trace[(size_t)blockIdx.x * 32 + slot] = t;
    }
}
#define TRACE(slot, cond) do { if (cond) trace_mark(p.trace, slot); } while (0)
#else
#define TRACE(slot, cond) do { } while (0)
#endif

// mbarrier / TMA bulk copy / PDL
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
#ifdef SQLLM_SPIN_WAIT
        asm volatile("{\n.reg .pred p;\nmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
#else
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
#endif
    } while (!ok);
}
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
__device__ __forceinline__ void tma_tile2d_g2s(uint32_t dst, const CUtensorMap *map, int col, int row, uint32_t bar, uint64_t pol) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
                 ::"r"(dst), "l"(map), "r"(col), "r"(row), "r"(bar), "l"(pol) : "memory");
}
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Maps a unit offset `o` (from the CTA's first unit) to (segment, unit-in-strip); advanced incrementally.
struct UnitIt {
    int o, rr, seg;
    __device__ __forceinline__ void init(int first, int r0, int R) {
        o = first;
        rr = r0 + first;
        seg = 0;
        while (rr >= R) { rr -= R; ++seg; }
    }
    __device__ __forceinline__ void advance(int step, int R) {
        o += step;
        rr += step;
        while (rr >= R) { rr -= R; ++seg; }
    }
};

// Walks, in order, the positions (unit pairs) one consumer warp owns: offset 2*warp + SU*p from the CTA's first unit.  Within a
// segment (= strip) consecutive positions are SU units apart, so callers keep running pointers and only `seek` at segment ends.
struct Cursor {
    int seg;   // current segment; == nseg when exhausted
    int left;  // positions left in this segment (including the current one)
    int rr;    // unit index inside the strip of the current position (the lane adds its own 0/1)
    __device__ __forceinline__ void seek(int from_seg, int warp2, int r0, int R, int len, int nseg) {
        for (int sg = from_seg; sg < nseg; ++sg) {
            const int b = sg == 0 ? 0 : sg * R - r0, e = min(len, (sg + 1) * R - r0);   // offsets [b, e) belong to segment sg
            const int pf = b <= warp2 ? 0 : (b - warp2 + SU - 1) / SU;                   // first position with offset >= b
            const int pl = e <= warp2 ? 0 : (e - warp2 + SU - 1) / SU;                   // positions with offset < e
            if (pl > pf) { seg = sg; left = pl - pf; rr = warp2 + SU * pf + r0 - sg * R; return; }
        }
        seg = nseg; left = 0; rr = 0;
    }
};

// =================================================================================================
// 4-bit: one 128-bit word-quad (4 columns x 8 inputs) -> 32 gathers + 16 packed FMAs.
//   E/O hold the even/odd nibbles of a word in separate bytes, already OR-ed with bits 12..15 of the
//   table address; PRMT then builds the complete LDS address: {ls.b3, ls.b2, E.b_n, ls.b0}.
// =================================================================================================
__device__ __forceinline__ void consume4(const uint4 q, const int jsel, const uint32_t lsb, const uint32_t segc,
                                         const uint32_t xaddr, uint64_t (&acc)[4]) {
    const float4 xa = lds_v4(xaddr), xb = lds_v4(xaddr + 16);
    const uint64_t x01 = pack2(xa.x, xa.y), x23 = pack2(xa.z, xa.w), x45 = pack2(xb.x, xb.y), x67 = pack2(xb.z, xb.w);
    // half-warp 1 walks its 4 columns in the order 1,0,3,2 so that the two half-warps never hit the same bank
    const uint32_t w[4] = {jsel ? q.y : q.x, jsel ? q.x : q.y, jsel ? q.w : q.z, jsel ? q.z : q.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const uint32_t E = (w[t] & 0x0F0F0F0Fu) | segc;
        const uint32_t O = ((w[t] >> 4) & 0x0F0F0F0Fu) | segc;
        const uint32_t l = lsb ^ (uint32_t)(t << 6);  // slot of column t (the lane's bank), see set_seg
        const float e0 = lds_f32(__byte_perm(E, l, 0x7604)), o0 = lds_f32(__byte_perm(O, l, 0x7604));
        const float e1 = lds_f32(__byte_perm(E, l, 0x7614)), o1 = lds_f32(__byte_perm(O, l, 0x7614));
        const float e2 = lds_f32(__byte_perm(E, l, 0x7624)), o2 = lds_f32(__byte_perm(O, l, 0x7624));
        const float e3 = lds_f32(__byte_perm(E, l, 0x7634)), o3 = lds_f32(__byte_perm(O, l, 0x7634));
        ffma2(acc[t], pack2(e0, o0), x01);
        ffma2(acc[t], pack2(e1, o1), x23);
        ffma2(acc[t], pack2(e2, o2), x45);
        ffma2(acc[t], pack2(e3, o3), x67);
    }
}

// =================================================================================================
// 3-bit: one group = 3 words per column = 32 inputs (10 | straddler | 10 | straddler | 10), the layout
// of squeezellm/quant.py:185-203.  Each index is moved to bits 8..10 (table row stride 256 B) by one
// shift (a funnel shift for the two straddlers) and merged with the lane's slot address by one LOP3.
// =================================================================================================
template <int SH>  // field at bit position SH of w -> bits 8..10
__device__ __forceinline__ uint32_t fld(uint32_t w) {
    if constexpr (SH < 8) return w << (8 - SH);
    else if constexpr (SH == 8) return w;
    else return w >> (SH - 8);
}
#define LK3(dst, word_expr, lsv) dst = lds_f32((((word_expr)) & 0x700u) | (lsv))

__device__ __forceinline__ void consume3_col(const uint32_t w0, const uint32_t w1, const uint32_t w2, const uint32_t lsv,
                                             const uint64_t (&xp)[16], uint64_t &acc) {
    float a, b;
    // inputs 0..9 from w0 (bits 3k), 10 straddles w0/w1
    LK3(a, fld<0>(w0), lsv);  LK3(b, fld<3>(w0), lsv);  ffma2(acc, pack2(a, b), xp[0]);
    LK3(a, fld<6>(w0), lsv);  LK3(b, fld<9>(w0), lsv);  ffma2(acc, pack2(a, b), xp[1]);
    LK3(a, fld<12>(w0), lsv); LK3(b, fld<15>(w0), lsv); ffma2(acc, pack2(a, b), xp[2]);
    LK3(a, fld<18>(w0), lsv); LK3(b, fld<21>(w0), lsv); ffma2(acc, pack2(a, b), xp[3]);
    LK3(a, fld<24>(w0), lsv); LK3(b, fld<27>(w0), lsv); ffma2(acc, pack2(a, b), xp[4]);
    LK3(a, __funnelshift_r(w0, w1, 22), lsv);            // input 10: bits 30,31 of w0 + bit 0 of w1
    LK3(b, fld<1>(w1), lsv);                             // input 11
    ffma2(acc, pack2(a, b), xp[5]);
    LK3(a, fld<4>(w1), lsv);  LK3(b, fld<7>(w1), lsv);  ffma2(acc, pack2(a, b), xp[6]);
    LK3(a, fld<10>(w1), lsv); LK3(b, fld<13>(w1), lsv); ffma2(acc, pack2(a, b), xp[7]);
    LK3(a, fld<16>(w1), lsv); LK3(b, fld<19>(w1), lsv); ffma2(acc, pack2(a, b), xp[8]);
    LK3(a, fld<22>(w1), lsv); LK3(b, fld<25>(w1), lsv); ffma2(acc, pack2(a, b), xp[9]);
    LK3(a, fld<28>(w1), lsv);                            // input 20
    LK3(b, __funnelshift_r(w1, w2, 23), lsv);            // input 21: bit 31 of w1 + bits 0,1 of w2
    ffma2(acc, pack2(a, b), xp[10]);
    LK3(a, fld<2>(w2), lsv);  LK3(b, fld<5>(w2), lsv);  ffma2(acc, pack2(a, b), xp[11]);
    LK3(a, fld<8>(w2), lsv);  LK3(b, fld<11>(w2), lsv); ffma2(acc, pack2(a, b), xp[12]);
    LK3(a, fld<14>(w2), lsv); LK3(b, fld<17>(w2), lsv); ffma2(acc, pack2(a, b), xp[13]);
    LK3(a, fld<20>(w2), lsv); LK3(b, fld<23>(w2), lsv); ffma2(acc, pack2(a, b), xp[14]);
    LK3(a, fld<26>(w2), lsv); LK3(b, fld<29>(w2), lsv); ffma2(acc, pack2(a, b), xp[15]);
}

template <int BITS> struct Words;
template <> struct Words<4> { uint4 a; };
template <> struct Words<3> { uint4 a, b, c; };

__device__ __forceinline__ void consume(const Words<4> &g, const int jsel, const uint32_t lsb, const uint32_t segc,
                                        const uint32_t (&)[4], const uint32_t xaddr, uint64_t (&acc)[4]) {
    consume4(g.a, jsel, lsb, segc, xaddr, acc);
}
__device__ __forceinline__ void consume(const Words<3> &g, const int jsel, const uint32_t, const uint32_t,
                                        const uint32_t (&lsv)[4], const uint32_t xaddr, uint64_t (&acc)[4]) {
    uint64_t xp[16];
#pragma unroll
    for (int v = 0; v < 8; ++v) {
        const float4 f = lds_v4(xaddr + 16 * v);
        xp[2 * v] = pack2(f.x, f.y);
        xp[2 * v + 1] = pack2(f.z, f.w);
    }
    const uint32_t a[4] = {jsel ? g.a.y : g.a.x, jsel ? g.a.x : g.a.y, jsel ? g.a.w : g.a.z, jsel ? g.a.z : g.a.w};
    const uint32_t b[4] = {jsel ? g.b.y : g.b.x, jsel ? g.b.x : g.b.y, jsel ? g.b.w : g.b.z, jsel ? g.b.z : g.b.w};
    const uint32_t c[4] = {jsel ? g.c.y : g.c.x, jsel ? g.c.x : g.c.y, jsel ? g.c.w : g.c.z, jsel ? g.c.z : g.c.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) consume3_col(a[t], b[t], c[t], lsv[t], xp, acc[t]);
}
__device__ __forceinline__ void gload_words(Words<4> &g, const uint32_t *q, size_t) { g.a = ldg_stream(q); }
__device__ __forceinline__ void gload_words(Words<3> &g, const uint32_t *q, size_t N) {
    g.a = ldg_stream(q);
    g.b = ldg_stream(q + N);
    g.c = ldg_stream(q + 2 * N);
}
__device__ __forceinline__ void zero_words(Words<4> &g) { g.a = make_uint4(0u, 0u, 0u, 0u); }
__device__ __forceinline__ void zero_words(Words<3> &g) { g.a = g.b = g.c = make_uint4(0u, 0u, 0u, 0u); }
__device__ __forceinline__ void load_words(Words<4> &g, uint32_t unit_addr) { g.a = lds_u4(unit_addr); }
__device__ __forceinline__ void load_words(Words<3> &g, uint32_t unit_addr) {
    g.a = lds_u4(unit_addr);
    g.b = lds_u4(unit_addr + STRIP * 4);
    g.c = lds_u4(unit_addr + 2 * STRIP * 4);
}

// ---- fused mode: who contributes to a strip, and the per-column final reduction ----------------------
__device__ __forceinline__ bool strip_has_hybrid(const Params &p, int strip) {
    if (!p.full_rows) return false;
    bool h = false;
    for (int j = 0; j < p.topX; ++j) {
        const int c = __ldg(p.fri + j);
        h |= (c >= 0 && c < p.N && c / STRIP == strip);
    }
    return h;
}
// Contributors that take a ticket on strip `strip` (deterministic fused mode): nd dense CTAs (stream-K), ncsr CTAs whose CSR row
// range touches the strip and - if a dense row lands in it - all hc dense-row contributors.
__device__ __forceinline__ int strip_contributors(const Params &p, int strip, int &nd, bool &hyb) {
    const int first = (int)(((long long)strip * p.R) / p.chunk);
    const int lastc = (int)((((long long)strip + 1) * p.R - 1) / p.chunk);
    nd = lastc - first + 1;
    hyb = strip_has_hybrid(p, strip);
    int ncsr = 0;
    if (p.rows) {
        const int c0 = strip * STRIP, c1 = min(p.N, c0 + STRIP) - 1;
        ncsr = c1 / p.csr_rpc - c0 / p.csr_rpc + 1;
    }
    return nd + ncsr + (hyb ? p.hc : 0);
}
// One warp: fixed-order totals of the dense-row partials ws_hyb[hc][topX] -> tot[topX] (shared memory).  All partials are
// pulled through the staging buffer in one go (one latency), then lanes = (slot, j) sum contributors slot, slot+nsl, ... and the
// slots are folded in fixed order: deterministic.  Callers guarantee every contributor has published (ticket) and fenced.
__device__ __forceinline__ void hybrid_totals(const Params &p, uint32_t stage_u32, const float *stage, float *tot, int lane) {
    const int tp = p.topX, tot_f = p.hc * tp;
    const int n16 = tot_f >> 2;  // ws_hyb and the staging buffer are 16-byte aligned
    for (int e = lane; e < n16; e += 32) cp_async16(stage_u32 + 16 * e, p.ws_hyb + 4 * e);
    for (int e = 4 * n16 + lane; e < tot_f; e += 32) cp_async4(stage_u32 + 4 * e, p.ws_hyb + e);
    cp_async_commit();
    cp_async_wait_all();
    __syncwarp();
    const int nsl = tp <= 16 ? 32 / tp : 1;
    for (int jb = 0; jb < (tp <= 16 ? 1 : tp); jb += 32) {
        const int sl = tp <= 16 ? lane / tp : 0, j = tp <= 16 ? lane - sl * tp : jb + lane;
        float t = 0.f;
        if (sl < nsl && j < tp)
            for (int b = sl; b < p.hc; b += nsl) t += stage[b * tp + j];
        for (int q = 1; q < nsl; ++q) {
            const float v = __shfl_sync(0xffffffffu, t, (j + q * tp) & 31);
            if (sl == 0) t += v;
        }
        if (sl == 0 && j < tp) tot[j] = t;
    }
    __syncwarp();
}
__device__ __forceinline__ void final_store(const Params &p, int strip, int c, int nd, const float *hyb_tot) {
    const int col = strip * STRIP + c;
    if (col >= p.N) return;
    const float *base = p.ws_part + (size_t)strip * p.maxc * STRIP + c;
    float tot = 0.f;
    for (int s = 0; s < nd; ++s) tot += ldcg_f32(base + s * STRIP);
    if (p.rows) tot += ldcg_f32(p.ws_csr + col);
    if (hyb_tot)
        for (int j = 0; j < p.topX; ++j)
            if (__ldg(p.fri + j) == col) tot += hyb_tot[j];
    if (p.bias) tot += p.bias[col];
    if (p.y_is_half) reinterpret_cast<__half *>(p.out)[col] = __float2half_rn(tot);
    else reinterpret_cast<float *>(p.out)[col] = tot;
}
// one warp takes a ticket on `strip` and, if it is the last contributor, reduces and stores the strip's 64 columns
__device__ __forceinline__ void warp_ticket(const Params &p, int strip, int lane, uint32_t hstage_u32, const float *hstage, float *hyb_tot) {
    int nd;
    bool hyb;
    const int expected = strip_contributors(p, strip, nd, hyb);
    int fin = 0;
    __syncwarp();
    if (lane == 0) {
        fin = (ticket_take(p.ws_cnt + strip) == expected - 1);
        if (fin) p.ws_cnt[strip] = 0;
    }
    fin = __shfl_sync(0xffffffffu, fin, 0);
    if (fin) {
        if (hyb) hybrid_totals(p, hstage_u32, hstage, hyb_tot, lane);
        final_store(p, strip, lane, nd, hyb ? hyb_tot : nullptr);
        final_store(p, strip, lane + 32, nd, hyb ? hyb_tot : nullptr);
    }
}

__device__ __forceinline__ float load_x(const Params &p, int k) {  // read-only path: x stays in L1 across the gathers
    return p.x_is_half ? __half2float(__ldg(reinterpret_cast<const __half *>(p.x) + k)) : __ldg(reinterpret_cast<const float *>(p.x) + k);
}

// =================================================================================================
// Sparse warp.  CSR rows (= output channels) are spread evenly over ALL CTAs (csr_rpc consecutive rows each, ~9 for a 4096-wide
// layer) and so are the k-rows of the topX dense rows; each warp therefore has a few hundred elements at most and every
// step is lane-parallel: row pointers live one-per-lane (shuffles / ballots instead of serial scans), cols/vals are staged
// with cp.async, x is gathered in batches of independent loads, per-row sums are taken in storage order (deterministic).
// Everything static (row pointers, cols/vals, dense-row values) is requested BEFORE griddepcontrol.wait.
// Results: accumulate mode -> red.add on mul; fused mode -> ws_csr[row] / dense-row partials + a ticket on the strips touched.
// =================================================================================================
template <int BITS, bool FUSED>
__device__ __forceinline__ void sparse_warp(const Params &p, unsigned char *sm, const uint32_t sm_u32, const int lane, float *hyb_tot,
                                            const int nseg, const int s0) {
    using C = Cfg<BITS>;
    const int N = p.N;
    const int cso = C::off_cstage(p.maxseg, p.xfloats);
    int *scols = reinterpret_cast<int *>(sm + cso);
    float *svals = reinterpret_cast<float *>(sm + cso + CSR_CH * 4);
    const uint32_t scols_u32 = sm_u32 + cso, svals_u32 = scols_u32 + CSR_CH * 4;

    // ---------------- phase A: static data ----------------
    float hfr[HYB_R];
    const bool hyb_on = p.full_rows && (int)blockIdx.x < p.hc;
    const bool hyb_multi = hyb_on && p.topX <= 32;  // 32/topX k-rows per warp step: lane = (row slot, column j)
    int kb = 0, ke = 0, nsl = 1, rs = 0, hj = lane;
    if (hyb_on) { kb = blockIdx.x * p.hrows; ke = min(p.K, kb + p.hrows); }
    if (hyb_multi) {
        nsl = 32 / p.topX;
        rs = lane / p.topX;
        hj = lane - rs * p.topX;
#pragma unroll
        for (int i = 0; i < HYB_R; ++i) {
            const int k = kb + rs + nsl * i;
            hfr[i] = (rs < nsl && k < ke) ? __ldg(p.full_rows + (size_t)k * p.topX + hj) : 0.f;
        }
    }
    // CSR: this CTA's rows [ra, rb) (rows are spread evenly over all CTAs), processed in groups of <= 31 rows / <= CSR_CH elements;
    // the first group is pre-staged before the dependency wait
    const int ra = p.rows ? min(N, (int)blockIdx.x * p.csr_rpc) : 0, rb = p.rows ? min(N, ra + p.csr_rpc) : 0;
    int r = ra, rp = 0, m = 0, base = 0, cnt = 0;
    auto group_begin = [&]() {  // row pointers one per lane, group size by ballot, then stage cols/vals
        rp = __ldg(p.rows + min(r + lane, rb));
        base = __shfl_sync(0xffffffffu, rp, 0);
        const bool ok = lane <= min(31, rb - r) && rp - base <= CSR_CH - 4;
        m = __popc(__ballot_sync(0xffffffffu, ok)) - 1;  // rp is non-decreasing: the ok lanes are a prefix that includes lane 0
        const int last = m > 0 ? __shfl_sync(0xffffffffu, rp, m) : base;
        if (p.csr_al16 && m > 0) {
            // 16-byte copies from the element-aligned-down start: up to 3 leading elements of earlier rows ride along (valid data,
            // never summed); the last quad is clipped with the src-size operand, so nothing past `last` is read
            base &= ~3;
            cnt = last - base;
            for (int e = 4 * lane; e < cnt; e += 128) {
                const int nb = min(16, 4 * (cnt - e));
                cp_async16_clip(scols_u32 + 4 * e, p.cols + base + e, nb);
                cp_async16_clip(svals_u32 + 4 * e, p.vals + base + e, nb);
            }
        } else {
            cnt = m > 0 ? last - base : 0;
            for (int e = lane; e < cnt; e += 32) {
                cp_async4(scols_u32 + 4 * e, p.cols + base + e);
                cp_async4(svals_u32 + 4 * e, p.vals + base + e);
            }
        }
        cp_async_commit();
    };
    if (r < rb) group_begin();

    TRACE(13, lane == 0);
#ifdef SQLLM_WAIT_ALL
    pdl_wait();
#else
    if (lane == 0) pdl_wait();
    __syncwarp();
#endif
    TRACE(14, lane == 0);

    // ---------------- phase B: needs x (and, in fused mode, the workspace) ----------------
    // (1) topX dense rows: CTA b < hc takes k-rows [kb, ke)
    if (hyb_on) {
        for (int jb = 0; jb < (hyb_multi ? 1 : p.topX); jb += 32) {
            float a = 0.f;
            int j;
            if (hyb_multi) {
                j = hj;
                float hx[HYB_R];
#pragma unroll
                for (int i = 0; i < HYB_R; ++i) {
                    const int k = kb + rs + nsl * i;
                    hx[i] = (rs < nsl && k < ke) ? load_x(p, k) : 0.f;
                }
#pragma unroll
                for (int i = 0; i < HYB_R; ++i) a += hfr[i] * hx[i];
                for (int k = kb + rs + nsl * HYB_R; rs < nsl && k < ke; k += nsl)
                    a += __ldg(p.full_rows + (size_t)k * p.topX + hj) * load_x(p, k);
                // fold the row slots onto slot 0 in fixed order
                for (int sl = 1; sl < nsl; ++sl) {
                    const float v = __shfl_sync(0xffffffffu, a, (hj + sl * p.topX) & 31);
                    if (rs == 0) a += v;
                }
                if (rs != 0) j = p.topX;  // only slot 0 publishes
            } else {
                j = jb + lane;
                if (j < p.topX) {
                    const float *fr = p.full_rows + (size_t)kb * p.topX + j;
#pragma unroll 8
                    for (int k = kb; k < ke; ++k, fr += p.topX) a += __ldg(fr) * load_x(p, k);
                }
            }
            if (j < p.topX) {
                if (FUSED && p.det) {
                    p.ws_hyb[(size_t)blockIdx.x * p.topX + j] = a;
                } else {
                    const int c = __ldg(p.fri + j);
                    if (c >= 0 && c < N) atomicAdd((FUSED ? p.ws_acc : reinterpret_cast<float *>(p.out)) + c, a);
                }
            }
        }
    }
    TRACE(15, lane == 0);

    // (2) CSR outliers
    float *const acc_out = FUSED ? p.ws_acc : reinterpret_cast<float *>(p.out);  // where red.add contributions go (non-deterministic modes)
    auto emit = [&](int row, float v) {
        if (FUSED && p.det) p.ws_csr[row] = v;
        else atomicAdd(acc_out + row, v);
    };
    while (r < rb) {
        if (m == 0) {  // a single row longer than the staging buffer: straight from global memory, whole warp
            const int e1 = __shfl_sync(0xffffffffu, rp, 1);
            float a = 0.f;
            for (int e = base + lane; e < e1; e += 32) a += __ldg(p.vals + e) * load_x(p, __ldg(p.cols + e));
            a = warp_sum(a);
            if (lane == 0) emit(r, a);
            r += 1;
        } else {
            cp_async_wait_all();
            __syncwarp();
            // products vals[e] * x[cols[e]] in place; gathers go out in batches of 8 independent loads per lane
            for (int e0 = lane; e0 < cnt; e0 += 32 * 8) {
                float xv[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int e = e0 + 32 * j;
                    xv[j] = e < cnt ? load_x(p, scols[e]) : 0.f;
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int e = e0 + 32 * j;
                    if (e < cnt) svals[e] *= xv[j];
                }
            }
            __syncwarp();
            // lane i < m owns row r+i: [a0, a1) in the staged arrays
            const int a0 = rp - base, a1 = __shfl_down_sync(0xffffffffu, rp, 1) - base;
            const int n = lane < m ? a1 - a0 : 0;
            if (lane < m && n <= 64) {  // short row: sequential sum in storage order (two interleaved chains)
                float ea = 0.f, eb = 0.f;
                int e = a0;
                for (; e + 1 < a1; e += 2) { ea += svals[e]; eb += svals[e + 1]; }
                if (e < a1) ea += svals[e];
                emit(r + lane, ea + eb);
            }
            unsigned longm = __ballot_sync(0xffffffffu, n > 64);  // long rows: the whole warp on each, fixed xor tree
            while (longm) {
                const int i = __ffs(longm) - 1;
                longm &= longm - 1;
                const int b0 = __shfl_sync(0xffffffffu, a0, i), b1 = __shfl_sync(0xffffffffu, a1, i);
                float a = 0.f;
                for (int e = b0 + lane; e < b1; e += 32) a += svals[e];
                a = warp_sum(a);
                if (lane == 0) emit(r + i, a);
            }
            __syncwarp();
            r += m;
        }
        if (r < rb) group_begin();
    }
    if (FUSED && p.det) {
        // publish: one fence for everything this warp wrote (CSR row sums, dense-row partials), then one ticket per strip touched
        const uint32_t hstage_u32 = svals_u32 + CSR_CH * 4;
        const float *hstage = svals + CSR_CH;
        __syncwarp();
        if (p.rows && ra < rb)
            for (int strip = ra / STRIP; strip <= (rb - 1) / STRIP; ++strip) warp_ticket(p, strip, lane, hstage_u32, hstage, hyb_tot);
        if (hyb_on) {  // every distinct strip that owns a dense-row output channel
            for (int j0 = 0; j0 < p.topX; ++j0) {
                const int cj0 = __ldg(p.fri + j0);
                if (cj0 < 0 || cj0 >= N) continue;
                const int strip = cj0 / STRIP;
                bool seen = false;
                for (int j = 0; j < j0; ++j) {
                    const int cj = __ldg(p.fri + j);
                    seen |= (cj >= 0 && cj < N && cj / STRIP == strip);
                }
                if (!seen) warp_ticket(p, strip, lane, hstage_u32, hstage, hyb_tot);
            }
        }
    }
}

// =================================================================================================
// The kernel
// =================================================================================================
template <int BITS, bool FUSED>
__global__ void __launch_bounds__(THREADS, BITS == 4 ? SQLLM_MINB4 : SQLLM_MINB3) lutgemv_kernel(const Params p, const __grid_constant__ CUtensorMap tmap) {
    using C = Cfg<BITS>;
    extern __shared__ unsigned char smem_raw[];
    // 4 KB aligned base, computed in the 32-bit shared window and pinned in a register (an opaque mov: otherwise the
    // compiler rematerialises it - S2UR + uniform adds - at every use once registers get tight)
    const uint32_t raw_u32 = smem_u32(smem_raw);
    uint32_t sm_u32 = (raw_u32 + 4095u) & ~4095u;
    asm volatile("mov.u32 %0, %0;" : "+r"(sm_u32));
    unsigned char *sm = smem_raw + (sm_u32 - raw_u32);
    const int maxseg = p.maxseg;
    float *part = reinterpret_cast<float *>(sm + C::off_part(maxseg));
    const uint32_t bar_u32 = sm_u32 + C::off_misc(maxseg);          // full[s] at +8s, empty[s] at +128+8s
    int *misc = reinterpret_cast<int *>(sm + C::off_misc(maxseg) + 256);
    float *hyb_tot = reinterpret_cast<float *>(sm + C::off_misc(maxseg) + 320);
    float *xs = reinterpret_cast<float *>(sm + C::off_x(maxseg));
    const uint32_t xs_u32 = sm_u32 + C::off_x(maxseg);
    const uint32_t stage_u32 = sm_u32 + C::off_stage(maxseg, p.xfloats, p.has_stage);
    const int nstage = p.nstage;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int i16 = lane & 15, jsel = lane >> 4;  // column group (4 columns) and unit-of-the-pair of this lane
    const int N = p.N, R = p.R;

    // ---- this CTA's chunk of the flattened [strip][unit] space ----
    const int g0 = min((int)blockIdx.x * p.chunk, p.T);
    const int g1 = (DBG(p) & 2) ? g0 : min(g0 + p.chunk, p.T);
    const int len = g1 - g0;
    const int s0 = g0 / R;
    const int r0 = g0 - s0 * R;
    const int nseg = len > 0 ? (g1 - 1) / R - s0 + 1 : 0;
    const int nst = (len + SU - 1) / SU;  // pipeline stages this CTA will consume

    TRACE(0, tid == 0);
#ifdef SQLLM_TRACE
    if (p.trace && tid == 0) { unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); p.trace[(size_t)blockIdx.x * 32 + 12] = smid + 1; }
#endif
    if (!LDG_MODE && tid == 0) {
        for (int s = 0; s < nstage; ++s) {
            mbar_init(bar_u32 + 8 * s, 1);          // full: the producer's arrive.expect_tx
            mbar_init(bar_u32 + 128 + 8 * s, NW);   // empty: one arrive per consumer warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    pdl_launch_dependents();  // the next kernel in the stream may start its own (independent) prologue now
    __syncthreads();
    TRACE(1, tid == 0);

    // ---- LDG mode: the first PF packed-word loads of every lane go out before anything else.  They do not depend on the
    //      previous kernel, so under PDL the register file of the next GEMV fills while this SM is still busy. ----
    constexpr int PF = LDG_MODE ? C::PF : 1;
    Words<BITS> ring[(LDG_MODE && !CPA_MODE) ? PF : 1];
    UnitIt ld;
    ld.init(2 * warp, r0, R);
    auto gload = [&](Words<BITS> &w) {  // fetch the pair `ld` points at (this lane's unit and 4 columns), then advance
        const int col0 = (s0 + ld.seg) * STRIP + 4 * (lane & 15);
        if (ld.o < len && col0 < N) gload_words(w, p.qw + (size_t)((ld.rr + (lane >> 4)) * C::ROWS_PER_UNIT) * N + col0, (size_t)N);
        else zero_words(w);
        ld.advance(SU, R);
    };
    // cp.async mode: slot u of this thread lives at ring_u32 + ((u * ROWS_PER_UNIT + row) * NW*32 + tid) * 16 (consecutive threads are
    // contiguous: coalesced fills, conflict-free 128-bit reads).  Exactly one group is committed per position, valid or not,
    // so "at most PF-1 groups pending" always means "the oldest position has landed".  A running global pointer follows the
    // load cursor; it is re-derived only when the cursor enters a new segment.
    const uint32_t ring_u32 = stage_u32 + tid * 16;
    constexpr uint32_t SLOT_STRIDE = C::ROWS_PER_UNIT * NW * 32 * 16;
    const int warp2 = 2 * warp;
    Cursor cl;
    cl.seg = 0; cl.left = 0; cl.rr = 0;
    const uint32_t *lptr = p.qw;
    bool lvalid = false;
    const size_t lstep = (size_t)SU * C::ROWS_PER_UNIT * N;  // words between consecutive positions of a warp
    auto cl_setup = [&]() {
        const int col0 = (s0 + cl.seg) * STRIP + 4 * i16;
        lvalid = cl.seg < nseg && col0 < N;  // lanes past a ragged last strip fetch nothing (their LUT columns are zero)
        if (lvalid) lptr = p.qw + (size_t)((cl.rr + jsel) * C::ROWS_PER_UNIT) * N + col0;
    };
    auto cpa_issue = [&](uint32_t dst) {
        if (lvalid) {
#pragma unroll
            for (int r = 0; r < C::ROWS_PER_UNIT; ++r) cp_async16(dst + r * (NW * 32 * 16), lptr + (size_t)r * N);
        }
        cp_async_commit();
        if (cl.seg < nseg) {
            lptr += lstep;
            if (--cl.left == 0) {
                cl.seek(cl.seg + 1, warp2, r0, R, len, nseg);
                cl_setup();
            }
        }
    };
    auto cpa_fetch = [&](Words<BITS> &w, uint32_t src) {
        w.a = lds_u4(src);
        if constexpr (BITS == 3) {
            w.b = lds_u4(src + NW * 32 * 16);
            w.c = lds_u4(src + 2 * NW * 32 * 16);
        }
    };
    if (warp == WARP_PRODUCER) {
        // =========================== TMA producer ===========================
        // Weights never depend on the previous kernel, so this runs ahead of pdl_wait().
        const uint64_t pol = l2_evict_first_policy();
        if (p.tma2d) {
            // One tensor-map box per BU units: hardware address generation.  The loop is a single latency-bound warp, so it
            // carries no divisions or re-derivations: ring slot, phase and box coordinates are all advanced incrementally.
            constexpr int BOXES = SU / C::BU;  // 1 (w4) / 4 (w3): lane b owns box b of every stage
            if (lane < BOXES) {
                constexpr uint32_t MASK = (1u << BOXES) - 1u;
                UnitIt it;
                it.init(lane * C::BU, r0, R);
                uint32_t full = bar_u32, empty = bar_u32 + 128, dst = stage_u32 + lane * C::BOX_BYTES;
                int s = 0;
                uint32_t ph = 0;
                bool refill = false;
                for (int n = 0; n < nst; ++n) {
                    if (refill) mbar_wait(empty, ph);
                    if (lane == 0) mbar_expect_tx(full, (uint32_t)min(BOXES, (len - it.o + C::BU - 1) / C::BU) * C::BOX_BYTES);
                    if (BOXES > 1) __syncwarp(MASK);
                    if (it.o < len) tma_tile2d_g2s(dst, &tmap, (s0 + it.seg) * STRIP, it.rr * C::ROWS_PER_UNIT, full, pol);
                    TRACE(8, lane == 0 && n == 0);
                    it.advance(SU, R);
                    full += 8; empty += 8; dst += C::STAGE_BYTES;
                    if (++s == nstage) {
                        s = 0;
                        full = bar_u32; empty = bar_u32 + 128; dst = stage_u32 + lane * C::BOX_BYTES;
                        if (refill) ph ^= 1u;
                        refill = true;
                    }
                }
            }
        } else {
            constexpr int COPIES = SU * C::ROWS_PER_UNIT;  // 16 (w4) / 48 (w3) row copies per stage
            for (int n = 0; n < nst; ++n) {
                const int use = n / nstage, s = n - use * nstage;
                const uint32_t full = bar_u32 + 8 * s, empty = bar_u32 + 128 + 8 * s;
                if (use > 0) mbar_wait(empty, (use - 1) & 1);
                // each lane describes up to 2 copies: copy id -> (unit, row-in-unit)
                uint32_t bytes[2] = {0u, 0u}, dst[2] = {0u, 0u};
                const uint32_t *src[2] = {nullptr, nullptr};
                uint32_t tot = 0;
    #pragma unroll
                for (int h = 0; h < (COPIES + 31) / 32; ++h) {
                    const int cid = lane + 32 * h;
                    if (cid < COPIES) {
                        const int u = cid / C::ROWS_PER_UNIT, rowin = cid - u * C::ROWS_PER_UNIT;
                        const int o = n * SU + u;
                        if (o < len) {
                            UnitIt it;
                            it.init(o, r0, R);
                            const int c0 = (s0 + it.seg) * STRIP;
                            bytes[h] = (uint32_t)min(STRIP, N - c0) * 4u;
                            src[h] = p.qw + (size_t)(it.rr * C::ROWS_PER_UNIT + rowin) * N + c0;
                            dst[h] = stage_u32 + s * C::STAGE_BYTES + cid * (STRIP * 4);
                        }
                    }
                    tot += bytes[h];
                }
                tot = __reduce_add_sync(0xffffffffu, tot);
                if (lane == 0) mbar_expect_tx(full, tot);
                __syncwarp();
    #pragma unroll
                for (int h = 0; h < (COPIES + 31) / 32; ++h)
                    if (bytes[h]) tma_bulk_g2s(dst[h], src[h], bytes[h], full, pol);
                TRACE(8, lane == 0 && n == 0);
            }
        }
        TRACE(9, lane == 0);
    } else if (warp == WARP_SPARSE) {
        sparse_warp<BITS, FUSED>(p, sm, sm_u32, lane, hyb_tot + maxseg * MAX_TOPX_FUSED, nseg, s0);
        TRACE(10, lane == 0);
    } else {
        // ---- LDG mode: the first PF packed-word loads of every lane go out before anything else ----
        if (CPA_MODE) {
            cl.seek(0, warp2, r0, R, len, nseg);
            cl_setup();
#pragma unroll
            for (int u = 0; u < PF; ++u) cpa_issue(ring_u32 + u * SLOT_STRIDE);
        } else if (LDG_MODE) {
#pragma unroll
            for (int u = 0; u < PF; ++u) gload(ring[u]);
        }
        // ---- consumers: stage the LUTs of this CTA's strips, transposed to [value][slot].  One 128-bit load per (column, value
        //      quad); a warp takes 32 columns whose slots fall in 32 different banks, so the four scalar stores are conflict-free.
        //      (4-byte cp.async would cost 16 shared-memory wavefronts per warp instruction - measured, profiles/r01.) ----
        constexpr int IPS = STRIP * C::L / 4;                 // (column, quad) items per strip: 256 (w4) / 128 (w3)
        constexpr int LQ = (MAXSEG * IPS + NW * 32 - 1) / (NW * 32);  // items per thread at most
        float4 lq[LQ];
#pragma unroll
        for (int n = 0; n < LQ; ++n) {
            const int it = tid + n * (NW * 32), seg = it / IPS, vw = (it % IPS) >> 5;
            const int c = ((lane >> 1) << 2) | ((vw & 1) << 1) | (lane & 1), q = vw >> 1;
            const int col = (s0 + seg) * STRIP + c;
            lq[n] = (seg < nseg && col < N && !(DBG(p) & 4)) ? __ldg(reinterpret_cast<const float4 *>(p.lut + (size_t)col * C::L) + q)
                                                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int e = tid; e < maxseg * NW * STRIP; e += NW * 32) part[e] = 0.f;
#pragma unroll
        for (int n = 0; n < LQ; ++n) {
            const int it = tid + n * (NW * 32), seg = it / IPS, vw = (it % IPS) >> 5;
            const int c = ((lane >> 1) << 2) | ((vw & 1) << 1) | (lane & 1), q = vw >> 1;
            const int slot = ((c & 3) << 4) | (c >> 2);
            if (seg < nseg) {
                float *t = reinterpret_cast<float *>(sm + seg * C::TAB) + (4 * q) * STRIP + slot;
                t[0] = lq[n].x; t[STRIP] = lq[n].y; t[2 * STRIP] = lq[n].z; t[3 * STRIP] = lq[n].w;
            }
        }

        TRACE(2, tid == 0);
        // Everything below reads data the previous kernel may have produced (x, mul, workspace).  One thread waits on the
        // programmatic dependency; the other consumers sleep on a hardware barrier instead of each polling it.
#ifdef SQLLM_WAIT_ALL
        pdl_wait();
#else
        if (tid == 0) pdl_wait();
        named_bar_sync(6, NW * 32);
#endif
        TRACE(3, tid == 0);

        // ---- stage the slice(s) of x this CTA needs, as fp32 ----
        for (int seg = 0; seg < nseg; ++seg) {
            const int ua = seg == 0 ? r0 : 0;                               // first unit of the segment inside its strip
            const int ub = min(R, r0 + len - seg * R);                      // one past the last
            const int dst_unit = p.x_direct ? ua : (seg * R + ua - r0);     // compact: indexed by unit offset
            const int nfl = (ub - ua) * C::XU;
            const int src_f = ua * C::XU, dst_f = dst_unit * C::XU;
            if (p.x_is_half) {
                const __half *xh = reinterpret_cast<const __half *>(p.x) + src_f;
                for (int e = tid; e < nfl / 4; e += NW * 32) {  // 4 halves in, one float4 out per thread: conflict-free stores
                    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(xh) + e);
                    const __half2 *h = reinterpret_cast<const __half2 *>(&u);
                    const float2 f0 = __half22float2(h[0]), f1 = __half22float2(h[1]);
                    reinterpret_cast<float4 *>(xs + dst_f)[e] = make_float4(f0.x, f0.y, f1.x, f1.y);
                }
            } else {
                const float *xf = reinterpret_cast<const float *>(p.x) + src_f;
                for (int e = tid; e < nfl / 4; e += NW * 32) cp_async16(xs_u32 + 4 * dst_f + 16 * e, xf + 4 * e);
            }
        }
        cp_async_commit();
        cp_async_wait_all();
        named_bar_sync(5, NW * 32);  // consumers only: LUTs, x slice, zeroed partials visible
        TRACE(4, tid == 0);
    }

    if (warp < NW) {
        // =========================== consumer warps ===========================
        // Everything in this loop is addressed through 32-bit shared-window addresses (no generic pointers: those make
        // the compiler rematerialise the window base through S2UR inside the loop when registers are tight).
        uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
        uint32_t lsb = 0u, segc = 0u;
        uint32_t lsv[4] = {0u, 0u, 0u, 0u};
        int cur_seg = -1;
        const uint32_t part_u32 = sm_u32 + C::off_part(maxseg) + (warp * STRIP + 4 * i16) * 4;
        const uint32_t lane_slot = (uint32_t)((jsel << 6) | (i16 << 2));  // column 0 of this lane: slot ((0^jsel)<<4 | i16), x4 bytes

        auto set_seg = [&](int seg) {
            const uint32_t tb = sm_u32 + seg * C::TAB;
            // 4-bit: byte 1 of the address comes from the nibble | segc (table 4 KB aligned); 3-bit: bits 8..10 are free (2 KB aligned)
            lsb = (BITS == 4 ? (tb & 0xFFFF0000u) : tb) | lane_slot;
            segc = ((tb >> 8) & 0xF0u) * 0x01010101u;
            if constexpr (BITS == 3) {
                // 3-bit: the four per-column slot addresses are pinned in registers for the whole segment.  Left to itself the
                // compiler folds the `^ (t << 6)` into a second LOP3 per lookup (96 extra instructions per 128-weight position).
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    lsv[t] = lsb ^ (uint32_t)(t << 6);
                    asm volatile("mov.u32 %0, %0;" : "+r"(lsv[t]));
                }
            }
        };
        auto deposit = [&](int seg) {
            float s[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) s[t] = sum2(acc[t]);
            // lane (i, j=1) holds column t^1 in slot t: hand it to lane (i, j=0)
            const float v0 = __shfl_xor_sync(0xffffffffu, s[1], 16);
            const float v1 = __shfl_xor_sync(0xffffffffu, s[0], 16);
            const float v2 = __shfl_xor_sync(0xffffffffu, s[3], 16);
            const float v3 = __shfl_xor_sync(0xffffffffu, s[2], 16);
            if (jsel == 0)
                asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(part_u32 + seg * (NW * STRIP * 4)), "f"(s[0] + v0),
                             "f"(s[1] + v1), "f"(s[2] + v2), "f"(s[3] + v3) : "memory");
#pragma unroll
            for (int t = 0; t < 4; ++t) acc[t] = 0ull;
        };

        const uint32_t xlane = xs_u32 + (C::XU * 4) * jsel;
        const bool xdir = p.x_direct != 0;
        UnitIt it;
        it.init(2 * warp, r0, R);
        if constexpr (CPA_MODE) {
            // private cp.async ring.  Outer loop: the segments (strips) this warp has positions in; inner loop: a fixed trip
            // count of positions with nothing but running pointers: wait for the slot, pull it into registers, do the math,
            // refill the slot PF positions ahead.
            Cursor cc;
            cc.seek(0, warp2, r0, R, len, nseg);
            uint32_t slot = ring_u32;
            const uint32_t slot_end = ring_u32 + PF * SLOT_STRIDE;
            while (cc.seg < nseg) {
                set_seg(cc.seg);
                uint32_t xptr = xlane + (C::XU * 4) * (xdir ? cc.rr : cc.rr + cc.seg * R - r0);
                for (int i = cc.left; i > 0; --i) {
                    cp_async_wait_pending<PF - 1>();
                    Words<BITS> cur;
                    cpa_fetch(cur, slot);
                    if (!(DBG(p) & 1)) consume(cur, jsel, lsb, segc, lsv, xptr, acc);
                    else acc[0] ^= cur.a.x;
                    cpa_issue(slot);  // the words are in registers (consumed above): the slot can be overwritten
                    slot += SLOT_STRIDE;
                    if (slot == slot_end) slot = ring_u32;
                    xptr += SU * C::XU * 4;
                }
                deposit(cc.seg);
                cc.seek(cc.seg + 1, warp2, r0, R, len, nseg);
            }
            cur_seg = -1;  // everything already deposited
        } else if constexpr (LDG_MODE) {
            // register ring: consume slot u, immediately refill it with the pair PF positions ahead
            while (it.o < len) {
#pragma unroll
                for (int u = 0; u < PF; ++u) {
                    if (it.o < len) {  // warp-uniform: len and o are even, a pair never straddles the end
                        if (it.seg != cur_seg) {
                            if (cur_seg >= 0) deposit(cur_seg);
                            cur_seg = it.seg;
                            set_seg(cur_seg);
                        }
                        if (!(DBG(p) & 1)) consume(ring[u], jsel, lsb, segc, lsv, xlane + (C::XU * 4) * (xdir ? it.rr : it.o), acc);
                        else acc[0] ^= ring[u].a.x;
                        gload(ring[u]);
                        it.advance(SU, R);
                    }
                }
            }
        } else {
            // this lane's unit inside a stage: 2*warp + jsel ; its 16 bytes at column group i16
            const uint32_t lane_off = stage_u32 + (2 * warp + jsel) * C::UNIT_BYTES + i16 * 16;
            Words<BITS> cur = {}, nxt = {};
            int s = 0;               // ring slot of the stage being fetched
            uint32_t par = 0;        // its phase parity
            auto fetch = [&](Words<BITS> &dst) {  // wait for ring slot s, pull this lane's words, release the slot, advance
                mbar_wait(bar_u32 + 8 * s, par);
                load_words(dst, lane_off + s * C::STAGE_BYTES);
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_u32 + 128 + 8 * s);
                if (++s == nstage) { s = 0; par ^= 1u; }
            };
            if (nst > 0) {
                fetch(cur);
                TRACE(5, tid == 0);
            }
            for (int n = 0; n < nst; ++n) {
                if (n + 1 < nst) {  // pull the next stage into registers before computing on this one
                    fetch(nxt);
                    TRACE(16 + (n + 1 < 15 ? n + 1 : 15), tid == 0);
                }
                if (it.o < len) {  // warp-uniform: len and o are even, a pair never straddles the end
                    if (it.seg != cur_seg) {
                        if (cur_seg >= 0) deposit(cur_seg);
                        cur_seg = it.seg;
                        set_seg(cur_seg);
                    }
                    if (!(DBG(p) & 1)) consume(cur, jsel, lsb, segc, lsv, xlane + (C::XU * 4) * (xdir ? it.rr : it.o), acc);
                    else acc[0] ^= cur.a.x;
                }
                it.advance(SU, R);
                cur = nxt;
            }
        }
        if (cur_seg >= 0) deposit(cur_seg);
        TRACE(6, tid == 0);
    }

    __syncthreads();  // all partials of this CTA are in shared memory
    TRACE(7, tid == 0);

    // =========================== flush ===========================
    if (tid < MAXSEG * STRIP) {
        const int seg = tid >> 6, c = tid & 63;
        const bool active = seg < nseg;
        float tot = 0.f;
        int strip = 0, nd = 1, slot = 0;
        bool hyb = false;
        if (active) {
            strip = s0 + seg;
#pragma unroll
            for (int w = 0; w < NW; ++w) tot += part[(seg * NW + w) * STRIP + c];
        }
        if (!FUSED) {
            const int col = strip * STRIP + c;
            if (active && col < N) atomicAdd(reinterpret_cast<float *>(p.out) + col, tot);
            TRACE(11, tid == 0);
            return;
        }
        if (!p.det) {  // fast fused mode: same red.add, into the zeroed scratch accumulator; conversion happens below
            const int col = strip * STRIP + c;
            if (active && col < N) atomicAdd(p.ws_acc + col, tot);
        } else {
        int expected = 1;
        if (active) {
            expected = strip_contributors(p, strip, nd, hyb);
            slot = (int)blockIdx.x - (int)(((long long)strip * R) / p.chunk);
            if (expected == 1) {  // this CTA is the strip's only contributor: store directly
                const int col = strip * STRIP + c;
                if (col < N) {
                    if (p.bias) tot += p.bias[col];
                    if (p.y_is_half) reinterpret_cast<__half *>(p.out)[col] = __float2half_rn(tot);
                    else reinterpret_cast<float *>(p.out)[col] = tot;
                }
            } else {
                p.ws_part[((size_t)strip * p.maxc + slot) * STRIP + c] = tot;
            }
        }
        // ticket: 64 threads (2 warps) per segment; sync them with a named barrier per segment
        const bool ticketed = active && expected > 1;
        named_bar_sync(seg + 1, 64);
        if (c == 0) {
            int fin = 0;
            if (ticketed) {
                fin = (ticket_take(p.ws_cnt + strip) == expected - 1);
                if (fin) p.ws_cnt[strip] = 0;
            }
            misc[seg] = fin;
        }
        named_bar_sync(seg + 1, 64);
        if (misc[seg]) {
            float *ht = hyb_tot + seg * MAX_TOPX_FUSED;
            if (hyb) {  // the first warp of this segment's pair stages and sums the dense-row partials, then both warps use them
                const int cso = C::off_cstage(maxseg, p.xfloats);
                if ((c >> 5) == 0) hybrid_totals(p, sm_u32 + cso + CSR_CH * 8, reinterpret_cast<const float *>(sm + cso + CSR_CH * 8), ht, lane);
                named_bar_sync(seg + 1, 64);
            }
            final_store(p, strip, c, nd, hyb ? ht : nullptr);
        }
        }  // det
        TRACE(11, tid == 0);
    }
    if (FUSED && !p.det) {
        // Fast fused mode.  Every CTA announces "my red.adds are out" with one fire-and-forget red.release on a gpu-scope counter
        // and leaves.  The last `nfin` CTAs of the grid (by index - they are dispatched last) stay, wait until the counter reaches
        // the grid size, and each turns its 1/nfin slice of the accumulator into y (+ bias, converted) and re-zeroes it.  One CTA
        // alone moves ~125 GB/s: 3.6 us for a 22016-wide layer (trace in profiles/r01); 16 of them need one L2 round trip.
        // All CTAs of a launch are co-resident by construction (make_plan sizes the grid to the occupancy), so the wait cannot
        // deadlock; the counter is reset by the last finisher for the next launch (kernel boundary orders it).
        __syncthreads();  // all red.adds of this CTA issued
        const int G = (int)gridDim.x, nfin = p.nfin;
        const int fidx = (int)blockIdx.x - (G - nfin);
        if (tid == 0) {
            asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(p.ws_hyb_cnt) : "memory");
            if (fidx >= 0) {
                int seen;
                do {
                    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(p.ws_hyb_cnt) : "memory");
                    if (seen < G) __nanosleep(40);
                } while (seen < G);
            }
        }
        TRACE(8, tid == 0);  // (slots 8 / 9 double as "announced / all arrived" and "finalizer done" outside the TMA mode)
        if (fidx < 0) return;
        __syncthreads();
        {
            const float4 *acc4 = reinterpret_cast<const float4 *>(p.ws_acc);
            const int n4 = N >> 2;
            const int per = (n4 + nfin - 1) / nfin;
            const int lo = min(n4, fidx * per), hi = min(n4, lo + per);
            for (int c0 = lo + tid; c0 < hi; c0 += 4 * THREADS) {
                float4 v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int c4 = c0 + u * THREADS;
                    v[u] = c4 < hi ? __ldcg(acc4 + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int c4 = c0 + u * THREADS;
                    if (c4 < hi) {
                        reinterpret_cast<float4 *>(p.ws_acc)[c4] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (p.bias) {
                            const float4 bv = __ldg(reinterpret_cast<const float4 *>(p.bias) + c4);
                            v[u].x += bv.x; v[u].y += bv.y; v[u].z += bv.z; v[u].w += bv.w;
                        }
                        uint2 pk = make_uint2(0u, 0u);
                        if (p.y_is_half) {
                            __half2 lo2 = __floats2half2_rn(v[u].x, v[u].y), hi2 = __floats2half2_rn(v[u].z, v[u].w);
                            pk.x = *reinterpret_cast<uint32_t *>(&lo2);
                            pk.y = *reinterpret_cast<uint32_t *>(&hi2);
                        }
                        if (p.xw_world == 0) {
                            if (p.y_is_half) reinterpret_cast<uint2 *>(p.out)[c4] = pk;
                            else reinterpret_cast<float4 *>(p.out)[c4] = v[u];
                        } else {
                            // local column 4*c4 of the stacked shard = column j of member m; it lands at [m][rank*w + j] of the
                            // [members][n_full] vector in EVERY rank's arena (w % 4 == 0: a quad never straddles members)
                            const int w = N / p.xw_members, col = 4 * c4, m = col / w, j = col - m * w;
                            const unsigned long long e = (unsigned long long)m * p.xw_nfull + (unsigned long long)p.xw_rank * w + j;
                            for (int pr = 0; pr < p.xw_world; ++pr) {
                                unsigned char *dst = reinterpret_cast<unsigned char *>(__ldg(p.xw_base + pr) + p.xw_out_off);
                                if (p.y_is_half) *reinterpret_cast<uint2 *>(dst + 2 * e) = pk;
                                else *reinterpret_cast<float4 *>(dst + 4 * e) = v[u];
                            }
                        }
                    }
                }
            }
        }
        TRACE(9, tid == 0);
        __syncthreads();
        if (tid == 0) {
            unsigned long long target = 0ull;
            if (p.xw_world) {
                // publish this finisher's stores on every rank (system-scope release), then wait until every finisher of every
                // rank has published on ours: when this grid completes, the local vector is whole.  Counters only grow
                // (expected arrivals so far live next to the flag), so nothing is ever reset across ranks.  The wait is bounded:
                // a rank that never shows up sets the error word instead of hanging the GPU.
                const unsigned long long self = __ldg(p.xw_base + p.xw_rank);
                target = *reinterpret_cast<volatile unsigned long long *>(self + p.xw_state_off) + (unsigned long long)p.xw_world * nfin;
                __threadfence_system();
                for (int pr = 0; pr < p.xw_world; ++pr)
                    atomicAdd_system(reinterpret_cast<unsigned long long *>(__ldg(p.xw_base + pr) + p.xw_flag_off), 1ull);
                unsigned long long seen, t0, t1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
                const bool broken = *reinterpret_cast<volatile unsigned int *>(self + p.xw_err_off) != 0u;  // an earlier wait gave up: do not wait again
                if (!broken) do {
                    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(self + p.xw_flag_off) : "memory");
                    if (seen >= target) break;
                    __nanosleep(100);
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    if (t1 - t0 > 2000000000ull) { *reinterpret_cast<volatile unsigned int *>(self + p.xw_err_off) = 1u; break; }
                } while (true);
            }
            // the finisher that completes the set puts both counters back to zero (and advances the expected arrivals)
            int done;
            asm volatile("atom.relaxed.gpu.global.add.s32 %0, [%1], 1;" : "=r"(done) : "l"(p.ws_hyb_cnt + 32) : "memory");
            if (done == nfin - 1) {
                p.ws_hyb_cnt[0] = 0;
                p.ws_hyb_cnt[32] = 0;
                if (p.xw_world) *reinterpret_cast<volatile unsigned long long *>(__ldg(p.xw_base + p.xw_rank) + p.xw_state_off) = target;
            }
        }
    }
}

// test hook: unpack exactly like the GEMV path (same shift/mask expressions)
__global__ void unpack_kernel(int bits, const uint32_t *__restrict__ q, int K, int N, uint8_t *__restrict__ idx) {
    const size_t n = (size_t)K * N;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(e / N), c = (int)(e % N);
        uint32_t v;
        if (bits == 4) {
            const uint32_t w = q[(size_t)(k >> 3) * N + c];
            const int n8 = k & 7;
            const uint32_t EO = (n8 & 1) ? ((w >> 4) & 0x0F0F0F0Fu) : (w & 0x0F0F0F0Fu);
            v = __byte_perm(EO, 0u, 0x4440 | (n8 >> 1)) & 0xFFu;
        } else {
            const int g = k >> 5, j = k & 31;
            const uint32_t *pq = q + (size_t)(3 * g) * N + c;
            const uint32_t w0 = pq[0], w1 = pq[N], w2 = pq[2 * (size_t)N];
            uint32_t f;  // field moved to bits 8..10, as in consume3_col
            if (j < 10) f = (3 * j < 8) ? (w0 << (8 - 3 * j)) : (w0 >> (3 * j - 8));
            else if (j == 10) f = __funnelshift_r(w0, w1, 22);
            else if (j < 21) { const int s = 1 + 3 * (j - 11); f = (s < 8) ? (w1 << (8 - s)) : (w1 >> (s - 8)); }
            else if (j == 21) f = __funnelshift_r(w1, w2, 23);
            else { const int s = 2 + 3 * (j - 22); f = (s < 8) ? (w2 << (8 - s)) : (w2 >> (s - 8)); }
            v = (f & 0x700u) >> 8;
        }
        idx[e] = (uint8_t)v;
    }
}

#include "lutgemv_v2.cuh"
#include "lutgemv_seq.cuh"
#include "lutgemm_batched.cuh"

// shared-window address at which a kernel without static shared memory sees its dynamic shared memory (the v2 carve-up aligns
// tables to their own size - up to 64 KB - so the host needs the real address, not a worst case; the kernel re-checks it)
__global__ void smem_base_probe(unsigned *out) {
    extern __shared__ unsigned char probe_smem[];
    *out = smem_u32(probe_smem);
}

// =================================================================================================
// Host side
// =================================================================================================
thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

struct DevInfo {
    int sm = 0;
    bool attr_set = false;
};
// Process-wide state (mode switches, lazily read environment knobs, per-device attributes) is guarded by g_state_mu: the entry
// points may be called from several host threads.  Switching a mode (sqllm_set_deterministic / sqllm_set_lut_mode) while other
// threads are launching is allowed but takes effect per call; do not switch while a CUDA graph that should keep the old mode is
// being captured.
std::recursive_mutex g_state_mu;
DevInfo g_dev[64];
int g_use_pdl = -1;
int g_det = -1;
int det_mode() {
    std::lock_guard<std::recursive_mutex> lk(g_state_mu);
    if (g_det < 0) { const char *e = getenv("SQLLM_DETERMINISTIC"); g_det = (e && e[0] == '1') ? 1 : 0; }
    return g_det;
}
// g_det - fused mode: 1 = deterministic per-strip tickets, 0 = red.add + one global ticket (default; SQLLM_DETERMINISTIC=1 or sqllm_set_deterministic)
int g_last_grid = 0;
unsigned long long *g_trace = nullptr;
size_t g_trace_stride = 0;

// ---- 2-D tensor maps for the packed matrix (one per (pointer, shape, box)), created through the driver entry point ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
struct TmKey {
    const void *ptr; int rows, cols, box_rows;
    bool operator==(const TmKey &o) const { return ptr == o.ptr && rows == o.rows && cols == o.cols && box_rows == o.box_rows; }
};
struct TmHash {
    size_t operator()(const TmKey &k) const {
        return std::hash<const void *>()(k.ptr) ^ ((size_t)k.rows * 1000003u) ^ ((size_t)k.cols * 10007u) ^ (size_t)k.box_rows;
    }
};
std::mutex g_tm_mutex;
std::unordered_map<TmKey, CUtensorMap, TmHash> g_tm_cache;
EncodeTiledFn g_encode = nullptr;

int get_tensor_map(const void *qweight, int rows, int cols, int box_rows, CUtensorMap &out) {
    std::lock_guard<std::mutex> lock(g_tm_mutex);
    const TmKey key{qweight, rows, cols, box_rows};
    auto it = g_tm_cache.find(key);
    if (it != g_tm_cache.end()) { out = it->second; return SQLLM_OK; }
    if (!g_encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn)
            return fail(SQLLM_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
        g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)cols * 4};
    const cuuint32_t box[2] = {(cuuint32_t)STRIP, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUtensorMap m;
    const CUresult r = g_encode(&m, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<void *>(qweight), gdim, gstride, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(SQLLM_ECUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    if (g_tm_cache.size() > 8192) g_tm_cache.clear();
    g_tm_cache.emplace(key, m);
    out = m;
    return SQLLM_OK;
}

struct Plan {
    int R, strips, T, chunk, G, maxc, hc, hrows, smem, maxseg, nstage, x_direct, xfloats, tma2d, box_rows;
    size_t ws_cnt_off, ws_hybcnt_off, ws_hyb_off, ws_part_off, ws_csr_off, ws_acc_off, ws_bytes;
    int csr_rpc, has_stage;
};

int make_plan(int bits, int K, int N, int topX, bool has_csr_in, bool fused, Plan &pl) {
    std::lock_guard<std::recursive_mutex> state_lock(g_state_mu);  // lazily initialised statics below
    const bool has_csr = has_csr_in || topX > 0;  // from here on: "a staging buffer is needed"
    // staging: CSR cols/vals chunks (8 KB); the deterministic fused mode also stages the dense-row partials there (8 KB more)
    pl.has_stage = has_csr ? CSR_CH * 8 + ((fused && det_mode() == 1) ? CSR_CH * 8 : 0) : 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return fail(SQLLM_ECUDA, "cudaGetDevice failed");
    if (dev < 0 || dev >= 64) return fail(SQLLM_EINVAL, "device ordinal %d out of range", dev);
    DevInfo &d = g_dev[dev];
    if (d.sm == 0) {
        if (cudaDeviceGetAttribute(&d.sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || d.sm <= 0)
            return fail(SQLLM_ECUDA, "cannot query SM count");
    }
    if (!d.attr_set) {
        const int mx = 227 * 1024;
        cudaFuncSetAttribute(lutgemv_kernel<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
        cudaFuncSetAttribute(lutgemv_kernel<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
        cudaFuncSetAttribute(lutgemv_kernel<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
        cudaFuncSetAttribute(lutgemv_kernel<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
        if (cudaGetLastError() != cudaSuccess) return fail(SQLLM_ECUDA, "cudaFuncSetAttribute failed");
        d.attr_set = true;
    }
    const int XU = bits == 4 ? 8 : 32;
    pl.R = bits == 4 ? K / 8 : K / 32;
    pl.strips = (N + STRIP - 1) / STRIP;
    const long long T = (long long)pl.strips * pl.R;
    if (T > 0x3fffffff) return fail(SQLLM_EINVAL, "problem too large");
    pl.T = (int)T;
    if (pl.strips > MAX_STRIPS || (fused && N > MAX_N_FUSED)) return fail(SQLLM_EINVAL, "out_features=%d exceeds the workspace header (max %d)", N, MAX_N_FUSED);

    // Each kernel takes only CPS CTA slots per SM (default 2 of the 4 that fit): the rest of the SM is left to the NEXT
    // GEMV in the stream, which - launched with programmatic dependent launch - streams its weights into shared memory
    // while this one is still computing.  All of a CTA's shared memory beyond the fixed part holds weight stages.
    static int cps = 0, budget = 0;
    if (!cps) {
        const char *e1 = getenv("SQLLM_CTAS_PER_SM"), *e2 = getenv("SQLLM_SMEM_BUDGET_KB");
        cps = e1 ? atoi(e1) : (LDG_MODE ? 3 : 2);
        if (cps < 1 || cps > 8) cps = LDG_MODE ? 3 : 2;
        budget = (e2 ? atoi(e2) : 56) * 1024;
        if (budget < 16 * 1024 || budget > 227 * 1024) budget = 56 * 1024;
    }
    // The grid must be co-resident: a plan whose shared memory lets fewer than `cps` CTAs onto an SM would run a second wave.
    // Plan for cps CTAs/SM, ask the occupancy calculator, and fall back to fewer CTAs per SM if it disagrees.
    int use_cps = cps;
replan:
    const int G0 = d.sm * use_cps;
    // 2-D TMA boxes need every box inside one strip and one CTA range: units per box BU divides R and the chunk.
    const int BU = bits == 4 ? Cfg<4>::BU : Cfg<3>::BU;
    static int no_tma2d = -1;
    if (no_tma2d < 0) { const char *e = getenv("SQLLM_NO_TMA2D"); no_tma2d = (e && e[0] == '1') ? 1 : 0; }
    pl.tma2d = (!LDG_MODE && !no_tma2d && K % 128 == 0 && pl.R % BU == 0) ? 1 : 0;
    pl.box_rows = bits == 4 ? Cfg<4>::BOX_ROWS : Cfg<3>::BOX_ROWS;
    const int gran = pl.tma2d ? (BU % 2 ? 2 * BU : BU) : 2;
    int chunk = (int)(gran * ((T + (long long)gran * G0 - 1) / ((long long)gran * G0)));
    if (chunk > 3 * pl.R) chunk = 3 * pl.R;  // a CTA may touch at most MAXSEG strips
    if (chunk < 2) chunk = 2;
    int maxseg = (chunk - 2) / pl.R + 2;      // worst case over start offsets (even offsets, even R)
    if (maxseg > MAXSEG) maxseg = MAXSEG;
    const bool direct = (long long)chunk * XU >= K;
    const int xfl = direct ? K : chunk * XU;
    pl.x_direct = direct ? 1 : 0;
    const int stage_bytes = bits == 4 ? Cfg<4>::STAGE_BYTES : Cfg<3>::STAGE_BYTES;
    const int fixed = bits == 4 ? Cfg<4>::total(maxseg, xfl, pl.has_stage, 0) : Cfg<3>::total(maxseg, xfl, pl.has_stage, 0);
    const int need = (chunk + SU - 1) / SU;
    int nstage = (budget - fixed) / stage_bytes;
    if (nstage > need) nstage = need;
    if (nstage > MAX_NSTAGE) nstage = MAX_NSTAGE;
    if (nstage < 2) nstage = 2;
    if (LDG_MODE) nstage = 0;  // weights go straight to registers
    const int smem = fixed + nstage * stage_bytes;
    if (smem > 227 * 1024) return fail(SQLLM_EINVAL, "in_features=%d needs %d B of shared memory (> 227 KB)", K, smem);
    {
        static std::mutex occ_mu;
        static std::unordered_map<unsigned long long, int> occ_cache;
        const unsigned long long key = ((unsigned long long)smem << 8) | (unsigned long long)((bits == 4 ? 2 : 0) | (fused ? 1 : 0));
        int occ = -1;
        {
            std::lock_guard<std::mutex> lk(occ_mu);
            auto it = occ_cache.find(key);
            if (it != occ_cache.end()) occ = it->second;
        }
        if (occ < 0) {
            const int threads = THREADS;
            cudaError_t e;
            if (bits == 4) e = fused ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lutgemv_kernel<4, true>, threads, smem)
                                     : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lutgemv_kernel<4, false>, threads, smem);
            else e = fused ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lutgemv_kernel<3, true>, threads, smem)
                           : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lutgemv_kernel<3, false>, threads, smem);
            if (e != cudaSuccess) return fail(SQLLM_ECUDA, "occupancy query failed: %s", cudaGetErrorString(e));
            std::lock_guard<std::mutex> lk(occ_mu);
            occ_cache[key] = occ;
        }
        if (occ < 1) return fail(SQLLM_EINVAL, "kernel does not fit an SM (shared memory %d B)", smem);
        if (occ < use_cps) { use_cps = occ; goto replan; }
    }
    pl.smem = smem;
    pl.maxseg = maxseg;
    pl.nstage = nstage;
    pl.xfloats = xfl;
    pl.chunk = chunk;
    pl.G = (int)((T + chunk - 1) / chunk);
    pl.maxc = (pl.R - 1) / chunk + 2;
    pl.hc = 0;
    pl.hrows = 0;
    int hc_det = 0;  // workspace is sized for the deterministic mode whatever the current mode
    if (topX > 0) {
        // dense-row contributors: as few k-rows per CTA as the grid allows, down to what one warp requests before the dependency
        // wait (HYB_R steps of 32/topX rows).  Deterministic mode also needs the partials (hc*topX floats) to fit the
        // 2*CSR_CH-float staging buffer of the finisher.
        const int rows_pre = HYB_R * (topX <= 32 ? 32 / topX : 1);
        int hc = pl.G;
        if (hc > (K + rows_pre - 1) / rows_pre) hc = (K + rows_pre - 1) / rows_pre;
        hc_det = hc;
        if (hc_det > 2 * CSR_CH / topX) hc_det = 2 * CSR_CH / topX;
        if (hc_det < 1) hc_det = 1;
        if (fused && det_mode() == 1) hc = hc_det;
        if (hc < 1) hc = 1;
        pl.hrows = (K + hc - 1) / hc;
        pl.hc = (K + pl.hrows - 1) / pl.hrows;
    }
    pl.csr_rpc = (N + pl.G - 1) / pl.G;
    if (pl.csr_rpc < 1) pl.csr_rpc = 1;
    // Fixed header: [0,4) dense-row ticket, [256, 256+4*MAX_STRIPS) per-strip tickets.  Tickets must never
    // share bytes with data regions of ANY shape (the workspace is reused across layers of different sizes).
    size_t off = WS_HEADER;
    pl.ws_hybcnt_off = 0;
    pl.ws_cnt_off = 256;
    pl.ws_hyb_off = off; off += (size_t)hc_det * (topX > 0 ? topX : 0) * 4;
    off = (off + 255) & ~(size_t)255;
    pl.ws_part_off = off; off += (size_t)pl.strips * pl.maxc * STRIP * 4;
    off = (off + 255) & ~(size_t)255;
    pl.ws_csr_off = off; off += (size_t)N * 4;
    pl.ws_acc_off = WS_ACC_OFF;
    pl.ws_bytes = off;
    return SQLLM_OK;
}

int check_common(const sqllm_lutgemv_args *a) {
    if (!a) return fail(SQLLM_EINVAL, "null args");
    if (a->bits != 3 && a->bits != 4) return fail(SQLLM_EINVAL, "bits must be 3 or 4 (got %d)", a->bits);
    if (a->in_features <= 0 || a->in_features % 64) return fail(SQLLM_EINVAL, "in_features=%d must be a positive multiple of 64", a->in_features);
    if (a->out_features <= 0 || a->out_features % 4) return fail(SQLLM_EINVAL, "out_features=%d must be a positive multiple of 4", a->out_features);
    if (!a->qweight || !a->lookup_table) return fail(SQLLM_EINVAL, "qweight / lookup_table must not be null");
    if (reinterpret_cast<uintptr_t>(a->qweight) & 15) return fail(SQLLM_EINVAL, "qweight must be 16-byte aligned");
    if (reinterpret_cast<uintptr_t>(a->lookup_table) & 15) return fail(SQLLM_EINVAL, "lookup_table must be 16-byte aligned");
    if (a->topX < 0) return fail(SQLLM_EINVAL, "topX < 0");
    if (a->full_rows && a->topX > 0 && !a->full_row_indices) return fail(SQLLM_EINVAL, "full_rows given without full_row_indices");
    return SQLLM_OK;
}

template <int BITS, bool FUSED>
cudaError_t launch_kernel(const Plan &pl, const Params &p, const CUtensorMap &tm, cudaStream_t st) {
    std::lock_guard<std::recursive_mutex> state_lock(g_state_mu);
    if (g_use_pdl < 0) {
        const char *e = getenv("SQLLM_NO_PDL");
        g_use_pdl = (e && e[0] == '1') ? 0 : 1;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    g_last_grid = pl.G;
    cfg.gridDim = dim3(pl.G);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = pl.smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_use_pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, lutgemv_kernel<BITS, FUSED>, p, tm);
}

template <bool FUSED>
int launch(const sqllm_lutgemv_args *a, const Plan &pl, Params &p, cudaStream_t st) {
    std::lock_guard<std::recursive_mutex> state_lock(g_state_mu);
    p.qw = reinterpret_cast<const uint32_t *>(a->qweight);
    p.lut = a->lookup_table;
    p.rows = a->rows; p.cols = a->cols; p.vals = a->vals;
    const bool hyb = a->full_rows && a->topX > 0;
    p.full_rows = hyb ? a->full_rows : nullptr;
    p.fri = hyb ? a->full_row_indices : nullptr;
    p.topX = hyb ? a->topX : 0;
    p.K = a->in_features; p.N = a->out_features;
    p.R = pl.R; p.strips = pl.strips; p.T = pl.T; p.chunk = pl.chunk;
    p.maxseg = pl.maxseg; p.nstage = pl.nstage; p.tma2d = pl.tma2d; p.x_direct = pl.x_direct; p.xfloats = pl.xfloats;
    p.hc = hyb ? pl.hc : 0; p.hrows = pl.hrows; p.maxc = pl.maxc;
    p.has_csr = a->rows ? 1 : 0;
    p.has_stage = pl.has_stage;
    p.csr_rpc = pl.csr_rpc;
    {   // ~1024 columns per finishing CTA, at most 16 of them (SQLLM_NFIN_COLS / SQLLM_NFIN_MAX override, for experiments)
        static int cols_per = 0, nmax = 0;
        if (!cols_per) {
            const char *e1 = getenv("SQLLM_NFIN_COLS"), *e2 = getenv("SQLLM_NFIN_MAX");
            cols_per = e1 && atoi(e1) > 0 ? atoi(e1) : 1024;
            nmax = e2 && atoi(e2) > 0 ? atoi(e2) : 16;
        }
        p.nfin = (a->out_features + cols_per - 1) / cols_per;
        if (p.nfin > nmax) p.nfin = nmax;
    }
    if (p.nfin > pl.G) p.nfin = pl.G;
    if (p.nfin < 1) p.nfin = 1;
    p.csr_al16 = (a->rows && ((reinterpret_cast<uintptr_t>(a->cols) | reinterpret_cast<uintptr_t>(a->vals)) & 15) == 0) ? 1 : 0;
    p.trace = g_trace;
    { static int dbg = -1; if (dbg < 0) { const char *e = getenv("SQLLM_DEBUG_FLAGS"); dbg = e ? atoi(e) : 0; } p.dbg = dbg; }
    if (g_trace) g_trace += g_trace_stride;
    CUtensorMap tm;
    memset(&tm, 0, sizeof(tm));
    if (pl.tma2d) {
        const int rc = get_tensor_map(a->qweight, a->in_features / 32 * a->bits, a->out_features, pl.box_rows, tm);
        if (rc) return rc;
    }
    const cudaError_t e = a->bits == 4 ? launch_kernel<4, FUSED>(pl, p, tm, st) : launch_kernel<3, FUSED>(pl, p, tm, st);
    if (e != cudaSuccess) return fail(SQLLM_ECUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    return SQLLM_OK;
}


// =================================================================================================
// v2 (lutgemv_v2.cuh): plan + launch.  One CTA per SM; all process-wide state behind one mutex / atomics.
// =================================================================================================
bool g_v2_attr[64] = {};
int g_lut_mode = -1;     // 0: exact fp32 table, 1: fp16 pair table when x is fp16 (SQLLM_LUT_MODE=fp16 / sqllm_set_lut_mode)
int g_kernel_sel = -1;   // 2: v2 (default), 1: v1 everywhere (SQLLM_KERNEL=v1; kept for A/B runs and as the deterministic mode's kernel)

int lut_mode() {
    std::lock_guard<std::recursive_mutex> lk(g_state_mu);
    if (g_lut_mode < 0) {
        const char *e = getenv("SQLLM_LUT_MODE");
        g_lut_mode = (e && (!strcmp(e, "fp16") || !strcmp(e, "pair") || !strcmp(e, "1"))) ? 1 : 0;
    }
    return g_lut_mode;
}
int kernel_sel() {
    std::lock_guard<std::recursive_mutex> lk(g_state_mu);
    if (g_kernel_sel < 0) {
        const char *e = getenv("SQLLM_KERNEL");
        g_kernel_sel = (e && !strcmp(e, "v1")) ? 1 : 2;
    }
    return g_kernel_sel;
}

typedef void (*K2)(const v2::P2, const CUtensorMap, const CUtensorMap);
struct K2Info { K2 fn; int tab, stage; };
// [bits==4][variant][fused] ; variant 0: exact, fp32 x ; 1: exact, fp16 x ; 2: fp16 pair table, fp16 x
K2Info k2_lookup(int bits, int variant, bool fused) {
#define K2E(B, M, XH, F) K2Info{v2::lutgemv2_kernel<B, M, XH, F>, v2::C2<B, M>::TAB, v2::C2<B, M>::STAGE}
    if (bits == 4) {
        if (variant == 0) return fused ? K2E(4, 0, false, true) : K2E(4, 0, false, false);
        if (variant == 1) return fused ? K2E(4, 0, true, true) : K2E(4, 0, true, false);
        return fused ? K2E(4, 1, true, true) : K2E(4, 1, true, false);
    }
    if (variant == 0) return fused ? K2E(3, 0, false, true) : K2E(3, 0, false, false);
    if (variant == 1) return fused ? K2E(3, 0, true, true) : K2E(3, 0, true, false);
    return fused ? K2E(3, 1, true, true) : K2E(3, 1, true, false);
#undef K2E
}

struct Plan2 {
    int R, strips, T, chunk, G, nstage, smem, hc, hrows, csr_rpc;
    unsigned smem_raw;
};
unsigned g_smem_raw[64] = {};

int make_plan2(int bits, int K, int N, int topX, int variant, bool fused, Plan2 &pl, K2Info &ki) {
    int dev = 0, sm = 0;
    unsigned smem_raw = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return fail(SQLLM_ECUDA, "cudaGetDevice failed");
    if (dev < 0 || dev >= 64) return fail(SQLLM_EINVAL, "device ordinal %d out of range", dev);
    {
        std::lock_guard<std::recursive_mutex> lk(g_state_mu);
        DevInfo &d = g_dev[dev];
        if (d.sm == 0 && (cudaDeviceGetAttribute(&d.sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || d.sm <= 0)) {
            d.sm = 0;
            return fail(SQLLM_ECUDA, "cannot query SM count");
        }
        sm = d.sm;
        if (!g_v2_attr[dev]) {
            for (int b = 3; b <= 4; ++b)
                for (int v = 0; v < 3; ++v)
                    for (int f = 0; f < 2; ++f)
                        if (cudaFuncSetAttribute(k2_lookup(b, v, f != 0).fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
                            return fail(SQLLM_ECUDA, "cudaFuncSetAttribute failed: %s", cudaGetErrorString(cudaGetLastError()));
            // one-time probe (synchronous; refused during stream capture, so the first call must come before capture - any warm-up does)
            unsigned *d_out = nullptr, h_out = 0;
            cudaError_t pe = cudaMalloc(&d_out, sizeof(unsigned));
            if (pe == cudaSuccess) {
                smem_base_probe<<<1, 1, 1024>>>(d_out);
                pe = cudaMemcpy(&h_out, d_out, sizeof(unsigned), cudaMemcpyDeviceToHost);
                cudaFree(d_out);
            }
            if (pe != cudaSuccess || h_out == 0) {
                cudaGetLastError();
                return fail(SQLLM_ECUDA, "shared-memory probe failed (first call inside a stream capture? run one call before capturing): %s", cudaGetErrorString(pe));
            }
            g_smem_raw[dev] = h_out;
            g_v2_attr[dev] = true;
        }
        smem_raw = g_smem_raw[dev];
    }
    ki = k2_lookup(bits, variant, fused);
    pl.R = bits == 4 ? K / 8 : K / 32;
    pl.strips = (N + STRIP - 1) / STRIP;
    const long long T = (long long)pl.strips * pl.R;
    if (T > 0x3fffffff) return fail(SQLLM_EINVAL, "problem too large");
    if (fused && N > MAX_N_FUSED) return fail(SQLLM_EINVAL, "out_features=%d exceeds the fused accumulator (max %d)", N, MAX_N_FUSED);
    pl.T = (int)T;
    int chunk = (int)(2 * ((T + 2LL * sm - 1) / (2LL * sm)));
    if (chunk < 2) chunk = 2;
    pl.chunk = chunk;
    pl.G = (int)((T + chunk - 1) / chunk);
    if (fused && pl.G > MAX_GRID_V2) return fail(SQLLM_EINVAL, "grid of %d CTAs exceeds the mailbox area (%d)", pl.G, MAX_GRID_V2);
    // shared memory, exactly as lutgemv2_kernel carves it: [fixed][x][ring stages ...][table 0][table 1][... ring stages]
    const unsigned raw = smem_raw;
    const unsigned base = (raw + 127u) & ~127u;
    const unsigned lo_base = base + v2::OFF_X + (unsigned)((K * (variant == 0 ? 4 : 2) + 127) & ~127);
    const unsigned tab0 = (lo_base + (unsigned)ki.tab - 1u) & ~((unsigned)ki.tab - 1u);
    const long long limit = (long long)raw + 227 * 1024;
    const long long hi_room = limit - ((long long)tab0 + 2LL * ki.tab);
    if (hi_room < 0) return fail(SQLLM_EINVAL, "in_features=%d does not fit the shared-memory carve-up of this table mode", K);
    const int lo_cap = (int)((tab0 - lo_base) / (unsigned)ki.stage), hi_cap = (int)(hi_room / ki.stage);
    int n = (chunk + v2::SU2 - 1) / v2::SU2 + 1;
    if (n > v2::MAXD) n = v2::MAXD;
    if (n > lo_cap + hi_cap) n = lo_cap + hi_cap;
    if (n < 2) return fail(SQLLM_EINVAL, "in_features=%d leaves no room for a weight ring in shared memory", K);
    const int n_lo = n < lo_cap ? n : lo_cap;
    pl.nstage = n;
    pl.smem = (int)((long long)tab0 + 2LL * ki.tab + (long long)(n - n_lo) * ki.stage - raw);
    pl.smem_raw = raw;
    pl.csr_rpc = (N + pl.G - 1) / pl.G;
    pl.hc = pl.hrows = 0;
    if (topX > 0) {
        pl.hrows = (K + pl.G - 1) / pl.G;
        pl.hc = (K + pl.hrows - 1) / pl.hrows;
    }
    return SQLLM_OK;
}

int launch2(const sqllm_lutgemv_args *a, int variant, bool fused, v2::P2 &p, cudaStream_t st) {
    const bool hyb = a->full_rows && a->topX > 0;
    Plan2 pl;
    K2Info ki;
    const int rc = make_plan2(a->bits, a->in_features, a->out_features, hyb ? a->topX : 0, variant, fused, pl, ki);
    if (rc) return rc;
    p.qw = reinterpret_cast<const uint32_t *>(a->qweight);
    p.lut = a->lookup_table;
    p.rows = a->rows; p.cols = a->cols; p.vals = a->vals;
    p.full_rows = hyb ? a->full_rows : nullptr;
    p.fri = hyb ? a->full_row_indices : nullptr;
    p.topX = hyb ? a->topX : 0;
    p.K = a->in_features; p.N = a->out_features;
    p.R = pl.R; p.T = pl.T; p.chunk = pl.chunk; p.nstage = pl.nstage; p.smem_raw = pl.smem_raw;
    p.hc = hyb ? pl.hc : 0; p.hrows = pl.hrows;
    p.csr_rpc = pl.csr_rpc;
    p.csr_al16 = (a->rows && ((reinterpret_cast<uintptr_t>(a->cols) | reinterpret_cast<uintptr_t>(a->vals)) & 15) == 0) ? 1 : 0;
    p.strips = pl.strips;
    p.nown_ctas = 0;
    if (p.xw_world)
        for (int b = 0; b < pl.G; ++b) {  // CTAs in whose range at least one strip starts
            const long long c0 = (long long)b * pl.chunk, c1 = std::min<long long>(pl.T, c0 + pl.chunk);
            if ((c0 + pl.R - 1) / pl.R < (c1 + pl.R - 1) / pl.R) ++p.nown_ctas;
        }
    {
        std::lock_guard<std::recursive_mutex> lk(g_state_mu);
        p.trace = g_trace;
        if (g_trace) g_trace += g_trace_stride;
        g_last_grid = pl.G;
        if (g_use_pdl < 0) {
            const char *e = getenv("SQLLM_NO_PDL");
            g_use_pdl = (e && e[0] == '1') ? 0 : 1;
        }
        static int l2pf = -1;
        if (l2pf < 0) {
            const char *e = getenv("SQLLM_L2PF");
            l2pf = e ? (e[0] == '1') : 0;
        }
        p.l2pf = l2pf;
        static int sp_w0 = -1;
        if (sp_w0 < 0) {
            const char *e = getenv("SQLLM_SP_W0");
            sp_w0 = e ? (e[0] == '1') : 0;
        }
        p.sp_w0 = sp_w0;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(pl.G);
    cfg.blockDim = dim3(v2::THREADS2);
    cfg.dynamicSmemBytes = pl.smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_use_pdl ? 1 : 0;
    // two tensor maps over the packed matrix: 64 columns x (32 units | 2 units) boxes
    const int rows_per_unit = a->bits == 4 ? 1 : 3, qrows = a->in_features / 32 * a->bits;
    CUtensorMap tm_big, tm_small;
    // (a matrix shorter than one full stage never issues the big box; its map is clamped so that the encoder accepts it)
    int trc = get_tensor_map(a->qweight, qrows, a->out_features, qrows < v2::SU2 * rows_per_unit ? 2 * rows_per_unit : v2::SU2 * rows_per_unit, tm_big);
    if (trc) return trc;
    trc = get_tensor_map(a->qweight, qrows, a->out_features, 2 * rows_per_unit, tm_small);
    if (trc) return trc;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, ki.fn, p, tm_big, tm_small);
    if (e != cudaSuccess) return fail(SQLLM_ECUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    return SQLLM_OK;
}


// ---- sequences (lutgemv_seq.cuh): plan + descriptors at create time, two launches per run -----------------------------
typedef void (*KSeq)(const seq::SeqCfg);
struct KSeqInfo { KSeq fn; int tab, stage, ntb; };
KSeqInfo kseq_lookup(int bits, int mode, bool multi) {
#define KSE(B, M, X) KSeqInfo{seq::lutgemv_seq_kernel<B, M, X>, v2::C2<B, M>::TAB, v2::C2<B, M>::STAGE, v2::C2<B, M>::TAB <= 16384 ? 4 : 2}
    if (bits == 4) {
        if (mode == 0) return multi ? KSE(4, 0, true) : KSE(4, 0, false);
        return multi ? KSE(4, 1, true) : KSE(4, 1, false);
    }
    if (mode == 0) return multi ? KSE(3, 0, true) : KSE(3, 0, false);
    return multi ? KSE(3, 1, true) : KSE(3, 1, false);
#undef KSE
}
constexpr int SEQ_MAX_ITEMS = 1023;  // the mailbox tag keeps 10 bits for the item

size_t seq_item_len(const sqllm_seq_item &it) {  // elements of the item's full-length output vector
    const int members = it.members > 0 ? it.members : 1;
    const int nfull = it.out_features_full > 0 ? it.out_features_full : it.a.out_features / members;
    return (size_t)members * nfull;
}
}  // namespace

struct sqllm_sequence {
    int dev = 0, n = 0, bits = 0, mode = 0, world = 1, rank = 0, grid = 0, smem = 0, coop = 1;
    seq::SeqCfg cfg;
    KSeq fn = nullptr;
    void *d_descs = nullptr, *d_exports = nullptr, *d_ws = nullptr, *d_arena = nullptr;
    bool own_arena = false;
};

namespace {
int seq_fail_free(sqllm_sequence *s, int rc) {
    if (s) sqllm_sequence_destroy(s);
    return rc;
}
}  // namespace

extern "C" size_t sqllm_sequence_arena_bytes(const sqllm_seq_item *items, int n_items) {
    if (!items || n_items <= 0) return 0;
    size_t off = 0;
    for (int i = 0; i < n_items; ++i) off += (seq_item_len(items[i]) * 4 + 127) / 128 * 128;
    return off;
}

extern "C" int sqllm_sequence_create(const sqllm_seq_item *items, int n_items, const sqllm_seq_options *opt, sqllm_sequence **out) {
    if (!items || !opt || !out || n_items <= 0) return fail(SQLLM_EINVAL, "sequence: null / empty arguments");
    if (n_items > SEQ_MAX_ITEMS) return fail(SQLLM_EINVAL, "sequence: at most %d items (got %d)", SEQ_MAX_ITEMS, n_items);
    const int world = opt->world > 0 ? opt->world : 1, rank = opt->rank;
    if (world > 64 || rank < 0 || rank >= world) return fail(SQLLM_EINVAL, "sequence: bad world / rank (%d / %d)", world, rank);
    if (world > 1 && (!opt->arena || !opt->peer_base)) return fail(SQLLM_EINVAL, "sequence: several GPUs need a peer-visible arena and peer_base");
    const int bits = items[0].a.bits, mode = opt->lut_mode == SQLLM_LUT_FP16_PAIR ? 1 : 0;
    int kmax = 0;
    for (int i = 0; i < n_items; ++i) {
        const sqllm_seq_item &it = items[i];
        sqllm_lutgemv_args a = it.a;
        a.batch = 1;
        a.vec = reinterpret_cast<const float *>(16);  // (vec / mul are not used by a sequence; check_common wants them non-null)
        a.mul = reinterpret_cast<float *>(16);
        const int rc = check_common(&a);
        if (rc) return rc;
        if (a.bits != bits) return fail(SQLLM_EINVAL, "sequence: item %d has bits=%d, item 0 has %d (one sequence, one width)", i, a.bits, bits);
        if (a.out_features < STRIP) return fail(SQLLM_EINVAL, "sequence: item %d: out_features=%d < %d", i, a.out_features, STRIP);
        if (a.out_features > MAX_N_FUSED) return fail(SQLLM_EINVAL, "sequence: item %d: out_features=%d exceeds %d", i, a.out_features, MAX_N_FUSED);
        if (a.full_rows && a.topX > MAX_TOPX_FUSED) return fail(SQLLM_EINVAL, "sequence: topX <= %d", MAX_TOPX_FUSED);
        const int members = it.members > 0 ? it.members : 1;
        if (a.out_features % members || (a.out_features / members) % 4) return fail(SQLLM_EINVAL, "sequence: item %d: %d columns are not %d members of a multiple of 4", i, a.out_features, members);
        if (world == 1 && seq_item_len(it) != (size_t)a.out_features) return fail(SQLLM_EINVAL, "sequence: item %d: members * out_features_full must equal out_features on one GPU", i);
        if (world > 1 && seq_item_len(it) < (size_t)world * a.out_features) return fail(SQLLM_EINVAL, "sequence: item %d: full length %zu < world * shard columns", i, seq_item_len(it));
        if (world > 1 && it.y) return fail(SQLLM_EINVAL, "sequence: item %d: plain y copies exist on one GPU only (use exports)", i);
        if (seq_item_len(it) % 4) return fail(SQLLM_EINVAL, "sequence: item %d: output length must be a multiple of 4", i);
        if (it.x_from >= i || it.x_from < -1) return fail(SQLLM_EINVAL, "sequence: item %d: x_from=%d must name an earlier item (or -1)", i, it.x_from);
        if (it.x_from < 0) {
            if (!it.x_ext || (reinterpret_cast<uintptr_t>(it.x_ext) & 15)) return fail(SQLLM_EINVAL, "sequence: item %d: x_ext must be a 16-byte aligned fp16 vector", i);
        } else {
            if (it.x_offset < 0 || it.x_offset % 4 || (size_t)it.x_offset + a.in_features > seq_item_len(items[it.x_from]))
                return fail(SQLLM_EINVAL, "sequence: item %d reads [%d, %d) of item %d's %zu outputs", i, it.x_offset, it.x_offset + a.in_features, it.x_from, seq_item_len(items[it.x_from]));
        }
        if ((reinterpret_cast<uintptr_t>(it.y) & 1) || (reinterpret_cast<uintptr_t>(it.bias) & 3)) return fail(SQLLM_EINVAL, "sequence: item %d: misaligned y / bias", i);
        kmax = std::max(kmax, a.in_features);
    }
    for (int e = 0; e < opt->n_export; ++e) {
        if (!opt->export_items || !opt->export_dst) return fail(SQLLM_EINVAL, "sequence: export arrays missing");
        const int it = opt->export_items[e];
        if (it < 0 || it >= n_items || !opt->export_dst[e] || (reinterpret_cast<uintptr_t>(opt->export_dst[e]) & 7))
            return fail(SQLLM_EINVAL, "sequence: export %d: bad item %d or destination (8-byte aligned fp16 vector)", e, it);
    }
    // device attributes, shared-memory window, kernel attribute (make_plan2 does the one-time probe)
    Plan2 probe;
    K2Info ki2;
    int rc = make_plan2(bits, items[0].a.in_features, items[0].a.out_features, 0, mode ? 2 : 1, true, probe, ki2);
    if (rc) return rc;
    const KSeqInfo ki = kseq_lookup(bits, mode, world > 1);
    int dev = 0, sm = 0;
    cudaGetDevice(&dev);
    {
        std::lock_guard<std::recursive_mutex> lk(g_state_mu);
        sm = g_dev[dev].sm;
    }
    if (cudaFuncSetAttribute(ki.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
        return fail(SQLLM_ECUDA, "cudaFuncSetAttribute failed: %s", cudaGetErrorString(cudaGetLastError()));
    // shared memory, exactly as lutgemv_seq_kernel carves it: [fixed][x][strip sums][ring stages ...][tables][... ring stages]
    const unsigned raw = probe.smem_raw, base = (raw + 127u) & ~127u;
    const int xbytes = (kmax * 2 + 127) & ~127;
    const unsigned lo_base = base + v2::OFF_X + (unsigned)xbytes + (unsigned)ki.ntb * STRIP * 4;
    const unsigned tab0 = (lo_base + (unsigned)ki.tab - 1u) & ~((unsigned)ki.tab - 1u);
    const long long limit = (long long)raw + 227 * 1024;
    const long long hi_room = limit - ((long long)tab0 + (long long)ki.ntb * ki.tab);
    if (hi_room < 0) return fail(SQLLM_EINVAL, "sequence: in_features=%d does not fit the shared-memory carve-up of this table mode", kmax);
    const int lo_cap = (int)((tab0 - lo_base) / (unsigned)ki.stage), hi_cap = (int)(hi_room / ki.stage);
    int nst = std::min(v2::MAXD, lo_cap + hi_cap);
    if (const char *e = getenv("SQLLM_SEQ_STAGES")) nst = std::max(2, std::min(nst, atoi(e)));  // experiments: a shallower weight ring
    if (nst < 2) return fail(SQLLM_EINVAL, "sequence: in_features=%d leaves no room for a weight ring in shared memory", kmax);
    const int n_lo = std::min(nst, lo_cap);
    const int smem = (int)((long long)tab0 + (long long)ki.ntb * ki.tab + (long long)(nst - n_lo) * ki.stage - raw);

    sqllm_sequence *s = new sqllm_sequence();
    s->dev = dev; s->n = n_items; s->bits = bits; s->mode = mode; s->world = world; s->rank = rank; s->grid = sm; s->smem = smem; s->fn = ki.fn;
    {
        const char *e = getenv("SQLLM_SEQ_COOP");
        s->coop = (e && e[0] == '0') ? 0 : 1;
    }
    // workspace: [0,4) token counter, [64,68) error word, per parity {flags [64 + MAX_STRIPS] ints, accumulator [MAX_N_FUSED] floats} (only
    // used by CTAs that own more than 8 strips), then EVERY item's own mailboxes: outlier row sums [N], partial strip sums [grid][64],
    // dense-row parts [topX][MAX_GRID_V2].  Mailboxes are not shared between items: an item may read only a slice of its predecessor's
    // output, so "x of item g+1 is complete" does not mean that every strip owner of item g has already taken its words.
    const size_t cnt_bytes = (size_t)(64 + MAX_STRIPS) * 4, acc_bytes = (size_t)MAX_N_FUSED * 4;
    const size_t par_off = 256, par_bytes = (cnt_bytes + acc_bytes + 255) / 256 * 256;
    std::vector<size_t> cbox_off(n_items), hbox_off(n_items), dbox_off(n_items);
    size_t ws_bytes = par_off + 2 * par_bytes;
    for (int i = 0; i < n_items; ++i) {
        const bool hyb = items[i].a.full_rows && items[i].a.topX > 0;
        cbox_off[i] = ws_bytes; ws_bytes += ((size_t)items[i].a.out_features * 8 + 255) / 256 * 256;
        hbox_off[i] = ws_bytes; ws_bytes += (size_t)MAX_GRID_V2 * 64 * 8;
        dbox_off[i] = ws_bytes; ws_bytes += hyb ? (size_t)items[i].a.topX * MAX_GRID_V2 * 8 : 0;
    }
    if (cudaMalloc(&s->d_ws, ws_bytes) != cudaSuccess || cudaMemset(s->d_ws, 0, ws_bytes) != cudaSuccess)
        return seq_fail_free(s, fail(SQLLM_ECUDA, "sequence: workspace allocation failed"));
    unsigned char *ws = static_cast<unsigned char *>(s->d_ws);
    const size_t arena_need = sqllm_sequence_arena_bytes(items, n_items);
    if (opt->arena) {
        if (opt->arena_bytes < arena_need || (reinterpret_cast<uintptr_t>(opt->arena) & 127))
            return seq_fail_free(s, fail(SQLLM_EINVAL, "sequence: arena of %zu bytes (128-byte aligned) needed, got %zu", arena_need, opt->arena_bytes));
        s->d_arena = opt->arena;
    } else {
        if (cudaMalloc(&s->d_arena, arena_need) != cudaSuccess || cudaMemset(s->d_arena, 0, arena_need) != cudaSuccess)
            return seq_fail_free(s, fail(SQLLM_ECUDA, "sequence: arena allocation failed"));
        s->own_arena = true;
    }
    std::vector<seq::SeqDesc> descs(n_items);
    std::vector<size_t> yoff(n_items);
    size_t off = 0;
    for (int i = 0; i < n_items; ++i) {
        yoff[i] = off;
        off += (seq_item_len(items[i]) * 4 + 127) / 128 * 128;
    }
    for (int i = 0; i < n_items; ++i) {
        const sqllm_seq_item &it = items[i];
        const sqllm_lutgemv_args &a = it.a;
        seq::SeqDesc &d = descs[i];
        memset(&d, 0, sizeof(d));
        v2::P2 &p = d.p;
        const bool hyb = a.full_rows && a.topX > 0;
        const int K = a.in_features, N = a.out_features;
        p.qw = reinterpret_cast<const uint32_t *>(a.qweight);
        p.lut = a.lookup_table;
        p.rows = a.rows; p.cols = a.cols; p.vals = a.vals;
        p.full_rows = hyb ? a.full_rows : nullptr;
        p.fri = hyb ? a.full_row_indices : nullptr;
        p.topX = hyb ? a.topX : 0;
        p.K = K; p.N = N;
        p.R = bits == 4 ? K / 8 : K / 32;
        p.strips = (N + STRIP - 1) / STRIP;
        const long long T = (long long)p.strips * p.R;
        if (T > 0x3fffffff) return seq_fail_free(s, fail(SQLLM_EINVAL, "sequence: item %d too large", i));
        p.T = (int)T;
        int chunk = (int)(2 * ((T + 2LL * sm - 1) / (2LL * sm)));
        if (chunk < 2) chunk = 2;
        p.chunk = chunk;
        const int G = (int)((T + chunk - 1) / chunk);
        if (G > MAX_GRID_V2) return seq_fail_free(s, fail(SQLLM_EINVAL, "sequence: grid of %d CTAs exceeds the mailbox area", G));
        p.nstage = nst; p.smem_raw = raw;
        p.csr_rpc = (N + G - 1) / G;
        if (a.rows && p.csr_rpc > v2::SP_ROWS) return seq_fail_free(s, fail(SQLLM_EINVAL, "sequence: item %d: %d outlier rows per CTA exceed %d", i, p.csr_rpc, v2::SP_ROWS));
        p.hc = p.hrows = 0;
        if (hyb) {
            p.hrows = (K + G - 1) / G;
            p.hc = (K + p.hrows - 1) / p.hrows;
        }
        p.csr_al16 = (a.rows && ((reinterpret_cast<uintptr_t>(a.cols) | reinterpret_cast<uintptr_t>(a.vals)) & 15) == 0) ? 1 : 0;
        p.y_is_half = 1;
        p.bias = it.bias;
        p.out = it.y;
        p.x = it.x_from < 0 ? it.x_ext : nullptr;
        unsigned char *par = ws + par_off + (size_t)(i & 1) * par_bytes;
        p.ws_cnt = reinterpret_cast<int *>(par);
        p.ws_acc = reinterpret_cast<float *>(par + cnt_bytes);
        p.ws_hbox = reinterpret_cast<unsigned long long *>(ws + hbox_off[i]);
        p.ws_cbox = reinterpret_cast<unsigned long long *>(ws + cbox_off[i]);
        p.ws_dbox = reinterpret_cast<unsigned long long *>(ws + dbox_off[i]);
        p.xw_world = world > 1 ? world : 0; p.xw_rank = rank;
        p.xw_members = it.members > 0 ? it.members : 1;
        p.xw_nfull = it.out_features_full > 0 ? it.out_features_full : N / p.xw_members;
        p.trace = opt->trace ? reinterpret_cast<unsigned long long *>(opt->trace) + (size_t)i * 1024 * 32 : nullptr;
        d.x_tag = it.x_from < 0 ? nullptr : reinterpret_cast<const uint32_t *>(static_cast<unsigned char *>(s->d_arena) + yoff[it.x_from]) + it.x_offset;
        d.y_off = yoff[i];
        const int rows_per_unit = bits == 4 ? 1 : 3, qrows = K / 32 * bits;
        rc = get_tensor_map(a.qweight, qrows, N, qrows < v2::SU2 * rows_per_unit ? 2 * rows_per_unit : v2::SU2 * rows_per_unit, d.tm_big);
        if (!rc) rc = get_tensor_map(a.qweight, qrows, N, 2 * rows_per_unit, d.tm_small);
        if (rc) return seq_fail_free(s, rc);
    }
    std::vector<seq::SeqExport> ex(std::max(1, opt->n_export));
    for (int e = 0; e < opt->n_export; ++e) {
        const int it = opt->export_items[e];
        ex[e].src = reinterpret_cast<const uint32_t *>(static_cast<unsigned char *>(s->d_arena) + yoff[it]);
        ex[e].dst = opt->export_dst[e];
        ex[e].n = (int)seq_item_len(items[it]);
    }
    if (cudaMalloc(&s->d_descs, descs.size() * sizeof(seq::SeqDesc)) != cudaSuccess ||
        cudaMemcpy(s->d_descs, descs.data(), descs.size() * sizeof(seq::SeqDesc), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMalloc(&s->d_exports, ex.size() * sizeof(seq::SeqExport)) != cudaSuccess ||
        cudaMemcpy(s->d_exports, ex.data(), ex.size() * sizeof(seq::SeqExport), cudaMemcpyHostToDevice) != cudaSuccess)
        return seq_fail_free(s, fail(SQLLM_ECUDA, "sequence: descriptor upload failed: %s", cudaGetErrorString(cudaGetLastError())));
    seq::SeqCfg &c = s->cfg;
    memset(&c, 0, sizeof(c));
    c.descs = static_cast<const seq::SeqDesc *>(s->d_descs);
    c.ngemv = n_items;
    c.epoch = reinterpret_cast<const unsigned *>(ws);
    c.err = reinterpret_cast<int *>(ws + 64);
    c.smem_raw = raw; c.xbytes = xbytes; c.nstage = nst;
    c.world = world; c.rank = rank;
    c.peer_base = reinterpret_cast<const unsigned long long *>(opt->peer_base);
    c.arena_base = reinterpret_cast<unsigned long long>(s->d_arena);
    c.exports = static_cast<const seq::SeqExport *>(s->d_exports);
    c.nexport = opt->n_export;
    *out = s;
    return SQLLM_OK;
}

extern "C" int sqllm_sequence_run(sqllm_sequence *s, void *stream) {
    if (!s) return fail(SQLLM_EINVAL, "sequence: null handle");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    seq::seq_bump_epoch<<<1, 1, 0, st>>>(reinterpret_cast<unsigned *>(s->d_ws));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(s->grid);
    cfg.blockDim = dim3(v2::THREADS2);
    cfg.dynamicSmemBytes = s->smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;  // every CTA waits on every other one: they must all be resident
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = s->coop ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, s->fn, s->cfg);
    if (e != cudaSuccess) return fail(SQLLM_ECUDA, "sequence launch failed: %s", cudaGetErrorString(e));
    return SQLLM_OK;
}

extern "C" int sqllm_sequence_error(sqllm_sequence *s, void *stream) {
    if (!s) return fail(SQLLM_EINVAL, "sequence: null handle");
    int h = 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (cudaMemcpyAsync(&h, static_cast<unsigned char *>(s->d_ws) + 64, 4, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess)
        return fail(SQLLM_ECUDA, "sequence: reading the error word failed: %s", cudaGetErrorString(cudaGetLastError()));
    return h != 0;
}

extern "C" int sqllm_sequence_reset_error(sqllm_sequence *s, void *stream) {
    if (!s) return fail(SQLLM_EINVAL, "sequence: null handle");
    if (cudaMemsetAsync(static_cast<unsigned char *>(s->d_ws) + 64, 0, 4, static_cast<cudaStream_t>(stream)) != cudaSuccess)
        return fail(SQLLM_ECUDA, "sequence: clearing the error word failed: %s", cudaGetErrorString(cudaGetLastError()));
    return SQLLM_OK;
}

extern "C" void sqllm_sequence_destroy(sqllm_sequence *s) {
    if (!s) return;
    cudaFree(s->d_descs);
    cudaFree(s->d_exports);
    cudaFree(s->d_ws);
    if (s->own_arena) cudaFree(s->d_arena);
    delete s;
}

namespace {

// ---- batched symbols: tile kernel + outlier kernels (lutgemm_batched.cuh) ----------------------------------------------
bool g_batched_attr[64] = {};
int launch_batched(const sqllm_lutgemv_args *a, cudaStream_t st) {
    using namespace batched;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return fail(SQLLM_ECUDA, "cudaGetDevice failed");
    {
        std::lock_guard<std::recursive_mutex> lk(g_state_mu);
        if (!g_batched_attr[dev]) {
            if (cudaFuncSetAttribute(lutgemm_batched_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess ||
                cudaFuncSetAttribute(lutgemm_batched_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
                return fail(SQLLM_ECUDA, "cudaFuncSetAttribute failed: %s", cudaGetErrorString(cudaGetLastError()));
            g_batched_attr[dev] = true;
        }
    }
    const int K = a->in_features, N = a->out_features, B = a->batch;
    const int XU = a->bits == 4 ? 8 : 32, tab = a->bits == 4 ? CB<4>::TAB : CB<3>::TAB;
    PB p;
    p.qw = reinterpret_cast<const uint32_t *>(a->qweight); p.lut = a->lookup_table; p.x = a->vec; p.mul = a->mul;
    p.K = K; p.N = N; p.B = B; p.R = K / XU;
    // K-slabs: the BT x rows of a slab sit in shared memory next to the table and the partial sums; <= 2048 inputs per slab keeps a
    // CTA under 90 KB, i.e. two CTAs (16 warps) per SM
    int slabs = (K + 2047) / 2048;
    p.ks = 2 * ((p.R + 2 * slabs - 1) / (2 * slabs));
    slabs = (p.R + p.ks - 1) / p.ks;
    const int kslab = p.ks * XU;
    const size_t smem = (size_t)2 * tab + (size_t)BT * (kslab * 4 + 16) + (size_t)BW * BT * STRIP * 4;
    if (smem > 227 * 1024) return fail(SQLLM_EINVAL, "batched tile needs %zu B of shared memory", smem);
    const int strips = (N + STRIP - 1) / STRIP, btiles = (B + BT - 1) / BT;
    if (btiles > 65535) return fail(SQLLM_EINVAL, "batch=%d is too large for one call (max %d)", B, 65535 * BT);
    const dim3 grid(strips, slabs, btiles);
    if (a->bits == 4) lutgemm_batched_kernel<4><<<grid, BTHREADS, smem, st>>>(p);
    else lutgemm_batched_kernel<3><<<grid, BTHREADS, smem, st>>>(p);
    if (a->rows) {
        const dim3 blk(32, 8), g((N + 7) / 8, std::min((B + 31) / 32, 64));
        csr_batched_kernel<<<g, blk, 0, st>>>(a->rows, a->cols, a->vals, a->vec, a->mul, K, N, B);
    }
    if (a->full_rows && a->topX > 0) {
        const int w = std::min(64, a->topX), per = 256 / w;  // blocks of at most 64 dense rows, any number of them
        dense_rows_batched_kernel<<<dim3(B, (a->topX + w - 1) / w), per * w, 0, st>>>(a->full_rows, a->full_row_indices, a->topX, w, a->vec, a->mul, K, N, B);
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(SQLLM_ECUDA, "batched launch failed: %s", cudaGetErrorString(e));
    return SQLLM_OK;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int sqllm_abi_version(void) { return SQLLM_ABI_VERSION; }
void sqllm_set_deterministic(int on) {
    std::lock_guard<std::recursive_mutex> lk(g_state_mu);
    g_det = on ? 1 : 0;
}
void sqllm_set_lut_mode(int mode) {
    std::lock_guard<std::recursive_mutex> lk(g_state_mu);
    g_lut_mode = mode == SQLLM_LUT_FP16_PAIR ? 1 : 0;
}
int sqllm_get_lut_mode(void) { return lut_mode(); }
int sqllm_workspace_error(const void *workspace, void *stream) {
    if (!workspace) return fail(SQLLM_EINVAL, "null workspace");
    int flag = 0;
    if (cudaMemcpyAsync(&flag, static_cast<const unsigned char *>(workspace) + 64, 4, cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)) != cudaSuccess ||
        cudaStreamSynchronize(static_cast<cudaStream_t>(stream)) != cudaSuccess)
        return fail(SQLLM_ECUDA, "cannot read the workspace error word: %s", cudaGetErrorString(cudaGetLastError()));
    return flag ? 1 : 0;
}

// debug hook (not in the public header): successive launches write their timeline at buf, buf+stride, ...
void sqllm_debug_set_trace(unsigned long long *buf, size_t stride_words) { g_trace = buf; g_trace_stride = stride_words; }
int sqllm_debug_last_grid(void) { return g_last_grid; }
const char *sqllm_last_error(void) { return g_err; }

int sqllm_device_sm_count(void) {
    int dev = 0, sm = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    return sm;
}

size_t sqllm_workspace_bytes(int bits, int in_features, int out_features, int topX) {
    Plan pl;
    if (bits != 3 && bits != 4) return 0;
    if (in_features <= 0 || in_features % 64 || out_features <= 0) return 0;
    // CSR staging changes the shared-memory footprint, hence occupancy, grid and chunk: take the max of both plans.
    size_t b = 0;
    for (int csr = 0; csr < 2; ++csr)
        if (make_plan(bits, in_features, out_features, topX, csr != 0, true, pl) == SQLLM_OK && pl.ws_bytes > b) b = pl.ws_bytes;
    return b;
}

int sqllm_lutgemv(const sqllm_lutgemv_args *a, void *stream) {
    int rc = check_common(a);
    if (rc) return rc;
    if (!a->vec || !a->mul) return fail(SQLLM_EINVAL, "vec / mul must not be null");
    if (a->batch < 1) return fail(SQLLM_EINVAL, "batch must be >= 1");
    if (reinterpret_cast<uintptr_t>(a->vec) & 15) return fail(SQLLM_EINVAL, "vec must be 16-byte aligned");
    const bool hyb = a->full_rows && a->topX > 0;
    if (a->batch >= 2) {
        static int loop_mode = -1;  // SQLLM_BATCHED=loop: one batch-1 launch per row, as in round 1 (A/B runs)
        {
            std::lock_guard<std::recursive_mutex> lk(g_state_mu);
            if (loop_mode < 0) { const char *e = getenv("SQLLM_BATCHED"); loop_mode = (e && !strcmp(e, "loop")) ? 1 : 0; }
        }
        if (!loop_mode) return launch_batched(a, static_cast<cudaStream_t>(stream));
    }
    if (kernel_sel() == 2 && a->out_features >= STRIP) {
        v2::P2 q;
        memset(&q, 0, sizeof(q));
        for (int b = 0; b < a->batch; ++b) {  // serial over batch rows, like the reference's in-kernel `for b` (:1011)
            q.x = a->vec + (size_t)b * a->in_features;
            q.out = a->mul + (size_t)b * a->out_features;
            rc = launch2(a, 0, false, q, static_cast<cudaStream_t>(stream));
            if (rc) return rc;
        }
        return SQLLM_OK;
    }
    Plan pl;
    rc = make_plan(a->bits, a->in_features, a->out_features, hyb ? a->topX : 0, a->rows != nullptr, false, pl);
    if (rc) return rc;
    Params p;
    memset(&p, 0, sizeof(p));
    for (int b = 0; b < a->batch; ++b) {  // serial over batch rows, like the reference's in-kernel `for b` (:1011)
        p.x = a->vec + (size_t)b * a->in_features;
        p.out = a->mul + (size_t)b * a->out_features;
        p.x_is_half = 0;
        rc = launch<false>(a, pl, p, static_cast<cudaStream_t>(stream));
        if (rc) return rc;
    }
    return SQLLM_OK;
}

int sqllm_lutgemv_fused(const sqllm_lutgemv_args *a, const void *x, int x_is_half, void *y, int y_is_half,
                        const float *bias, void *workspace, size_t workspace_bytes, void *stream) {
    int rc = check_common(a);
    if (rc) return rc;
    if (!x || !y) return fail(SQLLM_EINVAL, "x / y must not be null");
    if (reinterpret_cast<uintptr_t>(x) & 15) return fail(SQLLM_EINVAL, "x must be 16-byte aligned");
    if ((reinterpret_cast<uintptr_t>(y) & 15) || (reinterpret_cast<uintptr_t>(bias) & 15)) return fail(SQLLM_EINVAL, "y and bias must be 16-byte aligned");
    const bool hyb = a->full_rows && a->topX > 0;
    if (hyb && a->topX > MAX_TOPX_FUSED) return fail(SQLLM_EINVAL, "fused path supports topX <= %d", MAX_TOPX_FUSED);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    if (det_mode() == 0 && kernel_sel() == 2 && a->out_features >= STRIP) {
        if (!workspace || workspace_bytes < WS_HEADER) return fail(SQLLM_EWORKSPACE, "workspace too small: need %zu bytes, got %zu", (size_t)WS_HEADER, workspace_bytes);
        v2::P2 q;
        memset(&q, 0, sizeof(q));
        q.ws_cnt = reinterpret_cast<int *>(ws);
        q.ws_acc = reinterpret_cast<float *>(ws + WS_ACC_OFF);
        q.ws_hbox = reinterpret_cast<unsigned long long *>(ws + WS_HBOX_OFF);
        q.ws_cbox = reinterpret_cast<unsigned long long *>(ws + WS_CBOX_OFF);
        q.ws_dbox = reinterpret_cast<unsigned long long *>(ws + WS_DBOX_OFF);
        q.x = x; q.out = y; q.y_is_half = y_is_half; q.bias = bias;
        return launch2(a, x_is_half ? (lut_mode() == 1 ? 2 : 1) : 0, true, q, static_cast<cudaStream_t>(stream));
    }
    Plan pl;
    rc = make_plan(a->bits, a->in_features, a->out_features, hyb ? a->topX : 0, a->rows != nullptr, true, pl);
    if (rc) return rc;
    if (!workspace || workspace_bytes < pl.ws_bytes)
        return fail(SQLLM_EWORKSPACE, "workspace too small: need %zu bytes, got %zu", pl.ws_bytes, workspace_bytes);
    Params p;
    memset(&p, 0, sizeof(p));
    p.ws_cnt = reinterpret_cast<int *>(ws + pl.ws_cnt_off);
    p.ws_hyb_cnt = reinterpret_cast<int *>(ws + pl.ws_hybcnt_off);
    p.ws_hyb = reinterpret_cast<float *>(ws + pl.ws_hyb_off);
    p.ws_part = reinterpret_cast<float *>(ws + pl.ws_part_off);
    p.ws_csr = reinterpret_cast<float *>(ws + pl.ws_csr_off);
    p.ws_acc = reinterpret_cast<float *>(ws + pl.ws_acc_off);
    p.det = det_mode();
    p.x = x; p.x_is_half = x_is_half; p.out = y; p.y_is_half = y_is_half; p.bias = bias;
    return launch<true>(a, pl, p, static_cast<cudaStream_t>(stream));
}

int sqllm_lutgemv_fused_exchange(const sqllm_lutgemv_args *a, const void *x, int x_is_half, int y_is_half, const float *bias,
                                 void *workspace, size_t workspace_bytes, const sqllm_exchange *xc, void *stream) {
    int rc = check_common(a);
    if (rc) return rc;
    if (!x || !xc) return fail(SQLLM_EINVAL, "x / exchange descriptor must not be null");
    if (reinterpret_cast<uintptr_t>(x) & 15) return fail(SQLLM_EINVAL, "x must be 16-byte aligned");
    if (reinterpret_cast<uintptr_t>(bias) & 15) return fail(SQLLM_EINVAL, "bias must be 16-byte aligned");
    if (det_mode() == 1) return fail(SQLLM_EINVAL, "the exchange path needs the default (non-deterministic) fused mode");
    if (xc->world < 1 || xc->world > 64 || xc->rank < 0 || xc->rank >= xc->world) return fail(SQLLM_EINVAL, "bad world / rank (%d / %d)", xc->world, xc->rank);
    if (xc->members < 1 || a->out_features % xc->members) return fail(SQLLM_EINVAL, "out_features=%d is not %d equal members", a->out_features, xc->members);
    const int w = a->out_features / xc->members;
    if (w % 4) return fail(SQLLM_EINVAL, "shard width %d must be a multiple of 4", w);
    if (xc->out_features_full < xc->world * w) return fail(SQLLM_EINVAL, "out_features_full=%d < world * shard width = %d", xc->out_features_full, xc->world * w);
    if (!xc->peer_base) return fail(SQLLM_EINVAL, "peer_base must not be null");
    if ((xc->out_offset & 15) || (xc->flag_offset & 7) || (xc->state_offset & 7) || (xc->error_offset & 3)) return fail(SQLLM_EINVAL, "misaligned arena offsets");
    if ((xc->out_features_full * (y_is_half ? 2 : 4)) % 16 || (w * (y_is_half ? 2 : 4)) % 8) return fail(SQLLM_EINVAL, "vector sizes must keep 8/16-byte store alignment");
    const bool hyb = a->full_rows && a->topX > 0;
    if (hyb && a->topX > MAX_TOPX_FUSED) return fail(SQLLM_EINVAL, "fused path supports topX <= %d", MAX_TOPX_FUSED);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    if (kernel_sel() == 2 && a->out_features >= STRIP) {
        if (!workspace || workspace_bytes < WS_HEADER) return fail(SQLLM_EWORKSPACE, "workspace too small: need %zu bytes, got %zu", (size_t)WS_HEADER, workspace_bytes);
        v2::P2 q;
        memset(&q, 0, sizeof(q));
        q.ws_cnt = reinterpret_cast<int *>(ws);
        q.ws_acc = reinterpret_cast<float *>(ws + WS_ACC_OFF);
        q.ws_hbox = reinterpret_cast<unsigned long long *>(ws + WS_HBOX_OFF);
        q.ws_cbox = reinterpret_cast<unsigned long long *>(ws + WS_CBOX_OFF);
        q.ws_dbox = reinterpret_cast<unsigned long long *>(ws + WS_DBOX_OFF);
        q.x = x; q.out = nullptr; q.y_is_half = y_is_half; q.bias = bias;
        q.xw_world = xc->world; q.xw_rank = xc->rank; q.xw_members = xc->members; q.xw_nfull = xc->out_features_full;
        q.xw_base = reinterpret_cast<const unsigned long long *>(xc->peer_base);
        q.xw_out_off = xc->out_offset; q.xw_flag_off = xc->flag_offset; q.xw_state_off = xc->state_offset; q.xw_err_off = xc->error_offset;
        return launch2(a, x_is_half ? (lut_mode() == 1 ? 2 : 1) : 0, true, q, static_cast<cudaStream_t>(stream));
    }
    Plan pl;
    rc = make_plan(a->bits, a->in_features, a->out_features, hyb ? a->topX : 0, a->rows != nullptr, true, pl);
    if (rc) return rc;
    if (!workspace || workspace_bytes < pl.ws_bytes)
        return fail(SQLLM_EWORKSPACE, "workspace too small: need %zu bytes, got %zu", pl.ws_bytes, workspace_bytes);
    Params p;
    memset(&p, 0, sizeof(p));
    p.ws_cnt = reinterpret_cast<int *>(ws + pl.ws_cnt_off);
    p.ws_hyb_cnt = reinterpret_cast<int *>(ws + pl.ws_hybcnt_off);
    p.ws_hyb = reinterpret_cast<float *>(ws + pl.ws_hyb_off);
    p.ws_part = reinterpret_cast<float *>(ws + pl.ws_part_off);
    p.ws_csr = reinterpret_cast<float *>(ws + pl.ws_csr_off);
    p.ws_acc = reinterpret_cast<float *>(ws + pl.ws_acc_off);
    p.det = 0;
    p.x = x; p.x_is_half = x_is_half; p.out = nullptr; p.y_is_half = y_is_half; p.bias = bias;
    p.xw_world = xc->world; p.xw_rank = xc->rank; p.xw_members = xc->members; p.xw_nfull = xc->out_features_full;
    p.xw_base = reinterpret_cast<const unsigned long long *>(xc->peer_base);
    p.xw_out_off = xc->out_offset; p.xw_flag_off = xc->flag_offset; p.xw_state_off = xc->state_offset; p.xw_err_off = xc->error_offset;
    return launch<true>(a, pl, p, static_cast<cudaStream_t>(stream));
}

int sqllm_unpack_indices(int bits, const int32_t *qweight, int in_features, int out_features, uint8_t *idx, void *stream) {
    if ((bits != 3 && bits != 4) || !qweight || !idx || in_features % 32 || in_features <= 0 || out_features <= 0)
        return fail(SQLLM_EINVAL, "bad arguments to sqllm_unpack_indices");
    unpack_kernel<<<1024, 256, 0, static_cast<cudaStream_t>(stream)>>>(bits, reinterpret_cast<const uint32_t *>(qweight),
                                                                       in_features, out_features, idx);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(SQLLM_ECUDA, "unpack launch failed: %s", cudaGetErrorString(e));
    return SQLLM_OK;
}

// ---- the reference's 12 launchers -----------------------------------------------------------------
static int run12(int bits, const float *vec, const int32_t *mat, float *mul, const float *lut, int height, int width,
                 int batch, int vec_height, const int32_t *rows, const int32_t *cols, const float *vals, int num_rows,
                 const float *full_rows, const int32_t *fri, int fr_height, int fr_width, void *stream) {
    sqllm_lutgemv_args a;
    memset(&a, 0, sizeof(a));
    a.bits = bits;
    if (height <= 0 || height % bits) return fail(SQLLM_EINVAL, "height=%d is not a multiple of bits=%d", height, bits);
    a.in_features = height / bits * 32;
    a.out_features = width;
    a.batch = batch;
    if (vec_height >= 0 && vec_height != a.in_features)
        return fail(SQLLM_EINVAL, "vec has %d features, packed matrix implies %d", vec_height, a.in_features);
    if (rows && num_rows != width) return fail(SQLLM_EINVAL, "num_rows=%d must equal the matrix width %d", num_rows, width);
    if (full_rows && fr_height != a.in_features)
        return fail(SQLLM_EINVAL, "full_rows has %d rows, expected in_features=%d", fr_height, a.in_features);
    a.qweight = mat; a.lookup_table = lut; a.vec = vec; a.mul = mul;
    a.rows = rows; a.cols = cols; a.vals = vals;
    a.full_rows = full_rows; a.full_row_indices = fri; a.topX = full_rows ? fr_width : 0;
    return sqllm_lutgemv(&a, stream);
}

int sqllm_vecquant3matmul_nuq_perchannel(const float *vec, const int32_t *mat, float *mul, const float *lut, int height,
                                         int width, void *stream) {
    return run12(3, vec, mat, mul, lut, height, width, 1, -1, 0, 0, 0, 0, 0, 0, 0, 0, stream);
}
int sqllm_vecquant4matmul_nuq_perchannel(const float *vec, const int32_t *mat, float *mul, const float *lut, int height,
                                         int width, void *stream) {
    return run12(4, vec, mat, mul, lut, height, width, 1, -1, 0, 0, 0, 0, 0, 0, 0, 0, stream);
}
int sqllm_vecquant3matmul_nuq_perchannel_batched(const float *vec, const int32_t *mat, float *mul, const float *lut,
                                                 int height, int width, int batch, int vec_height, void *stream) {
    return run12(3, vec, mat, mul, lut, height, width, batch, vec_height, 0, 0, 0, 0, 0, 0, 0, 0, stream);
}
int sqllm_vecquant4matmul_nuq_perchannel_batched(const float *vec, const int32_t *mat, float *mul, const float *lut,
                                                 int height, int width, int batch, int vec_height, void *stream) {
    return run12(4, vec, mat, mul, lut, height, width, batch, vec_height, 0, 0, 0, 0, 0, 0, 0, 0, stream);
}
int sqllm_vecquant3matmul_spmv_nuq_perchannel(const int32_t *rows, const int32_t *cols, const float *mat, const float *vec,
                                              float *mul, int num_rows, const int32_t *mat3, const float *lut, int height,
                                              int width, void *stream) {
    return run12(3, vec, mat3, mul, lut, height, width, 1, -1, rows, cols, mat, num_rows, 0, 0, 0, 0, stream);
}
int sqllm_vecquant4matmul_spmv_nuq_perchannel(const int32_t *rows, const int32_t *cols, const float *mat, const float *vec,
                                              float *mul, int num_rows, const int32_t *mat4, const float *lut, int height,
                                              int width, void *stream) {
    return run12(4, vec, mat4, mul, lut, height, width, 1, -1, rows, cols, mat, num_rows, 0, 0, 0, 0, stream);
}
int sqllm_vecquant3matmul_spmv_nuq_perchannel_batched(const int32_t *rows, const int32_t *cols, const float *mat,
                                                      const float *vec, float *mul, int num_rows, const int32_t *mat3,
                                                      const float *lut, int height, int width, int batch, int vec_height,
                                                      void *stream) {
    return run12(3, vec, mat3, mul, lut, height, width, batch, vec_height, rows, cols, mat, num_rows, 0, 0, 0, 0, stream);
}
int sqllm_vecquant4matmul_spmv_nuq_perchannel_batched(const int32_t *rows, const int32_t *cols, const float *mat,
                                                      const float *vec, float *mul, int num_rows, const int32_t *mat4,
                                                      const float *lut, int height, int width, int batch, int vec_height,
                                                      void *stream) {
    return run12(4, vec, mat4, mul, lut, height, width, batch, vec_height, rows, cols, mat, num_rows, 0, 0, 0, 0, stream);
}
int sqllm_vecquant3matmul_spmv_hybrid_nuq_perchannel(const int32_t *rows, const int32_t *cols, const float *mat,
                                                     const float *vec, const float *full_rows, const int32_t *fri,
                                                     float *mul, int num_rows, const int32_t *mat3, const float *lut,
                                                     int height, int width, int fr_height, int fr_width, void *stream) {
    return run12(3, vec, mat3, mul, lut, height, width, 1, -1, rows, cols, mat, num_rows, full_rows, fri, fr_height, fr_width, stream);
}
int sqllm_vecquant4matmul_spmv_hybrid_nuq_perchannel(const int32_t *rows, const int32_t *cols, const float *mat,
                                                     const float *vec, const float *full_rows, const int32_t *fri,
                                                     float *mul, int num_rows, const int32_t *mat4, const float *lut,
                                                     int height, int width, int fr_height, int fr_width, void *stream) {
    return run12(4, vec, mat4, mul, lut, height, width, 1, -1, rows, cols, mat, num_rows, full_rows, fri, fr_height, fr_width, stream);
}
int sqllm_vecquant3matmul_spmv_hybrid_nuq_perchannel_batched(const int32_t *rows, const int32_t *cols, const float *mat,
                                                             const float *vec, const float *full_rows, const int32_t *fri,
                                                             float *mul, int num_rows, const int32_t *mat3, const float *lut,
                                                             int height, int width, int fr_height, int fr_width, int batch,
                                                             int vec_height, void *stream) {
    return run12(3, vec, mat3, mul, lut, height, width, batch, vec_height, rows, cols, mat, num_rows, full_rows, fri, fr_height, fr_width, stream);
}
int sqllm_vecquant4matmul_spmv_hybrid_nuq_perchannel_batched(const int32_t *rows, const int32_t *cols, const float *mat,
                                                             const float *vec, const float *full_rows, const int32_t *fri,
                                                             float *mul, int num_rows, const int32_t *mat4, const float *lut,
                                                             int height, int width, int fr_height, int fr_width, int batch,
                                                             int vec_height, void *stream) {
    return run12(4, vec, mat4, mul, lut, height, width, batch, vec_height, rows, cols, mat, num_rows, full_rows, fri, fr_height, fr_width, stream);
}

}  // extern "C"
