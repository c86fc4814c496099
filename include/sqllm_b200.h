/*
 * sqllm_b200.h - C ABI of the B200-native (sm_100a) dense-and-sparse LUT GEMV library
 *                (libsqllm_b200.so), a from-scratch replacement for the hot path of
 *                SqueezeAILab/SqueezeLLM:  squeezellm/quant_cuda_kernel.cu + quant_cuda.cpp.
 *
 * Boundary.  The reference exposes this path as a pybind11 C++ module `quant_cuda` whose 12
 * functions take torch::Tensor by value (squeezellm/quant_cuda.cpp:257-270) - there is no C ABI in
 * the reference.  This header is the C ABI that module sits on in our build: plain device
 * pointers, sizes and a stream; no torch types.  Each of the 12 entry points below replaces the
 * reference launcher named in its comment (same argument meaning, same accumulate-into-`mul`
 * contract); squeezellm_b200/csrc/quant_cuda_pybind.cpp is the thin torch::Tensor wrapper that
 * re-exports them under the reference's Python names.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the current CUDA device unless said otherwise;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - calls are asynchronous; nothing is retained after the call returns except `workspace`
 *     contents, which belong to the library between calls on the same stream;
 *   - return value: 0 on success, a negative SQLLM_E* code otherwise; sqllm_last_error() gives a
 *     thread-local human readable message.  (The reference performs no checks at all:
 *     squeezellm/quant_cuda_kernel.cu has no TORCH_CHECK / cudaGetLastError - SURVEY.md 8(b).)
 *   - shapes (reference: squeezellm/quant.py:48-95):
 *       vec           fp32 [batch, in]            (batch = 1 for the non-batched entry points)
 *       mat3 / mat4   int32 [in/32*bits, out]     packed indices, row-major
 *       lookup_table  fp32 [out, 2^bits]
 *       mul           fp32 [batch, out]           ACCUMULATED INTO (caller pre-fills zeros or bias)
 *       rows          int32 [out+1]   CSR row pointers, row = output channel
 *       cols          int32 [nnz]     input index of each non-zero
 *       vals          fp32  [nnz]
 *       full_rows     fp32 [in, topX] ; full_row_indices int32 [topX]  (output channel of column j)
 *     `height` = in/32*bits (rows of mat), `width` = out, as in the reference launchers.
 *   - requirements (checked, SQLLM_EINVAL otherwise): in % 64 == 0, out % 4 == 0, 16-byte aligned
 *     mat / vec, 1 <= batch.  The reference silently requires in % 128 == 0 and out % 128 == 0.
 */
#ifndef SQLLM_B200_H
#define SQLLM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SQLLM_OK 0
#define SQLLM_EINVAL (-1)   /* bad argument (shape, alignment, null pointer) */
#define SQLLM_ECUDA (-2)    /* a CUDA runtime call or launch failed */
#define SQLLM_EWORKSPACE (-3) /* workspace missing or too small */

#define SQLLM_ABI_VERSION 4   /* 2: + sqllm_lutgemv_fused_exchange, sqllm_set_deterministic ; 3: + sqllm_set_lut_mode, sqllm_workspace_error ; 4: + sqllm_sequence_* */

int sqllm_abi_version(void);
const char *sqllm_last_error(void);

/* Number of SMs x resident CTAs the persistent kernels will use on the current device
 * (informational; also used by bench.py to report the grid). */
int sqllm_device_sm_count(void);

/* ---------------------------------------------------------------------------------------------
 * Workspace.  Used only by the *_fused entry point (cross-CTA accumulator, counters, deterministic-mode partials).
 * Must be zero-filled once after allocation (cudaMemset); the library keeps it consistent afterwards.  One
 * workspace serves layers of any shape, but must not be used by two streams concurrently.  The size returned
 * does not depend on the summation mode.
 * ------------------------------------------------------------------------------------------- */
size_t sqllm_workspace_bytes(int bits, int in_features, int out_features, int topX);

/* ---------------------------------------------------------------------------------------------
 * Generic descriptor entry point (what all 12 wrappers below call).
 * ------------------------------------------------------------------------------------------- */
typedef struct sqllm_lutgemv_args {
    int bits;                 /* 3 or 4 */
    int in_features;          /* K */
    int out_features;         /* N */
    int batch;                /* rows of vec / mul */
    const int32_t *qweight;   /* [K/32*bits, N] */
    const float *lookup_table;/* [N, 2^bits] */
    const float *vec;         /* [batch, K] fp32 */
    float *mul;               /* [batch, N] fp32, accumulated into */
    /* optional CSR outliers (rows == NULL -> none) */
    const int32_t *rows;
    const int32_t *cols;
    const float *vals;
    /* optional dense rows (full_rows == NULL or topX == 0 -> none) */
    const float *full_rows;
    const int32_t *full_row_indices;
    int topX;
} sqllm_lutgemv_args;

int sqllm_lutgemv(const sqllm_lutgemv_args *args, void *stream);

/* Fused-path summation mode (process-wide).
 *   0 (default; env SQLLM_DETERMINISTIC unset): contributions are added with red.add.f32 into a workspace accumulator, like the
 *     reference's atomicAdd - results can differ in the last bits from run to run; the last CTAs of the grid convert it to y.
 *   1: per-strip partials reduced in a fixed order by the last-arriving contributor - bit-reproducible, 1.3-2x slower on
 *     layers with outliers. */
void sqllm_set_deterministic(int on);

/* Look-up-table precision of the fused path (process-wide; the 12 reference launchers below always use the exact table).
 *   SQLLM_LUT_EXACT (default): the per-channel codebook is used as stored, fp32 (squeezellm/quant_cuda_kernel.cu:779,866).
 *   SQLLM_LUT_FP16_PAIR      : north_star's "per-channel fp16 LUT" - centroids are rounded to fp16 (round-to-nearest-even) when a
 *     CTA builds its shared-memory table, which then holds PAIRS of centroids: one shared-memory read serves two weights and
 *     the products run as fp16 x fp16 -> fp32 FMAs (exact products, fp32 accumulation).  Only taken when x is fp16 (an fp32 x
 *     silently keeps the exact table); centroids must be finite in fp16 (|v| <= 65504).  Error against the exact result is that
 *     of the centroid rounding alone: <= 2^-11 relative per weight, ~2.5e-4 of max|y| on 4096-wide layers (tests/test_lut_fp16.py
 *     states and checks the bounds).  Environment: SQLLM_LUT_MODE=fp16.  Do not switch while other threads launch. */
#define SQLLM_LUT_EXACT 0
#define SQLLM_LUT_FP16_PAIR 1
void sqllm_set_lut_mode(int mode);
int sqllm_get_lut_mode(void);

/* Reads the workspace's error word (synchronises `stream`): 1 if a bounded in-kernel wait (2 s) ever gave up on this workspace -
 * the result of that call, and possibly later ones, is incomplete - else 0; negative on failure. */
int sqllm_workspace_error(const void *workspace, void *stream);

/* Fused module path behind QuantLinearLUT.forward (squeezellm/quant.py:211-312), batch-1 decode:
 *   y[c] = bias[c] + LUT-GEMV + CSR + dense rows, written (not accumulated) as fp16 or fp32,
 * from an fp16 or fp32 x, in ONE launch: replaces torch.zeros (quant.py:218), x.float() (:223,267),
 * the 1-3 reference launches and y.to(dtype) (:311).  Summation order: see sqllm_set_deterministic.
 * x_is_half / y_is_half select the element type of x / y.  bias may be NULL.  x, y and bias must be 16-byte aligned;
 * out_features <= SQLLM_MAX_N_FUSED and topX <= SQLLM_MAX_TOPX_FUSED on this path (and on the sequence and exchange paths);
 * sqllm_lutgemv has neither limit.  args->vec / args->mul / args->batch are ignored. */
#define SQLLM_MAX_TOPX_FUSED 128
#define SQLLM_MAX_N_FUSED 262144
int sqllm_lutgemv_fused(const sqllm_lutgemv_args *args,
                        const void *x, int x_is_half, void *y, int y_is_half, const float *bias,
                        void *workspace, size_t workspace_bytes, void *stream);

/* Fused forward of a COLUMN SHARD with the exchange built in (multi-GPU; the reference has none - north_star's
 * "column-shard each QuantLinear + all-reduce on the output vector", done by the kernel instead of a separate collective).
 * Every rank calls this with its shard (args->out_features = members * w columns: `members` sibling layers stacked, each
 * contributing this rank's w columns [rank*w, (rank+1)*w) of its out_features_full).  The CTAs that finish the GEMV store
 * their slice of y straight into EVERY rank's arena over NVLink peer memory - member m, column rank*w + j goes to element
 * [m][rank*w + j] of a [members][out_features_full] vector at out_offset - publish with a system-scope release on a
 * counter in each arena, and wait (bounded: 2 s, then *error_offset = 1) until all ranks' finishers have published on the
 * local one.  When the call's grid completes, the local vector is whole: the next stream-ordered consumer may read it.
 *   peer_base    device array [world] of the arenas' base addresses (e.g. torch symmetric memory's buffer_ptrs_dev)
 *   *_offset     byte offsets inside every arena: the destination vector, a u64 arrival counter (zero-initialised, only
 *                ever incremented), this rank's u64 expected-arrivals word (zero-initialised, local use), a u32 error word.
 * All ranks must issue the same sequence of exchange calls; consecutive calls must not target the same destination
 * (a fast rank may deliver call k+1 while a slow one still reads the result of call k).  Default summation mode only. */
typedef struct sqllm_exchange {
    int world, rank;
    int members;
    int out_features_full;
    const uint64_t *peer_base;
    size_t out_offset, flag_offset, state_offset, error_offset;
} sqllm_exchange;

int sqllm_lutgemv_fused_exchange(const sqllm_lutgemv_args *args,
                                 const void *x, int x_is_half, int y_is_half, const float *bias,
                                 void *workspace, size_t workspace_bytes, const sqllm_exchange *xchg, void *stream);

/* ---------------------------------------------------------------------------------------------
 * The reference's 12 launchers, one C entry point each.
 * ------------------------------------------------------------------------------------------- */
/* vecquant3matmul_nuq_perchannel_cuda  - squeezellm/quant_cuda_kernel.cu:132-154 */
int sqllm_vecquant3matmul_nuq_perchannel(const float *vec, const int32_t *mat, float *mul,
                                         const float *lookup_table, int height, int width, void *stream);
/* vecquant4matmul_nuq_perchannel_cuda  - squeezellm/quant_cuda_kernel.cu:157-179 */
int sqllm_vecquant4matmul_nuq_perchannel(const float *vec, const int32_t *mat, float *mul,
                                         const float *lookup_table, int height, int width, void *stream);
/* vecquant3matmul_nuq_perchannel_batched_cuda - :182-207 ; batch = vec.size(0), vec_height = vec.size(1) */
int sqllm_vecquant3matmul_nuq_perchannel_batched(const float *vec, const int32_t *mat, float *mul,
                                                 const float *lookup_table, int height, int width,
                                                 int batch, int vec_height, void *stream);
/* vecquant4matmul_nuq_perchannel_batched_cuda - :210-235 */
int sqllm_vecquant4matmul_nuq_perchannel_batched(const float *vec, const int32_t *mat, float *mul,
                                                 const float *lookup_table, int height, int width,
                                                 int batch, int vec_height, void *stream);
/* vecquant3matmul_spmv_nuq_perchannel_cuda - :238-282  (mat = CSR values, mat3 = packed weights) */
int sqllm_vecquant3matmul_spmv_nuq_perchannel(const int32_t *rows, const int32_t *cols, const float *mat,
                                              const float *vec, float *mul, int num_rows,
                                              const int32_t *mat3, const float *lookup_table,
                                              int height, int width, void *stream);
/* vecquant4matmul_spmv_nuq_perchannel_cuda - :285-327 */
int sqllm_vecquant4matmul_spmv_nuq_perchannel(const int32_t *rows, const int32_t *cols, const float *mat,
                                              const float *vec, float *mul, int num_rows,
                                              const int32_t *mat4, const float *lookup_table,
                                              int height, int width, void *stream);
/* vecquant3matmul_spmv_nuq_perchannel_batched_cuda - :331-381 */
int sqllm_vecquant3matmul_spmv_nuq_perchannel_batched(const int32_t *rows, const int32_t *cols, const float *mat,
                                                      const float *vec, float *mul, int num_rows,
                                                      const int32_t *mat3, const float *lookup_table,
                                                      int height, int width, int batch, int vec_height,
                                                      void *stream);
/* vecquant4matmul_spmv_nuq_perchannel_batched_cuda - :385-435 */
int sqllm_vecquant4matmul_spmv_nuq_perchannel_batched(const int32_t *rows, const int32_t *cols, const float *mat,
                                                      const float *vec, float *mul, int num_rows,
                                                      const int32_t *mat4, const float *lookup_table,
                                                      int height, int width, int batch, int vec_height,
                                                      void *stream);
/* vecquant3matmul_spmv_hybrid_nuq_perchannel_cuda - :439-507 ; full_rows is [fr_height=in, fr_width=topX] */
int sqllm_vecquant3matmul_spmv_hybrid_nuq_perchannel(const int32_t *rows, const int32_t *cols, const float *mat,
                                                     const float *vec, const float *full_rows,
                                                     const int32_t *full_row_indices, float *mul, int num_rows,
                                                     const int32_t *mat3, const float *lookup_table,
                                                     int height, int width, int fr_height, int fr_width,
                                                     void *stream);
/* vecquant4matmul_spmv_hybrid_nuq_perchannel_cuda - :511-577 */
int sqllm_vecquant4matmul_spmv_hybrid_nuq_perchannel(const int32_t *rows, const int32_t *cols, const float *mat,
                                                     const float *vec, const float *full_rows,
                                                     const int32_t *full_row_indices, float *mul, int num_rows,
                                                     const int32_t *mat4, const float *lookup_table,
                                                     int height, int width, int fr_height, int fr_width,
                                                     void *stream);
/* vecquant3matmul_spmv_hybrid_nuq_perchannel_batched_cuda - :580-657 */
int sqllm_vecquant3matmul_spmv_hybrid_nuq_perchannel_batched(const int32_t *rows, const int32_t *cols,
                                                             const float *mat, const float *vec,
                                                             const float *full_rows,
                                                             const int32_t *full_row_indices, float *mul,
                                                             int num_rows, const int32_t *mat3,
                                                             const float *lookup_table, int height, int width,
                                                             int fr_height, int fr_width, int batch,
                                                             int vec_height, void *stream);
/* vecquant4matmul_spmv_hybrid_nuq_perchannel_batched_cuda - :660-738 */
int sqllm_vecquant4matmul_spmv_hybrid_nuq_perchannel_batched(const int32_t *rows, const int32_t *cols,
                                                             const float *mat, const float *vec,
                                                             const float *full_rows,
                                                             const int32_t *full_row_indices, float *mul,
                                                             int num_rows, const int32_t *mat4,
                                                             const float *lookup_table, int height, int width,
                                                             int fr_height, int fr_width, int batch,
                                                             int vec_height, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Sequences: ONE persistent launch for a whole list of dependent matvecs.
 * Replaces the reference's per-layer launch loop during decode (squeezellm/llama.py:226-234 calls
 * QuantLinearLUT.forward once per layer; each forward is quant.py:212-312, i.e. 1-3 launches of
 * quant_cuda_kernel.cu:132-738).  Every item is one fused matvec (as sqllm_lutgemv_fused, fp16 in
 * and out); its input is either an external fp16 vector or a slice of an earlier item's output.
 * The kernel keeps the weight stream running across item boundaries and hands results from one
 * item to the next as self-validating tagged words in an arena (csrc/lutgemv_seq.cuh) - no
 * launch, no grid-wide barrier, no fence between two matvecs.  All items share `bits`.
 *
 * Several GPUs (column shards, one process per GPU): every rank creates the same sequence over
 * its own shards (items[i].a.out_features = members * shard width) and passes the peer-visible
 * arena of every rank; owners store their slice of each result into every rank's arena over
 * NVLink, the next item's input poll is the exchange.  All ranks must call sqllm_sequence_run the
 * same number of times.
 * ------------------------------------------------------------------------------------------- */
typedef struct sqllm_sequence sqllm_sequence;

typedef struct sqllm_seq_item {
    sqllm_lutgemv_args a;    /* the matrix: bits, in/out features, qweight, lookup_table, CSR, dense rows (vec/mul/batch ignored) */
    const float *bias;       /* optional, [out_features] */
    int x_from;              /* -1: x_ext ; i >= 0: the (full-length) output vector of item i < this item's index */
    int x_offset;            /* first element of that vector this item reads (multiple of 4); it reads in_features elements */
    const void *x_ext;       /* fp16 [in_features], read by every run (x_from == -1) */
    void *y;                 /* optional plain fp16 [out_features] copy of this item's own output columns */
    int members;             /* several GPUs: the item stacks `members` column shards of equal width (else 1) */
    int out_features_full;   /* several GPUs: full length of one member's output vector (else out_features) */
} sqllm_seq_item;

typedef struct sqllm_seq_options {
    int lut_mode;            /* SQLLM_LUT_EXACT / SQLLM_LUT_FP16_PAIR */
    int world, rank;         /* 1, 0 on a single GPU */
    void *arena;             /* world > 1: this rank's peer-visible arena (zero-filled once); NULL on one GPU: allocated here */
    size_t arena_bytes;
    const uint64_t *peer_base; /* world > 1: DEVICE array of `world` arena base addresses as seen from this rank */
    int n_export;            /* results wanted as plain fp16 vectors: item indices and destinations (full length) */
    const int *export_items;
    void *const *export_dst;
    uint64_t *trace;         /* debug builds (-DSQLLM_TRACE): [n_items][1024][32] time stamps, else NULL */
} sqllm_seq_options;

/* bytes of arena a sequence over these items needs (0 on error) */
size_t sqllm_sequence_arena_bytes(const sqllm_seq_item *items, int n_items);
int sqllm_sequence_create(const sqllm_seq_item *items, int n_items, const sqllm_seq_options *opt, sqllm_sequence **out);
/* two launches on `stream` (token counter, then the persistent kernel); CUDA-graph capturable */
int sqllm_sequence_run(sqllm_sequence *s, void *stream);
/* synchronises `stream`; 1 if a bounded in-kernel wait ever gave up (results incomplete), 0 if not, < 0 on error */
int sqllm_sequence_error(sqllm_sequence *s, void *stream);
/* clears the error word on `stream` (after a start-up skew between ranks has been dealt with: barrier, then reset on every rank) */
int sqllm_sequence_reset_error(sqllm_sequence *s, void *stream);
void sqllm_sequence_destroy(sqllm_sequence *s);

/* Test hook: unpack the packed indices on the GPU exactly as the GEMV kernels do
 * (idx uint8 [in, out]); lets tests prove the integer path bit-exact on its own. */
int sqllm_unpack_indices(int bits, const int32_t *qweight, int in_features, int out_features,
                         uint8_t *idx, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SQLLM_B200_H */
