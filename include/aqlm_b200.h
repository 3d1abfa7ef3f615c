/*
 * aqlm_b200 -- C-ABI of the B200-native (sm_100a) AQLM quantized-linear hot path.
 *
 * This header is the drop-in boundary (SURVEY.md §8b).  Every entry point takes plain device (or,
 * for *_host, pinned host) pointers, sizes and a CUstream/cudaStream_t passed as `void*`; no torch types.
 * Each function returns an aqlm_b200_status; on failure aqlm_b200_last_error() returns a message for
 * the calling thread.  Kernels never allocate or free: the caller owns every buffer, and nothing is
 * kept between calls (reference ownership model, cuda_kernel.cpp:159-163).  All launches go to the
 * stream given and are CUDA-graph capturable.
 *
 * Reference citations are relative to /root/reference/inference_lib/src/aqlm/inference_kernels/.
 *
 * Tensor layouts (identical to the reference module, inference.py:39-61):
 *   codes      [out_features, in_groups, num_codebooks]   int8 (nbits<=8) | int16 (nbits<=16), two's-complement
 *              storage of UNSIGNED codes (utils.py:23-31) -- kernels reinterpret, never sign-extend
 *   codebooks  [num_codebooks, 2^nbits, 1, in_group_size]  f16 | bf16
 *   scales     [out_features] (the module's [out,1,1,1])  f16 | bf16
 *   bias       [out_features] or NULL                      f16 | bf16
 *   input      [batch, in_features] row-major              f16 | bf16
 *   output     [batch, out_features] row-major             f16 | bf16 (or f32 partials, see flags)
 */
#ifndef AQLM_B200_H_
#define AQLM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AQLM_B200_VERSION 100 /* 0.1.0 */

typedef enum {
  AQLM_B200_OK = 0,
  AQLM_B200_ERR_DTYPE = 1,       /* not f16/bf16 -> NotImplementedError (cuda_kernel.cpp:9-25) */
  AQLM_B200_ERR_UNSUPPORTED = 2, /* scheme/group size not implemented -> NotImplementedError (cuda_kernel.cpp:137-144) */
  AQLM_B200_ERR_SHAPE = 3,       /* inconsistent sizes / misaligned pointers -> ValueError */
  AQLM_B200_ERR_CUDA = 4,        /* CUDA runtime error (the reference never checks; we do) -> RuntimeError */
  AQLM_B200_ERR_ARCH = 5         /* device is not sm_100 -> RuntimeError */
} aqlm_b200_status;

typedef enum { AQLM_B200_F16 = 0, AQLM_B200_BF16 = 1 } aqlm_b200_dtype;

/* flags for aqlm_b200_matmat_ex */
#define AQLM_B200_FLAG_PARTIAL_F32 1u /* write UNSCALED fp32 partial sums (no scale, no bias): the per-rank
                                          result of an in_features-sharded matvec, to be all-reduced */

/* One quantized weight matrix (all pointers are device pointers). */
typedef struct {
  const void* codes;
  const void* codebooks;
  const void* scales; /* may be NULL only with AQLM_B200_FLAG_PARTIAL_F32 */
  const void* bias;   /* NULL = no bias (Llama) */
  int64_t in_features;
  int64_t out_features;
  int32_t num_codebooks;
  int32_t nbits_per_codebook;
  int32_t in_group_size;  /* 8 or 16 */
  int32_t out_group_size; /* must be 1 (every reference CUDA kernel assumes it) */
  int32_t dtype;          /* aqlm_b200_dtype of codebooks/scales/bias/input/output */
  int32_t reserved;
} aqlm_b200_weight_t;

int aqlm_b200_version(void);
const char* aqlm_b200_last_error(void);
/* Number of kernels this library has launched in this process (bench.py's `gpu_launches`). */
uint64_t aqlm_b200_launch_count(void);
/* The AQLM_B200_* experiment switches (environment variables) are read once per process; tools that change the
 * environment at run time call this to re-read them.  Not needed in normal use. */
void aqlm_b200_reload_tunables(void);

/* ---- generic entry points -------------------------------------------------------------------- */

/* Fused code-gather + additive dequant + GEMV with the scale/bias epilogue in the same launch.
 * Replaces code1x16_matmat / code2x8_matmat / code1x8_matmat (cuda_kernel.cpp:148-182, 387-421,
 * 552-586: a host loop of one MatVec launch per batch row + 3-4 epilogue launches) and the Triton
 * path the reference uses for 8x8 (kernel_selector.py:91-94).  Any batch; intended for batch <= 6. */
int aqlm_b200_matmat(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, void* stream);
int aqlm_b200_matmat_ex(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, uint32_t flags,
                        void* stream);

/* Same with a caller-owned workspace (layout and zero-init contract as for aqlm_b200_matmat_dequant_ws below).  With a
 * workspace, batch-1 calls on 256-entry-codebook schemes (1x8, 2x8, 4x8, 8x8) use the dot-product-LUT kernel
 * (tensor-core-built LUT in shared memory, conflict-free 4-byte lookups) instead of per-code vector gathers. */
size_t aqlm_b200_matmat_workspace_bytes(const aqlm_b200_weight_t* w, int64_t batch);
int aqlm_b200_matmat_ws(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, uint32_t flags,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Grouped launch for several 1x16 linears that share the same input (q/k/v, gate/up): `w` describes the ROW-CONCATENATED
 * weights (codes [sum(seg_rows), in/8, 1], scales/bias [sum(seg_rows)]) and w->codebooks points to n_seg codebooks stacked
 * back to back (1 MiB each); output is [batch, sum(seg_rows)].  One launch instead of n_seg; batch <= 8.  New work (the
 * reference launches every linear separately); SURVEY §8f.2. */
int aqlm_b200_matmat_grouped(const aqlm_b200_weight_t* w, const int64_t* seg_rows, int n_seg, const void* input,
                             void* output, int64_t batch, uint32_t flags, void* stream);

/* Fused dequant + tensor-core GEMM for large batch: W never goes to HBM.  Replaces
 * code{1x16,2x8,1x8}_matmat_dequant (cuda_kernel.cpp:249-301, 450-484, 615-649: Dequant kernel ->
 * full W in HBM -> cuBLAS F::linear -> epilogue).  Tensor-core kernel for in_group_size 8 and for 1x16 with
 * in_group_size 16 (in_features % 128 == 0); other layouts run as passes of up to 8 rows through the fused GEMV. */
int aqlm_b200_matmat_dequant(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, void* stream);
/* Same with a caller-owned workspace, which lets the kernel split the K dimension across otherwise idle SMs
 * (the reduction is deterministic).  The first aqlm_b200_matmat_dequant_workspace_bytes() bytes... the whole
 * workspace must be ZERO before the first use and is left zero-initialised where it matters (tile counters),
 * so one persistent buffer per stream can be reused without memsets. */
size_t aqlm_b200_matmat_dequant_workspace_bytes(const aqlm_b200_weight_t* w, int64_t batch);
int aqlm_b200_matmat_dequant_ws(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch,
                                void* workspace, size_t workspace_bytes, void* stream);

/* Materialise W [out_features, in_features] (x scales when apply_scales != 0).  Replaces
 * code{1x16,2x8,1x8}_dequant (cuda_kernel.cpp:184-227, 423-448, 588-613). */
int aqlm_b200_dequant(const aqlm_b200_weight_t* w, void* weight_out, int apply_scales, void* stream);

/* Backward w.r.t. the input, fused: grad_input[batch, in] = (grad_output[batch, out] * scales) @ W_unscaled, with W
 * dequantized on chip (MN-major A tile, tcgen05 MMA, scale folded into the tile) -- W never goes to HBM and no library
 * GEMM is involved.  Replaces code*_matmat_dequant_transposed (cuda_kernel.cpp:303-354, 486-519, 651-684: Dequant
 * kernel -> full W in HBM -> cuBLAS), with the 2x8/1x8 unscaled-input defect (cuda_kernel.cpp:497,518,662,683) NOT
 * reproduced.  The optional workspace (same zero-init contract as aqlm_b200_matmat_dequant_ws) enables split-K over the
 * out rows.  Covers in_group_size 8 (8/16-bit codes, 1/2/4/8 codebooks) and in_group_size 16 for 1x16 with
 * in_features % 128 == 0; returns AQLM_B200_ERR_UNSUPPORTED for layouts the fused kernel does not cover (Kx8 or 2+
 * codebooks with in_group_size 16, code rows that are not a 16-byte multiple, out_features % 8 != 0, ...). */
size_t aqlm_b200_matmat_dequant_transposed_workspace_bytes(const aqlm_b200_weight_t* w, int64_t batch);
int aqlm_b200_matmat_dequant_transposed(const aqlm_b200_weight_t* w, const void* grad_output, void* grad_input,
                                        int64_t batch, void* workspace, size_t workspace_bytes, void* stream);

/* Epilogue of the sharded path: output[b,o] = (T)(partial[b,o] * scales[o] + bias[o]) after the
 * all-reduce of the fp32 partials (new work; the reference has no multi-GPU hot path, SURVEY §8e). */
int aqlm_b200_scale_bias(const float* partial, const void* scales, const void* bias, void* output, int64_t batch,
                         int64_t out_features, int32_t dtype, void* stream);

/* ---- multi-GPU: one-shot all-reduce over NVLink peer memory, fused with the epilogue ------------------------
 * One process per GPU.  Each rank allocates a shared buffer of aqlm_b200_comm_shared_bytes() with
 * aqlm_b200_shared_alloc (cudaMalloc + cudaIpcGetMemHandle; the 64-byte handle is exchanged out of band, e.g. with
 * torch.distributed.all_gather_object), opens every peer's handle with aqlm_b200_shared_open, and builds a communicator
 * from the W mapped pointers (peer_ptrs[rank] = its own buffer).  aqlm_b200_allreduce_scale_bias then does, in ONE
 * kernel: push my fp32 partials into every peer's buffer (P2P stores), publish a release flag, wait for all W flags,
 * add the W partials in rank order, apply scale + bias, write `output`.  Every rank must call it the same number of
 * times in the same order.  max_elems bounds batch*out_features of any call. */
typedef struct aqlm_b200_comm aqlm_b200_comm;
size_t aqlm_b200_comm_shared_bytes(int world, int64_t max_elems);
int aqlm_b200_shared_alloc(size_t bytes, void** ptr, void* handle64);
int aqlm_b200_shared_open(const void* handle64, void** ptr);
int aqlm_b200_comm_create(int rank, int world, void* const* peer_ptrs, int64_t max_elems, aqlm_b200_comm** out);
void* aqlm_b200_comm_partials(aqlm_b200_comm* comm); /* a device buffer of max_elems floats owned by the communicator */
int aqlm_b200_comm_destroy(aqlm_b200_comm* comm);
int aqlm_b200_allreduce_scale_bias(aqlm_b200_comm* comm, const float* partial, const void* scales, const void* bias,
                                   void* output, int64_t batch, int64_t out_features, int32_t dtype, void* stream);

/* The sharded linear as ONE kernel (1x16, in_group 8, batch <= 8): fused code-gather + dequant + GEMV on this rank's
 * in_features shard whose reduction epilogue performs the exchange over NVLink peer memory: every (row, batch) element
 * travels as one tagged 64-bit word {fp32 partial, step} stored into slot [step & 1][this rank] of EVERY rank's buffer
 * (8-byte P2P stores, coalesced per warp); the same thread then polls the W words of that element in its OWN buffer until
 * their tags equal the step, adds them in rank order (deterministic) and applies scale + bias -- no fence, flag or barrier
 * between push and reduction.  `w` describes the SHARD (in_features = local slice) with full-length scales/bias;
 * `seg_rows`/`n_seg` as in aqlm_b200_matmat_grouped (n_seg == 1: a plain linear, seg_rows may be NULL).  Every rank must
 * call it the same number of times in the same order (it shares the step counter with aqlm_b200_allreduce_scale_bias);
 * the grid is one CTA per SM so that all ranks' CTAs are resident while they wait for each other. */
int aqlm_b200_matmat_allreduce(aqlm_b200_comm* comm, const aqlm_b200_weight_t* w, const int64_t* seg_rows, int n_seg,
                               const void* input, void* output, int64_t batch, void* stream);

/* End-to-end variant with HOST buffers (pinned): H2D copy of `input_host` into `input_dev`, the fused
 * matmat, D2H copy of the result into `output_host`, and a stream synchronize.  `input_dev`/`output_dev`
 * are caller-owned device scratch of batch*in_features / batch*out_features elements. */
int aqlm_b200_matmat_host(const aqlm_b200_weight_t* w, const void* input_host, void* output_host, void* input_dev,
                          void* output_dev, int64_t batch, void* stream);

/* ---- flat wrappers named after the reference's pybind functions (cuda_kernel.cpp:686-699) ------
 * input [batch,in], codes, codebooks, scales, bias (nullable), output [batch,out]. */
int aqlm_b200_code1x16_matmat(const void* input, const void* codes, const void* codebooks, const void* scales,
                              const void* bias, void* output, int64_t batch, int64_t in_features,
                              int64_t out_features, int32_t in_group_size, int32_t dtype, void* stream);
int aqlm_b200_code2x8_matmat(const void* input, const void* codes, const void* codebooks, const void* scales,
                             const void* bias, void* output, int64_t batch, int64_t in_features,
                             int64_t out_features, int32_t dtype, void* stream);
int aqlm_b200_code1x8_matmat(const void* input, const void* codes, const void* codebooks, const void* scales,
                             const void* bias, void* output, int64_t batch, int64_t in_features,
                             int64_t out_features, int32_t dtype, void* stream);
int aqlm_b200_code1x16_matmat_dequant(const void* input, const void* codes, const void* codebooks,
                                      const void* scales, const void* bias, void* output, int64_t batch,
                                      int64_t in_features, int64_t out_features, int32_t in_group_size,
                                      int32_t dtype, void* stream);
int aqlm_b200_code2x8_matmat_dequant(const void* input, const void* codes, const void* codebooks,
                                     const void* scales, const void* bias, void* output, int64_t batch,
                                     int64_t in_features, int64_t out_features, int32_t dtype, void* stream);
int aqlm_b200_code1x8_matmat_dequant(const void* input, const void* codes, const void* codebooks,
                                     const void* scales, const void* bias, void* output, int64_t batch,
                                     int64_t in_features, int64_t out_features, int32_t dtype, void* stream);
int aqlm_b200_code1x16_dequant(const void* codes, const void* codebooks, const void* scales, void* weight_out,
                               int64_t in_features, int64_t out_features, int32_t in_group_size, int32_t dtype,
                               void* stream);
int aqlm_b200_code2x8_dequant(const void* codes, const void* codebooks, const void* scales, void* weight_out,
                              int64_t in_features, int64_t out_features, int32_t dtype, void* stream);
int aqlm_b200_code1x8_dequant(const void* codes, const void* codebooks, const void* scales, void* weight_out,
                              int64_t in_features, int64_t out_features, int32_t dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AQLM_B200_H_ */
