// C-ABI of aqlm_b200 (see include/aqlm_b200.h): argument validation, kernel selection, launches.
// The host-side role of the reference's cuda_kernel.cpp (dtype check 9-25, group-size switch 113-146,
// launch heuristics cuda_kernel.cu:476-516) without torch types.
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "common.cuh"
#include "dequant.cuh"
#include "gemm_tcgen05.cuh"
#include "gemm_tcgen05_t.cuh"
#include "gemv.cuh"
#include "gemv_lut.cuh"
#include "peer_allreduce.cuh"

namespace aqlm_b200 {

std::atomic<uint64_t> g_launch_count{0};

const DeviceInfo* device_info() {
  static DeviceInfo infos[kMaxDevices];
  static std::mutex mu;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) {
    fail(AQLM_B200_ERR_CUDA, "cudaGetDevice failed (no CUDA device / driver?)");
    return nullptr;
  }
  DeviceInfo& d = infos[dev];
  if (!d.ok) {
    std::lock_guard<std::mutex> lock(mu);
    if (!d.ok) {
      cudaError_t e = cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev);
      if (e == cudaSuccess) e = cudaDeviceGetAttribute(&d.cc_major, cudaDevAttrComputeCapabilityMajor, dev);
      if (e == cudaSuccess) e = cudaDeviceGetAttribute(&d.cc_minor, cudaDevAttrComputeCapabilityMinor, dev);
      if (e == cudaSuccess) e = cudaDeviceGetAttribute(&d.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
      if (e != cudaSuccess) {
        fail(AQLM_B200_ERR_CUDA, "cudaDeviceGetAttribute failed: %s", cudaGetErrorString(e));
        return nullptr;
      }
      d.index = dev;
      d.ok = true;
    }
  }
  if (d.cc_major != 10) {
    fail(AQLM_B200_ERR_ARCH, "aqlm_b200 is built for sm_100a only; device %d is sm_%d%d", dev, d.cc_major, d.cc_minor);
    return nullptr;
  }
  return &d;
}

static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

// Experiment switches (environment variables), read ONCE per process -- not per launch -- and again only when a tool
// calls aqlm_b200_reload_tunables() after changing the environment.  Defaults are the shipped configuration.
struct Tunables {
  int pdl, gemv_ctas_per_sm, gemv_threads, gather_mode, gemv_v2, force_generic;
  int disable_lut, lut_ctas_per_sm, lut_debug, lut_cluster, lut_batch_loop, lut_rb16, lut_c2_rb;
  int disable_tcgen05, gemm_stages, gemm_ksplit, gemm_cluster, gemm_debug, gemm_gather_mode, gemm_v2, gemm_tile_m, gemm_atmem, gemm_a_stages, gemm_groups;
  void load() {
    pdl = env_int("AQLM_B200_PDL", 1);
    gemv_ctas_per_sm = env_int("AQLM_B200_GEMV_CTAS_PER_SM", 1);
    gemv_threads = env_int("AQLM_B200_GEMV_THREADS", kGemv1x16Threads);
    gather_mode = env_int("AQLM_B200_GATHER_MODE", 0);
    gemv_v2 = env_int("AQLM_B200_GEMV_V2", 1);
    force_generic = env_int("AQLM_B200_FORCE_GENERIC", 0);
    disable_lut = env_int("AQLM_B200_DISABLE_LUT", 0);
    lut_ctas_per_sm = env_int("AQLM_B200_LUT_CTAS_PER_SM", 2);  // 128 regs x 256 threads: registers allow 2
    lut_debug = env_int("AQLM_B200_LUT_DEBUG", 0);
    lut_batch_loop = env_int("AQLM_B200_LUT_BATCH_LOOP", 1);  // batch 2-3 on 256-entry codebooks: one LUT launch per row
    lut_rb16 = env_int("AQLM_B200_LUT_RB16", 0);  // cluster kernel: 16-row warp batches on 768 threads (experiment)
    lut_c2_rb = env_int("AQLM_B200_LUT_C2_RB", 0);  // cluster kernel, second form: rows per warp batch (0: by row-block size; 16; 32)
    // K <= 2, in <= 4096: slab CTAs form a cluster, DSMEM reduction.  0: off (workspace kernel), 1: first form, 2: second form,
    // 3 (default): second form for row blocks of <= 768 rows = at most 24 warps of 32 rows, the 768-thread / 80-register
    // build (Llama-2-7B: 4096 -> 4096 / 11008; 15 clusters of 8 CTAs were resident on the measured boxes, i.e. blocks of
    // 288 and 736 rows), first form above, where the second form needs its 1024-thread / 64-register build and spills
    // (measured, profiles/r02/probe_lut2_n.jsonl: second form +12..+27 % up to 11008 rows, -2..-4 % at 12288 / 22016
    // rows = blocks of 832 / 1472 rows)
    lut_cluster = env_int("AQLM_B200_LUT_CLUSTER", 3);
    disable_tcgen05 = env_int("AQLM_B200_DISABLE_TCGEN05", 0);
    gemm_stages = env_int("AQLM_B200_GEMM_STAGES", 0);
    gemm_ksplit = env_int("AQLM_B200_GEMM_KSPLIT", 0);
    gemm_cluster = env_int("AQLM_B200_GEMM_CLUSTER", 0);  // 0: per plan (pairs of CTAs multicast the X tile: 52.7 vs 55.1 us at 4096->14336 bs=256; 4 is slower)
    gemm_debug = env_int("AQLM_B200_GEMM_DEBUG", 0);
    gemm_gather_mode = env_int("AQLM_B200_GEMM_GATHER_MODE", -1);  // -1: per scheme (1x16: ld.global.cg, no L1 allocation of the 1 MiB codebook's lines; 256-entry codebooks: L1-resident)
    gemm_v2 = env_int("AQLM_B200_GEMM_V2", -1);                   // -1: per-scheme default
    gemm_tile_m = env_int("AQLM_B200_GEMM_TILE_M", 0);            // 0: chosen by the plan
    gemm_a_stages = env_int("AQLM_B200_GEMM_A_STAGES", 0);        // ATMEM: A stages in tensor memory (0: 6)
    gemm_groups = env_int("AQLM_B200_GEMM_GROUPS", 0);            // ATMEM: producer groups of 4 warps (0: 3, max 4)
    gemm_atmem = env_int("AQLM_B200_GEMM_ATMEM", -1);             // A operand in tensor memory; -1: per-scheme default
  }
};
static Tunables& tun() {
  static Tunables t = [] { Tunables x; x.load(); return x; }();
  return t;
}

static int validate(const aqlm_b200_weight_t* w, bool need_scales) {
  if (!w) return fail(AQLM_B200_ERR_SHAPE, "weight descriptor is NULL");
  if (w->dtype != AQLM_B200_F16 && w->dtype != AQLM_B200_BF16)
    return fail(AQLM_B200_ERR_DTYPE,
                "AQLM CUDA kernels only support float16 and bfloat16. Please specify the correct `torch_dtype` "
                "when loading the model.");
  if (w->out_group_size != 1)
    return fail(AQLM_B200_ERR_UNSUPPORTED, "aqlm_b200 kernels require out_group_size == 1, got %d", w->out_group_size);
  if (w->in_group_size != 8 && w->in_group_size != 16)
    return fail(AQLM_B200_ERR_UNSUPPORTED, "AQLM CUDA kernels only support codebooks with 8 or 16 features. Got %d.",
                w->in_group_size);
  if (w->nbits_per_codebook < 1 || w->nbits_per_codebook > 16)
    return fail(AQLM_B200_ERR_UNSUPPORTED, "nbits_per_codebook must be in [1,16], got %d", w->nbits_per_codebook);
  if (w->num_codebooks < 1 || w->num_codebooks > 16)
    return fail(AQLM_B200_ERR_UNSUPPORTED, "num_codebooks must be in [1,16], got %d", w->num_codebooks);
  if (w->in_features <= 0 || w->out_features <= 0 || w->in_features % w->in_group_size != 0)
    return fail(AQLM_B200_ERR_SHAPE, "bad shape: in_features=%lld out_features=%lld in_group_size=%d",
                (long long)w->in_features, (long long)w->out_features, w->in_group_size);
  if (w->in_features > (1ll << 30) || w->out_features > (1ll << 30))
    return fail(AQLM_B200_ERR_SHAPE, "dimension too large");
  if (!w->codes || !w->codebooks) return fail(AQLM_B200_ERR_SHAPE, "codes/codebooks pointer is NULL");
  if (need_scales && !w->scales) return fail(AQLM_B200_ERR_SHAPE, "scales pointer is NULL");
  if ((reinterpret_cast<uintptr_t>(w->codebooks) & 15) != 0)
    return fail(AQLM_B200_ERR_SHAPE, "codebooks must be 16-byte aligned");
  return AQLM_B200_OK;
}

// Opt-in dynamic shared memory.  cudaFuncSetAttribute applies to the CURRENT device only, so the high-water mark is
// kept per (kernel instantiation, device): a process that drives several GPUs configures each of them.
struct SmemMarks {
  std::atomic<size_t> v[kMaxDevices];
};
template <typename KernelT>
static int ensure_smem(KernelT kernel, size_t smem, SmemMarks& marks, const DeviceInfo* di) {
  std::atomic<size_t>& m = marks.v[di->index];
  if (smem > 48 * 1024 && m.load(std::memory_order_relaxed) < smem) {
    AQLM_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    m.store(smem, std::memory_order_relaxed);
  }
  return AQLM_B200_OK;
}

// smem bytes of the vector GEMV: x tile + staged codebooks + per-(row,slice) partials
static size_t vec_smem_bytes(const GemvParams& p, int K, int code_bytes, int G, int BT, bool cbs, int grid) {
  const int gpc = 16 / (K * code_bytes);
  const int chunks = p.in_groups / gpc;
  const int slices = (chunks + kSliceChunks - 1) / kSliceChunks;
  const int rows_cta = (p.out_features + grid - 1) / grid;
  return (size_t)BT * p.in_features * 2 + (cbs ? ((size_t)K << p.nbits) * G * 2 : 0) +
         (size_t)rows_cta * slices * BT * 4;
}

template <typename T, int K, int CB, int G, int BT, bool CBS, int GM>
static int launch_vec(const GemvParams& p, const DeviceInfo* di, cudaStream_t st) {
  constexpr int THREADS = (BT <= 2) ? 1024 : 512;
  const int grid = di->sm_count * tun().gemv_ctas_per_sm;
  const size_t smem = vec_smem_bytes(p, K, CB, G, BT, CBS, grid);
  auto kernel = gemv_vec_kernel<T, K, CB, G, BT, CBS, GM, THREADS>;
  static SmemMarks marks;
  if (int rc = ensure_smem(kernel, smem, marks, di)) return rc;
  // PDL launch: this kernel's weight-only prologue may overlap the previous kernel's tail (see gemv.cuh).
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = tun().pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, p));
  count_launch();
  return AQLM_B200_OK;
}

template <typename T, int BT, int GM, int THREADS>
static int launch_1x16_t(const GemvParams& p, const DeviceInfo* di, cudaStream_t st) {
  const int grid = di->sm_count * (512 / THREADS);
  const size_t smem = vec_smem_bytes(p, 1, 2, 8, BT, false, grid);
  auto kernel = gemv_1x16_kernel<T, BT, GM, THREADS>;
  static SmemMarks marks;
  if (int rc = ensure_smem(kernel, smem, marks, di)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = tun().pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, p, GemvPeer{}));
  count_launch();
  return AQLM_B200_OK;
}

// Fused GEMV + peer-memory exchange (gemv_1x16_kernel<..., PEER = true>): contiguous row blocks, one CTA per SM.
template <typename T, int BT>
static int launch_1x16_peer(GemvParams p, const GemvPeer& pc, const DeviceInfo* di, cudaStream_t st) {
  const int grid = di->sm_count;
  if (grid > kPeerFlagStride) return fail(AQLM_B200_ERR_UNSUPPORTED, "fused exchange: more SMs than flag slots");
  int rb = (p.out_features + grid - 1) / grid;
  rb = (rb + 3) & ~3;
  p.row_block = rb;
  const int chunks = p.in_groups / 8;
  const int slices = (chunks + kSliceChunks - 1) / kSliceChunks;
  const size_t smem = (size_t)BT * p.in_features * 2 + (size_t)rb * slices * BT * 4;
  if (smem > (size_t)di->max_smem_optin - 1024)
    return fail(AQLM_B200_ERR_UNSUPPORTED, "fused exchange: activation tile + partials do not fit in shared memory");
  auto kernel = gemv_1x16_kernel<T, BT, 0, kGemv1x16Threads, true>;
  static SmemMarks marks;
  if (int rc = ensure_smem(kernel, smem, marks, di)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kGemv1x16Threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = tun().pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, p, pc));
  count_launch();
  return AQLM_B200_OK;
}

// 512-thread CTAs, one per SM (default), or 256-thread CTAs, two per SM (AQLM_B200_GEMV_THREADS=256; batch 1 only)
template <typename T, int BT, int GM>
static int launch_1x16(const GemvParams& p, const DeviceInfo* di, cudaStream_t st) {
  if constexpr (BT == 1 && GM == 0) {
    if (tun().gemv_threads == 256) return launch_1x16_t<T, BT, GM, 256>(p, di, st);
  }
  return launch_1x16_t<T, BT, GM, kGemv1x16Threads>(p, di, st);
}

template <typename T, int CB, int G, int BT>
static int launch_generic(const GemvParams& p, const DeviceInfo* di, cudaStream_t st) {
  int blocks = (p.out_features + 7) / 8;
  if (blocks > di->sm_count * 8) blocks = di->sm_count * 8;
  gemv_generic_kernel<T, CB, G, BT><<<blocks, kGemvThreads, 0, st>>>(p);
  count_launch();
  AQLM_CUDA_CHECK(cudaGetLastError());
  return AQLM_B200_OK;
}

template <typename T, int BT>
static int dispatch_bt(const aqlm_b200_weight_t* w, const GemvParams& p, const DeviceInfo* di, cudaStream_t st) {
  const int K = w->num_codebooks, nbits = w->nbits_per_codebook, G = w->in_group_size;
  const int code_bytes = nbits <= 8 ? 1 : 2;
  const size_t row_bytes = (size_t)p.in_groups * K * code_bytes;
  const bool vec_ok = (row_bytes % 16 == 0) && ((reinterpret_cast<uintptr_t>(w->codes) & 15) == 0) &&
                      ((reinterpret_cast<uintptr_t>(p.x) & 15) == 0) && !tun().force_generic;
  const size_t budget = (size_t)di->max_smem_optin - 1024;
  const int grid = di->sm_count * tun().gemv_ctas_per_sm;
  const bool pow2k = (K == 1 || K == 2 || K == 4 || K == 8);
  const size_t need = pow2k ? vec_smem_bytes(p, K, code_bytes, G, BT, nbits == 8, grid) : (size_t)-1;
  if (vec_ok && nbits == 16 && K == 1 && need <= budget) {
    const int gm = tun().gather_mode;
    if (G == 8 && tun().gemv_v2 && vec_smem_bytes(p, 1, 2, 8, BT, false, di->sm_count) <= budget) {
      if (gm == 1) return launch_1x16<T, BT, 1>(p, di, st);
      return launch_1x16<T, BT, 0>(p, di, st);
    }
    if (G == 8) {
      if (gm == 1) return launch_vec<T, 1, 2, 8, BT, false, 1>(p, di, st);
      if (gm == 2) return launch_vec<T, 1, 2, 8, BT, false, 2>(p, di, st);
      return launch_vec<T, 1, 2, 8, BT, false, 0>(p, di, st);
    }
    // g = 16: one codebook entry is fetched as ONE 256-bit request, which needs a 32-byte aligned table (any torch
    // allocation is); a 16-byte aligned table handed in through the C-ABI takes the generic kernel below
    if ((reinterpret_cast<uintptr_t>(w->codebooks) & 31) == 0) return launch_vec<T, 1, 2, 16, BT, false, 0>(p, di, st);
  }
  if (vec_ok && nbits == 8 && G == 8 && pow2k && need <= budget) {
    if (K == 1) return launch_vec<T, 1, 1, 8, BT, true, 0>(p, di, st);
    if (K == 2) return launch_vec<T, 2, 1, 8, BT, true, 0>(p, di, st);
    if (K == 4) return launch_vec<T, 4, 1, 8, BT, true, 0>(p, di, st);
    if (K == 8) return launch_vec<T, 8, 1, 8, BT, true, 0>(p, di, st);
  }
  if (code_bytes == 2) {
    if (G == 8) return launch_generic<T, 2, 8, BT>(p, di, st);
    return launch_generic<T, 2, 16, BT>(p, di, st);
  }
  if (G == 8) return launch_generic<T, 1, 8, BT>(p, di, st);
  return launch_generic<T, 1, 16, BT>(p, di, st);
}

template <typename T>
static int matmat_typed(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, uint32_t flags,
                        const DeviceInfo* di, cudaStream_t st) {
  const bool partial = (flags & AQLM_B200_FLAG_PARTIAL_F32) != 0;
  GemvParams p;
  p.codes = w->codes;
  p.codebooks = w->codebooks;
  p.scales = w->scales;
  p.bias = w->bias;
  p.out_features = (int)w->out_features;
  p.in_features = (int)w->in_features;
  p.in_groups = (int)(w->in_features / w->in_group_size);
  p.nbits = w->nbits_per_codebook;
  p.num_codebooks = w->num_codebooks;
  p.partial_f32 = partial ? 1 : 0;
  p.n_seg = 1;
  p.row_block = 0;
  p.seg_end[0] = p.seg_end[1] = p.seg_end[2] = p.seg_end[3] = p.out_features;
  const size_t out_elt = partial ? 4 : 2;
  // largest pass size whose x tile fits in shared memory
  int max_bt = 8;
  while (max_bt > 1 && (size_t)max_bt * w->in_features * 2 + 40 * 1024 > (size_t)di->max_smem_optin) max_bt >>= 1;
  for (int64_t b0 = 0; b0 < batch; b0 += max_bt) {
    const int nb = (int)((batch - b0) < max_bt ? (batch - b0) : max_bt);
    p.batch = nb;
    p.x = reinterpret_cast<const uint8_t*>(input) + (size_t)b0 * w->in_features * 2;
    p.y = reinterpret_cast<uint8_t*>(output) + (size_t)b0 * w->out_features * out_elt;
    int rc;
    if (nb == 1) rc = dispatch_bt<T, 1>(w, p, di, st);
    else if (nb == 2) rc = dispatch_bt<T, 2>(w, p, di, st);
    else if (nb <= 4) rc = dispatch_bt<T, 4>(w, p, di, st);
    else rc = dispatch_bt<T, 8>(w, p, di, st);
    if (rc) return rc;
  }
  return AQLM_B200_OK;
}

template <typename T>
static int dequant_typed(const aqlm_b200_weight_t* w, void* out, int apply_scales, cudaStream_t st) {
  const int in_groups = (int)(w->in_features / w->in_group_size);
  const int64_t n = w->out_features * in_groups;
  const int threads = 256;
  const int64_t blocks = (n + threads - 1) / threads;
  if (blocks > 0x7fffffffll) return fail(AQLM_B200_ERR_SHAPE, "weight too large for one dequant launch");
  const T* sc = apply_scales ? reinterpret_cast<const T*>(w->scales) : nullptr;
  const int cb = w->nbits_per_codebook <= 8 ? 1 : 2;
#define AQLM_DQ(CB, G)                                                                                        \
  dequant_kernel<T, CB, G><<<(unsigned)blocks, threads, 0, st>>>(w->codes, w->codebooks, sc, out,            \
                                                                   w->out_features, in_groups, w->num_codebooks, \
                                                                   w->nbits_per_codebook)
  if (cb == 2 && w->in_group_size == 8) AQLM_DQ(2, 8);
  else if (cb == 2) AQLM_DQ(2, 16);
  else if (w->in_group_size == 8) AQLM_DQ(1, 8);
  else AQLM_DQ(1, 16);
#undef AQLM_DQ
  count_launch();
  AQLM_CUDA_CHECK(cudaGetLastError());
  return AQLM_B200_OK;
}

// ---- Kx8 LUT GEMV: host side ------------------------------------------------------------------------
struct LutPlan {
  bool ok = false;
  int J = 32, n_slabs = 0, row_blocks = 0, rows_per_block = 0;
  size_t smem = 0, partials_bytes = 0;
};
constexpr size_t kWsCountersBytes = 65536;  // fixed counter region at the head of every workspace (16384 words)
constexpr int kGemmMaxTiles = 8192;  // split-K / LUT tickets use counter words [0, 8192); the LUT GEMV's generation words follow

static LutPlan lut_plan(const aqlm_b200_weight_t* w, int64_t batch, const DeviceInfo* di) {
  LutPlan L;
  const int K = w->num_codebooks;
  if (batch != 1 || w->nbits_per_codebook != 8 || w->in_group_size != 8) return L;
  if (!(K == 1 || K == 2 || K == 4 || K == 8)) return L;
  if (tun().disable_lut) return L;
  if ((reinterpret_cast<uintptr_t>(w->codes) & 7) != 0) return L;
  L.J = (K == 8) ? 16 : 32;
  const int in_groups = (int)(w->in_features / 8);
  L.n_slabs = (in_groups + L.J - 1) / L.J;
  L.smem = (size_t)K * 256 * L.J * 4 + 16;  // LUT + the "last CTA" flag word
  if (L.smem + 1024 > (size_t)di->max_smem_optin) return L;
  int per_sm = (int)((size_t)di->max_smem_optin / (L.smem + 1024));
  const int want = tun().lut_ctas_per_sm;
  if (per_sm > want) per_sm = want;
  if (per_sm < 1) per_sm = 1;
  // the whole grid must be resident at once (ONE wave): a few CTAs spilling into a second wave double the time
  int rb = (di->sm_count * per_sm) / L.n_slabs;
  if (rb < 1) rb = 1;
  int rpb = (int)((w->out_features + rb - 1) / rb);
  rpb = (rpb + 31) / 32 * 32;
  L.rows_per_block = rpb;
  L.row_blocks = (int)((w->out_features + rpb - 1) / rpb);
  if ((size_t)L.row_blocks > (size_t)kGemmMaxTiles) return L;  // tickets in words [0, 8192), generation words above
  L.partials_bytes = (size_t)L.n_slabs * w->out_features * 4;
  L.ok = true;
  return L;
}

template <typename T, int K, int J>
static int launch_lut(const aqlm_b200_weight_t* w, const void* input, void* output, uint32_t flags, const LutPlan& L,
                      void* workspace, cudaStream_t st) {
  const DeviceInfo* di = device_info();
  if (!di) return AQLM_B200_ERR_CUDA;
  LutParams p;
  p.codes = w->codes;
  p.codebooks = w->codebooks;
  p.scales = w->scales;
  p.bias = w->bias;
  p.x = input;
  p.y = output;
  p.ws_counters = reinterpret_cast<unsigned int*>(workspace);
  p.ws_gen = p.ws_counters + kGemmMaxTiles;  // generation words live in the upper half of the counter region
  p.ws_partials = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + kWsCountersBytes);
  p.out_features = (int)w->out_features;
  p.in_groups = (int)(w->in_features / 8);
  p.n_slabs = L.n_slabs;
  p.rows_per_block = L.rows_per_block;
  p.partial_f32 = (flags & AQLM_B200_FLAG_PARTIAL_F32) ? 1 : 0;
  p.debug = tun().lut_debug;
  constexpr int THREADS = (K <= 2) ? 256 : 512;  // K >= 4: one CTA per SM (128 KiB LUT), so give it 16 warps
  auto kernel = gemv_lut_kernel<T, K, J, THREADS>;
  static SmemMarks marks;
  if (int rc = ensure_smem(kernel, L.smem, marks, di)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(L.n_slabs, L.row_blocks);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = L.smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = tun().pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, p));
  count_launch();
  return AQLM_B200_OK;
}

template <typename T>
static int lut_typed(const aqlm_b200_weight_t* w, const void* input, void* output, uint32_t flags, const LutPlan& L,
                     void* workspace, cudaStream_t st) {
  switch (w->num_codebooks) {
    case 1: return launch_lut<T, 1, 32>(w, input, output, flags, L, workspace, st);
    case 2: return launch_lut<T, 2, 32>(w, input, output, flags, L, workspace, st);
    case 4: return launch_lut<T, 4, 32>(w, input, output, flags, L, workspace, st);
    default: return launch_lut<T, 8, 16>(w, input, output, flags, L, workspace, st);
  }
}

// Second form of the cluster kernel (gemv_lut_cluster2_kernel): LUT at absolute shared address 0x10000, one warp per
// row batch (the CTA size follows the row block), push-based cross-slab sum.
template <typename T, int K, int RB, int MAXT = 1024>
static int launch_lut_cluster2(const aqlm_b200_weight_t* w, const void* input, void* output, uint32_t flags,
                               const DeviceInfo* di, cudaStream_t st, int rpb, int row_blocks, int n_slabs) {
  int warps = (rpb + RB - 1) / RB;
  warps = warps < 8 ? 8 : (warps > 32 ? 32 : warps);
  if (MAXT == 1024 && warps <= 24)  // <= 768 threads: the 80-register build (the 64-register one spills ~50 words at RB = 32)
    return launch_lut_cluster2<T, K, RB, 768>(w, input, output, flags, di, st, rpb, row_blocks, n_slabs);
  auto kernel = gemv_lut_cluster2_kernel<T, K, RB, MAXT>;
  const size_t smem = (size_t)kLutAbs + (size_t)K * 256 * kLutCJ * 4;  // LUT ends at 0x10000 * (1 + K) whatever the window base
  static SmemMarks marks;
  if (int rc = ensure_smem(kernel, smem, marks, di)) return rc;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = n_slabs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = tun().pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  cfg.blockDim = dim3(warps * 32);
  cfg.gridDim = dim3(n_slabs, row_blocks);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  LutClusterParams p;
  p.codes = w->codes;
  p.codebooks = w->codebooks;
  p.scales = w->scales;
  p.bias = w->bias;
  p.x = input;
  p.y = output;
  p.out_features = (int)w->out_features;
  p.in_groups = (int)(w->in_features / 8);
  p.n_slabs = n_slabs;
  p.rows_per_block = rpb;
  p.partial_f32 = (flags & AQLM_B200_FLAG_PARTIAL_F32) ? 1 : 0;
  AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, p));
  count_launch();
  return AQLM_B200_OK;
}

// ---- Kx8 LUT GEMV, cluster / DSMEM variant (K <= 2, at most 8 slabs of 64 groups): host side ---------------
template <typename T, int K, int RB, int THREADS>
static int launch_lut_cluster(const aqlm_b200_weight_t* w, const void* input, void* output, uint32_t flags,
                              const DeviceInfo* di, cudaStream_t st, bool* taken) {
  *taken = false;
  const int in_groups = (int)(w->in_features / 8);
  const int n_slabs = (in_groups + kLutCJ - 1) / kLutCJ;
  auto kernel = gemv_lut_cluster_kernel<T, K, RB, THREADS>;
  const size_t lut_bytes = (size_t)K * 256 * kLutCJ * 4;
  // how many clusters of n_slabs CTAs can be resident at once: the grid must be ONE wave (a second wave doubles the time)
  static std::atomic<int> max_clusters[kMaxDevices][9];
  int mc = max_clusters[di->index][n_slabs].load(std::memory_order_relaxed);
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = n_slabs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = tun().pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.blockDim = dim3(THREADS);
  cfg.stream = st;
  static SmemMarks marks;
  if (mc == 0) {
    const size_t smem_max = lut_bytes + 8192;
    if (int rc = ensure_smem(kernel, smem_max, marks, di)) return rc;
    cfg.gridDim = dim3(n_slabs, di->sm_count);
    cfg.dynamicSmemBytes = smem_max;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess || n < 1) {
      (void)cudaGetLastError();
      n = -1;  // not launchable as a cluster here: use the workspace kernel
    }
    mc = n;
    max_clusters[di->index][n_slabs].store(mc, std::memory_order_relaxed);
  }
  if (mc < 1) return AQLM_B200_OK;
  int rpb = (int)((w->out_features + mc - 1) / mc);
  rpb = (rpb + 31) / 32 * 32;
  if (rpb > 2048) return AQLM_B200_OK;  // per-row partials live in shared memory
  const int row_blocks = (int)((w->out_features + rpb - 1) / rpb);
  if (tun().lut_cluster == 2 || (tun().lut_cluster >= 3 && rpb <= 768)) {  // second form: same grid / cluster shape, its own CTA size and shared-memory map
    const int rb_sel = tun().lut_c2_rb ? tun().lut_c2_rb : (rpb <= 512 ? 16 : 32);
    const int rc = rb_sel == 16 ? launch_lut_cluster2<T, K, 16>(w, input, output, flags, di, st, rpb, row_blocks, n_slabs)
                                : launch_lut_cluster2<T, K, 32>(w, input, output, flags, di, st, rpb, row_blocks, n_slabs);
    *taken = rc == AQLM_B200_OK;
    return rc;
  }
  const size_t smem = lut_bytes + (size_t)rpb * 4;
  if (int rc = ensure_smem(kernel, smem, marks, di)) return rc;
  LutClusterParams p;
  p.codes = w->codes;
  p.codebooks = w->codebooks;
  p.scales = w->scales;
  p.bias = w->bias;
  p.x = input;
  p.y = output;
  p.out_features = (int)w->out_features;
  p.in_groups = in_groups;
  p.n_slabs = n_slabs;
  p.rows_per_block = rpb;
  p.partial_f32 = (flags & AQLM_B200_FLAG_PARTIAL_F32) ? 1 : 0;
  cfg.gridDim = dim3(n_slabs, row_blocks);
  cfg.dynamicSmemBytes = smem;
  cfg.numAttrs = 2;
  AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, p));
  count_launch();
  *taken = true;
  return AQLM_B200_OK;
}

// Batch-1 call on a 1x8 / 2x8 weight whose in_features fit 8 slabs: no workspace needed.
static int try_lut_cluster(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, uint32_t flags,
                           const DeviceInfo* di, cudaStream_t st, bool* taken) {
  *taken = false;
  const int K = w->num_codebooks;
  const int in_groups = (int)(w->in_features / 8);
  if (batch != 1 || w->nbits_per_codebook != 8 || w->in_group_size != 8 || (K != 1 && K != 2)) return AQLM_B200_OK;
  if (!tun().lut_cluster || tun().disable_lut || tun().lut_debug) return AQLM_B200_OK;
  if ((in_groups & 1) || in_groups > 8 * kLutCJ) return AQLM_B200_OK;
  if ((reinterpret_cast<uintptr_t>(w->codes) & 3) || (reinterpret_cast<uintptr_t>(input) & 3)) return AQLM_B200_OK;
#define AQLM_LUTC(T)                                                                                              \
  (tun().lut_rb16 ? (K == 1 ? launch_lut_cluster<T, 1, 16, 768>(w, input, output, flags, di, st, taken)             \
                            : launch_lut_cluster<T, 2, 16, 768>(w, input, output, flags, di, st, taken))            \
                  : (K == 1 ? launch_lut_cluster<T, 1, 32, kLutCThreads>(w, input, output, flags, di, st, taken)    \
                            : launch_lut_cluster<T, 2, 32, kLutCThreads>(w, input, output, flags, di, st, taken)))
  if (w->dtype == AQLM_B200_F16) return AQLM_LUTC(__half);
  return AQLM_LUTC(__nv_bfloat16);
#undef AQLM_LUTC
}

// ---- fused dequant + tcgen05 GEMM: host side ------------------------------------------------------
typedef CUresult (*tmap_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static tmap_encode_fn get_tmap_encode() {
  static tmap_encode_fn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<tmap_encode_fn>(p);
  });
  return fn;
}

// cuTensorMapEncodeTiled is a DRIVER entry point: it needs a current context on the calling thread.  Threads that have
// only made runtime calls that do not bind one (e.g. an autograd worker thread: error 201, CUDA_ERROR_INVALID_CONTEXT)
// get the primary context bound by a no-op runtime call, once per thread.
static void ensure_driver_context() {
  static thread_local bool bound = false;
  if (!bound) {
    (void)cudaFree(nullptr);
    bound = true;
  }
}


struct GemmPlan {
  bool ok = false;       // tcgen05 path applicable
  int m_tiles = 0, n_tiles = 0, n_tile = 0, ksplit = 1, stages = 0, total_kblocks = 0, cluster = 1;
  int tile_m = kGemmBlockM;  // output rows per CTA tile
  bool v2 = false;           // producer mapping: one 4-warp group per stage, thread <-> row
  bool atmem = false;        // A operand written to tensor memory (needs v2)
  int a_stages = 0, groups = 0;  // ATMEM: A stages in TMEM (decoupled from the X stages) / V2: producer groups
  size_t counters_bytes = 0, partials_bytes = 0;
};

static GemmPlan gemm_plan(const aqlm_b200_weight_t* w, int64_t batch, const DeviceInfo* di, bool allow_split) {
  GemmPlan g;
  const int K = w->num_codebooks, nbits = w->nbits_per_codebook, gs = w->in_group_size;
  const int cb = nbits <= 8 ? 1 : 2;
  const bool g16 = gs == 16;
  if (nbits != 8 && nbits != 16) return g;
  // in_group_size 16: the 1x16 scheme only; its 256-bit gathers need a 32-byte aligned codebook (any torch allocation is)
  // No batch threshold: the tensor-core kernel beat the GEMV passes at every measured Llama-3-8B shape and batch, by
  // 2.2-4.0x at 7 rows and 28-75x at 256 (profiles/r03/probe_gemm_g16_matmat_dequant.jsonl)
  if (g16 && (K != 1 || nbits != 16 || (reinterpret_cast<uintptr_t>(w->codebooks) & 31) != 0)) return g;
  if (!(K == 1 || K == 2 || K == 4 || K == 8) || 8 * K * cb > kCodeTileBytes) return g;
  if (w->in_features % kGemmBlockK != 0) return g;
  if ((reinterpret_cast<uintptr_t>(w->codes) & 15) != 0) return g;
  // TMA needs a 16-byte multiple as the global row stride of the code matrix (1x8 and 1x16 g16: in_features % 128 == 0);
  // other shapes take the GEMV fallback in aqlm_b200_matmat_dequant_ws
  if (((size_t)(w->in_features / gs) * K * cb) % 16 != 0) return g;
  if (tun().disable_tcgen05) return g;
  g.total_kblocks = (int)(w->in_features / kGemmBlockK);
  if (batch <= 256) {
    g.n_tile = (int)((batch + 15) / 16 * 16);
    g.n_tiles = 1;
  } else {
    g.n_tile = 256;
    g.n_tiles = (int)((batch + 255) / 256);
  }
  // producer mapping V2 (one 4-warp group per stage) measured: 1x16 496 vs 505 TFLOP/s (V1), 2x8 134 vs 394, 8x8 196 vs 119
  // -> V2 for schemes with many codebooks; A-in-TMEM builds on V2 (profiles/r01/gemm_experiments.md, profiles/r02/)
  // A in tensor memory: measured 1x16 61.7 -> 55.1 us, 2x8 69.3 -> 49.2 us (4096->14336/11008, bs=256); 8x8 no gain
  g.atmem = (tun().gemm_atmem < 0 ? (K <= 2) : tun().gemm_atmem != 0) && !(tun().gemm_debug & 1);
  g.v2 = g.atmem || ((tun().gemm_v2 < 0 ? (K >= 4 ? 1 : 0) : tun().gemm_v2) != 0 && !(tun().gemm_debug & 1));
  // in_group_size 16 is built in the V2 + A-in-TMEM form only: switches that force another form leave it to the GEMV passes
  if (g16 && (!g.atmem || tun().gemm_v2 == 0)) return g;
  const size_t budget = (size_t)di->max_smem_optin;
  // At most 3 stages: shared memory taken here is L1 taken from the codebook gathers (outstanding misses need L1
  // lines); measured at N=256: 4 stages 335 TFLOP/s, 3 stages 484-503, 2 stages 470 (profiles/r01/gemm_experiments.md)
  int S = 3;
  while (S > 2 && gemm_smem_layout(S, g.n_tile, g.atmem).total > budget) --S;
  if (gemm_smem_layout(S, g.n_tile, g.atmem).total > budget) return g;
  const int forced_s = tun().gemm_stages;
  if (forced_s >= 2 && forced_s <= S) S = forced_s;
  if (forced_s == 4 && g.v2 && gemm_smem_layout(4, g.n_tile, g.atmem).total <= budget) S = 4;  // experiment: 4 X stages
  g.stages = S;
  g.groups = S;
  g.a_stages = S;
  if (g.atmem) {
    // tensor memory: accumulator columns [0, n_tile), then 32 columns per A stage; 512 columns in all
    const int room = (512 - ((g.n_tile + 31) & ~31)) / 32;
    int sa = tun().gemm_a_stages > 0 ? tun().gemm_a_stages : 6;
    if (sa > room) sa = room;
    if (sa > 8) sa = 8;
    if (sa < 2) sa = 2;
    g.a_stages = sa;
    g.groups = tun().gemm_groups > 0 ? (tun().gemm_groups > 4 ? 4 : tun().gemm_groups) : 3;
  }
  // ---- tile height and split-K: a small cost model over (tile_m, ksplit), in SM clocks ----
  //   per k-block of one CTA: max(gathers, tensor pipe, shared-memory traffic) + a fixed synchronisation cost;
  //   per CTA: its k-blocks + a fixed cost (launch ramp, TMEM alloc, pipeline fill, epilogue: ~5 us measured);
  //   per launch: waves x CTA time + split-K fix-up traffic (partials written and read once through L2).
  // The gather rate is the measured per-SM rate of random 16-byte codebook reads (profiles/: ~0.85/clk from L2 for the
  // 1 MiB 1x16 codebook; 256-entry codebooks are L1-resident and gather faster).  in_group_size 16 issues 4 gathers per
  // row per k-block, each one 32-byte request; the GEMM's rate of those is not measured, so the 16-byte rate stands in.
  const double clk = 1.9e9;
  const double gather_per_clk = (nbits == 16 ? 0.85 : 1.6) * (g.atmem ? 1.0 : 0.7);  // SS form: smaller L1 -> slower gathers
  const double gathers_per_row = (double)(kGemmBlockK / gs) * K;
  const double t_mma = 2.0 * g.n_tile;                                                 // 4 x (128 x N x 16) at 4096 MAC/clk
  int best_tm = kGemmBlockM, best_ks = 1;
  double best = 1e30;
  const int max_ks = !allow_split ? 1 : (g.total_kblocks / 2 < 16 ? (g.total_kblocks / 2 < 1 ? 1 : g.total_kblocks / 2) : 16);
  const bool want_pairs = (tun().gemm_cluster > 0 ? tun().gemm_cluster : (g.n_tile >= 128 ? 2 : 1)) > 1;
  for (int tm = kGemmBlockM; tm >= 32; tm -= (tm > 64 ? 1 : 8)) {
    const long long tiles = ((w->out_features + tm - 1) / tm) * (long long)g.n_tiles;
    if (tiles > kGemmMaxTiles) continue;
    // CTA pairs multicast the X tile: keep the number of M tiles even (full-height tiles stay as the fallback)
    if (want_pairs && tm != kGemmBlockM && (((w->out_features + tm - 1) / tm) & 1)) continue;
    const double t_gather = tm * gathers_per_row / gather_per_clk;
    const double t_smem = (g.atmem ? 0.0 : (128.0 + tm) * 128.0 / 128.0) + 2.0 * g.n_tile;  // bytes / (128 B/clk)
    const double t_kb = (t_gather > t_mma ? (t_gather > t_smem ? t_gather : t_smem) : (t_mma > t_smem ? t_mma : t_smem)) + 60.0;
    for (int c = 1; c <= max_ks; ++c) {
      const double ctas = (double)tiles * c;
      const double waves = (double)((long long)((ctas + di->sm_count - 1) / di->sm_count));
      const double kb_cta = (double)((g.total_kblocks + c - 1) / c);
      const double fix = c > 1 ? ctas * g.n_tile * kGemmBlockM * 4.0 * 2.0 / 4e12 * clk : 0.0;
      const double t = waves * (kb_cta * t_kb + 5e-6 * clk) + fix;
      if (t < best * (tm == kGemmBlockM && c == 1 ? 1.0 : 0.97)) {  // prefer full tiles / fewer splits unless the gain is real
        best = t;
        best_tm = tm;
        best_ks = c;
      }
    }
  }
  g.tile_m = best_tm;
  int ks = best_ks;
  if (tun().gemm_tile_m >= 8 && tun().gemm_tile_m <= kGemmBlockM) g.tile_m = tun().gemm_tile_m;
  g.m_tiles = (int)((w->out_features + g.tile_m - 1) / g.tile_m);
  if (allow_split && tun().gemm_ksplit > 0) ks = tun().gemm_ksplit;
  if (ks > g.total_kblocks) ks = g.total_kblocks;
  if (ks < 1) ks = 1;
  // fixed-size counter region (the partials of one plan must never overlap the counters of another plan that
  // reuses the same persistent workspace)
  g.counters_bytes = kWsCountersBytes;
  if ((size_t)g.m_tiles * g.n_tiles > (size_t)kGemmMaxTiles) ks = 1;
  g.ksplit = ks;
  // X-tile multicast: CTAs of a cluster (consecutive M tiles, same K range) each TMA-load 1/C of the X tile and
  // multicast it to all C, cutting the L2->SM traffic of X by C.
  int cl = tun().gemm_cluster > 0 ? tun().gemm_cluster : (g.n_tile >= 128 ? 2 : 1);
  while (cl > 1 && (g.m_tiles % cl != 0 || g.n_tile % (8 * cl) != 0)) cl >>= 1;
  g.cluster = cl < 1 ? 1 : cl;
  g.partials_bytes = ks > 1 ? (size_t)g.m_tiles * g.n_tiles * ks * g.n_tile * kGemmBlockM * 4 : 0;
  g.ok = true;
  return g;
}

template <typename T, int K, int CB, int GS = 8>
static int launch_gemm(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, const GemmPlan& g,
                       void* workspace, cudaStream_t st) {
  const size_t row_bytes = (size_t)(w->in_features / GS) * K * CB;
  const DeviceInfo* di = device_info();
  if (!di) return AQLM_B200_ERR_CUDA;
  tmap_encode_fn enc = get_tmap_encode();
  if (!enc) return fail(AQLM_B200_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  ensure_driver_context();
  CUtensorMap tx, tc;
  {
    cuuint64_t dims[2] = {(cuuint64_t)w->in_features, (cuuint64_t)batch};
    cuuint64_t strides[1] = {(cuuint64_t)w->in_features * 2};
    cuuint32_t box[2] = {(cuuint32_t)kGemmBlockK, (cuuint32_t)(g.n_tile / g.cluster)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&tx, DT<T>::is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                     const_cast<void*>(input), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(AQLM_B200_ERR_CUDA, "cuTensorMapEncodeTiled(x) failed: %d", (int)r);
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)row_bytes, (cuuint64_t)w->out_features};
    cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
    cuuint32_t box[2] = {(cuuint32_t)kCodeTileBytes, (cuuint32_t)g.tile_m};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&tc, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(w->codes), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(AQLM_B200_ERR_CUDA, "cuTensorMapEncodeTiled(codes) failed: %d", (int)r);
  }
  GemmParams p;
  p.codebooks = w->codebooks;
  p.scales = w->scales;
  p.bias = w->bias;
  p.y = output;
  p.ws_counters = g.ksplit > 1 ? reinterpret_cast<unsigned int*>(workspace) : nullptr;
  p.ws_partials = g.ksplit > 1 ? reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + g.counters_bytes) : nullptr;
  p.out_features = (int)w->out_features;
  p.batch = (int)batch;
  p.nbits = w->nbits_per_codebook;
  p.total_kblocks = g.total_kblocks;
  p.ksplit = g.ksplit;
  p.n_tile = g.n_tile;
  p.stages = g.stages;
  p.a_stages = g.a_stages;
  p.groups = g.groups;
  p.tile_m = g.tile_m;
  p.cluster = g.cluster;
  p.debug = tun().gemm_debug;
  p.gather_mode = tun().gemm_gather_mode >= 0 ? tun().gemm_gather_mode : (w->nbits_per_codebook > 8 ? 1 : 0);
  p.codes = w->codes;
  p.row_bytes = (long long)row_bytes;
  const size_t smem = gemm_smem_layout(g.stages, g.n_tile, g.atmem).total;
  const bool v2 = g.v2 && g.stages <= 4;
  const bool atmem = g.atmem && v2;
  decltype(&gemm_dequant_kernel<T, K, CB, true, true>) kernel;
  if constexpr (GS == 16) {
    if (!atmem) return fail(AQLM_B200_ERR_UNSUPPORTED, "in_group_size 16 GEMM is built in the V2 + A-in-TMEM form only");
    kernel = gemm_dequant_kernel<T, K, CB, true, true, 16>;
  } else {
    kernel = atmem ? gemm_dequant_kernel<T, K, CB, true, true>
                   : (v2 ? gemm_dequant_kernel<T, K, CB, true, false> : gemm_dequant_kernel<T, K, CB, false, false>);
  }
  static SmemMarks marks[3];
  if (int rc = ensure_smem(kernel, smem, marks[atmem ? 2 : (v2 ? 1 : 0)], di)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(g.m_tiles, g.ksplit, g.n_tiles);
  cfg.blockDim = dim3(v2 ? kGemmThreadsV2 : kGemmThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = g.cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = tun().pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, tx, tc, p));
  count_launch();
  return AQLM_B200_OK;
}

template <typename T>
static int gemm_typed(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, const GemmPlan& g,
                      void* workspace, cudaStream_t st) {
  const int K = w->num_codebooks, cb = w->nbits_per_codebook <= 8 ? 1 : 2;
  if (w->in_group_size == 16) return launch_gemm<T, 1, 2, 16>(w, input, output, batch, g, workspace, st);  // gemm_plan: 1x16 only
  if (cb == 2 && K == 1) return launch_gemm<T, 1, 2>(w, input, output, batch, g, workspace, st);
  if (cb == 2 && K == 2) return launch_gemm<T, 2, 2>(w, input, output, batch, g, workspace, st);
  if (cb == 2 && K == 4) return launch_gemm<T, 4, 2>(w, input, output, batch, g, workspace, st);
  if (cb == 2 && K == 8) return launch_gemm<T, 8, 2>(w, input, output, batch, g, workspace, st);
  if (K == 1) return launch_gemm<T, 1, 1>(w, input, output, batch, g, workspace, st);
  if (K == 2) return launch_gemm<T, 2, 1>(w, input, output, batch, g, workspace, st);
  if (K == 4) return launch_gemm<T, 4, 1>(w, input, output, batch, g, workspace, st);
  return launch_gemm<T, 8, 1>(w, input, output, batch, g, workspace, st);
}

// ---- fused dequant + TRANSPOSED tcgen05 GEMM (backward w.r.t. the input): host side ---------------------
struct GemmTPlan {
  bool ok = false;
  int m_tiles = 0, n_tiles = 0, n_tile = 0, ksplit = 1, stages = 0, total_kblocks = 0;
  size_t counters_bytes = 0, partials_bytes = 0;
};

static GemmTPlan gemm_t_plan(const aqlm_b200_weight_t* w, int64_t batch, const DeviceInfo* di, bool allow_split) {
  GemmTPlan g;
  const int K = w->num_codebooks, nbits = w->nbits_per_codebook, gs = w->in_group_size;
  const int cb = nbits <= 8 ? 1 : 2;
  if (nbits != 8 && nbits != 16) return g;
  // in_group_size 16: 1x16 only, 256-bit gathers from a 32-byte aligned codebook
  if (gs == 16 && (K != 1 || nbits != 16 || (reinterpret_cast<uintptr_t>(w->codebooks) & 31) != 0)) return g;
  if (!(K == 1 || K == 2 || K == 4 || K == 8) || 16 * K * cb > 256) return g;
  if (w->out_features % 8 != 0) return g;  // TMA row stride of grad_out
  if ((reinterpret_cast<uintptr_t>(w->codes) & 15) != 0) return g;
  if (((size_t)(w->in_features / gs) * K * cb) % 16 != 0) return g;  // 1x8 and 1x16 g16: in_features % 128 == 0
  if (tun().disable_tcgen05) return g;
  g.total_kblocks = (int)((w->out_features + kGemmBlockK - 1) / kGemmBlockK);
  g.m_tiles = (int)((w->in_features + kGemmBlockM - 1) / kGemmBlockM);
  if (batch <= 256) {
    g.n_tile = (int)((batch + 15) / 16 * 16);
    g.n_tiles = 1;
  } else {
    g.n_tile = 256;
    g.n_tiles = (int)((batch + 255) / 256);
  }
  const int ctile_row_bytes = (kGemmBlockM / gs) * K * cb;
  const size_t budget = (size_t)di->max_smem_optin;
  int S = 3;
  while (S > 2 && gemm_t_smem_layout(S, g.n_tile, ctile_row_bytes).total > budget) --S;
  if (gemm_t_smem_layout(S, g.n_tile, ctile_row_bytes).total > budget) return g;
  if (tun().gemm_stages >= 2 && tun().gemm_stages <= S) S = tun().gemm_stages;
  g.stages = S;
  if ((size_t)g.m_tiles * g.n_tiles > (size_t)kGemmMaxTiles) return g;
  int ks = 1;
  if (allow_split) {
    // same cost model as the forward plan: a k-block costs max(gathers, tensor pipe, smem traffic), every wave pays a
    // fixed ~5 us, split-K partials go through L2 once each way
    const double clk = 1.9e9;
    // (64 out rows x 128 / in_group_size gathers; the 32-byte gathers of in_group_size 16 are costed at the 16-byte rate)
    const double t_gather = 64.0 * (kGemmBlockM / gs) * K / ((nbits == 16 ? 0.85 : 1.6) * 0.7);
    const double t_smem = 256.0 + 2.0 * g.n_tile, t_mma = 2.0 * g.n_tile;
    const double t_kb = (t_gather > t_smem ? (t_gather > t_mma ? t_gather : t_mma) : (t_smem > t_mma ? t_smem : t_mma)) + 60.0;
    const double tiles = (double)g.m_tiles * g.n_tiles;
    double best = 1e30;
    const int max_ks = g.total_kblocks / 2 < 16 ? (g.total_kblocks / 2 < 1 ? 1 : g.total_kblocks / 2) : 16;
    for (int c = 1; c <= max_ks; ++c) {
      const double ctas = tiles * c;
      const double waves = (double)((long long)((ctas + di->sm_count - 1) / di->sm_count));
      const double kb_cta = (double)((g.total_kblocks + c - 1) / c);
      const double fix = c > 1 ? ctas * g.n_tile * kGemmBlockM * 4.0 * 2.0 / 4e12 * clk : 0.0;
      const double t = waves * (kb_cta * t_kb + 5e-6 * clk) + fix;
      if (t < best * 0.97) {
        best = t;
        ks = c;
      }
    }
    if (tun().gemm_ksplit > 0) ks = tun().gemm_ksplit;
    if (ks > g.total_kblocks) ks = g.total_kblocks;
    if (ks < 1) ks = 1;
  }
  g.ksplit = ks;
  g.counters_bytes = kWsCountersBytes;
  g.partials_bytes = ks > 1 ? (size_t)g.m_tiles * g.n_tiles * ks * g.n_tile * kGemmBlockM * 4 : 0;
  g.ok = true;
  return g;
}

template <typename T, int K, int CB, int GS = 8>
static int launch_gemm_t(const aqlm_b200_weight_t* w, const void* grad_output, void* grad_input, int64_t batch,
                         const GemmTPlan& g, void* workspace, cudaStream_t st) {
  const DeviceInfo* di = device_info();
  if (!di) return AQLM_B200_ERR_CUDA;
  tmap_encode_fn enc = get_tmap_encode();
  if (!enc) return fail(AQLM_B200_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  constexpr int GBT = (kGemmBlockM / GS) * K * CB;  // code bytes per out row per 128-in-feature tile (TMA box, >= 16)
  ensure_driver_context();
  CUtensorMap tg, tc;
  {
    cuuint64_t dims[2] = {(cuuint64_t)w->out_features, (cuuint64_t)batch};
    cuuint64_t strides[1] = {(cuuint64_t)w->out_features * 2};
    cuuint32_t box[2] = {(cuuint32_t)kGemmBlockK, (cuuint32_t)g.n_tile};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&tg, DT<T>::is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                     const_cast<void*>(grad_output), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(AQLM_B200_ERR_CUDA, "cuTensorMapEncodeTiled(grad_output) failed: %d", (int)r);
  }
  {
    const size_t row_bytes = (size_t)(w->in_features / GS) * K * CB;
    cuuint64_t dims[2] = {(cuuint64_t)row_bytes, (cuuint64_t)w->out_features};
    cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
    cuuint32_t box[2] = {(cuuint32_t)GBT, (cuuint32_t)kGemmTCtileRows};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&tc, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(w->codes), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(AQLM_B200_ERR_CUDA, "cuTensorMapEncodeTiled(codes, transposed) failed: %d", (int)r);
  }
  GemmTParams p;
  p.codebooks = w->codebooks;
  p.scales = w->scales;
  p.y = grad_input;
  p.ws_counters = g.ksplit > 1 ? reinterpret_cast<unsigned int*>(workspace) : nullptr;
  p.ws_partials = g.ksplit > 1 ? reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + g.counters_bytes) : nullptr;
  p.in_features = (int)w->in_features;
  p.out_features = (int)w->out_features;
  p.batch = (int)batch;
  p.nbits = w->nbits_per_codebook;
  p.total_kblocks = g.total_kblocks;
  p.ksplit = g.ksplit;
  p.n_tile = g.n_tile;
  p.stages = g.stages;
  p.gather_mode = tun().gemm_gather_mode >= 0 ? tun().gemm_gather_mode : (w->nbits_per_codebook > 8 ? 1 : 0);
  const size_t smem = gemm_t_smem_layout(g.stages, g.n_tile, GBT).total;
  auto kernel = gemm_dequant_t_kernel<T, K, CB, GS>;
  static SmemMarks marks;
  if (int rc = ensure_smem(kernel, smem, marks, di)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(g.m_tiles, g.ksplit, g.n_tiles);
  cfg.blockDim = dim3(kGemmTThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = tun().pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, tg, tc, p));
  count_launch();
  return AQLM_B200_OK;
}

template <typename T>
static int gemm_t_typed(const aqlm_b200_weight_t* w, const void* grad_output, void* grad_input, int64_t batch,
                        const GemmTPlan& g, void* workspace, cudaStream_t st) {
  const int K = w->num_codebooks, cb = w->nbits_per_codebook <= 8 ? 1 : 2;
  if (w->in_group_size == 16) return launch_gemm_t<T, 1, 2, 16>(w, grad_output, grad_input, batch, g, workspace, st);  // 1x16 only
  if (cb == 2 && K == 1) return launch_gemm_t<T, 1, 2>(w, grad_output, grad_input, batch, g, workspace, st);
  if (cb == 2 && K == 2) return launch_gemm_t<T, 2, 2>(w, grad_output, grad_input, batch, g, workspace, st);
  if (cb == 2 && K == 4) return launch_gemm_t<T, 4, 2>(w, grad_output, grad_input, batch, g, workspace, st);
  if (cb == 2 && K == 8) return launch_gemm_t<T, 8, 2>(w, grad_output, grad_input, batch, g, workspace, st);
  if (K == 1) return launch_gemm_t<T, 1, 1>(w, grad_output, grad_input, batch, g, workspace, st);
  if (K == 2) return launch_gemm_t<T, 2, 1>(w, grad_output, grad_input, batch, g, workspace, st);
  if (K == 4) return launch_gemm_t<T, 4, 1>(w, grad_output, grad_input, batch, g, workspace, st);
  return launch_gemm_t<T, 8, 1>(w, grad_output, grad_input, batch, g, workspace, st);
}

static aqlm_b200_weight_t make_weight(const void* codes, const void* codebooks, const void* scales, const void* bias,
                                      int64_t in_features, int64_t out_features, int K, int nbits, int g, int dtype) {
  aqlm_b200_weight_t w;
  memset(&w, 0, sizeof(w));
  w.codes = codes;
  w.codebooks = codebooks;
  w.scales = scales;
  w.bias = bias;
  w.in_features = in_features;
  w.out_features = out_features;
  w.num_codebooks = K;
  w.nbits_per_codebook = nbits;
  w.in_group_size = g;
  w.out_group_size = 1;
  w.dtype = dtype;
  return w;
}

}  // namespace aqlm_b200

using namespace aqlm_b200;

extern "C" {

int aqlm_b200_version(void) { return AQLM_B200_VERSION; }
void aqlm_b200_reload_tunables(void) { tun().load(); }
const char* aqlm_b200_last_error(void) { return tls_error_buf(); }
uint64_t aqlm_b200_launch_count(void) { return g_launch_count.load(); }

int aqlm_b200_matmat_ex(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, uint32_t flags,
                        void* stream) {
  const bool partial = (flags & AQLM_B200_FLAG_PARTIAL_F32) != 0;
  int rc = validate(w, !partial);
  if (rc) return rc;
  if (batch < 0) return fail(AQLM_B200_ERR_SHAPE, "negative batch");
  if (batch == 0) return AQLM_B200_OK;
  if (!input || !output) return fail(AQLM_B200_ERR_SHAPE, "input/output pointer is NULL");
  const DeviceInfo* di = device_info();
  if (!di) return (int)(strstr(tls_error_buf(), "sm_100a") ? AQLM_B200_ERR_ARCH : AQLM_B200_ERR_CUDA);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  {
    // batch 1 -- and batch 2-3 as one launch per row, like the reference's per-row host loop (cuda_kernel.cpp:387-421):
    // measured faster than one pass of the gather kernel up to 3 rows (profiles/r02/probe_lut_*.jsonl)
    const int64_t lut_rows = (batch == 1 || (tun().lut_batch_loop && batch <= 3)) ? batch : 0;
    const size_t out_elt = partial ? 4 : 2;
    int64_t done = 0;
    for (; done < lut_rows; ++done) {
      bool taken = false;
      rc = try_lut_cluster(w, reinterpret_cast<const uint8_t*>(input) + (size_t)done * w->in_features * 2,
                           reinterpret_cast<uint8_t*>(output) + (size_t)done * w->out_features * out_elt, 1, flags, di, st, &taken);
      if (rc) return rc;
      if (!taken) break;  // not applicable (decided before any launch: `taken` is the same for every row)
    }
    if (lut_rows > 0 && done == lut_rows) return AQLM_B200_OK;
  }
  if (w->dtype == AQLM_B200_F16) return matmat_typed<__half>(w, input, output, batch, flags, di, st);
  return matmat_typed<__nv_bfloat16>(w, input, output, batch, flags, di, st);
}

size_t aqlm_b200_matmat_workspace_bytes(const aqlm_b200_weight_t* w, int64_t batch) {
  if (validate(w, false) != AQLM_B200_OK || batch <= 0) return 0;
  const DeviceInfo* di = device_info();
  if (!di) return 0;
  if (batch > 2) return 0;
  const LutPlan L = lut_plan(w, 1, di);
  return L.ok ? kWsCountersBytes + L.partials_bytes : 0;
}

int aqlm_b200_matmat_ws(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, uint32_t flags,
                        void* workspace, size_t workspace_bytes, void* stream) {
  const bool partial = (flags & AQLM_B200_FLAG_PARTIAL_F32) != 0;
  int rc = validate(w, !partial);
  if (rc) return rc;
  const int64_t ws_rows = (batch == 1 || (tun().lut_batch_loop && batch == 2 && w->num_codebooks >= 4)) ? batch : 0;
  if (ws_rows > 0 && workspace && input && output && (reinterpret_cast<uintptr_t>(input) & 3) == 0) {
    const DeviceInfo* di = device_info();
    if (!di) return (int)(strstr(tls_error_buf(), "sm_100a") ? AQLM_B200_ERR_ARCH : AQLM_B200_ERR_CUDA);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (batch == 1) {  // K <= 2, in <= 4096: the cluster kernel needs no workspace (matmat_ex also loops it for batch 2-3)
      bool taken = false;
      rc = try_lut_cluster(w, input, output, 1, flags, di, st, &taken);
      if (rc || taken) return rc;
    }
    const LutPlan L = lut_plan(w, 1, di);
    const bool cluster_case = w->num_codebooks <= 2 && (w->in_features / 8) <= 8 * kLutCJ && tun().lut_cluster;
    if (L.ok && workspace_bytes >= kWsCountersBytes + L.partials_bytes && !(batch > 1 && cluster_case)) {
      const size_t out_elt = partial ? 4 : 2;
      for (int64_t b = 0; b < ws_rows; ++b) {  // launches are stream-ordered: the workspace is reused row after row
        const void* xin = reinterpret_cast<const uint8_t*>(input) + (size_t)b * w->in_features * 2;
        void* yout = reinterpret_cast<uint8_t*>(output) + (size_t)b * w->out_features * out_elt;
        rc = w->dtype == AQLM_B200_F16 ? lut_typed<__half>(w, xin, yout, flags, L, workspace, st)
                                       : lut_typed<__nv_bfloat16>(w, xin, yout, flags, L, workspace, st);
        if (rc) return rc;
      }
      return AQLM_B200_OK;
    }
  }
  return aqlm_b200_matmat_ex(w, input, output, batch, flags, stream);
}

int aqlm_b200_matmat_grouped(const aqlm_b200_weight_t* w, const int64_t* seg_rows, int n_seg, const void* input,
                             void* output, int64_t batch, uint32_t flags, void* stream) {
  const bool partial = (flags & AQLM_B200_FLAG_PARTIAL_F32) != 0;
  int rc = validate(w, !partial);
  if (rc) return rc;
  if (!seg_rows || n_seg < 1 || n_seg > 4) return fail(AQLM_B200_ERR_SHAPE, "grouped launch takes 1..4 segments");
  if (w->num_codebooks != 1 || w->nbits_per_codebook != 16 || w->in_group_size != 8)
    return fail(AQLM_B200_ERR_UNSUPPORTED, "grouped launch is implemented for the 1x16 (in_group 8) scheme only");
  if (batch < 1 || batch > 8) return fail(AQLM_B200_ERR_UNSUPPORTED, "grouped launch takes 1..8 batch rows");
  if (!input || !output) return fail(AQLM_B200_ERR_SHAPE, "input/output pointer is NULL");
  int64_t total = 0;
  for (int i = 0; i < n_seg; ++i) total += seg_rows[i];
  if (total != w->out_features) return fail(AQLM_B200_ERR_SHAPE, "segment rows do not add up to out_features");
  const size_t row_bytes = (size_t)(w->in_features / 8) * 2;
  if (row_bytes % 16 != 0 || (reinterpret_cast<uintptr_t>(w->codes) & 15) || (reinterpret_cast<uintptr_t>(input) & 15))
    return fail(AQLM_B200_ERR_UNSUPPORTED, "grouped launch needs 16-byte aligned code rows and input");
  const DeviceInfo* di = device_info();
  if (!di) return (int)(strstr(tls_error_buf(), "sm_100a") ? AQLM_B200_ERR_ARCH : AQLM_B200_ERR_CUDA);
  GemvParams p;
  p.codes = w->codes;
  p.codebooks = w->codebooks;
  p.scales = w->scales;
  p.bias = w->bias;
  p.x = input;
  p.y = output;
  p.out_features = (int)w->out_features;
  p.in_features = (int)w->in_features;
  p.in_groups = (int)(w->in_features / 8);
  p.nbits = 16;
  p.num_codebooks = 1;
  p.batch = (int)batch;
  p.partial_f32 = partial ? 1 : 0;
  p.n_seg = n_seg;
  p.row_block = 0;
  int64_t acc = 0;
  for (int i = 0; i < 4; ++i) {
    if (i < n_seg) acc += seg_rows[i];
    p.seg_end[i] = (int)acc;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int bt = batch == 1 ? 1 : (batch == 2 ? 2 : (batch <= 4 ? 4 : 8));
  if (vec_smem_bytes(p, 1, 2, 8, bt, false, di->sm_count) > (size_t)di->max_smem_optin - 1024)
    return fail(AQLM_B200_ERR_UNSUPPORTED, "grouped launch: activation tile does not fit in shared memory");
#define AQLM_GRP(T)                                                   \
  (bt == 1 ? launch_1x16<T, 1, 0>(p, di, st) : bt == 2 ? launch_1x16<T, 2, 0>(p, di, st) \
           : bt == 4 ? launch_1x16<T, 4, 0>(p, di, st) : launch_1x16<T, 8, 0>(p, di, st))
  if (w->dtype == AQLM_B200_F16) return AQLM_GRP(__half);
  return AQLM_GRP(__nv_bfloat16);
#undef AQLM_GRP
}

int aqlm_b200_matmat(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch, void* stream) {
  return aqlm_b200_matmat_ex(w, input, output, batch, 0, stream);
}

size_t aqlm_b200_matmat_dequant_workspace_bytes(const aqlm_b200_weight_t* w, int64_t batch) {
  if (validate(w, true) != AQLM_B200_OK || batch <= 0) return 0;
  const DeviceInfo* di = device_info();
  if (!di) return 0;
  const GemmPlan g = gemm_plan(w, batch, di, true);
  if (!g.ok || g.ksplit <= 1) return 0;
  return g.counters_bytes + g.partials_bytes;
}

int aqlm_b200_matmat_dequant_ws(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch,
                                void* workspace, size_t workspace_bytes, void* stream) {
  int rc = validate(w, true);
  if (rc) return rc;
  if (batch < 0) return fail(AQLM_B200_ERR_SHAPE, "negative batch");
  if (batch == 0) return AQLM_B200_OK;
  if (!input || !output) return fail(AQLM_B200_ERR_SHAPE, "input/output pointer is NULL");
  const DeviceInfo* di = device_info();
  if (!di) return (int)(strstr(tls_error_buf(), "sm_100a") ? AQLM_B200_ERR_ARCH : AQLM_B200_ERR_CUDA);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  GemmPlan g = gemm_plan(w, batch, di, workspace != nullptr);
  if (g.ok && g.ksplit > 1 && workspace_bytes < g.counters_bytes + g.partials_bytes) g = gemm_plan(w, batch, di, false);
  if (!g.ok || (reinterpret_cast<uintptr_t>(input) & 15) != 0) {
    // shapes the tensor-core kernel does not cover (in_features % 64 != 0, code rows not a 16-byte multiple, odd KxN,
    // in_group 16 other than 1x16):
    // batch passes of 8 rows through the fused gather+dequant+dot kernel
    return aqlm_b200_matmat_ex(w, input, output, batch, 0, stream);
  }
  if (w->dtype == AQLM_B200_F16) return gemm_typed<__half>(w, input, output, batch, g, workspace, st);
  return gemm_typed<__nv_bfloat16>(w, input, output, batch, g, workspace, st);
}

int aqlm_b200_matmat_dequant(const aqlm_b200_weight_t* w, const void* input, void* output, int64_t batch,
                             void* stream) {
  return aqlm_b200_matmat_dequant_ws(w, input, output, batch, nullptr, 0, stream);  // no workspace: no split-K
}

int aqlm_b200_dequant(const aqlm_b200_weight_t* w, void* weight_out, int apply_scales, void* stream) {
  int rc = validate(w, apply_scales != 0);
  if (rc) return rc;
  if (!weight_out || (reinterpret_cast<uintptr_t>(weight_out) & 15))
    return fail(AQLM_B200_ERR_SHAPE, "weight_out must be a 16-byte aligned device pointer");
  if (!device_info()) return (int)(strstr(tls_error_buf(), "sm_100a") ? AQLM_B200_ERR_ARCH : AQLM_B200_ERR_CUDA);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (w->dtype == AQLM_B200_F16) return dequant_typed<__half>(w, weight_out, apply_scales, st);
  return dequant_typed<__nv_bfloat16>(w, weight_out, apply_scales, st);
}

size_t aqlm_b200_matmat_dequant_transposed_workspace_bytes(const aqlm_b200_weight_t* w, int64_t batch) {
  if (validate(w, true) != AQLM_B200_OK || batch <= 0) return 0;
  const DeviceInfo* di = device_info();
  if (!di) return 0;
  const GemmTPlan g = gemm_t_plan(w, batch, di, true);
  if (!g.ok || g.ksplit <= 1) return 0;
  return g.counters_bytes + g.partials_bytes;
}

int aqlm_b200_matmat_dequant_transposed(const aqlm_b200_weight_t* w, const void* grad_output, void* grad_input,
                                        int64_t batch, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = validate(w, true);
  if (rc) return rc;
  if (batch < 0) return fail(AQLM_B200_ERR_SHAPE, "negative batch");
  if (batch == 0) return AQLM_B200_OK;
  if (!grad_output || !grad_input) return fail(AQLM_B200_ERR_SHAPE, "grad_output/grad_input pointer is NULL");
  if ((reinterpret_cast<uintptr_t>(grad_output) & 15) != 0)
    return fail(AQLM_B200_ERR_SHAPE, "grad_output must be 16-byte aligned");
  const DeviceInfo* di = device_info();
  if (!di) return (int)(strstr(tls_error_buf(), "sm_100a") ? AQLM_B200_ERR_ARCH : AQLM_B200_ERR_CUDA);
  GemmTPlan g = gemm_t_plan(w, batch, di, workspace != nullptr);
  if (g.ok && g.ksplit > 1 && workspace_bytes < g.counters_bytes + g.partials_bytes) g = gemm_t_plan(w, batch, di, false);
  if (!g.ok)
    return fail(AQLM_B200_ERR_UNSUPPORTED,
                "matmat_dequant_transposed: the fused kernel covers in_group_size 8 (8/16-bit codes, 1/2/4/8 codebooks) and "
                "in_group_size 16 (1x16, 32-byte aligned codebook), 16-byte aligned code rows and out_features %% 8 == 0");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (w->dtype == AQLM_B200_F16) return gemm_t_typed<__half>(w, grad_output, grad_input, batch, g, workspace, st);
  return gemm_t_typed<__nv_bfloat16>(w, grad_output, grad_input, batch, g, workspace, st);
}

int aqlm_b200_scale_bias(const float* partial, const void* scales, const void* bias, void* output, int64_t batch,
                         int64_t out_features, int32_t dtype, void* stream) {
  if (!partial || !scales || !output) return fail(AQLM_B200_ERR_SHAPE, "NULL pointer");
  if (dtype != AQLM_B200_F16 && dtype != AQLM_B200_BF16) return fail(AQLM_B200_ERR_DTYPE, "dtype must be f16/bf16");
  if (batch <= 0 || out_features <= 0) return AQLM_B200_OK;
  if (!device_info()) return (int)(strstr(tls_error_buf(), "sm_100a") ? AQLM_B200_ERR_ARCH : AQLM_B200_ERR_CUDA);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t n = batch * out_features;
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (dtype == AQLM_B200_F16)
    scale_bias_kernel<__half><<<blocks, 256, 0, st>>>(partial, (const __half*)scales, (const __half*)bias,
                                                      (__half*)output, batch, out_features);
  else
    scale_bias_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(partial, (const __nv_bfloat16*)scales,
                                                             (const __nv_bfloat16*)bias, (__nv_bfloat16*)output, batch,
                                                             out_features);
  count_launch();
  AQLM_CUDA_CHECK(cudaGetLastError());
  return AQLM_B200_OK;
}

// ---- peer-memory all-reduce (multi-GPU sharded path) -----------------------------------------------
struct aqlm_b200_comm {
  int rank, world;
  long long max_elems;
  uint8_t* peer_base[kPeerMaxWorld];
  unsigned int* local_state;  // [0] step, [1..2] tickets
  float* local_partials;      // [max_elems]
};

size_t aqlm_b200_comm_shared_bytes(int world, int64_t max_elems) {
  if (world < 1 || world > kPeerMaxWorld || max_elems <= 0) return 0;
  // flags + [set][src][max_elems] fp32 slots (stand-alone exchange kernel) + [set][src][max_elems] tagged 64-bit words
  // (exchange fused into the GEMV)
  return (size_t)kPeerFlagBytes + (size_t)2 * world * (size_t)max_elems * (sizeof(float) + sizeof(unsigned long long));
}

int aqlm_b200_shared_alloc(size_t bytes, void** ptr, void* handle64) {
  if (!ptr || !handle64 || bytes == 0) return fail(AQLM_B200_ERR_SHAPE, "bad shared_alloc arguments");
  AQLM_CUDA_CHECK(cudaMalloc(ptr, bytes));
  AQLM_CUDA_CHECK(cudaMemset(*ptr, 0, bytes));
  AQLM_CUDA_CHECK(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  AQLM_CUDA_CHECK(cudaIpcGetMemHandle(&h, *ptr));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle64, &h, 64);
  return AQLM_B200_OK;
}

int aqlm_b200_shared_open(const void* handle64, void** ptr) {
  if (!ptr || !handle64) return fail(AQLM_B200_ERR_SHAPE, "bad shared_open arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  AQLM_CUDA_CHECK(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return AQLM_B200_OK;
}

int aqlm_b200_comm_create(int rank, int world, void* const* peer_ptrs, int64_t max_elems, aqlm_b200_comm** out) {
  if (!out || !peer_ptrs || world < 1 || world > kPeerMaxWorld || rank < 0 || rank >= world || max_elems <= 0 || (max_elems & 3))
    return fail(AQLM_B200_ERR_SHAPE, "bad comm_create arguments");
  aqlm_b200_comm* c = new aqlm_b200_comm();
  c->rank = rank;
  c->world = world;
  c->max_elems = max_elems;
  for (int r = 0; r < world; ++r) c->peer_base[r] = reinterpret_cast<uint8_t*>(peer_ptrs[r]);
  AQLM_CUDA_CHECK(cudaMalloc(&c->local_state, 64));
  AQLM_CUDA_CHECK(cudaMemset(c->local_state, 0, 64));
  AQLM_CUDA_CHECK(cudaMalloc(&c->local_partials, (size_t)max_elems * sizeof(float)));
  AQLM_CUDA_CHECK(cudaDeviceSynchronize());
  *out = c;
  return AQLM_B200_OK;
}

void* aqlm_b200_comm_partials(aqlm_b200_comm* c) { return c ? c->local_partials : nullptr; }

int aqlm_b200_comm_destroy(aqlm_b200_comm* c) {
  if (!c) return AQLM_B200_OK;
  cudaFree(c->local_state);
  cudaFree(c->local_partials);
  delete c;
  return AQLM_B200_OK;
}

int aqlm_b200_allreduce_scale_bias(aqlm_b200_comm* c, const float* partial, const void* scales, const void* bias,
                                   void* output, int64_t batch, int64_t out_features, int32_t dtype, void* stream) {
  if (!c || !partial || !scales || !output) return fail(AQLM_B200_ERR_SHAPE, "NULL pointer");
  if (dtype != AQLM_B200_F16 && dtype != AQLM_B200_BF16) return fail(AQLM_B200_ERR_DTYPE, "dtype must be f16/bf16");
  const int64_t n = batch * out_features;
  if (n <= 0) return AQLM_B200_OK;
  if (n > c->max_elems || (out_features & 3)) return fail(AQLM_B200_ERR_SHAPE, "allreduce: %lld elements exceed the communicator's %lld (or out_features %% 4 != 0)", (long long)n, c->max_elems);
  const DeviceInfo* di = device_info();
  if (!di) return (int)(strstr(tls_error_buf(), "sm_100a") ? AQLM_B200_ERR_ARCH : AQLM_B200_ERR_CUDA);
  PeerParams p;
  for (int r = 0; r < kPeerMaxWorld; ++r) p.peer_base[r] = r < c->world ? c->peer_base[r] : nullptr;
  p.local = partial;
  p.scales = scales;
  p.bias = bias;
  p.y = output;
  p.step = c->local_state;
  p.tickets = c->local_state + 1;
  p.max_elems = c->max_elems;
  p.n = (int)n;
  p.out_features = (int)out_features;
  p.rank = c->rank;
  p.world = c->world;
  int grid = (int)((n / 4 + kPeerThreads - 1) / kPeerThreads);
  if (grid > kPeerMaxCtas) grid = kPeerMaxCtas;  // one flag per (source rank, CTA slice); every rank derives the same grid from n
  if (grid < 1) grid = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kPeerThreads);
  cfg.stream = reinterpret_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = tun().pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (dtype == AQLM_B200_F16) AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, peer_allreduce_epilogue_kernel<__half>, p));
  else AQLM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, peer_allreduce_epilogue_kernel<__nv_bfloat16>, p));
  count_launch();
  return AQLM_B200_OK;
}

int aqlm_b200_matmat_allreduce(aqlm_b200_comm* c, const aqlm_b200_weight_t* w, const int64_t* seg_rows, int n_seg,
                               const void* input, void* output, int64_t batch, void* stream) {
  if (!c) return fail(AQLM_B200_ERR_SHAPE, "communicator is NULL");
  int rc = validate(w, true);
  if (rc) return rc;
  if (w->num_codebooks != 1 || w->nbits_per_codebook != 16 || w->in_group_size != 8)
    return fail(AQLM_B200_ERR_UNSUPPORTED, "fused GEMV + exchange is implemented for the 1x16 (in_group 8) scheme");
  if (batch < 1 || batch > 8) return fail(AQLM_B200_ERR_UNSUPPORTED, "fused GEMV + exchange takes 1..8 batch rows");
  if (n_seg < 1 || n_seg > 4 || (n_seg > 1 && !seg_rows)) return fail(AQLM_B200_ERR_SHAPE, "1..4 segments");
  if (!input || !output) return fail(AQLM_B200_ERR_SHAPE, "input/output pointer is NULL");
  if ((w->out_features & 3) || batch * w->out_features > c->max_elems)
    return fail(AQLM_B200_ERR_SHAPE, "fused exchange: out_features %% 4 != 0 or batch*out_features exceeds the communicator's %lld",
                c->max_elems);
  const size_t row_bytes = (size_t)(w->in_features / 8) * 2;
  if (row_bytes % 16 != 0 || (reinterpret_cast<uintptr_t>(w->codes) & 15) || (reinterpret_cast<uintptr_t>(input) & 15))
    return fail(AQLM_B200_ERR_UNSUPPORTED, "fused exchange needs 16-byte aligned code rows and input");
  const DeviceInfo* di = device_info();
  if (!di) return (int)(strstr(tls_error_buf(), "sm_100a") ? AQLM_B200_ERR_ARCH : AQLM_B200_ERR_CUDA);
  GemvParams p;
  p.codes = w->codes;
  p.codebooks = w->codebooks;
  p.scales = w->scales;
  p.bias = w->bias;
  p.x = input;
  p.y = output;
  p.out_features = (int)w->out_features;
  p.in_features = (int)w->in_features;
  p.in_groups = (int)(w->in_features / 8);
  p.nbits = 16;
  p.num_codebooks = 1;
  p.batch = (int)batch;
  p.partial_f32 = 0;
  p.n_seg = n_seg;
  p.row_block = 0;
  int64_t acc = 0;
  for (int i = 0; i < 4; ++i) {
    if (i < n_seg) acc += (n_seg > 1 ? seg_rows[i] : w->out_features);
    p.seg_end[i] = (int)acc;
  }
  if (acc != w->out_features) return fail(AQLM_B200_ERR_SHAPE, "segment rows do not add up to out_features");
  GemvPeer pc;
  for (int r = 0; r < 16; ++r) pc.peer_base[r] = r < c->world ? c->peer_base[r] : nullptr;
  pc.step = c->local_state;
  pc.tickets = c->local_state + 1;
  pc.max_elems = c->max_elems;
  pc.rank = c->rank;
  pc.world = c->world;
  pc.ll_offset = (long long)kPeerFlagBytes + (long long)2 * c->world * c->max_elems * (long long)sizeof(float);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int bt = batch == 1 ? 1 : (batch == 2 ? 2 : (batch <= 4 ? 4 : 8));
#define AQLM_PEER(T)                                                                                    \
  (bt == 1 ? launch_1x16_peer<T, 1>(p, pc, di, st) : bt == 2 ? launch_1x16_peer<T, 2>(p, pc, di, st) \
           : bt == 4 ? launch_1x16_peer<T, 4>(p, pc, di, st) : launch_1x16_peer<T, 8>(p, pc, di, st))
  if (w->dtype == AQLM_B200_F16) return AQLM_PEER(__half);
  return AQLM_PEER(__nv_bfloat16);
#undef AQLM_PEER
}

int aqlm_b200_matmat_host(const aqlm_b200_weight_t* w, const void* input_host, void* output_host, void* input_dev,
                          void* output_dev, int64_t batch, void* stream) {
  int rc = validate(w, true);
  if (rc) return rc;
  if (!input_host || !output_host || !input_dev || !output_dev) return fail(AQLM_B200_ERR_SHAPE, "NULL buffer");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  AQLM_CUDA_CHECK(cudaMemcpyAsync(input_dev, input_host, (size_t)batch * w->in_features * 2, cudaMemcpyHostToDevice, st));
  rc = aqlm_b200_matmat_ex(w, input_dev, output_dev, batch, 0, stream);
  if (rc) return rc;
  AQLM_CUDA_CHECK(cudaMemcpyAsync(output_host, output_dev, (size_t)batch * w->out_features * 2, cudaMemcpyDeviceToHost, st));
  AQLM_CUDA_CHECK(cudaStreamSynchronize(st));
  return AQLM_B200_OK;
}

// ---- flat wrappers ------------------------------------------------------------------------------
#define AQLM_FLAT_MATMAT(NAME, K, NBITS, GEXPR, FN)                                                               \
  aqlm_b200_weight_t w = make_weight(codes, codebooks, scales, bias, in_features, out_features, K, NBITS, GEXPR, dtype); \
  return FN(&w, input, output, batch, stream)

int aqlm_b200_code1x16_matmat(const void* input, const void* codes, const void* codebooks, const void* scales,
                              const void* bias, void* output, int64_t batch, int64_t in_features,
                              int64_t out_features, int32_t in_group_size, int32_t dtype, void* stream) {
  AQLM_FLAT_MATMAT(code1x16_matmat, 1, 16, in_group_size, aqlm_b200_matmat);
}
int aqlm_b200_code2x8_matmat(const void* input, const void* codes, const void* codebooks, const void* scales,
                             const void* bias, void* output, int64_t batch, int64_t in_features,
                             int64_t out_features, int32_t dtype, void* stream) {
  AQLM_FLAT_MATMAT(code2x8_matmat, 2, 8, 8, aqlm_b200_matmat);
}
int aqlm_b200_code1x8_matmat(const void* input, const void* codes, const void* codebooks, const void* scales,
                             const void* bias, void* output, int64_t batch, int64_t in_features,
                             int64_t out_features, int32_t dtype, void* stream) {
  AQLM_FLAT_MATMAT(code1x8_matmat, 1, 8, 8, aqlm_b200_matmat);
}
int aqlm_b200_code1x16_matmat_dequant(const void* input, const void* codes, const void* codebooks,
                                      const void* scales, const void* bias, void* output, int64_t batch,
                                      int64_t in_features, int64_t out_features, int32_t in_group_size,
                                      int32_t dtype, void* stream) {
  AQLM_FLAT_MATMAT(code1x16_matmat_dequant, 1, 16, in_group_size, aqlm_b200_matmat_dequant);
}
int aqlm_b200_code2x8_matmat_dequant(const void* input, const void* codes, const void* codebooks,
                                     const void* scales, const void* bias, void* output, int64_t batch,
                                     int64_t in_features, int64_t out_features, int32_t dtype, void* stream) {
  AQLM_FLAT_MATMAT(code2x8_matmat_dequant, 2, 8, 8, aqlm_b200_matmat_dequant);
}
int aqlm_b200_code1x8_matmat_dequant(const void* input, const void* codes, const void* codebooks,
                                     const void* scales, const void* bias, void* output, int64_t batch,
                                     int64_t in_features, int64_t out_features, int32_t dtype, void* stream) {
  AQLM_FLAT_MATMAT(code1x8_matmat_dequant, 1, 8, 8, aqlm_b200_matmat_dequant);
}
#undef AQLM_FLAT_MATMAT

int aqlm_b200_code1x16_dequant(const void* codes, const void* codebooks, const void* scales, void* weight_out,
                               int64_t in_features, int64_t out_features, int32_t in_group_size, int32_t dtype,
                               void* stream) {
  aqlm_b200_weight_t w = make_weight(codes, codebooks, scales, nullptr, in_features, out_features, 1, 16, in_group_size, dtype);
  return aqlm_b200_dequant(&w, weight_out, 1, stream);
}
int aqlm_b200_code2x8_dequant(const void* codes, const void* codebooks, const void* scales, void* weight_out,
                              int64_t in_features, int64_t out_features, int32_t dtype, void* stream) {
  aqlm_b200_weight_t w = make_weight(codes, codebooks, scales, nullptr, in_features, out_features, 2, 8, 8, dtype);
  return aqlm_b200_dequant(&w, weight_out, 1, stream);
}
int aqlm_b200_code1x8_dequant(const void* codes, const void* codebooks, const void* scales, void* weight_out,
                              int64_t in_features, int64_t out_features, int32_t dtype, void* stream) {
  aqlm_b200_weight_t w = make_weight(codes, codebooks, scales, nullptr, in_features, out_features, 1, 8, 8, dtype);
  return aqlm_b200_dequant(&w, weight_out, 1, stream);
}

}  // extern "C"
