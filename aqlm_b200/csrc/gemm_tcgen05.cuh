// Fused additive-dequant + tensor-core GEMM for batch > 6:  Y[bs, out] = X[bs, in] . W^T, W never touches HBM.
//
// Replaces code{1x16,2x8,1x8}_matmat_dequant (reference cuda_kernel.cpp:249-301, 450-484, 615-649), which
// materialise W [out,in] in HBM with a Dequant kernel (cuda_kernel.cu:98-142) and then call cuBLAS.
//
// B200 design (tcgen05 / TMEM / TMA, hand-written PTX):
//   D[128 x N] (fp32, TMEM)  +=  A[128 x 64] (smem, K-major, SWIZZLE_128B)  x  B[N x 64]^T (smem, K-major, SWIZZLE_128B)
//   A = a 128-row tile of W, produced ON CHIP: producer warps read packed codes from a TMA-staged code tile,
//       gather the codebook vectors (L2/L1) and write them straight into the swizzled UMMA layout;
//   B = the activation tile X[n0:n0+N, k0:k0+64], TMA-loaded (OOB rows zero-filled, so any batch works);
//   one elected thread issues tcgen05.mma (128 x N x 16, kind::f16, fp16 or bf16 operands, fp32 accumulate),
//   tcgen05.commit releases smem stages through mbarriers; the epilogue reads TMEM with tcgen05.ld and
//   applies scale + bias.
// Grid = (M tiles, K splits, N tiles).  The kernel is bound by the per-SM codebook-gather rate (see
// profiles/), so the K dimension is split to put every SM to work; split partials go through an fp32
// workspace and the LAST-arriving CTA of each tile reduces them in a fixed order (deterministic).
#pragma once

#include <cuda.h>

#include "common.cuh"

namespace aqlm_b200 {

constexpr int kGemmProducerWarps = 16;
constexpr int kGemmThreads = 128 + 32 * kGemmProducerWarps;  // warps 0-3: TMA / MMA / TMEM-alloc, then epilogue; warps 4-19: dequant producers
// V2 producer mapping: one 4-warp group per smem stage (at most 4 stages), each group owns every S-th k-block entirely
constexpr int kGemmThreadsV2 = 128 + 32 * 4 * 4;
constexpr int kGemmBlockM = 128;
constexpr int kGemmBlockK = 64;          // 64 halves = 128 bytes = one swizzle row
constexpr int kCodeTileBytes = 128;      // bytes of codes per row per code tile (TMA box inner extent)
constexpr int kCodeTileStages = 2;

struct GemmParams {
  const void* codebooks;
  const void* scales;
  const void* bias;
  void* y;              // [batch, out_features]
  float* ws_partials;   // [m_tiles][n_tiles][ksplit][N][128] fp32 (ksplit > 1)
  unsigned int* ws_counters;  // [m_tiles * n_tiles], zero on entry
  int out_features;
  int batch;
  int nbits;
  int total_kblocks;    // in_features / 64
  int ksplit;
  int n_tile;           // N of the MMA (multiple of 16, <= 256)
  int stages;
  int cluster;          // CTAs per cluster along M that share (multicast) the X tiles
  int a_stages;         // ATMEM: number of 32-column A stages in tensor memory (decoupled from the X stages in smem)
  int groups;           // V2: producer groups of 4 warps (coupled form: = stages)
  int tile_m;           // output rows per CTA tile (<= 128): ragged tile heights balance the grid (e.g. 97 rows -> 148 tiles of 14336)
  int gather_mode;      // 0: ld.global.nc (L1 allocate), 1: ld.global.cg, 3: nc.L1::no_allocate
  int debug;            // bit0: read codes from global instead of the TMA code tile; bit1: no producer run-ahead
  const void* codes;    // (debug bit0)
  long long row_bytes;  // (debug bit0)
};

// ---- PTX wrappers -----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3}], [%4], %5;"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// one lane of a converged warp (uniform control flow around it lets ptxas keep descriptors in uniform registers)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// UMMA shared-memory descriptor, K-major, SWIZZLE_128B: start>>4 | LBO(=1)<<16 | SBO(1024 B >>4)<<32 | version 1<<46 | layout 2<<61
__device__ __forceinline__ uint64_t umma_desc_k128(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}
// UMMA instruction descriptor, kind::f16: D=f32, A/B = f16 (0) or bf16 (1), both K-major, M=128, N=n
__device__ __forceinline__ uint32_t umma_idesc(int ab_format, int n) {
  return (1u << 4) | ((uint32_t)ab_format << 7) | ((uint32_t)ab_format << 10) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(kGemmBlockM >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc),
      "r"(accumulate) : "memory");
}
// same with the A operand in tensor memory (lane = row, 32-bit column c holds K elements 2c, 2c+1)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc),
      "r"(accumulate) : "memory");
}
// 32 lanes x 32 columns: thread t of the warp writes r[0..31] to TMEM lane (32*(warp%4) + t), columns [col, col+32)
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
        "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
        "r"(r[30]), "r"(r[31])
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory carve-up (all offsets from a 1024-byte aligned base)
struct GemmSmem {
  uint32_t a, b, codes, full, empty, afull, aempty, cfull, cempty, tfull, tmem_slot, flag;
  size_t total;
};
__host__ __device__ inline GemmSmem gemm_smem_layout(int stages, int n_tile, bool a_in_tmem = false) {
  GemmSmem L;
  size_t off = 0;
  L.a = (uint32_t)off; off += a_in_tmem ? 0 : (size_t)stages * kGemmBlockM * 128;
  L.b = (uint32_t)off; off += (size_t)stages * n_tile * 128;
  off = (off + 1023) & ~(size_t)1023;
  L.codes = (uint32_t)off; off += (size_t)kCodeTileStages * kGemmBlockM * kCodeTileBytes;
  L.full = (uint32_t)off; off += 8 * 8;
  L.empty = (uint32_t)off; off += 8 * 8;
  L.afull = (uint32_t)off; off += 8 * 8;
  L.aempty = (uint32_t)off; off += 8 * 8;
  L.cfull = (uint32_t)off; off += 8 * kCodeTileStages;
  L.cempty = (uint32_t)off; off += 8 * kCodeTileStages;
  L.tfull = (uint32_t)off; off += 8;
  L.tmem_slot = (uint32_t)off; off += 4;
  L.flag = (uint32_t)off; off += 4;
  L.total = off + 1024;  // slack for manual 1024-byte alignment of the dynamic smem base
  return L;
}

// K = codebooks per group, CODE_BYTES = 1|2, GS = in_group_size (8, or 16 for 1x16 in the V2 + ATMEM form only).
// bytes of codes per row per 64-wide k-block: GB = (64 / GS) groups * K * CODE_BYTES
// GS = 16: a codebook entry is 16 halves = one 32-byte sector, fetched as ONE 256-bit request (ld_gather_v8), so a
// k-block costs 4 gather requests per row instead of 8; the entry fills 8 of the row's 32 TMEM columns unchanged.
// ATMEM (needs the V2 producer mapping, thread <-> row): the dequantized A tile is written to TENSOR MEMORY with tcgen05.st
// and the MMA takes A from TMEM.  Shared memory then carries only the X stages (and the code tiles): per k-block the
// shared-memory traffic drops from 96 KB (A write + A read + X write + X read at N=256) to 64 KB -- at 128 B/clk that was
// 768 clk against 512 clk of MMA, i.e. the SS form was shared-memory bound before any gather -- and the L1 the gathers
// run against grows by the 48 KB the A stages took.
template <typename T, int K, int CODE_BYTES, bool V2, bool ATMEM = false, int GS = 8>
__global__ void __launch_bounds__(V2 ? kGemmThreadsV2 : kGemmThreads, 1)
gemm_dequant_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_codes, const GemmParams p) {
  static_assert(!ATMEM || V2, "A-in-TMEM needs the thread <-> row producer mapping");
  static_assert(GS == 8 || (GS == 16 && K == 1 && CODE_BYTES == 2 && V2 && ATMEM), "in_group_size 16: 1x16, V2 + ATMEM only");
  constexpr int NTHREADS = V2 ? kGemmThreadsV2 : kGemmThreads;
  constexpr int GB = (kGemmBlockK / GS) * K * CODE_BYTES;  // code bytes per row per k-block
  constexpr int KB_PER_CTILE = kCodeTileBytes / GB;  // k-blocks covered by one code tile
  static_assert(KB_PER_CTILE >= 1, "scheme too wide for the code tile");
  extern __shared__ uint8_t smem_dyn[];
  const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
  uint8_t* gbase = smem_dyn + (base - smem_u32(smem_dyn));
  const GemmSmem L = gemm_smem_layout(p.stages, p.n_tile, ATMEM);
  const int S = p.stages;
  const int TM = p.tile_m;
  const int N = p.n_tile;
  const int C = p.cluster;
  const uint32_t crank = C > 1 ? cluster_ctarank() : 0u;
  const uint16_t cmask = (uint16_t)((1u << C) - 1u);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x, split = blockIdx.y, n_blk = blockIdx.z;
  const int m0 = m_tile * TM, n0 = n_blk * N;
  // PDL: the next kernel of the stream may be dispatched as soon as SM resources free up (no launch gap).  Everything this
  // kernel does before griddep_wait() touches WEIGHTS only (code tiles, codebook gathers); the X tiles are read and y /
  // the workspace written after it.
  griddep_launch_dependents();
  // k-block range of this split (balanced, contiguous)
  const int kb0 = (int)(((long long)p.total_kblocks * split) / p.ksplit);
  const int kb1 = (int)(((long long)p.total_kblocks * (split + 1)) / p.ksplit);
  const int nkb = kb1 - kb0;
  // code tiles: aligned to KB_PER_CTILE boundaries in absolute k-block index
  const int ct0 = kb0 / KB_PER_CTILE;
  const int ct1 = (kb1 + KB_PER_CTILE - 1) / KB_PER_CTILE;

  auto full_bar = [&](int s) { return base + L.full + 8 * s; };
  auto empty_bar = [&](int s) { return base + L.empty + 8 * s; };
  auto cfull_bar = [&](int s) { return base + L.cfull + 8 * s; };
  auto cempty_bar = [&](int s) { return base + L.cempty + 8 * s; };
  // ATMEM: the A stages (tensor memory) have their own full/empty barriers, decoupled from the X stages (shared memory):
  // the dequant producers run up to SA k-blocks ahead of the MMA no matter how late an X tile lands
  auto afull_bar = [&](int s) { return base + L.afull + 8 * s; };
  auto aempty_bar = [&](int s) { return base + L.aempty + 8 * s; };
  const int SA = ATMEM ? p.a_stages : S;
  const int G = V2 ? p.groups : 0;  // producer groups
  const uint32_t tfull_bar = base + L.tfull;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gbase + L.tmem_slot);

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      // X stage: the TMA thread's expect_tx arrival (+ the stage's producer warps when A shares the stage)
      mbar_init(full_bar(s), ATMEM ? 1 : (V2 ? 4 : kGemmProducerWarps) + 1);
      mbar_init(empty_bar(s), C);                      // tcgen05.commit of every CTA in the cluster
    }
    if constexpr (ATMEM) {
      for (int s = 0; s < SA; ++s) {
        mbar_init(afull_bar(s), 4);   // the 4 warps of the group that owns the k-block
        mbar_init(aempty_bar(s), 1);  // tcgen05.commit
      }
    }
    for (int s = 0; s < kCodeTileStages; ++s) {
      mbar_init(cfull_bar(s), 1);
      mbar_init(cempty_bar(s), V2 ? 4 * G : kGemmProducerWarps);
    }
    mbar_init(tfull_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // accumulator: columns [0, N); with ATMEM the A stages follow at a 32-column aligned offset, 32 columns per stage
  const uint32_t a_col0 = (uint32_t)((N + 31) & ~31);
  uint32_t tmem_cols = 32;
  while (tmem_cols < (ATMEM ? a_col0 + 32u * (uint32_t)p.a_stages : (uint32_t)N)) tmem_cols <<= 1;
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(base + L.tmem_slot), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (C > 1) cluster_sync_all();  // peers' barriers are initialised before anyone multicasts into them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (nkb > 0) {
    if (warp == 0) {
      // ===== TMA producer (whole warp, one elected lane issues): code tiles (one per KB_PER_CTILE k-blocks) and one X
      //       tile per k-block =====
      int ct_loaded = ct0;
      auto load_ctile = [&](int ct) {
        const int cs = (ct - ct0) % kCodeTileStages;
        const int it = (ct - ct0) / kCodeTileStages;
        if (it > 0) mbar_wait(cempty_bar(cs), (it - 1) & 1);  // every producer warp released the previous tenant
        if (elect_one()) {
          mbar_expect_tx(cfull_bar(cs), (uint32_t)TM * kCodeTileBytes);  // the TMA box is tile_m rows tall
          tma_load_2d(base + L.codes + cs * kGemmBlockM * kCodeTileBytes, &tmap_codes, ct * kCodeTileBytes, m0, cfull_bar(cs));
        }
        __syncwarp();
      };
      load_ctile(ct_loaded++);
      griddep_wait();  // X is produced by the previous kernel
      int s = 0, it = 0;  // X stage and its use count (no runtime division in this loop)
      for (int i = 0; i < nkb; ++i) {
        if (it > 0) mbar_wait(empty_bar(s), (it - 1) & 1);
        if (elect_one()) {
          if (p.debug & 4) {  // experiment: no X traffic (B tile keeps whatever it holds)
            mbar_arrive(full_bar(s));
          } else if (C == 1) {
            mbar_expect_tx(full_bar(s), (uint32_t)N * 128);
            tma_load_2d(base + L.b + s * N * 128, &tmap_x, (kb0 + i) * kGemmBlockK, n0, full_bar(s));
          } else {
            mbar_expect_tx(full_bar(s), (uint32_t)N * 128);  // all C slices land here
            // this CTA fetches rows [crank*N/C, (crank+1)*N/C) of the X tile and multicasts them to the whole cluster;
            // empty_bar(s) (count C) guarantees every CTA of the cluster has released stage s
            const int rows = N / C;
            tma_load_2d_mc(base + L.b + s * N * 128 + crank * rows * 128, &tmap_x, (kb0 + i) * kGemmBlockK, n0 + crank * rows,
                           full_bar(s), cmask);
          }
        }
        __syncwarp();
        // prefetch the NEXT code tile while the producers work on the current one
        const int ct_cur = (kb0 + i) / KB_PER_CTILE;
        if (ct_loaded < ct1 && ct_loaded <= ct_cur + 1) load_ctile(ct_loaded++);
        if (++s == S) { s = 0; ++it; }
      }
    } else if (warp == 1) {
      // ===== MMA issuer: the WHOLE warp runs the loop (uniform barrier waits, incremental stage counters), one elected
      //       lane issues.  A lane-0-only loop compiled to ~150 dependent scalar instructions per k-block (runtime
      //       modulo, R2UR moves, an election loop around every UTCHMMA): ~1000 clk per k-block against 512 clk of MMA --
      //       with gathers AND X loads switched off the kernel still took 44.6 us (profiles/r02/probe_gemm_e1.jsonl). =====
      const uint32_t idesc = umma_idesc(sizeof(T) == 2 && DT<T>::is_bf16 ? 1 : 0, N);
      int s = 0, sa = 0;
      uint32_t ph_b = 0, ph_a = 0;
      for (int i = 0; i < nkb; ++i) {
        mbar_wait(full_bar(s), ph_b);
        if constexpr (ATMEM) mbar_wait(afull_bar(sa), ph_a);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_addr = base + L.a + s * kGemmBlockM * 128;
          const uint32_t b_addr = base + L.b + s * N * 128;
          const uint64_t bdesc = umma_desc_k128(b_addr);
#pragma unroll
          for (int k = 0; k < kGemmBlockK / 16; ++k) {
            // advancing 16 K-elements = 32 bytes = +2 in the descriptor's (address >> 4) field
            if constexpr (ATMEM)
              umma_f16_ts(tmem_base, tmem_base + a_col0 + (uint32_t)(sa * 32 + k * 8), bdesc + (uint64_t)(2 * k), idesc, (i | k) ? 1u : 0u);
            else
              umma_f16(tmem_base, umma_desc_k128(a_addr) + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (i | k) ? 1u : 0u);
          }
          // frees this smem stage (in every CTA of the cluster) when the MMAs above have read it
          if (C == 1) umma_commit(empty_bar(s));
          else umma_commit_mc(empty_bar(s), cmask);
          if constexpr (ATMEM) umma_commit(aempty_bar(sa));  // and the A stage (this CTA's tensor memory only)
        }
        __syncwarp();
        if (++s == S) { s = 0; ph_b ^= 1u; }
        if (++sa == SA) { sa = 0; ph_a ^= 1u; }
      }
      if (elect_one()) umma_commit(tfull_bar);  // accumulator complete
      __syncwarp();
    } else if (warp >= 4) {
      if constexpr (V2) {
        // ===== V2 dequant producers: group g (4 warps, thread <-> row) owns stage g and every S-th k-block =====
        const int pw = warp - 4;
        const int g = pw >> 2;
        if (g < G) {
          const int row = (pw & 3) * 32 + lane;
          const bool active = row < TM;  // rows past the (ragged) tile height: no gathers, nothing to write
          const uint4* gcb = reinterpret_cast<const uint4*>(p.codebooks);
          constexpr int CWN = GB / 4 > 0 ? GB / 4 : 1;  // 32-bit words of codes per row per k-block
          constexpr bool INREG = (K <= 2);               // gather in issue() and hold the vectors in registers
          constexpr bool DB = (K == 1);                  // double-buffer across k-blocks
          int next_release = ct0;
          // arrive on cempty for every code tile in [next_release, upto): each producer warp arrives exactly once per
          // tile, in order, after the tile was loaded (phase bookkeeping) and after its own reads of it were consumed
          auto release_upto = [&](int upto) {
            for (; next_release < upto; ++next_release) {
              const int cs = (next_release - ct0) % kCodeTileStages, cit = (next_release - ct0) / kCodeTileStages;
              mbar_wait(cfull_bar(cs), cit & 1);
              __syncwarp();
              if (lane == 0) mbar_arrive(cempty_bar(cs));
            }
          };
          auto load_cw = [&](int i, uint32_t (&cw)[CWN]) {
            const int kb = kb0 + i;
            const int ct = kb / KB_PER_CTILE, st_in = kb % KB_PER_CTILE;
            release_upto(ct);
            const int cs = (ct - ct0) % kCodeTileStages, cit = (ct - ct0) / kCodeTileStages;
            mbar_wait(cfull_bar(cs), cit & 1);
            const uint8_t* crow = gbase + L.codes + cs * kGemmBlockM * kCodeTileBytes + row * 128;
            if (!active) {
#pragma unroll
              for (int q = 0; q < CWN; ++q) cw[q] = 0u;
            } else if constexpr (GB >= 16) {
#pragma unroll
              for (int q = 0; q < GB / 16; ++q) {
                const int chunk = ((st_in * GB) / 16 + q) ^ (row & 7);
                const uint4 v = *reinterpret_cast<const uint4*>(crow + (chunk << 4));
                cw[q * 4 + 0] = v.x; cw[q * 4 + 1] = v.y; cw[q * 4 + 2] = v.z; cw[q * 4 + 3] = v.w;
              }
            } else {  // GB == 8 (1x8; 1x16 with GS = 16)
              const int lb = st_in * GB;
              const int chunk = (lb >> 4) ^ (row & 7);
              const uint2 v = *reinterpret_cast<const uint2*>(crow + (chunk << 4) + (lb & 15));
              cw[0] = v.x; cw[1] = v.y;
            }
          };
          auto code_at = [&](const uint32_t (&cw)[CWN], int idx) -> uint32_t {
            if constexpr (CODE_BYTES == 2) return (cw[idx >> 1] >> ((idx & 1) * 16)) & 0xffffu;
            else return (cw[idx >> 2] >> ((idx & 3) * 8)) & 0xffu;
          };
          auto gather_all = [&](const uint32_t (&cw)[CWN], uint4 (&wv)[8][INREG ? K : 1]) {
            if constexpr (GS == 16) {
              // group q = 16 halves = TMEM columns [8q, 8q+8): one 256-bit gather into wv[2q] (lo) and wv[2q+1] (hi)
              if (active && !(p.debug & 8)) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const uint4* gp = gcb + 2 * (size_t)code_at(cw, q);
                  if (p.gather_mode == 1) ld_gather_v8<1>(gp, wv[2 * q][0], wv[2 * q + 1][0]);
                  else ld_gather_v8<0>(gp, wv[2 * q][0], wv[2 * q + 1][0]);
                }
              } else {
#pragma unroll
                for (int e = 0; e < 8; ++e) wv[e][0] = make_uint4(0u, 0u, 0u, 0u);
              }
            } else if constexpr (INREG) {
              if (active && !(p.debug & 8)) {
#pragma unroll
                for (int e = 0; e < 8; ++e)
#pragma unroll
                  for (int k = 0; k < K; ++k) {
                    const uint4* gp = gcb + (((size_t)k << p.nbits) + code_at(cw, e * K + k));
                    if (p.gather_mode == 1) wv[e][k] = ld_gather_v4<1>(gp);
                    else wv[e][k] = ld_gather_v4<0>(gp);
                  }
              } else {
#pragma unroll
                for (int e = 0; e < 8; ++e)
#pragma unroll
                  for (int k = 0; k < K; ++k) wv[e][k] = make_uint4(0u, 0u, 0u, 0u);
              }
            }
          };
          // this group's k-blocks are g, g+G, g+2G, ...: their A stage and use count advance incrementally
          const int NSTG = ATMEM ? SA : S;
          int st_next = g % NSTG, it_next = g / NSTG;
          auto commit = [&](int i, const uint32_t (&cw)[CWN], uint4 (&wv)[8][INREG ? K : 1]) {
            (void)i;
            const int s = st_next, it = it_next;
            st_next += G;
            while (st_next >= NSTG) { st_next -= NSTG; ++it_next; }
            if (it > 0) mbar_wait(ATMEM ? aempty_bar(s) : empty_bar(s), (it - 1) & 1);
            uint8_t* arow = gbase + L.a + s * kGemmBlockM * 128 + row * 128;
            uint32_t areg[32];  // ATMEM: the row's 64 halves in K order (= the TMEM column order)
            if constexpr (ATMEM) tc_fence_after();  // the stage's previous reader (MMA) is ordered before these writes
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              uint4 v;
              if constexpr (K == 1) {
                v = wv[e][0];
              } else {
                float f[8];
                if constexpr (INREG) {
                  unpack8<T>(wv[e][0], f);
#pragma unroll
                  for (int k = 1; k < K; ++k) accum8<T>(wv[e][k], f);
                } else if (active) {  // many codebooks: gather group by group (the 4-32 KiB codebooks are L1-resident)
                  uint4 t[K];
#pragma unroll
                  for (int k = 0; k < K; ++k) t[k] = ld_gather_v4<0>(gcb + (((size_t)k << p.nbits) + code_at(cw, e * K + k)));
                  unpack8<T>(t[0], f);
#pragma unroll
                  for (int k = 1; k < K; ++k) accum8<T>(t[k], f);
                } else {
#pragma unroll
                  for (int q = 0; q < 8; ++q) f[q] = 0.f;
                }
                v.x = DT<T>::pack2(f[0], f[1]); v.y = DT<T>::pack2(f[2], f[3]);
                v.z = DT<T>::pack2(f[4], f[5]); v.w = DT<T>::pack2(f[6], f[7]);
              }
              if constexpr (ATMEM) {
                areg[4 * e + 0] = v.x; areg[4 * e + 1] = v.y; areg[4 * e + 2] = v.z; areg[4 * e + 3] = v.w;
              } else {
                if (active) *reinterpret_cast<uint4*>(arow + ((e ^ (row & 7)) << 4)) = v;
              }
            }
            if constexpr (ATMEM) {
              // warp-collective store of 32 rows x 32 columns into this warp's TMEM quadrant, then make it visible to the
              // MMA thread: wait::st -> fence::before_thread_sync -> mbarrier arrive
              tmem_st_32x32b_x32(tmem_base + ((uint32_t)((pw & 3) * 32) << 16) + a_col0 + (uint32_t)(s * 32), areg);
              tc_fence_before();
            } else {
              fence_proxy_async();
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(ATMEM ? afull_bar(s) : full_bar(s));
          };
          if constexpr (DB) {
            uint32_t ca[CWN], cb[CWN];
            uint4 wa[8][K], wb[8][K];
            int i = g;
            if (i < nkb) { load_cw(i, ca); gather_all(ca, wa); }
            for (; i < nkb; i += 2 * G) {
              if (i + G < nkb) { load_cw(i + G, cb); gather_all(cb, wb); }
              commit(i, ca, wa);
              if (i + G < nkb) {
                if (i + 2 * G < nkb) { load_cw(i + 2 * G, ca); gather_all(ca, wa); }
                commit(i + G, cb, wb);
              }
            }
          } else {
            uint32_t ca[CWN];
            uint4 wa[8][INREG ? K : 1];
            for (int i = g; i < nkb; i += G) {
              load_cw(i, ca);
              gather_all(ca, wa);
              commit(i, ca, wa);
            }
          }
          release_upto(ct1);
        }
      } else {
      // ===== dequant producers: 512 threads, thread -> (row, quarter of the 8 groups of a k-block) =====
      // Software-pipelined: the gathers of k-block i+1 are in flight while k-block i is written to smem.
      const int pt = threadIdx.x - 128;
      const int row = pt >> 2, gq = pt & 3;
      const bool active = row < TM;  // rows past the (ragged) tile height: no gathers, nothing to write
      const uint4* gcb = reinterpret_cast<const uint4*>(p.codebooks);
      constexpr int CB2 = 2 * K * CODE_BYTES;  // code bytes of this thread's 2 groups
      constexpr int CW = (CB2 + 3) / 4;        // 32-bit words holding them
      constexpr int D = (K == 1) ? 4 : (K == 2 ? 2 : 1);  // k-blocks of gathers held in registers ahead of the writes

      // codes of k-block index i (relative) -> issue the 2*K gathers into wv
      auto issue = [&](int i, uint4 (&wv)[2][K]) {
        const int kb = kb0 + i;
        const int ct = kb / KB_PER_CTILE, st_in = kb % KB_PER_CTILE;
        const int cs = (ct - ct0) % kCodeTileStages, cit = (ct - ct0) / kCodeTileStages;
        mbar_wait(cfull_bar(cs), cit & 1);
        uint32_t cw[CW];
        if (!active) {
#pragma unroll
          for (int q = 0; q < CW; ++q) cw[q] = 0u;
        } else if (p.debug & 1) {
          const uint8_t* src = reinterpret_cast<const uint8_t*>(p.codes) + (size_t)(m0 + row) * p.row_bytes + (size_t)kb * GB + gq * CB2;
#pragma unroll
          for (int q = 0; q < CW; ++q) {
            uint32_t v = 0;
            if (m0 + row < p.out_features) {
              if constexpr (CB2 >= 4) v = reinterpret_cast<const uint32_t*>(src)[q];
              else v = reinterpret_cast<const uint16_t*>(src)[0];
            }
            cw[q] = v;
          }
        } else {
          // logical byte offset inside the 128-byte code row -> physical (SWIZZLE_128B: 16-byte chunk ^= row & 7)
          const int lbyte = st_in * GB + gq * CB2;
          const uint8_t* crow = gbase + L.codes + cs * kGemmBlockM * kCodeTileBytes + row * 128;
          if constexpr (CB2 >= 16) {
            const int chunk = (lbyte >> 4) ^ (row & 7);
            const uint4 v = *reinterpret_cast<const uint4*>(crow + (chunk << 4));
            cw[0] = v.x; cw[1] = v.y; cw[2] = v.z; cw[3] = v.w;
          } else {
            const int chunk = (lbyte >> 4) ^ (row & 7);
            const uint8_t* src = crow + (chunk << 4) + (lbyte & 15);
            if constexpr (CB2 == 8) { const uint2 v = *reinterpret_cast<const uint2*>(src); cw[0] = v.x; cw[1] = v.y; }
            else if constexpr (CB2 == 4) cw[0] = *reinterpret_cast<const uint32_t*>(src);
            else cw[0] = *reinterpret_cast<const uint16_t*>(src);
          }
        }
#pragma unroll
        for (int e = 0; e < 2; ++e) {
#pragma unroll
          for (int k = 0; k < K; ++k) {
            const int idx = e * K + k;
            uint32_t code;
            if constexpr (CODE_BYTES == 2) code = (cw[idx >> 1] >> ((idx & 1) * 16)) & 0xffffu;
            else code = (cw[idx >> 2] >> ((idx & 3) * 8)) & 0xffu;
            const uint4* gp = gcb + (((size_t)k << p.nbits) + code);
            if (!active || (p.debug & 8)) wv[e][k] = make_uint4(code, code, code, code);  // inactive row / experiment: no gathers
            else if (p.gather_mode == 1) wv[e][k] = ld_gather_v4<1>(gp);       // ld.global.cg (L2 only)
            else if (p.gather_mode == 3) wv[e][k] = ld_gather_v4<3>(gp);       // nc + L1::no_allocate
            else wv[e][k] = ld_gather_v4<0>(gp);
          }
        }
        // Release the code tile after its last k-block.  This MUST come after the gathers above were issued: their
        // addresses depend on the code registers, so the shared-memory loads of the codes have completed by now.
        // (Releasing right after issuing those loads lets the TMA refill the slot while they are still in flight.)
        if (st_in == KB_PER_CTILE - 1 || i == nkb - 1) {
          __syncwarp();
          if (lane == 0) mbar_arrive(cempty_bar(cs));
        }
      };
      // additive dequant + write the 2 groups of k-block i into the swizzled A stage, then signal the MMA thread
      auto commit = [&](int i, uint4 (&wv)[2][K]) {
        const int s = i % S, it = i / S;
        if (it > 0) mbar_wait(empty_bar(s), (it - 1) & 1);
        uint8_t* arow = gbase + L.a + s * kGemmBlockM * 128 + row * 128;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          uint4 v = wv[e][0];
          if constexpr (K > 1) {
            float f[8];
            unpack8<T>(wv[e][0], f);
#pragma unroll
            for (int k = 1; k < K; ++k) accum8<T>(wv[e][k], f);
            v.x = DT<T>::pack2(f[0], f[1]); v.y = DT<T>::pack2(f[2], f[3]);
            v.z = DT<T>::pack2(f[4], f[5]); v.w = DT<T>::pack2(f[6], f[7]);
          }
          const int j = gq * 2 + e;  // 16-byte chunk (= group) index inside the 128-byte K row
          if (active) *reinterpret_cast<uint4*>(arow + ((j ^ (row & 7)) << 4)) = v;
        }
        fence_proxy_async();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(full_bar(s));
      };
      // register ring of D k-blocks: the kernel is bound by gather LATENCY unless ~8+ gathers per thread are in flight
      // (ncu: long-scoreboard stalls dominate, L2/XBAR < 30% busy), so gathers run D k-blocks ahead of the smem writes.
      uint4 w[D][2][K];
#pragma unroll
      for (int d = 0; d < D; ++d)
        if (d < nkb) issue(d, w[d]);
      for (int i = 0; i < nkb; i += D) {
#pragma unroll
        for (int d = 0; d < D; ++d) {
          if (i + d < nkb) {
            commit(i + d, w[d]);
            if (i + d + D < nkb) issue(i + d + D, w[d]);
          }
        }
      }
      }
    }
  }

  // ===== epilogue: ALL warps (a warp may read the TMEM lanes 32*(warp%4)..+31, so the producer warps -- idle by now --
  //       take column chunks too: 5 warps per lane quadrant instead of 1), thread <-> TMEM lane <-> output row =====
  const size_t tile_id = (size_t)m_tile * gridDim.z + n_blk;
  T* y = reinterpret_cast<T*>(p.y);
  {
    __syncwarp();
    griddep_wait();  // before any global write (y, split-K partials): the previous kernel has completed
    constexpr int kParts = NTHREADS / 128;
    const int quad = warp & 3, part = warp >> 2;
    const int row_in_tile = quad * 32 + lane;
    const int row = m0 + row_in_tile;
    const bool row_ok = row_in_tile < TM && row < p.out_features;
    float sc = 1.f, bi = 0.f;
    if (row_ok && p.ksplit == 1) {
      sc = DT<T>::to_float(reinterpret_cast<const T*>(p.scales)[row]);
      if (p.bias) bi = DT<T>::to_float(reinterpret_cast<const T*>(p.bias)[row]);
    }
    if (nkb > 0) {
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
    }
    float* my_part = p.ws_partials ? p.ws_partials + ((tile_id * p.ksplit + split) * (size_t)N) * kGemmBlockM : nullptr;
    for (int c0 = part * 32; c0 < N; c0 += kParts * 32) {
      uint32_t r[32];
      if (nkb > 0) {
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, r);
      } else {
#pragma unroll
        for (int c = 0; c < 32; ++c) r[c] = 0u;
      }
      if (p.ksplit == 1) {
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          const int n = n0 + c0 + c;
          if (row_ok && c0 + c < N && n < p.batch && !(p.debug & 16)) y[(size_t)n * p.out_features + row] = DT<T>::from_float(fmaf(__uint_as_float(r[c]), sc, bi));
        }
      } else {
#pragma unroll
        for (int c = 0; c < 32; ++c)
          if (c0 + c < N) my_part[(size_t)(c0 + c) * kGemmBlockM + row_in_tile] = __uint_as_float(r[c]);
      }
    }
  }
  if (p.ksplit > 1) {
    // Split-K fix-up: the LAST-arriving split of this tile adds all partials in split order (deterministic) with the
    // whole CTA: thread -> (row, column phase); partials are [split][column][128 rows] so warps read 512 contiguous bytes.
    __threadfence();
    __syncthreads();
    uint32_t* flag = reinterpret_cast<uint32_t*>(gbase + L.flag);
    if (threadIdx.x == 0) {
      const unsigned int old = atomicAdd(p.ws_counters + tile_id, 1u);
      const bool last = (old == (unsigned int)p.ksplit - 1);
      *flag = last ? 1u : 0u;
      if (last) p.ws_counters[tile_id] = 0u;  // leave the counter clean for the next call
    }
    __syncthreads();
    if (*flag) {
      __threadfence();
      const float* parts = p.ws_partials + (tile_id * p.ksplit) * (size_t)N * kGemmBlockM;
      const int rrow = threadIdx.x & (kGemmBlockM - 1);
      const int cphase = threadIdx.x >> 7;
      constexpr int kPhases = NTHREADS / kGemmBlockM;
      const int row = m0 + rrow;
      if (rrow < TM && row < p.out_features) {
        const float sc = DT<T>::to_float(reinterpret_cast<const T*>(p.scales)[row]);
        const float bi = p.bias ? DT<T>::to_float(reinterpret_cast<const T*>(p.bias)[row]) : 0.f;
        const int ncols = min(N, p.batch - n0);
        for (int c = cphase; c < ncols; c += kPhases * 4) {
          float v[4] = {0.f, 0.f, 0.f, 0.f};
          for (int sp = 0; sp < p.ksplit; ++sp) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int cc = c + u * kPhases;
              if (cc < ncols) v[u] += __ldcg(parts + ((size_t)sp * N + cc) * kGemmBlockM + rrow);
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int cc = c + u * kPhases;
            if (cc < ncols) y[(size_t)(n0 + cc) * p.out_features + row] = DT<T>::from_float(fmaf(v[u], sc, bi));
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (C > 1) cluster_sync_all();  // no CTA exits while a peer can still signal its barriers
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

}  // namespace aqlm_b200
