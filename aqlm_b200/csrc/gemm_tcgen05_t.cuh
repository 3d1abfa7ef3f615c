// Fused additive-dequant + TRANSPOSED tensor-core GEMM (the backward w.r.t. the input):
//     grad_in[bs, in] = (grad_out[bs, out] * scales[out]) . W[out, in]          W never touches HBM.
//
// Replaces code{1x16,2x8,1x8}_matmat_dequant_transposed (reference cuda_kernel.cpp:303-354, 486-519, 651-684), which
// materialise W [out,in] in HBM with a Dequant kernel and call cuBLAS on (grad_out * scales); the reference's 2x8/1x8
// variants forget the scaled input (cuda_kernel.cpp:497,518,662,683) -- not reproduced.
//
// Same tcgen05 / TMEM / TMA skeleton as gemm_tcgen05.cuh with the contraction running over OUT rows:
//   D[128 in-features x N batch] (fp32, TMEM)  +=  A[128 x 64] . B[N x 64]^T        per k-block of 64 out rows
//   A = W^T tile, produced on chip.  A gathered codebook vector is 8 CONSECUTIVE in-features of ONE out row, i.e. 16
//       contiguous bytes along M: the A stage is therefore kept MN-MAJOR (canonical SWIZZLE_128B MN-major layout,
//       64 x 8 element atoms, instruction descriptor a_major = 1), so a gather still lands with ONE 16-byte store;
//       the per-row scale is applied to the vector before it is written (fp32 multiply, one rounding);
//   B = grad_out tile [N x 64 out columns], K-major, TMA-loaded with 128B swizzle (OOB rows/columns zero-filled);
//   code tiles: TMA boxes of 256 out rows x (128 / in_group_size groups * K codes) bytes, un-swizzled.
// Grid = (in/128 tiles, K splits over the out rows, N tiles); split partials and the deterministic last-CTA fix-up are
// the forward kernel's.
#pragma once

#include "gemm_tcgen05.cuh"

namespace aqlm_b200 {

constexpr int kGemmTCtileRows = 256;  // out rows per code tile (= 4 k-blocks)
constexpr int kGemmTThreads = 128 + 32 * 16;

struct GemmTParams {
  const void* codebooks;
  const void* scales;         // [out]
  void* y;                    // grad_in [batch, in_features]
  float* ws_partials;
  unsigned int* ws_counters;
  int in_features;
  int out_features;
  int batch;
  int nbits;
  int total_kblocks;          // ceil(out / 64)
  int ksplit;
  int n_tile;
  int stages;
  int gather_mode;
};

// UMMA shared-memory descriptor, MN-major, SWIZZLE_128B: atoms of 64 (MN) x 8 (K) elements = 1024 bytes;
// LBO = byte distance between atoms along MN, SBO = byte distance between atoms along K (both >> 4).
__device__ __forceinline__ uint64_t umma_desc_mn128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}

struct GemmTSmem {
  uint32_t a, b, codes, full, empty, cfull, cempty, tfull, tmem_slot, flag;
  size_t total;
};
__host__ __device__ inline GemmTSmem gemm_t_smem_layout(int stages, int n_tile, int ctile_row_bytes) {
  GemmTSmem L;
  size_t off = 0;
  L.a = (uint32_t)off; off += (size_t)stages * kGemmBlockM * 128;
  L.b = (uint32_t)off; off += (size_t)stages * n_tile * 128;
  off = (off + 1023) & ~(size_t)1023;
  L.codes = (uint32_t)off; off += (size_t)kCodeTileStages * kGemmTCtileRows * ctile_row_bytes;
  off = (off + 15) & ~(size_t)15;
  L.full = (uint32_t)off; off += 8 * 8;
  L.empty = (uint32_t)off; off += 8 * 8;
  L.cfull = (uint32_t)off; off += 8 * kCodeTileStages;
  L.cempty = (uint32_t)off; off += 8 * kCodeTileStages;
  L.tfull = (uint32_t)off; off += 8;
  L.tmem_slot = (uint32_t)off; off += 4;
  L.flag = (uint32_t)off; off += 4;
  L.total = off + 1024;
  return L;
}

// GS = in_group_size.  GS = 16 (1x16 only): a thread's 16 in-features are ONE codebook entry of 32 bytes, fetched as one
// 256-bit request and stored as the same two 16-byte chunks along M that two 8-wide groups fill.
template <typename T, int K, int CODE_BYTES, int GS = 8>
__global__ void __launch_bounds__(kGemmTThreads, 1)
gemm_dequant_t_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_codes, const GemmTParams p) {
  static_assert(GS == 8 || (GS == 16 && K == 1 && CODE_BYTES == 2), "in_group_size 16: 1x16 only");
  constexpr int GBT = (kGemmBlockM / GS) * K * CODE_BYTES;  // code bytes per out row per tile (128 in-features)
  constexpr int CB2 = GBT / 8;                              // code bytes of one thread's 16 in-features
  constexpr int CW = (CB2 + 3) / 4;
  constexpr int D = (K == 1) ? 4 : (K == 2 ? 2 : 1);  // k-blocks of gathers held in registers ahead of the writes
  constexpr int KB_PER_CTILE = kGemmTCtileRows / kGemmBlockK;
  extern __shared__ uint8_t smem_dyn[];
  const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
  uint8_t* gbase = smem_dyn + (base - smem_u32(smem_dyn));
  const GemmTSmem L = gemm_t_smem_layout(p.stages, p.n_tile, GBT);
  const int S = p.stages, N = p.n_tile;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x, split = blockIdx.y, n_blk = blockIdx.z;
  const int m0 = m_tile * kGemmBlockM, n0 = n_blk * N;
  const int kb0 = (int)(((long long)p.total_kblocks * split) / p.ksplit);
  const int kb1 = (int)(((long long)p.total_kblocks * (split + 1)) / p.ksplit);
  const int nkb = kb1 - kb0;
  const int ct0 = kb0 / KB_PER_CTILE, ct1 = (kb1 + KB_PER_CTILE - 1) / KB_PER_CTILE;
  griddep_launch_dependents();  // PDL, as in the forward kernel: weights before griddep_wait(), grad_out / outputs after

  auto full_bar = [&](int s) { return base + L.full + 8 * s; };
  auto empty_bar = [&](int s) { return base + L.empty + 8 * s; };
  auto cfull_bar = [&](int s) { return base + L.cfull + 8 * s; };
  auto cempty_bar = [&](int s) { return base + L.cempty + 8 * s; };
  const uint32_t tfull_bar = base + L.tfull;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gbase + L.tmem_slot);

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full_bar(s), 16 + 1);  // 16 producer warps + the TMA thread (expect_tx)
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < kCodeTileStages; ++s) {
      mbar_init(cfull_bar(s), 1);
      mbar_init(cempty_bar(s), 16);
    }
    mbar_init(tfull_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < N) tmem_cols <<= 1;
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(base + L.tmem_slot), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (nkb > 0) {
    if (warp == 0) {
      // ===== TMA producer (whole warp, one elected lane issues): code tiles (256 out rows x GBT bytes) and one grad_out
      //       tile per k-block =====
      int ct_loaded = ct0;
      auto load_ctile = [&](int ct) {
        const int cs = (ct - ct0) % kCodeTileStages, it = (ct - ct0) / kCodeTileStages;
        if (it > 0) mbar_wait(cempty_bar(cs), (it - 1) & 1);
        if (elect_one()) {
          mbar_expect_tx(cfull_bar(cs), kGemmTCtileRows * GBT);
          tma_load_2d(base + L.codes + cs * kGemmTCtileRows * GBT, &tmap_codes, m_tile * GBT, ct * kGemmTCtileRows, cfull_bar(cs));
        }
        __syncwarp();
      };
      load_ctile(ct_loaded++);
      griddep_wait();  // grad_out is produced by the previous kernel
      int s = 0, it = 0;
      for (int i = 0; i < nkb; ++i) {
        if (it > 0) mbar_wait(empty_bar(s), (it - 1) & 1);
        if (elect_one()) {
          mbar_expect_tx(full_bar(s), (uint32_t)N * 128);
          tma_load_2d(base + L.b + s * N * 128, &tmap_g, (kb0 + i) * kGemmBlockK, n0, full_bar(s));
        }
        __syncwarp();
        const int ct_cur = (kb0 + i) / KB_PER_CTILE;
        if (ct_loaded < ct1 && ct_loaded <= ct_cur + 1) load_ctile(ct_loaded++);
        if (++s == S) { s = 0; ++it; }
      }
    } else if (warp == 1) {
      // ===== MMA issuer (whole warp, one elected lane issues; see gemm_tcgen05.cuh): A MN-major (a_major bit 15), B K-major =====
      const uint32_t idesc = umma_idesc(DT<T>::is_bf16 ? 1 : 0, N) | (1u << 15);
      int s = 0;
      uint32_t ph = 0;
      for (int i = 0; i < nkb; ++i) {
        mbar_wait(full_bar(s), ph);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_addr = base + L.a + s * kGemmBlockM * 128;
          const uint32_t b_addr = base + L.b + s * N * 128;
          const uint64_t adesc = umma_desc_mn128(a_addr, 1024, 2048);
          const uint64_t bdesc = umma_desc_k128(b_addr);
#pragma unroll
          for (int k = 0; k < kGemmBlockK / 16; ++k) {
            // one MMA covers 16 out rows = 2 K-atoms of the stage: atoms are laid out [k_atom (8)][m_atom (2)][1024 B], so
            // A advances by 4096 bytes (+256 in the address field), B by 32 bytes (+2)
            umma_f16(tmem_base, adesc + (uint64_t)(256 * k), bdesc + (uint64_t)(2 * k), idesc, (i | k) ? 1u : 0u);
          }
          umma_commit(empty_bar(s));
        }
        __syncwarp();
        if (++s == S) { s = 0; ph ^= 1u; }
      }
      if (elect_one()) umma_commit(tfull_bar);
      __syncwarp();
    } else if (warp >= 4) {
      // ===== dequant producers: 512 threads, thread -> (out row kk of the k-block, 16 consecutive in-features: 2 adjacent
      //       groups of 8, or 1 group of 16) =====
      const int pt = threadIdx.x - 128;
      const int kk = pt >> 3, gp = pt & 7;  // kk: 0..63, gp: group pair 0..7 -> groups 2gp, 2gp+1 (of 16)
      const uint4* gcb = reinterpret_cast<const uint4*>(p.codebooks);
      const T* gsc = reinterpret_cast<const T*>(p.scales);

      auto issue = [&](int i, uint4 (&wv)[2][K], float& sc) {
        const int kb = kb0 + i;
        const int ct = kb / KB_PER_CTILE, st_in = kb % KB_PER_CTILE;
        const int cs = (ct - ct0) % kCodeTileStages, cit = (ct - ct0) / kCodeTileStages;
        const int o = kb * kGemmBlockK + kk;
        sc = o < p.out_features ? DT<T>::to_float(gsc[o]) : 0.f;  // rows past the end contribute nothing
        mbar_wait(cfull_bar(cs), cit & 1);
        const uint8_t* src = gbase + L.codes + cs * kGemmTCtileRows * GBT + (st_in * kGemmBlockK + kk) * GBT + gp * CB2;
        uint32_t cw[CW];
        if constexpr (CB2 >= 16) {
          const uint4 v = *reinterpret_cast<const uint4*>(src);
          cw[0] = v.x; cw[1] = v.y; cw[2] = v.z; cw[3] = v.w;
        } else if constexpr (CB2 == 8) {
          const uint2 v = *reinterpret_cast<const uint2*>(src);
          cw[0] = v.x; cw[1] = v.y;
        } else if constexpr (CB2 == 4) {
          cw[0] = *reinterpret_cast<const uint32_t*>(src);
        } else {
          cw[0] = *reinterpret_cast<const uint16_t*>(src);
        }
        if constexpr (GS == 16) {
          const uint4* gq = gcb + 2 * (size_t)(cw[0] & 0xffffu);
          if (p.gather_mode == 1) ld_gather_v8<1>(gq, wv[0][0], wv[1][0]);
          else ld_gather_v8<0>(gq, wv[0][0], wv[1][0]);
        } else {
#pragma unroll
          for (int e = 0; e < 2; ++e) {
#pragma unroll
            for (int k = 0; k < K; ++k) {
              const int idx = e * K + k;
              uint32_t code;
              if constexpr (CODE_BYTES == 2) code = (cw[idx >> 1] >> ((idx & 1) * 16)) & 0xffffu;
              else code = (cw[idx >> 2] >> ((idx & 3) * 8)) & 0xffu;
              const uint4* gq = gcb + (((size_t)k << p.nbits) + code);
              if (p.gather_mode == 1) wv[e][k] = ld_gather_v4<1>(gq);
              else wv[e][k] = ld_gather_v4<0>(gq);
            }
          }
        }
        if (st_in == KB_PER_CTILE - 1 || i == nkb - 1) {  // after the gathers were issued: the code reads have completed
          __syncwarp();
          if (lane == 0) mbar_arrive(cempty_bar(cs));
        }
      };
      int st_next = 0, it_next = 0;  // commit() runs for k-blocks 0, 1, 2, ... in order: stage / use count without division
      auto commit = [&](int i, uint4 (&wv)[2][K], float sc) {
        (void)i;
        const int s = st_next, it = it_next;
        if (++st_next == S) { st_next = 0; ++it_next; }
        if (it > 0) mbar_wait(empty_bar(s), (it - 1) & 1);
        // MN-major SWIZZLE_128B: atom (kk>>3, m_atom) at [(kk>>3)*2 + m_atom]*1024; inside an atom row kk&7 is 128 bytes of
        // 64 consecutive in-features, its 16-byte chunks XOR-swizzled with (kk&7)
        uint8_t* abase = gbase + L.a + s * kGemmBlockM * 128 + (kk >> 3) * 2048 + (kk & 7) * 128;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          uint4 v;
          if constexpr (K == 1) {
            // one codebook: scale the packed vector with 4 packed multiplies (a 16-bit x 16-bit product is exact in fp32, so
            // the packed multiply rounds exactly like fp32-multiply-then-round)
            v = wv[e][0];
            if constexpr (DT<T>::is_bf16) {
              const __nv_bfloat162 s2 = __float2bfloat162_rn(sc);
              __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
              for (int q = 0; q < 4; ++q) h[q] = __hmul2(h[q], s2);
            } else {
              const __half2 s2 = __float2half2_rn(sc);
              __half2* h = reinterpret_cast<__half2*>(&v);
#pragma unroll
              for (int q = 0; q < 4; ++q) h[q] = __hmul2(h[q], s2);
            }
          } else {
            float f[8];
            unpack8<T>(wv[e][0], f);
#pragma unroll
            for (int k = 1; k < K; ++k) accum8<T>(wv[e][k], f);
#pragma unroll
            for (int q = 0; q < 8; ++q) f[q] *= sc;
            v.x = DT<T>::pack2(f[0], f[1]); v.y = DT<T>::pack2(f[2], f[3]);
            v.z = DT<T>::pack2(f[4], f[5]); v.w = DT<T>::pack2(f[6], f[7]);
          }
          const int j = gp * 2 + e;  // group 0..15 of the tile = 16-byte chunk j along M
          *reinterpret_cast<uint4*>(abase + (j >> 3) * 1024 + (((j & 7) ^ (kk & 7)) << 4)) = v;
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(full_bar(s));
      };
      uint4 w[D][2][K];
      float scv[D];
#pragma unroll
      for (int d = 0; d < D; ++d)
        if (d < nkb) issue(d, w[d], scv[d]);
      for (int i = 0; i < nkb; i += D) {
#pragma unroll
        for (int d = 0; d < D; ++d) {
          if (i + d < nkb) {
            commit(i + d, w[d], scv[d]);
            if (i + d + D < nkb) issue(i + d + D, w[d], scv[d]);
          }
        }
      }
    }
  }

  // ===== epilogue: all warps (5 per TMEM lane quadrant), thread <-> TMEM lane <-> in-feature =====
  const size_t tile_id = (size_t)m_tile * gridDim.z + n_blk;
  T* y = reinterpret_cast<T*>(p.y);
  {
    __syncwarp();
    griddep_wait();  // before any global write
    constexpr int kParts = kGemmTThreads / 128;
    const int quad = warp & 3, part = warp >> 2;
    const int row_in_tile = quad * 32 + lane;
    const int col = m0 + row_in_tile;  // in-feature index
    const bool col_ok = col < p.in_features;
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
          if (col_ok && c0 + c < N && n < p.batch) y[(size_t)n * p.in_features + col] = DT<T>::from_float(__uint_as_float(r[c]));
        }
      } else {
#pragma unroll
        for (int c = 0; c < 32; ++c)
          if (c0 + c < N) my_part[(size_t)(c0 + c) * kGemmBlockM + row_in_tile] = __uint_as_float(r[c]);
      }
    }
  }
  if (p.ksplit > 1) {
    __threadfence();
    __syncthreads();
    uint32_t* flag = reinterpret_cast<uint32_t*>(gbase + L.flag);
    if (threadIdx.x == 0) {
      const unsigned int old = atomicAdd(p.ws_counters + tile_id, 1u);
      const bool last = (old == (unsigned int)p.ksplit - 1);
      *flag = last ? 1u : 0u;
      if (last) p.ws_counters[tile_id] = 0u;
    }
    __syncthreads();
    if (*flag) {
      __threadfence();
      const float* parts = p.ws_partials + (tile_id * p.ksplit) * (size_t)N * kGemmBlockM;
      const int rrow = threadIdx.x & (kGemmBlockM - 1);
      const int cphase = threadIdx.x >> 7;
      constexpr int kPhases = kGemmTThreads / kGemmBlockM;
      const int col = m0 + rrow;
      if (col < p.in_features) {
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
            if (cc < ncols) y[(size_t)(n0 + cc) * p.in_features + col] = DT<T>::from_float(v[u]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

}  // namespace aqlm_b200
