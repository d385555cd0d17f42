// Batched 16-bit GEMM on tcgen05 with fp32 accumulation in TMEM and fp32 output:
//
//   C[z][m, n] (+)= alpha * sum_{kb < KB} sum_{k < K} A[z][kb][m, k] * B[z][kb][n, k]
//
// One CTA per (128 * MT) x NT output tile (NT = 64 ... 256, MT * NT <= 512 TMEM columns).  Operands are read by TMA through 2-D tensor
// maps laid over the whole operand arrays; each operand is either K-major (array rows = m or n,
// columns = k) or MN-major (array rows = k, columns = m or n), so the transposes that the DAMSM
// backward needs (d img = dV^T beta, ...) cost nothing.  (z, kb) select sub-matrices through
// row / column offsets into the maps.  K must be a multiple of 64 (callers pad with zeros);
// ragged M / N edges are masked at the store.
//
// Warp roles: warp 4 = TMA producer, warp 5 = MMA issuer, warps 0-3 = epilogue (TMEM -> global).
#include <algorithm>
#include <atomic>

#include "tc_gemm_pairs.cuh"

namespace agb {
namespace tc {

constexpr int kGemmStages = 6;
constexpr int kGemmStageBytes = 2 * kChunkBytes16;   // A chunk + B chunk, 16 KB each
constexpr int kGemmSmem = kGemmStages * kGemmStageBytes + 1024;   // >= the 128 x 129 fp32 store tile

// SWIZZLE_128B descriptor for an MN-major operand: tile = [k rows][64 mn elements], 8-row groups
// 1024 B apart (SBO), successive 64-wide mn blocks `lbo_bytes` apart (LBO)
__device__ __forceinline__ uint64_t make_desc_sw128_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// kPairs: the per-batch K range / B operand of TcGemmPairArgs (all of it under if constexpr)
template <bool kPairs, typename Args>
__device__ __forceinline__ void tc_gemm_body(const CUtensorMap& mapA, const CUtensorMap& mapB, const CUtensorMap& mapA2,
                                             const CUtensorMap& mapB2, const Args& g) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = (unsigned char*)(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t full[kGemmStages], empty[kGemmStages], done;
  __shared__ uint32_t tmem_base_s;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int MT = g.MT;                                  // 128-row tiles per CTA sharing the B operand
  // output columns of this CTA: NT each, except that column 0 may be wider / narrower (NT0)
  const int NT = (g.NT0 && blockIdx.x == 0) ? g.NT0 : g.NT;
  const int n0 = g.NT0 ? (blockIdx.x == 0 ? 0 : g.NT0 + ((int)blockIdx.x - 1) * g.NT) : (int)blockIdx.x * g.NT;
  const int m0 = blockIdx.y * 128 * MT, z = blockIdx.z;
  int kchunks = g.K >> 6;
  int kb_begin = 0, kb_count = g.KB;
  const int zb = g.split_kb ? 0 : z;                   // batch index used for operand offsets
  if (g.split_kb) {
    kb_begin = z * g.KB;
    kb_count = max(0, min(g.KB, g.kb_total - kb_begin));
  }
  int krow0 = 0, zbB = zb;                             // kPairs: first K row of batch z, batch of the B operand
  if constexpr (kPairs) {
    if (g.koff) {
      const int lo = min(max(g.koff[z], g.kt0), g.kt0 + g.kct), hi = min(max(g.koff[z + 1], g.kt0), g.kt0 + g.kct);
      kchunks = max(0, hi - lo) * 2;
      krow0 = (lo - g.kt0) * 128;
    }
    if (g.bsel) {
      if (g.dyn_t0 + z >= g.dyn_tiles[0]) return;
      zbB = g.bsel[g.dyn_t0 + z];
    }
  }
  int m_valid = g.M;
  if (g.dyn_dim) {
    const int valid = max(0, (g.dyn_tiles[0] - g.dyn_t0) * 128);
    if (g.dyn_dim == 1) m_valid = min(g.M, valid);
    else kchunks = min(kchunks, (valid + 63) >> 6);
  }
  if (m0 >= m_valid) return;                           // whole CTA: nothing to do (before any barrier / alloc)
  const int per_src = kb_count * kchunks;
  const int total = g.nsrc * per_src;
  if (total == 0 && g.accumulate) return;              // empty reduction added to C: nothing to do
  const int stages = g.stages;
  const int nt_boxes = (NT + 63) >> 6;                 // B is staged in whole 64-column boxes (NT = 160: 2.5 -> 3)
  const int stage_bytes = MT * kChunkBytes16 + nt_boxes * 64 * 128;
  const uint32_t tmem_cols = MT * NT <= 128 ? 128u : (MT * NT <= 256 ? 256u : 512u);

  if (threadIdx.x == 0) {
    for (int i = 0; i < stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(&done, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&tmem_base_s, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  if (warp == 4) {
    if (elect_one()) {
      const uint32_t bytes = (uint32_t)stage_bytes;
      for (int it = 0; it < total; ++it) {
        const int s = it % stages, use = it / stages;
        const int src = it / per_src, r = it - src * per_src;
        const int kbl = r / kchunks, k0 = (r - kbl * kchunks) * 64;
        const int kb = kb_begin + kbl;
        const CUtensorMap* mA = src ? &mapA2 : &mapA;
        const CUtensorMap* mB = src ? &mapB2 : &mapB;
        mbar_wait(&empty[s], (use & 1) ^ 1);
        mbar_expect_tx(&full[s], bytes);
        unsigned char* sa = smem + s * stage_bytes;
        unsigned char* sb = sa + MT * kChunkBytes16;
        const int64_t azr = src ? g.a2_zrow : g.a_zrow, bzr = src ? g.b2_zrow : g.b_zrow;
        const int64_t azc = src ? g.a2_zcol : g.a_zcol, bzc = src ? g.b2_zcol : g.b_zcol;
        int arow = (int)(zb * azr + kb * g.a_kbrow), acol = (int)(zb * azc + kb * g.a_kbcol);
        int brow = (int)(zbB * bzr + kb * g.b_kbrow), bcol = (int)(zbB * bzc + kb * g.b_kbcol);
        if constexpr (kPairs) {
          (g.a_mn ? arow : acol) += krow0;
          (g.b_mn ? brow : bcol) += krow0;
        }
        for (int mt = 0; mt < MT; ++mt) {
          unsigned char* sam = sa + mt * kChunkBytes16;
          const int mm = m0 + mt * 128;
          if (!g.a_mn) {
            tma_load_2d(sam, mA, &full[s], acol + k0, arow + mm);                 // [128 m][64 k]
          } else {
            tma_load_2d(sam, mA, &full[s], acol + mm, arow + k0);                 // [64 k][64 m] x 2
            tma_load_2d(sam + 8192, mA, &full[s], acol + mm + 64, arow + k0);
          }
        }
        if (!g.b_mn) {
          tma_load_2d(sb, mB, &full[s], bcol + k0, brow + n0);                    // [NT n][64 k]
        } else {
          for (int nb = 0; nb < nt_boxes; ++nb)
            tma_load_2d(sb + nb * 8192, mB, &full[s], bcol + n0 + nb * 64, brow + k0);
        }
      }
    }
  } else if (warp == 5) {
    if (elect_one()) {
      const uint32_t idesc = make_idesc(128, NT, g.bf16) | ((uint32_t)g.a_mn << 15) | ((uint32_t)g.b_mn << 16);
      for (int it = 0; it < total; ++it) {
        const int s = it % stages, use = it / stages;
        mbar_wait(&full[s], use & 1);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + s * stage_bytes), sb = sa + MT * kChunkBytes16;
        for (int kk = 0; kk < 4; ++kk) {
          // K-major: +32 B per 16 k inside the 128-B row; MN-major: +16 rows = 2048 B
          const uint64_t db = g.b_mn ? make_desc_sw128_mn(sb + kk * 2048, 8192) : make_desc_sw128(sb) + 2 * kk;
          for (int mt = 0; mt < MT; ++mt) {
            const uint32_t sam = sa + mt * kChunkBytes16;
            const uint64_t da = g.a_mn ? make_desc_sw128_mn(sam + kk * 2048, 8192) : make_desc_sw128(sam) + 2 * kk;
            umma_f16(tmem + mt * NT, da, db, idesc, (it | kk) ? 1u : 0u);
          }
        }
        umma_commit(&empty[s]);
      }
      umma_commit(&done);
    }
  } else if (warp < 4) {
    if (total > 0) {
      mbar_wait(&done, 0);
      tc_fence_after();
    }
    float* Cz = g.C + (int64_t)z * g.c_z;
    for (int mt = 0; mt < MT; ++mt) {
      const int mbase = m0 + mt * 128;
      if (mbase >= m_valid) break;
      if (g.c_n == 1) {
        // n-contiguous output: transpose through shared memory (the operand ring is idle now) so that
        // every warp writes whole rows -- coalesced for any row pitch / alignment
        float* tile = reinterpret_cast<float*>(smem);          // [128][NT + 1]
        const int pitch = NT + 1;
        const int row = warp * 32 + lane;
        if (mt > 0) named_bar_sync(1, 128);                    // previous tile fully written out
        for (int c0 = 0; c0 < NT; c0 += 32) {
          float v[32];
          if (total > 0) {
            tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + mt * NT + c0, v);
            tmem_ld_wait();
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 0.f;           // empty reduction: the sum is zero
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) tile[row * pitch + c0 + j] = v[j];
        }
        named_bar_sync(1, 128);
        const int rows = min(128, m_valid - mbase);
        const int cols = min(NT, g.N - n0);
        if (!g.accumulate) {
          for (int r = warp; r < rows; r += 4) {
            float* prow = Cz + (int64_t)(mbase + r) * g.c_m + n0;
            for (int n = lane; n < cols; n += 32) prow[n] = g.alpha * tile[r * pitch + n];
          }
        } else {
          // read-modify-write of C: issue the loads of four rows (up to 32 per lane) before the first dependent
          // store.  One load per loop trip exposed a full memory round trip per 32 columns: the accumulating d img
          // launches took 8.7 ms against 5.1 ms for the same GEMM writing C (profiles/r2_launches_cfg4_n1.csv).
          constexpr int kRows = 4, kPer = 8;                   // NT <= 256 -> at most 8 columns per lane
          for (int r0 = warp * kRows; r0 < rows; r0 += 4 * kRows) {
            float old[kRows][kPer];
#pragma unroll
            for (int i = 0; i < kRows; ++i) {
              const float* prow = Cz + (int64_t)(mbase + r0 + i) * g.c_m + n0;
#pragma unroll
              for (int j = 0; j < kPer; ++j) {
                const int n = lane + 32 * j;
                old[i][j] = (r0 + i < rows && n < cols) ? prow[n] : 0.f;
              }
            }
#pragma unroll
            for (int i = 0; i < kRows; ++i) {
              float* prow = Cz + (int64_t)(mbase + r0 + i) * g.c_m + n0;
#pragma unroll
              for (int j = 0; j < kPer; ++j) {
                const int n = lane + 32 * j;
                if (r0 + i < rows && n < cols) prow[n] = old[i][j] + g.alpha * tile[(r0 + i) * pitch + n];
              }
            }
          }
        }
      } else {
        const int m = mbase + warp * 32 + lane;
        for (int c0 = 0; c0 < NT; c0 += 32) {
          float v[32];
          if (total > 0) {
            tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + mt * NT + c0, v);
            tmem_ld_wait();
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 0.f;
          }
          if (m < m_valid) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int n = n0 + c0 + j;
              if (n < g.N) {
                float* p = Cz + (int64_t)m * g.c_m + (int64_t)n * g.c_n;
                const float x = g.alpha * v[j];
                *p = g.accumulate ? (*p + x) : x;
              }
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, tmem_cols);
}

__global__ void __launch_bounds__(192)
tc_gemm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
               const __grid_constant__ CUtensorMap mapA2, const __grid_constant__ CUtensorMap mapB2,
               const TcGemmArgs g) {
  tc_gemm_body<false>(mapA, mapB, mapA2, mapB2, g);
}

__global__ void __launch_bounds__(192)
tc_gemm_pairs_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                     const __grid_constant__ CUtensorMap mapA2, const __grid_constant__ CUtensorMap mapB2,
                     const TcGemmPairArgs g) {
  tc_gemm_body<true>(mapA, mapB, mapA2, mapB2, g);
}

// launch configuration shared by both instantiations: validates g, sets g.stages, returns grid and smem size
template <typename Args>
static int tc_gemm_config(Args& g, int batch, dim3* grid_out, int* smem_out) {
  if (g.K <= 0 || g.K % 64 || g.KB <= 0) return fail_arg("tc_gemm: K=%d must be a positive multiple of 64", g.K);
  if (g.NT != 64 && g.NT != 128 && g.NT != 192 && g.NT != 256 && !(g.NT == 160 && g.b_mn))
    return fail_arg("tc_gemm: NT=%d", g.NT);
  if (g.NT0 && (g.NT0 % 64 || g.NT0 > 256 || !g.b_mn)) return fail_arg("tc_gemm: NT0=%d", g.NT0);
  if (g.MT != 1 && g.MT != 2) g.MT = 1;
  const int nt_max = std::max(g.NT, g.NT0);
  if (g.MT * nt_max > 512) return fail_arg("tc_gemm: MT*NT=%d exceeds TMEM", g.MT * nt_max);
  if (g.nsrc != 2) g.nsrc = 1;
  dim3 grid(g.NT0 ? 1 + cdiv(std::max(0, g.N - g.NT0), g.NT) : cdiv(g.N, g.NT), cdiv(g.M, 128 * g.MT), batch);
  if (grid.y > 65535 || grid.z > 65535) return fail_unsupported("tc_gemm grid too large");
  const int stage_bytes = g.MT * kChunkBytes16 + (nt_max + 63) / 64 * 64 * 128;
  const long long chunks = (long long)g.nsrc * g.KB * (g.K / 64);
  const int max_stages = std::min(kGemmStages, (kGemmSmem - 1024) / stage_bytes);
  g.stages = (int)std::min<long long>(max_stages, std::max<long long>(2, chunks));
  *grid_out = grid;
  *smem_out = std::max(g.stages * stage_bytes, 128 * (nt_max + 1) * 4) + 1024;
  return 0;
}

int tc_gemm_pairs(const TcGemmPairArgs& g_in, const CUtensorMap& mapA, const CUtensorMap& mapB, const CUtensorMap& mapA2,
                  const CUtensorMap& mapB2, int batch, cudaStream_t st) {
  TcGemmPairArgs g = g_in;
  if (g.M <= 0 || g.N <= 0 || batch <= 0) return 0;
  dim3 grid;
  int smem_bytes = 0;
  if (int rc = tc_gemm_config(g, batch, &grid, &smem_bytes)) return rc;
  {   // per device, once
    static std::atomic<bool> attr_set[64];
    int dev = 0;
    AGB_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_set[dev].load(std::memory_order_relaxed)) {
      AGB_CUDA(cudaFuncSetAttribute(tc_gemm_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGemmSmem));
      if (dev >= 0 && dev < 64) attr_set[dev].store(true, std::memory_order_relaxed);
    }
  }
  const int slot = prof_begin(g.prof_tag ? g.prof_tag : PROF_DAMSM_TC_BWD, st);
  tc_gemm_pairs_kernel<<<grid, 192, smem_bytes, st>>>(mapA, mapB, mapA2, mapB2, g);
  prof_end(slot, st);
  return check_launch("tc_gemm_pairs_kernel");
}

int tc_gemm2(const TcGemmArgs& g_in, const CUtensorMap& mapA, const CUtensorMap& mapB, const CUtensorMap& mapA2,
             const CUtensorMap& mapB2, int batch, cudaStream_t st) {
  TcGemmArgs g = g_in;
  if (g.M <= 0 || g.N <= 0 || batch <= 0) return 0;
  // NT = 160 (MN-major B only): two equal column tiles for N = 289...320, so that the CTAs sharing an A operand run
  // in lockstep and the second read of A hits the L2 (a 192 + 128 split drifts apart: 24 GB instead of 17 GB of DRAM
  // reads per d img launch, profiles/r2_ncu_attention_and_gemm_metrics.txt)
  dim3 grid;
  int smem_bytes = 0;
  if (int rc = tc_gemm_config(g, batch, &grid, &smem_bytes)) return rc;
  {   // per device, once
    static std::atomic<bool> attr_set[64];
    int dev = 0;
    AGB_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_set[dev].load(std::memory_order_relaxed)) {
      AGB_CUDA(cudaFuncSetAttribute(tc_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGemmSmem));
      if (dev >= 0 && dev < 64) attr_set[dev].store(true, std::memory_order_relaxed);
    }
  }
  const int slot = prof_begin(g.prof_tag ? g.prof_tag : PROF_DAMSM_TC_BWD, st);
  tc_gemm_kernel<<<grid, 192, smem_bytes, st>>>(mapA, mapB, mapA2, mapB2, g);
  prof_end(slot, st);
  return check_launch("tc_gemm_kernel");
}

int tc_gemm(const TcGemmArgs& g, const CUtensorMap& mapA, const CUtensorMap& mapB, int batch, cudaStream_t st) {
  TcGemmArgs h = g;
  h.nsrc = 1;
  return tc_gemm2(h, mapA, mapB, mapA, mapB, batch, st);
}

}  // namespace tc
}  // namespace agb

using namespace agb;

// Test hook: C[M,N] = A * B^T for one batch.  A is [M,K] row-major (a_mn = 0) or [K,M] (a_mn = 1);
// B likewise with N.  M, N arbitrary (<= one grid), K % 64 == 0.  `accumulate`: bit 0 = add to C; bits 8-15 /
// 16-23 / 24-31 select the tiling under test: NT / 32 (0 = default), NT0 / 64, MT.
extern "C" int agb_tc_gemm_test(const void* A, const void* B, float* C, int M, int N, int K, int a_mn, int b_mn,
                                int bf16, int accumulate, void* stream) {
  if (!A || !B || !C) return fail_arg("null pointer");
  CUtensorMap mapA, mapB;
  const int nt_sel = ((accumulate >> 8) & 0xff) * 32, nt0_sel = ((accumulate >> 16) & 0xff) * 64;
  const int mt_sel = (accumulate >> 24) & 0xff;
  accumulate &= 1;
  const int NT = nt_sel ? nt_sel : ((N % 128 == 0 || N > 64) ? 128 : 64);
  // box rows: K-major operands load [128 or NT rows x 64]; MN-major operands load [64 k rows x 64]
  if (int rc = tc::make_tmap_2d(&mapA, A, a_mn ? K : M, a_mn ? M : K, a_mn ? 64 : 128, bf16 != 0)) return rc;
  if (int rc = tc::make_tmap_2d(&mapB, B, b_mn ? K : N, b_mn ? N : K, b_mn ? 64 : NT, bf16 != 0)) return rc;
  tc::TcGemmArgs g{};
  g.a_mn = a_mn; g.b_mn = b_mn; g.bf16 = bf16 ? 1 : 0; g.M = M; g.N = N; g.K = K; g.KB = 1; g.NT = NT;
  g.C = C; g.c_z = 0; g.c_m = N; g.c_n = 1; g.alpha = 1.f; g.accumulate = accumulate;
  g.NT0 = nt0_sel; g.MT = mt_sel ? mt_sel : 1;
  return tc::tc_gemm(g, mapA, mapB, 1, (cudaStream_t)stream);
}
