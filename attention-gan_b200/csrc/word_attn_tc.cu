// Generator word-context attention on tcgen05 for 16-bit I/O (bf16 / fp16 feature maps).
//
// Replaces AttentionModule.forward (reference networks/attention.py:25-79).  At C = 32, T = 18 the
// CUDA-core formulation needs 1152 FMA per pixel forward against 164 B of HBM traffic, which puts
// its ceiling (fp32 FMA rate) below the HBM roofline; the two tiny contractions therefore run on
// the tensor cores and the SM only does the softmax and the stores:
//
//   tile       = 128 consecutive pixels of one sample (NCHW, HW contiguous)
//   TMA        h tile [C rows x 128 px] -> smem, 128B swizzle; used as the MN-major A operand
//   GEMM1      S[px, t]   = sum_c h[c, px] * (W.e)[c, t] * scale*log2(e)      (B operand: hi + lo split,
//                            so W.e enters with fp32 accuracy)                  M=128, N=NT, K=C
//   epilogue 1 thread = pixel: mask, softmax over the T words in registers (exp2), attn -> global,
//              P = attn as fp16 written back into TMEM (tcgen05.st) over the scores
//   GEMM2      ctx[px, c] = sum_t P[px, t] * (W.e)[c, t]        A operand from TMEM    M=128, N=C, K=NT
//   epilogue 2 thread = pixel: ctx -> global (lanes = consecutive pixels: coalesced)
//
// TMEM: 2 tile buffers x (NT score/P columns + C context columns) = 128 columns per CTA at
// T <= 32, C <= 32 (256 otherwise), so several CTAs share an SM and each keeps two tiles in flight.  The warp
// roles are listed at each kernel (forward: 10 warps; backward: 14 warps).
#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "tc_common.cuh"

namespace agb {
namespace tc {

__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ uint64_t make_desc_sw128_mn_lbo(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// ---- channels_last (NHWC) tiles ----
// A tile of 128 pixels x C channels is C/16 slabs of [128 px][16 ch] (32-byte rows, SWIZZLE_32B, 4 KB each),
// loaded by a 3-D TMA over (channel, pixel, sample), so pixels past the end of a sample read as zeros.
// Slab k holds channels 16k..16k+15: for a GEMM that contracts over channels it is the K-major operand of one
// K = 16 step; for a GEMM that contracts over pixels the slabs side by side are an MN-major operand (16
// channels per 32-byte row, 8-pixel groups 256 B apart, next 16 channels one slab = 4 KB further).
constexpr int kSlabBytes = 128 * 32;
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ uint64_t make_desc_sw32(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;   // MN-major: next 16 MN elements (K-major: ignored)
  d |= (uint64_t)(256 >> 4) << 32;                     // next group of 8 rows
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)6 << 61;                              // SWIZZLE_32B
  return d;
}

template <typename T16> __device__ __forceinline__ T16 f2h(float v);
template <> __device__ __forceinline__ __half f2h<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 f2h<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// ablation switches exist only in -DAGB_ABLATION builds (timing experiments; results are wrong when set)
#ifdef AGB_ABLATION
#define AGB_ABL(p, bit) ((p).dbg & (bit))
#else
#define AGB_ABL(p, bit) (false)
#endif

struct AttnFwdParams {
  const float* we;        // [B, C, T] fp32 projected words
  const int64_t* mask;    // [B, T]
  void* ctx;              // [B, C, HW] io dtype, batch stride ctx_bs
  void* attn;             // [B, T, HW] io dtype or null
  int64_t ctx_bs;
  int B, C, HW, T;
  float qscale;           // scale * log2(e)
  int tiles, ctas_per_sample;
  int stages;             // h-tile ring depth of the forward kernel
  int dbg;                // ablation switches for tuning (AGB_ATTN_DEBUG): 1 = no ctx stores, 2 = no attn stores
  int64_t ctx_ps;         // NHWC: pixel stride of ctx
};

constexpr int kAttnStages = 3;
constexpr int kMaxAttnStages = 8;
// first tile of CTA x when `tiles` tiles are split into `n` contiguous, balanced ranges
__device__ __forceinline__ int tile_range_begin(int tiles, int n, int x) { return (int)(((long long)tiles * x) / n); }
constexpr uint32_t kHalfLanes = 16u << 16;      // TMEM address of the second 16 lanes of a warp's quarter

// Epilogue layout (both kernels).  The epilogue warps read TMEM in the 16x256b fragment layout
// (tc_common.cuh): thread i of warp q owns the pixels q*32 + 16h + 8j + i/4 (h, j in {0,1}) and,
// per block k of 8 columns, the column pair 8k + 2(i%4) + {0,1}.  A softmax over the words is a
// reduction inside the thread plus two xor-shuffles over the quad.  Every 16-bit output is packed
// as one register per (pixel, column pair), which is exactly what
//   * tcgen05.st.16x128b needs to put P / ds back into TMEM as the A operand of the next GEMM, and
//   * stmatrix.trans needs to lay [column][8 pixels] 16-byte rows into shared memory, from where
//     the warp copies whole 64-byte row segments to global memory with 128-bit accesses
// so the epilogue issues ~1 instruction per 2 outputs instead of ~4 per output.
// Masked words get their -inf through the tensor core: an extra K = 16 block whose A operand is a
// constant (k = 0 row of ones) and whose B operand holds 0 / -inf per word.

// per-warp staging geometry inside a [rows x 128 px] tile stored as two swizzled [rows x 64 px] boxes
struct StageAddr {
  uint32_t st;      // stmatrix.x4 row address of this lane for row block 0 (add 1024 per block of 8 rows)
  uint32_t st2[2];  // stmatrix.x2 row addresses for the pixel halves h = 0, 1 (matrices j = 0, 1 of that half)
  uint32_t ld;      // ld.shared address of this lane's 16-byte chunk for row block 0
  int row, pxc;     // row (0..7) and pixel offset (multiple of 8, relative to the tile) of that chunk
};
__device__ __forceinline__ StageAddr stage_addr(uint32_t base, int rows, int q, int lane) {
  StageAddr a;
  const uint32_t box = base + (uint32_t)(q >> 1) * (uint32_t)(rows * 128);
  const int sr = lane & 7, sm = lane >> 3;
  a.st = box + sr * 128 + (((((q & 1) << 2) + sm) ^ sr) << 4);
  a.st2[0] = box + sr * 128 + (((((q & 1) << 2) + (sm & 1)) ^ sr) << 4);
  a.st2[1] = box + sr * 128 + (((((q & 1) << 2) + 2 + (sm & 1)) ^ sr) << 4);
  // rows r and r + 4 keep their chunks in opposite halves of the 128-byte line: pairing them inside a
  // quarter-warp makes the 128-bit reads conflict-free
  a.row = ((lane >> 2) & 1) * 4 + (lane >> 3);
  const int cq = lane & 3;
  a.ld = box + a.row * 128 + (((((q & 1) << 2) + cq) ^ (a.row & 7)) << 4);
  a.pxc = q * 32 + cq * 8;
  return a;
}

// softmax over the KB*8 columns of the two pixel rows (j = 0, 1) of one 16-lane half; v[4k + 2j + e]
template <int KB>
__device__ __forceinline__ void frag_softmax(float (&v)[4 * KB]) {
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    float mx = fmaxf(v[2 * j], v[2 * j + 1]);
#pragma unroll
    for (int k = 1; k < KB; ++k) mx = fmaxf(mx, fmaxf(v[4 * k + 2 * j], v[4 * k + 2 * j + 1]));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < KB; ++k)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float x = exp2f(v[4 * k + 2 * j + e] - mx);   // all masked: (-inf) - (-inf) = NaN, like the reference
        v[4 * k + 2 * j + e] = x;
        sum += x;
      }
    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
    const float inv = __fdividef(1.f, sum);
#pragma unroll
    for (int k = 0; k < KB; ++k)
#pragma unroll
      for (int e = 0; e < 2; ++e) v[4 * k + 2 * j + e] *= inv;
  }
}

// constant operands of the mask-bias MMA: sOnes = MN-major [16 k][128 px] (two 64-px halves, 2 KB
// apart) with k = 0 all ones; sBias = K-major [NT words][64 k] with k = 0 holding 0 or -inf
template <typename IO>
__device__ __forceinline__ void fill_mask_operands(unsigned char* sOnes, unsigned char* sBias, int NT,
                                                   const int64_t* mask_b, int T) {
  for (int i = threadIdx.x; i < 4096 / 16; i += blockDim.x) {
    const int row = (i >> 3) & 15;       // 16 rows of 128 B per half
    const uint32_t one2 = pack2<IO>(1.f, 1.f);
    reinterpret_cast<uint4*>(sOnes)[i] = row == 0 ? make_uint4(one2, one2, one2, one2) : make_uint4(0, 0, 0, 0);
  }
  for (int i = threadIdx.x; i < NT * 128 / 16; i += blockDim.x) reinterpret_cast<uint4*>(sBias)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  for (int t = threadIdx.x; t < NT; t += blockDim.x) {
    const bool keep = t < T && mask_b[t] != 0;
    *reinterpret_cast<IO*>(sBias + sw128_off(t, 0)) = f2h<IO>(keep ? 0.f : -INFINITY);
  }
}

// Persistent CTAs.  The B * tiles pixel tiles of the launch are split into gridDim.x contiguous,
// balanced ranges; a range that crosses a sample boundary is processed as two (or more) segments,
// each with its own W.e / mask operands.  Warp roles (320 threads): 0 = TMA producer (runs ahead across
// segments), 1 = MMA issuer, 2-5 = softmax warps (S -> P), 6-9 = output warps (ctx and attention maps
// -> global).  Warps 1-9 rebuild the operands between segments behind a named barrier.
// TL = word columns the epilogue touches (T rounded up to 8); NT = MMA N (32 or 64); CT = channels
constexpr int kFwdThreads = 320;
template <int NT, int CT> constexpr int fwd_min_ctas() { return (NT == 32 && CT <= 32) ? 3 : (CT <= 32 ? 2 : 1); }

// Persistent grid size: balanced contiguous ranges over all B * tiles tiles, one CTA per slot.  (A plan
// with k CTAs per sample never crosses a sample boundary, but its CTAs all walk the same offsets inside
// their rows at the same time and camp on a few DRAM channels: measured 1.4x slower at 128x128, B = 64.)
static int persistent_grid(long long slots, int B, int tiles) {
  return (int)std::min(slots, (long long)B * tiles);
}

struct Segment { int b, tile0, n; };
// next segment of the global tile range [g, g1): the tiles of one sample
__device__ __forceinline__ Segment next_segment(long long g, long long g1, int tiles) {
  Segment s;
  s.b = (int)(g / tiles);
  s.tile0 = (int)(g - (long long)s.b * tiles);
  s.n = (int)(((long long)(tiles - s.tile0) < g1 - g) ? (long long)(tiles - s.tile0) : g1 - g);
  return s;
}

// kNHWC: channels_last maps.  The h tile is C/16 K-major slabs (see kSlabBytes), and the output warps read
// ctx and the packed attention maps thread = pixel and store each pixel's contiguous C-vector and T-row.
template <typename IO, int NT, int TL, int CT, bool kNHWC = false>
__global__ void __launch_bounds__(kFwdThreads, (fwd_min_ctas<NT, CT>()))
word_attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap mapH, const AttnFwdParams p) {
  constexpr int KB = TL / 8;
  constexpr int C = CT;
  const int nst = p.stages;                      // depth of the h-tile ring (2..kMaxAttnStages)
  extern __shared__ __align__(1024) unsigned char smem[];
  constexpr int box_bytes = C * 128;             // one [C x 64 px] box
  constexpr int stage_bytes = 2 * box_bytes;
  unsigned char* sH = smem;
  unsigned char* sB1hi = smem + nst * stage_bytes;   // [NT rows t][64 k=c]  io type
  unsigned char* sB1lo = sB1hi + NT * 128;
  unsigned char* sB2hi = sB1lo + NT * 128;                   // [C rows c][64 k=t]   fp16
  unsigned char* sB2lo = sB2hi + box_bytes;
  unsigned char* sOnes = sB2lo + box_bytes;                  // 4 KB
  unsigned char* sBias = sOnes + 4096;                       // [NT rows t][64 k]
  unsigned char* sStA = sBias + NT * 128;                    // attn staging: 2 boxes x [TL rows][64 px]
  unsigned char* sStC = sStA + 2 * TL * 128;                 // ctx staging:  2 boxes x [C rows][64 px]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStC + 2 * box_bytes);
  uint64_t* h_full = bars;                                   // [kMaxAttnStages]
  uint64_t* h_empty = h_full + kMaxAttnStages;               // [kMaxAttnStages]
  uint64_t* s_full = h_empty + kMaxAttnStages;               // [2]
  uint64_t* p_ready = s_full + 2;                            // [2]
  uint64_t* c_full = p_ready + 2;                            // [2]
  uint64_t* c_empty = c_full + 2;                            // [2]
  uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(c_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int bufc = NT + C;                   // TMEM columns of one tile buffer: scores/P + context
  constexpr uint32_t tmem_cols = 2 * bufc <= 128 ? 128u : 256u;
  const long long total = (long long)p.B * p.tiles;
  const long long g0 = total * blockIdx.x / gridDim.x, g1 = total * (blockIdx.x + 1) / gridDim.x;

  if (threadIdx.x == 0) {
    for (int i = 0; i < nst; ++i) {
      mbar_init(&h_full[i], 1);
      mbar_init(&h_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 4);
      mbar_init(&c_full[i], 1);
      mbar_init(&c_empty[i], 4);
    }
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_base_s, tmem_cols);
  // constant operand of the mask-bias MMA; the per-sample bias column is rewritten per segment
  for (int i = threadIdx.x; i < 4096 / 16; i += blockDim.x) {
    const uint32_t one2 = pack2<IO>(1.f, 1.f);
    reinterpret_cast<uint4*>(sOnes)[i] = ((i >> 3) & 15) == 0 ? make_uint4(one2, one2, one2, one2) : make_uint4(0, 0, 0, 0);
  }
  for (int i = threadIdx.x; i < NT * 128 / 16; i += blockDim.x) reinterpret_cast<uint4*>(sBias)[i] = make_uint4(0, 0, 0, 0);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_base_s;
  constexpr int fmt_io = std::is_same<IO, __nv_bfloat16>::value ? 1 : 0;
  const int q = warp & 3;
  const uint32_t lane0 = (uint32_t)(q * 32) << 16;
  const size_t row8 = (size_t)8 * p.HW;

  if (warp == 0) {
    // ===================== TMA producer: h tiles of all segments =====================
    if (elect_one()) {
      int it = 0;
      for (long long g = g0; g < g1;) {
        const Segment sg = next_segment(g, g1, p.tiles);
        for (int i = 0; i < sg.n; ++i, ++it) {
          const int s = it % nst, use = it / nst;
          mbar_wait(&h_empty[s], (use & 1) ^ 1);
          mbar_expect_tx(&h_full[s], (uint32_t)stage_bytes);
          if constexpr (kNHWC) {
#pragma unroll
            for (int k = 0; k < C / 16; ++k)
              tma_load_3d(sH + s * stage_bytes + k * kSlabBytes, &mapH, &h_full[s], 16 * k, (sg.tile0 + i) * 128, sg.b);
          } else {
            tma_load_2d(sH + s * stage_bytes, &mapH, &h_full[s], (sg.tile0 + i) * 128, sg.b * C);
            tma_load_2d(sH + s * stage_bytes + box_bytes, &mapH, &h_full[s], (sg.tile0 + i) * 128 + 64, sg.b * C);
          }
        }
        g += sg.n;
      }
    }
  } else {
    const int tid = threadIdx.x - 32;            // 0..287 over warps 1-9
    int it0 = 0;                                 // tiles of earlier segments (mbarrier phases run on)
    for (long long g = g0; g < g1;) {
      const Segment sg = next_segment(g, g1, p.tiles);
      const int b = sg.b;
      const int ntile = (AGB_ABL(p, 16) && warp != 1) ? 0 : sg.n;
      // ---- operands of this sample: W.e hi + lo 16-bit split, K-major swizzled rows; mask bias ----
      {
        const float* we = p.we + (size_t)b * C * p.T;
        for (int i = tid; i < NT * C; i += kFwdThreads - 32) {        // B1[t][c]
          const int t = i / C, c = i - t * C;
          const float x = t < p.T ? we[c * p.T + t] * p.qscale : 0.f;
          const IO hi = f2h<IO>(x);
          const IO lo = f2h<IO>(x - to_f32(hi));
          *reinterpret_cast<IO*>(sB1hi + sw128_off(t, c)) = hi;
          *reinterpret_cast<IO*>(sB1lo + sw128_off(t, c)) = lo;
        }
        for (int i = tid; i < C * NT; i += kFwdThreads - 32) {        // B2[c][t]
          const int c = i / NT, t = i - c * NT;
          const float x = t < p.T ? we[c * p.T + t] : 0.f;
          const __half hi = __float2half_rn(x);
          const __half lo = __float2half_rn(x - __half2float(hi));
          *reinterpret_cast<__half*>(sB2hi + sw128_off(c, t)) = hi;
          *reinterpret_cast<__half*>(sB2lo + sw128_off(c, t)) = lo;
        }
        for (int t = tid; t < NT; t += kFwdThreads - 32) {
          const bool keep = t < p.T && p.mask[(size_t)b * p.T + t] != 0;
          *reinterpret_cast<IO*>(sBias + sw128_off(t, 0)) = f2h<IO>(keep ? 0.f : -INFINITY);
        }
        fence_proxy_async();
        named_bar_sync(1, kFwdThreads - 32);
      }
      if (warp == 1) {
        // ===================== MMA issuer =====================
        if (elect_one()) {
          constexpr uint32_t idesc1 = make_idesc(128, NT, fmt_io) | (1u << 15);   // A MN-major (pixels contiguous)
          constexpr uint32_t idesc2 = make_idesc(128, C, 0);                       // P (TMEM) x W.e, fp16
          constexpr int ks1 = C >> 4, ks2 = (TL + 15) >> 4;
          const uint64_t d_ones = make_desc_sw128_mn_lbo(smem_u32(sOnes), 2048u);
          const uint64_t d_bias = make_desc_sw128(smem_u32(sBias));
          tc_fence_after();
          // event-driven issue: GEMM1 of tile j1 needs its h tile and the TMEM buffer (output warps done
          // with tile j1 - 2); GEMM2 of tile j2 needs P from the softmax warps.  Neither blocks the other.
          int j1 = 0, j2 = 0;
          if (AGB_ABL(p, 16)) {                       // tuning: pure TMA streaming rate
            for (int j = 0; j < ntile; ++j) {
              mbar_wait(&h_full[(it0 + j) % nst], ((it0 + j) / nst) & 1);
              mbar_arrive(&h_empty[(it0 + j) % nst]);
            }
            j2 = ntile;
          }
          while (j2 < ntile) {
            const int i1 = it0 + j1, i2 = it0 + j2;
            if (j1 < ntile && j1 < j2 + 2 && mbar_try_wait(&h_full[i1 % nst], (i1 / nst) & 1) &&
                (i1 < 2 || mbar_try_wait(&c_empty[i1 & 1], ((i1 - 2) >> 1) & 1))) {
              const int s = i1 % nst, u = i1 & 1;
              tc_fence_after();
              const uint32_t a0 = smem_u32(sH + s * stage_bytes);
              umma_f16(tmem + u * bufc, d_ones, d_bias, idesc1, 0u);            // S = 0 / -inf per word
#pragma unroll
              for (int kk = 0; kk < ks1; ++kk) {
                if constexpr (kNHWC) {
                  constexpr uint32_t idesc1k = make_idesc(128, NT, fmt_io);                // A K-major (channels contiguous)
                  const uint64_t da = make_desc_sw32(a0 + kk * kSlabBytes, 0u);
                  umma_f16(tmem + u * bufc, da, make_desc_sw128(smem_u32(sB1hi)) + 2 * kk, idesc1k, 1u);
                  umma_f16(tmem + u * bufc, da, make_desc_sw128(smem_u32(sB1lo)) + 2 * kk, idesc1k, 1u);
                } else {
                const uint64_t da = make_desc_sw128_mn_lbo(a0 + kk * 2048, (uint32_t)box_bytes);
                umma_f16(tmem + u * bufc, da, make_desc_sw128(smem_u32(sB1hi)) + 2 * kk, idesc1, 1u);
                umma_f16(tmem + u * bufc, da, make_desc_sw128(smem_u32(sB1lo)) + 2 * kk, idesc1, 1u);
                }
              }
              umma_commit(&h_empty[s]);
              umma_commit(&s_full[u]);
              ++j1;
            }
            if (j2 < j1 && mbar_try_wait(&p_ready[i2 & 1], (i2 >> 1) & 1)) {
              const int u = i2 & 1;
              tc_fence_after();
#pragma unroll
              for (int kk = 0; kk < ks2; ++kk) {
                umma_f16_ts(tmem + u * bufc + NT, tmem + u * bufc + kk * 8, make_desc_sw128(smem_u32(sB2hi)) + 2 * kk,
                            idesc2, kk ? 1u : 0u);
                umma_f16_ts(tmem + u * bufc + NT, tmem + u * bufc + kk * 8, make_desc_sw128(smem_u32(sB2lo)) + 2 * kk,
                            idesc2, 1u);
              }
              umma_commit(&c_full[u]);
              ++j2;
            }
          }
        }
        __syncwarp();
      } else if (warp < 6) {
        // ===================== softmax warps: thread = pixel, no cross-lane traffic =====================
        // P (fp16 pairs) -> TMEM columns [0, NT/2) of the buffer = A operand of GEMM2.  The attention maps
        // in the caller's dtype go to columns [NT/2, NT) as packed pairs; the output warps read them back
        // in the 16x128b fragment layout, which transposes them for stmatrix (fp16 maps: P itself is read).
        const bool want_attn = p.attn != nullptr;
        for (int j = 0; j < ntile; ++j) {
          const int it = it0 + j, u = it & 1, k = it >> 1;
          mbar_wait(&s_full[u], k & 1);
          tc_fence_after();
          if (AGB_ABL(p, 4)) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&p_ready[u]);
            continue;
          }
          float v[TL];
          tmem_ld_cols<TL>(tmem + lane0 + u * bufc, v);
          tmem_ld_wait();
          float mx = fmaxf(v[0], v[1]);
#pragma unroll
          for (int t = 2; t < TL; t += 2) mx = fmaxf(mx, fmaxf(v[t], v[t + 1]));
          float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int t = 0; t < TL; ++t) {
            v[t] = exp2f(v[t] - mx);             // all masked: (-inf) - (-inf) = NaN, like the reference
            s4[t & 3] += v[t];
          }
          const float inv = __fdividef(1.f, (s4[0] + s4[1]) + (s4[2] + s4[3]));
          uint32_t pk[NT / 2];
#pragma unroll
          for (int t = 0; t < NT; t += 2) {
            if (t < TL) {
              v[t] *= inv;
              v[t + 1] *= inv;
              pk[t / 2] = pack2<__half>(v[t], v[t + 1]);
            } else {
              pk[t / 2] = 0u;
            }
          }
          tmem_st_n<NT / 2>(tmem + lane0 + u * bufc, pk);
          if constexpr (!std::is_same<IO, __half>::value) {
            if (want_attn) {
              uint32_t pa[TL / 2];
#pragma unroll
              for (int t = 0; t < TL; t += 2) pa[t / 2] = pack2<IO>(v[t], v[t + 1]);
              tmem_st_n<TL / 2>(tmem + lane0 + u * bufc + NT / 2, pa);
            }
          }
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&p_ready[u]);
        }
      } else {
        // ===================== output warps: ctx and attention maps -> global =====================
        IO* ctx = (IO*)p.ctx + (size_t)b * p.ctx_bs;
        IO* attn = p.attn ? (IO*)p.attn + (size_t)b * p.T * p.HW : nullptr;
        const StageAddr sc = stage_addr(smem_u32(sStC), C, q, lane);
        const StageAddr sa = stage_addr(smem_u32(sStA), TL, q, lane);
        constexpr int kAttnCol = std::is_same<IO, __half>::value ? 0 : NT / 2;
        for (int j = 0; j < ntile; ++j) {
          const int it = it0 + j, u = it & 1, k = it >> 1;
          mbar_wait(&c_full[u], k & 1);
          tc_fence_after();
          if (AGB_ABL(p, 8)) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&c_empty[u]);
            continue;
          }
          if constexpr (kNHWC) {
            // thread = pixel: its C context values and its T probabilities go to this warp's staging rows
            // ([32 px][C] and [32 px][T], 16-bit), TMEM read 16 columns at a time so the live set fits the 64
            // registers of three CTAs per SM; the warp then copies its 32 pixels out with 16-byte accesses on
            // consecutive addresses (a warp's maps are one contiguous block, its contexts C-vectors ctx_ps apart)
            unsigned char* wc = sStC + q * (32 * C * 2);
            unsigned char* wa = sStA + q * (32 * TL * 2);
#pragma unroll
            for (int c0 = 0; c0 < C; c0 += 16) {
              float cv[16];
              tmem_ld16(tmem + lane0 + u * bufc + NT + c0, cv);
              tmem_ld_wait();
#pragma unroll
              for (int c = 0; c < 16; c += 8)
                *reinterpret_cast<uint4*>(wc + (lane * C + c0 + c) * 2) =
                    make_uint4(pack2<IO>(cv[c], cv[c + 1]), pack2<IO>(cv[c + 2], cv[c + 3]),
                               pack2<IO>(cv[c + 4], cv[c + 5]), pack2<IO>(cv[c + 6], cv[c + 7]));
            }
            if (attn != nullptr) {
              float pv[TL / 2];
              tmem_ld_n<TL / 2>(tmem + lane0 + u * bufc + kAttnCol, pv);
              tmem_ld_wait();
              unsigned char* row = wa + lane * p.T * 2;
              if ((p.T & 1) == 0) {
#pragma unroll
                for (int t = 0; t < TL; t += 2)
                  if (t < p.T) *reinterpret_cast<uint32_t*>(row + t * 2) = __float_as_uint(pv[t / 2]);
              } else {           // odd T: rows are 2-byte aligned only
#pragma unroll
                for (int t = 0; t < TL; t += 2) {
                  const uint32_t pr = __float_as_uint(pv[t / 2]);
                  if (t < p.T) *reinterpret_cast<uint16_t*>(row + t * 2) = (uint16_t)(pr & 0xffffu);
                  if (t + 1 < p.T) *reinterpret_cast<uint16_t*>(row + t * 2 + 2) = (uint16_t)(pr >> 16);
                }
              }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&c_empty[u]);
            const int pix0 = (sg.tile0 + j) * 128 + q * 32;
            const int nvp = max(0, min(32, p.HW - pix0));         // a multiple of 8 (HW % 8 == 0)
            if (!AGB_ABL(p, 1)) {
              for (int i = lane; i < nvp * (C / 8); i += 32) {
                const int px = i / (C / 8), part = i - px * (C / 8);
                *reinterpret_cast<uint4*>(ctx + (size_t)(pix0 + px) * p.ctx_ps + part * 8) =
                    *reinterpret_cast<const uint4*>(wc + i * 16);
              }
            }
            if (attn != nullptr && !AGB_ABL(p, 2)) {
              uint4* dst = reinterpret_cast<uint4*>(attn + (size_t)pix0 * p.T);   // 16-byte aligned: pix0 % 8 == 0
              for (int i = lane; i < nvp * p.T / 8; i += 32) dst[i] = *reinterpret_cast<const uint4*>(wa + i * 16);
            }
            __syncwarp();
            continue;
          }
          float w[2][4 * (C / 8)];
          uint32_t pa[2][2 * KB];
          tmem_ld_frag<C / 8>(tmem + lane0 + u * bufc + NT, w[0]);
          tmem_ld_frag<C / 8>(tmem + lane0 + kHalfLanes + u * bufc + NT, w[1]);
          if (attn != nullptr) {
            tmem_ld_packed<KB>(tmem + lane0 + u * bufc + kAttnCol, pa[0]);
            tmem_ld_packed<KB>(tmem + lane0 + kHalfLanes + u * bufc + kAttnCol, pa[1]);
          }
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&c_empty[u]);
#pragma unroll
          for (int kk = 0; kk < C / 8; ++kk) {
            uint32_t r[4];
#pragma unroll
            for (int m = 0; m < 4; ++m)
              r[m] = pack2<IO>(w[m >> 1][4 * kk + 2 * (m & 1)], w[m >> 1][4 * kk + 2 * (m & 1) + 1]);
            stsm_x4_trans(sc.st + kk * 1024, r[0], r[1], r[2], r[3]);
          }
          if (attn != nullptr) {
#pragma unroll
            for (int kk = 0; kk < KB; ++kk)
              stsm_x4_trans(sa.st + kk * 1024, pa[0][2 * kk], pa[0][2 * kk + 1], pa[1][2 * kk], pa[1][2 * kk + 1]);
          }
          __syncwarp();
          {
            const int pix = (sg.tile0 + j) * 128 + sc.pxc;
            IO* dst = ctx + (size_t)sc.row * p.HW + pix;
#pragma unroll
            for (int i = 0; i < C / 8; ++i) {
              if (pix < p.HW && !AGB_ABL(p, 1)) *reinterpret_cast<uint4*>(dst) = lds128(sc.ld + i * 1024);
              dst += row8;
            }
          }
          if (attn != nullptr) {
            const int pix = (sg.tile0 + j) * 128 + sa.pxc;
            IO* dst = attn + (size_t)sa.row * p.HW + pix;
#pragma unroll
            for (int i = 0; i < KB; ++i) {
              if (sa.row + 8 * i < p.T && pix < p.HW && !AGB_ABL(p, 2)) *reinterpret_cast<uint4*>(dst) = lds128(sa.ld + i * 1024);
              dst += row8;
            }
          }
          __syncwarp();
        }
      }
      // the output warps have seen the last GEMM2 of the segment complete: operands may be rewritten
      named_bar_sync(1, kFwdThreads - 32);
      it0 += sg.n;
      g += sg.n;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, tmem_cols);
}

// 3-D map of a channels_last 16-bit tensor: element (c, p, b) at base + (c + p*ps + b*bs) elements; box =
// one [128 px][16 ch] slab, SWIZZLE_32B; pixels p >= HW (the tail of a sample's last tile) read as zeros
static int make_tmap_nhwc(CUtensorMap* map, const void* base, int C, int HW, int B, int64_t ps, int64_t bs, bool bf16) {
  static EncodeTiledFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || fn == nullptr) {
      set_error("cuTensorMapEncodeTiled entry point unavailable: %s", cudaGetErrorString(e));
      return e != cudaSuccess ? (int)e : (int)cudaErrorUnknown;
    }
    encode = (EncodeTiledFn)fn;
  }
  const cuuint64_t gdim[3] = {(cuuint64_t)C, (cuuint64_t)HW, (cuuint64_t)B};
  const cuuint64_t gstride[2] = {(cuuint64_t)ps * 2, (cuuint64_t)bs * 2};
  const cuuint32_t box[3] = {16, 128, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = encode(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                      const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (NHWC) failed with CUresult %d (C=%d HW=%d B=%d ps=%lld bs=%lld)", (int)r, C, HW,
              B, (long long)ps, (long long)bs);
    return (int)cudaErrorInvalidValue;
  }
  return 0;
}

template <typename IO, int CT, bool kNHWC>
static int launch_attn_fwd_tc_c(const CUtensorMap& mapH, const AttnFwdParams& p_in, int sms, cudaStream_t st) {
  const int NT = p_in.T <= 32 ? 32 : 64;
  const int TL = (p_in.T + 7) / 8 * 8;
  const int fixed = 2 * NT * 128 + 2 * CT * 128 + 4096 + NT * 128 + 2 * TL * 128 + 2 * CT * 128 + 256;
  const int per_sm = NT == 32 && CT <= 32 ? 3 : (CT <= 32 ? 2 : 1);
  // deepest h-tile ring that still lets per_sm CTAs share the SM's 227 KB (1 KB reserved per CTA)
  int stages = ((227 * 1024) / per_sm - 1024 - fixed) / (2 * CT * 128);
  stages = std::max(2, std::min(kMaxAttnStages, stages));
  if (options().attn_fwd_stages > 0) stages = std::max(2, std::min(kMaxAttnStages, options().attn_fwd_stages));   // tuning knob
  AttnFwdParams p = p_in;
  p.stages = stages;
  const int smem = stages * 2 * CT * 128 + fixed;
  int grid = persistent_grid((long long)sms * per_sm, p.B, p.tiles);
  if (options().attn_fwd_ctas > 0)   // tuning knob
    grid = (int)std::min<long long>(options().attn_fwd_ctas, (long long)p.B * p.tiles);
#define AGB_ATTN_FWD_CASE(NTV, TLV)                                                              \
  {                                                                                               \
    auto kern = word_attn_fwd_tc_kernel<IO, NTV, TLV, CT, kNHWC>;                                 \
    AGB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));      \
    kern<<<grid, kFwdThreads, smem, st>>>(mapH, p);                                               \
  }
  switch ((p.T + 7) / 8) {
    case 1: AGB_ATTN_FWD_CASE(32, 8) break;
    case 2: AGB_ATTN_FWD_CASE(32, 16) break;
    case 3: AGB_ATTN_FWD_CASE(32, 24) break;
    case 4: AGB_ATTN_FWD_CASE(32, 32) break;
    case 5: AGB_ATTN_FWD_CASE(64, 40) break;
    case 6: AGB_ATTN_FWD_CASE(64, 48) break;
    case 7: AGB_ATTN_FWD_CASE(64, 56) break;
    default: AGB_ATTN_FWD_CASE(64, 64) break;
  }
#undef AGB_ATTN_FWD_CASE
  return 0;
}

template <typename IO, bool kNHWC = false>
static int launch_attn_fwd_tc(const void* images, const AttnFwdParams& p, cudaStream_t st) {
  CUtensorMap mapH;
  if (int rc = kNHWC ? make_tmap_nhwc(&mapH, images, p.C, p.HW, p.B, p.C, (int64_t)p.HW * p.C,
                                      std::is_same<IO, __nv_bfloat16>::value)
                     : make_tmap_2d(&mapH, images, (uint64_t)p.B * p.C, (uint64_t)p.HW, (uint32_t)p.C,
                                    std::is_same<IO, __nv_bfloat16>::value))
    return rc;
  const int sms = device_sms();
  const int slot = prof_begin(PROF_ATTN_FWD, st);
  int rc = 0;
  switch (p.C) {
    case 16: rc = launch_attn_fwd_tc_c<IO, 16, kNHWC>(mapH, p, sms, st); break;
    case 32: rc = launch_attn_fwd_tc_c<IO, 32, kNHWC>(mapH, p, sms, st); break;
    case 48: rc = launch_attn_fwd_tc_c<IO, 48, kNHWC>(mapH, p, sms, st); break;
    default: rc = launch_attn_fwd_tc_c<IO, 64, kNHWC>(mapH, p, sms, st); break;
  }
  if (rc) return rc;
  prof_end(slot, st);
  return check_launch("word_attn_fwd_tc_kernel");
}

// =============================================================================================
// backward                                                   (SURVEY row a4: autograd of a3)
//
//   per tile of 128 pixels (thread = pixel in the epilogues):
//   GEMM1a  S[px,t] = h^T (W.e) scale log2e          GEMM1b  G[px,t] = dctx^T (W.e)
//   epilogue 1: a = softmax_t(S), g = G (+ dattn), ds = a (g - sum_t a g);
//               ds -> TMEM as bf16 hi + lo (A operand of GEMM3); [a | ds] -> smem, transposed
//               (B operand of GEMM4)
//   GEMM3   dh[px,c] = sum_t ds[px,t] (W.e)[c,t] scale                        (A from TMEM)
//   GEMM4   acc[(dctx rows; h rows), (a cols | ds cols)] += [dctx; h][., px] [a | ds][px, .]
//           accumulated in TMEM over all tiles of the CTA; d(W.e) = acc[dctx, a] + scale acc[h, ds]
//   epilogue 2: dh -> global
// TMEM (256 columns): two tile buffers of 96 (S|P, G, dh) + 64 accumulator columns.
// =============================================================================================
struct AttnBwdParams {
  const float* we;
  const int64_t* mask;
  const void* dattn;      // [B, T, HW] io dtype or null
  void* dh;               // [B, C, HW]
  float* part;            // [B, part_slots, C, T] per-CTA partial d(W.e)
  int part_slots, stages;
  int B, C, HW, T;
  float scale;
  int tiles, ctas_per_sample;
  int d_rows;             // rows of the dctx tensor map per sample (= dctx batch stride / HW; C when contiguous)
};

constexpr int kBwdNT = 32;      // word columns of the two-CTAs-per-SM variant (T <= 32)
constexpr int kBwdNTLong = 64;  // long captions (32 < T <= 64, bf16 maps): one CTA per SM, 448 of the 512 TMEM columns

// Persistent CTAs over contiguous, balanced ranges of the B * tiles pixel tiles (segments per sample,
// see the forward kernel).  Warp roles (448 threads): 0 = TMA producer, 1 = MMA issuer, 2-5 / 6-9 =
// softmax warpgroups for the even / odd tiles (tile buffer u = it & 1 belongs to warpgroup u), 10-13 =
// dh warps.  Softmax threads own one pixel: S and G rows come from TMEM with 32x32b loads, the softmax
// and its backward need no cross-lane traffic, and the 16-bit results go back to TMEM as packed pairs:
//   cols [0,16) ds hi, [16,32) ds lo (bf16; A operand of GEMM3), [32,48) a, [48,64) ds in fp16 (fp16 maps)
// The same warp reads a / ds back in the 16x128b fragment layout and stmatrix.trans-es them into the
// K-major (over pixels) B operand of GEMM4 -- the transposition costs ~12 instructions per warp.
constexpr int kBwdThreads = 448;
constexpr int kMaxBwdStages = 4;

// TMEM columns per tile buffer u (UB = 2 NT + 32):  [0,NT) S -> ds hi | ds lo (bf16 pairs, NT/2 columns each),
// [NT,2NT) G -> a (pairs, TL/2 columns) | ds in fp16 (fp16 maps, at NT + NT/2), [2NT, 2NT+32) dh;  the d(W.e)
// accumulator [a part | ds part] (2 TL columns) follows the two buffers at 2 UB.
// kNHWC: channels_last maps.  A stage is [dctx slabs | h slabs] (see kSlabBytes): K-major A operands of GEMM1,
// and side by side the MN-major A operand [dctx channels; h channels] x pixels of GEMM4.  dattn rows and dh
// are read / written thread = pixel.
template <typename IO, int NT, int TL, int CT, bool kNHWC = false>
__global__ void __launch_bounds__(kBwdThreads, NT <= 32 ? 2 : 1)
word_attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap mapH, const __grid_constant__ CUtensorMap mapD,
                        const AttnBwdParams p) {
  static_assert(NT == 32 || NT == 64, "NT");
  static_assert(TL <= NT && TL % 8 == 0, "TL");
  static_assert(NT == 32 || !std::is_same<IO, __half>::value, "long captions: bf16 maps only");
  constexpr uint32_t UB = 2 * NT + 32;
  constexpr uint32_t kTmemCols = NT == 32 ? 256 : 512;
  constexpr int KB = TL / 8;
  constexpr int C = CT;
  const int nst = p.stages;
  extern __shared__ __align__(1024) unsigned char smem[];
  constexpr int box = C * 128;                   // one [C x 64 px] box
  constexpr int stage_bytes = 4 * box;           // dctx_lo | h_lo | dctx_hi | h_hi
  constexpr int bt_box = 2 * TL * 128;           // one [a rows | ds rows][64 px] box of the GEMM4 B operand
  unsigned char* sIn = smem;
  unsigned char* sB1s = smem + nst * stage_bytes;              // [t][c] scaled*log2e   hi, lo (io type)
  unsigned char* sB1u = sB1s + 2 * NT * 128;                   // [t][c] unscaled       hi, lo (io type)
  unsigned char* sB2 = sB1u + 2 * NT * 128;                    // [c][t] * scale        hi, lo (bf16), 32 rows each
  unsigned char* sBt = sB2 + 2 * 32 * 128;                     // 2 buffers x 2 px-chunks x [2TL rows][64 px]
  unsigned char* sOnes = sBt + 2 * 2 * bt_box;                 // mask-bias MMA operands (see the forward kernel)
  unsigned char* sBias = sOnes + 4096;
  unsigned char* sStD = sBias + NT * 128;                      // dh staging: 2 boxes x [C rows][64 px]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStD + 2 * box);
  uint64_t* in_full = bars;                                    // [kMaxBwdStages]
  uint64_t* in_empty = in_full + kMaxBwdStages;                // [kMaxBwdStages]
  uint64_t* s_full = in_empty + kMaxBwdStages;                 // [2]
  uint64_t* p_ready = s_full + 2;                              // [2]
  uint64_t* dh_full = p_ready + 2;                             // [2]
  uint64_t* dh_empty = dh_full + 2;                            // [2]
  uint64_t* acc_done = dh_empty + 2;                           // [1]
  uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(acc_done + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long total = (long long)p.B * p.tiles;
  const long long g0 = total * blockIdx.x / gridDim.x, g1 = total * (blockIdx.x + 1) / gridDim.x;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kMaxBwdStages; ++i) {
      mbar_init(&in_full[i], 1);
      mbar_init(&in_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 4);
      mbar_init(&dh_full[i], 1);
      mbar_init(&dh_empty[i], 4);
    }
    mbar_init(acc_done, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_base_s, kTmemCols);
  for (int i = threadIdx.x; i < 4096 / 16; i += blockDim.x) {
    const uint32_t one2 = pack2<IO>(1.f, 1.f);
    reinterpret_cast<uint4*>(sOnes)[i] = ((i >> 3) & 15) == 0 ? make_uint4(one2, one2, one2, one2) : make_uint4(0, 0, 0, 0);
  }
  for (int i = threadIdx.x; i < NT * 128 / 16; i += blockDim.x) reinterpret_cast<uint4*>(sBias)[i] = make_uint4(0, 0, 0, 0);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_base_s;
  constexpr int fmt_io = std::is_same<IO, __nv_bfloat16>::value ? 1 : 0;
  constexpr uint32_t kAccCol = 2 * UB;
  const int q = warp & 3;
  const uint32_t lane0 = (uint32_t)(q * 32) << 16;

  if (warp == 0) {
    // ===================== TMA producer: dctx and h tiles of all segments =====================
    if (elect_one()) {
      int it = 0;
      for (long long g = g0; g < g1;) {
        const Segment sg = next_segment(g, g1, p.tiles);
        for (int i = 0; i < sg.n; ++i, ++it) {
          const int s = it % nst, use = it / nst;
          const int px0 = (sg.tile0 + i) * 128;
          mbar_wait(&in_empty[s], (use & 1) ^ 1);
          mbar_expect_tx(&in_full[s], (uint32_t)stage_bytes);
          unsigned char* st = sIn + s * stage_bytes;
          if constexpr (kNHWC) {
#pragma unroll
            for (int k = 0; k < C / 16; ++k) {
              tma_load_3d(st + k * kSlabBytes, &mapD, &in_full[s], 16 * k, px0, sg.b);
              tma_load_3d(st + (C / 16 + k) * kSlabBytes, &mapH, &in_full[s], 16 * k, px0, sg.b);
            }
          } else {
          tma_load_2d(st, &mapD, &in_full[s], px0, sg.b * p.d_rows);
          tma_load_2d(st + box, &mapH, &in_full[s], px0, sg.b * C);
          tma_load_2d(st + 2 * box, &mapD, &in_full[s], px0 + 64, sg.b * p.d_rows);
          tma_load_2d(st + 3 * box, &mapH, &in_full[s], px0 + 64, sg.b * C);
          }
        }
        g += sg.n;
      }
    }
  } else {
    constexpr int kWorkers = kBwdThreads - 32;
    const int tid = threadIdx.x - 32;
    int it0 = 0, seg = 0;
    for (long long g = g0; g < g1; ++seg) {
      const Segment sg = next_segment(g, g1, p.tiles);
      const int b = sg.b, ntile = sg.n;
      {
        const float* we = p.we + (size_t)b * C * p.T;
        const float qs = p.scale * kLog2e;
        for (int i = tid; i < NT * C; i += kWorkers) {
          const int t = i / C, c = i - t * C;
          const float w = t < p.T ? we[c * p.T + t] : 0.f;
          const float xs = w * qs;
          IO hi = f2h<IO>(xs);
          *reinterpret_cast<IO*>(sB1s + sw128_off(t, c)) = hi;
          *reinterpret_cast<IO*>(sB1s + NT * 128 + sw128_off(t, c)) = f2h<IO>(xs - to_f32(hi));
          hi = f2h<IO>(w);
          *reinterpret_cast<IO*>(sB1u + sw128_off(t, c)) = hi;
          *reinterpret_cast<IO*>(sB1u + NT * 128 + sw128_off(t, c)) = f2h<IO>(w - to_f32(hi));
        }
        for (int i = tid; i < C * NT; i += kWorkers) {
          const int c = i / NT, t = i - c * NT;
          const float x = t < p.T ? we[c * p.T + t] * p.scale : 0.f;
          const __nv_bfloat16 hi = __float2bfloat16_rn(x);
          *reinterpret_cast<__nv_bfloat16*>(sB2 + sw128_off(c, t)) = hi;
          *reinterpret_cast<__nv_bfloat16*>(sB2 + 32 * 128 + sw128_off(c, t)) = __float2bfloat16_rn(x - __bfloat162float(hi));
        }
        for (int t = tid; t < NT; t += kWorkers) {
          const bool keep = t < p.T && p.mask[(size_t)b * p.T + t] != 0;
          *reinterpret_cast<IO*>(sBias + sw128_off(t, 0)) = f2h<IO>(keep ? 0.f : -INFINITY);
        }
        fence_proxy_async();
        named_bar_sync(1, kWorkers);
      }
      if (warp == 1) {
        // ===================== MMA issuer (event driven, see the forward kernel) =====================
        if (elect_one()) {
          constexpr uint32_t idesc1 = make_idesc(128, NT, fmt_io) | (1u << 15);
          constexpr uint32_t idesc3 = make_idesc(128, C, 1);               // ds (bf16, TMEM) x W.e (bf16)
          constexpr uint32_t idesc4 = make_idesc(128, 2 * TL, fmt_io);     // [dctx; h] x [a | ds], K-major over pixels
          constexpr int ks1 = C >> 4;
          const uint64_t d_ones = make_desc_sw128_mn_lbo(smem_u32(sOnes), 2048u);
          const uint64_t d_bias = make_desc_sw128(smem_u32(sBias));
          tc_fence_after();
          int j1 = 0, j2 = 0;
          while (j2 < ntile) {
            const int i1 = it0 + j1, i2 = it0 + j2;
            if (j1 < ntile && j1 < j2 + 2 && mbar_try_wait(&in_full[i1 % nst], (i1 / nst) & 1)) {
              const int u = i1 & 1;
              tc_fence_after();
              const uint32_t st = smem_u32(sIn + (i1 % nst) * stage_bytes);
              umma_f16(tmem + u * UB, d_ones, d_bias, idesc1, 0u);        // S = 0 / -inf per word
#pragma unroll
              for (int kk = 0; kk < ks1; ++kk) {
                if constexpr (kNHWC) {
                  constexpr uint32_t idesc1k = make_idesc(128, NT, fmt_io);                          // A K-major
                  const uint64_t dh_ = make_desc_sw32(st + (C / 16 + kk) * kSlabBytes, 0u);           // h
                  const uint64_t dd_ = make_desc_sw32(st + kk * kSlabBytes, 0u);                      // dctx
                  umma_f16(tmem + u * UB, dh_, make_desc_sw128(smem_u32(sB1s)) + 2 * kk, idesc1k, 1u);
                  umma_f16(tmem + u * UB, dh_, make_desc_sw128(smem_u32(sB1s + NT * 128)) + 2 * kk, idesc1k, 1u);
                  umma_f16(tmem + u * UB + NT, dd_, make_desc_sw128(smem_u32(sB1u)) + 2 * kk, idesc1k, kk ? 1u : 0u);
                  umma_f16(tmem + u * UB + NT, dd_, make_desc_sw128(smem_u32(sB1u + NT * 128)) + 2 * kk, idesc1k, 1u);
                } else {
                const uint64_t dh_ = make_desc_sw128_mn_lbo(st + box + kk * 2048, (uint32_t)(2 * box));    // h
                const uint64_t dd_ = make_desc_sw128_mn_lbo(st + kk * 2048, (uint32_t)(2 * box));          // dctx
                umma_f16(tmem + u * UB, dh_, make_desc_sw128(smem_u32(sB1s)) + 2 * kk, idesc1, 1u);
                umma_f16(tmem + u * UB, dh_, make_desc_sw128(smem_u32(sB1s + NT * 128)) + 2 * kk, idesc1, 1u);
                umma_f16(tmem + u * UB + NT, dd_, make_desc_sw128(smem_u32(sB1u)) + 2 * kk, idesc1, kk ? 1u : 0u);
                umma_f16(tmem + u * UB + NT, dd_, make_desc_sw128(smem_u32(sB1u + NT * 128)) + 2 * kk, idesc1, 1u);
                }
              }
              umma_commit(&s_full[u]);
              ++j1;
            }
            if (j2 < j1 && mbar_try_wait(&p_ready[i2 & 1], (i2 >> 1) & 1) &&
                (i2 < 2 || mbar_try_wait(&dh_empty[i2 & 1], ((i2 - 2) >> 1) & 1))) {
              const int u = i2 & 1, s = i2 % nst;
              tc_fence_after();
#pragma unroll
              for (int kk = 0; kk < NT / 16; ++kk) {      // dh = ds (hi + lo) x W.e (hi + lo), lo*lo dropped
                const uint32_t a_hi = tmem + u * UB + kk * 8, a_lo = tmem + u * UB + NT / 2 + kk * 8;
                const uint64_t b_hi = make_desc_sw128(smem_u32(sB2)) + 2 * kk;
                const uint64_t b_lo = make_desc_sw128(smem_u32(sB2 + 32 * 128)) + 2 * kk;
                umma_f16_ts(tmem + u * UB + 2 * NT, a_hi, b_hi, idesc3, kk ? 1u : 0u);
                umma_f16_ts(tmem + u * UB + 2 * NT, a_lo, b_hi, idesc3, 1u);
                umma_f16_ts(tmem + u * UB + 2 * NT, a_hi, b_lo, idesc3, 1u);
              }
              umma_commit(&dh_full[u]);
              const uint32_t st = smem_u32(sIn + s * stage_bytes);
              const uint32_t bt = smem_u32(sBt + u * (2 * bt_box));
#pragma unroll
              for (int j = 0; j < 2; ++j)                  // two chunks of 64 pixels
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                  if constexpr (kNHWC) {
                    // [dctx; h] channels x 16 pixels: MN-major over the slabs (rows 2C..127 of M are not read back)
                    constexpr uint32_t idesc4m = make_idesc(128, 2 * TL, fmt_io) | (1u << 15);
                    umma_f16(tmem + kAccCol, make_desc_sw32(st + (4 * j + kk) * 512, (uint32_t)kSlabBytes),
                             make_desc_sw128(bt + j * bt_box) + 2 * kk, idesc4m, (j2 | j | kk) ? 1u : 0u);
                  } else {
                  umma_f16(tmem + kAccCol, make_desc_sw128(st + j * 2 * box) + 2 * kk,
                           make_desc_sw128(bt + j * bt_box) + 2 * kk, idesc4, (j2 | j | kk) ? 1u : 0u);
                  }
                }
              umma_commit(&in_empty[s]);
              ++j2;
            }
          }
          umma_commit(acc_done);
        }
        __syncwarp();
      } else if (warp < 10) {
        // ===================== softmax warpgroup u: thread = pixel =====================
        const int u = warp >= 6 ? 1 : 0;
        const IO* dattn = p.dattn ? (const IO*)p.dattn + (size_t)b * p.T * p.HW : nullptr;
        const uint32_t bt_st = stage_addr(smem_u32(sBt) + u * (2 * bt_box), 2 * TL, q, lane).st;
        constexpr bool kHalfIO = std::is_same<IO, __half>::value;
        for (int j = ((it0 & 1) == u ? 0 : 1); j < ntile; j += 2) {
          const int it = it0 + j, k = it >> 1;
          mbar_wait(&s_full[u], k & 1);
          tc_fence_after();
          if constexpr (NT <= 32) {
            float s[TL], g[TL];
            tmem_ld_cols<TL>(tmem + lane0 + u * UB, s);
            tmem_ld_cols<TL>(tmem + lane0 + u * UB + NT, g);
            tmem_ld_wait();
            float mx = fmaxf(s[0], s[1]);
#pragma unroll
            for (int t = 2; t < TL; t += 2) mx = fmaxf(mx, fmaxf(s[t], s[t + 1]));
            float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int t = 0; t < TL; ++t) {
              s[t] = exp2f(s[t] - mx);
              s4[t & 3] += s[t];
            }
            const float inv = __fdividef(1.f, (s4[0] + s4[1]) + (s4[2] + s4[3]));
            if (dattn != nullptr) {                      // rare: a gradient arrives through the attention maps too
              const int pix = (sg.tile0 + j) * 128 + q * 32 + lane;
#pragma unroll
              for (int t = 0; t < TL; ++t)
                if (t < p.T && pix < p.HW) g[t] += to_f32(dattn[kNHWC ? (size_t)pix * p.T + t : (size_t)t * p.HW + pix]);
            }
            float d4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int t = 0; t < TL; ++t) {
              s[t] *= inv;
              d4[t & 3] = fmaf(s[t], g[t], d4[t & 3]);
            }
            const float dot = (d4[0] + d4[1]) + (d4[2] + d4[3]);
            uint32_t hi[NT / 2], lo[NT / 2], pa[TL / 2];
            uint32_t ph[kHalfIO ? TL / 2 : 1];
#pragma unroll
            for (int t = 0; t < NT; t += 2) {
              if (t < TL) {
                const float d0 = s[t] * (g[t] - dot), d1 = s[t + 1] * (g[t + 1] - dot);
                const uint32_t h2 = pack2<__nv_bfloat16>(d0, d1);
                hi[t / 2] = h2;
                lo[t / 2] = pack2<__nv_bfloat16>(d0 - __uint_as_float(h2 << 16), d1 - __uint_as_float(h2 & 0xffff0000u));
                pa[t / 2] = pack2<IO>(s[t], s[t + 1]);
                if constexpr (kHalfIO) ph[t / 2] = pack2<IO>(d0, d1);
              } else {
                hi[t / 2] = 0u;
                lo[t / 2] = 0u;
              }
            }
            tmem_st_n<NT / 2>(tmem + lane0 + u * UB, hi);
            tmem_st_n<NT / 2>(tmem + lane0 + u * UB + NT / 2, lo);
            tmem_st_n<TL / 2>(tmem + lane0 + u * UB + NT, pa);
            if constexpr (kHalfIO) tmem_st_n<TL / 2>(tmem + lane0 + u * UB + NT + NT / 2, ph);
          } else {
            // long captions: the probabilities stay in registers (TL values), the upstream gradients G are streamed
            // from TMEM twice in chunks of 16 columns (dot product, then ds), so the live set stays near the
            // 128 registers of a one-CTA-per-SM kernel (the same chunking under the 72-register cap of the
            // two-CTAs-per-SM variant spills MORE than the straight version: measured with -Xptxas -v).  The packed results of chunk c land on columns that hold only consumed values:
            // ds hi / lo over S (already in registers), a over the first half of G (chunk c covers G columns
            // [16c, 16c+16), a of chunk c goes to [8c, 8c+8)).
            // The G chunks are double-buffered in registers: the load of chunk c+1 is issued before chunk c is
            // processed (and the first one before the exponentials), so one TMEM round trip per pass is exposed
            // instead of one per chunk.
            float s[TL];
            tmem_ld_cols<TL>(tmem + lane0 + u * UB, s);
            tmem_ld_wait();
            constexpr int kNch = (TL + 15) / 16;
            float gbuf[2][16];
            auto load_g = [&](float* g, int c0) {
              if (TL - c0 >= 16) tmem_ld16(tmem + lane0 + u * UB + NT + c0, g); else tmem_ld8(tmem + lane0 + u * UB + NT + c0, g);
            };
            load_g(gbuf[0], 0);
            float mx = fmaxf(s[0], s[1]);
#pragma unroll
            for (int t = 2; t < TL; t += 2) mx = fmaxf(mx, fmaxf(s[t], s[t + 1]));
            float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int t = 0; t < TL; ++t) {
              s[t] = exp2f(s[t] - mx);
              s4[t & 3] += s[t];
            }
            const float inv = __fdividef(1.f, (s4[0] + s4[1]) + (s4[2] + s4[3]));
            const int pix = (sg.tile0 + j) * 128 + q * 32 + lane;
            float d4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int c = 0; c < kNch; ++c) {
              const int c0 = c * 16;
              float* g = gbuf[c & 1];
              tmem_ld_wait();
              load_g(gbuf[(c + 1) & 1], c + 1 < kNch ? c0 + 16 : 0);      // next chunk, or chunk 0 again for the ds pass
#pragma unroll
              for (int t = 0; t < 16; ++t) {
                if (c0 + t < TL) {
                  if (dattn != nullptr && c0 + t < p.T && pix < p.HW)
                    g[t] += to_f32(dattn[kNHWC ? (size_t)pix * p.T + c0 + t : (size_t)(c0 + t) * p.HW + pix]);
                  s[c0 + t] *= inv;
                  d4[t & 3] = fmaf(s[c0 + t], g[t], d4[t & 3]);
                }
              }
            }
            const float dot = (d4[0] + d4[1]) + (d4[2] + d4[3]);
#pragma unroll
            for (int c = 0; c < NT / 16; ++c) {
              const int c0 = c * 16;
              uint32_t hi[8], lo[8], pa[8];
              if (c0 < TL) {
                float* g = gbuf[(kNch + c) & 1];
                tmem_ld_wait();
                if (c + 1 < kNch) load_g(gbuf[(kNch + c + 1) & 1], c0 + 16);
#pragma unroll
                for (int t = 0; t < 16; t += 2) {
                  if (c0 + t < TL) {
                    float g0 = g[t], g1 = g[t + 1];
                    if (dattn != nullptr && pix < p.HW) {
                      if (c0 + t < p.T) g0 += to_f32(dattn[kNHWC ? (size_t)pix * p.T + c0 + t : (size_t)(c0 + t) * p.HW + pix]);
                      if (c0 + t + 1 < p.T)
                        g1 += to_f32(dattn[kNHWC ? (size_t)pix * p.T + c0 + t + 1 : (size_t)(c0 + t + 1) * p.HW + pix]);
                    }
                    const float d0 = s[c0 + t] * (g0 - dot), d1 = s[c0 + t + 1] * (g1 - dot);
                    const uint32_t h2 = pack2<__nv_bfloat16>(d0, d1);
                    hi[t / 2] = h2;
                    lo[t / 2] = pack2<__nv_bfloat16>(d0 - __uint_as_float(h2 << 16), d1 - __uint_as_float(h2 & 0xffff0000u));
                    pa[t / 2] = pack2<IO>(s[c0 + t], s[c0 + t + 1]);
                  } else {
                    hi[t / 2] = 0u;
                    lo[t / 2] = 0u;
                    pa[t / 2] = 0u;
                  }
                }
                if (TL - c0 >= 16) tmem_st8(tmem + lane0 + u * UB + NT + c0 / 2, pa); else tmem_st4(tmem + lane0 + u * UB + NT + c0 / 2, pa);
              } else {
#pragma unroll
                for (int k = 0; k < 8; ++k) hi[k] = lo[k] = 0u;
              }
              tmem_st8(tmem + lane0 + u * UB + c0 / 2, hi);
              tmem_st8(tmem + lane0 + u * UB + NT / 2 + c0 / 2, lo);
            }
          }
          tmem_st_wait();
          // read a and ds back as stmatrix fragments: [a | ds] transposed into the B operand of GEMM4
          uint32_t fa[2][2 * KB], fd[2][2 * KB];
          constexpr int kDsCol = kHalfIO ? NT + NT / 2 : 0;
          tmem_ld_packed<KB>(tmem + lane0 + u * UB + NT, fa[0]);
          tmem_ld_packed<KB>(tmem + lane0 + kHalfLanes + u * UB + NT, fa[1]);
          tmem_ld_packed<KB>(tmem + lane0 + u * UB + kDsCol, fd[0]);
          tmem_ld_packed<KB>(tmem + lane0 + kHalfLanes + u * UB + kDsCol, fd[1]);
          tmem_ld_wait();
#pragma unroll
          for (int kk = 0; kk < KB; ++kk) {
            stsm_x4_trans(bt_st + kk * 1024, fa[0][2 * kk], fa[0][2 * kk + 1], fa[1][2 * kk], fa[1][2 * kk + 1]);
            stsm_x4_trans(bt_st + TL * 128 + kk * 1024, fd[0][2 * kk], fd[0][2 * kk + 1], fd[1][2 * kk], fd[1][2 * kk + 1]);
          }
          fence_proxy_async();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&p_ready[u]);
        }
      } else {
        // ===================== dh warps =====================
        const int px = q * 32 + lane;
        const int dtid = (warp - 10) * 32 + lane;
        IO* dh = (IO*)p.dh + (size_t)b * C * p.HW;
        const StageAddr sd = stage_addr(smem_u32(sStD), C, q, lane);
        const size_t row8 = (size_t)8 * p.HW;
        for (int j = 0; j < ntile; ++j) {
          const int it = it0 + j, u = it & 1, k = it >> 1;
          mbar_wait(&dh_full[u], k & 1);
          tc_fence_after();
          if constexpr (kNHWC) {
            // thread = pixel: its C gradient values go to this warp's staging rows [32 px][C], then the warp
            // copies its 32 pixels (one contiguous block of d images) out with 16-byte accesses
            unsigned char* wd = sStD + (px >> 5) * (32 * C * 2);
#pragma unroll
            for (int c0 = 0; c0 < C; c0 += 16) {
              float dv[16];
              tmem_ld16(tmem + lane0 + u * UB + 2 * NT + c0, dv);
              tmem_ld_wait();
#pragma unroll
              for (int c = 0; c < 16; c += 8)
                *reinterpret_cast<uint4*>(wd + (lane * C + c0 + c) * 2) =
                    make_uint4(pack2<IO>(dv[c], dv[c + 1]), pack2<IO>(dv[c + 2], dv[c + 3]),
                               pack2<IO>(dv[c + 4], dv[c + 5]), pack2<IO>(dv[c + 6], dv[c + 7]));
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&dh_empty[u]);
            const int pix0 = (sg.tile0 + j) * 128 + (px & ~31);
            const int nvp = max(0, min(32, p.HW - pix0));
            uint4* dst = reinterpret_cast<uint4*>((IO*)p.dh + ((size_t)b * p.HW + pix0) * C);
            for (int i = lane; i < nvp * C / 8; i += 32) dst[i] = *reinterpret_cast<const uint4*>(wd + i * 16);
            __syncwarp();
            continue;
          }
          float w[2][4 * (C / 8)];
          tmem_ld_frag<C / 8>(tmem + lane0 + u * UB + 2 * NT, w[0]);
          tmem_ld_frag<C / 8>(tmem + lane0 + kHalfLanes + u * UB + 2 * NT, w[1]);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&dh_empty[u]);
#pragma unroll
          for (int kk = 0; kk < C / 8; ++kk) {
            uint32_t r[4];
#pragma unroll
            for (int m = 0; m < 4; ++m)
              r[m] = pack2<IO>(w[m >> 1][4 * kk + 2 * (m & 1)], w[m >> 1][4 * kk + 2 * (m & 1) + 1]);
            stsm_x4_trans(sd.st + kk * 1024, r[0], r[1], r[2], r[3]);
          }
          __syncwarp();
          const int pix = (sg.tile0 + j) * 128 + sd.pxc;
          IO* dst = dh + (size_t)sd.row * p.HW + pix;
#pragma unroll
          for (int i = 0; i < C / 8; ++i) {
            if (pix < p.HW) *reinterpret_cast<uint4*>(dst) = lds128(sd.ld + i * 1024);
            dst += row8;
          }
          __syncwarp();
        }
        // ---- d(W.e) partial of this segment: part[b][slot], slot = index of this CTA among those of sample b ----
        {
          const long long first_cta = (((long long)b * p.tiles + 1) * gridDim.x + total - 1) / total - 1;
          float* part = p.part + ((size_t)b * p.part_slots + (size_t)(blockIdx.x - first_cta)) * C * p.T;
          float* sX = reinterpret_cast<float*>(sStD);          // [C][TL] exchange between the two row groups
          mbar_wait(acc_done, seg & 1);
          tc_fence_after();
          named_bar_sync(2, 128);                               // staging reads of the last tile are done
          {
            float vd[TL];
            tmem_ld_cols<TL>(tmem + lane0 + kAccCol + TL, vd);  // rows of h x columns of ds
            tmem_ld_wait();
            if (px >= C && px < 2 * C) {
#pragma unroll
              for (int t = 0; t < TL; ++t) sX[(px - C) * TL + t] = vd[t];
            }
          }
          named_bar_sync(2, 128);
          {
            float va[TL];
            tmem_ld_cols<TL>(tmem + lane0 + kAccCol, va);       // rows of dctx x columns of a
            tmem_ld_wait();
            tc_fence_before();
            if (px < C) {
#pragma unroll
              for (int t = 0; t < TL; ++t)
                if (t < p.T) part[px * p.T + t] = va[t] + p.scale * sX[px * TL + t];
            }
          }
          named_bar_sync(2, 128);
          (void)dtid;
        }
      }
      // dh warps have seen the accumulator of the segment complete: every MMA that reads the operands is done
      named_bar_sync(1, kWorkers);
      it0 += ntile;
      g += ntile;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, kTmemCols);
}

int word_attn_bwd_tc_supported(const void* images, const void* dctx, int64_t dctx_bs, const void* dattn, int C, int HW,
                               int T, int io_dtype) {
  if (io_dtype != AGB_BF16 && io_dtype != AGB_F16) return 0;
  if ((C != 16 && C != 32) || T > kBwdNTLong || HW % 8 != 0) return 0;
  if (T > kBwdNT && io_dtype != AGB_BF16) return 0;   // long captions: bf16 maps (fp16 would need a fourth packed operand in TMEM)
  // dctx may be a channel slice of a wider [B, C', HW] gradient (GenNextStage's concat buffer): whole rows only
  if (dctx_bs < (int64_t)C * HW || dctx_bs % HW != 0) return 0;
  if ((((uintptr_t)images | (uintptr_t)dctx) & 15) != 0) return 0;
  return 1;
}

// persistent grid of the backward kernel: 2 CTAs per SM (1 for long captions), never more CTAs than tiles
int word_attn_bwd_tc_grid(int B, int HW, int T) {
  const int sms = device_sms();
  if (options().attn_bwd_ctas > 0)   // tuning knob
    return (int)std::min<long long>(options().attn_bwd_ctas, (long long)B * cdiv(HW, 128));
  return persistent_grid((long long)sms * (T > kBwdNT ? 1 : 2), B, cdiv(HW, 128));
}

// number of per-sample partial-sum slots the backward kernel may write: the CTAs whose tile range
// overlaps one sample (ranges are floor(total/G) or one more tiles long)
int word_attn_bwd_tc_ctas(int B, int HW, int T) {
  const int tiles = cdiv(HW, 128);
  const long long total = (long long)B * tiles;
  const long long m = std::max<long long>(1, total / word_attn_bwd_tc_grid(B, HW, T));
  return (int)std::min<long long>(tiles, (tiles - 1) / m + 2);
}

// dwe[b][i] = sum over the slots sample b really has (fixed order -> deterministic)
__global__ void sum_range_partials_kernel(const float* __restrict__ part, int slots, int tiles, int G, long long total,
                                          int n, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
  if (i >= n) return;
  const long long first = (((long long)b * tiles + 1) * G + total - 1) / total - 1;
  const long long last = (((long long)(b + 1) * tiles) * G + total - 1) / total - 1;
  const float* p = part + (size_t)b * slots * n + i;
  float acc = 0.f;
  for (int k = 0; k <= (int)(last - first); ++k) acc += p[(size_t)k * n];
  out[(size_t)b * n + i] = acc;
}

// nhwc: channels_last maps, dctx with pixel stride dctx_ps
static int word_attn_bwd_tc_run(bool nhwc, const void* images, const float* we, const int64_t* mask, const void* dctx,
                                int64_t dctx_bs, int64_t dctx_ps, const void* dattn, void* dimages, float* part,
                                int part_slots, float* dwe, int B, int C, int HW, int T, int io_dtype, float scale,
                                cudaStream_t st) {
  const bool bf = io_dtype == AGB_BF16;
  CUtensorMap mapH, mapD;
  const int d_rows = nhwc ? 0 : (int)(dctx_bs / HW);
  if (nhwc) {
    if (int rc = make_tmap_nhwc(&mapH, images, C, HW, B, C, (int64_t)HW * C, bf)) return rc;
    if (int rc = make_tmap_nhwc(&mapD, dctx, C, HW, B, dctx_ps, dctx_bs, bf)) return rc;
  } else {
    if (int rc = make_tmap_2d(&mapH, images, (uint64_t)B * C, (uint64_t)HW, (uint32_t)C, bf)) return rc;
    if (int rc = make_tmap_2d(&mapD, dctx, (uint64_t)(B - 1) * d_rows + C, (uint64_t)HW, (uint32_t)C, bf)) return rc;
  }
  AttnBwdParams p;
  p.we = we; p.mask = mask; p.dattn = dattn; p.dh = dimages; p.part = part;
  p.B = B; p.C = C; p.HW = HW; p.T = T; p.scale = scale;
  p.tiles = cdiv(HW, 128);
  p.ctas_per_sample = 0;
  p.d_rows = d_rows;
  p.part_slots = part_slots;
  const int NT = T > kBwdNT ? kBwdNTLong : kBwdNT;
  const int per_sm = T > kBwdNT ? 1 : 2;
  const int TL = (T + 7) / 8 * 8;
  const int fixed = 4 * NT * 128 + 2 * 32 * 128 + 2 * 2 * (2 * TL) * 128 + 4096 + NT * 128 + 2 * C * 128 + 256;
  // deepest input ring that still lets per_sm CTAs share the SM's 227 KB (1 KB reserved per CTA)
  int stages = ((227 * 1024) / per_sm - 1024 - fixed) / (4 * C * 128);
  stages = std::max(2, std::min(kMaxBwdStages, stages));
  if (options().attn_bwd_stages > 0) stages = std::max(2, std::min(kMaxBwdStages, options().attn_bwd_stages));   // tuning knob
  p.stages = stages;
  const int smem = stages * 4 * C * 128 + fixed;
  const int grid = word_attn_bwd_tc_grid(B, HW, T);
  const int slot = prof_begin(PROF_ATTN_BWD, st);
#define AGB_ATTN_BWD_LAUNCH_L(IOT, NTV, TLV, CTV, L)                                              \
  {                                                                                               \
    auto kern = word_attn_bwd_tc_kernel<IOT, NTV, TLV, CTV, L>;                                   \
    AGB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));      \
    kern<<<grid, kBwdThreads, smem, st>>>(mapH, mapD, p);                                         \
  }
#define AGB_ATTN_BWD_LAUNCH(IOT, NTV, TLV, CTV)                                                    \
  if (nhwc) AGB_ATTN_BWD_LAUNCH_L(IOT, NTV, TLV, CTV, true) else AGB_ATTN_BWD_LAUNCH_L(IOT, NTV, TLV, CTV, false)
#define AGB_ATTN_BWD_CASE2(TLV, CTV)                                                              \
  if (bf) AGB_ATTN_BWD_LAUNCH(__nv_bfloat16, 32, TLV, CTV) else AGB_ATTN_BWD_LAUNCH(__half, 32, TLV, CTV)
#define AGB_ATTN_BWD_CASE(TLV)        \
  if (C == 16) {                      \
    AGB_ATTN_BWD_CASE2(TLV, 16)       \
  } else {                            \
    AGB_ATTN_BWD_CASE2(TLV, 32)       \
  }
#define AGB_ATTN_BWD_LONG(TLV)                                      \
  if (C == 16) AGB_ATTN_BWD_LAUNCH(__nv_bfloat16, 64, TLV, 16)      \
  else AGB_ATTN_BWD_LAUNCH(__nv_bfloat16, 64, TLV, 32)
  switch ((T + 7) / 8) {
    case 1: AGB_ATTN_BWD_CASE(8) break;
    case 2: AGB_ATTN_BWD_CASE(16) break;
    case 3: AGB_ATTN_BWD_CASE(24) break;
    case 4: AGB_ATTN_BWD_CASE(32) break;
    case 5: AGB_ATTN_BWD_LONG(40) break;
    case 6: AGB_ATTN_BWD_LONG(48) break;
    case 7: AGB_ATTN_BWD_LONG(56) break;
    default: AGB_ATTN_BWD_LONG(64) break;
  }
#undef AGB_ATTN_BWD_LAUNCH
#undef AGB_ATTN_BWD_LAUNCH_L
#undef AGB_ATTN_BWD_LONG
#undef AGB_ATTN_BWD_CASE2
#undef AGB_ATTN_BWD_CASE
  prof_end(slot, st);
  if (int rc = check_launch("word_attn_bwd_tc_kernel")) return rc;
  if (dwe == nullptr) return 0;                   // the caller reduces the partial slots itself
  sum_range_partials_kernel<<<dim3(cdiv(C * T, 128), B), 128, 0, st>>>(part, part_slots, p.tiles, grid,
                                                                       (long long)B * p.tiles, C * T, dwe);
  return check_launch("sum_range_partials_kernel");
}

int word_attn_bwd_tc(const void* images, const float* we, const int64_t* mask, const void* dctx, int64_t dctx_bs,
                     const void* dattn, void* dimages, float* part, int part_slots, float* dwe, int B, int C, int HW, int T, int io_dtype,
                     float scale, cudaStream_t st) {
  return word_attn_bwd_tc_run(false, images, we, mask, dctx, dctx_bs, 0, dattn, dimages, part, part_slots, dwe, B, C, HW,
                              T, io_dtype, scale, st);
}

int word_attn_bwd_tc_nhwc(const void* images, const float* we, const int64_t* mask, const void* dctx, int64_t dctx_bs,
                          int64_t dctx_ps, const void* dattn, void* dimages, float* part, int part_slots, int B, int C,
                          int HW, int T, int io_dtype, float scale, cudaStream_t st) {
  return word_attn_bwd_tc_run(true, images, we, mask, dctx, dctx_bs, dctx_ps, dattn, dimages, part, part_slots, nullptr,
                              B, C, HW, T, io_dtype, scale, st);
}

// NHWC takes the tensor-core kernels exactly where NCHW does (same dtype, C, T and HW rules, 16-byte aligned
// images and gradient), so the two layouts give the same results; the TMA map additionally needs 16-byte pixel and
// batch strides of dctx, which a channels_last tensor or its channel slice [:, C:] has whenever C % 16 == 0
int word_attn_bwd_tc_supported_nhwc(const void* images, const void* dctx, int64_t dctx_bs, int64_t dctx_ps,
                                    const void* dattn, int C, int HW, int T, int io_dtype) {
  if (!word_attn_bwd_tc_supported(images, dctx, (int64_t)C * HW, dattn, C, HW, T, io_dtype)) return 0;
  return dctx_ps % 8 == 0 && dctx_bs % 8 == 0;
}

// 1 when the tensor-core kernel can take this problem
int word_attn_tc_supported(const void* images, int C, int HW, int T, int io_dtype) {
  if (io_dtype != AGB_BF16 && io_dtype != AGB_F16) return 0;
  if (C % 16 != 0 || C < 16 || C > 64 || T > 64 || HW % 8 != 0) return 0;
  if (((uintptr_t)images & 15) != 0) return 0;
  return 1;
}

// the forward's NHWC rule: the NCHW one, plus 16-byte aligned ctx vectors and attention maps (the epilogue copies
// 16 bytes at a time)
int word_attn_tc_supported_nhwc(const void* images, const void* ctx, int64_t ctx_bs, int64_t ctx_ps, const void* attn,
                                int C, int HW, int T, int io_dtype) {
  if (!word_attn_tc_supported(images, C, HW, T, io_dtype)) return 0;
  return ((uintptr_t)ctx & 15) == 0 && ctx_ps % 8 == 0 && ctx_bs % 8 == 0 && ((uintptr_t)attn & 15) == 0;
}

int word_attn_fwd_tc_nhwc(const void* images, const float* we, const int64_t* mask, void* ctx, int64_t ctx_bs,
                          int64_t ctx_ps, void* attn, int B, int C, int HW, int T, int io_dtype, float qscale,
                          cudaStream_t st) {
  AttnFwdParams p;
  p.we = we; p.mask = mask; p.ctx = ctx; p.attn = attn; p.ctx_bs = ctx_bs; p.ctx_ps = ctx_ps;
  p.B = B; p.C = C; p.HW = HW; p.T = T; p.qscale = qscale;
  p.tiles = cdiv(HW, 128);
  p.ctas_per_sample = 0;
  p.dbg = 0;
#ifdef AGB_ABLATION
  if (const char* e = getenv("AGB_ATTN_DEBUG")) p.dbg = atoi(e);
#endif
  if (io_dtype == AGB_BF16) return launch_attn_fwd_tc<__nv_bfloat16, true>(images, p, st);
  return launch_attn_fwd_tc<__half, true>(images, p, st);
}

int word_attn_fwd_tc(const void* images, const float* we, const int64_t* mask, void* ctx, int64_t ctx_bs, void* attn,
                     int B, int C, int HW, int T, int io_dtype, float qscale, cudaStream_t st) {
  AttnFwdParams p;
  p.we = we; p.mask = mask; p.ctx = ctx; p.attn = attn; p.ctx_bs = ctx_bs; p.ctx_ps = 0;
  p.B = B; p.C = C; p.HW = HW; p.T = T; p.qscale = qscale;
  p.tiles = cdiv(HW, 128);
  p.ctas_per_sample = 0;   // the forward kernel is persistent over all samples
  p.dbg = 0;
#ifdef AGB_ABLATION
  if (const char* e = getenv("AGB_ATTN_DEBUG")) p.dbg = atoi(e);
#endif
  if (io_dtype == AGB_BF16) return launch_attn_fwd_tc<__nv_bfloat16>(images, p, st);
  return launch_attn_fwd_tc<__half>(images, p, st);
}

}  // namespace tc
}  // namespace agb
