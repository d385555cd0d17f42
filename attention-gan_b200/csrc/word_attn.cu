// Generator word-context attention, forward and backward (HBM-bound, CUDA cores).
//
// Replaces AttentionModule.forward (reference networks/attention.py:25-79) and its autograd.
// Data layout in HBM: images/ctx/attn/dctx/dimages are NCHW with HW contiguous, so a warp's
// lanes own consecutive pixels and every access is a full-width coalesced vector.  The projected
// word tile W.e [C x T] of one sample (2.3 KB at C=32, T=18) is fetched into shared memory by the
// TMA unit (cp.async.bulk, SASS UBLKCP), compacted to the unmasked words, and read as float4
// broadcasts.  Each thread owns V consecutive pixels and the whole T-vector of scores for them, so
// the softmax over words needs no cross-lane traffic at all.
//
// Algorithmic HBM bytes per pixel (es = bytes per element): fwd es*(2C+T), bwd es*3C (+es*T with
// dattn); see DESIGN.md.
#include <algorithm>
#include "agb_common.cuh"

namespace agb {

namespace tc {
int word_attn_tc_supported(const void* images, int C, int HW, int T, int io_dtype);
int word_attn_fwd_tc(const void* images, const float* we, const int64_t* mask, void* ctx, int64_t ctx_bs, void* attn,
                     int B, int C, int HW, int T, int io_dtype, float qscale, cudaStream_t st);
int word_attn_bwd_tc_supported(const void* images, const void* dctx, int64_t dctx_bs, const void* dattn, int C, int HW,
                               int T, int io_dtype);
int word_attn_tc_supported_nhwc(const void* images, const void* ctx, int64_t ctx_bs, int64_t ctx_ps, const void* attn,
                                int C, int HW, int T, int io_dtype);
int word_attn_fwd_tc_nhwc(const void* images, const float* we, const int64_t* mask, void* ctx, int64_t ctx_bs,
                          int64_t ctx_ps, void* attn, int B, int C, int HW, int T, int io_dtype, float qscale,
                          cudaStream_t st);
int word_attn_bwd_tc_supported_nhwc(const void* images, const void* dctx, int64_t dctx_bs, int64_t dctx_ps,
                                    const void* dattn, int C, int HW, int T, int io_dtype);
int word_attn_bwd_tc_nhwc(const void* images, const float* we, const int64_t* mask, const void* dctx, int64_t dctx_bs,
                          int64_t dctx_ps, const void* dattn, void* dimages, float* part, int part_slots, int B, int C,
                          int HW, int T, int io_dtype, float scale, cudaStream_t st);
int word_attn_bwd_tc_ctas(int B, int HW, int T);
int word_attn_bwd_tc_grid(int B, int HW, int T);
int word_attn_bwd_tc(const void* images, const float* we, const int64_t* mask, const void* dctx, int64_t dctx_bs,
                     const void* dattn, void* dimages, float* part, int part_slots, float* dwe, int B, int C, int HW, int T, int io_dtype,
                     float scale, cudaStream_t st);
}  // namespace tc

constexpr int kAttnThreads = 128;

// ---------------------------------------------------------------------------------------------
// we[b,c,t] = sum_e W[c,e] * words[b,e,t]                       (attention.py:50-52, conv1 1x1)
// ---------------------------------------------------------------------------------------------
__global__ void word_proj_fwd_kernel(const float* __restrict__ words, int64_t ws_b, int64_t ws_e,
                                     int64_t ws_t, const float* __restrict__ conv_w,
                                     float* __restrict__ we, int C, int E, int T) {
  const int b = blockIdx.x;
  const float* wb = words + (int64_t)b * ws_b;
  for (int i = threadIdx.x; i < C * T; i += blockDim.x) {
    const int c = i / T, t = i - c * T;
    const float* wr = conv_w + (size_t)c * E;
    const float* xr = wb + (int64_t)t * ws_t;
    float acc = 0.f;
    for (int e = 0; e < E; ++e) acc = fmaf(wr[e], xr[(int64_t)e * ws_e], acc);
    we[((size_t)b * C + c) * T + t] = acc;
  }
}

// shared prologue: TMA-load the [C,T] word tile of sample b, compact it to the unmasked words.
//   we_s[c*TMAX + j] = we[b, c, idx[j]]  (0 for j >= nv)
template <int TMAX>
__device__ __forceinline__ int stage_word_tile(const float* __restrict__ we, const int64_t* __restrict__ mask,
                                               int b, int C, int T, int use_tma, float* we_raw,
                                               float* we_s, uint64_t* bar, int* s_idx, int* s_midx,
                                               int* s_nv) {
  const int tid = threadIdx.x;
  const float* src = we + (size_t)b * C * T;
  if (tid == 0) {
    if (use_tma) {
      mbar_init(bar, 1);
      fence_barrier_init();
      mbar_expect_tx(bar, (uint32_t)(C * T * 4));
      tma_load_1d(we_raw, src, (uint32_t)(C * T * 4), bar);
    }
    int nv = 0, nm = 0;
    for (int t = 0; t < T; ++t) {
      if (mask[(size_t)b * T + t] != 0) s_idx[nv++] = t;
      else s_midx[nm++] = t;
    }
    *s_nv = nv;
  }
  if (!use_tma)
    for (int i = tid; i < C * T; i += blockDim.x) we_raw[i] = src[i];
  __syncthreads();
  if (use_tma) mbar_wait(bar, 0);
  const int nv = *s_nv;
  for (int i = tid; i < C * TMAX; i += blockDim.x) {
    const int c = i / TMAX, j = i - c * TMAX;
    we_s[i] = (j < nv) ? we_raw[c * T + s_idx[j]] : 0.f;
  }
  __syncthreads();
  return nv;
}

constexpr int kChanVec = 8;  // NHWC: channels one thread loads per access (pixel_scores' CU)
constexpr int kStoreVec = 4; // NHWC: channels one thread stores per access (fewer live accumulators)

// NHWC: V pixels x CU channels from pixel-major rows (pixel stride ps): per pixel, CU consecutive channels in
// one access when `vec` (C % CU == 0 and aligned), else one by one; pixels v >= n read as zero
template <typename IO, int CU, int V>
__device__ __forceinline__ void load_pixel_chans(const IO* __restrict__ p, int64_t ps, int nc, bool vec, int n,
                                                 float (&out)[CU][V]) {
#pragma unroll
  for (int v = 0; v < V; ++v) {
    float t[CU];
    if (v < n) load_vec<IO, CU>(p + (int64_t)v * ps, vec, nc, t);
#pragma unroll
    for (int u = 0; u < CU; ++u) out[u][v] = v < n ? t[u] : 0.f;
  }
}
template <typename IO, int CU, int V>
__device__ __forceinline__ void store_pixel_chans(IO* __restrict__ p, int64_t ps, int nc, bool vec, int n,
                                                  const float (&in)[CU][V]) {
#pragma unroll
  for (int v = 0; v < V; ++v) {
    float t[CU];
#pragma unroll
    for (int u = 0; u < CU; ++u) t[u] = in[u][v];
    if (v < n) store_vec<IO, CU>(p + (int64_t)v * ps, vec, nc, t);
  }
}

// scores for V pixels against the nv compacted words:  s[j][v] = sum_c h[c][p+v] * we_s[c][j]
// kNHWC: hb points at pixel p0 of a pixel-major map with pixel stride ps (HW unused); `vec` then means
// channel vectors of kChanVec.  The arithmetic (and its order) is the same for both layouts.
template <typename IO, int TMAX, int V, bool kNHWC = false>
__device__ __forceinline__ void pixel_scores(const IO* __restrict__ hb, int HW, int C, bool vec, int n,
                                             const float* we_s, int nv, float (&s)[TMAX][V], int64_t ps = 0) {
#pragma unroll
  for (int j = 0; j < TMAX; ++j)
#pragma unroll
    for (int v = 0; v < V; ++v) s[j][v] = 0.f;
  constexpr int CU = 8;  // channels fetched per batch: CU independent wide loads in flight
  for (int c0 = 0; c0 < C; c0 += CU) {
    float hv[CU][V];
    if constexpr (kNHWC) {
      load_pixel_chans<IO, CU, V>(hb + c0, ps, min(CU, C - c0), vec, n, hv);
    } else {
#pragma unroll
      for (int u = 0; u < CU; ++u) {
        if (c0 + u < C) load_vec<IO, V>(hb + (size_t)(c0 + u) * HW, vec, n, hv[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < CU; ++u) {
      if (c0 + u < C) {
        const float4* w4 = reinterpret_cast<const float4*>(we_s + (c0 + u) * TMAX);
#pragma unroll
        for (int j4 = 0; j4 < TMAX / 4; ++j4) {
          if (j4 * 4 < nv) {
            const float4 w = w4[j4];
#pragma unroll
            for (int v = 0; v < V; ++v) {
              s[j4 * 4 + 0][v] = fmaf(hv[u][v], w.x, s[j4 * 4 + 0][v]);
              s[j4 * 4 + 1][v] = fmaf(hv[u][v], w.y, s[j4 * 4 + 1][v]);
              s[j4 * 4 + 2][v] = fmaf(hv[u][v], w.z, s[j4 * 4 + 2][v]);
              s[j4 * 4 + 3][v] = fmaf(hv[u][v], w.w, s[j4 * 4 + 3][v]);
            }
          }
        }
      }
    }
  }
}

// in-register softmax over the nv valid words (attention.py:61-68); qscale = scale * log2(e)
template <int TMAX, int V>
__device__ __forceinline__ void softmax_words(float (&s)[TMAX][V], int nv, float qscale) {
#pragma unroll
  for (int v = 0; v < V; ++v) {
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < TMAX; ++j)
      if (j < nv) m = fmaxf(m, s[j][v]);
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < TMAX; ++j)
      if (j < nv) {
        const float e = exp2f((s[j][v] - m) * qscale);
        s[j][v] = e;
        sum += e;
      }
    const float inv = 1.f / sum;
#pragma unroll
    for (int j = 0; j < TMAX; ++j)
      if (j < nv) s[j][v] *= inv;
  }
}

// ---------------------------------------------------------------------------------------------
// forward                                                               attention.py:55-79
// ---------------------------------------------------------------------------------------------
// kNHWC: images / ctx / attn are pixel-major (channels_last); thread = V consecutive pixels as in NCHW, each
// moving its pixels' channel vectors.  ctx_bs is the batch stride of ctx and ctx_ps its pixel stride (C, or 2C
// for a channel slice of a concat buffer); vec_ok then says every channel vector is kChanVec-wide and aligned.
template <typename IO, int TMAX, int V, bool kNHWC = false>
__global__ void __launch_bounds__(kAttnThreads)
word_attn_fwd_kernel(const IO* __restrict__ h, const float* __restrict__ we,
                     const int64_t* __restrict__ mask, IO* __restrict__ ctx, int64_t ctx_bs,
                     IO* __restrict__ attn, int C, int HW, int T, float qscale, int use_tma, int vec_ok,
                     int64_t ctx_ps) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* we_raw = reinterpret_cast<float*>(smem_raw);
  float* we_s = we_raw + ((C * T + 3) & ~3);
  __shared__ uint64_t bar;
  __shared__ int s_idx[64], s_midx[64], s_nv;
  const int b = blockIdx.y;
  const int nv = stage_word_tile<TMAX>(we, mask, b, C, T, use_tma, we_raw, we_s, &bar, s_idx, s_midx, &s_nv);

  const int p0 = (blockIdx.x * kAttnThreads + threadIdx.x) * V;
  if (p0 >= HW) return;
  const int n = min(V, HW - p0);
  const bool vec = vec_ok != 0;
  if constexpr (kNHWC) {
    const IO* hb = h + ((size_t)b * HW + p0) * C;
    IO* cb = ctx + (size_t)b * ctx_bs + (size_t)p0 * ctx_ps;
    IO* ab = attn ? attn + ((size_t)b * HW + p0) * T : nullptr;
    const IO qnan = from_f32<IO>(__int_as_float(0x7fc00000));
    if (nv == 0) {  // every word masked: the reference's softmax over all -inf gives NaN
      for (int v = 0; v < n; ++v) {
        for (int c = 0; c < C; ++c) cb[(size_t)v * ctx_ps + c] = qnan;
        if (ab)
          for (int t = 0; t < T; ++t) ab[(size_t)v * T + t] = qnan;
      }
      return;
    }
    float s[TMAX][V];
    pixel_scores<IO, TMAX, V, true>(hb, HW, C, vec, n, we_s, nv, s, C);
    softmax_words<TMAX, V>(s, nv, qscale);
    // context = sum_j attn_j * we[:, j], kChanVec channels at a time              attention.py:73
    for (int c0 = 0; c0 < C; c0 += kStoreVec) {
      float acc[kStoreVec][V];
#pragma unroll
      for (int u = 0; u < kStoreVec; ++u) {
#pragma unroll
        for (int v = 0; v < V; ++v) acc[u][v] = 0.f;
        if (c0 + u < C) {
          const float4* w4 = reinterpret_cast<const float4*>(we_s + (c0 + u) * TMAX);
#pragma unroll
          for (int j4 = 0; j4 < TMAX / 4; ++j4) {
            if (j4 * 4 < nv) {
              const float4 w = w4[j4];
#pragma unroll
              for (int v = 0; v < V; ++v) {
                acc[u][v] = fmaf(s[j4 * 4 + 0][v], w.x, acc[u][v]);
                acc[u][v] = fmaf(s[j4 * 4 + 1][v], w.y, acc[u][v]);
                acc[u][v] = fmaf(s[j4 * 4 + 2][v], w.z, acc[u][v]);
                acc[u][v] = fmaf(s[j4 * 4 + 3][v], w.w, acc[u][v]);
              }
            }
          }
        }
      }
      store_pixel_chans<IO, kStoreVec, V>(cb + c0, ctx_ps, min(kStoreVec, C - c0), vec, n, acc);
    }
    if (ab) {  // a pixel's T probabilities are one contiguous row
      for (int v = 0; v < n; ++v) {
#pragma unroll
        for (int j = 0; j < TMAX; ++j)
          if (j < nv) ab[(size_t)v * T + s_idx[j]] = from_f32<IO>(s[j][v]);
        for (int k = 0; k < T - nv; ++k) ab[(size_t)v * T + s_midx[k]] = from_f32<IO>(0.f);
      }
    }
  } else {
  const IO* hb = h + (size_t)b * C * HW + p0;
  IO* cb = ctx + (size_t)b * ctx_bs + p0;

  if (nv == 0) {  // every word masked: the reference's softmax over all -inf gives NaN
    float nanv[V];
#pragma unroll
    for (int v = 0; v < V; ++v) nanv[v] = __int_as_float(0x7fc00000);
    for (int c = 0; c < C; ++c) store_vec<IO, V>(cb + (size_t)c * HW, vec, n, nanv);
    if (attn)
      for (int t = 0; t < T; ++t) store_vec<IO, V>(attn + ((size_t)b * T + t) * HW + p0, vec, n, nanv);
    return;
  }

  float s[TMAX][V];
  pixel_scores<IO, TMAX, V>(hb, HW, C, vec, n, we_s, nv, s);
  softmax_words<TMAX, V>(s, nv, qscale);

  // context = sum_j attn_j * we[:, j]                                    attention.py:73
  for (int c = 0; c < C; ++c) {
    float acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = 0.f;
    const float4* w4 = reinterpret_cast<const float4*>(we_s + c * TMAX);
#pragma unroll
    for (int j4 = 0; j4 < TMAX / 4; ++j4) {
      if (j4 * 4 < nv) {
        const float4 w = w4[j4];
#pragma unroll
        for (int v = 0; v < V; ++v) {
          acc[v] = fmaf(s[j4 * 4 + 0][v], w.x, acc[v]);
          acc[v] = fmaf(s[j4 * 4 + 1][v], w.y, acc[v]);
          acc[v] = fmaf(s[j4 * 4 + 2][v], w.z, acc[v]);
          acc[v] = fmaf(s[j4 * 4 + 3][v], w.w, acc[v]);
        }
      }
    }
    store_vec<IO, V>(cb + (size_t)c * HW, vec, n, acc);
  }
  if (attn) {
    IO* ab = attn + (size_t)b * T * HW + p0;
#pragma unroll
    for (int j = 0; j < TMAX; ++j)
      if (j < nv) store_vec<IO, V>(ab + (size_t)s_idx[j] * HW, vec, n, s[j]);
    float z[V];
#pragma unroll
    for (int v = 0; v < V; ++v) z[v] = 0.f;
    for (int k = 0; k < T - nv; ++k) store_vec<IO, V>(ab + (size_t)s_midx[k] * HW, vec, n, z);
  }
  }
}

// ---------------------------------------------------------------------------------------------
// backward, kernel 1: dimages + per-tile partial sums of d(W.e)              (SURVEY row a4)
//   g = we^T dctx (+ dattn);  ds = a * (g - sum_t a g);  dh = scale * we ds
//   dwe[c,t] = sum_p dctx[c,p] a[t,p] + scale * h[c,p] ds[t,p]
// Phase 1 is thread-per-pixel like the forward; a and ds of the tile are parked in shared memory
// and phase 2 re-maps threads to (channel, word-group) to contract over the tile's pixels.
// ---------------------------------------------------------------------------------------------
// kNHWC: images / dctx / dattn / dh pixel-major (dctx with pixel stride dctx_ps); vec_ok as in the forward
template <typename IO, int TMAX, int V, bool kNHWC = false>
__global__ void __launch_bounds__(kAttnThreads)
word_attn_bwd_kernel(const IO* __restrict__ h, const float* __restrict__ we,
                     const int64_t* __restrict__ mask, const IO* __restrict__ dctx, int64_t dctx_bs,
                     const IO* __restrict__ dattn, IO* __restrict__ dh, float* __restrict__ part,
                     int C, int HW, int T, float scale, int use_tma, int vec_ok, int vec4_ok, int64_t dctx_ps) {
  constexpr int PT = kAttnThreads * V;  // pixels per tile
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* we_raw = reinterpret_cast<float*>(smem_raw);
  float* we_s = we_raw + ((C * T + 3) & ~3);
  float* a_s = we_s + C * TMAX;   // [TMAX][PT]
  float* ds_s = a_s + TMAX * PT;  // [TMAX][PT]
  __shared__ uint64_t bar;
  __shared__ int s_idx[64], s_midx[64], s_nv;
  const int b = blockIdx.y, tid = threadIdx.x;
  const int nv = stage_word_tile<TMAX>(we, mask, b, C, T, use_tma, we_raw, we_s, &bar, s_idx, s_midx, &s_nv);
  const float qscale = scale * kLog2e;
  const int tile0 = blockIdx.x * PT;
  const int p0 = tile0 + tid * V;
  const int n = max(0, min(V, HW - p0));
  const bool vec = vec_ok != 0;
  const IO* hb = kNHWC ? h + ((size_t)b * HW + p0) * C : h + (size_t)b * C * HW + p0;
  const IO* db = kNHWC ? dctx + (size_t)b * dctx_bs + (size_t)p0 * dctx_ps : dctx + (size_t)b * dctx_bs + p0;

  if (nv == 0) {  // NaN forward: propagate NaN like autograd would
    float nanv[V];
#pragma unroll
    for (int v = 0; v < V; ++v) nanv[v] = __int_as_float(0x7fc00000);
    if constexpr (kNHWC) {
      for (int v = 0; v < n; ++v)
        for (int c = 0; c < C; ++c) dh[((size_t)b * HW + p0 + v) * C + c] = from_f32<IO>(nanv[0]);
    } else {
    if (n > 0)
      for (int c = 0; c < C; ++c) store_vec<IO, V>(dh + (size_t)b * C * HW + (size_t)c * HW + p0, vec, n, nanv);
    }
    float* pp = part + ((size_t)b * gridDim.x + blockIdx.x) * C * T;
    for (int i = tid; i < C * T; i += kAttnThreads) pp[i] = __int_as_float(0x7fc00000);
    return;
  }

  if (n > 0) {
    float a[TMAX][V];
    pixel_scores<IO, TMAX, V, kNHWC>(hb, HW, C, vec, n, we_s, nv, a, C);
    softmax_words<TMAX, V>(a, nv, qscale);
    float g[TMAX][V];
#pragma unroll
    for (int j = 0; j < TMAX; ++j)
#pragma unroll
      for (int v = 0; v < V; ++v) g[j][v] = 0.f;
    // g[j] = sum_c we[c][j] * dctx[c]
    pixel_scores<IO, TMAX, V, kNHWC>(db, HW, C, vec, n, we_s, nv, g, dctx_ps);
    if constexpr (kNHWC) {
      if (dattn) {  // a pixel's T gradients are one contiguous row
        const IO* ab = dattn + ((size_t)b * HW + p0) * T;
#pragma unroll
        for (int j = 0; j < TMAX; ++j)
          if (j < nv) {
#pragma unroll
            for (int v = 0; v < V; ++v) g[j][v] += v < n ? to_f32(ab[(size_t)v * T + s_idx[j]]) : 0.f;
          }
      }
    } else if (dattn) {
      const IO* ab = dattn + (size_t)b * T * HW + p0;
#pragma unroll
      for (int j = 0; j < TMAX; ++j)
        if (j < nv) {
          float t4[V];
          load_vec<IO, V>(ab + (size_t)s_idx[j] * HW, vec, n, t4);
#pragma unroll
          for (int v = 0; v < V; ++v) g[j][v] += t4[v];
        }
    }
#pragma unroll
    for (int v = 0; v < V; ++v) {
      float dot = 0.f;
#pragma unroll
      for (int j = 0; j < TMAX; ++j)
        if (j < nv) dot = fmaf(a[j][v], g[j][v], dot);
#pragma unroll
      for (int j = 0; j < TMAX; ++j)
        if (j < nv) g[j][v] = a[j][v] * (g[j][v] - dot);  // g now holds ds
    }
    // dh[c] = scale * sum_j we[c][j] ds[j]
    if constexpr (kNHWC) {
      IO* ob = dh + ((size_t)b * HW + p0) * C;
      for (int c0 = 0; c0 < C; c0 += kStoreVec) {
        float acc[kStoreVec][V];
#pragma unroll
        for (int u = 0; u < kStoreVec; ++u) {
#pragma unroll
          for (int v = 0; v < V; ++v) acc[u][v] = 0.f;
          if (c0 + u < C) {
            const float4* w4 = reinterpret_cast<const float4*>(we_s + (c0 + u) * TMAX);
#pragma unroll
            for (int j4 = 0; j4 < TMAX / 4; ++j4) {
              if (j4 * 4 < nv) {
                const float4 w = w4[j4];
#pragma unroll
                for (int v = 0; v < V; ++v) {
                  acc[u][v] = fmaf(g[j4 * 4 + 0][v], w.x, acc[u][v]);
                  acc[u][v] = fmaf(g[j4 * 4 + 1][v], w.y, acc[u][v]);
                  acc[u][v] = fmaf(g[j4 * 4 + 2][v], w.z, acc[u][v]);
                  acc[u][v] = fmaf(g[j4 * 4 + 3][v], w.w, acc[u][v]);
                }
              }
            }
#pragma unroll
            for (int v = 0; v < V; ++v) acc[u][v] *= scale;
          }
        }
        store_pixel_chans<IO, kStoreVec, V>(ob + c0, C, min(kStoreVec, C - c0), vec, n, acc);
      }
    } else {
    IO* ob = dh + (size_t)b * C * HW + p0;
    for (int c = 0; c < C; ++c) {
      float acc[V];
#pragma unroll
      for (int v = 0; v < V; ++v) acc[v] = 0.f;
      const float4* w4 = reinterpret_cast<const float4*>(we_s + c * TMAX);
#pragma unroll
      for (int j4 = 0; j4 < TMAX / 4; ++j4) {
        if (j4 * 4 < nv) {
          const float4 w = w4[j4];
#pragma unroll
          for (int v = 0; v < V; ++v) {
            acc[v] = fmaf(g[j4 * 4 + 0][v], w.x, acc[v]);
            acc[v] = fmaf(g[j4 * 4 + 1][v], w.y, acc[v]);
            acc[v] = fmaf(g[j4 * 4 + 2][v], w.z, acc[v]);
            acc[v] = fmaf(g[j4 * 4 + 3][v], w.w, acc[v]);
          }
        }
      }
#pragma unroll
      for (int v = 0; v < V; ++v) acc[v] *= scale;
      store_vec<IO, V>(ob + (size_t)c * HW, vec, n, acc);
    }
    }
    // park a and ds (pixels beyond HW contribute zero)
#pragma unroll
    for (int j = 0; j < TMAX; ++j)
      if (j < nv) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const bool live = v < n;
          a_s[j * PT + tid * V + v] = live ? a[j][v] : 0.f;
          ds_s[j * PT + tid * V + v] = live ? g[j][v] : 0.f;
        }
      }
  } else {
    for (int j = 0; j < nv; ++j)
#pragma unroll
      for (int v = 0; v < V; ++v) {
        a_s[j * PT + tid * V + v] = 0.f;
        ds_s[j * PT + tid * V + v] = 0.f;
      }
  }
  __syncthreads();

  // phase 2: thread -> (channel c, word group jg); words j = jg, jg+4, ...
  constexpr int JPT = TMAX / 4;  // words per thread
  const int jg = tid & 3;
  const int tile_pix = min(PT, HW - tile0);
  float* pp = part + ((size_t)b * gridDim.x + blockIdx.x) * C * T;
  for (int c = tid >> 2; c < C; c += kAttnThreads / 4) {
    float acc[JPT];
#pragma unroll
    for (int k = 0; k < JPT; ++k) acc[k] = 0.f;
    const IO* hr = h + (size_t)b * C * HW + (size_t)c * HW + tile0;
    const IO* dr = dctx + (size_t)b * dctx_bs + (size_t)c * HW + tile0;
    for (int p = 0; p < tile_pix; p += 4) {
      float h4[4], d4[4];
      const int nn = min(4, tile_pix - p);
      if constexpr (kNHWC) {   // one channel of 4 pixels: strided
        const IO* hq = h + ((size_t)b * HW + tile0 + p) * C + c;
        const IO* dq = dctx + (size_t)b * dctx_bs + (size_t)(tile0 + p) * dctx_ps + c;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          h4[i] = i < nn ? to_f32(hq[(size_t)i * C]) : 0.f;
          d4[i] = i < nn ? to_f32(dq[(size_t)i * dctx_ps]) : 0.f;
        }
      } else {
        load_vec<IO, 4>(hr + p, vec4_ok != 0, nn, h4);
        load_vec<IO, 4>(dr + p, vec4_ok != 0, nn, d4);
      }
#pragma unroll
      for (int k = 0; k < JPT; ++k) {
        const int j = jg + 4 * k;
        if (j < nv) {
          const float4 a4 = *reinterpret_cast<const float4*>(a_s + j * PT + p);
          const float4 s4 = *reinterpret_cast<const float4*>(ds_s + j * PT + p);
          float t = d4[0] * a4.x;
          t = fmaf(d4[1], a4.y, t);
          t = fmaf(d4[2], a4.z, t);
          t = fmaf(d4[3], a4.w, t);
          float u = h4[0] * s4.x;
          u = fmaf(h4[1], s4.y, u);
          u = fmaf(h4[2], s4.z, u);
          u = fmaf(h4[3], s4.w, u);
          acc[k] += fmaf(scale, u, t);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < JPT; ++k) {
      const int j = jg + 4 * k;
      if (j < nv) pp[c * T + s_idx[j]] = acc[k];
    }
    for (int k = jg; k < T - nv; k += 4) pp[c * T + s_midx[k]] = 0.f;
  }
}

// backward, kernel 2: dwe[b] = sum over tiles (fixed order -> deterministic), then
//   dwords[b,e,t] = sum_c W[c,e] dwe[b,c,t]                      (autograd of conv1, words side)
__global__ void word_attn_bwd_reduce_kernel(const float* __restrict__ part, int ntiles,
                                            const float* __restrict__ conv_w, float* __restrict__ dwe,
                                            float* __restrict__ dwords, int C, int E, int T) {
  extern __shared__ float s_dwe[];  // [C*T]
  const int b = blockIdx.x;
  const float* pb = part + (size_t)b * ntiles * C * T;
  for (int i = threadIdx.x; i < C * T; i += blockDim.x) {
    float acc = 0.f;
    for (int k = 0; k < ntiles; ++k) acc += pb[(size_t)k * C * T + i];
    s_dwe[i] = acc;
    dwe[(size_t)b * C * T + i] = acc;
  }
  __syncthreads();
  if (dwords == nullptr) return;
  for (int i = threadIdx.x; i < E * T; i += blockDim.x) {
    const int e = i / T, t = i - e * T;
    float acc = 0.f;
    for (int c = 0; c < C; ++c) acc = fmaf(conv_w[(size_t)c * E + e], s_dwe[c * T + t], acc);
    dwords[((size_t)b * E + e) * T + t] = acc;
  }
}

// dwe[b,i] = sum over the per-CTA partials (fixed order -> deterministic)
__global__ void sum_partials_kernel(const float* __restrict__ part, int nparts, int64_t part_stride,
                                    int64_t batch_stride, int n, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
  if (i >= n) return;
  const float* p = part + (int64_t)b * batch_stride + i;
  float acc = 0.f;
#pragma unroll 8
  for (int k = 0; k < nparts; ++k) acc += p[(int64_t)k * part_stride];
  out[(size_t)b * n + i] = acc;
}

// backward, kernel 3: dW[c,e] = sum_b sum_t dwe[b,c,t] * words[b,e,t]   (autograd of conv1, weight side)
__global__ void word_attn_bwd_dw_kernel(const float* __restrict__ dwe, const float* __restrict__ words,
                                        int64_t ws_b, int64_t ws_e, int64_t ws_t,
                                        float* __restrict__ dconv_w, int B, int C, int E, int T) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C * E) return;
  const int c = i / E, e = i - c * E;
  float acc = 0.f;
  for (int b = 0; b < B; ++b) {
    const float* d = dwe + ((size_t)b * C + c) * T;
    const float* x = words + (int64_t)b * ws_b + (int64_t)e * ws_e;
    for (int t = 0; t < T; ++t) acc = fmaf(d[t], x[(int64_t)t * ws_t], acc);
  }
  dconv_w[i] = acc;
}

// ---------------------------------------------------------------------------------------------
// small per-sample kernels around the pixel kernels (the conv1 projection and its autograd);
// one CTA per sample, everything staged in shared memory, fixed summation orders
// ---------------------------------------------------------------------------------------------
// we[b][c,t] = sum_e W[c,e] words[b][e,t]                              (attention.py:50-52, conv1 1x1)
// thread = one output (c, t); W and the sample's words sit in shared memory with padded rows
__device__ __forceinline__ void stage_words(float* x_s, const float* __restrict__ words, int64_t ws_b, int64_t ws_e,
                                            int64_t ws_t, int b, int E, int T) {
#pragma unroll 8
  for (int i = threadIdx.x; i < E * T; i += blockDim.x) {
    // walk the source along its contiguous dimension
    const int e = ws_e == 1 ? i % E : i / T, t = ws_e == 1 ? i / E : i % T;
    x_s[t * (E + 1) + e] = words[(int64_t)b * ws_b + (int64_t)e * ws_e + (int64_t)t * ws_t];
  }
}
__global__ void __launch_bounds__(1024)
project_words_kernel(const float* __restrict__ conv_w, const float* __restrict__ words, int64_t ws_b, int64_t ws_e,
                     int64_t ws_t, float* __restrict__ we, int C, int E, int T) {
  // gridDim.y CTAs per sample, each with a slice of the channels (the per-sample work is latency-bound: smaller
  // slices on more SMs finish sooner, and the weight slice is all a CTA has to stage)
  extern __shared__ float sm_[];
  const int b = blockIdx.x, P = E + 1;
  const int cs = (C + gridDim.y - 1) / gridDim.y, c0 = blockIdx.y * cs, nc = max(0, min(cs, C - c0));
  float* w_s = sm_;                               // [nc][E + 1]
  float* x_s = sm_ + (size_t)cs * (E + 1);        // [T][E + 1]
#pragma unroll 8
  for (int i = threadIdx.x; i < nc * E; i += blockDim.x) w_s[(i / E) * P + (i % E)] = conv_w[(size_t)c0 * E + i];
  stage_words(x_s, words, ws_b, ws_e, ws_t, b, E, T);
  __syncthreads();
  for (int i = threadIdx.x; i < nc * T; i += blockDim.x) {
    const int c = i / T, t = i - c * T;
    const float* w = w_s + c * P;
    const float* x = x_s + t * P;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int e = 0;
    for (; e + 4 <= E; e += 4) {
      a0 = fmaf(w[e], x[e], a0);
      a1 = fmaf(w[e + 1], x[e + 1], a1);
      a2 = fmaf(w[e + 2], x[e + 2], a2);
      a3 = fmaf(w[e + 3], x[e + 3], a3);
    }
    for (; e < E; ++e) a0 = fmaf(w[e], x[e], a0);
    we[(size_t)b * C * T + (size_t)c0 * T + i] = (a0 + a1) + (a2 + a3);
  }
}

// backward of the projection for one sample: dwe[b] = sum of the pixel kernel's partial slots;
// dwords[b][e,t] = sum_c W[c,e] dwe[b][c,t];  dwp[b][c,e] = sum_t dwe[b][c,t] words[b][e,t]
// (this sample's share of d conv1.weight; summed over b by sum_partials_kernel).
// slot count: G == 0: `slots` (every slot valid); G > 0: the CTAs of a persistent grid of G whose tile
// range overlaps sample b (word_attn_tc.cu).  thread = embedding index e.
__global__ void __launch_bounds__(1024)
project_words_bwd_kernel(const float* __restrict__ part, int slots, int tiles, int G, long long total,
                         const float* __restrict__ conv_w, const float* __restrict__ words, int64_t ws_b,
                         int64_t ws_e, int64_t ws_t, float* __restrict__ dwe, float* __restrict__ dwords,
                         float* __restrict__ dwp, int C, int E, int T) {
  // gridDim.y CTAs per sample, each with a slice [e0, e0 + ne) of the embedding index (both outputs are
  // independent per e); every slice re-forms the small dwe[b] (C*T values), slice 0 stores it
  extern __shared__ float sm_[];
  const int b = blockIdx.x;
  const int es = (E + gridDim.y - 1) / gridDim.y, e0 = blockIdx.y * es, ne = max(0, min(es, E - e0)), P = es + 1;
  float* d_s = sm_;                               // [C][T]
  float* w_s = d_s + C * T;                       // [C][es + 1]
  float* x_s = w_s + (size_t)C * P;               // [T][es + 1]
  int n = slots;
  if (G > 0) {
    const long long first = (((long long)b * tiles + 1) * G + total - 1) / total - 1;
    const long long last = (((long long)(b + 1) * tiles) * G + total - 1) / total - 1;
    n = (int)(last - first) + 1;
  }
  for (int i = threadIdx.x; i < C * T; i += blockDim.x) {
    const float* p = part + (size_t)b * slots * C * T + i;
    float acc = 0.f;
#pragma unroll 4
    for (int k = 0; k < n; ++k) acc += p[(size_t)k * C * T];
    d_s[i] = acc;
    if (blockIdx.y == 0) dwe[(size_t)b * C * T + i] = acc;
  }
  if (dwords != nullptr) {
#pragma unroll 8
    for (int i = threadIdx.x; i < C * ne; i += blockDim.x) w_s[(i / ne) * P + (i % ne)] = conv_w[(size_t)(i / ne) * E + e0 + (i % ne)];
  }
  if (dwp != nullptr) {
#pragma unroll 8
    for (int i = threadIdx.x; i < ne * T; i += blockDim.x) {
      // walk the source along its contiguous dimension
      const int e = ws_e == 1 ? i % ne : i / T, t = ws_e == 1 ? i / ne : i % T;
      x_s[t * P + e] = words[(int64_t)b * ws_b + (int64_t)(e0 + e) * ws_e + (int64_t)t * ws_t];
    }
  }
  __syncthreads();
  if (dwords != nullptr) {
    for (int i = threadIdx.x; i < ne * T; i += blockDim.x) {      // lanes = consecutive e: conflict-free
      const int t = i / ne, e = i - t * ne;
      float acc = 0.f;
      for (int c = 0; c < C; ++c) acc = fmaf(w_s[c * P + e], d_s[c * T + t], acc);
      dwords[((size_t)b * E + e0 + e) * T + t] = acc;
    }
  }
  if (dwp != nullptr) {
    for (int i = threadIdx.x; i < C * ne; i += blockDim.x) {
      const int c = i / ne, e = i - c * ne;
      float acc = 0.f;
      for (int t = 0; t < T; ++t) acc = fmaf(d_s[c * T + t], x_s[t * P + e], acc);
      dwp[((size_t)b * C + c) * E + e0 + e] = acc;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int pick_tmax(int T) {
  if (T <= 8) return 8;
  if (T <= 16) return 16;
  if (T <= 24) return 24;
  if (T <= 32) return 32;
  if (T <= 48) return 48;
  return 64;
}
static int fwd_v(int tmax) { return tmax <= 24 ? 4 : (tmax <= 32 ? 2 : 1); }
static int bwd_v(int tmax) { return tmax <= 24 ? 2 : 1; }

// NHWC: every channel vector of kChanVec elements starts aligned (pixel and batch strides included)
template <typename IO>
static bool chan_vec_ok(int C, int64_t ps, int64_t bs, const void* a, const void* b, const void* c) {
  const uintptr_t w = sizeof(IO) * kChanVec;
  return C % kChanVec == 0 && ps % kChanVec == 0 && bs % kChanVec == 0 && (uintptr_t)a % w == 0 &&
         (uintptr_t)b % w == 0 && (uintptr_t)c % w == 0;
}

template <typename IO, int TMAX, int V, bool kNHWC>
static int launch_fwd(const void* images, const float* we, const int64_t* mask, void* ctx,
                      int64_t ctx_bs, int64_t ctx_ps, void* attn, int B, int C, int HW, int T, float qscale,
                      int use_tma, cudaStream_t st) {
  const size_t smem = (size_t)(((C * T + 3) & ~3) + C * TMAX) * sizeof(float);
  const int vec_ok = kNHWC ? chan_vec_ok<IO>(C, ctx_ps, ctx_bs, images, ctx, images)
                           : (HW % V == 0) && (ctx_bs % V == 0) &&
                             ((uintptr_t)images % (sizeof(IO) * V) == 0) && ((uintptr_t)ctx % (sizeof(IO) * V) == 0) &&
                             (attn == nullptr || (uintptr_t)attn % (sizeof(IO) * V) == 0);
  dim3 grid(cdiv(HW, kAttnThreads * V), B);
  const int slot = prof_begin(PROF_ATTN_FWD, st);
  word_attn_fwd_kernel<IO, TMAX, V, kNHWC><<<grid, kAttnThreads, smem, st>>>(
      (const IO*)images, we, mask, (IO*)ctx, ctx_bs, (IO*)attn, C, HW, T, qscale, use_tma, vec_ok, ctx_ps);
  prof_end(slot, st);
  return check_launch("word_attn_fwd_kernel");
}

constexpr size_t kBwdStaticSmem = 1024;   // bound on word_attn_bwd_kernel's static shared memory (barrier, word lists)
template <typename IO, int TMAX, int V>
static size_t bwd_smem(int C, int T) {
  return (size_t)(((C * T + 3) & ~3) + C * TMAX + 2 * TMAX * kAttnThreads * V) * sizeof(float);
}

template <typename IO, int TMAX, int V, bool kNHWC>
static int launch_bwd(const void* images, const float* we, const int64_t* mask, const void* dctx,
                      int64_t dctx_bs, int64_t dctx_ps, const void* dattn, void* dimages, float* part, int B, int C,
                      int HW, int T, float scale, int use_tma, cudaStream_t st) {
  const size_t smem = bwd_smem<IO, TMAX, V>(C, T);
  auto kern = word_attn_bwd_kernel<IO, TMAX, V, kNHWC>;
  if (smem + kBwdStaticSmem > 48 * 1024)   // the opt-in counts the kernel's static shared memory too
    AGB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  auto ok = [&](int w) {
    return (HW % w == 0) && (dctx_bs % w == 0) && ((uintptr_t)images % (sizeof(IO) * w) == 0) &&
           ((uintptr_t)dctx % (sizeof(IO) * w) == 0) && ((uintptr_t)dimages % (sizeof(IO) * w) == 0) &&
           (dattn == nullptr || (uintptr_t)dattn % (sizeof(IO) * w) == 0);
  };
  dim3 grid(cdiv(HW, kAttnThreads * V), B);
  const int slot = prof_begin(PROF_ATTN_BWD, st);
  const int vec_ok = kNHWC ? chan_vec_ok<IO>(C, dctx_ps, dctx_bs, images, dctx, dimages) : ok(V);
  kern<<<grid, kAttnThreads, smem, st>>>((const IO*)images, we, mask, (const IO*)dctx, dctx_bs,
                                        (const IO*)dattn, (IO*)dimages, part, C, HW, T, scale,
                                        use_tma, vec_ok ? 1 : 0, ok(4) ? 1 : 0, dctx_ps);
  prof_end(slot, st);
  return check_launch("word_attn_bwd_kernel");
}

#define AGB_DISPATCH_TMAX(TM, ...)                     \
  switch (TM) {                                        \
    case 8: { constexpr int TMAX = 8; __VA_ARGS__; } break;   \
    case 16: { constexpr int TMAX = 16; __VA_ARGS__; } break; \
    case 24: { constexpr int TMAX = 24; __VA_ARGS__; } break; \
    case 32: { constexpr int TMAX = 32; __VA_ARGS__; } break; \
    case 48: { constexpr int TMAX = 48; __VA_ARGS__; } break; \
    default: { constexpr int TMAX = 64; __VA_ARGS__; } break; \
  }

static int check_common(int B, int C, int HW, int E, int T, int io_dtype) {
  if (B <= 0 || C <= 0 || HW <= 0 || E <= 0 || T <= 0) return fail_arg("non-positive size B=%d C=%d HW=%d E=%d T=%d", B, C, HW, E, T);
  if (T > 64) return fail_unsupported("T=%d > 64 words is outside the compiled range", T);
  if (C > 64) return fail_unsupported("C=%d > 64 channels is outside the compiled range", C);
  if (B > 65535) return fail_unsupported("B=%d > 65535", B);
  if (io_dtype != AGB_F32 && io_dtype != AGB_BF16 && io_dtype != AGB_F16) return fail_arg("bad io_dtype %d", io_dtype);
  return 0;
}

}  // namespace agb

using namespace agb;

// both layouts: nhwc = images / ctx / attn pixel-major, ctx with pixel stride ctx_ps
static int word_attn_fwd_impl(bool nhwc, const void* images, const float* words, int64_t ws_b, int64_t ws_e,
                              int64_t ws_t, const float* conv_w, const int64_t* mask, void* ctx, int64_t ctx_bs,
                              int64_t ctx_ps, void* attn, float* we, int B, int C, int HW, int E, int T, int io_dtype,
                              int scaled, void* stream) {
  if (int rc = check_common(B, C, HW, E, T, io_dtype)) return rc;
  if (!images || !words || !conv_w || !mask || !ctx || !we) return fail_arg("null pointer");
  if (nhwc && (ctx_ps < C || ctx_bs < (int64_t)HW * ctx_ps))
    return fail_arg("ctx strides overlap: pixel stride %lld < C=%d or batch stride %lld < HW * pixel stride",
                    (long long)ctx_ps, C, (long long)ctx_bs);
  cudaStream_t st = (cudaStream_t)stream;
  // we[b][c,t] = sum_e W[c,e] words[b][e,t]                     (attention.py:50-52, conv1 1x1)
  {
    // up to 4 channel slices per sample while the batch alone does not fill the GPU
    const int slices = std::max(1, std::min(std::min(4, C), (2 * device_sms() + B - 1) / B));
    const int cs = (C + slices - 1) / slices;
    const size_t smem = (size_t)(cs + T) * (E + 1) * sizeof(float);
    if (smem > 200 * 1024) return fail_unsupported("E=%d is outside the compiled range of the projection kernel", E);
    if (smem > 48 * 1024)
      AGB_CUDA(cudaFuncSetAttribute(project_words_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int threads = std::min(1024, (cs * T + 31) / 32 * 32);
    project_words_kernel<<<dim3(B, slices), threads, smem, st>>>(conv_w, words, ws_b, ws_e, ws_t, we, C, E, T);
    if (int rc = check_launch("project_words_kernel")) return rc;
  }
  const float qscale = (scaled ? 1.f / sqrtf((float)C) : 1.f) * kLog2e;
  // 16-bit feature maps: both contractions on tcgen05 (word_attn_tc.cu); fp32 maps and odd shapes:
  // CUDA cores.  Both are native sm_100a kernels of this library.
  if (nhwc) {
    if (tc::word_attn_tc_supported_nhwc(images, ctx, ctx_bs, ctx_ps, attn, C, HW, T, io_dtype))
      return tc::word_attn_fwd_tc_nhwc(images, we, mask, ctx, ctx_bs, ctx_ps, attn, B, C, HW, T, io_dtype, qscale, st);
  } else if (tc::word_attn_tc_supported(images, C, HW, T, io_dtype)) {
    return tc::word_attn_fwd_tc(images, we, mask, ctx, ctx_bs, attn, B, C, HW, T, io_dtype, qscale, st);
  }
  const int use_tma = ((C * T) % 4 == 0) && ((uintptr_t)we % 16 == 0);
  const int tm = pick_tmax(T);
  int rc = 0;
#define AGB_FWD_LAYOUT(L)                                                                                                   \
  AGB_DISPATCH_TMAX(tm, {                                                                                                   \
    constexpr int V = TMAX <= 24 ? 4 : (TMAX <= 32 ? 2 : 1);                                                                \
    if (io_dtype == AGB_F32) rc = launch_fwd<float, TMAX, V, L>(images, we, mask, ctx, ctx_bs, ctx_ps, attn, B, C, HW, T, qscale, use_tma, st); \
    else if (io_dtype == AGB_BF16) rc = launch_fwd<__nv_bfloat16, TMAX, V, L>(images, we, mask, ctx, ctx_bs, ctx_ps, attn, B, C, HW, T, qscale, use_tma, st); \
    else rc = launch_fwd<__half, TMAX, V, L>(images, we, mask, ctx, ctx_bs, ctx_ps, attn, B, C, HW, T, qscale, use_tma, st); \
  })
  if (nhwc) AGB_FWD_LAYOUT(true) else AGB_FWD_LAYOUT(false)
#undef AGB_FWD_LAYOUT
  return rc;
}

extern "C" int agb_word_attn_fwd(const void* images, const float* words, int64_t ws_b, int64_t ws_e,
                                 int64_t ws_t, const float* conv_w, const int64_t* mask, void* ctx,
                                 int64_t ctx_bs, void* attn, float* we, int B, int C, int HW, int E,
                                 int T, int io_dtype, int scaled, void* stream) {
  return word_attn_fwd_impl(false, images, words, ws_b, ws_e, ws_t, conv_w, mask, ctx, ctx_bs, 0, attn, we, B, C, HW,
                            E, T, io_dtype, scaled, stream);
}

extern "C" int agb_word_attn_fwd_nhwc(const void* images, const float* words, int64_t ws_b, int64_t ws_e,
                                      int64_t ws_t, const float* conv_w, const int64_t* mask, void* ctx,
                                      int64_t ctx_bs, int64_t ctx_ps, void* attn, float* we, int B, int C, int HW,
                                      int E, int T, int io_dtype, int scaled, void* stream) {
  return word_attn_fwd_impl(true, images, words, ws_b, ws_e, ws_t, conv_w, mask, ctx, ctx_bs, ctx_ps, attn, we, B, C,
                            HW, E, T, io_dtype, scaled, stream);
}

static int dw_splits(int B) {
  int s = 1;
  for (int k = 2; k <= 32 && k <= B; ++k)
    if (B % k == 0) s = k;
  return s;
}

extern "C" size_t agb_word_attn_bwd_workspace_bytes(int B, int C, int HW, int E, int T) {
  if (B <= 0 || C <= 0 || HW <= 0 || E <= 0 || T <= 0 || T > 64) return 0;
  const size_t ntiles = cdiv(HW, 128);   // upper bound of the partial sums either kernel family writes
  return (((size_t)B * ntiles + (size_t)B) * C * T + (size_t)B * C * E) * sizeof(float);
}

static int word_attn_bwd_impl(bool nhwc, const void* images, const float* words, int64_t ws_b, int64_t ws_e,
                              int64_t ws_t, const float* conv_w, const int64_t* mask, const float* we,
                              const void* dctx, int64_t dctx_bs, int64_t dctx_ps, const void* dattn, void* dimages,
                              float* dwords, float* dconv_w, void* workspace, size_t workspace_bytes, int B, int C,
                              int HW, int E, int T, int io_dtype, int scaled, void* stream) {
  if (int rc = check_common(B, C, HW, E, T, io_dtype)) return rc;
  if (!images || !words || !conv_w || !mask || !we || !dctx || !dimages || !workspace) return fail_arg("null pointer");
  if (nhwc && (dctx_ps < C || dctx_bs < (int64_t)HW * dctx_ps))
    return fail_arg("dctx strides overlap: pixel stride %lld < C=%d or batch stride %lld < HW * pixel stride",
                    (long long)dctx_ps, C, (long long)dctx_bs);
  if (workspace_bytes < agb_word_attn_bwd_workspace_bytes(B, C, HW, E, T)) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, agb_word_attn_bwd_workspace_bytes(B, C, HW, E, T));
    return AGB_E_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const float scale = scaled ? 1.f / sqrtf((float)C) : 1.f;
  const int use_tma = ((C * T) % 4 == 0) && ((uintptr_t)we % 16 == 0);
  const int tm = pick_tmax(T);
  const int V = bwd_v(tm);
  int ntiles = cdiv(HW, kAttnThreads * V);
  float* part = (float*)workspace;
  int rc = 0;
  const bool use_tc = (nhwc ? tc::word_attn_bwd_tc_supported_nhwc(images, dctx, dctx_bs, dctx_ps, dattn, C, HW, T, io_dtype)
                            : tc::word_attn_bwd_tc_supported(images, dctx, dctx_bs, dattn, C, HW, T, io_dtype)) != 0;
  if (use_tc) ntiles = tc::word_attn_bwd_tc_ctas(B, HW, T);
  float* dwe = part + (size_t)B * ntiles * C * T;
  int G = 0;                                      // 0: every partial slot is valid
  if (use_tc) {
    G = tc::word_attn_bwd_tc_grid(B, HW, T);
    rc = nhwc ? tc::word_attn_bwd_tc_nhwc(images, we, mask, dctx, dctx_bs, dctx_ps, dattn, dimages, part, ntiles, B, C,
                                          HW, T, io_dtype, scale, st)
              : tc::word_attn_bwd_tc(images, we, mask, dctx, dctx_bs, dattn, dimages, part, ntiles, nullptr, B, C, HW, T,
                                     io_dtype, scale, st);
    if (rc) return rc;
  } else {
#define AGB_BWD_LAYOUT(L)                                                                                                   \
    AGB_DISPATCH_TMAX(tm, {                                                                                                 \
      constexpr int VV = TMAX <= 24 ? 2 : 1;                                                                                \
      if (io_dtype == AGB_F32) rc = launch_bwd<float, TMAX, VV, L>(images, we, mask, dctx, dctx_bs, dctx_ps, dattn, dimages, part, B, C, HW, T, scale, use_tma, st); \
      else if (io_dtype == AGB_BF16) rc = launch_bwd<__nv_bfloat16, TMAX, VV, L>(images, we, mask, dctx, dctx_bs, dctx_ps, dattn, dimages, part, B, C, HW, T, scale, use_tma, st); \
      else rc = launch_bwd<__half, TMAX, VV, L>(images, we, mask, dctx, dctx_bs, dctx_ps, dattn, dimages, part, B, C, HW, T, scale, use_tma, st); \
    })
    if (nhwc) AGB_BWD_LAYOUT(true) else AGB_BWD_LAYOUT(false)
#undef AGB_BWD_LAYOUT
    if (rc) return rc;
  }
  // one CTA per sample: dwe[b] = sum of the partial slots; dwords[b][e,t] = sum_c W[c,e] dwe[b][c,t];
  // dwp[b][c,e] = sum_t dwe[b][c,t] words[b][e,t]; then dW[c,e] = sum_b dwp[b][c,e] in a fixed order
  float* dwp = dwe + (size_t)B * C * T;
  const int pslices = std::max(1, std::min(std::min(4, E / 32), (2 * device_sms() + B - 1) / B));   // slices of the embedding index
  const int pes = (E + pslices - 1) / pslices;
  const size_t psmem = ((size_t)C * T + (size_t)(C + T) * (pes + 1)) * sizeof(float);
  if (psmem > 200 * 1024) return fail_unsupported("E=%d is outside the compiled range of the projection kernel", E);
  if (psmem > 48 * 1024)
    AGB_CUDA(cudaFuncSetAttribute(project_words_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
  project_words_bwd_kernel<<<dim3(B, pslices), pes >= 128 ? 512 : 256, psmem, st>>>(
      part, ntiles, cdiv(HW, 128), G, (long long)B * cdiv(HW, 128), conv_w, words, ws_b, ws_e, ws_t, dwe, dwords,
      dconv_w ? dwp : nullptr, C, E, T);
  if ((rc = check_launch("project_words_bwd_kernel"))) return rc;
  if (dconv_w) {
    sum_partials_kernel<<<dim3(cdiv(C * E, 128), 1), 128, 0, st>>>(dwp, B, (int64_t)C * E, 0, C * E, dconv_w);
    if ((rc = check_launch("sum_partials_kernel"))) return rc;
  }
  return 0;
}

extern "C" int agb_word_attn_bwd(const void* images, const float* words, int64_t ws_b, int64_t ws_e,
                                 int64_t ws_t, const float* conv_w, const int64_t* mask,
                                 const float* we, const void* dctx, int64_t dctx_bs, const void* dattn,
                                 void* dimages, float* dwords, float* dconv_w, void* workspace,
                                 size_t workspace_bytes, int B, int C, int HW, int E, int T,
                                 int io_dtype, int scaled, void* stream) {
  return word_attn_bwd_impl(false, images, words, ws_b, ws_e, ws_t, conv_w, mask, we, dctx, dctx_bs, 0, dattn, dimages,
                            dwords, dconv_w, workspace, workspace_bytes, B, C, HW, E, T, io_dtype, scaled, stream);
}

extern "C" int agb_word_attn_bwd_nhwc(const void* images, const float* words, int64_t ws_b, int64_t ws_e,
                                      int64_t ws_t, const float* conv_w, const int64_t* mask,
                                      const float* we, const void* dctx, int64_t dctx_bs, int64_t dctx_ps,
                                      const void* dattn, void* dimages, float* dwords, float* dconv_w,
                                      void* workspace, size_t workspace_bytes, int B, int C, int HW, int E, int T,
                                      int io_dtype, int scaled, void* stream) {
  return word_attn_bwd_impl(true, images, words, ws_b, ws_e, ws_t, conv_w, mask, we, dctx, dctx_bs, dctx_ps, dattn,
                            dimages, dwords, dconv_w, workspace, workspace_bytes, B, C, HW, E, T, io_dtype, scaled,
                            stream);
}
