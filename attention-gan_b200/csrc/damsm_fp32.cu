// DAMSM word-region similarity, AGB_MATH_FP32 path: fp32 arithmetic on the CUDA cores.
//
// Replaces the loop body of WordsLoss.get_loss (reference losses/words_loss.py:43-86) with the
// func_attention it calls (networks/attention.py:82-121), and its autograd (SURVEY.md row a9).
// This path exists for 1e-5 parity and as the on-device cross-check of the tcgen05 path
// (damsm_tc.cu); it stages the per-pair intermediates of a chunk of captions in a workspace:
//
//   Wp  [Bc,T,D]   packed words, zero for t >= L_i            (words_loss.py:51)
//   S   [Bi,N,R]   raw scores <w_n, c_r>, N = chunk*T          (attention.py:99)
//   Bt  [Bi,N,R]   beta = softmax_r(gamma1 * softmax_t(S/sqrt(D)))  (attention.py:101-112)
//   V   [Bi,N,D]   weighted context sum_r beta c_r              (attention.py:119)
//
// and for backward additionally G [Bi,N,R] (d beta, then the dW operand) and per-word scalars.
// All contractions go through sgemm_strided (fixed summation order, no atomics).
#include <algorithm>
#include <cooperative_groups.h>
#include "agb_common.cuh"

namespace agb {

struct Fp32Plan {
  int nc;  // captions per chunk
  size_t off_wp, off_pn, off_S, off_Bt, off_G, off_V, off_stat, total;
};

static Fp32Plan make_plan(int Bi, int Bc, int T, int D, int R) {
  Fp32Plan p;
  const size_t per_cap = (size_t)Bi * T * ((size_t)3 * R + D + 4) * sizeof(float);
  const size_t budget = (size_t)1 << 30;
  size_t nc = budget / per_cap;
  if (nc < 1) nc = 1;
  if (nc > (size_t)Bc) nc = Bc;
  p.nc = (int)nc;
  const size_t N = nc * T;
  size_t o = 0;
  p.off_wp = o;   o = align_up(o + (size_t)Bc * T * D * 4, 256);
  p.off_pn = o;   o = align_up(o + (size_t)Bc * T * 4, 256);
  p.off_S = o;    o = align_up(o + (size_t)Bi * N * R * 4, 256);
  p.off_Bt = o;   o = align_up(o + (size_t)Bi * N * R * 4, 256);
  p.off_G = o;    o = align_up(o + (size_t)Bi * N * R * 4, 256);
  p.off_V = o;    o = align_up(o + (size_t)Bi * N * D * 4, 256);
  p.off_stat = o; o = align_up(o + (size_t)Bi * N * 4 * 4, 256);
  p.total = o;
  return p;
}

size_t damsm_fp32_workspace_bytes(int Bi, int Bc, int T, int D, int R) {
  return make_plan(Bi, Bc, T, D, R).total;
}

// ---------------------------------------------------------------------------------------------
// pack words: Wp[i,t,:] = words[i,:,t] for t < L_i else 0; pn[i,t] = |w_it|    (words_loss.py:51)
// ---------------------------------------------------------------------------------------------
__global__ void pack_words_kernel(const float* __restrict__ words, int64_t ws_b, int64_t ws_d,
                                  int64_t ws_t, const int32_t* __restrict__ cap_lens,
                                  float* __restrict__ Wp, float* __restrict__ pn, int T, int D) {
  const int i = blockIdx.x, t = blockIdx.y;
  const int L = min(max(cap_lens[i], 0), T);
  const float* src = words + (int64_t)i * ws_b + (int64_t)t * ws_t;
  float* dst = Wp + ((size_t)i * T + t) * D;
  float ss = 0.f;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const float v = (t < L) ? src[(int64_t)d * ws_d] : 0.f;
    dst[d] = v;
    ss = fmaf(v, v, ss);
  }
  __shared__ float red[32];
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < (blockDim.x + 31) / 32; ++w) tot += red[w];
    pn[(size_t)i * T + t] = sqrtf(tot);
  }
}

// block-wide sum over threads of TMAX per-thread values -> out_s[t] (shared), all threads synced
template <int TMAX>
__device__ __forceinline__ void block_sum_words(const float (&v)[TMAX], int L, float* red_s /*[32*TMAX]*/,
                                                float* out_s /*[TMAX]*/) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int t = 0; t < TMAX; ++t) {
    if (t < L) {
      const float s = warp_sum(v[t]);
      if (lane == 0) red_s[warp * TMAX + t] = s;
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < L; t += blockDim.x) {
    float tot = 0.f;
    for (int w = 0; w < nw; ++w) tot += red_s[w * TMAX + t];
    out_s[t] = tot;
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// alpha / beta of one (image b, caption i) pair; thread = region             attention.py:101-115
//   in : S  [Bi,N,R] raw scores          out: Bt [Bi,N,R] beta (0 for t >= L)
//   att_out [Bi,T,R]: beta of the matched pair (words_loss.py:63); row_offset < 0: every block
//   cap_lens == nullptr: every caption has T words (func_attention)
// ---------------------------------------------------------------------------------------------
template <int TMAX, int MAXT>
__global__ void __launch_bounds__(MAXT) pair_softmax_kernel(const float* __restrict__ S, float* __restrict__ Bt,
                                    const int32_t* __restrict__ cap_lens, int i0, int N, int T, int R,
                                    float inv_sqrt_d, float gamma1, int row_offset,
                                    float* __restrict__ att_out) {
  __shared__ float red_s[32 * TMAX];
  __shared__ float z_s[TMAX];
  const int ic = blockIdx.x, b = blockIdx.y, r = threadIdx.x;
  // i0 < 0: "matched pairs" mode, block b pairs image b with caption row_offset + b
  const int i = i0 < 0 ? row_offset + b : i0 + ic;
  const int L = cap_lens ? min(max(cap_lens[i], 0), T) : T;
  const bool live = r < R;
  const size_t base = ((size_t)b * N + (size_t)ic * T) * R + r;
  float e[TMAX];
  float mx = -INFINITY;
#pragma unroll
  for (int t = 0; t < TMAX; ++t) {
    e[t] = 0.f;
    if (t < L && live) {
      e[t] = S[base + (size_t)t * R] * inv_sqrt_d;
      mx = fmaxf(mx, e[t]);
    }
  }
  float sum = 0.f;
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < L && live) {
      e[t] = __expf(e[t] - mx);
      sum += e[t];
    }
  const float inv = live ? 1.f / sum : 0.f;
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < L) e[t] = live ? __expf(gamma1 * (e[t] * inv)) : 0.f;  // gamma1*alpha in [0,gamma1]
  block_sum_words<TMAX>(e, L, red_s, z_s);
  const bool diag = att_out != nullptr && (row_offset < 0 || i == row_offset + b);
#pragma unroll
  for (int t = 0; t < TMAX; ++t) {
    if (t < T && live) {
      const float beta = (t < L) ? e[t] / z_s[t] : 0.f;
      Bt[base + (size_t)t * R] = beta;
      if (diag) att_out[((size_t)b * T + t) * R + r] = beta;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// cosine + gamma2 log-sum-exp of one pair; warp = word, lane = feature     words_loss.py:20-27,77-79
// mode 0 (forward): m_out[b,i] = log sum_t exp(gamma2 cos_t)
// mode 1 (backward): V <- dV = dn w + (dq/q) v;  stat[b,n] = {dn, kappa, dp/p, 0}
// ---------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(128)
pair_cosine_kernel(float* __restrict__ V, const float* __restrict__ Wp, const float* __restrict__ pn,
                   const int32_t* __restrict__ cap_lens, int i0, int N, int T, int D, int Bc,
                   float gamma2, float eps, float* __restrict__ m_out, const float* __restrict__ dm,
                   const float* __restrict__ gscale, float* __restrict__ stat) {
  __shared__ float n_s[64], q_s[64], c_s[64], dn_s[64], dqq_s[64];
  __shared__ float sum_s;
  const int ic = blockIdx.x, b = blockIdx.y;
  const int i = i0 + ic;
  const int L = min(max(cap_lens[i], 0), T);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* Vp = V + ((size_t)b * N + (size_t)ic * T) * D;
  const float* Wi = Wp + (size_t)i * T * D;
  for (int t = warp; t < L; t += 4) {
    float n = 0.f, q2 = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float v = Vp[(size_t)t * D + d];
      n = fmaf(Wi[(size_t)t * D + d], v, n);
      q2 = fmaf(v, v, q2);
    }
    n = warp_sum(n);
    q2 = warp_sum(q2);
    if (lane == 0) {
      const float q = sqrtf(q2);
      const float den = fmaxf(pn[(size_t)i * T + t] * q, eps);
      n_s[t] = n;
      q_s[t] = q;
      c_s[t] = n / den;
    }
  }
  __syncthreads();
  if (warp == 0) {
    float s = 0.f;
    for (int t = lane; t < L; t += 32) s += __expf(gamma2 * c_s[t]);
    s = warp_sum(s);
    if (lane == 0) {
      sum_s = s;
      if (MODE == 0) m_out[(size_t)b * Bc + i] = logf(s);
    }
  }
  if (MODE == 0) return;
  __syncthreads();
  const float up = dm[(size_t)b * Bc + i] * (gscale ? *gscale : 1.f);
  if ((int)threadIdx.x < T) {
    const int t = threadIdx.x;
    float dn = 0.f, dqq = 0.f, dpp = 0.f, kappa = 0.f;
    if (t < L) {
      const float dcos = up * gamma2 * __expf(gamma2 * c_s[t]) / sum_s;
      const float p = pn[(size_t)i * T + t], q = q_s[t], n = n_s[t];
      const float pq = p * q;
      const float den = fmaxf(pq, eps);
      dn = dcos / den;
      if (pq > eps) {  // gradient flows through the norms only when the clamp is inactive
        dqq = -dcos * n / (den * q * q);
        dpp = -dcos * n / (den * p * p);
      }
      kappa = dn * n + dqq * q * q;  // = sum_r beta dbeta
    }
    dn_s[t] = dn;
    dqq_s[t] = dqq;
    float4 st = make_float4(dn, kappa, dpp, 0.f);
    reinterpret_cast<float4*>(stat)[(size_t)b * N + (size_t)ic * T + t] = st;
  }
  __syncthreads();
  for (int t = warp; t < T; t += 4) {
    const float dn = dn_s[t], dqq = dqq_s[t];
    for (int d = lane; d < D; d += 32) {
      const size_t o = (size_t)t * D + d;
      Vp[o] = (t < L) ? fmaf(dn, Wi[o], dqq * Vp[o]) : 0.f;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// backward through both softmaxes of one pair; thread = region                (SURVEY row a9)
//   in : S raw scores, Bt beta, G = dbeta [Bi,N,R], stat {dn, kappa}
//   out: S <- ds / sqrt(D)                      (operand of the dC GEMM)
//        G <- dn * beta + ds / sqrt(D)          (operand of the dW GEMM)
// ---------------------------------------------------------------------------------------------
template <int TMAX, int MAXT>
__global__ void __launch_bounds__(MAXT) pair_softmax_bwd_kernel(float* __restrict__ S, const float* __restrict__ Bt,
                                        float* __restrict__ G, const float* __restrict__ stat,
                                        const int32_t* __restrict__ cap_lens, int i0, int N, int T,
                                        int R, float inv_sqrt_d, float gamma1) {
  __shared__ float dn_s[TMAX], kap_s[TMAX];
  const int ic = blockIdx.x, b = blockIdx.y, r = threadIdx.x;
  const int i = i0 + ic;
  const int L = min(max(cap_lens[i], 0), T);
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    const float4 st = reinterpret_cast<const float4*>(stat)[(size_t)b * N + (size_t)ic * T + t];
    dn_s[t] = st.x;
    kap_s[t] = st.y;
  }
  __syncthreads();
  if (r >= R) return;
  const size_t base = ((size_t)b * N + (size_t)ic * T) * R + r;
  float a[TMAX];
  float mx = -INFINITY;
#pragma unroll
  for (int t = 0; t < TMAX; ++t) {
    a[t] = 0.f;
    if (t < L) {
      a[t] = S[base + (size_t)t * R] * inv_sqrt_d;
      mx = fmaxf(mx, a[t]);
    }
  }
  float sum = 0.f;
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < L) {
      a[t] = __expf(a[t] - mx);
      sum += a[t];
    }
  const float inv = 1.f / sum;
  float da[TMAX];
  float dot = 0.f;
#pragma unroll
  for (int t = 0; t < TMAX; ++t) {
    da[t] = 0.f;
    if (t < L) {
      a[t] *= inv;  // alpha
      const float beta = Bt[base + (size_t)t * R];
      da[t] = gamma1 * beta * (G[base + (size_t)t * R] - kap_s[t]);  // d alpha
      dot = fmaf(a[t], da[t], dot);
    }
  }
#pragma unroll
  for (int t = 0; t < TMAX; ++t) {
    if (t < T) {
      float ds = 0.f, g = 0.f;
      if (t < L) {
        ds = a[t] * (da[t] - dot) * inv_sqrt_d;
        g = fmaf(dn_s[t], Bt[base + (size_t)t * R], ds);
      }
      S[base + (size_t)t * R] = ds;
      G[base + (size_t)t * R] = g;
    }
  }
}

// dwords[n,:] += (sum_b dp/p [b,n]) * w_n                       (cosine backward, word-norm term)
__global__ void dwords_norm_term_kernel(float* __restrict__ dW, const float* __restrict__ Wp,
                                        const float* __restrict__ stat, int Bi, int N, int D) {
  const int n = blockIdx.x;
  __shared__ float tot_s;
  float acc = 0.f;
  for (int b = threadIdx.x; b < Bi; b += blockDim.x) acc += stat[((size_t)b * N + n) * 4 + 2];
  __shared__ float red[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < (blockDim.x + 31) / 32; ++w) t += red[w];
    tot_s = t;
  }
  __syncthreads();
  const float tot = tot_s;
  for (int d = threadIdx.x; d < D; d += blockDim.x) dW[(size_t)n * D + d] = fmaf(tot, Wp[(size_t)n * D + d], dW[(size_t)n * D + d]);
}

static int pick_tmax(int T) { return T <= 8 ? 8 : T <= 16 ? 16 : T <= 24 ? 24 : T <= 32 ? 32 : 64; }

#define AGB_TMAX_SWITCH(TM, ...)                                  \
  switch (TM) {                                                   \
    case 8: { constexpr int TMAX = 8; __VA_ARGS__; } break;       \
    case 16: { constexpr int TMAX = 16; __VA_ARGS__; } break;     \
    case 24: { constexpr int TMAX = 24; __VA_ARGS__; } break;     \
    case 32: { constexpr int TMAX = 32; __VA_ARGS__; } break;     \
    default: { constexpr int TMAX = 64; __VA_ARGS__; } break;     \
  }

// scores, beta and weighted context of captions [i0, i0+nc) against every image
static int chunk_forward(const float* img, const Fp32Plan& p, char* ws, const int32_t* cap_lens, int i0,
                         int nc, int Bi, int T, int D, int R, float gamma1, int row_offset,
                         float* att_out, cudaStream_t st) {
  const int N = nc * T;
  const float* Wp = (const float*)(ws + p.off_wp);
  float* S = (float*)(ws + p.off_S);
  float* Bt = (float*)(ws + p.off_Bt);
  float* V = (float*)(ws + p.off_V);
  // S[b][n,r] = sum_d Wp[i0*T+n, d] * img[b][d, r]                                attention.py:99
  SgemmArgs g{};
  g.A = Wp + (size_t)i0 * T * D; g.a_m = D; g.a_k = 1; g.a_kb = 0; g.a_batch = 0;
  g.B = img; g.b_k = R; g.b_n = 1; g.b_kb = 0; g.b_batch = (int64_t)D * R;
  g.C = S; g.c_m = R; g.c_n = 1; g.c_batch = (int64_t)N * R;
  g.M = N; g.N = R; g.K = D; g.KB = 1; g.alpha = 1.f; g.accumulate = 0;
  if (int rc = sgemm_strided(g, Bi, st)) return rc;
  const int threads = (R + 31) / 32 * 32;
  const int tm = pick_tmax(T);
  AGB_TMAX_SWITCH(tm, {
    if (threads <= 352) pair_softmax_kernel<TMAX, 352><<<dim3(nc, Bi), threads, 0, st>>>(
        S, Bt, cap_lens, i0, N, T, R, 1.f / sqrtf((float)D), gamma1, row_offset, att_out);
    else pair_softmax_kernel<TMAX, 1024><<<dim3(nc, Bi), threads, 0, st>>>(
        S, Bt, cap_lens, i0, N, T, R, 1.f / sqrtf((float)D), gamma1, row_offset, att_out);
  });
  if (int rc = check_launch("pair_softmax_kernel")) return rc;
  // V[b][n,d] = sum_r Bt[b][n,r] * img[b][d,r]                                    attention.py:119
  g.A = Bt; g.a_m = R; g.a_k = 1; g.a_batch = (int64_t)N * R;
  g.B = img; g.b_k = 1; g.b_n = R; g.b_batch = (int64_t)D * R;
  g.C = V; g.c_m = D; g.c_n = 1; g.c_batch = (int64_t)N * D;
  g.M = N; g.N = D; g.K = R;
  return sgemm_strided(g, Bi, st);
}

static int check_shape(int Bi, int Bc, int T, int D, int R) {
  if (Bi <= 0 || Bc <= 0 || T <= 0 || D <= 0 || R <= 0) return fail_arg("non-positive size Bi=%d Bc=%d T=%d D=%d R=%d", Bi, Bc, T, D, R);
  if (T > 64) return fail_unsupported("T=%d > 64 words is outside the compiled range", T);
  if (R > 1024) return fail_unsupported("R=%d > 1024 regions is outside the compiled range", R);
  if (Bi > 65535) return fail_unsupported("Bi=%d > 65535", Bi);
  return 0;
}

int damsm_fp32_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                   const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1,
                   float gamma2, float eps, int row_offset, float* m_out, float* att_out,
                   void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (int rc = check_shape(Bi, Bc, T, D, R)) return rc;
  const Fp32Plan p = make_plan(Bi, Bc, T, D, R);
  if (workspace_bytes < p.total) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, p.total);
    return AGB_E_WORKSPACE;
  }
  char* ws = (char*)workspace;
  float* Wp = (float*)(ws + p.off_wp);
  float* pn = (float*)(ws + p.off_pn);
  pack_words_kernel<<<dim3(Bc, T), 128, 0, st>>>(words, ws_b, ws_d, ws_t, cap_lens, Wp, pn, T, D);
  if (int rc = check_launch("pack_words_kernel")) return rc;
  for (int i0 = 0; i0 < Bc; i0 += p.nc) {
    const int nc = min(p.nc, Bc - i0);
    if (int rc = chunk_forward(img, p, ws, cap_lens, i0, nc, Bi, T, D, R, gamma1, row_offset, att_out, st)) return rc;
    pair_cosine_kernel<0><<<dim3(nc, Bi), 128, 0, st>>>((float*)(ws + p.off_V), Wp, pn, cap_lens, i0, nc * T, T,
                                                       D, Bc, gamma2, eps, m_out, nullptr, nullptr, nullptr);
    if (int rc = check_launch("pair_cosine_kernel<0>")) return rc;
  }
  return 0;
}

int damsm_fp32_bwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                   const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1,
                   float gamma2, float eps, const float* dm, const float* gscale, float* dimg,
                   float* dwords, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (int rc = check_shape(Bi, Bc, T, D, R)) return rc;
  const Fp32Plan p = make_plan(Bi, Bc, T, D, R);
  if (workspace_bytes < p.total) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, p.total);
    return AGB_E_WORKSPACE;
  }
  char* ws = (char*)workspace;
  float* Wp = (float*)(ws + p.off_wp);
  float* pn = (float*)(ws + p.off_pn);
  float* S = (float*)(ws + p.off_S);
  float* Bt = (float*)(ws + p.off_Bt);
  float* G = (float*)(ws + p.off_G);
  float* V = (float*)(ws + p.off_V);
  float* stat = (float*)(ws + p.off_stat);
  const float isd = 1.f / sqrtf((float)D);
  pack_words_kernel<<<dim3(Bc, T), 128, 0, st>>>(words, ws_b, ws_d, ws_t, cap_lens, Wp, pn, T, D);
  if (int rc = check_launch("pack_words_kernel")) return rc;
  const int threads = (R + 31) / 32 * 32;
  const int tm = pick_tmax(T);
  for (int i0 = 0; i0 < Bc; i0 += p.nc) {
    const int nc = min(p.nc, Bc - i0);
    const int N = nc * T;
    if (int rc = chunk_forward(img, p, ws, cap_lens, i0, nc, Bi, T, D, R, gamma1, 0, nullptr, st)) return rc;
    // dV and the per-word scalars of the cosine / LSE backward
    pair_cosine_kernel<1><<<dim3(nc, Bi), 128, 0, st>>>(V, Wp, pn, cap_lens, i0, N, T, D, Bc, gamma2, eps,
                                                       nullptr, dm, gscale, stat);
    if (int rc = check_launch("pair_cosine_kernel<1>")) return rc;
    // G[b][n,r] = dbeta = sum_d dV[b][n,d] * img[b][d,r]
    SgemmArgs g{};
    g.A = V; g.a_m = D; g.a_k = 1; g.a_batch = (int64_t)N * D;
    g.B = img; g.b_k = R; g.b_n = 1; g.b_batch = (int64_t)D * R;
    g.C = G; g.c_m = R; g.c_n = 1; g.c_batch = (int64_t)N * R;
    g.M = N; g.N = R; g.K = D; g.KB = 1; g.alpha = 1.f; g.accumulate = 0;
    if (int rc = sgemm_strided(g, Bi, st)) return rc;
    AGB_TMAX_SWITCH(tm, {
      if (threads <= 352) pair_softmax_bwd_kernel<TMAX, 352><<<dim3(nc, Bi), threads, 0, st>>>(
          S, Bt, G, stat, cap_lens, i0, N, T, R, isd, gamma1);
      else pair_softmax_bwd_kernel<TMAX, 1024><<<dim3(nc, Bi), threads, 0, st>>>(
          S, Bt, G, stat, cap_lens, i0, N, T, R, isd, gamma1);
    });
    if (int rc = check_launch("pair_softmax_bwd_kernel")) return rc;
    // dimg[b][d,r] (+)= sum_n dV[b][n,d] beta[b][n,r] + sum_n Wp[n,d] ds[b][n,r]/sqrt(D)
    g.A = V; g.a_m = 1; g.a_k = D; g.a_batch = (int64_t)N * D;
    g.B = Bt; g.b_k = R; g.b_n = 1; g.b_batch = (int64_t)N * R;
    g.C = dimg; g.c_m = R; g.c_n = 1; g.c_batch = (int64_t)D * R;
    g.M = D; g.N = R; g.K = N; g.accumulate = (i0 > 0);
    if (int rc = sgemm_strided(g, Bi, st)) return rc;
    g.A = Wp + (size_t)i0 * T * D; g.a_batch = 0;
    g.B = S; g.accumulate = 1;
    if (int rc = sgemm_strided(g, Bi, st)) return rc;
    if (dwords) {
      // dwords[n,d] = sum_b sum_r G[b][n,r] img[b][d,r]  (+ word-norm term)
      SgemmArgs h{};
      h.A = G; h.a_m = R; h.a_k = 1; h.a_kb = (int64_t)N * R; h.a_batch = 0;
      h.B = img; h.b_k = 1; h.b_n = R; h.b_kb = (int64_t)D * R; h.b_batch = 0;
      h.C = dwords + (size_t)i0 * T * D; h.c_m = D; h.c_n = 1; h.c_batch = 0;
      h.M = N; h.N = D; h.K = R; h.KB = Bi; h.alpha = 1.f; h.accumulate = 0;
      if (int rc = sgemm_strided(h, 1, st)) return rc;
      dwords_norm_term_kernel<<<N, 128, 0, st>>>(dwords + (size_t)i0 * T * D, Wp + (size_t)i0 * T * D, stat, Bi, N, D);
      if (int rc = check_launch("dwords_norm_term_kernel")) return rc;
    }
  }
  return 0;
}

}  // namespace agb

// =============================================================================================
// functional region-word attention on its own          reference networks/attention.py:82-121
// Same building blocks with one "caption" per sample (query b against context b only).
// =============================================================================================
namespace agb {

// backward of both softmaxes when the upstream gradient is arbitrary (dwc and optionally dattn):
//   G = dbeta (+ dattn);  kappa_t = sum_r beta dbeta (block reduction);  out: S <- ds (scaled)
template <int TMAX, int MAXT>
__global__ void __launch_bounds__(MAXT) func_softmax_bwd_kernel(float* __restrict__ S, const float* __restrict__ Bt,
                                        const float* __restrict__ G, const float* __restrict__ dattn,
                                        int T, int R, float scale, float gamma1) {
  __shared__ float red_s[32 * TMAX];
  __shared__ float kap_s[TMAX];
  const int b = blockIdx.x, r = threadIdx.x;
  const bool live = r < R;
  const size_t base = (size_t)b * T * R + r;
  float a[TMAX], be[TMAX], g[TMAX], bg[TMAX];
  float mx = -INFINITY;
#pragma unroll
  for (int t = 0; t < TMAX; ++t) {
    a[t] = be[t] = g[t] = bg[t] = 0.f;
    if (t < T && live) {
      a[t] = S[base + (size_t)t * R] * scale;
      mx = fmaxf(mx, a[t]);
      be[t] = Bt[base + (size_t)t * R];
      g[t] = G[base + (size_t)t * R] + (dattn ? dattn[base + (size_t)t * R] : 0.f);
      bg[t] = be[t] * g[t];
    }
  }
  block_sum_words<TMAX>(bg, T, red_s, kap_s);
  if (!live) return;
  float sum = 0.f;
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < T) {
      a[t] = __expf(a[t] - mx);
      sum += a[t];
    }
  const float inv = 1.f / sum;
  float dot = 0.f;
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < T) {
      a[t] *= inv;
      g[t] = gamma1 * be[t] * (g[t] - kap_s[t]);  // d alpha
      dot = fmaf(a[t], g[t], dot);
    }
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < T) S[base + (size_t)t * R] = a[t] * (g[t] - dot) * scale;
}

static int func_check(int B, int D, int L, int R) {
  if (B <= 0 || D <= 0 || L <= 0 || R <= 0) return fail_arg("non-positive size B=%d D=%d L=%d R=%d", B, D, L, R);
  if (L > 64) return fail_unsupported("L=%d > 64 words is outside the compiled range", L);
  if (R > 1024) return fail_unsupported("R=%d > 1024 regions is outside the compiled range", R);
  if (B > 65535) return fail_unsupported("B=%d > 65535", B);
  return 0;
}

// S[b][t,r] and beta[b][t,r] of the B diagonal pairs
static int func_scores(const float* query, int64_t qs_b, int64_t qs_d, int64_t qs_t, const float* context,
                       int B, int D, int L, int R, float gamma1, float scale, float* S, float* Bt,
                       float* attn_out, cudaStream_t st) {
  SgemmArgs g{};
  g.A = query; g.a_m = qs_t; g.a_k = qs_d; g.a_batch = qs_b;
  g.B = context; g.b_k = R; g.b_n = 1; g.b_batch = (int64_t)D * R;
  g.C = S; g.c_m = R; g.c_n = 1; g.c_batch = (int64_t)L * R;
  g.M = L; g.N = R; g.K = D; g.KB = 1; g.alpha = 1.f; g.accumulate = 0;
  if (int rc = sgemm_strided(g, B, st)) return rc;
  const int threads = (R + 31) / 32 * 32;
  AGB_TMAX_SWITCH(pick_tmax(L), {
    if (threads <= 352) pair_softmax_kernel<TMAX, 352><<<dim3(1, B), threads, 0, st>>>(
        S, Bt, nullptr, 0, L, L, R, scale, gamma1, -1, attn_out);
    else pair_softmax_kernel<TMAX, 1024><<<dim3(1, B), threads, 0, st>>>(
        S, Bt, nullptr, 0, L, L, R, scale, gamma1, -1, attn_out);
  });
  return check_launch("pair_softmax_kernel");
}

// beta of the matched pairs only (image b, caption row_offset + b), fp32: the att_maps output of
// WordsLoss (words_loss.py:63) for the tensor-core path.  One block per image, thread = region:
// scores over the feature dim with the caption's words broadcast from shared memory, both softmaxes
// in registers (S, Bt: unused scratch kept for ABI stability of the internal call).
// The feature dimension is split over the CTAs of a thread-block cluster (blockIdx.y = slice): every CTA
// accumulates the raw scores of its slice, the partial sums meet in the leader through distributed
// shared memory in a fixed order, and the leader finishes the two softmaxes.
// Body of one block.  pick(b, i, o) chooses image b, caption i and the att_out slot o of the block; when it returns
// false the block writes NaN maps instead (pick is the same for every CTA of a cluster, so the cluster returns as
// one).
template <int TMAX, class Pick>
__device__ __forceinline__ void att_maps_block(const float* __restrict__ img, const float* __restrict__ words,
                                               int64_t ws_b, int64_t ws_d, int64_t ws_t,
                                               const int32_t* __restrict__ cap_lens, int T, int D, int R,
                                               float inv_sqrt_d, float gamma1, Pick pick,
                                               float* __restrict__ att_out) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  extern __shared__ float w_s[];                  // [slice of D][TMAX] words, then [TMAX][blockDim.x] partial scores
  const int parts = gridDim.y, part = blockIdx.y, tpr = blockDim.x;
  const int d0 = (int)((long long)D * part / parts), d1 = (int)((long long)D * (part + 1) / parts);
  float* acc_s = w_s + (size_t)((D + parts - 1) / parts + 1) * TMAX;
  __shared__ float red_s[32 * TMAX];
  __shared__ float z_s[TMAX];
  int b, i, o;
  if (!pick(b, i, o)) {
    if (part == 0 && (int)threadIdx.x < R)
      for (int t = 0; t < T; ++t) att_out[((size_t)o * T + t) * R + threadIdx.x] = __int_as_float(0x7fc00000);
    return;
  }
  const int r = threadIdx.x;
  const int L = min(max(cap_lens[i], 0), T);
  for (int k = threadIdx.x; k < (d1 - d0) * TMAX; k += blockDim.x) {
    const int d = k / TMAX, t = k - d * TMAX;
    w_s[k] = (t < L) ? words[(int64_t)i * ws_b + (int64_t)(d0 + d) * ws_d + (int64_t)t * ws_t] : 0.f;
  }
  __syncthreads();
  const bool live = r < R;
  float e[TMAX];
#pragma unroll
  for (int t = 0; t < TMAX; ++t) e[t] = 0.f;
  if (live) {
    const float* c = img + (size_t)b * D * R + (size_t)d0 * R + r;
#pragma unroll 8
    for (int d = 0; d < d1 - d0; ++d) {
      const float cv = c[(size_t)d * R];
      const float4* w4 = reinterpret_cast<const float4*>(w_s + d * TMAX);
#pragma unroll
      for (int t4 = 0; t4 < TMAX / 4; ++t4) {
        const float4 w = w4[t4];
        e[4 * t4] = fmaf(cv, w.x, e[4 * t4]);
        e[4 * t4 + 1] = fmaf(cv, w.y, e[4 * t4 + 1]);
        e[4 * t4 + 2] = fmaf(cv, w.z, e[4 * t4 + 2]);
        e[4 * t4 + 3] = fmaf(cv, w.w, e[4 * t4 + 3]);
      }
    }
  }
  if (part > 0) {
#pragma unroll
    for (int t = 0; t < TMAX; ++t) acc_s[t * tpr + r] = e[t];
  }
  cluster.sync();
  if (part == 0) {
    for (int pp = 1; pp < parts; ++pp) {           // fixed order -> deterministic
      const float* remote = cluster.map_shared_rank(acc_s, pp);
#pragma unroll
      for (int t = 0; t < TMAX; ++t) e[t] += remote[t * tpr + r];
    }
  }
  cluster.sync();                                  // the slices' shared memory stays alive until it has been read
  if (part > 0) return;
  float mx = -INFINITY;
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < L) {
      e[t] *= inv_sqrt_d;
      mx = fmaxf(mx, e[t]);
    }
  float sum = 0.f;
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < L) {
      e[t] = __expf(e[t] - mx);
      sum += e[t];
    }
  const float inv = 1.f / sum;
#pragma unroll
  for (int t = 0; t < TMAX; ++t) e[t] = (t < L && live) ? __expf(gamma1 * (e[t] * inv)) : 0.f;
  block_sum_words<TMAX>(e, L, red_s, z_s);
  if (!live) return;
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < T) att_out[((size_t)o * T + t) * R + r] = (t < L) ? e[t] / z_s[t] : 0.f;
}

template <int TMAX>
__global__ void __launch_bounds__(1024)
diag_att_kernel(const float* __restrict__ img, const float* __restrict__ words, int64_t ws_b, int64_t ws_d,
                int64_t ws_t, const int32_t* __restrict__ cap_lens, int T, int D, int R, float inv_sqrt_d,
                float gamma1, int row_offset, float* __restrict__ att_out) {
  auto pick = [&](int& b, int& i, int& o) {
    b = blockIdx.x;
    i = row_offset + b;
    o = b;
    return true;
  };
  att_maps_block<TMAX>(img, words, ws_b, ws_d, ws_t, cap_lens, T, D, R, inv_sqrt_d, gamma1, pick, att_out);
}

// beta of listed pairs (agb_damsm_pairs_fwd): block p = image pair_img[p], caption pair_cap[p], with the arithmetic
// of diag_att_kernel.  A pair whose image or caption index is out of range, or whose caption has length 0, gets NaN
// maps.
template <int TMAX>
__global__ void __launch_bounds__(1024)
pair_att_kernel(const float* __restrict__ img, const float* __restrict__ words, int64_t ws_b, int64_t ws_d,
                int64_t ws_t, const int32_t* __restrict__ cap_lens, int Bi, int Bc, const int32_t* __restrict__ pair_img,
                const int32_t* __restrict__ pair_cap, int T, int D, int R, float inv_sqrt_d, float gamma1,
                float* __restrict__ att_out) {
  auto pick = [&](int& b, int& i, int& o) {
    o = blockIdx.x;
    b = pair_img[o];
    i = pair_cap[o];
    return b >= 0 && b < Bi && i >= 0 && i < Bc && cap_lens[i] > 0;
  };
  att_maps_block<TMAX>(img, words, ws_b, ws_d, ws_t, cap_lens, T, D, R, inv_sqrt_d, gamma1, pick, att_out);
}

int damsm_diag_att_maps(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                        const int32_t* cap_lens, int Bi, int T, int D, int R, float gamma1, int row_offset,
                        float* att_out, float* S, float* Bt, cudaStream_t st) {
  (void)S;
  (void)Bt;
  const int tpr = (R + 31) / 32 * 32;
  if (tpr > 1024) return fail_unsupported("R=%d regions > 1024", R);
  const int parts = D >= 64 ? 4 : 1;              // cluster size: slices of the feature dimension
  const float isd = 1.f / sqrtf((float)D);
  const int tm = pick_tmax(T);
  const size_t smem = ((size_t)((D + parts - 1) / parts + 1) * tm + (size_t)tm * tpr) * sizeof(float);
  AGB_TMAX_SWITCH(tm, {
    auto kern = diag_att_kernel<TMAX>;
    if (smem > 48 * 1024) AGB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(Bi, parts);
    cfg.blockDim = dim3(tpr);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 1;
    attr[0].val.clusterDim.y = parts;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    AGB_CUDA(cudaLaunchKernelEx(&cfg, kern, img, words, ws_b, ws_d, ws_t, cap_lens, T, D, R, isd, gamma1, row_offset,
                                att_out));
  });
  return check_launch("diag_att_kernel");
}

int damsm_pair_att_maps(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                        const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap,
                        int P, int T, int D, int R, float gamma1, float* att_out, cudaStream_t st) {
  const int tpr = (R + 31) / 32 * 32;
  if (tpr > 1024) return fail_unsupported("R=%d regions > 1024", R);
  const int parts = D >= 64 ? 4 : 1;              // the cluster split of damsm_diag_att_maps
  const float isd = 1.f / sqrtf((float)D);
  const int tm = pick_tmax(T);
  const size_t smem = ((size_t)((D + parts - 1) / parts + 1) * tm + (size_t)tm * tpr) * sizeof(float);
  AGB_TMAX_SWITCH(tm, {
    auto kern = pair_att_kernel<TMAX>;
    if (smem > 48 * 1024) AGB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(P, parts);
    cfg.blockDim = dim3(tpr);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 1;
    attr[0].val.clusterDim.y = parts;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    AGB_CUDA(cudaLaunchKernelEx(&cfg, kern, img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, pair_img, pair_cap, T, D, R,
                                isd, gamma1, att_out));
  });
  return check_launch("pair_att_kernel");
}

}  // namespace agb

using namespace agb;

extern "C" size_t agb_func_attention_workspace_bytes(int B, int L, int R) {
  if (B <= 0 || L <= 0 || R <= 0) return 0;
  return (size_t)3 * align_up((size_t)B * L * R * sizeof(float), 256);
}

extern "C" int agb_func_attention_fwd(const float* query, int64_t qs_b, int64_t qs_d, int64_t qs_t,
                                      const float* context, int B, int D, int L, int R, float gamma1,
                                      int scaled, float* wc_out, float* attn_out, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  if (int rc = func_check(B, D, L, R)) return rc;
  if (!query || !context || !wc_out || !workspace) return fail_arg("null pointer");
  if (workspace_bytes < agb_func_attention_workspace_bytes(B, L, R)) {
    set_error("workspace too small");
    return AGB_E_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const size_t blk = align_up((size_t)B * L * R * sizeof(float), 256);
  float* S = (float*)workspace;
  float* Bt = (float*)((char*)workspace + blk);
  const float scale = scaled ? 1.f / sqrtf((float)D) : 1.f;
  if (int rc = func_scores(query, qs_b, qs_d, qs_t, context, B, D, L, R, gamma1, scale, S, Bt, attn_out, st)) return rc;
  // wc[b][d,t] = sum_r context[b][d,r] beta[b][t,r]                              attention.py:119
  SgemmArgs g{};
  g.A = context; g.a_m = R; g.a_k = 1; g.a_batch = (int64_t)D * R;
  g.B = Bt; g.b_k = 1; g.b_n = R; g.b_batch = (int64_t)L * R;
  g.C = wc_out; g.c_m = L; g.c_n = 1; g.c_batch = (int64_t)D * L;
  g.M = D; g.N = L; g.K = R; g.KB = 1; g.alpha = 1.f; g.accumulate = 0;
  return sgemm_strided(g, B, st);
}

extern "C" int agb_func_attention_bwd(const float* query, int64_t qs_b, int64_t qs_d, int64_t qs_t,
                                      const float* context, int B, int D, int L, int R, float gamma1,
                                      int scaled, const float* dwc, const float* dattn, float* dquery,
                                      float* dcontext, void* workspace, size_t workspace_bytes,
                                      void* stream) {
  if (int rc = func_check(B, D, L, R)) return rc;
  if (!query || !context || !dwc || !workspace) return fail_arg("null pointer");
  if (workspace_bytes < agb_func_attention_workspace_bytes(B, L, R)) {
    set_error("workspace too small");
    return AGB_E_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const size_t blk = align_up((size_t)B * L * R * sizeof(float), 256);
  float* S = (float*)workspace;
  float* Bt = (float*)((char*)workspace + blk);
  float* G = (float*)((char*)workspace + 2 * blk);
  const float scale = scaled ? 1.f / sqrtf((float)D) : 1.f;
  if (int rc = func_scores(query, qs_b, qs_d, qs_t, context, B, D, L, R, gamma1, scale, S, Bt, nullptr, st)) return rc;
  // G[b][t,r] = sum_d dwc[b][d,t] context[b][d,r]
  SgemmArgs g{};
  g.A = dwc; g.a_m = 1; g.a_k = L; g.a_batch = (int64_t)D * L;
  g.B = context; g.b_k = R; g.b_n = 1; g.b_batch = (int64_t)D * R;
  g.C = G; g.c_m = R; g.c_n = 1; g.c_batch = (int64_t)L * R;
  g.M = L; g.N = R; g.K = D; g.KB = 1; g.alpha = 1.f; g.accumulate = 0;
  if (int rc = sgemm_strided(g, B, st)) return rc;
  const int threads = (R + 31) / 32 * 32;
  AGB_TMAX_SWITCH(pick_tmax(L), {
    if (threads <= 352) func_softmax_bwd_kernel<TMAX, 352><<<B, threads, 0, st>>>(S, Bt, G, dattn, L, R, scale, gamma1);
    else func_softmax_bwd_kernel<TMAX, 1024><<<B, threads, 0, st>>>(S, Bt, G, dattn, L, R, scale, gamma1);
  });
  if (int rc = check_launch("func_softmax_bwd_kernel")) return rc;
  if (dquery) {  // dquery[b][d,t] = sum_r context[b][d,r] ds[b][t,r]
    g.A = context; g.a_m = R; g.a_k = 1; g.a_batch = (int64_t)D * R;
    g.B = S; g.b_k = 1; g.b_n = R; g.b_batch = (int64_t)L * R;
    g.C = dquery; g.c_m = L; g.c_n = 1; g.c_batch = (int64_t)D * L;
    g.M = D; g.N = L; g.K = R;
    if (int rc = sgemm_strided(g, B, st)) return rc;
  }
  if (dcontext) {  // dcontext[b][d,r] = sum_t dwc[b][d,t] beta[b][t,r] + query[b][d,t] ds[b][t,r]
    g.A = dwc; g.a_m = L; g.a_k = 1; g.a_batch = (int64_t)D * L;
    g.B = Bt; g.b_k = R; g.b_n = 1; g.b_batch = (int64_t)L * R;
    g.C = dcontext; g.c_m = R; g.c_n = 1; g.c_batch = (int64_t)D * R;
    g.M = D; g.N = R; g.K = L; g.accumulate = 0;
    if (int rc = sgemm_strided(g, B, st)) return rc;
    g.A = query; g.a_m = qs_d; g.a_k = qs_t; g.a_batch = qs_b;
    g.B = S; g.accumulate = 1;
    if (int rc = sgemm_strided(g, B, st)) return rc;
  }
  return 0;
}
