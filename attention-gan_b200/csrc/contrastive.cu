// Two-way contrastive cross-entropy over the B x B similarity matrix, and the sentence cosine
// matrix with its backward.
//
// Replaces reference losses/words_loss.py:88-101 and losses/sentence_loss.py:14-25,33-49:
//   logits = gamma3 * raw;  logits[a,b] = -inf where class_ids[a]==class_ids[b], a != b;
//   loss = lambda * (mean_b CE(logits[b,:], labels[b]) + mean_i CE(logits[:,i], labels[i]))
// The gradient w.r.t. raw comes out of the same call (softmax weights are already at hand), so the
// DAMSM backward kernels start from dLoss/draw.  Fixed reduction order, no atomics.
#include "agb_common.cuh"

namespace agb {

__device__ __forceinline__ float logit_at(const float* __restrict__ raw, const int32_t* __restrict__ cls,
                                          int B, int a, int b, float gamma3) {
  if (cls != nullptr && a != b && cls[a] == cls[b]) return -INFINITY;
  return gamma3 * raw[(size_t)a * B + b];
}

__device__ __forceinline__ void lse_push(float& m, float& s, float x) {
  if (x == -INFINITY) return;
  if (x > m) {
    s = s * __expf(m - x) + 1.f;
    m = x;
  } else {
    s += __expf(x - m);
  }
}
__device__ __forceinline__ void lse_merge(float& m, float& s, float m2, float s2) {
  if (m2 == -INFINITY) return;
  if (m == -INFINITY) { m = m2; s = s2; return; }
  const float mm = fmaxf(m, m2);
  s = s * __expf(m - mm) + s2 * __expf(m2 - mm);
  m = mm;
}

// one block per row a: lse over the columns
__global__ void ce_row_kernel(const float* __restrict__ raw, int B, const int32_t* __restrict__ cls,
                              const int64_t* __restrict__ labels, float gamma3, float* __restrict__ lse_r,
                              float* __restrict__ part_r) {
  const int a = blockIdx.x;
  float m = -INFINITY, s = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) lse_push(m, s, logit_at(raw, cls, B, a, b, gamma3));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
    lse_merge(m, s, m2, s2);
  }
  __shared__ float ms[32], ss[32];
  if ((threadIdx.x & 31) == 0) { ms[threadIdx.x >> 5] = m; ss[threadIdx.x >> 5] = s; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float M = -INFINITY, S = 0.f;
    for (int w = 0; w < (blockDim.x + 31) / 32; ++w) lse_merge(M, S, ms[w], ss[w]);
    const float lse = M + logf(S);
    lse_r[a] = lse;
    part_r[a] = lse - logit_at(raw, cls, B, a, (int)labels[a], gamma3);
  }
}

// one block per 32 columns, 32 x 8 threads: thread (tx, ty) folds rows ty, ty+8, ... of column tx
// (adjacent threads read adjacent columns), then the 8 partial (max, sum) pairs are merged in order
__global__ void __launch_bounds__(256)
ce_col_kernel(const float* __restrict__ raw, int B, const int32_t* __restrict__ cls,
              const int64_t* __restrict__ labels, float gamma3, float* __restrict__ lse_c,
              float* __restrict__ part_c) {
  __shared__ float ms[8][33], ss[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int b = blockIdx.x * 32 + tx;
  float m = -INFINITY, s = 0.f;
  if (b < B)
    for (int a = ty; a < B; a += 8) lse_push(m, s, logit_at(raw, cls, B, a, b, gamma3));
  ms[ty][tx] = m;
  ss[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && b < B) {
    float M = -INFINITY, S = 0.f;
    for (int k = 0; k < 8; ++k) lse_merge(M, S, ms[k][tx], ss[k][tx]);
    const float lse = M + logf(S);
    lse_c[b] = lse;
    part_c[b] = lse - logit_at(raw, cls, B, (int)labels[b], b, gamma3);
  }
}

__global__ void ce_loss_kernel(const float* __restrict__ part_r, const float* __restrict__ part_c, int B,
                               float lambda, float* __restrict__ loss_out) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < B; i += blockDim.x) acc += part_r[i] + part_c[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < (blockDim.x + 31) / 32; ++w) t += red[w];
    loss_out[0] = lambda * t / (float)B;
  }
}

__global__ void ce_grad_kernel(const float* __restrict__ raw, int B, const int32_t* __restrict__ cls,
                               const int64_t* __restrict__ labels, float gamma3, float lambda,
                               const float* __restrict__ lse_r, const float* __restrict__ lse_c,
                               int row_begin, int row_count, float* __restrict__ draw) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int a = row_begin + blockIdx.y;
  if (b >= B || (int)blockIdx.y >= row_count) return;
  const float l = logit_at(raw, cls, B, a, b, gamma3);
  float d = 0.f;
  if (l != -INFINITY) {
    d = __expf(l - lse_r[a]) + __expf(l - lse_c[b]);
    if ((int)labels[a] == b) d -= 1.f;
    if ((int)labels[b] == a) d -= 1.f;
    d *= lambda * gamma3 / (float)B;
  }
  draw[(size_t)blockIdx.y * B + b] = d;
}

// Whole two-way CE in one CTA for B <= 128 (the reference's batch sizes: 16-64): logits live in
// shared memory, warp w folds rows w, w+32, ... and then columns w, w+32, ... with the same in-order
// merges as the multi-kernel path, loss and the requested gradient rows come out of the same launch.
__global__ void __launch_bounds__(1024)
ce_small_kernel(const float* __restrict__ raw, int B, const int32_t* __restrict__ cls,
                const int64_t* __restrict__ labels, float gamma3, float lambda, int row_begin, int row_count,
                float* __restrict__ loss_out, float* __restrict__ draw) {
  extern __shared__ float lg[];                 // [B][B+1] logits
  __shared__ float lse_r[128], lse_c[128], part[256];
  const int P = B + 1, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int i = threadIdx.x; i < B * B; i += blockDim.x) {
    const int a = i / B, b = i - a * B;
    lg[a * P + b] = logit_at(raw, cls, B, a, b, gamma3);
  }
  __syncthreads();
  for (int a = warp; a < B; a += nw) {          // rows
    float m = -INFINITY, s = 0.f;
    for (int b = lane; b < B; b += 32) lse_push(m, s, lg[a * P + b]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
      lse_merge(m, s, m2, s2);
    }
    if (lane == 0) {
      lse_r[a] = m + logf(s);
      part[a] = lse_r[a] - lg[a * P + (int)labels[a]];
    }
  }
  for (int b = warp; b < B; b += nw) {          // columns
    float m = -INFINITY, s = 0.f;
    for (int a = lane; a < B; a += 32) lse_push(m, s, lg[a * P + b]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
      lse_merge(m, s, m2, s2);
    }
    if (lane == 0) {
      lse_c[b] = m + logf(s);
      part[128 + b] = lse_c[b] - lg[(int)labels[b] * P + b];
    }
  }
  __syncthreads();
  if (warp == 0) {
    float acc = 0.f;
    for (int i = lane; i < B; i += 32) acc += part[i] + part[128 + i];
    acc = warp_sum(acc);
    if (lane == 0) loss_out[0] = lambda * acc / (float)B;
  }
  if (draw != nullptr) {
    for (int i = threadIdx.x; i < row_count * B; i += blockDim.x) {
      const int ra = i / B, b = i - ra * B, a = row_begin + ra;
      const float l = lg[a * P + b];
      float d = 0.f;
      if (l != -INFINITY) {
        d = __expf(l - lse_r[a]) + __expf(l - lse_c[b]);
        if ((int)labels[a] == b) d -= 1.f;
        if ((int)labels[b] == a) d -= 1.f;
        d *= lambda * gamma3 / (float)B;
      }
      draw[i] = d;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// sentence cosine matrix                                              sentence_loss.py:33-38
// MODE 0: scos[b,i] = <c_b,r_i> / max(|c_b||r_i|, eps)
// MODE 1: g[b,i] = dscos*gs/den,  gn[b,i] = g*num when the clamp is inactive
// ---------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256)
sent_cos_kernel(const float* __restrict__ cnn, const float* __restrict__ rnn, int Bc, int D, float eps,
                float* __restrict__ out0, float* __restrict__ out1, const float* __restrict__ dscos,
                const float* __restrict__ gscale) {
  extern __shared__ float c_s[];  // [D]
  __shared__ float red[8];
  __shared__ float p_s;
  const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float ss = 0.f;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const float v = cnn[(size_t)b * D + d];
    c_s[d] = v;
    ss = fmaf(v, v, ss);
  }
  ss = warp_sum(ss);
  if (lane == 0) red[warp] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    p_s = sqrtf(t);
  }
  __syncthreads();
  const float p = p_s;
  const float gs = (MODE == 1 && gscale) ? *gscale : 1.f;
  for (int i = warp; i < Bc; i += 8) {
    float num = 0.f, q2 = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float r = rnn[(size_t)i * D + d];
      num = fmaf(c_s[d], r, num);
      q2 = fmaf(r, r, q2);
    }
    num = warp_sum(num);
    q2 = warp_sum(q2);
    if (lane == 0) {
      const float pq = p * sqrtf(q2);
      const float den = fmaxf(pq, eps);
      if (MODE == 0) {
        out0[(size_t)b * Bc + i] = num / den;
      } else {
        const float g = dscos[(size_t)b * Bc + i] * gs / den;
        out0[(size_t)b * Bc + i] = g;
        out1[(size_t)b * Bc + i] = (pq > eps) ? g * num : 0.f;
      }
    }
  }
}

// Gradient of the cosine matrix w.r.t. one side, one block per row v of x (x = cnn for SIDE 0, rnn for
// SIDE 1; y is the other side, n_y rows):
//   g_j = dscos[v,j] * gs / max(|x_v||y_j|, eps),   dx_v = sum_j g_j y_j - (sum_j [clamp inactive] g_j <x_v,y_j>) / |x_v|^2 x_v
// The dots are recomputed here (B^2 D flop, negligible) so no workspace and no second launch is needed.
template <int SIDE>
__global__ void __launch_bounds__(256)
sent_grad_kernel(const float* __restrict__ x, const float* __restrict__ y, int n_x, int n_y, int D, float eps,
                 const float* __restrict__ dscos, const float* __restrict__ gscale, float* __restrict__ dx) {
  extern __shared__ float sm[];                 // x_v [D] | g [n_y]
  float* x_s = sm;
  float* g_s = sm + D;
  __shared__ float red[8];
  __shared__ float p2_s, gn_s;
  const int v = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float ss = 0.f;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const float t = x[(size_t)v * D + d];
    x_s[d] = t;
    ss = fmaf(t, t, ss);
  }
  ss = warp_sum(ss);
  if (lane == 0) red[warp] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    p2_s = t;
  }
  __syncthreads();
  const float p = sqrtf(p2_s);
  const float gs = gscale ? *gscale : 1.f;
  float gn = 0.f;
  for (int j = warp; j < n_y; j += 8) {
    float num = 0.f, q2 = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float r = y[(size_t)j * D + d];
      num = fmaf(x_s[d], r, num);
      q2 = fmaf(r, r, q2);
    }
    num = warp_sum(num);
    q2 = warp_sum(q2);
    if (lane == 0) {
      const float pq = p * sqrtf(q2);
      const float up = SIDE == 0 ? dscos[(size_t)v * n_y + j] : dscos[(size_t)j * n_x + v];
      const float g = up * gs / fmaxf(pq, eps);
      g_s[j] = g;
      if (pq > eps) gn += g * num;
    }
  }
  __syncthreads();
  if (lane == 0) red[warp] = gn;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    gn_s = p2_s > 0.f ? t / p2_s : 0.f;
  }
  __syncthreads();
  const float coef = gn_s;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float acc = 0.f;
    for (int j = 0; j < n_y; ++j) acc = fmaf(g_s[j], y[(size_t)j * D + d], acc);
    dx[(size_t)v * D + d] = acc - coef * x_s[d];
  }
}

// sentence cosine of candidate pairs: one warp per entry v = b*K + k, caption j = cand[v];
// out[v] = <c_b, r_j> / max(|c_b| |r_j|, eps), NaN when j is outside [0, Bc)
__global__ void __launch_bounds__(256)
sent_cos_cand_kernel(const float* __restrict__ cnn, const float* __restrict__ rnn, int Bc,
                     const int32_t* __restrict__ cand, int K, int n, int D, float eps, float* __restrict__ out) {
  const int v = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (v >= n) return;
  const int b = v / K, j = cand[v];
  if (j < 0 || j >= Bc) {
    if (lane == 0) out[v] = __int_as_float(0x7fc00000);
    return;
  }
  float num = 0.f, p2 = 0.f, q2 = 0.f;
  for (int d = lane; d < D; d += 32) {
    const float c = cnn[(size_t)b * D + d], r = rnn[(size_t)j * D + d];
    num = fmaf(c, r, num);
    p2 = fmaf(c, c, p2);
    q2 = fmaf(r, r, q2);
  }
  num = warp_sum(num);
  p2 = warp_sum(p2);
  q2 = warp_sum(q2);
  if (lane == 0) out[v] = num / fmaxf(sqrtf(p2) * sqrtf(q2), eps);
}

// sentence cosine of listed pairs: one warp per pair p, image b = pair_img[p], caption j = pair_cap[p], with the
// summation order of sent_cos_cand_kernel; NaN when b or j is out of range
__global__ void __launch_bounds__(256)
sent_cos_pairs_kernel(const float* __restrict__ cnn, const float* __restrict__ rnn, int Bi, int Bc,
                      const int32_t* __restrict__ pair_img, const int32_t* __restrict__ pair_cap, int n, int D,
                      float eps, float* __restrict__ out) {
  const long long v = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (v >= n) return;
  const int b = pair_img[v], j = pair_cap[v];
  if (b < 0 || b >= Bi || j < 0 || j >= Bc) {
    if (lane == 0) out[v] = __int_as_float(0x7fc00000);
    return;
  }
  float num = 0.f, p2 = 0.f, q2 = 0.f;
  for (int d = lane; d < D; d += 32) {
    const float c = cnn[(size_t)b * D + d], r = rnn[(size_t)j * D + d];
    num = fmaf(c, r, num);
    p2 = fmaf(c, c, p2);
    q2 = fmaf(r, r, q2);
  }
  num = warp_sum(num);
  p2 = warp_sum(p2);
  q2 = warp_sum(q2);
  if (lane == 0) out[v] = num / fmaxf(sqrtf(p2) * sqrtf(q2), eps);
}

}  // namespace agb

using namespace agb;

extern "C" int agb_sent_cos_pairs_fwd(const float* cnn, const float* rnn, int Bi, int Bc, const int32_t* pair_img,
                                      const int32_t* pair_cap, long long P, int D, float eps, float* scos_out,
                                      void* stream) {
  if (Bi <= 0 || Bc <= 0 || D <= 0 || P < 0) return fail_arg("non-positive size");
  if (P >= 0x7fffffffLL) return fail_unsupported("P=%lld >= 2^31", P);
  if (P == 0) return 0;
  if (!cnn || !rnn || !pair_img || !pair_cap || !scos_out) return fail_arg("null pointer");
  sent_cos_pairs_kernel<<<(unsigned)((P + 7) / 8), 256, 0, (cudaStream_t)stream>>>(cnn, rnn, Bi, Bc, pair_img, pair_cap,
                                                                                 (int)P, D, eps, scos_out);
  return check_launch("sent_cos_pairs_kernel");
}

extern "C" int agb_sent_cos_cand_fwd(const float* cnn, const float* rnn, int Bc, const int32_t* cand, int Bi, int K,
                                     int D, float eps, float* scos_out, void* stream) {
  if (Bi <= 0 || Bc <= 0 || K <= 0 || D <= 0) return fail_arg("non-positive size");
  if (!cnn || !rnn || !cand || !scos_out) return fail_arg("null pointer");
  const long long n = (long long)Bi * K;
  if (n >= 0x7fffffffLL - 8) return fail_unsupported("Bi*K=%lld >= 2^31", n);
  sent_cos_cand_kernel<<<(unsigned)((n + 7) / 8), 256, 0, (cudaStream_t)stream>>>(cnn, rnn, Bc, cand, K, (int)n, D, eps,
                                                                               scos_out);
  return check_launch("sent_cos_cand_kernel");
}

extern "C" size_t agb_contrastive_workspace_bytes(int B) { return B > 0 ? (size_t)4 * B * sizeof(float) : 0; }

extern "C" int agb_contrastive_fwd(const float* raw, int B, const int32_t* class_ids, const int64_t* labels,
                                   float gamma3, float lambda, int row_begin, int row_count,
                                   float* loss_out, float* draw, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  if (B <= 0) return fail_arg("B=%d", B);
  if (!raw || !labels || !loss_out || !workspace) return fail_arg("null pointer");
  if (workspace_bytes < agb_contrastive_workspace_bytes(B)) {
    set_error("workspace too small");
    return AGB_E_WORKSPACE;
  }
  if (draw && (row_begin < 0 || row_count < 0 || row_begin + row_count > B)) return fail_arg("bad row range [%d,+%d) of %d", row_begin, row_count, B);
  if (row_count > 65535) return fail_unsupported("row_count=%d > 65535", row_count);
  cudaStream_t st = (cudaStream_t)stream;
  if (B <= 128) {
    const size_t smem = (size_t)B * (B + 1) * sizeof(float);
    if (smem > 48 * 1024) AGB_CUDA(cudaFuncSetAttribute(ce_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ce_small_kernel<<<1, 1024, smem, st>>>(raw, B, class_ids, labels, gamma3, lambda, row_begin, row_count, loss_out,
                                          row_count > 0 ? draw : nullptr);
    return check_launch("ce_small_kernel");
  }
  float* lse_r = (float*)workspace;
  float* lse_c = lse_r + B;
  float* part_r = lse_c + B;
  float* part_c = part_r + B;
  ce_row_kernel<<<B, 256, 0, st>>>(raw, B, class_ids, labels, gamma3, lse_r, part_r);
  if (int rc = check_launch("ce_row_kernel")) return rc;
  ce_col_kernel<<<cdiv(B, 32), 256, 0, st>>>(raw, B, class_ids, labels, gamma3, lse_c, part_c);
  if (int rc = check_launch("ce_col_kernel")) return rc;
  ce_loss_kernel<<<1, 256, 0, st>>>(part_r, part_c, B, lambda, loss_out);
  if (int rc = check_launch("ce_loss_kernel")) return rc;
  if (draw && row_count > 0) {
    ce_grad_kernel<<<dim3(cdiv(B, 128), row_count), 128, 0, st>>>(raw, B, class_ids, labels, gamma3, lambda,
                                                                 lse_r, lse_c, row_begin, row_count, draw);
    if (int rc = check_launch("ce_grad_kernel")) return rc;
  }
  return 0;
}

namespace agb {
int sent_cos_fwd_launch(const float* cnn, const float* rnn, int Bi, int Bc, int D, float eps,
                        float* scos_out, cudaStream_t st) {
  sent_cos_kernel<0><<<Bi, 256, (size_t)D * sizeof(float), st>>>(cnn, rnn, Bc, D, eps, scos_out, nullptr, nullptr, nullptr);
  return check_launch("sent_cos_kernel<0>");
}
}  // namespace agb

extern "C" int agb_sent_cos_fwd(const float* cnn, const float* rnn, int Bi, int Bc, int D, float eps,
                                float* scos_out, void* stream) {
  if (Bi <= 0 || Bc <= 0 || D <= 0) return fail_arg("non-positive size");
  if (D > 8192) return fail_unsupported("D=%d > 8192", D);
  if (!cnn || !rnn || !scos_out) return fail_arg("null pointer");
  return sent_cos_fwd_launch(cnn, rnn, Bi, Bc, D, eps, scos_out, (cudaStream_t)stream);
}

extern "C" size_t agb_sent_cos_bwd_workspace_bytes(int Bi, int Bc) {
  (void)Bi;
  (void)Bc;
  return 0;   // kept for ABI stability: the backward kernels recompute what they need
}

extern "C" int agb_sent_cos_bwd(const float* cnn, const float* rnn, int Bi, int Bc, int D, float eps,
                                const float* dscos, const float* gscale, float* dcnn, float* drnn,
                                void* workspace, size_t workspace_bytes, void* stream) {
  (void)workspace;
  (void)workspace_bytes;
  if (Bi <= 0 || Bc <= 0 || D <= 0) return fail_arg("non-positive size");
  if (D > 8192 || Bi > 8192 || Bc > 8192) return fail_unsupported("D=%d Bi=%d Bc=%d exceed 8192", D, Bi, Bc);
  if (!cnn || !rnn || !dscos) return fail_arg("null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (dcnn) {   // dcnn[b] = sum_i g[b,i] r_i - (...) c_b
    const size_t smem = (size_t)(D + Bc) * sizeof(float);
    if (smem > 48 * 1024) AGB_CUDA(cudaFuncSetAttribute(sent_grad_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sent_grad_kernel<0><<<Bi, 256, smem, st>>>(cnn, rnn, Bi, Bc, D, eps, dscos, gscale, dcnn);
    if (int rc = check_launch("sent_grad_kernel<0>")) return rc;
  }
  if (drnn) {   // drnn[i] = sum_b g[b,i] c_b - (...) r_i   (partial over the local images when sharded)
    const size_t smem = (size_t)(D + Bi) * sizeof(float);
    if (smem > 48 * 1024) AGB_CUDA(cudaFuncSetAttribute(sent_grad_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sent_grad_kernel<1><<<Bc, 256, smem, st>>>(rnn, cnn, Bc, Bi, D, eps, dscos, gscale, drnn);
    if (int rc = check_launch("sent_grad_kernel<1>")) return rc;
  }
  return 0;
}
