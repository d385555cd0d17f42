// Shared device/host helpers for libattngan_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/attngan_b200.h"

namespace agb {

// ---- error plumbing -----------------------------------------------------------------------
void set_error(const char* fmt, ...);
int fail_arg(const char* fmt, ...);          // sets the message, returns AGB_E_BADARG
int fail_unsupported(const char* fmt, ...);  // returns AGB_E_UNSUPPORTED
int check_launch(const char* what);          // cudaGetLastError -> return code; counts the launch

// optional per-kernel timing for bench.py (agb_prof_enable / agb_prof_read); no-ops when disabled
enum ProfTag { PROF_SGEMM = 1, PROF_DAMSM_TC_FWD = 2, PROF_DAMSM_TC_BWD = 3, PROF_ATTN_FWD = 4, PROF_ATTN_BWD = 5,
               PROF_DAMSM_DIMG = 6, PROF_DAMSM_DWORDS = 7, PROF_DAMSM_PACK = 8, PROF_DAMSM_CAND = 9, PROF_MAX = 16 };
int prof_begin(int tag, cudaStream_t st);
void prof_end(int slot, cudaStream_t st);

// ---- process-wide options: read from the environment ONCE (first use), or set through agb_set_option() ----
struct Options {
  long long damsm_chunk_bytes;   // staging budget of one backward chunk of word tiles   (AGB_DAMSM_CHUNK_MB)
  long long damsm_save_bytes;    // budget of what the training forward saves            (AGB_DAMSM_SAVE_MB)
  int damsm_bwd;                 // 2 = always the recomputing backward                  (AGB_DAMSM_BWD)
  int damsm_uniform_split;       // != 0: equal item counts per CTA, not equal cost      (AGB_DAMSM_UNIFORM_SPLIT)
  int damsm_img_block;           // images per L2 block of the pair kernels, 0 = off     (AGB_DAMSM_IMG_BLOCK)
  int damsm_dw_splits;           // image slices of the d words reduction                (AGB_DAMSM_DW_SPLITS)
  int attn_fwd_stages, attn_fwd_ctas, attn_bwd_stages, attn_bwd_ctas;   // tuning knobs  (AGB_ATTN_*), 0 = automatic
};
const Options& options();
int device_sms();                // SM count of the current device (cached per device ordinal)

#define AGB_CUDA(expr)                                                         \
  do {                                                                         \
    cudaError_t _e = (expr);                                                   \
    if (_e != cudaSuccess) {                                                   \
      agb::set_error("%s failed: %s", #expr, cudaGetErrorString(_e));         \
      return (int)_e;                                                          \
    }                                                                          \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// ---- strided batched fp32 GEMM (sgemm.cu) ----------------------------------------------------
//   C[z][m,n] (+)= alpha * sum_{kb<KB} sum_{k<K} A[z][kb][m,k] * B[z][kb][k,n]      z < batch
struct SgemmArgs {
  const float* A;
  const float* B;
  float* C;
  int M, N, K, KB;
  int64_t a_m, a_k, a_kb, a_batch;
  int64_t b_k, b_n, b_kb, b_batch;
  int64_t c_m, c_n, c_batch;
  float alpha;
  int accumulate;
};
int sgemm_strided(const SgemmArgs& g, int batch, cudaStream_t st);

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// ---- device helpers -----------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

// V consecutive elements <-> fp32 registers.  `vec` (kernel-uniform) says the address is
// V*sizeof(T)-aligned and all V elements are in range, so one wide access is legal; otherwise
// `n` (0..V) elements are touched one by one.
template <typename T, int V> struct alignas(sizeof(T) * V) Pack { T v[V]; };

template <typename T, int V>
__device__ __forceinline__ void load_vec(const T* __restrict__ p, bool vec, int n, float (&out)[V]) {
  if (vec) {
    Pack<T, V> pk = *reinterpret_cast<const Pack<T, V>*>(p);
#pragma unroll
    for (int i = 0; i < V; ++i) out[i] = to_f32(pk.v[i]);
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i) out[i] = (i < n) ? to_f32(p[i]) : 0.f;
  }
}
template <typename T, int V>
__device__ __forceinline__ void store_vec(T* __restrict__ p, bool vec, int n, const float (&in)[V]) {
  if (vec) {
    Pack<T, V> pk;
#pragma unroll
    for (int i = 0; i < V; ++i) pk.v[i] = from_f32<T>(in[i]);
    *reinterpret_cast<Pack<T, V>*>(p) = pk;
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i)
      if (i < n) p[i] = from_f32<T>(in[i]);
  }
}

// ---- mbarrier / TMA bulk copy (1-D) ---------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// for single-thread roles (TMA producer, MMA issuer) whose waits are long: back off between polls so the
// spin does not compete with the working warps of the same scheduler for issue slots
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) __nanosleep(40);
}
// global -> shared bulk copy through the TMA unit (SASS: UBLKCP); bytes % 16 == 0, both 16B aligned
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

}  // namespace agb
