// C-ABI entry points of the DAMSM word-region similarity: argument checks and dispatch on the
// arithmetic (AGB_MATH_FP32 -> damsm_fp32.cu, AGB_MATH_TC_* -> damsm_tc.cu).
#include "agb_common.cuh"

namespace agb {
size_t damsm_fp32_workspace_bytes(int Bi, int Bc, int T, int D, int R);
int damsm_fp32_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                   const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1,
                   float gamma2, float eps, int row_offset, float* m_out, float* att_out,
                   void* workspace, size_t workspace_bytes, cudaStream_t st);
int damsm_fp32_bwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                   const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1,
                   float gamma2, float eps, const float* dm, const float* gscale, float* dimg,
                   float* dwords, void* workspace, size_t workspace_bytes, cudaStream_t st);
int sent_cos_fwd_launch(const float* cnn, const float* rnn, int Bi, int Bc, int D, float eps,
                        float* scos_out, cudaStream_t st);
#ifdef AGB_WITH_TC
size_t damsm_tc_workspace_bytes(int Bi, int Bc, int T, int D, int R, int math);
int damsm_tc_supported(int T, int D, int R);
int damsm_tc_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                 const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1,
                 float gamma2, float eps, int row_offset, float* m_out, float* att_out,
                 const float* cnn, const float* rnn, float* scos_out, void* workspace,
                 size_t workspace_bytes, int math, int save, cudaStream_t st);
int damsm_tc_bwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                 const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1,
                 float gamma2, float eps, const float* dm, const float* m_fwd, const float* gscale, float* dimg,
                 float* dwords, void* workspace, size_t workspace_bytes, int ws_from_fwd, int math, cudaStream_t st);
size_t damsm_tc_cand_workspace_bytes(int Bi, int K, int T, int math);
int damsm_tc_cand_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                      const int32_t* cap_lens, int Bc, const int32_t* cand, int Bi, int K, int T, int R, float gamma1,
                      float gamma2, float* m_out, void* workspace, size_t workspace_bytes, int math, cudaStream_t st);
size_t damsm_tc_pairs_workspace_bytes(int Bi, int Bc, long long P, int T, int math);
size_t damsm_tc_pairs_train_workspace_bytes(int Bi, int Bc, long long P, int T, int math);
int damsm_tc_pairs_train_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                             const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap,
                             long long P, int T, int R, float gamma1, float gamma2, float* m_out, void* workspace,
                             size_t workspace_bytes, int math, cudaStream_t st);
int damsm_tc_pairs_bwd(const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t, const int32_t* cap_lens, int Bi,
                       int Bc, long long P, int T, int R, float gamma1, float gamma2, const float* dm, float* dimg,
                       float* dwords, void* workspace, size_t workspace_bytes, int math, cudaStream_t st);
size_t sent_cos_pairs_bwd_workspace_bytes(int Bi, int Bc, long long P);
int sent_cos_pairs_bwd(const float* cnn, const float* rnn, int Bi, int Bc, const int32_t* pair_img,
                       const int32_t* pair_cap, long long P, int D, float eps, const float* dscos, float* dcnn,
                       float* drnn, void* workspace, size_t workspace_bytes, cudaStream_t st);
int damsm_tc_pairs_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                       const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap,
                       long long P, int T, int D, int R, float gamma1, float gamma2, float* m_out, float* att_out,
                       void* workspace, size_t workspace_bytes, int math, cudaStream_t st);
#endif
}  // namespace agb

using namespace agb;

extern "C" int agb_has_tcgen05(void) {
#ifdef AGB_WITH_TC
  return 1;
#else
  return 0;
#endif
}

extern "C" int agb_damsm_supported(int T, int D, int R, int math) {
  if (T <= 0 || D <= 0 || R <= 0) return 0;
  if (math == AGB_MATH_FP32) return (T <= 64 && R <= 1024) ? 1 : 0;
#ifdef AGB_WITH_TC
  if (math == AGB_MATH_TC_F16 || math == AGB_MATH_TC_BF16 || math == AGB_MATH_TC_F16X2) return damsm_tc_supported(T, D, R);
#endif
  return 0;
}

extern "C" size_t agb_damsm_workspace_bytes(int Bi, int Bc, int T, int D, int R, int math) {
  math &= ~AGB_MATH_SAVE;
  if (Bi <= 0 || Bc <= 0 || !agb_damsm_supported(T, D, R, math)) return 0;
  if (math == AGB_MATH_FP32) return damsm_fp32_workspace_bytes(Bi, Bc, T, D, R);
#ifdef AGB_WITH_TC
  return damsm_tc_workspace_bytes(Bi, Bc, T, D, R, math);
#else
  return 0;
#endif
}

extern "C" int agb_damsm_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d,
                             int64_t ws_t, const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R,
                             float gamma1, float gamma2, float eps, int row_offset, float* m_out,
                             float* att_out, const float* cnn, const float* rnn, float* scos_out,
                             void* workspace, size_t workspace_bytes, int math, void* stream) {
  if (!img || !words || !cap_lens || !m_out || !workspace) return fail_arg("null pointer");
  const int save = math & AGB_MATH_SAVE;
  math &= ~AGB_MATH_SAVE;
  if ((cnn != nullptr) != (rnn != nullptr) || (cnn != nullptr) != (scos_out != nullptr))
    return fail_arg("cnn, rnn and scos_out must be given together");
  if (!agb_damsm_supported(T, D, R, math)) return fail_unsupported("T=%d D=%d R=%d math=%d is outside the compiled range", T, D, R, math);
  cudaStream_t st = (cudaStream_t)stream;
  if (math == AGB_MATH_FP32) {
    if (int rc = damsm_fp32_fwd(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, D, R, gamma1, gamma2, eps,
                                row_offset, m_out, att_out, workspace, workspace_bytes, st))
      return rc;
    if (cnn) return sent_cos_fwd_launch(cnn, rnn, Bi, Bc, D, eps, scos_out, st);
    return 0;
  }
#ifdef AGB_WITH_TC
  return damsm_tc_fwd(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, D, R, gamma1, gamma2, eps, row_offset,
                      m_out, att_out, cnn, rnn, scos_out, workspace, workspace_bytes, math, save, st);
#else
  return fail_unsupported("library built without the tcgen05 kernels");
#endif
}

extern "C" int agb_damsm_bwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d,
                             int64_t ws_t, const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R,
                             float gamma1, float gamma2, float eps, const float* dm, const float* m_fwd,
                             const float* gscale, float* dimg, float* dwords, void* workspace,
                             size_t workspace_bytes, int ws_from_fwd, int math, void* stream) {
  if (!img || !words || !cap_lens || !dm || !dimg || !workspace) return fail_arg("null pointer");
  if (!agb_damsm_supported(T, D, R, math)) return fail_unsupported("T=%d D=%d R=%d math=%d is outside the compiled range", T, D, R, math);
  cudaStream_t st = (cudaStream_t)stream;
  if (math == AGB_MATH_FP32)
    return damsm_fp32_bwd(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, D, R, gamma1, gamma2, eps, dm,
                          gscale, dimg, dwords, workspace, workspace_bytes, st);
#ifdef AGB_WITH_TC
  return damsm_tc_bwd(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, D, R, gamma1, gamma2, eps, dm, m_fwd, gscale,
                      dimg, dwords, workspace, workspace_bytes, ws_from_fwd, math, st);
#else
  return fail_unsupported("library built without the tcgen05 kernels");
#endif
}

// candidate pairs run only on the tensor-core kernels (no fp32 path, no training forward)
static bool cand_math_ok(int math) {
  return math == AGB_MATH_TC_F16 || math == AGB_MATH_TC_BF16 || math == AGB_MATH_TC_F16X2;
}

extern "C" size_t agb_damsm_cand_workspace_bytes(int Bi, int K, int T, int D, int R, int math) {
  if (!cand_math_ok(math) || !agb_damsm_supported(T, D, R, math)) return 0;
#ifdef AGB_WITH_TC
  return damsm_tc_cand_workspace_bytes(Bi, K, T, math);
#else
  return 0;
#endif
}

extern "C" int agb_damsm_cand_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                                  const int32_t* cap_lens, int Bc, const int32_t* cand, int Bi, int K, int T, int D,
                                  int R, float gamma1, float gamma2, float* m_out, void* workspace,
                                  size_t workspace_bytes, int math, void* stream) {
  if (!img || !words || !cap_lens || !cand || !m_out || !workspace) return fail_arg("null pointer");
  if (!cand_math_ok(math)) return fail_unsupported("math=%d: candidate scores need a tensor-core inference mode", math);
  if (!agb_damsm_supported(T, D, R, math)) return fail_unsupported("T=%d D=%d R=%d math=%d is outside the compiled range", T, D, R, math);
#ifdef AGB_WITH_TC
  return damsm_tc_cand_fwd(img, words, ws_b, ws_d, ws_t, cap_lens, Bc, cand, Bi, K, T, R, gamma1, gamma2, m_out,
                           workspace, workspace_bytes, math, (cudaStream_t)stream);
#else
  return fail_unsupported("library built without the tcgen05 kernels");
#endif
}

extern "C" size_t agb_damsm_pairs_workspace_bytes(int Bi, int Bc, long long P, int T, int D, int R, int math) {
  if (!cand_math_ok(math) || !agb_damsm_supported(T, D, R, math)) return 0;
#ifdef AGB_WITH_TC
  return damsm_tc_pairs_workspace_bytes(Bi, Bc, P, T, math);
#else
  return 0;
#endif
}

extern "C" int agb_damsm_pairs_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                                   const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img,
                                   const int32_t* pair_cap, long long P, int T, int D, int R, float gamma1,
                                   float gamma2, float* m_out, float* att_out, void* workspace, size_t workspace_bytes,
                                   int math, void* stream) {
  if (!cand_math_ok(math)) return fail_unsupported("math=%d: pair scores need a tensor-core inference mode", math);
  if (!agb_damsm_supported(T, D, R, math)) return fail_unsupported("T=%d D=%d R=%d math=%d is outside the compiled range", T, D, R, math);
  if (P > 0 && (!img || !words || !cap_lens || !pair_img || !pair_cap || !m_out || !workspace))
    return fail_arg("null pointer");
#ifdef AGB_WITH_TC
  return damsm_tc_pairs_fwd(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, pair_img, pair_cap, P, T, D, R, gamma1,
                            gamma2, m_out, att_out, workspace, workspace_bytes, math, (cudaStream_t)stream);
#else
  return fail_unsupported("library built without the tcgen05 kernels");
#endif
}

extern "C" size_t agb_damsm_pairs_train_workspace_bytes(int Bi, int Bc, long long P, int T, int D, int R, int math) {
  if (!cand_math_ok(math) || !agb_damsm_supported(T, D, R, math)) return 0;
#ifdef AGB_WITH_TC
  return damsm_tc_pairs_train_workspace_bytes(Bi, Bc, P, T, math);
#else
  return 0;
#endif
}

extern "C" int agb_damsm_pairs_train_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                                         const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img,
                                         const int32_t* pair_cap, long long P, int T, int D, int R, float gamma1,
                                         float gamma2, float* m_out, void* workspace, size_t workspace_bytes, int math,
                                         void* stream) {
  if (!cand_math_ok(math)) return fail_unsupported("math=%d: pair training needs a tensor-core mode", math);
  if (!agb_damsm_supported(T, D, R, math)) return fail_unsupported("T=%d D=%d R=%d math=%d is outside the compiled range", T, D, R, math);
  if (P > 0 && (!img || !words || !cap_lens || !pair_img || !pair_cap || !m_out || !workspace))
    return fail_arg("null pointer");
#ifdef AGB_WITH_TC
  return damsm_tc_pairs_train_fwd(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, pair_img, pair_cap, P, T, R, gamma1,
                                  gamma2, m_out, workspace, workspace_bytes, math, (cudaStream_t)stream);
#else
  return fail_unsupported("library built without the tcgen05 kernels");
#endif
}

extern "C" int agb_damsm_pairs_bwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                                   const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img,
                                   const int32_t* pair_cap, long long P, int T, int D, int R, float gamma1, float gamma2,
                                   const float* dm, float* dimg, float* dwords, void* workspace,
                                   size_t workspace_bytes, int math, void* stream) {
  if (!cand_math_ok(math)) return fail_unsupported("math=%d: pair training needs a tensor-core mode", math);
  if (!agb_damsm_supported(T, D, R, math)) return fail_unsupported("T=%d D=%d R=%d math=%d is outside the compiled range", T, D, R, math);
  if (P > 0 && (!img || !words || !cap_lens || !pair_img || !pair_cap || !dm || !workspace))
    return fail_arg("null pointer");
#ifdef AGB_WITH_TC
  return damsm_tc_pairs_bwd(words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, P, T, R, gamma1, gamma2, dm, dimg, dwords,
                            workspace, workspace_bytes, math, (cudaStream_t)stream);
#else
  return fail_unsupported("library built without the tcgen05 kernels");
#endif
}

extern "C" size_t agb_sent_cos_pairs_bwd_workspace_bytes(int Bi, int Bc, long long P, int D) {
  if (D <= 0) return 0;
#ifdef AGB_WITH_TC
  return sent_cos_pairs_bwd_workspace_bytes(Bi, Bc, P);
#else
  return 0;
#endif
}

extern "C" int agb_sent_cos_pairs_bwd(const float* cnn, const float* rnn, int Bi, int Bc, const int32_t* pair_img,
                                      const int32_t* pair_cap, long long P, int D, float eps, const float* dscos,
                                      float* dcnn, float* drnn, void* workspace, size_t workspace_bytes, void* stream) {
  if (P > 0 && (!cnn || !rnn || !pair_img || !pair_cap || !dscos || !workspace)) return fail_arg("null pointer");
#ifdef AGB_WITH_TC
  return sent_cos_pairs_bwd(cnn, rnn, Bi, Bc, pair_img, pair_cap, P, D, eps, dscos, dcnn, drnn, workspace,
                            workspace_bytes, (cudaStream_t)stream);
#else
  return fail_unsupported("library built without the tcgen05 kernels");
#endif
}
