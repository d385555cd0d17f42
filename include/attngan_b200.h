/*
 * attngan_b200.h -- C ABI of libattngan_b200.so (B200 / sm_100a).
 *
 * The reference (ku222/Attention-GAN) has no FFI layer: its boundary for this hot path IS a set of
 * Python signatures.  Every entry point below names the reference interface it replaces
 * (file:line relative to the reference root).  The Python drop-ins under
 * attention-gan_b200/{networks,losses}/ bind these symbols with ctypes; INTEGRATION.md shows the
 * stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns int: 0 = ok, <0 = invalid argument / unsupported shape (AGB_E_*),
 *     >0 = a cudaError_t.  agb_last_error() returns a thread-local message for the last failure.
 *   - all pointers are DEVICE pointers unless the name ends in _host; nothing is allocated inside:
 *     the caller passes outputs and a workspace sized by the matching *_workspace_bytes() query.
 *   - launches go to the given stream (cudaStream_t passed as void*); no host synchronisation.
 *   - no torch types; layouts are given by explicit element strides where the reference accepts
 *     views.  "io dtype" is the storage type of the big per-pixel tensors only.
 *   - there is no CPU fallback: without a CUDA device the calls fail with a cudaError_t.
 */
#ifndef ATTNGAN_B200_H_
#define ATTNGAN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGB_VERSION 100 /* 0.1.0 */

/* storage type of images / ctx / attn / dctx / dimages in the generator attention */
enum agb_dtype { AGB_F32 = 0, AGB_BF16 = 1, AGB_F16 = 2 };

/* arithmetic used by the DAMSM pair kernels */
enum agb_math {
  AGB_MATH_FP32 = 0,    /* CUDA-core fp32 (bit-for-bit deterministic forward, 1e-6 parity)      */
  AGB_MATH_TC_F16 = 1,  /* tcgen05 kind::f16, fp16 operands, fp32 accumulate in TMEM (default)   */
  AGB_MATH_TC_BF16 = 2, /* tcgen05 kind::f16, bf16 operands                                      */
  /* split precision: every operand of the FORWARD enters the tensor core as hi + lo (two fp16 values) and the
   * partial products accumulate in fp32, so similarities and losses are as accurate as fp32 arithmetic (1e-4
   * on the loss for any batch, incl. the reference-derived fixtures); the backward runs the fp16 kernels. */
  AGB_MATH_TC_F16X2 = 3,
  /* flag, OR-ed into `math` of agb_damsm_fwd by a caller that will run agb_damsm_bwd on the same
   * workspace (ws_from_fwd = 2): the tensor-core forward then also saves the normalised context
   * vectors and their statistics in the workspace and the backward does not recompute them.
   * Ignored by the fp32 path. */
  AGB_MATH_SAVE = 0x100
};

enum agb_status {
  AGB_OK = 0,
  AGB_E_BADARG = -1,      /* null pointer, negative size, misaligned buffer                      */
  AGB_E_UNSUPPORTED = -2, /* shape outside the compiled range (see each call)                    */
  AGB_E_WORKSPACE = -3    /* workspace too small                                                 */
};

int agb_version(void);
const char* agb_last_error(void);
/* 1 when the library was built with the tcgen05 (sm_100a) DAMSM kernels */
int agb_has_tcgen05(void);

/* Process-wide tuning / test options.  Each is read from the environment ONCE (first use of the library) and can
 * be overridden here; none changes results, only how the work is staged:
 *   "damsm_chunk_mb"  (AGB_DAMSM_CHUNK_MB, 16384)  HBM staging budget of one chunk of word tiles in the tensor-core
 *                     DAMSM backward; a small value forces the multi-chunk path (tests do that)
 *   "damsm_save_mb"   (AGB_DAMSM_SAVE_MB, 65536)   budget for the context vectors the training forward saves;
 *                     above it the backward recomputes them (damsm_bwd2_kernel)
 *   "damsm_bwd"       (AGB_DAMSM_BWD, 0)           2 = always the recomputing backward
 *   "damsm_img_block" (AGB_DAMSM_IMG_BLOCK)      images per L2 block of the pair kernels' item order, 0 = off
 *   "damsm_dw_splits" (AGB_DAMSM_DW_SPLITS, 16)  image slices of the d words reduction
 *   "damsm_uniform_split", "attn_fwd_stages", "attn_fwd_ctas", "attn_bwd_stages", "attn_bwd_ctas": kernel tuning
 * Set an option BEFORE querying a workspace size that depends on it and keep it unchanged between a forward and its
 * backward.  Returns 0, or AGB_E_BADARG for an unknown name. */
int agb_set_option(const char* name, long long value);

/* Self-test of the tcgen05 / TMEM / TMA building blocks: one CTA computes
 * C[128,N] = A[128,K] * B[N,K]^T from 16-bit row-major device buffers (fp32 accumulate in TMEM).
 * K % 64 == 0, K <= 256, N in {128, 256}; manual_a != 0 stages A through the thread-written
 * swizzled shared-memory path instead of TMA. */
int agb_tc_selftest(const void* A, const void* B, float* C, int N, int K, int bf16, int manual_a,
                    void* stream);

/* Test hook of the batched tcgen05 GEMM (tc_gemm.cu): C[M,N] (+)= A * B^T for one batch, fp32 out.
 * A is [M,K] row-major (a_mn = 0, K-major) or [K,M] (a_mn = 1, MN-major); B likewise with N.
 * K % 64 == 0; operand row pitches must be multiples of 16 bytes. */
int agb_tc_gemm_test(const void* A, const void* B, float* C, int M, int N, int K, int a_mn, int b_mn,
                     int bf16, int accumulate, void* stream);

/* Measurement hooks (bench.py): number of kernels this library has launched so far, and optional
 * per-kernel timing with CUDA events recorded on the launching stream around the dominant kernels.
 * tag: 1 = fp32 sgemm, 2 = tcgen05 DAMSM forward pair kernel, 3 = tcgen05 DAMSM backward pair kernel,
 *      4 = word-attention forward, 5 = word-attention backward (main kernel),
 *      6 = d img reduction GEMM (tcgen05), 7 = d words reduction GEMM (tcgen05),
 *      9 = candidate pair kernel of agb_damsm_cand_fwd and agb_damsm_pairs_fwd (tcgen05).
 * agb_prof_read synchronises the recorded events and returns the summed duration and the count. */
long long agb_launch_count(void);
void agb_prof_enable(int on);
int agb_prof_read(int tag, double* total_ms, long long* launches);

/* ------------------------------------------------------------------------------------------------
 * Generator word-context attention
 * replaces AttentionModule.forward                       networks/attention.py:25-79
 *          (conv1 1x1 projection :50-52, bmm :59, scale :61, mask :65-66, softmax :68, bmm :73)
 *
 *   images  [B,C,HW]  io dtype, contiguous (NCHW feature map, HW = h*w)
 *   words   [B,E,T]   fp32, element strides (ws_b, ws_e, ws_t): the RNN hands over a transposed
 *                     view of [B,T,E] (rnn_encoder.py:92) and no copy is forced
 *   conv_w  [C,E]     fp32 contiguous (conv1.weight [C,E,1,1])
 *   mask    [B,T]     int64 contiguous, 0 = ignore the word (train.py:96-100)
 *   ctx     [B,C,HW]  io dtype; batch stride ctx_bs elements (so it can be a slice of a
 *                     [B,2C,HW] concat buffer, generator_submodules.py:116)
 *   attn    [B,T,HW]  io dtype, contiguous, or NULL to skip the attention-map output
 *   we      [B,C,T]   fp32 out: projected words W.e (saved for backward)
 *   scaled  != 0 -> scores / sqrt(C) (attention.py:61)
 * Limits: 1 <= T <= 64, 1 <= C <= 64.  A sample whose mask is all zero yields NaN like the
 * reference (softmax over an all -inf row).
 * ---------------------------------------------------------------------------------------------- */
int agb_word_attn_fwd(const void* images, const float* words, int64_t ws_b, int64_t ws_e,
                      int64_t ws_t, const float* conv_w, const int64_t* mask, void* ctx,
                      int64_t ctx_bs, void* attn, float* we, int B, int C, int HW, int E, int T,
                      int io_dtype, int scaled, void* stream);

/* bytes of scratch agb_word_attn_bwd needs (per-tile partial sums of d(W.e)) */
size_t agb_word_attn_bwd_workspace_bytes(int B, int C, int HW, int E, int T);

/* replaces autograd of AttentionModule.forward (SURVEY.md section 8 row a4)
 *   dctx    [B,C,HW] io dtype, batch stride dctx_bs;  dattn [B,T,HW] io dtype or NULL
 *   dimages [B,C,HW] io dtype out
 *   dwords  [B,E,T]  fp32 contiguous out, or NULL;  dconv_w [C,E] fp32 out (overwritten), or NULL
 *   we      [B,C,T]  as written by agb_word_attn_fwd
 * Deterministic: no floating-point atomics. */
int agb_word_attn_bwd(const void* images, const float* words, int64_t ws_b, int64_t ws_e,
                      int64_t ws_t, const float* conv_w, const int64_t* mask, const float* we,
                      const void* dctx, int64_t dctx_bs, const void* dattn, void* dimages,
                      float* dwords, float* dconv_w, void* workspace, size_t workspace_bytes, int B,
                      int C, int HW, int E, int T, int io_dtype, int scaled, void* stream);

/* ------------------------------------------------------------------------------------------------
 * DAMSM word-region similarity (all pairs of Bi images x Bc captions)
 * replaces the loop body of WordsLoss.get_loss           losses/words_loss.py:43-86
 *          and the func_attention it calls               networks/attention.py:82-121
 *
 *   img      [Bi,D,R]  fp32 contiguous (NCHW region features, R = ih*iw)
 *   words    [Bc,D,T]  fp32, element strides (ws_b, ws_d, ws_t)
 *   cap_lens [Bc]      int32, 1 <= L_i <= T
 *   m_out    [Bi,Bc]   fp32: m[b,i] = log sum_{t<L_i} exp(gamma2 * cos(w_it, wc_bit))  (:77-79)
 *   att_out  [Bi,T,R]  fp32 or NULL: beta of the matched pair (image b, caption row_offset+b),
 *                      rows t >= L zeroed (:63)
 *   cnn,rnn  [Bi,D],[Bc,D] fp32 contiguous or both NULL; when given, the raw cosine matrix
 *   scos_out [Bi,Bc]   of SentenceLoss (sentence_loss.py:33-38, before *gamma3) is produced by
 *                      the same call (its kernel runs on a forked stream beside the pair kernel
 *                      and is joined back into `stream` before the call returns)
 *   row_offset         global index of local image 0 when the batch is sharded over ranks
 * Limits: D % 32 == 0, D <= 256 (tcgen05: D == 256... see agb_damsm_supported), T <= 64.
 * ---------------------------------------------------------------------------------------------- */
size_t agb_damsm_workspace_bytes(int Bi, int Bc, int T, int D, int R, int math);

int agb_damsm_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                  const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1,
                  float gamma2, float eps, int row_offset, float* m_out, float* att_out,
                  const float* cnn, const float* rnn, float* scos_out, void* workspace,
                  size_t workspace_bytes, int math, void* stream);

/* replaces autograd of the same loop (SURVEY.md section 8 row a9)
 *   dm      [Bi,Bc]  fp32: dLoss/dm (already includes gamma3 and lambda, see agb_contrastive)
 *   m_fwd   [Bi,Bc]  fp32: m_out of the matching agb_damsm_fwd call, or NULL (then the tensor-core
 *                    path recomputes it; the fp32 path does not need it)
 *   ws_from_fwd      != 0: `workspace` is the untouched buffer the matching agb_damsm_fwd call (same
 *                    inputs, same math) used; the tensor-core path then reuses its packed operands
 *                    (1) and, if that call had AGB_MATH_SAVE set, its saved context vectors (2)
 *   gscale  device scalar (upstream d/dloss) or NULL for 1
 *   dimg    [Bi,D,R] fp32 out (overwritten)
 *   dwords  [Bc,T,D] fp32 contiguous out (note: word-major, the RNN's physical layout), or NULL
 *           when the text encoder is frozen (train.py:89); slots t >= L_i are zero.  In the
 *           sharded case this is the rank's partial sum over its images. */
int agb_damsm_bwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                  const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1,
                  float gamma2, float eps, const float* dm, const float* m_fwd, const float* gscale,
                  float* dimg, float* dwords, void* workspace, size_t workspace_bytes,
                  int ws_from_fwd, int math, void* stream);

/* returns 1 when (T, D, R, math) is inside the compiled range of the requested path */
int agb_damsm_supported(int T, int D, int R, int math);

/* ------------------------------------------------------------------------------------------------
 * DAMSM word-region similarity of candidate pairs (evaluation: R-precision)
 * every image b is scored against its own list of K captions, instead of all Bc of them
 *   m_out[b,k] = m(image b, caption cand[b,k]), defined exactly as agb_damsm_fwd's m_out (words_loss.py:43-79)
 *   img      [Bi,D,R] fp32 contiguous;  words [Bc,D,T] fp32, element strides (ws_b, ws_d, ws_t)
 *   cap_lens [Bc]     int32, 1 <= L <= T
 *   cand     [Bi,K]   int32 contiguous: an index outside [0,Bc) yields NaN for that entry (never a memory fault);
 *                     so does a caption of length 0
 *   m_out    [Bi,K]   fp32
 *   math: AGB_MATH_TC_F16 | AGB_MATH_TC_BF16 | AGB_MATH_TC_F16X2 (inference only: AGB_MATH_SAVE is rejected).
 *   A pair's m is bit for bit the m of the same pair from agb_damsm_fwd with the same math.
 * Limits: the tensor-core range of agb_damsm_supported (D = 256, T <= 32, R <= 320), Bi <= 65535, Bi*K < 2^31,
 * and at most 2^31 / 5508 word tiles in one call (the workspace query returns 0 beyond); otherwise
 * AGB_E_UNSUPPORTED.  The workspace size depends on the shapes only.  No host synchronisation, nothing
 * allocated: capturable in a CUDA graph.
 * ---------------------------------------------------------------------------------------------- */
size_t agb_damsm_cand_workspace_bytes(int Bi, int K, int T, int D, int R, int math);
int agb_damsm_cand_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                       const int32_t* cap_lens, int Bc, const int32_t* cand, int Bi, int K, int T, int D, int R,
                       float gamma1, float gamma2, float* m_out, void* workspace, size_t workspace_bytes,
                       int math, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Sentence cosine matrix on its own (SentenceLoss called without WordsLoss)
 * replaces sentence_loss.py:33-38 and its autograd
 *   scos_out [Bi,Bc] raw cosine <c_b, r_i> / max(|c_b||r_i|, eps)
 *   dscos    [Bi,Bc] dLoss/dcos;  dcnn [Bi,D], drnn [Bc,D] out, either may be NULL
 *            (drnn: partial sum over the local images when sharded)
 * ---------------------------------------------------------------------------------------------- */
int agb_sent_cos_fwd(const float* cnn, const float* rnn, int Bi, int Bc, int D, float eps,
                     float* scos_out, void* stream);
size_t agb_sent_cos_bwd_workspace_bytes(int Bi, int Bc);
int agb_sent_cos_bwd(const float* cnn, const float* rnn, int Bi, int Bc, int D, float eps,
                     const float* dscos, const float* gscale, float* dcnn, float* drnn,
                     void* workspace, size_t workspace_bytes, void* stream);
/* the same cosine for candidate pairs: cnn [Bi,D], rnn [Bc,D] fp32 contiguous, cand [Bi,K] int32 contiguous,
 *   scos_out[b,k] = <cnn_b, rnn_j> / max(|cnn_b| |rnn_j|, eps), j = cand[b,k]; NaN if j is outside [0,Bc) */
int agb_sent_cos_cand_fwd(const float* cnn, const float* rnn, int Bc, const int32_t* cand, int Bi, int K, int D,
                          float eps, float* scos_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Two-way contrastive cross-entropy over a B x B similarity matrix
 * replaces words_loss.py:88-101 and sentence_loss.py:14-25,40-49
 *   raw     [B,B] fp32: m (words) or cosine (sentence); all B rows (gathered over ranks)
 *   class_ids [B] int32 or NULL: entries (a,b), a != b, with equal ids become -inf
 *   labels  [B] int64: row b's target column / column i's target row (trainer.py:20-25: arange)
 *   loss_out[1]: lambda * (mean_b CE(gamma3*raw[b,:], labels[b]) + mean_i CE(gamma3*raw[:,i], labels[i]))
 *   draw    [row_count,B] out: dLoss/draw for rows [row_begin, row_begin+row_count) (incl. gamma3,
 *           lambda); 0 at masked entries
 *   workspace: 4*B floats
 * ---------------------------------------------------------------------------------------------- */
size_t agb_contrastive_workspace_bytes(int B);
int agb_contrastive_fwd(const float* raw, int B, const int32_t* class_ids, const int64_t* labels,
                        float gamma3, float lambda, int row_begin, int row_count, float* loss_out,
                        float* draw, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Region-feature head of the image encoder (SURVEY.md section 8, row f3)
 * replaces CNNEncoder.emb_features = conv1x1(Cin=768 -> Cout=256, no bias) on the Mixed_6e map and its autograd
 *          networks/cnn_encoder.py:56,101; utilities/layers.py:46-48
 *   x     [B,Cin,R]   fp32 contiguous (R = 17*17)         w  [Cout,Cin] fp32 (emb_features.weight [Cout,Cin,1,1])
 *   feat  [B,Cout,R]  fp32 out: what the reference hands to WordsLoss as img_features
 *   dfeat [B,Cout,R]  fp32;  dw [Cout,Cin] fp32 out or NULL;  dx [B,Cin,R] fp32 out or NULL (frozen trunk)
 *   ws_from_fwd != 0: `workspace` is the untouched buffer of the matching agb_region_head_fwd call (same x, w):
 *                     its 16-bit copies of x and w are reused
 * Both run on tcgen05 (bf16 operands cast once into the workspace, fp32 accumulation in TMEM): the forward in split
 * precision (hi + lo bf16 pairs: features within ~1e-5 of fp32 arithmetic), the backward with plain bf16 operands.
 * Limits: Cin % 64 == 0, Cout % 128 == 0.
 * ---------------------------------------------------------------------------------------------- */
size_t agb_region_head_workspace_bytes(int B, int Cin, int Cout, int R);
int agb_region_head_fwd(const float* x, const float* w, float* feat, void* workspace, size_t workspace_bytes,
                        int B, int Cin, int Cout, int R, void* stream);
int agb_region_head_bwd(const float* x, const float* w, const float* dfeat, float* dw, float* dx, void* workspace,
                        size_t workspace_bytes, int ws_from_fwd, int B, int Cin, int Cout, int R, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Functional region-word attention on its own
 * replaces func_attention(query, context, gamma1, scaled)    networks/attention.py:82-121
 *   query [B,D,L] fp32 strided, context [B,D,R] fp32 contiguous
 *   wc_out [B,D,L] fp32 contiguous, attn_out [B,L,R] fp32 contiguous
 *   backward: dwc [B,D,L] contiguous, dattn [B,L,R] contiguous or NULL
 *             -> dquery [B,D,L] contiguous (or NULL), dcontext [B,D,R] (or NULL)
 * Limits: L <= 64, R <= 1024.  fp32 arithmetic.
 * ---------------------------------------------------------------------------------------------- */
size_t agb_func_attention_workspace_bytes(int B, int L, int R);
int agb_func_attention_fwd(const float* query, int64_t qs_b, int64_t qs_d, int64_t qs_t,
                           const float* context, int B, int D, int L, int R, float gamma1,
                           int scaled, float* wc_out, float* attn_out, void* workspace,
                           size_t workspace_bytes, void* stream);
int agb_func_attention_bwd(const float* query, int64_t qs_b, int64_t qs_d, int64_t qs_t,
                           const float* context, int B, int D, int L, int R, float gamma1,
                           int scaled, const float* dwc, const float* dattn, float* dquery,
                           float* dcontext, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * DAMSM word-region similarity of an arbitrary list of (image, caption) pairs (evaluation: text-to-image
 * R-precision, hard-negative inspection, attention maps of chosen pairs)
 *   m_out[p] = m(image pair_img[p], caption pair_cap[p]), bit for bit agb_damsm_fwd's m of that pair in the same math
 *   img, words, cap_lens as in agb_damsm_cand_fwd
 *   pair_img, pair_cap [P] int32: any order, duplicates allowed.  A pair whose image is outside [0,Bi), whose caption
 *                      is outside [0,Bc) or whose caption has length 0 yields NaN (never a memory fault)
 *   m_out    [P]       fp32
 *   att_out  [P,T,R]   fp32 or NULL: beta of every pair (words_loss.py:63), the arithmetic of agb_damsm_fwd's matched
 *                      att_out; rows t >= L are 0, every row of an invalid pair is NaN
 *   The pairs are grouped by image on the device (stable counting sort: inside an image the list order is kept)
 *   and scored by the kernels of agb_damsm_cand_fwd.  P = 0 is a successful no-op.
 *   math: AGB_MATH_TC_F16 | AGB_MATH_TC_BF16 | AGB_MATH_TC_F16X2 (inference only: AGB_MATH_SAVE is rejected).
 * Limits: the tensor-core range of agb_damsm_supported (D = 256, T <= 32, R <= 320), Bi <= 65535, P < 2^31 and at
 * most 2^31 / 5508 work items; otherwise the workspace query returns 0 and the call AGB_E_UNSUPPORTED.  The
 * workspace size depends on (Bi, Bc, P, T, math) only.  No host synchronisation, nothing allocated: capturable in
 * a CUDA graph.
 * ---------------------------------------------------------------------------------------------- */
size_t agb_damsm_pairs_workspace_bytes(int Bi, int Bc, long long P, int T, int D, int R, int math);
int agb_damsm_pairs_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                        const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap,
                        long long P, int T, int D, int R, float gamma1, float gamma2, float* m_out, float* att_out,
                        void* workspace, size_t workspace_bytes, int math, void* stream);

/* sentence cosine of a pair list: scos_out[p] = the cosine (agb_sent_cos_fwd) of image pair_img[p] and caption pair_cap[p], bit for bit
 *   agb_sent_cos_cand_fwd's value for that pair; NaN if either index is out of range.  P = 0 is a no-op, P < 2^31 */
int agb_sent_cos_pairs_fwd(const float* cnn, const float* rnn, int Bi, int Bc, const int32_t* pair_img,
                           const int32_t* pair_cap, long long P, int D, float eps, float* scos_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training on a pair list: gradients of the pair scores m (agb_damsm_pairs_fwd) and of the pair cosines
 * (agb_sent_cos_pairs_fwd), so that a loss over a chosen set of pairs costs only those pairs
 *   agb_damsm_pairs_train_fwd: the arguments of agb_damsm_pairs_fwd without the maps; writes m_out [P] (bit for bit
 *     agb_damsm_pairs_fwd's m) and leaves in the workspace what agb_damsm_pairs_bwd reads: the sorted list, the
 *     packed tiles, the normalised context vectors and the row statistics of every packed word row
 *   agb_damsm_pairs_bwd: the same inputs, the same list and the workspace of the matching train forward, untouched
 *     in between; dm [P] = dLoss/dm in list order
 *     dimg   [Bi,D,R] fp32 contiguous (or NULL), every element written
 *     dwords [Bc,T,D] fp32 contiguous (word-major, as agb_damsm_bwd writes it) or NULL, every element written
 *     A pair with an invalid index or a caption of length 0 contributes nothing, whatever its dm.  An image or
 *     caption in no valid pair and the padded word slots t >= cap_lens get exactly 0.  The reductions have a fixed
 *     order (a stable integer sort of the entries by caption): the gradients are bit-reproducible.  fp16 operands
 *     (bf16 in AGB_MATH_TC_BF16) scaled by the dense backward's power-of-two gradient scale, fp32 accumulation.
 *   agb_sent_cos_pairs_bwd: dscos [P] -> dcnn [Bi,D], drnn [Bc,D] (either may be NULL), fp32 contiguous, with a
 *     workspace of its own; per image and per caption the pairs are summed in list order
 *   The workspace sizes depend on shapes only (no device query).  P = 0 is a no-op; the backward calls then write
 *   zero gradients.  Limits as agb_damsm_pairs_fwd (Bi <= 65535, P < 2^31).  No host synchronisation, nothing
 *   allocated: forward and backward can be captured in a CUDA graph.
 * ---------------------------------------------------------------------------------------------- */
size_t agb_damsm_pairs_train_workspace_bytes(int Bi, int Bc, long long P, int T, int D, int R, int math);
int agb_damsm_pairs_train_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                              const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap,
                              long long P, int T, int D, int R, float gamma1, float gamma2, float* m_out,
                              void* workspace, size_t workspace_bytes, int math, void* stream);
int agb_damsm_pairs_bwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                        const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap,
                        long long P, int T, int D, int R, float gamma1, float gamma2, const float* dm, float* dimg,
                        float* dwords, void* workspace, size_t workspace_bytes, int math, void* stream);
size_t agb_sent_cos_pairs_bwd_workspace_bytes(int Bi, int Bc, long long P, int D);
int agb_sent_cos_pairs_bwd(const float* cnn, const float* rnn, int Bi, int Bc, const int32_t* pair_img,
                           const int32_t* pair_cap, long long P, int D, float eps, const float* dscos, float* dcnn,
                           float* drnn, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ATTNGAN_B200_H_ */
