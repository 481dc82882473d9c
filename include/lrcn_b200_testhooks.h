/* lrcn_b200_testhooks.h -- kernel-level test hooks and diagnostics of liblrcn_b200_test.so.
 *
 * NOT part of the drop-in boundary: the product library liblrcn_b200.so exports none of these.  The parity tests
 * (tests/test_gpu_parity.py) load liblrcn_b200_test.so -- the same objects plus csrc/test_hooks.cu and csrc/probe_mma.cu --
 * when they need to drive a single kernel (a GEMM variant, the beam top-K / selection kernels) through the C ABI. */
#ifndef LRCN_B200_TESTHOOKS_H
#define LRCN_B200_TESTHOOKS_H

#include "lrcn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- kernel-level test hooks (parity tests call single kernels through the ABI) ---------------
 * C[M][N] (row-major, ldc=N) = op(A) * op(B) (+ C if beta) (+ bias[n]); a_kmajor: A is [M][K] else [K][M];
 * b_kmajor: B is [N][K] else [K][N].  precision selects the fp32 or the tcgen05 bf16x3 kernel. */
LRCN_API int lrcn_test_gemm(lrcn_handle* h, int precision, int a_kmajor, int b_kmajor, int M, int N, int K,
                   const float* A, const float* B, const float* bias, int beta, float* C);
/* diagnostics: average ms of `iters` back-to-back bf16x3 GEMM launches on scratch operands of this shape (no L2 flush);
 * dbg bits (pair kernel only): 1 = no epilogue stores, 2 = no TMA loads after the first ring fill, 4 = no MMAs */
LRCN_API int lrcn_test_gemm_time(lrcn_handle* h, int a_kmajor, int b_kmajor, int M, int N, int K, int with_shadow_out, int iters,
                        int dbg, float* avg_ms_out);
/* diagnostics: clocks to issue / complete a chain of n_mma tcgen05.mma (M x N x 16, bf16, smem operands) on every SM */
LRCN_API int lrcn_test_mma_rate(lrcn_handle* h, int M, int N, int n_mma, int commit_every, int issuers, int64_t* issue_clk_out,
                       int64_t* total_clk_out);
/* beam selection on caller-supplied probabilities: probs [rows][V], parent_prob [rows]; outputs per image */
LRCN_API int lrcn_test_beam_select(lrcn_handle* h, const float* probs, const float* parent_prob, int n_images, int K,
                          int V, int first_step, int64_t* tok_out, int32_t* parent_out, float* score_out);
/* the PRODUCTION top-K kernel of generation from logits [R][V]: tok_out/score_out/lp_out are [R][K] (ids 1-based) */
LRCN_API int lrcn_test_beam_topk_logits(lrcn_handle* h, const float* logits, const float* parent_prob, int R, int V, int K,
                               int64_t* tok_out, float* score_out, float* lp_out);
/* pre-ReLU output of CNN layer `layer` (1..15) for the n images of the last lrcn_extract_features call, as H x W x Cout x n
 * column-major (H = W = 224, 112, 56, 28, 14 for conv1..conv5, 1 for fc6 / fc7).  LRCN_ERR_STATE if that call ran more than
 * one internal chunk of images (only the last chunk is kept) or no call ran; LRCN_ERR_ARG if n differs from its n. */
LRCN_API int lrcn_test_cnn_activation(lrcn_handle* h, int layer, float* out, int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* LRCN_B200_TESTHOOKS_H */
