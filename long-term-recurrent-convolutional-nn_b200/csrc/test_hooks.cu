// test_hooks.cu -- kernel-level test hooks and diagnostics behind the C ABI (include/lrcn_b200_testhooks.h).
// Built ONLY into liblrcn_b200_test.so (the product library liblrcn_b200.so carries none of this).
#include "../../include/lrcn_b200_testhooks.h"
#include "lrcn_internal.h"

// ------------------------------------------------------------------------------------------ test hooks
extern "C" int lrcn_test_gemm(lrcn_handle* h, int precision, int a_kmajor, int b_kmajor, int M, int N, int K, const float* A, const float* B,
                              const float* bias, int beta, float* C) {
  if (!h || !A || !B || !C || M <= 0 || N <= 0 || K <= 0) return fail(LRCN_ERR_ARG, "bad argument");
  CK(cudaSetDevice(h->cfg.device));
  g_counter = &h->counter;
  // padded leading dimensions (multiples of 8) so the same buffers serve both kernels
  const int lda = ((a_kmajor ? K : M) + 7) / 8 * 8, ldb = ((b_kmajor ? K : N) + 7) / 8 * 8;
  const int ra = a_kmajor ? M : K, rb = b_kmajor ? N : K;
  const int ca = a_kmajor ? K : M, cb = b_kmajor ? K : N;
  float *dA = nullptr, *dB = nullptr, *dC = nullptr, *dbias = nullptr;
  bf16 *ah = nullptr, *al = nullptr, *bh = nullptr, *bl = nullptr;
  int rc = LRCN_OK;
  auto cleanup = [&] { for (void* p : {(void*)dA, (void*)dB, (void*)dC, (void*)dbias, (void*)ah, (void*)al, (void*)bh, (void*)bl}) if (p) cudaFree(p); };
#define CKT(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail(LRCN_ERR_CUDA, "%s -> %s", #call, cudaGetErrorString(e_)); cleanup(); return rc; } } while (0)
  const size_t na = ((size_t)ra * lda + 63) / 64 * 64, nb = ((size_t)rb * ldb + 63) / 64 * 64;
  CKT(cudaMalloc(&dA, na * 4)); CKT(cudaMalloc(&dB, nb * 4)); CKT(cudaMalloc(&dC, (size_t)M * N * 4));
  CKT(cudaMemset(dA, 0, na * 4)); CKT(cudaMemset(dB, 0, nb * 4));
  CKT(cudaMemcpy2D(dA, (size_t)lda * 4, A, (size_t)ca * 4, (size_t)ca * 4, ra, cudaMemcpyHostToDevice));
  CKT(cudaMemcpy2D(dB, (size_t)ldb * 4, B, (size_t)cb * 4, (size_t)cb * 4, rb, cudaMemcpyHostToDevice));
  CKT(cudaMemcpy(dC, C, (size_t)M * N * 4, cudaMemcpyHostToDevice));
  if (bias) { CKT(cudaMalloc(&dbias, (size_t)N * 4)); CKT(cudaMemcpy(dbias, bias, (size_t)N * 4, cudaMemcpyHostToDevice)); }
  if (precision == LRCN_PREC_FP32) {
    sgemm(h->stream, a_kmajor, b_kmajor, M, N, K, dA, lda, dB, ldb, dC, N, beta != 0, dbias);
  } else {
    CKT(cudaMalloc(&ah, na * 2)); CKT(cudaMalloc(&al, na * 2)); CKT(cudaMalloc(&bh, nb * 2)); CKT(cudaMalloc(&bl, nb * 2));
    split_bf16(h->stream, dA, na, ah, al);
    split_bf16(h->stream, dB, nb, bh, bl);
    if (!gemm_bf16x3(h->stream, a_kmajor, b_kmajor, M, N, K, ah, al, lda, bh, bl, ldb, dC, N, beta != 0, dbias, nullptr, nullptr)) {
      rc = fail(LRCN_ERR_CUDA, "%s", gemm_bf16x3_last_error());
      cudaStreamSynchronize(h->stream);
      cleanup();
      return rc;
    }
  }
  CKT(cudaStreamSynchronize(h->stream));
  CKT(cudaMemcpy(C, dC, (size_t)M * N * 4, cudaMemcpyDeviceToHost));
  cleanup();
  return LRCN_OK;
}

extern "C" int lrcn_test_gemm_time(lrcn_handle* h, int a_kmajor, int b_kmajor, int M, int N, int K, int with_shadow_out, int iters, int dbg,
                                   float* avg_ms_out) {
  if (!h || !avg_ms_out || M <= 0 || N <= 0 || K <= 0 || iters < 1) return fail(LRCN_ERR_ARG, "bad argument");
  CK(cudaSetDevice(h->cfg.device));
  g_counter = &h->counter;
  const int lda = ((a_kmajor ? K : M) + 7) / 8 * 8, ldb = ((b_kmajor ? K : N) + 7) / 8 * 8, ldc = (N + 7) / 8 * 8;
  const size_t na = (size_t)(a_kmajor ? M : K) * lda, nb = (size_t)(b_kmajor ? N : K) * ldb, nc = (size_t)M * ldc;
  float* dC = nullptr;
  bf16 *ah = nullptr, *al = nullptr, *bh = nullptr, *bl = nullptr, *ch = nullptr, *cl = nullptr;
  int rc = LRCN_OK;
  auto cleanup = [&] { for (void* p : {(void*)dC, (void*)ah, (void*)al, (void*)bh, (void*)bl, (void*)ch, (void*)cl}) if (p) cudaFree(p); g_gemm_dbg = 0; };
  CKT(cudaMalloc(&dC, nc * 4)); CKT(cudaMalloc(&ah, na * 2)); CKT(cudaMalloc(&al, na * 2)); CKT(cudaMalloc(&bh, nb * 2)); CKT(cudaMalloc(&bl, nb * 2));
  if (with_shadow_out) { CKT(cudaMalloc(&ch, nc * 2)); CKT(cudaMalloc(&cl, nc * 2)); }
  CKT(cudaMemset(ah, 0x3c, na * 2)); CKT(cudaMemset(al, 0x38, na * 2)); CKT(cudaMemset(bh, 0x3c, nb * 2)); CKT(cudaMemset(bl, 0x38, nb * 2));
  g_gemm_dbg = dbg;
  for (int i = -2; i < iters; i++) {
    if (i == 0) CKT(cudaEventRecord(h->ev0, h->stream));
    if (!gemm_bf16x3(h->stream, a_kmajor, b_kmajor, M, N, K, ah, al, lda, bh, bl, ldb, dC, ldc, false, nullptr, ch, cl)) {
      rc = fail(LRCN_ERR_CUDA, "%s", gemm_bf16x3_last_error());
      cudaStreamSynchronize(h->stream);
      cleanup();
      return rc;
    }
  }
  CKT(cudaEventRecord(h->ev1, h->stream));
  CKT(cudaEventSynchronize(h->ev1));
  float ms = 0.f;
  CKT(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  *avg_ms_out = ms / iters;
  cleanup();
  return LRCN_OK;
}

extern "C" int lrcn_test_mma_rate(lrcn_handle* h, int M, int N, int n_mma, int commit_every, int issuers, int64_t* issue_clk_out,
                                  int64_t* total_clk_out) {
  if (!h || !issue_clk_out || !total_clk_out || (M != 64 && M != 128) || N < 16 || N > 256 || (N % 16) || n_mma < 1 || (issuers & 15) < 1 || (issuers & 15) > 2 || commit_every < 0)
    return fail(LRCN_ERR_ARG, "bad argument");
  CK(cudaSetDevice(h->cfg.device));
  long long a = 0, b = 0;
  if (!probe_mma(h->stream, M, N, n_mma, commit_every, issuers, &a, &b)) return fail(LRCN_ERR_CUDA, "probe_mma failed: %s", cudaGetErrorString(cudaGetLastError()));
  *issue_clk_out = a; *total_clk_out = b;
  return LRCN_OK;
}

extern "C" int lrcn_test_beam_select(lrcn_handle* h, const float* probs, const float* parent_prob, int n_images, int K, int V, int first_step,
                                     int64_t* tok_out, int32_t* parent_out, float* score_out) {
  if (!h || !probs || !parent_prob || n_images <= 0 || K < 1 || K > 11 || V < K) return fail(LRCN_ERR_ARG, "bad argument");
  CK(cudaSetDevice(h->cfg.device));
  g_counter = &h->counter;
  const int R = n_images * K;
  float *dp = nullptr, *dpp = nullptr, *cs = nullptr, *clp = nullptr, *ss = nullptr, *slp = nullptr;
  int *ct = nullptr, *st = nullptr, *sp = nullptr;
  int rc = LRCN_OK;
  auto cleanup = [&] { for (void* p : {(void*)dp, (void*)dpp, (void*)cs, (void*)clp, (void*)ss, (void*)slp, (void*)ct, (void*)st, (void*)sp}) if (p) cudaFree(p); };
  CKT(cudaMalloc(&dp, (size_t)R * V * 4)); CKT(cudaMalloc(&dpp, (size_t)R * 4)); CKT(cudaMalloc(&cs, (size_t)R * K * 4)); CKT(cudaMalloc(&clp, (size_t)R * K * 4));
  CKT(cudaMalloc(&ss, (size_t)R * 4)); CKT(cudaMalloc(&slp, (size_t)R * 4)); CKT(cudaMalloc(&ct, (size_t)R * K * 4)); CKT(cudaMalloc(&st, (size_t)R * 4));
  CKT(cudaMalloc(&sp, (size_t)R * 4));
  CKT(cudaMemcpy(dp, probs, (size_t)R * V * 4, cudaMemcpyHostToDevice));
  CKT(cudaMemcpy(dpp, parent_prob, (size_t)R * 4, cudaMemcpyHostToDevice));
  beam_row_topk_probs(h->stream, dp, V, R, V, K, dpp, ct, cs, clp);
  beam_select(h->stream, ct, cs, clp, n_images, K, first_step, st, sp, ss, slp);
  CKT(cudaStreamSynchronize(h->stream));
  std::vector<int> t(R), p(R);
  CKT(cudaMemcpy(t.data(), st, (size_t)R * 4, cudaMemcpyDeviceToHost));
  CKT(cudaMemcpy(p.data(), sp, (size_t)R * 4, cudaMemcpyDeviceToHost));
  CKT(cudaMemcpy(score_out, ss, (size_t)R * 4, cudaMemcpyDeviceToHost));
  for (int i = 0; i < R; i++) { tok_out[i] = (int64_t)t[i] + 1; parent_out[i] = p[i]; }
  cleanup();
  return LRCN_OK;
}

// The PRODUCTION top-K kernel of generation, driven from logits exactly as enqueue_beam_step does (lrcn.jl:652-661):
// per row prob = exp(logp(a)), the K largest by (prob desc, index asc), score = prob * parent_prob (fp32), log-prob.
extern "C" int lrcn_test_beam_topk_logits(lrcn_handle* h, const float* logits, const float* parent_prob, int R, int V, int K, int64_t* tok_out,
                                          float* score_out, float* lp_out) {
  if (!h || !logits || !parent_prob || !tok_out || !score_out || !lp_out || R <= 0 || K < 1 || K > 11 || V < K) return fail(LRCN_ERR_ARG, "bad argument");
  if (!h->members.empty()) return fail(LRCN_ERR_ARG, "test hooks take a single-GPU handle");
  CK(cudaSetDevice(h->cfg.device));
  g_counter = &h->counter;
  const int ld = (V + 7) / 8 * 8;
  float *dl = nullptr, *dpp = nullptr, *cs = nullptr, *clp = nullptr;
  int* ct = nullptr;
  int rc = LRCN_OK;
  auto cleanup = [&] { for (void* p : {(void*)dl, (void*)dpp, (void*)cs, (void*)clp, (void*)ct}) if (p) cudaFree(p); };
  CKT(cudaMalloc(&dl, (size_t)R * ld * 4)); CKT(cudaMalloc(&dpp, (size_t)R * 4)); CKT(cudaMalloc(&cs, (size_t)R * K * 4)); CKT(cudaMalloc(&clp, (size_t)R * K * 4));
  CKT(cudaMalloc(&ct, (size_t)R * K * 4));
  CKT(cudaMemset(dl, 0, (size_t)R * ld * 4));
  CKT(cudaMemcpy2D(dl, (size_t)ld * 4, logits, (size_t)V * 4, (size_t)V * 4, R, cudaMemcpyHostToDevice));
  CKT(cudaMemcpy(dpp, parent_prob, (size_t)R * 4, cudaMemcpyHostToDevice));
  beam_row_topk(h->stream, dl, ld, R, V, K, dpp, ct, cs, clp);
  CKT(cudaStreamSynchronize(h->stream));
  std::vector<int> t((size_t)R * K);
  CKT(cudaMemcpy(t.data(), ct, (size_t)R * K * 4, cudaMemcpyDeviceToHost));
  CKT(cudaMemcpy(score_out, cs, (size_t)R * K * 4, cudaMemcpyDeviceToHost));
  CKT(cudaMemcpy(lp_out, clp, (size_t)R * K * 4, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < t.size(); i++) tok_out[i] = (int64_t)t[i] + 1;
  cleanup();
  return LRCN_OK;
}

extern "C" int lrcn_test_cnn_activation(lrcn_handle* h, int layer, float* out, int64_t n) {
  if (!h) return fail(LRCN_ERR_ARG, "null handle");
  if (!h->members.empty()) return fail(LRCN_ERR_ARG, "test hooks take a single-GPU handle");
  return cnn_activation(h, layer, out, n);
}
