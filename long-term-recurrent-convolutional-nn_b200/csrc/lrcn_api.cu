// lrcn_api.cu -- C ABI (include/lrcn_b200.h) and step orchestration of the LRCN decoder hot path.
//
// Data layout in HBM (row-major notation; the reference's column-major K x N matrix IS a row-major [N][K]):
//   parameter arena  w / g / m / v : four flat fp32 arenas with identical offsets, ordered by
//     backward readiness so each gradient bucket is one contiguous NCCL allreduce:
//       bucket 1: Wout [V][H2], bout [V]          (ready after the vocab backward)
//       bucket 2: W2 [4H2][2H2], b2, Wf [C][H1], Wcnn [C][4096]   (after layer-2 BPTT)
//       bucket 3: W1 [4H1][E+H1], b1, WembT [V][E]                 (after layer-1 BPTT)
//     Wemb is the only relayout (V x E column-major -> [V][E]) so a word vector is one coalesced row.
//     In bf16x3 mode w has bf16 hi/lo shadow arenas at the same element offsets (refreshed by Adam).
//   feature tables: [n][4096] fp32 resident per split + host id->row map.
//   workspace arena: time-major activations, row r = t*B + i (see Workspace below) + bf16 shadows.
// Reference call sites replaced: lrcn.jl:378 (lossgradient), :394 (update!), :452-474 (average_loss body),
// :585-678 (generate/beam_search).
#include "lrcn_internal.h"

#include <dlfcn.h>
#include <math.h>

#include <algorithm>
#include <chrono>

static thread_local std::string g_err;
static thread_local int g_last_code = 0;  // code of the last fail() on this thread (read by ApiGuard)
int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  g_last_code = code;
  return code;
}

// process-wide word in mapped host memory raised by a device-side wait that timed out (kernels.cuh)
static unsigned int* g_abort_host = nullptr;
static int check_device_abort() {
  if (g_abort_host && *reinterpret_cast<volatile unsigned int*>(g_abort_host))
    return fail(LRCN_ERR_CUDA, "device-side barrier time-out inside a persistent kernel (see stderr of the process); results are invalid");
  return LRCN_OK;
}
// stream synchronisation used by every ABI call: CUDA errors and device-side time-outs surface here
static int sync_stream(lrcn_handle* h) {
  CK(cudaStreamSynchronize(h->stream));
  return check_device_abort();
}

// ------------------------------------------------------------------------------------------ NCCL via dlopen
typedef struct { char internal[128]; } ncclUniqueId;
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(ncclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi* nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (api.lib) break;
    }
    if (api.lib) {
      api.GetUniqueId = (int (*)(ncclUniqueId*))dlsym(api.lib, "ncclGetUniqueId");
      api.CommInitRank = (int (*)(ncclComm_t*, int, ncclUniqueId, int))dlsym(api.lib, "ncclCommInitRank");
      api.CommDestroy = (int (*)(ncclComm_t))dlsym(api.lib, "ncclCommDestroy");
      api.AllReduce = (int (*)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(api.lib, "ncclAllReduce");
      api.GroupStart = (int (*)())dlsym(api.lib, "ncclGroupStart");
      api.GroupEnd = (int (*)())dlsym(api.lib, "ncclGroupEnd");
      api.GetErrorString = (const char* (*)(int))dlsym(api.lib, "ncclGetErrorString");
    }
  }
  return (api.lib && api.GetUniqueId && api.CommInitRank && api.AllReduce) ? &api : nullptr;
}
enum { NCCL_FLOAT32 = 7, NCCL_FLOAT64 = 8, NCCL_SUM = 0 };

struct GemmFail { std::string msg; };
// precision-dispatching GEMM on arena pointers (both are CUDA paths; no CPU fallback exists)
static void gemm(lrcn_handle* h, bool aK, bool bK, int M, int N, int K, const float* A, int lda, const float* B, int ldb, float* C,
                 int ldc, bool beta, const float* bias, bool split_out = false, bool c_zeroed = false) {
  if (!h->bf16mode) {
    sgemm(h->stream, aK, bK, M, N, K, A, lda, B, ldb, C, ldc, beta, bias);
    return;
  }
  bf16 *ah, *al, *bh, *bl, *ch = nullptr, *cl = nullptr;
  shadow(h, A, &ah, &al);
  shadow(h, B, &bh, &bl);
  if (split_out) shadow(h, C, &ch, &cl);
  if (!gemm_bf16x3(h->stream, aK, bK, M, N, K, ah, al, lda, bh, bl, ldb, C, ldc, beta, bias, ch, cl, c_zeroed))
    throw GemmFail{gemm_bf16x3_last_error()};
}

// weight gradient of one LSTM layer: dW[4H][N1+N2] = dG' * [X | Hprev] (column blocks of one matrix).  One CTA-pair launch
// with two B operands when the block boundary is tile aligned, else two GEMMs.  dW is zero on entry (step-start zeroing).
static void gemm_dw_dual(lrcn_handle* h, int M, int N1, int N2, int K, const float* dG, int ldg, const float* X, int ldx, const float* Hp, int ldh,
                         float* dW, int ldw) {
  if (h->bf16mode && !getenv("LRCN_NO_DUALB")) {
    bf16 *ah, *al, *b1h, *b1l, *b2h, *b2l;
    shadow(h, dG, &ah, &al);
    shadow(h, X, &b1h, &b1l);
    shadow(h, Hp, &b2h, &b2l);
    bool launched = false;
    if (!gemm2_bf16x3_dualB(h->stream, false, false, M, N1, N2, K, ah, al, ldg, b1h, b1l, ldx, b2h, b2l, ldh, dW, ldw, true, &launched))
      throw GemmFail{gemm_bf16x3_last_error()};
    if (launched) return;
  }
  gemm(h, false, false, M, N1, K, dG, ldg, X, ldx, dW, ldw, false, nullptr, false, true);
  gemm(h, false, false, M, N2, K, dG, ldg, Hp, ldh, dW + N1, ldw, false, nullptr, false, true);
}

// ------------------------------------------------------------------------------------------ misc ABI
extern "C" int lrcn_abi_version(void) { return LRCN_ABI_VERSION; }
extern "C" const char* lrcn_last_error(void) { return g_err.c_str(); }
extern "C" int lrcn_config_default(lrcn_config* c) {
  if (!c) return fail(LRCN_ERR_ARG, "null config");
  memset(c, 0, sizeof *c);
  c->embed = 1000; c->hidden1 = 1000; c->hidden2 = 1000;  // lrcn.jl:39-40
  c->vocab = 10636;
  c->max_batch = 256; c->max_len = 28;                    // lrcn.jl:353
  c->max_gen_rows = 1024; c->device = 0;
  c->precision = LRCN_PREC_BF16X3; c->use_graphs = 1;
  c->lr = 1e-3; c->beta1 = 0.9; c->beta2 = 0.999; c->eps = 1e-8;  // Knet Adam() via lrcn.jl:402 (Float64 hyper-parameters)
  c->n_gpus = 1;
  for (int i = 0; i < 8; i++) c->device_ids[i] = i;
  return LRCN_OK;
}

static void param_dims(const lrcn_handle* h, int k, int64_t* r, int64_t* c) {
  const int E = h->E, H1 = h->H1, H2 = h->H2, C = h->C, V = h->V;
  switch (k) {
    case 1: *r = E + H1; *c = 4 * H1; break;
    case 2: *r = 1; *c = 4 * H1; break;
    case 3: *r = 2 * H2; *c = 4 * H2; break;
    case 4: *r = 1; *c = 4 * H2; break;
    case 5: *r = H1; *c = C; break;
    case 6: *r = LRCN_F_CNN; *c = C; break;
    case 7: *r = V; *c = E; break;
    case 8: *r = H2; *c = V; break;
    default: *r = 1; *c = V; break;
  }
}

static int s_destroy(lrcn_handle* h) {
  if (!h) return LRCN_OK;
  if (!h->members.empty()) {  // single-process group: the parent owns only its members
    for (lrcn_handle* m : h->members) if (m) cudaSetDevice(m->cfg.device), cudaStreamSynchronize(m->stream);  // nobody unmaps while a peer may still run
    for (lrcn_handle* m : h->members) s_destroy(m);
    delete h;
    return LRCN_OK;
  }
  cudaSetDevice(h->cfg.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  cnn_free(h);
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second);
  if (h->comm && nccl_api()) nccl_api()->CommDestroy(h->comm);
  if (!h->peers_direct) for (void* q : h->p2p_opened) if (q) cudaIpcCloseMemHandle(q);
  for (cudaEvent_t e : h->sc_ev) if (e) cudaEventDestroy(e);
  void* ptrs[] = {h->w, h->g, h->m, h->v, h->w_hi, h->w_lo, h->wp1_hi, h->wp1_lo, h->wp2_hi, h->wp2_lo, h->wt1_hi, h->wt1_lo, h->wt2_hi, h->wt2_lo, h->tab[0].d, h->tab[1].d, h->ws.f, h->ws.hi, h->ws.lo, h->d_tok_in,
                  h->d_tok_tgt, h->d_rows, h->d_sc, h->p2p_ctl, h->d_loss_total, h->d_epoch, h->d_epoch_side, h->stage, h->d_counters, h->d_trace, h->g_last, h->g_ctok, h->g_stok, h->g_spar, h->g_hista, h->g_histb,
                  h->g_done, h->g_ndone, h->g_olen, h->g_rows, h->g_otok, h->l2_scratch, h->g_keep, h->g_omap, h->g_omap_s};
  for (void* p : ptrs) if (p) cudaFree(p);
  for (void* q : {(void*)h->ep_seq, (void*)h->ep_ids, (void*)h->ep_rows, (void*)h->ep_loss, (void*)h->ep_err, (void*)h->tab[0].d_ids, (void*)h->tab[0].d_rowof,
                  (void*)h->tab[1].d_ids, (void*)h->tab[1].d_rowof})
    if (q) cudaFree(q);
  for (auto& s : h->slots) { if (s.tok_in) cudaFree(s.tok_in); if (s.tok_tgt) cudaFree(s.tok_tgt); if (s.rows) cudaFree(s.rows); }
  if (h->h_stage) cudaFreeHost(h->h_stage);
  if (h->h_sc) cudaFreeHost(h->h_sc);
  if (h->h_loss) cudaFreeHost(h->h_loss);
  if (h->h_ndone) cudaFreeHost(h->h_ndone);
  if (h->h_keep) cudaFreeHost(h->h_keep);
  for (int i = 0; i < lrcn_handle::NSNAP; i++) { if (h->ev_snap[i]) cudaEventDestroy(h->ev_snap[i]); if (h->ev_keep[i]) cudaEventDestroy(h->ev_keep[i]); }
  for (cudaEvent_t e : {h->ev0, h->ev1, h->ev_seg[0], h->ev_seg[1], h->ev_seg[2], h->ev_seg[3], h->ev_comm}) if (e) cudaEventDestroy(e);
  if (h->ev_xfork) cudaEventDestroy(h->ev_xfork);
  for (int i = 0; i < lrcn_handle::NXFER; i++) { if (h->ev_xjoin[i]) cudaEventDestroy(h->ev_xjoin[i]); if (h->xfer[i]) cudaStreamDestroy(h->xfer[i]); }
  if (h->comm_stream) cudaStreamDestroy(h->comm_stream);
  if (h->side_stream) cudaStreamDestroy(h->side_stream);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev_zero) cudaEventDestroy(h->ev_zero);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return LRCN_OK;
}

static int create_impl(const lrcn_config* cfg, lrcn_handle* h) {
  h->cfg = *cfg;
  h->E = cfg->embed; h->H1 = cfg->hidden1; h->H2 = cfg->hidden2; h->V = cfg->vocab;
  h->C = (h->H2 + 1) / 2;
  h->ldV = (h->V + 7) / 8 * 8;
  h->ldv = (h->C + 7) / 8 * 8;
  h->bf16mode = cfg->precision == LRCN_PREC_BF16X3;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(LRCN_ERR_CUDA, "no CUDA device (%s); liblrcn_b200 has no CPU fallback", e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(LRCN_ERR_ARG, "device %d out of range (%d devices)", cfg->device, ndev);
  CK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg->device));
  if (h->bf16mode && prop.major != 10)
    return fail(LRCN_ERR_CUDA, "precision bf16x3 needs sm_100a (tcgen05); device is sm_%d%d", prop.major, prop.minor);
  init_simt_kernels();
  if (h->bf16mode && (!init_gemm_sm100() || !init_lstm_sm100())) return fail(LRCN_ERR_CUDA, "%s", gemm_bf16x3_last_error());
  if (!g_abort_host) {
    CK(cudaHostAlloc(&g_abort_host, sizeof(unsigned int), cudaHostAllocMapped | cudaHostAllocPortable));
    *g_abort_host = 0u;
  }
  if (!gemm_bind_abort(g_abort_host) || !gemm2_bind_abort(g_abort_host) || !lstm_bind_abort(g_abort_host) || !dp_bind_abort(g_abort_host))
    return fail(LRCN_ERR_CUDA, "binding the device-side time-out flag failed: %s", cudaGetErrorString(cudaGetLastError()));
  CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&h->comm_stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_zero, cudaEventDisableTiming));
  CK(cudaEventCreate(&h->ev0));
  CK(cudaEventCreate(&h->ev1));
  for (int i = 0; i < 4; i++) CK(cudaEventCreateWithFlags(&h->ev_seg[i], cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_comm, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_xfork, cudaEventDisableTiming));
  for (int i = 0; i < lrcn_handle::NXFER; i++) {
    CK(cudaStreamCreateWithFlags(&h->xfer[i], cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_xjoin[i], cudaEventDisableTiming));
  }

  // ---- parameter arenas, bucket order (1-based model index): [8,9 | 3,4,5,6 | 1,2,7]
  const int order[9] = {8, 9, 3, 4, 5, 6, 1, 2, 7};
  size_t pos = 0;
  for (int i = 0; i < 9; i++) {
    int k = order[i];
    if (i == 0) h->bucket_off[0] = pos;
    if (i == 2) h->bucket_off[1] = pos;
    if (i == 6) h->bucket_off[2] = pos;
    if (i == 8) h->bucket_off[3] = pos;
    param_dims(h, k, &h->rows[k - 1], &h->cols[k - 1]);
    h->nel[k - 1] = (size_t)(h->rows[k - 1] * h->cols[k - 1]);
    h->off[k - 1] = pos;
    pos += (h->nel[k - 1] + 63) / 64 * 64;
  }
  h->bucket_off[lrcn_handle::NBUCKET] = pos;
  h->P = pos;
  CK(cudaMalloc(&h->w, h->P * 4)); CK(cudaMalloc(&h->g, h->P * 4)); CK(cudaMalloc(&h->m, h->P * 4)); CK(cudaMalloc(&h->v, h->P * 4));
  CK(cudaMemset(h->w, 0, h->P * 4)); CK(cudaMemset(h->g, 0, h->P * 4)); CK(cudaMemset(h->m, 0, h->P * 4)); CK(cudaMemset(h->v, 0, h->P * 4));
  if (h->bf16mode) {
    CK(cudaMalloc(&h->w_hi, h->P * 2)); CK(cudaMalloc(&h->w_lo, h->P * 2));
    CK(cudaMemset(h->w_hi, 0, h->P * 2)); CK(cudaMemset(h->w_lo, 0, h->P * 2));
    CK(cudaMalloc(&h->wp1_hi, lstm_permuted_elems(h->H1) * 2)); CK(cudaMalloc(&h->wp1_lo, lstm_permuted_elems(h->H1) * 2));
    CK(cudaMalloc(&h->wp2_hi, lstm_permuted_elems(h->H2) * 2)); CK(cudaMalloc(&h->wp2_lo, lstm_permuted_elems(h->H2) * 2));
    CK(cudaMalloc(&h->wt1_hi, lstm_transposed_elems(h->H1) * 2)); CK(cudaMalloc(&h->wt1_lo, lstm_transposed_elems(h->H1) * 2));
    CK(cudaMalloc(&h->wt2_hi, lstm_transposed_elems(h->H2) * 2)); CK(cudaMalloc(&h->wt2_lo, lstm_transposed_elems(h->H2) * 2));
    CK(cudaMemset(h->wt1_hi, 0, lstm_transposed_elems(h->H1) * 2)); CK(cudaMemset(h->wt1_lo, 0, lstm_transposed_elems(h->H1) * 2));
    CK(cudaMemset(h->wt2_hi, 0, lstm_transposed_elems(h->H2) * 2)); CK(cudaMemset(h->wt2_lo, 0, lstm_transposed_elems(h->H2) * 2));
  }

  // ---- workspace arena
  const size_t B = cfg->max_batch, T = cfg->max_len + 1, R = B * T, R1 = B * (T + 1);
  const size_t E = h->E, H1 = h->H1, H2 = h->H2, C = h->C, ldV = h->ldV, ldv = h->ldv;
  Arena& a = h->ws;
  Workspace& o = h->o;
  o.X = a.take(B * LRCN_F_CNN); o.v = a.take(B * ldv); o.dv = a.take(B * ldv);
  o.Eall = a.take(R * E); o.dE = a.take(R * E);
  o.acts1 = a.take(R * 4 * H1); o.h1 = a.take(R1 * H1); o.c1 = a.take(R1 * H1);
  o.Z = a.take(R * 2 * C); o.dZ = a.take(R * 2 * C);
  o.acts2 = a.take(R * 4 * H2); o.h2 = a.take(R1 * H2); o.c2 = a.take(R1 * H2);
  o.logits = a.take(R * ldV); o.rowlp = a.take(R);
  o.colpart = a.take((size_t)COLPART_ROWS * ldV);  // per-CTA partial column sums of dA (softmax_ce_fused)
  o.dh2 = a.take(R * H2); o.dh1 = a.take(R * H1);
  o.dhrec1 = a.take(B * H1); o.dc1 = a.take(B * H1); o.dhrec2 = a.take(B * H2); o.dc2 = a.take(B * H2);
  const size_t G = cfg->max_gen_rows > 0 ? cfg->max_gen_rows : 1;
  const size_t ML = 64;  // max history length (nword+2 <= 64)
  o.gX = a.take(G * LRCN_F_CNN); o.gv = a.take(G * ldv); o.ge = a.take(G * E); o.gg1 = a.take(G * 4 * H1);
  o.gh1a = a.take(G * H1); o.gc1a = a.take(G * H1); o.gh1b = a.take(G * H1); o.gc1b = a.take(G * H1);
  o.gz = a.take(G * 2 * C); o.gg2 = a.take(G * 4 * H2);
  o.gh2a = a.take(G * H2); o.gc2a = a.take(G * H2); o.gh2b = a.take(G * H2); o.gc2b = a.take(G * H2);
  o.glogits = a.take(G * ldV); o.gprob = a.take(G); o.gcs = a.take(G * 16); o.gclp = a.take(G * 16); o.gss = a.take(G); o.gslp = a.take(G);
  o.glpa = a.take(G * ML); o.glpb = a.take(G * ML); o.goprob = a.take(G); o.golp = a.take(G * ML);
  o.gxh1 = a.take(G * (E + H1)); o.gxh2 = a.take(G * (2 * C + H2));  // [x|h] operands of the wide (many-row) generation path
  a.cap = a.used;
  CK(cudaMalloc(&a.f, a.cap * 4));
  CK(cudaMemset(a.f, 0, a.cap * 4));
  if (h->bf16mode) {
    CK(cudaMalloc(&a.hi, a.cap * 2)); CK(cudaMalloc(&a.lo, a.cap * 2));
    CK(cudaMemset(a.hi, 0, a.cap * 2)); CK(cudaMemset(a.lo, 0, a.cap * 2));
  }
  CK(cudaMalloc(&h->d_tok_in, R * 4)); CK(cudaMalloc(&h->d_tok_tgt, R * 4)); CK(cudaMalloc(&h->d_rows, B * 4));
  CK(cudaMallocHost(&h->h_stage, (2 * R + B) * 4));
  CK(cudaMalloc(&h->d_sc, sizeof(StepScalars))); CK(cudaMallocHost(&h->h_sc, lrcn_handle::SC_RING * sizeof(StepScalars)));
  memset(h->h_sc, 0, lrcn_handle::SC_RING * sizeof(StepScalars));
  for (int i = 0; i < lrcn_handle::SC_RING; i++) CK(cudaEventCreateWithFlags(&h->sc_ev[i], cudaEventDisableTiming));
  CK(cudaMalloc(&h->p2p_ctl, 4096)); CK(cudaMemset(h->p2p_ctl, 0, 4096));
  h->d_loss = &h->p2p_ctl->loss_partial;
  CK(cudaMalloc(&h->d_loss_total, 8)); CK(cudaMalloc(&h->d_epoch, 4)); CK(cudaMemset(h->d_epoch, 0, 4));
  CK(cudaMalloc(&h->d_epoch_side, 4)); CK(cudaMemset(h->d_epoch_side, 0, 4));
  // + the control words of the fused exchange + the two LL areas of the exposed bucket [W1, b1] (dp_p2p.cu): 2 lines of 16 bytes
  // per float4 and source rank, slices padded by up to 4 floats per rank
  h->ll_floats = 2 * (h->bucket_off[3] - h->bucket_off[2] + 4 * LRCN_P2P_MAX_RANKS + 64);
  CK(cudaMalloc(&h->stage, (h->P + 1024 + DP_XCTL_FLOATS + 2 * h->ll_floats) * 4));
  CK(cudaMemset(h->stage, 0, (h->P + 1024 + DP_XCTL_FLOATS + 2 * h->ll_floats) * 4));  // N staging rows of ~P/N floats each for the copy-engine gradient exchange
  CK(cudaMallocHost(&h->h_loss, 8));
  CK(cudaMalloc(&h->d_counters, 320 * sizeof(unsigned int)));  // [0,256): 4 LSTM launches x 64 (half-)tile barriers; [256,..): softmax
  CK(cudaMemset(h->d_counters, 0, 320 * sizeof(unsigned int)));
  if (getenv("LRCN_SEQ_TRACE") || getenv("LRCN_DP_STAMPS")) { CK(cudaMalloc(&h->d_trace, 64 * 32 * 8)); CK(cudaMemset(h->d_trace, 0, 64 * 32 * 8)); }
  CK(cudaMalloc(&h->g_last, G * 4)); CK(cudaMalloc(&h->g_ctok, G * 16 * 4)); CK(cudaMalloc(&h->g_stok, G * 4)); CK(cudaMalloc(&h->g_spar, G * 4));
  CK(cudaMalloc(&h->g_hista, G * ML * 4)); CK(cudaMalloc(&h->g_histb, G * ML * 4)); CK(cudaMalloc(&h->g_done, G * 4));
  CK(cudaMalloc(&h->g_ndone, 4)); CK(cudaMalloc(&h->g_olen, G * 4)); CK(cudaMalloc(&h->g_rows, G * 4)); CK(cudaMalloc(&h->g_otok, G * ML * 8));
  CK(cudaMallocHost(&h->h_ndone, (size_t)lrcn_handle::NSNAP * (G + 1) * 4));
  CK(cudaMallocHost(&h->h_keep, (size_t)lrcn_handle::NSNAP * G * 4));
  for (int i = 0; i < lrcn_handle::NSNAP; i++) {
    CK(cudaEventCreateWithFlags(&h->ev_snap[i], cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&h->ev_keep[i], cudaEventDisableTiming));
  }
  CK(cudaMalloc(&h->g_keep, G * 4)); CK(cudaMalloc(&h->g_omap, G * 4)); CK(cudaMalloc(&h->g_omap_s, 2 * G * 4));  // g_omap_s: [G] map scratch + [G] done scratch
  h->l2_n = (size_t)64 << 20;  // 256 MiB of floats > 126 MB L2
  CK(cudaMalloc(&h->l2_scratch, h->l2_n * 4));
  CK(cudaDeviceSynchronize());
  return LRCN_OK;
}

static int validate_config(const lrcn_config* cfg) {
  if (cfg->embed <= 0 || cfg->hidden1 <= 0 || cfg->hidden2 <= 0 || cfg->vocab < 4 || cfg->max_batch <= 0 || cfg->max_len <= 0)
    return fail(LRCN_ERR_ARG, "non-positive dimension in config");
  if (cfg->hidden2 % 2) return fail(LRCN_ERR_ARG, "hidden2 must be even (lrcn.jl:496-498,545-546: [x*Wf, x_cnn] must be H2 wide)");
  if (cfg->max_len > 60) return fail(LRCN_ERR_ARG, "max_len > 60 unsupported");
  if (cfg->precision != LRCN_PREC_FP32 && cfg->precision != LRCN_PREC_BF16X3) return fail(LRCN_ERR_ARG, "unknown precision %d", cfg->precision);
  if (cfg->precision == LRCN_PREC_BF16X3 && (cfg->embed % 8 || cfg->hidden1 % 8 || cfg->hidden2 % 8))
    return fail(LRCN_ERR_ARG, "precision bf16x3 needs embed, hidden1, hidden2 to be multiples of 8 (TMA 16-byte pitch); use LRCN_PREC_FP32");
  // softmax-CE and the beam top-K kernel stage one padded logits row in shared memory (200 KiB opt-in limit per CTA)
  if (((size_t)cfg->vocab + 8) * 4 > 200 * 1024)
    return fail(LRCN_ERR_ARG, "vocab %d too large: one logits row (%zu B) must fit the 200 KiB shared-memory row buffer of the softmax / top-K kernels (vocab <= 51192)",
                cfg->vocab, ((size_t)cfg->vocab + 8) * 4);
  if (cfg->n_gpus < 0 || cfg->n_gpus > LRCN_P2P_MAX_RANKS) return fail(LRCN_ERR_ARG, "n_gpus %d outside [0,%d]", cfg->n_gpus, LRCN_P2P_MAX_RANKS);
  return LRCN_OK;
}

// single-process data-parallel group: one member handle per GPU, direct peer pointers (no IPC, no launcher)
static int create_group(const lrcn_config* cfg, lrcn_handle* g) {
  const int N = cfg->n_gpus;
  g->cfg = *cfg;
  g->nranks = N;
  for (int i = 0; i < N; i++)
    for (int j = 0; j < i; j++)
      if (cfg->device_ids[i] == cfg->device_ids[j]) return fail(LRCN_ERR_ARG, "device_ids[%d] == device_ids[%d] == %d", i, j, cfg->device_ids[i]);
  for (int i = 0; i < N; i++) {
    lrcn_config c = *cfg;
    c.n_gpus = 1;
    c.device = cfg->device_ids[i];
    c.max_batch = (cfg->max_batch + N - 1) / N;
    c.max_gen_rows = (cfg->max_gen_rows + N - 1) / N;
    lrcn_handle* m = new lrcn_handle();
    g->members.push_back(m);
    m->parent = g;
    int rc = create_impl(&c, m);
    if (rc) return rc;
    m->rank = i; m->nranks = N;
  }
  for (int i = 0; i < N; i++) {
    CK(cudaSetDevice(cfg->device_ids[i]));
    for (int j = 0; j < N; j++) {
      if (i == j) continue;
      int can = 0;
      CK(cudaDeviceCanAccessPeer(&can, cfg->device_ids[i], cfg->device_ids[j]));
      if (!can) return fail(LRCN_ERR_CUDA, "GPU %d cannot access GPU %d as a peer (NVLink / P2P required for n_gpus > 1)", cfg->device_ids[i], cfg->device_ids[j]);
      cudaError_t e = cudaDeviceEnablePeerAccess(cfg->device_ids[j], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (e != cudaSuccess) return fail(LRCN_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", cfg->device_ids[i], cfg->device_ids[j], cudaGetErrorString(e));
    }
  }
  for (int i = 0; i < N; i++) {
    lrcn_handle* m = g->members[i];
    P2PPeers pe{};
    pe.nranks = N; pe.rank = i;
    for (int p = 0; p < N; p++) {
      lrcn_handle* q = g->members[p];
      pe.g[p] = q->g; pe.w[p] = q->w; pe.ctl[p] = q->p2p_ctl; m->peer_m[p] = q->m; m->peer_v[p] = q->v; m->peer_stage[p] = q->stage;
    }
    m->peers = pe;
    m->peers_direct = true;
    m->p2p_ready = true;
  }
  return LRCN_OK;
}

extern "C" int lrcn_create(const lrcn_config* cfg, lrcn_handle** out) {
  if (!cfg || !out) return fail(LRCN_ERR_ARG, "null argument");
  int rc = validate_config(cfg);
  if (rc) return rc;
  lrcn_handle* h = new lrcn_handle();
  rc = cfg->n_gpus > 1 ? create_group(cfg, h) : create_impl(cfg, h);
  if (rc != LRCN_OK) { std::string keep = g_err; s_destroy(h); g_err = keep; return rc; }
  *out = h;
  return LRCN_OK;
}

// ------------------------------------------------------------------------------------------ weights
static int s_param_shape(const lrcn_handle* h, int idx, int64_t* rows, int64_t* cols) {
  if (!h || idx < 1 || idx > 9 || !rows || !cols) return fail(LRCN_ERR_ARG, "bad param index %d", idx);
  *rows = h->rows[idx - 1]; *cols = h->cols[idx - 1];
  return LRCN_OK;
}
static int check_shape(lrcn_handle* h, int idx, const void* p, int64_t rows, int64_t cols) {
  if (!h || !p || idx < 1 || idx > 9) return fail(LRCN_ERR_ARG, "bad argument (idx=%d)", idx);
  if (rows != h->rows[idx - 1] || cols != h->cols[idx - 1])
    return fail(LRCN_ERR_ARG, "param %d shape mismatch: got %lldx%lld, expected %lldx%lld (lrcn.jl:489-510)", idx, (long long)rows,
                (long long)cols, (long long)h->rows[idx - 1], (long long)h->cols[idx - 1]);
  return LRCN_OK;
}
// host column-major <-> device arena.  Only Wemb (idx 7) is transposed.
static int upload(lrcn_handle* h, float* arena, int idx, const float* src) {
  CK(cudaSetDevice(h->cfg.device));
  size_t n = h->nel[idx - 1];
  float* dst = arena + h->off[idx - 1];
  if (idx == 7) {
    float* tmp = WS(h, h->o.logits);  // scratch: source memory is [E][V] row-major -> want [V][E]
    if (n > h->ws.cap - h->o.logits) {
      std::vector<float> t(n);
      const int64_t V = h->V, E = h->E;
      for (int64_t e = 0; e < E; e++) for (int64_t v = 0; v < V; v++) t[v * E + e] = src[e * V + v];
      CK(cudaMemcpyAsync(dst, t.data(), n * 4, cudaMemcpyHostToDevice, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      return LRCN_OK;
    }
    CK(cudaMemcpyAsync(tmp, src, n * 4, cudaMemcpyHostToDevice, h->stream));
    transpose2d(h->stream, tmp, h->E, h->V, dst);
  } else {
    CK(cudaMemcpyAsync(dst, src, n * 4, cudaMemcpyHostToDevice, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  return LRCN_OK;
}
static int download(lrcn_handle* h, const float* arena, int idx, float* dst) {
  CK(cudaSetDevice(h->cfg.device));
  size_t n = h->nel[idx - 1];
  const float* src = arena + h->off[idx - 1];
  if (idx == 7) {
    std::vector<float> t(n);
    CK(cudaMemcpyAsync(t.data(), src, n * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const int64_t V = h->V, E = h->E;
    for (int64_t v = 0; v < V; v++) for (int64_t e = 0; e < E; e++) dst[e * V + v] = t[v * E + e];
    return LRCN_OK;
  }
  CK(cudaMemcpyAsync(dst, src, n * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return LRCN_OK;
}
static int s_set_param(lrcn_handle* h, int idx, const float* p, int64_t rows, int64_t cols) {
  int rc = check_shape(h, idx, p, rows, cols);
  if (rc) return rc;
  g_counter = &h->counter;
  rc = upload(h, h->w, idx, p);
  if (rc) return rc;
  if (h->bf16mode) {
    size_t o = h->off[idx - 1];
    split_bf16(h->stream, h->w + o, h->nel[idx - 1], h->w_hi + o, h->w_lo + o);
    CK(cudaStreamSynchronize(h->stream));
  }
  return LRCN_OK;
}
static int s_get_param(lrcn_handle* h, int idx, float* p, int64_t rows, int64_t cols) {
  int rc = check_shape(h, idx, p, rows, cols);
  return rc ? rc : download(h, h->w, idx, p);
}
// Peer-memory data parallelism (dp_p2p.cu) leaves m, v -- and after a sharded train step the summed gradient -- current only
// in each owner's shard: collect the other shards from their owners.  All ranks must be idle (e.g. at a checkpoint barrier).
// copy-engine exchange: every gradient bucket k (arena range [bucket_off[k], bucket_off[k+1])) is split into N slices of
// per_k floats (multiples of 4); rank r owns [b, e) of it and its contributions sit at row offset pre_k of a staging row
struct BucketShard { size_t b, e, pre, per; };
static BucketShard bucket_shard(const lrcn_handle* h, int k, int r) {
  BucketShard s{};
  const int N = h->nranks;
  size_t pre = 0;
  for (int kk = 0; kk <= k; kk++) {
    const size_t n4 = (h->bucket_off[kk + 1] - h->bucket_off[kk]) / 4, per4 = (n4 + N - 1) / N;
    if (kk == k) {
      const size_t b4 = per4 * r < n4 ? per4 * r : n4, e4 = b4 + per4 < n4 ? b4 + per4 : n4;
      s.b = h->bucket_off[k] + 4 * b4; s.e = h->bucket_off[k] + 4 * e4; s.pre = pre; s.per = 4 * per4;
    }
    pre += 4 * per4;
  }
  return s;
}
static size_t stage_stride(const lrcn_handle* h) {
  const BucketShard s = bucket_shard(h, lrcn_handle::NBUCKET - 1, 0);
  return s.pre + s.per;
}

static int gather_shards(lrcn_handle* h, bool adam, bool grad) {
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));
  for (int r = 0; r < h->nranks; r++) {
    if (r == h->rank) continue;
    for (int k = 0; k < (h->shard_by_bucket ? lrcn_handle::NBUCKET : 1); k++) {
    size_t b, e;
    if (h->shard_by_bucket) { const BucketShard bs = bucket_shard(h, k, r); b = bs.b; e = bs.e; }
    else dp_p2p_shard(h->P, h->nranks, r, &b, &e);
    if (e <= b) continue;
    // on the handle's stream: device-to-device cudaMemcpy does not synchronise the host, and the download that follows is stream-ordered
    if (adam) {
      CK(cudaMemcpyAsync(h->m + b, h->peer_m[r] + b, (e - b) * 4, cudaMemcpyDefault, h->stream));
      CK(cudaMemcpyAsync(h->v + b, h->peer_v[r] + b, (e - b) * 4, cudaMemcpyDefault, h->stream));
    }
    if (grad) CK(cudaMemcpyAsync(h->g + b, h->peers.g[r] + b, (e - b) * 4, cudaMemcpyDefault, h->stream));
    }
  }
  CK(cudaStreamSynchronize(h->stream));
  if (adam) h->adam_sharded = false;
  if (grad) h->grad_sharded = false;
  return LRCN_OK;
}
static int s_get_grad(lrcn_handle* h, int idx, float* p, int64_t rows, int64_t cols) {
  int rc = check_shape(h, idx, p, rows, cols);
  if (rc) return rc;
  if (h->grad_sharded) { rc = gather_shards(h, false, true); if (rc) return rc; }
  return download(h, h->g, idx, p);
}
static int s_get_adam_state(lrcn_handle* h, int idx, int which, float* p, int64_t rows, int64_t cols) {
  int rc = check_shape(h, idx, p, rows, cols);
  if (rc) return rc;
  if (which != 0 && which != 1) return fail(LRCN_ERR_ARG, "which must be 0 (m) or 1 (v)");
  if (h->adam_sharded) { rc = gather_shards(h, true, false); if (rc) return rc; }
  return download(h, which ? h->v : h->m, idx, p);
}
static int s_set_adam_state(lrcn_handle* h, int idx, int which, const float* p, int64_t rows, int64_t cols) {
  int rc = check_shape(h, idx, p, rows, cols);
  if (rc) return rc;
  if (which != 0 && which != 1) return fail(LRCN_ERR_ARG, "which must be 0 (m) or 1 (v)");
  // a partial overwrite of sharded state would mix current and stale shards: make the local copy whole first
  if (h->adam_sharded) { rc = gather_shards(h, true, false); if (rc) return rc; }
  g_counter = &h->counter;
  return upload(h, which ? h->v : h->m, idx, p);
}
static int s_get_adam_step(lrcn_handle* h, int64_t* t) { if (!h || !t) return fail(LRCN_ERR_ARG, "null"); *t = h->adam_t; return LRCN_OK; }
static int s_set_adam_step(lrcn_handle* h, int64_t t) { if (!h || t < 0) return fail(LRCN_ERR_ARG, "bad step"); h->adam_t = t; return LRCN_OK; }

// ------------------------------------------------------------------------------------------ features
static int s_load_features(lrcn_handle* h, int split, const int64_t* ids, const float* feats, int64_t n) {
  if (!h || !ids || !feats || n <= 0 || split < 0 || split > 1) return fail(LRCN_ERR_ARG, "bad argument to lrcn_load_features");
  CK(cudaSetDevice(h->cfg.device));
  Table& t = h->tab[split];
  if (t.d) { CK(cudaStreamSynchronize(h->stream)); cudaFree(t.d); t.d = nullptr; cudaFree(t.d_ids); cudaFree(t.d_rowof); t.d_ids = nullptr; t.d_rowof = nullptr; }
  t.map.clear();
  CK(cudaMalloc(&t.d, (size_t)n * LRCN_F_CNN * 4));
  CK(cudaMemcpy(t.d, feats, (size_t)n * LRCN_F_CNN * 4, cudaMemcpyHostToDevice));
  t.n = n;
  t.map.reserve((size_t)n * 2);
  for (int64_t i = 0; i < n; i++) t.map[ids[i]] = (int)i;
  {  // device-side lookup for the epoch-level calls: ids sorted ascending + the table row of each (later duplicates win, like the map)
    std::vector<std::pair<long long, int>> pr;
    pr.reserve(t.map.size());
    for (auto& kv : t.map) pr.emplace_back((long long)kv.first, kv.second);
    std::sort(pr.begin(), pr.end());
    std::vector<long long> si(pr.size());
    std::vector<int> ro(pr.size());
    for (size_t i = 0; i < pr.size(); i++) { si[i] = pr[i].first; ro[i] = pr[i].second; }
    CK(cudaMalloc(&t.d_ids, si.size() * 8)); CK(cudaMalloc(&t.d_rowof, ro.size() * 4));
    CK(cudaMemcpy(t.d_ids, si.data(), si.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(t.d_rowof, ro.data(), ro.size() * 4, cudaMemcpyHostToDevice));
  }
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second);  // graphs bake the table pointer
  h->graphs.clear();
  return LRCN_OK;
}

// ------------------------------------------------------------------------------------------ step pieces
static int stage_host(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B, int* tok_in, int* tok_tgt,
                      int* rows) {
  if (!h || !image_ids || (!tokens && l > 0)) return fail(LRCN_ERR_ARG, "null argument");
  if (B <= 0 || B > h->cfg.max_batch) return fail(LRCN_ERR_ARG, "B=%d outside [1,%d]", B, h->cfg.max_batch);
  if (l < 0 || l > h->cfg.max_len) return fail(LRCN_ERR_ARG, "l=%d outside [0,%d]", l, h->cfg.max_len);
  if (split < 0 || split > 1 || !h->tab[split].d) return fail(LRCN_ERR_STATE, "no features loaded for split %d", split);
  const int T = l + 1;
  for (int i = 0; i < B; i++) tok_in[i] = 1;  // bos (0-based 1)                      lrcn.jl:556
  for (int t = 0; t < l; t++)
    for (int i = 0; i < B; i++) {
      int64_t tk = tokens[(size_t)t * B + i];
      if (tk < 1 || tk > h->V) return fail(LRCN_ERR_ARG, "token %lld at (t=%d,i=%d) outside [1,%d]", (long long)tk, t, i, h->V);
      tok_in[(size_t)(t + 1) * B + i] = (int)tk - 1;  // next input                   lrcn.jl:569
      tok_tgt[(size_t)t * B + i] = (int)tk - 1;       // target of step t            lrcn.jl:563-566
    }
  for (int i = 0; i < B; i++) tok_tgt[(size_t)(T - 1) * B + i] = 0;  // eos           lrcn.jl:572-577
  const Table& tb = h->tab[split];
  for (int i = 0; i < B; i++) {
    auto it = tb.map.find(image_ids[i]);
    if (it == tb.map.end()) return fail(LRCN_ERR_MISSING, "missing features for image id %lld (lrcn.jl:602-605)", (long long)image_ids[i]);
    rows[i] = it->second;
  }
  return LRCN_OK;
}

// one LSTM timestep of layer `layer` (1|2) on time-major buffers: acts [T*B][4H] (x-part + bias in, activations out),
// hs/cs [(T+1)*B][H] with slot 0 = zeros.  bf16x3: one fused tcgen05 kernel; fp32: SIMT GEMM + cell kernel.
static void lstm_step_fwd(lrcn_handle* h, int layer, int t, int B, float* acts, float* hs, float* cs) {
  const int H = layer == 1 ? h->H1 : h->H2;
  const int ldw = layer == 1 ? h->E + h->H1 : 2 * h->H2, x_off = layer == 1 ? h->E : 2 * h->C;
  float* g = acts + (size_t)t * B * 4 * H;
  float *hp = hs + (size_t)t * B * H, *hn = hs + (size_t)(t + 1) * B * H, *cp = cs + (size_t)t * B * H, *cn = cs + (size_t)(t + 1) * B * H;
  if (h->bf16mode) {
    bf16 *hp_hi, *hp_lo, *hn_hi, *hn_lo;
    shadow(h, hp, &hp_hi, &hp_lo);
    shadow(h, hn, &hn_hi, &hn_lo);
    if (!lstm_fwd_step(h->stream, B, H, t > 0, hp_hi, hp_lo, layer == 1 ? h->wp1_hi : h->wp2_hi, layer == 1 ? h->wp1_lo : h->wp2_lo, g, cp, cn,
                       hn, hn_hi, hn_lo))
      throw GemmFail{gemm_bf16x3_last_error()};
    return;
  }
  if (t > 0) sgemm(h->stream, true, true, B, 4 * H, H, hp, H, Wp(h, layer == 1 ? 1 : 3) + x_off, ldw, g, 4 * H, true, nullptr);
  lstm_cell_fwd(h->stream, g, cp, cn, hn, B, H);
}
static void lstm_step_bwd(lrcn_handle* h, int layer, int t, int T, int B, float* acts, float* cs, float* dh_all, float* dhrec, float* dc) {
  const int H = layer == 1 ? h->H1 : h->H2;
  const int ldw = layer == 1 ? h->E + h->H1 : 2 * h->H2, x_off = layer == 1 ? h->E : 2 * h->C;
  const float* W = Wp(h, layer == 1 ? 1 : 3);
  float* g = acts + (size_t)t * B * 4 * H;
  const float *cp = cs + (size_t)t * B * H, *cc = cs + (size_t)(t + 1) * B * H, *dh_in = dh_all + (size_t)t * B * H;
  const bool first = t == T - 1;
  if (h->bf16mode) {
    bf16 *g_hi, *g_lo, *gn_hi = nullptr, *gn_lo = nullptr;
    shadow(h, g, &g_hi, &g_lo);
    if (!first) shadow(h, g + (size_t)B * 4 * H, &gn_hi, &gn_lo);
    if (!lstm_bwd_step(h->stream, B, H, !first, layer == 1 ? h->wt1_hi : h->wt2_hi, layer == 1 ? h->wt1_lo : h->wt2_lo, gn_hi, gn_lo, g, g_hi, g_lo,
                       cp, cc, dh_in, dc))
      throw GemmFail{gemm_bf16x3_last_error()};
    return;
  }
  // fp32: dh_rec (from step t+1) was produced by the GEMM issued after the previous cell kernel
  lstm_cell_bwd(h->stream, g, cp, cc, dh_in, dhrec, dc, first, B, H);
  if (t > 0) sgemm(h->stream, true, false, B, H, 4 * H, g, 4 * H, W + x_off, ldw, dhrec, H, false, nullptr);
}

// all T steps of a layer: one persistent kernel when it applies (bf16x3, weights fit in smem, grid co-resident), else per step
static void lstm_layer_fwd(lrcn_handle* h, int layer, int T, int B, float* acts, float* hs, float* cs) {
  if (h->bf16mode && !getenv("LRCN_NO_PERSISTENT")) {
    const int H = layer == 1 ? h->H1 : h->H2;
    bf16 *hs_hi, *hs_lo;
    shadow(h, hs, &hs_hi, &hs_lo);
    bool launched = false;
    if (!lstm_fwd_seq(h->stream, B, H, T, layer == 1 ? h->wp1_hi : h->wp2_hi, layer == 1 ? h->wp1_lo : h->wp2_lo, acts, hs, cs, hs_hi, hs_lo,
                      h->d_counters + (layer == 1 ? 0 : 64), &launched, (layer == 2 && !getenv("LRCN_TRACE_BWD") && !getenv("LRCN_DP_STAMPS")) ? h->d_trace : nullptr))
      throw GemmFail{gemm_bf16x3_last_error()};
    if (launched) return;
  }
  for (int t = 0; t < T; t++) lstm_step_fwd(h, layer, t, B, acts, hs, cs);
}
// returns true when the bias gradient (column sums of dG) has already been accumulated into `dbias` by the LSTM kernel
static bool lstm_layer_bwd(lrcn_handle* h, int layer, int T, int B, float* acts, float* cs, float* dh_all, float* dhrec, float* dc, float* dbias) {
  if (h->bf16mode && !getenv("LRCN_NO_PERSISTENT")) {
    const int H = layer == 1 ? h->H1 : h->H2;
    bf16 *a_hi, *a_lo;
    shadow(h, acts, &a_hi, &a_lo);
    bool launched = false;
    if (!lstm_bwd_seq(h->stream, B, H, T, layer == 1 ? h->wt1_hi : h->wt2_hi, layer == 1 ? h->wt1_lo : h->wt2_lo, acts, a_hi, a_lo, cs, dh_all, dc,
                      h->d_counters + (layer == 2 ? 128 : 192), &launched, dbias, (layer == 2 && getenv("LRCN_TRACE_BWD") && !getenv("LRCN_DP_STAMPS")) ? h->d_trace : nullptr))
      throw GemmFail{gemm_bf16x3_last_error()};
    if (launched) return true;
  }
  for (int t = T - 1; t >= 0; t--) lstm_step_bwd(h, layer, t, T, B, acts, cs, dh_all, dhrec, dc);
  return false;
}

static void enqueue_forward(lrcn_handle* h, int split, int B, int l, bool train) {
  const int T = l + 1, R = T * B, E = h->E, H1 = h->H1, H2 = h->H2, C = h->C, V = h->V, ldV = h->ldV, ldv = h->ldv;
  const Workspace& o = h->o;
  cudaStream_t s = h->stream;
  float *X = WS(h, o.X), *v = WS(h, o.v), *Eall = WS(h, o.Eall), *acts1 = WS(h, o.acts1), *h1 = WS(h, o.h1), *c1 = WS(h, o.c1);
  float *Z = WS(h, o.Z), *acts2 = WS(h, o.acts2), *h2 = WS(h, o.h2), *c2 = WS(h, o.c2), *logits = WS(h, o.logits);
  // Step start.  (1) The recurrent-weight operands of the persistent LSTM kernels are rebuilt from the fp32 weights on a SIDE
  // stream (a fork/join that stream capture turns into a parallel graph branch): they depend on nothing but the weights, so
  // they overlap the zero-fill, the feature gather and the first GEMM.  The join sits before gather_embed, a kernel without
  // the PDL attribute, more than two launches upstream of the first LSTM kernel (which loads its weights before its
  // dependency wait).  (2) ONE launch zeroes every accumulation target of the step: grid-barrier counters and, for training,
  // the gradient arena behind dWout (bias column sums, split-K / stream-K weight gradients, the embedding scatter) and the
  // stream-K data-gradient buffers.
  if (h->bf16mode) {
    cudaEventRecord(h->ev_fork, s);
    cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0);
    lstm_prepare_weights2(h->side_stream, Wp(h, 1), E + H1, E, H1, h->wp1_hi, h->wp1_lo, train ? h->wt1_hi : nullptr, h->wt1_lo, Wp(h, 3), 2 * H2,
                          2 * C, H2, h->wp2_hi, h->wp2_lo, train ? h->wt2_hi : nullptr, h->wt2_lo);
    cudaEventRecord(h->ev_join, h->side_stream);
  }
  {
    // Two zeroing launches.  What the FORWARD pass needs (grid-barrier counters, slot 0 of the state buffers) is zeroed on the
    // main stream; the accumulation targets of the BACKWARD pass (~60 MB: the gradient arena behind dWout, the stream-K
    // data-gradient buffers) are zeroed on the side stream under the forward pass and joined before the softmax kernel, the
    // first kernel that accumulates into the gradient arena (dbout).
    ZeroSegs z, zb;
    z.add(h->d_counters, 256);
    // slot 0 of the h / c slot buffers is h_0 = c_0 = 0 (initstate, lrcn.jl:512-526).  Its POSITION is fixed (rows [0, B)), but
    // slot t of a call with a smaller B lands on rows [t*B_small, ...) -- inside slot 0 of a later, larger batch (average_loss
    // runs B = 10 on the handle that trains at 256).  So the first B rows (fp32 and bf16 shadows) are cleared every step.
    z.add(h1, (size_t)B * H1); z.add(c1, (size_t)B * H1); z.add(h2, (size_t)B * H2); z.add(c2, (size_t)B * H2);
    if (h->bf16mode) {  // two bf16 per float; B*H is even (H % 8 == 0 in this mode)
      z.add(SH(h, h1).hi, (size_t)B * H1 / 2); z.add(SH(h, h1).lo, (size_t)B * H1 / 2);
      z.add(SH(h, h2).hi, (size_t)B * H2 / 2); z.add(SH(h, h2).lo, (size_t)B * H2 / 2);
    }
    if (train) {
      ZeroSegs& t = h->bf16mode ? zb : z;
      t.add(h->g + h->off[8], h->P - h->off[8]);  // arena order [Wout, bout | W2, b2, Wf, Wcnn | W1, b1, Wemb]: everything from bout on
      t.add(WS(h, o.dh2), (size_t)R * H2);
      t.add(WS(h, o.dZ), (size_t)R * 2 * C);
      t.add(WS(h, o.dE), (size_t)R * E);
    }
    zero_multi(s, z);
    if (zb.count) {
      zero_multi(h->side_stream, zb);
      cudaEventRecord(h->ev_zero, h->side_stream);
    }
  }
  gather_features(s, h->tab[split].d, h->d_rows, B, X, SH(h, X).hi, SH(h, X).lo);
  gemm(h, true, true, B, C, LRCN_F_CNN, X, LRCN_F_CNN, Wp(h, 6), LRCN_F_CNN, v, ldv, false, nullptr);  // input*Wcnn  lrcn.jl:558
  if (h->bf16mode) cudaStreamWaitEvent(s, h->ev_join, 0);
  gather_embed(s, Wp(h, 7), h->d_tok_in, R, E, Eall, h->d_sc, train, SH(h, Eall).hi, SH(h, Eall).lo);
  gemm(h, true, true, R, 4 * H1, E, Eall, E, Wp(h, 1), E + H1, acts1, 4 * H1, false, Wp(h, 2));         // x-part of layer 1, all t
  lstm_layer_fwd(h, 1, T, B, acts1, h1, c1);
  gemm(h, true, true, R, C, H1, h1 + (size_t)B * H1, H1, Wp(h, 5), H1, Z, 2 * C, false, nullptr);         // x*w[end-4]  lrcn.jl:545
  z_finish(s, Z, v, ldv, R, B, C, h->d_sc, train, SH(h, Z).hi, SH(h, Z).lo);  // hcat(x,x_cnn) + dropout          lrcn.jl:546-547
  gemm(h, true, true, R, 4 * H2, 2 * C, Z, 2 * C, Wp(h, 3), 2 * H2, acts2, 4 * H2, false, Wp(h, 4));
  lstm_layer_fwd(h, 2, T, B, acts2, h2, c2);
  gemm(h, true, true, R, V, H2, h2 + (size_t)B * H2, H2, Wp(h, 8), H2, logits, ldV, false, Wp(h, 9));      // x*w[end-1] .+ w[end]  lrcn.jl:550
  // logp + gather + fp64 total  lrcn.jl:562-567; training in bf16x3 mode also folds dbout in and never writes dA in fp32
  h->dbout_fused = false;
  if (train && h->bf16mode) cudaStreamWaitEvent(s, h->ev_zero, 0);  // the backward pass's accumulation targets are zero from here on
  if (train && h->bf16mode && !getenv("LRCN_NO_FUSED_SOFTMAX"))
    h->dbout_fused = softmax_ce_fused(s, logits, ldV, R, V, h->d_tok_tgt, WS(h, o.rowlp), h->d_sc, SH(h, logits).hi, SH(h, logits).lo,
                                      WS(h, o.colpart), COLPART_ROWS, Gp(h, 9), h->d_loss, h->d_counters + 256);
  if (!h->dbout_fused)
    softmax_ce(s, logits, ldV, R, V, h->d_tok_tgt, WS(h, o.rowlp), h->d_sc, train, SH(h, logits).hi, SH(h, logits).lo, h->d_loss,
               h->d_counters + 256);
}

static void enqueue_backward_seg(lrcn_handle* h, int B, int l, bool train, int seg) {
  const int T = l + 1, R = T * B, E = h->E, H1 = h->H1, H2 = h->H2, C = h->C, V = h->V, ldV = h->ldV, ldv = h->ldv;
  const Workspace& o = h->o;
  cudaStream_t s = h->stream;
  float *X = WS(h, o.X), *Eall = WS(h, o.Eall), *acts1 = WS(h, o.acts1), *h1 = WS(h, o.h1), *c1 = WS(h, o.c1);
  float *Z = WS(h, o.Z), *dZ = WS(h, o.dZ), *acts2 = WS(h, o.acts2), *h2 = WS(h, o.h2), *c2 = WS(h, o.c2), *dA = WS(h, o.logits);
  float *dh2 = WS(h, o.dh2), *dh1 = WS(h, o.dh1), *dv = WS(h, o.dv), *dE = WS(h, o.dE);
  if (seg == 1) {
    gemm(h, false, false, V, H2, R, dA, ldV, h2 + (size_t)B * H2, H2, Gp(h, 8), H2, false, nullptr);      // dWout = h2' * dA
    if (!h->dbout_fused) colsum(s, dA, ldV, R, V, Gp(h, 9), true);                                                              // dbout
    gemm(h, true, false, R, H2, V, dA, ldV, Wp(h, 8), H2, dh2, H2, false, nullptr, false, true);                        // dh2 = dA * Wout'
  } else if (seg == 2) {
    float *dhrec = WS(h, o.dhrec2), *dc = WS(h, o.dc2);
    const bool db_done = lstm_layer_bwd(h, 2, T, B, acts2, c2, dh2, dhrec, dc, Gp(h, 4));
    gemm_dw_dual(h, 4 * H2, 2 * C, H2, R, acts2, 4 * H2, Z, 2 * C, h2, H2, Gp(h, 3), 2 * H2);  // dW2 = dG2' * [Z | h2_{t-1}] (slot 0 = 0)
    if (!db_done) colsum(s, acts2, 4 * H2, R, 4 * H2, Gp(h, 4), true);
    gemm(h, true, false, R, 2 * C, 4 * H2, acts2, 4 * H2, Wp(h, 3), 2 * H2, dZ, 2 * C, false, nullptr, false, true);
    dz_finish(s, dZ, dv, ldv, T, B, C, h->d_sc, train, SH(h, dZ).hi, SH(h, dZ).lo, SH(h, dv).hi, SH(h, dv).lo);
    gemm(h, false, false, C, H1, R, dZ, 2 * C, h1 + (size_t)B * H1, H1, Gp(h, 5), H1, false, nullptr, false, true);            // dWf
    gemm(h, true, false, R, H1, C, dZ, 2 * C, Wp(h, 5), H1, dh1, H1, false, nullptr);                             // dh1 = dq * Wf'
    gemm(h, false, false, C, LRCN_F_CNN, B, dv, ldv, X, LRCN_F_CNN, Gp(h, 6), LRCN_F_CNN, false, nullptr, false, true);        // dWcnn = X' * dv
  } else {
    // seg 3 = the whole layer-1 segment; the data-parallel step runs it as 31 (BPTT, then the embedding gradient: the largest
    // bucket of the segment is complete first and travels under 32) and 32 (the weight gradient of layer 1)
    float *dhrec = WS(h, o.dhrec1), *dc = WS(h, o.dc1);
    if (seg == 3 || seg == 31) {
      const bool db_done = lstm_layer_bwd(h, 1, T, B, acts1, c1, dh1, dhrec, dc, Gp(h, 2));
      if (!db_done) colsum(s, acts1, 4 * H1, R, 4 * H1, Gp(h, 2), true);
      gemm(h, true, false, R, E, 4 * H1, acts1, 4 * H1, Wp(h, 1), E + H1, dE, E, false, nullptr, false, true);
      scatter_add_embed(s, Gp(h, 7), h->d_tok_in, dE, R, E, h->d_sc, train);                                       // adjoint of Wemb[idx,:]
    }
    if (seg == 3 || seg == 32)
      gemm_dw_dual(h, 4 * H1, E, H1, R, acts1, 4 * H1, Eall, E, h1, H1, Gp(h, 1), E + H1);     // dW1 = dG1' * [E | h1_{t-1}]
  }
}

static void enqueue_adam(lrcn_handle* h) {
  adam_flat(h->stream, h->w, h->g, h->m, h->v, h->P, h->d_sc, h->w_hi, h->w_lo);
}

// run `fn` directly or as a cached CUDA graph keyed by (kind, B, l, flags)
template <class F>
static int run_cached(lrcn_handle* h, std::tuple<int, int, int, int> key, F fn) {
  g_counter = &h->counter;
  try {
    if (!h->cfg.use_graphs) { fn(); CK(cudaPeekAtLastError()); return LRCN_OK; }
    auto it = h->graphs.find(key);
    if (it == h->graphs.end()) {
      cudaGraph_t graph = nullptr;
      long long before = h->counter.n;
      CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
      fn();
      cudaError_t e = cudaStreamEndCapture(h->stream, &graph);
      if (e != cudaSuccess) return fail(LRCN_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
      long long launches = h->counter.n - before;
      h->counter.n = before;
      cudaGraphExec_t exec = nullptr;
      e = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) return fail(LRCN_ERR_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
      it = h->graphs.emplace(key, exec).first;
      h->graph_launches[key] = launches;
    }
    CK(cudaGraphLaunch(it->second, h->stream));
    h->counter.n += h->graph_launches[key];
  } catch (GemmFail& f) {
    cudaGraph_t junk = nullptr;
    cudaStreamCaptureStatus st;
    if (cudaStreamIsCapturing(h->stream, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone) { cudaStreamEndCapture(h->stream, &junk); if (junk) cudaGraphDestroy(junk); }
    return fail(LRCN_ERR_CUDA, "%s", f.msg.c_str());
  }
  return LRCN_OK;
}

// rows of the GLOBAL batch this step belongs to: the group dispatcher sets global_B; one process per GPU: equal shards
static double global_rows(const lrcn_handle* h, int B) { return h->global_B > 0 ? (double)h->global_B : (double)B * h->nranks; }

// fills the next pinned copy of the step scalars and enqueues its H2D copy; waits only if that ring entry's previous copy
// (SC_RING steps ago) has not executed yet
static int push_scalars(lrcn_handle* h, int B, int l, float pdrop, uint64_t seed, bool bump_adam) {
  const int slot = h->sc_next;
  h->sc_next = (slot + 1) % lrcn_handle::SC_RING;
  if (h->sc_busy[slot]) CK(cudaEventSynchronize(h->sc_ev[slot]));
  StepScalars* sc = h->h_sc + slot;
  const double ntok = global_rows(h, B) * (l + 1);
  sc->inv_ntok = (float)(1.0 / ntok);
  sc->pdrop = pdrop;
  sc->keep_scale = pdrop > 0.f ? 1.0f / (1.0f - pdrop) : 1.0f;
  sc->drop_thresh = pdrop > 0.f ? (uint32_t)((double)pdrop * 16777216.0) : 0u;
  sc->seed = seed + 0x9E3779B97F4A7C15ull * (uint64_t)h->rank;  // shards of one global batch draw different masks
  if (bump_adam) { h->adam_t += 1; h->dp_epoch += 1; }
  sc->xchg_epoch = h->dp_epoch; sc->pad_ = 0;
  const int64_t t = h->adam_t > 0 ? h->adam_t : 1;
  sc->adam_d1 = (float)(1.0 - pow(h->cfg.beta1, (double)t));
  sc->adam_d2 = (float)(1.0 - pow(h->cfg.beta2, (double)t));
  sc->lr = (float)h->cfg.lr; sc->beta1 = (float)h->cfg.beta1; sc->beta2 = (float)h->cfg.beta2; sc->eps = (float)h->cfg.eps;
  sc->one_m_beta1 = (float)(1.0 - h->cfg.beta1);
  sc->one_m_beta2 = (float)(1.0 - h->cfg.beta2);
  CK(cudaMemcpyAsync(h->d_sc, sc, sizeof(StepScalars), cudaMemcpyHostToDevice, h->stream));
  CK(cudaEventRecord(h->sc_ev[slot], h->stream));
  h->sc_busy[slot] = true;
  return LRCN_OK;
}

static int nccl_check(int r, const char* what) {
  if (r == 0) return LRCN_OK;
  NcclApi* n = nccl_api();
  return fail(LRCN_ERR_NCCL, "%s failed: %s", what, n && n->GetErrorString ? n->GetErrorString(r) : "nccl error");
}

// forward (+ backward (+ adam)) on the tokens currently in d_tok_in/d_tok_tgt/d_rows
static int run_step(lrcn_handle* h, int split, int B, int l, float pdrop, uint64_t seed, int mode /*0 loss,1 grad,2 train*/) {
  CK(cudaSetDevice(h->cfg.device));
  const bool train = mode >= 1;
  const bool drop = train && pdrop > 0.f;
  { int rc0 = push_scalars(h, B, l, train ? pdrop : 0.f, seed, mode == 2); if (rc0) return rc0; }
  h->last_B = B; h->last_l = l;
  const int fl = (split << 1) | (drop ? 1 : 0);
  int rc;
  h->loss_is_total = false;
  if (mode == 0) {
    return run_cached(h, std::make_tuple(0, B, l, fl), [&] { enqueue_forward(h, split, B, l, false); });
  }
  static const bool adam_overlap = getenv("LRCN_ADAM_NO_OVERLAP") == nullptr;
  if (h->nranks == 1 && mode == 2 && adam_overlap && h->bf16mode) {
    // One GPU: the Adam update (HBM-bound, 7.8 % of the step when it ran after the backward pass) is cut into the gradient
    // buckets of the data-parallel exchange and runs on a side stream -- a parallel branch of the step's graph -- UNDER the rest
    // of the backward pass, as soon as a bucket's gradient is complete and its weights have had their last use: [Wout, bout]
    // under the layer-2 BPTT kernel, [W2, b2, Wf, Wcnn] under the layer-1 BPTT kernel (on the 20 SMs the persistent LSTM
    // kernels leave free; those kernels are latency-bound and leave the HBM idle), Wemb under the dW1 GEMM.  Only [W1, b1]
    // (8.4 MB of 53) is updated after the last gradient kernel.  Same kernel, same per-element arithmetic as the flat update.
    static const int c_lstm = getenv("LRCN_ADAM_CTAS_LSTM") ? atoi(getenv("LRCN_ADAM_CTAS_LSTM")) : 20 * 8;
    static const int c_wemb = getenv("LRCN_ADAM_CTAS_WEMB") ? atoi(getenv("LRCN_ADAM_CTAS_WEMB")) : 148 * 8;
    return run_cached(h, std::make_tuple(25, B, l, fl), [&] {
      auto adam_bucket = [&](int k, cudaStream_t st, int grid) {
        const size_t b0 = h->bucket_off[k], n = h->bucket_off[k + 1] - b0;
        adam_range(st, h->w + b0, h->g + b0, h->m + b0, h->v + b0, n, h->d_sc, h->w_hi + b0, h->w_lo + b0, grid);
      };
      enqueue_forward(h, split, B, l, true);
      enqueue_backward_seg(h, B, l, true, 1);
      cudaEventRecord(h->ev_seg[0], h->stream);
      cudaStreamWaitEvent(h->comm_stream, h->ev_seg[0], 0);
      adam_bucket(0, h->comm_stream, c_lstm);
      enqueue_backward_seg(h, B, l, true, 2);
      cudaEventRecord(h->ev_seg[1], h->stream);
      cudaStreamWaitEvent(h->comm_stream, h->ev_seg[1], 0);
      adam_bucket(1, h->comm_stream, c_lstm);
      enqueue_backward_seg(h, B, l, true, 31);
      cudaEventRecord(h->ev_seg[2], h->stream);
      cudaStreamWaitEvent(h->comm_stream, h->ev_seg[2], 0);
      adam_bucket(3, h->comm_stream, c_wemb);
      cudaEventRecord(h->ev_comm, h->comm_stream);
      enqueue_backward_seg(h, B, l, true, 32);
      adam_bucket(2, h->stream, 148 * 8);
      cudaStreamWaitEvent(h->stream, h->ev_comm, 0);  // join the side branch
    });
  }
  if (h->nranks == 1) {
    return run_cached(h, std::make_tuple(mode == 2 ? 2 : 1, B, l, fl), [&] {
      enqueue_forward(h, split, B, l, true);
      for (int seg = 1; seg <= 3; seg++) enqueue_backward_seg(h, B, l, true, seg);
      if (mode == 2) enqueue_adam(h);
    });
  }
  static const bool force_nccl = getenv("LRCN_DP_NCCL") != nullptr;
  if (h->p2p_ready && !force_nccl) {
    h->loss_is_total = true;
    static const bool replicated = getenv("LRCN_DP_REPLICATED_ADAM") != nullptr;
    static const bool kernel_exchange = getenv("LRCN_DP_KERNEL_EXCHANGE") != nullptr;  // round-1 SM-driven exchange after the backward pass
    static const bool ce_exchange = getenv("LRCN_DP_CE") != nullptr;  // copy-engine exchange: measured slower (many small copies), kept for reference
    if (mode == 2 && !replicated) { h->adam_sharded = h->grad_sharded = true; h->shard_by_bucket = !kernel_exchange; }
    else h->grad_sharded = false;
    if (mode == 2 && !replicated && !kernel_exchange && !ce_exchange) {
      // Bucketed SM-driven exchange overlapped with the backward pass.  The owner-computes kernel of bucket 1 (Wout, bout) runs
      // on a side stream (a parallel branch of the step's graph) under the layer-2 BPTT kernel, that of bucket 2 (W2, b2, Wf, Wcnn)
      // under the layer-1 BPTT kernel: the persistent LSTM kernels hold 128 of the 148 SMs with one (register-file-filling) CTA
      // each, so the exchange CTAs land on the 20 SMs they leave free -- and because every exchange starts with a cross-GPU flag
      // barrier (a 1-warp kernel that co-resides anywhere), the LSTM grid is resident before the exchange kernel is launched.
      // The layer-1 segment ends with two buckets: the embedding gradient (Wemb, two thirds of the segment's bytes) is produced
      // FIRST (dE GEMM + scatter) and travels on the side stream under the layer-1 weight-gradient GEMM (whose CTAs leave room
      // for co-resident exchange CTAs on every SM); only bucket 3 (W1, b1) is exposed.
      static const int wemb_ctas = getenv("LRCN_DP_WEMB_CTAS") ? atoi(getenv("LRCN_DP_WEMB_CTAS")) : 148 * 4;
      static const bool stamps = getenv("LRCN_DP_STAMPS") != nullptr;
      return run_cached(h, std::make_tuple(24, B, l, fl), [&] {
        // stamps (tools/dp_timeline.py): main stream 0..7 = start, fwd done, seg1, seg2, seg31, seg32, last exchange done, joined;
        // bucket k: 8+4k .. = enter, first barrier passed, exchange kernel done, second barrier + split done
        auto stamp = [&](int id, cudaStream_t st) { if (stamps && h->d_trace) dp_stamp(st, h->d_trace + id); };
        static const bool pull = getenv("LRCN_DP_PULL") != nullptr;  // round-2a exchange: the owner LOADS its shard from every peer
        // measured at N = 2: 0.932 ms per step with the LL kernel on the exposed bucket vs 0.915 with the fused kernel (70 vs 50 us for
        // the bucket: 38 k threads polling their lines compete with the incoming stores), so it is opt-in
        static const bool ll = getenv("LRCN_DP_LL") != nullptr;
        static const bool fused = !pull && getenv("LRCN_DP_PUSH") == nullptr;  // default; LRCN_DP_PUSH=1: push / barrier / Adam / barrier as four kernels
        const size_t stride = stage_stride(h);
        auto exchange_bucket = [&](int k, cudaStream_t st, unsigned int* epoch, int flagset, bool last) {
          const int ctas = last ? 148 * 4 : (k == 3 ? wemb_ctas : 20 * 8);
          if (fused && last && ll) {
            // the exposed bucket: flag-in-data lines, no fences, no flag hops (dp_p2p.cu)
            stamp(8 + 4 * k, st);
            LLXArgs a{};
            for (int r = 0; r < h->nranks; r++) {
              const BucketShard bs = bucket_shard(h, k, r);
              a.stage[r] = h->peer_stage[r]; a.b4[r] = bs.b / 4; a.e4[r] = bs.e / 4; a.per4 = bs.per / 4;
            }
            a.llg4 = (h->P + 1024 + DP_XCTL_FLOATS) / 4; a.llw4 = a.llg4 + h->ll_floats / 4;
            dp_ll_exchange(st, h->peers, a, h->m, h->v, h->d_sc, h->d_loss_total, 148);
            stamp(10 + 4 * k, st);
            if (h->bf16mode) {
              const size_t b0 = h->bucket_off[k], nn = h->bucket_off[k + 1] - b0;
              split_bf16(st, h->w + b0, nn, h->w_hi + b0, h->w_lo + b0);
            }
            stamp(11 + 4 * k, st);
            return;
          }
          if (fused) {
            // ONE kernel per bucket: chunk-pipelined push -> flags -> owner sum + Adam -> weight push -> completion counters
            stamp(8 + 4 * k, st);
            FusedXArgs a{};
            for (int r = 0; r < h->nranks; r++) {
              const BucketShard bs = bucket_shard(h, k, r);
              a.stage[r] = h->peer_stage[r]; a.b4[r] = bs.b / 4; a.e4[r] = bs.e / 4;
              a.pre4 = bs.pre / 4;
            }
            a.stride4 = stride / 4; a.ctl4 = (h->P + 1024) / 4; a.bucket = k;
            dp_fused_exchange(st, h->peers, a, h->m, h->v, h->d_sc, last ? h->d_loss_total : nullptr, last ? 148 * 4 : (k == 3 ? wemb_ctas : 20 * 4));
            stamp(10 + 4 * k, st);
            if (h->bf16mode) {
              const size_t b0 = h->bucket_off[k], nn = h->bucket_off[k + 1] - b0;
              split_bf16(st, h->w + b0, nn, h->w_hi + b0, h->w_lo + b0);
            }
            stamp(11 + 4 * k, st);
            return;
          }
          if (!pull) {
            // PUSH exchange: (1) every rank stores its slices of the bucket's gradient into the owners' staging rows; (2) flag
            // barrier: all pushes have landed, and every rank is past its last use of the bucket's weights; (3) the owner sums the
            // N contributions in rank order, runs Adam on its slice and stores the new weights into every peer's arena;
            // (4) flag barrier: the new weights have landed everywhere; (5) local bf16 shadows.
            stamp(8 + 4 * k, st);
            float* dst[8]; const float* src[8]; size_t nf[8]; int n = 0;
            for (int d = 1; d < h->nranks; d++) {
              const int r = (h->rank + d) % h->nranks;  // staggered targets: no two ranks start on the same peer
              const BucketShard bs = bucket_shard(h, k, r);
              dst[n] = h->peer_stage[r] + (size_t)h->rank * stride + bs.pre; src[n] = h->g + bs.b; nf[n] = bs.e - bs.b; n++;
            }
            dp_push_slices(st, n, dst, src, nf, ctas);
            dp_xgpu_barrier(st, h->peers, epoch, flagset, stamps && h->d_trace ? h->d_trace + 32 + k : nullptr);
            stamp(9 + 4 * k, st);
            const BucketShard me = bucket_shard(h, k, h->rank);
            if (me.e > me.b || last)
              dp_adam_staged(st, h->w, h->g, h->m, h->v, h->stage, stride, me.pre, me.b, me.e, h->peers, h->d_sc, last ? h->d_loss_total : nullptr, true, ctas);
            stamp(10 + 4 * k, st);
            dp_xgpu_barrier(st, h->peers, epoch, flagset);
            if (h->bf16mode) {
              const size_t b0 = h->bucket_off[k], nn = h->bucket_off[k + 1] - b0;
              split_bf16(st, h->w + b0, nn, h->w_hi + b0, h->w_lo + b0);
            }
            stamp(11 + 4 * k, st);
            return;
          }
          stamp(8 + 4 * k, st);
          dp_xgpu_barrier(st, h->peers, epoch, flagset, stamps && h->d_trace ? h->d_trace + 32 + k : nullptr);  // every rank's gradients of this bucket are complete, and every rank is past its last use of the bucket's weights
          stamp(9 + 4 * k, st);
          const BucketShard me = bucket_shard(h, k, h->rank);
          if (me.e > me.b || last) dp_p2p_adam_range(st, h->peers, me.b, me.e, h->m, h->v, h->d_sc, last ? h->d_loss_total : nullptr, ctas);
          stamp(10 + 4 * k, st);
          dp_xgpu_barrier(st, h->peers, epoch, flagset);  // every owner's new weights of this bucket have landed everywhere
          if (h->bf16mode) {
            const size_t b0 = h->bucket_off[k], n = h->bucket_off[k + 1] - b0;
            split_bf16(st, h->w + b0, n, h->w_hi + b0, h->w_lo + b0);
          }
          stamp(11 + 4 * k, st);
        };
        stamp(0, h->stream);
        enqueue_forward(h, split, B, l, true);
        stamp(1, h->stream);
        enqueue_backward_seg(h, B, l, true, 1);
        stamp(2, h->stream);
        cudaEventRecord(h->ev_seg[0], h->stream);
        cudaStreamWaitEvent(h->comm_stream, h->ev_seg[0], 0);
        exchange_bucket(0, h->comm_stream, h->d_epoch_side, 1, false);
        enqueue_backward_seg(h, B, l, true, 2);
        stamp(3, h->stream);
        cudaEventRecord(h->ev_seg[1], h->stream);
        cudaStreamWaitEvent(h->comm_stream, h->ev_seg[1], 0);
        exchange_bucket(1, h->comm_stream, h->d_epoch_side, 1, false);
        enqueue_backward_seg(h, B, l, true, 31);
        stamp(4, h->stream);
        cudaEventRecord(h->ev_seg[2], h->stream);
        cudaStreamWaitEvent(h->comm_stream, h->ev_seg[2], 0);
        exchange_bucket(3, h->comm_stream, h->d_epoch_side, 1, false);
        cudaEventRecord(h->ev_comm, h->comm_stream);
        enqueue_backward_seg(h, B, l, true, 32);
        stamp(5, h->stream);
        exchange_bucket(2, h->stream, h->d_epoch, 0, true);
        stamp(6, h->stream);
        cudaStreamWaitEvent(h->stream, h->ev_comm, 0);  // join the side branch
        stamp(7, h->stream);
      });
    }
    if (mode == 2 && !replicated && !kernel_exchange) {
      // copy-engine exchange (dp_p2p.cu): bucket 1 (Wout, bout) travels under the layer-2 BPTT, bucket 2 (W2, b2, Wf, Wcnn)
      // under the layer-1 BPTT on a side stream (a parallel branch of the step's graph); only bucket 3 (W1, b1, Wemb) is exposed
      return run_cached(h, std::make_tuple(23, B, l, fl), [&] {
        const size_t stride = stage_stride(h);
        // the N-1 copies of a phase run on parallel branches of the graph (several DMA engines), forked from / joined into `st`
        auto parallel_copies = [&](cudaStream_t st, auto&& issue /* (rank r, stream) */) {
          if (h->nranks <= 2) { for (int r = 0; r < h->nranks; r++) if (r != h->rank) issue(r, st); return; }
          cudaEventRecord(h->ev_xfork, st);
          for (int i = 0; i < lrcn_handle::NXFER; i++) cudaStreamWaitEvent(h->xfer[i], h->ev_xfork, 0);
          int n = 0;
          for (int d = 1; d < h->nranks; d++, n++) issue((h->rank + d) % h->nranks, h->xfer[n % lrcn_handle::NXFER]);  // staggered targets: no two ranks start on the same peer
          for (int i = 0; i < lrcn_handle::NXFER; i++) { cudaEventRecord(h->ev_xjoin[i], h->xfer[i]); cudaStreamWaitEvent(st, h->ev_xjoin[i], 0); }
        };
        auto exchange_bucket = [&](int k, cudaStream_t st, unsigned int* epoch, int flagset, bool last) {
          parallel_copies(st, [&](int r, cudaStream_t cs) {  // reduce-scatter: push my gradient slices to their owners
            const BucketShard bs = bucket_shard(h, k, r);
            if (bs.e > bs.b) cudaMemcpyAsync(h->peer_stage[r] + (size_t)h->rank * stride + bs.pre, h->g + bs.b, (bs.e - bs.b) * 4, cudaMemcpyDeviceToDevice, cs);
          });
          dp_xgpu_barrier(st, h->peers, epoch, flagset);  // every rank's pushes of this bucket have landed (and every rank is past its last use of the bucket's weights)
          const BucketShard me = bucket_shard(h, k, h->rank);
          if (me.e > me.b || last)
            dp_adam_staged(st, h->w, h->g, h->m, h->v, h->stage, stride, me.pre, me.b, me.e, h->peers, h->d_sc, last ? h->d_loss_total : nullptr);
          if (me.e > me.b)
            parallel_copies(st, [&](int r, cudaStream_t cs) {  // all-gather: push the new weights of my slice
              cudaMemcpyAsync(h->peers.w[r] + me.b, h->w + me.b, (me.e - me.b) * 4, cudaMemcpyDeviceToDevice, cs);
            });
          dp_xgpu_barrier(st, h->peers, epoch, flagset);  // every owner's new weights of this bucket have landed everywhere
          if (h->bf16mode) {  // refresh the bf16 hi / lo shadows of the bucket (the exposed pass shrinks to the last bucket)
            const size_t b0 = h->bucket_off[k], n = h->bucket_off[k + 1] - b0;
            split_bf16(st, h->w + b0, n, h->w_hi + b0, h->w_lo + b0);
          }
        };
        enqueue_forward(h, split, B, l, true);
        enqueue_backward_seg(h, B, l, true, 1);
        cudaEventRecord(h->ev_seg[0], h->stream);
        cudaStreamWaitEvent(h->comm_stream, h->ev_seg[0], 0);
        exchange_bucket(0, h->comm_stream, h->d_epoch_side, 1, false);
        enqueue_backward_seg(h, B, l, true, 2);
        cudaEventRecord(h->ev_seg[1], h->stream);
        cudaStreamWaitEvent(h->comm_stream, h->ev_seg[1], 0);
        exchange_bucket(1, h->comm_stream, h->d_epoch_side, 1, false);
        cudaEventRecord(h->ev_comm, h->comm_stream);
        enqueue_backward_seg(h, B, l, true, 3);
        exchange_bucket(2, h->stream, h->d_epoch, 0, false);
        exchange_bucket(3, h->stream, h->d_epoch, 0, true);
        cudaStreamWaitEvent(h->stream, h->ev_comm, 0);  // join the side branch
      });
    }
    // backward pass, then ONE owner-computes exchange kernel over NVLink peer memory between two flag barriers (dp_p2p.cu),
    // then the replicated Adam: no NCCL kernels competing for SMs with the persistent GEMM / LSTM kernels
    return run_cached(h, std::make_tuple(mode == 2 ? 22 : 21, B, l, fl), [&] {
      enqueue_forward(h, split, B, l, true);
      for (int seg = 1; seg <= 3; seg++) enqueue_backward_seg(h, B, l, true, seg);
      if (mode == 2 && !replicated) {
        // reduce-scatter + Adam on the owned shard + all-gather of the new weights in one kernel; then the local bf16 shadows
        dp_p2p_adam(h->stream, h->peers, h->P, h->d_epoch, h->d_loss_total, h->m, h->v, h->d_sc);
        if (h->bf16mode) split_bf16(h->stream, h->w, h->P, h->w_hi, h->w_lo);
      } else {
        dp_p2p_allreduce(h->stream, h->peers, h->P, h->d_epoch, h->d_loss_total);
        if (mode == 2) enqueue_adam(h);
      }
    });
  }
  if (!h->comm) return fail(LRCN_ERR_ARG, "data-parallel group not initialised (lrcn_comm_init or lrcn_p2p_import)");
  NcclApi* n = nccl_api();
  static const bool bucketed = getenv("LRCN_DP_BUCKETS") != nullptr;  // measured: one allreduce after the backward pass beats 3 overlapped buckets
  if (!bucketed) {
    // one allreduce over the whole gradient arena after the backward pass (no overlap, but no SM contention between the NCCL
    // kernels and the persistent GEMM / LSTM kernels either)
    rc = run_cached(h, std::make_tuple(20, B, l, fl), [&] {
      enqueue_forward(h, split, B, l, true);
      for (int seg = 1; seg <= 3; seg++) enqueue_backward_seg(h, B, l, true, seg);
    });
    if (rc) return rc;
    rc = nccl_check(n->GroupStart(), "ncclGroupStart"); if (rc) return rc;
    rc = nccl_check(n->AllReduce(h->g, h->g, h->P, NCCL_FLOAT32, NCCL_SUM, h->comm, h->stream), "ncclAllReduce(grad)"); if (rc) return rc;
    rc = nccl_check(n->AllReduce(h->d_loss, h->d_loss, 1, NCCL_FLOAT64, NCCL_SUM, h->comm, h->stream), "ncclAllReduce(loss)"); if (rc) return rc;
    rc = nccl_check(n->GroupEnd(), "ncclGroupEnd"); if (rc) return rc;
    if (mode == 2) {
      rc = run_cached(h, std::make_tuple(14, 0, 0, 0), [&] { enqueue_adam(h); });
      if (rc) return rc;
    }
    return LRCN_OK;
  }
  // data-parallel: bucketed allreduce on the comm stream, overlapped with the remaining backward segments
  rc = run_cached(h, std::make_tuple(10, B, l, fl), [&] { enqueue_forward(h, split, B, l, true); enqueue_backward_seg(h, B, l, true, 1); });
  if (rc) return rc;
  for (int seg = 1; seg <= 3; seg++) {
    CK(cudaEventRecord(h->ev_seg[seg - 1], h->stream));
    CK(cudaStreamWaitEvent(h->comm_stream, h->ev_seg[seg - 1], 0));
    float* gb = h->g + h->bucket_off[seg - 1];
    size_t cnt = h->bucket_off[seg == 3 ? lrcn_handle::NBUCKET : seg] - h->bucket_off[seg - 1];  // the last allreduce takes (W1, b1) and Wemb
    if (seg == 3) { rc = nccl_check(n->GroupStart(), "ncclGroupStart"); if (rc) return rc; }
    rc = nccl_check(n->AllReduce(gb, gb, cnt, NCCL_FLOAT32, NCCL_SUM, h->comm, h->comm_stream), "ncclAllReduce(grad bucket)");
    if (rc) return rc;
    if (seg == 3) {
      rc = nccl_check(n->AllReduce(h->d_loss, h->d_loss, 1, NCCL_FLOAT64, NCCL_SUM, h->comm, h->comm_stream), "ncclAllReduce(loss)");
      if (rc) return rc;
      rc = nccl_check(n->GroupEnd(), "ncclGroupEnd");
      if (rc) return rc;
    }
    if (seg < 3) {
      rc = run_cached(h, std::make_tuple(10 + seg, B, l, fl), [&] { enqueue_backward_seg(h, B, l, true, seg + 1); });
      if (rc) return rc;
    }
  }
  CK(cudaEventRecord(h->ev_comm, h->comm_stream));
  CK(cudaStreamWaitEvent(h->stream, h->ev_comm, 0));
  if (mode == 2) {
    rc = run_cached(h, std::make_tuple(14, 0, 0, 0), [&] { enqueue_adam(h); });
    if (rc) return rc;
  }
  return LRCN_OK;
}

static int finish_loss(lrcn_handle* h, int B, int l, double* total_out) {
  CK(cudaMemcpyAsync(h->h_loss, h->loss_is_total ? h->d_loss_total : h->d_loss, 8, cudaMemcpyDeviceToHost, h->stream));
  int rc = sync_stream(h);
  if (rc) return rc;
  *total_out = *h->h_loss;
  return LRCN_OK;
}

static int stage_current(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B) {
  const size_t R = (size_t)(l + 1) * B;
  int* tin = h->h_stage;
  int* ttg = h->h_stage + R;
  int* rows = h->h_stage + 2 * R;
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));  // pinned staging buffer is reused
  int rc = stage_host(h, split, image_ids, tokens, l, B, tin, ttg, rows);
  if (rc) return rc;
  CK(cudaMemcpyAsync(h->d_tok_in, tin, R * 4, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_tok_tgt, ttg, R * 4, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_rows, rows, (size_t)B * 4, cudaMemcpyHostToDevice, h->stream));
  return LRCN_OK;
}

static int s_loss(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B, double* sum_logp_out,
                         int64_t* count_out) {
  int rc = stage_current(h, split, image_ids, tokens, l, B);
  if (rc) return rc;
  rc = run_step(h, split, B, l, 0.f, 0, 0);
  if (rc) return rc;
  double total;
  rc = finish_loss(h, B, l, &total);
  if (rc) return rc;
  if (sum_logp_out) *sum_logp_out = total;
  if (count_out) *count_out = (int64_t)B * (l + 1);
  return LRCN_OK;
}
static int s_grad(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B, float pdrop, uint64_t seed,
                         double* loss_out) {
  if (pdrop < 0.f || pdrop >= 1.f) return fail(LRCN_ERR_ARG, "pdrop must be in [0,1)");
  int rc = stage_current(h, split, image_ids, tokens, l, B);
  if (rc) return rc;
  rc = run_step(h, split, B, l, pdrop, seed, 1);
  if (rc) return rc;
  double total;
  rc = finish_loss(h, B, l, &total);
  if (rc) return rc;
  if (loss_out) *loss_out = -total / (global_rows(h, B) * (l + 1));
  return LRCN_OK;
}
static int s_train_step(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B, float pdrop,
                               uint64_t seed, double* loss_out) {
  if (pdrop < 0.f || pdrop >= 1.f) return fail(LRCN_ERR_ARG, "pdrop must be in [0,1)");
  int rc = stage_current(h, split, image_ids, tokens, l, B);
  if (rc) return rc;
  rc = run_step(h, split, B, l, pdrop, seed, 2);
  if (rc) return rc;
  double total;
  rc = finish_loss(h, B, l, &total);
  if (rc) return rc;
  if (loss_out) *loss_out = -total / (global_rows(h, B) * (l + 1));
  return LRCN_OK;
}
static int s_adam_update(lrcn_handle* h) {
  if (!h) return fail(LRCN_ERR_ARG, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  // Peer-memory data parallelism keeps m, v current only in each owner's shard, and after a sharded train step the summed
  // gradient too: a dense local Adam over the whole arena would silently diverge the replicas.
  if (h->nranks > 1 && h->adam_sharded)
    return fail(LRCN_ERR_STATE, "lrcn_adam_update after a sharded data-parallel train step: Adam state is distributed over the ranks; "
                                "call lrcn_get_adam_state (gathers it) on every rank first, or keep using lrcn_train_step");
  { int rc0 = push_scalars(h, 1, 0, 0.f, 0, true); if (rc0) return rc0; }
  g_counter = &h->counter;
  enqueue_adam(h);
  return sync_stream(h);
}
static int s_get_token_logps(lrcn_handle* h, float* out, int64_t n) {
  if (!h || !out) return fail(LRCN_ERR_ARG, "null");
  int64_t have = (int64_t)h->last_B * (h->last_l + 1);
  if (n != have) return fail(LRCN_ERR_ARG, "expected %lld values", (long long)have);
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpyAsync(out, WS(h, h->o.rowlp), (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return LRCN_OK;
}

static int s_stage_batch(lrcn_handle* h, int slot, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B) {
  if (!h || slot < 0 || slot >= 64) return fail(LRCN_ERR_ARG, "slot outside [0,64)");
  const size_t R = (size_t)(l + 1) * B;
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));
  int rc = stage_host(h, split, image_ids, tokens, l, B, h->h_stage, h->h_stage + R, h->h_stage + 2 * R);
  if (rc) return rc;
  Slot& s = h->slots[slot];
  if (!s.tok_in) {
    const size_t Rmax = (size_t)(h->cfg.max_len + 1) * h->cfg.max_batch;
    CK(cudaMalloc(&s.tok_in, Rmax * 4)); CK(cudaMalloc(&s.tok_tgt, Rmax * 4)); CK(cudaMalloc(&s.rows, (size_t)h->cfg.max_batch * 4));
  }
  s.l = l; s.B = B; s.split = split;
  CK(cudaMemcpyAsync(s.tok_in, h->h_stage, R * 4, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(s.tok_tgt, h->h_stage + R, R * 4, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(s.rows, h->h_stage + 2 * R, (size_t)B * 4, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return LRCN_OK;
}
static int s_train_step_staged(lrcn_handle* h, int slot, float pdrop, uint64_t seed, double* loss_out) {
  if (!h || slot < 0 || slot >= 64 || !h->slots[slot].tok_in) return fail(LRCN_ERR_ARG, "slot %d not staged", slot);
  if (pdrop < 0.f || pdrop >= 1.f) return fail(LRCN_ERR_ARG, "pdrop must be in [0,1)");
  Slot& s = h->slots[slot];
  const size_t R = (size_t)(s.l + 1) * s.B;
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpyAsync(h->d_tok_in, s.tok_in, R * 4, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_tok_tgt, s.tok_tgt, R * 4, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_rows, s.rows, (size_t)s.B * 4, cudaMemcpyDeviceToDevice, h->stream));
  int rc = run_step(h, s.split, s.B, s.l, pdrop, seed, 2);
  if (rc) return rc;
  if (loss_out) {
    double total;
    rc = finish_loss(h, s.B, s.l, &total);
    if (rc) return rc;
    *loss_out = -total / (global_rows(h, s.B) * (s.l + 1));
  }
  return LRCN_OK;
}

// ------------------------------------------------------------------------------------------ generation
static void beam_lstm_step(lrcn_handle* h, int layer, int step, int R, float* g, float* h_in, float* c_in, float* h_out, float* c_out) {
  const int H = layer == 1 ? h->H1 : h->H2;
  const int ldw = layer == 1 ? h->E + h->H1 : 2 * h->H2, x_off = layer == 1 ? h->E : 2 * h->C;
  if (h->bf16mode) {
    bf16 *hi_hi, *hi_lo, *ho_hi, *ho_lo;
    shadow(h, h_in, &hi_hi, &hi_lo);
    shadow(h, h_out, &ho_hi, &ho_lo);
    if (!lstm_fwd_step(h->stream, R, H, step > 1, hi_hi, hi_lo, layer == 1 ? h->wp1_hi : h->wp2_hi, layer == 1 ? h->wp1_lo : h->wp2_lo, g, c_in, c_out,
                       h_out, ho_hi, ho_lo))
      throw GemmFail{gemm_bf16x3_last_error()};
    return;
  }
  if (step > 1) sgemm(h->stream, true, true, R, 4 * H, H, h_in, H, Wp(h, layer == 1 ? 1 : 3) + x_off, ldw, g, 4 * H, true, nullptr);
  lstm_cell_fwd(h->stream, g, c_in, c_out, h_out, R, H);
}
// many rows in flight: throughput path.  The step's two gate GEMMs run on concatenated [x|h] operands (exactly the
// reference's hcat(input,hidden)*weight, lrcn.jl:529) so there is no accumulate pass over the gates.
static bool beam_wide(const lrcn_handle* h, int R) { return h->bf16mode && R > 512; }

// need_embed: gather the step's input embeddings here (first step, after a compaction, unfused mode); otherwise the previous
// step's advance kernel has already written them
static void enqueue_beam_step(lrcn_handle* h, int n_img, int K, int step, int nword, int maxlen, bool flip, float* out_lp, bool wide, const int* out_map,
                              bool need_embed) {
  const int R = n_img * K, E = h->E, H1 = h->H1, H2 = h->H2, C = h->C, V = h->V, ldV = h->ldV, ldv = h->ldv;
  const Workspace& o = h->o;
  cudaStream_t s = h->stream;
  float *e = WS(h, o.ge), *g1 = WS(h, o.gg1), *z = WS(h, o.gz), *g2 = WS(h, o.gg2), *logits = WS(h, o.glogits), *v = WS(h, o.gv);
  // state ping-pong: "a" holds the beams' current states; the cell writes advanced states into "b"; advance gathers b -> a
  float *h1a = WS(h, o.gh1a), *c1a = WS(h, o.gc1a), *h1b = WS(h, o.gh1b), *c1b = WS(h, o.gc1b);
  float *h2a = WS(h, o.gh2a), *c2a = WS(h, o.gc2a), *h2b = WS(h, o.gh2b), *c2b = WS(h, o.gc2b);
  int ld1 = H1, ld2 = H2;
  if (wide) {
    float *xh1 = WS(h, o.gxh1), *xh2 = WS(h, o.gxh2);
    ld1 = E + H1; ld2 = 2 * C + H2;
    if (need_embed) gather_embed(s, Wp(h, 7), h->g_last, R, E, xh1, h->d_sc, false, SH(h, xh1).hi, SH(h, xh1).lo, ld1);     // Wemb[tok:tok,:]  lrcn.jl:650
    gemm(h, true, true, R, 4 * H1, E + H1, xh1, ld1, Wp(h, 1), E + H1, g1, 4 * H1, false, Wp(h, 2));        // hcat(x,h)*W .+ b  lrcn.jl:529
    if (H1 % 4 == 0) lstm_cell_gen(s, g1, c1a, c1b, h1b, R, H1, SH(h, h1b).hi, SH(h, h1b).lo);
    else lstm_cell_fwd(s, g1, c1a, c1b, h1b, R, H1, SH(h, h1b).hi, SH(h, h1b).lo);
    // hcat(x*w[end-4], x_cnn) (lrcn.jl:545-546): the image half of a row is the same at every step, so it is written (with its
    // bf16 split) only at the first step and after a compaction; otherwise the GEMM's epilogue writes the split of its own half
    gemm(h, true, true, R, C, H1, h1b, H1, Wp(h, 5), H1, xh2, ld2, false, nullptr, !need_embed);
    if (need_embed) z_finish(s, xh2, v, ldv, R, -K, C, h->d_sc, false, SH(h, xh2).hi, SH(h, xh2).lo, ld2);
    gemm(h, true, true, R, 4 * H2, 2 * C + H2, xh2, ld2, Wp(h, 3), 2 * H2, g2, 4 * H2, false, Wp(h, 4));
    if (H2 % 4 == 0) lstm_cell_gen(s, g2, c2a, c2b, h2b, R, H2, SH(h, h2b).hi, SH(h, h2b).lo);
    else lstm_cell_fwd(s, g2, c2a, c2b, h2b, R, H2, SH(h, h2b).hi, SH(h, h2b).lo);
    h1a = xh1 + E;       // the gathered parent states go straight into the h columns of the next step's operands
    h2a = xh2 + 2 * C;
  } else {
    if (need_embed) gather_embed(s, Wp(h, 7), h->g_last, R, E, e, h->d_sc, false, SH(h, e).hi, SH(h, e).lo);                // Wemb[tok:tok,:]  lrcn.jl:650
    gemm(h, true, true, R, 4 * H1, E, e, E, Wp(h, 1), E + H1, g1, 4 * H1, false, Wp(h, 2));
    beam_lstm_step(h, 1, step, R, g1, h1a, c1a, h1b, c1b);
    gemm(h, true, true, R, C, H1, h1b, H1, Wp(h, 5), H1, z, 2 * C, false, nullptr, !need_embed);
    if (need_embed) z_finish(s, z, v, ldv, R, -K, C, h->d_sc, false, SH(h, z).hi, SH(h, z).lo);  // negative B => image index = row / K
    gemm(h, true, true, R, 4 * H2, 2 * C, z, 2 * C, Wp(h, 3), 2 * H2, g2, 4 * H2, false, Wp(h, 4));
    beam_lstm_step(h, 2, step, R, g2, h2a, c2a, h2b, c2b);
  }
  gemm(h, true, true, R, V, H2, h2b, H2, Wp(h, 8), H2, logits, ldV, false, Wp(h, 9));
  beam_row_topk(s, logits, ldV, R, V, K, WS(h, o.gprob), h->g_ctok, WS(h, o.gcs), WS(h, o.gclp));             // lrcn.jl:652-661
  static const bool unfused = getenv("LRCN_BEAM_UNFUSED") != nullptr;  // selection, advance and done-marking as three launches
  if (unfused) beam_select(s, h->g_ctok, WS(h, o.gcs), WS(h, o.gclp), n_img, K, step == 1, h->g_stok, h->g_spar, WS(h, o.gss), WS(h, o.gslp));  // :667-668
  BeamAdvanceArgs a;
  a.fused = unfused ? 0 : 1; a.cand_tok = h->g_ctok; a.cand_score = WS(h, o.gcs); a.cand_lp = WS(h, o.gclp);
  {
    float* ebuf = wide ? WS(h, o.gxh1) : e;
    a.wemb = unfused ? nullptr : Wp(h, 7); a.e_out = ebuf; a.e_hi = SH(h, ebuf).hi; a.e_lo = SH(h, ebuf).lo; a.E = E; a.lde = wide ? E + H1 : E;
  }
  a.n_img = n_img; a.K = K; a.H1 = H1; a.H2 = H2; a.maxlen = maxlen; a.step = step; a.nword = nword;
  a.ld1 = ld1; a.ld2 = ld2;
  a.sel_tok = h->g_stok; a.sel_parent = h->g_spar; a.sel_score = WS(h, o.gss); a.sel_lp = WS(h, o.gslp);
  a.h1_in = h1b; a.c1_in = c1b; a.h2_in = h2b; a.c2_in = c2b; a.h1_out = h1a; a.c1_out = c1a; a.h2_out = h2a; a.c2_out = c2a;
  a.hist_in = flip ? h->g_histb : h->g_hista; a.hist_out = flip ? h->g_hista : h->g_histb;
  a.lp_in = flip ? WS(h, o.glpb) : WS(h, o.glpa); a.lp_out = flip ? WS(h, o.glpa) : WS(h, o.glpb);
  a.h1_hi = SH(h, h1a).hi; a.h1_lo = SH(h, h1a).lo; a.h2_hi = SH(h, h2a).hi; a.h2_lo = SH(h, h2a).lo;
  a.prob = WS(h, o.gprob); a.last_tok = h->g_last; a.done = h->g_done; a.n_done = h->g_ndone;
  a.out_tokens = h->g_otok; a.out_len = h->g_olen; a.out_prob = WS(h, o.goprob); a.out_lp = out_lp; a.out_map = out_map;
  beam_advance(s, a);  // reorder/gather parent states (+ their bf16 split for the next recurrent GEMMs)                 lrcn.jl:670-677
}

__global__ void beam_init_kernel(int R, int maxlen, float* prob, int* last, int* hist, float* lp, int* done, int* n_done, int n_img, int* out_map) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r == 0) *n_done = 0;
  if (r < n_img) { done[r] = 0; out_map[r] = r; }  // compacted -> caller index: identity until the first compaction
  if (r >= R) return;
  prob[r] = 1.0f;  // (bos, 1.0)  lrcn.jl:627
  last[r] = 1;     // bos, 0-based
  hist[(size_t)r * maxlen] = 1;
  lp[(size_t)r * maxlen] = 0.f;
}

static int s_beam_search(lrcn_handle* h, int split, const int64_t* image_ids, int64_t n, int K, int nword, int64_t* tokens_out,
                                int32_t* len_out, float* prob_out, float* logp_out) {
  if (!h || !image_ids || !tokens_out || !len_out || !prob_out || n <= 0) return fail(LRCN_ERR_ARG, "bad argument to lrcn_beam_search");
  if (K < 1 || K > 11) return fail(LRCN_ERR_ARG, "beam_width %d outside [1,11]", K);
  if (nword < 1 || nword + 2 > 64) return fail(LRCN_ERR_ARG, "nword %d outside [1,62]", nword);
  if (split < 0 || split > 1 || !h->tab[split].d) return fail(LRCN_ERR_STATE, "no features loaded for split %d", split);
  if (K > h->cfg.max_gen_rows) return fail(LRCN_ERR_ARG, "max_gen_rows %d < beam_width", h->cfg.max_gen_rows);
  CK(cudaSetDevice(h->cfg.device));
  g_counter = &h->counter;
  const int maxlen = nword + 2;
  const int chunk = h->cfg.max_gen_rows / K;
  const Workspace& o = h->o;
  const Table& tb = h->tab[split];
  std::vector<int> rows;
  std::vector<long long> otok;
  for (int64_t base = 0; base < n; base += chunk) {
    const int ni = (int)((n - base) < chunk ? (n - base) : chunk);
    const int R = ni * K;
    rows.resize(ni);
    for (int i = 0; i < ni; i++) {
      auto it = tb.map.find(image_ids[base + i]);
      if (it == tb.map.end()) return fail(LRCN_ERR_MISSING, "missing features for image id %lld (lrcn.jl:602-605)", (long long)image_ids[base + i]);
      rows[i] = it->second;
    }
    { int rc0 = push_scalars(h, 1, 0, 0.f, 0, false); if (rc0) return rc0; }
    CK(cudaMemcpyAsync(h->g_rows, rows.data(), (size_t)ni * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    try {
      if (h->bf16mode) {
        lstm_prepare_weights2(h->stream, Wp(h, 1), h->E + h->H1, h->E, h->H1, h->wp1_hi, h->wp1_lo, nullptr, nullptr, Wp(h, 3), 2 * h->H2,
                              2 * h->C, h->H2, h->wp2_hi, h->wp2_lo, nullptr, nullptr);
      }
      gather_features(h->stream, tb.d, h->g_rows, ni, WS(h, o.gX), SH(h, WS(h, o.gX)).hi, SH(h, WS(h, o.gX)).lo);
      gemm(h, true, true, ni, h->C, LRCN_F_CNN, WS(h, o.gX), LRCN_F_CNN, Wp(h, 6), LRCN_F_CNN, WS(h, o.gv), h->ldv, false, nullptr);  // lrcn.jl:611
      beam_init_kernel<<<(R + 255) / 256, 256, 0, h->stream>>>(R, maxlen, WS(h, o.gprob), h->g_last, h->g_hista, WS(h, o.glpa), h->g_done, h->g_ndone, ni, h->g_omap);
      h->counter.n++;
      if (beam_wide(h, R)) {  // h_0 = 0 in the h columns of the [x|h] operands (fp32 and bf16 shadows)
        const size_t n1 = (size_t)R * (h->E + h->H1), n2 = (size_t)R * (2 * h->C + h->H2);
        CK(cudaMemsetAsync(WS(h, o.gxh1), 0, n1 * 4, h->stream)); CK(cudaMemsetAsync(WS(h, o.gxh2), 0, n2 * 4, h->stream));
        CK(cudaMemsetAsync(SH(h, WS(h, o.gxh1)).hi, 0, n1 * 2, h->stream)); CK(cudaMemsetAsync(SH(h, WS(h, o.gxh1)).lo, 0, n1 * 2, h->stream));
        CK(cudaMemsetAsync(SH(h, WS(h, o.gxh2)).hi, 0, n2 * 2, h->stream)); CK(cudaMemsetAsync(SH(h, WS(h, o.gxh2)).lo, 0, n2 * 2, h->stream));
      }
      CK(cudaMemsetAsync(WS(h, o.gc1a), 0, (size_t)R * h->H1 * 4, h->stream));
      CK(cudaMemsetAsync(WS(h, o.gc2a), 0, (size_t)R * h->H2 * 4, h->stream));
      bool flip = false;
      const bool wide = beam_wide(h, R);  // fixed for the chunk: the two paths keep the states in different buffers
      int n_act = ni;                     // images still in flight (compacted to the front)
      static const bool no_compact = getenv("LRCN_BEAM_NO_COMPACT") != nullptr;
      static const int den = getenv("LRCN_BEAM_COMPACT_DEN") ? atoi(getenv("LRCN_BEAM_COMPACT_DEN")) : 8;
      static const int lag = getenv("LRCN_BEAM_LAG") ? atoi(getenv("LRCN_BEAM_LAG")) : 1;  // 1..NSNAP-1 (measured: 1 = 162k, 2 = 157k, 3 = 152k captions/s: later decisions cost more than the queued step gains)
      // Asynchronous polling.  After EVERY step the done flags are copied into a ring of pinned snapshots (+ an event); the host
      // reads the snapshot of step s-1 right after it has enqueued step s, so the GPU always has a whole step queued while the
      // host waits, decides and enqueues -- the pipeline never drains (round 2a polled every 4 steps with a full
      // synchronisation and two more per compaction).  A decision taken from a one-step-old snapshot is safe: done flags only
      // ever rise, the compaction kernel carries the CURRENT flag of every survivor along, and an image that ended in between
      // simply rides until the next compaction.
      // Compaction: the reference decodes image by image and simply stops when an image ends (lrcn.jl:670); in a batch the
      // finished images would ride along until the slowest one ends (COCO captions end after ~10 of the 31 possible steps).
      // When at least 1/den of the images in flight have ended, the survivors move to the front and every later step (three
      // GEMMs, top-K, state gather) runs on the smaller batch.
      const int G1 = h->cfg.max_gen_rows + 1;
      int snap_gen[lrcn_handle::NSNAP], snap_n[lrcn_handle::NSNAP], gen = 0, n_compactions = 0;
      for (int q = 0; q < lrcn_handle::NSNAP; q++) snap_gen[q] = -1;
      bool all_done = false;
      static const bool beam_unfused = getenv("LRCN_BEAM_UNFUSED") != nullptr;
      bool need_embed = true;
      static const bool beam_debug = getenv("LRCN_BEAM_DEBUG") != nullptr;
      double wait_us = 0.0;
      const auto tl0 = std::chrono::steady_clock::now();
      int steps_run = 0;
      for (int step = 1; step <= nword + 1 && !all_done; step++) {
        steps_run = step;
        enqueue_beam_step(h, n_act, K, step, nword, maxlen, flip, logp_out ? WS(h, o.golp) : nullptr, wide, h->g_omap, need_embed);
        need_embed = beam_unfused;
        flip = !flip;
        const int q = step % lrcn_handle::NSNAP;
        int* snap = h->h_ndone + (size_t)q * G1;
        // the copies run on the side stream (an in-stream D2H copy stalls the kernel stream for ~5 us); the flags only ever rise,
        // so a copy that overlaps the next step is still a valid (older or newer) snapshot, and one that overlaps a compaction
        // belongs to the old numbering and is ignored (its done-count stays valid)
        CK(cudaEventRecord(h->ev_fork, h->stream));
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
        CK(cudaMemcpyAsync(snap, h->g_ndone, 4, cudaMemcpyDeviceToHost, h->side_stream));
        CK(cudaMemcpyAsync(snap + 1, h->g_done, (size_t)n_act * 4, cudaMemcpyDeviceToHost, h->side_stream));
        CK(cudaEventRecord(h->ev_snap[q], h->side_stream));
        snap_gen[q] = gen; snap_n[q] = n_act;
        if (step <= lag) continue;
        const int p = (step - lag) % lrcn_handle::NSNAP;  // an earlier step's snapshot: the GPU keeps `lag` steps queued while the host waits
        const auto tw0 = std::chrono::steady_clock::now();
        CK(cudaEventSynchronize(h->ev_snap[p]));
        if (beam_debug) wait_us += std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - tw0).count();
        const int* ps = h->h_ndone + (size_t)p * G1;
        if (ps[0] >= ni) { all_done = true; break; }      // (the step already enqueued runs on frozen images: a no-op)
        if (snap_gen[p] != gen || no_compact || step >= nword + 1) continue;  // indices of an older numbering
        int n_keep = 0;
        for (int i = 0; i < n_act; i++) n_keep += ps[1 + i] ? 0 : 1;
        if (n_keep == 0 || (n_act - n_keep) * den < n_act) continue;
        const int kq = n_compactions % lrcn_handle::NSNAP;
        if (n_compactions >= lrcn_handle::NSNAP) CK(cudaEventSynchronize(h->ev_keep[kq]));  // the list's previous upload has executed
        int* keep = h->h_keep + (size_t)kq * h->cfg.max_gen_rows;
        for (int i = 0, n = 0; i < n_act; i++) if (!ps[1 + i]) keep[n++] = i;
        CK(cudaMemcpyAsync(h->g_keep, keep, (size_t)n_keep * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaEventRecord(h->ev_keep[kq], h->stream));
        BeamCompactArgs ca{};
        ca.n_keep = n_keep; ca.K = K; ca.H1 = h->H1; ca.H2 = h->H2; ca.ldv = h->ldv; ca.maxlen = maxlen; ca.hist_len = step + 1;
        ca.ld1 = wide ? h->E + h->H1 : h->H1; ca.ld2 = wide ? 2 * h->C + h->H2 : h->H2;
        ca.keep = h->g_keep;
        ca.h1 = wide ? WS(h, o.gxh1) + h->E : WS(h, o.gh1a); ca.h2 = wide ? WS(h, o.gxh2) + 2 * h->C : WS(h, o.gh2a);
        ca.c1 = WS(h, o.gc1a); ca.c2 = WS(h, o.gc2a);
        ca.h1_s = WS(h, o.gh1b); ca.c1_s = WS(h, o.gc1b); ca.h2_s = WS(h, o.gh2b); ca.c2_s = WS(h, o.gc2b);  // the "advanced state" buffers are free between steps
        ca.h1_hi = SH(h, ca.h1).hi; ca.h1_lo = SH(h, ca.h1).lo; ca.h2_hi = SH(h, ca.h2).hi; ca.h2_lo = SH(h, ca.h2).lo;
        ca.hist_src = flip ? h->g_histb : h->g_hista; ca.hist_dst = flip ? h->g_hista : h->g_histb;
        ca.lp_src = flip ? WS(h, o.glpb) : WS(h, o.glpa); ca.lp_dst = flip ? WS(h, o.glpa) : WS(h, o.glpb);
        ca.prob = WS(h, o.gprob); ca.prob_s = WS(h, o.gss); ca.last = h->g_last; ca.last_s = h->g_stok;
        ca.v = WS(h, o.gv); ca.v_s = WS(h, o.gX);  // the gathered features are dead once v = X * Wcnn exists
        ca.out_map = h->g_omap; ca.out_map_s = h->g_omap_s; ca.done = h->g_done; ca.done_s = h->g_omap_s + h->cfg.max_gen_rows;
        beam_compact(h->stream, ca);
        flip = !flip;  // the compacted histories live in the other ping-pong buffer
        n_act = n_keep;
        need_embed = true;  // rows moved: the next step gathers its embeddings from the compacted token list
        gen++; n_compactions++;
      }
      if (beam_debug)
        fprintf(stderr, "[lrcn beam] %d images, %d steps enqueued, %d compactions: host loop %.0f us, of which %.0f us waiting for the GPU\n", ni, steps_run,
                n_compactions, std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - tl0).count(), wait_us);
    } catch (GemmFail& f) {
      return fail(LRCN_ERR_CUDA, "%s", f.msg.c_str());
    }
    CK(cudaPeekAtLastError());
    otok.resize((size_t)ni * maxlen);
    CK(cudaMemcpyAsync(otok.data(), h->g_otok, (size_t)ni * maxlen * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(len_out + base, h->g_olen, (size_t)ni * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(prob_out + base, WS(h, o.goprob), (size_t)ni * 4, cudaMemcpyDeviceToHost, h->stream));
    if (logp_out) CK(cudaMemcpyAsync(logp_out + base * (maxlen - 1), WS(h, o.golp), (size_t)ni * (maxlen - 1) * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < ni; i++) {
      int len = len_out[base + i];
      for (int j = 0; j < maxlen; j++) tokens_out[(base + i) * maxlen + j] = j < len ? (int64_t)otok[(size_t)i * maxlen + j] : 0;
    }
  }
  return LRCN_OK;
}

// ------------------------------------------------------------------------------------------ data-parallel group
extern "C" int lrcn_comm_unique_id(char id[LRCN_COMM_ID_BYTES]) {
  NcclApi* n = nccl_api();
  if (!n) return fail(LRCN_ERR_NCCL, "libnccl.so.2 not loadable: %s", dlerror() ? dlerror() : "?");
  ncclUniqueId u;
  int rc = nccl_check(n->GetUniqueId(&u), "ncclGetUniqueId");
  if (rc) return rc;
  memcpy(id, u.internal, LRCN_COMM_ID_BYTES);
  return LRCN_OK;
}
static int s_comm_init(lrcn_handle* h, const char id[LRCN_COMM_ID_BYTES], int rank, int nranks) {
  if (!h || !id || nranks < 1 || rank < 0 || rank >= nranks) return fail(LRCN_ERR_ARG, "bad rank/nranks");
  NcclApi* n = nccl_api();
  if (!n) return fail(LRCN_ERR_NCCL, "libnccl.so.2 not loadable");
  CK(cudaSetDevice(h->cfg.device));
  ncclUniqueId u;
  memcpy(u.internal, id, LRCN_COMM_ID_BYTES);
  int rc = nccl_check(n->CommInitRank(&h->comm, nranks, u, rank), "ncclCommInitRank");
  if (rc) return rc;
  h->rank = rank; h->nranks = nranks;
  return LRCN_OK;
}

struct P2PBlob {  // LRCN_P2P_BLOB_BYTES
  int magic, device;
  unsigned long long arena_floats;
  cudaIpcMemHandle_t g, ctl, w, m, v, stage;
};
static_assert(sizeof(P2PBlob) <= LRCN_P2P_BLOB_BYTES, "blob too large");
static int s_p2p_export(lrcn_handle* h, char blob[LRCN_P2P_BLOB_BYTES]) {
  if (!h || !blob) return fail(LRCN_ERR_ARG, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  P2PBlob b;
  memset(&b, 0, sizeof b);
  b.magic = 0x4C524350; b.device = h->cfg.device; b.arena_floats = h->P;
  CK(cudaIpcGetMemHandle(&b.g, h->g));
  CK(cudaIpcGetMemHandle(&b.ctl, h->p2p_ctl));
  CK(cudaIpcGetMemHandle(&b.w, h->w));
  CK(cudaIpcGetMemHandle(&b.m, h->m));
  CK(cudaIpcGetMemHandle(&b.v, h->v));
  CK(cudaIpcGetMemHandle(&b.stage, h->stage));
  memset(blob, 0, LRCN_P2P_BLOB_BYTES);
  memcpy(blob, &b, sizeof b);
  return LRCN_OK;
}
static int s_p2p_import(lrcn_handle* h, const char* blobs, int rank, int nranks) {
  if (!h || !blobs || nranks < 1 || nranks > LRCN_P2P_MAX_RANKS || rank < 0 || rank >= nranks)
    return fail(LRCN_ERR_ARG, "bad rank/nranks (at most %d ranks)", LRCN_P2P_MAX_RANKS);
  if (h->comm && (h->rank != rank || h->nranks != nranks)) return fail(LRCN_ERR_ARG, "rank/nranks differ from lrcn_comm_init");
  if (h->p2p_ready) return fail(LRCN_ERR_ARG, "peer memory already imported");
  CK(cudaSetDevice(h->cfg.device));
  P2PPeers pe{};
  pe.nranks = nranks; pe.rank = rank;
  for (int p = 0; p < nranks; p++) {
    P2PBlob b;
    memcpy(&b, blobs + (size_t)p * LRCN_P2P_BLOB_BYTES, sizeof b);
    if (b.magic != 0x4C524350 || b.arena_floats != h->P) return fail(LRCN_ERR_ARG, "blob %d does not describe a handle of this model", p);
    if (p == rank) { pe.g[p] = h->g; pe.w[p] = h->w; pe.ctl[p] = h->p2p_ctl; h->peer_m[p] = h->m; h->peer_v[p] = h->v; h->peer_stage[p] = h->stage; continue; }
    void* q[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    const cudaIpcMemHandle_t hs[6] = {b.g, b.ctl, b.w, b.m, b.v, b.stage};
    for (int k = 0; k < 6; k++) {
      cudaError_t e = cudaIpcOpenMemHandle(&q[k], hs[k], cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess)
        return fail(LRCN_ERR_CUDA, "cudaIpcOpenMemHandle(rank %d, device %d) -> %s (peer access over NVLink required)", p, b.device, cudaGetErrorString(e));
      h->p2p_opened[6 * p + k] = q[k];
    }
    pe.g[p] = (float*)q[0]; pe.ctl[p] = (P2PCtl*)q[1]; pe.w[p] = (float*)q[2]; h->peer_m[p] = (float*)q[3]; h->peer_v[p] = (float*)q[4];
    h->peer_stage[p] = (float*)q[5];
    if (getenv("LRCN_P2P_DEBUG")) fprintf(stderr, "[lrcn p2p] rank %d maps rank %d: g %p ctl %p w %p m %p v %p\n", rank, p, q[0], q[1], q[2], q[3], q[4]);
  }
  h->peers = pe;
  h->rank = rank; h->nranks = nranks;
  h->dp_epoch = 0;  // the fused exchange's flags / counters count the group's data-parallel steps: start them together
  CK(cudaMemset(h->stage + h->P + 1024, 0, (DP_XCTL_FLOATS + 2 * h->ll_floats) * 4));
  h->p2p_ready = true;
  return LRCN_OK;
}

// ------------------------------------------------------------------------------------------ measurement
static int s_sync(lrcn_handle* h) {
  if (!h) return fail(LRCN_ERR_ARG, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->comm_stream));
  return sync_stream(h);
}
static int s_timer_start(lrcn_handle* h) {
  if (!h) return fail(LRCN_ERR_ARG, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventRecord(h->ev0, h->stream));
  return LRCN_OK;
}
static int s_timer_stop(lrcn_handle* h, float* ms) {
  if (!h || !ms) return fail(LRCN_ERR_ARG, "null");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventRecord(h->ev1, h->stream));
  CK(cudaEventSynchronize(h->ev1));
  CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  return LRCN_OK;
}
static int s_kernel_launches(lrcn_handle* h, int64_t* n) {
  if (!h || !n) return fail(LRCN_ERR_ARG, "null");
  *n = h->counter.n;
  return LRCN_OK;
}
static int s_get_trace(lrcn_handle* h, uint64_t* out, int64_t n) {
  if (!h || !out || n <= 0 || n > 2048) return fail(LRCN_ERR_ARG, "bad argument");
  if (!h->d_trace) return fail(LRCN_ERR_STATE, "create the handle with LRCN_SEQ_TRACE=1 in the environment");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaMemcpy(out, h->d_trace, (size_t)n * 8, cudaMemcpyDeviceToHost));
  return LRCN_OK;
}
static int s_flush_l2(lrcn_handle* h) {
  if (!h) return fail(LRCN_ERR_ARG, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  fill_l2_scratch(h->stream, h->l2_scratch, h->l2_n, 0.f);
  return LRCN_OK;
}

static int s_time_kernel(lrcn_handle* h, const char* name, int reps, float* avg_ms, double* algo_bytes, double* algo_flops) {
  if (!h || !name || reps < 1 || !avg_ms) return fail(LRCN_ERR_ARG, "bad argument");
  CK(cudaSetDevice(h->cfg.device));
  g_counter = &h->counter;
  const int B = h->last_B > 0 ? h->last_B : h->cfg.max_batch, l = h->last_l > 0 ? h->last_l : h->cfg.max_len;
  const int T = l + 1, R = T * B;
  const Workspace& o = h->o;
  double bytes = 0, flops = 0;
  float total = 0.f;
  try {
    for (int i = 0; i < reps; i++) {
      fill_l2_scratch(h->stream, h->l2_scratch, h->l2_n, 0.f);  // evict L2 between timed launches
      CK(cudaEventRecord(h->ev0, h->stream));
      if (!strcmp(name, "adam")) {
        // algorithmic traffic: read w,g,m,v + write w,m,v = 28 B/param (+4 B/param of bf16 shadows in bf16x3 mode)
        enqueue_adam(h);
        bytes = (double)h->P * (h->bf16mode ? 32.0 : 28.0);
      } else if (!strcmp(name, "vocab_gemm")) {
        gemm(h, true, true, R, h->V, h->H2, WS(h, o.h2) + (size_t)B * h->H2, h->H2, Wp(h, 8), h->H2, WS(h, o.logits), h->ldV, false, Wp(h, 9));
        flops = 2.0 * R * h->V * h->H2;
        bytes = 4.0 * ((double)R * h->H2 + (double)h->V * h->H2 + (double)R * h->V);
      } else if (!strcmp(name, "gate_gemm")) {
        gemm(h, true, true, R, 4 * h->H1, h->E, WS(h, o.Eall), h->E, Wp(h, 1), h->E + h->H1, WS(h, o.acts1), 4 * h->H1, false, Wp(h, 2));
        flops = 2.0 * R * 4 * h->H1 * h->E;
        bytes = 4.0 * ((double)R * h->E + 4.0 * h->H1 * h->E + (double)R * 4 * h->H1);
      } else if (!strcmp(name, "lstm_bwd") || !strcmp(name, "lstm_fwd")) {
        // the layer-2 sequence kernel of the last step shape, alone: T-1 dependent recurrent steps (latency bound).  The buffers
        // hold whatever the last step left (timing is data independent); the grid-barrier counters must be zero on entry.
        CK(cudaMemsetAsync(h->d_counters, 0, 256 * sizeof(unsigned int), h->stream));
        CK(cudaEventRecord(h->ev0, h->stream));
        const int H = h->H2;
        if (!strcmp(name, "lstm_fwd")) lstm_layer_fwd(h, 2, T, B, WS(h, o.acts2), WS(h, o.h2), WS(h, o.c2));
        else lstm_layer_bwd(h, 2, T, B, WS(h, o.acts2), WS(h, o.c2), WS(h, o.dh2), WS(h, o.dhrec2), WS(h, o.dc2), Gp(h, 4));
        flops = 2.0 * B * 4.0 * H * H * (T - 1);
        bytes = 0;
      } else if (!strcmp(name, "gather")) {
        gather_embed(h->stream, Wp(h, 7), h->d_tok_in, R, h->E, WS(h, o.Eall), h->d_sc, false);
        bytes = 2.0 * 4.0 * R * h->E;
      } else if (!strcmp(name, "softmax_ce")) {
        bool fused = false;
        if (h->bf16mode)  // what the training step runs: read logits, write the bf16 hi/lo split of dA, dbout folded in
          fused = softmax_ce_fused(h->stream, WS(h, o.logits), h->ldV, R, h->V, h->d_tok_tgt, WS(h, o.rowlp), h->d_sc, SH(h, WS(h, o.logits)).hi,
                                   SH(h, WS(h, o.logits)).lo, WS(h, o.colpart), COLPART_ROWS, Gp(h, 9), nullptr, nullptr);
        if (!fused)
          softmax_ce(h->stream, WS(h, o.logits), h->ldV, R, h->V, h->d_tok_tgt, WS(h, o.rowlp), h->d_sc, true, SH(h, WS(h, o.logits)).hi, SH(h, WS(h, o.logits)).lo);
        bytes = 8.0 * R * h->V;  // read logits (4 B), write dA (fp32, or its bf16 hi/lo split: 4 B)
      } else {
        return fail(LRCN_ERR_ARG, "unknown kernel family '%s'", name);
      }
      CK(cudaEventRecord(h->ev1, h->stream));
      CK(cudaEventSynchronize(h->ev1));
      float ms;
      CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
      total += ms;
    }
  } catch (GemmFail& f) {
    return fail(LRCN_ERR_CUDA, "%s", f.msg.c_str());
  }
  *avg_ms = total / reps;
  if (algo_bytes) *algo_bytes = bytes;
  if (algo_flops) *algo_flops = flops;
  return LRCN_OK;
}

// ------------------------------------------------------------------------------------------ ABI wrappers
// Every exported call: argument check, sticky-failure check, dispatch (one GPU, or the members of a single-process group),
// and -- through ApiGuard -- promotion of a CUDA / NCCL failure to the handle's sticky state.
#include <thread>

#include <nvtx3/nvToolsExt.h>

// LRCN_NVTX=1: every ABI call is an NVTX range named after the entry point (header-only NVTX3: a no-op unless a tool is attached;
// `ncu --nvtx --nvtx-include "lrcn_train_step/"` then profiles exactly one call's kernels)
static const bool g_nvtx = getenv("LRCN_NVTX") != nullptr;
struct ApiGuard {
  lrcn_handle* h;
  bool pushed = false;
  explicit ApiGuard(lrcn_handle* h_, const char* name) : h(h_) {
    g_last_code = 0;
    if (g_nvtx) { nvtxRangePushA(name); pushed = true; }
  }
  ~ApiGuard() {
    if (pushed) nvtxRangePop();
    if (h && !h->sticky_code && (g_last_code == LRCN_ERR_CUDA || g_last_code == LRCN_ERR_NCCL)) { h->sticky_code = g_last_code; h->sticky_msg = g_err; }
  }
};
#define ENTER(h)                                                                                               \
  if (!(h)) return fail(LRCN_ERR_ARG, "null handle");                                                          \
  if ((h)->sticky_code) return fail((h)->sticky_code, "handle failed earlier and is unusable: %s", (h)->sticky_msg.c_str()); \
  ApiGuard guard_(const_cast<lrcn_handle*>(h), __func__)
static inline bool is_group(const lrcn_handle* h) { return !h->members.empty(); }
#define FOR_ALL(h, call)                                       \
  do {                                                         \
    for (lrcn_handle* m : (h)->members) { int rc_ = (call); if (rc_) return rc_; } \
    return LRCN_OK;                                            \
  } while (0)

// rows [off, off+b) of member i when a global batch of B rows is split over N members (sizes differ by at most one)
static inline void shard_rows(int B, int N, int i, int* off, int* b) {
  const int q = B / N, r = B % N;
  *b = q + (i < r ? 1 : 0);
  *off = i * q + (i < r ? i : r);
}
struct ShardBuf { std::vector<int64_t> tok; };
static const int64_t* shard_tokens(const int64_t* tokens, int l, int B, int off, int b, ShardBuf& buf) {
  if (!tokens || l == 0) return tokens;
  buf.tok.resize((size_t)l * b);
  for (int t = 0; t < l; t++) memcpy(buf.tok.data() + (size_t)t * b, tokens + (size_t)t * B + off, (size_t)b * sizeof(int64_t));
  return buf.tok.data();
}

extern "C" int lrcn_destroy(lrcn_handle* h) { return s_destroy(h); }
extern "C" int lrcn_param_shape(const lrcn_handle* h, int idx, int64_t* rows, int64_t* cols) {
  ENTER(h);
  return s_param_shape(is_group(h) ? h->members[0] : h, idx, rows, cols);
}
extern "C" int lrcn_set_param(lrcn_handle* h, int idx, const float* p, int64_t rows, int64_t cols) {
  ENTER(h);
  if (is_group(h)) FOR_ALL(h, s_set_param(m, idx, p, rows, cols));
  return s_set_param(h, idx, p, rows, cols);
}
extern "C" int lrcn_get_param(lrcn_handle* h, int idx, float* p, int64_t rows, int64_t cols) {
  ENTER(h);
  return s_get_param(is_group(h) ? h->members[0] : h, idx, p, rows, cols);
}
extern "C" int lrcn_get_grad(lrcn_handle* h, int idx, float* p, int64_t rows, int64_t cols) {
  ENTER(h);
  return s_get_grad(is_group(h) ? h->members[0] : h, idx, p, rows, cols);
}
extern "C" int lrcn_get_adam_state(lrcn_handle* h, int idx, int which, float* p, int64_t rows, int64_t cols) {
  ENTER(h);
  return s_get_adam_state(is_group(h) ? h->members[0] : h, idx, which, p, rows, cols);
}
extern "C" int lrcn_set_adam_state(lrcn_handle* h, int idx, int which, const float* p, int64_t rows, int64_t cols) {
  ENTER(h);
  if (is_group(h)) FOR_ALL(h, s_set_adam_state(m, idx, which, p, rows, cols));
  return s_set_adam_state(h, idx, which, p, rows, cols);
}
extern "C" int lrcn_get_adam_step(lrcn_handle* h, int64_t* t) {
  ENTER(h);
  return s_get_adam_step(is_group(h) ? h->members[0] : h, t);
}
extern "C" int lrcn_set_adam_step(lrcn_handle* h, int64_t t) {
  ENTER(h);
  if (is_group(h)) FOR_ALL(h, s_set_adam_step(m, t));
  return s_set_adam_step(h, t);
}
extern "C" int lrcn_load_features(lrcn_handle* h, int split, const int64_t* ids, const float* feats, int64_t n) {
  ENTER(h);
  if (is_group(h)) FOR_ALL(h, s_load_features(m, split, ids, feats, n));  // replicated: 0.5 GB (Flickr30k) / 2 GB (COCO) per GPU
  return s_load_features(h, split, ids, feats, n);
}

// forward / gradient / train step on a global batch, sharded by rows over the members of a group (SURVEY 8e)
static int group_step(lrcn_handle* g, int mode, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B, float pdrop, uint64_t seed,
                      double* loss_or_sum, int64_t* count_out) {
  const int N = (int)g->members.size();
  if (!image_ids || (!tokens && l > 0)) return fail(LRCN_ERR_ARG, "null argument");
  if (B <= 0 || B > g->cfg.max_batch) return fail(LRCN_ERR_ARG, "B=%d outside [1,%d]", B, g->cfg.max_batch);
  if (mode > 0 && B < N) return fail(LRCN_ERR_ARG, "a training batch of %d rows cannot be split over %d GPUs", B, N);
  std::vector<ShardBuf> bufs(N);
  // stage every member first (a bad token / unknown image id fails the call before anything is launched), then launch all
  for (int i = 0; i < N; i++) {
    int off, b;
    shard_rows(B, N, i, &off, &b);
    if (b == 0) continue;
    lrcn_handle* m = g->members[i];
    int rc = stage_current(m, split, image_ids + off, shard_tokens(tokens, l, B, off, b, bufs[i]), l, b);
    if (rc) return rc;
  }
  for (int i = 0; i < N; i++) {
    int off, b;
    shard_rows(B, N, i, &off, &b);
    if (b == 0) continue;
    lrcn_handle* m = g->members[i];
    m->global_B = B;
    int rc = run_step(m, split, b, l, pdrop, seed, mode);
    if (rc) return rc;
  }
  double total = 0.0;
  for (int i = 0; i < N; i++) {
    int off, b;
    shard_rows(B, N, i, &off, &b);
    if (b == 0) continue;
    double t;
    int rc = finish_loss(g->members[i], b, l, &t);  // synchronises member i
    if (rc) return rc;
    if (mode == 0 || i == 0) total = mode == 0 ? total + t : t;  // training: the exchange kernel already summed the loss over the members
  }
  if (mode == 0) {
    if (loss_or_sum) *loss_or_sum = total;
    if (count_out) *count_out = (int64_t)B * (l + 1);
  } else if (loss_or_sum) {
    *loss_or_sum = -total / ((double)B * (l + 1));
  }
  g->last_B = B; g->last_l = l;
  return LRCN_OK;
}

extern "C" int lrcn_loss(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B, double* sum_logp_out,
                         int64_t* count_out) {
  ENTER(h);
  if (is_group(h)) return group_step(h, 0, split, image_ids, tokens, l, B, 0.f, 0, sum_logp_out, count_out);
  return s_loss(h, split, image_ids, tokens, l, B, sum_logp_out, count_out);
}
extern "C" int lrcn_grad(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B, float pdrop, uint64_t seed,
                         double* loss_out) {
  ENTER(h);
  if (pdrop < 0.f || pdrop >= 1.f) return fail(LRCN_ERR_ARG, "pdrop must be in [0,1)");
  if (is_group(h)) return group_step(h, 1, split, image_ids, tokens, l, B, pdrop, seed, loss_out, nullptr);
  return s_grad(h, split, image_ids, tokens, l, B, pdrop, seed, loss_out);
}
extern "C" int lrcn_train_step(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B, float pdrop,
                               uint64_t seed, double* loss_out) {
  ENTER(h);
  if (pdrop < 0.f || pdrop >= 1.f) return fail(LRCN_ERR_ARG, "pdrop must be in [0,1)");
  if (is_group(h)) return group_step(h, 2, split, image_ids, tokens, l, B, pdrop, seed, loss_out, nullptr);
  return s_train_step(h, split, image_ids, tokens, l, B, pdrop, seed, loss_out);
}
extern "C" int lrcn_adam_update(lrcn_handle* h) {
  ENTER(h);
  if (is_group(h)) {
    // every member holds the all-reduced gradient after lrcn_grad; make the Adam state whole everywhere first (all idle here)
    for (lrcn_handle* m : h->members) if (m->adam_sharded) { int rc = gather_shards(m, true, false); if (rc) return rc; }
    FOR_ALL(h, s_adam_update(m));
  }
  return s_adam_update(h);
}
extern "C" int lrcn_get_token_logps(lrcn_handle* h, float* out, int64_t n) {
  ENTER(h);
  if (!is_group(h)) return s_get_token_logps(h, out, n);
  if (!out) return fail(LRCN_ERR_ARG, "null");
  const int B = h->last_B, T = h->last_l + 1, N = (int)h->members.size();
  if (n != (int64_t)B * T) return fail(LRCN_ERR_ARG, "expected %lld values", (long long)B * T);
  std::vector<float> tmp;
  for (int i = 0; i < N; i++) {
    int off, b;
    shard_rows(B, N, i, &off, &b);
    if (b == 0) continue;
    tmp.resize((size_t)b * T);
    int rc = s_get_token_logps(h->members[i], tmp.data(), (int64_t)b * T);
    if (rc) return rc;
    for (int t = 0; t < T; t++) memcpy(out + (size_t)t * B + off, tmp.data() + (size_t)t * b, (size_t)b * sizeof(float));
  }
  return LRCN_OK;
}
extern "C" int lrcn_stage_batch(lrcn_handle* h, int slot, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B) {
  ENTER(h);
  if (!is_group(h)) return s_stage_batch(h, slot, split, image_ids, tokens, l, B);
  const int N = (int)h->members.size();
  if (!image_ids || (!tokens && l > 0)) return fail(LRCN_ERR_ARG, "null argument");
  if (B < N || B > h->cfg.max_batch) return fail(LRCN_ERR_ARG, "B=%d outside [%d,%d]", B, N, h->cfg.max_batch);
  if (slot < 0 || slot >= 64) return fail(LRCN_ERR_ARG, "slot outside [0,64)");
  ShardBuf buf;
  for (int i = 0; i < N; i++) {
    int off, b;
    shard_rows(B, N, i, &off, &b);
    int rc = s_stage_batch(h->members[i], slot, split, image_ids + off, shard_tokens(tokens, l, B, off, b, buf), l, b);
    if (rc) return rc;
  }
  h->slots[slot].B = B; h->slots[slot].l = l;
  return LRCN_OK;
}
extern "C" int lrcn_train_step_staged(lrcn_handle* h, int slot, float pdrop, uint64_t seed, double* loss_out) {
  ENTER(h);
  if (!is_group(h)) return s_train_step_staged(h, slot, pdrop, seed, loss_out);
  if (slot < 0 || slot >= 64 || h->slots[slot].B == 0) return fail(LRCN_ERR_ARG, "slot %d not staged", slot);
  for (lrcn_handle* m : h->members) {
    m->global_B = h->slots[slot].B;
    int rc = s_train_step_staged(m, slot, pdrop, seed, m == h->members[0] ? loss_out : nullptr);
    if (rc) return rc;
  }
  return LRCN_OK;
}

extern "C" int lrcn_beam_search(lrcn_handle* h, int split, const int64_t* image_ids, int64_t n, int K, int nword, int64_t* tokens_out,
                                int32_t* len_out, float* prob_out, float* logp_out) {
  ENTER(h);
  if (!is_group(h)) return s_beam_search(h, split, image_ids, n, K, nword, tokens_out, len_out, prob_out, logp_out);
  // images are independent (lrcn.jl:152-155 loops them serially): contiguous slices, one worker thread per GPU, no collective
  if (!image_ids || !tokens_out || !len_out || !prob_out || n <= 0) return fail(LRCN_ERR_ARG, "bad argument to lrcn_beam_search");
  if (nword < 1 || nword + 2 > 64) return fail(LRCN_ERR_ARG, "nword %d outside [1,62]", nword);
  const int N = (int)h->members.size();
  const int maxlen = nword + 2;
  std::vector<int> rcs(N, LRCN_OK);
  std::vector<std::string> msgs(N);
  std::vector<std::thread> th;
  for (int i = 0; i < N; i++) {
    const int64_t lo = n * i / N, hi = n * (i + 1) / N;
    if (hi <= lo) continue;
    th.emplace_back([&, i, lo, hi] {
      rcs[i] = s_beam_search(h->members[i], split, image_ids + lo, hi - lo, K, nword, tokens_out + lo * maxlen, len_out + lo, prob_out + lo,
                             logp_out ? logp_out + lo * (maxlen - 1) : nullptr);
      if (rcs[i]) msgs[i] = g_err;  // thread-local message of the worker
    });
  }
  for (auto& t : th) t.join();
  for (int i = 0; i < N; i++) if (rcs[i]) return fail(rcs[i], "GPU %d: %s", h->members[i]->cfg.device, msgs[i].c_str());
  return LRCN_OK;
}

// ---- VGG-16 fc7 producer (row f-4, cnn_sm100.cu)
extern "C" int lrcn_set_cnn_param(lrcn_handle* h, int layer, int which, const float* data, const int64_t dims[4]) {
  ENTER(h);
  if (is_group(h)) FOR_ALL(h, cnn_set_param(m, layer, which, data, dims));
  return cnn_set_param(h, layer, which, data, dims);
}
extern "C" int lrcn_get_cnn_param(lrcn_handle* h, int layer, int which, float* data, const int64_t dims[4]) {
  ENTER(h);
  return cnn_get_param(is_group(h) ? h->members[0] : h, layer, which, data, dims);
}
extern "C" int lrcn_extract_features(lrcn_handle* h, const float* images, int64_t n, int flags, float* feats_out) {
  ENTER(h);
  if (!is_group(h)) return cnn_extract(h, images, n, flags, feats_out);
  // images are independent: contiguous slices, one worker thread per GPU, each writing its rows of feats_out
  if (!images || !feats_out || n <= 0) return fail(LRCN_ERR_ARG, "bad argument to lrcn_extract_features");
  const int N = (int)h->members.size();
  const int64_t img = (int64_t)3 * LRCN_CNN_IMAGE * LRCN_CNN_IMAGE;
  std::vector<int> rcs(N, LRCN_OK);
  std::vector<std::string> msgs(N);
  std::vector<std::thread> th;
  for (int i = 0; i < N; i++) {
    const int64_t lo = n * i / N, hi = n * (i + 1) / N;
    if (hi <= lo) continue;
    th.emplace_back([&, i, lo, hi] {
      rcs[i] = cnn_extract(h->members[i], images + lo * img, hi - lo, flags, feats_out + lo * LRCN_F_CNN);
      if (rcs[i]) msgs[i] = g_err;
    });
  }
  for (auto& t : th) t.join();
  for (int i = 0; i < N; i++) if (rcs[i]) return fail(rcs[i], "GPU %d: %s", h->members[i]->cfg.device, msgs[i].c_str());
  return LRCN_OK;
}

extern "C" int lrcn_comm_init(lrcn_handle* h, const char id[LRCN_COMM_ID_BYTES], int rank, int nranks) {
  ENTER(h);
  if (is_group(h)) return fail(LRCN_ERR_STATE, "this handle already drives %d GPUs by itself (cfg.n_gpus)", (int)h->members.size());
  return s_comm_init(h, id, rank, nranks);
}
extern "C" int lrcn_p2p_export(lrcn_handle* h, char blob[LRCN_P2P_BLOB_BYTES]) {
  ENTER(h);
  if (is_group(h)) return fail(LRCN_ERR_STATE, "this handle already drives %d GPUs by itself (cfg.n_gpus)", (int)h->members.size());
  return s_p2p_export(h, blob);
}
extern "C" int lrcn_p2p_import(lrcn_handle* h, const char* blobs, int rank, int nranks) {
  ENTER(h);
  if (is_group(h)) return fail(LRCN_ERR_STATE, "this handle already drives %d GPUs by itself (cfg.n_gpus)", (int)h->members.size());
  return s_p2p_import(h, blobs, rank, nranks);
}
extern "C" int lrcn_sync(lrcn_handle* h) {
  ENTER(h);
  if (is_group(h)) FOR_ALL(h, s_sync(m));
  return s_sync(h);
}
extern "C" int lrcn_timer_start(lrcn_handle* h) {
  ENTER(h);
  return s_timer_start(is_group(h) ? h->members[0] : h);
}
extern "C" int lrcn_timer_stop(lrcn_handle* h, float* ms) {
  ENTER(h);
  if (!is_group(h)) return s_timer_stop(h, ms);
  int rc = s_timer_stop(h->members[0], ms);  // the steps of all members end together (cross-GPU barrier inside the step)
  if (rc) return rc;
  FOR_ALL(h, s_sync(m));
}
extern "C" int lrcn_kernel_launches(lrcn_handle* h, int64_t* n) {
  ENTER(h);
  if (!is_group(h)) return s_kernel_launches(h, n);
  if (!n) return fail(LRCN_ERR_ARG, "null");
  *n = 0;
  for (lrcn_handle* m : h->members) *n += m->counter.n;
  return LRCN_OK;
}
extern "C" int lrcn_get_trace(lrcn_handle* h, uint64_t* out, int64_t n) {
  ENTER(h);
  return s_get_trace(is_group(h) ? h->members[0] : h, out, n);
}
extern "C" int lrcn_flush_l2(lrcn_handle* h) {
  ENTER(h);
  if (is_group(h)) FOR_ALL(h, s_flush_l2(m));
  return s_flush_l2(h);
}
extern "C" int lrcn_time_kernel(lrcn_handle* h, const char* name, int reps, float* avg_ms, double* algo_bytes, double* algo_flops) {
  ENTER(h);
  return s_time_kernel(is_group(h) ? h->members[0] : h, name, reps, avg_ms, algo_bytes, algo_flops);
}

// ------------------------------------------------------------------------------------------ epoch-level training (SURVEY 8 row f-1)
// The hot loop of train1 (lrcn.jl:351-396) for one epoch in ONE call: the epoch's token matrix and image ids are uploaded
// once, image ids are resolved to feature-table rows on the device, and every batch is staged by a small kernel from the
// resident data (inputs [bos, w..], targets [w.., eos], feature rows: lrcn.jl:369-376,556,563-577) right before its step
// graph -- no per-step host marshalling, H2D copy or synchronisation.  Batches longer than max_len are skipped like
// lrcn.jl:353 skips l > 28.  ldB / col0: this handle's columns of a wider (global) batch in the single-process group mode.
static int epoch_upload(lrcn_handle* h, int split, const int64_t* sequence, int64_t n_rows, const int64_t* input_ids, int64_t n_batches, int ldB) {
  CK(cudaSetDevice(h->cfg.device));
  if (split < 0 || split > 1 || !h->tab[split].d) return fail(LRCN_ERR_STATE, "no features loaded for split %d", split);
  const size_t ns = (size_t)n_rows * ldB, ni = (size_t)n_batches * ldB;
  if (ns > h->ep_seq_cap) { if (h->ep_seq) cudaFree(h->ep_seq); h->ep_seq = nullptr; CK(cudaMalloc(&h->ep_seq, ns * 8)); h->ep_seq_cap = ns; }
  if (ni > h->ep_ids_cap) {
    if (h->ep_ids) cudaFree(h->ep_ids);
    if (h->ep_rows) cudaFree(h->ep_rows);
    h->ep_ids = nullptr; h->ep_rows = nullptr;
    CK(cudaMalloc(&h->ep_ids, ni * 8)); CK(cudaMalloc(&h->ep_rows, ni * 4)); h->ep_ids_cap = ni;
  }
  if (!h->ep_err) { CK(cudaMalloc(&h->ep_err, 4)); }
  CK(cudaMemsetAsync(h->ep_err, 0, 4, h->stream));
  CK(cudaMemcpyAsync(h->ep_seq, sequence, ns * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->ep_ids, input_ids, ni * 8, cudaMemcpyHostToDevice, h->stream));
  g_counter = &h->counter;
  epoch_lookup_rows(h->stream, h->ep_ids, ni, h->tab[split].d_ids, h->tab[split].d_rowof, (int)h->tab[split].map.size(), h->ep_rows, h->ep_err);
  return LRCN_OK;
}
static int epoch_check(lrcn_handle* h) {
  int err = 0;
  CK(cudaMemcpyAsync(&err, h->ep_err, 4, cudaMemcpyDeviceToHost, h->stream));
  int rc = sync_stream(h);
  if (rc) return rc;
  if (err == 1) return fail(LRCN_ERR_MISSING, "missing features for an image id of the epoch (lrcn.jl:602-605)");
  if (err == 2) return fail(LRCN_ERR_ARG, "a token of the epoch lies outside [1,%d]", h->V);
  return LRCN_OK;
}

// mode 2: train steps (losses_out = mean NLL per step); mode 0: forward only (losses_out = SUM of log-probs per step, count_out = tokens)
static int epoch_run(lrcn_handle* h, int mode, int split, const int64_t* sequence, int64_t n_rows, const int64_t* input_ids, const int64_t* lengths,
                     int64_t n_batches, int B, const int64_t* order, int64_t n_order, float pdrop, uint64_t seed, double* losses_out,
                     int64_t* steps_out, int64_t* count_out) {
  if (!sequence || !input_ids || !lengths || n_rows < 0 || n_batches <= 0 || B <= 0 || (n_order > 0 && !order))
    return fail(LRCN_ERR_ARG, "bad argument to lrcn_train_epoch / lrcn_loss_epoch");
  if (pdrop < 0.f || pdrop >= 1.f) return fail(LRCN_ERR_ARG, "pdrop must be in [0,1)");
  std::vector<lrcn_handle*> hs;
  if (is_group(h)) hs = h->members; else hs.push_back(h);
  const int N = (int)hs.size();
  const int maxB = h->cfg.max_batch, max_len = h->cfg.max_len;
  if (B > maxB || B < N) return fail(LRCN_ERR_ARG, "B=%d outside [%d,%d]", B, N, maxB);
  int64_t count = 0;
  int last_l_run = -1;
  // start row of every batch in `sequence` (prefix sum of the lengths: lrcn.jl:336-342)
  std::vector<int64_t> start((size_t)n_batches + 1, 0);
  for (int64_t b = 0; b < n_batches; b++) {
    if (lengths[b] < 0) return fail(LRCN_ERR_ARG, "negative caption length");
    start[b + 1] = start[b] + lengths[b];
  }
  if (start[n_batches] > n_rows) return fail(LRCN_ERR_ARG, "lengths sum to %lld rows, sequence has %lld", (long long)start[n_batches], (long long)n_rows);
  int rc;
  for (lrcn_handle* m : hs) { rc = epoch_upload(m, split, sequence, n_rows, input_ids, n_batches, B); if (rc) return rc; }
  for (lrcn_handle* m : hs) { rc = epoch_check(m); if (rc) return rc; }  // unknown ids fail the call before any step runs (like the per-step call)
  const int64_t n_run_max = n_order > 0 ? n_order : n_batches;
  for (lrcn_handle* m : hs)
    if ((size_t)n_run_max > m->ep_loss_cap) { CK(cudaSetDevice(m->cfg.device)); if (m->ep_loss) cudaFree(m->ep_loss); m->ep_loss = nullptr; CK(cudaMalloc(&m->ep_loss, (size_t)n_run_max * 8)); m->ep_loss_cap = (size_t)n_run_max; }
  int64_t steps = 0;
  std::vector<double> denom;
  for (int64_t k = 0; k < n_run_max; k++) {
    const int64_t b = n_order > 0 ? order[k] : k;
    if (b < 0 || b >= n_batches) return fail(LRCN_ERR_ARG, "order[%lld] = %lld outside [0,%lld)", (long long)k, (long long)b, (long long)n_batches);
    const int l = (int)lengths[b];
    if (l > max_len) continue;  // lrcn.jl:353: batches of captions longer than 28 are skipped
    for (int i = 0; i < N; i++) {
      lrcn_handle* m = hs[i];
      int off = 0, bw = B;
      if (N > 1) shard_rows(B, N, i, &off, &bw);
      CK(cudaSetDevice(m->cfg.device));
      g_counter = &m->counter;
      epoch_stage_batch(m->stream, m->ep_seq, (size_t)start[b], l, B, off, bw, m->V, m->ep_rows, (size_t)b * B, m->d_tok_in, m->d_tok_tgt, m->d_rows, m->ep_err);
      m->global_B = N > 1 ? B : 0;
      rc = run_step(m, split, bw, l, pdrop, seed + (uint64_t)steps, mode);
      if (rc) return rc;
      CK(cudaMemcpyAsync(m->ep_loss + steps, m->loss_is_total ? m->d_loss_total : m->d_loss, 8, cudaMemcpyDeviceToDevice, m->stream));
    }
    denom.push_back((double)B * (l + 1) * (N > 1 ? 1 : hs[0]->nranks));
    count += (int64_t)B * (l + 1);
    last_l_run = l;
    steps++;
  }
  for (lrcn_handle* m : hs) { rc = epoch_check(m); if (rc) return rc; }  // synchronises; out-of-range tokens surface here
  if (losses_out && steps > 0) {
    std::vector<double> tot((size_t)steps);
    // training: the exchange kernel already summed the loss over the members; forward only: every member holds its columns' sum
    for (int i = 0; i < (mode == 0 ? N : 1); i++) {
      CK(cudaSetDevice(hs[i]->cfg.device));
      CK(cudaMemcpy(tot.data(), hs[i]->ep_loss, (size_t)steps * 8, cudaMemcpyDeviceToHost));
      for (int64_t k = 0; k < steps; k++) losses_out[k] = mode == 0 ? (i == 0 ? tot[k] : losses_out[k] + tot[k]) : -tot[k] / denom[k];
    }
  }
  if (steps_out) *steps_out = steps;
  if (count_out) *count_out = count;
  if (N > 1 && last_l_run >= 0) { h->last_B = B; h->last_l = last_l_run; }
  return LRCN_OK;
}
extern "C" int lrcn_train_epoch(lrcn_handle* h, int split, const int64_t* sequence, int64_t n_rows, const int64_t* input_ids, const int64_t* lengths,
                                int64_t n_batches, int B, const int64_t* order, int64_t n_order, float pdrop, uint64_t seed, double* losses_out,
                                int64_t* steps_out) {
  ENTER(h);
  return epoch_run(h, 2, split, sequence, n_rows, input_ids, lengths, n_batches, B, order, n_order, pdrop, seed, losses_out, steps_out, nullptr);
}
// average_loss (lrcn.jl:407-486) for a whole split in one call: forward only, pdrop = 0, batches in natural order
extern "C" int lrcn_loss_epoch(lrcn_handle* h, int split, const int64_t* sequence, int64_t n_rows, const int64_t* input_ids, const int64_t* lengths,
                               int64_t n_batches, int B, double* sum_logp_out, int64_t* count_out) {
  ENTER(h);
  if (n_batches <= 0) return fail(LRCN_ERR_ARG, "bad argument to lrcn_loss_epoch");
  std::vector<double> sums((size_t)n_batches, 0.0);
  int64_t steps = 0;
  int rc = epoch_run(h, 0, split, sequence, n_rows, input_ids, lengths, n_batches, B, nullptr, 0, 0.f, 0, sums.data(), &steps, count_out);
  if (rc) return rc;
  double s = 0.0;
  for (int64_t k = 0; k < steps; k++) s += sums[k];
  if (sum_logp_out) *sum_logp_out = s;
  return LRCN_OK;
}

// ------------------------------------------------------------------------------------------ checkpoint (SURVEY 8 row f-2)
// The reference saves `model` (Any[9] of Float32 matrices) and `vocab` (Dict) through JLD/HDF5 (lrcn.jl:88-93,183-186,
// 228-231,775-781).  No HDF5 exists in this image, so the library reads and writes a raw little-endian SIDECAR file with the
// same content plus the Adam state the reference never saved (SURVEY 5: resuming otherwise restarts Adam from zero):
//   "LRCNB2CK" | u32 version=1 | u32 flags (1: Adam state present) | i32 E,H1,H2,V | i64 adam_t | i64 aux_bytes
//   9 x { i64 rows, i64 cols, rows*cols float32 column-major }                    -- model[1..9], exactly what JLD holds
//   if flags&1: 9 x m then 9 x v in the same layout                               -- Knet Adam fstm / scndm
//   aux_bytes of caller data (the host writes the vocab Dict as "word\tindex\n" lines, UTF-8)
// julia/lrcn_b200.jl carries a pure-Julia reader/writer of the same file (read_checkpoint / write_checkpoint).
static int ck_write(FILE* f, const void* p, size_t n) { return fwrite(p, 1, n, f) == n ? 0 : 1; }
static int ck_read(FILE* f, void* p, size_t n) { return fread(p, 1, n, f) == n ? 0 : 1; }

extern "C" int lrcn_checkpoint_save(lrcn_handle* h, const char* path, int with_adam, const void* aux, int64_t aux_bytes) {
  ENTER(h);
  if (!path || aux_bytes < 0 || (aux_bytes > 0 && !aux)) return fail(LRCN_ERR_ARG, "bad argument to lrcn_checkpoint_save");
  lrcn_handle* m0 = is_group(h) ? h->members[0] : h;
  FILE* f = fopen(path, "wb");
  if (!f) return fail(LRCN_ERR_ARG, "cannot open %s for writing", path);
  const uint32_t version = 1, flags = with_adam ? 1u : 0u;
  const int32_t dims[4] = {m0->E, m0->H1, m0->H2, m0->V};
  int bad = ck_write(f, "LRCNB2CK", 8) | ck_write(f, &version, 4) | ck_write(f, &flags, 4) | ck_write(f, dims, 16) | ck_write(f, &m0->adam_t, 8) |
            ck_write(f, &aux_bytes, 8);
  std::vector<float> buf;
  int rc = LRCN_OK;
  for (int sect = 0; sect < (with_adam ? 3 : 1) && !bad && !rc; sect++)
    for (int k = 1; k <= 9 && !bad && !rc; k++) {
      const int64_t r = m0->rows[k - 1], c = m0->cols[k - 1];
      buf.resize((size_t)(r * c));
      rc = sect == 0 ? s_get_param(m0, k, buf.data(), r, c) : s_get_adam_state(m0, k, sect - 1, buf.data(), r, c);
      if (!rc) bad = ck_write(f, &r, 8) | ck_write(f, &c, 8) | ck_write(f, buf.data(), buf.size() * 4);
    }
  if (!bad && !rc && aux_bytes > 0) bad = ck_write(f, aux, (size_t)aux_bytes);
  if (fclose(f) != 0) bad = 1;
  if (rc) return rc;
  if (bad) return fail(LRCN_ERR_ARG, "short write to %s", path);
  return LRCN_OK;
}

extern "C" int lrcn_checkpoint_load(lrcn_handle* h, const char* path, int* had_adam, void* aux_out, int64_t aux_cap, int64_t* aux_bytes_out) {
  ENTER(h);
  if (!path) return fail(LRCN_ERR_ARG, "null path");
  lrcn_handle* m0 = is_group(h) ? h->members[0] : h;
  FILE* f = fopen(path, "rb");
  if (!f) return fail(LRCN_ERR_ARG, "cannot open %s", path);
  char magic[8];
  uint32_t version = 0, flags = 0;
  int32_t dims[4];
  int64_t adam_t = 0, aux_bytes = 0;
  int rc = LRCN_OK;
  if (ck_read(f, magic, 8) || memcmp(magic, "LRCNB2CK", 8) || ck_read(f, &version, 4) || version != 1 || ck_read(f, &flags, 4) || ck_read(f, dims, 16) ||
      ck_read(f, &adam_t, 8) || ck_read(f, &aux_bytes, 8) || adam_t < 0 || aux_bytes < 0) {
    fclose(f);
    return fail(LRCN_ERR_ARG, "%s is not an LRCNB2CK version-1 checkpoint", path);
  }
  if (dims[0] != m0->E || dims[1] != m0->H1 || dims[2] != m0->H2 || dims[3] != m0->V) {
    fclose(f);
    return fail(LRCN_ERR_ARG, "checkpoint is for embed %d hidden %d %d vocab %d; this handle has %d / %d %d / %d", dims[0], dims[1], dims[2], dims[3], m0->E,
                m0->H1, m0->H2, m0->V);
  }
  std::vector<float> buf;
  for (int sect = 0; sect < ((flags & 1u) ? 3 : 1) && !rc; sect++)
    for (int k = 1; k <= 9 && !rc; k++) {
      int64_t r = 0, c = 0;
      if (ck_read(f, &r, 8) || ck_read(f, &c, 8) || r != m0->rows[k - 1] || c != m0->cols[k - 1]) { rc = fail(LRCN_ERR_ARG, "%s: matrix %d has the wrong shape", path, k); break; }
      buf.resize((size_t)(r * c));
      if (ck_read(f, buf.data(), buf.size() * 4)) { rc = fail(LRCN_ERR_ARG, "%s is truncated", path); break; }
      if (is_group(h)) {
        for (lrcn_handle* m : h->members) { rc = sect == 0 ? s_set_param(m, k, buf.data(), r, c) : s_set_adam_state(m, k, sect - 1, buf.data(), r, c); if (rc) break; }
      } else {
        rc = sect == 0 ? s_set_param(h, k, buf.data(), r, c) : s_set_adam_state(h, k, sect - 1, buf.data(), r, c);
      }
    }
  if (!rc) {
    if (aux_bytes_out) *aux_bytes_out = aux_bytes;
    if (aux_out && aux_bytes > 0) {
      if (aux_cap < aux_bytes) rc = fail(LRCN_ERR_ARG, "aux buffer of %lld bytes < %lld stored", (long long)aux_cap, (long long)aux_bytes);
      else if (ck_read(f, aux_out, (size_t)aux_bytes)) rc = fail(LRCN_ERR_ARG, "%s is truncated", path);
    }
  }
  fclose(f);
  if (rc) return rc;
  if (had_adam) *had_adam = (flags & 1u) ? 1 : 0;
  if (flags & 1u) {  // resume Adam where it stopped; a model-only file leaves the optimizer as it is (the reference restarts it)
    if (is_group(h)) { for (lrcn_handle* m : h->members) m->adam_t = adam_t; }
    else h->adam_t = adam_t;
  }
  return LRCN_OK;
}
