// lrcn_internal.h -- the handle behind the C ABI (include/lrcn_b200.h), shared by lrcn_api.cu (product) and test_hooks.cu
// (kernel-level test hooks, built only into liblrcn_b200_test.so).
#pragma once
#include "../../include/lrcn_b200.h"
#include "kernels.cuh"

#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <tuple>
#include <unordered_map>
#include <vector>

typedef __nv_bfloat16 bf16;
typedef struct ncclComm* ncclComm_t;

int fail(int code, const char* fmt, ...);  // records the thread-local message of lrcn_last_error() and returns `code`
#define CK(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess) return fail(LRCN_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
  } while (0)

using namespace lrcn;
struct Arena {
  float* f = nullptr; bf16* hi = nullptr; bf16* lo = nullptr;
  size_t cap = 0, used = 0;
  size_t take(size_t n) { size_t o = used; used += (n + 63) / 64 * 64; return o; }
};
struct Table {
  float* d = nullptr; int64_t n = 0;
  std::unordered_map<int64_t, int> map;
  // device-side id -> row lookup (epoch-level calls): ids sorted ascending + the row of each
  long long* d_ids = nullptr; int* d_rowof = nullptr;
};
constexpr int COLPART_ROWS = 296;  // 2 CTAs per SM
struct Slot { int l = 0, B = 0, split = 0; int *tok_in = nullptr, *tok_tgt = nullptr, *rows = nullptr; };
struct Workspace {  // element offsets into the workspace arena
  size_t X, v, dv, Eall, dE, acts1, h1, c1, Z, dZ, acts2, h2, c2, logits, rowlp, dh2, dh1, dhrec1, dc1, dhrec2, dc2, colpart;
  // generation
  size_t gX, gv, ge, gg1, gh1a, gc1a, gh1b, gc1b, gz, gg2, gh2a, gc2a, gh2b, gc2b, glogits, gprob, gcs, gclp, gss, gslp, glpa, glpb, goprob, golp, gxh1, gxh2;
};
struct lrcn_handle {
  lrcn_config cfg;
  int E, H1, H2, C, V, ldV, ldv;
  bool bf16mode;
  cudaStream_t stream = nullptr, comm_stream = nullptr, side_stream = nullptr;  // side: weight prep, concurrent with the step's first kernels
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_zero = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_seg[4] = {nullptr, nullptr, nullptr, nullptr}, ev_comm = nullptr;
  // params
  static constexpr int NBUCKET = 4;   // gradient buckets in backward-readiness order: [Wout,bout | W2,b2,Wf,Wcnn | W1,b1 | Wemb]
  size_t P = 0, off[9], nel[9], bucket_off[NBUCKET + 1];
  int64_t rows[9], cols[9];
  float *w = nullptr, *g = nullptr, *m = nullptr, *v = nullptr;
  bf16 *w_hi = nullptr, *w_lo = nullptr;
  bf16 *wp1_hi = nullptr, *wp1_lo = nullptr, *wp2_hi = nullptr, *wp2_lo = nullptr;  // gate-interleaved recurrent weights (lstm_sm100.cu)
  bf16 *wt1_hi = nullptr, *wt1_lo = nullptr, *wt2_hi = nullptr, *wt2_lo = nullptr;  // transposed recurrent weights for the backward step
  int64_t adam_t = 0;
  // per-tensor gradient clipping (lrcn_set_gclip, kernels.cuh grad_sqnorm): one allocation holding norm[9] (fp64), scale[9],
  // the launch tickets (one per gradient bucket + one for whole-arena launches) and the chunk partial sums; gchunk0[k]: first
  // partial slot of tensor k (model order)
  double gclip = 0.0;
  bool have_grad = false;   // a gradient has been computed (lrcn_grad_norms)
  int gchunk0[9] = {};
  double *d_gnorm = nullptr, *d_gpart = nullptr; float* d_gscale = nullptr; unsigned int* d_gticket = nullptr;
  Table tab[2];
  Arena ws;
  Workspace o;
  int *d_tok_in = nullptr, *d_tok_tgt = nullptr, *d_rows = nullptr;
  // epoch-resident data of lrcn_train_epoch (row f-1: batch staging on the device)
  long long *ep_seq = nullptr, *ep_ids = nullptr; int* ep_rows = nullptr; double* ep_loss = nullptr; int* ep_err = nullptr;
  size_t ep_seq_cap = 0, ep_ids_cap = 0, ep_loss_cap = 0;
  int* h_stage = nullptr;  // pinned: tok_in | tok_tgt | rows
  // step scalars: one device struct (graphs read it through a fixed pointer), fed from a RING of pinned host copies so that
  // the host never rewrites a pinned buffer whose H2D copy has not executed yet (calls that do not synchronise, e.g.
  // lrcn_train_step_staged with loss_out = NULL, can be many steps ahead of the device)
  static constexpr int SC_RING = 16;
  StepScalars *d_sc = nullptr, *h_sc = nullptr;  // h_sc: SC_RING pinned structs
  cudaEvent_t sc_ev[SC_RING] = {};
  bool sc_busy[SC_RING] = {};
  int sc_next = 0;
  // sticky failure state (CUDA / NCCL errors, device-side barrier time-outs): every later call returns it
  int sticky_code = 0;
  std::string sticky_msg;
  // single-process multi-GPU group (cfg.n_gpus > 1): this handle then owns no device memory itself; members[i] is the
  // per-GPU handle of rank i (parent points back).  All API calls dispatch over the members.
  std::vector<lrcn_handle*> members;
  lrcn_handle* parent = nullptr;
  bool peers_direct = false;  // peers.* are direct peer pointers of this process (nothing to cudaIpcClose)
  double *d_loss = nullptr, *h_loss = nullptr;  // d_loss lives inside p2p_ctl (peers read it)
  // peer-memory data parallelism (dp_p2p.cu)
  P2PCtl* p2p_ctl = nullptr;          // exported control block: barrier flags + this rank's loss partial
  double* d_loss_total = nullptr;     // sum over ranks, written by the exchange kernel
  unsigned int* d_epoch = nullptr;    // barrier epoch counter (local)
  P2PPeers peers{};
  bool p2p_ready = false;
  bool loss_is_total = false;       // last step summed the loss over ranks into d_loss_total
  void* p2p_opened[6 * LRCN_P2P_MAX_RANKS] = {};  // IPC mappings to close
  float* peer_m[LRCN_P2P_MAX_RANKS] = {};
  float* peer_v[LRCN_P2P_MAX_RANKS] = {};
  bool adam_sharded = false;          // m, v are current only in each owner's shard (gathered on lrcn_get_adam_state)
  // fused exchange (dp_p2p.cu): staging rows for the gradient chunks the peers push to this rank, followed by the control
  // words (chunk flags, completion counters); and the peers' staging allocations
  float* stage = nullptr;
  float* peer_stage[LRCN_P2P_MAX_RANKS] = {};
  unsigned int dp_epoch = 0;          // data-parallel train steps run since the peer group was formed (the fused exchange's flag value)
  unsigned int* d_counters = nullptr;  // per-m-tile grid-barrier counters of the persistent LSTM kernels
  unsigned long long* d_trace = nullptr;  // LRCN_SEQ_TRACE=1: per-step timeline of the layer-2 forward sequence kernel
  Slot slots[64];
  std::map<std::tuple<int, int, int, int>, cudaGraphExec_t> graphs;
  std::map<std::tuple<int, int, int, int>, long long> graph_launches;
  LaunchCounter counter;
  int last_B = 0, last_l = 0;
  int global_B = 0;  // > 0: rows of the global batch of the current step (set by the single-process group dispatcher)
  bool grad_sharded = false;  // after a sharded train step the summed gradient is current only in each owner's shard
  bool dbout_fused = false;  // set by enqueue_forward: the softmax kernel already produced dbout
  // DP
  ncclComm_t comm = nullptr; int rank = 0, nranks = 1;
  // generation int buffers
  int *g_last = nullptr, *g_ctok = nullptr, *g_stok = nullptr, *g_spar = nullptr, *g_hista = nullptr, *g_histb = nullptr, *g_done = nullptr,
      *g_ndone = nullptr, *g_olen = nullptr, *g_rows = nullptr;
  long long* g_otok = nullptr;
  static constexpr int NSNAP = 4;   // ring of pinned snapshots of the done flags / survivor lists (asynchronous beam-search polling)
  cudaEvent_t ev_snap[NSNAP] = {nullptr, nullptr, nullptr, nullptr}, ev_keep[NSNAP] = {nullptr, nullptr, nullptr, nullptr};
  int* h_keep = nullptr;     // pinned: NSNAP survivor lists
  int* h_ndone = nullptr;    // pinned: [0] = images done so far, [1..] = done flags of the images in flight
  int *g_keep = nullptr, *g_omap = nullptr, *g_omap_s = nullptr;  // compaction: survivors, compacted -> caller index (+ scratch)
  float* l2_scratch = nullptr; size_t l2_n = 0;
  struct CnnState* cnn = nullptr;  // VGG-16 fc7 producer (cnn_sm100.cu): allocated by the first CNN call, null until then
};

// VGG-16 fc7 producer (cnn_sm100.cu), one GPU handle each; argument checks included, group dispatch in lrcn_api.cu
int cnn_set_param(lrcn_handle* h, int layer, int which, const float* data, const int64_t dims[4]);
int cnn_get_param(lrcn_handle* h, int layer, int which, float* data, const int64_t dims[4]);
int cnn_extract(lrcn_handle* h, const float* images, int64_t n, int flags, float* feats_out);
int cnn_activation(lrcn_handle* h, int layer, float* out, int64_t n);  // test hook lrcn_test_cnn_activation
void cnn_free(lrcn_handle* h);

static inline float* WS(lrcn_handle* h, size_t off) { return h->ws.f + off; }
static inline float* Wp(lrcn_handle* h, int idx1) { return h->w + h->off[idx1 - 1]; }
static inline float* Gp(lrcn_handle* h, int idx1) { return h->g + h->off[idx1 - 1]; }

static void shadow(lrcn_handle* h, const float* p, bf16** hi, bf16** lo) {
  if (p >= h->w && p < h->w + h->P) { *hi = h->w_hi + (p - h->w); *lo = h->w_lo + (p - h->w); return; }
  *hi = h->ws.hi + (p - h->ws.f);
  *lo = h->ws.lo + (p - h->ws.f);
}
struct ShadowPair { bf16* hi; bf16* lo; };
static ShadowPair SH(lrcn_handle* h, const float* p) {  // null pair in fp32 mode: producers then skip the split
  ShadowPair sp{nullptr, nullptr};
  if (h->bf16mode) shadow(h, p, &sp.hi, &sp.lo);
  return sp;
}
static void split_ws(lrcn_handle* h, const float* p, size_t n) {
  if (!h->bf16mode) return;
  bf16 *hi, *lo;
  shadow(h, p, &hi, &lo);
  split_bf16(h->stream, p, n, hi, lo);
}

