// kernels.cuh -- device-kernel launchers shared by the C-ABI layer (lrcn_api.cu).
// All matrices here are ROW-MAJOR device buffers; the reference's column-major K x N weight
// is the same memory as a row-major [N][K] matrix, so no relayout is needed except Wemb.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace lrcn {

// Scalars that change every step live in device memory so that a captured CUDA graph of the
// step can be replayed without re-baking kernel arguments.
struct StepScalars {
  float inv_ntok;       // 1 / (global token count) : dA scale (lrcn.jl:580 -total/count)
  float pdrop;          // dropout probability (lrcn.jl:542,547)
  float keep_scale;     // 1/(1-pdrop)
  uint32_t drop_thresh; // keep iff (hash>>8) >= drop_thresh ; drop_thresh = pdrop * 2^24
  uint64_t seed;
  float adam_d1;        // 1 - beta1^t
  float adam_d2;        // 1 - beta2^t
  float lr, beta1, beta2, eps;
  float one_m_beta1;    // (float)(1 - beta1), computed in double like Knet's axpy!(1-p.beta1, ...)
  float one_m_beta2;
  uint32_t xchg_epoch;  // data-parallel train steps run so far + 1 (same on every rank): the value of the fused exchange's chunk flags
  uint32_t pad_;
  double gclip;         // Knet Adam(gclip=...) per parameter tensor; 0 = off (lrcn_set_gclip)
};

// ---- programmatic dependent launch (PDL).  A kernel launched through launch_pdl may be scheduled while its predecessor in
// the stream is still draining; it must execute pdl_wait() before touching any global memory the predecessor reads or
// writes, and calls pdl_trigger() AFTER that wait, so at most two consecutive kernels overlap and everything two or more
// launches upstream is complete when a kernel starts.  LRCN_PDL=0 turns the launch attribute off.
extern int g_pdl;
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <int LEVEL = 1, typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = g_pdl >= LEVEL ? 1 : 0;  // LRCN_PDL: 0 off, 1 tcgen05 kernels (default), 2 all
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// ---- device-side time-outs.  Every spin wait in the persistent kernels (mbarrier, grid barrier, cross-GPU flag barrier) is
// clock-bounded.  A wait that times out does NOT trap (a trap destroys the CUDA context and every later call fails
// undiagnosed): it raises a flag -- one copy per translation unit in device memory, so that every other wait of that unit
// returns at once and the kernels drain, plus ONE process-wide word in mapped host memory that the C ABI checks after every
// synchronisation and turns into a sticky LRCN_ERR_CUDA "device-side barrier time-out" on the handle.
#ifdef __CUDACC__
static __device__ unsigned int g_dev_abort = 0;
static __device__ unsigned int* g_dev_abort_host = nullptr;
__device__ __forceinline__ bool dev_aborted() { return *reinterpret_cast<volatile unsigned int*>(&g_dev_abort) != 0u; }
static __device__ __noinline__ void dev_abort_set() {
  atomicExch(&g_dev_abort, 1u);
  if (g_dev_abort_host) { *reinterpret_cast<volatile unsigned int*>(g_dev_abort_host) = 1u; __threadfence_system(); }
}
// host: bind this translation unit's flag pointer on the CURRENT device (called from lrcn_create, never inside a capture)
static inline cudaError_t dev_abort_bind(unsigned int* host_flag) {
  const unsigned int zero = 0;
  cudaError_t e = cudaMemcpyToSymbol(g_dev_abort_host, &host_flag, sizeof host_flag);
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_dev_abort, &zero, sizeof zero);
  return e;
}
#endif
bool gemm_bind_abort(unsigned int* host_flag);   // gemm_sm100.cu
bool gemm2_bind_abort(unsigned int* host_flag);  // gemm2_sm100.cu
bool lstm_bind_abort(unsigned int* host_flag);   // lstm_sm100.cu
bool dp_bind_abort(unsigned int* host_flag);     // dp_p2p.cu

struct LaunchCounter { long long n = 0; };
extern thread_local LaunchCounter* g_counter;  // incremented by every launcher below

// ---------------------------------------------------------------- GEMM (fp32, CUDA cores)
// C[M][N] (ldc) = sum_k Aop[m][k] * Bop[k][n]  (+ C if beta) (+ bias[n])
//   a_kmajor: A[m*lda+k] else A[k*lda+m];  b_kmajor: B[n*ldb+k] else B[k*ldb+n]
void sgemm(cudaStream_t s, bool a_kmajor, bool b_kmajor, int M, int N, int K, const float* A, int lda,
           const float* B, int ldb, float* C, int ldc, bool beta, const float* bias);

// ---------------------------------------------------------------- elementwise / gather kernels
void gather_features(cudaStream_t s, const float* table, const int* rows, int B, float* X, __nv_bfloat16* hi = nullptr,
                     __nv_bfloat16* lo = nullptr);  // hi/lo: optional bf16 split of the output, same indexing
// E_all[r][:] = WembT[tok[r]][:] (* dropout mask site 0);  tok 0-based
void gather_embed(cudaStream_t s, const float* WembT, const int* tok, int R, int E, float* out,
                  const StepScalars* sc, bool train, __nv_bfloat16* hi = nullptr, __nv_bfloat16* lo = nullptr,
                  int ld_out = 0 /* row pitch of out (0 = E) */);
// Z[r][C+j] = v[r % B][j]; then dropout (site 1) over the whole row of 2C
void z_finish(cudaStream_t s, float* Z, const float* v, int ldv, int R, int B, int C, const StepScalars* sc, bool train,
              __nv_bfloat16* hi = nullptr, __nv_bfloat16* lo = nullptr, int ldz = 0 /* row pitch of Z (0 = 2C) */);
// LSTM cell forward for one step: gates (pre-activation, [B][4H], order f,i,o,g) are activated in place
void lstm_cell_fwd(cudaStream_t s, float* gates, const float* c_prev, float* c_out, float* h_out, int B, int H,
                   __nv_bfloat16* h_hi = nullptr, __nv_bfloat16* h_lo = nullptr);
// generation-only cell (bf16x3 mode, H % 4 == 0): 4 units per thread, fast sigmoid/tanh, gate activations not written back
void lstm_cell_gen(cudaStream_t s, const float* gates, const float* c_prev, float* c_out, float* h_out, int B, int H, __nv_bfloat16* h_hi,
                   __nv_bfloat16* h_lo);
// LSTM cell backward for one step; gates buffer holds activations and receives dG in place
void lstm_cell_bwd(cudaStream_t s, float* gates, const float* c_prev, const float* c_cur, const float* dh_in,
                   const float* dh_rec /*nullable*/, float* dc /*in/out*/, bool first /*dc,dh_rec are zero*/,
                   int B, int H);
// row-wise log-softmax cross-entropy: rowlp[r] = logp(a_r)[y_r]; if train, logits <- (softmax - onehot)*inv_ntok
void softmax_ce(cudaStream_t s, float* logits, int ld, int R, int V, const int* tgt, float* rowlp,
                const StepScalars* sc, bool train, __nv_bfloat16* hi = nullptr, __nv_bfloat16* lo = nullptr,
                double* total_out = nullptr /* fp64 sum of rowlp, written by the last CTA */, unsigned int* done_ctr = nullptr);
// bf16x3 training variant: writes only the bf16 hi/lo split of dA and folds the output-bias gradient (column sums of dA) in;
// colpart: scratch [colpart_rows][ld]; dbias must be zero on entry.  Returns false (nothing launched) if it does not apply.
bool softmax_ce_fused(cudaStream_t s, const float* logits, int ld, int R, int V, const int* tgt, float* rowlp, const StepScalars* sc,
                      __nv_bfloat16* hi, __nv_bfloat16* lo, float* colpart, int colpart_rows, float* dbias, double* total_out,
                      unsigned int* done_ctr);
void reduce_sum_double(cudaStream_t s, const float* x, int n, double* out);
void colsum(cudaStream_t s, const float* A, int ld, int R, int N, float* out, bool accumulate);
// dZ *= dropout mask (site 1); dv[i][j] = sum_t dZ[(t*B+i)][C+j]
void dz_finish(cudaStream_t s, float* dZ, float* dv, int ldv, int T, int B, int C, const StepScalars* sc, bool train,
               __nv_bfloat16* z_hi = nullptr, __nv_bfloat16* z_lo = nullptr, __nv_bfloat16* v_hi = nullptr, __nv_bfloat16* v_lo = nullptr);
// dWembT[tok[r]][:] += dE[r][:] (* dropout mask site 0)
void scatter_add_embed(cudaStream_t s, float* dWembT, const int* tok, const float* dE, int R, int E,
                       const StepScalars* sc, bool train);
// ---- per-tensor gradient clipping (Knet update!(w, g, ::Adam) -> gclip!(g, gclip)).  A range of whole parameter tensors of the
// arena; tensor j starts at float4 index off4[j] (tensor offsets are 64-element aligned, so no float4 straddles two tensors).
constexpr int GNORM_CHUNK4 = 4096;  // 16 Ki floats: one fp64 partial sum each, never straddling tensors
struct TensorRange {
  int n;                   // tensors in the range (<= 9)
  int k[9];                // 0-based model index of each (indexes norm[] / scale[])
  size_t off4[9];          // start, float4 units, relative to the pointer the kernel is given
  size_t nel[9];           // elements (the tail of the last float4 beyond nel is ignored)
  int chunk0[9];           // first partial-sum slot of each: a tensor's slots are the same whichever launch covers it
};
// norm[k] = sqrt(sum g^2) in fp64 and scale[k] = (gclip > 0 && norm > gclip) ? (float)(gclip / norm) : 1 for every tensor of the
// range.  The result depends neither on the grid nor on which other tensors the launch covers.  ticket: zero on entry, reset
// by the kernel (graph replay).
void grad_sqnorm(cudaStream_t s, const float* g, const TensorRange& r, double* part, double* norm, float* scale, unsigned int* ticket,
                 const StepScalars* sc, int grid_cap);
// Adam's view of the clip: the range's tensors as end offsets (float4 units, relative to the range start) and their scales
struct ClipMap {
  const float* scale;      // [9], model order (written by grad_sqnorm)
  size_t end4[9];
  int k[9];
  int n;
};
// fused dense Adam over one flat range (Knet defaults, lrcn.jl:394,402); optionally refreshes bf16 hi/lo shadows.
// clip != null: g is multiplied by its tensor's scale before the moments (g itself is not written)
void adam_flat(cudaStream_t s, float* w, const float* g, float* m, float* v, size_t n, const StepScalars* sc,
               __nv_bfloat16* w_hi, __nv_bfloat16* w_lo, const ClipMap* clip = nullptr);
void adam_range(cudaStream_t s, float* w, const float* g, float* m, float* v, size_t n, const StepScalars* sc, __nv_bfloat16* w_hi,
                __nv_bfloat16* w_lo, int grid, const ClipMap* clip = nullptr);
void split_bf16(cudaStream_t s, const float* x, size_t n, __nv_bfloat16* hi, __nv_bfloat16* lo);
// ---- batch staging on the device (SURVEY 8 row f-1; lrcn.jl:351-376): the epoch's token matrix and image ids are resident
// image id -> feature-table row for a whole epoch: ids [n] (1-based wire ids), sorted_ids/rowof [n_tab]; unknown ids raise *err
void epoch_lookup_rows(cudaStream_t s, const long long* ids, size_t n, const long long* sorted_ids, const int* rowof, int n_tab, int* rows_out, int* err);
// inputs [bos, w1..wl] / targets [w1..wl, eos] / feature rows of ONE batch from the resident epoch data (lrcn.jl:556,563-577):
// seq rows [row0, row0+l) of the [n_rows][ldB] int64 matrix, columns [col0, col0+B); tokens outside [1, V] raise *err
void epoch_stage_batch(cudaStream_t s, const long long* seq, size_t row0, int l, int ldB, int col0, int B, int V, const int* rows_all, size_t rows_off,
                       int* tok_in, int* tok_tgt, int* rows, int* err);
void transpose2d(cudaStream_t s, const float* in, int rows, int cols, float* out);  // out[c][r] = in[r][c]
void fill_l2_scratch(cudaStream_t s, float* buf, size_t n, float val);
// one launch zeroing up to 16 fp32 ranges (16-byte aligned starts): accumulation targets of the step (split-K / stream-K GEMM
// outputs, bias-gradient column sums, the embedding-gradient scatter, the LSTM grid-barrier counters)
struct ZeroSegs { float* p[16]; size_t n[16]; int count = 0; void add(void* ptr, size_t nfloats) { if (ptr && nfloats && count < 16) { p[count] = (float*)ptr; n[count] = nfloats; count++; } } };
void zero_multi(cudaStream_t s, const ZeroSegs& z);

// ---------------------------------------------------------------- beam search
// per row: prob = exp(logp(a)); top-K by (prob desc, index asc); cand_* are [R][K].  Needs 1 <= K <= TOPK_MAXK (11):
// lrcn_beam_search and the test hooks reject larger beam widths before any launch.
void beam_row_topk(cudaStream_t s, const float* logits, int ld, int R, int V, int K, const float* parent_prob,
                   int* cand_tok, float* cand_score, float* cand_lp);
// the same on given probabilities (test hook only)
void beam_row_topk_probs(cudaStream_t s, const float* probs, int ld, int R, int V, int K, const float* parent_prob,
                         int* cand_tok, float* cand_score, float* cand_lp);
// per image: pick K of the K*K (K at the first step) candidates by (score desc, list position asc).  Only the test hook calls
// it; in a decode step beam_advance makes the same picks with the same device code.
void beam_select(cudaStream_t s, const int* cand_tok, const float* cand_score, const float* cand_lp, int n_img, int K,
                 int first_step, int* sel_tok, int* sel_parent, float* sel_score, float* sel_lp);
struct BeamAdvanceArgs {
  int n_img, K, H1, H2, maxlen, step, nword;
  int ld1, ld2;  // row pitch of h1_out / h2_out (they are the h-columns of the [x|h] GEMM operand buffers)
  const float *h1_in, *c1_in, *h2_in, *c2_in; float *h1_out, *c1_out, *h2_out, *c2_out;
  const int* hist_in; int* hist_out; const float* lp_in; float* lp_out;
  __nv_bfloat16 *h1_hi, *h1_lo, *h2_hi, *h2_lo;  // optional bf16 split of the gathered h states (null in fp32 mode)
  float* prob; int* last_tok; int* done; int* n_done;
  long long* out_tokens; int* out_len; float* out_prob; float* out_lp;
  const int* out_map;  // compacted image index -> image index of the caller's chunk (outputs are written there); null = identity
  // the row's CTA picks its candidate by the image's stable selection over the K*K candidates (K at the first step), and the
  // k = 0 row marks the image done: one launch per decode step does all its bookkeeping
  const int* cand_tok; const float* cand_score; const float* cand_lp;
  // the row also gathers the embedding of its new token -- the next step's x operand (gather_embed_kernel's job, lrcn.jl:650);
  // skipped when wemb is null
  const float* wemb; float* e_out; __nv_bfloat16 *e_hi, *e_lo; int E, lde;
};
void beam_advance(cudaStream_t s, const BeamAdvanceArgs& a);
// Compaction of the generation batch: images whose best hypothesis has ended (lrcn.jl:670) leave the batch, the survivors'
// K rows (states, histories, scores) and per-image data move to the front.  Two launches (gather into scratch, copy back)
// because a parallel in-place move is not safe.
struct BeamCompactArgs {
  int n_keep, K, H1, H2, ld1, ld2, ldv, maxlen, hist_len;
  const int* keep;                                   // [n_keep] old (compacted) image index of the survivors, ascending
  float *h1, *c1, *h2, *c2;                          // current states: h with row pitch ld1 / ld2, c with H1 / H2
  float *h1_s, *c1_s, *h2_s, *c2_s;                  // scratch, contiguous rows
  __nv_bfloat16 *h1_hi, *h1_lo, *h2_hi, *h2_lo;      // bf16 split of h (row pitch ld1 / ld2), rebuilt on copy-back; may be null
  const int* hist_src; int* hist_dst; const float* lp_src; float* lp_dst;   // ping-pong history buffers: gathered into the other one
  float *prob, *prob_s; int *last, *last_s; float *v, *v_s; int *out_map, *out_map_s; int *done, *done_s;
};
void beam_compact(cudaStream_t s, const BeamCompactArgs& a);

// ---------------------------------------------------------------- tcgen05 path (gemm_sm100.cu)
// Same contract as sgemm, operands given as pre-split bf16 hi/lo pairs (ld in elements, multiple of 8).
bool gemm_bf16x3(cudaStream_t s, bool a_kmajor, bool b_kmajor, int M, int N, int K,
                 const __nv_bfloat16* A_hi, const __nv_bfloat16* A_lo, int lda,
                 const __nv_bfloat16* B_hi, const __nv_bfloat16* B_lo, int ldb,
                 float* C, int ldc, bool beta, const float* bias,
                 __nv_bfloat16* C_hi, __nv_bfloat16* C_lo /* optional split of the result, same ldc */,
                 bool c_zeroed = false /* C is known to be all zero: split-K / stream-K partial sums need no zero-fill */);
const char* gemm_bf16x3_last_error();
bool init_gemm_sm100();   // func attributes + driver entry point; call once outside any capture
bool init_gemm2_sm100();
// 2-CTA (cta_group::2) 256x256 pair-tile variant, same contract (gemm2_sm100.cu); gemm_bf16x3 dispatches to it
bool gemm_tma_epilogue_ok(const float* C, int ldc, bool beta, const void* C_hi);
extern int g_gemm_dbg;  // diagnostics for lrcn_bench_gemm only (0 in production)
bool gemm2_bf16x3(cudaStream_t s, bool a_kmajor, bool b_kmajor, int M, int N, int K, const __nv_bfloat16* A_hi, const __nv_bfloat16* A_lo,
                  int lda, const __nv_bfloat16* B_hi, const __nv_bfloat16* B_lo, int ldb, float* C, int ldc, bool beta, const float* bias,
                  __nv_bfloat16* C_hi, __nv_bfloat16* C_lo, bool c_zeroed = false);
bool gemm2_bf16x3_dualB(cudaStream_t s, bool a_kmajor, bool b_kmajor, int M, int N1, int N2, int K, const __nv_bfloat16* A_hi,
                        const __nv_bfloat16* A_lo, int lda, const __nv_bfloat16* B1_hi, const __nv_bfloat16* B1_lo, int ldb1,
                        const __nv_bfloat16* B2_hi, const __nv_bfloat16* B2_lo, int ldb2, float* C, int ldc, bool c_zeroed, bool* launched);
void init_simt_kernels();

// ---------------------------------------------------------------- data-parallel exchange over peer memory (dp_p2p.cu)
constexpr int LRCN_P2P_MAX_RANKS = 8;
struct P2PCtl {              // one per rank, in a small exported allocation
  unsigned int flags[64];    // flags[q]: last barrier epoch signalled by rank q
  double loss_partial;       // this rank's fp64 sum of token log-probs of the current step
};
struct P2PPeers { float* g[LRCN_P2P_MAX_RANKS]; float* w[LRCN_P2P_MAX_RANKS]; P2PCtl* ctl[LRCN_P2P_MAX_RANKS]; int nranks, rank; };
// barrier, in-place allreduce(sum) of the gradient arena (n_floats) + loss total, barrier
void dp_p2p_allreduce(cudaStream_t s, const P2PPeers& peers, size_t n_floats, unsigned int* epoch_ctr, double* loss_total);
// %globaltimer stamp at a point of a stream (LRCN_DP_STAMPS=1, tools/dp_timeline.py)
void dp_stamp(cudaStream_t s, unsigned long long* out);
// FUSED exchange of one gradient bucket (dp_p2p.cu): push of gradient chunks -> per-chunk flags -> owner-side sum + Adam ->
// push of the new weights -> completion counters, all in ONE kernel.  The control words live behind the staging rows.
constexpr int DP_XMAXCH = 512;                  // chunk flags per (bucket, source rank)
constexpr size_t DP_XCTL_FLOATS = 20480;        // control area at the end of every rank's staging allocation (u32 words): 64 + 4 * 8 * 512
struct FusedXArgs {
  float* stage[LRCN_P2P_MAX_RANKS];             // every rank's staging allocation (own included)
  size_t b4[LRCN_P2P_MAX_RANKS], e4[LRCN_P2P_MAX_RANKS];  // rank r's slice of the bucket, arena index in float4 units
  size_t stride4, pre4, ctl4;                   // staging row stride, the bucket's offset inside a row, start of the control area (float4 units)
  int bucket, sub;
};
void dp_fused_exchange(cudaStream_t s, const P2PPeers& peers, const FusedXArgs& a, float* m, float* v, const StepScalars* sc, double* loss_total, int grid_ctas);
// diagnostics (probe_mma.cu): clocks to issue / to complete a chain of n_mma tcgen05.mma M x N x 16 from resident smem operands
bool probe_mma(cudaStream_t s, int M, int N, int n_mma, int commit_every, int issuers, long long* issue_clk, long long* total_clk);

// ---------------------------------------------------------------- fused LSTM timestep (lstm_sm100.cu)
bool init_lstm_sm100();
size_t lstm_permuted_elems(int H);    // elements of the gate-interleaved forward operand (per hi / lo)
size_t lstm_transposed_elems(int H);  // elements of the transposed backward operand (per hi / lo)
// W_h = columns [x_off, x_off+H) of each layer weight W [4H][ldw] -> bf16 hi/lo step operands of both layers (t*_ may be null)
void lstm_prepare_weights2(cudaStream_t s, const float* W1, int ldw1, int x_off1, int H1, __nv_bfloat16* p1_hi, __nv_bfloat16* p1_lo,
                           __nv_bfloat16* t1_hi, __nv_bfloat16* t1_lo, const float* W2, int ldw2, int x_off2, int H2, __nv_bfloat16* p2_hi,
                           __nv_bfloat16* p2_lo, __nv_bfloat16* t2_hi, __nv_bfloat16* t2_lo);
// gates [B][4H] holds x-part + bias on entry and the activated gates on exit; has_rec=false at t=0 (h_0 = 0)
bool lstm_fwd_step(cudaStream_t s, int B, int H, bool has_rec, const __nv_bfloat16* hprev_hi, const __nv_bfloat16* hprev_lo,
                   const __nv_bfloat16* wperm_hi, const __nv_bfloat16* wperm_lo, float* gates, const float* c_prev, float* c_out,
                   float* h_out, __nv_bfloat16* h_hi, __nv_bfloat16* h_lo);
// gates [B][4H] holds the step's activations on entry and dG on exit (fp32 + bf16 hi/lo); has_rec=false at t=T-1
bool lstm_bwd_step(cudaStream_t s, int B, int H, bool has_rec, const __nv_bfloat16* wt_hi, const __nv_bfloat16* wt_lo,
                   const __nv_bfloat16* gnext_hi, const __nv_bfloat16* gnext_lo, float* gates, __nv_bfloat16* g_hi, __nv_bfloat16* g_lo,
                   const float* c_prev, const float* c_cur, const float* dh_in, float* dc);

// persistent whole-sequence variants (weights resident in tensor and shared memory, grid barrier per step).  *launched = false
// (and nothing enqueued) when they do not apply (H > 512, B > 2048, T < 2, grid not co-resident): use the per-step kernels then.
// counters: 64 uint32 in device memory, ZERO on entry (the caller zeroes them once per step; one region per launch).  hs/cs: [(T+1)*B][H] slot buffers; acts: [T*B][4H].
bool lstm_fwd_seq(cudaStream_t s, int B, int H, int T, const __nv_bfloat16* wperm_hi, const __nv_bfloat16* wperm_lo, float* acts, float* hs,
                  float* cs, __nv_bfloat16* hs_hi, __nv_bfloat16* hs_lo, unsigned int* counters, bool* launched,
                  unsigned long long* trace = nullptr /* optional [T][4 chains][8] globaltimer stamps of CTA (0,0) */);
bool lstm_bwd_seq(cudaStream_t s, int B, int H, int T, const __nv_bfloat16* wt_hi, const __nv_bfloat16* wt_lo, float* acts,
                  __nv_bfloat16* acts_hi, __nv_bfloat16* acts_lo, float* cs, const float* dh_all, float* dc, unsigned int* counters,
                  bool* launched, float* dbias = nullptr /* optional [4H], zero on entry: receives the bias gradient (column sums of dG) */,
                  unsigned long long* trace = nullptr);

}  // namespace lrcn
