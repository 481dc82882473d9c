/* lrcn_b200.h -- C ABI of liblrcn_b200.so: the B200-native LRCN caption-decoder hot path.
 *
 * Drop-in boundary for ekinakyurek/Long-Term-Recurrent-Convolutional-NN (`lrcn.jl`).  The
 * reference has no FFI layer; its seam is a set of Julia call sites (SURVEY.md §8b).  Each
 * entry point below names the reference call site (file:line) it replaces.  The Julia host
 * keeps its CLI flags, weight vector (9 column-major Float32 matrices), tokenizer and eval
 * code and reaches this library through `ccall` (julia/lrcn_b200.jl, INTEGRATION.md).
 *
 * Conventions
 *  - every function returns 0 on success, non-zero on failure; lrcn_last_error() returns a
 *    thread-local message.  No C++ exception crosses the ABI.  There is NO CPU fallback:
 *    without a CUDA device lrcn_create fails with LRCN_ERR_CUDA.
 *  - Int <-> int64_t, Float32 <-> float, Float64 <-> double; matrices are raw pointers to
 *    COLUMN-MAJOR storage exactly as Julia holds them; token / image ids are 1-based on the
 *    wire (eos=1,bos=2,unk=3: lrcn.jl:248-255).
 *  - the library owns all device memory, streams, CUDA graphs and NCCL communicators; the
 *    caller owns every host buffer and may free it as soon as the call returns (all calls
 *    are synchronous on return unless the name ends in _async).
 *  - one host thread per handle.  Two ways to use several GPUs of one NVLink node:
 *      (a) ONE process, ONE handle: set cfg.n_gpus / cfg.device_ids and the library drives all GPUs itself
 *          (peer access between its own devices, worker threads for generation): an unmodified single-process
 *          lrcn.jl gets data parallelism from lrcn_train_step alone -- batches are global, the library shards rows;
 *      (b) one process per GPU (torch.distributed / MPI launchers): one handle per rank, joined by
 *          lrcn_p2p_export/import (CUDA IPC) or lrcn_comm_init (NCCL).
 *  - CUDA / NCCL errors and device-side barrier time-outs are STICKY: once a handle has failed that way every later
 *    call on it returns the same code and message (the context may be unusable); destroy the handle.
 */
#ifndef LRCN_B200_H
#define LRCN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LRCN_API __attribute__((visibility("default")))
#else
#define LRCN_API
#endif

/* 2: lrcn_config gained n_gpus / device_ids (single-process multi-GPU group); sticky errors; lrcn_checkpoint_save / _load;
 *    lrcn_train_epoch / lrcn_loss_epoch (epoch-level calls, batches staged on the device: additive, same version);
 *    lrcn_set_cnn_param / lrcn_get_cnn_param / lrcn_extract_features (VGG-16 fc7 producer: additive, same version) */
#define LRCN_ABI_VERSION 2
#define LRCN_F_CNN 4096 /* lrcn.jl:28  const cnnout = 4096 */
#define LRCN_NUM_PARAMS 9

enum {
  LRCN_OK = 0,
  LRCN_ERR_ARG = 1,     /* bad argument / shape mismatch (the reference would throw) */
  LRCN_ERR_CUDA = 2,    /* CUDA runtime/driver error, incl. "no device" and device-side barrier time-outs; sticky on the handle */
  LRCN_ERR_NCCL = 3,
  LRCN_ERR_MISSING = 4, /* unknown image id: lrcn.jl:602-605 error("misssing features!!!!!!") */
  LRCN_ERR_STATE = 5
};

enum {
  LRCN_PREC_FP32 = 0,  /* fp32 CUDA-core GEMMs (exact-mode; bit-stable reductions) */
  LRCN_PREC_BF16X3 = 1 /* tcgen05 tensor cores, error-compensated bf16 hi/lo split, fp32 TMEM accumulate */
};

typedef struct lrcn_handle lrcn_handle;

/* Hot-path configuration.  Defaults mirror the reference: lrcn.jl:39-40 (--hidden 1000 1000,
 * --embed 1000), lrcn.jl:402 Adam() (lr 1e-3, b1 .9, b2 .999, eps 1e-8; --lr/--gclip are ignored
 * by the reference, lrcn.jl:330,386-393), lrcn.jl:353 (captions longer than 28 are skipped). */
typedef struct {
  int32_t embed;        /* E  */
  int32_t hidden1;      /* H1 */
  int32_t hidden2;      /* H2 (even; C = H2/2) */
  int32_t vocab;        /* V  */
  int32_t max_batch;    /* largest B per train/eval step on this GPU */
  int32_t max_len;      /* largest caption length l (decoder steps T = l+1) */
  int32_t max_gen_rows; /* largest images_in_flight * beam_width for generation */
  int32_t device;       /* CUDA device ordinal */
  int32_t precision;    /* LRCN_PREC_* */
  int32_t use_graphs;   /* 1: replay each (B,l) step shape as a CUDA graph */
  double lr, beta1, beta2, eps; /* Float64 like Knet's Adam fields: (float)(1-beta) must equal Knet's axpy! scalar */
  int32_t n_gpus;       /* 0 or 1: one GPU (`device`).  2..8: single-process data parallelism over device_ids[0..n_gpus) */
  int32_t device_ids[8];/* CUDA ordinals of the group; max_batch and max_gen_rows are then GLOBAL (summed over the GPUs) */
} lrcn_config;

LRCN_API int lrcn_abi_version(void);
LRCN_API const char* lrcn_last_error(void);
LRCN_API int lrcn_config_default(lrcn_config* cfg);

/* lifecycle.  Replaces nothing in the reference (Knet allocates implicitly). */
LRCN_API int lrcn_create(const lrcn_config* cfg, lrcn_handle** out);
LRCN_API int lrcn_destroy(lrcn_handle* h);

/* ---- weights: the frozen 9-matrix contract, idx = 1..9 in `model` order --------------------
 * replaces initweights() hand-off lrcn.jl:87, JLD load lrcn.jl:90, save lrcn.jl:185,230.
 *   1 W1 (E+H1)x4H1   2 b1 1x4H1   3 W2 2H2x4H2   4 b2 1x4H2   5 Wf H1xC   6 Wcnn 4096xC
 *   7 Wemb VxE        8 Wout H2xV  9 bout 1xV            (lrcn.jl:489-510)
 * get(set(x)) round-trips bit-exactly when no step intervened. */
LRCN_API int lrcn_param_shape(const lrcn_handle* h, int idx, int64_t* rows, int64_t* cols);
LRCN_API int lrcn_set_param(lrcn_handle* h, int idx, const float* colmajor, int64_t rows, int64_t cols);
LRCN_API int lrcn_get_param(lrcn_handle* h, int idx, float* colmajor, int64_t rows, int64_t cols);
/* gradient of the last lrcn_grad / lrcn_train_step, same shapes (what lossgradient returns, lrcn.jl:583) */
LRCN_API int lrcn_get_grad(lrcn_handle* h, int idx, float* colmajor, int64_t rows, int64_t cols);
/* Adam state extension (the reference never saves it, SURVEY.md §5): which = 0 -> m, 1 -> v */
LRCN_API int lrcn_get_adam_state(lrcn_handle* h, int idx, int which, float* colmajor, int64_t rows, int64_t cols);
LRCN_API int lrcn_set_adam_state(lrcn_handle* h, int idx, int which, const float* colmajor, int64_t rows, int64_t cols);
LRCN_API int lrcn_get_adam_step(lrcn_handle* h, int64_t* t);
LRCN_API int lrcn_set_adam_step(lrcn_handle* h, int64_t t);

/* ---- features: replaces the `feats` / `featsvl` Dict{Int,Array{Float32}} globals (lrcn.jl:121-123)
 * and the per-row staging loop lrcn.jl:369-376.  split 0 = train, 1 = val/test.  feats holds n rows
 * of 4096 contiguous floats.  The table stays resident in HBM; ids are mapped host-side. */
LRCN_API int lrcn_load_features(lrcn_handle* h, int split, const int64_t* ids, const float* feats, int64_t n);

/* ---- training (tokens: l x B int64, time-major: tokens[t*B+i], 1-based; image_ids: B) --------
 * lrcn_loss       = loss() forward only, lrcn.jl:553-581 / average_loss body lrcn.jl:452-474:
 *                   returns sum of target log-probs and the token count B*(l+1).
 * lrcn_grad       = lossgradient(...) lrcn.jl:378,583 (no update); loss_out = -total/count.
 * lrcn_adam_update= update!(param,gloss,optim) lrcn.jl:394 on the gradients currently held.
 * lrcn_train_step = lrcn.jl:378 + :394 fused (gradient, [allreduce], Adam).
 * pdrop: dropout probability at the two sites lrcn.jl:542,547 (0 => identity; parity is defined
 * at 0 since Knet's RNG is not reproducible); seed feeds the in-kernel counter RNG. */
LRCN_API int lrcn_loss(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B,
              double* sum_logp_out, int64_t* count_out);
LRCN_API int lrcn_grad(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B,
              float pdrop, uint64_t seed, double* loss_out);
LRCN_API int lrcn_adam_update(lrcn_handle* h);
LRCN_API int lrcn_train_step(lrcn_handle* h, int split, const int64_t* image_ids, const int64_t* tokens, int l, int B,
                    float pdrop, uint64_t seed, double* loss_out);
/* ---- one epoch of the train1 hot loop in ONE call (lrcn.jl:336-396; SURVEY 8 row f-1: batch staging on the device).
 * sequence: the [n_rows][B] time-major token matrix minibatch() builds (lrcn.jl:257-297: batch b owns lengths[b] consecutive
 * rows), input_ids: [n_batches][B], lengths: [n_batches], order: the host's shuffled batch order (lrcn.jl:351; NULL = 0..n-1).
 * The epoch is uploaded once, image ids are resolved to feature rows on the device, every batch is staged by a kernel from
 * the resident data, batches with l > max_len are skipped (lrcn.jl:353) and no step synchronises with the host.
 * losses_out (optional, n_order values): loss of every executed step, in execution order; steps_out: how many ran.
 * Step k uses dropout seed `seed + k`. */
LRCN_API int lrcn_train_epoch(lrcn_handle* h, int split, const int64_t* sequence, int64_t n_rows, const int64_t* input_ids,
                     const int64_t* lengths, int64_t n_batches, int B, const int64_t* order, int64_t n_order, float pdrop,
                     uint64_t seed, double* losses_out, int64_t* steps_out);
/* ---- average_loss over a whole split in ONE call (lrcn.jl:407-486): forward only, pdrop 0, batches in natural order, staged on
 * the device like lrcn_train_epoch; l > max_len batches are skipped (lrcn.jl:431).  Returns the sum of the target log-probs and
 * the token count, like lrcn_loss: average_loss = -sum / count (lrcn.jl:476-486). */
LRCN_API int lrcn_loss_epoch(lrcn_handle* h, int split, const int64_t* sequence, int64_t n_rows, const int64_t* input_ids,
                    const int64_t* lengths, int64_t n_batches, int B, double* sum_logp_out, int64_t* count_out);
/* per-token target log-probs of the last lrcn_loss/lrcn_grad call, (l+1) x B time-major */
LRCN_API int lrcn_get_token_logps(lrcn_handle* h, float* out, int64_t n);

/* device-resident variant for kernel-only timing: stage a batch once (H2D), then step on it
 * repeatedly with no host<->device traffic.  slot in [0, 64). */
LRCN_API int lrcn_stage_batch(lrcn_handle* h, int slot, int split, const int64_t* image_ids, const int64_t* tokens,
                     int l, int B);
LRCN_API int lrcn_train_step_staged(lrcn_handle* h, int slot, float pdrop, uint64_t seed, double* loss_out /* may be NULL: no D2H */);

/* ---- generation: generate()+beam_search() numeric part, lrcn.jl:585-632,644-678, for n images at
 * once (the reference loops images serially, lrcn.jl:152-155).  tokens_out: n x (nword+2) int64
 * incl. the leading bos; len_out[n] tokens used; prob_out[n] fp32 path probability of the best
 * hypothesis; logp_out (optional, n x (nword+1)) log-prob of each generated token.  The caller
 * prints tokens[2:] up to the first eos (lrcn.jl:633-640). */
LRCN_API int lrcn_beam_search(lrcn_handle* h, int split, const int64_t* image_ids, int64_t n, int beam_width, int nword,
                     int64_t* tokens_out, int32_t* len_out, float* prob_out, float* logp_out);

/* ---- fc7 producer (SURVEY 8 row f-4): VGG-16 up to relu7.  Replaces get_params_cnn / get_convnet / extract_features
 * (lrcn.jl:190-221, 697-773).  layer 1..13 = conv1_1..conv5_3, 14 = fc6, 15 = fc7; which 0 = filter, 1 = bias.
 * All arrays are column-major Float32 as Julia / MatConvNet hold them; indices below are 0-based.
 *  - images: 224 x 224 x 3 x n, already resized and mean-subtracted by the host (read_image_data); (y, x, c, i) is at
 *    y + 224 x + 224^2 c + 3 224^2 i.
 *  - filter: kh x kw x Cin x Cout, (dy, dx, c, o) at dy + kh dx + kh kw c + kh kw Cin o; dims {kh, kw, Cin, Cout}.
 *    bias: dims {Cout, 1, 1, 1}.  Shapes (MatConvNet's): conv1_x 3->64, 64->64; conv2_x 64->128, 128->128; conv3_x 128->256,
 *    256->256 x2; conv4_x 256->512, 512->512 x2; conv5_x 512->512 x3 (all 3x3); fc6 7x7x512x4096; fc7 1x1x4096x4096.
 *  - layer rule: out(y,x,o) = b(o) + sum_{dy,dx,c} w(dy,dx,c,o) in(y+dy-p, x+dx-p, c) (cross-correlation, zero padding,
 *    p = 1 for the 3x3 layers, 0 for fc6 / fc7); ReLU after every layer; 2x2 stride-2 max-pool after conv1_2, conv2_2,
 *    conv3_3, conv4_3 and conv5_3 (fc6 is a 7x7 convolution over the pooled 7x7x512 map).
 *  - feats_out: relu7 as 4096 x n (image i's 4096 floats contiguous): the layout lrcn_load_features takes.
 *    LRCN_FEAT_L1: each row divided by its sum; a row whose sum is 0 stays all zero.
 *  - images and feats_out may be host memory or device memory (unified addressing).
 *  - get(set(x)) is bit-exact.  LRCN_ERR_ARG: wrong dims, layer / which out of range, null pointers, n <= 0, unknown
 *    flags.  LRCN_ERR_STATE: extraction before all 30 tensors are set, get of a tensor never set.
 *  - the weights (fp32 + bf16 hi/lo, ~1.07 GB) and the extraction workspace (~2.7 GB) are allocated on the first
 *    lrcn_set_cnn_param / lrcn_extract_features and freed by lrcn_destroy.  Group handle: set goes to every GPU,
 *    extraction splits the images into contiguous slices, one per GPU. */
#define LRCN_CNN_LAYERS 15
#define LRCN_CNN_IMAGE 224
#define LRCN_FEAT_L1 1   /* f /= sum(f) per image, like the featsn files and lrcn.jl:597 */
LRCN_API int lrcn_set_cnn_param(lrcn_handle* h, int layer, int which, const float* data, const int64_t dims[4]);
LRCN_API int lrcn_get_cnn_param(lrcn_handle* h, int layer, int which, float* data, const int64_t dims[4]);
LRCN_API int lrcn_extract_features(lrcn_handle* h, const float* images, int64_t n, int flags, float* feats_out);

/* ---- checkpoint sidecar (SURVEY 8 row f-2).  Replaces save(file,"model",model,"vocab",vocab) lrcn.jl:185,230 and
 * load(file) lrcn.jl:88-93 (JLD/HDF5 is not available to a C library): a raw little-endian file
 *   "LRCNB2CK" | u32 version=1 | u32 flags (1 = Adam state) | i32 E,H1,H2,V | i64 adam_t | i64 aux_bytes |
 *   9 x {i64 rows, i64 cols, float32 column-major} [| 9 x m | 9 x v] | aux bytes
 * holding exactly the 9 matrices JLD holds, optionally Knet-Adam's m, v and step (which the reference never saved), and
 * `aux`: caller bytes (the hosts store the vocab Dict as "word\tindex\n" lines).  load validates magic, version, dims and
 * every shape; aux_out may be NULL to query aux_bytes_out first.  julia/lrcn_b200.jl has a pure-Julia reader/writer. */
LRCN_API int lrcn_checkpoint_save(lrcn_handle* h, const char* path, int with_adam, const void* aux, int64_t aux_bytes);
LRCN_API int lrcn_checkpoint_load(lrcn_handle* h, const char* path, int* had_adam, void* aux_out, int64_t aux_cap, int64_t* aux_bytes_out);

/* ---- data-parallel group (new; the reference is single-GPU).  One handle per rank.  The id is
 * produced on rank 0 and distributed by the host's own mechanism (torch.distributed, MPI, file). */
#define LRCN_COMM_ID_BYTES 128
LRCN_API int lrcn_comm_unique_id(char id[LRCN_COMM_ID_BYTES]);
LRCN_API int lrcn_comm_init(lrcn_handle* h, const char id[LRCN_COMM_ID_BYTES], int rank, int nranks);
/* Peer-memory data-parallel exchange (one process per GPU, all on one NVLink node).  Every rank exports a blob describing
 * its gradient arena (CUDA IPC handles), the launcher all-gathers the blobs, every rank imports all of them.  Afterwards
 * the gradient allreduce of lrcn_train_step / lrcn_grad is ONE owner-computes kernel over NVLink peer memory between two
 * flag barriers (csrc/dp_p2p.cu) instead of NCCL kernels; lrcn_comm_init is then optional.  LRCN_DP_NCCL=1 keeps NCCL. */
#define LRCN_P2P_BLOB_BYTES 512
LRCN_API int lrcn_p2p_export(lrcn_handle* h, char blob[LRCN_P2P_BLOB_BYTES]);
LRCN_API int lrcn_p2p_import(lrcn_handle* h, const char* blobs /* nranks x LRCN_P2P_BLOB_BYTES, rank order */, int rank, int nranks);

/* ---- measurement helpers: CUDA events on the library's own compute stream */
LRCN_API int lrcn_sync(lrcn_handle* h);
LRCN_API int lrcn_timer_start(lrcn_handle* h);
LRCN_API int lrcn_timer_stop(lrcn_handle* h, float* ms_out);
LRCN_API int lrcn_kernel_launches(lrcn_handle* h, int64_t* n_out); /* kernels launched (incl. inside graph replays) */
LRCN_API int lrcn_flush_l2(lrcn_handle* h);
/* LRCN_SEQ_TRACE=1 at create: [T][8] globaltimer (ns) stamps of CTA (0,0) of the layer-2 forward sequence kernel */
LRCN_API int lrcn_get_trace(lrcn_handle* h, uint64_t* out, int64_t n);                        /* writes a 256 MiB scratch buffer */
/* time `reps` launches of one named kernel family on the current buffers: "adam", "vocab_gemm", "gather" ... */
LRCN_API int lrcn_time_kernel(lrcn_handle* h, const char* name, int reps, float* avg_ms_out, double* algo_bytes_out,
                     double* algo_flops_out);

#ifdef __cplusplus
}
#endif
#endif /* LRCN_B200_H */
