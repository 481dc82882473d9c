// cnn_sm100.cu -- fc7 feature producer (SURVEY 8 row f-4): VGG-16 forward up to relu7 behind lrcn_extract_features.
// Replaces get_params_cnn / get_convnet / extract_features (lrcn.jl:190-221, 697-773).
//
// Every layer is one GEMM: C[M = pixels][N = Cout] = A[M][Kp] * W[Cout][Kp]^T + bias, with the existing gemm_bf16x3
// (tcgen05, bf16 hi/lo operands) or sgemm (fp32 mode).  What this file adds is the CUDA that feeds those GEMMs:
//   - the filters relaid K-major, W[o][(ky, kx, c)] with c fastest, zero-padded to Kp (a multiple of 8: the TMA pitch);
//   - one gather kernel per layer writing the zero-padded patch rows A (explicit im2col).  It reads the previous layer's
//     raw (pre-ReLU) fp32 GEMM output and applies that layer's ReLU and, where VGG has one, the 2x2 max-pool on the fly
//     (max of ReLU = ReLU of max).  conv1_1 reads the planar host image layout directly (K = 27 padded to 32); fc6's
//     gather is pool + ReLU + flatten of the 7x7x512 map (fc6 is a 7x7 convolution), fc7's is ReLU (+ split);
//   - the tail: relu7 and the optional per-image L1 normalisation, summed in a fixed order (deterministic).
// Pixel order inside a chunk: m = (i * W + x) * H + y (y fastest, like the column-major images), so every activation is
// [m][Cout] fp32.  Images run in chunks of CH; each layer keeps its own output buffer (the test hook reads any layer).
#include "lrcn_internal.h"

#include <algorithm>

namespace {

constexpr int NL = LRCN_CNN_LAYERS;
constexpr int CH = 16;  // images per chunk: conv1_2's patch matrix is then 16 * 224^2 x 576 fp32 = 1.85 GB
constexpr int IMG = LRCN_CNN_IMAGE;
constexpr int64_t IMG_ELEMS = (int64_t)3 * IMG * IMG;
constexpr int kCin[NL] = {3, 64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512, 512, 4096};
constexpr int kCout[NL] = {64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512, 512, 4096, 4096};
constexpr int kPoolIn[NL] = {0, 0, 1, 0, 1, 0, 0, 1, 0, 0, 1, 0, 0, 1, 0};  // input = 2x2 max-pool of the previous output

}  // namespace

struct CnnLayer {
  int cin, cout, k, pad;
  int hprev;  // spatial size of the previous layer's output (of the image for conv1_1)
  int pool;   // the input is the 2x2 max-pool of that output
  int hin, hout;
  int K, Kp;
};

struct CnnState {
  CnnLayer L[NL];
  size_t woff[NL], boff[NL];
  float* w = nullptr;  // [Cout][Kp] per layer, K-major
  bf16 *w_hi = nullptr, *w_lo = nullptr;
  float* b = nullptr;
  bool set[NL][2] = {};
  float* act[NL] = {};            // pre-ReLU output of every layer for one chunk: [CH * hout^2][Cout]
  void* patch = nullptr;          // fp32 [M][Kp], or bf16 hi [M][Kp] | lo [M][Kp]; also the raw-filter scratch of set / get
  size_t patch_elems = 0;
  float* img[2] = {};             // double-buffered chunk of images
  float* feat[2] = {};            // double-buffered relu7 rows of a chunk
  float* h_img[2] = {};           // pinned staging of host images
  cudaStream_t copy = nullptr;    // uploads from pinned staging, downloads of the features
  cudaEvent_t ev_read[2] = {}, ev_up[2] = {}, ev_feat[2] = {}, ev_copied[2] = {};
  int64_t last_n = 0, last_chunks = 0;  // images and chunks of the last extraction
};

namespace {

void build_layers(CnnLayer* L) {
  int h = IMG;
  for (int l = 0; l < NL; l++) {
    CnnLayer& y = L[l];
    y.cin = kCin[l]; y.cout = kCout[l];
    y.k = l < 13 ? 3 : (l == 13 ? 7 : 1);
    y.pad = l < 13 ? 1 : 0;
    y.hprev = h; y.pool = kPoolIn[l];
    y.hin = y.pool ? h / 2 : h;
    y.hout = y.hin + 2 * y.pad - y.k + 1;
    y.K = y.k * y.k * y.cin;
    y.Kp = (y.K + 7) / 8 * 8;
    h = y.hout;
  }
}

inline void count_launch() { if (g_counter) g_counter->n++; }
inline int grid_for(int64_t items) {
  const int64_t b = (items + 255) / 256;
  return (int)(b < 148 * 32 ? b : 148 * 32);
}

__device__ __forceinline__ void store8(float* f, bf16* hi, bf16* lo, size_t o, const float (&v)[8]) {
  if (hi) {
    __align__(16) bf16 h[8], l[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      h[j] = __float2bfloat16_rn(v[j]);
      l[j] = __float2bfloat16_rn(v[j] - __bfloat162float(h[j]));
    }
    *reinterpret_cast<uint4*>(hi + o) = *reinterpret_cast<const uint4*>(h);
    *reinterpret_cast<uint4*>(lo + o) = *reinterpret_cast<const uint4*>(l);
  } else {
    *reinterpret_cast<float4*>(f + o) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(f + o + 4) = make_float4(v[4], v[5], v[6], v[7]);
  }
}
__device__ __forceinline__ void max8(float (&v)[8], const float* p) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p + 4));
  v[0] = fmaxf(v[0], a.x); v[1] = fmaxf(v[1], a.y); v[2] = fmaxf(v[2], a.z); v[3] = fmaxf(v[3], a.w);
  v[4] = fmaxf(v[4], b.x); v[5] = fmaxf(v[5], b.y); v[6] = fmaxf(v[6], b.z); v[7] = fmaxf(v[7], b.w);
}

// conv1_1's patch rows straight from the planar images: one thread per output pixel writes its 32 columns
// (27 taps x channels in (ky, kx, c) order + 5 zeros)
__global__ void __launch_bounds__(256) cnn_gather_image_kernel(const float* __restrict__ img, int n_pix, float* __restrict__ f,
                                                               bf16* __restrict__ hi, bf16* __restrict__ lo) {
  for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < n_pix; m += gridDim.x * blockDim.x) {
    const int y = m % IMG, x = (m / IMG) % IMG, i = m / (IMG * IMG);
    const float* src = img + (size_t)i * IMG_ELEMS;
    float v[32];
#pragma unroll
    for (int tap = 0; tap < 9; tap++) {
      const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
      const bool in = yy >= 0 && yy < IMG && xx >= 0 && xx < IMG;
#pragma unroll
      for (int c = 0; c < 3; c++) v[tap * 3 + c] = in ? __ldg(src + (size_t)c * IMG * IMG + (size_t)xx * IMG + yy) : 0.f;
    }
#pragma unroll
    for (int j = 27; j < 32; j++) v[j] = 0.f;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      float w8[8];
#pragma unroll
      for (int j = 0; j < 8; j++) w8[j] = v[q * 8 + j];
      store8(f, hi, lo, (size_t)m * 32 + q * 8, w8);
    }
  }
}

// patch rows of layers 2..15: item t = ((m * k*k + tap) * Cin/8 + c8), 8 channels per thread (128-bit loads / stores).
// src: the previous layer's raw output [pixels][Cin] at hprev x hprev; the value read is ReLU(x) or ReLU(max of the 2x2
// window) at input position (y + ky - pad, x + kx - pad) of the hin x hin input, zero outside.
template <bool POOL>
__global__ void __launch_bounds__(256) cnn_gather_kernel(const float* __restrict__ src, int hprev, int hin, int k, int pad, int hout, int cin,
                                                         int n_items, int Kp, float* __restrict__ f, bf16* __restrict__ hi,
                                                         bf16* __restrict__ lo) {
  const unsigned c8n = (unsigned)cin >> 3, kk = (unsigned)(k * k);
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < (unsigned)n_items; t += gridDim.x * blockDim.x) {
    const unsigned c8 = t % c8n, r = t / c8n;
    const unsigned tap = r % kk, m = r / kk;
    const unsigned y = m % (unsigned)hout, r2 = m / (unsigned)hout;
    const unsigned x = r2 % (unsigned)hout, i = r2 / (unsigned)hout;
    const int yy = (int)y + (int)(tap / k) - pad, xx = (int)x + (int)(tap % k) - pad;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (yy >= 0 && yy < hin && xx >= 0 && xx < hin) {
      if (POOL) {
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = -INFINITY;
        const size_t p = ((size_t)i * hprev + 2 * xx) * hprev + 2 * yy;  // (2yy, 2xx); +1 along y, +hprev along x
        const float* s = src + c8 * 8;
        max8(v, s + p * cin); max8(v, s + (p + 1) * cin);
        max8(v, s + (p + hprev) * cin); max8(v, s + (p + hprev + 1) * cin);
      } else {
        const size_t p = ((size_t)i * hprev + xx) * hprev + yy;
        max8(v, src + p * cin + c8 * 8);  // max with 0 = ReLU
      }
#pragma unroll
      for (int j = 0; j < 8; j++) v[j] = fmaxf(v[j], 0.f);
    }
    store8(f, hi, lo, (size_t)m * Kp + (size_t)tap * cin + c8 * 8, v);
  }
}

// relu7 and the optional L1 normalisation of one image per CTA (4096 = 256 threads x 16); fixed-order sum
__global__ void __launch_bounds__(256) cnn_relu7_kernel(const float* __restrict__ fc7, int l1, float* __restrict__ out) {
  __shared__ float red[256];
  const float* row = fc7 + (size_t)blockIdx.x * LRCN_F_CNN;
  float* orow = out + (size_t)blockIdx.x * LRCN_F_CNN;
  float4 v[4];
  float s = 0.f;
#pragma unroll
  for (int q = 0; q < 4; q++) {
    v[q] = __ldg(reinterpret_cast<const float4*>(row) + q * 256 + threadIdx.x);
    v[q].x = fmaxf(v[q].x, 0.f); v[q].y = fmaxf(v[q].y, 0.f); v[q].z = fmaxf(v[q].z, 0.f); v[q].w = fmaxf(v[q].w, 0.f);
    s += (v[q].x + v[q].y) + (v[q].z + v[q].w);
  }
  if (l1) {
    red[threadIdx.x] = s;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
      if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
      __syncthreads();
    }
    const float tot = red[0];
    if (tot > 0.f) {  // a zero sum means an all-zero row: it stays zero (the reference would divide 0 by 0)
#pragma unroll
      for (int q = 0; q < 4; q++) { v[q].x /= tot; v[q].y /= tot; v[q].z /= tot; v[q].w /= tot; }
    }
  }
#pragma unroll
  for (int q = 0; q < 4; q++) reinterpret_cast<float4*>(orow)[q * 256 + threadIdx.x] = v[q];
}

// raw filter (dy, dx, c, o) column-major -> W[o][(dy * k + dx) * cin + c], zero-padded to Kp, + bf16 hi/lo split
__global__ void cnn_pack_filter_kernel(const float* __restrict__ raw, int k, int cin, int cout, int Kp, float* __restrict__ w,
                                       bf16* __restrict__ hi, bf16* __restrict__ lo) {
  const size_t total = (size_t)cout * Kp, K = (size_t)k * k * cin;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const size_t o = t / Kp, kk = t % Kp;
    float v = 0.f;
    if (kk < K) {
      const size_t tap = kk / cin, c = kk % cin, dy = tap / k, dx = tap % k;
      v = raw[dy + (size_t)k * dx + (size_t)k * k * c + K * o];
    }
    w[t] = v;
    if (hi) {
      const bf16 h = __float2bfloat16_rn(v);
      hi[t] = h;
      lo[t] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
  }
}
__global__ void cnn_unpack_filter_kernel(const float* __restrict__ w, int k, int cin, int cout, int Kp, float* __restrict__ raw) {
  const size_t K = (size_t)k * k * cin, total = K * cout;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += (size_t)gridDim.x * blockDim.x) {
    const size_t dy = j % k, dx = (j / k) % k, c = (j / ((size_t)k * k)) % cin, o = j / K;
    raw[j] = w[o * Kp + (dy * k + dx) * cin + c];
  }
}

int check_tensor(int layer, int which, const void* data, const int64_t dims[4], CnnLayer* out) {
  if (layer < 1 || layer > NL) return fail(LRCN_ERR_ARG, "CNN layer %d outside [1,%d]", layer, NL);
  if (which != 0 && which != 1) return fail(LRCN_ERR_ARG, "which must be 0 (filter) or 1 (bias)");
  if (!data || !dims) return fail(LRCN_ERR_ARG, "null argument");
  CnnLayer L[NL];
  build_layers(L);
  const CnnLayer& y = L[layer - 1];
  const int64_t want[4] = {which ? y.cout : y.k, which ? 1 : y.k, which ? 1 : y.cin, which ? 1 : y.cout};
  for (int d = 0; d < 4; d++)
    if (dims[d] != want[d])
      return fail(LRCN_ERR_ARG, "CNN layer %d %s dims {%lld,%lld,%lld,%lld}, expected {%lld,%lld,%lld,%lld}", layer, which ? "bias" : "filter",
                  (long long)dims[0], (long long)dims[1], (long long)dims[2], (long long)dims[3], (long long)want[0], (long long)want[1],
                  (long long)want[2], (long long)want[3]);
  *out = y;
  return LRCN_OK;
}

// weights + workspace, on the first CNN call of the handle
int ensure(lrcn_handle* h) {
  if (h->cnn) return LRCN_OK;
  CnnState* s = new CnnState();
  h->cnn = s;
  build_layers(s->L);
  size_t wn = 0, bn = 0;
  for (int l = 0; l < NL; l++) {
    const CnnLayer& y = s->L[l];
    s->woff[l] = wn; wn += ((size_t)y.cout * y.Kp + 63) / 64 * 64;
    s->boff[l] = bn; bn += ((size_t)y.cout + 63) / 64 * 64;
    s->patch_elems = std::max(s->patch_elems, (size_t)CH * y.hout * y.hout * y.Kp);
  }
  CK(cudaMalloc(&s->w, wn * 4)); CK(cudaMemset(s->w, 0, wn * 4));
  if (h->bf16mode) {
    CK(cudaMalloc(&s->w_hi, wn * 2)); CK(cudaMalloc(&s->w_lo, wn * 2));
    CK(cudaMemset(s->w_hi, 0, wn * 2)); CK(cudaMemset(s->w_lo, 0, wn * 2));
  }
  CK(cudaMalloc(&s->b, bn * 4)); CK(cudaMemset(s->b, 0, bn * 4));
  for (int l = 0; l < NL; l++) CK(cudaMalloc(&s->act[l], (size_t)CH * s->L[l].hout * s->L[l].hout * s->L[l].cout * 4));
  CK(cudaMalloc(&s->patch, s->patch_elems * 4));  // fp32, or bf16 hi | lo
  for (int j = 0; j < 2; j++) {
    CK(cudaMalloc(&s->img[j], (size_t)CH * IMG_ELEMS * 4));
    CK(cudaMalloc(&s->feat[j], (size_t)CH * LRCN_F_CNN * 4));
    CK(cudaMallocHost(&s->h_img[j], (size_t)CH * IMG_ELEMS * 4));
    for (cudaEvent_t* e : {&s->ev_read[j], &s->ev_up[j], &s->ev_feat[j], &s->ev_copied[j]}) CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  CK(cudaStreamCreateWithFlags(&s->copy, cudaStreamNonBlocking));
  return LRCN_OK;
}

struct PatchPtrs { float* f; bf16* hi; bf16* lo; };
PatchPtrs patch_ptrs(const lrcn_handle* h) {
  const CnnState* s = h->cnn;
  if (!h->bf16mode) return {static_cast<float*>(s->patch), nullptr, nullptr};
  bf16* hi = static_cast<bf16*>(s->patch);
  return {nullptr, hi, hi + s->patch_elems};
}

// gathers + GEMMs of all 15 layers for nc images in `img`; records ev_read once conv1_1 has consumed them
int run_chunk(lrcn_handle* h, const float* img, int nc, cudaEvent_t ev_read) {
  CnnState* s = h->cnn;
  const PatchPtrs P = patch_ptrs(h);
  for (int l = 0; l < NL; l++) {
    const CnnLayer& y = s->L[l];
    const int M = nc * y.hout * y.hout;
    if (l == 0) {
      cnn_gather_image_kernel<<<grid_for(M), 256, 0, h->stream>>>(img, M, P.f, P.hi, P.lo);
      CK(cudaEventRecord(ev_read, h->stream));
    } else {
      const int64_t items = (int64_t)M * y.k * y.k * (y.cin / 8);  // < 2^31 for CH images (largest: conv1_2, 57.8 M)
      if (y.pool)
        cnn_gather_kernel<true><<<grid_for(items), 256, 0, h->stream>>>(s->act[l - 1], y.hprev, y.hin, y.k, y.pad, y.hout, y.cin, (int)items, y.Kp,
                                                                         P.f, P.hi, P.lo);
      else
        cnn_gather_kernel<false><<<grid_for(items), 256, 0, h->stream>>>(s->act[l - 1], y.hprev, y.hin, y.k, y.pad, y.hout, y.cin, (int)items, y.Kp,
                                                                          P.f, P.hi, P.lo);
    }
    count_launch();
    const float* bias = s->b + s->boff[l];
    if (h->bf16mode) {
      if (!gemm_bf16x3(h->stream, true, true, M, y.cout, y.Kp, P.hi, P.lo, y.Kp, s->w_hi + s->woff[l], s->w_lo + s->woff[l], y.Kp, s->act[l], y.cout,
                       false, bias, nullptr, nullptr))
        return fail(LRCN_ERR_CUDA, "CNN layer %d GEMM: %s", l + 1, gemm_bf16x3_last_error());
    } else {
      sgemm(h->stream, true, true, M, y.cout, y.Kp, P.f, y.Kp, s->w + s->woff[l], y.Kp, s->act[l], y.cout, false, bias);
    }
  }
  CK(cudaPeekAtLastError());
  return LRCN_OK;
}

}  // namespace

void cnn_free(lrcn_handle* h) {
  CnnState* s = h->cnn;
  if (!s) return;
  if (s->copy) cudaStreamSynchronize(s->copy);
  for (void* p : {(void*)s->w, (void*)s->w_hi, (void*)s->w_lo, (void*)s->b, s->patch}) if (p) cudaFree(p);
  for (float* p : s->act) if (p) cudaFree(p);
  for (int j = 0; j < 2; j++) {
    if (s->img[j]) cudaFree(s->img[j]);
    if (s->feat[j]) cudaFree(s->feat[j]);
    if (s->h_img[j]) cudaFreeHost(s->h_img[j]);
    for (cudaEvent_t e : {s->ev_read[j], s->ev_up[j], s->ev_feat[j], s->ev_copied[j]}) if (e) cudaEventDestroy(e);
  }
  if (s->copy) cudaStreamDestroy(s->copy);
  delete s;
  h->cnn = nullptr;
}

int cnn_set_param(lrcn_handle* h, int layer, int which, const float* data, const int64_t dims[4]) {
  CnnLayer y;
  int rc = check_tensor(layer, which, data, dims, &y);
  if (rc) return rc;
  CK(cudaSetDevice(h->cfg.device));
  g_counter = &h->counter;
  rc = ensure(h);
  if (rc) return rc;
  CnnState* s = h->cnn;
  const int l = layer - 1;
  if (which == 1) {
    CK(cudaMemcpyAsync(s->b + s->boff[l], data, (size_t)y.cout * 4, cudaMemcpyDefault, h->stream));
  } else {
    float* raw = static_cast<float*>(s->patch);  // idle between calls
    CK(cudaMemcpyAsync(raw, data, (size_t)y.K * y.cout * 4, cudaMemcpyDefault, h->stream));
    cnn_pack_filter_kernel<<<grid_for((int64_t)y.cout * y.Kp), 256, 0, h->stream>>>(raw, y.k, y.cin, y.cout, y.Kp, s->w + s->woff[l],
                                                                                   s->w_hi ? s->w_hi + s->woff[l] : nullptr,
                                                                                   s->w_lo ? s->w_lo + s->woff[l] : nullptr);
    count_launch();
  }
  CK(cudaStreamSynchronize(h->stream));
  s->set[l][which] = true;
  return LRCN_OK;
}

int cnn_get_param(lrcn_handle* h, int layer, int which, float* data, const int64_t dims[4]) {
  CnnLayer y;
  int rc = check_tensor(layer, which, data, dims, &y);
  if (rc) return rc;
  const int l = layer - 1;
  CnnState* s = h->cnn;
  if (!s || !s->set[l][which]) return fail(LRCN_ERR_STATE, "CNN layer %d %s was never set", layer, which ? "bias" : "filter");
  CK(cudaSetDevice(h->cfg.device));
  g_counter = &h->counter;
  if (which == 1) {
    CK(cudaMemcpyAsync(data, s->b + s->boff[l], (size_t)y.cout * 4, cudaMemcpyDefault, h->stream));
  } else {
    float* raw = static_cast<float*>(s->patch);
    cnn_unpack_filter_kernel<<<grid_for((int64_t)y.K * y.cout), 256, 0, h->stream>>>(s->w + s->woff[l], y.k, y.cin, y.cout, y.Kp, raw);
    count_launch();
    CK(cudaMemcpyAsync(data, raw, (size_t)y.K * y.cout * 4, cudaMemcpyDefault, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  return LRCN_OK;
}

int cnn_extract(lrcn_handle* h, const float* images, int64_t n, int flags, float* feats_out) {
  if (!images || !feats_out || n <= 0) return fail(LRCN_ERR_ARG, "bad argument to lrcn_extract_features");
  if (flags & ~LRCN_FEAT_L1) return fail(LRCN_ERR_ARG, "unknown flags 0x%x", flags);
  for (int l = 0; l < NL; l++)
    for (int j = 0; j < 2; j++)
      if (!h->cnn || !h->cnn->set[l][j])
        return fail(LRCN_ERR_STATE, "CNN layer %d %s not set: lrcn_set_cnn_param all 30 tensors first", l + 1, j ? "bias" : "filter");
  CK(cudaSetDevice(h->cfg.device));
  g_counter = &h->counter;
  CnnState* s = h->cnn;
  cudaPointerAttributes pa;
  CK(cudaPointerGetAttributes(&pa, images));
  const bool dev_images = pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged;
  const int64_t nch = (n + CH - 1) / CH;
  s->last_n = n;
  s->last_chunks = nch;
  auto rows = [&](int64_t c) { return (int)std::min<int64_t>(CH, n - c * CH); };
  // chunk c's images into img[c % 2].  Host images go through pinned staging on the copy stream, so the upload of chunk
  // c + 1 (and the host-side memcpy into the staging buffer) overlaps the compute of chunk c.
  auto stage = [&](int64_t c) -> int {
    const int j = (int)(c & 1);
    const size_t bytes = (size_t)rows(c) * IMG_ELEMS * 4;
    const float* src = images + c * CH * IMG_ELEMS;
    if (dev_images) {
      CK(cudaMemcpyAsync(s->img[j], src, bytes, cudaMemcpyDefault, h->stream));  // stream order: chunk c - 2 has read img[j]
      return LRCN_OK;
    }
    CK(cudaEventSynchronize(s->ev_up[j]));  // h_img[j]'s previous upload is done
    memcpy(s->h_img[j], src, bytes);
    CK(cudaStreamWaitEvent(s->copy, s->ev_read[j], 0));  // conv1_1 of chunk c - 2 has read img[j]
    CK(cudaMemcpyAsync(s->img[j], s->h_img[j], bytes, cudaMemcpyHostToDevice, s->copy));
    CK(cudaEventRecord(s->ev_up[j], s->copy));
    CK(cudaStreamWaitEvent(h->stream, s->ev_up[j], 0));
    return LRCN_OK;
  };
  // relu7 rows of chunk c: copy stream, after the tail kernel (overlaps chunk c + 1)
  auto download = [&](int64_t c) -> int {
    const int j = (int)(c & 1);
    CK(cudaStreamWaitEvent(s->copy, s->ev_feat[j], 0));
    CK(cudaMemcpyAsync(feats_out + c * CH * LRCN_F_CNN, s->feat[j], (size_t)rows(c) * LRCN_F_CNN * 4, cudaMemcpyDefault, s->copy));
    CK(cudaEventRecord(s->ev_copied[j], s->copy));
    return LRCN_OK;
  };
  int rc = stage(0);
  for (int64_t c = 0; c < nch && !rc; c++) {
    const int j = (int)(c & 1);
    rc = run_chunk(h, s->img[j], rows(c), s->ev_read[j]);
    if (rc) break;
    if (c >= 2) CK(cudaStreamWaitEvent(h->stream, s->ev_copied[j], 0));  // feat[j] of chunk c - 2 has been copied out
    cnn_relu7_kernel<<<rows(c), 256, 0, h->stream>>>(s->act[NL - 1], flags & LRCN_FEAT_L1, s->feat[j]);
    count_launch();
    CK(cudaPeekAtLastError());
    CK(cudaEventRecord(s->ev_feat[j], h->stream));
    if (c + 1 < nch) rc = stage(c + 1);
    if (!rc && c >= 1) rc = download(c - 1);
  }
  if (!rc) rc = download(nch - 1);
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaStreamSynchronize(s->copy));
  return rc;
}

int cnn_activation(lrcn_handle* h, int layer, float* out, int64_t n) {
  if (!out || layer < 1 || layer > NL) return fail(LRCN_ERR_ARG, "bad argument to lrcn_test_cnn_activation");
  CnnState* s = h->cnn;
  if (!s || s->last_chunks != 1) return fail(LRCN_ERR_STATE, "the last lrcn_extract_features call did not run exactly one chunk of <= %d images", CH);
  if (n != s->last_n) return fail(LRCN_ERR_ARG, "n = %lld, the last extraction had %lld images", (long long)n, (long long)s->last_n);
  CK(cudaSetDevice(h->cfg.device));
  const CnnLayer& y = s->L[layer - 1];
  const size_t hw = (size_t)y.hout * y.hout, C = y.cout;
  std::vector<float> t(hw * C * n);
  CK(cudaMemcpy(t.data(), s->act[layer - 1], t.size() * 4, cudaMemcpyDeviceToHost));
  // [m = i * hw + x * H + y][o]  ->  (y, x, o, i) at y + H x + H W o + H W C i: pixel index x * H + y is the same
  for (int64_t i = 0; i < n; i++)
    for (size_t p = 0; p < hw; p++)
      for (size_t o = 0; o < C; o++) out[(size_t)i * hw * C + o * hw + p] = t[((size_t)i * hw + p) * C + o];
  return LRCN_OK;
}
