// kernels_simt.cu -- CUDA-core kernels of the LRCN decoder path for sm_100a:
// fp32 GEMM (exact mode / odd shapes), gathers, LSTM cell fwd/bwd, softmax-CE, reductions,
// scatter-add, fused Adam (+bf16 hi/lo shadow refresh), beam-search selection kernels.
// Reference semantics: lrcn.jl:528-581 (lstm, lrcn, loss), :644-678 (beam_search), Knet Adam.
#include "kernels.cuh"

#include <stdlib.h>
#include <math.h>

namespace lrcn {

thread_local LaunchCounter* g_counter = nullptr;
static inline void count_launch() { if (g_counter) g_counter->n++; }

// ------------------------------------------------------------------------------------------
// dropout mask: counter-based hash (SplitMix64 finaliser) of (seed, site, element index)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t drop_hash24(uint64_t seed, uint32_t site, uint64_t idx) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (idx + 1) + 0xD1B54A32D192ED03ull * (uint64_t)(site + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (uint32_t)(z >> 40);
}
__device__ __forceinline__ float drop_scale(const StepScalars* sc, uint32_t site, uint64_t idx) {
  if (sc->drop_thresh == 0) return 1.0f;
  return drop_hash24(sc->seed, site, idx) >= sc->drop_thresh ? sc->keep_scale : 0.0f;
}

__device__ __forceinline__ void split_one(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
__device__ __forceinline__ void store_split4(__nv_bfloat16* hi, __nv_bfloat16* lo, size_t idx, float4 x) {
  __nv_bfloat16 h[4], l[4];
  split_one(x.x, h[0], l[0]); split_one(x.y, h[1], l[1]); split_one(x.z, h[2], l[2]); split_one(x.w, h[3], l[3]);
  *reinterpret_cast<uint2*>(hi + idx) = *reinterpret_cast<uint2*>(h);
  *reinterpret_cast<uint2*>(lo + idx) = *reinterpret_cast<uint2*>(l);
}

// ------------------------------------------------------------------------------------------
// fp32 GEMM, 64x64x32 tiles, 256 threads, 4x4 micro-tile, register-prefetched k-tiles, split-K
// ------------------------------------------------------------------------------------------
constexpr int GBM = 64, GBN = 64, GBK = 32, GPAD = 4;

template <bool KMAJOR>
__device__ __forceinline__ void load_tile_regs(const float* __restrict__ P, int ld, int mn0, int MN, int k0, int kend,
                                               int tid, float (&r)[8]) {
#pragma unroll
  for (int i = 0; i < 8; i++) {
    int idx = tid + i * 256;
    int mm, kk;
    if (KMAJOR) { int kq = idx & 7; mm = (idx >> 3) & 63; kk = (idx >> 9) * 8 + kq; }
    else        { mm = idx & 63; kk = idx >> 6; }
    int gm = mn0 + mm, gk = k0 + kk;
    float v = 0.f;
    if (gm < MN && gk < kend) v = KMAJOR ? __ldg(P + (size_t)gm * ld + gk) : __ldg(P + (size_t)gk * ld + gm);
    r[i] = v;
  }
}
template <bool KMAJOR>
__device__ __forceinline__ void store_tile_smem(float (*S)[GBM + GPAD], int tid, const float (&r)[8]) {
#pragma unroll
  for (int i = 0; i < 8; i++) {
    int idx = tid + i * 256;
    int mm, kk;
    if (KMAJOR) { int kq = idx & 7; mm = (idx >> 3) & 63; kk = (idx >> 9) * 8 + kq; }
    else        { mm = idx & 63; kk = idx >> 6; }
    S[kk][mm] = r[i];
  }
}

template <bool AK, bool BKM>
__global__ void __launch_bounds__(256) sgemm_kernel(int M, int N, int K, const float* __restrict__ A, int lda,
                                                    const float* __restrict__ B, int ldb, float* __restrict__ C, int ldc,
                                                    int beta, const float* __restrict__ bias, int kper) {
  __shared__ __align__(16) float As[GBK][GBM + GPAD];
  __shared__ __align__(16) float Bs[GBK][GBN + GPAD];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * GBM, n0 = blockIdx.x * GBN;
  const int kbeg = blockIdx.z * kper;
  const int kend = min(K, kbeg + kper);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
  float ra[8], rb[8];
  load_tile_regs<AK>(A, lda, m0, M, kbeg, kend, tid, ra);
  load_tile_regs<BKM>(B, ldb, n0, N, kbeg, kend, tid, rb);
  for (int k0 = kbeg; k0 < kend; k0 += GBK) {
    store_tile_smem<AK>(As, tid, ra);
    store_tile_smem<BKM>(Bs, tid, rb);
    __syncthreads();
    if (k0 + GBK < kend) {
      load_tile_regs<AK>(A, lda, m0, M, k0 + GBK, kend, tid, ra);
      load_tile_regs<BKM>(B, ldb, n0, N, k0 + GBK, kend, tid, rb);
    }
#pragma unroll
    for (int kk = 0; kk < GBK; kk++) {
      float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  const bool split = gridDim.z > 1;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    int gm = m0 + ty * 4 + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      int gn = n0 + tx * 4 + j;
      if (gn >= N) continue;
      float v = acc[i][j];
      float* c = C + (size_t)gm * ldc + gn;
      if (split) {
        if (blockIdx.z == 0 && bias) v += bias[gn];
        atomicAdd(c, v);  // C was pre-zeroed by the launcher when !beta
      } else {
        if (bias) v += bias[gn];
        if (beta) v += *c;
        *c = v;
      }
    }
  }
}

void sgemm(cudaStream_t s, bool a_kmajor, bool b_kmajor, int M, int N, int K, const float* A, int lda, const float* B,
           int ldb, float* C, int ldc, bool beta, const float* bias) {
  if (M <= 0 || N <= 0) return;
  int tm = (M + GBM - 1) / GBM, tn = (N + GBN - 1) / GBN;
  int tiles = tm * tn;
  int splits = 1;
  if (tiles < 148 && K >= 256) {
    splits = (296 + tiles - 1) / tiles;
    int maxs = K / 128;
    if (splits > maxs) splits = maxs;
    if (splits < 1) splits = 1;
    if (splits > 32) splits = 32;
  }
  int kper = ((K + splits - 1) / splits + GBK - 1) / GBK * GBK;
  if (kper <= 0) kper = GBK;
  splits = (K + kper - 1) / kper;
  if (splits < 1) splits = 1;
  if (splits > 1 && !beta) {
    if (ldc == N) cudaMemsetAsync(C, 0, (size_t)M * N * sizeof(float), s);
    else cudaMemset2DAsync(C, (size_t)ldc * sizeof(float), 0, (size_t)N * sizeof(float), M, s);
  }
  dim3 grid(tn, tm, splits);
  int b = beta ? 1 : 0;
  if (a_kmajor && b_kmajor) sgemm_kernel<true, true><<<grid, 256, 0, s>>>(M, N, K, A, lda, B, ldb, C, ldc, b, bias, kper);
  else if (a_kmajor && !b_kmajor) sgemm_kernel<true, false><<<grid, 256, 0, s>>>(M, N, K, A, lda, B, ldb, C, ldc, b, bias, kper);
  else if (!a_kmajor && b_kmajor) sgemm_kernel<false, true><<<grid, 256, 0, s>>>(M, N, K, A, lda, B, ldb, C, ldc, b, bias, kper);
  else sgemm_kernel<false, false><<<grid, 256, 0, s>>>(M, N, K, A, lda, B, ldb, C, ldc, b, bias, kper);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// gathers
// ------------------------------------------------------------------------------------------
__global__ void gather_features_kernel(const float4* __restrict__ table, const int* __restrict__ rows, float4* __restrict__ X,
                                       __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  int i = blockIdx.x;
  const float4* src = table + (size_t)rows[i] * 1024;
  float4* dst = X + (size_t)i * 1024;
  for (int j = threadIdx.x; j < 1024; j += blockDim.x) {
    float4 x = __ldg(src + j);
    dst[j] = x;
    if (hi) store_split4(hi, lo, ((size_t)i * 1024 + j) * 4, x);
  }
}
void gather_features(cudaStream_t s, const float* table, const int* rows, int B, float* X, __nv_bfloat16* hi, __nv_bfloat16* lo) {
  launch_pdl<2>(gather_features_kernel, dim3(B), dim3(256), 0, s, (const float4*)table, rows, (float4*)X, hi, lo);
  count_launch();
}

// K1 (north_star): vectorised, coalesced word-embedding gather.  One warp per output row: 128-bit loads of the [V][E]
// row-major table (a word vector is one contiguous row), 128-bit fp32 stores and packed 64-bit bf16x4 hi / lo stores; the
// dropout mask of lrcn.jl:542 is applied on the fly.  Scalar tail / unaligned pitches fall back to 32-bit accesses.
__global__ void __launch_bounds__(256) gather_embed_kernel(const float* __restrict__ W, const int* __restrict__ tok, int R, int E, int ldo,
                                                           float* __restrict__ out, const StepScalars* __restrict__ sc, int train,
                                                           __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= R) return;
  const float* src = W + (size_t)tok[r] * E;
  float* dst = out + (size_t)r * ldo;
  const bool drop = train && sc->drop_thresh != 0;
  const bool vec = ((E | ldo) & 3) == 0;  // rows of W, out and the shadows are then 16 B (8 B for bf16) aligned
  const int E4 = vec ? (E >> 2) : 0;
  for (int q = lane; q < E4; q += 32) {
    float4 x = __ldg(reinterpret_cast<const float4*>(src) + q);
    if (drop) {
      const uint64_t idx = (uint64_t)r * E + 4 * q;
      x.x *= drop_scale(sc, 0, idx); x.y *= drop_scale(sc, 0, idx + 1); x.z *= drop_scale(sc, 0, idx + 2); x.w *= drop_scale(sc, 0, idx + 3);
    }
    reinterpret_cast<float4*>(dst)[q] = x;
    if (hi) store_split4(hi, lo, (size_t)r * ldo + 4 * q, x);
  }
  for (int e = 4 * E4 + lane; e < E; e += 32) {
    float v = __ldg(src + e);
    if (drop) v *= drop_scale(sc, 0, (uint64_t)r * E + e);
    dst[e] = v;
    if (hi) { __nv_bfloat16 h, l; split_one(v, h, l); hi[(size_t)r * ldo + e] = h; lo[(size_t)r * ldo + e] = l; }
  }
}
void gather_embed(cudaStream_t s, const float* WembT, const int* tok, int R, int E, float* out, const StepScalars* sc,
                  bool train, __nv_bfloat16* hi, __nv_bfloat16* lo, int ldo) {
  launch_pdl<2>(gather_embed_kernel, dim3((R + 7) / 8), dim3(256), 0, s, WembT, tok, R, E, ldo > 0 ? ldo : E, out, sc, train ? 1 : 0, hi, lo);
  count_launch();
}

__global__ void z_finish_kernel(float* __restrict__ Z, const float* __restrict__ v, int ldv, int R, int B, int C, int ldz,
                                const StepScalars* __restrict__ sc, int train, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  int r = blockIdx.x;
  int i = B > 0 ? r % B : r / (-B);  // B<0: generation, image index = row / beam_width
  float* z = Z + (size_t)r * ldz;
  for (int j = threadIdx.x; j < 2 * C; j += blockDim.x) {
    float x = (j < C) ? z[j] : v[(size_t)i * ldv + (j - C)];
    if (train) x *= drop_scale(sc, 1, (uint64_t)r * 2 * C + j);
    z[j] = x;
    if (hi) { __nv_bfloat16 h, l; split_one(x, h, l); hi[(size_t)r * ldz + j] = h; lo[(size_t)r * ldz + j] = l; }
  }
}
// vectorised variant (C, ldz, ldv multiples of 4): one warp per row, 128-bit accesses, packed bf16x4 shadow stores
__global__ void __launch_bounds__(256) z_finish_vec_kernel(float* __restrict__ Z, const float* __restrict__ v, int ldv, int R, int B, int C, int ldz,
                                                           const StepScalars* __restrict__ sc, int train, __nv_bfloat16* __restrict__ hi,
                                                           __nv_bfloat16* __restrict__ lo) {
  pdl_wait();
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= R) return;
  const int i = B > 0 ? r % B : r / (-B);  // B<0: generation, image index = row / beam_width
  float* z = Z + (size_t)r * ldz;
  const bool drop = train && sc->drop_thresh != 0;
  const int C4 = C >> 2;
  for (int q = lane; q < 2 * C4; q += 32) {
    float4 x = q < C4 ? reinterpret_cast<const float4*>(z)[q] : __ldg(reinterpret_cast<const float4*>(v + (size_t)i * ldv) + (q - C4));
    if (drop) {
      const uint64_t idx = (uint64_t)r * 2 * C + 4 * q;
      x.x *= drop_scale(sc, 1, idx); x.y *= drop_scale(sc, 1, idx + 1); x.z *= drop_scale(sc, 1, idx + 2); x.w *= drop_scale(sc, 1, idx + 3);
    }
    if (q >= C4 || drop) reinterpret_cast<float4*>(z)[q] = x;
    if (hi) store_split4(hi, lo, (size_t)r * ldz + 4 * q, x);
  }
}
void z_finish(cudaStream_t s, float* Z, const float* v, int ldv, int R, int B, int C, const StepScalars* sc, bool train,
              __nv_bfloat16* hi, __nv_bfloat16* lo, int ldz) {
  const int ld = ldz > 0 ? ldz : 2 * C;
  if (((C | ld | ldv) & 3) == 0)
    launch_pdl<2>(z_finish_vec_kernel, dim3((R + 7) / 8), dim3(256), 0, s, Z, v, ldv, R, B, C, ld, sc, train ? 1 : 0, hi, lo);
  else
    launch_pdl<2>(z_finish_kernel, dim3(R), dim3(128), 0, s, Z, v, ldv, R, B, C, ld, sc, train ? 1 : 0, hi, lo);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// LSTM cell (lrcn.jl:528-538): gate column order [forget | ingate | outgate | change]
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float sigm_f(float x) { return 1.0f / (1.0f + expf(-x)); }

__global__ void lstm_cell_fwd_kernel(float* __restrict__ gates, const float* __restrict__ c_prev, float* __restrict__ c_out,
                                     float* __restrict__ h_out, int B, int H, __nv_bfloat16* __restrict__ h_hi,
                                     __nv_bfloat16* __restrict__ h_lo) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  int i = idx / H, j = idx - i * H;
  float* g = gates + (size_t)i * 4 * H;
  float f = sigm_f(g[j]), in = sigm_f(g[H + j]), o = sigm_f(g[2 * H + j]), ch = tanhf(g[3 * H + j]);
  float c = c_prev[idx] * f + in * ch;
  g[j] = f; g[H + j] = in; g[2 * H + j] = o; g[3 * H + j] = ch;
  c_out[idx] = c;
  const float hv = o * tanhf(c);
  h_out[idx] = hv;
  if (h_hi) { __nv_bfloat16 hh, ll; split_one(hv, hh, ll); h_hi[idx] = hh; h_lo[idx] = ll; }
}
// generation (bf16x3 mode, H % 4 == 0): 4 units per thread, fast sigmoid / tanh like the tcgen05 step kernels, and the gate
// activations are NOT written back (only training's backward pass needs them)
__device__ __forceinline__ float sigm_fast_f(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_fast_f(float x) {
  const float ax = fabsf(x), e = __expf(-2.0f * ax);
  return copysignf(__fdividef(1.0f - e, 1.0f + e), x);
}
__global__ void lstm_cell_gen_kernel(const float* __restrict__ gates, const float* __restrict__ c_prev, float* __restrict__ c_out,
                                     float* __restrict__ h_out, int B, int H, __nv_bfloat16* __restrict__ h_hi,
                                     __nv_bfloat16* __restrict__ h_lo) {
  const int H4 = H >> 2;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H4) return;
  const int i = idx / H4, j = 4 * (idx - i * H4);
  const float* g = gates + (size_t)i * 4 * H + j;
  const float4 gf = *reinterpret_cast<const float4*>(g), gi = *reinterpret_cast<const float4*>(g + H);
  const float4 go = *reinterpret_cast<const float4*>(g + 2 * H), gc = *reinterpret_cast<const float4*>(g + 3 * H);
  const float4 cp = *reinterpret_cast<const float4*>(c_prev + (size_t)i * H + j);
  const float xf[4] = {gf.x, gf.y, gf.z, gf.w}, xi[4] = {gi.x, gi.y, gi.z, gi.w}, xo[4] = {go.x, go.y, go.z, go.w}, xc[4] = {gc.x, gc.y, gc.z, gc.w};
  const float cpv[4] = {cp.x, cp.y, cp.z, cp.w};
  float c[4], hv[4];
  __nv_bfloat16 hh[4], ll[4];
#pragma unroll
  for (int e = 0; e < 4; e++) {
    c[e] = cpv[e] * sigm_fast_f(xf[e]) + sigm_fast_f(xi[e]) * tanh_fast_f(xc[e]);
    hv[e] = sigm_fast_f(xo[e]) * tanh_fast_f(c[e]);
    split_one(hv[e], hh[e], ll[e]);
  }
  const size_t o = (size_t)i * H + j;
  *reinterpret_cast<float4*>(c_out + o) = make_float4(c[0], c[1], c[2], c[3]);
  *reinterpret_cast<float4*>(h_out + o) = make_float4(hv[0], hv[1], hv[2], hv[3]);
  *reinterpret_cast<uint2*>(h_hi + o) = *reinterpret_cast<uint2*>(hh);
  *reinterpret_cast<uint2*>(h_lo + o) = *reinterpret_cast<uint2*>(ll);
}
void lstm_cell_gen(cudaStream_t s, const float* gates, const float* c_prev, float* c_out, float* h_out, int B, int H, __nv_bfloat16* h_hi,
                   __nv_bfloat16* h_lo) {
  const int n = B * (H / 4);
  lstm_cell_gen_kernel<<<(n + 255) / 256, 256, 0, s>>>(gates, c_prev, c_out, h_out, B, H, h_hi, h_lo);
  count_launch();
}
void lstm_cell_fwd(cudaStream_t s, float* gates, const float* c_prev, float* c_out, float* h_out, int B, int H, __nv_bfloat16* h_hi,
                   __nv_bfloat16* h_lo) {
  int n = B * H;
  lstm_cell_fwd_kernel<<<(n + 255) / 256, 256, 0, s>>>(gates, c_prev, c_out, h_out, B, H, h_hi, h_lo);
  count_launch();
}

__global__ void lstm_cell_bwd_kernel(float* __restrict__ gates, const float* __restrict__ c_prev, const float* __restrict__ c_cur,
                                     const float* __restrict__ dh_in, const float* __restrict__ dh_rec, float* __restrict__ dc,
                                     int first, int B, int H) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  int i = idx / H, j = idx - i * H;
  float* g = gates + (size_t)i * 4 * H;
  float f = g[j], in = g[H + j], o = g[2 * H + j], ch = g[3 * H + j];
  float dh = dh_in[idx];
  if (!first && dh_rec) dh += dh_rec[idx];
  float tc = tanhf(c_cur[idx]);
  float dcv = (first ? 0.f : dc[idx]) + dh * o * (1.f - tc * tc);
  float dO = dh * tc;
  float dF = dcv * c_prev[idx];
  float dI = dcv * ch;
  float dG = dcv * in;
  dc[idx] = dcv * f;
  g[j] = dF * f * (1.f - f);
  g[H + j] = dI * in * (1.f - in);
  g[2 * H + j] = dO * o * (1.f - o);
  g[3 * H + j] = dG * (1.f - ch * ch);
}
void lstm_cell_bwd(cudaStream_t s, float* gates, const float* c_prev, const float* c_cur, const float* dh_in,
                   const float* dh_rec, float* dc, bool first, int B, int H) {
  int n = B * H;
  lstm_cell_bwd_kernel<<<(n + 255) / 256, 256, 0, s>>>(gates, c_prev, c_cur, dh_in, dh_rec, dc, first ? 1 : 0, B, H);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// block reductions
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  v = (l < nw) ? red[l] : -INFINITY;
  return warp_max(v);
}
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  v = (l < nw) ? red[l] : 0.f;
  return warp_sum(v);
}

// ------------------------------------------------------------------------------------------
// softmax cross-entropy, one CTA per row (Knet logp(x,2), lrcn.jl:562-567 and its adjoint)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512) softmax_ce_kernel(float* __restrict__ logits, int ld, int V, const int* __restrict__ tgt,
                                                         float* __restrict__ rowlp, const StepScalars* __restrict__ sc, int train,
                                                         __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                                         double* __restrict__ total_out, unsigned int* __restrict__ done_ctr) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  extern __shared__ __align__(16) float row[];
  __shared__ float red[32];
  __shared__ double dred[16];
  __shared__ int is_last;
  const int r = blockIdx.x;
  float* a = logits + (size_t)r * ld;
  const int V4 = V >> 2;  // ld % 8 == 0 and the arena is 256 B aligned -> rows are 16 B aligned
  float mx = -INFINITY;
  for (int q = threadIdx.x; q < V4; q += blockDim.x) {
    const float4 x = *reinterpret_cast<const float4*>(a + 4 * q);
    *reinterpret_cast<float4*>(row + 4 * q) = x;
    mx = fmaxf(fmaxf(mx, fmaxf(x.x, x.y)), fmaxf(x.z, x.w));
  }
  for (int j = 4 * V4 + threadIdx.x; j < V; j += blockDim.x) { const float x = a[j]; row[j] = x; mx = fmaxf(mx, x); }
  mx = block_max(mx, red);
  float sum = 0.f;
  for (int j = threadIdx.x; j < V; j += blockDim.x) sum += expf(row[j] - mx);
  sum = block_sum(sum, red);
  const float lse = logf(sum);
  const int y = tgt[r];
  if (threadIdx.x == 0) rowlp[r] = (row[y] - mx) - lse;
  if (train) {
    const float inv = sc->inv_ntok;
    const size_t base = (size_t)r * ld;
    for (int q = threadIdx.x; q < (ld >> 2); q += blockDim.x) {
      float p[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int j = 4 * q + e;
        float v = 0.f;  // padding columns [V, ld) stay clean
        if (j < V) { v = expf((row[j] - mx) - lse); if (j == y) v -= 1.0f; v *= inv; }
        p[e] = v;
      }
      const float4 o = make_float4(p[0], p[1], p[2], p[3]);
      *reinterpret_cast<float4*>(a + 4 * q) = o;
      if (hi) store_split4(hi, lo, base + 4 * q, o);
    }
  }
  // the last CTA to finish sums the per-row log-probs in a FIXED order (deterministic fp64 total: lrcn.jl:567 `total +=`)
  if (total_out) {
    if (threadIdx.x == 0) {
      __threadfence();
      const unsigned int prev = atomicAdd(done_ctr, 1u);
      is_last = (prev == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
      __threadfence();
      double acc = 0.0;
      const int R = gridDim.x;
      for (int i = threadIdx.x; i < R; i += blockDim.x) acc += (double)__ldcg(rowlp + i);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if ((threadIdx.x & 31) == 0) dred[threadIdx.x >> 5] = acc;
      __syncthreads();
      if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += dred[w];
        *total_out = t;
        *done_ctr = 0u;
      }
    }
  }
}
void softmax_ce(cudaStream_t s, float* logits, int ld, int R, int V, const int* tgt, float* rowlp, const StepScalars* sc,
                bool train, __nv_bfloat16* hi, __nv_bfloat16* lo, double* total_out, unsigned int* done_ctr) {
  size_t smem = (size_t)ld * sizeof(float);
  launch_pdl<2>(softmax_ce_kernel, dim3(R), dim3(512), smem, s, logits, ld, V, tgt, rowlp, sc, train ? 1 : 0, hi, lo, total_out, done_ctr);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// Training variant for the bf16x3 mode: persistent CTAs walk over rows with the row in REGISTERS, write only the bf16
// hi/lo split of dA = (softmax - onehot)/N (the fp32 dA is never needed: both consumers are tcgen05 GEMMs) and keep the
// column sums of dA (= the output-bias gradient) in registers, so the separate 100 MB column-sum pass disappears.
// colpart [gridDim.x][ld] receives one partial column sum per CTA; a (tiny) colsum over those rows finishes dbout.
// ------------------------------------------------------------------------------------------
template <int NV4>
__global__ void __launch_bounds__(512, NV4 <= 4 ? 2 : 1)
softmax_ce_fused_kernel(const float* __restrict__ logits, int ld, int V, int R, const int* __restrict__ tgt, float* __restrict__ rowlp,
                        const StepScalars* __restrict__ sc, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                        float* __restrict__ colpart, double* __restrict__ total_out, unsigned int* __restrict__ done_ctr) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(16) float colacc[];  // [ld]: this CTA's column sums (each thread owns its columns: no races)
  __shared__ float red[32];
  __shared__ double dred[16];
  __shared__ int is_last;
  const int ld4 = ld >> 2;
  const float inv = sc->inv_ntok;
#pragma unroll
  for (int i = 0; i < NV4; i++) {
    const int q = threadIdx.x + 512 * i;
    if (q < ld4) *reinterpret_cast<float4*>(colacc + 4 * q) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // the next row is loaded while the current one goes through its two block reductions
  float4 xn[NV4];
  auto load_row = [&](int r) {
    const float* a = logits + (size_t)r * ld;
#pragma unroll
    for (int i = 0; i < NV4; i++) {
      const int q = threadIdx.x + 512 * i;
      xn[i] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      if (q < ld4) xn[i] = __ldcs(reinterpret_cast<const float4*>(a + 4 * q));
    }
  };
  if ((int)blockIdx.x < R) load_row(blockIdx.x);
  for (int r = blockIdx.x; r < R; r += gridDim.x) {
    float4 x[NV4];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < NV4; i++) {
      const int j = 4 * (threadIdx.x + 512 * i);  // padding columns [V, ld) do not take part
      x[i] = xn[i];
      if (j + 1 >= V) x[i].y = -INFINITY;
      if (j + 2 >= V) x[i].z = -INFINITY;
      if (j + 3 >= V) x[i].w = -INFINITY;
      if (j >= V) x[i].x = -INFINITY;
      mx = fmaxf(fmaxf(mx, fmaxf(x[i].x, x[i].y)), fmaxf(x[i].z, x[i].w));
    }
    if (r + (int)gridDim.x < R) load_row(r + gridDim.x);
    mx = block_max(mx, red);
    // One exponential per element: e = exp(x - max) is kept in registers and scaled by 1/sum afterwards.  This kernel is
    // instruction bound otherwise (two precise expf per element = 60 us for 26 M logits); __expf (ex2.approx) has ~1e-7
    // relative error, far inside the 1e-4 budget of the bf16x3 mode (the exact fp32 mode uses softmax_ce_kernel).
    const int y = tgt[r];
    float xy = 0.f;  // the target logit, if this thread owns it
    bool own_y = false;
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < NV4; i++) {
      const int j = 4 * (threadIdx.x + 512 * i);
      if (y >= j && y < j + 4) { own_y = true; xy = y == j ? x[i].x : (y == j + 1 ? x[i].y : (y == j + 2 ? x[i].z : x[i].w)); }
      x[i].x = __expf(x[i].x - mx); x[i].y = __expf(x[i].y - mx); x[i].z = __expf(x[i].z - mx); x[i].w = __expf(x[i].w - mx);
      sum += (x[i].x + x[i].y) + (x[i].z + x[i].w);
    }
    sum = block_sum(sum, red);
    if (own_y) rowlp[r] = (xy - mx) - logf(sum);
    const float scale = inv / sum;
    const size_t base = (size_t)r * ld;
#pragma unroll
    for (int i = 0; i < NV4; i++) {
      const int q = threadIdx.x + 512 * i;
      if (q < ld4) {
        const int j = 4 * q;
        float p[4] = {x[i].x * scale, x[i].y * scale, x[i].z * scale, x[i].w * scale};  // padding columns: exp(-inf) = 0
        if (own_y && y >= j && y < j + 4) p[y - j] -= inv;
        const float4 o = make_float4(p[0], p[1], p[2], p[3]);
        store_split4(hi, lo, base + 4 * q, o);
        float4 c = *reinterpret_cast<float4*>(colacc + 4 * q);
        c.x += o.x; c.y += o.y; c.z += o.z; c.w += o.w;
        *reinterpret_cast<float4*>(colacc + 4 * q) = c;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < NV4; i++) {
    const int q = threadIdx.x + 512 * i;
    if (q < ld4) *reinterpret_cast<float4*>(colpart + (size_t)blockIdx.x * ld + 4 * q) = *reinterpret_cast<float4*>(colacc + 4 * q);
  }
  if (total_out) {  // deterministic fp64 total of the row log-probs by the last CTA (as in softmax_ce_kernel)
    // rowlp[r] is written by whichever thread owns the target column: every thread's stores must be ordered before thread 0's
    // release (fence + atomic) below, or the last CTA may sum a stale row log-prob
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      const unsigned int prev = atomicAdd(done_ctr, 1u);
      is_last = (prev == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
      __threadfence();
      double t = 0.0;
      for (int i = threadIdx.x; i < R; i += blockDim.x) t += (double)__ldcg(rowlp + i);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if ((threadIdx.x & 31) == 0) dred[threadIdx.x >> 5] = t;
      __syncthreads();
      if (threadIdx.x == 0) {
        double tt = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) tt += dred[w];
        *total_out = tt;
        *done_ctr = 0u;
      }
    }
  }
}
bool softmax_ce_fused(cudaStream_t s, const float* logits, int ld, int R, int V, const int* tgt, float* rowlp, const StepScalars* sc,
                      __nv_bfloat16* hi, __nv_bfloat16* lo, float* colpart, int colpart_rows, float* dbias, double* total_out,
                      unsigned int* done_ctr) {
  const int nv4 = ((ld >> 2) + 511) / 512;
  if (nv4 > 8 || (ld & 3) || !hi || !colpart) return false;
  int grid = R < colpart_rows ? R : colpart_rows;
#define LRCN_SMX(NV) launch_pdl<2>(softmax_ce_fused_kernel<NV>, dim3(grid), dim3(512), (size_t)ld * sizeof(float), s, logits, ld, V, R, tgt, rowlp, sc, hi, lo, colpart, total_out, done_ctr)
  if (nv4 <= 2) LRCN_SMX(2);
  else if (nv4 <= 4) LRCN_SMX(4);
  else if (nv4 <= 6) { if (grid > colpart_rows / 2) grid = colpart_rows / 2; LRCN_SMX(6); }
  else { if (grid > colpart_rows / 2) grid = colpart_rows / 2; LRCN_SMX(8); }
#undef LRCN_SMX
  count_launch();
  colsum(s, colpart, ld, grid, V, dbias, true);  // dbias is zeroed at step start
  return true;
}

__global__ void reduce_sum_double_kernel(const float* __restrict__ x, int n, double* __restrict__ out) {
  __shared__ double red[256];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += (double)x[i];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0];
}
void reduce_sum_double(cudaStream_t s, const float* x, int n, double* out) {
  reduce_sum_double_kernel<<<1, 256, 0, s>>>(x, n, out);
  count_launch();
}

// out[n] (+)= sum_r A[r][n] ; block = 32 float4-columns x 8 row-lanes, grid.y splits rows (atomic combine)
__global__ void colsum_kernel(const float* __restrict__ A, int ld, int R, int N, float* __restrict__ out, int rows_per) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  __shared__ float4 red[8][33];
  const int n4 = blockIdx.x * 32 + threadIdx.x;  // float4 column
  const int n = 4 * n4;
  const int r0 = blockIdx.y * rows_per, r1 = min(R, r0 + rows_per);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (n < N) {
    const bool full = n + 4 <= N;
    for (int r = r0 + threadIdx.y; r < r1; r += 8) {
      const float* p = A + (size_t)r * ld + n;
      if (full) { const float4 x = *reinterpret_cast<const float4*>(p); acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w; }
      else { acc.x += p[0]; if (n + 1 < N) acc.y += p[1]; if (n + 2 < N) acc.z += p[2]; }
    }
  }
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && n < N) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 8; k++) { const float4 x = red[k][threadIdx.x]; t.x += x.x; t.y += x.y; t.z += x.z; t.w += x.w; }
    atomicAdd(out + n, t.x);
    if (n + 1 < N) atomicAdd(out + n + 1, t.y);
    if (n + 2 < N) atomicAdd(out + n + 2, t.z);
    if (n + 3 < N) atomicAdd(out + n + 3, t.w);
  }
}
// requires ld % 4 == 0 and a 16-byte aligned A (all workspace matrices are)
void colsum(cudaStream_t s, const float* A, int ld, int R, int N, float* out, bool accumulate) {
  if (!accumulate) cudaMemsetAsync(out, 0, (size_t)N * sizeof(float), s);
  int gx = ((N + 3) / 4 + 31) / 32;
  int gy = 1;
  while (gx * gy < 592 && gy * 32 < R) gy *= 2;
  int rows_per = (R + gy - 1) / gy;
  launch_pdl<2>(colsum_kernel, dim3(gx, gy), dim3(32, 8), 0, s, A, ld, R, N, out, rows_per);
  count_launch();
}

__global__ void dz_finish_kernel(float* __restrict__ dZ, float* __restrict__ dv, int ldv, int T, int B, int C,
                                 const StepScalars* __restrict__ sc, int train, __nv_bfloat16* __restrict__ z_hi,
                                 __nv_bfloat16* __restrict__ z_lo, __nv_bfloat16* __restrict__ v_hi, __nv_bfloat16* __restrict__ v_lo) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  const int i = blockIdx.x;                                // batch row
  const int j = blockIdx.y * blockDim.x + threadIdx.x;     // column of Z
  if (j >= 2 * C) return;
  float acc = 0.f;
#pragma unroll 4
  for (int t = 0; t < T; t++) {
    const size_t idx = ((size_t)t * B + i) * 2 * C + j;
    float x = dZ[idx];
    if (train) { x *= drop_scale(sc, 1, (uint64_t)idx); dZ[idx] = x; }
    if (z_hi) { __nv_bfloat16 h, l; split_one(x, h, l); z_hi[idx] = h; z_lo[idx] = l; }
    acc += x;
  }
  if (j >= C) {
    dv[(size_t)i * ldv + (j - C)] = acc;
    if (v_hi) { __nv_bfloat16 h, l; split_one(acc, h, l); v_hi[(size_t)i * ldv + (j - C)] = h; v_lo[(size_t)i * ldv + (j - C)] = l; }
  }
}
// vectorised variant (C, ldv multiples of 4): a thread owns 4 columns of one batch row and walks the T steps with all loads of
// a group of steps in flight (the scalar kernel serialised T dependent load -> store round trips per thread)
__global__ void __launch_bounds__(128) dz_finish_vec_kernel(float* __restrict__ dZ, float* __restrict__ dv, int ldv, int T, int B, int C,
                                                            const StepScalars* __restrict__ sc, int train, __nv_bfloat16* __restrict__ z_hi,
                                                            __nv_bfloat16* __restrict__ z_lo, __nv_bfloat16* __restrict__ v_hi, __nv_bfloat16* __restrict__ v_lo) {
  pdl_wait();
  pdl_trigger();
  const int i = blockIdx.x;                                      // batch row
  const int q = blockIdx.y * blockDim.x + threadIdx.x;           // float4 column of Z
  if (q >= (2 * C) >> 2) return;
  const bool drop = train && sc->drop_thresh != 0;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  constexpr int U = 4;
  for (int t0 = 0; t0 < T; t0 += U) {
    float4 x[U];
#pragma unroll
    for (int u = 0; u < U; u++)
      if (t0 + u < T) x[u] = reinterpret_cast<const float4*>(dZ + ((size_t)(t0 + u) * B + i) * 2 * C)[q];
#pragma unroll
    for (int u = 0; u < U; u++) {
      if (t0 + u >= T) break;
      const size_t idx = ((size_t)(t0 + u) * B + i) * 2 * C + 4 * q;
      if (drop) {
        x[u].x *= drop_scale(sc, 1, idx); x[u].y *= drop_scale(sc, 1, idx + 1); x[u].z *= drop_scale(sc, 1, idx + 2); x[u].w *= drop_scale(sc, 1, idx + 3);
        *reinterpret_cast<float4*>(dZ + idx) = x[u];
      }
      if (z_hi) store_split4(z_hi, z_lo, idx, x[u]);
      acc.x += x[u].x; acc.y += x[u].y; acc.z += x[u].z; acc.w += x[u].w;
    }
  }
  const int j = 4 * q;
  if (j >= C) {
    *reinterpret_cast<float4*>(dv + (size_t)i * ldv + (j - C)) = acc;
    if (v_hi) store_split4(v_hi, v_lo, (size_t)i * ldv + (j - C), acc);
  }
}
void dz_finish(cudaStream_t s, float* dZ, float* dv, int ldv, int T, int B, int C, const StepScalars* sc, bool train,
               __nv_bfloat16* z_hi, __nv_bfloat16* z_lo, __nv_bfloat16* v_hi, __nv_bfloat16* v_lo) {
  if (((C | ldv) & 3) == 0) {
    dim3 grid(B, ((2 * C) / 4 + 127) / 128);
    launch_pdl<2>(dz_finish_vec_kernel, grid, dim3(128), 0, s, dZ, dv, ldv, T, B, C, sc, train ? 1 : 0, z_hi, z_lo, v_hi, v_lo);
  } else {
    dim3 grid(B, (2 * C + 127) / 128);
    launch_pdl<2>(dz_finish_kernel, grid, dim3(128), 0, s, dZ, dv, ldv, T, B, C, sc, train ? 1 : 0, z_hi, z_lo, v_hi, v_lo);
  }
  count_launch();
}

__global__ void scatter_add_embed_kernel(float* __restrict__ dW, const int* __restrict__ tok, const float* __restrict__ dE, int R,
                                         int E, const StepScalars* __restrict__ sc, int train) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  int r = blockIdx.x;
  float* dst = dW + (size_t)tok[r] * E;
  const float* src = dE + (size_t)r * E;
  for (int e = threadIdx.x; e < E; e += blockDim.x) {
    float v = src[e];
    if (train) v *= drop_scale(sc, 0, (uint64_t)r * E + e);
    atomicAdd(dst + e, v);
  }
}
void scatter_add_embed(cudaStream_t s, float* dWembT, const int* tok, const float* dE, int R, int E, const StepScalars* sc,
                       bool train) {
  launch_pdl<2>(scatter_add_embed_kernel, dim3(R), dim3(128), 0, s, dWembT, tok, dE, R, E, sc, train ? 1 : 0);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// fused Adam over the flat parameter arena (Knet Adam defaults; dense over every element)
// ------------------------------------------------------------------------------------------
// CLIP: g is scaled by its tensor's clip factor (grad_sqnorm) first -- one fp32 multiply, exact when the factor is 1.  The clip
// map is the LAST parameter so that the CLIP = false instantiation compiles to the kernel without it.
template <bool SPLIT, bool CLIP>
__global__ void __launch_bounds__(256) adam_kernel(float4* __restrict__ w, const float4* __restrict__ g, float4* __restrict__ m,
                                                   float4* __restrict__ v, size_t n4, const StepScalars* __restrict__ sc,
                                                   __nv_bfloat16* __restrict__ w_hi, __nv_bfloat16* __restrict__ w_lo, ClipMap cm) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  const float b1 = sc->beta1, b2 = sc->beta2, lr = sc->lr, eps = sc->eps, d1 = sc->adam_d1, d2 = sc->adam_d2;
  const float ob1 = sc->one_m_beta1, ob2 = sc->one_m_beta2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 W = w[i], G = __ldg(g + i), Mv = m[i], Vv = v[i];
    if (CLIP) {
      int k = cm.k[0];  // the tensor holding float4 i (constant indices: the map stays in the parameter bank)
#pragma unroll
      for (int t = 0; t < 8; t++) if (t + 1 < cm.n && i >= cm.end4[t]) k = cm.k[t + 1];
      const float s = __ldg(cm.scale + k);
      G.x = __fmul_rn(G.x, s); G.y = __fmul_rn(G.y, s); G.z = __fmul_rn(G.z, s); G.w = __fmul_rn(G.w, s);
    }
    float* wp = reinterpret_cast<float*>(&W);
    const float* gp = reinterpret_cast<const float*>(&G);
    float* mp = reinterpret_cast<float*>(&Mv);
    float* vp = reinterpret_cast<float*>(&Vv);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      float mm = __fadd_rn(__fmul_rn(b1, mp[k]), __fmul_rn(ob1, gp[k]));
      float vv = __fadd_rn(__fmul_rn(b2, vp[k]), __fmul_rn(ob2, __fmul_rn(gp[k], gp[k])));
      float mh = __fdiv_rn(mm, d1);
      float vh = __fdiv_rn(vv, d2);
      float upd = __fdiv_rn(mh, __fadd_rn(__fsqrt_rn(vh), eps));
      wp[k] = __fsub_rn(wp[k], __fmul_rn(lr, upd));
      mp[k] = mm; vp[k] = vv;
    }
    w[i] = W; m[i] = Mv; v[i] = Vv;
    if (SPLIT) {
      __nv_bfloat16 h[4], l[4];
#pragma unroll
      for (int k = 0; k < 4; k++) split_one(wp[k], h[k], l[k]);
      *reinterpret_cast<uint2*>(w_hi + 4 * i) = *reinterpret_cast<uint2*>(h);
      *reinterpret_cast<uint2*>(w_lo + 4 * i) = *reinterpret_cast<uint2*>(l);
    }
  }
}
void adam_flat(cudaStream_t s, float* w, const float* g, float* m, float* v, size_t n, const StepScalars* sc,
               __nv_bfloat16* w_hi, __nv_bfloat16* w_lo, const ClipMap* clip) {
  size_t n4 = n / 4;  // arena sizes are padded to multiples of 4
  int grid = 148 * 8;
  const ClipMap cm = clip ? *clip : ClipMap{};
#define LRCN_ADAM(SPLIT, CLIP) launch_pdl<2>(adam_kernel<SPLIT, CLIP>, dim3(grid), dim3(256), 0, s, (float4*)w, (const float4*)g, (float4*)m, \
                                             (float4*)v, n4, sc, SPLIT ? w_hi : (__nv_bfloat16*)nullptr, SPLIT ? w_lo : (__nv_bfloat16*)nullptr, cm)
  if (w_hi) { if (clip) LRCN_ADAM(true, true); else LRCN_ADAM(true, false); }
  else { if (clip) LRCN_ADAM(false, true); else LRCN_ADAM(false, false); }
#undef LRCN_ADAM
  count_launch();
}

// Adam on an arena range with a bounded grid and no PDL attribute: a bucket of the step's update, launched on a side stream under
// the rest of the backward pass (lrcn_api.cu)
void adam_range(cudaStream_t s, float* w, const float* g, float* m, float* v, size_t n, const StepScalars* sc, __nv_bfloat16* w_hi,
                __nv_bfloat16* w_lo, int grid, const ClipMap* clip) {
  const size_t n4 = n / 4;
  if (n4 == 0) return;
  const ClipMap cm = clip ? *clip : ClipMap{};
#define LRCN_ADAM(SPLIT, CLIP) adam_kernel<SPLIT, CLIP><<<grid, 256, 0, s>>>((float4*)w, (const float4*)g, (float4*)m, (float4*)v, n4, sc, \
                                                                            SPLIT ? w_hi : (__nv_bfloat16*)nullptr, SPLIT ? w_lo : (__nv_bfloat16*)nullptr, cm)
  if (w_hi) { if (clip) LRCN_ADAM(true, true); else LRCN_ADAM(true, false); }
  else { if (clip) LRCN_ADAM(false, true); else LRCN_ADAM(false, false); }
#undef LRCN_ADAM
  count_launch();
}

// ------------------------------------------------------------------------------------------
// per-tensor gradient norms for Knet's gclip (kernels.cuh: grad_sqnorm).  CTAs walk the range's 16 Ki-float chunks; a chunk's
// partial sum of squares (fp64) is reduced in a fixed order by whichever CTA takes it, and the last CTA (atomic ticket) sums each
// tensor's partials in a fixed order: the norms are bit-identical for any grid and any grouping of tensors into launches.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int gnorm_chunks(size_t nel) { return (int)(((nel + 3) / 4 + GNORM_CHUNK4 - 1) / GNORM_CHUNK4); }

__global__ void __launch_bounds__(256) grad_sqnorm_kernel(const float4* __restrict__ g, TensorRange r, double* __restrict__ part,
                                                          double* __restrict__ norm, float* __restrict__ scale,
                                                          unsigned int* __restrict__ ticket, const StepScalars* __restrict__ sc, int total) {
  __shared__ double red[8];
  __shared__ bool last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c = blockIdx.x; c < total; c += gridDim.x) {
    int j = 0, q = c;
    while (q >= gnorm_chunks(r.nel[j])) { q -= gnorm_chunks(r.nel[j]); j++; }
    const size_t nel = r.nel[j], n4 = (nel + 3) / 4, b = (size_t)q * GNORM_CHUNK4;
    const size_t e = b + GNORM_CHUNK4 < n4 ? b + GNORM_CHUNK4 : n4;
    const float4* p = g + r.off4[j];
    // all 16 loads of a thread in flight at once; then the sum in chunk order (a float4 past the chunk's end adds +0: exact)
    constexpr int PER = GNORM_CHUNK4 / 256;
    float4 x[PER];
#pragma unroll
    for (int u = 0; u < PER; u++) {
      const size_t i = b + threadIdx.x + 256 * u;
      x[u] = i < e ? __ldg(p + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < e && 4 * i + 4 > nel) {  // the tensor's last float4: ignore the padding
        if (4 * i + 1 >= nel) x[u].y = 0.f;
        if (4 * i + 2 >= nel) x[u].z = 0.f;
        if (4 * i + 3 >= nel) x[u].w = 0.f;
      }
    }
    double acc = 0.0;
#pragma unroll
    for (int u = 0; u < PER; u++) {
      acc += (double)x[u].x * x[u].x; acc += (double)x[u].y * x[u].y; acc += (double)x[u].z * x[u].z; acc += (double)x[u].w * x[u].w;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < 8; k++) s += red[k];
      part[r.chunk0[j] + q] = s;
    }
    __syncthreads();
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  for (int j = warp; j < r.n; j += 8) {  // one warp per tensor: lane-strided partials, then a fixed butterfly
    const int nch = gnorm_chunks(r.nel[j]);
    double s = 0.0;
    for (int q = lane; q < nch; q += 32) s += __ldcg(part + r.chunk0[j] + q);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      const double nrm = sqrt(s), gclip = sc->gclip;
      norm[r.k[j]] = nrm;
      scale[r.k[j]] = gclip > 0.0 && nrm > gclip ? (float)(gclip / nrm) : 1.0f;
    }
  }
  if (threadIdx.x == 0) *ticket = 0u;  // ready for the next launch (graph replay)
}
void grad_sqnorm(cudaStream_t s, const float* g, const TensorRange& r, double* part, double* norm, float* scale, unsigned int* ticket,
                 const StepScalars* sc, int grid_cap) {
  int total = 0;
  for (int j = 0; j < r.n; j++) total += (int)(((r.nel[j] + 3) / 4 + GNORM_CHUNK4 - 1) / GNORM_CHUNK4);
  const int grid = total < grid_cap ? total : grid_cap;
  grad_sqnorm_kernel<<<grid, 256, 0, s>>>((const float4*)g, r, part, norm, scale, ticket, sc, total);
  count_launch();
}

__global__ void split_bf16_kernel(const float4* __restrict__ x, size_t n4, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 X = __ldg(x + i);
    const float* xp = reinterpret_cast<const float*>(&X);
    __nv_bfloat16 h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; k++) split_one(xp[k], h[k], l[k]);
    *reinterpret_cast<uint2*>(hi + 4 * i) = *reinterpret_cast<uint2*>(h);
    *reinterpret_cast<uint2*>(lo + 4 * i) = *reinterpret_cast<uint2*>(l);
  }
}
void split_bf16(cudaStream_t s, const float* x, size_t n, __nv_bfloat16* hi, __nv_bfloat16* lo) {
  size_t n4 = (n + 3) / 4;  // buffers are padded to multiples of 64 elements
  if (n4 == 0) return;
  size_t want = (n4 + 255) / 256;
  int grid = (int)(want < (size_t)148 * 8 ? want : (size_t)148 * 8);
  split_bf16_kernel<<<grid, 256, 0, s>>>((const float4*)x, n4, hi, lo);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// batch staging on the device (row f-1)
// ------------------------------------------------------------------------------------------
__global__ void epoch_lookup_rows_kernel(const long long* __restrict__ ids, size_t n, const long long* __restrict__ sorted_ids,
                                         const int* __restrict__ rowof, int n_tab, int* __restrict__ rows_out, int* __restrict__ err) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long id = ids[i];
  int lo = 0, hi = n_tab - 1, found = -1;
  while (lo <= hi) {
    const int mid = (lo + hi) >> 1;
    const long long v = sorted_ids[mid];
    if (v == id) { found = mid; break; }
    if (v < id) lo = mid + 1; else hi = mid - 1;
  }
  if (found < 0) { atomicExch(err, 1); rows_out[i] = 0; }  // lrcn.jl:602-605 "misssing features"
  else rows_out[i] = rowof[found];
}
void epoch_lookup_rows(cudaStream_t s, const long long* ids, size_t n, const long long* sorted_ids, const int* rowof, int n_tab, int* rows_out, int* err) {
  if (n == 0) return;
  epoch_lookup_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(ids, n, sorted_ids, rowof, n_tab, rows_out, err);
  count_launch();
}
__global__ void epoch_stage_batch_kernel(const long long* __restrict__ seq, size_t row0, int l, int ldB, int col0, int B, int V,
                                         const int* __restrict__ rows_all, size_t rows_off, int* __restrict__ tok_in, int* __restrict__ tok_tgt,
                                         int* __restrict__ rows, int* __restrict__ err) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int T = l + 1;
  if (idx >= T * B) return;
  const int t = idx / B, i = idx - t * B;
  if (t == 0) { tok_in[i] = 1; rows[i] = rows_all[rows_off + col0 + i]; }  // bos (0-based 1)   lrcn.jl:556
  if (t < l) {
    const long long tk = seq[(row0 + t) * (size_t)ldB + col0 + i];
    int v = (int)tk - 1;
    if (tk < 1 || tk > V) { atomicExch(err, 2); v = 2; }  // out-of-range token: flagged, replaced by unk so that no kernel reads out of bounds
    tok_in[(size_t)(t + 1) * B + i] = v;   // next input              lrcn.jl:569
    tok_tgt[(size_t)t * B + i] = v;        // target of step t         lrcn.jl:563-566
  } else {
    tok_tgt[(size_t)t * B + i] = 0;        // eos                      lrcn.jl:572-577
  }
}
void epoch_stage_batch(cudaStream_t s, const long long* seq, size_t row0, int l, int ldB, int col0, int B, int V, const int* rows_all, size_t rows_off,
                       int* tok_in, int* tok_tgt, int* rows, int* err) {
  const int n = (l + 1) * B;
  epoch_stage_batch_kernel<<<(n + 255) / 256, 256, 0, s>>>(seq, row0, l, ldB, col0, B, V, rows_all, rows_off, tok_in, tok_tgt, rows, err);
  count_launch();
}

__global__ void transpose_kernel(const float* __restrict__ in, int rows, int cols, float* __restrict__ out) {
  __shared__ float tile[32][33];
  int c = blockIdx.x * 32 + threadIdx.x;
  for (int k = threadIdx.y; k < 32; k += 8) {
    int r = blockIdx.y * 32 + k;
    if (r < rows && c < cols) tile[k][threadIdx.x] = in[(size_t)r * cols + c];
  }
  __syncthreads();
  int r2 = blockIdx.y * 32 + threadIdx.x;
  for (int k = threadIdx.y; k < 32; k += 8) {
    int c2 = blockIdx.x * 32 + k;
    if (r2 < rows && c2 < cols) out[(size_t)c2 * rows + r2] = tile[threadIdx.x][k];
  }
}
void transpose2d(cudaStream_t s, const float* in, int rows, int cols, float* out) {
  dim3 grid((cols + 31) / 32, (rows + 31) / 32);
  transpose_kernel<<<grid, dim3(32, 8), 0, s>>>(in, rows, cols, out);
  count_launch();
}

__global__ void fill_kernel(float4* buf, size_t n4, float val) {
  float4 v = make_float4(val, val, val, val);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) buf[i] = v;
}
__global__ void zero_multi_kernel(const ZeroSegs z) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int k = 0; k < z.count; k++) {
    float* p = z.p[k];
    const size_t n = z.n[k], n4 = n / 4;
    float4* p4 = reinterpret_cast<float4*>(p);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) p4[i] = zero;
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) p[4 * n4 + threadIdx.x] = 0.f;
  }
}
void zero_multi(cudaStream_t s, const ZeroSegs& z) {
  if (z.count == 0) return;
  launch_pdl<2>(zero_multi_kernel, dim3(148 * 4), dim3(256), 0, s, z);
  count_launch();
}
void fill_l2_scratch(cudaStream_t s, float* buf, size_t n, float val) {
  fill_kernel<<<148 * 8, 256, 0, s>>>((float4*)buf, n / 4, val);
}

// ------------------------------------------------------------------------------------------
// beam search (lrcn.jl:644-678): fp32 probabilities exp(logp), ties -> lower index
// ------------------------------------------------------------------------------------------
struct BestPair { float v; int i; };
__device__ __forceinline__ BestPair better(BestPair a, BestPair b) {
  return (b.v > a.v || (b.v == a.v && b.i < a.i)) ? b : a;
}
__device__ __forceinline__ BestPair block_argmax(BestPair p, BestPair* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    BestPair q;
    q.v = __shfl_xor_sync(0xffffffffu, p.v, o);
    q.i = __shfl_xor_sync(0xffffffffu, p.i, o);
    p = better(p, q);
  }
  int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) red[w] = p;
  __syncthreads();
  BestPair q;
  q.v = -2.f; q.i = 0x7fffffff;
  if (l < nw) q = red[l];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    BestPair t;
    t.v = __shfl_xor_sync(0xffffffffu, q.v, o);
    t.i = __shfl_xor_sync(0xffffffffu, q.i, o);
    q = better(q, t);
  }
  return q;
}

constexpr int TOPK_MAX = 11;
constexpr int TOPK_CAP = 256;  // candidate list capacity of the threshold-select path
struct TopPair { float v; int i; };
__device__ __forceinline__ TopPair top_better(TopPair a, TopPair b) { return (b.v > a.v || (b.v == a.v && b.i < a.i)) ? b : a; }
__device__ __forceinline__ TopPair warp_top(TopPair p) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    TopPair q;
    q.v = __shfl_xor_sync(0xffffffffu, p.v, o);
    q.i = __shfl_xor_sync(0xffffffffu, p.i, o);
    p = top_better(p, q);
  }
  return p;
}
// block-wide (value desc, index asc) argmax; result valid in every thread
__device__ __forceinline__ TopPair block_top(TopPair p, TopPair* red) {
  p = warp_top(p);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) red[w] = p;
  __syncthreads();
  TopPair q;
  q.v = -INFINITY; q.i = 0x7fffffff;
  if (l < nw) q = red[l];
  return warp_top(q);
}

// per row: probabilities ynorm = exp(logp(ypred,2)) (fp32, lrcn.jl:652-654) and the K largest by (prob desc, index asc)
// (lrcn.jl:655-656: sortperm(rev=true) breaks ties by index).  Threshold select:
//   1. the row is staged once in shared memory; max and normaliser by block reductions (the normaliser uses __expf: its ~1e-7
//      relative error shifts every probability of the row alike, so no ordering changes);
//   2. tau = K-th largest of the per-thread maxima is a lower bound of the K-th largest element, so every top-K element is >= tau;
//   3. the (few) elements >= tau are appended to a candidate list; one warp evaluates their precise probabilities and picks the
//      K best by (prob desc, index asc).  Ties at tau are all candidates, so selection on given probabilities is exact.
//   A row with more than TOPK_CAP candidates (e.g. all-equal logits) falls back to K exact block-argmax rounds.
template <bool FROM_LOGITS>
__global__ void __launch_bounds__(512) beam_row_topk_kernel(const float* __restrict__ in, int ld, int R, int V, int K,
                                                            const float* __restrict__ parent_prob, int* __restrict__ cand_tok,
                                                            float* __restrict__ cand_score, float* __restrict__ cand_lp) {
  extern __shared__ __align__(16) float row[];  // V values (logits, or the given probabilities)
  __shared__ float red[32];
  __shared__ TopPair pred[32];
  __shared__ float cv[TOPK_CAP];
  __shared__ int ci[TOPK_CAP];
  __shared__ int ccount;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = blockIdx.x; r < R; r += gridDim.x) {  // persistent over rows
    const float* a = in + (size_t)r * ld;
    __syncthreads();  // previous row's shared state is no longer read
    if (threadIdx.x == 0) ccount = 0;
    float tmax = -INFINITY;
    const int V4 = ((reinterpret_cast<uintptr_t>(a) & 15) == 0) ? (V >> 2) : 0;
    for (int q = threadIdx.x; q < V4; q += blockDim.x) {
      const float4 x = *reinterpret_cast<const float4*>(a + 4 * q);
      *reinterpret_cast<float4*>(row + 4 * q) = x;
      tmax = fmaxf(fmaxf(tmax, fmaxf(x.x, x.y)), fmaxf(x.z, x.w));
    }
    for (int j = 4 * V4 + threadIdx.x; j < V; j += blockDim.x) { const float x = a[j]; row[j] = x; tmax = fmaxf(tmax, x); }
    float lse = 0.f, mx = 0.f;
    if (FROM_LOGITS) {
      mx = block_max(tmax, red);
      float sum = 0.f;
      for (int j = threadIdx.x; j < V; j += blockDim.x) sum += __expf(row[j] - mx);
      sum = block_sum(sum, red);
      lse = logf(sum);
    }
    // tau: K-th largest of the thread maxima (each thread covered a disjoint set of elements)
    float mine = tmax, tau = 0.f;
    for (int k = 0; k < K; k++) {
      TopPair p; p.v = mine; p.i = threadIdx.x;
      p = block_top(p, pred);
      tau = p.v;
      if (p.i == (int)threadIdx.x) mine = -INFINITY;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < V; j += blockDim.x) {
      const float x = row[j];
      if (x >= tau) {
        const int pos = atomicAdd(&ccount, 1);
        if (pos < TOPK_CAP) { cv[pos] = x; ci[pos] = j; }
      }
    }
    __syncthreads();
    const int nc = ccount;
    const float pp = parent_prob[r];
    if (nc <= TOPK_CAP) {
      if (warp == 0) {
        constexpr int PER = TOPK_CAP / 32;
        float pv[PER]; int pi[PER];
#pragma unroll
        for (int q = 0; q < PER; q++) {
          const int c = lane + 32 * q;
          pv[q] = -INFINITY; pi[q] = 0x7fffffff;
          if (c < nc) { const float x = cv[c]; pv[q] = FROM_LOGITS ? expf((x - mx) - lse) : x; pi[q] = ci[c]; }
        }
        for (int k = 0; k < K; k++) {
          TopPair best; best.v = -INFINITY; best.i = 0x7fffffff;
#pragma unroll
          for (int q = 0; q < PER; q++) { TopPair c; c.v = pv[q]; c.i = pi[q]; best = top_better(best, c); }
          best = warp_top(best);
#pragma unroll
          for (int q = 0; q < PER; q++) if (pi[q] == best.i) { pv[q] = -INFINITY; pi[q] = 0x7fffffff; }  // indices are unique
          if (lane == 0) {
            cand_tok[(size_t)r * K + k] = best.i;
            cand_score[(size_t)r * K + k] = __fmul_rn(best.v, pp);  // pmaxes = ynorm[xmaxes]*current_probability (lrcn.jl:657)
            cand_lp[(size_t)r * K + k] = FROM_LOGITS ? ((row[best.i] - mx) - lse) : logf(best.v);
          }
        }
      }
    } else {
      // exact fallback: K rounds of block argmax over the whole row on the probabilities themselves
      if (FROM_LOGITS) {
        __syncthreads();
        for (int j = threadIdx.x; j < V; j += blockDim.x) row[j] = expf((row[j] - mx) - lse);
      }
      for (int k = 0; k < K; k++) {
        __syncthreads();
        TopPair p; p.v = -INFINITY; p.i = 0x7fffffff;
        for (int j = threadIdx.x; j < V; j += blockDim.x) { TopPair c; c.v = row[j]; c.i = j; p = top_better(p, c); }
        p = block_top(p, pred);
        if (threadIdx.x == 0) {
          cand_tok[(size_t)r * K + k] = p.i;
          cand_score[(size_t)r * K + k] = __fmul_rn(p.v, pp);
          cand_lp[(size_t)r * K + k] = logf(p.v);
          row[p.i] = -1.f;  // exclude from later rounds
        }
      }
    }
  }
}
// Second-generation threshold select.  Like beam_row_topk_kernel the row is staged once in shared memory (40 KB at V = 10000,
// so 4 CTAs share an SM), but max and normaliser come from ONE block reduction of per-thread (max, sum exp) pairs and tau from
// per-warp top-K lists of the thread maxima: 4 block barriers per row instead of ~12.  Same results on given probabilities.
constexpr int TOPK_MAXK = 11;
template <bool FROM_LOGITS, int THREADS>
__global__ void __launch_bounds__(THREADS) beam_row_topk2_kernel(const float* __restrict__ in, int ld, int R, int V, int K,
                                                             const float* __restrict__ parent_prob, int* __restrict__ cand_tok,
                                                             float* __restrict__ cand_score, float* __restrict__ cand_lp) {
  extern __shared__ __align__(16) float row[];
  constexpr int NW = THREADS / 32;
  __shared__ float2 wred[NW];
  __shared__ float wtop[NW][TOPK_MAXK + 1];
  __shared__ float cv[TOPK_CAP];
  __shared__ int ci[TOPK_CAP];
  __shared__ int ccount;
  __shared__ TopPair pred[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = blockIdx.x; r < R; r += gridDim.x) {  // persistent over rows
    const float* a = in + (size_t)r * ld;
    __syncthreads();  // the previous row's shared state is no longer read
    if (threadIdx.x == 0) ccount = 0;
    float tmax = -INFINITY;
    const int V4 = ((reinterpret_cast<uintptr_t>(a) & 15) == 0) ? (V >> 2) : 0;
    for (int q = threadIdx.x; q < V4; q += blockDim.x) {
      const float4 x = *reinterpret_cast<const float4*>(a + 4 * q);
      *reinterpret_cast<float4*>(row + 4 * q) = x;
      tmax = fmaxf(fmaxf(tmax, fmaxf(x.x, x.y)), fmaxf(x.z, x.w));
    }
    for (int j = 4 * V4 + threadIdx.x; j < V; j += blockDim.x) { const float x = a[j]; row[j] = x; tmax = fmaxf(tmax, x); }
    // (max, sum exp) of this thread's own elements (it re-reads what it wrote: no barrier needed), then of the warp
    if (FROM_LOGITS) {
      float m = tmax, ssum = 0.f;
      if (tmax != -INFINITY) {
        for (int q = threadIdx.x; q < V4; q += blockDim.x) {
          const float4 x = *reinterpret_cast<const float4*>(row + 4 * q);
          ssum += (__expf(x.x - tmax) + __expf(x.y - tmax)) + (__expf(x.z - tmax) + __expf(x.w - tmax));
        }
        for (int j = 4 * V4 + threadIdx.x; j < V; j += blockDim.x) ssum += __expf(row[j] - tmax);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, ssum, o);
        const float mn = fmaxf(m, m2);
        ssum = (m == -INFINITY ? 0.f : ssum * __expf(m - mn)) + (m2 == -INFINITY ? 0.f : s2 * __expf(m2 - mn));
        m = mn;
      }
      if (lane == 0) wred[warp] = make_float2(m, ssum);
    }
    // per-warp top-K of the thread maxima (K rounds, one lane removed per round)
    {
      float cur = tmax;
      for (int k = 0; k < K; k++) {
        float best = cur;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o));
        const unsigned int holders = __ballot_sync(0xffffffffu, cur == best);
        if (lane == __ffs(holders) - 1) { cur = -INFINITY; wtop[warp][k] = best; }
      }
    }
    __syncthreads();
    float mx = 0.f, lse = 0.f;
    if (FROM_LOGITS) {
      float mm = -INFINITY;
#pragma unroll
      for (int w = 0; w < NW; w++) mm = fmaxf(mm, wred[w].x);
      float tot = 0.f;
#pragma unroll
      for (int w = 0; w < NW; w++) tot += wred[w].x == -INFINITY ? 0.f : wred[w].y * __expf(wred[w].x - mm);
      mx = mm; lse = logf(tot);
    }
    // tau = K-th largest of the NW*K per-warp values (every warp computes it redundantly): a lower bound of the K-th largest element
    float tau;
    {
      float mine[6];  // 16 * 11 = 176 <= 6 * 32
#pragma unroll
      for (int q = 0; q < 6; q++) {
        const int c = lane + 32 * q;
        mine[q] = (c < NW * K) ? wtop[c / K][c % K] : -INFINITY;
      }
      tau = -INFINITY;
      for (int k = 0; k < K; k++) {
        float best = -INFINITY;
#pragma unroll
        for (int q = 0; q < 6; q++) best = fmaxf(best, mine[q]);
        float wb = best;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wb = fmaxf(wb, __shfl_xor_sync(0xffffffffu, wb, o));
        tau = wb;
        const unsigned int holders = __ballot_sync(0xffffffffu, best == wb);
        if (lane == __ffs(holders) - 1) {
          bool removed = false;
#pragma unroll
          for (int q = 0; q < 6; q++) if (!removed && mine[q] == wb) { mine[q] = -INFINITY; removed = true; }
        }
      }
    }
    // candidates: every element >= tau (own elements again)
    for (int q = threadIdx.x; q < V4; q += blockDim.x) {
      const float4 x = *reinterpret_cast<const float4*>(row + 4 * q);
      const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
      for (int e = 0; e < 4; e++)
        if (xs[e] >= tau) {
          const int pos = atomicAdd(&ccount, 1);
          if (pos < TOPK_CAP) { cv[pos] = xs[e]; ci[pos] = 4 * q + e; }
        }
    }
    for (int j = 4 * V4 + threadIdx.x; j < V; j += blockDim.x) {
      const float x = row[j];
      if (x >= tau) {
        const int pos = atomicAdd(&ccount, 1);
        if (pos < TOPK_CAP) { cv[pos] = x; ci[pos] = j; }
      }
    }
    __syncthreads();
    const int nc = ccount;
    const float pp = parent_prob[r];
    if (nc <= TOPK_CAP) {
      if (warp == 0) {
        constexpr int PER = TOPK_CAP / 32;
        float pv[PER]; int pi[PER];
#pragma unroll
        for (int q = 0; q < PER; q++) {
          const int c = lane + 32 * q;
          pv[q] = -INFINITY; pi[q] = 0x7fffffff;
          if (c < nc) { const float x = cv[c]; pv[q] = FROM_LOGITS ? expf((x - mx) - lse) : x; pi[q] = ci[c]; }
        }
        for (int k = 0; k < K; k++) {
          TopPair best; best.v = -INFINITY; best.i = 0x7fffffff;
#pragma unroll
          for (int q = 0; q < PER; q++) { TopPair c; c.v = pv[q]; c.i = pi[q]; best = top_better(best, c); }
          best = warp_top(best);
#pragma unroll
          for (int q = 0; q < PER; q++) if (pi[q] == best.i) { pv[q] = -INFINITY; pi[q] = 0x7fffffff; }  // indices are unique
          if (lane == 0) {
            cand_tok[(size_t)r * K + k] = best.i;
            cand_score[(size_t)r * K + k] = __fmul_rn(best.v, pp);  // pmaxes = ynorm[xmaxes]*current_probability (lrcn.jl:657)
            cand_lp[(size_t)r * K + k] = FROM_LOGITS ? ((row[best.i] - mx) - lse) : logf(best.v);
          }
        }
      }
    } else {
      // exact fallback: K rounds of block argmax over the whole row on the probabilities themselves
      if (FROM_LOGITS) {
        for (int j = threadIdx.x; j < V; j += blockDim.x) row[j] = expf((row[j] - mx) - lse);
      }
      for (int k = 0; k < K; k++) {
        __syncthreads();
        TopPair p; p.v = -INFINITY; p.i = 0x7fffffff;
        for (int j = threadIdx.x; j < V; j += blockDim.x) { TopPair c; c.v = row[j]; c.i = j; p = top_better(p, c); }
        p = block_top(p, pred);
        if (threadIdx.x == 0) {
          cand_tok[(size_t)r * K + k] = p.i;
          cand_score[(size_t)r * K + k] = __fmul_rn(p.v, pp);
          cand_lp[(size_t)r * K + k] = logf(p.v);
          row[p.i] = -1.f;  // exclude from later rounds
        }
      }
    }
  }
}
// Third generation: the row lives in REGISTERS (NV4 float4 per thread, every load of the row in flight at once), shared memory
// holds only the candidate list; the row is dumped to shared memory only for the exact fallback.  The shared-memory staging of
// topk2 serialised a global round trip, three shared-memory passes and four block barriers per row with 4-5 CTAs per SM (0.30 of
// HBM at V = 10000); here the passes run on registers.  Same arithmetic in the same order per element => same results.
// Needs V % 4 == 0, 16-byte aligned rows and V <= 4 * THREADS * NV4.
template <bool FROM_LOGITS, int NV4>
__global__ void __launch_bounds__(256, 3) beam_row_topk3_kernel(const float* __restrict__ in, int ld, int R, int V, int K,
                                                             const float* __restrict__ parent_prob, int* __restrict__ cand_tok,
                                                             float* __restrict__ cand_score, float* __restrict__ cand_lp) {
  extern __shared__ __align__(16) float row[];  // fallback only
  constexpr int THREADS = 256, NW = THREADS / 32;
  __shared__ float2 wred[NW];
  __shared__ float wtop[NW][TOPK_MAXK + 1];
  __shared__ float cv[TOPK_CAP];
  __shared__ int ci[TOPK_CAP];
  __shared__ int ccount;
  __shared__ TopPair pred[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int V4 = V >> 2;
  for (int r = blockIdx.x; r < R; r += gridDim.x) {  // persistent over rows
    const float4* a4 = reinterpret_cast<const float4*>(in + (size_t)r * ld);
    float4 x[NV4];
#pragma unroll
    for (int i = 0; i < NV4; i++) {
      const int q = threadIdx.x + THREADS * i;
      x[i] = q < V4 ? __ldg(a4 + q) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    }
    __syncthreads();  // the previous row's shared state is no longer read
    if (threadIdx.x == 0) ccount = 0;
    float tmax = -INFINITY;
#pragma unroll
    for (int i = 0; i < NV4; i++) tmax = fmaxf(fmaxf(tmax, fmaxf(x[i].x, x[i].y)), fmaxf(x[i].z, x[i].w));
    if (FROM_LOGITS) {
      float m = tmax, ssum = 0.f;
      if (tmax != -INFINITY) {
#pragma unroll
        for (int i = 0; i < NV4; i++)
          if (threadIdx.x + THREADS * i < V4) ssum += (__expf(x[i].x - tmax) + __expf(x[i].y - tmax)) + (__expf(x[i].z - tmax) + __expf(x[i].w - tmax));
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, ssum, o);
        const float mn = fmaxf(m, m2);
        ssum = (m == -INFINITY ? 0.f : ssum * __expf(m - mn)) + (m2 == -INFINITY ? 0.f : s2 * __expf(m2 - mn));
        m = mn;
      }
      if (lane == 0) wred[warp] = make_float2(m, ssum);
    }
    {  // per-warp top-K of the thread maxima (K rounds, one lane removed per round)
      float cur = tmax;
      for (int k = 0; k < K; k++) {
        float best = cur;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o));
        const unsigned int holders = __ballot_sync(0xffffffffu, cur == best);
        if (lane == __ffs(holders) - 1) { cur = -INFINITY; wtop[warp][k] = best; }
      }
    }
    __syncthreads();
    float mx = 0.f, lse = 0.f;
    if (FROM_LOGITS) {
      float mm = -INFINITY;
#pragma unroll
      for (int w = 0; w < NW; w++) mm = fmaxf(mm, wred[w].x);
      float tot = 0.f;
#pragma unroll
      for (int w = 0; w < NW; w++) tot += wred[w].x == -INFINITY ? 0.f : wred[w].y * __expf(wred[w].x - mm);
      mx = mm; lse = logf(tot);
    }
    float tau;  // K-th largest of the NW*K per-warp values: a lower bound of the K-th largest element
    {
      float mine[3];  // 8 * 11 = 88 <= 3 * 32
#pragma unroll
      for (int q = 0; q < 3; q++) {
        const int c = lane + 32 * q;
        mine[q] = (c < NW * K) ? wtop[c / K][c % K] : -INFINITY;
      }
      tau = -INFINITY;
      for (int k = 0; k < K; k++) {
        float best = fmaxf(fmaxf(mine[0], mine[1]), mine[2]);
        float wb = best;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wb = fmaxf(wb, __shfl_xor_sync(0xffffffffu, wb, o));
        tau = wb;
        const unsigned int holders = __ballot_sync(0xffffffffu, best == wb);
        if (lane == __ffs(holders) - 1) {
          bool removed = false;
#pragma unroll
          for (int q = 0; q < 3; q++) if (!removed && mine[q] == wb) { mine[q] = -INFINITY; removed = true; }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NV4; i++) {  // candidates: every element >= tau (padding is -inf: never a candidate unless tau = -inf, where q < V4 guards)
      const int q = threadIdx.x + THREADS * i;
      const float xs[4] = {x[i].x, x[i].y, x[i].z, x[i].w};
#pragma unroll
      for (int e = 0; e < 4; e++)
        if (xs[e] >= tau && q < V4) {
          const int pos = atomicAdd(&ccount, 1);
          if (pos < TOPK_CAP) { cv[pos] = xs[e]; ci[pos] = 4 * q + e; }
        }
    }
    __syncthreads();
    const int nc = ccount;
    const float pp = parent_prob[r];
    if (nc <= TOPK_CAP) {
      if (warp == 0) {
        constexpr int PER = TOPK_CAP / 32;
        float pv[PER], pl[PER]; int pi[PER];
#pragma unroll
        for (int q = 0; q < PER; q++) {
          const int c = lane + 32 * q;
          pv[q] = -INFINITY; pi[q] = 0x7fffffff; pl[q] = 0.f;
          if (c < nc) {
            const float xc = cv[c];
            pl[q] = FROM_LOGITS ? ((xc - mx) - lse) : 0.f;
            pv[q] = FROM_LOGITS ? expf((xc - mx) - lse) : xc;
            pi[q] = ci[c];
          }
        }
        for (int k = 0; k < K; k++) {
          TopPair best; best.v = -INFINITY; best.i = 0x7fffffff;
#pragma unroll
          for (int q = 0; q < PER; q++) { TopPair c; c.v = pv[q]; c.i = pi[q]; best = top_better(best, c); }
          best = warp_top(best);
#pragma unroll
          for (int q = 0; q < PER; q++)
            if (pi[q] == best.i) {  // indices are unique: exactly one lane owns the winner and writes it
              cand_tok[(size_t)r * K + k] = best.i;
              cand_score[(size_t)r * K + k] = __fmul_rn(best.v, pp);  // pmaxes = ynorm[xmaxes]*current_probability (lrcn.jl:657)
              cand_lp[(size_t)r * K + k] = FROM_LOGITS ? pl[q] : logf(best.v);
              pv[q] = -INFINITY; pi[q] = 0x7fffffff;
            }
        }
      }
    } else {
      // exact fallback: K rounds of block argmax over the whole row on the probabilities themselves (row dumped to shared memory)
#pragma unroll
      for (int i = 0; i < NV4; i++) {
        const int q = threadIdx.x + THREADS * i;
        if (q < V4) {
          float4 y = x[i];
          if (FROM_LOGITS) { y.x = expf((y.x - mx) - lse); y.y = expf((y.y - mx) - lse); y.z = expf((y.z - mx) - lse); y.w = expf((y.w - mx) - lse); }
          *reinterpret_cast<float4*>(row + 4 * q) = y;
        }
      }
      for (int k = 0; k < K; k++) {
        __syncthreads();
        TopPair p; p.v = -INFINITY; p.i = 0x7fffffff;
        for (int j = threadIdx.x; j < V; j += blockDim.x) { TopPair c; c.v = row[j]; c.i = j; p = top_better(p, c); }
        p = block_top(p, pred);
        if (threadIdx.x == 0) {
          cand_tok[(size_t)r * K + k] = p.i;
          cand_score[(size_t)r * K + k] = __fmul_rn(p.v, pp);
          cand_lp[(size_t)r * K + k] = logf(p.v);
          row[p.i] = -1.f;  // exclude from later rounds
        }
      }
    }
  }
}
// Fourth generation: ONE WARP PER ROW, one streaming pass, no shared memory and no block barrier.  topk2 / topk3 process a row per
// CTA in phases separated by four block barriers with a serial last phase in warp 0: ~8 us of latency per row and 3 rows in
// flight per SM = 0.33 of the HBM peak (ncu launch list: 56 us for 3072 x 10000 logits).  Here every lane streams its float4
// columns (16 loads in flight per lane, 32 independent rows per SM), keeps an online (max, sum exp) pair and its own top-KM list
// in registers (sorted, strict '>' insertion in increasing column order: equal values keep the lower index first), and the warp
// then pops the K global winners from the 32 list heads by (value desc, index asc).  A member of the global top-K is always in its
// lane's top-K, so the selection is the exact top-K by (logit, index); probabilities are formed for the K winners only and winners
// whose probabilities round to the same float are re-ordered by index, which is the order the reference's stable sort of the
// probabilities gives (lrcn.jl:652-661).  Needs V % 4 == 0 and 16-byte aligned rows.
template <bool FROM_LOGITS, int KM, int U>
__global__ void __launch_bounds__(256) beam_row_topk4_kernel(const float* __restrict__ in, int ld, int R, int V, int K,
                                                             const float* __restrict__ parent_prob, int* __restrict__ cand_tok,
                                                             float* __restrict__ cand_score, float* __restrict__ cand_lp) {
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const int V4 = V >> 2;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < R; r += gridDim.x * wpb) {
    const float4* a4 = reinterpret_cast<const float4*>(in + (size_t)r * ld);
    float tv[KM]; int ti[KM];
#pragma unroll
    for (int k = 0; k < KM; k++) { tv[k] = -INFINITY; ti[k] = 0x7fffffff; }
    float m = -INFINITY, ssum = 0.f;
    auto consider = [&](float val, int idx) {
      if (val > tv[KM - 1]) {  // rare after the first few columns
        tv[KM - 1] = val; ti[KM - 1] = idx;
#pragma unroll
        for (int k = KM - 1; k > 0; k--) {
          if (tv[k] > tv[k - 1]) {  // strict: an equal earlier (lower-index) value stays in front
            const float fv = tv[k]; tv[k] = tv[k - 1]; tv[k - 1] = fv;
            const int iv = ti[k]; ti[k] = ti[k - 1]; ti[k - 1] = iv;
          }
        }
      }
    };
    for (int q0 = lane; q0 < V4; q0 += 32 * U) {
      float4 x[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const int q = q0 + 32 * u;
        x[u] = q < V4 ? __ldg(a4 + q) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const int q = q0 + 32 * u;
        if (q >= V4) break;
        if (FROM_LOGITS) {
          const float cm = fmaxf(fmaxf(x[u].x, x[u].y), fmaxf(x[u].z, x[u].w));
          if (cm > m) { ssum = (m == -INFINITY) ? 0.f : ssum * __expf(m - cm); m = cm; }
          if (m != -INFINITY) ssum += (__expf(x[u].x - m) + __expf(x[u].y - m)) + (__expf(x[u].z - m) + __expf(x[u].w - m));
        }
        consider(x[u].x, 4 * q); consider(x[u].y, 4 * q + 1); consider(x[u].z, 4 * q + 2); consider(x[u].w, 4 * q + 3);
      }
    }
    float mx = 0.f, lse = 0.f;
    if (FROM_LOGITS) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, ssum, o);
        const float mn = fmaxf(m, m2);
        ssum = (m == -INFINITY ? 0.f : ssum * __expf(m - mn)) + (m2 == -INFINITY ? 0.f : s2 * __expf(m2 - mn));
        m = mn;
      }
      mx = m; lse = logf(ssum);
    }
    // K rounds: the best list head of the warp by (value desc, index asc); the winning lane pops its list
    float wv = -INFINITY; int wi = 0x7fffffff;  // lane k keeps winner k
    for (int k = 0; k < K; k++) {
      TopPair best; best.v = tv[0]; best.i = ti[0];
      best = warp_top(best);
      if (ti[0] == best.i) {  // indices are unique: exactly one lane owns the winner
#pragma unroll
        for (int j = 0; j < KM - 1; j++) { tv[j] = tv[j + 1]; ti[j] = ti[j + 1]; }
        tv[KM - 1] = -INFINITY; ti[KM - 1] = 0x7fffffff;
      }
      if (lane == k) { wv = best.v; wi = best.i; }
    }
    const float lp = FROM_LOGITS ? ((wv - mx) - lse) : 0.f;
    const float pr = FROM_LOGITS ? expf(lp) : wv;
    // winners are ordered by (logit desc, index asc); probabilities are monotone in the logit, so only winners whose probabilities
    // round to the same float can be out of (probability desc, index asc) order: rank them explicitly
    int rank = 0;
    for (int j = 0; j < K; j++) {
      const float pj = __shfl_sync(0xffffffffu, pr, j);
      const int ij = __shfl_sync(0xffffffffu, wi, j);
      if (lane < K && j != lane && (pj > pr || (pj == pr && ij < wi))) rank++;
    }
    if (lane < K) {
      const float pp = parent_prob[r];
      cand_tok[(size_t)r * K + rank] = wi;
      cand_score[(size_t)r * K + rank] = __fmul_rn(pr, pp);  // pmaxes = ynorm[xmaxes]*current_probability (lrcn.jl:657)
      cand_lp[(size_t)r * K + rank] = FROM_LOGITS ? lp : logf(pr);
    }
  }
}
template <bool FROM_LOGITS>
static void beam_topk4_launch(cudaStream_t s, const float* in, int ld, int R, int V, int K, const float* parent_prob, int* cand_tok, float* cand_score,
                              float* cand_lp) {
  const int want = (R + 7) / 8;
  const int cap = 148 * 4;  // 48-64 registers per thread: four 256-thread CTAs per SM
  const int grid = want < cap ? want : cap;
  if (K <= 1) beam_row_topk4_kernel<FROM_LOGITS, 1, 8><<<grid, 256, 0, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
  else if (K <= 3) beam_row_topk4_kernel<FROM_LOGITS, 3, 8><<<grid, 256, 0, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
  else if (K <= 5) beam_row_topk4_kernel<FROM_LOGITS, 5, 8><<<grid, 256, 0, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
  else beam_row_topk4_kernel<FROM_LOGITS, TOPK_MAXK, 4><<<grid, 256, 0, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
  count_launch();
}
static void beam_topk_launch(cudaStream_t s, bool from_logits, const float* in, int ld, int R, int V, int K,
                             const float* parent_prob, int* cand_tok, float* cand_score, float* cand_lp) {
  const size_t smem = ((size_t)V + 4) * sizeof(float);
  const int grid = R < 148 * 4 ? R : 148 * 4;
  static const bool v1 = getenv("LRCN_TOPK_V1") != nullptr;
  static const bool no_v4 = getenv("LRCN_TOPK_V3") != nullptr || getenv("LRCN_TOPK_V2") != nullptr;
  // one warp per row needs many rows to fill the machine (a lone warp streams a 40 KB row in ~20 us); below that the CTA-per-row
  // kernels are faster (measured: COCO-shaped decode, i.e. compacted batches, 157 k captions/s with topk4 everywhere vs 163 k)
  static const int v4_rows = getenv("LRCN_TOPK_V4_ROWS") ? atoi(getenv("LRCN_TOPK_V4_ROWS")) : 2048;
  if (!v1 && !no_v4 && R >= v4_rows && K <= TOPK_MAXK && V % 4 == 0 && ld % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 && V >= 128) {
    if (from_logits) beam_topk4_launch<true>(s, in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
    else beam_topk4_launch<false>(s, in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
    return;
  }
  static const bool no_v3 = getenv("LRCN_TOPK_V2") != nullptr;
  constexpr int NV4 = 11;  // V <= 11264 (COCO: 10000 / 10636)
  if (!v1 && !no_v3 && K <= TOPK_MAXK && V % 4 == 0 && ld % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 && V > 4096 && V <= 4 * 256 * NV4) {
    const int g3 = R < 148 * 3 ? R : 148 * 3;  // 3 CTAs per SM (registers)
    if (from_logits) beam_row_topk3_kernel<true, NV4><<<g3, 256, smem, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
    else beam_row_topk3_kernel<false, NV4><<<g3, 256, smem, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
    count_launch();
    return;
  }
  if (!v1 && K <= TOPK_MAXK) {
    static const int th = getenv("LRCN_TOPK_THREADS") ? atoi(getenv("LRCN_TOPK_THREADS")) : 256;
    const int g2 = R < 148 * 8 ? R : 148 * 8;
    if (th == 512) {
      if (from_logits) beam_row_topk2_kernel<true, 512><<<grid, 512, smem, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
      else beam_row_topk2_kernel<false, 512><<<grid, 512, smem, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
    } else {
      if (from_logits) beam_row_topk2_kernel<true, 256><<<g2, 256, smem, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
      else beam_row_topk2_kernel<false, 256><<<g2, 256, smem, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
    }
    count_launch();
    return;
  }
  if (from_logits) beam_row_topk_kernel<true><<<grid, 512, smem, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
  else beam_row_topk_kernel<false><<<grid, 512, smem, s>>>(in, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
  count_launch();
}
void beam_row_topk(cudaStream_t s, const float* logits, int ld, int R, int V, int K, const float* parent_prob, int* cand_tok,
                   float* cand_score, float* cand_lp) {
  beam_topk_launch(s, true, logits, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
}
void beam_row_topk_probs(cudaStream_t s, const float* probs, int ld, int R, int V, int K, const float* parent_prob,
                         int* cand_tok, float* cand_score, float* cand_lp) {
  beam_topk_launch(s, false, probs, ld, R, V, K, parent_prob, cand_tok, cand_score, cand_lp);
}

// one thread per image: stable descending selection over the candidate list (beam-major, rank-minor)
__global__ void beam_select_kernel(const int* __restrict__ cand_tok, const float* __restrict__ cand_score,
                                   const float* __restrict__ cand_lp, int n_img, int K, int first_step, int* __restrict__ sel_tok,
                                   int* __restrict__ sel_parent, float* __restrict__ sel_score, float* __restrict__ sel_lp) {
  int img = blockIdx.x * blockDim.x + threadIdx.x;
  if (img >= n_img) return;
  int ncand = first_step ? K : K * K;
  const float* sc = cand_score + (size_t)img * K * K;
  unsigned long long used_lo = 0, used_hi = 0;  // K*K <= 128 candidates
  for (int k = 0; k < K; k++) {
    int best = -1;
    float bv = 0.f;
    for (int c = 0; c < ncand; c++) {
      bool used = c < 64 ? ((used_lo >> c) & 1ull) : ((used_hi >> (c - 64)) & 1ull);
      if (used) continue;
      float v = sc[c];
      if (best < 0 || v > bv) { best = c; bv = v; }  // strict > keeps the earlier list position on ties
    }
    if (best < 64) used_lo |= 1ull << best; else used_hi |= 1ull << (best - 64);
    size_t o = (size_t)img * K + k;
    sel_tok[o] = cand_tok[(size_t)img * K * K + best];
    sel_parent[o] = best / K;  // ceil((best+1)/K) - 1  (lrcn.jl:675)
    sel_score[o] = bv;
    sel_lp[o] = cand_lp[(size_t)img * K * K + best];
  }
}
void beam_select(cudaStream_t s, const int* cand_tok, const float* cand_score, const float* cand_lp, int n_img, int K,
                 int first_step, int* sel_tok, int* sel_parent, float* sel_score, float* sel_lp) {
  beam_select_kernel<<<(n_img + 63) / 64, 64, 0, s>>>(cand_tok, cand_score, cand_lp, n_img, K, first_step, sel_tok, sel_parent,
                                                      sel_score, sel_lp);
  count_launch();
}

// one CTA per (image, beam) row: reorder/gather the advanced states of the parents, extend histories,
// detect termination (best hypothesis ends in eos, or step > nword: lrcn.jl:670) and emit results.
__global__ void __launch_bounds__(128) beam_advance_kernel(BeamAdvanceArgs a) {
  int r = blockIdx.x;
  int img = r / a.K, k = r - img * a.K;
  if (a.done[img]) return;  // (fused: the k = 0 row of this launch may set the flag meanwhile -- either outcome is fine, the image is frozen from here on)
  __shared__ int s_tok, s_par;
  __shared__ float s_score, s_lp;
  if (a.fused) {
    // the image's selection, as beam_select_kernel does it: k+1 rounds of "best unused candidate", strict '>' keeps the earlier
    // list position (beam-major, rank-minor) on ties; this row takes the (k+1)-th
    if (threadIdx.x == 0) {
      const int ncand = a.step == 1 ? a.K : a.K * a.K;
      const float* sc = a.cand_score + (size_t)img * a.K * a.K;
      unsigned long long used_lo = 0, used_hi = 0;  // K*K <= 128 candidates
      int best = -1;
      float bv = 0.f;
      for (int kk = 0; kk <= k; kk++) {
        best = -1; bv = 0.f;
        for (int c = 0; c < ncand; c++) {
          const bool used = c < 64 ? ((used_lo >> c) & 1ull) : ((used_hi >> (c - 64)) & 1ull);
          if (used) continue;
          const float v = sc[c];
          if (best < 0 || v > bv) { best = c; bv = v; }
        }
        if (best < 64) used_lo |= 1ull << best; else used_hi |= 1ull << (best - 64);
      }
      s_tok = a.cand_tok[(size_t)img * a.K * a.K + best];
      s_par = best / a.K;  // ceil((best+1)/K) - 1  (lrcn.jl:675)
      s_score = bv;
      s_lp = a.cand_lp[(size_t)img * a.K * a.K + best];
    }
  } else if (threadIdx.x == 0) {
    s_tok = a.sel_tok[r]; s_par = a.sel_parent[r]; s_score = a.sel_score[r]; s_lp = a.sel_lp[r];
  }
  __syncthreads();
  int parent = img * a.K + s_par;
  // 128-bit copies when every row is 16-byte aligned (H, pitches and E multiples of 4: always in the bf16x3 mode)
  const bool vec = ((a.H1 | a.H2 | a.ld1 | a.ld2 | a.E | a.lde) & 3) == 0;
  if (vec) {
    for (int q = threadIdx.x; q < (a.H1 >> 2); q += blockDim.x) {
      const float4 hv = reinterpret_cast<const float4*>(a.h1_in + (size_t)parent * a.H1)[q];
      reinterpret_cast<float4*>(a.h1_out + (size_t)r * a.ld1)[q] = hv;
      reinterpret_cast<float4*>(a.c1_out + (size_t)r * a.H1)[q] = reinterpret_cast<const float4*>(a.c1_in + (size_t)parent * a.H1)[q];
      if (a.h1_hi) store_split4(a.h1_hi, a.h1_lo, (size_t)r * a.ld1 + 4 * q, hv);
    }
    for (int q = threadIdx.x; q < (a.H2 >> 2); q += blockDim.x) {
      const float4 hv = reinterpret_cast<const float4*>(a.h2_in + (size_t)parent * a.H2)[q];
      reinterpret_cast<float4*>(a.h2_out + (size_t)r * a.ld2)[q] = hv;
      reinterpret_cast<float4*>(a.c2_out + (size_t)r * a.H2)[q] = reinterpret_cast<const float4*>(a.c2_in + (size_t)parent * a.H2)[q];
      if (a.h2_hi) store_split4(a.h2_hi, a.h2_lo, (size_t)r * a.ld2 + 4 * q, hv);
    }
  } else {
  for (int j = threadIdx.x; j < a.H1; j += blockDim.x) {
    const float hv = a.h1_in[(size_t)parent * a.H1 + j];
    a.h1_out[(size_t)r * a.ld1 + j] = hv;
    a.c1_out[(size_t)r * a.H1 + j] = a.c1_in[(size_t)parent * a.H1 + j];
    if (a.h1_hi) { __nv_bfloat16 hh, ll; split_one(hv, hh, ll); a.h1_hi[(size_t)r * a.ld1 + j] = hh; a.h1_lo[(size_t)r * a.ld1 + j] = ll; }
  }
  for (int j = threadIdx.x; j < a.H2; j += blockDim.x) {
    const float hv = a.h2_in[(size_t)parent * a.H2 + j];
    a.h2_out[(size_t)r * a.ld2 + j] = hv;
    a.c2_out[(size_t)r * a.H2 + j] = a.c2_in[(size_t)parent * a.H2 + j];
    if (a.h2_hi) { __nv_bfloat16 hh, ll; split_one(hv, hh, ll); a.h2_hi[(size_t)r * a.ld2 + j] = hh; a.h2_lo[(size_t)r * a.ld2 + j] = ll; }
  }
  }
  // history so far has a.step tokens (bos + step-1 generated); append one
  int len = a.step;
  for (int j = threadIdx.x; j < len; j += blockDim.x) {
    a.hist_out[(size_t)r * a.maxlen + j] = a.hist_in[(size_t)parent * a.maxlen + j];
    a.lp_out[(size_t)r * a.maxlen + j] = a.lp_in[(size_t)parent * a.maxlen + j];
  }
  int tok = s_tok;
  if (a.fused && a.wemb) {  // the next step's input embedding Wemb[tok,:] (+ its bf16 split)
    const float* src = a.wemb + (size_t)tok * a.E;
    if (vec) {
      for (int q = threadIdx.x; q < (a.E >> 2); q += blockDim.x) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(src) + q);
        reinterpret_cast<float4*>(a.e_out + (size_t)r * a.lde)[q] = x;
        if (a.e_hi) store_split4(a.e_hi, a.e_lo, (size_t)r * a.lde + 4 * q, x);
      }
    } else
    for (int j = threadIdx.x; j < a.E; j += blockDim.x) {
      const float x = __ldg(src + j);
      a.e_out[(size_t)r * a.lde + j] = x;
      if (a.e_hi) { __nv_bfloat16 hh, ll; split_one(x, hh, ll); a.e_hi[(size_t)r * a.lde + j] = hh; a.e_lo[(size_t)r * a.lde + j] = ll; }
    }
  }
  if (threadIdx.x == 0) {
    a.hist_out[(size_t)r * a.maxlen + len] = tok;
    a.lp_out[(size_t)r * a.maxlen + len] = s_lp;
    a.prob[r] = s_score;
    a.last_tok[r] = tok;
  }
  if (k == 0) {
    bool stop = (tok == 0 /* eos, 0-based */) || (a.step > a.nword);
    if (stop) {
      __syncthreads();
      int total = len + 1;
      const int oimg = a.out_map ? a.out_map[img] : img;  // where the caller's chunk expects this image
      for (int j = threadIdx.x; j < total; j += blockDim.x) {
        a.out_tokens[(size_t)oimg * a.maxlen + j] = (long long)a.hist_out[(size_t)r * a.maxlen + j] + 1;
        if (a.out_lp && j >= 1) a.out_lp[(size_t)oimg * (a.maxlen - 1) + (j - 1)] = a.lp_out[(size_t)r * a.maxlen + j];
      }
      if (threadIdx.x == 0) {
        a.out_len[oimg] = total;
        a.out_prob[oimg] = s_score;
        if (a.fused) { a.done[img] = 1; atomicAdd(a.n_done, 1); }
      }
    }
  }
}
// second tiny kernel marks images done AFTER all K rows of the step were advanced (avoids a race on done[])
__global__ void beam_mark_done_kernel(const int* __restrict__ sel_tok, int n_img, int K, int step, int nword, int* __restrict__ done,
                                      int* __restrict__ n_done) {
  int img = blockIdx.x * blockDim.x + threadIdx.x;
  if (img >= n_img || done[img]) return;
  int tok = sel_tok[(size_t)img * K];
  if (tok == 0 || step > nword) {
    done[img] = 1;
    atomicAdd(n_done, 1);
  }
}
__global__ void __launch_bounds__(128) beam_compact_gather_kernel(BeamCompactArgs a) {
  const int rn = blockIdx.x, img = rn / a.K, k = rn - img * a.K;
  const int ro = a.keep[img] * a.K + k;
  const bool vec = ((a.H1 | a.H2 | a.ld1 | a.ld2) & 3) == 0;  // 128-bit copies when every row is 16-byte aligned
  if (vec) {
    for (int q = threadIdx.x; q < (a.H1 >> 2); q += blockDim.x) {
      reinterpret_cast<float4*>(a.h1_s + (size_t)rn * a.H1)[q] = reinterpret_cast<const float4*>(a.h1 + (size_t)ro * a.ld1)[q];
      reinterpret_cast<float4*>(a.c1_s + (size_t)rn * a.H1)[q] = reinterpret_cast<const float4*>(a.c1 + (size_t)ro * a.H1)[q];
    }
    for (int q = threadIdx.x; q < (a.H2 >> 2); q += blockDim.x) {
      reinterpret_cast<float4*>(a.h2_s + (size_t)rn * a.H2)[q] = reinterpret_cast<const float4*>(a.h2 + (size_t)ro * a.ld2)[q];
      reinterpret_cast<float4*>(a.c2_s + (size_t)rn * a.H2)[q] = reinterpret_cast<const float4*>(a.c2 + (size_t)ro * a.H2)[q];
    }
  } else {
  for (int j = threadIdx.x; j < a.H1; j += blockDim.x) {
    a.h1_s[(size_t)rn * a.H1 + j] = a.h1[(size_t)ro * a.ld1 + j];
    a.c1_s[(size_t)rn * a.H1 + j] = a.c1[(size_t)ro * a.H1 + j];
  }
  for (int j = threadIdx.x; j < a.H2; j += blockDim.x) {
    a.h2_s[(size_t)rn * a.H2 + j] = a.h2[(size_t)ro * a.ld2 + j];
    a.c2_s[(size_t)rn * a.H2 + j] = a.c2[(size_t)ro * a.H2 + j];
  }
  }
  for (int j = threadIdx.x; j < a.hist_len; j += blockDim.x) {
    a.hist_dst[(size_t)rn * a.maxlen + j] = a.hist_src[(size_t)ro * a.maxlen + j];
    a.lp_dst[(size_t)rn * a.maxlen + j] = a.lp_src[(size_t)ro * a.maxlen + j];
  }
  if (threadIdx.x == 0) { a.prob_s[rn] = a.prob[ro]; a.last_s[rn] = a.last[ro]; }
  if (k == 0) {
    const int io = a.keep[img];
    for (int j = threadIdx.x; j < a.ldv; j += blockDim.x) a.v_s[(size_t)img * a.ldv + j] = a.v[(size_t)io * a.ldv + j];
    if (threadIdx.x == 0) { a.out_map_s[img] = a.out_map[io]; a.done_s[img] = a.done[io]; }
  }
}
__global__ void __launch_bounds__(128) beam_compact_scatter_kernel(BeamCompactArgs a) {
  const int rn = blockIdx.x, img = rn / a.K, k = rn - img * a.K;
  const bool vec = ((a.H1 | a.H2 | a.ld1 | a.ld2) & 3) == 0;
  if (vec) {
    for (int q = threadIdx.x; q < (a.H1 >> 2); q += blockDim.x) {
      const float4 hv = reinterpret_cast<const float4*>(a.h1_s + (size_t)rn * a.H1)[q];
      reinterpret_cast<float4*>(a.h1 + (size_t)rn * a.ld1)[q] = hv;
      reinterpret_cast<float4*>(a.c1 + (size_t)rn * a.H1)[q] = reinterpret_cast<const float4*>(a.c1_s + (size_t)rn * a.H1)[q];
      if (a.h1_hi) store_split4(a.h1_hi, a.h1_lo, (size_t)rn * a.ld1 + 4 * q, hv);
    }
    for (int q = threadIdx.x; q < (a.H2 >> 2); q += blockDim.x) {
      const float4 hv = reinterpret_cast<const float4*>(a.h2_s + (size_t)rn * a.H2)[q];
      reinterpret_cast<float4*>(a.h2 + (size_t)rn * a.ld2)[q] = hv;
      reinterpret_cast<float4*>(a.c2 + (size_t)rn * a.H2)[q] = reinterpret_cast<const float4*>(a.c2_s + (size_t)rn * a.H2)[q];
      if (a.h2_hi) store_split4(a.h2_hi, a.h2_lo, (size_t)rn * a.ld2 + 4 * q, hv);
    }
  } else {
  for (int j = threadIdx.x; j < a.H1; j += blockDim.x) {
    const float hv = a.h1_s[(size_t)rn * a.H1 + j];
    a.h1[(size_t)rn * a.ld1 + j] = hv;
    a.c1[(size_t)rn * a.H1 + j] = a.c1_s[(size_t)rn * a.H1 + j];
    if (a.h1_hi) { __nv_bfloat16 hh, ll; split_one(hv, hh, ll); a.h1_hi[(size_t)rn * a.ld1 + j] = hh; a.h1_lo[(size_t)rn * a.ld1 + j] = ll; }
  }
  for (int j = threadIdx.x; j < a.H2; j += blockDim.x) {
    const float hv = a.h2_s[(size_t)rn * a.H2 + j];
    a.h2[(size_t)rn * a.ld2 + j] = hv;
    a.c2[(size_t)rn * a.H2 + j] = a.c2_s[(size_t)rn * a.H2 + j];
    if (a.h2_hi) { __nv_bfloat16 hh, ll; split_one(hv, hh, ll); a.h2_hi[(size_t)rn * a.ld2 + j] = hh; a.h2_lo[(size_t)rn * a.ld2 + j] = ll; }
  }
  }
  if (threadIdx.x == 0) { a.prob[rn] = a.prob_s[rn]; a.last[rn] = a.last_s[rn]; }
  if (k == 0) {
    for (int j = threadIdx.x; j < a.ldv; j += blockDim.x) a.v[(size_t)img * a.ldv + j] = a.v_s[(size_t)img * a.ldv + j];
    // the survivor list may be one step old (the host decides from an asynchronous snapshot): a survivor can have ended since
    if (threadIdx.x == 0) { a.out_map[img] = a.out_map_s[img]; a.done[img] = a.done_s[img]; }
  }
}
void beam_compact(cudaStream_t s, const BeamCompactArgs& a) {
  if (a.n_keep <= 0) return;
  beam_compact_gather_kernel<<<a.n_keep * a.K, 128, 0, s>>>(a);
  beam_compact_scatter_kernel<<<a.n_keep * a.K, 128, 0, s>>>(a);
  if (g_counter) g_counter->n += 2;
}

void beam_advance(cudaStream_t s, const BeamAdvanceArgs& a) {
  beam_advance_kernel<<<a.n_img * a.K, 128, 0, s>>>(a);
  count_launch();
  if (a.fused) return;
  beam_mark_done_kernel<<<(a.n_img + 127) / 128, 128, 0, s>>>(a.sel_tok, a.n_img, a.K, a.step, a.nword, a.done, a.n_done);
  count_launch();
}

// called once per process from lrcn_create (never inside a stream capture)
void init_simt_kernels() {
  cudaFuncSetAttribute(softmax_ce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(softmax_ce_fused_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  cudaFuncSetAttribute(softmax_ce_fused_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  cudaFuncSetAttribute(softmax_ce_fused_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024);
  cudaFuncSetAttribute(softmax_ce_fused_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024);
  cudaFuncSetAttribute(beam_row_topk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(beam_row_topk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(beam_row_topk2_kernel<true, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(beam_row_topk2_kernel<false, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(beam_row_topk2_kernel<true, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(beam_row_topk2_kernel<false, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
}

}  // namespace lrcn
