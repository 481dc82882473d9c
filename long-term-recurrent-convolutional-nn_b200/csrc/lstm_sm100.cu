// lstm_sm100.cu -- one LSTM timestep as ONE tcgen05 kernel: recurrent GEMM (bf16 hi/lo split, fp32 TMEM
// accumulate) fused with the sigmoid/tanh cell update (forward) or with the cell adjoint (backward).
// Reference semantics: lstm() lrcn.jl:528-538 (gate order [forget|ingate|outgate|change]) and its adjoint
// (SURVEY.md §10.2).  The x-part of the gates (input projection + bias) is precomputed for all timesteps by
// one large GEMM (teacher forcing), so a step only has the recurrent product left:
//   forward : G_t[m][n]     += sum_k h_{t-1}[m][k] * W_h[k][n]          (K = H,  N = 4H)
//   backward: dh_rec[m][j]   = sum_n dG_{t+1}[m][n] * W_h[j][n]         (K = 4H, N = H)
//
// These products are skinny (M = batch), strictly sequential and bound by operand delivery, not by MMA rate:
// a single SM's TMA engine sustains ~55 GB/s and its shared-memory port 128 B/clk (measured, profiles/).
// So the step is spread over as many SMs as possible with the smallest per-CTA operand footprint:
//   * CTA tile = 64 batch rows (UMMA M=64) x NT columns; grid = (N/NT, B/64), up to 128 CTAs;
//   * the 8 CTAs of a thread-block cluster share the same 64 batch rows: each one TMA-loads 1/8 of the
//     activation tile and MULTICASTS it to all 8 (cp.async.bulk.tensor ... .multicast::cluster), so the
//     activation tile costs every SM 1/8 of its bytes; stage release is a multicast tcgen05.commit to the
//     empty barriers of all 8 CTAs;
//   * the weight operand is a K-major bf16 hi/lo copy laid out for the step (gate-interleaved rows for the
//     forward step so one thread owns f,i,o,g of its 16 units; transposed for the backward step), refreshed
//     once per training step.
// Epilogue: thread = batch row (TMEM lane), finishes its units in registers and writes c_t/h_t (+bf16 split
// of h_t) or dG_t (fp32 in place over the stored activations, + bf16 split) and dc.
#include "kernels.cuh"
#include "sm100_ptx.cuh"

#include <stdlib.h>

#include <string>

namespace lrcn {
using namespace ptx;

constexpr int LBK = 64;          // k-block (bf16 elements) = one 128-byte swizzle row
constexpr int LM = 64;           // batch rows per CTA (UMMA M)
constexpr int CL = 4;            // cluster size (4 packs 32 clusters = 128 CTAs onto the 148 SMs in ONE wave; 8 does not)
constexpr int L_THREADS = 320;   // warp 0 TMA, warp 1 MMA/TMEM, warps 2-9 epilogue (two warps per TMEM lane quadrant)
constexpr int A_HALF = LM * LBK * 2;          // 8 KiB: one of {hi, lo} of the activation k-block
constexpr int A_SLICE = (LM / CL) * LBK * 2;  // 2 KiB: the 16 rows this CTA loads and multicasts (forward)
constexpr int NT = 64;                        // accumulator columns per CTA (fwd: 16 units x 4 gates; bwd: 64 units)
constexpr int B_HALF = NT * LBK * 2;          // 8 KiB
constexpr int STAGE = 2 * A_HALF + 2 * B_HALF;  // 32 KiB
constexpr int STAGES = 3;                       // 96 KiB of stages: TWO step CTAs are resident per SM (the grid of a large layer is > 148 CTAs)
constexpr int RED_BYTES = CL * LM * (NT / CL) * 4;  // 16 KiB: split-K partials received from the cluster (backward)
constexpr int L_SMEM = STAGES * STAGE + RED_BYTES + 256 + 768;  // 115712 B = (228 KiB - 2 x 1 KiB reserved) / 2
constexpr uint32_t L_TMEM_COLS = 128;           // stacked accumulator: 128 lanes {hi rows; lo rows} x 128 columns {* W_hi | * W_lo}
constexpr int XLD = 68;                         // padded row (floats) of the lo*hi hand-over buffer [64 rows][64 columns], aliased on stage 0

__device__ __forceinline__ uint32_t dsmem_addr(uint32_t local_smem_addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta));
  return r;
}
__device__ __forceinline__ void dsmem_st_f4(uint32_t addr, float4 v) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
#define LRCN_TMEM_LD_16(taddr, v)                                                                                           \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"      \
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), \
                 "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])                                \
               : "r"(taddr)                                                                                                  \
               : "memory")
#define LRCN_TMEM_LD_8(taddr, v)                                                                         \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"                  \
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) \
               : "r"(taddr)                                                                              \
               : "memory")

// bf16x3 mode only (the fp32 mode keeps expf/tanhf in kernels_simt.cu): ~1e-7 absolute error, far inside the 1e-4 budget
__device__ __forceinline__ float sigm_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_fast(float x) {
  const float ax = fabsf(x);
  const float e = __expf(-2.0f * ax);                 // in (0,1]: no overflow, no cancellation blow-up
  const float t = __fdividef(1.0f - e, 1.0f + e);
  return copysignf(t, x);
}

struct StepParams {
  int B, H, num_kb, has_rec;
  float* gates;              // [B][4H]: fwd: x-part + bias in, activations out;  bwd: activations in, dG out
  const float* c_prev;       // [B][H]  c_{t-1}
  float* c_out;              // fwd: c_t
  float* h_out;              // fwd: h_t
  __nv_bfloat16* o_hi;       // fwd: bf16 split of h_t [B][H];  bwd: bf16 split of dG_t [B][4H]   (may be null)
  __nv_bfloat16* o_lo;
  const float* c_cur;        // bwd: c_t
  const float* dh_in;        // bwd: dL/dh_t from the layer above
  float* dc;                 // bwd carry: in dL/dc_t, out dL/dc_{t-1}
};

struct StepSmem {
  uint32_t base, full_bar0, empty_bar0, tfull_bar;
  uint32_t* tmem_slot;
  float* red;
  float* x;   // hand-over buffer [LM][XLD]: stage 0, free once the accumulator is committed (every load into it has been consumed)
};
__device__ __forceinline__ StepSmem step_smem(uint8_t* smem_raw) {
  StepSmem s;
  s.base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // same offset in every CTA of the cluster
  uint8_t* al = smem_raw + (s.base - smem_u32(smem_raw));
  s.x = reinterpret_cast<float*>(al);
  s.red = reinterpret_cast<float*>(al + STAGES * STAGE);
  uint64_t* bars = reinterpret_cast<uint64_t*>(al + STAGES * STAGE + RED_BYTES);
  s.full_bar0 = smem_u32(bars);
  s.empty_bar0 = smem_u32(bars + STAGES);
  s.tfull_bar = smem_u32(bars + 2 * STAGES);
  s.tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 1);
  return s;
}
// MMA issue loop shared by both directions.  Called by the WHOLE (converged) warp: the loop runs on warp-uniform values and one
// elected lane issues, so the descriptors stay in uniform registers (see elect_one(); inside `if (lane == 0)` every
// tcgen05.mma was wrapped in an ELECT / R2UR / branch waterfall: ~125 clk per MMA instead of ~80).
// STACKED SPLIT MMA: the stage holds {A_hi 64 rows; A_lo 64 rows} and {B_hi 64; B_lo 64} back to
// back, each a valid 128-row K-major SWIZZLE_128B tile, so ONE 128x128x16 tcgen05.mma per k-step yields all split products:
//   lanes 0-63 x cols 0-63: A_hi*B_hi | lanes 0-63 x cols 64-127: A_hi*B_lo | lanes 64-127 x cols 0-63: A_lo*B_hi | (lo*lo ignored)
// -- a third of the instructions of three M=64 MMAs (the step is bound by MMA instructions and operand delivery, not flops).
__device__ __forceinline__ void step_mma_loop(const StepSmem& sm, uint32_t tmem_base_any, int num_kb, bool mcast_release) {
  const uint32_t idesc = idesc_bf16(128, 128, false, false);
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_base_any, 0);
  for (int i = 0; i < num_kb; i++) {
    const int s = i % STAGES;
    mbar_wait(sm.full_bar0 + 8 * s, (i / STAGES) & 1);
    tc_fence_after();
    const uint32_t st = sm.base + s * STAGE;
    const uint32_t a = desc_lo_kmajor(st), b = desc_lo_kmajor(st + 2 * A_HALF);
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < LBK / 16; k++) umma_bf16_lo(tmem_base, a + 2u * k, b + 2u * k, idesc, (i > 0 || k > 0) ? 1u : 0u);
      if (mcast_release) umma_commit_mcast(sm.empty_bar0 + 8 * s, (uint16_t)((1u << CL) - 1));  // free in MY smem: tell all CL producers
      else umma_commit(sm.empty_bar0 + 8 * s);
    }
    __syncwarp();
  }
  if (elect_one()) umma_commit(sm.tfull_bar);
  __syncwarp();
}
// pair barrier of the hi-row warp and the lo-row warp that hold the same 32 batch rows and column half (64 threads)
__device__ __forceinline__ void pair_bar_sync(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }

// ---------------------------------------------------------------------------------------------- forward step
// A = h_{t-1} tile [64 rows][K=H] (each CTA loads 16 rows and multicasts them to the 4 CTAs of its cluster),
// B = gate-interleaved W_h rows [64][K].  UMMA M=64 accumulator: tile row r lives in TMEM lane (r%16) + 32*(r/16).
// Epilogue: 8 warps; warp (quad, half) reads units [8*half, +8) of its 16 rows, lanes 16-31 take units 4-7 by shuffle,
// so all 256 threads finish 4 units each.
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(L_THREADS, 2)
lstm_fwd_step_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                     const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo, const StepParams p) {
  extern __shared__ uint8_t smem_raw[];
  const StepSmem sm = step_smem(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int nt = blockIdx.x, m0 = blockIdx.y * LM;
  const int num_kb = p.has_rec ? p.num_kb : 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; s++) { mbar_init(sm.full_bar0 + 8 * s, 1); mbar_init(sm.empty_bar0 + 8 * s, CL); }
    mbar_init(sm.tfull_bar, 1);
    mbar_init_fence();
  }
  if (warp == 0 && lane == 0 && num_kb > 0) {
    prefetch_tensormap(&tmA_hi); prefetch_tensormap(&tmA_lo); prefetch_tensormap(&tmB_hi); prefetch_tensormap(&tmB_lo);
  }
  if (warp == 1) tmem_alloc<L_TMEM_COLS>(smem_u32(sm.tmem_slot));
  tc_fence_before();
  __syncthreads();
  if (num_kb > 0) cluster_sync_all();  // every CTA's barriers are initialised before any peer multicasts into them
  tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < num_kb; i++) {
        const int s = i % STAGES;
        mbar_wait(sm.empty_bar0 + 8 * s, ((i / STAGES) & 1) ^ 1);  // all CL CTAs have consumed this stage
        const uint32_t full = sm.full_bar0 + 8 * s;
        mbar_expect_tx(full, STAGE);  // CL multicast slices of A (hi, lo) + own B (hi, lo)
        const uint32_t st = sm.base + s * STAGE;
        const int k0 = i * LBK;
        const int arow = m0 + (int)rank * (LM / CL);
        tma_load_2d_mcast(st + rank * A_SLICE, &tmA_hi, full, k0, arow, (uint16_t)((1u << CL) - 1));
        tma_load_2d_mcast(st + A_HALF + rank * A_SLICE, &tmA_lo, full, k0, arow, (uint16_t)((1u << CL) - 1));
        tma_load_2d(st + 2 * A_HALF, &tmB_hi, full, k0, nt * NT);
        tma_load_2d(st + 2 * A_HALF + B_HALF, &tmB_lo, full, k0, nt * NT);
      }
    }
  } else if (warp == 1) {
    if (num_kb > 0) step_mma_loop(sm, tmem_base, num_kb, true);
  } else {
    // warp%4 fixes the TMEM lane quadrant: quadrants 0,1 hold the h_hi rows 0-63, quadrants 2,3 the h_lo rows 0-63 of the tile.
    // The (quad, half) warp and the (quad+2, half) warp own the same 32 rows x 8 units (32 columns, unit-major: col = u*4 + gate):
    // the hi warp finishes units 0-3, the lo warp units 4-7; each hands the other its part of the sum through shared memory.
    const int ew = warp - 2, quad = warp & 3, half = ew >> 2, upper = quad >> 1;
    constexpr int NH = NT / 4;                                 // 16 units per CTA
    const int row = (quad & 1) * 32 + lane;
    float acc[4][4];  // [gate][unit]
    if (num_kb > 0) {
      mbar_wait(sm.tfull_bar, 0);
      tc_fence_after();
      const uint32_t tl = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(32 * half);
      float* xr = sm.x + (size_t)row * XLD + 32 * half;
      uint32_t keep[16], give[16];
      if (!upper) {
        uint32_t w[16];
        LRCN_TMEM_LD_16(tl + 16u, give);       // h_hi*W_hi, units 4-7
        LRCN_TMEM_LD_16(tl + 64u + 16u, w);    // h_hi*W_lo, units 4-7
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; q++)
          *reinterpret_cast<float4*>(xr + 16 + 4 * q) = make_float4(__uint_as_float(give[4 * q]) + __uint_as_float(w[4 * q]), __uint_as_float(give[4 * q + 1]) + __uint_as_float(w[4 * q + 1]),
                                                                     __uint_as_float(give[4 * q + 2]) + __uint_as_float(w[4 * q + 2]), __uint_as_float(give[4 * q + 3]) + __uint_as_float(w[4 * q + 3]));
        LRCN_TMEM_LD_16(tl, keep);             // units 0-3
        LRCN_TMEM_LD_16(tl + 64u, w);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 16; c++) keep[c] = __float_as_uint(__uint_as_float(keep[c]) + __uint_as_float(w[c]));
      } else {
        LRCN_TMEM_LD_16(tl, give);             // h_lo*W_hi, units 0-3
        LRCN_TMEM_LD_16(tl + 16u, keep);       // units 4-7
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; q++)
          *reinterpret_cast<float4*>(xr + 4 * q) = make_float4(__uint_as_float(give[4 * q]), __uint_as_float(give[4 * q + 1]), __uint_as_float(give[4 * q + 2]), __uint_as_float(give[4 * q + 3]));
      }
      pair_bar_sync(1 + (quad & 1) * 2 + half);
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const float4 o4 = *reinterpret_cast<const float4*>(xr + 16 * upper + 4 * e);
        acc[0][e] = __uint_as_float(keep[4 * e]) + o4.x; acc[1][e] = __uint_as_float(keep[4 * e + 1]) + o4.y;
        acc[2][e] = __uint_as_float(keep[4 * e + 2]) + o4.z; acc[3][e] = __uint_as_float(keep[4 * e + 3]) + o4.w;
      }
    } else {
#pragma unroll
      for (int e = 0; e < 4; e++)
#pragma unroll
        for (int g = 0; g < 4; g++) acc[g][e] = 0.f;
    }
    const int H = p.H;
    const int m = m0 + row;
    const int j = nt * NH + 8 * half + 4 * upper;  // first of this thread's 4 units (H % 4 == 0: a float4 never straddles H)
    if (m < p.B && j < H) {
      float* grow = p.gates + (size_t)m * 4 * H + j;
      const size_t hidx = (size_t)m * H + j;
      const float4 gf = *reinterpret_cast<const float4*>(grow);
      const float4 gi = *reinterpret_cast<const float4*>(grow + H);
      const float4 go = *reinterpret_cast<const float4*>(grow + 2 * H);
      const float4 gg = *reinterpret_cast<const float4*>(grow + 3 * H);
      const float4 cp = *reinterpret_cast<const float4*>(p.c_prev + hidx);
      float f[4] = {gf.x, gf.y, gf.z, gf.w}, in[4] = {gi.x, gi.y, gi.z, gi.w}, o[4] = {go.x, go.y, go.z, go.w}, ch[4] = {gg.x, gg.y, gg.z, gg.w};
      const float cpv[4] = {cp.x, cp.y, cp.z, cp.w};
      float cn[4], hn[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        f[e] = sigm_fast(f[e] + acc[0][e]);
        in[e] = sigm_fast(in[e] + acc[1][e]);
        o[e] = sigm_fast(o[e] + acc[2][e]);
        ch[e] = tanh_fast(ch[e] + acc[3][e]);
        cn[e] = cpv[e] * f[e] + in[e] * ch[e];
        hn[e] = o[e] * tanh_fast(cn[e]);
      }
      *reinterpret_cast<float4*>(grow) = make_float4(f[0], f[1], f[2], f[3]);
      *reinterpret_cast<float4*>(grow + H) = make_float4(in[0], in[1], in[2], in[3]);
      *reinterpret_cast<float4*>(grow + 2 * H) = make_float4(o[0], o[1], o[2], o[3]);
      *reinterpret_cast<float4*>(grow + 3 * H) = make_float4(ch[0], ch[1], ch[2], ch[3]);
      *reinterpret_cast<float4*>(p.c_out + hidx) = make_float4(cn[0], cn[1], cn[2], cn[3]);
      *reinterpret_cast<float4*>(p.h_out + hidx) = make_float4(hn[0], hn[1], hn[2], hn[3]);
      if (p.o_hi) {
        __nv_bfloat16 hh[4], ll[4];
#pragma unroll
        for (int e = 0; e < 4; e++) split_bf16(hn[e], hh[e], ll[e]);
        *reinterpret_cast<uint2*>(p.o_hi + hidx) = *reinterpret_cast<uint2*>(hh);
        *reinterpret_cast<uint2*>(p.o_lo + hidx) = *reinterpret_cast<uint2*>(ll);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (num_kb > 0) cluster_sync_all();  // no CTA leaves while a peer may still multicast into its smem / arrive on its barriers
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<L_TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------- backward step
// dh_rec[m][j] = sum_n dG_{t+1}[m][n] * W_h[j][n], K = 4H.  Tile = 64 rows x 64 units; the 4 CTAs of a cluster split K
// (each streams a quarter of dG_{t+1} and of the transposed weights: 4x fewer bytes per SM than sharing the tile), then
// exchange their fp32 partials through distributed shared memory: CTA r receives columns [16r,16r+16) from all four,
// sums them and runs the cell adjoint for those 16 units.
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(L_THREADS, 2)
lstm_bwd_step_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                     const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo, const StepParams p) {
  extern __shared__ uint8_t smem_raw[];
  const StepSmem sm = step_smem(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int nt = blockIdx.x / CL, m0 = blockIdx.y * LM;
  const int kb_per = (p.num_kb + CL - 1) / CL;
  const int kb_begin = (int)rank * kb_per;
  const int num_kb = p.has_rec ? max(0, min(p.num_kb, kb_begin + kb_per) - kb_begin) : 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; s++) { mbar_init(sm.full_bar0 + 8 * s, 1); mbar_init(sm.empty_bar0 + 8 * s, 1); }
    mbar_init(sm.tfull_bar, 1);
    mbar_init_fence();
  }
  if (warp == 0 && lane == 0 && num_kb > 0) {
    prefetch_tensormap(&tmA_hi); prefetch_tensormap(&tmA_lo); prefetch_tensormap(&tmB_hi); prefetch_tensormap(&tmB_lo);
  }
  if (warp == 1) tmem_alloc<L_TMEM_COLS>(smem_u32(sm.tmem_slot));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < num_kb; i++) {
        const int s = i % STAGES;
        mbar_wait(sm.empty_bar0 + 8 * s, ((i / STAGES) & 1) ^ 1);
        const uint32_t full = sm.full_bar0 + 8 * s;
        mbar_expect_tx(full, STAGE);
        const uint32_t st = sm.base + s * STAGE;
        const int k0 = (kb_begin + i) * LBK;
        tma_load_2d(st, &tmA_hi, full, k0, m0);
        tma_load_2d(st + A_HALF, &tmA_lo, full, k0, m0);
        tma_load_2d(st + 2 * A_HALF, &tmB_hi, full, k0, nt * NT);
        tma_load_2d(st + 2 * A_HALF + B_HALF, &tmB_lo, full, k0, nt * NT);
      }
    }
  } else if (warp == 1) {
    if (num_kb > 0) step_mma_loop(sm, tmem_base, num_kb, false);
  } else if (p.has_rec) {
    // phase 1: the lo-row warps hand their dG_lo*W_hi part to the hi-row warps of the same rows through shared memory; those
    // scatter the CTA's partial (64 rows x 64 units, over this K-quarter) to the four owners through DSMEM.
    // receive buffer layout in every CTA: red[src][row][16] fp32
    const int ew = warp - 2, quad = warp & 3, half = ew >> 2, upper = quad >> 1;
    const int row = (quad & 1) * 32 + lane;
    float* xr = sm.x + (size_t)row * XLD + 32 * half;
    if (num_kb > 0) {
      mbar_wait(sm.tfull_bar, 0);
      tc_fence_after();
      const uint32_t tl = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(32 * half);
      if (upper) {
        uint32_t v[32];
        LRCN_TMEM_LD_32(tl, v);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 8; q++)
          *reinterpret_cast<float4*>(xr + 4 * q) = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
        pair_bar_sync(1 + (quad & 1) * 2 + half);
      } else {
        const uint32_t local = smem_u32(sm.red) + (uint32_t)(((int)rank * LM + row) * (NT / CL)) * 4u;
        pair_bar_sync(1 + (quad & 1) * 2 + half);
#pragma unroll
        for (int d2 = 0; d2 < 2; d2++) {  // columns [32*half + 16*d2, +16) belong to CTA dst
          uint32_t v[16], w[16];
          LRCN_TMEM_LD_16(tl + 16u * d2, v);
          LRCN_TMEM_LD_16(tl + 64u + 16u * d2, w);
          tmem_ld_wait();
          const uint32_t ra = dsmem_addr(local, (uint32_t)(2 * half + d2));
#pragma unroll
          for (int q = 0; q < 4; q++) {
            const float4 x4 = *reinterpret_cast<const float4*>(xr + 16 * d2 + 4 * q);
            dsmem_st_f4(ra + 16u * q, make_float4(__uint_as_float(v[4 * q]) + __uint_as_float(w[4 * q]) + x4.x, __uint_as_float(v[4 * q + 1]) + __uint_as_float(w[4 * q + 1]) + x4.y,
                                                   __uint_as_float(v[4 * q + 2]) + __uint_as_float(w[4 * q + 2]) + x4.z, __uint_as_float(v[4 * q + 3]) + __uint_as_float(w[4 * q + 3]) + x4.w));
          }
        }
      }
    } else if (!upper) {  // this K-quarter is empty (short K): contribute zeros
      const uint32_t local = smem_u32(sm.red) + (uint32_t)(((int)rank * LM + row) * (NT / CL)) * 4u;
#pragma unroll
      for (int d2 = 0; d2 < 2; d2++) {
        const uint32_t ra = dsmem_addr(local, (uint32_t)(2 * half + d2));
#pragma unroll
        for (int q = 0; q < 4; q++) dsmem_st_f4(ra + 16u * q, make_float4(0.f, 0.f, 0.f, 0.f));
      }
    }
  }
  if (p.has_rec) cluster_sync_all();  // release/acquire: all partials have landed (also orders the DSMEM stores before exit)

  if (warp >= 2) {
    // phase 2: this CTA owns units [nt*64 + 16*rank, +16) of its 64 rows; 256 threads x 4 units
    const int ew = warp - 2, quad = warp & 3, half = ew >> 2, upper = quad >> 1;
    const int row = (quad & 1) * 32 + lane;
    const int ug = 2 * half + upper;  // group of 4 units within the 16
    const int H = p.H;
    const int m = m0 + row;
    const int j = nt * NT + 16 * (int)rank + 4 * ug;
    if (m < p.B && j < H) {
      float rec[4] = {0.f, 0.f, 0.f, 0.f};
      if (p.has_rec) {
#pragma unroll
        for (int src = 0; src < CL; src++) {
          const float4 x = *reinterpret_cast<const float4*>(sm.red + (size_t)(src * LM + row) * (NT / CL) + 4 * ug);
          rec[0] += x.x; rec[1] += x.y; rec[2] += x.z; rec[3] += x.w;
        }
      }
      float* grow = p.gates + (size_t)m * 4 * H + j;
      const size_t hidx = (size_t)m * H + j;
      const float4 gf = *reinterpret_cast<const float4*>(grow);
      const float4 gi = *reinterpret_cast<const float4*>(grow + H);
      const float4 go = *reinterpret_cast<const float4*>(grow + 2 * H);
      const float4 gg = *reinterpret_cast<const float4*>(grow + 3 * H);
      const float4 cpv4 = *reinterpret_cast<const float4*>(p.c_prev + hidx);
      const float4 ccv4 = *reinterpret_cast<const float4*>(p.c_cur + hidx);
      const float4 dhv4 = *reinterpret_cast<const float4*>(p.dh_in + hidx);
      float4 dcv4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p.has_rec) dcv4 = *reinterpret_cast<const float4*>(p.dc + hidx);
      const float f[4] = {gf.x, gf.y, gf.z, gf.w}, in[4] = {gi.x, gi.y, gi.z, gi.w}, o[4] = {go.x, go.y, go.z, go.w}, ch[4] = {gg.x, gg.y, gg.z, gg.w};
      const float cpv[4] = {cpv4.x, cpv4.y, cpv4.z, cpv4.w}, ccv[4] = {ccv4.x, ccv4.y, ccv4.z, ccv4.w};
      const float dhv[4] = {dhv4.x, dhv4.y, dhv4.z, dhv4.w}, dci[4] = {dcv4.x, dcv4.y, dcv4.z, dcv4.w};
      float r0[4], r1[4], r2[4], r3[4], dco[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const float dh = dhv[e] + rec[e];
        const float tc = tanh_fast(ccv[e]);
        const float dcv = dci[e] + dh * o[e] * (1.f - tc * tc);
        const float dO = dh * tc, dF = dcv * cpv[e], dI = dcv * ch[e], dG = dcv * in[e];
        dco[e] = dcv * f[e];
        r0[e] = dF * f[e] * (1.f - f[e]);
        r1[e] = dI * in[e] * (1.f - in[e]);
        r2[e] = dO * o[e] * (1.f - o[e]);
        r3[e] = dG * (1.f - ch[e] * ch[e]);
      }
      *reinterpret_cast<float4*>(p.dc + hidx) = make_float4(dco[0], dco[1], dco[2], dco[3]);
      *reinterpret_cast<float4*>(grow) = make_float4(r0[0], r0[1], r0[2], r0[3]);
      *reinterpret_cast<float4*>(grow + H) = make_float4(r1[0], r1[1], r1[2], r1[3]);
      *reinterpret_cast<float4*>(grow + 2 * H) = make_float4(r2[0], r2[1], r2[2], r2[3]);
      *reinterpret_cast<float4*>(grow + 3 * H) = make_float4(r3[0], r3[1], r3[2], r3[3]);
      if (p.o_hi) {
        const size_t gidx = (size_t)m * 4 * H + j;
        const float* rr[4] = {r0, r1, r2, r3};
#pragma unroll
        for (int g = 0; g < 4; g++) {
          __nv_bfloat16 hh[4], ll[4];
#pragma unroll
          for (int e = 0; e < 4; e++) split_bf16(rr[g][e], hh[e], ll[e]);
          *reinterpret_cast<uint2*>(p.o_hi + gidx + (size_t)g * H) = *reinterpret_cast<uint2*>(hh);
          *reinterpret_cast<uint2*>(p.o_lo + gidx + (size_t)g * H) = *reinterpret_cast<uint2*>(ll);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<L_TMEM_COLS>(tmem_base);
  }
}

// ============================================================================================================
// Persistent sequence kernels: ONE launch runs all T timesteps of a layer.  The CTA's slice of the recurrent weights
// (bf16 hi/lo) is loaded once and stays resident in tensor and shared memory; per step only the activation chunk streams in
// by TMA.  Steps are separated by a grid barrier per (m-tile, chain) (release/acquire counter in global memory): the
// h_t (or dG_t) rows a step produces are read by the TMA engines of the other CTAs in the next step, so the releasing
// thread fences generic->async proxy before the release and the reading producer fences after the acquire.
// All waits are clock-bounded and trap instead of hanging.
// ============================================================================================================
constexpr int MAX_RES_KB = 8;                  // resident weight k-blocks (16 KiB each)

struct SeqParams {
  int B, H, T, num_kb;          // num_kb: k-blocks of the full K (fwd: H/64, bwd: 4H/64)
  float* acts;                  // [T*B][4H]
  float* hs;                    // fwd: [(T+1)*B][H] h slots (slot 0 = zeros)
  float* cs;                    // [(T+1)*B][H] c slots
  __nv_bfloat16* o_hi;          // fwd: shadows of hs;  bwd: shadows of acts
  __nv_bfloat16* o_lo;
  const float* dh_all;          // bwd: [T*B][H]
  float* dc;                    // unused by the sequence kernels (dc is carried in registers)
  unsigned int* counters;       // one per (m-tile, chain), zeroed before launch
  unsigned long long* trace;    // optional [T][4 chains][8] globaltimer stamps of CTA (0,0) (LRCN_SEQ_TRACE=1), else null
  float* dbias;                 // bwd (optional): bias gradient [4H] += column sums of dG over all rows and steps (zero on entry)
  int sync_flags;               // diagnostics (LRCN_SEQ_SYNC): 8 = fwd issuer waits for the whole chunk, 16 = no anti-phase delay,
                                // bits 8 and up = the anti-phase delay in ns (0: 2800)
};

__device__ __forceinline__ void grid_arrive(unsigned int* ctr) {
  asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
}
__device__ __forceinline__ void grid_wait(const unsigned int* ctr, unsigned int target) {
  const long long t0 = clock64();
  unsigned int spins = 0;
  while (true) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
    if (v >= target) break;
    if ((++spins & 63u) == 0u) {
      if (dev_aborted()) break;
      if (clock64() - t0 > WAIT_LIMIT_CLK) {
        printf("lrcn lstm_seq: grid barrier timeout (block %d,%d have %u want %u)\n", blockIdx.x, blockIdx.y, v, target);
        dev_abort_set();
        break;
      }
    }
  }
}
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// ============================================================================================================
// TRANSPOSED, TWO-CHAIN forward sequence kernel, recurrent weights resident in TENSOR MEMORY + shared memory ("seq4", round 2).
//
// What bounded the round-1 kernels (ncu, globaltimer traces and probes: profiles/r02_lstm.md, tools/probe_mma_rate.py):
//   * a step is a dependent CHAIN -- grid barrier -> TMA of the new h tile -> 32 MMAs -> cell epilogue -> release -- of 6-7 us
//     during which the SM's tensor pipe is busy a quarter of the time;
//   * the MMA phase is bound by INSTRUCTIONS, not flops: one thread issues a tcgen05.mma every ~69 clk whatever its shape, and
//     the tensor pipe needs >= 40-64 clk per instruction just to fetch the 128-row operand (M = 64 costs as much as M = 128;
//     A from TMEM costs 64 clk per instruction).  So the number of MMAs per CTA and step is the currency: 32 k-steps per
//     row group, and every extra row group re-fetches the whole weight block;
//   * 128 KiB of weights in shared memory leave ~80 KiB: a ring that cannot hold a step's activations, whose stage-reuse
//     dependencies (cluster-wide "empty" barriers) serialise the TMA producer behind the MMA consumer.
// Hence:
//   * roles swapped: the weight block {W_hi 64 gate rows; W_lo 64 gate rows} is the A operand (M = 128); its first
//     T4_KB_TMEM k-blocks live in TMEM (tcgen05.mma A-from-TMEM form: 128 lanes x 32 columns per k-block), the rest in
//     shared memory -- which frees enough shared memory for BOTH chains' whole activation chunks to have a fixed home;
//   * the CTA's 64 rows are two independent chains of 32 rows: the streamed chunk {h_hi 32 rows; h_lo 32 rows} is the B
//     operand (N = 64), so one 128 x 64 x 16 MMA per k-step yields W_hi*h_hi, W_hi*h_lo, W_lo*h_hi (and an ignored
//     W_lo*h_lo): accumulator lane = gate column (0-63: W_hi, 64-127: W_lo), column = batch row (0-31: h_hi, 32-63: h_lo);
//   * every chain has its own grid-barrier counter, TMA-producer warp, MMA-issuer warp, TMEM accumulator, chunk buffer and
//     epilogue team: two issue loops and two epilogues run in parallel, one chain computes while the other communicates.
//     No stage ring and no "empty" barriers: chunk (t+1, c) may overwrite chunk (t, c) once chain c's grid barrier for step
//     t+1 is open, because every CTA of the cluster (the multicast group) arrives on it only after ITS MMAs of step t;
//   * all 128 threads of a team run the cell update (2 units x 2 rows each) after a transposing hand-over through shared
//     memory, with 64-byte-contiguous global accesses per (row, gate);
//   * small batches: B <= 128 runs ONE chain per CTA (32-row m-tiles, twice the CTAs).
// ============================================================================================================
constexpr int T4_MAXCH = 2;                       // chains per CTA (upper bound)
constexpr int T4_ROWS = 32;                       // batch rows per chain
constexpr int T4_BHALF = T4_ROWS * LBK * 2;       // 4 KiB: {hi | lo} of one k-block of a chain
constexpr int T4_BSTAGE = 2 * T4_BHALF;           // 8 KiB
constexpr int T4_CHUNK = MAX_RES_KB * T4_BSTAGE;  // 64 KiB: a chain's activations of one step
constexpr int T4_KB_TMEM = 4;                     // weight k-blocks held in TMEM; k-blocks [T4_KB_TMEM, 8) are held in shared memory
constexpr int T4_WSMEM = (MAX_RES_KB - T4_KB_TMEM) * 2 * B_HALF;  // 64 KiB
constexpr int T4_SLD = 33;                        // padded row (floats) of the transposing hand-over buffer [128 lanes][32 rows]
constexpr int T4_SBYTES = 128 * T4_SLD * 4;       // 16896 B per team
constexpr int T4_THREADS = 32 * (T4_MAXCH + T4_MAXCH + 4 * T4_MAXCH);  // warps 0-1 TMA producers, 2-3 MMA issuers (warp 2 owns TMEM), 4-11 epilogue (2 teams x 4 quadrants)
constexpr int T4_TEAM = 128;
constexpr uint32_t T4_TMEM_COLS = 256;            // [0,128): 2 accumulators x 64 columns; [128,256): the first 4 k-blocks of the stacked weight block
constexpr uint32_t T4_WCOL = 128;

struct Seq4Smem {
  uint32_t wres, chunk, full0, wbar, tfull0, tempty0, started0;
  uint32_t* tmem_slot;
  float* S;  // [2 teams][128][T4_SLD]
};
__device__ __forceinline__ Seq4Smem seq4_smem(uint8_t* smem_raw) {
  Seq4Smem s;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* al = smem_raw + (base - smem_u32(smem_raw));
  s.wres = base;                       // weight k-blocks [T4_KB_TMEM, 8): {W_hi 8 KiB | W_lo 8 KiB} each
  s.chunk = base + T4_WSMEM;           // [chain][k-block]{hi 4 KiB | lo 4 KiB}
  uint8_t* after = al + (size_t)T4_WSMEM + (size_t)T4_MAXCH * T4_CHUNK;
  s.S = reinterpret_cast<float*>(after);
  uint64_t* bars = reinterpret_cast<uint64_t*>(after + T4_MAXCH * T4_SBYTES);
  s.full0 = smem_u32(bars);                                        // [chain][k-block]
  s.wbar = smem_u32(bars + T4_MAXCH * MAX_RES_KB);
  s.tfull0 = smem_u32(bars + T4_MAXCH * MAX_RES_KB + 1);           // [chain]
  s.tempty0 = smem_u32(bars + T4_MAXCH * MAX_RES_KB + 1 + T4_MAXCH);
  s.started0 = smem_u32(bars + T4_MAXCH * MAX_RES_KB + 1 + 2 * T4_MAXCH);
  s.tmem_slot = reinterpret_cast<uint32_t*>(bars + T4_MAXCH * MAX_RES_KB + 1 + 3 * T4_MAXCH);
  return s;
}
static int seq4_smem_bytes() { return T4_WSMEM + T4_MAXCH * T4_CHUNK + T4_MAXCH * T4_SBYTES + 1024 + 256; }

#define T4_TRACE(c, slot) do { if (p.trace && blockIdx.x == 0 && blockIdx.y == 0) p.trace[((size_t)t * 4 + (c)) * 8 + (slot)] = gtime(); } while (0)
// named barriers of an epilogue team (128 threads): 2 + team
__device__ __forceinline__ void team_bar_sync(int team) { asm volatile("bar.sync %0, %1;" ::"r"(2 + team), "n"(T4_TEAM) : "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]: A is 128 lanes x 8 columns (16 bf16 of K per lane, two per 32-bit column, K ascending)
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(DESC_HI_SW128)
      : "memory");
}
#define LRCN_TMEM_ST_16(taddr, v)                                                                                       \
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" \
               ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), \
                 "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])                      \
               : "memory")

// wp_hi / wp_lo: the gate-interleaved recurrent weights [rows][w_ld] (lstm_prepare_weights2), K contiguous; tmB_*: their tensor maps
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T4_THREADS, 1)
lstm_fwd_seq4_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                     const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo, const __nv_bfloat16* __restrict__ wp_hi,
                     const __nv_bfloat16* __restrict__ wp_lo, const int w_rows, const int w_ld, const SeqParams p, const int nch) {
  extern __shared__ uint8_t smem_raw[];
  const Seq4Smem sm = seq4_smem(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int nt = blockIdx.x, mt = blockIdx.y, m0 = mt * T4_ROWS * nch;
  const int num_kb = p.num_kb, T = p.T, B = p.B, H = p.H;
  const int kb_tmem = min(num_kb, T4_KB_TMEM);
  const unsigned int ctas_per_mtile = gridDim.x;
  unsigned int* ctr = p.counters + T4_MAXCH * mt;  // [chain]

  if (threadIdx.x == 0) {
    for (int i = 0; i < T4_MAXCH * MAX_RES_KB; i++) mbar_init(sm.full0 + 8 * i, 1);
    mbar_init(sm.wbar, 1);
    for (int c = 0; c < T4_MAXCH; c++) { mbar_init(sm.tfull0 + 8 * c, 2); mbar_init(sm.tempty0 + 8 * c, 1); mbar_init(sm.started0 + 8 * c, 1); }
    mbar_init_fence();
  }
  if (warp == 0 && lane == 0) { prefetch_tensormap(&tmA_hi); prefetch_tensormap(&tmA_lo); prefetch_tensormap(&tmB_hi); prefetch_tensormap(&tmB_lo); }
  if (warp == T4_MAXCH) tmem_alloc<T4_TMEM_COLS>(smem_u32(sm.tmem_slot));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_slot;

  // Resident weights, once.  They were written by the prep kernels more than two launches upstream (PDL discipline, kernels.cuh),
  // so they are read BEFORE the dependency wait and the load overlaps the previous kernel's tail.
  // (1) k-blocks [T4_KB_TMEM, num_kb) -> shared memory by TMA;
  if (warp == 0 && lane == 0) {
    const int n_sm = num_kb - kb_tmem;
    if (n_sm > 0) {
      mbar_expect_tx(sm.wbar, (uint32_t)n_sm * 2 * B_HALF);
      for (int i = 0; i < n_sm; i++) {
        tma_load_2d(sm.wres + i * 2 * B_HALF, &tmB_hi, sm.wbar, (kb_tmem + i) * LBK, nt * NT);
        tma_load_2d(sm.wres + i * 2 * B_HALF + B_HALF, &tmB_lo, sm.wbar, (kb_tmem + i) * LBK, nt * NT);
      }
    } else {
      mbar_arrive(sm.wbar);
    }
  }
  // (2) k-blocks [0, kb_tmem) -> TMEM by the epilogue warps, which own the TMEM lanes of their quadrant: lane = stacked weight row
  // (0-63: W_hi rows of this n-tile, 64-127: W_lo rows), 32-bit column j = K elements 2j, 2j+1 -- exactly the uint32 words of the
  // K-contiguous bf16 row.
  if (warp >= 2 * T4_MAXCH) {
    const int quad = warp & 3, khalf = (warp - 2 * T4_MAXCH) >> 2;  // the two warps of a quadrant split the K range
    const int srow = 32 * quad + lane;                              // stacked row = TMEM lane
    const int wrow = nt * NT + (srow & 63);
    const __nv_bfloat16* src = (srow < 64 ? wp_hi : wp_lo) + (size_t)wrow * w_ld;
    const bool row_ok = wrow < w_rows;
    const int ncol = kb_tmem * (LBK / 2);                           // 32-bit columns in use (32 per k-block)
    for (int c0 = khalf * 16; c0 < ncol; c0 += 32) {
      uint32_t v[16];
#pragma unroll
      for (int q = 0; q < 4; q++) {
        uint4 x = make_uint4(0u, 0u, 0u, 0u);
        const int k0 = 2 * (c0 + 4 * q);  // first K element of this 16-byte piece; rows are padded to multiples of 8 elements
        if (row_ok && k0 < w_ld) x = __ldg(reinterpret_cast<const uint4*>(src + k0));
        v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
      }
      LRCN_TMEM_ST_16(tmem_base + ((uint32_t)(quad * 32) << 16) + T4_WCOL + (uint32_t)c0, v);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // every CTA's barriers are initialised before any peer multicasts into them
  tc_fence_after();
  pdl_wait();
  pdl_trigger();

  if (warp < T4_MAXCH) {
    // ===================== TMA producers: warp c serves chain c -- and issues the SECOND half of the chain's MMAs =====================
    // 32 dependent-issue MMAs at ~80 clk each were the longest phase of a step.  The producer warp is idle between its TMA
    // issue and the next grid barrier, so it issues k-blocks [num_kb/2, num_kb) into the SAME accumulator while the issuer
    // warp does [0, num_kb/2): tcgen05.mma executes in issue order, so accumulating from two threads is safe once the
    // issuer's first MMA of the step (the one that overwrites the accumulator) has been issued (`started` barrier).
    const int c = __shfl_sync(0xffffffffu, warp, 0);
    if (c < nch) {
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc = idesc_bf16(128, 2 * T4_ROWS, false, false);
      const uint32_t acc = tb + (uint32_t)(2 * T4_ROWS * c);
      const uint32_t buf = sm.chunk + (uint32_t)c * T4_CHUNK;
      const uint32_t fullc = sm.full0 + 8 * (c * MAX_RES_KB);
      const int kb_split = (num_kb + 1) / 2;
      mbar_wait(sm.wbar, 0);
      for (int t = 1; t < T; t++) {
        if (lane == 0) {
          grid_wait(ctr + c, (unsigned int)t * ctas_per_mtile);  // h_{t-1} rows of this chain are complete; the cluster's MMAs of step t-1 are done
          T4_TRACE(c, 0);
          fence_proxy_async_global();
          const int arow = t * B + m0 + T4_ROWS * c;  // slot t of hs = h_{t-1}
          for (int kb = 0; kb < num_kb; kb++) mbar_expect_tx(fullc + 8 * kb, T4_BSTAGE);
          for (int kb = (int)rank; kb < num_kb; kb += CL) {  // k-block kb is fetched by rank kb % CL and multicast to the cluster
            const uint32_t st = buf + kb * T4_BSTAGE;
            tma_load_2d_mcast(st, &tmA_hi, fullc + 8 * kb, kb * LBK, arow, (uint16_t)((1u << CL) - 1));
            tma_load_2d_mcast(st + T4_BHALF, &tmA_lo, fullc + 8 * kb, kb * LBK, arow, (uint16_t)((1u << CL) - 1));
          }
          T4_TRACE(c, 1);
        }
        __syncwarp();
        // second half of the k-blocks (converged warp, elected lane: see elect_one())
        mbar_wait(sm.started0 + 8 * c, (t - 1) & 1);  // the issuer warp has issued this step's first (overwriting) MMA
        tc_fence_after();
        for (int kb = kb_split; kb < num_kb; kb++) {
          mbar_wait(fullc + 8 * kb, (t - 1) & 1);
          tc_fence_after();
          const uint32_t b_lo = desc_lo_kmajor(buf + kb * T4_BSTAGE);
          if (kb < T4_KB_TMEM) {
            const uint32_t a_col = tb + T4_WCOL + (uint32_t)(kb * (LBK / 2));
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < LBK / 16; k++) umma_bf16_ts(acc, a_col + 8u * k, b_lo + 2u * k, idesc, 1u);
            }
          } else {
            const uint32_t a_lo = desc_lo_kmajor(sm.wres + (kb - T4_KB_TMEM) * 2 * B_HALF);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < LBK / 16; k++) umma_bf16_lo(acc, a_lo + 2u * k, b_lo + 2u * k, idesc, 1u);
            }
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(sm.tfull0 + 8 * c);  // tfull counts two commits: this warp's and the issuer warp's
        __syncwarp();
      }
    }
  } else if (warp < 2 * T4_MAXCH) {
    // ===================== MMA issuers: warp 2 + c serves chain c =====================
    // The whole warp runs the loops CONVERGED on warp-uniform values and one elected lane issues (see elect_one()).
    const int c = __shfl_sync(0xffffffffu, warp - T4_MAXCH, 0);
    if (c < nch) {
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc = idesc_bf16(128, 2 * T4_ROWS, false, false);
      const uint32_t acc = tb + (uint32_t)(2 * T4_ROWS * c);
      const uint32_t buf = sm.chunk + (uint32_t)c * T4_CHUNK;
      const uint32_t fullc = sm.full0 + 8 * (c * MAX_RES_KB);
      mbar_wait(sm.wbar, 0);
      for (int t = 1; t < T; t++) {
        if (t >= 2) mbar_wait(sm.tempty0 + 8 * c, (t - 2) & 1);  // epilogue (t-1, c) has drained this accumulator
        tc_fence_after();
        if (p.sync_flags & 8) {  // diagnostics: wait for the whole chunk first, so that slot 3 = data arrival and slot 4 - slot 3 = pure MMA issue
          for (int kb = 0; kb < num_kb; kb++) { mbar_wait(fullc + 8 * kb, (t - 1) & 1); if (kb == 0 && lane == 0) T4_TRACE(c, 2); }
          if (lane == 0) T4_TRACE(c, 3);
        }
        const int kb_split = (num_kb + 1) / 2;  // this warp: k-blocks [0, kb_split); the producer warp: the rest
        for (int kb = 0; kb < kb_split; kb++) {
          if (!(p.sync_flags & 8)) {
            mbar_wait(fullc + 8 * kb, (t - 1) & 1);
            if (lane == 0) { if (kb == 0) T4_TRACE(c, 2); else if (kb == kb_split - 1) T4_TRACE(c, 3); }
          }
          tc_fence_after();
          const uint32_t b_lo = desc_lo_kmajor(buf + kb * T4_BSTAGE);
          if (kb < T4_KB_TMEM) {
            const uint32_t a_col = tb + T4_WCOL + (uint32_t)(kb * (LBK / 2));
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < LBK / 16; k++) umma_bf16_ts(acc, a_col + 8u * k, b_lo + 2u * k, idesc, (kb | k) ? 1u : 0u);
              if (kb == 0) mbar_arrive(sm.started0 + 8 * c);
            }
          } else {
            const uint32_t a_lo = desc_lo_kmajor(sm.wres + (kb - T4_KB_TMEM) * 2 * B_HALF);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < LBK / 16; k++) umma_bf16_lo(acc, a_lo + 2u * k, b_lo + 2u * k, idesc, 1u);
            }
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(sm.tfull0 + 8 * c);
        __syncwarp();
        if (lane == 0) T4_TRACE(c, 4);
      }
    }
  } else {
    // ===================== epilogue teams: team c finishes chain c =====================
    const int ew = warp - 2 * T4_MAXCH, quad = warp & 3, c = ew >> 2;
    const int tid = (ew & 3) * 32 + lane;           // 0..127 inside the team (its four warps cover the four TMEM lane quadrants)
    float* S = sm.S + (size_t)c * 128 * T4_SLD;
    if (c < nch) {
      // cell ownership: rows rr and rr + 16 of the chain, units 2*up, 2*up+1 of the CTA's 16
      const int rr = tid >> 3, up = tid & 7;
      const int j = nt * (NT / 4) + 2 * up;
      float creg[2][2];
      float2 xg[2][4];
      bool active[2];
      int mrow[2];
#pragma unroll
      for (int q = 0; q < 2; q++) {
        mrow[q] = m0 + T4_ROWS * c + rr + 16 * q;
        active[q] = mrow[q] < B && j < H;
        creg[q][0] = creg[q][1] = 0.f;
#pragma unroll
        for (int g = 0; g < 4; g++) xg[q][g] = make_float2(0.f, 0.f);
        if (active[q]) {
          const float* g0 = p.acts + (size_t)mrow[q] * 4 * H + j;
#pragma unroll
          for (int g = 0; g < 4; g++) xg[q][g] = *reinterpret_cast<const float2*>(g0 + g * H);
        }
      }
      for (int t = 0; t < T; t++) {
        if (t > 0) {
          mbar_wait(sm.tfull0 + 8 * c, (t - 1) & 1);
          if (tid == 0) T4_TRACE(c, 5);
          tc_fence_after();
          // accumulator lane = 32*quad + lane: gate column (W_hi: 0-63 | W_lo: 64-127); columns 0-31: * h_hi, 32-63: * h_lo
          const uint32_t tl = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(2 * T4_ROWS * c);
          float* dst = S + (size_t)(32 * quad + lane) * T4_SLD;
          uint32_t v[32];
          LRCN_TMEM_LD_32(tl, v);
          if (quad < 2) {
            uint32_t w[32];
            LRCN_TMEM_LD_32(tl + T4_ROWS, w);
            tmem_ld_wait();
#pragma unroll
            for (int r = 0; r < T4_ROWS; r++) dst[r] = __uint_as_float(v[r]) + __uint_as_float(w[r]);
          } else {
            tmem_ld_wait();
#pragma unroll
            for (int r = 0; r < T4_ROWS; r++) dst[r] = __uint_as_float(v[r]);
          }
          tc_fence_before();
          team_bar_sync(c);
        }
        float gf[2][2], gi[2][2], go[2][2], gc[2][2], hn[2][2];
#pragma unroll
        for (int q = 0; q < 2; q++) {
          float a[4][2];  // [gate][unit] recurrent part of the pre-activations
#pragma unroll
          for (int e = 0; e < 2; e++)
#pragma unroll
            for (int g = 0; g < 4; g++) {
              const int gl = 4 * (2 * up + e) + g;  // weight rows are unit-major: row u*4 + gate
              a[g][e] = t > 0 ? S[(size_t)gl * T4_SLD + rr + 16 * q] + S[(size_t)(64 + gl) * T4_SLD + rr + 16 * q] : 0.f;
            }
          if (active[q]) {
            const float xf[2] = {xg[q][0].x, xg[q][0].y}, xi[2] = {xg[q][1].x, xg[q][1].y};
            const float xo[2] = {xg[q][2].x, xg[q][2].y}, xc[2] = {xg[q][3].x, xg[q][3].y};
            __nv_bfloat16 hh[2], ll[2];
#pragma unroll
            for (int e = 0; e < 2; e++) {
              gf[q][e] = sigm_fast(xf[e] + a[0][e]);
              gi[q][e] = sigm_fast(xi[e] + a[1][e]);
              go[q][e] = sigm_fast(xo[e] + a[2][e]);
              gc[q][e] = tanh_fast(xc[e] + a[3][e]);
              creg[q][e] = creg[q][e] * gf[q][e] + gi[q][e] * gc[q][e];
              hn[q][e] = go[q][e] * tanh_fast(creg[q][e]);
              split_bf16(hn[q][e], hh[e], ll[e]);
            }
            const size_t hnext = ((size_t)(t + 1) * B + mrow[q]) * H + j;
            *reinterpret_cast<uint32_t*>(p.o_hi + hnext) = *reinterpret_cast<uint32_t*>(hh);
            *reinterpret_cast<uint32_t*>(p.o_lo + hnext) = *reinterpret_cast<uint32_t*>(ll);
          }
        }
        // every thread of the team is past its reads of S and its h stores: one thread frees the accumulator for the issuer
        // and publishes h_t of this chain (bar.sync orders the team's stores before the gpu-scope release; the reading
        // producers fence generic->async proxy after their acquire)
        team_bar_sync(c);
        if (tid == 0) {
          T4_TRACE(c, 6);
          // Anti-phase the two chains once: they are symmetric and would otherwise run in lockstep, sharing the tensor pipe
          // during the same 2 us and idling together through release / barrier / TMA latency.  A one-off delay of chain 1's
          // first publish by about half a step makes one chain compute while the other communicates; nothing pulls them back.
          if (t == 0 && c == 1 && nch > 1 && !(p.sync_flags & 16)) {
            const unsigned long long t0 = gtime();
            while (gtime() - t0 < (unsigned long long)(p.sync_flags >> 8 ? (p.sync_flags >> 8) : 2800)) {}
          }
          if (t > 0) mbar_arrive(sm.tempty0 + 8 * c);
          if (t + 1 < T) { fence_proxy_async_global(); grid_arrive(ctr + c); }
          T4_TRACE(c, 7);
        }
#pragma unroll
        for (int q = 0; q < 2; q++) {
          if (active[q]) {  // off the critical path: what only later kernels read
            const size_t hnext = ((size_t)(t + 1) * B + mrow[q]) * H + j;
            float* grow = p.acts + ((size_t)t * B + mrow[q]) * 4 * H + j;
            *reinterpret_cast<float2*>(grow) = make_float2(gf[q][0], gf[q][1]);
            *reinterpret_cast<float2*>(grow + H) = make_float2(gi[q][0], gi[q][1]);
            *reinterpret_cast<float2*>(grow + 2 * H) = make_float2(go[q][0], go[q][1]);
            *reinterpret_cast<float2*>(grow + 3 * H) = make_float2(gc[q][0], gc[q][1]);
            *reinterpret_cast<float2*>(p.cs + hnext) = make_float2(creg[q][0], creg[q][1]);
            *reinterpret_cast<float2*>(p.hs + hnext) = make_float2(hn[q][0], hn[q][1]);
            if (t + 1 < T) {  // prefetch the next step's x-part
              const float* gn = p.acts + ((size_t)(t + 1) * B + mrow[q]) * 4 * H + j;
#pragma unroll
              for (int g = 0; g < 4; g++) xg[q][g] = *reinterpret_cast<const float2*>(gn + g * H);
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // no CTA leaves while a peer may still multicast into its shared memory
  if (warp == T4_MAXCH) {
    tc_fence_after();
    tmem_dealloc<T4_TMEM_COLS>(tmem_base);
  }
}

// ============================================================================================================
// TRANSPOSED, TWO-CHAIN backward sequence kernel, recurrent weights resident in TENSOR MEMORY ("bwd4", round 2).
// Same construction as lstm_fwd_seq4_kernel (see there for the measurements behind it), for
//   dh_rec[m][j] = sum_n dG_{t+1}[m][n] * W_h[j][n],  K = 4H.
//   * the 4 CTAs of a cluster are the K-quarters of one 64-unit output tile (K = 4H is too long for one CTA's weights);
//     each holds its slice of the transposed weights {WhT_hi 64 units; WhT_lo 64 units} x K/4 as the A operand (M = 128)
//     entirely in TMEM (128 lanes x 32 columns per k-block, <= 8 k-blocks) -- shared memory holds no weights;
//   * the CTA's 64 batch rows are two independent chains of 32 rows: B operand = {dG_hi 32 rows; dG_lo 32 rows} (N = 64) of
//     the K-slice, 64 KiB per chain and step with a fixed home (plain TMA: every K-quarter streams different bytes);
//     accumulator lane = unit (0-63: * WhT_hi, 64-127: * WhT_lo), column = batch row (0-31: dG_hi, 32-63: dG_lo);
//   * per chain: own grid-barrier counter, producer warp, issuer warp (converged elect loop), accumulator and epilogue team.
//     The team drops the accumulator into a shared-memory buffer [128 lanes][32 rows] and one thread SENDS every cluster
//     rank the rows of the 16 units that rank finishes (W_hi part and W_lo part: two 2 KiB cp.async.bulk copies
//     shared::cta -> shared::cluster per rank, completing bytes on the receiver's mbarrier -- per-thread st.shared::cluster
//     stores cost 3 us per step here); every thread then waits for the 4 x 2 partials of ITS units, sums them and runs the
//     cell adjoint (4 units x 1 row per thread, 16-byte global accesses).  No "buffer free" handshake is needed: a rank sends step n+1 only after the grid barrier of that step,
//     which every CTA of the m-tile passes after it has consumed the partials of step n.
// ============================================================================================================
constexpr int B4_PART = 16 * T4_SLD * 4;            // 2112 B: 16 unit rows of the hand-over buffer = one bulk copy
constexpr int B4_RED = CL * 2 * B4_PART;            // 16896 B per chain: receive buffer [src][hi-part | lo-part][16 units][T4_SLD]
constexpr uint32_t B4_TMEM_COLS = 512;              // [0,128): 2 accumulators x 64 columns; [128,384): the weight slice, up to 8 k-blocks
constexpr uint32_t B4_WCOL = 128;

struct Bwd4Smem {
  uint32_t chunk, full0, tfull0, tempty0, redfull0, started0;
  uint32_t* tmem_slot;
  float* S;    // [2 teams][128][T4_SLD]
  float* red;  // [2 chains][CL src][2 parts][16][T4_SLD]
};
__device__ __forceinline__ Bwd4Smem bwd4_smem(uint8_t* smem_raw) {
  Bwd4Smem s;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* al = smem_raw + (base - smem_u32(smem_raw));
  s.chunk = base;  // [chain][k-block]{hi 4 KiB | lo 4 KiB}
  uint8_t* after = al + (size_t)T4_MAXCH * T4_CHUNK;
  s.S = reinterpret_cast<float*>(after);
  s.red = reinterpret_cast<float*>(after + T4_MAXCH * T4_SBYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(after + T4_MAXCH * T4_SBYTES + T4_MAXCH * B4_RED);
  s.full0 = smem_u32(bars);                                        // [chain][k-block]
  s.tfull0 = smem_u32(bars + T4_MAXCH * MAX_RES_KB);               // [chain]
  s.tempty0 = smem_u32(bars + T4_MAXCH * MAX_RES_KB + T4_MAXCH);
  s.redfull0 = smem_u32(bars + T4_MAXCH * MAX_RES_KB + 2 * T4_MAXCH);
  s.started0 = smem_u32(bars + T4_MAXCH * MAX_RES_KB + 3 * T4_MAXCH);
  s.tmem_slot = reinterpret_cast<uint32_t*>(bars + T4_MAXCH * MAX_RES_KB + 4 * T4_MAXCH);
  return s;
}
static int bwd4_smem_bytes() { return T4_MAXCH * T4_CHUNK + T4_MAXCH * T4_SBYTES + T4_MAXCH * B4_RED + 1024 + 256; }
// bulk copy of local shared memory into a cluster peer's shared memory (DMA engine); completes bytes on the PEER's mbarrier
__device__ __forceinline__ void dsmem_bulk_copy(uint32_t dst_cluster_addr, uint32_t src_cta_addr, uint32_t bytes, uint32_t mbar_cluster_addr) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst_cluster_addr), "r"(src_cta_addr), "r"(bytes), "r"(mbar_cluster_addr) : "memory");
}

// wt_hi / wt_lo: transposed recurrent weights [w_rows units][K = 4H] (lstm_prepare_weights2), K contiguous
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T4_THREADS, 1)
lstm_bwd_seq4_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo, const __nv_bfloat16* __restrict__ wt_hi,
                     const __nv_bfloat16* __restrict__ wt_lo, const int w_rows, const SeqParams p, const int nch) {
  extern __shared__ uint8_t smem_raw[];
  const Bwd4Smem sm = bwd4_smem(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int nt = blockIdx.x / CL, mt = blockIdx.y, m0 = mt * T4_ROWS * nch;
  const int T = p.T, B = p.B, H = p.H;
  const int kb_per = (p.num_kb + CL - 1) / CL;                                   // k-blocks of the full K = 4H per rank (<= 8)
  const int kb_begin = (int)rank * kb_per;
  const int nkb = max(0, min(p.num_kb, kb_begin + kb_per) - kb_begin);
  const unsigned int ctas_per_mtile = gridDim.x;
  unsigned int* ctr = p.counters + T4_MAXCH * mt;  // [chain]

  if (threadIdx.x == 0) {
    for (int i = 0; i < T4_MAXCH * MAX_RES_KB; i++) mbar_init(sm.full0 + 8 * i, 1);
    for (int c = 0; c < T4_MAXCH; c++) {
      mbar_init(sm.tfull0 + 8 * c, 2); mbar_init(sm.tempty0 + 8 * c, 1); mbar_init(sm.redfull0 + 8 * c, 1); mbar_init(sm.started0 + 8 * c, 1);
    }
    mbar_init_fence();
  }
  if (warp == 0 && lane == 0) { prefetch_tensormap(&tmA_hi); prefetch_tensormap(&tmA_lo); }
  if (warp == T4_MAXCH) tmem_alloc<B4_TMEM_COLS>(smem_u32(sm.tmem_slot));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_slot;

  // Resident weight slice -> TMEM, once, by the epilogue warps (lane = stacked weight row: 0-63 WhT_hi units of this tile,
  // 64-127 WhT_lo; 32-bit column j = K elements 2j, 2j+1 of this rank's K-quarter).  Written by the prep kernels more than two
  // launches upstream (PDL discipline, kernels.cuh): read BEFORE the dependency wait.
  if (warp >= 2 * T4_MAXCH) {
    const int quad = warp & 3, khalf = (warp - 2 * T4_MAXCH) >> 2;
    const int srow = 32 * quad + lane;
    const int wrow = nt * NT + (srow & 63);
    const size_t K = 4 * (size_t)H;
    const __nv_bfloat16* src = (srow < 64 ? wt_hi : wt_lo) + (size_t)wrow * K + (size_t)kb_begin * LBK;
    const bool row_ok = wrow < w_rows;
    const int klim = (int)K - kb_begin * LBK;                        // K elements of this row from the slice start (K % 32 == 0)
    const int ncol = nkb * (LBK / 2);
    for (int c0 = khalf * 16; c0 < ncol; c0 += 32) {
      uint32_t v[16];
#pragma unroll
      for (int q = 0; q < 4; q++) {
        uint4 x = make_uint4(0u, 0u, 0u, 0u);
        const int k0 = 2 * (c0 + 4 * q);
        if (row_ok && k0 < klim) x = __ldg(reinterpret_cast<const uint4*>(src + k0));
        v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
      }
      LRCN_TMEM_ST_16(tmem_base + ((uint32_t)(quad * 32) << 16) + B4_WCOL + (uint32_t)c0, v);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // every CTA's barriers are initialised before any peer arrives on them
  tc_fence_after();
  pdl_wait();
  pdl_trigger();

  if (warp < T4_MAXCH) {
    // ===================== TMA producers: warp c serves chain c -- and issues the second half of the chain's MMAs (see the forward kernel) =====================
    const int c = __shfl_sync(0xffffffffu, warp, 0);
    if (c < nch && nkb > 0) {
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc = idesc_bf16(128, 2 * T4_ROWS, false, false);
      const uint32_t acc = tb + (uint32_t)(2 * T4_ROWS * c);
      const uint32_t buf = sm.chunk + (uint32_t)c * T4_CHUNK;
      const uint32_t fullc = sm.full0 + 8 * (c * MAX_RES_KB);
      const int kb_split = (nkb + 1) / 2;
      int n = 0;
      for (int t = T - 2; t >= 0; t--, n++) {
        if (lane == 0) {
          grid_wait(ctr + c, (unsigned int)(T - 1 - t) * ctas_per_mtile);  // dG_{t+1} rows of this chain are complete
          T4_TRACE(c, 0);
          fence_proxy_async_global();
          const int arow = (t + 1) * B + m0 + T4_ROWS * c;
          for (int i = 0; i < nkb; i++) {
            const uint32_t full = fullc + 8 * i, st = buf + i * T4_BSTAGE;
            mbar_expect_tx(full, T4_BSTAGE);
            tma_load_2d(st, &tmA_hi, full, (kb_begin + i) * LBK, arow);
            tma_load_2d(st + T4_BHALF, &tmA_lo, full, (kb_begin + i) * LBK, arow);
          }
          T4_TRACE(c, 1);
        }
        __syncwarp();
        mbar_wait(sm.started0 + 8 * c, n & 1);  // the issuer warp has issued this step's first (overwriting) MMA
        tc_fence_after();
        for (int i = kb_split; i < nkb; i++) {
          mbar_wait(fullc + 8 * i, n & 1);
          tc_fence_after();
          const uint32_t b_lo = desc_lo_kmajor(buf + i * T4_BSTAGE);
          const uint32_t a_col = tb + B4_WCOL + (uint32_t)(i * (LBK / 2));
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < LBK / 16; k++) umma_bf16_ts(acc, a_col + 8u * k, b_lo + 2u * k, idesc, 1u);
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(sm.tfull0 + 8 * c);  // tfull counts two commits
        __syncwarp();
      }
    }
  } else if (warp < 2 * T4_MAXCH) {
    // ===================== MMA issuers: warp 2 + c serves chain c (converged warp, elected lane: see elect_one()) =====================
    const int c = __shfl_sync(0xffffffffu, warp - T4_MAXCH, 0);
    if (c < nch && nkb > 0) {
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc = idesc_bf16(128, 2 * T4_ROWS, false, false);
      const uint32_t acc = tb + (uint32_t)(2 * T4_ROWS * c);
      const uint32_t buf = sm.chunk + (uint32_t)c * T4_CHUNK;
      const uint32_t fullc = sm.full0 + 8 * (c * MAX_RES_KB);
      int n = 0;  // index of the recurrent step
      for (int t = T - 2; t >= 0; t--, n++) {
        if (n >= 1) mbar_wait(sm.tempty0 + 8 * c, (n - 1) & 1);  // the epilogue of the previous step has drained this accumulator
        tc_fence_after();
        const int kb_split = (nkb + 1) / 2;  // this warp: k-blocks [0, kb_split); the producer warp: the rest
        for (int i = 0; i < kb_split; i++) {
          mbar_wait(fullc + 8 * i, n & 1);
          if (lane == 0) { if (i == 0) T4_TRACE(c, 2); else if (i == kb_split - 1) T4_TRACE(c, 3); }
          tc_fence_after();
          const uint32_t b_lo = desc_lo_kmajor(buf + i * T4_BSTAGE);
          const uint32_t a_col = tb + B4_WCOL + (uint32_t)(i * (LBK / 2));
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < LBK / 16; k++) umma_bf16_ts(acc, a_col + 8u * k, b_lo + 2u * k, idesc, (i | k) ? 1u : 0u);
            if (i == 0) mbar_arrive(sm.started0 + 8 * c);
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(sm.tfull0 + 8 * c);
        __syncwarp();
        if (lane == 0) T4_TRACE(c, 4);
      }
    }
  } else {
    // ===================== epilogue teams: team c finishes chain c =====================
    const int ew = warp - 2 * T4_MAXCH, quad = warp & 3, c = ew >> 2;
    const int tid = (ew & 3) * 32 + lane;  // 0..127 inside the team
    float* S = sm.S + (size_t)c * 128 * T4_SLD;
    float* red = sm.red + (size_t)c * (B4_RED / 4);
    if (c < nch) {
      // finisher mapping: row fr of the chain, units 4*ug .. 4*ug+3 of this rank's 16
      const int fr = tid >> 2, ug = tid & 3;
      const int m = m0 + T4_ROWS * c + fr;
      const int j = nt * NT + 16 * (int)rank + 4 * ug;
      const bool active = m < B && j < H;
      float dcreg[4] = {0.f, 0.f, 0.f, 0.f};
      float bsum[4][4];  // [gate][unit]: this thread's share of the bias gradient (sum of dG over its row and all steps)
#pragma unroll
      for (int g = 0; g < 4; g++)
#pragma unroll
        for (int e = 0; e < 4; e++) bsum[g][e] = 0.f;
      float4 pf, pi, po, pg, pcp, pcc, pdh;
      pf = pi = po = pg = pcp = pcc = pdh = make_float4(0.f, 0.f, 0.f, 0.f);
      auto prefetch = [&](int tt) {
        const float* g0 = p.acts + ((size_t)tt * B + m) * 4 * H + j;
        pf = *reinterpret_cast<const float4*>(g0); pi = *reinterpret_cast<const float4*>(g0 + H);
        po = *reinterpret_cast<const float4*>(g0 + 2 * H); pg = *reinterpret_cast<const float4*>(g0 + 3 * H);
        pcp = *reinterpret_cast<const float4*>(p.cs + ((size_t)tt * B + m) * H + j);
        pcc = *reinterpret_cast<const float4*>(p.cs + ((size_t)(tt + 1) * B + m) * H + j);
        pdh = *reinterpret_cast<const float4*>(p.dh_all + ((size_t)tt * B + m) * H + j);
      };
      if (active) prefetch(T - 1);
      int n = 0;
      for (int t = T - 1; t >= 0; t--) {
        const bool has_rec = t < T - 1;
        float rec[4] = {0.f, 0.f, 0.f, 0.f};
        if (has_rec) {
          // phase 1: accumulator -> S (the three split products summed: lanes 0-63 hold hi*hi + hi*lo, lanes 64-127 lo*hi)
          float* dst = S + (size_t)(32 * quad + lane) * T4_SLD;
          if (nkb > 0) {
            mbar_wait(sm.tfull0 + 8 * c, n & 1);
            if (tid == 0) T4_TRACE(c, 5);
            tc_fence_after();
            const uint32_t tl = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(2 * T4_ROWS * c);
            uint32_t v[32];
            LRCN_TMEM_LD_32(tl, v);
            if (quad < 2) {
              uint32_t w[32];
              LRCN_TMEM_LD_32(tl + T4_ROWS, w);
              tmem_ld_wait();
#pragma unroll
              for (int r = 0; r < T4_ROWS; r++) dst[r] = __uint_as_float(v[r]) + __uint_as_float(w[r]);
            } else {
              tmem_ld_wait();
#pragma unroll
              for (int r = 0; r < T4_ROWS; r++) dst[r] = __uint_as_float(v[r]);
            }
            tc_fence_before();
          } else {
#pragma unroll
            for (int r = 0; r < T4_ROWS; r++) dst[r] = 0.f;
          }
          fence_async_smem();  // the team's generic-proxy writes of S become visible to the bulk-copy (async proxy) reads
          team_bar_sync(c);
          // phase 2: one thread sends every rank the partials (over this K-quarter) of the 16 units it finishes
          if (tid == 0) {
            if (nkb > 0) mbar_arrive(sm.tempty0 + 8 * c);  // every thread of the team is past its TMEM reads
            mbar_expect_tx(sm.redfull0 + 8 * c, (CL - 1) * 2 * B4_PART);   // what the three other ranks will deliver to me (my own part stays in S)
            const uint32_t s_hi = smem_u32(S), s_lo = smem_u32(S) + 64 * T4_SLD * 4;
            const uint32_t r_mine = smem_u32(red) + (uint32_t)((int)rank * 2 * B4_PART);
#pragma unroll
            for (int d = 0; d < CL; d++) {
              if (d == (int)rank) continue;
              const uint32_t dst = dsmem_addr(r_mine, (uint32_t)d), bar = dsmem_addr(sm.redfull0 + 8 * c, (uint32_t)d);
              dsmem_bulk_copy(dst, s_hi + (uint32_t)(d * B4_PART), B4_PART, bar);
              dsmem_bulk_copy(dst + B4_PART, s_lo + (uint32_t)(d * B4_PART), B4_PART, bar);
            }
            T4_TRACE(c, 6);   // partials sent
          }
          // phase 3: the 4 x 2 partials of my units
          mbar_wait(sm.redfull0 + 8 * c, n & 1);
          if (tid == 0) T4_TRACE(c, 7);   // received
#pragma unroll
          for (int src = 0; src < CL; src++) {  // fixed order: deterministic sums
            // the other ranks' partials arrived in `red`; this rank's own (W_hi part, W_lo part) are still in S
            const float* p_hi = src == (int)rank ? S + (size_t)(16 * src) * T4_SLD : red + (size_t)(2 * src) * 16 * T4_SLD;
            const float* p_lo = src == (int)rank ? S + (size_t)(64 + 16 * src) * T4_SLD : red + (size_t)(2 * src + 1) * 16 * T4_SLD;
#pragma unroll
            for (int e = 0; e < 4; e++) rec[e] += p_hi[(size_t)(4 * ug + e) * T4_SLD + fr] + p_lo[(size_t)(4 * ug + e) * T4_SLD + fr];
          }
          n++;
        }
        float r0[4], r1[4], r2[4], r3[4];
        const size_t gidx = ((size_t)t * B + m) * 4 * H + j;
        if (active) {
          const float f[4] = {pf.x, pf.y, pf.z, pf.w}, in[4] = {pi.x, pi.y, pi.z, pi.w}, o[4] = {po.x, po.y, po.z, po.w}, ch[4] = {pg.x, pg.y, pg.z, pg.w};
          const float cpv[4] = {pcp.x, pcp.y, pcp.z, pcp.w}, ccv[4] = {pcc.x, pcc.y, pcc.z, pcc.w}, dhv[4] = {pdh.x, pdh.y, pdh.z, pdh.w};
#pragma unroll
          for (int e = 0; e < 4; e++) {
            const float dh = dhv[e] + rec[e];
            const float tc = tanh_fast(ccv[e]);
            const float dcv = dcreg[e] + dh * o[e] * (1.f - tc * tc);
            const float dO = dh * tc, dF = dcv * cpv[e], dI = dcv * ch[e], dG = dcv * in[e];
            dcreg[e] = dcv * f[e];
            r0[e] = dF * f[e] * (1.f - f[e]);
            r1[e] = dI * in[e] * (1.f - in[e]);
            r2[e] = dO * o[e] * (1.f - o[e]);
            r3[e] = dG * (1.f - ch[e] * ch[e]);
          }
          const float* rr[4] = {r0, r1, r2, r3};
#pragma unroll
          for (int g = 0; g < 4; g++)
#pragma unroll
            for (int e = 0; e < 4; e++) bsum[g][e] += rr[g][e];
#pragma unroll
          for (int g = 0; g < 4; g++) {  // the bf16 split of dG_t is what the next step's TMA reads: store it first
            __nv_bfloat16 hh[4], ll[4];
#pragma unroll
            for (int e = 0; e < 4; e++) split_bf16(rr[g][e], hh[e], ll[e]);
            *reinterpret_cast<uint2*>(p.o_hi + gidx + (size_t)g * H) = *reinterpret_cast<uint2*>(hh);
            *reinterpret_cast<uint2*>(p.o_lo + gidx + (size_t)g * H) = *reinterpret_cast<uint2*>(ll);
          }
        }
        if (t > 0) {  // publish dG_t of this chain
          team_bar_sync(c);  // orders the team's stores before the release below; also: every reader is done with `red`
          if (tid == 0) {
            // anti-phase the two chains once (see lstm_fwd_seq4_kernel)
            if (t == T - 1 && c == 1 && nch > 1 && !(p.sync_flags & 16)) {
              const unsigned long long t0 = gtime();
              while (gtime() - t0 < (unsigned long long)(p.sync_flags >> 8 ? (p.sync_flags >> 8) : 2800)) {}
            }
            fence_proxy_async_global(); grid_arrive(ctr + c);
          }
        }
        if (active) {  // off the critical path
          float* grow = p.acts + gidx;
          *reinterpret_cast<float4*>(grow) = make_float4(r0[0], r0[1], r0[2], r0[3]);
          *reinterpret_cast<float4*>(grow + H) = make_float4(r1[0], r1[1], r1[2], r1[3]);
          *reinterpret_cast<float4*>(grow + 2 * H) = make_float4(r2[0], r2[1], r2[2], r2[3]);
          *reinterpret_cast<float4*>(grow + 3 * H) = make_float4(r3[0], r3[1], r3[2], r3[3]);
          if (t > 0) prefetch(t - 1);
        }
      }
      if (p.dbias) {
        // bias gradient: sum over the rows of a warp by shuffles (lanes with equal ug), over the team's four warps through S
        // (free now), then one atomic per (gate, unit) and team onto the zero-initialised gradient
#pragma unroll
        for (int g = 0; g < 4; g++)
#pragma unroll
          for (int e = 0; e < 4; e++) {
            float v = active ? bsum[g][e] : 0.f;
            v += __shfl_xor_sync(0xffffffffu, v, 4); v += __shfl_xor_sync(0xffffffffu, v, 8); v += __shfl_xor_sync(0xffffffffu, v, 16);
            bsum[g][e] = v;
          }
        team_bar_sync(c);
        if (lane < 4) {
#pragma unroll
          for (int g = 0; g < 4; g++)
#pragma unroll
            for (int e = 0; e < 4; e++) S[((ew & 3) * 4 + lane) * 16 + g * 4 + e] = bsum[g][e];  // [warp][ug][gate][unit]
        }
        team_bar_sync(c);
        if (tid < 64) {
          const int ugq = tid >> 4, ge = tid & 15, g = ge >> 2, e = ge & 3;
          float v = 0.f;
#pragma unroll
          for (int w4 = 0; w4 < 4; w4++) v += S[(w4 * 4 + ugq) * 16 + ge];
          const int jj = nt * NT + 16 * (int)rank + 4 * ugq + e;
          if (jj < H) atomicAdd(p.dbias + (size_t)g * H + jj, v);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // no CTA leaves while a peer may still store into its shared memory / arrive on its barriers
  if (warp == T4_MAXCH) {
    tc_fence_after();
    tmem_dealloc<B4_TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------- weight copies
constexpr int F_NT = NT, F_NH = NT / 4;  // forward: 16 hidden units x 4 gates per CTA
constexpr int R_NT = NT;                // backward: 64 hidden units per cluster, 16 finished by each CTA

// forward operand: rows = gate columns n = g*H + j of the layer weight W [4H][ldw] (columns [x_off, x_off+H) = W_h),
// permuted UNIT-major so that CTA nt's 64 rows are its 16 units x [f i o g]:  row jt*64 + u*4 + g  <-  n = g*H + jt*16 + u
struct PrepLayer { const float* W; int ldw, x_off, H; __nv_bfloat16 *p_hi, *p_lo, *t_hi, *t_lo; };
struct PrepArgs { PrepLayer l[2]; };

__global__ void permute_split_kernel(const PrepArgs a) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  const PrepLayer& L = a.l[blockIdx.y];
  const float* __restrict__ W = L.W;
  const int ldw = L.ldw, x_off = L.x_off, H = L.H, Hp = (L.H + 7) / 8 * 8;
  __nv_bfloat16* __restrict__ hi = L.p_hi;
  __nv_bfloat16* __restrict__ lo = L.p_lo;
  if ((int)blockIdx.x >= (H + F_NH - 1) / F_NH * F_NT) return;
  const int row = blockIdx.x;
  const int jt = row / F_NT, r = row % F_NT, u = r / 4, g = r % 4;
  const int j = jt * F_NH + u;
  for (int k = threadIdx.x; k < Hp; k += blockDim.x) {
    float x = 0.f;
    if (j < H && k < H) x = W[(size_t)(g * H + j) * ldw + x_off + k];
    __nv_bfloat16 h, l;
    split_bf16(x, h, l);
    hi[(size_t)row * Hp + k] = h;
    lo[(size_t)row * Hp + k] = l;
  }
}
// backward operand: WhT[j][n] = W[n][x_off + j]  ([Hr rows][4H], K-major over the gate columns n)
__global__ void transpose_split_kernel(const PrepArgs a) {
  pdl_wait();  // PDL: launched while the previous kernel drains (kernels.cuh)
  pdl_trigger();
  const PrepLayer& L = a.l[blockIdx.z];
  const float* __restrict__ W = L.W;
  const int ldw = L.ldw, x_off = L.x_off, H = L.H;
  __nv_bfloat16* __restrict__ hi = L.t_hi;
  __nv_bfloat16* __restrict__ lo = L.t_lo;
  if (!hi || (int)blockIdx.x * 32 >= 4 * H || (int)blockIdx.y * 32 >= (H + 63) / 64 * 64) return;  // uniform per block
  __shared__ float tile[32][33];
  const int n0 = blockIdx.x * 32, j0 = blockIdx.y * 32;  // n over 4H, j over Hr
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int n = n0 + r, j = j0 + threadIdx.x;
    tile[r][threadIdx.x] = (n < 4 * H && j < H) ? W[(size_t)n * ldw + x_off + j] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int j = j0 + r, n = n0 + threadIdx.x;
    if (n < 4 * H) {
      __nv_bfloat16 h, l;
      split_bf16(tile[threadIdx.x][r], h, l);
      hi[(size_t)j * 4 * H + n] = h;
      lo[(size_t)j * 4 * H + n] = l;
    }
  }
}
static int fwd_rows(int H) { return (H + F_NH - 1) / F_NH * F_NT; }
static int bwd_rows(int H) { return (H + 63) / 64 * 64; }
size_t lstm_permuted_elems(int H) { return (size_t)fwd_rows(H) * ((H + 7) / 8 * 8); }
size_t lstm_transposed_elems(int H) { return (size_t)bwd_rows(H) * 4 * H; }

// both layers in one launch each (perm_* for the forward step, tr_* (may be null) for the backward step)
void lstm_prepare_weights2(cudaStream_t s, const float* W1, int ldw1, int x_off1, int H1, __nv_bfloat16* p1_hi, __nv_bfloat16* p1_lo,
                           __nv_bfloat16* t1_hi, __nv_bfloat16* t1_lo, const float* W2, int ldw2, int x_off2, int H2, __nv_bfloat16* p2_hi,
                           __nv_bfloat16* p2_lo, __nv_bfloat16* t2_hi, __nv_bfloat16* t2_lo) {
  PrepArgs a;
  a.l[0] = PrepLayer{W1, ldw1, x_off1, H1, p1_hi, p1_lo, t1_hi, t1_lo};
  a.l[1] = PrepLayer{W2, ldw2, x_off2, H2, p2_hi, p2_lo, t2_hi, t2_lo};
  const int Hm = H1 > H2 ? H1 : H2;
  launch_pdl<2>(permute_split_kernel, dim3(fwd_rows(Hm), 2), dim3(128), 0, s, a);
  if (g_counter) g_counter->n++;
  if (t1_hi || t2_hi) {
    launch_pdl<2>(transpose_split_kernel, dim3((4 * Hm + 31) / 32, bwd_rows(Hm) / 32, 2), dim3(32, 8), 0, s, a);
    if (g_counter) g_counter->n++;
  }
}

static bool check_launch(const char* what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) { set_sm100_error((std::string(what) + ": " + cudaGetErrorString(e)).c_str()); return false; }
  return true;
}

bool lstm_fwd_step(cudaStream_t s, int B, int H, bool has_rec, const __nv_bfloat16* hprev_hi, const __nv_bfloat16* hprev_lo,
                   const __nv_bfloat16* wperm_hi, const __nv_bfloat16* wperm_lo, float* gates, const float* c_prev, float* c_out, float* h_out,
                   __nv_bfloat16* h_hi, __nv_bfloat16* h_lo) {
  const int Hp = (H + 7) / 8 * 8, rows = fwd_rows(H);
  CUtensorMap ta_hi, ta_lo, tb_hi, tb_lo;
  if (!get_tensor_map_bf16(&tb_hi, wperm_hi, H, rows, Hp, F_NT) || !get_tensor_map_bf16(&tb_lo, wperm_lo, H, rows, Hp, F_NT)) return false;
  if (has_rec) {
    if (!get_tensor_map_bf16(&ta_hi, hprev_hi, H, B, H, LM / CL) || !get_tensor_map_bf16(&ta_lo, hprev_lo, H, B, H, LM / CL)) return false;
  } else {  // never dereferenced (no mainloop), but kernel parameters must be valid maps
    ta_hi = tb_hi; ta_lo = tb_lo;
  }
  StepParams p{};
  p.B = B; p.H = H; p.num_kb = (H + LBK - 1) / LBK; p.has_rec = has_rec ? 1 : 0;
  p.gates = gates; p.c_prev = c_prev; p.c_out = c_out; p.h_out = h_out; p.o_hi = h_hi; p.o_lo = h_lo;
  const int nt = (H + F_NH - 1) / F_NH;
  dim3 grid((nt + CL - 1) / CL * CL, (B + LM - 1) / LM);
  lstm_fwd_step_kernel<<<grid, L_THREADS, L_SMEM, s>>>(ta_hi, ta_lo, tb_hi, tb_lo, p);
  if (g_counter) g_counter->n++;
  return check_launch("lstm_fwd_step launch");
}

// wt_hi/wt_lo: transposed recurrent weights from lstm_prepare_weights; gnext: bf16 split of dG_{t+1} [B][4H]
bool lstm_bwd_step(cudaStream_t s, int B, int H, bool has_rec, const __nv_bfloat16* wt_hi, const __nv_bfloat16* wt_lo,
                   const __nv_bfloat16* gnext_hi, const __nv_bfloat16* gnext_lo, float* gates, __nv_bfloat16* g_hi, __nv_bfloat16* g_lo,
                   const float* c_prev, const float* c_cur, const float* dh_in, float* dc) {
  CUtensorMap ta_hi, ta_lo, tb_hi, tb_lo;
  const uint64_t K = 4 * (uint64_t)H;
  if (!get_tensor_map_bf16(&tb_hi, wt_hi, K, bwd_rows(H), K, R_NT) || !get_tensor_map_bf16(&tb_lo, wt_lo, K, bwd_rows(H), K, R_NT)) return false;
  if (has_rec) {
    if (!get_tensor_map_bf16(&ta_hi, gnext_hi, K, B, K, LM) || !get_tensor_map_bf16(&ta_lo, gnext_lo, K, B, K, LM)) return false;
  } else {
    ta_hi = tb_hi; ta_lo = tb_lo;
  }
  StepParams p{};
  p.B = B; p.H = H; p.num_kb = (int)((K + LBK - 1) / LBK); p.has_rec = has_rec ? 1 : 0;
  p.gates = gates; p.o_hi = g_hi; p.o_lo = g_lo; p.c_prev = c_prev; p.c_cur = c_cur; p.dh_in = dh_in; p.dc = dc;
  const int nt = (H + R_NT - 1) / R_NT;
  dim3 grid(nt * CL, (B + LM - 1) / LM);  // CL k-slices per 64x64 output tile
  lstm_bwd_step_kernel<<<grid, L_THREADS, L_SMEM, s>>>(ta_hi, ta_lo, tb_hi, tb_lo, p);
  if (g_counter) g_counter->n++;
  return check_launch("lstm_bwd_step launch");
}

static int g_lstm_sms = 0;
// Can the persistent kernel be used?  (its weight k-blocks must fit on chip; the whole grid must be co-resident)
static bool seq_fits(const void* kernel, int res_kb, dim3 grid, int smem_bytes) {
  if (res_kb > MAX_RES_KB) return false;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = dim3(T4_THREADS); cfg.dynamicSmemBytes = smem_bytes;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int nclusters = 0;
  if (cudaOccupancyMaxActiveClusters(&nclusters, kernel, &cfg) != cudaSuccess) { cudaGetLastError(); return false; }
  return (long long)nclusters * CL >= (long long)grid.x * grid.y;
}

// whole-sequence forward of one layer; returns true with *launched = false when the persistent kernel does not apply
bool lstm_fwd_seq(cudaStream_t s, int B, int H, int T, const __nv_bfloat16* wperm_hi, const __nv_bfloat16* wperm_lo, float* acts, float* hs,
                  float* cs, __nv_bfloat16* hs_hi, __nv_bfloat16* hs_lo, unsigned int* counters, bool* launched, unsigned long long* trace) {
  *launched = false;
  if (T < 2) return true;
  const int num_kb = (H + LBK - 1) / LBK;
  const int nt = (H + F_NH - 1) / F_NH;
  // the fewest chains per CTA (= the most CTAs) whose grid is still co-resident
  for (int nch = 1; nch <= T4_MAXCH; nch *= 2) {
    const int rows = T4_ROWS * nch;
    dim3 grid4((nt + CL - 1) / CL * CL, (B + rows - 1) / rows);
    if (grid4.y * T4_MAXCH > 64) continue;  // one counter per (m-tile, chain)
    if (!seq_fits((const void*)lstm_fwd_seq4_kernel, num_kb, grid4, seq4_smem_bytes())) continue;
    const int Hp = (H + 7) / 8 * 8, wrows = fwd_rows(H);
    CUtensorMap ta_hi, ta_lo, tb_hi, tb_lo;
    if (!get_tensor_map_bf16(&tb_hi, wperm_hi, H, wrows, Hp, F_NT) || !get_tensor_map_bf16(&tb_lo, wperm_lo, H, wrows, Hp, F_NT)) return false;
    const uint64_t R = (uint64_t)(T + 1) * B;
    if (!get_tensor_map_bf16(&ta_hi, hs_hi, H, R, H, T4_ROWS) || !get_tensor_map_bf16(&ta_lo, hs_lo, H, R, H, T4_ROWS)) return false;
    SeqParams p{};
    p.B = B; p.H = H; p.T = T; p.num_kb = num_kb; p.acts = acts; p.hs = hs; p.cs = cs; p.o_hi = hs_hi; p.o_lo = hs_lo; p.counters = counters;
    p.trace = trace;
    static const int dbg_flags = getenv("LRCN_SEQ_SYNC") ? atoi(getenv("LRCN_SEQ_SYNC")) : 0;
    p.sync_flags = dbg_flags;
    launch_pdl(lstm_fwd_seq4_kernel, grid4, dim3(T4_THREADS), seq4_smem_bytes(), s, ta_hi, ta_lo, tb_hi, tb_lo, wperm_hi, wperm_lo, wrows, Hp, p, nch);
    if (g_counter) g_counter->n++;
    *launched = true;
    return check_launch("lstm_fwd_seq4 launch");
  }
  return true;
}

// whole-sequence backward of one layer; same contract as lstm_fwd_seq
bool lstm_bwd_seq(cudaStream_t s, int B, int H, int T, const __nv_bfloat16* wt_hi, const __nv_bfloat16* wt_lo, float* acts,
                  __nv_bfloat16* acts_hi, __nv_bfloat16* acts_lo, float* cs, const float* dh_all, float* dc, unsigned int* counters,
                  bool* launched, float* dbias, unsigned long long* trace) {
  *launched = false;
  const uint64_t K = 4 * (uint64_t)H;
  const int num_kb = (int)((K + LBK - 1) / LBK);
  const int kb_per = (num_kb + CL - 1) / CL;
  const int nt = (H + R_NT - 1) / R_NT;
  if (T < 2 || kb_per > MAX_RES_KB) return true;
  for (int nch = 1; nch <= T4_MAXCH; nch *= 2) {
    const int rows = T4_ROWS * nch;
    dim3 grid4(nt * CL, (B + rows - 1) / rows);
    if (grid4.y * T4_MAXCH > 64) continue;  // one counter per (m-tile, chain)
    if (!seq_fits((const void*)lstm_bwd_seq4_kernel, kb_per, grid4, bwd4_smem_bytes())) continue;
    CUtensorMap ta_hi, ta_lo;
    const uint64_t R = (uint64_t)T * B;
    if (!get_tensor_map_bf16(&ta_hi, acts_hi, K, R, K, T4_ROWS) || !get_tensor_map_bf16(&ta_lo, acts_lo, K, R, K, T4_ROWS)) return false;
    SeqParams p{};
    p.B = B; p.H = H; p.T = T; p.num_kb = num_kb; p.acts = acts; p.cs = cs; p.o_hi = acts_hi; p.o_lo = acts_lo; p.dh_all = dh_all; p.dc = dc;
    p.counters = counters; p.dbias = dbias; p.trace = trace;
    static const int dbg_flags = getenv("LRCN_SEQ_SYNC") ? atoi(getenv("LRCN_SEQ_SYNC")) : 0;
    p.sync_flags = dbg_flags;
    launch_pdl(lstm_bwd_seq4_kernel, grid4, dim3(T4_THREADS), bwd4_smem_bytes(), s, ta_hi, ta_lo, wt_hi, wt_lo, bwd_rows(H), p, nch);
    if (g_counter) g_counter->n++;
    *launched = true;
    return check_launch("lstm_bwd_seq4 launch");
  }
  return true;
}

bool lstm_bind_abort(unsigned int* host_flag) { return dev_abort_bind(host_flag) == cudaSuccess; }

bool init_lstm_sm100() {
  cudaError_t e = cudaFuncSetAttribute(lstm_fwd_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(lstm_bwd_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(lstm_fwd_seq4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, seq4_smem_bytes());
  if (e == cudaSuccess) e = cudaFuncSetAttribute(lstm_bwd_seq4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd4_smem_bytes());
  if (e != cudaSuccess) { set_sm100_error((std::string("cudaFuncSetAttribute(lstm): ") + cudaGetErrorString(e)).c_str()); return false; }
  return true;
}

}  // namespace lrcn
