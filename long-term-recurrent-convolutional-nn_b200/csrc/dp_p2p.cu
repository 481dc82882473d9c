// dp_p2p.cu -- data-parallel gradient exchange over NVLink peer memory, without NCCL kernels.
//
// One handle per GPU; every rank maps its peers' gradient and weight arenas, control blocks and staging allocations (CUDA IPC,
// or direct peer pointers in a single-process group).  Rank r OWNS a contiguous 1/N slice of what is exchanged and sums it over
// all ranks in fixed rank order, so the sum is deterministic and identical everywhere.
//   training step      one fused_exchange_kernel launch per gradient bucket: every rank pushes its gradient chunks into the
//                      owners' staging rows, the owner sums them, runs Adam on its slice and pushes the new weights into every
//                      rank's arena; per-chunk flags and completion counters order it (see the section above the kernel).
//   gradient-only step flag barrier  ->  allreduce_p2p_kernel: the owner loads its shard of the arena from every rank and stores
//                      the sum into every rank's arena in place  ->  flag barrier (every rank's stores have landed).
// Why not NCCL here: its kernels compete for SMs with the persistent tcgen05 GEMM / LSTM kernels (which need their whole
// grid co-resident), so a "bucketed, overlapped" allreduce ends up serialising; measured in profiles/r01_progress.md.
#include "kernels.cuh"

#include <stdlib.h>

#include <stdio.h>

namespace lrcn {

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_sys_add(unsigned int* p, unsigned int x) {
  asm volatile("red.release.sys.global.add.u32 [%0], %1;" ::"l"(p), "r"(x) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ float4 ld_peer_f4(const float4* p) {  // peer memory is cached in L1 only and L1 is not coherent: bypass it
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}

// one warp: lane q signals rank q and waits for rank q's signal
__global__ void xgpu_barrier_kernel(P2PPeers peers, unsigned int* epoch_ctr) {
  __shared__ unsigned int epoch;
  if (threadIdx.x == 0) { epoch = *epoch_ctr + 1u; *epoch_ctr = epoch; }
  __syncwarp();
  const unsigned int e = epoch;
  const int q = threadIdx.x;
  __threadfence_system();
  if (q < peers.nranks) {
    st_release_sys(&peers.ctl[q]->flags[peers.rank], e);
    const unsigned int* mine = &peers.ctl[peers.rank]->flags[q];
    const long long t0 = clock64();
    while ((int)(ld_acquire_sys(mine) - e) < 0) {
      if (dev_aborted()) break;
      if (clock64() - t0 > 40000000000ll) {  // ~20 s: a peer died or never reached the barrier
        printf("lrcn dp_p2p: barrier timeout, rank %d waiting for rank %d (epoch %u)\n", peers.rank, q, e);
        dev_abort_set();  // flag + drain instead of a trap (kernels.cuh): the ABI reports a sticky error
        break;
      }
    }
  }
}

// in-place allreduce(sum) of the gradient arena by owner-computes shards + fp64 loss total
__global__ void __launch_bounds__(256) allreduce_p2p_kernel(P2PPeers peers, size_t begin4, size_t end4, double* loss_total) {
  const int N = peers.nranks;
  for (size_t i = begin4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < end4; i += (size_t)gridDim.x * blockDim.x) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
    for (int p = 0; p < N; p++) {
      const float4 x = ld_peer_f4(reinterpret_cast<const float4*>(peers.g[p]) + i);
      acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
    }
    for (int p = 0; p < N; p++) reinterpret_cast<float4*>(peers.g[p])[i] = acc;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && loss_total) {
    double t = 0.0;
    for (int p = 0; p < N; p++) {
      double v;
      asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(&peers.ctl[p]->loss_partial) : "memory");
      t += v;
    }
    *loss_total = t;
  }
  __threadfence_system();  // my stores into peer memory are performed before this kernel ends (the second barrier follows)
}

bool dp_bind_abort(unsigned int* host_flag) { return dev_abort_bind(host_flag) == cudaSuccess; }

// [begin, end) of rank r's shard of an arena of n_floats, in floats
static void dp_p2p_shard(size_t n_floats, int nranks, int r, size_t* begin, size_t* end) {
  const size_t n4 = n_floats / 4, per = (n4 + nranks - 1) / nranks;
  const size_t b = per * r < n4 ? per * r : n4;
  const size_t e = b + per < n4 ? b + per : n4;
  *begin = 4 * b; *end = 4 * e;
}

void dp_p2p_allreduce(cudaStream_t s, const P2PPeers& peers, size_t n_floats, unsigned int* epoch_ctr, double* loss_total) {
  size_t b, e;  // arena sizes are multiples of 64 floats
  dp_p2p_shard(n_floats, peers.nranks, peers.rank, &b, &e);
  xgpu_barrier_kernel<<<1, 32, 0, s>>>(peers, epoch_ctr);
  allreduce_p2p_kernel<<<148 * 4, 256, 0, s>>>(peers, b / 4, e / 4, loss_total);
  xgpu_barrier_kernel<<<1, 32, 0, s>>>(peers, epoch_ctr);
  if (g_counter) g_counter->n += 3;
}

// ---------------------------------------------------------------------------------------------------------------------
// FUSED bucket exchange: reduce-scatter, sharded Adam and all-gather of one gradient bucket in ONE kernel over NVLink peer
// memory, pipelined per 32 KiB chunk (tools/dp_timeline.py showed the multi-kernel exchange spending most of its time in launch
// gaps, whole-kernel system fences and two cross-GPU barrier kernels per bucket).  CTA j of G:
//   A  for every peer r and every chunk c = j, j+G, .. of r's slice: store my gradient chunk into r's staging row `rank`, fence,
//      then st.release.sys  flag_r[bucket][rank][c] = epoch                                  (posted stores, nothing waits here)
//   B  for every chunk c = j, j+G, .. of MY slice: wait until flag[bucket][q][c] == epoch for all q, sum the contributions in
//      rank order, Adam (same operation order as adam_kernel: replicas stay bit-identical), store the new weights into every
//      peer's arena, fence, then red.release.sys  done_p[bucket][rank] += 1 on every peer p
//   C  CTA 0 waits until done[bucket][q] == epoch * chunks(q) for all q: every owner's new weights have landed here.
// A never waits, so B's waits are always satisfied by the peers' A phases (no co-residency requirement, no deadlock).  A peer's
// weights are overwritten only after ITS gradient chunk arrived, i.e. after its backward pass is done with them; a staging row is
// rewritten only in the next step, after the owner's done-counter said it had consumed the row.
constexpr int XSUB = 1024;       // float4 per sub-block (16 KiB): 4 per thread; a chunk = a.sub sub-blocks (1 unless a slice exceeds 8 MiB)
constexpr int XMAXCH = DP_XMAXCH;  // chunks per slice the flag area has room for
__device__ __forceinline__ unsigned int* xflag(float* stage, size_t ctl4, int bucket, int src, int chunk) {
  return reinterpret_cast<unsigned int*>(reinterpret_cast<float4*>(stage) + ctl4) + 64 + ((size_t)(bucket * LRCN_P2P_MAX_RANKS + src) * XMAXCH + chunk);
}
__device__ __forceinline__ unsigned int* xdone(float* stage, size_t ctl4, int bucket, int owner) {
  return reinterpret_cast<unsigned int*>(reinterpret_cast<float4*>(stage) + ctl4) + bucket * LRCN_P2P_MAX_RANKS + owner;
}
__device__ __forceinline__ bool xwait(const unsigned int* p, unsigned int want, const char* what, int q) {
  const long long t0 = clock64();
  unsigned int spins = 0;
  while ((int)(ld_acquire_sys(p) - want) < 0) {
    if ((++spins & 255u) == 0u) {
      if (dev_aborted()) return false;
      if (clock64() - t0 > 40000000000ll) {
        printf("lrcn dp_p2p: fused exchange timeout waiting for %s of rank %d (want %u)\n", what, q, want);
        dev_abort_set();
        return false;
      }
    }
  }
  return true;
}
__global__ void __launch_bounds__(256) fused_exchange_kernel(const P2PPeers peers, const FusedXArgs a, float4* __restrict__ m, float4* __restrict__ v,
                                                             const StepScalars* __restrict__ sc, double* loss_total) {
  const int N = peers.nranks, me = peers.rank, G = gridDim.x, tid = threadIdx.x;
  const unsigned int epoch = sc->xchg_epoch;
  const float4* gl = reinterpret_cast<const float4*>(peers.g[me]);
  // ---- A: push my gradient chunks to their owners
  for (int d = 1; d < N; d++) {
    const int r = (me + d) % N;  // staggered targets: no two ranks start on the same peer
    const size_t n4 = a.e4[r] - a.b4[r];
    const size_t XCH = (size_t)XSUB * a.sub;
    const int nch = (int)((n4 + XCH - 1) / XCH);
    float4* row = reinterpret_cast<float4*>(a.stage[r]) + (size_t)me * a.stride4 + a.pre4;
    for (int c = blockIdx.x; c < nch; c += G) {
      for (int sb = 0; sb < a.sub; sb++) {
        const size_t o = (size_t)c * XCH + (size_t)sb * XSUB;
        float4 x[XSUB / 256];
#pragma unroll
        for (int u = 0; u < XSUB / 256; u++) { const size_t i = o + tid + 256 * u; if (i < n4) x[u] = gl[a.b4[r] + i]; }
#pragma unroll
        for (int u = 0; u < XSUB / 256; u++) { const size_t i = o + tid + 256 * u; if (i < n4) row[i] = x[u]; }
      }
    }
  }
  // ONE system-scope fence per CTA for all its pushes (a sys-scope release costs ~10 us here: per chunk it dominated), then the
  // chunk flags as relaxed stores behind it.  bar.sync makes the fence cumulative over the whole CTA's stores.
  __syncthreads();
  if (tid == 0) {
    __threadfence_system();
    for (int d = 1; d < N; d++) {
      const int r = (me + d) % N;
      const size_t n4 = a.e4[r] - a.b4[r];
      const int nch = (int)((n4 + (size_t)XSUB * a.sub - 1) / ((size_t)XSUB * a.sub));
      for (int c = blockIdx.x; c < nch; c += G) st_relaxed_sys(xflag(a.stage[r], a.ctl4, a.bucket, me, c), epoch);
    }
  }
  // ---- B: my slice
  {
    const float b1 = sc->beta1, b2 = sc->beta2, lr = sc->lr, eps = sc->eps, d1 = sc->adam_d1, d2 = sc->adam_d2;
    const float ob1 = sc->one_m_beta1, ob2 = sc->one_m_beta2;
    const size_t b4 = a.b4[me], n4 = a.e4[me] - a.b4[me];
    const size_t XCH = (size_t)XSUB * a.sub;
    const int nch = (int)((n4 + XCH - 1) / XCH);
    const float4* st = reinterpret_cast<const float4*>(a.stage[me]) + a.pre4;
    float4* wl = reinterpret_cast<float4*>(peers.w[me]);
    float4* gw = reinterpret_cast<float4*>(peers.g[me]);
    int mine = 0;
    for (int c = blockIdx.x; c < nch; c += G) {
      if (tid < N && tid != me) xwait(xflag(a.stage[me], a.ctl4, a.bucket, tid, c), epoch, "a gradient chunk", tid);
      __syncthreads();
      const size_t o = (size_t)c * XCH;
#pragma unroll 2
      for (int u = 0; u < (int)(XCH / 256); u++) {
        const size_t i = o + tid + 256 * u;
        if (i >= n4) break;
        float4 Gs = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int q = 0; q < N; q++) {  // fixed rank order: deterministic, identical on every rank
          const float4 x = q == me ? gl[b4 + i] : ld_peer_f4(st + (size_t)q * a.stride4 + i);   // staged rows were written by a peer: bypass L1
          Gs.x += x.x; Gs.y += x.y; Gs.z += x.z; Gs.w += x.w;
        }
        float4 W = wl[b4 + i], Mv = m[b4 + i], Vv = v[b4 + i];
        float* wp = reinterpret_cast<float*>(&W);
        const float* gp = reinterpret_cast<const float*>(&Gs);
        float* mp = reinterpret_cast<float*>(&Mv);
        float* vp = reinterpret_cast<float*>(&Vv);
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const float mm = __fadd_rn(__fmul_rn(b1, mp[k]), __fmul_rn(ob1, gp[k]));
          const float vv = __fadd_rn(__fmul_rn(b2, vp[k]), __fmul_rn(ob2, __fmul_rn(gp[k], gp[k])));
          const float upd = __fdiv_rn(__fdiv_rn(mm, d1), __fadd_rn(__fsqrt_rn(__fdiv_rn(vv, d2)), eps));
          wp[k] = __fsub_rn(wp[k], __fmul_rn(lr, upd));
          mp[k] = mm; vp[k] = vv;
        }
        for (int p = 0; p < N; p++) reinterpret_cast<float4*>(peers.w[p])[b4 + i] = W;   // all-gather by posted stores (own arena included)
        m[b4 + i] = Mv; v[b4 + i] = Vv;
        gw[b4 + i] = Gs;  // the summed gradient of the owned slice stays readable (lrcn_get_grad gathers the slices)
      }
      __syncthreads();  // the chunk's staging rows and flags are consumed before the next wait
      mine++;
    }
    if (mine > 0 && tid < N && tid != me) red_release_sys_add(xdone(a.stage[tid], a.ctl4, a.bucket, me), (unsigned int)mine);  // one release per CTA
  }
  // ---- C: all owners' new weights of this bucket have landed in my arena
  if (blockIdx.x == 0) {
    if (tid < N && tid != me) {
      const size_t n4 = a.e4[tid] - a.b4[tid];
      const size_t XCH = (size_t)XSUB * a.sub;
      const unsigned int nch = (unsigned int)((n4 + XCH - 1) / XCH);
      if (nch) xwait(xdone(a.stage[me], a.ctl4, a.bucket, tid), epoch * nch, "the new weights", tid);
    }
    if (tid == 0 && loss_total) {
      double t = 0.0;
      for (int p = 0; p < N; p++) {
        double x;
        asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(x) : "l"(&peers.ctl[p]->loss_partial) : "memory");
        t += x;
      }
      *loss_total = t;
    }
  }
}
void dp_fused_exchange(cudaStream_t s, const P2PPeers& peers, const FusedXArgs& a0, float* m, float* v, const StepScalars* sc, double* loss_total, int grid_ctas) {
  FusedXArgs a = a0;
  size_t longest = 0;
  for (int r = 0; r < peers.nranks; r++) longest = a.e4[r] - a.b4[r] > longest ? a.e4[r] - a.b4[r] : longest;
  a.sub = (int)((longest + (size_t)XSUB * XMAXCH - 1) / ((size_t)XSUB * XMAXCH));  // at most XMAXCH chunks per slice
  if (a.sub < 1) a.sub = 1;
  fused_exchange_kernel<<<grid_ctas, 256, 0, s>>>(peers, a, reinterpret_cast<float4*>(m), reinterpret_cast<float4*>(v), sc, loss_total);
  if (g_counter) g_counter->n++;
}

// timeline stamps of the data-parallel step (LRCN_DP_STAMPS=1, tools/dp_timeline.py): %globaltimer at a point of a stream
__global__ void stamp_kernel(unsigned long long* out) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  *out = t;
}
void dp_stamp(cudaStream_t s, unsigned long long* out) { stamp_kernel<<<1, 1, 0, s>>>(out); }


}  // namespace lrcn
