// step_tail.cuh — everything of reverse_once that follows the rollouts (mbd_planner.py:110-135), for ANY number of
// ranks, in TWO launches (round 1: three kernels on one GPU, six plus two exchange kernels when sharded):
//
//   k_step_weights   ONE thread-block cluster of 8 CTAs x 1024 threads.  Sharded runs first rendezvous with the peer
//                    GPUs (system-scope release/acquire flags in the peers' symmetric buffers) and pull the peers'
//                    per-sample returns (and demo log-densities) over NVLink straight into the statistics pass — the
//                    exchange IS the first read of the data, there is no separate gather kernel.  Then the global mean /
//                    population std / demo blend / softmax of mbd_planner.py:110-127: every reduction is a block
//                    butterfly followed by a DSMEM exchange of the eight CTA partials (cluster barrier), so 65,536
//                    samples (8 GPUs x 8192) cost eight elements per thread instead of sixty-four in one CTA.
//   k_step_update    weighted-mean runs (64 samples, sequential fmaf) on ceil(n/64) x ceil(HNu/256) CTAs; the LAST CTA of
//                    each column block (atomic ticket) folds the runs with the adjacent-pairwise tree and, on one rank,
//                    applies the update lines 130-133 at once; sharded, it publishes the rank partial, the last column
//                    block rendezvous with the peers, reads their partials over NVLink, folds them in rank order and
//                    applies the update.
//
// Both kernels take the step's parameters (PRNG key, sigma, the five schedule scalars) from a DEVICE table indexed by a
// DEVICE step counter, and the last thread of k_step_update decrements that counter: a diffusion step is three
// parameterless launches that can be captured once in a CUDA graph and replayed Ndiffuse-1 times.
//
// Determinism: every reduction order is a function of (N, n_local / 64) only — never of the rank count — so sharded and
// unsharded runs agree bit for bit whenever N/P is 64 * 2^k (same guarantee as round 1).
#pragma once

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "mbd_b200.h"
#include "mbd_fp32.h"

namespace mbd {

namespace cg = cooperative_groups;

constexpr int kClusterCtas = 8;         // portable cluster size
constexpr int kWeightsThreads = 1024;
constexpr int kTailRun = 64;            // samples per sequential run (== kRun in mbd_b200.cu)
constexpr int kUpdThreads = 256;

struct TailArgs {
  // step parameters (device)
  const mbd_step_params* sp;
  mbd_step_ctl* ctl;
  float* Ybars;           // [Ndiffuse][HNu]
  float* rew_hist;        // [Ndiffuse] or null
  int N, n_begin, n_local, HNu;
  float temp, rew_xref;
  int demo;
  // buffers
  const float* Y0s;       // [n_local][HNu]
  const float* rews;      // local returns [n_local]
  const float* logpd;     // local demo log-densities or null
  float* rews_all;        // [N]   (P == 1: aliases rews)
  float* logpd_all;       // [N]   (P == 1: aliases logpd)
  float* logp;            // [N] scratch
  float* weights;         // [n_local]
  float* runs;            // [nruns][HNu]
  float* partial;         // [HNu] this rank's partial (P > 1: lives in the symmetric buffer)
  float* scalars;         // [4]
  // exchange
  float* peer[8];
  int P, rank;
  unsigned long long off_rews, off_logpd, off_partial, off_flags;   // word offsets in the symmetric buffer
  unsigned long long timeout_cycles;
  // batched solves (one rank): solve s owns row s of every per-solve array (mbd_step_plan layout); nd = Ndiffuse
  const float* temps;     // [S] or null (one solve: `temp`)
  int nd;
};

// Moves every per-solve pointer of `a` to solve s (s = 0: no-op) and takes that solve's temperature.  Each solve then runs
// exactly the code, and therefore the reduction trees, of a lone solve.
__device__ __forceinline__ void tail_solve(TailArgs& a, int s) {
  if (a.temps) a.temp = a.temps[s];
  const size_t n = (size_t)s * a.n_local, N = (size_t)s * a.N, HNu = a.HNu;
  const size_t nruns = (a.n_local + kTailRun - 1) / kTailRun;
  a.sp += (size_t)s * a.nd; a.ctl += s; a.Ybars += (size_t)s * a.nd * HNu;
  if (a.rew_hist) a.rew_hist += (size_t)s * a.nd;
  a.Y0s += n * HNu; a.rews += n; a.weights += n;
  if (a.logpd) a.logpd += n;
  a.rews_all += N; a.logp += N;
  if (a.logpd_all) a.logpd_all += N;
  a.runs += (size_t)s * nruns * HNu; a.partial += (size_t)s * HNu; a.scalars += (size_t)s * 4;
}

__device__ __forceinline__ void tail_st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int tail_ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Cross-GPU rendezvous, executed by threads 0..P-1 of ONE CTA: publish `epoch` into slot [rank] of flag row `row` of every
// peer, then wait until the own row shows `epoch` from every peer.  Stream order on each rank guarantees that the
// producer kernel of the data finished before its flag is published.  Returns false on timeout (a peer died or diverged):
// the caller then POISONS its output with NaN so that the failure cannot go unnoticed, and sets ctl->err.
__device__ __forceinline__ bool peer_rendezvous(const TailArgs& a, int row, unsigned int epoch) {
  bool ok = true;
  if ((int)threadIdx.x < a.P) {
    __threadfence_system();
    tail_st_release_sys(reinterpret_cast<unsigned int*>(a.peer[threadIdx.x]) + a.off_flags + 8 * row + a.rank, epoch);
    const unsigned int* f = reinterpret_cast<const unsigned int*>(a.peer[a.rank]) + a.off_flags + 8 * row + threadIdx.x;
    const long long t0 = clock64();
    while ((int)(tail_ld_acquire_sys(f) - epoch) < 0) {
      if ((unsigned long long)(clock64() - t0) > a.timeout_cycles) { ok = false; break; }
    }
  }
  return ok;
}

enum { TOP_SUM = 0, TOP_MAX = 1 };

// deterministic block reduction (butterfly inside the warp, then warp 0 over the warp results); every thread gets the result
template <int OP>
__device__ __forceinline__ float tail_block_reduce(float v, float* sh) {
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_xor_sync(0xffffffffu, v, o);
    v = OP == TOP_SUM ? v + t : fmaxf(v, t);
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = sh[threadIdx.x & 31];
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_xor_sync(0xffffffffu, r, o);
    r = OP == TOP_SUM ? r + t : fmaxf(r, t);
  }
  return r;
}

// cluster-wide reduction: block result -> this CTA's slot `pass` in shared memory -> cluster barrier -> lanes 0..7 of warp 0
// read the eight slots through distributed shared memory and fold them with a butterfly (fixed order) -> broadcast
template <int OP>
__device__ __forceinline__ float cluster_reduce(float v, float* sh, float* slots, float* bcast, int pass, cg::cluster_group& cl) {
  float b = tail_block_reduce<OP>(v, sh);
  if (threadIdx.x == 0) slots[pass] = b;
  cl.sync();
  if (threadIdx.x < 32) {
    float r = OP == TOP_SUM ? 0.0f : -INFINITY;
    if (threadIdx.x < kClusterCtas) r = cl.map_shared_rank(slots, threadIdx.x)[pass];
    for (int o = 1; o < kClusterCtas; o <<= 1) {
      float t = __shfl_xor_sync(0xffffffffu, r, o);
      r = OP == TOP_SUM ? r + t : fmaxf(r, t);
    }
    if (threadIdx.x == 0) *bcast = r;
  }
  __syncthreads();
  float r = *bcast;
  __syncthreads();   // *bcast may be rewritten by the next pass
  return r;
}

// mbd_planner.py:110-127.  One cluster; thread g of the 8192 cluster threads owns the elements i = g (mod 8192): it re-reads
// only its own elements in every pass, so the passes need no memory barrier beyond the reductions themselves.
// BATCH: one cluster per solve of a batched step (the single-solve instantiation is the kernel as it was)
template <bool BATCH>
__global__ void __cluster_dims__(kClusterCtas, 1, 1) __launch_bounds__(kWeightsThreads, 1) k_step_weights(TailArgs a) {
  __shared__ float sh[32];
  __shared__ float slots[16];
  __shared__ float bcast;
  __shared__ int s_ok;
  cg::cluster_group cl = cg::this_cluster();
  if constexpr (BATCH) tail_solve(a, (int)(blockIdx.x / kClusterCtas));
  const int g =(int)cl.block_rank() * kWeightsThreads + threadIdx.x;
  constexpr int G = kClusterCtas * kWeightsThreads;
  const int N = a.N;
  const float fN = (float)N;
  const int step = a.ctl->i;
  bool ok = true;
  if (a.P > 1) {
    // rendezvous #1 of the step (flag row 0), then pull every rank's returns over NVLink into rews_all / logpd_all
    if (cl.block_rank() == 0) {
      bool mine = peer_rendezvous(a, 0, 2u * a.ctl->epoch + 1u);
      int all = __syncthreads_and(mine ? 1 : 0);
      if (threadIdx.x == 0) s_ok = all;
    }
    cl.sync();
    ok = cl.map_shared_rank(&s_ok, 0)[0] != 0;
    const int nl = a.n_local;
    // eight NVLink loads in flight per thread (one round trip for the 65,536 returns of an 8 x 8192 run instead of eight)
    for (int i0 = g; i0 < N; i0 += 8 * G) {
      float vr[8], vl[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int i = i0 + k * G;
        const int r = i < N ? i / nl : 0, j = i < N ? i - r * nl : 0;
        float* base = a.peer[0];
#pragma unroll
        for (int q = 1; q < 8; ++q) base = (r == q) ? a.peer[q] : base;    // select instead of a dynamically indexed parameter array
        vr[k] = (ok && i < N) ? __ldcv(base + a.off_rews + j) : __int_as_float(0x7fc00000);
        vl[k] = (ok && i < N && a.demo) ? __ldcv(base + a.off_logpd + j) : __int_as_float(0x7fc00000);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int i = i0 + k * G;
        if (i < N) {
          a.rews_all[i] = vr[k];
          if (a.demo) a.logpd_all[i] = vl[k];
        }
      }
    }
    if (!ok && g == 0) a.ctl->err = 1u;
  }
  const float* rews = a.rews_all;
  float acc = 0.0f;
  for (int i = g; i < N; i += G) acc += rews[i];
  const float rew_mean = cluster_reduce<TOP_SUM>(acc, sh, slots, &bcast, 0, cl) / fN;
  acc = 0.0f;
  for (int i = g; i < N; i += G) { float d = rews[i] - rew_mean; acc = fmaf(d, d, acc); }
  float rew_std = sqrtf(cluster_reduce<TOP_SUM>(acc, sh, slots, &bcast, 1, cl) / fN);   // population std (ddof 0)
  rew_std = rew_std < 1e-4f ? 1.0f : rew_std;
  float* logp = a.logp;
  int pass = 2;
  if (a.demo) {
    const float* logpd = a.logpd_all;
    float mxd = -INFINITY;
    for (int i = g; i < N; i += G) mxd = fmaxf(mxd, logpd[i]);
    mxd = cluster_reduce<TOP_MAX>(mxd, sh, slots, &bcast, pass++, cl);
    acc = 0.0f;
    for (int i = g; i < N; i += G) {
      float l0 = (rews[i] - rew_mean) / rew_std / a.temp;
      float ld = ((logpd[i] - mxd) + a.rew_xref - rew_mean) / rew_std / a.temp;
      float l = ld > l0 ? ld : l0;
      logp[i] = l;
      acc += l;
    }
    const float lmean = cluster_reduce<TOP_SUM>(acc, sh, slots, &bcast, pass++, cl) / fN;
    acc = 0.0f;
    for (int i = g; i < N; i += G) { float d = logp[i] - lmean; acc = fmaf(d, d, acc); }
    const float lstd = sqrtf(cluster_reduce<TOP_SUM>(acc, sh, slots, &bcast, pass++, cl) / fN);
    for (int i = g; i < N; i += G) logp[i] = (logp[i] - lmean) / lstd / a.temp;
  } else {
    for (int i = g; i < N; i += G) logp[i] = (rews[i] - rew_mean) / rew_std / a.temp;
  }
  float mx = -INFINITY;
  for (int i = g; i < N; i += G) mx = fmaxf(mx, logp[i]);
  mx = cluster_reduce<TOP_MAX>(mx, sh, slots, &bcast, pass++, cl);
  acc = 0.0f;
  for (int i = g; i < N; i += G) acc += mbd_expf(logp[i] - mx);
  const float S = cluster_reduce<TOP_SUM>(acc, sh, slots, &bcast, pass++, cl);
  for (int i = g; i < N; i += G) {
    const int j = i - a.n_begin;
    if (j >= 0 && j < a.n_local) a.weights[j] = mbd_expf(logp[i] - mx) / S;
  }
  if (g == 0) {
    a.scalars[0] = rew_mean; a.scalars[1] = rew_std; a.scalars[2] = mx; a.scalars[3] = S;
    if (a.rew_hist) a.rew_hist[step] = rew_mean;
  }
  cl.sync();   // no CTA may exit while its shared memory can still be read by a peer CTA
}

// adjacent-pairwise tree over `count` rows (binary-counter stack, aligned blocks of 8 rows loaded together) — the same
// association as tree_sum_rows in mbd_b200.cu, but with L2 (cache-global) loads: the rows were written by OTHER CTAs of the
// SAME launch, so the non-coherent L1 / read-only path must not be used.
template <bool PEER>
__device__ __forceinline__ float tail_tree_rows(const float* const* bases, const float* rows, int count, size_t stride, int j) {
  auto ld = [&](int r) -> float { return PEER ? __ldcv(bases[r] + j) : __ldcg(rows + (size_t)r * stride + j); };
  float stack[32];
  int depth = 0, r = 0;
  // aligned blocks of 32 rows: 32 loads in flight, folded in registers in adjacent-pair order (5 levels) and pushed at level 5 —
  // the association of the binary counter, with a quarter of the L2 round trips of the 8-row blocks
  for (; r + 32 <= count; r += 32) {
    float v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = ld(r + k);
#pragma unroll
    for (int w = 1; w < 32; w <<= 1)
#pragma unroll
      for (int k = 0; k < 32; k += 2 * w) v[k] = v[k] + v[k + w];
    float b = v[0];
    int rr = r >> 5;
    int lvl = 0;
    while (rr & 1) { b = stack[--depth] + b; rr >>= 1; ++lvl; }
    (void)lvl;
    stack[depth++] = b;
  }
  // after the 32-blocks the counter holds one entry per set bit of (r >> 5), all at levels >= 5; the rest (< 32 rows) is
  // folded by 8-row blocks (level 3) and single rows exactly as before, then merged top-down
  float sub[4];      // sub-stack of the ragged part, levels 3..4 (at most 3 blocks of 8)
  int sd = 0;
  for (int q = 0; r + 8 <= count; r += 8, ++q) {
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = ld(r + k);
    float b = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
    int rr = q;
    while (rr & 1) { b = sub[--sd] + b; rr >>= 1; }
    sub[sd++] = b;
  }
  float tail_v = 0.0f;
  bool has_tail = false;
  if (r < count) {
    float tstack[4];
    int td = 0;
    for (int q = 0; r + q < count; ++q) {
      float v = ld(r + q);
      int rr = q;
      while (rr & 1) { v = tstack[--td] + v; rr >>= 1; }
      tstack[td++] = v;
    }
    float v = tstack[--td];
    while (td > 0) v = tstack[--td] + v;
    tail_v = v;
    has_tail = true;
  }
  // merge: ragged singles into the 8-block sub-stack, that into the main stack, then the main stack top-down
  float acc = 0.0f;
  bool have = false;
  if (has_tail) { acc = tail_v; have = true; }
  while (sd > 0) { float t = sub[--sd]; acc = have ? t + acc : t; have = true; }
  while (depth > 0) { float t = stack[--depth]; acc = have ? t + acc : t; have = true; }
  return acc;
}

// mbd_planner.py:100,130-133 literally (k_update in mbd_b200.cu)
__device__ __forceinline__ float diffusion_update(float Ybar, float Ybar_i, const mbd_step_params& p) {
  float Yi = Ybar_i * p.coef[0];
  float score = p.coef[1] * (-Yi + p.coef[0] * Ybar);
  float Yim1 = p.coef[3] * (Yi + p.coef[2] * score);
  return Yim1 / p.coef[4];
}

// grid (nruns, ceil(HNu / 256), S); block 256.  ctl->ticket[y]: per column block y; ctl->ticket[MBD_STEP_MAX_COLBLOCKS]: over the
// column blocks.  Batched: blockIdx.z is the solve, and the tickets and the counter are that solve's.
template <bool BATCH>
__global__ void __launch_bounds__(kUpdThreads) k_step_update(TailArgs a) {
  __shared__ int s_flag;
  if constexpr (BATCH) tail_solve(a, (int)blockIdx.z);
  const int tid = threadIdx.x;
  const int j = blockIdx.y * kUpdThreads + tid;
  const int HNu = a.HNu;
  const int nruns = gridDim.x;
  const int step = a.ctl->i;
  {
    const int r = blockIdx.x;
    const int n0 = r * kTailRun, n1 = min(n0 + kTailRun, a.n_local);
    if (j < HNu) {
      const float* __restrict__ w = a.weights;
      const float* __restrict__ Y = a.Y0s;
      float acc;
      if (n1 - n0 == kTailRun) {
        // full run: 16 loads in flight per thread (the accumulation order stays sequential)
        float y[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) y[k] = Y[(size_t)(n0 + k) * HNu + j];
        acc = w[n0] * y[0];
#pragma unroll
        for (int k = 1; k < 16; ++k) acc = fmaf(w[n0 + k], y[k], acc);
#pragma unroll
        for (int b = 16; b < kTailRun; b += 16) {
#pragma unroll
          for (int k = 0; k < 16; ++k) y[k] = Y[(size_t)(n0 + b + k) * HNu + j];
#pragma unroll
          for (int k = 0; k < 16; ++k) acc = fmaf(w[n0 + b + k], y[k], acc);
        }
      } else {
        acc = w[n0] * Y[(size_t)n0 * HNu + j];
        for (int n = n0 + 1; n < n1; ++n) acc = fmaf(w[n], Y[(size_t)n * HNu + j], acc);
      }
      a.runs[(size_t)r * HNu + j] = acc;
    }
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) s_flag = (atomicAdd(&a.ctl->ticket[blockIdx.y], 1u) == (unsigned)(nruns - 1));
  __syncthreads();
  if (!s_flag) return;
  // ---- last CTA of this column block: every run row of these columns is complete -------------------------------------
  __threadfence();
  const mbd_step_params p = a.sp[step];
  float* out = a.Ybars + (size_t)(step - 1) * HNu;
  const float* Ybar_i = a.Ybars + (size_t)step * HNu;
  if (j < HNu) {
    const float v = tail_tree_rows<false>(nullptr, a.runs, nruns, (size_t)HNu, j);
    if (a.P == 1) out[j] = diffusion_update(v, Ybar_i[j], p);
    else a.partial[j] = v;
  }
  if (tid == 0) a.ctl->ticket[blockIdx.y] = 0u;
  __threadfence();
  __syncthreads();
  if (tid == 0) s_flag = (atomicAdd(&a.ctl->ticket[MBD_STEP_MAX_COLBLOCKS], 1u) == gridDim.y - 1);
  __syncthreads();
  if (!s_flag) return;
  // ---- the very last CTA of the launch ----------------------------------------------------------------------------------
  __threadfence();
  if (a.P > 1) {
    // rendezvous #2 (flag row 1): every rank's partial is complete; fold them in rank order and apply the update
    bool mine = peer_rendezvous(a, 1, 2u * a.ctl->epoch + 2u);
    const bool ok = __syncthreads_and(mine ? 1 : 0) != 0;
    const float* bases[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) bases[r] = a.peer[r < a.P ? r : 0] + a.off_partial;
    for (int c = tid; c < HNu; c += kUpdThreads) {
      const float v = tail_tree_rows<true>(bases, nullptr, a.P, 0, c);
      out[c] = ok ? diffusion_update(v, Ybar_i[c], p) : __int_as_float(0x7fc00000);
    }
    if (!ok && tid == 0) a.ctl->err = 1u;
  }
  __syncthreads();
  if (tid == 0) {
    a.ctl->ticket[MBD_STEP_MAX_COLBLOCKS] = 0u;
    a.ctl->epoch = a.ctl->epoch + 1u;
    a.ctl->i = step - 1;
  }
}

// ---- measured fp32 peak (bench.py roofline_fp32 denominator; SURVEY 8d asks for an FFMA micro-benchmark) ---------------
// 16 independent FFMA chains per thread, 1024 threads per CTA, two CTAs per SM: the fp32 pipe is the only limiter.
__global__ void __launch_bounds__(1024, 2) k_ffma_peak(float* out, int iters, float a, float b) {
  float x[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) x[k] = (float)(threadIdx.x + k) * 1e-3f;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int k = 0; k < 16; ++k) x[k] = fmaf(x[k], a, b);
    }
  }
  float s = 0.0f;
#pragma unroll
  for (int k = 0; k < 16; ++k) s += x[k];
  if (s == 123.456f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;   // never true: keeps the chains alive
}

}  // namespace mbd
