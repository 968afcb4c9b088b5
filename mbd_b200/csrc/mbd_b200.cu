// mbd_b200.cu — kernels + C ABI (include/mbd_b200.h) of the B200-native MBD hot path.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo (see build.py).
//
// Kernels
//   k_rollout<FUSED>   sampling (threefry + erfinv, optional) + Nsample x H env steps of the
//                      Brax-positional pipeline, one link per lane, model staged by TMA.
//   k_car2d            the self-contained kinematic car env, one sample per thread.
//   k_sample           stand-alone jax.random.normal sampling.
//   k_softmax_weights  global reward statistics, demo blend and softmax (single CTA).
//   k_wsum_runs / k_wsum_tree / k_update   deterministic weighted mean + diffusion update.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stddef.h>
#include <string.h>

#include <type_traits>

#include <cooperative_groups.h>

#include "mbd_b200.h"
#include "mbd_fp32.h"
#include "mbd_model.h"
#include "xpbd_device.cuh"
#include "xpbd_wpl.cuh"
#include "xpbd_pk.cuh"
#include "step_tail.cuh"

namespace mbd {

constexpr int kLPS = MBD_MAXL;          // lanes per sample group
constexpr int kRolloutThreads = 128;    // 8 sample groups per CTA
constexpr int kSPB = kRolloutThreads / kLPS;
constexpr int kRun = 64;                // samples per sequential run in the weighted sum

// ---- TMA bulk copy of the model blob into shared memory ---------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void stage_model_tma(float* sblob, uint64_t* mbar, const uint32_t* gblob) {
  constexpr uint32_t kBytes = MBD_BLOB_WORDS * 4;
  static_assert(kBytes % 16 == 0, "bulk copy size must be a multiple of 16 bytes");
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(kBytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sblob)),
                 "l"(gblob), "r"(kBytes), "r"(smem_u32(mbar))
                 : "memory");
  }
  // every thread waits for phase 0 to complete
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(mbar))
        : "memory");
  }
}

// ---- sampling helper: one element of clip(normal*sigma + Ybar, -1, 1) -----------------------------
__device__ __forceinline__ float sample_elem(uint32_t k0, uint32_t k1, uint32_t idx, uint32_t total, float sigma, float ybar) {
  float eps = mbd_bits_to_normal(mbd_random_bits_at(k0, k1, idx, total));
  float y = eps * sigma + ybar;
  return clampf(y, -1.0f, 1.0f);
}

struct SampleParams { uint32_t k0, k1; float sigma; const float* Ybar; };

__global__ void k_sample(uint32_t k0, uint32_t k1, uint32_t total, uint32_t begin, uint32_t count, int HNu, float sigma,
                         const float* __restrict__ Ybar, float* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  uint32_t idx = begin + i;
  out[i] = sample_elem(k0, k1, idx, total, sigma, Ybar[idx % (uint32_t)HNu]);
}

// ---- batched solves (mbd_step_plan.n_solves > 1): the solve is blockIdx.y of the fused launch -----------------------
// Per-solve strides in elements of the arrays that carry a leading solve axis; all zero (and gridDim.y == 1) outside a
// batched step, so the offsets below vanish.  The noise index stays n_begin + ns inside the solve: solve s draws exactly
// the noise of a lone solve with its key.
struct SolveStride { unsigned int state, y0s, n, nd, ybars; };
template <class St>
__device__ __forceinline__ void solve_offsets(const SolveStride& z, St*& state, float*& Y0s, float*& rews, float*& logpd,
                                              const mbd_step_params*& sp, const mbd_step_ctl*& ctl, const float*& Ybars) {
  const size_t s = blockIdx.y;
  state += s * z.state; Y0s += s * z.y0s; rews += s * z.n;
  if (logpd) logpd += s * z.n;
  sp += s * z.nd; ctl += s; Ybars += s * z.ybars;
}

// ---- the rollout kernel ----------------------------------------------------------------------------
struct RolloutArgs {
  const uint32_t* blob;    // device copy of the model blob
  const float* state_init; // [L,13]
  float* Y0s;              // [n,H,nu]  (input, or output+input when FUSED)
  int n, H;
  float* rewss;            // [n,H] or null
  float* rews;             // [n]
  const float* xref;       // [ntrack,href,3] or null
  int href;
  float* logpd;            // [n] or null
  float* final_state;      // [n,L,13] or null
  float* track_pos;        // [n,H,ntrack,3] or null
  int nsub_override;
  // fused sampling
  uint32_t k0, k1;
  int n_total, n_begin;
  float sigma;
  const float* Ybar;       // [H*nu]
  // fused sampling with DEVICE-resident step parameters (graph-capturable step, step_tail.cuh): when sp != null the key,
  // sigma and the iterate row are taken from sp[ctl->i] / Ybars + ctl->i * HNu instead of the by-value fields above
  const mbd_step_params* sp;
  const mbd_step_ctl* ctl;
  const float* Ybars;
  int prng_part;           // 1: partitionable threefry layout (mbd_set_prng_layout), 0: legacy
  // v2 mapping: link owned by (warp, half) and the half-warp offset (in units of 4 lanes) of every link's row
  signed char wl[MBD_MAXL][2];
  unsigned long long offs;
  // warp-uniform link topology, copied from the blob by the host: read through the constant bank with a warp-uniform
  // index (the warp id is taken through __shfl_sync(.., 0), which the compiler tracks as uniform), so ndof / parent /
  // children / contact count live in UNIFORM registers and every branch on them is a uniform branch — no BSSY / BSYNC /
  // WARPSYNC convergence bookkeeping around code that can never diverge (22 % of the stall samples of the round-1 kernel)
  struct LinkCfgP { signed char ndof, parent, ncon, smask, child[MBD_MAXCHILD]; } cfg[MBD_MAXL];
  // multi-group CTAs: warp -> (group << 4) | link slot
  signed char gw[32];
  int count_x;             // group barriers: 32 * (links that are not leaves with contacts), see SyncGroup
  int stagger;             // two-group CTA: cycles group 1 waits before its first step (experiment: de-phase the groups)
  SolveStride ss;          // batched step: per-solve strides (FUSED kernels only; zero otherwise)
};
// the per-solve pointers of a fused rollout launch, formed where they are used: the kernel parameter itself is never
// written (a written parameter struct is copied to local memory as a whole), and the output pointers are not kept live
// across the rollout loop (they would cost registers in the single-solve kernels)
template <bool FUSED>
__device__ __forceinline__ size_t solve_index() { return FUSED ? (size_t)blockIdx.y : 0; }
template <bool FUSED>
struct SolvePtrs {   // blockIdx.y is re-read at every use instead of being held in a register
  const RolloutArgs& a;
  __device__ __forceinline__ const float* state_init() const { return a.state_init + solve_index<FUSED>() * a.ss.state; }
  __device__ __forceinline__ float* Y0s() const { return a.Y0s + solve_index<FUSED>() * a.ss.y0s; }
  __device__ __forceinline__ float* rews() const { return a.rews + solve_index<FUSED>() * a.ss.n; }
  __device__ __forceinline__ float* logpd() const { return a.logpd + solve_index<FUSED>() * a.ss.n; }
};
template <bool FUSED>
__device__ __forceinline__ SolvePtrs<FUSED> solve_ptrs(const RolloutArgs& a) { return SolvePtrs<FUSED>{a}; }

__device__ __forceinline__ SampleParams sample_params(const RolloutArgs& a, int HNu) {
  SampleParams q;
  q.k0 = a.k0; q.k1 = a.k1; q.sigma = a.sigma; q.Ybar = a.Ybar;
  if (a.sp != nullptr) {
    const size_t s = blockIdx.y;   // solve of a batched step (0 otherwise)
    const mbd_step_params* sp = a.sp + s * a.ss.nd;
    const int i = a.ctl[s].i;
    q.k0 = sp[i].key[0]; q.k1 = sp[i].key[1]; q.sigma = sp[i].sigma;
    q.Ybar = a.Ybars + s * a.ss.ybars + (size_t)i * HNu;
  }
  return q;
}

template <bool FUSED, int CMAX>
__global__ void __launch_bounds__(kRolloutThreads) k_rollout(RolloutArgs a) {
  __shared__ __align__(128) float sblob[MBD_BLOB_WORDS];
  __shared__ __align__(8) uint64_t mbar;
  const SolvePtrs<FUSED> so = solve_ptrs<FUSED>(a);
  stage_model_tma(sblob, &mbar, a.blob);
  ModelSmem M;
  M.f = sblob;

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int L = M.hi(MBD_H_NLINK), nu = M.hi(MBD_H_NU);
  const int HNu = a.H * nu;
  const int nsub = a.nsub_override > 0 ? a.nsub_override : M.hi(MBD_H_NFRAMES);
  const int reward_kind = M.hi(MBD_H_REWARD);
  const int ntrack = M.hi(MBD_H_NTRACK);

  if (FUSED) {
    // each CTA draws the noise of exactly its own samples, then reads it back after the barrier
    const uint32_t total = a.prng_part ? 0u : (uint32_t)a.n_total * (uint32_t)HNu;   // 0 selects the partitionable layout
    const SampleParams sq = sample_params(a, HNu);
    const int first = blockIdx.x * kSPB;
    const int cnt = min(kSPB, a.n - first) * HNu;
    for (int e = tid; e < cnt; e += kRolloutThreads) {
      int ns = first + e / HNu, j = e % HNu;
      uint32_t idx = (uint32_t)(a.n_begin + ns) * (uint32_t)HNu + (uint32_t)j;
      so.Y0s()[(size_t)ns * HNu + j] = sample_elem(sq.k0, sq.k1, idx, total, sq.sigma, sq.Ybar[j]);
    }
    __syncthreads();
  }

  LaneCfg c;
  load_lane_cfg(M, lane, kLPS, c);
  StepConsts K;
  load_step_consts(M, K);

  const int n_local = blockIdx.x * kSPB + tid / kLPS;
  const bool active = n_local < a.n;
  const int n_rd = active ? n_local : 0;
  const bool live = c.l < L;

  LinkState s;
  {
    const float* st = so.state_init() + (live ? c.l : 0) * MBD_STATE_STRIDE;
    s.p = V3(st[0], st[1], st[2]);
    s.q = Q4(st[3], st[4], st[5], st[6]);
    s.w = V3(st[7], st[8], st[9]);
    s.v = V3(st[10], st[11], st[12]);
    if (!live) { s.p = V3(0, 0, 0); s.q = Q4(1, 0, 0, 0); s.w = V3(0, 0, 0); s.v = V3(0, 0, 0); }
  }
  // actuator.to_tau constants of this lane's dofs
  int aid[MBD_MAXDOF];
  float gear[MBD_MAXDOF], clo[MBD_MAXDOF], chi[MBD_MAXDOF];
#pragma unroll
  for (int k = 0; k < MBD_MAXDOF; ++k) {
    int base = MBD_F_DOF0 + k * MBD_DOF_STRIDE;
    bool has = live && k < c.ndof;
    aid[k] = has ? M.li(base + MBD_D_ACT, c.l) : -1;
    gear[k] = M.lf(base + MBD_D_GEAR, live ? c.l : 0);
    clo[k] = M.lf(base + MBD_D_CLO, live ? c.l : 0);
    chi[k] = M.lf(base + MBD_D_CHI, live ? c.l : 0);
  }
  int my_track = -1;
  for (int k = 0; k < ntrack; ++k)
    if (live && M.hi(MBD_H_TRACK0 + k) == c.l) my_track = k;

  float rsum = 0.0f, tacc = 0.0f;
  const float* urow = so.Y0s() + (size_t)n_rd * HNu;
  for (int t = 0; t < a.H; ++t) {
    float tau[MBD_MAXDOF];
#pragma unroll
    for (int k = 0; k < MBD_MAXDOF; ++k) {
      float u = aid[k] >= 0 ? urow[t * nu + aid[k]] : 0.0f;
      tau[k] = aid[k] >= 0 ? gear[k] * clampf(u, clo[k], chi[k]) : 0.0f;
    }
    float r_pre = 0.0f;
    if (reward_kind == MBD_REWARD_HUMANOIDTRACK && c.l == 0) {
      v3 x0 = link_origin(M, c, s);
      v3 v0 = link_origin_vel(M, c, s);
      r_pre = 1.0f + ((-fabsf(v0.x - 1.6f) - fabsf(x0.z - 1.3f)) - fabsf(x0.y) * 0.1f);
    }
    if (reward_kind == MBD_REWARD_ANT && c.l == 0) r_pre = link_origin(M, c, s).x;   // root x before the step
    for (int f = 0; f < nsub; ++f) positional_step<CMAX>(M, c, K, s, tau);
    const q4 q_link1 = shfl4(s.q, c.gbase + 1);   // cartpole reward: the pole's rotation (all lanes shuffle)
    if (c.l == 0) {
      float r;
      if (reward_kind == MBD_REWARD_HUMANOIDTRACK) {
        r = r_pre;
      } else if (reward_kind == MBD_REWARD_ANT) {
        r = reward_ant(M, r_pre, link_origin(M, c, s).x, urow + t * nu, nu);
      } else if (reward_kind == MBD_REWARD_HOPPER) {
        r = reward_hopper(M, link_origin(M, c, s));
      } else if (reward_kind == MBD_REWARD_CARTPOLE) {
        r = reward_cartpole(M, s, q_link1);
      } else {
        r = reward_post(reward_kind, link_origin(M, c, s));
      }
      rsum += r;
      if (a.rewss && active) a.rewss[(size_t)n_local * a.H + t] = r;
    }
    if (my_track >= 0) {
      v3 x = link_origin(M, c, s);
      if (a.track_pos && active) {
        float* o = a.track_pos + (((size_t)n_local * a.H + t) * ntrack + my_track) * 3;
        o[0] = x.x; o[1] = x.y; o[2] = x.z;
      }
      if (a.xref) {
        int tt = t < a.href ? t : a.href - 1;
        const float* xr = a.xref + ((size_t)my_track * a.href + tt) * 3;
        v3 d = V3(x.x - xr[0], x.y - xr[1], x.z - xr[2]);
        float nr = sqrtf(vdot(d, d));
        float cl = nr < 0.5f ? nr : 0.5f;
        float q = cl / 0.5f;
        tacc = fmaf(q, q, tacc);
      }
    }
  }
  if (c.l == 0 && active) so.rews()[n_local] = rsum / (float)a.H;
  if (a.logpd && a.xref) {
    // sum the per-body accumulators in track order on lane 0 of the group
    float tot = 0.0f;
    for (int k = 0; k < ntrack; ++k) {
      int src = c.gbase + M.hi(MBD_H_TRACK0 + k);
      float v = __shfl_sync(0xffffffffu, tacc, src);
      tot += v;
    }
    if (c.l == 0 && active) so.logpd()[n_local] = 0.0f - tot / (float)(ntrack * a.H);
  }
  if (a.final_state && active && live) {
    float* o = a.final_state + ((size_t)n_local * L + c.l) * MBD_STATE_STRIDE;
    o[0] = s.p.x; o[1] = s.p.y; o[2] = s.p.z;
    o[3] = s.q.w; o[4] = s.q.x; o[5] = s.q.y; o[6] = s.q.z;
    o[7] = s.w.x; o[8] = s.w.y; o[9] = s.w.z;
    o[10] = s.v.x; o[11] = s.v.y; o[12] = s.v.z;
  }
}

// ---- v2 rollout kernel: warp per link, lane per sample (xpbd_wpl.cuh) -------------------------------------
template <bool FUSED, int SYNC, int SPLIT, int CMAX, int GROUPS = 1, int kGroupLinks = MBD_MAXL>
__device__ __forceinline__ void rollout_wpl_body(const RolloutArgs& a, float* sblob, uint64_t* mbar_p, uint64_t* edge_bars, float* dyn) {
  stage_model_tma(sblob, mbar_p, a.blob);
  ModelSmem M;
  M.f = sblob;
  const SolvePtrs<FUSED> so = solve_ptrs<FUSED>(a);

  static_assert(SPLIT == 1 || SPLIT == 2, "links per warp");
  static_assert(SPLIT == 1 || SYNC == 0, "edge barriers assume one link per warp");
  static_assert(GROUPS == 1 || (SPLIT == 1 && SYNC == 0), "sample groups: one link per warp, group barriers");
  constexpr int kLpl = kWplLanes / SPLIT;                      // lanes (= samples) per link
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);   // the warp id as a value the compiler knows to be warp-uniform
  // GROUPS independent 32-sample groups share the CTA with their warps INTERLEAVED (warp w -> group w % GROUPS,
  // link slot w / GROUPS), so the links that the mapping marks critical (highest slots) have the highest warp ids
  // of the whole CTA — the SM arbiter issues the highest eligible warp id first.
  const int gwe = GROUPS == 1 ? warp_u : a.gw[warp_u];
  const int grp = GROUPS == 1 ? 0 : (gwe >> 4);
  const int l = a.wl[gwe & 15][SPLIT == 1 ? 0 : lane / kLpl];  // warp (and half) -> link
  const int slot = lane % kLpl;                                // sample index inside the CTA
  const int L = M.hi(MBD_H_NLINK), nu = M.hi(MBD_H_NU);
  const int HNu = a.H * nu;
  const int nsub = a.nsub_override > 0 ? a.nsub_override : M.hi(MBD_H_NFRAMES);
  const int reward_kind = M.hi(MBD_H_REWARD);
  const int ntrack = M.hi(MBD_H_NTRACK);
  const int nthreads = blockDim.x;

  if (FUSED) {
    const uint32_t total = a.prng_part ? 0u : (uint32_t)a.n_total * (uint32_t)HNu;   // 0 selects the partitionable layout
    const SampleParams sq = sample_params(a, HNu);
    const int first = blockIdx.x * kLpl * GROUPS;
    const int cnt = min(kLpl * GROUPS, a.n - first) * HNu;
    for (int e = tid; e < cnt; e += nthreads) {
      int ns = first + e / HNu, j = e % HNu;
      uint32_t idx = (uint32_t)(a.n_begin + ns) * (uint32_t)HNu + (uint32_t)j;
      so.Y0s()[(size_t)ns * HNu + j] = sample_elem(sq.k0, sq.k1, idx, total, sq.sigma, sq.Ybar[j]);
    }
    __syncthreads();
  }

  WplSmem S;
  S.X = dyn + grp * L * (kXF + kEF) * kWplLanes;
  S.E = S.X + L * kXF * kWplLanes;
  S.lane = slot;
  S.offs = a.offs;
  // a thread whose half owns no link (odd link count) shadows its partner's link into the unused half of
  // that row: it executes the same code, nobody reads what it writes, and it produces no output
  const bool owner = (S.off(l) == (lane / kLpl) * kLpl);
  if (!owner) S.offs = (S.offs & ~(0xFull << (4 * l))) | ((unsigned long long)(((lane / kLpl) * kLpl) >> 2) << (4 * l));
  WarpCfg c;
  if constexpr (SPLIT == 1) {
    c.l = l; c.ndof = a.cfg[l].ndof; c.parent = a.cfg[l].parent; c.ncon = a.cfg[l].ncon; c.smask = a.cfg[l].smask;
#pragma unroll
    for (int k = 0; k < MBD_MAXCHILD; ++k) c.child[k] = a.cfg[l].child[k];
  } else {
    load_warp_cfg(M, l, c);   // two links per warp: the topology differs between the half-warps
  }

  const int n_local = (blockIdx.x * GROUPS + grp) * kLpl + slot;
  const bool active = n_local < a.n && owner;
  const int n_rd = n_local < a.n ? n_local : a.n - 1;

  LinkState s;
  {
    const float* st = so.state_init() + l * MBD_STATE_STRIDE;
    s.p = V3(st[0], st[1], st[2]);
    s.q = Q4(st[3], st[4], st[5], st[6]);
    s.w = V3(st[7], st[8], st[9]);
    s.v = V3(st[10], st[11], st[12]);
  }
  S.put_p(l, s.p); S.put_q(l, s.q); S.put_w(l, s.w);
  typename std::conditional<GROUPS != 1, SyncGroup<kGroupLinks>,
      typename std::conditional<SYNC == 2, SyncNamed, SyncCta>::type>::type Y;
  if constexpr (GROUPS != 1) { Y.base = 1 + 4 * grp; Y.count_x = a.count_x; }
  if constexpr (SYNC == 2) Y.setup(M, l, L);
  int aid[MBD_MAXDOF];
#pragma unroll
  for (int k = 0; k < MBD_MAXDOF; ++k) aid[k] = k < c.ndof ? M.li(MBD_F_DOF0 + k * MBD_DOF_STRIDE + MBD_D_ACT, l) : -1;
  int my_track = -1;
  for (int k = 0; k < ntrack; ++k)
    if (M.hi(MBD_H_TRACK0 + k) == l) my_track = k;
  __syncthreads();
  if constexpr (SYNC != 0) Y.arrive_pose(l);  // the initial pose is published
  if constexpr (GROUPS != 1) {
    if (grp == 1 && a.stagger > 0) {
      const long long t0 = clock64();
      while (clock64() - t0 < (long long)a.stagger) {}
    }
  }
  float rsum = 0.0f, tacc = 0.0f;
  const float* urow = so.Y0s() + (size_t)n_rd * HNu;
  for (int t = 0; t < a.H; ++t) {
    float tau[MBD_MAXDOF];
#pragma unroll
    for (int k = 0; k < MBD_MAXDOF; ++k) {
      const int base = MBD_F_DOF0 + k * MBD_DOF_STRIDE;
      float u = aid[k] >= 0 ? urow[t * nu + aid[k]] : 0.0f;
      tau[k] = aid[k] >= 0 ? M.lf(base + MBD_D_GEAR, l) * clampf(u, M.lf(base + MBD_D_CLO, l), M.lf(base + MBD_D_CHI, l)) : 0.0f;
    }
    float r_pre = 0.0f;
    if (reward_kind == MBD_REWARD_HUMANOIDTRACK && l == 0) {
      v3 x0 = link_origin_w(M, 0, s);
      v3 v0 = link_origin_vel_w(M, 0, s);
      r_pre = 1.0f + ((-fabsf(v0.x - 1.6f) - fabsf(x0.z - 1.3f)) - fabsf(x0.y) * 0.1f);
    }
    if (reward_kind == MBD_REWARD_ANT && l == 0) r_pre = link_origin_w(M, 0, s).x;   // root x before the step
    for (int f = 0; f < nsub; ++f) positional_step_wpl<CMAX>(M, c, S, Y, s, tau);
    if (l == 0) {
      float r;
      if (reward_kind == MBD_REWARD_HUMANOIDTRACK) {
        r = r_pre;
      } else if (reward_kind == MBD_REWARD_ANT) {
        r = reward_ant(M, r_pre, link_origin_w(M, 0, s).x, urow + t * nu, nu);
      } else if (reward_kind == MBD_REWARD_HOPPER) {
        r = reward_hopper(M, link_origin_w(M, 0, s));
      } else if (reward_kind == MBD_REWARD_CARTPOLE) {
        r = reward_cartpole(M, s, S.xq(1));   // link 1 published its rotation before the end-of-substep barrier
      } else {
        r = reward_post(reward_kind, link_origin_w(M, 0, s));
      }
      rsum += r;
      if (a.rewss && active) a.rewss[(size_t)n_local * a.H + t] = r;
    }
    if (my_track >= 0) {
      v3 x = link_origin_w(M, l, s);
      if (a.track_pos && active) {
        float* o = a.track_pos + (((size_t)n_local * a.H + t) * ntrack + my_track) * 3;
        o[0] = x.x; o[1] = x.y; o[2] = x.z;
      }
      if (a.xref) {
        int tt = t < a.href ? t : a.href - 1;
        const float* xr = a.xref + ((size_t)my_track * a.href + tt) * 3;
        v3 d = V3(x.x - xr[0], x.y - xr[1], x.z - xr[2]);
        float nr = sqrtf(vdot(d, d));
        float cl = nr < 0.5f ? nr : 0.5f;
        float q = cl / 0.5f;
        tacc = fmaf(q, q, tacc);
      }
    }
  }
  if (l == 0 && active) so.rews()[n_local] = rsum / (float)a.H;
  if (a.logpd && a.xref) {
    // per-body accumulators -> shared (reuse E), summed in track order by warp 0
    __syncthreads();  // every warp is done with E
    if (my_track >= 0 && owner) S.E[my_track * kWplLanes + slot] = tacc;
    __syncthreads();
    if (l == 0 && active) {
      float tot = 0.0f;
      for (int k = 0; k < ntrack; ++k) tot += S.E[k * kWplLanes + slot];
      so.logpd()[n_local] = 0.0f - tot / (float)(ntrack * a.H);
    }
  }
  if (a.final_state && active) {
    float* o = a.final_state + ((size_t)n_local * L + l) * MBD_STATE_STRIDE;
    o[0] = s.p.x; o[1] = s.p.y; o[2] = s.p.z;
    o[3] = s.q.w; o[4] = s.q.x; o[5] = s.q.y; o[6] = s.q.z;
    o[7] = s.w.x; o[8] = s.w.y; o[9] = s.w.z;
    o[10] = s.v.x; o[11] = s.v.y; o[12] = s.v.z;
  }
}

template <bool FUSED, int NWARPS, int MINB, int SYNC, int SPLIT, int CMAX, int GROUPS = 1>
__global__ void __launch_bounds__(32 * NWARPS, MINB) k_rollout_wpl(RolloutArgs a) {
  __shared__ __align__(128) float sblob[MBD_BLOB_WORDS];
  __shared__ __align__(8) uint64_t mbar;
  __shared__ __align__(8) uint64_t edge_bars[2 * MBD_MAXL];
  extern __shared__ __align__(16) float dyn[];
  rollout_wpl_body<FUSED, SYNC, SPLIT, CMAX, GROUPS, NWARPS / GROUPS>(a, sblob, &mbar, edge_bars, dyn);
}

// ---- packed rollout kernel: warp per link, TWO samples per lane on FFMA2 / FMUL2 / FADD2 (xpbd_pk.cuh) -----------------
// One 64-sample group per CTA, one CTA per SM (11 warps, no register cap).  The fp32 pipe does the same work per sample
// as the scalar kernels, but every packed instruction advances two rollouts: half the issue slots and half the
// dependent-latency steps per sample.  Model constants are read from a duplicated (c, c) copy of the blob so that they are
// packed operands without a repack; exchange rows are 64-bit per lane (LDS.64 / STS.64).
template <int CMAX, class Sync>
__device__ __forceinline__ void positional_step_pk(const pk::Model<pk::f2>& M, const pk::Cfg& c, const pk::Smem<pk::f2>& S, Sync& Y,
                                                   pk::State<pk::f2>& s, const pk::f2 tau[MBD_MAXDOF]) {
  pk::Carry<pk::f2, CMAX> k;
  MBD_PH_BEGIN
  Y.wait_pose(c.ndof > 0 ? c.parent : -1);
  pk::phase_A<pk::f2, CMAX>(M, c, S, s, tau, k);
  MBD_PH(0)
  Y.arrive_terms(c.l);
  Y.end_A(c);
  MBD_PH(1)
  Y.wait_terms(c.child);
  pk::phase_B<pk::f2, CMAX>(M, c, S, s, k);
  MBD_PH(2)
  Y.arrive_pose(c.l);
  Y.end_B(c);
  MBD_PH(3)
  Y.wait_pose(c.ndof > 0 ? c.parent : -1);
  pk::phase_C<pk::f2, CMAX>(M, c, S, s, k);
  MBD_PH(4)
  Y.arrive_terms(c.l);
  Y.end_C(c);
  MBD_PH(5)
  Y.wait_terms(c.child);
  pk::phase_D<pk::f2, CMAX>(M, c, S, s, k);
  MBD_PH(6)
  Y.arrive_pose(c.l);
  Y.end_D(c);
  MBD_PH(7)
}

__device__ __forceinline__ v3 pk_lo(pk::V<pk::f2> a) { return V3(pk::lo(a.x), pk::lo(a.y), pk::lo(a.z)); }
__device__ __forceinline__ v3 pk_hi(pk::V<pk::f2> a) { return V3(pk::hi(a.x), pk::hi(a.y), pk::hi(a.z)); }

constexpr int kPkLinks = 11;       // links (= warps) per CTA the packed kernel is built for
constexpr int kPkSamples = 64;     // samples per CTA
constexpr size_t kPkDynBytes = (size_t)(MBD_BLOB_WORDS + kPkLinks * (pk::kXF + pk::kEF) * pk::kLanes) * sizeof(pk::f2);

template <bool FUSED, int CMAX, int SYNC>
__global__ void __launch_bounds__(32 * kPkLinks, 1) k_rollout_pk(RolloutArgs a) {
  __shared__ __align__(128) float sblob[MBD_BLOB_WORDS];
  __shared__ __align__(8) uint64_t mbar;
  extern __shared__ __align__(16) float dyn[];
  const SolvePtrs<FUSED> so = solve_ptrs<FUSED>(a);
  stage_model_tma(sblob, &mbar, a.blob);
  ModelSmem Ms;
  Ms.f = sblob;
  const int tid = threadIdx.x, lane = tid & 31, nthreads = blockDim.x;
  pk::f2* tab = reinterpret_cast<pk::f2*>(dyn);
  for (int i = tid; i < MBD_BLOB_WORDS; i += nthreads) tab[i] = pk::mk2(sblob[i], sblob[i]);
  pk::Model<pk::f2> M;
  M.t = tab;
  M.f = sblob;
  const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp id, known-uniform to the compiler (see RolloutArgs::cfg)
  const int l = a.wl[warp_u][0];   // warp -> link (scheduler-balanced order, build_pairing)
  const int L = M.hi(MBD_H_NLINK), nu = M.hi(MBD_H_NU);
  const int HNu = a.H * nu;
  const int nsub = a.nsub_override > 0 ? a.nsub_override : M.hi(MBD_H_NFRAMES);
  const int reward_kind = M.hi(MBD_H_REWARD);
  const int ntrack = M.hi(MBD_H_NTRACK);

  if (FUSED) {
    const uint32_t total = a.prng_part ? 0u : (uint32_t)a.n_total * (uint32_t)HNu;   // 0 selects the partitionable layout
    const SampleParams sq = sample_params(a, HNu);
    const int first = blockIdx.x * kPkSamples;
    const int cnt = min(kPkSamples, a.n - first) * HNu;
    for (int e = tid; e < cnt; e += nthreads) {
      int ns = first + e / HNu, j = e % HNu;
      uint32_t idx = (uint32_t)(a.n_begin + ns) * (uint32_t)HNu + (uint32_t)j;
      so.Y0s()[(size_t)ns * HNu + j] = sample_elem(sq.k0, sq.k1, idx, total, sq.sigma, sq.Ybar[j]);
    }
  }
  __syncthreads();   // the duplicated table and (FUSED) this CTA's action rows are complete

  pk::Smem<pk::f2> S;
  S.X = tab + MBD_BLOB_WORDS;
  S.E = S.X + L * pk::kXF * pk::kLanes;
  S.lane = lane;
  pk::Cfg c;   // topology through the parameter bank: uniform registers, uniform branches
  c.l = l; c.ndof = a.cfg[l].ndof; c.parent = a.cfg[l].parent; c.ncon = a.cfg[l].ncon;
#pragma unroll
  for (int k = 0; k < MBD_MAXCHILD; ++k) c.child[k] = a.cfg[l].child[k];

  // lane holds samples 2*lane (low half) and 2*lane + 1 (high half) of the CTA
  const int n0 = blockIdx.x * kPkSamples + 2 * lane;
  const bool act0 = n0 < a.n, act1 = n0 + 1 < a.n;
  const int r0 = act0 ? n0 : a.n - 1, r1 = act1 ? n0 + 1 : a.n - 1;

  pk::State<pk::f2> s;
  {
    const float* st = so.state_init() + l * MBD_STATE_STRIDE;
    auto b = [&](int i) { return pk::mk2(st[i], st[i]); };
    s.p = pk::mkV(b(0), b(1), b(2));
    s.q = pk::mkQ(b(3), b(4), b(5), b(6));
    s.w = pk::mkV(b(7), b(8), b(9));
    s.v = pk::mkV(b(10), b(11), b(12));
  }
  S.put_p(l, s.p); S.put_q(l, s.q); S.put_w(l, s.w);
  typename std::conditional<SYNC == 2, SyncNamedFenced, SyncGroup<kPkLinks>>::type Y;
  if constexpr (SYNC == 2) Y.setup(Ms, l, L);
  else { Y.base = 1; Y.count_x = a.count_x; }
  int my_track = -1;
  for (int k = 0; k < ntrack; ++k)
    if (M.hi(MBD_H_TRACK0 + k) == l) my_track = k;
  __syncthreads();
  if constexpr (SYNC == 2) Y.arrive_pose(l);  // the initial pose is published
  float rsum0 = 0.0f, rsum1 = 0.0f, tacc0 = 0.0f, tacc1 = 0.0f;
  const float* urow0 = so.Y0s() + (size_t)r0 * HNu;
  const float* urow1 = so.Y0s() + (size_t)r1 * HNu;
  for (int t = 0; t < a.H; ++t) {
    pk::f2 tau[MBD_MAXDOF];
#pragma unroll
    for (int k = 0; k < MBD_MAXDOF; ++k) {
      const int base = MBD_F_DOF0 + k * MBD_DOF_STRIDE;
      const int ak = k < c.ndof ? M.li(base + MBD_D_ACT, l) : -1;
      tau[k] = pk::mk2(0.0f, 0.0f);
      if (ak >= 0) {
        pk::f2 u = pk::mk2(urow0[t * nu + ak], urow1[t * nu + ak]);
        tau[k] = pk::mul(M.l(base + MBD_D_GEAR, l), pk::clamp_(u, M.l(base + MBD_D_CLO, l), M.l(base + MBD_D_CHI, l)));
      }
    }
    float rp0 = 0.0f, rp1 = 0.0f;
    if (reward_kind == MBD_REWARD_HUMANOIDTRACK && l == 0) {
      pk::V<pk::f2> x0 = pk::link_origin_w(M, 0, s), v0 = pk::link_origin_vel_w(M, 0, s);
      v3 xa = pk_lo(x0), xb = pk_hi(x0), va = pk_lo(v0), vb = pk_hi(v0);
      rp0 = 1.0f + ((-fabsf(va.x - 1.6f) - fabsf(xa.z - 1.3f)) - fabsf(xa.y) * 0.1f);
      rp1 = 1.0f + ((-fabsf(vb.x - 1.6f) - fabsf(xb.z - 1.3f)) - fabsf(xb.y) * 0.1f);
    }
    if (reward_kind == MBD_REWARD_ANT && l == 0) {   // root x before the step
      pk::V<pk::f2> x0 = pk::link_origin_w(M, 0, s);
      rp0 = pk::lo(x0.x); rp1 = pk::hi(x0.x);
    }
    for (int f = 0; f < nsub; ++f) positional_step_pk<CMAX>(M, c, S, Y, s, tau);
    if (l == 0) {
      float ra = rp0, rb = rp1;
      if (reward_kind == MBD_REWARD_ANT) {
        pk::V<pk::f2> x0 = pk::link_origin_w(M, 0, s);
        ra = reward_ant(Ms, rp0, pk::lo(x0.x), urow0 + t * nu, nu);
        rb = reward_ant(Ms, rp1, pk::hi(x0.x), urow1 + t * nu, nu);
      } else if (reward_kind != MBD_REWARD_HUMANOIDTRACK) {
        pk::V<pk::f2> x0 = pk::link_origin_w(M, 0, s);
        ra = reward_post(reward_kind, pk_lo(x0));
        rb = reward_post(reward_kind, pk_hi(x0));
      }
      rsum0 += ra; rsum1 += rb;
      if (a.rewss) {
        if (act0) a.rewss[(size_t)n0 * a.H + t] = ra;
        if (act1) a.rewss[(size_t)(n0 + 1) * a.H + t] = rb;
      }
    }
    if (my_track >= 0) {
      pk::V<pk::f2> xx = pk::link_origin_w(M, l, s);
      const v3 xs[2] = {pk_lo(xx), pk_hi(xx)};
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const v3 x = xs[i];
        if (a.track_pos && (i == 0 ? act0 : act1)) {
          float* o = a.track_pos + (((size_t)(n0 + i) * a.H + t) * ntrack + my_track) * 3;
          o[0] = x.x; o[1] = x.y; o[2] = x.z;
        }
        if (a.xref) {
          int tt = t < a.href ? t : a.href - 1;
          const float* xr = a.xref + ((size_t)my_track * a.href + tt) * 3;
          v3 d = V3(x.x - xr[0], x.y - xr[1], x.z - xr[2]);
          float nr = sqrtf(vdot(d, d));
          float cl = nr < 0.5f ? nr : 0.5f;
          float q = cl / 0.5f;
          if (i == 0) tacc0 = fmaf(q, q, tacc0); else tacc1 = fmaf(q, q, tacc1);
        }
      }
    }
  }
  if (l == 0) {
    if (act0) so.rews()[n0] = rsum0 / (float)a.H;
    if (act1) so.rews()[n0 + 1] = rsum1 / (float)a.H;
  }
  if (a.logpd && a.xref) {
    float* Ef = reinterpret_cast<float*>(S.E);   // per-body accumulators -> shared (reuse E), summed in track order by warp 0
    __syncthreads();
    if (my_track >= 0) { Ef[my_track * kPkSamples + 2 * lane] = tacc0; Ef[my_track * kPkSamples + 2 * lane + 1] = tacc1; }
    __syncthreads();
    if (l == 0) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        float tot = 0.0f;
        for (int k = 0; k < ntrack; ++k) tot += Ef[k * kPkSamples + 2 * lane + i];
        if (i == 0 ? act0 : act1) so.logpd()[n0 + i] = 0.0f - tot / (float)(ntrack * a.H);
      }
    }
  }
  if (a.final_state) {
    const pk::f2 f[13] = {s.p.x, s.p.y, s.p.z, s.q.w, s.q.x, s.q.y, s.q.z, s.w.x, s.w.y, s.w.z, s.v.x, s.v.y, s.v.z};
    if (act0) {
      float* o = a.final_state + ((size_t)n0 * L + l) * MBD_STATE_STRIDE;
#pragma unroll
      for (int j = 0; j < 13; ++j) o[j] = pk::lo(f[j]);
    }
    if (act1) {
      float* o = a.final_state + ((size_t)(n0 + 1) * L + l) * MBD_STATE_STRIDE;
#pragma unroll
      for (int j = 0; j < 13; ++j) o[j] = pk::hi(f[j]);
    }
  }
}

// ---- car2d (/root/reference/mbd/envs/car2d.py) ---------------------------------------------------------
constexpr int kCarObs = 11;
__device__ __forceinline__ void car_dynamics(const float* x, const float* u, float* o) {
  float s, c;
  mbd_sincosf(x[2], &s, &c);
  o[0] = u[1] * s * 3.0f;
  o[1] = u[1] * c * 3.0f;
  o[2] = u[0] * 3.14159274101257324f / 3.0f * 2.0f;
}
struct CarArgs {
  const float* params; const float* x0; float* Y0s; int n, H;
  float* rewss; float* rews; const float* xref; int href; float* logpd; float* traj;
  int fused; uint32_t k0, k1; int n_total, n_begin; float sigma; const float* Ybar;
  const mbd_step_params* sp; const mbd_step_ctl* ctl; const float* Ybars;   // device-resident step parameters (see RolloutArgs)
  int prng_part;
  SolveStride ss;          // batched step: per-solve strides (zero otherwise)
};
template <bool BATCH = false>   // BATCH: blockIdx.y is the solve of a batched step
__global__ void k_car2d(CarArgs a) {
  __shared__ float sp[2 * kCarObs + 4];
  if constexpr (BATCH) solve_offsets(a.ss, a.x0, a.Y0s, a.rews, a.logpd, a.sp, a.ctl, a.Ybars);
  if (threadIdx.x < 2 * kCarObs + 4) sp[threadIdx.x] = a.params[threadIdx.x];
  __syncthreads();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const float orad = sp[2 * kCarObs], dt = sp[2 * kCarObs + 1], hdt = sp[2 * kCarObs + 2], sdt = sp[2 * kCarObs + 3];
  const int HNu = a.H * 2;
  const uint32_t total = a.prng_part ? 0u : (uint32_t)a.n_total * (uint32_t)HNu;   // 0 selects the partitionable layout
  uint32_t ck0 = a.k0, ck1 = a.k1; float csigma = a.sigma; const float* cYbar = a.Ybar;
  if (a.sp != nullptr) {
    const int si = a.ctl->i;
    ck0 = a.sp[si].key[0]; ck1 = a.sp[si].key[1]; csigma = a.sp[si].sigma; cYbar = a.Ybars + (size_t)si * HNu;
  }
  float q[3] = {a.x0[0], a.x0[1], a.x0[2]};
  float sum = 0.0f, acc = 0.0f;
  for (int t = 0; t < a.H; ++t) {
    float* ur = a.Y0s + ((size_t)i * a.H + t) * 2;
    float u0, u1;
    if (a.fused) {
      uint32_t idx = (uint32_t)(a.n_begin + i) * (uint32_t)HNu + (uint32_t)(2 * t);
      u0 = sample_elem(ck0, ck1, idx, total, csigma, cYbar[2 * t]);
      u1 = sample_elem(ck0, ck1, idx + 1, total, csigma, cYbar[2 * t + 1]);
      ur[0] = u0; ur[1] = u1;
    } else {
      u0 = ur[0]; u1 = ur[1];
    }
    float u[2] = {clampf(u0, -1.0f, 1.0f), clampf(u1, -1.0f, 1.0f)};
    float k1[3], k2[3], k3[3], k4[3], y[3], qn[3];
    car_dynamics(q, u, k1);
    for (int d = 0; d < 3; ++d) y[d] = q[d] + hdt * k1[d];
    car_dynamics(y, u, k2);
    for (int d = 0; d < 3; ++d) y[d] = q[d] + hdt * k2[d];
    car_dynamics(y, u, k3);
    for (int d = 0; d < 3; ++d) y[d] = q[d] + dt * k3[d];
    car_dynamics(y, u, k4);
    for (int d = 0; d < 3; ++d) qn[d] = q[d] + sdt * (((k1[d] + 2.0f * k2[d]) + 2.0f * k3[d]) + k4[d]);
    bool collide = false;
    for (int k = 0; k < kCarObs; ++k) {
      float dx = qn[0] - sp[2 * k], dy = qn[1] - sp[2 * k + 1];
      if (sqrtf(dx * dx + dy * dy) < orad) collide = true;
    }
    if (!collide) { q[0] = qn[0]; q[1] = qn[1]; q[2] = qn[2]; }
    float dx = q[0] - 0.5f, dy = q[1] - 0.0f;
    float d = sqrtf(dx * dx + dy * dy);
    float cc = clampf(d, 0.0f, 0.2f) / 0.2f;
    float r = 1.0f - cc * cc;
    if (a.rewss) a.rewss[(size_t)i * a.H + t] = r;
    sum += r;
    if (a.traj) { float* o = a.traj + ((size_t)i * a.H + t) * 3; o[0] = q[0]; o[1] = q[1]; o[2] = q[2]; }
    if (a.xref) {
      int tt = t < a.href ? t : a.href - 1;
      float ex = q[0] - a.xref[2 * tt], ey = q[1] - a.xref[2 * tt + 1];
      float dd = sqrtf(ex * ex + ey * ey);
      float c2 = clampf(dd, 0.0f, 0.5f) / 0.5f;
      acc += c2 * c2;
    }
  }
  a.rews[i] = sum / (float)a.H;
  if (a.logpd && a.xref) a.logpd[i] = 0.0f - acc / (float)a.H;
}

}  // namespace mbd
#include "pusht.cuh"   // k_pusht: the pushT env (planar generalized pipeline), uses sample_elem / clampf from above
namespace mbd {

// ---- test hook: the exact div / rcp / sqrt device sequences on arrays (tests/test_rollout_gpu.py) ----------
__global__ void k_test_arith(int op, const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ o, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (op == 0) o[i] = MBD_DIV(a[i], b[i]);
  else if (op == 1) o[i] = MBD_RCP(a[i]);
  else if (op == 2) o[i] = MBD_SQRT(a[i]);
  else o[i] = mbd_atan2f(a[i], b[i]);
}

// ---- reward statistics + softmax (mbd_planner.py:110-127), single CTA ------------------------------------
constexpr int kStatThreads = 1024;
enum { OP_SUM = 0, OP_MAX = 1 };

template <int OP>
__device__ __forceinline__ float block_reduce(float v, float* sh) {
  // deterministic: butterfly inside the warp, then warp 0 over the 32 warp results
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_xor_sync(0xffffffffu, v, o);
    v = OP == OP_SUM ? v + t : fmaxf(v, t);
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = sh[threadIdx.x & 31];
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_xor_sync(0xffffffffu, r, o);
    r = OP == OP_SUM ? r + t : fmaxf(r, t);
  }
  return r;  // every thread holds the result
}

__global__ void __launch_bounds__(kStatThreads) k_softmax_weights(const float* __restrict__ rews, const float* __restrict__ logpd,
                                                                  int N, int n_begin, int n_local, float temp, float rew_xref,
                                                                  float* __restrict__ weights, float* __restrict__ scalars,
                                                                  float* __restrict__ logp_scratch) {
  __shared__ float sh[32];
  const int tid = threadIdx.x;
  const float fN = (float)N;
  float acc = 0.0f;
  for (int i = tid; i < N; i += kStatThreads) acc += rews[i];
  const float rew_mean = block_reduce<OP_SUM>(acc, sh) / fN;
  acc = 0.0f;
  for (int i = tid; i < N; i += kStatThreads) { float d = rews[i] - rew_mean; acc = fmaf(d, d, acc); }
  float rew_std = sqrtf(block_reduce<OP_SUM>(acc, sh) / fN);  // population std (ddof 0)
  rew_std = rew_std < 1e-4f ? 1.0f : rew_std;
  float* logp = logp_scratch;  // [N]
  if (logpd != nullptr) {
    float mx = -INFINITY;
    for (int i = tid; i < N; i += kStatThreads) mx = fmaxf(mx, logpd[i]);
    mx = block_reduce<OP_MAX>(mx, sh);
    acc = 0.0f;
    for (int i = tid; i < N; i += kStatThreads) {
      float l0 = (rews[i] - rew_mean) / rew_std / temp;
      float ld = ((logpd[i] - mx) + rew_xref - rew_mean) / rew_std / temp;
      float l = ld > l0 ? ld : l0;
      logp[i] = l;
      acc += l;
    }
    const float lmean = block_reduce<OP_SUM>(acc, sh) / fN;
    acc = 0.0f;
    for (int i = tid; i < N; i += kStatThreads) { float d = logp[i] - lmean; acc = fmaf(d, d, acc); }
    const float lstd = sqrtf(block_reduce<OP_SUM>(acc, sh) / fN);
    for (int i = tid; i < N; i += kStatThreads) logp[i] = (logp[i] - lmean) / lstd / temp;
  } else {
    for (int i = tid; i < N; i += kStatThreads) logp[i] = (rews[i] - rew_mean) / rew_std / temp;
  }
  __syncthreads();
  float mx = -INFINITY;
  for (int i = tid; i < N; i += kStatThreads) mx = fmaxf(mx, logp[i]);
  mx = block_reduce<OP_MAX>(mx, sh);
  acc = 0.0f;
  for (int i = tid; i < N; i += kStatThreads) acc += mbd_expf(logp[i] - mx);
  const float S = block_reduce<OP_SUM>(acc, sh);
  for (int i = tid; i < n_local; i += kStatThreads) weights[i] = mbd_expf(logp[n_begin + i] - mx) / S;
  if (tid == 0) { scalars[0] = rew_mean; scalars[1] = rew_std; scalars[2] = mx; scalars[3] = S; }
}

// ---- weighted mean, deterministic order -----------------------------------------------------------------------
// run r covers samples [r*kRun, (r+1)*kRun): out[r][j] = sum_n w[n]*Y[n][j] sequentially (fmaf)
// SQERR: accumulate w[n] * (Y[n][j] - mu[j])^2 instead (CMA-ES sigma update, path_integral.py:39-45)
template <bool SQERR>
__global__ void k_wsum_runs(const float* __restrict__ w, const float* __restrict__ Y, const float* __restrict__ mu, int n_local, int HNu,
                            float* __restrict__ runs) {
  int j = blockIdx.y * blockDim.x + threadIdx.x;
  int r = blockIdx.x;
  if (j >= HNu) return;
  int n0 = r * kRun, n1 = min(n0 + kRun, n_local);
  const float m = SQERR ? mu[j] : 0.0f;
  auto term = [&](int n) { float y = Y[(size_t)n * HNu + j]; if (SQERR) { float d = y - m; return d * d; } return y; };
  float acc = w[n0] * term(n0);
  for (int n = n0 + 1; n < n1; ++n) acc = fmaf(w[n], term(n), acc);
  runs[(size_t)r * HNu + j] = acc;
}
// pairwise (adjacent) tree over `count` rows of [count][stride] -> value for column j; binary-counter
// stack.  Aligned blocks of 8 rows are loaded together (8 loads in flight) and folded in registers in the
// same adjacent-pair order, then pushed at level 3 — identical association, 8x fewer serialized loads.
__device__ __forceinline__ float tree_sum_rows(const float* __restrict__ rows, int count, int stride, int j) {
  float stack[32];
  int depth = 0;
  int r = 0;
  for (; r + 8 <= count; r += 8) {
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = rows[(size_t)(r + k) * stride + j];
    float b = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
    int rr = r >> 3;
    while (rr & 1) { b = stack[--depth] + b; rr >>= 1; }
    stack[depth++] = b;
  }
  if (r < count) {
    // ragged tail (< 8 rows): plain binary counter over single rows, then merged as ONE block below
    float tstack[4];
    int td = 0;
    for (int q = 0; r + q < count; ++q) {
      float v = rows[(size_t)(r + q) * stride + j];
      int rr = q;
      while (rr & 1) { v = tstack[--td] + v; rr >>= 1; }
      tstack[td++] = v;
    }
    float v = tstack[--td];
    while (td > 0) v = tstack[--td] + v;
    stack[depth++] = v;
  }
  float v = stack[--depth];
  while (depth > 0) v = stack[--depth] + v;
  return v;
}
__global__ void k_wsum_tree(const float* __restrict__ runs, int nruns, int HNu, float* __restrict__ out) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= HNu) return;
  out[j] = tree_sum_rows(runs, nruns, HNu, j);
}
__global__ void k_update(const float* __restrict__ partials, int P, int HNu, const float* __restrict__ Ybar_i, float c_sqrt_ab,
                         float c_inv_1mab, float c_1mab, float c_inv_sqrt_a, float c_sqrt_abm1, float* __restrict__ out) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= HNu) return;
  float Ybar = tree_sum_rows(partials, P, HNu, j);
  // mbd_planner.py:100,130-133 literally
  float Yi = Ybar_i[j] * c_sqrt_ab;
  float score = c_inv_1mab * (-Yi + c_sqrt_ab * Ybar);
  float Yim1 = c_inv_sqrt_a * (Yi + c_1mab * score);
  out[j] = Yim1 / c_sqrt_abm1;
}



// ---- ONE kernel per diffusion step (single GPU, no demo): rollouts + statistics + weighted mean + update ------
// reverse_once (mbd_planner.py:97-135) as a single cooperative launch: the rollout body above, a grid barrier,
// then every CTA recomputes the global reward statistics redundantly (so no broadcast barrier is needed),
// CTA r reduces run r of the weighted mean, a second grid barrier, and the first CTAs finish the pairwise tree
// and the update.  The arithmetic replays k_softmax_weights / k_wsum_runs / k_wsum_tree / k_update exactly
// (the 1024-thread strided partial sums + butterfly of k_softmax_weights are emulated with 1024 virtual threads and
// an adjacent-pairwise shared-memory tree, which is the same association), so the fused step is bit-identical
// to the multi-kernel path.
struct StepTail {
  float temp;
  const float* Ybar_i;  // [HNu]
  float c0, c1, c2, c3, c4;
  float* weights;       // [n]
  float* scalars;       // [4]
  float* runs;          // [ceil(n/64)][HNu]
  float* out;           // [HNu]
};

template <int OP, class F>
__device__ __forceinline__ float vreduce1024(float* vp, int N, F term) {
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int v = tid; v < kStatThreads; v += nt) {
    float acc = OP == OP_SUM ? 0.0f : -INFINITY;
    for (int i = v; i < N; i += kStatThreads) acc = term(acc, i);
    vp[v] = acc;
  }
  __syncthreads();
  for (int o = 1; o < kStatThreads; o <<= 1) {
    for (int v = tid; v < kStatThreads; v += nt)
      if ((v & (2 * o - 1)) == 0) vp[v] = OP == OP_SUM ? vp[v] + vp[v + o] : fmaxf(vp[v], vp[v + o]);
    __syncthreads();
  }
  float r = vp[0];
  __syncthreads();
  return r;
}

template <int NWARPS, int MINB, int CMAX>
__global__ void __launch_bounds__(32 * NWARPS, MINB) k_reverse_step_wpl(RolloutArgs a, StepTail t) {
  __shared__ __align__(128) float sblob[MBD_BLOB_WORDS];
  __shared__ __align__(8) uint64_t mbar;
  __shared__ __align__(8) uint64_t edge_bars[2 * MBD_MAXL];
  __shared__ float vp[kStatThreads];
  __shared__ float wrun[kRun];
  extern __shared__ __align__(16) float dyn[];
  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  rollout_wpl_body<true, 0, 1, CMAX>(a, sblob, &mbar, edge_bars, dyn);
  __threadfence();
  grid.sync();
  // ---- mbd_planner.py:110-127 (k_softmax_weights replayed) ------------------------------------------------
  const int N = a.n, tid = threadIdx.x, nt = blockDim.x;
  const int HNu = a.H * reinterpret_cast<const int*>(sblob)[MBD_H_NU];
  const float* rews = a.rews;
  const float fN = (float)N;
  const float rew_mean = vreduce1024<OP_SUM>(vp, N, [&](float acc, int i) { return acc + rews[i]; }) / fN;
  float rew_std = sqrtf(vreduce1024<OP_SUM>(vp, N, [&](float acc, int i) { float d = rews[i] - rew_mean; return fmaf(d, d, acc); }) / fN);
  rew_std = rew_std < 1e-4f ? 1.0f : rew_std;
  auto logp = [&](int i) { return (rews[i] - rew_mean) / rew_std / t.temp; };
  const float mx = vreduce1024<OP_MAX>(vp, N, [&](float acc, int i) { return fmaxf(acc, logp(i)); });
  const float S = vreduce1024<OP_SUM>(vp, N, [&](float acc, int i) { return acc + mbd_expf(logp(i) - mx); });
  if (blockIdx.x == 0 && tid == 0) { t.scalars[0] = rew_mean; t.scalars[1] = rew_std; t.scalars[2] = mx; t.scalars[3] = S; }
  // ---- mbd_planner.py:128, run r = this CTA (k_wsum_runs replayed) ------------------------------------------------
  const int nruns = (N + kRun - 1) / kRun;
  if ((int)blockIdx.x < nruns) {
    const int n0 = blockIdx.x * kRun, n1 = min(n0 + kRun, N);
    if (tid < n1 - n0) {
      float w = mbd_expf(logp(n0 + tid) - mx) / S;
      wrun[tid] = w;
      t.weights[n0 + tid] = w;
    }
    __syncthreads();
    for (int j = tid; j < HNu; j += nt) {
      float acc = wrun[0] * a.Y0s[(size_t)n0 * HNu + j];
      for (int n = n0 + 1; n < n1; ++n) acc = fmaf(wrun[n - n0], a.Y0s[(size_t)n * HNu + j], acc);
      t.runs[(size_t)blockIdx.x * HNu + j] = acc;
    }
  }
  __threadfence();
  grid.sync();
  // ---- pairwise tree over the runs + mbd_planner.py:100,130-133 (k_wsum_tree, k_update replayed) ----------------
  const int j = blockIdx.x * nt + tid;
  if (j < HNu) {
    float Ybar = tree_sum_rows(t.runs, nruns, HNu, j);
    float Yi = t.Ybar_i[j] * t.c0;
    float score = t.c1 * (-Yi + t.c0 * Ybar);
    float Yim1 = t.c3 * (Yi + t.c2 * score);
    t.out[j] = Yim1 / t.c4;
  }
}

// ---- fused cross-GPU exchange over NVLink peer memory ----------------------------------------------------
// Replaces NCCL all_gather for the two tiny per-step exchanges (per-sample returns, rank partials):
// every rank owns a symmetric buffer (torch symmetric memory: peer-mapped, same layout on all ranks).
// One kernel = in-kernel barrier (system-scope release/acquire on per-peer flag words) + direct peer loads:
//   1. CTA 0 publishes `epoch` into slot [rank] of every peer's flag row        (st.release.sys)
//   2. every CTA waits until its own flag row shows `epoch` from all P peers     (ld.acquire.sys)
//   3. dst[r][j] = peer_r[src_off + j] for all ranks r                           (ld.global.cv over NVLink)
// Stream order guarantees the producer kernel of the data finished before step 1 runs on each rank.
struct PeerArgs {
  float* peer[8];
  int P, rank, count;
  unsigned long long src_off, flag_off;  // in 4-byte words from the buffer base
  unsigned int epoch;
  float* dst;        // [P*count] local
  unsigned int* err; // local error word (set to 1 on a barrier timeout instead of hanging the GPU)
};

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__global__ void k_peer_gather(PeerArgs a) {
  if (blockIdx.x == 0 && threadIdx.x < a.P) {
    __threadfence_system();
    st_release_sys(reinterpret_cast<unsigned int*>(a.peer[threadIdx.x]) + a.flag_off + a.rank, a.epoch);
  }
  if (threadIdx.x < a.P) {
    const unsigned int* f = reinterpret_cast<const unsigned int*>(a.peer[a.rank]) + a.flag_off + threadIdx.x;
    long long t0 = clock64();
    while (ld_acquire_sys(f) < a.epoch) {
      if (clock64() - t0 > 4000000000LL) { *a.err = 1u; break; }  // ~2 s: never hang the device
    }
  }
  __syncthreads();
  const int total = a.P * a.count;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int r = i / a.count, j = i - r * a.count;
    a.dst[i] = __ldcv(a.peer[r] + a.src_off + j);
  }
}

}  // namespace mbd

// =====================================================================================================
// C ABI
// =====================================================================================================
struct mbd_model {
  int device;           // the device the blob lives on: launches on another current device are refused
  uint32_t* blob_dev;
  int L, nu, n_frames, ntrack, max_ncon;
  // v2 kernel mappings (host side): one link per warp, and two same-type links per warp
  signed char wl1[MBD_MAXL][2], wl2[MBD_MAXL][2], wl6[MBD_MAXL][2];
  unsigned long long offs1, offs2;
  int nwarps2;
  signed char gw2[32];  // two-group CTA: warp -> (group << 4) | slot
  int nlate;            // jointed leaf links with contacts (SyncGroup's late leaves)
  bool named_ok;        // SyncNamed needs two hardware barrier ids (1..15) per link that has children: at most 7 such links
  bool pk_ok;           // the packed kernel (xpbd_pk.cuh) covers this model: 11 links, hinge dofs only, a reward it implements
  mbd::RolloutArgs::LinkCfgP cfg[MBD_MAXL];   // warp-uniform topology handed to the kernels through the parameter bank
};

// Pairs links with the same (ndof, #contacts, has-children) signature so that the two halves of a warp run
// the same code path (right/left limbs); leftovers are paired jointed-with-jointed, the root stays alone.
static void build_pairing(mbd_model* m, const uint32_t* blob) {
  const int32_t* bi = reinterpret_cast<const int32_t*>(blob);
  auto li = [&](int f, int l) { return bi[MBD_HDR_WORDS + f * MBD_MAXL + l]; };
  const int L = m->L;
  int sig[MBD_MAXL];
  bool used[MBD_MAXL] = {false};
  for (int l = 0; l < L; ++l) sig[l] = li(MBD_F_NDOF, l) * 64 + li(MBD_F_NCON, l) * 4 + (li(MBD_F_CHILD0, l) >= 0 ? 1 : 0);
  m->offs1 = 0; m->offs2 = 0; m->nwarps2 = 0;
  m->nlate = 0;
  for (int l = 0; l < MBD_MAXL; ++l) {
    const bool live = l < L;
    m->cfg[l].ndof = (signed char)(live ? li(MBD_F_NDOF, l) : -1);
    m->cfg[l].parent = (signed char)(live ? li(MBD_F_PARENT, l) : -1);
    m->cfg[l].ncon = (signed char)(live ? li(MBD_F_NCON, l) : 0);
    m->cfg[l].smask = (signed char)((live && li(MBD_F_NDOF, l) > 0) ? li(MBD_F_SLIDE, l) : 0);
    for (int k = 0; k < MBD_MAXCHILD; ++k) m->cfg[l].child[k] = (signed char)(live ? li(MBD_F_CHILD0 + k, l) : -1);
  }
  // must be the predicate SyncGroup::end_D uses (leaf && contacts; a single-link free body with contacts counts too)
  for (int l = 0; l < L; ++l) m->nlate += (li(MBD_F_CHILD0, l) < 0 && li(MBD_F_NCON, l) > 0) ? 1 : 0;
  // two-group CTA: warp w -> (group, slot).  Both groups sit on ALL FOUR SM sub-partition schedulers (group = bit 0 xor bit 2
  // of the warp id) and group 1 starts ~half a substep late (g_group_stagger): the two groups then demand the fp32 pipe in
  // different phases.  Measured on humanoidrun 8192 x 50 (scripts/gpu_stagger_sweep.py, profiles/r02_experiments.md):
  // dedicated scheduler pairs 1.386 ms; shared schedulers in lockstep 1.408 ms; shared + 3500..5000 cycles offset 1.353-1.358 ms.
  for (int w = 0; w < 32; ++w) m->gw2[w] = (signed char)((((w ^ (w >> 2)) & 1) << 4) | ((w >> 1) & 15));
  for (int l = 0; l < MBD_MAXL; ++l) { m->wl1[l][0] = (signed char)(l < L ? l : 0); m->wl1[l][1] = m->wl1[l][0]; m->wl2[l][0] = m->wl2[l][1] = 0; }
  {
    // One link per warp: warps are issued by SM sub-partition (warp id % 4).  Spread the joint work
    // (weight ~ ndof) evenly over the four schedulers and keep links with contacts on different ones
    // (longest-processing-time greedy; slot s of scheduler q is warp 4*s + q).
    int order[MBD_MAXL], nslot[4] = {0, 0, 0, 0};
    float load[4] = {0, 0, 0, 0}, conload[4] = {0, 0, 0, 0};
    int cap[4];
    for (int q = 0; q < 4; ++q) cap[q] = (L - q + 3) / 4;
    auto weight = [&](int l) { int nd = li(MBD_F_NDOF, l); return nd <= 0 ? 0.0f : (nd == 1 ? 0.6f : (nd == 2 ? 0.93f : 1.0f)); };
    for (int l = 0; l < L; ++l) order[l] = l;
    for (int i = 0; i < L; ++i)       // sort: contacts first, then by weight, descending (stable)
      for (int j = i + 1; j < L; ++j) {
        float wi = weight(order[i]) + 10.0f * li(MBD_F_NCON, order[i]), wj = weight(order[j]) + 10.0f * li(MBD_F_NCON, order[j]);
        if (wj > wi) { int t = order[i]; order[i] = order[j]; order[j] = t; }
      }
    for (int i = 0; i < L; ++i) {
      int l = order[i], best = -1;
      for (int q = 0; q < 4; ++q) {
        if (nslot[q] >= cap[q]) continue;
        float cost = load[q] + 100.0f * (li(MBD_F_NCON, l) > 0 ? conload[q] : 0.0f);
        if (best < 0 || cost < load[best] + 100.0f * (li(MBD_F_NCON, l) > 0 ? conload[best] : 0.0f)) best = q;
      }
      // the SM arbiter favours the highest warp id among eligible warps (B300_MICROARCH.md): the critical
      // links (assigned first) take the highest slot of their scheduler
      int w = 4 * (cap[best] - 1 - nslot[best]) + best;
      m->wl1[w][0] = m->wl1[w][1] = (signed char)l;
      nslot[best]++; load[best] += weight(l); conload[best] += li(MBD_F_NCON, l) > 0 ? 1.0f : 0.0f;
    }
  }
  {
    // Two-group CTA (SyncGroup): the leaves with contacts are decoupled from the end-of-substep barrier, their long
    // contact phase overlaps everybody else's torque phase — they take the LOWEST warp ids so that they do not steal
    // issue slots from it; the links above them (the chain that waits for their terms) take the highest.
    // Order: late leaves, root, other leaves, links that are no ancestor of a late leaf, ancestors by depth.
    bool late[MBD_MAXL], anc[MBD_MAXL] = {false}, leaf[MBD_MAXL];
    int depth[MBD_MAXL];
    for (int l = 0; l < L; ++l) {
      leaf[l] = li(MBD_F_CHILD0, l) < 0;
      late[l] = leaf[l] && li(MBD_F_NCON, l) > 0 && li(MBD_F_NDOF, l) > 0;
      depth[l] = 0;
      for (int p = li(MBD_F_PARENT, l); p >= 0; p = li(MBD_F_PARENT, p)) ++depth[l];
    }
    for (int l = 0; l < L; ++l)
      if (late[l]) for (int p = li(MBD_F_PARENT, l); p >= 0; p = li(MBD_F_PARENT, p)) anc[p] = true;
    auto rank = [&](int l) { return late[l] ? 0 : (li(MBD_F_NDOF, l) == 0 ? 1 : (leaf[l] ? 2 : (!anc[l] ? 3 : 4 + depth[l]))); };
    int order[MBD_MAXL];
    for (int l = 0; l < L; ++l) order[l] = l;
    for (int i = 0; i < L; ++i)
      for (int j = i + 1; j < L; ++j)
        if (rank(order[j]) < rank(order[i])) { int t = order[i]; order[i] = order[j]; order[j] = t; }   // stable: ties keep link order
    for (int w = 0; w < MBD_MAXL; ++w) m->wl6[w][0] = m->wl6[w][1] = (signed char)(w < L ? order[w] : 0);
  }
  auto add_pair = [&](int a, int b) {
    int w = m->nwarps2++;
    m->wl2[w][0] = (signed char)a;
    m->wl2[w][1] = (signed char)(b >= 0 ? b : a);
    if (b >= 0) m->offs2 |= (unsigned long long)(16 >> 2) << (4 * b);
    used[a] = true;
    if (b >= 0) used[b] = true;
  };
  for (int a = 0; a < L; ++a) {
    if (used[a]) continue;
    for (int b = a + 1; b < L; ++b)
      if (!used[b] && sig[b] == sig[a]) { add_pair(a, b); break; }
  }
  int prev = -1;
  for (int a = 0; a < L; ++a) {  // leftovers: jointed with jointed
    if (used[a] || li(MBD_F_NDOF, a) <= 0) continue;
    if (prev < 0) prev = a; else { add_pair(prev, a); prev = -1; }
  }
  if (prev >= 0) add_pair(prev, -1);
  for (int a = 0; a < L; ++a)
    if (!used[a]) add_pair(a, -1);
}

static int g_group_stagger = 4000;   // cycles group 1 of a two-group CTA waits before its first step (see build_pairing)
static int g_prng_part = 0;       // threefry layout of the samplers: 0 legacy, 1 partitionable (mbd_set_prng_layout)
static int g_kernel_variant = 0;  // 0 = auto, 1 = v1 (lane per link), 2..4 = v2 (warp per link; CTA / named / mbarrier sync)
static thread_local char g_err[256] = "";
static int set_err(const char* where, cudaError_t e) {
  snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
  return MBD_ECUDA;
}
#define CK(call)                                  \
  do {                                            \
    cudaError_t e_ = (call);                      \
    if (e_ != cudaSuccess) return set_err(#call, e_); \
  } while (0)

extern "C" {

const char* mbd_last_error(void) { return g_err; }

int mbd_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int mbd_set_prng_layout(int partitionable) {
  g_prng_part = partitionable ? 1 : 0;
  return MBD_OK;
}

int mbd_set_kernel_variant(int v) {
  if (v < 0 || v > 9 || v == 7 || v == 4) return MBD_EINVAL;   // 4 (mbarrier polling) and 10 / 11 (neighbourhood barriers) were removed in round 2
  g_kernel_variant = v;
  return MBD_OK;
}

// experiment hook: override the slot -> link order of the one-link-per-warp mapping (slot L-1 = highest warp id)
int mbd_model_set_warp_order(mbd_model* m, const int* order, int n) {
  if (!m || !order || n != m->L) return MBD_EINVAL;
  for (int w = 0; w < n; ++w) { if (order[w] < 0 || order[w] >= n) return MBD_EINVAL; m->wl1[w][0] = m->wl1[w][1] = m->wl6[w][0] = m->wl6[w][1] = (signed char)order[w]; }
  return MBD_OK;
}

// experiment hook: warp -> (group, slot) table of the two-group CTA; map[w] = (group << 4) | slot
int mbd_model_set_group_map(mbd_model* m, const int* map, int n) {
  if (!m || !map || n != 2 * m->L || n > 32) return MBD_EINVAL;
  int seen[2][MBD_MAXL] = {{0}};
  for (int w = 0; w < n; ++w) {
    int g = map[w] >> 4, sl = map[w] & 15;
    if (g < 0 || g > 1 || sl >= m->L || seen[g][sl]) return MBD_EINVAL;
    seen[g][sl] = 1;
  }
  for (int w = 0; w < n; ++w) m->gw2[w] = (signed char)map[w];
  return MBD_OK;
}

int mbd_set_group_stagger(int cycles) {
  if (cycles < 0) return MBD_EINVAL;
  g_group_stagger = cycles;
  return MBD_OK;
}

int mbd_layout_info(int32_t* out, int n) {
  const int32_t v[] = {(int32_t)MBD_MODEL_MAGIC, MBD_HDR_WORDS, MBD_NFIELDS, MBD_MAXL, MBD_MAXCHILD, MBD_MAXDOF, MBD_MAXCON,
                       MBD_MAXTRACK, MBD_DOF_STRIDE, MBD_CON_STRIDE, MBD_H_DT, MBD_H_RW0, MBD_F_MASS, MBD_F_COM, MBD_F_RC,
                       MBD_F_JQ, MBD_F_RP, MBD_F_PQ, MBD_F_PARITY, MBD_F_SLIDE, MBD_F_DOF0, MBD_F_NCON, MBD_F_CON0, MBD_BLOB_WORDS,
                       MBD_STATE_STRIDE};
  const int cnt = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < cnt && i < n; ++i) out[i] = v[i];
  return cnt;
}

int mbd_abi_batch_offsets(int32_t* out, int n) {
  const int32_t v[] = {(int32_t)offsetof(mbd_step_plan, n_solves), (int32_t)offsetof(mbd_step_plan, n_diffuse),
                       (int32_t)offsetof(mbd_step_plan, temps_dev)};
  const int cnt = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < cnt && i < n; ++i) out[i] = v[i];
  return cnt;
}

// sizeof / offsetof of the structs that cross the ABI by pointer (cross-checked against the ctypes mirrors in tests/test_abi.py)
int mbd_abi_sizes(int32_t* out, int n) {
  const int32_t v[] = {(int32_t)sizeof(mbd_step_params), (int32_t)sizeof(mbd_step_ctl), (int32_t)sizeof(mbd_step_plan),
                       (int32_t)offsetof(mbd_step_plan, n_total), (int32_t)offsetof(mbd_step_plan, xref_dev),
                       (int32_t)offsetof(mbd_step_plan, Y0s_dev), (int32_t)offsetof(mbd_step_plan, P),
                       (int32_t)offsetof(mbd_step_plan, peer_base_ptrs), (int32_t)offsetof(mbd_step_plan, timeout_cycles),
                       (int32_t)offsetof(mbd_step_ctl, ticket)};
  const int cnt = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < cnt && i < n; ++i) out[i] = v[i];
  return cnt;
}

mbd_model* mbd_model_create(const uint32_t* blob_host, size_t nwords) {
  if (!blob_host || nwords != MBD_BLOB_WORDS || blob_host[MBD_H_MAGIC] != MBD_MODEL_MAGIC) {
    snprintf(g_err, sizeof(g_err), "mbd_model_create: bad blob (words=%zu)", nwords);
    return nullptr;
  }
  if (mbd_device_count() <= 0) {
    snprintf(g_err, sizeof(g_err), "mbd_model_create: no CUDA device (there is no CPU fallback)");
    return nullptr;
  }
  mbd_model* m = new mbd_model();
  const int32_t* hi = reinterpret_cast<const int32_t*>(blob_host);
  m->L = hi[MBD_H_NLINK]; m->nu = hi[MBD_H_NU]; m->n_frames = hi[MBD_H_NFRAMES]; m->ntrack = hi[MBD_H_NTRACK];
  if (m->L < 1 || m->L > MBD_MAXL || m->ntrack > MBD_MAXTRACK) { delete m; snprintf(g_err, sizeof(g_err), "bad link count"); return nullptr; }
  build_pairing(m, blob_host);
  if (cudaGetDevice(&m->device) != cudaSuccess) m->device = 0;
  m->max_ncon = 0;
  for (int l = 0; l < m->L; ++l) { int nc = hi[MBD_HDR_WORDS + MBD_F_NCON * MBD_MAXL + l]; if (nc > m->max_ncon) m->max_ncon = nc; }
  if (m->max_ncon > MBD_MAXCON) { delete m; snprintf(g_err, sizeof(g_err), "too many contacts on one link"); return nullptr; }
  {
    // the packed (two samples per lane) physics has no slide-dof path and evaluates only the rewards of the free-root envs
    const int rk = hi[MBD_H_REWARD];
    bool slides = false;
    for (int l = 0; l < m->L; ++l) slides = slides || m->cfg[l].smask != 0;
    int nparents = 0;
    for (int l = 0; l < m->L; ++l) nparents += m->cfg[l].child[0] >= 0 ? 1 : 0;
    m->named_ok = 2 * nparents <= 15;
    m->pk_ok = m->L == mbd::kPkLinks && !slides &&
               (rk == MBD_REWARD_HUMANOIDRUN || rk == MBD_REWARD_HUMANOIDTRACK || rk == MBD_REWARD_HUMANOIDSTANDUP || rk == MBD_REWARD_ANT);
  }
  if (cudaMalloc(&m->blob_dev, nwords * 4) != cudaSuccess || cudaMemcpy(m->blob_dev, blob_host, nwords * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "mbd_model_create: cudaMalloc/cudaMemcpy failed");
    delete m;
    return nullptr;
  }
  return m;
}

void mbd_model_destroy(mbd_model* m) {
  if (!m) return;
  cudaFree(m->blob_dev);
  delete m;
}

int mbd_sample(const uint32_t key[2], int n_total, int n_begin, int n_local, int HNu, float sigma, const float* Ybar_dev,
               float* Y0s_dev, mbd_stream s) {
  if (!key || n_local <= 0 || HNu <= 0 || n_begin < 0 || n_begin + n_local > n_total) return MBD_EINVAL;
  if ((uint64_t)n_total * (uint64_t)HNu >= 0xffffffffull) return MBD_EINVAL;
  uint32_t count = (uint32_t)n_local * (uint32_t)HNu;
  mbd::k_sample<<<(count + 255) / 256, 256, 0, (cudaStream_t)s>>>(key[0], key[1], g_prng_part ? 0u : (uint32_t)n_total * (uint32_t)HNu,
                                                                (uint32_t)n_begin * (uint32_t)HNu, count, HNu, sigma, Ybar_dev, Y0s_dev);
  CK(cudaGetLastError());
  return MBD_OK;
}

#define MBD_LAUNCH_WPL_C(NW, MINB, SYNC, SPLIT, CMAX, GRID, THREADS)                                     \
  do {                                                                                                 \
    if (fused)                                                                                         \
      mbd::k_rollout_wpl<true, NW, MINB, SYNC, SPLIT, CMAX><<<GRID, THREADS, dyn, st>>>(a);            \
    else                                                                                               \
      mbd::k_rollout_wpl<false, NW, MINB, SYNC, SPLIT, CMAX><<<GRID, THREADS, dyn, st>>>(a);           \
  } while (0)
// contact arrays are sized by the model's worst link: 2 (humanoidrun/track) or MBD_MAXCON (humanoidstandup)
#define MBD_LAUNCH_WPL(NW, MINB, SYNC, SPLIT, GRID, THREADS)                                           \
  do {                                                                                                 \
    if (m->max_ncon <= 2) MBD_LAUNCH_WPL_C(NW, MINB, SYNC, SPLIT, 2, GRID, THREADS);                   \
    else MBD_LAUNCH_WPL_C(NW, MINB, SYNC, SPLIT, MBD_MAXCON, GRID, THREADS);                           \
  } while (0)

// cudaFuncSetAttribute and occupancy are PER DEVICE: one process may drive several GPUs (PipelineEnv.device_model caches a
// model per device), so the "already done" flags are kept per device ordinal (ADVICE r1)
static int current_device_slot() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
  return dev;
}

// S > 1: S solves of a batched step in one launch (blockIdx.y = solve, fused only); the selector sees the whole launch
static int launch_rollout(bool fused, mbd::RolloutArgs a, const mbd_model* m, cudaStream_t st, int S = 1) {
  const int L = m->L;
  {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != m->device) {
      snprintf(g_err, sizeof(g_err), "model lives on device %d but the current device is %d", m->device, dev);
      return MBD_EINVAL;
    }
  }
  memcpy(a.cfg, m->cfg, sizeof(a.cfg));
  a.prng_part = g_prng_part;
  int variant = g_kernel_variant;
  // auto (measured on humanoidrun, profiles/r02_shard_sweep.md): the step is latency-bound below one 32-sample CTA per SM
  // and throughput-bound above.
  //   n <= 148 * 8   one 8-sample CTA (4 warps, lane per link, no barriers) per SM: shortest dependent chain   -> v1
  //   n <= 148 * 32  one 32-sample CTA per SM, warp per link, named edge barriers, uncapped registers           -> v3
  //   larger         64 samples per SM, two per lane on the packed FFMA2 / FMUL2 / FADD2 path (half the issue slots per
  //                  sample; with the topology in uniform registers it beats the two-group scalar CTA by 8 %)      -> v9
  // A batch of S solves is decided on its total sample count S * n (all variants give identical bits).
  const int ntot = a.n * S;
  if (variant == 0) variant = (L == 11) ? (ntot <= 148 * 8 ? 1 : (ntot <= 148 * 32 ? 3 : ((m->max_ncon <= 2 && m->pk_ok) ? 9 : 2))) : 2;   // contact-heavy models (humanoidstandup): CTA barriers
  if (!m->named_ok) variant = variant == 3 ? 2 : (variant == 9 ? 8 : variant);   // deep trees: not enough named barriers
  if ((variant == 8 || variant == 9) && !m->pk_ok) variant = 2;   // the packed kernel is built for 11-link hinge-only models (no slide dofs)
  if (variant == 8 || variant == 9) {
    // packed kernel: 64 samples per CTA, two per lane (variant 8: group barriers with decoupled leaves, 9: named edge barriers)
    memcpy(a.wl, m->wl1, sizeof(a.wl));
    a.count_x = 32 * (L - m->nlate);
    const dim3 grid((a.n + mbd::kPkSamples - 1) / mbd::kPkSamples, S);
    const int dyn = (int)mbd::kPkDynBytes;
#define MBD_PK_ATTR(F, C, S) CK(cudaFuncSetAttribute(mbd::k_rollout_pk<F, C, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn))
#define MBD_PK_LAUNCH(C, S)                                                                     \
  do {                                                                                          \
    if (fused) mbd::k_rollout_pk<true, C, S><<<grid, 32 * mbd::kPkLinks, dyn, st>>>(a);         \
    else mbd::k_rollout_pk<false, C, S><<<grid, 32 * mbd::kPkLinks, dyn, st>>>(a);              \
  } while (0)
    static bool pk_attr_set_dev[64] = {false};
    bool& pk_attr_set = pk_attr_set_dev[current_device_slot()];
    if (!pk_attr_set) {
      MBD_PK_ATTR(true, 2, 0); MBD_PK_ATTR(false, 2, 0); MBD_PK_ATTR(true, 2, 2); MBD_PK_ATTR(false, 2, 2);
      MBD_PK_ATTR(true, MBD_MAXCON, 0); MBD_PK_ATTR(false, MBD_MAXCON, 0); MBD_PK_ATTR(true, MBD_MAXCON, 2); MBD_PK_ATTR(false, MBD_MAXCON, 2);
      pk_attr_set = true;
    }
    if (m->max_ncon <= 2) { if (variant == 8) MBD_PK_LAUNCH(2, 0); else MBD_PK_LAUNCH(2, 2); }
    else { if (variant == 8) MBD_PK_LAUNCH(MBD_MAXCON, 0); else MBD_PK_LAUNCH(MBD_MAXCON, 2); }
#undef MBD_PK_ATTR
#undef MBD_PK_LAUNCH
  } else if (variant >= 2) {
    size_t dyn = (size_t)L * (mbd::kXF + mbd::kEF) * mbd::kWplLanes * sizeof(float);
    const bool split = (variant == 5);
    memcpy(a.wl, split ? m->wl2 : m->wl1, sizeof(a.wl));
    a.offs = split ? m->offs2 : m->offs1;
    memcpy(a.gw, m->gw2, sizeof(a.gw));
    a.count_x = 32 * (L - m->nlate);
    if (split) {
      const dim3 grid((a.n + 15) / 16, S);
      const int nw = m->nwarps2;
      if (nw <= 6) MBD_LAUNCH_WPL(6, 4, 0, 2, grid, 32 * nw);     // humanoids: 6 warps, 4 CTAs/SM
      else MBD_LAUNCH_WPL(MBD_MAXL, 1, 0, 2, grid, 32 * nw);
    } else {
      const int gx = (a.n + mbd::kWplLanes - 1) / mbd::kWplLanes;
      const dim3 grid(gx, S);
      if (L == 11 && variant == 6 && m->max_ncon <= 2) {  // two interleaved 32-sample groups per 704-thread CTA
        const dim3 grid2((a.n + 63) / 64, S);
        size_t dyn2 = 2 * dyn;
        memcpy(a.wl, m->wl6, sizeof(a.wl));
        a.stagger = g_group_stagger;
        static bool attr_set_dev[64] = {false};
        bool& attr_set = attr_set_dev[current_device_slot()];
        if (!attr_set) {
          CK(cudaFuncSetAttribute(mbd::k_rollout_wpl<true, 22, 1, 0, 1, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn2));
          CK(cudaFuncSetAttribute(mbd::k_rollout_wpl<false, 22, 1, 0, 1, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn2));
          attr_set = true;
        }
        if (fused) mbd::k_rollout_wpl<true, 22, 1, 0, 1, 2, 2><<<grid2, 64 * L, dyn2, st>>>(a);
        else mbd::k_rollout_wpl<false, 22, 1, 0, 1, 2, 2><<<grid2, 64 * L, dyn2, st>>>(a);
      } else if (L == 11 && variant == 2) MBD_LAUNCH_WPL(11, 2, 0, 1, grid, 32 * L);       // CTA-wide barriers
      else if (L == 11 && variant == 3 && gx * S <= 148) MBD_LAUNCH_WPL(11, 1, 2, 1, grid, 32 * L);  // one CTA per SM (whole launch): no register cap
      else if (L == 11 && variant == 3) MBD_LAUNCH_WPL(11, 2, 2, 1, grid, 32 * L);  // named edge barriers
      else MBD_LAUNCH_WPL(MBD_MAXL, 1, 0, 1, grid, 32 * L);
    }
  } else {
    const dim3 grid((a.n + mbd::kSPB - 1) / mbd::kSPB, S);
    if (m->max_ncon <= 2) {
      if (fused) mbd::k_rollout<true, 2><<<grid, mbd::kRolloutThreads, 0, st>>>(a);
      else mbd::k_rollout<false, 2><<<grid, mbd::kRolloutThreads, 0, st>>>(a);
    } else {
      if (fused) mbd::k_rollout<true, MBD_MAXCON><<<grid, mbd::kRolloutThreads, 0, st>>>(a);
      else mbd::k_rollout<false, MBD_MAXCON><<<grid, mbd::kRolloutThreads, 0, st>>>(a);
    }
  }
  CK(cudaGetLastError());
  return MBD_OK;
}

int mbd_rollout(const mbd_model* m, const float* state_init_dev, const float* Y0s_dev, int n, int H, float* rewss_dev,
                float* rews_dev, const float* xref_dev, int href, float* logpd_dev, float* final_state_dev, float* track_pos_dev,
                int nsub_override, mbd_stream s) {
  if (!m || !state_init_dev || !Y0s_dev || !rews_dev || n <= 0 || H <= 0) return MBD_EINVAL;
  if (xref_dev && href <= 0) return MBD_EINVAL;
  mbd::RolloutArgs a;
  memset(&a, 0, sizeof(a));
  a.blob = m->blob_dev; a.state_init = state_init_dev; a.Y0s = const_cast<float*>(Y0s_dev); a.n = n; a.H = H;
  a.rewss = rewss_dev; a.rews = rews_dev; a.xref = xref_dev; a.href = href; a.logpd = logpd_dev;
  a.final_state = final_state_dev; a.track_pos = track_pos_dev; a.nsub_override = nsub_override;
  return launch_rollout(false, a, m, (cudaStream_t)s);
}

int mbd_sample_rollout(const mbd_model* m, const float* state_init_dev, const uint32_t key[2], int n_total, int n_begin, int n_local,
                       int H, float sigma, const float* Ybar_dev, float* Y0s_dev, float* rews_dev, const float* xref_dev, int href,
                       float* logpd_dev, mbd_stream s) {
  if (!m || !state_init_dev || !key || !Ybar_dev || !Y0s_dev || !rews_dev || n_local <= 0 || H <= 0) return MBD_EINVAL;
  if (n_begin < 0 || n_begin + n_local > n_total) return MBD_EINVAL;
  if ((uint64_t)n_total * (uint64_t)H * (uint64_t)m->nu >= 0xffffffffull) return MBD_EINVAL;
  if (xref_dev && href <= 0) return MBD_EINVAL;
  mbd::RolloutArgs a;
  memset(&a, 0, sizeof(a));
  a.blob = m->blob_dev; a.state_init = state_init_dev; a.Y0s = Y0s_dev; a.n = n_local; a.H = H;
  a.rews = rews_dev; a.xref = xref_dev; a.href = href; a.logpd = logpd_dev;
  a.k0 = key[0]; a.k1 = key[1]; a.n_total = n_total; a.n_begin = n_begin; a.sigma = sigma; a.Ybar = Ybar_dev;
  return launch_rollout(true, a, m, (cudaStream_t)s);
}

int mbd_reverse_step(const mbd_model* m, const float* state_init_dev, const uint32_t key[2], int n, int H, float sigma,
                     const float* Ybar_i_dev, float temp, const float coef[5], float* Y0s_dev, float* rews_dev, float* weights_dev,
                     float* scalars_dev, float* runs_dev, float* Ybar_im1_dev, mbd_stream s) {
  if (!m || !state_init_dev || !key || !Ybar_i_dev || !coef || !Y0s_dev || !rews_dev || !weights_dev || !scalars_dev || !runs_dev ||
      !Ybar_im1_dev || n <= 0 || H <= 0)
    return MBD_EINVAL;
  if ((uint64_t)n * (uint64_t)H * (uint64_t)m->nu >= 0xffffffffull) return MBD_EINVAL;
  // the single-kernel step exists for the one-link-per-warp mapping of 11-link models with <= 2 contacts per link
  if (m->L != 11 || m->max_ncon > 2 || g_kernel_variant == 1) return MBD_EUNSUPPORTED;
  const int grid = (n + mbd::kWplLanes - 1) / mbd::kWplLanes;
  const size_t dyn = (size_t)m->L * (mbd::kXF + mbd::kEF) * mbd::kWplLanes * sizeof(float);
  static int max_coresident_dev[64];
  static bool max_coresident_init = false;
  if (!max_coresident_init) { for (int i = 0; i < 64; ++i) max_coresident_dev[i] = -1; max_coresident_init = true; }
  int& max_coresident = max_coresident_dev[current_device_slot()];
  if (max_coresident < 0) {
    int per_sm = 0, dev = 0, sms = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mbd::k_reverse_step_wpl<11, 2, 2>, 32 * 11, dyn));
    max_coresident = per_sm * sms;
  }
  if (grid > max_coresident || grid * mbd::kWplLanes < 2048) return MBD_EUNSUPPORTED;  // needs co-residency; tiny shards use v1
  mbd::RolloutArgs a;
  memset(&a, 0, sizeof(a));
  a.blob = m->blob_dev; a.state_init = state_init_dev; a.Y0s = Y0s_dev; a.n = n; a.H = H; a.rews = rews_dev;
  a.k0 = key[0]; a.k1 = key[1]; a.n_total = n; a.n_begin = 0; a.sigma = sigma; a.Ybar = Ybar_i_dev;
  memcpy(a.wl, m->wl1, sizeof(a.wl));
  memcpy(a.cfg, m->cfg, sizeof(a.cfg));
  a.prng_part = g_prng_part;
  a.offs = m->offs1;
  mbd::StepTail t;
  t.temp = temp; t.Ybar_i = Ybar_i_dev; t.c0 = coef[0]; t.c1 = coef[1]; t.c2 = coef[2]; t.c3 = coef[3]; t.c4 = coef[4];
  t.weights = weights_dev; t.scalars = scalars_dev; t.runs = runs_dev; t.out = Ybar_im1_dev;
  void* args[] = {&a, &t};
  CK(cudaLaunchCooperativeKernel((const void*)mbd::k_reverse_step_wpl<11, 2, 2>, dim3(grid), dim3(32 * 11), args, dyn, (cudaStream_t)s));
  return MBD_OK;
}

int mbd_car2d_rollout(const float* params_dev, const float* x0_dev, const uint32_t* key, int n_total, int n_begin, int n_local, int H,
                      float sigma, const float* Ybar_dev, float* Y0s_dev, float* rewss_dev, float* rews_dev, const float* xref_dev,
                      int href, float* logpd_dev, float* traj_dev, mbd_stream s) {
  if (!params_dev || !x0_dev || !Y0s_dev || !rews_dev || n_local <= 0 || H <= 0) return MBD_EINVAL;
  if (key && (!Ybar_dev || n_begin < 0 || n_begin + n_local > n_total)) return MBD_EINVAL;
  mbd::CarArgs a;
  memset(&a, 0, sizeof(a));
  a.params = params_dev; a.x0 = x0_dev; a.Y0s = Y0s_dev; a.n = n_local; a.H = H; a.rewss = rewss_dev; a.rews = rews_dev;
  a.xref = xref_dev; a.href = href; a.logpd = logpd_dev; a.traj = traj_dev;
  a.fused = key != nullptr;
  a.prng_part = g_prng_part;
  if (key) { a.k0 = key[0]; a.k1 = key[1]; a.n_total = n_total; a.n_begin = n_begin; a.sigma = sigma; a.Ybar = Ybar_dev; }
  mbd::k_car2d<false><<<(n_local + 63) / 64, 64, 0, (cudaStream_t)s>>>(a);
  CK(cudaGetLastError());
  return MBD_OK;
}

int mbd_pusht_rollout(const float* params_dev, const float* x0_dev, const uint32_t* key, int n_total, int n_begin, int n_local, int H,
                      float sigma, const float* Ybar_dev, float* Y0s_dev, float* rewss_dev, float* rews_dev, float* final_state_dev,
                      float* traj_dev, mbd_stream s) {
  if (!params_dev || !x0_dev || !Y0s_dev || !rews_dev || n_local <= 0 || H <= 0) return MBD_EINVAL;
  if (key && (!Ybar_dev || n_begin < 0 || n_begin + n_local > n_total)) return MBD_EINVAL;
  if (key && (uint64_t)n_total * (uint64_t)H * 2ull >= 0xffffffffull) return MBD_EINVAL;
  mbd::PushTArgs a;
  memset(&a, 0, sizeof(a));
  a.params = params_dev; a.x0 = x0_dev; a.Y0s = Y0s_dev; a.n = n_local; a.H = H; a.rewss = rewss_dev; a.rews = rews_dev;
  a.final_state = final_state_dev; a.traj = traj_dev;
  a.fused = key != nullptr;
  a.prng_part = g_prng_part;
  if (key) { a.k0 = key[0]; a.k1 = key[1]; a.n_total = n_total; a.n_begin = n_begin; a.sigma = sigma; a.Ybar = Ybar_dev; }
  mbd::k_pusht<<<(n_local + 63) / 64, 64, 0, (cudaStream_t)s>>>(a);
  CK(cudaGetLastError());
  return MBD_OK;
}

int mbd_softmax_weights(const float* rews_all_dev, const float* logpd_all_dev, int n_total, int n_begin, int n_local, float temp,
                        float rew_xref, float* weights_dev, float* scalars_dev, float* logp_scratch_dev, mbd_stream s) {
  if (!rews_all_dev || !weights_dev || !scalars_dev || !logp_scratch_dev || n_total <= 0 || n_begin < 0 || n_begin + n_local > n_total)
    return MBD_EINVAL;
  mbd::k_softmax_weights<<<1, mbd::kStatThreads, 0, (cudaStream_t)s>>>(rews_all_dev, logpd_all_dev, n_total, n_begin, n_local, temp,
                                                                    rew_xref, weights_dev, scalars_dev, logp_scratch_dev);
  CK(cudaGetLastError());
  return MBD_OK;
}

static int weighted_sum_impl(const float* weights_dev, const float* Y0s_dev, const float* mu_dev, int n_local, int HNu, float* scratch_dev,
                             float* partial_dev, mbd_stream s) {
  if (!weights_dev || !Y0s_dev || !scratch_dev || !partial_dev || n_local <= 0 || HNu <= 0) return MBD_EINVAL;
  int nruns = (n_local + mbd::kRun - 1) / mbd::kRun;
  dim3 grid(nruns, (HNu + 255) / 256);
  if (mu_dev)
    mbd::k_wsum_runs<true><<<grid, 256, 0, (cudaStream_t)s>>>(weights_dev, Y0s_dev, mu_dev, n_local, HNu, scratch_dev);
  else
    mbd::k_wsum_runs<false><<<grid, 256, 0, (cudaStream_t)s>>>(weights_dev, Y0s_dev, nullptr, n_local, HNu, scratch_dev);
  CK(cudaGetLastError());
  mbd::k_wsum_tree<<<(HNu + 127) / 128, 128, 0, (cudaStream_t)s>>>(scratch_dev, nruns, HNu, partial_dev);
  CK(cudaGetLastError());
  return MBD_OK;
}

int mbd_weighted_sum(const float* weights_dev, const float* Y0s_dev, int n_local, int HNu, float* scratch_dev, float* partial_dev,
                     mbd_stream s) {
  return weighted_sum_impl(weights_dev, Y0s_dev, nullptr, n_local, HNu, scratch_dev, partial_dev, s);
}

int mbd_weighted_sum_runs(const float* weights_dev, const float* Y0s_dev, int n_local, int HNu, float* runs_dev, mbd_stream s) {
  if (!weights_dev || !Y0s_dev || !runs_dev || n_local <= 0 || HNu <= 0) return MBD_EINVAL;
  int nruns = (n_local + mbd::kRun - 1) / mbd::kRun;
  dim3 grid(nruns, (HNu + 255) / 256);
  mbd::k_wsum_runs<false><<<grid, 256, 0, (cudaStream_t)s>>>(weights_dev, Y0s_dev, nullptr, n_local, HNu, runs_dev);
  CK(cudaGetLastError());
  return nruns;
}

int mbd_weighted_sqerr_sum(const float* weights_dev, const float* Y0s_dev, const float* mu_dev, int n_local, int HNu, float* scratch_dev,
                           float* partial_dev, mbd_stream s) {
  if (!mu_dev) return MBD_EINVAL;
  return weighted_sum_impl(weights_dev, Y0s_dev, mu_dev, n_local, HNu, scratch_dev, partial_dev, s);
}

int mbd_peer_gather(const uint64_t* peer_base_ptrs, int P, int rank, size_t src_off_words, int count, size_t flag_off_words,
                    uint32_t epoch, float* dst_dev, uint32_t* err_dev, mbd_stream s) {
  if (!peer_base_ptrs || P < 1 || P > 8 || rank < 0 || rank >= P || count <= 0 || !dst_dev || !err_dev || epoch == 0) return MBD_EINVAL;
  mbd::PeerArgs a;
  memset(&a, 0, sizeof(a));
  for (int r = 0; r < P; ++r) a.peer[r] = reinterpret_cast<float*>(peer_base_ptrs[r]);
  a.P = P; a.rank = rank; a.count = count; a.src_off = src_off_words; a.flag_off = flag_off_words; a.epoch = epoch;
  a.dst = dst_dev; a.err = err_dev;
  int total = P * count;
  int grid = (total + 1023) / 1024;
  if (grid > 64) grid = 64;
  mbd::k_peer_gather<<<grid, 256, 0, (cudaStream_t)s>>>(a);
  CK(cudaGetLastError());
  return MBD_OK;
}

// launches (2) and (3) of a step: statistics / softmax (one cluster) and weighted mean + update ("last CTA done")
static int step_tail_launch(const mbd_step_plan* pl, cudaStream_t st, cudaEvent_t ev_mid2 = nullptr) {
  const int HNu = pl->H * pl->nu;
  const bool demo = pl->xref_dev != nullptr;
  mbd::TailArgs t;
  memset(&t, 0, sizeof(t));
  t.sp = pl->params_dev; t.ctl = pl->ctl_dev; t.Ybars = pl->Ybars_dev; t.rew_hist = pl->rew_hist_dev;
  t.N = pl->n_total; t.n_begin = pl->n_begin; t.n_local = pl->n_local; t.HNu = HNu;
  t.temp = pl->temp; t.rew_xref = pl->rew_xref; t.demo = demo ? 1 : 0;
  t.Y0s = pl->Y0s_dev; t.rews = pl->rews_dev; t.logpd = pl->logpd_dev;
  t.rews_all = pl->P == 1 ? pl->rews_dev : pl->rews_all_dev;
  t.logpd_all = pl->P == 1 ? pl->logpd_dev : pl->logpd_all_dev;
  t.logp = pl->logp_dev; t.weights = pl->weights_dev; t.runs = pl->runs_dev; t.partial = pl->partial_dev; t.scalars = pl->scalars_dev;
  t.P = pl->P; t.rank = pl->rank;
  for (int r = 0; r < pl->P && pl->peer_base_ptrs; ++r) t.peer[r] = reinterpret_cast<float*>(pl->peer_base_ptrs[r]);
  t.off_rews = pl->off_rews_words; t.off_logpd = pl->off_logpd_words; t.off_partial = pl->off_partial_words; t.off_flags = pl->off_flags_words;
  t.timeout_cycles = pl->timeout_cycles ? pl->timeout_cycles : 40000000000ull;   // ~20 s: a dead peer, not a slow one
  const int S = pl->n_solves > 1 ? pl->n_solves : 1;
  if (S > 1) { t.temps = pl->temps_dev; t.nd = pl->n_diffuse; }   // one cluster / one z-slice of the update grid per solve
  if (S > 1) mbd::k_step_weights<true><<<mbd::kClusterCtas * S, mbd::kWeightsThreads, 0, st>>>(t);
  else mbd::k_step_weights<false><<<mbd::kClusterCtas, mbd::kWeightsThreads, 0, st>>>(t);
  CK(cudaGetLastError());
  if (ev_mid2) CK(cudaEventRecord(ev_mid2, st));
  const int nruns = (pl->n_local + mbd::kTailRun - 1) / mbd::kTailRun;
  dim3 grid(nruns, (HNu + mbd::kUpdThreads - 1) / mbd::kUpdThreads, S);
  if (S > 1) mbd::k_step_update<true><<<grid, mbd::kUpdThreads, 0, st>>>(t);
  else mbd::k_step_update<false><<<grid, mbd::kUpdThreads, 0, st>>>(t);
  CK(cudaGetLastError());
  return MBD_OK;
}

// ---- one diffusion step with device-resident parameters: three launches, CUDA-graph capturable --------------------------
static int step_launch_impl(const mbd_step_plan* pl, cudaStream_t st, cudaEvent_t ev_mid, cudaEvent_t ev_mid2 = nullptr) {
#define STEP_REQUIRE(cond, msg)                                             \
  do {                                                                      \
    if (!(cond)) { snprintf(g_err, sizeof(g_err), "mbd_step_launch: %s", msg); return MBD_EINVAL; } \
  } while (0)
  STEP_REQUIRE(pl != nullptr, "plan is NULL");
  STEP_REQUIRE(pl->state_init_dev && pl->params_dev && pl->ctl_dev && pl->Ybars_dev, "state_init / params / ctl / Ybars must be set");
  STEP_REQUIRE(pl->Y0s_dev && pl->rews_dev && pl->rews_all_dev && pl->logp_dev && pl->weights_dev && pl->runs_dev && pl->partial_dev &&
               pl->scalars_dev, "a work buffer is NULL");
  STEP_REQUIRE(pl->n_local > 0 && pl->H > 0 && pl->nu > 0 && pl->n_begin >= 0 && pl->n_begin + pl->n_local <= pl->n_total,
               "bad sample range (n_begin + n_local must lie inside n_total)");
  STEP_REQUIRE(pl->P >= 1 && pl->P <= 8 && pl->rank >= 0 && pl->rank < pl->P, "rank count must be 1..8");
  STEP_REQUIRE(pl->P == 1 || pl->peer_base_ptrs != nullptr, "sharded step needs the peers' symmetric-buffer addresses");
  const int HNu = pl->H * pl->nu;
  STEP_REQUIRE((HNu + mbd::kUpdThreads - 1) / mbd::kUpdThreads <= MBD_STEP_MAX_COLBLOCKS, "H * Nu exceeds 27 * 256 columns");
  STEP_REQUIRE((uint64_t)pl->n_total * (uint64_t)HNu < 0xffffffffull, "Nsample * H * Nu must stay below 2^32 (threefry counter layout)");
  const bool demo = pl->xref_dev != nullptr;
  STEP_REQUIRE(!demo || (pl->href > 0 && pl->logpd_dev && pl->logpd_all_dev), "demo step needs href, logpd and logpd_all");
  STEP_REQUIRE(pl->n_solves >= 0, "n_solves must be >= 0");
  const int S = pl->n_solves > 1 ? pl->n_solves : 1;
  STEP_REQUIRE(S == 1 || pl->P == 1, "a batch of solves (n_solves > 1) cannot be sharded over ranks (P must be 1)");
  STEP_REQUIRE(S == 1 || pl->temps_dev != nullptr, "n_solves > 1 needs temps_dev (one temperature per solve)");
  STEP_REQUIRE(S == 1 || pl->n_diffuse >= 2, "n_solves > 1 needs n_diffuse >= 2 (rows per solve of params / Ybars / rew_hist)");
  STEP_REQUIRE(S <= 65535, "n_solves exceeds the grid's y / z extent (65535)");
  // per-solve strides of the arrays with a leading solve axis (all zero for one solve: the kernels then add nothing)
  mbd::SolveStride ss;
  memset(&ss, 0, sizeof(ss));
  if (S > 1) {
    ss.state = pl->model ? (unsigned)(pl->model->L * MBD_STATE_STRIDE) : (pl->env_kind == MBD_ENV_PUSHT ? (unsigned)MBD_PT_STATE : 3u);
    ss.y0s = (unsigned)pl->n_local * (unsigned)HNu; ss.n = (unsigned)pl->n_local;
    ss.nd = (unsigned)pl->n_diffuse; ss.ybars = (unsigned)pl->n_diffuse * (unsigned)HNu;
  }
#undef STEP_REQUIRE
  // 1. sampling + rollouts
  if (pl->model) {
    if (pl->model->nu != pl->nu) return MBD_EINVAL;
    mbd::RolloutArgs a;
    memset(&a, 0, sizeof(a));
    a.blob = pl->model->blob_dev; a.state_init = pl->state_init_dev; a.Y0s = pl->Y0s_dev; a.n = pl->n_local; a.H = pl->H;
    a.rews = pl->rews_dev; a.xref = pl->xref_dev; a.href = pl->href; a.logpd = demo ? pl->logpd_dev : nullptr;
    a.n_total = pl->n_total; a.n_begin = pl->n_begin;
    a.sp = pl->params_dev; a.ctl = pl->ctl_dev; a.Ybars = pl->Ybars_dev; a.ss = ss;
    int rc = launch_rollout(true, a, pl->model, st, S);
    if (rc != MBD_OK) return rc;
  } else if (pl->env_kind == MBD_ENV_PUSHT) {
    if (!pl->car_params_dev || pl->nu != 2 || demo) return MBD_EINVAL;
    mbd::PushTArgs a;
    memset(&a, 0, sizeof(a));
    a.params = pl->car_params_dev; a.x0 = pl->state_init_dev; a.Y0s = pl->Y0s_dev; a.n = pl->n_local; a.H = pl->H;
    a.rews = pl->rews_dev;
    a.fused = 1; a.n_total = pl->n_total; a.n_begin = pl->n_begin; a.prng_part = g_prng_part;
    a.sp = pl->params_dev; a.ctl = pl->ctl_dev; a.Ybars = pl->Ybars_dev; a.ss = ss;
    mbd::k_pusht<<<dim3((pl->n_local + 63) / 64, S), 64, 0, st>>>(a);
    CK(cudaGetLastError());
  } else {
    if (!pl->car_params_dev || pl->nu != 2) return MBD_EINVAL;
    mbd::CarArgs a;
    memset(&a, 0, sizeof(a));
    a.params = pl->car_params_dev; a.x0 = pl->state_init_dev; a.Y0s = pl->Y0s_dev; a.n = pl->n_local; a.H = pl->H;
    a.rews = pl->rews_dev; a.xref = pl->xref_dev; a.href = pl->href; a.logpd = demo ? pl->logpd_dev : nullptr;
    a.fused = 1; a.n_total = pl->n_total; a.n_begin = pl->n_begin; a.prng_part = g_prng_part;
    a.sp = pl->params_dev; a.ctl = pl->ctl_dev; a.Ybars = pl->Ybars_dev; a.ss = ss;
    if (S > 1) mbd::k_car2d<true><<<dim3((pl->n_local + 63) / 64, S), 64, 0, st>>>(a);
    else mbd::k_car2d<false><<<(pl->n_local + 63) / 64, 64, 0, st>>>(a);
    CK(cudaGetLastError());
  }
  if (ev_mid) CK(cudaEventRecord(ev_mid, st));
  return step_tail_launch(pl, st, ev_mid2);
}
int mbd_step_launch(const mbd_step_plan* pl, mbd_stream s) { return step_launch_impl(pl, (cudaStream_t)s, nullptr); }

// mbd_step_launch with CUDA events recorded before launch (1), between launch (1) and launch (2), and after launch (3):
// bench.py times the rollout kernel inside the real step with them (torch.cuda.Event exposes no handle that a C launch
// sequence could record into; the events come from mbd_event_create)
int mbd_step_launch_ev(const mbd_step_plan* pl, void* ev_before, void* ev_mid, void* ev_mid2, void* ev_after, mbd_stream s) {
  cudaStream_t st = (cudaStream_t)s;
  if (ev_before) CK(cudaEventRecord((cudaEvent_t)ev_before, st));
  int rc = step_launch_impl(pl, st, (cudaEvent_t)ev_mid, (cudaEvent_t)ev_mid2);
  if (rc != MBD_OK) return rc;
  if (ev_after) CK(cudaEventRecord((cudaEvent_t)ev_after, st));
  return MBD_OK;
}
void* mbd_event_create(void) {
  cudaEvent_t e = nullptr;
  if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
  return (void*)e;
}
void mbd_event_destroy(void* e) { if (e) cudaEventDestroy((cudaEvent_t)e); }
int mbd_event_record(void* e, mbd_stream s) { CK(cudaEventRecord((cudaEvent_t)e, (cudaStream_t)s)); return MBD_OK; }
int mbd_event_sync(void* e) { CK(cudaEventSynchronize((cudaEvent_t)e)); return MBD_OK; }
float mbd_event_elapsed_ms(void* a, void* b) {
  float ms = -1.0f;
  if (cudaEventElapsedTime(&ms, (cudaEvent_t)a, (cudaEvent_t)b) != cudaSuccess) return -1.0f;
  return ms;
}

// measured fp32 FFMA throughput of the current device in TFLOP/s (FMA = 2 flop); synchronises the stream
int mbd_ffma_peak(float* scratch_dev, int iters, float* tflops_out, mbd_stream s) {
  if (!scratch_dev || !tflops_out || iters <= 0) return MBD_EINVAL;
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t st = (cudaStream_t)s;
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  const int grid = 2 * sms;
  mbd::k_ffma_peak<<<grid, 1024, 0, st>>>(scratch_dev, iters / 8 + 1, 1.0000001f, 1e-9f);   // warm-up
  float best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    CK(cudaEventRecord(e0, st));
    mbd::k_ffma_peak<<<grid, 1024, 0, st>>>(scratch_dev, iters, 1.0000001f, 1e-9f);
    CK(cudaEventRecord(e1, st));
    CK(cudaEventSynchronize(e1));
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    if (ms < best) best = ms;
  }
  CK(cudaGetLastError());
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  const double flop = 2.0 * 64.0 * (double)iters * 1024.0 * (double)grid;
  *tflops_out = (float)(flop / (best * 1e-3) / 1e12);
  return MBD_OK;
}

int mbd_test_arith(int op, const float* a_dev, const float* b_dev, float* out_dev, int n, mbd_stream s) {
  if (!a_dev || !b_dev || !out_dev || n <= 0 || op < 0 || op > 3) return MBD_EINVAL;
  mbd::k_test_arith<<<(n + 255) / 256, 256, 0, (cudaStream_t)s>>>(op, a_dev, b_dev, out_dev, n);
  CK(cudaGetLastError());
  return MBD_OK;
}

#ifdef MBD_PROFILE_PHASES
int mbd_prof_read(unsigned long long* out) { return (int)cudaMemcpyFromSymbol(out, g_phase_cycles, sizeof(unsigned long long) * 16 * 8); }
int mbd_prof_reset(void) {
  static unsigned long long z[16 * 8] = {0};
  return (int)cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z));
}
#endif

int mbd_update(const float* partials_dev, int P, int HNu, const float* Ybar_i_dev, const float coef[5], float* Ybar_im1_dev,
               mbd_stream s) {
  if (!partials_dev || !Ybar_i_dev || !coef || !Ybar_im1_dev || P <= 0 || HNu <= 0) return MBD_EINVAL;
  mbd::k_update<<<(HNu + 127) / 128, 128, 0, (cudaStream_t)s>>>(partials_dev, P, HNu, Ybar_i_dev, coef[0], coef[1], coef[2], coef[3],
                                                              coef[4], Ybar_im1_dev);
  CK(cudaGetLastError());
  return MBD_OK;
}

}  // extern "C"
