// pusht.cuh — the pushT env (/root/reference/mbd/envs/pushT.py:16-66) on the GPU: one sample per thread.
//
// pushT is the reference's only env on Brax's `generalized` backend (reduced coordinates, mass matrix, constraint solve).  Its
// model (mbd/assets/pushT.xml) is three world-parented planar bodies with 8 dofs, so a whole physics step — smooth forces,
// closed-form 3x3 inverse mass matrix of the slider, up to 10 soft constraint rows (4 joint limits, 2 sphere-box contacts x 3 rows
// of the 4-sided friction pyramid, its out-of-plane pair merged), at most 100 projected Gauss-Seidel sweeps, semi-implicit Euler with implicit joint damping — fits in one
// thread's registers / local memory; there is nothing to exchange between threads and no tensor-core shaped work (the "mass
// matrix" is 3x3).  Layout and the restated algorithm: include/mbd_pusht.h; the arithmetic (association order included) is
// the one of oracle/pusht_oracle.c, which the tests compare bit for bit.  Division and square root are the IEEE ones (nvcc
// defaults -prec-div / -prec-sqrt; this kernel is latency-trivial next to the XPBD rollouts).
#pragma once

#include "mbd_pusht.h"

namespace mbd {

struct PushTArgs {
  const float* params; const float* x0; float* Y0s; int n, H;
  float* rewss; float* rews; float* final_state; float* traj;
  int fused; uint32_t k0, k1; int n_total, n_begin; float sigma; const float* Ybar;
  const mbd_step_params* sp; const mbd_step_ctl* ctl; const float* Ybars;   // device-resident step parameters (see RolloutArgs)
  int prng_part;
  SolveStride ss;          // batched step: per-solve strides (zero otherwise; mbd_b200.cu)
};

__device__ __forceinline__ void pt_imp_aref(const float* P, float pos, float vel, float& imp, float& aref) {
  const float dmin = P[MBD_PT_DMIN], dmax = P[MBD_PT_DMAX], mid = P[MBD_PT_MID];
  const float x = fabsf(pos) / P[MBD_PT_WIDTH];
  const float a = (1.0f / mid) * (x * x);
  const float omx = 1.0f - x;
  const float b = 1.0f - (1.0f / (1.0f - mid)) * (omx * omx);
  const float y = x < mid ? a : b;
  float d = clampf(dmin + y * (dmax - dmin), dmin, dmax);
  if (x > 1.0f) d = dmax;
  imp = d;
  aref = (0.0f - P[MBD_PT_KB] * vel) - (P[MBD_PT_KK] * d) * pos;
}

// inverse mass matrix of the slider block (symmetric 3x3) and of the pusher (1/m on both dofs)
struct PtMinv { float imp, A00, A01, A02, A11, A12, A22; };

// The padded NRP x NRP constraint system and its projected Gauss-Seidel sweeps.  Jc / posc hold the nr ACTIVE rows compacted to
// the front.  For NRP = 4 and 8 every array below — and Jc itself when the caller built it in registers — is indexed by
// compile-time constants after unrolling, i.e. lives in registers.  The sweeps stop when none of the multipliers moved by more than
// MBD_PT_TOL of the largest one (with TOL = 0: at an exact fixed point, where all later sweeps would be no-ops).
template <int NRP>
__device__ __forceinline__ void pt_solve(const float* P, const float (*Jc)[5], const float* posc, const float* rsc, int nr, const PtMinv& M,
                                         const float* Mif, const float* qd, int iters, float* xout) {
  float A[NRP][NRP], bq[NRP], invD[NRP], x[NRP], MiJ[NRP][5];
#pragma unroll
  for (int i = 0; i < NRP; ++i) {
    if (i < nr) {
      MiJ[i][0] = M.imp * Jc[i][0]; MiJ[i][1] = M.imp * Jc[i][1];
      MiJ[i][2] = (M.A00 * Jc[i][2] + M.A01 * Jc[i][3]) + M.A02 * Jc[i][4];
      MiJ[i][3] = (M.A01 * Jc[i][2] + M.A11 * Jc[i][3]) + M.A12 * Jc[i][4];
      MiJ[i][4] = (M.A02 * Jc[i][2] + M.A12 * Jc[i][3]) + M.A22 * Jc[i][4];
    } else {
#pragma unroll
      for (int k = 0; k < 5; ++k) MiJ[i][k] = 0.0f;
    }
  }
#pragma unroll
  for (int i = 0; i < NRP; ++i) {
    float Ji[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    if (i < nr) { Ji[0] = Jc[i][0]; Ji[1] = Jc[i][1]; Ji[2] = Jc[i][2]; Ji[3] = Jc[i][3]; Ji[4] = Jc[i][4]; }
#pragma unroll
    for (int j = 0; j < NRP; ++j) {
      float a = 0.0f;
      if (i < nr && j < nr) a = (((Ji[0] * MiJ[j][0] + Ji[1] * MiJ[j][1]) + Ji[2] * MiJ[j][2]) + Ji[3] * MiJ[j][3]) + Ji[4] * MiJ[j][4];
      A[i][j] = a;
    }
    x[i] = 0.0f;
    if (i < nr) {
      const float vel = (((Ji[0] * qd[0] + Ji[1] * qd[1]) + Ji[2] * qd[2]) + Ji[3] * qd[3]) + Ji[4] * qd[4];
      float imp, aref;
      pt_imp_aref(P, posc[i], vel, imp, aref);
      const float arr = A[i][i];
      A[i][i] = arr + (rsc[i] * ((1.0f - imp) / imp)) * arr;
      invD[i] = 1.0f / A[i][i];
      bq[i] = ((((Ji[0] * Mif[0] + Ji[1] * Mif[1]) + Ji[2] * Mif[2]) + Ji[3] * Mif[3]) + Ji[4] * Mif[4]) - aref;
    } else {
      A[i][i] = 1.0f; invD[i] = 1.0f; bq[i] = 0.0f;
    }
  }
  // convergence is judged on the constraint force J^T x (the rows of a contact are linearly dependent: x keeps redistributing
  // along the null space of J^T long after the force has converged — see the oracle)
  const float tol = P[MBD_PT_TOL];
  float F[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
  for (int it = 0; it < iters; ++it) {
    float dF[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int i = 0; i < NRP; ++i) {
      float r0 = bq[i], r1 = 0.0f;   // two interleaved fused accumulators (even / odd columns): half the dependent chain
#pragma unroll
      for (int j = 0; j < NRP; j += 2) { r0 = fmaf(A[i][j], x[j], r0); r1 = fmaf(A[i][j + 1], x[j + 1], r1); }
      const float res = r0 + r1;
      const float xn = x[i] - res * invD[i];
      const float xc = xn > 0.0f ? xn : 0.0f;
      const float dxi = xc - x[i];
      if (i < nr) {
#pragma unroll
        for (int k = 0; k < 5; ++k) dF[k] = fmaf(Jc[i][k], dxi, dF[k]);
      }
      x[i] = xc;
    }
    float dmax = 0.0f, fmx = 0.0f;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      dmax = fmaxf(dmax, fabsf(dF[k]));
      F[k] = F[k] + dF[k];
      fmx = fmaxf(fmx, fabsf(F[k]));
    }
    if (dmax <= tol * fmx) break;   // converged (tol = 0: the force did not move at all)
  }
#pragma unroll
  for (int i = 0; i < NRP; ++i) xout[i] = x[i];
}

// geometry of one sphere-box pair: world normal (box -> sphere), arm of the contact point from the slider origin, distance
struct PtContact { float nx, ny, rhox, rhoy, dist; };

__device__ __forceinline__ PtContact pt_contact(const float* B, const float* q, float s, float c, float rp) {
  const float bx = q[2] + (c * B[0] - s * B[1]), by = q[3] + (s * B[0] + c * B[1]);
  const float dx = q[0] - bx, dy = q[1] - by;
  const float lx = c * dx + s * dy, ly = c * dy - s * dx;
  const float clx = clampf(lx, -B[2], B[2]), cly = clampf(ly, -B[3], B[3]);
  const float ex = lx - clx, ey = ly - cly;
  const float d2 = ex * ex + ey * ey;
  float nlx, nly, dist, sx = clx, sy = cly;
  if (d2 > 0.0f) {
    const float d = sqrtf(d2);
    nlx = ex / d; nly = ey / d;
    dist = d - rp;
  } else {
    const float px = B[2] - fabsf(lx), py = B[3] - fabsf(ly);
    if (px < py) { nlx = lx < 0.0f ? -1.0f : 1.0f; nly = 0.0f; dist = (0.0f - px) - rp; sx = nlx * B[2]; }
    else { nlx = 0.0f; nly = ly < 0.0f ? -1.0f : 1.0f; dist = (0.0f - py) - rp; sy = nly * B[3]; }
  }
  PtContact o;
  o.nx = c * nlx - s * nly; o.ny = s * nlx + c * nly;
  const float half = 0.5f * dist;
  const float ax = B[0] + (sx + nlx * half), ay = B[1] + (sy + nly * half);
  o.rhox = c * ax - s * ay; o.rhoy = s * ax + c * ay;
  o.dist = dist;
  return o;
}

// the rows of a contact: n - mu t, n + mu t, and n standing for the out-of-plane pyramid pair (regulariser weight 1/2, see the
// oracle) (pusher x, y | slider x, y, theta)
__device__ __forceinline__ void pt_contact_row(const PtContact& k, float mu, int j, float* Jr) {
  const float tx = 0.0f - k.ny, ty = k.nx;
  float ddx = k.nx, ddy = k.ny;
  if (j == 0) { ddx = k.nx - mu * tx; ddy = k.ny - mu * ty; }
  if (j == 1) { ddx = k.nx + mu * tx; ddy = k.ny + mu * ty; }
  Jr[0] = ddx; Jr[1] = ddy;
  Jr[2] = 0.0f - ddx; Jr[3] = 0.0f - ddy;
  Jr[4] = 0.0f - (k.rhox * ddy - k.rhoy * ddx);
}

// one brax.generalized.pipeline.step of the planar model; P = parameter table in shared memory
__device__ void pusht_substep(const float* P, float* q, float* qd, float u0, float u1) {
  const float dt = P[MBD_PT_DT];
  const float ms = P[MBD_PT_MS], ims = P[MBD_PT_IMS], Is = P[MBD_PT_IS], iIs = P[MBD_PT_IIS];
  float s, c;
  mbd_sincosf(q[4], &s, &c);
  const float rx = c * P[MBD_PT_CX] - s * P[MBD_PT_CY];
  const float ry = s * P[MBD_PT_CX] + c * P[MBD_PT_CY];
  // qf_smooth
  float f[5];
  const float w = qd[4], mw2 = ms * (w * w);
  f[0] = P[MBD_PT_GEAR0] * u0 - P[MBD_PT_DPX] * qd[0];
  f[1] = P[MBD_PT_GEAR1] * u1 - P[MBD_PT_DPY] * qd[1];
  f[2] = mw2 * rx - P[MBD_PT_DSX] * qd[2];
  f[3] = mw2 * ry - P[MBD_PT_DSY] * qd[3];
  f[4] = 0.0f - P[MBD_PT_DSTH] * w;
  float ftot[5] = {f[0], f[1], f[2], f[3], f[4]};
  // which constraints are active?  (registers only; rows are built afterwards, and only for the active ones)
  float limpos[MBD_PT_NLIM], limside[MBD_PT_NLIM];
  bool limact[MBD_PT_NLIM], anylim = false;
#pragma unroll
  for (int k = 0; k < MBD_PT_NLIM; ++k) {
    const float pmin = q[k] - P[MBD_PT_LIM0 + 2 * k], pmax = P[MBD_PT_LIM0 + 2 * k + 1] - q[k];
    const float pm = pmin < pmax ? pmin : pmax;
    limpos[k] = pm < 0.0f ? pm : 0.0f;
    limact[k] = pm < 0.0f;
    limside[k] = pmin < pmax ? 1.0f : -1.0f;
    anylim = anylim || limact[k];
  }
  const float mu = P[MBD_PT_MU], rp = P[MBD_PT_RP];
  const PtContact c0 = pt_contact(P + MBD_PT_BOX0, q, s, c, rp), c1 = pt_contact(P + MBD_PT_BOX0 + 4, q, s, c, rp);
  const bool act0 = c0.dist < 0.0f, act1 = c1.dist < 0.0f;
  if (anylim || act0 || act1) {
    PtMinv M;
    M.imp = P[MBD_PT_IMP];
    M.A00 = ims + (ry * ry) * iIs; M.A01 = 0.0f - (rx * ry) * iIs; M.A02 = ry * iIs;
    M.A11 = ims + (rx * rx) * iIs; M.A12 = 0.0f - rx * iIs; M.A22 = iIs;
    float Mif[5];
    Mif[0] = M.imp * f[0]; Mif[1] = M.imp * f[1];
    Mif[2] = (M.A00 * f[2] + M.A01 * f[3]) + M.A02 * f[4];
    Mif[3] = (M.A01 * f[2] + M.A11 * f[3]) + M.A12 * f[4];
    Mif[4] = (M.A02 * f[2] + M.A12 * f[3]) + M.A22 * f[4];
    const int iters = (int)P[MBD_PT_ITERS];
    if (!anylim && (act0 != act1)) {
      // the common case — the pusher touches exactly one box, no joint limit: four rows, everything in registers
      PtContact k = c0;
      if (act1) k = c1;
      float Jc[4][5], posc[4], rsc[4], x[4];
#pragma unroll
      for (int j = 0; j < MBD_PT_NCROW; ++j) { pt_contact_row(k, mu, j, Jc[j]); posc[j] = k.dist; rsc[j] = j == 2 ? 0.5f : 1.0f; }
#pragma unroll
      for (int kk = 0; kk < 5; ++kk) Jc[3][kk] = 0.0f;
      posc[3] = 0.0f; rsc[3] = 1.0f;
      pt_solve<4>(P, Jc, posc, rsc, MBD_PT_NCROW, M, Mif, qd, iters, x);
#pragma unroll
      for (int i = 0; i < MBD_PT_NCROW; ++i)
#pragma unroll
        for (int kk = 0; kk < 5; ++kk) ftot[kk] = ftot[kk] + Jc[i][kk] * x[i];
    } else {
      // general case: compact the active rows (limits, box 0, box 1 — the oracle's order) into local arrays
      float Jc[12][5], posc[12], rsc[12], x[12];
      int nr = 0;
      for (int k = 0; k < MBD_PT_NLIM; ++k)
        if (limact[k]) {
          for (int kk = 0; kk < 5; ++kk) Jc[nr][kk] = 0.0f;
          Jc[nr][k] = limside[k];
          posc[nr] = limpos[k]; rsc[nr] = 1.0f;
          ++nr;
        }
      for (int b = 0; b < MBD_PT_NBOX; ++b) {
        const PtContact k = b == 0 ? c0 : c1;
        if (k.dist < 0.0f)
          for (int j = 0; j < MBD_PT_NCROW; ++j) { pt_contact_row(k, mu, j, Jc[nr]); posc[nr] = k.dist; rsc[nr] = j == 2 ? 0.5f : 1.0f; ++nr; }
      }
      if (nr <= 4) pt_solve<4>(P, Jc, posc, rsc, nr, M, Mif, qd, iters, x);
      else if (nr <= 8) pt_solve<8>(P, Jc, posc, rsc, nr, M, Mif, qd, iters, x);
      else pt_solve<12>(P, Jc, posc, rsc, nr, M, Mif, qd, iters, x);
      for (int i = 0; i < nr; ++i)
        for (int kk = 0; kk < 5; ++kk) ftot[kk] = ftot[kk] + Jc[i][kk] * x[i];
    }
  }
  // (M + dt D) qdd = ftot
  float qdd[5];
  qdd[0] = ftot[0] / (P[MBD_PT_MP] + dt * P[MBD_PT_DPX]);
  qdd[1] = ftot[1] / (P[MBD_PT_MP] + dt * P[MBD_PT_DPY]);
  {
    const float m1 = ms + dt * P[MBD_PT_DSX], m2 = ms + dt * P[MBD_PT_DSY];
    const float a = 0.0f - ms * ry, b = ms * rx;
    const float J3 = (Is + ms * (rx * rx + ry * ry)) + dt * P[MBD_PT_DSTH];
    const float g1 = ftot[2] / m1, g2 = ftot[3] / m2;
    const float den = (J3 - (a * a) / m1) - (b * b) / m2;
    const float x3 = ((ftot[4] - a * g1) - b * g2) / den;
    qdd[2] = g1 - (a * x3) / m1;
    qdd[3] = g2 - (b * x3) / m2;
    qdd[4] = x3;
  }
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    qd[k] = qd[k] + qdd[k] * dt;
    q[k] = q[k] + qd[k] * dt;
  }
}

// pushT.py:50-62
__device__ __forceinline__ float pusht_reward(const float* q) {
  const float gx = q[5] - q[2], gy = q[6] - q[3];
  const float px = q[0] - q[2], py = q[1] - q[3];
  const float dps = sqrtf(px * px + py * py) - 0.2f;
  const float d_pusher2slider = dps > 0.0f ? dps : 0.0f;
  return 1.0f - ((sqrtf(gx * gx + gy * gy) + fabsf(q[7] - q[4]) / MBD_PI_F) + d_pusher2slider);
}

// sample_elem: the planner's per-element sampler (defined in mbd_b200.cu before this header is included)
__global__ void __launch_bounds__(64) k_pusht(PushTArgs a) {
  __shared__ float P[MBD_PT_NPARAM];
  {
    float* no_logpd = nullptr;
    solve_offsets(a.ss, a.x0, a.Y0s, a.rews, no_logpd, a.sp, a.ctl, a.Ybars);
  }
  for (int k = threadIdx.x; k < MBD_PT_NPARAM; k += blockDim.x) P[k] = a.params[k];
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const int HNu = a.H * MBD_PT_NU;
  const int nsub = (int)P[MBD_PT_NSUB];
  const uint32_t total = a.prng_part ? 0u : (uint32_t)a.n_total * (uint32_t)HNu;
  uint32_t ck0 = a.k0, ck1 = a.k1; float csigma = a.sigma; const float* cYbar = a.Ybar;
  if (a.sp != nullptr) {
    const int si = a.ctl->i;
    ck0 = a.sp[si].key[0]; ck1 = a.sp[si].key[1]; csigma = a.sp[si].sigma; cYbar = a.Ybars + (size_t)si * HNu;
  }
  float q[MBD_PT_NQ], qd[MBD_PT_NQ];
  for (int k = 0; k < MBD_PT_NQ; ++k) { q[k] = a.x0[k]; qd[k] = a.x0[MBD_PT_NQ + k]; }
  float sum = 0.0f;
  for (int t = 0; t < a.H; ++t) {
    float* ur = a.Y0s + ((size_t)i * a.H + t) * 2;
    float u0, u1;
    if (a.fused) {
      const uint32_t idx = (uint32_t)(a.n_begin + i) * (uint32_t)HNu + (uint32_t)(2 * t);
      u0 = sample_elem(ck0, ck1, idx, total, csigma, cYbar[2 * t]);
      u1 = sample_elem(ck0, ck1, idx + 1, total, csigma, cYbar[2 * t + 1]);
      ur[0] = u0; ur[1] = u1;
    } else {
      u0 = ur[0]; u1 = ur[1];
    }
    u0 = clampf(u0, -1.0f, 1.0f); u1 = clampf(u1, -1.0f, 1.0f);   // motor ctrlrange
    for (int k = 0; k < nsub; ++k) pusht_substep(P, q, qd, u0, u1);
    const float r = pusht_reward(q);
    if (a.rewss) a.rewss[(size_t)i * a.H + t] = r;
    sum += r;
    if (a.traj) {
      float* o = a.traj + ((size_t)i * a.H + t) * MBD_PT_STATE;
      for (int k = 0; k < MBD_PT_NQ; ++k) { o[k] = q[k]; o[MBD_PT_NQ + k] = qd[k]; }
    }
  }
  a.rews[i] = sum / (float)a.H;
  if (a.final_state)
    for (int k = 0; k < MBD_PT_NQ; ++k) { a.final_state[(size_t)i * MBD_PT_STATE + k] = q[k]; a.final_state[(size_t)i * MBD_PT_STATE + MBD_PT_NQ + k] = qd[k]; }
}

}  // namespace mbd
