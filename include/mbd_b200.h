/* mbd_b200.h — C ABI of the B200-native MBD hot path (libmbd_b200.so).
 *
 * The reference has no FFI layer (it is pure Python/JAX); the seams this library replaces are
 * the Python call sites of the jitted hot path.  Each entry point cites the reference
 * interface it stands in for.  Conventions: one host thread; every pointer marked `_dev` is
 * device memory owned by the caller (torch tensors on the Python side); the stream is passed
 * explicitly; return 0 on success, a negative MBD_E* code otherwise (no exceptions cross the
 * ABI, nothing is allocated after *_create).  See INTEGRATION.md for the ctypes stub.
 */
#ifndef MBD_B200_H_
#define MBD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MBD_OK 0
#define MBD_EINVAL (-1)  /* bad argument / bad blob */
#define MBD_ECUDA (-2)   /* CUDA runtime error (see mbd_last_error) */
#define MBD_ENOGPU (-3)  /* no CUDA device: there is deliberately NO CPU fallback */
#define MBD_EUNSUPPORTED (-4) /* this fused entry point does not cover the configuration: use the separate calls */

typedef struct mbd_model mbd_model;
typedef void* mbd_stream; /* cudaStream_t */

/* ABI/layout self-description (cross-checked against the Python packer in tests/test_abi.py) */
int mbd_layout_info(int32_t* out, int n);
/* sizeof / offsetof of the structs passed by pointer (mbd_step_params, mbd_step_ctl, mbd_step_plan), same cross-check */
int mbd_abi_sizes(int32_t* out, int n);
/* offsetof(mbd_step_plan, n_solves / n_diffuse / temps_dev): the batched-solve fields, same cross-check */
int mbd_abi_batch_offsets(int32_t* out, int n);
const char* mbd_last_error(void);
int mbd_device_count(void);
/* rollout kernel mapping: 0 = auto (by shard size), 1 = v1 (one link per lane), 2/3 = v2 (one link per
 * warp, lane = sample) with CTA-wide / named-barrier phase synchronisation (4, mbarrier polling, was removed), 5 = v2 with two
 * same-type links per warp (16 samples per CTA), 6 = v2 with two interleaved 32-sample groups per 704-thread CTA
 * (leaf links decoupled from the group barriers), 8/9 = packed kernel: two samples per lane on FFMA2/FMUL2/FADD2,
 * 64 samples per CTA, group barriers / named edge barriers (11-link models; others fall back to 2).  4 and 7 are unused
 * (as are 10 / 11, a round-2 experiment that lost and was removed).
 * All variants produce bit-identical results; the switch exists for tests and profiling. */
int mbd_set_kernel_variant(int v);
/* threefry counter layout of every in-kernel sampler (process-wide): 0 = legacy (jax_threefry_partitionable=False, what the JAX
 * known-answer vectors in tests/test_prng.py pin), 1 = partitionable (the default of JAX >= 0.5; [jax-recalled], unpinned).
 * The host-side key chain must use the same layout (mbd_b200.prng.set_layout). */
int mbd_set_prng_layout(int partitionable);
/* tuning hook: slot -> link order of the one-link-per-warp mapping (slot L-1 gets the highest warp id) */
int mbd_model_set_warp_order(mbd_model* m, const int* order, int n);
/* tuning hook: cycles the second sample group of a two-group CTA waits before its first step (de-phases the groups) */
int mbd_set_group_stagger(int cycles);
/* tuning hook: two-group CTA warp table, map[w] = (group << 4) | slot for the 2*L warps */
int mbd_model_set_group_map(mbd_model* m, const int* map, int n);

/* brax.io.mjcf.load(...) result made device resident — replaces the `sys` captured by the
 * jitted env.step (/root/reference/mbd/envs/humanoidrun.py:15-17).  blob: include/mbd_model.h */
mbd_model* mbd_model_create(const uint32_t* blob_host, size_t nwords);
void mbd_model_destroy(mbd_model*);

/* eps = jax.random.normal(key,(Nsample,H,Nu)); Y0s = clip(eps*sigma + Ybar_i, -1, 1)
 * (/root/reference/mbd/planners/mbd_planner.py:103-106) for global samples
 * [n_begin, n_begin+n_local) of n_total.  Y0s_dev [n_local, HNu]. */
int mbd_sample(const uint32_t key[2], int n_total, int n_begin, int n_local, int HNu, float sigma,
               const float* Ybar_dev, float* Y0s_dev, mbd_stream s);

/* jax.vmap(rollout_us, in_axes=(None,0))(state_init, Y0s)  (mbd_planner.py:109, utils.py:14-20)
 * for a Brax-positional env (HumanoidRun.step humanoidrun.py:34-41, HumanoidTrack.step
 * humanoidtrack.py:63-82).  state_init_dev [L,13]; Y0s_dev [n,H,Nu].
 * Outputs (NULL = not wanted): rewss_dev [n,H]; rews_dev [n] = rewss.mean(-1) (required);
 * logpd_dev [n] = vmap(env.eval_xref_logpd)(qs) when xref_dev [ntrack,href,3] is given;
 * final_state_dev [n,L,13]; track_pos_dev [n,H,ntrack,3].  nsub_override>0 replaces n_frames. */
int mbd_rollout(const mbd_model* m, const float* state_init_dev, const float* Y0s_dev, int n, int H,
                float* rewss_dev, float* rews_dev, const float* xref_dev, int href, float* logpd_dev,
                float* final_state_dev, float* track_pos_dev, int nsub_override, mbd_stream s);

/* mbd_sample + mbd_rollout fused in ONE kernel (each CTA draws the noise of its own samples,
 * writes Y0s once, then rolls them out): the hot path of reverse_once, mbd_planner.py:103-110. */
int mbd_sample_rollout(const mbd_model* m, const float* state_init_dev, const uint32_t key[2], int n_total,
                       int n_begin, int n_local, int H, float sigma, const float* Ybar_dev, float* Y0s_dev,
                       float* rews_dev, const float* xref_dev, int href, float* logpd_dev, mbd_stream s);

/* The whole of reverse_once (mbd_planner.py:97-135, enable_demo False, one GPU) as ONE cooperative kernel:
 * sampling + rollouts, grid barrier, reward statistics + softmax (recomputed per CTA), weighted-mean runs, grid
 * barrier, pairwise tree + update.  Bit-identical to mbd_sample_rollout + mbd_softmax_weights + mbd_weighted_sum
 * + mbd_update.  Returns MBD_EUNSUPPORTED when the configuration is not covered (model shape, shard too large
 * for co-residency or too small to benefit): the caller then uses the separate entry points.
 * runs_dev: ceil(n/64)*H*Nu floats; scalars_dev[4] as in mbd_softmax_weights. */
int mbd_reverse_step(const mbd_model* m, const float* state_init_dev, const uint32_t key[2], int n, int H, float sigma,
                     const float* Ybar_i_dev, float temp, const float coef[5], float* Y0s_dev, float* rews_dev,
                     float* weights_dev, float* scalars_dev, float* runs_dev, float* Ybar_im1_dev, mbd_stream s);

/* Car2d (self-contained env, /root/reference/mbd/envs/car2d.py:77-102).
 * params_dev: [obs_center(11x2), obs_radius, dt, dt/2, dt/6]; x0_dev [3]; xref_dev [href,2] or NULL.
 * key == NULL: Y0s_dev is an input; else it is sampled first (fused) as in mbd_sample. */
int mbd_car2d_rollout(const float* params_dev, const float* x0_dev, const uint32_t* key, int n_total, int n_begin,
                      int n_local, int H, float sigma, const float* Ybar_dev, float* Y0s_dev, float* rewss_dev,
                      float* rews_dev, const float* xref_dev, int href, float* logpd_dev, float* traj_dev,
                      mbd_stream s);

/* rews.mean(), rews.std() (guard <1e-4 -> 1), logp0, demo blend, softmax
 * (mbd_planner.py:110-127) over the GLOBAL reward vector rews_all_dev [n_total] (all ranks'
 * samples, all-gathered by the caller); writes the softmax weights of the local slice
 * weights_dev [n_local] and scalars_dev[4] = {rews.mean(), rew_std, max logit, sum exp}.
 * logpd_all_dev NULL = enable_demo False.  logp_scratch_dev: n_total floats (receives logp0). */
int mbd_softmax_weights(const float* rews_all_dev, const float* logpd_all_dev, int n_total, int n_begin,
                        int n_local, float temp, float rew_xref, float* weights_dev, float* scalars_dev,
                        float* logp_scratch_dev, mbd_stream s);

/* partial of Ybar = einsum("n,nij->ij", weights, Y0s) over the local samples
 * (mbd_planner.py:128), deterministic order (64-sample runs, then a pairwise tree) so that
 * sharded and unsharded runs agree bit for bit.  scratch_dev: ceil(n_local/64)*HNu floats. */
int mbd_weighted_sum(const float* weights_dev, const float* Y0s_dev, int n_local, int HNu, float* scratch_dev,
                     float* partial_dev, mbd_stream s);

/* First stage of mbd_weighted_sum only: runs_dev [ceil(n_local/64)][HNu].  Returns the number of runs (> 0) or a
 * negative error.  With one rank the pairwise tree over the runs is the same tree mbd_update applies to its
 * `partials`, so `mbd_update(runs, P = nruns, ...)` finishes the weighted mean and the update in one launch. */
int mbd_weighted_sum_runs(const float* weights_dev, const float* Y0s_dev, int n_local, int HNu, float* runs_dev, mbd_stream s);

/* einsum("n,nij->ij", weights, (Y0s - mu_0t)**2): the CMA-ES spread update of
 * /root/reference/mbd/planners/path_integral.py:39-45, same deterministic order as mbd_weighted_sum. */
int mbd_weighted_sqerr_sum(const float* weights_dev, const float* Y0s_dev, const float* mu_dev, int n_local, int HNu,
                           float* scratch_dev, float* partial_dev, mbd_stream s);

/* Fused exchange over NVLink peer memory (replaces ncclAllGather for the two small per-step exchanges of
 * reverse_once when the Nsample axis is sharded): an in-kernel cross-GPU barrier (system-scope flags in
 * the peers' symmetric buffers) followed by direct peer loads.  peer_base_ptrs [P] are the base addresses
 * of every rank's symmetric buffer (identical layout); dst_dev [P*count] receives rank-ordered data read
 * from word offset src_off_words; flag rows live at flag_off_words (P words, zero-initialised, one row
 * per call site); epoch must increase by one per call on the same row.  err_dev: set to 1 on timeout. */
int mbd_peer_gather(const uint64_t* peer_base_ptrs, int P, int rank, size_t src_off_words, int count,
                    size_t flag_off_words, uint32_t epoch, float* dst_dev, uint32_t* err_dev, mbd_stream s);

/* Test hook: element-wise MBD_DIV (op 0), MBD_RCP (1), MBD_SQRT (2), mbd_atan2f (3) — the branch-free
 * exact device sequences of include/mbd_fp32.h — so tests can compare them with IEEE results bit for bit. */
int mbd_test_arith(int op, const float* a_dev, const float* b_dev, float* out_dev, int n, mbd_stream s);

/* Ybar = tree-sum of the P rank partials; then score / Yim1 / Ybar_im1 literally as
 * mbd_planner.py:100,130-133.  coef = {sqrt(ab_i), 1/(1-ab_i), 1-ab_i, 1/sqrt(alpha_i), sqrt(ab_{i-1})}. */
int mbd_update(const float* partials_dev, int P, int HNu, const float* Ybar_i_dev, const float coef[5],
               float* Ybar_im1_dev, mbd_stream s);

/* pushT (/root/reference/mbd/envs/pushT.py:16-66, the reference's one env on Brax's `generalized` backend; planar
 * reduced-coordinate pipeline restated in include/mbd_pusht.h).  params_dev [MBD_PT_NPARAM], x0_dev [16] = q | qd.
 * key != NULL: fused sampling exactly as mbd_car2d_rollout.  final_state_dev [n,16], traj_dev [n,H,16] optional. */
int mbd_pusht_rollout(const float* params_dev, const float* x0_dev, const uint32_t* key, int n_total, int n_begin,
                      int n_local, int H, float sigma, const float* Ybar_dev, float* Y0s_dev, float* rewss_dev,
                      float* rews_dev, float* final_state_dev, float* traj_dev, mbd_stream s);
enum { MBD_ENV_CAR2D = 0, MBD_ENV_PUSHT = 1 };

/* ---- one diffusion step as THREE parameterless launches (CUDA-graph capturable) -------------------------------------
 * reverse_once (mbd_planner.py:97-135) for any rank count: (1) sampling + rollouts, (2) global reward statistics /
 * demo blend / softmax in one 8-CTA thread-block cluster that pulls the peers' per-sample returns over NVLink itself,
 * (3) weighted-mean runs whose last CTA folds the tree, exchanges the rank partials over NVLink and applies the update
 * lines 130-133.  Everything that changes from step to step lives in DEVICE memory: params_dev[i] = {Y0s_rng key
 * (mbd_planner.py:103), sigmas[i], the five schedule scalars of mbd_update}, ctl_dev->i = the step index (the host loop
 * variable of mbd_planner.py:141), decremented by the last thread of launch (3); the iterate Ybar_i is row i of Ybars_dev
 * and the result is written to row i - 1, rews.mean() to rew_hist_dev[i].  The host therefore launches the same three
 * kernels Ndiffuse-1 times (or replays one captured graph) without touching a parameter. */
typedef struct mbd_step_params { uint32_t key[2]; float sigma; float coef[5]; } mbd_step_params; /* 32 bytes */
#define MBD_STEP_MAX_COLBLOCKS 27 /* H*Nu <= 27*256 */
typedef struct mbd_step_ctl {      /* 128 bytes, zero-initialised by the caller except `i` */
  int32_t i;                       /* current step index (Ndiffuse-1 ... 1) */
  uint32_t epoch;                  /* cross-GPU rendezvous counter (advanced once per step) */
  uint32_t err;                    /* set to 1 when a cross-GPU rendezvous timed out (outputs are NaN-poisoned) */
  uint32_t pad;
  uint32_t ticket[28];             /* "last CTA done" tickets: per column block, [27] over the column blocks... see step_tail.cuh */
} mbd_step_ctl;
typedef struct mbd_step_plan {
  const mbd_model* model;            /* Brax-positional env; NULL = a flat-state env selected by env_kind: car2d (car_params_dev,
                                      * state_init_dev = x0[3]) or pushT (car_params_dev = the MBD_PT_* table, state_init_dev = q|qd [16]) */
  const float* car_params_dev;
  const float* state_init_dev;       /* [L,13] */
  const mbd_step_params* params_dev; /* [Ndiffuse] */
  mbd_step_ctl* ctl_dev;
  float* Ybars_dev;                  /* [Ndiffuse, H*Nu] */
  float* rew_hist_dev;               /* [Ndiffuse] or NULL */
  int32_t n_total, n_begin, n_local, H, nu;
  float temp, rew_xref;
  const float* xref_dev;             /* demo reference (enable_demo) or NULL */
  int32_t href;
  int32_t env_kind;                  /* model == NULL: MBD_ENV_CAR2D (0, the default) or MBD_ENV_PUSHT; sits in what was padding */
  float* Y0s_dev;                    /* [n_local, H*Nu] */
  float* rews_dev;                   /* [n_local]; P > 1: inside this rank's symmetric buffer at off_rews_words */
  float* logpd_dev;                  /* [n_local] or NULL; P > 1: at off_logpd_words */
  float* rews_all_dev;               /* [n_total] (unused when P == 1) */
  float* logpd_all_dev;              /* [n_total] or NULL */
  float* logp_dev;                   /* [n_total] scratch */
  float* weights_dev;                /* [n_local] */
  float* runs_dev;                   /* [ceil(n_local/64), H*Nu] */
  float* partial_dev;                /* [H*Nu]; P > 1: inside the symmetric buffer at off_partial_words */
  float* scalars_dev;                /* [4] = {rews.mean(), rew_std, max logit, sum exp} of the last step */
  int32_t P, rank;
  const uint64_t* peer_base_ptrs;    /* host array [P]: base address of every rank's symmetric buffer (NULL when P == 1) */
  uint64_t off_rews_words, off_logpd_words, off_partial_words, off_flags_words;  /* flags: 2 rows of 8 words, zeroed */
  uint64_t timeout_cycles;           /* cross-GPU rendezvous timeout in SM cycles; 0 = default (~20 s) */
  /* ---- batched solves (appended; a zero-initialised plan is one solve, exactly as before) ----
   * n_solves = S > 1 runs S independent solves (same env, N, H, Ndiffuse, schedule, demo flag; own state_init, key chain,
   * temperature) in the same three launches.  Every per-solve array then has the solve as its leading axis:
   * state_init [S, L*13 | 3 | 16], params [S, Nd], ctl [S], Ybars [S, Nd, HNu], rew_hist [S, Nd], Y0s [S, n, HNu],
   * rews / logpd / weights [S, n], logp [S, N], runs [S, nruns, HNu], partial [S, HNu], scalars [S, 4]; xref is shared.
   * Batches are single-rank only (P == 1). */
  int32_t n_solves;                  /* 0 or 1 = one solve */
  int32_t n_diffuse;                 /* rows per solve of params / Ybars / rew_hist (required, >= 2, when n_solves > 1) */
  const float* temps_dev;            /* [n_solves] sampling temperatures (required when n_solves > 1; `temp` is then unused) */
} mbd_step_plan;
int mbd_step_launch(const mbd_step_plan* plan, mbd_stream s);
/* the same three launches with CUDA events (mbd_event_create; NULL = skip) recorded before (1), between (1) and (2), between
 * (2) and (3), after (3): lets a caller time each kernel inside the real step on the launching stream (bench.py's roofline
 * and its per-kernel breakdown at every rank count) */
int mbd_step_launch_ev(const mbd_step_plan* plan, void* ev_before, void* ev_mid, void* ev_mid2, void* ev_after, mbd_stream s);
void* mbd_event_create(void);
void mbd_event_destroy(void* ev);
int mbd_event_record(void* ev, mbd_stream s);
int mbd_event_sync(void* ev);
float mbd_event_elapsed_ms(void* ev_a, void* ev_b);

/* Measured fp32 FFMA throughput of the current device in TFLOP/s (16 independent chains per thread, 2048 threads per SM):
 * the denominator of bench.py's fp32 roofline (SURVEY 8d).  Synchronises the stream. */
int mbd_ffma_peak(float* scratch_dev, int iters, float* tflops_out, mbd_stream s);

#ifdef __cplusplus
}
#endif
#endif /* MBD_B200_H_ */
