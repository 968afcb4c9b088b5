#!/usr/bin/env python
"""bench.py — env-steps/s of the MBD reverse-diffusion step (BASELINE.json metric).

A "step" is ONE diffusion step `reverse_once` (/root/reference/mbd/planners/mbd_planner.py:97-135)
on humanoidrun: Nsample x Hsample env steps (x n_frames=7 XPBD substeps) + reward statistics +
softmax weighted mean + update.  value = Nsample*Hsample / t_step, whole job over all ranks.

  python bench.py [--gpus N --steps K --warmup W]        # under torchrun for N > 1
  python bench.py --impl reference ...                   # the CPU restatement (oracle) arm
  python bench.py --dump-outputs DIR ...                 # also save what the last timed step computed, for comparing builds

Timing: CUDA events recorded on the launching stream by the C launch sequence itself (before the step, after the
rollout kernel, after the step), >= 3 warm-ups, L2 flushed (256 MiB memset, untimed) between steps, barrier +
synchronize on both sides, max over ranks.

What the one JSON line carries beyond the contract:
  value / e2e        weak scaling (8192 samples per GPU); `strong` = the same measurement with 8192 samples IN TOTAL
                     (BASELINE config 4: "humanoidrun Nsample=8192 sample-sharded across 8 GPUs")
  parity_ok          N > 1: rank 0 re-runs the first steps of the chain UNSHARDED and compares the iterates bit for bit
  e2e_solve          wall clock of run_diffusion(Args(env_name="humanoidrun", not_render=True)) / 299 — what the reference's
                     own timing script measures (/root/reference/mbd/scripts/run_mbd.py:20-39)
  roofline           the mandated HBM figure; roofline_fp32 (against the FFMA peak MEASURED in this run) and
                     roofline_issue are the ones that bind (SURVEY F7)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

ENV_NAME, NSAMPLE, HSAMPLE, NDIFFUSE, TEMP = "humanoidrun", 8192, 50, 300, 0.1
NU, NFRAMES = 17, 7
BYTES_PER_ENV_STEP = 4 * NU + 4  # SURVEY 8(d): action row read once + reward written once = 72 B
FLOP_PER_SUBSTEP = 9336          # algorithmic flops per sample and XPBD substep (tests/test_pk_host.py::test_algorithmic_operation_count)
METRIC = "env-steps/sec (Nsample x Hsample per diffusion step) on humanoidrun"
WORKLOAD = f"{ENV_NAME} Nsample={NSAMPLE} Hsample={HSAMPLE} n_frames={NFRAMES} Ndiffuse={NDIFFUSE}"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _ncu_summary():
    """numbers of the rollout kernel from the committed ncu --set full capture (profiles/)."""
    p = os.path.join(ROOT, "profiles", "rollout_kernel_summary.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:  # noqa: BLE001
            return {}
    return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 6 and r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on all host threads
# ---------------------------------------------------------------------------------------------------------------------
def _host_threads() -> int:
    """every hardware thread this process may USE: the affinity mask capped by the cgroup CPU quota (a container can see 128
    CPUs and be allowed 32 of them; 128 OpenMP threads then only oversubscribe).  torchrun exports OMP_NUM_THREADS=1,
    which round 1 obeyed by accident — the count is passed to the oracle explicitly."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except Exception:  # noqa: BLE001
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                q, per = int(f.read()), int(g.read())
            if q > 0:
                n = min(n, max(1, int(q / per + 0.5)))
        except Exception:  # noqa: BLE001
            pass
    return max(1, n)


def time_cpu_oracle(n_samples: int, steps: int, warmup: int):
    """The CPU restatement of the same diffusion step (sampling + rollouts + statistics) on `n_samples` of the Nsample
    rollouts per step.  Threads are set explicitly; `warmup` >= 3 untimed steps bring up the OpenMP team, the pages and the
    clocks (round 1's readings moved 5x without them); the value is the MEDIAN step time.  Returns (env-steps/s, s, threads)."""
    import mbd_b200
    from mbd_b200 import prng
    from oracle import oracle as orc
    from oracle import planner as opl
    native = orc.use_native()
    simd = orc.use_simd() is not None     # SIMD across samples (what XLA-CPU under vmap would do); scalar fallback if it cannot be built here
    env = mbd_b200.envs.get_env(ENV_NAME)
    rng, rng_reset = prng.split(prng.PRNGKey(0))
    q = env.sys.init_q.astype(np.float32)
    r, r1, r2 = prng.split(rng_reset, 3)   # humanoidrun.reset on the host (no GPU needed for this arm)
    st = env.pipeline_init(q + prng.uniform(r1, (env.sys.q_size(),), minval=-0.01, maxval=0.01),
                           prng.uniform(r2, (env.sys.qd_size(),), minval=-0.01, maxval=0.01)).raw
    key, _ = prng.split(rng)
    _, alphas, alphas_bar, sigmas = opl.make_schedule(1e-4, 1e-2, NDIFFUSE)
    oenv = opl.OracleEnv("xpbd", NU, blob=env.blob, state=st, simd=simd)
    threads = _host_threads()
    Yb = np.zeros(HSAMPLE * NU, np.float32)
    times = []
    i = NDIFFUSE - 1
    for it in range(max(warmup, 3) + steps):
        key, k = prng.split(key)
        t0 = time.perf_counter()
        o = opl.reverse_once(oenv, k, n_samples, HSAMPLE, float(sigmas[i]), Yb, TEMP, alphas, alphas_bar, i, nthreads=threads)
        dt = time.perf_counter() - t0
        Yb = o["Ybar_im1"]
        i -= 1
        if it >= max(warmup, 3):
            times.append(dt)
    t = float(np.median(times))
    how = (f"{orc.use_simd().orc_simd_width()}-lane SIMD across samples (g++ -O3 -march=native; the templated physics of csrc/xpbd_pk.cuh on a host "
           "lane type, bit-identical to the scalar C oracle)") if simd else ("scalar C oracle, " + ("-O2 -march=native" if native else "-O2 -mavx2 -mfma"))
    return n_samples * HSAMPLE / t, t, threads, how


def run_reference(args):
    """--impl reference: the reference's CPU path.  JAX/Brax are not installable here (no network, no
    wheels), so this is the CPU restatement (oracle port, OpenMP over samples), labelled as such."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.cpu_samples
    val, t, threads, flags = time_cpu_oracle(n, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "note": f"CPU restatement (JAX/Brax unavailable): {flags}; OpenMP over {threads} threads, median of {args.steps} steps; "
                           f"each step = sampling + a bounded sample of {n} of the {NSAMPLE} rollouts + statistics"},
        "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{n} of {NSAMPLE} rollouts x {HSAMPLE} env steps per step, median of {args.steps} steps after "
                                   f"{max(args.warmup, 3)} warm-ups"},
        "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    import mbd_b200
    from mbd_b200 import ops, prng
    from mbd_b200.planners import engine as eng
    from mbd_b200.planners.mbd_planner import Args, run_diffusion

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    env = mbd_b200.envs.get_env(ENV_NAME)
    rng, rng_reset = prng.split(prng.PRNGKey(0))
    state_init = env.reset(rng_reset)
    _, alphas, alphas_bar, sigmas = eng.make_schedule(1e-4, 1e-2, NDIFFUSE)
    rng_exp, _ = prng.split(rng)
    keys = eng.key_chain(rng_exp, NDIFFUSE)
    HNu = HSAMPLE * NU
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    align = torch.zeros(1, device=dev)
    ev = [ops.Event() for _ in range(4)]   # before | after rollouts | after statistics | after update

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_engine(n_total, single=False):
        e = eng.DiffusionEngine(env, n_total, HSAMPLE, TEMP, False, state_init, Ndiffuse=NDIFFUSE, emulate=(1, 0, None) if single else None)
        e.load_schedule(keys, sigmas, alphas, alphas_bar)
        e.set_step(NDIFFUSE - 1)
        return e

    def chain(e, nsteps, timed, host_io):
        """nsteps diffusion steps of the real seed-0 chain from wherever the device step counter stands; returns summed
        (step ms, rollout-kernel ms)"""
        h_in = torch.zeros(HNu, dtype=torch.float32).pin_memory()
        h_out = torch.zeros(HNu + 1, dtype=torch.float32).pin_memory()
        tot, kern, kw = 0.0, 0.0, 0.0
        i = int(e.ctl[0].item())
        if host_io:
            h_in.copy_(e.Ybars[i].cpu())
        for _ in range(nsteps):
            flush.fill_(1)
            if world > 1:
                # the untimed 256 MiB flush ends at a different moment on every GPU; without re-alignment that skew is paid
                # inside the timed step at the first cross-GPU rendezvous (measured: ~80 us at 8 ranks).  A stream-ordered
                # one-word NCCL all-reduce (no host sync) lines the ranks up again BEFORE the first timed event — in a real
                # solve there is no flush and the previous step's rendezvous keeps the ranks aligned.
                dist.all_reduce(align)
            if host_io:   # the reference-facing call with HOST buffers: H2D of the iterate, D2H of result + reward
                ev[0].record()
                e.Ybars[i].copy_(h_in, non_blocking=True)
                ops.step_launch(e._plan_c)
                h_out[:HNu].copy_(e.Ybars[i - 1], non_blocking=True)
                h_out[HNu:].copy_(e.rew_hist[i:i + 1], non_blocking=True)
                ev[2].record()
            else:
                ops.step_launch_timed(e._plan_c, ev[0], ev[1], ev[3], ev[2])
            ev[2].synchronize()
            if host_io:
                h_in.copy_(h_out[:HNu])
            if timed:
                tot += ev[0].elapsed_ms(ev[2])
                if not host_io:
                    kern += ev[0].elapsed_ms(ev[1])
                    kw += ev[1].elapsed_ms(ev[3])
            i -= 1
        return tot, kern, kw

    breakdown = {}
    outputs = {}

    def measure(n_total, keep_outputs=False):
        """(ms per step, rollout-kernel ms, e2e ms per step, parity_ok or None, engine) for n_total samples over `world` ranks;
        keep_outputs: copy what the last timed step returned into `outputs` before later steps overwrite it"""
        e = make_engine(n_total)
        chain(e, args.warmup, False, False)
        barrier()
        tot, kern, kw = chain(e, args.steps, True, False)
        barrier()
        if keep_outputs:
            i = int(e.ctl[0].item()) + 1     # the last timed step read Ybars[i] and wrote Ybars[i - 1]
            outputs.update(ybar_im1=e.Ybars[i - 1].view(HSAMPLE, NU).cpu().numpy(), rew_mean=e.rew_hist[i].cpu().numpy(),
                           returns=e.rews_all.cpu().numpy())
        chain(e, 1, False, True)
        barrier()
        e2e, _, _ = chain(e, args.steps, True, True)
        barrier()
        e.check_exchange()
        t = torch.tensor([tot, kern, e2e, kw], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tot, kern, e2e, kw = (float(v) / args.steps for v in t.tolist())
        breakdown.clear()
        breakdown.update({"rollout_ms": kern, "statistics_ms": kw, "update_ms": tot - kern - kw,
                          "note": "CUDA events between the three launches of the step, max over ranks; the statistics kernel includes "
                                  "the cross-GPU rendezvous + NVLink pull of the returns, the update kernel the exchange of the rank partials"})
        parity = None
        if world > 1:
            # rank 0 re-runs the first steps of the same chain UNSHARDED: the sharded iterates must be the same bits
            ok = 1
            ncheck = min(3, args.warmup + args.steps)
            if rank == 0:
                e1 = make_engine(n_total, single=True)
                for _ in range(ncheck):
                    e1.step()
                torch.cuda.synchronize()
                a = e.Ybars[NDIFFUSE - 1 - ncheck:NDIFFUSE - 1].cpu().numpy().view(np.uint32)
                b = e1.Ybars[NDIFFUSE - 1 - ncheck:NDIFFUSE - 1].cpu().numpy().view(np.uint32)
                ok = int(np.array_equal(a, b))
                del e1
            okt = torch.tensor([ok], device=dev)
            dist.broadcast(okt, 0)
            parity = bool(okt.item())
        return tot, kern, e2e, parity, e

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n_weak = NSAMPLE * world if args.scaling == "weak" else NSAMPLE
    ms_step, kern_ms, e2e_ms, parity_ok, e = measure(n_weak, keep_outputs=bool(args.dump_outputs))
    weak_breakdown = dict(breakdown)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        # float32; the chain is the fixed seed-0 one, so the same arguments give the same inputs on every run and every build
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    n_local = e.n_local
    del e
    strong = None
    if world > 1 and args.scaling == "weak":
        # optional blocks never cost the main line: every rank takes the same path (the failure modes are deterministic — a
        # configuration error raises on all ranks alike), and the error is reported in place of the block
        try:
            s_ms, s_kern, s_e2e, s_par, es = measure(NSAMPLE)
            strong = {"metric": METRIC, "value": NSAMPLE * HSAMPLE / (s_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": s_ms,
                      "kernel_ms": s_kern, "e2e_value": NSAMPLE * HSAMPLE / (s_e2e * 1e-3), "global_samples": NSAMPLE,
                      "samples_per_gpu": es.n_local, "parity_ok": s_par, "kernels": dict(breakdown),
                      "note": "BASELINE config 4: humanoidrun Nsample=8192 sample-sharded across the ranks (strong scaling)"}
            del es
        except Exception as ex:  # noqa: BLE001
            strong = {"error": f"{type(ex).__name__}: {ex}"}
    # ---- the whole solve through the reference-facing API (run_mbd.py:20-39 times exactly this call)
    solve = None
    if not args.no_solve:
        import gc
        gc.collect()          # the engines of the step measurements (CUDA graphs, symmetric buffers) are torn down HERE, not inside the timed solve
        barrier()
        try:
            t0 = time.perf_counter()
            rew_final = run_diffusion(Args(env_name=ENV_NAME, not_render=True), log_every=10 ** 9)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            w = torch.tensor([wall], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(w, op=dist.ReduceOp.MAX)
            wall = float(w.item())
            solve = {"wall_s": wall, "ms_per_step": wall / (NDIFFUSE - 1) * 1e3, "value": NSAMPLE * HSAMPLE * (NDIFFUSE - 1) / wall,
                     "unit": "env-steps/s", "rew_final": float(rew_final), "global_samples": NSAMPLE,
                     "what": "time.time() around run_diffusion(Args(env_name='humanoidrun', not_render=True)): env + model construction, "
                             "schedule upload, graph capture, 299 steps, final rollout"}
        except Exception as ex:  # noqa: BLE001
            solve = {"error": f"{type(ex).__name__}: {ex}"}
    if rank == 0:
        value = n_weak * HSAMPLE / (ms_step * 1e-3)
        kern_s = kern_ms * 1e-3
        alg_bytes = n_local * HSAMPLE * BYTES_PER_ENV_STEP  # per launch of the rollout kernel (per rank)
        peak, peak_src = _peaks()
        achieved = alg_bytes / kern_s / 1e9
        summ = _ncu_summary()
        line = {
            "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "chain": f"steps i={NDIFFUSE - 1 - args.warmup}..{NDIFFUSE - args.warmup - args.steps} of the real seed-0 chain",
                       "global_samples": n_weak, "samples_per_gpu": n_local, "parallelism": f"sample-shard x{world}",
                       "exchange": "none" if world == 1 else "NVLink peer loads inside the tail kernels (symmetric memory)",
                       "l2": "flushed between steps (256 MiB memset, untimed" + ("; ranks re-aligned after the flush by an untimed stream-ordered NCCL all-reduce)" if world > 1 else ")"), "substeps_per_s": value * NFRAMES},
            "clocks": clocks,
            "e2e": {"value": n_weak * HSAMPLE / (e2e_ms * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": HNu * 4,
                    "d2h_bytes_per_step": HNu * 4 + 4},
            "gpu_launches": 3 * args.steps,
            "kernels": weak_breakdown,
            "roofline": {"bound": "hbm", "kernel": f"{summ.get('kernel', 'k_rollout_wpl<true,...>')} (fused sampling + rollouts)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": summ.get("dram_bytes_per_launch"), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kern_ms,
                         "note": "path is fp32-issue bound, not HBM bound (SURVEY F7): see roofline_fp32 / roofline_issue and DESIGN.md"},
        }
        if parity_ok is not None:
            line["parity_ok"] = parity_ok
        if strong is not None:
            line["strong"] = strong
        if solve is not None:
            line["e2e_solve"] = solve
        wi = summ.get("warp_instructions")
        clk = float((clocks or {}).get("sm_mhz") or 1965.0)
        if wi and n_local == NSAMPLE:
            peak_issue = 148 * 4 * clk * 1e6  # 1 warp-instruction per SM sub-partition per cycle
            line["roofline_issue"] = {"bound": "fp32 issue slots", "achieved": wi / kern_s, "peak": peak_issue, "unit": "warp-inst/s",
                                      "frac": wi / kern_s / peak_issue, "warp_instructions_per_launch": wi,
                                      "source": "profiles/rollout_kernel_summary.json (ncu smsp__inst_executed.sum)"}
        try:
            measured_tf = ops.ffma_peak(dev)
            flop = float(n_local) * HSAMPLE * NFRAMES * FLOP_PER_SUBSTEP
            nominal_tf = 148 * 128 * 2 * clk * 1e6 / 1e12
            line["roofline_fp32"] = {"bound": "fp32 pipe", "achieved": flop / kern_s / 1e12, "peak": measured_tf, "unit": "TFLOP/s",
                                     "frac": flop / kern_s / 1e12 / measured_tf, "peak_source": "measured in this run (mbd_ffma_peak: 16 "
                                     "independent FFMA chains per thread, 2048 threads per SM)", "nominal_peak": nominal_tf,
                                     "flop_per_sample_substep": FLOP_PER_SUBSTEP,
                                     "note": "algorithmic flops (mul, add 1; fma 2; div, rcp, sqrt 1); the device executes ~15 % more"}
        except Exception as ex:  # noqa: BLE001 - never lose the bench line over an explanatory field
            line["roofline_fp32"] = {"error": str(ex)}
        if world == 1 and not args.no_cpu_baseline:
            try:
                val, tcpu, threads, flags = time_cpu_oracle(args.cpu_samples, 5, 3)
                line["cpu_baseline"] = {"value": val, "unit": "env-steps/s", "cores": threads, "kind": "port",
                                        "sample": f"{args.cpu_samples} of {NSAMPLE} rollouts x {HSAMPLE} env steps per step, median of 5 steps "
                                                  f"after 3 warm-ups (CPU restatement: {flags}; JAX/Brax unavailable)"}
            except Exception as ex:  # noqa: BLE001
                line["cpu_baseline"] = {"error": f"{type(ex).__name__}: {ex}"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-samples", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-solve", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if 2 * args.steps + args.warmup + 2 >= NDIFFUSE:
        raise SystemExit("2*steps + warmup + 2 must be < Ndiffuse")
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs saves the outputs of the GPU arm; --impl reference times a sample of the rollouts only")
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
