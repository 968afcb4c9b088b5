"""Batched solves against solves run one after another, on one GPU.

    python scripts/gpu_batch_timing.py build-parent [REV]   # needs nvcc + git: mbd_b200/_C/libmbd_b200_parent.so from REV (HEAD)
    python scripts/gpu_batch_timing.py run [OUT.json]       # GPU: batch sweep + run_mbd wall clocks + single-solve A/B

`run` writes one JSON document (default profiles/r03_batch_timing.json) with the card's name and power limit, read in the
same process, and three parts:
  step    device time of ONE diffusion step (CUDA events around graph replays after warm-up, median of 60 steps) of a batch
          of S solves, next to S x the single-solve step time measured in the same process;
  run_mbd wall clock of `run_mbd --mode seed` (8 seeds, recommended parameters) as one batch and as the sequential loop of
          run_diffusion, twice each, alternating; the final rewards of both must be equal;
  ab      single-solve step time of this tree's library and of the parent's, alternated in fresh subprocesses (3 rounds).
"""
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
PARENT_SO = os.path.join(ROOT, "mbd_b200", "_C", "libmbd_b200_parent.so")

STEP_CONFIGS = [("car2d", 64, 40, (1, 2, 4, 8)), ("hopper", 1024, 50, (1, 2, 4, 8)), ("ant", 2048, 50, (1, 2, 4, 8)),
                ("pushT", 2048, 40, (1, 2, 4, 8)), ("humanoidrun", 1024, 50, (1, 2, 4)), ("humanoidrun", 8192, 50, (1, 2, 4))]
AB_CONFIGS = [("humanoidrun", 8192, 50), ("hopper", 1024, 50), ("car2d", 64, 40)]
RUN_MBD_ENVS = ["car2d", "hopper", "ant", "pushT", "humanoidrun"]


def build_parent(rev: str):
    from mbd_b200 import build as b
    with tempfile.TemporaryDirectory() as td:
        files = subprocess.run(["git", "-C", ROOT, "ls-tree", "-r", "--name-only", rev, "mbd_b200/csrc", "include"],
                               capture_output=True, text=True, check=True).stdout.split()
        for f in files:
            os.makedirs(os.path.join(td, os.path.dirname(f)), exist_ok=True)
            with open(os.path.join(td, f), "wb") as fh:
                fh.write(subprocess.run(["git", "-C", ROOT, "show", f"{rev}:{f}"], capture_output=True, check=True).stdout)
        flags = [x for x in b.NVCC_FLAGS if not x.startswith("-I")] + ["-I" + os.path.join(td, "include"), "-I" + os.path.join(td, "mbd_b200", "csrc")]
        subprocess.run([b.nvcc_path()] + flags + ["-o", PARENT_SO, os.path.join(td, "mbd_b200", "csrc", "mbd_b200.cu")], check=True)
    print("built", PARENT_SO, "from", rev)


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else None)


def step_ms(name, N, H, S, nsteps=60, warm=10):
    """median device time of one step of a batch of S solves (S = 1: the single-solve engine), graph replays"""
    import numpy as np
    import torch
    import mbd_b200
    from mbd_b200 import prng
    from mbd_b200.planners import engine as eng
    env = mbd_b200.envs.get_env(name)
    Nd = nsteps + warm + 2
    states = [env.reset(prng.split(prng.PRNGKey(s))[1]) for s in range(S)]
    temps = [0.1] * S
    keys = np.stack([eng.key_chain(prng.split(prng.PRNGKey(s))[0], Nd) for s in range(S)])
    _, alphas, alphas_bar, sigmas = eng.make_schedule(1e-4, 1e-2, Nd)
    e = eng.DiffusionEngine(env, N, H, temps if S > 1 else temps[0], False, states if S > 1 else states[0], Ndiffuse=Nd)
    e.load_schedule(keys if S > 1 else keys[0], sigmas, alphas, alphas_bar)
    e.set_step(Nd - 1)
    e.capture()
    for _ in range(warm):
        e.step()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(nsteps + 1)]
    ev[0].record()
    for k in range(nsteps):
        e.step()
        ev[k + 1].record()
    torch.cuda.synchronize()
    return statistics.median(ev[k].elapsed_time(ev[k + 1]) for k in range(nsteps))


def run_mbd_walls(name):
    import torch
    from mbd_b200.planners import mbd_planner as mp
    mp.tqdm = None
    mk = lambda k: mp.Args(seed=k, env_name=name, not_render=True)   # noqa: E731
    out = dict(seq_s=[], batch_s=[])
    rews = {}
    for _ in range(2):
        for mode in ("seq", "batch"):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                r = [mp.run_diffusion(mk(k)) for k in range(8)] if mode == "seq" else mp.run_diffusion_batch([mk(k) for k in range(8)])
            torch.cuda.synchronize()
            out[f"{mode}_s"].append(time.perf_counter() - t0)
            rews[mode] = r
    out["rewards_equal"] = rews["seq"] == rews["batch"]
    out["speedup_best"] = min(out["seq_s"]) / min(out["batch_s"])
    return out


def ab_child(which):
    """prints one JSON line: single-solve step ms of each AB config with this tree's (new) or the parent's library"""
    if which == "parent":
        import ctypes
        import types
        from mbd_b200 import build as b

        class Lenient(ctypes.CDLL):   # the parent library lacks the symbols this tree added
            def __getattr__(self, n):
                try:
                    return super().__getattr__(n)
                except AttributeError:
                    return types.SimpleNamespace()
        ctypes.CDLL = Lenient
        b.OUT = PARENT_SO
        b.is_stale = lambda: False
    print(json.dumps({f"{n} {N}x{H}": step_ms(n, N, H, 1) for n, N, H in AB_CONFIGS}), flush=True)


def main_run(out_path):
    import torch
    torch.cuda.set_device(0)
    res = dict(gpu=gpu_info(), step=[], run_mbd={}, ab=None)
    for name, N, H, Ss in STEP_CONFIGS:
        single = step_ms(name, N, H, 1)
        for S in Ss:
            t = single if S == 1 else step_ms(name, N, H, S)
            row = dict(env=name, N=N, H=H, S=S, batch_step_ms=t, single_step_ms=single, S_x_single_ms=S * single,
                       speedup=S * single / t, not_slower=t <= S * single)
            res["step"].append(row)
            print(json.dumps(row), flush=True)
    for name in RUN_MBD_ENVS:
        res["run_mbd"][name] = run_mbd_walls(name)
        print(name, json.dumps(res["run_mbd"][name]), flush=True)
    if os.path.exists(PARENT_SO):
        ab = dict(new=[], parent=[])
        for _ in range(3):
            for which in ("parent", "new"):
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "ab-child", which], capture_output=True, text=True, cwd=ROOT)
                line = [l for l in p.stdout.splitlines() if l.startswith("{")]
                ab[which].append(json.loads(line[-1]) if line else p.stderr[-2000:])
        summ = {}
        for k in ab["new"][0] if isinstance(ab["new"][0], dict) else []:
            nv = [r[k] for r in ab["new"]]
            pv = [r[k] for r in ab["parent"]]
            summ[k] = dict(new_ms=nv, parent_ms=pv, new_spread_ms=max(nv) - min(nv), parent_spread_ms=max(pv) - min(pv),
                           median_diff_ms=statistics.median(nv) - statistics.median(pv))
        ab["summary"] = summ
        res["ab"] = ab
        print(json.dumps(summ, indent=1), flush=True)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    mode = sys.argv[1]
    if mode == "build-parent":
        build_parent(sys.argv[2] if len(sys.argv) > 2 else "HEAD")
    elif mode == "ab-child":
        ab_child(sys.argv[2])
    elif mode == "run":
        main_run(sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "profiles", "r03_batch_timing.json"))
    else:
        raise SystemExit(__doc__)
