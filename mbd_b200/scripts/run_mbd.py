"""Seed and temperature sweeps — port of the reference's mbd/scripts/run_mbd.py.

    python -m mbd_b200.scripts.run_mbd --algo mbd --mode seed --env_name hopper

mode=seed runs 8 seeds (not_render=True); mode=temp runs the 8 temperatures of the reference at seed 0 with
disable_recommended_params=True.  The printed lines are the reference's: `rew: m \\pm s` and `time: m \\pm s` (seed),
`rews: [...]` and `best_temp: t` (temp).

One difference: with algo=mbd the 8 solves run as ONE batch on the GPU (`run_diffusion_batch`: shared launches, every
solve bit-identical to running it alone), so there are no per-solve wall times.  `time:` then prints the batch wall
clock divided by the number of solves with `\\pm 0.00`, and one extra line `batch: S solves in X s` gives the batch
wall clock itself.  algo=path_integral keeps the reference's sequential loop over run_path_integral.
"""
from __future__ import annotations

from dataclasses import dataclass
from time import time

import numpy as np

from mbd_b200.planners import mbd_planner, path_integral

SEEDS = 8
TEMPS = np.array([0.01, 0.03, 0.06, 0.1, 0.2, 0.4, 0.6, 0.8])


@dataclass
class Args:
    algo: str = "mbd"  # path_integral, mbd
    update_method: str = "mppi"  # softmax, cma-es, cem
    mode: str = "seed"  # temp
    env_name: str = "ant"


def _run_batch(args_list):
    t0 = time()
    rews = mbd_planner.run_diffusion_batch(args_list)
    wall = time() - t0
    print(f"batch: {len(args_list)} solves in {wall:.2f} s")
    return rews, wall


def run_multiple_seed(args: Args):
    if args.algo == "mbd":
        rews, wall = _run_batch([mbd_planner.Args(seed=seed, env_name=args.env_name, not_render=True) for seed in range(SEEDS)])
        times = np.full(SEEDS, wall / SEEDS)
    elif args.algo == "path_integral":
        rews, times = [], []
        for seed in range(SEEDS):
            t0 = time()
            local_args = path_integral.Args(seed=seed, env_name=args.env_name, update_method=args.update_method)
            rews.append(path_integral.run_path_integral(local_args))
            times.append(time() - t0)
    else:
        raise NotImplementedError(args.algo)
    rews, times = np.array(rews), np.array(times)
    print(f"rew: {rews.mean():.2f} \\pm {rews.std():.2f}")
    print(f"time: {times.mean():.2f} \\pm {times.std():.2f}")
    return rews


def run_multiple_temp(args: Args):
    if args.algo == "mbd":
        rews, _ = _run_batch([mbd_planner.Args(seed=0, env_name=args.env_name, temp_sample=float(temp), not_render=True,
                                               disable_recommended_params=True) for temp in TEMPS])
    elif args.algo == "path_integral":
        rews = [path_integral.run_path_integral(path_integral.Args(seed=0, env_name=args.env_name, temp_sample=float(temp)))
                for temp in TEMPS]
    else:
        raise NotImplementedError(args.algo)
    rews = np.array(rews)
    best_temp = TEMPS[np.argmax(rews)]
    print(f"rews: {rews}")
    print(f"best_temp: {best_temp:.2f}")
    return rews


def main(args: Args):
    if args.mode == "seed":
        return run_multiple_seed(args)
    if args.mode == "temp":
        return run_multiple_temp(args)
    raise ValueError(f"mode must be seed or temp, got {args.mode!r}")


if __name__ == "__main__":
    import tyro

    main(tyro.cli(Args))
