"""MBD planner — drop-in for /root/reference/mbd/planners/mbd_planner.py.

Same `Args` fields, same recommended-parameter override, same `run_diffusion(args) -> rew_final`
signature, stdout lines and `results/{env}/mu_0ts.npy` artefact; the jitted `reverse_once` is
replaced by `DiffusionEngine.reverse_once` (hand-written sm_100a CUDA behind the C ABI).
Under torchrun (WORLD_SIZE > 1) the Nsample axis is sharded over ranks.

`run_diffusion_batch(args_list)` runs several independent solves (own seed and temperature; shared env, sizes, schedule
and demo flag) as one batch: the S solves share the three launches of every step, and each returns exactly what
`run_diffusion` returns for it alone.
"""
from __future__ import annotations

import contextlib
import io
import os
from dataclasses import dataclass

import numpy as np
import torch
import torch.distributed as dist

import mbd_b200
from mbd_b200 import ops, prng
from mbd_b200.planners.engine import DiffusionEngine, key_chain, make_schedule

try:  # tqdm is cosmetic
    from tqdm import tqdm
except Exception:  # noqa: BLE001
    tqdm = None


## load config
@dataclass
class Args:
    # exp
    seed: int = 0
    disable_recommended_params: bool = False
    not_render: bool = False
    # env
    env_name: str = (
        "ant"  # "humanoidstandup", "ant", "halfcheetah", "hopper", "walker2d", "car2d"
    )
    # diffusion
    Nsample: int = 2048  # number of samples
    Hsample: int = 50  # horizon
    Ndiffuse: int = 100  # number of diffusion steps
    temp_sample: float = 0.1  # temperature for sampling
    beta0: float = 1e-4  # initial beta
    betaT: float = 1e-2  # final beta
    enable_demo: bool = False


# recommended parameters (mbd_planner.py:45-63)
TEMP_RECOMMEND = {"ant": 0.1, "halfcheetah": 0.4, "hopper": 0.1, "humanoidstandup": 0.1, "humanoidrun": 0.1, "walker2d": 0.1,
                  "pushT": 0.2}
NDIFFUSE_RECOMMEND = {"pushT": 200, "humanoidrun": 300}
NSAMPLE_RECOMMEND = {"humanoidrun": 8192}
HSAMPLE_RECOMMEND = {"pushT": 40}


def apply_recommended_params(args: Args) -> Args:
    """mbd_planner.py:64-69 — mutates args in place exactly like the reference."""
    if not args.disable_recommended_params:
        args.temp_sample = TEMP_RECOMMEND.get(args.env_name, args.temp_sample)
        args.Ndiffuse = NDIFFUSE_RECOMMEND.get(args.env_name, args.Ndiffuse)
        args.Nsample = NSAMPLE_RECOMMEND.get(args.env_name, args.Nsample)
        args.Hsample = HSAMPLE_RECOMMEND.get(args.env_name, args.Hsample)
        if _is_main():   # one line per job, as in the single-process reference (every rank of a torchrun job runs this)
            print(f"override temp_sample to {args.temp_sample}")
    return args


def _is_main() -> bool:
    return not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0


def run_diffusion(args: Args, log_every: int = 10, return_trajectory: bool = False):
    rng = prng.PRNGKey(seed=args.seed)

    ## setup env
    apply_recommended_params(args)
    env = mbd_b200.envs.get_env(args.env_name)
    Nu = env.action_size

    rng, rng_reset = prng.split(rng)  # NOTE: rng_reset should never be changed.
    state_init = env.reset(rng_reset)

    ## run diffusion
    betas, alphas, alphas_bar, sigmas = make_schedule(args.beta0, args.betaT, args.Ndiffuse)
    if _is_main():
        print(f"init sigma = {sigmas[-1]:.2e}")

    engine = DiffusionEngine(env, args.Nsample, args.Hsample, args.temp_sample, args.enable_demo, state_init, Ndiffuse=args.Ndiffuse)
    HNu = args.Hsample * Nu
    # Everything the loop of mbd_planner.py:138-148 feeds into reverse_once is uploaded ONCE: the Y0s_rng chain
    # (rng, Y0s_rng = split(rng) per step, :103), sigmas[i] and the schedule scalars.  engine.Ybars row N-1 = YN = 0 and
    # row i-1 receives Ybar_{i-1}; one step is captured in a CUDA graph and replayed, nothing is copied to the host inside
    # the loop.
    rng_exp, rng = prng.split(rng)
    engine.load_schedule(key_chain(rng_exp, args.Ndiffuse), sigmas, alphas, alphas_bar)
    engine.set_step(args.Ndiffuse - 1)
    if os.environ.get("MBD_GRAPH", "1") != "0":
        engine.capture()
    steps = range(args.Ndiffuse - 1, 0, -1)
    pbar = tqdm(steps, desc="Diffusing") if (tqdm is not None and _is_main()) else None
    for n_done, i in enumerate(pbar if pbar is not None else steps):
        engine.step()
        if pbar is not None and (n_done % log_every == log_every - 1 or i == 1):
            # the reference formats rew every step (a device->host sync each step, mbd_planner.py:147);
            # here the sync is paid every `log_every` steps only
            pbar.set_postfix({"rew": f"{engine.rew_hist[i].item():.2e}"})
            engine.check_exchange()
    engine.check_exchange()
    Ybars = engine.Ybars
    Yi = Ybars[: args.Ndiffuse - 1].flip(0).reshape(args.Ndiffuse - 1, args.Hsample, Nu)  # jnp.array(Ybars) order

    if not args.not_render and _is_main():
        _save_results(args, env, state_init, Yi)
    rew_final = final_reward(env, engine, Yi[-1])
    if return_trajectory:
        return rew_final, Yi
    return rew_final


# Args fields that every solve of one batch must share (they size the buffers or are part of the shared schedule)
BATCH_SHARED_FIELDS = ("env_name", "Nsample", "Hsample", "Ndiffuse", "beta0", "betaT", "enable_demo")


def _prepare_batch(args_list):
    """apply_recommended_params to every Args (in place, as run_diffusion does) and check the shared fields; returns the
    stdout text each call produced, so the caller can print it at the point the sequential loop would.  No GPU call."""
    args_list = list(args_list)
    if not args_list:
        raise ValueError("run_diffusion_batch needs at least one Args")
    printed = []
    for a in args_list:
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            apply_recommended_params(a)
        printed.append(buf.getvalue())
    for field in BATCH_SHARED_FIELDS:
        vals = [getattr(a, field) for a in args_list]
        if any(v != vals[0] for v in vals[1:]):
            raise ValueError(f"run_diffusion_batch: every solve must share `{field}` (got {vals})")
    return args_list, printed


def run_diffusion_batch(args_list, log_every: int = 10, return_trajectory: bool = False):
    """`[run_diffusion(a) for a in args_list]` as ONE batch of independent solves on one GPU.

    The solves must agree on env_name, Nsample, Hsample, Ndiffuse, beta0, betaT and enable_demo (after the recommended
    parameters are applied; ValueError otherwise); each keeps its own seed (reset noise and key chain) and temp_sample.
    All of them run through one captured graph, three launches per diffusion step.  Returns the list of final rewards, or
    with return_trajectory the list of (rew_final, Yi) — bit for bit what the sequential loop returns.  Prints the same
    lines and writes the same results/{env}/ files as that loop (later solves overwrite earlier ones)."""
    args_list, printed = _prepare_batch(args_list)
    ops._lib.require_gpu()
    a0 = args_list[0]
    env = mbd_b200.envs.get_env(a0.env_name)
    Nu = env.action_size
    betas, alphas, alphas_bar, sigmas = make_schedule(a0.beta0, a0.betaT, a0.Ndiffuse)
    states, keys = [], []
    for a, text in zip(args_list, printed):
        # run_diffusion's key handling, solve by solve
        rng = prng.PRNGKey(seed=a.seed)
        if _is_main():
            print(text, end="")
        rng, rng_reset = prng.split(rng)
        states.append(env.reset(rng_reset))
        if _is_main():
            print(f"init sigma = {sigmas[-1]:.2e}")
        rng_exp, rng = prng.split(rng)
        keys.append(key_chain(rng_exp, a.Ndiffuse))
    S = len(args_list)
    engine = DiffusionEngine(env, a0.Nsample, a0.Hsample, [a.temp_sample for a in args_list], a0.enable_demo,
                             states if S > 1 else states[0], Ndiffuse=a0.Ndiffuse)
    engine.load_schedule(np.stack(keys) if S > 1 else keys[0], sigmas, alphas, alphas_bar)
    engine.set_step(a0.Ndiffuse - 1)
    if os.environ.get("MBD_GRAPH", "1") != "0":
        engine.capture()
    steps = range(a0.Ndiffuse - 1, 0, -1)
    pbar = tqdm(steps, desc=f"Diffusing x{S}") if (tqdm is not None and _is_main()) else None
    for n_done, i in enumerate(pbar if pbar is not None else steps):
        engine.step()
        if pbar is not None and (n_done % log_every == log_every - 1 or i == 1):
            pbar.set_postfix({"rew": f"{engine.solve(0).rew_hist[i].item():.2e}"})
    out = []
    for s, a in enumerate(args_list):
        v = engine.solve(s)
        Yi = v.Ybars[: a.Ndiffuse - 1].flip(0).reshape(a.Ndiffuse - 1, a.Hsample, Nu)
        if not a.not_render and _is_main():
            _save_results(a, env, states[s], Yi)
        rew_final = final_reward(env, engine, Yi[-1], state_init=v.state_init)
        out.append((rew_final, Yi) if return_trajectory else rew_final)
    return out


def _save_results(args: Args, env, state_init, Yi: torch.Tensor):
    """the results/{env}/ artefacts of one solve (mbd_planner.py:157-178)"""
    path = f"{mbd_b200.__path__[0]}/../results/{args.env_name}"
    if not os.path.exists(path):
        os.makedirs(path)
    np.save(f"{path}/mu_0ts.npy", Yi.cpu().numpy())
    if args.env_name == "car2d":
        _render_car2d(env, state_init, Yi[-1].cpu().numpy(), args, path)
    elif env.kind in ("xpbd", "pusht"):
        # mbd_planner.py:168-178: rollout.html = brax.io.html.render(sys with opt.timestep = env.dt, rollout).  The same
        # page (and the JSON document inside it, which vis_diffusion.py / brax.io.html.render_from_json consume) is written
        # by mbd_b200.io.brax_json; rollout_states.npz keeps the plain arrays
        from ..io import brax_json
        from ..utils import rollout_states, trajectory_arrays
        rollout = rollout_states(env.step, state_init, Yi[-1].cpu().numpy())
        with open(f"{path}/rollout.html", "w") as f:
            f.write(brax_json.render(env.sys, rollout, env.dt))
        with open(f"{path}/rollout.json", "w") as f:
            f.write(brax_json.dumps(env.sys, rollout, env.dt))
        np.savez(f"{path}/rollout_states.npz", **trajectory_arrays(env, rollout))


def final_reward(env, engine: DiffusionEngine, us: torch.Tensor, state_init: torch.Tensor = None) -> float:
    """rollout_us(state_init, Yi[-1])[0].mean()  (mbd_planner.py:179-180) — one n=1 launch.  state_init: the device state
    of one solve of a batched engine (default: the engine's own state)."""
    us = us.reshape(1, engine.H, engine.Nu).contiguous()
    st = engine.state_init if state_init is None else state_init
    if env.kind == "xpbd":
        out = ops.rollout(engine.model, st, us)
    elif env.kind == "pusht":
        out = ops.pusht_rollout(engine.params_car, st, us)
    else:
        out = ops.car2d_rollout(engine.params_car, st, us)
    return float(out["rews"][0].item())


def _render_car2d(env, state_init, us, args, path):
    try:
        import matplotlib
        matplotlib.use("Agg")
        from matplotlib import pyplot as plt
    except Exception:  # noqa: BLE001
        return
    fig, ax = plt.subplots(1, 1, figsize=(3, 3))
    xs = [np.asarray(state_init.pipeline_state)]
    state = state_init
    for t in range(us.shape[0]):
        state = env.step(state, us[t])
        xs.append(np.asarray(state.pipeline_state))
    env.render(ax, np.stack(xs))
    if args.enable_demo:
        ax.plot(env.xref[:, 0], env.xref[:, 1], "g--", label="RRT path")
    ax.legend()
    plt.savefig(f"{path}/rollout.png")


def _maybe_init_distributed():
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and not dist.is_initialized():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")


if __name__ == "__main__":
    import tyro

    _maybe_init_distributed()
    rew_final = run_diffusion(args=tyro.cli(Args))
    if _is_main():
        print(f"final reward = {rew_final:.2e}")
