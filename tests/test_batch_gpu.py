"""Batched solves on the GPU: S independent solves in the same three launches per step give, solve for solve, exactly the
bits of S separate single-solve engines (each with its own initial state, key chain and temperature) — over two steps, for
every env family, every rollout-kernel variant and under CUDA-graph replay; run_diffusion_batch equals the sequential
loop of run_diffusion; the launch refuses what it does not cover; one batch is tied to the numpy planner oracle."""
import ctypes

import numpy as np
import pytest
import torch

import mbd_b200
from mbd_b200 import _lib, ops, prng
from mbd_b200.planners import engine as eng
from mbd_b200.planners.mbd_planner import Args, run_diffusion, run_diffusion_batch
from oracle import planner as opl
from tests.conftest import assert_bit_exact

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def N(t):
    return t.detach().cpu().numpy()


def _states(env, S):
    """S distinct initial states: the env's reset with solve-specific keys (car2d's reset is deterministic, so its start
    point is nudged per solve)"""
    out = []
    for s in range(S):
        st = env.reset(prng.split(prng.PRNGKey(s + 1))[1])
        if env.kind == "car2d":
            raw = np.asarray(st.pipeline_state, np.float32) + np.float32(0.01 * s)
        else:
            raw = np.array(st.pipeline_state.raw, np.float32)
        out.append(raw)
    return out


def _setup(env, S, Nn, H, Nd, demo):
    states = _states(env, S)
    temps = [0.05 + 0.03 * s for s in range(S)]
    keys = [eng.key_chain(np.uint32([11 + s, 3 * s + 5]), Nd) for s in range(S)]
    _, alphas, alphas_bar, sigmas = eng.make_schedule(1e-4, 1e-2, Nd)
    sched = (sigmas, alphas, alphas_bar)
    b = eng.DiffusionEngine(env, Nn, H, temps, demo, states, Ndiffuse=Nd)
    b.load_schedule(np.stack(keys), *sched)
    b.set_step(Nd - 1)
    singles = []
    for s in range(S):
        e = eng.DiffusionEngine(env, Nn, H, temps[s], demo, states[s], Ndiffuse=Nd)
        e.load_schedule(keys[s], *sched)
        e.set_step(Nd - 1)
        singles.append(e)
    return b, singles


def _compare(b, singles, what):
    torch.cuda.synchronize()
    for s, e in enumerate(singles):
        v = b.solve(s)
        tag = f"{what} solve {s}"
        assert_bit_exact(N(v.Y0s), N(e.Y0s), f"{tag}: Y0s")
        assert_bit_exact(N(v.rews_local), N(e.rews_local), f"{tag}: rews")
        if e.logpd_local is not None:
            assert_bit_exact(N(v.logpd_local), N(e.logpd_local), f"{tag}: logpd")
        assert_bit_exact(N(v.weights), N(e.weights), f"{tag}: weights")
        assert_bit_exact(N(v.scalars), N(e.scalars), f"{tag}: scalars")
        assert_bit_exact(N(v.Ybars), N(e.Ybars), f"{tag}: Ybars")
        assert_bit_exact(N(v.rew_hist), N(e.rew_hist), f"{tag}: rew_hist")
        assert int(v.ctl[0].item()) == int(e.ctl[0].item()), f"{tag}: step counter"


def _two_steps(b, singles):
    for _ in range(2):
        b.step()
        for e in singles:
            e.step()


ENVS = [("car2d", False, 200, 12), ("car2d", True, 200, 12), ("humanoidrun", False, 100, 10), ("hopper", False, 100, 10),
        ("humanoidtrack", True, 100, 10), ("pushT", False, 100, 8)]


@pytest.mark.parametrize("S", [1, 3, 8])
@pytest.mark.parametrize("name,demo,Nn,H", ENVS, ids=[f"{n}{'-demo' if d else ''}" for n, d, _, _ in ENVS])
def test_batch_equals_separate_engines(name, demo, Nn, H, S):
    env = mbd_b200.envs.get_env(name)
    Nd = 6
    b, singles = _setup(env, S, Nn, H, Nd, demo)
    assert b.S == S
    if S == 1:
        assert b.Y0s.shape == singles[0].Y0s.shape and b.Ybars.shape == singles[0].Ybars.shape
    _two_steps(b, singles)
    _compare(b, singles, f"{name} S={S}")
    assert int(b.solve(0).ctl[0].item()) == Nd - 3


@pytest.mark.parametrize("variant", [1, 2, 3, 5, 6, 8, 9])
def test_batch_every_kernel_variant(variant):
    env = mbd_b200.envs.get_env("humanoidrun")
    ops.set_kernel_variant(variant)
    try:
        b, singles = _setup(env, 3, 100, 8, 5, False)   # 100 samples: not a multiple of 64 (ragged last CTA)
        _two_steps(b, singles)
        _compare(b, singles, f"variant {variant}")
    finally:
        ops.set_kernel_variant(0)


def test_batch_graph_replay_equals_direct_launches():
    env = mbd_b200.envs.get_env("hopper")
    Nd = 6
    g, _ = _setup(env, 4, 128, 10, Nd, False)
    d, _ = _setup(env, 4, 128, 10, Nd, False)
    g.capture()
    for _ in range(3):
        g.step()
        d.step()
    torch.cuda.synchronize()
    assert_bit_exact(N(g.Ybars), N(d.Ybars), "graph vs direct: Ybars")
    assert_bit_exact(N(g.rew_hist), N(d.rew_hist), "graph vs direct: rew_hist")
    assert torch.equal(g.ctl[:, 0], d.ctl[:, 0]) and int(g.ctl[0, 0].item()) == Nd - 4


def _strip_tqdm(text):
    return [l for l in text.splitlines() if l.strip() and "Diffusing" not in l]


def test_run_diffusion_batch_car2d_equals_sequential_loop(capsys):
    mk = lambda k: Args(seed=k, env_name="car2d", not_render=True)   # noqa: E731
    seq = [run_diffusion(mk(k), return_trajectory=True) for k in range(4)]
    out_seq = capsys.readouterr().out
    bat = run_diffusion_batch([mk(k) for k in range(4)], return_trajectory=True)
    out_bat = capsys.readouterr().out
    assert [r for r, _ in bat] == [r for r, _ in seq]
    for (_, yb), (_, ys) in zip(bat, seq):
        assert_bit_exact(N(yb), N(ys), "trajectory")
    assert _strip_tqdm(out_bat) == _strip_tqdm(out_seq)
    assert run_diffusion_batch([mk(k) for k in range(4)]) == [r for r, _ in seq]


def test_run_diffusion_batch_hopper_temperature_sweep(capsys):
    mk = lambda t: Args(seed=0, env_name="hopper", not_render=True, disable_recommended_params=True, Nsample=256, Hsample=20,  # noqa: E731
                        Ndiffuse=8, temp_sample=t)
    temps = [0.05, 0.1, 0.4]
    seq = [run_diffusion(mk(t), return_trajectory=True) for t in temps]
    out_seq = capsys.readouterr().out
    bat = run_diffusion_batch([mk(t) for t in temps], return_trajectory=True)
    out_bat = capsys.readouterr().out
    assert [r for r, _ in bat] == [r for r, _ in seq]
    for (_, yb), (_, ys) in zip(bat, seq):
        assert_bit_exact(N(yb), N(ys), "trajectory")
    assert _strip_tqdm(out_bat) == _strip_tqdm(out_seq)


def test_step_launch_refuses_uncovered_batches():
    env = mbd_b200.envs.get_env("car2d")
    b, _ = _setup(env, 2, 64, 8, 4, False)
    peers = (ctypes.c_uint64 * 2)(1, 2)

    def refused(**fields):
        p = _lib.StepPlan.from_buffer_copy(b._plan_c)
        for k, v in fields.items():
            setattr(p, k, v)
        rc = _lib.lib().mbd_step_launch(ctypes.byref(p), ops._stream())
        return rc, _lib.lib().mbd_last_error().decode()

    rc, msg = refused(P=2, rank=0, peer_base_ptrs=ctypes.cast(peers, ctypes.POINTER(ctypes.c_uint64)))
    assert rc == -1 and "cannot be sharded" in msg
    rc, msg = refused(temps_dev=None)
    assert rc == -1 and "temps_dev" in msg
    rc, msg = refused(n_diffuse=1)
    assert rc == -1 and "n_diffuse" in msg
    rc, msg = refused(n_solves=-1)
    assert rc == -1 and "n_solves" in msg
    with pytest.raises(ops.MbdError):
        eng.DiffusionEngine(env, 64, 8, [0.1, 0.2], False, _states(env, 2), emulate=(1, 0, None))


def test_batch_car2d_vs_oracle(orc):
    """one batched step of three car2d solves against the numpy planner oracle, solve by solve (rtol 1e-4)"""
    car = mbd_b200.envs.get_env("car2d")
    S, Nn, H, Nd = 3, 256, 50, 10
    states = _states(car, S)
    temps = [0.05, 0.1, 0.3]
    keys = [eng.key_chain(np.uint32([21 + s, 2]), Nd) for s in range(S)]
    _, alphas, alphas_bar, sigmas = opl.make_schedule(1e-4, 1e-2, Nd)
    b = eng.DiffusionEngine(car, Nn, H, temps, False, states, Ndiffuse=Nd)
    b.load_schedule(np.stack(keys), sigmas, alphas, alphas_bar)
    b.set_step(Nd - 1)
    b.step()
    torch.cuda.synchronize()
    i = Nd - 1
    for s in range(S):
        oenv = opl.OracleEnv("car2d", 2, params=car.params, x0=states[s])
        ref = opl.reverse_once(oenv, keys[s][i], Nn, H, float(sigmas[i]), np.zeros(H * 2, np.float32), temps[s], alphas, alphas_bar, i)
        v = b.solve(s)
        assert_bit_exact(N(v.Y0s), ref["Y0s"], f"solve {s}: Y0s"); assert_bit_exact(N(v.rews_local), ref["rews"], f"solve {s}: rews")
        for got, exp, what in ((N(v.weights), ref["weights"], "weights"), (N(v.Ybars[i - 1]), ref["Ybar_im1"], "Ybar_im1"),
                               (N(v.scalars)[0], ref["rew_mean"], "rews.mean()")):
            got, exp = np.asarray(got, np.float64), np.asarray(exp, np.float64)
            err = np.abs(got - exp).max() / max(np.abs(exp).max(), 1e-6)
            assert err <= 1e-4, f"solve {s} {what}: {err:.3e}"
