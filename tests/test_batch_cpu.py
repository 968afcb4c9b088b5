"""Batched solves without a GPU: shared-field validation of run_diffusion_batch, the C-ABI offsets of the batch fields of
mbd_step_plan, the run_mbd port's defaults, and the no-CPU-fallback failure mode of the batch API."""
import ctypes
import dataclasses

import numpy as np
import pytest
import torch

from mbd_b200 import _lib
from mbd_b200.planners import mbd_planner
from mbd_b200.scripts import run_mbd

SHARED_MISMATCH = [
    ("env_name", dict(env_name="hopper")),
    ("Nsample", dict(Nsample=128)),
    ("Hsample", dict(Hsample=20)),
    ("Ndiffuse", dict(Ndiffuse=7)),
    ("beta0", dict(beta0=2e-4)),
    ("betaT", dict(betaT=2e-2)),
    ("enable_demo", dict(enable_demo=True)),
]


@pytest.mark.parametrize("field,override", SHARED_MISMATCH, ids=[f for f, _ in SHARED_MISMATCH])
def test_batch_rejects_mismatched_shared_field(field, override):
    base = dict(env_name="car2d", not_render=True, disable_recommended_params=True, Nsample=64, Hsample=10, Ndiffuse=5)
    args = [mbd_planner.Args(seed=0, **base), mbd_planner.Args(seed=1, **{**base, **override})]
    with pytest.raises(ValueError, match=field):
        mbd_planner.run_diffusion_batch(args)


def test_batch_mismatch_after_recommended_params():
    """the check runs on the arguments as the solves would see them: pushT's recommended Hsample (40) against the
    default one (50) of a solve with disable_recommended_params is a mismatch"""
    a = mbd_planner.Args(seed=0, env_name="pushT", not_render=True)
    b = mbd_planner.Args(seed=1, env_name="pushT", not_render=True, disable_recommended_params=True)
    with pytest.raises(ValueError, match="Hsample"):
        mbd_planner.run_diffusion_batch([a, b])


def test_batch_rejects_empty():
    with pytest.raises(ValueError):
        mbd_planner.run_diffusion_batch([])


def test_batch_offsets_match_ctypes_mirror():
    out = np.zeros(8, np.int32)
    n = _lib.lib().mbd_abi_batch_offsets(out.ctypes.data_as(_lib.c_i32p), 8)
    P = _lib.StepPlan
    assert n == 3
    assert out[:3].tolist() == [P.n_solves.offset, P.n_diffuse.offset, P.temps_dev.offset]
    # appended after the last field of the single-solve plan
    assert P.n_solves.offset >= P.timeout_cycles.offset + 8


def test_run_mbd_args_match_reference_defaults():
    a = run_mbd.Args()
    assert dataclasses.asdict(a) == dict(algo="mbd", update_method="mppi", mode="seed", env_name="ant")
    assert run_mbd.SEEDS == 8
    assert run_mbd.TEMPS.tolist() == [0.01, 0.03, 0.06, 0.1, 0.2, 0.4, 0.6, 0.8]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_batch_has_no_cpu_fallback():
    args = [mbd_planner.Args(seed=k, env_name="car2d", not_render=True, Nsample=64, Hsample=10, Ndiffuse=5) for k in range(2)]
    with pytest.raises(_lib.MbdError):
        mbd_planner.run_diffusion_batch(args)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_run_mbd_has_no_cpu_fallback():
    with pytest.raises(_lib.MbdError):
        run_mbd.main(run_mbd.Args(env_name="car2d"))


def test_step_plan_default_is_one_solve():
    p = _lib.StepPlan()
    assert p.n_solves == 0 and p.n_diffuse == 0 and not p.temps_dev
    assert ctypes.sizeof(p) == _lib.StepPlan.temps_dev.offset + 8
