"""Small workloads for compute-sanitizer (racecheck / synccheck / memcheck): every rollout kernel variant on 64 samples x 5
env steps of humanoidrun (plus hopper for the slide-dof path and the generic instantiation), one full diffusion step (cluster
statistics kernel + last-CTA update), two emulated ranks exchanging through peer loads, and a batched step of three solves
(hopper and humanoidrun: solve axis on every launch, one cluster per solve, per-solve tickets).
    compute-sanitizer --tool racecheck python scripts/gpu_sanitize.py"""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import mbd_b200
from mbd_b200 import ops, prng
from mbd_b200.planners import engine as eng

which = sys.argv[1] if len(sys.argv) > 1 else "all"
env = mbd_b200.envs.get_env("humanoidrun")
st = env.reset(prng.split(prng.PRNGKey(0))[1]).pipeline_state.raw
m = env.device_model(torch.device("cuda:0"))
sti = torch.as_tensor(st, device="cuda:0")
n, H = 64, 5
us = torch.as_tensor(np.clip(np.random.default_rng(0).normal(size=(n, H, 17)), -1, 1).astype(np.float32), device="cuda:0")
if which in ("all", "rollout"):
    ref = None
    for v in (2, 1, 3, 5, 6, 8, 9):
        ops.set_kernel_variant(v)
        out = ops.rollout(m, sti, us, want_final=True)["final"].cpu().numpy()
        ref = out if ref is None else ref
        print("variant", v, "bit-identical:", bool(np.array_equal(out, ref)), flush=True)
    ops.set_kernel_variant(0)
    hop = mbd_b200.envs.get_env("hopper")
    hs = torch.as_tensor(hop.reset(prng.split(prng.PRNGKey(0))[1]).pipeline_state.raw, device="cuda:0")
    hu = torch.as_tensor(np.clip(np.random.default_rng(1).normal(size=(n, H, 3)), -1, 1).astype(np.float32), device="cuda:0")
    a = None
    for v in (2, 1):
        ops.set_kernel_variant(v)
        o = ops.rollout(hop.device_model(torch.device("cuda:0")), hs, hu, want_final=True)["final"].cpu().numpy()
        a = o if a is None else a
        print("hopper variant", v, "bit-identical:", bool(np.array_equal(o, a)), flush=True)
    ops.set_kernel_variant(0)
if which in ("all", "rollout", "pusht"):
    # pushT kernel (one sample per thread, constraint rows and the padded solver systems in registers / local memory): a scripted
    # push that touches both boxes (8-row system) plus random actions, and two diffusion steps through the step API
    pt = mbd_b200.envs.get_env("pushT")
    x0 = pt.reset(prng.split(prng.PRNGKey(0))[1]).pipeline_state.raw.copy(); x0[0:2] = [-0.21, 0.0]
    pu = np.clip(np.random.default_rng(2).normal(size=(70, 8, 2)) * 0.8 + [0.6, 0.1], -1.5, 1.5).astype(np.float32)
    o = ops.pusht_rollout(pt.device_params(), torch.as_tensor(x0, device="cuda:0"), torch.as_tensor(pu, device="cuda:0"), want_final=True, want_traj=True)
    print("pushT rollouts finite:", bool(torch.isfinite(o["final"]).all().item()), "slider moved:", float(o["final"][:, 2].abs().max().item()), flush=True)
    _, al, ab, sg = eng.make_schedule(1e-4, 1e-2, 6)
    ep = eng.DiffusionEngine(pt, 128, 8, 0.2, False, x0, Ndiffuse=6)
    ep.load_schedule(eng.key_chain(np.uint32([3, 4]), 6), sg, al, ab); ep.set_step(5)
    ep.step(); ep.step(); torch.cuda.synchronize()
    print("pushT steps done, ctl.i =", int(ep.ctl[0].item()), flush=True)
if which in ("all", "step"):
    Nd = 6
    _, alphas, alphas_bar, sigmas = eng.make_schedule(1e-4, 1e-2, Nd)
    keys = eng.key_chain(np.uint32([1, 2]), Nd)
    e = eng.DiffusionEngine(env, 128, H, 0.1, False, st, Ndiffuse=Nd)
    e.load_schedule(keys, sigmas, alphas, alphas_bar); e.set_step(Nd - 1)
    e.step(); e.step()
    torch.cuda.synchronize()
    print("single-rank steps done, ctl.i =", int(e.ctl[0].item()), flush=True)
    ranks = eng.DiffusionEngine.make_emulated_ranks(env, 128, H, 0.1, False, st, 2, Ndiffuse=Nd)
    for r in ranks:
        r.load_schedule(keys, sigmas, alphas, alphas_bar); r.set_step(Nd - 1)
    eng.DiffusionEngine.step_emulated_ranks(ranks); eng.DiffusionEngine.step_emulated_ranks(ranks)
    torch.cuda.synchronize()
    print("emulated 2-rank steps equal the single-rank ones:", bool(torch.equal(ranks[0].Ybars, e.Ybars) and torch.equal(ranks[1].Ybars, e.Ybars)),
          "err", int(ranks[0].ctl[2].item()), flush=True)
if which in ("all", "batch"):
    Nd = 6
    _, alphas, alphas_bar, sigmas = eng.make_schedule(1e-4, 1e-2, Nd)
    for name in ("hopper", "humanoidrun"):
        be = mbd_b200.envs.get_env(name)
        sts = [be.reset(prng.split(prng.PRNGKey(s))[1]) for s in range(3)]
        b = eng.DiffusionEngine(be, 100, H, [0.05, 0.1, 0.2], False, sts, Ndiffuse=Nd)
        b.load_schedule(np.stack([eng.key_chain(np.uint32([s, 9]), Nd) for s in range(3)]), sigmas, alphas, alphas_bar)
        b.set_step(Nd - 1)
        b.step(); b.step(); torch.cuda.synchronize()
        print(f"batched {name} steps done (S=3), ctl.i =", b.ctl[:, 0].tolist(), flush=True)
print("done")
