"""Device-side engine of one reverse-diffusion step (`reverse_once`,
/root/reference/mbd/planners/mbd_planner.py:97-135), sample-sharded over ranks.

A step is THREE launches at any rank count (`mbd_step_launch`, csrc/step_tail.cuh):
  1. fused sampling + rollouts                      -> Y0s_local, rews_local (+logpd_local)
  2. k_step_weights: one 8-CTA cluster; sharded, it rendezvous with the peer GPUs and pulls their per-sample returns
     over NVLink itself, then global mean / std / demo blend / softmax           -> weights_local
  3. k_step_update: weighted-mean runs; the last CTA folds the tree, exchanges the rank partials over NVLink (sharded)
     and applies the update lines 130-133                                         -> Ybars[i - 1], ctl.i -= 1
Everything that changes from step to step (PRNG key, sigma, schedule scalars, the step index, the iterate) lives in DEVICE
memory, so the three launches take no per-step host arguments: `load_schedule` uploads the whole solve once, `capture`
records one step in a CUDA graph and `step` replays it — the host loop of mbd_planner.py:138-148 no longer bounds a solve.
Rank r of P owns samples [r*N/P, (r+1)*N/P); noise is addressed by GLOBAL index, all reduction orders depend on N only,
so the result does not depend on P.  Sharded runs need torch symmetric memory (NVLink peer access); there is no NCCL call
on the path (NCCL only bootstraps the rendezvous of the symmetric buffer).
"""
from __future__ import annotations

import ctypes
import os
import types
from typing import Optional

import numpy as np
import torch

from .. import _lib, ops, prng
from .sharding import ShardPlan


def linspace_f32(start: float, stop: float, num: int) -> np.ndarray:
    """`jnp.linspace(start, stop, num)` with x64 disabled (mbd_planner.py:13-14 leaves it off) **[jax-recalled]**: JAX does not
    compute `start + k * delta`; it blends the endpoints in float32, `start * (1 - k/(num-1)) + stop * (k/(num-1))`, and appends
    `stop` itself as the last element.  NumPy's float64 formula rounded to float32 differs from this by an ulp in a few entries
    (VERDICT r1, row a2); `MBD_LINSPACE=numpy` restores it."""
    import os
    f = np.float32
    if os.environ.get("MBD_LINSPACE", "jax") == "numpy" or num < 2:
        return np.linspace(start, stop, num, dtype=f)
    div = f(num - 1)
    step = (np.arange(num - 1, dtype=f) / div).astype(f)
    out = (f(start) * (f(1.0) - step)).astype(f) + (f(stop) * step).astype(f)
    return np.concatenate([out.astype(f), np.array([stop], dtype=f)])


def make_schedule(beta0: float, betaT: float, Ndiffuse: int):
    """mbd_planner.py:84-87 in float32."""
    betas = linspace_f32(beta0, betaT, Ndiffuse)
    alphas = (np.float32(1.0) - betas).astype(np.float32)
    alphas_bar = np.cumprod(alphas, dtype=np.float32)
    sigmas = np.sqrt(np.float32(1.0) - alphas_bar).astype(np.float32)
    return betas, alphas, alphas_bar, sigmas


def update_coef(alphas, alphas_bar, i: int):
    """The float32 scalars of mbd_planner.py:100,130-133 for step i."""
    one = np.float32(1.0)
    ab = np.float32(alphas_bar[i])
    return [np.sqrt(ab), one / (one - ab), one - ab, one / np.sqrt(np.float32(alphas[i])), np.sqrt(np.float32(alphas_bar[i - 1]))]


def key_chain(rng_exp, Ndiffuse: int) -> np.ndarray:
    """The Y0s_rng of every step: `rng, Y0s_rng = split(rng)` per step starting from rng_exp (mbd_planner.py:103,150).
    Returns [Ndiffuse, 2] uint32 with row i = key of step i (rows 0 and beyond the chain are zero)."""
    keys = np.zeros((Ndiffuse, 2), np.uint32)
    r = np.asarray(rng_exp, np.uint32)
    for i in range(Ndiffuse - 1, 0, -1):
        r, k = prng.split2(r)
        keys[i] = k
    return keys


def _is_state_batch(state_init) -> bool:
    """a list / tuple of states (not a list of numbers, which is one flat state)"""
    return isinstance(state_init, (list, tuple)) and len(state_init) > 0 and not np.isscalar(state_init[0])


class DiffusionEngine:
    def __init__(self, env, Nsample: int, Hsample: int, temp_sample, enable_demo: bool, state_init,
                 device: Optional[torch.device] = None, group=None, Ndiffuse: int = 2, emulate=None):
        """emulate = (P, rank, bufs): rank `rank` of P ranks that all live on THIS device and exchange through the plain
        device buffers `bufs` (one per rank) — the same kernels, flags and peer loads as a real sharded run, used by the
        single-GPU tests (`make_emulated_ranks`).

        Batched solves: `state_init` may be a sequence of S states and / or `temp_sample` a sequence of S temperatures (a
        single value is shared).  The S independent solves then run in the same three launches per step; every per-solve
        buffer gains a leading solve axis (`solve(s)` gives the views of one solve) and each solve gives exactly the bits it
        gives alone.  S == 1 is the single-solve engine.  Batches run on one rank only."""
        self.env = env
        states = list(state_init) if _is_state_batch(state_init) else [state_init]
        temps = [float(t) for t in np.atleast_1d(np.asarray(temp_sample, dtype=np.float64))]
        S = max(len(states), len(temps))
        if len(states) == 1:
            states = states * S
        if len(temps) == 1:
            temps = temps * S
        if len(states) != S or len(temps) != S:
            raise ValueError(f"{len(states)} initial states but {len(temps)} temperatures")
        if S > 1 and (emulate is not None or group is not None):
            raise ops.MbdError("a batch of solves runs on one rank: emulate= / group= are not supported with several solves")
        self.S, self.temps = S, temps
        self.N, self.H = int(Nsample), int(Hsample)
        self.temp = temps[0] if S == 1 else temps
        self.enable_demo = bool(enable_demo)
        self.plan = ShardPlan.from_env(self.N, group) if emulate is None else ShardPlan(self.N, emulate[0], emulate[1], None)
        self.group, self.P, self.rank = group, self.plan.P, self.plan.rank
        if S > 1 and self.P > 1:
            raise ops.MbdError("a batch of solves runs on one rank (WORLD_SIZE > 1 shards a single solve instead)")
        lead = () if S == 1 else (S,)      # leading solve axis of every per-solve buffer
        self.n_local, self.n_begin = self.plan.n_local, self.plan.n_begin
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.Nu = env.action_size
        self.HNu = self.H * self.Nu
        self.Nd = max(int(Ndiffuse), 2)
        d = self.device
        f = dict(device=d, dtype=torch.float32)
        self.Y0s = torch.empty(lead + (self.n_local, self.HNu), **f)
        # ---- exchange: P > 1 needs ONE peer-mapped symmetric buffer per rank, [rews n_local | logpd n_local | partial HNu |
        #      2 flag rows of 8 words]; the tail kernels read the peers' slices over NVLink themselves.
        self.sym, self.peer_ptrs = None, None
        self.exchange = "none" if self.P == 1 else "p2p"
        self.off_rews, self.off_logpd, self.off_partial = 0, self.n_local, 2 * self.n_local
        self.off_flags = 2 * self.n_local + self.HNu
        if self.P > 1 and emulate is not None:
            self.exchange = "p2p-emulated"
            self.sym = emulate[2][self.rank]
            assert self.sym.numel() == 2 * self.n_local + self.HNu + 16 and self.sym.device == d
            self.peer_ptrs = (ctypes.c_uint64 * self.P)(*[int(b.data_ptr()) for b in emulate[2]])
        elif self.P > 1:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm_mem
            words = 2 * self.n_local + self.HNu + 16
            self.sym = symm_mem.empty(words, dtype=torch.float32, device=d)
            self.sym.zero_()
            self.sym_hdl = symm_mem.rendezvous(self.sym, dist.group.WORLD if group is None else group)
            self.peer_ptrs = (ctypes.c_uint64 * self.P)(*[int(p) for p in self.sym_hdl.buffer_ptrs])
            torch.cuda.synchronize()
            dist.barrier(group=group)
        if self.P > 1:
            self.rews_local = self.sym[self.off_rews:self.off_rews + self.n_local]
            self.logpd_local = self.sym[self.off_logpd:self.off_logpd + self.n_local] if self.enable_demo else None
            self.partial = self.sym[self.off_partial:self.off_partial + self.HNu]
            self.rews_all = torch.empty(self.N, **f)
            self.logpd_all = torch.empty(self.N, **f) if self.enable_demo else None
        else:
            self.rews_local = torch.empty(lead + (self.n_local,), **f)
            self.logpd_local = torch.empty(lead + (self.n_local,), **f) if self.enable_demo else None
            self.partial = torch.empty(lead + (self.HNu,), **f)
            self.rews_all, self.logpd_all = self.rews_local, self.logpd_local
        self.weights = torch.empty(lead + (self.n_local,), **f)
        self.scalars = torch.zeros(lead + (4,), **f)
        self.logp_scratch = torch.empty(lead + (self.N,), **f)
        self.run_scratch = torch.empty(S * ((self.n_local + ops.RUN - 1) // ops.RUN) * self.HNu, **f)
        # ---- device-resident solve state
        self.Ybars = torch.zeros(lead + (self.Nd, self.HNu), **f)  # row i = input of step i, row i-1 = its output (row Nd-1 = YN = 0)
        self.rew_hist = torch.zeros(lead + (self.Nd,), **f)        # rews.mean() of step i
        self.params = torch.zeros(lead + (self.Nd, _lib.STEP_PARAMS_WORDS), device=d, dtype=torch.int32)
        self.ctl = torch.zeros(lead + (_lib.STEP_CTL_WORDS,), device=d, dtype=torch.int32)
        self.temps_dev = torch.tensor(temps, **f) if S > 1 else None
        self.launches_per_step = 3
        self.launches_last_step = 3
        self.graph = None
        if env.kind == "xpbd":
            self.model = env.device_model(d)
            self.state_init = self._stack_states(states, lambda st: st.pipeline_state.raw if hasattr(st, "pipeline_state") else st)
            self.xref = torch.as_tensor(env.xref, device=d).contiguous() if self.enable_demo else None
            self.params_car = None
        elif env.kind == "car2d":
            self.model = None
            self.params_car, xref = env.device_params()
            self.state_init = self._stack_states(states, lambda st: st.pipeline_state if hasattr(st, "pipeline_state") else st)
            self.xref = xref if self.enable_demo else None
        elif env.kind == "pusht":
            if self.enable_demo:
                raise ValueError("pushT has no demonstration (mbd_planner.py:118 applies to humanoidtrack / car2d)")
            self.model = None
            self.params_car = env.device_params()
            self.state_init = self._stack_states(states, lambda st: st.pipeline_state.raw if hasattr(st, "pipeline_state") else st)
            self.xref = None
        else:
            raise ValueError(env.kind)
        self.rew_xref = float(getattr(env, "rew_xref", 0.0))
        self._plan_c = self._make_plan()

    def _stack_states(self, states, raw_of) -> torch.Tensor:
        """one state -> its array as today; S states -> [S, ...] (the solve is the leading axis)"""
        arrs = [np.ascontiguousarray(raw_of(st), dtype=np.float32) for st in states]
        a = arrs[0] if self.S == 1 else np.ascontiguousarray(np.stack(arrs))
        return torch.as_tensor(a, device=self.device)

    def solve(self, s: int) -> types.SimpleNamespace:
        """views of solve s's buffers (with one solve: the buffers themselves)"""
        if not 0 <= s < self.S:
            raise IndexError(f"solve {s} of {self.S}")
        pick = (lambda t: t) if self.S == 1 else (lambda t: None if t is None else t[s])   # noqa: E731
        return types.SimpleNamespace(Ybars=pick(self.Ybars), rew_hist=pick(self.rew_hist), rews_local=pick(self.rews_local),
                                     logpd_local=pick(self.logpd_local), weights=pick(self.weights), scalars=pick(self.scalars),
                                     Y0s=pick(self.Y0s), ctl=pick(self.ctl), state_init=pick(self.state_init), temp=self.temps[s])

    def _single(self, what: str):
        if self.S > 1:
            raise ops.MbdError(f"{what} drives one solve; this engine holds a batch of {self.S} (use load_schedule / set_step / step)")

    # ---- C-ABI plan ----------------------------------------------------------------------------------------------
    def _make_plan(self) -> "_lib.StepPlan":
        p = _lib.StepPlan()
        vp = lambda t: None if t is None else t.data_ptr()   # noqa: E731
        p.model = self.model._h if self.model is not None else None
        p.car_params_dev = vp(self.params_car)
        p.state_init_dev = vp(self.state_init)
        p.params_dev, p.ctl_dev, p.Ybars_dev, p.rew_hist_dev = vp(self.params), vp(self.ctl), vp(self.Ybars), vp(self.rew_hist)
        p.n_total, p.n_begin, p.n_local, p.H, p.nu = self.N, self.n_begin, self.n_local, self.H, self.Nu
        p.temp, p.rew_xref = self.temps[0], self.rew_xref
        p.xref_dev = vp(self.xref)
        p.env_kind = _lib.ENV_PUSHT if self.env.kind == "pusht" else _lib.ENV_CAR2D
        p.href = 0 if self.xref is None else int(self.xref.shape[1] if self.env.kind == "xpbd" else self.xref.shape[0])
        p.Y0s_dev, p.rews_dev, p.logpd_dev = vp(self.Y0s), vp(self.rews_local), vp(self.logpd_local)
        p.rews_all_dev, p.logpd_all_dev, p.logp_dev = vp(self.rews_all), vp(self.logpd_all), vp(self.logp_scratch)
        p.weights_dev, p.runs_dev, p.partial_dev, p.scalars_dev = vp(self.weights), vp(self.run_scratch), vp(self.partial), vp(self.scalars)
        p.P, p.rank = self.P, self.rank
        if self.peer_ptrs is not None:
            p.peer_base_ptrs = ctypes.cast(self.peer_ptrs, ctypes.POINTER(ctypes.c_uint64))
        p.off_rews_words, p.off_logpd_words, p.off_partial_words, p.off_flags_words = self.off_rews, self.off_logpd, self.off_partial, self.off_flags
        p.timeout_cycles = int(float(os.environ.get("MBD_XCHG_TIMEOUT_S", "20")) * 2.0e9)
        p.n_solves, p.n_diffuse, p.temps_dev = self.S, self.Nd, vp(self.temps_dev)
        return p

    # ---- solve-level API -----------------------------------------------------------------------------------------
    def load_schedule(self, keys: np.ndarray, sigmas: np.ndarray, alphas: np.ndarray, alphas_bar: np.ndarray):
        """uploads the per-step parameters of a whole solve: row i = {Y0s_rng of step i, sigmas[i], update_coef(i)}.
        A batch takes one key chain per solve, keys [S, Nd, 2] (the schedule is shared)."""
        Nd, S = self.Nd, self.S
        keys = np.asarray(keys)
        if keys.shape == (S, Nd, 2) and S == 1:
            keys = keys[0]
        kshape = (Nd, 2) if S == 1 else (S, Nd, 2)
        if len(sigmas) != Nd or keys.shape != kshape:
            raise ops.MbdError(f"schedule of {len(sigmas)} steps / keys {keys.shape} do not match the engine (Ndiffuse={Nd}, solves={S})")
        tab = np.zeros((Nd, _lib.STEP_PARAMS_WORDS), np.uint32)
        tab[:, 2] = np.asarray(sigmas, np.float32).view(np.uint32)
        for i in range(1, Nd):
            tab[i, 3:8] = np.asarray(update_coef(alphas, alphas_bar, i), np.float32).view(np.uint32)
        tab = np.broadcast_to(tab, keys.shape[:-1] + (_lib.STEP_PARAMS_WORDS,)).copy()
        tab[..., 0:2] = keys
        self.params.copy_(torch.from_numpy(tab.view(np.int32)))

    def set_step(self, i: int):
        """device step counter <- i (the next `step()` runs diffusion step i: reads Ybars[i], writes Ybars[i-1])"""
        self.ctl.view(-1, _lib.STEP_CTL_WORDS)[:, 0].fill_(int(i))

    def step(self):
        """one diffusion step at the device-resident step index (three launches, or one replay of the captured graph)"""
        if self.graph is not None:
            self.graph.replay()
        else:
            ops.step_launch(self._plan_c)

    def capture(self):
        """records one step in a CUDA graph; later `step()` calls replay it (parameters come from device memory)"""
        i0 = int(self.ctl.view(-1, _lib.STEP_CTL_WORDS)[0, 0].item())
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            ops.step_launch(self._plan_c)        # warm-up outside capture (module load, func attributes)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        if self.P > 1:
            import torch.distributed as dist
            dist.barrier(group=self.group)       # every rank finished its warm-up step before anybody re-arms the counter
        self.set_step(i0)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            ops.step_launch(self._plan_c)
        self.graph = g
        return g

    def check_exchange(self):
        """Raises if a cross-GPU rendezvous ever timed out (a peer died or diverged; the outputs are NaN-poisoned).
        Synchronises: call it outside the step loop."""
        if int(self.ctl.view(-1, _lib.STEP_CTL_WORDS)[:, 2].abs().sum().item()) != 0:
            raise ops.MbdError("cross-GPU rendezvous timed out (a peer rank stopped participating); outputs are NaN")

    @classmethod
    def make_emulated_ranks(cls, env, Nsample, Hsample, temp_sample, enable_demo, state_init, P: int, Ndiffuse: int = 2, device=None):
        """P engines = P ranks on ONE device, each with its own stream, exchanging through plain device buffers with the very
        kernels, flags and peer loads of a real sharded run.  Drive them with `step_emulated_ranks`."""
        d = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        HNu = int(Hsample) * env.action_size
        n_local = int(Nsample) // P
        bufs = [torch.zeros(2 * n_local + HNu + 16, device=d) for _ in range(P)]
        engines = [cls(env, Nsample, Hsample, temp_sample, enable_demo, state_init, device=d, Ndiffuse=Ndiffuse, emulate=(P, r, bufs))
                   for r in range(P)]
        for e in engines:
            e.stream = torch.cuda.Stream(device=d)
        return engines

    @staticmethod
    def step_emulated_ranks(engines, ranks=None):
        """launches one step of every (or the given) emulated rank on its own stream — they rendezvous on the device"""
        cur = torch.cuda.current_stream()
        for e in engines:
            e.stream.wait_stream(cur)
        for r, e in enumerate(engines):
            if ranks is None or r in ranks:
                with torch.cuda.stream(e.stream):
                    e.step()
        for e in engines:
            cur.wait_stream(e.stream)

    def rollout_phase(self, key, sigma: float, Ybar_i: torch.Tensor):
        """sampling + rollouts with host-side parameters (path_integral.py's update_once shares it)"""
        self._single("rollout_phase")
        if self.env.kind == "xpbd":
            ops.sample_rollout(self.model, self.state_init, key, self.N, self.n_begin, self.n_local, self.H, float(sigma), Ybar_i,
                               self.Y0s, self.rews_local, xref=self.xref, logpd_out=self.logpd_local)
        elif self.env.kind == "pusht":
            ops.pusht_rollout(self.params_car, self.state_init, self.Y0s.view(self.n_local, self.H, 2), key=key, n_total=self.N,
                              n_begin=self.n_begin, sigma=float(sigma), Ybar=Ybar_i, rews_out=self.rews_local)
        else:
            ops.car2d_rollout(self.params_car, self.state_init, self.Y0s.view(self.n_local, self.H, 2), xref=self.xref, key=key,
                              n_total=self.N, n_begin=self.n_begin, sigma=float(sigma), Ybar=Ybar_i, rews_out=self.rews_local,
                              logpd_out=self.logpd_local)

    def stage_step(self, key, sigma: float, Ybar_i: torch.Tensor, coef, i: int = 1):
        """host-side parameters of ONE step -> row i of the device tables; the next `step()` runs it"""
        self._single("stage_step")
        row = np.zeros(_lib.STEP_PARAMS_WORDS, np.uint32)
        row[0:2] = np.asarray(key, np.uint32)
        row[2] = np.float32(sigma).view(np.uint32)
        row[3:8] = np.asarray(coef, np.float32).view(np.uint32)
        self.params[i].copy_(torch.from_numpy(row.view(np.int32)))
        self.Ybars[i].copy_(Ybar_i)
        self.set_step(i)

    # ---- single-step API (tests, bench, path-compatible with round 1) ---------------------------------------------
    def reverse_once(self, key, sigma: float, Ybar_i: torch.Tensor, coef, out: Optional[torch.Tensor] = None):
        """One diffusion step with host-side parameters: stages them into row 1 of the device tables, runs the step,
        returns (Ybar_im1 [HNu] device tensor, rews.mean() device scalar view)."""
        self.stage_step(key, sigma, Ybar_i, coef, 1)
        g, self.graph = self.graph, None
        try:
            self.step()
        finally:
            self.graph = g
        res = self.Ybars[0]
        if out is not None:
            out.copy_(res)
            res = out
        return res, self.scalars[0]
