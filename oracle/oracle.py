"""ctypes front-end of the CPU oracle (oracle/libmbd_oracle.so) — TEST INFRASTRUCTURE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this module.  The product package (mbd_b200) never does.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

_f32p = ctypes.POINTER(ctypes.c_float)
_u32p = ctypes.POINTER(ctypes.c_uint32)


def build(force: bool = False) -> str:
    """Compiles oracle/libmbd_oracle.so (gcc, see oracle/Makefile) when it is missing, stale or forced."""
    import fcntl
    so = os.path.join(_HERE, "libmbd_oracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("mbd_oracle.c", "pusht_oracle.c", "Makefile")]
    hdrs = [os.path.join(_HERE, "..", "include", h) for h in ("mbd_fp32.h", "mbd_model.h", "mbd_pusht.h")]

    def stale():
        return (not os.path.exists(so)) or any(os.path.getmtime(p) > os.path.getmtime(so) for p in srcs + hdrs if os.path.exists(p))

    if force or stale():
        with open(os.path.join(_HERE, ".build.lock"), "w") as lock:
            fcntl.flock(lock, fcntl.LOCK_EX)
            if force or stale():
                subprocess.run(["make", "-C", _HERE, "-B"], check=True, capture_output=True)
    return so


_HOST_DIR = None


def _host_build_dir() -> str:
    """Scratch directory of this process for the libraries compiled for THIS host at run time (-march=native).  They
    never go into the source tree, which may be read-only where bench.py runs; the directory is removed at exit."""
    global _HOST_DIR
    if _HOST_DIR is None:
        import atexit
        import shutil
        import tempfile
        _HOST_DIR = tempfile.mkdtemp(prefix="mbd_oracle_")
        atexit.register(shutil.rmtree, _HOST_DIR, True)
    return _HOST_DIR


def use_native() -> bool:
    """Switches this process to libmbd_oracle_native.so: the same source built `-O2 -march=native` ON THIS HOST
    (bench.py's timed CPU arm; -ffp-contract=off is kept, so the results are the same bits).  Returns False — and keeps
    the portable build — when the compile fails."""
    global _LIB
    so = os.path.join(_host_build_dir(), "libmbd_oracle_native.so")
    try:
        subprocess.run(["make", "-C", _HERE, "-B", "native", "NATIVE_OUT=" + so], check=True, capture_output=True)
        L = ctypes.CDLL(so)
        L.orc_num_threads.restype = ctypes.c_int
        _LIB = L
        return True
    except Exception:  # noqa: BLE001
        return False


_SIMD = None


def use_simd():
    """Builds (on THIS host, -march=native) and loads libmbd_oracle_simd.so — the SIMD-across-samples CPU arm of
    bench.py (mbd_oracle_simd.cpp: the templated physics of csrc/xpbd_pk.cuh instantiated with a 16-lane host type; same
    bits as the scalar oracle).  Returns the library or None when it cannot be built."""
    global _SIMD
    if _SIMD is not None:
        return _SIMD or None
    root = os.path.join(_HERE, "..")
    so = os.path.join(_host_build_dir(), "libmbd_oracle_simd.so")
    flags = ["-O3", "-march=native", "-std=c++17", "-ffp-contract=off", "-fno-math-errno", "-fopenmp", "-shared", "-fPIC", "-fvisibility=hidden"]
    try:
        with open("/proc/cpuinfo") as f:
            if "avx512f" in f.read():
                flags.append("-mprefer-vector-width=512")   # gcc splits 512-bit vectors in two by default on most Xeons: 6x slower here
    except OSError:
        pass
    try:
        subprocess.run(["g++"] + flags + ["-I" + os.path.join(root, "include"), "-I" + os.path.join(root, "mbd_b200", "csrc"),
                                          os.path.join(_HERE, "mbd_oracle_simd.cpp"), "-o", so], check=True, capture_output=True)
        _SIMD = ctypes.CDLL(so)
    except Exception:  # noqa: BLE001
        _SIMD = False
    return _SIMD or None


def simd_rollout(blob, state_init, Y0s, want_final=False, nthreads=0):
    """vmap(rollout_us) through the SIMD CPU arm (humanoidrun / humanoidstandup); None when it does not cover the model"""
    L_ = use_simd()
    if L_ is None:
        return None
    blob = np.ascontiguousarray(blob, dtype=np.uint32)
    nl = int(blob.view(np.int32)[1])
    state_init = np.ascontiguousarray(state_init, dtype=np.float32).reshape(nl, 13)
    Y0s = np.ascontiguousarray(Y0s, dtype=np.float32)
    n, H, _ = Y0s.shape
    rews = np.zeros(n, dtype=np.float32)
    final = np.zeros((n, nl, 13), dtype=np.float32) if want_final else None
    rc = L_.orc_simd_rollout(_up(blob), _fp(state_init), _fp(Y0s), n, H, _fp(rews), _fp(final), nthreads)
    if rc != 0:
        return None
    return dict(rews=rews, final=final, logpd=None, rewss=None, track=None)


def lib():
    global _LIB
    if _LIB is None:
        _LIB = ctypes.CDLL(build())
        _LIB.orc_num_threads.restype = ctypes.c_int
    return _LIB


def _fp(a):
    return None if a is None else a.ctypes.data_as(_f32p)


def _up(a):
    return a.ctypes.data_as(_u32p)


def num_threads() -> int:
    return int(lib().orc_num_threads())


# ---- PRNG (jax.random restated) -------------------------------------------------------
def threefry2x32(key, ctr):
    key = np.ascontiguousarray(key, dtype=np.uint32)
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32)
    out = np.zeros(2, dtype=np.uint32)
    lib().orc_threefry2x32(_up(key), _up(ctr), _up(out))
    return out


def random_bits(key, total):
    key = np.ascontiguousarray(key, dtype=np.uint32)
    out = np.zeros(total, dtype=np.uint32)
    lib().orc_random_bits(_up(key), ctypes.c_uint32(total), _up(out))
    return out


def prng_key(seed: int):
    """jax.random.PRNGKey(seed) for 0 <= seed < 2**32 (x64 disabled)."""
    return np.array([0, seed & 0xFFFFFFFF], dtype=np.uint32)


_PART = False


def set_prng_layout(partitionable: bool):
    """legacy (default, pinned by JAX's KATs) or partitionable [jax-recalled] threefry layout for every sampler of the oracle"""
    global _PART
    _PART = bool(partitionable)
    lib().orc_set_prng_layout(1 if partitionable else 0)


def split(key, num=2):
    """jax.random.split: legacy threefry_2x32(key, iota(2*num)).reshape(num, 2); partitionable: key i = block(key, (0, i))."""
    if _PART:
        key = np.ascontiguousarray(key, dtype=np.uint32)
        return np.stack([threefry2x32(key, np.uint32([0, i])) for i in range(num)])
    return random_bits(key, 2 * num).reshape(num, 2)


def normal(key, shape, begin=None, end=None, nthreads=0):
    total = int(np.prod(shape)) if len(shape) else 1
    b = 0 if begin is None else begin
    e = total if end is None else end
    out = np.zeros(e - b, dtype=np.float32)
    key = np.ascontiguousarray(key, dtype=np.uint32)
    lib().orc_normal(_up(key), ctypes.c_uint32(total), ctypes.c_uint32(b), ctypes.c_uint32(e), _fp(out), nthreads)
    return out.reshape(shape) if begin is None and end is None else out


def uniform(key, shape, minval=0.0, maxval=1.0):
    """jax.random.uniform (f32): max(minval, unit * (maxval - minval) + minval)."""
    total = int(np.prod(shape)) if len(shape) else 1
    bits = random_bits(key, total)
    unit = ((bits >> np.uint32(9)) | np.uint32(0x3F800000)).view(np.float32) - np.float32(1.0)
    lo, hi = np.float32(minval), np.float32(maxval)
    return np.maximum(lo, unit * (hi - lo) + lo).reshape(shape)


def sample_Y0s(key, n_total, HNu, sigma, Ybar, n_begin=0, n_end=None, nthreads=0):
    """mbd_planner.py:103-106 for samples [n_begin, n_end) of n_total."""
    n_end = n_total if n_end is None else n_end
    key = np.ascontiguousarray(key, dtype=np.uint32)
    Ybar = np.ascontiguousarray(Ybar, dtype=np.float32).reshape(-1)
    out = np.zeros((n_end - n_begin, HNu), dtype=np.float32)
    lib().orc_sample_Y0s(_up(key), n_total, n_begin, n_end, HNu, ctypes.c_float(sigma), _fp(Ybar), _fp(out), nthreads)
    return out


# ---- rollouts ------------------------------------------------------------------------------
def xpbd_rollout(blob, state_init, Y0s, xref=None, want_rewss=False, want_final=False, want_track=False,
                 nsub_override=0, nthreads=0):
    """vmap(rollout_us)(state_init, Y0s) for a Brax-positional env.  Y0s [n,H,nu] float32."""
    blob = np.ascontiguousarray(blob, dtype=np.uint32)
    L = int(blob.view(np.int32)[1])
    ntrack = int(blob.view(np.int32)[5])
    state_init = np.ascontiguousarray(state_init, dtype=np.float32).reshape(L, 13)
    Y0s = np.ascontiguousarray(Y0s, dtype=np.float32)
    n, H, nu = Y0s.shape
    rews = np.zeros(n, dtype=np.float32)
    rewss = np.zeros((n, H), dtype=np.float32) if want_rewss else None
    final = np.zeros((n, L, 13), dtype=np.float32) if want_final else None
    track = np.zeros((n, H, ntrack, 3), dtype=np.float32) if want_track else None
    logpd, href = None, 0
    if xref is not None:
        xref = np.ascontiguousarray(xref, dtype=np.float32)
        href = xref.shape[1]
        logpd = np.zeros(n, dtype=np.float32)
    rc = lib().orc_xpbd_rollout(_up(blob), _fp(state_init), _fp(Y0s), n, H, _fp(rewss), _fp(rews), _fp(xref), href,
                                _fp(logpd), _fp(final), _fp(track), nsub_override, nthreads)
    if rc != 0:
        raise RuntimeError(f"orc_xpbd_rollout failed: {rc}")
    return dict(rews=rews, rewss=rewss, logpd=logpd, final=final, track=track)


def car2d_rollout(params, x0, Y0s, xref=None, want_rewss=False, want_traj=False, nthreads=0):
    params = np.ascontiguousarray(params, dtype=np.float32)
    x0 = np.ascontiguousarray(x0, dtype=np.float32)
    Y0s = np.ascontiguousarray(Y0s, dtype=np.float32)
    n, H, _ = Y0s.shape
    rews = np.zeros(n, dtype=np.float32)
    rewss = np.zeros((n, H), dtype=np.float32) if want_rewss else None
    traj = np.zeros((n, H, 3), dtype=np.float32) if want_traj else None
    logpd, href = None, 0
    if xref is not None:
        xref = np.ascontiguousarray(xref, dtype=np.float32)
        href = xref.shape[0]
        logpd = np.zeros(n, dtype=np.float32)
    lib().orc_car2d_rollout(_fp(params), _fp(x0), _fp(Y0s), n, H, _fp(rewss), _fp(rews), _fp(xref), href, _fp(logpd),
                            _fp(traj), nthreads)
    return dict(rews=rews, rewss=rewss, logpd=logpd, traj=traj)


def pusht_rollout(params, x0, Y0s, want_rewss=False, want_final=False, want_traj=False, nthreads=0):
    """vmap(rollout_us) of the pushT env (oracle/pusht_oracle.c): params [MBD_PT_NPARAM], x0 [16] = q | qd, Y0s [n, H, 2]"""
    params = np.ascontiguousarray(params, dtype=np.float32)
    x0 = np.ascontiguousarray(x0, dtype=np.float32).reshape(16)
    Y0s = np.ascontiguousarray(Y0s, dtype=np.float32)
    n, H, _ = Y0s.shape
    rews = np.zeros(n, dtype=np.float32)
    rewss = np.zeros((n, H), dtype=np.float32) if want_rewss else None
    final = np.zeros((n, 16), dtype=np.float32) if want_final else None
    traj = np.zeros((n, H, 16), dtype=np.float32) if want_traj else None
    lib().orc_pusht_rollout(_fp(params), _fp(x0), _fp(Y0s), n, H, _fp(rewss), _fp(rews), _fp(final), _fp(traj), nthreads)
    return dict(rews=rews, rewss=rewss, final=final, traj=traj, logpd=None)


def fmap(fn: str, a, b=None):
    idx = dict(atan2=0, sin=1, cos=2, log=3, exp=4, erfinv=5)[fn]
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = a if b is None else np.ascontiguousarray(b, dtype=np.float32)
    out = np.zeros_like(a)
    lib().orc_map(idx, _fp(a), _fp(b), _fp(out), a.size)
    return out
