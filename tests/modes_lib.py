"""ctypes bindings of tests/modes: the CPU oracle and the host build of the device code with per-env game modes.

TEST INFRASTRUCTURE: `ModeOracleBatch` / `ModeHostSimBatch` are `OracleBatch` / `HostSimBatch` whose every reset
(masked or automatic) starts the next episode of env i in the mode `reset_modes[i]` says, like hk_set_reset_modes,
and whose state records carry word HK_S_MODE.  The libraries are built on first use, next to their sources when that
directory is writable, else in a temporary directory.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import hostsim_lib as H
import oracle_lib as O

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_DIR = os.path.join(_ROOT, "tests", "modes")
_FLAGS = ["-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-pthread"]
_p = O._p


def _build(name, srcs, deps):
    out_dir = _DIR if os.access(_DIR, os.W_OK) else os.path.join(tempfile.gettempdir(), f"hk_modes_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"lib{name}.so")
    if not (os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(s) for s in srcs + deps)):
        subprocess.check_call(["g++"] + _FLAGS + ["-o", so] + srcs)
    return C.CDLL(so)


def _headers():
    csrc = os.path.join(_ROOT, "hockey_env_b200", "csrc")
    return [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")] + [os.path.join(_ROOT, "include", "hockey_b200.h")]


def _copy_decls(L, ref, names):
    for n in names:
        f, g = getattr(L, n), getattr(ref, n)
        f.argtypes, f.restype = g.argtypes, g.restype


_oracle = _hostsim = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        odir = os.path.join(_ROOT, "oracle")
        L = _build("oracle_modes", [os.path.join(_DIR, "oracle_modes.cpp"), os.path.join(odir, "b2mini.cpp")],
                   [os.path.join(odir, f) for f in ("hockey_oracle.cpp", "b2mini.h")] + _headers())
        _copy_decls(L, O.lib(), ["hko_get_obs", "hko_get_stats", "hko_clear_stats", "hko_set_obs_state"])
        vp, i64, u64, i32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int
        L.hkm_create.restype = vp
        L.hkm_create.argtypes = [i64, i32, i32, u64, i64]
        for n in ("hkm_destroy",):
            getattr(L, n).argtypes = [vp]
        for n in ("hkm_set_reset_modes", "hkm_get_modes", "hkm_get_state", "hkm_set_state"):
            getattr(L, n).argtypes = [vp, vp]
        L.hkm_reset_seeded.argtypes = [vp, vp, vp, vp, vp]
        L.hkm_step.argtypes = [vp, vp, i32, i32, i32, i32] + [vp] * 8
        _oracle = L
    return _oracle


def hostsim_lib():
    global _hostsim
    if _hostsim is None:
        L = _build("hostsim_modes", [os.path.join(_DIR, "hostsim_modes.cpp")],
                   [os.path.join(_ROOT, "tests", "hostsim", "hostsim.cpp")] + _headers())
        _copy_decls(L, H.lib(), ["hs_create", "hs_get_obs", "hs_get_stats", "hs_clear_stats", "hs_set_fast",
                                 "hs_fast_counts", "hs_set_obs_state"])
        vp = C.c_void_p
        L.hsm_destroy.argtypes = [vp]
        for n in ("hsm_set_reset_modes", "hsm_get_modes", "hsm_get_state", "hsm_set_state"):
            getattr(L, n).argtypes = [vp, vp]
        L.hsm_reset_seeded.argtypes = [vp, vp, vp, vp, vp]
        L.hsm_step.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int] + [vp] * 8
        _hostsim = L
    return _hostsim


class _ModeCalls:
    """The calls both bindings share; `_fn(name)` maps a base name to the library's symbol."""

    def set_reset_modes(self, modes):
        """Per-env mode of the episode each later reset starts (None = keep).  The array is kept and read by every
        later reset, like the device tensor of hk_set_reset_modes: rewrite `self.reset_modes` in place."""
        self.reset_modes = None if modes is None else np.ascontiguousarray(modes, np.uint8)
        self._fn("set_reset_modes")(self.h, _p(self.reset_modes))

    def modes(self):
        m = np.zeros(self.n, np.uint8)
        self._fn("get_modes")(self.h, _p(m))
        return m

    def reset(self, mask=None, one_starting=None, seeds=None):
        obs = np.zeros((self.n, O.OBS_DIM), np.float32)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        o = None if one_starting is None else np.ascontiguousarray(one_starting, np.int8)
        sd = None if seeds is None else np.ascontiguousarray(seeds, np.int64)
        self._fn("reset_seeded")(self.h, _p(m), _p(o), _p(sd), _p(obs))
        return obs

    def get_state(self):
        s = np.zeros((self.n, O.STATE_WORDS), np.uint32)
        self._fn("get_state")(self.h, _p(s))
        return s

    def set_state(self, s):
        s = np.ascontiguousarray(s, np.uint32)
        assert s.shape == (self.n, O.STATE_WORDS)
        self._fn("set_state")(self.h, _p(s))


class ModeOracleBatch(_ModeCalls, O.OracleBatch):
    def __init__(self, n, mode=O.MODE_NORMAL, keep_mode=True, seed=0, env_id_offset=0):
        self.n = int(n)
        self.L = oracle_lib()
        self.h = self.L.hkm_create(self.n, int(mode), int(bool(keep_mode)), int(seed), int(env_id_offset))
        self.reset_modes = None

    def _fn(self, name):
        return getattr(self.L, "hkm_" + name)

    def __del__(self):
        try:
            if self.h:
                self.L.hkm_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def step(self, action=None, p1=O.POL_EXTERNAL, p2=O.POL_EXTERNAL, flags=0):
        n = self.n
        a, stride = None, 0
        if action is not None:
            a = np.ascontiguousarray(action, np.float32)
            stride = a.shape[1]
        out = dict(obs=np.zeros((n, 18), np.float32), obs2=np.zeros((n, 18), np.float32),
                   reward=np.zeros(n, np.float64), reward2=np.zeros(n, np.float64), done=np.zeros(n, np.uint8),
                   info=np.zeros((n, 4), np.float64), info2=np.zeros((n, 4), np.float64),
                   final_obs=np.zeros((n, 18), np.float32))
        self.L.hkm_step(self.h, _p(a), stride, p1, p2, flags, _p(out["obs"]), _p(out["obs2"]), _p(out["reward"]),
                        _p(out["reward2"]), _p(out["done"]), _p(out["info"]), _p(out["info2"]), _p(out["final_obs"]))
        return out


class ModeHostSimBatch(_ModeCalls, H.HostSimBatch):
    def __init__(self, n, mode=0, keep_mode=True, seed=0, env_id_offset=0, fast=False):
        self.n = int(n)
        self.L = hostsim_lib()
        self.h = self.L.hs_create(self.n, int(mode), int(bool(keep_mode)), int(seed), int(env_id_offset))
        self.L.hs_set_fast(self.h, int(bool(fast)))
        self.reset_modes = None

    def _fn(self, name):
        return getattr(self.L, "hsm_" + name)

    def __del__(self):
        try:
            if self.h:
                self.L.hsm_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def step(self, action=None, p1=0, p2=0, flags=0):
        n = self.n
        a, stride = None, 0
        if action is not None:
            a = np.ascontiguousarray(action, np.float32)
            stride = a.shape[1]
        out = dict(obs=np.zeros((n, 18), np.float32), obs2=np.zeros((n, 18), np.float32),
                   reward=np.zeros(n, np.float32), reward2=np.zeros(n, np.float32), done=np.zeros(n, np.uint8),
                   info=np.zeros((n, 4), np.float32), info2=np.zeros((n, 4), np.float32),
                   final_obs=np.zeros((n, 18), np.float32))
        self.L.hsm_step(self.h, _p(a), stride, p1, p2, flags, _p(out["obs"]), _p(out["obs2"]), _p(out["reward"]),
                        _p(out["reward2"]), _p(out["done"]), _p(out["info"]), _p(out["info2"]), _p(out["final_obs"]))
        return out
