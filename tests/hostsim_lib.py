"""ctypes binding of tests/hostsim (the product's device headers compiled for the host).

TEST INFRASTRUCTURE: lets the CPU test tier compare the kernel arithmetic with the oracle bit-for-bit.
Never imported by the hockey_env_b200 package.
"""
import ctypes as C
import os
import subprocess
import numpy as np
import oracle_lib as O

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build(force=False, root=_ROOT):
    """compile <root>/tests/hostsim/hostsim.cpp (which includes <root>/hockey_env_b200/csrc and <root>/include by
    relative path) into libhostsim.so next to it; `root` other than the repository builds a copy, e.g. a mutant"""
    d = os.path.join(root, "tests", "hostsim")
    so = os.path.join(d, "libhostsim.so")
    csrc = os.path.join(root, "hockey_env_b200", "csrc")
    srcs = [os.path.join(d, "hostsim.cpp"), os.path.join(root, "include", "hockey_b200.h")]
    srcs += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not force and os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(s) for s in srcs):
        return so
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                           "-x", "c++", "-o", so, os.path.join(d, "hostsim.cpp")])
    return so


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = load(build())
    return _lib


def load(so):
    """ctypes handle of a built libhostsim.so with the argument types set"""
    L = C.CDLL(so)
    vp, i64, u64, i32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int
    L.hs_create.restype = vp
    L.hs_create.argtypes = [i64, i32, i32, u64, i64]
    L.hs_destroy.argtypes = [vp]
    L.hs_reset.argtypes = [vp, vp, vp, vp]
    L.hs_reset_seeded.argtypes = [vp, vp, vp, vp, vp]
    L.hs_get_obs.argtypes = [vp, vp, vp]
    L.hs_step.argtypes = [vp, vp, i32, i32, i32, i32] + [vp] * 8
    L.hs_get_state.argtypes = [vp, vp]
    L.hs_set_state.argtypes = [vp, vp]
    L.hs_set_obs_state.argtypes = [vp, vp]
    L.hs_get_stats.argtypes = [vp, vp]
    L.hs_clear_stats.argtypes = [vp]
    L.hs_scene.argtypes = [vp, vp, i64]
    L.hs_scene_size.restype = i64
    L.hs_set_fast.argtypes = [vp, i32]
    L.hs_fast_counts.argtypes = [vp, vp]
    L.hs_set_mid_budget.argtypes = [vp, i32]
    L.hs_last_work.argtypes = [vp, vp]
    return L


_p = O._p

# columns of HostSimBatch.last_work(): what each env's last tick did (tests/hostsim/hostsim.cpp, hk_world.cuh WorkRecord)
W_KIND, W_SHAPE, W_SWEEPS, W_TOI, W_MAXSUB, W_SKIP_AFTER, W_EVENTS, W_GOAL, W_TIER = range(9)
# W_KIND: 1..8 = solveKind (two contacts (1,1) (1,2) (2,1) (2,2), three contacts (1,1,1) (1,1,2) (1,2,1) (2,1,1)),
# 9 = one contact with one point, 10 = one contact with two points, 11 = the generic loop, 0 = no island solve;
# W_SHAPE: contacts | points << 4 of that solve; W_EVENTS: bit 0 a puck x static TOI event, bit 1 a racket x static one
KIND_1C1P, KIND_1C2P, KIND_GENERIC = 9, 10, 11
TIER_FAST, TIER_TOUCH, TIER_GENERAL = 0, 1, 2


class HostSimBatch:
    def __init__(self, n, mode=0, keep_mode=True, seed=0, env_id_offset=0, fast=False, L=None):
        self.n = int(n)
        self.L = lib() if L is None else L  # L: another build (load()), e.g. of a mutated copy of the headers
        self.h = self.L.hs_create(self.n, int(mode), int(bool(keep_mode)), int(seed), int(env_id_offset))
        self.L.hs_set_fast(self.h, int(bool(fast)))

    def __del__(self):
        try:
            if self.h:
                self.L.hs_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def reset(self, mask=None, one_starting=None, seeds=None):
        obs = np.zeros((self.n, 18), np.float32)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        o = None if one_starting is None else np.ascontiguousarray(one_starting, np.int8)
        sd = None if seeds is None else np.ascontiguousarray(seeds, np.int64)
        self.L.hs_reset_seeded(self.h, _p(m), _p(o), _p(sd), _p(obs))
        return obs

    def get_obs(self):
        obs = np.zeros((self.n, 18), np.float32)
        obs2 = np.zeros((self.n, 18), np.float32)
        self.L.hs_get_obs(self.h, _p(obs), _p(obs2))
        return obs, obs2

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
        self.L.hs_step(self.h, _p(a), stride, p1, p2, flags, _p(out["obs"]), _p(out["obs2"]), _p(out["reward"]),
                       _p(out["reward2"]), _p(out["done"]), _p(out["info"]), _p(out["info2"]), _p(out["final_obs"]))
        return out

    def get_state(self):
        s = np.zeros((self.n, O.STATE_WORDS), np.uint32)
        self.L.hs_get_state(self.h, _p(s))
        return s

    def set_state(self, s):
        s = np.ascontiguousarray(s, np.uint32)
        self.L.hs_set_state(self.h, _p(s))

    def set_obs_state(self, obs18):
        s = np.ascontiguousarray(obs18, np.float32)
        self.L.hs_set_obs_state(self.h, _p(s))

    def fast_counts(self):
        c = np.zeros(4, np.int64)
        self.L.hs_fast_counts(self.h, _p(c))
        return int(c[0]), int(c[1]), int(c[2])

    def touch_count(self):
        c = np.zeros(4, np.int64)
        self.L.hs_fast_counts(self.h, _p(c))
        return int(c[3])

    def last_work(self):
        """[n, 9] int32 record of each env's last tick (columns W_*)"""
        w = np.zeros((self.n, 9), np.int32)
        self.L.hs_last_work(self.h, _p(w))
        return w

    def stats(self):
        s = np.zeros(16, np.float64)
        self.L.hs_get_stats(self.h, _p(s))
        return s
