"""Harvests a corpus of rare general-tier ticks: python tests/golden/make_general_corpus.py

The general tier selects specialised code per env and per tick by the shape of that tick's work: fixed-shape register
loops for two and three contacts, the generic loop for larger islands, the re-pack cuts of the one-point solve, the
180-sweep creeping solves, multi-event TOI ticks and the exact skips around an event.  Ordinary games reach several of
these a handful of times per hundred thousand env-steps, or never.  This script drives the host build of the kernel
headers (tests/hostsim) with external-action programs that make them likely, reads the per-env work record of every
tick (HostSimBatch.last_work), and keeps, per class, the full state record of the tick before the class occurred.

Written: general_corpus.npz (byte for byte reproducible: everything is seeded numpy, the zip entries carry a fixed date)
  state    [R, HK_STATE_WORDS] uint32  the record the class tick starts from (warm-start cache included)
  mode     [R] int32                   creation mode of the batch it was harvested in (what record mode 0 stands for)
  actions  [R, T, 8] float32           external actions of both players; row 0 produces the class
  cls      [R] int32                   index into `classes`
  classes  [C] str                     class names (CLASSES below)
  work     [R, 9] int32                the host work record of row 0's tick (hostsim_lib.W_*), for the coverage checks
tests/test_general_corpus.py replays it against the oracle on the host build and on the GPU.
"""
import io
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import hostsim_lib as H  # noqa: E402
import oracle_lib as O  # noqa: E402

T = 16              # ticks per record
HK_MAX_SUBSTEPS = 8  # hk_math.cuh
OUT = os.path.join(HERE, "general_corpus.npz")


def _kind(k):
    return lambda w: w[H.W_KIND] == k


# (name, predicate on the work record of row 0's tick, minimum count); every class must also finish in the general tier.
# Harvest order is this order: a tick that matches several classes is filed under the first one that still needs records.
CLASSES = [
    ("3c(2,1,1)", _kind(8), 64),
    ("3c(1,2,1)", _kind(7), 64),
    ("3c(1,1,2)", _kind(6), 64),
    ("3c(1,1,1)", _kind(5), 64),
    ("generic", _kind(H.KIND_GENERIC), 64),
    ("toi4+", lambda w: w[H.W_TOI] >= 4, 64),
    ("toi3", lambda w: w[H.W_TOI] == 3, 64),
    ("max_substeps", lambda w: w[H.W_MAXSUB] >= HK_MAX_SUBSTEPS, 64),
    ("sensor", lambda w: (w[H.W_EVENTS] & 1) != 0 and w[H.W_GOAL] != 0, 64),
    ("skip_after_event", lambda w: w[H.W_SKIP_AFTER] > 0, 64),
    ("toi2", lambda w: w[H.W_TOI] == 2, 64),
    ("creep180", lambda w: w[H.W_SWEEPS] == 180 and w[H.W_TOI] == 0, 64),
    ("cut12", lambda w: w[H.W_KIND] == H.KIND_1C1P and w[H.W_TOI] == 0 and w[H.W_SWEEPS] == 12, 24),
    ("cut24", lambda w: w[H.W_KIND] == H.KIND_1C1P and w[H.W_TOI] == 0 and w[H.W_SWEEPS] == 24, 24),
    ("cut48", lambda w: w[H.W_KIND] == H.KIND_1C1P and w[H.W_TOI] == 0 and w[H.W_SWEEPS] == 48, 24),
    ("2c(2,2)", _kind(4), 64),
    ("2c(2,1)", _kind(3), 64),
    ("2c(1,2)", _kind(2), 64),
    ("2c(1,1)", _kind(1), 64),
    ("1c2p", _kind(H.KIND_1C2P), 64),
    ("puck_static", lambda w: (w[H.W_EVENTS] & 1) != 0, 64),
]
# the three re-pack cuts together form the "cut" class of at least 64 records
CUT_CLASSES = ("cut12", "cut24", "cut48")
# what the committed corpus must hold where the harvest falls short of the quota above: ticks with four or more TOI
# events are the rarest class (about one in 3,000 of the fast corner starts' three-event ticks); no pair reaches
# HK_MAX_SUBSTEPS in any of these programs (the highest sub-step count seen is 2), so that class stays empty
REQUIRED = {"toi4+": 48, "max_substeps": 0}
NAMES = [c[0] for c in CLASSES]


def classify(w):
    """names of every class the work record w (one env's tick) belongs to"""
    if w[H.W_TIER] != H.TIER_GENERAL:
        return []
    return [name for name, pred, _ in CLASSES if pred(w)]


# ---- external-action programs ----------------------------------------------------------------------------------
# obs (player 1's view) and obs2 (player 2's mirrored view) both hold [own x, y, angle, vx, vy, w, other ..., puck x, y,
# vx, vy, ...] relative to the rink centre; an action's force is in the player's own view, so "towards the puck" is the
# same expression in both.
def _toward(o, gain):
    return np.clip(gain * (o[:, 12:14] - o[:, 0:2]), -1.0, 1.0)


def prog_uniform(rng, obs, obs2, t):
    return rng.uniform(-1.4, 1.4, (obs.shape[0], 8))


def prog_squeeze(rng, obs, obs2, t):
    n = obs.shape[0]
    a = np.zeros((n, 8))
    a[:, 0:2] = _toward(obs, 3.0) + rng.normal(0, 0.15, (n, 2))
    a[:, 4:6] = _toward(obs2, 3.0) + rng.normal(0, 0.15, (n, 2))
    a[:, 2] = rng.uniform(-1, 1, n)
    a[:, 6] = rng.uniform(-1, 1, n)
    a[:, 3] = rng.uniform(-1, 1, n)
    a[:, 7] = rng.uniform(-1, 1, n)
    return a


def prog_pin(rng, obs, obs2, t):
    # player 1 presses the puck on, past it towards the nearest side wall (or its own goal line), and keeps pressing
    n = obs.shape[0]
    a = np.zeros((n, 8))
    tgt = obs[:, 12:14] + np.stack([np.where(obs[:, 12] < 0, -0.4, 0.4), np.where(obs[:, 13] < 0, -0.4, 0.4)], 1)
    a[:, 0:2] = np.clip(4.0 * (tgt - obs[:, 0:2]), -1, 1)
    a[:, 2] = np.sign(np.sin(0.3 * t + np.arange(n)))
    a[:, 3] = (rng.random(n) < 0.2) * 1.0
    a[:, 4:8] = rng.uniform(-1, 1, (n, 4))
    return a


def prog_ram(rng, obs, obs2, t):
    # full-speed crossing runs with rotation: direction flips every 12 ticks, torque saturated
    n = obs.shape[0]
    a = np.zeros((n, 8))
    phase = ((t // 12) + np.arange(n)) % 4
    d = np.array([[1, 0.3], [-1, -0.3], [0.4, 1], [-0.4, -1]])[phase]
    a[:, 0:2] = d
    a[:, 4:6] = -d[:, ::-1]
    a[:, 2] = np.where(np.arange(n) % 2 == 0, 1.0, -1.0)
    a[:, 6] = -a[:, 2]
    return a


# ---- starting states (set_obs_state) ---------------------------------------------------------------------------
XW, YW = 4.4, 3.4  # roughly the inner rink extent from the centre


def starts_corner(rng, n, speed):
    """puck near a wall or corner, both rackets close to it; the puck moves at `speed` towards the corner"""
    s = np.zeros((n, 18))
    cx = rng.choice([-1, 1], n) * rng.uniform(2.5, XW, n)
    cy = rng.choice([-1, 1], n) * rng.uniform(1.5, YW, n)
    corner = np.stack([np.sign(cx) * XW, np.sign(cy) * YW], 1)
    pk = np.stack([cx, cy], 1)
    d = corner - pk
    d /= np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-3)
    s[:, 12:14] = pk
    s[:, 14:16] = d * speed[:, None]
    for k, off in ((0, -1.0), (6, 1.0)):
        ang = rng.uniform(0, 2 * np.pi, n)
        r = rng.uniform(0.5, 1.4, n)
        s[:, k] = cx - np.sign(cx) * r * np.abs(np.cos(ang)) + 0.3 * off
        s[:, k + 1] = cy - np.sign(cy) * r * np.abs(np.sin(ang))
        s[:, k + 2] = rng.uniform(-0.8, 0.8, n)
        s[:, k + 3:k + 5] = rng.normal(0, 2.0, (n, 2))
        s[:, k + 5] = rng.normal(0, 2.0, n)
    return s.astype(np.float32)


# (program, mode, start (None: the env's own reset), batch, ticks, seed)
RUNS = []
for _r in range(24):  # the late rounds only still look for the rarest classes (ticks with four or more TOI events)
    RUNS += [
        (prog_squeeze, O.MODE_NORMAL, "corner_slow", 2048, 60, 100 + _r),
        (prog_squeeze, O.MODE_TRAIN_SHOOTING, "corner_fast", 2048, 40, 200 + _r),
        (prog_pin, O.MODE_TRAIN_DEFENSE, None, 2048, 80, 300 + _r),
        (prog_ram, O.MODE_NORMAL, None, 2048, 80, 400 + _r),
        (prog_uniform, O.MODE_TRAIN_SHOOTING, None, 2048, 80, 500 + _r),
        (prog_squeeze, O.MODE_TRAIN_DEFENSE, "corner_fast", 2048, 40, 600 + _r),
    ]


def harvest(runs=RUNS, verbose=True):
    quota = {name: m for name, _, m in CLASSES}
    got = {name: [] for name in NAMES}
    seen = {name: 0 for name in NAMES}
    for ri, (prog, mode, start, n, ticks, seed) in enumerate(runs):
        if all(len(got[k]) >= quota[k] for k in NAMES):
            break
        rng = np.random.default_rng(seed)
        h = H.HostSimBatch(n, mode=mode, seed=seed, env_id_offset=1_000_000 * seed, fast=True)
        h.reset()
        if start is not None:
            speed = rng.uniform(1.0, 6.0, n) if start == "corner_slow" else rng.uniform(10.0, 40.0, n)
            h.set_obs_state(starts_corner(rng, n, speed))
        pending = {}  # env -> (class, state, [action rows], work)
        for t in range(ticks):
            obs, obs2 = h.get_obs()
            a = prog(rng, obs, obs2, t).astype(np.float32)
            pre = h.get_state()
            h.step(a, O.POL_EXTERNAL, O.POL_EXTERNAL, O.STEP_AUTORESET)
            w = h.last_work()
            for i, rec in list(pending.items()):
                rec[2].append(a[i].copy())
                if len(rec[2]) == T:
                    got[rec[0]].append((rec[1], mode, np.stack(rec[2]), rec[3]))
                    del pending[i]
            for i in np.flatnonzero(w[:, H.W_TIER] == H.TIER_GENERAL):
                if i in pending:
                    continue
                names = classify(w[i])
                for k in names:
                    seen[k] += 1
                for k in names:
                    if len(got[k]) + sum(1 for r in pending.values() if r[0] == k) < quota[k]:
                        pending[i] = (k, pre[i].copy(), [a[i].copy()], w[i].copy())
                        break
        if verbose:
            print(f"run {ri:2d} {prog.__name__:14s} mode {mode} start {start}: " +
                  " ".join(f"{k}={len(got[k])}" for k in NAMES), flush=True)
    return got, seen


def _npz_bytes(arrays):
    buf = io.BytesIO()
    with zipfile.ZipFile(buf, "w", zipfile.ZIP_DEFLATED) as z:
        for k, v in arrays.items():
            b = io.BytesIO()
            np.lib.format.write_array(b, np.ascontiguousarray(v), allow_pickle=False)
            zi = zipfile.ZipInfo(k + ".npy", date_time=(1980, 1, 1, 0, 0, 0))
            zi.compress_type = zipfile.ZIP_DEFLATED
            z.writestr(zi, b.getvalue())
    return buf.getvalue()


def main():
    H.build()
    got, seen = harvest()
    present = [k for k in NAMES if got[k]]
    st, md, ac, cl, wk = [], [], [], [], []
    for ci, k in enumerate(present):
        for s, m, a, w in got[k]:
            st.append(s); md.append(m); ac.append(a); cl.append(ci); wk.append(w)
    arrays = dict(state=np.array(st, np.uint32), mode=np.array(md, np.int32), actions=np.array(ac, np.float32),
                  cls=np.array(cl, np.int32), classes=np.array(present), work=np.array(wk, np.int32))
    data = _npz_bytes(arrays)
    with open(OUT, "wb") as f:
        f.write(data)
    print(f"wrote {OUT}: {len(st)} records, {len(data)} bytes")
    for k in NAMES:
        print(f"  {k:18s} kept {len(got[k]):4d}   ticks seen {seen[k]}")


if __name__ == "__main__":
    main()
