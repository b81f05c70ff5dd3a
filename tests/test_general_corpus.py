"""The general tier's rare paths, reached on purpose: a corpus of harvested ticks replayed against the oracle.

tests/golden/general_corpus.npz (tests/golden/make_general_corpus.py) holds, per class, state records from which the
next tick takes one rare path: the fixed-shape two- and three-contact loops, the generic loop, the one-contact loops with
their re-pack cuts, 180-sweep creeping solves, ticks with two, three and four or more TOI events, TOI evaluations skipped
after an event, puck x static events and goals scored in an event tick.  Each record carries 16 ticks of external
actions.  Every output of every tick and the full state record after every tick must equal the oracle's (-0 == +0).

CPU tier: the corpus still produces its classes on the host build of the kernel headers, the host build equals the
oracle on all of it, and textual mutants of the headers (built from a copy) make the comparison fail in the class they
target.  GPU tier: the CUDA library against the oracle on the corpus in several layouts and cascade variants, with the
lane trace proving that every class ran in the general tier with its contacts, points and TOI events.
"""
import os
import shutil

import numpy as np
import pytest

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_CORPUS = os.path.join(_HERE, "golden", "general_corpus.npz")


def _corpus():
    z = np.load(_CORPUS)
    return dict(state=z["state"], mode=z["mode"], actions=z["actions"], cls=z["cls"], classes=[str(c) for c in z["classes"]],
                work=z["work"])


def _gen():
    import sys
    sys.path.insert(0, os.path.join(_HERE, "golden"))
    import make_general_corpus as G
    return G


def _replay_host(O, H, C, idx, mode, L=None):
    """host build vs oracle on records idx (all harvested in `mode`), T ticks.  Returns {record: first differing tick}."""
    from parity_util import state_mismatches, outputs_equal
    n = len(idx)
    h = H.HostSimBatch(n, mode=mode, seed=11, fast=True, L=L)
    ora = O.OracleBatch(n, mode=mode, seed=11)
    s = C["state"][idx]
    h.set_state(s)
    ora.set_state(s)
    bad = {}
    for t in range(C["actions"].shape[1]):
        a = np.ascontiguousarray(C["actions"][idx, t])
        rh = h.step(a, 0, 0, O.STEP_AUTORESET)
        ro = ora.step(a, O.POL_EXTERNAL, O.POL_EXTERNAL, O.STEP_AUTORESET)
        rows = set(state_mismatches(ora.get_state(), h.get_state())[:, 0].tolist())
        if outputs_equal(ro, rh):
            for k in ("obs", "obs2", "done", "final_obs", "reward", "reward2", "info", "info2"):
                x, y = ro[k], rh[k]
                if x.dtype == np.float64:
                    x = x.astype(np.float32)
                d = x != y
                rows |= set(np.flatnonzero(d.reshape(n, -1).any(1)).tolist())
        for r in rows:
            bad.setdefault(int(idx[r]), t)
    if not bad:
        s1, s2 = h.stats(), ora.stats()
        for i in (0, 1, 2, 3, 4, 12, 13):
            assert s1[i] == s2[i], f"stats[{i}] {s1[i]} != {s2[i]}"
    return bad


def _replay_all_host(O, H, C, L=None):
    bad = {}
    for m in np.unique(C["mode"]):
        bad.update(_replay_host(O, H, C, np.flatnonzero(C["mode"] == m), int(m), L))
    return bad


def _by_class(C, bad, first_tick_only=False):
    out = {}
    for r, t in bad.items():
        if first_tick_only and t != 0:
            continue
        k = C["classes"][C["cls"][r]]
        out[k] = out.get(k, 0) + 1
    return out


# ---- CPU tier ----------------------------------------------------------------------------------------------------

def test_corpus_classes_and_counts(oracle, hostsim):
    """every class has its minimum number of records, and stepping each record once on the host build reproduces its
    class -- and the very work record stored with it (catches a corpus made stale by a change to the physics)"""
    G, H, O = _gen(), hostsim, oracle
    C = _corpus()
    counts = {k: int((C["cls"] == i).sum()) for i, k in enumerate(C["classes"])}
    for name, _, minimum in G.CLASSES:
        minimum = G.REQUIRED.get(name, minimum)
        if minimum > 0:
            assert counts.get(name, 0) >= minimum, f"class {name}: {counts.get(name, 0)} records < {minimum}"
    assert sum(counts[k] for k in G.CUT_CLASSES) >= 64
    assert os.path.getsize(_CORPUS) < 1_600_000
    for m in np.unique(C["mode"]):
        idx = np.flatnonzero(C["mode"] == m)
        h = H.HostSimBatch(len(idx), mode=int(m), seed=11, fast=True)
        h.set_state(C["state"][idx])
        h.step(np.ascontiguousarray(C["actions"][idx, 0]), 0, 0, O.STEP_AUTORESET)
        w = h.last_work()
        for j, r in enumerate(idx):
            name = C["classes"][C["cls"][r]]
            assert name in G.classify(w[j]), f"record {r} no longer produces {name}: work {w[j].tolist()}"
        assert np.array_equal(w, C["work"][idx]), "host work records differ from the stored ones"


def test_host_build_equals_oracle_on_corpus(oracle, hostsim):
    C = _corpus()
    bad = _replay_all_host(oracle, hostsim, C)
    assert not bad, f"host build differs from the oracle, per class: {_by_class(C, bad)}; first: {sorted(bad.items())[:8]}"


# Textual mutants of the headers: (name, file, text, replacement, class whose first tick must then differ).
_MUTANTS = [
    # the three contacts of the (1,2,1) loop visited in reverse order (the shape is symmetric, so the loop still fits)
    ("reverse_3c121", "hk_world.cuh",
     "    case 7: return runVelocityIterationsFixedCore<1, 2, 1>(vcs, v, budget, velIters, sweepsOut);\n",
     "    case 7: { VC t0 = vcs[0]; vcs[0] = vcs[2]; vcs[2] = t0;\n"
     "      const int r = runVelocityIterationsFixedCore<1, 2, 1>(vcs, v, budget, velIters, sweepsOut);\n"
     "      t0 = vcs[0]; vcs[0] = vcs[2]; vcs[2] = t0; return r; }\n",
     "3c(1,2,1)"),
    # a period-2 cycle of the fixed-shape loops resolved to the other state of the cycle
    ("period2_parity", "hk_world.cuh",
     "      const int remaining = velIters - 1 - it;  // period-2 cycle: state after sweep it == state after sweep it - 2\n"
     "      if (remaining & 1) {",
     "      const int remaining = velIters - 1 - it;  // period-2 cycle: state after sweep it == state after sweep it - 2\n"
     "      if (!(remaining & 1)) {",
     "3c(1,2,1)"),
    # the skip after an event ignores how far the rest of the sweep approaches the static face
    ("skip_after_event_weak", "hk_world.cuh",
     "  return sepBoundOf(e, pid) - corr - disp > target + 0.25f * HK_LINEAR_SLOP + 0.004f;",
     "  return sepBoundOf(e, pid) - corr > target + 0.25f * HK_LINEAR_SLOP + 0.004f;",
     "toi2"),
]


def _copy_tree(dst):
    for rel in ("hockey_env_b200/csrc", "include"):
        shutil.copytree(os.path.join(_ROOT, rel), os.path.join(dst, rel))
    os.makedirs(os.path.join(dst, "tests", "hostsim"))
    shutil.copy(os.path.join(_HERE, "hostsim", "hostsim.cpp"), os.path.join(dst, "tests", "hostsim", "hostsim.cpp"))


@pytest.mark.parametrize("mutant", [None] + [m[0] for m in _MUTANTS])
def test_corpus_comparison_has_teeth(oracle, hostsim, tmp_path, mutant):
    """a copy of the headers with one planted mistake must fail the corpus comparison in the class the mistake targets
    (at that class's own first tick); the unmutated copy must pass"""
    H = hostsim
    root = str(tmp_path / "src")
    _copy_tree(root)
    target = None
    if mutant is not None:
        _, fname, old, new, target = next(m for m in _MUTANTS if m[0] == mutant)
        p = os.path.join(root, "hockey_env_b200", "csrc", fname)
        text = open(p).read()
        assert text.count(old) == 1, f"mutant {mutant}: the text to replace is not unique in {fname}"
        open(p, "w").write(text.replace(old, new))
    L = H.load(H.build(force=True, root=root))
    C = _corpus()
    bad = _replay_all_host(oracle, H, C, L)
    if mutant is None:
        assert not bad, f"unmutated copy differs: {_by_class(C, bad)}"
    else:
        first = _by_class(C, bad, first_tick_only=True)
        assert first.get(target, 0) > 0, f"mutant {mutant} not caught in {target} at its first tick: {_by_class(C, bad)}"


# ---- GPU tier ----------------------------------------------------------------------------------------------------

_ORACLE_CACHE = {}


def _oracle_run(O, key, states, actions, mode):
    """oracle outputs / states of every tick for one layout (shared by all cascade variants of that layout)"""
    if key not in _ORACLE_CACHE:
        n = states.shape[0]
        ora = O.OracleBatch(n, mode=mode, seed=13, n_threads=8)
        ora.set_state(states)
        ticks = []
        for t in range(actions.shape[1]):
            ro = ora.step(np.ascontiguousarray(actions[:, t]), O.POL_EXTERNAL, O.POL_EXTERNAL, O.STEP_AUTORESET)
            ticks.append((ro, ora.get_state()))
        _ORACLE_CACHE[key] = (ticks, ora.stats())
    return _ORACLE_CACHE[key]


def _gpu_env(hk, n, mode, var):
    knobs = ("HK_TIERS", "HK_PHASE_SYNC", "HK_TOUCH", "HK_LANE_TRACE")
    old = {k: os.environ.get(k) for k in knobs}
    for k in knobs:
        os.environ.pop(k, None)
    os.environ.update(var)
    try:
        return hk.HockeyVecEnv(n, mode=hk.Mode(mode), device="cuda:0", seed=13, want_agent_two=True)
    finally:
        for k, v in old.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v


def _run_gpu(O, key, states, actions, mode, var, trace=False):
    """the CUDA library against the oracle on one layout; returns the per-env lane-trace words of tick 0 if traced"""
    import torch
    import hockey_env_b200 as hk
    from parity_util import state_mismatches
    n = states.shape[0]
    ticks, ostats = _oracle_run(O, key, states, actions, mode)
    env = _gpu_env(hk, n, mode, dict(var, **({"HK_LANE_TRACE": "1"} if trace else {})))
    env.set_full_state(torch.from_numpy(states.view(np.int32)).cuda())
    rec0 = None
    for t in range(actions.shape[1]):
        env.step(torch.from_numpy(np.ascontiguousarray(actions[:, t])).cuda())
        if trace and t == 0:
            torch.cuda.synchronize()
            nw = n // 32 + 8
            buf = np.zeros(20 * nw + 2 * n, np.uint32)
            hk._lib.check(env.L.hk_debug_lane_trace(env._h, buf.ctypes.data, buf.size))
            rec0 = buf[4 * nw:4 * nw + 2 * n].reshape(n, 2)[:, 0].copy()
        ro, ost = ticks[t]
        for k, ten in (("obs", env.obs), ("obs2", env.obs2), ("done", env.done), ("final_obs", env.final_obs)):
            assert np.array_equal(ten.cpu().numpy(), ro[k]), f"{key} {var}: {k} differs at tick {t}"
        for k, ten in (("reward", env.reward), ("reward2", env.reward2), ("info", env.info), ("info2", env.info2)):
            assert np.array_equal(ten.cpu().numpy(), ro[k].astype(np.float32)), f"{key} {var}: {k} differs at tick {t}"
        bad = state_mismatches(ost, env.get_full_state().cpu().numpy().view(np.uint32))
        assert len(bad) == 0, f"{key} {var}: state differs at tick {t}: {bad[:8].tolist()}"
    s = env.stats()
    assert s["overflows"] == 0
    for k, i in (("episodes", 0), ("wins", 1), ("losses", 2), ("draws", 3), ("env_steps", 4), ("toi_events", 12)):
        assert s[k] == ostats[i], f"{key} {var}: stats {k}"
    return rec0


def _interleaved(C, m, n):
    idx = np.flatnonzero(C["mode"] == m)
    rows = np.resize(idx, n)  # records in corpus order, classes interleaved by repetition
    return rows


_VARIANTS = [{}, {"HK_TIERS": "3"}, {"HK_PHASE_SYNC": "0"}, {"HK_TOUCH": "1"}]


@pytest.mark.gpu
@pytest.mark.parametrize("var", _VARIANTS, ids=["default", "tiers3", "phase_sync0", "touch"])
def test_gpu_corpus_interleaved(oracle, var):
    """all classes interleaved at 4,096 envs, one batch per mode, in each cascade variant"""
    C = _corpus()
    for m in np.unique(C["mode"]):
        rows = _interleaved(C, m, 4096)
        _run_gpu(oracle, ("interleaved", int(m)), C["state"][rows], C["actions"][rows], int(m), var)


@pytest.mark.gpu
def test_gpu_corpus_each_class_tiled(oracle):
    """each class alone, tiled to 4,096 envs: one block holds many units of the same rare shape"""
    C = _corpus()
    for ci, name in enumerate(C["classes"]):
        for m in np.unique(C["mode"][C["cls"] == ci]):
            idx = np.flatnonzero((C["cls"] == ci) & (C["mode"] == m))
            rows = np.resize(idx, 4096)
            _run_gpu(oracle, ("tiled", name, int(m)), C["state"][rows], C["actions"][rows], int(m), {})


@pytest.mark.gpu
@pytest.mark.parametrize("var", [{}, {"HK_TOUCH": "1"}], ids=["default", "touch"])
def test_gpu_corpus_among_fast_envs(oracle, var):
    """every record placed among quiet fast-tier envs at 16,384: few general lanes, small automatic block shapes and the
    staged wide k_fast"""
    C = _corpus()
    n = 16384
    for m in np.unique(C["mode"]):
        idx = np.flatnonzero(C["mode"] == m)
        base = oracle.OracleBatch(n, mode=int(m), seed=13, n_threads=8)
        states = base.get_state()
        pos = (np.arange(len(idx)) * (n // len(idx))) + 7
        states[pos] = C["state"][idx]
        actions = np.zeros((n,) + C["actions"].shape[1:], np.float32)
        actions[pos] = C["actions"][idx]
        _run_gpu(oracle, ("sparse", int(m)), states, actions, int(m), var)


@pytest.mark.gpu
def test_gpu_corpus_coverage_trace(oracle):
    """HK_LANE_TRACE=1 on the interleaved batch: every record's class tick ran in the general tier with the contacts,
    manifold points and TOI events the host build recorded for it -- and the traced run still equals the oracle"""
    import hostsim_lib as H
    C = _corpus()
    seen = set()
    for m in np.unique(C["mode"]):
        rows = _interleaved(C, m, 4096)
        rec = _run_gpu(oracle, ("interleaved", int(m)), C["state"][rows], C["actions"][rows], int(m), {}, trace=True)
        for j, r in enumerate(rows):
            w = C["work"][r]
            name = C["classes"][C["cls"][r]]
            assert rec[j] != 0, f"record {r} ({name}) did not run in the general tier"
            toi, shape = (rec[j] >> 12) & 0xF, (rec[j] >> 20) & 0xFF
            assert toi == min(w[H.W_TOI], 15), f"record {r} ({name}): {toi} TOI events, host {w[H.W_TOI]}"
            if w[H.W_KIND] != 0:
                assert shape == (w[H.W_SHAPE] & 0xFF), f"record {r} ({name}): shape {shape:#x}, host {w[H.W_SHAPE]:#x}"
            seen.add(name)
    assert seen == set(C["classes"])
