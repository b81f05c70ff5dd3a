"""CPU tier of per-env game modes: the device code (tests/hostsim) against the oracle when envs of one batch play
different modes and switch mode at explicit and automatic resets; the record rule for word HK_S_MODE.
Both sides take the per-env modes through tests/modes (modes_lib)."""
import numpy as np
import pytest

import modes_lib as M
from parity_util import state_mismatches, outputs_equal

S_MODE = 56


def _pair(O, H, n, seed, fast, create_mode=0, modes=None):
    o = M.ModeOracleBatch(n, mode=create_mode, seed=seed, env_id_offset=3_000_000)
    h = M.ModeHostSimBatch(n, mode=create_mode, seed=seed, env_id_offset=3_000_000, fast=fast)
    if modes is not None:
        o.set_reset_modes(modes.copy())
        h.set_reset_modes(modes.copy())
    return o, h


def _check(o, h, t):
    bad = state_mismatches(o.get_state(), h.get_state())
    assert len(bad) == 0, f"state differs at tick {t}: {bad[:6].tolist()}"
    assert np.array_equal(o.modes(), h.modes()), f"modes differ at tick {t}"


@pytest.mark.parametrize("fast", [False, True])
def test_fixed_mix_matches_oracle(oracle, hostsim, fast):
    O, H = oracle, hostsim
    n = 96
    modes = (np.arange(n) % 3).astype(np.uint8)
    o, h = _pair(O, H, n, seed=11, fast=fast, modes=modes)
    ro, rh = o.reset(one_starting=np.ones(n, np.int8)), h.reset(one_starting=np.ones(n, np.int8))
    assert np.array_equal(ro, rh)
    assert np.array_equal(h.modes(), modes)
    _check(o, h, -1)
    for t in range(270):
        ro = o.step(None, O.POL_STRONG, O.POL_STRONG, O.STEP_AUTORESET)
        rh = h.step(None, O.POL_STRONG, O.POL_STRONG, O.STEP_AUTORESET)
        assert outputs_equal(ro, rh) == [], f"outputs differ at tick {t}"
        if t % 30 == 0:
            _check(o, h, t)
    _check(o, h, "end")
    so, sh = o.stats(), h.stats()
    assert np.array_equal(so[:11], sh[:11]) and so[12] == sh[12] and so[0] > n
    s = h.get_state()
    assert np.array_equal(s[:, S_MODE], np.where(modes == 0, 0, modes.astype(np.uint32) + 1))


@pytest.mark.parametrize("fast", [False, True])
def test_switching_at_explicit_and_auto_resets_matches_oracle(oracle, hostsim, fast):
    """Codes rewritten in place every few ticks: auto-resets and masked resets pick up the code of that moment."""
    O, H = oracle, hostsim
    n = 80
    rng = np.random.default_rng(5)
    modes = rng.integers(0, 3, n).astype(np.uint8)
    o, h = _pair(O, H, n, seed=23, fast=fast, create_mode=2, modes=modes)
    seen = set()
    for t in range(330):
        if t % 7 == 0:
            new = rng.integers(0, 3, n).astype(np.uint8)
            o.reset_modes[:] = new
            h.reset_modes[:] = new
        if t % 50 == 25:
            mask = (rng.random(n) < 0.3).astype(np.uint8)
            one = rng.integers(-1, 2, n).astype(np.int8)
            assert np.array_equal(o.reset(mask=mask, one_starting=one), h.reset(mask=mask, one_starting=one))
        ro = o.step(None, O.POL_STRONG, O.POL_WEAK, O.STEP_AUTORESET)
        rh = h.step(None, O.POL_STRONG, O.POL_WEAK, O.STEP_AUTORESET)
        assert outputs_equal(ro, rh) == [], f"outputs differ at tick {t}"
        seen.update(np.unique(h.modes()).tolist())
        if t % 25 == 0:
            _check(o, h, t)
    _check(o, h, "end")
    assert seen == {0, 1, 2}
    so, sh = o.stats(), h.stats()
    assert np.array_equal(so[:11], sh[:11]) and so[12] == sh[12] and so[0] > 0


def test_clearing_the_codes_keeps_each_env_mode(oracle, hostsim):
    O, H = oracle, hostsim
    n = 30
    modes = (np.arange(n) % 3).astype(np.uint8)
    o, h = _pair(O, H, n, seed=3, fast=True, modes=modes)
    o.reset(one_starting=np.ones(n, np.int8))
    h.reset(one_starting=np.ones(n, np.int8))
    o.set_reset_modes(None)
    h.set_reset_modes(None)
    for t in range(200):
        ro = o.step(None, O.POL_STRONG, O.POL_STRONG, O.STEP_AUTORESET)
        rh = h.step(None, O.POL_STRONG, O.POL_STRONG, O.STEP_AUTORESET)
        assert outputs_equal(ro, rh) == [], f"outputs differ at tick {t}"
    assert np.array_equal(h.modes(), modes) and np.array_equal(o.modes(), modes)
    _check(o, h, "end")


@pytest.mark.parametrize("create_mode", [0, 2])
def test_mode_word_of_the_record(oracle, hostsim, create_mode):
    """Word 56: 0 = the creation mode, m + 1 = mode m; on reading, 0 and values above 3 mean the creation mode."""
    O, H = oracle, hostsim
    n = 12
    modes = (np.arange(n) % 3).astype(np.uint8)
    o, h = _pair(O, H, n, seed=8, fast=True, create_mode=create_mode, modes=modes)
    o.reset(one_starting=np.ones(n, np.int8))
    h.reset(one_starting=np.ones(n, np.int8))
    for _ in range(30):
        o.step(None, O.POL_STRONG, O.POL_STRONG, O.STEP_AUTORESET)
        h.step(None, O.POL_STRONG, O.POL_STRONG, O.STEP_AUTORESET)
    want = np.where(modes == create_mode, 0, modes.astype(np.uint32) + 1)
    for impl in (o, h):
        s = impl.get_state()
        assert np.array_equal(s[:, S_MODE], want)
        # round trip into a fresh batch of the same creation mode
        for Batch in (M.ModeOracleBatch, M.ModeHostSimBatch):
            b = Batch(n, mode=create_mode, seed=8, env_id_offset=3_000_000)
            b.set_state(s)
            assert np.array_equal(b.modes(), modes)
            assert len(state_mismatches(s, b.get_state())) == 0
    # records of builds without per-env modes (word 56 = 0) and out-of-range words read as the creation mode
    s = h.get_state()
    s[:, S_MODE] = np.where(np.arange(n) % 2 == 0, 0, 4 + np.arange(n)).astype(np.uint32)
    for Batch in (M.ModeOracleBatch, M.ModeHostSimBatch):
        b = Batch(n, mode=create_mode, seed=8, env_id_offset=3_000_000)
        b.set_state(s)
        assert np.array_equal(b.modes(), np.full(n, create_mode, np.uint8))
        assert np.array_equal(b.get_state()[:, S_MODE], np.zeros(n, np.uint32))


def test_single_mode_records_keep_word_56_zero(oracle, hostsim):
    O, H = oracle, hostsim
    for mode in (0, 1, 2):
        o, h = _pair(O, H, 16, seed=4, fast=True, create_mode=mode)
        for _ in range(90):
            o.step(None, O.POL_STRONG, O.POL_STRONG, O.STEP_AUTORESET)
            h.step(None, O.POL_STRONG, O.POL_STRONG, O.STEP_AUTORESET)
        assert not o.get_state()[:, S_MODE].any() and not h.get_state()[:, S_MODE].any()
        assert np.array_equal(h.modes(), np.full(16, mode, np.uint8))
