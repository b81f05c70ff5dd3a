"""Per-env game modes on the GPU: a mixed batch equals, env for env, single-mode batches of each env's mode; mode
switches at explicit and automatic resets match the CPU oracle; every execution path agrees; the Python surface
(HockeyEnv mode setter, reset(mode=...), HockeyGymVectorEnv options, training.ModeMix)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import modes_lib as M  # noqa: E402  (the CPU oracle with per-env modes)

S_MODE = 56
_KNOBS = ("HK_MONO", "HK_TIERS", "HK_TOUCH", "HK_FUSED", "HK_FAST_WIDE")


def _state(env):
    return env.get_full_state().cpu().numpy().view(np.uint32)


def _with_env(var, make):
    """make() with exactly the execution knobs in `var` set (they are read when a handle is created)."""
    old = {k: os.environ.get(k) for k in _KNOBS}
    for k in _KNOBS:
        os.environ.pop(k, None)
    os.environ.update(var)
    try:
        return make()
    finally:
        for k, v in old.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v


_OUT = ("obs", "obs2", "reward", "reward2", "done", "info", "info2", "final_obs")


@pytest.mark.parametrize("n,var", [(4096, {}), (16384, {}), (4096, {"HK_TOUCH": "1"})])
def test_mixed_batch_equals_single_mode_batches(n, var):
    import hockey_env_b200 as hk
    from parity_util import state_mismatches
    modes = torch.arange(n, device="cuda:0") % 3
    kw = dict(device="cuda:0", seed=19, env_id_offset=40_000, p1="strong", p2="strong", want_agent_two=True)
    mixed = _with_env(var, lambda: hk.HockeyVecEnv(n, mode=modes.to(torch.uint8), **kw))
    single = [_with_env(var, lambda m=m: hk.HockeyVecEnv(n, mode=hk.Mode(m), **kw)) for m in range(3)]
    for s in single:
        s.reset(one_starting=True)
    assert torch.equal(mixed.modes(), modes.to(torch.uint8))
    sel = [(modes == m) for m in range(3)]

    def pick(name):
        t = [getattr(s, name) for s in single]
        shape = (-1,) + (1,) * (t[0].dim() - 1)
        return torch.where(sel[0].view(shape), t[0], torch.where(sel[1].view(shape), t[1], t[2]))

    for name in ("obs", "obs2", "info", "info2"):
        assert torch.equal(getattr(mixed, name), pick(name)), f"{name} differs after the first reset"
    for t in range(300):
        mixed.step()
        for s in single:
            s.step()
        for name in _OUT:
            assert torch.equal(getattr(mixed, name), pick(name)), f"{name} differs at tick {t}"
    ref = np.where(sel[0].cpu().numpy()[:, None], _state(single[0]),
                   np.where(sel[1].cpu().numpy()[:, None], _state(single[1]), _state(single[2])))
    got = _state(mixed)
    assert np.array_equal(got[:, S_MODE], np.where(modes.cpu().numpy() == 0, 0, modes.cpu().numpy() + 1))
    got[:, S_MODE] = 0
    bad = state_mismatches(ref, got)
    assert len(bad) == 0, f"state differs: {bad[:8].tolist()}"
    st = mixed.stats()
    assert st["episodes"] > n and st["overflows"] == 0


def test_mode_switching_matches_oracle(oracle):
    import hockey_env_b200 as hk
    from parity_util import state_mismatches, outputs_equal
    O = oracle
    n, seed = 384, 61
    rng = np.random.default_rng(3)
    env = hk.HockeyVecEnv(n, mode=hk.Mode.TRAIN_SHOOTING, device="cuda:0", seed=seed, env_id_offset=9_000, p1="strong",
                          p2="weak", want_agent_two=True)
    ora = M.ModeOracleBatch(n, mode=O.MODE_TRAIN_SHOOTING, seed=seed, env_id_offset=9_000)
    codes = rng.integers(0, 3, n).astype(np.uint8)
    env.set_reset_modes(torch.from_numpy(codes))
    ora.set_reset_modes(codes.copy())
    seen = set()
    for t in range(400):
        if t % 20 == 0:
            codes = rng.integers(0, 3, n).astype(np.uint8)
            env.reset_modes.copy_(torch.from_numpy(codes))
            ora.reset_modes[:] = codes
        if t == 130:  # explicit masked reset with per-env modes: also rewrites those envs' codes
            mask = rng.random(n) < 0.4
            m = rng.integers(0, 3, n).astype(np.uint8)
            env.reset(mask=torch.from_numpy(mask), mode=torch.from_numpy(m))
            ora.reset_modes[mask] = m[mask]
            ora.reset(mask=mask.astype(np.uint8))
            assert np.array_equal(env.obs.cpu().numpy(), ora.get_obs()[0])
            assert np.array_equal(env.reset_modes.cpu().numpy(), ora.reset_modes)
        env.step()
        ro = ora.step(None, O.POL_STRONG, O.POL_WEAK, O.STEP_AUTORESET)
        rh = {k: getattr(env, k).cpu().numpy() for k in _OUT}
        assert outputs_equal(ro, rh) == [], f"outputs differ at tick {t}"
        if t % 40 == 0 or t == 399:
            assert np.array_equal(env.modes().cpu().numpy(), ora.modes()), f"modes differ at tick {t}"
            bad = state_mismatches(ora.get_state(), _state(env))
            assert len(bad) == 0, f"state differs at tick {t}: {bad[:8].tolist()}"
        seen.update(np.unique(ora.modes()).tolist())
    assert seen == {0, 1, 2}
    s, so = env.stats(), ora.stats()
    for k, i in (("episodes", 0), ("wins", 1), ("losses", 2), ("draws", 3), ("env_steps", 4), ("toi_events", 12)):
        assert s[k] == so[i], k
    assert s["episodes"] > n


def test_execution_variants_agree_on_a_switching_batch():
    """Monolithic kernel, 3-tier cascade and hk_rollout (per-tick cascade and fused) read the reset codes alike."""
    import hockey_env_b200 as hk
    from parity_util import state_mismatches
    n = 4096
    rng = np.random.default_rng(12)
    draws = [torch.from_numpy(rng.integers(0, 3, n).astype(np.uint8)).cuda() for _ in range(16)]
    first = torch.from_numpy(rng.integers(0, 3, n).astype(np.uint8)).cuda()
    variants = ({}, {"HK_TIERS": "3"}, {"HK_MONO": "1"}, {"HK_FUSED": "1"}, {"HK_TOUCH": "1", "HK_FAST_WIDE": "1"})
    envs = [_with_env(v, lambda: hk.HockeyVecEnv(n, mode=first.clone(), device="cuda:0", seed=5, p1="strong", p2="strong"))
            for v in variants]
    for k in range(15):  # 15 x 20 ticks, codes rewritten every 20 ticks
        for e in envs:
            e.reset_modes.copy_(draws[k])
        envs[0].rollout(20, "strong", "strong")  # per-tick cascade
        envs[1].rollout(20, "strong", "strong")  # 3 tiers
        envs[2].rollout(20, "strong", "strong")  # HK_MONO: K ticks in one launch
        envs[3].rollout(20, "strong", "strong")  # HK_FUSED: k_rollout_fused
        for _ in range(20):
            envs[4].step()
    ref = _state(envs[0])
    assert len(np.unique(ref[:, S_MODE])) > 1
    for v, e in zip(variants[1:], envs[1:]):
        bad = state_mismatches(ref, _state(e))
        assert len(bad) == 0, f"{v}: state differs {bad[:8].tolist()}"
    s = [e.stats() for e in envs]
    assert s[0]["episodes"] > 0
    assert all(x["episodes"] == s[0]["episodes"] and x["wins"] == s[0]["wins"] for x in s[1:])


def test_hockey_env_mode_setter_and_reset_mode(oracle):
    import hockey_env_b200 as hk
    O = oracle
    for how in ("setter", "reset"):
        env = hk.HockeyEnv(mode=hk.Mode.NORMAL, seed=123)
        ora = M.ModeOracleBatch(1, mode=O.MODE_NORMAL, seed=123)
        ora.set_reset_modes(np.array([2], np.uint8))
        if how == "setter":
            env.mode = hk.Mode.TRAIN_DEFENSE
            assert env.max_timesteps == 250  # the setter only records the mode; reset applies it
            obs, info = env.reset()
        else:
            obs, info = env.reset(mode="TRAIN_DEFENSE")
        assert env.mode == hk.Mode.TRAIN_DEFENSE and env.max_timesteps == 80
        ro = ora.reset()
        assert np.array_equal(obs.astype(np.float32), ro[0])
        assert env._vec.modes().tolist() == [2]
        rng = np.random.default_rng(1)
        factors = []
        for episode in range(6):
            if episode:
                env.reset()
                assert np.array_equal(env._obs_np(env._vec.obs).astype(np.float32), ora.reset()[0])
            steps, done = 0, False
            while not done:
                a = np.concatenate([rng.uniform(-0.3, 0.3, 4), np.zeros(4)])  # player 1 barely moves
                obs, r, done, _, info = env.step(a)
                ro = ora.step(a.astype(np.float32)[None], O.POL_EXTERNAL, O.POL_EXTERNAL, 0)
                assert np.array_equal(obs.astype(np.float32), ro["obs"][0])
                assert np.float32(r) == ro["reward"].astype(np.float32)[0] and done == bool(ro["done"][0])
                steps += 1
                c = info["reward_closeness_to_puck"]
                if c != 0:
                    d = obs[0:2].astype(np.float32) - obs[12:14].astype(np.float32)
                    factors.append(c / np.hypot(float(d[0]), float(d[1])))
            # time runs 0..80: done once time >= max_timesteps = 80 (hockey_env.py:690), earlier only on a goal
            assert steps == 81 if info["winner"] == 0 else steps < 81
        # closeness factor of an 80-step episode: -30 / ((250/60) * 80 / 2) = -0.18 per unit of distance
        assert factors and np.allclose(factors, -0.18, rtol=1e-4)
        # back to NORMAL at the next reset
        env.mode = hk.Mode.NORMAL
        env.reset()
        assert env.max_timesteps == 250 and env._vec.modes().tolist() == [0]
        env.close()


def test_gym_vector_env_mode_option():
    import hockey_env_b200 as hk
    from hockey_env_b200.vector import HockeyGymVectorEnv
    n = 64
    v = HockeyGymVectorEnv(n, mode=[hk.Mode(i % 3) for i in range(n)], opponent="weak", seed=2)
    assert v.env.modes().cpu().tolist() == [i % 3 for i in range(n)]
    v.reset(options={"mode": "TRAIN_DEFENSE"})
    assert v.env.modes().cpu().tolist() == [2] * n
    mask = np.arange(n) % 2 == 0
    v.reset(options={"mode": hk.Mode.NORMAL, "reset_mask": mask})
    assert v.env.modes().cpu().tolist() == [0 if i % 2 == 0 else 2 for i in range(n)]
    for _ in range(260):  # the modes hold across auto-resets
        v.step(np.zeros((n, 4), np.float32))
    assert v.env.modes().cpu().tolist() == [0 if i % 2 == 0 else 2 for i in range(n)]
    v.close()


def test_mode_mix_draws_and_counters():
    import hockey_env_b200 as hk
    from hockey_env_b200.training import ModeMix
    n = 8192
    env = hk.HockeyVecEnv(n, device="cuda:0", seed=4, p1="strong", p2="weak")
    probs = (0.5, 0.3, 0.2)
    mix = ModeMix(env, probs=probs, seed=9)
    mix.reset(one_starting=True)
    env.clear_stats()
    drawn = torch.zeros(3, dtype=torch.float64, device="cuda:0")  # codes drawn for the envs that auto-reset
    for _ in range(600):
        _, _, done, _, info = env.step()
        mix.update(done, info["winner"])
        drawn += torch.bincount(mix.codes[done.bool()].long(), minlength=3).to(torch.float64)
    c = mix.counts.cpu().numpy()
    s = env.stats()
    total = c[:, 0].sum()
    assert total == s["episodes"] > n
    assert c[:, 1].sum() == s["wins"] and c[:, 2].sum() == s["losses"] and c[:, 3].sum() == s["draws"]
    assert np.array_equal(c[:, 0], c[:, 1:].sum(1))
    # finished episodes by mode are skewed (NORMAL episodes last longer); the draws themselves follow `probs`
    f = drawn.cpu().numpy()
    k = f.sum()
    assert k == total
    for m in range(3):
        sd = np.sqrt(k * probs[m] * (1 - probs[m]))
        assert abs(f[m] - k * probs[m]) < 5 * sd, (m, f[m], k * probs[m])
    # curriculum: after set_probs every new draw is TRAIN_DEFENSE.  Drawn one episode ahead: an env finishes its running
    # episode and the one already drawn for it (at most 251 ticks each) before it plays a draw made after set_probs.
    mix.set_probs((0, 0, 1))
    for _ in range(520):
        mix.step()
    assert bool((mix.codes == 2).all())
    assert bool((env.modes() == 2).all())
    # each finished episode is credited to the mode it was played in
    for m, row in zip(hk.Mode, mix.counts.cpu().numpy()):
        assert row[0] > 0, m
