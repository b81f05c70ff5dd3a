"""Exploration noise with on-device state in the fused actor epilogue: hk_actor_forward_explore /
hk_actor_forward_pool_explore (a per-slot AR(1) process, x' = rho x + scale z, that covers Gaussian and Ornstein-Uhlenbeck
noise), `ExplorationNoise`, noise= / reset= on `FusedActor` and `FusedActorPool`, and the training loops above them:
collect(noise=), td3.train(fused=True, noise=) and td3.train_population(noise=) with one slot per member."""
import math
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_actor_train import NPZ, _golden, _obs, _random_actor, _zero_actor  # noqa: E402  actors and observations

F32 = np.float32


# ---- CPU ------------------------------------------------------------------------------------------------------------

def test_explore_abi_error_convention_without_gpu():
    import hockey_env_b200 as hk
    L = hk.load_library()
    INV = hk._lib.HK_E_INVALID
    A = 0x10000  # an aligned address: every call below is rejected before anything is read through it

    def fwd(params=A, obs=A, act=A, stride=4, n=100, seed=1, counter=A, slots=A, state=A, reset=None, row0=0, device=0):
        return L.hk_actor_forward_explore(params, obs, act, stride, n, seed, counter, slots, state, reset, row0, device, None)

    def pool(params=A, k=2, choice=A, obs=A, act=A, stride=4, n=100, scratch=A, seed=1, counter=A, slots=A, state=A, reset=None,
             row0=0, device=0):
        return L.hk_actor_forward_pool_explore(params, k, choice, obs, act, stride, n, scratch, seed, counter, slots, state, reset,
                                               row0, device, None)

    explore_cases = [(dict(counter=None), b"NULL"), (dict(slots=None), b"NULL"), (dict(state=None), b"NULL"),
                     (dict(counter=A + 4), b"counter needs 8-byte"), (dict(slots=A + 8), b"16-byte"), (dict(state=A + 4), b"16-byte"),
                     (dict(row0=-1), b"row0")]
    fwd_cases = [(dict(params=None), b"NULL"), (dict(obs=None), b"NULL"), (dict(act=None), b"NULL"), (dict(n=0), b"n must be"),
                 (dict(n=-5), b"n must be"), (dict(stride=3), b"act_stride"), (dict(params=A + 8), b"alignment"),
                 (dict(obs=A + 4), b"alignment")]
    pool_cases = [(dict(params=None), b"NULL"), (dict(choice=None), b"NULL"), (dict(obs=None), b"NULL"), (dict(act=None), b"NULL"),
                  (dict(scratch=None), b"NULL"), (dict(n=0), b"n must be"), (dict(n=2**31), b"n must be"),
                  (dict(stride=3), b"act_stride"), (dict(k=0), b"k must be"), (dict(k=4097), b"k must be"),
                  (dict(choice=A + 2), b"alignment"), (dict(scratch=A + 4), b"alignment")]
    for fn, name, cases in ((fwd, b"hk_actor_forward_explore", fwd_cases + explore_cases),
                            (pool, b"hk_actor_forward_pool_explore", pool_cases + explore_cases)):
        for kw, msg in cases:
            assert fn(**kw) == INV, (name, kw)
            err = L.hk_last_error()
            assert name + b":" in err and msg in err, (kw, err)
        if not torch.cuda.is_available():
            # valid arguments, with and without a reset mask (u8: any address), reach the device probe
            for reset in (None, A, A + 1):
                assert fn(reset=reset) == hk._lib.HK_E_NODEVICE, (name, reset)
                assert b"no CUDA device" in L.hk_last_error()


@pytest.mark.parametrize("kw, msg", [
    (dict(sigma=-0.1), "sigma"), (dict(sigma=float("nan")), "sigma"), (dict(sigma=float("inf")), "sigma"),
    (dict(theta=-0.5), "theta"), (dict(theta=float("nan")), "theta"), (dict(theta=float("inf")), "theta"),
    (dict(dt=0.0), "dt"), (dict(dt=-1e-2), "dt"), (dict(dt=float("nan")), "dt"),
    (dict(theta=150.0, dt=1e-2), r"theta \* dt"), (dict(clip=-0.1), "clip"), (dict(clip=float("nan")), "clip"),
    (dict(slots=2, sigma=[0.1, -0.1]), "sigma"), (dict(slots=2, theta=[0.15, -1.0]), "theta"),
    (dict(slots=3, sigma=[0.1, 0.2]), "2 entries for 3 slots"), (dict(n=0), "n >= 1"), (dict(slots=0), "slots >= 1"),
])
def test_exploration_noise_validates_before_touching_a_device(kw, msg):
    import hockey_env_b200 as hk
    args = dict(n=16, device="cpu")  # a valid call on the CPU would raise HockeyLibraryError, not ValueError
    args.update(kw)
    with pytest.raises(ValueError, match=msg):
        hk.ExplorationNoise(**args)
    if not torch.cuda.is_available():
        with pytest.raises(hk.HockeyLibraryError):
            hk.ExplorationNoise(16, device="cpu")


def test_slot_mapping_gaussian_and_ou():
    from hockey_env_b200 import ExplorationNoise
    row = ExplorationNoise.slot_row
    inf = math.inf
    assert row(0.3) == (0.0, float(F32(0.3)), inf)                             # Gaussian: rho 0, scale sigma, no clip
    assert row(0.3, clip=0.5, dt=0.7) == (0.0, float(F32(0.3)), float(F32(0.5)))  # dt does not enter a Gaussian slot
    assert row(0.0, clip=0.0) == (0.0, 0.0, 0.0)
    # OU: rho = 1 - theta dt, scale = sigma sqrt(dt), each computed in float64 and rounded to float32 once
    assert row(0.2, theta=0.15, dt=1e-2) == (float(F32(1 - 0.15 * 1e-2)), float(F32(0.2 * math.sqrt(1e-2))), inf)
    assert row(0.5, clip=0.3, theta=2.0, dt=0.05) == (float(F32(0.9)), float(F32(0.5 * math.sqrt(0.05))), float(F32(0.3)))
    assert row(1.0, theta=0.0, dt=0.25) == (1.0, 0.5, inf)   # theta 0: a random walk
    assert row(1.0, theta=100.0, dt=0.01) == (0.0, float(F32(0.1)), inf)  # theta dt = 1: the bound is allowed
    # float64 then one rounding: sigma sqrt(dt) rounded once differs from float32 arithmetic here
    scale32 = F32(0.2) * np.sqrt(F32(1e-2))
    assert row(0.2, theta=0.15, dt=1e-2)[1] == float(F32(0.2 * math.sqrt(1e-2))) != float(scale32)
    for v in row(0.37, clip=0.11, theta=0.3, dt=0.013):
        assert float(F32(v)) == v


def test_training_loops_reject_noise_with_noise_scale_or_unfused():
    from hockey_env_b200 import td3
    from hockey_env_b200.td3 import TD3Config
    noise = SimpleNamespace(n=10, slots=2)
    with pytest.raises(ValueError, match="not both"):
        td3.train(SimpleNamespace(), SimpleNamespace(), 1, noise_scale=0.2, fused=True, noise=noise)
    with pytest.raises(ValueError, match="fused=True"):
        td3.train(SimpleNamespace(), SimpleNamespace(), 1, noise=noise)
    pop = SimpleNamespace(k=2, configs=[TD3Config(action_noise_scale=0.2), TD3Config(action_noise_scale=0.3)])
    with pytest.raises(ValueError, match="not both"):
        td3.train_population(SimpleNamespace(num_envs=10), pop, ticks=1, noise_scale=0.2, noise=noise)
    with pytest.raises(ValueError, match="2 slots"):
        td3.train_population(SimpleNamespace(num_envs=10), pop, ticks=1, noise=SimpleNamespace(n=10, slots=3))
    with pytest.raises(ValueError, match="10 rows"):
        td3.train_population(SimpleNamespace(num_envs=10), pop, ticks=1, noise=SimpleNamespace(n=12, slots=2))


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _bits(t):
    return t.contiguous().view(torch.int32).cpu()


def _slots(*rows):
    """[S, 4] float32 table of (rho, scale, clip) rows."""
    return torch.tensor([list(r) + [0.0] for r in rows], dtype=torch.float32, device="cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129, 65_536 + 5])
def test_gaussian_slot_equals_the_noisy_launch(n):
    import hockey_env_b200 as hk
    f = hk.FusedActor(_golden("cuda:0")[0], seed=0xABCDEF0123)
    obs = _obs(n, n)
    for sigma, clip, row0, ctr in ((0.3, 0.5, 0, 7), (1.0, None, 3_000_000_000, (2 << 32) + 5)):
        a8 = torch.full((n, 8), 5.0, device="cuda:0")
        f.counter.fill_(ctr)
        f(obs, out=a8[:, 4:], noise=sigma, noise_clip=clip, row0=row0)
        ex = hk.ExplorationNoise(n, sigma=sigma, clip=clip)
        b8 = torch.full((n, 8), 5.0, device="cuda:0")
        f.counter.fill_(ctr)
        f(obs, out=b8[:, 4:], noise=ex, row0=row0)
        assert int(f.counter) == ctr + 1
        assert torch.equal(_bits(a8), _bits(b8)), (sigma, clip)
    # the state of a Gaussian slot is the unclipped sigma z: with a zero actor and no clip, act = clamp(state)
    z = hk.FusedActor(_zero_actor(), seed=5)
    ex = hk.ExplorationNoise(n, sigma=0.5)
    act = z(obs, noise=ex).clone()
    assert torch.equal(act, ex.state.clamp(-1, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 16])
@pytest.mark.parametrize("n", [1, 129, 65_536 + 5])
def test_pool_gaussian_slots_equal_the_noisy_pool_launch(n, k):
    import hockey_env_b200 as hk
    actors = [_golden("cuda:0")[s % 2] if s < 2 else _random_actor(s) for s in range(k)]
    pool = hk.FusedActorPool(actors, seed=99)
    obs = _obs(n, n + k)
    g = torch.Generator(device="cuda:0").manual_seed(n + k)
    choice = torch.randint(-1, k, (n,), device="cuda:0", generator=g, dtype=torch.int32)
    a8 = torch.full((n, 8), 3.0, device="cuda:0")
    pool.counter.fill_(11)
    pool(obs, choice, out=a8[:, 4:], noise=0.25, noise_clip=0.4, row0=17)
    ex = hk.ExplorationNoise(n, slots=k, sigma=0.25, clip=0.4)
    ex.state.fill_(-7.0)
    b8 = torch.full((n, 8), 3.0, device="cuda:0")
    pool.counter.fill_(11)
    pool(obs, choice, out=b8[:, 4:], noise=ex, row0=17)
    assert torch.equal(_bits(a8), _bits(b8))
    skipped = (choice < 0).cpu()
    assert bool((ex.state.cpu()[skipped] == -7.0).all())  # rows that are not written keep their state


def _unit_z(call, ex, ctr):
    """The normals z_ctr of every row: one call with every slot (rho 0, scale 1, no clip) leaves z in the state."""
    table = ex.table.clone()
    ex.table.copy_(_slots(*[(0.0, 1.0, math.inf)] * ex.slots))
    call(ctr, None)
    z = ex.state.clone()
    ex.table.copy_(table)
    return z


def _ar1(rho, scale, x, z, reset=None):
    """fl(fl(rho x) + fl(scale z)) in float32 torch ops (x = 0 where reset), and fl(scale z) where rho == 0; rho / scale
    are scalars or per-row [n, 1]."""
    if reset is not None:
        x = torch.where(reset.bool().unsqueeze(1), torch.zeros_like(x), x)
    sz = torch.mul(scale, z)
    return torch.where(torch.as_tensor(rho) == 0, sz, torch.add(torch.mul(rho, x), sz))


@pytest.mark.gpu
def test_exact_recurrence_and_reset():
    import hockey_env_b200 as hk
    n, ctr = 10_003, (1 << 32) + 77
    f = hk.FusedActor(_golden("cuda:0")[1], seed=4242)
    obs = _obs(n, 8)
    base = f(obs).clone()
    ex = hk.ExplorationNoise(n, sigma=0.6, clip=0.45, theta=3.0, dt=0.05)
    rho, scale, clip = [float(v) for v in ex.table[0, :3].cpu()]
    assert (rho, scale) == (float(F32(0.85)), float(F32(0.6 * math.sqrt(0.05))))

    def call(c, reset):
        f.counter.fill_(c)
        return f(obs, noise=ex, reset=reset).clone()

    z = _unit_z(call, ex, ctr).cpu()
    g = torch.Generator().manual_seed(3)
    x0 = torch.randn((n, 4), generator=g) * 0.7
    reset = torch.rand(n, generator=g) < 0.3
    for rst in (None, reset.cuda(), reset.to(torch.uint8).cuda()):
        ex.state.copy_(x0)
        act = call(ctr, rst).cpu()
        want = _ar1(torch.tensor(rho), torch.tensor(scale), x0, z, None if rst is None else reset)
        got = ex.state.cpu()
        assert torch.equal(_bits(got), _bits(want)), rst
        if rst is not None:  # reset rows start from 0: exactly fl(scale z)
            assert torch.equal(_bits(got[reset]), _bits(torch.mul(torch.tensor(scale), z[reset])))
        want_act = (base.cpu() + want.clamp(-clip, clip)).clamp(-1.0, 1.0)
        assert torch.equal(_bits(act), _bits(want_act))
    # the reset tensor is read, not written, and the counter advanced once per call
    assert int(f.counter) == ctr + 1


@pytest.mark.gpu
def test_pool_rows_use_their_own_slot_and_grouping_does_not_matter():
    import hockey_env_b200 as hk
    k, n, ctr = 3, 40_000 + 11, 9
    actors = [_golden("cuda:0")[0], _golden("cuda:0")[1], _random_actor(41)]
    obs = _obs(n, 21)
    g = torch.Generator(device="cuda:0").manual_seed(2)
    choice = torch.randint(-1, k, (n,), device="cuda:0", generator=g, dtype=torch.int32)
    reset = torch.rand(n, device="cuda:0", generator=g) < 0.2
    slot_args = dict(sigma=[0.3, 0.5, 0.8], clip=[0.5, None, 0.2], theta=[None, 0.15, 2.0], dt=[1e-2, 1e-2, 0.1])
    x0 = torch.randn((n, 4), device="cuda:0", generator=g) * 0.5

    def run(perm):
        """Snapshot s of the pool and slot s of the table become label perm[s]: other groups and tile order, same rows."""
        inv = [perm.index(s) for s in range(k)]
        pool = hk.FusedActorPool([actors[inv[s]] for s in range(k)], seed=31)
        ex = hk.ExplorationNoise(n, slots=k, **{key: [v[inv[s]] for s in range(k)] for key, v in slot_args.items()})
        ch = torch.where(choice >= 0, torch.tensor(perm, device="cuda:0", dtype=torch.int32)[choice.long().clamp(min=0)], choice)

        def call(c, rst):
            pool.counter.fill_(c)
            return pool(obs, ch, out=out, noise=ex, reset=rst)

        out = torch.full((n, 4), 6.0, device="cuda:0")
        z = _unit_z(call, ex, ctr)
        ex.state.copy_(x0)
        out = torch.full((n, 4), 6.0, device="cuda:0")
        call(ctr, reset)
        base = pool(obs, ch, out=torch.full((n, 4), 6.0, device="cuda:0")).clone()
        return out.clone(), ex.state.clone(), z, base, ex.table[ch.long().clamp(min=0)].clone()

    out, state, z, base, tab = run([0, 1, 2])
    rows = choice >= 0
    want = _ar1(tab[:, :1], tab[:, 1:2], x0, z, reset)
    assert torch.equal(_bits(state[rows]), _bits(want[rows]))
    clip = tab[:, 2:3]
    want_act = torch.minimum(torch.maximum(base + torch.minimum(torch.maximum(want, -clip), clip), torch.tensor(-1.0, device="cuda:0")),
                             torch.tensor(1.0, device="cuda:0"))
    assert torch.equal(_bits(out[rows]), _bits(want_act[rows]))
    # choice -1 rows: act and state byte-identical
    assert bool((out[~rows] == 6.0).all()) and torch.equal(_bits(state[~rows]), _bits(x0[~rows]))
    # three different slot parameterisations are in use
    assert len({tuple(r) for r in tab[rows].cpu().tolist()}) == 3
    for perm in ([2, 0, 1], [1, 2, 0]):
        o2, s2, _, _, _ = run(perm)
        assert torch.equal(_bits(o2), _bits(out)) and torch.equal(_bits(s2), _bits(state)), perm


@pytest.mark.gpu
def test_ou_statistics():
    import hockey_env_b200 as hk
    n, rho, scale, calls = 65_536, 0.9, 0.2, 100
    f = hk.FusedActor(_zero_actor(), seed=123)
    obs = _obs(n, 1)
    ex = hk.ExplorationNoise(n, sigma=scale / math.sqrt(0.01), theta=(1 - rho) / 0.01, dt=0.01)
    r, s, _ = [float(v) for v in ex.table[0, :3].cpu()]
    assert abs(r - rho) < 1e-7 and abs(s - scale) < 1e-7
    for _ in range(calls - 1):
        f(obs, noise=ex)
    prev = ex.state.double().cpu().flatten().numpy()
    act = f(obs, noise=ex).double().cpu().flatten().numpy()
    x = ex.state.double().cpu().flatten().numpy()
    assert np.array_equal(act, np.clip(x, -1, 1))  # a zero actor with no clip: the action is the clamped state
    m = x.size
    var, want = x.var(), s * s / (1 - r * r)
    assert abs(var - want) < 5 * want * math.sqrt(2.0 / (m - 1)), (var, want)
    ac = np.corrcoef(prev, x)[0, 1]
    assert abs(ac - r) < 5 * (1 - r * r) / math.sqrt(m), (ac, r)


@pytest.mark.gpu
def test_captured_pool_graph_follows_the_counter_state_and_table():
    import hockey_env_b200 as hk
    k, n = 3, 20_000
    pool = hk.FusedActorPool([_golden("cuda:0")[0], _golden("cuda:0")[1], _random_actor(7)], seed=12)
    obs = _obs(n, 5)
    choice = (torch.arange(n, device="cuda:0") % k).to(torch.int32)
    choice[::7] = -1
    ex = hk.ExplorationNoise(n, slots=k, sigma=0.4, theta=0.5, dt=0.1)
    out = torch.zeros((n, 4), device="cuda:0")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pool(obs, choice, out=out, noise=ex)  # warm-up: kernel attributes set, scratch allocated
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        pool(obs, choice, out=out, noise=ex)
    plain = pool(obs, choice, out=torch.zeros((n, 4), device="cuda:0")).clone()

    def sequence():
        pool.counter.fill_(1000)
        ex.reset()
        for m in range(k):
            ex.set(m, sigma=0.4, theta=0.5)
        rec = []
        for j in range(4):
            if j == 2:
                ex.set(1, sigma=0.0, theta=None)  # member 1 stops exploring from the next replay on
            graph.replay()
            rec.append((out.clone(), ex.state.clone()))
        torch.cuda.synchronize()
        assert int(pool.counter) == 1004
        return rec

    rec = sequence()
    for j in range(1, 4):  # every replay advances the counter and the state
        assert not torch.equal(rec[j][1], rec[j - 1][1]) and not torch.equal(rec[j][0], rec[j - 1][0])
    one = choice == 1
    for j in (2, 3):
        assert bool((rec[j][1][one] == 0).all()) and torch.equal(rec[j][0][one], plain[one])
    assert not torch.equal(rec[1][0][one], plain[one]) and bool((rec[1][1][one] != 0).any())
    others = (choice == 0) | (choice == 2)
    assert not torch.equal(rec[3][0][others], plain[others])
    again = sequence()
    for (a, sa), (b, sb) in zip(rec, again):
        assert torch.equal(_bits(a), _bits(b)) and torch.equal(_bits(sa), _bits(sb))


@pytest.mark.gpu
def test_train_population_explores_per_member():
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    k, n, ticks = 2, 1024, 5
    env = hk.HockeyVecEnv(n, device="cuda:0", seed=6, p2="weak")
    cfgs = [td3.TD3Config(buffer_size=n // k * ticks, action_noise_scale=s) for s in (0.0, 0.3)]  # differing sigmas are fine with noise=
    pop = td3.FusedTD3Population(k, configs=cfgs, device="cuda:0", seeds=[3, 4])
    noise = hk.ExplorationNoise(n, slots=k, sigma=[0.0, 0.3], theta=[None, 0.15], dt=[1e-2, 0.05])
    td3.train_population(env, pop, ticks=ticks, warmup_ticks=ticks, noise=noise)  # no update: the actors stay as built
    assert int(pop.fused_pool.counter) == ticks
    buf, b = pop.replay_buffer, n // k
    for m in range(k):
        rows = slice(m * buf.capacity, m * buf.capacity + ticks * b)
        obs, act = buf.obs[rows].contiguous(), buf.action[rows]
        plain = pop.fused_pool(obs, torch.full((ticks * b,), m, dtype=torch.int32, device="cuda:0")).clone()
        if m == 0:
            assert torch.equal(act, plain)
        else:
            assert not torch.equal(act, plain) and float((act - plain).abs().max()) > 0.05
    assert bool((noise.state[:b] == 0).all()) and bool((noise.state[b:] != 0).any())
    env.close()


@pytest.mark.gpu
def test_train_and_collect_with_ou_noise():
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    n = 512
    env = hk.HockeyVecEnv(n, device="cuda:0", seed=2, p2="weak")
    buf = hk.DeviceReplayBuffer(n * 20, device="cuda:0", seed=1)
    actor = hk.load_td3_actor(NPZ, device="cuda:0", name="stage_3").train()
    learner = td3.DeviceTD3Learner(actor=actor, config=td3.TD3Config(batch_size=256), replay_buffer=buf, device="cuda:0")
    noise = hk.ExplorationNoise(n, sigma=0.2, theta=0.15)
    loss = td3.train(env, learner, ticks=12, warmup_ticks=8, fused=True, noise=noise)
    assert torch.isfinite(loss) and len(buf) == n * 12 and int(learner.fused_actor.counter) == 12
    assert bool((noise.state != 0).any()) and float(buf.action[:len(buf)].abs().max()) <= 1.0
    env.close()
    env = hk.HockeyVecEnv(n, device="cuda:0", seed=4, p2="weak")
    f = hk.FusedActor(_golden("cuda:0")[0], seed=1)
    buf = hk.DeviceReplayBuffer(n * 10, device="cuda:0")
    noise = hk.ExplorationNoise(n, sigma=0.3, clip=0.5, theta=0.15)
    hk.collect(env, f, buf, 10, noise=noise)
    assert len(buf) == n * 10 and int(f.counter) == 10
    a = buf.action[:n]
    assert not torch.equal(a, f(buf.obs[:n].contiguous()))
    env.close()


@pytest.mark.gpu
def test_loops_called_in_chunks_start_every_episode_from_zero_state():
    """One-tick calls of collect / train / train_population: an env whose episode ended on a call's last tick starts the
    next call with zero noise state (the loops zero those rows before returning), every other env keeps its state."""
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    n, calls = 512, 90  # TRAIN_SHOOTING episodes last at most 80 ticks: every env finishes at least one
    f = hk.FusedActor(_golden("cuda:0")[0], seed=1)
    learner = td3.DeviceTD3Learner(actor=hk.load_td3_actor(NPZ, device="cuda:0", name="stage_3").train(),
                                   replay_buffer=hk.DeviceReplayBuffer(n * calls, device="cuda:0"), device="cuda:0")
    pop = td3.FusedTD3Population(2, configs=td3.TD3Config(buffer_size=n // 2 * calls), device="cuda:0")
    loops = {
        "collect": (1, lambda env, nz, buf=hk.DeviceReplayBuffer(n * calls, device="cuda:0"): hk.collect(env, f, buf, 1, noise=nz)),
        "train": (1, lambda env, nz: td3.train(env, learner, ticks=1, warmup_ticks=8, fused=True, noise=nz)),
        "train_population": (2, lambda env, nz: td3.train_population(env, pop, ticks=1, warmup_ticks=8, noise=nz)),
    }
    for name, (slots, call) in loops.items():
        env = hk.HockeyVecEnv(n, mode=hk.Mode.TRAIN_SHOOTING, device="cuda:0", seed=7, p2="weak")
        noise = hk.ExplorationNoise(n, slots=slots, sigma=0.3, theta=0.15)
        ended = 0
        for _ in range(calls):
            before = noise.state.clone()
            call(env, noise)
            done = env.done.bool()
            ended += int(done.sum())
            assert bool((noise.state[done] == 0).all()), name
            assert bool((noise.state[~done] != before[~done]).any()), name
        assert ended >= n, (name, ended)
        env.close()
