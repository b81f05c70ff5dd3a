"""FusedTD3Population: K TD3 learners in one multi-cluster launch (hk_td3_update_population), the population replay buffer,
hk_actor_pack_many and td3.train_population.  The population launch is checked byte for byte against K single-member
hk_td3_update calls on the same local batches."""
import copy
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_td3_fused import HP_DISTINCT, _batch, _start_state  # noqa: E402  seeded batches and mid-training start states

A = 0x10000  # an aligned address: every invalid call below is rejected before anything is read through it


# ---- CPU ------------------------------------------------------------------------------------------------------------

def test_population_abi_error_convention_without_gpu():
    import ctypes as C
    import hockey_env_b200 as hk
    from hockey_env_b200 import _lib
    L = hk.load_library()
    INV = _lib.HK_E_INVALID
    k0 = 4

    def call(arenas=A, scratch=A, b=256, k=k0, losses=A, low=None, rng=None, seeds=True, do_actor=True, member=None, **kw):
        bt = _lib.TD3Batch(A, A, A, A, A, A, None, None, 0)
        hp = (_lib.TD3HParams * k0)(*[_lib.TD3HParams(0.99, 0.005, 0.005, 4e-4, 4e-4, 0.0, 0.0, 0.15, 0.2, 0.3)] * k0)
        lows, rngs = (C.c_void_p * k0)(*[A] * k0), (C.c_void_p * k0)(*[A] * k0)
        for key, v in kw.items():
            if key in dict(_lib.TD3Batch._fields_):
                setattr(bt, key, v)
            else:
                setattr(hp[member], key, v)
        if low is not None:
            lows[member] = low
        if rng is not None:
            rngs[member] = rng
        sd = (C.c_uint64 * k0)(*range(k0)) if seeds else None
        da = (C.c_uint8 * k0)(1, 0, 1, 0) if do_actor else None
        return L.hk_td3_update_population(arenas, scratch, C.byref(bt), b, k, hp, lows, rngs, sd, da, losses, 0, None)

    nan, inf = float("nan"), float("inf")
    cases = [(dict(arenas=None), b"NULL"), (dict(scratch=None), b"NULL"), (dict(losses=None), b"NULL"), (dict(seeds=False), b"NULL"),
             (dict(do_actor=False), b"NULL"), (dict(obs=None), b"NULL batch"), (dict(idx=None), b"NULL batch"),
             (dict(prio_weights=A), b"prio_idx"), (dict(arenas=A + 8), b"16-byte"), (dict(scratch=A + 4), b"16-byte"),
             (dict(idx=A + 4), b"8-byte"), (dict(prio_weights=A, prio_idx=A + 4, prio_n=5), b"8-byte"), (dict(reward=A + 2), b"4-byte"),
             (dict(k=0), b"k must be"), (dict(k=65), b"k must be"), (dict(b=0), b"batch"), (dict(b=1025), b"batch"),
             (dict(prio_weights=A, prio_idx=A, prio_n=0), b"prio_n"),
             (dict(member=2, low=0), b"member 2: NULL"), (dict(member=3, rng=A + 2), b"member 3: action_low / action_range need 4-byte")]
    for m, name in enumerate(("gamma", "tau_actor", "tau_critic", "lr_actor", "lr_critic", "wd_actor", "wd_critic", "beta",
                              "target_noise", "target_noise_clip")):
        for v in (-0.1, nan, inf):
            cases.append(({name: v, "member": m % k0}, f"member {m % k0}: {name} must be finite and >= 0".encode()))
    for kw, msg in cases:
        assert call(**kw) == INV, kw
        err = L.hk_last_error()
        assert b"hk_td3_update_population:" in err and msg in err, (kw, err)
    assert L.hk_td3_population_cluster_size(0, 0) == INV and b"k must be in [1, 64]" in L.hk_last_error()
    assert L.hk_td3_population_cluster_size(65, 0) == INV
    for args, msg in (((None, 862_784, 4, A), b"NULL"), ((A, 862_784, 4, None), b"NULL"), ((A, 862_784, 0, A), b"k must be"),
                      ((A, 862_784, 4097, A), b"k must be"), ((A, 71_683, 4, A), b"stride_floats"), ((A, 862_784, 4, A + 8), b"16-byte"),
                      ((A + 2, 862_784, 4, A), b"4-byte")):
        assert L.hk_actor_pack_many(*args, 0, None) == INV, args
        err = L.hk_last_error()
        assert b"hk_actor_pack_many:" in err and msg in err, (args, err)
    if not torch.cuda.is_available():
        assert call() == _lib.HK_E_NODEVICE and b"no CUDA device" in L.hk_last_error()
        assert call(k=1, b=1, prio_weights=A, prio_idx=A, prio_n=3) == _lib.HK_E_NODEVICE
        assert L.hk_td3_population_cluster_size(1, 0) == _lib.HK_E_NODEVICE
        assert L.hk_actor_pack_many(A, 71_684, 4096, A, 0, None) == _lib.HK_E_NODEVICE


def _cpu_buffer(k, cap, prio=False, seed=0):
    from hockey_env_b200.td3 import PopulationReplayBuffer
    return PopulationReplayBuffer(k, cap, device="cpu", seed=seed, prioritized=prio)


def _tagged(k, n, tick):
    """A batch of K * n transitions whose reward encodes (tick, member block, row in block)."""
    rows = torch.arange(k * n)
    rew = (tick * 10_000 + (rows // n) * 100 + rows % n).float()
    obs = rew.unsqueeze(1).repeat(1, 18)
    return obs, torch.zeros(k * n, 4) + rew.unsqueeze(1), rew, obs + 0.5, ((rows % n) % 3 == 0).to(torch.uint8)


def test_population_buffer_layout_and_wrap_around():
    k, n, cap = 3, 4, 10
    buf = _cpu_buffer(k, cap)
    for tick in range(4):  # 16 rows per member into rings of 10: ticks 2 and 3 wrap
        buf.push(*_tagged(k, n, tick))
    assert buf.pos == 16 % cap and buf.size == cap and len(buf) == cap
    for m in range(k):
        got = buf.reward[m * cap:(m + 1) * cap]
        want = torch.empty(cap)
        for tick in range(4):
            for j in range(n):
                want[(tick * n + j) % cap] = tick * 10_000 + m * 100 + j
        assert torch.equal(got, want), m
        assert torch.equal(buf.obs[m * cap:(m + 1) * cap], want.unsqueeze(1).repeat(1, 18))
        assert torch.equal(buf.next_obs[m * cap:(m + 1) * cap], want.unsqueeze(1).repeat(1, 18) + 0.5)
        assert torch.equal(buf.done[m * cap:(m + 1) * cap], ((want % 100) % 3 == 0).float())
    with pytest.raises(ValueError, match="equal blocks"):
        buf.push(*_tagged(1, 7, 0))
    with pytest.raises(ValueError, match="larger"):
        buf.push(*_tagged(k, cap + 1, 0))


@pytest.mark.parametrize("prio", [False, True])
def test_member_views_alias_the_member_rows(prio):
    from hockey_env_b200.td3 import DevicePrioritizedReplayBuffer
    from hockey_env_b200.training import DeviceReplayBuffer
    k, cap = 4, 16
    buf = _cpu_buffer(k, cap, prio)
    buf.push(*_tagged(k, 5, 0))
    for m in range(k):
        v = buf.member(m)
        assert type(v) is (DevicePrioritizedReplayBuffer if prio else DeviceReplayBuffer)
        assert (v.pos, v.size, v.capacity) == (buf.pos, buf.size, cap)
        arrays = ("obs", "action", "reward", "next_obs", "done") + (("weights",) if prio else ())
        for name in arrays:
            t, full = getattr(v, name), getattr(buf, name)
            assert t.data_ptr() == full[m * cap].data_ptr() and t.shape[0] == cap, (m, name)
        v.reward[2] = -7.0  # a write through the view lands in member m's rows of the population buffer
        assert float(buf.reward[m * cap + 2]) == -7.0
        idx = v.sample_indices(50)
        assert int(idx.min()) >= 0 and int(idx.max()) < buf.size
    with pytest.raises(IndexError):
        buf.member(k)


@pytest.mark.parametrize("prio", [False, True])
def test_indices_stay_inside_each_members_rows(prio):
    k, cap = 5, 40
    buf = _cpu_buffer(k, cap, prio, seed=3)
    buf.push(*_tagged(k, 25, 0))
    if prio:  # member m's weight mass all on its row m: a prioritized draw then picks exactly that row
        buf.weights.zero_()
        for m in range(k):
            buf.weights[m * cap + m] = 1e6  # the others are clamped to 1e-6 before the draw
    for b in (1, 64):
        idx = buf.sample_indices(b)
        assert idx.dtype == torch.int64 and tuple(idx.shape) == (k, min(b, 25))
        lo = torch.arange(k).unsqueeze(1) * cap
        assert bool(((idx >= lo) & (idx < lo + 25)).all())
        if prio:
            assert torch.equal(idx, (lo + torch.arange(k).unsqueeze(1)).expand_as(idx))


def test_prioritized_push_uses_each_members_own_max():
    k, cap, n = 3, 8, 3
    buf = _cpu_buffer(k, cap, prio=True)
    buf.push(*_tagged(k, n, 0))
    assert torch.equal(buf.weights, torch.full((k * cap,), 1e8))  # empty buffer: the init weight
    w = buf.weights.view(k, cap)
    w[:, :n] = torch.tensor([[0.5, 3.0, 1.0], [7.0, 0.1, 0.2], [0.3, 0.3, 0.4]])
    w[:, n:] = 99.0  # rows beyond the stored ones do not count
    buf.push(*_tagged(k, n, 1))
    assert torch.equal(w[:, n:2 * n], torch.tensor([3.0, 7.0, 0.4]).unsqueeze(1).expand(k, n))
    buf.push(*_tagged(k, n, 2))  # wraps: rows 6, 7, 0
    assert torch.equal(w[:, 6:8], torch.tensor([3.0, 7.0, 0.4]).unsqueeze(1).expand(k, 2))
    assert torch.equal(w[:, 0], torch.tensor([3.0, 7.0, 0.4]))


def test_population_rejects_mismatched_settings_and_uneven_env_split():
    from hockey_env_b200 import td3
    from hockey_env_b200.td3 import FusedTD3Population, TD3Config
    for field, a, b in (("batch_size", 256, 128), ("buffer_size", 1000, 2000), ("prioritized_replay", False, True)):
        with pytest.raises(ValueError, match=field):  # checked before anything touches a device
            FusedTD3Population(2, configs=[TD3Config(**{field: a}), TD3Config(**{field: b})])
    with pytest.raises(ValueError, match="k = 3"):
        FusedTD3Population(3, configs=[TD3Config()] * 2)
    with pytest.raises(ValueError, match="k must be"):
        FusedTD3Population(65)
    pop = SimpleNamespace(k=3, configs=[TD3Config()] * 3)
    with pytest.raises(ValueError, match="equal blocks"):
        td3.train_population(SimpleNamespace(num_envs=10), pop, ticks=1)
    pop = SimpleNamespace(k=2, configs=[TD3Config(action_noise_scale=0.2), TD3Config(action_noise_scale=0.3)])
    with pytest.raises(ValueError, match="action_noise_scale"):
        td3.train_population(SimpleNamespace(num_envs=10), pop, ticks=1)


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _member_cfg(m, prio, **kw):
    """Member m's TD3Config: every one of the ten hyper-parameters moved off HP_DISTINCT by a member-dependent factor,
    policy_update_freq 1, 2 or 3 (so one launch mixes critic-only and actor steps)."""
    from hockey_env_b200.td3 import TD3Config
    f = 1.0 + 0.1 * m
    hp = {key: v * f for key, v in HP_DISTINCT.items()}
    hp["gamma"] = 0.99 - 0.005 * m
    return TD3Config(**{"policy_update_freq": 1 + m % 3, "prioritized_replay": prio, "batch_size": 256, "buffer_size": 300, **hp, **kw})


def _population(k, prio, seed=0, seeds=None, cap=300, configs=None):
    """A population in distinct mid-training start states (Adam moments, step counts, noise counters near 2^32, distinct
    action bounds per member), with a full, seeded buffer of `cap` rows per member."""
    from hockey_env_b200.actor import ActorNetwork
    from hockey_env_b200.td3 import FusedTD3Population, PopulationReplayBuffer, TwinQNetwork
    buf = PopulationReplayBuffer(k, cap, device="cuda:0", seed=seed + 1, prioritized=prio)
    buf.push(*_batch(k * cap, seed=seed + 2, device="cuda:0"))
    if prio:
        buf.weights.copy_(torch.rand(k * cap, generator=torch.Generator().manual_seed(seed + 3)).cuda() + 0.05)
    states = []
    for m in range(k):
        bounds = ([-2.0 + 0.1 * m, -1.0, -0.5, -3.0], [4.0, 2.0 + 0.2 * m, 1.0, 6.0]) if m % 2 else None
        states.append(_start_state(seed + 100 + m, bounds=bounds, counters=(999 + m, 333 + m, 2**32 - 1 - (m % 3))))
    actors, critics = [], []
    for nets, _ in states:
        a, c = ActorNetwork(), TwinQNetwork()
        a.load_state_dict(nets["policy"])
        c.load_state_dict(nets["critic"])
        actors.append(a)
        critics.append(c)
    pop = FusedTD3Population(k, configs=configs or [_member_cfg(m, prio) for m in range(k)], actors=actors, critics=critics,
                             seeds=seeds or [(m << 40) + 17 * m + seed for m in range(k)], replay_buffer=buf, device="cuda:0")
    for mem, (nets, adam) in zip(pop.members, states):
        mem.target_actor.load_state_dict(nets["target_policy"])
        mem.target_critic.load_state_dict(nets["target_critic"])
        for key in ("m_actor", "v_actor", "m_critic", "v_critic"):
            mem.blocks[key].copy_(adam[key])
        mem.counters.copy_(torch.tensor(adam["t"], dtype=torch.int64))
    return pop


def _oracle_update(pop, idx):
    """Member m's update as one hk_td3_update on pop.replay_buffer.member(m)'s views with idx[m]'s local rows."""
    buf = pop.replay_buffer
    out = []
    for m, mem in enumerate(pop.members):
        v = buf.member(m)
        local = (idx[m] - m * buf.capacity).contiguous()
        prio = (v.weights, local, v.size) if buf.prioritized else None
        out.append(mem._launch((v.obs, v.action, v.reward, v.next_obs, v.done), local, prio))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 8, 17])
@pytest.mark.parametrize("prio", [False, True])
def test_population_launch_equals_single_member_oracle(k, prio):
    """Three population updates against 3 x K hk_td3_update calls from the same start state, byte for byte: arenas
    (weights, targets, Adam moments, step counts, noise counters crossing 2^32), losses, importance weights and the
    buffer's priorities.  300 draws of 256 rows per member: duplicate indices in every prioritized batch."""
    pops = [_population(k, prio, seed=7), _population(k, prio, seed=7)]
    assert torch.equal(pops[0].arenas, pops[1].arenas)
    gen = torch.Generator(device="cuda:0").manual_seed(5)
    for step in range(3):
        b = 256 if step < 2 else 37
        idx = pops[0].replay_buffer.sample_indices(b) if prio else \
            torch.randint(0, 300, (k, b), device="cuda:0", generator=gen) + pops[0].replay_buffer.offsets
        assert prio is False or any(len(set(r.tolist())) < b for r in idx)
        al, cl = pops[0].update(idx)
        want = _oracle_update(pops[1], idx)
        torch.cuda.synchronize()
        for m in range(k):
            assert pops[0].last_do_actor[m] == (want[m][0] is not None), (step, m)
            assert torch.equal(pops[0].arenas[m], pops[1].arenas[m]), (step, m)
            assert cl[m].view(1).view(torch.int32).item() == want[m][1].view(1).view(torch.int32).item(), (step, m)
            if want[m][0] is None:
                assert torch.isnan(al[m]), (step, m)
            else:
                assert al[m].view(1).view(torch.int32).item() == want[m][0].view(1).view(torch.int32).item(), (step, m)
            assert torch.equal(pops[0].last_importance_weights()[m], pops[1].members[m].last_importance_weights()), (step, m)
        if prio:
            assert torch.equal(pops[0].replay_buffer.weights, pops[1].replay_buffer.weights), step
    acts = [sum(1 for s in range(1, 4) if s % (1 + m % 3) == 0) for m in range(k)]
    for m, mem in enumerate(pops[0].members):
        assert [int(v) for v in mem.counters.cpu()] == [999 + m + 3, 333 + m + acts[m], 2**32 - 1 - (m % 3) + 3]
    if k > 1:
        assert not torch.equal(pops[0].arenas[0], pops[0].arenas[1])


def _cluster_run(path):
    """Three prioritized population updates (K = 3; batches 1024, 1024 and 37); saves arenas, priorities, losses and the
    cluster size the launches used."""
    import hockey_env_b200 as hk
    pop = _population(3, True, seed=41, cap=1100, configs=[_member_cfg(m, True, buffer_size=1100) for m in range(3)])
    losses = []
    for b in (1024, 1024, 37):
        al, cl = pop.update_from_buffer(b)
        losses += [al, cl]
    torch.cuda.synchronize()
    np.savez(path, arenas=pop.arenas.cpu().numpy(), weights=pop.replay_buffer.weights.cpu().numpy(),
             losses=torch.stack(losses).cpu().numpy(), cluster=int(hk.load_library().hk_td3_population_cluster_size(3, 0)))


@pytest.mark.gpu
def test_population_results_do_not_depend_on_the_cluster_size(tmp_path):
    """The same population run at its default cluster size and at 8, 4 and 1 (HK_TD3_CLUSTER, one process each) leaves
    byte-identical arenas, priorities and losses."""
    import hockey_env_b200 as hk
    from hockey_env_b200 import _lib
    L = hk.load_library()
    sizes = [L.hk_td3_population_cluster_size(k, 0) for k in range(1, 65)]
    assert set(sizes) <= {16, 8} and sizes[0] == 16 == L.hk_td3_cluster_size(0)
    assert L.hk_td3_population_cluster_size(3, -1) == _lib.HK_E_INVALID
    _cluster_run(tmp_path / "default.npz")
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([here, os.path.dirname(here)]))
    want = np.load(tmp_path / "default.npz")
    runs = [16, 8, 4, 1] if int(want["cluster"]) == 8 else [8, 4, 1]
    for n in runs:
        r = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) +
                           ["-c", "import sys, test_td3_population as t; t._cluster_run(sys.argv[1])", str(tmp_path / f"{n}.npz")],
                           env=dict(env, HK_TD3_CLUSTER=str(n)), cwd=here, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (n, r.stderr[-3000:])
    seen = {int(want["cluster"])}
    for n in runs:
        got = np.load(tmp_path / f"{n}.npz")
        assert int(got["cluster"]) == min(n, int(want["cluster"]))
        seen.add(int(got["cluster"]))
        for key in ("arenas", "weights", "losses"):
            assert got[key].tobytes() == want[key].tobytes(), (n, key)
    assert seen >= {8, 4, 1}


@pytest.mark.gpu
def test_population_determinism_graph_replay_and_no_sync():
    runs = []
    for _ in range(2):
        pop = _population(4, True, seed=61)
        for _ in range(6):
            pop.update_from_buffer()
        torch.cuda.synchronize()
        runs.append((pop.arenas.clone(), pop.replay_buffer.weights.clone()))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])

    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        pop.update_from_buffer()
    finally:
        torch.cuda.set_sync_debug_mode("default")

    cfgs = [_member_cfg(m, False, policy_update_freq=1) for m in range(4)]  # a captured launch fixes each member's actor step
    eager, graphed = (_population(4, False, seed=62, configs=copy.deepcopy(cfgs)) for _ in range(2))
    buf = eager.replay_buffer
    static = buf.sample_indices(256)
    for p in (eager, graphed):  # warm-up outside the capture: scratch allocation, first-launch set-up
        p.update(static)
    draws = [buf.sample_indices(256) for _ in range(6)]
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            graphed.update(static)
    torch.cuda.current_stream().wait_stream(s)
    for d in draws:
        static.copy_(d)
        graph.replay()
        eager.update(d)
        torch.cuda.synchronize()
        assert torch.equal(eager.arenas, graphed.arenas)


@pytest.mark.gpu
def test_actor_pack_many_equals_host_pack_and_leaves_other_slots():
    from hockey_env_b200.actor import FusedActor, FusedActorPool
    pop = _population(5, False, seed=71)
    for _ in range(3):
        pop.update_from_buffer()  # actors that moved from their start weights
    spare = [m.actor for m in pop.members] + [pop.members[0].target_actor, pop.members[1].target_actor]
    pool = FusedActorPool(spare, device="cuda:0")
    noise = torch.randint(0, 256, tuple(pool.table.shape), dtype=torch.uint8, generator=torch.Generator().manual_seed(3)).cuda()
    pool.table.copy_(noise)
    pop.refresh_pool(pool)
    torch.cuda.synchronize()
    for m, mem in enumerate(pop.members):
        sd = {key: v.detach().cpu() for key, v in mem.actor.state_dict().items()}
        assert torch.equal(pool.table[m].cpu(), FusedActor.pack(sd)), m
    assert torch.equal(pool.table[5:], noise[5:])
    with pytest.raises(ValueError, match="slots"):
        pop.refresh_pool(FusedActorPool(spare[:4], device="cuda:0"))


@pytest.mark.gpu
def test_train_population_blocks_act_through_their_member():
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    from hockey_env_b200.actor import FusedActor
    k, n = 4, 256
    env = hk.HockeyVecEnv(k * n, device="cuda:0", seed=3, p2="weak")
    cfgs = [td3.TD3Config(buffer_size=512, lr_pol=1e-3 * (m + 1)) for m in range(k)]
    pop = td3.FusedTD3Population(k, configs=cfgs, device="cuda:0", seeds=[11, 12, 13, 14])
    obs = env.obs.clone()
    td3.train_population(env, pop, ticks=1, warmup_ticks=8)  # warm-up only: no update, one noisy pooled launch
    assert pop.fused_pool.seed == 11 and int(pop.fused_pool.counter) == 1
    buf = pop.replay_buffer
    for m, mem in enumerate(pop.members):
        fa = FusedActor(mem.actor, device="cuda:0", seed=pop.fused_pool.seed)
        want = fa(obs[m * n:(m + 1) * n].contiguous(), noise=0.2, row0=m * n)
        got = buf.action[m * buf.capacity:m * buf.capacity + n]
        assert torch.equal(got, want), m
        assert torch.equal(buf.obs[m * buf.capacity:m * buf.capacity + n], obs[m * n:(m + 1) * n])
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("prio", [False, True])
def test_train_population_short_run(prio):
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    k, n = 4, 2048
    env = hk.HockeyVecEnv(n, device="cuda:0", seed=5, p2="weak")
    cfgs = [td3.TD3Config(prioritized_replay=prio, buffer_size=n // k * 20, policy_update_freq=1 + m % 2, lr_q=4e-4 * (1 + m))
            for m in range(k)]
    pop = td3.FusedTD3Population(k, configs=cfgs, device="cuda:0")
    before = pop.arenas.clone()
    ticks, upt, warm = 20, 2, 8
    loss = td3.train_population(env, pop, ticks=ticks, updates_per_tick=upt, warmup_ticks=warm)
    torch.cuda.synchronize()
    updates = upt * (ticks - warm)
    assert tuple(loss.shape) == (k,) and bool(torch.isfinite(loss).all())
    assert len(pop.replay_buffer) == n // k * ticks and env.stats()["env_steps"] == n * ticks
    blocks, ctr, _ = pop.members[0].arena_layout()
    for m, mem in enumerate(pop.members):
        assert [int(v) for v in mem.counters.cpu()] == [updates, updates // (1 + m % 2), updates]
        o, cnt = blocks["actor"]
        assert not torch.equal(pop.arenas[m].view(torch.float32)[o:o + cnt], before[m].view(torch.float32)[o:o + cnt]), m
        assert bool(torch.isfinite(pop.arenas[m].view(torch.float32)[:ctr]).all())
    if prio:
        assert bool((pop.replay_buffer.weights < 1e8).any())
    env.close()


@pytest.mark.gpu
def test_copy_member_makes_arenas_equal_and_seeds_decide_the_rest():
    from hockey_env_b200 import td3
    k, cap = 3, 300
    cfgs = [td3.TD3Config(buffer_size=cap, policy_update_freq=1)] * k
    pop = td3.FusedTD3Population(k, configs=[copy.copy(c) for c in cfgs], seeds=[5, 5, 6], device="cuda:0")
    one = _batch(cap, seed=9, device="cuda:0")
    pop.replay_buffer.push(*[torch.cat([t] * k) for t in one])  # every member holds the same rows
    pop.update_from_buffer()
    assert not torch.equal(pop.arenas[0], pop.arenas[1])  # different start weights
    pop.copy_member(1, 0)
    pop.copy_member(2, 0)
    assert torch.equal(pop.arenas[1], pop.arenas[0]) and torch.equal(pop.arenas[2], pop.arenas[0])
    assert pop.members[1].train_step == pop.members[0].train_step
    local = torch.randint(0, cap, (1, 256), device="cuda:0").expand(k, 256)
    pop.update((local + pop.replay_buffer.offsets).contiguous())
    torch.cuda.synchronize()
    assert torch.equal(pop.arenas[1], pop.arenas[0])      # same arena, rows and seed: the same update
    assert not torch.equal(pop.arenas[2], pop.arenas[0])  # only the target-noise seed differs
