"""FusedTD3Learner: one TD3 update in one sm_100a launch (csrc/hk_td3.cuh, hk_td3_update), against torch learners in
float32 and float64 built from the same weights, batch indices and target noise."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_actor_train import philox, uniforms  # noqa: E402  the host restatement of hk::philox and the uniform mapping

STREAM_TD3_TARGET = 5
A = 0x10000  # an aligned address: every invalid call below is rejected before anything is read through it


def td3_noise_key(counter):
    """Philox counter words 2 and 3 of the target noise of the update with noise counter `counter`."""
    return counter & 0xFFFFFFFF, STREAM_TD3_TARGET | (((counter >> 32) & 0xFFFFFF) << 8)


def td3_normals(seed, batch, counter):
    """float64 [batch, 4]: the target-policy noise normals of rows 0 .. batch - 1."""
    c2, c3 = td3_noise_key(counter)
    x, y, z, w = philox(seed, np.arange(batch, dtype=np.uint64), c2, c3)
    out = []
    for a, b in ((x, y), (z, w)):
        u1, u2 = uniforms(a, b)
        r = np.sqrt(-2.0 * np.log(u1))
        out += [r * np.cos(2 * np.pi * u2), r * np.sin(2 * np.pi * u2)]
    return np.stack(out, 1)


def _p64(n):
    return (n + 63) // 64 * 64


def scratch_floats(b):
    bh = b * 256
    return (4 * _p64(b) + 3 * _p64(2 * b) + _p64(b) + 2 * _p64(20 * b) + 3 * _p64(24 * b) + 2 * _p64(bh) + 6 * _p64(2 * bh)
            + 2 * _p64(bh) + _p64(4 * b) + 4 * _p64(bh) + _p64(4 * b) + 2 * _p64(bh) + _p64(71684) + _p64(143874))


def _batch(n, seed=0, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    out = (torch.randn(n, 18, generator=g), torch.rand(n, 4, generator=g) * 2 - 1, torch.randn(n, generator=g),
           torch.randn(n, 18, generator=g), (torch.rand(n, generator=g) < 0.1).float())
    return tuple(t.to(device) for t in out)


# ---- CPU ------------------------------------------------------------------------------------------------------------

def test_target_noise_key_and_known_answers():
    assert td3_noise_key(0) == (0, 5)
    assert td3_noise_key((3 << 32) | 11) == (11, 5 | (3 << 8))
    got = philox(0, [0], 0, 0)  # Random123 known answers (also checked in test_actor_train)
    assert [int(v[0]) for v in got] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    z = td3_normals(7, 50_000, 3)
    assert np.isfinite(z).all() and abs(z.mean()) < 0.02 and abs(z.std() - 1) < 0.02
    assert not np.array_equal(td3_normals(7, 10, 4), z[:10])  # the counter changes the draw
    assert np.array_equal(td3_normals(7, 10, 3), z[:10])      # a row's noise depends on its index, not on the batch size


def test_arena_and_scratch_sizes():
    import hockey_env_b200 as hk
    from hockey_env_b200.td3 import FusedTD3Learner
    L = hk.load_library()
    blocks, ctr, nbytes = FusedTD3Learner.arena_layout()
    assert int(L.hk_td3_arena_bytes()) == nbytes == 4 * (862_720 + 64)
    want = {"actor": 0, "critic": 71_744, "target_actor": 215_680, "target_critic": 287_424, "m_actor": 431_360,
            "v_actor": 503_104, "m_critic": 574_848, "v_critic": 718_784}  # include/hockey_b200.h
    assert {k: o for k, (o, _) in blocks.items()} == want and ctr == 862_720
    assert all(o % 64 == 0 for o, _ in blocks.values())
    for b in (1, 2, 37, 256, 1000, 1024):
        assert int(L.hk_td3_scratch_bytes(b)) == 4 * scratch_floats(b)


def test_arena_layout_is_state_dict_order():
    from hockey_env_b200.actor import ActorNetwork
    from hockey_env_b200.td3 import FusedTD3Learner, TwinQNetwork
    blocks, _, _ = FusedTD3Learner.arena_layout()
    for name, net in (("actor", ActorNetwork()), ("critic", TwinQNetwork())):
        params = dict(net.named_parameters())
        keys = [k for k in net.state_dict() if k in params]  # state_dict order; the critic's action buffers are not params
        assert keys == list(params)
        assert sum(p.numel() for p in params.values()) == blocks[name][1]
    sd = TwinQNetwork().state_dict()
    assert [k for k in sd if not k.startswith("action")] == [f"{h}.fc{i}.{w}" for h in ("q1", "q2") for i in (1, 2, 3)
                                                             for w in ("weight", "bias")]
    assert tuple(sd["q1.fc1.weight"].shape) == (256, 22) and tuple(ActorNetwork().state_dict()["fc1.weight"].shape) == (256, 18)


def test_abi_error_convention_without_gpu():
    import ctypes as C
    import hockey_env_b200 as hk
    from hockey_env_b200 import _lib
    L = hk.load_library()
    INV = _lib.HK_E_INVALID
    assert L.hk_td3_scratch_bytes(0) == INV and b"hk_td3_scratch_bytes:" in L.hk_last_error()
    assert L.hk_td3_scratch_bytes(1025) == INV

    def call(arena=A, scratch=A, batch=None, b=256, hp=None, low=A, rng=A, losses=A, **kw):
        bt = _lib.TD3Batch(A, A, A, A, A, A, None, None, 0)
        h = _lib.TD3HParams(0.99, 0.005, 0.005, 4e-4, 4e-4, 0.0, 0.0, 0.15, 0.2, 0.3)
        for k, v in kw.items():
            setattr(bt if k in dict(_lib.TD3Batch._fields_) else h, k, v)
        return L.hk_td3_update(arena, scratch, C.byref(bt) if batch is None else batch, b, C.byref(h) if hp is None else hp,
                               low, rng, 1, 1, losses, 0, None)

    nan, inf = float("nan"), float("inf")
    cases = [(dict(arena=None), b"NULL"), (dict(scratch=None), b"NULL"), (dict(low=None), b"NULL"), (dict(rng=None), b"NULL"),
             (dict(losses=None), b"NULL"), (dict(obs=None), b"NULL"), (dict(idx=None), b"NULL"), (dict(done=None), b"NULL"),
             (dict(prio_weights=A), b"prio_idx"), (dict(arena=A + 8), b"16-byte"), (dict(scratch=A + 4), b"16-byte"),
             (dict(idx=A + 4), b"8-byte"), (dict(obs=A + 2), b"4-byte"), (dict(b=0), b"batch"), (dict(b=1025), b"batch"),
             (dict(prio_weights=A, prio_idx=A, prio_n=0), b"prio_n")]
    for name in ("gamma", "tau_actor", "tau_critic", "lr_actor", "lr_critic", "wd_actor", "wd_critic", "beta", "target_noise",
                 "target_noise_clip"):
        cases += [({name: -0.1}, name.encode()), ({name: nan}, name.encode()), ({name: inf}, name.encode())]
    for kw, msg in cases:
        assert call(**kw) == INV, kw
        err = L.hk_last_error()
        assert b"hk_td3_update:" in err and msg in err, (kw, err)
    assert L.hk_td3_update(A, A, None, 256, None, A, A, 1, 1, A, 0, None) == INV
    if not torch.cuda.is_available():
        assert call() == _lib.HK_E_NODEVICE and b"no CUDA device" in L.hk_last_error()
        assert call(prio_weights=A, prio_idx=A, prio_n=5, b=1, target_noise=0.0) == _lib.HK_E_NODEVICE


def test_fused_learner_needs_cuda_and_the_reference_architecture():
    import hockey_env_b200 as hk
    from hockey_env_b200.actor import ActorNetwork
    from hockey_env_b200.td3 import FusedTD3Learner
    with pytest.raises(hk.HockeyLibraryError, match="CUDA"):
        FusedTD3Learner(device="cpu")
    if torch.cuda.is_available():
        with pytest.raises(ValueError, match="reference architecture"):
            FusedTD3Learner(actor=ActorNetwork(hidden=128))


@pytest.mark.parametrize("prio", [False, True])
def test_sample_indices_gather_equals_sample(prio):
    from hockey_env_b200.td3 import DevicePrioritizedReplayBuffer
    from hockey_env_b200.training import DeviceReplayBuffer
    Buf = DevicePrioritizedReplayBuffer if prio else DeviceReplayBuffer
    bufs = [Buf(500, device="cpu", seed=4) for _ in range(2)]
    for k in range(3):
        for b in bufs:
            b.push(*_batch(200, seed=k))
    if prio:
        for b in bufs:
            b.weights[:] = torch.rand(500, generator=torch.Generator().manual_seed(1)) + 0.01
    for _ in range(3):
        want = bufs[0].sample(64)
        idx = bufs[1].sample_indices(64)
        got = (bufs[1].obs[idx], bufs[1].action[idx], bufs[1].reward[idx], bufs[1].next_obs[idx], bufs[1].done[idx])
        assert all(torch.equal(x, y) for x, y in zip(want, got))
        if prio:
            assert torch.equal(bufs[0].last_batch_inds, bufs[1].last_batch_inds)


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _learner_pair(cfg, seed=0, buf=None):
    """A FusedTD3Learner and its start state (a CPU state dict) from seeded random networks."""
    from hockey_env_b200.actor import ActorNetwork
    from hockey_env_b200.td3 import FusedTD3Learner, TwinQNetwork
    torch.manual_seed(seed)
    actor, critic = ActorNetwork(), TwinQNetwork()
    L = FusedTD3Learner(actor=actor, critic=critic, config=cfg, replay_buffer=buf, device="cuda:0", seed=seed + 11)
    with torch.no_grad():  # targets that differ from the online nets, so Polyak is visible
        for p in list(L.target_actor.parameters()) + list(L.target_critic.parameters()):
            p.add_(0.01 * torch.randn_like(p))
    return L, {k: {n: t.detach().cpu().clone() for n, t in v.items()} for k, v in L.state_dict().items()}


def _reference(state, batch, z, cfg, dtype, do_actor, weights=None):
    """DeviceTD3Learner.update written out for `dtype` with the target noise z given: returns the nets, the Adam
    moments, the losses and the priorities."""
    from hockey_env_b200.actor import ActorNetwork
    from hockey_env_b200.td3 import TwinQNetwork, huber_weighted
    dev = "cuda:0"
    nets = {"policy": ActorNetwork(), "critic": TwinQNetwork(), "target_policy": ActorNetwork(), "target_critic": TwinQNetwork()}
    for k, n in nets.items():
        n.load_state_dict(state[k])
        n.to(dev, dtype)
    actor, critic, ta, tc = nets["policy"], nets["critic"], nets["target_policy"], nets["target_critic"]
    aopt = torch.optim.Adam(actor.parameters(), lr=cfg.lr_pol, weight_decay=cfg.wd_pol)
    copt = torch.optim.Adam(critic.parameters(), lr=cfg.lr_q, weight_decay=cfg.wd_q)
    s, a, r, s2, d = (t.to(dev, dtype) for t in batch)
    w = None if weights is None else weights.to(dev, dtype)
    with torch.no_grad():
        a2 = ta(s2)
        noise = (z.to(dev, dtype) * cfg.target_action_noise_scale).clamp(-cfg.target_action_noise_clip, cfg.target_action_noise_clip)
        q1t, q2t = tc(s2, (a2 + noise).clamp(-1.0, 1.0))
        y = r + cfg.gamma * (1 - d) * torch.minimum(q1t, q2t)
    q1, q2 = critic(s, a)
    closs = 0.5 * (huber_weighted(q1, y, w) + huber_weighted(q2, y, w))
    closs.backward()
    copt.step()
    prio = (0.5 * ((q1 - y).abs() + (q2 - y).abs())).detach().clamp(1e-6, 1e6)
    aloss = None
    if do_actor:
        q, _ = critic(s, actor(s))
        aloss = -q.mean()
        aloss.backward()
        aopt.step()
        with torch.no_grad():
            for net, tgt, tau in ((actor, ta, cfg.tau_actor), (critic, tc, cfg.tau_critic)):
                for tp, p in zip(tgt.parameters(), net.parameters()):
                    tp.mul_(1 - tau).add_(p, alpha=tau)
    flat = lambda ps: torch.cat([p.detach().reshape(-1) for p in ps])  # noqa: E731
    mom = lambda opt, net, k: torch.cat([opt.state[p][k].reshape(-1) if p in opt.state else torch.zeros_like(p).reshape(-1)  # noqa: E731
                                         for p in net.parameters()])
    return {"actor": flat(actor.parameters()), "critic": flat(critic.parameters()), "target_actor": flat(ta.parameters()),
            "target_critic": flat(tc.parameters()), "m_actor": mom(aopt, actor, "exp_avg"), "v_actor": mom(aopt, actor, "exp_avg_sq"),
            "m_critic": mom(copt, critic, "exp_avg"), "v_critic": mom(copt, critic, "exp_avg_sq"),
            "closs": closs.detach().reshape(1), "aloss": None if aloss is None else aloss.detach().reshape(1), "prio": prio}


def _check_against_float64(L, got_losses, ref32, ref64, lr):
    for name in ("m_actor", "v_actor", "m_critic", "v_critic", "target_actor", "target_critic"):
        e_f = float((L.blocks[name].double() - ref64[name]).abs().max())
        e_t = float((ref32[name].double() - ref64[name]).abs().max())
        assert e_f <= 4 * e_t + 1e-7, (name, e_f, e_t)
    for name, got in (("closs", got_losses[1]), ("aloss", got_losses[0])):
        if ref64[name] is None:
            assert got is None
            continue
        e_f = float((got.double() - ref64[name]).abs().max())
        e_t = float((ref32[name].double() - ref64[name]).abs().max())
        assert e_f <= 4 * e_t + 1e-7, (name, e_f, e_t)
    for name in ("actor", "critic"):
        err = (L.blocks[name].double() - ref64[name]).abs()
        assert float((err <= 1e-6).double().mean()) >= 0.999, (name, float((err <= 1e-6).double().mean()))
        assert float(err.max()) <= 2 * lr, (name, float(err.max()))


@pytest.mark.gpu
@pytest.mark.parametrize("b", [1, 37, 256, 1024])
@pytest.mark.parametrize("actor_step", [False, True])
@pytest.mark.parametrize("wd", [0.0, 1e-2])
def test_one_update_against_float64(b, actor_step, wd):
    from hockey_env_b200.td3 import TD3Config
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = TD3Config(policy_update_freq=1 if actor_step else 2, wd_q=wd, wd_pol=wd)
    L, state = _learner_pair(cfg, seed=b)
    batch = _batch(b, seed=b + 1, device="cuda:0")
    z = torch.from_numpy(td3_normals(L.seed, b, 0))
    losses = L.update(*batch)
    torch.cuda.synchronize()
    assert int(L.counters[0]) == 1 and int(L.counters[1]) == int(actor_step) and int(L.counters[2]) == 1
    ref64 = _reference(state, batch, z, cfg, torch.float64, actor_step)
    ref32 = _reference(state, batch, z.float(), cfg, torch.float32, actor_step)
    _check_against_float64(L, losses, ref32, ref64, cfg.lr_q)


@pytest.mark.gpu
def test_policy_update_freq_and_polyak():
    from hockey_env_b200.td3 import TD3Config
    cfg = TD3Config(policy_update_freq=3)
    L, _ = _learner_pair(cfg, seed=5)
    batch = _batch(256, seed=6, device="cuda:0")
    for step in range(1, 7):
        before = {k: L.blocks[k].clone() for k in ("actor", "critic", "target_actor", "target_critic")}
        al, cl = L.update(*batch)
        assert torch.isfinite(cl)
        assert not torch.equal(L.blocks["critic"], before["critic"])
        if step % 3:
            assert al is None
            for k in ("actor", "target_actor", "target_critic"):
                assert torch.equal(L.blocks[k], before[k]), (step, k)
        else:
            assert al is not None and torch.isfinite(al) and not torch.equal(L.blocks["actor"], before["actor"])
            for k, tau in (("actor", cfg.tau_actor), ("critic", cfg.tau_critic)):
                want = before["target_" + k] * (1 - tau) + tau * L.blocks[k]
                assert torch.allclose(L.blocks["target_" + k], want, rtol=0, atol=1e-7), (step, k)
    assert [int(v) for v in L.counters.cpu()] == [6, 2, 6] and L.train_step == 6


def _filled_prio_buffer(size, seed):
    from hockey_env_b200.td3 import DevicePrioritizedReplayBuffer
    buf = DevicePrioritizedReplayBuffer(size, device="cuda:0", seed=seed)
    buf.push(*_batch(size, seed=seed, device="cuda:0"))
    buf.weights.copy_(torch.rand(size, generator=torch.Generator().manual_seed(seed)).cuda() + 0.05)
    return buf


@pytest.mark.gpu
def test_prioritized_weights_priorities_and_no_sync():
    from hockey_env_b200.td3 import DeviceTD3Learner, TD3Config
    cfg = TD3Config(prioritized_replay=True, policy_update_freq=1)
    buf = _filled_prio_buffer(40, seed=3)  # 40 draws with replacement from 40 rows: many duplicate indices
    L, state = _learner_pair(cfg, seed=8, buf=buf)
    gstate = buf.gen.get_state()
    idx = buf.sample_indices(256)  # capped at the 40 stored rows, like sample()
    b = idx.shape[0]
    ref_w = DeviceTD3Learner.importance_weights(L)  # the torch formula on the same indices (host sync: outside the check)
    batch = (buf.obs[idx], buf.action[idx], buf.reward[idx], buf.next_obs[idx], buf.done[idx])
    weights_before = buf.weights.clone()
    buf.gen.set_state(gstate)
    buf.last_batch_inds = None
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        al, cl = L.update_from_buffer(256)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert buf.last_batch_inds is None
    assert torch.allclose(L.last_importance_weights(), ref_w, rtol=1e-5, atol=0)
    assert b == 40 and torch.isfinite(cl) and torch.isfinite(al)
    z = torch.from_numpy(td3_normals(L.seed, b, 0))
    ref = _reference(state, batch, z, cfg, torch.float64, True, weights=ref_w.double())
    idx_c, prio = idx.cpu().numpy(), ref["prio"].float()
    last = {int(ix): r for r, ix in enumerate(idx_c)}
    first = {}
    for r, ix in enumerate(idx_c):
        first.setdefault(int(ix), r)
    spread = 0.0
    for ix, r in last.items():
        assert torch.allclose(buf.weights[ix], prio[r], rtol=1e-4, atol=1e-6), (ix, float(buf.weights[ix]), float(prio[r]))
        spread = max(spread, float((prio[first[ix]] - prio[r]).abs() / prio[r]))
    assert spread > 1e-2  # occurrences of one index differ (target noise is per row): last-wins is what was checked
    untouched = torch.ones(40, dtype=torch.bool)
    untouched[list(last)] = False
    assert torch.equal(buf.weights[untouched.cuda()], weights_before[untouched.cuda()])


@pytest.mark.gpu
def test_bit_identical_run_to_run():
    from hockey_env_b200.td3 import TD3Config
    arenas = []
    for _ in range(2):
        buf = _filled_prio_buffer(5000, seed=1)
        L, _ = _learner_pair(TD3Config(prioritized_replay=True), seed=2, buf=buf)
        for _ in range(50):
            L.update_from_buffer(256)
        torch.cuda.synchronize()
        arenas.append((L.arena.clone(), buf.weights.clone()))
    assert torch.equal(arenas[0][0], arenas[1][0]) and torch.equal(arenas[0][1], arenas[1][1])


@pytest.mark.gpu
def test_graph_replay_equals_eager():
    from hockey_env_b200.training import DeviceReplayBuffer
    from hockey_env_b200.td3 import TD3Config
    cfg = TD3Config()
    buf = DeviceReplayBuffer(4096, device="cuda:0", seed=3)
    buf.push(*_batch(4096, seed=4, device="cuda:0"))  # full
    eager, _ = _learner_pair(cfg, seed=9)
    graphed, _ = _learner_pair(cfg, seed=9)
    draws = [[buf.sample_indices(256) for _ in range(cfg.policy_update_freq)] for _ in range(4)]
    static = [tuple(t.clone() for t in (buf.obs[i], buf.action[i], buf.reward[i], buf.next_obs[i], buf.done[i])) for i in draws[0]]
    for i in draws[0]:  # warm-up (first-call set-up outside the capture), same updates on both
        for L in (eager, graphed):
            L.update(buf.obs[i], buf.action[i], buf.reward[i], buf.next_obs[i], buf.done[i])
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            outs = [graphed.update(*st) for st in static]
    torch.cuda.current_stream().wait_stream(s)
    for rnd in range(1, 4):
        for st, i in zip(static, draws[rnd]):
            for dst, src in zip(st, (buf.obs[i], buf.action[i], buf.reward[i], buf.next_obs[i], buf.done[i])):
                dst.copy_(src)
            eager.update(buf.obs[i], buf.action[i], buf.reward[i], buf.next_obs[i], buf.done[i])
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(eager.arena, graphed.arena), rnd
        assert outs[-1][1].isfinite()
    assert [int(v) for v in graphed.counters.cpu()] == [8, 4, 8]


@pytest.mark.gpu
def test_critic_loss_halves_on_a_fixed_batch():
    from hockey_env_b200.td3 import TD3Config
    L, _ = _learner_pair(TD3Config(), seed=12)
    s, a, r, s2, d = _batch(64, device="cuda:0")
    _, cl = L.update(s, a, r, s2, d)
    first = float(cl)
    for _ in range(200):
        _, cl = L.update(s, a, r, s2, d)
    assert float(cl) < 0.5 * first


@pytest.mark.gpu
def test_td3_training_loop_with_fused_learner():
    import os
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    npz = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "td3_actors.npz")
    for prio in (False, True):
        env = hk.HockeyVecEnv(512, device="cuda:0", seed=2, p2="weak")
        cfg = td3.TD3Config(prioritized_replay=prio, batch_size=256)
        Buf = td3.DevicePrioritizedReplayBuffer if prio else hk.DeviceReplayBuffer
        buf = Buf(512 * 40, device="cuda:0", seed=1)
        actor = hk.load_td3_actor(npz, device="cuda:0", name="stage_3").train()
        L = hk.FusedTD3Learner(actor=actor, config=cfg, replay_buffer=buf, device="cuda:0")
        before = [p.clone() for p in L.actor.parameters()]
        loss = td3.train(env, L, ticks=60, updates_per_tick=2, fused=True)
        assert torch.isfinite(loss) and len(buf) == 512 * 40 and L.train_step == 2 * (60 - 8)
        assert any(not torch.equal(p, q) for p, q in zip(L.actor.parameters(), before))
        assert env.stats()["env_steps"] == 512 * 60
        assert [int(v) for v in L.counters.cpu()] == [104, 52, 104]
        if prio:
            assert (buf.weights[:len(buf)] < 1e8).any()
        env.close()


@pytest.mark.gpu
def test_checkpoints_move_between_learners():
    from hockey_env_b200.actor import FusedActor
    from hockey_env_b200.td3 import DeviceTD3Learner, TD3Config
    L, _ = _learner_pair(TD3Config(policy_update_freq=1), seed=13)
    L.update(*_batch(128, seed=2, device="cuda:0"))
    T = DeviceTD3Learner(device="cuda:0")
    T.load_state_dict(L.state_dict())
    x = torch.randn(100, 18, device="cuda:0")
    with torch.no_grad():
        assert torch.equal(T.actor(x), L.actor(x))
        assert all(torch.equal(u, v) for u, v in zip(T.critic(x, L.actor(x)), L.critic(x, L.actor(x))))
    T.update(*_batch(128, seed=3, device="cuda:0"))
    F, _ = _learner_pair(TD3Config(), seed=14)
    F.load_state_dict(T.state_dict())
    with torch.no_grad():
        assert torch.equal(F.actor(x), T.actor(x)) and torch.equal(F.target_actor(x), T.target_actor(x))
    assert F.blocks["actor"].data_ptr() == F.actor.fc1.weight.data_ptr()  # loading wrote into the arena
    assert torch.equal(FusedActor(T.actor).refresh(F.actor).params, FusedActor(T.actor).params)  # refresh reads the arena views
