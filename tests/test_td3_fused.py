"""FusedTD3Learner: one TD3 update in one sm_100a launch (csrc/hk_td3.cuh, hk_td3_update), against torch learners in
float32 and float64 built from the same weights, batch indices and target noise."""
import copy
import os
import subprocess
import sys
from dataclasses import replace

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
        assert L.hk_td3_cluster_size(0) == _lib.HK_E_NODEVICE and b"hk_td3_cluster_size:" in L.hk_last_error()


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


def _reference(state, batch, z, cfg, dtype, do_actor, weights=None, adam=None, device="cuda:0", a_clamp=1.0):
    """DeviceTD3Learner.update written out for `dtype` on `device` with the target noise z given: returns the nets, the
    Adam moments, the losses, the priorities and the share of entries at the noise clip and at the a' clamp ("edges").
    Every net, the critics' action bounds included, comes from `state`.  adam: the optimizers' start state
    ({m,v}_{actor,critic} flat in state_dict order, "t": (critic steps, actor steps, ...)); None: fresh optimizers.
    a_clamp: the bound of a' (the reference clamps to [-1, 1]; inf stands for an update that drops the clamp)."""
    from hockey_env_b200.actor import ActorNetwork
    from hockey_env_b200.td3 import TwinQNetwork, huber_weighted
    dev = device
    nets = {"policy": ActorNetwork(), "critic": TwinQNetwork(), "target_policy": ActorNetwork(), "target_critic": TwinQNetwork()}
    for k, n in nets.items():
        n.load_state_dict(state[k])
        n.to(dev, dtype)
    actor, critic, ta, tc = nets["policy"], nets["critic"], nets["target_policy"], nets["target_critic"]
    aopt = torch.optim.Adam(actor.parameters(), lr=cfg.lr_pol, weight_decay=cfg.wd_pol)
    copt = torch.optim.Adam(critic.parameters(), lr=cfg.lr_q, weight_decay=cfg.wd_q)
    if adam is not None:
        for opt, net, key, steps in ((copt, critic, "critic", adam["t"][0]), (aopt, actor, "actor", adam["t"][1])):
            o = 0
            for p in net.parameters():
                m, v = (adam[f"{k}_{key}"][o:o + p.numel()].view(p.shape).to(dev, dtype).clone() for k in ("m", "v"))
                opt.state[p] = {"step": torch.tensor(float(steps)), "exp_avg": m, "exp_avg_sq": v}
                o += p.numel()
    s, a, r, s2, d = (t.to(dev, dtype) for t in batch)
    w = None if weights is None else weights.to(dev, dtype)
    with torch.no_grad():
        a2 = ta(s2)
        raw = z.to(dev, dtype) * cfg.target_action_noise_scale
        noise = raw.clamp(-cfg.target_action_noise_clip, cfg.target_action_noise_clip)
        q1t, q2t = tc(s2, (a2 + noise).clamp(-a_clamp, a_clamp))
        y = r + cfg.gamma * (1 - d) * torch.minimum(q1t, q2t)
        edges = {"noise_clip": float((raw.abs() > cfg.target_action_noise_clip).double().mean()),
                 "a_clamp": float(((a2 + noise).abs() > 1).double().mean())}
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
            "closs": closs.detach().reshape(1), "aloss": None if aloss is None else aloss.detach().reshape(1), "prio": prio,
            "edges": edges}


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
    bad = T.state_dict()
    bad["target_critic"] = dict(bad["target_critic"], action_range=bad["target_critic"]["action_range"] * 2)
    before = F.arena.clone()
    with pytest.raises(ValueError, match="action_range"):  # the kernel would normalise the target critic's input wrongly
        F.load_state_dict(bad)
    assert torch.equal(F.arena, before)
    assert torch.equal(FusedActor(T.actor).refresh(F.actor).params, FusedActor(T.actor).params)  # refresh reads the arena views


# ---- start states away from the defaults --------------------------------------------------------------------------------
# Every pair of hyper-parameters equal, Adam at step 1 (update = lr sign(g)), noise counter 0 and the default action bounds
# (normalisation = identity) hide whole classes of one-line mistakes.  These cases move each of them off its default.

HP_DISTINCT = dict(lr_q=7e-4, lr_pol=2e-4, tau_critic=0.02, tau_actor=0.003, wd_q=3e-3, wd_pol=1e-2, gamma=0.95, beta=0.4,
                   target_action_noise_scale=0.35, target_action_noise_clip=0.12)
BOUNDS = ([-2.0, -1.0, -0.5, -3.0], [4.0, 2.0, 1.0, 6.0])             # action_low, action_range per column
BOUNDS_INF = ([-2.0, -1.0, -0.5, -3.0], [4.0, float("inf"), 1.0, 6.0])  # an infinite range: no normalisation
CASES = {
    "midtrain": {},
    "hparams": dict(cfg=HP_DISTINCT),
    "hparams_prio": dict(cfg=HP_DISTINCT, prio=True),
    "bounds": dict(bounds=BOUNDS),
    "bounds_ckpt": dict(bounds=BOUNDS, ckpt=True),  # bounds arriving through FusedTD3Learner.load_state_dict
    "bounds_inf": dict(bounds=BOUNDS_INF),
    "saturated": dict(target_bias=4.0),             # tanh(target fc3) ~ +-1: a' + noise is clamped on about half the entries
    "noise_clip": dict(cfg=dict(target_action_noise_scale=1.0, target_action_noise_clip=0.05)),
    "sigma0": dict(cfg=dict(target_action_noise_scale=0.0)),
    "clip0": dict(cfg=dict(target_action_noise_clip=0.0)),
}
COUNTERS = (999, 333, 77)  # critic steps, actor steps and noise counter of the start state
BLOCKS = ("actor", "critic", "target_actor", "target_critic", "m_actor", "v_actor", "m_critic", "v_critic")


def _case_cfg(case, actor_step, **kw):
    from hockey_env_b200.td3 import TD3Config
    c = CASES[case]
    return TD3Config(policy_update_freq=1 if actor_step else 2, prioritized_replay=c.get("prio", False), **{**c.get("cfg", {}), **kw})


def _start_state(seed, bounds=None, target_bias=None, counters=COUNTERS):
    """Seeded CPU start state: the four nets in checkpoint form (targets perturbed away from the online nets; both critics
    with `bounds`; the target actor's fc3.bias +-target_bias) and a mid-training Adam state: v log-uniform in
    [1e-7, 1e-4], m ~ N(0, 1) sqrt(v) / 2, so that the update is far from Adam's sign-like first step."""
    from hockey_env_b200.actor import ActorNetwork
    from hockey_env_b200.td3 import TwinQNetwork
    torch.manual_seed(seed)
    nets = {"policy": ActorNetwork(), "critic": TwinQNetwork()}
    nets["target_policy"], nets["target_critic"] = copy.deepcopy(nets["policy"]), copy.deepcopy(nets["critic"])
    with torch.no_grad():
        for k in ("target_policy", "target_critic"):
            for p in nets[k].parameters():
                p.add_(0.01 * torch.randn_like(p))
        if bounds is not None:
            low, rng = torch.tensor(bounds[0]), torch.tensor(bounds[1])
            for k in ("critic", "target_critic"):
                nets[k].action_low.copy_(low)
                nets[k].action_range.copy_(rng)
                nets[k].action_high.copy_(low + rng)
        if target_bias is not None:
            nets["target_policy"].fc3.bias.copy_(target_bias * torch.tensor([1.0, -1.0, 1.0, -1.0]))
    g = torch.Generator().manual_seed(seed + 1)
    adam = {"t": tuple(counters)}
    for name, net in (("actor", nets["policy"]), ("critic", nets["critic"])):
        n = sum(p.numel() for p in net.parameters())
        v = 10.0 ** (torch.rand(n, generator=g) * 3 - 7)
        adam["v_" + name], adam["m_" + name] = v, 0.5 * v.sqrt() * torch.randn(n, generator=g)
    return {k: {n: t.detach().clone() for n, t in v.state_dict().items()} for k, v in nets.items()}, adam


def _case_state(case, seed):
    c = CASES[case]
    return _start_state(seed, c.get("bounds"), c.get("target_bias"))


def _fused_learner(nets, adam, cfg, buf=None, seed=11, ckpt=False):
    """A FusedTD3Learner on cuda:0 in the start state: the online nets through the constructor and the targets loaded
    into its modules, or (ckpt=True) a default learner that loads the whole checkpoint; Adam moments and counters are
    written into the arena."""
    from hockey_env_b200.actor import ActorNetwork
    from hockey_env_b200.td3 import FusedTD3Learner, TwinQNetwork
    if ckpt:
        L = FusedTD3Learner(config=cfg, replay_buffer=buf, device="cuda:0", seed=seed)
        L.load_state_dict(nets)
    else:
        actor, critic = ActorNetwork(), TwinQNetwork()
        actor.load_state_dict(nets["policy"])
        critic.load_state_dict(nets["critic"])
        L = FusedTD3Learner(actor=actor, critic=critic, config=cfg, replay_buffer=buf, device="cuda:0", seed=seed)
        L.target_actor.load_state_dict(nets["target_policy"])
        L.target_critic.load_state_dict(nets["target_critic"])
    for k in ("m_actor", "v_actor", "m_critic", "v_critic"):
        L.blocks[k].copy_(adam[k])
    L.counters.copy_(torch.tensor(adam["t"], dtype=torch.int64))
    return L


def _snapshot(L):
    """The learner's state in the form of _start_state: checkpoint, Adam moments and counters (CPU copies)."""
    nets = {k: {n: t.detach().cpu().clone() for n, t in v.items()} for k, v in L.state_dict().items()}
    adam = {k: L.blocks[k].cpu().clone() for k in ("m_actor", "v_actor", "m_critic", "v_critic")}
    adam["t"] = tuple(int(v) for v in L.counters.cpu())
    return nets, adam


def _importance_weights(pw, n, beta):
    """DeviceTD3Learner.importance_weights in pw's dtype, from the buffer weights pw of the batch's indices."""
    w = (1.0 / (pw / pw.sum() * n)) ** beta
    return w / w.max()


def _draw_batch(buf, b):
    """The indices and rows that the next update_from_buffer(b) draws, and the buffer's weights before it; the buffer's
    generator is left as it was."""
    g = buf.gen.get_state()
    idx = buf.sample_indices(b)
    buf.gen.set_state(g)
    buf.last_batch_inds = None
    return idx, tuple(t[idx].clone() for t in (buf.obs, buf.action, buf.reward, buf.next_obs, buf.done)), buf.weights.clone()


def _tolerances(ref32, ref64):
    """The fused learner's allowance against float64, per output: 4x torch fp32's own error plus 1e-7."""
    return {k: 4 * float((ref32[k].double().cpu() - ref64[k].cpu()).abs().max()) + 1e-7
            for k in BLOCKS + ("closs", "aloss", "prio") if ref64[k] is not None}


def _excess(got, ref64, tol):
    """{output: max |got - ref64| / tolerance} over the outputs in both; above 1 fails the comparison."""
    return {k: float((got[k].double().cpu() - ref64[k].cpu()).abs().max()) / tol[k] for k in tol if got.get(k) is not None}


def _check_tight(L, losses, ref32, ref64):
    """Every arena block, parameters included, and both losses within _tolerances: with a mid-training Adam state the
    update is well conditioned, unlike the sign-like first step that _check_against_float64 allows 2 lr for."""
    assert (losses[0] is None) == (ref64["aloss"] is None)
    bad = {k: r for k, r in _excess(dict(L.blocks, closs=losses[1], aloss=losses[0]), ref64, _tolerances(ref32, ref64)).items()
           if r > 1}
    assert not bad, bad


def _check_priorities(buf, idx, before, ref32, ref64):
    """The written-back priorities (last occurrence of an index wins) against float64; other rows untouched."""
    last = {int(ix): r for r, ix in enumerate(idx.tolist())}
    ixs, rows = torch.tensor(list(last)), torch.tensor(list(last.values()))
    err = float((buf.weights.cpu()[ixs].double() - ref64["prio"].cpu()[rows]).abs().max())
    assert err <= _tolerances(ref32, ref64)["prio"], err
    untouched = torch.ones(buf.weights.shape[0], dtype=torch.bool)
    untouched[ixs] = False
    assert torch.equal(buf.weights.cpu()[untouched], before.cpu()[untouched])


# ---- the reference has teeth at every edge (CPU) ---------------------------------------------------------------------
# For each one-line mistake the GPU tests below must catch, the float64 reference computed with the mistaken semantics
# differs from the correct one by far more than the tolerance the fused learner is held to at that configuration.

SEED_HI, CTR_HI = (1 << 40) + 5, (1 << 32) + 1  # a seed and a noise counter with non-zero high words

MUTANTS = {  # name: the case it needs, and the reference arguments that compute the mistaken semantics
    "bounds_dropped": ("bounds", dict(state=dict(bounds=None))),
    "a_clamp_dropped": ("saturated", dict(a_clamp=float("inf"))),
    "noise_clip_dropped": ("noise_clip", dict(cfg=dict(target_action_noise_clip=float("inf")))),
    "lr_swapped": ("hparams", dict(cfg=dict(lr_q=HP_DISTINCT["lr_pol"], lr_pol=HP_DISTINCT["lr_q"]))),
    "tau_swapped": ("hparams", dict(cfg=dict(tau_critic=HP_DISTINCT["tau_actor"], tau_actor=HP_DISTINCT["tau_critic"]))),
    "wd_swapped": ("hparams", dict(cfg=dict(wd_q=HP_DISTINCT["wd_pol"], wd_pol=HP_DISTINCT["wd_q"]))),
    "gamma_default": ("hparams", dict(cfg=dict(gamma=0.99))),
    "sigma_default": ("hparams", dict(cfg=dict(target_action_noise_scale=0.2))),
    "beta_default": ("hparams_prio", dict(beta=0.15)),
    "adam_steps_swapped": ("midtrain", dict(t=(COUNTERS[1], COUNTERS[0], COUNTERS[2]))),
    "counter_high_word_dropped": ("midtrain", dict(z=(SEED_HI, CTR_HI & 0xFFFFFFFF))),
    "seed_truncated": ("midtrain", dict(z=(SEED_HI & 0xFFFFFFFF, CTR_HI))),
}


@pytest.mark.parametrize("mutant", list(MUTANTS))
def test_reference_edges_have_teeth(mutant):
    case, mut = MUTANTS[mutant]
    b = 256
    c = CASES[case]
    cfg = _case_cfg(case, True)
    nets, adam = _case_state(case, seed=71)
    batch = _batch(b, seed=72)
    pw = torch.rand(b, generator=torch.Generator().manual_seed(73), dtype=torch.float64) + 0.05 if cfg.prioritized_replay else None

    def run(dtype, **m):
        st = nets
        if "state" in m:
            st, _ = _start_state(71, **{**dict(bounds=c.get("bounds"), target_bias=c.get("target_bias")), **m["state"]})
        seed, ctr = m.get("z", (SEED_HI, CTR_HI))
        z = torch.from_numpy(td3_normals(seed, b, ctr))
        w = None if pw is None else _importance_weights(pw.to(dtype), 3000, m.get("beta", cfg.beta))
        return _reference(st, batch, z.to(dtype), replace(cfg, **m.get("cfg", {})), dtype, True, weights=w,
                          adam=dict(adam, t=m.get("t", adam["t"])), device="cpu", a_clamp=m.get("a_clamp", 1.0))

    ref64, ref32 = run(torch.float64), run(torch.float32)
    tol = _tolerances(ref32, ref64)
    worst = max(_excess(run(torch.float64, **mut), ref64, tol).values())
    assert worst > 100, worst
    if case == "saturated":
        assert ref64["edges"]["a_clamp"] > 0.4, ref64["edges"]
    if case == "noise_clip":
        assert ref64["edges"]["noise_clip"] > 0.9, ref64["edges"]


def test_fused_learner_rejects_unequal_target_critic_bounds():
    from hockey_env_b200.td3 import FusedTD3Learner
    nets, _ = _start_state(61, bounds=BOUNDS)
    FusedTD3Learner._check_action_bounds(nets["critic"], nets["target_critic"])
    for k in ("action_low", "action_range"):
        bad = {n: dict(sd) for n, sd in nets.items()}
        bad["target_critic"][k] = bad["target_critic"][k] + torch.tensor([0.0, 0.5, 0.0, 0.0])
        with pytest.raises(ValueError, match=k):  # checked before anything is loaded, so no device is needed
            FusedTD3Learner.load_state_dict(FusedTD3Learner.__new__(FusedTD3Learner), bad)


# ---- GPU: the fused learner away from the defaults ------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("actor_step", [False, True])
def test_update_cases_against_float64(case, actor_step):
    """One update from a mid-training start state (Adam moments, step counts 999 / 333, noise counter 77) in each case,
    against the float64 reference started from the same state."""
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    b = 256
    cfg = _case_cfg(case, actor_step)
    nets, adam = _case_state(case, seed=21)
    buf = _filled_prio_buffer(3000, seed=22) if cfg.prioritized_replay else None
    L = _fused_learner(nets, adam, cfg, buf, ckpt=CASES[case].get("ckpt", False))
    if buf is not None:
        idx, batch, before = _draw_batch(buf, b)
        pw = before[idx]
        w64, w32 = _importance_weights(pw.double(), buf.size, cfg.beta), _importance_weights(pw, buf.size, cfg.beta)
        losses = L.update_from_buffer(b)
    else:
        batch, w64, w32 = _batch(b, seed=23, device="cuda:0"), None, None
        losses = L.update(*batch)
    torch.cuda.synchronize()
    assert [int(v) for v in L.counters.cpu()] == [COUNTERS[0] + 1, COUNTERS[1] + int(actor_step), COUNTERS[2] + 1]
    z = torch.from_numpy(td3_normals(L.seed, b, COUNTERS[2]))
    ref64 = _reference(nets, batch, z, cfg, torch.float64, actor_step, weights=w64, adam=adam)
    ref32 = _reference(nets, batch, z.float(), cfg, torch.float32, actor_step, weights=w32, adam=adam)
    _check_tight(L, losses, ref32, ref64)
    if buf is not None:
        err = float((L.last_importance_weights().double() - w64).abs().max())
        assert err <= 4 * float((w32.double() - w64).abs().max()) + 1e-7, err
        _check_priorities(buf, idx, before, ref32, ref64)
    edges = ref64["edges"]
    if case == "saturated":
        assert edges["a_clamp"] > 0.4, edges
    elif case in ("noise_clip", "clip0"):
        assert edges["noise_clip"] > 0.9, edges


@pytest.mark.gpu
def test_stepwise_across_the_noise_counter_high_word():
    """Six prioritized updates with policy_update_freq 3 (actor steps with tA != tC), a seed >= 2^32 and the noise counter
    crossing 2^32: each update against the float64 reference started from a snapshot taken just before it."""
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    from hockey_env_b200.td3 import TD3Config
    b = 256
    cfg = TD3Config(prioritized_replay=True, policy_update_freq=3, **HP_DISTINCT)
    nets, adam = _start_state(31, counters=(999, 333, 2**32 - 3))
    buf = _filled_prio_buffer(3000, seed=32)
    L = _fused_learner(nets, adam, cfg, buf, seed=SEED_HI)
    for step in range(1, 7):
        nets, adam = _snapshot(L)
        idx, batch, before = _draw_batch(buf, b)
        pw = before[idx]
        w64, w32 = _importance_weights(pw.double(), buf.size, cfg.beta), _importance_weights(pw, buf.size, cfg.beta)
        losses = L.update_from_buffer(b)
        torch.cuda.synchronize()
        do_actor = step % 3 == 0
        tC, tA, ctr = adam["t"]
        assert [int(v) for v in L.counters.cpu()] == [tC + 1, tA + int(do_actor), ctr + 1]
        z = torch.from_numpy(td3_normals(SEED_HI, b, ctr))
        ref64 = _reference(nets, batch, z, cfg, torch.float64, do_actor, weights=w64, adam=adam)
        ref32 = _reference(nets, batch, z.float(), cfg, torch.float32, do_actor, weights=w32, adam=adam)
        _check_tight(L, losses, ref32, ref64)
        err = float((L.last_importance_weights().double() - w64).abs().max())
        assert err <= 4 * float((w32.double() - w64).abs().max()) + 1e-7, (step, err)
        _check_priorities(buf, idx, before, ref32, ref64)
    assert [int(v) for v in L.counters.cpu()] == [1005, 335, 2**32 + 3]


@pytest.mark.gpu
def test_sample_then_update_equals_update_from_buffer():
    """update() on a prioritized buffer's sample() (last_batch_inds set) and update_from_buffer() are the same update:
    the same draws, a bit-identical arena, priorities and importance weights, and last_batch_inds cleared."""
    from hockey_env_b200.td3 import TD3Config
    cfg = TD3Config(prioritized_replay=True, policy_update_freq=2)
    nets, adam = _start_state(51)
    runs = []
    for via_sample in (True, False):
        buf = _filled_prio_buffer(3000, seed=52)
        L = _fused_learner(nets, adam, cfg, buf)
        draws = []
        for _ in range(3):
            if via_sample:
                batch = buf.sample(256)
                draws.append(buf.last_batch_inds.clone())
                L.update(*batch)
            else:
                draws.append(_draw_batch(buf, 256)[0])
                L.update_from_buffer(256)
            assert buf.last_batch_inds is None
        torch.cuda.synchronize()
        runs.append((draws, L.arena.clone(), buf.weights.clone(), L.last_importance_weights().clone()))
    assert all(torch.equal(u, v) for u, v in zip(runs[0][0], runs[1][0]))
    for u, v in zip(runs[0][1:], runs[1][1:]):
        assert torch.equal(u, v)
    assert not torch.equal(runs[0][2], _filled_prio_buffer(3000, seed=52).weights)  # priorities were written back


def _cluster_run(path):
    """Seeded prioritized updates at B = 1024 and 37, two of them actor steps; saves the arena, the buffer's weights, the
    losses and the cluster size the launches used."""
    import hockey_env_b200 as hk
    from hockey_env_b200.td3 import TD3Config
    nets, adam = _start_state(41)
    buf = _filled_prio_buffer(3000, seed=42)
    L = _fused_learner(nets, adam, TD3Config(prioritized_replay=True, policy_update_freq=2), buf)
    losses = []
    for b in (1024, 1024, 37, 37):
        al, cl = L.update_from_buffer(b)
        losses += [cl] if al is None else [al, cl]
    torch.cuda.synchronize()
    np.savez(path, arena=L.arena.cpu().numpy(), weights=buf.weights.cpu().numpy(), losses=torch.stack(losses).cpu().numpy(),
             cluster=int(hk.load_library().hk_td3_cluster_size(0)))


@pytest.mark.gpu
def test_results_do_not_depend_on_the_cluster_size(tmp_path):
    """The same updates at cluster sizes 16 (the default on a B200), 8, 4, 3 and 1 (HK_TD3_CLUSTER, one process each,
    since the library reads it once) leave byte-identical arenas, priorities and losses."""
    import hockey_env_b200 as hk
    from hockey_env_b200 import _lib
    L = hk.load_library()
    assert L.hk_td3_cluster_size(0) == 16 and L.hk_td3_cluster_size(-1) == _lib.HK_E_INVALID
    _cluster_run(tmp_path / "16.npz")
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([here, os.path.dirname(here)]))
    sizes = (8, 4, 3, 1)
    for n in sizes:
        r = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) +
                           ["-c", "import sys, test_td3_fused as t; t._cluster_run(sys.argv[1])", str(tmp_path / f"{n}.npz")],
                           env=dict(env, HK_TD3_CLUSTER=str(n)), cwd=here, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (n, r.stderr[-3000:])
    want = np.load(tmp_path / "16.npz")
    assert int(want["cluster"]) == 16
    for n in sizes:
        got = np.load(tmp_path / f"{n}.npz")
        assert int(got["cluster"]) == n
        for k in ("arena", "weights", "losses"):
            assert got[k].tobytes() == want[k].tobytes(), (n, k)
