"""The training-time side of the fused actor: hk_actor_pack (the parameter block packed on the device from a module's
live fp32 parameters, byte-identical to FusedActor.pack), the noisy epilogue of hk_actor_forward_noisy /
hk_actor_forward_pool_noisy (Philox + Box-Muller exploration noise keyed on seed, row and a device counter), and the
Python layers above them: FusedActor.refresh, FusedActorPool.set, noise= on both callables, collect(noise=) and
td3.train(fused=True)."""
import math
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

NPZ = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "td3_actors.npz")
P = 256 * 24 * 4 + 256 * 256 * 2 + 16 * 256 * 2 + 2 * 256 * 4 + 16 * 4  # bytes of one packed actor
M32 = np.uint64(0xFFFFFFFF)
STREAM_ACTOR_NOISE = 4


# ---- host restatement of the noise (csrc/hk_actor.cuh NoiseKey, hk_math.cuh philox) -----------------------------------

def philox(seed, c0c1, c2, c3):
    """Philox4x32-10 as hk::philox(seed, c0c1, c2, c3), vectorised over c0c1 (uint64 array); returns 4 uint64 arrays."""
    with np.errstate(over="ignore"):
        k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
        c0c1 = np.asarray(c0c1, dtype=np.uint64)
        c0, c1 = c0c1 & M32, c0c1 >> np.uint64(32)
        c2 = np.full_like(c0, np.uint64(c2))
        c3 = np.full_like(c0, np.uint64(c3))
        for _ in range(10):
            p0 = np.uint64(0xD2511F53) * c0
            p1 = np.uint64(0xCD9E8D57) * c2
            c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
            k0 = (k0 + np.uint64(0x9E3779B9)) & M32
            k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c0, c1, c2, c3


def noise_key(counter):
    """Philox counter words 2 and 3 of a call with device counter `counter`."""
    return counter & 0xFFFFFFFF, STREAM_ACTOR_NOISE | (((counter >> 32) & 0xFFFFFF) << 8)


def uniforms(a, b):
    """Box-Muller inputs from two Philox words: u1 in (0, 1], u2 in [0, 1) (24-bit, exact in float32)."""
    return ((a >> np.uint64(8)) + np.uint64(1)).astype(np.float64) * 2.0**-24, (b >> np.uint64(8)).astype(np.float64) * 2.0**-24


def host_normals(seed, rows, counter):
    """float64 [len(rows), 4]: the four standard normals of each row (global row index = row0 + i)."""
    c2, c3 = noise_key(counter)
    x, y, z, w = philox(seed, np.asarray(rows, dtype=np.uint64), c2, c3)
    out = []
    for a, b in ((x, y), (z, w)):
        u1, u2 = uniforms(a, b)
        r = np.sqrt(-2.0 * np.log(u1))
        out += [r * np.cos(2 * np.pi * u2), r * np.sin(2 * np.pi * u2)]
    return np.stack(out, 1)


# ---- CPU ------------------------------------------------------------------------------------------------------------

def test_philox_restatement_known_answers():
    """Random123's known-answer vectors for Philox4x32-10 (key = (k0, k1), counter = (c0, c1, c2, c3))."""
    got = philox(0, [0], 0, 0)
    assert [int(v[0]) for v in got] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    got = philox(0xFFFFFFFFFFFFFFFF, [0xFFFFFFFFFFFFFFFF], 0xFFFFFFFF, 0xFFFFFFFF)
    assert [int(v[0]) for v in got] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]


def test_noise_key_and_uniform_mapping():
    assert noise_key(0) == (0, 4)
    assert noise_key(7) == (7, 4)
    assert noise_key((5 << 32) | 9) == (9, 4 | (5 << 8))  # the counter's high bits go above the stream tag
    words = np.array([0, 0xFF, 0x100, 0x7FFFFFFF, 0xFFFFFF00, 0xFFFFFFFF], dtype=np.uint64)
    u1, u2 = uniforms(words, words)
    assert (u1 > 0).all() and (u1 <= 1).all() and u1[-1] == 1.0 and u1[0] == 2.0**-24
    assert (u2 >= 0).all() and (u2 < 1).all() and u2[0] == 0.0
    # every uniform is a multiple of 2^-24 below 2^24 * 2^-24: exact in float32, so device and host start equal
    assert np.array_equal(u1.astype(np.float32).astype(np.float64), u1)
    z = host_normals(123, np.arange(100_000), 5)
    assert np.isfinite(z).all() and np.abs(z).max() <= math.sqrt(48 * math.log(2)) + 1e-12
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1) < 0.02
    # a row's normals depend on its global index only
    assert np.array_equal(host_normals(123, np.arange(40_000, 40_010), 5), z[40_000:40_010])


def test_new_abi_error_convention_without_gpu():
    import hockey_env_b200 as hk
    L = hk.load_library()
    INV = hk._lib.HK_E_INVALID
    A = 0x10000  # an aligned address: every call below is rejected before anything is read through it

    def fwd(params=A, obs=A, act=A, stride=4, n=100, seed=1, counter=A, sigma=0.2, clip=0.5, row0=0, device=0):
        return L.hk_actor_forward_noisy(params, obs, act, stride, n, seed, counter, sigma, clip, row0, device, None)

    def pool(params=A, k=2, choice=A, obs=A, act=A, stride=4, n=100, scratch=A, seed=1, counter=A, sigma=0.2, clip=0.5, row0=0,
             device=0):
        return L.hk_actor_forward_pool_noisy(params, k, choice, obs, act, stride, n, scratch, seed, counter, sigma, clip, row0,
                                             device, None)

    def pack(w1=A, b1=A, w2=A, b2=A, w3=A, b3=A, params=A, device=0):
        return L.hk_actor_pack(w1, b1, w2, b2, w3, b3, params, device, None)

    noise_cases = [(dict(counter=None), b"NULL"), (dict(counter=A + 4), b"counter needs 8-byte"),
                   (dict(sigma=-0.1), b"sigma"), (dict(sigma=float("nan")), b"sigma"), (dict(sigma=float("inf")), b"sigma"),
                   (dict(clip=float("nan")), b"clip"), (dict(row0=-1), b"row0")]
    fwd_cases = [(dict(params=None), b"NULL"), (dict(obs=None), b"NULL"), (dict(act=None), b"NULL"), (dict(n=0), b"n must be"),
                 (dict(stride=3), b"act_stride"), (dict(params=A + 8), b"alignment"), (dict(obs=A + 4), b"alignment")]
    pool_cases = [(dict(params=None), b"NULL"), (dict(choice=None), b"NULL"), (dict(scratch=None), b"NULL"),
                  (dict(n=2**31), b"n must be"), (dict(stride=3), b"act_stride"), (dict(k=0), b"k must be"),
                  (dict(k=4097), b"k must be"), (dict(choice=A + 2), b"alignment"), (dict(scratch=A + 4), b"alignment")]
    pack_cases = [(dict(w1=None), b"NULL"), (dict(b1=None), b"NULL"), (dict(w2=None), b"NULL"), (dict(b2=None), b"NULL"),
                  (dict(w3=None), b"NULL"), (dict(b3=None), b"NULL"), (dict(params=None), b"NULL"),
                  (dict(params=A + 4), b"16-byte"), (dict(w2=A + 2), b"4-byte"), (dict(b3=A + 1), b"4-byte")]
    for fn, name, cases in ((fwd, b"hk_actor_forward_noisy", fwd_cases + noise_cases),
                            (pool, b"hk_actor_forward_pool_noisy", pool_cases + noise_cases),
                            (pack, b"hk_actor_pack", pack_cases)):
        for kw, msg in cases:
            assert fn(**kw) == INV, (name, kw)
            err = L.hk_last_error()
            assert name + b":" in err and msg in err, (kw, err)
        if not torch.cuda.is_available():
            assert fn() == hk._lib.HK_E_NODEVICE, name
            assert b"no CUDA device" in L.hk_last_error()
    # clip <= 0 and +inf mean "no clip": valid arguments
    if not torch.cuda.is_available():
        for clip in (0.0, -1.0, float("inf")):
            assert fwd(clip=clip) == hk._lib.HK_E_NODEVICE


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _golden(device):
    from hockey_env_b200.actor import load_td3_actor
    return [load_td3_actor(NPZ, device=device, name=nm) for nm in ("stage_3", "competition")]


def _random_actor(seed, device="cuda:0", scale=1.0):
    from hockey_env_b200.actor import ActorNetwork
    torch.manual_seed(seed)
    a = ActorNetwork().to(device)
    with torch.no_grad():
        for p in a.parameters():
            p.mul_(scale)
    return a


def _rounding_ties_actor(device="cuda:0"):
    """Weights whose low 16 bits sit at and next to the bf16 rounding tie (0x8000), with both parities of the kept
    part, signed zeros and subnormals: the cases where a conversion other than round-to-nearest-even would differ."""
    a = _random_actor(77, device)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for p in a.parameters():
            hi = torch.randint(0x3A00, 0x4000, p.shape, generator=g, dtype=torch.int32)
            hi = hi | (torch.randint(0, 2, p.shape, generator=g, dtype=torch.int32) << 15)
            lo = torch.tensor([0x8000, 0x7FFF, 0x8001, 0x0000, 0xFFFF], dtype=torch.int32)[
                torch.randint(0, 5, p.shape, generator=g)]
            bits = (hi << 16) | lo
            flat = bits.flatten()
            flat[:4] = torch.tensor([0, -2**31, 1, 0x00008000], dtype=torch.int32)  # +0, -0, subnormals
            p.copy_(flat.view(p.shape).view(torch.float32).to(device))
    return a


def _host_pack(actor):
    from hockey_env_b200.actor import FusedActor, _reference_state_dict
    return FusedActor.pack(_reference_state_dict(actor, "test"))


def _obs(n, seed, device="cuda:0"):
    g = torch.Generator(device=device).manual_seed(seed)
    scale = torch.tensor([2, 2, .5, 4, 4, 3, 2, 2, .5, 4, 4, 3, 3, 2, 8, 8, 4, 4], device=device)
    return torch.randn((n, 18), device=device, generator=g) * scale


def _zero_actor(device="cuda:0"):
    """All weights and biases zero: the kernel outputs tanh(0) = 0, so a noisy call returns the clamped noise itself."""
    a = _random_actor(0, device)
    with torch.no_grad():
        for p in a.parameters():
            p.zero_()
    return a


@pytest.mark.gpu
def test_device_pack_equals_host_pack_byte_for_byte():
    import hockey_env_b200 as hk
    modules = _golden("cuda:0") + [_random_actor(s) for s in (1, 2, 3)] + [_random_actor(4, scale=300.0),
                                                                           _random_actor(5, scale=1e-30), _rounding_ties_actor()]
    f = hk.FusedActor(_random_actor(99))
    for i, m in enumerate(modules):
        f.refresh(m)
        torch.cuda.synchronize()
        want = _host_pack(m)
        got = f.params.cpu()
        bad = (got != want).nonzero().flatten()
        assert bad.numel() == 0, f"module {i}: {bad.numel()} bytes differ, first at {bad[:8].tolist()}"


@pytest.mark.gpu
def test_pool_set_repacks_one_slot_only():
    import hockey_env_b200 as hk
    actors = _golden("cuda:0") + [_random_actor(11)]
    pool = hk.FusedActorPool(actors)
    before = pool.table.clone()
    new = _random_actor(12)
    pool.set(1, new)
    torch.cuda.synchronize()
    t = pool.table.cpu()
    assert torch.equal(t[1], _host_pack(new))
    assert torch.equal(t[0], before[0].cpu()) and torch.equal(t[2], before[2].cpu())
    with pytest.raises(IndexError):
        pool.set(3, new)


@pytest.mark.gpu
def test_refresh_then_forward_equals_fresh_fused_actor():
    import hockey_env_b200 as hk
    a, b = _golden("cuda:0")
    f = hk.FusedActor(a)
    obs = _obs(50_000, 3)
    f.refresh(b)
    assert torch.equal(f(obs).clone(), hk.FusedActor(b)(obs))
    # a module trained in place: refresh follows its live parameters
    m = _random_actor(21)
    f.refresh(m)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(0.01)
    f.refresh(m)
    assert torch.equal(f(obs).clone(), hk.FusedActor(m)(obs))


def _call_noisy(L, f, obs, out, sigma, clip, row0, counter, seed):
    import ctypes as C
    import hockey_env_b200 as hk
    hk._lib.check(L.hk_actor_forward_noisy(C.c_void_p(f.params.data_ptr()), C.c_void_p(obs.data_ptr()), C.c_void_p(out.data_ptr()),
                                           int(out.stride(0)), obs.shape[0], seed, C.c_void_p(counter.data_ptr()), sigma, clip, row0, 0,
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129, 4096, 100_003])
def test_sigma_zero_is_bit_identical_to_the_plain_kernel(n):
    import hockey_env_b200 as hk
    L = hk.load_library()
    a = _golden("cuda:0")[0]
    f = hk.FusedActor(a)
    obs = _obs(n, n)
    counter = torch.tensor([12345], dtype=torch.int64, device="cuda:0")
    got = _call_noisy(L, f, obs, torch.full((n, 4), 9.0, device="cuda:0"), 0.0, 0.3, 0, counter, 7)
    assert torch.equal(got, f(obs))
    assert torch.equal(f(obs, noise=0.0), f(obs)) and int(f.counter) == 0  # noise=0: the plain call, counter untouched


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 16])
@pytest.mark.parametrize("n", [1, 129, 100_003])
def test_pool_sigma_zero_is_bit_identical(n, k):
    import ctypes as C
    import hockey_env_b200 as hk
    L = hk.load_library()
    actors = [_golden("cuda:0")[s % 2] if s < 2 else _random_actor(s) for s in range(k)]
    pool = hk.FusedActorPool(actors)
    obs = _obs(n, n + k)
    g = torch.Generator(device="cuda:0").manual_seed(n + k)
    choice = torch.randint(-1, k + 1, (n,), device="cuda:0", generator=g, dtype=torch.int32)
    want = pool(obs, choice, out=torch.full((n, 4), 2.0, device="cuda:0")).clone()
    out = torch.full((n, 4), 2.0, device="cuda:0")
    scratch = torch.empty(int(L.hk_actor_pool_scratch_bytes(n, k)), dtype=torch.uint8, device="cuda:0")
    counter = torch.tensor([3], dtype=torch.int64, device="cuda:0")
    hk._lib.check(L.hk_actor_forward_pool_noisy(C.c_void_p(pool.table.data_ptr()), k, C.c_void_p(choice.data_ptr()),
                                                C.c_void_p(obs.data_ptr()), C.c_void_p(out.data_ptr()), 4, n,
                                                C.c_void_p(scratch.data_ptr()), 5, C.c_void_p(counter.data_ptr()), 0.0, 0.0, 0, 0,
                                                C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert torch.equal(out, want)


@pytest.mark.gpu
def test_noise_repeats_and_depends_on_the_key_only():
    import hockey_env_b200 as hk
    a = _golden("cuda:0")[1]
    f = hk.FusedActor(a, seed=2024)
    n = 10_000
    obs = _obs(n, 1)
    f.counter.fill_(41)
    x = f(obs, noise=0.2).clone()
    assert int(f.counter) == 42
    y = f(obs, noise=0.2).clone()
    assert not torch.equal(x, y)                       # a new counter: fresh noise
    f.counter.fill_(41)
    assert torch.equal(f(obs, noise=0.2), x)           # the same (seed, counter): the same draw, bit for bit
    # shards: rows [0, 3000) and [3000, n) with row0 = 3000 draw what one call over the batch draws
    f.counter.fill_(41)
    lo = f(obs[:3000].contiguous(), noise=0.2).clone()
    f.counter.fill_(41)
    hi = f(obs[3000:].contiguous(), noise=0.2, row0=3000).clone()
    assert torch.equal(torch.cat([lo, hi]), x)
    # a shorter batch: its rows draw what the same rows of the longer one draw
    f.counter.fill_(41)
    assert torch.equal(f(obs[:1234].contiguous(), noise=0.2), x[:1234])
    # another seed: another draw
    g = hk.FusedActor(a, seed=2025)
    g.counter.fill_(41)
    assert not torch.equal(g(obs, noise=0.2), x)


@pytest.mark.gpu
def test_noise_matches_host_box_muller():
    import hockey_env_b200 as hk
    f = hk.FusedActor(_zero_actor(), seed=0xDEADBEEF12345678)
    n, row0, ctr = 200_003, 5_000_000_000, (3 << 32) + 17
    obs = _obs(n, 2)
    f.counter.fill_(ctr)
    # sigma = 1/8: |sigma z| <= 0.73 never reaches the [-1, 1] clamp, and the scaling is exact
    z = (f(obs, noise=0.125, row0=row0) * 8).double().cpu().numpy()
    want = host_normals(f.seed, row0 + np.arange(n, dtype=np.uint64), ctr)
    err = np.abs(z - want)
    assert err.max() < 1e-5, (err.max(), np.unravel_index(err.argmax(), err.shape))


@pytest.mark.gpu
def test_noise_is_standard_normal_and_clip_holds():
    from scipy import stats
    import hockey_env_b200 as hk
    f = hk.FusedActor(_zero_actor(), seed=99)
    n = 1_000_000
    obs = _obs(n, 4)
    z = (f(obs, noise=0.125) * 8).double().cpu().numpy()
    for col in range(4):
        p = stats.kstest(z[:, col], "norm").pvalue
        assert p > 1e-3, (col, p)
    assert abs(np.corrcoef(z[:, 0], z[:, 1])[0, 1]) < 5e-3 and abs(np.corrcoef(z[:, 0], z[:, 2])[0, 1]) < 5e-3
    clip = 0.3
    c = f(obs, noise=1.0, noise_clip=clip).cpu()
    assert float(c.abs().max()) <= np.float32(clip)
    assert float((c.abs() == np.float32(clip)).float().mean()) > 0.7  # P(|z| >= 0.3) = 0.76
    # no clip (None, <= 0, +inf): the [-1, 1] action clamp only
    for nc in (None, 0.0, -1.0, float("inf")):
        f.counter.fill_(0)
        u = f(obs, noise=1.0, noise_clip=nc).cpu()
        assert float(u.abs().max()) == 1.0 and float((u.abs() == 1).float().mean()) > 0.3


@pytest.mark.gpu
def test_noise_on_real_actor_is_clamped_sum():
    """act = clamp(actor(obs) + sigma z, -1, 1) with the plain kernel's actor(obs), to float32 rounding."""
    import hockey_env_b200 as hk
    f = hk.FusedActor(_golden("cuda:0")[0], seed=8)
    n = 50_000
    obs = _obs(n, 6)
    base = f(obs).double().cpu().numpy()
    got = f(obs, noise=0.2, noise_clip=0.5).double().cpu().numpy()
    want = np.clip(base + np.clip(0.2 * host_normals(8, np.arange(n), 0), -0.5, 0.5), -1, 1)
    assert np.abs(got - want).max() < 1e-5


@pytest.mark.gpu
def test_pool_noise_is_keyed_on_the_row_not_the_group():
    import hockey_env_b200 as hk
    actors = _golden("cuda:0") + [_random_actor(31)]
    pool = hk.FusedActorPool(actors, seed=77)
    fused = [hk.FusedActor(a, seed=77) for a in actors]
    n = 30_001
    obs = _obs(n, 9)
    g = torch.Generator(device="cuda:0").manual_seed(1)
    choice = torch.randint(-1, 3, (n,), device="cuda:0", generator=g, dtype=torch.int32)
    pool.counter.fill_(5)
    got = pool(obs, choice, out=torch.full((n, 4), 4.0, device="cuda:0"), noise=0.2, noise_clip=0.5).clone()
    assert int(pool.counter) == 6
    want = torch.full((n, 4), 4.0, device="cuda:0")
    for s, f in enumerate(fused):
        f.counter.fill_(5)
        m = choice == s
        want[m] = f(obs, noise=0.2, noise_clip=0.5)[m]
    assert torch.equal(got, want)


@pytest.mark.gpu
def test_captured_graph_draws_fresh_reproducible_noise():
    import hockey_env_b200 as hk
    f = hk.FusedActor(_golden("cuda:0")[0], seed=3)
    n = 20_000
    obs = _obs(n, 12)
    out = torch.zeros((n, 4), device="cuda:0")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        f(obs, out=out, noise=0.2)  # warm-up: kernel attributes set
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        f(obs, out=out, noise=0.2)
    f.counter.fill_(100)
    draws = []
    for _ in range(3):
        graph.replay()
        draws.append(out.clone())
    torch.cuda.synchronize()
    assert int(f.counter) == 103
    assert not torch.equal(draws[0], draws[1]) and not torch.equal(draws[1], draws[2])
    for j, d in enumerate(draws):  # replay j drew with counter 100 + j
        f.counter.fill_(100 + j)
        assert torch.equal(f(obs, noise=0.2), d)


@pytest.mark.gpu
def test_collect_with_fused_actor_and_noise():
    import hockey_env_b200 as hk
    env = hk.HockeyVecEnv(1024, device="cuda:0", seed=4, p2="weak")
    f = hk.FusedActor(_golden("cuda:0")[0], seed=1)
    buf = hk.DeviceReplayBuffer(1024 * 10, device="cuda:0")
    hk.collect(env, f, buf, 10, noise=0.2)
    assert len(buf) == 1024 * 10 and int(f.counter) == 10
    a = buf.action[:1024]
    assert float(a.abs().max()) <= 1.0
    assert not torch.equal(a, f(buf.obs[:1024].contiguous()))  # the stored actions carry the exploration noise
    env.close()


@pytest.mark.gpu
def test_td3_training_loop_fused():
    """td3.train(fused=True) set up like the unfused loop test: the plumbing runs, losses stay finite, the buffers fill,
    parameters move, and the mirror ends equal to the host pack of the trained actor."""
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    from hockey_env_b200.actor import FusedActor
    for prio in (False, True):
        env = hk.HockeyVecEnv(512, device="cuda:0", seed=2, p2="weak")
        cfg = td3.TD3Config(prioritized_replay=prio, batch_size=256)
        Buf = td3.DevicePrioritizedReplayBuffer if prio else hk.DeviceReplayBuffer
        buf = Buf(512 * 40, device="cuda:0", seed=1)
        actor = hk.load_td3_actor(NPZ, device="cuda:0", name="stage_3").train()
        L = td3.DeviceTD3Learner(actor=actor, config=cfg, replay_buffer=buf, device="cuda:0")
        before = [p.clone() for p in L.actor.parameters()]
        loss = td3.train(env, L, ticks=60, updates_per_tick=2, fused=True)
        assert torch.isfinite(loss) and len(buf) == 512 * 40 and L.train_step == 2 * (60 - 8)
        assert any(not torch.equal(p, q) for p, q in zip(L.actor.parameters(), before))
        assert env.stats()["env_steps"] == 512 * 60
        assert isinstance(L.fused_actor, FusedActor) and int(L.fused_actor.counter) == 60
        torch.cuda.synchronize()
        assert torch.equal(L.fused_actor.params.cpu(), _host_pack(L.actor))
        assert float(buf.action[:len(buf)].abs().max()) <= 1.0
        if prio:
            assert (buf.weights[:len(buf)] < 1e8).any()
        env.close()
