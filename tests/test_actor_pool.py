"""The snapshot-pool actor kernel (csrc/hk_actor.cuh k_actor_pool_mlp, hk_actor_forward_pool): row i through snapshot
choice[i] of K packed actors, rows grouped on the device.  Every written row must equal the single-actor kernel
(FusedActor) of its snapshot bit for bit -- a row's result depends only on its own observation and its weights -- and
every skipped row must be untouched.  Above it: FusedActorPool, OpponentPool's fused snapshot path and cross_play."""
import ctypes
import math
import os

import pytest

torch = pytest.importorskip("torch")

NPZ = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "td3_actors.npz")
P = 256 * 24 * 4 + 256 * 256 * 2 + 16 * 256 * 2 + 2 * 256 * 4 + 16 * 4  # bytes of one packed actor


def _a4(words):
    return (words + 3) // 4 * 4


def _actors(k, device):
    """The two reference checkpoints, then seeded perturbations of them: k distinct actors."""
    from hockey_env_b200.actor import load_td3_actor
    base = [load_td3_actor(NPZ, device=device, name=nm) for nm in ("stage_3", "competition")]
    out = base[:k]
    g = torch.Generator().manual_seed(1234)
    while len(out) < k:
        a = load_td3_actor(NPZ, device=device, name=("stage_3", "competition")[len(out) % 2])
        with torch.no_grad():
            for p in a.parameters():
                p.add_((0.05 * torch.randn(p.shape, generator=g)).to(p.device))
        out.append(a)
    return out


def _obs(n, seed, device="cuda:0"):
    g = torch.Generator(device=device).manual_seed(seed)
    scale = torch.tensor([2, 2, .5, 4, 4, 3, 2, 2, .5, 4, 4, 3, 3, 2, 8, 8, 4, 4], device=device)
    return torch.randn((n, 18), device=device, generator=g) * scale


# ---- CPU ------------------------------------------------------------------------------------------------------------

def test_scratch_bytes_formula():
    import hockey_env_b200 as hk
    L = hk.load_library()
    for n, k in ((1, 1), (127, 3), (100_003, 16), (262_144, 4096), (2**31 - 1, 7)):
        words = _a4(k) + _a4(k + 1) + _a4(k + 1) + _a4(k) + _a4(n)  # counts | group offsets | tile offsets | cursors | rows
        assert L.hk_actor_pool_scratch_bytes(n, k) == 4 * words
    for n, k in ((0, 1), (-5, 1), (2**31, 1), (10, 0), (10, -1), (10, 4097)):
        assert L.hk_actor_pool_scratch_bytes(n, k) == hk._lib.HK_E_INVALID
        assert b"hk_actor_pool_scratch_bytes" in L.hk_last_error()


def test_pool_error_convention_without_gpu():
    import hockey_env_b200 as hk
    L = hk.load_library()
    INV = hk._lib.HK_E_INVALID
    A = 0x10000  # an aligned address: every call below is rejected before anything is read through it

    def call(params=A, k=2, choice=A, obs=A, act=A, stride=4, n=100, scratch=A, device=0):
        return L.hk_actor_forward_pool(params, k, choice, obs, act, stride, n, scratch, device, None)

    cases = [(dict(params=None), b"NULL"), (dict(choice=None), b"NULL"), (dict(obs=None), b"NULL"), (dict(act=None), b"NULL"),
             (dict(scratch=None), b"NULL"), (dict(n=0), b"n must be"), (dict(n=-3), b"n must be"), (dict(n=2**31), b"n must be"),
             (dict(stride=3), b"act_stride"), (dict(k=0), b"k must be"), (dict(k=4097), b"k must be"),
             (dict(params=A + 8), b"alignment"), (dict(obs=A + 4), b"alignment"), (dict(choice=A + 2), b"alignment"),
             (dict(scratch=A + 4), b"alignment")]
    for kw, msg in cases:
        assert call(**kw) == INV, kw
        err = L.hk_last_error()
        assert b"hk_actor_forward_pool" in err and msg in err, (kw, err)
    if not torch.cuda.is_available():
        assert call() == hk._lib.HK_E_NODEVICE
        assert b"no CUDA device" in L.hk_last_error()
        with pytest.raises(hk.HockeyLibraryError):
            hk.FusedActorPool([])


def test_pool_table_is_the_concatenated_blocks():
    import hockey_env_b200 as hk
    from hockey_env_b200.actor import FusedActor, FusedActorPool
    assert FusedActor.PARAM_BYTES == P == hk.load_library().hk_actor_param_bytes()
    actors = _actors(3, "cpu")
    table = FusedActorPool.pack(actors)
    assert table.dtype == torch.uint8 and tuple(table.shape) == (3, P)
    flat = table.flatten()
    for s, a in enumerate(actors):  # snapshot s starts at byte s * hk_actor_param_bytes()
        blk = FusedActor.pack({k: v.float() for k, v in a.state_dict().items()})
        assert torch.equal(flat[s * P:(s + 1) * P], blk)
    assert tuple(FusedActorPool.pack([]).shape) == (0, P)
    bad = torch.nn.Sequential()
    bad.fc1, bad.fc2, bad.fc3 = torch.nn.Linear(18, 64), torch.nn.Linear(64, 64), torch.nn.Linear(64, 4)
    with pytest.raises(ValueError, match="18 -> 256 -> 256 -> 4"):
        FusedActorPool.pack([bad])


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _expected(fused, obs, choice, base):
    """What the pool must produce: row i = FusedActor(snapshot choice[i])(obs)[i], other rows = base."""
    want = base.clone()
    for s, f in enumerate(fused):
        m = choice == s
        want[m] = f(obs)[m]
    return want


def _mismatch_report(got, want):
    bad = (got != want).any(1).nonzero().flatten()
    return f"{bad.numel()} rows differ, first {bad[:8].tolist()}: got {got[bad[:4]].tolist()} want {want[bad[:4]].tolist()}"


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 16])
@pytest.mark.parametrize("n", [1, 127, 128, 129, 4096, 100_003])
def test_pool_matches_fused_actor_bit_for_bit(n, k):
    import hockey_env_b200 as hk
    actors = _actors(k, "cuda:0")
    fused = [hk.FusedActor(a) for a in actors]
    pool = hk.FusedActorPool(actors)
    assert len(pool) == k
    obs = _obs(n, 100 + n)
    g = torch.Generator(device="cuda:0").manual_seed(n * 31 + k)
    # snapshots, skipped rows (-1, large negative, >= K) and, for K >= 3, an empty group (snapshot 1)
    choice = torch.randint(-1, k + 2, (n,), device="cuda:0", generator=g, dtype=torch.int64)
    choice[torch.rand(n, device="cuda:0", generator=g) < 0.05] = -(2**40)
    if k >= 3:
        choice[choice == 1] = 2
    for dtype in (torch.int64, torch.int32):  # as int32, -2^40 wraps to 0: those rows then choose snapshot 0
        c = choice.to(dtype)
        out = torch.full((n, 4), 7.0, device="cuda:0")
        got = pool(obs, c, out=out)
        want = _expected(fused, obs, c.long(), torch.full((n, 4), 7.0, device="cuda:0"))
        torch.cuda.synchronize()
        assert torch.equal(got, want), _mismatch_report(got, want)
    # out=None: the persistent buffer, skipped rows zero -- also after a call that wrote them
    pool(obs, torch.zeros(n, dtype=torch.int32, device="cuda:0"))
    got = pool(obs, choice)
    assert torch.equal(got, _expected(fused, obs, choice, torch.zeros((n, 4), device="cuda:0")))
    if k == 1:  # every row chosen: the whole batch of hk_actor_forward
        assert torch.equal(pool(obs, torch.zeros(n, dtype=torch.int32, device="cuda:0")), fused[0](obs))


@pytest.mark.gpu
def test_pool_writes_into_out_views():
    import hockey_env_b200 as hk
    actors = _actors(2, "cuda:0")
    fused = [hk.FusedActor(a) for a in actors]
    pool = hk.FusedActorPool()
    assert len(pool) == 0 and pool.add(actors[0]) == 0 and pool.add(actors[1]) == 1 and len(pool) == 2
    n = 5000
    obs = _obs(n, 7)
    choice = (torch.arange(n, device="cuda:0") % 3 - 1).to(torch.int32)  # -1, 0, 1, ...
    a8 = torch.full((n, 8), 3.0, device="cuda:0")
    got = pool(obs, choice, out=a8[:, 4:])
    assert got.data_ptr() == a8[:, 4:].data_ptr()
    assert (a8[:, :4] == 3.0).all()
    assert torch.equal(a8[:, 4:], _expected(fused, obs, choice.long(), torch.full((n, 4), 3.0, device="cuda:0")))


@pytest.mark.gpu
def test_pool_call_is_graph_capturable():
    """The grouping runs on the device: a captured call follows a choice tensor rewritten in place."""
    import hockey_env_b200 as hk
    actors = _actors(3, "cuda:0")
    fused = [hk.FusedActor(a) for a in actors]
    pool = hk.FusedActorPool(actors)
    n = 20_000
    obs = _obs(n, 11)
    choice = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    out = torch.zeros((n, 4), device="cuda:0")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pool(obs, choice, out=out)  # warm-up: scratch allocated, kernel attributes set
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        pool(obs, choice, out=out)
    for seed in (1, 2):
        g = torch.Generator(device="cuda:0").manual_seed(seed)
        choice.copy_(torch.randint(-1, 4, (n,), device="cuda:0", generator=g, dtype=torch.int32))
        out.fill_(5.0)
        graph.replay()
        torch.cuda.synchronize()
        want = _expected(fused, obs, choice.long(), torch.full((n, 4), 5.0, device="cuda:0"))
        assert torch.equal(out, want), _mismatch_report(out, want)


@pytest.mark.gpu
def test_opponent_pool_fused_path_matches_module_list():
    """The same self-play run with snapshots as a list of FusedActor and as one FusedActorPool ends in the same state."""
    import hockey_env_b200 as hk
    a, b = _actors(2, "cuda:0")
    p1 = hk.FusedActor(a)
    results = []
    for snaps in ([hk.FusedActor(a), hk.FusedActor(b)], hk.FusedActorPool([a, b])):
        env = hk.HockeyVecEnv(4096, device="cuda:0", seed=21, p2="per_env")
        pool = hk.OpponentPool(env, p_weak=0.2, p_strong=0.2, snapshots=snaps, p_snapshot=0.6, seed=3)
        obs = env.obs
        for _ in range(300):
            obs, *_ = pool.step(p1(obs))
        torch.cuda.synchronize()
        results.append((env.get_full_state().cpu(), env.stats(), pool.choice.cpu()))
        assert int(((pool.choice >= 2)).sum()) > 0
    (s0, st0, c0), (s1, st1, c1) = results
    assert torch.equal(c0, c1)
    assert torch.equal(s0, s1)
    # the counters are exact; the float64 return sums are accumulated with atomics, so their last bits follow the
    # order in which blocks flush (two runs of the same path differ there too)
    assert st0.keys() == st1.keys()
    for key in st0:
        if key.startswith("sum_return"):
            assert st0[key] == pytest.approx(st1[key], rel=1e-12, abs=1e-9), key
        else:
            assert st0[key] == st1[key], key


def _binom_sd(p, m):
    return math.sqrt(max(p * (1 - p), 1e-4) / max(m, 1))


@pytest.mark.gpu
def test_cross_play_league_table():
    import hockey_env_b200 as hk
    s3, comp = _actors(2, "cuda:0")
    num_envs, per_pair_eps = 4096, 2048
    for actors in ([s3, s3], [s3, comp]):
        r = hk.cross_play(actors, episodes_per_pair=per_pair_eps, num_envs=num_envs, seed=5)
        k = len(actors)
        per_pair = num_envs // (k * k)
        total = r["win_rate"] + r["draw_rate"] + r["loss_rate"]
        assert torch.allclose(total, torch.ones_like(total), atol=1e-12), total
        # every env filled its quota: exactly quota * envs episodes per pair were counted
        assert (r["episodes"] == r["episodes_per_env"] * per_pair).all() and r["episodes_per_env"] * per_pair >= per_pair_eps
        W, L, E = r["win_rate"].cpu(), r["loss_rate"].cpu(), r["episodes"].cpu()
        print("win", W.tolist(), "draw", r["draw_rate"].tolist(), "loss", L.tolist(), "ret", r["mean_return"].tolist())
        if actors[0] is actors[1]:
            for i in range(k):
                for j in range(k):  # the same policy on both sides: wins and losses agree
                    w, l, m = float(W[i, j]), float(L[i, j]), float(E[i, j])
                    sd = math.sqrt(max(w + l - (w - l) ** 2, 1e-4) / m)
                    assert abs(w - l) <= 4.5 * sd, (i, j, w, l, m)
        else:
            for i in range(k):
                for j in range(k):  # i beats j as player 1 as often as j loses to i with the sides swapped
                    w, l = float(W[i, j]), float(L[j, i])
                    sd = math.hypot(_binom_sd(w, float(E[i, j])), _binom_sd(l, float(E[j, i])))
                    assert abs(w - l) <= 4.5 * sd, (i, j, w, l)
