"""The fused actor kernel (csrc/hk_actor.cuh, hk_actor_forward) layer by layer, against exact probes and against a float64
reference that rounds its operands the way the kernel does.

test_actor_kernel.py compares the kernel with the fp32 module, whose differences from the kernel (TF32 / bf16 operands)
reach ~0.3 on single outputs of a trained policy: bounds that wide cannot see a rounding-mode slip, one misplaced
weight or a wrong output bias.  Here:

* `reference` models every operand rounding of the kernel, so what is left between the two is the tensor core's fp32
  accumulation order and tanh.approx.f32: small enough that per-weight-set bounds on max / RMS / mean error catch
  truncation in place of rounding and a shifted output bias (`check_realistic`).
* three probes isolate one layer each, with every other layer's arithmetic exact (saturated +-1 activations, dyadic
  weights), so a single misplaced element, bias or row moves an output by far more than the tolerance
  (`check_w3_probe`, `check_w2_probe`, `check_w1_probe`).  The W3 probe measures the tanh.approx error on the device.
* a probe tells apart how the tensor core consumes the raw f32 bits of W1 under kind::tf32 (`check_w1_operand`).
* every check also runs on the CPU with the reference standing in for the kernel, once plainly (it must pass) and once
  with a planted mistake (it must fail): `test_checks_have_teeth`.
"""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

NPZ = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "td3_actors.npz")

# The PTX ISA (Floating Point Instructions: tanh) bounds the relative error of tanh.approx.f32 by 2^-10.987.  Every
# tolerance below is built from this bound, not from the error a B200 shows (2^-16.6 at most on the W3 probe).
TANH_APPROX_REL = 2.0 ** -10.987

# How kind::tf32 consumes the raw f32 bits FusedActor.pack stores for W1, as test_w1_operand_probe measured it on a B200:
# the low 13 significand bits are dropped (truncation toward zero), not rounded.
W1_OPERAND = "truncate"


# ---- operand roundings ------------------------------------------------------------------------------------------------

def _f32_bits(x):
    return x.to(torch.float32).view(torch.int32)


def _from_bits(i):
    return i.view(torch.float32).to(torch.float64)


def tf32_rna(x):
    """cvt.rna.tf32.f32 of finite values: nearest, ties away from zero, to 10 fraction bits.  On sign-magnitude bits,
    adding half an ulp to the pattern and clearing the low 13 bits rounds the magnitude half away from zero."""
    return _from_bits((_f32_bits(x) + 0x1000) & ~0x1FFF)


def tf32_rne(x):
    i = _f32_bits(x)
    return _from_bits((i + 0xFFF + ((i >> 13) & 1)) & ~0x1FFF)


def tf32_trunc(x):
    return _from_bits(_f32_bits(x) & ~0x1FFF)


def bf16_rne(x):
    return x.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def bf16_trunc(x):
    return _from_bits(_f32_bits(x) & ~0xFFFF)


W1_OPERANDS = {"truncate": tf32_trunc, "rne": tf32_rne, "rna": tf32_rna, "fp32": lambda x: x.to(torch.float32).to(torch.float64)}


def _f32(x):
    return x.to(torch.float32).to(torch.float64)


def reference(sd, obs, w1=None, act=bf16_rne, wq=bf16_rne, full=False):
    """The kernel's forward pass in float64 with the kernel's operand roundings:
        obs  -> TF32 (cvt.rna: nearest, ties away);   W1 -> the tensor core's kind::tf32 reading of f32 bits (W1_OPERAND);
        W2, W3 and both hidden activations -> bf16 round to nearest even (the pack and the epilogue's cvt.rn.bf16x2);
        each layer's accumulator rounded to fp32, then the fp32 bias add;
        float64 matrix products and exact tanh.
    Not modelled: the order in which the tensor core accumulates in fp32, and the error of tanh.approx.f32.
    `w1` / `act` / `wq` override the roundings (the probes' candidates and the planted mistakes); full=True returns the
    intermediates too."""
    p = {k: v.to(torch.float64) for k, v in sd.items()}
    x = tf32_rna(obs.to(torch.float64))
    z1 = _f32(_f32(x @ W1_OPERANDS[w1 or W1_OPERAND](p["fc1.weight"]).T) + _f32(p["fc1.bias"]))
    t1 = torch.tanh(z1)
    h1 = act(t1)
    z2 = _f32(_f32(h1 @ wq(p["fc2.weight"]).T) + _f32(p["fc2.bias"]))
    t2 = torch.tanh(z2)
    h2 = act(t2)
    z3 = _f32(_f32(h2 @ wq(p["fc3.weight"]).T) + _f32(p["fc3.bias"]))
    out = torch.tanh(z3)
    return dict(z1=z1, t1=t1, h1=h1, z2=z2, t2=t2, h2=h2, z3=z3, out=out) if full else out


def _bf16_ulp(a):
    """The bf16 spacing at magnitude a (7 fraction bits): one rounding of a value near a, or two roundings of values
    within it of each other, differ by at most this much."""
    a = a.abs().clamp_min(2.0 ** -120)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


# ---- weights, observations, forward passes ---------------------------------------------------------------------------

def _sd(w1, b1, w2, b2, w3, b3):
    t = dict(zip(("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias"), (w1, b1, w2, b2, w3, b3)))
    return {k: v.to(torch.float32).contiguous() for k, v in t.items()}


def weight_set(name):
    """stage_3 / competition: the trained policies; default_init: a seeded ActorNetwork as training starts it;
    default_init_x3: those weights x3, which saturates most hidden units."""
    from hockey_env_b200.actor import ActorNetwork, load_td3_actor
    if name in ("stage_3", "competition"):
        return {k: v.float() for k, v in load_td3_actor(NPZ, device="cpu", name=name).state_dict().items()}
    with torch.random.fork_rng():
        torch.manual_seed(1234)
        sd = {k: v.detach().float() for k, v in ActorNetwork().state_dict().items()}
    return {k: v * 3 for k, v in sd.items()} if name == "default_init_x3" else sd


WEIGHT_SETS = ("stage_3", "competition", "default_init", "default_init_x3")
_OBS_SCALE = torch.tensor([2, 2, .5, 4, 4, 3, 2, 2, .5, 4, 4, 3, 3, 2, 8, 8, 4, 4], dtype=torch.float32)


def realistic_obs(n, n_wide, seed):
    """n rows of test_actor_kernel.py's observation distribution (positions +-4, velocities +-10, angles, timers), then
    n_wide rows uniform in [-30, 30]."""
    g = torch.Generator().manual_seed(seed)
    return torch.cat([torch.randn((n, 18), generator=g) * _OBS_SCALE, (torch.rand((n_wide, 18), generator=g) * 2 - 1) * 30])


def _signs(shape, g):
    return torch.randint(0, 2, shape, generator=g).to(torch.float64) * 2 - 1


def _dyadic(shape, lo, hi, g):
    """+-m * 2^-10 with m uniform in [lo, hi]: bf16-exact for hi < 256, and sums of a few hundred stay exact in fp32."""
    return _signs(shape, g) * torch.randint(lo, hi + 1, shape, generator=g).to(torch.float64) * 2.0 ** -10


def kernel_forward(sd, obs):
    """hk_actor_forward of the FusedActor packed from `sd` (through FusedActor.pack, as every caller packs)."""
    import hockey_env_b200 as hk
    net = hk.ActorNetwork()
    net.load_state_dict(sd)
    out = hk.FusedActor(net)(obs.to(torch.float32).contiguous().cuda())
    return out.to(torch.float64).cpu()


def reference_forward(sd, obs):
    """The reference with exact tanh in place of the kernel: every check must pass it (see test_checks_have_teeth)."""
    return reference(sd, obs)


# ---- probe: how kind::tf32 reads W1 ----------------------------------------------------------------------------------
# Hidden unit u gets W1[u, 0] = a_u, W1[u, 1] = b_u = -+1 and obs[0] = obs[1] = 2^8, so z1_u = 2^8 (q(a_u) - 1) is exact
# for every reading q of a_u, and W2 / W3 one-hot carry unit u to output u.  a_0 separates truncation from rounding,
# a_1 (a tie above an even neighbour) ties away from ties to even, a_2 is a_0 negated (truncation toward zero vs
# toward -inf), a_3 is a tie above an odd neighbour.  z1 per reading (truncate, rne, rna, fp32):
#   u0: 0, .25, .25, .15625   u1: 0, 0, .25, .125   u2: 0, -.25, -.25, -.15625   u3: .25, .5, .5, .375
W1_PROBE = ((1 + 2 ** -11 + 2 ** -13, -1.0), (1 + 2 ** -11, -1.0), (-(1 + 2 ** -11 + 2 ** -13), 1.0), (1 + 2 ** -10 + 2 ** -11, -1.0))


def w1_operand_probe():
    w1 = torch.zeros(256, 18, dtype=torch.float64)
    for u, (a, b) in enumerate(W1_PROBE):
        w1[u, 0], w1[u, 1] = a, b
    w2 = torch.zeros(256, 256, dtype=torch.float64)
    w2[:4, :4] = torch.eye(4)
    w3 = torch.zeros(4, 256, dtype=torch.float64)
    w3[:, :4] = torch.eye(4)
    obs = torch.zeros(128, 18)
    obs[:, :2] = 2.0 ** 8
    return _sd(w1, torch.zeros(256), w2, torch.zeros(256), w3, torch.zeros(4)), obs


def check_w1_operand(forward):
    """The readings of W1 whose prediction the output matches (to 4e-3; the candidates are >= 0.1 apart)."""
    sd, obs = w1_operand_probe()
    got = forward(sd, obs)
    return [m for m in W1_OPERANDS if (got - reference(sd, obs, w1=m)).abs().max().item() <= 4e-3]


# ---- probe: W3 / b3, and the tanh.approx error -----------------------------------------------------------------------
# obs in {+-1} on columns 0..16 and W1 = +-16 there: |z1| = 16 |odd sum| >= 16, h1 = +-1 exactly.  Each W2 row has three
# +-8 entries: |z2| >= 8, h2 = +-1 exactly (bf16 rounds tanh(8) to 1).  W3 and b3 are multiples of 2^-10 below 2^-2,
# so z3 = W3 h2 + b3 is exact in fp32 in any order, spread over about [-6, 6], and the output must be tanh.approx(z3).

def w3_probe(n=4096, seed=31):
    g = torch.Generator().manual_seed(seed)
    w1 = torch.zeros(256, 18, dtype=torch.float64)
    w1[:, :17] = 16 * _signs((256, 17), g)
    w2 = torch.zeros(256, 256, dtype=torch.float64)
    for j in range(256):
        w2[j, torch.randperm(256, generator=g)[:3]] = 8 * _signs((3,), g)
    w3 = _dyadic((4, 256), 16, 255, g)
    b3 = _dyadic((4,), 0, 255, g)
    obs = torch.zeros(n, 18)
    obs[:, :17] = _signs((n, 17), g).float()
    return _sd(w1, torch.zeros(256), w2, torch.zeros(256), w3, b3), obs


def _w3_probe_z3(sd, obs):
    p = {k: v.to(torch.float64) for k, v in sd.items()}
    h1 = torch.sign(obs.to(torch.float64) @ p["fc1.weight"].T)
    h2 = torch.sign(h1 @ p["fc2.weight"].T)
    return h2 @ p["fc3.weight"].T + p["fc3.bias"]


def check_w3_probe(forward):
    """Returns the largest relative error of the outputs against tanh(z3); asserts it within the PTX ISA's bound."""
    sd, obs = w3_probe()
    want = torch.tanh(_w3_probe_z3(sd, obs))
    got = forward(sd, obs)
    assert torch.equal(got == 0, want == 0), "tanh(+-0) must be +-0"
    rel = ((got - want).abs() / want.abs().clamp_min(1e-300))[want != 0]
    assert rel.max().item() <= TANH_APPROX_REL, (rel.max().item(), TANH_APPROX_REL)
    return rel.max().item()


# Large |z3|: W3 = 0, b3 = z, so the four outputs are tanh.approx(z) directly.
TANH_SATURATED = ((10.0, 16.0, 1e30, float("inf")), (-10.0, -16.0, -1e30, float("-inf")))


def check_tanh_saturates(forward):
    """The fp32 outputs are exactly +-1 (tanh(10) is 1 - 4e-9: 1.0 in fp32)."""
    for z in TANH_SATURATED:
        sd, obs = w3_probe(n=128)
        sd["fc3.weight"] = torch.zeros(4, 256)
        sd["fc3.bias"] = torch.tensor(z, dtype=torch.float32)
        got = forward(sd, obs).to(torch.float32)
        assert torch.equal(got, torch.tensor(z).sign().expand(128, 4)), (z, got[0].tolist())


# ---- probe: W2 / b2 --------------------------------------------------------------------------------------------------
# h1 = sign(16 R obs) is an exact +-1 pattern per row, different for every unit.  W2 and b2 are multiples of 2^-10 with
# |W2| in [2^-5, 2^-4] and |b2| in [2^-5, 2^-2]: bf16-exact, and z2 = W2 h1 + b2 is exact in fp32 in any order, so a
# zeroed or misplaced element moves some z2 by >= 2^-5.  W3 is one-hot on 4 layer-2 units per launch, b3 = 0, so the
# outputs are tanh.approx(bf16(tanh.approx(z2))) of those units; 64 launches (repacks) cover all 256.

W2_PROBE_ROWS = 300


def w2_probe(seed=32):
    g = torch.Generator().manual_seed(seed)
    w1 = torch.zeros(256, 18, dtype=torch.float64)
    w1[:, :17] = 16 * _signs((256, 17), g)
    w2 = _dyadic((256, 256), 32, 64, g)
    b2 = _dyadic((256,), 32, 256, g)
    obs = torch.zeros(W2_PROBE_ROWS, 18)
    obs[:, :17] = _signs((W2_PROBE_ROWS, 17), g).float()
    return _sd(w1, torch.zeros(256), w2, b2, torch.zeros(4, 256), torch.zeros(4)), obs


def _one_hot_w3(units):
    w3 = torch.zeros(4, 256)
    w3[torch.arange(4), torch.as_tensor(units)] = 1.0
    return w3


def _chain_tol(tol, t):
    """Bound on |kernel - reference| after one epilogue (tanh, then bf16) when the inputs differ by `tol`: the tanh.approx
    error, then one bf16 spacing for a rounding that may fall either side; t is the reference's tanh."""
    return tol + TANH_APPROX_REL * t.abs() + _bf16_ulp(t.abs() + tol + TANH_APPROX_REL)


def check_w2_probe(forward):
    """Returns the largest |kernel - expected| / tolerance over all 256 layer-2 units; asserts it <= 1."""
    sd, obs = w2_probe()
    p = {k: v.to(torch.float64) for k, v in sd.items()}
    h1 = torch.sign(obs.to(torch.float64) @ p["fc1.weight"].T)
    z2 = h1 @ p["fc2.weight"].T + p["fc2.bias"]
    worst = 0.0
    for blk in range(64):
        units = list(range(4 * blk, 4 * blk + 4))
        t2 = torch.tanh(z2[:, units])
        want = torch.tanh(bf16_rne(t2))
        tol = _chain_tol(torch.zeros_like(t2), t2) + TANH_APPROX_REL * want.abs()
        got = forward(dict(sd, **{"fc3.weight": _one_hot_w3(units)}), obs)
        excess = ((got - want).abs() / tol).max().item()
        assert excess <= 1.0, (units, excess)
        worst = max(worst, excess)
    return worst


# ---- probe: W1 / b1 --------------------------------------------------------------------------------------------------
# Realistic W1, b1 (stage_3) and observations; W2 a permutation (h2_j = bf16(tanh.approx(h1_perm(j))), exact: one
# product of 1.0, b2 = 0) and W3 one-hot on 4 units per launch.  Expected: the reference's tanh o bf16 o tanh o bf16 o
# tanh; the tolerance carries the fp32 accumulation of layer 1, E and one bf16 spacing per rounding through the chain.

W1_PROBE_ROWS = 300


def w1_probe(seed=33):
    g = torch.Generator().manual_seed(seed)
    base = weight_set("stage_3")
    perm = torch.randperm(256, generator=g)
    w2 = torch.zeros(256, 256, dtype=torch.float64)
    w2[torch.arange(256), perm] = 1.0
    obs = realistic_obs(W1_PROBE_ROWS - 44, 44, seed)
    return _sd(base["fc1.weight"], base["fc1.bias"], w2, torch.zeros(256), torch.zeros(4, 256), torch.zeros(4)), obs


def check_w1_probe(forward):
    """Returns the largest |kernel - expected| / tolerance over all 256 layer-1 units; asserts it <= 1."""
    sd, obs = w1_probe()
    r = reference(sd, obs, full=True)
    x = tf32_rna(obs.to(torch.float64))
    w1 = W1_OPERANDS[W1_OPERAND](sd["fc1.weight"].to(torch.float64))
    # fp32 accumulation in any order of 18 products and the bias: a few ulps of the largest partial sum, generously
    acc = 2.0 ** -20 * ((x.abs() @ w1.abs().T) + sd["fc1.bias"].to(torch.float64).abs())
    tol1 = _chain_tol(acc, r["t1"])
    worst = 0.0
    for blk in range(64):
        units = list(range(4 * blk, 4 * blk + 4))
        src = sd["fc2.weight"][units].argmax(dim=1)          # the layer-1 unit each read-out layer-2 unit copies
        t2 = torch.tanh(r["h1"][:, src])
        want = torch.tanh(bf16_rne(t2))
        tol = _chain_tol(tol1[:, src], t2) + TANH_APPROX_REL * want.abs()
        got = forward(dict(sd, **{"fc3.weight": _one_hot_w3(units)}), obs)
        excess = ((got - want).abs() / tol).max().item()
        assert excess <= 1.0, (units, excess)
        worst = max(worst, excess)
    return worst


# ---- realistic weights -----------------------------------------------------------------------------------------------
# Kernel minus reference per weight set over `realistic_inputs`: max |err|, RMS and mean signed error.  Bounds: what one
# B200 (148 SMs) measured, with a margin of 1.5x on max and RMS and 2x on |mean|, floored at 1e-5:
#   stage_3          max 3.004e-2  rms 3.543e-4  mean +2.8e-7
#   competition      max 2.216e-2  rms 3.328e-4  mean -7.6e-7
#   default_init     max 1.019e-3  rms 7.092e-5  mean +4.8e-8
#   default_init_x3  max 5.931e-3  rms 1.591e-4  mean -5.0e-7
# The reference with a planted mistake (exact tanh) exceeds every set's bounds: bf16 truncation in place of rounding
# gives 16x-53x the measured RMS, b3 += 0.02 a mean above 1e-3, one row with its neighbour's observation a max above 0.4.

REALISTIC_BOUNDS = {
    #                  max      rms      |mean|
    "stage_3":         (4.5e-2, 5.3e-4, 1e-5),
    "competition":     (3.3e-2, 5.0e-4, 1e-5),
    "default_init":    (1.5e-3, 1.1e-4, 1e-5),
    "default_init_x3": (8.9e-3, 2.4e-4, 1e-5),
}


def realistic_inputs():
    return realistic_obs(16384, 4096, seed=34)


def error_stats(got, want):
    d = got - want
    return dict(max=d.abs().max().item(), rms=d.pow(2).mean().sqrt().item(), mean=d.mean().item())


def realistic_errors(forward):
    """{weight set: stats} and the weight sets whose stats exceed REALISTIC_BOUNDS."""
    obs = realistic_inputs()
    stats, bad = {}, []
    for name in WEIGHT_SETS:
        s = stats[name] = error_stats(forward(weight_set(name), obs), _realistic_reference(name))
        bmax, brms, bmean = REALISTIC_BOUNDS[name]
        if not (s["max"] <= bmax and s["rms"] <= brms and abs(s["mean"]) <= bmean):
            bad.append(name)
    return stats, bad


def check_realistic(forward):
    """Returns {weight set: stats}; asserts every statistic within REALISTIC_BOUNDS."""
    stats, bad = realistic_errors(forward)
    assert not bad, {name: stats[name] for name in bad}
    return stats


_REF_CACHE = {}


def _realistic_reference(name):
    if name not in _REF_CACHE:
        _REF_CACHE[name] = reference(weight_set(name), realistic_inputs())
    return _REF_CACHE[name]


# ---- CPU: the probes' preconditions ----------------------------------------------------------------------------------

def _exact_bf16(t):
    return torch.equal(bf16_rne(t.to(torch.float64)), t.to(torch.float64))


def _exact_tf32(t):
    return all(torch.equal(f(t.to(torch.float64)), t.to(torch.float64)) for f in (tf32_trunc, tf32_rna))


def _fp32_sums_exact(terms, total):
    """Every partial sum of `terms` ([rows, k]), in any order, is exact in fp32, and the sum is `total`: the terms are
    multiples of 2^-10 whose magnitudes sum below 2^14, so every partial sum is a multiple of 2^-10 below 2^14 in
    magnitude, which a 24-bit significand holds."""
    m = terms * 1024
    c = terms.cumsum(-1)
    return (torch.equal(m, m.round()) and bool((terms.abs().sum(-1) < 2 ** 14).all()) and torch.equal(_f32(c), c)
            and torch.equal(c[..., -1], total))


def test_w1_operand_probe_separates_the_readings():
    sd, obs = w1_operand_probe()
    assert _exact_tf32(obs) and _exact_bf16(sd["fc2.weight"]) and _exact_bf16(sd["fc3.weight"])
    outs = {m: reference(sd, obs, w1=m) for m in W1_OPERANDS}
    for a in outs:
        for b in outs:
            if a < b:
                assert (outs[a] - outs[b]).abs().max().item() >= 0.1, (a, b)
    assert check_w1_operand(reference_forward) == [W1_OPERAND]


def test_w3_probe_preconditions():
    sd, obs = w3_probe()
    p = {k: v.to(torch.float64) for k, v in sd.items()}
    x = obs.to(torch.float64)
    assert _exact_tf32(x) and _exact_tf32(p["fc1.weight"])
    for k in ("fc2.weight", "fc3.weight", "fc3.bias"):
        assert _exact_bf16(p[k]), k
    z1 = x @ p["fc1.weight"].T
    assert z1.abs().min().item() >= 16                      # h1 = +-1: tanh(16) is 1 in fp32 and in bf16
    h1 = torch.sign(z1)
    z2 = h1 @ p["fc2.weight"].T
    assert z2.abs().min().item() >= 8                       # h2 = +-1: bf16 rounds tanh(8) to 1
    assert bf16_rne(torch.tanh(torch.tensor(8.0, dtype=torch.float64)) * (1 - TANH_APPROX_REL)).item() == 1.0
    h2 = torch.sign(z2)
    z3 = _w3_probe_z3(sd, obs)
    for i in range(4):
        assert _fp32_sums_exact(torch.cat([h2 * p["fc3.weight"][i], p["fc3.bias"][i].expand(len(x), 1)], 1), z3[:, i])
    assert z3.min().item() < -5 and z3.max().item() > 5, (z3.min().item(), z3.max().item())
    assert (z3.abs() < 0.5).sum().item() >= 100            # enough rows where a shifted z3 is visible at the output
    assert p["fc3.weight"].abs().min().item() >= 2.0 ** -6
    assert torch.equal(reference(sd, obs), torch.tanh(z3))  # the reference agrees: every rounding on this probe is exact


def test_w2_probe_preconditions():
    sd, obs = w2_probe()
    p = {k: v.to(torch.float64) for k, v in sd.items()}
    x = obs.to(torch.float64)
    assert _exact_tf32(x) and _exact_tf32(p["fc1.weight"])
    assert _exact_bf16(p["fc2.weight"]) and _exact_bf16(p["fc2.bias"])
    assert p["fc2.weight"].abs().max().item() <= 2.0 ** -4
    assert p["fc2.weight"].abs().min().item() >= 2.0 ** -5 and p["fc2.bias"].abs().min().item() >= 2.0 ** -5
    z1 = x @ p["fc1.weight"].T
    assert z1.abs().min().item() >= 16
    h1 = torch.sign(z1)
    # the 256 units' sign patterns over the rows are pairwise distinct (and no unit is constant)
    cols = {tuple(h1[:, j].tolist()) for j in range(256)}
    assert len(cols) == 256 and all(len(set(c)) == 2 for c in cols)
    z2 = h1 @ p["fc2.weight"].T + p["fc2.bias"]
    for j in range(0, 256, 5):
        assert _fp32_sums_exact(torch.cat([h1 * p["fc2.weight"][j], p["fc2.bias"][j].expand(len(x), 1)], 1), z2[:, j])
    # every unit has rows where its z2 is in tanh's steep part, so a shift of 2^-5 there is visible
    assert ((z2.abs() < 0.75).sum(0) >= 20).all()
    r = reference(dict(sd, **{"fc3.weight": _one_hot_w3([0, 1, 2, 3])}), obs, full=True)
    assert torch.equal(r["z2"], z2) and torch.equal(r["h1"], h1)


def test_w1_probe_preconditions():
    sd, obs = w1_probe()
    w2 = sd["fc2.weight"]
    assert torch.equal(w2.sum(0), torch.ones(256)) and torch.equal(w2.sum(1), torch.ones(256)) and _exact_bf16(w2)
    r = reference(dict(sd, **{"fc3.weight": _one_hot_w3([0, 1, 2, 3])}), obs, full=True)
    assert torch.equal(r["z2"], r["h1"][:, w2.argmax(1)])  # layer 2 copies layer-1 activations exactly
    # every layer-1 unit is off saturation on some rows, where its W1 row and b1 entry show at the output
    assert ((r["t1"].abs() < 0.9).sum(0) >= 10).all()


# ---- CPU: every check fails on a planted mistake ---------------------------------------------------------------------

def _obs_from_neighbour(obs, row=127):
    o = obs.clone()
    o[row] = obs[row - 1]
    return o


def _zero(key, idx):
    def f(sd):
        t = sd[key].clone()
        t[idx] = 0.0
        return dict(sd, **{key: t})
    return f


def _add(key, v):
    return lambda sd: dict(sd, **{key: sd[key] + v})


# name: (the reference with the mistake, the checks that must fail)
MUTANTS = {
    "act_bf16_truncated": (lambda sd, obs: reference(sd, obs, act=bf16_trunc), ("realistic",)),
    "weights_bf16_truncated": (lambda sd, obs: reference(sd, obs, wq=bf16_trunc), ("realistic",)),
    "b3_plus_0.02": (lambda sd, obs: reference(_add("fc3.bias", 0.02)(sd), obs), ("realistic", "w3")),
    "w2_element_zeroed": (lambda sd, obs: reference(_zero("fc2.weight", (255, 255))(sd), obs), ("w2",)),
    "b2_entry_zeroed": (lambda sd, obs: reference(_zero("fc2.bias", 200)(sd), obs), ("w2",)),
    "row_takes_neighbour_obs": (lambda sd, obs: reference(sd, _obs_from_neighbour(obs)), ("realistic", "w1", "w2", "w3")),
    "w1_element_zeroed": (lambda sd, obs: reference(_zero("fc1.weight", (77, 17))(sd), obs), ("w1",)),
    "b1_entry_zeroed": (lambda sd, obs: reference(_zero("fc1.bias", 131)(sd), obs), ("w1",)),
    "w3_element_zeroed": (lambda sd, obs: reference(_zero("fc3.weight", (3, 255))(sd), obs), ("w3",)),
}

CHECKS = {"realistic": check_realistic, "w1": check_w1_probe, "w2": check_w2_probe, "w3": check_w3_probe,
          "tanh_saturates": check_tanh_saturates}


@pytest.mark.parametrize("check", list(CHECKS))
def test_checks_pass_the_reference(check):
    CHECKS[check](reference_forward)


@pytest.mark.parametrize("mutant", list(MUTANTS))
def test_checks_have_teeth(mutant):
    forward, catchers = MUTANTS[mutant]
    for name in catchers:
        if name == "realistic":  # every weight set's bounds catch it on their own
            stats, bad = realistic_errors(forward)
            assert bad == list(WEIGHT_SETS), stats
        else:
            with pytest.raises(AssertionError):
                CHECKS[name](forward)


# ---- GPU: the kernel -------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_w1_operand_probe():
    assert check_w1_operand(kernel_forward) == [W1_OPERAND]


@pytest.mark.gpu
def test_w3_probe_and_tanh_approx_error():
    e = check_w3_probe(kernel_forward)
    print(f"tanh.approx.f32: max relative error {e:.4g} = 2^{np.log2(e):.3f} (ISA bound 2^-10.987)")
    check_tanh_saturates(kernel_forward)


@pytest.mark.gpu
def test_w2_probe():
    print("W2 probe: worst error / tolerance", check_w2_probe(kernel_forward))


@pytest.mark.gpu
def test_w1_probe():
    print("W1 probe: worst error / tolerance", check_w1_probe(kernel_forward))


@pytest.mark.gpu
def test_realistic_weights_against_reference():
    for name, s in check_realistic(kernel_forward).items():
        print(f"{name:16s} max {s['max']:.4e} rms {s['rms']:.4e} mean {s['mean']:+.4e}")


def _sentinel(shape):
    return torch.full(shape, 0x7FC0DEAD, dtype=torch.int32, device="cuda:0").view(torch.float32)


@pytest.mark.gpu
def test_grid_sizes_and_rows_past_n():
    """The grid is min(tiles, SMs) and each CTA walks tiles with one mbarrier phase bit: every n from one row to past
    two full waves gives each row the result of one launch over all rows, and writes nothing outside rows [0, n) x
    columns [0, 4) of an [n + 256, 8] buffer.  Observation rows past n (same allocation) are NaN: never read into a
    written row."""
    import hockey_env_b200 as hk
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    sizes = (1, 127, 129, sms * 128 - 1, sms * 128, sms * 128 + 1, 2 * sms * 128 + 1)
    net = hk.ActorNetwork()
    net.load_state_dict(weight_set("default_init"))
    fused = hk.FusedActor(net)
    nmax = max(sizes)
    obs = realistic_obs(nmax, 0, seed=35).cuda()
    full = fused(obs).clone()
    torch.cuda.synchronize()
    assert torch.isfinite(full).all()
    for n in sizes:
        o = torch.full((n + 256, 18), float("nan"), device="cuda:0")
        o[:n] = obs[:n]
        buf = _sentinel((n + 256, 8))
        fused(o[:n], out=buf[:n])
        torch.cuda.synchronize()
        bits = buf.view(torch.int32)
        assert torch.equal(buf[:n, :4].view(torch.int32), full[:n].view(torch.int32)), n
        assert (bits[:n, 4:] == 0x7FC0DEAD).all() and (bits[n:] == 0x7FC0DEAD).all(), n


@pytest.mark.gpu
def test_non_finite_rows_stay_in_their_row():
    """NaN, +-inf and +-1e30 observation rows (whole rows and single elements) inside a tile change only their own
    outputs: every other row is bit-identical to the launch without them."""
    import hockey_env_b200 as hk
    net = hk.ActorNetwork()
    net.load_state_dict(weight_set("stage_3"))
    fused = hk.FusedActor(net)
    n = 3 * 128 + 17
    obs = realistic_obs(n, 0, seed=36).cuda()
    clean = fused(obs).clone()
    bad = obs.clone()
    rows = {130: float("nan"), 131: float("inf"), 132: float("-inf"), 133: 1e30, 134: -1e30, 255: float("nan"), 256: 1e30}
    for r, v in rows.items():
        bad[r] = v
    bad[140, 7], bad[141, 0], bad[142, 17] = float("nan"), float("inf"), -1e30
    got = fused(bad).clone()
    torch.cuda.synchronize()
    keep = torch.ones(n, dtype=torch.bool)
    keep[list(rows) + [140, 141, 142]] = False
    keep = keep.cuda()
    assert torch.equal(got[keep].view(torch.int32), clean[keep].view(torch.int32))
