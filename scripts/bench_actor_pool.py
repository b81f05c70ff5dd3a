"""Cost of the self-play snapshot opponents per tick: python scripts/bench_actor_pool.py [--rows 65536,262144]
[--ks 1,2,4,8,16] [--iters 20] [--repeats 5] [--out FILE]

Inputs: N observation rows (seeded, in the env's range) and a choice per row, uniform over K snapshots with 40 % of the
rows set to -1 (envs that play an in-kernel BasicOpponent, as in a weak / strong / snapshot mix).  The K snapshots are
the reference checkpoint stage_3 and seeded perturbations of it.  Arms, each on the same rows and choices:
  (a) torch_list   OpponentPool.opponent_actions with the snapshots as torch fp32 modules: K full-batch MLPs + torch.where
  (b) fused_list   the same with K FusedActor (hk_actor_forward) launches over all N rows + torch.where
  (c) pooled       OpponentPool.opponent_actions with a FusedActorPool: one hk_actor_forward_pool over the env's
                   obs_agent_two(), snapshot index per env, -1 for the BasicOpponent envs
  pool_call        the bare FusedActorPool call on a fixed obs tensor (no obs_agent_two, no index conversion)
  (a) and (c) also as complete OpponentPool.step ticks (env step with p2='per_env' and re-draws; p_weak = p_strong =
  0.2, p_snapshot = 0.6) on an env of N envs.
K = 1 overhead: the pooled call with K = 1 and every row chosen against hk_actor_forward (FusedActor) over the same rows.

Method: CUDA events around `--iters` back-to-back calls of one arm, the arms alternating, `--repeats` rounds after a
warm-up; the median ms per call is reported.  The obs tensor (N x 72 B <= 19 MB) and the weights stay L2-resident, as
they are when the env step has just written the observations.  Prints one JSON line per measurement, the card name
and power limit first; --out also writes them to FILE.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, _ROOT)
NPZ = os.path.join(_ROOT, "tests", "golden", "td3_actors.npz")
FLOP_PER_ROW = 2 * (18 * 256 + 256 * 256 + 256 * 4)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # measurement still runs; the line says what is unknown
        return f"unknown ({e})"


def snapshots(k, device):
    import torch
    import hockey_env_b200 as hk
    g = torch.Generator().manual_seed(99)
    out = []
    for s in range(k):
        a = hk.load_td3_actor(NPZ, device=device, name="stage_3")
        if s:
            with torch.no_grad():
                for p in a.parameters():
                    p.add_((0.05 * torch.randn(p.shape, generator=g)).to(p.device))
        out.append(a)
    return out


def time_arms(arms, iters, repeats, warmup=3):
    """{name: median ms per call} for zero-argument callables, alternating the arms round by round."""
    import torch
    for f in arms.values():
        for _ in range(warmup):
            f()
    torch.cuda.synchronize()
    ms = {name: [] for name in arms}
    for _ in range(repeats):
        for name, f in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                f()
            b.record()
            torch.cuda.synchronize()
            ms[name].append(a.elapsed_time(b) / iters)
    return {name: (statistics.median(v), (max(v) - min(v)) / statistics.median(v)) for name, v in ms.items()}


def choices(n, k, device, seed):
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    c = torch.randint(0, k, (n,), device=device, generator=g)
    c[torch.rand(n, device=device, generator=g) < 0.4] = -1
    return c


def run(n, k, args, emit):
    import torch
    import hockey_env_b200 as hk
    dev = "cuda:0"
    actors = snapshots(k, dev)
    fused = [hk.FusedActor(a) for a in actors]
    table = hk.FusedActorPool(actors)
    c = choices(n, k, dev, seed=n + k)

    # opponent_actions: one env, three OpponentPools over it, all with the same per-env draw
    env = hk.HockeyVecEnv(n, device=dev, seed=1, p2="per_env")
    pools = {"torch_list": hk.OpponentPool(env, 0.2, 0.2, actors, 0.6, seed=2),
             "fused_list": hk.OpponentPool(env, 0.2, 0.2, fused, 0.6, seed=2),
             "pooled": hk.OpponentPool(env, 0.2, 0.2, table, 0.6, seed=2)}
    for p in pools.values():
        p.choice.copy_(torch.where(c >= 0, c + hk.OpponentPool.SNAPSHOT0, torch.zeros_like(c)))
    obs = env.obs_agent_two().clone()
    c32 = c.to(torch.int32)
    out = torch.empty((n, 4), device=dev)
    arms = {name: p.opponent_actions for name, p in pools.items()}
    arms["pool_call"] = lambda: table(obs, c32, out=out)
    t = time_arms(arms, args.iters, args.repeats)
    with torch.no_grad():  # the arms agree where they must: (b) and (c) bit for bit on the snapshot rows
        ref = pools["fused_list"].opponent_actions().clone()
        got = pools["pooled"].opponent_actions().clone()
    same = bool(torch.equal(ref, got))
    for name, (ms, spread) in t.items():
        emit({"what": "opponent_actions", "arm": name, "rows": n, "k": k, "ms": round(ms, 5), "spread": round(spread, 3),
              "snapshot_rows": int((c >= 0).sum())} | ({"tflops_on_snapshot_rows": round(int((c >= 0).sum()) * FLOP_PER_ROW / ms / 1e9, 1)}
                                                      if name == "pool_call" else {}))
    emit({"what": "check", "rows": n, "k": k, "fused_list_equals_pooled": same})

    # complete OpponentPool.step ticks for (a) and (c): one env each, same seeds
    ticks = {}
    a1 = torch.zeros((n, 4), device=dev)
    for name, snaps in (("torch_list", actors), ("pooled", table)):
        e = hk.HockeyVecEnv(n, device=dev, seed=1, p2="per_env")
        p = hk.OpponentPool(e, 0.2, 0.2, snaps, 0.6, seed=2)
        ticks[name] = (e, p)
    t = time_arms({name: (lambda p=p: p.step(a1)) for name, (e, p) in ticks.items()}, args.iters, args.repeats)
    for name, (ms, spread) in t.items():
        emit({"what": "opponent_pool_step", "arm": name, "rows": n, "k": k, "ms": round(ms, 5), "spread": round(spread, 3)})
    for e, _ in ticks.values():
        e.close()
    env.close()

    if k == 1:  # grouping overhead: K = 1, every row chosen, against the single-actor kernel on the same rows
        zeros = torch.zeros(n, dtype=torch.int32, device=dev)
        out2 = torch.empty((n, 4), device=dev)
        t = time_arms({"hk_actor_forward": lambda: fused[0](obs, out=out), "pool_k1_all_rows": lambda: table(obs, zeros, out=out2)},
                      args.iters, args.repeats)
        torch.cuda.synchronize()
        emit({"what": "k1_overhead", "rows": n, "hk_actor_forward_ms": round(t["hk_actor_forward"][0], 5),
              "pool_ms": round(t["pool_k1_all_rows"][0], 5),
              "overhead_ms": round(t["pool_k1_all_rows"][0] - t["hk_actor_forward"][0], 5),
              "spreads": [round(t["hk_actor_forward"][1], 3), round(t["pool_k1_all_rows"][1], 3)],
              "bit_equal": bool(torch.equal(out, out2))})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="65536,262144")
    ap.add_argument("--ks", default="1,2,4,8,16")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_actor_pool.py measures the B200 kernels: no CUDA device")
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(json.dumps(d))

    emit({"gpu": gpu_info(), "torch": torch.__version__, "tf32_matmul": torch.backends.cuda.matmul.allow_tf32})
    for n in (int(x) for x in args.rows.split(",")):
        for k in (int(x) for x in args.ks.split(",")):
            run(n, k, args, emit)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
