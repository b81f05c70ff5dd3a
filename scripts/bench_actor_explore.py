"""Cost of exploration noise with on-device state: python scripts/bench_actor_explore.py [--rows 65536,262144] [--pool-k 8]
[--train-k 8] [--train-rows 65536] [--iters 20] [--repeats 7] [--train-ticks 5] [--out FILE]

The actor is the reference checkpoint stage_3 (the pool: stage_3 / competition alternating).  At each row count N it
measures, with the arms of one measurement alternating round by round:
  single       one behaviour-policy launch on a fixed obs [N, 18]:
                 noisy          hk_actor_forward_noisy, sigma 0.2 (FusedActor(obs, noise=0.2))
                 explore_gauss  hk_actor_forward_explore with a Gaussian slot (rho 0, scale 0.2): reads no state, writes it
                 explore_ou     hk_actor_forward_explore with an OU slot (theta 0.15, dt 0.01) and a reset mask with 1 % of
                                rows set: reads and writes the state and reads the mask
  pool         K = --pool-k snapshots, choice = row // (N / K):
                 shared_sigma   hk_actor_forward_pool_noisy, sigma 0.2
                 ou_per_slot    hk_actor_forward_pool_explore with K distinct OU slots and the reset mask
  train_tick   one td3.train_population tick of K = --train-k members on --train-rows envs (pooled actor launch, env
               tick, push, population update, pack): one shared sigma against per-member OU slots; ms per tick
Method: CUDA events around `--iters` back-to-back calls of one arm after a warm-up, `--repeats` alternating rounds; the
median ms per call and the spread (max - min) / median of the rounds.  The obs (N x 72 B) and state (N x 16 B) tensors
stay L2-resident, as they are in a training tick.  Prints one JSON line per measurement, the card's name, power limit and
max SM clock first (read in the same process); --out also writes them to FILE.
"""
import argparse
import json
import os
import sys

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, _ROOT)
sys.path.insert(0, os.path.join(_ROOT, "scripts"))
from bench_actor_pool import gpu_info, time_arms  # noqa: E402

NPZ = os.path.join(_ROOT, "tests", "golden", "td3_actors.npz")
SIGMA = 0.2


def run(n, args, emit):
    import torch
    import hockey_env_b200 as hk
    dev = "cuda:0"
    actors = [hk.load_td3_actor(NPZ, device=dev, name=nm) for nm in ("stage_3", "competition")]
    fused = hk.FusedActor(actors[0], seed=1)
    g = torch.Generator(device=dev).manual_seed(n)
    obs = torch.randn((n, 18), device=dev, generator=g) * 2
    reset = torch.rand(n, device=dev, generator=g) < 0.01
    out = torch.empty((n, 4), device=dev)
    gauss = hk.ExplorationNoise(n, sigma=SIGMA)
    ou = hk.ExplorationNoise(n, sigma=SIGMA, theta=0.15, dt=0.01)
    with torch.no_grad():
        t = time_arms({"noisy": lambda: fused(obs, out=out, noise=SIGMA),
                       "explore_gauss": lambda: fused(obs, out=out, noise=gauss),
                       "explore_ou": lambda: fused(obs, out=out, noise=ou, reset=reset)}, args.iters, args.repeats)
    for name, (ms, spread) in t.items():
        emit({"what": "single", "arm": name, "rows": n, "ms": round(ms, 5), "spread": round(spread, 3)})

    k = args.pool_k
    pool = hk.FusedActorPool([actors[s % 2] for s in range(k)], seed=2)
    choice = (torch.arange(n, device=dev) // (n // k)).clamp(max=k - 1).to(torch.int32)
    per = hk.ExplorationNoise(n, slots=k, sigma=[0.1 + 0.05 * s for s in range(k)], theta=[0.05 + 0.05 * s for s in range(k)],
                              dt=0.01)
    with torch.no_grad():
        t = time_arms({"shared_sigma": lambda: pool(obs, choice, out=out, noise=SIGMA),
                       "ou_per_slot": lambda: pool(obs, choice, out=out, noise=per, reset=reset)}, args.iters, args.repeats)
    for name, (ms, spread) in t.items():
        emit({"what": "pool", "arm": name, "rows": n, "k": k, "ms": round(ms, 5), "spread": round(spread, 3)})


def run_train(n, k, args, emit):
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    dev = "cuda:0"
    per = n // k
    arms = {}
    envs = []
    for name in ("shared_sigma", "ou_per_member"):
        env = hk.HockeyVecEnv(n, device=dev, seed=4, p2="weak")
        pop = td3.FusedTD3Population(k, configs=td3.TD3Config(buffer_size=4 * per), device=dev)
        noise = None if name == "shared_sigma" else hk.ExplorationNoise(
            n, slots=k, sigma=[0.1 + 0.05 * m for m in range(k)], theta=[0.05 + 0.05 * m for m in range(k)], dt=0.01)
        td3.train_population(env, pop, ticks=1, warmup_ticks=1, noise=noise)  # fill the buffers with one tick
        envs.append(env)
        arms[name] = lambda env=env, pop=pop, noise=noise: td3.train_population(env, pop, ticks=args.train_ticks, warmup_ticks=0,
                                                                                noise=noise)
    t = time_arms(arms, max(1, args.iters // args.train_ticks), args.repeats, warmup=1)
    for name, (ms, spread) in t.items():
        emit({"what": "train_tick", "arm": name, "k": k, "rows": n, "ms": round(ms / args.train_ticks, 5),
              "spread": round(spread, 3), "updates_per_tick": 1, "batch_size": 256})
    for e in envs:
        e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="65536,262144")
    ap.add_argument("--pool-k", type=int, default=8)
    ap.add_argument("--train-k", type=int, default=8)
    ap.add_argument("--train-rows", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--train-ticks", type=int, default=5)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_actor_explore.py measures the B200 kernels: no CUDA device")
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(json.dumps(d))

    emit({"gpu": gpu_info(), "torch": torch.__version__})
    for n in (int(x) for x in args.rows.split(",") if x):
        run(n, args, emit)
    if args.train_rows:
        run_train(args.train_rows, args.train_k, args, emit)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
