"""Cost of a population of K TD3 learners: python scripts/bench_td3_population.py [--ks 1,2,4,8,16,32] [--batches 256,1024]
[--rows 65536,262144] [--train-k 8] [--iters 20] [--repeats 7] [--train-ticks 5] [--out FILE]

Measures, with the arms of one measurement alternating round by round:
  update       K learner updates: K FusedTD3Learner.update_from_buffer calls one after another (K launches of one cluster,
               each learner with its own replay buffer) against one FusedTD3Population.update_from_buffer (one index draw,
               one launch of K clusters), at each K and batch size, uniform replay.  ms per K updates.  Every member
               uses policy_update_freq 2, so half of the updates are actor steps.
  train_tick   one training tick of K = --train-k learners on --rows envs in total: td3.train_population (one pooled noisy
               actor launch, one env tick, one push, one population launch, one pack of all K actors) against K
               sequential td3.train(fused=True) ticks, each on its own env of rows / K envs.  ms per population tick.
The cluster size that each population launch uses is recorded with the update rows; the occupancy line gives the K up
to which the device keeps all clusters of 16 (and of 8) CTAs resident, read off hk_td3_population_cluster_size.
Method: CUDA events around back-to-back calls of one arm after a warm-up, `--repeats` alternating rounds; the median ms
per call and the spread (max - min) / median of the rounds.  Replay buffers of 100,000 rows per learner stay L2-resident
at small K.  Prints one JSON line per measurement, the card's name, power limit and max SM clock first (read in the same
process); --out also writes them to FILE.
"""
import argparse
import json
import os
import sys

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, _ROOT)
sys.path.insert(0, os.path.join(_ROOT, "scripts"))
from bench_actor_pool import gpu_info, time_arms  # noqa: E402

CAPACITY = 100_000


def _fill(buf, rows, dev, seed):
    import torch
    g = torch.Generator(device=dev).manual_seed(seed)
    buf.push(torch.randn(rows, 18, device=dev, generator=g), torch.rand(rows, 4, device=dev, generator=g) * 2 - 1,
             torch.randn(rows, device=dev, generator=g), torch.randn(rows, 18, device=dev, generator=g),
             (torch.rand(rows, device=dev, generator=g) < 0.01).float())


def run_updates(k, b, args, emit):
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    dev = "cuda:0"
    cfg = td3.TD3Config(batch_size=b, buffer_size=CAPACITY)
    learners = []
    for m in range(k):
        buf = hk.DeviceReplayBuffer(CAPACITY, device=dev, seed=m)
        _fill(buf, CAPACITY, dev, 100 + m)
        learners.append(td3.FusedTD3Learner(config=cfg, replay_buffer=buf, device=dev, seed=m))
    pbuf = td3.PopulationReplayBuffer(k, CAPACITY, device=dev, seed=1)
    _fill(pbuf, k * CAPACITY, dev, 7)
    pop = td3.FusedTD3Population(k, configs=cfg, replay_buffer=pbuf, device=dev)

    def sequential():
        for lr in learners:
            lr.update_from_buffer()

    t = time_arms({"sequential": sequential, "population": pop.update_from_buffer}, args.iters, args.repeats, warmup=4)
    cluster = int(hk.load_library().hk_td3_population_cluster_size(k, 0))
    for name, (ms, spread) in t.items():
        emit({"what": "update", "arm": name, "k": k, "batch": b, "ms": round(ms, 5), "spread": round(spread, 3),
              "cluster": cluster if name == "population" else int(hk.load_library().hk_td3_cluster_size(0))})


def run_train(n, k, args, emit):
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    dev = "cuda:0"
    per = n // k
    envs = [hk.HockeyVecEnv(per, device=dev, seed=4 + m, p2="weak") for m in range(k)]
    learners = [td3.FusedTD3Learner(replay_buffer=hk.DeviceReplayBuffer(4 * per, device=dev, seed=m), device=dev, seed=m)
                for m in range(k)]
    penv = hk.HockeyVecEnv(n, device=dev, seed=4, p2="weak")
    pop = td3.FusedTD3Population(k, configs=td3.TD3Config(buffer_size=4 * per), device=dev)
    for e, lr in zip(envs, learners):
        td3.train(e, lr, ticks=1, warmup_ticks=1, fused=True)  # fill the buffers with one tick
    td3.train_population(penv, pop, ticks=1, warmup_ticks=1)
    tt = args.train_ticks

    def sequential():
        for e, lr in zip(envs, learners):
            td3.train(e, lr, ticks=tt, warmup_ticks=0, fused=True)

    t = time_arms({"sequential": sequential, "population": lambda: td3.train_population(penv, pop, ticks=tt, warmup_ticks=0)},
                  max(1, args.iters // tt), args.repeats, warmup=1)
    for name, (ms, spread) in t.items():
        emit({"what": "train_tick", "arm": name, "k": k, "rows": n, "ms": round(ms / tt, 5), "spread": round(spread, 3),
              "updates_per_tick": 1, "batch_size": 256})
    for e in envs + [penv]:
        e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="1,2,4,8,16,32")
    ap.add_argument("--batches", default="256,1024")
    ap.add_argument("--rows", default="65536,262144")
    ap.add_argument("--train-k", type=int, default=8)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--train-ticks", type=int, default=5)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    args.iters += args.iters % 2
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_td3_population.py measures the B200 kernels: no CUDA device")
    import hockey_env_b200 as hk
    L = hk.load_library()
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(json.dumps(d))

    sizes = {k: int(L.hk_td3_population_cluster_size(k, 0)) for k in range(1, 65)}
    occ16 = max([k for k, s in sizes.items() if s == 16 and all(sizes[j] == 16 for j in range(1, k + 1))], default=0)
    occ8 = max([k for k, s in sizes.items() if s == 8], default=0)
    emit({"gpu": gpu_info(), "torch": torch.__version__, "td3_cluster_size": int(L.hk_td3_cluster_size(0)),
          "max_resident_clusters_16": occ16, "max_resident_clusters_8": occ8 if occ8 else "not above the 16-CTA count",
          "population_cluster_size": {k: sizes[k] for k in (1, 2, 4, 8, 9, 12, 16, 17, 24, 32, 48, 64)}})
    for b in (int(x) for x in args.batches.split(",") if x):
        for k in (int(x) for x in args.ks.split(",") if x):
            run_updates(k, b, args, emit)
    for n in (int(x) for x in args.rows.split(",") if x):
        run_train(n, args.train_k, args, emit)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
