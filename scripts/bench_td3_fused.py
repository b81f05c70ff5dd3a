"""Cost of the TD3 learner update: python scripts/bench_td3_fused.py [--batches 256,1024] [--rows 65536,262144]
[--iters 50] [--repeats 7] [--train-ticks 10] [--out FILE]

Measures, with the arms of one measurement alternating round by round:
  update       one learner update from a full replay buffer (update_from_buffer: index draw, gather, target, critic step,
               and on every second call the actor step and Polyak), DeviceTD3Learner (torch modules, autograd,
               torch.optim.Adam; TF32 off) against FusedTD3Learner (one hk_td3_update launch), at each batch size, uniform
               and prioritized replay.  ms per update, averaged over `--iters` consecutive updates (an even number, so
               actor steps are half of them).
  train_tick   td3.train ticks at each env count (noisy FusedActor launch -> env.step -> push -> one learner update of
               batch 256), fused=True with the torch learner against fused=True with the fused learner; --train-ticks
               ticks per call, ms per tick reported.
Method: CUDA events around back-to-back calls of one arm after a warm-up, `--repeats` alternating rounds; the median ms
per call and the spread (max - min) / median of the rounds.  The replay buffer (300,000 rows) and the weights stay
L2-resident.  Prints one JSON line per measurement, the card name and power limit first; --out also writes them to FILE.
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


def _buffer(prio, dev, capacity=300_000):
    import torch
    from hockey_env_b200 import td3
    from hockey_env_b200.training import DeviceReplayBuffer
    buf = (td3.DevicePrioritizedReplayBuffer if prio else DeviceReplayBuffer)(capacity, device=dev, seed=3)
    g = torch.Generator(device=dev).manual_seed(4)
    buf.push(torch.randn(capacity, 18, device=dev, generator=g), torch.rand(capacity, 4, device=dev, generator=g) * 2 - 1,
             torch.randn(capacity, device=dev, generator=g), torch.randn(capacity, 18, device=dev, generator=g),
             (torch.rand(capacity, device=dev, generator=g) < 0.01).float())
    if prio:
        buf.weights.copy_(torch.rand(capacity, device=dev, generator=g) + 0.01)
    return buf


def run_updates(b, prio, args, emit):
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    dev = "cuda:0"
    arms = {}
    for name, cls in (("torch", td3.DeviceTD3Learner), ("fused", td3.FusedTD3Learner)):
        buf = _buffer(prio, dev)
        learner = cls(actor=hk.load_td3_actor(NPZ, device=dev, name="stage_3").train(), replay_buffer=buf, device=dev, seed=6,
                      config=td3.TD3Config(prioritized_replay=prio, batch_size=b))
        arms[name] = lambda lr=learner: lr.update_from_buffer()
    t = time_arms(arms, args.iters, args.repeats, warmup=4)
    for name, (ms, spread) in t.items():
        emit({"what": "update", "arm": name, "batch": b, "prioritized": prio, "ms": round(ms, 5), "spread": round(spread, 3)})


def run_train(n, args, emit):
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    dev = "cuda:0"
    arms, envs = {}, []
    for name, cls in (("torch_learner", td3.DeviceTD3Learner), ("fused_learner", td3.FusedTD3Learner)):
        e = hk.HockeyVecEnv(n, device=dev, seed=4, p2="weak")
        buf = hk.DeviceReplayBuffer(4 * n, device=dev, seed=5)
        learner = cls(actor=hk.load_td3_actor(NPZ, device=dev, name="stage_3").train(), replay_buffer=buf, device=dev, seed=6)
        td3.train(e, learner, ticks=1, warmup_ticks=1, fused=True)  # fill the buffer with one tick
        envs.append(e)
        arms[name] = lambda e=e, lr=learner: td3.train(e, lr, ticks=args.train_ticks, warmup_ticks=0, fused=True)
    t = time_arms(arms, max(1, args.iters // args.train_ticks), args.repeats, warmup=1)
    for name, (ms, spread) in t.items():
        emit({"what": "train_tick", "arm": name, "rows": n, "ms": round(ms / args.train_ticks, 5), "spread": round(spread, 3),
              "updates_per_tick": 1, "batch_size": 256, "fused_actor": True})
    for e in envs:
        e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="256,1024")
    ap.add_argument("--rows", default="65536,262144")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--train-ticks", type=int, default=10)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    args.iters += args.iters % 2
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_td3_fused.py measures the B200 kernels: no CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(json.dumps(d))

    emit({"gpu": gpu_info(), "torch": torch.__version__, "tf32_matmul": torch.backends.cuda.matmul.allow_tf32})
    for b in (int(x) for x in args.batches.split(",") if x):
        for prio in (False, True):
            run_updates(b, prio, args, emit)
    for n in (int(x) for x in args.rows.split(",") if x):
        run_train(n, args, emit)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
