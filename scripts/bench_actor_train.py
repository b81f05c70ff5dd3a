"""Cost of the learner's own behaviour policy per tick: python scripts/bench_actor_train.py [--rows 65536,262144]
[--iters 20] [--repeats 5] [--train-ticks 10] [--out FILE]

The actor is the reference checkpoint stage_3; the exploration noise has std 0.2 (TD3Config.action_noise_scale).  At each
row count N it measures, with the arms of one measurement alternating round by round:
  behaviour      one tick's exploring actions on a fixed obs [N, 18]:
                   torch_noise   the fp32 torch module, then randn / add / clamp (td3._explore, collect(noise=) on a module)
                   fused_noisy   one hk_actor_forward_noisy launch (FusedActor(obs, noise=0.2))
                   fused_plain   hk_actor_forward without noise (for the cost of the noise epilogue)
  pack           FusedActor.refresh (hk_actor_pack on the device) against the host path FusedActor.pack + copy to the
                 device (host clock around the call and a device synchronise)
  collect_tick   one training.collect tick (actor -> env.step -> buffer push) with noise 0.2, the module against a FusedActor
  train_tick     td3.train ticks (explore -> env.step -> push -> one learner update with batch 256), fused=False against
                 fused=True; --train-ticks ticks per call, ms per tick reported
Method: CUDA events around `--iters` back-to-back calls of one arm after a warm-up, `--repeats` alternating rounds; the
median ms per call and the spread (max - min) / median of the rounds are reported.  The obs tensor (N x 72 B <= 19 MB) and
the weights stay L2-resident, as they are when the env step has just written the observations.  Prints one JSON line per
measurement, the card name and power limit first; --out also writes them to FILE.
"""
import argparse
import json
import os
import statistics
import sys
import time

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, _ROOT)
sys.path.insert(0, os.path.join(_ROOT, "scripts"))
from bench_actor_pool import gpu_info, time_arms  # noqa: E402

NPZ = os.path.join(_ROOT, "tests", "golden", "td3_actors.npz")
SIGMA = 0.2


def run(n, args, emit):
    import torch
    import hockey_env_b200 as hk
    from hockey_env_b200 import td3
    from hockey_env_b200.actor import FusedActor, _reference_state_dict
    from hockey_env_b200.training import behaviour_actions
    dev = "cuda:0"
    module = hk.load_td3_actor(NPZ, device=dev, name="stage_3")
    fused = hk.FusedActor(module, seed=1)
    env = hk.HockeyVecEnv(n, device=dev, seed=1, p2="weak")
    obs = env.obs.clone()
    out = torch.empty((n, 4), device=dev)

    # behaviour policy of one tick
    with torch.no_grad():
        t = time_arms({"torch_noise": lambda: behaviour_actions(module, obs, SIGMA),
                       "fused_noisy": lambda: fused(obs, out=out, noise=SIGMA),
                       "fused_plain": lambda: fused(obs, out=out)}, args.iters, args.repeats)
        diff = float((fused(obs) - module(obs)).abs().mean())
    for name, (ms, spread) in t.items():
        emit({"what": "behaviour", "arm": name, "rows": n, "ms": round(ms, 5), "spread": round(spread, 3)})
    emit({"what": "check", "rows": n, "mean_abs_fused_minus_fp32": round(diff, 6)})

    # weight refresh: device pack against the host round trip
    t = time_arms({"refresh": lambda: fused.refresh(module)}, args.iters, args.repeats)
    host = []
    for _ in range(args.repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.iters):
            fused.params.copy_(FusedActor.pack(_reference_state_dict(module, "bench")).to(dev))
        torch.cuda.synchronize()
        host.append((time.perf_counter() - t0) * 1e3 / args.iters)
    hm = statistics.median(host)
    emit({"what": "pack", "arm": "hk_actor_pack", "rows": n, "ms": round(t["refresh"][0], 5), "spread": round(t["refresh"][1], 3)})
    emit({"what": "pack", "arm": "host_pack_and_copy", "rows": n, "ms": round(hm, 5), "spread": round((max(host) - min(host)) / hm, 3)})
    env.close()

    # one collect tick: separate envs and buffers per arm, same seeds
    arms, envs = {}, []
    for name, actor in (("module", module), ("fused", fused)):
        e = hk.HockeyVecEnv(n, device=dev, seed=2, p2="weak")
        buf = hk.DeviceReplayBuffer(4 * n, device=dev, seed=3)
        envs.append(e)
        arms[name] = lambda e=e, actor=actor, buf=buf: hk.collect(e, actor, buf, 1, noise=SIGMA)
    t = time_arms(arms, args.iters, args.repeats)
    for name, (ms, spread) in t.items():
        emit({"what": "collect_tick", "arm": name, "rows": n, "ms": round(ms, 5), "spread": round(spread, 3)})

    # td3.train ticks: one learner update per tick after the replay buffer holds a batch
    arms = {}
    for fz in (False, True):
        e = hk.HockeyVecEnv(n, device=dev, seed=4, p2="weak")
        buf = hk.DeviceReplayBuffer(4 * n, device=dev, seed=5)
        learner = td3.DeviceTD3Learner(actor=hk.load_td3_actor(NPZ, device=dev, name="stage_3").train(), replay_buffer=buf,
                                       device=dev, seed=6)
        td3.train(e, learner, ticks=1, warmup_ticks=1, fused=fz)  # fill the buffer with one tick
        envs.append(e)
        arms["fused" if fz else "torch"] = lambda e=e, lr=learner, fz=fz: td3.train(e, lr, ticks=args.train_ticks, warmup_ticks=0,
                                                                                     fused=fz)
    t = time_arms(arms, max(1, args.iters // args.train_ticks), args.repeats, warmup=1)
    for name, (ms, spread) in t.items():
        emit({"what": "train_tick", "arm": name, "rows": n, "ms": round(ms / args.train_ticks, 5), "spread": round(spread, 3),
              "updates_per_tick": 1, "batch_size": 256})
    for e in envs:
        e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="65536,262144")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--train-ticks", type=int, default=10)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_actor_train.py measures the B200 kernels: no CUDA device")
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(json.dumps(d))

    emit({"gpu": gpu_info(), "torch": torch.__version__, "tf32_matmul": torch.backends.cuda.matmul.allow_tf32})
    for n in (int(x) for x in args.rows.split(",")):
        run(n, args, emit)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
