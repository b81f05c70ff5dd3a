"""Throughput of per-env game modes: python scripts/bench_modes.py [--steps K] [--warmup W] [--envs N] [--ab PARENT_TREE]

Mixed mode: N envs (default 65,536) split a third per mode (NORMAL / TRAIN_SHOOTING / TRAIN_DEFENSE, env i plays
mode i % 3), strong vs strong in-kernel BasicOpponents with auto-reset, stepped
  * as ONE handle with per-env modes, and
  * as three single-mode handles of N // 3 envs stepped back to back on one stream,
with env-steps/s from CUDA events around K timed steps and per-kernel times from hk_kernel_times.

--ab PARENT_TREE: the single-mode workloads of bench.py (normal65k, defense65k, normal1M), run alternately from
PARENT_TREE (a built checkout of the commit to compare with: its own bench.py, package and library) and from this
tree, --repeats times each, so that any difference can be read against the spread of repeated runs.
Prints one JSON line per measurement; the card name and power limit first.
"""
import argparse
import json
import os
import subprocess
import sys

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, _ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # measurement still runs; the line says what is unknown
        return f"unknown ({e})"


def timed(step_fns, envs, steps, warmup):
    import torch
    for _ in range(warmup):
        for f in step_fns:
            f()
    torch.cuda.synchronize()
    for e in envs:
        e.kernel_timing(True)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        for f in step_fns:
            f()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    kern = {}
    for e in envs:
        t, _ = e.kernel_times()
        for k, v in t.items():
            kern[k] = kern.get(k, 0.0) + v / steps
        e.kernel_timing(False)
    return ms, {k: round(v, 4) for k, v in kern.items()}


def mixed(args):
    import torch
    import hockey_env_b200 as hk
    n = args.envs
    modes = (torch.arange(n, device="cuda:0") % 3).to(torch.uint8)
    env = hk.HockeyVecEnv(n, mode=modes, device="cuda:0", seed=args.seed, p1="strong", p2="strong")
    ms, kern = timed([env.step], [env], args.steps, args.warmup)
    print(json.dumps({"layout": "one mixed handle", "envs": n, "steps": args.steps, "ms_per_step": ms / args.steps,
                      "env_steps_per_s": n * args.steps / (ms / 1e3), "kernel_ms_per_tick": kern,
                      "modes_now": torch.bincount(env.modes().long(), minlength=3).tolist()}), flush=True)
    env.close()
    k = n // 3
    envs = [hk.HockeyVecEnv(k, mode=hk.Mode(m), device="cuda:0", seed=args.seed, env_id_offset=m * k, p1="strong",
                            p2="strong") for m in range(3)]
    ms, kern = timed([e.step for e in envs], envs, args.steps, args.warmup)
    print(json.dumps({"layout": "three single-mode handles, back to back", "envs": 3 * k, "steps": args.steps,
                      "ms_per_step": ms / args.steps, "env_steps_per_s": 3 * k * args.steps / (ms / 1e3),
                      "kernel_ms_per_tick": kern}), flush=True)
    for e in envs:
        e.close()


def ab(args):
    trees = [("parent", os.path.abspath(args.ab)), ("this", _ROOT)]
    for r in range(args.repeats):
        for config in args.configs.split(","):
            for name, tree in trees:
                out = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--config", config, "--steps",
                                      str(args.bench_steps), "--warmup", str(args.bench_warmup), "--no-e2e",
                                      "--no-cpu-baseline", "--rollout-k", "0"], cwd=tree, capture_output=True, text=True)
                try:
                    d = json.loads(out.stdout.strip().splitlines()[-1])
                    print(json.dumps({"config": config, "lib": name, "repeat": r, "value": d.get("value"),
                                      "ms_per_step": d.get("ms_per_step"), "kernel_ms_per_tick": d.get("kernel_ms_per_tick")}),
                          flush=True)
                except Exception as e:
                    print(json.dumps({"config": config, "lib": name, "repeat": r, "error": str(e),
                                      "stderr": out.stderr[-2000:]}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--ab", metavar="PARENT_TREE", help="also run bench.py's single-mode workloads from this built checkout")
    ap.add_argument("--configs", default="normal65k,defense65k,normal1M")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=200)
    ap.add_argument("--bench-warmup", type=int, default=30)
    args = ap.parse_args()
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    mixed(args)
    if args.ab:
        ab(args)


if __name__ == "__main__":
    main()
