#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched HockeyEnv hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--config NAME]   # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...         # the CPU path (oracle restatement) on the host cores
  python bench.py ... --dump-outputs DIR                          # also save the last timed step's outputs (see dump_outputs)

A "step" is one tick of every env of the batch (one hk_step call per GPU): physics, contact sensing, rewards,
observation write, in-kernel opponents and auto-reset.  Workloads (`--config`, BASELINE.json `configs`):

  normal65k   (default) 65,536 NORMAL envs per GPU, strong-vs-strong in-kernel BasicOpponent  -- the headline metric
  shooting4k  4,096 TRAIN_SHOOTING envs per GPU, U(-1,1) random actions for both players      -- configs[1]
  defense65k  65,536 TRAIN_DEFENSE envs per GPU, strong BasicOpponent vs zero action          -- configs[2]
  defense65k_weak  same with a weak BasicOpponent as player 2
  normal1M    1,048,576 NORMAL envs IN TOTAL (sharded over the GPUs), strong vs strong        -- configs[3], north_star target
  actor262k   262,144 NORMAL envs in total, player 1 = the reference's trained TD3 actor (stage_3 weights, torch
              matmuls on the obs tensor in place), player 2 = in-kernel strong BasicOpponent  -- configs[4]

Envs are independent: contiguous global-env-id shards, no per-step communication; episode statistics are all-reduced
once at the end (NCCL).

Steady state: episodes start synchronised after a reset, and the first ticks (no puck has reached a wall or a racket
yet) are far cheaper than the stationary mix.  Both arms therefore run an UNTIMED pre-roll of >= 400 ticks first,
independent of --warmup, extended until the TOI-event rate of two consecutive 100-tick windows agrees within 20 %.
Timing: W untimed warm-up steps through the timed call path, then K steps each bracketed by CUDA events on the launching
stream with an L2 flush (256 MiB memset, untimed) between steps, barrier + synchronize on both sides, MAX over ranks.
"""
import argparse
import json
import os
import sys
import threading
import time

_ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, _ROOT)

# SURVEY.md section 8(d): algorithmic bytes per env-step (96 B state record read + written, obs 72, reward 4, done 1,
# info 16; + 32 B action read when actions are external).  STORED_* is what this implementation actually keeps per env
# in HBM (256 B core record incl. fat AABBs, contact list, RNG counters, episode returns) -- reported beside it.
ALGO_BYTES_FUSED, ALGO_BYTES_EXTERNAL = 285, 317
STORED_BYTES_FUSED = 256 + 256 + 72 + 4 + 1 + 16
ISSUE_PEAK_WARP_INST_PER_S = 148 * 4 * 1.965e9  # SURVEY 8(d): 148 SMs x 4 schedulers x 1 warp-inst/clk x 1.965 GHz
PREROLL_TICKS = 400
DUMP_BYTES = 60 << 20  # --dump-outputs: above this, a fixed sample of env rows is written (keeps a dump under 64 MB)
DUMP_SAMPLE_SEED = 0

CONFIGS = {
    "normal65k": dict(mode="NORMAL", p1="strong", p2="strong", per_gpu=65536, total=None,
                      text="65536 NORMAL envs per GPU, strong-vs-strong in-kernel BasicOpponent"),
    "shooting4k": dict(mode="TRAIN_SHOOTING", p1="random", p2="random", per_gpu=4096, total=None,
                       text="4096 TRAIN_SHOOTING envs per GPU, U(-1,1) random actions for both players"),
    "defense65k": dict(mode="TRAIN_DEFENSE", p1="strong", p2="zero", per_gpu=65536, total=None,
                       text="65536 TRAIN_DEFENSE envs per GPU, strong BasicOpponent vs zero action"),
    "defense65k_weak": dict(mode="TRAIN_DEFENSE", p1="strong", p2="weak", per_gpu=65536, total=None,
                            text="65536 TRAIN_DEFENSE envs per GPU, strong vs weak BasicOpponent"),
    "normal1M": dict(mode="NORMAL", p1="strong", p2="strong", per_gpu=None, total=1048576,
                     text="1048576 NORMAL envs in total, strong-vs-strong in-kernel BasicOpponent"),
    "normal1M_weak": dict(mode="NORMAL", p1="weak", p2="strong", per_gpu=None, total=1048576,
                          text="1048576 NORMAL envs in total, weak-vs-strong in-kernel BasicOpponent"),
    "actor262k": dict(mode="NORMAL", p1="actor", p2="strong", per_gpu=None, total=262144,
                      text="262144 NORMAL envs in total, player 1 = TD3 actor (stage_3 weights, on device), player 2 = "
                           "in-kernel strong BasicOpponent"),
}


def resolve(args, world):
    c = dict(CONFIGS[args.config])
    if args.envs:
        n, scaling = args.envs, "weak"
    elif c["total"]:
        n, scaling = c["total"] // world, "strong"
    else:
        n, scaling = c["per_gpu"], "weak"
    c["n"], c["scaling"] = n, scaling
    return c


def config_dict(args, c, world):
    """Identical for both arms (the driver compares them)."""
    return {"workload": f"{args.config}: {c['text']}, auto-reset, all per-tick outputs (obs/reward/done/info) written",
            "name": args.config, "envs_per_gpu": c["n"], "mode": c["mode"], "p1": c["p1"], "p2": c["p2"],
            "parallelism": f"env-sharded x{world}, no per-step communication",
            "steady_state": f">= {PREROLL_TICKS} untimed pre-roll ticks before warm-up",
            "l2": "no flush" if args.no_l2_flush else "flushed between timed steps (256 MiB memset, untimed)"}


def _peaks():
    p = os.path.join(_ROOT, "MEASURED_PEAKS.json")
    try:
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _capture(name):
    """ncu numbers of the dominant kernel for this workload, extracted from the committed capture of this build
    (scripts/extract_profiles.py -> profiles/roofline_capture.json); None if there is no capture for it."""
    try:
        return json.load(open(os.path.join(_ROOT, "profiles", "roofline_capture.json"))).get(name)
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            pass

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=1.0)
        s = sorted(self.samples)
        med = s[len(s) // 2] if s else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ---- CPU legs (the oracle restatement; the one place outside tests/ and smoke() that executes oracle/) -------------------
def _oracle_batch(c, n, seed, cores):
    sys.path.insert(0, os.path.join(_ROOT, "tests"))
    import numpy as np
    import oracle_lib as O
    mode = {"NORMAL": O.MODE_NORMAL, "TRAIN_SHOOTING": O.MODE_TRAIN_SHOOTING, "TRAIN_DEFENSE": O.MODE_TRAIN_DEFENSE}[c["mode"]]
    pol = {"strong": O.POL_STRONG, "weak": O.POL_WEAK, "random": O.POL_RANDOM, "zero": O.POL_ZERO,
           "actor": O.POL_STRONG}  # CPU legs: the actor's GEMMs are not part of the env path; a strong BasicOpponent stands in
    b = O.OracleBatch(n, mode=mode, seed=seed, n_threads=cores)
    b.reset(one_starting=(np.arange(n) % 2).astype(np.int8))
    return b, pol[c["p1"]], pol[c["p2"]]


def _oracle_preroll(b, p1, p2):
    """Pre-roll to the stationary episode-phase mix; returns TOI events per env-step of the last 100-tick window."""
    b.rollout(PREROLL_TICKS - 200, p1, p2)
    rate = []
    for _ in range(12):
        b.clear_stats()
        b.rollout(100, p1, p2)
        s = b.stats()
        rate.append(s[12] / max(s[4], 1))
        if len(rate) >= 2 and abs(rate[-1] - rate[-2]) <= 0.2 * max(rate[-2], 1e-9):
            break
    b.clear_stats()
    return rate[-1]


def run_reference(args, rank, world):
    """Reference arm for this tier: the CPU implementation of the path (the oracle restatement of hockey_env.py + the
    Box2D step; the reference's own pybox2d build is not installable here, DESIGN.md section 1) on all host threads, same
    workload; one step = one tick of a bounded sample of the batch, advanced in rollout chunks."""
    if rank != 0:
        return
    c = resolve(args, world)
    cores = os.cpu_count() or 1
    n = min(c["n"], 2048 * cores)
    b, p1, p2 = _oracle_batch(c, n, args.seed, cores)
    toi_tail = _oracle_preroll(b, p1, p2)
    chunk = 5
    for _ in range((args.warmup + chunk - 1) // chunk):
        b.rollout(chunk, p1, p2)
    b.clear_stats()
    done, t0 = 0, time.perf_counter()
    while done < args.steps:
        k = min(chunk, args.steps - done)
        b.rollout(k, p1, p2)
        done += k
    dt = time.perf_counter() - t0
    s = b.stats()
    value = n * args.steps / dt
    sample = f"{n} of {c['n']} envs x {args.steps} ticks in rollout chunks of {chunk}, {cores} threads"
    print(json.dumps({
        "impl": "reference", "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": c["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, c, world),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "episode_stats": {"episodes": s[0], "env_steps": s[4], "toi_events_per_step": s[12] / max(s[4], 1),
                          "toi_events_per_step_preroll_tail": toi_tail},
    }), flush=True)


def cpu_baseline(args, c, budget_s=12.0):
    """Oracle ("port") timed on the host cores on a bounded sample of the same workload, in steady state."""
    cores = os.cpu_count() or 1
    n = min(c["n"], 256 * cores)
    b, p1, p2 = _oracle_batch(c, n, args.seed, cores)
    _oracle_preroll(b, p1, p2)
    steps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s:
        b.rollout(25, p1, p2)
        steps += 25
    dt = time.perf_counter() - t0
    return {"value": n * steps / dt, "unit": "env-steps/s", "cores": cores, "kind": "port",
            "sample": f"{n} of {c['n']} envs x {steps} ticks after a {PREROLL_TICKS}+ tick pre-roll, {cores} threads, {dt:.1f} s"}


def dump_outputs(out_dir, arrays, rank, world):
    """--dump-outputs: writes what the last timed step returned to its caller as out_dir/<name>.npy (float32), in global
    env order (gathered from all ranks), so that two builds can be compared output for output.  env_index.npy (float64)
    names the rows: all envs, or, when that would exceed DUMP_BYTES, one fixed seeded sample of them for every array."""
    import numpy as np
    import torch
    import torch.distributed as dist
    arrays = {k: v.to(torch.float32).contiguous() for k, v in arrays.items()}
    if world > 1:
        for k, v in arrays.items():
            g = v.new_empty((world * v.shape[0],) + tuple(v.shape[1:]))
            dist.all_gather_into_tensor(g, v)
            arrays[k] = g
    if rank != 0:
        return None
    total = next(iter(arrays.values())).shape[0]
    row_bytes = 8 + sum(4 * v[0].numel() for v in arrays.values())
    rows = min(total, DUMP_BYTES // row_bytes)
    idx = np.arange(total)
    if rows < total:
        idx = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(total, rows, replace=False))
    dev_idx = torch.from_numpy(idx).to(next(iter(arrays.values())).device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v.index_select(0, dev_idx).cpu().numpy())
    return {"dir": out_dir, "arrays": ["env_index"] + sorted(arrays), "rows": int(rows), "of_envs": int(total)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="normal65k", choices=sorted(CONFIGS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (overrides the config's size)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-l2-flush", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--actor-impl", default="fused", choices=["fused", "torch"],
                    help="config actor262k: the fused tcgen05 kernel (hk_actor_forward) or the fp32 torch module")
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--e2e-mode", default="copy", choices=["copy", "overlap", "zero_copy"],
                    help="HockeyVecEnv.step_host mode: one D2H copy of the packed record after the tick (default), DMA of the fast "
                         "tier's rows overlapped with the general tier, or zero-copy stores only")
    ap.add_argument("--rollout-k", type=int, default=64, help="ticks per hk_rollout call of the fused-rollout leg (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import hockey_env_b200 as hk

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    c = resolve(args, world)
    n = c["n"]
    mode = hk.Mode[c["mode"]]
    actor = None
    if c["p1"] == "actor":
        module = hk.load_td3_actor(os.path.join(_ROOT, "tests", "golden", "td3_actors.npz"), device=dev, name="stage_3")
        actor = module if args.actor_impl == "torch" else hk.FusedActor(module, device=dev)
    env = hk.HockeyVecEnv(n, mode=mode, device=dev, seed=args.seed, env_id_offset=rank * n,
                          p1=None if actor is not None else c["p1"], p2=c["p2"])
    env.reset(one_starting=(torch.arange(n, device=dev) % 2).to(torch.int8))
    flush = None if args.no_l2_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ev_actor = []

    def tick(timed=False):
        """Returns what the step hands its caller: HockeyVecEnv.step's tuple and player 1's actions (None if in-kernel)."""
        if actor is None:
            return env.step(), None
        with torch.no_grad():
            if timed:
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
            a = actor(env.obs)
            if timed:
                a1.record()
                ev_actor.append((a0, a1))
            return env.step(a), a

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- untimed pre-roll to the stationary episode-phase mix --------------------------------------------------------------
    def advance(k):
        if actor is None:
            env.rollout(k, c["p1"], c["p2"])
        else:
            for _ in range(k):
                tick()

    advance(PREROLL_TICKS - 200)
    rates = []
    for _ in range(12):
        env.clear_stats()
        advance(100)
        s = env.stats()
        rates.append(s["toi_events"] / max(s["env_steps"], 1))
        if len(rates) >= 2 and abs(rates[-1] - rates[-2]) <= 0.2 * max(rates[-2], 1e-9):
            break
    preroll_ticks = PREROLL_TICKS - 200 + 100 * len(rates)

    for _ in range(args.warmup):
        tick()
    env.clear_stats()
    env.kernel_timing(True)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for k in range(args.steps):
        if flush is not None:
            flush.zero_()
        ev[k][0].record()
        last = tick(timed=True)
        ev[k][1].record()
    barrier()
    clocks = sampler.stop()
    dumped = None
    if args.dump_outputs:  # before the legs below step the env again and overwrite its output buffers
        (obs, reward, done, truncated, info), action = last
        arrays = {"obs": obs, "reward": reward, "done": done, "truncated": truncated}
        arrays.update({f"info_{k}": v for k, v in info.items()})
        if action is not None:
            arrays["action"] = action
        dumped = dump_outputs(args.dump_outputs, arrays, rank, world)
    kernel_ms = sum(a.elapsed_time(b) for a, b in ev)
    actor_ms = sum(a.elapsed_time(b) for a, b in ev_actor)
    ktimes, ksteps = env.kernel_times()
    env.kernel_timing(False)
    t = torch.tensor([kernel_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    kernel_ms = float(t.item())
    value = world * n * args.steps / (kernel_ms * 1e-3)
    st = env.stats_tensor()

    # ---- fused rollout (hk_rollout): K ticks per call, no per-tick outputs -- reported beside the headline, never as it ----
    rollout = None
    if args.rollout_k > 0 and actor is None:
        calls = max(2, min(8, (args.steps + args.rollout_k - 1) // args.rollout_k))
        env.rollout(args.rollout_k, c["p1"], c["p2"])
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(calls):
            env.rollout(args.rollout_k, c["p1"], c["p2"])
        r1.record()
        barrier()
        t = torch.tensor([r0.elapsed_time(r1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rollout = {"value": world * n * calls * args.rollout_k / (float(t.item()) * 1e-3), "unit": "env-steps/s",
                   "k_steps": args.rollout_k, "calls": calls,
                   "note": "hk_rollout: in-kernel policies, auto-reset, statistics only (no per-tick outputs, no L2 flush)"}

    # ---- end to end through the public API with HOST buffers.  Same workload as the device-timed leg: player 1's actions
    # come from pinned host memory every tick (H2D inside the timed region), obs/reward/done/info go back to pinned host
    # memory every tick, host sync every tick (what a host-side agent does).  To keep the dynamics those of the named
    # workload, player 1's policy (the vectorised BasicOpponent / uniform noise / the actor) is run closed-loop ONCE,
    # untimed, from a snapshot of the steady state and its actions are recorded to host memory; the timed pass restores
    # the snapshot and replays them from the host, which reproduces that trajectory exactly.
    e2e = None
    if not args.no_e2e:
        p2 = c["p2"]
        e2e_env = hk.HockeyVecEnv(n, mode=mode, device=dev, seed=args.seed + 1, env_id_offset=rank * n, p2=p2)
        obs, _ = e2e_env.reset(one_starting=(torch.arange(n, device=dev) % 2).to(torch.int8))
        if actor is not None:
            policy = lambda o: actor(o)
        elif c["p1"] == "random":
            gen = torch.Generator(device=dev)
            gen.manual_seed(args.seed + rank)
            policy = lambda o: torch.rand((n, 4), device=dev, generator=gen) * 2 - 1
        else:
            host_opp = hk.BasicOpponent(weak=c["p1"] == "weak")
            policy = lambda o: host_opp.act(o)
        e2e_warm = max(3, args.warmup)
        e2e_steps = max(1, min(args.e2e_steps, (512 << 20) // (16 * n) - e2e_warm))
        with torch.no_grad():
            for _ in range(PREROLL_TICKS):
                obs, *_ = e2e_env.step(policy(obs).contiguous())
            snap = e2e_env.get_full_state()
            h_acts = torch.empty((e2e_warm + e2e_steps, n, 4), dtype=torch.float32).pin_memory()
            for k in range(e2e_warm + e2e_steps):
                a = policy(obs).contiguous()
                h_acts[k].copy_(a)
                obs, *_ = e2e_env.step(a)
        e2e_env.set_full_state(snap)
        host = e2e_env.host_buffers()
        for k in range(e2e_warm):
            e2e_env.step_host(h_acts[k], host, mode=args.e2e_mode)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(e2e_steps):
            e2e_env.step_host(h_acts[e2e_warm + k], host, mode=args.e2e_mode)  # H2D, tick, D2H, stream sync
        e1.record()
        barrier()
        same = bool(torch.equal(host["host"]["obs"], obs.cpu()))  # the replay ended where the recording pass ended
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": world * n * e2e_steps / (float(t.item()) * 1e-3), "unit": "env-steps/s",
               "h2d_bytes_per_step": n * 16, "d2h_bytes_per_step": e2e_env.host_bytes_per_step(),
               "steps": e2e_steps, "ms_per_step": float(t.item()) / e2e_steps, "replay_matches_recording": same,
               "note": "HockeyVecEnv.step_host: player-1 actions from pinned host memory (recorded closed-loop from the same "
                       f"steady state: p1 = {c['p1']}), obs/reward/done/info "
                       + {"overlap": "reach pinned host memory by a DMA of the fast tier's rows that overlaps the general tier plus the "
                                     "general tier's own stores into the mapped record (hk_step_host)",
                          "copy": "are packed and copied with ONE D2H copy to pinned host memory",
                          "zero_copy": "are stored by the kernels straight into mapped pinned host memory"}[args.e2e_mode]
                       + f", host sync every tick; player 2 = in-kernel {p2}", "mode": args.e2e_mode}
        e2e_env.close()

    # ---- end-of-run statistics: the only collective on this path (NCCL all-reduce of 16 doubles)
    if world > 1:
        dist.all_reduce(st, op=dist.ReduceOp.SUM)
    st = st.cpu().tolist()

    if rank == 0:
        peak, peak_src = _peaks()
        ms_tick = kernel_ms / args.steps
        algo = ALGO_BYTES_EXTERNAL if actor is not None else ALGO_BYTES_FUSED
        # dominant kernel = the one with the largest summed device time in the timed region (events on the launching stream)
        dom = max(ktimes, key=lambda k: ktimes[k])
        dom_ms = ktimes[dom] / max(ksteps, 1)
        # units one launch of it processes: all envs for k_fast, the queued envs for the general tier
        gen_units = st[14] / max(args.steps * world, 1)
        units = float(n) if dom == "k_fast" else gen_units
        achieved = algo * units / (dom_ms * 1e-3) / 1e9
        cap = _capture(args.config)
        issue = None
        if cap and cap.get("warp_inst_per_tick"):
            issue = {"achieved": cap["warp_inst_per_tick"] / (ms_tick * 1e-3), "peak": ISSUE_PEAK_WARP_INST_PER_S, "unit": "warp-inst/s",
                     "frac": cap["warp_inst_per_tick"] / (ms_tick * 1e-3) / ISSUE_PEAK_WARP_INST_PER_S,
                     "capture_frac": cap["warp_inst_per_tick"] / (cap["capture_ms_per_tick"] * 1e-3) / ISSUE_PEAK_WARP_INST_PER_S
                     if cap.get("capture_ms_per_tick") else None,
                     "note": f"warp instructions per tick from the steady-state ncu capture of this build ({cap.get('source')}), "
                             "divided by the tick time measured in this run; capture_frac uses the capture run's own tick time"}
        out = {
            "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_tick, "higher_is_better": True, "scaling": c["scaling"],
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, c, world),
            "e2e": e2e,
            "rollout": rollout,
            # kernels of this repo launched in the timed region: k_fast (+ k_touch) + the general tier(s) per tick
            "gpu_launches": args.steps * (env.launches_per_step() + (1 if actor is not None and args.actor_impl == "fused" else 0)),
            "clocks": clocks,
            "kernel_ms_per_tick": {k: v / max(ksteps, 1) for k, v in ktimes.items()},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": cap.get("dram_bytes_per_launch") if cap else None,
                         "traffic_unit": "dram bytes per launch of the dominant kernel (ncu --set full capture of this build, profiles/)",
                         "algorithmic_bytes_per_env_step": algo, "units_per_launch": units,
                         "algorithmic_bytes_per_launch": algo * units, "kernel_ms_per_launch": dom_ms,
                         "stored_bytes_per_env_step": STORED_BYTES_FUSED + (32 if actor is not None else 0),
                         "whole_tick": {"achieved": algo * n / (ms_tick * 1e-3) / 1e9, "frac": algo * n / (ms_tick * 1e-3) / 1e9 / peak,
                                        "note": "all kernels of the tick, all envs"},
                         "peak_source": peak_src, "issue": issue,
                         "note": "achieved = SURVEY 8(d) algorithmic bytes x env-steps one launch of the dominant kernel completes / "
                                 "its mean launch duration (CUDA events on the launching stream, this run); the path is "
                                 "latency/issue bound, not HBM-bound (DESIGN.md section 4)"},
            "episode_stats": {"episodes": st[0], "wins": st[1], "losses": st[2], "draws": st[3], "env_steps": st[4],
                              "mean_len": st[8] / max(st[0], 1), "velocity_iters_per_step": st[11] / max(st[4], 1),
                              "toi_events_per_step": st[12] / max(st[4], 1), "overflows": st[13],
                              "general_tier_share": st[14] / max(st[4], 1),
                              "toi_events_per_step_preroll_tail": rates[-1], "preroll_ticks": preroll_ticks},
        }
        if actor is not None:
            out["actor"] = {"impl": "fused tcgen05 kernel (hk_actor_forward: TF32 layer 1, bf16 layers 2-3, fp32 accumulation in TMEM)"
                            if args.actor_impl == "fused" else "torch fp32 module (cuBLAS GEMMs + elementwise tanh)",
                            "ms_per_step": actor_ms / args.steps, "share_of_step": actor_ms / max(kernel_ms, 1e-9),
                            "weights": "tests/golden/td3_actors.npz:stage_3 (pretrained/stage_3/models/td3_best.pt)",
                            "flops_per_env": 2 * (18 * 256 + 256 * 256 + 256 * 4)}
        if dumped is not None:
            out["dump_outputs"] = dumped
        if st[0] <= 0:
            out["warning"] = "no episode finished in the timed region"
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(args, c)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
