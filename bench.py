#!/usr/bin/env python
"""bench.py — env-turns/sec of the batched Everglades turn step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs-per-gpu E] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

It runs what __graft_entry__.build() compiled and writes nothing into the tree (the tree may be read-only).

One "step" = one game turn for every match of the batch: the random_actions agent kernel for both
players + the turn-step kernel (--agents fused: one launch of evg_step_agents does both).  Workload (config.workload): BASELINE.json configs[4] at
N = 1 — DemoMap, both players random_actions, 1,048,576 lock-step matches per GPU with in-place
auto-reset; matches shard across ranks with NO collective on the step path (weak scaling; the
only exchange is an end-of-run all_gather of episode statistics).

Before anything is timed the batch is SETTLED into its steady state (--phase staggered, the default): one episode
of untimed turns during which block b (128 consecutive matches) is reset after turn b mod 150, so that afterwards
every phase of the game is present in equal shares and a timed window of ANY length sees the same mix of marching,
fighting and in-place resets — the full-episode mean, not whichever turns the window happens to cover.  Inside a
block the matches stay in lock-step, as they do in this workload (99.6 % of random-vs-random matches run to the turn
limit, so matches started together end together).  --phase staggered-match offsets every single match instead (32
different game phases inside every warp: a harder, artificial mix, reported in profiles/); --phase lockstep keeps all
matches on the same turn.

Printed JSON (rank 0, one line): value = device-timed whole-job env-turns/s with state and inputs
resident in HBM; e2e = the same metric through the public host-buffer API (pinned host actions
H2D + step + D2H of every match's observations/rewards/done flags each step, in the packed wire
format of include/evgsim.h by default; e2e_f32 = the same with float32 observation vectors);
roofline = the step kernel's algorithmic bytes FOR THE TURNS THAT WERE TIMED (1331 B + 16 B per
unit slot that fought, counted on the device) / its CUDA-event duration against the measured HBM
peak; cpu_baseline = the unmodified Python reference (oracle/_ref, staged by oracle/stage_ref.py)
on all host cores, with the C oracle port (oracle/evg_oracle.c) next to it.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env_turns_per_sec"
UNIT = "env-turns/s"
# Algorithmic bytes per match-turn (SURVEY.md §8d / DESIGN.md §4.4): 1331 B fixed (state 227 B read +
# written, actions 28 B, observations 840 B, rewards 8 B, done 1 B) + 16 B (8 read + 8 written) per unit
# slot of the groups that fought that turn.  The slots are COUNTED ON THE DEVICE over the timed turns
# (EvgEpisodeStats.fought_unit_slots), not assumed: a full random-vs-random episode averages 21.6.
B_ALG_FIXED = 1331
B_ALG_PER_FOUGHT_SLOT = 16
# --dump-outputs: at most this many matches, drawn with a fixed seed, so that two builds run with the same arguments
# dump the same matches.  A match's outputs take at most 892 B as float32 (obs 840, reward 8, done and status 4 each,
# scores 8, action rows 28 where the step returns them), so the dump stays under 64 MB.
DUMP_MATCHES = 65536
DUMP_SEED = 1234


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=450)   # 3 full 150-turn episodes
    ap.add_argument("--warmup", type=int, default=150)  # 1 episode
    ap.add_argument("--envs-per-gpu", type=int, default=1 << 20)
    ap.add_argument("--total-envs", type=int, default=0,
                    help="strong scaling: this many matches in total, split evenly over the ranks (overrides --envs-per-gpu)")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--phase", default="staggered", choices=["staggered", "staggered-match", "lockstep"],
                    help="staggered: settle so that block b of 128 consecutive matches is b mod 150 turns into its game (every phase "
                         "of the game present at once, lock-step inside a block); staggered-match: match i is i mod 150 turns in "
                         "(32 different phases inside every warp); lockstep: all matches on the same turn")
    ap.add_argument("--e2e-format", default="wire", choices=["wire", "i16", "f32"],
                    help="observation transport of the headline e2e number (all lossless; f32 is always reported as e2e_f32 too)")
    ap.add_argument("--agents", default="kernel", choices=["kernel", "fused"],
                    help="random_actions rows from the agent kernel (2 launches/step) or generated inside the step kernel (1 launch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (observations, rewards, done flags and "
                         "the info arrays) for a fixed sample of rank 0's matches as DIR/<name>.npy, float32, plus the "
                         "sampled match ids as DIR/match_id.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path's outputs; --impl reference has none")
    return args


def workload_config(args, world):
    return {
        "workload": "DemoMap random_actions self-match, %d lock-step matches per GPU, auto-reset "
                    "(BASELINE.json configs[4] at N=1; weak-scaled over ranks)" % args.envs_per_gpu,
        "envs_per_gpu": args.envs_per_gpu, "total_envs": args.envs_per_gpu * world,
        "map": "DemoMap.json", "agents": "random_actions vs random_actions (on-device, Philox tape; %s)" % args.agents,
        "turn_limit": 150, "auto_reset": "terminal-obs", "seed": args.seed,
        "phase": {"staggered": "staggered: the matches of block b (128 consecutive matches) are (b mod 150) turns into their games "
                               "when timing starts (settled over 150 untimed turns), lock-step inside a block",
                  "staggered-match": "staggered-match: match i is (i mod 150) turns into its game when timing starts",
                  "lockstep": "lockstep: every match on the same game turn"}[args.phase],
        "l2": "resident state %.2f GB/GPU >> 126 MB L2; no flush between steps" % (args.envs_per_gpu * (256 + 1600) / 1e9),
        "parallelism": "match-sharded x%d, no step-path collective" % world,
    }


# ------------------------------------------------------------------------------------------------
# CPU oracle port on the host cores (cpu_baseline leg and --impl reference arm)
# ------------------------------------------------------------------------------------------------
def cpu_oracle_rate(seconds, seed=0, threads=None, turns=150):
    """Time oracle/evg_oracle.c (evo_run_random: both players random_actions, in-place reset) on
    `threads` host threads for about `seconds`.  Returns (env_turns_per_s, threads, sample, elapsed)."""
    import evgsim
    from oracle import evg_oracle as eo

    cfg = evgsim.load_config()
    threads = threads or os.cpu_count() or 1
    eo.lib()
    t0 = time.perf_counter()
    n, _, _ = eo.run_random(cfg, seed, 0, 64, turns)  # calibration, single thread
    per_thread_rate = n / (time.perf_counter() - t0)
    matches = max(16, int(per_thread_rate * seconds / turns))
    results = [0] * threads

    def work(k):
        results[k] = eo.run_random(cfg, seed, 1_000_000 + k * matches, matches, turns)[0]

    ths = [threading.Thread(target=work, args=(k,)) for k in range(threads)]
    t0 = time.perf_counter()
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    el = time.perf_counter() - t0
    total = sum(results)
    sample = "%d threads x %d matches x %d turns of the same workload (oracle/evg_oracle.c, gcc -O2)" % (threads, matches, turns)
    return total / el, threads, sample, el


def cpu_reference_rate(seconds):
    """The UNMODIFIED Python reference (oracle/_ref or /root/reference) on all host cores: env-turns/s through its own
    EvergladesEnv.reset/step.  Returns None where no copy of the reference is present."""
    from oracle import ref_harness as rh
    if not rh.reference_available():
        return None
    rate, procs, rate_one, sample = rh.time_reference(seconds)
    return {"value": rate, "unit": UNIT, "cores": procs, "kind": "reference", "sample": sample,
            "one_process": rate_one, "source": rh.REFERENCE_ROOT}


def cpu_baselines(seconds, seed):
    """cpu_baseline (the real reference when a copy is present, else the port) and the port line next to it."""
    rate, threads, sample, _ = cpu_oracle_rate(seconds, seed=seed)
    port = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample}
    try:
        ref = cpu_reference_rate(seconds)
    except Exception as e:  # a broken multiprocessing setup must not cost the GPU line
        print("[bench] timing the Python reference failed: %r" % (e,), file=sys.stderr)
        ref = None
    return (ref or port), port


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores — the unmodified
    Python server + gym wrapper staged under oracle/_ref (one process per core), each step a bounded sample of the
    same workload; the compiled C restatement (the oracle port) is reported next to it as `cpu_baseline_port`."""
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    budget = min(30.0, max(5.0, 0.03 * (steps + warm)))
    t0 = time.perf_counter()
    main_line, port = cpu_baselines(budget, args.seed)
    rate = main_line["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "i32/f64", "data": "synthetic", "config": workload_config(args, world),
        "cpu_baseline": main_line, "cpu_baseline_port": port,
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "elapsed_s": time.perf_counter() - t0,
    }
    _emit(line)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons of one GPU, polled through NVML from a thread for the whole run (started before
    the warm-up); `report(t0, t1)` summarises the samples whose timestamps fall inside the timed region."""
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, device):
        self.samples = []  # (perf_counter, sm_mhz, reasons bitmask)
        self.stop_flag = False
        self.thread = None
        self.h = None
        self.max_mhz = None
        try:
            import pynvml
            import torch
            self.nv = pynvml
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(device).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                idx = int(vis.split(",")[device.index]) if vis and vis.split(",")[0].isdigit() else device.index
                self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:
            print("[bench] NVML unavailable: %r" % (e,), file=sys.stderr)
            self.h = None

    def _poll(self):
        nv = self.nv
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = reasons_fn(self.h)
                self.samples.append((time.perf_counter(), float(mhz), int(rs)))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.h is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=2)

    def report(self, t0, t1):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0, "source": "NVML, polled every ~2 ms"}
        inside = [x for x in self.samples if t0 <= x[0] <= t1]
        if not inside and self.samples:
            # a region shorter than one poll: the nearest samples on either side of it
            before = [x for x in self.samples if x[0] < t0][-2:]
            after = [x for x in self.samples if x[0] > t1][:2]
            inside = before + after
            out["source"] += "; region shorter than a poll, nearest samples used"
        if inside:
            mhz = sorted(x[1] for x in inside)
            bits = 0
            for x in inside:
                bits |= x[2]
            out.update(sm_mhz=mhz[len(mhz) // 2], samples=len(inside), reasons=sorted(k for k, v in self.BAD.items() if bits & v))
        return out


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(envs_per_gpu, phase):
    """DRAM bytes per step-kernel launch (dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture)
    for THIS batch size and phase mix from profiles/step_kernel_traffic.json, else None: traffic measured on another
    batch size or another part of the game is not this run's traffic."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")))
        for c in d.get("captures", []):
            if int(c["envs"]) == int(envs_per_gpu) and c.get("phase") == phase:
                return float(c["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


def capture_outputs(step_out, first):
    """Host copies of what one step returned, (obs, reward, done, info), for --dump-outputs: the rows of min(N,
    DUMP_MATCHES) matches drawn with DUMP_SEED (sorted), every array as float32 (the integer ones hold values far below
    2**24, so the conversion is exact), and the global ids of those matches as float64."""
    import numpy as np
    import torch

    obs, rew, done, info = step_out
    n = obs.shape[0]
    idx = np.arange(n)
    if n > DUMP_MATCHES:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_MATCHES, replace=False))
    sel = torch.as_tensor(idx, device=obs.device)
    out = {"match_id": (first + idx).astype(np.float64)}
    for name, t in [("obs", obs), ("reward", rew), ("done", done)] + sorted(info.items()):
        out[name] = t.index_select(0, sel).cpu().numpy().astype(np.float32)
    return out


def write_outputs(directory, arrays):
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
def _emit(line: dict) -> None:
    """The ONE JSON line goes to the real stdout; everything else any library prints (NCCL's version banner,
    build messages) was diverted to stderr by _quiet_stdout()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def _quiet_stdout() -> None:
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def main():
    args = parse_args()
    _quiet_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.scaling = "weak"
    if args.total_envs:
        assert args.total_envs % (world * 128) == 0, "--total-envs must split into whole 128-match blocks per rank"
        args.envs_per_gpu = args.total_envs // world
        args.scaling = "strong"
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    import evgsim
    from evgsim import dist as evd

    assert torch.cuda.is_available(), "bench.py measures the CUDA path; no GPU visible"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    E = args.envs_per_gpu
    first, _ = rank * E, E
    clocks = ClockSampler(dev)
    clocks.start()  # before the warm-up: a poll thread needs no start-up time inside the timed region
    env = evgsim.BatchedEvergladesEnv(E, device=dev, seed=args.seed, auto_reset=evgsim._capi.AUTORESET_TERMINAL,
                                      env_id_offset=first)
    env.reset()
    stream = torch.cuda.current_stream(dev)
    TL = env.num_turns

    fused = args.agents == "fused"

    def one_step():
        if fused:
            env.step_agents()                   # ONE launch: both players' random_actions rows + the whole turn
        else:
            env.step(env.random_actions())      # agent kernel, then the turn-step kernel

    # ---- settle into the steady state (untimed, not part of --warmup): after turn t the matches with i mod TL == t
    # start over, so match i ends up (TL - 1 - i mod TL) turns into its game and every phase is equally represented
    if args.phase != "lockstep":
        phase_of = torch.arange(E, device=dev, dtype=torch.int32)
        phase_of = (phase_of // 128 if args.phase == "staggered" else phase_of) % TL
        for t in range(TL):
            one_step()
            env.reset(mask=(phase_of == t))
        del phase_of
    for _ in range(args.warmup):
        one_step()
    torch.cuda.synchronize(dev)

    # ---- device-timed region: EXACTLY K steps, barrier + synchronize on both sides
    K = args.steps
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    stats0 = env.episode_stats()
    launches0 = env.launch_count
    wall0 = time.perf_counter()
    torch.cuda.profiler.start()  # `ncu --profile-from-start off` then lists exactly the timed region's launches
    t_begin.record(stream)
    for k in range(K):
        a = None if fused else env.random_actions()
        ev[k][0].record(stream)
        if fused:
            out = env.step_agents()
        else:
            out = env.step(a)
        ev[k][1].record(stream)
    t_end.record(stream)
    torch.cuda.synchronize(dev)
    torch.cuda.profiler.stop()
    wall1 = time.perf_counter()
    # the step's tensors are overwritten by the steps below: copy the last timed step's outputs now
    dumped = capture_outputs(out, first) if args.dump_outputs and rank == 0 else None
    if world > 1:
        dist.barrier()
    clk = clocks.report(wall0, wall1)
    launches = env.launch_count - launches0
    stats1 = env.episode_stats()
    fought = stats1["fought_unit_slots"] - stats0["fought_unit_slots"]  # unit slots that fought in the K timed turns
    step_kernel_name = {0: "evg_step_kernel (warp per match)",
                        1: "evg_step_tpm_kernel (thread per match)"}.get(env._lib.evg_step_kernel_kind(env._h), "?")
    total_ms = t_begin.elapsed_time(t_end)
    step_kernel_ms = sum(a.elapsed_time(b) for a, b in ev) / K

    # ---- end-to-end through the public host-buffer API (pinned host memory, copies inside)
    Ke = max(1, min(args.e2e_steps, K))
    ring = []
    for _ in range(4):  # pre-drawn host-side action rows (random_actions ignores observations)
        ring.append(env.random_actions().cpu().pin_memory())
        env.step(env._actions)

    def time_e2e(fmt):
        from evgsim import hostmem
        env.host_buffers(fmt)
        placement = hostmem.last_placement()
        for _ in range(3):
            env.step_host(ring[0], obs_format=fmt)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sink = 0.0
        e0.record(stream)
        for k in range(Ke):
            obs_h, rew_h, done_h, _ = env.step_host(ring[k % 4], sync=True, obs_format=fmt)
            sink += float(obs_h[0, 0].sum()) + float(rew_h[0, 0])  # the host reads the step's result
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1), placement

    def d2h_probe(nbytes):
        """Plain pinned D2H copy of as many bytes as the headline e2e format moves per step: the link's own speed."""
        from evgsim import hostmem
        src = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        dst = hostmem.pinned_empty((nbytes,), torch.uint8, dev.index)
        for _ in range(2):
            dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(5):
            dst.copy_(src, non_blocking=True)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / 5

    e2e_ms, placement = time_e2e(args.e2e_format)
    e2e_f32_ms, _ = time_e2e("f32") if args.e2e_format != "f32" else (e2e_ms, None)
    probe_ms = d2h_probe(env.d2h_bytes_per_step(args.e2e_format))
    clocks.stop()

    # ---- extra (not the metric): the same self-play as ONE launch per 150-turn rollout (evg_rollout: the batch stays in
    # shared memory between turns, only the last turn's observations are written) — what a consumer that needs no
    # per-turn observations gets (scripted evaluation matches, BASELINE.json configs[1] and [2])
    KR = 150
    env.rollout(10, evgsim._capi.AGENT_RANDOM, evgsim._capi.AGENT_RANDOM)
    torch.cuda.synchronize(dev)
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record(stream)
    env.rollout(KR, evgsim._capi.AGENT_RANDOM, evgsim._capi.AGENT_RANDOM)
    r1.record(stream)
    torch.cuda.synchronize(dev)
    rollout_ms = r0.elapsed_time(r1)

    # ---- max over ranks
    t = torch.tensor([total_ms, step_kernel_ms, e2e_ms, e2e_f32_ms, probe_ms, rollout_ms], dtype=torch.float64, device=dev)
    f = torch.tensor([fought], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(f, op=dist.ReduceOp.SUM)
    total_ms, step_kernel_ms, e2e_ms, e2e_f32_ms, probe_ms, rollout_ms = (float(x) for x in t.tolist())
    fought_all = int(f.item())
    stats = evd.gather_episode_stats(stats1, device=dev)  # the only collective; not timed

    if rank == 0:
        total_envs = E * world
        value = total_envs * K / (total_ms / 1e3)
        e2e_value = total_envs * Ke / (e2e_ms / 1e3)
        peak, peak_src = measured_hbm_peak()
        slots_per_env_turn = fought_all / float(total_envs * K)
        b_alg = B_ALG_FIXED + B_ALG_PER_FOUGHT_SLOT * slots_per_env_turn
        achieved = E * b_alg / (step_kernel_ms / 1e3) / 1e9  # GB/s per GPU, step kernel alone
        d2h = env.d2h_bytes_per_step(args.e2e_format)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "i32/f64", "data": "synthetic", "config": workload_config(args, world),
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": env.h2d_bytes_per_step() * world,
                    "d2h_bytes_per_step": d2h * world, "steps": Ke, "ms_per_step": e2e_ms / Ke,
                    "obs_format": args.e2e_format,
                    "api": "BatchedEvergladesEnv.step_host(obs_format=%r) (evg_step_host_fmt), pinned host buffers; the host gets "
                           "every match's observations (lossless; evgsim.wire.expand == the float32 vector), rewards and done flags" % args.e2e_format,
                    "pinned_placement": placement,
                    "link": {"d2h_probe_ms": probe_ms, "d2h_probe_gbs_per_gpu": d2h / (probe_ms / 1e3) / 1e9,
                             "e2e_d2h_gbs_per_gpu": d2h / (e2e_ms / Ke / 1e3) / 1e9,
                             "note": "a plain pinned D2H copy of the same bytes per step on every rank at once: what the host link "
                                     "allows; e2e_d2h_gbs_per_gpu / d2h_probe_gbs_per_gpu is how close the step gets to it"}},
            "e2e_f32": {"value": total_envs * Ke / (e2e_f32_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_f32_ms / Ke,
                        "d2h_bytes_per_step": env.d2h_bytes_per_step("f32") * world, "obs_format": "f32"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": step_kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(E, args.phase), "peak_source": peak_src,
                         "bytes_per_env_turn": b_alg, "fought_unit_slots_per_env_turn": slots_per_env_turn,
                         "bytes_formula": "1331 + 16 * fought unit slots per env-turn, slots counted on the device over the timed turns",
                         "kernel_ms": step_kernel_ms, "kernel_env_turns_per_s": E / (step_kernel_ms / 1e3)},
            "episode_stats": stats,
            "scripted_rollout": {"value": total_envs * KR / (rollout_ms / 1e3), "unit": UNIT, "turns_per_launch": KR,
                                 "note": "extra, not the metric: evg_rollout, one launch per 150 turns of the same self-play; "
                                         "only the last turn's observations are written"},
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"], line["cpu_baseline_port"] = cpu_baselines(args.cpu_seconds, args.seed)
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
