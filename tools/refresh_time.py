#!/usr/bin/env python
"""What it costs to keep a fused policy's weight images current during training.  One JSON line per case, each with the
GPU's name and power limit:

- refresh: FusedDQN / FusedPPO / FusedRPPO.refresh() (evg_pack_*: one kernel, no host sync), CUDA events around 200
  back-to-back calls after 5 warm-up calls; DQN 105 -> 528 -> 132, PPO and the recurrent actor at L = 128 and 248.
  Beside it the alternative without it, constructing the wrapper again (parameters to the host, numpy packing, images
  back), host clock around 10 constructions each ending in a device synchronise, and the bytes one refresh writes.
- dqn_training_turn: DQN's online-training turn at `matches` matches as a CUDA graph of refresh -> forward -> decode ->
  step, against the same graph without refresh: the per-turn price of acting with the current network.  Both graphs
  replayed 300 times per round, alternating, 3 rounds; the median round of each.

    python tools/refresh_time.py [matches=32768]
"""
import json
import os
import statistics
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import evgsim
from evgsim import policy
from tools.policy_rollout import RecurrentActor
from tools.ppo_time import gpu_info, timed_us


def build(kind, latent):
    torch.manual_seed(0)
    if kind == "dqn":
        net = torch.nn.Sequential(torch.nn.Linear(105, 528), torch.nn.ReLU(), torch.nn.Linear(528, 132))
        return net.cuda(), (lambda env: policy.FusedDQN(env, net))
    if kind == "ppo":
        net = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                                  torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
        return net.cuda(), (lambda env: policy.FusedPPO(env, net))
    net = RecurrentActor(latent).cuda()
    return net, (lambda env: policy.FusedRPPO(env, net))


def image_bytes(fused):
    ts = [fused._w1, fused._w2] if isinstance(fused, policy.FusedDQN) else fused._w
    return sum(t.numel() * t.element_size() for t in ts)


def rebuild_ms(make, env, reps=10):
    for _ in range(2):
        make(env)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        make(env)
        torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps * 1e3


def graph_of(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    return g


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
    gpu = gpu_info()
    env = evgsim.BatchedEvergladesEnv(1024, seed=0)
    env.reset()
    for kind, latent in (("dqn", 528), ("ppo", 128), ("ppo", 248), ("rppo", 128), ("rppo", 248)):
        net, make = build(kind, latent)
        fused = make(env)
        print(json.dumps({"gpu": gpu, "case": "refresh", "policy": kind, "hidden" if kind == "dqn" else "latent": latent,
                          "refresh_us": timed_us(fused.refresh, reps=200), "rebuild_ms": rebuild_ms(make, env),
                          "bytes_written": image_bytes(fused)}), flush=True)

    env = evgsim.BatchedEvergladesEnv(n, seed=0, auto_reset=1)
    env.reset()
    net, make = build("dqn", 528)
    fused = make(env)

    def turn():
        fused()
        env.step(env._actions)

    def turn_with_refresh():
        fused.refresh()
        turn()

    graphs = {"without_refresh": graph_of(turn), "with_refresh": graph_of(turn_with_refresh)}
    times = {k: [] for k in graphs}
    reps = 300
    for _ in range(3):
        for k, g in graphs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                g.replay()
            b.record()
            torch.cuda.synchronize()
            times[k].append(a.elapsed_time(b) / reps * 1e3)
    med = {k: statistics.median(v) for k, v in times.items()}
    print(json.dumps({"gpu": gpu, "case": "dqn_training_turn", "matches": n, "hidden": 528,
                      "turn_us": med["without_refresh"], "turn_with_refresh_us": med["with_refresh"],
                      "refresh_cost_us": med["with_refresh"] - med["without_refresh"], "rounds_us": times}), flush=True)


if __name__ == "__main__":
    main()
