#!/usr/bin/env python
"""CUDA-event times of the policy-in-the-loop turn's kernels with float32 observations against wire rows.

    python tools/wire_policy_time.py [--envs 32768 1048576] [--reps 20]

One JSON line per measurement, each with the card's name and power limit:
- the step (evg_step_fmt) writing float32 observations against writing wire rows;
- each fused policy (evg_policy_mlp, evg_policy_ppo and evg_policy_rppo at L = 128 and 248) on float32 against on wire;
- evg_wire_expand of every row without an index and through a random permutation, in GB/s of the bytes it must move
  (rows read + float32 observations written + reward and done + the index) against 6,538 GB/s, a device-to-device
  copy measured on a B200.
Each pair is timed alternating, the mean over --reps launches of each, after a warm-up of both.  At 32,768 matches the
float32 observations (27.5 MB) stay in the 126 MB L2 between step and policy; at 1,048,576 (880 MB) they do not."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import evgsim
from evgsim import policy

COPY_GBS = 6538.0


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return {"gpu": torch.cuda.get_device_name(0), "power_limit": pl}


def timed(fns, reps):
    """mean ms per call of each function in fns, alternating them call by call"""
    for f in fns:
        f()
    torch.cuda.synchronize()
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)] for _ in fns]
    for r in range(reps):
        for i, f in enumerate(fns):
            ev[i][r][0].record()
            f()
            ev[i][r][1].record()
    torch.cuda.synchronize()
    return [sum(a.elapsed_time(b) for a, b in e) / reps for e in ev]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[32768, 1048576])
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    info = card()
    for n in args.envs:
        env = evgsim.BatchedEvergladesEnv(n, seed=1)
        env.reset()
        env.reset(obs_format="wire")
        rows = env.obs_rows("wire")
        acts = env.random_actions().clone()

        def emit(what, f32_ms, wire_ms, **kw):
            print(json.dumps(dict(info, envs=n, kernel=what, f32_ms=round(f32_ms, 4), wire_ms=round(wire_ms, 4),
                                  wire_over_f32=round(wire_ms / f32_ms, 4), **kw)), flush=True)

        # the step: the turn counter moves on, the matches' state stays mid-game (auto-reset off keeps every match alive)
        t = timed([lambda: env.step(acts), lambda: env.step(acts, obs_format="wire")], args.reps)
        emit("evg_step", *t, obs_bytes_f32=n * 2 * env.obs_len * 4, obs_bytes_wire=rows.numel())
        env.expand_wire(rows, out=env.obs)  # both inputs describe the same state
        torch.manual_seed(0)
        dqn = torch.nn.Sequential(torch.nn.Linear(105, 528), torch.nn.ReLU(), torch.nn.Linear(528, 132)).cuda()
        f = policy.FusedDQN(env, dqn)
        t = timed([lambda: f.forward_t(), lambda: f.forward_t(obs_format="wire")], args.reps)
        emit("evg_policy_mlp", *t, rows=2 * n)
        for latent in (128, 248):
            ppo = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                                      torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1)).cuda()
            p = policy.FusedPPO(env, ppo)
            t = timed([lambda: p(), lambda: p(obs_format="wire")], args.reps)
            emit("evg_policy_ppo", *t, rows=2 * n, latent=latent)
            actor = torch.nn.Module()
            actor.action_head = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
            actor.action_gru = torch.nn.GRU(latent, latent)
            actor.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
            actor.cuda()
            q = policy.FusedRPPO(env, actor)
            t = timed([lambda: q(), lambda: q(obs_format="wire")], max(3, args.reps // 4))
            emit("evg_policy_rppo", *t, rows=2 * n, latent=latent)
            del p, q
        perm = torch.randperm(n, device=env.device)
        out = torch.empty_like(env.obs)
        reward = torch.empty_like(env.reward)
        done = torch.empty_like(env.done)
        t = timed([lambda: env.expand_wire(rows, out=out, reward=reward, done=done),
                   lambda: env.expand_wire(rows, index=perm, out=out, reward=reward, done=done)], args.reps)
        moved = rows.numel() + out.numel() * 4 + n * 9
        for name, ms, extra in (("evg_wire_expand", t[0], 0), ("evg_wire_expand indexed", t[1], n * 8)):
            gbs = (moved + extra) / ms / 1e6
            print(json.dumps(dict(info, envs=n, kernel=name, ms=round(ms, 4), bytes=moved + extra, gb_per_s=round(gbs, 1),
                                  of_copy_bandwidth=round(gbs / COPY_GBS, 3))), flush=True)
        del env, f
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
