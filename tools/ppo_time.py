#!/usr/bin/env python
"""Time of the fused PPO actor (evg_policy_ppo: forward, sampling and unravel in one kernel) against the torch path of
tools/policy_rollout.py --policy ppo --dtype bf16 (bf16 forward, torch.multinomial without replacement, evg_decode_indices),
each piece of the latter timed alone too.  CUDA events around 50 back-to-back calls after 5 warm-up calls; mid-game
observations (40 random turns).  Prints one JSON line with the GPU's name and power limit.

    python tools/ppo_time.py [matches=32768] [latent=128]
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import evgsim
from evgsim import policy


def timed_us(fn, reps=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e3


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
    latent = int(sys.argv[2]) if len(sys.argv) > 2 else 128
    env = evgsim.BatchedEvergladesEnv(n, seed=0, auto_reset=1)
    env.reset()
    for _ in range(40):
        env.step(env.random_actions())
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                              torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1)).cuda()
    fused = policy.FusedPPO(env, net)
    nb = net.to(torch.bfloat16).eval()
    x = env.obs.view(-1, 105)
    probs = nb(x.to(torch.bfloat16)).float()
    idx = torch.multinomial(probs, 7, replacement=False)

    @torch.no_grad()
    def torch_turn():
        p = nb(x.to(torch.bfloat16)).float()
        i = torch.multinomial(p, 7, replacement=False)
        return env.decode_indices(i.view(n, 2, 7), div=12, mod=11)

    print(json.dumps({"gpu": gpu_info(), "rows": 2 * n, "latent": latent,
                      "fused_ppo_us": timed_us(fused), "fused_ppo_with_logp_us": timed_us(lambda: fused(want_logp=True)),
                      "fused_ppo_with_probs_us": timed_us(lambda: fused(want_probs=True)),
                      "torch_bf16_forward_us": timed_us(lambda: nb(x.to(torch.bfloat16))),
                      "torch_multinomial_us": timed_us(lambda: torch.multinomial(probs, 7, replacement=False)),
                      "decode_indices_us": timed_us(lambda: env.decode_indices(idx.view(n, 2, 7), div=12, mod=11)),
                      "torch_path_us": timed_us(torch_turn)}))


if __name__ == "__main__":
    main()
