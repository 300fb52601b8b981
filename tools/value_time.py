#!/usr/bin/env python
"""Time of the fused PPO critic (evg_policy_value) on float32 observations and on wire rows, against torch's float32 and
bf16 forward of the same Sequential(Linear(105, L), Tanh, Linear(L, L), Tanh, Linear(L, 1)) on the same observations.
CUDA events around 50 back-to-back calls after 5 warm-up calls; mid-game observations (40 random turns, stepped in the
wire format and expanded, so both inputs hold the same state).  Prints one JSON line with the GPU's name and power limit.

    python tools/value_time.py [matches=32768] [latent=128]
"""
import copy
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch
import evgsim
from evgsim import policy
from ppo_time import gpu_info, timed_us


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
    latent = int(sys.argv[2]) if len(sys.argv) > 2 else 128
    env = evgsim.BatchedEvergladesEnv(n, seed=0, auto_reset=1)
    env.reset(obs_format="wire")
    for _ in range(40):
        env.step(env.random_actions(), obs_format="wire")
    env.expand_wire(env.obs_rows("wire"), out=env.obs)
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                              torch.nn.Linear(latent, 1)).cuda().eval()
    critic = policy.FusedValue(env, net)
    nb = copy.deepcopy(net).to(torch.bfloat16)
    x = env.obs.view(-1, 105)
    with torch.no_grad():
        v = critic().clone()
        diff = (v.view(-1) - net(x).view(-1)).abs().max().item()
        assert torch.equal(critic(obs_format="wire"), v)
        print(json.dumps({"gpu": gpu_info(), "matches": n, "rows": 2 * n, "latent": latent,
                          "fused_value_f32_us": timed_us(critic), "fused_value_wire_us": timed_us(lambda: critic(obs_format="wire")),
                          "torch_fp32_forward_us": timed_us(lambda: net(x)),
                          "torch_bf16_forward_us": timed_us(lambda: nb(x.to(torch.bfloat16))),
                          "max_abs_diff_vs_torch_fp32": diff}))


if __name__ == "__main__":
    main()
