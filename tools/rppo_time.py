#!/usr/bin/env python
"""Time of the fused recurrent PPO actor (evg_policy_rppo: head, 7 GRU steps, 7 draws, unravel and the state update in
one kernel) against the torch path of tools/policy_rollout.py --policy rppo --dtype bf16 (bf16 head, cuDNN GRU over 7
steps, output layer, torch.multinomial(probs, 1) per step, evg_decode_indices), each piece of the latter timed alone
too.  CUDA events around 50 back-to-back calls after 5 warm-up calls; mid-game observations (40 random turns).  Prints
one JSON line with the GPU's name and power limit, and the fused kernel's weight stream: the bytes of bf16 weights each
128-row tile reads from L2 (W1 + W2 once, then per step the six GRU matrices and W3) and that total over the kernel time.

    python tools/rppo_time.py [matches=32768] [latent=128]
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import evgsim
from evgsim import policy
from tools.policy_rollout import RecurrentActor
from tools.ppo_time import gpu_info, timed_us


def weight_bytes_per_tile(latent):
    """bf16 bytes the kernel streams per tile: W1 [Lp x 128], W2 [Lp x Ka], per step W_i and W_h (3 x [Lp x Ka] each)
    and W3 [144 x Ka], padded as the images are."""
    lp, ka = -(-latent // 16) * 16, -(-latent // 64) * 64
    return 2 * (lp * 128 + lp * ka + 7 * (6 * lp * ka + 144 * ka))


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
    latent = int(sys.argv[2]) if len(sys.argv) > 2 else 128
    env = evgsim.BatchedEvergladesEnv(n, seed=0, auto_reset=1)
    env.reset()
    for _ in range(40):
        env.step(env.random_actions())
    torch.manual_seed(0)
    actor = RecurrentActor(latent).cuda().eval()
    fused = policy.FusedRPPO(env, actor)
    nb = RecurrentActor(latent).cuda().to(torch.bfloat16).eval()
    nb.load_state_dict(actor.state_dict())
    x = env.obs.view(-1, 105)
    hidden = torch.zeros((1, 2 * n, latent), dtype=torch.bfloat16, device=env.device)
    with torch.no_grad():
        probs, _ = nb(x.to(torch.bfloat16), hidden)
        probs = probs.float().view(-1, 132)
        head = nb.action_head(x.to(torch.bfloat16))
        seq = head.unsqueeze(0).expand(7, -1, -1).contiguous()
        out, _ = nb.action_gru(seq, hidden)
    idx = torch.multinomial(probs, 1).view(7, n, 2).permute(1, 2, 0).contiguous()

    @torch.no_grad()
    def torch_turn():
        p, h = nb(x.to(torch.bfloat16), hidden)
        hidden.copy_(h)
        i = torch.multinomial(p.float().view(-1, 132), 1).view(7, n, 2).permute(1, 2, 0).contiguous()
        return env.decode_indices(i, div=12, mod=11)

    fused_us = timed_us(fused)
    tiles = -(-2 * n // 128)
    stream = weight_bytes_per_tile(latent) * tiles
    with torch.no_grad():
        print(json.dumps({"gpu": gpu_info(), "rows": 2 * n, "latent": latent,
                          "fused_rppo_us": fused_us, "fused_rppo_with_logp_us": timed_us(lambda: fused(want_logp=True)),
                          "fused_rppo_with_logp_and_hidden_in_us": timed_us(lambda: fused(want_logp=True, want_hidden_in=True)),
                          "fused_rppo_with_probs_us": timed_us(lambda: fused(want_probs=True)),
                          "weight_stream_bytes": stream, "weight_stream_gb_per_s": stream / fused_us / 1e3,
                          "torch_bf16_head_us": timed_us(lambda: nb.action_head(x.to(torch.bfloat16))),
                          "torch_bf16_gru_us": timed_us(lambda: nb.action_gru(seq, hidden)),
                          "torch_bf16_layer_us": timed_us(lambda: nb.action_layer(out)),
                          "torch_multinomial_us": timed_us(lambda: torch.multinomial(probs, 1)),
                          "decode_indices_us": timed_us(lambda: env.decode_indices(idx, div=12, mod=11)),
                          "torch_path_us": timed_us(torch_turn)}))


if __name__ == "__main__":
    main()
