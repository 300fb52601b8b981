#!/usr/bin/env python
"""CUDA-event kernel times of the fused PPO actors with and without their optional outputs, at 32,768 matches (65,536
rows, both players), L = 128 and 248, on float32 observations and on wire rows:

    python tools/logp_time.py [--envs 32768] [--reps 20] [--rounds 3]

  none      the call as a rollout that keeps only the draws makes it
  logp      want_logp (each draw's log-probability, [N, 2, 7] float32)
  logp_hin  want_logp + want_hidden_in (evg_policy_rppo only: the state each row started from, [N, 2, L] float32)
  probs     want_probs ([N, 2, 132] / [N, 2, 7, 132] float32)

The variants of one (actor, L, format) are timed alternating call by call (tools/wire_policy_time.py's timed), the mean
over --reps calls each, and the whole comparison is repeated --rounds times so that the spread between rounds can be
read next to the differences between variants.  One JSON line per (actor, L, format, round), with the card's name and
power limit.  Mid-game observations (30 random turns); the rppo state is carried from call to call."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import evgsim
from evgsim import policy
from tools.wire_policy_time import card, timed


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    info = card()
    n = args.envs
    env = evgsim.BatchedEvergladesEnv(n, seed=1)
    env.reset(obs_format="wire")
    for _ in range(30):
        env.step(env.random_actions(), obs_format="wire")
    env.expand_wire(env.obs_rows("wire"), out=env.obs)  # both inputs describe the same state
    for kind in ("ppo", "rppo"):
        for latent in (128, 248):
            torch.manual_seed(0)
            if kind == "ppo":
                net = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                                          torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
                f = policy.FusedPPO(env, net)
                variants = {"none": {}, "logp": {"want_logp": True}, "probs": {"want_probs": True}}
            else:
                from tools.policy_rollout import RecurrentActor
                f = policy.FusedRPPO(env, RecurrentActor(latent))
                variants = {"none": {}, "logp": {"want_logp": True}, "logp_hin": {"want_logp": True, "want_hidden_in": True},
                            "probs": {"want_probs": True}}
            for fmt in ("f32", "wire"):
                fns = [lambda kw=kw: f(obs_format=fmt, **kw) for kw in variants.values()]
                for rnd in range(args.rounds):
                    ms = timed(fns, args.reps)
                    print(json.dumps(dict(info, kernel="evg_policy_" + kind, rows=2 * n, latent=latent, obs_format=fmt, round=rnd,
                                          **{v + "_us": round(t * 1e3, 2) for v, t in zip(variants, ms)})), flush=True)


if __name__ == "__main__":
    main()
