"""Time the recurrent actor's acting call (FusedRPPO, evg_policy_rppo) on one library, for A/B runs of a change that
must not move it: EVGSIM_LIB=<lib> python tools/rppo_act_time.py [--matches 32768] [--latent 128 248].
One JSON line per (latent, variant): the median of 50 calls timed with CUDA events, L2 overwritten before each."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--matches", type=int, default=32768)
    ap.add_argument("--latent", type=int, nargs="+", default=[128, 248])
    a = ap.parse_args()
    import evgsim
    from evgsim import policy
    env = evgsim.BatchedEvergladesEnv(a.matches, device=0, seed=2)
    env.reset()
    for _ in range(5):
        env.step(env.random_actions())
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=env.device)
    for L in a.latent:
        torch.manual_seed(L)
        actor = torch.nn.Module()
        actor.action_head = torch.nn.Sequential(torch.nn.Linear(env.obs_len, L), torch.nn.Tanh(), torch.nn.Linear(L, L), torch.nn.Tanh())
        actor.action_gru = torch.nn.GRU(L, L)
        actor.action_layer = torch.nn.Sequential(torch.nn.Linear(L, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
        fused = policy.FusedRPPO(env, actor.to(env.device))
        for variant, kw in (("plain", {}), ("logp_hidden_in", dict(want_logp=True, want_hidden_in=True))):
            ts = []
            for i in range(55):
                flush.fill_(i & 0xFF)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fused(**kw)
                e1.record()
                torch.cuda.synchronize()
                if i >= 5:
                    ts.append(e0.elapsed_time(e1))
            ts.sort()
            print(json.dumps(dict(lib=os.path.basename(evgsim._capi.lib_path()), rows=2 * a.matches, latent=L, variant=variant,
                                  ms=round(ts[len(ts) // 2], 4))), flush=True)


if __name__ == "__main__":
    main()
