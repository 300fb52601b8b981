#!/usr/bin/env python
"""Time of the fused PPO loss head (evg_ppo_loss + evg_ppo_loss_grad, BatchedEvergladesEnv.ppo_loss) against the same
loss in plain torch (tests/ppo_loss.py: torch_loss, float32), forward plus backward from z, eager and replayed from a
CUDA graph.  One JSON line per case, each naming the card and its power limit:

- "head": B in {65,536, 8,388,608} rows, K = 1 (z [B, 132]) and K = 7 (z [B, 7, 132]).  fused_us and torch_us are
  forward + backward to dz (torch.autograd.grad of surr and ent with given upstream gradients), fwd_us / bwd_us the two
  launches alone with outputs given.  Every timed pass is one CUDA event pair after a 256 MB buffer is overwritten, so no
  pass finds z in the 126 MB L2 (at B = 65,536 z is 35 MB for K = 1); the median of `reps` passes after 3 warm-up passes.
  bytes: from the shapes, what each launch must move: forward z (528 B a distribution) + idx 56 + old_logp 28 + adv 4
  + surr, ent, ratio 12 + logp 28 per row; backward z + dz (1,056 B a distribution) + idx 56 + adv, ratio, g_surr,
  g_ent 16 per row.  share = bytes / 7.7 TB/s (the data sheet's HBM3e bandwidth) / time: the memory-bound share.  A
  torch case that runs out of memory is reported as such, not timed.
- "step": one minibatch step of 65,536 rows, expand_wire of stored wire rows -> actor up to its last Linear -> loss head
  -> backward -> Adam step, with the fused head and with the torch head (FusedPPO's actor, L = 128, and FusedRPPO's,
  whose GRU is stepped seven times from the stored hidden_in), eager.

    python tools/ppo_loss_time.py [reps=20]
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch
import evgsim
from ppo_loss import torch_loss
from ppo_time import gpu_info

N_ACT, CLIP, HBM = 132, 0.2, 7.7e12


def timed_us(fn, flush, reps):
    for _ in range(3):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        flush.add_(1)
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return sorted(a.elapsed_time(b) for a, b in ev)[reps // 2] * 1e3


def graphed(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):  # warm-up of the autograd path on a side stream, as torch.cuda.graph asks
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    torch.cuda.synchronize()
    return g.replay


def inputs(B, K, gen):
    dev = "cuda"
    shape = (B, N_ACT) if K == 1 else (B, 7, N_ACT)
    z = (torch.randn(shape, device=dev, generator=gen) * 1.5).requires_grad_(True)
    if K == 1:
        idx = torch.rand((B, N_ACT), device=dev, generator=gen).argsort(dim=1)[:, :7].contiguous()
    else:
        idx = torch.randint(0, N_ACT, (B, 7), device=dev, generator=gen)
    old = torch.randn((B, 7), device=dev, generator=gen) * 0.05 - 4.9
    adv = torch.randn(B, device=dev, generator=gen)
    gs, ge = torch.randn(B, device=dev, generator=gen), torch.randn(B, device=dev, generator=gen)
    return z, idx, old, adv, gs, ge


def head_cases(env, gpu, flush, reps):
    gen = torch.Generator(device="cuda").manual_seed(0)
    for K in (1, 7):
        for B in (65536, 8388608):
            z, idx, old, adv, gs, ge = inputs(B, K, gen)
            per_dist = 4 * N_ACT
            fwd_bytes = B * (K * per_dist + 56 + 28 + 4 + 12 + 28)
            bwd_bytes = B * (2 * K * per_dist + 56 + 16)

            def fused():
                surr, ent, _ = env.ppo_loss(z, idx, old, adv, clip=CLIP)
                return torch.autograd.grad((surr, ent), z, (gs, ge))

            def plain():
                surr, ent, _, _ = torch_loss(z, idx, old, adv, CLIP)
                return torch.autograd.grad((surr, ent), z, (gs, ge))

            zd = z.detach()
            o = [torch.empty(B, device="cuda") for _ in range(3)]
            logp = torch.empty((B, 7), device="cuda")
            dz = torch.empty_like(zd)
            n = N_ACT
            env._ppo_loss_launch(zd, idx, old, adv, CLIP, K, n, o[0], o[1], logp, o[2])
            out = {"kind": "head", "gpu": gpu, "rows": B, "K": K, "n": n, "fwd_bytes": fwd_bytes, "bwd_bytes": bwd_bytes}
            fwd_us = timed_us(lambda: env._ppo_loss_launch(zd, idx, old, adv, CLIP, K, n, o[0], o[1], logp, o[2]), flush, reps)
            bwd_us = timed_us(lambda: env._ppo_loss_grad_launch(zd, idx, adv, o[2], CLIP, K, n, gs, ge, dz), flush, reps)
            out.update(fwd_us=round(fwd_us, 2), bwd_us=round(bwd_us, 2), fwd_share=round(fwd_bytes / HBM / (fwd_us * 1e-6), 3),
                       bwd_share=round(bwd_bytes / HBM / (bwd_us * 1e-6), 3))
            out["fused_us"] = round(timed_us(fused, flush, reps), 2)
            out["fused_graph_us"] = round(timed_us(graphed(fused), flush, reps), 2)
            torch.cuda.empty_cache()
            d_fused = fused()[0]
            try:
                d_torch = plain()[0]
                out["max_abs_dz_diff_vs_torch"] = (d_fused - d_torch).abs().max().item()
                del d_torch, d_fused
                out["torch_us"] = round(timed_us(plain, flush, max(5, reps // 4)), 2)
                if B <= 65536:  # the graph's private pool would hold a second copy of every intermediate
                    out["torch_graph_us"] = round(timed_us(graphed(plain), flush, reps), 2)
            except torch.cuda.OutOfMemoryError:
                out["torch_us"] = "out of memory"
            d_fused = None
            print(json.dumps(out), flush=True)
            del z, idx, old, adv, gs, ge, zd, o, logp, dz, d_fused
            torch.cuda.empty_cache()


def step_cases(gpu, flush, reps, R=65536, latent=128):
    from evgsim import policy
    n = R // 2
    env = evgsim.BatchedEvergladesEnv(n, seed=0, auto_reset=evgsim._capi.AUTORESET_NEXT)
    env.reset(obs_format="wire")
    for _ in range(20):
        env.step(env.random_actions(), obs_format="wire")
    torch.manual_seed(0)
    for kind in ("ppo", "rppo"):
        if kind == "ppo":
            actor = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                                        torch.nn.Linear(latent, N_ACT), torch.nn.Tanh(), torch.nn.Softmax(dim=-1)).cuda()
            fused = policy.FusedPPO(env, actor)
            fused(obs_format="wire", want_logp=True)
            hidden_in = None
        else:
            actor = torch.nn.Module()
            actor.action_head = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
            actor.action_gru = torch.nn.GRU(latent, latent)
            actor.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, N_ACT), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
            actor = actor.cuda()
            fused = policy.FusedRPPO(env, actor)
            fused(obs_format="wire", want_logp=True, want_hidden_in=True)
            hidden_in = fused.hidden_in.view(1, R, latent).clone()
        rows = env.obs_rows("wire").clone()
        idx, logp = fused.idx.view(R, 7).clone(), fused.logp.view(R, 7).clone()
        adv = torch.randn(R, device="cuda")
        opt = torch.optim.Adam(actor.parameters(), lr=1e-5)

        def z_of():
            obs = env.expand_wire(rows).view(R, 105)
            if kind == "ppo":
                return actor[:-2](obs)
            x = actor.action_head(obs)
            out, _ = actor.action_gru(x.unsqueeze(0).expand(7, -1, -1).contiguous(), hidden_in)
            return actor.action_layer[0](out).permute(1, 0, 2).contiguous()

        def step(head):
            z = z_of()
            if head == "fused":
                surr, ent, _ = env.ppo_loss(z, idx, logp, adv, clip=CLIP)
            else:
                surr, ent, _, _ = torch_loss(z, idx, logp, adv, CLIP)
            opt.zero_grad()
            (surr.mean() - 0.01 * ent.mean()).backward()
            opt.step()

        res = {"kind": "step", "gpu": gpu, "actor": kind, "rows": R, "latent": latent}
        for head in ("fused", "torch"):
            res[head + "_step_us"] = round(timed_us(lambda: step(head), flush, reps), 1)
        print(json.dumps(res), flush=True)
    env.close()


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    gpu = gpu_info()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    env = evgsim.BatchedEvergladesEnv(8, seed=0)
    head_cases(env, gpu, flush, reps)
    step_cases(gpu, flush, reps)


if __name__ == "__main__":
    main()
