"""Time PPO's feed-forward minibatch update step from stored wire rows: the fused actor and critic (FusedPPO.evaluate,
FusedValue.evaluate) against torch float32 on env.expand_wire's observations, eager and as a CUDA graph; the fused
kernels and the torch reductions alone; and the recurrent step (tools/rppo_update_time.py's) with the head fused or in
torch.

    python tools/ppo_update_time.py --rows 65536 1048576 --latent 128 248 [--out OUT.jsonl]

Every pass overwrites L2 first (a 512 MB buffer is written) and is timed with CUDA events; each line is the median of
--reps passes, with the card's name and power limit read in the same run.  The feed-forward step is: actor z and critic
v, env.ppo_loss (K = 1), 0.5 MSE of v, backward, Adam over both networks."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def mlp(obs_len, L, out, dev, tail):
    lin = torch.nn.Linear
    return torch.nn.Sequential(lin(obs_len, L), torch.nn.Tanh(), lin(L, L), torch.nn.Tanh(), lin(L, out), *tail).to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[65536, 1048576])
    ap.add_argument("--latent", type=int, nargs="+", default=[128, 248])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import evgsim
    from evgsim import _capi, policy
    from rppo_update_time import make_actor
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda", 0)
    name = card()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    # stored rows: 4 turns of a 4096-match self-play env, repeated to the batch
    src = evgsim.BatchedEvergladesEnv(4096, device=0, seed=1, auto_reset=_capi.AUTORESET_NEXT)
    src.reset(obs_format="wire")
    torch.manual_seed(0)
    play = policy.FusedPPO(src, mlp(src.obs_len, 64, 132, dev, [torch.nn.Tanh(), torch.nn.Softmax(dim=-1)]))
    store = []
    for _ in range(4):
        store.append(src.obs_rows("wire").clone())
        play(obs_format="wire")
        src.step(src._actions, obs_format="wire")
    store = torch.cat(store)
    env = src
    lines = []

    def timed(fn, before=None):
        ts = []
        for i in range(a.reps + 3):
            if before:
                before()
            flush.fill_(i & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2]

    def record(**kw):
        d = dict(card=name, **kw)
        lines.append(d)
        print(json.dumps(d), flush=True)

    for R in a.rows:
        M = R // 2
        rows = store.repeat((M + store.shape[0] - 1) // store.shape[0], 1)[:M].contiguous()
        gen = torch.Generator(device=dev).manual_seed(R)
        idx = torch.stack([torch.randperm(132, device=dev, generator=gen)[:7] for _ in range(64)]).repeat(R // 64, 1)
        old = -torch.rand((R, 7), device=dev, generator=gen) * 5
        adv = torch.randn(R, device=dev, generator=gen)
        ret = torch.randn(R, device=dev, generator=gen)
        for L in a.latent:
            torch.manual_seed(L)
            actor = mlp(env.obs_len, L, 132, dev, [torch.nn.Tanh(), torch.nn.Softmax(dim=-1)])
            critic = mlp(env.obs_len, L, 1, dev, [])
            fa, fc = policy.FusedPPO(env, actor), policy.FusedValue(env, critic)
            params = list(actor.parameters()) + list(critic.parameters())
            old_ = old.clone()

            def loss(kind):
                if kind == "fused":
                    z, v = fa.evaluate(rows), fc.evaluate(rows).view(-1)
                else:
                    obs = env.expand_wire(rows).view(-1, env.obs_len)
                    z, v = actor[:-2](obs), critic(obs).view(-1)
                surr, ent, _ = env.ppo_loss(z, idx, old_, adv, clip=0.2)
                return surr.mean() - 0.01 * ent.mean() + 0.5 * torch.nn.functional.mse_loss(v, ret)

            for kind in ("fused", "torch_f32"):
                opt = torch.optim.Adam(params, lr=1e-6, capturable=True)

                def run():
                    opt.zero_grad(set_to_none=False)
                    loss(kind).backward()
                    opt.step()
                run()
                record(rows=R, latent=L, case="ff_step_%s_eager" % kind, ms=round(timed(run), 4))
                s = torch.cuda.Stream()
                s.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s):
                    for _ in range(2):
                        run()
                torch.cuda.current_stream().wait_stream(s)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    run()
                record(rows=R, latent=L, case="ff_step_%s_graph" % kind, ms=round(timed(graph.replay), 4))
                del graph
            # the fused pieces alone: each network's pack + forward kernel, the backward kernel, the torch reductions
            for net, fused, mod in (("actor", fa, actor), ("critic", fc, critic)):
                kind = _capi.PPO_TRAIN_ACTOR if net == "actor" else _capi.PPO_TRAIN_CRITIC
                prm = list(mod.parameters())
                f = policy._ff_train_function()
                out_dim = 132 if net == "actor" else 1
                with torch.no_grad():
                    record(rows=R, latent=L, case="fused_%s_forward_pack_and_kernel" % net,
                           ms=round(timed(lambda: f.apply(rows, fused, kind, _capi.OBS_WIRE, -1, out_dim, *prm)), 4))
            h = torch.rand((R, L), device=dev, generator=gen)
            g2 = torch.randn((R, L), device=dev, generator=gen)
            dd2, dd1 = torch.empty_like(h), torch.empty_like(h)
            import ctypes as C
            p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
            w2t = policy._ff_train_images(fa, _capi.PPO_TRAIN_ACTOR)[3]
            record(rows=R, latent=L, case="fused_backward_kernel", bytes_moved_per_row=4 * 5 * L,
                   ms=round(timed(lambda: _capi.check(env._lib.evg_ppo_train_backward(env._h, R, L, p(w2t), p(g2), p(h), p(h), p(dd2), p(dd1),
                                                                                      env._stream()))), 4))
            obs = env.expand_wire(rows).view(-1, env.obs_len)
            dz = torch.randn((R, 132), device=dev, generator=gen)
            w3 = actor[4].weight.detach()

            def reductions():
                bf = lambda t: t.to(torch.bfloat16).float()  # noqa: E731
                return (dz @ bf(w3), dd1.t() @ bf(obs), dd1.sum(0), dd2.t() @ bf(h), dd2.sum(0), dz.t() @ bf(h), dz.sum(0),
                        env.expand_wire(rows))
            record(rows=R, latent=L, case="fused_actor_torch_reductions_and_expand", ms=round(timed(reductions), 4))
            del actor, critic, fa, fc, params, obs
        # the recurrent step at 65,536 rows: head fused or in torch, the GRU fused (FusedRPPO.evaluate) in both
        if R <= 65536:
            for L in a.latent:
                ractor = make_actor(env.obs_len, L, dev)
                fr = policy.FusedRPPO(env, ractor)
                h0 = torch.rand((R, L), device=dev, generator=gen) * 2 - 1
                opt = torch.optim.Adam(ractor.parameters(), lr=1e-6)

                def rstep(kind):
                    def run():
                        opt.zero_grad(set_to_none=True)
                        x = fr.evaluate_head(rows) if kind == "fused" else ractor.action_head(env.expand_wire(rows).view(-1, env.obs_len))
                        surr, ent, _ = env.ppo_loss(fr.evaluate(x, h0), idx, old, adv, clip=0.2)
                        (surr.mean() - 0.01 * ent.mean()).backward()
                        opt.step()
                    return run
                for kind in ("fused", "torch_f32"):
                    record(rows=R, latent=L, case="rppo_step_head_%s_eager" % kind, ms=round(timed(rstep(kind)), 4))
    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
