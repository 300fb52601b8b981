"""Time the recurrent PPO actor's minibatch update step: the fused GRU + action layer (FusedRPPO.evaluate) against
cuDNN's GRU in float32 (torch's defaults), cuDNN under bf16 autocast, and a plain 7-step torch loop without cuDNN.

    python tools/rppo_update_time.py --rows 65536 --latent 128 248 [--out OUT.jsonl] [--profile PROFILE.txt]

Every pass overwrites L2 first (a 512 MB buffer is written) and is timed with CUDA events; each line is the median of
--reps passes.  One JSON line per (latent, case), with the card's name and power limit, on stdout and, with --out,
into that file.  --profile runs the cuDNN float32 step once more under torch.profiler, separately from the timings, and
writes the kernels' time split.
The step is: head (Linear-Tanh x 2) forward, the GRU and action_layer[0], env.ppo_loss (K = 7), backward, Adam."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def make_actor(obs_len, L, dev, seed=0):
    torch.manual_seed(seed)
    a = torch.nn.Module()
    a.action_head = torch.nn.Sequential(torch.nn.Linear(obs_len, L), torch.nn.Tanh(), torch.nn.Linear(L, L), torch.nn.Tanh())
    a.action_gru = torch.nn.GRU(L, L)
    a.action_layer = torch.nn.Sequential(torch.nn.Linear(L, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
    return a.to(dev)


def z_cudnn(actor, x, h0):
    out, _ = actor.action_gru(x.unsqueeze(0).expand(7, -1, -1).contiguous(), h0.unsqueeze(0))
    return actor.action_layer[0](out).permute(1, 0, 2).contiguous()


def z_loop(actor, x, h0):
    g = actor.action_gru
    L = x.shape[1]
    gi = torch.nn.functional.linear(x, g.weight_ih_l0, g.bias_ih_l0)
    h, zs = h0, []
    for _ in range(7):
        gh = torch.nn.functional.linear(h, g.weight_hh_l0, g.bias_hh_l0)
        r = torch.sigmoid(gi[:, :L] + gh[:, :L])
        u = torch.sigmoid(gi[:, L:2 * L] + gh[:, L:2 * L])
        n = torch.tanh(gi[:, 2 * L:] + r * gh[:, 2 * L:])
        h = (1 - u) * n + u * h
        zs.append(actor.action_layer[0](h))
    return torch.stack(zs, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=65536)
    ap.add_argument("--latent", type=int, nargs="+", default=[128, 248])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    import evgsim
    from evgsim import policy
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda", 0)
    env = evgsim.BatchedEvergladesEnv(64, device=0, seed=1)
    env.reset()
    name = card()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    R = a.rows
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

    for L in a.latent:
        actor = make_actor(env.obs_len, L, dev)
        fused = policy.FusedRPPO(env, actor)
        gen = torch.Generator(device=dev).manual_seed(L)
        obs = torch.rand((R, env.obs_len), device=dev, generator=gen)
        h0 = torch.rand((R, L), device=dev, generator=gen) * 2 - 1
        idx = torch.randint(0, 132, (R, 7), device=dev, generator=gen)
        old = -torch.rand((R, 7), device=dev, generator=gen) * 5
        adv = torch.randn(R, device=dev, generator=gen)
        opt = torch.optim.Adam(actor.parameters(), lr=1e-6)

        def step(kind):
            def run():
                opt.zero_grad(set_to_none=True)
                x = actor.action_head(obs)
                if kind == "fused":
                    z = fused.evaluate(x, h0)
                elif kind == "cudnn_bf16":
                    with torch.autocast("cuda", dtype=torch.bfloat16):
                        z = z_cudnn(actor, x, h0)
                    z = z.float().contiguous()
                elif kind == "loop":
                    z = z_loop(actor, x, h0)
                else:
                    z = z_cudnn(actor, x, h0)
                surr, ent, _ = env.ppo_loss(z, idx, old, adv, clip=0.2)
                (surr.mean() - 0.01 * ent.mean()).backward()
                opt.step()
            return run

        def record(case, ms, **kw):
            d = dict(card=name, rows=R, latent=L, case=case, ms=round(ms, 4), **kw)
            lines.append(d)
            print(json.dumps(d), flush=True)

        # the fused pieces alone
        x = actor.action_head(obs).detach().contiguous()
        z = torch.empty((R, 7, 132), device=dev)
        h = torch.empty((R, 7, L), device=dev)
        p = policy._rppo_params(actor)[4:]
        record("fused_forward_pack_and_kernel", timed(lambda: fused._train_forward(x, h0, *p, z, h)))
        dz = torch.randn((R, 7, 132), device=dev, generator=gen) * 1e-3
        w3b = p[4].detach().to(torch.bfloat16).float()
        g0 = (dz.view(-1, 132) @ w3b).view(R, 7, L)
        g = torch.empty_like(g0)
        dgh = torch.empty((R, 7, 3 * L), device=dev)
        s = torch.empty((R, 3 * L), device=dev)
        record("fused_backward_kernel", timed(lambda: fused._train_backward(x, h0, h, g, dgh, s), before=lambda: g.copy_(g0)),
               bytes_written_per_row=4 * (7 * 3 * L + 3 * L))

        def reductions():
            bf = lambda t: t.to(torch.bfloat16).float()  # noqa: E731
            d = dgh.view(-1, 3 * L)
            hp = bf(torch.cat([h0.unsqueeze(1), h[:, :6]], 1)).view(-1, L)
            return (dz.view(-1, 132) @ w3b, s @ bf(p[0].detach()), s.t() @ bf(x), s.sum(0), d.t() @ hp, d.sum(0),
                    dz.view(-1, 132).t() @ bf(h).view(-1, L), dz.sum((0, 1)))
        record("fused_weight_grad_reductions_torch_fp32", timed(reductions))
        for kind in ("fused", "cudnn_f32", "cudnn_bf16", "loop"):
            record("step_" + kind, timed(step(kind)))
        del x, z, h, dgh, s, g, g0

        if a.profile:
            from torch.profiler import ProfilerActivity, profile
            run = step("cudnn_f32")
            run()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run()
                torch.cuda.synchronize()
            tot, rnn, rows = 0.0, 0.0, []
            for ev in prof.key_averages():
                t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                if t <= 0:
                    continue
                tot += t
                if any(w in ev.key.lower() for w in ("rnn", "gru", "cudnn", "persist", "lstm")):
                    rnn += t
                rows.append((t, ev.key))
            rows.sort(reverse=True)
            with open(a.profile, "a") as f:
                f.write("# %s, %d rows, L = %d: cuDNN float32 step, device time %.3f ms, cuDNN RNN kernels %.3f ms (%.1f %%)\n"
                        % (name, R, L, tot / 1e3, rnn / 1e3, 100 * rnn / max(tot, 1e-9)))
                for t, k in rows[:25]:
                    f.write("%10.3f ms  %s\n" % (t / 1e3, k[:140]))
    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
