"""evg_ppo_loss / evg_ppo_loss_grad (BatchedEvergladesEnv.ppo_loss) on the GPU: PPO's policy loss from the actor's last
Linear output, and its gradient.

1. Forward against the float64 statement within the derived bound (tests/ppo_loss.py: loss_bound), for K = 1 and 7 and
   n = 7, 132, 256, at batch sizes on each side of a CTA's rows and of one pass of the persistent grid; draws at 0 and
   n - 1, repeated draws for K = 7; clip 0, 0.2, 0.99; A negative, zero and positive; z = 0 (ent = log n) and +-20.
2. dz against torch's float64 autograd of the torch statement within grad_bound, on the rows whose clip branch the
   kernel's float32 ratio and the float64 one agree on; dz exactly +0 where both upstream gradients are 0, a clipped
   row's dz bit for bit its entropy part, and g_ent alone giving the entropy gradient alone.
3. The kernel's own logp fed back as old_logp: ratio == 1 and surr == -A bit for bit.
4. Stored wire-row rollouts of FusedPPO (self-play, and player 0 against the SwarmAgent) and FusedRPPO (hidden_in)
   re-evaluated in float32 torch: the new logp within LOGP_BF16 of the stored one, parameter gradients through the
   fused loss equal to those through the torch statement, then an optimiser step, refresh() and the next rollout.
5. A CUDA graph of the forward and backward launches replays the eager result; with outputs given they allocate
   nothing, and neither they nor the autograd path synchronise.
6. An index outside [0, n) gives a NaN row and a NaN dz row, the other rows unchanged; every ValueError of the wrapper
   comes before a launch, and the C ABI refuses every bad argument.

LOGP_BF16 = 0.1 per draw: the actors sample from their bf16 network, a float32 re-evaluation differs from it by rounding.
On the golden games' observations the largest gap of any log-probability between the bf16 statement
(policy.reference_forward_ppo / _rppo) and float32 is 0.023 (feed-forward, L = 128) and 0.013 (recurrent); a draw's
logp = log p_j - log T_k moves by at most twice that, and the tolerance doubles it again."""
import ctypes as C

import numpy as np
import pytest

from ppo_loss import clipped, grad_bound, grad_float64, loss_bound, loss_float64, torch_loss

pytestmark = pytest.mark.gpu

LOGP_BF16 = 0.1
CTA_ROWS = 8  # K = 1 forward: a warp per row, 8 warps a CTA; K = 7: a CTA per row


@pytest.fixture(scope="module")
def evg():
    import __graft_entry__ as g
    g.build()
    import evgsim
    return evgsim


@pytest.fixture(scope="module")
def env(evg):
    return evg.BatchedEvergladesEnv(8, seed=1)


@pytest.fixture(scope="module")
def sms(evg):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def bits(a):
    a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
    return np.ascontiguousarray(a).view(np.uint32)


def make_rows(rng, B, K, n):
    """z [B, n] or [B, 7, n] at scale 1.5 with rows of 0 and of +-20, draws with 0 and n - 1 among them (distinct for
    K = 1, repeats for K = 7), old_logp near log(1/n), A cycling through negative, zero and positive."""
    z = (rng.standard_normal((B, n) if K == 1 else (B, 7, n)) * 1.5).astype(np.float32)
    z[0::11] = 0.0
    z[5::11] = 20.0 * np.where(rng.random(z[5::11].shape) < 0.5, -1.0, 1.0)
    if K == 1:
        idx = np.argsort(rng.random((B, n)), axis=1)[:, :7].astype(np.int64)
        for b in range(1, B, 4):    # action 0 drawn first
            idx[b] = np.concatenate([[0], 1 + rng.permutation(n - 1)[:6]])
        for b in range(2, B, 4):    # action n - 1 drawn last
            idx[b] = np.concatenate([rng.permutation(n - 1)[:6], [n - 1]])
    else:
        idx = rng.integers(0, n, (B, 7)).astype(np.int64)
        idx[1::4] = idx[1::4, :1]          # the same draw seven times
        idx[2::4, 3], idx[3::4, 5] = 0, n - 1
    old = (rng.standard_normal((B, 7)) * 0.05 - np.log(n)).astype(np.float32)
    adv = rng.standard_normal(B).astype(np.float32) * 3
    adv[0::3] = -np.abs(adv[0::3])
    adv[1::3] = 0.0
    adv[2::3] = np.abs(adv[2::3])
    return z, idx, old, adv


def run(env, z, idx, old, adv, clip, requires_grad=False):
    import torch
    dev = env.device
    zt = torch.from_numpy(z).to(dev).requires_grad_(requires_grad)
    it, ot, at = (torch.from_numpy(x).to(dev) for x in (idx, old, adv))
    surr, ent, info = env.ppo_loss(zt, it, ot, at, clip=clip)
    return zt, surr, ent, info


def batch_sizes(K, sms):
    """One row, a CTA's rows and one more, and around one pass of the persistent grid at 3 and 4 resident CTAs an SM."""
    rows = CTA_ROWS if K == 1 else 1
    out = {1, 2, rows - 1, rows, rows + 1, 3 * sms * rows + 1, 4 * sms * rows - 1, 4 * sms * rows + 1}
    return sorted(b for b in out if b >= 1)


@pytest.mark.parametrize("K", [1, 7])
@pytest.mark.parametrize("n", [7, 132, 256])
def test_forward_within_the_derived_bound_of_float64(env, sms, K, n):
    rng = np.random.default_rng(100 * K + n)
    for B in batch_sizes(K, sms):
        z, idx, old, adv = make_rows(rng, B, K, n)
        for clip in (0.0, 0.2, 0.99):
            _, surr, ent, info = run(env, z, idx, old, adv, clip)
            got = [t.cpu().numpy() for t in (surr, ent, info["logp"], info["ratio"])]
            want = loss_float64(z, idx, old, adv, clip)
            bound = loss_bound(z, idx, old, adv, clip)
            for name, g, w, b in zip(("surr", "ent", "logp", "ratio"), got, want, bound):
                assert g.shape == w.shape and np.all(np.abs(g - w) <= b), (name, B, K, n, clip, np.max(np.abs(g - w) - b))
            assert np.all(np.abs(got[1][0::11] - np.log(n)) <= bound[1][0::11])  # z = 0: uniform


@pytest.mark.parametrize("K", [1, 7])
@pytest.mark.parametrize("n", [7, 132, 256])
def test_gradient_against_torch_float64_autograd(env, K, n):
    import torch
    rng = np.random.default_rng(7 * K + n)
    B = 517
    z, idx, old, adv = make_rows(rng, B, K, n)
    old += (rng.standard_normal((B, 7)) * 0.1).astype(np.float32)  # ratios on both sides of the clip range
    gs = rng.standard_normal(B).astype(np.float32)
    ge = rng.standard_normal(B).astype(np.float32)
    gs[3::10], ge[3::10] = 0.0, 0.0
    for clip in (0.0, 0.2, 0.99):
        zt, surr, ent, info = run(env, z, idx, old, adv, clip, requires_grad=True)
        dev = zt.device
        gst, get_ = torch.from_numpy(gs).to(dev), torch.from_numpy(ge).to(dev)
        dz, = torch.autograd.grad((surr, ent), zt, (gst, get_), retain_graph=True)
        r32 = info["ratio"].cpu().numpy()
        z64 = torch.tensor(z, dtype=torch.float64, requires_grad=True)
        s64, e64, _, r64 = torch_loss(z64, torch.from_numpy(idx), torch.from_numpy(old), torch.from_numpy(adv), clip)
        want, = torch.autograd.grad((s64, e64), z64, (torch.from_numpy(gs).double(), torch.from_numpy(ge).double()))
        want = want.numpy()
        r64 = r64.detach().numpy()
        same = clipped(r32, adv, clip) == clipped(r64, adv, clip)
        assert same.mean() > 0.95, (K, n, clip)
        b = grad_bound(z, idx, adv, r64, clip, old, gs, ge)
        d = dz.cpu().numpy()
        assert np.all(np.abs(d - want)[same] <= b[same]), (K, n, clip, np.max((np.abs(d - want) - b)[same]))
        # the analytic float64 gradient on the kernel's own branch, on every row
        mine = grad_float64(z, idx, adv, r32, clip, gs, ge)
        assert np.all(np.abs(d - mine) <= grad_bound(z, idx, adv, r32, clip, old, gs, ge))
        # exact values: +0 where both upstream gradients are 0
        zero_rows = (gs == 0) & (ge == 0)
        assert (bits(d[zero_rows]) == 0).all()
        # g_ent alone: the entropy gradient alone, and a clipped row's dz is that bit for bit
        de, = torch.autograd.grad(ent, zt, get_)
        de = de.cpu().numpy()
        assert np.all(np.abs(de - grad_float64(z, idx, adv, r32, clip, None, ge)) <= grad_bound(z, idx, adv, r32, clip, old, None, ge))
        cl = clipped(r32, adv, clip)
        assert cl.any() or clip == 0.99, (K, n, clip)
        assert np.array_equal(bits(d[cl]), bits(de[cl]))
        dz0 = torch.empty_like(zt)
        env._ppo_loss_grad_launch(zt.detach(), torch.from_numpy(idx).to(dev), torch.from_numpy(adv).to(dev), info["ratio"], clip, K, n,
                                  torch.zeros_like(gst), get_, dz0)
        assert np.array_equal(bits(dz0), bits(de))


@pytest.mark.parametrize("K", [1, 7])
def test_own_logp_gives_ratio_one(env, K):
    import torch
    rng = np.random.default_rng(K)
    z, idx, old, adv = make_rows(rng, 1000, K, 132)
    _, _, _, info = run(env, z, idx, old, adv, 0.2)
    _, surr, _, info2 = run(env, z, idx, info["logp"].cpu().numpy(), adv, 0.2)
    assert (info2["ratio"] == 1.0).all()
    assert np.array_equal(bits(surr), bits(-torch.from_numpy(adv)))


def store_rollout(evg, kind, player, n=500, T=6, latent=64, seed=5):
    import torch
    from evgsim import _capi, policy
    env = evg.BatchedEvergladesEnv(n, seed=seed, auto_reset=_capi.AUTORESET_NEXT)
    env.reset(obs_format="wire")
    torch.manual_seed(seed)
    if kind == "ppo":
        actor = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                                    torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1)).to(env.device)
        fused = policy.FusedPPO(env, actor, player=player)
        extra = {}
    else:
        actor = torch.nn.Module()
        actor.action_head = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
        actor.action_gru = torch.nn.GRU(latent, latent)
        actor.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
        actor = actor.to(env.device)
        fused = policy.FusedRPPO(env, actor, player=player)
        extra = {"want_hidden_in": True}

    def rollout(turns):
        rec = dict(rows=[], idx=[], logp=[], hidden_in=[])
        for _ in range(turns):
            rec["rows"].append(env.obs_rows("wire").clone())
            fused(obs_format="wire", want_logp=True, **extra)
            rec["idx"].append(fused.idx.clone())
            rec["logp"].append(fused.logp.clone())
            if kind == "rppo":
                rec["hidden_in"].append(fused.hidden_in.clone())
            if player == 0:
                env.agent_actions(_capi.AGENT_EXTERNAL, _capi.AGENT_SWARM)
            env.step(env._actions, obs_format="wire")
        return {k: torch.stack(v) for k, v in rec.items() if v}

    return env, actor, fused, rollout


def last_linear(env, actor, kind, rows, hidden_in, player):
    """float32 torch from the stored rows: z of the actor's last Linear, [R, 132] or [R, 7, 132]."""
    T, M = rows.shape[:2]
    obs = env.expand_wire(rows.view(T * M, -1), player=player).view(-1, 105)
    if kind == "ppo":
        return actor[:-2](obs)
    x = actor.action_head(obs)
    h0 = hidden_in.reshape(1, -1, x.shape[1])
    out, _ = actor.action_gru(x.unsqueeze(0).expand(7, -1, -1).contiguous(), h0)
    return actor.action_layer[0](out).permute(1, 0, 2).contiguous()


@pytest.mark.parametrize("kind,player", [("ppo", -1), ("ppo", 0), ("rppo", -1)])
def test_a_stored_rollout_updates_the_actor(evg, kind, player):
    import torch
    env, actor, fused, rollout = store_rollout(evg, kind, player)
    rec = rollout(6)
    idx, logp = rec["idx"].view(-1, 7), rec["logp"].view(-1, 7)
    R = idx.shape[0]
    adv = torch.randn(R, device=env.device, generator=torch.Generator(device=env.device).manual_seed(3))
    z = last_linear(env, actor, kind, rec["rows"], rec.get("hidden_in"), player)
    assert z.shape == ((R, 132) if kind == "ppo" else (R, 7, 132))
    surr, ent, info = env.ppo_loss(z, idx, logp, adv, clip=0.2)
    gap = (info["logp"] - logp).abs().max().item()
    assert gap <= LOGP_BF16, gap
    assert (info["ratio"] - 1).abs().max().item() <= np.expm1(7 * LOGP_BF16)
    params = [p for p in actor.parameters()]
    fused_grads = torch.autograd.grad(surr.mean() - 0.01 * ent.mean(), params, retain_graph=True)
    s_t, e_t, l_t, _ = torch_loss(z, idx, logp, adv, 0.2)
    assert (l_t - info["logp"]).abs().max().item() < 1e-4
    torch_grads = torch.autograd.grad(s_t.mean() - 0.01 * e_t.mean(), params, retain_graph=True)
    for a, b in zip(fused_grads, torch_grads):
        scale = b.abs().max().item()
        assert (a - b).abs().max().item() <= 1e-3 * scale + 1e-7, (a.shape, (a - b).abs().max().item(), scale)
    opt = torch.optim.Adam(actor.parameters(), lr=1e-3)
    opt.zero_grad()
    (surr.mean() - 0.01 * ent.mean()).backward()
    opt.step()
    fused.refresh()
    nxt = rollout(3)
    assert ((nxt["idx"] >= 0) & (nxt["idx"] < 132)).all()
    assert torch.isfinite(nxt["logp"]).all()


@pytest.mark.parametrize("K", [1, 7])
def test_cuda_graph_and_no_allocation(env, K):
    import torch
    rng = np.random.default_rng(11 + K)
    B, n = 3000, 132
    z, idx, old, adv = make_rows(rng, B, K, n)
    dev = env.device
    zt = torch.from_numpy(z).to(dev).requires_grad_(True)
    it, ot, at = (torch.from_numpy(x).to(dev) for x in (idx, old, adv))
    gs = torch.randn(B, device=dev)
    ge = torch.randn(B, device=dev)

    def run_once():
        surr, ent, info = env.ppo_loss(zt, it, ot, at, clip=0.2)
        dz, = torch.autograd.grad((surr, ent), zt, (gs, ge))
        return surr, ent, info["logp"], info["ratio"], dz

    want = [t.clone() for t in run_once()]
    torch.cuda.synchronize()
    # the launches themselves, outputs given: nothing allocated, no synchronisation; the autograd path: no synchronisation
    outs = [torch.empty(B, device=dev) for _ in range(3)] + [torch.empty((B, 7), device=dev), torch.empty_like(zt)]
    before = torch.cuda.memory_stats(dev)["allocation.all.allocated"]
    torch.cuda.set_sync_debug_mode("error")
    try:
        env._ppo_loss_launch(zt.detach(), it, ot, at, 0.2, K, n, outs[0], outs[1], outs[3], outs[2])
        env._ppo_loss_grad_launch(zt.detach(), it, at, outs[2], 0.2, K, n, gs, ge, outs[4])
        assert torch.cuda.memory_stats(dev)["allocation.all.allocated"] == before
        run_once()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    for a, b in zip(outs, (want[0], want[1], want[3], want[2], want[4])):
        assert np.array_equal(bits(a), bits(b))
    # the two launches in a CUDA graph, outputs given (tools/ppo_loss_time.py also captures the autograd path)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            env._ppo_loss_launch(zt.detach(), it, ot, at, 0.2, K, n, outs[0], outs[1], outs[3], outs[2])
            env._ppo_loss_grad_launch(zt.detach(), it, at, outs[2], 0.2, K, n, gs, ge, outs[4])
    torch.cuda.current_stream(dev).wait_stream(side)
    for _ in range(2):
        for t in outs:
            t.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(outs, (want[0], want[1], want[3], want[2], want[4])):
            assert np.array_equal(bits(a), bits(b))


@pytest.mark.parametrize("K", [1, 7])
def test_index_out_of_range_gives_a_nan_row(env, K):
    import torch
    rng = np.random.default_rng(21 + K)
    B, n = 64, 132
    z, idx, old, adv = make_rows(rng, B, K, n)
    bad_rows = [3, 17, 40]
    idx_bad = idx.copy()
    idx_bad[3, 0], idx_bad[17, 6], idx_bad[40, 2] = -1, n, 1 << 40
    zt, surr, ent, info = run(env, z, idx_bad, old, adv, 0.2, requires_grad=True)
    dz, = torch.autograd.grad((surr, ent), zt, (torch.ones_like(surr), torch.ones_like(ent)))
    _, s0, e0, i0 = run(env, z, idx, old, adv, 0.2)
    keep = np.setdiff1d(np.arange(B), bad_rows)
    for a, b in ((surr, s0), (ent, e0), (info["logp"], i0["logp"]), (info["ratio"], i0["ratio"])):
        a, b = a.detach().cpu().numpy(), b.cpu().numpy()
        assert np.isnan(a[bad_rows]).all()
        assert np.array_equal(bits(a[keep]), bits(b[keep]))
    d = dz.cpu().numpy()
    assert np.isnan(d[bad_rows]).all() and np.isfinite(d[keep]).all()


def test_wrapper_refuses_before_launching(env):
    import torch
    dev = env.device
    B, n = 16, 132
    z = torch.zeros((B, n), device=dev)
    idx = torch.zeros((B, 7), dtype=torch.int64, device=dev)
    old = torch.zeros((B, 7), device=dev)
    adv = torch.zeros(B, device=dev)
    before = env.launch_count
    bad = [
        dict(z=z.double()), dict(z=z.cpu()), dict(z=z.t().contiguous().t()), dict(z=z[:, :6].contiguous()),
        dict(z=torch.zeros((B, 257), device=dev)), dict(z=torch.zeros((B, 6, n), device=dev)), dict(z=torch.zeros((B,), device=dev)),
        dict(z=torch.zeros((0, n), device=dev), idx=idx[:0], old_logp=old[:0], adv=adv[:0]),
        dict(idx=idx.int()), dict(idx=idx[:, :6].contiguous()), dict(idx=idx[:-1]), dict(idx=idx.cpu()),
        dict(old_logp=old.double()), dict(old_logp=old[:-1]), dict(old_logp=old.t().contiguous().t()),
        dict(adv=adv.double()), dict(adv=adv[:-1]), dict(adv=adv[:, None]),
        dict(clip=-0.1), dict(clip=1.0), dict(clip=float("nan")), dict(clip=0.99999999), dict(clip="0.2"),
    ]
    for kw in bad:
        a = dict(z=z, idx=idx, old_logp=old, adv=adv, clip=0.2)
        a.update(kw)
        with pytest.raises(ValueError):
            env.ppo_loss(**a)
    assert env.launch_count == before
    env.ppo_loss(z, idx, old, adv)
    assert env.launch_count == before + 1


def test_abi_refuses_bad_arguments(env):
    import torch
    dev = env.device
    B, n = 16, 132
    z = torch.zeros((B, n), device=dev)
    idx = torch.zeros((B, 7), dtype=torch.int64, device=dev)
    f = [torch.zeros(B * 7 + 1, device=dev) for _ in range(6)]
    dz = torch.zeros(B * n + 1, device=dev)
    p = lambda t, off=0: C.c_void_p(t.data_ptr() + off)  # noqa: E731
    lib, h, s = env._lib, env._h, env._stream()
    base = dict(B=B, K=1, n=n, z=p(z), idx=p(idx), old=p(f[0]), adv=p(f[1]), clip=0.2, surr=p(f[2]), ent=p(f[3]), logp=p(f[4]), ratio=p(f[5]),
                dz=p(dz))

    def fwd(**kw):
        a = dict(base, **kw)
        return lib.evg_ppo_loss(h, a["B"], a["K"], a["n"], a["z"], a["idx"], a["old"], a["adv"], a["clip"], a["surr"], a["ent"], a["logp"],
                                a["ratio"], s)

    def bwd(**kw):
        a = dict(dict(base, gs=None, ge=None), **kw)
        return lib.evg_ppo_loss_grad(h, a["B"], a["K"], a["n"], a["z"], a["idx"], a["adv"], a["ratio"], a["clip"], a["gs"], a["ge"],
                                     a["dz"], s)

    null = C.c_void_p()
    before = env.launch_count
    cases = [dict(B=0), dict(B=-5), dict(B=1 << 31), dict(K=0), dict(K=2), dict(K=8), dict(n=6), dict(n=257),
             dict(clip=-1e-7), dict(clip=1.0), dict(clip=float("nan")), dict(clip=float("inf")),
             dict(z=null), dict(idx=null), dict(old=null), dict(adv=null), dict(surr=null), dict(ent=null), dict(logp=null), dict(ratio=null),
             dict(z=p(z, 2)), dict(idx=p(idx, 4)), dict(old=p(f[0], 1)), dict(adv=p(f[1], 2)), dict(surr=p(f[2], 3)), dict(ratio=p(f[5], 1))]
    for kw in cases:
        assert fwd(**kw) == -1, kw
        if not set(kw) & {"old", "surr", "ent", "logp"}:
            assert bwd(**kw) == -1, kw
    assert bwd(gs=p(f[0], 2)) == -1 and bwd(ge=p(f[0], 1)) == -1 and bwd(dz=null) == -1 and bwd(dz=p(dz, 2)) == -1
    assert lib.evg_ppo_loss(None, B, 1, n, p(z), p(idx), p(f[0]), p(f[1]), 0.2, p(f[2]), p(f[3]), p(f[4]), p(f[5]), s) == -1
    assert env.launch_count == before
    assert fwd() == 0 and bwd(gs=p(f[0]), ge=p(f[1])) == 0 and env.launch_count == before + 2
    # float32 operands 4-byte but not 8-byte aligned are accepted
    assert fwd(old=p(f[0], 4), adv=p(f[1], 4)) == 0 and bwd(adv=p(f[1], 4), dz=p(dz, 4)) == 0
    torch.cuda.synchronize()
