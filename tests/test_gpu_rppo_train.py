"""The recurrent actor's update operation on the B200 (evg_rppo_train_forward / _backward, FusedRPPO.evaluate).

1. Exact forward: on the exact module's saturating network (x = +-1 exactly) h_7 is bit for bit the acting kernel's
   FusedRPPO.hidden from the same stored state, at every width and at the tiling edges, for float32 and wire rows.
2. Forward bound: on random actors every step's h_k lies within rppo_train.step_bound of float64 from the kernel's own
   h_{k-1}, and z_k within z_bound of float64 from the kernel's own h_k.
3. Gradients: dx and the six parameter gradients against the float64 analytic backward with the kernel's bf16 operands
   (rppo_train.backward64 with rnd = bf16).  The two differ by float32 accumulation and by the rare operand that rounds
   to the other bf16 neighbour (2^-8 relative of one term): GRAD_TOL of the largest entry holds it with margin.  dz = 0
   gives exact zeros, dz on one step leaves the other steps out of dW3, and a call repeats bit for bit.  What the
   kernel writes (every dgh_k, g_k and S) is held element by element to a derived bound and to exact values in
   tests/test_gpu_rppo_train_steps.py, and evaluate's reductions of it to gamma_m bounds: GRAD_TOL stands for the
   bf16 operands and float32 accumulation the float64 reference leaves out, not for the kernel's own arithmetic.
4. A stored FusedRPPO rollout against the SwarmAgent: the minibatch step with evaluate + ppo_loss is within UPDATE_TOL of
   the cuDNN float32 path's gradients (bf16 operands against float32), then Adam, refresh() and the next rollout.
5. A CUDA graph of the whole minibatch step equals eager; sync debug mode "error" passes; every refusal.
"""
import numpy as np
import pytest

import rppo_train as rt
from test_gpu_policy_rppo_exact import ExactNet, LATENTS, actor_of, float_net
from test_gpu_policy_tiling import mid_game
from test_gpu_ppo_loss import last_linear, store_rollout

gpu = pytest.mark.gpu
GRAD_TOL = 4e-3
UPDATE_TOL = 3e-2
WIDTHS = [1, 16, 127, 128, 129, 248, 256]


@pytest.fixture(scope="module")
def evg():
    import __graft_entry__ as g
    g.build()
    import evgsim
    return evgsim


@pytest.fixture(scope="module")
def sms(evg):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def env(evg, cfg):
    return mid_game(evg, cfg, 45)


def forward(fused, x, h0):
    """The kernel's (z [R, 7, out], h [R, 7, L]) through the wrapper's own launch path."""
    import torch
    R, L = x.shape
    z = torch.empty((R, 7, fused.out_dim), dtype=torch.float32, device=x.device)
    h = torch.empty((R, 7, L), dtype=torch.float32, device=x.device)
    fused._train_forward(x, h0, *fused_params(fused._net), z, h)
    return z, h


def grads(fused, x, h0, dz):
    """dx and the six parameter gradients of evaluate from dz, as numpy (float64)."""
    import torch
    actor = fused._net
    params = fused_params(actor)
    xt = x.clone().requires_grad_(True)
    z = fused.evaluate(xt, h0)
    got = torch.autograd.grad(z, [xt] + params, dz)
    return [g.double().cpu().numpy() for g in got]


def fused_params(actor):
    from evgsim import policy
    p = policy._rppo_params(actor)
    return [p[4], p[5], p[6], p[7], p[8], p[9]]


def exact_x(weights, obs):
    """The head's output on the saturating network from the kernel's bf16 observations: +-1 exactly."""
    w1, b1, w2, b2 = (np.asarray(a, np.float64) for a in weights[:4])
    x = np.tanh(np.tanh(rt.bf16(obs).astype(np.float64) @ w1.T + b1) @ w2.T + b2).astype(np.float32)
    assert np.all(np.abs(x) == 1)
    return x


# ---------------------------------------------------------------- 1. exact forward

def check_exact_forward(evg, env, latent, player, obs_format, seed):
    import torch
    rng = np.random.default_rng(seed)
    net = ExactNet(rng, env.obs_len, latent)
    fused = evg.policy.FusedRPPO(env, net.actor().to(env.device), player=player)
    rows = fused.hidden.numel() // latent
    fused.hidden.copy_(torch.from_numpy(net.h0(rng, rows)).view(fused.hidden.shape))
    if obs_format == "wire":  # a turn stepped in wire rows, and the float32 observations they expand to
        env.step(env.random_actions(), obs_format="wire")
        obs = env.expand_wire(env.obs_rows("wire"), player=player).cpu().numpy()
    else:
        obs = env.obs.cpu().numpy()
    obs = obs.reshape(-1, env.obs_len) if player < 0 else obs.reshape(-1, 2, env.obs_len)[:, player] if obs.ndim == 3 else obs
    fused(obs_format=obs_format, want_hidden_in=True)
    h0 = fused.hidden_in.view(rows, latent).clone()
    x = torch.from_numpy(exact_x(net.weights, obs)).to(env.device)
    z, h = forward(fused, x, h0)
    assert torch.equal(h[:, 6], fused.hidden.view(rows, latent)), (latent, (h[:, 6] != fused.hidden.view(rows, latent)).sum().item())


@gpu
@pytest.mark.parametrize("latent", LATENTS)
@pytest.mark.parametrize("obs_format", ["f32", "wire"])
def test_exact_forward_equals_the_acting_state_at_every_width(evg, env, latent, obs_format):
    check_exact_forward(evg, env, latent, -1, obs_format, latent)


@gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129, "big"])
@pytest.mark.parametrize("latent", [64, 128, 129, 256])
def test_exact_forward_at_the_tiling_edges(evg, cfg, sms, n, latent):
    m = ((5 * sms + 1) // 2 - 1) * 128 + 54 if n == "big" else n
    check_exact_forward(evg, mid_game(evg, cfg, m, seed=m), latent, 0, "f32", latent + m)


# ---------------------------------------------------------------- 2. forward bound

def random_case(evg, env, L, out, R, seed):
    import torch
    rng = np.random.default_rng(seed)
    weights = float_net(rng, env.obs_len, L, out)
    fused = evg.policy.FusedRPPO(env, actor_of(weights).to(env.device))
    x = torch.from_numpy(rng.uniform(-1, 1, (R, L)).astype(np.float32)).to(env.device)
    h0 = torch.from_numpy(rng.uniform(-1, 1, (R, L)).astype(np.float32)).to(env.device)
    return fused, weights, x, h0, rng


@gpu
@pytest.mark.parametrize("L", WIDTHS)
@pytest.mark.parametrize("out", [7, 132, 144])
def test_forward_within_the_step_bound(evg, env, L, out):
    fused, w, x, h0, _ = random_case(evg, env, L, out, 300, L * 1000 + out)
    z, h = (t.cpu().numpy() for t in forward(fused, x, h0))
    xs, h0s = x.cpu().numpy(), h0.cpu().numpy()
    wb = [rt.bf16(w[4]), w[5], rt.bf16(w[6]), w[7], rt.bf16(w[8]), w[9]]
    for k in range(7):
        hp = h0s if k == 0 else h[:, k - 1]
        _, h64, _ = rt.forward64(xs, hp, wb, rnd=rt.bf16)
        assert np.all(np.abs(h[:, k] - h64[:, 0]) <= rt.step_bound(xs, hp, wb)), (k, np.abs(h[:, k] - h64[:, 0]).max())
        z64 = rt.bf16(h[:, k].astype(np.float64)) @ wb[4].astype(np.float64).T + w[9]
        assert np.all(np.abs(z[:, k] - z64) <= rt.z_bound(h[:, k], w[8], w[9])), k


# ---------------------------------------------------------------- 3. gradients

def check_grads(evg, env, L, out, R, seed):
    import torch
    fused, w, x, h0, rng = random_case(evg, env, L, out, R, seed)
    dz = torch.from_numpy(rng.normal(size=(R, 7, out)).astype(np.float32)).to(env.device)
    got = grads(fused, x, h0, dz)
    wb = [rt.bf16(w[4]), w[5], rt.bf16(w[6]), w[7], rt.bf16(w[8]), w[9]]
    want = rt.backward64(x.cpu().numpy(), h0.cpu().numpy(), wb, dz.cpu().numpy(), rnd=rt.bf16)
    for name, a, b in zip(["dx", "dw_ih", "db_ih", "dw_hh", "db_hh", "dw3", "db3"], got, want):
        scale = np.abs(b).max()
        assert np.abs(a - b).max() <= GRAD_TOL * scale + 1e-6, (name, L, out, R, np.abs(a - b).max() / scale)
    return fused, x, h0, dz


@gpu
@pytest.mark.parametrize("L", WIDTHS)
@pytest.mark.parametrize("out", [7, 132, 144])
def test_gradients_against_float64(evg, env, L, out):
    check_grads(evg, env, L, out, 129, L * 7 + out)


@gpu
@pytest.mark.parametrize("R", [1, 127, 128, 129, "big"])
@pytest.mark.parametrize("L", [17, 128, 129, 256])
def test_gradients_at_the_tiling_edges(evg, env, sms, L, R):
    """One row block and a carry of one atom group (L = 17), one row block and two groups (128), two row blocks and
    groups of 4, 4, 1 atoms (129), two full row blocks, groups of 4, 4, 4 and a full piece table (256)."""
    check_grads(evg, env, L, 132, int(2.5 * sms) * 128 + 54 if R == "big" else R, 11)


@gpu
def test_zero_dz_single_step_and_repeatability(evg, env):
    import torch
    fused, w, x, h0, rng = random_case(evg, env, 129, 132, 300, 5)
    zero = torch.zeros((300, 7, 132), device=env.device)
    assert all(np.all(g == 0) for g in grads(fused, x, h0, zero))
    dz = torch.from_numpy(rng.normal(size=(300, 7, 132)).astype(np.float32)).to(env.device)
    a, b = grads(fused, x, h0, dz), grads(fused, x, h0, dz)
    assert all(np.array_equal(p, q) for p, q in zip(a, b))
    _, h = forward(fused, x, h0)
    for k in range(7):
        one = torch.zeros_like(dz)
        one[:, k] = dz[:, k]
        dw3 = grads(fused, x, h0, one)[5]
        hb = h[:, k].to(torch.bfloat16).double()
        assert np.allclose(dw3, (dz[:, k].double().t() @ hb).cpu().numpy(), rtol=1e-5, atol=1e-5), k


# ---------------------------------------------------------------- 4. a real update

def minibatch(env, actor, fused, rec, adv, use_fused):
    x = actor.action_head(env.expand_wire(rec["rows"].view(-1, rec["rows"].shape[-1]), player=-1).view(-1, env.obs_len))
    h0 = rec["hidden_in"].reshape(-1, x.shape[1])
    z = fused.evaluate(x, h0) if use_fused else last_linear(env, actor, "rppo", rec["rows"], rec["hidden_in"], -1)
    surr, ent, _ = env.ppo_loss(z, rec["idx"].view(-1, 7), rec["logp"].view(-1, 7), adv, clip=0.2)
    return surr.mean() - 0.01 * ent.mean()


@gpu
@pytest.mark.parametrize("latent", [64, 248])
def test_a_stored_rollout_updates_the_actor(evg, latent):
    import torch
    env, actor, fused, rollout = store_rollout(evg, "rppo", -1, latent=latent)
    rec = rollout(6)
    R = rec["idx"].numel() // 7
    adv = torch.randn(R, device=env.device, generator=torch.Generator(device=env.device).manual_seed(3))
    params = list(actor.parameters())
    ours = torch.autograd.grad(minibatch(env, actor, fused, rec, adv, True), params)
    ref = torch.autograd.grad(minibatch(env, actor, fused, rec, adv, False), params)
    for a, b in zip(ours, ref):
        err = ((a - b).norm() / b.norm()).item()
        assert err <= UPDATE_TOL, (a.shape, err)
    opt = torch.optim.Adam(actor.parameters(), lr=1e-3)
    opt.zero_grad()
    minibatch(env, actor, fused, rec, adv, True).backward()
    opt.step()
    fused.refresh()
    nxt = rollout(3)
    assert ((nxt["idx"] >= 0) & (nxt["idx"] < 132)).all() and torch.isfinite(nxt["logp"]).all()


# ---------------------------------------------------------------- 5. graph, sync, refusals

@gpu
def test_cuda_graph_and_no_synchronisation(evg):
    import torch
    env, actor, fused, rollout = store_rollout(evg, "rppo", -1, latent=128)
    rec = rollout(3)
    R = rec["idx"].numel() // 7
    adv = torch.randn(R, device=env.device, generator=torch.Generator(device=env.device).manual_seed(1))
    params = list(actor.parameters())

    def step():
        for p in params:
            p.grad = None
        minibatch(env, actor, fused, rec, adv, True).backward()
        return [p.grad.clone() for p in params]

    eager = step()
    torch.cuda.set_sync_debug_mode("error")
    try:
        again = step()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert all(torch.equal(a, b) for a, b in zip(eager, again))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    for p in params:
        p.grad = None
    with torch.cuda.graph(g):
        minibatch(env, actor, fused, rec, adv, True).backward()
    for p in params:
        p.grad.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(p.grad, a) for p, a in zip(params, eager))


@gpu
def test_evaluate_refuses_before_launching(evg, env):
    import torch
    fused, _, x, h0, _ = random_case(evg, env, 64, 132, 10, 1)
    n = env.launch_count
    bad = [(x.double(), h0), (x.cpu(), h0), (x[:, :32], h0), (x.t().contiguous().t(), h0), (x, h0[:5]), (x, h0.double()),
           (x.view(2, 5, 64), h0), ("x", h0)]
    for a, b in bad:
        with pytest.raises(ValueError):
            fused.evaluate(a, b)
    assert env.launch_count == n
    z = fused.evaluate(x[:0], h0[:0])
    assert z.shape == (0, 7, 132) and env.launch_count == n
    fused._net.action_gru.weight_hh_l0.data = fused._net.action_gru.weight_hh_l0.data.double()
    with pytest.raises(ValueError):
        fused.evaluate(x, h0)
    assert env.launch_count == n


@gpu
def test_device_pack_writes_the_host_images(evg, env):
    import torch
    fused, w, x, h0, _ = random_case(evg, env, 129, 132, 10, 2)
    forward(fused, x, h0)
    img = fused._train_images()
    imgs = evg.policy.pack_rppo(*w)
    assert np.array_equal(img[0].cpu().numpy(), imgs[2]) and np.array_equal(img[1].cpu().numpy(), imgs[3])
    assert np.array_equal(img[2].cpu().numpy(), rt.pack_wht(w[6]))
    assert np.array_equal(img[3].cpu().numpy(), imgs[4])
    b = img[4].cpu().numpy()
    assert np.array_equal(b[:144], imgs[5][512:656]) and np.array_equal(b[144:], imgs[5][656:])
