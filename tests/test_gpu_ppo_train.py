"""evg_ppo_train_forward / _backward (FusedPPO.evaluate, FusedValue.evaluate, FusedRPPO.evaluate_head) on the GPU.

0. The exact networks of the *_exact tests: z and v equal float64 exactly, bf16(x) too, at 15 widths from 1 to 256,
   f32 and wire input, players -1, 0 and 1, R = 1, 127, 128, 129, 130 and several tiles per CTA; the device training
   images equal the host packers' bytes.
1. The acting kernels, bit for bit, at L in LATENTS, on float32 and wire rows, for players -1, 0 and 1, at R = 1, 127,
   128, 129 and ~2.5 tiles per CTA: the critic's evaluate is its acting call; the head's bf16(x), fed to the unchanged
   recurrent update forward from the acting call's hidden_in, leaves h_7 equal to the acting call's .hidden; the actor's
   z through env.ppo_loss gives |ratio - 1| within ppo_train.ratio_bound (printed beside the torch float32 path's).
2. Every h1, h2 and output within ppo_train's float64 bounds of its own layer's bf16 operands.
3. dD2, dD1 and every parameter gradient against float64 on the kernel's bf16 operands within the derived bounds, at
   L in {1, 17, 64, 128, 129, 248, 256}, actor out in {7, 132, 144}, the critic and the head, at the row edges; exact
   zeros for a zero upstream gradient; repeat calls bit for bit.  The ~2.5-tiles-per-CTA edge runs at L = 64 and 256.
4. A stored wire-row rollout's update (actor + critic + ppo_loss + MSE, and the recurrent pipeline with evaluate_head)
   against torch on the kernels' bf16 operands within UPDATE_TOL relative norm, and against plain torch float32 within
   F32_TOL, each plus the two paths' largest ratio difference; then Adam, refresh() and the next rollout.
5. The whole update in a CUDA graph equals eager bit for bit and runs under sync-debug "error"; every ValueError comes
   before any launch."""
import numpy as np
import pytest

import ppo_train as pt
from test_gpu_policy_ppo_exact import ExactPPO, machine
from test_gpu_policy_rppo_exact import LATENTS as EXACT_LATENTS
from test_gpu_policy_value import exact_critic, true_value
from test_gpu_policy_wire import wire_env
from test_gpu_ppo_loss import bits, evg, store_rollout  # noqa: F401

pytestmark = pytest.mark.gpu

LATENTS = [1, 17, 64, 128, 129, 248, 256]
# (matches, player): R = 1, 127, 128, 129 rows, and ~2.5 tiles per CTA of 148 SMs
EDGES = [(1, 1), (127, 0), (64, -1), (129, 1), (23680, -1)]
# relative norm of a parameter gradient's difference between the fused update and torch float32 with the kernels' bf16
# operands (straight-through rounding: the same forward definition, float32 sums in torch's order), plus the largest
# difference between the two paths' ratios (the surrogate's gradient is proportional to the ratio)
UPDATE_TOL = 3e-2
# the same against plain torch float32: a sanity bound, not a precision claim.  The first layer's gradient flows through
# tanh units that large integer observations saturate, where 1 - h1^2 is tiny and bf16 operands move it by a large
# relative amount (on a B200 the actor's and the critic's dW1 and db1 differ by up to 7.9 % at L = 64, every other
# parameter by under 3 %, while against the bf16-operand path every gradient agrees within 0.4 %)
F32_TOL = 0.1


def st_bf16(t):
    """t rounded to bf16 in the forward, the identity in the backward."""
    import torch
    return t + (t.to(torch.bfloat16).float() - t).detach()


def mlp_bf16(net, x, n_layers):
    """The first n_layers Linear layers of a Sequential with Tanh after the hidden ones, on bf16 operands."""
    import torch
    lin = [m for m in net if isinstance(m, torch.nn.Linear)]
    for i, m in enumerate(lin[:n_layers]):
        x = torch.nn.functional.linear(st_bf16(x), st_bf16(m.weight), m.bias)
        x = torch.tanh(x) if i < 2 else x
    return x


def nets(torch, L, out, dev, seed):
    torch.manual_seed(seed)
    lin = torch.nn.Linear
    actor = torch.nn.Sequential(lin(105, L), torch.nn.Tanh(), lin(L, L), torch.nn.Tanh(), lin(L, out), torch.nn.Tanh(),
                                torch.nn.Softmax(dim=-1)).to(dev)
    critic = torch.nn.Sequential(lin(105, L), torch.nn.Tanh(), lin(L, L), torch.nn.Tanh(), lin(L, 1)).to(dev)
    ractor = torch.nn.Module()
    ractor.action_head = torch.nn.Sequential(lin(105, L), torch.nn.Tanh(), lin(L, L), torch.nn.Tanh())
    ractor.action_gru = torch.nn.GRU(L, L)
    ractor.action_layer = torch.nn.Sequential(lin(L, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
    return actor, critic, ractor.to(dev)


_GAMES = {}


def game(evg, n):
    """A self-play env of n matches after 3 random-policy turns: (env, wire rows of the current turn)."""
    if n not in _GAMES:
        import torch
        from evgsim import _capi, policy
        env = evg.BatchedEvergladesEnv(n, seed=7 + n, auto_reset=_capi.AUTORESET_NEXT)
        env.reset(obs_format="wire")
        play = policy.FusedPPO(env, nets(torch, 32, 132, env.device, 1)[0])
        for _ in range(3):
            play(obs_format="wire")
            env.step(env._actions, obs_format="wire")
        _GAMES[n] = env
    return _GAMES[n]


def np64(t):
    return t.detach().double().cpu().numpy()


@pytest.mark.parametrize("n,player", EDGES)
@pytest.mark.parametrize("L", LATENTS)
def test_the_acting_kernels_bit_for_bit(evg, n, player, L):
    import torch
    from evgsim import policy
    env = game(evg, n)
    dev = env.device
    rows = env.obs_rows("wire").clone()
    obs = env.expand_wire(rows)
    R = n * (2 if player < 0 else 1)
    actor, critic, ractor = nets(torch, L, 132, dev, L)
    # the critic
    fc = policy.FusedValue(env, critic, player=player)
    for o, fmt in ((rows, "wire"), (obs, "f32")):
        v = fc.evaluate(o, obs_format=fmt)
        assert v.shape == fc._shape(n)
        assert np.array_equal(bits(v), bits(fc(o, obs_format=fmt)))
    # the head: h_7 of the update forward from the acting call's hidden_in is the acting call's .hidden
    fr = policy.FusedRPPO(env, ractor, player=player)
    fr(obs_format="wire")  # a state that is not zero
    fr(obs_format="wire", want_hidden_in=True)
    params = policy._rppo_params(ractor)
    for o, fmt in ((rows, "wire"), (obs, "f32")):
        x = fr.evaluate_head(o, obs_format=fmt)
        assert x.shape == (R, L)
        z = torch.empty((R, 7, 132), device=dev)
        h = torch.empty((R, 7, L), device=dev)
        fr._train_forward(x.detach().contiguous(), fr.hidden_in.view(R, L), *params[4:], z, h)
        assert np.array_equal(bits(h[:, 6]), bits(fr.hidden.view(R, L))), fmt
    # the actor: its own draws' log-probabilities give ratio 1 within the summation-order bound
    fa = policy.FusedPPO(env, actor, player=player)
    fa(obs_format="wire", want_logp=True)
    idx, logp = fa.idx.view(R, 7), fa.logp.view(R, 7)
    adv = torch.ones(R, device=dev)
    for o, fmt in ((rows, "wire"), (obs, "f32")):
        z = fa.evaluate(o, obs_format=fmt)
        assert z.shape == (R, 132)
        _, _, info = env.ppo_loss(z.detach(), idx, logp, adv)
        dev_fused = (info["ratio"] - 1).abs().max().item()
        assert dev_fused <= pt.ratio_bound(132), (fmt, dev_fused)
    x32 = obs.view(-1, 105) if player < 0 else obs[:, player]
    _, _, info = env.ppo_loss(actor[:-2](x32).detach().contiguous(), idx, logp, adv)
    print("L=%d R=%d |ratio-1|: fused %.3g (bound %.3g), torch float32 %.3g"
          % (L, R, dev_fused, pt.ratio_bound(132), (info["ratio"] - 1).abs().max().item()))


def load(module, weights):
    """Copy float32 arrays (torch.nn.Linear's layout, in order) into the Linear layers of a Sequential."""
    import torch
    lin = [m for m in module if isinstance(m, torch.nn.Linear)]
    with torch.no_grad():
        for i, m in enumerate(lin):
            m.weight.copy_(torch.from_numpy(np.asarray(weights[2 * i], np.float32)))
            m.bias.copy_(torch.from_numpy(np.asarray(weights[2 * i + 1], np.float32)))
    return module


@pytest.fixture(scope="module")
def exact_env(evg):
    """Mid-game matches stepped in the wire format (env.obs their expansion): both players' rows make ~5 tiles per CTA."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return wire_env(evg, evg.load_config(), ((5 * sms + 1) // 2 - 1) * 128 + 54)


# (matches, player): R = 1, 127, 128, 129, 128 and 130 rows, and every match (several tiles per CTA on every SM)
EXACT_EDGES = [(1, 0), (127, 1), (128, 0), (129, 1), (64, -1), (65, -1), (None, -1)]


@pytest.mark.parametrize("L", EXACT_LATENTS)
def test_exact_networks_equal_float64(evg, exact_env, L):
    """The saturating constructions of the *_exact tests (test_gpu_policy_ppo_exact.ExactPPO, whose every hidden
    activation has one bf16 value and whose last layer's sums are exact in any order, and its critic): z and v equal
    the float64 truth exactly, for f32 and wire input, players -1, 0 and 1, at every row edge.  The head's x = h2 is
    tanhf's fp32 value, which no construction makes exact: bf16(x) equals the truth's H2 exactly, and x lies within
    tanhf's 2 ulp (4 u |x|) of float64 tanh of the exact pre-activation."""
    import torch
    from evgsim import policy
    env = exact_env
    dev = env.device
    rng = np.random.default_rng(L + 1000)
    anet, cnet, hnet = ExactPPO(rng, 105, L), exact_critic(rng, 105, L), ExactPPO(rng, 105, L)
    obs = env.obs.cpu().numpy().reshape(-1, 105)
    _, H2, _ = machine(obs, anet)
    w3, b3 = (np.asarray(a, np.float64) for a in anet.weights[4:])
    z_true = H2.astype(np.float64) @ w3.T + b3
    assert np.array_equal(z_true.astype(np.float32).astype(np.float64), z_true)
    v_true = true_value(obs, cnet)
    H1h, H2h, _ = machine(obs, hnet)
    w2, b2 = (np.asarray(a, np.float64) for a in hnet.weights[2:4])
    x_exact = np.tanh(H1h.astype(np.float64) @ w2.T + b2)
    actor, critic, ractor = nets(torch, L, 132, dev, L)
    load(actor, anet.weights)
    load(critic, cnet.weights)
    load(ractor.action_head, hnet.weights[:4])
    M = env.num_envs
    rows_all = env.obs_rows("wire")
    for m, player in EXACT_EDGES:
        m = M if m is None else m
        sel = np.arange(2 * m) if player < 0 else 2 * np.arange(m) + player
        fa, fc, fr = (policy.FusedPPO(env, actor, player=player), policy.FusedValue(env, critic, player=player),
                      policy.FusedRPPO(env, ractor, player=player))
        for src, fmt in ((env.obs[:m], "f32"), (rows_all[:m], "wire")):
            z = fa.evaluate(src, obs_format=fmt).detach().cpu().numpy()
            assert np.array_equal(z, z_true[sel].astype(np.float32)), (m, player, fmt, "z")
            v = fc.evaluate(src, obs_format=fmt).detach().cpu().numpy().reshape(-1)
            assert np.array_equal(v, v_true[sel].astype(np.float32)), (m, player, fmt, "v")
            x = fr.evaluate_head(src, obs_format=fmt).detach().cpu().numpy()
            assert np.array_equal(policy.bf16_round(x), H2h[sel]), (m, player, fmt, "bf16(x)")
            assert np.all(np.abs(x - x_exact[sel]) <= 4 * pt.U32 * np.abs(x_exact[sel])), (m, player, fmt, "x")


@pytest.mark.parametrize("L", [1, 17, 64, 129, 256])
@pytest.mark.parametrize("net", ["actor", "critic", "head"])
def test_device_training_images_are_the_host_packers_bytes(evg, net, L):
    """evg_ppo_train_pack's W1, W2, W3 (or w3) and bias vector are pack_ppo's / pack_value's bytes, and its W2^T is
    ppo_train.pack_w2t's, every byte of each written (the images start as 0xFF)."""
    import torch
    from evgsim import _capi, policy
    env = game(evg, 64)
    actor, critic, ractor = nets(torch, L, 132, env.device, L + 7)
    fused = {"actor": lambda: policy.FusedPPO(env, actor), "critic": lambda: policy.FusedValue(env, critic),
             "head": lambda: policy.FusedRPPO(env, ractor)}[net]()
    kind = {"actor": _capi.PPO_TRAIN_ACTOR, "critic": _capi.PPO_TRAIN_CRITIC, "head": _capi.PPO_TRAIN_HEAD}[net]
    for t in policy._ff_train_images(fused, kind):
        t.view(torch.uint8).fill_(0xFF)
    (fused.evaluate_head if net == "head" else fused.evaluate)(env.obs_rows("wire"))
    torch.cuda.synchronize()
    i1, i2, i3, i2t, bias = (t.cpu().numpy() for t in policy._ff_train_images(fused, kind))
    if net == "critic":
        w = [p_.detach().cpu().numpy() for p_ in policy._value_params(critic)]
        h1, h2, h3, hb, _ = policy.pack_value(*w)
    else:
        w = [p_.detach().cpu().numpy() for p_ in (policy._rppo_params(ractor)[:4] if net == "head" else fused._params(actor))]
        h1, h2, h3, hb, _, _ = policy.pack_ppo(*(w if net == "actor" else w + [np.zeros((7, L), np.float32), np.zeros(7, np.float32)]))
    same = lambda a, b: np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))  # noqa: E731
    assert same(i1, h1) and same(i2, h2) and same(i2t, pt.pack_w2t(w[2]))
    if net == "head":
        assert same(bias, hb[:2 * policy.PPO_MAX_LATENT])
    else:
        assert same(i3, h3) and same(bias, hb)


def run_net(env, fused, net, obs, player, dy_seed=0, dy_zero=False):
    """Forward and backward of one network through autograd (rows of `player`, a random or zero upstream gradient):
    (y, params with their .grad, dy)."""
    import torch
    from evgsim import _capi, policy
    kind = {"actor": _capi.PPO_TRAIN_ACTOR, "critic": _capi.PPO_TRAIN_CRITIC, "head": _capi.PPO_TRAIN_HEAD}[net]
    params = (policy._value_params(fused._net) if net == "critic" else policy._rppo_params(fused._net)[:4] if net == "head"
              else fused._params(fused._net))
    for p_ in params:
        p_.grad = None
    y = policy._ff_train_function().apply(obs, fused, kind, _capi.OBS_WIRE, player, fused.out_dim if net == "actor" else 1 if net == "critic"
                                          else fused.latent, *params)
    g = torch.Generator(device=env.device).manual_seed(dy_seed)
    dy = torch.zeros_like(y) if dy_zero else torch.randn(y.shape, device=env.device, generator=g)
    y.backward(dy)
    return y, params, dy


def kernel_outputs(env, fused, net, rows, player, params, dy):
    """What the kernels write for these parameters and upstream gradient, by direct calls (they are deterministic:
    the same as inside autograd): h1, h2, g2, dD2, dD1."""
    import ctypes as C
    import torch
    from evgsim import _capi, policy
    kind = {"actor": _capi.PPO_TRAIN_ACTOR, "critic": _capi.PPO_TRAIN_CRITIC, "head": _capi.PPO_TRAIN_HEAD}[net]
    out_dim = fused.out_dim if net == "actor" else 1 if net == "critic" else fused.latent
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    i1, i2, i3, i2t, bias = policy._ff_train_images(fused, kind)
    w = list(params) + [None, None] * (net == "head")
    lib, L = env._lib, fused.latent
    R = rows.shape[0] * (2 if player < 0 else 1)
    _capi.check(lib.evg_ppo_train_pack(env._h, kind, *[p(t) for t in w], L, out_dim, p(i1), p(i2), None if net == "head" else p(i3), p(i2t),
                                       p(bias), env._stream()))
    h1, h2 = torch.empty((R, L), device=env.device), torch.empty((R, L), device=env.device)
    out = torch.empty((R, out_dim), device=env.device)
    _capi.check(lib.evg_ppo_train_forward(env._h, kind, _capi.OBS_WIRE, p(rows), rows.shape[0], player, L, out_dim, p(i1), p(i2),
                                          None if net == "head" else p(i3), p(bias), p(out), p(h1), p(h2), env._stream()))
    bf = lambda t: t.detach().to(torch.bfloat16).float()  # noqa: E731
    d = dy.reshape(R, -1)
    g2 = (d @ bf(params[4]) if net == "actor" else d * bf(params[4]) if net == "critic" else d).contiguous()
    dd2, dd1 = torch.empty_like(h1), torch.empty_like(h1)
    _capi.check(lib.evg_ppo_train_backward(env._h, R, L, p(i2t), p(g2), p(h1), p(h2), p(dd2), p(dd1), env._stream()))
    torch.cuda.synchronize()
    return h1, h2, g2, dd2, dd1


@pytest.mark.parametrize("n,player", EDGES[:4] + [(2000, -1), EDGES[4]])
@pytest.mark.parametrize("L", LATENTS)
@pytest.mark.parametrize("net,out", [("actor", 7), ("actor", 132), ("actor", 144), ("critic", 1), ("head", 0)])
def test_forward_and_gradients_against_float64(evg, n, player, L, net, out):
    """... and at ~2.5 tiles per CTA (EDGES[4]), where every CTA of both kernels runs its persistent loop past the first
    tile, at one width of one 128-row piece and one of two."""
    import torch
    from evgsim import policy
    if n == EDGES[4][0] and L not in (64, 256):
        pytest.skip("the multi-tile batch runs at L = 64 and 256")
    if L not in (1, 129, 256) and n not in (2000, EDGES[4][0]) and net == "actor" and out != 132:
        pytest.skip("out 7 and 144 run at the extreme widths and the multi-tile batches")
    env = game(evg, n)
    dev = env.device
    rows = env.obs_rows("wire").clone()
    R = n * (2 if player < 0 else 1)
    obs = env.expand_wire(rows).view(-1, 105) if player < 0 else env.expand_wire(rows, player=player)
    actor, critic, ractor = nets(torch, L, max(out, 7), dev, L + out)
    fused = {"actor": lambda: policy.FusedPPO(env, actor, player=player), "critic": lambda: policy.FusedValue(env, critic, player=player),
             "head": lambda: policy.FusedRPPO(env, ractor, player=player)}[net]()
    y, params, dy = run_net(env, fused, net, rows, player)
    h1, h2, g2, dd2, dd1 = kernel_outputs(env, fused, net, rows, player, params, dy)
    w = [np64(p_) for p_ in params]
    x = np64(obs)
    H1, H2 = np64(h1), np64(h2)
    # forward: each layer from its own bf16 inputs, and the last
    for hk, xin, wi, bi in ((H1, x, w[0], w[1]), (H2, H1, w[2], w[3])):
        exact = np.tanh(pt.bf16(xin) @ pt.bf16(wi).T + bi)
        assert np.all(np.abs(hk - exact) <= pt.layer_bound(xin.astype(np.float32), wi, bi))
    Y = np64(y).reshape(R, -1)
    if net != "head":
        exact = pt.bf16(H2) @ pt.bf16(w[4]).T + w[5]
        bound = 2 * pt.gamma(L + 1) * (np.abs(pt.bf16(H2)) @ np.abs(pt.bf16(w[4])).T + np.abs(w[5])) + 1e-30
        assert np.all(np.abs(Y - exact) <= bound)
    else:
        assert np.array_equal(bits(y), bits(h2))
    # backward: dD2 = g2 (1 - h2^2) in float32 (3 u), dD1 from the kernel's own bf16(dD2)
    G2, D2, D1 = np64(g2), np64(dd2), np64(dd1)
    assert np.all(np.abs(D2 - G2 * (1 - H2 * H2)) <= 3 * pt.U32 * np.abs(G2) + 1e-30)
    exact = (pt.bf16(D2) @ pt.bf16(w[2])) * (1 - H1 * H1)
    assert np.all(np.abs(D1 - exact) <= pt.dd1_bound(D2, w[2]))
    # parameter gradients: float32 reductions of what the kernels wrote
    DY = np64(dy).reshape(R, -1)
    want = [(D1, pt.bf16(x)), (D2, pt.bf16(H1))] + ([] if net == "head" else [(DY, pt.bf16(H2))])
    for i, (a, bmat) in enumerate(want):
        gw, gb = np64(params[2 * i].grad), np64(params[2 * i + 1].grad)
        assert np.all(np.abs(gw - a.T @ bmat) <= pt.matmul_bound(a, bmat)), i
        assert np.all(np.abs(gb - a.sum(0)) <= pt.matmul_bound(a, np.ones((R, 1)))[:, 0]), i


@pytest.mark.parametrize("net", ["actor", "critic", "head"])
def test_zero_upstream_gives_zero_and_repeats_are_bitwise(evg, net):
    import torch
    from evgsim import policy
    env = game(evg, 500)
    rows = env.obs_rows("wire").clone()
    actor, critic, ractor = nets(torch, 129, 132, env.device, 9)
    fused = {"actor": lambda: policy.FusedPPO(env, actor), "critic": lambda: policy.FusedValue(env, critic),
             "head": lambda: policy.FusedRPPO(env, ractor)}[net]()
    _, params, _ = run_net(env, fused, net, rows, -1, dy_zero=True)
    for p_ in params:
        assert not p_.grad.any(), p_.shape
    runs = []
    for _ in range(2):
        y, params, _ = run_net(env, fused, net, rows, -1, dy_seed=4)
        runs.append([bits(y)] + [bits(p_.grad) for p_ in params])
    for a, b in zip(*runs):
        assert np.array_equal(a, b)


def update_step(env, fa, fc, rec, adv, ret, path):
    """One PPO minibatch loss from stored wire rows: "fused" networks, or torch on expand_wire, "f32" or "bf16"
    (the kernels' operands): (loss, ratio)."""
    import torch
    rows = rec["rows"].view(-1, rec["rows"].shape[-1])
    idx, logp = rec["idx"].view(-1, 7), rec["logp"].view(-1, 7)
    if path == "fused":
        z, v = fa.evaluate(rows), fc.evaluate(rows)
    else:
        obs = env.expand_wire(rows).view(-1, 105)
        obs_a = obs if fa.player < 0 else env.expand_wire(rows, player=fa.player)
        if path == "f32":
            z, v = fa._net[:-2](obs_a), fc._net(obs).view(-1, 2)
        else:
            z, v = mlp_bf16(fa._net, obs_a, 3), mlp_bf16(fc._net, obs, 3).view(-1, 2)
    surr, ent, info = env.ppo_loss(z, idx, logp, adv)
    return surr.mean() - 0.01 * ent.mean() + 0.5 * torch.nn.functional.mse_loss(v.view(-1), ret), info["ratio"]


@pytest.mark.parametrize("player", [-1, 0])
def test_a_stored_rollout_updates_actor_and_critic(evg, player):
    import torch
    from evgsim import policy
    env, actor, fa, rollout = store_rollout(evg, "ppo", player)
    critic = torch.nn.Sequential(torch.nn.Linear(105, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                                 torch.nn.Linear(64, 1)).to(env.device)
    fc = policy.FusedValue(env, critic)
    rec = rollout(6)
    R = rec["idx"].view(-1, 7).shape[0]
    g = torch.Generator(device=env.device).manual_seed(3)
    adv, ret = torch.randn(R, device=env.device, generator=g), torch.randn(R, device=env.device, generator=g)
    if player == 0:  # the critic values both players' rows; the actor's rows are player 0's
        ret = torch.randn(R * 2, device=env.device, generator=g)
    params = list(actor.parameters()) + list(critic.parameters())
    loss_f, ratio_f = update_step(env, fa, fc, rec, adv, ret, "fused")
    gf = torch.autograd.grad(loss_f, params)
    for path, base in (("bf16", UPDATE_TOL), ("f32", F32_TOL)):
        loss_t, ratio_t = update_step(env, fa, fc, rec, adv, ret, path)
        gt = torch.autograd.grad(loss_t, params)
        tol = base + (ratio_f - ratio_t).abs().max().item()
        rels = [((a - b).norm() / b.norm().clamp_min(1e-12)).item() for a, b in zip(gf, gt)]
        print("player %d, torch %s: gradient relative norms %s (tolerance %.3g)" % (player, path, ["%.2g" % r for r in rels], tol))
        assert max(rels) <= tol, (path, rels, tol)
    opt = torch.optim.Adam(params, lr=1e-3)
    opt.zero_grad()
    update_step(env, fa, fc, rec, adv, ret, "fused")[0].backward()
    opt.step()
    fa.refresh()
    fc.refresh()
    nxt = rollout(3)
    assert ((nxt["idx"] >= 0) & (nxt["idx"] < 132)).all() and torch.isfinite(nxt["logp"]).all()


def test_a_stored_rollout_updates_the_recurrent_actor(evg):
    import torch
    env, actor, fr, rollout = store_rollout(evg, "rppo", -1)
    rec = rollout(6)
    rows = rec["rows"].view(-1, rec["rows"].shape[-1])
    idx, logp, h0 = rec["idx"].view(-1, 7), rec["logp"].view(-1, 7), rec["hidden_in"].view(-1, fr.latent)
    R = idx.shape[0]
    adv = torch.randn(R, device=env.device, generator=torch.Generator(device=env.device).manual_seed(3))
    params = list(actor.parameters())

    def loss(head):
        obs = env.expand_wire(rows).view(-1, 105)
        x = fr.evaluate_head(rows) if head == "fused" else actor.action_head(obs) if head == "f32" else mlp_bf16(actor.action_head, obs, 2)
        surr, ent, info = env.ppo_loss(fr.evaluate(x, h0), idx, logp, adv)
        return surr.mean() - 0.01 * ent.mean(), info

    lf, info = loss("fused")
    assert (info["ratio"] - 1).abs().max().item() <= pt.ratio_bound(132)
    gf = torch.autograd.grad(lf, params)
    for path, base in (("bf16", UPDATE_TOL), ("f32", F32_TOL)):
        lt, info_t = loss(path)
        gt = torch.autograd.grad(lt, params)
        tol = base + (info["ratio"] - info_t["ratio"]).abs().max().item()
        rels = [((a - b).norm() / b.norm().clamp_min(1e-12)).item() for a, b in zip(gf, gt)]
        print("recurrent, torch %s head: gradient relative norms %s (tolerance %.3g)" % (path, ["%.2g" % r for r in rels], tol))
        assert max(rels) <= tol, (path, rels, tol)
    opt = torch.optim.Adam(params, lr=1e-3)
    opt.zero_grad()
    loss("fused")[0].backward()
    opt.step()
    fr.refresh()
    nxt = rollout(3)
    assert torch.isfinite(nxt["logp"]).all()


def test_cuda_graph_and_no_sync(evg):
    import torch
    from evgsim import policy
    env, actor, fa, rollout = store_rollout(evg, "ppo", -1, n=300)
    critic = torch.nn.Sequential(torch.nn.Linear(105, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                                 torch.nn.Linear(64, 1)).to(env.device)
    fc = policy.FusedValue(env, critic)
    rec = rollout(4)
    R = rec["idx"].view(-1, 7).shape[0]
    g = torch.Generator(device=env.device).manual_seed(5)
    adv, ret = torch.randn(R, device=env.device, generator=g), torch.randn(R, device=env.device, generator=g)
    params = list(actor.parameters()) + list(critic.parameters())

    def step():
        for p_ in params:
            p_.grad = None
        update_step(env, fa, fc, rec, adv, ret, "fused")[0].backward()
        return [p_.grad.clone() for p_ in params]

    eager = step()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        step()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for p_ in params:
            p_.grad = None
        update_step(env, fa, fc, rec, adv, ret, "fused")[0].backward()
    graph.replay()
    torch.cuda.synchronize()
    for a, p_ in zip(eager, params):
        assert np.array_equal(bits(a), bits(p_.grad))


def test_refusals_before_any_launch(evg):
    import torch
    from evgsim import policy
    env = game(evg, 64)
    rows = env.obs_rows("wire").clone()
    obs = env.expand_wire(rows)
    actor, critic, ractor = nets(torch, 32, 132, env.device, 2)
    fa, fc, fr = policy.FusedPPO(env, actor), policy.FusedValue(env, critic), policy.FusedRPPO(env, ractor)
    for ev in (fa.evaluate, fc.evaluate, fr.evaluate_head):
        for args in [(rows, "i16"), (rows, "f32"), (obs, "wire"), (rows.float(), "wire"), (rows[:, :-16], "wire"), (rows.cpu(), "wire"),
                     (rows.t().contiguous().t(), "wire"), (obs.double(), "f32"), (obs[:, :1].contiguous(), "f32"),
                     (obs.transpose(0, 1).contiguous().transpose(0, 1), "f32"), ([1, 2], "wire")]:
            before = env.launch_count
            with pytest.raises(ValueError):
                ev(*args[:1], obs_format=args[1])
            assert env.launch_count == before, args[1]
        assert ev(rows[:0]).shape[0] == 0
    for fused in (policy.FusedPPO(env, weights=[p_.detach().cpu().numpy() for p_ in fa._params(actor)]),
                  policy.FusedValue(env, weights=[p_.detach().cpu().numpy() for p_ in policy._value_params(critic)])):
        before = env.launch_count
        with pytest.raises(ValueError, match="weights="):
            fused.evaluate(rows)
        assert env.launch_count == before
    actor.double()
    before = env.launch_count
    with pytest.raises(ValueError, match="parameter"):
        fa.evaluate(rows)
    assert env.launch_count == before
