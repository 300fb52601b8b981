"""The fused PPO critic (evg_policy_value, evgsim.policy.FusedValue) on the GPU.

1. The exact network: test_gpu_policy_ppo_exact.py's hidden layers (boolean and analog units, every H one exact value
   on a 2^-11 grid), with a last layer of eighths on the boolean units and +-1/2 or +-1 on every analog unit and b3 in
   eighths.  Every product and partial sum of the last layer is then a multiple of 2^-12 below 2^11 in magnitude, exact
   in float32 in any order, so every value must EQUAL the float64 truth: at every width, at the tile edges (1, 127,
   128, 129 rows, and CTAs with several tiles), on float32 and wire rows, for player -1, 0 and 1.  The CPU checks at the
   top show that a kernel with H rounded toward zero, a tanh on the output, bf16-rounded biases or a dropped K chunk
   gives other values.
2. Random torch critics: within tests/test_policy_value_cpu.py's derived bound of the float64 truth, and within a
   bf16 tolerance of torch's float32 forward.
3. Wire rows give the float32 call's values bit for bit: env rows across automatic resets, DemoMap and the 16-node ring,
   and a stored [T, N] rollout evaluated in one call against T per-turn calls.
4. refresh(): the device images are pack_value's bytes (special values included), refresh() equals a rebuilt wrapper,
   allocates nothing and does not synchronise, and a CUDA graph of refresh -> FusedPPO -> FusedValue -> step replays
   the same turns as eager calls while the weights change.
5. Calling the critic every turn changes nothing else in a rollout.
6. The argument errors: ValueError from the wrapper, EVG_E_ARG from the C ABI."""
import ctypes as C

import numpy as np
import pytest

from evgsim import policy
from test_gpu_policy_ppo_exact import ExactPPO, machine
from test_gpu_policy_refresh import crafted, sgd_step
from test_gpu_policy_tiling import evg, sms  # noqa: F401
from test_gpu_policy_wire import config, same, wire_env
from test_policy_value_cpu import LATENTS, critic_weights, value_bound

gpu = pytest.mark.gpu
VALUE_MUTANTS = ["H1_rz", "H2_rz", "tanh_out", "bias_bf16", "l2_chunk", "l3_chunk"]
TORCH_ATOL = 5e-2  # bf16 operands against torch's float32 forward, nn.Linear's init: 0.018 at most over 20,000 synthetic rows


# ---------------------------------------------------------------- the exact critic (checked on the CPU)

def exact_critic(rng, in_dim, latent):
    """ExactPPO's hidden layers with one output: eighths on about 36 boolean units, +-1/2 or +-1 on every analog unit,
    b3 in eighths."""
    net = ExactPPO(rng, in_dim, latent, out_dim=1)
    a2 = net.analog2
    w3 = rng.choice([-1.0, 1.0], latent) * (rng.random(latent) < min(1.0, 36 / max(1, (~a2).sum()))) / 8
    w3[a2] = rng.choice([-1, -0.5, 0.5, 1], a2.sum())
    net.weights[4] = w3.reshape(1, latent).astype(np.float32)
    net.weights[5] = (rng.integers(-8, 9, 1) / 8).astype(np.float32)
    return net


def true_value(obs, net, mutant=None):
    """The exact critic in float64 (machine's H2, checked), or a defect: H1 / H2 rounded toward zero, b1 / b2 rounded to
    bf16, layer 2 missing its second K chunk (machine's mutants), a tanh on the output, the dot product missing H2's
    columns from 128 on."""
    _, H2, _ = machine(obs, net, mutant if mutant in ("H1_rz", "H2_rz", "bias_bf16", "l2_chunk") else None)
    H2 = H2.astype(np.float64)
    if mutant == "l3_chunk":
        H2[:, 128:] = 0
    w3, b3 = (np.asarray(a, dtype=np.float64) for a in net.weights[4:])
    assert (np.abs(H2) @ np.abs(w3[0])).max() + 1 < 2 ** 11, "output sums too wide"
    v = H2 @ w3[0] + b3[0]
    return np.tanh(v) if mutant == "tanh_out" else v


def obs_ints(rng, rows, in_dim):
    x = rng.integers(-100, 151, (rows, in_dim)).astype(np.float32)
    x[:, 0] = rng.integers(0, 600, rows)
    return x


@pytest.mark.parametrize("latent", [1, 17, 128, 129, 200, 256])
def test_exact_value_is_exact_and_sees_every_defect(latent):
    """The truth is a float32 number (exact in any order), reference_forward_value gives it bit for bit, and each
    defect changes it in more than 20 % of rows."""
    rng = np.random.default_rng(latent)
    net = exact_critic(rng, 105, latent)
    x = obs_ints(rng, 600, 105)
    v = true_value(x, net)
    assert np.array_equal(v.astype(np.float32).astype(np.float64), v)
    assert np.array_equal(policy.reference_forward_value(x, *net.weights), v.astype(np.float32))
    if latent == 1:
        return
    for mutant in VALUE_MUTANTS:
        if mutant.endswith("chunk") and latent <= 128:
            continue
        caught = (true_value(x, net, mutant) != v).mean()
        assert caught > 0.2, (mutant, caught)


# ---------------------------------------------------------------- GPU helpers

@pytest.fixture(scope="module")
def small(evg, cfg):
    """45 mid-game matches stepped in the wire format, env.obs their expansion: 90 rows, one partial tile."""
    return wire_env(evg, cfg, 45)


@pytest.fixture(scope="module")
def big(evg, cfg, sms):
    """One player's rows make ~2.5 tiles per CTA, both players' ~5, the last tile partial."""
    return wire_env(evg, cfg, ((5 * sms + 1) // 2 - 1) * 128 + 54)


def values(critic, m=None, fmt="f32"):
    """The critic of the env's first m matches ([m, 2] or [m] as numpy), from float32 or wire rows."""
    env = critic.env
    if m is None:
        return critic(obs_format=fmt).cpu().numpy()
    src = env.obs if fmt == "f32" else env.obs_rows("wire")
    return critic(src[:m], obs_format=fmt).cpu().numpy()


def check_exact_values(env, net, m=None):
    """Every player and format equal to the float64 truth of env.obs's rows."""
    m = env.num_envs if m is None else m
    obs = env.obs[:m].cpu().numpy()
    want = true_value(obs.reshape(-1, env.obs_len), net).reshape(m, 2).astype(np.float32)
    for player in (-1, 0, 1):
        critic = policy.FusedValue(env, weights=net.weights, player=player)
        for fmt in ("f32", "wire"):
            got = values(critic, None if m == env.num_envs else m, fmt)
            w = want if player < 0 else want[:, player]
            assert np.array_equal(got, w), (player, fmt, np.abs(got - w).max())


# ---------------------------------------------------------------- 1. the exact network

@gpu
@pytest.mark.parametrize("latent", LATENTS)
def test_exact_at_every_width(small, latent):
    check_exact_values(small, exact_critic(np.random.default_rng(latent), 105, latent))


@gpu
@pytest.mark.parametrize("latent", [64, 128, 129, 256])
def test_exact_at_the_tile_edges(big, sms, latent):
    """1, 127, 128 and 129 rows (player 0 or 1 over that many matches; both players over 64 and 65), and the whole
    batch: several tiles per CTA on every SM."""
    net = exact_critic(np.random.default_rng(latent + 1), 105, latent)
    assert 2 * big.num_envs > 4 * 128 * sms
    for m in (1, 64, 65, 127, 128, 129):
        check_exact_values(big, net, m)
    check_exact_values(big, net)


@gpu
def test_exact_on_the_16_node_ring(evg, tmp_path):
    env = wire_env(evg, config(evg, tmp_path, "ring16"), 300)
    assert env.obs_len == 125
    check_exact_values(env, exact_critic(np.random.default_rng(16), 125, 129))


# ---------------------------------------------------------------- 2. random torch critics

def torch_critic(torch, width, latent, seed):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Linear(width, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                               torch.nn.Linear(latent, 1)).cuda()


@gpu
@pytest.mark.parametrize("latent", [128, 248])
def test_random_critics_within_the_bound_and_of_torch(big, latent):
    """Within value_bound of the float64 truth (so within twice that of reference_forward_value, which is inside it
    too), and within TORCH_ATOL of torch's float32 forward."""
    import torch
    net = torch_critic(torch, 105, latent, latent)
    critic = policy.FusedValue(big, net)
    got = critic().cpu().numpy().reshape(-1).astype(np.float64)
    x = big.obs.view(-1, 105).cpu().numpy()
    w = policy._host_arrays(policy._value_params(net))
    v, bound = value_bound(x, *w)
    assert (np.abs(got - v) <= bound).all(), (np.abs(got - v) / bound).max()
    ref = policy.reference_forward_value(x, *w).astype(np.float64)
    assert (np.abs(got - ref) <= 2 * bound).all()
    with torch.no_grad():
        want = net(big.obs.view(-1, 105)).view(-1).cpu().numpy()
    assert np.abs(got - want).max() <= TORCH_ATOL, np.abs(got - want).max()


# ---------------------------------------------------------------- 3. wire rows = float32, bit for bit

@gpu
@pytest.mark.parametrize("which", ["demo", "ring16"])
def test_wire_equals_f32_across_resets(evg, tmp_path, which):
    """Both formats every turn of matches that end and start over (turn limit 30, automatic reset)."""
    import torch
    cfg = config(evg, tmp_path, which)
    cfg.turn_limit = 30
    env = evg.BatchedEvergladesEnv(300, seed=4, config=cfg, auto_reset=1)
    critics = [policy.FusedValue(env, torch_critic(torch, env.obs_len, latent, latent), player=p)
               for latent, p in ((1, -1), (128, 0), (256, 1))]
    env.reset(obs_format="wire")
    for t in range(70):
        env.step(env.random_actions(), obs_format="wire")
        env.expand_wire(env.obs_rows("wire"), out=env.obs)
        for c in critics:
            assert same(c().clone(), c(obs_format="wire")), t
    assert env.episode_stats()["episodes"] > 0


@gpu
def test_a_stored_rollout_in_one_call(evg, cfg):
    """[T, N] wire rows (and their float32 expansion) evaluated as T * N matches in one call equal T per-turn calls."""
    import torch
    T, n = 12, 700
    env = evg.BatchedEvergladesEnv(n, seed=9, auto_reset=1)
    critic = policy.FusedValue(env, torch_critic(torch, 105, 200, 3))
    rb = int(env._lib.evg_obs_row_bytes(env._h, 2))  # EVG_OBS_WIRE
    rows = torch.empty((T, n, rb), dtype=torch.uint8, device=env.device)
    per_turn = torch.empty((T, n, 2), device=env.device)
    env.reset(obs_format="wire")
    for t in range(T):
        env.step(env.random_actions(), obs_format="wire")
        rows[t].copy_(env.obs_rows("wire"))
        critic(obs_format="wire", out=per_turn[t])
    got = critic(rows.view(T * n, rb), obs_format="wire")
    assert got.shape == (T * n, 2) and same(got.view(T, n, 2), per_turn)
    obs = env.expand_wire(rows.view(T * n, rb))
    assert same(critic(obs.view(T * n, 2, 105)), got)
    out = torch.full((T * n,), 7.0, device=env.device)
    one = policy.FusedValue(env, critic._net, player=1)
    assert one(rows.view(T * n, rb), obs_format="wire", out=out) is out and same(out, got[:, 1].contiguous())


# ---------------------------------------------------------------- 4. refresh

def images(critic):
    return list(critic._w)


@gpu
@pytest.mark.parametrize("latent", LATENTS)
def test_device_images_are_the_host_packers_bytes(evg, latent):
    """Special values in every parameter (ties, +-0, subnormals, overflow to +-Inf); the images start as 0xFF."""
    import torch
    env = evg.BatchedEvergladesEnv(16, seed=1)
    rng = np.random.default_rng(latent)
    shapes = [(latent, 105), (latent,), (latent, latent), (latent,), (1, latent), (1,)]
    ws = [crafted(rng, s) for s in shapes]
    net = torch_critic(torch, 105, latent, 0)
    with torch.no_grad():
        for p, w in zip(policy._value_params(net), ws):
            p.copy_(torch.from_numpy(w))
    critic = policy.FusedValue(env, weights=critic_weights(rng, 105, latent))
    for t in critic._w:
        t.view(torch.uint8).fill_(0xFF)
    critic.refresh(net)
    want = policy.pack_value(*ws)[:4]
    for got, w in zip(images(critic), want):
        assert np.array_equal(got.cpu().numpy().view(np.uint8), np.ascontiguousarray(w).view(np.uint8))


def mid_game(evg, n=300, seed=3, turns=12):
    env = evg.BatchedEvergladesEnv(n, seed=seed)
    env.reset()
    for _ in range(turns):
        env.step(env.random_actions())
    return env


@gpu
def test_refresh_equals_a_rebuilt_wrapper(evg):
    import torch
    env = mid_game(evg)
    net = torch_critic(torch, 105, 248, 11)
    critic = policy.FusedValue(env, net)
    gen = torch.Generator(device=env.device).manual_seed(1)
    for _ in range(2):
        sgd_step(list(net.parameters()), gen)
    critic.refresh()
    fresh = policy.FusedValue(env, net)
    assert same(critic().clone(), fresh())
    for x, y in zip(images(critic), images(fresh)):
        assert torch.equal(x, y)


@gpu
def test_refresh_and_calls_allocate_nothing_and_do_not_synchronise(evg):
    import torch
    env = mid_game(evg, n=64, turns=1)
    critic = policy.FusedValue(env, torch_critic(torch, 105, 128, 2))
    ptrs = [t.data_ptr() for t in images(critic)] + [critic.value.data_ptr()]
    critic.refresh()
    critic()
    torch.cuda.synchronize()
    before = torch.cuda.memory_stats()["allocation.all.allocated"]
    launches = env.launch_count
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            critic.refresh()
            critic()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert env.launch_count == launches + 6
    assert torch.cuda.memory_stats()["allocation.all.allocated"] == before
    assert [t.data_ptr() for t in images(critic)] + [critic.value.data_ptr()] == ptrs


@gpu
def test_cuda_graph_of_refresh_actor_critic_step(evg, cfg):
    """One capture of refresh (actor and critic) -> FusedPPO -> FusedValue -> step; optimiser steps on both modules
    between turns.  The replays equal the same turns run eagerly: actions, observations, rewards, log-probabilities and
    values."""
    import torch
    n = 1000
    cfg.turn_limit = 30
    try:
        envs = [evg.BatchedEvergladesEnv(n, seed=14, config=cfg, auto_reset=1) for _ in range(2)]
    finally:
        cfg.turn_limit = 150
    torch.manual_seed(21)
    actor = torch.nn.Sequential(torch.nn.Linear(105, 128), torch.nn.Tanh(), torch.nn.Linear(128, 128), torch.nn.Tanh(),
                                torch.nn.Linear(128, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1)).cuda()
    net = torch_critic(torch, 105, 248, 22)
    ppo = [policy.FusedPPO(e, actor) for e in envs]
    critic = [policy.FusedValue(e, net) for e in envs]
    for e in envs:
        e.reset()

    def turn(k):
        ppo[k].refresh()
        critic[k].refresh()
        acts = ppo[k](want_logp=True)
        critic[k]()
        envs[k].step(acts)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            turn(1)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            turn(1)
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(3):
        turn(0)
    start = [t.clone() for t in images(critic[1])]
    gen = torch.Generator(device=envs[0].device).manual_seed(5)
    for t in range(40):
        sgd_step(list(actor.parameters()) + list(net.parameters()), gen, lr=0.02)
        turn(0)
        g.replay()
        for a, b in ((envs[0]._actions, envs[1]._actions), (envs[0].obs, envs[1].obs), (envs[0].reward, envs[1].reward),
                     (ppo[0].logp, ppo[1].logp), (critic[0].value, critic[1].value)):
            assert torch.equal(a, b), t
    for x, y, s in zip(images(critic[0]), images(critic[1]), start):
        assert torch.equal(x, y) and not torch.equal(y, s)
    torch.cuda.synchronize()
    assert (envs[0].get_state()["episode"] > 0).any()


# ---------------------------------------------------------------- 5. no effect elsewhere

@gpu
@pytest.mark.parametrize("obs_format", ["f32", "wire"])
def test_the_critic_changes_nothing_else_in_a_rollout(evg, cfg, obs_format):
    import torch
    cfg.turn_limit = 40
    try:
        envs = [evg.BatchedEvergladesEnv(600, seed=31, config=cfg, auto_reset=1) for _ in range(2)]
    finally:
        cfg.turn_limit = 150
    torch.manual_seed(3)
    actor = torch.nn.Sequential(torch.nn.Linear(105, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                                torch.nn.Linear(64, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1)).cuda()
    ppo = [policy.FusedPPO(e, actor) for e in envs]
    critic = policy.FusedValue(envs[1], torch_critic(torch, 105, 128, 4))
    for e in envs:
        e.reset(obs_format=obs_format)
    for t in range(100):
        outs = []
        for k, e in enumerate(envs):
            acts = ppo[k](obs_format=obs_format, want_logp=True)
            if k == 1:
                critic(obs_format=obs_format)
            outs.append(e.step(acts, obs_format=obs_format))
        for a, b in zip(outs[0][:3], outs[1][:3]):
            assert same(a, b), t
        assert same(ppo[0].logp, ppo[1].logp) and same(envs[0]._actions, envs[1]._actions), t
    s0, s1 = envs[0].episode_stats(), envs[1].episode_stats()
    assert s0 == s1 and s0["episodes"] > 0


# ---------------------------------------------------------------- 6. argument errors

@gpu
def test_wrapper_refusals(evg, cfg):
    import torch
    env = wire_env(evg, cfg, 64, turns=2)
    net = torch_critic(torch, 105, 64, 0)
    critic = policy.FusedValue(env, net)
    before = env.launch_count
    rows, obs = env.obs_rows("wire"), env.obs
    with pytest.raises(ValueError):
        critic(obs_format="i16")
    for bad in (rows[:, :96].clone(), rows.to(torch.int8), rows.cpu(), rows.float(), rows.t().contiguous().t(), rows.view(-1)):
        with pytest.raises(ValueError, match="obs must be"):
            critic(bad, obs_format="wire")
    for bad in (obs.double(), obs.cpu(), obs.view(-1, 105), obs.transpose(0, 1).contiguous().transpose(0, 1), obs[:, :, :100].clone()):
        with pytest.raises(ValueError, match="obs must be"):
            critic(bad)
    for out in (torch.empty((64, 2), device=env.device, dtype=torch.float64), torch.empty((64, 2)), torch.empty((64,), device=env.device),
                torch.empty((2, 64), device=env.device).t(), torch.empty((63, 2), device=env.device)):
        with pytest.raises(ValueError, match="out must be"):
            critic(obs, out=out)
    for bad_net in (torch_critic(torch, 104, 64, 0), torch.nn.Sequential(*list(net)[:-1], torch.nn.Linear(64, 2)).cuda(),
                    torch.nn.Sequential(*list(net)[:2], torch.nn.Linear(64, 1)).cuda()):
        with pytest.raises(ValueError):
            policy.FusedValue(env, bad_net)
    wrong = torch_critic(torch, 105, 32, 0)
    with pytest.raises(ValueError, match="shape"):
        critic.refresh(wrong)
    with pytest.raises(ValueError, match="float32"):
        critic.refresh(torch_critic(torch, 105, 64, 0).double())
    assert env.launch_count == before


@gpu
def test_abi_argument_errors(evg, cfg, tmp_path):
    """Bad arguments return EVG_E_ARG (-1) and launch nothing; n_matches = 0 launches nothing and succeeds; a map wider
    than the tiling (32 nodes, 189 values) is refused."""
    import torch
    from evgsim import _capi
    from test_gpu_generic import write_ring32
    env = wire_env(evg, cfg, 64, turns=2)
    net = torch_critic(torch, 105, 64, 0)
    critic = policy.FusedValue(env, net)
    lib, h, s = env._lib, env._h, env._stream()
    ptr = lambda t, off=0: C.c_void_p(t.data_ptr() + off)  # noqa: E731
    imgs = [ptr(t) for t in critic._w]
    rows, out = env.obs_rows("wire"), critic.value

    def value(fmt=_capi.OBS_WIRE, obs=None, m=64, player=-1, imgs=imgs, latent=64, dst=None, e=env):
        return e._lib.evg_policy_value(e._h, fmt, ptr(rows) if obs is None else obs, m, player, *imgs, latent,
                                       ptr(out) if dst is None else dst, s)

    n = env.launch_count
    assert value(fmt=_capi.OBS_I16) == -1 and value(fmt=7) == -1
    assert value(obs=C.c_void_p()) == -1 and value(dst=C.c_void_p()) == -1 and value(obs=ptr(rows, 8)) == -1
    for k in range(4):
        assert value(imgs=imgs[:k] + [C.c_void_p()] + imgs[k + 1:]) == -1, k
        assert value(imgs=imgs[:k] + [ptr(critic._w[k], 8)] + imgs[k + 1:]) == -1, k
    for kw in ({"m": -1}, {"player": -2}, {"player": 2}, {"latent": 0}, {"latent": 257}):
        assert value(**kw) == -1, kw
    assert value(m=0) == 0
    assert env.launch_count == n
    assert value() == 0 and env.launch_count == n + 1
    ps = [ptr(t) for t in policy._value_params(net)]

    def pack(ps=ps, imgs=imgs, latent=64, e=env):
        return e._lib.evg_pack_value(e._h, *ps, latent, *imgs, s)

    n = env.launch_count
    for k in range(6):
        assert pack(ps=ps[:k] + [C.c_void_p()] + ps[k + 1:]) == -1, k
    for k in range(4):
        assert pack(imgs=imgs[:k] + [C.c_void_p()] + imgs[k + 1:]) == -1, k
        assert pack(imgs=imgs[:k] + [ptr(critic._w[k], 8)] + imgs[k + 1:]) == -1, k
    assert pack(latent=0) == -1 and pack(latent=257) == -1
    assert env.launch_count == n
    assert pack() == 0 and env.launch_count == n + 1
    cfg32 = evg.load_config(write_ring32(tmp_path), "Ring32.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")
    wide = evg.BatchedEvergladesEnv(64, seed=2, config=cfg32)
    wide.reset()
    assert wide.obs_len == 189
    assert value(fmt=_capi.OBS_F32, obs=ptr(wide.obs), e=wide) == -1 and b"189" in lib.evg_last_error()
    assert pack(e=wide) == -1 and b"189" in lib.evg_last_error()
    torch.cuda.synchronize()
