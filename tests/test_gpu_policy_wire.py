"""The fused policies on wire rows (obs_format='wire', the _fmt entry points) against the same policies on the float32
observations of the same state, bit for bit: the wire stager must build exactly the bf16 tile the float32 stager builds.

The state: a simulator stepped in the wire format whose rows are then expanded into its own float32 tensor
(expand_wire, checked bit for bit against the float32 step in tests/test_gpu_wire_expand.py), so both inputs describe
the same matches and the draws read the same records.  Batch sizes sit at the 128-row tile edges and past one tile per
CTA; maps are DemoMap and the 7- and 16-node maps (89 and 125 values per row, the widest that fits)."""
import numpy as np
import pytest

from test_gpu_generic import write_configs
from test_gpu_policy_tiling import write_ring16

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def evg():
    import __graft_entry__ as g
    g.build()
    import evgsim
    return evgsim


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def config(evg, tmp_path, which):
    if which == "demo":
        return evg.load_config()
    if which == "map7":
        return evg.load_config(write_configs(tmp_path, 100), "Map7.json", "Units4.json", "Setup.json")
    return evg.load_config(write_ring16(tmp_path), "Ring16.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")


def wire_env(evg, cfg, n, seed=17, turns=30):
    """n matches played for `turns` turns in the wire format; env.obs holds the expansion of the last rows."""
    env = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg)
    env.reset(obs_format="wire")
    for _ in range(turns):
        env.step(env.random_actions(), obs_format="wire")
    env.expand_wire(env.obs_rows("wire"), out=env.obs)
    return env


def nets(torch, width, latent, seed=0):
    torch.manual_seed(seed)
    dqn = torch.nn.Sequential(torch.nn.Linear(width, 528), torch.nn.ReLU(), torch.nn.Linear(528, 132))
    ppo = torch.nn.Sequential(torch.nn.Linear(width, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                              torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
    actor = torch.nn.Module()
    actor.action_head = torch.nn.Sequential(torch.nn.Linear(width, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
    actor.action_gru = torch.nn.GRU(latent, latent)
    actor.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
    for m in (dqn, ppo, actor):
        m.to("cuda")
    return dqn, ppo, actor


def same(a, b):
    a, b = a.detach().cpu().numpy(), b.detach().cpu().numpy()
    return a.dtype == b.dtype and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def same_state(a, b):
    """EvgEnvState arrays equal field by field (the struct's padding bytes are not written by the export)"""
    return all(np.array_equal(a[k], b[k]) for k in a.dtype.names)


def check_dqn(evg, env, dqn):
    from evgsim import policy
    f = policy.FusedDQN(env, dqn)
    q = f.forward().clone()
    qt = f.forward_t().clone()
    assert same(f.forward(obs_format="wire"), q) and same(f.forward_t(obs_format="wire"), qt)
    assert same(f.forward(obs=env.obs_rows("wire").clone(), obs_format="wire"), q)
    acts = f().clone()
    assert same(f(obs_format="wire"), acts)


def run_actor(wrapper, fmt):
    acts = wrapper(want_probs=True, obs_format=fmt).clone()
    return acts, wrapper.idx.clone(), wrapper.probs.clone()


def check_actor(cls, env, net, player):
    import torch
    a = cls(env, net, player=player)
    h0 = getattr(a, "hidden", None)
    if h0 is not None:  # a carried state to start from, the same for both calls
        a.hidden.copy_(torch.rand_like(a.hidden) * 2 - 1)
        h0 = a.hidden.clone()
    ref = run_actor(a, "f32")
    if h0 is not None:
        ref, h1 = ref + (a.hidden.clone(),), a.hidden.copy_(h0)
    got = run_actor(a, "wire")
    if h0 is not None:
        got = got + (a.hidden.clone(),)
    for x, y in zip(ref, got):
        assert same(x, y), (cls.__name__, player)


@pytest.mark.parametrize("n", [1, 63, 64, 65, 127, 128, 129, "big"])
def test_tile_edges_on_demomap(evg, cfg, sms, n):
    import torch
    from evgsim import policy
    n = (5 * sms + 1) // 2 * 64 + 27 if n == "big" else n  # "big": ~2.5 tiles per CTA for one player, ~5 for both
    env = wire_env(evg, cfg, n)
    dqn, _, _ = nets(torch, env.obs_len, 128)
    check_dqn(evg, env, dqn)
    for latent in (1, 128, 256):
        _, ppo, actor = nets(torch, env.obs_len, latent, seed=latent)
        for player in (-1, 0, 1):
            check_actor(policy.FusedPPO, env, ppo, player)
            check_actor(policy.FusedRPPO, env, actor, player)


@pytest.mark.parametrize("which", ["map7", "ring16"])
def test_other_observation_widths(evg, tmp_path, which):
    import torch
    from evgsim import policy
    env = wire_env(evg, config(evg, tmp_path, which), 300)
    dqn, ppo, actor = nets(torch, env.obs_len, 129)
    check_dqn(evg, env, dqn)
    for player in (-1, 0, 1):
        check_actor(policy.FusedPPO, env, ppo, player)
        check_actor(policy.FusedRPPO, env, actor, player)


@pytest.mark.parametrize("latent", [1, 128, 256])
def test_recurrent_state_across_turns_with_resets(evg, cfg, latent):
    """20 turns of the recurrent actor, each on the wire rows of a twin and on the float32 observations of the other;
    masked resets in between restart some rows' state.  The state, draws and probabilities agree every turn."""
    import torch
    from evgsim import policy
    n = 333
    envs = [evg.BatchedEvergladesEnv(n, seed=8, config=cfg) for _ in range(2)]
    envs[0].reset()
    envs[1].reset(obs_format="wire")
    _, _, actor = nets(torch, envs[0].obs_len, latent, seed=3)
    fa = [policy.FusedRPPO(e, actor) for e in envs]
    for t in range(20):
        out = [run_actor(fa[0], "f32"), run_actor(fa[1], "wire")]
        for x, y in zip(*out):
            assert same(x, y), t
        assert same(fa[0].hidden, fa[1].hidden), t
        if t % 6 == 5:
            mask = torch.zeros(n, dtype=torch.uint8, device=envs[0].device)
            mask[t::7] = 1
            envs[0].reset(mask)
            envs[1].reset(mask, obs_format="wire")
        else:
            acts = envs[0]._actions.clone()
            envs[0].step(acts)
            envs[1].step(acts, obs_format="wire")


@pytest.mark.parametrize("family", ["dqn", "ppo", "rppo"])
def test_rollouts_on_wire_end_where_float32_rollouts_end(evg, family):
    """200 turns under AUTORESET_TERMINAL, each turn driven by the wrapper: on float32 observations with the float32 step,
    and on wire rows with the wire step.  Same records and same episode statistics at the end."""
    import torch
    from evgsim import policy
    cfg = evg.load_config(auto_reset=1)
    n = 700
    envs = [evg.BatchedEvergladesEnv(n, seed=21, config=cfg, auto_reset=1) for _ in range(2)]
    envs[0].reset()
    envs[1].reset(obs_format="wire")
    dqn, ppo, actor = nets(torch, envs[0].obs_len, 128, seed=4)
    make = {"dqn": lambda e: policy.FusedDQN(e, dqn), "ppo": lambda e: policy.FusedPPO(e, ppo),
            "rppo": lambda e: policy.FusedRPPO(e, actor)}[family]
    wr = [make(e) for e in envs]
    for _ in range(200):
        envs[0].step(wr[0](obs_format="f32"))
        envs[1].step(wr[1](obs_format="wire"), obs_format="wire")
    assert same_state(envs[0].get_state(), envs[1].get_state())
    sa, sb = envs[0].episode_stats(), envs[1].episode_stats()
    assert sa == sb and sa["episodes"] > 0


def test_cuda_graph_of_refresh_policy_and_wire_step(evg, cfg):
    """refresh -> FusedPPO(wire) -> wire step captured once and replayed equals the same turns run eagerly."""
    import torch
    from evgsim import policy
    n = 500
    envs = [evg.BatchedEvergladesEnv(n, seed=12, config=cfg) for _ in range(2)]
    _, ppo, _ = nets(torch, envs[0].obs_len, 128, seed=5)
    wr = [policy.FusedPPO(e, ppo) for e in envs]
    for e in envs:
        e.reset(obs_format="wire")

    def turn(e, w):
        w.refresh()
        e.step(w(obs_format="wire"), obs_format="wire")

    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        turn(envs[0], wr[0])  # warm-up outside the capture
        turn(envs[1], wr[1])
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            turn(envs[0], wr[0])
    torch.cuda.current_stream().wait_stream(stream)
    for _ in range(15):
        g.replay()
        turn(envs[1], wr[1])
    torch.cuda.synchronize()
    assert same(envs[0].obs_rows("wire"), envs[1].obs_rows("wire")) and same(wr[0].idx, wr[1].idx)
    assert same_state(envs[0].get_state(), envs[1].get_state())


def test_refusals(evg, cfg, tmp_path):
    import torch
    from evgsim import policy, _capi
    from test_gpu_generic import write_ring32
    env = wire_env(evg, cfg, 64, turns=2)
    dqn, ppo, actor = nets(torch, env.obs_len, 64)
    wrappers = [policy.FusedDQN(env, dqn), policy.FusedPPO(env, ppo), policy.FusedRPPO(env, actor)]
    before = env.launch_count
    for w in wrappers:
        with pytest.raises(ValueError):
            w(obs_format="i16")
    rows = env.obs_rows("wire")
    f = wrappers[0]
    for bad in (rows[:, :96].clone(), rows.to(torch.int8), rows.cpu(), rows.float(), rows[:32].clone(), rows.t().contiguous().t()):
        with pytest.raises(ValueError):
            f.forward(obs=bad, obs_format="wire")
    assert env.launch_count == before
    # EVG_OBS_I16 at the C ABI, and the 32-node map (189 values) for every wrapper's wire input
    assert env._lib.evg_policy_ppo_fmt(env._h, _capi.OBS_I16, rows.data_ptr(), -1, *[w.data_ptr() for w in wrappers[1]._w], 64, 132, 12, 11,
                                       env._actions.data_ptr(), None, None, None) == -1
    wide = evg.load_config(write_ring32(tmp_path), "Ring32.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")
    env32 = evg.BatchedEvergladesEnv(64, seed=2, config=wide)
    env32.reset(obs_format="wire")
    with pytest.raises(ValueError, match="189"):
        policy._wire_rows(env32, None, "wire")
