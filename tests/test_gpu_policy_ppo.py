"""The fused PPO actor (evg_policy_ppo: tcgen05 + TMEM forward, sampling on the tape) against the numpy statement of its
arithmetic, against torch, against the CPU sampler of tests/ppo_sampling.py and, in the loop, against the oracle.

Tolerances.  The kernel and evgsim.policy.reference_forward_ppo round the same operands to bf16 and accumulate in fp32;
they differ in summation order and in the last bit of tanh / exp, which moves a hidden activation across a bf16 rounding
boundary only rarely.  One such move changes a logit by about one bf16 ulp of the activation times a weight (~1e-3 at
most for these nets) and a probability by about that relative amount, so the bar against the reference is 5e-3 of each
probability.  Against the plain fp32 torch network the difference is the bf16 rounding of operands and activations
itself (2^-9 relative each, through three layers): 3e-2 of the largest probability, as in tests/test_policy_ppo_cpu.py.
Rows sum to 1 within 1e-5 (132 float32 quotients)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def evg():
    import __graft_entry__ as g
    g.build()
    import evgsim
    return evgsim


def make_net(torch, seed, latent):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                               torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))


def weights_of(net):
    return [t.detach().float().cpu().numpy() for m in (net[0], net[2], net[4]) for t in (m.weight, m.bias)]


def mid_game(evg, cfg, n, seed=3, offset=0, turns=30):
    env = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg, env_id_offset=offset)
    env.reset()
    for _ in range(turns):  # real mid-game observations (turn counter, control states, unit counts)
        env.step(env.random_actions())
    return env


def expected_idx(env, probs, player=-1):
    """ppo_sampling.ppo_sample of the kernel's own probabilities with the tape's uniforms of every row."""
    import ppo_sampling as ps
    st = env.get_state()
    players = (0, 1) if player < 0 else (player,)
    u = np.stack([[ps.policy_uniforms(env.seed, env.env_id_offset + m, int(st[m]["turn"]), p, int(st[m]["episode"])) for p in players]
                  for m in range(env.num_envs)])
    return ps.ppo_sample_rows(probs.reshape(-1, probs.shape[-1]), u.reshape(-1, 7)).reshape(env.num_envs, len(players), 7)


@pytest.mark.parametrize("n", [64, 1037, 4096])
@pytest.mark.parametrize("latent", [128, 248, 100, 1, 15, 16, 17, 63, 64, 65, 129, 160, 192, 193, 255, 256])
def test_probabilities_and_exact_sampling(evg, cfg, n, latent):
    import torch
    from evgsim import policy
    from oracle import policy_decode
    env = mid_game(evg, cfg, n)
    net = make_net(torch, n + latent, latent)
    fused = policy.FusedPPO(env, net)
    acts = fused(want_probs=True).cpu().numpy()
    probs = fused.probs.cpu().numpy().reshape(2 * n, 132)
    idx = fused.idx.cpu().numpy()
    obs = env.obs.view(-1, 105)
    want = policy.reference_forward_ppo(obs.cpu().numpy(), *weights_of(net))
    assert np.isfinite(probs).all() and (probs > 0).all()
    assert np.abs(probs.sum(-1) - 1).max() <= 1e-5
    assert (np.abs(probs - want) <= 5e-3 * want).all(), np.abs(probs / want - 1).max()
    with torch.no_grad():
        ref32 = net.to(env.device)(obs).cpu().numpy()
    assert np.abs(probs - ref32).max() <= 3e-2 * ref32.max()
    # every row's indices are ppo_sample of its probabilities with its own uniforms, and its rows their unravel
    assert np.array_equal(idx, expected_idx(env, probs))
    assert np.array_equal(acts, policy_decode.ppo_unravel(idx).astype(np.int8))
    assert np.array_equal(env.decode_indices(fused.idx.clone(), div=12, mod=11, out=torch.empty_like(env._actions)).cpu().numpy(), acts)


def test_single_player_writes_only_its_own_rows(evg, cfg):
    import torch
    from evgsim import policy
    n = 777
    env = mid_game(evg, cfg, n, seed=8)
    net = make_net(torch, 4, 128)
    both = policy.FusedPPO(env, net)
    a_both = both(want_probs=True).clone()
    for p in (0, 1):
        one = policy.FusedPPO(env, net, player=p)
        env._actions.fill_(-7)  # sentinel
        a = one(want_probs=True)
        assert (a[:, 1 - p] == -7).all()
        # the draws are keyed on (match, turn, episode, player): the same rows as the two-player call's
        assert torch.equal(a[:, p], a_both[:, p])
        assert torch.equal(one.idx, both.idx[:, p]) and torch.equal(one.probs, both.probs[:, p])
        assert one.idx.shape == (n, 7) and one.probs.shape == (n, 132)
        assert np.array_equal(one.idx.cpu().numpy()[:, None], expected_idx(env, one.probs.cpu().numpy(), player=p))


def test_sharding_and_repeat_independence(evg, cfg):
    import torch
    from evgsim import policy
    n = 2 * 1500
    net = make_net(torch, 6, 248)
    whole = mid_game(evg, cfg, n, seed=12)
    halves = [mid_game(evg, cfg, n // 2, seed=12, offset=o) for o in (0, n // 2)]
    fw = policy.FusedPPO(whole, net)
    aw = fw(want_probs=True).clone()
    idx, probs = fw.idx.clone(), fw.probs.clone()
    fw(want_probs=True)
    assert torch.equal(fw.idx, idx) and torch.equal(fw.probs, probs) and torch.equal(whole._actions, aw)
    parts = []
    for h in halves:
        f = policy.FusedPPO(h, net)
        a = f(want_probs=True)
        parts.append((f.idx.cpu(), f.probs.cpu(), a.cpu()))
    assert torch.equal(torch.cat([p[0] for p in parts]), idx.cpu())
    assert torch.equal(torch.cat([p[1] for p in parts]), probs.cpu())
    assert torch.equal(torch.cat([p[2] for p in parts]), aw.cpu())


def test_first_draw_follows_the_probabilities(evg, cfg):
    """65,536 freshly reset matches share one player-0 observation and so one distribution; their first draws differ
    only through the tape (their global ids).  Chi-square of the 132-bin histogram against the probabilities."""
    import torch
    from scipy import stats
    from evgsim import policy
    n = 65536
    env = evg.BatchedEvergladesEnv(n, seed=21, config=cfg)
    env.reset()
    fused = policy.FusedPPO(env, make_net(torch, 2, 128), player=0)
    fused(want_probs=True)
    probs = fused.probs.cpu().numpy()
    assert (probs == probs[0]).all()
    first = fused.idx[:, 0].cpu().numpy()
    counts = np.bincount(first, minlength=132)
    exp = probs[0].astype(np.float64) / probs[0].astype(np.float64).sum() * n
    assert stats.chisquare(counts, exp).pvalue > 1e-4
    assert len(np.unique(fused.idx.cpu().numpy()[:100], axis=0)) == 100  # the matches do draw differently


@pytest.mark.parametrize("opponent", ["self", "swarm"])
def test_in_the_loop_bit_exact_against_the_oracle(evg, cfg, opponent):
    """FusedPPO self-play, and FusedPPO(player=0) against the on-device SwarmAgent: the oracle replays the rows both
    players played, turn by turn, across automatic resets (auto_reset=2, turn_limit=50); sampled rows are checked
    against ppo_sample of the kernel's probabilities."""
    import torch
    from evgsim import _capi, policy
    from oracle import evg_oracle as eo
    import ppo_sampling as ps
    from oracle import policy_decode
    n = 384
    cfg.auto_reset = 2
    cfg.turn_limit = 50
    try:
        env = evg.BatchedEvergladesEnv(n, seed=5, config=cfg, auto_reset=2, env_id_offset=40)
        ora = eo.OracleBatch(cfg, n, seed=5, first=40)
        assert np.array_equal(env.reset().cpu().numpy(), ora.reset().astype(np.float32))
        player = -1 if opponent == "self" else 0
        fused = policy.FusedPPO(env, make_net(torch, 3, 128), player=player)
        moved = 0
        for t in range(120):
            st = env.get_state()
            fused(want_probs=True)
            if opponent == "self":
                obs, rew, done, info = env.step(env._actions)
                acts = env._actions.cpu().numpy()
            else:
                obs, rew, done, info = env.step_agents(_capi.AGENT_EXTERNAL, _capi.AGENT_SWARM, actions=env._actions)
                acts = info["actions"].cpu().numpy()
            probs = fused.probs.cpu().numpy().reshape(n, -1, 132)
            idx = fused.idx.cpu().numpy().reshape(n, -1, 7)
            for m in range(t % 7, n, 37):
                for k in range(probs.shape[1]):
                    p = k if player < 0 else player
                    u = ps.policy_uniforms(5, 40 + m, int(st[m]["turn"]), p, int(st[m]["episode"]))
                    assert np.array_equal(idx[m, k], ps.ppo_sample(probs[m, k], u)), (t, m, p)
                    assert np.array_equal(acts[m, p], policy_decode.ppo_unravel(idx[m, k]).astype(np.int8)), (t, m, p)
            oobs, orew, odone = ora.step(acts)
            assert np.array_equal(obs.cpu().numpy(), oobs.astype(np.float32)), t
            assert np.array_equal(rew.cpu().numpy(), orew.astype(np.float32)), t
            assert np.array_equal(done.cpu().numpy(), odone), t
            moved += int((obs[:, :, 48::5] != 0).sum())
        assert moved > 0
        gs, os_ = env.get_state(), ora.states
        for name in ("turn", "episode", "control_state", "controlled_by", "health"):
            assert np.array_equal(gs[name], os_[name]), name
        assert env.episode_stats()["episodes"] > 0
    finally:
        cfg.auto_reset = 0
        cfg.turn_limit = 150


def test_cuda_graph_turn_equals_eager_turns(evg, cfg):
    import torch
    from evgsim import policy
    n = 1000
    net = make_net(torch, 9, 248)
    envs = [evg.BatchedEvergladesEnv(n, seed=14, config=cfg, auto_reset=1) for _ in range(2)]
    fused = [policy.FusedPPO(e, net) for e in envs]
    for e in envs:
        e.reset()

    def turn(k):
        fused[k]()
        envs[k].step(envs[k]._actions)

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
    for t in range(60):
        turn(0)
        g.replay()
        assert torch.equal(fused[0].idx, fused[1].idx), t
        assert torch.equal(envs[0].obs, envs[1].obs), t
    torch.cuda.synchronize()
    s0, s1 = envs[0].get_state(), envs[1].get_state()
    for name in ("turn", "episode", "control_state", "controlled_by", "health"):
        assert np.array_equal(s0[name], s1[name]), name
