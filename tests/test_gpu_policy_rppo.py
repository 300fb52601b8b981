"""The fused recurrent PPO actor (evg_policy_rppo: tcgen05 + TMEM head and GRU, 7 draws on the tape, state carried in
FusedRPPO.hidden) against the numpy statement of its arithmetic, against torch, against the CPU sampler of
tests/ppo_sampling.py and, in the loop, against the oracle.

Tolerances.  The kernel and evgsim.policy.reference_forward_rppo round the same operands to bf16 and accumulate in fp32;
they differ in summation order (the kernel sums X W_i^T and H W_h^T in one accumulator) and in the last bit of tanh / exp /
the sigmoid.  As for the feed-forward actor (tests/test_gpu_policy_ppo.py) that rarely moves an activation or an element
of h across a bf16 rounding boundary; one such move changes a pre-activation by about one bf16 ulp of the operand times a
weight.  Here h is rounded again at each of the 7 steps and the fp32 state carries any such move into the later steps;
the bar stays the feed-forward actor's 5e-3 of each probability, and 5e-3 absolute on the final h (|h| < 1).
Against the plain fp32 torch network the difference is the bf16 rounding itself: 3e-2 of the largest probability, as in
tests/test_policy_rppo_cpu.py.  Rows sum to 1 within 1e-5 (132 float32 quotients)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LATENTS = [1, 15, 16, 17, 63, 64, 65, 127, 128, 129, 160, 192, 248, 255, 256]
P_REL, H_ABS = 5e-3, 5e-3


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


class Actor:
    """The reference ActorCritic's actor (use_recurrent), as tools/policy_rollout.py: RecurrentActor."""

    def __init__(self, torch, latent, seed):
        torch.manual_seed(seed)
        self.action_head = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
        self.action_gru = torch.nn.GRU(latent, latent)
        self.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))

    def torch_fp32(self, obs, h0):
        """probs [rows, 7, 132] and h [rows, L] of the fp32 torch network (on the CPU)."""
        import torch
        with torch.no_grad():
            x = self.action_head(torch.from_numpy(obs))
            seq, h = self.action_gru(x.unsqueeze(0).expand(7, -1, -1).contiguous(), torch.from_numpy(h0).unsqueeze(0))
            return self.action_layer(seq).permute(1, 0, 2).numpy(), h[0].numpy()


def mid_game(evg, cfg, n, seed=3, offset=0, turns=30):
    env = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg, env_id_offset=offset)
    env.reset()
    for _ in range(turns):  # real mid-game observations (turn counter, control states, unit counts)
        env.step(env.random_actions())
    return env


def uniforms(env, player=-1, matches=None):
    """The tape's 7 uniforms of every row (float32 [rows, 7]), rows in the kernel's order."""
    import ppo_sampling as ps
    st = env.get_state()
    players = (0, 1) if player < 0 else (player,)
    ms = range(env.num_envs) if matches is None else matches
    return np.stack([ps.policy_uniforms(env.seed, env.env_id_offset + m, int(st[m]["turn"]), p, int(st[m]["episode"]))
                     for m in ms for p in players])


def check_draws(idx, probs, u, acts_rows):
    """Every draw k is ppo_sample(probs_k, [u_k]), every action row its unravel."""
    import ppo_sampling as ps
    from oracle import policy_decode
    for k in range(7):
        assert np.array_equal(idx[:, k], ps.ppo_sample_rows(probs[:, k], u[:, k:k + 1])[:, 0]), k
    assert np.array_equal(acts_rows, policy_decode.ppo_unravel(idx).astype(np.int8))


def check_against_reference(actor, obs, h0, probs, h):
    from evgsim import policy
    want, want_h = policy.reference_forward_rppo(obs, h0, policy.rppo_weights(actor))
    assert np.isfinite(probs).all() and (probs > 0).all() and np.isfinite(h).all()
    assert np.abs(probs.sum(-1) - 1).max() <= 1e-5
    assert (np.abs(probs - want) <= P_REL * want).all(), np.abs(probs / want - 1).max()
    assert np.abs(h - want_h).max() <= H_ABS, np.abs(h - want_h).max()
    ref32, _ = actor.torch_fp32(obs, h0)
    assert np.abs(probs - ref32).max() <= 3e-2 * ref32.max(), (np.abs(probs - ref32).max(), ref32.max())


def run(env, actor, h0, player=-1):
    """One FusedRPPO call from state h0 (numpy, the shape of .hidden): (fused, actions, idx, probs, hidden) as numpy."""
    import torch
    from evgsim import policy
    fused = policy.FusedRPPO(env, actor, player=player)
    fused.hidden.copy_(torch.from_numpy(h0))
    acts = fused(want_probs=True).cpu().numpy()
    return fused, acts, fused.idx.cpu().numpy(), fused.probs.cpu().numpy(), fused.hidden.cpu().numpy()


@pytest.mark.parametrize("n", [64, 1037, 4096])
@pytest.mark.parametrize("latent", LATENTS)
def test_probabilities_state_and_exact_draws(evg, cfg, n, latent):
    """The kernel's own h0 (random, every match is mid-game) fed to the reference: the 7 distributions, the final state,
    and every draw bit for bit."""
    import torch
    env = mid_game(evg, cfg, n)
    actor = Actor(torch, latent, n + latent)
    h0 = np.random.default_rng(latent).uniform(-1, 1, (n, 2, latent)).astype(np.float32)
    assert (env.get_state()["turn"] > 0).all()
    _, acts, idx, probs, h = run(env, actor, h0)
    obs = env.obs.view(-1, 105).cpu().numpy()
    check_against_reference(actor, obs, h0.reshape(-1, latent), probs.reshape(-1, 7, 132), h.reshape(-1, latent))
    check_draws(idx.reshape(-1, 7), probs.reshape(-1, 7, 132), uniforms(env), acts.reshape(-1, 7, 2))


@pytest.mark.parametrize("latent,player", [(128, -1), (248, 0)])
def test_multi_tile_batches(evg, cfg, sms, latent, player):
    """Matches of ~2.5 tiles per CTA: player 0's rows give each CTA 2 or 3 tiles, both players' rows 4 or 5, the last
    tile partial.  Rows of the first, second, ... tile of the first CTAs and the last tile are checked in full."""
    import torch
    tiles = (5 * sms + 1) // 2
    n = (tiles - 1) * 128 + 54
    env = mid_game(evg, cfg, n, seed=17)
    actor = Actor(torch, latent, 40 + latent)
    shape = (n, 2, latent) if player < 0 else (n, latent)
    h0 = np.random.default_rng(1).uniform(-1, 1, shape).astype(np.float32)
    _, acts, idx, probs, h = run(env, actor, h0, player)
    rows_total = n * (2 if player < 0 else 1)
    n_tiles = -(-rows_total // 128)
    pick = sorted({t for c in (0, 1, 2) for t in range(c, n_tiles, sms)} | {n_tiles - 1})
    rows = np.concatenate([np.arange(t * 128, min((t + 1) * 128, rows_total)) for t in pick])
    per = 2 if player < 0 else 1
    obs = env.obs.cpu().numpy()
    obs_rows = obs.reshape(-1, 105)[rows] if player < 0 else obs[rows, player]
    check_against_reference(actor, obs_rows, h0.reshape(-1, latent)[rows], probs.reshape(-1, 7, 132)[rows], h.reshape(-1, latent)[rows])
    u_all = uniforms(env, player, matches=sorted(set((rows // per).tolist())))
    m_index = {m: i for i, m in enumerate(sorted(set((rows // per).tolist())))}
    u = u_all.reshape(-1, per, 7)[[m_index[r // per] for r in rows], rows % per]
    acts_rows = acts.reshape(-1, 7, 2)[rows] if player < 0 else acts[rows, player]
    check_draws(idx.reshape(-1, 7)[rows], probs.reshape(-1, 7, 132)[rows], u, acts_rows)


def test_turn_zero_rows_start_from_zero(evg, cfg):
    """Freshly reset matches ignore whatever .hidden holds (NaN included); after automatic resets in the middle of a
    batch exactly the rows of the matches that started over run from zero, the others from their state."""
    import torch
    n, latent = 1500, 128
    actor = Actor(torch, latent, 5)
    env = evg.BatchedEvergladesEnv(n, seed=9, config=cfg)
    env.reset()
    garbage = np.random.default_rng(2).uniform(-50, 50, (n, 2, latent)).astype(np.float32)
    garbage[::7] = np.nan
    got = run(env, actor, garbage)[1:]
    zero = run(env, actor, np.zeros_like(garbage))[1:]
    for a, b in zip(got, zero):
        assert np.array_equal(a, b)
    cfg.turn_limit = 20
    try:
        env = evg.BatchedEvergladesEnv(n, seed=9, config=cfg, auto_reset=1)
        env.reset()
        for t in range(20):  # every third match starts over at turn 10, the others reach the limit at turn 20
            if t == 10:
                env.reset(mask=(np.arange(n) % 3 == 0).astype(np.uint8))
            env.step(env.random_actions())
    finally:
        cfg.turn_limit = 150
    turn = env.get_state()["turn"]
    assert 0 < (turn == 0).sum() < n
    h0 = np.random.default_rng(3).uniform(-1, 1, (n, 2, latent)).astype(np.float32)
    _, acts, idx, probs, h = run(env, actor, h0)
    eff = np.where((turn == 0)[:, None, None], 0, h0).astype(np.float32)
    _, acts_e, idx_e, probs_e, h_e = run(env, actor, eff)
    assert np.array_equal(idx, idx_e) and np.array_equal(probs, probs_e) and np.array_equal(h, h_e)
    check_against_reference(actor, env.obs.view(-1, 105).cpu().numpy(), eff.reshape(-1, latent), probs.reshape(-1, 7, 132), h.reshape(-1, latent))


def test_single_player_sharding_and_repeats(evg, cfg):
    import torch
    n, latent = 2 * 777, 248
    actor = Actor(torch, latent, 4)
    env = mid_game(evg, cfg, n, seed=8)
    h0 = np.random.default_rng(4).uniform(-1, 1, (n, 2, latent)).astype(np.float32)
    fused, acts, idx, probs, h = run(env, actor, h0)
    # a second call from the same state is bit-identical
    again = run(env, actor, h0)[1:]
    for a, b in zip(again, (acts, idx, probs, h)):
        assert np.array_equal(a, b)
    # one player: only its own rows, the same draws, distributions and state as the two-player call
    for p in (0, 1):
        env._actions.fill_(-7)
        _, a1, i1, p1, h1 = run(env, actor, np.ascontiguousarray(h0[:, p]), player=p)
        assert (a1[:, 1 - p] == -7).all() and np.array_equal(a1[:, p], acts[:, p])
        assert np.array_equal(i1, idx[:, p]) and np.array_equal(p1, probs[:, p]) and np.array_equal(h1, h[:, p])
    # the whole batch equals two shards
    parts = [run(mid_game(evg, cfg, n // 2, seed=8, offset=o), actor, h0[o:o + n // 2])[1:] for o in (0, n // 2)]
    for k, whole in enumerate((acts, idx, probs, h)):
        assert np.array_equal(np.concatenate([q[k] for q in parts]), whole), k


def test_draws_follow_the_probabilities(evg, cfg):
    """65,536 freshly reset matches share one player-0 observation and a zero state, so one distribution per step; the
    draws of step 0 and step 6 differ only through the tape.  Chi-square of each 132-bin histogram."""
    import torch
    from scipy import stats
    from evgsim import policy
    n = 65536
    env = evg.BatchedEvergladesEnv(n, seed=21, config=cfg)
    env.reset()
    fused = policy.FusedRPPO(env, Actor(torch, 128, 2), player=0)
    fused(want_probs=True)
    probs = fused.probs.cpu().numpy()
    idx = fused.idx.cpu().numpy()
    assert (probs == probs[0]).all()
    for k in (0, 6):
        counts = np.bincount(idx[:, k], minlength=132)
        exp = probs[0, k].astype(np.float64) / probs[0, k].astype(np.float64).sum() * n
        assert stats.chisquare(counts, exp).pvalue > 1e-4, k
    assert len(np.unique(idx[:100], axis=0)) == 100


@pytest.mark.parametrize("opponent", ["self", "swarm"])
def test_in_the_loop_bit_exact_against_the_oracle(evg, cfg, opponent):
    """FusedRPPO self-play, and FusedRPPO(player=0) against the on-device SwarmAgent, 120 turns across automatic resets
    (auto_reset=2, turn_limit=50) with the state carried by the kernel: the oracle replays the rows played (duplicate
    indices included), and sampled rows are checked against ppo_sample of the kernel's distributions."""
    import torch
    from evgsim import _capi, policy
    from oracle import evg_oracle as eo
    from oracle import policy_decode
    import ppo_sampling as ps
    n = 384
    cfg.auto_reset = 2
    cfg.turn_limit = 50
    try:
        env = evg.BatchedEvergladesEnv(n, seed=5, config=cfg, auto_reset=2, env_id_offset=40)
        ora = eo.OracleBatch(cfg, n, seed=5, first=40)
        assert np.array_equal(env.reset().cpu().numpy(), ora.reset().astype(np.float32))
        player = -1 if opponent == "self" else 0
        fused = policy.FusedRPPO(env, Actor(torch, 128, 3), player=player)
        dups = 0
        for t in range(120):
            st = env.get_state()
            fused(want_probs=True)
            if opponent == "self":
                obs, rew, done, info = env.step(env._actions)
                acts = env._actions.cpu().numpy()
            else:
                obs, rew, done, info = env.step_agents(_capi.AGENT_EXTERNAL, _capi.AGENT_SWARM, actions=env._actions)
                acts = info["actions"].cpu().numpy()
            probs = fused.probs.cpu().numpy().reshape(n, -1, 7, 132)
            idx = fused.idx.cpu().numpy().reshape(n, -1, 7)
            dups += sum(len(set(r.tolist())) < 7 for r in idx.reshape(-1, 7))
            for m in range(t % 7, n, 37):
                for k in range(probs.shape[1]):
                    p = k if player < 0 else player
                    u = ps.policy_uniforms(5, 40 + m, int(st[m]["turn"]), p, int(st[m]["episode"]))
                    for s in range(7):
                        assert idx[m, k, s] == ps.ppo_sample(probs[m, k, s], u[s:s + 1])[0], (t, m, p, s)
                    assert np.array_equal(acts[m, p], policy_decode.ppo_unravel(idx[m, k]).astype(np.int8)), (t, m, p)
            oobs, orew, odone = ora.step(acts)
            assert np.array_equal(obs.cpu().numpy(), oobs.astype(np.float32)), t
            assert np.array_equal(rew.cpu().numpy(), orew.astype(np.float32)), t
            assert np.array_equal(done.cpu().numpy(), odone), t
        assert dups > 0  # rows with a repeated index were played and replayed
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
    actor = Actor(torch, 248, 9)
    cfg.turn_limit = 40
    try:
        envs = [evg.BatchedEvergladesEnv(n, seed=14, config=cfg, auto_reset=1) for _ in range(2)]
    finally:
        cfg.turn_limit = 150
    fused = [policy.FusedRPPO(e, actor) for e in envs]
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
    assert torch.equal(fused[0].hidden, fused[1].hidden)
    for t in range(60):
        turn(0)
        g.replay()
        assert torch.equal(fused[0].idx, fused[1].idx), t
        assert torch.equal(fused[0].hidden, fused[1].hidden), t
        assert torch.equal(envs[0].obs, envs[1].obs), t
    torch.cuda.synchronize()
    s0, s1 = envs[0].get_state(), envs[1].get_state()
    assert (s0["episode"] > 0).any()
    for name in ("turn", "episode", "control_state", "controlled_by", "health"):
        assert np.array_equal(s0[name], s1[name]), name


def test_argument_errors(evg, cfg):
    import torch
    from evgsim import policy
    env = evg.BatchedEvergladesEnv(64, seed=1, config=cfg)
    env.reset()
    fused = policy.FusedRPPO(env, Actor(torch, 128, 1))
    ptr = lambda t: C.c_void_p(t.data_ptr())
    w1, w2, wi, wh, w3, bias = (ptr(t) for t in fused._w)

    def call(hidden, latent=128, out_dim=132):
        return env._lib.evg_policy_rppo(env._h, ptr(env.obs), -1, w1, w2, wi, wh, w3, bias, latent, out_dim, 12, 11, hidden,
                                        ptr(env._actions), ptr(fused.idx), None, env._stream())

    h = ptr(fused.hidden)
    assert call(None) == -1  # EVG_E_ARG
    for latent in (0, 257):
        assert call(h, latent=latent) == -1
    for out_dim in (6, 145):
        assert call(h, out_dim=out_dim) == -1
    assert call(h) == 0
