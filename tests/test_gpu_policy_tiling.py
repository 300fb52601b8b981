"""The fused DQN and PPO kernels (evg_policy_mlp, evg_policy_ppo) past one tile per CTA and at every tiling edge.

Both kernels are persistent (grid = min(tiles, SMs), 128-row tiles), and most of their pipelining only runs when a CTA
handles a second tile: the next tile's observations are loaded under this tile's epilogue or sampling, DQN queues the
next tile's first MMAs early, and the weight-image and mbarrier parities carry over from tile to tile.  The large batch
here is sized from the device's SM count so that CTAs handle 2 to 5 tiles of distinct, real mid-game rows, unevenly,
with a partial last tile.

What each check compares against:
- DQN, exact integer Q: integer observations and weights chosen so that every value the kernel forms is exact in its
  format (bf16-exact operands, every partial sum an integer below 2^22, exact in fp32 whatever the order).  Q then has
  one correct value: the integer computation below, with the kernel's only roundings (bf16 round-to-nearest-even of the
  observations and of the hidden activations), compared bit for bit.  Two variants put bf16 ties into the hidden
  activations and into the observations, where round-toward-zero or round-half-away would change Q.
- DQN, float nets: a float64 evaluation of the bf16-rounded operands with a per-element bound (see q_and_bound).
- PPO: probabilities within 5e-3 of each of evgsim.policy.reference_forward_ppo's (tests/test_gpu_policy_ppo.py gives
  the reasoning), the drawn indices equal to tests/ppo_sampling.py's sampler bit for bit, the action rows their unravel.
- Both: results that do not depend on where a row sits in the batch (permuted rows, shards), bit for bit.
The CPU tests at the top check the generators of the exact cases."""
import ctypes as C
import json

import numpy as np
import pytest

from evgsim import policy

gpu = pytest.mark.gpu
EXACT = 2 ** 22     # bound on every partial sum of the exact cases (fp32 holds integers up to 2^24: two bits to spare)
HIDDEN = [1, 190, 191, 192, 383, 528, 12288]
OUTS = [1, 12, 36, 37, 132, 144]


# ---------------------------------------------------------------- exact integer cases (checked on the CPU below)

def bf16_exact(a):
    a = np.asarray(a, dtype=np.float32)
    return np.array_equal(policy.bf16_round(a), a)


def bf16_rz(a):
    """bf16 rounding toward zero (truncation), as float32: the conversion the exact cases must tell apart from RNE."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    return (u & np.uint32(0xFFFF0000)).view(np.float32)


def exact_q(x, w1, b1, w2, b2, round_h=policy.bf16_round, round_a=policy.bf16_round):
    """(Q int64 [rows, out], hidden pre-activations z) of integer weights, computed exactly: A and H rounded to bf16 as
    the kernel rounds them, every product and sum in integers (float64 BLAS on integers far below 2^53 is exact).
    Asserts what makes the kernel's own fp32 arithmetic exact as well: integer, bf16-exact weights and biases (b2 rides
    through the bf16 image) and every partial sum of both layers below 2^22."""
    w1, b1, w2, b2 = (np.asarray(a, dtype=np.float64) for a in (w1, b1, w2, b2))
    for a in (w1, b1, w2, b2):
        assert np.array_equal(a, np.round(a)) and bf16_exact(a)
    xb = round_a(np.asarray(x, dtype=np.float32)).astype(np.float64)
    assert np.array_equal(xb, np.round(xb))
    assert (np.abs(xb) @ np.abs(w1).T + np.abs(b1)).max() < EXACT
    z = xb @ w1.T + b1
    h = round_h(np.maximum(z, 0).astype(np.float32)).astype(np.float64)
    assert (h @ np.abs(w2).T + np.abs(b2)).max() < EXACT
    return (h @ w2.T + b2).astype(np.int64), z


def small_obs(rng, rows, in_dim):
    return rng.integers(-2, 3, (rows, in_dim)).astype(np.float32)


def int_net(rng, in_dim, hidden, out):
    """W1, W2 in {-1, 0, 1}, |b1| <= 40, |b2| <= 100: with small_obs every hidden pre-activation is an integer of at most
    8 significant bits (|z| <= 2 * 105 + 40), so ReLU then bf16 is the identity."""
    return (rng.integers(-1, 2, (hidden, in_dim)).astype(np.float32), rng.integers(-40, 41, hidden).astype(np.float32),
            rng.integers(-1, 2, (out, hidden)).astype(np.float32), rng.integers(-100, 101, out).astype(np.float32))


def hidden_ties(rng, rows, in_dim, hidden, out):
    """Every hidden pre-activation an integer in [258, 510], about half of them odd: bf16 ties, which round to even
    (257 -> 256, 259 -> 260).  40 weights of +-1 per hidden unit on small_obs, b1 even in [338, 430]."""
    w1 = np.zeros((hidden, in_dim), dtype=np.float32)
    for j in range(hidden):
        w1[j, rng.choice(in_dim, 40, replace=False)] = rng.choice([-1, 1], 40)
    b1 = (2 * rng.integers(169, 216, hidden)).astype(np.float32)
    return small_obs(rng, rows, in_dim), (w1, b1, *int_net(rng, in_dim, hidden, out)[2:])


def input_ties(rng, rows, in_dim, hidden, out):
    """Observation features +-odd integers in [259, 507], ties of the bf16 conversion of A; each hidden unit reads one
    feature with weight +-1 and b1 in {-2, 0, 2}, so its pre-activation +-bf16(x) + b1 is exact in bf16 again."""
    x = rng.choice([-1, 1], (rows, in_dim)) * (2 * rng.integers(129, 254, (rows, in_dim)) + 1)
    w1 = np.zeros((hidden, in_dim), dtype=np.float32)
    w1[np.arange(hidden), rng.integers(0, in_dim, hidden)] = rng.choice([-1, 1], hidden)
    b1 = rng.choice([-2, 0, 2], hidden).astype(np.float32)
    return x.astype(np.float32), (w1, b1, *int_net(rng, in_dim, hidden, out)[2:])


@pytest.mark.parametrize("hidden", HIDDEN)
def test_exact_cases_are_exact_in_every_format(hidden):
    """Every constructed operand and pre-activation is what the case claims, the integer Q equals
    evgsim.policy.reference_forward (float32 numpy) exactly, and the rounding the tie cases target changes Q."""
    rng = np.random.default_rng(hidden)
    rows = 40 if hidden > 4096 else 300
    x, w = small_obs(rng, rows, 105), int_net(rng, 105, hidden, 144)
    q, z = exact_q(x, *w)
    assert bf16_exact(x) and np.abs(z).max() <= 256 and bf16_exact(z)
    assert np.array_equal(policy.reference_forward(x, *w), q.astype(np.float32))
    if hidden > 4096:
        return
    x, w = hidden_ties(rng, rows, 105, hidden, 144)
    q, z = exact_q(x, *w)
    assert bf16_exact(x) and z.min() >= 257 and z.max() <= 511 and (z % 2 == 1).mean() > 0.4
    assert np.array_equal(policy.reference_forward(x, *w), q.astype(np.float32))
    assert (exact_q(x, *w, round_h=bf16_rz)[0] != q).any(1).mean() > 0.15  # H rounded toward zero gives another Q
    x, w = input_ties(rng, rows, 105, hidden, 144)
    q, z = exact_q(x, *w)
    assert (np.abs(x) % 2 == 1).all() and np.abs(x).min() > 256 and bf16_exact(np.maximum(z, 0))
    assert np.array_equal(policy.reference_forward(x, *w), q.astype(np.float32))
    assert (exact_q(x, *w, round_a=bf16_rz)[0] != q).any(1).mean() > 0.15  # A rounded toward zero gives another Q


def linear(rng, out, inp, scale=1.0):
    """(weight, bias) of torch.nn.Linear's default initialisation (uniform in +-1/sqrt(fan_in)) times `scale`."""
    s = scale / np.sqrt(inp)
    return [rng.uniform(-s, s, (out, inp)).astype(np.float32), rng.uniform(-s, s, out).astype(np.float32)]


def float_dqn(rng, in_dim, hidden, out):
    return linear(rng, hidden, in_dim, 3.0) + linear(rng, out, hidden, 3.0)


def ppo_net(rng, in_dim, latent, out):
    return linear(rng, latent, in_dim) + linear(rng, latent, latent) + linear(rng, out, latent)


def q_and_bound(x, w1, b1, w2, b2, block=8192):
    """float64 Q of the bf16-rounded operands, and a per-element bound on the kernel's distance from it.  An fp32 sum of
    K terms is within K * 2^-23 of the sum of their magnitudes (round-to-nearest or truncating adders; the zero padding
    adds nothing): K = inputs + 1 (b1) in layer 1, hidden units + 1 (b2) in layer 2.  A hidden activation is
    bf16(relu(D1)) with D1 within that error e1 of the exact pre-activation z, so it lies between bf16(relu(z - e1)) and
    bf16(relu(z + e1)) (both roundings are monotone): the two differ only where z is that close to a rounding boundary,
    and only there does the bound grant a flipped activation (one bf16 step)."""
    f = lambda a: policy.bf16_round(np.asarray(a, dtype=np.float32)).astype(np.float64)  # noqa: E731
    w1b, b1b, w2b, b2b = map(f, (w1, b1, w2, b2))
    k1, k2 = w1.shape[1] + 1, w1.shape[0] + 1
    q, bound = [], []
    for r0 in range(0, len(x), block):
        xb = f(x[r0:r0 + block])
        z = xb @ w1b.T + b1b
        e1 = k1 * 2.0 ** -23 * (np.abs(xb) @ np.abs(w1b).T + np.abs(b1b))
        e1 += (np.abs(z) + e1) * 2.0 ** -22  # the float32 conversion inside f
        lo, hi = f(np.maximum(z - e1, 0)), f(np.maximum(z + e1, 0))
        q.append(f(np.maximum(z, 0)) @ w2b.T + b2b)
        bound.append((hi - lo) @ np.abs(w2b).T + k2 * 2.0 ** -23 * (hi @ np.abs(w2b).T + np.abs(b2b)))
    return np.concatenate(q), np.concatenate(bound)


def test_float_bound_holds_for_the_float32_reference():
    """reference_forward (the kernel's arithmetic in float32 numpy, another summation order) stays within the bound,
    which scales with each element's own terms and for most elements lies below half the earlier bar of 2e-3 of the
    batch's largest |Q|."""
    rng = np.random.default_rng(2)
    x = rng.integers(-3, 300, (500, 105)).astype(np.float32)
    for hidden in (1, 191, 528):
        w = float_dqn(rng, 105, hidden, 132)
        q, bound = q_and_bound(x, *w)
        assert (np.abs(policy.reference_forward(x, *w) - q) <= bound).all()
        assert np.median(bound) < 1e-3 * np.abs(q).max()


# ---------------------------------------------------------------- GPU fixtures and helpers

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


def mid_game(evg, cfg, n, seed=17, offset=0, turns=30):
    env = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg, env_id_offset=offset)
    env.reset()
    for _ in range(turns):  # real mid-game observations, different in every row
        env.step(env.random_actions())
    return env


@pytest.fixture(scope="module")
def big(evg, cfg, sms):
    """Matches whose per-player rows make ~2.5 tiles per CTA, the last one partial (CTAs handle 2 or 3 tiles); the rows
    of both players make ~5 (CTAs handle 4 or 5)."""
    tiles = (5 * sms + 1) // 2
    return mid_game(evg, cfg, (tiles - 1) * 128 + 54)


@pytest.fixture(scope="module")
def env_of(evg, cfg):
    made = {}

    def get(n):
        if n not in made:
            made[n] = evg.BatchedEvergladesEnv(n, seed=1, config=cfg)
        return made[n]
    return get


def dqn_q(env, w, obs=None):
    """FusedDQN's Q [rows, out] for obs (float32 numpy [rows, obs_len]; default env.obs), both layouts (checked equal)."""
    import torch
    fused = policy.FusedDQN(env, weights=w)
    o = None if obs is None else torch.from_numpy(np.ascontiguousarray(obs)).to(env.device).view(env.num_envs, 2, env.obs_len)
    q = fused.forward(o).cpu().numpy().reshape(-1, fused.out_dim)
    assert np.array_equal(fused.forward_t(o).cpu().numpy(), q.T)
    return q


def checked_tiles(rows, sms):
    """The tiles whose draws are replayed on the CPU: the first CTAs' first, second and third tiles, the last CTA's
    first and second, every 23rd tile and the last, partial one."""
    n = -(-rows // 128)
    t = {0, 1, sms - 1, sms, sms + 1, 2 * sms - 1, 2 * sms, 2 * sms + 1, n - 2, n - 1} | set(range(0, n, 23))
    return sorted(x for x in t if x < n)


def expected_draws(env, probs, player, tiles=None):
    """(rows, ppo_sample of those rows' probabilities with the tape's uniforms): every row, or the rows of `tiles`.
    Rows are (match, player) pairs for player -1, matches otherwise."""
    import ppo_sampling as ps
    per = 2 if player < 0 else 1
    spans = [(0, len(probs))] if tiles is None else [(128 * t, min(128 * t + 128, len(probs))) for t in tiles]
    rows, u = [], []
    for r0, r1 in spans:
        m0 = r0 // per
        st = env.get_state(m0, (r1 - 1) // per + 1 - m0)
        for r in range(r0, r1):
            s = st[r // per - m0]
            rows.append(r)
            u.append(ps.policy_uniforms(env.seed, env.env_id_offset + r // per, int(s["turn"]), r % 2 if per == 2 else player, int(s["episode"])))
    rows = np.array(rows)
    return rows, ps.ppo_sample_rows(probs[rows], np.stack(u))


def check_ppo(env, w, player=-1, div=12, mod=11, tiles=None):
    """FusedPPO against reference_forward_ppo (5e-3 of every probability, rows summing to 1), its draws against
    ppo_sample_rows and its action rows against their unravel."""
    from oracle import policy_decode
    fused = policy.FusedPPO(env, weights=w, player=player, div=div, mod=mod)
    acts = fused(want_probs=True).cpu().numpy()
    out = fused.out_dim
    probs, idx = fused.probs.cpu().numpy().reshape(-1, out), fused.idx.cpu().numpy().reshape(-1, 7)
    obs = env.obs.cpu().numpy()
    want = policy.reference_forward_ppo(obs.reshape(-1, env.obs_len) if player < 0 else obs[:, player], *w)
    assert np.isfinite(probs).all() and (probs > 0).all()
    assert np.abs(probs.sum(-1) - 1).max() <= 1e-5
    assert (np.abs(probs - want) <= 5e-3 * want).all(), np.abs(probs / want - 1).max()
    rows, draws = expected_draws(env, probs, player, tiles)
    assert np.array_equal(idx[rows], draws)
    played = acts.reshape(-1, 7, 2) if player < 0 else acts[:, player]
    assert np.array_equal(played, policy_decode.ppo_unravel(idx, div, mod).astype(np.int8))
    return fused


# ---------------------------------------------------------------- DQN

@gpu
@pytest.mark.parametrize("out", OUTS)
@pytest.mark.parametrize("hidden", HIDDEN)
def test_dqn_exact_q_at_every_width(env_of, hidden, out):
    """One partial tile (two for 12,288 hidden units, 65 chunks): bias unit in every position of its chunk, 1 to 144
    outputs across the 36-column quarters each thread stores."""
    env = env_of(100 if hidden > 4096 else 45)
    rng = np.random.default_rng(hidden * 1000 + out)
    x, w = small_obs(rng, 2 * env.num_envs, 105), int_net(rng, 105, hidden, out)
    assert np.array_equal(dqn_q(env, w, x), exact_q(x, *w)[0])


@gpu
@pytest.mark.parametrize("hidden,out", [(1, 144), (191, 37), (192, 1), (383, 12), (528, 132), (528, 36)])
def test_dqn_exact_q_multi_tile(big, hidden, out):
    rng = np.random.default_rng(hidden + out)
    x, w = small_obs(rng, 2 * big.num_envs, 105), int_net(rng, 105, hidden, out)
    assert np.array_equal(dqn_q(big, w, x), exact_q(x, *w)[0])


@gpu
@pytest.mark.parametrize("multi", [False, True])
@pytest.mark.parametrize("case", [hidden_ties, input_ties])
def test_dqn_rounds_ties_to_nearest_even(env_of, big, case, multi):
    env = big if multi else env_of(45)
    hidden, out = (528, 132) if multi else (191, 37)
    x, w = case(np.random.default_rng(7), 2 * env.num_envs, 105, hidden, out)
    assert np.array_equal(dqn_q(env, w, x), exact_q(x, *w)[0])


@gpu
def test_dqn_multi_tile_real_observations(big):
    """Mid-game rows: exact with integer weights, within the per-element float64 bound with a float net, and the same
    bits for every row wherever it sits (rows permuted)."""
    rng = np.random.default_rng(3)
    x = big.obs.cpu().numpy().reshape(-1, 105)
    assert len(np.unique(x, axis=0)) > len(x) // 2  # distinct rows
    w = int_net(rng, 105, 528, 132)
    assert np.array_equal(dqn_q(big, w), exact_q(x, *w)[0])
    wf = float_dqn(rng, 105, 528, 132)
    q = dqn_q(big, wf)
    want, bound = q_and_bound(x, *wf)
    assert np.isfinite(q).all() and (np.abs(q - want) <= bound).all(), np.abs(q - want).max()
    perm = rng.permutation(len(x))
    assert np.array_equal(dqn_q(big, wf, x[perm]), q[perm])


@gpu
def test_dqn_float_bound_holds_at_every_width(env_of):
    env = env_of(45)
    rng = np.random.default_rng(11)
    for hidden, out in ((1, 144), (191, 37), (12288, 132)):
        x = rng.integers(-3, 60, (2 * env.num_envs, 105)).astype(np.float32)
        wf = float_dqn(rng, 105, hidden, out)
        q = dqn_q(env, wf, x)
        want, bound = q_and_bound(x, *wf)
        assert (np.abs(q - want) <= bound).all(), (hidden, out, np.abs(q - want).max())


# ---------------------------------------------------------------- PPO

@gpu
@pytest.mark.parametrize("player,latent", [(-1, 256), (0, 129), (1, 64)])
def test_ppo_multi_tile(big, sms, player, latent):
    rows = big.num_envs * (2 if player < 0 else 1)
    check_ppo(big, ppo_net(np.random.default_rng(latent), 105, latent, 132), player, tiles=checked_tiles(rows, sms))


@gpu
@pytest.mark.parametrize("out_dim,div,mod", [(7, 2, 3), (16, 4, 4), (17, 5, 3), (131, 11, 12), (144, 12, 12)])
@pytest.mark.parametrize("latent", [16, 193])
def test_ppo_output_widths(evg, cfg, out_dim, div, mod, latent):
    env = mid_game(evg, cfg, 333)
    check_ppo(env, ppo_net(np.random.default_rng(out_dim + latent), 105, latent, out_dim), div=div, mod=mod)


# ---------------------------------------------------------------- both: bitwise independence of the batch layout

@gpu
def test_shards_agree_bit_for_bit(evg, cfg, big):
    """The whole batch against three shards (env_id_offset) that put every row into another tile and CTA."""
    import torch
    m = big.num_envs
    cuts = [0, m // 7 + 1, m // 2 + 37, m]
    shards = [mid_game(evg, cfg, b - a, offset=a) for a, b in zip(cuts, cuts[1:])]
    for s, a, b in zip(shards, cuts, cuts[1:]):
        assert torch.equal(s.obs, big.obs[a:b])
    rng = np.random.default_rng(5)
    wf = float_dqn(rng, 105, 528, 132)
    q = dqn_q(big, wf)
    assert np.array_equal(np.concatenate([dqn_q(s, wf) for s in shards]), q)
    wp = ppo_net(rng, 105, 256, 132)
    whole = policy.FusedPPO(big, weights=wp)
    acts = whole(want_probs=True).clone()
    parts = []
    for s in shards:
        f = policy.FusedPPO(s, weights=wp)
        a = f(want_probs=True)
        parts.append((f.idx.clone(), f.probs.clone(), a.clone()))
    assert torch.equal(torch.cat([p[0] for p in parts]), whole.idx)
    assert torch.equal(torch.cat([p[1] for p in parts]), whole.probs)
    assert torch.equal(torch.cat([p[2] for p in parts]), acts)


# ---------------------------------------------------------------- other observation widths

def write_ring16(tmp_path):
    """16 nodes on a ring with chords, bases at 1 and 9, mirror map i -> ((i + 7) % 16) + 1: 125-value observations,
    DQN's bias input in the last 8 columns of the second swizzle atom."""
    n = 16
    nodes = []
    for i in range(1, n + 1):
        nb = {(i % n) + 1: 2 + i % 3, ((i - 2) % n) + 1: 2 + (i - 1) % 3, ((i + 7) % n) + 1: 5}
        nodes.append({"ID": i, "Connections": [{"ConnectedID": d, "Distance": w} for d, w in sorted(nb.items())],
                      "ControlPoints": 300 if i in (1, 9) else 50 + i, "Resource": ["DEFEND"] if i % 5 == 0 else [],
                      "StructureDefense": 1 + (i % 4) * 0.25, "TeamStart": {1: 0, 9: 1}.get(i, -1)})
    p1 = [0] + [((i + 7) % n) + 1 for i in range(1, n + 1)]
    (tmp_path / "Ring16.json").write_text(json.dumps({"MapName": "ring16", "nodes": nodes, "P1NodeMap": p1}))
    (tmp_path / "Setup.json").write_text(json.dumps({"TurnLimit": 50, "CaptureBonus": 700, "UnitBudget": 100}))
    return str(tmp_path)


@gpu
@pytest.mark.parametrize("nodes", [7, 16])
def test_other_observation_widths(evg, tmp_path, nodes):
    """7 nodes: 89 values, DQN's bias input off an 8-column boundary; 16 nodes: 125 values, the widest map that fits."""
    from test_gpu_generic import write_configs
    if nodes == 7:
        cfg = evg.load_config(write_configs(tmp_path, 100), "Map7.json", "Units4.json", "Setup.json")
    else:
        cfg = evg.load_config(write_ring16(tmp_path), "Ring16.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")
    env = mid_game(evg, cfg, 1500)
    width = 1 + 4 * nodes + 60
    assert env.obs_len == width
    x = env.obs.cpu().numpy().reshape(-1, width)
    rng = np.random.default_rng(nodes)
    w = int_net(rng, width, 191, 37)
    assert np.array_equal(dqn_q(env, w), exact_q(x, *w)[0])
    wf = float_dqn(rng, width, 528, 132)
    want, bound = q_and_bound(x, *wf)
    assert (np.abs(dqn_q(env, wf) - want) <= bound).all()
    check_ppo(env, ppo_net(rng, width, 130, 132))


@gpu
def test_observations_wider_than_the_tiling_are_refused(evg, tmp_path):
    """32 nodes make 189-value rows, more than the 128 input columns both kernels are tiled for.  The wrappers refuse a
    network of another width; the C API itself refuses the map, here with images packed for a 105-wide network."""
    import torch
    from evgsim import _capi
    from test_gpu_generic import write_ring32
    cfg = evg.load_config(write_ring32(tmp_path), "Ring32.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")
    env = evg.BatchedEvergladesEnv(64, seed=2, config=cfg)
    env.reset()
    assert env.obs_len == 189
    rng = np.random.default_rng(0)
    wd, wp = int_net(rng, 105, 528, 132), ppo_net(rng, 105, 128, 132)
    with pytest.raises(ValueError, match="105 inputs"):
        policy.FusedDQN(env, weights=wd)
    with pytest.raises(ValueError, match="105 inputs"):
        policy.FusedPPO(env, weights=wp)
    dev = env.device
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    img1, img2, hidden, out = policy.pack_mlp(*wd)
    i1, i2 = torch.from_numpy(img1).to(dev), torch.from_numpy(img2).to(dev)
    q = torch.zeros((128, out), dtype=torch.float32, device=dev)
    assert env._lib.evg_policy_mlp(env._h, ptr(env.obs), 128, ptr(i1), ptr(i2), hidden, out, ptr(q), 0, env._stream()) == -1  # EVG_E_ARG
    assert b"189" in _capi.load().evg_last_error()
    p1, p2, p3, bias = (torch.from_numpy(a).to(dev) for a in policy.pack_ppo(*wp)[:4])
    idx = torch.zeros((64, 2, 7), dtype=torch.int64, device=dev)
    assert env._lib.evg_policy_ppo(env._h, ptr(env.obs), -1, ptr(p1), ptr(p2), ptr(p3), ptr(bias), 128, 132, 12, 11, ptr(env._actions),
                                   ptr(idx), None, env._stream()) == -1  # EVG_E_ARG
    assert b"189" in _capi.load().evg_last_error()
    torch.cuda.synchronize()
    assert not q.any() and not idx.any()


# ---------------------------------------------------------------- the wrappers' own checks

@gpu
def test_wrappers_check_widths_and_observations(env_of):
    import torch
    env = env_of(45)
    rng = np.random.default_rng(1)
    with pytest.raises(ValueError, match="100 inputs"):  # b1 would meet observation feature 100 instead of the constant 1
        policy.FusedDQN(env, weights=int_net(rng, 100, 64, 12))
    with pytest.raises(ValueError, match="100 inputs"):
        policy.FusedDQN(env, torch.nn.Sequential(torch.nn.Linear(100, 64), torch.nn.ReLU(), torch.nn.Linear(64, 12)))
    with pytest.raises(ValueError, match="100 inputs"):
        policy.FusedPPO(env, weights=ppo_net(rng, 100, 32, 132))
    w = int_net(rng, 105, 64, 12)
    fused = policy.FusedDQN(env, weights=w)
    x = small_obs(rng, 90, 105)
    good = torch.from_numpy(x).to(env.device).view(45, 2, 105)
    bad = {"float64": good.double(), "on the host": good.cpu(), "not contiguous": good.transpose(0, 1),
           "short": good.reshape(-1)[:-1], "long": torch.zeros((46, 2, 105), device=env.device)}
    for name, obs in bad.items():
        for run in (fused.forward, fused.forward_t):
            with pytest.raises(ValueError):
                run(obs)
    assert np.array_equal(fused.forward(good).cpu().numpy().reshape(90, 12), exact_q(x, *w)[0])
