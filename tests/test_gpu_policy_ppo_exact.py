"""The fused PPO actor (evg_policy_ppo) on a network whose every hidden activation has one exact value, with its
probabilities within a derived bound of float64 and its log-probabilities within a derived bound of the float64 truth,
at every tiling edge.

The exact network.  Each hidden layer has two kinds of units:
- Boolean units: W in 40 {-1, 0, 1} over integer observations (bf16 rounding keeps them integers) or over the previous
  layer's boolean units, b = +-20.  Every pre-activation is an odd multiple of 20, so H = bf16(tanhf(z)) = +-1 even if
  tanhf stops an ulp short of 1.
- Analog units: a layer-1 analog unit reads one observation feature with a weight +-2^-e, e in 8..10, plus a bias on
  the 2^-12 grid; a layer-2 analog unit reads one layer-1 analog unit with a weight in {+-1/2, +-1}, up to two boolean
  units with +-1/8, and a bias on the same grid.  Each product and sum is then exact in float32 in any order, and so is
  z.  The generator picks every analog bias so that tanh(z) sits at least M = 8 float32 ulps from every bf16 rounding
  midpoint for every z the unit can reach (layer 1: every bf16-rounded integer in [-700, 700]; layer 2: every value its
  inputs can take), and |H| >= 2^-4.  tanhf is within 2 ulp of tanh (CUDA Programming Guide, single-precision maximum
  ulp errors), so H = bf16_rne(tanhf(z)) has one value, and it is a multiple of 2^-11: every later sum sits on a grid.
- Output layer: eighths on the boolean layer-2 units and one weight in {+-1/2, +-1} on one analog layer-2 unit per
  output, b3 in eighths.  The argument of tanh is exact; only tanhf, expf, the sum and the division round.  A one-ulp
  error in an analog H2 moves a probability by 1e-4 to 1e-3, 10 to 100 times the bound below.
machine() is that network in float64 numpy, asserting every condition above on the rows it is given: the exact H1 and
H2, and float64 probabilities.

The probability bound is tests/test_gpu_policy_rppo_exact.py's P_REL (about 9.6e-6): the same tanhf, expf, float32 sum
of at most 144 terms and correctly rounded division.  Most of it is the sum's worst case, 143 u.  The probabilities of a
row share that one computed sum, so their ratios are free of it: q_i / q_j = (e_i / e_j)(1 + d_i) / (1 + d_j) with
|d| <= u (the divisions), and each e within EPS_E of exp(tanh t) (tanhf, expf).  Every ratio to the row's largest
probability is therefore within R_REL = ((1 + EPS_E)(1 + u) / ((1 - EPS_E)(1 - u)))^2 - 1, about 2.1e-6, of the exact
ratio: the bound that sees an approximate tanh or exp on the output layer.

The log-probability bound.  The kernel writes logf(q_s / T_k) for draw k, where q_j are its probabilities and T_k is
its float32 sum, in ascending j, of the q_j not drawn before draw k.  The truth is log(p_s / R_k), with p the exact
probabilities and R_k = 1 - sum_{i<k} p_{s_i}, the sum of the exact p_j not drawn before.
- q_j = p_j (1 + th_j) with |th_j| <= P_REL, so the exact sum of the q_j not drawn lies within a factor 1 +- P_REL of
  R_k; T_k, a float32 sum of at most 144 positive terms, is within GAMMA = 143 u / (1 - 143 u) of that sum (u = 2^-24).
- The quotient q_s / T_k is correctly rounded: relative error u.
- So q_s / T_k lies within a factor (1 + P_REL)(1 + u) / ((1 - P_REL)(1 - GAMMA)) of p_s / R_k, and its log within the
  log of that factor, about 2 P_REL + GAMMA = 2.8e-5.
- logf is within 1 ulp (CUDA Programming Guide) of a value of magnitude at most 7 (every p_j >= e^-2 / 144, so the log
  of p_s / R_k >= log p_s >= -7): 2^-21 more.
LOGP_ABS, the sum, is about 2.8e-5, 350 times tighter than the 1e-2 to which tests/test_gpu_policy_logp.py re-evaluates
a stored rollout.  Unlike that module's 2e-6 check of logp against the kernel's own probabilities, it ties logp to the
network: a wrong forward pass no longer gives a "correct" logp.

The CPU tests at the top check the construction: its margins, that the float32 reference agrees with the machine, that
each plausible defect of the kernel leaves the bound, and that the machine refuses rows it cannot vouch for."""
import numpy as np
import pytest

from evgsim import policy
from test_gpu_policy_rppo_exact import EPS_E, GAMMA, LATENTS, OUT_CASES, P_REL, U, obs_rows, synthetic_obs
from test_gpu_policy_tiling import big, bf16_rz, checked_tiles, evg, expected_draws, mid_game, sms, write_ring16  # noqa: F401

gpu = pytest.mark.gpu
M = 8                   # margin of every analog tanh from a bf16 rounding midpoint, in float32 ulps
X_MAX = 700             # layer-1 analog units keep their margins for every bf16-rounded integer in [-X_MAX, X_MAX]
GRID = 2.0 ** -12       # the analog biases' grid
R_REL = ((1 + EPS_E) * (1 + U) / ((1 - EPS_E) * (1 - U))) ** 2 - 1
LOGP_ABS = np.log((1 + P_REL) * (1 + U) / ((1 - P_REL) * (1 - GAMMA))) + 2.0 ** -21
TIE_LATENTS = [129, 256]  # wide enough that most rows carry a changed H1 on to the probabilities
MUTANTS = ["H1_rz", "H2_rz", "tanh_approx_hidden", "tanh_approx_out", "bias_bf16", "l2_chunk", "l3_chunk"]
DOMAIN = np.unique(policy.bf16_round(np.arange(-X_MAX, X_MAX + 1, dtype=np.float32))).astype(np.float64)


# ---------------------------------------------------------------- the exact network and its machine (checked on the CPU)

def margin(z):
    """Distance, in float32 ulps, from tanh(z) to the nearest bf16 rounding midpoint (half an ulp for the float32
    rounding of tanh(z) itself subtracted)."""
    t = np.abs(np.tanh(np.asarray(z, dtype=np.float64))).astype(np.float32)
    return np.abs((t.view(np.uint32) & 0xFFFF).astype(np.int64) - 0x8000) - 0.5


def bf16_tanh(z, rnd=policy.bf16_round):
    return rnd(np.tanh(np.asarray(z, dtype=np.float64)).astype(np.float32)).astype(np.float64)


def analog_bias(rng, reach):
    """A bias on the 2^-12 grid such that every z = b + reach keeps the margin M and |bf16(tanh z)| >= 2^-4: z keeps one
    sign, at least 0.07 from 0."""
    lo = np.abs(reach).max() + 0.07
    for _ in range(200):
        b = rng.choice([-1, 1]) * rng.integers(int(np.ceil(lo / GRID)), int((lo + 1.5) / GRID)) * GRID
        z = b + reach
        if margin(z).min() >= M and np.abs(bf16_tanh(z)).min() >= 2.0 ** -4:
            return b
    raise AssertionError("no bias keeps the margins")


class ExactPPO:
    """Weights (float32, torch.nn.Linear's layout: w1, b1, w2, b2, w3, b3) of the network of the module docstring, and
    which units of each hidden layer are analog (about a third, at least one)."""

    def __init__(self, rng, in_dim, latent, out_dim=132):
        L = latent
        tern = lambda *shape: 40.0 * rng.integers(-1, 2, shape)  # noqa: E731
        pm20 = lambda *shape: 20.0 * rng.choice([-1, 1], shape)  # noqa: E731
        self.analog1, self.analog2 = np.zeros(L, dtype=bool), np.zeros(L, dtype=bool)
        self.analog1[rng.choice(L, max(1, L // 3), replace=False)] = True
        self.analog2[rng.choice(L, max(1, L // 3), replace=False)] = True
        a1, a2 = np.flatnonzero(self.analog1), np.flatnonzero(self.analog2)
        b1 = np.flatnonzero(~self.analog1)
        w1, bias1 = tern(L, in_dim), pm20(L)
        w1[a1] = 0
        h1_values = {}  # every H a layer-1 analog unit can take
        for j in a1:
            f, s = rng.integers(in_dim), rng.choice([-1, 1]) * 2.0 ** -rng.integers(8, 11)
            w1[j, f] = s
            bias1[j] = analog_bias(rng, s * DOMAIN)
            h1_values[j] = np.unique(bf16_tanh(bias1[j] + s * DOMAIN))
        w2, bias2 = tern(L, L), pm20(L)
        w2[:, a1] = 0
        w2[a2] = 0
        for j in a2:
            src = rng.choice(a1)
            w2[j, src] = rng.choice([-1, -0.5, 0.5, 1])
            reach = w2[j, src] * h1_values[src]
            for k in rng.choice(b1, min(2, len(b1)), replace=False):
                w2[j, k] = rng.choice([-1, 1]) / 8
                reach = np.concatenate([reach + 1 / 8, reach - 1 / 8])
            bias2[j] = analog_bias(rng, np.unique(reach))
        n_bool = L - len(a2)
        w3 = rng.choice([-1.0, 1.0], (out_dim, L)) * (rng.random((out_dim, L)) < min(1.0, 36 / max(1, n_bool))) / 8
        w3[:, a2] = 0
        w3[np.arange(out_dim), rng.choice(a2, out_dim)] = rng.choice([-1, -0.5, 0.5, 1], out_dim)
        self.weights = [np.asarray(a, dtype=np.float32) for a in (w1, bias1, w2, bias2, w3, rng.integers(-8, 9, out_dim) / 8)]


def on_grid(a, step):
    return np.array_equal(np.asarray(a, dtype=np.float64) / step, np.round(np.asarray(a, dtype=np.float64) / step))


def check_exactness(net):
    """The weight conditions under which every sum of the kernel is exact in float32, in any order."""
    w1, b1, w2, b2, w3, b3 = (np.asarray(a, dtype=np.float64) for a in net.weights)
    a1, a2 = net.analog1, net.analog2
    for w in (w1, w2, w3):
        assert np.array_equal(policy.bf16_round(w.astype(np.float32)), w), "weights not bf16-exact"
    assert on_grid(w1[~a1], 40) and on_grid(w2[~a2], 40) and not w2[np.ix_(~a2, a1)].any(), "boolean units off their grid"
    assert (np.abs(b1[~a1]) == 20).all() and (np.abs(b2[~a2]) == 20).all(), "boolean biases"
    assert ((w1[a1] != 0).sum(1) == 1).all() and on_grid(w1[a1], 2.0 ** -10), "layer-1 analog weights off their grid"
    assert on_grid(w2[np.ix_(a2, a1)], 0.5) and on_grid(w2[a2], 1 / 8), "layer-2 analog weights off their grid"
    assert on_grid(b1, GRID) and on_grid(b2, GRID), "analog biases off their grid"
    assert on_grid(w3[:, a2], 0.5) and on_grid(w3, 1 / 8) and on_grid(b3, 1 / 8), "output layer off its grid"


def hidden(z, analog, check, rnd, approx):
    """bf16(tanh(z)) of one hidden layer; with check, asserts the boolean margins, the analog margins and |H| >= 2^-4."""
    if check:
        assert np.abs(z[:, ~analog]).min(initial=20) >= 20, "boolean pre-activation inside +-20"
        assert margin(z[:, analog]).min() >= M, "analog margin below M ulps"
    t = np.tanh(z)
    if approx:  # tanh.approx.f32: relative error about 2^-11
        t = t * (1 + 2.0 ** -11 * np.random.default_rng(1).choice([-1, 1], t.shape))
    H = rnd(t.astype(np.float32)).astype(np.float64)
    if check:
        assert np.abs(H[:, analog]).min() >= 2.0 ** -4, "analog activation below 2^-4"
    return H


def machine(obs, net, mutant=None):
    """The exact network on observation rows: (H1, H2 float32 [rows, L], probabilities float64 [rows, out]).  Asserts
    integer observations, the weight grids, every sum within float32's exact range and every margin.  `mutant` runs a
    defect instead (without the assertions on rows): H1 or H2 rounded toward zero, a tanh.approx-sized error in the
    hidden epilogue or on the output tanh, b1 and b2 rounded to bf16 before the add, or (L > 128) layer 2 or 3 missing
    its second K chunk."""
    check = mutant is None
    check_exactness(net)
    w1, b1, w2, b2, w3, b3 = (np.asarray(a, dtype=np.float64) for a in net.weights)
    if mutant == "bias_bf16":
        b1, b2 = (policy.bf16_round(b.astype(np.float32)).astype(np.float64) for b in (b1, b2))
    x = policy.bf16_round(np.asarray(obs, dtype=np.float32)).astype(np.float64)
    assert np.array_equal(x, np.round(x)), "observations not integers"
    assert (np.abs(x) @ np.abs(w1[~net.analog1]).T).max(initial=0) + 20 < 2 ** 24, "layer-1 sums beyond float32's integers"
    approx = mutant == "tanh_approx_hidden"
    H1 = hidden(x @ w1.T + b1, net.analog1, check, bf16_rz if mutant == "H1_rz" else policy.bf16_round, approx)
    H1in = H1.copy()
    if mutant == "l2_chunk":
        H1in[:, 128:] = 0
    assert (np.abs(H1in) @ np.abs(w2[net.analog2]).T).max() + np.abs(b2).max() < 2 ** 11, "layer-2 analog sums too wide"
    H2 = hidden(H1in @ w2.T + b2, net.analog2, check, bf16_rz if mutant == "H2_rz" else policy.bf16_round, approx)
    H2in = H2.copy()
    if mutant == "l3_chunk":
        H2in[:, 128:] = 0
    assert (np.abs(H2in) @ np.abs(w3).T).max() + 1 < 2 ** 11, "output sums too wide"
    y = np.tanh(H2in @ w3.T + b3)
    if mutant == "tanh_approx_out":
        y = y * (1 + 2.0 ** -11 * np.random.default_rng(2).choice([-1, 1], y.shape))
    e = np.exp(y)
    return H1.astype(np.float32), H2.astype(np.float32), e / e.sum(-1, keepdims=True)


def true_logp(p, idx):
    """float64 log(p[s_k] / (1 - sum_{i<k} p[s_i])) of the draws idx [rows, 7] from the exact probabilities p."""
    ps = np.take_along_axis(p, np.asarray(idx, dtype=np.int64), axis=1)
    return np.log(ps / (1 - (np.cumsum(ps, axis=1) - ps)))


def ratio_error(q, p):
    """Largest relative distance of q_i / q_j from p_i / p_j, with j each row's largest q."""
    q = np.asarray(q, dtype=np.float64)
    j = np.argmax(q, axis=-1)[:, None]
    want = p / np.take_along_axis(p, j, axis=1)
    return (np.abs(q / np.take_along_axis(q, j, axis=1) - want) / want).max()


def float32_hidden(obs, weights):
    """H1 and H2 as reference_forward_ppo computes them (float32 numpy, bf16-rounded operands)."""
    f32, rnd = np.float32, policy.bf16_round
    w1, b1, w2, b2 = weights[:4]
    h1 = rnd(np.tanh((rnd(np.asarray(obs, dtype=f32)) @ rnd(w1).T).astype(f32) + b1).astype(f32))
    return h1, rnd(np.tanh((h1 @ rnd(w2).T).astype(f32) + b2).astype(f32))


@pytest.mark.parametrize("latent", [1, 17, 128, 129, 200, 256])
def test_machine_is_the_float32_reference_and_sees_every_defect(latent):
    """The float32 statement of the kernel (reference_forward_ppo) gives the machine's probabilities within P_REL,
    their ratios within R_REL and its log-probabilities, for the sampler's draws, within LOGP_ABS; the machine's H1 and
    H2 are the float32 statement's bit for bit, and the analog units do take fractional values; each defect leaves the
    bound in more than 20 % of rows."""
    import ppo_logp
    import ppo_sampling as ps
    rng = np.random.default_rng(latent)
    rows = 600
    net = ExactPPO(rng, 105, latent)
    x = synthetic_obs(rng, rows, 105)
    H1, H2, p = machine(x, net)
    ref_p = policy.reference_forward_ppo(x, *net.weights)
    assert (np.abs(ref_p - p) <= P_REL * p).all(), np.abs(ref_p / p - 1).max()
    assert ratio_error(ref_p, p) <= R_REL
    h1, h2 = float32_hidden(x, net.weights)
    assert np.array_equal(h1, H1) and np.array_equal(h2, H2)
    for H, analog in ((H1, net.analog1), (H2, net.analog2)):
        assert (np.abs(H[:, ~analog]) == 1).all()
        frac = np.abs(H[:, analog]) < 1
        assert frac.mean() > 0.5 and len(np.unique(H[:, analog][frac])) > min(20, analog.sum())
    idx = ps.ppo_sample_rows(ref_p, rng.random((rows, 7)).astype(np.float32))
    assert np.abs(ppo_logp.ppo_logp_rows(ref_p, idx) - true_logp(p, idx)).max() <= LOGP_ABS
    assert 4e-6 < P_REL < 1.1e-5 and 2e-6 < R_REL < 2.5e-6 and 2.5e-5 < LOGP_ABS < 3.5e-5
    if latent == 1:
        return
    for mutant in MUTANTS:
        if mutant.endswith("chunk") and latent <= 128:
            continue
        caught = (np.abs(machine(x, net, mutant)[2] - p) > P_REL * p).any(1)
        assert caught.mean() > 0.2, (mutant, caught.mean())


def test_the_margins_are_checked():
    """machine() refuses what it could not vouch for: a fractional observation, an analog pre-activation within M ulps
    of a bf16 rounding midpoint, a bias off the 2^-12 grid."""
    rng = np.random.default_rng(0)
    net = ExactPPO(rng, 105, 40)
    x = synthetic_obs(rng, 10, 105)
    machine(x, net)
    with pytest.raises(AssertionError, match="integers"):
        machine(x + 0.5, net)
    j = np.flatnonzero(net.analog1)[0]
    f = np.flatnonzero(net.weights[0][j])[0]
    s, b = float(net.weights[0][j, f]), float(net.weights[1][j])
    near = b + GRID * np.arange(-4096, 4097)
    near = near[margin(near + s * policy.bf16_round(x[0, f])) < M]
    assert len(near)
    net.weights[1] = net.weights[1].copy()
    net.weights[1][j] = near[np.argmin(np.abs(near - b))]
    with pytest.raises(AssertionError, match="margin"):
        machine(x, net)
    net.weights[1][j] = b + 2.0 ** -20
    with pytest.raises(AssertionError, match="grid"):
        machine(x, net)


def tie_rows(latent, rows):
    """(an exact network, integer observation rows) whose values are odd in +-[259, 599] on every feature an analog
    layer-1 unit reads and on about half the others: bf16 ties (259 -> 260) and other inexact values, which the kernel
    must round to nearest even.  The others are integers in [-100, 150]."""
    rng = np.random.default_rng(latent)
    net = ExactPPO(rng, 105, latent)
    x = rng.integers(-100, 151, (rows, 105))
    odd = rng.random(x.shape) < 0.5
    odd[:, net.weights[0][net.analog1].any(0)] = True
    x[odd] = rng.choice([-1, 1], odd.sum()) * (2 * rng.integers(129, 300, odd.sum()) + 1)
    return net, x.astype(np.float32)


@pytest.mark.parametrize("latent", TIE_LATENTS)
def test_observation_ties_change_H1_and_the_probabilities(latent):
    """Observations rounded toward zero instead of to nearest even change H1 in nearly every tie row and move a
    probability outside P_REL in more than 20 % of them: the GPU test on these rows sees a truncating stager."""
    net, x = tie_rows(latent, 300)
    H1, _, p = machine(x, net)
    H1_rz, _, p_rz = machine(bf16_rz(x), net)
    assert (H1_rz != H1).any(1).mean() > 0.9
    assert (np.abs(p_rz - p) > P_REL * p).any(1).mean() > 0.2


# ---------------------------------------------------------------- GPU fixtures and helpers

@pytest.fixture(scope="module")
def small(evg, cfg):
    """45 mid-game matches: 90 rows, one partial tile."""
    return mid_game(evg, cfg, 45)


def call(fused):
    """One kernel call: (actions, idx [rows, 7], probs [rows, out], logp [rows, 7]) as numpy."""
    acts = fused(want_probs=True, want_logp=True).cpu().numpy()
    return (acts, fused.idx.cpu().numpy().reshape(-1, 7), fused.probs.cpu().numpy().reshape(-1, fused.out_dim),
            fused.logp.cpu().numpy().reshape(-1, 7))


def check_exact(net, obs, idx, probs, logp, block=8192):
    """Every probability within P_REL of the machine's and every ratio to its row's largest within R_REL, rows summing
    to 1, every logp within LOGP_ABS of the float64 truth of the kernel's own draws."""
    for r0 in range(0, len(obs), block):
        s = slice(r0, r0 + block)
        want = machine(obs[s], net)[2]
        assert (np.abs(probs[s] - want) <= P_REL * want).all(), (r0, np.abs(probs[s] / want - 1).max())
        assert ratio_error(probs[s], want) <= R_REL, (r0, ratio_error(probs[s], want))
        assert np.abs(probs[s].sum(-1) - 1).max() <= 1e-5
        err = np.abs(logp[s].astype(np.float64) - true_logp(want, idx[s]))
        assert err.max() <= LOGP_ABS, (r0, err.max())


def check_draws(env, acts, idx, probs, player=-1, div=12, mod=11, tiles=None):
    """The draws of every row (or the rows of `tiles`) are ppo_sample_rows of the kernel's probabilities with the tape's
    uniforms, and the action rows their unravel."""
    from oracle import policy_decode
    rows, draws = expected_draws(env, probs, player, tiles)
    assert np.array_equal(idx[rows], draws)
    played = acts.reshape(-1, 7, 2) if player < 0 else acts[:, player]
    assert np.array_equal(played, policy_decode.ppo_unravel(idx, div, mod).astype(np.int8))


# ---------------------------------------------------------------- the exact network on the GPU

@gpu
@pytest.mark.parametrize("latent", LATENTS)
def test_exact_at_every_width(small, latent):
    net = ExactPPO(np.random.default_rng(latent), 105, latent)
    acts, idx, probs, logp = call(policy.FusedPPO(small, weights=net.weights))
    check_exact(net, obs_rows(small), idx, probs, logp)
    check_draws(small, acts, idx, probs)


@gpu
@pytest.mark.parametrize("latent", [64, 128, 129, 256])
def test_exact_multi_tile(big, sms, latent):
    """Both players' rows make CTAs handle 4 or 5 tiles, the last one partial: every row against the machine, the draws
    of the tiles checked_tiles picks.  One player's rows (2 or 3 tiles per CTA, other tile edges) give that player's
    column of the two-player call bit for bit, and leave the other side's action rows."""
    net = ExactPPO(np.random.default_rng(latent), 105, latent)
    acts, idx, probs, logp = call(policy.FusedPPO(big, weights=net.weights))
    check_exact(net, obs_rows(big), idx, probs, logp)
    check_draws(big, acts, idx, probs, tiles=checked_tiles(len(idx), sms))
    for p in (0, 1):
        big._actions.fill_(-7)
        a1, i1, p1, l1 = call(policy.FusedPPO(big, weights=net.weights, player=p))
        assert np.array_equal(p1, probs[p::2]) and np.array_equal(i1, idx[p::2]) and np.array_equal(l1, logp[p::2]), p
        assert np.array_equal(a1[:, p], acts[:, p]) and (a1[:, 1 - p] == -7).all(), p
        check_draws(big, a1, i1, p1, player=p, tiles=checked_tiles(len(i1), sms))


@gpu
@pytest.mark.parametrize("out_dim,div,mod", OUT_CASES)
@pytest.mark.parametrize("latent", [16, 193])
def test_output_widths(small, latent, out_dim, div, mod):
    net = ExactPPO(np.random.default_rng(out_dim + latent), 105, latent, out_dim)
    acts, idx, probs, logp = call(policy.FusedPPO(small, weights=net.weights, div=div, mod=mod))
    check_exact(net, obs_rows(small), idx, probs, logp)
    check_draws(small, acts, idx, probs, div=div, mod=mod)


@gpu
@pytest.mark.parametrize("latent", TIE_LATENTS)
def test_observation_ties_reach_the_analog_units(evg, cfg, latent):
    """tie_rows written into env.obs: the tile stager must round them to nearest even, or H1 and the probabilities
    change (test_observation_ties_change_H1_and_the_probabilities)."""
    import torch
    env = mid_game(evg, cfg, 150, turns=3)
    net, x = tie_rows(latent, 300)
    env.obs.copy_(torch.from_numpy(x).view(env.obs.shape))
    acts, idx, probs, logp = call(policy.FusedPPO(env, weights=net.weights))
    check_exact(net, x, idx, probs, logp)
    check_draws(env, acts, idx, probs)


@gpu
@pytest.mark.parametrize("nodes", [7, 16])
def test_other_observation_widths(evg, tmp_path, nodes):
    """7 nodes: 89 values per row; 16 nodes: 125, the widest map the 128 input columns hold."""
    from test_gpu_generic import write_configs
    if nodes == 7:
        cfg = evg.load_config(write_configs(tmp_path, 100), "Map7.json", "Units4.json", "Setup.json")
    else:
        cfg = evg.load_config(write_ring16(tmp_path), "Ring16.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")
    env = mid_game(evg, cfg, 300)
    width = 1 + 4 * nodes + 60
    assert env.obs_len == width
    net = ExactPPO(np.random.default_rng(nodes), width, 129)
    acts, idx, probs, logp = call(policy.FusedPPO(env, weights=net.weights))
    check_exact(net, obs_rows(env), idx, probs, logp)
    check_draws(env, acts, idx, probs)
