"""The fused recurrent PPO actor (evg_policy_rppo) on a network whose every gate and state has one exact value, at every
tiling edge and across carried turns.

The exact network.  The kernel's own arithmetic is exact when every product and sum is exact in its format and every
pre-activation of a saturating function sits at least 20 from 0, so that tanh and the sigmoid land on their limits
(1 + expf(-20) rounds to 1 in float32, tanhf(20) is 1).  ExactNet builds such a network:
- Head: W1, W2 in 40 {-1, 0, 1}, b1, b2 = +-20.  Observations are integers (bf16 rounding keeps them integers), so each
  head pre-activation is an odd multiple of 20 and x = +-1, exactly in bf16 even if tanhf stops an ulp short of 1.
- Carry units (a third of them): their z row is 0 in W_iz and W_hz with b_iz + b_hz = +20, so z = 1 exactly and
  h' = 0 n + 1 h = h bit for bit, contracted into an FMA or not.  Their columns of W_hh are 0: they feed no gate.  Their
  h is any float32 with 2^-4 <= |h| <= 1 that bf16 does not hold exactly (ties included), so H = bf16(h) has a right
  and a wrong rounding.
- Boolean units: h in {-1, 0, 1}.  W_i, and W_h on their columns, in 40 {-1, 0, 1}; b_ir + b_hr and b_iz + b_hz = +-20,
  b_in = +-20, b_hn in 40 {-1, 0, 1}.  Every r / z pre-activation is an odd multiple of 20, so r and z are 1 or below
  2.1e-9 (0 when expf overflows).  With a = W_in x + b_in (an odd multiple of 20) and c = W_hn H + b_hn (a multiple of
  40), n = sign(a + c) when r = 1 and tanh(a + r c) = sign(a) when r is tiny (|r c| < 3e-5).  h' = (1 - z) n + z h is
  then h when z = 1 and exactly n when z is tiny (1 - z rounds to 1, z h is below half an ulp of 1).
- Output layer: W3 in eighths on the boolean units and one weight in {+-1/2, +-1} on one carry unit per output, b3 in
  eighths.  Every term of D3 + b3 is a multiple of 2^-12 and every partial sum below 2^12, so the argument of tanh is
  exact in float32 in any order; only tanhf, expf, the sum and the division round.
machine() is that network as integer sign logic in numpy: the exact state, bit for bit, and float64 probabilities.

The probability bound, from documented error bounds with u = 2^-24 (no fast-math: the kernel is built without it):
- y = tanhf(t) is within 2 ulp of tanh(t) (CUDA Programming Guide, single-precision maximum ulp errors), relative error
  2^-22 at most, so |y - tanh t| <= 2^-22 and exp(y) is within a factor exp(2^-22) of exp(tanh t);
- expf is within 2 ulp as well: each e_j is within eps_e = (1 + 2^-22) exp(2^-22) - 1 (about 2^-21) of its exact value;
- S, the float32 sum of at most 144 positive terms in any order (the kernel adds four partial sums in a fixed order), is
  within gamma = 143 u / (1 - 143 u) of the sum of the e_j it adds, so within (1 + eps_e)(1 + gamma) of the exact sum;
- p_j = e_j / S is correctly rounded (IEEE division): relative error u.
So p_j / p_j(exact) lies within (1 + eps_e)(1 + u) / ((1 - eps_e)(1 - gamma)) - 1 = P_REL, about 160 u = 9.6e-6, 500
times tighter than the 5e-3 of tests/test_gpu_policy_rppo.py.  The state is compared bit for bit, the draws bit for bit
with tests/ppo_sampling.py's sampler on the kernel's own probabilities.  Float networks, where the rounding of bf16
operands is not exact, are held to that module's 5e-3 against evgsim.policy.reference_forward_rppo.

The CPU tests at the top check the construction: its margins, that the float32 reference agrees with the machine, and
that each plausible defect of the kernel moves the state or leaves the bound."""
import ctypes as C

import numpy as np
import pytest

from evgsim import policy
from test_gpu_policy_tiling import bf16_rz, checked_tiles, linear, mid_game, write_ring16

gpu = pytest.mark.gpu
LATENTS = [1, 15, 16, 17, 63, 64, 65, 127, 128, 129, 160, 192, 248, 255, 256]
OUT_CASES = [(7, 2, 3), (16, 4, 4), (17, 5, 3), (131, 11, 12), (144, 12, 12)]
U = 2.0 ** -24
EPS_E = (1 + 2.0 ** -22) * np.exp(2.0 ** -22) - 1
GAMMA = 143 * U / (1 - 143 * U)
P_REL = (1 + EPS_E) * (1 + U) / ((1 - EPS_E) * (1 - GAMMA)) - 1
F_REL, F_ABS = 5e-3, 5e-3  # float networks: tests/test_gpu_policy_rppo.py's bars
MUTANTS = ["h_bf16", "H_rz", "bhn_outside_r", "r_z_swapped", "H_stale", "H_early"]


# ---------------------------------------------------------------- the exact network and its machine (checked on the CPU)

class ExactNet:
    """Weights (float32, rppo_weights' order) of the saturating network of the module docstring, and its carry units."""

    def __init__(self, rng, in_dim, latent, out_dim=132):
        L = latent
        tern = lambda *shape: 40.0 * rng.integers(-1, 2, shape)  # noqa: E731
        pm20 = lambda *shape: 20.0 * rng.choice([-1, 1], shape)  # noqa: E731
        self.carry = np.zeros(L, dtype=bool)
        self.carry[rng.choice(L, L // 3, replace=False)] = True
        c = np.flatnonzero(self.carry)
        w_ih, w_hh, b_hh = tern(3 * L, L), tern(3 * L, L), tern(3 * L)
        w_hh[:, c] = 0
        b_ih = np.concatenate([pm20(2 * L) - b_hh[:2 * L], pm20(L)])  # b_ir + b_hr, b_iz + b_hz = +-20; b_in = +-20
        w_ih[L + c] = w_hh[L + c] = 0
        b_ih[L + c] = 20 - b_hh[L + c]
        n_bool = L - len(c)
        w3 = rng.choice([-1.0, 1.0], (out_dim, L)) * (rng.random((out_dim, L)) < min(1.0, 36 / n_bool)) / 8
        w3[:, c] = 0
        if len(c):
            w3[np.arange(out_dim), rng.choice(c, out_dim)] = rng.choice([-1, -0.5, 0.5, 1], out_dim)
        self.weights = [np.asarray(a, dtype=np.float32) for a in (
            tern(L, in_dim), pm20(L), tern(L, L), pm20(L), w_ih, b_ih, w_hh, b_hh, w3, rng.integers(-8, 9, out_dim) / 8)]

    def h0(self, rng, rows):
        """A state of the kind the network keeps exact: boolean units in {-1, 0, 1}; carry units +-[2^-4, 1), never
        bf16-exact, an eighth of them bf16 ties (low half 0x8000)."""
        h = rng.integers(-1, 2, (rows, len(self.carry))).astype(np.float32)
        k = int(self.carry.sum())
        bits = rng.uniform(2.0 ** -4, 1, (rows, k)).astype(np.float32).view(np.uint32) | np.uint32(1)
        tie = rng.random((rows, k)) < 1 / 8
        bits[tie] = (bits[tie] & np.uint32(0xFFFF0000)) | np.uint32(0x8000)
        h[:, self.carry] = bits.view(np.float32) * rng.choice(np.float32([-1, 1]), (rows, k))
        return h

    def actor(self):
        """A torch module with the reference ActorCritic's action_head, action_gru and action_layer holding the weights."""
        return actor_of(self.weights)


def actor_of(weights):
    import torch
    w1, w3 = weights[0], weights[8]
    latent = w1.shape[0]
    m = torch.nn.Module()
    m.action_head = torch.nn.Sequential(torch.nn.Linear(w1.shape[1], latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
    m.action_gru = torch.nn.GRU(latent, latent)
    m.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, w3.shape[0]), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
    with torch.no_grad():
        for p, w in zip(policy._rppo_params(m), weights):
            p.copy_(torch.from_numpy(np.asarray(w, dtype=np.float32)))
    return m


def machine(obs, h0, net, mutant=None):
    """The exact network's 7 steps: (probs float64 [rows, 7, out], h float32 [rows, L]).  Asserts what makes the kernel
    exact: integer observations with head sums below 2^24, every margin at least 20, carry states 0 or in [2^-4, 1].
    Every sum of integers below 2^24, and of multiples of 2^-12 below 2^12, is exact in float32 BLAS.  `mutant` runs a
    defect instead: h carried in bf16, H rounded toward zero, b_hn added outside r *, r and z swapped, the gates reading
    the previous step's H, or (L > 128) the second pass reading the H the first pass has just updated."""
    f32 = np.float32
    w1, b1, w2, b2, w_ih, b_ih, w_hh, b_hh, w3, b3 = net.weights
    L = w1.shape[0]
    B = np.flatnonzero(~net.carry)
    nb = len(B)
    g = np.concatenate([B, L + B, 2 * L + B])
    x0 = policy.bf16_round(np.asarray(obs, dtype=f32))
    assert np.array_equal(x0, np.round(x0)) and 40 * np.abs(x0).sum(1).max() + 20 < 2 ** 24
    z1 = x0 @ w1.T + b1
    z2 = np.sign(z1) @ w2.T + b2
    assert np.abs(z1).min() >= 20 and np.abs(z2).min() >= 20
    gi = np.sign(z2) @ w_ih[g].T
    b_rz = (b_ih + b_hh)[g[:2 * nb]]
    b_in, b_hn = b_ih[2 * L + B], b_hh[2 * L + B]
    whh = w_hh[np.ix_(g, B)]
    rnd = bf16_rz if mutant == "H_rz" else policy.bf16_round
    h = np.array(h0, dtype=f32)
    hc = np.abs(h[:, net.carry])
    assert ((hc == 0) | ((hc >= 2.0 ** -4) & (hc <= 1))).all()

    def update(Hb, hb):
        gh = Hb @ whh.T
        pre = gi[:, :2 * nb] + gh[:, :2 * nb] + b_rz
        a, c = gi[:, 2 * nb:] + b_in, gh[:, 2 * nb:] + b_hn
        assert min(np.abs(pre).min(), np.abs(a).min(), np.abs(a + c).min()) >= 20
        r, z = pre[:, :nb] > 0, pre[:, nb:] > 0
        if mutant == "r_z_swapped":
            r, z = z, r
        n = np.sign(np.where(r, a + c, a + b_hn if mutant == "bhn_outside_r" else a))
        return np.where(z, hb, n).astype(f32)

    def bf16_h(h):  # H = bf16(h): the boolean units are exact already
        H = h.copy()
        H[:, net.carry] = rnd(h[:, net.carry])
        return H

    probs = []
    H_prev = H = bf16_h(h)
    for _ in range(7):
        hb = update((H_prev if mutant == "H_stale" else H)[:, B], h[:, B])
        if mutant == "H_early" and L > 128:
            first = B < 128
            H_mixed = H.copy()
            H_mixed[:, B[first]] = hb[:, first]
            hb = np.where(first, hb, update(H_mixed[:, B], h[:, B]))
        h = h.copy()
        h[:, B] = hb
        if mutant == "h_bf16":
            h = policy.bf16_round(h)
        H_prev, H = H, bf16_h(h)
        e = np.exp(np.tanh((H @ w3.T + b3).astype(np.float64)))
        probs.append(e / e.sum(-1, keepdims=True))
    return np.stack(probs, axis=1), h


def synthetic_obs(rng, rows, in_dim):
    """Integer rows in the observations' range, a few above 256 (rounded to even integers by bf16)."""
    x = rng.integers(-100, 151, (rows, in_dim)).astype(np.float32)
    x[:, 0] = rng.integers(0, 600, rows)
    return x


@pytest.mark.parametrize("latent", [1, 17, 128, 129, 200, 256])
def test_machine_is_the_float32_reference_and_sees_every_defect(latent):
    """The float32 numpy statement of the kernel (reference_forward_rppo) gives the machine's state bit for bit and its
    probabilities within P_REL; the boolean units really move; each defect moves the state or leaves the bound."""
    rng = np.random.default_rng(latent)
    rows = 600
    net = ExactNet(rng, 105, latent)
    x, h0 = synthetic_obs(rng, rows, 105), net.h0(rng, rows)
    p, h = machine(x, h0, net)
    with np.errstate(over="ignore"):  # the sigmoid's exp overflows to inf by design: 1 / (1 + inf) = 0
        ref_p, ref_h = policy.reference_forward_rppo(x, h0, net.weights)
    assert np.array_equal(ref_h, h) and np.array_equal(h[:, net.carry], h0[:, net.carry])
    assert (np.abs(ref_p - p) <= P_REL * p).all(), np.abs(ref_p / p - 1).max()
    assert 4e-6 < P_REL < 1.1e-5
    if latent == 1:
        return
    assert (h[:, ~net.carry] != h0[:, ~net.carry]).mean() > 0.25
    for mutant in MUTANTS:
        if mutant == "H_early" and latent <= 128:
            continue
        mp, mh = machine(x, h0, net, mutant)
        caught = (mh != h).any(1) | (np.abs(mp - p) > P_REL * p).any((1, 2))
        assert caught.mean() > 0.2, (mutant, caught.mean())


def test_the_margins_are_checked():
    """machine() refuses what would not be exact: a fractional observation, a carry state below 2^-4, a bias that
    leaves a gate pre-activation at 0."""
    rng = np.random.default_rng(0)
    net = ExactNet(rng, 105, 40)
    x, h0 = synthetic_obs(rng, 10, 105), net.h0(rng, 10)
    machine(x, h0, net)
    with pytest.raises(AssertionError):
        machine(x + 0.5, h0, net)
    h1 = h0.copy()
    h1[0, np.flatnonzero(net.carry)[0]] = 2.0 ** -6
    with pytest.raises(AssertionError):
        machine(x, h1, net)
    net.weights[5] = net.weights[5] + 20  # b_ir + b_hr in {0, 40}: some r pre-activation at 0
    with pytest.raises(AssertionError):
        machine(x, h0, net)


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


@pytest.fixture(scope="module")
def small(evg, cfg):
    """45 mid-game matches: 90 rows, one partial tile."""
    return mid_game(evg, cfg, 45)


@pytest.fixture(scope="module")
def big(evg, cfg, sms):
    """Matches whose per-player rows make ~2.5 tiles per CTA, the last one partial; both players' rows ~5."""
    return mid_game(evg, cfg, ((5 * sms + 1) // 2 - 1) * 128 + 54)


def float_net(rng, in_dim, latent, out_dim=132):
    """torch's default initialisation of the head, the GRU (uniform in +-1/sqrt(L)) and the output layer."""
    s = 1 / np.sqrt(latent)
    gru = [rng.uniform(-s, s, shape).astype(np.float32) for shape in ((3 * latent, latent), 3 * latent) * 2]
    return linear(rng, latent, in_dim) + linear(rng, latent, latent) + gru + linear(rng, out_dim, latent)


def obs_rows(env, player=-1):
    obs = env.obs.cpu().numpy()
    return obs.reshape(-1, env.obs_len) if player < 0 else obs[:, player]


def call(fused, h0=None):
    """One kernel call (from state h0 if given): (records before it, actions, idx [rows, 7], probs [rows, 7, out],
    hidden [rows, L]) as numpy."""
    import torch
    if h0 is not None:
        fused.hidden.copy_(torch.from_numpy(np.ascontiguousarray(h0, dtype=np.float32)).view(fused.hidden.shape))
    st = fused.env.get_state()
    acts = fused(want_probs=True).cpu().numpy()
    return (st, acts, fused.idx.cpu().numpy().reshape(-1, 7), fused.probs.cpu().numpy().reshape(-1, 7, fused.out_dim),
            fused.hidden.cpu().numpy().reshape(-1, fused.latent))


def check_exact(net, obs, h0, probs, h, block=8192):
    """The state bit for bit and every probability within P_REL of the machine's, every row."""
    for r0 in range(0, len(obs), block):
        s = slice(r0, r0 + block)
        want, want_h = machine(obs[s], h0[s], net)
        assert np.array_equal(h[s], want_h), (r0, np.argwhere(h[s] != want_h)[:5])
        assert (np.abs(probs[s] - want) <= P_REL * want).all(), (r0, np.abs(probs[s] / want - 1).max())
        assert np.abs(probs[s].sum(-1) - 1).max() <= 1e-5


def check_float(weights, obs, h0, probs, h):
    want, want_h = policy.reference_forward_rppo(obs, h0, weights)
    assert np.isfinite(probs).all() and np.isfinite(h).all()
    assert (np.abs(probs - want) <= F_REL * want).all(), np.abs(probs / want - 1).max()
    assert np.abs(h - want_h).max() <= F_ABS, np.abs(h - want_h).max()


def check_draws(env, st, acts, idx, probs, div=12, mod=11, rows=None):
    """Every draw of the two-player rows `rows` (default all) is ppo_sample of the kernel's distribution with the tape's
    uniform of the records `st` the call read, and every action row its unravel."""
    import ppo_sampling as ps
    from oracle import policy_decode
    rows = np.arange(len(idx)) if rows is None else np.asarray(rows)
    u = np.stack([ps.policy_uniforms(env.seed, env.env_id_offset + r // 2, int(st[r // 2]["turn"]), r % 2, int(st[r // 2]["episode"]))
                  for r in rows])
    for k in range(7):
        assert np.array_equal(idx[rows, k], ps.ppo_sample_rows(probs[rows, k], u[:, k:k + 1])[:, 0]), k
    assert np.array_equal(acts.reshape(-1, 7, 2)[rows], policy_decode.ppo_unravel(idx[rows], div, mod).astype(np.int8))


# ---------------------------------------------------------------- the exact network on the GPU

@gpu
@pytest.mark.parametrize("latent", LATENTS)
def test_exact_state_at_every_width(small, latent):
    rng = np.random.default_rng(latent)
    net = ExactNet(rng, 105, latent)
    h0 = net.h0(rng, 90)
    st, acts, idx, probs, h = call(policy.FusedRPPO(small, net.actor()), h0)
    check_exact(net, obs_rows(small), h0, probs, h)
    check_draws(small, st, acts, idx, probs)


@gpu
@pytest.mark.parametrize("latent", [64, 128, 129, 256])
def test_exact_state_multi_tile(big, sms, latent):
    """Both players' rows make CTAs handle 4 or 5 tiles, the last one partial: the state and probabilities of every
    row against the machine, the draws of the tiles checked_tiles picks.  One player's rows (2 or 3 tiles per CTA, other
    tile edges) give that player's rows of the two-player call bit for bit, and leave the other side's action rows."""
    rng = np.random.default_rng(latent)
    net = ExactNet(rng, 105, latent)
    actor = net.actor()
    h0 = net.h0(rng, 2 * big.num_envs)
    st, acts, idx, probs, h = call(policy.FusedRPPO(big, actor), h0)
    check_exact(net, obs_rows(big), h0, probs, h)
    rows = 2 * big.num_envs
    check_draws(big, st, acts, idx, probs, rows=np.concatenate([np.arange(128 * t, min(128 * t + 128, rows)) for t in checked_tiles(rows, sms)]))
    for p in (0, 1):
        big._actions.fill_(-7)
        _, a1, i1, p1, h1 = call(policy.FusedRPPO(big, actor, player=p), h0.reshape(-1, 2, latent)[:, p])
        assert np.array_equal(h1, h[p::2]) and np.array_equal(p1, probs[p::2]) and np.array_equal(i1, idx[p::2]), p
        assert np.array_equal(a1[:, p], acts[:, p]) and (a1[:, 1 - p] == -7).all(), p


@gpu
@pytest.mark.parametrize("latent", [17, 128, 129, 256])
def test_turn_zero_rows_start_from_zero(evg, cfg, latent):
    """Freshly reset matches ignore what .hidden holds (garbage, NaN) and write back the state of a zero start, units
    128.. (kept in .hidden itself) included; after a masked reset mid-game exactly the restarted matches' rows do."""
    n = 300
    rng = np.random.default_rng(latent)
    net = ExactNet(rng, 105, latent)
    env = evg.BatchedEvergladesEnv(n, seed=9, config=cfg)
    env.reset()
    fused = policy.FusedRPPO(env, net.actor())
    garbage = rng.uniform(-50, 50, (2 * n, latent)).astype(np.float32)
    garbage[::7] = np.nan
    st, acts, idx, probs, h = call(fused, garbage)
    assert (st["turn"] == 0).all()
    check_exact(net, obs_rows(env), np.zeros_like(garbage), probs, h)
    check_draws(env, st, acts, idx, probs)
    for _ in range(10):
        env.step(env.random_actions())
    env.reset(mask=(np.arange(n) % 3 == 0).astype(np.uint8))
    h0 = net.h0(rng, 2 * n)
    st, acts, idx, probs, h = call(fused, h0)
    fresh = np.repeat(st["turn"] == 0, 2)
    assert 0 < fresh.sum() < 2 * n
    check_exact(net, obs_rows(env), np.where(fresh[:, None], 0, h0).astype(np.float32), probs, h)
    check_draws(env, st, acts, idx, probs)


@gpu
@pytest.mark.parametrize("mode", ["off", "terminal", "next"])
@pytest.mark.parametrize("latent", [64, 129, 256])
def test_carried_turns_follow_the_machine(evg, cfg, latent, mode):
    """30 turns of kernel call then env.step, the state carried by the kernel and, independently, by the machine (zero
    where the records read turn 0 before the call), compared after every turn.  A 12-turn limit ends every match
    twice: TERMINAL and NEXT restart them, OFF keeps stepping the finished matches, whose state keeps evolving."""
    import torch
    from evgsim import _capi
    auto = {"off": _capi.AUTORESET_OFF, "terminal": _capi.AUTORESET_TERMINAL, "next": _capi.AUTORESET_NEXT}[mode]
    n = 150
    saved = cfg.turn_limit, cfg.auto_reset
    cfg.turn_limit = 12
    try:
        env = evg.BatchedEvergladesEnv(n, seed=31, config=cfg, auto_reset=auto)
    finally:
        cfg.turn_limit, cfg.auto_reset = saved
    env.reset()
    for _ in range(5):
        env.step(env.random_actions())
    rng = np.random.default_rng(latent)
    net = ExactNet(rng, 105, latent)
    fused = policy.FusedRPPO(env, net.actor())
    state = net.h0(rng, 2 * n)
    fused.hidden.copy_(torch.from_numpy(state).view(fused.hidden.shape))
    restarts = finished = 0
    for t in range(30):
        st, acts, idx, probs, h = call(fused)
        fresh = np.repeat(st["turn"] == 0, 2)
        restarts += fresh.sum()
        want, state = machine(obs_rows(env), np.where(fresh[:, None], 0, state).astype(np.float32), net)
        assert np.array_equal(h, state), (t, np.argwhere(h != state)[:5])
        assert (np.abs(probs - want) <= P_REL * want).all(), (t, np.abs(probs / want - 1).max())
        check_draws(env, st, acts, idx, probs)
        finished += int(env.step(env._actions)[2].sum())
    assert finished > 0
    if mode == "off":
        assert restarts == 0
        assert (np.abs(state[:, net.carry]) >= 2.0 ** -4).all()  # never zeroed: the carry units still hold h0
    else:
        assert 0 < restarts


@gpu
@pytest.mark.parametrize("out_dim,div,mod", OUT_CASES)
@pytest.mark.parametrize("latent", [16, 193])
def test_output_widths(small, latent, out_dim, div, mod):
    rng = np.random.default_rng(out_dim + latent)
    net = ExactNet(rng, 105, latent, out_dim)
    h0 = net.h0(rng, 90)
    st, acts, idx, probs, h = call(policy.FusedRPPO(small, net.actor(), div=div, mod=mod), h0)
    check_exact(net, obs_rows(small), h0, probs, h)
    check_draws(small, st, acts, idx, probs, div, mod)
    w = float_net(rng, 105, latent, out_dim)
    h0 = rng.uniform(-1, 1, (90, latent)).astype(np.float32)
    st, acts, idx, probs, h = call(policy.FusedRPPO(small, actor_of(w), div=div, mod=mod), h0)
    check_float(w, obs_rows(small), h0, probs, h)
    check_draws(small, st, acts, idx, probs, div, mod)


# ---------------------------------------------------------------- other observation widths

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
    rng = np.random.default_rng(nodes)
    net = ExactNet(rng, width, 129)
    h0 = net.h0(rng, 600)
    st, acts, idx, probs, h = call(policy.FusedRPPO(env, net.actor()), h0)
    check_exact(net, obs_rows(env), h0, probs, h)
    check_draws(env, st, acts, idx, probs)
    w = float_net(rng, width, 64)
    h0 = rng.uniform(-1, 1, (600, 64)).astype(np.float32)
    st, acts, idx, probs, h = call(policy.FusedRPPO(env, actor_of(w)), h0)
    check_float(w, obs_rows(env), h0, probs, h)
    check_draws(env, st, acts, idx, probs)


@gpu
def test_observations_wider_than_the_tiling_are_refused(evg, tmp_path):
    """32 nodes make 189-value rows.  FusedRPPO refuses a network of another width; the C API refuses the map itself
    (here with images packed for 105 inputs) and writes nothing."""
    import torch
    from evgsim import _capi
    from test_gpu_generic import write_ring32
    cfg = evg.load_config(write_ring32(tmp_path), "Ring32.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")
    env = evg.BatchedEvergladesEnv(64, seed=2, config=cfg)
    env.reset()
    assert env.obs_len == 189
    w = float_net(np.random.default_rng(0), 105, 128)
    with pytest.raises(ValueError, match="105 inputs"):
        policy.FusedRPPO(env, actor_of(w))
    dev = env.device
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    images = [torch.from_numpy(a).to(dev) for a in policy.pack_rppo(*w)[:6]]
    hidden = torch.full((64, 2, 128), 3.0, device=dev)
    idx = torch.zeros((64, 2, 7), dtype=torch.int64, device=dev)
    probs = torch.full((64, 2, 7, 132), 5.0, device=dev)
    env._actions.fill_(-7)
    assert env._lib.evg_policy_rppo(env._h, ptr(env.obs), -1, *map(ptr, images), 128, 132, 12, 11, ptr(hidden), ptr(env._actions),
                                    ptr(idx), ptr(probs), env._stream()) == -1  # EVG_E_ARG
    assert b"189" in _capi.load().evg_last_error()
    torch.cuda.synchronize()
    assert (hidden == 3).all() and not idx.any() and (probs == 5).all() and (env._actions == -7).all()


# ---------------------------------------------------------------- bitwise independence of the batch layout

@gpu
def test_shards_agree_bit_for_bit(evg, cfg, big):
    """The whole multi-tile batch against three uneven shards (env_id_offset) that put every row into another tile and
    CTA, a float network at L = 256: idx, probs, actions and the state, bit for bit."""
    import torch
    m = big.num_envs
    cuts = [0, m // 7 + 1, m // 2 + 37, m]
    shards = [mid_game(evg, cfg, b - a, offset=a) for a, b in zip(cuts, cuts[1:])]
    for s, a, b in zip(shards, cuts, cuts[1:]):
        assert torch.equal(s.obs, big.obs[a:b])
    rng = np.random.default_rng(5)
    actor = actor_of(float_net(rng, 105, 256))
    h0 = rng.uniform(-1, 1, (m, 2, 256)).astype(np.float32)
    whole = call(policy.FusedRPPO(big, actor), h0)[1:]
    parts = [call(policy.FusedRPPO(s, actor), h0[a:b])[1:] for s, a, b in zip(shards, cuts, cuts[1:])]
    for k, name in enumerate(("actions", "idx", "probs", "hidden")):
        assert np.array_equal(np.concatenate([p[k] for p in parts]), whole[k]), name
