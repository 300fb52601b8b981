"""The fused recurrent PPO actor (evg_policy_rppo) on GRU units whose gates are fractional: their float32 state within a
derived bound of float64 and the log-probabilities of its draws within a derived bound of the float64 truth, at every
width and tiling edge, across carried turns, and in the instantiation a PPO training loop runs (want_logp and
want_hidden_in, without probabilities).

The network.  AnalogNet is tests/test_gpu_policy_rppo_exact.py's ExactNet (boolean units with h in {-1, 0, 1}, carry
units whose h never changes, an output layer that reads only those) with about a third of its units, at least one from
L = 3 up and on both sides of unit 128 above L = 128 (units 128.. keep their state in d_hidden between passes), turned
analog:
- Gate inputs.  Each of an analog unit's r, z and n rows reads 2 to 4 columns of x (the head output, +-1) with +-1/8,
  one or two carry units' H with +-1/2 and up to two boolean units' H with +-1/8.  b_ih and b_hh lie on the 2^-12 grid
  within +-0.6, so every pre-activation lies within +-3: r, z and n are fractional.
- Exactness.  Carry H is bf16_rne of a float32 state in [2^-4, 1] (or 0) that the kernel keeps bit for bit, a multiple
  of 2^-11.  Every term of a gate pre-activation, of the kernel's pre-summed b_ir + b_hr and b_iz + b_hz, and of
  W_hn H + b_hn is then a multiple of 2^-12, and the sum of their magnitudes stays below 2^11: each is exact in float32
  in any summation order.  Only the gate functions, the product r c, the add in n's argument and h' round.
- Leaf units.  An analog unit's own H feeds nothing: its columns of W_hh and W3 are 0.  The boolean and carry units keep
  their bit-exact states and the probabilities ExactNet's P_REL; the analog units are seen through the float32 state the
  kernel writes back.
machine() steps this network in float64 (boolean and carry units as exact sign logic, as the exact module's machine
does), asserts its preconditions on the rows it is given, and bounds the kernel's float32 analog state element by element.

The state bound E, from documented error bounds, with u = 2^-24 (the kernel is built without fast-math):
- expf and tanhf are within 2 ulp (CUDA Programming Guide, single-precision maximum ulp errors): relative error at most
  F = 2^-22.  __frcp_rn, IEEE add and IEEE multiply are correctly rounded: relative error at most u.
- The sigmoid __frcp_rn(1 + expf(-v)) of an exact v: expf moves 1 + e^-v by at most F relative, the add and the
  reciprocal round once each, so it is within S = (1 + u) / ((1 - F)(1 - u)) - 1 (about 3.6e-7) relative of
  1 / (1 + e^-v): dr = S r, dz = S z.
- n = tanh(t), t = a + r c with a = W_in x + b_in and c = W_hn H + b_hn exact.  The product r~ c is within
  e1 = |r c| ((1 + S)(1 + u) - 1) of r c, and the add rounds once (or not at all when contracted into an FMA):
  |t~ - t| <= dt = e1 + u (|t| + e1).  tanh is 1-Lipschitz and tanhf adds F relative: |n~ - n| <= dn = dt + F (|n| + dt).
- h' = (1 - z) n + z h.  With n~ = n + d_n, z~ = z + d_z and h~ = h + d_h (the previous step's error),
  (1 - z~) n~ + z~ h~ - h' = (1 - z~) d_n + z~ d_h + d_z (h - n) exactly.  Evaluating it rounds at most four quantities
  of magnitude at most 2 in the kernel's form and in any algebraically equal one (an FMA contraction, n + z (h - n),
  h + (1 - z)(n - h)): RHO = 8 u more, so that a legitimate rewrite keeps the bound.  Hence, per step k,
      E_k = (1 - z + dz) dn + (z + dz) E_{k-1} + dz |h - n| + RHO,   E_0 = 0 (the kernel starts from the same float32 h),
  an earlier error propagating with factor z~ <= 1.  machine() evaluates E in float64, whose own rounding (~1e-16) is
  far below RHO.  With |t| <= 3 and |c| <= 1.85, a step adds at most dn + RHO = 1.8e-6 (z = 0) or 2 dz + RHO = 1.2e-6
  on top of E_{k-1} (z = 1), so E stays below 1e-5 after 7 steps; on the tests' rows it reaches 4.5e-6 (median 1.2e-6),
  and the float32 statement reference_forward_rppo stays within 0.16 E.
Each of these defects leaves E in more than 20 % of rows at L >= 17 (the CPU tests): r, z or n rounded to bf16, a
tanh.approx-sized error (2^-11 relative) on n, the sigmoid computed as 0.5 + 0.5 tanh.approx(v / 2), h' = z n + (1 - z) h,
b_hn added outside r *, the pre-summed r / z bias without b_hh, h kept in bf16 between steps.  An __expf-sized error (a
few ulp) is below what E resolves: this module does not claim to see it.

The log-probability bound.  Step k draws once, with replacement, from its own distribution; the kernel writes
logf(q_s / T_k), T_k its float32 ascending sum of all of step k's probabilities q_j.  The truth is log p*_k[s], which is
tests/test_gpu_policy_ppo_exact.py's log(p_s / R_k) with R_k = 1.  That module's derivation of LOGP_ABS holds for any
R_k, and every step here is the case of its first draw: the output layer is the feed-forward actor's (tanhf, expf, a
float32 sum of at most 144 terms, a correctly rounded division), so each q_j is within P_REL of p_j; T_k, the float32
sum of all q_j, is within (1 +- P_REL)(1 +- GAMMA) of 1 = R_k; the quotient rounds once; logf adds one ulp of a value
of magnitude at most 7 (p_j >= e^-2 / 144).  So LOGP_ABS (about 2.8e-5) carries over unchanged, and so do P_REL for the
probabilities and R_REL for their ratios to the row's largest.

The CPU tests at the top check the construction, the bound and its margin; the GPU tests hold the kernel to them."""
from collections import namedtuple
from types import SimpleNamespace

import numpy as np
import pytest

from evgsim import policy
from test_gpu_policy_logp import wire_env
from test_gpu_policy_ppo_exact import LOGP_ABS, R_REL, on_grid, ratio_error
from test_gpu_policy_rppo_exact import LATENTS, OUT_CASES, P_REL, U, ExactNet, check_draws, obs_rows, synthetic_obs
from test_gpu_policy_rppo_exact import machine as exact_machine
from test_gpu_policy_tiling import big, checked_tiles, evg, sms  # noqa: F401

gpu = pytest.mark.gpu
F = 2.0 ** -22                                # expf, tanhf: 2 ulp, relative
S = (1 + U) / ((1 - F) * (1 - U)) - 1         # the sigmoid's relative error
RHO = 8 * U                                   # the rounding of h' in any of its forms
GRID = 2.0 ** -12                             # the analog biases' grid
MUTANTS = ["r_bf16", "z_bf16", "n_bf16", "n_tanh_approx", "sigmoid_tanh_approx", "z_swapped", "bhn_outside_r",
           "b_rz_without_hh", "h_bf16"]


# ---------------------------------------------------------------- the network and its machine (checked on the CPU)

class AnalogNet(ExactNet):
    """ExactNet with analog units (the module docstring): .analog marks them; the weights are ExactNet's otherwise, with
    the analog units' columns of W_hh and W3 zeroed."""

    def __init__(self, rng, in_dim, latent, out_dim=132):
        L = latent
        super().__init__(rng, in_dim, L, out_dim)
        while L > 128 and self.carry[128:].all():  # L = 129 with unit 128 a carry unit: no analog unit could sit there
            super().__init__(rng, in_dim, L, out_dim)
        free = np.flatnonzero(~self.carry)
        k = max(1, L // 3) if self.carry.any() else 0  # the analog rows read carry units: ExactNet has none below L = 3
        chosen = [rng.choice(side) for side in ([free[free < 128], free[free >= 128]] if L > 128 else [free])][:k]
        chosen += list(rng.choice(np.setdiff1d(free, chosen), k - len(chosen), replace=False))
        self.analog = np.zeros(L, dtype=bool)
        self.analog[chosen] = True
        c, b = np.flatnonzero(self.carry), np.flatnonzero(~self.carry & ~self.analog)
        w_ih, b_ih, w_hh, b_hh, w3 = (a.copy() for a in self.weights[4:9])
        w_hh[:, self.analog] = 0
        w3[:, self.analog] = 0
        pm = lambda n: rng.choice([-1.0, 1.0], n)  # noqa: E731
        for row in np.flatnonzero(np.tile(self.analog, 3)):
            w_ih[row], w_hh[row] = 0, 0
            cols = rng.choice(L, min(L, rng.integers(2, 5)), replace=False)
            w_ih[row, cols] = pm(len(cols)) / 8
            cols = rng.choice(c, min(len(c), rng.integers(1, 3)), replace=False)
            w_hh[row, cols] = pm(len(cols)) / 2
            cols = rng.choice(b, min(len(b), rng.integers(0, 3)), replace=False)
            w_hh[row, cols] = pm(len(cols)) / 8
            b_ih[row], b_hh[row] = rng.integers(-2458, 2459, 2) * GRID  # within +-0.6
        self.weights[4:9] = [w_ih, b_ih, w_hh, b_hh, w3]

    def h0(self, rng, rows):
        """ExactNet's state, with the analog units anywhere in [-1, 1]."""
        h = super().h0(rng, rows)
        h[:, self.analog] = rng.uniform(-1, 1, (rows, self.analog.sum())).astype(np.float32)
        return h


Truth = namedtuple("Truth", "probs h E steps bounds gates")


def bf16(v):
    return policy.bf16_round(np.asarray(v, dtype=np.float32)).astype(np.float64)


def machine(obs, h0, net, mutant=None):
    """The network's 7 steps from state h0 (float32 [rows, L]) as a Truth: probs float64 [rows, 7, out]; the final state
    h float64 [rows, L] (the kernel's float32 bit for bit outside the analog units, float64 on them) and its bound E (0
    outside the analog units); the analog units' states `steps` and their bounds after each step (float64 [rows, 7,
    analog units]) and their gates r, z, n at each step ([3, rows, 7, analog units]).  Asserts what makes the kernel's
    sums exact and E a bound: integer observations, the head's and the boolean units' margins of 20, bf16-exact analog
    weights on their grids, analog biases on the 2^-12 grid, analog sums below 2^11, analog units feeding nothing,
    boolean states in {-1, 0, 1}, carry states 0 or in [2^-4, 1] and analog states in [-1, 1].  `mutant` runs one of
    MUTANTS on the analog units instead."""
    f64 = np.float64
    w1, b1, w2, b2, w_ih, b_ih, w_hh, b_hh, w3, b3 = (np.asarray(a, dtype=f64) for a in net.weights)
    L = w1.shape[0]
    A, C = net.analog, net.carry
    B = ~A & ~C
    ga = np.tile(A, 3)
    assert not w_hh[:, A].any() and not w3[:, A].any(), "an analog unit feeds a gate or an output"
    wa = np.concatenate([w_ih[ga], w_hh[ga]], axis=1)
    assert np.array_equal(bf16(wa), wa) and on_grid(wa, 1 / 8) and on_grid(w_hh[np.ix_(ga, C)], 0.5), "analog weights off their grid"
    assert on_grid(b_ih[ga], GRID) and on_grid(b_hh[ga], GRID), "analog biases off their grid"
    h = np.array(h0, dtype=np.float32).astype(f64)
    hc = np.abs(h[:, C])
    assert ((hc == 0) | ((hc >= 2.0 ** -4) & (hc <= 1))).all(), "carry state neither 0 nor in [2^-4, 1]"
    assert (np.abs(h[:, A]) <= 1).all(), "analog state outside [-1, 1]"
    assert np.isin(h[:, B], (-1, 0, 1)).all(), "boolean state outside {-1, 0, 1}"
    # |x| = 1 and |H| <= 1: every analog sum's terms add up to at most its weights' and biases' magnitudes
    assert (np.abs(w_ih[ga]).sum(1) + np.abs(w_hh[ga]).sum(1) + np.abs(b_ih[ga]) + np.abs(b_hh[ga])).max(initial=0) < 2 ** 11, \
        "analog sums too wide"
    x0 = bf16(obs)
    assert np.array_equal(x0, np.round(x0)) and 40 * np.abs(x0).sum(1).max() + 20 < 2 ** 24, "observations not integers"
    z1 = x0 @ w1.T + b1
    z2 = np.sign(z1) @ w2.T + b2
    assert min(np.abs(z1).min(), np.abs(z2).min()) >= 20, "head margin below 20"
    x = np.sign(z2)
    b_rz = b_ih[:2 * L] + b_hh[:2 * L]

    def gate_inputs(units, b_r, b_z):
        """(r and z pre-activations, a = W_in x + b_in, c = W_hn H + b_hn) of `units` as functions of H."""
        k = len(units)
        rows = np.concatenate([units, L + units, 2 * L + units])
        base = x @ w_ih[rows].T + np.concatenate([b_r, b_z, b_ih[2 * L + units]])
        w, b_hn = w_hh[rows], b_hh[2 * L + units]

        def at(H):
            gh = H @ w.T
            return base[:, :k] + gh[:, :k], base[:, k:2 * k] + gh[:, k:2 * k], base[:, 2 * k:], gh[:, 2 * k:] + b_hn
        return at

    iB, iA = np.flatnonzero(B), np.flatnonzero(A)
    boolean = gate_inputs(iB, b_rz[iB], b_rz[L + iB])
    if mutant == "b_rz_without_hh":
        analog = gate_inputs(iA, b_ih[iA], b_ih[L + iA])
    else:
        analog = gate_inputs(iA, b_rz[iA], b_rz[L + iA])
    b_hn = b_hh[2 * L + iA]
    flip = np.random.default_rng(1)  # the signs of the tanh.approx-sized errors

    def sig(v):
        if mutant == "sigmoid_tanh_approx":
            return 0.5 + 0.5 * np.tanh(v / 2) * (1 + 2.0 ** -11 * flip.choice([-1, 1], v.shape))
        return 1 / (1 + np.exp(-v))

    rows, na = len(h), len(iA)
    probs, gates = np.empty((rows, 7, len(b3))), np.empty((3, rows, 7, na))
    steps, bounds = np.empty((rows, 7, na)), np.empty((rows, 7, na))
    E = np.zeros((rows, na))
    H = h.copy()
    H[:, C] = bf16(h[:, C])  # the carry units' H never changes; the analog units keep h here, read by nothing
    for k in range(7):
        pr, pz, a, c = boolean(H)
        assert min(np.abs(v).min(initial=20) for v in (pr, pz, a, a + c)) >= 20, "boolean margin below 20"
        hb = np.where(pz > 0, H[:, iB], np.sign(np.where(pr > 0, a + c, a)))
        pr, pz, a, c = analog(H)
        r, z, ha = sig(pr), sig(pz), H[:, iA]
        if mutant == "r_bf16":
            r = bf16(r)
        if mutant == "z_bf16":
            z = bf16(z)
        t = a + (b_hn + r * (c - b_hn) if mutant == "bhn_outside_r" else r * c)
        n = np.tanh(t)
        if mutant == "n_bf16":
            n = bf16(n)
        if mutant == "n_tanh_approx":
            n = n * (1 + 2.0 ** -11 * flip.choice([-1, 1], n.shape))
        ha_next = z * n + (1 - z) * ha if mutant == "z_swapped" else (1 - z) * n + z * ha
        if mutant == "h_bf16":
            ha_next = bf16(ha_next)
        e1 = np.abs(r * c) * ((1 + S) * (1 + U) - 1)
        dt = e1 + U * (np.abs(t) + e1)
        dn = dt + F * (np.abs(n) + dt)
        dz = S * z
        E = (1 - z + dz) * dn + (z + dz) * E + dz * np.abs(ha - n) + RHO
        H[:, iB], H[:, iA] = hb, ha_next
        e = np.exp(np.tanh(H @ w3.T + b3))
        probs[:, k] = e / e.sum(-1, keepdims=True)
        steps[:, k], bounds[:, k], gates[:, :, k] = ha_next, E, (r, z, n)
    H[:, C] = h[:, C]
    E_all = np.zeros_like(h)
    E_all[:, A] = E
    return Truth(probs, H, E_all, steps, bounds, gates)


def true_logp(probs, idx):
    """float64 log p*_k[s_k] of each step's draw idx [rows, 7] from the exact probabilities [rows, 7, out]."""
    return np.log(np.take_along_axis(probs, np.asarray(idx, dtype=np.int64)[:, :, None], axis=2)[:, :, 0])


@pytest.mark.parametrize("latent", [1, 3, 17, 128, 129, 200, 256])
def test_machine_is_the_float32_reference_and_sees_every_defect(latent):
    """reference_forward_rppo (the kernel's arithmetic in float32 numpy) gives the non-analog state bit for bit, the
    analog state within E and the probabilities within P_REL and R_REL; its logp of sampled draws is within LOGP_ABS of
    the float64 truth; the machine's non-analog part is the exact module's machine; the gates are fractional; every
    defect leaves E in more than 20 % of rows."""
    import ppo_logp
    import ppo_sampling as ps
    rng = np.random.default_rng(latent)
    rows = 600
    net = AnalogNet(rng, 105, latent)
    A = net.analog
    assert A.sum() == (max(1, latent // 3) if latent >= 3 else 0)
    if latent > 128:
        assert A[:128].any() and A[128:].any()
    x, h0 = synthetic_obs(rng, rows, 105), net.h0(rng, rows)
    t = machine(x, h0, net)
    with np.errstate(over="ignore"):  # the boolean sigmoids' exp overflows to inf by design: 1 / (1 + inf) = 0
        ref_p, ref_h = policy.reference_forward_rppo(x, h0, net.weights)
    assert np.array_equal(ref_h[:, ~A], t.h[:, ~A])
    assert (np.abs(ref_h - t.h) <= t.E).all(), (np.abs(ref_h - t.h) - t.E).max()
    assert (np.abs(ref_p - t.probs) <= P_REL * t.probs).all() and ratio_error(ref_p.reshape(-1, 132), t.probs.reshape(-1, 132)) <= R_REL
    p_old, h_old = exact_machine(x, np.where(A, 0, h0).astype(np.float32), SimpleNamespace(weights=net.weights, carry=net.carry | A))
    assert np.array_equal(p_old, t.probs) and np.array_equal(h_old[:, ~A], t.h[:, ~A])
    u = rng.random((rows, 7)).astype(np.float32)
    idx = np.stack([ps.ppo_sample_rows(ref_p[:, k], u[:, k:k + 1])[:, 0] for k in range(7)], axis=1)
    assert np.abs(ppo_logp.rppo_logp_rows(ref_p, idx) - true_logp(t.probs, idx)).max() <= LOGP_ABS
    assert 3e-7 < S < 4e-7 and t.E.max() < 1e-5
    if latent < 3:
        return
    assert (np.abs(ref_h - t.h) <= 0.25 * t.E)[:, A].all()  # a correct float32 evaluation keeps a margin
    for g in (t.gates[0], t.gates[1], np.abs(t.gates[2])):
        assert ((0.02 < g) & (g < 0.98)).mean() > 0.5
    assert len(np.unique(t.steps[:, -1])) > 0.9 * t.steps[:, -1].size
    if latent < 17:
        return
    for mutant in MUTANTS:
        caught = (np.abs(machine(x, h0, net, mutant).h - t.h) > t.E)[:, A].any(1)
        assert caught.mean() > 0.2, (mutant, caught.mean())


def test_the_preconditions_are_checked():
    """machine() refuses what would make a sum inexact or E no bound: an analog bias off the 2^-12 grid, an analog
    weight too large for the sums, an analog unit read by W_hh or by W3, a carry state below 2^-4."""
    rng = np.random.default_rng(0)
    net = AnalogNet(rng, 105, 40)
    x, h0 = synthetic_obs(rng, 10, 105), net.h0(rng, 10)
    machine(x, h0, net)
    j = np.flatnonzero(net.analog)[0]
    for k, row, col, value, match in ((5, j, None, 2.0 ** -20, "grid"), (7, 80 + j, None, 2.0 ** -13, "grid"),
                                      (4, 40 + j, 0, 2.0 ** 11, "wide"), (6, np.flatnonzero(~net.analog & ~net.carry)[0], j, 40.0, "feeds"),
                                      (8, 3, j, 0.125, "feeds")):
        bad = SimpleNamespace(weights=[w.copy() for w in net.weights], carry=net.carry, analog=net.analog)
        if col is None:
            bad.weights[k][row] += value
        else:
            bad.weights[k][row, col] = value
        with pytest.raises(AssertionError, match=match):
            machine(x, h0, bad)
    h1 = h0.copy()
    h1[0, np.flatnonzero(net.carry)[0]] = 2.0 ** -6
    with pytest.raises(AssertionError, match="carry"):
        machine(x, h1, net)


# ---------------------------------------------------------------- GPU fixtures and helpers

@pytest.fixture(scope="module")
def small(evg, cfg):
    """45 mid-game matches (90 rows, one partial tile) stepped on wire rows, env.obs their expansion: the f32 and the
    wire call read the same observations."""
    return wire_env(evg, cfg, 45)


Out = namedtuple("Out", "st acts idx probs logp hidden_in hidden")


def call(fused, h0=None, obs_format="f32", want_probs=False, want_hidden_in=True):
    """One call with want_logp (from state h0 if given), every output asked for as numpy with rows flattened (None where
    not asked for), and the records it read.  The optional outputs are NaN before the call: each must be written."""
    import torch
    if h0 is not None:
        fused.hidden.copy_(torch.from_numpy(np.ascontiguousarray(h0, dtype=np.float32)).view(fused.hidden.shape))
    for t in (fused.probs, fused.logp, fused.hidden_in):
        t.fill_(float("nan"))
    st = fused.env.get_state()
    acts = fused(want_probs=want_probs, obs_format=obs_format, want_logp=True, want_hidden_in=want_hidden_in).cpu().numpy()
    L, out = fused.latent, fused.out_dim
    return Out(st, acts, fused.idx.cpu().numpy().reshape(-1, 7), fused.probs.cpu().numpy().reshape(-1, 7, out) if want_probs else None,
               fused.logp.cpu().numpy().reshape(-1, 7), fused.hidden_in.cpu().numpy().reshape(-1, L) if want_hidden_in else None,
               fused.hidden.cpu().numpy().reshape(-1, L))


def start_state(st, h0):
    """The state two-player rows start from: h0, +0.0 where the records read turn 0."""
    return np.where(np.repeat(st["turn"] == 0, 2)[:, None], np.float32(0), h0).astype(np.float32)


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def check(net, env, start, o, div=12, mod=11, rows=None, block=8192):
    """A two-player call o from state `start` against the machine: the analog state within E and every other unit bit
    for bit, logp within LOGP_ABS of the float64 truth of the kernel's draws, hidden_in = start bit for bit; with
    probabilities, each within P_REL and its ratio to the row's largest within R_REL, and the draws of `rows` (default
    all) ppo_sample_rows of them with the tape's uniforms, the action rows their unravel."""
    A = net.analog
    obs = obs_rows(env)
    if o.hidden_in is not None:
        assert same_bits(o.hidden_in, start)
    for r0 in range(0, len(obs), block):
        s = slice(r0, r0 + block)
        t = machine(obs[s], start[s], net)
        h = o.hidden[s]
        assert np.array_equal(h[:, ~A], t.h[:, ~A]), (r0, np.argwhere(h[:, ~A] != t.h[:, ~A])[:5])
        err = np.abs(h - t.h)
        assert (err <= t.E).all(), (r0, np.argwhere(err > t.E)[:5], (err / np.maximum(t.E, 1e-30))[:, A].max())
        err = np.abs(o.logp[s].astype(np.float64) - true_logp(t.probs, o.idx[s]))
        assert err.max() <= LOGP_ABS, (r0, err.max())
        if o.probs is not None:
            q = o.probs[s]
            assert (np.abs(q - t.probs) <= P_REL * t.probs).all(), (r0, np.abs(q / t.probs - 1).max())
            assert ratio_error(q.reshape(-1, q.shape[-1]), t.probs.reshape(-1, q.shape[-1])) <= R_REL
            assert np.abs(q.sum(-1) - 1).max() <= 1e-5
    if o.probs is not None:
        check_draws(env, o.st, o.acts, o.idx, o.probs, div, mod, rows)


# ---------------------------------------------------------------- the analog network on the GPU

@gpu
@pytest.mark.parametrize("fmt", ["f32", "wire"])
@pytest.mark.parametrize("latent", LATENTS)
def test_every_width(small, latent, fmt):
    """As a training loop calls it (want_logp, want_hidden_in, no probabilities) and with probabilities as well: the two
    calls agree bit for bit, and hold to the machine."""
    rng = np.random.default_rng(latent)
    net = AnalogNet(rng, 105, latent)
    h0 = net.h0(rng, 90)
    fused = policy.FusedRPPO(small, net.actor())
    train = call(fused, h0, fmt)
    full = call(fused, h0, fmt, want_probs=True)
    for k in ("acts", "idx", "logp", "hidden_in", "hidden"):
        assert same_bits(getattr(train, k), getattr(full, k)), k
    check(net, small, start_state(full.st, h0), full)


@gpu
@pytest.mark.parametrize("latent", [64, 128, 129, 256])
def test_multi_tile(big, sms, latent):
    """Both players' rows make CTAs handle 4 or 5 tiles, the last one partial: every row against the machine, the draws
    of the tiles checked_tiles picks.  Each player's own call equals its column of the two-player call bit for bit,
    logp and hidden_in included, and leaves the other side's action rows."""
    rng = np.random.default_rng(latent)
    net = AnalogNet(rng, 105, latent)
    actor = net.actor()
    h0 = net.h0(rng, 2 * big.num_envs)
    o = call(policy.FusedRPPO(big, actor), h0, want_probs=True)
    rows = 2 * big.num_envs
    check(net, big, start_state(o.st, h0), o,
          rows=np.concatenate([np.arange(128 * t, min(128 * t + 128, rows)) for t in checked_tiles(rows, sms)]))
    for p in (0, 1):
        big._actions.fill_(-7)
        o1 = call(policy.FusedRPPO(big, actor, player=p), h0.reshape(-1, 2, latent)[:, p], want_probs=True)
        for k in ("idx", "probs", "logp", "hidden_in", "hidden"):
            assert same_bits(getattr(o1, k), getattr(o, k)[p::2]), (p, k)
        assert np.array_equal(o1.acts[:, p], o.acts[:, p]) and (o1.acts[:, 1 - p] == -7).all(), p


@gpu
@pytest.mark.parametrize("latent", [17, 128, 129, 256])
def test_turn_zero_rows_start_from_zero(evg, cfg, latent):
    """Fresh matches ignore what .hidden holds (garbage, NaN): the analog units restart from +0.0 and hidden_in is +0.0;
    after a masked reset mid-game exactly the restarted matches' rows do."""
    n = 300
    rng = np.random.default_rng(latent)
    net = AnalogNet(rng, 105, latent)
    env = evg.BatchedEvergladesEnv(n, seed=9, config=cfg)
    env.reset()
    fused = policy.FusedRPPO(env, net.actor())
    garbage = rng.uniform(-50, 50, (2 * n, latent)).astype(np.float32)
    garbage[::7] = np.nan
    o = call(fused, garbage, want_probs=True)
    assert (o.st["turn"] == 0).all() and not o.hidden_in.view(np.uint32).any()
    check(net, env, np.zeros_like(garbage), o)
    for _ in range(10):
        env.step(env.random_actions())
    env.reset(mask=(np.arange(n) % 3 == 0).astype(np.uint8))
    h0 = net.h0(rng, 2 * n)
    o = call(fused, h0, want_probs=True)
    start = start_state(o.st, h0)
    assert 0 < (o.st["turn"] == 0).sum() < n
    check(net, env, start, o)


@gpu
@pytest.mark.parametrize("mode", ["off", "terminal", "next"])
@pytest.mark.parametrize("latent", [64, 129, 256])
def test_carried_turns(evg, cfg, latent, mode):
    """30 turns of kernel call then env.step under a 12-turn limit (test_gpu_policy_rppo_exact.py's
    test_carried_turns_follow_the_machine).  Each turn starts the machine from the kernel's own previous state (bit-exact
    outside the analog units), zero where the records read turn 0; hidden_in is that start bit for bit."""
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
    net = AnalogNet(rng, 105, latent)
    fused = policy.FusedRPPO(env, net.actor())
    state = net.h0(rng, 2 * n)
    fused.hidden.copy_(torch.from_numpy(state).view(fused.hidden.shape))
    restarts = finished = 0
    for _ in range(30):
        o = call(fused, want_probs=True)
        restarts += (o.st["turn"] == 0).sum()
        check(net, env, start_state(o.st, state), o)
        state = o.hidden
        finished += int(env.step(env._actions)[2].sum())
    assert finished > 0
    if mode == "off":
        assert restarts == 0
    else:
        assert 0 < restarts


@gpu
@pytest.mark.parametrize("out_dim,div,mod", [OUT_CASES[0], OUT_CASES[-1]])
@pytest.mark.parametrize("latent", [16, 193])
def test_output_widths(small, latent, out_dim, div, mod):
    rng = np.random.default_rng(out_dim + latent)
    net = AnalogNet(rng, 105, latent, out_dim)
    h0 = net.h0(rng, 90)
    o = call(policy.FusedRPPO(small, net.actor(), div=div, mod=mod), h0, want_probs=True)
    check(net, small, start_state(o.st, h0), o, div, mod)
