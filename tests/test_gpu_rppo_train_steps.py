"""The recurrent actor's update backward (evg_rppo_train_kernel<true>) step by step: every element of what it writes.

tests/test_gpu_rppo_train.py checks the backward through the reduced gradients only.  Here the kernel's own outputs are
compared element by element, from fused._train_forward and fused._train_backward called directly with an entry value G
of d_g the test writes itself:
1. Step bound: on random float networks every dgh_k, every g_{k-1} and S lie within rppo_train.backward_step_bound of
   float64, each step evaluated from the kernel's own inputs to it (its g_k, its h_{k-1}, its dgh_k as the carry's
   operand), at every width and out_dim, and at the row edges R = 1, 127, 128, 129 and ~2.5 tiles per CTA (last tile
   partial) at L = 17 .. 256: one and two row blocks, carry groups of 1 .. 4 atoms (4, 4, 1 at L = 129 .. 192 and
   4, 4, 4 at L > 192, where the piece table is full), several tiles per CTA.  Large batches are checked on the rows of
   the tiles checked_tiles picks (first and second tiles of the first and last CTAs, the partial last tile).
2. Bits: on DyadicNet, a GRU whose every float32 operation is exact or one IEEE rounding numpy repeats, d_h, d_g,
   d_dgh and S equal dyadic_machine's value for value (a zero's sign set aside) at every width and the same row edges.
3. Writes: outputs are the first R rows of longer buffers.  Every element below R is written finite (d_dgh and S
   start as NaN: the wrapper hands the kernel torch.empty buffers), every byte past R is left, g_7 = G_7 bit for bit.
4. Wiring: FusedRPPO.evaluate's gradients are float64 reductions of the kernel's own S and dgh within gamma_m bounds
   (torch's float32 matmul, TF32 off), so GRAD_TOL in tests/test_gpu_rppo_train.py only stands for the bf16 operands.
The CPU tests check the dyadic construction: its premises, that the machine is rppo_train.backward32 bit for bit, and
which of rppo_train.BACKWARD_MUTANTS move its bits."""
import numpy as np
import pytest

import rppo_train as rt
from test_gpu_policy_rppo_exact import LATENTS, actor_of
from test_gpu_policy_tiling import bf16_rz, checked_tiles, linear, mid_game
from test_gpu_rppo_train import WIDTHS, fused_params, grads, random_case

gpu = pytest.mark.gpu
F = np.float32
TAIL = 131             # rows past R in every output buffer
SENTINEL = 0x5AA5C33C  # their bit pattern (a finite float32), which no kernel write may change
R_EDGES = [1, 127, 128, 129, "big"]
STEP_LATENTS = [17, 64, 128, 129, 248, 256]
DYADIC_LATENTS = [64, 128, 129, 192, 256]
# the mutants the dyadic network cannot see: dgh_r is always 0 (r is 0 or 1) and n = 0, so c and 1 - n^2 never matter
DYADIC_BLIND = {"dar_without_c", "dtanh_1mn"}


# ---------------------------------------------------------------- the dyadic GRU (checked on the CPU)

class DyadicNet:
    """A GRU whose backward the kernel computes exactly or with roundings numpy float32 repeats (W_ih = 0, x unused).
    - Half units (every odd-indexed unit is constant, every even one half; L = 1 is one half unit): r fixed per unit,
      exactly 1 (b_ir = +40: 1 + expf(-40) rounds to 1) or exactly 0 (b_ir = -120: expf(120) overflows, 1 / inf = 0).
      Their z row and n row each read at most one constant unit, with a weight in {+-1/2, +-1/4}, and b_iz (b_hn)
      cancels that product of bf16(h_const) exactly, so u = sigmoid(0) = 1/2 and c = 0, n = tanh(+-0) = 0.  Then
      h_k = h_{k-1} / 2, dgh = [0, fl(g h_{k-1}) / 4, (g / 2) r], dgi = [0, fl(g h_{k-1}) / 4, g / 2] and the carry
      adds g_k / 2.
    - Constant units: b_ir = b_iz = +40, every weight 0, b_in = b_hn = 0: r = u = 1, n = 0, so h_k = h_{k-1} (one value
      per unit in every row, never bf16-exact: a wrong rounding of H moves the half units' u off 1/2) and dgh = 0; the
      carry adds g_k and bf16(dgh) of the one half-unit gate that reads the unit, times its weight.
    Every column of W_hh has at most one nonzero, so the carry's tensor-core sums are exact in any order, and every
    product the compiler could contract into an FMA is exact (u, 1 - u in {1/2, 1}, n = 0, r (1 - r) = 0).  Half units
    sit in every 64-column atom of gates z and n, constant units in every 16-column group on both sides of unit 128:
    every (gate, atom) of the staged dgh and every 16-column group of the carry's output carries a value.
    Left out, and covered by the step bound instead: dgh_r is always zero (so da_r's c and 1 - n^2 are never seen), and
    no carry sums more than one nonzero term."""

    def __init__(self, rng, in_dim, latent, out_dim=132):
        L = latent
        self.latent = L
        self.const = np.arange(L) % 2 == 1
        half, const = np.flatnonzero(~self.const), np.flatnonzero(self.const)
        self.r = np.ones(L, dtype=F)
        self.r[half] = rng.integers(0, 2, len(half))
        self.hc = (rng.uniform(0.5, 2, L).astype(F).view(np.uint32) | np.uint32(0x11)).view(F) * rng.choice(F([-1, 1]), L)
        self.hc[~self.const] = 0
        slots = rng.permutation(2 * len(half))[:len(const)]  # (half unit, gate z or n) slots, one per constant unit
        self.reads = (const, 1 + slots % 2, half[slots // 2], rng.choice(F([-0.5, -0.25, 0.25, 0.5]), len(const)))
        w_ih, w_hh = np.zeros((3 * L, L), F), np.zeros((3 * L, L), F)
        b_ih, b_hh = np.zeros(3 * L, F), np.zeros(3 * L, F)
        b_ih[:L] = np.where(self.r > 0, 40, -120)
        b_ih[L + const] = 40
        for j, gate, i, wt in zip(*self.reads):
            w_hh[gate * L + i, j] = wt
            cancel = -(rt.bf16(self.hc[j:j + 1])[0] * wt)
            if gate == 1:
                b_ih[L + i] = cancel
            else:
                b_hh[2 * L + i] = cancel
        self.weights = linear(rng, L, in_dim) + linear(rng, L, L) + [w_ih, b_ih, w_hh, b_hh] + linear(rng, out_dim, L)

    def h0(self, rng, rows):
        """Half units +-[1/4, 1) with full float32 mantissas, constant units their one value."""
        h = (rng.uniform(0.25, 1, (rows, self.latent)) * rng.choice([-1, 1], (rows, self.latent))).astype(F)
        h[:, self.const] = self.hc[self.const]
        return h

    def G(self, rng, rows):
        """An entry value of d_g: full float32 mantissas in +-[1/8, 4)."""
        return (rng.uniform(0.125, 4, (rows, rt.K, self.latent)) * rng.choice([-1, 1], (rows, rt.K, self.latent))).astype(F)


def dyadic_machine(net, G, h0, mutant=None):
    """The dyadic network's forward and backward in numpy float32: (d_h [R, 7, L], d_g [R, 7, L], d_dgh [R, 7, 3L],
    S [R, 3L]), bit for bit what the kernel writes.  Asserts the construction's premises on the given rows and weights.
    `mutant` runs one of rppo_train.BACKWARD_MUTANTS as backward32 does (DYADIC_BLIND ones leave every bit)."""
    L = net.latent
    w_ih, b_ih, w_hh, b_hh = net.weights[4:8]
    half, const = ~net.const, net.const
    j, gate, i, wt = net.reads
    # premises: no input path, r rows empty, one nonzero per carry column, biases cancelling the one product exactly
    assert not w_ih.any() and not w_hh[:L].any() and (np.count_nonzero(w_hh, axis=0) <= 1).all()
    assert np.array_equal(w_hh[gate * L + i, j], wt) and np.count_nonzero(w_hh) == len(j)
    assert np.array_equal(b_ih[L + i[gate == 1]] + b_hh[L + i[gate == 1]], -(rt.bf16(net.hc[j[gate == 1]]) * wt[gate == 1]))
    assert np.array_equal(b_hh[2 * L + i[gate == 2]], -(rt.bf16(net.hc[j[gate == 2]]) * wt[gate == 2]))
    assert ((b_ih + b_hh)[:L][net.r > 0] >= 40).all() and ((b_ih + b_hh)[:L][net.r == 0] <= -120).all()
    assert ((b_ih + b_hh)[L:2 * L][const] >= 40).all() and not b_ih[2 * L:].any() and not b_hh[L:2 * L].any()
    h0, G = np.asarray(h0, F), np.asarray(G, F)
    assert np.array_equal(h0[:, const], np.broadcast_to(net.hc[const], h0[:, const].shape))
    assert ((np.abs(h0[:, half]) >= 0.25) & (np.abs(h0[:, half]) <= 1)).all()
    assert ((np.abs(G) >= 2.0 ** -4) & (np.abs(G) <= 4)).all()  # g stays far from float32's subnormals and overflow
    hs = [h0]
    for _ in range(rt.K):
        hs.append(np.where(half, hs[-1] * F(0.5), hs[-1]))
    u = np.where(half, F(0.5), F(1))
    keep = rt.carry_columns(L, mutant == "carry_last_group_dropped")
    g, dgh, s = G.copy(), np.zeros((len(G), rt.K, 3 * L), F), None
    zero = np.zeros((len(G), L), F)
    for k in range(rt.K, 0, -1):
        gk = g[:, k - 1]
        hp = hs[k] if mutant == "reads_h_k" else hs[k - 1]
        dau = np.where(half, gk * (-hp if mutant == "dau_n_minus_h" else hp) * F(0.25), F(0))
        dan = np.where(half, gk * F(0.5), F(0))
        d = np.concatenate([zero, dau, dan if mutant == "dgh_n_without_r" else dan * net.r], 1)
        dgh[:, k - 1] = d
        dgi = d if mutant == "s_sums_dgh" else np.concatenate([zero, dau, dan], 1)
        s = dgi if k == rt.K else s + dgi
        if k > 1:
            gu = gk if mutant == "carry_g" else gk * (F(1) - u) if mutant == "carry_g_1mu" else gk * u
            staged = np.where(keep, bf16_rz(d) if mutant == "dgh_rz" else rt.bf16(d), F(0))
            D = np.zeros_like(zero)
            if mutant == "carry_untransposed":  # W_hg's column j for row i: the constant units' dgh, all zero
                for q in (1, 2):
                    D[:, i[gate == q]] += staged[:, q * L + j[gate == q]] * wt[gate == q]
            else:
                D[:, j] = staged[:, gate * L + i] * wt
            g[:, k - 2] = (g[:, k - 2] + gu) + D
    return np.stack(hs[1:], 1), g, dgh, s


def dyadic_case(L, R, seed):
    rng = np.random.default_rng(seed)
    net = DyadicNet(rng, 105, L)
    return net, rng.uniform(-1, 1, (R, L)).astype(F), net.h0(rng, R), net.G(rng, R)


@pytest.mark.parametrize("L", [1, 16, 17, 64, 65, 129, 192, 256])
def test_dyadic_machine_is_the_float32_statement(L):
    """forward32 and backward32 (the kernel's float32 statement, numpy's summation order) give the machine's every bit;
    the network has what the docstring claims: half units in every 64-column atom of z and n, a carry value in every
    16-column group, r both 0 and 1, staged dgh that bf16 rounds (RNE and toward zero differ)."""
    net, x, h0, G = dyadic_case(L, 200, L)
    h, g, dgh, s = dyadic_machine(net, G, h0)
    with np.errstate(over="ignore"):  # expf(120) = inf by design: 1 / (1 + inf) = 0
        _, h32 = rt.forward32(x, h0, net.weights[4:10])
    assert np.array_equal(h32, h)
    for a, b in zip(rt.backward32(x, h0, h, net.weights[4:10], G), (g, dgh, s)):
        assert np.array_equal(a, b)
    if L == 1:
        return
    half = ~net.const
    for c in range(0, L, 64):
        assert half[c:c + 64].any() and (dgh[:, :, L + c:L + c + 64] != 0).any() and (dgh[:, :, 2 * L + c:2 * L + c + 64] != 0).any()
    assert np.array_equal(np.sort(net.reads[0]), np.flatnonzero(net.const))  # every constant unit takes a carry value
    for c in range(0, L - 1, 16):
        assert net.const[c:c + 16].any(), c
    assert set(net.r[half]) == {0, 1} and (rt.bf16(dgh) != bf16_rz(dgh)).mean() > 0.1


@pytest.mark.parametrize("L", [17, 129, 256])
def test_dyadic_machine_sees_every_defect_it_claims(L):
    """Each mutant of BACKWARD_MUTANTS outside DYADIC_BLIND changes d_g, d_dgh or S in over half of the rows, as
    backward32 runs it, bit for bit; the blind ones change nothing (the step bound sees them).  The carry without its
    last atom group is claimed at L > 64 only."""
    net, x, h0, G = dyadic_case(L, 200, L + 1)
    want = dyadic_machine(net, G, h0)[1:]
    for mutant in rt.BACKWARD_MUTANTS:
        got = dyadic_machine(net, G, h0, mutant)
        for a, b in zip(rt.backward32(x, h0, got[0], net.weights[4:10], G, mutant), got[1:]):
            assert np.array_equal(a, b), mutant
        moved = np.zeros(len(G), bool)
        for a, b in zip(got[1:], want):
            moved |= (a != b).reshape(len(G), -1).any(1)
        if mutant in DYADIC_BLIND or (mutant == "carry_last_group_dropped" and L <= 64):
            assert not moved.any(), mutant
        else:
            assert moved.mean() > 0.5, (mutant, moved.mean())


def test_the_dyadic_premises_are_checked():
    """The machine refuses rows and weights it would not compute exactly."""
    net, x, h0, G = dyadic_case(40, 10, 0)
    dyadic_machine(net, G, h0)
    bad_h = h0.copy()
    bad_h[3, 1] += 1  # a constant unit that differs between rows
    bad_G = G.copy()
    bad_G[0, 0, 0] = 2.0 ** -30
    for args in ((G, bad_h), (bad_G, h0)):
        with pytest.raises(AssertionError):
            dyadic_machine(net, *args)
    net.weights[6][0, 0] = 0.5  # a half unit's r row that reads a unit
    with pytest.raises(AssertionError):
        dyadic_machine(net, G, h0)


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
def env(evg, cfg):
    return mid_game(evg, cfg, 45)


@pytest.fixture(scope="module")
def seen():
    """The worst bound ratio of each quantity over the module's step-bound cases, printed at the end (pytest -s)."""
    worst = {}
    yield worst
    for name, (ratio, where) in sorted(worst.items()):
        print("worst %s ratio %.4g at %s" % (name, ratio, where))


def batch_rows(R, sms):
    """R, or for "big" ~2.5 tiles per CTA with the last tile partial (test_gpu_policy_tiling.big's rows)."""
    return ((5 * sms + 1) // 2 - 1) * 128 + 54 if R == "big" else R


def run(fused, x, h0, G):
    """fused._train_forward then fused._train_backward into the first R rows of buffers TAIL rows longer, whose tails
    hold SENTINEL and whose outputs start as NaN (d_g as G).  Checks the writes: every element below R finite, every
    tail byte unchanged, g_7 = G_7 bit for bit.  -> (h, g, dgh, s), the first R rows, on the device."""
    import torch
    R, L = x.shape

    def buf(*shape):
        t = torch.full((R + TAIL,) + shape, float("nan"), device=x.device)
        t[R:].view(torch.int32).fill_(SENTINEL)
        return t

    z, h, g, dgh, s = buf(rt.K, fused.out_dim), buf(rt.K, L), buf(rt.K, L), buf(rt.K, 3 * L), buf(3 * L)
    g[:R] = G
    fused._train_forward(x, h0, *fused_params(fused._net), z[:R], h[:R])
    fused._train_backward(x, h0, h[:R], g[:R], dgh[:R], s[:R])
    for name, t in (("z", z), ("h", h), ("g", g), ("dgh", dgh), ("s", s)):
        assert torch.isfinite(t[:R]).all(), (name, R, torch.isfinite(t[:R]).view(R, -1).all(1).logical_not().nonzero()[:5].tolist())
        assert (t[R:].view(torch.int32) == SENTINEL).all(), (name, R)
    assert torch.equal(g[:R, 6].view(torch.int32), G[:, 6].view(torch.int32))
    return h[:R], g[:R], dgh[:R], s[:R]


# ---------------------------------------------------------------- 1. every element within the step bound

def check_steps(evg, env, sms, L, out, R, seed, seen):
    import torch
    fused, w, x, h0, rng = random_case(evg, env, L, out, R, seed)
    G = torch.from_numpy(rng.normal(size=(R, rt.K, L)).astype(F)).to(x.device)
    h, g, dgh, s = run(fused, x, h0, G)
    rows = np.arange(R) if R <= 1024 else np.concatenate([np.arange(128 * t, min(128 * t + 128, R)) for t in checked_tiles(R, sms)])
    idx = torch.from_numpy(rows).to(x.device)
    got = [t.index_select(0, idx).cpu().numpy() for t in (x, h0, h, G, g, dgh, s)]
    wb = [rt.bf16(w[4]), w[5], rt.bf16(w[6]), w[7]]
    worst = rt.worst(rt.backward_ratios(got[0], got[1], got[2], wb, *got[3:]))
    for name, (ratio, where) in worst.items():
        at = (int(rows[where[0]]),) + where[1:]  # (row, slot of d_dgh or d_g, column) or, for S, (row, column)
        if ratio > seen.get(name, (-1,))[0]:
            seen[name] = (ratio, dict(L=L, out=out, R=R, at=at))
        assert ratio <= 1, (name, L, out, R, "ratio %.3g at (row, slot, column) %s" % (ratio, at))


@gpu
@pytest.mark.parametrize("L", WIDTHS)
@pytest.mark.parametrize("out", [7, 132, 144])
def test_backward_steps_within_the_bound_at_every_width(evg, env, sms, seen, L, out):
    check_steps(evg, env, sms, L, out, 300, 31 * L + out, seen)


@gpu
@pytest.mark.parametrize("R", R_EDGES)
@pytest.mark.parametrize("L", STEP_LATENTS)
def test_backward_steps_within_the_bound_at_the_tiling_edges(evg, env, sms, seen, L, R):
    check_steps(evg, env, sms, L, 132, batch_rows(R, sms), 7 * L + 3, seen)


# ---------------------------------------------------------------- 2. bit for bit on the dyadic network

def check_dyadic(evg, env, L, R, seed, block=8192):
    import torch
    net, x, h0, G = dyadic_case(L, R, seed)
    fused = evg.policy.FusedRPPO(env, actor_of(net.weights).to(env.device))
    dev = lambda a: torch.from_numpy(a).to(env.device)  # noqa: E731
    got = run(fused, dev(x), dev(h0), dev(G))
    for r0 in range(0, R, block):
        sl = slice(r0, r0 + block)
        want = dyadic_machine(net, G[sl], h0[sl])
        for name, a, b in zip(("h", "g", "dgh", "s"), (t[sl].cpu().numpy() for t in got), want):
            assert np.array_equal(a, b), (name, L, R, np.argwhere(a != b)[:5].tolist())


@gpu
@pytest.mark.parametrize("L", LATENTS)
def test_dyadic_backward_bit_for_bit_at_every_width(evg, env, L):
    check_dyadic(evg, env, L, 300, L)


@gpu
@pytest.mark.parametrize("R", R_EDGES)
@pytest.mark.parametrize("L", DYADIC_LATENTS)
def test_dyadic_backward_bit_for_bit_at_the_tiling_edges(evg, env, sms, L, R):
    check_dyadic(evg, env, L, batch_rows(R, sms), 3 * L + 1)


# ---------------------------------------------------------------- 3. evaluate's reductions of the kernel's S and dgh

@gpu
@pytest.mark.parametrize("L,R", [(17, 300), (129, 1000), (256, 129)])
def test_evaluate_reduces_the_kernels_own_s_and_dgh(evg, env, L, R):
    """dx = S bf16(W_ih), dW_ih = S^T bf16(x), db_ih = sum S, dW_hh = sum_k dgh_k^T bf16(h_{k-1}), db_hh = sum dgh,
    dW3 = sum_k dz_k^T bf16(h_k), db3 = sum dz, each against float64 of the kernel's own float32 S, dgh and h within
    gamma_m sum |a_i b_i| (m terms, any order: torch's float32 matmul and sum without TF32)."""
    import torch
    fused, w, x, h0, rng = random_case(evg, env, L, 132, R, L + R)
    kept = {}
    launch = fused._train_backward

    def spy(x_, h0_, h_, g_, dgh_, s_):
        launch(x_, h0_, h_, g_, dgh_, s_)
        kept.update(h=h_.clone(), dgh=dgh_.clone(), s=s_.clone())

    fused._train_backward = spy
    dz = torch.from_numpy(rng.normal(size=(R, rt.K, 132)).astype(F)).to(x.device)
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        got = grads(fused, x, h0, dz)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    f64 = lambda t: np.asarray(t, np.float64)  # noqa: E731
    s, dgh, h = (f64(kept[k].cpu().numpy()) for k in ("s", "dgh", "h"))
    dgh = dgh.reshape(R * rt.K, 3 * L)
    xb, hb = rt.bf16(f64(x.cpu().numpy())), rt.bf16(h).reshape(R * rt.K, L)
    hprev = rt.bf16(np.concatenate([f64(h0.cpu().numpy())[:, None], h[:, :rt.K - 1]], 1)).reshape(R * rt.K, L)
    dzs = f64(dz.cpu().numpy()).reshape(R * rt.K, 132)
    wih = rt.bf16(f64(w[4]))
    ones = lambda n: np.ones((n, 1))  # noqa: E731
    want = [(s, wih), (s.T, xb), (s.T, ones(R)), (dgh.T, hprev), (dgh.T, ones(R * rt.K)), (dzs.T, hb), (dzs.T, ones(R * rt.K))]
    for name, a, (p, q) in zip(["dx", "dw_ih", "db_ih", "dw_hh", "db_hh", "dw3", "db3"], got, want):
        ref = (p @ q).reshape(a.shape)
        bound = rt._gamma(p.shape[1]) * (np.abs(p) @ np.abs(q)).reshape(a.shape)
        err = np.abs(a - ref)
        assert (err <= bound).all(), (name, L, R, float((err / np.maximum(bound, 1e-300)).max()))
