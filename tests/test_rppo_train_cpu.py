"""CPU checks of the recurrent actor's update operation: its analytic backward against torch float64 autograd and central
differences, the float32 forward within the derived step bound, the float32 backward within the derived backward step
bound and each of its plausible defects outside it, the transposed image layout, and the C ABI's refusals."""
import ctypes as C

import numpy as np
import pytest

import rppo_train as rt
from evgsim import _capi, policy


def weights(rng, L, out, scale=1.0):
    s = scale / np.sqrt(L)
    return [rng.uniform(-s, s, shape) for shape in ((3 * L, L), 3 * L, (3 * L, L), 3 * L, (out, L), out)]


@pytest.mark.parametrize("L,out", [(1, 7), (5, 9), (16, 7), (33, 20)])
def test_analytic_backward_equals_torch_float64_autograd(L, out):
    rng = np.random.default_rng(L)
    R = 6
    w = weights(rng, L, out, scale=2.0)
    x, h0, dz = rng.uniform(-1, 1, (R, L)), rng.uniform(-1, 1, (R, L)), rng.normal(size=(R, 7, out))
    z_t, g_t = rt.torch_reference(x, h0, w, dz)
    z, _, _ = rt.forward64(x, h0, w)
    assert np.allclose(z, z_t, rtol=0, atol=1e-12)
    for a, b in zip(rt.backward64(x, h0, w, dz), g_t):
        assert np.allclose(a, b, rtol=1e-10, atol=1e-12)


def test_analytic_backward_equals_central_differences():
    rng = np.random.default_rng(3)
    R, L, out = 3, 4, 7
    w = weights(rng, L, out, scale=2.0)
    x, h0, dz = rng.uniform(-1, 1, (R, L)), rng.uniform(-1, 1, (R, L)), rng.normal(size=(R, 7, out))
    grads = rt.backward64(x, h0, w, dz)
    loss = lambda x_, w_: float((rt.forward64(x_, h0, w_)[0] * dz).sum())  # noqa: E731
    eps = 1e-6
    for idx in [(0, 0), (2, 3), (1, 1)]:
        xp, xm = x.copy(), x.copy()
        xp[idx] += eps
        xm[idx] -= eps
        assert abs((loss(xp, w) - loss(xm, w)) / (2 * eps) - grads[0][idx]) < 1e-7
    for i, gi in zip(range(6), grads[1:]):
        for _ in range(3):
            j = tuple(rng.integers(0, n) for n in np.shape(w[i]))
            wp = [a.copy() for a in w]
            wm = [a.copy() for a in w]
            wp[i][j] += eps
            wm[i][j] -= eps
            assert abs((loss(x, wp) - loss(x, wm)) / (2 * eps) - gi[j]) < 1e-7, (i, j)


@pytest.mark.parametrize("L", [1, 16, 128, 248])
def test_float32_statement_within_the_step_bound(L):
    rng = np.random.default_rng(L)
    R, out = 64, 132
    w = [a.astype(np.float32) for a in weights(rng, L, out)]
    wb = [rt.bf16(w[0]), w[1], rt.bf16(w[2]), w[3], rt.bf16(w[4]), w[5]]
    x, h0 = rng.uniform(-1, 1, (R, L)).astype(np.float32), rng.uniform(-1, 1, (R, L)).astype(np.float32)
    z32, h32 = rt.forward32(x, h0, w)
    worst = 0.0
    for k in range(7):
        hp = h0 if k == 0 else h32[:, k - 1]
        _, h64, _ = rt.forward64(x, hp, wb, rnd=rt.bf16)
        b = rt.step_bound(x, hp, wb)
        assert np.all(np.abs(h32[:, k] - h64[:, 0]) <= b), k
        worst = max(worst, float((np.abs(h32[:, k] - h64[:, 0]) / b).max()))
        zb = rt.z_bound(h32[:, k], w[4], w[5])
        z64 = rt.bf16(h32[:, k].astype(np.float64)) @ wb[4].astype(np.float64).T + w[5]
        assert np.all(np.abs(z32[:, k] - z64) <= zb), k
    assert worst < 0.5, worst  # margin: the statement uses under half the bound
    assert np.max(rt.step_bound(x, h0, wb)) < 1e-3  # and the bound is tight enough to catch a bf16-sized error


@pytest.mark.parametrize("L", [1, 17, 64, 129, 256])
def test_transposed_image_layout_at_every_swizzle_position(L):
    """Element (j, i) of gate g's W_hg^T block is w_hh[g L + i][j], at the swizzled offset of every (row, column)."""
    rng = np.random.default_rng(L)
    w_hh = rng.normal(size=(3 * L, L)).astype(np.float32)
    img = rt.pack_wht(w_hh)
    lp, ka = -(-L // 16) * 16, -(-L // 64) * 64
    blk = ka // 64 * lp * 128
    assert img.size == 3 * blk
    bits = img.view(np.uint16)
    for g in range(3):
        j, i = np.meshgrid(np.arange(lp), np.arange(ka), indexing="ij")
        got = bits[(g * blk + policy.swz_offset(lp, j, i)) // 2]
        want = np.zeros((lp, ka), dtype=np.float32)
        want[:L, :L] = w_hh[g * L:(g + 1) * L].T
        assert np.array_equal(got, policy.to_bf16_bits(want)), g
    # every 16-byte chunk position is written exactly once
    j, i = np.meshgrid(np.arange(lp), np.arange(ka), indexing="ij")
    offs = np.sort(policy.swz_offset(lp, j, i).ravel())
    assert np.array_equal(offs, np.arange(0, blk, 2))


def test_rppo_train_is_in_the_binding():
    rows_ = {s[0]: s for s in _capi.SYMBOLS}
    assert len(rows_["evg_rppo_train_pack"][2]) == 15
    assert len(rows_["evg_rppo_train_forward"][2]) == 13 and rows_["evg_rppo_train_forward"][2][1] is C.c_int64
    assert len(rows_["evg_rppo_train_backward"][2]) == 15 and rows_["evg_rppo_train_backward"][2][1] is C.c_int64


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    return _capi.load()


def test_abi_refuses_bad_arguments_without_a_device(lib):
    """The argument checks come before the handle's, so each refusal names its argument even with a NULL handle."""
    buf = (C.c_double * 64)()
    a = C.addressof(buf)
    a = a + (-a) % 16
    good = dict(B=4, L=128, o=132, x=a, h0=a, wi=a, wh=a, wht=a, w3=a, bias=a, z=a, h=a, g=a, dgh=a, s=a)

    def fwd(**kw):
        v = dict(good, **kw)
        p = lambda n: C.c_void_p(v[n])  # noqa: E731
        rc = lib.evg_rppo_train_forward(None, v["B"], v["L"], v["o"], p("x"), p("h0"), p("wi"), p("wh"), p("w3"), p("bias"), p("z"), p("h"), None)
        return rc, lib.evg_last_error().decode()

    def bwd(**kw):
        v = dict(good, **kw)
        p = lambda n: C.c_void_p(v[n])  # noqa: E731
        rc = lib.evg_rppo_train_backward(None, v["B"], v["L"], v["o"], p("x"), p("h0"), p("h"), p("wi"), p("wh"), p("wht"), p("bias"),
                                         p("g"), p("dgh"), p("s"), None)
        return rc, lib.evg_last_error().decode()

    def pack(**kw):
        v = dict(good, **kw)
        p = lambda n: C.c_void_p(v[n])  # noqa: E731
        rc = lib.evg_rppo_train_pack(None, p("x"), p("x"), p("h0"), p("h0"), p("h"), p("h"), v["L"], v["o"], p("wi"), p("wh"), p("wht"), p("w3"),
                                     p("bias"), None)
        return rc, lib.evg_last_error().decode()

    common = [(dict(L=0), "latent"), (dict(L=257), "latent"), (dict(o=6), "out_dim"), (dict(o=145), "out_dim"),
              (dict(wi=None), "null image"), (dict(wi=a + 8), "16-byte"), (dict(wh=a + 4), "16-byte"), (dict(bias=None), "null image")]
    for call, extra in [(fwd, [(dict(w3=None), "null image"), (dict(x=None), "null float32"), (dict(x=a + 2), "4-byte"), (dict(h0=None), "null float32"),
                               (dict(z=a + 1), "4-byte"), (dict(h=None), "null float32")]),
                        (bwd, [(dict(wht=a + 8), "16-byte"), (dict(x=None), "null float32"), (dict(h=a + 2), "4-byte"), (dict(g=None), "null float32"),
                               (dict(dgh=None), "null float32"), (dict(s=a + 1), "4-byte")]),
                        (pack, [(dict(wht=None), "null image"), (dict(w3=a + 4), "16-byte"), (dict(h0=None), "null float32"), (dict(h=a + 2), "4-byte")])]:
        for kw, word in common + extra:
            rc, msg = call(**kw)
            assert rc == -1 and word in msg, (call.__name__, kw, msg)
        if call is not pack:
            for B in (0, -1, 1 << 31):
                rc, msg = call(B=B)
                assert rc == -1 and "n_rows" in msg, (call.__name__, B, msg)
        rc, msg = call()
        assert rc == -1 and "null EvgSim handle" in msg, (call.__name__, msg)


def backward_case(L, R=64, seed=None):
    """A random float network, its float32 forward and an entry value G of d_g: (x, h0, h, w, wb, G)."""
    rng = np.random.default_rng(L if seed is None else seed)
    w = [a.astype(np.float32) for a in weights(rng, L, 132)]
    wb = [rt.bf16(w[0]), w[1], rt.bf16(w[2]), w[3], rt.bf16(w[4]), w[5]]
    x, h0 = rng.uniform(-1, 1, (R, L)).astype(np.float32), rng.uniform(-1, 1, (R, L)).astype(np.float32)
    _, h = rt.forward32(x, h0, w)
    G = rng.normal(size=(R, 7, L)).astype(np.float32)
    return x, h0, h, w, wb, G


@pytest.mark.parametrize("L", [1, 16, 17, 128, 129, 248])
def test_float32_backward_within_the_backward_step_bound(L):
    """backward32 (the kernel's statement in numpy's summation order) keeps dgh_k, g_{k-1} and S of every step within
    under half of backward_step_bound, leaves g_7 as it came in, and the bound is far below a bf16-sized error."""
    x, h0, h, w, wb, G = backward_case(L)
    g, dgh, s = rt.backward32(x, h0, h, w, G)
    assert np.array_equal(g[:, 6], G[:, 6])
    worst = rt.worst(rt.backward_ratios(x, h0, h, wb, G, g, dgh, s))
    assert all(v[0] < 0.5 for v in worst.values()), worst
    b = rt.backward_step_bound(x, h[:, 5], wb, g[:, 6], G[:, 5], dgh[:, 6])
    assert b.dgh_b.max() < 2.0 ** -12 * np.abs(b.dgh).max() and b.g_b.max() < 2.0 ** -12 * np.abs(b.g).max()


@pytest.mark.parametrize("L", [17, 129, 248])
def test_each_backward_mutant_leaves_the_bound(L):
    """Every plausible defect of BACKWARD_MUTANTS takes every row out of the bound (share 1.0), in the quantity it
    corrupts: dgh for the gradient formulas, g_{k-1} for the carry, S for its sum.  The carry without its last group of
    atoms is only a defect for L > 64 (one group below); nothing is claimed for it at L = 17."""
    x, h0, h, w, wb, G = backward_case(L)
    where = {"carry_g": "g", "carry_g_1mu": "g", "carry_untransposed": "g", "carry_last_group_dropped": "g", "dgh_rz": "g",
             "s_sums_dgh": "S"}
    for mutant in rt.BACKWARD_MUTANTS:
        if mutant == "carry_last_group_dropped" and L <= 64:
            continue
        g, dgh, s = rt.backward32(x, h0, h, w, G, mutant)
        ratio = rt.backward_ratios(x, h0, h, wb, G, g, dgh, s)[where.get(mutant, "dgh")]
        caught = ~(ratio.reshape(len(x), -1) <= 1).all(1)
        assert caught.mean() == 1.0, (mutant, caught.mean())


def test_gate_bounds_are_the_step_bounds():
    """step_bound is gate_bounds' e_n and e_u carried through h' = (1 - u) n + u h, and e_c holds c's one dot product."""
    x, h0, h, w, wb, G = backward_case(33, R=8)
    e_r, e_u, e_n, e_c = rt.gate_bounds(x, h0, wb)
    assert np.array_equal(rt.step_bound(x, h0, wb), e_n + e_u * (1 + np.abs(h0)) + 4 * rt.U32 * (1 + np.abs(h0)))
    assert (e_r >= 8 * rt.U32).all() and (e_u >= 8 * rt.U32).all() and (e_c > 0).all()
