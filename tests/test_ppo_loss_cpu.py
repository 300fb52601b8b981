"""tests/ppo_loss.py on the CPU: the log-probability of the ordered seven draws against an enumeration in float64, the
analytic gradient against torch's float64 autograd and central differences, the float32 statement within the derived
bound, and the C ABI entries: in the binding, and refusing bad arguments without a GPU."""
import ctypes as C
import itertools

import numpy as np
import pytest

from evgsim import _capi
from ppo_loss import grad_float64, loss_bound, loss_float64, reference_loss, torch_loss


def rows(rng, B, K, n, scale=1.5):
    z = (rng.standard_normal((B, n) if K == 1 else (B, 7, n)) * scale).astype(np.float32)
    if K == 1:
        idx = np.stack([rng.permutation(n)[:7] for _ in range(B)]).astype(np.int64)
    else:
        idx = rng.integers(0, n, (B, 7)).astype(np.int64)
    old = (rng.standard_normal((B, 7)) * 0.1 - np.log(n)).astype(np.float32)
    adv = rng.standard_normal(B).astype(np.float32)
    return z, idx, old, adv


def test_ell_is_the_log_probability_of_the_ordered_draws():
    """n = 8: every ordered 7-tuple of distinct actions.  Sequential sampling without replacement gives the tuple
    probability prod_k p_{j_k} / (1 - sum of the p drawn before k); those add up to 1, and the statements' ell (the sum of
    the seven logp) is its log."""
    n = 8
    rng = np.random.default_rng(0)
    z1 = (rng.standard_normal(n) * 2).astype(np.float32)
    p = np.exp(np.tanh(z1.astype(np.float64)))
    p /= p.sum()
    tuples = np.array(list(itertools.permutations(range(n), 7)), dtype=np.int64)
    prob = np.ones(len(tuples))
    gone = np.zeros(len(tuples))
    for k in range(7):
        pj = p[tuples[:, k]]
        prob *= pj / (1.0 - gone)
        gone += pj
    assert abs(prob.sum() - 1.0) < 1e-12
    B = len(tuples)
    z = np.repeat(z1[None], B, axis=0)
    old = np.zeros((B, 7), np.float32)
    adv = np.ones(B, np.float32)
    _, _, logp64, _ = loss_float64(z, tuples, old, adv, 0.2)
    assert np.allclose(logp64.sum(-1), np.log(prob), rtol=0, atol=1e-12)
    _, _, logp32, _ = reference_loss(z, tuples, old, adv, 0.2)
    _, _, b_logp, _ = loss_bound(z, tuples, old, adv, 0.2)
    assert np.all(np.abs(logp32 - logp64) <= b_logp)
    assert np.all(np.abs(logp32.astype(np.float64).sum(-1) - np.log(prob)) <= b_logp.sum(-1) + 7 * 2 ** -23 * 8)


@pytest.mark.parametrize("K", [1, 7])
def test_gradient_equals_torch_float64_and_central_differences(K):
    import torch
    rng = np.random.default_rng(K)
    B, n = 24, 11
    z, idx, old, adv = rows(rng, B, K, n)
    adv[:4] = [2.0, -2.0, 0.0, 1.0]
    old[0] += 0.3  # row 0 (A > 0, r < 1): unclipped; row 1 (A < 0, r > 1): unclipped
    g_s = rng.standard_normal(B)
    g_e = rng.standard_normal(B)
    for clip in (0.2, 0.0, 0.99):
        zt = torch.tensor(z, dtype=torch.float64, requires_grad=True)
        surr, ent, logp, ratio = torch_loss(zt, torch.tensor(idx), torch.tensor(old), torch.tensor(adv), clip)
        (surr * torch.tensor(g_s)).sum().add((ent * torch.tensor(g_e)).sum()).backward()
        s64, e64, l64, r64 = loss_float64(z, idx, old, adv, clip)
        assert np.allclose(surr.detach().numpy(), s64, rtol=1e-12, atol=1e-12)
        assert np.allclose(ent.detach().numpy(), e64, rtol=1e-12, atol=1e-12)
        assert np.allclose(logp.detach().numpy(), l64, rtol=1e-12, atol=1e-12)
        want = grad_float64(z, idx, adv, r64, clip, g_s, g_e)
        assert np.allclose(zt.grad.numpy(), want, rtol=1e-10, atol=1e-12), clip
    # central differences of the float64 definition, on rows away from the clip boundary
    clip = 0.2
    _, _, _, r64 = loss_float64(z, idx, old, adv, clip)
    ok = (np.abs(r64 - 0.8) > 1e-3) & (np.abs(r64 - 1.2) > 1e-3)
    want = grad_float64(z, idx, adv, r64, clip, g_s, g_e)
    h = 1e-6
    zf = z.astype(np.float64)
    flat = zf.reshape(B, -1)
    for col in range(flat.shape[1]):
        up, dn = flat.copy(), flat.copy()
        up[:, col] += h
        dn[:, col] -= h
        fu = loss_float64(up.reshape(z.shape), idx, old, adv, clip)
        fd = loss_float64(dn.reshape(z.shape), idx, old, adv, clip)
        num = ((fu[0] - fd[0]) * g_s + (fu[1] - fd[1]) * g_e) / (2 * h)
        assert np.allclose(num[ok], want.reshape(B, -1)[ok, col], rtol=1e-6, atol=1e-7), col


@pytest.mark.parametrize("K,n", [(1, 7), (1, 132), (1, 256), (7, 7), (7, 132), (7, 256)])
def test_float32_statement_within_the_derived_bound(K, n):
    rng = np.random.default_rng(n + K)
    z, idx, old, adv = rows(rng, 300, K, n)
    z[:10] = 0.0
    z[10:20] = 20.0 * np.sign(z[10:20])
    for clip in (0.0, 0.2, 0.99):
        got = reference_loss(z, idx, old, adv, clip)
        want = loss_float64(z, idx, old, adv, clip)
        bound = loss_bound(z, idx, old, adv, clip)
        for g, w, b in zip(got, want, bound):
            assert np.all(np.abs(g - w) <= b), (K, n, clip)
    assert np.allclose(want[1][:10], np.log(n), rtol=0, atol=1e-12)  # z = 0: the uniform distribution


def test_ppo_loss_is_in_the_binding():
    rows_ = {s[0]: s for s in _capi.SYMBOLS}
    _, res, args = rows_["evg_ppo_loss"]
    assert res is C.c_int and len(args) == 14 and args[1] is C.c_int64 and args[8] is C.c_float
    _, res, args = rows_["evg_ppo_loss_grad"]
    assert res is C.c_int and len(args) == 13 and args[1] is C.c_int64 and args[8] is C.c_float


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    return _capi.load()


def test_abi_refuses_bad_arguments_without_a_device(lib):
    """The argument checks come before the handle's, so each refusal names its argument even with a NULL handle."""
    buf = (C.c_double * 64)()
    a = C.addressof(buf)
    good = dict(B=4, K=1, n=132, z=a, idx=a, old=a, adv=a, clip=0.2, surr=a, ent=a, logp=a, ratio=a)

    def fwd(**kw):
        x = dict(good, **kw)
        rc = lib.evg_ppo_loss(None, x["B"], x["K"], x["n"], C.c_void_p(x["z"]), C.c_void_p(x["idx"]), C.c_void_p(x["old"]),
                              C.c_void_p(x["adv"]), x["clip"], C.c_void_p(x["surr"]), C.c_void_p(x["ent"]), C.c_void_p(x["logp"]),
                              C.c_void_p(x["ratio"]), None)
        return rc, lib.evg_last_error().decode()

    cases = [(dict(B=0), "n_rows"), (dict(B=-1), "n_rows"), (dict(B=1 << 31), "n_rows"), (dict(K=2), "n_dist"), (dict(K=0), "n_dist"),
             (dict(n=6), "n_actions"), (dict(n=257), "n_actions"), (dict(clip=-0.1), "clip"), (dict(clip=1.0), "clip"),
             (dict(clip=float("nan")), "clip"), (dict(idx=None), "idx"), (dict(idx=a + 4), "idx"), (dict(z=None), "operand 0"),
             (dict(z=a + 2), "operand 0"), (dict(old=None), "operand 1"), (dict(adv=None), "operand 2"), (dict(surr=None), "operand 3"),
             (dict(ent=None), "operand 4"), (dict(logp=a + 1), "operand 5"), (dict(ratio=None), "operand 6")]
    for kw, word in cases:
        rc, msg = fwd(**kw)
        assert rc == -1 and word in msg, (kw, msg)
    rc, msg = fwd()
    assert rc == -1 and "null EvgSim handle" in msg
    rc, msg = fwd(K=7, n=7, clip=0.0)
    assert rc == -1 and "null EvgSim handle" in msg

    def bwd(**kw):
        x = dict(dict(good, gs=None, ge=None), **kw)
        rc = lib.evg_ppo_loss_grad(None, x["B"], x["K"], x["n"], C.c_void_p(x["z"]), C.c_void_p(x["idx"]), C.c_void_p(x["adv"]),
                                   C.c_void_p(x["ratio"]), x["clip"], C.c_void_p(x["gs"]), C.c_void_p(x["ge"]), C.c_void_p(x["surr"]), None)
        return rc, lib.evg_last_error().decode()

    for kw, word in [(dict(K=3), "n_dist"), (dict(n=300), "n_actions"), (dict(clip=2.0), "clip"), (dict(idx=None), "idx"),
                     (dict(z=None), "operand 0"), (dict(adv=None), "operand 1"), (dict(ratio=None), "operand 2"),
                     (dict(surr=None), "operand 3"), (dict(gs=a + 2), "g_surr"), (dict(ge=a + 1), "g_ent")]:
        rc, msg = bwd(**kw)
        assert rc == -1 and word in msg, (kw, msg)
    rc, msg = bwd(gs=a, ge=a)
    assert rc == -1 and "null EvgSim handle" in msg
