"""CPU checks of the feed-forward update networks (evg_ppo_train_*): the analytic backward against torch float64
autograd and central differences, the float32 statement within its derived per-layer bound, the W2^T image at every
swizzle position, and the C ABI's refusals without a device."""
import ctypes as C

import numpy as np
import pytest

import ppo_train as pt
from evgsim import _capi, policy

NETS = ["actor", "critic", "head"]


def weights(rng, net, L, out=7, in_dim=9, scale=2.0):
    s1, s = scale / np.sqrt(in_dim), scale / np.sqrt(L)
    w = [rng.uniform(-s1, s1, (L, in_dim)), rng.uniform(-s1, s1, L), rng.uniform(-s, s, (L, L)), rng.uniform(-s, s, L)]
    if net == "actor":
        w += [rng.uniform(-s, s, (out, L)), rng.uniform(-s, s, out)]
    elif net == "critic":
        w += [rng.uniform(-s, s, (1, L)), rng.uniform(-s, s, 1)]
    return w


def upstream(rng, net, R, L, out=7):
    return rng.normal(size={"actor": (R, out), "critic": (R,), "head": (R, L)}[net])


@pytest.mark.parametrize("net", NETS)
@pytest.mark.parametrize("L", [1, 5, 17])
def test_analytic_backward_equals_torch_float64_autograd(net, L):
    rng = np.random.default_rng(L)
    R = 6
    w = weights(rng, net, L)
    obs, dy = rng.uniform(-1, 1, (R, 9)), upstream(rng, net, R, L)
    y_t, g_t = pt.torch_reference(obs, w, net, dy)
    assert np.allclose(pt.forward64(obs, w, net)[0], y_t, rtol=0, atol=1e-12)
    got = pt.backward64(obs, w, net, dy)
    assert len(got) == len(w)
    for a, b, p in zip(got, g_t, w):
        assert np.shape(a) == np.shape(p)
        assert np.allclose(a, b, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("net", NETS)
def test_analytic_backward_equals_central_differences(net):
    rng = np.random.default_rng(3)
    R, L = 3, 4
    w = weights(rng, net, L)
    obs, dy = rng.uniform(-1, 1, (R, 9)), upstream(rng, net, R, L)
    grads = pt.backward64(obs, w, net, dy)
    loss = lambda w_: float((pt.forward64(obs, w_, net)[0] * dy).sum())  # noqa: E731
    eps = 1e-6
    for i, gi in enumerate(grads):
        for _ in range(3):
            j = tuple(rng.integers(0, n) for n in np.shape(w[i]))
            wp, wm = [a.copy() for a in w], [a.copy() for a in w]
            wp[i][j] += eps
            wm[i][j] -= eps
            assert abs((loss(wp) - loss(wm)) / (2 * eps) - gi[j]) < 1e-7, (i, j)


@pytest.mark.parametrize("L", [1, 16, 128, 248, 256])
def test_float32_statement_within_the_layer_bound(L):
    """Each hidden layer of forward32 within layer_bound of float64 on the same bf16 operands, using under half of it;
    and the bound is far below a bf16-sized error."""
    rng = np.random.default_rng(L)
    R = 64
    w = [a.astype(np.float32) for a in weights(rng, "head", L, in_dim=105, scale=1.0)]
    obs = rng.integers(0, 20, (R, 105)).astype(np.float32)
    _, h1, h2 = pt.forward32(obs, w, "head")
    worst = 0.0
    for x, h, wi, bi in ((obs, h1, w[0], w[1]), (h1, h2, w[2], w[3])):
        exact = np.tanh(pt.bf16(x.astype(np.float64)) @ pt.bf16(wi.astype(np.float64)).T + bi)
        b = pt.layer_bound(x, wi, bi)
        assert np.all(np.abs(h - exact) <= b)
        worst = max(worst, float((np.abs(h - exact) / b).max()))
        assert b.max() < 2.0 ** -10
    assert worst < 0.5, worst


@pytest.mark.parametrize("L", [1, 17, 64, 129, 256])
def test_w2t_image_at_every_swizzle_position(L):
    """Element (j, i) of the W2^T block is w2[i][j], at the swizzled offset of every (row, column); every 16-byte chunk
    position is written exactly once."""
    rng = np.random.default_rng(L)
    w2 = rng.normal(size=(L, L)).astype(np.float32)
    img = pt.pack_w2t(w2)
    lp, ka = -(-L // 16) * 16, -(-L // 64) * 64
    assert img.size == ka // 64 * lp * 128
    j, i = np.meshgrid(np.arange(lp), np.arange(ka), indexing="ij")
    want = np.zeros((lp, ka), dtype=np.float32)
    want[:L, :L] = w2.T
    assert np.array_equal(img.view(np.uint16)[policy.swz_offset(lp, j, i) // 2], policy.to_bf16_bits(want))
    assert np.array_equal(np.sort(policy.swz_offset(lp, j, i).ravel()), np.arange(0, img.size, 2))


def test_ppo_train_is_in_the_binding():
    rows_ = {s[0]: s for s in _capi.SYMBOLS}
    assert len(rows_["evg_ppo_train_pack"][2]) == 16
    assert len(rows_["evg_ppo_train_forward"][2]) == 16 and rows_["evg_ppo_train_forward"][2][4] is C.c_int64
    assert len(rows_["evg_ppo_train_backward"][2]) == 10 and rows_["evg_ppo_train_backward"][2][1] is C.c_int64


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
    A, CR, H = _capi.PPO_TRAIN_ACTOR, _capi.PPO_TRAIN_CRITIC, _capi.PPO_TRAIN_HEAD
    good = dict(net=A, fmt=_capi.OBS_WIRE, obs=a, M=4, player=-1, B=4, L=128, o=132, w1=a, w2=a, w3=a, w2t=a, bias=a, out=a, h1=a, h2=a,
                g2=a, dd2=a, dd1=a, s=a)

    def fwd(**kw):
        v = dict(good, **kw)
        p = lambda n: C.c_void_p(v[n])  # noqa: E731
        rc = lib.evg_ppo_train_forward(None, v["net"], v["fmt"], p("obs"), v["M"], v["player"], v["L"], v["o"], p("w1"), p("w2"), p("w3"), p("bias"),
                                       p("out"), p("h1"), p("h2"), None)
        return rc, lib.evg_last_error().decode()

    def bwd(**kw):
        v = dict(good, **kw)
        p = lambda n: C.c_void_p(v[n])  # noqa: E731
        rc = lib.evg_ppo_train_backward(None, v["B"], v["L"], p("w2t"), p("g2"), p("h1"), p("h2"), p("dd2"), p("dd1"), None)
        return rc, lib.evg_last_error().decode()

    def pack(**kw):
        v = dict(good, **kw)
        p = lambda n: C.c_void_p(v[n])  # noqa: E731
        rc = lib.evg_ppo_train_pack(None, v["net"], p("s"), p("s"), p("s"), p("s"), p("g2"), p("g2"), v["L"], v["o"], p("w1"), p("w2"), p("w3"),
                                    p("w2t"), p("bias"), None)
        return rc, lib.evg_last_error().decode()

    net_cases = [(dict(net=3), "unknown network"), (dict(net=-1), "unknown network"), (dict(L=0), "latent"), (dict(L=257), "latent"),
                 (dict(o=6), "out_dim"), (dict(o=145), "out_dim"), (dict(net=CR, o=2), "out_dim"), (dict(net=H, o=132), "out_dim"),
                 (dict(w1=None), "null image"), (dict(w2=a + 8), "16-byte"), (dict(w3=None), "null image"), (dict(bias=a + 4), "16-byte")]
    cases = {
        fwd: net_cases + [(dict(player=2), "player"), (dict(player=-2), "player"), (dict(M=0), "n_matches"), (dict(M=-1), "n_matches"),
                          (dict(M=1 << 30), "n_matches"), (dict(fmt=_capi.OBS_I16), "format"), (dict(fmt=7), "format"),
                          (dict(obs=None), "null observations"), (dict(obs=a + 4), "16-byte"), (dict(fmt=_capi.OBS_F32, obs=a + 2), "4-byte"),
                          (dict(out=None), "null float32"), (dict(h1=a + 2), "4-byte"), (dict(h2=None), "null float32")],
        pack: net_cases + [(dict(w2t=None), "null image"), (dict(s=None), "null float32"), (dict(g2=a + 1), "4-byte")],
        bwd: [(dict(B=0), "n_rows"), (dict(B=-1), "n_rows"), (dict(B=1 << 31), "n_rows"), (dict(L=0), "latent"), (dict(L=257), "latent"),
              (dict(w2t=None), "null image"), (dict(w2t=a + 8), "16-byte"), (dict(g2=None), "null float32"), (dict(h1=a + 2), "4-byte"),
              (dict(h2=None), "null float32"), (dict(dd2=a + 1), "4-byte"), (dict(dd1=None), "null float32")],
    }
    for call, cs in cases.items():
        for kw, word in cs:
            rc, msg = call(**kw)
            assert rc == -1 and word in msg, (call.__name__, kw, msg)
        rc, msg = call()
        assert rc == -1 and "null EvgSim handle" in msg, (call.__name__, msg)
    # the head needs no last layer: its w3 / b3 / out may be NULL, and the critic's M x 2 rows may reach 2^31 - 1 only
    for kw in (dict(net=H, o=128, w3=None, out=None), dict(net=CR, o=1, M=(1 << 30) - 1)):
        rc, msg = fwd(**kw)
        assert rc == -1 and "null EvgSim handle" in msg, (kw, msg)
    rc, msg = pack(net=H, o=128, w3=None, g2=None)
    assert rc == -1 and "null EvgSim handle" in msg, msg
