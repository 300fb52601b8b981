"""tests/ppo_gae.py on the CPU: the float32 reference on a rollout worked by hand, its distance to the float64 textbook
form against the derived bound, and the C ABI entry in the binding."""
import numpy as np

from evgsim import _capi
from ppo_gae import gae_bound, gae_float64, reference_gae


def test_reference_equals_a_rollout_worked_by_hand():
    """gamma = lam = 1/2 (gl = 1/4) and binary fractions, so every step is exact.  Column 0 holds two episodes, done at
    t = 0 and at t = T-1 = 4 (its bootstrap V_5 = 8 is cut); column 1 is never done and bootstraps from V_5.
      column 0: t=4 delta = -1 - 4 = -5, A = -5;  t=3 delta = 2 + 2 - 1/2 = 7/2, A = 7/2 - 5/4 = 9/4;
                t=2 delta = 1/2 + 1/4 + 1 = 7/4, A = 7/4 + 9/16 = 37/16;  t=1 delta = 0 - 1/2 - 2 = -5/2,
                A = -5/2 + 37/64 = -123/64;  t=0 (done) delta = 1 - 1 = 0, A = 0.
      column 1: t=4 delta = -1 + 4 - 4 = -1;  t=3 A = 7/2 - 1/4 = 13/4;  t=2 A = 7/4 + 13/16 = 41/16;
                t=1 A = -5/2 + 41/64 = -119/64;  t=0 delta = 1 + 1 - 1 = 1, A = 1 - 119/256 = 137/256.
    R_t = A_t + V_t."""
    v = np.array([1.0, 2.0, -1.0, 0.5, 4.0, 8.0], dtype=np.float32)
    r = np.array([1.0, 0.0, 0.5, 2.0, -1.0], dtype=np.float32)
    values = np.stack([v, v], axis=1)  # [T+1, M = 2]
    reward = np.stack([r, r], axis=1)
    done = np.array([[1, 0], [0, 0], [0, 0], [0, 0], [1, 0]], dtype=np.uint8)
    adv, ret = reference_gae(values, reward, done, 0.5, 0.5)
    want_a = np.array([[0.0, 137 / 256], [-123 / 64, -119 / 64], [37 / 16, 41 / 16], [9 / 4, 13 / 4], [-5.0, -1.0]])
    assert adv.dtype == np.float32 and np.array_equal(adv, want_a.astype(np.float32))
    assert np.array_equal(ret, (want_a + v[:5, None]).astype(np.float32))
    a64, r64 = gae_float64(values, reward, done, 0.5, 0.5)
    assert np.array_equal(a64, want_a) and np.array_equal(r64, want_a + v[:5, None])


def random_rollout(rng, T, M, cols=2, p_done=0.05, scale=10.0):
    values = (rng.standard_normal((T + 1, M, cols)) * scale).astype(np.float32)
    reward = (rng.standard_normal((T, M, cols)) * scale / 4).astype(np.float32)
    done = (rng.random((T, M)) < p_done).astype(np.uint8)
    return values, reward, done


def test_reference_within_the_derived_bound_of_float64():
    rng = np.random.default_rng(0)
    worst = 0.0
    for gamma, lam in ((0.99, 0.95), (1.0, 1.0), (0.9, 0.0), (0.0, 0.7), (0.999, 0.99)):
        for p_done in (0.0, 0.02, 0.5):
            values, reward, done = random_rollout(rng, 300, 64, p_done=p_done)
            adv, ret = reference_gae(values, reward, done, gamma, lam)
            a64, r64 = gae_float64(values, reward, done, gamma, lam)
            ea, er = gae_bound(values, reward, done, gamma, lam)
            assert np.all(np.abs(adv - a64) <= ea), (gamma, lam, p_done)
            assert np.all(np.abs(ret - r64) <= er), (gamma, lam, p_done)
            worst = max(worst, float(np.max(np.abs(adv - a64) / ea)))
    assert worst > 1e-3  # the bound is not vacuous: the float32 pass does leave the float64 value


def test_bound_weights_the_trace_behind_each_turn():
    """With gl = 0 the bound is a few roundings of the turn itself; with gl near 1 and no done it grows with the length of
    the trace behind it, as (c gl)^k weights say."""
    rng = np.random.default_rng(1)
    values, reward, done = random_rollout(rng, 200, 8, p_done=0.0)
    e0, _ = gae_bound(values, reward, done, 0.9, 0.0)
    e1, _ = gae_bound(values, reward, done, 1.0, 1.0)
    mag = np.abs(values[:-1]) + np.abs(reward) + np.abs(values[1:])
    assert np.all(e0 <= 6 * 2.0 ** -24 * mag * 1.0001)
    assert e1[0].mean() > 50 * e1[-1].mean()


def test_gae_is_in_the_binding():
    import ctypes as C
    row = [s for s in _capi.SYMBOLS if s[0] == "evg_gae"]
    assert len(row) == 1
    _, res, args = row[0]
    assert res is C.c_int and len(args) == 13
    assert args[8] is C.c_float and args[9] is C.c_float and args[2] is C.c_int64
