"""CPU statements of PPO's advantages and returns (evg_gae, BatchedEvergladesEnv.gae, DESIGN.md §4.11), for their tests.
TEST INFRASTRUCTURE ONLY.

reference_gae is the kernel's float32 recurrence operation by operation (numpy rounds each float32 operation on its own,
like the kernel's __fmul_rn / __fadd_rn / __fsub_rn), so the kernel must equal it bit for bit.  gae_float64 is the
textbook form in float64, multiplying by (1 - d); gae_bound is the derived bound on the distance between the two.
"""
import numpy as np

U = 2.0 ** -24 + 2.0 ** -53  # float32's unit roundoff, plus float64's for the reference the kernel is compared with


def _mask(done, like):
    d = np.asarray(done).astype(bool)
    return d.reshape(d.shape + (1,) * (like.ndim - d.ndim))


def reference_gae(values, reward, done, gamma, lam):
    """values float32 [T+1, M, ...], reward float32 [T, M, ...] (the same columns), done [T, M] (non-zero = done) ->
    (adv, ret) float32 [T, M, ...]: include/evgsim.h's recurrence, gl = fl(gamma * lam), backward from A_T = 0."""
    v = np.asarray(values, dtype=np.float32)
    r = np.asarray(reward, dtype=np.float32)
    g, gl = np.float32(gamma), np.float32(gamma) * np.float32(lam)
    zero = np.float32(0.0)
    adv, ret = np.empty_like(r), np.empty_like(r)
    a = np.zeros_like(v[0])
    with np.errstate(over="ignore", invalid="ignore"):
        for t in range(r.shape[0] - 1, -1, -1):
            d = _mask(done[t], v[t])
            nv = np.where(d, zero, v[t + 1])
            na = np.where(d, zero, a)
            delta = (r[t] + g * nv) - v[t]
            a = delta + gl * na
            adv[t], ret[t] = a, a + v[t]
    return adv, ret


def gae_float64(values, reward, done, gamma, lam):
    """The textbook GAE in float64, with the float32 gamma and lam the kernel is given: delta_t = r_t + gamma V_{t+1}
    (1 - d_t) - V_t, A_t = delta_t + gamma lam (1 - d_t) A_{t+1}, R_t = A_t + V_t."""
    v = np.asarray(values, dtype=np.float64)
    r = np.asarray(reward, dtype=np.float64)
    g, lm = float(np.float32(gamma)), float(np.float32(lam))
    adv, ret = np.empty_like(r), np.empty_like(r)
    a = np.zeros_like(v[0])
    for t in range(r.shape[0] - 1, -1, -1):
        nd = 1.0 - _mask(done[t], v[t])
        a = r[t] + g * v[t + 1] * nd - v[t] + g * lm * nd * a
        adv[t], ret[t] = a, a + v[t]
    return adv, ret


def gae_bound(values, reward, done, gamma, lam):
    """Per element (adv_bound, ret_bound), float64 [T, M, ...]: how far the float32 recurrence can lie from
    gae_float64 on the same float32 inputs.

    With u = 2^-24 and every float32 operation fl(x) = x (1 + e), |e| <= u, the kernel's errors at turn t are, for
    p = gamma nv, s = r + p, delta = s - V, q = gl na (gl = gamma lam (1 + e_g)), A = delta + q, R = A + V, and E_{t+1}
    the error carried in A_{t+1}:
        |p^ - p| <= u|p|,  |s^ - s| <= (1 + u)|p^ - p| + u|s|,  |delta^ - delta| <= (1 + u)|s^ - s| + u|delta|,
        |q^ - q| <= gamma lam ((2u + u^2)|na| + (1 + u)^2 E_{t+1}),
        E_t = |A^ - A| <= (1 + u)(|delta^ - delta| + |q^ - q|) + u|A|,   |R^ - R| <= (1 + u) E_t + u|R|.
    Collecting terms with c = (1 + u)^3 >= every product of (1 + u) factors above:
        E_t <= c u (|p| + |s| + |delta| + 3 gamma lam |na| + |A_t|) + c gamma lam E_{t+1}   (na = 0 and no carry if d_t),
    so a turn k steps before t weighs (c gamma lam)^k: a few roundings per turn, weighted by (gamma lam)^k.  gae_float64
    runs the same operations in the same order, so the same bound holds for it with u = 2^-53; the two bounds together are
    at most this one with u = 2^-24 + 2^-53 (U), which is what is returned, on the float64 evaluation's magnitudes."""
    v = np.asarray(values, dtype=np.float64)
    r = np.asarray(reward, dtype=np.float64)
    g, lm = float(np.float32(gamma)), float(np.float32(lam))
    gl, c = g * lm, (1.0 + U) ** 3
    eb, rb = np.empty_like(r), np.empty_like(r)
    a = np.zeros_like(v[0])
    e = np.zeros_like(v[0])
    for t in range(r.shape[0] - 1, -1, -1):
        nd = 1.0 - _mask(done[t], v[t])
        na = nd * a
        p = g * v[t + 1] * nd
        s = r[t] + p
        delta = s - v[t]
        a = delta + gl * na
        e = c * U * (np.abs(p) + np.abs(s) + np.abs(delta) + 3.0 * gl * np.abs(na) + np.abs(a)) + c * gl * nd * e
        eb[t], rb[t] = e, (1.0 + U) * e + U * np.abs(a + v[t])
    return eb, rb
