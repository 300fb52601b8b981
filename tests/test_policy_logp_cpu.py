"""Host side of the fused actors' log-probabilities (d_logp of evg_policy_ppo_logp / evg_policy_rppo_logp): the statement
in tests/ppo_logp.py against an independent float64 enumeration of sequential sampling without replacement, and
the entry points' refusal of a null handle.  The kernels are checked against the statement in
tests/test_gpu_policy_logp.py."""
import itertools

import numpy as np
import pytest

import ppo_logp as pl
import ppo_sampling as ps
from evgsim import _capi


def enumerated_probability(p, tup):
    """P(the ordered draws `tup`) of sequential sampling without replacement from p, in float64 from scratch."""
    p = np.asarray(p, dtype=np.float64)
    left, out = p.sum(), 1.0
    for j in tup:
        out *= p[j] / left
        left -= p[j]
    return out


def dyadic(n, seed):
    """n float32 probabilities that are multiples of 2^-10 summing to 1: every float32 partial sum of them is exact."""
    w = np.random.default_rng(seed).integers(1, 40, n)
    w[-1] += 1024 - w.sum()
    assert w[-1] > 0
    return (w / 1024.0).astype(np.float32)


@pytest.mark.parametrize("draws", [2, 3])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_ordered_tuples_sum_to_one(draws, seed):
    """out_dim 9: exp(sum of logp) over every ordered tuple of distinct indices is the enumerated probability and the
    tuples' probabilities add up to 1, both to 1e-12 (exact float32 sums, so T is the float64 remainder)."""
    p = dyadic(9, seed)
    tuples = list(itertools.permutations(range(9), draws))
    lp = pl.ppo_logp_rows(np.repeat(p[None], len(tuples), 0), np.array(tuples))
    got = np.exp(lp.sum(1))
    want = np.array([enumerated_probability(p, t) for t in tuples])
    assert np.abs(got - want).max() <= 1e-12
    assert abs(got.sum() - 1.0) <= 1e-12


@pytest.mark.parametrize("seed", range(4))
def test_float32_normaliser_against_float64_enumeration(seed):
    """Probabilities as the kernel makes them (float32 quotients of exp(tanh(.)), not exactly summing to 1): each
    tuple's probability differs from the float64 enumeration only by the float32 rounding of the T_k (relative 1e-6)."""
    rng = np.random.default_rng(seed)
    e = np.exp(np.tanh(rng.standard_normal(9))).astype(np.float32)
    p = (e / e.sum(dtype=np.float32)).astype(np.float32)
    tuples = np.array(list(itertools.permutations(range(9), 3)))
    got = np.exp(pl.ppo_logp_rows(np.repeat(p[None], len(tuples), 0), tuples).sum(1))
    want = np.array([enumerated_probability(p, t) for t in tuples])
    assert np.abs(got / want - 1).max() <= 1e-6
    assert abs(got.sum() - 1.0) <= 1e-6


@pytest.mark.parametrize("seed", range(6))
def test_sampler_logp_is_that_of_its_own_draws(seed):
    """ppo_sample_logp: the indices of ppo_sample, T_0 the float32 sum of every probability, each T_k the previous one's
    float32 remainder recomputed in ascending order, every logp in [-7, 0] for tanh-bounded logits over 132 outputs."""
    rng = np.random.default_rng(seed)
    e = np.exp(np.tanh(3 * rng.standard_normal(132))).astype(np.float32)
    p = (e / e.sum(dtype=np.float32)).astype(np.float32)
    u = rng.random(7).astype(np.float32)
    if seed == 0:
        u[3] = np.float32(1 - 2 ** -24)  # the largest uniform: a draw that may run past the float32 prefix sums
    idx, t, lp = pl.ppo_sample_logp(p, u)
    assert np.array_equal(idx, ps.ppo_sample(p, u)) and len(set(idx.tolist())) == 7
    acc = np.float32(0)
    for v in p:
        acc = np.float32(acc + v)
    assert t[0] == acc
    for k in range(1, 7):
        rest = np.float32(0)
        for j in range(132):
            if j not in idx[:k]:
                rest = np.float32(rest + p[j])
        assert t[k] == rest
    assert np.array_equal(lp, np.log(p[idx].astype(np.float64) / t.astype(np.float64)))
    assert (lp <= 0).all() and (lp >= -7).all()


def test_recurrent_one_draw_per_step():
    """rppo_sample_logp: one draw with replacement, T the float32 ascending sum; over every index the exp(logp) add up
    to 1 (dyadic probabilities), and the rows form agrees with the scalar one."""
    p = dyadic(9, 5)
    assert abs(sum(np.exp(pl.rppo_logp_rows(np.repeat(p[None, None], 9, 0).repeat(7, 1), np.tile(np.arange(9)[:, None], 7))[:, 0]))
               - 1.0) <= 1e-12
    rng = np.random.default_rng(7)
    probs = np.empty((5, 7, 132), dtype=np.float32)
    idx = np.empty((5, 7), dtype=np.int64)
    want = np.empty((5, 7))
    for r in range(5):
        for k in range(7):
            e = np.exp(np.tanh(2 * rng.standard_normal(132))).astype(np.float32)
            probs[r, k] = (e / e.sum(dtype=np.float32)).astype(np.float32)
            idx[r, k], t, want[r, k] = pl.rppo_sample_logp(probs[r, k], np.float32(rng.random()))
            assert t == pl.ppo_totals(probs[r, k][None], np.array([[0]]))[0, 0]
    assert np.array_equal(pl.rppo_logp_rows(probs, idx), want)
    assert (want <= 0).all() and (want >= -7).all()


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    return _capi.load()


def test_null_handles_are_refused(lib):
    for fmt in (_capi.OBS_F32, _capi.OBS_I16, _capi.OBS_WIRE):
        assert lib.evg_policy_ppo_logp(None, fmt, None, -1, None, None, None, None, 128, 132, 12, 11, None, None, None, None, None) == -1
        assert lib.evg_policy_rppo_logp(None, fmt, None, -1, None, None, None, None, None, None, 128, 132, 12, 11, None, None, None, None,
                                        None, None, None) == -1
    assert b"null" in lib.evg_last_error()
