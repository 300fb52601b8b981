"""CPU statement of the fused PPO actors' log-probabilities (d_logp of evg_policy_ppo_logp / evg_policy_rppo_logp,
DESIGN.md §4.6 and §4.7), for their tests.  TEST INFRASTRUCTURE ONLY.

Each draw's log(p_j / T_k) in float64 on the float32 operands the kernels use: p_j the probability drawn, T_k the
sampler's own float32 normaliser of draw k (tests/ppo_sampling.py's ppo_sample states the draws themselves).
"""
import numpy as np

from ppo_sampling import ppo_sample


def ppo_sample_logp(probs, u):
    """ppo_sample with what the kernel writes to d_logp: (indices int64 [k], T float32 [k], logp float64 [k]).  T[k] is
    the float32 sum, in ascending j, of the probabilities not chosen before draw k (the normaliser draw k used, also
    when rounding left no j and the largest not-chosen j was taken); logp[k] = log(p[idx[k]] / T[k]) in float64 on those
    float32 operands."""
    p = np.asarray(probs, dtype=np.float32)
    idx = ppo_sample(p, u)
    t = ppo_totals(p[None], idx[None])[0]
    return idx, t, np.log(p[idx].astype(np.float64) / t.astype(np.float64))


def ppo_totals(probs, idx):
    """T of every draw of every row: probs float32 [rows, n], idx int64 [rows, k] (the draws made, in order) -> float32
    [rows, k], draw k's float32 ascending sum of the probabilities not in idx[:, :k] (a chosen entry adds nothing)."""
    p = np.asarray(probs, dtype=np.float32)
    idx = np.asarray(idx, dtype=np.int64)
    rows, n = p.shape
    taken = np.zeros((rows, n), dtype=bool)
    out = np.empty(idx.shape, dtype=np.float32)
    zero = np.float32(0.0)
    for k in range(idx.shape[1]):
        t = np.zeros(rows, dtype=np.float32)
        for j in range(n):
            t += np.where(taken[:, j], zero, p[:, j])
        out[:, k] = t
        taken[np.arange(rows), idx[:, k]] = True
    return out


def ppo_logp_rows(probs, idx):
    """The log-probabilities of the draws idx int64 [rows, k] made without replacement from probs float32 [rows, n]:
    float64 [rows, k], log(p_j / T_k) with ppo_totals' T."""
    p = np.asarray(probs, dtype=np.float32)
    idx = np.asarray(idx, dtype=np.int64)
    pj = np.take_along_axis(p, idx, axis=1).astype(np.float64)
    return np.log(pj / ppo_totals(p, idx).astype(np.float64))


def rppo_logp_rows(probs, idx):
    """The recurrent actor's log-probabilities: probs float32 [rows, 7, n] (step k's distribution), idx int64 [rows, 7]
    (one draw per step, with replacement) -> float64 [rows, 7], log(p_k[j] / T_k) with T_k the float32 ascending sum
    of p_k (what the kernel's draw uses, ppo_sample's T of a single draw)."""
    p = np.asarray(probs, dtype=np.float32)
    t = np.zeros(p.shape[:2], dtype=np.float32)
    for j in range(p.shape[2]):
        t += p[:, :, j]
    pj = np.take_along_axis(p, np.asarray(idx, dtype=np.int64)[:, :, None], axis=2)[:, :, 0].astype(np.float64)
    return np.log(pj / t.astype(np.float64))


def rppo_sample_logp(probs, u):
    """One draw of the recurrent actor from probs float32 [n] with uniform u: (index, T float32, logp float64)."""
    p = np.asarray(probs, dtype=np.float32)
    j = int(ppo_sample(p, [u])[0])
    t = ppo_totals(p[None], np.array([[j]]))[0, 0]
    return j, t, float(np.log(np.float64(p[j]) / np.float64(t)))
