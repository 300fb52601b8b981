"""CPU statement of evg_policy_ppo's action sampling (DESIGN.md §4.6), for the tests of the fused PPO actor.
TEST INFRASTRUCTURE ONLY.

policy_uniforms: the tape's domain 3 (DESIGN.md §2) — the 7 uniforms of one (match, turn, player, episode), from the
same Philox4x32-10 as oracle/tape.py.
ppo_sample: PPOAgent.get_action's 7 draws without replacement (agents/PPO/PPOAgent.py:122-127) as the kernel makes
them from those uniforms, in float32 scalar arithmetic, bit for bit.
"""
import numpy as np

from oracle.tape import MASK, philox4x32

DOMAIN_POLICY_SAMPLE = 3  # after oracle/tape.py's 0 combat, 1 random_actions, 2 SwarmAgent


def policy_uniforms(seed: int, env: int, turn: int, player: int, episode: int = 0):
    """The 7 float32 uniforms in [0, 1) of evg_policy_ppo's draws for (global match id, turn, player, episode): words
    0..3 of the block with c2 = player, 4..7 of c2 = player | 1<<8 (domain 3), u_k = (w_k >> 8) * 2^-24."""
    key = (seed & MASK, (seed >> 32) & MASK)
    c3 = DOMAIN_POLICY_SAMPLE | (episode & 0xFFFFFF) << 8
    w = philox4x32((env & MASK, turn & MASK, player & MASK, c3), key) + philox4x32((env & MASK, turn & MASK, (player | 1 << 8) & MASK, c3), key)
    return np.array([(x >> 8) * 2.0 ** -24 for x in w[:7]], dtype=np.float32)


def ppo_sample(probs, u):
    """Distinct indices (one per uniform in u, float32) drawn from `probs` (float32 [n]) without replacement.  Draw k:
    T = float32 sum, in ascending j, of the probabilities not chosen yet; x = u[k] * T; walk the not-chosen j in
    ascending order accumulating c += p[j] in float32 and take the first j with x < c; if rounding leaves none, the
    largest j not chosen yet.  The distribution is that of sequential sampling without replacement
    (torch.multinomial(probs, 7, replacement=False)); the stream is not torch's."""
    p = [np.float32(v) for v in np.asarray(probs, dtype=np.float32)]
    chosen, taken = [], set()
    for k in range(len(u)):
        t = np.float32(0.0)
        for j, v in enumerate(p):
            if j not in taken:
                t = np.float32(t + v)
        x = np.float32(np.float32(u[k]) * t)
        c = np.float32(0.0)
        sel = None
        for j, v in enumerate(p):
            if j in taken:
                continue
            c = np.float32(c + v)
            if x < c:
                sel = j
                break
        if sel is None:
            sel = max(j for j in range(len(p)) if j not in taken)
        chosen.append(sel)
        taken.add(sel)
    return np.array(chosen, dtype=np.int64)


def ppo_sample_rows(probs, u):
    """ppo_sample of every row at once: probs float32 [rows, n], u float32 [rows, k] -> int64 [rows, k].  The same
    float32 sums in the same order, each row's vectorised across the rows (a chosen entry adds nothing: x + 0 = x)."""
    p = np.asarray(probs, dtype=np.float32)
    u = np.asarray(u, dtype=np.float32)
    rows, n = p.shape
    taken = np.zeros((rows, n), dtype=bool)
    out = np.empty(u.shape, dtype=np.int64)
    zero = np.float32(0.0)
    for k in range(u.shape[1]):
        t = np.zeros(rows, dtype=np.float32)
        for j in range(n):
            t += np.where(taken[:, j], zero, p[:, j])
        x = u[:, k] * t
        c = np.zeros(rows, dtype=np.float32)
        sel = np.full(rows, -1, dtype=np.int64)
        for j in range(n):
            c += np.where(taken[:, j], zero, p[:, j])
            sel[(sel < 0) & ~taken[:, j] & (x < c)] = j
        last = n - 1 - np.argmax(~taken[:, ::-1], axis=1)
        sel = np.where(sel < 0, last, sel)
        taken[np.arange(rows), sel] = True
        out[:, k] = sel
    return out
