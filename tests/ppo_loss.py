"""CPU statements of PPO's policy loss from the actor's last Linear output (evg_ppo_loss / evg_ppo_loss_grad,
BatchedEvergladesEnv.ppo_loss, DESIGN.md §4.12), for its tests and tools/ppo_loss_time.py.  TEST INFRASTRUCTURE ONLY.

- reference_loss: the float32 statement in the kernel's order (every sum over the n actions is a lane's ascending sum
  over the slots s, element lane + 32 s, then the xor butterfly 16, 8, 4, 2, 1).  numpy's tanh / exp / log are not
  CUDA's, so the kernel is held to the float64 statement within the derived bound, not to this bit for bit.
- loss_float64 / grad_float64: the definition in float64, the gradient written out analytically.
- loss_bound / grad_bound: first-order bounds on |float32 kernel - float64| from the roundings of the kernel's
  operations (tanhf and expf within 2 ulp, logf within 1 ulp, the division and every add and multiply within 1 ulp),
  doubled to cover second-order terms.
- torch_loss: the same loss in plain torch (float32 or float64), for autograd comparisons and the timing tool.

z is float32 [B, n] (K = 1: one distribution, 7 draws without replacement) or [B, 7, n] (K = 7: distribution k serves
draw k, with replacement); idx int64 [B, 7], old_logp float32 [B, 7], adv float32 [B], clip = epsilon in [0, 1).
"""
import numpy as np

DRAWS = 7
U = 2.0 ** -24


def _dists(z):
    """z as [B, K, n] and K."""
    z = np.asarray(z)
    return (z[:, None, :], 1) if z.ndim == 2 else (z, z.shape[1])


def warp_sum(x):
    """float32 [..., n], n <= 256 -> float32 [...]: lane l adds x[l + 32 s] for s = 0..7 in order (0 past n), then
    the butterfly over xor 16, 8, 4, 2, 1 (lane l adds lane l ^ w; both orders give the same float)."""
    x = np.asarray(x, dtype=np.float32)
    n = x.shape[-1]
    xp = np.zeros(x.shape[:-1] + (256,), dtype=np.float32)
    xp[..., :n] = x
    xp = xp.reshape(x.shape[:-1] + (8, 32))
    part = np.zeros(x.shape[:-1] + (32,), dtype=np.float32)
    for s in range(8):
        part = part + xp[..., s, :]
    for w in (16, 8, 4, 2, 1):
        part = part[..., :w] + part[..., w:2 * w]
    return part[..., 0]


def _counted(idx, n):
    """bool [B, 7, n]: whether element i counts in T_k for K = 1 (not among idx[:, :k])."""
    B = idx.shape[0]
    c = np.ones((B, DRAWS, n), dtype=bool)
    for k in range(1, DRAWS):
        c[:, k] = c[:, k - 1]
        c[np.arange(B), k, idx[:, k - 1]] = False
    return c


def _clip_bounds(clip):
    one, e = np.float32(1), np.float32(clip)
    return one - e, one + e


def reference_loss(z, idx, old_logp, adv, clip):
    """The float32 statement: (surr [B], ent [B], logp [B, 7], ratio [B])."""
    f32 = np.float32
    z3, K = _dists(np.asarray(z, dtype=f32))
    idx = np.asarray(idx, dtype=np.int64)
    B, _, n = z3.shape
    y = np.tanh(z3).astype(f32)
    e = np.exp(y).astype(f32)
    S = warp_sum(e)
    L = np.log(S).astype(f32)
    p = (e / S[..., None]).astype(f32)
    lp = (y - L[..., None]).astype(f32)
    H = -warp_sum((p * lp).astype(f32))
    if K == 1:
        T = warp_sum(np.where(_counted(idx, n), p, f32(0)))  # [B, 7]
        yj = np.take_along_axis(y[:, 0], idx, axis=1)
        Lk = np.repeat(L, DRAWS, axis=1)
    else:
        T = warp_sum(p)
        yj = np.take_along_axis(y, idx[:, :, None], axis=2)[:, :, 0]
        Lk = L
    logp = ((yj - Lk).astype(f32) - np.log(T).astype(f32)).astype(f32)
    ell, ell_old, hs = np.zeros(B, f32), np.zeros(B, f32), np.zeros(B, f32)
    old = np.asarray(old_logp, dtype=f32)
    for k in range(DRAWS):
        ell = ell + logp[:, k]
        ell_old = ell_old + old[:, k]
    for k in range(K):
        hs = hs + H[:, k]
    ratio = np.exp(ell - ell_old).astype(f32)
    lo, hi = _clip_bounds(clip)
    A = np.asarray(adv, dtype=f32)
    surr = -np.minimum(ratio * A, np.clip(ratio, lo, hi) * A)
    return surr.astype(f32), (hs / f32(K)).astype(f32), logp, ratio


def _float64_parts(z, idx):
    z3, K = _dists(np.asarray(z, dtype=np.float64))
    idx = np.asarray(idx, dtype=np.int64)
    B, _, n = z3.shape
    y = np.tanh(z3)
    e = np.exp(y)
    p = e / e.sum(-1, keepdims=True)
    lp = y - np.log(e.sum(-1, keepdims=True))
    H = -(p * lp).sum(-1)  # [B, K]
    if K == 1:
        cnt = _counted(idx, n)
        T = (p[:, 0][:, None, :] * cnt).sum(-1)
        lpj = np.take_along_axis(lp[:, 0], idx, axis=1)
    else:
        cnt = np.ones((B, DRAWS, n), dtype=bool)
        T = p.sum(-1)
        lpj = np.take_along_axis(lp, idx[:, :, None], axis=2)[:, :, 0]
    return dict(K=K, n=n, y=y, p=p, lp=lp, H=H, T=T, cnt=cnt, logp=lpj - np.log(T))


def loss_float64(z, idx, old_logp, adv, clip):
    """The definition in float64 on the same inputs: (surr, ent, logp, ratio)."""
    q = _float64_parts(z, idx)
    ratio = np.exp(q["logp"].sum(-1) - np.asarray(old_logp, dtype=np.float64).sum(-1))
    lo, hi = (np.float64(v) for v in _clip_bounds(clip))
    A = np.asarray(adv, dtype=np.float64)
    surr = -np.minimum(ratio * A, np.clip(ratio, lo, hi) * A)
    return surr, q["H"].mean(-1), q["logp"], ratio


def clipped(ratio, adv, clip):
    """Where the surrogate's gradient is 0: the clipped branch is the minimum (ties take the unclipped branch)."""
    lo, hi = (np.float64(v) for v in _clip_bounds(clip))
    A = np.asarray(adv, dtype=np.float64)
    r = np.asarray(ratio, dtype=np.float64)
    return ((A > 0) & (r > hi)) | ((A < 0) & (r < lo))


def grad_float64(z, idx, adv, ratio, clip, g_surr=None, g_ent=None):
    """d(g_surr . surr + g_ent . ent)/dz in float64, with the branch and the factor r taken from `ratio` (pass the
    kernel's ratio to follow its branch, or loss_float64's): float64 of z's shape."""
    q = _float64_parts(z, idx)
    K, n, p, y = q["K"], q["n"], q["p"], q["y"]
    B = p.shape[0]
    idx = np.asarray(idx, dtype=np.int64)
    A = np.asarray(adv, dtype=np.float64)
    r = np.asarray(ratio, dtype=np.float64)
    gs = np.zeros(B) if g_surr is None else np.asarray(g_surr, dtype=np.float64)
    ge = np.zeros(B) if g_ent is None else np.asarray(g_ent, dtype=np.float64)
    G = np.where(clipped(r, A, clip), 0.0, -A * r * gs)
    if K == 1:
        c = np.zeros((B, 1, n))
        for k in range(DRAWS):
            c[np.arange(B), 0, idx[:, k]] += 1
        Q = (q["cnt"] / q["T"][:, :, None]).sum(1)[:, None, :]  # sum of 1 / T_k over the draws that count i
    else:
        c = np.zeros((B, DRAWS, n))
        c[np.arange(B)[:, None], np.arange(DRAWS)[None, :], idx] = 1
        Q = 1.0 / q["T"][:, :, None]
    dy = G[:, None, None] * (c - p * Q) - (ge / K)[:, None, None] * p * (q["lp"] + q["H"][:, :, None])
    dz = (1 - y * y) * dy
    return dz[:, 0] if np.asarray(z).ndim == 2 else dz


def _bound_parts(z, idx, old_logp):
    """The float64 values and the first-order error terms shared by the two bounds."""
    q = _float64_parts(z, idx)
    n = q["n"]
    D = -(-n // 32) + 5                 # additions on a sum's longest path: the lane's slots, then 5 butterfly steps
    e_S = (8 + D) * U                   # relative: e from tanhf (4u absolute in y) and expf (2 ulp), then the sum
    e_p = 8 * U + e_S + 2 * U           # relative
    L = q["lp"] - q["y"]                # -log S
    e_L = e_S + 2 * U * np.abs(L)       # absolute, logf within 1 ulp
    e_lp = 4 * U + e_L + 2 * U * np.abs(q["lp"])
    e_T = e_p + D * U                   # relative
    e_logT = e_T + 2 * U * np.abs(np.log(q["T"]))
    if q["K"] == 1:
        e_lpj = np.max(e_lp[:, 0], axis=-1, keepdims=True)
    else:
        e_lpj = np.max(e_lp, axis=-1)
    e_logp = e_lpj + e_logT + 2 * U * np.abs(q["logp"])
    old = np.asarray(old_logp, dtype=np.float64)
    e_ell = e_logp.sum(-1) + 2 * U * DRAWS * (np.abs(q["logp"]).sum(-1) + np.abs(old).sum(-1))
    d = q["logp"].sum(-1) - old.sum(-1)
    e_r = e_ell + 2 * U * np.abs(d) + 4 * U     # relative error of the ratio
    e_H = np.max(e_lp, axis=-1) + (e_p + (D + 4) * U) * (q["p"] * np.abs(q["lp"])).sum(-1)  # [B, K]
    return q, dict(e_p=e_p, e_lp=e_lp, e_T=e_T, e_logp=e_logp, e_r=e_r, e_H=e_H, D=D)


def loss_bound(z, idx, old_logp, adv, clip):
    """Bounds on |kernel - loss_float64| for (surr, ent, logp, ratio)."""
    surr, ent, logp, ratio = loss_float64(z, idx, old_logp, adv, clip)
    q, e = _bound_parts(z, idx, old_logp)
    K = q["K"]
    A = np.abs(np.asarray(adv, dtype=np.float64))
    b_ratio = ratio * e["e_r"]
    b_surr = A * b_ratio + 4 * U * np.abs(surr)
    b_ent = e["e_H"].mean(-1) + 2 * U * (K + 1) * np.abs(q["H"]).sum(-1) / K
    return 2 * b_surr, 2 * b_ent, 2 * e["e_logp"], 2 * b_ratio


def grad_bound(z, idx, adv, ratio, clip, old_logp, g_surr=None, g_ent=None):
    """Bound on |kernel dz - grad_float64(z, idx, adv, ratio, ...)|, ratio being the one whose branch both follow."""
    q, e = _bound_parts(z, idx, old_logp)
    K, n, p, y = q["K"], q["n"], q["p"], q["y"]
    B = p.shape[0]
    idx = np.asarray(idx, dtype=np.int64)
    A = np.asarray(adv, dtype=np.float64)
    r = np.asarray(ratio, dtype=np.float64)
    gs = np.zeros(B) if g_surr is None else np.abs(np.asarray(g_surr, dtype=np.float64))
    ge = np.zeros(B) if g_ent is None else np.abs(np.asarray(g_ent, dtype=np.float64))
    G = np.where(clipped(r, A, clip), 0.0, np.abs(A * r) * gs)[:, None, None]
    e_G = (e["e_r"] + 4 * U)[:, None, None]
    if K == 1:
        c = np.zeros((B, 1, n))
        for k in range(DRAWS):
            c[np.arange(B), 0, idx[:, k]] += 1
        Q = (q["cnt"] / q["T"][:, :, None]).sum(1)[:, None, :]
        e_Q = e["e_T"] + (2 + 2 * DRAWS) * U
    else:
        c = np.zeros((B, DRAWS, n))
        c[np.arange(B)[:, None], np.arange(DRAWS)[None, :], idx] = 1
        Q = 1.0 / q["T"][:, :, None]
        e_Q = e["e_T"] + 2 * U
    pQ = p * Q
    t1 = np.abs(c - pQ)
    b1 = G * ((e["e_p"] + e_Q + 2 * U) * pQ + 2 * U * t1) + G * e_G * t1 + 2 * U * G * t1
    h = np.abs(q["lp"] + q["H"][:, :, None])
    Ek = (ge / K)[:, None, None]
    b2 = Ek * p * (e["e_lp"] + e["e_H"][:, :, None] + 2 * U * h + (e["e_p"] + 6 * U) * h)
    v = np.abs(G * t1) + Ek * p * h
    w = 1 - y * y
    b = w * (b1 + b2 + 2 * U * v) + v * 10 * U + 2 * U * w * v
    b = 2 * b
    return b[:, 0] if np.asarray(z).ndim == 2 else b


def torch_loss(z, idx, old_logp, adv, clip):
    """The loss in plain torch, in z's dtype: (surr, ent, logp, ratio), differentiable through autograd.  lo and hi are
    the kernel's float32 fl(1 - clip) and fl(1 + clip)."""
    import torch
    y = torch.tanh(z)
    p = torch.softmax(y, dim=-1)
    lo, hi = (float(v) for v in _clip_bounds(clip))  # float32 values, exact in z's dtype
    if z.dim() == 2:
        keep = torch.ones_like(p)
        logps = []
        for k in range(DRAWS):
            j = idx[:, k:k + 1]
            T = (p * keep).sum(-1)
            logps.append(torch.log(p.gather(1, j)[:, 0]) - torch.log(T))
            keep = keep.scatter(1, j, 0.0)
        logp = torch.stack(logps, dim=1)
        ent = -(p * torch.log(p)).sum(-1)
    else:
        T = p.sum(-1)
        logp = torch.log(p.gather(2, idx[:, :, None])[:, :, 0]) - torch.log(T)
        ent = -(p * torch.log(p)).sum(-1).mean(-1)
    ratio = torch.exp(logp.sum(-1) - old_logp.to(z.dtype).sum(-1))
    A = adv.to(z.dtype)
    surr = -torch.min(ratio * A, torch.clamp(ratio, lo, hi) * A)
    return surr, ent, logp, ratio
