"""Reference of the recurrent actor's update operation (evg_rppo_train_forward / _backward, FusedRPPO.evaluate;
include/evgsim.h states the definition).

- ``forward64`` / ``backward64``: the definition and its analytic backward in float64.  ``rnd`` is applied where the
  kernel rounds an MMA operand (x, h_{k-1} for W_hh, h_k for W3, dgh_k for the carry, and the weights by the caller), so
  with ``rnd = bf16`` they state what the kernel computes up to float32 accumulation and transcendentals, and with the
  identity they are the textbook GRU.
- ``torch_reference``: torch.nn.GRU + Linear in float64 autograd, the truth the analytic backward is checked against.
- ``forward32``: the float32 statement in the kernel's order, from x.
- ``step_bound``: a first-order bound on one float32 step of the kernel against ``forward64`` from the same h_{k-1}.
"""
import numpy as np

K = 7
U32 = 2.0 ** -24


def bf16(a):
    """Round to bf16 (nearest even) and back, in the input's precision (float32 rounding first for float64 input)."""
    a32 = np.ascontiguousarray(a, dtype=np.float32)
    u = a32.view(np.uint32).astype(np.uint64)
    r = (((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16).astype(np.uint32).view(np.float32)
    return r.astype(np.asarray(a).dtype if np.asarray(a).dtype == np.float64 else np.float32)


def _ident(a):
    return a


def _sig(v):
    return 1.0 / (1.0 + np.exp(-v))


def forward64(x, h0, w, rnd=_ident):
    """x, h0 [R, L]; w = (w_ih, b_ih, w_hh, b_hh, w3, b3) -> (z [R, 7, out], h [R, 7, L], gates: list of (r, u, n, c))."""
    w_ih, b_ih, w_hh, b_hh, w3, b3 = (np.asarray(a, dtype=np.float64) for a in w)
    L = x.shape[1]
    gi = rnd(np.asarray(x, np.float64)) @ w_ih.T
    h = np.asarray(h0, dtype=np.float64)
    zs, hs, gates = [], [], []
    for _ in range(K):
        gh = rnd(h) @ w_hh.T
        r = _sig(gi[:, :L] + gh[:, :L] + b_ih[:L] + b_hh[:L])
        u = _sig(gi[:, L:2 * L] + gh[:, L:2 * L] + b_ih[L:2 * L] + b_hh[L:2 * L])
        c = gh[:, 2 * L:] + b_hh[2 * L:]
        n = np.tanh(gi[:, 2 * L:] + b_ih[2 * L:] + r * c)
        gates.append((r, u, n, c))
        h = (1 - u) * n + u * h
        hs.append(h)
        zs.append(rnd(h) @ w3.T + b3)
    return np.stack(zs, 1), np.stack(hs, 1), gates


def backward64(x, h0, w, dz, rnd=_ident):
    """The analytic backward of include/evgsim.h from dz [R, 7, out] -> (dx, dw_ih, db_ih, dw_hh, db_hh, dw3, db3)."""
    w_ih, b_ih, w_hh, b_hh, w3, b3 = (np.asarray(a, dtype=np.float64) for a in w)
    dz = np.asarray(dz, dtype=np.float64)
    _, hs, gates = forward64(x, h0, w, rnd)
    h_prev = np.concatenate([np.asarray(h0, np.float64)[:, None], hs[:, :K - 1]], 1)
    carry = 0.0
    s = 0.0
    dw_hh = np.zeros_like(w_hh)
    db_hh = np.zeros_like(b_hh)
    for k in range(K - 1, -1, -1):
        r, u, n, c = gates[k]
        g = dz[:, k] @ w3 + carry
        dn = g * (1 - u)
        da_n = dn * (1 - n * n)
        da_u = g * (h_prev[:, k] - n) * u * (1 - u)
        da_r = da_n * c * r * (1 - r)
        dgi = np.concatenate([da_r, da_u, da_n], 1)
        dgh = np.concatenate([da_r, da_u, da_n * r], 1)
        s = s + dgi
        dw_hh += dgh.T @ rnd(h_prev[:, k])
        db_hh += dgh.sum(0)
        carry = g * u + rnd(dgh) @ w_hh
    xr = rnd(np.asarray(x, np.float64))
    dw3 = np.einsum("rko,rkl->ol", dz, rnd(hs))
    return s @ w_ih, s.T @ xr, s.sum(0), dw_hh, db_hh, dw3, dz.sum((0, 1))


def torch_reference(x, h0, w, dz):
    """torch.nn.GRU + Linear in float64 autograd on the given operands: (z, (dx, dw_ih, db_ih, dw_hh, db_hh, dw3, db3))."""
    import torch
    w_ih, b_ih, w_hh, b_hh, w3, b3 = w
    L = np.shape(x)[1]
    gru = torch.nn.GRU(L, L).double()
    lin = torch.nn.Linear(L, np.shape(w3)[0]).double()
    with torch.no_grad():
        for p, a in zip((gru.weight_ih_l0, gru.bias_ih_l0, gru.weight_hh_l0, gru.bias_hh_l0, lin.weight, lin.bias), w):
            p.copy_(torch.from_numpy(np.asarray(a, np.float64)))
    xt = torch.from_numpy(np.asarray(x, np.float64)).requires_grad_(True)
    out, _ = gru(xt.unsqueeze(0).expand(K, -1, -1), torch.from_numpy(np.asarray(h0, np.float64)).unsqueeze(0))
    z = lin(out).permute(1, 0, 2)
    z.backward(torch.from_numpy(np.asarray(dz, np.float64)))
    grads = (xt.grad, gru.weight_ih_l0.grad, gru.bias_ih_l0.grad, gru.weight_hh_l0.grad, gru.bias_hh_l0.grad, lin.weight.grad, lin.bias.grad)
    return z.detach().numpy(), tuple(g.numpy() for g in grads)


def forward32(x, h0, w):
    """The float32 statement in the kernel's order, from x: bf16 operands, float32 products, X W_ir^T + H W_hr^T summed
    before the pre-summed bias, h in float32 -> (z [R, 7, out], h [R, 7, L]).  Its float32 products sum in numpy's
    order, not the tensor core's: it agrees with the kernel to the bound, not bit for bit."""
    f = np.float32
    w_ih, b_ih, w_hh, b_hh, w3, b3 = (np.asarray(a, dtype=f) for a in w)
    L = x.shape[1]
    gi = (bf16(np.asarray(x, f)) @ bf16(w_ih).T).astype(f)
    h = np.asarray(h0, dtype=f)
    zs, hs = [], []
    for _ in range(K):
        gh = (bf16(h) @ bf16(w_hh).T).astype(f)
        r = (f(1) / (f(1) + np.exp(-((gi[:, :L] + gh[:, :L]) + (b_ih[:L] + b_hh[:L]))))).astype(f)
        u = (f(1) / (f(1) + np.exp(-((gi[:, L:2 * L] + gh[:, L:2 * L]) + (b_ih[L:2 * L] + b_hh[L:2 * L]))))).astype(f)
        n = np.tanh((gi[:, 2 * L:] + b_ih[2 * L:]) + r * (gh[:, 2 * L:] + b_hh[2 * L:])).astype(f)
        h = ((f(1) - u) * n + u * h).astype(f)
        hs.append(h)
        zs.append(((bf16(h) @ bf16(w3).T).astype(f) + b3).astype(f))
    return np.stack(zs, 1), np.stack(hs, 1)


def step_bound(x, h_prev, w):
    """Per-element bound on one float32 step of the kernel (h_k and z_k) against forward64 run one step from the same
    h_{k-1}, with bf16 operands.  A float32 dot product of m terms is within gamma_m sum |a_i b_i| (gamma_m = m u / (1 - m u),
    any summation order); the kernel adds two of them for r and u and the bias afterwards.  Through sigmoid (slope <= 1/4)
    and tanh (slope <= 1) the pre-activation error passes at most unchanged; expf, tanhf and the reciprocal add a few ulp
    (8 u on each gate, generously), and h' = (1 - u) n + u h four roundings.  The bound is first order: the terms it drops
    are below u^2 times the same sums.
    Returns the bound on h_k [R, L]; z_bound gives z_k's from the kernel's own h_k."""
    w_ih, b_ih, w_hh, b_hh, w3, b3 = (np.abs(np.asarray(a, dtype=np.float64)) for a in w)
    L = x.shape[1]
    ax, ah = np.abs(bf16(np.asarray(x, np.float64))), np.abs(bf16(np.asarray(h_prev, np.float64)))
    gam = lambda m: m * U32 / (1 - m * U32)  # noqa: E731
    ei = ax @ w_ih.T * gam(L)
    eh = ah @ w_hh.T * gam(L)
    pre = ax @ w_ih.T + ah @ w_hh.T + b_ih + b_hh
    e_rz = ei[:, :2 * L] + eh[:, :2 * L] + 3 * U32 * pre[:, :2 * L]  # products, their sum and the bias add
    e_r = 0.25 * e_rz[:, :L] + 8 * U32
    e_u = 0.25 * e_rz[:, L:] + 8 * U32
    c_abs = (ah @ w_hh.T)[:, 2 * L:] + b_hh[2 * L:]
    e_n = ei[:, 2 * L:] + eh[:, 2 * L:] + e_r * c_abs + 4 * U32 * (c_abs + (ax @ w_ih.T)[:, 2 * L:] + b_ih[2 * L:]) + 8 * U32
    e_h = e_n + e_u * (1 + np.abs(h_prev)) + 4 * U32 * (1 + np.abs(h_prev))
    return e_h


def z_bound(h_k, w3, b3):
    """Bound on z_k = fl(bf16(h_k) bf16(W3)^T) + b3 against float64 of the same bf16 operands."""
    ah = np.abs(bf16(np.asarray(h_k, np.float64)))
    a3 = np.abs(bf16(np.asarray(w3, np.float64)))
    m = a3.shape[1]
    return ah @ a3.T * (m * U32 / (1 - m * U32)) + U32 * (ah @ a3.T + np.abs(b3))


def pack_wht(w_hh):
    """The transposed image evg_rppo_train_pack writes (d_wht_img), built on the host: gate g's block holds
    W_hg^T = w_hh[g L:(g + 1) L].T as an [Lp x Ka] K-major swizzled image."""
    from evgsim import policy
    w_hh = np.asarray(w_hh, dtype=np.float32)
    L = w_hh.shape[1]
    lp, ka = -(-L // 16) * 16, -(-L // 64) * 64
    return np.concatenate([policy._image(w_hh[g * L:(g + 1) * L].T, lp, ka) for g in range(3)])
