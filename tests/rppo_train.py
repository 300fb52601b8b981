"""Reference of the recurrent actor's update operation (evg_rppo_train_forward / _backward, FusedRPPO.evaluate;
include/evgsim.h states the definition).

- ``forward64`` / ``backward64``: the definition and its analytic backward in float64.  ``rnd`` is applied where the
  kernel rounds an MMA operand (x, h_{k-1} for W_hh, h_k for W3, dgh_k for the carry, and the weights by the caller), so
  with ``rnd = bf16`` they state what the kernel computes up to float32 accumulation and transcendentals, and with the
  identity they are the textbook GRU.
- ``torch_reference``: torch.nn.GRU + Linear in float64 autograd, the truth the analytic backward is checked against.
- ``forward32``: the float32 statement in the kernel's order, from x.
- ``gate_bounds`` / ``step_bound``: first-order bounds on the float32 gates and on one float32 step of the kernel
  against ``forward64`` from the same h_{k-1}.
- ``backward32``: the backward's float32 statement in the kernel's order, with BACKWARD_MUTANTS, its plausible defects.
- ``backward_step_bound`` / ``s_bound`` / ``backward_ratios``: a first-order bound on each backward step (dgh_k,
  g_{k-1}) and on S against float64, each step evaluated from the kernel's own inputs to it.
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


def _gamma(m):
    return m * U32 / (1 - m * U32)


def gate_bounds(x, h_prev, w):
    """Per-element bounds (e_r, e_u, e_n, e_c), each [R, L], on the kernel's float32 gates r, u, n and c = W_hn H + b_hn
    of one step against forward64's from the same h_{k-1}, with bf16 operands.  A float32 dot product of m terms is within
    gamma_m sum |a_i b_i| (gamma_m = m u / (1 - m u), u = 2^-24, any summation order); the kernel adds two of them for r
    and u and the bias afterwards.  Through sigmoid (slope <= 1/4) and tanh (slope <= 1) the pre-activation error passes
    at most unchanged.  expf and tanhf are within 2 ulp (CUDA Programming Guide, single-precision maximum ulp errors; the
    library is built without fast-math) and __frcp_rn is correctly rounded, so sigmoid = __frcp_rn(1 + expf(-v)) is
    within 6 u relative and tanhf within 4 u of its value: 8 u on each gate covers both.  c is one dot product and one
    bias add.  The bounds are first order: the terms they drop are below u^2 times the same sums."""
    w_ih, b_ih, w_hh, b_hh = (np.abs(np.asarray(a, dtype=np.float64)) for a in w[:4])
    L = x.shape[1]
    ax, ah = np.abs(bf16(np.asarray(x, np.float64))), np.abs(bf16(np.asarray(h_prev, np.float64)))
    ei = ax @ w_ih.T * _gamma(L)
    eh = ah @ w_hh.T * _gamma(L)
    pre = ax @ w_ih.T + ah @ w_hh.T + b_ih + b_hh
    e_rz = ei[:, :2 * L] + eh[:, :2 * L] + 3 * U32 * pre[:, :2 * L]  # products, their sum and the bias add
    e_r = 0.25 * e_rz[:, :L] + 8 * U32
    e_u = 0.25 * e_rz[:, L:] + 8 * U32
    c_abs = (ah @ w_hh.T)[:, 2 * L:] + b_hh[2 * L:]
    e_n = ei[:, 2 * L:] + eh[:, 2 * L:] + e_r * c_abs + 4 * U32 * (c_abs + (ax @ w_ih.T)[:, 2 * L:] + b_ih[2 * L:]) + 8 * U32
    e_c = eh[:, 2 * L:] + U32 * c_abs
    return e_r, e_u, e_n, e_c


def step_bound(x, h_prev, w):
    """Per-element bound on one float32 step of the kernel (h_k and z_k) against forward64 run one step from the same
    h_{k-1}, with bf16 operands: gate_bounds' e_n and e_u through h' = (1 - u) n + u h, and its four roundings.
    Returns the bound on h_k [R, L]; z_bound gives z_k's from the kernel's own h_k."""
    _, e_u, e_n, _ = gate_bounds(x, h_prev, w)
    return e_n + e_u * (1 + np.abs(h_prev)) + 4 * U32 * (1 + np.abs(h_prev))


def z_bound(h_k, w3, b3):
    """Bound on z_k = fl(bf16(h_k) bf16(W3)^T) + b3 against float64 of the same bf16 operands."""
    ah = np.abs(bf16(np.asarray(h_k, np.float64)))
    a3 = np.abs(bf16(np.asarray(w3, np.float64)))
    m = a3.shape[1]
    return ah @ a3.T * (m * U32 / (1 - m * U32)) + U32 * (ah @ a3.T + np.abs(b3))


BACKWARD_MUTANTS = ["dgh_n_without_r", "carry_g", "carry_g_1mu", "dau_n_minus_h", "dar_without_c", "dtanh_1mn",
                    "s_sums_dgh", "carry_untransposed", "carry_last_group_dropped", "reads_h_k", "dgh_rz"]


def _sig32(v):
    f = np.float32
    with np.errstate(over="ignore"):  # expf(120) = inf by design in the dyadic network: 1 / (1 + inf) = 0
        return (f(1) / (f(1) + np.exp(-v))).astype(f)


def carry_columns(L, last_group_dropped=False):
    """The carry's 3L operand columns (gate g's unit j at g L + j) as the kernel stages them: 64-column atoms q = gate
    q // ka, units 64 (q % ka) .., in groups of four.  With last_group_dropped, a mask without the last group's atoms
    (L > 64; at L <= 64 there is one group and the mask keeps it)."""
    ka = -(-L // 64)
    keep = np.ones(3 * L, dtype=bool)
    if last_group_dropped and L > 64:
        first = 4 * ((3 * ka - 1) // 4)
        for q in range(first, 3 * ka):
            g, c = divmod(q, ka)
            keep[g * L + 64 * c:g * L + min(64 * c + 64, L)] = False
    return keep


def backward32(x, h0, h, w, G, mutant=None):
    """The kernel's float32 statement of the backward (evg_rppo_train_kernel<true>), in its order, step k = 7 .. 1:
    the gates recomputed from bf16(x) and bf16(h_{k-1}) as forward32 computes them,
        dn = g_k (1 - u), da_n = dn (1 - n n), da_u = g_k (h_{k-1} - n) (u (1 - u)), da_r = da_n c (r (1 - r)),
        dgh_k = [da_r, da_u, da_n r], dgi_k = [da_r, da_u, da_n], S = dgi_7 + dgi_6 + .. + dgi_1,
        g_{k-1} = fl(fl(G_{k-1} + g_k u) + bf16(dgh_k) bf16(W_hh))   (the carry contracts with the transposed W_hh).
    x, h0 [R, L]; h [R, 7, L] (h_1 .. h_7, the forward's); w = (w_ih, b_ih, w_hh, b_hh, ...); G [R, 7, L], the entry
    value of d_g (W3^T dz_k with bf16(W3)) -> (d_g [R, 7, L], d_dgh [R, 7, 3L], S [R, 3L]).  Its float32 products sum
    in numpy's order, not the tensor core's.  `mutant` (one of BACKWARD_MUTANTS) runs a plausible defect instead:
    dgh_n = da_n without r; the carry with g_k or g_k (1 - u) for g_k u; da_u with (n - h) for (h - n); da_r without c;
    (1 - n) for (1 - n^2); S summing dgh for dgi; the carry through W_hg for W_hg^T; the carry without its last group
    of atoms; the step reading h_k for h_{k-1} (the staged operand and h in da_u); bf16(dgh) rounded toward zero."""
    from test_gpu_policy_tiling import bf16_rz
    f = np.float32
    w_ih, b_ih, w_hh, b_hh = (np.asarray(a, dtype=f) for a in w[:4])
    L = x.shape[1]
    R = x.shape[0]
    gi = (bf16(np.asarray(x, f)) @ bf16(w_ih).T).astype(f)
    whb = bf16(w_hh)
    hs = np.concatenate([np.asarray(h0, f)[:, None], np.asarray(h, f)], 1)
    g = np.array(G, dtype=f)
    dgh = np.zeros((R, K, 3 * L), dtype=f)
    keep = carry_columns(L, mutant == "carry_last_group_dropped")
    s = None
    for k in range(K, 0, -1):
        hp = hs[:, k] if mutant == "reads_h_k" else hs[:, k - 1]
        gh = (bf16(hp) @ whb.T).astype(f)
        r = _sig32((gi[:, :L] + gh[:, :L]) + (b_ih[:L] + b_hh[:L]))
        u = _sig32((gi[:, L:2 * L] + gh[:, L:2 * L]) + (b_ih[L:2 * L] + b_hh[L:2 * L]))
        c = (gh[:, 2 * L:] + b_hh[2 * L:]).astype(f)
        n = np.tanh((gi[:, 2 * L:] + b_ih[2 * L:]) + r * c).astype(f)
        gk = g[:, k - 1]
        dn = gk * (f(1) - u)
        dan = dn * (f(1) - (n if mutant == "dtanh_1mn" else n * n))
        dau = gk * ((n - hp) if mutant == "dau_n_minus_h" else (hp - n)) * (u * (f(1) - u))
        dar = (dan if mutant == "dar_without_c" else dan * c) * (r * (f(1) - r))
        d = np.concatenate([dar, dau, dan if mutant == "dgh_n_without_r" else dan * r], 1)
        dgh[:, k - 1] = d
        dgi = d if mutant == "s_sums_dgh" else np.concatenate([dar, dau, dan], 1)
        s = dgi if k == K else s + dgi
        if k > 1:
            gu = gk if mutant == "carry_g" else gk * (f(1) - u) if mutant == "carry_g_1mu" else gk * u
            staged = np.where(keep, bf16_rz(d) if mutant == "dgh_rz" else bf16(d), f(0))
            if mutant == "carry_untransposed":
                D = sum(staged[:, q * L:(q + 1) * L] @ whb[q * L:(q + 1) * L].T for q in range(3))
            else:
                D = staged @ whb
            g[:, k - 2] = (g[:, k - 2] + gu) + D.astype(f)
    return g, dgh, s


def _mul(a, b):
    """(value, bound) of a float32 product of two (float64 value, error bound) pairs: the error of the operands times
    the other's largest magnitude, and one rounding of the largest product."""
    (va, ea), (vb, eb) = a, b
    ma, mb = np.abs(va) + ea, np.abs(vb) + eb
    return va * vb, ea * mb + np.abs(va) * eb + U32 * ma * mb


def _sub(a, b):
    (va, ea), (vb, eb) = a, b
    return va - vb, ea + eb + U32 * (np.abs(va) + ea + np.abs(vb) + eb)


class StepBound:
    """backward_step_bound's result: float64 references and per-element bounds of one backward step."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def backward_step_bound(x, h_prev, w, g_k, G_prev=None, dgh_k=None):
    """A first-order bound on one float32 backward step of the kernel, evaluated from the kernel's own inputs to that
    step, so that an error in one step is not blamed on the next.  x, h_prev = h_{k-1} [R, L]; w with bf16 weights;
    g_k [R, L], the kernel's (d_g[:, k - 1] after the call).  Returns a StepBound with
    - dgh, dgh_b [R, 3L]: float64 dgh_k from g_k and float64 gates of h_{k-1}, and the bound on the kernel's dgh_k;
    - dgi, dgi_b [R, 3L]: the same for dgi_k, the step's term of S;
    - with G_prev (the entry value of d_g[:, k - 2]) and dgh_k (the kernel's): g, g_b [R, L], float64 of
      G_{k-1} + g_k u + bf16(dgh_k) bf16(W_hh), and the bound on the kernel's g_{k-1}.
    The gates carry gate_bounds' errors (expf and tanhf within 2 ulp, __frcp_rn correctly rounded).  Each product and
    difference of the gradient formulas adds its operands' errors times the other operand's magnitude and one rounding
    (_mul, _sub): a rounding the compiler removes by contracting a product into an FMA (nvcc's default --fmad=true, no
    fast-math) only makes the error smaller.  The carry is a float32 dot product of 3L terms of exact bf16 products on
    the tensor core: gamma_3L sum |bf16(dgh)| |bf16(W_hh)|; g_k u is off by |g_k| e_u; fl(G + g_k u) and the add of the
    carry are two roundings, and the product g_k u a third where it is not contracted."""
    f64 = np.float64
    L = x.shape[1]
    wb = [np.asarray(a, f64) for a in w[:4]]
    w_ih, b_ih, w_hh, b_hh = wb
    gi = bf16(np.asarray(x, f64)) @ w_ih.T
    gh = bf16(np.asarray(h_prev, f64)) @ w_hh.T
    r = _sig(gi[:, :L] + gh[:, :L] + b_ih[:L] + b_hh[:L])
    u = _sig(gi[:, L:2 * L] + gh[:, L:2 * L] + b_ih[L:2 * L] + b_hh[L:2 * L])
    c = gh[:, 2 * L:] + b_hh[2 * L:]
    n = np.tanh(gi[:, 2 * L:] + b_ih[2 * L:] + r * c)
    e_r, e_u, e_n, e_c = gate_bounds(x, h_prev, wb)
    g = (np.asarray(g_k, f64), 0.0)
    one = (1.0, 0.0)
    R_, U_, N_, C_ = (r, e_r), (u, e_u), (n, e_n), (c, e_c)
    omu = _sub(one, U_)
    dn = _mul(g, omu)
    dan = _mul(dn, _sub(one, _mul(N_, N_)))
    dau = _mul(_mul(g, _sub((np.asarray(h_prev, f64), 0.0), N_)), _mul(U_, omu))
    dar = _mul(_mul(dan, C_), _mul(R_, _sub(one, R_)))
    dgn = _mul(dan, R_)
    out = StepBound(dgh=np.concatenate([dar[0], dau[0], dgn[0]], 1), dgh_b=np.concatenate([dar[1], dau[1], dgn[1]], 1),
                    dgi=np.concatenate([dar[0], dau[0], dan[0]], 1), dgi_b=np.concatenate([dar[1], dau[1], dan[1]], 1))
    if G_prev is not None:
        db = bf16(np.asarray(dgh_k, f64))
        D = db @ w_hh
        Dabs = np.abs(db) @ np.abs(w_hh)
        gu = g[0] * u
        out.g = np.asarray(G_prev, f64) + gu + D
        out.g_b = _gamma(3 * L) * Dabs + np.abs(g[0]) * e_u + 3 * U32 * (np.abs(G_prev) + np.abs(g[0]) * (u + e_u) + Dabs)
    return out


def s_bound(steps):
    """The float64 S = sum of the steps' dgi and the bound on the kernel's S: the steps' own bounds and seven roundings
    of the partial sums (dgi_7 + dgi_6 + .. + dgi_1) -> (S, bound)."""
    S = sum(b.dgi for b in steps)
    mag = sum(np.abs(b.dgi) + b.dgi_b for b in steps)
    return S, sum(b.dgi_b for b in steps) + 7 * U32 * mag


def _ratio(err, bound):
    return np.where(err == 0, 0.0, err / np.maximum(bound, 1e-300))


def backward_ratios(x, h0, h, w, G, g, dgh, s):
    """A backward's d_g, d_dgh and S (the kernel's or backward32's) against backward_step_bound, each step from its own
    inputs -> {'dgh': [R, 7, 3L] (step k at k - 1), 'g': [R, 6, L] (g_{k-1} of step k at k - 2), 'S': [R, 3L]} of
    |got - float64| / bound: within the bound where <= 1 (NaN where the result is not finite)."""
    f64 = np.float64
    hs = np.concatenate([np.asarray(h0, f64)[:, None], np.asarray(h, f64)], 1)
    g, dgh, s, G = (np.asarray(a, f64) for a in (g, dgh, s, G))
    rd, rg, steps = np.zeros(dgh.shape), np.zeros(g[:, 1:].shape), []
    for k in range(K, 0, -1):
        b = backward_step_bound(x, hs[:, k - 1], w, g[:, k - 1], G[:, k - 2] if k > 1 else None, dgh[:, k - 1] if k > 1 else None)
        rd[:, k - 1] = _ratio(np.abs(dgh[:, k - 1] - b.dgh), b.dgh_b)
        if k > 1:
            rg[:, k - 2] = _ratio(np.abs(g[:, k - 2] - b.g), b.g_b)
        steps.append(b)
    S, sb = s_bound(steps)
    return {"dgh": rd, "g": rg, "S": _ratio(np.abs(s - S), sb)}


def worst(ratios):
    """{name: (largest ratio, its index (row, k, column) or (row, column))}, NaN counted as the largest."""
    out = {}
    for name, r in ratios.items():
        i = np.unravel_index(np.argmax(np.where(np.isnan(r), np.inf, r)), r.shape)
        out[name] = (float(r[i]), tuple(int(v) for v in i))
    return out


def pack_wht(w_hh):
    """The transposed image evg_rppo_train_pack writes (d_wht_img), built on the host: gate g's block holds
    W_hg^T = w_hh[g L:(g + 1) L].T as an [Lp x Ka] K-major swizzled image."""
    from evgsim import policy
    w_hh = np.asarray(w_hh, dtype=np.float32)
    L = w_hh.shape[1]
    lp, ka = -(-L // 16) * 16, -(-L // 64) * 64
    return np.concatenate([policy._image(w_hh[g * L:(g + 1) * L].T, lp, ka) for g in range(3)])
