"""The feed-forward update networks of evg_ppo_train_forward / _backward (include/evgsim.h) in numpy: the float64
statement, its analytic backward, torch float64 autograd of the same expression, the float32 statement in the kernels'
order, the W2^T image as the host packs it, and the bounds the GPU tests hold the kernels to.

Per row, L = 1..256:  h1 = tanh(W1 obs + b1),  h2 = tanh(W2 h1 + b2),  then z = W3 h2 + b3 (actor), v = w3 . h2 + b3
(critic) or nothing (head: x = h2).  In the kernels every product's operands are bf16 (`rnd`).  Backward with the bf16
roundings taken as the identity:  g2 = dz W3 | dv w3 | dx,  dD2 = g2 (1 - h2^2),  dD1 = (dD2 W2) (1 - h1^2),
dW3 = dz^T h2, dW2 = dD2^T h1, dW1 = dD1^T obs, the biases' the column sums."""
import numpy as np

from evgsim import policy

U32 = 2.0 ** -24  # unit roundoff of float32


def bf16(a):
    """a rounded to bf16 (float64 stays float64, anything else becomes float32)."""
    a = np.asarray(a)
    return policy.bf16_round(a.astype(np.float32)).astype(np.float64 if a.dtype == np.float64 else np.float32)


def gamma(n):
    return n * U32 / (1 - n * U32)


def forward64(obs, w, net, rnd=lambda a: a):
    """float64 forward: w = (w1, b1, w2, b2[, w3, b3]); returns (y, h1, h2), y = z [R, out], v [R] or x = h2."""
    f = np.float64
    w1, b1, w2, b2 = (np.asarray(a, f) for a in w[:4])
    h1 = np.tanh(rnd(np.asarray(obs, f)) @ rnd(w1).T + b1)
    h2 = np.tanh(rnd(h1) @ rnd(w2).T + b2)
    if net == "head":
        return h2, h1, h2
    w3, b3 = (np.asarray(a, f) for a in w[4:])
    y = rnd(h2) @ rnd(w3).T + b3
    return (y[:, 0] if net == "critic" else y), h1, h2


def backward64(obs, w, net, dy):
    """The analytic backward of forward64 (no rounding): gradients of sum(y * dy) for w's parameters, in w's order."""
    f = np.float64
    obs, dy = np.asarray(obs, f), np.asarray(dy, f)
    _, h1, h2 = forward64(obs, w, net)
    if net == "actor":
        g2 = dy @ np.asarray(w[4], f)
    elif net == "critic":
        g2 = dy[:, None] * np.asarray(w[4], f)
    else:
        g2 = dy
    dd2 = g2 * (1 - h2 * h2)
    dd1 = (dd2 @ np.asarray(w[2], f)) * (1 - h1 * h1)
    grads = [dd1.T @ obs, dd1.sum(0), dd2.T @ h1, dd2.sum(0)]
    if net == "actor":
        grads += [dy.T @ h2, dy.sum(0)]
    elif net == "critic":
        grads += [(dy @ h2)[None, :], np.array([dy.sum()])]
    return grads


def torch_reference(obs, w, net, dy):
    """torch float64 autograd of the same expression: (y, gradients in w's order)."""
    import torch
    t = [torch.tensor(np.asarray(a, np.float64), requires_grad=True) for a in w]
    o = torch.tensor(np.asarray(obs, np.float64))
    h = torch.tanh(o @ t[0].T + t[1])
    h = torch.tanh(h @ t[2].T + t[3])
    y = h if net == "head" else h @ t[4].T + t[5]
    if net == "critic":
        y = y[:, 0]
    (y * torch.tensor(np.asarray(dy, np.float64))).sum().backward()
    return y.detach().numpy(), [a.grad.numpy() for a in t]


def forward32(obs, w, net):
    """The float32 statement: bf16 operands, float32 products and sums (numpy's order), float32 biases and tanh."""
    f = np.float32
    w1, b1, w2, b2 = (np.asarray(a, f) for a in w[:4])
    h1 = np.tanh((bf16(np.asarray(obs, f)) @ bf16(w1).T).astype(f) + b1).astype(f)
    h2 = np.tanh((bf16(h1) @ bf16(w2).T).astype(f) + b2).astype(f)
    if net == "head":
        return h2, h1, h2
    w3, b3 = (np.asarray(a, f) for a in w[4:])
    y = ((bf16(h2) @ bf16(w3).T).astype(f) + b3).astype(f)
    return (y[:, 0] if net == "critic" else y), h1, h2


def layer_bound(x, w, b):
    """|float32 h - tanh(bf16(x) . bf16(w) + b) in float64| of one hidden layer from its float32 input x: the dot product
    of K terms and the bias add within gamma_{K+1} sum |a||b| for any order of round-to-nearest sums, taken twice over
    because the tensor core's accumulation order and rounding are not documented; tanh does not grow it (|tanh'| <= 1);
    tanhf's own error within 2 ulp (CUDA's accurate tanhf; numpy's is better): 4 u |h|."""
    xb, wb = bf16(np.asarray(x, np.float64)), bf16(np.asarray(w, np.float64))
    a = xb @ wb.T + np.asarray(b, np.float64)
    return 2 * gamma(xb.shape[1] + 1) * (np.abs(xb) @ np.abs(wb).T + np.abs(np.asarray(b, np.float64))) + 4 * U32 * np.abs(np.tanh(a))


def pack_w2t(w2):
    """The W2^T image evg_ppo_train_pack writes: element (j, i) = w2[i][j] of an [Lp x Ka] block, zero padded."""
    L = np.shape(w2)[0]
    return policy._image(np.asarray(w2, np.float32).T, -(-L // 16) * 16, -(-L // 64) * 64)


def dd1_bound(dd2_kernel, w2):
    """|dD1 - float64 of the kernel's own bf16(dD2) . bf16(W2) (1 - h1^2)|: the tensor core's fp32 accumulation of L
    products, taken at twice the round-to-nearest gamma_L sum |a||b| (the order and the rounding inside the MMA are
    not documented), then the epilogue's float32 (1 - h1^2), within 2 u absolute, and its product, u relative:
    (2 gamma_L + 3 u) sum |a||b|, as 0 <= 1 - h1^2 <= 1."""
    a, b = np.abs(bf16(np.asarray(dd2_kernel, np.float64))), np.abs(bf16(np.asarray(w2, np.float64)))
    return (2 * gamma(a.shape[1]) + 3 * U32) * (a @ b) + 1e-30


def matmul_bound(a, b):
    """|fl32(a^T b) - (a^T b)| for any summation order of R terms: gamma_R sum |a||b|."""
    a, b = np.abs(np.asarray(a, np.float64)), np.abs(np.asarray(b, np.float64))
    return gamma(a.shape[0]) * (a.T @ b) + 1e-30


def ratio_bound(n):
    """|ratio - 1| of env.ppo_loss fed z bit for bit the acting kernel's pre-tanh values: y = tanh(z) is the same float,
    so only the summation orders differ (ppo_loss's butterfly against the sampler's ascending sums).  Per draw
    logp = log p_j - log T_k: p_j = e_j / S with S a sum of n terms (each order within gamma_{n-1} of the exact sum, so
    the two within 2 gamma_{n-1}), T_k a sum of up to n of the p (2 gamma_{n-1} again, plus the p's own rounding), and the
    division, log and subtraction a few u each: |d logp| <= 4 gamma_n + 8 u per draw, 7 draws, then exp."""
    return float(np.expm1(7 * (4 * gamma(n) + 8 * U32)))
