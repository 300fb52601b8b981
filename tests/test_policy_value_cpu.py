"""The fused PPO critic's host side (no GPU): evgsim.policy.pack_value's images, reference_forward_value against a float64
evaluation within a derived bound, and the refusals of FusedValue that need no device.

The bound (value_bound).  Let x, W1, W2, w3 be the bf16-rounded operands.  The truth v is the critic in float64 on them
with each hidden activation rounded to bf16 (nearest even) as the kernel rounds it: H1 = bf16(tanh(W1 x + b1)),
H2 = bf16(tanh(W2 H1 + b2)), v = w3 . H2 + b3.  A computation with float32 sums in any order and a float32 tanh (the
numpy reference, or the kernel's tensor cores, whose fp32 accumulation may truncate: unit error u = 2^-23 per operation
rather than 2^-24) differs from it by at most, unit by unit (absolute values; gamma_n = n u / (1 - n u)):
- layer 1: the pre-activation is off by e1 <= gamma_K |W1| |x| + u |z1| (K = obs_len products, then b1); tanh's slope
  on [|z1| - e1, |z1| + e1] is at most sech^2(max(|z1| - e1, 0)) and a float32 tanh is within E_T = 4 u of tanh, so t1 is
  off by d1 = e1 (1 + u) sech^2(max(|z1| - e1, 0)) + E_T (tanh_error).  The computed H1 is the
  truth's unless a bf16 rounding midpoint lies within d1 of t1; where one does, it is off by at most d1 + 2 ulp(t1)
  (bf16_shift).  Call that D1 (0 for most units).
- layer 2: e2 <= |W2| D1 + gamma_L |W2| (|H1| + D1) + u (|z2| + e2), then d2 and D2 as for layer 1.
- output: |dv| <= |w3| D2 + gamma_L |w3| (|H2| + D2) + u (|v| + |dv|).
Where no rounding can flip, the bound is float32 accumulation error only; a unit that can flip allows one bf16 step of
it through w3."""
import numpy as np
import pytest

from evgsim import policy

LATENTS = [1, 15, 16, 17, 63, 64, 65, 128, 129, 255, 256]
U = 2.0 ** -23          # float32 unit error per operation, with room for truncating accumulation
E_T = 4 * 2.0 ** -24    # a float32 tanh within a few ulps of tanh, |tanh| <= 1


def gamma(n):
    return n * U / (1 - n * U)


def bf16_shift(t, d):
    """How far bf16(t') can be from bf16(t) for any |t' - t| <= d: 0 unless a bf16 rounding midpoint lies within d of t,
    else d + 2 ulp(t) (room for a binade edge)."""
    a = np.abs(t)
    ulp = np.exp2(np.floor(np.log2(np.maximum(a, 2.0 ** -120))) - 7)
    r = a / ulp
    dist = np.abs(r - np.floor(r) - 0.5) * ulp
    return np.where(dist <= d, d + 2 * ulp, 0.0)


def tanh_error(z, e):
    """How far a float32 tanh of a value within e of z can be from tanh(z)."""
    return e * (1 + U) * 4 / (np.exp(np.minimum(np.maximum(np.abs(z) - e, 0.0), 300)) + np.exp(-np.maximum(np.abs(z) - e, 0.0))) ** 2 + E_T


def value_bound(obs, w1, b1, w2, b2, w3, b3):
    """(v float64 [rows], bound float64 [rows]) of the module docstring."""
    f64 = np.float64
    rnd = lambda a: policy.bf16_round(np.asarray(a, dtype=np.float32)).astype(f64)  # noqa: E731
    x, W1, W2, w3 = rnd(obs), rnd(w1), rnd(w2), rnd(w3).reshape(-1)
    b1, b2, b3 = (np.asarray(b, dtype=np.float32).astype(f64) for b in (b1, b2, b3))
    K, L = W1.shape[1], W1.shape[0]
    z1 = x @ W1.T + b1
    t1 = np.tanh(z1)
    H1 = rnd(t1)
    e1 = gamma(K) * (np.abs(x) @ np.abs(W1).T) + U * np.abs(z1)
    D1 = bf16_shift(t1, tanh_error(z1, e1))
    z2 = H1 @ W2.T + b2
    t2 = np.tanh(z2)
    H2 = rnd(t2)
    e2 = D1 @ np.abs(W2).T + gamma(L) * ((np.abs(H1) + D1) @ np.abs(W2).T)
    e2 = e2 + U * (np.abs(z2) + e2)
    D2 = bf16_shift(t2, tanh_error(z2, e2))
    v = H2 @ w3 + b3[0]
    dv = D2 @ np.abs(w3) + gamma(L) * ((np.abs(H2) + D2) @ np.abs(w3))
    return v, dv + U * (np.abs(v) + 2 * dv)


def critic_weights(rng, in_dim, latent, scale=1.0):
    """Random float32 weights in torch.nn.Linear's init range (uniform +-1/sqrt(fan_in)), times `scale`."""
    def lin(o, i):
        k = scale / np.sqrt(i)
        return rng.uniform(-k, k, (o, i)).astype(np.float32), rng.uniform(-k, k, o).astype(np.float32)
    w1, b1 = lin(latent, in_dim)
    w2, b2 = lin(latent, latent)
    w3, b3 = lin(1, latent)
    return [w1, b1, w2, b2, w3, b3]


def obs_like(rng, rows, in_dim):
    """Integer rows in the observations' range, a few above 256 (rounded to even integers by bf16)."""
    x = rng.integers(-100, 151, (rows, in_dim)).astype(np.float32)
    x[:, 0] = rng.integers(0, 600, rows)
    return x


def block_bytes(mat, rows, cols):
    """The [rows x cols] block of `mat` (zero padded) written element by element at policy.swz_offset, independently of
    policy._image: uint8 [(cols / 64) * rows * 128]."""
    full = np.zeros((rows, cols), dtype=np.float32)
    full[:mat.shape[0], :mat.shape[1]] = mat
    out = np.full((cols // 64) * rows * 128, 0xAB, dtype=np.uint8)
    bits = policy.to_bf16_bits(full)
    for r in range(rows):
        for k in range(cols):
            o = policy.swz_offset(rows, r, k)
            out[o], out[o + 1] = bits[r, k] & 0xFF, bits[r, k] >> 8
    return out


@pytest.mark.parametrize("latent", LATENTS)
def test_pack_value_bytes(latent):
    """Every element of W1, W2 and w3 at its swizzle position, every other byte zero (block_bytes starts from 0xAB, so
    a byte no element covers would show), W1 and W2 exactly pack_ppo's, and the bias vector's layout."""
    rng = np.random.default_rng(latent)
    w = critic_weights(rng, 105, latent, scale=7.0)
    img1, img2, img3, bias, L = policy.pack_value(*w)
    lp, ka = -(-latent // 16) * 16, -(-latent // 64) * 64
    assert L == latent
    for img, mat, rows, cols in ((img1, w[0], lp, 128), (img2, w[2], lp, ka), (img3, w[4], 16, ka)):
        assert img.dtype == np.uint8
        assert np.array_equal(img, block_bytes(mat, rows, cols)), (rows, cols)
    p1, p2, _, _, _, _ = policy.pack_ppo(w[0], w[1], w[2], w[3], np.ones((7, latent), np.float32), np.zeros(7, np.float32))
    assert np.array_equal(img1, p1) and np.array_equal(img2, p2)
    want = np.zeros(2 * 256 + 16, dtype=np.float32)
    want[:latent], want[256:256 + latent], want[512] = w[1], w[3], w[5][0]
    assert bias.dtype == np.float32 and np.array_equal(bias.view(np.uint32), want.view(np.uint32))


def test_pack_value_refuses_other_shapes():
    w = critic_weights(np.random.default_rng(0), 105, 32)
    for k, bad in ((4, np.zeros((2, 32), np.float32)), (5, np.zeros(2, np.float32)), (2, np.zeros((32, 31), np.float32))):
        with pytest.raises(AssertionError):
            policy.pack_value(*(w[:k] + [bad] + w[k + 1:]))
    with pytest.raises(AssertionError):
        policy.pack_value(*critic_weights(np.random.default_rng(0), 105, 257))


@pytest.mark.parametrize("latent", [1, 17, 128, 248, 256])
@pytest.mark.parametrize("scale", [1.0, 4.0])
def test_reference_within_the_derived_bound(latent, scale):
    """reference_forward_value within value_bound of the float64 truth, and (L > 128) the second 128 columns of H2
    dropped from the dot product leave it."""
    rng = np.random.default_rng(latent + int(scale))
    w = critic_weights(rng, 105, latent, scale)
    x = obs_like(rng, 500, 105)
    got = policy.reference_forward_value(x, *w)
    assert got.dtype == np.float32 and got.shape == (500,)
    v, bound = value_bound(x, *w)
    assert (np.abs(got - v) <= bound).all(), (np.abs(got - v) / bound).max()
    if latent > 128:  # the subtler defects are left to the exact network of tests/test_gpu_policy_value.py
        f32, rnd = np.float32, policy.bf16_round
        h = rnd(np.tanh((rnd(x) @ rnd(w[0]).T).astype(f32) + w[1]).astype(f32))
        h = rnd(np.tanh((h @ rnd(w[2]).T).astype(f32) + w[3]).astype(f32))
        h[:, 128:] = 0
        dropped = (h @ rnd(w[4]).T).astype(f32).reshape(-1) + w[5]
        assert (np.abs(dropped - v) > bound).mean() > 0.2


# ---------------------------------------------------------------- FusedValue's refusals without a device

class HostEnv:
    """What FusedValue reads of an env before it launches anything, on the CPU."""

    def __init__(self, n=4, obs_len=105):
        import torch
        self.num_envs, self.obs_len, self.device = n, obs_len, torch.device("cpu")
        self.obs = torch.zeros((n, 2, obs_len))


def critic(torch, width=105, latent=32, last=1, hidden_layers=2):
    layers = [torch.nn.Linear(width, latent), torch.nn.Tanh()]
    for _ in range(hidden_layers - 1):
        layers += [torch.nn.Linear(latent, latent), torch.nn.Tanh()]
    return torch.nn.Sequential(*layers, torch.nn.Linear(latent, last))


def test_fused_value_refuses_networks_it_cannot_run():
    torch = pytest.importorskip("torch")
    env = HostEnv()
    policy.FusedValue(env, critic(torch))  # the shape it runs
    for net, match in ((critic(torch, last=2), "Linear\\(L, 1\\)"), (critic(torch, hidden_layers=1), "3 Linear|Linear layers"),
                       (critic(torch, hidden_layers=3), "Linear layers"), (critic(torch, width=104), "104 inputs"),
                       (critic(torch, latent=257), "257")):
        with pytest.raises(ValueError, match=match):
            policy.FusedValue(env, net)
    w = policy._host_arrays(policy._value_params(critic(torch)))
    with pytest.raises(ValueError, match="shape"):
        policy.FusedValue(env, weights=w[:4] + [np.zeros((2, 32), np.float32), np.zeros(2, np.float32)])
    with pytest.raises(ValueError, match="6 arrays"):
        policy.FusedValue(env, weights=w[:4])
    with pytest.raises(ValueError, match="player"):
        policy.FusedValue(env, weights=w, player=2)
    with pytest.raises(ValueError, match="input columns"):
        wide = HostEnv(obs_len=189)
        policy.FusedValue(wide, critic(torch, width=189))


def test_fused_value_refuses_bad_inputs_before_launching():
    torch = pytest.importorskip("torch")
    env = HostEnv()
    f = policy.FusedValue(env, critic(torch))
    with pytest.raises(ValueError, match="obs_format"):
        f(obs_format="i16")
    good = torch.zeros((3, 2, 105))
    for bad in (good.double(), good[:, :, :104].clone(), good.view(6, 105), good.transpose(0, 1).contiguous().transpose(0, 1),
                good.numpy()):
        with pytest.raises(ValueError, match="obs must be"):
            f(bad)
    for out in (torch.zeros((3, 2), dtype=torch.float64), torch.zeros((3,)), torch.zeros((2, 3)).t(), torch.zeros((4, 2))):
        with pytest.raises(ValueError, match="out must be"):
            f(good, out=out)
    with pytest.raises(ValueError, match="out must be"):
        f(out=torch.zeros((4,)))
    one = policy.FusedValue(env, critic(torch), player=1)
    assert tuple(one.value.shape) == (4,) and tuple(f.value.shape) == (4, 2)
    with pytest.raises(ValueError, match="out must be"):
        one(good, out=torch.zeros((3, 2)))
    assert f(good[:0]).shape == (0, 2)  # no matches: nothing to launch
