"""Host side of the fused PPO actor (evg_policy_ppo): the weight images and bias vector pack_ppo builds, the numpy
statement of the kernel's arithmetic, the tape's domain 3 and the sampler it feeds.  The kernel itself is checked in
tests/test_gpu_policy_ppo.py."""
import numpy as np
import pytest

from evgsim import _capi, policy
import ppo_sampling as ps
from oracle import tape


def _weights(rng, latent, out=132, in_dim=105, scale=1.0):
    return [(rng.standard_normal(s) * scale).astype(np.float32)
            for s in ((latent, in_dim), (latent,), (latent, latent), (latent,), (out, latent), (out,))]


@pytest.mark.parametrize("latent", [128, 248, 100, 1, 15, 16, 17, 63, 64, 65, 129, 160, 192, 193, 255, 256])
def test_pack_ppo_places_every_weight_where_the_header_says(latent):
    w1, b1, w2, b2, w3, b3 = _weights(np.random.default_rng(latent), latent)
    img1, img2, img3, bias, L, out = policy.pack_ppo(w1, b1, w2, b2, w3, b3)
    lp, ka = -(-latent // 16) * 16, -(-latent // 64) * 64
    assert (L, out) == (latent, 132)
    assert img1.nbytes == 2 * lp * 128 and img2.nbytes == (ka // 64) * lp * 128 and img3.nbytes == (ka // 64) * 144 * 128
    i1, i2, i3 = img1.view(np.uint16), img2.view(np.uint16), img3.view(np.uint16)
    bits = policy.to_bf16_bits
    # every weight, each at its swizzled byte
    n, k = np.meshgrid(np.arange(latent), np.arange(105), indexing="ij")
    assert np.array_equal(i1[policy.swz_offset(lp, n, k) // 2], bits(w1))
    n, k = np.meshgrid(np.arange(latent), np.arange(latent), indexing="ij")
    assert np.array_equal(i2[policy.swz_offset(lp, n, k) // 2], bits(w2))
    o, k = np.meshgrid(np.arange(132), np.arange(latent), indexing="ij")
    assert np.array_equal(i3[policy.swz_offset(144, o, k) // 2], bits(w3))
    # ... and nothing else: the padding is zero
    for img, w in ((i1, w1), (i2, w2), (i3, w3)):
        assert np.count_nonzero(img) == np.count_nonzero(bits(w))
    # biases stay float32: b1 at 0, b2 at 256, b3 at 512, zero padded
    assert bias.dtype == np.float32 and bias.shape == (2 * 256 + 144,)
    assert np.array_equal(bias[:latent], b1) and np.array_equal(bias[256:256 + latent], b2) and np.array_equal(bias[512:644], b3)
    assert not bias[latent:256].any() and not bias[256 + latent:512].any() and not bias[644:].any()


@pytest.mark.parametrize("latent", [128, 248, 100])
def test_reference_forward_ppo_agrees_with_the_fp32_torch_net(latent):
    """The only difference to fp32 torch is the bf16 rounding of the operands and hidden activations: the largest
    probability error stays within 3e-2 of the largest probability."""
    import torch
    torch.manual_seed(latent)
    net = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                              torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
    rng = np.random.default_rng(0)
    obs = rng.integers(-3, 40, size=(300, 105)).astype(np.float32)  # integer-valued, like the game's observations
    w = [t.detach().numpy() for m in (net[0], net[2], net[4]) for t in (m.weight, m.bias)]
    got = policy.reference_forward_ppo(obs, *w)
    with torch.no_grad():
        want = net(torch.from_numpy(obs)).numpy()
    assert got.dtype == np.float32 and got.shape == want.shape
    assert np.abs(got.sum(-1) - 1).max() < 1e-5
    assert np.abs(got - want).max() <= 3e-2 * want.max(), (np.abs(got - want).max(), want.max())


def test_policy_uniforms_are_keyed_on_every_field():
    base = (7, 1234, 15, 0, 2)  # seed, global match id, turn, player, episode
    u = ps.policy_uniforms(*base)
    assert u.dtype == np.float32 and u.shape == (7,) and (u >= 0).all() and (u < 1).all()
    for f in range(5):
        other = list(base)
        other[f] += 1
        assert not np.array_equal(ps.policy_uniforms(*other), u), f
    # u_k = (w_k >> 8) * 2^-24 of domain 3's blocks; domain 1 (random_actions) on the same counters is another stream
    seed, env, turn, player, episode = base
    h3 = tape.block_halves(seed, env, turn, player, ps.DOMAIN_POLICY_SAMPLE, episode)
    h1 = tape.block_halves(seed, env, turn, player, tape.DOMAIN_AGENT_RANDOM, episode)
    w0 = h3[0] | h3[1] << 16
    assert u[0] == np.float32((w0 >> 8) * 2.0 ** -24)
    assert h3 != h1
    assert ps.DOMAIN_POLICY_SAMPLE == 3


def test_ppo_sample_draws_distinct_indices_and_falls_back_to_the_largest_open_index():
    rng = np.random.default_rng(3)
    for _ in range(50):
        p = rng.random(132).astype(np.float32)
        p /= p.sum()
        idx = ps.ppo_sample(p, rng.random(7).astype(np.float32))
        assert len(set(idx.tolist())) == 7 and idx.min() >= 0 and idx.max() < 132
    # only three indices carry mass: after them T = 0, no x < c is ever met, and each later draw takes the largest
    # index not chosen yet
    p = np.zeros(10, dtype=np.float32)
    p[[1, 4, 6]] = np.float32(1 / 3)
    idx = ps.ppo_sample(p, np.full(7, 0.5, dtype=np.float32))
    assert sorted(idx[:3].tolist()) == [1, 4, 6] and idx[3:].tolist() == [9, 8, 7, 5]
    # u = 0 takes the first open index with mass, the largest u below 1 the last one
    q = np.full(8, np.float32(1 / 8))
    assert ps.ppo_sample(q, np.zeros(7, dtype=np.float32)).tolist() == [0, 1, 2, 3, 4, 5, 6]
    assert ps.ppo_sample(q, np.full(7, 1 - 2 ** -24, dtype=np.float32)).tolist() == [7, 6, 5, 4, 3, 2, 1]


def test_ppo_sample_rows_equals_ppo_sample_row_by_row():
    """The vectorised sampler the GPU tests check whole batches with makes the same draws as the scalar statement,
    including rows whose mass runs out (the fallback to the largest open index) and uniforms at both ends."""
    rng = np.random.default_rng(5)
    for n in (7, 17, 132, 144):
        p = rng.random((300, n)).astype(np.float32) ** 4  # a few large entries, many tiny ones
        p[:20] = 0
        p[np.arange(20), rng.integers(0, n, 20)] = 1  # one index with all the mass
        p[20:40, : n // 2] = 0
        p /= p.sum(-1, dtype=np.float32, keepdims=True)
        u = rng.random((300, 7)).astype(np.float32)
        u[40:60] = 0
        u[60:80] = 1 - 2 ** -24
        want = np.stack([ps.ppo_sample(p[i], u[i]) for i in range(300)])
        assert np.array_equal(ps.ppo_sample_rows(p, u), want), n


def test_ppo_sample_matches_sequential_sampling_without_replacement():
    """Ordered triples of 5 items: frequencies over 200,000 draws against the exact probabilities
    p_i * p_j / (1 - p_i) * p_k / (1 - p_i - p_j) (chi-square, fixed seed)."""
    from scipy import stats
    p = np.array([0.35, 0.25, 0.2, 0.12, 0.08], dtype=np.float32)
    rng = np.random.default_rng(11)
    n = 200_000
    u = ((rng.integers(0, 1 << 24, size=(n, 3))).astype(np.float64) * 2.0 ** -24).astype(np.float32)
    counts = {}
    for k in range(n):
        t = tuple(ps.ppo_sample(p, u[k]).tolist())
        counts[t] = counts.get(t, 0) + 1
    pd = p.astype(np.float64)
    keys, exp = [], []
    for i in range(5):
        for j in range(5):
            for m in range(5):
                if len({i, j, m}) == 3:
                    keys.append((i, j, m))
                    exp.append(pd[i] * pd[j] / (1 - pd[i]) * pd[m] / (1 - pd[i] - pd[j]))
    assert set(counts) <= set(keys)
    obs = np.array([counts.get(k, 0) for k in keys], dtype=np.float64)
    exp = np.array(exp) / np.sum(exp) * n
    assert stats.chisquare(obs, exp).pvalue > 1e-4


def test_null_handle_call_fails():
    import __graft_entry__ as g
    g.build()
    lib = _capi.load()
    assert lib.evg_policy_ppo(None, None, -1, None, None, None, None, 128, 132, 12, 11, None, None, None, None) == -1
