"""Host side of the fused recurrent PPO actor (evg_policy_rppo): the numpy statement of the kernel's arithmetic against
torch.nn.GRU, the images pack_rppo builds, and the checks FusedRPPO makes before any device call.  The kernel itself is
checked in tests/test_gpu_policy_rppo.py."""
import types

import numpy as np
import pytest

from evgsim import _capi, policy


class Actor:
    """The reference ActorCritic's actor (use_recurrent): action_head, action_gru, action_layer; forward over 7 steps
    as tools/policy_rollout.py: RecurrentActor."""

    def __init__(self, torch, latent, seed=0, in_dim=105, out=132, **gru_kw):
        torch.manual_seed(seed)
        self.action_head = torch.nn.Sequential(torch.nn.Linear(in_dim, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
        self.action_gru = torch.nn.GRU(gru_kw.pop("input_size", latent), latent, **gru_kw)
        self.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, out), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))

    def __call__(self, x, hidden):
        seq, hidden = self.action_gru(self.action_head(x).unsqueeze(0).expand(7, -1, -1).contiguous(), hidden)
        return self.action_layer(seq), hidden


@pytest.mark.parametrize("latent", [1, 17, 128, 248, 256])
def test_reference_forward_rppo_matches_torch_gru_over_carried_turns(latent):
    """bf16=False is torch's network in fp32 (gate order r, z, n; r multiplies W_hn h + b_hn), to 1e-5 over three turns
    whose state is carried from one to the next; bf16=True stays within 3e-2 of the largest probability."""
    import torch
    actor = Actor(torch, latent, seed=latent)
    w = policy.rppo_weights(actor)
    rng = np.random.default_rng(latent)
    rows = 200
    h = rng.uniform(-1, 1, (rows, latent)).astype(np.float32)
    h_bf = h.copy()
    for turn in range(3):
        obs = rng.integers(-3, 40, size=(rows, 105)).astype(np.float32)  # integer-valued, like the game's observations
        with torch.no_grad():
            p_t, h_t = actor(torch.from_numpy(obs), torch.from_numpy(h).unsqueeze(0))
        p_t, h_t = p_t.permute(1, 0, 2).numpy(), h_t[0].numpy()
        probs, h_new = policy.reference_forward_rppo(obs, h, w, bf16=False)
        assert probs.dtype == np.float32 and probs.shape == (rows, 7, 132) and h_new.shape == (rows, latent)
        assert np.abs(probs - p_t).max() <= 1e-5, (turn, np.abs(probs - p_t).max())
        assert np.abs(h_new - h_t).max() <= 1e-5, (turn, np.abs(h_new - h_t).max())
        pb, h_bf = policy.reference_forward_rppo(obs, h_bf, w, bf16=True)
        assert np.abs(pb.sum(-1) - 1).max() < 1e-5
        assert np.abs(pb - p_t).max() <= 3e-2 * p_t.max(), (turn, np.abs(pb - p_t).max(), p_t.max())
        h = h_t


@pytest.mark.parametrize("latent", [1, 15, 16, 17, 63, 64, 65, 127, 128, 129, 160, 192, 248, 255, 256])
def test_pack_rppo_places_every_weight_where_the_header_says(latent):
    rng = np.random.default_rng(latent)
    shapes = ((latent, 105), (latent,), (latent, latent), (latent,), (3 * latent, latent), (3 * latent,), (3 * latent, latent),
              (3 * latent,), (132, latent), (132,))
    w1, b1, w2, b2, w_ih, b_ih, w_hh, b_hh, w3, b3 = [rng.standard_normal(s).astype(np.float32) for s in shapes]
    img1, img2, imgi, imgh, img3, bias, L, out = policy.pack_rppo(w1, b1, w2, b2, w_ih, b_ih, w_hh, b_hh, w3, b3)
    lp, ka = -(-latent // 16) * 16, -(-latent // 64) * 64
    assert (L, out) == (latent, 132)
    # the head and the output layer are pack_ppo's
    for got, want in zip((img1, img2, img3, bias[:656]), policy.pack_ppo(w1, b1, w2, b2, w3, b3)[:4]):
        assert np.array_equal(got, want)
    block = (ka // 64) * lp * 128
    assert imgi.nbytes == imgh.nbytes == 3 * block
    n, k = np.meshgrid(np.arange(latent), np.arange(latent), indexing="ij")
    for img, w in ((imgi, w_ih), (imgh, w_hh)):
        for g in range(3):
            gate = img[g * block:(g + 1) * block].view(np.uint16)
            assert np.array_equal(gate[policy.swz_offset(lp, n, k) // 2], policy.to_bf16_bits(w[g * latent:(g + 1) * latent]))
            assert np.count_nonzero(gate) == np.count_nonzero(policy.to_bf16_bits(w[g * latent:(g + 1) * latent]))
    # the GRU's biases stay float32: b_ih gate g at 656 + 256 g, b_hh gate g at 1424 + 256 g, zero padded
    assert bias.dtype == np.float32 and bias.shape == (656 + 6 * 256,)
    for base, b in ((656, b_ih), (1424, b_hh)):
        for g in range(3):
            seg = bias[base + 256 * g:base + 256 * (g + 1)]
            assert np.array_equal(seg[:latent], b[g * latent:(g + 1) * latent]) and not seg[latent:].any()


def _env(obs_len=105, num_envs=4):
    """Only what FusedRPPO reads before its first device call."""
    return types.SimpleNamespace(obs_len=obs_len, num_envs=num_envs, device="cpu")


@pytest.mark.parametrize("case", ["layers", "bidirectional", "input_size", "no_bias", "obs_width", "too_wide"])
def test_fused_rppo_refuses_a_network_the_kernel_does_not_run(case):
    import torch
    kw = {"layers": dict(num_layers=2), "bidirectional": dict(bidirectional=True), "input_size": dict(input_size=16),
          "no_bias": dict(bias=False)}.get(case, {})
    latent = 257 if case == "too_wide" else 32
    actor = Actor(torch, latent, in_dim=100 if case == "obs_width" else 105, **kw)
    with pytest.raises(ValueError):
        policy.FusedRPPO(_env(), actor)


def test_null_handle_call_fails():
    import __graft_entry__ as g
    g.build()
    lib = _capi.load()
    assert lib.evg_policy_rppo(None, None, -1, None, None, None, None, None, None, 128, 132, 12, 11, None, None, None, None, None) == -1
