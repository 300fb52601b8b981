"""Policy-in-the-loop glue: the reference's two networks evaluated by libevgsim's fused tensor-core kernels (tcgen05 +
TMEM, bf16 operands, fp32 accumulation) on the observation tensor the step kernel writes.

- DQN (agents/DQN/QNetwork.py:37,42 — Linear(105, 528) - ReLU - Linear(528, 132)): evg_policy_mlp, decoded by
  evg_decode_dqn.  ``pack_mlp`` builds its weight images, ``FusedDQN`` wraps a torch ``Sequential(Linear, ReLU, Linear)``.
- PPO's actor (agents/PPO/ActorCritic.py:33-50 without the GRU — Linear(105, L) - Tanh - Linear(L, L) - Tanh -
  Linear(L, 132) - Tanh - Softmax): evg_policy_ppo, which also draws PPOAgent.get_action's 7 indices on the tape and
  writes the action rows.  ``pack_ppo`` builds its images, ``FusedPPO`` wraps the torch ``Sequential``.
- PPO's recurrent actor (agents/PPO/ActorCritic.py:33-60 with use_recurrent — the same head, then GRU(L, L) stepped 7
  times on the head's output, Linear(L, 132) - Tanh - Softmax after every step, one draw per step): evg_policy_rppo, which
  carries the GRU state across turns and zeroes it when a match starts over.  ``pack_rppo`` builds its images,
  ``FusedRPPO`` wraps a module with the reference ActorCritic's ``action_head``, ``action_gru`` and ``action_layer``.
- PPO's critic (agents/PPO/ActorCritic.py, value_layer — Linear(105, L) - Tanh - Linear(L, L) - Tanh - Linear(L, 1)):
  evg_policy_value, the state values of the env's observations or of any number of stored rows.  ``pack_value`` builds
  its images, ``FusedValue`` wraps the torch ``Sequential``.

The images are what the kernels copy straight into shared memory (bf16, K-major, 128-byte swizzle; layout in
include/evgsim.h).  The constructors pack them on the host; each wrapper's ``refresh()`` re-packs them in place on the
device (evg_pack_mlp / _ppo / _rppo / _value) after an optimiser step.  Plumbing only; the networks themselves are the caller's.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi

IN_PAD, CHUNK, OUT_PAD, ATOM = _capi.MLP_IN_PAD, _capi.MLP_CHUNK, _capi.MLP_OUT_PAD, 64
PPO_IN_PAD, PPO_MAX_LATENT, PPO_OUT_PAD = _capi.PPO_IN_PAD, _capi.PPO_MAX_LATENT, _capi.PPO_OUT_PAD
VALUE_OUT_PAD = _capi.VALUE_OUT_PAD


def to_bf16_bits(x):
    """float32 array -> uint16 bf16 bit patterns, round to nearest even (what __float2bfloat16_rn does)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def bf16_round(x):
    """float32 array rounded to bf16 precision (as float32): the operands the kernel multiplies."""
    return (to_bf16_bits(x).astype(np.uint32) << 16).view(np.float32).reshape(np.shape(x))


def swz_offset(rows, r, k):
    """Byte offset of element (row r, column k) in a K-major [rows x K] bf16 block with the 128-byte swizzle."""
    return (k // ATOM) * rows * 128 + r * 128 + ((((k % ATOM) >> 3) ^ (r & 7)) << 4) + (k & 7) * 2


def _image(mat, rows, cols):
    """mat [<=rows, <=cols] float32 -> the uint8 image of a zero-padded [rows x cols] block."""
    full = np.zeros((rows, cols), dtype=np.float32)
    full[:mat.shape[0], :mat.shape[1]] = mat
    bits = to_bf16_bits(full)
    r, k = np.meshgrid(np.arange(rows), np.arange(cols), indexing="ij")
    img = np.zeros((cols // ATOM) * rows * 128 // 2, dtype=np.uint16)
    img[swz_offset(rows, r, k) // 2] = bits
    return img.view(np.uint8)


def pack_mlp(w1, b1, w2, b2):
    """w1 [hidden, in], b1 [hidden], w2 [out, hidden], b2 [out] (float32, torch.nn.Linear's layout) ->
    (w1_img uint8, w2_img uint8, hidden, out) as evg_policy_mlp expects them.  The biases ride inside the images:
    input feature `in` is the constant 1 (its weights are b1), hidden unit `hidden` is wired to relu(1) = 1 (its outgoing
    weights are b2)."""
    w1, b1, w2, b2 = (np.asarray(a, dtype=np.float32) for a in (w1, b1, w2, b2))
    hidden, in_dim = w1.shape
    out = w2.shape[0]
    assert in_dim < IN_PAD and out <= OUT_PAD and w2.shape[1] == hidden and b1.shape == (hidden,) and b2.shape == (out,)
    n_chunks = -(-(hidden + 1) // CHUNK)
    w1p = np.zeros((n_chunks * CHUNK, in_dim + 1), dtype=np.float32)
    w1p[:hidden, :in_dim] = w1
    w1p[:hidden, in_dim] = b1
    w1p[hidden, in_dim] = 1.0
    w2p = np.zeros((out, n_chunks * CHUNK), dtype=np.float32)
    w2p[:, :hidden] = w2
    w2p[:, hidden] = b2
    img1 = np.concatenate([_image(w1p[c * CHUNK:(c + 1) * CHUNK], CHUNK, IN_PAD) for c in range(n_chunks)])
    img2 = np.concatenate([_image(w2p[:, c * CHUNK:(c + 1) * CHUNK], OUT_PAD, CHUNK) for c in range(n_chunks)])
    return img1, img2, hidden, out


def reference_forward(obs, w1, b1, w2, b2):
    """What the kernel computes, in numpy: bf16-rounded operands (weights, biases, observations, hidden activations),
    float32 accumulation."""
    x = bf16_round(np.asarray(obs, dtype=np.float32))
    h = np.maximum(x @ bf16_round(w1).T + bf16_round(b1), 0.0).astype(np.float32)
    return bf16_round(h) @ bf16_round(w2).T + bf16_round(b2)


def _check_input_width(w1, env):
    """The kernels read env.obs_len features per row (and DQN's bias input sits right behind them): a first layer of
    another width would silently multiply the wrong columns."""
    if np.shape(w1)[1] != env.obs_len:
        raise ValueError("the network takes %d inputs, the environment's observations have %d values" % (np.shape(w1)[1], env.obs_len))


def _linear_params(net, n, expected):
    """(weight, bias) of each of the `n` nn.Linear layers of a Sequential, in order."""
    import torch
    lin = [m for m in net if isinstance(m, torch.nn.Linear)]
    assert len(lin) == n, "expected " + expected
    return [t for m in lin for t in (m.weight, m.bias)]


def _host_arrays(params):
    return [t.detach().float().cpu().numpy() for t in params]


def _refresh_sources(fused, net, params_of, shapes):
    """The parameters `refresh` packs from, as device pointers: ValueError, before anything is launched, unless each is
    a contiguous float32 tensor on the env's device of exactly the shape the wrapper's images were sized for."""
    import torch
    net = fused._net if net is None else net
    if net is None:
        raise ValueError("this wrapper was built from weights= arrays: pass the module to refresh(net)")
    params = params_of(net)
    env = fused.env
    for i, (t, shape) in enumerate(zip(params, shapes)):
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != env.device:
            raise ValueError("parameter %d must be a contiguous float32 tensor on %s, got %s%s on %s"
                             % (i, env.device, t.dtype, "" if t.is_contiguous() else " (not contiguous)", t.device))
        if tuple(t.shape) != shape:
            raise ValueError("parameter %d has shape %s, the wrapper's images were built for %s" % (i, tuple(t.shape), shape))
    return [C.c_void_p(t.data_ptr()) for t in params]


def _wire_rows(env, obs, obs_format):
    """The observations a fused policy reads: (format code, tensor).  'f32' is env.obs; 'wire' is env.obs_rows('wire'),
    or `obs` when given, a contiguous uint8 [num_envs, row_bytes] tensor on the env's device (ValueError otherwise, and
    for a map whose observations do not fit the kernels' 128 input columns, before anything is launched)."""
    import torch
    if obs_format not in ("f32", "wire"):
        raise ValueError("obs_format must be 'f32' or 'wire', got %r" % (obs_format,))
    if obs_format == "f32":
        return _capi.OBS_F32, obs
    if env.obs_len >= PPO_IN_PAD:
        raise ValueError("observations of %d values do not fit the %d input columns of the fused kernels" % (env.obs_len, PPO_IN_PAD))
    rb = int(env._lib.evg_obs_row_bytes(env._h, _capi.OBS_WIRE))
    if obs is None:
        return _capi.OBS_WIRE, env.obs_rows("wire")
    if not isinstance(obs, torch.Tensor) or obs.dtype != torch.uint8 or not obs.is_contiguous() or obs.device != env.device \
            or tuple(obs.shape) != (env.num_envs, rb):
        raise ValueError("wire rows must be a contiguous uint8 tensor of shape (%d, %d) on %s, got %s" % (
            env.num_envs, rb, env.device, "%s %s%s on %s" % (obs.dtype, tuple(obs.shape), "" if obs.is_contiguous() else " (not contiguous)",
                                                          obs.device) if isinstance(obs, torch.Tensor) else type(obs).__name__))
    return _capi.OBS_WIRE, obs


def _ptr(t, wanted):
    """An optional output of a fused actor: the tensor's address when it is asked for, else NULL (not written)."""
    return C.c_void_p(t.data_ptr()) if wanted else None


class FusedDQN:
    """Q-network forward + decode for a BatchedEvergladesEnv: ``actions = FusedDQN(env, net)()`` reads env.obs in place."""

    def __init__(self, env, net=None, weights=None):
        import torch
        self._net = net if weights is None else None
        if weights is None:
            weights = _host_arrays(self._params(net))
        _check_input_width(weights[0], env)
        img1, img2, self.hidden, self.out_dim = pack_mlp(*weights)
        self.env = env
        dev = env.device
        self._w1 = torch.from_numpy(img1).to(dev)
        self._w2 = torch.from_numpy(img2).to(dev)
        self.q = torch.empty((env.num_envs, 2, self.out_dim), dtype=torch.float32, device=dev)
        self.qt = torch.empty((self.out_dim, env.num_envs * 2), dtype=torch.float32, device=dev)

    @staticmethod
    def _params(net):
        return _linear_params(net, 2, "Sequential(Linear, ReLU, Linear)")

    def refresh(self, net=None):
        """Re-pack the weight images in place from `net` (default: the module this wrapper was built with), on the device:
        one kernel on the env's current stream, no allocation, no host synchronisation; the images are byte for byte
        those the constructor would build.  Call it after each optimiser step.  It can be captured in a CUDA graph, which
        then holds the parameters' addresses: it stays valid across in-place updates (optimizer.step(), load_state_dict),
        while replacing a parameter tensor needs a new capture.  The parameters must be contiguous float32 tensors on the
        env's device, of the shapes the wrapper was built with (ValueError otherwise, before anything is launched)."""
        h, o, w = self.hidden, self.out_dim, self.env.obs_len
        w1, b1, w2, b2 = _refresh_sources(self, net, self._params, [(h, w), (h,), (o, h), (o,)])
        env = self.env
        _capi.check(env._lib.evg_pack_mlp(env._h, w1, b1, w2, b2, h, o, C.c_void_p(self._w1.data_ptr()),
                                          C.c_void_p(self._w2.data_ptr()), env._stream()))

    def _run(self, obs, out, transposed, obs_format="f32"):
        env = self.env
        fmt, obs = _wire_rows(env, obs, obs_format)
        if obs is None:
            obs = env.obs
        elif fmt == _capi.OBS_F32:  # the kernel reads num_envs * 2 rows of obs_len float32 values from obs.data_ptr(), whatever obs is
            import torch
            if obs.dtype != torch.float32 or not obs.is_contiguous() or obs.device != env.device \
                    or obs.numel() != env.num_envs * 2 * env.obs_len:
                raise ValueError("obs must be a contiguous float32 tensor of %d x 2 x %d values on %s, got %s %s%s on %s"
                                 % (env.num_envs, env.obs_len, env.device, obs.dtype, tuple(obs.shape),
                                    "" if obs.is_contiguous() else " (not contiguous)", obs.device))
        _capi.check(env._lib.evg_policy_mlp_fmt(env._h, fmt, C.c_void_p(obs.data_ptr()), env.num_envs * 2, C.c_void_p(self._w1.data_ptr()),
                                                C.c_void_p(self._w2.data_ptr()), self.hidden, self.out_dim, C.c_void_p(out.data_ptr()),
                                                int(transposed), env._stream()))
        return out

    def forward(self, obs=None, obs_format="f32"):
        """Q-values float32 [N, 2, out] for `obs` (default: the environment's own observation tensor).  obs_format 'wire':
        the wire rows of env.obs_rows('wire'), or `obs` as uint8 [N, row_bytes] rows (e.g. a replay minibatch gathered
        with index_select); the Q-values are bit for bit those of the float32 observations the rows expand to."""
        return self._run(obs, self.q, False, obs_format)

    def forward_t(self, obs=None, obs_format="f32"):
        """The same Q-values transposed, float32 [out, N * 2]: what the decode reads coalesced."""
        return self._run(obs, self.qt, True, obs_format)

    def __call__(self, obs_format="f32"):
        """Action rows int8 [N, 2, 7, 2] for both players: forward, then DQNAgent.filter_actions on the device."""
        env = self.env
        qt = self.forward_t(obs_format=obs_format)
        assert self.out_dim % _capi.NUM_GROUPS == 0
        _capi.check(env._lib.evg_decode_dqn_layout(env._h, C.c_void_p(qt.data_ptr()), self.out_dim // _capi.NUM_GROUPS, -1, 1,
                                                   C.c_void_p(env._actions.data_ptr()), env._stream()))
        return env._actions


def pack_ppo(w1, b1, w2, b2, w3, b3):
    """w1 [L, in], b1 [L], w2 [L, L], b2 [L], w3 [out, L], b3 [out] (float32, torch.nn.Linear's layout) ->
    (w1_img, w2_img, w3_img uint8, bias float32, latent, out) as evg_policy_ppo expects them: W1 as an [Lp x 128] block,
    W2 as [Lp x Ka], W3 as [144 x Ka] (Lp = L rounded up to 16, Ka = L rounded up to 64), zero padded; the biases stay
    float32, b1 | b2 | b3 at 0, 256 and 512 of one zero-padded vector (the kernel adds them in fp32)."""
    w1, b1, w2, b2, w3, b3 = (np.asarray(a, dtype=np.float32) for a in (w1, b1, w2, b2, w3, b3))
    latent, in_dim = w1.shape
    out = w3.shape[0]
    assert in_dim < PPO_IN_PAD and 1 <= latent <= PPO_MAX_LATENT and 7 <= out <= PPO_OUT_PAD
    assert w2.shape == (latent, latent) and w3.shape[1] == latent and b1.shape == b2.shape == (latent,) and b3.shape == (out,)
    lp, ka = -(-latent // 16) * 16, -(-latent // ATOM) * ATOM
    bias = np.zeros(2 * PPO_MAX_LATENT + PPO_OUT_PAD, dtype=np.float32)
    bias[:latent] = b1
    bias[PPO_MAX_LATENT:PPO_MAX_LATENT + latent] = b2
    bias[2 * PPO_MAX_LATENT:2 * PPO_MAX_LATENT + out] = b3
    return _image(w1, lp, PPO_IN_PAD), _image(w2, lp, ka), _image(w3, PPO_OUT_PAD, ka), bias, latent, out


def reference_forward_ppo(obs, w1, b1, w2, b2, w3, b3):
    """What evg_policy_ppo computes, in numpy: bf16-rounded operands (observations, weights, both hidden activations),
    float32 accumulation, biases added in float32 (not rounded), y = tanh(z), probabilities exp(y) / sum(exp(y)) in
    float32.  Returns float32 [rows, out]."""
    f32 = np.float32
    x = bf16_round(np.asarray(obs, dtype=f32))
    h = np.tanh((x @ bf16_round(w1).T).astype(f32) + np.asarray(b1, f32)).astype(f32)
    h = np.tanh((bf16_round(h) @ bf16_round(w2).T).astype(f32) + np.asarray(b2, f32)).astype(f32)
    y = np.tanh((bf16_round(h) @ bf16_round(w3).T).astype(f32) + np.asarray(b3, f32)).astype(f32)
    e = np.exp(y).astype(f32)
    return (e / e.sum(axis=-1, dtype=f32, keepdims=True)).astype(f32)


def pack_value(w1, b1, w2, b2, w3, b3):
    """The critic's weights w1 [L, in], b1 [L], w2 [L, L], b2 [L], w3 [1, L], b3 [1] (float32, torch.nn.Linear's layout)
    -> (w1_img, w2_img, w3_img uint8, bias float32, latent) as evg_policy_value expects them: W1 and W2 exactly as
    pack_ppo packs them, w3 as row 0 of a zero [16 x Ka] block, b1 | b2 | b3 at 0, 256 and 512 of one zero-padded
    float32 vector of 528."""
    w1, b1, w2, b2, w3, b3 = (np.asarray(a, dtype=np.float32) for a in (w1, b1, w2, b2, w3, b3))
    latent, in_dim = w1.shape
    assert in_dim < PPO_IN_PAD and 1 <= latent <= PPO_MAX_LATENT
    assert w2.shape == (latent, latent) and w3.shape == (1, latent) and b1.shape == b2.shape == (latent,) and b3.shape == (1,)
    lp, ka = -(-latent // 16) * 16, -(-latent // ATOM) * ATOM
    bias = np.zeros(2 * PPO_MAX_LATENT + VALUE_OUT_PAD, dtype=np.float32)
    bias[:latent] = b1
    bias[PPO_MAX_LATENT:PPO_MAX_LATENT + latent] = b2
    bias[2 * PPO_MAX_LATENT] = b3[0]
    return _image(w1, lp, PPO_IN_PAD), _image(w2, lp, ka), _image(w3, VALUE_OUT_PAD, ka), bias, latent


def reference_forward_value(obs, w1, b1, w2, b2, w3, b3):
    """What evg_policy_value computes, in numpy: bf16-rounded operands (observations, W1, W2, w3, both hidden
    activations), float32 accumulation, b1, b2 and b3 added in float32 (not rounded), no tanh after the last layer.
    Returns float32 [rows]."""
    f32 = np.float32
    x = bf16_round(np.asarray(obs, dtype=f32))
    h = np.tanh((x @ bf16_round(w1).T).astype(f32) + np.asarray(b1, f32)).astype(f32)
    h = np.tanh((bf16_round(h) @ bf16_round(w2).T).astype(f32) + np.asarray(b2, f32)).astype(f32)
    v = (bf16_round(h) @ bf16_round(np.asarray(w3, f32)).T).astype(f32) + np.asarray(b3, f32)
    return v.astype(f32).reshape(-1)


class FusedPPO:
    """PPO actor forward + PPOAgent.get_action's sampling for a BatchedEvergladesEnv, in one kernel:
    ``actions = FusedPPO(env, net)()`` reads env.obs in place (or, with obs_format='wire', the env's wire rows) and
    writes env._actions.  The draws come from the tape (seed, global match id, turn, episode, player), not from torch's
    generator: the rows do not depend on batch size, sharding or call order.  `player` -1 plays both sides, 0 or 1 only
    that side's rows (the other side's rows are left as they are, e.g. for a scripted opponent)."""

    def __init__(self, env, net=None, weights=None, player=-1, latent=None, div=12, mod=11):
        import torch
        self._net = net if weights is None else None
        if weights is None:
            weights = _host_arrays(self._params(net))
        _check_input_width(weights[0], env)
        img1, img2, img3, bias, self.latent, self.out_dim = pack_ppo(*weights)
        assert latent is None or latent == self.latent, "latent %s != the weights' %d" % (latent, self.latent)
        assert player in (-1, 0, 1)
        self.env, self.player, self.div, self.mod = env, int(player), int(div), int(mod)
        dev = env.device
        self._w = [torch.from_numpy(a).to(dev) for a in (img1, img2, img3, bias)]
        shape = (env.num_envs, 2) if self.player < 0 else (env.num_envs,)
        self.idx = torch.empty(shape + (_capi.MAX_ACTIONS,), dtype=torch.int64, device=dev)
        self.probs = torch.empty(shape + (self.out_dim,), dtype=torch.float32, device=dev)
        self.logp = torch.empty(shape + (_capi.MAX_ACTIONS,), dtype=torch.float32, device=dev)

    @staticmethod
    def _params(net):
        return _linear_params(net, 3, "Sequential(Linear, Tanh, Linear, Tanh, Linear, Tanh, Softmax)")

    def refresh(self, net=None):
        """Re-pack the weight images and the bias vector in place from `net` (default: the module this wrapper was built
        with), on the device; see FusedDQN.refresh (CUDA graphs, the ValueError checks)."""
        L, o, w = self.latent, self.out_dim, self.env.obs_len
        src = _refresh_sources(self, net, self._params, [(L, w), (L,), (L, L), (L,), (o, L), (o,)])
        env = self.env
        w1, w2, w3, bias = (C.c_void_p(t.data_ptr()) for t in self._w)
        _capi.check(env._lib.evg_pack_ppo(env._h, *src, L, o, w1, w2, w3, bias, env._stream()))

    def evaluate(self, obs, obs_format="wire"):
        """The actor for a PPO update, on the tensor cores (evg_ppo_train_forward / _backward): stored observations, wire
        rows uint8 [M, row_bytes] ('wire') or float32 [M, 2, obs_len] ('f32'), -> z float32 [R, out], the output of the
        actor's last Linear before its Tanh (what env.ppo_loss takes), R = 2M rows ordered like .idx / .logp for player -1
        (row i = match i // 2, player i % 2), else M.  Differentiable with respect to the wrapped net's six parameters
        (autograd accumulates their .grad).  The arithmetic and the MMAs are the acting kernel's, so with the parameters
        the acting images were packed from, tanh(z) is what the acting call took its softmax of, bit for bit.  The net's
        current parameters are packed into images of this call's own (one device launch); the acting images stay the
        behaviour policy until refresh().  See _ff_evaluate for the backward and the ValueError checks."""
        L, o = self.latent, self.out_dim
        return _ff_evaluate(self, _capi.PPO_TRAIN_ACTOR, obs, obs_format, self.player, o, [(o, L), (o,)], self._params)

    def __call__(self, want_probs=False, obs_format="f32", want_logp=False):
        """Action rows int8 [N, 2, 7, 2] (env._actions); fills .idx (int64 [N, 2, 7] or [N, 7]) and, with want_probs,
        .probs (float32 [N, 2, out] or [N, out]).  With want_logp, .logp (float32 [N, 2, 7] or [N, 7]): draw k's
        log-probability log(p_j / T_k), T_k the sampler's float32 sum of the probabilities not drawn before it, so that
        .logp.sum(-1) is the log-probability of the ordered 7 draws without replacement (the behaviour policy's term of
        a PPO ratio).  No other output depends on want_probs / want_logp.  obs_format 'wire' reads env.obs_rows('wire')
        (the env stepped with obs_format='wire'), with results bit for bit those of the float32 observations."""
        env = self.env
        fmt, obs = _wire_rows(env, None, obs_format)
        obs = env.obs if obs is None else obs
        w1, w2, w3, bias = (C.c_void_p(t.data_ptr()) for t in self._w)
        _capi.check(env._lib.evg_policy_ppo_logp(env._h, fmt, C.c_void_p(obs.data_ptr()), self.player, w1, w2, w3, bias, self.latent,
                                                 self.out_dim, self.div, self.mod, C.c_void_p(env._actions.data_ptr()),
                                                 C.c_void_p(self.idx.data_ptr()), _ptr(self.probs, want_probs), _ptr(self.logp, want_logp),
                                                 env._stream()))
        return env._actions


def rppo_weights(actor):
    """(w1, b1, w2, b2, w_ih, b_ih, w_hh, b_hh, w3, b3) float32 numpy arrays of a module with the reference ActorCritic's
    action_head (Linear, Tanh, Linear, Tanh), action_gru and action_layer (Linear, Tanh, Softmax).  ValueError for a GRU
    the kernel does not run: more than one layer, bidirectional, an input width other than the hidden width, no biases."""
    return _host_arrays(_rppo_params(actor))


def _rppo_params(actor):
    """rppo_weights' parameters as the module's own tensors, after its checks."""
    import torch
    gru = actor.action_gru
    if gru.num_layers != 1 or gru.bidirectional or gru.input_size != gru.hidden_size or not gru.bias:
        raise ValueError("the fused recurrent actor runs one unidirectional GRU layer with biases and input width = hidden "
                         "width; got num_layers=%d bidirectional=%s input_size=%d hidden_size=%d bias=%s"
                         % (gru.num_layers, gru.bidirectional, gru.input_size, gru.hidden_size, gru.bias))
    head = [m for m in actor.action_head if isinstance(m, torch.nn.Linear)]
    out = [m for m in actor.action_layer if isinstance(m, torch.nn.Linear)]
    if len(head) != 2 or len(out) != 1:
        raise ValueError("expected action_head = (Linear, Tanh, Linear, Tanh) and action_layer = (Linear, Tanh, Softmax)")
    latent = gru.hidden_size
    if not 1 <= latent <= PPO_MAX_LATENT:
        raise ValueError("the GRU's width %d is outside 1..%d" % (latent, PPO_MAX_LATENT))
    if head[1].weight.shape[0] != latent:
        raise ValueError("the head's output width %d is not the GRU's %d" % (head[1].weight.shape[0], latent))
    return [head[0].weight, head[0].bias, head[1].weight, head[1].bias, gru.weight_ih_l0, gru.bias_ih_l0, gru.weight_hh_l0,
            gru.bias_hh_l0, out[0].weight, out[0].bias]


def pack_rppo(w1, b1, w2, b2, w_ih, b_ih, w_hh, b_hh, w3, b3):
    """The recurrent actor's weights (float32, torch's layouts: w_ih / w_hh [3L, L] and b_ih / b_hh [3L] with gates r, z, n
    as torch.nn.GRU's weight_ih_l0 ...) -> (w1_img, w2_img, wi_img, wh_img, w3_img uint8, bias float32, latent, out) as
    evg_policy_rppo expects them.  W1, W2, W3 and b1 | b2 | b3 are pack_ppo's; each GRU matrix is three [Lp x Ka] blocks,
    one per gate; b_ih gate g follows b3 at 656 + 256 g, b_hh gate g at 1424 + 256 g (include/evgsim.h)."""
    img1, img2, img3, bias, latent, out = pack_ppo(w1, b1, w2, b2, w3, b3)
    w_ih, b_ih, w_hh, b_hh = (np.asarray(a, dtype=np.float32) for a in (w_ih, b_ih, w_hh, b_hh))
    assert w_ih.shape == w_hh.shape == (3 * latent, latent) and b_ih.shape == b_hh.shape == (3 * latent,)
    lp, ka = -(-latent // 16) * 16, -(-latent // ATOM) * ATOM
    gates = [np.concatenate([_image(w[g * latent:(g + 1) * latent], lp, ka) for g in range(3)]) for w in (w_ih, w_hh)]
    gb = np.zeros(6 * PPO_MAX_LATENT, dtype=np.float32)
    for g in range(3):
        gb[g * PPO_MAX_LATENT:g * PPO_MAX_LATENT + latent] = b_ih[g * latent:(g + 1) * latent]
        gb[(3 + g) * PPO_MAX_LATENT:(3 + g) * PPO_MAX_LATENT + latent] = b_hh[g * latent:(g + 1) * latent]
    return img1, img2, gates[0], gates[1], img3, np.concatenate([bias, gb]), latent, out


def reference_forward_rppo(obs, h0, weights, bf16=True):
    """What evg_policy_rppo computes, in numpy: obs float32 [rows, in], h0 float32 [rows, L], weights as rppo_weights
    returns them -> (probs float32 [rows, 7, out], h float32 [rows, L]).  With bf16 the operands of every product are
    rounded to bf16 as the kernel's are (observations, weights, both head activations, h at each step), products
    accumulate in float32, and the biases, gate arithmetic and h stay float32; r and z add X W_i^T + H W_h^T first and
    then b_i + b_h, as the kernel's shared accumulator does.  Without bf16 it is plain float32 in torch.nn.GRU's order."""
    f32 = np.float32
    w1, b1, w2, b2, w_ih, b_ih, w_hh, b_hh, w3, b3 = (np.asarray(a, dtype=f32) for a in weights)
    rnd = bf16_round if bf16 else (lambda v: np.asarray(v, dtype=f32))
    latent = w1.shape[0]

    def sig(v):
        return (f32(1) / (f32(1) + np.exp(-v))).astype(f32)

    a1 = np.tanh((rnd(obs) @ rnd(w1).T).astype(f32) + b1).astype(f32)
    x = rnd(np.tanh((rnd(a1) @ rnd(w2).T).astype(f32) + b2).astype(f32))
    gi = (x @ rnd(w_ih).T).astype(f32)  # the same every step
    h = np.array(h0, dtype=f32)
    probs = []
    for _ in range(7):
        gh = (rnd(h) @ rnd(w_hh).T).astype(f32)
        s = slice(0, latent), slice(latent, 2 * latent), slice(2 * latent, 3 * latent)
        if bf16:
            r = sig((gi[:, s[0]] + gh[:, s[0]]) + (b_ih[s[0]] + b_hh[s[0]]))
            z = sig((gi[:, s[1]] + gh[:, s[1]]) + (b_ih[s[1]] + b_hh[s[1]]))
        else:
            r = sig(gi[:, s[0]] + b_ih[s[0]] + gh[:, s[0]] + b_hh[s[0]])
            z = sig(gi[:, s[1]] + b_ih[s[1]] + gh[:, s[1]] + b_hh[s[1]])
        n = np.tanh((gi[:, s[2]] + b_ih[s[2]]) + r * (gh[:, s[2]] + b_hh[s[2]])).astype(f32)
        h = ((f32(1) - z) * n + z * h).astype(f32)
        e = np.exp(np.tanh((rnd(h) @ rnd(w3).T).astype(f32) + b3)).astype(f32)
        probs.append((e / e.sum(axis=-1, dtype=f32, keepdims=True)).astype(f32))
    return np.stack(probs, axis=1), h


class FusedRPPO:
    """PPO's recurrent actor + its 7 draws for a BatchedEvergladesEnv, in one kernel: ``actions = FusedRPPO(env, actor)()``
    reads env.obs in place (or, with obs_format='wire', the env's wire rows), steps the GRU state ``.hidden`` and writes
    env._actions.  ``.hidden`` (float32 [N, 2, L], or [N, L] for one player; zero at construction) is read and written
    back by every call, and a row restarts from zero when its match's record is at turn 0 (after reset() and after an
    automatic reset): under AUTORESET_TERMINAL / _NEXT that is the ``hidden *= 1 - done`` mask of a torch rollout.  Under
    AUTORESET_OFF a finished match keeps its state until it is reset.  Step k draws one index from its distribution with
    replacement (ActorCritic.act: one torch.multinomial(probs, 1) per step), keyed on the tape as FusedPPO's draws.
    `player` -1 plays both sides, 0 or 1 only that side's rows."""

    def __init__(self, env, actor, player=-1, div=12, mod=11):
        import torch
        weights = rppo_weights(actor)
        self._net = actor
        _check_input_width(weights[0], env)
        if player not in (-1, 0, 1):
            raise ValueError("player must be -1, 0 or 1, got %r" % (player,))
        img1, img2, imgi, imgh, img3, bias, self.latent, self.out_dim = pack_rppo(*weights)
        self.env, self.player, self.div, self.mod = env, int(player), int(div), int(mod)
        dev = env.device
        self._w = [torch.from_numpy(a).to(dev) for a in (img1, img2, imgi, imgh, img3, bias)]
        shape = (env.num_envs, 2) if self.player < 0 else (env.num_envs,)
        self.hidden = torch.zeros(shape + (self.latent,), dtype=torch.float32, device=dev)
        self.idx = torch.empty(shape + (_capi.MAX_ACTIONS,), dtype=torch.int64, device=dev)
        self.probs = torch.empty(shape + (_capi.MAX_ACTIONS, self.out_dim), dtype=torch.float32, device=dev)
        self.logp = torch.empty(shape + (_capi.MAX_ACTIONS,), dtype=torch.float32, device=dev)
        self.hidden_in = torch.zeros_like(self.hidden)
        self._t = None

    def refresh(self, actor=None):
        """Re-pack the weight images and the bias vector in place from `actor` (default: the module this wrapper was built
        with), on the device; .hidden is left as it is.  ValueError for a GRU the kernel does not run (as the constructor),
        otherwise as FusedDQN.refresh (CUDA graphs, the checks)."""
        L, o, w = self.latent, self.out_dim, self.env.obs_len
        w1, b1, w2, b2, wi, bi, wh, bh, w3, b3 = _refresh_sources(
            self, actor, _rppo_params, [(L, w), (L,), (L, L), (L,), (3 * L, L), (3 * L,), (3 * L, L), (3 * L,), (o, L), (o,)])
        env = self.env
        i1, i2, ii, ih, i3, bias = (C.c_void_p(t.data_ptr()) for t in self._w)
        _capi.check(env._lib.evg_pack_rppo(env._h, w1, b1, w2, b2, w3, b3, wi, bi, wh, bh, L, o, i1, i2, ii, ih, i3, bias,
                                           env._stream()))

    def evaluate(self, x, hidden_in):
        """The GRU's 7 steps and action_layer[0] for a PPO update, on the tensor cores (evg_rppo_train_forward / _backward):
        x float32 [R, L], the action head's output, and hidden_in float32 [R, L], the state each stored row started from
        (the acting call's .hidden_in) -> z float32 [R, 7, out], step k's output of action_layer[0] before its Tanh, as
        env.ppo_loss takes it with K = 7.  Differentiable with respect to x and the wrapped actor's weight_ih_l0,
        weight_hh_l0, bias_ih_l0, bias_hh_l0, action_layer[0].weight and .bias (autograd accumulates their .grad); no
        gradient flows to hidden_in.  The arithmetic is the acting kernel's (bf16 operands, fp32 accumulation and gates),
        so from the same x and state h_7 is what an acting call leaves in .hidden.  The actor's current parameters are
        packed into images of this call's own (one device launch); the acting images stay as they are until refresh().
        The backward's weight-gradient reductions are float32 torch.matmul calls on what the kernel writes (torch's
        default precision: TF32 is used only where the caller enabled it).  ValueError, before any launch, for a tensor
        of the wrong dtype, shape, device or contiguity; R = 0 gives an empty tensor.  No host synchronisation."""
        import torch
        env, L, o = self.env, self.latent, self.out_dim
        for name, t in (("x", x), ("hidden_in", hidden_in)):
            if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or not t.is_contiguous() or t.device != env.device \
                    or t.dim() != 2 or t.shape[1] != L:
                raise ValueError("%s must be a contiguous float32 tensor [R, %d] on %s, got %s" % (name, L, env.device, _describe(t)))
        if hidden_in.shape != x.shape:
            raise ValueError("hidden_in has %d rows, x has %d" % (hidden_in.shape[0], x.shape[0]))
        params = _rppo_params(self._net)
        for i, (t, shape) in enumerate(zip(params, [(L, env.obs_len), (L,), (L, L), (L,), (3 * L, L), (3 * L,), (3 * L, L), (3 * L,), (o, L), (o,)])):
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != env.device or tuple(t.shape) != shape:
                raise ValueError("parameter %d must be a contiguous float32 tensor of shape %s on %s, got %s" % (i, shape, env.device, _describe(t)))
        if x.shape[0] == 0:
            return torch.empty((0, _capi.MAX_ACTIONS, o), dtype=torch.float32, device=env.device)
        return _rppo_train_function().apply(x, hidden_in, self, *params[4:])

    def evaluate_head(self, obs, obs_format="wire"):
        """The action head for a PPO update, on the tensor cores (evg_ppo_train_forward / _backward): stored observations,
        wire rows uint8 [M, row_bytes] ('wire') or float32 [M, 2, obs_len] ('f32'), -> x float32 [R, L] = tanh(W2
        bf16(tanh(W1 bf16(obs) + b1)) + b2), rows ordered like .idx / .hidden_in, ready for evaluate(x, hidden_in).
        Differentiable with respect to action_head's four parameters.  bf16(x) is the operand the acting kernel's GRU
        read, bit for bit, so from the acting call's .hidden_in, evaluate's h_7 is what that call left in .hidden.  See
        _ff_evaluate for the images, the backward and the ValueError checks."""
        return _ff_evaluate(self, _capi.PPO_TRAIN_HEAD, obs, obs_format, self.player, self.latent, [],
                            lambda actor: _rppo_params(actor)[:4])

    def _train_images(self):
        """The training images (wi, wh, wht, w3 uint8, bias float32), allocated on first use."""
        import torch
        if self._t is None:
            lp, ka = -(-self.latent // 16) * 16, -(-self.latent // ATOM) * ATOM
            dev = self.env.device
            gate_bytes = 3 * (ka // ATOM) * lp * 128
            self._t = [torch.empty(gate_bytes, dtype=torch.uint8, device=dev) for _ in range(3)]
            self._t.append(torch.empty((ka // ATOM) * PPO_OUT_PAD * 128, dtype=torch.uint8, device=dev))
            self._t.append(torch.empty(PPO_OUT_PAD + 6 * PPO_MAX_LATENT, dtype=torch.float32, device=dev))
        return self._t

    def _train_forward(self, x, h0, w_ih, b_ih, w_hh, b_hh, w3, b3, z, h):
        env, p = self.env, (lambda t: C.c_void_p(t.data_ptr()))
        wi, wh, wht, i3, bias = (p(t) for t in self._train_images())
        _capi.check(env._lib.evg_rppo_train_pack(env._h, p(w3), p(b3), p(w_ih), p(b_ih), p(w_hh), p(b_hh), self.latent, self.out_dim,
                                                 wi, wh, wht, i3, bias, env._stream()))
        _capi.check(env._lib.evg_rppo_train_forward(env._h, x.shape[0], self.latent, self.out_dim, p(x), p(h0), wi, wh, i3, bias, p(z), p(h),
                                                    env._stream()))

    def _train_backward(self, x, h0, h, g, dgh, s):
        env, p = self.env, (lambda t: C.c_void_p(t.data_ptr()))
        wi, wh, wht, _, bias = (p(t) for t in self._train_images())
        _capi.check(env._lib.evg_rppo_train_backward(env._h, x.shape[0], self.latent, self.out_dim, p(x), p(h0), p(h), wi, wh, wht, bias,
                                                     p(g), p(dgh), p(s), env._stream()))

    def __call__(self, want_probs=False, obs_format="f32", want_logp=False, want_hidden_in=False):
        """Action rows int8 [N, 2, 7, 2] (env._actions); steps .hidden, fills .idx (int64 [N, 2, 7] or [N, 7]) and, with
        want_probs, .probs (float32 [N, 2, 7, out] or [N, 7, out]: step k's distribution).  With want_logp, .logp
        (float32 [N, 2, 7] or [N, 7]): step k's log(p_k[j] / T_k), T_k the sampler's float32 sum of p_k.  With
        want_hidden_in, .hidden_in (.hidden's shape): the state each row started this call from (zero for a row whose
        match is at turn 0), which is what a PPO update re-evaluates the stored turn from.  No other output depends on
        want_probs / want_logp / want_hidden_in.  obs_format 'wire' reads env.obs_rows('wire'), as FusedPPO does."""
        env = self.env
        fmt, obs = _wire_rows(env, None, obs_format)
        obs = env.obs if obs is None else obs
        w1, w2, wi, wh, w3, bias = (C.c_void_p(t.data_ptr()) for t in self._w)
        _capi.check(env._lib.evg_policy_rppo_logp(env._h, fmt, C.c_void_p(obs.data_ptr()), self.player, w1, w2, wi, wh, w3, bias, self.latent,
                                                  self.out_dim, self.div, self.mod, C.c_void_p(self.hidden.data_ptr()),
                                                  _ptr(self.hidden_in, want_hidden_in), C.c_void_p(env._actions.data_ptr()),
                                                  C.c_void_p(self.idx.data_ptr()), _ptr(self.probs, want_probs), _ptr(self.logp, want_logp),
                                                  env._stream()))
        return env._actions


_RPPO_TRAIN = None


def _rppo_train_function():
    """The torch.autograd.Function of FusedRPPO.evaluate (defined on first use: torch is imported lazily)."""
    global _RPPO_TRAIN
    if _RPPO_TRAIN is None:
        import torch

        def bf16(t):
            return t.to(torch.bfloat16).to(torch.float32)

        class RPPOTrain(torch.autograd.Function):
            @staticmethod
            def forward(ctx, x, hidden_in, fused, w_ih, b_ih, w_hh, b_hh, w3, b3):
                R, L = x.shape
                z = torch.empty((R, _capi.MAX_ACTIONS, fused.out_dim), dtype=torch.float32, device=x.device)
                h = torch.empty((R, _capi.MAX_ACTIONS, L), dtype=torch.float32, device=x.device)
                fused._train_forward(x, hidden_in, w_ih, b_ih, w_hh, b_hh, w3, b3, z, h)
                ctx.save_for_backward(x, hidden_in, h, w_ih, w_hh, w3)
                ctx.fused = fused
                return z

            @staticmethod
            def backward(ctx, dz):
                x, h0, h, w_ih, w_hh, w3 = ctx.saved_tensors
                R, L = x.shape
                K, o = _capi.MAX_ACTIONS, w3.shape[0]
                dz = dz.to(torch.float32).contiguous().view(R * K, o)
                g = (dz @ bf16(w3)).view(R, K, L)  # W3^T dz_k; the kernel adds the carries in place
                dgh = torch.empty((R, K, 3 * L), dtype=torch.float32, device=x.device)
                s = torch.empty((R, 3 * L), dtype=torch.float32, device=x.device)
                ctx.fused._train_backward(x, h0, h, g, dgh, s)
                dgh = dgh.view(R * K, 3 * L)
                h_prev = bf16(torch.cat([h0.unsqueeze(1), h[:, :K - 1]], dim=1)).view(R * K, L)
                return (s @ bf16(w_ih), None, None, s.t() @ bf16(x), s.sum(0), dgh.t() @ h_prev, dgh.sum(0),
                        dz.t() @ bf16(h).view(R * K, L), dz.sum(0))

        _RPPO_TRAIN = RPPOTrain
    return _RPPO_TRAIN


def _value_params(net):
    """The critic's (w1, b1, w2, b2, w3, b3) tensors of a Sequential(Linear, Tanh, Linear, Tanh, Linear(L, 1));
    ValueError for another layer count or a last layer that is not Linear(L, 1)."""
    import torch
    lin = [m for m in net if isinstance(m, torch.nn.Linear)]
    if len(lin) != 3:
        raise ValueError("expected Sequential(Linear, Tanh, Linear, Tanh, Linear(L, 1)), got %d Linear layers" % len(lin))
    if lin[2].out_features != 1:
        raise ValueError("the critic's last layer must be Linear(L, 1), got Linear(%d, %d)" % (lin[2].in_features, lin[2].out_features))
    return [t for m in lin for t in (m.weight, m.bias)]


class FusedValue:
    """PPO's critic for a BatchedEvergladesEnv, in one kernel: ``v = FusedValue(env, net)()`` is V of env.obs (float32
    [N, 2] for player -1, [N] for player 0 or 1), written into ``.value``.  Called with stored rows it evaluates any
    number M of matches in one launch: wire rows uint8 [M, row_bytes] or float32 observations [M, 2, obs_len] -> [M, 2]
    (or [M]), e.g. a whole [T, N] rollout flattened.  bf16 operands and fp32 accumulation like the actors
    (reference_forward_value); like FusedPPO.logp, values agree with a float32 torch critic to bf16 accuracy only."""

    def __init__(self, env, net=None, weights=None, player=-1):
        import torch
        self._net = net if weights is None else None
        if weights is None:
            weights = _host_arrays(_value_params(net))
        if len(weights) != 6:
            raise ValueError("expected the 6 arrays (w1, b1, w2, b2, w3, b3), got %d" % len(weights))
        _check_input_width(weights[0], env)
        L = np.shape(weights[0])[0]
        if not 1 <= L <= PPO_MAX_LATENT:
            raise ValueError("the critic's width %d is outside 1..%d" % (L, PPO_MAX_LATENT))
        shapes = [(L, env.obs_len), (L,), (L, L), (L,), (1, L), (1,)]
        for i, (w, shape) in enumerate(zip(weights, shapes)):
            if np.shape(w) != shape:
                raise ValueError("parameter %d has shape %s, a critic of width %d needs %s (the last layer is Linear(L, 1))"
                                 % (i, np.shape(w), L, shape))
        if player not in (-1, 0, 1):
            raise ValueError("player must be -1, 0 or 1, got %r" % (player,))
        if env.obs_len >= PPO_IN_PAD:
            raise ValueError("observations of %d values do not fit the %d input columns of the fused kernels" % (env.obs_len, PPO_IN_PAD))
        img1, img2, img3, bias, self.latent = pack_value(*weights)
        self.env, self.player = env, int(player)
        dev = env.device
        self._w = [torch.from_numpy(a).to(dev) for a in (img1, img2, img3, bias)]
        self.value = torch.empty(self._shape(env.num_envs), dtype=torch.float32, device=dev)

    def _shape(self, m):
        return (m, 2) if self.player < 0 else (m,)

    def refresh(self, net=None):
        """Re-pack the weight images and the bias vector in place from `net` (default: the module this wrapper was built
        with), on the device; see FusedDQN.refresh (CUDA graphs, the ValueError checks)."""
        L, w = self.latent, self.env.obs_len
        src = _refresh_sources(self, net, _value_params, [(L, w), (L,), (L, L), (L,), (1, L), (1,)])
        env = self.env
        i1, i2, i3, bias = (C.c_void_p(t.data_ptr()) for t in self._w)
        _capi.check(env._lib.evg_pack_value(env._h, *src, L, i1, i2, i3, bias, env._stream()))

    def evaluate(self, obs, obs_format="wire"):
        """The critic for a PPO update, on the tensor cores (evg_ppo_train_forward / _backward): stored observations, wire
        rows uint8 [M, row_bytes] ('wire') or float32 [M, 2, obs_len] ('f32'), -> V float32 [M, 2] (player -1) or [M],
        bit for bit what self(obs, obs_format) gives with the acting images packed from the same parameters.
        Differentiable with respect to the wrapped net's six parameters.  See _ff_evaluate for the images, the backward
        and the ValueError checks."""
        L = self.latent
        return _ff_evaluate(self, _capi.PPO_TRAIN_CRITIC, obs, obs_format, self.player, 1, [(1, L), (1,)], _value_params)

    def __call__(self, obs=None, obs_format="f32", out=None):
        """State values float32 [M, 2] (player -1) or [M].  obs None: the env's own observations (M = num_envs; 'wire'
        reads env.obs_rows('wire'), the env stepped with obs_format='wire'), into .value unless `out` is given.
        Otherwise `obs` is float32 [M, 2, obs_len] ('f32') or uint8 wire rows [M, row_bytes] ('wire'), contiguous on the
        env's device, and the values go to `out` (allocated when None).  Wire rows give bit for bit the values of the
        float32 observations they expand to.  ValueError, before anything is launched, for another format (the kernels
        read no 'i16'), a tensor of the wrong dtype, shape or device, or one that is not contiguous."""
        import torch
        env = self.env
        if obs_format not in ("f32", "wire"):
            raise ValueError("obs_format must be 'f32' or 'wire', got %r" % (obs_format,))
        fmt = _capi.OBS_F32 if obs_format == "f32" else _capi.OBS_WIRE
        if obs is None:
            obs = env.obs if fmt == _capi.OBS_F32 else env.obs_rows("wire")
            m = env.num_envs
            out = self.value if out is None else out
        else:
            if fmt == _capi.OBS_F32:
                dtype, tail, what = torch.float32, (2, env.obs_len), "float32 observations [M, 2, %d]" % env.obs_len
            else:
                rb = int(env._lib.evg_obs_row_bytes(env._h, _capi.OBS_WIRE))
                dtype, tail, what = torch.uint8, (rb,), "uint8 wire rows [M, %d]" % rb
            if not isinstance(obs, torch.Tensor) or obs.dtype != dtype or not obs.is_contiguous() or obs.device != env.device \
                    or obs.dim() != 1 + len(tail) or tuple(obs.shape[1:]) != tail:
                raise ValueError("obs must be contiguous %s on %s, got %s" % (what, env.device, _describe(obs)))
            m = obs.shape[0]
            if out is None:
                out = torch.empty(self._shape(m), dtype=torch.float32, device=env.device)
        if not isinstance(out, torch.Tensor) or out.dtype != torch.float32 or not out.is_contiguous() or out.device != env.device \
                or tuple(out.shape) != self._shape(m):
            raise ValueError("out must be a contiguous float32 tensor of shape %s on %s, got %s" % (self._shape(m), env.device, _describe(out)))
        if m == 0:
            return out
        i1, i2, i3, bias = (C.c_void_p(t.data_ptr()) for t in self._w)
        _capi.check(env._lib.evg_policy_value(env._h, fmt, C.c_void_p(obs.data_ptr()), m, self.player, i1, i2, i3, bias, self.latent,
                                              C.c_void_p(out.data_ptr()), env._stream()))
        return out


def _ff_evaluate(fused, net, obs, obs_format, player, out_dim, last_shapes, params_of):
    """FusedPPO.evaluate, FusedValue.evaluate and FusedRPPO.evaluate_head: the network `net` (_capi.PPO_TRAIN_*) of the
    wrapper's module on stored observations.  ValueError, before any launch, for a wrapper built from weights= (no module
    to differentiate), an obs_format other than 'wire' or 'f32' (the kernels read no 'i16'), observations of the wrong
    dtype, shape, device or contiguity, and parameters that are not contiguous float32 tensors on the env's device of the
    wrapper's shapes.  M = 0 gives an empty tensor.  No host synchronisation: the call can be captured in a CUDA graph.

    The forward packs the current parameters (evg_ppo_train_pack) and runs evg_ppo_train_forward, which also writes h1 and
    h2.  The backward computes g2 = dL/dh2 in float32 torch (dz bf16(W3), dv bf16(w3) or the upstream dx), runs
    evg_ppo_train_backward for dD2 and dD1, and reduces the parameter gradients with float32 torch.matmul / sum on what
    the kernels wrote (torch's default precision: TF32 only where the caller enabled it): dW3 = dz^T bf16(h2), dW2 =
    dD2^T bf16(h1), dW1 = dD1^T bf16(obs), the biases' the column sums.  Wire rows are expanded for dW1 on the device
    (env.expand_wire).  No gradient flows to the observations.  The backward reads the wrapper's one W2^T image, packed
    by the latest call: W2 is saved for backward, so changing it in place between a call and its backward (an
    optimiser step under retain_graph) raises torch's version-counter error instead of using the newer W2; W3 is
    saved for the same reason.  Several calls with unchanged parameters may be backpropagated in any order."""
    import torch
    env = fused.env
    if fused._net is None:
        raise ValueError("this wrapper was built from weights= arrays: it has no module to differentiate")
    if obs_format not in ("f32", "wire"):
        raise ValueError("obs_format must be 'f32' or 'wire', got %r" % (obs_format,))
    if env.obs_len >= PPO_IN_PAD:
        raise ValueError("observations of %d values do not fit the %d input columns of the fused kernels" % (env.obs_len, PPO_IN_PAD))
    if obs_format == "f32":
        fmt, dtype, tail, what = _capi.OBS_F32, torch.float32, (2, env.obs_len), "float32 observations [M, 2, %d]" % env.obs_len
    else:
        rb = int(env._lib.evg_obs_row_bytes(env._h, _capi.OBS_WIRE))
        fmt, dtype, tail, what = _capi.OBS_WIRE, torch.uint8, (rb,), "uint8 wire rows [M, %d]" % rb
    if not isinstance(obs, torch.Tensor) or obs.dtype != dtype or not obs.is_contiguous() or obs.device != env.device \
            or obs.dim() != 1 + len(tail) or tuple(obs.shape[1:]) != tail:
        raise ValueError("obs must be contiguous %s on %s, got %s" % (what, env.device, _describe(obs)))
    L = fused.latent
    params = params_of(fused._net)
    for i, (t, shape) in enumerate(zip(params, [(L, env.obs_len), (L,), (L, L), (L,)] + last_shapes)):
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != env.device or tuple(t.shape) != shape:
            raise ValueError("parameter %d must be a contiguous float32 tensor of shape %s on %s, got %s" % (i, shape, env.device, _describe(t)))
    rows = obs.shape[0] * (2 if player < 0 else 1)
    if obs.shape[0] == 0:
        shape = {_capi.PPO_TRAIN_ACTOR: (0, out_dim), _capi.PPO_TRAIN_HEAD: (0, L)}.get(net, (0, 2) if player < 0 else (0,))
        return torch.empty(shape, dtype=torch.float32, device=env.device)
    y = _ff_train_function().apply(obs, fused, net, fmt, player, out_dim, *params)
    return y.view(-1, 2) if net == _capi.PPO_TRAIN_CRITIC and player < 0 else y


def _ff_train_images(fused, net):
    """The training images of a wrapper (w1, w2, w3, w2t uint8, bias float32; w3 empty for the head), allocated on first use."""
    import torch
    if getattr(fused, "_ft", None) is None:
        lp, ka = -(-fused.latent // 16) * 16, -(-fused.latent // ATOM) * ATOM
        dev = fused.env.device
        w3_rows = {_capi.PPO_TRAIN_ACTOR: PPO_OUT_PAD, _capi.PPO_TRAIN_CRITIC: VALUE_OUT_PAD}.get(net, 0)
        b3 = {_capi.PPO_TRAIN_ACTOR: PPO_OUT_PAD, _capi.PPO_TRAIN_CRITIC: VALUE_OUT_PAD}.get(net, 0)
        fused._ft = [torch.empty(n, dtype=torch.uint8, device=dev)
                     for n in ((PPO_IN_PAD // ATOM) * lp * 128, (ka // ATOM) * lp * 128, max(1, (ka // ATOM) * w3_rows * 128), (ka // ATOM) * lp * 128)]
        fused._ft.append(torch.empty(2 * PPO_MAX_LATENT + b3, dtype=torch.float32, device=dev))
    return fused._ft


_FF_TRAIN = None


def _ff_train_function():
    """The torch.autograd.Function of _ff_evaluate (defined on first use: torch is imported lazily)."""
    global _FF_TRAIN
    if _FF_TRAIN is None:
        import torch

        def bf16(t):
            return t.to(torch.bfloat16).to(torch.float32)

        def p(t):
            return C.c_void_p(t.data_ptr()) if t is not None else None

        class FFTrain(torch.autograd.Function):
            @staticmethod
            def forward(ctx, obs, fused, net, fmt, player, out_dim, w1, b1, w2, b2, w3=None, b3=None):
                env, L = fused.env, fused.latent
                R = obs.shape[0] * (2 if player < 0 else 1)
                i1, i2, i3, i2t, bias = _ff_train_images(fused, net)
                head = net == _capi.PPO_TRAIN_HEAD
                _capi.check(env._lib.evg_ppo_train_pack(env._h, net, p(w1), p(b1), p(w2), p(b2), p(w3), p(b3), L, out_dim, p(i1), p(i2),
                                                        None if head else p(i3), p(i2t), p(bias), env._stream()))
                h1 = torch.empty((R, L), dtype=torch.float32, device=obs.device)
                h2 = torch.empty((R, L), dtype=torch.float32, device=obs.device)
                out = None if head else torch.empty((R, out_dim) if net == _capi.PPO_TRAIN_ACTOR else (R,), dtype=torch.float32, device=obs.device)
                _capi.check(env._lib.evg_ppo_train_forward(env._h, net, fmt, p(obs), obs.shape[0], player, L, out_dim, p(i1), p(i2),
                                                           None if head else p(i3), p(bias), p(out), p(h1), p(h2), env._stream()))
                # w2 is saved for its version counter: the backward reads the wrapper's W2^T image, which the next
                # evaluate re-packs, so a parameter changed in place in between must raise, as torch's own layers do
                ctx.save_for_backward(obs, h1, h2, w2, w3)
                ctx.fused, ctx.net, ctx.fmt, ctx.player = fused, net, fmt, player
                return h2 if head else out

            @staticmethod
            def backward(ctx, dy):
                obs, h1, h2, _, w3 = ctx.saved_tensors
                fused, net, player = ctx.fused, ctx.net, ctx.player
                env, (R, L) = fused.env, h1.shape
                dy = dy.to(torch.float32).reshape(R, -1).contiguous()
                if net == _capi.PPO_TRAIN_ACTOR:
                    g2 = dy @ bf16(w3)
                elif net == _capi.PPO_TRAIN_CRITIC:
                    g2 = dy * bf16(w3)  # [R, 1] x [1, L]: dv_i w3_j
                else:
                    g2 = dy
                g2 = g2.contiguous()
                dd2 = torch.empty_like(h1)
                dd1 = torch.empty_like(h1)
                _capi.check(env._lib.evg_ppo_train_backward(env._h, R, L, p(_ff_train_images(fused, net)[3]), p(g2), p(h1), p(h2), p(dd2), p(dd1),
                                                            env._stream()))
                if ctx.fmt == _capi.OBS_WIRE:
                    x = env.expand_wire(obs, player=player)
                else:
                    x = obs if player < 0 else obs[:, player]
                x = bf16(x.reshape(R, env.obs_len))
                grads = [dd1.t() @ x, dd1.sum(0), dd2.t() @ bf16(h1), dd2.sum(0)]
                if net != _capi.PPO_TRAIN_HEAD:
                    grads += [dy.t() @ bf16(h2), dy.sum(0)]
                return (None,) * 6 + tuple(grads)

        _FF_TRAIN = FFTrain
    return _FF_TRAIN


def _describe(t):
    import torch
    if not isinstance(t, torch.Tensor):
        return type(t).__name__
    return "%s %s%s on %s" % (t.dtype, tuple(t.shape), "" if t.is_contiguous() else " (not contiguous)", t.device)
