"""Host-side mirror of the reference's gym wrapper on top of libevgsim (CUDA, sm_100a).

``EvergladesEnv``         — same attributes, ``reset(**kwargs)`` / ``step(actions)`` signatures, dict-in
                            / dict-out types and error behaviour as
                            gym_everglades/envs/everglades_env.py:13-116, for ONE match (N = 1).
``BatchedEvergladesEnv``  — N matches in lockstep on one GPU; tensors in, tensors out.

PyTorch is plumbing only (device memory, streams); every game rule runs in the kernels of
csrc/evg_kernels.cu through the C ABI of include/evgsim.h.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi
from .config import load_config, UNIT_CLASSES, MAX_SCORE  # noqa: F401  (MAX_SCORE re-exported, env.py:11)


def _torch():
    import torch
    return torch


OBS_FORMATS = {"f32": _capi.OBS_F32, "i16": _capi.OBS_I16, "wire": _capi.OBS_WIRE}


class BatchedEvergladesEnv:
    """N Everglades matches stepped in lockstep by one CUDA launch per turn.

    Shapes (L = obs_len = 1 + 4*num_nodes + 60; 105 on DemoMap):
        actions int8    [N, 2, 7, 2]   (group id, node id in the acting player's own numbering)
        obs     float32 [N, 2, L]      layout of env.py:158-171 (board_state[0:45] ++ player_state[1:61])
        reward  float32 [N, 2]         env.py:37-60
        done    uint8   [N]            status != 0 (server.py:321-328)
    Output tensors are allocated once and overwritten in place by every call.
    """

    def __init__(self, num_envs, device=0, seed=0, config_dir=None, map_file="DemoMap.json",
                 unit_file="UnitDefinitions.json", setup_file="GameSetup.json", auto_reset=_capi.AUTORESET_OFF,
                 env_id_offset=0, config=None):
        torch = _torch()
        self._lib = _capi.load()
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedEvergladesEnv needs a CUDA device: the game step has no CPU implementation")
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.cfg = config if config is not None else load_config(config_dir, map_file, unit_file, setup_file, auto_reset)
        if config is not None:
            self.cfg.auto_reset = int(auto_reset) if auto_reset is not None else self.cfg.auto_reset
        self.num_envs = int(num_envs)
        self.seed = int(seed)
        self.env_id_offset = int(env_id_offset)
        self._h = C.c_void_p()
        _capi.check(self._lib.evg_create(C.byref(self.cfg), self.num_envs, self.seed, self.env_id_offset, dev_index,
                                         C.byref(self._h)))
        lay = _capi.EvgLayout()
        _capi.check(self._lib.evg_layout(self._h, C.byref(lay)))
        self.layout = lay
        self.obs_len = int(lay.obs_len)
        # reference attributes (env.py:17-22)
        self.num_turns = int(self.cfg.turn_limit)
        self.num_groups = _capi.NUM_GROUPS
        self.num_nodes = int(self.cfg.n_nodes)
        self.num_units = int(sum(self.cfg.group_size[0]))
        self.num_actions_per_turn = _capi.MAX_ACTIONS
        self.unit_classes = list(UNIT_CLASSES)
        N = self.num_envs
        with torch.cuda.device(self.device):
            # resident state: owned here, only ever touched by the kernels
            self._records = torch.empty(lay.records_bytes, dtype=torch.uint8, device=self.device)
            self._health = torch.empty(lay.health_bytes // 8, dtype=torch.float64, device=self.device)
            self._stats = torch.zeros(lay.stats_bytes // 8, dtype=torch.int64, device=self.device)
            self._tables = torch.zeros(lay.tables_bytes // 8, dtype=torch.float64, device=self.device)
            self._agents = torch.zeros(lay.agents_bytes // 4, dtype=torch.int32, device=self.device)
            self.obs = torch.empty((N, 2, self.obs_len), dtype=torch.float32, device=self.device)
            self.reward = torch.empty((N, 2), dtype=torch.float32, device=self.device)
            self.done = torch.empty((N,), dtype=torch.uint8, device=self.device)
            self.status = torch.empty((N,), dtype=torch.uint8, device=self.device)
            self.scores = torch.empty((N, 2), dtype=torch.int32, device=self.device)
            self._actions = torch.zeros((N, 2, _capi.MAX_ACTIONS, 2), dtype=torch.int8, device=self.device)
        ptrs = (C.c_void_p * _capi.BIND_COUNT)(self._records.data_ptr(), self._health.data_ptr(), self._stats.data_ptr(),
                                               self._tables.data_ptr(), self._agents.data_ptr())
        _capi.check(self._lib.evg_bind(self._h, ptrs, _capi.BIND_COUNT))
        self._host = {}
        self._rows = {}
        self._is_reset = False

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.evg_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(self._lib.evg_launch_count(self._h))

    def _to_int8_rows(self, actions, device):
        """Any numeric [N,2,7,2] array -> int8 rows on `device`: astype(int) truncation toward zero (server.py:232),
        then SATURATION into int8, so that ids beyond the int8 range stay out of range (no-op rows) instead of wrapping
        into valid commands.  The one conversion both step() and step_host() use."""
        torch = _torch()
        shape = (self.num_envs, 2, _capi.MAX_ACTIONS, 2)
        a = torch.as_tensor(actions)
        if tuple(a.shape) != shape:
            raise ValueError("actions must have shape %s, got %s" % (shape, tuple(a.shape)))
        a = a.to(device)
        if a.dtype == torch.int8:
            return a
        if a.is_floating_point():
            a = a.trunc()
        return a.clamp(-128, 127).to(torch.int8)

    def _as_actions(self, actions):
        torch = _torch()
        shape = (self.num_envs, 2, _capi.MAX_ACTIONS, 2)
        if isinstance(actions, torch.Tensor) and actions.dtype == torch.int8 and actions.device == self.device \
                and tuple(actions.shape) == shape and actions.is_contiguous():
            return actions
        self._actions.copy_(self._to_int8_rows(actions, self.device))
        return self._actions

    def _fmt(self, obs_format):
        try:
            return OBS_FORMATS[obs_format]
        except KeyError:
            raise ValueError("obs_format must be one of %s" % sorted(OBS_FORMATS))

    def obs_rows(self, obs_format):
        """The device tensor a non-float32 observation format is written into (allocated on first use):
        'i16' int16 [N,2,L] (same layout as `obs`), 'wire' uint8 [N, row_bytes] (evgsim.wire / include/evgsim.h)."""
        torch = _torch()
        fmt = self._fmt(obs_format)
        if fmt == _capi.OBS_F32:
            return self.obs
        if obs_format not in self._rows:
            if fmt == _capi.OBS_I16:
                self._rows[obs_format] = torch.empty((self.num_envs, 2, self.obs_len), dtype=torch.int16, device=self.device)
            else:
                rb = int(self._lib.evg_obs_row_bytes(self._h, fmt))
                self._rows[obs_format] = torch.empty((self.num_envs, rb), dtype=torch.uint8, device=self.device)
        return self._rows[obs_format]

    # ------------------------------------------------------------------ reference-shaped API
    def reset(self, mask=None, obs_format="f32"):
        """All matches (mask None) or the masked ones go back to the game_init state; returns obs (or, with another
        obs_format, obs_rows(obs_format)).  A masked reset starts the slot's next episode (new combat tape)."""
        torch = _torch()
        fmt = self._fmt(obs_format)
        mptr = None
        if mask is not None:
            if not self._is_reset:
                raise RuntimeError("the first reset() must cover all matches (mask=None)")
            mask = torch.as_tensor(mask).to(self.device).ne(0).to(torch.uint8).contiguous()
            if tuple(mask.shape) != (self.num_envs,):
                raise ValueError("mask must have shape (%d,)" % self.num_envs)
            mptr = C.c_void_p(mask.data_ptr())
        rows = self.obs_rows(obs_format)
        scratch = C.c_void_p(self.obs.data_ptr()) if fmt == _capi.OBS_I16 else None
        _capi.check(self._lib.evg_reset_fmt(self._h, fmt, mptr, C.c_void_p(rows.data_ptr()), scratch, self._stream()))
        self._is_reset = True
        return rows

    def step(self, actions, obs_format="f32"):
        """One game turn for every match. Returns (obs, reward, done, info) — tensors, overwritten in place.
        obs_format 'wire' / 'i16': the observations come as obs_rows(obs_format) instead (lossless, fewer bytes)."""
        if not self._is_reset:
            raise RuntimeError("call reset() before step()")
        a = self._as_actions(actions)
        fmt = self._fmt(obs_format)
        rows = self.obs_rows(obs_format)
        scratch = C.c_void_p(self.obs.data_ptr()) if fmt == _capi.OBS_I16 else None
        _capi.check(self._lib.evg_step_fmt(self._h, fmt, C.c_void_p(a.data_ptr()), C.c_void_p(rows.data_ptr()), scratch,
                                           C.c_void_p(self.reward.data_ptr()), C.c_void_p(self.done.data_ptr()),
                                           C.c_void_p(self.status.data_ptr()), C.c_void_p(self.scores.data_ptr()),
                                           self._stream()))
        return rows, self.reward, self.done, {"status": self.status, "scores": self.scores}

    def step_agents(self, agent0=_capi.AGENT_RANDOM, agent1=_capi.AGENT_RANDOM, actions=None, want_actions=False):
        """One turn with scripted opponents fused into the step kernel (evg_step_agents).

        agentN: _capi.AGENT_EXTERNAL (rows of that player are taken from `actions`), AGENT_RANDOM, AGENT_BASE_RUSH or
        AGENT_SWARM (agents/State_Machine/*.py on the device).
        With both players scripted and want_actions=False the turn is a single launch that reads no action
        buffer; want_actions=True also writes the generated rows into the returned info["actions"]."""
        if not self._is_reset:
            raise RuntimeError("call reset() before step()")
        ext = agent0 == _capi.AGENT_EXTERNAL or agent1 == _capi.AGENT_EXTERNAL
        aptr = None
        rows_t = self._actions  # the tensor the kernels read external rows from and write generated rows into
        if ext:
            rows_t = self._as_actions(actions)
            aptr = C.c_void_p(rows_t.data_ptr())
        elif (want_actions or self._lib.evg_step_kernel_kind(self._h) == 0
              or (self.num_nodes > 15 and _capi.AGENT_RANDOM in (int(agent0), int(agent1)))):
            # next to the warp-per-match kernel (small batches), and for the random agent on maps too large for its
            # register-only variant, the agents run as their own kernel and hand their rows over in the action buffer
            aptr = C.c_void_p(self._actions.data_ptr())
        _capi.check(self._lib.evg_step_agents(self._h, int(agent0), int(agent1), aptr, C.c_void_p(self.obs.data_ptr()),
                                              C.c_void_p(self.reward.data_ptr()), C.c_void_p(self.done.data_ptr()),
                                              C.c_void_p(self.status.data_ptr()), C.c_void_p(self.scores.data_ptr()),
                                              self._stream()))
        info = {"status": self.status, "scores": self.scores}
        if aptr is not None:
            info["actions"] = rows_t
        return self.obs, self.reward, self.done, info

    def rollout(self, turns, agent0=_capi.AGENT_RANDOM, agent1=_capi.AGENT_RANDOM, graph_turns=50):
        """`turns` self-play turns with both players scripted on the device, in ONE launch of evg_rollout.

        Small batches run the warp-per-match multi-turn kernel (a warp keeps its match for the whole rollout), larger ones
        the thread-per-match kernel, whose CTAs keep each batch of 128 matches in shared memory for all the turns: only the
        last turn pays for observations and the record write-back, none for a launch.  Results are those of calling
        step_agents(agent0, agent1) `turns` times: the tensors hold the last turn's outputs, episode statistics accumulate
        on the device.  (Only the random agent on maps of more than 15 nodes still runs turn by turn: agent kernel + step,
        captured into a CUDA graph of `graph_turns` turns; graph_turns=0 disables the graph.)"""
        if not self._is_reset:
            raise RuntimeError("call reset() before rollout()")
        torch = _torch()
        agent0, agent1 = int(agent0), int(agent1)
        if _capi.AGENT_EXTERNAL in (agent0, agent1):
            raise ValueError("rollout() needs both players scripted (AGENT_RANDOM / AGENT_BASE_RUSH / AGENT_SWARM)")
        left = int(turns)
        if not (self.num_nodes > 15 and _capi.AGENT_RANDOM in (agent0, agent1)):
            _capi.check(self._lib.evg_rollout(self._h, agent0, agent1, left, C.c_void_p(self._actions.data_ptr()),
                                              C.c_void_p(self.obs.data_ptr()), C.c_void_p(self.reward.data_ptr()),
                                              C.c_void_p(self.done.data_ptr()), C.c_void_p(self.status.data_ptr()),
                                              C.c_void_p(self.scores.data_ptr()), self._stream()))
            return self.obs, self.reward, self.done, {"status": self.status, "scores": self.scores}
        if graph_turns and left >= graph_turns:
            key = (agent0, agent1, int(graph_turns))
            graphs = self.__dict__.setdefault("_graphs", {})
            if key not in graphs:
                cur = torch.cuda.current_stream(self.device)
                side = torch.cuda.Stream(self.device)
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    self.step_agents(agent0, agent1)  # warm-up outside the capture (lazy module loading)
                    left -= 1
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=side):
                        for _ in range(graph_turns):
                            self.step_agents(agent0, agent1)
                cur.wait_stream(side)
                graphs[key] = g  # (capturing does not run the turns)
            g = graphs[key]
            while left >= graph_turns:
                g.replay()
                left -= graph_turns
        for _ in range(left):
            self.step_agents(agent0, agent1)
        return self.obs, self.reward, self.done, {"status": self.status, "scores": self.scores}

    # ------------------------------------------------------------------ host-buffer path (end-to-end)
    def host_buffers(self, obs_format="f32"):
        """Pinned host arrays for step_host: actions int8[N,2,7,2] in; obs (in `obs_format`), reward, done out.
        They are allocated by evgsim.hostmem (page-locked, on the NUMA node next to this GPU where the kernel allows)."""
        if obs_format not in self._host:
            torch = _torch()
            from . import hostmem
            fmt = self._fmt(obs_format)
            N = self.num_envs
            dev = self.device.index if self.device.index is not None else torch.cuda.current_device()
            if fmt == _capi.OBS_F32:
                obs = hostmem.pinned_empty((N, 2, self.obs_len), torch.float32, dev)
            elif fmt == _capi.OBS_I16:
                obs = hostmem.pinned_empty((N, 2, self.obs_len), torch.int16, dev)
            else:
                obs = hostmem.pinned_empty((N, int(self._lib.evg_obs_row_bytes(self._h, fmt))), torch.uint8, dev)
            first = next(iter(self._host.values()), None)
            self._host[obs_format] = {
                "actions": first["actions"] if first else hostmem.pinned_empty((N, 2, _capi.MAX_ACTIONS, 2), torch.int8, dev).zero_(),
                "obs": obs,
                "reward": first["reward"] if first else hostmem.pinned_empty((N, 2), torch.float32, dev),
                "done": first["done"] if first else hostmem.pinned_empty((N,), torch.uint8, dev),
            }
        return self._host[obs_format]

    def step_host(self, actions=None, sync=True, obs_format="f32"):
        """Same turn through HOST memory: H2D actions, step, D2H obs/reward/done (evg_step_host_fmt).

        `actions`: None (use host_buffers()['actions'] as filled by the caller) or an array copied into
        it.  obs_format: 'f32' (the reference's vector, 840 B per match on DemoMap), 'i16' (same layout, 420 B) or
        'wire' (one packed 128-byte row per match that also carries reward and done; evgsim.wire.expand rebuilds the
        float32 vector exactly).  Returns the pinned host tensors (valid after the stream is synchronised; sync=True
        does it); with 'wire' the reward and done tensors are views into the rows.
        """
        if not self._is_reset:
            raise RuntimeError("call reset() before step()")
        torch = _torch()
        fmt = self._fmt(obs_format)
        hb = self.host_buffers(obs_format)
        src = hb["actions"]
        if actions is not None:
            if isinstance(actions, torch.Tensor) and actions.dtype == torch.int8 and actions.device.type == "cpu" \
                    and actions.is_pinned() and actions.is_contiguous() and tuple(actions.shape) == tuple(src.shape):
                src = actions  # already page-locked: DMA straight from the caller's buffer
            else:
                src.copy_(self._to_int8_rows(actions, "cpu"))
        rows = self.obs_rows(obs_format)
        scratch = C.c_void_p(self.obs.data_ptr()) if fmt == _capi.OBS_I16 else None
        wire = fmt == _capi.OBS_WIRE  # the row carries the rewards and the done flag: no separate copies
        _capi.check(self._lib.evg_step_host_fmt(
            self._h, fmt, C.c_void_p(src.data_ptr()), C.c_void_p(hb["obs"].data_ptr()),
            None if wire else C.c_void_p(hb["reward"].data_ptr()), None if wire else C.c_void_p(hb["done"].data_ptr()),
            C.c_void_p(self._actions.data_ptr()), C.c_void_p(rows.data_ptr()), scratch,
            C.c_void_p(self.reward.data_ptr()), C.c_void_p(self.done.data_ptr()), self._stream()))
        if sync:
            torch.cuda.current_stream(self.device).synchronize()
        if wire:
            g = _capi.WIRE_NODE0 + 4 * self.num_nodes + 3 * 2 * _capi.NUM_GROUPS
            rew = hb["obs"][:, g:g + 8].view(torch.float32)  # views into the pinned rows: [N,2] float32, [N] uint8
            return hb["obs"], rew, hb["obs"][:, 2], {}
        return hb["obs"], hb["reward"], hb["done"], {}

    def h2d_bytes_per_step(self) -> int:
        return self.num_envs * int(self.layout.action_bytes)

    def d2h_bytes_per_step(self, obs_format="f32") -> int:
        fmt = self._fmt(obs_format)
        extra = 0 if fmt == _capi.OBS_WIRE else 2 * 4 + 1  # separate reward and done copies (a wire row has them inside)
        return self.num_envs * (int(self._lib.evg_obs_row_bytes(self._h, fmt)) + extra)

    # ------------------------------------------------------------------ scripted agents on the device
    def random_actions(self, player=-1, out=None):
        """random_actions agent (agents/State_Machine/random_actions.py:38-46) for `player` (-1 = both)."""
        out = self._actions if out is None else out
        _capi.check(self._lib.evg_agent_random(self._h, C.c_void_p(out.data_ptr()), int(player), self._stream()))
        return out

    def agent_actions(self, agent0, agent1, out=None):
        """Rows of the scripted agents (_capi.AGENT_RANDOM / AGENT_BASE_RUSH / AGENT_SWARM) for both players into an
        int8 [N,2,7,2] tensor; AGENT_EXTERNAL players' rows are left as they are."""
        out = self._actions if out is None else out
        _capi.check(self._lib.evg_agents(self._h, int(agent0), int(agent1), C.c_void_p(out.data_ptr()), self._stream()))
        return out

    # ------------------------------------------------------------------ policy-in-the-loop glue
    def decode_dqn(self, q, player=-1, out=None):
        """Q-values float32 [N,2,12*C] (player=-1) or [N,12*C] -> action rows, exactly like DQNAgent.filter_actions
        (agents/DQN/DQNAgent.py:161-197).  The policy forward itself is the caller's torch module on `self.obs`."""
        torch = _torch()
        out = self._actions if out is None else out
        q = q.to(self.device, torch.float32).contiguous()
        rows = self.num_envs * (2 if player < 0 else 1)
        if q.numel() % (rows * _capi.NUM_GROUPS):
            raise ValueError("q must hold 12*C values per (match, player)")
        cols = q.numel() // (rows * _capi.NUM_GROUPS)
        _capi.check(self._lib.evg_decode_dqn(self._h, C.c_void_p(q.data_ptr()), cols, int(player), C.c_void_p(out.data_ptr()),
                                             self._stream()))
        return out

    def decode_indices(self, idx, div=12, mod=11, player=-1, out=None):
        """Flat action indices int64 [N,2,7] (or [N,7]) -> rows (idx // div, idx % mod); defaults are PPOAgent.get_action's
        (agents/PPO/PPOAgent.py:122-127)."""
        torch = _torch()
        out = self._actions if out is None else out
        idx = idx.to(self.device, torch.int64).contiguous()
        assert idx.numel() == self.num_envs * (2 if player < 0 else 1) * _capi.MAX_ACTIONS
        _capi.check(self._lib.evg_decode_indices(self._h, C.c_void_p(idx.data_ptr()), int(div), int(mod), int(player),
                                                 C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def shape_reward(self, mode, out=None):
        """utils/reward_shaping.py on the device: mode = _capi.SHAPE_* ; returns float32 [N,2] from the last step's
        reward/done/obs tensors (turnNum = observed turn - 1)."""
        torch = _torch()
        if out is None:
            if getattr(self, "_shaped", None) is None:
                self._shaped = torch.empty((self.num_envs, 2), dtype=torch.float32, device=self.device)
            out = self._shaped
        _capi.check(self._lib.evg_shape_reward(self._h, int(mode), C.c_void_p(self.reward.data_ptr()), C.c_void_p(self.done.data_ptr()),
                                               C.c_void_p(self.obs.data_ptr()), C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def expand_wire(self, rows, index=None, player=-1, out=None, reward=None, done=None):
        """Wire rows uint8 [M, row_bytes] (obs_rows('wire') of some turn, or rows stored since) -> the float32
        observations on the device, bit for bit what the step writes in the f32 format (evg_wire_expand).  Output row i
        expands rows[index[i]] (index: int64 [K] on the device; None: row i), so a replay memory expands a sampled
        minibatch in one launch; an index outside [0, M) gives a row of zeros (reward 0, done 0).  player -1: float32
        [K, 2, L]; 0 or 1: [K, L].  reward (float32 [K, 2]) and done (uint8 [K]) are filled when given.  Returns `out`
        (allocated when None).  ValueError, before anything is launched, for a tensor of the wrong dtype, width, shape or
        device, or one that is not contiguous."""
        torch = _torch()
        rb = int(self._lib.evg_obs_row_bytes(self._h, _capi.OBS_WIRE))

        def need(name, t, dtype, shape):
            if not isinstance(t, torch.Tensor) or t.dtype != dtype or t.device != self.device or not t.is_contiguous() \
                    or (shape is not None and tuple(t.shape) != shape):
                raise ValueError("%s must be a contiguous %s tensor%s on %s, got %s" % (
                    name, dtype, "" if shape is None else " of shape %s" % (shape,), self.device,
                    "%s %s%s on %s" % (t.dtype, tuple(t.shape), "" if t.is_contiguous() else " (not contiguous)", t.device)
                    if isinstance(t, torch.Tensor) else type(t).__name__))

        need("rows", rows, torch.uint8, None)
        if rows.dim() != 2 or rows.shape[1] != rb:
            raise ValueError("rows must be [M, %d] wire rows of this map, got shape %s" % (rb, tuple(rows.shape)))
        if player not in (-1, 0, 1):
            raise ValueError("player must be -1, 0 or 1, got %r" % (player,))
        if index is not None:
            need("index", index, torch.int64, None)
            if index.dim() != 1:
                raise ValueError("index must be one-dimensional, got shape %s" % (tuple(index.shape),))
        k = rows.shape[0] if index is None else index.shape[0]
        shape = (k, 2, self.obs_len) if player < 0 else (k, self.obs_len)
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=self.device)
        need("out", out, torch.float32, shape)
        if reward is not None:
            need("reward", reward, torch.float32, (k, 2))
        if done is not None:
            need("done", done, torch.uint8, (k,))

        def ptr(t):
            return None if t is None else C.c_void_p(t.data_ptr())

        _capi.check(self._lib.evg_wire_expand(self._h, ptr(rows), rows.shape[0], ptr(index), k, int(player), ptr(out), ptr(reward),
                                              ptr(done), self._stream()))
        return out

    # ------------------------------------------------------------------ snapshots
    def get_state(self, first=0, count=None):
        """numpy structured array (dtype _capi.env_state_dtype()) of matches [first, first+count)."""
        torch = _torch()
        count = self.num_envs - first if count is None else count
        dt = _capi.env_state_dtype()
        buf = torch.empty(count * dt.itemsize, dtype=torch.uint8, device=self.device)
        _capi.check(self._lib.evg_export_state(self._h, first, count, C.c_void_p(buf.data_ptr()), self._stream()))
        return buf.cpu().numpy().view(dt).copy()

    def set_state(self, states, first=0):
        """Import EvgEnvState records (get_state's dtype) into matches [first, first+len).  Before the first reset() only
        an import that covers ALL matches is accepted (the others would be uninitialised memory); fields that the
        kernels use as indices are validated here and raise ValueError."""
        torch = _torch()
        dt = _capi.env_state_dtype()
        states = np.ascontiguousarray(states)
        assert states.dtype == dt
        if not self._is_reset and not (first == 0 and len(states) == self.num_envs):
            raise RuntimeError("set_state() before reset() must cover all %d matches" % self.num_envs)
        n = self.num_nodes
        g = states["groups"]
        cp = np.array(list(self.cfg.node_control_points)[:n + 1])
        if ((g["location"] < 1) | (g["location"] > n)).any() or (g["travel_destination"] > n).any() \
                or ((g["distance_remaining"] < 0) | (g["distance_remaining"] > 255)).any() \
                or (np.abs(states["control_state"][:, 1:n + 1].astype(np.int64)) > cp[1:]).any() \
                or ((states["controlled_by"][:, 1:n + 1] < -1) | (states["controlled_by"][:, 1:n + 1] > 1)).any():
            raise ValueError("set_state: location must be 1..%d, travel_destination <= %d, distance_remaining 0..255, "
                             "|control_state| <= ControlPoints and controlled_by -1..1" % (n, n))
        buf = torch.from_numpy(states.view(np.uint8).reshape(-1).copy()).to(self.device)
        _capi.check(self._lib.evg_import_state(self._h, first, len(states), C.c_void_p(buf.data_ptr()), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()
        self._is_reset = True

    def episode_stats(self) -> dict:
        st = _capi.EvgEpisodeStats()
        _capi.check(self._lib.evg_episode_stats(self._h, C.byref(st), self._stream()))
        return {"episodes": st.episodes, "wins": [st.wins[0], st.wins[1]], "ties": st.ties,
                "total_turns": st.total_turns, "total_score": [st.total_score[0], st.total_score[1]],
                "status_count": [st.status_count[i] for i in range(4)], "env_turns": st.env_turns,
                "fought_unit_slots": st.fought_unit_slots}


class EvergladesEnv:
    """Drop-in for ``gym_everglades.envs.EvergladesEnv`` (env.py:13-116), one match on the GPU.

    Same attributes (env.py:17-28, with ``observation_space`` a Box[105] and ``action_space`` a Tuple of
    (Discrete 12, Discrete 12) x 7 — gym's classes when gym/gymnasium is installed, stand-ins with the same attributes
    otherwise), ``reset(**kwargs) -> {pid: float64[105]}`` and ``step({pid: array[k,2]}) -> (obs, reward, done, {})``
    with the reference's types and error behaviour: AssertionError for != 2 players (env.py:87) or != 2 action columns
    (server.py:226), IndexError for group ids outside [-12, 11] and player-1 node ids outside [-12, 11]
    (server.py:92,235; negative ids wrap like Python lists).  ``render``/``close`` are no-ops (the pyglet viewer is out
    of scope).  Combat randomness comes from the Philox tape keyed on (`seed`, match id, EPISODE, ...): the simulator is
    kept across ``reset()`` calls and every reset starts the next episode of the slot, so successive episodes draw
    different combat targets, like the reference's global numpy stream that carries on across resets.
    """

    metadata = {"render.modes": ["human"]}

    def __init__(self, device=0, seed=0):
        self.num_turns = 150
        self.num_units = 100
        self.num_groups = 12
        self.num_nodes = 11
        self.num_actions_per_turn = 7
        self.unit_classes = list(UNIT_CLASSES)
        from .spaces import space_classes
        Box, Discrete, Tuple = space_classes()
        self.action_space = Tuple((Discrete(self.num_groups), Discrete(self.num_nodes + 1)) * self.num_actions_per_turn)  # env.py:25
        self.observation_space = self._build_observation_space(Box)
        self.viewer = None
        self._device, self._seed = device, seed
        self._env = None
        self._env_key = None

    def _build_observation_space(self, Box):
        """Box bounds as env.py:124-143 declares them (controlState of bases exceeds them: SURVEY A.5)."""
        group_low = np.array([1, 0, 0, 0, 0])
        group_high = np.array([self.num_nodes, len(self.unit_classes), 100, 1, self.num_units])
        cp_low = np.array([0, 0, -100, -1])
        cp_high = np.array([1, 1, 100, self.num_units])
        low = np.concatenate([[1], np.tile(cp_low, self.num_nodes), np.tile(group_low, self.num_groups)])
        high = np.concatenate([[self.num_turns + 1], np.tile(cp_high, self.num_nodes), np.tile(group_high, self.num_groups)])
        return Box(low=low.astype(np.float32), high=high.astype(np.float32))

    def reset(self, **kwargs):
        self.players = kwargs.get("players")
        config_dir = kwargs.get("config_dir")
        map_file = kwargs.get("map_file") or "DemoMap.json"
        unit_file = kwargs.get("unit_file") or "UnitDefinitions.json"
        self.debug = kwargs.get("debug", False)  # accepted and, as in the reference, without effect on obs
        assert len(self.players) == 2, "Must have exactly two players"  # env.py:87
        self.pks = self.players.keys()
        self.sorted_pks = sorted(self.pks)
        for p in self.pks:
            assert p in (0, 1), "Given player number not included in map configuration file starting locations"
        cfg = load_config(config_dir, map_file, unit_file, kwargs.get("setup_file", "GameSetup.json"))
        key = (bytes(cfg), int(kwargs.get("env_id", 0)))
        if self._env is None or key != self._env_key:
            # first game, or other config files than last time: a new simulator (episode counter back to 0)
            if self._env is not None:
                self._env.close()
            self._env = BatchedEvergladesEnv(1, device=self._device, seed=self._seed, config=cfg,
                                             auto_reset=_capi.AUTORESET_OFF, env_id_offset=key[1])
            self._env_key = key
            obs = self._env.reset()
        else:
            obs = self._env.reset(mask=[1])  # same game files: next episode of the same slot, nothing reallocated
        self.num_nodes = self._env.num_nodes
        self.num_turns = self._env.num_turns
        self.num_units = self._env.num_units
        return self._obs_dict(obs)
    def _obs_dict(self, obs):
        o = obs[0].to("cpu").numpy().astype(np.float64)
        return {p: o[p].copy() for p in self.players}

    def step(self, actions):
        rows = np.zeros((1, 2, _capi.MAX_ACTIONS, 2), dtype=np.int8)
        for player in (0, 1):  # server.py:218-221
            if player not in actions:
                print("Player {} not found in input action dictionary".format(player))
                continue
            action = np.asarray(actions[player])
            r, c = action.shape[:2]
            assert c == 2, "Did not receive 2 columns for player {}s action".format(player)  # server.py:226
            action = action[:7, :].astype(int)  # server.py:227,232
            for i, (gid, nid) in enumerate(action):
                if not -self.num_groups <= gid < self.num_groups:
                    raise IndexError("list index out of range")  # players[player].groups[gid], server.py:235
                gid = gid % self.num_groups
                if player == 1:
                    if not -(self.num_nodes + 1) <= nid <= self.num_nodes:
                        raise IndexError("list index out of range")  # p1_node_map[int(nid)], server.py:92
                    nid = nid % (self.num_nodes + 1)
                rows[0, player, i] = (gid, nid if 0 <= nid <= 127 else 0)
        obs, _, done, info = self._env.step(rows)
        scores = info["scores"][0].to("cpu").numpy()
        status = int(info["status"][0])
        reward = {i: 0 for i in self.players}
        done = 0
        if status != 0:  # env.py:39-46
            done = 1
            if scores[0] != scores[1]:
                reward[0] = 1 if scores[0] > scores[1] else 0
                reward[1] = 1 if scores[1] > scores[0] else -1
        else:  # env.py:58-60
            reward[0] = int(scores[0]) / MAX_SCORE
            reward[1] = int(scores[1]) / MAX_SCORE
        return self._obs_dict(obs), reward, done, {}

    def render(self, mode="human"):
        return None

    def close(self):
        if self._env is not None:
            self._env.close()
            self._env = None
            self._env_key = None
