"""The fused PPO actors' log-probabilities (FusedPPO / FusedRPPO want_logp, evg_policy_*_logp d_logp) and the recurrent
actor's starting state (want_hidden_in, d_hidden_in): against the statement of tests/ppo_logp.py on the kernel's own
probabilities and draws, at every tiling edge, on f32 and wire input; every other output unchanged by asking for them;
and a stored rollout (wire rows, draws, logp, starting state) re-evaluated by the numpy reference.

Tolerances.  The kernel computes logf(p_j / T_k) in fp32 (one correctly rounded quotient, accurate logf); the statement
computes log(p_j / T_k) in float64 on the same fp32 operands: 2e-6 absolute (about 4 ulp of a value of magnitude <= 7).
Re-evaluation from the stored rollout uses the probability tolerance of tests/test_gpu_policy_rppo.py, P_REL = 5e-3 of
each probability (so of p_j / T_k twice that, T_k being a sum of such probabilities)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LOGP_ABS, P_REL = 2e-6, 5e-3


@pytest.fixture(scope="module")
def evg():
    import __graft_entry__ as g
    g.build()
    import evgsim
    return evgsim


@pytest.fixture(scope="module")
def sms(evg):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def ppo_net(torch, latent, seed):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                               torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))


def rppo_actor(torch, latent, seed):
    torch.manual_seed(seed)
    actor = torch.nn.Module()
    actor.action_head = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
    actor.action_gru = torch.nn.GRU(latent, latent)
    actor.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
    return actor


def wire_env(evg, cfg, n, seed=17, turns=30, **kw):
    """n matches played for `turns` turns in the wire format; env.obs holds the expansion of the last rows, so the f32
    and the wire call read the same observations."""
    env = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg, **kw)
    env.reset(obs_format="wire")
    for _ in range(turns):
        env.step(env.random_actions(), obs_format="wire")
    env.expand_wire(env.obs_rows("wire"), out=env.obs)
    return env


def bits(t):
    a = np.ascontiguousarray(t.detach().cpu().numpy())
    return a.view(np.uint8)


def call(fused, h0=None, **kw):
    """One call from state h0 (FusedRPPO): every output as numpy, the outputs not asked for as None."""
    import torch
    if h0 is not None:
        fused.hidden.copy_(h0)
    fused.env._actions.fill_(-7)
    for t in [fused.logp, fused.probs] + ([fused.hidden_in] if h0 is not None else []):
        t.fill_(float("nan"))
    acts = fused(**kw).clone()
    torch.cuda.synchronize()
    out = {"actions": acts, "idx": fused.idx.clone(), "logp": fused.logp.clone() if kw.get("want_logp") else None,
           "probs": fused.probs.clone() if kw.get("want_probs") else None}
    if h0 is not None:
        out["hidden"] = fused.hidden.clone()
        out["hidden_in"] = fused.hidden_in.clone() if kw.get("want_hidden_in") else None
    return out


def statement(kind, probs, idx):
    import ppo_logp as pl
    p = probs.cpu().numpy()
    i = idx.cpu().numpy().reshape(-1, 7)
    if kind == "ppo":
        return pl.ppo_logp_rows(p.reshape(-1, 132), i)
    return pl.rppo_logp_rows(p.reshape(-1, 7, 132), i)


def check_values(kind, res):
    logp = res["logp"].cpu().numpy().reshape(-1, 7).astype(np.float64)
    want = statement(kind, res["probs"], res["idx"])
    assert np.isfinite(logp).all()
    assert np.abs(logp - want).max() <= LOGP_ABS, np.abs(logp - want).max()
    assert (logp <= 0).all() and (logp >= -7).all(), (logp.min(), logp.max())


def check_unchanged(kind, fused, fmt, h0, full):
    """actions, idx, probs and hidden bit for bit with and without the new outputs; logp with and without probs."""
    bare = call(fused, h0, obs_format=fmt)
    for k in ("actions", "idx") + (("hidden",) if kind == "rppo" else ()):
        assert np.array_equal(bits(bare[k]), bits(full[k])), k
    extra = {"want_hidden_in": True} if kind == "rppo" else {}
    probs_only = call(fused, h0, obs_format=fmt, want_probs=True)
    assert np.array_equal(bits(probs_only["probs"]), bits(full["probs"]))
    logp_only = call(fused, h0, obs_format=fmt, want_logp=True, **extra)
    assert np.array_equal(bits(logp_only["logp"]), bits(full["logp"]))
    for k in ("actions", "idx") + (("hidden", "hidden_in") if kind == "rppo" else ()):
        assert np.array_equal(bits(logp_only[k]), bits(full[k])), k


@pytest.mark.parametrize("fmt", ["f32", "wire"])
@pytest.mark.parametrize("latent", [1, 128, 248, 256])
@pytest.mark.parametrize("kind", ["ppo", "rppo"])
def test_logp_is_the_statement_of_the_kernels_own_draws(evg, cfg, kind, latent, fmt):
    """Every logp within 2e-6 of log(p_j / T_k) on the kernel's probs and idx, in [-7, 0]; nothing else changes."""
    import torch
    from evgsim import policy
    n = 1037
    env = wire_env(evg, cfg, n, seed=latent)
    if kind == "ppo":
        fused, h0, extra = policy.FusedPPO(env, ppo_net(torch, latent, latent)), None, {}
    else:
        fused = policy.FusedRPPO(env, rppo_actor(torch, latent, latent))
        h0 = torch.from_numpy(np.random.default_rng(latent).uniform(-1, 1, (n, 2, latent)).astype(np.float32)).to(env.device)
        extra = {"want_hidden_in": True}
    full = call(fused, h0, obs_format=fmt, want_probs=True, want_logp=True, **extra)
    check_values(kind, full)
    if kind == "rppo":
        assert np.array_equal(bits(full["hidden_in"]), bits(expect_hidden_in(env, h0)))
    check_unchanged(kind, fused, fmt, h0, full)
    other = call(fused, h0, obs_format="wire" if fmt == "f32" else "f32", want_logp=True, **extra)
    assert np.array_equal(bits(other["logp"]), bits(full["logp"]))  # wire rows stage the same bf16 tile


@pytest.mark.parametrize("player", [-1, 0, 1])
@pytest.mark.parametrize("kind", ["ppo", "rppo"])
def test_tiling_edges_and_single_players(evg, cfg, sms, kind, player):
    """Batches at and around the 128-row tile and past several tiles per CTA (test_multi_tile_batches' size); a one-player
    call writes [N, 7] that equals its column of the two-player call, and leaves the other player's action rows alone."""
    import torch
    from evgsim import policy
    tiles = (5 * sms + 1) // 2
    latent = 248 if kind == "rppo" else 128
    make = (lambda env, p: policy.FusedRPPO(env, rppo_actor(torch, latent, 3), player=p)) if kind == "rppo" else \
        (lambda env, p: policy.FusedPPO(env, ppo_net(torch, latent, 3), player=p))
    for n in (1, 63, 64, 65, 127, 128, 129, (tiles - 1) * 128 + 54):
        env = wire_env(evg, cfg, n, seed=n, turns=12)
        h0 = None
        if kind == "rppo":
            h_both = torch.from_numpy(np.random.default_rng(n).uniform(-1, 1, (n, 2, latent)).astype(np.float32)).to(env.device)
            h0 = h_both if player < 0 else h_both[:, player].contiguous()
        extra = {"want_hidden_in": True} if kind == "rppo" else {}
        fused = make(env, player)
        res = call(fused, h0, want_probs=True, want_logp=True, **extra)
        assert tuple(res["logp"].shape) == ((n, 2, 7) if player < 0 else (n, 7))
        check_values(kind, res)
        if player >= 0:
            assert (res["actions"][:, 1 - player] == -7).all()
            both = call(make(env, -1), h_both if kind == "rppo" else None, want_logp=True, **extra)
            assert np.array_equal(bits(res["logp"]), bits(both["logp"][:, player])), n
            assert np.array_equal(bits(res["idx"]), bits(both["idx"][:, player])), n
            if kind == "rppo":
                assert np.array_equal(bits(res["hidden_in"]), bits(both["hidden_in"][:, player])), n


def expect_hidden_in(env, h0):
    turn = torch_turn(env, h0.device)
    shape = (-1,) + (1,) * (h0.dim() - 1)
    return torch_where(turn.view(shape) == 0, h0)


def torch_turn(env, device):
    import torch
    return torch.as_tensor(env.get_state()["turn"].astype(np.int64), device=device)


def torch_where(fresh, h0):
    import torch
    return torch.where(fresh, torch.zeros_like(h0), h0)


@pytest.mark.parametrize("latent", [128, 248])
def test_hidden_in_is_the_state_each_row_started_from(evg, cfg, latent):
    """hidden_in = where(turn == 0, +0.0, hidden before the call), bit for bit: fresh matches with NaN and garbage in
    .hidden, automatic resets in the middle of a batch, a masked reset under AUTORESET_OFF (where a finished match keeps
    its state); at L = 248 units 128.. live in d_hidden itself."""
    import torch
    from evgsim import policy
    n = 1500
    actor = rppo_actor(torch, latent, 5)
    env = evg.BatchedEvergladesEnv(n, seed=9, config=cfg)
    env.reset()
    fused = policy.FusedRPPO(env, actor)
    garbage = np.random.default_rng(2).uniform(-50, 50, (n, 2, latent)).astype(np.float32)
    garbage[::7] = np.nan
    res = call(fused, torch.from_numpy(garbage).to(env.device), want_hidden_in=True)
    assert (bits(res["hidden_in"]) == 0).all()  # +0.0 everywhere
    for auto in (1, 0):
        cfg.turn_limit = 20
        try:
            env = evg.BatchedEvergladesEnv(n, seed=9, config=cfg, auto_reset=auto)
            env.reset()
            # every third match starts over at turn 10, the others reach the limit at turn 20: under AUTORESET_TERMINAL
            # they restart with the last step; under AUTORESET_OFF they stay finished for 5 more steps, then every fifth
            # match is reset by hand
            for t in range(20 if auto else 25):
                if t == 10:
                    env.reset(mask=(np.arange(n) % 3 == 0).astype(np.uint8))
                env.step(env.random_actions())
            if auto == 0:
                env.reset(mask=(np.arange(n) % 5 == 0).astype(np.uint8))
        finally:
            cfg.turn_limit = 150
        turn = env.get_state()["turn"]
        assert 0 < (turn == 0).sum() < n, auto
        fused = policy.FusedRPPO(env, actor)
        h0 = torch.from_numpy(np.random.default_rng(3).uniform(-1, 1, (n, 2, latent)).astype(np.float32)).to(env.device)
        res = call(fused, h0, want_hidden_in=True, want_logp=True)
        assert np.array_equal(bits(res["hidden_in"]), bits(expect_hidden_in(env, h0))), auto
        bare = call(fused, h0)
        assert np.array_equal(bits(bare["hidden"]), bits(res["hidden"])) and np.array_equal(bits(bare["idx"]), bits(res["idx"]))


def near_limit_env(evg, cfg, n, seed):
    """n matches under AUTORESET_TERMINAL whose every fifth match is 2..9 turns from the limit: a 24-turn rollout
    crosses automatic resets in the middle of the batch."""
    env = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg, auto_reset=1)
    env.reset(obs_format="wire")
    st = env.get_state()
    st["turn"][::5] = cfg.turn_limit - 2 - np.arange(len(st["turn"][::5])) % 8
    env.set_state(st)
    env.step(env.random_actions(), obs_format="wire")  # rows of the imported state
    return env


@pytest.mark.parametrize("kind", ["ppo", "rppo"])
def test_a_stored_rollout_is_enough_to_re_evaluate_it(evg, cfg, kind):
    """Player 0 against the SwarmAgent on wire rows for 24 turns across automatic resets; per turn the pre-turn rows,
    idx, logp (and hidden_in) are stored.  The numpy reference on expand_wire(rows) (and hidden_in) gives back every
    stored logp; hidden_in of turn t + 1 is .hidden after turn t, or zero where the match restarted."""
    import torch
    import ppo_logp as pl
    from evgsim import _capi, policy
    n, latent = 600, 128
    env = near_limit_env(evg, cfg, n, seed=31)
    if kind == "ppo":
        net = ppo_net(torch, latent, 8)
        fused = policy.FusedPPO(env, net, player=0)
        weights = [t.detach().numpy() for m in net if isinstance(m, torch.nn.Linear) for t in (m.weight, m.bias)]
        extra = {}
    else:
        actor = rppo_actor(torch, latent, 8)
        fused = policy.FusedRPPO(env, actor, player=0)
        weights = policy.rppo_weights(actor)
        extra = {"want_hidden_in": True}
    store = []
    restarted = 0
    for t in range(24):
        rows = env.obs_rows("wire").clone()
        turn = env.get_state()["turn"]
        restarted += int(((turn == 0) & (t > 0)).sum())
        fused(obs_format="wire", want_logp=True, **extra)
        rec = {"rows": rows, "turn": turn, "idx": fused.idx.cpu().numpy(), "logp": fused.logp.cpu().numpy()}
        if kind == "rppo":
            rec["hidden_in"], rec["hidden"] = fused.hidden_in.cpu().numpy(), fused.hidden.cpu().numpy()
        store.append(rec)
        env.agent_actions(_capi.AGENT_EXTERNAL, _capi.AGENT_SWARM)
        env.step(env._actions, obs_format="wire")
    assert restarted > 0
    for t, rec in enumerate(store):
        obs = env.expand_wire(rec["rows"], player=0).cpu().numpy()
        if kind == "ppo":
            p = policy.reference_forward_ppo(obs, *weights)
            want = pl.ppo_logp_rows(p, rec["idx"])
            assert np.abs(rec["logp"] - want).max() <= 2 * P_REL, (t, np.abs(rec["logp"] - want).max())
        else:
            p, _ = policy.reference_forward_rppo(obs, rec["hidden_in"], weights)
            pj = np.take_along_axis(p, rec["idx"][:, :, None], axis=2)[:, :, 0]
            assert (np.abs(np.exp(rec["logp"].astype(np.float64)) - pj) <= P_REL * pj).all(), t
            if t + 1 < len(store):
                nxt = store[t + 1]
                fresh = nxt["turn"] == 0
                assert np.array_equal(nxt["hidden_in"][~fresh], rec["hidden"][~fresh]), t
                assert (nxt["hidden_in"][fresh].view(np.uint32) == 0).all(), t


@pytest.mark.parametrize("kind", ["ppo", "rppo"])
def test_cuda_graph_of_refresh_actor_step(evg, cfg, kind):
    """refresh -> actor(want_logp, want_hidden_in) -> step captured once; the replays give the eager turns' logp and
    hidden_in bit for bit, across automatic resets."""
    import torch
    from evgsim import policy
    n = 1000
    cfg.turn_limit = 30
    try:
        envs = [evg.BatchedEvergladesEnv(n, seed=14, config=cfg, auto_reset=1) for _ in range(2)]
    finally:
        cfg.turn_limit = 150
    if kind == "ppo":
        net = ppo_net(torch, 128, 21).to(envs[0].device)
        fused = [policy.FusedPPO(e, net) for e in envs]
        extra = {}
    else:
        net = rppo_actor(torch, 248, 21).to(envs[0].device)
        fused = [policy.FusedRPPO(e, net) for e in envs]
        extra = {"want_hidden_in": True}
    for e in envs:
        e.reset()

    def turn(k):
        fused[k].refresh()
        fused[k](want_logp=True, **extra)
        envs[k].step(envs[k]._actions)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            turn(1)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            turn(1)
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(3):
        turn(0)
    for t in range(45):
        turn(0)
        g.replay()
        assert torch.equal(fused[0].idx, fused[1].idx), t
        assert np.array_equal(bits(fused[0].logp), bits(fused[1].logp)), t
        if kind == "rppo":
            assert np.array_equal(bits(fused[0].hidden_in), bits(fused[1].hidden_in)), t
            assert torch.equal(fused[0].hidden, fused[1].hidden), t
    torch.cuda.synchronize()
    assert (envs[0].get_state()["episode"] > 0).any()


def test_argument_errors(evg, cfg):
    """An overlap of d_hidden_in and d_hidden (whole or partial), EVG_OBS_I16 and a null handle are refused with EVG_E_ARG
    before anything is launched; adjacent buffers are fine."""
    import torch
    from evgsim import _capi, policy
    n, latent = 64, 128
    env = evg.BatchedEvergladesEnv(n, seed=1, config=cfg)
    env.reset()
    fused = policy.FusedRPPO(env, rppo_actor(torch, latent, 1))
    ppo = policy.FusedPPO(env, ppo_net(torch, latent, 1))
    ptr = lambda t: C.c_void_p(t.data_ptr())
    w1, w2, wi, wh, w3, bias = (ptr(t) for t in fused._w)
    buf = torch.zeros((3 * n * 2 * latent,), dtype=torch.float32, device=env.device)
    size = n * 2 * latent

    def rcall(hidden, hidden_in, fmt=_capi.OBS_F32, h=env._h):
        return env._lib.evg_policy_rppo_logp(h, fmt, ptr(env.obs), -1, w1, w2, wi, wh, w3, bias, latent, 132, 12, 11, hidden, hidden_in,
                                             ptr(env._actions), ptr(fused.idx), None, ptr(fused.logp), env._stream())

    h = ptr(buf[size:])
    for off in (0, 1, size - 1, -size + 1):
        assert rcall(h, ptr(buf[size + off:])) == -1, off
        assert b"overlaps" in env._lib.evg_last_error()
    assert rcall(h, ptr(buf[2 * size:])) == 0 and rcall(h, ptr(buf)) == 0
    assert rcall(h, None) == 0
    assert rcall(h, ptr(buf[2 * size:]), fmt=_capi.OBS_I16) == -1
    assert rcall(h, ptr(buf[2 * size:]), h=None) == -1
    p1, p2, p3, pb = (ptr(t) for t in ppo._w)

    def pcall(fmt=_capi.OBS_F32, h=env._h):
        return env._lib.evg_policy_ppo_logp(h, fmt, ptr(env.obs), -1, p1, p2, p3, pb, latent, 132, 12, 11, ptr(env._actions),
                                            ptr(ppo.idx), None, ptr(ppo.logp), env._stream())

    assert pcall() == 0
    assert pcall(fmt=_capi.OBS_I16) == -1
    assert pcall(h=None) == -1
    torch.cuda.synchronize()
