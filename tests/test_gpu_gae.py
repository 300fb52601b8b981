"""evg_gae (BatchedEvergladesEnv.gae) on the GPU: PPO's advantages and returns of a stored rollout.

1. Random float inputs: bit for bit tests/ppo_gae.py's reference_gae (compared as uint32 patterns, so -0.0 shows) at
   every edge of the kernel's batching (T = 1, 2, K-1, K, K+1, 2K+1, 300 with K = 16 turns a batch) and of its one-warp
   CTAs (M = 1, 31, 32, 33, and an odd 40,001), for players -1, 0 and 1, gamma and lam in {0, 1, 0.99 / 0.95}, columns
   never done, always done, done only at t = 0 or only at t = T-1, values from 1e-40 (subnormal) to 1e30.
2. Wire rows of real rollouts under AUTORESET_TERMINAL and _NEXT, the matches staggered by masked resets so that dones
   fall on every turn of the window: rows alone, the float tensors that expand_wire gives for rows[1:], and the two mixed
   (the caller's rewards with the rows' done flags, and the reverse) all equal reference_gae.  Under AUTORESET_OFF the
   rows' done flags are taken as written: from the turn limit on every turn is its own episode, A_t = r_t - V_t.
3. The pipeline: FusedValue over the (T+1) * M stored rows, then gae, equals reference_gae on those values and lies
   within the derived bound (gae_bound) of the float64 textbook form.
4. A CUDA graph of critic -> gae replays the eager result; with outputs given gae allocates nothing.
5. Every ValueError of the wrapper is raised before a launch; every EVG_E_ARG case of the C ABI is refused."""
import ctypes as C

import numpy as np
import pytest

from ppo_gae import gae_bound, gae_float64, reference_gae
from test_gpu_policy_tiling import evg  # noqa: F401

pytestmark = pytest.mark.gpu

K = 16  # kGaeBatch of csrc/evg_gae.cu: turns whose loads one batch issues
BLOCK = 32  # kGaeThreads: matches per CTA
GAMMAS = [(0.0, 0.0), (1.0, 1.0), (0.99, 0.95), (0.0, 1.0), (1.0, 0.0)]


def bits(a):
    a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
    return np.ascontiguousarray(a).view(np.uint32)


def col(a, player):
    return a if player < 0 else np.ascontiguousarray(a[..., player])


@pytest.fixture(scope="module")
def env(evg):  # noqa: F811
    e = evg.BatchedEvergladesEnv(8, seed=1)
    e.reset()
    return e


def float_rollout(rng, T, M):
    """values [T+1, M, 2], reward [T, M, 2], done [T, M]: column m never done (m % 5 == 0), always done (1), done only at
    t = 0 (2), only at t = T-1 (3), or at random (4); magnitudes per column from 1e-40 to 1e30."""
    scale = np.array([1.0, 1e3, 1e30, 1e-40, 0.5], dtype=np.float64)[rng.integers(0, 5, M)]
    values = (rng.standard_normal((T + 1, M, 2)) * scale[None, :, None]).astype(np.float32)
    reward = (rng.standard_normal((T, M, 2)) * scale[None, :, None]).astype(np.float32)
    kind = np.arange(M) % 5
    done = np.zeros((T, M), dtype=np.uint8)
    done[:, kind == 1] = 1
    done[0, kind == 2] = 1
    done[T - 1, kind == 3] = 1
    done[:, kind == 4] = rng.random((T, int((kind == 4).sum()))) < 0.1
    return values, reward, done


def test_random_inputs_bit_for_bit(env):
    import torch
    rng = np.random.default_rng(0)
    dev = env.device
    n = 0
    for T in (1, 2, K - 1, K, K + 1, 2 * K + 1, 300):
        for M in (1, BLOCK - 1, BLOCK, BLOCK + 1, 40001):
            values, reward, done = float_rollout(rng, T, M)
            tv, tr, td = (torch.from_numpy(x).to(dev) for x in (values, reward, done))
            for player in (-1, 0, 1):
                v = tv if player < 0 else tv[..., player].contiguous()
                for gamma, lam in GAMMAS:
                    adv, ret = env.gae(v, reward=tr, done=td, gamma=gamma, lam=lam, player=player)
                    want_a, want_r = reference_gae(col(values, player), col(reward, player), done, gamma, lam)
                    assert adv.shape == want_a.shape and ret.shape == want_r.shape
                    assert np.array_equal(bits(adv), bits(want_a)), (T, M, player, gamma, lam)
                    assert np.array_equal(bits(ret), bits(want_r)), (T, M, player, gamma, lam)
                    n += 1
    assert n == 7 * 5 * 3 * len(GAMMAS)


def staggered_rollout(evg, mode, n=1000, T=40, seed=3, turn_limit=25):  # noqa: F811
    """n matches under auto-reset `mode`, each slot at its own phase (masked resets at random turns before the window),
    then T turns of scripted play stored as T+1 wire rows.  Returns env, rows [T+1, n, row_bytes] and what the step
    wrote as reward [T, n, 2] / done [T, n]."""
    import torch
    cfg = evg.load_config()
    cfg.turn_limit = turn_limit
    env = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg, auto_reset=mode)
    env.reset(obs_format="wire")
    g = torch.Generator(device=env.device).manual_seed(seed)
    for _ in range(turn_limit):
        env.step(env.agent_actions(evg._capi.AGENT_SWARM, evg._capi.AGENT_RANDOM), obs_format="wire")
        env.reset(mask=torch.rand(n, device=env.device, generator=g) < 0.08, obs_format="wire")
    rb = int(env._lib.evg_obs_row_bytes(env._h, evg._capi.OBS_WIRE))
    rows = torch.empty((T + 1, n, rb), dtype=torch.uint8, device=env.device)
    reward = torch.empty((T, n, 2), dtype=torch.float32, device=env.device)
    done = torch.empty((T, n), dtype=torch.uint8, device=env.device)
    rows[0].copy_(env.obs_rows("wire"))
    for t in range(T):
        _, r, d, _ = env.step(env.agent_actions(evg._capi.AGENT_SWARM, evg._capi.AGENT_BASE_RUSH), obs_format="wire")
        rows[t + 1].copy_(env.obs_rows("wire"))
        reward[t].copy_(r)
        done[t].copy_(d)
    return env, rows, reward, done


@pytest.mark.parametrize("mode", ["terminal", "next"])
def test_wire_rows_of_a_real_rollout(evg, mode):  # noqa: F811
    import torch
    env, rows, reward, done = staggered_rollout(evg, {"terminal": evg._capi.AUTORESET_TERMINAL, "next": evg._capi.AUTORESET_NEXT}[mode])
    T, n = done.shape
    per_t = done.sum(1).cpu().numpy()
    assert per_t[0] > 0 and per_t[-1] > 0 and (per_t > 0).all(), per_t  # dones on every turn of the window
    # the float tensors of the same turns, from the stored rows on the device
    rb = rows.shape[2]
    r = torch.empty((T * n, 2), dtype=torch.float32, device=env.device)
    d = torch.empty((T * n,), dtype=torch.uint8, device=env.device)
    env.expand_wire(rows[1:].reshape(T * n, rb), reward=r, done=d)
    r, d = r.view(T, n, 2), d.view(T, n)
    assert torch.equal(d, done) and np.array_equal(bits(r), bits(reward))
    rng = np.random.default_rng(7)
    values = torch.from_numpy(rng.standard_normal((T + 1, n, 2)).astype(np.float32)).to(env.device)
    shaped = torch.from_numpy(rng.standard_normal((T, n, 2)).astype(np.float32)).to(env.device)
    other = torch.from_numpy((rng.random((T, n)) < 0.3).astype(np.uint8)).to(env.device)
    rn, dn, sn, on = (x.cpu().numpy() for x in (r, d, shaped, other))
    for player in (-1, 0, 1):
        v = values if player < 0 else values[..., player].contiguous()
        vn = v.cpu().numpy()
        want = reference_gae(vn, col(rn, player), dn, 0.99, 0.95)
        for got in (env.gae(v, rows=rows, player=player), env.gae(v, reward=r, done=d, player=player),
                    env.gae(v, rows=rows, reward=r, done=d, player=player)):
            assert np.array_equal(bits(got[0]), bits(want[0])) and np.array_equal(bits(got[1]), bits(want[1])), (mode, player)
        # the caller's rewards with the rows' done flags, and the rows' rewards with the caller's done flags
        got = env.gae(v, rows=rows, reward=shaped, player=player)
        want = reference_gae(vn, col(sn, player), dn, 0.99, 0.95)
        assert np.array_equal(bits(got[0]), bits(want[0])) and np.array_equal(bits(got[1]), bits(want[1])), (mode, player)
        got = env.gae(v, rows=rows, done=other, player=player)
        want = reference_gae(vn, col(rn, player), on, 0.99, 0.95)
        assert np.array_equal(bits(got[0]), bits(want[0])) and np.array_equal(bits(got[1]), bits(want[1])), (mode, player)


def test_autoreset_off_keeps_the_done_flag(evg):  # noqa: F811
    """From a common reset, 25-turn matches under AUTORESET_OFF over a 40-turn window: the pass takes the rows' done flags
    as written, done is 1 on every turn from the turn limit on (t >= 24: row t+1 is turn t+1), and on every done turn
    A_t = fl(r_t - V_t) and R_t = fl(A_t + V_t)."""
    import torch
    cfg = evg.load_config()
    cfg.turn_limit = 25
    n, T = 512, 40
    env = evg.BatchedEvergladesEnv(n, seed=5, config=cfg, auto_reset=evg._capi.AUTORESET_OFF)
    rb = int(env._lib.evg_obs_row_bytes(env._h, evg._capi.OBS_WIRE))
    rows = torch.empty((T + 1, n, rb), dtype=torch.uint8, device=env.device)
    rows[0].copy_(env.reset(obs_format="wire"))
    for t in range(T):
        env.step(env.agent_actions(evg._capi.AGENT_RANDOM, evg._capi.AGENT_SWARM), obs_format="wire")
        rows[t + 1].copy_(env.obs_rows("wire"))
    r = torch.empty((T * n, 2), dtype=torch.float32, device=env.device)
    d = torch.empty((T * n,), dtype=torch.uint8, device=env.device)
    env.expand_wire(rows[1:].reshape(T * n, rb), reward=r, done=d)
    rn, dn = r.view(T, n, 2).cpu().numpy(), d.view(T, n).cpu().numpy().astype(bool)
    assert dn[24:].all() and not dn[0].all()
    values = np.random.default_rng(2).standard_normal((T + 1, n, 2)).astype(np.float32)
    adv, ret = env.gae(torch.from_numpy(values).to(env.device), rows=rows)
    adv, ret = adv.cpu().numpy(), ret.cpu().numpy()
    want = reference_gae(values, rn, dn, 0.99, 0.95)
    assert np.array_equal(bits(adv), bits(want[0])) and np.array_equal(bits(ret), bits(want[1]))
    one_turn = rn - values[:-1]  # float32 r_t - V_t
    assert np.array_equal(bits(adv[dn]), bits(one_turn[dn])) and np.array_equal(bits(ret[dn]), bits((one_turn + values[:-1])[dn]))


def critic_for(env, seed=0, latent=64):
    import torch
    from evgsim import policy
    torch.manual_seed(seed)
    net = torch.nn.Sequential(torch.nn.Linear(env.obs_len, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                              torch.nn.Linear(latent, 1)).to(env.device)
    return policy.FusedValue(env, net)


def test_pipeline_critic_then_gae(evg):  # noqa: F811
    import torch
    env, rows, reward, done = staggered_rollout(evg, evg._capi.AUTORESET_TERMINAL, n=777, T=50, seed=11)
    T1, n, rb = rows.shape
    critic = critic_for(env)
    with torch.no_grad():
        values = critic(rows.view(T1 * n, rb), obs_format="wire").view(T1, n, 2)
    vn, rn, dn = values.cpu().numpy(), reward.cpu().numpy(), done.cpu().numpy()
    for gamma, lam in ((0.99, 0.95), (1.0, 1.0)):
        adv, ret = env.gae(values, rows=rows, gamma=gamma, lam=lam)
        want = reference_gae(vn, rn, dn, gamma, lam)
        assert np.array_equal(bits(adv), bits(want[0])) and np.array_equal(bits(ret), bits(want[1])), (gamma, lam)
        a64, r64 = gae_float64(vn, rn, dn, gamma, lam)
        ea, er = gae_bound(vn, rn, dn, gamma, lam)
        a, r = adv.cpu().numpy().astype(np.float64), ret.cpu().numpy().astype(np.float64)
        assert np.all(np.abs(a - a64) <= ea) and np.all(np.abs(r - r64) <= er), (gamma, lam)


def test_cuda_graph_and_no_allocation(evg):  # noqa: F811
    import torch
    env, rows, reward, done = staggered_rollout(evg, evg._capi.AUTORESET_NEXT, n=300, T=33, seed=4)
    T1, n, rb = rows.shape
    critic = critic_for(env, seed=1)
    flat = rows.view(T1 * n, rb)
    vals = torch.empty((T1 * n, 2), dtype=torch.float32, device=env.device)
    adv = torch.empty((T1 - 1, n, 2), dtype=torch.float32, device=env.device)
    ret = torch.empty_like(adv)

    def run():
        critic(flat, obs_format="wire", out=vals)
        return env.gae(vals.view(T1, n, 2), rows=rows, adv=adv, ret=ret)

    with torch.no_grad():
        a, r = run()
        assert a is adv and r is ret
        torch.cuda.synchronize()
        want_a, want_r = adv.clone(), ret.clone()
        before = torch.cuda.memory_allocated(env.device)
        torch.cuda.set_sync_debug_mode("error")
        try:
            env.gae(vals.view(T1, n, 2), rows=rows, adv=adv, ret=ret)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert torch.cuda.memory_allocated(env.device) == before
        cur = torch.cuda.current_stream(env.device)
        side = torch.cuda.Stream(env.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            run()  # warm-up outside the capture
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                run()
        cur.wait_stream(side)
        for _ in range(2):
            adv.fill_(float("nan"))
            ret.fill_(float("nan"))
            vals.fill_(float("nan"))
            g.replay()
            torch.cuda.synchronize()
            assert np.array_equal(bits(adv), bits(want_a)) and np.array_equal(bits(ret), bits(want_r))


def test_wrapper_refuses_before_launching(evg):  # noqa: F811
    import torch
    env, rows, reward, done = staggered_rollout(evg, evg._capi.AUTORESET_TERMINAL, n=64, T=4, seed=2, turn_limit=10)
    dev = env.device
    T1, n, rb = rows.shape
    values = torch.zeros((T1, n, 2), device=dev)
    before = env.launch_count
    bad = [
        dict(values=values.double(), rows=rows),                             # dtype
        dict(values=values.cpu(), rows=rows),                                # device
        dict(values=values.transpose(0, 1).contiguous().transpose(0, 1), rows=rows),  # not contiguous
        dict(values=values[:1], rows=rows[:1]),                              # T = 0
        dict(values=values, rows=rows, player=0),                            # [T+1, M, 2] for one player
        dict(values=values[..., 0].contiguous(), rows=rows),                 # [T+1, M] for both
        dict(values=values, rows=rows, player=2),
        dict(values=values, rows=rows[:, :, :64].contiguous()),              # row width
        dict(values=values, rows=rows[:-1]),                                 # T+1 rows
        dict(values=values, rows=rows.view(T1 * n, rb)),                     # flattened rows
        dict(values=values, rows=rows.float()),
        dict(values=values),                                                 # no rows, no float tensors
        dict(values=values, reward=reward),                                  # no rows, no done
        dict(values=values, done=done),                                      # no rows, no reward
        dict(values=values, rows=rows, reward=reward[:, :, :1].contiguous()),
        dict(values=values, rows=rows, reward=reward.double()),
        dict(values=values, rows=rows, done=done.bool()),
        dict(values=values, rows=rows, done=done[1:]),
        dict(values=values, rows=rows, adv=torch.empty((T1, n, 2), device=dev)),
        dict(values=values, rows=rows, ret=torch.empty((T1 - 1, n, 2), device=dev, dtype=torch.float64)),
        dict(values=values, rows=rows, adv=torch.empty((T1 - 1, n, 2))),
        dict(values=values, rows=rows, gamma=1.5),
        dict(values=values, rows=rows, gamma=float("nan")),
        dict(values=values, rows=rows, lam=-0.1),
        dict(values=values, rows=rows, lam=float("inf")),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            env.gae(**kw)
    assert env.launch_count == before
    env.gae(values, rows=rows)
    assert env.launch_count == before + 1


def test_abi_refuses_bad_arguments(evg):  # noqa: F811
    import torch
    env, rows, reward, done = staggered_rollout(evg, evg._capi.AUTORESET_TERMINAL, n=64, T=4, seed=2, turn_limit=10)
    dev = env.device
    T1, n, _ = rows.shape
    values = torch.zeros((T1, n, 2), device=dev)
    adv = torch.empty((T1 - 1, n, 2), device=dev)
    ret = torch.empty_like(adv)
    ptr = lambda t, off=0: C.c_void_p(t.data_ptr() + off)  # noqa: E731
    null = C.c_void_p()
    lib, h, s = env._lib, env._h, env._stream()
    base = dict(T=T1 - 1, M=n, player=-1, rows=ptr(rows), reward=null, done=null, values=ptr(values), gamma=0.99, lam=0.95,
                adv=ptr(adv), ret=ptr(ret))

    def call(**kw):
        a = dict(base, **kw)
        return lib.evg_gae(h, a["T"], a["M"], a["player"], a["rows"], a["reward"], a["done"], a["values"], a["gamma"], a["lam"],
                           a["adv"], a["ret"], s)

    before = env.launch_count
    cases = [
        dict(T=0), dict(T=-3), dict(M=0), dict(M=-1), dict(M=1 << 31),
        dict(player=-2), dict(player=2),
        dict(values=null), dict(adv=null), dict(ret=null),
        dict(rows=null), dict(rows=null, reward=ptr(reward)), dict(rows=null, done=ptr(done)),
        dict(rows=ptr(rows, 8)),
        dict(values=ptr(values, 4)), dict(adv=ptr(adv, 4)), dict(ret=ptr(ret, 4)), dict(reward=ptr(reward, 4)),
        dict(gamma=-0.5), dict(gamma=1.0001), dict(gamma=float("nan")), dict(gamma=float("inf")),
        dict(lam=-1e-7), dict(lam=2.0), dict(lam=float("nan")), dict(lam=float("-inf")),
    ]
    for kw in cases:
        assert call(**kw) == -1, kw
    assert lib.evg_gae(None, T1 - 1, n, -1, ptr(rows), null, null, ptr(values), 0.99, 0.95, ptr(adv), ptr(ret), s) == -1
    assert env.launch_count == before
    assert call() == 0 and env.launch_count == before + 1
    # one player's float operands need only 4-byte alignment
    v1 = torch.zeros((T1 * n + 1,), device=dev)
    assert call(player=1, values=ptr(v1, 4), reward=ptr(reward), done=ptr(done)) == 0
    torch.cuda.synchronize()
