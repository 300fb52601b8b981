"""refresh() of FusedDQN / FusedPPO / FusedRPPO: the weight images packed on the device (evg_pack_mlp / _ppo / _rppo,
csrc/evg_policy_pack.cu) from the module's float32 parameters, into the wrapper's own image tensors.

- The device images are byte for byte evgsim.policy.pack_mlp / pack_ppo / pack_rppo's, padding included (the images are
  filled with 0xFF first), for hidden / latent widths at every chunk and swizzle-atom edge, on three observation widths,
  with weights that hold bf16 ties of both parities, signed zeros, subnormals, values that round to +-Inf and +-Inf.
- A NaN weight packs to a bf16 NaN at its byte.
- refresh() + call equals a freshly constructed wrapper, bit for bit; it allocates nothing and does not synchronise.
- A CUDA graph of refresh -> policy -> step, replayed with in-place optimiser steps between turns, equals the same turns
  run eagerly, bit for bit.
- refresh() refuses what the kernel cannot pack (ValueError, images untouched); the ABI returns EVG_E_ARG."""
import copy
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# float32 bit patterns and what round-to-nearest-even makes of them (evgsim.policy.to_bf16_bits)
CRAFTED = np.array([
    0x3F808000, 0xBF808000,  # ties with an even lower bit: stay at 0x3F80 (round-half-up would give 0x3F81)
    0x3F818000, 0xBF818000,  # ties with an odd lower bit: go to 0x3F82 (round-toward-zero would give 0x3F81)
    0x00000000, 0x80000000,  # +-0
    0x00000001, 0x80000001, 0x00008000, 0x00018000, 0x007FFFFF, 0x80408000,  # subnormals, ties among them
    0x7F7FFFFF, 0xFF7FFFFF, 0x7F7F8000, 0xFF7F8000,  # round up to +-Inf
    0x7F800000, 0xFF800000,  # +-Inf
    0x7F7F7FFF,  # the largest value that stays finite
], dtype=np.uint32)
LATENTS = [1, 15, 16, 17, 63, 64, 65, 127, 128, 129, 248, 255, 256]


@pytest.fixture(scope="module")
def evg():
    import __graft_entry__ as g
    g.build()
    import evgsim
    return evgsim


@pytest.fixture(scope="module")
def envs(evg, tmp_path_factory):
    """One small env per observation width: DemoMap (105), the 7-node map (89), the 16-node ring (125)."""
    from test_gpu_generic import write_configs
    from test_gpu_policy_tiling import write_ring16
    cfgs = {105: evg.load_config(),
            89: evg.load_config(write_configs(tmp_path_factory.mktemp("map7"), 100), "Map7.json", "Units4.json", "Setup.json"),
            125: evg.load_config(write_ring16(tmp_path_factory.mktemp("ring16")), "Ring16.json",
                                 evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")}
    out = {}
    for width, cfg in cfgs.items():
        env = evg.BatchedEvergladesEnv(16, seed=1, config=cfg)
        env.reset()
        assert env.obs_len == width
        out[width] = env
    return out


def crafted(rng, shape):
    """Random normals with CRAFTED's values at random places (as many as fit)."""
    a = rng.standard_normal(shape).astype(np.float32)
    flat = a.reshape(-1).view(np.uint32)
    k = min(flat.size, 2 * len(CRAFTED))
    flat[rng.choice(flat.size, k, replace=False)] = CRAFTED[rng.permutation(np.arange(k) % len(CRAFTED))]
    return a


def dqn_net(torch, width, hidden, out):
    return torch.nn.Sequential(torch.nn.Linear(width, hidden), torch.nn.ReLU(), torch.nn.Linear(hidden, out))


def ppo_net(torch, width, latent, out):
    return torch.nn.Sequential(torch.nn.Linear(width, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh(),
                               torch.nn.Linear(latent, out), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))


class Actor:
    """The reference ActorCritic's recurrent actor, as tests/test_gpu_policy_rppo.py: Actor."""

    def __init__(self, torch, width, latent, out, **gru_kw):
        self.action_head = torch.nn.Sequential(torch.nn.Linear(width, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
        self.action_gru = torch.nn.GRU(latent, latent, **gru_kw)
        self.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, out), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))

    def modules(self):
        return (self.action_head, self.action_gru, self.action_layer)

    def parameters(self):
        return [p for m in self.modules() for p in m.parameters()]

    def to(self, dev):
        for m in self.modules():
            m.to(dev)
        return self


def make(family, width, size, out, dev, seed=0):
    """(module on dev, wrapper class) of one family."""
    import torch
    from evgsim import policy
    torch.manual_seed(seed)
    if family == "dqn":
        net, cls = dqn_net(torch, width, size, out), policy.FusedDQN
    elif family == "ppo":
        net, cls = ppo_net(torch, width, size, out), policy.FusedPPO
    else:
        net, cls = Actor(torch, width, size, out), policy.FusedRPPO
    return net.to(dev), cls


def params(family, net):
    from evgsim import policy
    return policy._rppo_params(net) if family == "rppo" else list(net.parameters())


def images(fused):
    return [fused._w1, fused._w2] if hasattr(fused, "_w1") else list(fused._w)


def host_pack(family, ws):
    """What the numpy packer makes of the arrays ws (in module order): images uint8, bias vectors float32."""
    from evgsim import policy
    if family == "dqn":
        return list(policy.pack_mlp(*ws)[:2])
    if family == "ppo":
        return list(policy.pack_ppo(*ws)[:4])
    return list(policy.pack_rppo(*ws)[:6])


def as_bytes(t):
    import torch
    return t.contiguous().view(-1).view(torch.uint8).cpu().numpy()


def load(family, net, rng):
    """Crafted float32 values into every parameter, in place; returns them as numpy arrays (module order)."""
    import torch
    ws = []
    with torch.no_grad():
        for p in params(family, net):
            a = crafted(rng, tuple(p.shape))
            p.copy_(torch.from_numpy(a))
            ws.append(a)
    return ws


def check_refresh_bytes(env, family, size, out, seed):
    import torch
    rng = np.random.default_rng(seed)
    net, cls = make(family, env.obs_len, size, out, env.device, seed)
    fused = cls(env, net)
    ws = load(family, net, rng)
    for t in images(fused):
        t.view(torch.uint8).fill_(0xFF)
    fused.refresh()
    want = host_pack(family, ws)
    got = images(fused)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(as_bytes(g), np.ascontiguousarray(w).view(np.uint8)), (family, i)


@pytest.mark.parametrize("width", [105, 89, 125])
@pytest.mark.parametrize("out", [1, 12, 132, 144])
@pytest.mark.parametrize("hidden", [1, 16, 190, 191, 192, 383, 528, 12288])
def test_dqn_images_are_the_host_packers_bytes(evg, envs, width, hidden, out):
    check_refresh_bytes(envs[width], "dqn", hidden, out, hidden * 7 + out)


@pytest.mark.parametrize("width", [105, 89, 125])
@pytest.mark.parametrize("out", [7, 132, 144])
@pytest.mark.parametrize("latent", LATENTS)
@pytest.mark.parametrize("family", ["ppo", "rppo"])
def test_ppo_images_are_the_host_packers_bytes(evg, envs, family, width, latent, out):
    check_refresh_bytes(envs[width], family, latent, out, latent * 5 + out)


@pytest.mark.parametrize("family", ["dqn", "ppo", "rppo"])
def test_nan_packs_to_a_bf16_nan_at_its_byte(evg, envs, family):
    """NaNs (quiet and signalling) in the first layer's weights and in the last: a bf16 NaN at each one's swizzled byte;
    every other byte is the host packer's."""
    import torch
    from evgsim import policy
    env = envs[105]
    size, out = (528, 132) if family == "dqn" else (129, 132)
    net, cls = make(family, 105, size, out, env.device, 3)
    fused = cls(env, net)
    ws = load(family, net, np.random.default_rng(3))
    last = 2 if family == "dqn" else -2  # w2 / w3
    spots = [(0, size - 9, 17, 0x7FC00000), (0, 5, 104, 0x7F800001), (last, 100, size - 1, 0xFFC00001)]
    for i, r, k, bits in spots:
        ws[i][r, k] = np.uint32(bits).view(np.float32)
        with torch.no_grad():
            params(family, net)[i][r, k] = torch.from_numpy(np.array([bits], dtype=np.uint32).view(np.float32))[0]
    for t in images(fused):
        t.view(torch.uint8).fill_(0xFF)
    fused.refresh()
    got = [as_bytes(t) for t in images(fused)]
    want = [np.ascontiguousarray(w).view(np.uint8).copy() for w in host_pack(family, ws)]
    if family == "dqn":
        c = 192 * 128 * 2, 144 * 192 * 2  # chunk sizes of W1' and W2'
        where = [(0, (r // 192) * c[0] + policy.swz_offset(192, r % 192, k)) for _, r, k, _ in spots[:2]]
        where.append((1, (spots[2][2] // 192) * c[1] + policy.swz_offset(144, spots[2][1], spots[2][2] % 192)))
    else:
        lp = -(-size // 16) * 16
        where = [(0, policy.swz_offset(lp, r, k)) for _, r, k, _ in spots[:2]]
        where.append((len(want) - 2, policy.swz_offset(144, spots[2][1], spots[2][2])))
    for img, off in where:
        v = int(got[img][off:off + 2].view(np.uint16)[0])
        assert v & 0x7F80 == 0x7F80 and v & 0x7F, hex(v)  # exponent all ones, mantissa not zero
        got[img][off:off + 2] = want[img][off:off + 2] = 0
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


def mid_game(evg, n=300, seed=3, turns=12):
    env = evg.BatchedEvergladesEnv(n, seed=seed)
    env.reset()
    for _ in range(turns):
        env.step(env.random_actions())
    return env


def sgd_step(net_params, gen, lr=0.05):
    """An optimiser step: SGD on seeded random gradients, in place."""
    import torch
    opt = torch.optim.SGD(net_params, lr=lr)
    for p in net_params:
        p.grad = torch.randn(p.shape, generator=gen, device=p.device)
    opt.step()


def outputs(family, fused):
    """Everything a call of the wrapper produces, cloned."""
    if family == "dqn":
        q = fused.forward().clone()
        return [q, fused().clone()]
    acts = fused(want_probs=True).clone()
    res = [acts, fused.idx.clone(), fused.probs.clone()]
    if family == "rppo":
        res.append(fused.hidden.clone())
    return res


@pytest.mark.parametrize("family", ["dqn", "ppo", "rppo"])
def test_refresh_equals_a_rebuilt_wrapper(evg, family):
    import torch
    env = mid_game(evg)
    size = {"dqn": 528, "ppo": 128, "rppo": 248}[family]
    net, cls = make(family, 105, size, 132, env.device, 11)
    fused = cls(env, net)
    gen = torch.Generator(device=env.device).manual_seed(1)
    for _ in range(2):
        sgd_step(params(family, net), gen)
    h0 = torch.rand((env.num_envs, 2, size), generator=gen, device=env.device) * 2 - 1
    fused.refresh()
    fresh = cls(env, net)
    if family == "rppo":
        fused.hidden.copy_(h0)
        fresh.hidden.copy_(h0)
    a, b = outputs(family, fused), outputs(family, fresh)
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), i
    for x, y in zip(images(fused), images(fresh)):
        assert torch.equal(x, y)


@pytest.mark.parametrize("family", ["dqn", "ppo", "rppo"])
def test_refresh_allocates_nothing_and_does_not_synchronise(evg, family):
    import torch
    env = mid_game(evg, n=64, turns=1)
    net, cls = make(family, 105, 128, 132, env.device, 2)
    fused = cls(env, net)
    ptrs = [t.data_ptr() for t in images(fused)]
    fused.refresh()  # anything lazily set up on a first call is set up now
    torch.cuda.synchronize()
    before = torch.cuda.memory_stats()["allocation.all.allocated"]
    launches = env.launch_count
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            fused.refresh()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert env.launch_count == launches + 3
    assert torch.cuda.memory_stats()["allocation.all.allocated"] == before
    assert [t.data_ptr() for t in images(fused)] == ptrs


@pytest.mark.parametrize("family", ["dqn", "ppo", "rppo"])
def test_cuda_graph_of_refresh_policy_step_follows_in_place_updates(evg, cfg, family):
    """One capture of refresh -> policy -> step; an optimiser step on the shared module between turns.  The replays equal
    the same turns run eagerly, and the graph's images follow the updates."""
    import torch
    n, size = 1000, {"dqn": 528, "ppo": 128, "rppo": 248}[family]
    cfg.turn_limit = 30
    try:
        envs = [evg.BatchedEvergladesEnv(n, seed=14, config=cfg, auto_reset=1) for _ in range(2)]
    finally:
        cfg.turn_limit = 150
    net, cls = make(family, 105, size, 132, envs[0].device, 21)
    fused = [cls(e, net) for e in envs]
    for e in envs:
        e.reset()

    def turn(k):
        fused[k].refresh()
        fused[k]()
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
    start = [t.clone() for t in images(fused[1])]
    gen = torch.Generator(device=envs[0].device).manual_seed(5)
    for t in range(40):
        sgd_step(params(family, net), gen, lr=0.02)
        turn(0)
        g.replay()
        assert torch.equal(envs[0]._actions, envs[1]._actions), t
        assert torch.equal(envs[0].obs, envs[1].obs), t
        assert torch.equal(envs[0].reward, envs[1].reward), t
        if family == "rppo":
            assert torch.equal(fused[0].hidden, fused[1].hidden), t
    for x, y, s in zip(images(fused[0]), images(fused[1]), start):
        assert torch.equal(x, y) and not torch.equal(y, s)
    torch.cuda.synchronize()
    s0, s1 = envs[0].get_state(), envs[1].get_state()
    assert (s0["episode"] > 0).any()
    for name in ("turn", "episode", "control_state", "controlled_by", "health"):
        assert np.array_equal(s0[name], s1[name]), name


def test_refusals_leave_the_images_untouched(evg, envs):
    import torch
    from evgsim import policy
    env = envs[105]
    rng = np.random.default_rng(0)
    cases = []
    for family, size in (("dqn", 64), ("ppo", 32), ("rppo", 32)):
        net, cls = make(family, 105, size, 132, env.device, 1)
        fused = cls(env, net)
        other, _ = make(family, 105, size + 1, 132, env.device, 1)
        wrong_out, _ = make(family, 105, size, 133, env.device, 1)
        bad = [copy.deepcopy(net).to("cpu"), other, wrong_out]
        dbl = copy.deepcopy(net)
        for m in (dbl.modules() if family == "rppo" else (dbl,)):
            m.double()
        bad.append(dbl)
        nc = copy.deepcopy(net)
        p = params(family, nc)[0]
        p.data = p.data.t().contiguous().t()  # same values and shape, column-major
        assert not p.is_contiguous()
        bad.append(nc)
        if family == "rppo":
            two = Actor(torch, 105, size, 132, num_layers=2).to(env.device)
            bad.append(two)
        cases.append((fused, bad))
    wd = [rng.standard_normal(s).astype(np.float32) for s in ((64, 105), (64,), (132, 64), (132,))]
    from_arrays = policy.FusedDQN(env, weights=wd)
    before = [[t.clone() for t in images(f)] for f, _ in cases] + [[t.clone() for t in images(from_arrays)]]
    for fused, bad in cases:
        for b in bad:
            with pytest.raises(ValueError):
                fused.refresh(b)
    with pytest.raises(ValueError, match="weights="):
        from_arrays.refresh()
    torch.cuda.synchronize()
    after = [[t for t in images(f)] for f, _ in cases] + [images(from_arrays)]
    for x, y in zip(before, after):
        for a, b in zip(x, y):
            assert torch.equal(a, b)
    from_arrays.refresh(dqn_net(torch, 105, 64, 132).to(env.device))  # an explicit module of the right shape is fine


def test_abi_argument_errors_and_launch_count(evg, envs, tmp_path):
    """Bad arguments return EVG_E_ARG (-1) and launch nothing; a good call is one launch.  A map whose observations are
    wider than the kernels' tiling (32 nodes, 189 values) is refused by all three."""
    import torch
    from test_gpu_generic import write_ring32
    env = envs[105]
    dev = env.device
    ptr = lambda t, off=0: C.c_void_p(t.data_ptr() + off)  # noqa: E731
    cfg32 = evg.load_config(write_ring32(tmp_path), "Ring32.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")
    wide = evg.BatchedEvergladesEnv(64, seed=2, config=cfg32)
    assert wide.obs_len == 189
    wide_launches = wide.launch_count

    net, cls = make("dqn", 105, 528, 132, dev, 1)
    fd = cls(env, net)
    w1, b1, w2, b2 = (ptr(t) for t in params("dqn", net))

    def mlp(hidden=528, out=132, i1=None, i2=None, first=None, e=env):
        return e._lib.evg_pack_mlp(e._h, w1 if first is None else first, b1, w2, b2, hidden, out,
                                   i1 or ptr(fd._w1), i2 or ptr(fd._w2), e._stream())

    n = env.launch_count
    assert mlp(first=C.c_void_p()) == -1
    for h, o in ((0, 132), (12289, 132), (528, 0), (528, 145)):
        assert mlp(h, o) == -1, (h, o)
    assert mlp(i1=ptr(fd._w1, 8)) == -1 and mlp(i2=ptr(fd._w2, 8)) == -1
    assert env.launch_count == n
    assert mlp() == 0 and env.launch_count == n + 1
    assert mlp(e=wide) == -1 and b"189" in env._lib.evg_last_error()

    for family in ("ppo", "rppo"):
        net, cls = make(family, 105, 128, 132, dev, 1)
        f = cls(env, net)
        ps = [ptr(t) for t in params(family, net)]
        imgs = [ptr(t) for t in f._w]

        def call(latent=128, out=132, imgs=imgs, ps=ps, e=env):
            if family == "ppo":
                return e._lib.evg_pack_ppo(e._h, *ps, latent, out, *imgs, e._stream())
            w1_, b1_, w2_, b2_, wi, bi, wh, bh, w3_, b3_ = ps
            return e._lib.evg_pack_rppo(e._h, w1_, b1_, w2_, b2_, w3_, b3_, wi, bi, wh, bh, latent, out, *imgs, e._stream())

        n = env.launch_count
        for k in range(len(ps)):
            assert call(ps=ps[:k] + [C.c_void_p()] + ps[k + 1:]) == -1, (family, k)
        for k in range(len(imgs)):
            assert call(imgs=imgs[:k] + [C.c_void_p()] + imgs[k + 1:]) == -1, (family, k)
            assert call(imgs=imgs[:k] + [ptr(f._w[k], 8)] + imgs[k + 1:]) == -1, (family, k)
        for latent, out in ((0, 132), (257, 132), (128, 6), (128, 145)):
            assert call(latent, out) == -1, (family, latent, out)
        assert env.launch_count == n
        assert call() == 0 and env.launch_count == n + 1
        assert call(e=wide) == -1 and b"189" in env._lib.evg_last_error()
    assert wide.launch_count == wide_launches
    torch.cuda.synchronize()
