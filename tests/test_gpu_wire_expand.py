"""evg_wire_expand (BatchedEvergladesEnv.expand_wire): wire rows back into the float32 observations on the device.

A simulator stepped in the wire format and a twin stepped in float32, with the same seed and the same actions, hold the
same matches; on every turn the expansion of the first's rows must equal the twin's observations bit for bit (compared
as uint32 patterns, so -0.0 or a NaN payload would show), and equal evgsim.wire.expand on the host.  Reward and done
come out of the row too.  Then the index: duplicates, a reversed order, indices out of range (zeros), one player, n = 1."""
import numpy as np
import pytest

from test_gpu_generic import write_configs, write_ring32

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def evg():
    import __graft_entry__ as g
    g.build()
    import evgsim
    return evgsim


def bits(t):
    return np.ascontiguousarray(t.cpu().numpy()).view(np.uint32)


def twins(evg, cfg, n, seed=5):
    cfg.auto_reset = 1
    saved = cfg.turn_limit
    cfg.turn_limit = 25  # several episodes per slot in the turns below: the automatic resets are expanded too
    try:
        a = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg, auto_reset=1)
        b = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg, auto_reset=1)
    finally:
        cfg.turn_limit, cfg.auto_reset = saved, 0
    return a, b


def maps(evg, tmp_path, which):
    if which == "demo":
        return evg.load_config()
    if which == "map7":
        return evg.load_config(write_configs(tmp_path, 120), "Map7.json", "Units4.json", "Setup.json")
    return evg.load_config(write_ring32(tmp_path), "Ring32.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json")


@pytest.mark.parametrize("which", ["demo", "map7", "ring32"])
@pytest.mark.parametrize("kernel", ["warp", "tpm", "tpm128"])
def test_expansion_equals_the_float32_step(evg, tmp_path, monkeypatch, kernel, which):
    import torch
    from evgsim import wire
    monkeypatch.setenv("EVG_TPM_SMALL_MAX", "0" if kernel == "tpm128" else str(1 << 30))
    monkeypatch.setenv("EVG_STEP_KERNEL", "tpm" if kernel == "tpm128" else kernel)
    cfg = maps(evg, tmp_path, which)
    w, f = twins(evg, cfg, 300)
    rows = w.reset(obs_format="wire")
    f.reset()
    reward = torch.empty((300, 2), dtype=torch.float32, device=w.device)
    done = torch.empty((300,), dtype=torch.uint8, device=w.device)
    ndone = 0
    for t in range(60):
        acts = f.random_actions().clone()
        w.step(acts, obs_format="wire")
        obs, rew, dn, _ = f.step(acts)
        got = w.expand_wire(rows, reward=reward, done=done)
        assert got.shape == (300, 2, f.obs_len) and got.dtype == torch.float32 and got.device == w.device
        assert np.array_equal(bits(got), bits(obs)), (which, kernel, t)
        assert np.array_equal(bits(reward), bits(rew)) and torch.equal(done, dn), (which, kernel, t)
        hobs, hrew, hdone, _ = wire.expand(rows.cpu().numpy(), cfg)
        assert np.array_equal(bits(got), hobs.view(np.uint32)) and np.array_equal(hdone, done.cpu().numpy())
        ndone += int(dn.sum())
    assert ndone >= 300  # every slot went through at least one automatic reset


@pytest.mark.parametrize("which", ["demo", "map7", "ring32"])
def test_index_player_and_out_of_range(evg, tmp_path, which):
    import torch
    cfg = maps(evg, tmp_path, which)
    w, f = twins(evg, cfg, 257)
    rows = w.reset(obs_format="wire")
    f.reset()
    for _ in range(12):
        acts = f.random_actions().clone()
        w.step(acts, obs_format="wire")
        f.step(acts)
    full = f.obs
    dev = w.device
    n = 257
    cases = {
        "dups": torch.tensor([3, 3, 0, 256, 3, 17, 17], device=dev),
        "reversed": torch.arange(n - 1, -1, -1, device=dev),
        "one": torch.tensor([200], device=dev),
        "out": torch.tensor([5, -1, n, 1 << 40, -(1 << 40), 6], device=dev),
    }
    for name, idx in cases.items():
        ok = (idx >= 0) & (idx < n)
        safe = torch.where(ok, idx, torch.zeros_like(idx))
        for player in (-1, 0, 1):
            want = full[safe] if player < 0 else full[safe, player]
            want = torch.where(ok.view(-1, *([1] * (want.dim() - 1))), want, torch.zeros_like(want))
            reward = torch.full((idx.numel(), 2), 7.0, device=dev)
            done = torch.full((idx.numel(),), 9, dtype=torch.uint8, device=dev)
            got = w.expand_wire(rows, index=idx, player=player, reward=reward, done=done)
            assert np.array_equal(bits(got), bits(want)), (name, player)
            assert np.array_equal(bits(reward), bits(torch.where(ok[:, None], f.reward[safe], torch.zeros_like(reward)))), name
            assert torch.equal(done, torch.where(ok, f.done[safe], torch.zeros_like(done))), name
    # n = 1, no index: one stored row on its own
    one = rows[200:201].clone()
    assert np.array_equal(bits(w.expand_wire(one)), bits(full[200:201]))
    assert np.array_equal(bits(w.expand_wire(one, player=1)), bits(full[200:201, 1]))


def test_expand_wire_refuses_bad_tensors_before_launching(evg):
    import torch
    env = evg.BatchedEvergladesEnv(8, seed=1)
    rows = env.reset(obs_format="wire")
    before = env.launch_count
    bad = [
        dict(rows=rows.float()),                       # dtype
        dict(rows=rows[:, :64].clone()),               # width
        dict(rows=rows.cpu()),                         # device
        dict(rows=rows.t().contiguous().t()),          # not contiguous
        dict(rows=rows, index=torch.zeros(3, dtype=torch.int32, device=env.device)),
        dict(rows=rows, index=torch.zeros(3, dtype=torch.int64)),
        dict(rows=rows, out=torch.empty((8, 2, 104), device=env.device)),
        dict(rows=rows, player=2),
        dict(rows=rows, reward=torch.empty((8, 3), device=env.device)),
        dict(rows=rows, done=torch.empty((8,), dtype=torch.int32, device=env.device)),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            env.expand_wire(**kw)
    assert env.launch_count == before
