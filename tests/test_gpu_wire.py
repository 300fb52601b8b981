"""Compact observation formats of the step (include/evgsim.h EVG_OBS_*): the packed wire row written by the step
kernels themselves and the int16 vector must carry EXACTLY the float32 observations of the oracle — on every step
kernel, with auto-reset, on another map, and through the host-facing chunk pipeline."""
import numpy as np
import pytest

from test_gpu_parity import adjacent_actions
from test_gpu_generic import write_configs, write_ring32

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def evg():
    import __graft_entry__ as g
    g.build()
    import evgsim
    return evgsim


@pytest.fixture(scope="module")
def eo():
    from oracle import evg_oracle
    return evg_oracle


def follow(evg, eo, cfg, n, turns, seed, first, fmt, auto_reset=1):
    from evgsim import wire
    cfg.auto_reset = auto_reset
    env = evg.BatchedEvergladesEnv(n, seed=seed, config=cfg, auto_reset=auto_reset, env_id_offset=first)
    ora = eo.OracleBatch(cfg, n, seed=seed, first=first)
    rows = env.reset(obs_format=fmt).cpu().numpy()
    oobs = ora.reset().astype(np.float32)

    def check(rows, oobs, orew=None, odone=None, ostatus=None, where=""):
        if fmt == "wire":
            obs, rew, done, status = wire.expand(rows, cfg)
            assert np.array_equal(obs, oobs), where
            if orew is not None:
                assert np.array_equal(rew, orew.astype(np.float32)), where
                assert np.array_equal(done, odone) and np.array_equal(status, ostatus), where
        else:
            assert rows.dtype == np.int16 and np.array_equal(rows.astype(np.float32), oobs), where

    check(rows, oobs, where="reset")
    rng = np.random.default_rng(seed)
    ndone = 0
    for t in range(turns):
        acts = adjacent_actions(rng, ora.states, cfg)
        rows, rew, done, info = env.step(acts, obs_format=fmt)
        oobs, orew, odone = ora.step(acts)
        check(rows.cpu().numpy(), oobs.astype(np.float32), orew, odone, ora.status, "turn %d" % (t + 1))
        assert np.array_equal(rew.cpu().numpy(), orew.astype(np.float32)) and np.array_equal(done.cpu().numpy(), odone)
        ndone += int(odone.sum())
    return env, ndone


@pytest.mark.parametrize("fmt", ["wire", "i16"])
@pytest.mark.parametrize("kernel", ["warp", "tpm", "tpm128"])
def test_compact_rows_expand_to_the_oracle_observations(evg, eo, cfg, monkeypatch, kernel, fmt):
    monkeypatch.setenv("EVG_TPM_SMALL_MAX", "0" if kernel == "tpm128" else str(1 << 30))  # "tpm" = one-warp CTAs, forced
    kernel = "tpm" if kernel == "tpm128" else kernel
    monkeypatch.setenv("EVG_STEP_KERNEL", kernel)
    cfg.turn_limit = 70
    try:
        env, ndone = follow(evg, eo, cfg, 1000 + 37, 150, seed=77, first=123, fmt=fmt, auto_reset=2 if fmt == "wire" else 1)
        assert ndone >= 2 * 1037
    finally:
        cfg.turn_limit = 150
        cfg.auto_reset = 0


@pytest.mark.parametrize("kernel", ["warp", "tpm"])
def test_wire_rows_on_other_maps(evg, eo, tmp_path, monkeypatch, kernel):
    """Run-time-sized kernels: a 7-node map with four unit types (112-byte rows) and the
    32-node ring (224-byte rows, two staging chunks per row in the thread-per-match kernel)."""
    monkeypatch.setenv("EVG_STEP_KERNEL", kernel)
    from evgsim import wire
    d = write_configs(tmp_path, 120)
    cfg7 = evg.load_config(d, "Map7.json", "Units4.json", "Setup.json", auto_reset=1)
    env, ndone = follow(evg, eo, cfg7, 300, 130, seed=5, first=0, fmt="wire")
    assert env.obs_rows("wire").shape[1] == wire.row_bytes(7) == 112 and ndone > 300
    d = write_ring32(tmp_path)
    cfg32 = evg.load_config(d, "Ring32.json", evg.DEFAULT_CONFIG_DIR + "/UnitDefinitions.json", "Setup.json", auto_reset=1)
    env, ndone = follow(evg, eo, cfg32, 200, 110, seed=6, first=50, fmt="wire")
    assert env.obs_rows("wire").shape[1] == wire.row_bytes(32) == 224 and ndone >= 400


@pytest.mark.parametrize("fmt", ["wire", "i16"])
def test_step_host_compact_formats_through_the_chunk_pipeline(evg, cfg, fmt):
    """evg_step_host_fmt on a batch large enough for the sub-range launches: host rows == expand-equal to the float32
    observations of a twin simulator stepped on the device, reward and done included (the wire row carries them)."""
    import torch
    from evgsim import wire
    n = 66000 + 21
    a = evg.BatchedEvergladesEnv(n, seed=4, config=cfg, env_id_offset=9)
    b = evg.BatchedEvergladesEnv(n, seed=4, config=cfg, env_id_offset=9)
    a.reset()
    b.reset()
    for t in range(40):
        acts = b.random_actions().clone()
        rows, rew, done, _ = a.step_host(acts.cpu(), obs_format=fmt)
        bobs, brew, bdone, info = b.step(acts)
        torch.cuda.synchronize()
        if fmt == "wire":
            obs, wrew, wdone, wstatus = wire.expand(rows.numpy(), cfg)
            assert np.array_equal(obs, bobs.cpu().numpy()), t
            assert np.array_equal(wrew, brew.cpu().numpy()) and np.array_equal(wdone, bdone.cpu().numpy()), t
            assert np.array_equal(wstatus, info["status"].cpu().numpy()), t
        else:
            assert bool((rows.to(torch.float32) == bobs.cpu()).all()), t
        assert bool((rew == brew.cpu()).all()) and bool((done == bdone.cpu()).all()), t
    assert a.d2h_bytes_per_step(fmt) == n * {"wire": 128, "i16": 420 + 9}[fmt]


def test_wire_with_fused_agents_takes_the_runtime_sized_kernel(evg, cfg, monkeypatch):
    """Scripted agents fused into a wire-row step are not instantiated on the compile-time DemoMap kernel, and no C ABI
    entry point asks for them (evg_step_agents and evg_rollout write float32; the launcher refuses the combination).  The
    wire step with rows from outside (here: random_actions) takes the DemoMap wire instantiation of 128-thread CTAs."""
    monkeypatch.setenv("EVG_STEP_KERNEL", "tpm")
    env = evg.BatchedEvergladesEnv(512, seed=1, config=cfg)
    env.reset()
    rows, _, _, _ = env.step(env.random_actions(), obs_format="wire")
    assert rows.shape == (512, 128)
