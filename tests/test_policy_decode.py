"""Policy-in-the-loop glue (SURVEY §8 f-2): the reference agents' action decoding, pinned to the reference's own
code by tests/golden/policy_decode_v1.npz (DQNAgent.filter_actions called unbound on 400 Q-vectors)."""
import os

import numpy as np
import pytest

from oracle import policy_decode as pd

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "policy_decode_v1.npz")


def test_numpy_restatement_matches_reference_filter_actions():
    z = np.load(GOLD)
    for q, a in zip(z["q"], z["actions"]):
        assert np.array_equal(pd.dqn_filter_actions(q), a)
    assert np.array_equal(pd.ppo_unravel(z["ppo_idx"]), z["ppo_actions"])


@pytest.mark.gpu
def test_device_decode_matches_reference():
    import torch
    import __graft_entry__ as g
    g.build()
    import evgsim
    z = np.load(GOLD)
    n = 200
    env = evgsim.BatchedEvergladesEnv(n)
    env.reset()
    q = torch.from_numpy(z["q"][:2 * n].reshape(n, 2, 132))
    rows = env.decode_dqn(q).cpu().numpy()
    assert np.array_equal(rows, z["actions"][:2 * n].reshape(n, 2, 7, 2))
    rows1 = env.decode_dqn(torch.from_numpy(z["q"][2 * n - n:2 * n]), player=1).cpu().numpy()
    assert np.array_equal(rows1[:, 1], z["actions"][n:2 * n]) and np.array_equal(rows1[:, 0], rows[:, 0])
    idx = torch.from_numpy(z["ppo_idx"][:2 * n].astype(np.int64).reshape(n, 2, 7))
    assert np.array_equal(env.decode_indices(idx).cpu().numpy(), z["ppo_actions"][:2 * n].reshape(n, 2, 7, 2))
    # policy in the loop: a DQN-shaped MLP (105 -> 528 -> 132, agents/DQN/QNetwork.py:37,42) on the obs tensor, both players
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(105, 528), torch.nn.ReLU(), torch.nn.Linear(528, 132)).to(env.device)
    obs = env.obs
    for t in range(5):
        with torch.no_grad():
            qv = net(obs.reshape(-1, 105)).reshape(n, 2, 132)
        a = env.decode_dqn(qv)
        want = np.stack([pd.dqn_filter_actions(v) for v in qv.cpu().numpy().reshape(-1, 132)]).reshape(n, 2, 7, 2)
        assert np.array_equal(a.cpu().numpy(), want)
        obs, _, _, _ = env.step(a)


def test_reward_shaping_restatement_matches_reference_functions():
    import importlib.util
    from oracle import ref_harness as rh
    path = os.path.join(rh.REFERENCE_ROOT, "utils", "reward_shaping.py")
    if not os.path.isfile(path):
        pytest.skip("reference checkout not present")
    spec = importlib.util.spec_from_file_location("ref_reward_shaping", path)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    fns = {0: ref.normalized_score, 1: ref.basic_reward, 2: ref.penalize_long_games, 3: ref.reward_short_games}
    rng = np.random.default_rng(0)
    for _ in range(500):
        rew = {0: float(rng.choice([0, 1, -1, 0.3, 0.31])), 1: float(rng.choice([0, 1, -1, 0.3, 0.29]))}
        done, turn = bool(rng.integers(2)), int(rng.integers(0, 150))
        for mode, fn in fns.items():
            for p in (0, 1):
                assert pd.shape_reward(mode, p, rew, done, turn) == fn(p, rew, done, turn)


@pytest.mark.gpu
def test_device_reward_shaping():
    import __graft_entry__ as g
    g.build()
    import evgsim
    cfg = evgsim.load_config(turn_limit=30, auto_reset=1)
    n = 256
    env = evgsim.BatchedEvergladesEnv(n, seed=3, config=cfg, auto_reset=1)
    env.reset()
    for t in range(65):
        obs, rew, done, _ = env.step_agents()
        o, r, d = obs.cpu().numpy(), rew.cpu().numpy().astype(np.float64), done.cpu().numpy()
        for mode in range(4):
            got = env.shape_reward(mode).cpu().numpy()
            want = np.array([[pd.shape_reward(mode, p, r[i], bool(d[i]), float(o[i, 0, 0]) - 1.0) for p in range(2)] for i in range(n)])
            assert np.array_equal(got, want.astype(np.float32)), (t, mode)
