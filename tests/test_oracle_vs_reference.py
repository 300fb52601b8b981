"""The oracle against the unmodified reference: live where a checkout of the reference is present (see
oracle/ref_harness.py), against the reference's stored results everywhere else.  The committed golden fixtures
(test_oracle_golden.py) carry the random-game comparison to machines without a checkout."""
import numpy as np
import pytest

from conftest import state_fields, flat_health
from oracle import ref_harness as rh, evg_oracle as eo

needs_reference = pytest.mark.skipif(not rh.reference_available(), reason="reference checkout not present")

# (location, travel_destination, distance_remaining, ready, moving) of player 0's group 0 in the reference after the
# turn of test_float_actions_truncate_like_astype_int
FLOAT_ACTION_GROUP0 = [1, 2, 6, 0, 1]


@needs_reference
@pytest.mark.parametrize("seed", [11, 12, 13])
def test_random_game_matches_live_reference(cfg, seed):
    rng = np.random.default_rng(seed)
    acts = np.zeros((150, 2, 7, 2), dtype=np.int64)
    for t in range(150):
        for p in range(2):
            acts[t, p, :, 0] = rng.permutation(12)[:7]
            acts[t, p, :, 1] = rng.permutation(np.arange(1, 12))[:7]
    ref = rh.run_reference_game(seed, seed * 7, acts)
    o = eo.OracleEnv(cfg, seed, seed * 7)
    for t in range(len(ref["done"])):
        obs, rew, done, _, _ = o.step(acts[t])
        assert np.array_equal(obs, ref["obs"][t + 1])
        assert np.array_equal(rew, ref["reward"][t]) and done == ref["done"][t]
        assert np.array_equal(state_fields(o.state[0]), ref["grp"][t + 1])
        assert np.array_equal(flat_health(o.state[0], cfg), ref["health"][t + 1])
        assert np.array_equal(eo.list_rank(o.state[0]), ref["rank"][t + 1])


def test_float_actions_truncate_like_astype_int(cfg):
    """server.py:232 `action.astype(int)`: (0.9, 2.9) commands group 0 to node 2.  The oracle is checked against the
    reference's result stored above; the reference itself too where a checkout is present."""
    acts = np.zeros((1, 2, 7, 2))
    acts[0, 0, 0] = (0.9, 2.9)
    o = eo.OracleEnv(cfg, 1, 0)
    o.step(acts[0])
    assert state_fields(o.state[0])[0, 0].tolist()[:5] == FLOAT_ACTION_GROUP0
    if rh.reference_available():
        ref = rh.run_reference_game(1, 0, acts)
        assert ref["grp"][1][0, 0].tolist()[:5] == FLOAT_ACTION_GROUP0
