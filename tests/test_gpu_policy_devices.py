"""The fused policies (FusedDQN, FusedPPO, FusedRPPO) with simulators on two GPUs in one process.

The policy kernels need more than 48 KB of dynamic shared memory, and the opt-in to it is a per-device attribute of the
kernel: evg_create makes it on the simulator's own device.  Each family plays a few turns on cuda:0 and on cuda:1, turn
by turn in that order, and every device's action rows and outputs must equal those of a run on cuda:0 alone with the same
seed (the draws are keyed on the tape, so the device does not change them).  Skipped with fewer than two GPUs."""
import pytest

pytestmark = pytest.mark.gpu

TURNS = 4


@pytest.fixture(scope="module")
def evg():
    import __graft_entry__ as g
    g.build()
    import evgsim
    return evgsim


def play(evg, family, device):
    """Per turn of self-play on `device` (300 matches: 600 rows, the last tile partial): the wrapper's outputs and the
    action rows, on the host."""
    from test_gpu_policy_refresh import make
    env = evg.BatchedEvergladesEnv(300, device=device, seed=5)
    env.reset()
    net, cls = make(family, env.obs_len, 528 if family == "dqn" else 128, 132, env.device, seed=1)
    fused = cls(env, net)
    for _ in range(TURNS):
        if family == "dqn":
            out = [fused.forward().clone(), fused.forward_t().clone()]
            actions = fused()
        else:
            actions = fused(want_probs=True)
            out = [fused.idx.clone(), fused.probs.clone()] + ([fused.hidden.clone()] if family == "rppo" else [])
        out.append(actions.clone())
        env.step(actions)
        yield [t.cpu() for t in out]


@pytest.mark.parametrize("family", ["dqn", "ppo", "rppo"])
def test_two_devices_equal_one(evg, family):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    alone = list(play(evg, family, 0))
    on0, on1 = play(evg, family, 0), play(evg, family, 1)
    for t, ref in enumerate(alone):
        a, b = next(on0), next(on1)  # cuda:0's turn, then cuda:1's
        for k, (r, x, y) in enumerate(zip(ref, a, b)):
            assert torch.equal(r, x) and torch.equal(r, y), (family, t, k)
