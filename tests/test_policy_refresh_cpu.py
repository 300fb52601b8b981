"""Host side of refresh() (FusedDQN / FusedPPO / FusedRPPO): the entry points it calls refuse a null handle, and every
check it makes on the module's parameters is made before any device call.  The packing itself is checked against the
numpy packers in tests/test_gpu_policy_refresh.py."""
import copy
import types

import pytest

from evgsim import _capi, policy


def _env(device="cpu", obs_len=105, num_envs=4):
    """Only what the wrappers read before their first device call."""
    import torch
    return types.SimpleNamespace(obs_len=obs_len, num_envs=num_envs, device=torch.device(device))


class Actor:
    """The reference ActorCritic's recurrent actor."""

    def __init__(self, torch, latent, **gru_kw):
        torch.manual_seed(0)
        self.action_head = torch.nn.Sequential(torch.nn.Linear(105, latent), torch.nn.Tanh(), torch.nn.Linear(latent, latent), torch.nn.Tanh())
        self.action_gru = torch.nn.GRU(latent, latent, **gru_kw)
        self.action_layer = torch.nn.Sequential(torch.nn.Linear(latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))


def _nets(torch, family, size):
    if family == "dqn":
        return policy.FusedDQN, torch.nn.Sequential(torch.nn.Linear(105, size), torch.nn.ReLU(), torch.nn.Linear(size, 132))
    if family == "ppo":
        return policy.FusedPPO, torch.nn.Sequential(torch.nn.Linear(105, size), torch.nn.Tanh(), torch.nn.Linear(size, size), torch.nn.Tanh(),
                                                    torch.nn.Linear(size, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
    return policy.FusedRPPO, Actor(torch, size)


def _first_weight(family, net):
    return net.action_head[0] if family == "rppo" else net[0]


@pytest.mark.parametrize("case", ["float64", "not_contiguous", "wider", "other_out", "other_device"])
@pytest.mark.parametrize("family", ["dqn", "ppo", "rppo"])
def test_refresh_refuses_parameters_the_images_were_not_built_for(family, case):
    import torch
    cls, net = _nets(torch, family, 32)
    fused = cls(_env(), net)
    bad = copy.deepcopy(net)
    lin = _first_weight(family, bad)
    if case == "float64":
        lin.weight.data = lin.weight.data.double()
    elif case == "not_contiguous":
        lin.weight.data = lin.weight.data.t().contiguous().t()
    elif case == "wider":
        bad = _nets(torch, family, 33)[1]
    elif case == "other_out":
        out_layer = bad.action_layer[0] if family == "rppo" else bad[-3 if family == "ppo" else 2]
        out_layer.weight.data = torch.zeros((144, 32))
    else:
        fused = cls(_env("meta"), net)
    with pytest.raises(ValueError):
        fused.refresh(bad)


def test_refresh_of_a_wrapper_built_from_arrays_needs_a_module():
    import torch
    _, net = _nets(torch, "dqn", 16)
    fused = policy.FusedDQN(_env(), weights=[t.detach().numpy() for t in net.parameters()])
    with pytest.raises(ValueError, match="weights="):
        fused.refresh()
    _, net = _nets(torch, "ppo", 16)
    fused = policy.FusedPPO(_env(), weights=[t.detach().numpy() for t in net.parameters()])
    with pytest.raises(ValueError, match="weights="):
        fused.refresh()


@pytest.mark.parametrize("kw", [dict(num_layers=2), dict(bidirectional=True), dict(bias=False)])
def test_rppo_refresh_refuses_a_gru_the_kernel_does_not_run(kw):
    import torch
    fused = policy.FusedRPPO(_env(), Actor(torch, 32))
    with pytest.raises(ValueError):
        fused.refresh(Actor(torch, 32, **kw))


def test_null_handle_calls_fail():
    import __graft_entry__ as g
    g.build()
    lib = _capi.load()
    assert lib.evg_pack_mlp(None, None, None, None, None, 528, 132, None, None, None) == -1
    assert lib.evg_pack_ppo(None, None, None, None, None, None, None, 128, 132, None, None, None, None, None) == -1
    assert lib.evg_pack_rppo(None, None, None, None, None, None, None, None, None, None, None, 128, 132, None, None, None, None, None,
                             None, None) == -1
