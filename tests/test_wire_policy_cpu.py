"""Host side of the wire-row inputs: evg_wire_expand and the policies' _fmt entry points refuse a null handle, and the
wrappers refuse an unknown format or a map too wide for the kernels before any device call."""
import types

import pytest

from evgsim import _capi, policy


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    return _capi.load()


def test_null_handles_are_refused(lib):
    assert lib.evg_wire_expand(None, None, 0, None, 0, -1, None, None, None, None) == -1
    for fmt in (_capi.OBS_F32, _capi.OBS_I16, _capi.OBS_WIRE, 7):
        assert lib.evg_policy_mlp_fmt(None, fmt, None, 0, None, None, 528, 132, None, 0, None) == -1
        assert lib.evg_policy_ppo_fmt(None, fmt, None, -1, None, None, None, None, 128, 132, 12, 11, None, None, None, None) == -1
        assert lib.evg_policy_rppo_fmt(None, fmt, None, -1, None, None, None, None, None, None, 128, 132, 12, 11, None, None, None, None,
                                       None) == -1
    assert b"null" in lib.evg_last_error()


@pytest.mark.parametrize("fmt", ["i16", "F32", "float32", None])
def test_wrappers_refuse_other_formats(fmt):
    with pytest.raises(ValueError, match="obs_format"):
        policy._wire_rows(types.SimpleNamespace(obs_len=105), None, fmt)


def test_wire_input_refuses_observations_wider_than_the_tiling():
    """32 nodes: 189 values per player, past the kernels' 128 input columns."""
    with pytest.raises(ValueError, match="189 values"):
        policy._wire_rows(types.SimpleNamespace(obs_len=189), None, "wire")
