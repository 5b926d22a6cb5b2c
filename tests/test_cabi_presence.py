"""The presence-aware tick entry points and their Python front door reject bad arguments before any CUDA work (no
GPU needed)."""
import ctypes

import pytest
import torch


def _lib():
    from deepdish_b200 import _lib, build
    build.build()
    return _lib, _lib.lib()


def test_presence_entry_points_reject_bad_arguments_without_touching_cuda():
    _l, lib = _lib()
    assert lib.dd_engine_step_present(None, None, None, None, None, None, None, 0, None) == _l.DD_ERR_INVALID
    assert lib.dd_engine_step_host_present(None, None, None, None, None, None) == _l.DD_ERR_INVALID
    # the layout grew by the tick_present word, appended after every other array
    cfg = _l.make_config(10, 16, 8, 20, ["person"])
    lay = _l.TrackerLayout()
    assert lib.dd_tracker_layout_query(ctypes.byref(cfg), ctypes.byref(lay)) == 0
    assert _l.LAYOUT_FIELDS[-1] == "tick_present" and _l.field_specs(cfg)["tick_present"] == ("int32", (10,))
    assert max(getattr(lay, n) for n in _l.LAYOUT_FIELDS) == lay.tick_present
    assert lay.tick_present + 4 * 10 <= lay.total_bytes


class _Fake:
    """Just what BatchedTracker._check_present reads."""
    n_streams = 4
    device = torch.device("cuda", 0)


@pytest.mark.parametrize("present", [torch.ones(4, dtype=torch.int32), torch.ones(5, dtype=torch.bool),
                                     torch.ones(4, dtype=torch.bool), [1, 1, 1, 1], None])
def test_step_present_validation(present):
    from deepdish_b200.batched import BatchedTracker
    with pytest.raises(ValueError):
        BatchedTracker._check_present(_Fake(), present)
