"""The crossing-record section of the state blob and its entry point, without a GPU: appended after every other array,
0 bytes when off, every other offset independent of event_cap; bad arguments rejected before any CUDA work."""
import ctypes

import pytest


def _lib():
    from deepdish_b200 import _lib, build
    build.build()
    return _lib, _lib.lib()


def _layout(lib, cfg):
    from deepdish_b200 import _lib as L
    lay = L.TrackerLayout()
    rc = lib.dd_tracker_layout_query(ctypes.byref(cfg), ctypes.byref(lay))
    return rc, lay


@pytest.mark.parametrize("cap", [1, 7, 4096])
def test_events_section_is_appended_and_free_when_off(cap):
    _l, lib = _lib()
    mk = lambda c: _l.make_config(10, 16, 8, 20, ["person", "bicycle", "motorbike"], event_cap=c)
    rc0, off = _layout(lib, mk(0))
    rc1, on = _layout(lib, mk(cap))
    assert rc0 == rc1 == _l.DD_OK
    for n in _l.LAYOUT_FIELDS:
        assert getattr(off, n) == getattr(on, n), n
    # off: no bytes, the blob ends where it ended before the section existed
    assert off.events == off.total_bytes == (off.tick_present + 4 * 10 + 255) // 256 * 256
    # on: header + cap records of 16 bytes, behind every other array
    assert on.events == off.total_bytes and on.total_bytes == (on.events + 16 * (1 + cap) + 255) // 256 * 256
    assert _l.field_specs(mk(cap))["events"] == ("int32", (cap + 1, 4))
    assert _l.field_specs(mk(0))["events"] == ("int32", (0, 4))


def test_negative_event_cap_is_rejected():
    _l, lib = _lib()
    cfg = _l.make_config(4, 16, 8, 20, ["person"], event_cap=-1)
    assert _layout(lib, cfg)[0] == _l.DD_ERR_INVALID
    assert lib.dd_tracker_init(None, ctypes.byref(cfg), None) == _l.DD_ERR_INVALID


def test_copy_events_is_exported_and_checks_its_arguments():
    _l, lib = _lib()
    assert hasattr(lib, "dd_engine_copy_events")
    assert lib.dd_engine_copy_events(None, None, None) == _l.DD_ERR_INVALID


def test_tracker_rejects_a_negative_capacity_before_touching_cuda():
    from deepdish_b200.batched import BatchedTracker
    with pytest.raises(ValueError):
        BatchedTracker(4, ["person"], crossing_capacity=-1)
