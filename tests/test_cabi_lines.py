"""Several count lines per stream in the state blob, without a GPU: n_lines 0 and 1 keep the one-line layout, L lines
grow only `counts` (i64 [S,L,C,4]) and shift what follows by the same amount, n_lines outside 1..32 is rejected, and
BatchedTracker rejects bad `lines` arguments before any CUDA work."""
import ctypes

import pytest

LABELS = ["person", "bicycle", "motorbike"]
S = 10


def _lib():
    from deepdish_b200 import _lib, build
    build.build()
    return _lib, _lib.lib()


def _layout(lib, cfg):
    from deepdish_b200 import _lib as L
    lay = L.TrackerLayout()
    rc = lib.dd_tracker_layout_query(ctypes.byref(cfg), ctypes.byref(lay))
    return rc, lay


def _align(x):
    return (x + 255) // 256 * 256


@pytest.mark.parametrize("cap", [0, 64])
def test_zero_and_one_line_are_the_one_line_layout(cap):
    _l, lib = _lib()
    cfg0 = _l.make_config(S, 16, 8, 20, LABELS, event_cap=cap, n_lines=0)
    rc0, a = _layout(lib, cfg0)
    rc1, b = _layout(lib, _l.make_config(S, 16, 8, 20, LABELS, event_cap=cap, n_lines=1))
    assert rc0 == rc1 == _l.DD_OK
    for n in ["total_bytes"] + _l.LAYOUT_FIELDS + [_l.EVENTS_FIELD]:
        assert getattr(a, n) == getattr(b, n), n
    assert a.mean - a.counts == _align(8 * S * len(LABELS) * 4)
    assert _l.field_specs(cfg0)["counts"] == ("int64", (S, len(LABELS), 4))


@pytest.mark.parametrize("n_lines", [2, 5, 32])
def test_lines_grow_only_counts(n_lines):
    _l, lib = _lib()
    _, one = _layout(lib, _l.make_config(S, 16, 8, 20, LABELS, event_cap=16))
    cfg = _l.make_config(S, 16, 8, 20, LABELS, event_cap=16, n_lines=n_lines)
    rc, many = _layout(lib, cfg)
    assert rc == _l.DD_OK
    shift = _align(8 * S * n_lines * len(LABELS) * 4) - _align(8 * S * len(LABELS) * 4)
    assert shift > 0
    names = _l.LAYOUT_FIELDS + [_l.EVENTS_FIELD]
    k = names.index("counts")
    for n in names[:k + 1]:
        assert getattr(many, n) == getattr(one, n), n
    for n in names[k + 1:] + ["total_bytes"]:
        assert getattr(many, n) == getattr(one, n) + shift, n
    assert _l.field_specs(cfg)["counts"] == ("int64", (S, n_lines, len(LABELS), 4))
    assert _l.field_specs(cfg)["path_crossed"] == ("int32", (S, 16))


@pytest.mark.parametrize("n_lines", [33, -1])
def test_out_of_range_line_counts_are_rejected(n_lines):
    _l, lib = _lib()
    cfg = _l.make_config(4, 16, 8, 20, ["person"], n_lines=n_lines)
    assert _layout(lib, cfg)[0] == _l.DD_ERR_INVALID
    assert lib.dd_tracker_init(None, ctypes.byref(cfg), None) == _l.DD_ERR_INVALID


@pytest.mark.parametrize("kw", [
    dict(line=(0.0, 0.0, 1.0, 1.0), lines=[(0.0, 0.0, 1.0, 1.0)]),       # both
    dict(lines=[[0.0, 0.0, 1.0, 1.0]] * 33),                              # too many
    dict(lines=[[0.0, 0.0, 1.0]] * 2),                                     # not segments
    dict(lines=[[[0.0, 0.0, 1.0, 1.0]] * 2] * 3),                          # per stream, wrong stream count
    dict(lines=[(0.0, 0.0, 1.0, 1.0)] * 0),                               # none
])
def test_tracker_rejects_bad_lines_before_touching_cuda(kw):
    from deepdish_b200.batched import BatchedTracker
    with pytest.raises(ValueError):
        BatchedTracker(4, ["person"], **kw)
