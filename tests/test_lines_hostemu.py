"""Several count lines per camera on the CPU: the count-line body k_countline_lines runs, compiled with a one-lane group,
counts every line of every stream exactly as an oracle LineCounter of that line counts it, tick by tick, across
frame-presence drops; with records on it lists them merged in the device's order (tracker.tracks, each track's lines
ascending, then the deletion records, lines ascending) and an overflowing list counts every record and writes the first
event_cap.  The line sets hold the default mid-line, the frame's diagonal twice, a horizontal line, a line outside the
frame and a line of each stream's own."""
import numpy as np
import pytest

from deepdish_b200 import _lib as L
from tests import crossings as X
from tests import lines as LN
from tests import presence as P
from tests.hostemu.lines import HostEmuLinesTracker
from tests.parity import compare_stream


@pytest.fixture(scope="module")
def scene():
    return LN.LinesScene(LN.per_stream_lines())


def _emu(scene, cap):
    n = scene.lines.shape[1]
    return HostEmuLinesTracker(L.make_config(X.S, X.T, X.DMAX, P.BUDGET, X.LABELS, max_age=P.MAX_AGE, event_cap=cap,
                                             n_lines=n), scene.lines)


def _tick(emu, b, p):
    return emu.tick(b.tlwh.numpy(), b.conf.numpy(), b.label.numpy(), b.feat.numpy(), b.count.numpy(), p)


def _check_counts(emu, scene, f):
    want = scene.counts_at[f]
    assert emu.v["counts"].shape == want.shape
    for s in range(X.S):
        for l in range(want.shape[1]):
            np.testing.assert_array_equal(emu.v["counts"][s, l], want[s, l], err_msg="tick %d stream %d line %d" % (f, s, l))


def test_scene_has_every_case(scene):
    c = scene.cases()
    assert all(v > 0 for v in c.values()), c
    cnt = scene.counts()
    for s in range(X.S):
        ls = [tuple(x) for x in scene.lines[s]]
        d = [l for l, x in enumerate(ls) if x == LN.DIAG]
        assert len(d) == 2
        np.testing.assert_array_equal(cnt[s, d[0]], cnt[s, d[1]])          # the duplicate counts identically
        assert not cnt[s, ls.index(LN.OUTSIDE)].any()                      # the line outside the frame counts zero
    assert cnt[..., 2].sum() > 500 and cnt[..., 3].sum() > 20


def test_counts_match_a_line_counter_per_line_every_tick(scene):
    emu = _emu(scene, 0)
    assert emu.lay.events == emu.lay.total_bytes
    for f, (b, p, exp) in enumerate(zip(scene.frames, scene.present, scene.ids)):
        P.check_tick_ids(_tick(emu, b, p), exp, p, f)
        _check_counts(emu, scene, f)
    for s in range(X.S):
        compare_stream(scene.orc.trk[s], None, emu.v, s, X.LABELS)


def test_records_match_the_merged_oracle_records(scene):
    emu = _emu(scene, 1024)
    n_rec = 0
    for f, (b, p, exp) in enumerate(zip(scene.frames, scene.present, scene.ids)):
        P.check_tick_ids(_tick(emu, b, p), exp, p, f)
        n, rec = emu.events()
        want = scene.tick_records(f)
        assert n == len(want), f
        np.testing.assert_array_equal(rec, want, err_msg="tick %d" % f)
        total = (0 if f == 0 else total) + LN.fold(rec, X.S, scene.lines.shape[1], len(X.LABELS))
        np.testing.assert_array_equal(total, emu.v["counts"], err_msg="fold, tick %d" % f)
        n_rec += n
    assert n_rec > 800
    _check_counts(emu, scene, len(scene.frames) - 1)


def test_overflow_counts_every_record_and_writes_cap(scene):
    cap = 5
    emu = _emu(scene, cap)
    over = 0
    for f, (b, p) in enumerate(zip(scene.frames, scene.present)):
        _tick(emu, b, p)
        n, rec = emu.events()
        want = scene.tick_records(f)
        assert n == len(want), f
        assert len(rec) == min(n, cap)
        np.testing.assert_array_equal(rec, want[:cap], err_msg="tick %d" % f)
        over += int(n > cap)
    assert over > 5
    _check_counts(emu, scene, len(scene.frames) - 1)
