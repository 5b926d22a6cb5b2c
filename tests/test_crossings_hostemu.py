"""Crossing records on the CPU: the count-line body k_countline<true> runs, compiled with a one-lane group, lists
one record per counter increment -- live crossings in tracker.tracks order, then the deletion record -- exactly as the
oracle's process_results counts them, tick by tick, across frame-presence drops; an overflowing list counts every
record and writes the first event_cap."""
import numpy as np
import pytest

from deepdish_b200 import _lib as L
from tests import crossings as X
from tests import presence as P
from tests.hostemu.driver import HostEmuTracker
from tests.parity import compare_stream


@pytest.fixture(scope="module")
def scene():
    return X.CrossingScene()


def _emu(cap):
    return HostEmuTracker(L.make_config(X.S, X.T, X.DMAX, P.BUDGET, X.LABELS, max_age=P.MAX_AGE, event_cap=cap),
                          line=X.LINE)


def _tick(emu, b, p):
    return emu.tick(b.tlwh.numpy(), b.conf.numpy(), b.label.numpy(), b.feat.numpy(), b.count.numpy(), p)


def test_scene_has_every_case(scene):
    c = scene.cases()
    assert all(v > 0 for v in c.values()), c


def test_records_match_the_oracle_tick_by_tick(scene):
    emu = _emu(512)
    total = np.zeros((X.S, len(X.LABELS), 4), np.int64)
    n_rec = 0
    for f, (b, p, exp) in enumerate(zip(scene.frames, scene.present, scene.ids)):
        P.check_tick_ids(_tick(emu, b, p), exp, p, f)
        n, rec = emu.events()
        want = scene.tick_records(f)
        assert n == len(want), f
        np.testing.assert_array_equal(rec, want, err_msg="tick %d" % f)
        total += X.fold(rec, X.S, len(X.LABELS))
        np.testing.assert_array_equal(total, emu.v["counts"], err_msg="fold, tick %d" % f)
        n_rec += n
    assert n_rec > 200
    for s in range(X.S):
        compare_stream(scene.orc.trk[s], scene.orc.cnt[s], emu.v, s, X.LABELS)


def test_overflow_counts_every_record_and_writes_cap(scene):
    cap = 3
    emu = _emu(cap)
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
    # the records never touch the tracking: same counters as the oracle
    for s in range(X.S):
        np.testing.assert_array_equal(emu.v["counts"][s], scene.orc.cnt[s].counts(X.LABELS))
