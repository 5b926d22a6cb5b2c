"""Crossing records on the B200: every tick's records of every stream against the oracle's process_results (live
crossings in tracker.tracks order, then the deletion record), through step() with one and three chunks, captured
graphs and plain launches, gallery turns, step_host_packed running ahead, frame-presence drops and the per-call path;
records off change nothing; an overflowing list raises; the records fold into the device counters."""
import numpy as np
import pytest
import torch

from deepdish_b200.scene import Scene
from tests import crossings as X
from tests import presence as P
from tests.parity import OracleStreams, compare_stream

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
CAP = 256


@pytest.fixture(scope="module")
def scene():
    return X.CrossingScene()


def _tracker(n_chunks=1, cap=CAP, **kw):
    from deepdish_b200.batched import BatchedTracker
    return BatchedTracker(X.S, X.LABELS, max_tracks=X.T, max_dets=X.DMAX, budget=P.BUDGET, max_age=P.MAX_AGE,
                          n_chunks=n_chunks, line=X.LINE, device=DEV, crossing_capacity=cap, **kw)


def _check(got, want, f):
    np.testing.assert_array_equal(np.stack([got.stream, got.track_id, got.label, got.column], axis=1).reshape(-1, 4),
                                  want, err_msg="tick %d" % f)


@pytest.mark.parametrize("graphs", [True, False])
@pytest.mark.parametrize("n_chunks", [1, 3])
def test_step_records_match_the_oracle(scene, n_chunks, graphs):
    bt = _tracker(n_chunks, engine_graphs=graphs)
    assert bt.gallery_turns and all(v > 0 for v in scene.cases().values())
    buf = bt.new_crossings_buffer()
    for f, (b, p, exp) in enumerate(zip(scene.frames, scene.present, scene.ids)):
        ids = bt.step(b.to(DEV), present=torch.from_numpy(p).to(DEV), reduce=True, out_events_host=buf)
        P.check_tick_ids(ids.cpu().numpy(), exp, p, f)
        torch.cuda.synchronize()
        want = scene.tick_records(f)
        _check(bt.crossings(buf), want, f)
        _check(bt.crossings(), want, f)
    bt.check()
    v = bt.host_view()
    for s in range(X.S):
        compare_stream(scene.orc.trk[s], scene.orc.cnt[s], v, s, X.LABELS)


def test_host_path_running_ahead(scene):
    """step_host_packed ticks enqueued back to back without a host synchronisation, three upload buffers in rotation,
    each tick's ids and records copied into pinned buffers of its own; every tick checked after the final join."""
    bt = _tracker(3)
    bt.UPLOAD_BUFFERS = 3
    packed = [bt.pack_host(b, p) for b, p in zip(scene.frames, scene.present)]
    ids = [torch.full((X.S, X.DMAX), -7, dtype=torch.int32).pin_memory() for _ in packed]
    evs = [bt.new_crossings_buffer() for _ in packed]
    for f, pk in enumerate(packed):
        bt.step_host_packed(pk, ids[f], out_events_host=evs[f])
    bt.join()
    torch.cuda.synchronize()
    assert all(len(c.blob_dev) == 3 for c in bt.chunks)
    for f in range(len(packed)):
        P.check_tick_ids(ids[f].numpy(), scene.ids[f], scene.present[f], f)
        _check(bt.crossings(evs[f]), scene.tick_records(f), f)
    bt.check()
    np.testing.assert_array_equal(bt.total_counts.cpu().numpy(), sum(c.counts(X.LABELS) for c in scene.orc.cnt))


def test_per_call_path(scene):
    """predict / update / countline: every stream present, the records of each countline() call."""
    bt = _tracker(2)
    orc = OracleStreams(X.S, X.LABELS, budget=P.BUDGET, max_age=P.MAX_AGE, line=X.LINE)
    orc.cnt = [X.EventCounter(c.line, X.LABELS) for c in orc.cnt]
    n = 0
    for f, b in enumerate(scene.frames[:90]):
        exp = orc.step(b)
        d = b.to(DEV)
        bt.predict()
        got = bt.update(d.tlwh, d.conf, d.label, d.feat, d.count).cpu().numpy()
        bt.countline()
        for s in range(X.S):
            assert list(got[s, :int(b.count[s])]) == exp[s], (f, s)
        want = np.concatenate([X.records(orc.cnt[s], s) for s in range(X.S)])
        _check(bt.crossings(), want, f)
        n += len(want)
    assert n > 50


def _state(bt):
    names = ["n_tracks", "next_id", "n_deleted", "order", "deleted", "counts", "track_id", "hits", "age", "tsu", "state",
             "gal_len", "gal_pos", "mean", "cov", "path_n", "path_last", "path_crossed", "lab_cnt", "lab_sum", "err"]
    return bt.host_view(names)


def test_off_is_off(scene):
    """crossing_capacity 0 and > 0 on the same scene: bit-identical ids, state and total_counts, the same launches."""
    runs = []
    for cap in (0, CAP):
        bt = _tracker(2, cap=cap)
        ids = []
        for b, p in zip(scene.frames, scene.present):
            ids.append(bt.step(b.to(DEV), present=torch.from_numpy(p).to(DEV), reduce=True).cpu().numpy().copy())
        runs.append((ids, _state(bt), bt.total_counts.cpu().numpy(), bt.engine_stats()[1]))
        if cap == 0:
            with pytest.raises(RuntimeError):
                bt.crossings()
            with pytest.raises(RuntimeError):
                bt.new_crossings_buffer()
    (ia, sa, ta, la), (ib, sb, tb, lb) = runs
    for f in range(len(ia)):
        np.testing.assert_array_equal(ia[f], ib[f], err_msg="tick %d" % f)
    for k in sa:
        np.testing.assert_array_equal(sa[k], sb[k], err_msg=k)
    np.testing.assert_array_equal(ta, tb)
    # per tick: 2 chunks x (7 kernels + the partial count reduction) + the count summation
    assert la == lb == len(ia) * (2 * 8 + 1)


def test_overflow_raises_and_tracking_is_unaffected(scene):
    a, b_ = _tracker(2, cap=1), _tracker(2, cap=0)
    raised = 0
    for f, (b, p) in enumerate(zip(scene.frames, scene.present)):
        pr = torch.from_numpy(p).to(DEV)
        ia = a.step(b.to(DEV), present=pr).cpu().numpy()
        ib = b_.step(b.to(DEV), present=pr).cpu().numpy()
        np.testing.assert_array_equal(ia, ib, err_msg="tick %d" % f)
        if max(sum(len(scene.rec[f][s]) for s in range(c.lo, c.hi)) for c in a.chunks) > 1:
            with pytest.raises(RuntimeError, match="chunk"):
                a.crossings()
            raised += 1
        else:
            _check(a.crossings(), scene.tick_records(f), f)
    assert raised > 10
    sa, sb = _state(a), _state(b_)
    for k in sa:
        np.testing.assert_array_equal(sa[k], sb[k], err_msg=k)


def test_fold_invariant_at_256_streams():
    """256 streams on two chunks, 120 ticks: all records since init folded into [S, C, 4] equal the device counters."""
    from deepdish_b200.batched import BatchedTracker
    S, D, TICKS = 256, 24, 120
    bt = BatchedTracker(S, X.LABELS, max_tracks=64, max_dets=D, budget=30, max_age=12, n_chunks=2, line=X.LINE,
                        device=DEV, crossing_capacity=4096)
    sc = Scene(S, 14, D, n_labels=3, seed=9, respawn_prob=0.02)
    sc.vel = sc.vel * 2.0
    bufs = [bt.new_crossings_buffer() for _ in range(3)]
    total = np.zeros((S, len(X.LABELS), 4), np.int64)
    n = 0
    for f in range(TICKS):
        buf = bufs[f % 3]
        bt.step(sc.step().to(DEV), out_events_host=buf)
        torch.cuda.synchronize()
        r = bt.crossings(buf)
        rec = np.stack([r.stream, r.track_id, r.label, r.column], axis=1)
        assert (np.diff(r.stream) >= 0).all()
        total += X.fold(rec, S, len(X.LABELS))
        n += len(rec)
    bt.check()
    np.testing.assert_array_equal(total, bt.host_view(["counts"])["counts"])
    assert n > 1000 and (total[:, :, 3] > 0).any()
