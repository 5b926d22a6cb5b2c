"""Several count lines per camera on the B200: every line's counters of every stream and tick against an oracle
LineCounter of that line, and the merged crossing records (tracker.tracks order, each track's lines ascending, then the
deletion records, lines ascending), through step() with one and three chunks, captured graphs and plain launches, gallery
turns, step_host_packed running ahead and the per-call path, for per-stream and shared line sets; tracking is the
single-line tracker's; lines=[l] is line=l bit for bit with the same launches; state_dict round trip; overflow."""
import numpy as np
import pytest
import torch

from tests import crossings as X
from tests import lines as LN
from tests import presence as P
from tests.parity import OracleStreams, compare_stream

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
CAP = 1024


@pytest.fixture(scope="module")
def scene():
    return LN.LinesScene(LN.per_stream_lines())


@pytest.fixture(scope="module")
def shared():
    return LN.LinesScene(np.broadcast_to(LN.shared_lines(), (X.S,) + LN.shared_lines().shape), ticks=100)


def _tracker(n_chunks=1, cap=CAP, **kw):
    from deepdish_b200.batched import BatchedTracker
    return BatchedTracker(X.S, X.LABELS, max_tracks=X.T, max_dets=X.DMAX, budget=P.BUDGET, max_age=P.MAX_AGE,
                          n_chunks=n_chunks, device=DEV, crossing_capacity=cap, **kw)


def _records(got):
    return np.stack([got.stream, got.track_id, got.label, got.column + 4 * got.line], axis=1).reshape(-1, 4)


def _run_step(bt, sc, check_counts=True):
    from deepdish_b200.batched import LineCrossings
    buf = bt.new_crossings_buffer() if bt.crossing_capacity else None
    for f, (b, p, exp) in enumerate(zip(sc.frames, sc.present, sc.ids)):
        ids = bt.step(b.to(DEV), present=torch.from_numpy(p).to(DEV), reduce=True, out_events_host=buf)
        P.check_tick_ids(ids.cpu().numpy(), exp, p, f)
        torch.cuda.synchronize()
        if buf is not None:
            got = bt.crossings(buf)
            assert isinstance(got, LineCrossings)
            np.testing.assert_array_equal(_records(got), sc.tick_records(f), err_msg="tick %d" % f)
        if check_counts:
            np.testing.assert_array_equal(bt.v["counts"].cpu().numpy(), sc.counts_at[f], err_msg="tick %d" % f)
            np.testing.assert_array_equal(bt.total_counts.cpu().numpy(), sc.counts_at[f].sum(axis=0),
                                          err_msg="tick %d" % f)
    bt.check()


@pytest.mark.parametrize("graphs", [True, False])
@pytest.mark.parametrize("n_chunks", [1, 3])
def test_step_per_stream_lines_match_the_oracle(scene, n_chunks, graphs):
    bt = _tracker(n_chunks, lines=scene.lines, engine_graphs=graphs)
    assert bt.gallery_turns and all(v > 0 for v in scene.cases().values())
    assert tuple(bt.total_counts.shape) == scene.lines.shape[1:2] + (len(X.LABELS), 4)
    _run_step(bt, scene)
    v = bt.host_view()
    for s in range(X.S):
        compare_stream(scene.orc.trk[s], None, v, s, X.LABELS)


def test_step_shared_lines_match_the_oracle(shared):
    bt = _tracker(2, lines=LN.shared_lines())
    assert bt.line_per_stream == 0
    _run_step(bt, shared)


def test_host_path_running_ahead(scene):
    """step_host_packed ticks enqueued back to back without a host synchronisation, three upload buffers in rotation,
    each tick's ids and records copied into pinned buffers of its own; every tick checked after the final join."""
    bt = _tracker(3, lines=scene.lines)
    bt.UPLOAD_BUFFERS = 3
    packed = [bt.pack_host(b, p) for b, p in zip(scene.frames, scene.present)]
    ids = [torch.full((X.S, X.DMAX), -7, dtype=torch.int32).pin_memory() for _ in packed]
    evs = [bt.new_crossings_buffer() for _ in packed]
    for f, pk in enumerate(packed):
        bt.step_host_packed(pk, ids[f], out_events_host=evs[f])
    bt.join()
    torch.cuda.synchronize()
    for f in range(len(packed)):
        P.check_tick_ids(ids[f].numpy(), scene.ids[f], scene.present[f], f)
        np.testing.assert_array_equal(_records(bt.crossings(evs[f])), scene.tick_records(f), err_msg="tick %d" % f)
    bt.check()
    np.testing.assert_array_equal(bt.total_counts.cpu().numpy(), scene.counts_at[-1].sum(axis=0))
    np.testing.assert_array_equal(bt.host_view(["counts"])["counts"], scene.counts_at[-1])


@pytest.mark.parametrize("per_stream", [True, False])
def test_per_call_path(scene, per_stream):
    """predict / update / countline, every stream present: each countline() call's records and every line's counters,
    reduce_counts() summed over streams."""
    lines = scene.lines if per_stream else np.broadcast_to(LN.shared_lines(), (X.S,) + LN.shared_lines().shape)
    bt = _tracker(2, lines=scene.lines if per_stream else LN.shared_lines())
    orc = OracleStreams(X.S, X.LABELS, budget=P.BUDGET, max_age=P.MAX_AGE)
    cnt = [[X.EventCounter(lines[s, l].reshape(2, 2), X.LABELS) for l in range(lines.shape[1])] for s in range(X.S)]
    n = 0
    for f, b in enumerate(scene.frames[:90]):
        exp = [LN._oracle_update(orc.trk[s], b, s, X.LABELS) for s in range(X.S)]
        for s in range(X.S):
            for c in cnt[s]:
                c.step(orc.trk[s])
        d = b.to(DEV)
        bt.predict()
        got = bt.update(d.tlwh, d.conf, d.label, d.feat, d.count).cpu().numpy()
        bt.countline()
        for s in range(X.S):
            assert list(got[s, :int(b.count[s])]) == exp[s], (f, s)
        want = np.concatenate([LN.merged_records(cnt[s], s) for s in range(X.S)])
        np.testing.assert_array_equal(_records(bt.crossings()), want, err_msg="tick %d" % f)
        n += len(want)
    assert n > 200
    want = np.array([[c.counts(X.LABELS) for c in cs] for cs in cnt])
    np.testing.assert_array_equal(bt.host_view(["counts"])["counts"], want)
    np.testing.assert_array_equal(bt.reduce_counts().cpu().numpy(), want.sum(axis=0))
    np.testing.assert_array_equal(bt.all_reduce_counts().cpu().numpy(), want.sum(axis=0))


_TRACKING = ["n_tracks", "next_id", "n_deleted", "order", "deleted", "track_id", "hits", "age", "tsu", "state",
             "gal_len", "gal_pos", "mean", "cov", "path_n", "path_last", "lab_cnt", "lab_sum", "err"]


def _run_plain(bt, sc):
    ids = []
    for b, p in zip(sc.frames, sc.present):
        ids.append(bt.step(b.to(DEV), present=torch.from_numpy(p).to(DEV), reduce=True).cpu().numpy().copy())
    return ids


def test_tracking_is_the_single_line_trackers(scene):
    """ids and every tracking array equal those of a one-line tracker; only counters and path_crossed differ."""
    a, b_ = _tracker(2, cap=0, lines=scene.lines), _tracker(2, cap=0, line=X.LINE)
    ia, ib = _run_plain(a, scene), _run_plain(b_, scene)
    for f in range(len(ia)):
        np.testing.assert_array_equal(ia[f], ib[f], err_msg="tick %d" % f)
    sa, sb = a.host_view(_TRACKING), b_.host_view(_TRACKING)
    for k in _TRACKING:
        np.testing.assert_array_equal(sa[k], sb[k], err_msg=k)


@pytest.mark.parametrize("per_stream", [False, True])
def test_one_line_in_lines_is_line(scene, per_stream):
    """lines=[l] and line=l: bit-identical ids, state, counters and records, the same kernel launches."""
    from deepdish_b200.batched import Crossings
    one = np.array(X.LINE, np.float64)
    line = np.broadcast_to(one, (X.S, 4)).copy() if per_stream else one
    lines = line[:, None, :].copy() if per_stream else line[None, :]
    runs = []
    for kw in (dict(line=line), dict(lines=lines)):
        bt = _tracker(2, cap=256, **kw)
        assert bt.n_lines == 1 and bt.line_per_stream == int(per_stream)
        buf = bt.new_crossings_buffer()
        ids, recs = [], []
        for b, p in zip(scene.frames, scene.present):
            ids.append(bt.step(b.to(DEV), present=torch.from_numpy(p).to(DEV), reduce=True,
                               out_events_host=buf).cpu().numpy().copy())
            torch.cuda.synchronize()
            r = bt.crossings(buf)
            assert isinstance(r, Crossings)
            recs.append(np.stack(r, axis=1))
        runs.append((ids, bt.host_view(_TRACKING + ["counts", "path_crossed"]), bt.total_counts.cpu().numpy(), recs,
                     bt.engine_stats()[1]))
    (ia, sa, ta, ra, la), (ib, sb, tb, rb, lb) = runs
    for f in range(len(ia)):
        np.testing.assert_array_equal(ia[f], ib[f], err_msg="tick %d" % f)
        np.testing.assert_array_equal(ra[f], rb[f], err_msg="tick %d" % f)
    for k in sa:
        np.testing.assert_array_equal(sa[k], sb[k], err_msg=k)
    assert ta.shape == (len(X.LABELS), 4)
    np.testing.assert_array_equal(ta, tb)
    # per tick: 2 chunks x (7 kernels + the partial count reduction) + the count summation
    assert la == lb == len(ia) * (2 * 8 + 1)


def test_state_dict_round_trip(scene):
    half = len(scene.frames) // 2
    a = _tracker(2, cap=0, lines=scene.lines)
    for b, p in zip(scene.frames[:half], scene.present[:half]):
        a.step(b.to(DEV), present=torch.from_numpy(p).to(DEV))
    sd = a.state_dict()
    assert sd["n_lines"] == scene.lines.shape[1]
    b_ = _tracker(2, cap=0, lines=scene.lines)
    b_.load_state_dict(sd)
    for t in (a, b_):
        for b, p in zip(scene.frames[half:], scene.present[half:]):
            t.step(b.to(DEV), present=torch.from_numpy(p).to(DEV))
    np.testing.assert_array_equal(a.host_view(["counts"])["counts"], scene.counts_at[-1])
    np.testing.assert_array_equal(b_.host_view(["counts"])["counts"], scene.counts_at[-1])
    # a different number of lines, and a checkpoint without the key (one line), are refused by a multi-line tracker
    with pytest.raises(ValueError, match="count lines"):
        _tracker(2, cap=0, lines=scene.lines[:, :2]).load_state_dict(sd)
    old = {k: v for k, v in sd.items() if k != "n_lines"}
    with pytest.raises(ValueError, match="count lines"):
        _tracker(2, cap=0, lines=scene.lines).load_state_dict(old)


def test_overflow_raises_and_counting_is_unaffected(scene):
    a = _tracker(2, cap=2, lines=scene.lines)
    raised = 0
    for f, (b, p) in enumerate(zip(scene.frames, scene.present)):
        a.step(b.to(DEV), present=torch.from_numpy(p).to(DEV))
        if max(sum(len(scene.rec[f][s]) for s in range(c.lo, c.hi)) for c in a.chunks) > 2:
            with pytest.raises(RuntimeError, match="chunk"):
                a.crossings()
            raised += 1
        else:
            np.testing.assert_array_equal(_records(a.crossings()), scene.tick_records(f), err_msg="tick %d" % f)
    assert raised > 10
    np.testing.assert_array_equal(a.host_view(["counts"])["counts"], scene.counts_at[-1])
