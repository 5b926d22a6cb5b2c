"""bench.py --dump-outputs: the arrays last_step_outputs takes from the timed path (det -> track ids, counters, live
tracks in track order) against the oracle on a small scene with more streams than the covariance sample."""
import numpy as np
import pytest
import torch

import bench
from tests.parity import OracleStreams, LABELS3

pytestmark = pytest.mark.gpu


def test_last_step_outputs_match_oracle():
    from deepdish_b200.batched import BatchedTracker
    from deepdish_b200.scene import Scene
    S = bench.DUMP_COV_STREAMS + 16
    bt = BatchedTracker(S, LABELS3, max_tracks=48, max_dets=16, budget=20, max_age=30, device="cuda:0", n_chunks=2)
    orc = OracleStreams(S, LABELS3, budget=20, max_age=30)
    sc = Scene(S, 12, 16, n_labels=3, seed=5)
    for _ in range(30):
        b = sc.step()
        ids = orc.step(b)
        dev = b.to("cuda:0")
        got = bt.step(dev, join=False, reduce=True)
        counts = bt.all_reduce_counts(reduced=True, async_op=True)
    bt.join()
    bt.wait_counts()
    torch.cuda.synchronize()
    d = bench.last_step_outputs(bt, dev, got, counts)
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in d.values())
    pick = d["track_cov_streams"].astype(int)
    assert len(pick) == bench.DUMP_COV_STREAMS and np.all(np.diff(pick) > 0)
    np.testing.assert_array_equal(d["counts"], sum(c.counts(LABELS3) for c in orc.cnt))
    for s in range(S):
        n, trk = len(ids[s]), orc.trk[s].tracks
        nt = len(trk)
        assert list(d["det_track_id"][s, :n]) == ids[s] and np.all(d["det_track_id"][s, n:] == -1), s
        assert list(d["track_id"][s, :nt]) == [t.track_id for t in trk] and np.all(d["track_id"][s, nt:] == -1), s
        assert list(d["track_state"][s, :nt]) == [t.state for t in trk]
        assert list(d["track_tsu"][s, :nt]) == [t.time_since_update for t in trk]
        np.testing.assert_array_equal(d["stream_counts"][s], orc.cnt[s].counts(LABELS3))
        assert not d["track_mean"][s, nt:].any()
        if nt:
            np.testing.assert_allclose(d["track_mean"][s, :nt], np.stack([t.mean for t in trk]), rtol=1e-4, atol=1e-9)
    for i, s in enumerate(pick):
        trk = orc.trk[s].tracks
        assert not d["track_cov"][i, len(trk):].any()
        if trk:
            np.testing.assert_allclose(d["track_cov"][i, :len(trk)], np.stack([t.covariance for t in trk]),
                                       rtol=1e-4, atol=1e-12)
