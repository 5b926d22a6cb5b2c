"""Capacity corners on the B200, against the oracle (ids, track table, lifecycle, counters, gallery rows) and against
the exact gallery pass (ids, gate words and the bits of every gate-passing cost): 1024 slots with 988 and 992
detections (31 gate words, the solver at n = 1024, set tables of 4096 slots) on each matching kernel, 960 slots with
1024 detections (32 gate words, the last bit of the last word set), one track passing exactly 64 and 65 gates, one slot
per stream, gallery rings of 1 to 1000 rows and nn_budget=0, and 128 labels counted on 32 lines in two chunks."""
import numpy as np
import pytest
import torch

from deepdish_b200 import _lib as L
from deepdish_b200.scene import Scene, SceneBatch
from tests import capacity as CP
from tests.parity import OracleStreams, compare_stream, compare_costs, LABELS3
from tests.test_gpu_gallery import _history, _compare

pytestmark = pytest.mark.gpu


def _tracker(S, T, D, budget, labels=LABELS3, **kw):
    from deepdish_b200.batched import BatchedTracker
    return BatchedTracker(S, labels, max_tracks=T, max_dets=D, budget=budget, max_age=30, **kw)


def _crowd_tracker(D, match_warps):
    """A crowd's first tick starts ~950 tracks, each taking a gallery page: a pool sized for every slot."""
    return _tracker(1, 1024, D, 4, match_warps=match_warps, pool_fraction=1.0)


def _oracle_run(bt, orc, sc, frames, labels=LABELS3, counters=None, gallery_every=0, costs_from=None, reduce=False):
    """Step the tracker and the oracle on the same batches and compare every tick.  Returns the tracker's history in
    _history's form (for _compare) and the per-tick batches and host views."""
    hist, seen = [], []
    for f in range(frames):
        b = sc.step()
        S = b.count.shape[0]
        pre = bt.host_view(["n_tracks", "order", "track_id"]) if costs_from is not None and f >= costs_from else None
        ids = orc.step(b)
        got = bt.step(b.to("cuda"), reduce=reduce).cpu().numpy().copy()
        bt.maintain(wait=True)
        v = bt.host_view()
        if counters is not None:
            for s in range(S):
                for c in counters[s]:
                    c.step(orc.trk[s])
        post = {"gate": bt.v["gate"].cpu().numpy(), "cost": bt.v["cost"].cpu().numpy()}
        for s in range(S):
            n = int(b.count[s])
            assert list(got[s, :n]) == ids[s], (f, s)
            rows = None
            if gallery_every and (f % gallery_every == gallery_every - 1 or f == frames - 1):
                rows = lambda s_, sl: bt.gallery(s_, sl).cpu().numpy()          # noqa: E731
            compare_stream(orc.trk[s], orc.cnt[s] if counters is None else None, v, s, labels, gallery_rows=rows)
            if pre is not None:
                compare_costs(orc.trk[s], pre, post, s)
        if counters is not None:
            want = CP.line_counts(counters)
            np.testing.assert_array_equal(v["counts"], want, err_msg="counts tick %d" % f)
            if reduce:
                torch.cuda.synchronize()
                np.testing.assert_array_equal(bt.total_counts.cpu().numpy(), want.sum(axis=0))
        hist.append((got, post["gate"].astype(np.uint32), post["cost"], v["state"], int(bt.v["work_ctl"][0])))
        seen.append((b, v))
    bt.check()
    return hist, seen


def _popcounts(gate):
    """Gate-passing detections of every (stream, slot) of a gate array [S, T, DW]."""
    return np.unpackbits(np.ascontiguousarray(gate).view(np.uint8), axis=-1).sum(axis=-1)


@pytest.fixture(scope="module")
def crowd_988():
    """The 1024 x 988 crowd on the one-warp matching kernel, compared with the oracle (costs on the last ticks)."""
    bt = _crowd_tracker(988, 1)
    return _oracle_run(bt, OracleStreams(1, LABELS3, budget=4), CP.crowd(950, 988, seed=3), 12, gallery_every=6,
                       costs_from=10)


def _crowd_reached(hist, seen):
    live = max(int(v["n_tracks"][0]) for _, v in seen)
    dets = max(int(b.count[0]) for b, _ in seen)
    many = max(int(_popcounts(h[1]).max()) for h in hist)
    assert hist[0][1].shape[-1] == 31 and live >= 700 and dets >= 900 and many > 4, (live, dets, many)


def test_crowd_1024_slots_one_warp(crowd_988):
    _crowd_reached(*crowd_988)


@pytest.mark.parametrize("match_warps", [4, 8])
def test_crowd_1024_slots_cta_kernels(crowd_988, match_warps):
    """The 4- and 8-warp matching kernels on the crowd: the oracle's decisions and the one-warp kernel's ids, gate
    words and costs bit for bit."""
    bt = _crowd_tracker(988, match_warps)
    hist, seen = _oracle_run(bt, OracleStreams(1, LABELS3, budget=4), CP.crowd(950, 988, seed=3), 12)
    _crowd_reached(hist, seen)
    checked, _ = _compare("crowd_988_w%d" % match_warps, hist, crowd_988[0])
    assert checked > 2000


def test_crowd_1024_slots_992_detections():
    """Past 988 detections the CTA kernels' 256 extra bytes do not fit and the tick runs the one-warp kernel whatever
    match_warps asks: the same decisions as the oracle, and bit for bit what match_warps=1 computes."""
    runs = []
    for mw in (1, 4):
        bt = _crowd_tracker(992, mw)
        runs.append(_oracle_run(bt, OracleStreams(1, LABELS3, budget=4), CP.crowd(950, 992, seed=3), 12))
    _crowd_reached(*runs[0])
    checked, _ = _compare("crowd_992", runs[1][0], runs[0][0])
    assert checked > 2000


class _Ramp:
    """crowd(900, 1024) without misses or clutter (900 tracks in 960 slots) until tick `full`, then with all 124
    clutter boxes: 1024 detections, 32 gate words, the new tracks overflow the track table (flagged)."""

    def __init__(self, full):
        self.sc = CP.crowd(900, 1024, seed=12, miss_prob=0.0)
        self.sc.clutter_mean = 0.0
        self.f, self.full = 0, full

    def step(self):
        if self.f == self.full:
            self.sc.clutter_mean = 1e9
        self.f += 1
        return self.sc.step()


def test_960_slots_1024_detections_half_prepass_equals_exact():
    kw = dict(S=1, nobj=900, dmax=1024, tmax=960, budget=4, frames=12, seed=12, feat_noise=0.02,
              scene=lambda: _Ramp(9), flags=L.FLAG_TRACK_OVERFLOW, pool_fraction=1.0)
    half, exact = _history("default", **kw), _history("exact", **kw)
    checked, many = _compare("960x1024", half, exact)
    gate = np.stack([h[1] for h in half[9:]])                     # [ticks, S, T, 32]
    assert gate.shape[-1] == 32 and (gate[..., 31] >> 31).any()  # detection 1023 passed a gate
    assert checked > 2000 and many > 4


class _Cluster:
    """One object seen alone for six ticks (a confirmed track), then on one tick `nd` detections inside its gate (all
    of them gate-passing but the one at index `hole`: a full first and second gate word for nd = 64, one detection in
    the third for nd = 65), then alone again."""

    D = 80

    def __init__(self, nd, hole=None):
        self.nd, self.hole, self.f = nd, hole, 0
        g = torch.Generator().manual_seed(nd)
        base = torch.randn(128, generator=g)
        feat = base[None] + 0.01 * torch.randn(nd, 128, generator=g)
        self.feat = feat / feat.norm(dim=1, keepdim=True)

    def step(self):
        n = self.nd if self.f == 6 else 1
        self.f += 1
        tlwh = torch.zeros(1, self.D, 4, dtype=torch.float64)
        i = torch.arange(n)
        tlwh[0, :n, 0] = 300.0 + (i % 8).double() - 4.0
        tlwh[0, :n, 1] = 200.0 + (i // 8).double() - 4.0
        tlwh[0, :n, 2], tlwh[0, :n, 3] = 40.0, 100.0
        if n > 1 and self.hole is not None:
            tlwh[0, self.hole, 0] = 500.0                        # far outside the gate
        conf = torch.zeros(1, self.D)
        conf[0, :n] = 0.9 - 0.001 * i.float()
        feat = torch.zeros(1, self.D, 128)
        feat[0, :n] = self.feat[:n]
        return SceneBatch(tlwh, conf, torch.zeros(1, self.D, dtype=torch.int32), feat,
                          torch.tensor([n], dtype=torch.int32))


@pytest.mark.parametrize("nd,hole", [(64, None), (65, None), (65, 32)])
def test_one_track_passing_64_and_65_gates(nd, hole):
    """The producer walks gate words 0 and 1 from the work record and stops at the detection count (64), or reads
    word 2 from the gate array (65; with a hole at detection 32, word 2 differs from word 1): oracle decisions, and
    costs bit for bit those of the exact pass."""
    hist, _ = _oracle_run(_tracker(1, 128, _Cluster.D, 8), OracleStreams(1, LABELS3, budget=8), _Cluster(nd, hole), 9,
                          costs_from=6)
    kw = dict(S=1, nobj=1, dmax=_Cluster.D, tmax=128, budget=8, frames=9, seed=0, feat_noise=0.0,
              scene=lambda: _Cluster(nd, hole))
    passing = nd - (hole is not None)
    checked, many = _compare("cluster_%d_%s" % (nd, hole), hist, _history("exact", **kw))
    assert many == passing and checked >= passing
    g = hist[6][1][0]
    row = g[np.argmax(_popcounts(g))]
    assert row[0] == 0xFFFFFFFF and row[1] == (0xFFFFFFFE if hole == 32 else 0xFFFFFFFF)
    assert row[2] == (1 if nd == 65 else 0)


def test_one_slot():
    """max_tracks = max_dets = 1 follows the oracle; with more detections than slots the overflow is flagged and
    check() raises."""
    bt = _tracker(1, 1, 1, 4)
    _oracle_run(bt, OracleStreams(1, LABELS3, budget=4), Scene(1, 1, 1, n_labels=3, seed=8, respawn_prob=0.0), 30)
    assert int(bt.v["state"][0, 0]) == 2
    bt = _tracker(1, 1, 4, 4)
    sc = Scene(1, 3, 4, n_labels=3, seed=9)
    for _ in range(3):
        bt.step(sc.step().to("cuda"))
    assert bt.status() & L.FLAG_TRACK_OVERFLOW and int(bt.v["n_tracks"][0]) <= 1
    with pytest.raises(RuntimeError, match="track capacity exceeded"):
        bt.check()


def _ring_scene(seed):
    return lambda: Scene(2, 8, 12, n_labels=3, seed=seed, respawn_prob=0.0, miss_prob=0.0)


@pytest.mark.parametrize("budget", [1, 15, 16, 17, 127, 128, 129, 256, 257, 1000])
def test_gallery_ring_budgets(budget):
    """Rings that wrap inside one page, at the 16-row page and 128-row block edges, and longer than one block: gallery
    rows are the oracle's samples[-budget:], and the half pre-pass's costs the exact pass's, bit for bit."""
    frames = budget + budget // 4 + 60
    hist, seen = _oracle_run(_tracker(2, 32, 12, budget), OracleStreams(2, LABELS3, budget=budget),
                             _ring_scene(61)(), frames, gallery_every=max(16, budget // 4))
    assert max(int(v["gal_len"].max()) for _, v in seen) == budget
    kw = dict(S=2, nobj=8, dmax=12, tmax=32, budget=budget, frames=frames, seed=61, feat_noise=0.02,
              scene=_ring_scene(61))
    checked, _ = _compare("ring_%d" % budget, hist, _history("exact", **kw))
    assert checked > 500


def test_budget_zero_keeps_every_sample():
    """nn_budget=0 keeps every sample (the reference's samples[-0:]): galleries past 16 and 128 rows equal to the
    oracle's, and ids, gate words and costs bit for bit those of budget=None."""
    frames = 150
    hist, seen = _oracle_run(_tracker(2, 32, 12, 0), OracleStreams(2, LABELS3, budget=0), _ring_scene(62)(), frames,
                             gallery_every=10)
    assert max(int(v["gal_len"].max()) for _, v in seen) > 128
    kw = dict(S=2, nobj=8, dmax=12, tmax=32, budget=None, frames=frames, seed=62, feat_noise=0.02,
              scene=_ring_scene(62))
    checked, _ = _compare("budget0", hist, _history("default", **kw))
    assert checked > 500


def test_128_labels_32_lines_two_chunks():
    """Exact vote ties decided by the name order (not the index order), the motorbike/bicycle rule at label indices
    126 and 127, counters [S, 32, 128, 4] of every line against an oracle counter of it, and their reduction over
    streams (16,384 counters) against the oracle's sum."""
    S = 4
    bt = _tracker(S, 64, 40, 8, labels=CP.LABELS128, lines=CP.LINES32, n_chunks=2)
    orc = OracleStreams(S, CP.LABELS128, budget=8)
    counters = CP.line_counters(S)
    sc = CP.LabelScene(S, 30, 40, seed=5)
    ties = rule = 0

    class _Counting:
        def step(self):
            nonlocal ties, rule
            t, r = CP.vote_corners(orc.trk)
            ties, rule = ties + t, rule + r
            return sc.step()

    _, seen = _oracle_run(bt, orc, _Counting(), 80, labels=CP.LABELS128, counters=counters, reduce=True)
    assert seen[-1][1]["counts"].shape == (S, 32, 128, 4) and bt.total_counts.shape == (32, 128, 4)
    assert ties > 20 and rule > 5 and int(seen[-1][1]["counts"].sum()) > 300, (ties, rule)
