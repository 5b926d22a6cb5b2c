"""Matching edge scenarios shared by the CPU (host emulation) and GPU tests: scripted streams whose every matching
decision sits on an edge of the rules -- costs exactly at a threshold or one ulp either side of it, raw costs in the
clip band (thr, thr + 1e-5), all-clip cascade levels, ties, the last cascade level, the CPython set order that feeds
the IoU stage -- run next to the oracle (real scipy, real sets) and compared bit for bit.

Exact costs by construction.  An identity feature is a positive multiple of a basis vector e_k (k < K_IDENT); a mixed
feature is p e_k + q e_u for a Pythagorean triple (p, q, r) and a private component u >= K_IDENT that nothing else in
the stream uses.  Normalised on either side they are e_k and (f32(p/r), f32(q/r)).  A gallery row and a detection then
share at most one non-zero component (the exactness guard asserts it for every pair the cascade could compare), so the
f32 cost 1 - f32(p/r) is the same whatever the summation order: numpy's BLAS, the fmaf chain of the exact pass and the
half pre-pass with exact re-check of the gallery kernel.  Boxes are integer with a dyadic aspect ratio and never move:
every Kalman update has a zero innovation, so track means are those boxes exactly and IoU costs are computed from the
same doubles on both sides.  Gating is never near its edge: a detection sits on a track's box (d^2 = 0) or far away.

State edits (applied before a tick, identically to the oracle's Trk objects and to the implementation's SoA state):
("tsu", i, v) sets time_since_update of track index i; ("confirm", i) turns the tentative track i into a confirmed one
(the device gallery already holds every feature of its updates; the oracle's Trk.features move to metric.samples)."""
import numpy as np
import torch
from scipy.optimize import linear_sum_assignment

from deepdish_b200 import _lib as L
from deepdish_b200.scene import SceneBatch
from oracle import deepsort as od, countline as oc
from tests.parity import compare_stream, LABELS3

K_IDENT = 32              # identity components 0..31; private components of mixed features K_IDENT..127
BUDGET = 100
TRIPLES = ((4, 3, 5), (3, 4, 5), (12, 5, 13), (5, 12, 13), (15, 8, 17), (8, 15, 17), (24, 7, 25), (7, 24, 25),
           (21, 20, 29), (20, 21, 29))
COUNTERS = ("at_thr", "clip_band", "all_clip", "transposed", "noncontig", "set_not_ascending", "iou_at_thr",
            "set_boundary", "lanes_33")


def basis(k, scale=1.0):
    f = np.zeros(128, np.float32)
    f[k] = scale
    return f


def cos_cost(tri):
    """f32 cosine cost of e_k against the mixed feature (p e_k + q e_u) / r, as a double."""
    p, q, r = tri
    return float(np.float32(1) - np.float32(p) / np.float32(r))


def cell(i, dx=0):
    """Integer tlwh box of grid cell i (12 x 4 cells, 30 x 40 boxes: aspect 3/4, far apart for the gate)."""
    return (10.0 + (i % 12) * 52 + dx, 10.0 + (i // 12) * 115, 30.0, 40.0)


class Scn:
    """One scripted stream.  knobs: tracker-wide settings (max_age, max_cosine_distance, max_iou_distance); streams
    with the same knobs and track capacity run in one tracker."""

    def __init__(self, name, max_age=30, cos=0.2, iou=0.7, max_tracks=64, pin_tracks=False, port=True):
        self.name = name
        self.knobs = (int(max_age), float(cos), float(iou))
        self.max_tracks, self.pin_tracks, self.port = max_tracks, pin_tracks, port
        self.ticks = []            # [(dets [(tlwh, feat)], edits)]
        self.expect = {}           # tick -> {det index: track id, or 0 for "a new track"}
        self.overflow_at = None    # tick at which the track table overflows (the stream ends there)
        self.priv = K_IDENT

    def mix(self, k, tri):
        """p e_k + q e_u with the stream's next private component u."""
        assert k < K_IDENT and self.priv < 128, self.name
        f = np.zeros(128, np.float32)
        f[k], f[self.priv] = tri[0], tri[1]
        self.priv += 1
        return f

    def tick(self, dets, edits=(), expect=None):
        self.ticks.append((list(dets), list(edits)))
        if expect:
            self.expect[len(self.ticks) - 1] = dict(expect)
        return len(self.ticks) - 1

    def confirm(self, objs):
        """Three ticks of the same detections [(cell box, feature or feature list per tick)]: the tracks are confirmed
        at the third, with ids 1.. in detection order."""
        for f in range(3):
            self.tick([(b, ft[f] if isinstance(ft, list) else ft) for b, ft in objs])


# --------------------------------------------------------------------------------------------------- the oracle side
class OracleStream:
    """One od.Trkr (real scipy and real sets, or the pure-Python port of both) and its count-line, plus what the
    comparisons and coverage counters read from each update."""

    def __init__(self, knobs, port=False):
        max_age, cos, iou = knobs
        self.thr_cos, self.thr_iou = cos, iou
        self.lsaps = []
        solver = od.lsap_port if port else linear_sum_assignment

        def lsap(c):
            self.lsaps.append(np.array(c, copy=True))
            return solver(c)
        kw = dict(set_order=od.cpython_set_difference_order) if port else {}
        self.trk = od.Trkr(od.Metric("cosine", cos, BUDGET), iou, max_age, 3, lsap=lsap, **kw)
        self.cnt = oc.LineCounter(oc.default_line(640, 480), LABELS3)

    def edit(self, e):
        t = self.trk.tracks[e[1]]
        if e[0] == "tsu":
            assert int(e[2]) >= t.time_since_update       # only raised: a track that missed more ticks
            t.time_since_update = int(e[2])
        elif e[0] == "confirm":
            assert t.state == od.TENTATIVE
            t.state = od.CONFIRMED
            self.trk.metric.samples[t.track_id] = list(t.features)[-BUDGET:]
            t.features = []
        else:
            raise ValueError(e)

    def guard(self, dets):
        """Every (gallery row, detection) pair the cascade could compare shares at most one non-zero component."""
        if not dets:
            return
        fz = np.stack([d.feature != 0 for d in dets]).astype(np.int32)
        for t in self.trk.tracks:
            if t.is_confirmed():
                g = np.asarray(self.trk.metric.samples[t.track_id]) != 0
                assert (g.astype(np.int32) @ fz.T).max() <= 1, t.track_id

    def step(self, dets_spec, cnt):
        dets = [od.Det(np.asarray(b, float), LABELS3[0], 0.9, f) for b, f in dets_spec]
        t = self.trk
        confirmed = [i for i, x in enumerate(t.tracks) if x.is_confirmed()]
        nxt0 = t._next_id
        t.trace, self.lsaps = {}, []
        t.predict()
        self.guard(dets)
        t.update(dets)
        self.cnt.step(t)
        ids = [-1] * len(dets)
        for tid, d in t.trace["match_ids"]:
            ids[d] = tid
        nxt = t._next_id - len(t.trace["unmatched_detections"])
        for k, d in enumerate(t.trace["unmatched_detections"]):
            ids[d] = nxt + k
        # coverage, from the trace
        gated = t.trace.get("gated_costs", [])
        for _, _, c in gated:
            cnt["at_thr"] += int((c == self.thr_cos).sum())
            cnt["clip_band"] += int(((c > self.thr_cos) & (c < self.thr_cos + 1e-5)).sum())
            cnt["all_clip"] += int(c.shape[1] >= 2 and bool((c > self.thr_cos).all()))
        cnt["transposed"] += sum(int(c.shape[0] > c.shape[1]) for c in self.lsaps)
        for c in self.lsaps[len(gated):]:
            cnt["iou_at_thr"] += int((c == self.thr_iou).sum())
        cnt["noncontig"] += int(confirmed != list(range(len(confirmed))))
        matched = [k for k, _ in t.trace["matches_a"]]
        un = list(set(confirmed) - set(matched))          # the expression of linear_assignment.py:140
        cnt["set_not_ascending"] += int(un != sorted(un))
        nc = len(confirmed)
        cnt["set_boundary"] += int(nc >= 40 and abs(len(matched) - (nc >> 2)) <= 1)
        cnt["lanes_33"] += int(len(dets) >= 33 and len(t.tracks) >= 33)
        return ids, nxt0


def compare_gate_costs(o_trk, pre, post, s):
    """Gate bits and cost entries of every pair the oracle's cascade compared, bit for bit (the exactness guard makes
    every cost exact).  pre: n_tracks / order / track_id before the update; post: gate / cost after it."""
    n = int(pre["n_tracks"][s])
    slot_of = {int(pre["track_id"][s, sl]): int(sl) for sl in pre["order"][s, :n]}
    checked = 0
    for tids, dets, cost in o_trk.trace.get("gated_costs", []):
        for r, tid in enumerate(tids):
            sl = slot_of[tid]
            for c, d in enumerate(dets):
                bit = (int(post["gate"][s, sl, d >> 5]) >> (d & 31)) & 1
                if cost[r, c] >= od.INFTY_COST:
                    assert bit == 0, (tid, d)
                else:
                    assert bit == 1, (tid, d)
                    got = float(post["cost"][s, sl, d])
                    assert got == cost[r, c], (tid, d, got, cost[r, c])
                    checked += 1
    return checked


# ---------------------------------------------------------------------------------------------------- running groups
def groups(scns, max_tracks=None):
    """Scenarios that can share one tracker: same knobs and track capacity (max_tracks overrides every capacity that
    the scenario does not pin)."""
    out = {}
    for sc in scns:
        t = sc.max_tracks if (sc.pin_tracks or max_tracks is None) else max_tracks
        out.setdefault((sc.knobs, t), []).append(sc)
    return [(k[0], k[1], v) for k, v in out.items()]


def make_batch(scns, f, D):
    S = len(scns)
    tlwh = np.zeros((S, D, 4))
    conf = np.zeros((S, D), np.float32)
    label = np.zeros((S, D), np.int32)
    feat = np.zeros((S, D, 128), np.float32)
    count = np.zeros(S, np.int32)
    for s, sc in enumerate(scns):
        dets = sc.ticks[f][0] if f < len(sc.ticks) else []
        count[s] = len(dets)
        for i, (b, ft) in enumerate(dets):
            tlwh[s, i], feat[s, i], conf[s, i] = b, ft, 0.9
    return SceneBatch(*(torch.from_numpy(a) for a in (tlwh, conf, label, feat, count)))


LIFECYCLE = ("n_tracks", "order", "track_id", "state", "hits", "age", "tsu", "deleted", "n_deleted", "next_id", "mean",
             "cov", "gal_len", "counts", "gate", "cost", "err")


def run_group(knobs, T, scns, impl_factory, port=False, cnt=None):
    """Run scenarios (one stream each) through an implementation and the oracle, comparing every tick.

    impl_factory(S, T, D, max_age, max_cos, max_iou) -> object with tick(SceneBatch on the host) -> ids numpy [S, D],
    view(names) -> {name: numpy copy}, set(name, s, slot, value) (a state edit), gallery(s, slot) -> numpy [len, 128].
    Returns the number of cost entries compared bit for bit."""
    cnt = cnt if cnt is not None else dict.fromkeys(COUNTERS, 0)
    S = len(scns)
    n_ticks = max(len(sc.ticks) for sc in scns)
    D = max(1, max(len(d) for sc in scns for d, _ in sc.ticks))
    impl = impl_factory(S, T, D, *knobs)
    orc = [OracleStream(knobs, port=port) for _ in scns]
    done = [False] * S
    checked = 0
    for f in range(n_ticks):
        pre = impl.view(("n_tracks", "order", "track_id"))
        for s, sc in enumerate(scns):
            for e in (sc.ticks[f][1] if f < len(sc.ticks) else []):
                orc[s].edit(e)
                slot = int(pre["order"][s, e[1]])
                if e[0] == "tsu":
                    impl.set("tsu", s, slot, int(e[2]))
                else:
                    impl.set("state", s, slot, od.CONFIRMED)
        exp = [orc[s].step(sc.ticks[f][0] if f < len(sc.ticks) else [], cnt) for s, sc in enumerate(scns)]
        got = impl.tick(make_batch(scns, f, D))
        post = impl.view(LIFECYCLE)
        last = f == n_ticks - 1
        for s, sc in enumerate(scns):
            if done[s]:
                continue
            ids, nxt0 = exp[s]
            what = (sc.name, f, s)
            for d, want in sc.expect.get(f, {}).items():        # the scenario reaches the edge it is written for
                assert (ids[d] >= nxt0) if want == 0 else (ids[d] == want), (what, d, ids[d], want)
            row = [int(x) for x in got[s, :len(ids)]]
            if sc.overflow_at == f:
                # the first free slots take the first unmatched detections; the rest get no track
                lost = [d for d in range(len(ids)) if row[d] == -1]
                assert lost and all(row[d] in (ids[d], -1) for d in range(len(ids))), (what, row, ids)
                assert int(post["err"][s]) == L.FLAG_TRACK_OVERFLOW, what
                done[s] = True
                continue
            assert row == ids, (what, row, ids)
            assert int(post["err"][s]) == 0, (what, int(post["err"][s]))
            compare_stream(orc[s].trk, orc[s].cnt, post, s, LABELS3,
                           gallery_rows=impl.gallery if last or f == len(sc.ticks) - 1 else None)
            checked += compare_gate_costs(orc[s].trk, pre, post, s)
    return checked


def run_all(scns, impl_factory, port=False, max_tracks=None):
    cnt = dict.fromkeys(COUNTERS, 0)
    checked = 0
    for knobs, T, grp in groups(scns, max_tracks):
        checked += run_group(knobs, T, grp, impl_factory, port=port, cnt=cnt)
    return checked, cnt


# ------------------------------------------------------------------------------------------------ hand-written streams
def s_cos_threshold(thr, label):
    """A confirmed track A (gallery e0, gate-passing detections 0..3 and 35: its pair sits at gate-passing rank 4 >=
    DD_CVAL, in the second gate word) and B (gallery e1, its pair at rank 0), one missed tick each so that the IoU stage
    cannot rescue them; both pairs cost exactly c = 1 - f32(4/5).  They match iff c <= thr."""
    sc = Scn("cos_thr_" + label, cos=thr)
    sc.confirm([(cell(0), basis(0)), (cell(1), basis(1))])
    c = cos_cost((4, 3, 5))
    dets = [(cell(0), basis(10 + i)) for i in range(4)] + [(cell(1), sc.mix(1, (4, 3, 5)))]
    dets += [(cell(2 + i), basis(20)) for i in range(30)] + [(cell(0), sc.mix(0, (4, 3, 5)))]
    dets += [(cell(32 + i), basis(21)) for i in range(4)]
    m = c <= thr
    sc.tick(dets, [("tsu", 0, 1), ("tsu", 1, 1)], expect={35: 1 if m else 0, 4: 2 if m else 0})
    return sc


def s_clip_band():
    """Raw costs in (thr, thr + 1e-5) are clipped to the value the gated-out pairs get: the assignment solver ties
    them, and the tie (not the raw cost) decides which detection the track's row takes and so the order of new ids."""
    c = cos_cost((4, 3, 5))
    sc = Scn("clip_band", cos=c - 5e-6)
    sc.confirm([(cell(0), basis(0)), (cell(1), basis(1))])
    # track 0: [gated out, clip band, gated out, gated out]; track 1: one plain clipped pair (cost 0.4), the rest gated
    sc.tick([(cell(5), basis(7)), (cell(0), sc.mix(0, (4, 3, 5))), (cell(6), basis(8)),
             (cell(1), sc.mix(1, (3, 4, 5)))], [("tsu", 0, 1), ("tsu", 1, 1)])
    # square level: track 1 matches below the threshold, track 0's only gate-passing pair is in the clip band
    sc.tick([(cell(1), sc.mix(1, (12, 5, 13))), (cell(0), sc.mix(0, (4, 3, 5)))], [("tsu", 0, 2), ("tsu", 1, 2)])
    return sc


def s_clip_magnitude():
    """2 x 2 level: r1c1 = 0, r1c2 = x, r2c1 = y (exact mixed costs), r2c2 clipped; thr = x + y - 1.5e-5 puts 0 + clip
    just below x + y, so the diagonal wins only if the clip is exactly thr + 1e-5."""
    x, y = cos_cost((4, 3, 5)), cos_cost((12, 5, 13))
    sc = Scn("clip_magnitude", cos=x + y - 1.5e-5)
    # A (id 1) gallery {e2, mix(3, 4-3-5), e2}; B (id 2) gallery {mix(2, 12-5-13) x 3}; both on cell 0
    sc.confirm([(cell(0), [basis(2), sc.mix(3, (4, 3, 5)), basis(2)]),
                (cell(0), [sc.mix(2, (12, 5, 13)), sc.mix(2, (12, 5, 13)), sc.mix(2, (12, 5, 13))])])
    sc.tick([(cell(0), basis(2)), (cell(0), basis(3))], [("tsu", 0, 1), ("tsu", 1, 1)], expect={0: 1, 1: 0})
    return sc


def s_all_clip(shape):
    """A level where every pair is clipped or gated, then a deeper level whose track Z ties on every detection: the
    detection Z takes is the first of the rewritten unmatched list (unassigned columns first, then the rejected ones
    in row order).  wide: 1 x 3; square: a 1 x 3 level reorders the columns a 3 x 3 level then sees; tall: 3 x 2."""
    sc = Scn("all_clip_" + shape)
    n0, n1, nc, first = {"wide": (0, 1, 3, 1), "square": (1, 3, 3, 1), "tall": (0, 3, 2, 0)}[shape]
    sc.confirm([(cell(0), basis(5 + i)) for i in range(n0 + n1)] + [(cell(0), basis(9))])
    edits = [("tsu", n0 + i, 1) for i in range(n1)] + [("tsu", n0 + n1, 2)]
    sc.tick([(cell(0), basis(9)) for _ in range(nc)], edits, expect={first: n0 + n1 + 1})
    return sc


def s_tied():
    """Identical galleries x identical detection features: transposed, wide and square levels, one level and across
    levels."""
    sc = Scn("tied")
    sc.confirm([(cell(0), basis(4))] * 3)
    sc.tick([(cell(0), basis(4))] * 2, [("tsu", i, 1) for i in range(3)])           # 3 x 2, one level
    sc.tick([(cell(0), basis(4))] * 2, [("tsu", 0, 2), ("tsu", 1, 1)])              # level 1, then 2 x 1 at level 2
    sc.tick([(cell(0), basis(4))] * 4)                                              # 2 x 4, then 1 x 2 at level 3
    sc.tick([(cell(0), basis(4))] * 3)                                              # 3 x 3
    return sc


def s_depth(max_age):
    """Track A at tsu = max_age (the last cascade level: it can match) and B at max_age + 1 (never matched, deleted);
    with max_age 70 also tracks on the sparse levels 1, 5 and 30.  Raised time_since_update stands for missed ticks;
    a track with tsu > 1 gets no IoU rescue."""
    sc = Scn("depth_%d" % max_age, max_age=max_age)
    n = 5 if max_age == 70 else 2
    sc.confirm([(cell(i), basis(i)) for i in range(n)])
    edits, expect = [("tsu", 1, max_age)], {1: 0}
    if max_age >= 1:
        edits.append(("tsu", 0, max_age - 1))
        expect[0] = 1
    else:
        expect = {}                # no cascade at all: the IoU stage rescues both tracks (tsu == 1)
    if n == 5:
        edits += [("tsu", 3, 4), ("tsu", 4, 29)]
        expect.update({2: 3, 3: 4, 4: 5})
    sc.tick([(cell(i), basis(i)) for i in range(n)], edits, expect=expect)
    sc.tick([(cell(i), basis(i)) for i in range(n)])
    return sc


def s_depth_limit():
    """max_age = 32766: tsu 32766 is the last level, 32767 (the largest time_since_update the matching stores) is
    deleted."""
    sc = Scn("depth_limit", max_age=32766)
    sc.confirm([(cell(0), basis(0)), (cell(1), basis(1))])
    sc.tick([(cell(0), basis(0)), (cell(1), basis(1))], [("tsu", 0, 32765), ("tsu", 1, 32766)], expect={0: 1, 1: 0})
    return sc


def s_set_order(nmatched):
    """44 confirmed tracks; tracks 3 and 8 share a box, survive the cascade with tsu == 1 and tie on one detection's
    IoU: the first of them in the CPython set order of the unmatched confirmed tracks takes it.  nmatched around
    (44 >> 2) = 11 straddles the copy-and-difference fast path; 40 leaves 4 survivors whose set order is not
    ascending ([8, 33, 3, 38])."""
    sc = Scn("set_order_%d" % nmatched)
    cells = [3 if i == 8 else i for i in range(44)]
    sc.confirm([(cell(cells[i]), basis(i % 30)) for i in range(44)])
    if nmatched == 40:
        match = [i for i in range(44) if i not in (3, 8, 33, 38)]
    else:
        match = list(range(10, 10 + nmatched))
    dets = [(cell(3), basis(31))] + [(cell(cells[i]), basis(i % 30)) for i in match]
    sc.tick(dets, expect={0: 9 if nmatched == 40 else 4})
    return sc


def s_noncontig():
    """A later tentative track (index 8) is confirmed by a host edit while earlier ones are tentative: the confirmed
    list [1, 8] takes the general set-order path, whose order [8, 1] hands the IoU tie on their shared box to 8."""
    sc = Scn("noncontig", port=False)
    cells = [1 if i == 8 else i for i in range(10)]
    objs = [(cell(cells[i]), basis(i)) for i in range(10)]
    sc.tick(objs)
    sc.tick(objs)
    dets = [(cell(1), basis(31))] + [(cell(cells[i]), basis(i)) for i in range(10) if i not in (1, 8)]
    sc.tick(dets, [("confirm", 1), ("confirm", 8)], expect={0: 9})
    sc.tick(dets)
    return sc


def s_iou_threshold(thr, label):
    """A one-tick-old tentative track on an exact box and a detection shifted by 10 px: IoU cost exactly 0.5.  Two
    tentative tracks sharing a box and one detection on it: a transposed IoU problem with a tie."""
    sc = Scn("iou_thr_" + label, iou=thr)
    sc.tick([(cell(0), basis(0)), (cell(1), basis(1)), (cell(1), basis(2))])
    sc.tick([(cell(0, dx=10), basis(0)), (cell(1), basis(1))], expect={0: 1 if 0.5 <= thr else 0, 1: 2})
    return sc


def s_iou_clip_magnitude():
    """IoU 2 x 2: track A's box is the disjoint union of track B's box and detection d1, so r1c2 = r2c1 = 0.5 and
    r2c2 = 1 = r1c2 + r2c1 (the IoU distance is a metric: this is its triangle inequality with equality), r1c1 = 0.
    thr = 1 - 1.5e-5 clips r2c2 only, and the diagonal 0 + clip beats 0.5 + 0.5 only if the clip is thr + 1e-5."""
    sc = Scn("iou_clip_magnitude", iou=1 - 1.5e-5)
    x, y = cell(0)[:2]
    sc.tick([((x, y, 30.0, 40.0), basis(0)), ((x, y, 30.0, 20.0), basis(1))])
    sc.tick([((x, y, 30.0, 40.0), basis(0)), ((x, y + 20, 30.0, 20.0), basis(1))], expect={0: 1, 1: 0})
    return sc


def s_counts(n):
    """n objects (31 / 32 / 33: the lane boundaries), ticks with n - 1 and n detections and an empty tick."""
    sc = Scn("counts_%d" % n)
    sc.confirm([(cell(i), basis(i % 30)) for i in range(n)])
    sc.tick([(cell(i), basis(i % 30)) for i in range(1, n)])
    sc.tick([])
    sc.tick([(cell(i), basis(i % 30)) for i in range(n)])
    return sc


def s_first_tick():
    """Detections with no tracks, then tracks with no detections."""
    sc = Scn("first_tick")
    sc.tick([(cell(i), basis(i)) for i in range(3)])
    sc.tick([])
    sc.tick([(cell(i), basis(i)) for i in range(3)])
    return sc


def s_overflow():
    """8 slots: 4 tentative tracks, 4 others replace them (nnew == nfree), then 5 new detections with 4 free slots."""
    sc = Scn("overflow", max_tracks=8, pin_tracks=True)
    sc.tick([(cell(i), basis(i)) for i in range(4)])
    sc.tick([(cell(4 + i), basis(4 + i)) for i in range(4)], expect={0: 0, 3: 0})
    sc.tick([(cell(8 + i), basis(8 + i)) for i in range(5)])
    sc.overflow_at = 2
    return sc


def hand_scenarios():
    c = cos_cost((4, 3, 5))
    out = [s_cos_threshold(np.nextafter(c, 0), "below"), s_cos_threshold(c, "at"),
           s_cos_threshold(np.nextafter(c, 1), "above"), s_clip_band(), s_clip_magnitude()]
    out += [s_all_clip(k) for k in ("wide", "square", "tall")]
    out += [s_tied()] + [s_depth(a) for a in (0, 1, 3, 70)] + [s_depth_limit()]
    out += [s_set_order(m) for m in (10, 11, 12, 40)] + [s_noncontig()]
    out += [s_iou_threshold(0.5, "at"), s_iou_threshold(np.nextafter(0.5, 0), "below"), s_iou_clip_magnitude()]
    out += [s_counts(n) for n in (31, 32, 33)] + [s_first_tick(), s_overflow()]
    return out


# ----------------------------------------------------------------------------------------------------------- fuzzing
def thresholds():
    """Exact costs of single mixed pairs, their f64 neighbours and points 5e-6 below them (costs in the clip band)."""
    out = []
    for tri in TRIPLES:
        c = cos_cost(tri)
        out += [c, np.nextafter(c, 0), np.nextafter(c, 1), c - 5e-6]
    return out


def fuzz_scenarios(seed, n_streams=4, ticks=30):
    """Clustered objects on shared boxes, random misses, identity / mixed / foreign features, clutter; one threshold
    drawn from the exact costs and their neighbours and one max_age per seed (tracker-wide)."""
    rng = np.random.default_rng(seed)
    thr = float(rng.choice(thresholds()))
    max_age = int(rng.choice([1, 2, 3, 5]))
    out = []
    for s in range(n_streams):
        sc = Scn("fuzz%d.%d" % (seed, s), max_age=max_age, cos=thr)
        n_cl = int(rng.integers(2, 4))
        cl_cells = rng.choice(40, n_cl, replace=False)
        objs = [(int(rng.integers(n_cl)), int(rng.integers(12))) for _ in range(int(rng.integers(3, 9)))]
        for f in range(ticks):
            dets = []
            for c, k in objs:
                if rng.random() < 0.25:
                    continue
                u = rng.random()
                if u < 0.3 and sc.priv < 128:
                    ft = sc.mix(k, TRIPLES[int(rng.integers(len(TRIPLES)))])
                elif u < 0.4:
                    ft = basis(int(rng.integers(12)))
                else:
                    ft = basis(k, float(rng.integers(1, 4)))
                dets.append((cell(int(cl_cells[c])), ft))
            if rng.random() < 0.3:
                dets.append((cell(int(cl_cells[int(rng.integers(n_cl))])), basis(int(rng.integers(12, 20)))))
            order = rng.permutation(len(dets))
            sc.tick([dets[i] for i in order])
        out.append(sc)
    return out
