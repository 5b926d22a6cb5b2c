"""Scenes with several count lines per camera, shared by the CPU (host emulation) and GPU tests: the crossing scene of
tests/crossings.py (more than 32 live tracks crossing in one tick, frame-presence drops, an absence right after a
counted deletion) counted by one oracle LineCounter per line and stream, and the merged crossing records each stream's
lines produce (tracker.tracks order, each track's lines ascending, then the deletion records, lines ascending)."""
import numpy as np

from deepdish_b200.scene import Scene
from oracle import countline as oc
from tests import crossings as X
from tests import presence as P
from tests.parity import OracleStreams

MID = tuple(oc.default_line(640, 480).reshape(-1))      # the reference's default vertical mid-line
DIAG = X.LINE                                          # the frame's diagonal
HORIZ = (0.0, 240.0, 640.0, 240.0)
OUTSIDE = (1000.0, 0.0, 1000.0, 480.0)                 # right of the frame: never crossed
BASE = [MID, DIAG, HORIZ, DIAG, OUTSIDE]               # DIAG twice: a duplicate line counts identically


def per_stream_lines(n_streams=X.S):
    """f64 [S,6,4]: BASE plus a horizontal line of the stream's own height, rotated by the stream index so that every
    stream's set differs and the duplicates sit at different line indices."""
    out = []
    for s in range(n_streams):
        own = (0.0, 100.0 + 25.0 * s, 640.0, 100.0 + 25.0 * s)
        ls = BASE + [own]
        k = s % len(ls)
        out.append(ls[k:] + ls[:k])
    return np.array(out, np.float64)


def shared_lines():
    """f64 [5,4]: BASE, one set for every stream."""
    return np.array(BASE, np.float64)


def merged_records(counters, s, labels=X.LABELS):
    """The records stream s's lines produced in their last step, merged as the device lists them: int32 [n, 4]
    (stream, track_id, label, column + 4 line)."""
    live, dels = [], []
    for l, c in enumerate(counters):
        ev = c.events[-1]
        idx = c.index[-1]
        for k, (tid, lbl, d) in enumerate(ev):
            if d == "del":
                dels.append((l, (s, tid, labels.index(lbl), 3 + 4 * l)))
            else:
                live.append((idx[k], l, (s, tid, labels.index(lbl), (0 if d == 1 else 1) + 4 * l)))
    live.sort(key=lambda r: (r[0], r[1]))
    dels.sort(key=lambda r: r[0])
    out = [r[2] for r in live] + [r[1] for r in dels]
    return np.array(out, dtype=np.int32).reshape(-1, 4)


def fold(rec, n_streams, n_lines, n_labels):
    """Records -> [S, L, C, 4] counter increments."""
    out = np.zeros((n_streams, n_lines, n_labels, 4), np.int64)
    np.add.at(out, (rec[:, 0], rec[:, 3] >> 2, rec[:, 2], rec[:, 3] & 3), 1)
    out[..., 2] = out[..., 0] + out[..., 1]
    return out


class LinesScene:
    """The frames of tests/crossings.py's CrossingScene, with per-stream line sets lines f64 [S,L,4]: one tracker and
    L EventCounters per stream, stepped only for the streams that have a frame.  A stream whose tick counted a deletion
    on any line has no frame on the next tick."""

    def __init__(self, lines, seed=5, ticks=P.TICKS):
        self.lines = np.asarray(lines, np.float64)
        S, L = X.S, self.lines.shape[1]
        big = Scene(len(X.BIG), X.BIG_NOBJ, X.DMAX, n_labels=3, seed=seed, label_noise=0.5, clutter_mean=1.0,
                    respawn_prob=0.03)
        big.vel = big.vel * 2.0
        small = Scene(S - len(X.BIG), X.NOBJ, X.DMAX, n_labels=3, seed=seed + 1, respawn_prob=0.02, clutter_mean=0.5)
        small.vel = small.vel * 2.0
        self.orc = OracleStreams(S, X.LABELS, budget=P.BUDGET, max_age=P.MAX_AGE)
        self.cnt = [[X.EventCounter(self.lines[s, l].reshape(2, 2), X.LABELS) for l in range(L)] for s in range(S)]
        masks = P.base_masks()
        masks[:, list(X.BIG)] = masks[:, [0, 9]]
        self.frames, self.present, self.ids, self.rec, self.counts_at = [], [], [], [], []
        self.absent_after_del = 0
        force = np.zeros(S, bool)
        for f in range(ticks):
            b = X._concat(big.step(), small.step(), X.BIG)
            p = masks[f] & ~force
            self.absent_after_del += int(force.sum())
            before = np.array([sum(c.counts(X.LABELS)[:, 3].sum() for c in cs) for cs in self.cnt])
            ids = []
            for s in range(S):
                if not p[s]:
                    ids.append(None)
                    continue
                t = self.orc.trk[s]
                ids.append(_oracle_update(t, b, s, X.LABELS))
                for c in self.cnt[s]:
                    c.step(t)
            after = np.array([sum(c.counts(X.LABELS)[:, 3].sum() for c in cs) for cs in self.cnt])
            self.rec.append([merged_records(self.cnt[s], s) if p[s] else np.zeros((0, 4), np.int32) for s in range(S)])
            force = after > before
            force[0] = False
            self.frames.append(b)
            self.present.append(p)
            self.ids.append(ids)
            self.counts_at.append(self.counts())

    def tick_records(self, f):
        """All streams' records of tick f in stream order: int32 [n, 4]."""
        return np.concatenate(self.rec[f])

    def counts(self):
        """The oracle's counters now (counts_at[f]: after tick f): int64 [S, L, C, 4]."""
        return np.array([[c.counts(X.LABELS) for c in cs] for cs in self.cnt])

    def cases(self):
        """How often each case the lines must get right occurs in the scene: crossings past the first warp round of one
        tick, a track crossing distinct lines in one tick, a deletion counted on several lines, an absence right after
        a counted deletion."""
        c = dict(multi_round=0, distinct_lines_one_track=0, del_several_lines=0, absent_after_del=self.absent_after_del)
        for s in range(X.S):
            k = 0
            for f in range(len(self.frames)):
                if not self.present[f][s]:
                    continue
                r = self.rec[f][s]
                live = r[(r[:, 3] & 3) != 3]
                idx = [i for cnt in self.cnt[s] for i in cnt.index[k]]
                c["multi_round"] += int(bool(idx) and min(idx) < 32 <= max(idx))
                if len(live):
                    c["distinct_lines_one_track"] += int(np.unique(live[:, 1], return_counts=True)[1].max() >= 3)
                c["del_several_lines"] += int(((r[:, 3] & 3) == 3).sum() >= 2)
                k += 1
        return c


def _oracle_update(t, batch, s, labels):
    """predict + update of one oracle tracker; -> the stream's det -> track id list."""
    from oracle import deepsort as od
    tlwh, conf, lab, feat = batch.stream(s)
    dets = [od.Det(tlwh[i], labels[lab[i]], conf[i], feat[i]) for i in range(len(conf))]
    t.trace = {}
    t.predict()
    t.update(dets)
    ids = [-1] * len(dets)
    for tid, d in t.trace["match_ids"]:
        ids[d] = tid
    nxt = t._next_id - len(t.trace["unmatched_detections"])
    for k, d in enumerate(t.trace["unmatched_detections"]):
        ids[d] = nxt + k
    return ids
