"""Crossing-record scenes shared by the CPU (host emulation) and GPU tests of the per-tick count-line crossings: an
oracle counter that also records the deletion record, and a frame-presence scene whose streams produce the cases the
records must get right (more than 32 live tracks crossing in several lane rounds of one tick, deletions with and
without live crossings, the motorbike/bicycle label rule at a crossing, an absence right after a counted deletion)."""
import numpy as np
import torch

from deepdish_b200.scene import Scene, SceneBatch
from oracle import countline as oc
from tests import presence as P
from tests.parity import OracleStreams

LABELS = ["person", "bicycle", "motorbike"]
S, DMAX, T, TICKS = P.S, 48, 96, P.TICKS
BIG = (0, 5)                 # streams with 40 objects (the others have 10)
BIG_NOBJ, NOBJ = 40, 10
LINE = (0.0, 0.0, 640.0, 480.0)    # the frame's diagonal: more crossings per tick than the default mid-line


class EventCounter(oc.LineCounter):
    """LineCounter whose per-step event list ends with the deletion record: (track_id, label name, "del") for the
    last deleted track when its del count survives (deepdish.py:1041-1044).  Also notes, per step, the index in
    tracker.tracks of each crossing track and whether the motorbike/bicycle rule decided a crossing's label."""

    def __init__(self, line, labels):
        super().__init__(line, labels)
        self.index = []           # per step: tracker.tracks index of each live crossing
        self.rule = []            # per step: number of crossings whose label the motorbike/bicycle rule decided

    def _check_deleted(self, trk):
        out = super()._check_deleted(trk)
        self._last_del = (trk.track_id, out)
        return out

    def step(self, tracker):
        self._last_del = None
        super().step(tracker)
        ids = [t.track_id for t in tracker.tracks]
        by_id = dict(zip(ids, tracker.tracks))
        ev = self.events[-1]
        self.index.append([ids.index(tid) for tid, _, _ in ev])
        self.rule.append(sum(_rule_decides(by_id[tid]) for tid, _, _ in ev))
        if self._last_del is not None and self._last_del[1]:
            (lbl,) = self._last_del[1].keys()
            ev.append((self._last_del[0], lbl, "del"))


def _rule_decides(trk):
    """track.py:175-183 applies: the two best labels are motorbike then bicycle."""
    if not trk.labels:
        return False
    stats = [(lbl, len(s), np.average(s)) for lbl, s in trk.dist.items()]
    alphas = np.array([a for _, _, a in stats])
    cnt = np.array([c for _, c, _ in stats])
    ranked = list(reversed(sorted(zip((alphas + cnt) / (cnt.sum() + alphas.sum()), [l for l, _, _ in stats]))))
    return len(ranked) > 1 and ranked[0][1] == "motorbike" and ranked[1][1] == "bicycle"


def records(counter, s, labels=LABELS):
    """The oracle's crossing records of its last step for stream s: int32 [n, 4] (stream, track_id, label, column)."""
    out = [(s, tid, labels.index(lbl), 3 if d == "del" else (0 if d == 1 else 1)) for tid, lbl, d in counter.events[-1]]
    return np.array(out, dtype=np.int32).reshape(-1, 4)


def fold(rec, n_streams, n_labels):
    """Records -> [S, C, 4] counter increments."""
    out = np.zeros((n_streams, n_labels, 4), np.int64)
    np.add.at(out, (rec[:, 0], rec[:, 2], rec[:, 3]), 1)
    out[:, :, 2] = out[:, :, 0] + out[:, :, 1]
    return out


def _concat(a, b, idx_a):
    """Stream-wise merge of two SceneBatches: streams idx_a from a, the rest from b, in stream order."""
    n = a.count.shape[0] + b.count.shape[0]
    ia, ib = 0, 0
    order = []
    for s in range(n):
        if s in idx_a:
            order.append((0, ia)); ia += 1
        else:
            order.append((1, ib)); ib += 1
    return SceneBatch(*(torch.stack([(getattr(a, k) if w == 0 else getattr(b, k))[i] for w, i in order])
                        for k in SceneBatch.__slots__))


class CrossingScene:
    """Frames, presence per tick and the oracle's crossing records per tick and stream, computed once.  The two big
    streams carry 40 objects moving twice as fast as the default scene and labels that flip half of the time
    (so motorbike tracks collect bicycle votes); presence follows tests/presence.py (base_masks, and an absence right
    after a tick that counted a deletion)."""

    def __init__(self, seed=5):
        big = Scene(len(BIG), BIG_NOBJ, DMAX, n_labels=3, seed=seed, label_noise=0.5, clutter_mean=1.0,
                    respawn_prob=0.03)
        big.vel = big.vel * 2.0
        small = Scene(S - len(BIG), NOBJ, DMAX, n_labels=3, seed=seed + 1, respawn_prob=0.02, clutter_mean=0.5)
        small.vel = small.vel * 2.0
        self.orc = OracleStreams(S, LABELS, budget=P.BUDGET, max_age=P.MAX_AGE, line=LINE)
        self.orc.cnt = [EventCounter(c.line, LABELS) for c in self.orc.cnt]
        masks = P.base_masks()
        masks[:, list(BIG)] = masks[:, [0, 9]]          # one big stream always present, one dropping ~10 %
        self.frames, self.present, self.ids, self.rec = [], [], [], []
        self.absent_after_del = 0
        force = np.zeros(S, bool)
        for f in range(TICKS):
            b = _concat(big.step(), small.step(), BIG)
            p = masks[f] & ~force
            self.absent_after_del += int(force.sum())
            before = np.array([c.counts(LABELS)[:, 3].sum() for c in self.orc.cnt])
            self.ids.append(P.oracle_tick(self.orc, b, p))
            after = np.array([c.counts(LABELS)[:, 3].sum() for c in self.orc.cnt])
            self.rec.append([records(self.orc.cnt[s], s) if p[s] else np.zeros((0, 4), np.int32) for s in range(S)])
            force = after > before
            force[0] = False
            self.frames.append(b)
            self.present.append(p)

    def tick_records(self, f):
        """All streams' records of tick f in stream order: int32 [n, 4]."""
        return np.concatenate(self.rec[f])

    def cases(self):
        """How often each case the records must get right occurs in the scene."""
        c = dict(multi_round=0, del_alone=0, del_with_live=0, rule=0, absent_after_del=self.absent_after_del)
        for s, cnt in enumerate(self.orc.cnt):
            k = 0
            for f in range(TICKS):
                if not self.present[f][s]:
                    continue
                idx, r = cnt.index[k], self.rec[f][s]
                c["multi_round"] += int(bool(idx) and min(idx) < 32 <= max(idx))
                has_del = bool(len(r)) and r[-1, 3] == 3
                c["del_alone"] += int(has_del and len(r) == 1)
                c["del_with_live"] += int(has_del and len(r) > 1)
                c["rule"] += cnt.rule[k]
                k += 1
        return c
