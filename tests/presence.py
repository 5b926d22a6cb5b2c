"""Frame-presence scenes shared by the CPU (host emulation) and GPU tests of ticks in which some streams have no
frame: a fixed mix of presence patterns, the oracle stepped only for the streams that have a frame (the reference
calls nothing on the tracker of a camera that delivers no frame), and the per-stream state of one stream."""
import numpy as np

from deepdish_b200 import _lib
from deepdish_b200.scene import Scene
from tests.parity import OracleStreams, LABELS3
from oracle import deepsort as od

S, NOBJ, DMAX, MAX_AGE, BUDGET, TICKS = 12, 10, 16, 8, 20, 160
ALL_ABSENT_TICKS = (30, 31, 77, 120)
# per-tick scratch and the presence word itself: exempt from "an absent stream is left bit for bit as it was"
SCRATCH = {"gate", "cost", "det_xyah", "det_featn", "det_feath", "det_slot", "det_kind", "cdesc", "work", "work_ctl",
           "work_rec", "tick_args", "timeline", "tick_present"}


def base_masks(seed=3):
    """[TICKS, S] bool: stream 0 always present; stream 1 absent until tick 50; streams 2-5 drop ~30 % of their
    frames at random; streams 6-8 have bursts of absence far longer than MAX_AGE; streams 9-11 drop ~10 %; no stream
    has a frame on ALL_ABSENT_TICKS."""
    rng = np.random.default_rng(seed)
    m = np.ones((TICKS, S), bool)
    m[:50, 1] = False
    m[:, 2:6] = rng.random((TICKS, 4)) >= 0.3
    for s, (a, n) in zip((6, 7, 8), ((20, 3 * MAX_AGE), (60, MAX_AGE + 3), (90, 5 * MAX_AGE))):
        m[a:a + n, s] = False
    m[:, 9:] = rng.random((TICKS, S - 9)) >= 0.1
    m[list(ALL_ABSENT_TICKS), :] = False
    return m


def oracle_tick(orc, batch, present):
    """OracleStreams.step for the present streams only; -> per-stream id lists (None for an absent stream)."""
    out = []
    for s, (t, c) in enumerate(zip(orc.trk, orc.cnt)):
        if not present[s]:
            out.append(None)
            continue
        tlwh, conf, lab, feat = batch.stream(s)
        dets = [od.Det(tlwh[i], orc.labels[lab[i]], conf[i], feat[i]) for i in range(len(conf))]
        t.trace = {}
        t.predict()
        t.update(dets)
        c.step(t)
        ids = [-1] * len(dets)
        for tid, d in t.trace["match_ids"]:
            ids[d] = tid
        nxt = t._next_id - len(t.trace["unmatched_detections"])
        for k, d in enumerate(t.trace["unmatched_detections"]):
            ids[d] = nxt + k
        out.append(ids)
    return out


class PresenceScene:
    """Frames, the presence actually used per tick and the oracle's ids, computed once.  Besides base_masks: a stream
    (other than stream 0) whose tick counted a deleted track at the line (the `del` counter rose) has no frame on the
    next tick -- that tick must not count the same deletion again."""

    def __init__(self, seed=17):
        # little clutter: a frame whose last deleted track is a tentative one counts no deletion (deepdish.py:1041-1044)
        sc = Scene(S, NOBJ, DMAX, n_labels=3, seed=seed, respawn_prob=0.02, clutter_mean=0.3)
        self.orc = OracleStreams(S, LABELS3, budget=BUDGET, max_age=MAX_AGE)
        masks = base_masks()
        self.frames, self.present, self.ids = [], [], []
        self.absent_after_del = 0
        force = np.zeros(S, bool)
        for f in range(TICKS):
            b = sc.step()
            p = masks[f] & ~force
            self.absent_after_del += int(force.sum())
            before = np.array([c.counts(LABELS3)[:, 3].sum() for c in self.orc.cnt])
            self.ids.append(oracle_tick(self.orc, b, p))
            after = np.array([c.counts(LABELS3)[:, 3].sum() for c in self.orc.cnt])
            force = after > before
            force[0] = False
            self.frames.append(b)
            self.present.append(p)

    def total_counts(self):
        return sum(c.counts(LABELS3) for c in self.orc.cnt)


def check_tick_ids(got, exp, present, f):
    """got i32 [S,Dmax] (numpy): present rows match the oracle, absent rows are -1 throughout."""
    for s in range(S):
        if present[s]:
            assert list(got[s, :len(exp[s])]) == exp[s], (f, s)
        else:
            assert (got[s] == -1).all(), (f, s)


def stream_state(v, cfg, s, pages):
    """Every per-stream and per-slot array of stream s (scratch excluded) from the typed views v (name -> numpy array),
    and the f32 and half rows of the gallery pages its slots hold: pages(pid) -> (f32 bytes, half bytes)."""
    out = {}
    for name, (dt, shape) in _lib.field_specs(cfg).items():
        if name in SCRATCH or shape[0] != cfg.n_streams or name == "work":
            continue
        out[name] = np.array(v[name][s], copy=True)
    for slot in range(cfg.max_tracks):
        for k in range(int(v["gal_np"][s, slot])):
            pid = int(v["ptab"][s, slot, k])
            f32, f16 = pages(pid)
            out["page%d.%d.f32" % (slot, k)] = np.array(f32, copy=True)
            out["page%d.%d.f16" % (slot, k)] = np.array(f16, copy=True)
    return out


def assert_same_state(a, b, what):
    assert a.keys() == b.keys(), what
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), (what, k)
