"""Frame presence on the CPU: the fused tick of the host emulation (the kernel bodies compiled with a one-lane group)
leaves a stream without a frame untouched, and matches the oracle that simply does not step such a stream."""
import numpy as np
import pytest

from deepdish_b200 import _lib as L
from tests import presence as P
from tests.hostemu.tick import HostEmuTickTracker
from tests.parity import compare_stream, LABELS3


@pytest.fixture(scope="module")
def scene():
    return P.PresenceScene()


def _emu():
    return HostEmuTickTracker(L.make_config(P.S, 48, P.DMAX, P.BUDGET, LABELS3, max_age=P.MAX_AGE))


def _tick(emu, b, present):
    return emu.tick(b.tlwh.numpy(), b.conf.numpy(), b.label.numpy(), b.feat.numpy(), b.count.numpy(), present)


def test_presence_patterns_against_the_oracle(scene):
    assert scene.absent_after_del > 0          # a deletion counted at the line, then a tick without a frame
    emu = _emu()
    for f, (b, p, exp) in enumerate(zip(scene.frames, scene.present, scene.ids)):
        got = _tick(emu, b, p)
        P.check_tick_ids(got, exp, p, f)
        np.testing.assert_array_equal(emu.v["tick_present"], p.astype(np.int32))
    for s in range(P.S):
        compare_stream(scene.orc.trk[s], scene.orc.cnt[s], emu.v, s, LABELS3, gallery_rows=emu.gallery)
    np.testing.assert_array_equal(emu.v["counts"].sum(axis=0), scene.total_counts())
    assert int(emu.v["err"].sum()) == 0
    ctl = emu.v["pool_ctl"]
    assert int(ctl[0]) + int(emu.v["gal_np"].sum()) == int(ctl[1])


def _pages(emu):
    return lambda pid: (emu.pool_f32[pid * L.PAGE_F32_BYTES:(pid + 1) * L.PAGE_F32_BYTES],
                        emu.pool_f16[pid * L.PAGE_F16_BYTES:(pid + 1) * L.PAGE_F16_BYTES])


def test_absent_stream_state_is_bit_for_bit_unchanged(scene):
    """Across every tick in which a stream has no frame -- bursts far longer than max_age included -- each of its
    per-stream and per-slot arrays and the rows of its gallery pages stay exactly as they were, whatever the detection
    arrays hold for it (garbage, a count above max_dets)."""
    emu = _emu()
    rng = np.random.default_rng(0)
    checked = 0
    for f, (b, p) in enumerate(zip(scene.frames, scene.present)):
        before = {s: P.stream_state(emu.v, emu.cfg, s, _pages(emu)) for s in range(P.S) if not p[s]}
        tlwh, conf, label, feat, count = (b.tlwh.numpy().copy(), b.conf.numpy().copy(), b.label.numpy().copy(),
                                          b.feat.numpy().copy(), b.count.numpy().copy())
        for s in np.flatnonzero(~p):
            tlwh[s] = rng.normal(size=tlwh[s].shape) * 1e6
            feat[s] = np.nan
            label[s] = -5
            count[s] = P.DMAX + 7
        emu.tick(tlwh, conf, label, feat, count, p)
        for s, st in before.items():
            P.assert_same_state(st, P.stream_state(emu.v, emu.cfg, s, _pages(emu)), (f, s))
            assert (emu.det_track_id[s] == -1).all()
            checked += 1
    assert checked > 200 and int(emu.v["err"].sum()) == 0


def test_all_present_equals_no_presence(scene):
    """present all ones and present=None: the same ids every tick and the same blob, byte for byte."""
    a, b_ = _emu(), _emu()
    ones = np.ones(P.S, np.uint8)
    for f, b in enumerate(scene.frames[:60]):
        ia = _tick(a, b, ones).copy()
        ib = _tick(b_, b, None)
        np.testing.assert_array_equal(ia, ib)
    assert a.blob.tobytes() == b_.blob.tobytes()
    assert a.pool_f32.tobytes() == b_.pool_f32.tobytes()


def test_per_call_update_steps_every_stream_after_absent_ticks(scene):
    """The per-call update marks every stream present: after fused ticks with absences, predict / update / count-line
    step each stream again, as the reference's per-camera Tracker would."""
    emu = _emu()
    from tests.parity import OracleStreams
    orc = OracleStreams(P.S, LABELS3, budget=P.BUDGET, max_age=P.MAX_AGE)
    for f in range(40):
        b, p = scene.frames[f], scene.present[f]
        P.check_tick_ids(_tick(emu, b, p), P.oracle_tick(orc, b, p), p, f)
    for f in range(40, 70):
        b = scene.frames[f]
        exp = P.oracle_tick(orc, b, np.ones(P.S, bool))
        emu.predict()
        got = emu.update(b.tlwh.numpy(), b.conf.numpy(), b.label.numpy(), b.feat.numpy(), b.count.numpy())
        emu.countline()
        assert (emu.v["tick_present"] == 1).all()
        P.check_tick_ids(got, exp, np.ones(P.S, bool), f)
    for s in range(P.S):
        compare_stream(orc.trk[s], orc.cnt[s], emu.v, s, LABELS3)
