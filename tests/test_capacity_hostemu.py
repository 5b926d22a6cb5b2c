"""Capacity corners on the CPU.  The layout check: every (max_tracks, max_dets) whose matching step fits the 227 KB of
shared memory a block can have is accepted and the next larger max_dets is rejected, by the product's layout query and
the host emulation's alike, and BatchedTracker refuses a shape that does not fit before it touches the GPU.  Then the
kernel bodies (compiled with a one-lane group) against the oracle, tick by tick, at the corners: a crowd of about a
thousand objects at 1024 slots x 992 detections, gallery rings across the 16-row page and 128-row block edges and
nn_budget=0, 128 labels on 32 count lines, and one slot per stream."""
import ctypes

import numpy as np
import pytest

from deepdish_b200 import _lib as L
from deepdish_b200.scene import Scene
from tests import capacity as CP
from tests.hostemu import driver as hd
from tests.parity import OracleStreams, compare_stream, compare_costs, LABELS3


def _smem(T, D):
    f = hd.emu().ddh_match_smem_bytes
    f.argtypes, f.restype = [ctypes.c_int, ctypes.c_int], ctypes.c_longlong
    return f(T, D)


@pytest.fixture(scope="module")
def queries():
    from deepdish_b200 import build
    build.build()            # no-op when up to date; nvcc cross-compiles without a GPU
    return {"product": L.lib().dd_tracker_layout_query, "hostemu": hd.emu().ddh_tracker_layout_query}


def _rc(query, T, D):
    cfg = L.make_config(1, T, D, None, LABELS3)
    return query(ctypes.byref(cfg), ctypes.byref(L.TrackerLayout()))


def test_layout_boundary_corners(queries):
    for name, q in queries.items():
        for T, D in ((1024, 992), (960, 1024), (991, 1024), (1, 1), (1, 1024), (1024, 1), (1024, 988)):
            assert _rc(q, T, D) == L.DD_OK, (name, T, D)
        for T, D in ((1024, 993), (1024, 1024), (992, 1024), (1025, 1), (1, 1025)):
            assert _rc(q, T, D) == L.DD_ERR_INVALID, (name, T, D)


@pytest.mark.parametrize("T", [1, 64, 256, 512, 900, 960, 961, 976, 991, 992, 1000, 1008, 1016, 1023, 1024])
def test_layout_boundary_follows_the_matching_step(queries, T):
    """The largest accepted max_dets of each max_tracks is the largest whose matching step fits the limit."""
    sizes = [_smem(T, D) for D in range(1, 1025)]
    assert all(a <= b for a, b in zip(sizes, sizes[1:]))          # the layout only grows with max_dets
    fit = [D for D, b in zip(range(1, 1025), sizes) if b <= L.SMEM_OPTIN_BYTES]
    dmax = fit[-1]
    assert (dmax == 1024) == (T <= 991)
    for name, q in queries.items():
        assert _rc(q, T, dmax) == L.DD_OK, (name, T, dmax)
        if dmax < 1024:
            assert _rc(q, T, dmax + 1) == L.DD_ERR_INVALID, (name, T, dmax + 1)
    if dmax < 1024:
        with pytest.raises(ValueError, match="largest max_dets that fits max_tracks=%d is %d\\b" % (T, dmax)):
            L.check_shape(L.lib(), T, dmax + 1)
    L.check_shape(L.lib(), T, dmax)


def test_batched_tracker_rejects_a_shape_the_matching_step_cannot_run(queries):
    from deepdish_b200.batched import BatchedTracker
    with pytest.raises(ValueError, match=r"232448 bytes \(227 KB\).*max_tracks=1024 is 992"):
        BatchedTracker(1, LABELS3, max_tracks=1024, max_dets=1024)
    with pytest.raises(ValueError, match="max_tracks=1024 is 992"):
        BatchedTracker(1, LABELS3, max_tracks=1024, max_dets=993)


def _run(emu, orc, frames_or_batches, S, labels=LABELS3, counters=None, costs_from=None, gallery_every=0):
    """Tick the host emulation and the oracle on the same batches; compare ids, track table, lifecycle, counters and
    (every gallery_every ticks) gallery rows.  Yields (tick, batch) after each comparison."""
    for f, b in enumerate(frames_or_batches):
        pre = {k: emu.v[k].copy() for k in ("n_tracks", "order", "track_id")}
        ids = orc.step(b)
        got = emu.tick(b.tlwh.numpy(), b.conf.numpy(), b.label.numpy(), b.feat.numpy(), b.count.numpy())
        if counters is not None:
            for s in range(S):
                for c in counters[s]:
                    c.step(orc.trk[s])
        for s in range(S):
            n = int(b.count[s])
            assert list(got[s, :n]) == ids[s], (f, s)
            rows = emu.gallery if gallery_every and f % gallery_every == gallery_every - 1 else None
            compare_stream(orc.trk[s], orc.cnt[s] if counters is None else None, emu.v, s, labels, gallery_rows=rows)
            if costs_from is not None and f >= costs_from:
                compare_costs(orc.trk[s], pre, emu.v, s)
        if counters is not None:
            np.testing.assert_array_equal(emu.v["counts"], CP.line_counts(counters), err_msg="counts tick %d" % f)
        yield f, b


def _scene_batches(sc, frames):
    for _ in range(frames):
        yield sc.step()


def test_crowd_1024_slots_992_detections_host_emulation():
    """31 gate words per track, tracks with more than DD_CVAL gate-passing detections, the solver at n = 1024 and set
    tables of 4096 slots; gate bits and costs of the last ticks against the oracle."""
    cfg = L.make_config(1, 1024, 992, 4, LABELS3, max_age=30)
    emu = hd.HostEmuTracker(cfg)
    orc = OracleStreams(1, LABELS3, budget=4, max_age=30)
    live = dets = many = high_word = 0
    for f, b in _run(emu, orc, _scene_batches(CP.crowd(950, 992, seed=3), 12), 1, costs_from=9, gallery_every=6):
        live, dets = max(live, int(emu.v["n_tracks"][0])), max(dets, int(b.count[0]))
        bits = np.unpackbits(emu.v["gate"][0].view(np.uint8), bitorder="little").reshape(1024, -1)
        many = max(many, int(bits.sum(axis=1).max()))
        high_word = max(high_word, int(np.nonzero(bits.any(axis=0))[0].max()) >> 5 if bits.any() else 0)
    assert int(emu.v["err"][0]) == 0
    assert emu.v["gate"].shape[-1] == 31 and live >= 700 and dets >= 900 and many > 4 and high_word >= 27, \
        (live, dets, many, high_word)


@pytest.mark.parametrize("budget", [0, 1, 15, 16, 17, 127, 128, 129])
def test_gallery_rings_host_emulation(budget):
    """Rings that wrap inside one page, at the 16-row page edge and at the 128-row block edge, and nn_budget=0, which
    keeps every sample as nn_budget=None does (the oracle's samples[-0:])."""
    frames = 150 if budget in (0, 127, 128, 129) else 60
    # the C config's budget 0 is the unbounded gallery; the oracle runs the reference's nn_budget as given
    cfg = L.make_config(2, 32, 12, budget or None, LABELS3, max_age=30, page_cap=(frames + 15) // 16 + 1)
    emu = hd.HostEmuTracker(cfg)
    orc = OracleStreams(2, LABELS3, budget=budget, max_age=30)
    longest = 0
    for f, b in _run(emu, orc, _scene_batches(Scene(2, 8, 12, n_labels=3, seed=31, respawn_prob=0.0), frames), 2,
                     gallery_every=10):
        longest = max(longest, int(emu.v["gal_len"].max()))
    assert int(emu.v["err"].sum()) == 0
    assert longest == budget if budget else longest > 128, longest


def test_128_labels_32_lines_host_emulation():
    """Vote ties between labels seen equally often, decided by the name order, which is not the index order, and the
    motorbike/bicycle rule at label indices 126 and 127; every line's counters against an oracle counter of it."""
    S = 2
    cfg = L.make_config(S, 64, 40, 8, CP.LABELS128, max_age=30, n_lines=32)
    emu = hd.HostEmuTracker(cfg, line=CP.LINES32)
    orc = OracleStreams(S, CP.LABELS128, budget=8, max_age=30)
    counters = CP.line_counters(S)
    sc = CP.LabelScene(S, 30, 40, seed=5)
    ties = rule = 0
    for f, b in _run(emu, orc, (sc.step() for _ in range(80)), S, labels=CP.LABELS128, counters=counters):
        t, r = CP.vote_corners(orc.trk)
        ties, rule = ties + t, rule + r
    assert emu.v["counts"].shape == (S, 32, 128, 4)
    assert ties > 20 and rule > 5, (ties, rule)
    assert int(emu.v["counts"].sum()) > 200 and int(emu.v["err"].sum()) == 0


def test_one_slot_host_emulation():
    """max_tracks = max_dets = 1: one object is tracked as the oracle tracks it; with several detections the track
    table overflows and the stream's flag says so."""
    emu = hd.HostEmuTracker(L.make_config(1, 1, 1, 4, LABELS3, max_age=30))
    orc = OracleStreams(1, LABELS3, budget=4, max_age=30)
    for f, b in _run(emu, orc, _scene_batches(Scene(1, 1, 1, n_labels=3, seed=8, respawn_prob=0.0), 30), 1):
        pass
    assert int(emu.v["err"][0]) == 0 and int(emu.v["state"][0, 0]) == 2
    emu = hd.HostEmuTracker(L.make_config(1, 1, 4, 4, LABELS3, max_age=30))
    sc = Scene(1, 3, 4, n_labels=3, seed=9)
    for _ in range(3):
        b = sc.step()
        emu.tick(b.tlwh.numpy(), b.conf.numpy(), b.label.numpy(), b.feat.numpy(), b.count.numpy())
    assert int(emu.v["err"][0]) & L.FLAG_TRACK_OVERFLOW and int(emu.v["n_tracks"][0]) <= 1
