"""GPU parity: the CUDA BatchedTracker (through the C ABI) against the oracle, tick by tick.

Bit-exact: track ids, states, hits/age/time_since_update, deleted lists, det->track assignment,
pos/neg/int/del counters.  Tolerance: Kalman mean / covariance rtol 1e-4 (north_star)."""
import numpy as np
import pytest
import torch

from deepdish_b200.scene import Scene
from tests.parity import OracleStreams, compare_stream, compare_costs, LABELS3

pytestmark = pytest.mark.gpu


def _run(S, nobj, dmax, tmax, frames, max_age, seed, budget=100, check_every=1, per_call=False, **kw):
    """per_call: every tick issued call by call (predict, update, countline) instead of through the engine."""
    from deepdish_b200.batched import BatchedTracker
    bt = BatchedTracker(S, LABELS3, max_tracks=tmax, max_dets=dmax, budget=budget, max_age=max_age, **kw)
    orc = OracleStreams(S, LABELS3, budget=budget, max_age=max_age)
    sc = Scene(S, nobj, dmax, n_labels=3, seed=seed)
    for f in range(frames):
        b = sc.step()
        ids = orc.step(b)
        d = b.to("cuda")
        if per_call:
            bt.predict()
            got = bt.update(d.tlwh, d.conf, d.label, d.feat, d.count).cpu().numpy()
            bt.countline()
        else:
            got = bt.step(d).cpu().numpy()
        for s in range(S):
            n = int(b.count[s])
            assert list(got[s, :n]) == ids[s], (f, s)
        if f % check_every == 0 or f == frames - 1:
            bt.check()
            v = bt.host_view()
            rows = (lambda s, slot: bt.gallery(s, slot).cpu().numpy()) if (f % 25 == 24 or f == frames - 1) else None
            for s in range(S):
                compare_stream(orc.trk[s], orc.cnt[s], v, s, LABELS3, gallery_rows=rows)
    bt.check()
    ctl = [c.v["pool_ctl"].cpu().numpy() for c in bt.chunks]       # every page is free or in exactly one slot's table
    assert sum(int(c[0]) for c in ctl) + int(bt.v["gal_np"].sum()) == sum(int(c[1]) for c in ctl)
    return bt, orc


def test_c1_single_stream_300_frames():
    """BASELINE config 0: 1 stream, 300 frames, <=20 dets, budget 100."""
    bt, orc = _run(1, 20, 24, 64, 300, 30, seed=11)
    assert orc.trk[0]._next_id > 100          # clutter created and deleted many tentative tracks


def test_streams_20_objects_max_age_60():
    _run(8, 20, 24, 64, 150, 60, seed=3, check_every=5)


def test_c3_like_50_objects():
    """BASELINE config 2 shape (50 dets/frame, budget 100) on a sample of streams."""
    bt, orc = _run(16, 50, 64, 128, 80, 60, seed=5, check_every=10)
    tot = bt.reduce_counts().cpu().numpy()
    exp = sum(c.counts(LABELS3) for c in orc.cnt)
    np.testing.assert_array_equal(tot, exp)
    assert tot[:, 2].sum() > 0


def test_small_budget_and_short_age():
    """Ring wrap-around (budget 5) and early deletion (max_age 3)."""
    _run(4, 12, 16, 48, 120, 3, seed=9, budget=5, check_every=4)


def test_unbounded_galleries_and_pool_growth_multi_stream():
    """nn_budget=None on several streams and two chunks, starting from a pool and page tables that are far too small:
    pool segments are attached and the page tables re-laid out while the run goes on -- between engine ticks from the
    engine's pool polls, and in a second run by update() from the exact counters --; parity with the oracle
    throughout."""
    for per_call in (False, True):
        bt, orc = _run(6, 10, 14, 40, 260, 20, seed=21, budget=None, check_every=13, n_chunks=2,
                       pool_pages=64, seg_pages=64, page_cap=2, per_call=per_call)
        assert all(len(c.segs) > 1 for c in bt.chunks) and all(c.v["ptab"].shape[2] >= 16 for c in bt.chunks), per_call
        assert max(len(g) for t in orc.trk for g in t.metric.samples.values()) > 200


def test_pool_exhaustion_is_reported_not_silent():
    from deepdish_b200.batched import BatchedTracker
    bt = BatchedTracker(2, LABELS3, max_tracks=32, max_dets=12, budget=40, max_age=30, pool_pages=8, seg_pages=8)
    bt._poll_pool = False                          # no growth: the 8-page pool must run dry
    sc = Scene(2, 10, 12, n_labels=3, seed=5)
    from deepdish_b200 import _lib
    for _ in range(30):
        bt.step(sc.step().to("cuda"))
    # which appends are dropped once the pool is dry depends on the order the CTAs reach it, so what follows (ids, even a
    # track overflow) is not deterministic -- the flag and the error are
    assert bt.status() & _lib.FLAG_POOL_EXHAUSTED
    with pytest.raises(RuntimeError, match="pool exhausted"):
        bt.check()


def test_bad_label_is_flagged_and_not_counted():
    from deepdish_b200.batched import BatchedTracker
    bt = BatchedTracker(1, LABELS3, max_tracks=16, max_dets=4, budget=10)
    b = Scene(1, 3, 4, n_labels=3, seed=2).step().to("cuda")
    b.label[0, 0] = 7
    bt.step(b)
    assert int(bt.v["lab_cnt"].sum()) == int(b.count[0]) - 1
    with pytest.raises(ValueError, match="label"):
        bt.check()


def test_empty_frames_and_capacity_flags():
    from deepdish_b200.batched import BatchedTracker
    S, D, T = 2, 8, 8
    bt = BatchedTracker(S, ["person"], max_tracks=T, max_dets=D, budget=4)
    z = dict(tlwh=torch.zeros(S, D, 4, dtype=torch.float64, device="cuda"),
             conf=torch.zeros(S, D, device="cuda"), label=torch.zeros(S, D, dtype=torch.int32, device="cuda"),
             feat=torch.ones(S, D, 128, device="cuda"), count=torch.zeros(S, dtype=torch.int32, device="cuda"))
    bt.predict(); bt.update(**z); bt.countline()
    assert bt.status() == 0 and int(bt.v["n_tracks"].sum()) == 0
    # 8 detections in stream 0, twice -> 8 tentative + 8 deleted slots cannot fit T=8 the 2nd time
    z["tlwh"][0, :, 0] = torch.arange(D, dtype=torch.float64, device="cuda") * 70
    z["tlwh"][0, :, 2:] = 10
    z["count"][0] = D
    bt.predict(); bt.update(**z)
    assert bt.status() == 0 and int(bt.v["n_tracks"][0]) == 8
    z["tlwh"][0, :, 1] = 300                     # nothing matches -> 8 deleted + 8 new > T
    bt.predict(); bt.update(**z)
    with pytest.raises(RuntimeError):
        bt.check()
    with pytest.raises(ValueError):
        bt.update(z["tlwh"].float(), z["conf"], z["label"], z["feat"], z["count"])


def test_gated_cost_matrices_match_oracle():
    """Distance matrices: every (track, detection) the reference would not gate out has the same
    min-cosine cost within 1e-4 relative (+2e-6 absolute: the reference's own BLAS summation noise)."""
    from deepdish_b200.batched import BatchedTracker
    S = 4
    bt = BatchedTracker(S, LABELS3, max_tracks=128, max_dets=64, budget=100, max_age=60)
    orc = OracleStreams(S, LABELS3, budget=100, max_age=60)
    sc = Scene(S, 50, 64, n_labels=3, seed=21)
    checked = 0
    for f in range(50):
        b = sc.step()
        pre = bt.host_view(["n_tracks", "order", "track_id"])
        orc.step(b)
        bt.step(b.to("cuda"))
        if f >= 5 and f % 3 == 0:
            post = bt.host_view(["gate", "cost"])
            for s in range(S):
                checked += compare_costs(orc.trk[s], pre, post, s)
    assert checked > 1000


def test_stream_chunks_engine_host_and_per_call_ticks():
    """n_chunks > 1, switching tick by tick between the engine on device batches (enqueue-only steps), the engine on
    ragged pinned host batches and the per-call path (predict, update, countline, reduce_counts): the same ids / state /
    counters as the oracle, and the chunked count reduction equals the sum over streams."""
    from deepdish_b200.batched import BatchedTracker
    S = 7
    bt = BatchedTracker(S, LABELS3, max_tracks=64, max_dets=24, budget=30, max_age=30, n_chunks=3)
    orc = OracleStreams(S, LABELS3, budget=30, max_age=30)
    sc = Scene(S, 16, 24, n_labels=3, seed=31)
    ids_host = torch.empty((S, 24), dtype=torch.int32).pin_memory()
    for f in range(60):
        b = sc.step()
        ids = orc.step(b)
        if f % 3 == 0:
            bt.step(b.to("cuda"), join=False, reduce=True)
            bt.join()
            got = bt.det_track_id.cpu().numpy()
        elif f % 3 == 1:              # ragged pinned host batch: one H2D copy per chunk + unpack kernel
            bt.step_host_packed(bt.pack_host(b), ids_host)
            bt.join()
            torch.cuda.synchronize()
            got = ids_host.numpy().copy()
        else:
            d = b.to("cuda")
            bt.predict()
            got = bt.update(d.tlwh, d.conf, d.label, d.feat, d.count).cpu().numpy()
            bt.countline()
            bt.reduce_counts()
        for s in range(S):
            n = int(b.count[s])
            assert list(got[s, :n]) == ids[s], (f, s)
        exp = sum(c.counts(LABELS3) for c in orc.cnt)
        np.testing.assert_array_equal(bt.total_counts.cpu().numpy(), exp)
    v = bt.host_view()
    for s in range(S):
        compare_stream(orc.trk[s], orc.cnt[s], v, s, LABELS3)
    bt.check()


def test_c4_like_crowd_200_dets():
    """BASELINE config 3 shape (crowd: ~200 dets/frame, up to 256+ tracks, budget 100) on a few streams:
    multi-word gate masks, transposed and non-transposed LSAPs up to ~200 x 200, CTA-sized shared memory."""
    bt, orc = _run(3, 190, 224, 384, 45, 60, seed=17, check_every=5)
    assert max(len(t.tracks) for t in orc.trk) > 200


def test_label_vote_motorbike_bicycle_rule_and_per_stream_lines():
    """track.py:154-188: Dirichlet vote with the motorbike / bicycle special case (30 % label noise makes
    the vote matter), counters keyed by the voted label; one count-line per stream (vertical, horizontal,
    diagonal) -- counters bit-exact."""
    from deepdish_b200.batched import BatchedTracker
    labels = ["motorbike", "bicycle", "person"]
    S = 6
    lines = np.array([[320, 0, 320, 480], [0, 240, 640, 240], [0, 0, 640, 480], [100, 0, 500, 480],
                      [640, 100, 0, 300], [320, 480, 320, 0]], dtype=np.float64)
    bt = BatchedTracker(S, labels, max_tracks=64, max_dets=24, budget=40, max_age=25, line=lines, n_chunks=2)
    orc = OracleStreams(S, labels, budget=40, max_age=25, line=lines)
    sc = Scene(S, 16, 24, n_labels=3, seed=41, label_noise=0.3)
    for f in range(140):
        b = sc.step()
        ids = orc.step(b)
        got = bt.step(b.to("cuda")).cpu().numpy()
        for s in range(S):
            assert list(got[s, :int(b.count[s])]) == ids[s], (f, s)
        if f % 10 == 9:
            v = bt.host_view()
            for s in range(S):
                compare_stream(orc.trk[s], orc.cnt[s], v, s, labels)
    tot = bt.reduce_counts().cpu().numpy()
    assert tot[:, 2].sum() > 20 and (tot[:, 2] > 0).sum() >= 2         # several labels were counted
    bt.check()


@pytest.mark.parametrize("n_init,max_age", [(1, 1), (2, 4), (5, 12)])
def test_n_init_and_max_age_variants(n_init, max_age):
    from deepdish_b200.batched import BatchedTracker
    from oracle import deepsort as od, countline as oc
    S = 3
    bt = BatchedTracker(S, LABELS3, max_tracks=96, max_dets=24, budget=10, max_age=max_age, n_init=n_init)
    trk = [od.Trkr(od.Metric("cosine", 0.2, 10), 0.7, max_age, n_init) for _ in range(S)]
    cnt = [oc.LineCounter(oc.default_line(640, 480), LABELS3) for _ in range(S)]
    sc = Scene(S, 14, 24, n_labels=3, seed=50 + n_init, miss_prob=0.2)
    for f in range(70):
        b = sc.step()
        if 30 <= f < 30 + max_age + 3:
            b.count[1] = 0                         # stream 1 goes blind: every track ages out, ids restart later
        got = bt.step(b.to("cuda")).cpu().numpy()
        for s in range(S):
            tlwh, conf, lab, feat = b.stream(s)
            dets = [od.Det(tlwh[i], LABELS3[lab[i]], conf[i], feat[i]) for i in range(len(conf))]
            trk[s].trace = {}
            trk[s].predict(); trk[s].update(dets); cnt[s].step(trk[s])
            exp = [-1] * len(dets)
            for tid, d in trk[s].trace["match_ids"]:
                exp[d] = tid
            nxt = trk[s]._next_id - len(trk[s].trace["unmatched_detections"])
            for k, d in enumerate(trk[s].trace["unmatched_detections"]):
                exp[d] = nxt + k
            assert list(got[s, :len(dets)]) == exp, (f, s)
        if f % 7 == 0:
            v = bt.host_view()
            for s in range(S):
                compare_stream(trk[s], cnt[s], v, s, LABELS3)
    bt.check()


def test_checkpoint_resume_is_bit_identical():
    from deepdish_b200.batched import BatchedTracker
    S = 5
    kw = dict(max_tracks=64, max_dets=24, budget=20, max_age=20, n_chunks=2)
    a = BatchedTracker(S, LABELS3, **kw)
    sc = Scene(S, 14, 24, n_labels=3, seed=77)
    frames = [sc.step().to("cuda") for _ in range(45)]
    for b in frames[:25]:
        a.step(b)
    sd = a.state_dict()
    ids_a = [a.step(b).clone() for b in frames[25:]]
    b2 = BatchedTracker(S, LABELS3, **kw)
    b2.load_state_dict(sd)
    for k, b in enumerate(frames[25:]):
        assert torch.equal(b2.step(b), ids_a[k])
    va, vb = a.host_view(), b2.host_view()
    for name in ("n_tracks", "order", "track_id", "state", "mean", "cov", "counts", "next_id"):
        np.testing.assert_array_equal(va[name], vb[name])
    assert torch.equal(a.reduce_counts(), b2.reduce_counts())


@pytest.mark.parametrize("match_warps", [4, 8])
@pytest.mark.parametrize("shape", ["crowd", "c3", "small_budget"])
def test_cta_matching_kernel(shape, match_warps):
    """k_match_cta (4 warps per stream, picked automatically for crowded scenes; 8 on request) forced on for several
    shapes: the same oracle parity as the one-warp kernel."""
    if shape == "crowd":
        bt, orc = _run(3, 190, 224, 384, 40, 60, seed=18, check_every=5, match_warps=match_warps)
        assert max(len(t.tracks) for t in orc.trk) > 200
    elif shape == "c3":
        _run(12, 50, 64, 128, 70, 60, seed=6, check_every=10, match_warps=match_warps)
    else:
        _run(4, 12, 16, 48, 100, 3, seed=10, budget=5, check_every=4, match_warps=match_warps)


def test_unpack_detections_entry():
    """dd_unpack_detections (ragged blob -> padded arrays) on its own: equals the padded batch it was packed from."""
    import ctypes
    from deepdish_b200 import _lib
    from deepdish_b200.batched import BatchedTracker
    S, D = 9, 24
    bt = BatchedTracker(S, LABELS3, max_tracks=32, max_dets=D, budget=10)
    b = Scene(S, 16, D, n_labels=3, seed=5).step()
    (blob, total, offs), = bt.pack_host(b)
    dev = blob[:total].cuda()
    t = torch.zeros((S, D, 4), dtype=torch.float64, device="cuda"); cf = torch.zeros((S, D), device="cuda")
    lb = torch.zeros((S, D), dtype=torch.int32, device="cuda"); ft = torch.zeros((S, D, 128), device="cuda")
    ct = torch.zeros((S,), dtype=torch.int32, device="cuda")
    _lib.check(bt.lib.dd_unpack_detections(dev.data_ptr(), S, D, *offs, t.data_ptr(), cf.data_ptr(), lb.data_ptr(),
                                           ft.data_ptr(), ct.data_ptr(), ctypes.c_void_p(0)), "dd_unpack_detections")
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ct.cpu().numpy(), b.count.numpy())
    valid = (torch.arange(D)[None, :] < b.count[:, None]).numpy()
    for got, exp in ((t, b.tlwh), (cf, b.conf), (lb, b.label), (ft, b.feat)):
        np.testing.assert_array_equal(got.cpu().numpy()[valid], exp.numpy()[valid])


def test_engine_counts_launches_and_survives_mode_switches():
    """The native tick engine (dd_engine_*): one captured graph per chunk and tick.  Its launch counter is what
    bench.py reports as gpu_launches; ticks issued through it and call by call from Python (update / countline) can be
    interleaved on the same tracker and still equal a tracker that only ever used one path."""
    from deepdish_b200.batched import BatchedTracker
    S = 6
    a = BatchedTracker(S, LABELS3, max_tracks=48, max_dets=16, budget=20, max_age=30, n_chunks=2)
    b = BatchedTracker(S, LABELS3, max_tracks=48, max_dets=16, budget=20, max_age=30, n_chunks=1)
    sc = Scene(S, 10, 16, n_labels=3, seed=5)
    for f in range(24):
        fr = sc.step().to("cuda")
        if f % 4 == 3:               # the per-call path: predict + update + countline
            a.predict()
            ia = a.update(fr.tlwh, fr.conf, fr.label, fr.feat, fr.count).cpu().numpy().copy()
            a.countline()
        else:
            ia = a.step(fr, join=True, reduce=True).cpu().numpy().copy()
        ib = b.step(fr, join=True, reduce=True).cpu().numpy().copy()
        np.testing.assert_array_equal(ia, ib, err_msg="tick %d" % f)
    ticks, launches, blocked = a.engine_stats()
    assert ticks == 18 and launches == 18 * (2 * 8 + 1) and blocked >= 0.0
    assert b.engine_stats()[1] == 24 * (8 + 1)
    assert torch.equal(a.reduce_counts(), b.reduce_counts())
    va, vb = a.host_view(["track_id", "state", "hits", "mean"]), b.host_view(["track_id", "state", "hits", "mean"])
    for k in va:
        np.testing.assert_array_equal(va[k], vb[k], err_msg=k)
    a.check()
    b.check()


def test_engine_plain_launches_equal_graph_replay():
    """dd_engine_set_graphs(0): the engine launches the tick's kernels plainly instead of replaying captured graphs --
    same kernels, same order, same streams, so ids, counters and state are identical tick by tick."""
    from deepdish_b200.batched import BatchedTracker
    S = 6
    kw = dict(max_tracks=48, max_dets=16, budget=20, max_age=30, n_chunks=2)
    a = BatchedTracker(S, LABELS3, engine_graphs=False, **kw)
    b = BatchedTracker(S, LABELS3, **kw)
    c = BatchedTracker(S, LABELS3, engine_graphs=False, gallery_turns=False, **kw)
    sc = Scene(S, 10, 16, n_labels=3, seed=11)
    for f in range(30):
        fr = sc.step().to("cuda")
        ia = a.step(fr, join=True, reduce=True).cpu().numpy().copy()
        ib = b.step(fr, join=True, reduce=True).cpu().numpy().copy()
        ic = c.step(fr, join=True, reduce=True).cpu().numpy().copy()
        np.testing.assert_array_equal(ia, ib, err_msg="tick %d" % f)
        np.testing.assert_array_equal(ic, ib, err_msg="tick %d (no turns)" % f)
    assert a.engine_stats()[:2] == b.engine_stats()[:2]
    assert torch.equal(a.reduce_counts(), b.reduce_counts()) and torch.equal(c.reduce_counts(), b.reduce_counts())
    va, vb = a.host_view(["track_id", "state", "hits", "mean"]), b.host_view(["track_id", "state", "hits", "mean"])
    for k in va:
        np.testing.assert_array_equal(va[k], vb[k], err_msg=k)
    a.check()
    c.check()
