"""Frame presence on the B200: ticks in which only some streams have a frame (``step(present=...)``,
``pack_host(batch, present)`` + ``step_host_packed``) against the oracle that does not step the absent streams, the
state of an absent stream bit for bit, and the equivalence of all-present with no presence."""
import numpy as np
import pytest
import torch

from deepdish_b200 import _lib
from tests import presence as P
from tests.parity import OracleStreams, compare_stream, LABELS3

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def scene():
    return P.PresenceScene()


def _tracker(n_chunks=1, **kw):
    from deepdish_b200.batched import BatchedTracker
    kw.setdefault("budget", P.BUDGET)
    return BatchedTracker(P.S, LABELS3, max_tracks=48, max_dets=P.DMAX, max_age=P.MAX_AGE, n_chunks=n_chunks,
                          device=DEV, **kw)


def _tick(bt, b, p, path):
    """One tick with presence p (numpy bool [S]); -> the det -> track ids (numpy)."""
    if path == "step":
        bt.step(b.to(DEV), present=torch.from_numpy(p).to(DEV), reduce=True)
        return bt.det_track_id.cpu().numpy()
    out = torch.full((P.S, P.DMAX), -7, dtype=torch.int32).pin_memory()
    bt.step_host_packed(bt.pack_host(b, p), out)
    bt.join()
    torch.cuda.synchronize()
    return out.numpy().copy()


def _final(bt, orc, gallery_streams=(0, 6, 11)):
    bt.check()
    v = bt.host_view()
    rows = lambda s, slot: bt.gallery(s, slot).cpu().numpy()
    for s in range(P.S):
        compare_stream(orc.trk[s], orc.cnt[s], v, s, LABELS3, gallery_rows=rows if s in gallery_streams else None)
    bt.join()
    np.testing.assert_array_equal(bt.total_counts.cpu().numpy(), sum(c.counts(LABELS3) for c in orc.cnt))


@pytest.mark.parametrize("path", ["step", "host"])
@pytest.mark.parametrize("n_chunks", [1, 3])
def test_presence_parity(scene, n_chunks, path):
    """~30 % random drops, bursts of absence far longer than max_age, a stream always present, a stream absent until
    tick 50, ticks without any frame and a tick without a frame right after one that counted a deletion at the line:
    ids every tick (absent rows all -1), then the state of every stream and the counters against the oracle."""
    assert scene.absent_after_del > 0
    bt = _tracker(n_chunks)
    for f, (b, p, exp) in enumerate(zip(scene.frames, scene.present, scene.ids)):
        P.check_tick_ids(_tick(bt, b, p, path), exp, p, f)
    _final(bt, scene.orc)


def test_absent_stream_state_is_bit_for_bit_unchanged(scene):
    """Across every tick in which a stream has no frame, each of its per-stream and per-slot arrays and the f32 and half
    rows of its gallery pages stay exactly as they were -- also for absences far longer than max_age, and whatever its
    rows of the detection batch hold (garbage, a count above max_dets: no overflow flag)."""
    bt = _tracker(2)
    rng = np.random.default_rng(0)

    def pages(s):
        c = bt._chunk_of(s)
        sp = c.cfg.seg_pages

        def get(pid):
            f32, f16 = c.segs[pid // sp]
            k = pid % sp
            return (f32[k * _lib.PAGE_F32_BYTES:(k + 1) * _lib.PAGE_F32_BYTES].cpu().numpy(),
                    f16[k * _lib.PAGE_F16_BYTES:(k + 1) * _lib.PAGE_F16_BYTES].cpu().numpy())
        return get

    names = [n for n in bt.v.keys() if n not in P.SCRATCH]
    checked = 0
    for f, (b, p) in enumerate(zip(scene.frames, scene.present)):
        v = bt.host_view(names)
        before = {s: P.stream_state(v, bt.cfg, s, pages(s)) for s in np.flatnonzero(~p)}
        b = b.to(DEV)
        for s in np.flatnonzero(~p):
            b.tlwh[s] = torch.randn_like(b.tlwh[s]) * 1e6
            b.feat[s] = float("nan")
            b.label[s] = -5
            b.count[s] = P.DMAX + 7
        ids = bt.step(b, present=torch.from_numpy(p).to(DEV)).cpu().numpy()
        v = bt.host_view(names)
        for s, st in before.items():
            P.assert_same_state(st, P.stream_state(v, bt.cfg, s, pages(s)), (f, s))
            assert (ids[s] == -1).all()
            checked += 1
        assert list(bt.v["tick_present"].cpu().numpy()) == list(p.astype(np.int32))
    assert checked > 200
    bt.check()


def test_all_present_equals_no_presence(scene):
    """present all ones (bool and uint8) is bit-identical to present=None: ids every tick and the whole state."""
    a, b_, c = _tracker(3), _tracker(3), _tracker(3)
    ones_b = torch.ones(P.S, dtype=torch.bool, device=DEV)
    ones_u = torch.ones(P.S, dtype=torch.uint8, device=DEV)
    for f, b in enumerate(scene.frames[:80]):
        b = b.to(DEV)
        ia = a.step(b, present=ones_b).cpu().numpy()
        ib = b_.step(b).cpu().numpy()
        ic = c.step(b, present=ones_u).cpu().numpy()
        np.testing.assert_array_equal(ia, ib)
        np.testing.assert_array_equal(ic, ib)
    # host_view() leaves out the page tables and the free stack: which page an append takes depends on the order in
    # which CTAs reach the pool, so the gallery rows themselves are compared instead
    va, vb, vc = a.host_view(), b_.host_view(), c.host_view()
    assert va.keys() == vb.keys() == vc.keys()
    for n in va:
        assert va[n].tobytes() == vb[n].tobytes() == vc[n].tobytes(), n
    for t in (a, b_, c):
        assert (t.v["tick_present"].cpu().numpy() == 1).all()
    for s in range(P.S):
        for slot in np.flatnonzero(va["gal_len"][s] > 0):
            ga = a.gallery(s, int(slot)).cpu().numpy()
            assert ga.tobytes() == b_.gallery(s, int(slot)).cpu().numpy().tobytes() == \
                c.gallery(s, int(slot)).cpu().numpy().tobytes(), (s, slot)


def test_unbounded_galleries_from_a_small_pool_with_absences_running_ahead(scene):
    """nn_budget=None on three chunks from a pool and page tables far too small, host-path ticks with presence enqueued
    back to back without a host synchronisation: pool growth and page-table re-layouts keep up, nothing overflows,
    and ids and state equal the oracle."""
    bt = _tracker(3, budget=None, pool_pages=64, seg_pages=64, page_cap=2)
    orc = OracleStreams(P.S, LABELS3, budget=None, max_age=P.MAX_AGE)
    packed = [bt.pack_host(b, p) for b, p in zip(scene.frames, scene.present)]
    out = [torch.full((P.S, P.DMAX), -7, dtype=torch.int32).pin_memory() for _ in packed]
    for f, pk in enumerate(packed):
        bt.step_host_packed(pk, out[f])
    bt.join()
    torch.cuda.synchronize()
    bt.check()
    for f, (b, p) in enumerate(zip(scene.frames, scene.present)):
        P.check_tick_ids(out[f].numpy(), P.oracle_tick(orc, b, p), p, f)
    assert any(len(c.segs) > 1 for c in bt.chunks) and any(_lib.page_cap(c.cfg) > 2 for c in bt.chunks)
    _final(bt, orc)


@pytest.mark.parametrize("kw", [dict(gallery_impl=1), dict(engine_graphs=False)])
def test_exact_gallery_pass_and_plain_launches(scene, kw):
    """gallery_impl=1 (the exact f32 pass, k_cosine) and plain kernel launches instead of graphs give the same ids."""
    bt = _tracker(3, **kw)
    for f, (b, p, exp) in enumerate(zip(scene.frames, scene.present, scene.ids)):
        P.check_tick_ids(_tick(bt, b, p, "step" if f % 2 else "host"), exp, p, f)
    _final(bt, scene.orc, gallery_streams=())


def test_per_call_update_steps_every_stream_after_absent_ticks(scene):
    """After engine ticks with absences, the per-call predict / update / count-line step every stream again."""
    bt = _tracker(2)
    orc = OracleStreams(P.S, LABELS3, budget=P.BUDGET, max_age=P.MAX_AGE)
    for f in range(40):
        b, p = scene.frames[f], scene.present[f]
        P.check_tick_ids(_tick(bt, b, p, "step"), P.oracle_tick(orc, b, p), p, f)
    allp = np.ones(P.S, bool)
    for f in range(40, 70):
        b = scene.frames[f]
        exp = P.oracle_tick(orc, b, allp)
        bd = b.to(DEV)
        bt.predict()
        ids = bt.update(bd.tlwh, bd.conf, bd.label, bd.feat, bd.count).cpu().numpy()
        bt.countline()
        P.check_tick_ids(ids, exp, allp, f)
    assert (bt.v["tick_present"].cpu().numpy() == 1).all()
    bt.check()
    v = bt.host_view()
    for s in range(P.S):
        compare_stream(orc.trk[s], orc.cnt[s], v, s, LABELS3)


def test_presence_input_validation(scene):
    bt = _tracker(2)
    b = scene.frames[0].to(DEV)
    S = P.S
    for bad in (torch.ones(S, dtype=torch.int32, device=DEV), torch.ones(S, dtype=torch.float32, device=DEV),
                torch.ones(S + 1, dtype=torch.bool, device=DEV), torch.ones((S, 1), dtype=torch.bool, device=DEV),
                torch.ones(S, dtype=torch.bool), torch.ones(2 * S, dtype=torch.bool, device=DEV)[::2],
                np.ones(S, bool)):
        with pytest.raises(ValueError):
            bt.step(b, present=bad)
    with pytest.raises(ValueError):
        bt.pack_host(scene.frames[0], np.ones(S + 1, bool))
    p = np.ones(S, bool)
    with_p, without = bt.pack_host(scene.frames[0], p), bt.pack_host(scene.frames[0])
    with pytest.raises(ValueError):                  # chunks must agree on carrying presence
        bt.step_host_packed([with_p[0], without[1]])
    blob, total, sec = with_p[0]
    with pytest.raises(ValueError):                  # the presence section must lie inside the uploaded bytes
        bt.step_host_packed([(blob, total, sec[:4] + (total - 1,)), with_p[1]])
    with pytest.raises(ValueError):
        bt.step_host_packed(with_p[:1])
    # nothing above reached the device: the tracker still matches the oracle from its first tick
    orc = OracleStreams(S, LABELS3, budget=P.BUDGET, max_age=P.MAX_AGE)
    for f in range(5):
        fb, fp = scene.frames[f], scene.present[f]
        P.check_tick_ids(_tick(bt, fb, fp, "host"), P.oracle_tick(orc, fb, fp), fp, f)
