"""The end-to-end host path as a deployment drives it: ``step_host_packed`` ticks enqueued back to back while the host
never synchronises, so that uploads, ticks, read-backs, pool polls and storage growth of many ticks are in flight at
once.  Every frame is packed first (each pinned blob stays alive) and every tick writes its ids into its own pinned
buffer; the loop does no oracle work (that would slow the host until it never runs ahead).  After one join and
synchronisation every tick's ids are compared bit for bit, and the final state with the oracle or with a tracker driven
through ``step()``."""
import numpy as np
import pytest
import torch

from deepdish_b200 import _lib
from deepdish_b200.scene import Scene, SceneBatch
from tests.parity import OracleStreams, compare_stream, LABELS3

pytestmark = pytest.mark.gpu


def _frames(S, nobj, dmax, n, seed):
    sc = Scene(S, nobj, dmax, n_labels=3, seed=seed)
    return [sc.step() for _ in range(n)]


class _Busy:
    """Ordinary work queued on the caller's stream in front of a tick or an edit (a few large matrix products): an
    edit the tracker makes on that stream then runs well after the host has enqueued the next tick."""

    def __init__(self, n=3):
        g = torch.Generator(device="cuda").manual_seed(0)
        self.a = torch.randn(4096, 4096, device="cuda", generator=g)
        self.c = torch.empty_like(self.a)
        self.n = n

    def __call__(self):
        for _ in range(self.n):
            torch.matmul(self.a, self.a, out=self.c)


def _run_ahead(bt, frames, before_tick=None, after_tick=None):
    """Enqueue one host-path tick per frame without synchronising; return each tick's ids (numpy) and the packed
    blobs.  before_tick(f) / after_tick(f) enqueue more work around tick f."""
    S, D = bt.n_streams, bt.max_dets
    packed = [bt.pack_host(b) for b in frames]
    out = [torch.full((S, D), -7, dtype=torch.int32).pin_memory() for _ in frames]
    for f, p in enumerate(packed):
        if before_tick is not None:
            before_tick(f)
        bt.step_host_packed(p, out[f])
        if after_tick is not None:
            after_tick(f)
    bt.join()
    torch.cuda.synchronize()
    return [o.numpy().copy() for o in out], packed


def _check_oracle(bt, frames, got, orc, gallery_streams=()):
    bt.check()                      # a capacity flag explains a mismatch below
    for f, b in enumerate(frames):
        exp = orc.step(b)
        for s in range(bt.n_streams):
            assert list(got[f][s, :int(b.count[s])]) == exp[s], (f, s)
    v = bt.host_view()
    rows = lambda s, slot: bt.gallery(s, slot).cpu().numpy()
    for s in range(bt.n_streams):
        compare_stream(orc.trk[s], orc.cnt[s], v, s, LABELS3, gallery_rows=rows if s in gallery_streams else None)
    np.testing.assert_array_equal(bt.total_counts.cpu().numpy(), sum(c.counts(LABELS3) for c in orc.cnt))


@pytest.mark.parametrize("busy_caller", [False, True])
def test_unbounded_galleries_grow_while_running_ahead(busy_caller):
    """nn_budget=None on three chunks from a pool and page tables far too small: the engine's pool polls make
    maintain() attach segments and re-lay out the page tables between host-path ticks the host is still running ahead
    of.  busy_caller: matrix products queued on the caller's stream before every tick.  The re-layout's copies into the
    new blob run on that stream, well after the next tick has been enqueued on the chunk's stream, and the chunk streams
    lag the host by several ticks, so storage grows from polls that complete late."""
    from deepdish_b200.batched import BatchedTracker
    S, D, T, MAX_AGE, TICKS = 6, 14, 40, 20, 260
    bt = BatchedTracker(S, LABELS3, max_tracks=T, max_dets=D, budget=None, max_age=MAX_AGE, n_chunks=3,
                        pool_pages=64, seg_pages=64, page_cap=2)
    frames = _frames(S, 10, D, TICKS, seed=21)
    busy = _Busy() if busy_caller else None
    caps = []
    got, _ = _run_ahead(bt, frames, before_tick=(lambda f: busy()) if busy else None,
                        after_tick=lambda f: caps.append([_lib.page_cap(c.cfg) for c in bt.chunks]))
    orc = OracleStreams(S, LABELS3, budget=None, max_age=MAX_AGE)
    _check_oracle(bt, frames, got, orc, gallery_streams=(0, 3, 5))
    assert all(len(c.segs) > 1 for c in bt.chunks)
    grew = [f for f in range(1, TICKS) if caps[f] != caps[f - 1]]
    assert grew and max(grew) > 100, grew                   # a re-layout in the middle of the run-ahead stretch
    assert max(len(g) for t in orc.trk for g in t.metric.samples.values()) > 128


@pytest.mark.parametrize("upload_buffers", [2, 3, 4])
def test_upload_buffer_rotation(upload_buffers):
    """UPLOAD_BUFFERS device blobs per chunk (2 .. 4) in rotation: an upload must wait for the tick that last read its
    buffer, however far ahead the host is."""
    from deepdish_b200.batched import BatchedTracker
    S, D = 6, 16
    bt = BatchedTracker(S, LABELS3, max_tracks=48, max_dets=D, budget=20, max_age=30, n_chunks=2, pool_fraction=1.0)
    assert not bt._poll_pool
    bt.UPLOAD_BUFFERS = upload_buffers
    frames = _frames(S, 12, D, 60, seed=60 + upload_buffers)
    got, _ = _run_ahead(bt, frames)
    assert all(len(c.blob_dev) == upload_buffers for c in bt.chunks)
    _check_oracle(bt, frames, got, OracleStreams(S, LABELS3, budget=20, max_age=30), gallery_streams=(1, 4))


def test_split_upload_single_chunk():
    """A chunk blob over 4 MiB is uploaded in two halves on two copy streams; the tick waits for both."""
    from deepdish_b200.batched import BatchedTracker
    S, D = 192, 56
    bt = BatchedTracker(S, LABELS3, max_tracks=96, max_dets=D, budget=100, max_age=30)
    frames = _frames(S, 48, D, 12, seed=71)
    got, packed = _run_ahead(bt, frames)
    assert all(p[0][1] > 4 << 20 for p in packed), [p[0][1] for p in packed]
    _check_oracle(bt, frames, got, OracleStreams(S, LABELS3, budget=100, max_age=30), gallery_streams=(0, 191))


def test_split_upload_two_chunks_against_device_ticks():
    """Two chunks, each blob over 4 MiB: every stream bit-identical to a tracker driven through step() on the padded
    device batches, and a sample of streams replayed through the oracle."""
    from deepdish_b200.batched import BatchedTracker
    S, D, T = 384, 56, 96
    kw = dict(max_tracks=T, max_dets=D, budget=100, max_age=30, n_chunks=2)
    frames = _frames(S, 48, D, 12, seed=72)
    a = BatchedTracker(S, LABELS3, **kw)
    got, packed = _run_ahead(a, frames)
    assert all(p[k][1] > 4 << 20 for p in packed for k in range(2)), [[q[1] for q in p] for p in packed]
    b = BatchedTracker(S, LABELS3, **kw)
    sample = list(range(0, S, 24))
    orc = OracleStreams(len(sample), LABELS3, budget=100, max_age=30)
    idx = torch.as_tensor(sample)
    for f, fr in enumerate(frames):
        ib = b.step(fr.to("cuda")).cpu().numpy()
        np.testing.assert_array_equal(got[f], ib, err_msg="tick %d" % f)
        exp = orc.step(SceneBatch(*(getattr(fr, k)[idx] for k in SceneBatch.__slots__)))
        for k, s in enumerate(sample):
            assert list(got[f][s, :int(fr.count[s])]) == exp[k], (f, s)
    a.check()
    b.check()
    va, vb = a.host_view(), b.host_view()
    for name in ("n_tracks", "next_id", "n_deleted", "counts"):
        np.testing.assert_array_equal(va[name], vb[name], err_msg=name)
    live = np.arange(T)[None, :] < va["n_tracks"][:, None]
    np.testing.assert_array_equal(va["order"][live], vb["order"][live])
    rows, slots = np.repeat(np.arange(S), va["n_tracks"]), va["order"][live]
    for name in ("track_id", "state", "hits", "age", "tsu", "gal_len", "gal_pos", "mean", "cov"):
        np.testing.assert_array_equal(va[name][rows, slots], vb[name][rows, slots], err_msg=name)
    sub = {k: v[sample] for k, v in va.items()}
    for k in range(len(sample)):
        compare_stream(orc.trk[k], orc.cnt[k], sub, k, LABELS3)
    np.testing.assert_array_equal(a.total_counts.cpu().numpy(), va["counts"].sum(axis=0))


def test_gallery_insert_between_host_ticks():
    """gallery_insert runs on the caller's stream; host-path ticks do not fork from it.  With a pool that covers the
    worst case nothing else orders the two, and matrix products queued in front of every tick and insert keep the
    insert late.  Ids, track tables and gallery rows bit-identical to a tracker driven through step() that receives the
    same inserts."""
    from deepdish_b200.batched import BatchedTracker
    S, D, T, TICKS = 6, 16, 48, 70
    kw = dict(max_tracks=T, max_dets=D, budget=20, max_age=30, n_chunks=2, pool_fraction=1.0)
    frames = _frames(S, 12, D, TICKS, seed=81)
    rng = np.random.default_rng(81)
    # the reference run decides where the inserts go: a confirmed track's slot, in a stream of either chunk
    b = BatchedTracker(S, LABELS3, **kw)
    inserts, ids_b = {}, []
    for f, fr in enumerate(frames):
        ids_b.append(b.step(fr.to("cuda")).cpu().numpy().copy())
        if f >= 8 and f % 5 == 3:
            s = (f // 5) % S
            v = b.host_view(["n_tracks", "order", "state"], streams=[s])
            conf = [int(sl) for sl in v["order"][0, :int(v["n_tracks"][0])] if v["state"][0, sl] == 2]
            if conf:
                feat = rng.standard_normal(128).astype(np.float32)
                feat /= np.linalg.norm(feat)
                inserts[f] = (s, conf[len(conf) // 2], feat, (f // 5) % 2 == 1)
                b.gallery_insert(*inserts[f][:3], before_newest=inserts[f][3])
    assert len(inserts) >= 8 and any(x[3] for x in inserts.values()) and not all(x[3] for x in inserts.values())
    a = BatchedTracker(S, LABELS3, **kw)
    assert not a._poll_pool
    busy = _Busy()

    def insert(f):
        if f in inserts:
            busy()
            s, slot, feat, before = inserts[f]
            a.gallery_insert(s, slot, feat, before_newest=before)

    got, _ = _run_ahead(a, frames, before_tick=lambda f: busy(), after_tick=insert)
    for f in range(TICKS):
        np.testing.assert_array_equal(got[f], ids_b[f], err_msg="tick %d" % f)
    a.check()
    b.check()
    names = ["n_tracks", "order", "track_id", "state", "hits", "age", "tsu", "gal_len", "gal_pos", "mean", "cov",
             "next_id", "n_deleted", "deleted", "counts"]
    va, vb = a.host_view(names), b.host_view(names)
    for k in names:
        np.testing.assert_array_equal(va[k], vb[k], err_msg=k)
    checked = 0
    for s in range(S):
        for sl in va["order"][s, :int(va["n_tracks"][s])]:
            if va["state"][s, sl] == 2:
                ra, rb = a.gallery(s, int(sl)).cpu().numpy(), b.gallery(s, int(sl)).cpu().numpy()
                np.testing.assert_array_equal(ra.view(np.uint32), rb.view(np.uint32), err_msg="stream %d slot %d" % (s, sl))
                checked += len(ra)
    assert checked > 0
