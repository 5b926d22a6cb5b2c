"""Matching edges on the GPU: every scenario of tests/matching_edges.py and the seeded exact-cost fuzz streams through
the CUDA BatchedTracker against the oracle -- ids, lifecycle, Kalman state, error flags, gate bits and cost entries
bit for bit after every tick -- with the one-warp matching kernel and the CTA kernels (4 and 8 warps), one and two
stream chunks, both gallery implementations, the per-call update path and a track capacity that picks the CTA kernel
automatically.  The lane-parallel parts (ballot compaction, the tie key of the assignment scans, the fast path of
each row's first scan) only run here."""
import pytest
import torch

from tests import matching_edges as M
from tests.parity import LABELS3

pytestmark = pytest.mark.gpu

FUZZ_SEEDS = tuple(range(12))


class _Bt:
    """run_group's implementation interface over a BatchedTracker (engine ticks, or predict / update / countline)."""

    def __init__(self, S, T, D, max_age, cos, iou, per_call=False, **kw):
        from deepdish_b200.batched import BatchedTracker
        self.bt = BatchedTracker(S, LABELS3, max_tracks=T, max_dets=D, budget=M.BUDGET, max_age=max_age,
                                 max_cosine_distance=cos, max_iou_distance=iou, **kw)
        self.per_call = per_call

    def tick(self, b):
        d = b.to("cuda")
        if self.per_call:
            self.bt.predict()
            ids = self.bt.update(d.tlwh, d.conf, d.label, d.feat, d.count)
            self.bt.countline()
        else:
            ids = self.bt.step(d)
        return ids.cpu().numpy()

    def view(self, names):
        return self.bt.host_view(list(names))

    def set(self, name, s, slot, value):
        c = self.bt._chunk_of(s)
        self.bt.join()
        c.v[name][s - c.lo, slot] = value           # on the caller's stream, which the next tick waits for

    def gallery(self, s, slot):
        return self.bt.gallery(s, slot).cpu().numpy()


def _factory(**kw):
    return lambda *a: _Bt(*a, **kw)


@pytest.fixture(scope="module")
def scenarios():
    fuzz = [sc for seed in FUZZ_SEEDS for sc in M.fuzz_scenarios(seed)]
    return M.hand_scenarios(), fuzz


def _run(scenarios, max_tracks=None, **kw):
    hand, fuzz = scenarios
    checked, cnt = M.run_all(hand, _factory(**kw), max_tracks=max_tracks)
    for k in M.COUNTERS:
        assert cnt[k] > 0, (k, cnt)
    checked += M.run_all(fuzz, _factory(**kw), max_tracks=max_tracks)[0]
    assert checked > 1000


@pytest.mark.parametrize("gallery_impl", ["default", "exact"])
@pytest.mark.parametrize("n_chunks", [1, 2])
@pytest.mark.parametrize("match_warps", [1, 4, 8])
def test_matching_edges_engine(scenarios, match_warps, n_chunks, gallery_impl):
    _run(scenarios, match_warps=match_warps, n_chunks=n_chunks, gallery_impl=gallery_impl)


def test_matching_edges_per_call(scenarios):
    _run(scenarios, per_call=True)


def test_matching_edges_automatic_cta_kernel(scenarios):
    """max_tracks 192 (> 160): the matching kernel is chosen automatically, and it is the 4-warp CTA kernel."""
    _run(scenarios, max_tracks=192)
