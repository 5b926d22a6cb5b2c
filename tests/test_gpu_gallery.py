"""The gallery kernel's half-precision pre-pass must be invisible: its cost entries (min cosine distance of every
gate-passing (track, detection) pair) are compared BIT FOR BIT with the exact f32 pass on the same tracker history,
on scenes built to stress the re-check: identical gallery rows (every row inside the window), near-duplicates,
short galleries (fewer rows than one 16-row step), budgets that are not multiples of 16, more than 8 gate-passing
detections per track (several query groups) and more than 32 detections (several gate words)."""
import functools

import numpy as np
import pytest
import torch

from deepdish_b200.scene import Scene
from tests.parity import LABELS3

pytestmark = pytest.mark.gpu

# BatchedTracker knobs of the half pre-pass (k_gallery_stream) under test; each must leave the costs bit-identical.
# gallery_stages: ring stages per triple (1 = the producer and the mma warp hand one stage back and forth);
# cosine_ctas_per_sm: triples per CTA (per SM), or with gallery_waves one-triple CTAs per SM and wave;
# gallery_waves: grid of SMs x triples x waves one-triple CTAs, each claiming a bounded quota of the work list.
KNOBS = {
    "default": {},
    "stages1": dict(gallery_stages=1),
    "stages2": dict(gallery_stages=2),
    "stages3": dict(gallery_stages=3),
    "stages5": dict(gallery_stages=5),
    "stages16": dict(gallery_stages=16),
    "ctas1": dict(cosine_ctas_per_sm=1),
    "ctas2": dict(cosine_ctas_per_sm=2),
    "waves1_ctas1": dict(gallery_waves=1, cosine_ctas_per_sm=1),
    "waves1_ctas8": dict(gallery_waves=1, cosine_ctas_per_sm=8),
    "waves2_ctas1": dict(gallery_waves=2, cosine_ctas_per_sm=1),
    "waves2_ctas8": dict(gallery_waves=2, cosine_ctas_per_sm=8),
}


def _history(impl, S, nobj, dmax, tmax, budget, frames, seed, feat_noise, big_boxes=False, scene=None, flags=0,
             pool_fraction=0.5):
    """impl: "exact" (the f32 pass) or a KNOBS key (the half pre-pass with those knobs).  scene: a factory of the
    scene to run instead of Scene(S, nobj, dmax, ...); flags: the status the run must end with (0: bt.check())."""
    from deepdish_b200.batched import BatchedTracker
    knobs = dict(gallery_impl="exact") if impl == "exact" else KNOBS[impl]
    bt = BatchedTracker(S, LABELS3, max_tracks=tmax, max_dets=dmax, budget=budget, max_age=30, page_cap=8,
                        pool_fraction=pool_fraction, **knobs)
    sc = scene() if scene is not None else Scene(S, nobj, dmax, n_labels=3, seed=seed, feat_noise=feat_noise)
    if big_boxes:                      # large slow boxes: many detections pass each track's Mahalanobis gate
        sc.size = sc.size * 4.0
        sc.vel = sc.vel * 0.2
    out = []
    for f in range(frames):
        b = sc.step().to("cuda")
        ids = bt.step(b).cpu().numpy().copy()
        bt.maintain(wait=True)
        gate = bt.v["gate"].cpu().numpy().astype(np.uint32)
        cost = bt.v["cost"].cpu().numpy()
        state = bt.v["state"].cpu().numpy()
        out.append((ids, gate, cost, state, int(bt.v["work_ctl"][0])))
    if flags:
        assert bt.status() == flags
    else:
        bt.check()
    return out


@functools.lru_cache(maxsize=None)
def _exact(name):
    """The exact pass's history of a scene, shared by every knob set compared with it."""
    return _history("exact", **SCENES[name])


def _compare(name, half, exact):
    """Bit-identical ids, gate words and costs of every gate-passing entry, tick by tick.  Returns (entries checked,
    most gate-passing detections of one track on one tick)."""
    checked = many = 0
    for f, ((ih, gh, ch, sh, _), (ie, ge, ce, se, _)) in enumerate(zip(half, exact)):
        np.testing.assert_array_equal(ih, ie, err_msg="%s ids frame %d" % (name, f))
        np.testing.assert_array_equal(gh, ge)
        S, T, D = ch.shape
        bits = ((gh[:, :, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(S, T, -1)[:, :, :D].astype(bool)
        # gate words of slots that were not confirmed at gating time are stale; ids equal => same tracks were gated.
        # Compare every entry both runs wrote this tick: identical bit patterns.
        a, b = ch.view(np.uint32), ce.view(np.uint32)
        np.testing.assert_array_equal(a[bits], b[bits], err_msg="%s cost bits frame %d" % (name, f))
        checked += int(bits.sum())
        many = max(many, int(bits.sum(axis=2).max()))
    return checked, many


SCENES = dict([
    ("plain", dict(S=6, nobj=20, dmax=24, tmax=64, budget=100, frames=70, seed=41, feat_noise=0.02)),
    ("identical_rows", dict(S=4, nobj=12, dmax=16, tmax=48, budget=37, frames=60, seed=42, feat_noise=0.0)),
    ("near_duplicates", dict(S=4, nobj=12, dmax=16, tmax=48, budget=20, frames=50, seed=43, feat_noise=2e-4)),
    ("short_gallery_budget_5", dict(S=4, nobj=12, dmax=16, tmax=48, budget=5, frames=40, seed=44, feat_noise=0.02)),
    ("many_candidates_two_gate_words", dict(S=3, nobj=40, dmax=48, tmax=128, budget=33, frames=40, seed=45,
                                            feat_noise=0.05, big_boxes=True)),
    # identical rows x up to 8 gate-passing detections: more window candidates than a checker message lists (240), so
    # the checker's evaluate-everything fallback runs
    ("identical_rows_many_candidates", dict(S=3, nobj=30, dmax=40, tmax=96, budget=100, frames=115, seed=48,
                                            feat_noise=0.0, big_boxes=True)),
    # a crowd: more than 16 gate-passing detections per track (three and more jobs per gallery), five gate words, the
    # four-warp matching kernel
    ("crowd_many_jobs_per_track", dict(S=2, nobj=70, dmax=144, tmax=192, budget=33, frames=30, seed=49,
                                      feat_noise=0.05, big_boxes=True)),
    # nn_budget=None: galleries of ~300 rows span several 256-row blocks of the half pre-pass (running maximum)
    ("unbounded_multi_block", dict(S=2, nobj=8, dmax=12, tmax=32, budget=None, frames=340, seed=46, feat_noise=0.01)),
    ("unbounded_identical_rows", dict(S=2, nobj=6, dmax=8, tmax=32, budget=None, frames=300, seed=47, feat_noise=0.0)),
])
# every knob set runs the scenes with a ragged last page, the checker's evaluate-everything fallback, several jobs per
# track and several 128-row blocks; the default knobs run every scene
CORE = ("short_gallery_budget_5", "identical_rows_many_candidates", "crowd_many_jobs_per_track", "unbounded_multi_block")
CASES = [(impl, name) for impl in KNOBS for name in SCENES if impl == "default" or name in CORE]


@pytest.mark.parametrize("impl,name,kw", [(impl, name, SCENES[name]) for impl, name in CASES],
                         ids=["%s-%s-kw%d" % (impl, name, list(SCENES).index(name)) for impl, name in CASES])
def test_half_prepass_costs_are_bit_identical_to_the_exact_pass(name, kw, impl):
    checked, many = _compare(name, _history(impl, **kw), _exact(name))
    assert checked > 500
    if name == "many_candidates_two_gate_words":
        assert many > 8
    if name == "identical_rows_many_candidates":
        assert many >= 3
    if name == "crowd_many_jobs_per_track":
        assert many > 16


def test_bounded_claim_loop_stops_mid_list():
    """gallery_waves=1, one triple per CTA: the grid is one CTA per SM and each claims an even share of the work list
    (quota = ceil(entries / grid) rounded up to even).  With more than two entries per CTA the producers stop claiming
    mid-list; with an empty list (the first ticks: no confirmed track yet) every CTA only posts its stop job.  Costs and
    ids bit-identical to the exact pass."""
    kw = dict(S=12, nobj=50, dmax=64, tmax=128, budget=100, frames=20, seed=51, feat_noise=0.02)
    half = _history("waves1_ctas1", **kw)
    checked, _ = _compare("bounded_claims", half, _history("exact", **kw))
    grid = torch.cuda.get_device_properties(0).multi_processor_count * 1 * 1       # SMs x triples x waves
    entries = [h[4] for h in half]
    assert entries[0] == 0 and max(entries) > 2 * grid, (grid, entries)
    assert checked > 500
