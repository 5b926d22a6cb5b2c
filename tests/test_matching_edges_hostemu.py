"""Matching edges on the CPU: every scenario of tests/matching_edges.py and the seeded exact-cost fuzz streams through
the host emulation (the kernel bodies compiled with a one-lane group) against the oracle -- ids, lifecycle, Kalman
state, gate bits and cost entries bit for bit -- and coverage counters that show each edge was reached."""
import numpy as np
import pytest

from deepdish_b200 import _lib as L
from tests import matching_edges as M
from tests.hostemu.driver import HostEmuTracker
from tests.parity import LABELS3

FUZZ_SEEDS = tuple(range(40))


class _Emu:
    """run_group's implementation interface over the host emulation (fused tick, or the per-call order)."""

    def __init__(self, S, T, D, max_age, cos, iou, per_call=False):
        cfg = L.make_config(S, T, D, M.BUDGET, LABELS3, max_age=max_age, max_cosine_distance=cos,
                            max_iou_distance=iou)
        self.emu, self.per_call = HostEmuTracker(cfg), per_call

    def tick(self, b):
        a = (b.tlwh.numpy(), b.conf.numpy(), b.label.numpy(), b.feat.numpy(), b.count.numpy())
        if not self.per_call:
            return self.emu.tick(*a).copy()
        self.emu.predict()
        ids = self.emu.update(*a).copy()
        self.emu.countline()
        return ids

    def view(self, names):
        return {n: self.emu.v[n].copy() for n in names}

    def set(self, name, s, slot, value):
        self.emu.v[name][s, slot] = value

    def gallery(self, s, slot):
        return self.emu.gallery(s, slot)


def _factory(per_call=False):
    return lambda *a: _Emu(*a, per_call=per_call)


@pytest.fixture(scope="module")
def hand():
    return M.hand_scenarios()


def test_hand_scenarios_host_emulation(hand):
    checked, cnt = M.run_all(hand, _factory())
    assert checked > 200
    # every edge the scenarios are written for was reached
    for k in M.COUNTERS:
        assert cnt[k] > 0, (k, cnt)


def test_hand_scenarios_port_oracle_host_emulation(hand):
    """The same scenarios against the oracle built on the pure-Python LSAP and set-order ports (their set order
    assumes confirmed indices 0..n-1, so the non-contiguous scenario stays out)."""
    M.run_all([sc for sc in hand if sc.port], _factory(), port=True)


def test_hand_scenarios_per_call_host_emulation(hand):
    """predict / update / count-line issued call by call: the same decisions."""
    M.run_all([sc for sc in hand if sc.name.startswith(("cos_thr_at", "clip_", "all_clip", "set_order_40",
                                                         "noncontig", "iou_"))], _factory(per_call=True))


def test_fuzz_exact_costs_host_emulation():
    cnt = dict.fromkeys(M.COUNTERS, 0)
    checked = 0
    for seed in FUZZ_SEEDS:
        c, k = M.run_all(M.fuzz_scenarios(seed), _factory())
        checked += c
        for n in cnt:
            cnt[n] += k[n]
    assert checked > 1000
    for k in ("at_thr", "clip_band", "all_clip", "transposed"):
        assert cnt[k] > 0, (k, cnt)


def test_cost_construction_is_exact():
    """The premise of the module: each mixed cost is an exact f32 value that numpy's BLAS, a sequential fmaf-free sum
    and a reversed sum all give, and the thresholds drawn from them straddle it as intended."""
    for tri in M.TRIPLES:
        p, q, r = tri
        sc = M.Scn("x")
        f = sc.mix(3, tri)
        g = M.basis(3, 2.0)
        fn, gn = f / np.linalg.norm(f), g / np.linalg.norm(g)
        c = M.cos_cost(tri)
        assert float(np.float32(1) - np.dot(gn[None], fn[:, None])[0, 0]) == c
        assert float(np.float32(1) - np.float32(sum(gn[::-1] * fn[::-1]))) == c
        assert np.nextafter(c, 0) < c < np.nextafter(c, 1) and c - 5e-6 < c < c - 5e-6 + 1e-5
