"""The presence section of the ragged detection batch (deepdish_b200/ragged.py): layout, round trip, and a blob
without presence unchanged byte for byte."""
import numpy as np
import pytest

from deepdish_b200 import ragged


def _batch(rng, n, D, counts):
    tlwh = rng.integers(0, 600, (n, D, 4)).astype(np.float64)
    conf = rng.uniform(0.5, 1, (n, D)).astype(np.float32)
    label = rng.integers(0, 3, (n, D)).astype(np.int32)
    feat = rng.normal(size=(n, D, 128)).astype(np.float32)
    return tlwh, conf, label, feat, np.asarray(counts, np.int64)


@pytest.mark.parametrize("counts,present", [([3, 0, 5, 1], [1, 1, 0, 1]), ([2, 2, 2], [0, 0, 0]), ([6, 6], [1, 1]),
                                            ([1], [0]), ([4, 99, -3, 2, 0], [1, 0, 0, 1, 1])])
def test_presence_round_trip(counts, present):
    rng = np.random.default_rng(1)
    n, D = len(counts), 6
    tlwh, conf, label, feat, cnt = _batch(rng, n, D, counts)
    pres = np.asarray(present, bool)
    blob, total, sections = ragged.pack(tlwh, conf, label, feat, cnt, present=pres)
    assert len(sections) == 5
    o_tlwh, o_conf, o_label, o_feat, o_present = sections
    eff = np.where(pres, cnt, 0)                     # an absent stream owns no entries; its count is never read
    N = int(eff.sum())
    assert (o_tlwh, o_conf, o_label, o_feat) == ragged.section_offsets(n, N)[0]
    assert o_present % 16 == 0 and o_present >= o_feat + 512 * N and total == o_present + n
    assert list(blob[:4 * (n + 1)].view(np.int32)) == [0] + list(np.cumsum(eff))
    np.testing.assert_array_equal(blob[o_present:total], pres.astype(np.uint8))
    t2, c2, l2, f2, k2, p2 = ragged.unpack(blob, n, D, present=True)
    np.testing.assert_array_equal(p2, pres)
    np.testing.assert_array_equal(k2, eff)
    sel = np.arange(D)[None, :] < eff[:, None]
    for got, exp in ((t2, tlwh), (c2, conf), (l2, label), (f2, feat)):
        np.testing.assert_array_equal(got[sel], exp[sel])
        assert not got[~sel].any()


@pytest.mark.parametrize("counts", [[3, 0, 5, 1], [0, 0], [6]])
def test_no_presence_is_byte_identical(counts):
    """present=None packs exactly the blob, size and four offsets of a batch without presence, and unpack's default
    return value is unchanged; an all-present section only appends bytes."""
    rng = np.random.default_rng(2)
    n, D = len(counts), 6
    args = _batch(rng, n, D, counts)
    a, ta, sa = ragged.pack(*args)
    b, tb, sb = ragged.pack(*args, present=None)
    assert ta == tb and sa == sb and len(sa) == 4 and a[:ta].tobytes() == b[:tb].tobytes()
    assert ragged.section_offsets(n, int(sum(counts))) == ragged.section_offsets(n, int(sum(counts)), False)
    assert len(ragged.unpack(a, n, D)) == 5
    c, tc, sc = ragged.pack(*args, present=np.ones(n, bool))
    assert sc[:4] == sa and c[:ta].tobytes() == a[:ta].tobytes()


def test_presence_shape_is_checked_and_absent_counts_are_not():
    rng = np.random.default_rng(3)
    tlwh, conf, label, feat, cnt = _batch(rng, 3, 4, [1, 2, 3])
    with pytest.raises(ValueError):
        ragged.pack(tlwh, conf, label, feat, cnt, present=[1, 0])
    cnt[1] = 50                                      # over capacity, but the stream is absent
    ragged.pack(tlwh, conf, label, feat, cnt, present=[1, 0, 1])
    with pytest.raises(ValueError):
        ragged.pack(tlwh, conf, label, feat, cnt, present=[1, 1, 1])
