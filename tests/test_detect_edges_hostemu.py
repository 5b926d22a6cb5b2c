"""Host-emulation counterpart of tests/test_gpu_detect_edges.py: the same generated NMS, YOLOv5 row and Keras YOLOv3
cases through the host build of the kernel bodies (tests/hostemu) against the oracle, so that the case generators and
the device functions the two builds share (dd_nms_suppresses, dd_yolo_row, dd_y3_suppresses) are checked without a
GPU.  The host build runs the serial #else branches of dd_nms_frame, not its device-only batch and scan paths."""
import numpy as np
import pytest

from oracle import detect as odet
from tests import detect_edges as de
from tests.hostemu import driver as hd


def _nms_check(boxes, scores, thr):
    exp = odet.non_max_suppression(boxes, thr, scores)
    assert hd.nms(boxes, scores, thr) == exp
    return exp


@pytest.mark.parametrize("thr", de.BIG_THRS)
def test_nms_big_frames_host_emulation(thr):
    b, s, counts = de.big_batch(np.random.default_rng(31))
    resumes = 0
    for f, c in enumerate(counts):
        n = min(int(c), de.NMS_NMAX)
        exp = _nms_check(b[f, :n], s[f, :n], thr)
        keep, r = de.nms_batches(b[f, :n], s[f, :n], thr)
        assert keep == exp
        resumes += r
    assert (counts > 1024).any() and (counts == de.NMS_NMAX).any() and (counts > de.NMS_NMAX).any()
    assert resumes > 0                   # some batch of 32 survivors filled inside a 32-rank window


@pytest.mark.parametrize("thr", de.FRAC_THRS)
def test_nms_fractional_and_mixed_host_emulation(thr):
    frames = de.fractional_frames(np.random.default_rng(32))
    for name, (b, s) in frames.items():
        _nms_check(b, s, thr)
    cov = de.fractional_coverage(frames)
    assert all(cov.values()), cov


@pytest.mark.parametrize("thr", de.EXACT_THRS)
def test_nms_exact_overlap_host_emulation(thr):
    B, S, C, pairs = de.exact_frames(np.random.default_rng(33), thr)
    for f in range(2):
        _nms_check(B[f, :C[f]], S[f, :C[f]], thr)
    exact, below, above = de.exact_coverage(pairs, thr)
    assert exact >= 100 and below >= 20 and above >= 20, (exact, below, above)


@pytest.mark.parametrize("thr", (0.6, 0.3))
def test_nms_tied_scores_host_emulation(thr):
    for b, s in de.tied_frames(np.random.default_rng(34)):
        assert len(np.unique(s)) <= 8
        _nms_check(b, s, thr)


def test_yolo_rows_edges_host_emulation():
    head, kinds = de.yolo_edge_head(np.random.default_rng(35))
    de.assert_yolo_coverage(head, kinds, 0.25)
    tl, sc, cl, an, nan = hd.yolo_rows(head, de.YOLO_MASK, 0.25, (640, 480), (640, 480))
    ib, score, cls, anchor = de.yolo_reference(head, 0.25)
    assert nan == 0
    np.testing.assert_array_equal(an, anchor)
    np.testing.assert_array_equal(tl, ib)
    np.testing.assert_array_equal(sc, score)
    np.testing.assert_array_equal(cl, cls)
    u8, kinds = de.yolo_u8_edge_head(np.random.default_rng(36))
    head = odet.yolo_dequant(u8, de.u8_scale(), 0)
    de.assert_yolo_coverage(head, kinds, 0.25, step=2.0 ** -16)
    tl, sc, cl, an, nan = hd.yolo_rows(head, de.YOLO_MASK, 0.25, (640, 480), (640, 480))
    ib, score, cls, anchor = de.yolo_reference(head, 0.25)
    np.testing.assert_array_equal(an, anchor)
    np.testing.assert_array_equal(cl, cls)
    np.testing.assert_array_equal(sc, score)
    np.testing.assert_array_equal(tl, ib)


def test_yolo3_threshold_and_iou_edges_host_emulation():
    maps, thr = de.yolo3_edge_maps(np.random.default_rng(37))
    assert (de.yolo3_probabilities(maps) == np.float32(thr)).sum() >= 2
    v = de.yolo3_exact_iou(maps, thr)
    wm = np.array([1 if n in de.Y3_WANTED else 0 for n in de.Y3_NAMES], np.uint8)
    for nms in (v, float(np.nextafter(v, 1.0))):
        b, s, l, fl = hd.yolo3(maps, de.Y3_ANCHORS, len(de.Y3_NAMES), wm, thr, (640, 480), (de.Y3_NET, de.Y3_NET),
                               nms_thresh=nms)
        eb, el, es = de.yolo3_reference(maps, thr, nms)
        assert fl == 0
        np.testing.assert_array_equal(b, eb.astype(float))
        np.testing.assert_array_equal(l, el)
        np.testing.assert_array_equal(s.view(np.uint32), es.view(np.uint32))
