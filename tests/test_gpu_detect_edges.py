"""GPU parity of the detector post-processing at the edges the synthetic heads never reach: NMS above the register
path (up to the 3049-candidate limit) and on fractional, huge, negative and degenerate boxes, overlaps exactly on the
threshold and within 2 ulp of it, tied scores at n > 16 and n > 1024; YOLOv5 decode (f32 and u8) with scores exactly
on the threshold, tied top classes and NaN rows; the SSD, TFLite and Keras YOLOv3 thresholds hit exactly; and the
argument checks of the detector wrappers.  Everything is compared bit-exactly with oracle/detect.py, and every edge is
asserted in numpy to be present (tests/detect_edges.py builds the cases; tests/test_detect_edges_hostemu.py runs the
same cases through the host emulation)."""
import numpy as np
import pytest
import torch

from oracle import detect as odet
from oracle.make_golden import synth_yolo_head
from tests import detect_edges as de

pytestmark = pytest.mark.gpu

F32 = np.float32


def _nms(boxes, scores, counts, thr):
    from deepdish_b200 import ops
    keep, nkeep = ops.nms(torch.from_numpy(np.ascontiguousarray(boxes, np.float64)).cuda(),
                          torch.from_numpy(np.ascontiguousarray(scores, F32)).cuda(),
                          torch.from_numpy(np.asarray(counts, np.int32)).cuda(), thr)
    return keep.cpu().numpy(), nkeep.cpu().numpy()


def _pack(frames):
    nmax = max(len(b) for b, _ in frames)
    B = np.zeros((len(frames), nmax, 4))
    S = np.zeros((len(frames), nmax), F32)
    for f, (b, s) in enumerate(frames):
        B[f, :len(b)], S[f, :len(b)] = b, s
    return B, S, np.array([len(b) for b, _ in frames], np.int32)


def _check_frames(B, S, C, thr):
    keep, nkeep = _nms(B, S, C, thr)
    for f in range(len(C)):
        n = min(int(C[f]), B.shape[1])
        exp = odet.non_max_suppression(B[f, :n], thr, S[f, :n])
        assert int(nkeep[f]) == len(exp), (f, thr)
        assert list(keep[f, :nkeep[f]]) == exp, (f, thr)


@pytest.mark.parametrize("thr", de.BIG_THRS)
def test_nms_above_register_path(thr):
    """Frame counts 0 .. 3049 and one above nmax (clamped) in one launch: the register path (<= 1024) and the
    shared-memory window scan mixed; clustered boxes make batches of 32 survivors fill inside a 32-rank window."""
    B, S, C = de.big_batch(np.random.default_rng(31))
    assert B.shape[1] == de.NMS_NMAX and (C > 1024).any() and (C == de.NMS_NMAX).any() and (C > de.NMS_NMAX).any()
    _check_frames(B, S, C, thr)
    resumes = sum(de.nms_batches(B[f, :min(c, de.NMS_NMAX)], S[f, :min(c, de.NMS_NMAX)], thr)[1]
                  for f, c in enumerate(C) if c > 1024)
    assert resumes > 0


def test_nms_capacity_limit():
    """One candidate more than fits shared memory: refused by the API (DD_ERR_CAPACITY) before any launch."""
    with pytest.raises(RuntimeError, match="capacity"):
        _nms(np.zeros((1, de.NMS_NMAX + 1, 4)), np.zeros((1, de.NMS_NMAX + 1), F32), [1], 0.6)


@pytest.mark.parametrize("thr", de.FRAC_THRS)
def test_nms_fractional_and_mixed_boxes(thr):
    """Non-integer frames (n = 17 .. 2048), an integer frame with one fractional box, integer boxes beyond 2^20 and
    negative ones, nested / touching / sliver / degenerate pairs; thresholds 0.0 (the boundary of the disjointness
    shortcut), -0.1 (shortcut off) and 1.0."""
    frames = de.fractional_frames(np.random.default_rng(32))
    cov = de.fractional_coverage(frames)
    assert all(cov.values()), cov
    _check_frames(*_pack(list(frames.values())), thr)


@pytest.mark.parametrize("thr", de.EXACT_THRS)
def test_nms_exact_overlap_edges(thr):
    """Hundreds of non-interacting pairs per frame whose overlap is exactly thr in f64 (suppression is `>`), their
    +-1 px neighbours, and fractional pairs 1-2 ulp either side of thr (inside the guard band: the division decides);
    one frame on the register path, one above it."""
    B, S, C, pairs = de.exact_frames(np.random.default_rng(33), thr)
    exact, below, above = de.exact_coverage(pairs, thr)
    assert exact >= 100 and below >= 20 and above >= 20, (exact, below, above)
    assert C[0] <= 1024 < C[1]
    _check_frames(B, S, C, thr)


@pytest.mark.parametrize("thr", (0.6, 0.3))
def test_nms_tied_scores_large_frames(thr):
    """Scores from 8 distinct values at n = 17 .. 1500.  The reference leaves the order of tied scores at n > 16
    implementation-defined (numpy's argsort is unstable there); the project's declared rule -- the higher original
    index is picked first, what the oracle's stable sort gives -- is pinned at these sizes too."""
    frames = de.tied_frames(np.random.default_rng(34))
    assert all(len(np.unique(s)) <= 8 for _, s in frames) and max(len(b) for b, _ in frames) > 1024
    _check_frames(*_pack(frames), thr)


def _mask():
    return torch.from_numpy(de.YOLO_MASK).cuda()


def _yolo_compare(out, f, exp):
    n = int(out["count"][f])
    ib, score, cls, anchor = exp
    assert n == len(anchor), f
    np.testing.assert_array_equal(out["anchor"][f, :n], anchor)
    np.testing.assert_array_equal(out["tlwh"][f, :n], ib)
    np.testing.assert_array_equal(out["score"][f, :n], score)
    np.testing.assert_array_equal(out["cls"][f, :n], cls)


def test_yolo_decode_edges_f32():
    """Scores exactly on the threshold (0.5 * 0.5, 0.25 * 1) and one ulp either side, tied top classes (equal raw
    values, and equal products of different raw values) between a wanted and an unwanted class in both orders, rows
    with NaN objectness / a NaN class score (dropped: np.argmax returns the first NaN); frame 1 also has a NaN box
    coordinate in a passing row, which drops the whole frame."""
    from deepdish_b200 import ops
    head, kinds = de.yolo_edge_head(np.random.default_rng(35))
    de.assert_yolo_coverage(head, kinds, 0.25)
    bad = head.copy()
    bad[kinds["exact"][0], 0] = np.nan
    out = ops.yolo_decode(torch.from_numpy(np.stack([head, bad])).cuda(), _mask(), 0.25, (640, 480), (640, 480),
                          ncap=1024)
    o = {k: v.cpu().numpy() for k, v in out.items()}
    assert int(o["flags"][0]) == 0 and int(o["flags"][1]) == 0
    _yolo_compare(o, 0, de.yolo_reference(head, 0.25))
    assert len(odet.box_filter(list(odet.yolo_decode(bad, 640, 480, de.YOLO_NAMES, de.YOLO_WANTED, 0.25)[0]),
                               640, 480)[1]) == 0
    assert int(o["count"][1]) == 0


def test_yolo_decode_edges_u8_and_nms():
    """u8 head (scale 2^-8, zero point 0): products 128 * 128 / 2^16 exactly on 0.25 and one quantization step either
    side, many tied top classes (256 levels over 80 classes); the quantized scores then go through NMS, where tied
    scores at n > 16 are common."""
    from deepdish_b200 import ops
    q, kinds = de.yolo_u8_edge_head(np.random.default_rng(36))
    head = odet.yolo_dequant(q, de.u8_scale(), 0)
    de.assert_yolo_coverage(head, kinds, 0.25, step=2.0 ** -16)
    out = ops.yolo_decode(torch.from_numpy(q[None]).cuda(), _mask(), 0.25, (640, 480), (640, 480), ncap=2048,
                          quant=(float(de.u8_scale()), 0))
    keep, nkeep = ops.nms(out["tlwh"], out["score"], out["count"], 0.6)
    o = {k: v.cpu().numpy() for k, v in out.items()}
    exp = de.yolo_reference(head, 0.25)
    _yolo_compare(o, 0, exp)
    ib, score = exp[0], exp[1]
    assert len(score) > 16 and len(np.unique(score)) < len(score)          # tied scores reach NMS
    assert list(keep[0, :nkeep[0]].cpu().numpy()) == odet.non_max_suppression(ib, 0.6, score)


@pytest.mark.parametrize("ncap,hot,lo,hi", [(2048, 0.07, 1100, 2000), (4096, 0.14, 2049, 4096)])
def test_yolo_crowd_decode_and_nms(ncap, hot, lo, hi):
    """Crowd heads (25200 anchors): 1100-2000 candidates after the box filter through yolo_decode(ncap=2048) and NMS with
    the same nmax, and more than 2048 candidates for the anchor-order pass at ncap = 4096 (decode only: NMS takes at most
    3049 candidates)."""
    from deepdish_b200 import ops
    from tests.test_gpu_detect import COCO
    rng = np.random.default_rng(38)
    head = synth_yolo_head(rng, 2, 25200, hot=hot)
    wanted = ["person", "bicycle", "car", "motorbike", "bus", "truck"]
    mask = torch.tensor([1 if n in wanted else 0 for n in COCO], dtype=torch.uint8, device="cuda")
    out = ops.yolo_decode(torch.from_numpy(head).cuda(), mask, 0.25, (640, 480), (640, 480), ncap=ncap)
    kn = ops.nms(out["tlwh"], out["score"], out["count"], 0.6) if ncap <= de.NMS_NMAX else None
    o = {k: v.cpu().numpy() for k, v in out.items()}
    assert int(o["flags"].sum()) == 0
    for f in range(2):
        tlwh, cls, score, anchor = odet.yolo_decode(head[f], 640, 480, COCO, wanted, 0.25)
        ib, kept = odet.box_filter(list(tlwh), 640, 480)
        assert lo <= len(kept) <= hi
        _yolo_compare(o, f, (ib.astype(float).reshape(-1, 4), score[kept], cls[kept], anchor[kept]))
        if kn is not None:
            keep, nkeep = kn[0].cpu().numpy(), kn[1].cpu().numpy()
            assert list(keep[f, :nkeep[f]]) == odet.non_max_suppression(ib, 0.6, score[kept])


def test_ssd_score_and_iou_edges():
    """Custom anchors whose decoded boxes are exact (raw box offsets 0, dyadic anchors): best class scores exactly 0.5
    (kept: >= confidence) and one ulp below (dropped); box pairs of different classes with an f32 IoU exactly 0.6
    (the op suppresses at >, so both stay) and just above it (the second is suppressed)."""
    from deepdish_b200 import ops
    ncls, na = 8, 64
    names = ["???", "person", "bicycle", "car", "c04", "c05", "c06", "c07"]
    wanted = ["person", "bicycle", "car"]
    anchors = np.zeros((na, 4), F32)
    for a in range(na):                                   # background anchors: small boxes on a grid
        anchors[a] = (0.0625 * (a // 8) + 0.03125, 0.0625 * (a % 8) + 0.03125, 0.03125, 0.03125)
    hot = [(0.375, 0.375, 0.25, 0.25, 1, 0.9),            # (yc, xc, h, w, class column, score)
           (0.375, 0.4375, 0.25, 0.25, 3, 0.8),           # shifted by 1/16: IoU with the first exactly 0.6f
           (0.75, 0.375, 0.125, 0.25, 1, 0.85),
           (0.75, 0.4375 - 2.0 ** -10, 0.125, 0.25, 3, 0.75),      # IoU with the third just above 0.6f
           (0.125, 0.75, 0.125, 0.125, 2, 0.5),           # exactly on the confidence threshold
           (0.375, 0.875, 0.125, 0.125, 2, float(np.nextafter(F32(0.5), F32(0))))]   # one ulp below it
    slots = [9 * k + 2 for k in range(len(hot))]
    sc = np.full((2, na, ncls), 0.01, F32)
    for k, (yc, xc, h, w, c, s) in enumerate(hot):
        anchors[slots[k]] = (yc, xc, h, w)
        sc[:, slots[k], c] = F32(s)
    sc[1, slots[0], 1], sc[1, slots[1], 3] = F32(0.8), F32(0.9)     # frame 1: the other box of the 0.6f pair picks first
    rb = np.zeros((2, na, 4), F32)
    dec = np.stack([anchors[:, 0] - anchors[:, 2] / 2, anchors[:, 1] - anchors[:, 3] / 2,
                    anchors[:, 0] + anchors[:, 2] / 2, anchors[:, 1] + anchors[:, 3] / 2], 1).astype(F32)
    assert odet._iou_f32(dec[slots[0]], dec[slots[1]]) == F32(0.6)
    assert odet._iou_f32(dec[slots[2]], dec[slots[3]]) > F32(0.6)
    best = sc[:, :, 1:].max(axis=2)
    assert (best == F32(0.5)).sum() >= 2 and (best == np.nextafter(F32(0.5), F32(0))).sum() >= 2
    c2l = np.array([(c + 1) if names[c + 1] in wanted else -1 for c in range(ncls - 1)], np.int32)
    out = ops.ssd_decode(torch.from_numpy(rb).cuda(), torch.from_numpy(sc).cuda(), torch.from_numpy(anchors).cuda(),
                         torch.from_numpy(c2l).cuda(), 0.5, 0.5, (640, 480), (640, 480))
    o = {k: v.cpu().numpy() for k, v in out.items()}
    for b in range(2):
        ob, oc, os_, _ = odet.tflite_detection_postprocess(rb[b], sc[b], anchors)
        tlwh, labels, scores = odet.ssd_postprocess(ob, oc, os_, 640, 480, names, wanted)
        ib, kept = odet.box_filter([tuple(r) for r in tlwh], 640, 480)
        n = int(o["count"][b])
        assert n == len(kept) == 4, (b, n)
        np.testing.assert_array_equal(o["score"][b, :n], scores[kept])
        assert list(o["label"][b, :n]) == [names.index(labels[i]) for i in kept]
        np.testing.assert_array_equal(o["tlwh"][b, :n], ib.astype(float).reshape(-1, 4))


def test_tflite_adapter_score_edges():
    """Op scores exactly on the adapter's threshold (kept: >=) and one ulp below (dropped), at 0.5 and at the
    non-dyadic 0.3 (both sides round it to the same f32), with tied scores (stable order)."""
    from deepdish_b200 import ops
    rng = np.random.default_rng(39)
    names = ["person", "bicycle", "car", "dog", "cat"]
    wanted = ["person", "car", "cat"]
    b, n = 4, 16
    yx = np.sort(rng.uniform(0, 1, (b, n, 2, 2)), axis=3)                # per box: sorted (y0, y1), (x0, x1)
    boxes = np.stack([yx[..., 0, 0], yx[..., 1, 0], yx[..., 0, 1], yx[..., 1, 1]], -1).astype(F32)
    classes = rng.integers(0, len(names), (b, n)).astype(F32)
    count = np.array([16, 12, 16, 9], np.int32)
    ok = torch.ones(len(names), dtype=torch.uint8, device="cuda")
    wm = torch.tensor([1 if x in wanted else 0 for x in names], dtype=torch.uint8, device="cuda")
    on_thr = 0
    for thr in (0.5, 0.3):
        t = F32(thr)
        scores = rng.choice(np.array([0.2, 0.45, 0.6, 0.9], F32), (b, n))
        scores[:, 0:3] = t
        scores[:, 3:5] = np.nextafter(t, F32(0))
        scores[:, 5] = np.nextafter(t, F32(1))
        assert (scores == t).sum() >= 8
        out = ops.tflite_postprocess(*(torch.from_numpy(x).cuda() for x in (boxes, classes, scores, count)), ok, wm,
                                     thr, (640, 480))
        o = {k: v.cpu().numpy() for k, v in out.items()}
        for f in range(b):
            eb, el, es = odet.tflite_adapter_postprocess(boxes[f], classes[f], scores[f], count[f], 640, 480, names,
                                                         wanted, thr)
            k = int(o["count"][f])
            assert k == len(el), (thr, f)
            on_thr += sum(1 for s in es if s == t)
            np.testing.assert_array_equal(o["tlwh"][f, :k], np.array(eb, float).reshape(-1, 4))
            assert [names[i] for i in o["label"][f, :k]] == el
            np.testing.assert_array_equal(o["score"][f, :k], np.array(es, F32))
    assert on_thr >= 2


def test_yolo3_threshold_and_iou_edges():
    """Keras YOLOv3 adapter: a class probability exactly equal to the score threshold (zeroed: decode_netout keeps
    `> thr`) and an nms_thresh equal to the IoU of a returned pair at which the reference's `>=` decides the output;
    the next larger nms_thresh too."""
    from deepdish_b200 import ops
    maps, thr = de.yolo3_edge_maps(np.random.default_rng(37))
    assert (de.yolo3_probabilities(maps) == F32(thr)).sum() >= 2
    v = de.yolo3_exact_iou(maps, thr)
    wm = torch.tensor([1 if n in de.Y3_WANTED else 0 for n in de.Y3_NAMES], dtype=torch.uint8, device="cuda")
    dev = [torch.from_numpy(m[None].copy()).cuda() for m in maps]
    for nms in (v, float(np.nextafter(v, 1.0))):
        out = ops.yolo3_decode(dev, de.Y3_ANCHORS, wm, thr, nms, (640, 480), (de.Y3_NET, de.Y3_NET))
        o = {k: x.cpu().numpy() for k, x in out.items()}
        eb, el, es = de.yolo3_reference(maps, thr, nms)
        k = int(o["count"][0])
        assert int(o["flags"][0]) == 0 and k == len(el)
        np.testing.assert_array_equal(o["box"][0, :k], eb.astype(float))
        np.testing.assert_array_equal(o["label"][0, :k], el)
        np.testing.assert_array_equal(o["score"][0, :k].view(np.uint32), es.view(np.uint32))


def test_detector_wrappers_reject_bad_inputs():
    """The five detector wrappers read their inputs as dense arrays of one dtype: a slice, another dtype, another
    shape or a host tensor is refused instead of being misread."""
    from deepdish_b200 import ops
    cuda = dict(device="cuda")
    boxes = torch.zeros((2, 8, 4), dtype=torch.float64, **cuda)
    scores = torch.zeros((2, 8), dtype=torch.float32, **cuda)
    counts = torch.full((2,), 8, dtype=torch.int32, **cuda)
    wide = torch.zeros((2, 8, 6), dtype=torch.float64, **cuda)
    for args in ((wide[:, :, :4], scores, counts), (boxes.float(), scores, counts), (boxes, scores.double(), counts),
                 (boxes, scores[:, :4], counts), (boxes, scores, counts.long()), (boxes, scores, counts.cpu()),
                 (boxes.transpose(0, 1).contiguous().transpose(0, 1), scores, counts)):
        with pytest.raises(ValueError):
            ops.nms(*args, 0.6)
    with pytest.raises(ValueError):
        ops.nms(boxes, scores, counts, 0.6, out=(torch.zeros((2, 4), dtype=torch.int32, **cuda), counts.clone()))
    with pytest.raises(ValueError):
        ops.box_filter(wide[:, :, :4])
    with pytest.raises(ValueError):
        ops.box_filter(boxes.float())
    with pytest.raises(ValueError):
        ops.box_filter(boxes, counts.long())
    head = torch.zeros((2, 64, 85), dtype=torch.float32, **cuda)
    mask = torch.ones(80, dtype=torch.uint8, **cuda)
    for h, m in ((head.double(), mask), (head[:, ::2], mask), (head, mask[:40]), (head, mask.bool()),
                 (head.to(torch.int8), mask)):
        with pytest.raises(ValueError):
            ops.yolo_decode(h, m)
    with pytest.raises(ValueError):
        ops.yolo_decode(head, mask, ncap=32, out=ops.yolo_decode(head, mask, ncap=16))
    rb = torch.zeros((2, 64, 4), dtype=torch.float32, **cuda)
    rs = torch.zeros((2, 64, 8), dtype=torch.float32, **cuda)
    an = torch.zeros((64, 4), dtype=torch.float32, **cuda)
    c2l = torch.zeros(7, dtype=torch.int32, **cuda)
    for args in ((rb.double(), rs, an, c2l), (rb, rs[:, :32], an, c2l), (rb, rs, an[:32], c2l), (rb, rs, an, c2l[:6]),
                 (rb, rs, an.t().contiguous().t(), c2l), (rb, rs, an, c2l.cpu())):
        with pytest.raises(ValueError):
            ops.ssd_decode(*args)
    ob = torch.zeros((2, 10, 4), dtype=torch.float32, **cuda)
    oc = torch.zeros((2, 10), dtype=torch.float32, **cuda)
    cnt = torch.full((2,), 10, dtype=torch.int32, **cuda)
    ok = torch.ones(5, dtype=torch.uint8, **cuda)
    for args in ((ob.double(), oc, oc, cnt, ok, ok), (ob, oc.int(), oc, cnt, ok, ok), (ob, oc, oc[:, :5], cnt, ok, ok),
                 (ob, oc, oc, cnt.long(), ok, ok), (ob, oc, oc, cnt, ok, ok[:3]), (ob[:, ::2], oc, oc, cnt, ok, ok)):
        with pytest.raises(ValueError):
            ops.tflite_postprocess(*args)
