"""GPU parity of the detector post-processing at larger sizes than the fixtures: YOLOv5 head decode
(f32 and u8), NMS at up to 1024 candidates, SSD-MobileNet decode; checked against the oracle."""
import numpy as np
import pytest
import torch

from oracle import detect as odet
from oracle.make_golden import synth_yolo_head

pytestmark = pytest.mark.gpu

COCO = [l.strip() for l in """person bicycle car motorbike aeroplane bus train truck boat trafficlight firehydrant
stopsign parkingmeter bench bird cat dog horse sheep cow elephant bear zebra giraffe backpack umbrella handbag tie
suitcase frisbee skis snowboard sportsball kite baseballbat baseballglove skateboard surfboard tennisracket bottle
wineglass cup fork knife spoon bowl banana apple sandwich orange broccoli carrot hotdog pizza donut cake chair sofa
pottedplant bed diningtable toilet tvmonitor laptop mouse remote keyboard cellphone microwave oven toaster sink
refrigerator book clock vase scissors teddybear hairdrier toothbrush""".split()]


def test_yolo_full_head_f32_and_nms():
    """25200 x 85 head (BASELINE config 1 shape, 4 frames): decode + filter + NMS keep-lists bit-exact."""
    from deepdish_b200 import ops
    assert len(COCO) == 80
    rng = np.random.default_rng(11)
    head = synth_yolo_head(rng, 4, 25200, hot=0.01)
    wanted = ["person", "bicycle", "car", "motorbike", "bus", "truck"]
    mask = torch.tensor([1 if n in wanted else 0 for n in COCO], dtype=torch.uint8, device="cuda")
    out = ops.yolo_decode(torch.from_numpy(head).cuda(), mask, 0.25, (640, 480), (640, 480), ncap=1024)
    keep, nkeep = ops.nms(out["tlwh"], out["score"], out["count"], 0.6)
    o = {k: v.cpu().numpy() for k, v in out.items()}
    keep, nkeep = keep.cpu().numpy(), nkeep.cpu().numpy()
    assert int(o["flags"].sum()) == 0
    for f in range(4):
        tlwh, cls, score, anchor = odet.yolo_decode(head[f], 640, 480, COCO, wanted, 0.25)
        ib, kept = odet.box_filter(list(tlwh), 640, 480)
        n = int(o["count"][f])
        assert n == len(kept) and n > 50
        np.testing.assert_array_equal(o["tlwh"][f, :n], ib.astype(np.float64))
        np.testing.assert_array_equal(o["score"][f, :n], score[kept])
        np.testing.assert_array_equal(o["cls"][f, :n], cls[kept])
        np.testing.assert_array_equal(o["anchor"][f, :n], anchor[kept])
        exp_keep = odet.non_max_suppression(ib, 0.6, score[kept])
        assert list(keep[f, :nkeep[f]]) == exp_keep


def test_yolo_u8_head_and_overflow_flag():
    from deepdish_b200 import ops, _lib
    rng = np.random.default_rng(12)
    q = rng.integers(0, 256, (2, 2000, 85), dtype=np.uint8)
    q[..., 4] = (q[..., 4] * 0.4).astype(np.uint8)
    scale, zp = 1.0 / 255, 3
    wanted = COCO[:10]
    mask = torch.tensor([1 if n in wanted else 0 for n in COCO], dtype=torch.uint8, device="cuda")
    out = ops.yolo_decode(torch.from_numpy(q).cuda(), mask, 0.25, (640, 480), (640, 480), ncap=2048, quant=(scale, zp))
    o = {k: v.cpu().numpy() for k, v in out.items()}
    for f in range(2):
        head = odet.yolo_dequant(q[f], np.float32(scale), zp)
        tlwh, cls, score, anchor = odet.yolo_decode(head, 640, 480, COCO, wanted, 0.25)
        ib, kept = odet.box_filter(list(tlwh), 640, 480)
        n = int(o["count"][f])
        assert n == len(kept) and n > 20
        np.testing.assert_array_equal(o["tlwh"][f, :n], ib.astype(np.float64))
        np.testing.assert_array_equal(o["score"][f, :n], score[kept])
        np.testing.assert_array_equal(o["cls"][f, :n], cls[kept])          # u8 ties for the top class: first one wins
        np.testing.assert_array_equal(o["anchor"][f, :n], anchor[kept])
    small = ops.yolo_decode(torch.from_numpy(q).cuda(), mask, 0.25, (640, 480), (640, 480), ncap=8, quant=(scale, zp))
    assert int(small["flags"].cpu()[0]) & _lib.FLAG_DET_OVERFLOW          # never silently truncated


def test_nms_1024_candidates_and_empty():
    from deepdish_b200 import ops
    rng = np.random.default_rng(13)
    B, N = 6, 1024
    counts = np.array([1024, 1000, 513, 64, 1, 0], np.int32)
    boxes = np.zeros((B, N, 4)); scores = np.zeros((B, N), np.float32)
    for b in range(B):
        n = counts[b]
        k = max(1, n // 6)
        cx, cy = rng.uniform(30, 600, k), rng.uniform(30, 440, k)
        p = rng.integers(0, k, n)
        boxes[b, :n] = np.stack([np.clip(cx[p] + rng.normal(0, 8, n), 0, 630).astype(int),
                                 np.clip(cy[p] + rng.normal(0, 8, n), 0, 470).astype(int),
                                 rng.integers(10, 60, n), rng.integers(20, 120, n)], 1)
        scores[b, :n] = (0.25 + 0.75 * (rng.permutation(n) + rng.uniform(0.1, 0.9, n)) / max(n, 1)).astype(np.float32)
    keep, nkeep = ops.nms(ops._dev(boxes, torch.float64), ops._dev(scores, torch.float32), ops._dev(counts, torch.int32), 0.6)
    keep, nkeep = keep.cpu().numpy(), nkeep.cpu().numpy()
    for b in range(B):
        n = counts[b]
        exp = odet.non_max_suppression(boxes[b, :n].astype(np.int64), 0.6, scores[b, :n])
        assert list(keep[b, :nkeep[b]]) == exp


def test_ssd_decode_vs_oracle():
    """1917 anchors x 91 classes.  The anchor decode is a third-party TFLite op (parity unpinned): the
    oracle restates it; expf may differ from numpy's exp by an ulp, so a frame may differ by one pixel."""
    from deepdish_b200 import ops
    rng = np.random.default_rng(14)
    B, A, C = 48, 1917, 91
    anchors = odet.ssd_anchors()
    rb = rng.normal(0, 0.8, (B, A, 4)).astype(np.float32)
    sc = (rng.beta(0.4, 12, (B, A, C))).astype(np.float32)
    names = ["???"] + ["c%02d" % i for i in range(1, C)]
    names[1], names[2], names[3], names[4], names[6] = "person", "bicycle", "car", "motorcycle", "bus"
    wanted = ["person", "bicycle", "car", "motorcycle", "bus"]
    for b in range(B):                          # a few confident, clustered anchors per frame
        hot = rng.choice(A, 24, replace=False)
        sc[b, hot, 1 + rng.choice([0, 1, 2, 3, 5, 7], 24)] = rng.uniform(0.4, 1.0, 24).astype(np.float32)
    c2l = np.array([(c + 1) if names[c + 1] in wanted else -1 for c in range(C - 1)], np.int32)
    out = ops.ssd_decode(torch.from_numpy(rb).cuda(), torch.from_numpy(sc).cuda(), torch.from_numpy(anchors).cuda(),
                         torch.from_numpy(c2l).cuda(), 0.5, 0.5, (640, 480), (640, 480))
    o = {k: v.cpu().numpy() for k, v in out.items()}
    total = 0
    for b in range(B):
        ob, oc, os_, _ = odet.tflite_detection_postprocess(rb[b], sc[b], anchors)
        tlwh, labels, scores = odet.ssd_postprocess(ob, oc, os_, 640, 480, names, wanted)
        ib, kept = odet.box_filter([tuple(r) for r in tlwh], 640, 480)
        n = int(o["count"][b])
        assert n == len(kept), b
        np.testing.assert_array_equal(o["score"][b, :n], scores[kept])
        assert list(o["label"][b, :n]) == [names.index(labels[i]) for i in kept]
        np.testing.assert_array_equal(o["tlwh"][b, :n], ib.astype(float).reshape(-1, 4))     # bit-exact boxes
        total += n
    assert total > 100


def test_tflite_adapter_golden_batched_and_facade():
    """TFLITE adapter (tools/tflite.py + tflite_object_detector._postprocess) against the reference's own outputs."""
    from deepdish_b200.tools.tflite import TFLITE, ObjectDetectorOptions
    from tests import goldens
    g = goldens.load("tflite_adapter.npz")
    names, wanted = list(g["names"]), list(g["wanted"])
    total = 0
    for c in range(len(g["count"])):
        thr, maxr, use_deny, use_allow = g["opts"][c]
        opt = ObjectDetectorOptions(score_threshold=float(thr), max_results=int(maxr),
                                    label_deny_list=list(g["deny"]) if use_deny else None,
                                    label_allow_list=list(g["allow"]) if use_allow else None)
        ad = TFLITE(wanted_labels=wanted, label_list=names, options=opt,
                    outputs_fn=lambda img, c=c: (g["op_boxes"][c], g["op_classes"][c], g["op_scores"][c], g["count"][c]))
        boxes, labels, scores = ad.detect_image(np.zeros((480, 640, 3), np.uint8))
        np.testing.assert_array_equal(np.array(boxes, np.int64).reshape(-1, 4), g["tlwh%d" % c])
        assert [names.index(l) for l in labels] == list(g["lab%d" % c])
        np.testing.assert_array_equal(np.array(scores, np.float32), g["score%d" % c])
        total += len(labels)
    assert total > 100
    # batched call: every third case shares the same options
    ad = TFLITE(wanted_labels=wanted, label_list=names, options=ObjectDetectorOptions(score_threshold=0.5))
    sel = [c for c in range(len(g["count"])) if tuple(g["opts"][c]) == (0.5, -1.0, 0.0, 0.0)]
    res = ad.detect_outputs(g["op_boxes"][sel], g["op_classes"][sel], g["op_scores"][sel], g["count"][sel], (640, 480))
    for c, (boxes, labels, scores) in zip(sel, res):
        np.testing.assert_array_equal(np.array(boxes, np.int64).reshape(-1, 4), g["tlwh%d" % c])
    assert len(sel) >= 4
