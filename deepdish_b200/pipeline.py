"""Detector heads -> NMS -> tracker, batched over streams, all on the device.

The batched counterpart of the reference's per-camera chain ``detect_objects`` (detector adapter +
box filter, deepdish.py:935-960) -> ``encode_features`` (NMS, deepdish.py:995-998; Detection list,
:1014) -> ``track_objects`` (:1028-1029) -> ``process_results`` counting (:1041-1112).  The CNNs
themselves (detector body, re-ID encoder) are out of scope: the pipeline consumes raw detector heads
and a caller-supplied feature provider.

A pipeline owns one BatchedTracker and a list of front-ends, each decoding the heads of a contiguous
range of streams (YOLOv5 or SSD-MobileNet) straight into the tracker's padded detection batch.
"""
import ctypes

import torch

from . import _lib, ops


class _FrontEnd:
    def __init__(self, lo, hi, class_names, wanted_labels, tracker_labels, ncap, frame_size, img_size,
                 nms_max_overlap):
        self.lo, self.hi = lo, hi
        self.ncap, self.frame_size, self.img_size = ncap, frame_size, img_size
        self.nms_max_overlap = nms_max_overlap
        self.class_names = list(class_names)
        self.wanted = set(wanted_labels)
        self.tracker_labels = list(tracker_labels)

    def _label_map(self, names, device):
        m = [self.tracker_labels.index(n) if (n in self.wanted and n in self.tracker_labels) else -1 for n in names]
        return torch.tensor(m, dtype=torch.int32, device=device)


class YoloFrontEnd(_FrontEnd):
    """tools/yolov5.py:115-146 + deepdish.py:946-955 + preprocessing.non_max_suppression."""

    def __init__(self, lo, hi, class_names, wanted_labels, tracker_labels, score_threshold=0.25, ncap=1024,
                 frame_size=(640, 480), img_size=None, nms_max_overlap=0.6, quant=None, device="cuda"):
        super().__init__(lo, hi, class_names, wanted_labels, tracker_labels, ncap, frame_size,
                         img_size or frame_size, nms_max_overlap)
        self.thr, self.quant = score_threshold, quant
        self.mask = torch.tensor([1 if n in self.wanted else 0 for n in self.class_names], dtype=torch.uint8,
                                 device=device)
        self.map = self._label_map(self.class_names, device)

    def candidates(self, head):
        self._out = out = ops.yolo_decode(head, self.mask, self.thr, self.img_size, self.frame_size, self.ncap,
                                          self.quant, out=getattr(self, "_out", None))
        return out["tlwh"], out["score"], out["cls"], out["count"], out["flags"]


class SsdFrontEnd(_FrontEnd):
    """TFLite_Detection_PostProcess (restated) + tools/ssd_mobilenet.py:59-150,198-213 + deepdish.py:946-955 +
    preprocessing.non_max_suppression.  label_names = the detector's label file (labels[c+1] is class c)."""

    def __init__(self, lo, hi, label_names, wanted_labels, tracker_labels, anchors, score_threshold=0.5,
                 iou_threshold=0.5, ncap=16, frame_size=(640, 480), img_size=None, nms_max_overlap=0.6, device="cuda"):
        super().__init__(lo, hi, label_names, wanted_labels, tracker_labels, ncap, frame_size,
                         img_size or frame_size, nms_max_overlap)
        self.thr, self.iou = score_threshold, iou_threshold
        self.anchors = anchors.to(device).contiguous()
        n = len(self.class_names)
        # class c of the op -> label id c+1 of the label file when that name is wanted, else -1
        c2l = [(c + 1) if (c + 1 < n and self.class_names[c + 1] in self.wanted) else -1 for c in range(n - 1)]
        self.c2l = torch.tensor(c2l, dtype=torch.int32, device=device)
        self.map = self._label_map(self.class_names, device)

    def candidates(self, heads):
        raw_boxes, raw_scores = heads
        self._out = out = ops.ssd_decode(raw_boxes, raw_scores, self.anchors, self.c2l, self.thr, self.iou,
                                         self.img_size, self.frame_size, self.ncap, out=getattr(self, "_out", None))
        return out["tlwh"], out["score"], out["label"], out["count"], out["flags"]


class DetectTrackPipeline:
    def __init__(self, tracker, frontends):
        self.bt = tracker
        self.frontends = list(frontends)
        S, D = tracker.n_streams, tracker.max_dets
        dev = tracker.device
        self.det_tlwh = torch.zeros((S, D, 4), dtype=torch.float64, device=dev)
        self.det_conf = torch.zeros((S, D), dtype=torch.float32, device=dev)
        self.det_label = torch.zeros((S, D), dtype=torch.int32, device=dev)
        self.det_count = torch.zeros((S,), dtype=torch.int32, device=dev)
        self.flags = torch.zeros((S,), dtype=torch.int32, device=dev)
        self.lib = _lib.lib()

    def detect(self, heads):
        """heads: one entry per front-end (YOLO: head tensor [n,na,5+nc]; SSD: (raw_boxes, raw_scores)).
        Fills the padded detection batch (boxes, confidences, labels, counts) in NMS pick order."""
        D = self.bt.max_dets
        st = ctypes.c_void_p(torch.cuda.current_stream(self.bt.device).cuda_stream)
        self.flags.zero_()
        for fe, h in zip(self.frontends, heads):
            tlwh, score, label, count, flags = fe.candidates(h)
            fe._keep = ops.nms(tlwh, score, count, fe.nms_max_overlap, out=getattr(fe, "_keep", None))
            keep, nkeep = fe._keep
            self.flags[fe.lo:fe.hi] |= flags
            n = fe.hi - fe.lo
            _lib.check(self.lib.dd_gather_detections(
                tlwh.data_ptr(), score.data_ptr(), label.data_ptr(), fe.map.data_ptr(), fe.map.numel(), fe.ncap,
                keep.data_ptr(), nkeep.data_ptr(), keep.shape[1], n, D,
                self.det_tlwh.data_ptr() + fe.lo * D * 32, self.det_conf.data_ptr() + fe.lo * D * 4,
                self.det_label.data_ptr() + fe.lo * D * 4, self.det_count.data_ptr() + fe.lo * 4,
                self.flags.data_ptr() + fe.lo * 4, st), "dd_gather_detections")
        return self.det_tlwh, self.det_conf, self.det_label, self.det_count

    def step(self, heads, features, join=True, present=None):
        """detect() + one tracker tick.  features: f32 [S,Dmax,128] tensor or callable(tlwh, count) -> tensor
        (the re-ID encoder's output for the kept boxes, in the same order).  present: frame presence of each stream
        (BatchedTracker.step): the tick leaves the streams without a frame untouched."""
        tlwh, conf, label, count = self.detect(heads)
        feat = features(tlwh, count) if callable(features) else features

        class _B:
            pass
        b = _B()
        b.tlwh, b.conf, b.label, b.feat, b.count = tlwh, conf, label, feat, count
        return self.bt.step(b, join=join, reduce=True, present=present)

    def check(self):
        if int(self.flags.max()) & _lib.FLAG_DET_OVERFLOW:
            raise RuntimeError("detection capacity exceeded in the detector front-end / gather")
        self.bt.check()
