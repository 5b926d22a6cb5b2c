"""numpy driver for the host emulation of the kernel bodies.  TEST SCAFFOLDING (see dd_hostemu.cpp)."""
import ctypes

import numpy as np

from deepdish_b200 import _lib as L
from . import build as _build

_emu = None


def emu():
    global _emu
    if _emu is None:
        _emu = ctypes.CDLL(_build.build())
    return _emu


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class HostEmuTracker:
    """Same call sequence as deepdish_b200.batched.BatchedTracker, on host memory."""

    def __init__(self, cfg, line=(320.0, 0.0, 320.0, 480.0)):
        self.cfg = cfg
        # gallery page pool in host memory: one segment that covers the worst case (every slot's table full)
        need = cfg.n_streams * cfg.max_tracks * L.page_cap(cfg)
        seg = 1
        while seg < need:
            seg <<= 1
        cfg.seg_pages, cfg.n_segs = seg, 1
        self.pool_f32 = np.zeros(seg * L.PAGE_F32_BYTES, dtype=np.uint8)
        self.pool_f16 = np.zeros(seg * L.PAGE_F16_BYTES, dtype=np.uint8)
        cfg.pool_f32[0], cfg.pool_f16[0] = self.pool_f32.ctypes.data, self.pool_f16.ctypes.data
        self.lay = L.TrackerLayout()
        assert emu().ddh_tracker_layout_query(ctypes.byref(cfg), ctypes.byref(self.lay)) == 0
        self.blob = np.zeros(self.lay.total_bytes, dtype=np.uint8)
        self.v = {}
        for name, (dt, shape) in L.field_specs(cfg).items():
            off = getattr(self.lay, name)
            n = int(np.prod(shape)) * np.dtype(dt).itemsize
            self.v[name] = self.blob[off:off + n].view(dt).reshape(shape)
        assert emu().ddh_tracker_init(_p(self.blob), ctypes.byref(cfg)) == 0
        self.line = np.asarray(line, dtype=np.float64)
        self.det_track_id = np.zeros((cfg.n_streams, cfg.max_dets), dtype=np.int32)

    def predict(self):
        assert emu().ddh_tracker_predict(_p(self.blob), ctypes.byref(self.cfg)) == 0

    def update(self, tlwh, conf, label, feat, count):
        self._keep = [np.ascontiguousarray(tlwh, np.float64), np.ascontiguousarray(conf, np.float32),
                      np.ascontiguousarray(label, np.int32), np.ascontiguousarray(feat, np.float32),
                      np.ascontiguousarray(count, np.int32)]
        a = self._keep
        rc = emu().ddh_tracker_update(_p(self.blob), ctypes.byref(self.cfg), _p(a[0]), _p(a[1]), _p(a[2]),
                                      _p(a[3]), _p(a[4]), _p(self.det_track_id))
        assert rc == 0
        return self.det_track_id

    def gallery(self, s, slot):
        n = int(self.v["gal_len"][s, slot])
        out = np.zeros((max(n, 1), 128), dtype=np.float32)
        got = emu().ddh_gallery_read(_p(self.blob), ctypes.byref(self.cfg), int(s), int(slot), _p(out), n)
        assert got == n
        return out[:n]

    def countline(self):
        assert emu().ddh_tracker_countline(_p(self.blob), ctypes.byref(self.cfg), _p(self.line), 0) == 0


def lsap(cost):
    cost = np.ascontiguousarray(cost, np.float64)
    nr, nc = cost.shape
    out = np.full(nr, -1, dtype=np.int32)
    rc = emu().ddh_lsap(_p(cost), nr, nc, _p(out))
    return rc, out


def set_difference_order(a, m):
    a = np.ascontiguousarray(a, np.int32)
    m = np.ascontiguousarray(m, np.int32)
    out = np.zeros(max(len(a), 1), dtype=np.int32)
    n = emu().ddh_set_difference_order(_p(a), len(a), _p(m), len(m), _p(out))
    return out[:n].tolist()


def intersection(segs):
    segs = np.ascontiguousarray(segs, np.float64).reshape(-1, 8)
    out = np.zeros(len(segs), dtype=np.int32)
    emu().ddh_intersection(_p(segs), len(segs), _p(out))
    return out


def ssd_post(sel_box, sel_cls, sel_score, class_to_label, conf_thr=0.5, nms_iou=0.5, img=(640, 480), frame=(640, 480)):
    sel_box = np.ascontiguousarray(sel_box, np.float32).reshape(-1, 4)
    n = len(sel_box)
    sel_cls = np.ascontiguousarray(sel_cls, np.int32)
    sel_score = np.ascontiguousarray(sel_score, np.float32)
    c2l = np.ascontiguousarray(class_to_label, np.int32)
    tl = np.zeros((16, 4)); sc = np.zeros(16, np.float32); lb = np.zeros(16, np.int32)
    emu().ddh_ssd_post.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_float, ctypes.c_double] + [ctypes.c_int] * 4 + [ctypes.c_void_p] * 3
    k = emu().ddh_ssd_post(_p(sel_box), _p(sel_cls), _p(sel_score), n, _p(c2l), conf_thr, nms_iou, img[0], img[1],
                           frame[0], frame[1], _p(tl), _p(sc), _p(lb))
    return tl[:k], sc[:k], lb[:k]


def yolo3(maps, anchors, nc, wanted_mask, thr, image, net, ncap=256, nms_thresh=0.5):
    m = [np.ascontiguousarray(x, np.float32) for x in maps]
    grids = np.array([x.shape[0] for x in m], np.int32)
    anch = np.ascontiguousarray(anchors, np.int32).reshape(-1)
    wm = np.ascontiguousarray(wanted_mask, np.uint8)
    box = np.zeros((ncap, 4)); sc = np.zeros(ncap, np.float32); lb = np.zeros(ncap, np.int32); fl = np.zeros(1, np.int32)
    emu().ddh_yolo3.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int, ctypes.c_void_p, ctypes.c_float, ctypes.c_double] + \
        [ctypes.c_int] * 5 + [ctypes.c_void_p] * 4
    k = emu().ddh_yolo3(_p(m[0]), _p(m[1]), _p(m[2]), _p(grids), _p(anch), nc, _p(wm), thr, nms_thresh, image[0], image[1],
                        net[0], net[1], ncap, _p(box), _p(sc), _p(lb), _p(fl))
    return box[:k], sc[:k], lb[:k], int(fl[0])


def box_filter(boxes, frame=(640, 480)):
    boxes = np.ascontiguousarray(boxes, np.float64).reshape(-1, 4)
    n = len(boxes)
    out = np.zeros((max(n, 1), 4)); idx = np.zeros(max(n, 1), np.int32)
    k = emu().ddh_box_filter(_p(boxes), n, frame[0], frame[1], _p(out), _p(idx))
    return out[:k], idx[:k]


def nms(boxes, scores, max_overlap):
    boxes = np.ascontiguousarray(boxes, np.float64).reshape(-1, 4)
    scores = np.ascontiguousarray(scores, np.float32)
    keep = np.zeros(max(len(boxes), 1), np.int32)
    emu().ddh_nms.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_void_p]
    k = emu().ddh_nms(_p(boxes), _p(scores), len(boxes), max_overlap, _p(keep))
    return keep[:k].tolist()


def yolo_rows(head, wanted_mask, thr, img, frame):
    head = np.ascontiguousarray(head, np.float32)
    na, rw = head.shape
    wanted_mask = np.ascontiguousarray(wanted_mask, np.uint8)
    tl = np.zeros((na, 4)); sc = np.zeros(na, np.float32); cl = np.zeros(na, np.int32); an = np.zeros(na, np.int32)
    nan = np.zeros(1, np.int32)
    emu().ddh_yolo_rows.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_float] + \
        [ctypes.c_int] * 4 + [ctypes.c_void_p] * 5
    k = emu().ddh_yolo_rows(_p(head), na, rw - 5, _p(wanted_mask), thr, img[0], img[1], frame[0], frame[1],
                            _p(tl), _p(sc), _p(cl), _p(an), _p(nan))
    return tl[:k], sc[:k], cl[:k], an[:k], int(nan[0])
