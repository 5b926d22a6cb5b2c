"""Thin torch wrappers over the stand-alone C-ABI operators (device tensors in, device tensors out).

These are what the per-function ``deep_sort`` mirror (deepdish_b200/deep_sort/*.py) and the detector
adapters call.  Every function launches on the current CUDA stream of the tensors' device and returns
without synchronising.  No CPU implementation exists behind any of them.
"""
import ctypes

import numpy as np
import torch

from . import _lib


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _dev(x, dtype, device="cuda"):
    """Host array / tensor -> contiguous CUDA tensor of `dtype`."""
    if isinstance(x, torch.Tensor):
        t = x.to(device=device, dtype=dtype)
    else:
        t = torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).to(device)
    return t.contiguous()


def _need_cuda(t):
    if not t.is_cuda:
        raise RuntimeError("deepdish_b200 operators run on CUDA tensors only (no CPU fallback)")


def _arg(t, name, dtype, shape, device):
    """The kernels read `t` as a dense row-major array of `dtype` on `device`: anything else (a slice, a
    transposed view, another dtype or device, other extents) would be silently misread.  shape: ints, None = any."""
    if not isinstance(t, torch.Tensor):
        raise ValueError("%s must be a torch.Tensor" % name)
    dtypes = dtype if isinstance(dtype, tuple) else (dtype,)
    if t.dtype not in dtypes:
        raise ValueError("%s must be %s, got %s" % (name, " or ".join(str(d) for d in dtypes), t.dtype))
    if t.device != device:
        raise ValueError("%s must be on %s, got %s" % (name, device, t.device))
    if t.dim() != len(shape) or any(s is not None and s != n for s, n in zip(shape, t.shape)):
        raise ValueError("%s must have shape [%s], got %s" % (
            name, ",".join("*" if s is None else str(s) for s in shape), list(t.shape)))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return t


# ------------------------------------------------------------------------------------- Kalman
def kalman_initiate(xyah):
    """KalmanFilter.initiate (kalman_filter.py:55-86).  xyah f64 [n,4] -> mean [n,8], cov [n,8,8]."""
    _need_cuda(xyah)
    n = xyah.shape[0]
    mean = torch.empty((n, 8), dtype=torch.float64, device=xyah.device)
    cov = torch.empty((n, 8, 8), dtype=torch.float64, device=xyah.device)
    _lib.check(_lib.lib().dd_kalman_initiate(xyah.data_ptr(), mean.data_ptr(), cov.data_ptr(), n,
                                             _stream(xyah.device)), "dd_kalman_initiate")
    return mean, cov


def kalman_predict_(mean, cov):
    """KalmanFilter.predict (kalman_filter.py:88-123), in place."""
    _need_cuda(mean)
    _lib.check(_lib.lib().dd_kalman_predict(mean.data_ptr(), cov.data_ptr(), mean.shape[0],
                                            _stream(mean.device)), "dd_kalman_predict")
    return mean, cov


def kalman_project(mean, cov):
    """KalmanFilter.project (kalman_filter.py:125-152) -> pmean [n,4], pcov [n,4,4]."""
    _need_cuda(mean)
    n = mean.shape[0]
    pm = torch.empty((n, 4), dtype=torch.float64, device=mean.device)
    pc = torch.empty((n, 4, 4), dtype=torch.float64, device=mean.device)
    _lib.check(_lib.lib().dd_kalman_project(mean.data_ptr(), cov.data_ptr(), pm.data_ptr(), pc.data_ptr(), n,
                                            _stream(mean.device)), "dd_kalman_project")
    return pm, pc


def kalman_update_(mean, cov, xyah):
    """KalmanFilter.update (kalman_filter.py:154-186), in place, one measurement per row."""
    _need_cuda(mean)
    _lib.check(_lib.lib().dd_kalman_update(mean.data_ptr(), cov.data_ptr(), xyah.data_ptr(), mean.shape[0],
                                           _stream(mean.device)), "dd_kalman_update")
    return mean, cov


def kalman_gating_distance(mean, cov, xyah, only_position=False):
    """KalmanFilter.gating_distance (kalman_filter.py:188-229): n tracks x m measurements -> [n,m]."""
    _need_cuda(mean)
    n, m = mean.shape[0], xyah.shape[0]
    out = torch.empty((n, m), dtype=torch.float64, device=mean.device)
    _lib.check(_lib.lib().dd_kalman_gating_distance(mean.data_ptr(), cov.data_ptr(), xyah.data_ptr(), n, m,
                                                    1 if only_position else 0, out.data_ptr(),
                                                    _stream(mean.device)), "dd_kalman_gating_distance")
    return out


# ------------------------------------------------------------------------------------- metric / IoU
def nn_distance(gallery, offsets, feats, metric="cosine"):
    """NearestNeighborDistanceMetric.distance (nn_matching.py:156-177): gallery f32 [G,128] grouped by
    offsets i32 [n+1], feats f32 [m,128] -> f64 [n,m]."""
    _need_cuda(feats)
    n, m = offsets.shape[0] - 1, feats.shape[0]
    out = torch.zeros((n, m), dtype=torch.float64, device=feats.device)
    code = {"cosine": 0, "euclidean": 1}[metric]
    _lib.check(_lib.lib().dd_nn_distance(gallery.data_ptr() if gallery.numel() else None, offsets.data_ptr(),
                                         feats.data_ptr(), n, m, code, out.data_ptr(), _stream(feats.device)),
               "dd_nn_distance")
    return out


def iou_cost(track_tlwh, tsu, det_tlwh):
    """iou_matching.iou_cost (iou_matching.py:42-81) -> f64 [n,m]."""
    _need_cuda(track_tlwh)
    n, m = track_tlwh.shape[0], det_tlwh.shape[0]
    out = torch.zeros((n, m), dtype=torch.float64, device=track_tlwh.device)
    _lib.check(_lib.lib().dd_iou_cost(track_tlwh.data_ptr(), tsu.data_ptr(), det_tlwh.data_ptr(), n, m,
                                      out.data_ptr(), _stream(track_tlwh.device)), "dd_iou_cost")
    return out


# ------------------------------------------------------------------------------------- assignment
def lsap(cost):
    """scipy.optimize.linear_sum_assignment with scipy's tie-breaking (linear_assignment.py:58).
    cost f64 [b,nr,nc] -> col4row i32 [b,nr] (-1 = unassigned row), status i32 [b]."""
    _need_cuda(cost)
    b, nr, nc = cost.shape
    out = torch.full((b, nr), -1, dtype=torch.int32, device=cost.device)
    st = torch.zeros((b,), dtype=torch.int32, device=cost.device)
    _lib.check(_lib.lib().dd_lsap(cost.data_ptr(), b, nr, nc, out.data_ptr(), st.data_ptr(),
                                  _stream(cost.device)), "dd_lsap")
    return out, st


def linear_sum_assignment(cost):
    """Drop-in for scipy's function on ONE host matrix: returns (row_ind, col_ind) numpy arrays."""
    c = np.asarray(cost, dtype=np.float64)
    if c.ndim != 2:
        raise ValueError("expected a matrix (2-D array), got a %r array" % (c.shape,))
    if c.size == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    if np.isnan(c).any() or np.isneginf(c).any():
        raise ValueError("matrix contains invalid numeric entries")
    out, st = lsap(_dev(c[None], torch.float64))
    if int(st[0]) != 0:
        raise ValueError("cost matrix is infeasible")
    col = out[0].cpu().numpy().astype(np.int64)
    rows = np.nonzero(col >= 0)[0]
    return rows.astype(np.int64), col[rows]


def set_difference_order(a, na, m, nm):
    """CPython `list(set(a) - set(m))` iteration order for batches of small ints (device tensors)."""
    _need_cuda(a)
    b, na_max = a.shape
    out = torch.zeros((b, na_max), dtype=torch.int32, device=a.device)
    on = torch.zeros((b,), dtype=torch.int32, device=a.device)
    _lib.check(_lib.lib().dd_set_difference_order(a.data_ptr(), na.data_ptr(), na_max, m.data_ptr(), nm.data_ptr(),
                                                  m.shape[1], b, out.data_ptr(), on.data_ptr(),
                                                  _stream(a.device)), "dd_set_difference_order")
    return out, on


def segments_intersect(seg):
    """tools/intersection.py:4-24 for seg f64 [n,8] = (p, pr, q, qs) -> i32 [n]."""
    _need_cuda(seg)
    out = torch.zeros((seg.shape[0],), dtype=torch.int32, device=seg.device)
    _lib.check(_lib.lib().dd_intersection(seg.data_ptr(), seg.shape[0], out.data_ptr(), _stream(seg.device)),
               "dd_intersection")
    return out


# ------------------------------------------------------------------------------------- detection
def nms(boxes, scores, counts, max_overlap, out=None):
    """preprocessing.non_max_suppression for b frames (preprocessing.py:6-73).
    boxes f64 [b,nmax,4] tlwh, scores f32 [b,nmax], counts i32 [b] -> keep i32 [b,nmax], nkeep i32 [b].
    out = (keep, nkeep) reuses caller buffers (entries past nkeep are then left untouched)."""
    _need_cuda(boxes)
    dev = boxes.device
    _arg(boxes, "boxes", torch.float64, (None, None, 4), dev)
    b, nmax = boxes.shape[:2]
    _arg(scores, "scores", torch.float32, (b, nmax), dev)
    _arg(counts, "counts", torch.int32, (b,), dev)
    if out is None:
        keep = torch.full((b, nmax), -1, dtype=torch.int32, device=dev)
        nkeep = torch.zeros((b,), dtype=torch.int32, device=dev)
    else:
        keep, nkeep = out
        _arg(keep, "out keep", torch.int32, (b, nmax), dev)
        _arg(nkeep, "out nkeep", torch.int32, (b,), dev)
    _lib.check(_lib.lib().dd_nms(boxes.data_ptr(), scores.data_ptr(), counts.data_ptr(), b, nmax,
                                 float(max_overlap), keep.data_ptr(), nkeep.data_ptr(), _stream(boxes.device)),
               "dd_nms")
    return keep, nkeep


def box_filter(boxes, counts=None, frame_size=(640, 480)):
    """The pre-NMS box filter of Pipeline.detect_objects (deepdish.py:941-960) for b frames of float tlwh boxes.
    boxes f64 [b,nmax,4], counts i32 [b] or None -> (tlwh f64 [b,nmax,4] integer-valued, index i32 [b,nmax], count i32 [b])."""
    _need_cuda(boxes)
    _arg(boxes, "boxes", torch.float64, (None, None, 4), boxes.device)
    b, nmax = boxes.shape[:2]
    if counts is not None:
        _arg(counts, "counts", torch.int32, (b,), boxes.device)
    out = torch.zeros((b, nmax, 4), dtype=torch.float64, device=boxes.device)
    idx = torch.full((b, nmax), -1, dtype=torch.int32, device=boxes.device)
    cnt = torch.zeros((b,), dtype=torch.int32, device=boxes.device)
    _lib.check(_lib.lib().dd_box_filter(boxes.data_ptr(), counts.data_ptr() if counts is not None else None, b, nmax,
                                        int(frame_size[0]), int(frame_size[1]), out.data_ptr(), idx.data_ptr(),
                                        cnt.data_ptr(), _stream(boxes.device)), "dd_box_filter")
    return out, idx, cnt


def yolo_decode(head, wanted_mask, score_thr=0.25, img_size=(640, 480), frame_size=(640, 480), ncap=1024,
                quant=None, out=None):
    """YOLOv5 head decode + box filter for b frames (tools/yolov5.py:115-146, deepdish.py:946-955).
    head f32 [b,na,5+nc] (or u8 with quant=(scale, zero_point)); wanted_mask u8 [nc].
    Returns dict(tlwh f64 [b,ncap,4], score f32, cls i32, anchor i32, count i32 [b], flags i32 [b])."""
    _need_cuda(head)
    dev = head.device
    _arg(head, "head", (torch.float32, torch.uint8), (None, None, None), dev)
    b, na, rw = head.shape
    nc = rw - 5
    _arg(wanted_mask, "wanted_mask", torch.uint8, (nc,), dev)
    spec = dict(tlwh=(torch.float64, (b, ncap, 4)), score=(torch.float32, (b, ncap)), cls=(torch.int32, (b, ncap)),
                anchor=(torch.int32, (b, ncap)), count=(torch.int32, (b,)), flags=(torch.int32, (b,)))
    if out is None:      # pass the previous result back as `out` to reuse its buffers (rows past count are stale)
        out = {k: torch.zeros(s, dtype=dt, device=dev) for k, (dt, s) in spec.items()}
    for k, (dt, s) in spec.items():
        _arg(out[k], "out[%r]" % k, dt, s, dev)
    is_u8 = head.dtype == torch.uint8
    if is_u8 and quant is None:
        raise ValueError("u8 head needs quant=(scale, zero_point)")
    scale, zp = quant if is_u8 else (1.0, 0)
    _lib.check(_lib.lib().dd_yolo_decode(head.data_ptr(), 1 if is_u8 else 0, float(scale), int(zp), b, na, nc,
                                         wanted_mask.data_ptr(), float(score_thr), int(img_size[0]),
                                         int(img_size[1]), int(frame_size[0]), int(frame_size[1]), ncap,
                                         out["tlwh"].data_ptr(), out["score"].data_ptr(), out["cls"].data_ptr(),
                                         out["anchor"].data_ptr(), out["count"].data_ptr(),
                                         out["flags"].data_ptr(), _stream(dev)), "dd_yolo_decode")
    return out


def yolo3_decode(maps, anchors, wanted_mask, score_thr=0.5, nms_thresh=0.5, image_size=(640, 480), net_size=(416, 416),
                 ncap=256):
    """Keras YOLOv3 adapter post-processing for b frames (tools/yolo.py:48-153,207-237).  maps: three f32 CUDA tensors
    [b,g,g,3*(5+nc)]; anchors: 3 x 6 ints.  Returns dict(box f64 [b,ncap,4] (x, y, w, h), score f32, label i32,
    count i32 [b], flags i32 [b])."""
    import ctypes
    m = [_need_cuda(t) or t.contiguous() for t in maps]
    b, nc = m[0].shape[0], m[0].shape[-1] // 3 - 5
    dev = m[0].device
    out = dict(box=torch.zeros((b, ncap, 4), dtype=torch.float64, device=dev),
               score=torch.zeros((b, ncap), dtype=torch.float32, device=dev),
               label=torch.zeros((b, ncap), dtype=torch.int32, device=dev),
               count=torch.zeros((b,), dtype=torch.int32, device=dev), flags=torch.zeros((b,), dtype=torch.int32, device=dev))
    grids = (ctypes.c_int32 * 3)(*[int(t.shape[1]) for t in m])
    anch = (ctypes.c_int32 * 18)(*[int(a) for row in anchors for a in row])
    _lib.check(_lib.lib().dd_yolo3_decode(m[0].data_ptr(), m[1].data_ptr(), m[2].data_ptr(), grids, anch, b, nc,
                                          wanted_mask.data_ptr(), float(score_thr), float(nms_thresh), int(image_size[0]),
                                          int(image_size[1]), int(net_size[0]), int(net_size[1]), ncap, out["box"].data_ptr(),
                                          out["score"].data_ptr(), out["label"].data_ptr(), out["count"].data_ptr(),
                                          out["flags"].data_ptr(), _stream(dev)), "dd_yolo3_decode")
    return out


def ssd_decode(raw_boxes, raw_scores, anchors, class_to_label, conf_thr=0.5, nms_iou=0.5, img_size=(640, 480),
               frame_size=(640, 480), ncap=16, out=None):
    """SSD-MobileNet post-processing for b frames (TFLite_Detection_PostProcess restated +
    tools/ssd_mobilenet.py:59-150,198-213 + deepdish.py:946-955).  raw_boxes f32 [b,na,4], raw_scores f32
    [b,na,ncls], anchors f32 [na,4], class_to_label i32 [ncls-1].
    Returns dict(tlwh f64 [b,ncap,4], score f32, label i32, count i32 [b], flags i32 [b])."""
    _need_cuda(raw_boxes)
    dev = raw_boxes.device
    _arg(raw_boxes, "raw_boxes", torch.float32, (None, None, 4), dev)
    b, na, _ = raw_boxes.shape
    _arg(raw_scores, "raw_scores", torch.float32, (b, na, None), dev)
    ncls = raw_scores.shape[2]
    _arg(anchors, "anchors", torch.float32, (na, 4), dev)
    _arg(class_to_label, "class_to_label", torch.int32, (ncls - 1,), dev)
    spec = dict(tlwh=(torch.float64, (b, ncap, 4)), score=(torch.float32, (b, ncap)), label=(torch.int32, (b, ncap)),
                count=(torch.int32, (b,)), flags=(torch.int32, (b,)))
    if out is None:
        out = dict(tlwh=torch.zeros((b, ncap, 4), dtype=torch.float64, device=dev),
                   score=torch.zeros((b, ncap), dtype=torch.float32, device=dev),
                   label=torch.full((b, ncap), -1, dtype=torch.int32, device=dev),
                   count=torch.zeros((b,), dtype=torch.int32, device=dev),
                   flags=torch.zeros((b,), dtype=torch.int32, device=dev))
    for k, (dt, s) in spec.items():
        _arg(out[k], "out[%r]" % k, dt, s, dev)
    _lib.check(_lib.lib().dd_ssd_decode(raw_boxes.data_ptr(), raw_scores.data_ptr(), anchors.data_ptr(), b, na, ncls,
                                        class_to_label.data_ptr(), float(conf_thr), float(nms_iou),
                                        int(img_size[0]), int(img_size[1]), int(frame_size[0]), int(frame_size[1]),
                                        ncap, out["tlwh"].data_ptr(), out["score"].data_ptr(),
                                        out["label"].data_ptr(), out["count"].data_ptr(), out["flags"].data_ptr(),
                                        _stream(dev)), "dd_ssd_decode")
    return out


def tflite_postprocess(op_boxes, op_classes, op_scores, op_count, list_ok, wanted, score_thr=0.5, img_size=(640, 480),
                       max_results=-1, ncap=None):
    """TFLite object-detector adapter for b frames (tools/tflite_object_detector.py:234-295, tools/tflite.py:26-41).
    op_boxes f32 [b,n,4], op_classes f32 [b,n], op_scores f32 [b,n], op_count i32 [b]; list_ok / wanted u8 [n_labels].
    Returns dict(tlwh f64 [b,ncap,4], score f32, label i32, count i32 [b], flags i32 [b])."""
    _need_cuda(op_boxes)
    dev = op_boxes.device
    _arg(op_boxes, "op_boxes", torch.float32, (None, None, 4), dev)
    b, n, _ = op_boxes.shape
    _arg(op_classes, "op_classes", torch.float32, (b, n), dev)
    _arg(op_scores, "op_scores", torch.float32, (b, n), dev)
    _arg(op_count, "op_count", torch.int32, (b,), dev)
    _arg(list_ok, "list_ok", torch.uint8, (None,), dev)
    _arg(wanted, "wanted", torch.uint8, list_ok.shape, dev)
    ncap = n if ncap is None else ncap

    out = dict(tlwh=torch.zeros((b, ncap, 4), dtype=torch.float64, device=dev),
               score=torch.zeros((b, ncap), dtype=torch.float32, device=dev),
               label=torch.full((b, ncap), -1, dtype=torch.int32, device=dev),
               count=torch.zeros((b,), dtype=torch.int32, device=dev),
               flags=torch.zeros((b,), dtype=torch.int32, device=dev))
    _lib.check(_lib.lib().dd_tflite_postprocess(op_boxes.data_ptr(), op_classes.data_ptr(), op_scores.data_ptr(),
                                                op_count.data_ptr(), b, n, int(img_size[0]), int(img_size[1]),
                                                float(score_thr), list_ok.data_ptr(), wanted.data_ptr(),
                                                list_ok.shape[0], int(max_results), ncap, out["tlwh"].data_ptr(),
                                                out["score"].data_ptr(), out["label"].data_ptr(),
                                                out["count"].data_ptr(), out["flags"].data_ptr(), _stream(dev)),
               "dd_tflite_postprocess")
    return out


# ------------------------------------------------------------------------------------- encoder input
def extract_patches(frames, boxes, counts=None, patch_shape=(128, 64), boxes_are_int=True, out=None):
    """extract_image_patch for every box of b frames (tools/generate_detections.py:40-84, 198-205).
    frames u8 [b,H,W,3], boxes f64 [b,dmax,4] tlwh, counts i32 [b] or None.
    Returns (patches u8 [b,dmax,ph,pw,3], valid i32 [b,dmax]); out = (patches, valid) reuses buffers."""
    _need_cuda(frames)
    if frames.dtype != torch.uint8 or boxes.dtype != torch.float64:
        raise ValueError("frames must be uint8 and boxes float64")
    b, H, W, ch = frames.shape
    if ch != 3:
        raise ValueError("frames must be [b,H,W,3]")
    dmax = boxes.shape[1]
    ph, pw = int(patch_shape[0]), int(patch_shape[1])
    if out is None:
        patches = torch.zeros((b, dmax, ph, pw, 3), dtype=torch.uint8, device=frames.device)
        valid = torch.zeros((b, dmax), dtype=torch.int32, device=frames.device)
    else:
        patches, valid = out
    _lib.check(_lib.lib().dd_extract_patches(frames.data_ptr(), b, H, W, boxes.data_ptr(),
                                             counts.data_ptr() if counts is not None else None, dmax,
                                             1 if boxes_are_int else 0, ph, pw, patches.data_ptr(),
                                             valid.data_ptr(), _stream(frames.device)), "dd_extract_patches")
    return patches, valid


def dummy_encode(patches, out=None):
    """DummyImageEncoder.__call__ (tools/generate_detections.py:86-105): u8 [...,16,8,3] -> f32 [...,128]."""
    _need_cuda(patches)
    if patches.dtype != torch.uint8 or tuple(patches.shape[-3:]) != (16, 8, 3):
        raise ValueError("patches must be uint8 [...,16,8,3]")
    lead = tuple(patches.shape[:-3])
    n = int(np.prod(lead)) if lead else 1
    if out is None:
        out = torch.empty(lead + (128,), dtype=torch.float32, device=patches.device)
    _lib.check(_lib.lib().dd_dummy_encode(patches.data_ptr(), n, out.data_ptr(), _stream(patches.device)),
               "dd_dummy_encode")
    return out
