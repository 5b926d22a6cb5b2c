"""ctypes binding of libdeepdish_b200.so (the C ABI declared in include/deepdish_b200.h).

There is deliberately no fallback: if the CUDA library has not been built, importing any operator
raises.  Build it with ``python -m deepdish_b200.build`` (nvcc, sm_100a).
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdeepdish_b200.so")

DD_OK, DD_ERR_INVALID, DD_ERR_CUDA, DD_ERR_CAPACITY = 0, -1, -2, -3
DD_MAX_LABELS = 128
DD_MAX_LINES = 32
DD_MAX_SEGS = 16
PAGE_ROWS, PAGE_F32_BYTES, PAGE_F16_BYTES = 16, 8192, 4096
FLAG_TRACK_OVERFLOW, FLAG_DET_OVERFLOW, FLAG_LSAP_INFEASIBLE = 1, 2, 4
FLAG_POOL_EXHAUSTED, FLAG_GALLERY_OVERFLOW, FLAG_BAD_LABEL = 8, 16, 32
GALLERY_IMPLS = {"default": 0, "exact": 1}

_i32, _f64, _u64, _vp = ctypes.c_int32, ctypes.c_double, ctypes.c_uint64, ctypes.c_void_p


class TrackerConfig(ctypes.Structure):
    _fields_ = [("n_streams", _i32), ("max_tracks", _i32), ("max_dets", _i32), ("budget", _i32),
                ("feat_dim", _i32), ("n_labels", _i32), ("max_age", _i32), ("n_init", _i32),
                ("max_cosine_distance", _f64), ("max_iou_distance", _f64),
                ("label_motorbike", _i32), ("label_bicycle", _i32),
                ("label_rank", _i32 * DD_MAX_LABELS),
                ("page_cap", _i32), ("seg_pages", _i32), ("n_segs", _i32),
                ("gallery_impl", _i32), ("cosine_ctas_per_sm", _i32), ("match_warps", _i32),
                ("gallery_stages", _i32), ("gallery_waves", _i32), ("event_cap", _i32), ("timeline", _i32),
                ("n_lines", _i32), ("pool_f32", _u64 * DD_MAX_SEGS), ("pool_f16", _u64 * DD_MAX_SEGS)]


LAYOUT_FIELDS = ["n_tracks", "next_id", "n_deleted", "err", "order", "deleted", "counts", "mean", "cov",
                 "track_id", "hits", "age", "tsu", "state", "gal_len", "gal_pos", "gal_np", "ptab", "free_stack",
                 "pool_ctl", "lab_cnt", "lab_sum", "path_n", "path_last", "path_crossed", "gate", "cost", "det_xyah",
                 "det_featn", "det_slot", "det_kind", "cdesc", "work", "work_ctl", "work_rec", "det_feath", "tick_args", "timeline",
                 "tick_present"]
# the crossing records: appended after every array above, 0 bytes (offset == total_bytes) unless event_cap > 0
EVENTS_FIELD = "events"


class TrackerLayout(ctypes.Structure):
    _fields_ = [("total_bytes", _u64)] + [(n, _u64) for n in LAYOUT_FIELDS + [EVENTS_FIELD]]


def n_lines(cfg):
    """Count lines per stream (config.n_lines, 0 read as 1)."""
    return cfg.n_lines or 1


def counts_shape(cfg):
    """Shape of one stream's counters: [C,4] with one count line, [L,C,4] with L > 1."""
    L = n_lines(cfg)
    return (cfg.n_labels, 4) if L == 1 else (L, cfg.n_labels, 4)


def field_specs(cfg):
    """name -> (dtype string, shape) of every array in the state blob."""
    S, T, D, C = cfg.n_streams, cfg.max_tracks, cfg.max_dets, cfg.n_labels
    DW = (D + 31) // 32
    PT = page_cap(cfg)
    i, f, d = "int32", "float32", "float64"
    return {
        "n_tracks": (i, (S,)), "next_id": (i, (S,)), "n_deleted": (i, (S,)), "err": (i, (S,)),
        "order": (i, (S, T)), "deleted": (i, (S, T)), "counts": ("int64", (S,) + counts_shape(cfg)),
        "mean": (d, (S, T, 8)), "cov": (d, (S, T, 8, 8)), "track_id": (i, (S, T)),
        "hits": (i, (S, T)), "age": (i, (S, T)), "tsu": (i, (S, T)), "state": (i, (S, T)),
        "gal_len": (i, (S, T)), "gal_pos": (i, (S, T)), "gal_np": (i, (S, T)), "ptab": (i, (S, T, PT)),
        "free_stack": (i, (DD_MAX_SEGS * cfg.seg_pages,)), "pool_ctl": (i, (64,)),
        "lab_cnt": (i, (S, T, C)), "lab_sum": (d, (S, T, C)), "path_n": (i, (S, T)),
        "path_last": (d, (S, T, 2)), "path_crossed": (i, (S, T)), "gate": (i, (S, T, DW)),
        "cost": (f, (S, T, D)), "det_xyah": (d, (S, D, 4)), "det_featn": (f, (S, D, 128)),
        "det_slot": (i, (S, D)), "det_kind": (i, (S, D)), "cdesc": (i, (S, T, 4)),
        "work": (i, (S * T,)), "work_ctl": (i, (64,)), "work_rec": (i, (S * T, 16)),
        "det_feath": ("float16", (S, D, 128)), "tick_args": (i, (64,)), "timeline": ("int64", (64, 8, 2)),
        "tick_present": (i, (S,)),
        # row 0 = header (records this count-line step produced), rows 1.. = {stream, track_id, label, column + 4 line}
        "events": (i, (cfg.event_cap + 1 if cfg.event_cap > 0 else 0, 4)),
    }


def page_cap(cfg):
    """Page-table entries per slot (dd_page_cap in csrc/dd_view.h)."""
    need = (cfg.budget + PAGE_ROWS - 1) // PAGE_ROWS if cfg.budget > 0 else 1
    return max(cfg.page_cap, need)


def make_config(n_streams, max_tracks, max_dets, budget, labels, max_age=30, n_init=3,
                max_cosine_distance=0.2, max_iou_distance=0.7, page_cap=0, seg_pages=1024,
                gallery_impl=0, cosine_ctas_per_sm=0, match_warps=0, gallery_stages=0, gallery_waves=0,
                timeline=0, event_cap=0, n_lines=1):
    """Fill a dd_tracker_config from Python values; ``labels`` is the ordered list of label names.
    ``budget=None`` is the reference's nn_budget=None (deepdish.py:515): unbounded galleries (budget 0 in the C
    struct).  The pool segment pointers are filled in by the caller that allocates them."""
    labels = list(labels)
    if not 0 < len(labels) <= DD_MAX_LABELS:
        raise ValueError("need 1..%d labels" % DD_MAX_LABELS)
    if budget is not None and budget <= 0:
        raise ValueError("nn_budget must be positive or None")
    if seg_pages <= 0 or seg_pages & (seg_pages - 1):
        raise ValueError("seg_pages must be a power of two")
    cfg = TrackerConfig()
    cfg.n_streams, cfg.max_tracks, cfg.max_dets, cfg.budget = n_streams, max_tracks, max_dets, budget or 0
    cfg.page_cap, cfg.seg_pages, cfg.n_segs = page_cap, seg_pages, 1
    cfg.gallery_impl = GALLERY_IMPLS[gallery_impl] if isinstance(gallery_impl, str) else int(gallery_impl)
    cfg.cosine_ctas_per_sm, cfg.match_warps, cfg.gallery_stages = cosine_ctas_per_sm, match_warps, gallery_stages
    cfg.gallery_waves, cfg.timeline, cfg.event_cap, cfg.n_lines = gallery_waves, timeline, event_cap, n_lines
    cfg.feat_dim, cfg.n_labels, cfg.max_age, cfg.n_init = 128, len(labels), max_age, n_init
    cfg.max_cosine_distance, cfg.max_iou_distance = max_cosine_distance, max_iou_distance
    cfg.label_motorbike = labels.index("motorbike") if "motorbike" in labels else -1
    cfg.label_bicycle = labels.index("bicycle") if "bicycle" in labels else -1
    ranks = {n: r for r, n in enumerate(sorted(labels))}
    for k, n in enumerate(labels):
        cfg.label_rank[k] = ranks[n]
    return cfg


_lib = None


def lib():
    """Load the CUDA library or raise -- never falls back to a CPU implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("deepdish_b200: CUDA library %s is missing; build it with "
                           "`python -m deepdish_b200.build` (nvcc, sm_100a). There is no CPU fallback."
                           % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    L.dd_version.restype = ctypes.c_char_p
    cfgp, layp = ctypes.POINTER(TrackerConfig), ctypes.POINTER(TrackerLayout)
    sigs = {
        "dd_tracker_layout_query": [cfgp, layp],
        "dd_tracker_init": [_vp, cfgp, _vp],
        "dd_tracker_predict": [_vp, cfgp, _vp],
        "dd_tracker_update": [_vp, cfgp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
        "dd_tracker_update_profiled": [_vp, cfgp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.POINTER(_vp)],
        "dd_tracker_pool_attach": [_vp, cfgp, _vp],
        "dd_tracker_gallery_read": [_vp, cfgp, _i32, _i32, _vp, _i32, _vp],
        "dd_tracker_gallery_insert": [_vp, cfgp, _i32, _i32, _vp, _i32, _vp],
        "dd_event_create": [ctypes.POINTER(_vp)],
        "dd_event_destroy": [_vp],
        "dd_event_elapsed_ms": [_vp, _vp, ctypes.POINTER(ctypes.c_float)],
        "dd_event_record": [_vp, _vp],
        "dd_tracker_countline": [_vp, cfgp, _vp, _i32, _vp],
        "dd_unpack_detections": [_vp, _i32, _i32, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                 _vp, _vp, _vp, _vp, _vp, _vp],
        "dd_tracker_count_reduce": [_vp, cfgp, _vp, _vp],
        "dd_tracker_status": [_vp, cfgp, ctypes.POINTER(_i32), _vp],
        "dd_engine_create": [_i32, ctypes.POINTER(_vp), ctypes.POINTER(cfgp), ctypes.POINTER(_i32), ctypes.POINTER(_vp), _vp,
                             _vp, _i32, _vp, _vp, _vp, _i32, _i32, ctypes.POINTER(_vp)],
        "dd_engine_destroy": [_vp],
        "dd_engine_set_graphs": [_vp, _i32],
        "dd_engine_rebind": [_vp, _i32, _vp, cfgp],
        "dd_engine_bind_host": [_vp, _i32, ctypes.POINTER(_vp), _i32, _u64, _vp, _vp, _vp, _vp],
        "dd_engine_step": [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp],
        "dd_engine_step_host": [_vp, ctypes.POINTER(_vp), ctypes.POINTER(_u64), ctypes.POINTER(ctypes.c_int64), _vp, _vp],
        "dd_engine_step_present": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp],
        "dd_engine_step_host_present": [_vp, ctypes.POINTER(_vp), ctypes.POINTER(_u64), ctypes.POINTER(ctypes.c_int64), _vp,
                                        _vp],
        "dd_engine_copy_events": [_vp, _vp, _vp],
        "dd_engine_join": [_vp, _vp],
        "dd_engine_wait_counts": [_vp, _vp],
        "dd_engine_pool_latest": [_vp, _i32, _i32, ctypes.POINTER(_i32), ctypes.POINTER(ctypes.c_int64)],
        "dd_engine_stats": [_vp, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64),
                            ctypes.POINTER(ctypes.c_double)],
        "dd_kalman_initiate": [_vp, _vp, _vp, _i32, _vp],
        "dd_kalman_predict": [_vp, _vp, _i32, _vp],
        "dd_kalman_project": [_vp, _vp, _vp, _vp, _i32, _vp],
        "dd_kalman_update": [_vp, _vp, _vp, _i32, _vp],
        "dd_kalman_gating_distance": [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp],
        "dd_nn_distance": [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp],
        "dd_iou_cost": [_vp, _vp, _vp, _i32, _i32, _vp, _vp],
        "dd_lsap": [_vp, _i32, _i32, _i32, _vp, _vp, _vp],
        "dd_set_difference_order": [_vp, _vp, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp],
        "dd_intersection": [_vp, _i32, _vp, _vp],
        "dd_nms": [_vp, _vp, _vp, _i32, _i32, _f64, _vp, _vp, _vp],
        "dd_ssd_decode": [_vp, _vp, _vp, _i32, _i32, _i32, _vp, ctypes.c_float, _f64, _i32, _i32, _i32, _i32, _i32,
                          _vp, _vp, _vp, _vp, _vp, _vp],
        "dd_yolo3_decode": [_vp, _vp, _vp, ctypes.POINTER(_i32), ctypes.POINTER(_i32), _i32, _i32, _vp, ctypes.c_float, _f64,
                            _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp],
        "dd_box_filter": [_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp],
        "dd_gather_detections": [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp],
        "dd_tflite_postprocess": [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, ctypes.c_float, _vp, _vp, _i32, _i32, _i32,
                                  _vp, _vp, _vp, _vp, _vp, _vp],
        "dd_extract_patches": [_vp, _i32, _i32, _i32, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp],
        "dd_dummy_encode": [_vp, _i32, _vp, _vp],
        "dd_yolo_decode": [_vp, _i32, ctypes.c_float, _i32, _i32, _i32, _i32, _vp, ctypes.c_float,
                           _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    }
    for name, args in sigs.items():
        fn = getattr(L, name)
        fn.argtypes = args
        fn.restype = ctypes.c_int
    _lib = L
    return L


def check(rc, what):
    if rc == DD_OK:
        return
    msg = {DD_ERR_INVALID: "invalid argument", DD_ERR_CUDA: "CUDA error",
           DD_ERR_CAPACITY: "capacity exceeded"}.get(rc, "error %d" % rc)
    if rc == DD_ERR_INVALID:
        raise ValueError("%s: %s" % (what, msg))
    raise RuntimeError("%s: %s" % (what, msg))
