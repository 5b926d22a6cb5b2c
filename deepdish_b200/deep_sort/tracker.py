"""``deep_sort.tracker`` mirror (reference deep_sort/tracker.py): ``Tracker`` is the S = 1 view of
``deepdish_b200.batched.BatchedTracker``.  ``predict()`` / ``update(detections)`` launch the same CUDA
kernels as the batched path and return without reading the state back; ``tracks`` / ``deleted_tracks`` are LAZY
host views (lists of Track in the reference's list order), materialised from the device state with one packed
device-to-host copy the first time they are looked at after a device call."""
import ctypes

import numpy as np
import torch

from .. import _lib
from ..batched import BatchedTracker
from . import kalman_filter
from .track import Track, TrackState  # noqa: F401  (TrackState re-exported like the reference module)

# state arrays a host view needs, all inside the packed prefix of the blob (everything before the per-tick scratch)
_VIEW_FIELDS = ("n_tracks", "n_deleted", "order", "deleted", "mean", "cov", "track_id", "hits", "age", "tsu", "state",
                "lab_cnt", "lab_sum")


class Tracker:
    MAX_TRACKS = 256          # slots (live + deleted-this-tick + new); overflow raises, never truncates
    MAX_DETS = 256

    def __init__(self, metric, max_iou_distance=0.7, max_age=30, n_init=3):
        self.metric = metric
        self.max_iou_distance = max_iou_distance
        self.max_age = max_age
        self.n_init = n_init
        self.kf = kalman_filter.KalmanFilter()
        self._tracks = []
        self._deleted = []
        self._objs = {}                        # track id -> Track: the host objects persist across frames
        self._stale = False                    # the device state is newer than the host lists
        self._device_ids = []                  # track ids of the device's live list, in its order (as last materialised)
        self._late_features = []               # (track_id, unit feature) to enter the gallery after the next matching
        self._labels = []                      # label vocabulary in first-seen order
        self._bt = None
        self._host_blob = None
        if getattr(metric, "_metric_name", "cosine") != "cosine":
            # the device tick computes the cosine metric only (deepdish.py:516 never builds another one); the
            # euclidean metric stays available through NearestNeighborDistanceMetric.distance
            raise NotImplementedError("Tracker runs the 'cosine' metric on the device; got %r" % metric._metric_name)

    # -- lazy host views ------------------------------------------------------------------------
    @property
    def tracks(self):
        self._sync()
        return self._tracks

    @tracks.setter
    def tracks(self, value):
        """``tracker.tracks = [...]`` (deepdish.py:1047): tracks missing from the new list are dropped from the
        device's live list at the next device call."""
        self._sync()
        self._tracks = list(value)

    @property
    def deleted_tracks(self):
        self._sync()
        return self._deleted

    @deleted_tracks.setter
    def deleted_tracks(self, value):
        self._sync()
        self._deleted = list(value)

    def _sync(self):
        if self._stale:
            self._stale = False
            self._materialize()

    def _materialize(self):
        """One packed device-to-host copy of the blob's state prefix, then the Track lists in the reference's order."""
        bt = self._bt
        c = bt.chunks[0]
        nbytes = int(c.lay.gate)                                   # the per-tick scratch starts at `gate`
        if self._host_blob is None or self._host_blob.numel() != nbytes:
            self._host_blob = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        self._host_blob.copy_(c.blob[:nbytes], non_blocking=True)
        torch.cuda.current_stream(bt.device).synchronize()
        raw = self._host_blob.numpy()
        v = {}
        specs = _lib.field_specs(c.cfg)
        for name in _VIEW_FIELDS:
            dt, shape = specs[name]
            off = int(getattr(c.lay, name))
            n = int(np.prod(shape)) * np.dtype(dt).itemsize
            v[name] = raw[off:off + n].view(dt).reshape(shape)[0]
        nlab = len(self._labels)

        def make(slot):
            tid = int(v["track_id"][slot])
            t = self._objs.get(tid)
            if t is None:
                t = self._objs[tid] = Track(None, None, tid, self.n_init, self.max_age)
            t.mean = v["mean"][slot].copy()
            t.covariance = v["cov"][slot].copy()
            t.hits, t.age = int(v["hits"][slot]), int(v["age"][slot])
            t.time_since_update, t.state = int(v["tsu"][slot]), int(v["state"][slot])
            t._slot = int(slot)
            cnt = v["lab_cnt"][slot, :nlab]
            t._label_stats = {self._labels[k]: (int(cnt[k]), float(v["lab_sum"][slot, k])) for k in np.nonzero(cnt)[0]}
            if t.state == TrackState.Confirmed:
                t.features = []                                    # moved to metric.samples (tracker.py:84-93)
            return t

        self._tracks = [make(s) for s in v["order"][:int(v["n_tracks"])]]
        self._device_ids = [t.track_id for t in self._tracks]
        self._deleted = [make(s) for s in v["deleted"][:int(v["n_deleted"])]]
        keep = set(self._device_ids) | {t.track_id for t in self._deleted}
        if len(self._objs) > 2 * len(keep) + 64:                   # forget tracks that left both lists
            self._objs = {k: t for k, t in self._objs.items() if k in keep}

    # -- host edits written back to the device ------------------------------------------------
    def _flush(self):
        """Write host-side edits back before the device runs again: tracks dropped from ``tracks`` leave the live
        list (their slots become free), and tracks updated through ``Track.update(kf, detection)`` outside the tracker
        (framerecords.py:157-160) get their Kalman state, hits, time_since_update, state and label votes stored.
        Their features join the gallery after the NEXT matching, exactly when the reference's partial_fit would
        move them from ``track.features`` to ``metric.samples`` (tracker.py:84-93).  Nothing can have been edited
        when the lists were not looked at since the last device call."""
        if self._bt is None or self._stale:
            return
        v = self._bt.chunks[0].v
        keep = {t.track_id for t in self._tracks}
        if any(tid not in keep for tid in self._device_ids):
            n = int(v["n_tracks"][0])
            order = v["order"][0, :n].cpu().numpy()
            ids = v["track_id"][0].cpu().numpy()
            live = [int(s) for s in order if int(ids[s]) in keep]
            for s in order:
                if int(ids[s]) not in keep:
                    v["state"][0, int(s)] = 0                                   # DD_STATE_FREE
            if live:
                v["order"][0, :len(live)] = torch.as_tensor(live, dtype=torch.int32, device=v["order"].device)
            v["n_tracks"][0] = len(live)
            self._device_ids = [int(ids[s]) for s in live]
        for t in self._tracks:
            if not t._pending:
                continue
            s = t._slot
            dev = v["mean"].device
            v["mean"][0, s] = torch.as_tensor(np.asarray(t.mean, np.float64), device=dev)
            v["cov"][0, s] = torch.as_tensor(np.asarray(t.covariance, np.float64), device=dev)
            v["hits"][0, s], v["tsu"][0, s], v["state"][0, s] = int(t.hits), int(t.time_since_update), int(t.state)
            for d in t._pending:
                c = self._label_id(d.label)
                v["lab_cnt"][0, s, c] += 1
                v["lab_sum"][0, s, c] += float(d.confidence)
                f = np.asarray(d.feature, np.float32)
                self._late_features.append((t.track_id, f / np.float32(np.sqrt(np.sum(f * f, dtype=np.float32)))))
            t._pending = []

    def _apply_late_features(self, matched_ids):
        """Gallery surgery after a matching: a late feature goes in BEFORE the feature the update just appended for
        the same track (the order partial_fit would produce), or at the end if the track was not matched."""
        self._sync()
        slot_of = {t.track_id: t._slot for t in self._tracks}
        for tid, f in self._late_features:
            if tid in slot_of:
                self._bt.gallery_insert(0, slot_of[tid], f, before_newest=tid in matched_ids)
        self._late_features = []

    # -- device state -----------------------------------------------------------------------
    def _ensure(self):
        if self._bt is None:
            names = ["\x00unused%03d" % i for i in range(_lib.DD_MAX_LABELS)]
            bt = self._bt = BatchedTracker(1, names, max_tracks=self.MAX_TRACKS, max_dets=self.MAX_DETS,
                                           budget=self.metric.budget, max_cosine_distance=self.metric.matching_threshold,
                                           max_iou_distance=self.max_iou_distance, max_age=self.max_age,
                                           n_init=self.n_init, pool_pages=2048, seg_pages=2048, page_cap=64)
            D = self.MAX_DETS
            # persistent staging: pinned host arrays (numpy views) + device arrays; a call copies only its n rows
            self._h = (torch.zeros((1, D, 4), dtype=torch.float64).pin_memory(), torch.zeros((1, D), dtype=torch.float32).pin_memory(),
                       torch.zeros((1, D), dtype=torch.int32).pin_memory(), torch.zeros((1, D, 128), dtype=torch.float32).pin_memory(),
                       torch.zeros((1,), dtype=torch.int32).pin_memory())
            self._hn = tuple(t.numpy() for t in self._h)
            self._d = tuple(torch.zeros(t.shape, dtype=t.dtype, device=bt.device) for t in self._h)
            self._ids_host = torch.zeros((D,), dtype=torch.int32).pin_memory()
        return self._bt

    @property
    def _next_id(self):
        return 1 if self._bt is None else int(self._bt.v["next_id"][0])

    def _label_id(self, label):
        if label not in self._labels:
            if len(self._labels) >= _lib.DD_MAX_LABELS:
                raise RuntimeError("more than %d distinct labels" % _lib.DD_MAX_LABELS)
            self._labels.append(label)
            cfg = self._bt.cfg                  # ranks follow ascending label-name order (track.py:170)
            order = sorted(range(len(self._labels)), key=lambda i: self._labels[i])
            for r, i in enumerate(order):
                cfg.label_rank[i] = r
            cfg.label_motorbike = self._labels.index("motorbike") if "motorbike" in self._labels else -1
            cfg.label_bicycle = self._labels.index("bicycle") if "bicycle" in self._labels else -1
        return self._labels.index(label)

    # -- reference API ----------------------------------------------------------------------
    def predict(self):
        """tracker.py:51-57."""
        if self._bt is None:
            return
        self._flush()
        self._bt.predict()
        self._stale = True

    def update(self, detections):
        """tracker.py:59-93."""
        bt = self._ensure()
        self._flush()
        D = bt.cfg.max_dets
        n = len(detections)
        if n > D:
            raise RuntimeError("detection capacity exceeded (%d > %d)" % (n, D))
        tlwh, conf, lab, feat, cnt = self._hn
        for i, d in enumerate(detections):
            tlwh[0, i], conf[0, i], lab[0, i] = d.tlwh, d.confidence, self._label_id(d.label)
            feat[0, i] = d.feature
        cnt[0] = n
        if n:
            for dv, hv in zip(self._d[:4], self._h[:4]):
                dv[0, :n].copy_(hv[0, :n], non_blocking=True)
        self._d[4].copy_(self._h[4], non_blocking=True)
        ids = bt.update(*self._d)
        if n:
            self._ids_host[:n].copy_(ids[0, :n], non_blocking=True)
        flags = ctypes.c_int32(0)                   # dd_tracker_status synchronises the stream: the ids are on the host after it
        c = bt.chunks[0]
        _lib.check(bt.lib.dd_tracker_status(c.state, c.cfgp, ctypes.byref(flags),
                                            ctypes.c_void_p(torch.cuda.current_stream(bt.device).cuda_stream)), "dd_tracker_status")
        self.last_detection_track_ids = self._ids_host[:n].numpy().copy()
        self._stale = True
        self.metric.samples = _LazySamples(self)
        if flags.value:
            bt.check()                              # raises with the reason
        if self._late_features:
            self._apply_late_features({int(i) for i in self.last_detection_track_ids})
        for i, d in enumerate(detections):          # host-side caches kept like track.py:75-80,147-151
            tid = int(self.last_detection_track_ids[i])
            if tid < 0:
                continue
            t = self._objs.get(tid)
            if t is None:
                t = self._objs[tid] = Track(None, None, tid, self.n_init, self.max_age)
            t.labels.append(d.label)
            t.dist.setdefault(d.label, []).append(d.confidence)
            t.detections.append(d)
            t.features.append(d.feature)            # emptied for confirmed tracks when the views are materialised


class _LazySamples(dict):
    """``metric.samples``: {track_id: [unit-normalised gallery vectors, oldest first]} read from the
    device galleries on first access (nn_matching.py:132-154 keeps only confirmed targets)."""

    def __init__(self, trk):
        super().__init__()
        self._trk, self._loaded = trk, False

    def _load(self):
        if self._loaded:
            return
        self._loaded = True
        trk = self._trk
        for t in trk.tracks:
            if t.is_confirmed():
                dict.__setitem__(self, t.track_id, list(trk._bt.gallery(0, t._slot).cpu().numpy()))

    def __getitem__(self, k):
        self._load(); return dict.__getitem__(self, k)

    def __iter__(self):
        self._load(); return dict.__iter__(self)

    def __len__(self):
        self._load(); return dict.__len__(self)

    def keys(self):
        self._load(); return dict.keys(self)

    def values(self):
        self._load(); return dict.values(self)

    def items(self):
        self._load(); return dict.items(self)

    def get(self, k, default=None):
        self._load(); return dict.get(self, k, default)

    def __contains__(self, k):
        self._load(); return dict.__contains__(self, k)
