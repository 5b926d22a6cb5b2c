"""BatchedTracker -- S independent DeepSORT trackers stepped together on one B200.

The batched extension of the reference's ``deep_sort.tracker.Tracker`` (SURVEY.md section 8b): same
``predict()`` / ``update(detections)`` call sequence (tracker.py:51-93), plus the count-line step of
``Pipeline.process_results`` (deepdish.py:1035-1114).  All state lives in caller-owned device blobs
whose layout is defined by the C ABI (include/deepdish_b200.h); this class only allocates them with
torch, passes raw pointers + a CUDA stream to libdeepdish_b200.so, and exposes typed torch views for
inspection.  There is no CPU path.

Stream chunks.  Streams never interact, so the S streams can be split into ``n_chunks`` contiguous
chunks, each with its own state blob and its own CUDA stream.  A chunk's tick is a strictly ordered
kernel sequence on its stream; different chunks overlap freely, so the latency-bound per-stream
matching kernel of one chunk runs under the HBM-bound gallery kernel of another, also across tick
boundaries.  ``step(..., join=False)`` only enqueues; ``join()`` makes the caller's stream wait for
every chunk.  With ``n_chunks=1`` everything runs on the caller's current stream.
"""
import collections
import ctypes

import numpy as np
import torch

from . import _lib

_DT = {"int32": torch.int32, "int64": torch.int64, "float32": torch.float32,
       "float64": torch.float64, "float16": torch.float16}


Crossings = collections.namedtuple("Crossings", "stream track_id label column")
Crossings.__doc__ = """Count-line crossings of one tick, numpy int32 arrays sorted by stream (tracker-wide index) and within a stream
in the order the reference's ``process_results`` counts them (``tracker.tracks``, then the deleted track): column 0 /
1 = a live track crossed the line (pos / neg, and int, of ``label``), 3 = the del count of the last deleted track."""

LineCrossings = collections.namedtuple("LineCrossings", "stream track_id label column line")
LineCrossings.__doc__ = """Crossings of a tracker with several count lines per stream: as ``Crossings``, plus the line each record
counts on.  Within a stream: ``tracker.tracks`` order, each track's lines ascending, then the deletion records, lines
ascending."""


def _pow2_at_least(n):
    p = 1
    while p < n:
        p <<= 1
    return p


class _Chunk:
    """One contiguous block of streams: config, state blob, gallery page pool, typed views, CUDA stream.

    Gallery storage is a pool of 16-row pages (f32 page + half page) in up to ``DD_MAX_SEGS`` equal segments
    allocated with torch; the blob only holds the page tables.  ``grow_pool`` attaches one more segment,
    ``grow_page_table`` re-lays the blob out with a larger per-slot page table (unbounded galleries)."""

    def __init__(self, owner, lo, hi, stream):
        self.lo, self.hi = lo, hi
        self.stream = stream
        self.owner = o = owner
        n = hi - lo
        rows = o.budget if o.budget is not None else 64
        worst = n * o.max_tracks * ((rows + _lib.PAGE_ROWS - 1) // _lib.PAGE_ROWS)
        seg_pages = o.seg_pages or _pow2_at_least(max(64, -(-worst // (_lib.DD_MAX_SEGS - 4))))
        want = o.pool_pages if o.pool_pages is not None else max(1, int(worst * o.pool_fraction))
        n_segs = max(1, min(_lib.DD_MAX_SEGS, -(-want // seg_pages)))
        self.cfg = _lib.make_config(n, o.max_tracks, o.max_dets, o.budget, o.labels, max_age=o.max_age,
                                    n_init=o.n_init, max_cosine_distance=o.max_cosine_distance,
                                    max_iou_distance=o.max_iou_distance, page_cap=o.page_cap, seg_pages=seg_pages,
                                    gallery_impl=o.gallery_impl, cosine_ctas_per_sm=o.cosine_ctas_per_sm,
                                    match_warps=o.match_warps, gallery_stages=o.gallery_stages,
                                    gallery_waves=o.gallery_waves,
                                    timeline=o.timeline, event_cap=o.crossing_capacity, n_lines=o.n_lines)
        self.cfgp = ctypes.byref(self.cfg)
        self.segs = []
        for _ in range(n_segs):
            self._alloc_seg()
        self.cfg.n_segs = n_segs
        self._bind()
        self.done = torch.cuda.Event()

    def _alloc_seg(self):
        k = len(self.segs)
        if k >= _lib.DD_MAX_SEGS:
            raise RuntimeError("gallery page pool cannot grow beyond %d segments of %d pages; construct the tracker "
                               "with a larger seg_pages" % (_lib.DD_MAX_SEGS, self.cfg.seg_pages))
        dev = self.owner.device
        f32 = torch.empty(self.cfg.seg_pages * _lib.PAGE_F32_BYTES, dtype=torch.uint8, device=dev)
        f16 = torch.empty(self.cfg.seg_pages * _lib.PAGE_F16_BYTES, dtype=torch.uint8, device=dev)
        self.segs.append((f32, f16))
        self.cfg.pool_f32[k], self.cfg.pool_f16[k] = f32.data_ptr(), f16.data_ptr()

    def _bind(self):
        """(Re)compute the layout for self.cfg, allocate the blob and make the typed views."""
        self.lay = _lib.TrackerLayout()
        _lib.check(self.owner.lib.dd_tracker_layout_query(self.cfgp, ctypes.byref(self.lay)), "dd_tracker_layout_query")
        self.blob = torch.empty(self.lay.total_bytes, dtype=torch.uint8, device=self.owner.device)
        self.state = self.blob.data_ptr()
        self.v = {}
        for name, (dt, shape) in _lib.field_specs(self.cfg).items():
            off = getattr(self.lay, name)
            n = torch.empty((), dtype=_DT[dt]).element_size()
            for d in shape:
                n *= d
            self.v[name] = self.blob[off:off + n].view(_DT[dt]).view(shape)

    def pool_bytes(self):
        return sum(a.numel() + b.numel() for a, b in self.segs)

    def grow_pool(self, sp):
        """Attach one more pool segment (enqueued on the chunk's stream: ordered after the ticks already there)."""
        self._alloc_seg()
        self.cfg.n_segs = len(self.segs)
        _lib.check(self.owner.lib.dd_tracker_pool_attach(self.state, self.cfgp, sp), "dd_tracker_pool_attach")

    def grow_page_table(self, page_cap):
        """Re-layout with a larger per-slot page table.  The caller has synchronised the chunk's stream."""
        old = self.v
        old_blob = self.blob  # noqa: F841  (keeps the old views alive while copying)
        self.cfg.page_cap = int(page_cap)
        self._bind()
        pt = old["ptab"].shape[2]
        for name, t in self.v.items():
            if name == "ptab":
                t[:, :, :pt].copy_(old[name])
            else:
                t.copy_(old[name])


class _CatView:
    """``bt.v[name]``: the state array of all streams (concatenation over chunks; a view when there
    is a single chunk).  Read-only for n_chunks > 1."""

    def __init__(self, owner):
        self._o = owner

    def __getitem__(self, name):
        o = self._o
        if len(o.chunks) == 1:
            return o.chunks[0].v[name]
        o.join()
        return torch.cat([c.v[name] for c in o.chunks], dim=0)

    def __iter__(self):
        return iter(self._o.chunks[0].v)

    def keys(self):
        return self._o.chunks[0].v.keys()


class BatchedTracker:
    def __init__(self, n_streams, labels, max_tracks=128, max_dets=64, budget=100,
                 max_cosine_distance=0.2, max_iou_distance=0.7, max_age=30, n_init=3,
                 line=None, frame_size=(640, 480), device="cuda", n_chunks=1,
                 pool_pages=None, pool_fraction=0.5, seg_pages=None, page_cap=0,
                 gallery_impl="default", cosine_ctas_per_sm=0, match_warps=0, gallery_stages=0, gallery_waves=0,
                 timeline=0, gallery_turns=True, engine_graphs=True, crossing_capacity=0, lines=None):
        """budget=None is the reference's nn_budget=None (deepdish.py:515-516): galleries grow without bound; the
        page pool and the per-slot page tables are grown between ticks (``maintain``).

        Gallery memory: ``pool_pages`` 16-row pages per chunk (default: ``pool_fraction`` of the worst case
        streams x max_tracks x ceil(budget / 16)), in segments of ``seg_pages``; more segments are attached when
        fewer than 1/8 of the pages are free.  A pool that still runs dry raises in ``check()``.

        crossing_capacity > 0: every count-line step also lists its crossings (``crossings()``), up to that many
        records per chunk and tick; 0 (the default) leaves the count-line step exactly as without it.

        Count lines: ``line`` is one segment (x1, y1, x2, y2) for all streams or one per stream ([S,4]); default the
        reference's vertical mid-line of ``frame_size``.  ``lines`` (instead of ``line``) gives several lines per
        stream: [L,4] shared by all streams or [S,L,4] per stream, 1 <= L <= 32.  Each line is counted as the reference
        counts its one line; with L > 1 the counters gain a line axis (``total_counts`` [L,C,4], ``v["counts"]``
        [S,L,C,4]) and ``crossings()`` returns ``LineCrossings``.  ``lines`` with one line is the tracker ``line=``
        with that line builds."""
        if int(crossing_capacity) < 0:
            raise ValueError("crossing_capacity must be >= 0")
        if lines is not None:
            if line is not None:
                raise ValueError("give line or lines, not both")
            lt = torch.as_tensor(lines, dtype=torch.float64)
            if lt.dim() not in (2, 3) or lt.shape[-1] != 4 or (lt.dim() == 3 and lt.shape[0] != n_streams):
                raise ValueError("lines: expected [L,4] or [%d,L,4], got %s" % (n_streams, tuple(lt.shape)))
            if not 1 <= lt.shape[-2] <= _lib.DD_MAX_LINES:
                raise ValueError("lines: need 1..%d lines per stream, got %d" % (_lib.DD_MAX_LINES, lt.shape[-2]))
            self.n_lines = int(lt.shape[-2])
            line = lt[..., 0, :] if self.n_lines == 1 else lt
        else:
            self.n_lines = 1
        self.crossing_capacity = int(crossing_capacity)
        self.lib = _lib.lib()
        self.pool_pages, self.pool_fraction, self.seg_pages, self.page_cap = pool_pages, pool_fraction, seg_pages, page_cap
        self.gallery_impl, self.cosine_ctas_per_sm, self.match_warps = gallery_impl, cosine_ctas_per_sm, match_warps
        self.gallery_stages, self.gallery_waves = gallery_stages, gallery_waves
        self.timeline, self.gallery_turns, self.engine_graphs = timeline, gallery_turns, engine_graphs
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("BatchedTracker runs on a CUDA device only (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.labels = list(labels)
        self.n_streams, self.max_tracks, self.max_dets, self.budget = n_streams, max_tracks, max_dets, budget
        self.max_age, self.n_init = max_age, n_init
        self.max_cosine_distance, self.max_iou_distance = max_cosine_distance, max_iou_distance
        n_chunks = max(1, min(int(n_chunks), n_streams))
        from .sharding import shard_range
        self.chunks = []
        with torch.cuda.device(self.device):
            for i in range(n_chunks):
                lo, hi = shard_range(n_streams, i, n_chunks)
                st = None if n_chunks == 1 else torch.cuda.Stream(device=self.device)
                self.chunks.append(_Chunk(self, lo, hi, st))
        self.cfg = self.chunks[0].cfg          # shape-independent fields (labels, thresholds, capacities per stream)
        self.v = _CatView(self)
        if line is None:                      # deepdish.py:739-744
            w, h = frame_size
            line = (float(int(w / 2)), 0.0, float(int(w / 2)), float(int(h)))
        lt = torch.as_tensor(line, dtype=torch.float64)
        self.line_per_stream = 1 if lt.dim() == (2 if self.n_lines == 1 else 3) else 0
        self.line = lt.to(self.device).contiguous()
        S, D = n_streams, max_dets
        cs = _lib.counts_shape(self.cfg)
        self.det_track_id = torch.full((S, D), -1, dtype=torch.int32, device=self.device)
        self.partial_counts = torch.zeros((2, n_chunks) + cs, dtype=torch.int64, device=self.device)
        self.total_counts = torch.zeros(cs, dtype=torch.int64, device=self.device)
        self._tick = 0
        self._aux = torch.cuda.Stream(device=self.device) if n_chunks > 1 else None
        self._poll_pool = any(len(c.segs) * c.cfg.seg_pages < self._worst_pages(c) for c in self.chunks) or budget is None
        self._engine = None           # native tick engine (csrc/dd_engine.cu), created at the first step()
        self._mode = None             # "eng": the last tick ran through the engine, "py": through the per-call path
        torch.cuda.synchronize(self.device)
        for c in self.chunks:
            _lib.check(self.lib.dd_tracker_init(c.state, c.cfgp, self._sp(c)), "dd_tracker_init")
        self.join()

    # ------------------------------------------------------------------------------------------
    def _eng(self):
        """The native tick engine of this tracker (dd_engine_create): one captured CUDA graph per chunk and tick, the
        event plumbing between chunk streams, the count summation and the pool polls behind ONE C call per tick."""
        if self._engine is None:
            P = len(self.chunks)
            states = (ctypes.c_void_p * P)(*[c.state for c in self.chunks])
            cfgs = (ctypes.POINTER(_lib.TrackerConfig) * P)(*[ctypes.pointer(c.cfg) for c in self.chunks])
            los = (ctypes.c_int32 * P)(*[c.lo for c in self.chunks])
            sts = (ctypes.c_void_p * P)(*[c.stream.cuda_stream if c.stream is not None else 0 for c in self.chunks])
            h = ctypes.c_void_p()
            _lib.check(self.lib.dd_engine_create(P, states, cfgs, los, sts,
                                                 ctypes.c_void_p(self._aux.cuda_stream if self._aux is not None else 0),
                                                 self.line.data_ptr(), self.line_per_stream, self.partial_counts.data_ptr(),
                                                 self.total_counts.data_ptr(), self.det_track_id.data_ptr(),
                                                 self.POLL_EVERY if self._poll_pool else 0, 1 if self.gallery_turns else 0,
                                                 ctypes.byref(h)),
                       "dd_engine_create")
            self._engine = h
            if not self.engine_graphs:        # the tick's kernels launched plainly by the engine instead of replayed graphs
                _lib.check(self.lib.dd_engine_set_graphs(h, 0), "dd_engine_set_graphs")
        return self._engine

    def __del__(self):
        try:
            if getattr(self, "_engine", None) is not None:
                torch.cuda.synchronize(self.device)
                self.lib.dd_engine_destroy(self._engine)
                self._engine = None
        except Exception:
            pass

    def _enter(self, mode):
        """Work is issued through the engine ("eng": step(), step_host_packed()) or call by call from Python ("py":
        predict(), update(), countline(), reduce_counts()).  A switch re-orders every stream first: dd_engine_step_host
        does not fork from the caller's stream, and the engine's count summation on the auxiliary stream writes
        total_counts, which reduce_counts() writes on the caller's stream."""
        if mode == self._mode:
            return
        if self._mode is not None and len(self.chunks) > 1:
            self.join()
            ev = self._cur().record_event()
            for c in self.chunks:
                c.stream.wait_event(ev)
            self._aux.wait_event(ev)
        self._mode = mode

    def _rebind(self, c):
        if self._engine is not None:
            _lib.check(self.lib.dd_engine_rebind(self._engine, self.chunks.index(c), c.state, c.cfgp), "dd_engine_rebind")

    def engine_stats(self):
        """(ticks stepped, kernels launched, host ms blocked in the run-ahead throttle) of the native engine."""
        if self._engine is None:
            return 0, 0, 0.0
        t, n, b = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_double(0)
        _lib.check(self.lib.dd_engine_stats(self._engine, ctypes.byref(t), ctypes.byref(n), ctypes.byref(b)), "dd_engine_stats")
        return t.value, n.value, b.value

    def _worst_pages(self, c):
        if self.budget is None:
            return float("inf")
        return (c.hi - c.lo) * self.max_tracks * ((self.budget + _lib.PAGE_ROWS - 1) // _lib.PAGE_ROWS)

    UPLOAD_BUFFERS = 2    # device blobs a chunk's ragged host batches rotate through (step_host_packed); 3 and 4 measured
                          # slower end to end (0.587 / 0.603 vs 0.569 ms per tick): the link, not the buffer depth, is the bound
    POLL_EVERY = 2        # ticks between the engine's polls of the pool counters (the forecast covers 8 appends ahead)

    def maintain(self, wait=False):
        """Grow gallery storage ahead of need, from the engine's latest poll of every chunk's pool counters
        (``wait=True``: from the state right now, synchronising).  A poll that is 3 ticks old is waited for, so the host
        never runs further ahead of the device than the 8-append forecast covers.
        Pool: segments are attached until the free pages cover the forecast (pages the live tracks can take within
        their next 8 appends) plus one page per detection slot (new tracks).  Unbounded galleries: the page table is doubled when the
        longest gallery is within 128 rows of its capacity."""
        for i, c in enumerate(self.chunks):
            st = c.stream if c.stream is not None else self._cur()
            if wait:
                st.synchronize()
                ctl = c.v["pool_ctl"][:4].cpu()
            elif self._mode == "eng" and self._engine is not None:
                out, tick = (ctypes.c_int32 * 4)(), ctypes.c_int64(-1)
                _lib.check(self.lib.dd_engine_pool_latest(self._engine, i, 3, out, ctypes.byref(tick)), "dd_engine_pool_latest")
                if tick.value < 0 or tick.value == getattr(c, "eng_poll_seen", -1):
                    continue
                c.eng_poll_seen = tick.value
                ctl = out
            else:
                continue
            free, attached, longest, forecast = int(ctl[0]), int(ctl[1]), int(ctl[2]), int(ctl[3])
            # new tracks take one page each: keep one worst-case tick of them (every detection a new track) in hand
            want = forecast + forecast // 4 + (c.hi - c.lo) * min(self.max_dets, self.max_tracks)
            grown = False
            while attached == len(c.segs) * c.cfg.seg_pages and free < want \
                    and attached < self._worst_pages(c) and len(c.segs) < _lib.DD_MAX_SEGS:
                c.grow_pool(ctypes.c_void_p(st.cuda_stream))
                free += c.cfg.seg_pages
                attached += c.cfg.seg_pages
                grown = True
            cap_rows = _lib.page_cap(c.cfg) * _lib.PAGE_ROWS
            if self.budget is None and longest + 128 >= cap_rows:
                st.synchronize()
                c.grow_page_table(2 * _lib.page_cap(c.cfg))
                grown = True
            if grown:
                self._rebind(c)
                c.eng_poll_seen = -1
                self._after_caller(c)

    def memory_bytes(self):
        """Device bytes of the tracker state: blobs + gallery page pool."""
        return sum(c.blob.numel() + c.pool_bytes() for c in self.chunks)

    def _cur(self):
        return torch.cuda.current_stream(self.device)

    def _sp(self, c):
        s = c.stream if c.stream is not None else self._cur()
        return ctypes.c_void_p(s.cuda_stream)

    def _after_caller(self, c):
        """Chunk c's stream waits for what the caller's stream holds now: a state edit made there (a re-laid-out blob
        filled by copies, new pool segments taken from the caller's stream's allocations, a gallery insert).
        dd_engine_step_host does not fork from the caller's stream, so without this a host-path tick could read the
        state before the edit.  The blob and the segments are only freed after a host synchronisation of the chunk's
        stream (re-layout, load_state_dict, the tracker's end), so using them on it needs no record_stream."""
        if c.stream is not None:
            c.stream.wait_stream(self._cur())

    def _fork(self, tensors=()):
        """Chunk streams wait for everything already enqueued on the caller's stream."""
        if len(self.chunks) == 1:
            return
        ev = self._cur().record_event()
        for c in self.chunks:
            c.stream.wait_event(ev)
            for t in tensors:
                t.record_stream(c.stream)

    def join(self):
        """Make the caller's current stream wait for all chunk streams and for the count summation (no host
        synchronisation)."""
        if len(self.chunks) == 1:
            return
        cur = self._cur()
        for c in self.chunks:
            c.done.record(c.stream)
            cur.wait_event(c.done)
        if self._engine is not None:
            _lib.check(self.lib.dd_engine_join(self._engine, ctypes.c_void_p(cur.cuda_stream)), "dd_engine_join")

    def _line_ptr(self, c):
        return self.line.data_ptr() + (c.lo * 32 * self.n_lines if self.line_per_stream else 0)

    def _check_batch(self, tlwh, conf, label, feat, count):
        S, D = self.n_streams, self.max_dets
        for t, dt, shape in ((tlwh, torch.float64, (S, D, 4)), (conf, torch.float32, (S, D)),
                             (label, torch.int32, (S, D)), (feat, torch.float32, (S, D, 128)),
                             (count, torch.int32, (S,))):
            if t.dtype != dt or tuple(t.shape) != shape or not t.is_cuda or not t.is_contiguous():
                raise ValueError("expected contiguous CUDA %s %s, got %s %s on %s"
                                 % (dt, shape, t.dtype, tuple(t.shape), t.device))

    @staticmethod
    def _ptrs(c, tlwh, conf, label, feat, count, ids):
        D = conf.shape[1]
        lo = c.lo
        return (tlwh.data_ptr() + lo * D * 32, conf.data_ptr() + lo * D * 4, label.data_ptr() + lo * D * 4,
                feat.data_ptr() + lo * D * 512, count.data_ptr() + lo * 4, ids.data_ptr() + lo * D * 4)

    # ------------------------------------------------------------------------------------------
    def predict(self):
        """Tracker.predict for every stream (tracker.py:51-57)."""
        self._enter("py")
        self._fork()
        for c in self.chunks:
            _lib.check(self.lib.dd_tracker_predict(c.state, c.cfgp, self._sp(c)), "dd_tracker_predict")
        self.join()

    def update(self, tlwh, conf, label, feat, count):
        """Tracker.update for every stream (tracker.py:59-93).

        tlwh f64 [S,Dmax,4], conf f32 [S,Dmax], label i32 [S,Dmax], feat f32 [S,Dmax,128], count i32 [S]
        -- device tensors, padded.  Returns det_track_id i32 [S,Dmax] (device; -1 = padding).

        When the gallery storage can grow (a pool smaller than the worst case, or unbounded galleries), the update first
        grows it from the exact counters (``maintain(wait=True)``): the call blocks until the work already enqueued on
        the tracker's streams has run."""
        self._check_batch(tlwh, conf, label, feat, count)
        self._enter("py")
        if self._poll_pool:
            self.maintain(wait=True)
        self._fork((tlwh, conf, label, feat, count))
        for c in self.chunks:
            p = self._ptrs(c, tlwh, conf, label, feat, count, self.det_track_id)
            _lib.check(self.lib.dd_tracker_update(c.state, c.cfgp, *p, self._sp(c)), "dd_tracker_update")
        self.join()
        return self.det_track_id

    def update_profiled(self, tlwh, conf, label, feat, count, events6):
        """update() that records 6 CUDA events (see dd_tracker_update_profiled); single chunk only."""
        if len(self.chunks) != 1:
            raise RuntimeError("update_profiled needs n_chunks=1")
        c = self.chunks[0]
        p = self._ptrs(c, tlwh, conf, label, feat, count, self.det_track_id)
        _lib.check(self.lib.dd_tracker_update_profiled(c.state, c.cfgp, *p, self._sp(c), events6),
                   "dd_tracker_update_profiled")
        return self.det_track_id

    def new_events(self, n=6):
        arr = (ctypes.c_void_p * n)()
        for i in range(n):
            h = ctypes.c_void_p()
            _lib.check(self.lib.dd_event_create(ctypes.byref(h)), "dd_event_create")
            arr[i] = h
        return arr

    def elapsed_ms(self, start, end):
        ms = ctypes.c_float(0)
        _lib.check(self.lib.dd_event_elapsed_ms(start, end, ctypes.byref(ms)), "dd_event_elapsed_ms")
        return ms.value

    def countline(self):
        """Count-line step (deepdish.py:1041-1112) on the state left by update()."""
        self._enter("py")
        self._fork()
        for c in self.chunks:
            _lib.check(self.lib.dd_tracker_countline(c.state, c.cfgp, self._line_ptr(c), self.line_per_stream,
                                                     self._sp(c)), "dd_tracker_countline")
        self.join()

    def _check_present(self, present):
        S = self.n_streams
        if not isinstance(present, torch.Tensor) or present.dtype not in (torch.bool, torch.uint8) \
                or tuple(present.shape) != (S,) or present.device != self.device or not present.is_contiguous():
            raise ValueError("present: expected a contiguous bool or uint8 tensor (%d,) on %s, got %s"
                             % (S, self.device, "%s %s on %s" % (present.dtype, tuple(present.shape), present.device)
                                if isinstance(present, torch.Tensor) else type(present).__name__))

    def step(self, batch, join=True, reduce=False, present=None, out_events_host=None):
        """One tick (predict + update + count-line [+ count reduction into total_counts]) for a SceneBatch-like object
        of device tensors: ONE call into the native engine, which launches one captured graph per chunk.  join=False
        only enqueues (call join()).

        present: frame presence of each stream this tick, a contiguous CUDA bool / uint8 tensor [S] on the tracker's
        device (None: every stream has a frame).  A stream without a frame is left exactly as it is -- no predict, no
        update, no gallery append, no count-line step, as the reference leaves the tracker of a camera that delivers no
        frame --, its rows of the batch (count included) are ignored and its det_track_id row is -1.  Its tracks
        survive any length of absence and are predicted once at its next frame.

        out_events_host: a buffer of ``new_crossings_buffer()``; the tick's crossing records are copied into it behind
        the tick (read them with ``crossings(out_events_host)`` once the caller's stream has been synchronised after
        join())."""
        tlwh, conf, label, feat, count = batch.tlwh, batch.conf, batch.label, batch.feat, batch.count
        if out_events_host is not None:
            self._check_crossings_buffer(out_events_host)
        self._check_batch(tlwh, conf, label, feat, count)
        if present is not None:
            self._check_present(present)
        self._enter("eng")
        if self._poll_pool:
            self.maintain()
        if len(self.chunks) > 1:
            for t in (tlwh, conf, label, feat, count) + ((present,) if present is not None else ()):
                for c in self.chunks:
                    t.record_stream(c.stream)
        _lib.check(self.lib.dd_engine_step_present(self._eng(), tlwh.data_ptr(), conf.data_ptr(), label.data_ptr(),
                                                   feat.data_ptr(), count.data_ptr(),
                                                   present.data_ptr() if present is not None else None,
                                                   1 if reduce else 0, ctypes.c_void_p(self._cur().cuda_stream)),
                   "dd_engine_step_present")
        if out_events_host is not None:
            self._copy_events(out_events_host)
        self._tick += 1
        if join:
            self.join()
        return self.det_track_id

    # ------------------------------------------------------------------------------------------
    def _staging_small(self, c):
        if getattr(c, "staging_small", None) is None:
            n, D = c.hi - c.lo, self.max_dets
            c.staging_small = (torch.empty((n, D, 4), dtype=torch.float64, device=self.device),
                               torch.empty((n, D), dtype=torch.float32, device=self.device),
                               torch.empty((n, D), dtype=torch.int32, device=self.device),
                               torch.empty((n,), dtype=torch.int32, device=self.device))
        return c.staging_small

    def pack_host(self, batch, present=None):
        """Ragged host form of a padded batch (the batched equivalent of the reference's per-stream list of
        Detection objects, deepdish.py:1014): per chunk ONE pinned byte blob
        ``[i32 offsets[n+1] | f64 tlwh[N,4] | f32 conf[N] | i32 label[N] | f32 feat[N,128]]`` holding only the
        detections that exist, so a tick uploads one copy per chunk and no padding.
        present: frame presence of each stream (bool-like [S], host or device; see step()).  Each blob then ends with
        a ``u8 present[n]`` section, absent streams own no entries and their counts are ignored; the presence rides in
        the tick's one upload."""
        from . import ragged
        cnt = batch.count.cpu().numpy()
        tlwh, conf = batch.tlwh.cpu().numpy(), batch.conf.cpu().numpy()
        label, feat = batch.label.cpu().numpy(), batch.feat.cpu().numpy()
        if present is not None:
            present = (present.cpu().numpy() if isinstance(present, torch.Tensor) else np.asarray(present)).astype(bool)
            if present.shape != (self.n_streams,):
                raise ValueError("present must have shape (%d,), got %s" % (self.n_streams, present.shape))
            cnt = np.where(present, cnt, 0)
        if int(cnt.max(initial=0)) > self.max_dets:
            raise RuntimeError("detection capacity exceeded (max_dets=%d)" % self.max_dets)
        out = []
        for c in self.chunks:
            pr = present[c.lo:c.hi] if present is not None else None
            _, total = ragged.section_offsets(c.hi - c.lo, int(cnt[c.lo:c.hi].sum()), pr is not None)
            blob = torch.empty(max(total, 16), dtype=torch.uint8).pin_memory()
            _, total, sections = ragged.pack(tlwh[c.lo:c.hi], conf[c.lo:c.hi], label[c.lo:c.hi], feat[c.lo:c.hi],
                                             cnt[c.lo:c.hi], out=blob.numpy(), present=pr)
            out.append((blob, total, sections))
        return out

    @staticmethod
    def packed_nbytes(packed):
        return sum(p[1] for p in packed)

    def step_host_packed(self, packed, out_ids_host=None, out_events_host=None):
        """End-to-end tick from a ragged pinned host batch (``pack_host``): one call into the native engine
        (dd_engine_step_host).  Per chunk: ONE H2D copy on the chunk's own copy stream into a double-buffered device
        blob -- so the upload of tick k + 1 runs under the kernels of tick k --, then on the chunk's compute stream the
        captured tick reading the blob in place, its partial count reduction and (optionally) the D2H copy of the
        det->track ids.  The pinned blobs must stay alive until their copy has run.  Unlike step(), the chunk streams do
        not wait for the caller's stream; this tracker's own edits made there (maintain(), gallery_insert) are ordered
        before the next tick of the chunk they touch.  Returns total_counts (device;
        valid on the caller's stream after join() or all_reduce_counts()).
        A batch packed with frame presence (``pack_host(batch, present)``) runs the tick of step(present=...)
        (dd_engine_step_host_present); every chunk of it must carry the presence section or none.
        out_events_host: as in step(); the copy runs beside the ids' read-back, off the chunks' compute streams."""
        if out_events_host is not None:
            self._check_crossings_buffer(out_events_host)
        kinds = {len(p[2]) for p in packed}
        if len(packed) != len(self.chunks) or not kinds <= {4, 5} or len(kinds) != 1:
            raise ValueError("packed: expected one blob per chunk (%d), all with or all without a presence section"
                             % len(self.chunks))
        n_off = kinds.pop()
        self._enter("eng")
        if self._poll_pool:
            self.maintain()
        eng = self._eng()
        P = len(self.chunks)
        if getattr(self, "_host_bound", None) is None:
            for i, c in enumerate(self.chunks):
                n = c.hi - c.lo
                cap = 4 * (n + 1) + 64 + n * self.max_dets * (32 + 4 + 4 + 512) + n + 16
                c.blob_dev = [torch.empty(cap, dtype=torch.uint8, device=self.device) for _ in range(self.UPLOAD_BUFFERS)]
                ptrs = (ctypes.c_void_p * len(c.blob_dev))(*[b.data_ptr() for b in c.blob_dev])
                t, cf, lb, ct = self._staging_small(c)
                _lib.check(self.lib.dd_engine_bind_host(eng, i, ptrs, len(c.blob_dev), cap,
                                                        t.data_ptr(), cf.data_ptr(), lb.data_ptr(), ct.data_ptr()),
                           "dd_engine_bind_host")
            self._host_bound = ((ctypes.c_void_p * P)(), (ctypes.c_uint64 * P)(), (ctypes.c_int64 * (5 * P))())
        blobs, sizes, offs = self._host_bound
        for i, (blob, total, sec) in enumerate(packed):
            blobs[i], sizes[i] = blob.data_ptr(), total
            offs[n_off * i:n_off * (i + 1)] = list(sec)
        fn = self.lib.dd_engine_step_host_present if n_off == 5 else self.lib.dd_engine_step_host
        _lib.check(fn(eng, blobs, sizes, offs, out_ids_host.data_ptr() if out_ids_host is not None else None,
                      ctypes.c_void_p(self._cur().cuda_stream)), fn.__name__)
        if out_events_host is not None:
            self._copy_events(out_events_host)
        self._tick += 1
        return self.total_counts

    # ------------------------------------------------------------------------------------------
    def _crossings_words(self):
        return len(self.chunks) * 4 * (1 + self.crossing_capacity)

    def new_crossings_buffer(self):
        """Pinned host buffer for ``step(..., out_events_host=)`` / ``step_host_packed(..., out_events_host=)``: every
        chunk's crossing list (header + ``crossing_capacity`` records)."""
        if self.crossing_capacity <= 0:
            raise RuntimeError("crossing records are off: construct the tracker with crossing_capacity > 0")
        return torch.zeros(self._crossings_words(), dtype=torch.int32).pin_memory()

    def _check_crossings_buffer(self, buf):
        if self.crossing_capacity <= 0:
            raise RuntimeError("crossing records are off: construct the tracker with crossing_capacity > 0")
        if not isinstance(buf, torch.Tensor) or buf.dtype != torch.int32 or buf.is_cuda or not buf.is_pinned() \
                or not buf.is_contiguous() or buf.numel() != self._crossings_words():
            raise ValueError("out_events_host: expected a buffer of new_crossings_buffer() (pinned int32 [%d])"
                             % self._crossings_words())

    def _copy_events(self, buf):
        _lib.check(self.lib.dd_engine_copy_events(self._eng(), buf.data_ptr(), ctypes.c_void_p(self._cur().cuda_stream)),
                   "dd_engine_copy_events")

    def crossings(self, host_buffer=None):
        """The count-line crossings of the last tick (or per-call ``countline()``) as ``Crossings`` arrays
        (``LineCrossings`` with several lines per stream).
        host_buffer: a buffer a step copied them into (valid once that copy has completed: after join() and a
        synchronisation of the caller's stream); None: read from the device, which joins and synchronises.
        Raises RuntimeError naming the chunk whose list overflowed crossing_capacity (records are never dropped
        silently), and when the tracker was built without crossing records."""
        if self.crossing_capacity <= 0:
            raise RuntimeError("crossing records are off: construct the tracker with crossing_capacity > 0")
        cap = self.crossing_capacity
        if host_buffer is None:
            self.join()
            torch.cuda.synchronize(self.device)
            lists = [c.v["events"].cpu().numpy() for c in self.chunks]
        else:
            self._check_crossings_buffer(host_buffer)
            lists = host_buffer.numpy().reshape(len(self.chunks), cap + 1, 4)
        parts = []
        for i, (c, ev) in enumerate(zip(self.chunks, lists)):
            n = int(ev[0, 0])
            if n > cap:
                raise RuntimeError("crossing list of chunk %d (streams %d..%d) overflowed: %d records this tick, "
                                   "crossing_capacity=%d" % (i, c.lo, c.hi - 1, n, cap))
            rec = ev[1:1 + n]
            rec = rec[np.argsort(rec[:, 0], kind="stable")]          # by stream; positions keep the order within one
            parts.append(rec + np.array([c.lo, 0, 0, 0], dtype=np.int32))
        r = np.concatenate(parts).astype(np.int32, copy=False)
        if self.n_lines > 1:          # column word = column + 4 line
            return LineCrossings(r[:, 0].copy(), r[:, 1].copy(), r[:, 2].copy(), r[:, 3] & 3, r[:, 3] >> 2)
        return Crossings(r[:, 0].copy(), r[:, 1].copy(), r[:, 2].copy(), r[:, 3].copy())

    def reduce_counts(self):
        """Sum the per-stream counters -> i64 [C,4] (pos, neg, int, del per label; [L,C,4] with L > 1 lines), this GPU
        only.  Runs on the caller's stream, behind every chunk."""
        self._enter("py")
        self.join()
        sp = ctypes.c_void_p(self._cur().cuda_stream)
        for i, c in enumerate(self.chunks):
            _lib.check(self.lib.dd_tracker_count_reduce(c.state, c.cfgp, self.partial_counts[0, i].data_ptr(), sp),
                       "dd_tracker_count_reduce")
        torch.sum(self.partial_counts[0], dim=0, out=self.total_counts)
        return self.total_counts

    def all_reduce_counts(self, reduced=False, async_op=False):
        """[C,4] ([L,C,4]) counters summed over streams and, over NCCL, ranks (the path's only collective).
        reduced=True: total_counts already holds this tick's local sum (step(reduce=True) / step_host_packed).
        async_op=True: the all-reduce runs on NCCL's own stream on a copy of the counters (two alternating buffers)
        and the caller's stream is not made to wait, so ranks do not rendezvous every tick; the returned tensor is
        valid after wait_counts()."""
        t = self.total_counts if reduced else self.reduce_counts()
        import torch.distributed as dist
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        if async_op and not multi:
            return t                    # one rank: nothing to exchange, total_counts is the result (valid after join())
        if not async_op:
            self._wait_sum()
            if multi:
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return t
        if not hasattr(self, "_ar_buf"):
            self._ar_buf = [torch.zeros_like(self.total_counts) for _ in range(2)]
            self._ar_work = [None, None]
            self._ar_turn = 0
        k = self._ar_turn
        self._ar_turn ^= 1
        # the stream total_counts is produced on: the engine sums several chunks on the auxiliary stream, reduce_counts()
        # on the caller's
        side = self._aux if self._mode == "eng" and self._aux is not None else self._cur()
        with torch.cuda.stream(side):
            if self._ar_work[k] is not None:
                self._ar_work[k].wait()
            self._ar_buf[k].copy_(t)
            self._ar_work[k] = dist.all_reduce(self._ar_buf[k], op=dist.ReduceOp.SUM, async_op=True) if multi else None
            self._ar_done = side.record_event()
        return self._ar_buf[k]

    def _wait_sum(self):
        """The caller's stream waits for the engine's latest count summation (reduce_counts() sums on the caller's
        stream)."""
        if self._engine is not None:
            _lib.check(self.lib.dd_engine_wait_counts(self._engine, ctypes.c_void_p(self._cur().cuda_stream)),
                       "dd_engine_wait_counts")

    def wait_counts(self):
        """Make the caller's stream wait for every outstanding asynchronous count all-reduce."""
        for k, w in enumerate(getattr(self, "_ar_work", [])):
            if w is not None:
                w.wait()
                self._ar_work[k] = None
        if getattr(self, "_ar_done", None) is not None:
            self._cur().wait_event(self._ar_done)

    def status(self):
        self.join()
        out = 0
        for c in self.chunks:
            flags = ctypes.c_int32(0)
            _lib.check(self.lib.dd_tracker_status(c.state, c.cfgp, ctypes.byref(flags), self._sp(c)),
                       "dd_tracker_status")
            out |= flags.value
        return out

    def check(self):
        """Raise if any stream overflowed its capacities (never silently truncated)."""
        f = self.status()
        # storage first: once appends are dropped the tracks that got no gallery depend on the order the CTAs reached the
        # pool, and what follows (spurious new tracks, even a track overflow) is a consequence
        if f & _lib.FLAG_POOL_EXHAUSTED:
            raise RuntimeError("gallery page pool exhausted (a feature was not appended); construct the tracker with a "
                               "larger pool_pages / pool_fraction")
        if f & _lib.FLAG_TRACK_OVERFLOW:
            raise RuntimeError("track capacity exceeded (max_tracks=%d)" % self.max_tracks)
        if f & _lib.FLAG_DET_OVERFLOW:
            raise RuntimeError("detection capacity exceeded (max_dets=%d)" % self.max_dets)
        if f & _lib.FLAG_LSAP_INFEASIBLE:
            raise ValueError("cost matrix is infeasible")
        if f & _lib.FLAG_GALLERY_OVERFLOW:
            raise RuntimeError("a gallery outgrew its page table (page_cap); call maintain() more often")
        if f & _lib.FLAG_BAD_LABEL:
            raise ValueError("a detection label is outside [0, n_labels)")

    # ------------------------------------------------------------------------------------------
    def state_dict(self):
        """Checkpoint of the whole tracker state (SURVEY.md section 5: the reference never saves tracker
        state; only its counters survive a restart).  Host copies of every chunk's blob + the tick counter."""
        self.join()
        torch.cuda.synchronize(self.device)
        return {"blobs": [c.blob.cpu() for c in self.chunks], "tick": self._tick,
                "pools": [[(a.cpu(), b.cpu()) for a, b in c.segs] for c in self.chunks],
                "page_caps": [_lib.page_cap(c.cfg) for c in self.chunks],
                "shape": (self.n_streams, self.max_tracks, self.max_dets, self.budget, len(self.labels),
                          len(self.chunks), self.chunks[0].cfg.seg_pages), "total_counts": self.total_counts.cpu(),
                "n_lines": self.n_lines}

    def load_state_dict(self, sd):
        if int(sd.get("n_lines", 1)) != self.n_lines:       # checkpoints from before count lines had one line
            raise ValueError("checkpoint has %d count lines per stream, this tracker %d"
                             % (int(sd.get("n_lines", 1)), self.n_lines))
        shape = (self.n_streams, self.max_tracks, self.max_dets, self.budget, len(self.labels), len(self.chunks),
                 self.chunks[0].cfg.seg_pages)
        if tuple(sd["shape"]) != shape:
            raise ValueError("checkpoint shape %s does not match tracker %s" % (tuple(sd["shape"]), shape))
        self.join()
        torch.cuda.synchronize(self.device)
        for c, b, pool, cap in zip(self.chunks, sd["blobs"], sd["pools"], sd["page_caps"]):
            if len(pool) < len(c.segs):
                raise ValueError("checkpoint has fewer pool segments (%d) than this tracker (%d)" % (len(pool), len(c.segs)))
            while len(c.segs) < len(pool):        # page ids in the checkpoint refer to every segment it had
                c._alloc_seg()
            c.cfg.n_segs = len(c.segs)
            if cap != _lib.page_cap(c.cfg):
                c.cfg.page_cap = cap
                c._bind()
            c.blob.copy_(b.to(self.device))
            for (a, h), (pa, ph) in zip(c.segs, pool):
                a.copy_(pa.to(self.device))
                h.copy_(ph.to(self.device))
            c.eng_poll_seen = -1
            self._rebind(c)
        self.total_counts.copy_(sd["total_counts"].to(self.device))
        self._tick = int(sd["tick"])
        torch.cuda.synchronize(self.device)

    def host_view(self, names=None, streams=None):
        """numpy copies of state arrays (optionally a subset of streams) for inspection / tests."""
        names = names or [n for n in self.v.keys() if n not in ("ptab", "free_stack", "pool_ctl", "work_rec", "cost", "gate", "det_featn", "det_feath", "work", "work_ctl", "tick_args", "timeline", "tick_present", "events")]
        out = {}
        for n in names:
            t = self.v[n]
            if streams is not None:
                t = t[torch.as_tensor(streams, device=self.device)]
            out[n] = t.cpu().numpy()
        return out

    def _chunk_of(self, stream):
        for c in self.chunks:
            if c.lo <= stream < c.hi:
                return c
        raise IndexError("stream %d out of range" % stream)

    def gallery(self, stream, slot):
        """metric.samples of one slot (nn_matching.py:132-154): its unit-normalised gallery rows, oldest first, as a
        float32 CUDA tensor [len, 128] (dd_tracker_gallery_read)."""
        c = self._chunk_of(stream)
        self.join()
        n = int(c.v["gal_len"][stream - c.lo, slot])
        out = torch.empty((n, 128), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.dd_tracker_gallery_read(c.state, c.cfgp, stream - c.lo, slot, out.data_ptr(), n,
                                                    ctypes.c_void_p(self._cur().cuda_stream)), "dd_tracker_gallery_read")
        return out

    def gallery_insert(self, stream, slot, feature, before_newest=False):
        """Host edit: append one unit-normalised feature to a slot's gallery (before its newest row when
        ``before_newest``), as metric.partial_fit would (dd_tracker_gallery_insert)."""
        c = self._chunk_of(stream)
        self.join()
        f = torch.as_tensor(feature, dtype=torch.float32).to(self.device).contiguous()
        if f.numel() != 128:
            raise ValueError("feature must have 128 components")
        _lib.check(self.lib.dd_tracker_gallery_insert(c.state, c.cfgp, stream - c.lo, slot, f.data_ptr(),
                                                      1 if before_newest else 0,
                                                      ctypes.c_void_p(self._cur().cuda_stream)), "dd_tracker_gallery_insert")
        self._after_caller(c)
        if self._poll_pool:
            self.maintain(wait=True)

    def gallery_vectors(self):
        """Total gallery vectors of confirmed live tracks (G in SURVEY.md section 8d), per stream."""
        self.join()
        outs = []
        for c in self.chunks:
            S, T = c.hi - c.lo, self.max_tracks
            valid = torch.arange(T, device=self.device)[None, :] < c.v["n_tracks"][:, None]
            rows = torch.arange(S, device=self.device)[:, None].expand(S, T)[valid]
            slots = c.v["order"].long()[valid]
            live = torch.zeros((S, T), dtype=torch.bool, device=self.device)
            live[rows, slots] = True
            outs.append((c.v["gal_len"] * (live & (c.v["state"] == 2))).sum(dim=1))
        return torch.cat(outs)
