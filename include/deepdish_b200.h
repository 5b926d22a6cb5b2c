/* deepdish_b200.h -- C ABI of the B200-native tracking-by-detection hot path of AdaptiveCity/deepdish.
 *
 * Drop-in boundary (SURVEY.md section 8b).  The reference is 100 % Python and has no FFI of its own;
 * each entry point below names the reference interface (file:line under /root/reference) whose
 * arithmetic it replaces.  The reference-side binding a maintainer would add is a ctypes stub, shown in
 * INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name starts with `host_`;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls are asynchronous
 *     with respect to the host, outputs are valid after the stream is synchronised;
 *   - return value: DD_OK or a negative DD_ERR_* code; nothing is thrown across the ABI;
 *   - the caller (PyTorch, cudaMalloc, ...) owns every buffer; the library keeps no state of its own beyond per-device
 *     caches of the kernel attributes it has opted into (shared-memory sizes, carve-out);
 *   - row-major, densely packed arrays; f64 = double, f32 = float, i32 = int32_t, i64 = int64_t.
 */
#ifndef DEEPDISH_B200_H
#define DEEPDISH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DD_OK             0
#define DD_ERR_INVALID   (-1)   /* bad argument (size, NULL, unsupported feature dim ...)            */
#define DD_ERR_CUDA      (-2)   /* a CUDA runtime call / launch failed                               */
#define DD_ERR_CAPACITY  (-3)   /* T > max_tracks or D > max_dets: never silently truncated          */

#define DD_MAX_LABELS   128
#define DD_FEAT_DIM     128     /* MARS re-ID feature width (tools/generate_detections.py:137-140)   */

/* track states, deep_sort/track.py:15-17 (0 = slot unused) */
#define DD_STATE_FREE       0
#define DD_STATE_TENTATIVE  1
#define DD_STATE_CONFIRMED  2
#define DD_STATE_DELETED    3

/* per-stream error bits in the `err` state array (sticky; read with dd_tracker_status) */
#define DD_FLAG_TRACK_OVERFLOW  1   /* needed more than max_tracks slots              */
#define DD_FLAG_DET_OVERFLOW    2   /* det_count[s] > max_dets                        */
#define DD_FLAG_LSAP_INFEASIBLE 4   /* scipy would raise ValueError (NaN / inf cost)  */
#define DD_FLAG_POOL_EXHAUSTED  8   /* the gallery page pool had no free page: a feature was NOT appended */
#define DD_FLAG_GALLERY_OVERFLOW 16 /* an unbounded gallery outgrew its page table (page_cap): not appended */
#define DD_FLAG_BAD_LABEL       32  /* det_label outside [0, n_labels): the vote was skipped                */

/* Gallery storage: 16-row pages drawn from a pool (nn_matching.py:137-154 keeps a growing Python list per
 * track; nn_budget=None -- the only way deepdish.py:515-516 builds its metric -- never trims it). */
#define DD_PAGE_ROWS        16
#define DD_PAGE_F32_BYTES   8192    /* 16 rows x 128 f32, row-major                                          */
#define DD_PAGE_F16_BYTES   4096    /* the same rows rounded to half, stored in mma fragment order (below)   */
#define DD_MAX_SEGS         16      /* pool segments (equal size, attached one by one as the pool grows)     */

const char* dd_version(void);

/* ------------------------------------------------------------------------------------------------
 * Batched DeepSORT tracker: S independent streams, one `deep_sort.tracker.Tracker` each.
 * Replaces deep_sort/tracker.py:40-138 (+ track.py, kalman_filter.py, nn_matching.py,
 * iou_matching.py, linear_assignment.py and scipy.optimize.linear_sum_assignment underneath).
 * ---------------------------------------------------------------------------------------------- */
typedef struct dd_tracker_config {
    int32_t n_streams;          /* S                                                                */
    int32_t max_tracks;         /* Tmax: slots per stream (live + deleted-this-tick + new)          */
    int32_t max_dets;           /* Dmax: detections per stream per tick                             */
    int32_t budget;             /* nn_budget: gallery vectors kept per track (nn_matching.py:150);
                                   0 = None: unbounded, what deepdish.py:515-516 always passes      */
    int32_t feat_dim;           /* must be DD_FEAT_DIM                                              */
    int32_t n_labels;           /* C <= DD_MAX_LABELS                                               */
    int32_t max_age;            /* tracker.py:40 (deepdish.py:1418 default 60)                      */
    int32_t n_init;             /* tracker.py:40                                                    */
    double  max_cosine_distance;/* metric.matching_threshold (deepdish.py:1412 default 0.2)         */
    double  max_iou_distance;   /* tracker.py:40 default 0.7                                        */
    int32_t label_motorbike;    /* label ids for the track.py:175-183 special case, -1 if absent    */
    int32_t label_bicycle;
    int32_t label_rank[DD_MAX_LABELS]; /* rank of each label NAME in ascending string order
                                          (tie-break of the reverse sort in track.py:170)           */
    /* gallery page pool (caller-owned device memory, like the blob) */
    int32_t page_cap;           /* page-table entries per slot; budget > 0: ceil(budget / 16) (0 = that default);
                                   budget == 0: rows a gallery can reach before the caller must re-layout with a
                                   larger page_cap (DD_FLAG_GALLERY_OVERFLOW when it does not)          */
    int32_t seg_pages;          /* pages per pool segment, a power of two                               */
    int32_t n_segs;             /* segments attached so far, 1..DD_MAX_SEGS (dd_tracker_pool_attach)    */
    /* per-tracker tuning (A/B measurements; 0 = default everywhere) */
    int32_t gallery_impl;       /* 0 = default (the half-precision producer / mma / checker stream), 1 = exact f32
                                   pass (bit-identical to 0; defines the result)                        */
    int32_t cosine_ctas_per_sm; /* impl 0: warp triples (producer, mma, checker) per SM (default 7; at most 7, 8 with
                                   gallery_waves)                                                       */
    int32_t match_warps;        /* matching kernel: 0 = by problem size, 1 / 4 / 8 warps per stream     */
    int32_t gallery_stages;     /* impl 0: 4 KB ring stages per warp triple (default 4)                 */
    int32_t gallery_waves;      /* impl 0: 0 = one persistent CTA per SM holding all the triples (default); W > 0 = one
                                   triple per CTA, SMs x triples x W CTAs that each stream a bounded share of the work
                                   list and exit (measured equal on C3, kept as an A/B knob)                         */
    int32_t event_cap;          /* crossing records kept per tick (count-line events, `events` below); 0 = off: no
                                   `events` section and the count-line step exactly as without it; < 0 is invalid */
    int32_t timeline;           /* != 0: every tick kernel stamps its first CTA's start and its last CTA's end
                                   (%globaltimer, ns) into the blob's `timeline` words (benchmarks/timeline.py)    */
    uint64_t pool_f32[DD_MAX_SEGS]; /* device pointers, seg_pages x DD_PAGE_F32_BYTES each, 16-byte aligned */
    uint64_t pool_f16[DD_MAX_SEGS]; /* device pointers, seg_pages x DD_PAGE_F16_BYTES each, 16-byte aligned */
} dd_tracker_config;

/* Half page layout ("fragment order"): the 16-byte chunk c (= 8 consecutive halves, c = 0..15) of row r sits at
 * byte ((c >> 2) * 2 + (r >> 3)) * 512 + ((r & 7) * 4 + (c & 3)) * 16 of the page, so that lane 4 g + t of a warp
 * reads its mma.m16n8k16 A operands for rows g and g + 8 with fully coalesced (and, from shared memory,
 * conflict-free) 16-byte loads. */

/* Byte offsets of every array inside the caller-owned state blob (all multiples of 256). */
typedef struct dd_tracker_layout {
    uint64_t total_bytes;
    /* per stream */
    uint64_t n_tracks;      /* i32 [S]            live tracks                                       */
    uint64_t next_id;       /* i32 [S]            tracker.py:49 _next_id                            */
    uint64_t n_deleted;     /* i32 [S]            len(tracker.deleted_tracks)                       */
    uint64_t err;           /* i32 [S]            DD_FLAG_* bits                                    */
    uint64_t order;         /* i32 [S,Tmax]       slot of the k-th live track (creation order)      */
    uint64_t deleted;       /* i32 [S,Tmax]       slots deleted by the last update (creation order) */
    uint64_t counts;        /* i64 [S,C,4]        pos, neg, int, del per label                      */
    /* per slot */
    uint64_t mean;          /* f64 [S,Tmax,8]                                                       */
    uint64_t cov;           /* f64 [S,Tmax,8,8]                                                     */
    uint64_t track_id;      /* i32 [S,Tmax]                                                         */
    uint64_t hits;          /* i32 [S,Tmax]                                                         */
    uint64_t age;           /* i32 [S,Tmax]                                                         */
    uint64_t tsu;           /* i32 [S,Tmax]       time_since_update                                 */
    uint64_t state;         /* i32 [S,Tmax]       DD_STATE_*                                        */
    uint64_t gal_len;       /* i32 [S,Tmax]       valid gallery vectors (<= budget when budget > 0)  */
    uint64_t gal_pos;       /* i32 [S,Tmax]       next write position (ring position when budget > 0) */
    uint64_t gal_np;        /* i32 [S,Tmax]       pages the slot holds                              */
    uint64_t ptab;          /* i32 [S,Tmax,page_cap]  page ids: gallery row p lives in page ptab[p / 16], row p % 16;
                                                  rows are unit-normalised features                 */
    uint64_t free_stack;    /* i32 [DD_MAX_SEGS * seg_pages]  free page ids                         */
    uint64_t pool_ctl;      /* i32 [64]           [0] free pages, [1] pages attached, [2] longest gallery so far,
                                                  [3] forecast: tracks updated this tick that need another page within
                                                  their next 8 appends (rebuilt every tick; tracks not updated this
                                                  tick and new tracks come on top) */
    uint64_t lab_cnt;       /* i32 [S,Tmax,C]     votes per label (track.py:75-80,147-151)          */
    uint64_t lab_sum;       /* f64 [S,Tmax,C]     sum of confidences per label                      */
    uint64_t path_n;        /* i32 [S,Tmax]       points in the count-line path db                  */
    uint64_t path_last;     /* f64 [S,Tmax,2]     last bottom-centre point                          */
    uint64_t path_crossed;  /* i32 [S,Tmax]       any path segment crossed the line                 */
    /* per-tick scratch / outputs */
    uint64_t gate;          /* u32 [S,Tmax,ceil(Dmax/32)]  bit d set: d^2 <= chi2inv95[4]           */
    uint64_t cost;          /* f32 [S,Tmax,Dmax]  min cosine distance (valid where gate bit set)    */
    uint64_t det_xyah;      /* f64 [S,Dmax,4]                                                       */
    uint64_t det_featn;     /* f32 [S,Dmax,128]   unit-normalised detection features                */
    uint64_t det_slot;      /* i32 [S,Dmax]       slot the detection was applied to                 */
    uint64_t det_kind;      /* i32 [S,Dmax]       0 none, 1 Kalman update, 2 new track              */
    uint64_t cdesc;         /* i32 [S,Tmax,4]     per track index: slot, gallery rows, #gate-passing detections
                                                  (0 = nothing to stream), pages                            */
    uint64_t work;          /* i32 [S*Tmax]       work list of the gallery kernel: s * Tmax + track index of
                                                  every track with a gate-passing detection (any order)     */
    uint64_t work_ctl;      /* i32 [64]           [0] = entries in `work`, [32] = claim cursor              */
    uint64_t work_rec;      /* i32 [S*Tmax,16]    one self-contained record per work-list entry (same order): stream * Tmax
                                                  + slot, stream, gallery rows, #gate-passing detections, pages, gate
                                                  words 0 and 1, detections this tick, page ids 0..7 -- all the gallery
                                                  kernel's producer warps need to start the bulk copies of a track   */
    uint64_t det_feath;     /* f16 [S,Dmax,128]   half copy of det_featn                                     */
    uint64_t tick_args;     /* 256 bytes          per-tick input pointers of a captured tick (written by dd_engine_step) */
    uint64_t timeline;      /* u64 [64,8,2]       config.timeline: per engine tick (mod 64) and kernel (prep, gate, gallery, match,
                                                  apply, count-line, count-reduce): min start / max end in ns; the caller
                                                  initialises starts to ~0 and ends to 0                         */
    uint64_t tick_present;  /* i32 [S]            1: the stream had a frame in the last tick (written by every tick's
                                                  detection prep; the per-call update marks every stream present)  */
    uint64_t events;        /* i32 [4 + 4 event_cap] crossing records of the last count-line step, 0 bytes when event_cap = 0
                                                  (then events == total_bytes).  header[0] = records the step produced (may
                                                  exceed event_cap: the list overflowed, records past event_cap are counted
                                                  but not written), header[1..3] unused; then event_cap records
                                                  {stream (index within this blob), track_id, label, column}, one per counter
                                                  increment of the step: column 0 / 1 = a live track crossed the line and
                                                  added 1 to pos / neg and to int of `label` (the label get_label gave the
                                                  counter), column 3 = the del increment of the last deleted track.  A
                                                  stream's records keep the order of tracker.tracks, its deletion record
                                                  last; streams interleave.  Reset at the start of every count-line step */
} dd_tracker_layout;

/* Host-only arithmetic: fills `host_out`.  No CUDA call. */
int dd_tracker_layout_query(const dd_tracker_config* host_cfg, dd_tracker_layout* host_out);

/* Zero the blob, set _next_id = 1 (tracker.py:46-49) and put the pages of the host_cfg->n_segs attached
 * segments on the free stack. */
int dd_tracker_init(void* state, const dd_tracker_config* host_cfg, void* stream);

/* Grow the page pool: the caller has allocated segment number host_cfg->n_segs - 1 (pool_f32 / pool_f16 entries
 * filled, n_segs already incremented); its seg_pages page ids go on the free stack.  Must not run concurrently
 * with a tick of the same tracker (same stream, or ordered by events). */
int dd_tracker_pool_attach(void* state, const dd_tracker_config* host_cfg, void* stream);

/* metric.samples[track] (nn_matching.py:132-154): the gallery of one slot, oldest row first, as unit-normalised
 * f32 rows.  out f32 [max_rows,128]; rows written = min(gallery length, max_rows) (the length is gal_len). */
int dd_tracker_gallery_read(void* state, const dd_tracker_config* host_cfg, int32_t stream_index, int32_t slot,
                            float* out, int32_t max_rows, void* stream);

/* Host edit of one gallery (the FrameRecords hook, deepdish/framerecords.py:157-160, lets a caller run
 * Track.update outside the tracker; the feature then reaches metric.samples at the next partial_fit,
 * tracker.py:84-93): append unit-normalised feat f32 [128] to the slot's gallery -- before its newest row when
 * before_newest != 0 -- with the page allocation, budget trim and half copy an append in the tick performs. */
int dd_tracker_gallery_insert(void* state, const dd_tracker_config* host_cfg, int32_t stream_index, int32_t slot,
                              const float* feat, int32_t before_newest, void* stream);

/* Tracker.predict (tracker.py:51-57 -> track.py:113-125 -> kalman_filter.py:88-123). */
int dd_tracker_predict(void* state, const dd_tracker_config* host_cfg, void* stream);

/* Tracker.update (tracker.py:59-93): gating + cosine cost, matching cascade, IoU stage, Kalman update,
 * mark_missed, _initiate_track, deleted/live split, partial_fit.
 *   det_tlwh  f64 [S,Dmax,4]   Detection.tlwh        (detection.py:30)
 *   det_conf  f32 [S,Dmax]     Detection.confidence
 *   det_label i32 [S,Dmax]     index into the label list
 *   det_feat  f32 [S,Dmax,128] Detection.feature
 *   det_count i32 [S]          detections present this tick (<= Dmax)
 *   out_det_track_id i32 [S,Dmax]  (may be NULL) track id each detection was matched to / created as */
int dd_tracker_update(void* state, const dd_tracker_config* host_cfg,
                      const double* det_tlwh, const float* det_conf, const int32_t* det_label,
                      const float* det_feat, const int32_t* det_count,
                      int32_t* out_det_track_id, void* stream);

/* dd_tracker_update that also records six caller-supplied CUDA events on `stream`: before the
 * detection prep kernel and after each of prep / gate / cosine / match / apply (no synchronisation), so a
 * benchmark can time each kernel inside its own timed region.  host_events6: host array of 6 events
 * made by dd_event_create. */
int dd_tracker_update_profiled(void* state, const dd_tracker_config* host_cfg,
                               const double* det_tlwh, const float* det_conf, const int32_t* det_label,
                               const float* det_feat, const int32_t* det_count,
                               int32_t* out_det_track_id, void* stream, void* const* host_events6);
int dd_event_create(void** host_out);
int dd_event_destroy(void* ev);
int dd_event_elapsed_ms(void* start, void* end, float* host_ms);   /* both events must have completed */
int dd_event_record(void* ev, void* stream);

/* Count-line step (deepdish.py:1035-1114 counting part, :1303-1312; tools/intersection.py:4-30).  Skips a stream
 * that had no frame in the last tick (tick_present; only dd_engine_step_present / _host_present leave one).  With
 * event_cap > 0 it also lists its crossing records (layout `events`), as every tick's count-line step does.
 *   line f64 [S,4] (x1,y1,x2,y2 per stream) or, with line_per_stream = 0, one f64[4] for all streams. */
int dd_tracker_countline(void* state, const dd_tracker_config* host_cfg, const double* line,
                         int line_per_stream, void* stream);

/* Ragged detection batch -> the padded arrays dd_tracker_update consumes.  The reference hands Tracker.update a
 * Python list of Detection objects per stream (deepdish.py:1014); its batched equivalent is one contiguous blob
 * (what a host uploads with a single copy):  i32 offsets[S+1] (stream s owns entries offsets[s]..offsets[s+1]),
 * then at the given byte offsets f64 tlwh[N][4], f32 conf[N], i32 label[N], f32 feat[N][128], N = offsets[S].
 * Writes det_count[s] and the first det_count[s] rows of each padded array (rows beyond are left untouched;
 * a stream with more than max_dets entries gets det_count > max_dets, which the tick reports as
 * DD_FLAG_DET_OVERFLOW).  blob and off_feat must be 16-byte aligned. */
int dd_unpack_detections(const void* blob, int32_t n_streams, int32_t max_dets, int64_t off_tlwh, int64_t off_conf,
                         int64_t off_label, int64_t off_feat, double* det_tlwh, float* det_conf,
                         int32_t* det_label, float* det_feat, int32_t* det_count, void* stream);

/* Sum the per-stream counters into out_counts i64 [C,4] (the tensor handed to the NCCL all-reduce). */
int dd_tracker_count_reduce(void* state, const dd_tracker_config* host_cfg, int64_t* out_counts,
                            void* stream);

/* OR of all per-stream DD_FLAG_* bits -> *host_flags.  Synchronises `stream`.  (The pool counters a caller polls
 * to grow the pool ahead of need are the blob's pool_ctl words.) */
int dd_tracker_status(void* state, const dd_tracker_config* host_cfg, int32_t* host_flags, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Tick engine: the native executor of the batched per-frame loop (the batched form of the reference's driver loop,
 * deepdish.py:1245-1262 -> Pipeline.process_results :1035-1114 around Tracker.predict / update).  One engine drives
 * the n_chunks trackers ("stream chunks": contiguous blocks of streams with their own state blob and CUDA stream) of
 * one GPU: per chunk and tick the detection-prep kernel launched with the tick's inputs by value -- it publishes them into the
 * blob's tick_args words -- followed by ONE captured CUDA graph of the remaining kernels of the tick; chunks overlap freely across tick
 * boundaries; the chunks' partial counters are summed into total_counts on the auxiliary stream.
 * The engine is a HOST object owning only CUDA events / graphs / one capture stream / per-chunk copy streams and 32
 * bytes of pinned memory per chunk; all device buffers stay caller-owned.  Not thread-safe.
 * ---------------------------------------------------------------------------------------------- */
/*   host_states[i], host_cfgs[i]  blob and config of chunk i (configs are copied), host_first_stream[i] its first stream;
 *   host_streams[i]               the chunk's CUDA stream, aux_stream the summation stream (both ignored -- everything runs
 *                                 on the caller's stream -- when n_chunks == 1);
 *   line f64 [4] or [S,4]; partial_counts i64 [2,n_chunks,C,4]; total_counts i64 [C,4]; det_track_id i32 [S,Dmax];
 *   poll_every > 0: every that many ticks the chunk's pool counters are copied to pinned memory behind its tick
 *   (dd_engine_pool_latest reads them without synchronising);
 *   gallery_turns != 0 (n_chunks > 1): the chunks take turns on the HBM-bound gallery stream -- each one waits for the
 *   previously enqueued one --, which keeps the chunks in anti-phase: the latency-bound matching of one chunk always
 *   runs under the gallery stream of another (the tick is then captured as three graphs per chunk). */
int dd_engine_create(int32_t n_chunks, void* const* host_states, const dd_tracker_config* const* host_cfgs,
                     const int32_t* host_first_stream, void* const* host_streams, void* aux_stream, const double* line,
                     int32_t line_per_stream, int64_t* partial_counts, int64_t* total_counts, int32_t* det_track_id,
                     int32_t poll_every, int32_t gallery_turns, void** host_out_engine);
int dd_engine_destroy(void* engine);
/* use_graphs != 0 (the default): the tick's kernels behind the detection-prep kernel are replayed from captured CUDA
 * graphs; 0: the same kernels are launched plainly from the engine's C++ loop.  Same results, same order on the same
 * streams; graphs cost the host less per tick, plain launches leave shorter gaps where a tick is cut into several
 * graphs (gallery_turns).  May be switched between ticks. */
int dd_engine_set_graphs(void* engine, int32_t use_graphs);
/* A chunk's blob was re-laid out or its pool grew (cfg->n_segs / page_cap / segment pointers changed): its captured
 * graphs are dropped and re-captured at the next tick. */
int dd_engine_rebind(void* engine, int32_t chunk, void* state, const dd_tracker_config* host_cfg);
/* Buffers of the end-to-end path of one chunk: n_blobs (2 .. 4) device blobs of blob_capacity bytes (16-byte aligned;
 * host_dev_blobs is a HOST array of their device pointers) the ragged host batches are uploaded into in rotation -- the
 * upload of tick k + n_blobs can start as soon as tick k has consumed its blob, so more buffers decouple the host link
 * from the device tick --, and the small padded arrays (f64 [n,Dmax,4], f32 [n,Dmax], i32 [n,Dmax], i32 [n]) the
 * tick's first kernel expands box / confidence / label / count into. */
int dd_engine_bind_host(void* engine, int32_t chunk, void* const* host_dev_blobs, int32_t n_blobs, uint64_t blob_capacity,
                        double* det_tlwh, float* det_conf, int32_t* det_label, int32_t* det_count);
/* One tick of every chunk from a padded, HBM-resident batch of all S streams (arrays as dd_tracker_update);
 * det_track_id is written; reduce != 0: counters reduced into total_counts (valid after dd_engine_join).  Only
 * enqueues: chunk streams wait for what is already on caller_stream, nothing waits for the chunks. */
int dd_engine_step(void* engine, const double* det_tlwh, const float* det_conf, const int32_t* det_label,
                   const float* det_feat, const int32_t* det_count, int32_t reduce, void* caller_stream);
/* dd_engine_step for a tick in which only some streams have a frame (cameras at different frame rates, dropped
 * frames): present u8 [S] (nonzero = the stream has a frame; NULL = every stream, which is dd_engine_step).  A stream
 * without a frame is left exactly as it is, as the reference leaves the Tracker of a camera that delivers no frame:
 * no Track.predict, no matching or lifecycle change, no gallery append, no count-line step; its rows of the detection
 * arrays and its det_count are ignored (never used) and its det_track_id row is set to -1.  Its counters still take part in the
 * count reduction.  Tracks survive any length of absence and are predicted once at the stream's next frame. */
int dd_engine_step_present(void* engine, const double* det_tlwh, const float* det_conf, const int32_t* det_label,
                           const float* det_feat, const int32_t* det_count, const uint8_t* present, int32_t reduce,
                           void* caller_stream);
/* One end-to-end tick from ragged PINNED host blobs (one per chunk, dd_unpack_detections' format; host_offsets4[4 i ..]
 * = byte offsets of chunk i's tlwh / conf / label / feat sections): upload on the chunk's copy stream (the upload of
 * tick k + 1 runs under the kernels of tick k), the tick reading the blob in place, the count reduction, and -- when
 * host_out_ids (pinned, i32 [S,Dmax]) is given -- the device-to-host copy of the det -> track ids.  The host blobs
 * must stay untouched until their copy has run.  With n_chunks > 1 the chunk streams do NOT wait for caller_stream,
 * so a tick is not held up by whatever the caller queued there: a host that edits a chunk's state or pool on
 * another stream (re-layout, pool segments, gallery insert) makes the chunk's stream wait for that edit itself, as
 * BatchedTracker does. */
int dd_engine_step_host(void* engine, const void* const* host_blobs, const uint64_t* host_blob_bytes,
                        const int64_t* host_offsets4, int32_t* host_out_ids, void* caller_stream);
/* dd_engine_step_host with frame presence (semantics as dd_engine_step_present): host_offsets5[5 i ..] = chunk i's
 * tlwh / conf / label / feat offsets and the byte offset of a u8 present[n] section (n = the chunk's streams) inside
 * its blob, which must lie within host_blob_bytes[i].  An absent stream owns no entries of the blob. */
int dd_engine_step_host_present(void* engine, const void* const* host_blobs, const uint64_t* host_blob_bytes,
                                const int64_t* host_offsets5, int32_t* host_out_ids, void* caller_stream);
/* Crossing records of every chunk's latest tick -> host_out (pinned i32): chunk i's block, the 4 + 4 event_cap words of
 * its `events` section (header, then the records), starts after the blocks of chunks 0 .. i - 1.  Enqueued behind the
 * chunk's latest tick on a read-back stream of its own, like the det -> track ids of dd_engine_step_host (everything on
 * caller_stream when n_chunks == 1); the chunk's next tick waits for the copy before its count-line step rewrites the
 * list, dd_engine_join makes caller_stream wait for it.  Call it right after an engine step (dd_engine_step*): it is
 * ordered behind the engine's ticks only, so after the per-call path (dd_tracker_countline on a stream of the caller's)
 * read the `events` section on that stream instead.  DD_ERR_INVALID for a NULL host_out or when a chunk has
 * event_cap == 0. */
int dd_engine_copy_events(void* engine, int32_t* host_out, void* caller_stream);
/* caller_stream waits for every chunk and for the latest count summation (no host synchronisation). */
int dd_engine_join(void* engine, void* caller_stream);
/* caller_stream waits for the latest count summation only (total_counts of the last reduced tick). */
int dd_engine_wait_counts(void* engine, void* caller_stream);
/* Latest completed poll of chunk's pool counters -> host_out4 (free pages, pages attached, longest gallery, forecast)
 * and the tick it was taken behind (-1: none yet).  If neither of the two most recent polls has completed and the
 * engine is already max_age_ticks ticks past one of them, waits for the more recent such poll: the host never runs
 * further ahead than the forecast covers. */
int dd_engine_pool_latest(void* engine, int32_t chunk, int32_t max_age_ticks, int32_t* host_out4, int64_t* host_out_tick);
/* Ticks stepped, kernels launched (prep kernels + graph nodes + count summations), host milliseconds spent blocked in the run-ahead
 * throttle.  Any output may be NULL. */
int dd_engine_stats(void* engine, int64_t* host_out_ticks, int64_t* host_out_launches, double* host_out_blocked_ms);

/* ------------------------------------------------------------------------------------------------
 * Stand-alone batched operators behind the per-function deep_sort API.
 * ---------------------------------------------------------------------------------------------- */
/* KalmanFilter.initiate (kalman_filter.py:55-86): xyah f64[n,4] -> mean f64[n,8], cov f64[n,64]. */
int dd_kalman_initiate(const double* xyah, double* mean, double* cov, int32_t n, void* stream);
/* KalmanFilter.predict (kalman_filter.py:88-123), in place. */
int dd_kalman_predict(double* mean, double* cov, int32_t n, void* stream);
/* KalmanFilter.project (kalman_filter.py:125-152): -> pmean f64[n,4], pcov f64[n,16]. */
int dd_kalman_project(const double* mean, const double* cov, double* pmean, double* pcov, int32_t n,
                      void* stream);
/* KalmanFilter.update (kalman_filter.py:154-186), in place, one measurement per track. */
int dd_kalman_update(double* mean, double* cov, const double* xyah, int32_t n, void* stream);
/* KalmanFilter.gating_distance (kalman_filter.py:188-229): n tracks x m measurements -> f64[n,m]. */
int dd_kalman_gating_distance(const double* mean, const double* cov, const double* xyah, int32_t n,
                              int32_t m, int32_t only_position, double* out, void* stream);

/* NearestNeighborDistanceMetric.distance (nn_matching.py:156-177), dense.
 *   gallery f32 [G,128] raw sample vectors, gal_offsets i32 [n+1] (target i owns rows off[i]..off[i+1]),
 *   feats f32 [m,128] raw, out f64 [n,m].  metric: 0 = cosine (nn_matching.py:78-96),
 *   1 = euclidean (nn_matching.py:57-75). */
int dd_nn_distance(const float* gallery, const int32_t* gal_offsets, const float* feats, int32_t n,
                   int32_t m, int32_t metric, double* out, void* stream);

/* iou_matching.iou_cost (iou_matching.py:42-81): track_tlwh f64[n,4], tsu i32[n], det_tlwh f64[m,4]
 * -> f64[n,m] (1 - IoU, rows with tsu > 1 = 1e5). */
int dd_iou_cost(const double* track_tlwh, const int32_t* tsu, const double* det_tlwh, int32_t n,
                int32_t m, double* out, void* stream);

/* scipy.optimize.linear_sum_assignment as called at linear_assignment.py:58, INCLUDING scipy's
 * tie-breaking (scipy 1.18.1 rectangular_lsap.cpp).  cost f64 [b,nr,nc]; out_col4row i32 [b,nr]
 * (-1 = row unassigned, only when nr > nc); out_status i32 [b] (0 ok, 1 infeasible). */
int dd_lsap(const double* cost, int32_t b, int32_t nr, int32_t nc, int32_t* out_col4row,
            int32_t* out_status, void* stream);

/* Iteration order of CPython 3.12 `list(set(a) - set(m))` (linear_assignment.py:140) for batches of
 * small non-negative ints: a i32 [b,na_max] with na i32 [b]; m i32 [b,nm_max] with nm i32 [b];
 * out i32 [b,na_max], out_n i32 [b].  Values must be < 1024. */
int dd_set_difference_order(const int32_t* a, const int32_t* na, int32_t na_max, const int32_t* m,
                            const int32_t* nm, int32_t nm_max, int32_t b, int32_t* out,
                            int32_t* out_n, void* stream);

/* tools/intersection.py:4-24 for n segment pairs: seg f64 [n,8] = p,pr,q,qs -> out i32 [n]. */
int dd_intersection(const double* seg, int32_t n, int32_t* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Detector post-processing.
 * ---------------------------------------------------------------------------------------------- */
/* preprocessing.non_max_suppression (deep_sort/preprocessing.py:6-73), one block per frame.
 *   boxes f64 [b,nmax,4] tlwh, scores f32 [b,nmax] (unique per frame), counts i32 [b],
 *   out_keep i32 [b,nmax] original indices in pick order (descending score), out_nkeep i32 [b]. */
int dd_nms(const double* boxes, const float* scores, const int32_t* counts, int32_t b, int32_t nmax,
           double max_overlap, int32_t* out_keep, int32_t* out_nkeep, void* stream);

/* YOLOV5.detect_image post-processing (tools/yolov5.py:115-146) fused with the box filter
 * (deepdish.py:946-955) for b frames:
 *   head: f32 [b,na,5+nc], or u8 with (scale, zero_point) when head_is_u8 != 0 (yolov5.py:115-118);
 *   wanted u8 [nc] (1 = label in wanted_labels); img_w/img_h = PIL image size (yolov5.py:98,131);
 *   frame_w/frame_h = camera viewport of the box filter (deepdish.py:945); frame_w <= 0 skips the box
 *   filter and emits detect_image's own float boxes (adapter mode, tools/yolov5.py:137-146).
 *   Candidates are emitted in ascending anchor order, at most ncap per frame (more -> DD_FLAG_DET_OVERFLOW
 *   in out_flags[b]):  out_tlwh f64 [b,ncap,4] integer-valued boxes after the filter, out_score f32,
 *   out_class i32, out_anchor i32, out_count i32 [b]. */
int dd_yolo_decode(const void* head, int32_t head_is_u8, float scale, int32_t zero_point, int32_t b,
                   int32_t na, int32_t nc, const uint8_t* wanted, float score_thr, int32_t img_w,
                   int32_t img_h, int32_t frame_w, int32_t frame_h, int32_t ncap, double* out_tlwh,
                   float* out_score, int32_t* out_class, int32_t* out_anchor, int32_t* out_count,
                   int32_t* out_flags, void* stream);

/* Keras YOLOv3 adapter post-processing for b frames (tools/yolo.py: decode_netout :48-81, correct_yolo_boxes :83-91,
 * do_nms :122-137, get_boxes :140-153 and the tail of YOLO.detect_image :207-237, including its quirks: transposed
 * boxes x = box[1], y = box[0]; a box with two labels above the threshold is returned twice; reversed order).
 *   map0..2 f32 [b,g,g,3*(5+nc)] raw output maps (g = host_grids3[k]), host_anchors18 = the model's 3 x 6 anchor sizes
 *   (host arrays); wanted u8 [nc].  out_box f64 [b,ncap,4] (x, y, w, h integers), out_score f32, out_label i32 (class
 *   index), out_count i32 [b]; out_flags i32 [b]: DD_FLAG_DET_OVERFLOW (more than ncap results or more than 128 boxes
 *   above the threshold), 64 = two zero-area boxes met in do_nms (the reference raises ZeroDivisionError).
 *   float32 exp is correctly rounded by declaration (see dd_ssd_decode). */
int dd_yolo3_decode(const float* map0, const float* map1, const float* map2, const int32_t* host_grids3,
                    const int32_t* host_anchors18, int32_t b, int32_t nc, const uint8_t* wanted, float score_thr,
                    double nms_thresh, int32_t image_w, int32_t image_h, int32_t net_w, int32_t net_h, int32_t ncap,
                    double* out_box, float* out_score, int32_t* out_label, int32_t* out_count, int32_t* out_flags,
                    void* stream);

/* SSD-MobileNet post-processing for b frames: the TFLite custom op TFLite_Detection_PostProcess
 * (1917-anchor centre-size decode, best non-background class per anchor, greedy IoU NMS at 0.6, <= 10
 * boxes; third-party, restated -- see DESIGN.md "parity unpinned") followed by SSDMobileNet.predict /
 * nms_boxes / SSD_MOBILENET.detect_image (tools/ssd_mobilenet.py:100-150, 59-98, 198-213) and the box
 * filter (deepdish.py:946-955).
 *   raw_boxes f32 [b,na,4] (ty,tx,th,tw), raw_scores f32 [b,na,ncls] (column 0 = background),
 *   anchors f32 [na,4] (ycenter,xcenter,h,w), class_to_label i32 [ncls-1]: output label id of 0-based
 *   class c (the reference's labels[c+1]) or -1 when that label is not wanted.
 *   out_tlwh f64 [b,ncap,4], out_score f32 [b,ncap], out_label i32 [b,ncap], out_count i32 [b]; ncap >= 10;
 *   out_flags i32 [b]: DD_FLAG_DET_OVERFLOW when more than 1024 anchors of a frame reach conf_thr.
 *   raw_scores must be 16-byte aligned (TMA bulk copies).  frame_w <= 0 skips the box filter (adapter mode:
 *   the float boxes SSD_MOBILENET.detect_image returns). */
int dd_ssd_decode(const float* raw_boxes, const float* raw_scores, const float* anchors, int32_t b,
                  int32_t na, int32_t ncls, const int32_t* class_to_label, float conf_thr, double nms_iou,
                  int32_t img_w, int32_t img_h, int32_t frame_w, int32_t frame_h, int32_t ncap,
                  double* out_tlwh, float* out_score, int32_t* out_label, int32_t* out_count,
                  int32_t* out_flags, void* stream);

/* TFLite object-detector adapter for b frames: ObjectDetector._postprocess (tools/tflite_object_detector.py:234-295)
 * followed by TFLITE.detect_image (tools/tflite.py:26-41), on the outputs of the model's own detection post-process op:
 *   op_boxes f32 [b,n,4] (ymin,xmin,ymax,xmax normalised), op_classes f32 [b,n], op_scores f32 [b,n], op_count i32 [b];
 *   list_ok u8 [n_labels]: 1 where the label passes label_deny_list / label_allow_list; wanted u8 [n_labels]: 1 where
 *   the label is in wanted_labels; max_results <= 0 = unlimited.  Output in the reference's order (stable descending
 *   score): out_tlwh f64 [b,ncap,4] = [left, top, right-left, bottom-top] (integers), out_score f32, out_label i32
 *   (class id), out_count i32 [b]; out_flags i32 [b]: DD_FLAG_DET_OVERFLOW when more than ncap detections survive
 *   or a class id is outside the label list (IndexError in the reference). */
int dd_tflite_postprocess(const float* op_boxes, const float* op_classes, const float* op_scores,
                          const int32_t* op_count, int32_t b, int32_t n, int32_t img_w, int32_t img_h,
                          float score_thr, const uint8_t* list_ok, const uint8_t* wanted, int32_t n_labels,
                          int32_t max_results, int32_t ncap, double* out_tlwh, float* out_score, int32_t* out_label,
                          int32_t* out_count, int32_t* out_flags, void* stream);

/* The pre-NMS box filter of Pipeline.detect_objects (deepdish.py:941-960, motion test excluded) on the float boxes a
 * detector adapter returns, for b frames: a NaN anywhere in a frame's boxes drops the whole frame; x, y, w, h are
 * clipped to the camera viewport and truncated toward zero; boxes larger than 0.9 W H are rejected.
 *   boxes f64 [b,nmax,4] tlwh, counts i32 [b] (NULL = nmax); out_tlwh f64 [b,nmax,4] (integers), out_index i32 [b,nmax]
 *   (input index of each survivor, input order kept), out_count i32 [b].  (dd_yolo_decode / dd_ssd_decode fuse the
 *   same filter when given frame_w > 0.) */
int dd_box_filter(const double* boxes, const int32_t* counts, int32_t b, int32_t nmax, int32_t frame_w, int32_t frame_h,
                  double* out_tlwh, int32_t* out_index, int32_t* out_count, void* stream);

/* The step between NMS and the tracker (deepdish.py:996-998,1014): gather the kept candidates, in NMS pick
 * order, into the tracker's padded detection batch for b streams.
 *   cand_* [b,ncap] candidate arrays (dd_yolo_decode / dd_ssd_decode outputs), keep i32 [b,nmax] + nkeep i32 [b]
 *   from dd_nms; label_map i32 [n_map] (may be NULL): detector class / label id -> tracker label id.
 *   Writes det_tlwh f64 [b,dmax,4], det_conf f32 [b,dmax], det_label i32 [b,dmax], det_count i32 [b];
 *   nkeep > dmax sets DD_FLAG_DET_OVERFLOW in out_flags[b] (never silently truncated). */
int dd_gather_detections(const double* cand_tlwh, const float* cand_score, const int32_t* cand_label,
                         const int32_t* label_map, int32_t n_map, int32_t ncap, const int32_t* keep,
                         const int32_t* nkeep, int32_t nmax, int32_t b, int32_t dmax, double* det_tlwh,
                         float* det_conf, int32_t* det_label, int32_t* det_count, int32_t* out_flags,
                         void* stream);

/* ------------------------------------------------------------------------------------------------
 * Re-ID encoder input (the step between NMS and the tracker's feature input).
 * ---------------------------------------------------------------------------------------------- */
/* extract_image_patch (tools/generate_detections.py:40-84) for every detection box of b frames, as the
 * encoder loop calls it (generate_detections.py:198-205): aspect-corrected crop, clip to the frame, 8-bit
 * bilinear cv2.resize to (patch_h, patch_w) -- OpenCV's fixed-point arithmetic, bit-exact.
 *   frames u8 [b,img_h,img_w,3]; boxes f64 [b,dmax,4] tlwh; counts i32 [b] boxes present per frame (NULL = dmax);
 *   boxes_are_int != 0: numpy int64 box semantics (what deepdish.py:993-1008 passes: the aspect correction
 *   truncates toward zero at each item assignment), 0: float box semantics (one truncation at astype(int));
 *   out_patches u8 [b,dmax,patch_h,patch_w,3]; out_valid i32 [b,dmax]: 0 where the reference returns None
 *   (empty or fully outside box; the patch is zero-filled -- the reference substitutes np.random noise) and
 *   for slots >= counts (patch left untouched).  patch_w must be a multiple of 4 and <= 512. */
int dd_extract_patches(const uint8_t* frames, int32_t b, int32_t img_h, int32_t img_w, const double* boxes,
                       const int32_t* counts, int32_t dmax, int32_t boxes_are_int, int32_t patch_h,
                       int32_t patch_w, uint8_t* out_patches, int32_t* out_valid, void* stream);

/* DummyImageEncoder.__call__ (tools/generate_detections.py:86-105), the reference's arithmetic stand-in for the
 * MARS CNN: patches u8 [n,16,8,3] -> out_feat f32 [n,128] (channel mean - 128, L2-normalised; bit-exact). */
int dd_dummy_encode(const uint8_t* patches, int32_t n, float* out_feat, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DEEPDISH_B200_H */
