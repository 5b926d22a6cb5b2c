// dd_view.h -- typed view of the caller-owned tracker state blob + gallery page pool (layout in
// include/deepdish_b200.h).
#pragma once
#include "../../include/deepdish_b200.h"
#include "dd_common.cuh"
#include "dd_lsap.cuh"

// Per-tick inputs of the tick kernels: by value in the kernel parameters or, for a captured tick (dd_engine.cu),
// read from the blob's tick_args words (indirect != 0), so that one CUDA graph serves every tick.
struct DDTickArgs {
    const double* det_tlwh;      // f64 [S,D,4]   (ragged: written by the first kernel, read by the later ones)
    const float* det_conf;       // f32 [S,D]
    const int* det_label;        // i32 [S,D]
    const float* det_feat;       // f32 [S,D,128] (NULL when blob != NULL)
    const int* det_count;        // i32 [S]
    int* out_ids;                // i32 [S,D] or NULL
    long long* out_counts;       // i64 [C,4] or NULL
    const unsigned char* blob;   // ragged batch (dd_unpack_detections' format) or NULL
    const unsigned char* present;// u8 [S]: frame presence of each stream, NULL = every stream present (read by the
                                 // detection-prep kernel only, which records it in the blob's tick_present words)
    long long off_tlwh, off_conf, off_label, off_feat;
    int indirect;
    int tick;                    // engine tick number (timeline slot)
    int publish;                 // detection-prep kernel only: copy these arguments into the blob's tick_args words for
                                 // the captured kernels behind it
};
#define DD_ARG(f) (A.indirect ? V.targs->f : A.f)
// timeline stamps (config.timeline, captured ticks only): kernel k's earliest CTA start / latest CTA end of this tick
#if defined(__CUDACC__)
__device__ __forceinline__ unsigned long long dd_globaltimer() {
    unsigned long long t = 0;
#if defined(__CUDA_ARCH__)
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
#endif
    return t;
}
#define DD_TL_SLOT_AT(tick, k) (V.tl + (size_t)((((tick) & 63) * 8 + (k)) * 2))
#define DD_TL_SLOT(k) DD_TL_SLOT_AT(V.targs->tick, k)
#define DD_TL_BEGIN(k) do { if (V.tl && threadIdx.x == 0) atomicMin(DD_TL_SLOT(k), dd_globaltimer()); } while (0)
#define DD_TL_END(k) do { if (V.tl && threadIdx.x == 0) atomicMax(DD_TL_SLOT(k) + 1, dd_globaltimer()); } while (0)
#endif

struct DDView {
    int S, T, D, B, C, DW;           // streams, slots, det capacity, budget (0 = unbounded), labels, gate words / row
    int PT;                          // page-table entries per slot
    int seg_shift, seg_mask, n_segs; // page id -> (segment, page in segment)
    int tab_cap;                     // slots of each CPython-set emulation table (dd_set_table_slots(T))
    int max_age, n_init;
    double thr_cos, thr_iou;
    int lbl_motorbike, lbl_bicycle;
    int *n_tracks, *next_id, *n_deleted, *err, *order, *deleted;
    long long* counts;
    double *mean, *cov;
    int *track_id, *hits, *age, *tsu, *state, *gal_len, *gal_pos, *gal_np, *ptab, *free_stack, *pool_ctl;
    int* lab_cnt;
    double* lab_sum;
    int* path_n;
    double* path_last;
    int* path_crossed;
    unsigned* gate;
    float* cost;
    double* det_xyah;
    float* det_featn;
    int *det_slot, *det_kind;
    int* cdesc;
    int *work, *work_ctl, *work_rec;
    int* tick_present;               // [S] 1: the stream has a frame this tick (see dd_prep_presence)
    unsigned short* det_feath;
    const DDTickArgs* targs;         // the blob's tick_args words
    unsigned long long* tl;          // timeline words, NULL unless config.timeline
    char* segf[DD_MAX_SEGS];         // f32 pages of each pool segment
    char* segh[DD_MAX_SEGS];         // half pages
    int label_rank[DD_MAX_LABELS];
    int* ev;                         // crossing records: i32 header[4] + [ev_cap][4] (layout `events`), NULL unless
    int ev_cap;                      // config.event_cap > 0
    int n_lines;                     // count lines per stream (counts [S,n_lines,C,4])
};

// ---- gallery pages ----------------------------------------------------------------------------------
DD_HD float4* dd_page_f32(const DDView& V, int pid) {
    return (float4*)(V.segf[pid >> V.seg_shift] + (size_t)(pid & V.seg_mask) * DD_PAGE_F32_BYTES);
}
DD_HD char* dd_page_f16(const DDView& V, int pid) {
    return V.segh[pid >> V.seg_shift] + (size_t)(pid & V.seg_mask) * DD_PAGE_F16_BYTES;
}
// f32 gallery row `row` of the slot whose page table is pt (a row = 32 float4)
DD_HD const float4* dd_gallery_row(const DDView& V, const int* pt, int row) {
    return dd_page_f32(V, pt[row >> 4]) + (size_t)(row & 15) * (DD_FEAT_DIM / 4);
}
// byte offset, inside a half page, of 16-byte chunk c (8 halves) of row r: "fragment order" (deepdish_b200.h)
DD_HD int dd_half_chunk_off(int r, int c) {
    return (((c >> 2) * 2 + (r >> 3)) * 32 + (r & 7) * 4 + (c & 3)) * 16;
}

#if defined(__CUDACC__)
// stamps kernel k's timeline slot at construction and at scope exit (early returns included); thread 0 of each CTA
struct DDTlScope {
    const DDView& V;
    const int k;
    int tick;
    __device__ __forceinline__ DDTlScope(const DDView& v, int k_) : V(v), k(k_), tick(0) {
        if (V.tl && threadIdx.x == 0) { tick = V.targs->tick; atomicMin(DD_TL_SLOT_AT(tick, k), dd_globaltimer()); }
    }
    // the detection-prep kernel publishes the tick's arguments itself: it takes the tick number from its own copy
    __device__ __forceinline__ DDTlScope(const DDView& v, int k_, int tick_) : V(v), k(k_), tick(tick_) {
        if (V.tl && threadIdx.x == 0) atomicMin(DD_TL_SLOT_AT(tick, k), dd_globaltimer());
    }
    __device__ __forceinline__ ~DDTlScope() {
        if (V.tl && threadIdx.x == 0) atomicMax(DD_TL_SLOT_AT(tick, k) + 1, dd_globaltimer());
    }
};
#endif

static inline uint64_t dd_align256(uint64_t x) { return (x + 255u) & ~(uint64_t)255u; }

static inline int dd_page_cap(const dd_tracker_config* c) {
    const int need = c->budget > 0 ? (c->budget + DD_PAGE_ROWS - 1) / DD_PAGE_ROWS : 1;
    return c->page_cap > need ? c->page_cap : need;
}

// config.n_lines, 0 read as 1 (zero-initialised configs)
static inline int dd_n_lines(const dd_tracker_config* c) { return c->n_lines == 0 ? 1 : c->n_lines; }

static inline int dd_layout_compute(const dd_tracker_config* c, dd_tracker_layout* L) {
    if (!c || !L) return DD_ERR_INVALID;
    if (c->n_streams <= 0 || c->max_tracks <= 0 || c->max_dets <= 0 || c->budget < 0) return DD_ERR_INVALID;
    if (c->feat_dim != DD_FEAT_DIM) return DD_ERR_INVALID;
    if (c->n_labels <= 0 || c->n_labels > DD_MAX_LABELS) return DD_ERR_INVALID;
    if (c->max_tracks > 1024 || c->max_dets > 1024) return DD_ERR_INVALID;
    /* the matching kernel keeps time_since_update in 16-bit shared-memory arrays */
    if (c->max_age < 0 || c->max_age > 32766 || c->n_init < 1) return DD_ERR_INVALID;
    if (c->event_cap < 0) return DD_ERR_INVALID;
    if (dd_n_lines(c) < 1 || dd_n_lines(c) > DD_MAX_LINES) return DD_ERR_INVALID;
    if (c->seg_pages <= 0 || (c->seg_pages & (c->seg_pages - 1)) != 0) return DD_ERR_INVALID;
    if (c->n_segs < 1 || c->n_segs > DD_MAX_SEGS || c->page_cap < 0) return DD_ERR_INVALID;
    const uint64_t S = c->n_streams, T = c->max_tracks, D = c->max_dets, PT = dd_page_cap(c),
                   C = c->n_labels, F = DD_FEAT_DIM, DW = (D + 31) / 32, NLN = dd_n_lines(c);
    uint64_t off = 0;
#define DD_PUT(name, bytes) do { L->name = off; off = dd_align256(off + (uint64_t)(bytes)); } while (0)
    DD_PUT(n_tracks, 4 * S);
    DD_PUT(next_id, 4 * S);
    DD_PUT(n_deleted, 4 * S);
    DD_PUT(err, 4 * S);
    DD_PUT(order, 4 * S * T);
    DD_PUT(deleted, 4 * S * T);
    DD_PUT(counts, 8 * S * NLN * C * 4);
    DD_PUT(mean, 8 * S * T * 8);
    DD_PUT(cov, 8 * S * T * 64);
    DD_PUT(track_id, 4 * S * T);
    DD_PUT(hits, 4 * S * T);
    DD_PUT(age, 4 * S * T);
    DD_PUT(tsu, 4 * S * T);
    DD_PUT(state, 4 * S * T);
    DD_PUT(gal_len, 4 * S * T);
    DD_PUT(gal_pos, 4 * S * T);
    DD_PUT(gal_np, 4 * S * T);
    DD_PUT(ptab, 4 * S * T * PT);
    DD_PUT(free_stack, 4 * (uint64_t)DD_MAX_SEGS * c->seg_pages);
    DD_PUT(pool_ctl, 4 * 64);
    DD_PUT(lab_cnt, 4 * S * T * C);
    DD_PUT(lab_sum, 8 * S * T * C);
    DD_PUT(path_n, 4 * S * T);
    DD_PUT(path_last, 8 * S * T * 2);
    DD_PUT(path_crossed, 4 * S * T);
    DD_PUT(gate, 4 * S * T * DW);
    DD_PUT(cost, 4 * S * T * D);
    DD_PUT(det_xyah, 8 * S * D * 4);
    DD_PUT(det_featn, 4 * S * D * F);
    DD_PUT(det_slot, 4 * S * D);
    DD_PUT(det_kind, 4 * S * D);
    DD_PUT(cdesc, 4 * S * T * 4);
    DD_PUT(work, 4 * S * T);
    DD_PUT(work_ctl, 4 * 64);
    DD_PUT(work_rec, 4 * S * T * 16);
    DD_PUT(det_feath, 2 * S * D * F);
    DD_PUT(tick_args, 256);
    DD_PUT(timeline, 8 * 64 * 8 * 2);
    DD_PUT(tick_present, 4 * S);
    DD_PUT(events, c->event_cap > 0 ? 16 * (1 + (uint64_t)c->event_cap) : 0);     // 0 bytes when off: total_bytes unchanged
#undef DD_PUT
    L->total_bytes = off;
    return DD_OK;
}

static inline int dd_make_view(void* blob, const dd_tracker_config* c, DDView* v) {
    dd_tracker_layout L;
    int rc = dd_layout_compute(c, &L);
    if (rc != DD_OK) return rc;
    if (!blob) return DD_ERR_INVALID;
    char* b = (char*)blob;
    v->S = c->n_streams; v->T = c->max_tracks; v->D = c->max_dets; v->B = c->budget;
    v->C = c->n_labels; v->DW = (c->max_dets + 31) / 32;
    v->PT = dd_page_cap(c);
    v->seg_mask = c->seg_pages - 1;
    v->seg_shift = 0;
    while ((1 << v->seg_shift) < c->seg_pages) ++v->seg_shift;
    v->n_segs = c->n_segs;
    v->tab_cap = dd_set_table_slots(c->max_tracks);
    v->max_age = c->max_age; v->n_init = c->n_init;
    v->thr_cos = c->max_cosine_distance; v->thr_iou = c->max_iou_distance;
    v->lbl_motorbike = c->label_motorbike; v->lbl_bicycle = c->label_bicycle;
    v->n_tracks = (int*)(b + L.n_tracks); v->next_id = (int*)(b + L.next_id);
    v->n_deleted = (int*)(b + L.n_deleted); v->err = (int*)(b + L.err);
    v->order = (int*)(b + L.order); v->deleted = (int*)(b + L.deleted);
    v->counts = (long long*)(b + L.counts);
    v->mean = (double*)(b + L.mean); v->cov = (double*)(b + L.cov);
    v->track_id = (int*)(b + L.track_id); v->hits = (int*)(b + L.hits); v->age = (int*)(b + L.age);
    v->tsu = (int*)(b + L.tsu); v->state = (int*)(b + L.state);
    v->gal_len = (int*)(b + L.gal_len); v->gal_pos = (int*)(b + L.gal_pos);
    v->gal_np = (int*)(b + L.gal_np); v->ptab = (int*)(b + L.ptab);
    v->free_stack = (int*)(b + L.free_stack); v->pool_ctl = (int*)(b + L.pool_ctl);
    v->lab_cnt = (int*)(b + L.lab_cnt); v->lab_sum = (double*)(b + L.lab_sum);
    v->path_n = (int*)(b + L.path_n); v->path_last = (double*)(b + L.path_last);
    v->path_crossed = (int*)(b + L.path_crossed);
    v->gate = (unsigned*)(b + L.gate); v->cost = (float*)(b + L.cost);
    v->det_xyah = (double*)(b + L.det_xyah); v->det_featn = (float*)(b + L.det_featn);
    v->det_slot = (int*)(b + L.det_slot); v->det_kind = (int*)(b + L.det_kind);
    v->cdesc = (int*)(b + L.cdesc);
    v->tick_present = (int*)(b + L.tick_present);
    v->det_feath = (unsigned short*)(b + L.det_feath);
    v->targs = (const DDTickArgs*)(b + L.tick_args);
    v->tl = c->timeline ? (unsigned long long*)(b + L.timeline) : nullptr;
    v->ev = c->event_cap > 0 ? (int*)(b + L.events) : nullptr;
    v->ev_cap = c->event_cap;
    v->n_lines = dd_n_lines(c);
    v->work = (int*)(b + L.work); v->work_ctl = (int*)(b + L.work_ctl); v->work_rec = (int*)(b + L.work_rec);
    for (int i = 0; i < DD_MAX_SEGS; ++i) {
        const bool on = i < c->n_segs;
        v->segf[i] = on ? (char*)(uintptr_t)c->pool_f32[i] : nullptr;
        v->segh[i] = on ? (char*)(uintptr_t)c->pool_f16[i] : nullptr;
        if (on && (!v->segf[i] || !v->segh[i] || (c->pool_f32[i] & 15) || (c->pool_f16[i] & 15))) return DD_ERR_INVALID;
    }
    for (int i = 0; i < DD_MAX_LABELS; ++i) v->label_rank[i] = i < c->n_labels ? c->label_rank[i] : 0;
    return DD_OK;
}
