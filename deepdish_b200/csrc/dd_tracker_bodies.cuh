// dd_tracker_bodies.cuh -- per-unit bodies of the batched DeepSORT tick (group-generic, see dd_common.cuh).
//
//   dd_prep_det        (stream, det)    frame presence + Detection.to_xyah + feature normalisation
//   dd_predict_track   (stream, track)  Track.predict
//   dd_gate_track      (stream, track)  gating_distance -> gate bitmask + stream descriptor
//   dd_cosine_track    (stream, track)  gallery min cosine distance for the gate-passing pairs
//   dd_match_stream    (stream)         matching cascade + IoU stage + track lifecycle
//   dd_apply_det       (stream, det)    Kalman update / initiate + gallery append + label vote
//   dd_countline       (stream)         count-line crossing + per-label counters
//   dd_countline_lines (stream)         the same for several count lines per stream (config.n_lines > 1)
#pragma once
#include "dd_view.h"
#include "dd_kalman.cuh"
#include "dd_lsap.cuh"
#if defined(__CUDACC__)
#include <cuda_fp16.h>
#endif

#define DD_INFTY_COST 1e5          // deep_sort/linear_assignment.py:8
#define DD_POOL_LOOKAHEAD 8        // appends ahead that the page-demand forecast (pool_ctl[3]) covers

#if defined(__CUDA_ARCH__)
// half copies of unit vectors for the gallery kernel's pre-pass (device only; the host emulation runs the
// exact pass and never reads them)
DD_D void dd_store_half4(unsigned short* dst, const float4& x) {
    const __half2 lo = __floats2half2_rn(x.x, x.y), hi = __floats2half2_rn(x.z, x.w);
    uint2 u;
    u.x = *reinterpret_cast<const unsigned*>(&lo);
    u.y = *reinterpret_cast<const unsigned*>(&hi);
    *reinterpret_cast<uint2*>(dst) = u;
}
DD_D void dd_atomic_add_ll(long long* p, long long v) { atomicAdd((unsigned long long*)p, (unsigned long long)v); }
DD_D void dd_atomic_or(int* p, int v) { atomicOr(p, v); }
DD_D int dd_atomic_add_i(int* p, int v) { return atomicAdd(p, v); }
DD_D void dd_atomic_max_i(int* p, int v) { atomicMax(p, v); }
#else
inline void dd_store_half4(unsigned short*, const float4&) {}
inline void dd_atomic_add_ll(long long* p, long long v) { *p += v; }
inline void dd_atomic_or(int* p, int v) { *p |= v; }
inline int dd_atomic_add_i(int* p, int v) { const int o = *p; *p = o + v; return o; }
inline void dd_atomic_max_i(int* p, int v) { if (v > *p) *p = v; }
#endif

// ------------------------------------------------------------------------------------------------
// Gallery page pool: a stack of free page ids.  Pages are popped only while features are appended (k_apply, the
// host-edit insert) and pushed only while slots are recycled (k_match, pool attach): never both in one kernel, so
// a counter and plain stores suffice.
// ------------------------------------------------------------------------------------------------
DD_HD int dd_page_alloc(const DDView& V) {
    const int i = dd_atomic_add_i(V.pool_ctl, -1) - 1;
    if (i < 0) {
        dd_atomic_add_i(V.pool_ctl, 1);
        return -1;
    }
    return V.free_stack[i];
}
DD_HD void dd_page_free(const DDView& V, int pid) { V.free_stack[dd_atomic_add_i(V.pool_ctl, 1)] = pid; }

// one gallery row -> f32 page + half page (chunks x[kk] = float4 number lane + kk * NL of the row)
template <class G, int KP>
DD_HD void dd_gallery_store_row(const G& g, const DDView& V, int pid, int r, const float4 (&x)[KP]) {
    float4* dst = dd_page_f32(V, pid) + (size_t)r * (DD_FEAT_DIM / 4);
    char* dsth = dd_page_f16(V, pid);
    int kk = 0;
    for (int k = g.lane; k < DD_FEAT_DIM / 4; k += G::NL, ++kk) {
        dst[k] = x[kk];
        dd_store_half4((unsigned short*)(dsth + dd_half_chunk_off(r, k >> 1) + (k & 1) * 8), x[kk]);
    }
}

// Append one unit-normalised feature (chunks x[kk] = float4 number lane + kk * NL) to the gallery of `slot`:
// what metric.partial_fit does for one (feature, target) pair (nn_matching.py:148-151).  pos / len / np are the
// slot's gal_pos / gal_len / gal_np as read by the caller (all lanes hold the same values).
// pid_hint: the id of page pos / 16 when the caller has already read it (>= 0), else -1.
template <class G, int KP>
DD_HD void dd_gallery_append(const G& g, const DDView& V, int s, size_t slot, int pos, int len, int np,
                             const float4 (&x)[KP], int pid_hint = -1) {
    const int pg = pos >> 4;
    int pid = -1;
    bool ok = true;
    if (pg < np) {
        pid = pid_hint >= 0 ? pid_hint : V.ptab[slot * V.PT + pg];
    } else if (pg >= V.PT) {
        ok = false;
        if (g.lane == 0) dd_atomic_or(V.err + s, DD_FLAG_GALLERY_OVERFLOW);
    } else {
        if (g.lane == 0) pid = dd_page_alloc(V);
        pid = g.imax(g.lane == 0 ? pid : (int)0x80000000);
        if (pid < 0) {
            ok = false;
            if (g.lane == 0) dd_atomic_or(V.err + s, DD_FLAG_POOL_EXHAUSTED);
        } else if (g.lane == 0) {
            V.ptab[slot * V.PT + pg] = pid;
            V.gal_np[slot] = np + 1;
        }
    }
    if (!ok) return;
    dd_gallery_store_row<G, KP>(g, V, pid, pos & 15, x);
    if (g.lane == 0) {
        const int nlen = V.B > 0 ? (len < V.B ? len + 1 : V.B) : len + 1;
        const int npos = V.B > 0 ? ((pos + 1 == V.B) ? 0 : pos + 1) : pos + 1;
        V.gal_pos[slot] = npos;
        V.gal_len[slot] = nlen;
        if (V.B == 0 && nlen > V.pool_ctl[2]) dd_atomic_max_i(V.pool_ctl + 2, nlen);     // longest gallery so far
        // page-demand forecast (pool_ctl[3]): does this gallery need another page within its next few appends?
        const int ring_pages = V.B > 0 ? (V.B + DD_PAGE_ROWS - 1) / DD_PAGE_ROWS : 0x7fffffff;
        const int have = pg < np ? np : np + 1;
        if (dd_imin((npos + DD_POOL_LOOKAHEAD - 1) >> 4, ring_pages - 1) >= have) dd_atomic_add_i(V.pool_ctl + 3, 1);
    }
}

// ------------------------------------------------------------------------------------------------
// Detection.to_xyah (deep_sort/detection.py:43-50) and b / |b| (deep_sort/nn_matching.py:53).
// ------------------------------------------------------------------------------------------------
// box = the detection's tlwh (4 doubles), feat = its raw 128-d feature row; results go to slot (s, d) of the scratch
template <class G>
DD_HD void dd_prep_det_at(const G& g, const DDView& V, int s, int d, const double* box, const float* feat) {
    const size_t sd = (size_t)s * V.D + d;
    if (g.lane == 0) {
        const double* b = box;
        double* o = V.det_xyah + sd * 4;
        o[0] = dd_add(b[0], dd_div(b[2], 2.0));
        o[1] = dd_add(b[1], dd_div(b[3], 2.0));
        o[2] = dd_div(b[2], b[3]);
        o[3] = b[3];
    }
    const float4* f4 = (const float4*)feat;
    float4* o4 = (float4*)(V.det_featn + sd * DD_FEAT_DIM);
    float ss = 0.f;
    for (int k = g.lane; k < DD_FEAT_DIM / 4; k += G::NL) {
        const float4 x = f4[k];
        ss = dd_fmaf(x.x, x.x, ss); ss = dd_fmaf(x.y, x.y, ss);
        ss = dd_fmaf(x.z, x.z, ss); ss = dd_fmaf(x.w, x.w, ss);
    }
    const float nrm = dd_sqrtf(g.sum(ss));
    for (int k = g.lane; k < DD_FEAT_DIM / 4; k += G::NL) {
        float4 x = f4[k];
        x.x = dd_divf(x.x, nrm); x.y = dd_divf(x.y, nrm);
        x.z = dd_divf(x.z, nrm); x.w = dd_divf(x.w, nrm);
        o4[k] = x;
        dd_store_half4(V.det_feath + sd * DD_FEAT_DIM + 4 * k, x);
    }
}

// Frame presence (present u8 [S], NULL = every stream): the detection prep of every tick records it in tick_present,
// which every later step of the tick reads.  A stream without a frame is left exactly as it is -- what the reference
// does to the tracker of a camera that delivers no frame: no predict, no update, no count-line step -- and its
// detection inputs are never used.  Returns whether stream s is present.
template <class G>
DD_HD bool dd_prep_presence(const G& g, const DDView& V, int s, int d, const unsigned char* present) {
    const bool p = present == nullptr || present[s] != 0;
    if (d == 0 && g.lane == 0) V.tick_present[s] = p ? 1 : 0;
    return p;
}

template <class G>
DD_HD void dd_prep_det(const G& g, const DDView& V, int s, int d, const double* det_tlwh,
                       const float* det_feat, const int* det_count, const unsigned char* present = nullptr) {
    if (!dd_prep_presence(g, V, s, d, present)) return;
    int nd = det_count[s];
    if (nd > V.D) nd = V.D;
    if (d >= nd) return;
    const size_t sd = (size_t)s * V.D + d;
    dd_prep_det_at(g, V, s, d, det_tlwh + sd * 4, det_feat + sd * DD_FEAT_DIM);
}

// ------------------------------------------------------------------------------------------------
// Track.predict (deep_sort/track.py:113-125).
// ------------------------------------------------------------------------------------------------
template <class G>
DD_HD void dd_predict_live_track(const G& g, const DDView& V, int s, int t) {
    const size_t slot = (size_t)s * V.T + V.order[(size_t)s * V.T + t];
    dd_kf_predict(g, V.mean + slot * 8, V.cov + slot * 64);
    if (g.lane == 0) {
        V.age[slot] += 1;
        V.tsu[slot] += 1;
    }
}
template <class G>
DD_HD void dd_predict_track(const G& g, const DDView& V, int s, int t) {
    if (t < V.n_tracks[s]) dd_predict_live_track(g, V, s, t);
}

// Track.predict inside a tick: only the tracks of a stream that has a frame (the per-call predict steps every stream).
// The presence word is loaded beside the track count, not in front of it: no extra memory round trip on the chain.
template <class G>
DD_HD void dd_tick_predict_track(const G& g, const DDView& V, int s, int t) {
    const int nt = V.n_tracks[s], present = V.tick_present[s];
    if (present && t < nt) dd_predict_live_track(g, V, s, t);
}

// ------------------------------------------------------------------------------------------------
// Gate-first appearance cost for one confirmed track:
//   gate bit d  = not (gating_distance > chi2inv95[4])     (linear_assignment.py:182-189)
//   cost[d]     = min over the track's gallery of 1 - a.b   (nn_matching.py:78-96), only where the
//                 gate bit is set -- every other entry of the reference cost matrix is overwritten
//                 with INFTY_COST before it is read, so it is never computed here.
// Gallery rows are unit vectors (normalised when appended); each lane owns one float4 of the 128-d
// row, up to DD_CH candidates share one pass over the gallery.
// ------------------------------------------------------------------------------------------------
#define DD_CH 4          // candidates sharing one pass over the gallery
#define DD_ROWS 8        // gallery rows per step (8 x 512 B = 4 KB); fold size = DD_ROWS x NC

// Cross-lane sum of N = ROWS * NC per-lane partials v[r * NC + c] by a transposing butterfly
// (N - 1 + log2(32 / N) shuffles instead of 5 N), folded into a running maximum over rows per candidate.
// WarpG: after the butterfly lane L owns the total of value index idx(L) = L >> log2(32 / N), so its
// candidate is idx(L) % NC; the running maximum lives in acc[0] and dd_fold_finish combines lanes.
// HostG: one lane owns everything, acc[c] is the maximum for candidate c.
#if defined(__CUDACC__)
template <int NC, int N>
__device__ __forceinline__ void dd_fold_max(const WarpG& g, float (&v)[N], float (&acc)[NC]) {
    int n = N, o = 16;
#pragma unroll
    for (; n > 1; n >>= 1, o >>= 1) {
        const bool up = (g.lane & o) != 0;
        const int half = n >> 1;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float send = up ? v[i] : v[i + half];
            const float keep = up ? v[i + half] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
#pragma unroll
    for (; o > 0; o >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
    acc[0] = v[0] > acc[0] ? v[0] : acc[0];
}
template <int NC, int N>
__device__ __forceinline__ void dd_fold_finish(const WarpG& g, float (&acc)[NC], float (&best)[NC]) {
    constexpr int SH = N >= 32 ? 0 : (N == 16 ? 1 : (N == 8 ? 2 : (N == 4 ? 3 : 4)));   // idx(L) = L >> SH
    const int mine = (g.lane >> SH) % NC;
#pragma unroll
    for (int c = 0; c < NC; ++c) best[c] = g.fmax(mine == c ? acc[0] : -3.0e38f);
}
#endif
template <int NC, int N>
inline void dd_fold_max(const HostG&, float (&v)[N], float (&acc)[NC]) {
    for (int r = 0; r < N / NC; ++r)
        for (int c = 0; c < NC; ++c) acc[c] = v[r * NC + c] > acc[c] ? v[r * NC + c] : acc[c];
}
template <int NC, int N>
inline void dd_fold_finish(const HostG&, float (&acc)[NC], float (&best)[NC]) {
    for (int c = 0; c < NC; ++c) best[c] = acc[c];
}

// max over the gallery rows of row . q[c] for NC query vectors; rows are unit vectors, each lane owns
// float4 chunk(s) of the 128-d row; DD_ROWS rows (4 KB) are loaded back to back before any arithmetic.
// Rows past glen re-read the last row (duplicates do not change a max).  This is the exact f32 pass: the
// arithmetic that DEFINES the cost entries (the half-precision gallery kernel re-evaluates its candidates with
// exactly these operations), the host emulation's path and gallery_impl = 1.  pt = the slot's page table.
template <class G, int NC>
DD_HD void dd_cosine_pass(const G& g, const DDView& V, const int* __restrict__ pt, int glen,
                          const float4* const (&qp)[DD_CH], float (&best)[DD_CH]) {
    constexpr int ROWS = DD_ROWS;
    constexpr int DD_FOLD = DD_ROWS * NC;
    constexpr int KP = (DD_FEAT_DIM / 4) / G::NL;          // float4 chunks per lane (1 on a warp)
    float4 q[NC][KP];
    for (int c = 0; c < NC; ++c) {
        int kk = 0;
        for (int k = g.lane; k < DD_FEAT_DIM / 4; k += G::NL, ++kk) q[c][kk] = qp[c][k];
    }
    float acc[NC];
    for (int c = 0; c < NC; ++c) acc[c] = -3.0e38f;
    for (int g0 = 0; g0 < glen; g0 += ROWS) {
        float v[DD_FOLD];
#pragma unroll
        for (int i = 0; i < DD_FOLD; ++i) v[i] = 0.f;
        int kk = 0;
        for (int k = g.lane; k < DD_FEAT_DIM / 4; k += G::NL, ++kk) {
            float4 a[ROWS];
#pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                const int row = dd_imin(g0 + r, glen - 1);
                a[r] = dd_gallery_row(V, pt, row)[k];
            }
#pragma unroll
            for (int r = 0; r < ROWS; ++r)
#pragma unroll
                for (int c = 0; c < NC; ++c) {
                    float p = v[r * NC + c];
                    p = dd_fmaf(a[r].x, q[c][kk].x, p);
                    p = dd_fmaf(a[r].y, q[c][kk].y, p);
                    p = dd_fmaf(a[r].z, q[c][kk].z, p);
                    p = dd_fmaf(a[r].w, q[c][kk].w, p);
                    v[r * NC + c] = p;
                }
        }
        dd_fold_max<NC, DD_FOLD>(g, v, acc);
    }
    float b[NC];
    dd_fold_finish<NC, DD_FOLD>(g, acc, b);
    for (int c = 0; c < NC; ++c) best[c] = b[c];
}

template <class G>
struct DDDirectPass {
    template <int NC>
    DD_HD void run(const G& g, const DDView& V, const int* pt, int glen, const float4* const (&qp)[DD_CH],
                   float (&best)[DD_CH]) {
        dd_cosine_pass<G, NC>(g, V, pt, glen, qp, best);
    }
};

// Gate of one track index (every t < Tmax is visited so that inactive entries get an empty descriptor):
// f64 projection + 4x4 Cholesky per lane (redundant), lanes sweep the detections, ballot -> gate words.
// A stream without a frame this tick gets empty descriptors only: nothing of it reaches the gallery kernel.
template <class G>
DD_HD int dd_gate_track(const G& g, const DDView& V, int s, int t, const int* det_count) {
    int* desc = V.cdesc + ((size_t)s * V.T + t) * 4;
    const int nt = V.n_tracks[s], present = V.tick_present[s];
    bool active = present != 0 && t < nt;
    size_t slot = 0;
    if (active) {
        slot = (size_t)s * V.T + V.order[(size_t)s * V.T + t];
        active = V.state[slot] == DD_STATE_CONFIRMED;
    }
    if (!active) {
        if (g.lane == 0) { desc[0] = 0; desc[1] = 0; desc[2] = 0; desc[3] = 0; }
        return 0;
    }
    int nd = det_count[s];
    if (nd > V.D) nd = V.D;
    const double* mean = V.mean + slot * 8;
    double S[16], L[16], rinv[4];
    dd_kf_project_cov(mean, V.cov + slot * 64, S);
    dd_chol<4>(S, L, rinv);
    const double pm[4] = {mean[0], mean[1], mean[2], mean[3]};
    int ncand = 0;
    for (int base = 0; base < nd; base += 32) {
        unsigned word = 0;
        const int lim = dd_imin(base + 32, nd);
        for (int j = base + g.lane; j < lim; j += G::NL) {
            const double d2 = dd_maha_sq<4>(L, rinv, pm, V.det_xyah + ((size_t)s * V.D + j) * 4);
            if (!(d2 > DD_CHI2INV95_4)) word |= 1u << (j - base);
        }
        word = g.bor(word);
        if (g.lane == 0) V.gate[slot * V.DW + (base >> 5)] = word;
#if defined(__CUDA_ARCH__)
        ncand += __popc(word);
#else
        ncand += __builtin_popcount(word);
#endif
    }
    if (g.lane == 0) {
        desc[0] = (int)(slot - (size_t)s * V.T);
        desc[1] = V.gal_len[slot];
        desc[2] = ncand;
        desc[3] = V.gal_np[slot];
    }
    return ncand;       // > 0: the track index goes on the gallery kernel's work list
}

// Appearance cost of one track index for its gate-passing detections: one descriptor load decides
// whether anything is streamed; the gallery is then read once per group of <= DD_CH candidates.
template <class G, class Pass>
DD_HD void dd_cosine_track(const G& g, const DDView& V, int s, int t, const int* det_count, Pass& pass) {
    const int* desc = V.cdesc + ((size_t)s * V.T + t) * 4;
    if (desc[2] <= 0) return;
    const size_t slot = (size_t)s * V.T + desc[0];
    const int glen = desc[1];
    int nd = det_count[s];
    if (nd > V.D) nd = V.D;
    const int* pt = V.ptab + slot * V.PT;
    for (int base = 0; base < nd; base += 32) {
        unsigned word = V.gate[slot * V.DW + (base >> 5)];
        while (word) {
            int cj[DD_CH];
            int nc = 0;
            while (word && nc < DD_CH) {
                const int b = dd_ctz(word);
                word &= word - 1;
                cj[nc++] = base + b;
            }
            const float4* qp[DD_CH];
            for (int c = 0; c < DD_CH; ++c)
                qp[c] = (const float4*)(V.det_featn + ((size_t)s * V.D + cj[c < nc ? c : 0]) * DD_FEAT_DIM);
            float best[DD_CH];
            if (glen <= 0) {
                for (int c = 0; c < DD_CH; ++c) best[c] = -3.0e38f;
            } else if (nc == 1) {
                pass.template run<1>(g, V, pt, glen, qp, best);
            } else if (nc == 2) {
                pass.template run<2>(g, V, pt, glen, qp, best);
            } else {
                pass.template run<4>(g, V, pt, glen, qp, best);
            }
            if (g.lane == 0)
                for (int c = 0; c < nc; ++c) V.cost[slot * V.D + cj[c]] = dd_subf(1.0f, best[c]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Per-stream matching + lifecycle.  Shared-memory plan (bytes, n = max(T, D)):
//   LSAP scratch | trk_slot[T] trk_tsu[T] trk_det[T] rows[T] lista[T] listb[T] | cols/undA[D] undB[D]
//   | trk_state[T] flag[T] (bytes) | three set tables of dd_set_table_slots(T) shorts
// ------------------------------------------------------------------------------------------------
struct DDMatchSmem {
    DDLsapScratch ls;
    short *trk_slot, *trk_tsu, *trk_det, *rows, *lista, *listb, *undA, *undB, *r2c, *c2r;
    unsigned char *trk_state, *flag;
    short *tabA, *tabB, *tabC;
    int tab_cap;
    double* tbox;      // [T][5]  x, y, x2, y2, area of the IoU-stage rows (Track.to_tlwh, track.py:84-97)
    unsigned* gate_sm; // [T][DW] gate words of the live tracks, by track index
    float* cval;       // [T][DD_CVAL] cost of the first DD_CVAL gate-passing detections of each track
    double* dbox;      // [D][4]  this stream's detection boxes (the IoU-stage scan reads them per column)
};

// Three regions are never live at the same time and share one union: the gate words + staged costs (matching cascade
// only), the three CPython-set tables (set-order step between the cascade and the IoU stage) and tbox (IoU stage
// only).  The matching warp's shared memory decides how many streams fit on an SM beside another chunk's gallery
// stream, so every kilobyte here is occupancy.
#ifndef DD_CVAL
#define DD_CVAL 4       // gate-passing costs per track kept in shared memory (the rest is read from global)
#endif
#ifndef DD_MB
#define DD_MB 4         // iterations per batch of the matching warp's staging loops (loads first, then stores)
#endif
DD_HD size_t dd_match_union_bytes(int T, int D, int tab_cap) {
    const size_t a = (size_t)T * ((D + 31) / 32) * 4 + (size_t)T * DD_CVAL * 4;
    const size_t b = (size_t)tab_cap * 2 * 3;
    const size_t c = (size_t)T * 5 * 8;
    size_t m = a > b ? a : b;
    m = m > c ? m : c;
    return (m + 15) & ~(size_t)15;
}
DD_HD size_t dd_match_smem_base_bytes(int T, int D, int tab_cap) {
    const int n = T > D ? T : D;
    size_t b = dd_lsap_scratch_bytes(n);
    b += (size_t)T * 2 * 6 + (size_t)D * 2 * 2 + (size_t)n * 2 * 2;
    b += (size_t)T * 2;
    return (b + 15) & ~(size_t)15;
}
DD_HD size_t dd_match_smem_bytes(int T, int D, int tab_cap) {
    return dd_match_smem_base_bytes(T, D, tab_cap) + (size_t)D * 32 + dd_match_union_bytes(T, D, tab_cap) + 16;
}

DD_HD void dd_match_carve(char* mem, int T, int D, int tab_cap, DDMatchSmem& m) {
    const int n = T > D ? T : D;
    dd_lsap_carve(mem, n, m.ls);
    char* p = mem + dd_lsap_scratch_bytes(n);
    m.trk_slot = (short*)p; p += T * 2;
    m.trk_tsu = (short*)p; p += T * 2;
    m.trk_det = (short*)p; p += T * 2;
    m.rows = (short*)p; p += T * 2;
    m.lista = (short*)p; p += T * 2;
    m.listb = (short*)p; p += T * 2;
    m.undA = (short*)p; p += D * 2;
    m.undB = (short*)p; p += D * 2;
    m.r2c = (short*)p; p += n * 2;
    m.c2r = (short*)p; p += n * 2;
    m.trk_state = (unsigned char*)p; p += T;
    m.flag = (unsigned char*)p; p += T;
    p = mem + dd_match_smem_base_bytes(T, D, tab_cap);
    m.dbox = (double*)p; p += (size_t)D * 32;
    // the union
    m.tab_cap = tab_cap;
    m.gate_sm = (unsigned*)p;
    m.cval = (float*)(m.gate_sm + (size_t)T * ((D + 31) / 32));
    m.tabA = (short*)p;
    m.tabB = m.tabA + tab_cap;
    m.tabC = m.tabB + tab_cap;
    m.tbox = (double*)p;
}

// cost functors: (r, c) are positions in the rows[] / cols[] lists of the current sub-problem.
struct DDCosineCost {      // tracker.py:97-105 + linear_assignment.py:57
    const unsigned* gate;  // shared memory [T, DW], indexed by TRACK INDEX
    const float* cval;     // shared memory [T, DD_CVAL]: costs of the first gate-passing detections
    const float* cost;     // stream base [T, D] in global memory, indexed by slot (overflow of cval only)
    const short *trk_slot, *rows, *cols;
    int D, DW;
    double thr, clip;
    DD_HD double raw(int r, int c) const {
        const int t = rows[r];
        const int d = cols[c];
        const unsigned* gw = gate + t * DW;
        const unsigned word = gw[d >> 5];
        if (!((word >> (d & 31)) & 1u)) return DD_INFTY_COST;
        int k = dd_popc(word & ((1u << (d & 31)) - 1u));          // rank of d among the track's set bits
        for (int w = 0; w < (d >> 5); ++w) k += dd_popc(gw[w]);
        return (double)(k < DD_CVAL ? cval[t * DD_CVAL + k] : cost[trk_slot[t] * D + d]);
    }
    DD_HD double operator()(int r, int c) const {
        const double v = raw(r, c);
        return v > thr ? clip : v;
    }
};

struct DDIouCost {         // iou_matching.py:7-81 + linear_assignment.py:57
    const double* tbox;    // [nr][5] per row: x, y, x2, y2, area (INFTY rows: area < 0)
    const double* det_tlwh;// stream's boxes [D, 4] (shared-memory copy)
    const short* cols;
    double thr, clip;
    DD_HD double raw(int r, int c) const {
        const double* t = tbox + r * 5;
        if (t[4] < 0.0) return DD_INFTY_COST;          // time_since_update > 1 (iou_matching.py:74-76)
        const double* b = det_tlwh + (size_t)cols[c] * 4;
        const double tlx = dd_max(t[0], b[0]), tly = dd_max(t[1], b[1]);
        const double brx = dd_min(t[2], dd_add(b[0], b[2]));
        const double bry = dd_min(t[3], dd_add(b[1], b[3]));
        const double iw = dd_max(0.0, dd_sub(brx, tlx)), ih = dd_max(0.0, dd_sub(bry, tly));
        const double inter = dd_mul(iw, ih);
        const double uni = dd_sub(dd_add(t[4], dd_mul(b[2], b[3])), inter);
        return dd_sub(1.0, dd_div(inter, uni));
    }
    DD_HD double operator()(int r, int c) const {
        const double v = raw(r, c);
        return v > thr ? clip : v;
    }
};

template <class F>
struct DDTransposed {
    const F& f;
    DD_HD explicit DDTransposed(const F& f_) : f(f_) {}
    DD_HD double operator()(int i, int j) const { return f(j, i); }
};

// linear_assignment.py:11-75.  rows[nr] = track indices, cols = *und (ordered unmatched detections,
// nund entries).  Records matches in trk_det[], rewrites *und / nund with the new ordered
// unmatched-detection list.  Returns 0 or -1 (infeasible).
template <class G, class F>
DD_HD int dd_min_cost_matching(const G& g, const F& cost, double thr, DDMatchSmem& m, int nr,
                               short*& und, short*& und_next, int& nund) {
    const int nc = nund;
    if (nr == 0 || nc == 0) return 0;
    int rc;
    if (nc < nr) {
        DDTransposed<F> ct(cost);
        rc = dd_lsap_solve(g, nc, nr, ct, m.ls);
        for (int c = g.lane; c < nc; c += G::NL) m.c2r[c] = m.ls.col4row[c];
        for (int r = g.lane; r < nr; r += G::NL) m.r2c[r] = m.ls.row4col[r];
    } else {
        rc = dd_lsap_solve(g, nr, nc, cost, m.ls);
        for (int r = g.lane; r < nr; r += G::NL) m.r2c[r] = m.ls.col4row[r];
        for (int c = g.lane; c < nc; c += G::NL) m.c2r[c] = m.ls.row4col[c];
    }
    g.sync();
    if (rc != 0) return rc;
    int n2 = 0;
    for (int base = 0; base < nc; base += G::NL) {       // columns without a row, in column order
        const int c = base + g.lane;
        const bool p = c < nc && m.c2r[c] < 0;
        int tot;
        const int pos = g.scan_excl(p, tot);
        if (p) und_next[n2 + pos] = und[c];
        n2 += tot;
    }
    for (int base = 0; base < nr; base += G::NL) {       // assigned but over threshold, in row order
        const int r = base + g.lane;
        bool p = false;
        int c = -1;
        if (r < nr) {
            c = m.r2c[r];
            if (c >= 0) {
                p = cost(r, c) > thr;
                if (!p) m.trk_det[m.rows[r]] = und[c];
            }
        }
        int tot;
        const int pos = g.scan_excl(p, tot);
        if (p) und_next[n2 + pos] = und[c];
        n2 += tot;
    }
    g.sync();
    short* t = und; und = und_next; und_next = t;
    nund = n2;
    return 0;
}

template <class G>
DD_HD void dd_match_stream(const G& g, const DDView& V, int s, const double* det_tlwh,
                           const int* det_count, int* out_det_track_id, char* smem) {
    DDMatchSmem m;
    dd_match_carve(smem, V.T, V.D, V.tab_cap, m);
    const size_t sT = (size_t)s * V.T, sD = (size_t)s * V.D;
    // the count is loaded beside the presence word, off the warp's dependency chain; it is used only when present
    const int present = V.tick_present[s], nT = V.n_tracks[s], ndel_prev = V.n_deleted[s];
    int nd = det_count[s];
    if (!present) {                    // no frame: no detections to report, every track and slot stays as it is
        if (out_det_track_id)
            for (int d = g.lane; d < V.D; d += G::NL) out_det_track_id[sD + d] = -1;
        return;
    }
    if (nd > V.D) {
        nd = V.D;
        if (g.lane == 0) V.err[s] |= DD_FLAG_DET_OVERFLOW;
    }
    if (nd < 0) nd = 0;
    // slots deleted by the previous update become free now
    for (int k = g.lane; k < ndel_prev; k += G::NL) V.state[sT + V.deleted[sT + k]] = DD_STATE_FREE;
    // Staging loops of this function: the compiler cannot move a global load over the shared-memory store of the
    // iteration before it, so a plain loop pays one memory round trip per iteration -- and this warp is all latency.
    // They are therefore written in batches of DD_MB iterations: all loads of a batch first, then its stores.
    for (int t0 = g.lane; t0 < nT; t0 += DD_MB * G::NL) {
        int slot[DD_MB], tsu[DD_MB], st[DD_MB];
#pragma unroll
        for (int u = 0; u < DD_MB; ++u) slot[u] = t0 + u * G::NL < nT ? V.order[sT + t0 + u * G::NL] : 0;
#pragma unroll
        for (int u = 0; u < DD_MB; ++u) {
            tsu[u] = V.tsu[sT + slot[u]];
            st[u] = V.state[sT + slot[u]];
        }
#pragma unroll
        for (int u = 0; u < DD_MB; ++u) {
            const int t = t0 + u * G::NL;
            if (t >= nT) break;
            m.trk_slot[t] = (short)slot[u];
            m.trk_tsu[t] = (short)tsu[u];
            m.trk_state[t] = (unsigned char)st[u];
            m.trk_det[t] = -1;
        }
    }
    for (int d = g.lane; d < nd; d += G::NL) m.undA[d] = (short)d;
    for (int e0 = g.lane; e0 < nd * 4; e0 += DD_MB * G::NL) {
        double b[DD_MB];
#pragma unroll
        for (int u = 0; u < DD_MB; ++u) b[u] = e0 + u * G::NL < nd * 4 ? det_tlwh[sD * 4 + e0 + u * G::NL] : 0.0;
#pragma unroll
        for (int u = 0; u < DD_MB; ++u)
            if (e0 + u * G::NL < nd * 4) m.dbox[e0 + u * G::NL] = b[u];
    }
    g.sync();
    short *und = m.undA, *und_next = m.undB;
    int nund = nd;
    int infeasible = 0;

    // ---- confirmed tracks (tracker.py:108-111) -> lista, and the deepest occupied cascade level
    int nconf = 0, max_tsu = 0;
    for (int base = 0; base < nT; base += G::NL) {
        const int t = base + g.lane;
        const bool p = t < nT && m.trk_state[t] == DD_STATE_CONFIRMED;
        int tot;
        const int pos = g.scan_excl(p, tot);
        if (p) {
            m.lista[nconf + pos] = (short)t;
            max_tsu = dd_imax(max_tsu, (int)m.trk_tsu[t]);
        }
        nconf += tot;
    }
    max_tsu = g.imax(max_tsu);
    g.sync();

    // ---- matching cascade (linear_assignment.py:121-139)
    {
        for (int e0 = g.lane; e0 < nT * V.DW; e0 += DD_MB * G::NL) {      // stage the gate words (by track index)
            unsigned gw[DD_MB];
#pragma unroll
            for (int u = 0; u < DD_MB; ++u) {
                const int e = e0 + u * G::NL;
                gw[u] = 0u;
                if (e < nT * V.DW) {
                    const int t = e / V.DW, w = e - t * V.DW;
                    if (m.trk_state[t] == DD_STATE_CONFIRMED) gw[u] = V.gate[(sT + m.trk_slot[t]) * V.DW + w];
                }
            }
#pragma unroll
            for (int u = 0; u < DD_MB; ++u)
                if (e0 + u * G::NL < nT * V.DW) m.gate_sm[e0 + u * G::NL] = gw[u];
        }
        g.sync();
        // stage the first DD_CVAL gate-passing costs of every track: one track per lane, a cursor over its gate words,
        // the (<= DD_CVAL) loads of a track issued together from one 4*D-byte cost row
        for (int t = g.lane; t < nT; t += G::NL) {
            const float* crow = V.cost + (sT + m.trk_slot[t]) * V.D;
            const unsigned* gwp = m.gate_sm + t * V.DW;
            float cv[DD_CVAL];
            bool has[DD_CVAL];
            int w = 0;
            unsigned word = gwp[0];
#pragma unroll
            for (int k = 0; k < DD_CVAL; ++k) {
                while (!word && ++w < V.DW) word = gwp[w];
                has[k] = word != 0u;
                cv[k] = 0.0f;
                if (has[k]) {
                    cv[k] = crow[w * 32 + dd_ctz(word)];
                    word &= word - 1;
                }
            }
#pragma unroll
            for (int k = 0; k < DD_CVAL; ++k)
                if (has[k]) m.cval[t * DD_CVAL + k] = cv[k];
        }
        g.sync();
        DDCosineCost cc;
        cc.gate = m.gate_sm; cc.cval = m.cval; cc.cost = V.cost + sT * V.D;
        cc.trk_slot = m.trk_slot; cc.rows = m.rows; cc.D = V.D; cc.DW = V.DW;
        cc.thr = V.thr_cos; cc.clip = dd_add(V.thr_cos, 1e-5);
        const int depth = dd_imin(V.max_age, max_tsu);
        for (int level = 0; level < depth; ++level) {
            if (nund == 0) break;
            {   // jump to the next occupied level (levels without tracks are skipped by the reference too)
                int nxt = 0x7fffffff;
                for (int k = g.lane; k < nconf; k += G::NL) {
                    const int ts = m.trk_tsu[m.lista[k]];
                    if (ts >= 1 + level && ts < nxt) nxt = ts;
                }
                nxt = g.imin(nxt);
                if (nxt > depth) break;
                level = nxt - 1;
            }
            int nr = 0;
            for (int base = 0; base < nconf; base += G::NL) {
                const int k = base + g.lane;
                const bool p = k < nconf && m.trk_tsu[m.lista[k]] == 1 + level;
                int tot;
                const int pos = g.scan_excl(p, tot);
                if (p) m.rows[nr + pos] = m.lista[k];
                nr += tot;
            }
            g.sync();
            if (nr == 0) continue;
            cc.cols = und;
            if (dd_min_cost_matching(g, cc, V.thr_cos, m, nr, und, und_next, nund) != 0) infeasible = 1;
        }
    }

    // ---- unmatched confirmed tracks in CPython set order (linear_assignment.py:140)
    int n_unm_a = 0;
    {
        // ascending survivors by ordered compaction; is the confirmed list 0..nconf-1 (always, in this flow)?
        bool contig = true;
        int nsurv = 0;
        for (int base = 0; base < nconf; base += G::NL) {
            const int k = base + g.lane;
            bool p = false;
            if (k < nconf) {
                const int t = m.lista[k];
                contig = contig && (t == k);
                p = m.trk_det[t] < 0;
            }
            int tot;
            const int pos = g.scan_excl(p, tot);
            if (p) m.rows[nsurv + pos] = m.lista[k];
            nsurv += tot;
        }
        contig = g.all(contig);
        const int nmatched = nconf - nsurv;
        g.sync();
        if (contig && ((nconf >> 2) > nmatched || nsurv <= 1)) {
            for (int k = g.lane; k < nsurv; k += G::NL) m.listb[k] = m.rows[k];
            n_unm_a = nsurv;
        } else if (contig) {
            // one lane inserts (serial by nature), the group reads the slots back in order
            int tm = 0;
            if (g.lane == 0) tm = dd_set_build_from_survivors(m.rows, nsurv, m.tabA, m.tabB);
            tm = g.imax(tm);
            g.sync();
            const short* R = (tm >> 16) ? m.tabB : m.tabA;
            const int slots = (tm & 0xffff) + 1;
            for (int base = 0; base < slots; base += G::NL) {
                const int i = base + g.lane;
                const int e = i < slots ? R[i] : 0;
                int tot;
                const int pos = g.scan_excl(e != 0, tot);
                if (e) m.listb[n_unm_a + pos] = (short)(e - 1);
                n_unm_a += tot;
            }
        } else {
            for (int k = g.lane; k < nT; k += G::NL) m.flag[k] = 0;
            g.sync();
            for (int k = g.lane; k < nconf; k += G::NL)
                if (m.trk_det[m.lista[k]] >= 0) m.flag[m.lista[k]] = 1;
            g.sync();
            if (g.lane == 0)
                n_unm_a = dd_set_difference_order_serial(m.lista, nconf, m.flag, nmatched, m.listb,
                                                         m.tabA, m.tabB, m.tabC, m.tab_cap);
            n_unm_a = g.imax(n_unm_a);
        }
        g.sync();
    }

    // ---- IoU stage rows: unconfirmed (ascending) + set-ordered unmatched confirmed with tsu == 1
    int nr = 0;
    for (int base = 0; base < nT; base += G::NL) {
        const int t = base + g.lane;
        const bool p = t < nT && m.trk_state[t] != DD_STATE_CONFIRMED;
        int tot;
        const int pos = g.scan_excl(p, tot);
        if (p) m.rows[nr + pos] = (short)t;
        nr += tot;
    }
    for (int base = 0; base < n_unm_a; base += G::NL) {
        const int k = base + g.lane;
        const bool p = k < n_unm_a && m.trk_tsu[m.listb[k]] == 1;
        int tot;
        const int pos = g.scan_excl(p, tot);
        if (p) m.rows[nr + pos] = m.listb[k];
        nr += tot;
    }
    g.sync();
    if (nr > 0 && nund > 0) {
        for (int r = g.lane; r < nr; r += G::NL) {       // Track.to_tlwh of every IoU row, once
            const int t = m.rows[r];
            const double* mu = V.mean + (sT + m.trk_slot[t]) * 8;
            const double w = dd_mul(mu[2], mu[3]), h = mu[3];
            const double x = dd_sub(mu[0], dd_div(w, 2.0)), y = dd_sub(mu[1], dd_div(h, 2.0));
            double* o = m.tbox + r * 5;
            o[0] = x; o[1] = y; o[2] = dd_add(x, w); o[3] = dd_add(y, h);
            o[4] = m.trk_tsu[t] > 1 ? -1.0 : dd_mul(w, h);
        }
        g.sync();
        DDIouCost ic;
        ic.tbox = m.tbox; ic.det_tlwh = m.dbox; ic.cols = und;
        ic.thr = V.thr_iou; ic.clip = dd_add(V.thr_iou, 1e-5);
        if (dd_min_cost_matching(g, ic, V.thr_iou, m, nr, und, und_next, nund) != 0) infeasible = 1;
    }
    if (infeasible && g.lane == 0) V.err[s] |= DD_FLAG_LSAP_INFEASIBLE;

    // ---- lifecycle (tracker.py:72-81, track.py:127-152,190-196)
    for (int d = g.lane; d < V.D; d += G::NL) {
        V.det_kind[sD + d] = 0;
        V.det_slot[sD + d] = -1;
        if (out_det_track_id) out_det_track_id[sD + d] = -1;
    }
    g.sync();
    for (int t0 = g.lane; t0 < nT; t0 += DD_MB * G::NL) {
        int hit[DD_MB], tid[DD_MB];
#pragma unroll
        for (int u = 0; u < DD_MB; ++u) {        // hits and ids of the matched tracks of the batch, loaded together
            const int t = t0 + u * G::NL;
            hit[u] = tid[u] = 0;
            if (t < nT && m.trk_det[t] >= 0) {
                const size_t slot = sT + m.trk_slot[t];
                hit[u] = V.hits[slot];
                tid[u] = V.track_id[slot];
            }
        }
#pragma unroll
        for (int u = 0; u < DD_MB; ++u) {
            const int t = t0 + u * G::NL;
            if (t >= nT) break;
            const size_t slot = sT + m.trk_slot[t];
            const int d = m.trk_det[t];
            int st = m.trk_state[t];
            if (d >= 0) {
                const int hits = hit[u] + 1;
                V.hits[slot] = hits;
                V.tsu[slot] = 0;
                if (st == DD_STATE_TENTATIVE && hits >= V.n_init) st = DD_STATE_CONFIRMED;
                V.det_kind[sD + d] = 1;
                V.det_slot[sD + d] = m.trk_slot[t];
                if (out_det_track_id) out_det_track_id[sD + d] = tid[u];
            } else {
                if (st == DD_STATE_TENTATIVE) st = DD_STATE_DELETED;
                else if (m.trk_tsu[t] > V.max_age) st = DD_STATE_DELETED;
            }
            V.state[slot] = st;
            m.trk_state[t] = (unsigned char)st;
        }
    }
    g.sync();
    // free slots in ascending slot order -> lista; a free slot that still holds gallery pages (its track was
    // deleted by the previous update, or dropped by a host edit) returns them to the pool first
    int nfree = 0;
    for (int base0 = 0; base0 < V.T; base0 += DD_MB * G::NL) {
        int sst[DD_MB], snp[DD_MB];
#pragma unroll
        for (int u = 0; u < DD_MB; ++u) {
            const int k = base0 + u * G::NL + g.lane;
            sst[u] = k < V.T ? V.state[sT + k] : -1;
            snp[u] = k < V.T ? V.gal_np[sT + k] : 0;
        }
#pragma unroll
        for (int u = 0; u < DD_MB; ++u) {
            if (base0 + u * G::NL >= V.T) break;
            const int k = base0 + u * G::NL + g.lane;
            const bool p = k < V.T && sst[u] == DD_STATE_FREE;
            if (p && snp[u] > 0) {
                const int* pt = V.ptab + (sT + k) * V.PT;
                for (int i = 0; i < snp[u]; ++i) dd_page_free(V, pt[i]);
                V.gal_np[sT + k] = 0;
                V.gal_len[sT + k] = 0;
                V.gal_pos[sT + k] = 0;
            }
            int tot;
            const int pos = g.scan_excl(p, tot);
            if (p) m.lista[nfree + pos] = (short)k;
            nfree += tot;
        }
    }
    g.sync();
    int nnew = nund;
    if (nnew > nfree) {
        nnew = nfree;
        if (g.lane == 0) V.err[s] |= DD_FLAG_TRACK_OVERFLOW;
    }
    const int id0 = V.next_id[s];
    for (int k = g.lane; k < nnew; k += G::NL) {          // tracker.py:135-138, ids in list order
        const int d = und[k];
        const size_t slot = sT + m.lista[k];
        V.track_id[slot] = id0 + k;
        V.hits[slot] = 1;
        V.age[slot] = 1;
        V.tsu[slot] = 0;
        V.state[slot] = DD_STATE_TENTATIVE;
        V.det_kind[sD + d] = 2;
        V.det_slot[sD + d] = m.lista[k];
        if (out_det_track_id) out_det_track_id[sD + d] = id0 + k;
    }
    // stable split of the old list into live / deleted (tracker.py:80-81), then append new tracks
    int nlive = 0, ndel = 0;
    for (int base = 0; base < nT; base += G::NL) {
        const int t = base + g.lane;
        const bool in = t < nT;
        const bool dead = in && m.trk_state[t] == DD_STATE_DELETED;
        int tot_l, tot_d;
        const int pl = g.scan_excl(in && !dead, tot_l);
        const int pd = g.scan_excl(dead, tot_d);
        if (in && !dead) V.order[sT + nlive + pl] = m.trk_slot[t];
        if (dead) V.deleted[sT + ndel + pd] = m.trk_slot[t];
        nlive += tot_l;
        ndel += tot_d;
    }
    g.sync();
    for (int k = g.lane; k < nnew; k += G::NL) V.order[sT + nlive + k] = m.lista[k];
    if (g.lane == 0) {
        V.n_tracks[s] = nlive + nnew;
        V.n_deleted[s] = ndel;
        V.next_id[s] = id0 + nnew;
    }
}

// ------------------------------------------------------------------------------------------------
// Per-detection state update: Track.update (track.py:127-152) or Tracker._initiate_track
// (tracker.py:135-138 -> kalman_filter.py:55-86, track.py:67-82), then the gallery append that
// metric.partial_fit performs (nn_matching.py:137-154; ring of `budget` unit vectors) and the label
// vote.  scratch: >= 64 doubles per group.
// ------------------------------------------------------------------------------------------------
template <class G>
DD_HD void dd_apply_det(const G& g, const DDView& V, int s, int d, const float* det_conf,
                        const int* det_label, double* scratch) {
    const size_t sd = (size_t)s * V.D + d;
    // det_kind of a stream without a frame still holds what its last present tick matched
    const int present = V.tick_present[s], kind = V.det_kind[sd];
    if (!present || kind == 0) return;
    const size_t slot = (size_t)s * V.T + V.det_slot[sd];
    const double* z = V.det_xyah + sd * 4;
    // everything the tail needs is loaded before the Kalman arithmetic (independent of it; the compiler cannot
    // hoist these loads over the state stores itself): the feature chunks, the ring position, label and confidence
    constexpr int KP = (DD_FEAT_DIM / 4 + G::NL - 1) / G::NL;
    float4 x[KP];
    {
        const float4* src = (const float4*)(V.det_featn + sd * DD_FEAT_DIM);
        int kk = 0;
        for (int k = g.lane; k < DD_FEAT_DIM / 4; k += G::NL, ++kk) x[kk] = src[k];
    }
    int pos = V.gal_pos[slot];
    int len = V.gal_len[slot];
    int np = V.gal_np[slot];
    // the page the feature will land in, read ahead of the Kalman arithmetic like the other operands of the tail
    const int pid_hint = (kind == 1 && (pos >> 4) < np) ? V.ptab[slot * V.PT + (pos >> 4)] : -1;
    const int lbl = det_label[sd];
    const double conf = (double)det_conf[sd];
    const bool lbl_ok = lbl >= 0 && lbl < V.C;
    if (!lbl_ok && g.lane == 0) dd_atomic_or(V.err + s, DD_FLAG_BAD_LABEL);   // never counted for another class
    int lcnt = 0;
    double lsum = 0.0;
    if (kind == 1) {
        if (lbl_ok) {
            lcnt = V.lab_cnt[slot * V.C + lbl];
            lsum = V.lab_sum[slot * V.C + lbl];
        }
        dd_kf_update(g, V.mean + slot * 8, V.cov + slot * 64, z, scratch);
    } else {
        dd_kf_initiate(g, z, V.mean + slot * 8, V.cov + slot * 64);
        for (int c = g.lane; c < V.C; c += G::NL) {
            if (c == lbl) continue;                      // written below with the first vote
            V.lab_cnt[slot * V.C + c] = 0;
            V.lab_sum[slot * V.C + c] = 0.0;
        }
        if (g.lane == 0) {
            V.path_n[slot] = 0;
            V.path_crossed[slot] = 0;
        }
        pos = 0;       // a recycled slot gave its pages back in the matching kernel (np == 0 already)
        len = 0;
    }
    dd_gallery_append<G, KP>(g, V, s, slot, pos, len, np, x, pid_hint);
    if (g.lane == 0 && lbl_ok) {
        V.lab_cnt[slot * V.C + lbl] = lcnt + 1;
        V.lab_sum[slot * V.C + lbl] = dd_add(lsum, conf);
    }
}

// ------------------------------------------------------------------------------------------------
// Count-line (tools/intersection.py:4-24, deepdish.py:1041-1112,1303-1312, track.py:154-188).
// ------------------------------------------------------------------------------------------------
DD_HD double dd_cross2(double a0, double a1, double b0, double b1) {
    return dd_sub(dd_mul(a0, b1), dd_mul(a1, b0));
}

// intersection(p, pr, q, qs) with points given as (x, y) pairs.
DD_HD bool dd_segments_intersect(double px, double py, double prx, double pry, double qx, double qy,
                                 double qsx, double qsy) {
    const double eps = 2.220446049250313e-16;            // sys.float_info.epsilon
    const double rx = dd_sub(prx, px), ry = dd_sub(pry, py);
    const double sx = dd_sub(qsx, qx), sy = dd_sub(qsy, qy);
    const double rxs = dd_cross2(rx, ry, sx, sy);
    const double qmpx = dd_sub(qx, px), qmpy = dd_sub(qy, py);
    const double qpxr = dd_cross2(qmpx, qmpy, rx, ry);
    if (fabs(rxs) < eps) {
        if (fabs(qpxr) < eps) {
            const double rr = dd_add(dd_mul(rx, rx), dd_mul(ry, ry));
            const double ax = dd_div(rx, rr), ay = dd_div(ry, rr);
            double t0 = dd_add(dd_mul(qmpx, ax), dd_mul(qmpy, ay));
            double t1 = dd_add(t0, dd_add(dd_mul(sx, ax), dd_mul(sy, ay)));
            if (t0 > t1) { const double tmp = t0; t0 = t1; t1 = tmp; }
            return !(t1 < 0.0 || t0 > 1.0);
        }
        return false;
    }
    const double t = dd_div(dd_cross2(qmpx, qmpy, sx, sy), rxs);
    const double u = dd_div(qpxr, rxs);
    return 0.0 <= t && t <= 1.0 && 0.0 <= u && u <= 1.0;
}

// Track.get_label (track.py:154-188): Dirichlet-expected vote, reverse (value, name) order,
// motorbike/bicycle rule.  Returns the label index (or -1 when the track has no votes).
DD_HD int dd_get_label(const DDView& V, size_t slot) {
    const int* cnt = V.lab_cnt + slot * V.C;
    const double* sum = V.lab_sum + slot * V.C;
    double tot_c = 0.0, tot_a = 0.0;
    for (int c = 0; c < V.C; ++c)
        if (cnt[c] > 0) {
            tot_c = dd_add(tot_c, (double)cnt[c]);
            tot_a = dd_add(tot_a, dd_div(sum[c], (double)cnt[c]));
        }
    const double den = dd_add(tot_c, tot_a);
    int b1 = -1, b2 = -1;
    double v1 = 0.0, v2 = 0.0;
    for (int c = 0; c < V.C; ++c) {
        if (cnt[c] <= 0) continue;
        const double v = dd_div(dd_add(dd_div(sum[c], (double)cnt[c]), (double)cnt[c]), den);
        const bool gt1 = b1 < 0 || v > v1 || (v == v1 && V.label_rank[c] > V.label_rank[b1]);
        if (gt1) {
            b2 = b1; v2 = v1;
            b1 = c; v1 = v;
        } else {
            const bool gt2 = b2 < 0 || v > v2 || (v == v2 && V.label_rank[c] > V.label_rank[b2]);
            if (gt2) { b2 = c; v2 = v; }
        }
    }
    if (b2 >= 0 && b1 == V.lbl_motorbike && b2 == V.lbl_bicycle && V.lbl_motorbike >= 0)
        return (v1 > dd_mul(v2, 4.0)) ? b1 : b2;
    return b1;
}

// One live track's count-line step (deepdish.py:1046-1112): path point, crossing test, counters.  Returns the counter
// column its crossing incremented (0 pos, 1 neg; int as well) with its label in *label, or -1.
DD_HD int dd_countline_track(const DDView& V, size_t slot, double p1x, double p1y, double q1x, double q1y,
                             long long* cnt, int* label) {
    if (V.state[slot] != DD_STATE_CONFIRMED || V.tsu[slot] > 1) return -1;
    int col = -1;
    const double* m = V.mean + slot * 8;
    // Track.to_tlbr (track.py:84-111) and the bottom-centre point (deepdish.py:1060-1063)
    const double w = dd_mul(m[2], m[3]), h = m[3];
    const double x = dd_sub(m[0], dd_div(w, 2.0)), y = dd_sub(m[1], dd_div(h, 2.0));
    const double x2 = dd_add(x, w), y2 = dd_add(y, h);
    const double bx = dd_div(dd_add(x, x2), 2.0), by = y2;
    const int n = V.path_n[slot];
    if (n >= 1) {
        const double lx = V.path_last[slot * 2], ly = V.path_last[slot * 2 + 1];
        // p2 = latest, q2 = previous (deepdish.py:1073-1075)
        const double cp = dd_cross2(dd_sub(q1x, p1x), dd_sub(q1y, p1y), dd_sub(lx, bx), dd_sub(ly, by));
        if (dd_segments_intersect(p1x, p1y, q1x, q1y, bx, by, lx, ly)) {
            const int l = dd_get_label(V, slot);
            if (l >= 0) {
                col = cp >= 0.0 ? 0 : 1;
                dd_atomic_add_ll(cnt + l * 4 + col, 1);
                dd_atomic_add_ll(cnt + l * 4 + 2, 1);
                *label = l;
            }
        }
        // any_intersection walks the path forwards: segment (previous, latest)
        if (dd_segments_intersect(p1x, p1y, q1x, q1y, lx, ly, bx, by)) V.path_crossed[slot] = 1;
    }
    V.path_last[slot * 2] = bx;
    V.path_last[slot * 2 + 1] = by;
    V.path_n[slot] = n + 1;
    return col;
}

DD_HD void dd_put_event(const DDView& V, int pos, int s, int track_id, int label, int col) {
    if (pos >= V.ev_cap) return;                     // overflow: counted in header[0], not written
    int* r = V.ev + 4 + (size_t)pos * 4;
    r[0] = s; r[1] = track_id; r[2] = label; r[3] = col;
}

// EV (config.event_cap > 0, V.ev set): the same counter increments, and one crossing record per increment (layout
// `events`).  The track loop then runs in warp-uniform rounds: each round's crossings are compacted in order and take
// their positions with one atomicAdd on header[0], so a stream's records keep the order of tracker.tracks.
template <class G, bool EV = false>
DD_HD void dd_countline(const G& g, const DDView& V, int s, const double* line) {
    const size_t sT = (size_t)s * V.T;
    const double p1x = line[0], p1y = line[1], q1x = line[2], q1y = line[3];
    long long* cnt = V.counts + (size_t)s * V.C * 4;
    const int present = V.tick_present[s], ndel = V.n_deleted[s], nT = V.n_tracks[s];
    // a stream without a frame in the last tick takes no count-line step: in particular the last track its previous
    // present tick deleted is not counted a second time
    if (!present) return;
    // deleted tracks (deepdish.py:1041-1044): only the LAST one's result survives the overwrite
    int del_label = -1, del_id = 0;
    if (g.lane == 0 && ndel > 0) {
        const size_t slot = sT + V.deleted[sT + ndel - 1];
        if (V.path_n[slot] > 1 && V.path_crossed[slot]) {
            const int l = dd_get_label(V, slot);
            if (l >= 0) dd_atomic_add_ll(cnt + l * 4 + 3, 1);
            if (EV) { del_label = l; del_id = V.track_id[slot]; }
        }
    }
    if constexpr (!EV) {
        for (int t = g.lane; t < nT; t += G::NL) {
            int l;
            dd_countline_track(V, sT + V.order[sT + t], p1x, p1y, q1x, q1y, cnt, &l);
        }
    } else {
        for (int t0 = 0; t0 < nT; t0 += G::NL) {
            const int t = t0 + g.lane;
            int l = -1, col = -1;
            size_t slot = 0;
            if (t < nT) {
                slot = sT + V.order[sT + t];
                col = dd_countline_track(V, slot, p1x, p1y, q1x, q1y, cnt, &l);
            }
            int total = 0;
            const int rank = g.scan_excl(col >= 0, total);
            if (total == 0) continue;
            int base = 0;
            if (g.lane == 0) base = dd_atomic_add_i(V.ev, total);
            base = g.imax(g.lane == 0 ? base : 0);        // lane 0's reservation to every lane (base >= 0)
            if (col >= 0) dd_put_event(V, base + rank, s, V.track_id[slot], l, col);
        }
        if (g.lane == 0 && del_label >= 0) dd_put_event(V, dd_atomic_add_i(V.ev, 1), s, del_id, del_label, 3);
    }
}

// ------------------------------------------------------------------------------------------------
// Several count lines per stream (config.n_lines = L > 1).  Line l is counted into counts[s][l] exactly as the
// reference's process_results counts its one line; dd_countline above stays the one-line step.
// ------------------------------------------------------------------------------------------------
// One live track's step against the stream's L lines (lines[4 l ..] = x1, y1, x2, y2): the bottom-centre point once,
// each line's crossing and direction test against the previous point, get_label once if some line was crossed, the
// path_crossed bits and the path point once.  Returns the mask of the lines whose counters it incremented (bit l), with
// the neg direction of each in *neg (bit l set: column 1, else 0) and its label in *label.
DD_HD unsigned dd_countline_track_lines(const DDView& V, size_t slot, const double* lines, long long* cnt,
                                        unsigned* neg, int* label) {
    if (V.state[slot] != DD_STATE_CONFIRMED || V.tsu[slot] > 1) return 0u;
    unsigned hit = 0u;
    const double* m = V.mean + slot * 8;
    const double w = dd_mul(m[2], m[3]), h = m[3];
    const double x = dd_sub(m[0], dd_div(w, 2.0)), y = dd_sub(m[1], dd_div(h, 2.0));
    const double x2 = dd_add(x, w), y2 = dd_add(y, h);
    const double bx = dd_div(dd_add(x, x2), 2.0), by = y2;
    const int n = V.path_n[slot];
    if (n >= 1) {
        const double lx = V.path_last[slot * 2], ly = V.path_last[slot * 2 + 1];
        unsigned ng = 0u, crossed = 0u;
        for (int l = 0; l < V.n_lines; ++l) {
            const double p1x = lines[l * 4], p1y = lines[l * 4 + 1], q1x = lines[l * 4 + 2], q1y = lines[l * 4 + 3];
            if (dd_segments_intersect(p1x, p1y, q1x, q1y, bx, by, lx, ly)) {
                const double cp = dd_cross2(dd_sub(q1x, p1x), dd_sub(q1y, p1y), dd_sub(lx, bx), dd_sub(ly, by));
                hit |= 1u << l;
                if (!(cp >= 0.0)) ng |= 1u << l;
            }
            if (dd_segments_intersect(p1x, p1y, q1x, q1y, lx, ly, bx, by)) crossed |= 1u << l;
        }
        if (hit) {
            const int lab = dd_get_label(V, slot);
            if (lab >= 0) {
                for (int l = 0; l < V.n_lines; ++l) {
                    if (!((hit >> l) & 1u)) continue;
                    long long* c = cnt + ((size_t)l * V.C + lab) * 4;
                    dd_atomic_add_ll(c + ((ng >> l) & 1u), 1);
                    dd_atomic_add_ll(c + 2, 1);
                }
                *neg = ng;
                *label = lab;
            } else {
                hit = 0u;
            }
        }
        if (crossed) V.path_crossed[slot] |= (int)crossed;
    }
    V.path_last[slot * 2] = bx;
    V.path_last[slot * 2 + 1] = by;
    V.path_n[slot] = n + 1;
    return hit;
}

// dd_countline for L lines; `lines` = the stream's [L,4] segments (the kernel stages them in shared memory).  EV: one
// record per counter increment, column word = column + 4 line.  A lane writes up to L records in a round, so the
// round's records are placed with a warp prefix sum of the per-lane counts: a stream's records follow tracker.tracks,
// each track's lines ascending, then the deletion records, lines ascending.
template <class G, bool EV = false>
DD_HD void dd_countline_lines(const G& g, const DDView& V, int s, const double* lines) {
    const size_t sT = (size_t)s * V.T;
    long long* cnt = V.counts + (size_t)s * V.n_lines * V.C * 4;
    const int present = V.tick_present[s], ndel = V.n_deleted[s], nT = V.n_tracks[s];
    if (!present) return;
    // deleted tracks (deepdish.py:1041-1044): only the LAST one's result survives the overwrite, on every line whose
    // bit its path set
    int del_label = -1, del_id = 0;
    unsigned del_lines = 0u;
    if (g.lane == 0 && ndel > 0) {
        const size_t slot = sT + V.deleted[sT + ndel - 1];
        const unsigned crossed = (unsigned)V.path_crossed[slot];
        if (V.path_n[slot] > 1 && crossed) {
            const int l = dd_get_label(V, slot);
            if (l >= 0)
                for (int k = 0; k < V.n_lines; ++k)
                    if ((crossed >> k) & 1u) dd_atomic_add_ll(cnt + ((size_t)k * V.C + l) * 4 + 3, 1);
            if (EV) { del_label = l; del_id = V.track_id[slot]; del_lines = crossed; }
        }
    }
    if constexpr (!EV) {
        for (int t = g.lane; t < nT; t += G::NL) {
            unsigned ng;
            int l;
            dd_countline_track_lines(V, sT + V.order[sT + t], lines, cnt, &ng, &l);
        }
    } else {
        for (int t0 = 0; t0 < nT; t0 += G::NL) {
            const int t = t0 + g.lane;
            unsigned hit = 0u, ng = 0u;
            int l = -1;
            size_t slot = 0;
            if (t < nT) {
                slot = sT + V.order[sT + t];
                hit = dd_countline_track_lines(V, slot, lines, cnt, &ng, &l);
            }
            int total = 0;
            const int rank = g.scan_excl_sum(dd_popc(hit), total);
            if (total == 0) continue;
            int base = 0;
            if (g.lane == 0) base = dd_atomic_add_i(V.ev, total);
            base = g.imax(g.lane == 0 ? base : 0);        // lane 0's reservation to every lane (base >= 0)
            if (hit) {
                int pos = base + rank;
                const int tid = V.track_id[slot];
                for (int k = 0; k < V.n_lines; ++k)
                    if ((hit >> k) & 1u) dd_put_event(V, pos++, s, tid, l, (int)((ng >> k) & 1u) + 4 * k);
            }
        }
        if (g.lane == 0 && del_label >= 0) {
            int pos = dd_atomic_add_i(V.ev, dd_popc(del_lines));
            for (int k = 0; k < V.n_lines; ++k)
                if ((del_lines >> k) & 1u) dd_put_event(V, pos++, s, del_id, del_label, 3 + 4 * k);
        }
    }
}
