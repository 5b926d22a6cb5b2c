// dd_detect_bodies.cuh -- detector post-processing bodies (group-generic, see dd_common.cuh).
//
//   dd_nms_frame        one CTA per frame: preprocessing.non_max_suppression as sort + bitmask + scan
//   dd_yolo_rows        one thread per anchor row of a staged tile: YOLOv5 head decode + box filter
//   dd_order_frame      one CTA per frame: put the appended candidates back into anchor order
#pragma once
#include "dd_common.cuh"
#include "dd_lsap.cuh"
#include "../../include/deepdish_b200.h"

// ---- order-preserving f32 <-> u32 key (ascending key == ascending float) ---------------------
DD_HD unsigned dd_f32_key(float f) {
    union { float f; unsigned u; } c;
    c.f = f;
    return (c.u & 0x80000000u) ? ~c.u : (c.u | 0x80000000u);
}

// In-place ascending bitonic sort of P (power of two) 64-bit keys by the whole group.
template <class G>
DD_HD void dd_bitonic_sort(const G& g, unsigned long long* keys, int P) {
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = g.lane; i < P; i += g.nl) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = keys[i], b = keys[ixj];
                    const bool up = (i & k) == 0;
                    if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
                }
            }
            g.sync();
        }
    }
}

DD_HD int dd_next_pow2(int n) {
    int p = 1;
    while (p < n) p <<= 1;
    return p;
}

struct alignas(16) DDIBox { int x1, y1, x2, y2; };

// Shared-memory plan of dd_nms_frame for up to nmax candidates.
#define DD_NMS_BATCH 32          // survivors-so-far whose suppression rows are evaluated together
struct DDNmsSmem {
    unsigned long long* ukeys;  // [nmax] unsorted (score desc, index asc) keys
    unsigned long long* keys;   // [nmax] sorted
    unsigned* remv;             // [nh]   removed bits by rank (32 per word)
    unsigned* rows;             // [DD_NMS_BATCH][nh] suppression rows of the current batch
    int* batch;                 // [DD_NMS_BATCH + 2] ranks of the batch, then {count, next cursor}
    double *x1, *y1, *x2, *y2, *area;   // [nmax] in rank order
    DDIBox* ibox;                       // [nmax] integer copies (valid when every box is integer-valued)
    int* allint;                        // [1]
};
DD_HD size_t dd_nms_smem_bytes(int nmax) {
    const int nh = (nmax + 31) / 32;
    return (size_t)nmax * 16 + (size_t)nh * 4 * (1 + DD_NMS_BATCH) + (DD_NMS_BATCH + 2) * 4 + 16 +
           (size_t)nmax * 5 * 8 + (size_t)nmax * 16 + 32;
}
DD_HD void dd_nms_carve(char* mem, int nmax, DDNmsSmem& m) {
    const int nh = (nmax + 31) / 32;
    m.ukeys = (unsigned long long*)mem;
    m.keys = m.ukeys + nmax;
    m.x1 = (double*)(m.keys + nmax);
    m.y1 = m.x1 + nmax; m.x2 = m.y1 + nmax; m.y2 = m.x2 + nmax; m.area = m.y2 + nmax;
    m.ibox = (DDIBox*)(((uintptr_t)(m.area + nmax) + 15) & ~(uintptr_t)15);
    m.remv = (unsigned*)(m.ibox + nmax);
    m.rows = m.remv + nh;
    m.batch = (int*)(m.rows + (size_t)DD_NMS_BATCH * nh);
    m.allint = m.batch + DD_NMS_BATCH + 2;
}

// Does box A (the higher-ranked pick) suppress box J:  fl(inter / area_J) > max_overlap, +1 px convention
// (preprocessing.py:59-71), all f64.  Exact without a division in the common cases: disjoint boxes never
// suppress (for thresholds >= 0); otherwise inter is compared against max_overlap * area_J with a 2^-40
// relative guard band and only inside the band the division decides.
DD_HD bool dd_nms_suppresses(double ax1, double ay1, double ax2, double ay2, double jx1, double jy1, double jx2,
                             double jy2, double aj, double max_overlap, bool fast) {
    double iw = dd_add(dd_sub(dd_min(ax2, jx2), dd_max(ax1, jx1)), 1.0);
    if (fast && !(iw > 0.0)) return false;
    double ih = dd_add(dd_sub(dd_min(ay2, jy2), dd_max(ay1, jy1)), 1.0);
    if (fast && !(ih > 0.0)) return false;
    iw = dd_max(0.0, iw);
    ih = dd_max(0.0, ih);
    const double inter = dd_mul(iw, ih);
    if (fast && aj > 0.0) {
        const double t = max_overlap * aj;
        if (inter > t * (1.0 + 9.094947017729282e-13)) return true;
        if (inter < t * (1.0 - 9.094947017729282e-13)) return false;
    }
    return dd_div(inter, aj) > max_overlap;
}

// deep_sort/preprocessing.py:6-73.  boxes f64 [n,4] tlwh, scores f32 [n].  keep[] receives the
// original indices in pick order (descending score); returns their number through *nkeep.
//   rank     : descending score; among equal scores the HIGHER original index is picked first.  That is what the
//              reference does for the frame sizes deepdish sees: np.argsort(scores) (preprocessing.py:50) is a
//              stable insertion sort for n <= 16 and the loop pops from the end of the ascending order.  For
//              n > 16 numpy switches to an unstable (SIMD) sort and the order of tied scores is numpy's
//              implementation detail; this rule is kept there too.  Ranks by counting smaller keys (n^2 / 32 warp ops);
//   greedy   : the reference keeps a candidate unless an earlier survivor suppresses it
//              (inter(i,j) / area(j) > max_overlap, +1 pixel convention, f64 like boxes.astype(float)).  Only
//              survivors' suppression rows are ever needed, so they are built lazily: take the next <= 32
//              candidates that are still alive, build their rows over all later candidates in parallel
//              (one warp per 32 candidates, ballots give the bits; integer-valued boxes -- the pipeline's
//              case -- are tested for disjointness in int32 first), then scan the batch serially with the
//              removed bits held in the scanning warp's registers.
// (Measured and dropped, round 2: building the WHOLE upper-triangular suppression matrix in one parallel sweep followed by
// a single serial scan -- no barrier per 32 survivors -- takes 0.135 ms for C2's 64 frames x 540 candidates against
// 0.125 ms for the lazy batches below: the frame's CTA is bound by its instruction count, and the full matrix tests 3x
// the pairs.)
template <class G>
DD_HD void dd_nms_frame(const G& g, const double* boxes, const float* scores, int n, int nmax,
                        double max_overlap, int* keep, int* nkeep, char* smem) {
    if (n > nmax) n = nmax;
    if (n <= 0) {
        if (g.lane == 0) *nkeep = 0;
        return;
    }
    DDNmsSmem m;
    dd_nms_carve(smem, nmax, m);
    const int nh = (n + 31) / 32;
    for (int i = g.lane; i < n; i += g.nl)
        m.ukeys[i] = ((unsigned long long)(~dd_f32_key(scores[i])) << 32) | (0xffffffffu - (unsigned)i);
    for (int w = g.lane; w < nh; w += g.nl) m.remv[w] = 0u;
    if (g.lane == 0) { *m.allint = 1; m.batch[DD_NMS_BATCH + 1] = 0; }
    g.sync();
    for (int i = g.lane; i < n; i += g.nl) {                 // rank = number of smaller keys (keys are distinct)
        const unsigned long long k = m.ukeys[i];
        int r = 0;
        for (int j = 0; j < n; ++j) r += m.ukeys[j] < k;
        m.keys[r] = k;
        const int o = (int)(0xffffffffu - (unsigned)(k & 0xffffffffu));
        const double x = boxes[o * 4 + 0], y = boxes[o * 4 + 1], w = boxes[o * 4 + 2], h = boxes[o * 4 + 3];
        const double xx2 = dd_add(w, x), yy2 = dd_add(h, y);
        m.x1[r] = x; m.y1[r] = y; m.x2[r] = xx2; m.y2[r] = yy2;
        m.area[r] = dd_mul(dd_add(dd_sub(xx2, x), 1.0), dd_add(dd_sub(yy2, y), 1.0));
        // |coords| < 2^20 keeps every int32 intermediate of the disjointness test exact
        const bool isint = x == (double)(int)x && y == (double)(int)y && xx2 == (double)(int)xx2 && yy2 == (double)(int)yy2 &&
                           fabs(x) < 1048576.0 && fabs(y) < 1048576.0 && fabs(xx2) < 1048576.0 && fabs(yy2) < 1048576.0;
        if (isint) { DDIBox q; q.x1 = (int)x; q.y1 = (int)y; q.x2 = (int)xx2; q.y2 = (int)yy2; m.ibox[r] = q; }
        else *m.allint = 0;
    }
    g.sync();
    const bool fast = max_overlap >= 0.0;
    const bool ints = fast && *m.allint != 0;
    int nk = 0;
#if defined(__CUDA_ARCH__)
    // first warp: removed bits live in registers (lane w owns ranks 32w..32w+31) when they fit
    const bool regpath = nh <= 32;
    unsigned remv_reg = 0u;
    int cursor_reg = 0;
#endif
    while (true) {
        // ---- next batch: up to DD_NMS_BATCH ranks >= cursor whose removed bit is clear (first warp)
        if (g.lane < 32) {
            int nb = 0;
#if defined(__CUDA_ARCH__)
            int cursor = regpath ? cursor_reg : m.batch[DD_NMS_BATCH + 1];
            while (nb < DD_NMS_BATCH && cursor < n) {
                const int r = cursor + g.lane;
                const unsigned word = regpath ? __shfl_sync(0xffffffffu, remv_reg, (r >> 5) & 31)
                                              : (r < n ? m.remv[r >> 5] : 0u);
                const bool alive = r < n && !((word >> (r & 31)) & 1u);
                const unsigned bal = __ballot_sync(0xffffffffu, alive);
                const int pos = nb + __popc(bal & ((1u << g.lane) - 1u));
                if (alive && pos < DD_NMS_BATCH) m.batch[pos] = r;
                const int tot = __popc(bal);
                if (nb + tot > DD_NMS_BATCH) {              // batch full inside this window: resume after its last rank
                    const int last = __fns(bal, 0, DD_NMS_BATCH - nb);      // bit of the (BATCH-nb)-th set bit
                    cursor += last + 1;
                    nb = DD_NMS_BATCH;
                } else {
                    nb += tot;
                    cursor += 32;
                }
            }
            cursor_reg = cursor;
#else
            int cursor = m.batch[DD_NMS_BATCH + 1];
            while (nb < DD_NMS_BATCH && cursor < n) {
                if (!((m.remv[cursor >> 5] >> (cursor & 31)) & 1u)) m.batch[nb++] = cursor;
                ++cursor;
            }
#endif
            dd_first_warp_sync();
            if (g.lane == 0) { m.batch[DD_NMS_BATCH] = nb; m.batch[DD_NMS_BATCH + 1] = cursor < n ? cursor : n; }
        }
        g.sync();
        const int nb = m.batch[DD_NMS_BATCH];
        if (nb == 0) break;
        // ---- suppression rows of the batch over the later candidates
#if defined(__CUDA_ARCH__)
        {
            // one warp per batch member: its box stays in registers while the warp sweeps the later candidates, 32 per
            // step; candidates already removed need no bit (OR-ing them into the removed set again changes nothing)
            const int wid = g.lane >> 5, ln = g.lane & 31, nwarp = g.nl >> 5;
            for (int b = wid; b < nb; b += nwarp) {
                const int i = m.batch[b];
                DDIBox bi;
                bi.x1 = bi.y1 = bi.x2 = bi.y2 = 0;
                if (ints) bi = m.ibox[i];
                for (int hw = i >> 5; hw < nh; ++hw) {
                    const int j = hw * 32 + ln;
                    const unsigned gone = m.remv[hw];
                    bool sup = false;
                    if (j > i && j < n && !((gone >> ln) & 1u)) {
                        bool test = true;
                        if (ints) {
                            const DDIBox bj = m.ibox[j];
                            test = (min(bi.x2, bj.x2) - max(bi.x1, bj.x1) + 1 > 0) &&
                                   (min(bi.y2, bj.y2) - max(bi.y1, bj.y1) + 1 > 0);
                        }
                        if (test)
                            sup = dd_nms_suppresses(m.x1[i], m.y1[i], m.x2[i], m.y2[i], m.x1[j], m.y1[j], m.x2[j],
                                                    m.y2[j], m.area[j], max_overlap, fast);
                    }
                    const unsigned bits = __ballot_sync(0xffffffffu, sup);
                    if (ln == 0) m.rows[b * nh + hw] = bits;
                }
            }
        }
#else
        for (int e = g.lane; e < nb * nh; e += g.nl) {
            const int b = e / nh, hw = e - b * nh;
            const int i = m.batch[b];
            unsigned bits = 0;
            for (int j = dd_imax(i + 1, hw * 32); j < dd_imin(n, hw * 32 + 32); ++j)
                if (dd_nms_suppresses(m.x1[i], m.y1[i], m.x2[i], m.y2[i], m.x1[j], m.y1[j], m.x2[j], m.y2[j],
                                      m.area[j], max_overlap, fast))
                    bits |= 1u << (j - hw * 32);
            m.rows[e] = bits;
        }
#endif
        g.sync();
        // ---- serial scan of the batch (first warp)
        if (g.lane < 32) {
#if defined(__CUDA_ARCH__)
            if (regpath) {
                const int mine = g.lane < nb ? m.batch[g.lane] : 0;
                for (int b = 0; b < nb; ++b) {
                    const int i = __shfl_sync(0xffffffffu, mine, b);
                    const unsigned word = __shfl_sync(0xffffffffu, remv_reg, i >> 5);
                    if ((word >> (i & 31)) & 1u) continue;                 // suppressed inside the batch
                    if (g.lane == 0) keep[nk] = (int)(0xffffffffu - (unsigned)(m.keys[i] & 0xffffffffu));
                    ++nk;
                    if (g.lane >= (i >> 5) && g.lane < nh) remv_reg |= m.rows[b * nh + g.lane];
                }
                if (g.lane < nh) m.remv[g.lane] = remv_reg;                // the next batch's row builders skip removed candidates
            } else
#endif
            {
                const int nscan = g.nl < 32 ? g.nl : 32;
                for (int b = 0; b < nb; ++b) {
                    const int i = m.batch[b];
                    if ((m.remv[i >> 5] >> (i & 31)) & 1u) continue;       // suppressed inside the batch
                    if (g.lane == 0) keep[nk] = (int)(0xffffffffu - (unsigned)(m.keys[i] & 0xffffffffu));
                    ++nk;
                    for (int w = (i >> 5) + g.lane; w < nh; w += nscan) m.remv[w] |= m.rows[b * nh + w];
                    dd_first_warp_sync();
                }
            }
        }
        g.sync();
    }
    if (g.lane == 0) *nkeep = nk;
}

// ------------------------------------------------------------------------------------------------
// The pre-NMS box filter of Pipeline.detect_objects for ONE box (deepdish.py:950-955):
//   x, y = int(np.clip(x, 0, W)), int(np.clip(y, 0, H));  w, h = int(np.clip(w, 0, W - x)), int(np.clip(h, 0, H - y))
//   reject w * h > 0.9 * W * H.   int() truncates toward zero; f32 inputs are widened exactly.
// The frame-level NaN rule (:947-949: one NaN anywhere drops every box of the frame) is the caller's.
// ------------------------------------------------------------------------------------------------
DD_HD bool dd_box_clip(double x, double y, double w, double h, int frame_w, int frame_h, double max_area, int* o) {
    const double fx = x < 0.0 ? 0.0 : (x > (double)frame_w ? (double)frame_w : x);
    const double fy = y < 0.0 ? 0.0 : (y > (double)frame_h ? (double)frame_h : y);
    const int ix = (int)fx, iy = (int)fy;
    const double mw = (double)(frame_w - ix), mh = (double)(frame_h - iy);
    const double fw = w < 0.0 ? 0.0 : (w > mw ? mw : w);
    const double fh = h < 0.0 ? 0.0 : (h > mh ? mh : h);
    const int iw = (int)fw, ih = (int)fh;
    if ((double)((long long)iw * ih) > max_area) return false;
    o[0] = ix; o[1] = iy; o[2] = iw; o[3] = ih;
    return true;
}

// ------------------------------------------------------------------------------------------------
// YOLOv5 head row decode (tools/yolov5.py:120-146) + box filter (deepdish.py:946-955).
// row: 5+nc f32 values (x, y, w, h normalised, obj, cls...).  Returns true when the row survives
// every filter; the emitted box is the integer-valued tlwh after clipping.
// ------------------------------------------------------------------------------------------------
struct DDYoloParams {
    int nc;
    float thr;
    float img_w, img_h;       // PIL image size the head is scaled to (yolov5.py:131)
    int frame_w, frame_h;     // camera viewport of the box filter (deepdish.py:945)
    double max_area;          // 0.9 * frame_w * frame_h
};

template <class Row>
DD_HD bool dd_yolo_row(const Row& row, const DDYoloParams& p, const unsigned char* wanted,
                       double* out_tlwh, float* out_score, int* out_class, bool* out_nan) {
    const float obj = row(4);
    float best = dd_mulf(row(5), obj);
    int bi = 0;
    bool nan = best != best;
    for (int c = 1; c < p.nc; ++c) {
        const float v = dd_mulf(row(5 + c), obj);
        if (v > best) { best = v; bi = c; }              // np.argmax: first maximum wins
        nan = nan || v != v;
    }
    // np.argmax returns the first NaN when there is one, and a NaN score fails the threshold: a NaN product anywhere
    // in the row drops it, even when another class passes
    if (nan || !(best >= p.thr)) return false;           // yolov5.py:130
    if (!wanted[bi]) return false;                       // yolov5.py:139
    const float cx = row(0), cy = row(1), w = row(2), h = row(3);
    const float hx = dd_divf(w, 2.0f), hy = dd_divf(h, 2.0f);
    const float x1 = dd_mulf(dd_subf(cx, hx), p.img_w), y1 = dd_mulf(dd_subf(cy, hy), p.img_h);
    const float x2 = dd_mulf(dd_addf(cx, hx), p.img_w), y2 = dd_mulf(dd_addf(cy, hy), p.img_h);
    const float bw = dd_subf(x2, x1), bh = dd_subf(y2, y1);       // yolov5.py:141-142
    if (p.frame_w <= 0) {            // adapter mode: detect_image's own output, no box filter
        out_tlwh[0] = x1; out_tlwh[1] = y1; out_tlwh[2] = bw; out_tlwh[3] = bh;
        *out_score = best;
        *out_class = bi;
        return true;
    }
    *out_nan = (x1 != x1) || (y1 != y1) || (bw != bw) || (bh != bh);
    int ib[4];
    if (!dd_box_clip(x1, y1, bw, bh, p.frame_w, p.frame_h, p.max_area, ib)) return false;      // deepdish.py:950-953
    out_tlwh[0] = ib[0]; out_tlwh[1] = ib[1]; out_tlwh[2] = ib[2]; out_tlwh[3] = ib[3];
    *out_score = best;
    *out_class = bi;
    return true;
}

// ------------------------------------------------------------------------------------------------
// SSD-MobileNet: TFLite_Detection_PostProcess (third-party op, restated from its published algorithm,
// fast-NMS mode; PARITY UNPINNED -- see oracle/detect.py) followed by the reference's own
// post-processing (tools/ssd_mobilenet.py:100-150,59-98,198-213) and the box filter
// (deepdish.py:946-955).
// ------------------------------------------------------------------------------------------------
struct DDSsdParams {
    int na, ncls;              // anchors (1917), classes incl. background column 0 (91)
    int max_det;               // 10
    float score_thr, iou_thr;  // 1e-8, 0.6 (op attributes)
    float sy, sx, sh, sw;      // box coder scales 10, 10, 5, 5
    float conf_thr;            // ssd_mobilenet.py:100 confidence 0.5 (also score_threshold :207)
    double nms_iou;            // ssd_mobilenet.py:100 iou_threshold 0.5
    int img_w, img_h, frame_w, frame_h;
    double max_area;
};
#define DD_SSD_MAXDET 16

// The op's exp is DECLARED correctly rounded in f32: exp evaluated in f64 (<= 1 ulp there, on the device as in glibc)
// and rounded once to f32.  An f32 libm expf may differ from that in the last bit on either side; the oracle
// (oracle/detect.py) uses the same definition, which makes the decoded boxes bit-exact between the two.
#if defined(__CUDA_ARCH__)
DD_D float dd_expf(float x) { return (float)exp((double)x); }
#else
inline float dd_expf(float x) { return (float)exp((double)x); }
#endif

// DecodeCenterSizeBoxes for one anchor: raw (ty,tx,th,tw), anchor (yc,xc,h,w) -> (ymin,xmin,ymax,xmax) f32.
DD_HD void dd_ssd_decode_box(const float* raw, const float* an, const DDSsdParams& p, float* out) {
    const float yc = dd_addf(dd_mulf(dd_divf(raw[0], p.sy), an[2]), an[0]);
    const float xc = dd_addf(dd_mulf(dd_divf(raw[1], p.sx), an[3]), an[1]);
    const float hh = dd_mulf(dd_mulf(0.5f, dd_expf(dd_divf(raw[2], p.sh))), an[2]);
    const float hw = dd_mulf(dd_mulf(0.5f, dd_expf(dd_divf(raw[3], p.sw))), an[3]);
    out[0] = dd_subf(yc, hh); out[1] = dd_subf(xc, hw); out[2] = dd_addf(yc, hh); out[3] = dd_addf(xc, hw);
}

// ComputeIntersectionOverUnion (f32).
DD_HD float dd_ssd_iou(const float* a, const float* b) {
    const float aa = dd_mulf(dd_subf(a[2], a[0]), dd_subf(a[3], a[1]));
    const float ab = dd_mulf(dd_subf(b[2], b[0]), dd_subf(b[3], b[1]));
    if (aa <= 0.f || ab <= 0.f) return 0.f;
    const float ih = fmaxf(dd_subf(fminf(a[2], b[2]), fmaxf(a[0], b[0])), 0.f);
    const float iw = fmaxf(dd_subf(fminf(a[3], b[3]), fmaxf(a[1], b[1])), 0.f);
    const float inter = dd_mulf(ih, iw);
    return dd_divf(inter, dd_subf(dd_addf(aa, ab), inter));
}

// Everything after the op's greedy selection, serial (<= max_det boxes):
//   sel_box [n][4] (ymin,xmin,ymax,xmax normalised f32), sel_cls [n] (0-based, background removed),
//   sel_score [n] in descending score order.  class_to_label[c] = output label id or -1 (label unknown
//   or not wanted).  Writes <= n rows (tlwh integer-valued f64 after the box filter, score, label) in
//   the reference's output order; returns the count.
DD_HD int dd_ssd_post(const float* sel_box, const int* sel_cls, const float* sel_score, int n,
                      const DDSsdParams& p, const int* class_to_label, double* out_tlwh,
                      float* out_score, int* out_label) {
    double bx[DD_SSD_MAXDET][4];
    int cls[DD_SSD_MAXDET];
    float sc[DD_SSD_MAXDET];
    int m = 0;
    // NaN scrub (:111-116).  Reference quirk kept: np.where on the [n,4] box array yields (rows, cols) and
    // BOTH index lists are used to zero scores, so a NaN in column k also zeroes score[k].
    unsigned zero = 0;
    for (int i = 0; i < n; ++i)
        for (int k = 0; k < 4; ++k)
            if (sel_box[i * 4 + k] != sel_box[i * 4 + k]) zero |= (1u << i) | (1u << k);
    for (int i = 0; i < n; ++i) {                       // confidence filter (:119)
        float s = sel_score[i];
        if (((zero >> i) & 1u) || s != s) s = 0.f;
        if (!(s >= p.conf_thr)) continue;
        // reorder [1,0,3,2] * [w,h,w,h] -> f64 (xmin, ymin, xmax, ymax)  (:121-127)
        bx[m][0] = dd_mul((double)sel_box[i * 4 + 1], (double)p.img_w);
        bx[m][1] = dd_mul((double)sel_box[i * 4 + 0], (double)p.img_h);
        bx[m][2] = dd_mul((double)sel_box[i * 4 + 3], (double)p.img_w);
        bx[m][3] = dd_mul((double)sel_box[i * 4 + 2], (double)p.img_h);
        cls[m] = sel_cls[i];
        sc[m] = s;
        ++m;
    }
    // class iteration order = CPython set(labels) order (:61): emulate the small-int set
    short tabA[64], tabB[64];
    short *R = tabA, *Rt = tabB;
    int mask = 7, fill = 0;
    for (int i = 0; i < 8; ++i) R[i] = 0;
    for (int i = 0; i < m; ++i) {
        bool dup = false;
        for (int k = 0; k < i; ++k) dup = dup || cls[k] == cls[i];
        if (!dup) dd_set_add(R, Rt, mask, fill, cls[i]);
    }
    int n_out = 0;
    bool any_nan = false;
    double cand[DD_SSD_MAXDET][4];
    float cand_s[DD_SSD_MAXDET];
    int cand_l[DD_SSD_MAXDET];
    int nc = 0;
    for (int slot = 0; slot <= mask; ++slot) {
        if (!R[slot]) continue;
        const int c = R[slot] - 1;
        int idx[DD_SSD_MAXDET];
        int k = 0;
        for (int i = 0; i < m; ++i)
            if (cls[i] == c) idx[k++] = i;               // already in descending score order (stable)
        bool dead[DD_SSD_MAXDET];
        for (int i = 0; i < k; ++i) dead[i] = false;
        for (int a = 0; a < k; ++a) {                    // per-class greedy NMS, IoU with +1 px (:59-98)
            if (dead[a]) continue;
            const double* A = bx[idx[a]];
            const double wa = dd_sub(A[2], A[0]), ha = dd_sub(A[3], A[1]);
            const double area_a = dd_mul(wa, ha);
            for (int b = a + 1; b < k; ++b) {
                if (dead[b]) continue;
                const double* B = bx[idx[b]];
                const double wb = dd_sub(B[2], B[0]), hb = dd_sub(B[3], B[1]);
                const double xx1 = dd_max(A[0], B[0]), yy1 = dd_max(A[1], B[1]);
                const double xx2 = dd_min(dd_add(A[0], wa), dd_add(B[0], wb));
                const double yy2 = dd_min(dd_add(A[1], ha), dd_add(B[1], hb));
                const double w1 = dd_max(0.0, dd_add(dd_sub(xx2, xx1), 1.0));
                const double h1 = dd_max(0.0, dd_add(dd_sub(yy2, yy1), 1.0));
                const double inter = dd_mul(w1, h1);
                const double ovr = dd_div(inter, dd_sub(dd_add(area_a, dd_mul(wb, hb)), inter));
                if (!(ovr <= p.nms_iou)) dead[b] = true;
            }
            // label map (+1) / wanted filter / tlwh (:143-147, :207-212)
            const int lab = class_to_label[c];
            if (lab < 0 || !(sc[idx[a]] >= p.conf_thr)) continue;
            cand[nc][0] = A[0]; cand[nc][1] = A[1]; cand[nc][2] = wa; cand[nc][3] = ha;
            for (int q = 0; q < 4; ++q) any_nan = any_nan || (cand[nc][q] != cand[nc][q]);
            cand_s[nc] = sc[idx[a]];
            cand_l[nc] = lab;
            ++nc;
        }
    }
    if (p.frame_w <= 0) {                                // adapter mode: detect_image's own output
        for (int i = 0; i < nc; ++i) {
            for (int q = 0; q < 4; ++q) out_tlwh[i * 4 + q] = cand[i][q];
            out_score[i] = cand_s[i];
            out_label[i] = cand_l[i];
        }
        return nc;
    }
    if (any_nan) return 0;                               // deepdish.py:947-949
    for (int i = 0; i < nc; ++i) {                       // box filter (deepdish.py:950-955)
        int ib[4];
        if (!dd_box_clip(cand[i][0], cand[i][1], cand[i][2], cand[i][3], p.frame_w, p.frame_h, p.max_area, ib)) continue;
        out_tlwh[n_out * 4 + 0] = ib[0]; out_tlwh[n_out * 4 + 1] = ib[1];
        out_tlwh[n_out * 4 + 2] = ib[2]; out_tlwh[n_out * 4 + 3] = ib[3];
        out_score[n_out] = cand_s[i];
        out_label[n_out] = cand_l[i];
        ++n_out;
    }
    return n_out;
}

// ------------------------------------------------------------------------------------------------
// Keras YOLOv3 adapter (tools/yolo.py): decode_netout (:48-81), correct_yolo_boxes (:83-91), do_nms (:122-137),
// get_boxes (:140-153) and the tail of YOLO.detect_image (:207-237).  Quirks kept on purpose: every cell emits a box
// (the `objectness.all() <= obj_thresh` test only skips an objectness of exactly 0), y uses the FRACTIONAL row
// i / grid_w, a box with two labels above the threshold is returned twice (both times with its arg-max label), the
// returned boxes are transposed (x = box[1], y = box[0]) and come out in reversed get_boxes order.  Scalar arithmetic
// follows numpy 2 (Python ints / floats do not widen float32); exp is dd_expf (correctly rounded f32 by declaration).
// ------------------------------------------------------------------------------------------------
#define DD_Y3_MAX_ACTIVE 128      // boxes of one frame with a class score above the threshold (more -> DD_FLAG_DET_OVERFLOW)
#define DD_Y3_BAD_BOX 64          // flag: two zero-area boxes met in do_nms (ZeroDivisionError in the reference)

struct DDYolo3Params {
    int nc;                       // classes
    int g[3];                     // grid size of each output map (g x g cells, 3 boxes per cell)
    int anchors[3][6];            // tools/yolo.py:166
    float thr;                    // score_threshold (obj_thresh of decode_netout and get_boxes' thresh)
    double nms_thresh;            // 0.5 (:205)
    int image_w, image_h, net_w, net_h;
};

DD_HD float dd_sigmoid_f32(float x) { return dd_divf(1.0f, dd_addf(1.0f, dd_expf(-x))); }      // yolo.py:45-46

// box (map k, cell i, anchor b) of a frame: raw = its 5 + nc logits.  Integer box (xmin, ymin, xmax, ymax) after
// correct_yolo_boxes; returns the objectness sigmoid.
DD_HD float dd_yolo3_box(const float* raw, int k, int i, int b, const DDYolo3Params& p, int* box) {
    const int gw = p.g[k], gh = p.g[k];
    const int col = i % gw;
    const float rowf = (float)((double)i / (double)gw);                    // python float row (:59), narrowed at :67
    const float sx = dd_sigmoid_f32(raw[0]), sy = dd_sigmoid_f32(raw[1]);
    const float x = dd_divf(dd_addf((float)col, sx), (float)gw);
    const float y = dd_divf(dd_addf(rowf, sy), (float)gh);
    const float w = dd_divf(dd_mulf((float)p.anchors[k][2 * b], dd_expf(raw[2])), (float)p.net_w);
    const float h = dd_divf(dd_mulf((float)p.anchors[k][2 * b + 1], dd_expf(raw[3])), (float)p.net_h);
    const float hw = dd_divf(w, 2.0f), hh = dd_divf(h, 2.0f);
    box[0] = (int)dd_mulf(dd_subf(x, hw), (float)p.image_w);               // int() truncates toward zero (:88-91)
    box[1] = (int)dd_mulf(dd_subf(y, hh), (float)p.image_h);
    box[2] = (int)dd_mulf(dd_addf(x, hw), (float)p.image_w);
    box[3] = (int)dd_mulf(dd_addf(y, hh), (float)p.image_h);
    return dd_sigmoid_f32(raw[4]);
}

DD_HD int dd_y3_overlap(int a1, int a2, int b1, int b2) {                  // _interval_overlap (:93-107)
    if (b1 < a1) return b2 < a1 ? 0 : dd_imin(a2, b2) - a1;
    return a2 < b1 ? 0 : dd_imin(a2, b2) - b1;
}

// bbox_iou (:109-116) >= nms_thresh; *bad is set when the reference would divide by zero
DD_HD bool dd_y3_suppresses(const int* p, const int* q, double nms_thresh, int* bad) {
    const long long iw = dd_y3_overlap(p[0], p[2], q[0], q[2]), ih = dd_y3_overlap(p[1], p[3], q[1], q[3]);
    const long long inter = iw * ih;
    const long long uni = (long long)(p[2] - p[0]) * (p[3] - p[1]) + (long long)(q[2] - q[0]) * (q[3] - q[1]) - inter;
    if (uni == 0) { *bad = 1; return false; }
    return dd_div((double)inter, (double)uni) >= nms_thresh;
}

// do_nms for one class c over the n active boxes (in box order): cls [n][nc] thresholded scores, box [n][4].
// scratch: n ints.  Sort by descending score, stable (equal scores: lower box index first).
DD_HD void dd_y3_nms_class(int c, int n, int nc, float* cls, const int* box, double nms_thresh, int* order, int* bad) {
    int m = 0;
    for (int i = 0; i < n; ++i)
        if (cls[i * nc + c] != 0.f) {                                      // zero scores sort last and never suppress
            int j = m++;
            while (j > 0 && cls[order[j - 1] * nc + c] < cls[i * nc + c]) { order[j] = order[j - 1]; --j; }
            order[j] = i;
        }
    for (int a = 0; a < m; ++a) {
        const int p = order[a];
        if (cls[p * nc + c] == 0.f) continue;
        for (int e = a + 1; e < m; ++e) {
            const int q = order[e];
            if (dd_y3_suppresses(box + p * 4, box + q * 4, nms_thresh, bad)) cls[q * nc + c] = 0.f;
        }
        // boxes whose score for c is already zero stay zero whatever their IoU: nothing to do for them
    }
}

// get_boxes + the detect_image tail over the n active boxes (box order); returns the number of detections written
// (at most ncap; *overflow set beyond).  out_box [ncap][4] = x, y, w, h (ints, transposed like the reference).
DD_HD int dd_y3_emit(int n, int nc, const float* cls, const int* box, float thr, const unsigned char* wanted, int ncap,
                     double* out_box, float* out_score, int* out_label, int* overflow) {
    int k = 0;
    for (int p = n - 1; p >= 0; --p) {
        int lab = 0, above = 0;
        for (int c = 0; c < nc; ++c) {
            if (cls[p * nc + c] > cls[p * nc + lab]) lab = c;              // np.argmax: first maximum
            above += cls[p * nc + c] > thr ? 1 : 0;
        }
        const float score = cls[p * nc + lab];
        if (!wanted[lab] || score < thr) continue;
        int x = box[p * 4 + 1], y = box[p * 4 + 0];
        int w = box[p * 4 + 3] - box[p * 4 + 1], h = box[p * 4 + 2] - box[p * 4 + 0];
        if (x < 0) { w += x; x = 0; }
        if (y < 0) { h += y; y = 0; }
        for (int rep = 0; rep < above; ++rep) {                            // once per label above the threshold (:145-152)
            if (k >= ncap) { *overflow = 1; return k; }
            out_box[k * 4 + 0] = x; out_box[k * 4 + 1] = y; out_box[k * 4 + 2] = w; out_box[k * 4 + 3] = h;
            out_score[k] = score; out_label[k] = lab;
            ++k;
        }
    }
    return k;
}
