// dd_hostemu.cpp -- TEST SCAFFOLDING ONLY (built by tests/hostemu/build.py, loaded only by tests/).
//
// Compiles the group-generic kernel bodies of deepdish_b200/csrc with HostG (one lane, trivial
// collectives) so that the serial logic of the CUDA path -- scipy-exact LSAP, CPython set order,
// cascade / lifecycle bookkeeping, count-line -- can be exercised against the oracle on a machine
// without a GPU.  It shares no code with oracle/, is never linked into libdeepdish_b200.so and is
// never imported by the deepdish_b200 package: the product path has no CPU fallback.
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../deepdish_b200/csrc/dd_tracker_bodies.cuh"
#include "../../deepdish_b200/csrc/dd_detect_bodies.cuh"

extern "C" {

int ddh_tracker_layout_query(const dd_tracker_config* cfg, dd_tracker_layout* out) {
    return dd_layout_compute(cfg, out);
}

// shared memory of the matching step for T slots and D detections (what the layout check compares with the limit)
long long ddh_match_smem_bytes(int T, int D) { return (long long)dd_match_smem_bytes(T, D, dd_set_table_slots(T)); }

int ddh_tracker_init(void* state, const dd_tracker_config* cfg) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    dd_tracker_layout L;
    dd_layout_compute(cfg, &L);
    memset(state, 0, L.total_bytes);
    for (int s = 0; s < V.S; ++s) V.next_id[s] = 1;
    const int n_pages = cfg->n_segs * cfg->seg_pages;
    for (int i = 0; i < n_pages; ++i) V.free_stack[i] = n_pages - 1 - i;
    V.pool_ctl[0] = n_pages; V.pool_ctl[1] = n_pages;
    return DD_OK;
}

int ddh_tracker_predict(void* state, const dd_tracker_config* cfg) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    HostG g;
    for (int s = 0; s < V.S; ++s)
        for (int t = 0; t < V.T; ++t) dd_predict_track(g, V, s, t);
    return DD_OK;
}

int ddh_tracker_update(void* state, const dd_tracker_config* cfg, const double* det_tlwh,
                       const float* det_conf, const int32_t* det_label, const float* det_feat,
                       const int32_t* det_count, int32_t* out_det_track_id) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    HostG g;
    for (int s = 0; s < V.S; ++s)
        for (int d = 0; d < V.D; ++d) dd_prep_det(g, V, s, d, det_tlwh, det_feat, det_count);
    for (int s = 0; s < V.S; ++s)
        for (int t = 0; t < V.T; ++t) dd_gate_track(g, V, s, t, det_count);
    for (int s = 0; s < V.S; ++s)
        for (int t = 0; t < V.T; ++t) { DDDirectPass<HostG> pass; dd_cosine_track(g, V, s, t, det_count, pass); }
    std::vector<char> smem(dd_match_smem_bytes(V.T, V.D, V.tab_cap) + 16);
    for (int s = 0; s < V.S; ++s)
        dd_match_stream(g, V, s, det_tlwh, det_count, out_det_track_id, smem.data());
    double scratch[64];
    for (int s = 0; s < V.S; ++s)
        for (int d = 0; d < V.D; ++d) dd_apply_det(g, V, s, d, det_conf, det_label, scratch);
    return DD_OK;
}

// metric.samples of one slot, oldest row first (what dd_tracker_gallery_read returns on the device).
int ddh_gallery_read(void* state, const dd_tracker_config* cfg, int s, int slot_in_stream, float* out, int max_rows) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    const size_t slot = (size_t)s * V.T + slot_in_stream;
    const int len = V.gal_len[slot], pos = V.gal_pos[slot];
    const int n = len < max_rows ? len : max_rows;
    for (int i = 0; i < n; ++i) {
        int row = i;
        if (V.B > 0) { row = pos - len + i; if (row < 0) row += V.B; }
        memcpy(out + (size_t)i * DD_FEAT_DIM, dd_gallery_row(V, V.ptab + slot * V.PT, row), DD_FEAT_DIM * 4);
    }
    return n;
}

// The count-line step as dd_tick_tail issues it: a new crossing list when the records are on, then the step of every
// stream.  lines f64 [S,L,4].
static void ddh_countline_step(const DDView& V, const double* lines) {
    HostG g;
    if (V.ev) V.ev[0] = 0;
    for (int s = 0; s < V.S; ++s) {
        const double* l = lines + (size_t)s * V.n_lines * 4;
        if (V.ev)
            dd_countline<HostG, true>(g, V, s, l);
        else
            dd_countline<HostG, false>(g, V, s, l);
    }
}

int ddh_tracker_countline(void* state, const dd_tracker_config* cfg, const double* lines) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    ddh_countline_step(V, lines);
    return DD_OK;
}

// One fused tick as the engine runs it (k_prep, k_gate<true>, gallery, k_match, k_apply, k_countline), with frame
// presence.  present u8 [S] (NULL = every stream present); lines f64 [S,L,4].
int ddh_tracker_tick(void* state, const dd_tracker_config* cfg, const double* det_tlwh, const float* det_conf,
                     const int32_t* det_label, const float* det_feat, const int32_t* det_count, const uint8_t* present,
                     const double* lines, int32_t* out_det_track_id) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    HostG g;
    for (int s = 0; s < V.S; ++s)
        for (int d = 0; d < V.D; ++d) dd_prep_det(g, V, s, d, det_tlwh, det_feat, det_count, present);
    for (int s = 0; s < V.S; ++s)
        for (int t = 0; t < V.T; ++t) {
            dd_tick_predict_track(g, V, s, t);
            dd_gate_track(g, V, s, t, det_count);
        }
    for (int s = 0; s < V.S; ++s)
        for (int t = 0; t < V.T; ++t) { DDDirectPass<HostG> pass; dd_cosine_track(g, V, s, t, det_count, pass); }
    std::vector<char> smem(dd_match_smem_bytes(V.T, V.D, V.tab_cap) + 16);
    for (int s = 0; s < V.S; ++s)
        dd_match_stream(g, V, s, det_tlwh, det_count, out_det_track_id, smem.data());
    double scratch[64];
    for (int s = 0; s < V.S; ++s)
        for (int d = 0; d < V.D; ++d) dd_apply_det(g, V, s, d, det_conf, det_label, scratch);
    ddh_countline_step(V, lines);
    return DD_OK;
}

// scipy-exact LSAP on one dense f64 matrix (the device code path of dd_lsap).
int ddh_lsap(const double* cost, int nr, int nc, int32_t* out_col4row) {
    HostG g;
    const int n = nr > nc ? nr : nc;
    std::vector<char> mem(dd_lsap_scratch_bytes(n) + 16);
    DDLsapScratch s;
    dd_lsap_carve(mem.data(), n, s);
    struct Dense { const double* c; int nc; double operator()(int i, int j) const { return c[i * nc + j]; } };
    struct DenseT { const double* c; int nc; double operator()(int i, int j) const { return c[j * nc + i]; } };
    int rc;
    if (nc < nr) {
        DenseT f{cost, nc};
        rc = dd_lsap_solve(g, nc, nr, f, s);
        for (int r = 0; r < nr; ++r) out_col4row[r] = s.row4col[r];
    } else {
        Dense f{cost, nc};
        rc = dd_lsap_solve(g, nr, nc, f, s);
        for (int r = 0; r < nr; ++r) out_col4row[r] = s.col4row[r];
    }
    return rc;
}

int ddh_set_difference_order(const int32_t* a, int na, const int32_t* m, int nm, int32_t* out) {
    int maxv = 0;
    for (int i = 0; i < na; ++i) if (a[i] > maxv) maxv = a[i];
    for (int i = 0; i < nm; ++i) if (m[i] > maxv) maxv = m[i];
    std::vector<unsigned char> flag(maxv + 1, 0);
    for (int i = 0; i < nm; ++i) flag[m[i]] = 1;
    std::vector<short> av(na), o(na + 1);
    for (int i = 0; i < na; ++i) av[i] = (short)a[i];
    const int cap = dd_set_table_slots(na > 0 ? na : 1);
    std::vector<short> A(cap), B(cap), C(cap);
    bool contig = true;
    for (int i = 0; i < na; ++i) contig = contig && a[i] == i;
    int n;
    if (contig) {
        std::vector<short> surv;
        for (int i = 0; i < na; ++i) if (!flag[i]) surv.push_back((short)i);
        if ((na >> 2) > nm) { n = (int)surv.size(); for (int i = 0; i < n; ++i) o[i] = surv[i]; }
        else n = dd_set_order_from_survivors(surv.data(), (int)surv.size(), o.data(), A.data(), B.data());
    } else {
        n = dd_set_difference_order_serial(av.data(), na, flag.data(), nm, o.data(), A.data(), B.data(),
                                           C.data(), cap);
    }
    for (int i = 0; i < n; ++i) out[i] = o[i];
    return n;
}

int ddh_intersection(const double* seg, int n, int32_t* out) {
    for (int i = 0; i < n; ++i) {
        const double* p = seg + (size_t)i * 8;
        out[i] = dd_segments_intersect(p[0], p[1], p[2], p[3], p[4], p[5], p[6], p[7]) ? 1 : 0;
    }
    return 0;
}

// SSD: the post-processing of the op's outputs (device function dd_ssd_post) on host arrays.
int ddh_ssd_post(const float* sel_box, const int32_t* sel_cls, const float* sel_score, int n,
                 const int32_t* class_to_label, float conf_thr, double nms_iou, int img_w, int img_h,
                 int frame_w, int frame_h, double* out_tlwh, float* out_score, int32_t* out_label) {
    DDSsdParams P;
    P.na = 0; P.ncls = 0; P.max_det = 10; P.score_thr = 1e-8f; P.iou_thr = 0.6f;
    P.sy = 10.f; P.sx = 10.f; P.sh = 5.f; P.sw = 5.f;
    P.conf_thr = conf_thr; P.nms_iou = nms_iou;
    P.img_w = img_w; P.img_h = img_h; P.frame_w = frame_w; P.frame_h = frame_h;
    P.max_area = 0.9 * frame_w * frame_h;
    return dd_ssd_post(sel_box, sel_cls, sel_score, n, P, class_to_label, out_tlwh, out_score, out_label);
}

// The box filter device function (dd_box_clip + the frame-level NaN rule) on one frame of host boxes.
int ddh_box_filter(const double* boxes, int n, int frame_w, int frame_h, double* out_tlwh, int32_t* out_index) {
    for (int e = 0; e < n * 4; ++e) if (boxes[e] != boxes[e]) return 0;
    int nk = 0;
    for (int i = 0; i < n; ++i) {
        int ib[4];
        if (!dd_box_clip(boxes[i * 4], boxes[i * 4 + 1], boxes[i * 4 + 2], boxes[i * 4 + 3], frame_w, frame_h,
                         0.9 * frame_w * frame_h, ib)) continue;
        for (int q = 0; q < 4; ++q) out_tlwh[nk * 4 + q] = ib[q];
        out_index[nk++] = i;
    }
    return nk;
}

// Keras YOLOv3 post-processing device functions on one frame of host maps (same helpers as k_yolo3_post, serial).
int ddh_yolo3(const float* m0, const float* m1, const float* m2, const int32_t* grids, const int32_t* anchors18, int nc,
              const uint8_t* wanted, float thr, double nms_thresh, int image_w, int image_h, int net_w, int net_h, int ncap,
              double* out_box, float* out_score, int32_t* out_label, int32_t* out_flags) {
    DDYolo3Params P;
    P.nc = nc; P.thr = thr; P.nms_thresh = nms_thresh;
    P.image_w = image_w; P.image_h = image_h; P.net_w = net_w; P.net_h = net_h;
    for (int k = 0; k < 3; ++k) { P.g[k] = grids[k]; for (int a = 0; a < 6; ++a) P.anchors[k][a] = anchors18[k * 6 + a]; }
    const float* maps[3] = {m0, m1, m2};
    const int rw = 5 + nc;
    std::vector<int> box;
    std::vector<float> cls;
    for (int k = 0; k < 3; ++k)
        for (int e = 0; e < P.g[k] * P.g[k] * 3; ++e) {
            const float* raw = maps[k] + (size_t)e * rw;
            if (!(dd_sigmoid_f32(raw[4]) > thr)) continue;
            int b4[4];
            dd_yolo3_box(raw, k, e / 3, e % 3, P, b4);
            box.insert(box.end(), b4, b4 + 4);
            for (int c = 0; c < nc; ++c) {
                const float v = dd_mulf(dd_sigmoid_f32(raw[4]), dd_sigmoid_f32(raw[5 + c]));
                cls.push_back(v > thr ? v : 0.f);
            }
        }
    const int n = (int)box.size() / 4;
    std::vector<int> order(n + 1);
    int bad = 0, over = 0;
    for (int c = 0; c < nc; ++c) dd_y3_nms_class(c, n, nc, cls.data(), box.data(), nms_thresh, order.data(), &bad);
    const int k = dd_y3_emit(n, nc, cls.data(), box.data(), thr, wanted, ncap, out_box, out_score, out_label, &over);
    *out_flags = (over ? DD_FLAG_DET_OVERFLOW : 0) | (bad ? DD_Y3_BAD_BOX : 0);
    return k;
}

// NMS device body on host arrays (one frame).
int ddh_nms(const double* boxes, const float* scores, int n, double max_overlap, int32_t* keep) {
    HostG g;
    std::vector<char> smem(dd_nms_smem_bytes(n > 0 ? n : 1) + 64);
    int nk = 0;
    dd_nms_frame(g, boxes, scores, n, n > 0 ? n : 1, max_overlap, keep, &nk, smem.data());
    return nk;
}

// YOLO row decode + box filter device body on host arrays: head [na, 5+nc] f32.
int ddh_yolo_rows(const float* head, int na, int nc, const uint8_t* wanted, float thr, int img_w, int img_h,
                  int frame_w, int frame_h, double* out_tlwh, float* out_score, int32_t* out_class,
                  int32_t* out_anchor, int32_t* out_nan) {
    DDYoloParams P;
    P.nc = nc; P.thr = thr; P.img_w = (float)img_w; P.img_h = (float)img_h;
    P.frame_w = frame_w; P.frame_h = frame_h; P.max_area = 0.9 * frame_w * frame_h;
    struct Row { const float* p; float operator()(int k) const { return p[k]; } };
    int n = 0;
    *out_nan = 0;
    for (int a = 0; a < na; ++a) {
        Row row{head + (size_t)a * (5 + nc)};
        bool isnan = false;
        double tl[4]; float sc; int cl;
        const bool ok = dd_yolo_row(row, P, wanted, tl, &sc, &cl, &isnan);
        if (isnan) *out_nan = 1;
        if (!ok) continue;
        for (int q = 0; q < 4; ++q) out_tlwh[n * 4 + q] = tl[q];
        out_score[n] = sc; out_class[n] = cl; out_anchor[n] = a;
        ++n;
    }
    return n;
}

}  // extern "C"
