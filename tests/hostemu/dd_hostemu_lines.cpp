// dd_hostemu_lines.cpp -- TEST SCAFFOLDING ONLY (built by tests/hostemu/lines.py, loaded only by tests/).
//
// The fused tick of dd_hostemu_tick.cpp with several count lines per stream (config.n_lines > 1): the count-line step
// is the body k_countline_lines runs, compiled with the one-lane HostG, with the crossing records when
// config.event_cap > 0 (behind the same reset of the list's header that dd_tick_tail makes).  Never linked into
// libdeepdish_b200.so.
#include <vector>
#include "../../deepdish_b200/csrc/dd_tracker_bodies.cuh"

extern "C" {

// lines f64 [S,L,4]; present u8 [S] (NULL = every stream present)
int ddh_tracker_tick_lines(void* state, const dd_tracker_config* cfg, const double* det_tlwh, const float* det_conf,
                           const int32_t* det_label, const float* det_feat, const int32_t* det_count,
                           const uint8_t* present, const double* lines, int32_t* out_det_track_id) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    if (V.n_lines < 2) return DD_ERR_INVALID;
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
    if (V.ev) V.ev[0] = 0;
    for (int s = 0; s < V.S; ++s) {
        const double* l = lines + (size_t)s * V.n_lines * 4;
        if (V.ev)
            dd_countline_lines<HostG, true>(g, V, s, l);
        else
            dd_countline_lines<HostG, false>(g, V, s, l);
    }
    return DD_OK;
}

}  // extern "C"
