// dd_hostemu_tick.cpp -- TEST SCAFFOLDING ONLY (built by tests/hostemu/tick.py, loaded only by tests/).
//
// One fused tick of the batched tracker as the engine runs it (k_prep, k_gate<true>, gallery, k_match, k_apply,
// k_countline), with frame presence, compiled from the same group-generic kernel bodies with the one-lane HostG.  It
// works on the blob and page pool of a tests/hostemu/driver.py HostEmuTracker.  Never linked into libdeepdish_b200.so.
#include <vector>
#include "../../deepdish_b200/csrc/dd_tracker_bodies.cuh"

extern "C" {

// present u8 [S] (NULL = every stream present)
int ddh_tracker_tick(void* state, const dd_tracker_config* cfg, const double* det_tlwh, const float* det_conf,
                     const int32_t* det_label, const float* det_feat, const int32_t* det_count, const uint8_t* present,
                     const double* line, int line_per_stream, int32_t* out_det_track_id) {
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
    for (int s = 0; s < V.S; ++s) dd_countline(g, V, s, line + (line_per_stream ? (size_t)s * 4 : 0));
    return DD_OK;
}

}  // extern "C"
