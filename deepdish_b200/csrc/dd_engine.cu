// dd_engine.cu -- native host-side executor of the batched tick: per stream chunk ONE captured CUDA graph per tick
// (prep -> gate -> gallery -> match -> apply -> count-line -> count reduce), launched on the chunk's own stream, plus
// the event plumbing between chunks, the count summation on an auxiliary stream, the double-buffered upload of ragged
// host batches on per-chunk copy streams and the asynchronous polling of the page-pool counters.
//
// Why native: the reference's per-frame driver loop is Python (deepdish.py:1245-1262); batched over 1024 streams the
// tick is 0.5 ms of device time, and 14 launches + a dozen event / stream calls per tick through ctypes cost as much on
// the host.  Here a tick costs the host one C call: per chunk one plain kernel launch (detection prep, which carries the tick's inputs) + the
// captured graph(s) of the rest.
// A graph's kernel parameters are frozen at capture, so the per-tick inputs (detection arrays, the ragged blob and
// its section offsets, the output slots) travel through the blob's tick_args words (DDTickArgs, dd_view.h).
#include <cuda_runtime.h>
#include <new>
#include <vector>
#include "dd_view.h"

// dd_tracker.cu
int dd_capture_tick(void* state, const dd_tracker_config* cfg, int ragged, int reduce, int parts, const double* line,
                    int line_per_stream, cudaStream_t st);
int dd_tick_prepare_host(void* state, const dd_tracker_config* cfg);
int dd_launch_prep_publishing(void* state, const dd_tracker_config* cfg, const DDTickArgs* A, cudaStream_t st);
enum { PART_PREP = 1, PART_GATE = 2, PART_GALLERY = 4, PART_POST = 8, PART_TAIL = 16 };      // DD_PART_* of dd_tracker.cu
size_t dd_tick_args_offset(const dd_tracker_config* cfg);

#define DD_CU(x) do { if ((x) != cudaSuccess) return DD_ERR_CUDA; } while (0)

#include <chrono>
extern "C" int dd_engine_destroy(void* engine);

// total[e] = sum over chunks of partial[c][e]
__global__ void k_sum_partials(const long long* __restrict__ partial, int n_chunks, int n, long long* __restrict__ total) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    long long acc = 0;
    for (int c = 0; c < n_chunks; ++c) acc += partial[(size_t)c * n + e];
    total[e] = acc;
}

namespace {

struct Chunk {
    void* state = nullptr;
    dd_tracker_config cfg;
    int lo = 0, n = 0;
    size_t events_off = 0;       // byte offset of the blob's `events` section (crossing records)
    cudaStream_t st = nullptr, copy_st = nullptr, copy_st2 = nullptr, d2h_st = nullptr;
    cudaEvent_t done = nullptr, copied = nullptr, copied2 = nullptr, unpacked[4] = {nullptr, nullptr, nullptr, nullptr}, gal_done = nullptr;
    cudaEvent_t tick_end = nullptr, d2h_done = nullptr;      // the det -> track ids leave on their own stream
    bool d2h_valid = false;
    bool unpacked_valid[4] = {false, false, false, false};
    // captured pieces of a tick, [ragged][reduce][piece]: 0 = everything (or, with gallery turns, the kernels before the
    // gallery stream), 1 = the gallery stream, 2 = the kernels behind it
    cudaGraphExec_t graph[2][2][3] = {};
    // host path (dd_engine_bind_host): double-buffered device blob + the small padded arrays the tick fills
    unsigned char* dev_blob[4] = {nullptr, nullptr, nullptr, nullptr};
    int n_blob = 0;              // upload buffers in rotation (2 .. 4)
    size_t blob_cap = 0;
    double* s_tlwh = nullptr;
    float* s_conf = nullptr;
    int *s_label = nullptr, *s_count = nullptr;
    // pool polling: two pinned copies of pool_ctl[0..3], alternating
    int* poll_host = nullptr;
    cudaEvent_t poll_ev[2] = {nullptr, nullptr};
    long long poll_tick[2] = {-1, -1};
    int poll_turn = 0;
};

struct Engine {
    int P = 0, D = 0, C4 = 0, line_per_stream = 0, poll_every = 0;
    int n_lines = 1;                 // count lines per stream: line is [L,4] or [S,L,4], C4 = L * C * 4
    bool turns = false;              // chunks take turns on the gallery stream (see dd_engine_create)
    bool graphs = true;              // replay captured graphs (dd_engine_set_graphs(0): launch the tick's kernels plainly)
    cudaEvent_t last_gal = nullptr;  // end of the most recently enqueued gallery stream
    std::vector<Chunk> ch;
    cudaStream_t aux = nullptr, cap = nullptr;
    cudaEvent_t fork_ev = nullptr, sum_done[2] = {nullptr, nullptr};
    bool sum_valid[2] = {false, false};
    int last_sum = -1;
    const double* line = nullptr;
    long long *partial = nullptr, *total = nullptr;
    int* ids = nullptr;
    long long tick = 0;
    long long launches = 0;          // kernels launched: prep kernels + graph nodes + count summations (bench.py gpu_launches)
    double blocked_ms = 0.0;         // host time spent waiting on the run-ahead throttle (pool polls)
};

// cudaEventSynchronize that accounts the time the host was blocked
cudaError_t blocked_sync(Engine& E, cudaEvent_t ev) {
    if (cudaEventQuery(ev) == cudaSuccess) return cudaSuccess;
    cudaGetLastError();
    const auto t0 = std::chrono::steady_clock::now();
    const cudaError_t e = cudaEventSynchronize(ev);
    E.blocked_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return e;
}

void drop_graphs(Chunk& c) {
    for (int a = 0; a < 2; ++a)
        for (int b = 0; b < 2; ++b)
            for (int k = 0; k < 3; ++k)
                if (c.graph[a][b][k]) { cudaGraphExecDestroy(c.graph[a][b][k]); c.graph[a][b][k] = nullptr; }
}

int capture_piece(Engine& E, Chunk& c, int ragged, int reduce, int parts, cudaGraphExec_t* out) {
    const double* line = E.line + (E.line_per_stream ? (size_t)c.lo * E.n_lines * 4 : 0);
    DD_CU(cudaStreamBeginCapture(E.cap, cudaStreamCaptureModeRelaxed));
    const int rc = dd_capture_tick(c.state, &c.cfg, ragged, reduce, parts, line, E.line_per_stream, E.cap);
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(E.cap, &g);
    if (rc != DD_OK || e != cudaSuccess || !g) {
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        return rc != DD_OK ? rc : DD_ERR_CUDA;
    }
    cudaGraphExec_t x = nullptr;
    const cudaError_t e2 = cudaGraphInstantiate(&x, g, 0);
    cudaGraphDestroy(g);
    if (e2 != cudaSuccess) return DD_ERR_CUDA;
    *out = x;
    return DD_OK;
}

int ensure_graphs(Engine& E, Chunk& c, int ragged, int reduce) {
    cudaGraphExec_t* g = c.graph[ragged][reduce];
    if (g[0]) return DD_OK;
    static bool carve_set[64] = {};      // per device; see dd_tick_prepare: every kernel of the tick asks for the maximum carve-out
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64 && !carve_set[dev]) {
        cudaFuncSetAttribute(k_sum_partials, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        carve_set[dev] = true;
    }
    int rc = dd_tick_prepare_host(c.state, &c.cfg);        // function attributes: outside the capture
    if (rc != DD_OK) return rc;
    // the detection-prep kernel runs in front of the graphs (launch_tick): it carries the tick's arguments by value
    if (!E.turns) return capture_piece(E, c, ragged, reduce, PART_GATE | PART_GALLERY | PART_POST | PART_TAIL, &g[0]);
    rc = capture_piece(E, c, ragged, reduce, PART_GALLERY, &g[1]);
    if (rc == DD_OK) rc = capture_piece(E, c, ragged, reduce, PART_POST | PART_TAIL, &g[2]);
    if (rc == DD_OK) rc = capture_piece(E, c, ragged, reduce, PART_GATE, &g[0]);
    if (rc != DD_OK)                     // all pieces or none: g[0] is what marks the set as captured
        for (int k = 0; k < 3; ++k)
            if (g[k]) { cudaGraphExecDestroy(g[k]); g[k] = nullptr; }
    return rc;
}

// consumed: (ragged ticks) recorded right behind the detection-prep kernel, the only reader of the uploaded blob
int launch_tick(Engine& E, Chunk& c, const DDTickArgs& A, int ragged, int reduce, cudaStream_t st,
                cudaEvent_t consumed = nullptr) {
    int rc = E.graphs ? ensure_graphs(E, c, ragged, reduce) : dd_tick_prepare_host(c.state, &c.cfg);
    if (rc != DD_OK) return rc;
    cudaGraphExec_t* g = c.graph[ragged][reduce];
    const double* line = E.line + (E.line_per_stream ? (size_t)c.lo * E.n_lines * 4 : 0);
    // one piece of the tick behind the prep kernel: its captured graph, or the same kernels launched plainly (they read
    // the tick's inputs through tick_args either way)
    auto piece = [&](int k, int parts) -> int {
        if (E.graphs) return cudaGraphLaunch(g[k], st) == cudaSuccess ? DD_OK : DD_ERR_CUDA;
        return dd_capture_tick(c.state, &c.cfg, ragged, reduce, parts, line, E.line_per_stream, st);
    };
    if (c.d2h_valid) {                       // the previous tick's ids must have left before this tick's matching rewrites them
        DD_CU(cudaStreamWaitEvent(st, c.d2h_done, 0));
        c.d2h_valid = false;
    }
    // the first kernel of the tick is launched plainly with the tick's arguments by value; it publishes them into the
    // blob's tick_args words, from which the captured kernels behind it read (a graph's parameters are frozen)
    rc = dd_launch_prep_publishing(c.state, &c.cfg, &A, st);
    if (rc != DD_OK) return rc;
    if (ragged && consumed) DD_CU(cudaEventRecord(consumed, st));
    rc = piece(0, E.turns ? PART_GATE : PART_GATE | PART_GALLERY | PART_POST | PART_TAIL);
    if (rc != DD_OK) return rc;
    if (E.turns) {
        // the gallery stream is the HBM-bound kernel: two of them side by side gain nothing, and chunks that drift into
        // phase run their gallery streams AND their latency-bound kernels at the same time.  So every gallery stream
        // waits for the previously enqueued one (of another chunk): chunks stay in anti-phase, the matching of one runs
        // under the gallery stream of the other.
        if (E.last_gal && E.last_gal != c.gal_done) DD_CU(cudaStreamWaitEvent(st, E.last_gal, 0));
        rc = piece(1, PART_GALLERY);
        if (rc != DD_OK) return rc;
        DD_CU(cudaEventRecord(c.gal_done, st));
        E.last_gal = c.gal_done;
        rc = piece(2, PART_POST | PART_TAIL);
        if (rc != DD_OK) return rc;
    }
    E.launches += 7 + (reduce ? 1 : 0);      // the tick's 7 (8) kernels
    if (E.poll_every > 0 && E.tick % E.poll_every == 0) {
        // the slot written two polls ago is reused: its copy has long completed unless the host runs far ahead
        const int k = c.poll_turn;
        if (c.poll_tick[k] >= 0) DD_CU(blocked_sync(E, c.poll_ev[k]));
        dd_tracker_layout L;
        dd_layout_compute(&c.cfg, &L);
        DD_CU(cudaMemcpyAsync(c.poll_host + 4 * k, (char*)c.state + L.pool_ctl, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
        DD_CU(cudaEventRecord(c.poll_ev[k], st));
        c.poll_tick[k] = E.tick;
        c.poll_turn ^= 1;
    }
    return DD_OK;
}

int sum_partials(Engine& E, int par, cudaStream_t cur) {
    const long long* src = E.partial + (size_t)par * E.P * E.C4;
    if (E.P == 1) {
        k_sum_partials<<<(E.C4 + 127) / 128, 128, 0, cur>>>(src, 1, E.C4, E.total);
        DD_CU(cudaGetLastError());
        ++E.launches;
        return DD_OK;
    }
    // on the auxiliary stream, NOT the caller's: the caller's stream must not wait for every chunk each tick, or the
    // next tick's fork event would serialise the chunks tick by tick
    for (auto& c : E.ch) DD_CU(cudaStreamWaitEvent(E.aux, c.done, 0));
    k_sum_partials<<<(E.C4 + 127) / 128, 128, 0, E.aux>>>(src, E.P, E.C4, E.total);
    DD_CU(cudaGetLastError());
    DD_CU(cudaEventRecord(E.sum_done[par], E.aux));
    ++E.launches;
    E.sum_valid[par] = true;
    E.last_sum = par;
    return DD_OK;
}

}  // namespace

extern "C" {

int dd_engine_create(int32_t n_chunks, void* const* host_states, const dd_tracker_config* const* host_cfgs,
                     const int32_t* host_first_stream, void* const* host_streams, void* aux_stream, const double* line,
                     int32_t line_per_stream, int64_t* partial_counts, int64_t* total_counts, int32_t* det_track_id,
                     int32_t poll_every, int32_t gallery_turns, void** host_out_engine) {
    if (n_chunks <= 0 || !host_states || !host_cfgs || !host_first_stream || !line || !partial_counts || !total_counts ||
        !det_track_id || !host_out_engine)
        return DD_ERR_INVALID;
    if (n_chunks > 1 && (!host_streams || !aux_stream)) return DD_ERR_INVALID;
    Engine* E = new (std::nothrow) Engine();
    if (!E) return DD_ERR_INVALID;
    E->P = n_chunks;
    E->line = line;
    E->line_per_stream = line_per_stream;
    E->partial = (long long*)partial_counts;
    E->total = (long long*)total_counts;
    E->ids = det_track_id;
    E->aux = (cudaStream_t)aux_stream;
    E->poll_every = poll_every;
    E->turns = gallery_turns != 0 && n_chunks > 1;
    E->ch.resize(n_chunks);
    bool ok = cudaStreamCreateWithFlags(&E->cap, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&E->fork_ev, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&E->sum_done[0], cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&E->sum_done[1], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok && i < n_chunks; ++i) {
        Chunk& c = E->ch[i];
        dd_tracker_layout L;
        if (!host_states[i] || !host_cfgs[i] || dd_layout_compute(host_cfgs[i], &L) != DD_OK) { ok = false; break; }
        c.state = host_states[i];
        c.cfg = *host_cfgs[i];
        c.lo = host_first_stream[i];
        c.n = c.cfg.n_streams;
        c.events_off = L.events;
        c.st = n_chunks > 1 ? (cudaStream_t)host_streams[i] : nullptr;
        if (i == 0) { E->D = c.cfg.max_dets; E->n_lines = dd_n_lines(&c.cfg); E->C4 = E->n_lines * c.cfg.n_labels * 4; }
        ok = c.cfg.max_dets == E->D && dd_n_lines(&c.cfg) == E->n_lines && E->n_lines * c.cfg.n_labels * 4 == E->C4 &&
             cudaEventCreateWithFlags(&c.done, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.copied, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.copied2, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.tick_end, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.d2h_done, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.gal_done, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.unpacked[0], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.unpacked[1], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.unpacked[2], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.unpacked[3], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.poll_ev[0], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c.poll_ev[1], cudaEventDisableTiming) == cudaSuccess &&
             cudaHostAlloc((void**)&c.poll_host, 8 * sizeof(int), cudaHostAllocDefault) == cudaSuccess;
    }
    if (!ok) {
        cudaGetLastError();
        dd_engine_destroy(E);
        *host_out_engine = nullptr;
        return DD_ERR_CUDA;
    }
    *host_out_engine = E;
    return DD_OK;
}

int dd_engine_destroy(void* engine) {
    Engine* E = (Engine*)engine;
    if (!E) return DD_ERR_INVALID;
    for (auto& c : E->ch) {
        drop_graphs(c);
        if (c.copy_st) cudaStreamDestroy(c.copy_st);
        if (c.copy_st2) cudaStreamDestroy(c.copy_st2);
        if (c.d2h_st) cudaStreamDestroy(c.d2h_st);
        for (cudaEvent_t e : {c.done, c.copied, c.copied2, c.gal_done, c.tick_end, c.d2h_done, c.unpacked[0], c.unpacked[1], c.unpacked[2], c.unpacked[3], c.poll_ev[0], c.poll_ev[1]})
            if (e) cudaEventDestroy(e);
        if (c.poll_host) cudaFreeHost(c.poll_host);
    }
    for (cudaEvent_t e : {E->fork_ev, E->sum_done[0], E->sum_done[1]})
        if (e) cudaEventDestroy(e);
    if (E->cap) cudaStreamDestroy(E->cap);
    delete E;
    return DD_OK;
}

int dd_engine_set_graphs(void* engine, int32_t use_graphs) {
    Engine* E = (Engine*)engine;
    if (!E) return DD_ERR_INVALID;
    E->graphs = use_graphs != 0;
    return DD_OK;
}

int dd_engine_rebind(void* engine, int32_t chunk, void* state, const dd_tracker_config* host_cfg) {
    Engine* E = (Engine*)engine;
    if (!E || chunk < 0 || chunk >= E->P || !state || !host_cfg) return DD_ERR_INVALID;
    Chunk& c = E->ch[chunk];
    drop_graphs(c);                  // the DDView frozen in the captured kernels is stale
    dd_tracker_layout L;
    c.state = state;
    c.cfg = *host_cfg;
    c.events_off = dd_layout_compute(host_cfg, &L) == DD_OK ? L.events : 0;     // (an invalid config fails at the next tick)
    c.poll_tick[0] = c.poll_tick[1] = -1;
    return DD_OK;
}

int dd_engine_bind_host(void* engine, int32_t chunk, void* const* host_dev_blobs, int32_t n_blobs, uint64_t blob_capacity,
                        double* det_tlwh, float* det_conf, int32_t* det_label, int32_t* det_count) {
    Engine* E = (Engine*)engine;
    if (!E || chunk < 0 || chunk >= E->P || !host_dev_blobs || n_blobs < 2 || n_blobs > 4 || !det_tlwh || !det_conf ||
        !det_label || !det_count)
        return DD_ERR_INVALID;
    for (int k = 0; k < n_blobs; ++k)
        if (!host_dev_blobs[k] || ((uintptr_t)host_dev_blobs[k] & 15)) return DD_ERR_INVALID;
    Chunk& c = E->ch[chunk];
    for (int k = 0; k < n_blobs; ++k) c.dev_blob[k] = (unsigned char*)host_dev_blobs[k];
    c.n_blob = n_blobs;
    c.blob_cap = blob_capacity;
    c.s_tlwh = det_tlwh; c.s_conf = det_conf; c.s_label = det_label; c.s_count = det_count;
    if (!c.copy_st) DD_CU(cudaStreamCreateWithFlags(&c.copy_st, cudaStreamNonBlocking));
    if (!c.copy_st2) DD_CU(cudaStreamCreateWithFlags(&c.copy_st2, cudaStreamNonBlocking));
    if (!c.d2h_st) DD_CU(cudaStreamCreateWithFlags(&c.d2h_st, cudaStreamNonBlocking));
    return DD_OK;
}

int dd_engine_step(void* engine, const double* det_tlwh, const float* det_conf, const int32_t* det_label,
                   const float* det_feat, const int32_t* det_count, int32_t reduce, void* caller_stream) {
    return dd_engine_step_present(engine, det_tlwh, det_conf, det_label, det_feat, det_count, nullptr, reduce, caller_stream);
}

int dd_engine_step_present(void* engine, const double* det_tlwh, const float* det_conf, const int32_t* det_label,
                           const float* det_feat, const int32_t* det_count, const uint8_t* present, int32_t reduce,
                           void* caller_stream) {
    Engine* E = (Engine*)engine;
    if (!E || !det_tlwh || !det_conf || !det_label || !det_feat || !det_count) return DD_ERR_INVALID;
    cudaStream_t cur = (cudaStream_t)caller_stream;
    const int par = (int)(E->tick & 1);
    const bool multi = E->P > 1;
    reduce = reduce ? 1 : 0;
    if (multi) {
        DD_CU(cudaEventRecord(E->fork_ev, cur));
        for (auto& c : E->ch) DD_CU(cudaStreamWaitEvent(c.st, E->fork_ev, 0));
        if (reduce && E->sum_valid[par])            // partial_counts[par] of tick - 2 must have been summed
            for (auto& c : E->ch) DD_CU(cudaStreamWaitEvent(c.st, E->sum_done[par], 0));
    }
    for (int i = 0; i < E->P; ++i) {
        Chunk& c = E->ch[i];
        const size_t o = (size_t)c.lo * E->D;
        DDTickArgs A;
        A.det_tlwh = det_tlwh + o * 4; A.det_conf = det_conf + o; A.det_label = det_label + o;
        A.det_feat = det_feat + o * DD_FEAT_DIM; A.det_count = det_count + c.lo;
        A.out_ids = E->ids + o;
        A.out_counts = reduce ? E->partial + ((size_t)par * E->P + i) * E->C4 : nullptr;
        A.blob = nullptr;
        A.present = present ? present + c.lo : nullptr;
        A.off_tlwh = A.off_conf = A.off_label = A.off_feat = 0;
        A.indirect = 0;
        A.tick = (int)E->tick;
        cudaStream_t st = multi ? c.st : cur;
        const int rc = launch_tick(*E, c, A, 0, reduce, st);
        if (rc != DD_OK) return rc;
        if (multi) DD_CU(cudaEventRecord(c.done, st));
    }
    if (reduce) {
        const int rc = sum_partials(*E, par, cur);
        if (rc != DD_OK) return rc;
    }
    ++E->tick;
    return DD_OK;
}

}  // extern "C"

namespace {

// n_off: offsets per chunk in host_offsets, 4 (tlwh, conf, label, feat) or 5 (+ the u8 present[n] section)
int step_host(Engine* E, const void* const* host_blobs, const uint64_t* host_blob_bytes, const int64_t* host_offsets,
              int n_off, int32_t* host_out_ids, void* caller_stream) {
    if (!E || !host_blobs || !host_blob_bytes || !host_offsets) return DD_ERR_INVALID;
    cudaStream_t cur = (cudaStream_t)caller_stream;
    const int par = (int)(E->tick & 1);
    const bool multi = E->P > 1;
    for (int i = 0; i < E->P; ++i) {
        const int64_t* of = host_offsets + n_off * i;
        if (!host_blobs[i] || E->ch[i].n_blob < 2 || host_blob_bytes[i] > E->ch[i].blob_cap) return DD_ERR_INVALID;
        if ((of[0] & 7) || (of[1] & 3) || (of[2] & 3) || (of[3] & 15)) return DD_ERR_INVALID;
        if (n_off == 5 && (of[4] < 0 || (uint64_t)of[4] + (uint64_t)E->ch[i].n > host_blob_bytes[i])) return DD_ERR_INVALID;
    }
    if (multi && E->sum_valid[par])
        for (auto& c : E->ch) DD_CU(cudaStreamWaitEvent(c.st, E->sum_done[par], 0));
    for (int i = 0; i < E->P; ++i) {
        Chunk& c = E->ch[i];
        cudaStream_t st = multi ? c.st : cur;
        // upload on the chunk's copy streams into the buffer the tick before last has finished reading.  Two halves on
        // two streams: one DMA stream alone does not saturate the host link on every box (41 vs 54 GB/s measured), and
        // the chunks' uploads do not otherwise overlap in time
        const size_t total = (size_t)host_blob_bytes[i];
        size_t half = total > ((size_t)4 << 20) ? ((total / 2 + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1)) : total;
        if (half > total) half = total;
        const int bi = (int)(E->tick % c.n_blob);         // upload buffer of this tick: free once the tick n_blob back consumed it
        if (c.unpacked_valid[bi]) {
            DD_CU(cudaStreamWaitEvent(c.copy_st, c.unpacked[bi], 0));
            if (half < total) DD_CU(cudaStreamWaitEvent(c.copy_st2, c.unpacked[bi], 0));
        }
        DD_CU(cudaMemcpyAsync(c.dev_blob[bi], host_blobs[i], half, cudaMemcpyHostToDevice, c.copy_st));
        DD_CU(cudaEventRecord(c.copied, c.copy_st));
        DD_CU(cudaStreamWaitEvent(st, c.copied, 0));
        if (half < total) {
            DD_CU(cudaMemcpyAsync(c.dev_blob[bi] + half, (const char*)host_blobs[i] + half, total - half, cudaMemcpyHostToDevice,
                                  c.copy_st2));
            DD_CU(cudaEventRecord(c.copied2, c.copy_st2));
            DD_CU(cudaStreamWaitEvent(st, c.copied2, 0));
        }
        const size_t o = (size_t)c.lo * E->D;
        const int64_t* of = host_offsets + n_off * i;
        DDTickArgs A;
        A.det_tlwh = c.s_tlwh; A.det_conf = c.s_conf; A.det_label = c.s_label; A.det_feat = nullptr; A.det_count = c.s_count;
        A.out_ids = E->ids + o;
        A.out_counts = E->partial + ((size_t)par * E->P + i) * E->C4;
        A.blob = c.dev_blob[bi];
        A.off_tlwh = of[0]; A.off_conf = of[1]; A.off_label = of[2]; A.off_feat = of[3];
        A.present = n_off == 5 ? c.dev_blob[bi] + of[4] : nullptr;     // rides in the same upload
        A.indirect = 0;
        A.tick = (int)E->tick;
        // only the tick's first kernel reads the blob (later kernels read the small padded arrays it fills)
        const int rc = launch_tick(*E, c, A, 1, 1, st, c.unpacked[bi]);
        if (rc != DD_OK) return rc;
        c.unpacked_valid[bi] = true;
        if (host_out_ids) {
            const size_t nb = (size_t)c.n * E->D * sizeof(int);
            if (multi) {
                // off the chunk's stream: the read-back would otherwise sit in the chunk's chain in front of the next tick
                DD_CU(cudaEventRecord(c.tick_end, st));
                DD_CU(cudaStreamWaitEvent(c.d2h_st, c.tick_end, 0));
                DD_CU(cudaMemcpyAsync(host_out_ids + o, E->ids + o, nb, cudaMemcpyDeviceToHost, c.d2h_st));
                DD_CU(cudaEventRecord(c.d2h_done, c.d2h_st));
                c.d2h_valid = true;
            } else {
                DD_CU(cudaMemcpyAsync(host_out_ids + o, E->ids + o, nb, cudaMemcpyDeviceToHost, st));
            }
        }
        if (multi) DD_CU(cudaEventRecord(c.done, st));
    }
    const int rc = sum_partials(*E, par, cur);
    if (rc != DD_OK) return rc;
    ++E->tick;
    return DD_OK;
}

}  // namespace

extern "C" {

int dd_engine_step_host(void* engine, const void* const* host_blobs, const uint64_t* host_blob_bytes,
                        const int64_t* host_offsets4, int32_t* host_out_ids, void* caller_stream) {
    return step_host((Engine*)engine, host_blobs, host_blob_bytes, host_offsets4, 4, host_out_ids, caller_stream);
}

int dd_engine_step_host_present(void* engine, const void* const* host_blobs, const uint64_t* host_blob_bytes,
                                const int64_t* host_offsets5, int32_t* host_out_ids, void* caller_stream) {
    return step_host((Engine*)engine, host_blobs, host_blob_bytes, host_offsets5, 5, host_out_ids, caller_stream);
}

int dd_engine_copy_events(void* engine, int32_t* host_out, void* caller_stream) {
    Engine* E = (Engine*)engine;
    if (!E || !host_out) return DD_ERR_INVALID;
    for (auto& c : E->ch)
        if (c.cfg.event_cap <= 0) return DD_ERR_INVALID;
    const bool multi = E->P > 1;
    size_t o = 0;
    for (auto& c : E->ch) {
        const size_t words = 4 + 4 * (size_t)c.cfg.event_cap;
        const void* src = (const char*)c.state + c.events_off;
        if (multi) {
            // off the chunk's stream, as the ids of dd_engine_step_host: the next tick waits for d2h_done
            if (!c.d2h_st) DD_CU(cudaStreamCreateWithFlags(&c.d2h_st, cudaStreamNonBlocking));
            DD_CU(cudaEventRecord(c.tick_end, c.st));
            DD_CU(cudaStreamWaitEvent(c.d2h_st, c.tick_end, 0));
            DD_CU(cudaMemcpyAsync(host_out + o, src, words * sizeof(int32_t), cudaMemcpyDeviceToHost, c.d2h_st));
            DD_CU(cudaEventRecord(c.d2h_done, c.d2h_st));
            c.d2h_valid = true;
        } else {
            DD_CU(cudaMemcpyAsync(host_out + o, src, words * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                  (cudaStream_t)caller_stream));
        }
        o += words;
    }
    return DD_OK;
}

int dd_engine_join(void* engine, void* caller_stream) {
    Engine* E = (Engine*)engine;
    if (!E) return DD_ERR_INVALID;
    if (E->P == 1) return DD_OK;
    cudaStream_t cur = (cudaStream_t)caller_stream;
    for (auto& c : E->ch) {
        DD_CU(cudaEventRecord(c.done, c.st));
        DD_CU(cudaStreamWaitEvent(cur, c.done, 0));
        if (c.d2h_valid) DD_CU(cudaStreamWaitEvent(cur, c.d2h_done, 0));
    }
    if (E->last_sum >= 0) DD_CU(cudaStreamWaitEvent(cur, E->sum_done[E->last_sum], 0));
    return DD_OK;
}

int dd_engine_wait_counts(void* engine, void* caller_stream) {
    Engine* E = (Engine*)engine;
    if (!E) return DD_ERR_INVALID;
    if (E->P > 1 && E->last_sum >= 0) DD_CU(cudaStreamWaitEvent((cudaStream_t)caller_stream, E->sum_done[E->last_sum], 0));
    return DD_OK;
}

int dd_engine_pool_latest(void* engine, int32_t chunk, int32_t max_age_ticks, int32_t* host_out4, int64_t* host_out_tick) {
    Engine* E = (Engine*)engine;
    if (!E || chunk < 0 || chunk >= E->P || !host_out4 || !host_out_tick) return DD_ERR_INVALID;
    Chunk& c = E->ch[chunk];
    *host_out_tick = -1;
    const int newest = c.poll_turn ^ 1, older = c.poll_turn;          // poll_turn = the slot the NEXT poll writes
    int use = -1;
    for (const int k : {newest, older}) {                             // the most recent poll that has completed
        if (use >= 0 || c.poll_tick[k] < 0) continue;
        const cudaError_t q = cudaEventQuery(c.poll_ev[k]);
        if (q == cudaSuccess) use = k;
        else if (q != cudaErrorNotReady) return DD_ERR_CUDA;
    }
    cudaGetLastError();
    if (use < 0) {
        // none has: the host is too far ahead if one of them is max_age_ticks old -- wait for the most recent such poll.
        // (Waiting only for the newest would never happen once polls come more often than max_age_ticks: a newer poll
        // always replaces it before it gets that old, and a device that lags a few ticks would never be polled.)
        for (const int k : {newest, older}) {
            if (use >= 0 || c.poll_tick[k] < 0 || E->tick - c.poll_tick[k] < max_age_ticks) continue;
            DD_CU(blocked_sync(*E, c.poll_ev[k]));
            use = k;
        }
    }
    if (use < 0) return DD_OK;
    for (int k = 0; k < 4; ++k) host_out4[k] = c.poll_host[4 * use + k];
    *host_out_tick = c.poll_tick[use];
    return DD_OK;
}

int dd_engine_stats(void* engine, int64_t* host_out_ticks, int64_t* host_out_launches, double* host_out_blocked_ms) {
    Engine* E = (Engine*)engine;
    if (!E) return DD_ERR_INVALID;
    if (host_out_ticks) *host_out_ticks = E->tick;
    if (host_out_launches) *host_out_launches = E->launches;
    if (host_out_blocked_ms) *host_out_blocked_ms = E->blocked_ms;
    return DD_OK;
}

}  // extern "C"
