// dd_tracker.cu -- sm_100a kernels + C ABI of the batched DeepSORT tick.
//
// Launch shapes (S streams, T = max_tracks, D = max_dets; small per-item kernels use 8 lanes per item):
//   k_prep         (stream, detection) -> 8 lanes         xyah + unit feature (+ half copy)
//   k_gate         (stream, track index) -> 8 lanes       Track.predict + Mahalanobis gate + work list
//   gallery kernel persistent grid over the work list     <- the HBM-bound kernel (dd_gallery.cuh)
//   k_match        stream -> 1 warp (4 / 8 for crowds)    cascade + IoU stage + lifecycle, dynamic shared memory
//   k_apply        (stream, detection) -> 8 lanes         Kalman update / initiate + gallery append + label vote
//   k_countline    stream -> 1 warp                       (k_countline_ev: + the crossing records)
//   k_count_reduce one CTA per counter
#include <cuda_runtime.h>
#include "dd_gallery.cuh"

#define DD_CHECK_LAUNCH()                                         \
    do {                                                          \
        cudaError_t e__ = cudaGetLastError();                     \
        if (e__ != cudaSuccess) return DD_ERR_CUDA;               \
    } while (0)

// Small per-item kernels: DD_SUB lanes per item, 32 / DD_SUB items per warp (SubG).
#ifndef DD_MATCH_MIN_CTAS
#define DD_MATCH_MIN_CTAS 24     // <= 80 registers: a matching warp must fit beside the gallery stream of another chunk
#endif
#ifndef DD_APPLY_MIN_CTAS
#define DD_APPLY_MIN_CTAS 8      // <= 128 registers, no spills: an apply warp (4 K registers) must fit into what a
#endif                           // register-file partition has left beside five 72-register gallery warps of another chunk
#define DD_SUB 8
#define DD_ITEMS_PER_CTA (DD_WARPS * 32 / DD_SUB)

__global__ void __launch_bounds__(DD_WARPS * 32)
k_prep(const DDView V, const DDTickArgs A) {
    DDTlScope tl_(V, 0, A.tick);
    if (A.publish && blockIdx.x == 0 && threadIdx.x == 0) *const_cast<DDTickArgs*>(V.targs) = A;
    const double* __restrict__ det_tlwh = DD_ARG(det_tlwh);
    const float* __restrict__ det_feat = DD_ARG(det_feat);
    const int* __restrict__ det_count = DD_ARG(det_count);
    const int w = blockIdx.x * DD_ITEMS_PER_CTA + threadIdx.x / DD_SUB;
    if (blockIdx.x == 0 && threadIdx.x == 0) {      // new tick: empty work list, claim cursor at 0
        V.work_ctl[0] = 0;
        V.work_ctl[32] = 0;
        V.pool_ctl[3] = 0;                          // page-demand forecast, rebuilt by the apply kernel
    }
    if (w >= V.S * V.D) return;
    SubG<DD_SUB> g;
    dd_prep_det(g, V, w / V.D, w % V.D, det_tlwh, det_feat, det_count, DD_ARG(present));
}

__global__ void __launch_bounds__(DD_WARPS * 32) k_predict(const DDView V) {
    const int w = blockIdx.x * DD_ITEMS_PER_CTA + threadIdx.x / DD_SUB;
    if (w >= V.S * V.T) return;
    SubG<DD_SUB> g;
    dd_predict_track(g, V, w / V.T, w % V.T);
}

// PREDICT = true: Tracker.predict of the same track index first (the fused tick): the 8 lanes that gate a track
// have just written its predicted mean / covariance, so the state is read back from L1 instead of HBM and one
// launch disappears.
// k_prep fed by a ragged blob (dd_unpack_detections' format): expands box / confidence / label / count into the
// padded arrays the later kernels read and normalises the feature straight from the blob, so the 512-byte feature
// rows are never copied to a padded staging buffer.
struct DDRagged {
    const unsigned char* blob;
    long long off_tlwh, off_conf, off_label, off_feat;
    double* det_tlwh;
    float* det_conf;
    int *det_label, *det_count;
};

__global__ void __launch_bounds__(DD_WARPS * 32)
k_prep_ragged(const DDView V, const DDTickArgs A) {
    DDTlScope tl_(V, 0, A.tick);
    if (A.publish && blockIdx.x == 0 && threadIdx.x == 0) *const_cast<DDTickArgs*>(V.targs) = A;
    DDRagged R;
    R.blob = DD_ARG(blob);
    R.off_tlwh = DD_ARG(off_tlwh); R.off_conf = DD_ARG(off_conf); R.off_label = DD_ARG(off_label); R.off_feat = DD_ARG(off_feat);
    R.det_tlwh = (double*)DD_ARG(det_tlwh); R.det_conf = (float*)DD_ARG(det_conf);
    R.det_label = (int*)DD_ARG(det_label); R.det_count = (int*)DD_ARG(det_count);
    const int w = blockIdx.x * DD_ITEMS_PER_CTA + threadIdx.x / DD_SUB;
    if (blockIdx.x == 0 && threadIdx.x == 0) {      // new tick: empty work list, claim cursor at 0
        V.work_ctl[0] = 0;
        V.work_ctl[32] = 0;
        V.pool_ctl[3] = 0;                          // page-demand forecast, rebuilt by the apply kernel
    }
    if (w >= V.S * V.D) return;
    SubG<DD_SUB> g;
    const int s = w / V.D, d = w - s * V.D;
    if (!dd_prep_presence(g, V, s, d, DD_ARG(present))) return;     // an absent stream owns no entries
    const int* offs = (const int*)R.blob;
    const int o0 = offs[s];
    const int n = offs[s + 1] - o0;
    if (d == 0 && g.lane == 0) R.det_count[s] = n;     // n > max_dets: the tick raises DD_FLAG_DET_OVERFLOW
    if (d >= n) return;
    const size_t src = (size_t)o0 + d, dst = (size_t)s * V.D + d;
    const double* box = (const double*)(R.blob + R.off_tlwh) + src * 4;
    if (g.lane < 4) R.det_tlwh[dst * 4 + g.lane] = box[g.lane];
    if (g.lane == 4) R.det_conf[dst] = ((const float*)(R.blob + R.off_conf))[src];
    if (g.lane == 5) R.det_label[dst] = ((const int*)(R.blob + R.off_label))[src];
    dd_prep_det_at(g, V, s, d, box, (const float*)(R.blob + R.off_feat) + src * DD_FEAT_DIM);
}

#ifndef DD_GATE_MIN_CTAS
#define DD_GATE_MIN_CTAS 8      // 64 registers, no spills: 32 warps per SM instead of 28 (the kernel is bound by f64 dependency latency)
#endif
#if DD_GATE_MIN_CTAS > 0
#define DD_GATE_BOUNDS __launch_bounds__(DD_WARPS * 32, DD_GATE_MIN_CTAS)
#else
#define DD_GATE_BOUNDS __launch_bounds__(DD_WARPS * 32)
#endif
template <bool PREDICT>
__global__ void DD_GATE_BOUNDS
k_gate(const DDView V, const DDTickArgs A) {
    DDTlScope tl_(V, 1);
    const int* __restrict__ det_count = DD_ARG(det_count);
    // gate, then append the track indices that have something to stream to the work list of the gallery
    // kernel: one atomicAdd per CTA (16 track indices), entries of a CTA stay in ascending order.
    __shared__ int s_has[DD_ITEMS_PER_CTA];
    __shared__ int s_base;
    const int item = threadIdx.x / DD_SUB;
    const int w = blockIdx.x * DD_ITEMS_PER_CTA + item;
    SubG<DD_SUB> g;
    int has = 0;
    if (w < V.S * V.T) {
        if (PREDICT) {
            dd_tick_predict_track(g, V, w / V.T, w % V.T);
            g.sync();
        }
        has = dd_gate_track(g, V, w / V.T, w % V.T, det_count) > 0 ? 1 : 0;
    }
    if (g.lane == 0) s_has[item] = has;
    __syncthreads();
    if (threadIdx.x < 32) {
        const int h = threadIdx.x < DD_ITEMS_PER_CTA ? s_has[threadIdx.x] : 0;
        const unsigned m = __ballot_sync(0xffffffffu, h != 0);
        if (threadIdx.x == 0) s_base = m ? atomicAdd(V.work_ctl, __popc(m)) : 0;
        if (threadIdx.x < DD_ITEMS_PER_CTA) s_has[threadIdx.x] = __popc(m & ((1u << threadIdx.x) - 1u));
    }
    __syncthreads();
    if (has) {
        // work-list entry + its self-contained record (see work_rec in deepdish_b200.h): lane L writes words L, 8 + L
        const int idx = s_base + s_has[item];
        const int s = w / V.T;
        g.sync();                                   // the descriptor and gate words lane 0 wrote are visible
        const int4 dsc = *(const int4*)(V.cdesc + (size_t)w * 4);
        const size_t slotg = (size_t)s * V.T + dsc.x;
        int nd = det_count[s];
        if (nd > V.D) nd = V.D;
        int v = 0;
        switch (g.lane) {
            case 0: v = (int)slotg; V.work[idx] = w; break;
            case 1: v = s; break;
            case 2: v = dsc.y; break;
            case 3: v = dsc.z; break;
            case 4: v = dsc.w; break;
            case 5: v = (int)V.gate[slotg * V.DW]; break;
            case 6: v = V.DW > 1 ? (int)V.gate[slotg * V.DW + 1] : 0; break;
            default: v = nd; break;
        }
        int* rec = V.work_rec + (size_t)idx * 16;
        rec[g.lane] = v;
        rec[8 + g.lane] = g.lane < dsc.w ? V.ptab[slotg * V.PT + g.lane] : 0;
    }
}

static int dd_sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
    }
    return n;
}

__global__ void __launch_bounds__(32, DD_MATCH_MIN_CTAS)
k_match(const DDView V, const DDTickArgs A) {
    DDTlScope tl_(V, 3);
    extern __shared__ __align__(128) char smem[];
    WarpG g;
    // timeline slot 7 (config.timeline only): [0] = latest CTA start, [1] = longest single CTA, both relative quantities
    // that tell a placement delay (CTAs waiting for room on an SM) from a slow-down of the matching itself
    unsigned long long t0 = 0;
    if (V.tl && threadIdx.x == 0) t0 = dd_globaltimer();
    dd_match_stream(g, V, blockIdx.x, DD_ARG(det_tlwh), DD_ARG(det_count), DD_ARG(out_ids), smem);
    if (V.tl && threadIdx.x == 0) {
        atomicMax(DD_TL_SLOT(7), t0);
        atomicMax(DD_TL_SLOT(7) + 1, dd_globaltimer() - t0);
    }
}

// Crowded scenes (C4: ~260 tracks x ~180 detections per stream): the same matching body run by 4 (or 8) warps of
// one CTA per stream, so every column scan, list compaction and staging loop is 4x (8x) wider.
template <int NW>
__global__ void __launch_bounds__(NW * 32)
k_match_cta(const DDView V, const DDTickArgs A) {
    DDTlScope tl_(V, 3);
    extern __shared__ __align__(128) char smem[];
    CtaG<NW> g(smem);
    dd_match_stream(g, V, blockIdx.x, DD_ARG(det_tlwh), DD_ARG(det_count), DD_ARG(out_ids), smem + 256);
}

// 64-thread CTAs at <= 128 registers: at ~150 registers per thread a warp would not fit into any register-file
// partition beside the persistent gallery CTA of another chunk, and the whole kernel would wait for it to drain.
#define DD_APPLY_WARPS 2
#define DD_APPLY_ITEMS (DD_APPLY_WARPS * 32 / DD_SUB)
__global__ void __launch_bounds__(DD_APPLY_WARPS * 32, DD_APPLY_MIN_CTAS)
k_apply(const DDView V, const DDTickArgs A) {
    DDTlScope tl_(V, 4);
    const float* __restrict__ det_conf = DD_ARG(det_conf);
    const int* __restrict__ det_label = DD_ARG(det_label);
    __shared__ double scratch[DD_APPLY_ITEMS][64];
    const int w = blockIdx.x * DD_APPLY_ITEMS + threadIdx.x / DD_SUB;
    if (w >= V.S * V.D) return;
    SubG<DD_SUB> g;
    dd_apply_det(g, V, w / V.D, w % V.D, det_conf, det_label, scratch[threadIdx.x / DD_SUB]);
}

__global__ void __launch_bounds__(DD_WARPS * 32)
k_countline(const DDView V, const double* __restrict__ line, int line_per_stream) {
    DDTlScope tl_(V, 5);
    const int w = blockIdx.x * DD_WARPS + (threadIdx.x >> 5);
    if (w >= V.S) return;
    WarpG g;
    dd_countline(g, V, w, line + (line_per_stream ? (size_t)w * 4 : 0));
}

// k_countline that also writes the crossing records (config.event_cap > 0); a kernel of its own so that k_countline
// stays exactly what it is when the records are off
__global__ void __launch_bounds__(DD_WARPS * 32)
k_countline_ev(const DDView V, const double* __restrict__ line, int line_per_stream) {
    DDTlScope tl_(V, 5);
    const int w = blockIdx.x * DD_WARPS + (threadIdx.x >> 5);
    if (w >= V.S) return;
    WarpG g;
    dd_countline<WarpG, true>(g, V, w, line + (line_per_stream ? (size_t)w * 4 : 0));
}

// counts [S, C*4] -> out [C*4]; one CTA per output element, tree reduction over streams.
__global__ void __launch_bounds__(256)
k_count_reduce(const long long* __restrict__ counts, int S, int n, long long* __restrict__ out,
               const DDTickArgs* __restrict__ ind) {
    if (ind) out = ind->out_counts;                  // captured tick: the output alternates between ticks
    __shared__ long long sh[256];
    const int e = blockIdx.x;
    long long acc = 0;
    for (int s = threadIdx.x; s < S; s += blockDim.x) acc += counts[(size_t)s * n + e];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[e] = sh[0];
}

__global__ void __launch_bounds__(256) k_init(const DDView V, int n_pages) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V.S) V.next_id[i] = 1;
    if (i < n_pages) V.free_stack[i] = n_pages - 1 - i;        // page 0 is handed out first
    if (i == 0) { V.pool_ctl[0] = n_pages; V.pool_ctl[1] = n_pages; V.pool_ctl[2] = 0; }
}

// a new segment's page ids go on top of the free stack (the counters are bumped by k_pool_commit afterwards)
__global__ void __launch_bounds__(256) k_pool_attach(const DDView V, int first_page, int n_pages) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pages) V.free_stack[V.pool_ctl[0] + i] = first_page + n_pages - 1 - i;
}
__global__ void k_pool_commit(const DDView V, int n_pages) {
    V.pool_ctl[0] += n_pages;
    V.pool_ctl[1] += n_pages;
}

// metric.samples[track], oldest row first: one warp per output row
__global__ void __launch_bounds__(DD_WARPS * 32)
k_gallery_read(const DDView V, int s, int slot_in_stream, float* __restrict__ out, int max_rows) {
    const size_t slot = (size_t)s * V.T + slot_in_stream;
    const int len = V.gal_len[slot], pos = V.gal_pos[slot];
    const int n = len < max_rows ? len : max_rows;
    const int i = blockIdx.x * DD_WARPS + (threadIdx.x >> 5);
    if (i >= n) return;
    int row = i;
    if (V.B > 0) {
        row = pos - len + i;
        if (row < 0) row += V.B;
    }
    ((float4*)(out + (size_t)i * DD_FEAT_DIM))[threadIdx.x & 31] = dd_gallery_row(V, V.ptab + slot * V.PT, row)[threadIdx.x & 31];
}

// host edit: append (or insert before the newest row) one unit feature; one warp
__global__ void __launch_bounds__(32)
k_gallery_insert(const DDView V, int s, int slot_in_stream, const float* __restrict__ feat, int before_newest) {
    WarpG g;
    const size_t slot = (size_t)s * V.T + slot_in_stream;
    const int pos = V.gal_pos[slot], len = V.gal_len[slot], np = V.gal_np[slot];
    float4 x[1];
    x[0] = ((const float4*)feat)[g.lane];
    if (before_newest && len > 0) {
        int last = pos - 1;
        if (last < 0) last += V.B;                       // only a ring wraps
        const int pid = V.ptab[slot * V.PT + (last >> 4)];
        float4 newest[1];
        newest[0] = dd_page_f32(V, pid)[(size_t)(last & 15) * (DD_FEAT_DIM / 4) + g.lane];
        __syncwarp();
        dd_gallery_store_row<WarpG, 1>(g, V, pid, last & 15, x);
        __syncwarp();
        dd_gallery_append<WarpG, 1>(g, V, s, slot, pos, len, np, newest);
    } else {
        dd_gallery_append<WarpG, 1>(g, V, s, slot, pos, len, np, x);
    }
}

__global__ void __launch_bounds__(256)
k_status(const DDView V) {
    __shared__ int sh;
    if (threadIdx.x == 0) sh = 0;
    __syncthreads();
    int acc = 0;
    for (int s = threadIdx.x; s < V.S; s += blockDim.x) acc |= V.err[s];
    acc = __reduce_or_sync(0xffffffffu, acc);
    if ((threadIdx.x & 31) == 0 && acc) atomicOr(&sh, acc);
    __syncthreads();
    if (threadIdx.x == 0) V.pool_ctl[8] = sh;
}

// Ragged host batch -> the padded arrays of the tick.  One warp per detection (512 B feature + box + conf + label).
__global__ void __launch_bounds__(DD_WARPS * 32)
k_unpack(const unsigned char* __restrict__ blob, int S, int dmax, long long off_tlwh, long long off_conf,
         long long off_label, long long off_feat, double* __restrict__ det_tlwh, float* __restrict__ det_conf,
         int* __restrict__ det_label, float* __restrict__ det_feat, int* __restrict__ det_count) {
    const int* offs = (const int*)blob;                           // [S + 1]
    const int w = blockIdx.x * DD_WARPS + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= S * dmax) return;
    const int s = w / dmax, d = w - s * dmax;
    const int o0 = offs[s];
    const int n = offs[s + 1] - o0;
    if (d == 0 && lane == 0) det_count[s] = n;                    // n > dmax: the tick raises DD_FLAG_DET_OVERFLOW
    if (d >= n) return;
    const size_t src = (size_t)o0 + d, dst = (size_t)s * dmax + d;
    ((float4*)(det_feat + dst * DD_FEAT_DIM))[lane] = ((const float4*)(blob + off_feat) + src * (DD_FEAT_DIM / 4))[lane];
    if (lane < 4) det_tlwh[dst * 4 + lane] = ((const double*)(blob + off_tlwh))[src * 4 + lane];
    if (lane == 4) det_conf[dst] = ((const float*)(blob + off_conf))[src];
    if (lane == 5) det_label[dst] = ((const int*)(blob + off_label))[src];
}

static inline int warps_to_blocks(long long n_warps) { return (int)((n_warps + DD_WARPS - 1) / DD_WARPS); }
static inline int items_to_blocks(long long n) { return (int)((n + DD_ITEMS_PER_CTA - 1) / DD_ITEMS_PER_CTA); }

// ---- the launches of one update (shared by every entry point) --------------------------------------------
template <class... KArgs, class... Args>
static void dd_launch(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t st, Args... args) {
    kernel<<<grid, block, smem, st>>>(KArgs(args)...);
}
// Function attributes (opt-in shared memory) are set here, outside any stream capture.
static int dd_tick_prepare(const DDView& V, const dd_tracker_config* cfg, int* triples_out, int* stages_out, int* mw_out) {
    const size_t smem = dd_match_smem_bytes(V.T, V.D, V.tab_cap);
    if (smem > 227 * 1024) return DD_ERR_INVALID;
    int mw = cfg->match_warps;
    if (mw != 1 && mw != 4 && mw != 8) mw = (V.T > 160 || V.D > 160) ? 4 : 1;
    if (mw > 1 && smem + 256 > 227 * 1024) mw = 1;
    // Function attributes belong to a device: the caches below (what has been opted in so far; the attributes only ever
    // grow) are kept per device, so a process that drives several GPUs sets them on each.
    struct Opted { size_t match = 0, cta = 0, gsm = 0; bool carve = false; };
    static Opted opted[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return DD_ERR_CUDA;
    size_t &match_set = opted[dev].match, &cta_set = opted[dev].cta, &gsm_set = opted[dev].gsm;
    bool& carve_set = opted[dev].carve;
    // Shared-memory carve-out: an SM's L1 / shared split is fixed by the first CTA that lands on it and cannot change
    // while CTAs are resident.  The driver would give the gallery stream the smallest configuration that holds ONE of
    // its CTAs (196 KB for 170 KB), leaving 25 KB -- one matching warp -- for everything else of the other stream
    // chunks.  Every tick kernel therefore asks for the maximum carve-out (228 KB), whichever reaches an idle SM first.
    if (!carve_set) {
        const int mx = cudaSharedmemCarveoutMaxShared;
        const void* ks[] = {(const void*)k_prep, (const void*)k_prep_ragged, (const void*)k_gate<true>, (const void*)k_gate<false>,
                            (const void*)k_gallery_stream, (const void*)k_cosine, (const void*)k_match,
                            (const void*)k_match_cta<4>, (const void*)k_match_cta<8>, (const void*)k_apply,
                            (const void*)k_countline, (const void*)k_countline_ev, (const void*)k_count_reduce,
                            (const void*)k_predict};
        for (const void* k : ks)
            if (cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, mx) != cudaSuccess) return DD_ERR_CUDA;
        carve_set = true;
    }
    if (mw == 1 && smem > 48 * 1024 && smem > match_set) {
        if (cudaFuncSetAttribute(k_match, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return DD_ERR_CUDA;
        match_set = smem;
    }
    if (mw > 1 && smem + 256 > 48 * 1024 && smem + 256 > cta_set) {
        if (cudaFuncSetAttribute(k_match_cta<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem + 256)) != cudaSuccess ||
            cudaFuncSetAttribute(k_match_cta<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem + 256)) != cudaSuccess)
            return DD_ERR_CUDA;
        cta_set = smem + 256;
    }
    int triples = 0, stages = 0;
    if (cfg->gallery_impl == 0) {
        const bool split = cfg->gallery_waves > 0;             // one triple per CTA
        triples = cfg->cosine_ctas_per_sm > 0 ? cfg->cosine_ctas_per_sm : 7;
        if (triples > (split ? 8 : 7)) triples = split ? 8 : 7;
        stages = cfg->gallery_stages > 0 ? cfg->gallery_stages : 4;
        if (stages > 16) stages = 16;
        const size_t per = dd_gs_triple_bytes(stages);
        while (triples > 1 && (split ? (per + 1024) * triples > 228 * 1024 : per * triples > 226 * 1024)) --triples;
        const size_t gsm = split ? per : per * triples;
        if (gsm > 227 * 1024) return DD_ERR_INVALID;
        if (gsm > gsm_set) {
            if (cudaFuncSetAttribute(k_gallery_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm) != cudaSuccess)
                return DD_ERR_CUDA;
            gsm_set = gsm;
        }
    }
    *triples_out = triples; *stages_out = stages; *mw_out = mw;
    return DD_OK;
}

static int dd_launch_gallery(const DDView& V, const dd_tracker_config* cfg, const DDTickArgs& A, int triples, int stages,
                             cudaStream_t st) {
    const int impl = cfg->gallery_impl;
    if (impl == 1) {
        k_cosine<<<warps_to_blocks((long long)V.S * V.T), DD_WARPS * 32, 0, st>>>(V, A);
    } else if (impl == 0) {
        if (cfg->gallery_waves > 0)
            k_gallery_stream<<<dd_sm_count() * triples * cfg->gallery_waves, 96, dd_gs_triple_bytes(stages), st>>>(V, stages, 1);
        else
            k_gallery_stream<<<dd_sm_count(), triples * 96, dd_gs_triple_bytes(stages) * triples, st>>>(V, stages, 0);
    } else {
        return DD_ERR_INVALID;
    }
    DD_CHECK_LAUNCH();
    return DD_OK;
}

// parts: which kernels of the update to launch (the engine captures a tick in pieces so that it can put events between them)
#define DD_PART_PREP 1      // detection prep (the only reader of a ragged blob)
#define DD_PART_GATE 2      // Track.predict + gating + work list
#define DD_PART_GALLERY 4   // the gallery stream
#define DD_PART_POST 8      // matching + apply
#define DD_PART_TAIL 16     // count-line (+ count reduce): dd_tick_tail
#define DD_PART_ALL 31
static int dd_update_impl(void* state, const dd_tracker_config* cfg, const DDTickArgs& A, cudaStream_t st,
                          cudaEvent_t* ev, bool with_predict, int parts = DD_PART_ALL) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    if (!A.indirect && (!A.det_tlwh || !A.det_conf || !A.det_label || (!A.det_feat && !A.blob) || !A.det_count))
        return DD_ERR_INVALID;
    int triples = 0, stages = 0, mw = 1;
    rc = dd_tick_prepare(V, cfg, &triples, &stages, &mw);
    if (rc != DD_OK) return rc;
    const size_t smem = dd_match_smem_bytes(V.T, V.D, V.tab_cap);
    const bool ragged = A.blob != nullptr;       // (captured tick: a non-NULL marker, the kernels read V.targs->blob)
    if (ev) cudaEventRecord(ev[0], st);
    if (parts & DD_PART_PREP) {
        if (ragged)
            dd_launch(k_prep_ragged, items_to_blocks((long long)V.S * V.D), DD_WARPS * 32, 0, st, V, A);
        else
            dd_launch(k_prep, items_to_blocks((long long)V.S * V.D), DD_WARPS * 32, 0, st, V, A);
        DD_CHECK_LAUNCH();
    }
    if (ev) cudaEventRecord(ev[1], st);
    if (parts & DD_PART_GATE) {
        if (with_predict)
            dd_launch(k_gate<true>, items_to_blocks((long long)V.S * V.T), DD_WARPS * 32, 0, st, V, A);
        else
            dd_launch(k_gate<false>, items_to_blocks((long long)V.S * V.T), DD_WARPS * 32, 0, st, V, A);
        DD_CHECK_LAUNCH();
    }
    if (ev) cudaEventRecord(ev[2], st);
    if (parts & DD_PART_GALLERY) {
        rc = dd_launch_gallery(V, cfg, A, triples, stages, st);
        if (rc != DD_OK) return rc;
    }
    if (ev) cudaEventRecord(ev[3], st);
    if (parts & DD_PART_POST) {
        if (mw == 1)
            dd_launch(k_match, V.S, 32, smem, st, V, A);
        else if (mw == 8)
            dd_launch(k_match_cta<8>, V.S, 8 * 32, smem + 256, st, V, A);
        else
            dd_launch(k_match_cta<4>, V.S, 4 * 32, smem + 256, st, V, A);
        DD_CHECK_LAUNCH();
    }
    if (ev) cudaEventRecord(ev[4], st);
    if (parts & DD_PART_POST) {
        dd_launch(k_apply, (unsigned)(((long long)V.S * V.D + DD_APPLY_ITEMS - 1) / DD_APPLY_ITEMS), DD_APPLY_WARPS * 32, 0, st, V, A);
        DD_CHECK_LAUNCH();
    }
    if (ev) cudaEventRecord(ev[5], st);
    return DD_OK;
}

// reduce (captured tick): the count reduction into the tick's out_counts, read from the blob's tick_args words
static int dd_tick_tail(void* state, const dd_tracker_config* cfg, const double* line, int line_per_stream, bool reduce,
                        cudaStream_t st) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    if (V.ev) {
        // a new crossing list (a memset node in a captured tick)
        if (cudaMemsetAsync(V.ev, 0, sizeof(int), st) != cudaSuccess) return DD_ERR_CUDA;
        dd_launch(k_countline_ev, warps_to_blocks(V.S), DD_WARPS * 32, 0, st, V, line, line_per_stream);
    } else {
        dd_launch(k_countline, warps_to_blocks(V.S), DD_WARPS * 32, 0, st, V, line, line_per_stream);
    }
    DD_CHECK_LAUNCH();
    if (reduce) {
        dd_launch(k_count_reduce, V.C * 4, 256, 0, st, (const long long*)V.counts, V.S, V.C * 4, (long long*)nullptr,
                  (const DDTickArgs*)V.targs);
        DD_CHECK_LAUNCH();
    }
    return DD_OK;
}

static DDTickArgs dd_args_padded(const double* det_tlwh, const float* det_conf, const int* det_label, const float* det_feat,
                                 const int* det_count, int* out_ids) {
    DDTickArgs A;
    A.det_tlwh = det_tlwh; A.det_conf = det_conf; A.det_label = det_label; A.det_feat = det_feat; A.det_count = det_count;
    A.out_ids = out_ids; A.out_counts = nullptr; A.blob = nullptr; A.present = nullptr;
    A.off_tlwh = A.off_conf = A.off_label = A.off_feat = 0;
    A.indirect = 0;
    A.tick = 0;
    A.publish = 0;
    return A;
}

// One captured tick (dd_engine.cu): every per-tick input comes from the blob's tick_args words.
// The kernels `parts` (DD_PART_*) of one tick, every per-tick input read from the blob's tick_args words: what the engine
// captures (a ragged tick's prep kernel runs in front of the graphs so that "blob consumed" can be recorded behind it).
int dd_capture_tick(void* state, const dd_tracker_config* cfg, int ragged, int reduce, int parts, const double* line,
                    int line_per_stream, cudaStream_t st) {
    DDTickArgs A = dd_args_padded(nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
    A.indirect = 1;
    A.blob = ragged ? (const unsigned char*)(uintptr_t)16 : nullptr;      // marker only: the kernels read V.targs->blob
    if (parts & (DD_PART_ALL & ~DD_PART_TAIL)) {
        const int rc = dd_update_impl(state, cfg, A, st, nullptr, true, parts);
        if (rc != DD_OK) return rc;
    }
    if (parts & DD_PART_TAIL) return dd_tick_tail(state, cfg, line, line_per_stream, reduce != 0, st);
    return DD_OK;
}
#ifdef DD_GS_VARIANTS
// Benchmark hook (A/B builds only, benchmarks/gallery_variants.py): run gallery-stream variant `skip` again on the work
// list the last tick left behind.  Variants other than 0 write wrong costs -- nothing reads them before the next tick.
extern "C" int dd_gallery_replay(void* state, const dd_tracker_config* cfg, int skip, void* stream) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    int triples = 0, stages = 0, mw = 1;
    rc = dd_tick_prepare(V, cfg, &triples, &stages, &mw);
    if (rc != DD_OK || cfg->gallery_impl != 0) return DD_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t gsm = dd_gs_triple_bytes(stages) * triples;
    k_reset_cursor<<<1, 1, 0, st>>>(V);
#define DD_VARIANT(S) case S: \
        cudaFuncSetAttribute(k_gallery_stream_dbg<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm); \
        cudaFuncSetAttribute(k_gallery_stream_dbg<S>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); \
        k_gallery_stream_dbg<S><<<dd_sm_count(), triples * 96, gsm, st>>>(V, stages, 0); break;
    switch (skip) {
        DD_VARIANT(0) DD_VARIANT(1) DD_VARIANT(2) DD_VARIANT(3) DD_VARIANT(4) DD_VARIANT(7) DD_VARIANT(8) DD_VARIANT(15)
        DD_VARIANT(16) DD_VARIANT(31)
        default: return DD_ERR_INVALID;
    }
#undef DD_VARIANT
    DD_CHECK_LAUNCH();
    return DD_OK;
}
// read (and reset) the role-level cycle counters of the variant kernels: host_out16 u64[16]
extern "C" int dd_gallery_prof(unsigned long long* host_out16, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaStreamSynchronize(st) != cudaSuccess) return DD_ERR_CUDA;
    if (cudaMemcpyFromSymbol(host_out16, dd_gs_prof, 16 * sizeof(unsigned long long)) != cudaSuccess) return DD_ERR_CUDA;
    unsigned long long z[16] = {0};
    if (cudaMemcpyToSymbol(dd_gs_prof, z, sizeof(z)) != cudaSuccess) return DD_ERR_CUDA;
    return DD_OK;
}
#endif

// The detection-prep kernel of an engine tick: launched plainly (not captured) with the tick's arguments by value, which
// it publishes into the blob's tick_args words for the captured kernels behind it.
int dd_launch_prep_publishing(void* state, const dd_tracker_config* cfg, const DDTickArgs* A, cudaStream_t st) {
    DDTickArgs a = *A;
    a.indirect = 0;
    a.publish = 1;
    return dd_update_impl(state, cfg, a, st, nullptr, true, DD_PART_PREP);
}

int dd_tick_prepare_host(void* state, const dd_tracker_config* cfg) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    int a, b, c;
    return dd_tick_prepare(V, cfg, &a, &b, &c);
}
size_t dd_tick_args_offset(const dd_tracker_config* cfg) {
    dd_tracker_layout L;
    return dd_layout_compute(cfg, &L) == DD_OK ? (size_t)L.tick_args : 0;
}

extern "C" {

const char* dd_version(void) { return "deepdish_b200 0.2.0 (sm_100a)"; }

int dd_tracker_layout_query(const dd_tracker_config* cfg, dd_tracker_layout* out) {
    return dd_layout_compute(cfg, out);
}

int dd_tracker_init(void* state, const dd_tracker_config* cfg, void* stream) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    dd_tracker_layout L;
    dd_layout_compute(cfg, &L);
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(state, 0, L.total_bytes, st) != cudaSuccess) return DD_ERR_CUDA;
    const int n_pages = cfg->n_segs * cfg->seg_pages;
    const int n = n_pages > V.S ? n_pages : V.S;
    k_init<<<(n + 255) / 256, 256, 0, st>>>(V, n_pages);
    DD_CHECK_LAUNCH();
    return DD_OK;
}

int dd_tracker_pool_attach(void* state, const dd_tracker_config* cfg, void* stream) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    if (cfg->n_segs < 2) return DD_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    const int n = cfg->seg_pages;
    k_pool_attach<<<(n + 255) / 256, 256, 0, st>>>(V, (cfg->n_segs - 1) * n, n);
    DD_CHECK_LAUNCH();
    k_pool_commit<<<1, 1, 0, st>>>(V, n);
    DD_CHECK_LAUNCH();
    return DD_OK;
}

int dd_tracker_gallery_read(void* state, const dd_tracker_config* cfg, int32_t stream_index, int32_t slot,
                            float* out, int32_t max_rows, void* stream) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    if (!out || stream_index < 0 || stream_index >= V.S || slot < 0 || slot >= V.T || max_rows < 0) return DD_ERR_INVALID;
    if (max_rows == 0) return DD_OK;
    k_gallery_read<<<warps_to_blocks(max_rows), DD_WARPS * 32, 0, (cudaStream_t)stream>>>(V, stream_index, slot, out, max_rows);
    DD_CHECK_LAUNCH();
    return DD_OK;
}

int dd_tracker_gallery_insert(void* state, const dd_tracker_config* cfg, int32_t stream_index, int32_t slot,
                              const float* feat, int32_t before_newest, void* stream) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    if (!feat || stream_index < 0 || stream_index >= V.S || slot < 0 || slot >= V.T) return DD_ERR_INVALID;
    k_gallery_insert<<<1, 32, 0, (cudaStream_t)stream>>>(V, stream_index, slot, feat, before_newest);
    DD_CHECK_LAUNCH();
    return DD_OK;
}

int dd_tracker_predict(void* state, const dd_tracker_config* cfg, void* stream) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    k_predict<<<items_to_blocks((long long)V.S * V.T), DD_WARPS * 32, 0, (cudaStream_t)stream>>>(V);
    DD_CHECK_LAUNCH();
    return DD_OK;
}

int dd_tracker_update(void* state, const dd_tracker_config* cfg, const double* det_tlwh,
                      const float* det_conf, const int32_t* det_label, const float* det_feat,
                      const int32_t* det_count, int32_t* out_det_track_id, void* stream) {
    const DDTickArgs in = dd_args_padded(det_tlwh, det_conf, det_label, det_feat, det_count, out_det_track_id);
    return dd_update_impl(state, cfg, in, (cudaStream_t)stream, nullptr, false);
}

int dd_tracker_update_profiled(void* state, const dd_tracker_config* cfg, const double* det_tlwh,
                               const float* det_conf, const int32_t* det_label, const float* det_feat,
                               const int32_t* det_count, int32_t* out_det_track_id, void* stream,
                               void* const* host_events6) {
    if (!host_events6) return DD_ERR_INVALID;
    cudaEvent_t ev[6];
    for (int i = 0; i < 6; ++i) ev[i] = (cudaEvent_t)host_events6[i];
    const DDTickArgs in = dd_args_padded(det_tlwh, det_conf, det_label, det_feat, det_count, out_det_track_id);
    return dd_update_impl(state, cfg, in, (cudaStream_t)stream, ev, false);
}

int dd_event_create(void** host_out) {
    if (!host_out) return DD_ERR_INVALID;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return DD_ERR_CUDA;
    *host_out = (void*)e;
    return DD_OK;
}

int dd_event_destroy(void* ev) { return cudaEventDestroy((cudaEvent_t)ev) == cudaSuccess ? DD_OK : DD_ERR_CUDA; }

int dd_event_elapsed_ms(void* start, void* end, float* host_ms) {
    if (!host_ms) return DD_ERR_INVALID;
    return cudaEventElapsedTime(host_ms, (cudaEvent_t)start, (cudaEvent_t)end) == cudaSuccess ? DD_OK : DD_ERR_CUDA;
}

int dd_event_record(void* ev, void* stream) {
    return cudaEventRecord((cudaEvent_t)ev, (cudaStream_t)stream) == cudaSuccess ? DD_OK : DD_ERR_CUDA;
}

int dd_tracker_countline(void* state, const dd_tracker_config* cfg, const double* line,
                         int line_per_stream, void* stream) {
    if (!line) return DD_ERR_INVALID;
    return dd_tick_tail(state, cfg, line, line_per_stream, false, (cudaStream_t)stream);
}

int dd_unpack_detections(const void* blob, int32_t n_streams, int32_t max_dets, int64_t off_tlwh, int64_t off_conf,
                         int64_t off_label, int64_t off_feat, double* det_tlwh, float* det_conf,
                         int32_t* det_label, float* det_feat, int32_t* det_count, void* stream) {
    if (!blob || !det_tlwh || !det_conf || !det_label || !det_feat || !det_count) return DD_ERR_INVALID;
    if (n_streams <= 0 || max_dets <= 0) return DD_ERR_INVALID;
    if ((off_tlwh & 7) || (off_conf & 3) || (off_label & 3) || (off_feat & 15) || ((uintptr_t)blob & 15)) return DD_ERR_INVALID;
    k_unpack<<<warps_to_blocks((long long)n_streams * max_dets), DD_WARPS * 32, 0, (cudaStream_t)stream>>>(
        (const unsigned char*)blob, n_streams, max_dets, off_tlwh, off_conf, off_label, off_feat, det_tlwh, det_conf,
        det_label, det_feat, det_count);
    DD_CHECK_LAUNCH();
    return DD_OK;
}

int dd_tracker_count_reduce(void* state, const dd_tracker_config* cfg, int64_t* out_counts, void* stream) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    if (!out_counts) return DD_ERR_INVALID;
    k_count_reduce<<<V.C * 4, 256, 0, (cudaStream_t)stream>>>(V.counts, V.S, V.C * 4, (long long*)out_counts, nullptr);
    DD_CHECK_LAUNCH();
    return DD_OK;
}

int dd_tracker_status(void* state, const dd_tracker_config* cfg, int32_t* host_flags, void* stream) {
    DDView V;
    int rc = dd_make_view(state, cfg, &V);
    if (rc != DD_OK) return rc;
    if (!host_flags) return DD_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    k_status<<<1, 256, 0, st>>>(V);                   // the OR lands in a scratch word of the blob: no allocation
    cudaError_t e = cudaMemcpyAsync(host_flags, V.pool_ctl + 8, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    return e == cudaSuccess ? DD_OK : DD_ERR_CUDA;
}

}  // extern "C"
