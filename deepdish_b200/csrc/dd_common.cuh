// dd_common.cuh -- thread-group abstraction + exact-arithmetic helpers shared by all kernels.
//
// Every kernel body is a template over a "group" G: the set of threads that cooperate on one unit
// of work (a track, a stream, a frame).  On the device G is a warp (WarpG) or a whole CTA (BlockG).
// tests/hostemu compiles the very same bodies with HostG (one lane, all collectives trivial) into a
// host library so the serial logic (scipy-exact LSAP, CPython set order, lifecycle) can be checked
// on a machine without a GPU.  HostG is test scaffolding only: the product library never runs it.
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define DD_HD __host__ __device__ __forceinline__
#define DD_D __device__ __forceinline__
#else
#define DD_HD inline
#define DD_D inline
struct alignas(16) float4 { float x, y, z, w; };      // host emulation build only
#endif

// ---- f64/f32 arithmetic that must round like numpy's element-wise ops (no FMA contraction) -------
// The library is compiled with -fmad=false; these wrappers additionally pin the intent where an
// operation order decides a thresholded (bit-exact) output.
#if defined(__CUDA_ARCH__)
DD_D double dd_mul(double a, double b) { return __dmul_rn(a, b); }
DD_D double dd_add(double a, double b) { return __dadd_rn(a, b); }
DD_D double dd_sub(double a, double b) { return __dsub_rn(a, b); }
DD_D double dd_div(double a, double b) { return __ddiv_rn(a, b); }
DD_D double dd_sqrt(double a) { return __dsqrt_rn(a); }
DD_D float dd_fmaf(float a, float b, float c) { return __fmaf_rn(a, b, c); }
DD_D float dd_mulf(float a, float b) { return __fmul_rn(a, b); }
DD_D float dd_addf(float a, float b) { return __fadd_rn(a, b); }
DD_D float dd_subf(float a, float b) { return __fsub_rn(a, b); }
DD_D float dd_divf(float a, float b) { return __fdiv_rn(a, b); }
DD_D float dd_sqrtf(float a) { return __fsqrt_rn(a); }
#else
inline double dd_mul(double a, double b) { volatile double r = a * b; return r; }
inline double dd_add(double a, double b) { return a + b; }
inline double dd_sub(double a, double b) { return a - b; }
inline double dd_div(double a, double b) { return a / b; }
inline double dd_sqrt(double a) { return sqrt(a); }
inline float dd_fmaf(float a, float b, float c) { return fmaf(a, b, c); }
inline float dd_mulf(float a, float b) { volatile float r = a * b; return r; }
inline float dd_addf(float a, float b) { return a + b; }
inline float dd_subf(float a, float b) { return a - b; }
inline float dd_divf(float a, float b) { return a / b; }
inline float dd_sqrtf(float a) { return sqrtf(a); }
#endif

DD_HD double dd_max(double a, double b) { return a > b ? a : b; }   // np.maximum for non-NaN input
DD_HD double dd_min(double a, double b) { return a < b ? a : b; }
#if defined(__CUDA_ARCH__)
DD_D int dd_ctz(unsigned w) { return __ffs((int)w) - 1; }
#else
inline int dd_ctz(unsigned w) { return __builtin_ctz(w); }
#endif
#if defined(__CUDA_ARCH__)
DD_D int dd_popc(unsigned w) { return __popc(w); }
#else
inline int dd_popc(unsigned w) { return __builtin_popcount(w); }
#endif
DD_HD int dd_imin(int a, int b) { return a < b ? a : b; }
DD_HD int dd_imax(int a, int b) { return a > b ? a : b; }

// __syncwarp for code that only the first warp of a CTA executes (no-op on the host emulation)
#if defined(__CUDA_ARCH__)
DD_D void dd_first_warp_sync() { __syncwarp(); }
#else
inline void dd_first_warp_sync() {}
#endif

// (value, preference) pair used by the LSAP column scan: lower value wins, ties -> higher pref.
struct DDKey {
    double val;
    int pref;
};
DD_HD bool dd_key_better(const DDKey& a, const DDKey& b) {   // is a strictly better than b
    return (a.val < b.val) || (a.val == b.val && a.pref > b.pref);
}

#if defined(__CUDACC__)
// ---------------------------------------------------------------------------------------- WarpG
struct WarpG {
    static constexpr int NL = 32;
    int lane;
    __device__ explicit WarpG() : lane(threadIdx.x & 31) {}
    __device__ void sync() const { __syncwarp(); }
    __device__ float sum(float v) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    }
    __device__ double sum(double v) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    }
    __device__ int sum(int v) const { return __reduce_add_sync(0xffffffffu, v); }
    __device__ int imax(int v) const { return __reduce_max_sync(0xffffffffu, v); }
    __device__ int imin(int v) const { return __reduce_min_sync(0xffffffffu, v); }
    __device__ float fmax(float v) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = ::fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
        return v;
    }
    __device__ unsigned bor(unsigned v) const { return __reduce_or_sync(0xffffffffu, v); }
    __device__ bool any(bool p) const { return __any_sync(0xffffffffu, p); }
    // exclusive prefix count of a per-lane predicate + total (ordered compaction)
    __device__ int scan_excl(bool p, int& total) const {
        unsigned m = __ballot_sync(0xffffffffu, p);
        total = __popc(m);
        return __popc(m & ((1u << lane) - 1u));
    }
    // exclusive prefix sum of a per-lane count 0 <= v < 2^bits + total (ordered compaction of several items per lane):
    // one ballot per bit, so counts of 0 / 1 cost what scan_excl costs
    __device__ int scan_excl_sum(int v, int bits, int& total) const {
        int rank = 0;
        total = 0;
        for (int b = 0; b < bits; ++b) {
            const unsigned m = __ballot_sync(0xffffffffu, (v >> b) & 1);
            total += __popc(m) << b;
            rank += __popc(m & ((1u << lane) - 1u)) << b;
        }
        return rank;
    }
    // Warp-wide best key in 3 REDUX ops: min over an order-preserving 64-bit image of the double
    // (hi word, then lo word among the hi-minimal lanes), then max pref among the value-minimal lanes.
    // -0.0 is folded into +0.0 first so that bit equality == IEEE equality (NaN sorts above +inf).
    __device__ DDKey best(DDKey k) const {
        long long b = __double_as_longlong(k.val + 0.0);
        unsigned long long key = (unsigned long long)b ^ ((unsigned long long)(b >> 63) | 0x8000000000000000ull);
        const unsigned hi = (unsigned)(key >> 32), lo = (unsigned)key;
        const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
        const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xffffffffu);
        const bool tie = (hi == mhi) && (lo == mlo);
        const int mp = __reduce_max_sync(0xffffffffu, tie ? k.pref : (int)0x80000000);
        key = ((unsigned long long)mhi << 32) | mlo;
        key = (key & 0x8000000000000000ull) ? (key ^ 0x8000000000000000ull) : ~key;
        DDKey r;
        r.val = __longlong_as_double((long long)key);
        r.pref = mp;
        return r;
    }
    __device__ bool all(bool p) const { return __all_sync(0xffffffffu, p); }
};

// ---------------------------------------------------------------------------------------- SubG<W>
// W adjacent lanes of a warp (W = 8: four independent work items per warp for the small per-track /
// per-detection kernels).  Every collective names only the group's own lanes, so groups of one warp
// may diverge (different item kinds, early exits) without deadlocking each other.
template <int W>
struct SubG {
    static constexpr int NL = W;
    int lane;          // lane within the group
    unsigned mask;     // the group's lanes within the warp
    __device__ explicit SubG() {
        const int wl = threadIdx.x & 31;
        lane = wl & (W - 1);
        mask = ((W == 32) ? 0xffffffffu : ((1u << W) - 1u)) << (wl & ~(W - 1));
    }
    __device__ void sync() const { __syncwarp(mask); }
    __device__ float sum(float v) const {
#pragma unroll
        for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
        return v;
    }
    __device__ unsigned bor(unsigned v) const { return __reduce_or_sync(mask, v); }
    __device__ int imax(int v) const { return __reduce_max_sync(mask, v); }
};

// ---------------------------------------------------------------------------------------- CtaG<NW>
// NW warps of one CTA cooperating on one unit of work (the per-stream matching of crowded scenes, where the
// column scans of the assignment solver are hundreds of entries wide).  Same interface as WarpG; every
// collective is a warp-level step, one shared-memory slot per warp and ONE __syncthreads: the slots are
// double-buffered (a thread can only reach the collective after next once everybody has left this one).
// All threads of the CTA must execute the same sequence of collectives.
template <int NW>
struct CtaG {
    static constexpr int NL = NW * 32;
    int lane;                  // thread index in the CTA
    mutable int phase;         // which half of the scratch the next collective uses
    int* scr_i;                // [2][NW] ints
    double* scr_d;             // [2][NW] doubles
    __device__ CtaG(void* scratch) : lane(threadIdx.x), phase(0) {
        scr_d = (double*)scratch;
        scr_i = (int*)(scr_d + 2 * NW);
    }
    static constexpr int scratch_bytes() { return 2 * NW * 8 + 2 * NW * 4 * 2; }
    __device__ void sync() const { __syncthreads(); }
    __device__ int* slot_i() const { int* p = scr_i + phase * NW; return p; }
    __device__ int imax(int v) const {
        int* sl = slot_i();
        const int w = __reduce_max_sync(0xffffffffu, v);
        if ((lane & 31) == 0) sl[lane >> 5] = w;
        __syncthreads();
        int r = sl[0];
#pragma unroll
        for (int k = 1; k < NW; ++k) r = r > sl[k] ? r : sl[k];
        phase ^= 1;
        return r;
    }
    __device__ int imin(int v) const { return -imax(-v); }
    __device__ bool all(bool p) const { return imax(p ? 0 : 1) == 0; }
    __device__ bool any(bool p) const { return imax(p ? 1 : 0) != 0; }
    __device__ int scan_excl(bool p, int& total) const {
        int* sl = slot_i();
        const unsigned m = __ballot_sync(0xffffffffu, p);
        if ((lane & 31) == 0) sl[lane >> 5] = __popc(m);
        __syncthreads();
        int before = 0, tot = 0;
#pragma unroll
        for (int k = 0; k < NW; ++k) {
            const int c = sl[k];
            before += (k < (lane >> 5)) ? c : 0;
            tot += c;
        }
        phase ^= 1;
        total = tot;
        return before + __popc(m & ((1u << (lane & 31)) - 1u));
    }
    __device__ DDKey best(DDKey k) const {
        WarpG wg;
        const DDKey w = wg.best(k);
        double* sd = scr_d + phase * NW;
        int* si = scr_i + 2 * NW + phase * NW;
        if ((lane & 31) == 0) { sd[lane >> 5] = w.val; si[lane >> 5] = w.pref; }
        __syncthreads();
        DDKey r;
        r.val = sd[0]; r.pref = si[0];
#pragma unroll
        for (int q = 1; q < NW; ++q) {
            DDKey c;
            c.val = sd[q]; c.pref = si[q];
            if (dd_key_better(c, r)) r = c;
        }
        phase ^= 1;
        return r;
    }
};

// ---------------------------------------------------------------------------------------- BlockG
// Whole CTA; collectives go through a small shared-memory scratch supplied by the kernel.
struct BlockG {
    int lane;      // thread index in the CTA
    int nl;        // blockDim.x
    __device__ explicit BlockG() : lane(threadIdx.x), nl(blockDim.x) {}
    __device__ void sync() const { __syncthreads(); }
};
#endif

// ---------------------------------------------------------------------------------------- HostG
struct HostG {
    static constexpr int NL = 1;
    int lane = 0;
    int nl = 1;
    void sync() const {}
    float sum(float v) const { return v; }
    double sum(double v) const { return v; }
    int sum(int v) const { return v; }
    int imax(int v) const { return v; }
    int imin(int v) const { return v; }
    float fmax(float v) const { return v; }
    unsigned bor(unsigned v) const { return v; }
    bool any(bool p) const { return p; }
    bool all(bool p) const { return p; }
    int scan_excl(bool p, int& total) const { total = p ? 1 : 0; return 0; }
    int scan_excl_sum(int v, int, int& total) const { total = v; return 0; }
    DDKey best(DDKey k) const { return k; }
};
