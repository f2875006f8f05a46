// Analyses on the trace hot path (analyses.py:16-30,60-97,118-133) and order-preserving
// vignetting compaction (transformations.py:214-225).  All kernels are HBM-streaming:
// persistent grids, double2 loads, warp-shuffle + shared-memory block reductions, a
// fixed-shape two-level tree (deterministic, no floating-point atomics).
#include "pxf_internal.h"
#include "pxf_ray.cuh"

namespace pxf {

#define NSUM 9
#define SUM_BLOCKS_MAX 2048   // >= SM count x resident CTAs

// ------------------------------------------------------------------ sums
template <int MODE>
PXF_DEV void sums_accum(double acc[NSUM], double x, double y, double l, double m, double n, double w,
                        bool has_w, double a, double b, double z = 0., double c = 0.)
{
    if (MODE == PXF_SUMS_CENTROID) {
        acc[0] += w;
        acc[1] += has_w ? x * w : x;
        acc[2] += has_w ? y * w : y;
        acc[3] += 1.;
    } else if (MODE == PXF_SUMS_RMS) {
        double rho = sq(x - a) + sq(y - b);
        acc[0] += w;
        acc[1] += has_w ? rho * w : rho;
    } else if (MODE == PXF_SUMS_POINT) {
        // analyses.py:33-45: (x-px)**2 + (y-py)**2 + (z-pz)**2
        double rho = sq(x - a) + sq(y - b) + sq(z - c);
        acc[0] += w;
        acc[1] += has_w ? rho * w : rho;
    } else {
        double ln = l / n, mn = m / n;
        if (MODE == PXF_SUMS_IMAGEPLANE_Z) {
            // where the ray crosses z = 0: the literal plane scan (move the plane by dz, trace to it) propagates a
            // ray by (dz - z)/n, so in terms of (x0, y0) its footprint at offset dz is (x0 + dz l/n, y0 + dz m/n)
            x = x - ln * z;
            y = y - mn * z;
        }
        double t1 = x * l / n, t2 = y * m / n, t3 = sq(ln), t4 = sq(mn);
        acc[0] += w;
        acc[1] += has_w ? x * w : x;
        acc[2] += has_w ? y * w : y;
        acc[3] += has_w ? ln * w : ln;
        acc[4] += has_w ? mn * w : mn;
        acc[5] += has_w ? t1 * w : t1;
        acc[6] += has_w ? t2 * w : t2;
        acc[7] += has_w ? t3 * w : t3;
        acc[8] += has_w ? t4 * w : t4;
    }
}

// One pass, HBM bound: each thread keeps U independent accumulator sets (a single fp64 add chain per
// quantity would be latency bound: 8 cycles per element) fed by U batched 16-byte loads per row, and
// folds them in a fixed order at the end -- same bits on every run and for every grid of the same
// size (the grid is a function of num only).
template <int MODE, bool VEC2>
__global__ void __launch_bounds__(PXF_BLOCK)
k_sums(const double *__restrict__ x, const double *__restrict__ y, const double *__restrict__ l,
       const double *__restrict__ m, const double *__restrict__ n, const double *__restrict__ w,
       int64_t num, double a, double b, const double *__restrict__ ab_dev, double *__restrict__ partial,
       const double *__restrict__ z = nullptr, double c = 0.)
{
    constexpr int NS = MODE == PXF_SUMS_CENTROID ? 4 : ((MODE == PXF_SUMS_RMS || MODE == PXF_SUMS_POINT) ? 2 : 9);
    constexpr bool IP = MODE == PXF_SUMS_IMAGEPLANE || MODE == PXF_SUMS_IMAGEPLANE_Z;
    constexpr bool ZZ = MODE == PXF_SUMS_IMAGEPLANE_Z || MODE == PXF_SUMS_POINT;
    constexpr int U = IP ? 2 : 4;
    if (ab_dev) { a = ab_dev[0]; b = ab_dev[1]; }
    double acc[U][NSUM];
#pragma unroll
    for (int u = 0; u < U; u++)
#pragma unroll
        for (int k = 0; k < NSUM; k++) acc[u][k] = 0.;
    const bool has_w = w != nullptr;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    if (VEC2) {
        const int64_t npair = num >> 1;
        for (int64_t q0 = tid; q0 < npair; q0 += U * nthr) {
            double2 xv[U], yv[U], lv[U], mv[U], nv[U], wv[U], zv[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const int64_t q = q0 + u * nthr;
                const bool in = q < npair;
                const double2 z2 = make_double2(0., 0.), o2 = make_double2(1., 1.);
                xv[u] = in ? *reinterpret_cast<const double2 *>(x + 2 * q) : z2;
                yv[u] = in ? *reinterpret_cast<const double2 *>(y + 2 * q) : z2;
                if (IP) {
                    lv[u] = in ? *reinterpret_cast<const double2 *>(l + 2 * q) : z2;
                    mv[u] = in ? *reinterpret_cast<const double2 *>(m + 2 * q) : z2;
                    nv[u] = in ? *reinterpret_cast<const double2 *>(n + 2 * q) : o2;
                } else { lv[u] = z2; mv[u] = z2; nv[u] = o2; }
                zv[u] = (ZZ && in) ? *reinterpret_cast<const double2 *>(z + 2 * q) : z2;
                wv[u] = (in && has_w) ? *reinterpret_cast<const double2 *>(w + 2 * q) : o2;
            }
#pragma unroll
            for (int u = 0; u < U; u++)
                if (q0 + u * nthr < npair) {
                    sums_accum<MODE>(acc[u], xv[u].x, yv[u].x, lv[u].x, mv[u].x, nv[u].x, wv[u].x, has_w, a, b, zv[u].x, c);
                    sums_accum<MODE>(acc[u], xv[u].y, yv[u].y, lv[u].y, mv[u].y, nv[u].y, wv[u].y, has_w, a, b, zv[u].y, c);
                }
        }
        if ((num & 1) && tid == 0) {
            const int64_t i = num - 1;
            sums_accum<MODE>(acc[0], x[i], y[i], IP ? l[i] : 0., IP ? m[i] : 0.,
                             IP ? n[i] : 1., has_w ? w[i] : 1., has_w, a, b, ZZ ? z[i] : 0., c);
        }
    } else {
        for (int64_t i0 = tid; i0 < num; i0 += U * nthr) {
            double xv[U], yv[U], lv[U], mv[U], nv[U], wv[U], zv[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const int64_t i = i0 + u * nthr;
                const bool in = i < num;
                xv[u] = in ? x[i] : 0.;
                yv[u] = in ? y[i] : 0.;
                lv[u] = (in && IP) ? l[i] : 0.;
                mv[u] = (in && IP) ? m[i] : 0.;
                nv[u] = (in && IP) ? n[i] : 1.;
                zv[u] = (in && ZZ) ? z[i] : 0.;
                wv[u] = (in && has_w) ? w[i] : 1.;
            }
#pragma unroll
            for (int u = 0; u < U; u++)
                if (i0 + u * nthr < num) sums_accum<MODE>(acc[u], xv[u], yv[u], lv[u], mv[u], nv[u], wv[u], has_w, a, b, zv[u], c);
        }
    }
#pragma unroll
    for (int k = 0; k < NS; k++) {
        double t = acc[0][k];
#pragma unroll
        for (int u = 1; u < U; u++) t += acc[u][k];
        acc[0][k] = t;
    }
    __shared__ double sh[NSUM][PXF_BLOCK / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NS; k++) {
        double v = acc[0][k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) sh[k][warp] = v;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < NS; k++) {
            double v = lane < PXF_BLOCK / 32 ? sh[k][lane] : 0.;
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) partial[(int64_t)blockIdx.x * NSUM + k] = v;
        }
    }
}

__global__ void __launch_bounds__(PXF_BLOCK)
k_sums_final(const double *__restrict__ partial, int nblocks, int ns, double *__restrict__ out)
{
    __shared__ double sh[PXF_BLOCK / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = 0; k < ns; k++) {
        double v = 0.;
        for (int b = threadIdx.x; b < nblocks; b += blockDim.x) v += partial[(int64_t)b * NSUM + k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) sh[warp] = v;
        __syncthreads();
        if (warp == 0) {
            v = lane < PXF_BLOCK / 32 ? sh[lane] : 0.;
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) out[k] = v;
        }
        __syncthreads();
    }
}

static int sums_launch(int mode, const double *x, const double *y, const double *l, const double *m,
                       const double *n, const double *w, int64_t num, double a, double b,
                       const double *ab_dev, double *out_dev, void *scratch, cudaStream_t s, const double *z = nullptr,
                       double c = 0.)
{
    if (num < 0 || !x || !y || !out_dev || !scratch) { set_error("pxf_sums: bad argument"); return PXF_ERR_INVALID; }
    const bool ip = mode == PXF_SUMS_IMAGEPLANE || mode == PXF_SUMS_IMAGEPLANE_Z;
    if (ip && (!l || !m || !n)) { set_error("pxf_sums: l,m,n required"); return PXF_ERR_INVALID; }
    if ((mode == PXF_SUMS_IMAGEPLANE_Z || mode == PXF_SUMS_POINT) && !z) { set_error("pxf_sums: z required"); return PXF_ERR_INVALID; }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    int grid = grid_for(num, PXF_BLOCK * 8, 4);
    if (grid > SUM_BLOCKS_MAX) grid = SUM_BLOCKS_MAX;
    double *partial = static_cast<double *>(scratch);
    uintptr_t al = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(w);
    if (mode == PXF_SUMS_POINT) al |= reinterpret_cast<uintptr_t>(z);
    if (ip)
        al |= reinterpret_cast<uintptr_t>(l) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(n) |
              reinterpret_cast<uintptr_t>(z);
    const bool v2 = (al & 15) == 0;
    int ns;
#define PXF_SUMS_GO(M)                                                                                         \
    do {                                                                                                       \
        if (v2) k_sums<M, true><<<grid, PXF_BLOCK, 0, s>>>(x, y, l, m, n, w, num, a, b, ab_dev, partial, z, c);  \
        else k_sums<M, false><<<grid, PXF_BLOCK, 0, s>>>(x, y, l, m, n, w, num, a, b, ab_dev, partial, z, c);    \
    } while (0)
    if (mode == PXF_SUMS_CENTROID) { ns = 4; PXF_SUMS_GO(PXF_SUMS_CENTROID); }
    else if (mode == PXF_SUMS_RMS) { ns = 2; PXF_SUMS_GO(PXF_SUMS_RMS); }
    else if (mode == PXF_SUMS_IMAGEPLANE) { ns = 9; PXF_SUMS_GO(PXF_SUMS_IMAGEPLANE); }
    else if (mode == PXF_SUMS_IMAGEPLANE_Z) { ns = 9; PXF_SUMS_GO(PXF_SUMS_IMAGEPLANE_Z); }
    else if (mode == PXF_SUMS_POINT) { ns = 2; PXF_SUMS_GO(PXF_SUMS_POINT); }
    else {
        set_error("pxf_sums: bad mode");
        return PXF_ERR_INVALID;
    }
#undef PXF_SUMS_GO
    k_sums_final<<<1, PXF_BLOCK, 0, s>>>(partial, grid, ns, out_dev);
    count_launch(2);
    return check_launch("k_sums");
}

int sums_finalize(const double *partial, int nblocks, int ns, double *out_dev, cudaStream_t s)
{
    if (nblocks > SUM_BLOCKS_MAX) { set_error("sums_finalize: too many partials"); return PXF_ERR_INVALID; }
    k_sums_final<<<1, PXF_BLOCK, 0, s>>>(partial, nblocks, ns, out_dev);
    count_launch();
    return check_launch("k_sums_final");
}

// cxy[0] = S1/S0, cxy[1] = S2/S0 (np.average: sum(w*x)/sum(w); unweighted: sum(x)/N)
__global__ void k_centroid_from_sums(const double *__restrict__ sums, double *__restrict__ cxy)
{
    cxy[0] = sums[1] / sums[0];
    cxy[1] = sums[2] / sums[0];
}

// ------------------------------------------------------------------ rho
__global__ void __launch_bounds__(PXF_BLOCK)
k_rho(const double *__restrict__ x, const double *__restrict__ y, int64_t num, double cx, double cy,
      const double *__restrict__ cxy_dev, double *__restrict__ out)
{
    if (cxy_dev) { cx = cxy_dev[0]; cy = cxy_dev[1]; }
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < num; i += nthr) out[i] = sqrt(sq(x[i] - cx) + sq(y[i] - cy));
}

// ------------------------------------------------------------------ exact radix select
// Device-resident state so that no pass needs a host round trip.
struct SelectState {
    unsigned long long prefix[2];   // resolved high bits of each chain (right aligned)
    unsigned long long rank[2];     // 0-based rank still to resolve inside the prefix group
    int nprefix;                    // 1 while both order statistics share a prefix, else 2
    int valid;                      // 0 when a bracketed select missed its bracket (caller falls back)
};

PXF_DEV unsigned long long key_of(double r) { return (unsigned long long)__double_as_longlong(r); }


// Warp-aggregated shared-memory histogram update (bin < 0: nothing to add; every lane of the warp must call).
// The early select passes see almost every key in ONE bin: the lanes that share lane 0's bin are counted by a ballot and
// added once, the rest add themselves.  (__match_any_sync would aggregate every bin, but it runs at a few hundred
// cycles per warp on this part -- it bounded this kernel at 2.4 TB/s, profiles/r02_notes.md.)
PXF_DEV void hist_add_warp(unsigned int *sh, int bin)
{
    const int b0 = __shfl_sync(0xffffffffu, bin, 0);
    const unsigned same = __ballot_sync(0xffffffffu, bin == b0);
    if (bin == b0) {
        if ((threadIdx.x & 31) == 0 && bin >= 0) atomicAdd(&sh[bin], (unsigned)__popc(same));
    } else if (bin >= 0) {
        atomicAdd(&sh[bin], 1u);
    }
}

template <bool FROM_KEYS>
__global__ void __launch_bounds__(PXF_BLOCK)
k_select_hist(const double *__restrict__ x, const double *__restrict__ y, const double *__restrict__ keys,
              int64_t num, const unsigned long long *__restrict__ count_dev,
              const double *__restrict__ cxy, int shift, int bits,
              const SelectState *__restrict__ st, unsigned long long *__restrict__ hist,
              unsigned long long *__restrict__ nan_count)
{
    extern __shared__ unsigned int sh[];
    const int nbins = 1 << bits;
    const int np = st->nprefix;
    const unsigned long long p0 = st->prefix[0], p1 = st->prefix[1];
    const int hi = shift + bits;
    for (int t = threadIdx.x; t < np * nbins; t += blockDim.x) sh[t] = 0;
    __syncthreads();
    double cx = 0., cy = 0.;
    if (!FROM_KEYS) { cx = cxy[0]; cy = cxy[1]; }
    if (FROM_KEYS && count_dev) {
        unsigned long long c = *count_dev;
        if ((unsigned long long)num > c) num = (int64_t)c;
    }
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    unsigned int nans = 0;
    // whole warps iterate together so that __match_any_sync sees a full mask
    const int64_t nround = (num + nthr - 1) / nthr;
    for (int64_t it = 0; it < nround; it++) {
        const int64_t i = tid + it * nthr;
        int bin = -1;
        if (i < num) {
            double r = FROM_KEYS ? keys[i] : sqrt(sq(x[i] - cx) + sq(y[i] - cy));
            if (r != r) {
                nans++;
            } else {
                unsigned long long k = key_of(r);
                unsigned long long top = hi >= 64 ? 0ull : (k >> hi);
                int d = (int)((k >> shift) & (unsigned long long)(nbins - 1));
                if (top == p0) bin = d;
                else if (np == 2 && top == p1) bin = nbins + d;
            }
        }
        hist_add_warp(sh, bin);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < np * nbins; t += blockDim.x) {
        unsigned int v = sh[t];
        if (v) atomicAdd(&hist[t], (unsigned long long)v);
    }
    if (nan_count) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) nans += __shfl_down_sync(0xffffffffu, nans, o);
        if ((threadIdx.x & 31) == 0 && nans) atomicAdd(nan_count, (unsigned long long)nans);
    }
}

// One CTA walks the (all-reduced) histogram and narrows each chain by `bits` bits.
__global__ void __launch_bounds__(1024)
k_select_scan(unsigned long long *__restrict__ hist, int bits, SelectState *__restrict__ st)
{
    __shared__ unsigned long long wsum[32];
    __shared__ int found_bin[2];
    __shared__ unsigned long long found_base[2];
    const int nbins = 1 << bits;
    const int np = st->nprefix;
    const int per = (nbins + blockDim.x - 1) / blockDim.x;
    if (threadIdx.x < 2) { found_bin[threadIdx.x] = 0; found_base[threadIdx.x] = 0ull; }
    __syncthreads();
    for (int j = 0; j < 2; j++) {
        const int hsel = (np == 2) ? j : 0;
        const unsigned long long *h = hist + (size_t)hsel * nbins;
        const unsigned long long rank = st->rank[j];
        // block-wide exclusive scan over contiguous chunks of `per` bins per thread
        const int b0 = threadIdx.x * per;
        unsigned long long local = 0;
        for (int b = b0; b < b0 + per && b < nbins; b++) local += h[b];
        unsigned long long incl = local;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            unsigned long long v = lane < (int)(blockDim.x >> 5) ? wsum[lane] : 0ull;
            unsigned long long iv = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                unsigned long long t = __shfl_up_sync(0xffffffffu, iv, o);
                if (lane >= o) iv += t;
            }
            wsum[lane] = iv - v;
        }
        __syncthreads();
        unsigned long long excl = wsum[warp] + incl - local;
        if (rank >= excl && rank < excl + local) {
            unsigned long long c = excl;
            for (int b = b0; b < b0 + per && b < nbins; b++) {
                unsigned long long hb = h[b];
                if (rank < c + hb) { found_bin[j] = b; found_base[j] = c; break; }
                c += hb;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        unsigned long long pa = st->prefix[0], pb = (np == 2) ? st->prefix[1] : st->prefix[0];
        st->prefix[0] = (pa << bits) | (unsigned long long)found_bin[0];
        st->prefix[1] = (pb << bits) | (unsigned long long)found_bin[1];
        st->rank[0] -= found_base[0];
        st->rank[1] -= found_base[1];
        st->nprefix = (st->prefix[0] == st->prefix[1]) ? 1 : 2;
    }
    __syncthreads();
    // zero the histogram for the next pass
    for (int t = threadIdx.x; t < 2 * nbins; t += blockDim.x) hist[t] = 0ull;
}

__global__ void k_select_init(SelectState *st, unsigned long long k0, unsigned long long k1,
                              unsigned long long *hist, int nh, unsigned long long *nan_count)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        st->prefix[0] = 0; st->prefix[1] = 0; st->rank[0] = k0; st->rank[1] = k1; st->nprefix = 1; st->valid = 1;
        if (nan_count) *nan_count = 0;
    }
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nh; t += gridDim.x * blockDim.x) hist[t] = 0ull;
}

// out[0] = 2*median (np.median(r)*2., analyses.py:96); out[1], out[2] = the two middle order statistics
__global__ void k_select_result(const SelectState *st, const unsigned long long *nan_count, int64_t num,
                                double *out)
{
    double a = __longlong_as_double((long long)st->prefix[0]);
    double b = __longlong_as_double((long long)st->prefix[1]);
    double med = (a + b) / 2.;
    if (num == 0 || (nan_count && *nan_count > 0)) med = __longlong_as_double(0x7ff8000000000000ll);
    out[0] = med * 2.;
    out[1] = a;
    out[2] = b;
    out[3] = st->valid ? 1. : 0.;
}

// ------------------------------------------------------------------ bracketed select
// np.median over 1e8 radii does not need five full passes: a strided sample of S radii gives
// (by an exact select on the sample) a bracket [lo,hi] that holds the two middle order
// statistics with overwhelming probability; ONE pass over the bundle then counts the radii
// below lo and collects the few per cent inside the bracket, and the exact select finishes on
// that small buffer.  If the bracket misses (or the candidate buffer overflows) the state is
// flagged invalid and the caller reruns the full five-pass select -- the result is exact
// either way.
#define BRACKET_SAMPLES 65536
#define BRACKET_MIN_NUM (int64_t(1) << 21)

__global__ void __launch_bounds__(PXF_BLOCK)
k_select_sample(const double *__restrict__ x, const double *__restrict__ y, int64_t num,
                const double *__restrict__ cxy, int nsamp, double *__restrict__ keys)
{
    const double cx = cxy[0], cy = cxy[1];
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < nsamp; j += gridDim.x * blockDim.x) {
        const int64_t i = (int64_t)(((unsigned long long)j * (unsigned long long)num) / (unsigned long long)nsamp);
        keys[j] = sqrt(sq(x[i] - cx) + sq(y[i] - cy));
    }
}

// counters: [0] #(r < lo), [1] #(lo <= r <= hi) (may exceed cap), [2] #NaN, [3] #shards whose buffer overflowed
// HBM-streaming pass (16 B/ray).  Each thread issues COLLECT_U independent 16-byte load pairs
// before touching any of them (memory-level parallelism).  The few per cent of radii inside the
// bracket are appended to a per-CTA shared-memory buffer (shared-memory atomics) that is
// flushed to the global candidate buffer with ONE global atomic per flush: appending through a
// single global counter directly serialises at L2 (measured 1.2 TB/s instead of ~5).
#define COLLECT_U 4
#define COLLECT_SCAP 4096     // shared staging capacity (doubles); a batch adds at most 2048
template <bool VEC2>
__global__ void __launch_bounds__(PXF_BLOCK)
k_bracket_collect(const double *__restrict__ x, const double *__restrict__ y, int64_t num,
                  const double *__restrict__ cxy, const double *__restrict__ lohi,
                  double *__restrict__ cand, unsigned long long cap, unsigned long long *__restrict__ counters)
{
    __shared__ double sbuf[COLLECT_SCAP];
    __shared__ unsigned int scount;
    __shared__ unsigned long long sbase;
    const double cx = cxy[0], cy = cxy[1];
    const double lo = lohi[1], hi = lohi[2];
    const int lane = threadIdx.x & 31;
    unsigned int below = 0, nans = 0;
    constexpr int PER = VEC2 ? 2 : 1;
    constexpr int NE = COLLECT_U * PER;
    static_assert(NE * PXF_BLOCK <= COLLECT_SCAP / 2, "staging buffer too small for one batch");
    const int64_t items = VEC2 ? (num >> 1) : num;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * COLLECT_U;
    if (threadIdx.x == 0) scount = 0;
    __syncthreads();
    auto flush = [&]() {                 // block-uniform
        if (threadIdx.x == 0) sbase = atomicAdd(&counters[1], (unsigned long long)scount);
        __syncthreads();
        const unsigned int n = scount;
        for (unsigned int t = threadIdx.x; t < n; t += blockDim.x) {
            const unsigned long long dst = sbase + t;
            if (dst < cap) cand[dst] = sbuf[t];
        }
        __syncthreads();
        if (threadIdx.x == 0) scount = 0;
        __syncthreads();
    };
    // block-uniform trip count
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x * COLLECT_U; base < items; base += stride) {
        double r[NE];
        if (VEC2) {
            double2 xv[COLLECT_U], yv[COLLECT_U];
#pragma unroll
            for (int u = 0; u < COLLECT_U; u++) {
                const int64_t q = base + (int64_t)u * blockDim.x + threadIdx.x;
                if (q < items) {
                    xv[u] = *reinterpret_cast<const double2 *>(x + 2 * q);
                    yv[u] = *reinterpret_cast<const double2 *>(y + 2 * q);
                } else {
                    xv[u] = make_double2(0., 0.); yv[u] = make_double2(0., 0.);
                }
            }
#pragma unroll
            for (int u = 0; u < COLLECT_U; u++) {
                r[2 * u] = sqrt(sq(xv[u].x - cx) + sq(yv[u].x - cy));
                r[2 * u + (PER - 1)] = sqrt(sq(xv[u].y - cx) + sq(yv[u].y - cy));
            }
        } else {
            double xv[COLLECT_U], yv[COLLECT_U];
#pragma unroll
            for (int u = 0; u < COLLECT_U; u++) {
                const int64_t q = base + (int64_t)u * blockDim.x + threadIdx.x;
                xv[u] = q < items ? x[q] : 0.;
                yv[u] = q < items ? y[q] : 0.;
            }
#pragma unroll
            for (int u = 0; u < COLLECT_U; u++) r[u * PER] = sqrt(sq(xv[u] - cx) + sq(yv[u] - cy));
        }
#pragma unroll
        for (int e = 0; e < NE; e++) {
            const int64_t q = base + (int64_t)(e / PER) * blockDim.x + threadIdx.x;
            if (q < items) {
                if (r[e] != r[e]) nans++;
                else if (r[e] < lo) below++;
                else if (r[e] <= hi) sbuf[atomicAdd(&scount, 1u)] = r[e];
            }
        }
        __syncthreads();
        if (scount > COLLECT_SCAP / 2) flush();
    }
    if (VEC2 && (num & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
        const double rr = sqrt(sq(x[num - 1] - cx) + sq(y[num - 1] - cy));
        if (rr != rr) nans++;
        else if (rr < lo) below++;
        else if (rr <= hi) sbuf[atomicAdd(&scount, 1u)] = rr;
    }
    __syncthreads();
    if (scount > 0) flush();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        below += __shfl_down_sync(0xffffffffu, below, o);
        nans += __shfl_down_sync(0xffffffffu, nans, o);
    }
    if (lane == 0) {
        if (below) atomicAdd(&counters[0], (unsigned long long)below);
        if (nans) atomicAdd(&counters[2], (unsigned long long)nans);
    }
}

// ranks inside the candidate buffer = global ranks - #below; flags the state invalid when the
// bracket does not contain both ranks or the buffer overflowed.  counters are the (possibly
// all-reduced) totals.
__global__ void k_select_begin_bracket(SelectState *st, unsigned long long k0, unsigned long long k1,
                                       const unsigned long long *__restrict__ counters, unsigned long long cap_total,
                                       unsigned long long *hist, int nh, unsigned long long *nan_count)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const unsigned long long below = counters[0], ncand = counters[1];
        if (cap_total == ~0ull) cap_total = counters[4];       // summed capacities travel with the counters
        const bool ok = counters[3] == 0 && ncand <= cap_total && k0 >= below && k1 < below + ncand;
        st->prefix[0] = 0; st->prefix[1] = 0;
        st->rank[0] = ok ? k0 - below : 0; st->rank[1] = ok ? k1 - below : 0;
        st->nprefix = 1; st->valid = ok ? 1 : 0;
        if (nan_count) *nan_count = counters[2];
    }
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nh; t += gridDim.x * blockDim.x) hist[t] = 0ull;
}

// ------------------------------------------------------------------ single-GPU fast path
// The pass-wise select above is built for the multi-GPU driver (a histogram all-reduce between
// passes) and costs 11 launches of ~10 us for each of its two small selects.  On one GPU the
// same result comes from four launches around the one big pass:
//   k_select_sample_sums   centroid from the sums + strided sample of radii        (multi-CTA)
//   k_bracket_small        ONE CTA: three 13-bit radix passes over the 64 Ki sample keys with
//                          shared-memory histograms -> bracket [lo,hi] (the sample order statistics
//                          ra, rb rounded outwards to 39-bit prefixes); zeroes the counters
//   k_bracket_collect      the HBM pass (unchanged)
//   k_cand_hist            candidates -> 4096 LINEAR bins over [lo,hi] (monotone, so bin order is
//                          value order); the last CTA to finish scans the bins and picks the one or
//                          two bins holding the middle ranks
//   k_cand_finish          collects the few hundred keys of those bins; the last CTA sorts them in
//                          shared memory and writes {2*median, lower, upper, valid}
// Exact: every step either narrows by a monotone map or sorts; anything unexpected (bracket miss,
// buffer overflow, ties piling into one bin) clears `valid` and the caller reruns the five-pass
// select.
#define FAST_NBINS 4096
#define FAST_FINCAP 4096
struct FastSel {
    unsigned int ticket_hist, ticket_fin;
    unsigned int bin_a, bin_b;
    unsigned long long base_a;       // candidates in bins below bin_a
    unsigned long long r0, r1;       // ranks of the two middle order statistics among the candidates
    unsigned int nfin;
    int valid;
    int is_nan;
    int pad;
};

__global__ void __launch_bounds__(PXF_BLOCK)
k_select_sample_sums(const double *__restrict__ x, const double *__restrict__ y, int64_t num,
                     const double *__restrict__ sums, double *__restrict__ cxy, int nsamp, double *__restrict__ keys)
{
    // same arithmetic as k_centroid_from_sums; every thread computes it, thread 0 publishes it
    const double cx = sums[1] / sums[0], cy = sums[2] / sums[0];
    if (blockIdx.x == 0 && threadIdx.x == 0) { cxy[0] = cx; cxy[1] = cy; }
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < nsamp; j += gridDim.x * blockDim.x) {
        const int64_t i = (int64_t)(((unsigned long long)j * (unsigned long long)num) / (unsigned long long)nsamp);
        keys[j] = sqrt(sq(x[i] - cx) + sq(y[i] - cy));
    }
}

// block-wide: find the bin holding 0-based rank `rank` in the nbins-entry shared histogram h
// (nbins <= 8 * blockDim.x).  Returns through found[0] = bin, found[1] = count below the bin
// (both untouched when rank >= total).  All threads must call.
PXF_DEV void block_find_bin(const unsigned int *h, int nbins, unsigned long long rank, unsigned long long *wsum,
                            unsigned long long *found)
{
    const int per = (nbins + blockDim.x - 1) / blockDim.x;
    const int b0 = threadIdx.x * per;
    unsigned long long local = 0;
    for (int b = b0; b < b0 + per && b < nbins; b++) local += h[b];
    unsigned long long incl = local;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned long long v = lane < (int)(blockDim.x >> 5) ? wsum[lane] : 0ull;
        unsigned long long iv = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, iv, o);
            if (lane >= o) iv += t;
        }
        wsum[lane] = iv - v;
    }
    __syncthreads();
    const unsigned long long excl = wsum[warp] + incl - local;
    if (rank >= excl && rank < excl + local) {
        unsigned long long c = excl;
        for (int b = b0; b < b0 + per && b < nbins; b++) {
            const unsigned long long hb = h[b];
            if (rank < c + hb) { found[0] = (unsigned long long)b; found[1] = c; break; }
            c += hb;
        }
    }
    __syncthreads();
}

// ONE-CTA radix select of two order statistics of a small key set (<= ~1e6 keys, L2 resident):
// npass = 3 resolves 39 bits and rounds the pair outwards over the other 25 (a bracket), npass = 5
// resolves all 64 (the exact values).  The keys are nseg segments of seg_cap doubles of which the
// first seg_counts[s] are valid (seg_counts == NULL: all of them) -- the layout an all-gather of
// per-rank buffers produces.  ranks: (ra, rb), or taken from a FastSel (r0-base_a, r1-base_a) when
// `fs` is given, in which case its valid / is_nan flags and any overflowed segment decide the
// outcome first.  out = {a+b, a, b, valid}.  `hk_*` (nullable): buffers of the single-GPU pipeline
// that this launch also resets.
__global__ void __launch_bounds__(1024)
k_small_select(const double *__restrict__ keys, const int *__restrict__ seg_counts, int nseg, int seg_cap,
               unsigned long long ra, unsigned long long rb, int npass, const FastSel *__restrict__ fs,
               double *__restrict__ out, unsigned long long *__restrict__ hk_counters,
               FastSel *__restrict__ hk_fs, unsigned int *__restrict__ hk_fhist)
{
    extern __shared__ unsigned int sh[];                // [2][8192]
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long found[2][2];
    __shared__ unsigned long long prefix[2], rank[2];
    __shared__ int np, verdict;                         // verdict: 0 run, 1 invalid, 2 NaN
    const int NB = 8192;
    if (hk_fhist) for (int t = threadIdx.x; t < FAST_NBINS; t += blockDim.x) hk_fhist[t] = 0u;
    if (hk_counters && threadIdx.x < 8) hk_counters[threadIdx.x] = 0ull;
    if (threadIdx.x == 0) {
        if (hk_fs) { hk_fs->ticket_hist = 0; hk_fs->ticket_fin = 0; hk_fs->nfin = 0; hk_fs->valid = 0; hk_fs->is_nan = 0; }
        int v = 0;
        if (fs) {
            ra = fs->r0 - fs->base_a; rb = fs->r1 - fs->base_a;
            if (fs->is_nan) v = 2;
            else if (!fs->valid) v = 1;
        }
        unsigned long long have = 0;
        for (int sgm = 0; sgm < nseg; sgm++) {
            const int c = seg_counts ? seg_counts[sgm] : seg_cap;
            if (c > seg_cap && v == 0) v = 1;            // a rank's buffer overflowed
            have += (unsigned long long)(c < seg_cap ? c : seg_cap);
        }
        if (v == 0 && rb >= have) v = 1;
        verdict = v;
        prefix[0] = prefix[1] = 0ull; rank[0] = ra; rank[1] = rb; np = 1;
    }
    __syncthreads();
    if (verdict != 0) {
        if (threadIdx.x == 0) {
            const double nanv = __longlong_as_double(0x7ff8000000000000ll);
            const bool isn = verdict == 2;
            out[0] = isn ? nanv : 0.; out[1] = isn ? nanv : 0.; out[2] = isn ? nanv : 0.; out[3] = isn ? 1. : 0.;
        }
        return;
    }
    const int total = nseg * seg_cap;
    const int shifts[5] = {51, 38, 25, 12, 0};
    const int nbits[5] = {13, 13, 13, 13, 12};
    for (int pass = 0; pass < npass; pass++) {
        const int shift = shifts[pass], bits = nbits[pass], hi = shift + bits;
        const int nb = 1 << bits;
        const int npl = np;
        const unsigned long long p0 = prefix[0], p1 = prefix[1];
        for (int t = threadIdx.x; t < 2 * NB; t += blockDim.x) sh[t] = 0u;
        if (threadIdx.x < 2) { found[threadIdx.x][0] = 0ull; found[threadIdx.x][1] = 0ull; }
        __syncthreads();
        // warp-aggregated (the first pass sees almost every key in the same one or two bins); loads
        // issued eight at a time so the single CTA is not bound by one L2 latency per key
        for (int j0 = 0; j0 < total; j0 += 8 * blockDim.x) {
            double rv[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int j = j0 + u * blockDim.x + threadIdx.x;
                bool ok = j < total;
                if (ok && seg_counts) ok = (j % seg_cap) < seg_counts[j / seg_cap];
                rv[u] = ok ? keys[j] : __longlong_as_double(0x7ff8000000000000ll);
            }
#pragma unroll
            for (int u = 0; u < 8; u++) {
                int bin = -1;
                const double r = rv[u];
                if (r == r) {
                    const unsigned long long k = key_of(r);
                    const unsigned long long top = hi >= 64 ? 0ull : (k >> hi);
                    const int d = (int)((k >> shift) & (unsigned long long)(nb - 1));
                    if (top == p0) bin = d;
                    else if (npl == 2 && top == p1) bin = NB + d;
                }
                hist_add_warp(sh, bin);
            }
        }
        __syncthreads();
        for (int j = 0; j < 2; j++)
            block_find_bin(sh + ((npl == 2) ? j : 0) * NB, nb, rank[j], wsum, found[j]);
        if (threadIdx.x == 0) {
            const unsigned long long pa = prefix[0], pb = (npl == 2) ? prefix[1] : prefix[0];
            prefix[0] = (pa << bits) | found[0][0];
            prefix[1] = (pb << bits) | found[1][0];
            rank[0] -= found[0][1];
            rank[1] -= found[1][1];
            np = (prefix[0] == prefix[1]) ? 1 : 2;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // unresolved low bits (25 after three passes, none after five): round the pair outwards
        const int rem = npass >= 5 ? 0 : 64 - 13 * npass;
        const unsigned long long ones = rem ? ((1ull << rem) - 1ull) : 0ull;
        const double a = __longlong_as_double((long long)(rem ? (prefix[0] << rem) : prefix[0]));
        const double b = __longlong_as_double((long long)(rem ? ((prefix[1] << rem) | ones) : prefix[1]));
        out[0] = ((a + b) / 2.) * 2.;
        out[1] = a; out[2] = b; out[3] = 1.;
    }
}

PXF_DEV int cand_bin(double r, double lo, double scale)
{
    const double t = (r - lo) * scale;          // monotone in r; NaN (hi == lo) -> bin 0
    int b = t > 0. ? (t < (double)FAST_NBINS ? (int)t : FAST_NBINS - 1) : 0;
    return b;
}
PXF_DEV double cand_scale(double lo, double hi)
{
    const double w = hi - lo;
    return w > 0. ? (double)FAST_NBINS / w : 0.;
}

// validity of the bracket + the bin(s) holding the two middle ranks; h = the (global) histogram in
// shared memory.  All threads of the CTA call.  cap_total == ~0: the summed capacities travel in
// counters[4] (multi-GPU).
PXF_DEV void cand_scan_block(const unsigned int *h, const unsigned long long *__restrict__ counters,
                             unsigned long long cap_total, unsigned long long k0, unsigned long long k1,
                             FastSel *__restrict__ fs, unsigned long long *wsum, unsigned long long (*found)[2])
{
    const unsigned long long below = counters[0], ncand = counters[1], nnan = counters[2];
    if (cap_total == ~0ull) cap_total = counters[4];
    const bool ok = nnan == 0 && counters[3] == 0 && ncand <= cap_total && k0 >= below && k1 < below + ncand;
    if (threadIdx.x < 2) { found[threadIdx.x][0] = 0ull; found[threadIdx.x][1] = 0ull; }
    __syncthreads();
    const unsigned long long r0 = ok ? k0 - below : 0ull, r1 = ok ? k1 - below : 0ull;
    block_find_bin(h, FAST_NBINS, r0, wsum, found[0]);
    block_find_bin(h, FAST_NBINS, r1, wsum, found[1]);
    if (threadIdx.x == 0) {
        fs->bin_a = (unsigned int)found[0][0];
        fs->bin_b = (unsigned int)found[1][0];
        fs->base_a = found[0][1];
        fs->r0 = r0; fs->r1 = r1;
        fs->valid = (ok || nnan) ? 1 : 0;
        fs->is_nan = nnan ? 1 : 0;
        fs->nfin = 0; fs->ticket_fin = 0; fs->ticket_hist = 0;
    }
}

// SCAN: single GPU -- the last CTA to finish also scans (counters are already global).
template <bool SCAN>
__global__ void __launch_bounds__(PXF_BLOCK)
k_cand_hist(const double *__restrict__ cand, unsigned long long cap, const unsigned long long *__restrict__ ncand_ptr,
            const unsigned long long *__restrict__ counters, const double *__restrict__ lohi,
            unsigned long long k0, unsigned long long k1, unsigned int *__restrict__ fhist, FastSel *__restrict__ fs)
{
    __shared__ unsigned int sh[FAST_NBINS];
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long found[2][2];
    __shared__ bool last;
    unsigned long long ncand = *ncand_ptr;
    if (ncand > cap) ncand = cap;                    // overflow is flagged through the counters
    const double lo = lohi[1], scale = cand_scale(lo, lohi[2]);
    for (int t = threadIdx.x; t < FAST_NBINS; t += blockDim.x) sh[t] = 0u;
    __syncthreads();
    const unsigned long long nthr = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < ncand; i0 += 8 * nthr) {
        double rv[8];
#pragma unroll
        for (int u = 0; u < 8; u++) { const unsigned long long i = i0 + u * nthr; rv[u] = i < ncand ? cand[i] : 0.; }
#pragma unroll
        for (int u = 0; u < 8; u++)
            if (i0 + u * nthr < ncand) atomicAdd(&sh[cand_bin(rv[u], lo, scale)], 1u);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < FAST_NBINS; t += blockDim.x) {
        const unsigned int v = sh[t];
        if (v) atomicAdd(&fhist[t], v);
    }
    if (!SCAN) return;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(&fs->ticket_hist, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    for (int t = threadIdx.x; t < FAST_NBINS; t += blockDim.x) sh[t] = __ldcg(&fhist[t]);
    __syncthreads();
    cand_scan_block(sh, counters, cap, k0, k1, fs, wsum, found);
}

// multi-GPU: the scan alone, on the all-reduced histogram and counters
__global__ void __launch_bounds__(PXF_BLOCK)
k_cand_scan(const unsigned int *__restrict__ fhist, const unsigned long long *__restrict__ counters,
            unsigned long long k0, unsigned long long k1, FastSel *__restrict__ fs)
{
    __shared__ unsigned int sh[FAST_NBINS];
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long found[2][2];
    for (int t = threadIdx.x; t < FAST_NBINS; t += blockDim.x) sh[t] = fhist[t];
    __syncthreads();
    cand_scan_block(sh, counters, ~0ull, k0, k1, fs, wsum, found);
}

// ascending bitonic sort of m (a power of two) NaN-free keys in shared memory; all threads of the CTA call
PXF_DEV void block_bitonic_sort(double *srt, unsigned int m)
{
    for (unsigned int k = 2; k <= m; k <<= 1) {
        for (unsigned int j = k >> 1; j > 0; j >>= 1) {
            for (unsigned int t = threadIdx.x; t < m; t += blockDim.x) {
                const unsigned int u = t ^ j;
                if (u > t) {
                    const double a = srt[t], b = srt[u];
                    const bool up = (t & k) == 0;
                    if ((a > b) == up) { srt[t] = b; srt[u] = a; }
                }
            }
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(PXF_BLOCK)
k_cand_finish(const double *__restrict__ cand, unsigned long long cap, const unsigned long long *__restrict__ ncand_ptr,
              const double *__restrict__ lohi, FastSel *__restrict__ fs, double *__restrict__ fin,
              double *__restrict__ out, int *__restrict__ fin_count)
{
    // fin_count != NULL (multi-GPU): gather this shard's keys of the chosen bins and report how many;
    // the sort happens after the all-gather (k_small_select).  Otherwise the last CTA sorts in place.
    __shared__ double srt[FAST_FINCAP];
    __shared__ bool last;
    const int valid = fs->valid;
    if (!valid || fs->is_nan) {
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            if (fin_count) { *fin_count = 0; return; }
            const double nanv = __longlong_as_double(0x7ff8000000000000ll);
            out[0] = nanv; out[1] = nanv; out[2] = nanv; out[3] = valid ? 1. : 0.;
        }
        return;
    }
    unsigned long long ncand = *ncand_ptr;
    if (ncand > cap) ncand = cap;
    const double lo = lohi[1], scale = cand_scale(lo, lohi[2]);
    const int ba = (int)fs->bin_a, bb = (int)fs->bin_b;
    const unsigned long long nthr = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < ncand; i0 += 8 * nthr) {
        double rv[8];
#pragma unroll
        for (int u = 0; u < 8; u++) { const unsigned long long i = i0 + u * nthr; rv[u] = i < ncand ? cand[i] : 0.; }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int b = cand_bin(rv[u], lo, scale);
            if (i0 + u * nthr < ncand && b >= ba && b <= bb) {
                const unsigned int slot = atomicAdd(&fs->nfin, 1u);
                if (slot < FAST_FINCAP) fin[slot] = rv[u];
            }
        }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(&fs->ticket_fin, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    const unsigned int n = *reinterpret_cast<volatile unsigned int *>(&fs->nfin);
    if (fin_count) {
        if (threadIdx.x == 0) *fin_count = (int)(n < 0x7fffffffu ? n : 0x7fffffffu);    // > FAST_FINCAP = overflow
        return;
    }
    const unsigned long long i0 = fs->r0 - fs->base_a, i1 = fs->r1 - fs->base_a;
    if (n > FAST_FINCAP || i1 >= n) {
        if (threadIdx.x == 0) { out[0] = 0.; out[1] = 0.; out[2] = 0.; out[3] = 0.; }
        return;
    }
    // bitonic sort of n keys padded with +Inf to a power of two
    unsigned int m = 1;
    while (m < n) m <<= 1;
    for (unsigned int t = threadIdx.x; t < m; t += blockDim.x)
        srt[t] = t < n ? __ldcg(&fin[t]) : __longlong_as_double(0x7ff0000000000000ll);
    __syncthreads();
    block_bitonic_sort(srt, m);
    if (threadIdx.x == 0) {
        const double a = srt[i0], b = srt[i1];
        out[0] = ((a + b) / 2.) * 2.;
        out[1] = a; out[2] = b; out[3] = 1.;
    }
}

// ------------------------------------------------------------------ compaction
#define CTILE 2048   // rays per CTA tile: 8 warps x 8 chunks x 32 lanes

__global__ void __launch_bounds__(PXF_BLOCK)
k_vignette_flags(const double *__restrict__ l, const double *__restrict__ m, const double *__restrict__ n,
                 int64_t num, uint8_t *__restrict__ flags)
{
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < num; i += nthr) {
        double mag = sq(l[i]) + sq(m[i]) + sq(n[i]);
        flags[i] = mag > .1 ? 1 : 0;
    }
}

// per-tile survivor counts
__global__ void __launch_bounds__(PXF_BLOCK)
k_compact_count(const uint8_t *__restrict__ flags, int64_t num, unsigned int *__restrict__ tile_count)
{
    __shared__ unsigned int sh[PXF_BLOCK / 32];
    const int64_t base = (int64_t)blockIdx.x * CTILE;
    unsigned int c = 0;
#pragma unroll
    for (int j = 0; j < CTILE / PXF_BLOCK; j++) {
        int64_t i = base + j * PXF_BLOCK + threadIdx.x;
        if (i < num && flags[i]) c++;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = 0;
        for (int w = 0; w < PXF_BLOCK / 32; w++) t += sh[w];
        tile_count[blockIdx.x] = t;
    }
}

// exclusive scan of the tile counts into 64-bit offsets; total at offsets[ntiles]
__global__ void __launch_bounds__(1024)
k_compact_scan(const unsigned int *__restrict__ tile_count, int64_t ntiles, long long *__restrict__ offsets)
{
    __shared__ long long wsum[32];
    __shared__ long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t b0 = 0; b0 < ntiles; b0 += blockDim.x) {
        int64_t b = b0 + threadIdx.x;
        long long v = b < ntiles ? (long long)tile_count[b] : 0;
        long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            long long w = wsum[lane];
            long long iw = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                long long t = __shfl_up_sync(0xffffffffu, iw, o);
                if (lane >= o) iw += t;
            }
            wsum[lane] = iw - w;
        }
        __syncthreads();
        long long excl = carry + wsum[warp] + incl - v;
        if (b < ntiles) offsets[b] = excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) offsets[ntiles] = carry;
}

// Each warp owns 8 consecutive 32-ray chunks of the tile; ballot + popc give the rank inside a
// chunk, a 64-entry shared scan gives the chunk base, the tile offset comes from k_compact_scan.
// row pointers travel as a kernel argument (no pointer loads in the loop, no H2D staging copy)
struct RowTable { const double *in[16]; double *out[16]; };

template <int MODE>   // 0: scatter rows, 1: write indices
__global__ void __launch_bounds__(PXF_BLOCK)
k_compact_scatter(const __grid_constant__ RowTable T, int nrows,
                  const uint8_t *__restrict__ flags, int64_t num, const long long *__restrict__ offsets,
                  long long *__restrict__ idx_out)
{
    __shared__ unsigned int chunk_cnt[CTILE / 32];
    __shared__ unsigned int chunk_base[CTILE / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t base = (int64_t)blockIdx.x * CTILE;
    unsigned int ballots[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int chunk = warp * 8 + j;
        const int64_t i = base + chunk * 32 + lane;
        const bool f = i < num && flags[i] != 0;
        ballots[j] = __ballot_sync(0xffffffffu, f);
        if (lane == 0) chunk_cnt[chunk] = __popc(ballots[j]);
    }
    __syncthreads();
    if (warp == 0) {
        unsigned int a = chunk_cnt[lane], b = chunk_cnt[lane + 32];
        unsigned int ia = a, ib = b;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned int ta = __shfl_up_sync(0xffffffffu, ia, o);
            unsigned int tb = __shfl_up_sync(0xffffffffu, ib, o);
            if (lane >= o) { ia += ta; ib += tb; }
        }
        unsigned int total_a = __shfl_sync(0xffffffffu, ia, 31);
        chunk_base[lane] = ia - a;
        chunk_base[lane + 32] = total_a + ib - b;
    }
    __syncthreads();
    const long long tile_off = offsets[blockIdx.x];
    long long dst[8];
    bool keep[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int chunk = warp * 8 + j;
        keep[j] = (ballots[j] >> lane) & 1u;
        dst[j] = tile_off + chunk_base[chunk] + __popc(ballots[j] & ((1u << lane) - 1));
    }
    const int64_t i0 = base + warp * 256 + lane;
    if (MODE == 0) {
        // row-outer: the eight loads of a row are issued together, then the eight stores
        for (int r = 0; r < nrows; r++) {
            const double *__restrict__ src = T.in[r];
            double *__restrict__ out = T.out[r];
            double v[8];
#pragma unroll
            for (int j = 0; j < 8; j++) v[j] = keep[j] ? src[i0 + j * 32] : 0.;
#pragma unroll
            for (int j = 0; j < 8; j++)
                if (keep[j]) out[dst[j]] = v[j];
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (keep[j]) idx_out[dst[j]] = i0 + j * 32;
    }
}

__global__ void __launch_bounds__(PXF_BLOCK)
k_gather_rows(const __grid_constant__ RowTable T, int nrows, const long long *__restrict__ idx, int64_t count)
{
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < count; i += nthr) {
        const long long s = idx[i];
        for (int r = 0; r < nrows; r++) T.out[r][i] = T.in[r][s];
    }
}

// ------------------------------------------------------------------ segmented bundles
// Per-segment versions of the analyses for a bundle that is a concatenation of segments (seg_start[0..nseg],
// the layout of SegmentedProgram).  Every kernel walks the bundle in tiles with seg_tile_pieces; the launch count
// does not depend on nseg.
//
// Sums: a tile of SEGSUM_TILE rays splits into pieces (tile t, segment s); walking the bundle in order, each
// piece advances t or s or both, so slot = t + s is unique and the slots of one segment are contiguous
// ([start/T + s, (end-1)/T + s]).  One partial per slot, then one CTA per segment folds its slots in a fixed
// tree: the same bits on every run for the same bundle and layout, whatever the grid.
#define SEGSUM_TILE 4096

PXF_DEV void block_sum_store(const double *acc, int ns, double *__restrict__ out, double (*sh)[PXF_BLOCK / 32])
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = 0; k < ns; k++) {
        double v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) sh[k][warp] = v;
    }
    __syncthreads();
    if (warp == 0) {
        for (int k = 0; k < ns; k++) {
            double v = lane < PXF_BLOCK / 32 ? sh[k][lane] : 0.;
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) out[k] = v;
        }
    }
    __syncthreads();
}

template <int MODE, bool VEC2>
__global__ void __launch_bounds__(PXF_BLOCK)
k_sums_seg(const double *__restrict__ x, const double *__restrict__ y, const double *__restrict__ z,
           const double *__restrict__ l, const double *__restrict__ m, const double *__restrict__ n,
           const double *__restrict__ w, int64_t num, const long long *__restrict__ seg_start, int nseg,
           const double *__restrict__ ab_dev, double *__restrict__ partial)
{
    constexpr int NS = MODE == PXF_SUMS_CENTROID ? 4 : ((MODE == PXF_SUMS_RMS || MODE == PXF_SUMS_POINT) ? 2 : 9);
    constexpr bool IP = MODE == PXF_SUMS_IMAGEPLANE || MODE == PXF_SUMS_IMAGEPLANE_Z;
    constexpr bool ZZ = MODE == PXF_SUMS_IMAGEPLANE_Z || MODE == PXF_SUMS_POINT;
    constexpr int U = IP ? 2 : 4;
    __shared__ double sh[NSUM][PXF_BLOCK / 32];
    const bool has_w = w != nullptr;
    // one ray through sums_accum, loaded with scalar loads (odd ends of a piece, unaligned rows)
    auto one = [&](double *acc, int64_t i, double a, double b, double c) {
        sums_accum<MODE>(acc, x[i], y[i], IP ? l[i] : 0., IP ? m[i] : 0., IP ? n[i] : 1., has_w ? w[i] : 1., has_w, a, b,
                         ZZ ? z[i] : 0., c);
    };
    for (int64_t t0 = (int64_t)blockIdx.x * SEGSUM_TILE; t0 < num; t0 += (int64_t)gridDim.x * SEGSUM_TILE) {
        const int64_t t1 = t0 + SEGSUM_TILE < num ? t0 + SEGSUM_TILE : num;
        const int64_t tile = t0 / SEGSUM_TILE;
        seg_tile_pieces(t0, t1, seg_start, nseg, [&](int seg, int64_t pa, int64_t pb) {
            double a = 0., b = 0., c = 0.;
            if (MODE == PXF_SUMS_RMS) { a = ab_dev[2 * seg]; b = ab_dev[2 * seg + 1]; }
            if (MODE == PXF_SUMS_POINT) { a = ab_dev[3 * seg]; b = ab_dev[3 * seg + 1]; c = ab_dev[3 * seg + 2]; }
            double acc[U][NSUM];
#pragma unroll
            for (int u = 0; u < U; u++)
#pragma unroll
                for (int k = 0; k < NSUM; k++) acc[u][k] = 0.;
            if (VEC2) {
                // pairs at even bundle indices (the 16-byte alignment of the rows), odd ends one by one
                const int64_t q0 = (pa + 1) >> 1, q1 = pb >> 1;
                for (int64_t qb = q0 + threadIdx.x; qb < q1; qb += U * blockDim.x) {
                    double2 xv[U], yv[U], lv[U], mv[U], nv[U], wv[U], zv[U];
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        const int64_t q = qb + u * blockDim.x;
                        const bool in = q < q1;
                        const double2 z2 = make_double2(0., 0.), o2 = make_double2(1., 1.);
                        xv[u] = in ? *reinterpret_cast<const double2 *>(x + 2 * q) : z2;
                        yv[u] = in ? *reinterpret_cast<const double2 *>(y + 2 * q) : z2;
                        if (IP) {
                            lv[u] = in ? *reinterpret_cast<const double2 *>(l + 2 * q) : z2;
                            mv[u] = in ? *reinterpret_cast<const double2 *>(m + 2 * q) : z2;
                            nv[u] = in ? *reinterpret_cast<const double2 *>(n + 2 * q) : o2;
                        } else { lv[u] = z2; mv[u] = z2; nv[u] = o2; }
                        zv[u] = (ZZ && in) ? *reinterpret_cast<const double2 *>(z + 2 * q) : z2;
                        wv[u] = (in && has_w) ? *reinterpret_cast<const double2 *>(w + 2 * q) : o2;
                    }
#pragma unroll
                    for (int u = 0; u < U; u++)
                        if (qb + u * blockDim.x < q1) {
                            sums_accum<MODE>(acc[u], xv[u].x, yv[u].x, lv[u].x, mv[u].x, nv[u].x, wv[u].x, has_w, a, b, zv[u].x, c);
                            sums_accum<MODE>(acc[u], xv[u].y, yv[u].y, lv[u].y, mv[u].y, nv[u].y, wv[u].y, has_w, a, b, zv[u].y, c);
                        }
                }
                if (threadIdx.x == 0 && (pa & 1)) one(acc[0], pa, a, b, c);
                if (threadIdx.x == 1 && (pb & 1) && pb - 1 >= 2 * q0) one(acc[0], pb - 1, a, b, c);
            } else {
                for (int64_t i = pa + threadIdx.x; i < pb; i += blockDim.x) one(acc[0], i, a, b, c);
            }
#pragma unroll
            for (int k = 0; k < NS; k++) {
                double t = acc[0][k];
#pragma unroll
                for (int u = 1; u < U; u++) t += acc[u][k];
                acc[0][k] = t;
            }
            block_sum_store(acc[0], NS, partial + (tile + seg) * NSUM, sh);
        });
    }
}

// one CTA per segment: fixed-order fold of its slots; out[16 s + k], k >= ns zeroed
__global__ void __launch_bounds__(PXF_BLOCK)
k_sums_seg_fold(const double *__restrict__ partial, const long long *__restrict__ seg_start, int ns,
                double *__restrict__ out)
{
    __shared__ double sh[NSUM][PXF_BLOCK / 32];
    const int s = blockIdx.x;
    const long long a = seg_start[s], b = seg_start[s + 1];
    const long long first = b > a ? a / SEGSUM_TILE + s : 0, last = b > a ? (b - 1) / SEGSUM_TILE + s : -1;
    double acc[NSUM];
    for (int k = 0; k < NSUM; k++) acc[k] = 0.;
    for (long long q = first + threadIdx.x; q <= last; q += blockDim.x)
        for (int k = 0; k < ns; k++) acc[k] += partial[q * NSUM + k];
    double v[NSUM];
    block_sum_store(acc, ns, v, sh);
    if (threadIdx.x == 0)
        for (int k = 0; k < 16; k++) out[16 * (int64_t)s + k] = k < ns ? v[k] : 0.;
}

// cxy[2 s..] = sums[16 s + 1] / sums[16 s], sums[16 s + 2] / sums[16 s] (k_centroid_from_sums per segment)
__global__ void k_centroids_seg(const double *__restrict__ sums, int nseg, double *__restrict__ cxy)
{
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < nseg; s += gridDim.x * blockDim.x) {
        cxy[2 * s] = sums[16 * (int64_t)s + 1] / sums[16 * (int64_t)s];
        cxy[2 * s + 1] = sums[16 * (int64_t)s + 2] / sums[16 * (int64_t)s];
    }
}

// survivors per segment: counts[s] += #flags != 0 (zeroed by the caller)
__global__ void __launch_bounds__(PXF_BLOCK)
k_seg_counts(const uint8_t *__restrict__ flags, int64_t num, const long long *__restrict__ seg_start, int nseg,
             unsigned long long *__restrict__ counts)
{
    __shared__ unsigned int cnt;
    for (int64_t t0 = (int64_t)blockIdx.x * SEGSUM_TILE; t0 < num; t0 += (int64_t)gridDim.x * SEGSUM_TILE) {
        const int64_t t1 = t0 + SEGSUM_TILE < num ? t0 + SEGSUM_TILE : num;
        seg_tile_pieces(t0, t1, seg_start, nseg, [&](int seg, int64_t pa, int64_t pb) {
            if (threadIdx.x == 0) cnt = 0;
            __syncthreads();
            unsigned int c = 0;
            for (int64_t i = pa + threadIdx.x; i < pb; i += blockDim.x) c += flags[i] != 0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
            if ((threadIdx.x & 31) == 0 && c) atomicAdd(&cnt, c);
            __syncthreads();
            if (threadIdx.x == 0 && cnt) atomicAdd(&counts[seg], (unsigned long long)cnt);
            __syncthreads();
        });
    }
}

// ---- segmented unweighted HPD: exact 2*median of every segment's radii about its own centroid
// k_hpdseg_prepare  one CTA per segment.  Up to SEG_DIRECT rays: all radii in shared memory, bitonic sort, done.
//                   Larger: a strided sample of SEG_DIRECT radii, sorted -> bracket [lo, hi] around the median
//                   (sample ranks 0.5 +- 6 sigma, pxf_bracket_sample_ranks).
// k_hpdseg_collect  ONE pass over the bundle: per bracketed segment, #(r < lo), #NaN, and the radii inside the
//                   bracket appended to the segment's slice of the candidate buffer (capacity ~1/8 of the segment)
// k_hpdseg_finish   one CTA per bracketed segment: 4096 linear bins over [lo, hi] locate the middle ranks, the
//                   keys of those bins are sorted in shared memory.
// A bracket miss, a candidate overflow or ties piling up in one bin leave valid = 0 for that segment only; the
// caller resolves those segments with the five-pass select on their slice.
#define SEG_DIRECT 8192
#define SEG_CAND_DIV 8
#define SEG_FINCAP 8192

PXF_DEV double nan_d() { return __longlong_as_double(0x7ff8000000000000ll); }

__global__ void __launch_bounds__(1024)
k_hpdseg_prepare(const double *__restrict__ x, const double *__restrict__ y, const long long *__restrict__ seg_start,
                 const double *__restrict__ sums, int ra, int rb, double *__restrict__ cxy, double *__restrict__ lohi,
                 unsigned long long *__restrict__ counters, int *__restrict__ state, double *__restrict__ out)
{
    extern __shared__ double keys[];
    const int s = blockIdx.x;
    const long long a = seg_start[s], n = seg_start[s + 1] - a;
    const double cx = sums[16 * (int64_t)s + 1] / sums[16 * (int64_t)s], cy = sums[16 * (int64_t)s + 2] / sums[16 * (int64_t)s];
    double *o = out + 4 * (int64_t)s;
    if (threadIdx.x == 0) {
        cxy[2 * s] = cx; cxy[2 * s + 1] = cy;
        counters[3 * (int64_t)s] = 0; counters[3 * (int64_t)s + 1] = 0; counters[3 * (int64_t)s + 2] = 0;
        state[s] = 0;
    }
    if (n == 0) {                                       // np.median([]) is nan
        if (threadIdx.x == 0) { o[0] = nan_d(); o[1] = nan_d(); o[2] = nan_d(); o[3] = 1.; }
        return;
    }
    const int mcnt = n <= SEG_DIRECT ? (int)n : SEG_DIRECT;
    bool nan = false;
    for (int j = threadIdx.x; j < mcnt; j += blockDim.x) {
        const long long i = a + (n <= SEG_DIRECT ? j : (long long)(((unsigned long long)j * (unsigned long long)n) / SEG_DIRECT));
        const double r = sqrt(sq(x[i] - cx) + sq(y[i] - cy));
        keys[j] = r;
        nan = nan || r != r;
    }
    if (__syncthreads_or(nan)) {                        // a NaN radius: np.median is nan
        if (threadIdx.x == 0) { o[0] = nan_d(); o[1] = nan_d(); o[2] = nan_d(); o[3] = 1.; }
        return;
    }
    unsigned int m2 = 1;
    while (m2 < (unsigned)mcnt) m2 <<= 1;
    for (unsigned int t = mcnt + threadIdx.x; t < m2; t += blockDim.x) keys[t] = __longlong_as_double(0x7ff0000000000000ll);
    __syncthreads();
    block_bitonic_sort(keys, m2);
    if (threadIdx.x == 0) {
        if (n <= SEG_DIRECT) {
            const double lo = keys[(n - 1) / 2], hi = keys[n / 2];
            o[0] = ((lo + hi) / 2.) * 2.; o[1] = lo; o[2] = hi; o[3] = 1.;
        } else {
            lohi[2 * s] = keys[ra]; lohi[2 * s + 1] = keys[rb];
            state[s] = 1;
        }
    }
}

#define SEGCOL_TILE 4096
template <bool VEC2>
__global__ void __launch_bounds__(PXF_BLOCK)
k_hpdseg_collect(const double *__restrict__ x, const double *__restrict__ y, int64_t num,
                 const long long *__restrict__ seg_start, int nseg, const int *__restrict__ state,
                 const double *__restrict__ cxy, const double *__restrict__ lohi, double *__restrict__ cand,
                 unsigned long long *__restrict__ counters)
{
    __shared__ double sbuf[SEGCOL_TILE];
    __shared__ unsigned int scount, sbelow, snan;
    __shared__ unsigned long long sbase;
    for (int64_t t0 = (int64_t)blockIdx.x * SEGCOL_TILE; t0 < num; t0 += (int64_t)gridDim.x * SEGCOL_TILE) {
        const int64_t t1 = t0 + SEGCOL_TILE < num ? t0 + SEGCOL_TILE : num;
        seg_tile_pieces(t0, t1, seg_start, nseg, [&](int seg, int64_t pa, int64_t pb) {
            if (state[seg] != 1) return;               // block-uniform
            const double cx = cxy[2 * seg], cy = cxy[2 * seg + 1], lo = lohi[2 * seg], hi = lohi[2 * seg + 1];
            if (threadIdx.x == 0) { scount = 0; sbelow = 0; snan = 0; }
            __syncthreads();
            unsigned int below = 0, nans = 0;
            auto put = [&](double r) {
                if (r != r) nans++;
                else if (r < lo) below++;
                else if (r <= hi) sbuf[atomicAdd(&scount, 1u)] = r;
            };
            if (VEC2) {
                const int64_t q0 = (pa + 1) >> 1, q1 = pb >> 1;
                for (int64_t qb = q0 + threadIdx.x; qb < q1; qb += 4 * blockDim.x) {
                    double2 xv[4], yv[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int64_t q = qb + u * blockDim.x;
                        xv[u] = q < q1 ? *reinterpret_cast<const double2 *>(x + 2 * q) : make_double2(0., 0.);
                        yv[u] = q < q1 ? *reinterpret_cast<const double2 *>(y + 2 * q) : make_double2(0., 0.);
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++)
                        if (qb + u * blockDim.x < q1) {
                            put(sqrt(sq(xv[u].x - cx) + sq(yv[u].x - cy)));
                            put(sqrt(sq(xv[u].y - cx) + sq(yv[u].y - cy)));
                        }
                }
                if (threadIdx.x == 0 && (pa & 1)) put(sqrt(sq(x[pa] - cx) + sq(y[pa] - cy)));
                if (threadIdx.x == 1 && (pb & 1) && pb - 1 >= 2 * q0) put(sqrt(sq(x[pb - 1] - cx) + sq(y[pb - 1] - cy)));
            } else {
                for (int64_t i = pa + threadIdx.x; i < pb; i += blockDim.x) put(sqrt(sq(x[i] - cx) + sq(y[i] - cy)));
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                below += __shfl_down_sync(0xffffffffu, below, o);
                nans += __shfl_down_sync(0xffffffffu, nans, o);
            }
            if ((threadIdx.x & 31) == 0) {
                if (below) atomicAdd(&sbelow, below);
                if (nans) atomicAdd(&snan, nans);
            }
            __syncthreads();
            unsigned long long *c = counters + 3 * (int64_t)seg;
            if (threadIdx.x == 0) {
                sbase = scount ? atomicAdd(&c[1], (unsigned long long)scount) : 0ull;
                if (sbelow) atomicAdd(&c[0], (unsigned long long)sbelow);
                if (snan) atomicAdd(&c[2], (unsigned long long)snan);
            }
            __syncthreads();
            const long long a = seg_start[seg];
            const unsigned long long cap = (unsigned long long)(seg_start[seg + 1] / SEG_CAND_DIV - a / SEG_CAND_DIV);
            double *dst = cand + a / SEG_CAND_DIV;
            for (unsigned int t = threadIdx.x; t < scount; t += blockDim.x)
                if (sbase + t < cap) dst[sbase + t] = sbuf[t];
            __syncthreads();
        });
    }
}

__global__ void __launch_bounds__(1024)
k_hpdseg_finish(const long long *__restrict__ seg_start, const int *__restrict__ state,
                const unsigned long long *__restrict__ counters, const double *__restrict__ lohi,
                const double *__restrict__ cand, double *__restrict__ out)
{
    extern __shared__ double fin[];                                   // [SEG_FINCAP] then the bins
    unsigned int *h = reinterpret_cast<unsigned int *>(fin + SEG_FINCAP);
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long found[2][2];
    __shared__ unsigned int nfin;
    const int s = blockIdx.x;
    if (state[s] != 1) return;
    double *o = out + 4 * (int64_t)s;
    const long long a = seg_start[s], b = seg_start[s + 1], n = b - a;
    const unsigned long long k0 = (n - 1) / 2, k1 = n / 2;
    const unsigned long long below = counters[3 * (int64_t)s], nc = counters[3 * (int64_t)s + 1];
    const unsigned long long cap = (unsigned long long)(b / SEG_CAND_DIV - a / SEG_CAND_DIV);
    if (counters[3 * (int64_t)s + 2]) {
        if (threadIdx.x == 0) { o[0] = nan_d(); o[1] = nan_d(); o[2] = nan_d(); o[3] = 1.; }
        return;
    }
    if (!(nc <= cap && k0 >= below && k1 < below + nc)) {
        if (threadIdx.x == 0) { o[0] = 0.; o[1] = 0.; o[2] = 0.; o[3] = 0.; }
        return;
    }
    const double *c = cand + a / SEG_CAND_DIV;
    const double lo = lohi[2 * s], scale = cand_scale(lo, lohi[2 * s + 1]);
    for (int t = threadIdx.x; t < FAST_NBINS; t += blockDim.x) h[t] = 0u;
    if (threadIdx.x < 2) { found[threadIdx.x][0] = 0ull; found[threadIdx.x][1] = 0ull; }
    if (threadIdx.x == 0) nfin = 0;
    __syncthreads();
    for (unsigned long long i = threadIdx.x; i < nc; i += blockDim.x) atomicAdd(&h[cand_bin(c[i], lo, scale)], 1u);
    __syncthreads();
    const unsigned long long r0 = k0 - below, r1 = k1 - below;
    block_find_bin(h, FAST_NBINS, r0, wsum, found[0]);
    block_find_bin(h, FAST_NBINS, r1, wsum, found[1]);
    const int ba = (int)found[0][0], bb = (int)found[1][0];
    const unsigned long long base_a = found[0][1];
    for (unsigned long long i = threadIdx.x; i < nc; i += blockDim.x) {
        const double r = c[i];
        const int bin = cand_bin(r, lo, scale);
        if (bin >= ba && bin <= bb) {
            const unsigned int slot = atomicAdd(&nfin, 1u);
            if (slot < SEG_FINCAP) fin[slot] = r;
        }
    }
    __syncthreads();
    const unsigned int nf = nfin;
    if (nf > SEG_FINCAP || r1 - base_a >= nf) {                       // ties piled up in the middle bins
        if (threadIdx.x == 0) { o[0] = 0.; o[1] = 0.; o[2] = 0.; o[3] = 0.; }
        return;
    }
    unsigned int m2 = 1;
    while (m2 < nf) m2 <<= 1;
    for (unsigned int t = nf + threadIdx.x; t < m2; t += blockDim.x) fin[t] = __longlong_as_double(0x7ff0000000000000ll);
    __syncthreads();
    block_bitonic_sort(fin, m2);
    if (threadIdx.x == 0) {
        const double va = fin[r0 - base_a], vb = fin[r1 - base_a];
        o[0] = ((va + vb) / 2.) * 2.; o[1] = va; o[2] = vb; o[3] = 1.;
    }
}

static int need_device()
{
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    return PXF_OK;
}

static int select_smem_bytes(int bits) { return 2 * (1 << bits) * (int)sizeof(unsigned int); }

static int select_pass(const double *x, const double *y, const double *keys, int64_t num,
                       const unsigned long long *count_dev, const double *cxy, int shift, int bits,
                       SelectState *st, unsigned long long *hist, unsigned long long *nan_count, cudaStream_t s)
{
    static bool attr_set[64] = {};
    if (first_on_device(attr_set)) {
        cudaFuncSetAttribute(k_select_hist<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, select_smem_bytes(13));
        cudaFuncSetAttribute(k_select_hist<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, select_smem_bytes(13));
    }
    int grid = grid_for(num, PXF_BLOCK * 8, 3);
    if (keys)
        k_select_hist<true><<<grid, PXF_BLOCK, select_smem_bytes(bits), s>>>(x, y, keys, num, count_dev, cxy, shift,
                                                                           bits, st, hist, nan_count);
    else
        k_select_hist<false><<<grid, PXF_BLOCK, select_smem_bytes(bits), s>>>(x, y, keys, num, count_dev, cxy, shift,
                                                                            bits, st, hist, nan_count);
    count_launch();
    return check_launch("k_select_hist");
}

}  // namespace pxf

using namespace pxf;

extern "C" {

size_t pxf_sums_scratch_bytes(void) { return (size_t)SUM_BLOCKS_MAX * NSUM * sizeof(double); }

int pxf_sums(int32_t mode, const double *x, const double *y, const double *l, const double *m,
             const double *n, const double *w, int64_t num, double a, double b,
             double *out_dev, void *scratch, pxf_stream_t stream)
{
    return sums_launch(mode, x, y, l, m, n, w, num, a, b, nullptr, out_dev, scratch,
                       reinterpret_cast<cudaStream_t>(stream));
}

int pxf_sums_z(const double *x, const double *y, const double *z, const double *l, const double *m,
               const double *n, const double *w, int64_t num, double *out_dev, void *scratch, pxf_stream_t stream)
{
    return sums_launch(PXF_SUMS_IMAGEPLANE_Z, x, y, l, m, n, w, num, 0., 0., nullptr, out_dev, scratch,
                       reinterpret_cast<cudaStream_t>(stream), z);
}

int pxf_rho(const double *x, const double *y, int64_t num, double cx, double cy, double *rho_out,
            pxf_stream_t stream)
{
    if (num == 0) return PXF_OK;
    if (num < 0 || !x || !y || !rho_out) { set_error("pxf_rho: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_rho<<<grid_for(num, PXF_BLOCK * 2, 8), PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        x, y, num, cx, cy, nullptr, rho_out);
    count_launch();
    return check_launch("k_rho");
}

// ---- radix-select primitives (device-resident state; used directly by the sharded path) ----
size_t pxf_select_state_bytes(void) { return sizeof(SelectState) + 8 /*nan*/ + 2 * 8192 * 8 /*hist*/ + 64; }

/* state layout inside the caller's buffer: [SelectState][nan u64][pad][hist u64 x 2*8192] */
static inline SelectState *st_of(void *buf) { return reinterpret_cast<SelectState *>(buf); }
static inline unsigned long long *nan_of(void *buf) { return reinterpret_cast<unsigned long long *>((char *)buf + 48); }
static inline unsigned long long *hist_of(void *buf) { return reinterpret_cast<unsigned long long *>((char *)buf + 64); }

int pxf_select_begin(void *state, int64_t k0, int64_t k1, pxf_stream_t stream)
{
    if (!state || k0 < 0 || k1 < k0) { set_error("pxf_select_begin: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_select_init<<<16, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        st_of(state), (unsigned long long)k0, (unsigned long long)k1, hist_of(state), 2 * 8192, nan_of(state));
    count_launch();
    return check_launch("k_select_init");
}

/* histogram of one digit of the local shard into the state's histogram (device uint64[2<<13]) */
int pxf_select_hist(const double *x, const double *y, const double *keys, int64_t num, const double *cxy_dev,
                    int32_t shift, int32_t bits, void *state, pxf_stream_t stream)
{
    if (!state || bits < 1 || bits > 13 || shift < 0 || shift + bits > 64 || num < 0 ||
        (!keys && (!x || !y || !cxy_dev))) {
        set_error("pxf_select_hist: bad argument");
        return PXF_ERR_INVALID;
    }
    int rc = need_device();
    if (rc) return rc;
    if (num == 0) return PXF_OK;
    return select_pass(x, y, keys, num, nullptr, cxy_dev, shift, bits, st_of(state), hist_of(state), nan_of(state),
                       reinterpret_cast<cudaStream_t>(stream));
}

uint64_t *pxf_select_hist_ptr(void *state) { return reinterpret_cast<uint64_t *>(hist_of(state)); }
uint64_t *pxf_select_nan_ptr(void *state) { return reinterpret_cast<uint64_t *>(nan_of(state)); }

/* narrow both chains by `bits` using the (possibly all-reduced) histogram, then clear it */
int pxf_select_narrow(int32_t bits, void *state, pxf_stream_t stream)
{
    if (!state || bits < 1 || bits > 13) { set_error("pxf_select_narrow: bad argument"); return PXF_ERR_INVALID; }
    k_select_scan<<<1, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(hist_of(state), bits, st_of(state));
    count_launch();
    return check_launch("k_select_scan");
}

/* out_dev[0] = 2*median, out_dev[1..2] = the two middle order statistics */
int pxf_select_finish(void *state, int64_t num_total, double *out_dev, pxf_stream_t stream)
{
    if (!state || !out_dev) { set_error("pxf_select_finish: bad argument"); return PXF_ERR_INVALID; }
    k_select_result<<<1, 1, 0, reinterpret_cast<cudaStream_t>(stream)>>>(st_of(state), nan_of(state), num_total, out_dev);
    count_launch();
    return check_launch("k_select_result");
}

int pxf_centroid_from_sums(const double *sums_dev, double *cxy_dev, pxf_stream_t stream)
{
    if (!sums_dev || !cxy_dev) { set_error("pxf_centroid_from_sums: bad argument"); return PXF_ERR_INVALID; }
    k_centroid_from_sums<<<1, 1, 0, reinterpret_cast<cudaStream_t>(stream)>>>(sums_dev, cxy_dev);
    count_launch();
    return check_launch("k_centroid_from_sums");
}

// The digit schedule of the 64-bit key: 13+13+13+13+12.
static const int kShift[5] = {51, 38, 25, 12, 0};
static const int kBits[5] = {13, 13, 13, 13, 12};

int pxf_select_schedule(int32_t pass, int32_t *shift, int32_t *bits)
{
    if (pass < 0 || pass >= 5) return 0;
    *shift = kShift[pass]; *bits = kBits[pass];
    return 5;
}

// ---- single-GPU convenience entry points --------------------------------------------------
int pxf_centroid(const double *x, const double *y, const double *w, int64_t num,
                 double *cx_host, double *cy_host, pxf_stream_t stream)
{
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    int rc = need_device();
    if (rc) return rc;
    Scratch sc;
    if ((rc = sc.alloc(pxf_sums_scratch_bytes() + 16 * sizeof(double), s))) return rc;
    double *out = reinterpret_cast<double *>((char *)sc.p + pxf_sums_scratch_bytes());
    if ((rc = sums_launch(PXF_SUMS_CENTROID, x, y, nullptr, nullptr, nullptr, w, num, 0., 0., nullptr, out, sc.p, s)))
        return rc;
    double h[4];
    PXF_CUDA(cudaMemcpyAsync(h, out, sizeof(h), cudaMemcpyDeviceToHost, s));
    PXF_CUDA(cudaStreamSynchronize(s));
    *cx_host = h[1] / h[0];
    *cy_host = h[2] / h[0];
    return PXF_OK;
}

int pxf_rmscentroid(const double *x, const double *y, const double *w, int64_t num,
                    double *rms_host, pxf_stream_t stream)
{
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    int rc = need_device();
    if (rc) return rc;
    Scratch sc;
    if ((rc = sc.alloc(pxf_sums_scratch_bytes() + 32 * sizeof(double), s))) return rc;
    double *out = reinterpret_cast<double *>((char *)sc.p + pxf_sums_scratch_bytes());
    double *cxy = out + 16;
    if ((rc = sums_launch(PXF_SUMS_CENTROID, x, y, nullptr, nullptr, nullptr, w, num, 0., 0., nullptr, out, sc.p, s)))
        return rc;
    k_centroid_from_sums<<<1, 1, 0, s>>>(out, cxy);
    count_launch();
    if ((rc = sums_launch(PXF_SUMS_RMS, x, y, nullptr, nullptr, nullptr, w, num, 0., 0., cxy, out, sc.p, s)))
        return rc;
    double h[2];
    PXF_CUDA(cudaMemcpyAsync(h, out, sizeof(h), cudaMemcpyDeviceToHost, s));
    PXF_CUDA(cudaStreamSynchronize(s));
    *rms_host = sqrt(h[1] / h[0]);
    return PXF_OK;
}

int pxf_rmspoint(const double *x, const double *y, const double *z, const double *w, int64_t num,
                 double px, double py, double pz, double *rms_host, pxf_stream_t stream)
{
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    int rc = need_device();
    if (rc) return rc;
    if (!rms_host) { set_error("pxf_rmspoint: null result"); return PXF_ERR_INVALID; }
    Scratch sc;
    if ((rc = sc.alloc(pxf_sums_scratch_bytes() + 16 * sizeof(double), s))) return rc;
    double *out = reinterpret_cast<double *>((char *)sc.p + pxf_sums_scratch_bytes());
    if ((rc = sums_launch(PXF_SUMS_POINT, x, y, nullptr, nullptr, nullptr, w, num, px, py, nullptr, out, sc.p, s, z, pz)))
        return rc;
    double h[2];
    PXF_CUDA(cudaMemcpyAsync(h, out, sizeof(h), cudaMemcpyDeviceToHost, s));
    PXF_CUDA(cudaStreamSynchronize(s));
    *rms_host = sqrt(h[1] / h[0]);
    return PXF_OK;
}

int pxf_analyticimageplane(const double *x, const double *y, const double *l, const double *m,
                           const double *n, const double *w, int64_t num, double *dz_host,
                           pxf_stream_t stream)
{
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    int rc = need_device();
    if (rc) return rc;
    Scratch sc;
    if ((rc = sc.alloc(pxf_sums_scratch_bytes() + 16 * sizeof(double), s))) return rc;
    double *out = reinterpret_cast<double *>((char *)sc.p + pxf_sums_scratch_bytes());
    if ((rc = sums_launch(PXF_SUMS_IMAGEPLANE, x, y, l, m, n, w, num, 0., 0., nullptr, out, sc.p, s))) return rc;
    double h[9];
    PXF_CUDA(cudaMemcpyAsync(h, out, sizeof(h), cudaMemcpyDeviceToHost, s));
    PXF_CUDA(cudaStreamSynchronize(s));
    // analyses.py:123-131 with <q> = S_q/S_0
    const double W = h[0];
    double ax_ = h[1] / W, ay_ = h[2] / W, aln = h[3] / W, amn = h[4] / W;
    double bx = h[5] / W - ax_ * aln;
    double ax = h[7] / W - aln * aln;
    double by = h[6] / W - ay_ * amn;
    double ay = h[8] / W - amn * amn;
    *dz_host = -(bx + by) / (ax + ay);
    return PXF_OK;
}

// ---- bracketed-select primitives (also used by the sharded path) ----------------------------
int64_t pxf_bracket_min_num(void) { return BRACKET_MIN_NUM; }
int32_t pxf_bracket_samples(void) { return BRACKET_SAMPLES; }
/* candidate-buffer capacity (doubles) for a shard of num rays: 4 % of the shard */
int64_t pxf_bracket_capacity(int64_t num) { int64_t c = num / 25; return c < 65536 ? 65536 : c; }
/* sample ranks whose order statistics bracket the median: 0.5 +- 6 sigma of the sample quantile */
void pxf_bracket_sample_ranks(int32_t nsamp, int64_t *a, int64_t *b)
{
    double sigma = 0.5 / sqrt((double)nsamp);
    int64_t d = (int64_t)ceil(6. * sigma * nsamp) + 1;
    *a = nsamp / 2 - d; *b = nsamp / 2 + d;
    if (*a < 0) *a = 0;
    if (*b > nsamp - 1) *b = nsamp - 1;
}

/* keys_out[j] = radius of ray floor(j*num/nsamp) about the device centroid, j < nsamp */
int pxf_select_sample(const double *x, const double *y, int64_t num, const double *cxy_dev, int32_t nsamp,
                      double *keys_out, pxf_stream_t stream)
{
    if (num <= 0 || nsamp <= 0 || !x || !y || !cxy_dev || !keys_out) { set_error("pxf_select_sample: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_select_sample<<<grid_for(nsamp, PXF_BLOCK, 4), PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        x, y, num, cxy_dev, nsamp, keys_out);
    count_launch();
    return check_launch("k_select_sample");
}

/* One pass: counters[0] += #(r<lo), counters[1] += #(lo<=r<=hi) with those radii appended to
 * cand (capacity cap; overflow only counted), counters[2] += #NaN.  lohi_dev = the 4-double
 * output of pxf_select_finish on the sample ([1]=lo, [2]=hi).  counters: device uint64[4],
 * zeroed by the caller. */
int pxf_bracket_collect(const double *x, const double *y, int64_t num, const double *cxy_dev,
                        const double *lohi_dev, double *cand, int64_t cap, uint64_t *counters, pxf_stream_t stream)
{
    if (num < 0 || !cxy_dev || !lohi_dev || !cand || cap <= 0 || !counters) { set_error("pxf_bracket_collect: bad argument"); return PXF_ERR_INVALID; }
    if (num == 0) return PXF_OK;
    if (!x || !y) { set_error("pxf_bracket_collect: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const bool aligned = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
    unsigned long long *c = reinterpret_cast<unsigned long long *>(counters);
    if (aligned)
        k_bracket_collect<true><<<grid_for(((num + 1) >> 1) / COLLECT_U + 1, PXF_BLOCK, 4), PXF_BLOCK, 0, s>>>(x, y, num, cxy_dev, lohi_dev, cand, (unsigned long long)cap, c);
    else
        k_bracket_collect<false><<<grid_for(num / COLLECT_U + 1, PXF_BLOCK, 4), PXF_BLOCK, 0, s>>>(x, y, num, cxy_dev, lohi_dev, cand, (unsigned long long)cap, c);
    count_launch();
    return check_launch("k_bracket_collect");
}

/* Begin the select over the candidate buffers: ranks k0,k1 are GLOBAL ranks, counters the
 * (all-reduced) totals, cap_total the summed capacities (< 0: read it from counters[4], so a
 * sharded caller can all-reduce it together with the counters and never sync the host).
 * Marks the state invalid on a miss. */
int pxf_select_begin_bracket(void *state, int64_t k0, int64_t k1, const uint64_t *counters, int64_t cap_total,
                             pxf_stream_t stream)
{
    if (!state || k0 < 0 || k1 < k0 || !counters) { set_error("pxf_select_begin_bracket: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_select_begin_bracket<<<16, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        st_of(state), (unsigned long long)k0, (unsigned long long)k1, reinterpret_cast<const unsigned long long *>(counters),
        cap_total < 0 ? ~0ull : (unsigned long long)cap_total, hist_of(state), 2 * 8192, nan_of(state));
    count_launch();
    return check_launch("k_select_begin_bracket");
}

// pack = [count, sum x, sum y, count | x of nsamp strided rays | y of the same rays]: what one rank
// contributes to the all-gather that replaces "all-reduce the centroid sums" + "all-gather the sample"
__global__ void __launch_bounds__(PXF_BLOCK)
k_sample_pack(const double *__restrict__ x, const double *__restrict__ y, int64_t num, const double *__restrict__ sums,
              int nsamp, double *__restrict__ pack)
{
    if (blockIdx.x == 0 && threadIdx.x < 4) pack[threadIdx.x] = sums[threadIdx.x];
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < nsamp; j += gridDim.x * blockDim.x) {
        const int64_t i = num > 0 ? (int64_t)(((unsigned long long)j * (unsigned long long)num) / (unsigned long long)nsamp) : 0;
        pack[4 + j] = num > 0 ? x[i] : __longlong_as_double(0x7ff8000000000000ll);
        pack[4 + nsamp + j] = num > 0 ? y[i] : __longlong_as_double(0x7ff8000000000000ll);
    }
}
// gathered = world packs.  Every thread adds the per-rank sums in rank order (identical on every rank
// and every thread), thread 0 publishes the global sums and centroid, all compute the sample radii.
__global__ void __launch_bounds__(PXF_BLOCK)
k_sample_radii(const double *__restrict__ gathered, int world, int nsamp, double *__restrict__ sums_out,
               double *__restrict__ cxy, double *__restrict__ keys)
{
    const int stride = 4 + 2 * nsamp;
    double s0 = 0., s1 = 0., s2 = 0.;
    for (int r = 0; r < world; r++) {
        s0 += gathered[(size_t)r * stride];
        s1 += gathered[(size_t)r * stride + 1];
        s2 += gathered[(size_t)r * stride + 2];
    }
    const double cx = s1 / s0, cy = s2 / s0;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        sums_out[0] = s0; sums_out[1] = s1; sums_out[2] = s2; sums_out[3] = s0;
        cxy[0] = cx; cxy[1] = cy;
    }
    const int total = world * nsamp;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < total; j += gridDim.x * blockDim.x) {
        const int r = j / nsamp, q = j - r * nsamp;
        const double xs = gathered[(size_t)r * stride + 4 + q], ys = gathered[(size_t)r * stride + 4 + nsamp + q];
        keys[j] = sqrt(sq(xs - cx) + sq(ys - cy));
    }
}

int pxf_sample_pack(const double *x, const double *y, int64_t num, const double *sums_dev, int32_t nsamp,
                    double *pack_out, pxf_stream_t stream)
{
    if (num < 0 || nsamp <= 0 || (num > 0 && (!x || !y)) || !sums_dev || !pack_out) { set_error("pxf_sample_pack: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_sample_pack<<<grid_for(nsamp, PXF_BLOCK, 4), PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        x, y, num, sums_dev, nsamp, pack_out);
    count_launch();
    return check_launch("k_sample_pack");
}
int pxf_sample_radii(const double *gathered, int32_t world, int32_t nsamp, double *sums_out, double *cxy_out,
                     double *keys_out, pxf_stream_t stream)
{
    if (!gathered || world < 1 || nsamp <= 0 || !sums_out || !cxy_out || !keys_out) { set_error("pxf_sample_radii: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_sample_radii<<<grid_for((int64_t)world * nsamp, PXF_BLOCK, 4), PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        gathered, world, nsamp, sums_out, cxy_out, keys_out);
    count_launch();
    return check_launch("k_sample_radii");
}

/* ---- building blocks of the fused bracketed select, for callers that put a collective between
 * them (pyxfocus_b200/dist.py): sample -> all-gather -> pxf_small_select(3 passes) = bracket ->
 * pxf_bracket_collect -> all-reduce counters -> pxf_cand_hist -> all-reduce 4096 bins ->
 * pxf_cand_scan -> pxf_cand_gather -> all-gather -> pxf_small_select(5 passes) = exact pair. ---- */
size_t pxf_fastsel_bytes(void) { return sizeof(FastSel); }
int32_t pxf_fast_nbins(void) { return FAST_NBINS; }
int32_t pxf_fast_fincap(void) { return FAST_FINCAP; }

int pxf_small_select(const double *keys, const int32_t *seg_counts, int32_t nseg, int32_t seg_cap, int64_t ra, int64_t rb,
                     int32_t npass, const void *fastsel, double *out_dev, pxf_stream_t stream)
{
    if (!keys || nseg < 1 || seg_cap < 1 || (int64_t)nseg * seg_cap > (int64_t(1) << 24) || (npass != 3 && npass != 5) ||
        !out_dev || (!fastsel && (ra < 0 || rb < ra))) {
        set_error("pxf_small_select: bad argument");
        return PXF_ERR_INVALID;
    }
    int rc = need_device();
    if (rc) return rc;
    static bool smem_set[64] = {};
    if (first_on_device(smem_set))
        PXF_CUDA(cudaFuncSetAttribute(k_small_select, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 8192 * 4));
    k_small_select<<<1, 1024, 2 * 8192 * 4, reinterpret_cast<cudaStream_t>(stream)>>>(
        keys, seg_counts, nseg, seg_cap, (unsigned long long)ra, (unsigned long long)rb, npass,
        static_cast<const FastSel *>(fastsel), out_dev, nullptr, nullptr, nullptr);
    count_launch();
    return check_launch("k_small_select");
}

/* fhist (pxf_fast_nbins() uint32, zeroed by the caller) += this shard's candidates in linear bins over [lo,hi] */
int pxf_cand_hist(const double *cand, int64_t cap, const uint64_t *count_dev, const double *lohi_dev,
                  uint32_t *fhist, pxf_stream_t stream)
{
    if (!cand || cap < 1 || !count_dev || !lohi_dev || !fhist) { set_error("pxf_cand_hist: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_cand_hist<false><<<grid_for(cap, PXF_BLOCK * 8, 2), PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        cand, (unsigned long long)cap, reinterpret_cast<const unsigned long long *>(count_dev), nullptr, lohi_dev, 0ull, 0ull,
        fhist, nullptr);
    count_launch();
    return check_launch("k_cand_hist");
}

/* counters: the all-reduced [below, inside, nan, overflowed, capacity]; fhist: the all-reduced bins */
int pxf_cand_scan(const uint32_t *fhist, const uint64_t *counters, int64_t k0, int64_t k1, void *fastsel,
                  pxf_stream_t stream)
{
    if (!fhist || !counters || !fastsel || k0 < 0 || k1 < k0) { set_error("pxf_cand_scan: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_cand_scan<<<1, PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        fhist, reinterpret_cast<const unsigned long long *>(counters), (unsigned long long)k0, (unsigned long long)k1,
        static_cast<FastSel *>(fastsel));
    count_launch();
    return check_launch("k_cand_scan");
}

/* fin (pxf_fast_fincap() doubles) <- this shard's candidates in the chosen bins; *fin_count = how many
 * (more than the capacity = overflow, the final select then reports invalid) */
int pxf_cand_gather(const double *cand, int64_t cap, const uint64_t *count_dev, const double *lohi_dev, void *fastsel,
                    double *fin, int32_t *fin_count, pxf_stream_t stream)
{
    if (!cand || cap < 1 || !count_dev || !lohi_dev || !fastsel || !fin || !fin_count) { set_error("pxf_cand_gather: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_cand_finish<<<grid_for(cap, PXF_BLOCK * 8, 2), PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        cand, (unsigned long long)cap, reinterpret_cast<const unsigned long long *>(count_dev), lohi_dev,
        static_cast<FastSel *>(fastsel), fin, nullptr, fin_count);
    count_launch();
    return check_launch("k_cand_gather");
}

/* histogram pass over a key buffer whose length lives on the device (min(*count_dev, cap)) */
int pxf_select_hist_keys(const double *keys, int64_t cap, const uint64_t *count_dev, int32_t shift, int32_t bits,
                         void *state, pxf_stream_t stream)
{
    if (!state || !keys || cap <= 0 || bits < 1 || bits > 13 || shift < 0 || shift + bits > 64) {
        set_error("pxf_select_hist_keys: bad argument");
        return PXF_ERR_INVALID;
    }
    int rc = need_device();
    if (rc) return rc;
    return select_pass(nullptr, nullptr, keys, cap, reinterpret_cast<const unsigned long long *>(count_dev), nullptr,
                       shift, bits, st_of(state), hist_of(state), nullptr, reinterpret_cast<cudaStream_t>(stream));
}

// workspace layout of the device-side HPD
struct HpdWs {
    char *sums_scr; double *sums, *cxy, *lohi, *samp; void *stA, *stB; unsigned long long *counters; double *cand;
    int64_t cap;
    FastSel *fs; unsigned int *fhist; double *fin;
};
static size_t a256(size_t v) { return (v + 255) & ~(size_t)255; }
static size_t hpd_ws_carve(HpdWs &w, char *base, int64_t num)
{
    size_t off = 0;
    w.sums_scr = base + off; off += a256(pxf_sums_scratch_bytes());
    w.sums = (double *)(base + off); off += 256;
    w.cxy = (double *)(base + off); off += 256;
    w.lohi = (double *)(base + off); off += 256;
    w.counters = (unsigned long long *)(base + off); off += 256;
    w.stA = base + off; off += a256(pxf_select_state_bytes());
    w.stB = base + off; off += a256(pxf_select_state_bytes());
    w.samp = (double *)(base + off); off += a256((size_t)BRACKET_SAMPLES * 8);
    w.fs = (FastSel *)(base + off); off += a256(sizeof(FastSel));
    w.fhist = (unsigned int *)(base + off); off += a256((size_t)FAST_NBINS * 4);
    w.fin = (double *)(base + off); off += a256((size_t)FAST_FINCAP * 8);
    w.cap = num >= BRACKET_MIN_NUM ? pxf_bracket_capacity(num) : 0;
    w.cand = (double *)(base + off); off += a256((size_t)w.cap * 8);
    return off;
}
size_t pxf_hpd_workspace_bytes(int64_t num)
{
    HpdWs w;
    return hpd_ws_carve(w, nullptr, num < 0 ? 0 : num) + 256;
}

static int hpd_full(const double *x, const double *y, int64_t num, const double *cxy, void *state, double *out_dev,
                    pxf_stream_t stream)
{
    int rc;
    int64_t k0 = num > 0 ? (num - 1) / 2 : 0, k1 = num > 0 ? num / 2 : 0;
    if ((rc = pxf_select_begin(state, k0, k1, stream))) return rc;
    for (int p = 0; p < 5 && num > 0; p++) {
        if ((rc = pxf_select_hist(x, y, nullptr, num, cxy, kShift[p], kBits[p], state, stream))) return rc;
        if ((rc = pxf_select_narrow(kBits[p], state, stream))) return rc;
    }
    return pxf_select_finish(state, num, out_dev, stream);
}

/* Unweighted HPD entirely on the device.  out_dev: double[4] = {2*median, lower middle, upper
 * middle, valid}.  mode 0 = automatic (bracketed select for large bundles: one full pass
 * instead of five, small selects fused into single kernels), 1 = force the five-pass select,
 * 2 = the bracketed select built from the pass-wise entry points (what the multi-GPU driver
 * runs with all-reduces in between).  With mode 0/2 the caller must check out_dev[3]: 0 means
 * the bracket missed (probability ~1e-9) or ties overflowed a bin, and the call has to be
 * repeated with mode 1.  workspace: pxf_hpd_workspace_bytes(num). */
int pxf_hpd_from_sums_dev(const double *x, const double *y, int64_t num, const double *sums_dev, double *out_dev,
                          void *workspace, int32_t mode, pxf_stream_t stream);

int pxf_hpd_unweighted_dev(const double *x, const double *y, int64_t num, double *out_dev,
                           void *workspace, int32_t mode, pxf_stream_t stream)
{
    return pxf_hpd_from_sums_dev(x, y, num, nullptr, out_dev, workspace, mode, stream);
}

/* Same, with the centroid sums {count, sum x, sum y} already on the device (sums_dev, e.g. from
 * pxf_trace_program_sums); sums_dev == NULL computes them with one extra pass over x,y. */
int pxf_hpd_from_sums_dev(const double *x, const double *y, int64_t num, const double *sums_dev, double *out_dev,
                          void *workspace, int32_t mode, pxf_stream_t stream)
{
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    int rc = need_device();
    if (rc) return rc;
    if (num < 0 || !out_dev || !workspace || (num > 0 && (!x || !y))) { set_error("pxf_hpd_unweighted_dev: bad argument"); return PXF_ERR_INVALID; }
    HpdWs w;
    hpd_ws_carve(w, static_cast<char *>(workspace), num);
    if (!sums_dev) {
        if ((rc = sums_launch(PXF_SUMS_CENTROID, x, y, nullptr, nullptr, nullptr, nullptr, num, 0., 0., nullptr, w.sums, w.sums_scr, s)))
            return rc;
        sums_dev = w.sums;
    }
    int64_t ra, rb;
    pxf_bracket_sample_ranks(BRACKET_SAMPLES, &ra, &rb);
    if (mode == 0 && num >= BRACKET_MIN_NUM) {
        // single-GPU fast path (see k_bracket_small): 5 launches in all
        static bool smem_set[64] = {};
        if (first_on_device(smem_set))
            PXF_CUDA(cudaFuncSetAttribute(k_small_select, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 8192 * 4));
        k_select_sample_sums<<<grid_for(BRACKET_SAMPLES, PXF_BLOCK, 4), PXF_BLOCK, 0, s>>>(
            x, y, num, sums_dev, w.cxy, BRACKET_SAMPLES, w.samp);
        k_small_select<<<1, 1024, 2 * 8192 * 4, s>>>(w.samp, nullptr, 1, BRACKET_SAMPLES, (unsigned long long)ra,
                                                      (unsigned long long)rb, 3, nullptr, w.lohi, w.counters, w.fs, w.fhist);
        count_launch(2);
        if ((rc = check_launch("k_small_select"))) return rc;
        if ((rc = pxf_bracket_collect(x, y, num, w.cxy, w.lohi, w.cand, w.cap, reinterpret_cast<uint64_t *>(w.counters), stream))) return rc;
        const int g = grid_for(w.cap, PXF_BLOCK * 8, 2);     // few CTAs: each flushes a 4096-bin histogram
        k_cand_hist<true><<<g, PXF_BLOCK, 0, s>>>(w.cand, (unsigned long long)w.cap, w.counters + 1, w.counters, w.lohi,
                                                  (unsigned long long)((num - 1) / 2), (unsigned long long)(num / 2), w.fhist, w.fs);
        k_cand_finish<<<g, PXF_BLOCK, 0, s>>>(w.cand, (unsigned long long)w.cap, w.counters + 1, w.lohi, w.fs, w.fin, out_dev, nullptr);
        count_launch(2);
        return check_launch("k_cand_finish");
    }
    k_centroid_from_sums<<<1, 1, 0, s>>>(sums_dev, w.cxy);
    count_launch();
    if (mode == 1 || num < BRACKET_MIN_NUM) return hpd_full(x, y, num, w.cxy, w.stA, out_dev, stream);
    // mode 2: the pass-wise bracketed select (what the multi-GPU driver runs, with all-reduces between passes)
    // 1. bracket from a strided sample (exact select of two sample order statistics)
    if ((rc = pxf_select_sample(x, y, num, w.cxy, BRACKET_SAMPLES, w.samp, stream))) return rc;
    if ((rc = pxf_select_begin(w.stA, ra, rb, stream))) return rc;
    for (int p = 0; p < 5; p++) {
        if ((rc = pxf_select_hist(nullptr, nullptr, w.samp, BRACKET_SAMPLES, nullptr, kShift[p], kBits[p], w.stA, stream))) return rc;
        if ((rc = pxf_select_narrow(kBits[p], w.stA, stream))) return rc;
    }
    if ((rc = pxf_select_finish(w.stA, BRACKET_SAMPLES, w.lohi, stream))) return rc;
    // 2. one pass: count below, collect the bracket
    PXF_CUDA(cudaMemsetAsync(w.counters, 0, 64, s));
    if ((rc = pxf_bracket_collect(x, y, num, w.cxy, w.lohi, w.cand, w.cap, reinterpret_cast<uint64_t *>(w.counters), stream))) return rc;
    // 3. exact select among the candidates
    if ((rc = pxf_select_begin_bracket(w.stB, (num - 1) / 2, num / 2, reinterpret_cast<uint64_t *>(w.counters), w.cap, stream))) return rc;
    for (int p = 0; p < 5; p++) {
        if ((rc = pxf_select_hist_keys(w.cand, w.cap, reinterpret_cast<uint64_t *>(w.counters + 1), kShift[p], kBits[p], w.stB, stream))) return rc;
        if ((rc = pxf_select_narrow(kBits[p], w.stB, stream))) return rc;
    }
    return pxf_select_finish(w.stB, num, out_dev, stream);
}

/* analyses.hpd (unweighted) with the centroid sums optionally supplied on the device */
int pxf_hpd_with_sums(const double *x, const double *y, int64_t num, const double *sums_dev, double *hpd_host,
                      pxf_stream_t stream)
{
    if (num == 0 && hpd_host) { *hpd_host = __builtin_nan(""); return PXF_OK; }   // np.median([]) is nan
    if (num < 0 || !x || !y || !hpd_host) { set_error("pxf_hpd: bad argument"); return PXF_ERR_INVALID; }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    int rc = need_device();
    if (rc) return rc;
    Scratch sc;
    const size_t wb = pxf_hpd_workspace_bytes(num);
    if ((rc = sc.alloc(wb + 64, s))) return rc;
    double *out = reinterpret_cast<double *>((char *)sc.p + wb);
    double h[4];
    for (int mode = 0; mode < 2; mode++) {
        if ((rc = pxf_hpd_from_sums_dev(x, y, num, sums_dev, out, sc.p, mode, stream))) return rc;
        PXF_CUDA(cudaMemcpyAsync(h, out, sizeof(h), cudaMemcpyDeviceToHost, s));
        PXF_CUDA(cudaStreamSynchronize(s));
        if (h[3] != 0.) break;          // valid (always the case for mode 1)
    }
    *hpd_host = h[0];
    return PXF_OK;
}

int pxf_hpd(const double *x, const double *y, const double *w, int64_t num, double *hpd_host,
            pxf_stream_t stream)
{
    if (w) {
        if (num <= 0 || !x || !y || !hpd_host) { set_error("pxf_hpd: bad argument"); return PXF_ERR_INVALID; }
        return pxf_hpd_weighted(x, y, w, num, hpd_host, stream);
    }
    return pxf_hpd_with_sums(x, y, num, nullptr, hpd_host, stream);
}

// ---- compaction ---------------------------------------------------------------------------
size_t pxf_compact_scratch_bytes(int64_t num)
{
    int64_t ntiles = (num + CTILE - 1) / CTILE;
    if (ntiles < 1) ntiles = 1;
    // [offsets int64 x (ntiles+1)] [tile_count u32 x ntiles] [row table]
    return (size_t)(ntiles + 1) * 8 + (size_t)ntiles * 4 + 16 + sizeof(RowTable);
}

static inline long long *coff(const void *scratch) { return (long long *)scratch; }
static inline unsigned int *ccnt(const void *scratch, int64_t ntiles)
{
    return (unsigned int *)((char *)scratch + (size_t)(ntiles + 1) * 8);
}

int pxf_vignette_flags(const double *l, const double *m, const double *n, int64_t num,
                       uint8_t *flags, pxf_stream_t stream)
{
    if (num == 0) return PXF_OK;
    if (num < 0 || !l || !m || !n || !flags) { set_error("pxf_vignette_flags: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_vignette_flags<<<grid_for(num, PXF_BLOCK * 2, 8), PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        l, m, n, num, flags);
    count_launch();
    return check_launch("k_vignette_flags");
}

int pxf_compact_count(const uint8_t *flags, int64_t num, void *scratch, int64_t *count_host,
                      pxf_stream_t stream)
{
    if (num == 0 && count_host) { *count_host = 0; return PXF_OK; }
    if (num < 0 || !flags || !scratch || !count_host) { set_error("pxf_compact_count: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    int64_t ntiles = (num + CTILE - 1) / CTILE;
    k_compact_count<<<(unsigned)ntiles, PXF_BLOCK, 0, s>>>(flags, num, ccnt(scratch, ntiles));
    k_compact_scan<<<1, 1024, 0, s>>>(ccnt(scratch, ntiles), ntiles, coff(scratch));
    count_launch(2);
    if ((rc = check_launch("k_compact_count"))) return rc;
    long long total = 0;
    PXF_CUDA(cudaMemcpyAsync(&total, coff(scratch) + ntiles, 8, cudaMemcpyDeviceToHost, s));
    PXF_CUDA(cudaStreamSynchronize(s));
    *count_host = total;
    return PXF_OK;
}

int pxf_compact_scatter(const double *const *rows_in, double *const *rows_out, int32_t nrows,
                        const uint8_t *flags, int64_t num, const void *scratch, pxf_stream_t stream)
{
    if (num == 0) return PXF_OK;
    if (num < 0 || !rows_in || !rows_out || nrows < 1 || nrows > 16 || !flags || !scratch) {
        set_error("pxf_compact_scatter: bad argument");
        return PXF_ERR_INVALID;
    }
    int rc = need_device();
    if (rc) return rc;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    int64_t ntiles = (num + CTILE - 1) / CTILE;
    RowTable h;
    memset(&h, 0, sizeof(h));
    for (int r = 0; r < nrows; r++) { h.in[r] = rows_in[r]; h.out[r] = rows_out[r]; }
    k_compact_scatter<0><<<(unsigned)ntiles, PXF_BLOCK, 0, s>>>(h, nrows, flags, num, coff(scratch), nullptr);
    count_launch();
    return check_launch("k_compact_scatter");
}

int pxf_compact_indices(const uint8_t *flags, int64_t num, const void *scratch, int64_t *idx_out,
                        pxf_stream_t stream)
{
    if (num == 0) return PXF_OK;
    if (num < 0 || !flags || !scratch) { set_error("pxf_compact_indices: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    // idx_out may be NULL only if no ray survives (nothing is written then)
    int64_t ntiles = (num + CTILE - 1) / CTILE;
    RowTable none;
    memset(&none, 0, sizeof(none));
    k_compact_scatter<1><<<(unsigned)ntiles, PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        none, 0, flags, num, coff(scratch), reinterpret_cast<long long *>(idx_out));
    count_launch();
    return check_launch("k_compact_indices");
}

int pxf_gather_rows(const double *const *rows_in, double *const *rows_out, int32_t nrows,
                    const int64_t *idx, int64_t count, void *table_scratch /* >= 256 B device */,
                    pxf_stream_t stream)
{
    if (count < 0 || !rows_in || !rows_out || nrows < 1 || nrows > 16 || !idx || !table_scratch) {
        set_error("pxf_gather_rows: bad argument");
        return PXF_ERR_INVALID;
    }
    int rc = need_device();
    if (rc) return rc;
    if (count == 0) return PXF_OK;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    RowTable h;
    memset(&h, 0, sizeof(h));
    for (int r = 0; r < nrows; r++) { h.in[r] = rows_in[r]; h.out[r] = rows_out[r]; }
    (void)table_scratch;
    k_gather_rows<<<grid_for(count, PXF_BLOCK, 8), PXF_BLOCK, 0, s>>>(h, nrows, reinterpret_cast<const long long *>(idx), count);
    count_launch();
    return check_launch("k_gather_rows");
}

// ---- segmented bundles ------------------------------------------------------------------------
static int seg_args(int64_t num, const int64_t *seg_start_dev, int32_t nseg, const char *what)
{
    if (num < 0 || !seg_start_dev || nseg < 1) { set_error("%s: bad argument", what); return PXF_ERR_INVALID; }
    return need_device();
}

int pxf_segment_counts(const uint8_t *flags, int64_t num, const int64_t *seg_start_dev, int32_t nseg,
                       int64_t *counts_dev, pxf_stream_t stream)
{
    int rc = seg_args(num, seg_start_dev, nseg, "pxf_segment_counts");
    if (rc) return rc;
    if (!counts_dev || (num > 0 && !flags)) { set_error("pxf_segment_counts: bad argument"); return PXF_ERR_INVALID; }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    PXF_CUDA(cudaMemsetAsync(counts_dev, 0, (size_t)nseg * 8, s));
    if (num == 0) return PXF_OK;
    k_seg_counts<<<grid_for(num, SEGSUM_TILE, 4), PXF_BLOCK, 0, s>>>(flags, num, reinterpret_cast<const long long *>(seg_start_dev),
                                                                    nseg, reinterpret_cast<unsigned long long *>(counts_dev));
    count_launch();
    return check_launch("k_seg_counts");
}

size_t pxf_sums_segmented_scratch_bytes(int64_t num, int32_t nseg)
{
    const int64_t ntiles = (num > 0 ? num : 0) / SEGSUM_TILE + 1;
    return (size_t)(ntiles + (nseg > 0 ? nseg : 0)) * NSUM * sizeof(double);
}

int pxf_sums_segmented(int32_t mode, const double *x, const double *y, const double *z, const double *l, const double *m,
                       const double *n, const double *w, int64_t num, const int64_t *seg_start_dev, int32_t nseg,
                       const double *ab_dev, double *out_dev, void *scratch, pxf_stream_t stream)
{
    int rc = seg_args(num, seg_start_dev, nseg, "pxf_sums_segmented");
    if (rc) return rc;
    const bool ip = mode == PXF_SUMS_IMAGEPLANE || mode == PXF_SUMS_IMAGEPLANE_Z;
    const bool zz = mode == PXF_SUMS_IMAGEPLANE_Z || mode == PXF_SUMS_POINT;
    if (!out_dev || !scratch || (num > 0 && (!x || !y || (ip && (!l || !m || !n)) || (zz && !z))) ||
        ((mode == PXF_SUMS_RMS || mode == PXF_SUMS_POINT) && !ab_dev) || mode < PXF_SUMS_CENTROID || mode > PXF_SUMS_POINT) {
        set_error("pxf_sums_segmented: bad argument");
        return PXF_ERR_INVALID;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const long long *ss = reinterpret_cast<const long long *>(seg_start_dev);
    double *partial = static_cast<double *>(scratch);
    const int ns = mode == PXF_SUMS_CENTROID ? 4 : ((mode == PXF_SUMS_RMS || mode == PXF_SUMS_POINT) ? 2 : 9);
    if (num > 0) {
        uintptr_t al = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(w);
        if (zz) al |= reinterpret_cast<uintptr_t>(z);
        if (ip) al |= reinterpret_cast<uintptr_t>(l) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(n);
        const bool v2 = (al & 15) == 0;
        const int grid = grid_for(num, SEGSUM_TILE, 4);
#define PXF_SEGSUMS_GO(M)                                                                                          \
        do {                                                                                                       \
            if (v2) k_sums_seg<M, true><<<grid, PXF_BLOCK, 0, s>>>(x, y, z, l, m, n, w, num, ss, nseg, ab_dev, partial);   \
            else k_sums_seg<M, false><<<grid, PXF_BLOCK, 0, s>>>(x, y, z, l, m, n, w, num, ss, nseg, ab_dev, partial);    \
        } while (0)
        if (mode == PXF_SUMS_CENTROID) PXF_SEGSUMS_GO(PXF_SUMS_CENTROID);
        else if (mode == PXF_SUMS_RMS) PXF_SEGSUMS_GO(PXF_SUMS_RMS);
        else if (mode == PXF_SUMS_IMAGEPLANE) PXF_SEGSUMS_GO(PXF_SUMS_IMAGEPLANE);
        else if (mode == PXF_SUMS_IMAGEPLANE_Z) PXF_SEGSUMS_GO(PXF_SUMS_IMAGEPLANE_Z);
        else PXF_SEGSUMS_GO(PXF_SUMS_POINT);
#undef PXF_SEGSUMS_GO
        count_launch();
    }
    k_sums_seg_fold<<<nseg, PXF_BLOCK, 0, s>>>(partial, ss, ns, out_dev);
    count_launch();
    return check_launch("k_sums_seg");
}

int pxf_centroids_segmented(const double *sums_dev, int32_t nseg, double *cxy_dev, pxf_stream_t stream)
{
    if (!sums_dev || !cxy_dev || nseg < 1) { set_error("pxf_centroids_segmented: bad argument"); return PXF_ERR_INVALID; }
    int rc = need_device();
    if (rc) return rc;
    k_centroids_seg<<<grid_for(nseg, PXF_BLOCK, 4), PXF_BLOCK, 0, reinterpret_cast<cudaStream_t>(stream)>>>(sums_dev, nseg, cxy_dev);
    count_launch();
    return check_launch("k_centroids_seg");
}

struct HpdSegWs { double *cxy, *lohi, *cand; unsigned long long *counters; int *state; void *fallback; };
static size_t hpdseg_carve(HpdSegWs &w, char *base, int64_t num, int32_t nseg)
{
    size_t off = 0;
    w.cxy = (double *)(base + off); off += a256((size_t)nseg * 16);
    w.lohi = (double *)(base + off); off += a256((size_t)nseg * 16);
    w.counters = (unsigned long long *)(base + off); off += a256((size_t)nseg * 24);
    w.state = (int *)(base + off); off += a256((size_t)nseg * 4);
    w.fallback = base + off; off += a256(pxf_hpd_workspace_bytes(0));
    w.cand = (double *)(base + off); off += a256((size_t)(num / SEG_CAND_DIV + 1) * 8);
    return off;
}

size_t pxf_hpd_segmented_workspace_bytes(int64_t num, int32_t nseg, int32_t weighted)
{
    HpdSegWs w;
    if (num < 0) num = 0;
    if (nseg < 1) nseg = 1;
    if (weighted) return hpd_weighted_segmented_bytes(num) + 256;
    return hpdseg_carve(w, nullptr, num, nseg) + 256;
}

int pxf_hpd_segmented(const double *x, const double *y, const double *w, int64_t num, const int64_t *seg_start_dev,
                      int32_t nseg, const double *sums_dev, double *out_dev, void *workspace, int32_t mode,
                      pxf_stream_t stream)
{
    int rc = seg_args(num, seg_start_dev, nseg, "pxf_hpd_segmented");
    if (rc) return rc;
    if (!sums_dev || !out_dev || !workspace || (num > 0 && (!x || !y)) || (mode != 0 && mode != 1)) {
        set_error("pxf_hpd_segmented: bad argument");
        return PXF_ERR_INVALID;
    }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const long long *ss = reinterpret_cast<const long long *>(seg_start_dev);
    if (w) return hpd_weighted_segmented(x, y, w, num, ss, nseg, sums_dev, out_dev, workspace, s);
    HpdSegWs ws;
    hpdseg_carve(ws, static_cast<char *>(workspace), num, nseg);
    if (mode == 1) {
        // every segment through the five-pass select on its slice (reads the layout back: a testing aid)
        int64_t *hs = static_cast<int64_t *>(malloc((size_t)(nseg + 1) * 8));
        if (!hs) { set_error("pxf_hpd_segmented: out of host memory"); return PXF_ERR_INVALID; }
        cudaError_t e = cudaMemcpyAsync(hs, seg_start_dev, (size_t)(nseg + 1) * 8, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) { free(hs); set_error("pxf_hpd_segmented: %s", cudaGetErrorString(e)); return PXF_ERR_CUDA; }
        for (int sg = 0; sg < nseg && rc == 0; sg++) {
            const int64_t a = hs[sg], cnt = hs[sg + 1] - hs[sg];
            rc = pxf_hpd_from_sums_dev(cnt > 0 ? x + a : x, cnt > 0 ? y + a : y, cnt, sums_dev + 16 * (int64_t)sg,
                                       out_dev + 4 * (int64_t)sg, ws.fallback, 1, stream);
        }
        free(hs);
        return rc;
    }
    static bool smem_set[64] = {};
    if (first_on_device(smem_set)) {
        PXF_CUDA(cudaFuncSetAttribute(k_hpdseg_prepare, cudaFuncAttributeMaxDynamicSharedMemorySize, SEG_DIRECT * 8));
        PXF_CUDA(cudaFuncSetAttribute(k_hpdseg_finish, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      SEG_FINCAP * 8 + FAST_NBINS * 4));
    }
    int64_t ra, rb;
    pxf_bracket_sample_ranks(SEG_DIRECT, &ra, &rb);
    k_hpdseg_prepare<<<nseg, 1024, SEG_DIRECT * 8, s>>>(x, y, ss, sums_dev, (int)ra, (int)rb, ws.cxy, ws.lohi, ws.counters,
                                                         ws.state, out_dev);
    count_launch();
    if (num > 0) {
        const bool v2 = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
        const int grid = grid_for(num, SEGCOL_TILE, 4);
        if (v2) k_hpdseg_collect<true><<<grid, PXF_BLOCK, 0, s>>>(x, y, num, ss, nseg, ws.state, ws.cxy, ws.lohi, ws.cand, ws.counters);
        else k_hpdseg_collect<false><<<grid, PXF_BLOCK, 0, s>>>(x, y, num, ss, nseg, ws.state, ws.cxy, ws.lohi, ws.cand, ws.counters);
        count_launch();
    }
    k_hpdseg_finish<<<nseg, 1024, SEG_FINCAP * 8 + FAST_NBINS * 4, s>>>(ss, ws.state, ws.counters, ws.lohi, ws.cand, out_dev);
    count_launch();
    return check_launch("pxf_hpd_segmented");
}

}  // extern "C"
