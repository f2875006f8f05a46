// Hand-written stable LSD radix sort (8-bit digits) of fp64 keys with an index payload, the
// gathered inclusive scan, and the weighted-HPD reduction built on them
// (analyses.rhocdf / hpd weighted branch, analyses.py:73-97: argsort -> cumsum -> argmin).
//
// Sort: one-sweep passes.  k_sort_hist_all histograms all eight key bytes in one read of the
// input; k_sort_plan (one CTA) turns the histograms into per-pass digit bases, drops the passes
// on constant bytes and fixes the ping-pong order on the device (nothing is read back); every
// remaining pass is ONE kernel, k_onesweep: a tile of keys is ranked in shared memory (ranks
// inside a 32-key slice from eight ballots, stable), its digit counts are published and the
// counts of all earlier tiles are summed by a decoupled look-back, and the tile is written out
// digit run by digit run.  The first pass converts the doubles and synthesises the indices, the
// last pass writes doubles and int64 indices.
// Scan: the array is cut into G contiguous chunks, one CTA per chunk: chunk sums, one-CTA scan,
// rescan.
#include "pxf_internal.h"
#include "pxf_ray.cuh"

namespace pxf {

#define SORT_THREADS 256
#define SORT_WARPS (SORT_THREADS / 32)
#define SORT_ITEMS 8                       // 32-key slices per warp per tile
#define SORT_TILE (SORT_THREADS * SORT_ITEMS)
#define SORT_MAXG 1024

typedef unsigned long long u64;
typedef unsigned int u32;

// np.sort order: -inf < ... < -0 == +0 < ... < +inf < NaN (all NaNs last, equal among themselves); a stable sort
// keeps the input order of keys that compare equal, so -0 and +0 share one key, as do all NaNs (the sorted-key
// output re-reads the original value for those, see SortPlan::gather)
PXF_DEV u64 sort_key(double v)
{
    if (v != v) return ~0ull;
    u64 b = (u64)__double_as_longlong(v);
    if (b == 0x8000000000000000ull) b = 0;
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
PXF_DEV bool sort_key_lossy(double v) { return v != v || (u64)__double_as_longlong(v) == 0x8000000000000000ull; }
PXF_DEV double unsort_key(u64 k, double nanv)
{
    if (k == ~0ull) return nanv;
    u64 b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

struct Chunking { int64_t num; int64_t per; int G; };   // chunk g = [g*per, min(num,(g+1)*per)), per % SORT_TILE == 0

// ------------------------------------------------------------------ one-sweep LSD passes
// One up-front pass histograms all eight digits of every key (8 B/key read, nothing written); a one-CTA plan
// kernel turns the histograms into per-pass digit bases, drops the digits that are constant over the array and
// fixes the ping-pong order on the device (no read-back).  Each remaining pass is ONE kernel: a tile of
// OS_TILE keys is ranked in shared memory, its digit counts are published, the tile's global offsets come from
// a decoupled look-back over the preceding tiles' published counts (tiles are handed out by a ticket counter, so
// every predecessor is already running), and the tile is written out digit run by digit run.  The first pass
// converts the doubles and synthesises the indices, the last one writes doubles and int64 indices: 8 + 20 +
// 24 (passes-2) + 28 B/key instead of 32 B/key/pass + 48.
#define OS_LOOKBACK 16
#define OS_FLAG_SHIFT 56
#define OS_VALUE_MASK ((1ull << OS_FLAG_SHIFT) - 1)

struct SortPlan {
    u64 base[8][256];      // exclusive scan of digit d's histogram
    int active[8];         // pass on digit d runs
    int src[8];            // 0: reads buffer A, 1: reads buffer B (ignored by the first pass)
    int first[8], last[8];
    int npass;
    int gather;            // some key is -0 or NaN: the sorted keys are re-read from the input by index
    unsigned ticket[8];    // next tile of pass d
};

__global__ void __launch_bounds__(SORT_THREADS)
k_sort_hist_all(const double *__restrict__ in, int64_t num, u64 *__restrict__ ghist /*[8][256]*/)
{
    __shared__ u32 sh[8 * 256];
    for (int t = threadIdx.x; t < 8 * 256; t += blockDim.x) sh[t] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    // whole warps stay in the loop together (the match below is warp-wide)
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < num; i0 += 4 * nthr) {
        u64 k[4];
        bool in_range[4];
        bool lossy = false;
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int64_t i = i0 + u * nthr + lane;
            in_range[u] = i0 + u * nthr < num && i < num;
            const double v = in_range[u] ? in[i] : 0.;
            k[u] = in_range[u] ? sort_key(v) : 0ull;
            lossy = lossy || sort_key_lossy(v);
        }
        if (lossy) ghist[8 * 256] = 1;
#pragma unroll
        for (int u = 0; u < 4; u++) {
            if (i0 + u * nthr >= num) break;
            // the top two bytes (sign, exponent, four mantissa bits) take few values: one atomic per warp when
            // the warp agrees, instead of 32 serialised ones on a single address
            const unsigned act = __ballot_sync(0xffffffffu, in_range[u]);
            const unsigned top = (unsigned)(k[u] >> 48);
            const bool same = act == 0xffffffffu && __all_sync(0xffffffffu, top == __shfl_sync(0xffffffffu, top, 0));
            if (same) {
                if (lane == 0) { atomicAdd(&sh[7 * 256 + (top >> 8)], 32u); atomicAdd(&sh[6 * 256 + (top & 255)], 32u); }
            } else if (in_range[u]) {
                atomicAdd(&sh[7 * 256 + (top >> 8)], 1u);
                atomicAdd(&sh[6 * 256 + (top & 255)], 1u);
            }
            if (in_range[u]) {
#pragma unroll
                for (int d = 0; d < 6; d++) atomicAdd(&sh[d * 256 + (int)((k[u] >> (8 * d)) & 255)], 1u);
            }
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 8 * 256; t += blockDim.x)
        if (sh[t]) atomicAdd(&ghist[t], (u64)sh[t]);
}

// digits: 0 = skip every digit that is constant over the array, else the caller's mask
__global__ void __launch_bounds__(256) k_sort_plan(const u64 *__restrict__ ghist, int64_t num, int digits, SortPlan *plan)
{
    __shared__ u64 wsum[8];
    __shared__ int trivial[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 8) trivial[threadIdx.x] = 0;
    __syncthreads();
    for (int d = 0; d < 8; d++) {
        const u64 v = ghist[d * 256 + threadIdx.x];
        if (v == (u64)num) trivial[d] = 1;
        u64 incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            u64 t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        u64 b = 0;
        for (int q = 0; q < warp; q++) b += wsum[q];
        plan->base[d][threadIdx.x] = b + incl - v;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int np = 0, lastd = -1;
        for (int d = 0; d < 8; d++) {
            const int on = digits ? (digits >> d) & 1 : !trivial[d];
            plan->active[d] = on;
            plan->first[d] = on && np == 0;
            plan->last[d] = 0;
            plan->src[d] = np >= 1 ? (np - 1) & 1 : 0;     // pass 0 writes A, pass 1 reads A writes B, ...
            plan->ticket[d] = 0;
            if (on) { np++; lastd = d; }
        }
        if (lastd >= 0) plan->last[lastd] = 1;
        plan->npass = np;
        plan->gather = ghist[8 * 256] != 0;
    }
}

PXF_DEV u64 os_ld(const u64 *p) { return *reinterpret_cast<const volatile u64 *>(p); }
PXF_DEV void os_st(u64 *p, u64 v) { *reinterpret_cast<volatile u64 *>(p) = v; }

template <int OS_THREADS, int OS_ITEMS>
struct OsSmem {
    static constexpr int OS_TILE = OS_THREADS * OS_ITEMS, OS_WARPS = OS_THREADS / 32;
    u64 sk[OS_TILE];                  // the tile, sorted by digit
    u32 sv[OS_TILE];
    u32 whist[OS_WARPS][256];         // per-warp digit counts, then exclusive offsets over warps
    u64 run[256];                     // global position of the tile's first key of each digit
    u32 tbase[256];                   // position of each digit's run inside the sorted tile
    u32 twarp[8];
    unsigned tile;
};

// byte d (0..7) of a 64-bit key
PXF_DEV int key_byte(u64 k, unsigned sel) { return (int)(__byte_perm((u32)k, (u32)(k >> 32), sel) & 255u); }

// FULL: the tile has OS_TILE keys (no bounds checks, loads at constant offsets from one base address)
template <int OS_THREADS, int OS_ITEMS, bool FULL>
PXF_DEV void onesweep_tile(OsSmem<OS_THREADS, OS_ITEMS> &sm, const double *__restrict__ in, const u64 *__restrict__ kin,
                           const u32 *__restrict__ vin, u64 *__restrict__ kout, u32 *__restrict__ vout,
                           double *__restrict__ keys_out, long long *__restrict__ idx_out, const int64_t num, const int d,
                           const bool first, const bool last, const SortPlan *__restrict__ plan,
                           u64 *__restrict__ status, const int64_t tile)
{
    constexpr int OS_TILE = OS_THREADS * OS_ITEMS, OS_WARPS = OS_THREADS / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned sel = (unsigned)d;
    const int64_t t0 = tile * OS_TILE;
    const int cnt = FULL ? OS_TILE : (int)(num - t0);
    const int wofs = warp * (32 * OS_ITEMS) + lane;        // this lane's first key inside the tile
    u64 k[OS_ITEMS];
    u32 rank[OS_ITEMS];
    // warp w owns tile elements [w*32*ITEMS, (w+1)*32*ITEMS) as ITEMS consecutive 32-key slices
    if (first) {
        const double *p = in + t0 + wofs;
#pragma unroll
        for (int j = 0; j < OS_ITEMS; j++) k[j] = (FULL || wofs + j * 32 < cnt) ? sort_key(p[j * 32]) : ~0ull;
    } else {
        const u64 *p = kin + t0 + wofs;
#pragma unroll
        for (int j = 0; j < OS_ITEMS; j++) k[j] = (FULL || wofs + j * 32 < cnt) ? p[j * 32] : ~0ull;
    }
    u32 *wh = sm.whist[warp];
#pragma unroll
    for (int j = 0; j < OS_ITEMS; j++) {
        const bool valid = FULL || wofs + j * 32 < cnt;
        const int dd = key_byte(k[j], sel);
        // lanes holding the same digit: eight ballots (match.any runs at a few hundred cycles per warp on this part:
        // the first version of this kernel spent most of its time in it, profiles/r02_notes.md)
        unsigned peers = FULL ? 0xffffffffu : __ballot_sync(0xffffffffu, valid);
#pragma unroll
        for (int b = 0; b < 8; b++) {
            const bool bit = (dd >> b) & 1;
            const unsigned m = __ballot_sync(0xffffffffu, bit);
            peers &= bit ? m : ~m;
        }
        if (!FULL && !valid) peers = 1u << lane;
        // every lane reads its digit's running count (lanes of one digit read one word: a broadcast), then the first
        // lane of each group adds the group's size -- the load precedes the store in the warp's instruction order
        const u32 base = wh[dd];
        __syncwarp();
        if (valid && lane == __ffs(peers) - 1) wh[dd] = base + __popc(peers);
        rank[j] = base + __popc(peers & ((1u << lane) - 1));
        __syncwarp();
    }
    __syncthreads();
    // thread dg = digit dg: counts over warps -> exclusive offsets over warps, tile total acc; the total is
    // published at once so that later tiles can add it while this one is still staging
    const int dg = threadIdx.x;
    const u64 aggf = (u64)(2 * d + 3), incf = aggf + 1;
    u64 *mine = status + (size_t)tile * 256 + (dg & 255);
    u32 acc = 0, total = 0;
    if (dg < 256) {
#pragma unroll
        for (int w = 0; w < OS_WARPS; w++) {
            const u32 c = sm.whist[w][dg];
            sm.whist[w][dg] = acc;
            acc += c;
        }
        total = acc;
        os_st(mine, ((tile == 0 ? incf : aggf) << OS_FLAG_SHIFT) | (u64)acc);
        // where each digit's run starts inside the tile once it is sorted by digit
        u32 incl = acc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            u32 t_ = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t_;
        }
        if (lane == 31) sm.twarp[warp] = incl;
        acc = incl - acc;                     // exclusive within the warp's 32 digits
    }
    __syncthreads();
    if (dg < 256) {
        u32 b = 0;
        for (int q = 0; q < warp; q++) b += sm.twarp[q];
        sm.tbase[dg] = b + acc;
    }
    __syncthreads();
    // stage the tile in shared memory in digit order; the payload goes straight from global memory to its slot
#pragma unroll
    for (int j = 0; j < OS_ITEMS; j++) {
        if (FULL || wofs + j * 32 < cnt) {
            const int dd = key_byte(k[j], sel);
            rank[j] += sm.tbase[dd] + wh[dd];
            sm.sk[rank[j]] = k[j];
        }
    }
    if (first) {
#pragma unroll
        for (int j = 0; j < OS_ITEMS; j++)
            if (FULL || wofs + j * 32 < cnt) sm.sv[rank[j]] = (u32)(t0 + wofs + j * 32);
    } else {
        const u32 *p = vin + t0 + wofs;
#pragma unroll
        for (int j = 0; j < OS_ITEMS; j++)
            if (FULL || wofs + j * 32 < cnt) sm.sv[rank[j]] = p[j * 32];
    }
    // look back for the number of keys of digit dg in all earlier tiles
    if (dg < 256) {
        u64 excl = 0;
        if (tile != 0) {
            int64_t t = tile - 1;
            for (;;) {
                u64 sw[OS_LOOKBACK];
#pragma unroll
                for (int u = 0; u < OS_LOOKBACK; u++)
                    sw[u] = t - u >= 0 ? os_ld(status + (size_t)(t - u) * 256 + dg) : 0ull;
                bool done = false;
#pragma unroll
                for (int u = 0; u < OS_LOOKBACK; u++) {
                    if (done || t - u < 0) break;
                    u64 w_ = sw[u];
                    while ((w_ >> OS_FLAG_SHIFT) < aggf) w_ = os_ld(status + (size_t)(t - u) * 256 + dg);
                    excl += w_ & OS_VALUE_MASK;
                    if ((w_ >> OS_FLAG_SHIFT) == incf) done = true;
                }
                if (done) break;
                t -= OS_LOOKBACK;
            }
            os_st(mine, (incf << OS_FLAG_SHIFT) | (excl + (u64)total));
        }
        // destination of tile position p of digit dg: run[dg] + p, with the tile-local start folded in
        sm.run[dg] = plan->base[d][dg] + excl - (u64)sm.tbase[dg];
    }
    __syncthreads();
    // write the tile out position by position: keys of one digit are consecutive in the tile AND at their
    // destination, so a warp's store covers a few contiguous runs instead of 32 scattered keys
    if (last) {
        const double nanv = __longlong_as_double(0x7ff8000000000000ll);
        const bool gather = plan->gather != 0;
#pragma unroll 4
        for (int p = threadIdx.x; p < cnt; p += OS_THREADS) {
            const u64 kk = sm.sk[p];
            const u64 dst = sm.run[key_byte(kk, sel)] + (u32)p;
            const u32 vv = sm.sv[p];
            if (keys_out) keys_out[dst] = gather ? in[vv] : unsort_key(kk, nanv);
            if (idx_out) idx_out[dst] = (long long)vv;
        }
    } else {
#pragma unroll 4
        for (int p = threadIdx.x; p < cnt; p += OS_THREADS) {
            const u64 kk = sm.sk[p];
            const u64 dst = sm.run[key_byte(kk, sel)] + (u32)p;
            kout[dst] = kk;
            vout[dst] = sm.sv[p];
        }
    }
}

template <int OS_THREADS, int OS_ITEMS, int OS_MINB>
__global__ void __launch_bounds__(OS_THREADS, OS_MINB)
k_onesweep(const double *__restrict__ in, u64 *__restrict__ kA, u64 *__restrict__ kB, u32 *__restrict__ vA,
           u32 *__restrict__ vB, double *__restrict__ keys_out, long long *__restrict__ idx_out, int64_t num, int d,
           SortPlan *__restrict__ plan, u64 *__restrict__ status /*[tiles][256]*/)
{
    if (!plan->active[d]) return;
    constexpr int OS_TILE = OS_THREADS * OS_ITEMS;
    extern __shared__ __align__(16) unsigned char os_raw[];
    OsSmem<OS_THREADS, OS_ITEMS> &sm = *reinterpret_cast<OsSmem<OS_THREADS, OS_ITEMS> *>(os_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool first = plan->first[d] != 0, last = plan->last[d] != 0;
    const bool fromB = plan->src[d] != 0;
    const u64 *kin = fromB ? kB : kA;
    const u32 *vin = fromB ? vB : vA;
    u64 *kout = first ? kA : (fromB ? kA : kB);
    u32 *vout = first ? vA : (fromB ? vA : vB);
    if (threadIdx.x == 0) sm.tile = atomicAdd(&plan->ticket[d], 1u);
#pragma unroll
    for (int q = 0; q < 256 / 32; q++) sm.whist[warp][q * 32 + lane] = 0;
    __syncthreads();
    const int64_t tile = sm.tile;
    if ((tile + 1) * OS_TILE <= num)
        onesweep_tile<OS_THREADS, OS_ITEMS, true>(sm, in, kin, vin, kout, vout, keys_out, idx_out, num, d, first, last, plan,
                                                  status, tile);
    else
        onesweep_tile<OS_THREADS, OS_ITEMS, false>(sm, in, kin, vin, kout, vout, keys_out, idx_out, num, d, first, last, plan,
                                                   status, tile);
}

// every digit constant (all keys equal, or a single key): the order is the input order
__global__ void __launch_bounds__(SORT_THREADS)
k_sort_identity(const double *__restrict__ in, int64_t num, const SortPlan *__restrict__ plan,
                double *__restrict__ keys_out, long long *__restrict__ idx_out)
{
    if (plan->npass != 0) return;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    const double nanv = __longlong_as_double(0x7ff8000000000000ll);
    (void)nanv;
    for (int64_t i = tid; i < num; i += nthr) {
        if (keys_out) keys_out[i] = in[i];
        if (idx_out) idx_out[i] = (long long)i;
    }
}

// ------------------------------------------------------------------ gathered inclusive scan
// out[i] = sum_{j<=i} (w ? w[idx[j]] : 1).  Same chunking: chunk sums, one-CTA scan, rescan.
__global__ void __launch_bounds__(SORT_THREADS)
k_scan_chunk_sums(const double *__restrict__ w, const long long *__restrict__ idx, Chunking ck,
                  double *__restrict__ csum)
{
    __shared__ double sh[SORT_WARPS];
    const int64_t lo = (int64_t)blockIdx.x * ck.per;
    const int64_t hi = lo + ck.per < ck.num ? lo + ck.per : ck.num;
    double acc = 0.;
    for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) acc += w ? w[idx ? idx[i] : i] : 1.;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.;
        for (int q = 0; q < SORT_WARPS; q++) t += sh[q];
        csum[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024) k_scan_chunk_offsets(double *__restrict__ csum, int G)
{
    // serial exclusive scan of <= 1024 chunk sums (left-to-right like np.cumsum), staged through shared
    // memory so that the one scanning thread does not chain G global-memory round trips
    __shared__ double sh[SORT_MAXG + 1];
    for (int g = threadIdx.x; g < G; g += blockDim.x) sh[g] = csum[g];
    __syncthreads();
    if (threadIdx.x == 0) {
        double run = 0.;
        for (int g = 0; g < G; g++) { double t = sh[g]; sh[g] = run; run += t; }
        sh[G] = run;
    }
    __syncthreads();
    for (int g = threadIdx.x; g <= G; g += blockDim.x) csum[g] = sh[g];
}

__global__ void __launch_bounds__(SORT_THREADS)
k_scan_apply(const double *__restrict__ w, const long long *__restrict__ idx, Chunking ck,
             const double *__restrict__ csum, double *__restrict__ out)
{
    __shared__ double wtot[SORT_WARPS];
    __shared__ double carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = csum[blockIdx.x];
    __syncthreads();
    const int64_t lo = (int64_t)blockIdx.x * ck.per;
    const int64_t hi = lo + ck.per < ck.num ? lo + ck.per : ck.num;
    for (int64_t t0 = lo; t0 < hi; t0 += SORT_THREADS) {
        const int64_t i = t0 + threadIdx.x;
        double v = 0.;
        if (i < hi) v = w ? w[idx ? idx[i] : i] : 1.;
        double incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            double t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wtot[warp] = incl;
        __syncthreads();
        double base = carry;
        for (int q = 0; q < warp; q++) base += wtot[q];
        if (i < hi) out[i] = base + incl;
        __syncthreads();
        if (threadIdx.x == SORT_THREADS - 1) carry = base + incl;
        __syncthreads();
    }
}

// ------------------------------------------------------------------ argmin |cdf/max - q|
// np.argmin returns the first minimiser; NaN handling follows numpy (first NaN wins).
struct ArgMin { double v; long long i; };
PXF_DEV bool am_better(double v, long long i, double bv, long long bi)
{
    const bool vn = v != v, bn = bv != bv;
    if (vn || bn) { if (vn && bn) return i < bi; return vn; }
    return v < bv || (v == bv && i < bi);
}

__global__ void __launch_bounds__(SORT_THREADS)
k_cdf_argmin(const double *__restrict__ cdf, int64_t num, const double *__restrict__ maxv_ptr, double q0, double q1,
             ArgMin *__restrict__ partial /*[grid][2]*/)
{
    const double mx = *maxv_ptr;
    double bv[2] = {__longlong_as_double(0x7ff0000000000000ll), __longlong_as_double(0x7ff0000000000000ll)};
    long long bi[2] = {0x7fffffffffffffffll, 0x7fffffffffffffffll};
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < num; i += nthr) {
        const double c = cdf[i] / mx;
        const double d0 = fabs(c - q0), d1 = fabs(c - q1);
        if (am_better(d0, i, bv[0], bi[0])) { bv[0] = d0; bi[0] = i; }
        if (am_better(d1, i, bv[1], bi[1])) { bv[1] = d1; bi[1] = i; }
    }
    __shared__ double shv[2][SORT_WARPS];
    __shared__ long long shi[2][SORT_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < 2; c++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double ov = __shfl_down_sync(0xffffffffu, bv[c], o);
            long long oi = __shfl_down_sync(0xffffffffu, bi[c], o);
            if (am_better(ov, oi, bv[c], bi[c])) { bv[c] = ov; bi[c] = oi; }
        }
        if (lane == 0) { shv[c][warp] = bv[c]; shi[c][warp] = bi[c]; }
    }
    __syncthreads();
    if (threadIdx.x < 2) {
        const int c = threadIdx.x;
        double v = shv[c][0];
        long long i = shi[c][0];
        for (int w = 1; w < SORT_WARPS; w++)
            if (am_better(shv[c][w], shi[c][w], v, i)) { v = shv[c][w]; i = shi[c][w]; }
        partial[blockIdx.x * 2 + c].v = v;
        partial[blockIdx.x * 2 + c].i = i;
    }
}

// cdf.max(): numpy max propagates NaN
__global__ void __launch_bounds__(SORT_THREADS)
k_max_partial(const double *__restrict__ a, int64_t num, double *__restrict__ partial)
{
    double m = -__longlong_as_double(0x7ff0000000000000ll);
    bool nan = false;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < num; i += nthr) {
        double v = a[i];
        if (v != v) nan = true;
        else if (v > m) m = v;
    }
    if (nan) m = __longlong_as_double(0x7ff8000000000000ll);
    __shared__ double sh[SORT_WARPS];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ov = __shfl_down_sync(0xffffffffu, m, o);
        if (ov != ov || (m == m && ov > m)) m = ov;
    }
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = sh[0];
        for (int w = 1; w < SORT_WARPS; w++) {
            double ov = sh[w];
            if (ov != ov || (r == r && ov > r)) r = ov;
        }
        partial[blockIdx.x] = r;
    }
}

__global__ void k_hpdw_final(const double *__restrict__ maxpart, int nmax, double *__restrict__ maxv)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double r = maxpart[0];
        for (int w = 1; w < nmax; w++) {
            double ov = maxpart[w];
            if (ov != ov || (r == r && ov > r)) r = ov;
        }
        *maxv = r;
    }
}

__global__ void k_hpdw_result(const ArgMin *__restrict__ partial, int nblk, const double *__restrict__ rsorted,
                              double *__restrict__ out /*[3]: hpd, r75, r25*/)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double v0 = partial[0].v, v1 = partial[1].v;
        long long i0 = partial[0].i, i1 = partial[1].i;
        for (int b = 1; b < nblk; b++) {
            if (am_better(partial[2 * b].v, partial[2 * b].i, v0, i0)) { v0 = partial[2 * b].v; i0 = partial[2 * b].i; }
            if (am_better(partial[2 * b + 1].v, partial[2 * b + 1].i, v1, i1)) { v1 = partial[2 * b + 1].v; i1 = partial[2 * b + 1].i; }
        }
        double r75 = rsorted[i0], r25 = rsorted[i1];
        out[0] = r75 - r25;
        out[1] = r75;
        out[2] = r25;
    }
}

static Chunking make_chunking(int64_t num)
{
    Chunking ck;
    int G = sm_count() * 4;
    if (G > SORT_MAXG) G = SORT_MAXG;
    if (G < 1) G = 1;
    int64_t per = (num + G - 1) / G;
    per = ((per + SORT_TILE - 1) / SORT_TILE) * SORT_TILE;
    if (per < SORT_TILE) per = SORT_TILE;
    ck.num = num; ck.per = per;
    ck.G = (int)((num + per - 1) / per);
    if (ck.G < 1) ck.G = 1;
    return ck;
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Tile shape of the one-sweep pass: 512 threads x 12 keys, 2 CTAs/SM.  Argsort of 5e7 keys, steady state, threads x keys
// (CTAs/SM) 512 x 12 (2) / 256 x 12 (3) / 512 x 16 (2) / 1024 x 8 (1) / 256 x 16 (3): 4.16 / 4.60 / 5.60 / 5.02 / 4.24 ms
// (profiles/r02k_sort_variants.txt); after the full-tile fast path 512 x 12 / 256 x 16 / 256 x 12: 3.49 / 3.47 / 3.94 ms
// (profiles/r02n_sort_variants.txt)
#define OS_T 512
#define OS_I 12
#define OS_B 2

static int onesweep_passes(const double *keys_in, u64 *kA, u64 *kB, u32 *vA, u32 *vB, double *keys_out, long long *idx_out,
                           int64_t num, int digits, SortPlan *plan, u64 *status, cudaStream_t s)
{
    constexpr int T = OS_T, I = OS_I;
    const size_t tiles = ((size_t)num + (size_t)T * I - 1) / ((size_t)T * I);
    auto kern = k_onesweep<T, I, OS_B>;
    static bool smem_set[64] = {};
    if (first_on_device(smem_set))
        PXF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(OsSmem<T, I>)));
    for (int d = 0; d < 8; d++) {
        if (digits && !(digits & (1 << d))) continue;
        kern<<<(unsigned)tiles, T, sizeof(OsSmem<T, I>), s>>>(keys_in, kA, kB, vA, vB, keys_out, idx_out, num, d, plan, status);
        count_launch();
    }
    return PXF_OK;
}


// ------------------------------------------------------------------ segmented weighted HPD
// analyses.hpd(rays, weights) of every segment of a segmented bundle: radii about each segment's centroid, ONE
// stable sort by (segment, radius) -- the radius digits first, then a stable sort of the segment ids, so every
// segment's rays end up in its own slice [seg_start[s], seg_start[s+1]) in radius order, ties in input order as
// in the single-bundle sort -- then one CTA per segment: cumulative weights restarted at the segment, its max,
// and the first minimisers of |cdf/max - .75| and |cdf/max - .25|.
#define HPDW_SEG_TILE 4096
__global__ void __launch_bounds__(SORT_THREADS)
k_rho_seg(const double *__restrict__ x, const double *__restrict__ y, int64_t num, const long long *__restrict__ seg_start,
          int nseg, const double *__restrict__ sums, double *__restrict__ rho)
{
    for (int64_t t0 = (int64_t)blockIdx.x * HPDW_SEG_TILE; t0 < num; t0 += (int64_t)gridDim.x * HPDW_SEG_TILE) {
        const int64_t t1 = t0 + HPDW_SEG_TILE < num ? t0 + HPDW_SEG_TILE : num;
        seg_tile_pieces(t0, t1, seg_start, nseg, [&](int seg, int64_t a, int64_t b) {
            const double cx = sums[16 * (int64_t)seg + 1] / sums[16 * (int64_t)seg];
            const double cy = sums[16 * (int64_t)seg + 2] / sums[16 * (int64_t)seg];
            for (int64_t i = a + threadIdx.x; i < b; i += blockDim.x) rho[i] = sqrt(sq(x[i] - cx) + sq(y[i] - cy));
        });
    }
}

// key[i] = segment of ray idx[i] (exact as a double)
__global__ void __launch_bounds__(SORT_THREADS)
k_seg_of(const long long *__restrict__ idx, int64_t num, const long long *__restrict__ seg_start, int nseg,
         double *__restrict__ key)
{
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < num; i += nthr) {
        const long long r = idx[i];
        int lo = 0, hi = nseg - 1;                      // last segment starting at or before r
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (seg_start[mid] <= r) lo = mid; else hi = mid - 1;
        }
        key[i] = (double)lo;
    }
}

__global__ void __launch_bounds__(SORT_THREADS)
k_seg_compose(const long long *__restrict__ idx1, const double *__restrict__ rs1, const long long *__restrict__ idx2,
              int64_t num, long long *__restrict__ idx, double *__restrict__ rs)
{
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < num; i += nthr) {
        const long long j = idx2[i];
        idx[i] = idx1[j];
        rs[i] = rs1[j];
    }
}

#define HPDW_SEG_THREADS 1024
__global__ void __launch_bounds__(HPDW_SEG_THREADS)
k_hpdw_seg(const double *__restrict__ w, const long long *__restrict__ idx, const double *__restrict__ rs,
           const long long *__restrict__ seg_start, const double *__restrict__ sums, double *__restrict__ cdf,
           double *__restrict__ out)
{
    constexpr int NW = HPDW_SEG_THREADS / 32;
    __shared__ double wtot[NW];
    __shared__ double carry, mxs;
    __shared__ double shv[2][NW];
    __shared__ long long shi[2][NW];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int s = blockIdx.x;
    const long long a = seg_start[s], b = seg_start[s + 1];
    double *o = out + 4 * (int64_t)s;
    const double nanv = __longlong_as_double(0x7ff8000000000000ll);
    if (b == a || sums[16 * (int64_t)s] == 0.) {       // no rays / no weight: documented as NaN
        if (threadIdx.x == 0) { o[0] = nanv; o[1] = nanv; o[2] = nanv; o[3] = 1.; }
        return;
    }
    if (threadIdx.x == 0) carry = 0.;
    __syncthreads();
    // inclusive scan of w[idx[i]] over the slice (block scan with a running carry, as k_scan_apply) and its max
    double m = -__longlong_as_double(0x7ff0000000000000ll);
    bool nan = false;
    for (long long t0 = a; t0 < b; t0 += HPDW_SEG_THREADS) {
        const long long i = t0 + threadIdx.x;
        const double v = i < b ? w[idx[i]] : 0.;
        double incl = v;
#pragma unroll
        for (int q = 1; q < 32; q <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, incl, q);
            if (lane >= q) incl += t;
        }
        if (lane == 31) wtot[warp] = incl;
        __syncthreads();
        double base = carry;
        for (int q = 0; q < warp; q++) base += wtot[q];
        if (i < b) {
            const double c = base + incl;
            cdf[i] = c;
            if (c != c) nan = true;
            else if (c > m) m = c;
        }
        __syncthreads();
        if (threadIdx.x == HPDW_SEG_THREADS - 1) carry = base + incl;
        __syncthreads();
    }
    if (nan) m = nanv;
#pragma unroll
    for (int q = 16; q > 0; q >>= 1) {
        const double ov = __shfl_down_sync(0xffffffffu, m, q);
        if (ov != ov || (m == m && ov > m)) m = ov;
    }
    if (lane == 0) wtot[warp] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = wtot[0];
        for (int q = 1; q < NW; q++) {
            const double ov = wtot[q];
            if (ov != ov || (r == r && ov > r)) r = ov;
        }
        mxs = r;
    }
    __syncthreads();
    const double mx = mxs;
    double bv[2] = {__longlong_as_double(0x7ff0000000000000ll), __longlong_as_double(0x7ff0000000000000ll)};
    long long bi[2] = {0x7fffffffffffffffll, 0x7fffffffffffffffll};
    for (long long i = a + threadIdx.x; i < b; i += HPDW_SEG_THREADS) {
        const double c = cdf[i] / mx;
        const double d0 = fabs(c - .75), d1 = fabs(c - .25);
        if (am_better(d0, i, bv[0], bi[0])) { bv[0] = d0; bi[0] = i; }
        if (am_better(d1, i, bv[1], bi[1])) { bv[1] = d1; bi[1] = i; }
    }
#pragma unroll
    for (int c = 0; c < 2; c++) {
#pragma unroll
        for (int q = 16; q > 0; q >>= 1) {
            const double ov = __shfl_down_sync(0xffffffffu, bv[c], q);
            const long long oi = __shfl_down_sync(0xffffffffu, bi[c], q);
            if (am_better(ov, oi, bv[c], bi[c])) { bv[c] = ov; bi[c] = oi; }
        }
        if (lane == 0) { shv[c][warp] = bv[c]; shi[c][warp] = bi[c]; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long ii[2];
        for (int c = 0; c < 2; c++) {
            double v = shv[c][0];
            long long i = shi[c][0];
            for (int q = 1; q < NW; q++)
                if (am_better(shv[c][q], shi[c][q], v, i)) { v = shv[c][q]; i = shi[c][q]; }
            ii[c] = i;
        }
        const double r75 = rs[ii[0]], r25 = rs[ii[1]];
        o[0] = r75 - r25; o[1] = r75; o[2] = r25; o[3] = 1.;
    }
}

size_t hpd_weighted_segmented_bytes(int64_t num)
{
    const size_t n = (size_t)(num > 0 ? num : 1);
    return 7 * align256(n * 8) + align256(pxf_sort_scratch_bytes(num)) + 256;
}

int hpd_weighted_segmented(const double *x, const double *y, const double *w, int64_t num, const long long *seg_start,
                           int nseg, const double *sums, double *out, void *workspace, cudaStream_t s)
{
    const size_t n = (size_t)(num > 0 ? num : 1);
    char *p = static_cast<char *>(workspace);
    double *rho = (double *)p; p += align256(n * 8);      // radii, then the segment keys, then the cdf
    double *rs1 = (double *)p; p += align256(n * 8);
    long long *idx1 = (long long *)p; p += align256(n * 8);
    double *kout = (double *)p; p += align256(n * 8);
    long long *idx2 = (long long *)p; p += align256(n * 8);
    long long *idx = (long long *)p; p += align256(n * 8);
    double *rs = (double *)p; p += align256(n * 8);
    void *sort_scr = p;
    pxf_stream_t st = reinterpret_cast<pxf_stream_t>(s);
    int rc;
    if (num > 0) {
        k_rho_seg<<<grid_for(num, HPDW_SEG_TILE, 4), SORT_THREADS, 0, s>>>(x, y, num, seg_start, nseg, sums, rho);
        count_launch();
        if ((rc = pxf_argsort(rho, num, rs1, reinterpret_cast<int64_t *>(idx1), sort_scr, st))) return rc;
        k_seg_of<<<grid_for(num, SORT_THREADS * 4, 8), SORT_THREADS, 0, s>>>(idx1, num, seg_start, nseg, rho);
        count_launch();
        if ((rc = pxf_argsort(rho, num, kout, reinterpret_cast<int64_t *>(idx2), sort_scr, st))) return rc;
        k_seg_compose<<<grid_for(num, SORT_THREADS * 4, 8), SORT_THREADS, 0, s>>>(idx1, rs1, idx2, num, idx, rs);
        count_launch();
    }
    k_hpdw_seg<<<nseg, HPDW_SEG_THREADS, 0, s>>>(w, idx, rs, seg_start, sums, rho, out);
    count_launch();
    return check_launch("pxf_hpd_segmented (weighted)");
}

}  // namespace pxf

using namespace pxf;

extern "C" {

size_t pxf_sort_scratch_bytes(int64_t num)
{
    size_t n = (size_t)(num > 0 ? num : 1);
    const size_t tiles = (n + 256 * 12 - 1) / (256 * 12);       // 256 x 12-key tiles: room for any tile shape of 3072 keys or more
    return 2 * align256(n * 8) + 2 * align256(n * 4) + align256(tiles * 256 * 8) + align256(8 * 256 * 8 + 64) +
           align256(sizeof(SortPlan)) + 1024;
}

// digits: bit d set = sort on byte d of the 64-bit key (LSD order).  0 = automatic: bytes that are constant over the
// array are skipped (decided on the device from the up-front histogram of all eight bytes: nothing is read back,
// the call is asynchronous on `stream`).  A caller that knows which bytes can differ (e.g. keys from a narrow
// bracket) passes the mask.
int pxf_argsort_digits(const double *keys_in, int64_t num, double *keys_out, int64_t *idx_out,
                       void *scratch, int32_t digits, pxf_stream_t stream)
{
    if (num < 0 || !keys_in || !scratch || num > 0xffffffffll || digits < 0 || digits > 255) { set_error("pxf_argsort: bad argument"); return PXF_ERR_INVALID; }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    if (keys_out == keys_in) { set_error("pxf_argsort: keys_out must not alias keys_in (the input is read by the first and the last pass)"); return PXF_ERR_INVALID; }
    if (num == 0) return PXF_OK;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const size_t n = (size_t)num;
    const size_t tiles = (n + OS_T * OS_I - 1) / (OS_T * OS_I);
    char *p = static_cast<char *>(scratch);
    u64 *kA = (u64 *)p; p += align256(n * 8);
    u64 *kB = (u64 *)p; p += align256(n * 8);
    u32 *vA = (u32 *)p; p += align256(n * 4);
    u32 *vB = (u32 *)p; p += align256(n * 4);
    u64 *status = (u64 *)p; p += align256(tiles * 256 * 8);
    u64 *ghist = (u64 *)p; p += align256(8 * 256 * 8 + 64);   // [8][256] + the lossy-key flag
    SortPlan *plan = (SortPlan *)p;
    // one memset covers the tile status words and the histogram (they are adjacent)
    PXF_CUDA(cudaMemsetAsync(status, 0, align256(tiles * 256 * 8) + 8 * 256 * 8 + 64, s));
    k_sort_hist_all<<<grid_for(num, SORT_THREADS * 4, 8), SORT_THREADS, 0, s>>>(keys_in, num, ghist);
    k_sort_plan<<<1, 256, 0, s>>>(ghist, num, digits, plan);
    count_launch(2);
    long long *io = reinterpret_cast<long long *>(idx_out);
    const int rc = onesweep_passes(keys_in, kA, kB, vA, vB, keys_out, io, num, digits, plan, status, s);
    if (rc) return rc;
    k_sort_identity<<<grid_for(num, SORT_THREADS * 2, 8), SORT_THREADS, 0, s>>>(keys_in, num, plan, keys_out, io);
    count_launch();
    return check_launch("pxf_argsort");
}

int pxf_argsort(const double *keys_in, int64_t num, double *keys_out, int64_t *idx_out,
                void *scratch, pxf_stream_t stream)
{
    return pxf_argsort_digits(keys_in, num, keys_out, idx_out, scratch, 0, stream);
}

size_t pxf_scan_scratch_bytes(int64_t num) { (void)num; return (size_t)(SORT_MAXG + 8) * 8; }

int pxf_cumsum_gather(const double *w, const int64_t *idx, int64_t num, double *out,
                      void *scratch, pxf_stream_t stream)
{
    if (num < 0 || !out || !scratch) { set_error("pxf_cumsum_gather: bad argument"); return PXF_ERR_INVALID; }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    if (num == 0) return PXF_OK;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    Chunking ck = make_chunking(num);
    double *csum = static_cast<double *>(scratch);
    const long long *ix = reinterpret_cast<const long long *>(idx);
    k_scan_chunk_sums<<<ck.G, SORT_THREADS, 0, s>>>(w, ix, ck, csum);
    k_scan_chunk_offsets<<<1, 1024, 0, s>>>(csum, ck.G);
    k_scan_apply<<<ck.G, SORT_THREADS, 0, s>>>(w, ix, ck, csum, out);
    count_launch(3);
    return check_launch("pxf_cumsum_gather");
}

// analyses.hpd weighted branch (analyses.py:88-94): r,cdf = rhocdf(...); r[argmin|cdf-.75|]-r[argmin|cdf-.25|]
int pxf_hpd_weighted_sorted(const double *x, const double *y, const double *w, int64_t num, double *hpd_host,
                     pxf_stream_t stream)
{
    if (num <= 0 || !x || !y || !w || !hpd_host) { set_error("pxf_hpd_weighted_sorted: bad argument"); return PXF_ERR_INVALID; }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    int rc;
    const size_t n = (size_t)num;
    const int RG = 1024;
    Scratch sc;
    size_t bytes = pxf_sums_scratch_bytes() + 64 * 8 + 3 * align256(n * 8) + pxf_sort_scratch_bytes(num) +
                   pxf_scan_scratch_bytes(num) + align256(RG * 2 * sizeof(ArgMin)) + align256(RG * 8) + 1024;
    if ((rc = sc.alloc(bytes, s))) return rc;
    char *p = static_cast<char *>(sc.p);
    void *sum_scr = p; p += pxf_sums_scratch_bytes();
    double *sums = (double *)p; p += 32 * 8;
    double *small = (double *)p; p += 32 * 8;       // [0]=max, [4..6]=result
    double *rho = (double *)p; p += align256(n * 8);   // later reused for the cdf
    double *rs = (double *)p; p += align256(n * 8);
    long long *idx = (long long *)p; p += align256(n * 8);
    void *sort_scr = p; p += pxf_sort_scratch_bytes(num);
    void *scan_scr = p; p += align256(pxf_scan_scratch_bytes(num));
    ArgMin *am = (ArgMin *)p; p += align256(RG * 2 * sizeof(ArgMin));
    double *maxpart = (double *)p;
    // centroid with weights, then radii about it (analyses.py:60-71 with cent=True)
    if ((rc = pxf_sums(PXF_SUMS_CENTROID, x, y, nullptr, nullptr, nullptr, w, num, 0., 0., sums, sum_scr, stream))) return rc;
    double h[4];
    PXF_CUDA(cudaMemcpyAsync(h, sums, sizeof(h), cudaMemcpyDeviceToHost, s));
    PXF_CUDA(cudaStreamSynchronize(s));
    double cx = h[1] / h[0], cy = h[2] / h[0];
    if ((rc = pxf_rho(x, y, num, cx, cy, rho, stream))) return rc;
    if ((rc = pxf_argsort(rho, num, rs, reinterpret_cast<int64_t *>(idx), sort_scr, stream))) return rc;
    double *cdf = rho;
    if ((rc = pxf_cumsum_gather(w, reinterpret_cast<int64_t *>(idx), num, cdf, scan_scr, stream))) return rc;
    int grid = grid_for(num, SORT_THREADS * 4, 4);
    if (grid > RG) grid = RG;
    k_max_partial<<<grid, SORT_THREADS, 0, s>>>(cdf, num, maxpart);
    k_hpdw_final<<<1, 32, 0, s>>>(maxpart, grid, small);
    k_cdf_argmin<<<grid, SORT_THREADS, 0, s>>>(cdf, num, small, .75, .25, am);
    k_hpdw_result<<<1, 32, 0, s>>>(am, grid, rs, small + 4);
    count_launch(4);
    if ((rc = check_launch("pxf_hpd_weighted_sorted"))) return rc;
    double r[3];
    PXF_CUDA(cudaMemcpyAsync(r, small + 4, sizeof(r), cudaMemcpyDeviceToHost, s));
    PXF_CUDA(cudaStreamSynchronize(s));
    *hpd_host = r[0];
    return PXF_OK;
}

}  // extern "C"
