// Statically specialised fused kernels for the reference's canonical op chains.
//
// The generic interpreter (pxf_fused.cu) pays for its generality: every scalar parameter is an
// indexed constant load (ADU pipe), the opcode switch costs branches and i-cache, and the
// register allocation is the maximum over all ops (pow, sincos, ...).  For the chains the
// reference's example scripts actually run -- Wolter-I pair to the focal plane
// (examples/axro/singlePassAlignment.py:246-269), Wolter-Schwarzschild pair
// (examples/axro/axialHeights.py:77-113), SPO pair (examples/arcus/cat.py:219-280) -- the op
// list is known at compile time: a variadic template composes the SAME per-op device functions
// (pxf_ray.cuh) into one straight-line kernel whose parameters are direct constant-bank operands.
// Results are bit-identical to the interpreter and to the per-routine kernels.
#include <stdlib.h>
#include <string>
#include "pxf_program.h"
#include "pxf_chain_ops.cuh"

namespace pxf {

// host side of a compile-time chain: does an op list match it, and its parameter pack from the folded op table
template <class... Ops> struct ChainHost;
template <> struct ChainHost<> {
    static void fill(ChainP<> &, const FusedOp *) {}
    static bool match(const FusedOp *, int n) { return n == 0; }
};
template <class Op, class... Rest> struct ChainHost<Op, Rest...> {
    static void fill(ChainP<Op, Rest...> &cp, const FusedOp *ops)
    {
        static_assert(sizeof(typename Op::P) <= sizeof(ops->q), "parameter block too large");
        memcpy(&cp.head, ops->q, sizeof(typename Op::P));
        ChainHost<Rest...>::fill(cp.tail, ops + 1);
    }
    static bool match(const FusedOp *ops, int n)
    {
        return n >= 1 && ops->code == Op::CODE && ChainHost<Rest...>::match(ops + 1, n - 1);
    }
};

// ---- kernel -------------------------------------------------------------------------------
// MODE 1: one ray per thread-iteration (8-byte accesses, the path for unaligned rows)
// MODE 2: two rays per thread-iteration (double2 accesses), traced one after the other
// PF    : (MODE 1) software prefetch -- the loads of the NEXT iteration are issued before the current
//         ray is traced, so every warp keeps ~1.5-3 KB of loads in flight during its compute
//         phase.  Without it the kernel is limited by bytes in flight: a warp is either waiting
//         for its loads or computing, and with ~70 % of the time spent computing too few loads
//         are outstanding to keep HBM busy (measured: 4.1 ms vs 2.6 ms for the same traffic
//         with trivial compute, profiles/r01_notes.md).
// LMc/SMc: row masks known at compile time (0 = use the runtime masks LM/SM), so that rows the
//         chain never loads cost no registers in the prefetch buffer.
// Registers are capped for 3 resident CTAs per SM.  Tuned on B200 (profiles/r01_notes.md): on aligned rows two
// rays in sequence, 3 CTAs/SM, no prefetch is the fastest shape; a bulk-async variant that streams the rows
// into a shared-memory ring (cp.async.bulk, one producer thread) removes every load stall and is no faster.
#define CHAIN_MINB 3
template <unsigned M>
PXF_DEV void cload1(Ray &r, const RowPtrs &P, unsigned LM, int64_t i)
{
    if (M == 0) { fload1(r, P, LM, i); return; }
    r.opd = (M & R_OPD) ? P.p[0][i] : 0.;
    r.x = (M & R_X) ? P.p[1][i] : 0.;  r.y = (M & R_Y) ? P.p[2][i] : 0.;  r.z = (M & R_Z) ? P.p[3][i] : 0.;
    r.l = (M & R_L) ? P.p[4][i] : 0.;  r.m = (M & R_M) ? P.p[5][i] : 0.;  r.n = (M & R_N) ? P.p[6][i] : 0.;
    r.ux = (M & R_UX) ? P.p[7][i] : 0.; r.uy = (M & R_UY) ? P.p[8][i] : 0.; r.uz = (M & R_UZ) ? P.p[9][i] : 0.;
}
#define CLD2(bit, k, f)                                                               \
    if (M & bit) { double2 v = *reinterpret_cast<const double2 *>(P.p[k] + i); a.f = v.x; b.f = v.y; } \
    else { a.f = 0.; b.f = 0.; }
template <unsigned M>
PXF_DEV void cload2(Ray &a, Ray &b, const RowPtrs &P, unsigned LM, int64_t i)
{
    if (M == 0) { fload2(a, b, P, LM, i); return; }
    CLD2(R_OPD, 0, opd) CLD2(R_X, 1, x) CLD2(R_Y, 2, y) CLD2(R_Z, 3, z) CLD2(R_L, 4, l)
    CLD2(R_M, 5, m) CLD2(R_N, 6, n) CLD2(R_UX, 7, ux) CLD2(R_UY, 8, uy) CLD2(R_UZ, 9, uz)
}
template <unsigned M>
PXF_DEV void cstore1(const Ray &r, const RowPtrs &P, unsigned SM, int64_t i)
{
    fstore1(r, P, M ? M : SM, i);
}
template <unsigned M>
PXF_DEV void cstore2(const Ray &a, const Ray &b, const RowPtrs &P, unsigned SM, int64_t i)
{
    fstore2(a, b, P, M ? M : SM, i);
}

template <class C, class CP, int MODE, bool PF, unsigned LMc, unsigned SMc>
__global__ void __launch_bounds__(PXF_BLOCK, CHAIN_MINB)
k_chain(const RowPtrs P, const RowPtrs Q, const int64_t num, uint8_t *__restrict__ alive,
        double *__restrict__ partials, const unsigned LM, const unsigned SM, const __grid_constant__ CP prm)
{
    double cnt = 0., sx = 0., sy = 0.;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    if (MODE >= 2) {
        const int64_t npair = num >> 1;
        int64_t q = tid;
        Ray cur[2];
        while (q < npair) {
            const int64_t qn = q + nthr;
            cload2<LMc>(cur[0], cur[1], P, LM, q << 1);
            C::run(cur[0], prm);
            C::run(cur[1], prm);
            const int64_t i = q << 1;
            cstore2<SMc>(cur[0], cur[1], Q, SM, i);
            if (alive) { alive[i] = 1; alive[i + 1] = 1; }
            cnt += 2.; sx += cur[0].x; sx += cur[1].x; sy += cur[0].y; sy += cur[1].y;
            q = qn;
        }
        if ((num & 1) && tid == 0) {
            const int64_t i = num - 1;
            Ray a;
            cload1<LMc>(a, P, LM, i);
            const bool ka = C::run(a, prm);
            cstore1<SMc>(a, Q, SM, i);
            if (alive) alive[i] = ka ? 1 : 0;
            if (ka) { cnt += 1.; sx += a.x; sy += a.y; }
        }
    } else {
        int64_t i = tid;
        Ray cur, nxt;
        if (PF && i < num) cload1<LMc>(cur, P, LM, i);
        while (i < num) {
            const int64_t in = i + nthr;
            if (PF) {
                if (in < num) cload1<LMc>(nxt, P, LM, in);
            } else {
                cload1<LMc>(cur, P, LM, i);
            }
            const bool ka = C::run(cur, prm);
            cstore1<SMc>(cur, Q, SM, i);
            if (alive) alive[i] = ka ? 1 : 0;
            if (ka) { cnt += 1.; sx += cur.x; sy += cur.y; }
            if (PF) cur = nxt;
            i = in;
        }
    }
    if (partials) centroid_block_reduce(cnt, sx, sy, partials);
}

template <class C, class CP, int MODE, bool PF, unsigned LMc, unsigned SMc>
static int launch_k_chain(const RowPtrs &P, const RowPtrs &Q, int64_t num, uint8_t *alive, unsigned LM, unsigned SM,
                          const CP &cp, cudaStream_t s, double *partials, int *grid_out)
{
    static int ctas = 0;
    auto kern = k_chain<C, CP, MODE, PF, LMc, SMc>;
    if (ctas == 0) {
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, PXF_BLOCK, 0) != cudaSuccess || nb <= 0) {
            cudaGetLastError();
            nb = CHAIN_MINB;
        }
        ctas = nb;
    }
    const int64_t items = MODE >= 2 ? ((num + 1) >> 1) : num;
    const int grid = grid_for(items, PXF_BLOCK, ctas);
    if (grid_out) *grid_out = grid;
    kern<<<grid, PXF_BLOCK, 0, s>>>(P, Q, num, alive, partials, LM, SM, cp);
    count_launch();
    return check_launch("k_chain");
}

// LMc/SMc: the row masks this chain has when traced in place or out of place (checked against
// build_program's liveness result at run time; any other masks take the runtime-mask kernel).
template <unsigned LMc, unsigned SMc, class... Ops>
static int try_chain(const RowPtrs &P, const RowPtrs &Q, int64_t num, const FusedProgram &fp, uint8_t *alive,
                     bool aligned, cudaStream_t s, double *partials, int *grid_out)
{
    using C = Chain<Ops...>;
    using CP = ChainP<Ops...>;
    if (fp.nops != C::N || !ChainHost<Ops...>::match(fp.ops, fp.nops)) return PXF_ERR_UNSUPPORTED;
    CP cp;
    memset(&cp, 0, sizeof(cp));
    ChainHost<Ops...>::fill(cp, fp.ops);
    const unsigned LM = fp.load_mask, SM = fp.store_mask;
    {
        std::string nm = "k_chain<Chain<";
        const char *names[] = {Ops::NAME...};
        for (size_t k = 0; k < sizeof...(Ops); k++) { if (k) nm += ", "; nm += names[k]; }
        note_kernel((nm + ">> (built into libpxf)").c_str());
    }
    if constexpr (LMc != 0) {
        if (LM == LMc && SM == SMc) {
            if (!aligned) return launch_k_chain<C, CP, 1, true, LMc, SMc>(P, Q, num, alive, LM, SM, cp, s, partials, grid_out);
            return launch_k_chain<C, CP, 2, false, LMc, SMc>(P, Q, num, alive, LM, SM, cp, s, partials, grid_out);
        }
    }
    if (!aligned) return launch_k_chain<C, CP, 1, false, 0u, 0u>(P, Q, num, alive, LM, SM, cp, s, partials, grid_out);
    return launch_k_chain<C, CP, 2, false, 0u, 0u>(P, Q, num, alive, LM, SM, cp, s, partials, grid_out);
}

int launch_chain(const RowPtrs &P, const RowPtrs &Q, int64_t num, const FusedProgram &fp, uint8_t *alive,
                 bool aligned, cudaStream_t s, double *partials, int *grid_out)
{
    static int disabled = -1;
    if (disabled < 0) {
        const char *e = getenv("PXF_NO_SPECIALIZE");     // force the generic interpreter (tests, A/B timing)
        disabled = (e && e[0] == '1') ? 1 : 0;
    }
    if (disabled || fp.has_vignette) return PXF_ERR_UNSUPPORTED;
    int rc;
    // Wolter-I pair to the focal plane (BASELINE config 1)
    rc = try_chain<(R_POS | R_DIR), R_NINE, CTransform, CWolterPrimary, CReflect, CWolterSecondary, CReflect, CFlat>(P, Q, num, fp, alive, aligned, s, partials, grid_out);
    if (rc != PXF_ERR_UNSUPPORTED) return rc;
    rc = try_chain<0u, 0u, CWolterPrimary, CReflect, CWolterSecondary, CReflect, CFlat>(P, Q, num, fp, alive, aligned, s, partials, grid_out);
    if (rc != PXF_ERR_UNSUPPORTED) return rc;
    rc = try_chain<0u, 0u, CTransform, CWolterPrimary, CReflect, CWolterSecondary, CReflect>(P, Q, num, fp, alive, aligned, s, partials, grid_out);
    if (rc != PXF_ERR_UNSUPPORTED) return rc;
    // Wolter-Schwarzschild pair with the field-angle kick (BASELINE config 2)
    rc = try_chain<0u, 0u, CTransform, CWsPrimary, CKick, CReflect, CWsSecondary, CReflect>(P, Q, num, fp, alive, aligned, s, partials, grid_out);
    if (rc != PXF_ERR_UNSUPPORTED) return rc;
    // SPO primary/secondary pair (BASELINE config 4, per-shell part)
    rc = try_chain<0u, 0u, CTransform, CSpoCone, CReflect, CSpoCone, CReflect, CTransform>(P, Q, num, fp, alive, aligned, s, partials, grid_out);
    if (rc != PXF_ERR_UNSUPPORTED) return rc;
    // focus step: move the plane and trace to it (surfaces.focus, surfaces.py:502-510)
    rc = try_chain<0u, 0u, CTransform, CFlat>(P, Q, num, fp, alive, aligned, s, partials, grid_out);
    return rc;
}

// ---- segmented specialised chain (nested assemblies) --------------------------------------------
// Same tiling as k_program_seg (pxf_fused.cu) with the op list known at compile time: the per-segment
// parameter pack ChainP (not an op table) is staged in shared memory and the chain runs straight-line.
// Registers capped for 4 resident CTAs per SM: measured at 2e7 rays, 260 shells, caps 2 / 3 / 4 / 5: 0.92 / 0.78 /
// 0.72 / 0.76 ms.
#define CSEG_TILE (PXF_BLOCK * 8)
template <class C, class CP>
__global__ void __launch_bounds__(PXF_BLOCK, 4)
k_chain_seg(const RowPtrs P, const RowPtrs Q, const int64_t num, uint8_t *__restrict__ alive,
            const long long *__restrict__ seg_start, const CP *__restrict__ table, const int nseg,
            const unsigned LM, const unsigned SM)
{
    __shared__ __align__(16) CP sp;
    static_assert(sizeof(CP) % 8 == 0, "parameter pack must be a whole number of doubles");
    int staged = -1;
    for (int64_t t0 = (int64_t)blockIdx.x * CSEG_TILE; t0 < num; t0 += (int64_t)gridDim.x * CSEG_TILE) {
        const int64_t t1 = t0 + CSEG_TILE < num ? t0 + CSEG_TILE : num;
        int lo = 0, hi = nseg - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (seg_start[mid] <= t0) lo = mid; else hi = mid - 1;
        }
        int seg = lo;
        int64_t pos = t0;
        while (pos < t1 && seg < nseg) {
            int64_t send = seg_start[seg + 1];
            if (send <= pos) { seg++; continue; }
            if (send > t1) send = t1;
            if (seg != staged) {
                __syncthreads();
                const double *src = reinterpret_cast<const double *>(table + seg);
                double *dst = reinterpret_cast<double *>(&sp);
                for (int t = threadIdx.x; t < (int)(sizeof(CP) / 8); t += blockDim.x) dst[t] = src[t];
                __syncthreads();
                staged = seg;
            }
            for (int64_t i = pos + threadIdx.x; i < send; i += blockDim.x) {
                Ray a;
                fload1(a, P, LM, i);
                const bool keep = C::run(a, sp);
                fstore1(a, Q, SM, i);
                if (alive) alive[i] = keep ? 1 : 0;
            }
            pos = send;
            seg++;
        }
    }
}

using SegWolter = Chain<CTransform, CWolterPrimary, CReflect, CWolterSecondary, CReflect, CFlat>;
using SegWolterP = ChainP<CTransform, CWolterPrimary, CReflect, CWolterSecondary, CReflect, CFlat>;
using SegWolterH = ChainHost<CTransform, CWolterPrimary, CReflect, CWolterSecondary, CReflect, CFlat>;

size_t seg_chain_bytes(int nseg) { return (size_t)nseg * sizeof(SegWolterP); }

// ops: segment-major folded op table.  Returns the chain id (1 = Wolter-I pair to the focal plane) after filling
// dst with one parameter pack per segment, or 0 when no specialisation matches.
int seg_chain_fill(const FusedOp *ops, int nops, int nseg, void *dst)
{
    static int disabled = -1;
    if (disabled < 0) {
        const char *e = getenv("PXF_NO_SPECIALIZE");
        disabled = (e && e[0] == '1') ? 1 : 0;
    }
    if (disabled || nops != SegWolter::N || !SegWolterH::match(ops, nops)) return 0;
    SegWolterP *out = static_cast<SegWolterP *>(dst);
    for (int sgm = 0; sgm < nseg; sgm++) {
        memset(&out[sgm], 0, sizeof(SegWolterP));
        SegWolterH::fill(out[sgm], ops + (size_t)sgm * nops);
    }
    return 1;
}

int seg_chain_launch(int chain_id, const RowPtrs &P, const RowPtrs &Q, int64_t num, uint8_t *alive,
                     const long long *seg_start_dev, const void *table_dev, int nseg, unsigned LM, unsigned SM,
                     cudaStream_t s)
{
    if (chain_id != 1) return PXF_ERR_UNSUPPORTED;
    auto kern = k_chain_seg<SegWolter, SegWolterP>;
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, PXF_BLOCK, 0) != cudaSuccess || nb <= 0) { cudaGetLastError(); nb = 3; }
    const int grid = grid_for(num, CSEG_TILE, nb);
    kern<<<grid, PXF_BLOCK, 0, s>>>(P, Q, num, alive, seg_start_dev, static_cast<const SegWolterP *>(table_dev), nseg, LM, SM);
    count_launch();
    note_kernel("k_chain_seg<Chain<CTransform,CWolterPrimary,CReflect,CWolterSecondary,CReflect,CFlat>>");
    return check_launch("k_chain_seg");
}

}  // namespace pxf
