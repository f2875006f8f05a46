// Compile-time op chains: one functor per fused-program opcode and a variadic template that composes them into
// straight-line per-ray code.  Device code only (no host headers): included by pxf_chain.cu for the chains that are
// instantiated when libpxf.so is built, and compiled by NVRTC at run time for every other op list (pxf_jit.cu).
//
// A functor's parameter block P is exactly what build_program (pxf_fused.cu) stores at the start of FusedOp::q for
// that opcode; every P is a whole number of doubles with 8-byte alignment, so the parameter pack of a chain,
// ChainP<Ops...>, is the plain concatenation of the blocks followed by 8 bytes -- the host builds it without
// knowing the C++ type (pxf_jit.cu).
#pragma once
#include "pxf_rows.cuh"

namespace pxf {

struct NoP { double unused; };

// what an op may need besides the ray and its parameters
struct ChainCtx {
    const ZernP *zt;          // Zernike table staged in shared memory (PXF_OP_ZERNSURF / ZERNPHASE)
    const LLTab *llt;         // LL tables staged in shared memory, by slot (PXF_OP_LLSURF)
    int64_t i;                // index of the ray in the bundle (side arrays)
    const double *aux_wave;   // pxf_program_aux
    int *aux_count;
    int *aux_count_max;
};
PXF_DEV ChainCtx chain_ctx_none()
{
    ChainCtx c; c.zt = nullptr; c.llt = nullptr; c.i = 0; c.aux_wave = nullptr; c.aux_count = nullptr; c.aux_count_max = nullptr;
    return c;
}

PXF_DEV double chain_ray_row(const Ray &r, int row)
{
    switch (row) {
        case 0: return r.opd; case 1: return r.x; case 2: return r.y; case 3: return r.z;
        case 4: return r.l; case 5: return r.m; case 6: return r.n; case 7: return r.ux;
        case 8: return r.uy; default: return r.uz;
    }
}
// one atomic per warp: the largest grating count seen by the lanes that are here together
PXF_DEV void chain_count_max(int *dst, int k)
{
    const unsigned act = __activemask();
    const int m = __reduce_max_sync(act, k);
    if ((threadIdx.x & 31) == (__ffs(act) - 1)) atomicMax(dst, m);
}

// ---- op functors (CODE = the PXF_OP_* value, include/pxf.h) ----
#define PXF_CHAIN_OP(FUNCTOR, CODEV, PTYPE, CALL)                                                     \
    struct FUNCTOR {                                                                                  \
        using P = PTYPE;                                                                              \
        static constexpr int CODE = CODEV;                                                            \
        static constexpr const char *NAME = #FUNCTOR;                                                 \
        PXF_DEV static bool apply(Ray &r, const P &p, const ChainCtx &ctx) { (void)p; (void)ctx; CALL; return true; } \
    };
PXF_CHAIN_OP(CTransform, 1, TransformP, op_transform(r, p))
PXF_CHAIN_OP(CITransform, 2, TransformP, op_itransform(r, p))
PXF_CHAIN_OP(CReflect, 3, NoP, op_reflect(r))
PXF_CHAIN_OP(CRefract, 4, RefractP, op_refract(r, p))
PXF_CHAIN_OP(CRadgrat, 5, RadgratP, op_radgrat(r, p, p.wave, false))
PXF_CHAIN_OP(CFlat, 6, NoP, op_flat(r, false, 0.))
struct FlatOpdP { double nr; };
PXF_CHAIN_OP(CFlatOpd, 7, FlatOpdP, op_flat(r, true, p.nr))
PXF_CHAIN_OP(CConic, 8, ConicP, op_conic(r, p))
PXF_CHAIN_OP(CConicOpd, 9, ConicP, op_conic(r, p))
PXF_CHAIN_OP(CWolterPrimary, 10, WolterP, op_wolterprimary(r, p))
PXF_CHAIN_OP(CWolterPrimaryOpd, 11, WolterP, op_wolterprimary(r, p))
PXF_CHAIN_OP(CWolterSecondary, 12, WolterP, op_woltersecondary(r, p))
PXF_CHAIN_OP(CWolterSine, 13, WolterSineP, op_woltersine(r, p))
PXF_CHAIN_OP(CWsPrimary, 14, WSP, op_wsprimary(r, p))
PXF_CHAIN_OP(CWsSecondary, 15, WSP, op_wssecondary(r, p))
PXF_CHAIN_OP(CSpoCone, 16, SpoP, op_spocone(r, p))
struct KickP { double dl, dm, sn; };
PXF_CHAIN_OP(CKick, 20, KickP,
             r.l = r.l + p.dl; r.m = r.m + p.dm; r.n = p.sn * sqrt(1. - sq(r.l) - sq(r.m)))
PXF_CHAIN_OP(CKickN, 22, KickNP, op_kickn(r, p))
PXF_CHAIN_OP(CTraceSphere, 27, SphereP, op_tracesphere(r, p))
PXF_CHAIN_OP(CTraceSphereOpd, 28, SphereP, op_tracesphere(r, p))
PXF_CHAIN_OP(CTraceCyl, 29, SphereP, op_tracecyl(r, p))
PXF_CHAIN_OP(CTraceCylOpd, 30, SphereP, op_tracecyl(r, p))
PXF_CHAIN_OP(CCylConic, 31, CylConicP, op_cylconic(r, p))
PXF_CHAIN_OP(CParaxial, 32, ParaxialP, op_paraxial(r, p))
PXF_CHAIN_OP(CParaxialY, 33, ParaxialP, op_paraxial(r, p))
PXF_CHAIN_OP(CTorus, 34, TorusP, op_torus(r, p))
PXF_CHAIN_OP(CWsPrimaryBack, 35, WSP, op_wsprimary_t<true>(r, p))
PXF_CHAIN_OP(CWsSecondaryBack, 36, WSP, op_wssecondary_t<true>(r, p))
// CONICPLUS[OPD] / LEGSURF: q = the device address of the folded block
struct ConicPlusTabP { const ConicPlusP *t; };
struct LegSurfTabP { const LegSurfP *t; };
PXF_CHAIN_OP(CConicPlus, 38, ConicPlusTabP, op_conicplus(r, *p.t))
PXF_CHAIN_OP(CConicPlusOpd, 39, ConicPlusTabP, op_conicplus(r, *p.t))
PXF_CHAIN_OP(CLegSurf, 40, LegSurfTabP, op_legsurf(r, *p.t))
// RADGRATW / GRAT: q = the scalars and the device addresses of the per-ray arrays, read at the ray's index
PXF_CHAIN_OP(CRadgratW, 41, RadgratWP, op_radgrat(r, p.g, p.wave[ctx.i], true))
PXF_CHAIN_OP(CGrat, 42, GratOpP, op_grat(r, p.d, p.order[ctx.i], p.wave[ctx.i]))
#undef PXF_CHAIN_OP

// predicates: the ray stops at the op when apply() returns false
struct CVignetteMag {
    using P = NoP;
    static constexpr int CODE = 17;
    PXF_DEV static bool apply(Ray &r, const P &, const ChainCtx &) { double mag = sq(r.l) + sq(r.m) + sq(r.n); return mag > .1; }
};
struct VigBoxP { double lo, hi; };
template <int ROW> struct CVignetteBox {
    using P = VigBoxP;
    static constexpr int CODE = 18;
    PXF_DEV static bool apply(Ray &r, const P &p, const ChainCtx &) { double v = chain_ray_row(r, ROW); return (v > p.lo) && (v < p.hi); }
};
struct VigAbsP { double hi, centre, has_centre; };
template <int ROW> struct CVignetteAbs {
    using P = VigAbsP;
    static constexpr int CODE = 19;
    PXF_DEV static bool apply(Ray &r, const P &p, const ChainCtx &)
    {
        double v = chain_ray_row(r, ROW);
        if (p.has_centre != 0.) v = v - p.centre;
        return fabs(v) < p.hi;
    }
};
struct VigRhoP { double rho0; };
struct CVignetteRhoGt {
    using P = VigRhoP;
    static constexpr int CODE = 23;
    PXF_DEV static bool apply(Ray &r, const P &p, const ChainCtx &) { double rho = sqrt(sq(r.x) + sq(r.y)); return rho > p.rho0; }
};
// ZERNSURF: q = {0, opd flag}; the table comes through the context
struct ZernOpP { double unused, with_opd; };
struct CZernSurf {
    using P = ZernOpP;
    static constexpr int CODE = 21;
    PXF_DEV static bool apply(Ray &r, const P &p, const ChainCtx &ctx)
    {
        const ZernP *zt = ctx.zt;
        if (zt) op_tracezern<7>(r, zt->rad, zt->nr, zt->tol, zt->nmax, p.with_opd != 0., reinterpret_cast<const double *>(zt->e));
        return true;
    }
};
// ZERNPHASE: q = {wave}; the table comes through the context, as for ZERNSURF
struct ZernPhaseOpP { double wave; };
struct CZernPhase {
    using P = ZernPhaseOpP;
    static constexpr int CODE = 37;
    PXF_DEV static bool apply(Ray &r, const P &p, const ChainCtx &ctx)
    {
        const ZernP *zt = ctx.zt;
        if (zt) op_zernphase<7>(r, zt->rad, p.wave, zt->nmax, reinterpret_cast<const double *>(zt->e));
        return true;
    }
};
// LLSURF: q = {N, slot}; the table comes through the context.  Both are template arguments: N is the op's order as
// make_ll rounds it (3, 5, 7), read from the zero-padded 8x8 block with static offsets -- the same bits as the
// per-routine kernel of that order (pxf_ray.cuh, LLTab)
struct LLOpP { double n, slot; };
template <int N, int SLOT> struct CLLSurf {
    using P = LLOpP;
    static constexpr int CODE = 26;
    PXF_DEV static bool apply(Ray &r, const P &, const ChainCtx &ctx)
    {
        const LLTab &t = ctx.llt[SLOT];
        op_ll<N, PXF_LL_PROG_MAXN + 1>(r, t.s, t.C);
        return true;
    }
};
struct CGratFan {
    using P = GratFanP;
    static constexpr int CODE = 24;
    PXF_DEV static bool apply(Ray &r, const P &p, const ChainCtx &ctx)
    {
        const int k = op_gratfan(r, p, p.wave_array ? ctx.aux_wave[ctx.i] : p.g.wave);
        if (ctx.aux_count) ctx.aux_count[ctx.i] = k;
        if (ctx.aux_count_max) chain_count_max(ctx.aux_count_max, k < 0 ? p.cap + 1 : k);
        return true;
    }
};
struct RotxP { TransformP rot; double total; };
struct CRotxRemaining {
    using P = RotxP;
    static constexpr int CODE = 25;
    PXF_DEV static bool apply(Ray &r, const P &p, const ChainCtx &ctx)
    {
        const int k = ctx.aux_count[ctx.i];
        if (k >= 0) op_rotx_repeat(r, p.rot, (int)p.total - k);
        return true;
    }
};

// ---- parameter pack and straight-line composition ----
template <class... Ops> struct ChainP;
template <> struct ChainP<> { double unused; };
template <class Op, class... Rest> struct ChainP<Op, Rest...> {
    typename Op::P head;
    ChainP<Rest...> tail;
};

template <class... Ops> struct Chain;
template <> struct Chain<> {
    static constexpr int N = 0;
    PXF_DEV static bool run(Ray &, const ChainP<> &, const ChainCtx &) { return true; }
};
template <class Op, class... Rest> struct Chain<Op, Rest...> {
    static constexpr int N = 1 + sizeof...(Rest);
    static_assert(sizeof(typename Op::P) % 8 == 0 && alignof(typename Op::P) == 8, "parameter blocks are whole doubles");
    PXF_DEV static bool run(Ray &r, const ChainP<Op, Rest...> &p, const ChainCtx &ctx)
    {
        if (!Op::apply(r, p.head, ctx)) return false;
        return Chain<Rest...>::run(r, p.tail, ctx);
    }
    PXF_DEV static bool run(Ray &r, const ChainP<Op, Rest...> &p) { return run(r, p, chain_ctx_none()); }
};

// ---- kernel bodies for the run-time specialised chains ----
// MODE 2: two rays per thread-iteration (double2 rows), 1: one ray (also the path for unaligned rows).
// LMc/SMc: the program's row masks as compile-time constants.  NLL: the number of PXF_OP_LLSURF ops (tables ll0, ll1).
template <class C, class CP, int MODE, bool ZERN, int NLL, unsigned LMc, unsigned SMc>
PXF_DEV void chain_body(const RowPtrs &P, const RowPtrs &Q, const int64_t num, uint8_t *__restrict__ alive,
                        double *__restrict__ partials, const CP &prm, const ZernP *__restrict__ zern_dev,
                        const double *__restrict__ aux_wave, int *__restrict__ aux_count, int *__restrict__ aux_count_max,
                        const LLTab *__restrict__ ll0, const LLTab *__restrict__ ll1)
{
    __shared__ __align__(16) unsigned char zraw[ZERN ? sizeof(ZernP) : NLL ? NLL * sizeof(LLTab) : 16];
    ChainCtx ctx = chain_ctx_none();
    ctx.aux_wave = aux_wave; ctx.aux_count = aux_count; ctx.aux_count_max = aux_count_max;
    if (ZERN && zern_dev) {
        const double *src = reinterpret_cast<const double *>(zern_dev);
        double *dst = reinterpret_cast<double *>(zraw);
        for (int t = threadIdx.x; t < (int)(sizeof(ZernP) / 8); t += blockDim.x) dst[t] = src[t];
        __syncthreads();
        ctx.zt = reinterpret_cast<const ZernP *>(zraw);
    }
    if (NLL) {
        double *dst = reinterpret_cast<double *>(zraw);
        for (int j = 0; j < NLL; j++) {
            const double *src = reinterpret_cast<const double *>(j ? ll1 : ll0);
            for (int t = threadIdx.x; t < (int)(sizeof(LLTab) / 8); t += blockDim.x) dst[j * (int)(sizeof(LLTab) / 8) + t] = src[t];
        }
        __syncthreads();
    }
    double cnt = 0., sx = 0., sy = 0.;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    if (MODE >= 2) {
        const int64_t npair = num >> 1;
        for (int64_t q = tid; q < npair; q += nthr) {
            const int64_t i = q << 1;
            Ray a, b;
            fload2(a, b, P, LMc, i);
            ctx.i = i;
            const bool ka = C::run(a, prm, ctx);
            ctx.i = i + 1;
            const bool kb = C::run(b, prm, ctx);
            fstore2(a, b, Q, SMc, i);
            if (alive) { alive[i] = ka ? 1 : 0; alive[i + 1] = kb ? 1 : 0; }
            if (ka) { cnt += 1.; sx += a.x; sy += a.y; }
            if (kb) { cnt += 1.; sx += b.x; sy += b.y; }
        }
        if ((num & 1) && tid == 0) {
            const int64_t i = num - 1;
            Ray a;
            fload1(a, P, LMc, i);
            ctx.i = i;
            const bool ka = C::run(a, prm, ctx);
            fstore1(a, Q, SMc, i);
            if (alive) alive[i] = ka ? 1 : 0;
            if (ka) { cnt += 1.; sx += a.x; sy += a.y; }
        }
    } else {
        for (int64_t i = tid; i < num; i += nthr) {
            Ray a;
            fload1(a, P, LMc, i);
            ctx.i = i;
            // NLL (one ray per thread): the staged tables are addressed per ray through an opaque zero, as in
            // chain_seg_body.  Hoisted out of the loop, their scalars and coefficients stay in registers (ptxas for the
            // LL pair at N = 5, no cap: 254 registers against 154 with the re-addressing).
            if (NLL) {
                int z = 0;
                asm volatile("" : "+r"(z));
                ctx.llt = reinterpret_cast<const LLTab *>(zraw) + z;
            }
            const bool ka = C::run(a, prm, ctx);
            fstore1(a, Q, SMc, i);
            if (alive) alive[i] = ka ? 1 : 0;
            if (ka) { cnt += 1.; sx += a.x; sy += a.y; }
        }
    }
    if (partials) centroid_block_reduce(cnt, sx, sy, partials);
}

// Segmented form (nested assemblies): the bundle is walked in tiles of CHAIN_SEG_TILE consecutive rays; a CTA stages
// the parameter pack of the segment its tile lies in (re-staged only when the segment changes).  ZERN: zern holds one
// Zernike table per segment, staged with the pack.  NLL: ll holds NLL LL tables per segment (segment-major), staged
// likewise.
#define CHAIN_SEG_TILE (PXF_BLOCK * 8)
template <class C, class CP, bool ZERN, int NLL, unsigned LMc, unsigned SMc>
PXF_DEV void chain_seg_body(const RowPtrs &P, const RowPtrs &Q, const int64_t num, uint8_t *__restrict__ alive,
                            const long long *__restrict__ seg_start, const CP *__restrict__ table, const int nseg,
                            const unsigned LMr, const unsigned SMr, const ZernP *__restrict__ zern,
                            const LLTab *__restrict__ ll)
{
    __shared__ __align__(16) CP sp;
    __shared__ __align__(16) unsigned char zraw[ZERN ? sizeof(ZernP) : NLL ? NLL * sizeof(LLTab) : 16];
    const unsigned LM = LMc ? LMc : LMr, SM = SMc ? SMc : SMr;
    ChainCtx ctx = chain_ctx_none();
    int staged = -1;
    for (int64_t t0 = (int64_t)blockIdx.x * CHAIN_SEG_TILE; t0 < num; t0 += (int64_t)gridDim.x * CHAIN_SEG_TILE) {
        const int64_t t1 = t0 + CHAIN_SEG_TILE < num ? t0 + CHAIN_SEG_TILE : num;
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
                if (ZERN) {
                    const double *zsrc = reinterpret_cast<const double *>(zern + seg);
                    double *zdst = reinterpret_cast<double *>(zraw);
                    for (int t = threadIdx.x; t < (int)(sizeof(ZernP) / 8); t += blockDim.x) zdst[t] = zsrc[t];
                }
                if (NLL) {
                    const double *lsrc = reinterpret_cast<const double *>(ll + (int64_t)seg * NLL);
                    double *ldst = reinterpret_cast<double *>(zraw);
                    for (int t = threadIdx.x; t < NLL * (int)(sizeof(LLTab) / 8); t += blockDim.x) ldst[t] = lsrc[t];
                }
                __syncthreads();
                staged = seg;
            }
            for (int64_t i = pos + threadIdx.x; i < send; i += blockDim.x) {
                Ray a;
                fload1(a, P, LM, i);
                // ZERN: the staged pack and table are addressed per ray through an opaque zero.  Hoisted out of this
                // loop their loads would hold ~90 more registers than the fused Zernike kernel does (ptxas, no cap:
                // 242 vs 150) and spill at its 3 CTAs/SM.  NLL: likewise (the LL pair at N = 5, no cap: 255 registers
                // and spills, against 154 with the re-addressing).  Otherwise z is the constant 0.
                int z = 0;
                if (ZERN || NLL) asm volatile("" : "+r"(z));
                if (ZERN) ctx.zt = reinterpret_cast<const ZernP *>(zraw) + z;
                if (NLL) ctx.llt = reinterpret_cast<const LLTab *>(zraw) + z;
                ctx.i = i;                             // (the per-ray arrays are indexed in the whole bundle)
                const bool keep = C::run(a, (&sp)[z], ctx);
                fstore1(a, Q, SM, i);
                if (alive) alive[i] = keep ? 1 : 0;
            }
            pos = send;
            seg++;
        }
    }
}

}  // namespace pxf
