// Fused per-ray program: one kernel loads a ray once, runs a whole op list in registers and
// stores once -- no HBM round trip per optical element.  The per-op arithmetic is the same
// device code as the per-routine kernels (pxf_ray.cuh), so the result is bit-identical to
// issuing the routines one by one.  Every ray runs the same program, so the opcode switch is
// warp-uniform; only Newton trip counts and vignetting diverge.
#include "pxf_program.h"

namespace pxf {

PXF_DEV double ray_row(const Ray &r, int row)
{
    switch (row) {
        case 0: return r.opd; case 1: return r.x; case 2: return r.y; case 3: return r.z;
        case 4: return r.l; case 5: return r.m; case 6: return r.n; case 7: return r.ux;
        case 8: return r.uy; default: return r.uz;
    }
}

// returns false when the ray is vignetted at this op
// ZERN: whether this instantiation carries the Zernike evaluation at all -- it needs ~3x the registers of every
// other op, so programs without a PXF_OP_ZERNSURF op run a kernel compiled without it
// one atomic per warp: the largest grating count seen by the lanes that are here together
PXF_DEV void count_max_update(int *dst, int k)
{
    const unsigned act = __activemask();
    const int m = __reduce_max_sync(act, k);
    if ((threadIdx.x & 31) == (__ffs(act) - 1)) atomicMax(dst, m);
}

// i: the ray's index in the bundle (side arrays); aux_*: FusedProgram::aux_* (null unless the program uses them)
// AUX: whether this instantiation carries the side-array ops (the grating fan: asin + a data-dependent loop) -- like
// ZERN they get their own kernel so that every other program keeps its register budget
// LL: whether it carries the Legendre-Legendre shells (PXF_OP_LLSURF); llt: their tables in shared memory, by slot
// SURF: whether it carries the remaining scalar surfaces (PXF_OP_TRACESPHERE .. PXF_OP_WSSECONDARYBACK)
// TAB: whether it also carries the surfaces read through a device table (PXF_OP_CONICPLUS[OPD], PXF_OP_LEGSURF)
// ZPH: whether it carries the Zernike phase surface (PXF_OP_ZERNPHASE; zt as for ZERN)
// GRAT: whether it carries the gratings with per-ray arrays (PXF_OP_RADGRATW / GRAT) without the fan; AUX carries them too
template <bool ZERN = false, bool AUX = false, bool LL = false, bool SURF = false, bool TAB = false, bool ZPH = false,
          bool GRAT = false>
PXF_DEV bool run_op(Ray &r, const FusedOp &op, const ZernP *zt = nullptr, int64_t i = 0,
                    const double *aux_wave = nullptr, int *aux_count = nullptr, int *aux_count_max = nullptr,
                    const LLTab *llt = nullptr)
{
    switch (op.code) {
        case PXF_OP_KICKN: op_kickn(r, *reinterpret_cast<const KickNP *>(op.q)); break;
        case PXF_OP_VIGNETTE_RHOGT: {
            double rho = sqrt(sq(r.x) + sq(r.y));
            return rho > op.q[0];
        }
        case PXF_OP_GRATFAN:
            if constexpr (AUX) {
                const GratFanP &p = *reinterpret_cast<const GratFanP *>(op.q);
                const int k = op_gratfan(r, p, p.wave_array ? aux_wave[i] : p.g.wave);
                if (aux_count) aux_count[i] = k;
                if (aux_count_max) count_max_update(aux_count_max, k < 0 ? p.cap + 1 : k);
            }
            break;
        case PXF_OP_ROTX_REMAINING:
            if constexpr (AUX) {
                const int k = aux_count[i];
                if (k >= 0) op_rotx_repeat(r, *reinterpret_cast<const TransformP *>(op.q), op.row - k);
            }
            break;
        case PXF_OP_TRANSFORM: op_transform(r, *reinterpret_cast<const TransformP *>(op.q)); break;
        case PXF_OP_ITRANSFORM: op_itransform(r, *reinterpret_cast<const TransformP *>(op.q)); break;
        case PXF_OP_REFLECT: op_reflect(r); break;
        case PXF_OP_REFRACT: op_refract(r, *reinterpret_cast<const RefractP *>(op.q)); break;
        case PXF_OP_RADGRAT: {
            const RadgratP &p = *reinterpret_cast<const RadgratP *>(op.q);
            op_radgrat(r, p, p.wave, false);
            break;
        }
        // the arrays are read at the ray's index i, as the stand-alone kernels read them
        case PXF_OP_RADGRATW:
            if constexpr (AUX || GRAT) {
                const RadgratWP &p = *reinterpret_cast<const RadgratWP *>(op.q);
                op_radgrat(r, p.g, p.wave[i], true);
            }
            break;
        case PXF_OP_GRAT:
            if constexpr (AUX || GRAT) {
                const GratOpP &p = *reinterpret_cast<const GratOpP *>(op.q);
                op_grat(r, p.d, p.order[i], p.wave[i]);
            }
            break;
        case PXF_OP_FLAT: op_flat(r, false, 0.); break;
        case PXF_OP_FLATOPD: op_flat(r, true, op.q[0]); break;
        case PXF_OP_CONIC:
        case PXF_OP_CONICOPD: op_conic(r, *reinterpret_cast<const ConicP *>(op.q)); break;
        // (parameter blocks of the Newton surfaces are copied to registers once: read through the
        // op-indexed constant bank they would be re-fetched by an LDC on every use in every pass)
        case PXF_OP_WOLTERPRIMARY:
        case PXF_OP_WOLTERPRIMARYOPD: { const WolterP p = *reinterpret_cast<const WolterP *>(op.q); op_wolterprimary(r, p); break; }
        case PXF_OP_WOLTERSECONDARY: { const WolterP p = *reinterpret_cast<const WolterP *>(op.q); op_woltersecondary(r, p); break; }
        case PXF_OP_WOLTERSINE: op_woltersine(r, *reinterpret_cast<const WolterSineP *>(op.q)); break;
        case PXF_OP_WSPRIMARY: op_wsprimary(r, *reinterpret_cast<const WSP *>(op.q)); break;
        case PXF_OP_WSSECONDARY: op_wssecondary(r, *reinterpret_cast<const WSP *>(op.q)); break;
        case PXF_OP_SPOCONE: op_spocone(r, *reinterpret_cast<const SpoP *>(op.q)); break;
        case PXF_OP_VIGNETTE_MAG: {
            double mag = sq(r.l) + sq(r.m) + sq(r.n);
            return mag > .1;
        }
        case PXF_OP_VIGNETTE_BOX: {
            double v = ray_row(r, op.row);
            return (v > op.q[0]) && (v < op.q[1]);
        }
        case PXF_OP_VIGNETTE_ABS: {
            double v = ray_row(r, op.row);
            if (op.q[2] != 0.) v = v - op.q[1];        // |row - centre| < hi (the centre is optional: v - 0 is v, but skip it)
            return fabs(v) < op.q[0];
        }
        case PXF_OP_ZERNSURF:
            // zt: the table in shared memory (k_program); same device code as the per-routine kernel (nmax <= 7)
            if constexpr (ZERN) {
                if (zt) op_tracezern<7>(r, zt->rad, zt->nr, zt->tol, zt->nmax, op.q[1] != 0., reinterpret_cast<const double *>(zt->e));
            }
            break;
        case PXF_OP_LLSURF:
            // every table is an 8x8 block padded with zeros: the order-7 evaluation gives the bits of the per-routine
            // kernel of the table's own order (pxf_ray.cuh, LLTab)
            if constexpr (LL) op_ll<PXF_LL_PROG_MAXN, PXF_LL_PROG_MAXN + 1>(r, llt[op.row].s, llt[op.row].C);
            break;
        case PXF_OP_TRACESPHERE:
        case PXF_OP_TRACESPHEREOPD:
            if constexpr (SURF) op_tracesphere(r, *reinterpret_cast<const SphereP *>(op.q));
            break;
        case PXF_OP_TRACECYL:
        case PXF_OP_TRACECYLOPD:
            if constexpr (SURF) op_tracecyl(r, *reinterpret_cast<const SphereP *>(op.q));
            break;
        case PXF_OP_CYLCONIC:
            if constexpr (SURF) { const CylConicP p = *reinterpret_cast<const CylConicP *>(op.q); op_cylconic(r, p); }
            break;
        case PXF_OP_PARAXIAL:
        case PXF_OP_PARAXIALY:
            if constexpr (SURF) op_paraxial(r, *reinterpret_cast<const ParaxialP *>(op.q));
            break;
        case PXF_OP_TORUS:
            if constexpr (SURF) { const TorusP p = *reinterpret_cast<const TorusP *>(op.q); op_torus(r, p); }
            break;
        case PXF_OP_WSPRIMARYBACK:
            if constexpr (SURF) op_wsprimary_t<true>(r, *reinterpret_cast<const WSP *>(op.q));
            break;
        case PXF_OP_WSSECONDARYBACK:
            if constexpr (SURF) op_wssecondary_t<true>(r, *reinterpret_cast<const WSP *>(op.q));
            break;
        // q[0]: the device address of the folded block (warp-uniform, read through L1)
        case PXF_OP_CONICPLUS:
        case PXF_OP_CONICPLUSOPD:
            if constexpr (TAB) op_conicplus(r, **reinterpret_cast<const ConicPlusP *const *>(op.q));
            break;
        case PXF_OP_LEGSURF:
            if constexpr (TAB) op_legsurf(r, **reinterpret_cast<const LegSurfP *const *>(op.q));
            break;
        case PXF_OP_ZERNPHASE:
            // zt: the table in shared memory; q[0] = wave.  Same device code as pxf_zernphase (nmax <= 7)
            if constexpr (ZPH) {
                if (zt) op_zernphase<7>(r, zt->rad, op.q[0], zt->nmax, reinterpret_cast<const double *>(zt->e));
            }
            break;
        case PXF_OP_KICK: {
            r.l = r.l + op.q[0];
            r.m = r.m + op.q[1];
            r.n = op.q[2] * sqrt(1. - sq(r.l) - sq(r.m));
            break;
        }
        default: break;
    }
    return true;
}

template <bool ZERN = false, bool AUX = false, bool LL = false, bool SURF = false, bool TAB = false, bool ZPH = false>
PXF_DEV bool run_program(Ray &r, const FusedProgram &prog, const ZernP *zt = nullptr, int64_t i = 0,
                         const LLTab *llt = nullptr)
{
    for (int k = 0; k < prog.nops; k++)
        if (!run_op<ZERN, AUX, LL, SURF, TAB, ZPH>(r, prog.ops[k], zt, i, prog.aux_wave, prog.aux_count, prog.aux_count_max, llt))
            return false;
    return true;
}

template <int MINB, bool ZERN = false, bool AUX = false, bool LL = false, bool SURF = false, bool TAB = false,
          bool ZPH = false>
__global__ void __launch_bounds__(PXF_BLOCK, MINB)
k_program(const RowPtrs P, const RowPtrs Q, const int64_t num, uint8_t *__restrict__ alive,
          double *__restrict__ partials, const __grid_constant__ FusedProgram prog)
{
    double cnt = 0., sx = 0., sy = 0.;
    // the Zernike table of a PXF_OP_ZERNSURF / ZERNPHASE op, or the tables of the PXF_OP_LLSURF ops, staged once per CTA
    __shared__ __align__(16) unsigned char zraw[(ZERN || ZPH) ? sizeof(ZernP) : LL ? PXF_PROG_MAX_LL * sizeof(LLTab) : 16];
    const ZernP *zt = nullptr;
    const LLTab *llt = nullptr;
    if ((ZERN || ZPH) && prog.zern) {
        const double *src = reinterpret_cast<const double *>(prog.zern);
        double *dst = reinterpret_cast<double *>(zraw);
        for (int t = threadIdx.x; t < (int)(sizeof(ZernP) / 8); t += blockDim.x) dst[t] = src[t];
        __syncthreads();
        zt = reinterpret_cast<const ZernP *>(zraw);
    }
    if (LL) {
        double *dst = reinterpret_cast<double *>(zraw);
        for (int j = 0; j < prog.nll; j++) {
            const double *src = reinterpret_cast<const double *>(prog.ll[j]);
            for (int t = threadIdx.x; t < (int)(sizeof(LLTab) / 8); t += blockDim.x) dst[j * (sizeof(LLTab) / 8) + t] = src[t];
        }
        __syncthreads();
        llt = reinterpret_cast<const LLTab *>(zraw);
    }
    // P: rows read, Q: rows written (Q == P for the in-place f2py semantics)
    const unsigned LM = prog.load_mask, SM = prog.store_mask;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < num; i += nthr) {
        Ray a;
        fload1(a, P, LM, i);
        const bool ka = run_program<ZERN, AUX, LL, SURF, TAB, ZPH>(a, prog, zt, i, llt);
        fstore1(a, Q, SM, i);
        if (alive) alive[i] = ka ? 1 : 0;
        if (ka) { cnt += 1.; sx += a.x; sy += a.y; }
    }
    if (partials) centroid_block_reduce(cnt, sx, sy, partials);
}

// ---------------------------------------------------------------- segmented execution
// Nested assemblies (BASELINE config 5; examples/axro/axialHeights.py:215-322, SMARTX.py:163-259): the bundle
// is a concatenation of segments (one mirror shell each) and every segment runs the SAME opcode sequence with
// its own folded scalars.  The reference loops over shells in Python; one launch per shell is launch bound at
// 260 shells (measured 12 ms of launches for 1e7 rays).  Here one persistent grid walks the bundle in tiles of
// SEG_TILE consecutive rays; a CTA stages the op table of the segment its tile lies in into shared memory
// (re-staged only when the segment changes; a tile that straddles segments is processed piecewise).
// A program with a PXF_OP_ZERNSURF op carries one Zernike table per segment (zern_off: their offset in the table,
// 0 = none); the table of the segment is staged next to its op table.  A program with nll PXF_OP_LLSURF ops carries
// nll LL tables per segment (ll_off), staged the same way.
#define SEG_TILE (PXF_BLOCK * 8)
struct SegHeader {
    unsigned load_mask, store_mask; int nops, nseg; int chain_id, jit_pack_bytes; long long zern_off;
    long long ll_off; int nll, surf;
};
static_assert(sizeof(ZernP) % 16 == 0, "per-segment Zernike tables are laid out back to back, 16-byte aligned");
static_assert(sizeof(LLTab) % 8 == 0, "per-segment LL tables are laid out back to back, whole doubles");

// shared-memory offset of the staged Zernike or LL tables: behind the op table, 16-byte aligned
__host__ __device__ __forceinline__ int seg_zern_smem_offset(int nops) { return (nops * (int)sizeof(FusedOp) + 15) & ~15; }

// ZERN: zern = nseg Zernike tables, one per segment (the Zernike instantiation of run_op, as k_program<.., ZERN = true>)
// LL: ll = nseg * nll LL tables, segment-major (the LL instantiation of run_op, as k_program<.., LL = true>)
// SURF: the remaining scalar surfaces (as k_program<.., SURF = true>); TAB: and the table surfaces (TAB = true)
// ZPH: zern = nseg Zernike tables of PXF_OP_ZERNPHASE ops (as k_program<.., ZPH = true>)
// GRAT: the gratings with per-ray arrays (PXF_OP_RADGRATW / GRAT), read at the ray's index in the whole bundle
template <int MINB, bool ZERN = false, bool LL = false, bool SURF = false, bool TAB = false, bool ZPH = false,
          bool GRAT = false>
__global__ void __launch_bounds__(PXF_BLOCK, MINB)
k_program_seg(const RowPtrs P, const RowPtrs Q, const int64_t num, uint8_t *__restrict__ alive,
              const long long *__restrict__ seg_start, const FusedOp *__restrict__ ops, const int nops, const int nseg,
              const unsigned LM, const unsigned SM, const ZernP *__restrict__ zern, const LLTab *__restrict__ ll,
              const int nll)
{
    extern __shared__ __align__(16) unsigned char seg_smem[];
    FusedOp *sops = reinterpret_cast<FusedOp *>(seg_smem);
    ZernP *zt = (ZERN || ZPH) ? reinterpret_cast<ZernP *>(seg_smem + seg_zern_smem_offset(nops)) : nullptr;
    LLTab *llt = LL ? reinterpret_cast<LLTab *>(seg_smem + seg_zern_smem_offset(nops)) : nullptr;
    int staged = -1;
    const int words = nops * (int)(sizeof(FusedOp) / 8);
    for (int64_t t0 = (int64_t)blockIdx.x * SEG_TILE; t0 < num; t0 += (int64_t)gridDim.x * SEG_TILE) {
        const int64_t t1 = t0 + SEG_TILE < num ? t0 + SEG_TILE : num;
        seg_tile_pieces(t0, t1, seg_start, nseg, [&](int seg, int64_t pos, int64_t send) {
            if (seg != staged) {                       // block-uniform
                __syncthreads();
                const double *src = reinterpret_cast<const double *>(ops + (int64_t)seg * nops);
                double *dst = reinterpret_cast<double *>(sops);
                for (int t = threadIdx.x; t < words; t += blockDim.x) dst[t] = src[t];
                if (ZERN || ZPH) {
                    const double *zsrc = reinterpret_cast<const double *>(zern + seg);
                    double *zdst = reinterpret_cast<double *>(zt);
                    for (int t = threadIdx.x; t < (int)(sizeof(ZernP) / 8); t += blockDim.x) zdst[t] = zsrc[t];
                }
                if (LL) {
                    const double *lsrc = reinterpret_cast<const double *>(ll + (int64_t)seg * nll);
                    double *ldst = reinterpret_cast<double *>(llt);
                    for (int t = threadIdx.x; t < nll * (int)(sizeof(LLTab) / 8); t += blockDim.x) ldst[t] = lsrc[t];
                }
                __syncthreads();
                staged = seg;
            }
            for (int64_t i = pos + threadIdx.x; i < send; i += blockDim.x) {
                Ray a;
                fload1(a, P, LM, i);
                bool keep = true;
                for (int k = 0; k < nops; k++)
                    if (!run_op<ZERN, false, LL, SURF, TAB, ZPH, GRAT>(a, sops[k], zt, i, nullptr, nullptr, nullptr, llt)) { keep = false; break; }
                fstore1(a, Q, SM, i);
                if (alive) alive[i] = keep ? 1 : 0;
            }
        });
    }
}

// rows read (use) / possibly written (st) / unconditionally overwritten (kill) by each op
static void op_masks(int code, int row, unsigned &use, unsigned &st, unsigned &kill)
{
    switch (code) {
        case PXF_OP_TRANSFORM: case PXF_OP_ITRANSFORM: use = R_NINE; st = R_NINE; kill = R_NINE; break;
        case PXF_OP_REFLECT: use = R_DIR | R_NRM; st = R_DIR; kill = R_DIR; break;
        case PXF_OP_REFRACT: use = R_DIR | R_NRM; st = R_DIR | R_NRM; kill = 0; break;
        case PXF_OP_RADGRAT: case PXF_OP_RADGRATW: use = R_X | R_Y | R_DIR; st = R_DIR; kill = R_DIR; break;
        // a ray whose kick leaves l^2+m^2 > 1 gets l = m = n = 0: the direction is written either way
        case PXF_OP_GRAT: use = R_DIR; st = R_DIR; kill = R_DIR; break;
        case PXF_OP_FLAT: use = R_POS | R_DIR; st = R_POS | R_NRM; kill = R_POS | R_NRM; break;
        case PXF_OP_FLATOPD: use = R_POS | R_DIR | R_OPD; st = R_POS | R_NRM | R_OPD; kill = R_POS | R_NRM; break;
        case PXF_OP_CONIC: case PXF_OP_SPOCONE: use = R_NINE; st = R_NINE; kill = 0; break;
        case PXF_OP_CONICOPD: use = R_ALL; st = R_ALL; kill = 0; break;
        case PXF_OP_WOLTERPRIMARY: case PXF_OP_WOLTERSECONDARY: case PXF_OP_WOLTERSINE:
            use = R_POS | R_DIR; st = R_POS | R_NRM; kill = R_POS | R_NRM; break;
        case PXF_OP_WOLTERPRIMARYOPD:
            use = R_POS | R_DIR | R_OPD; st = R_POS | R_NRM | R_OPD; kill = R_POS | R_NRM; break;
        case PXF_OP_WSPRIMARY: case PXF_OP_WSSECONDARY: use = R_NINE; st = R_POS | R_NRM; kill = R_POS; break;
        case PXF_OP_VIGNETTE_MAG: use = R_DIR; st = 0; kill = 0; break;
        case PXF_OP_VIGNETTE_BOX: case PXF_OP_VIGNETTE_ABS: use = 1u << row; st = 0; kill = 0; break;
        case PXF_OP_KICK: use = R_L | R_M; st = R_DIR; kill = R_N; break;
        case PXF_OP_KICKN: use = R_DIR; st = R_DIR; kill = 0; break;
        case PXF_OP_VIGNETTE_RHOGT: use = R_X | R_Y; st = 0; kill = 0; break;
        case PXF_OP_GRATFAN: case PXF_OP_ROTX_REMAINING: use = R_NINE; st = R_NINE; kill = 0; break;
        case PXF_OP_ZERNSURF: use = R_POS | R_DIR | (row ? R_OPD : 0u); st = R_POS | R_NRM | (row ? R_OPD : 0u); kill = R_POS | R_NRM; break;
        case PXF_OP_LLSURF: use = R_POS | R_DIR; st = R_POS | R_NRM; kill = R_POS | R_NRM; break;
        // a ray that misses the sphere / cylinder is zeroed, direction included: the direction is stored, not killed
        case PXF_OP_TRACESPHERE: case PXF_OP_TRACECYL: use = R_POS | R_DIR; st = R_NINE; kill = R_POS | R_NRM; break;
        case PXF_OP_TRACESPHEREOPD: case PXF_OP_TRACECYLOPD:
            use = R_POS | R_DIR | R_OPD; st = R_NINE | R_OPD; kill = R_POS | R_NRM; break;
        case PXF_OP_CYLCONIC: case PXF_OP_TORUS: use = R_POS | R_DIR; st = R_POS | R_NRM; kill = R_POS | R_NRM; break;
        case PXF_OP_PARAXIAL: use = R_X | R_Y | R_L | R_M; st = R_L | R_M; kill = R_L | R_M; break;
        case PXF_OP_PARAXIALY: use = R_Y | R_M; st = R_M; kill = R_M; break;
        case PXF_OP_WSPRIMARYBACK: case PXF_OP_WSSECONDARYBACK: use = R_NINE; st = R_POS | R_NRM; kill = R_POS; break;
        case PXF_OP_CONICPLUS: use = R_POS | R_DIR; st = R_POS | R_NRM; kill = R_POS | R_NRM; break;
        case PXF_OP_CONICPLUSOPD: use = R_POS | R_DIR | R_OPD; st = R_POS | R_NRM | R_OPD; kill = R_POS | R_NRM; break;
        // the phase surfaces kick the direction they read (legsurf keeps the sign of n): nothing is killed
        case PXF_OP_LEGSURF: use = R_X | R_Y | R_DIR; st = R_DIR; kill = 0; break;
        case PXF_OP_ZERNPHASE: use = R_X | R_Y | R_DIR | R_OPD; st = R_DIR | R_OPD; kill = 0; break;
        default: use = 0; st = 0; kill = 0; break;
    }
}

static bool is_table_surface_op(int code)
{
    return code == PXF_OP_CONICPLUS || code == PXF_OP_CONICPLUSOPD || code == PXF_OP_LEGSURF;
}
// the surface family: ops 27..36 and the table surfaces
static bool is_surface_op(int code)
{
    return (code >= PXF_OP_TRACESPHERE && code <= PXF_OP_WSSECONDARYBACK) || is_table_surface_op(code);
}
// which of the interpreters of the newer table ops an op list needs (read from the ops, so that FusedProgram, the
// parameter of every k_program, keeps its layout)
static void new_table_kinds(const FusedOp *ops, int nops, bool &zphase, bool &tabsurf)
{
    zphase = tabsurf = false;
    for (int k = 0; k < nops; k++) {
        zphase = zphase || ops[k].code == PXF_OP_ZERNPHASE;
        tabsurf = tabsurf || is_table_surface_op(ops[k].code);
    }
}
// the gratings with per-ray arrays, which run in the side-array interpreters
static bool is_array_op(int code) { return code == PXF_OP_RADGRATW || code == PXF_OP_GRAT; }
static bool has_array_ops(const FusedOp *ops, int nops)
{
    for (int k = 0; k < nops; k++)
        if (is_array_op(ops[k].code)) return true;
    return false;
}
static bool is_table_or_aux_op(int code)
{
    return code == PXF_OP_ZERNSURF || code == PXF_OP_LLSURF || code == PXF_OP_GRATFAN || code == PXF_OP_ROTX_REMAINING ||
           code == PXF_OP_ZERNPHASE;
}

int build_program(FusedProgram &fp, const pxf_op *ops, int nops, const pxf_program_aux *aux)
{
    if (!ops || nops < 1 || nops > PXF_MAX_OPS) { set_error("program: need 1..%d ops", PXF_MAX_OPS); return PXF_ERR_INVALID; }
    memset(&fp, 0, sizeof(fp));
    fp.nops = nops;
    // the remaining scalar surfaces run in an interpreter of their own, which holds no table or side-array op: refused
    // before anything else is checked, so the verdict does not depend on the order of the ops
    bool surf = false, other = false, arrays = false, zll = false;
    int zphase = 0, tables = 0;                // PXF_OP_ZERNPHASE ops; ops with a Zernike or LL table or a side array
    for (int k = 0; k < nops; k++) {
        arrays = arrays || is_array_op(ops[k].code);
        zll = zll || ops[k].code == PXF_OP_ZERNSURF || ops[k].code == PXF_OP_ZERNPHASE || ops[k].code == PXF_OP_LLSURF;
        surf = surf || is_surface_op(ops[k].code);
        other = other || is_table_or_aux_op(ops[k].code);
        zphase += ops[k].code == PXF_OP_ZERNPHASE;
        tables += is_table_or_aux_op(ops[k].code);
    }
    // the gratings with per-ray arrays run in the side-array interpreters, which hold no table op and no surface of the
    // family: the combinations would need interpreters of their own
    if (arrays && (surf || zll)) {
        set_error("program: PXF_OP_RADGRATW / GRAT cannot share a program with a Zernike surface or phase, a "
                  "Legendre-Legendre shell or the sphere / cylinder / cylconic / paraxial / torus / W-S back-surface / "
                  "conicplus / legsurf ops");
        return PXF_ERR_UNSUPPORTED;
    }
    if (surf && other) {
        set_error("program: the sphere / cylinder / cylconic / paraxial / torus / W-S back-surface / conicplus / legsurf "
                  "ops cannot share a program with a Zernike surface or phase, a Legendre-Legendre shell or a grating fan");
        return PXF_ERR_UNSUPPORTED;
    }
    // the Zernike phase surface runs in an interpreter of its own, which holds no other table or side-array op
    if (zphase && tables > 1) {
        set_error("program: a Zernike phase surface cannot share a program with another Zernike surface or phase, a "
                  "Legendre-Legendre shell or a grating fan");
        return PXF_ERR_UNSUPPORTED;
    }
    fp.surf = surf ? 1 : 0;
    if (aux) { fp.aux_wave = aux->wave; fp.aux_count = aux->count; fp.aux_count_max = aux->count_max; }
    unsigned store = 0;
    for (int k = 0; k < nops; k++) {
        const pxf_op &o = ops[k];
        FusedOp &f = fp.ops[k];
        f.code = o.code;
        f.row = 0;
        const double *p = o.p;
        switch (o.code) {
            case PXF_OP_TRANSFORM: { TransformP t = make_transform(p[0], p[1], p[2], p[3], p[4], p[5]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_ITRANSFORM: { TransformP t = make_itransform(p[0], p[1], p[2], p[3], p[4], p[5]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_REFLECT: case PXF_OP_FLAT: case PXF_OP_VIGNETTE_MAG: break;
            case PXF_OP_REFRACT: { RefractP t; t.ratio = p[0] / p[1]; memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_RADGRAT: { RadgratP t = make_radgrat(p[0], p[1], p[2]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_FLATOPD: f.q[0] = p[0]; break;
            // the arrays' device addresses, bit-cast into the doubles; folded as pxf_radgratw / pxf_grat fold the scalars
            case PXF_OP_RADGRATW: {
                RadgratWP t;
                t.g = make_radgrat(0., p[1], p[2]);
                memcpy(&t.wave, &p[0], sizeof(t.wave));
                if (!t.wave) { set_error("program: PXF_OP_RADGRATW needs a device wave array"); return PXF_ERR_INVALID; }
                memcpy(f.q, &t, sizeof(t));
                break;
            }
            case PXF_OP_GRAT: {
                GratOpP t;
                t.d = p[0];
                memcpy(&t.order, &p[1], sizeof(t.order));
                memcpy(&t.wave, &p[2], sizeof(t.wave));
                if (!t.order || !t.wave) { set_error("program: PXF_OP_GRAT needs device order and wave arrays"); return PXF_ERR_INVALID; }
                memcpy(f.q, &t, sizeof(t));
                break;
            }
            case PXF_OP_CONIC: { ConicP t = make_conic(p[0], p[1], false, 0.); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_CONICOPD: { ConicP t = make_conic(p[0], p[1], true, p[2]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_WOLTERPRIMARY: { WolterP t = make_wolter(p[0], p[1], p[2], false, 0.); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_WOLTERPRIMARYOPD: { WolterP t = make_wolter(p[0], p[1], p[2], true, p[3]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_WOLTERSECONDARY: { WolterP t = make_wolter(p[0], p[1], p[2], false, 0.); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_WOLTERSINE: { WolterSineP t = make_woltersine(p[0], p[1], p[2], p[3]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_WSPRIMARY: case PXF_OP_WSSECONDARY: { WSP t = make_ws(p[0], p[1], p[2]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_SPOCONE: { SpoP t = make_spo(p[0], p[1]); memcpy(f.q, &t, sizeof(t)); break; }
            // folded as the stand-alone entry points of pxf_ops.cu fold them
            case PXF_OP_TRACESPHERE: case PXF_OP_TRACECYL: { SphereP t = make_sphere(p[0], false, 0.); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_TRACESPHEREOPD: case PXF_OP_TRACECYLOPD: { SphereP t = make_sphere(p[0], true, p[1]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_CYLCONIC: { CylConicP t = make_cylconic(p[0], p[1]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_PARAXIAL: { ParaxialP t{p[0], 0, 0}; memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_PARAXIALY: { ParaxialP t{p[0], 1, 0}; memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_TORUS: { TorusP t = make_torus(p[0], p[1]); memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_WSPRIMARYBACK: case PXF_OP_WSSECONDARYBACK: { WSP t = make_ws(p[0], p[1], p[2], p[3]); memcpy(f.q, &t, sizeof(t)); break; }
            // the device table's address (folded by pxf_conicplus_table_fill / pxf_legsurf_table_fill)
            case PXF_OP_CONICPLUS: case PXF_OP_CONICPLUSOPD: case PXF_OP_LEGSURF: {
                const void *tab;
                memcpy(&tab, &p[0], sizeof(tab));
                if (!tab) { set_error("program: PXF_OP_CONICPLUS / CONICPLUSOPD / LEGSURF need a device table"); return PXF_ERR_INVALID; }
                memcpy(f.q, &tab, sizeof(tab));
                break;
            }
            case PXF_OP_ZERNPHASE: {
                const ZernP *tab;
                memcpy(&tab, &p[0], sizeof(tab));
                if (!tab) { set_error("program: PXF_OP_ZERNPHASE needs a device table"); return PXF_ERR_INVALID; }
                if (!(p[2] >= 0. && p[2] <= 7.)) { set_error("program: PXF_OP_ZERNPHASE supports radial orders <= 7 (use pxf_zernphase)"); return PXF_ERR_UNSUPPORTED; }
                fp.zern = tab;
                f.q[0] = p[1];                         // wave
                break;
            }
            case PXF_OP_VIGNETTE_BOX:
                f.row = (int)p[0];
                if (f.row < 0 || f.row > 9) { set_error("program: bad row in VIGNETTE_BOX"); return PXF_ERR_INVALID; }
                f.q[0] = p[1]; f.q[1] = p[2];
                break;
            case PXF_OP_VIGNETTE_ABS:
                f.row = (int)p[0];
                if (f.row < 0 || f.row > 9) { set_error("program: bad row in VIGNETTE_ABS"); return PXF_ERR_INVALID; }
                f.q[0] = p[1]; f.q[1] = p[2]; f.q[2] = (p[2] != 0.) ? 1. : 0.;
                break;
            case PXF_OP_KICK: f.q[0] = p[0]; f.q[1] = p[1]; f.q[2] = p[2]; break;
            case PXF_OP_KICKN: { KickNP t; t.dl = p[0]; t.dm = p[1]; t.dl2 = p[0] * p[0]; t.dm2 = p[1] * p[1]; memcpy(f.q, &t, sizeof(t)); break; }
            case PXF_OP_VIGNETTE_RHOGT: f.q[0] = p[0]; break;
            case PXF_OP_GRATFAN: {
                // p: ang, hubdist, l, dpermm, order, wave (NaN: per-ray wavelengths).  The script's
                // tran.transform(rays,0,0,0,ang,0,0) reaches the Fortran negated (transformations.py:29).
                GratFanP t;
                memset(&t, 0, sizeof(t));
                t.rot = make_transform(0., 0., 0., -p[0], 0., 0.);
                t.wave_array = (p[5] != p[5]) ? 1 : 0;
                t.g = make_radgrat(t.wave_array ? 0. : p[5], p[3], p[4]);
                t.hub = p[1]; t.hub_l = p[2] + p[1]; t.thresh = .001;
                t.cap = (aux && aux->cap > 0) ? aux->cap : 4096;
                if (t.wave_array && !(aux && aux->wave)) { set_error("program: PXF_OP_GRATFAN with wave = NaN needs aux.wave"); return PXF_ERR_INVALID; }
                memcpy(f.q, &t, sizeof(t));
                fp.uses_aux = 1;
                break;
            }
            case PXF_OP_ROTX_REMAINING: {
                if (!(aux && aux->count)) { set_error("program: PXF_OP_ROTX_REMAINING needs aux.count"); return PXF_ERR_INVALID; }
                if (!(p[1] >= 0. && p[1] <= 1.e6)) { set_error("program: PXF_OP_ROTX_REMAINING: bad total"); return PXF_ERR_INVALID; }
                TransformP t = make_transform(0., 0., 0., -p[0], 0., 0.);
                memcpy(f.q, &t, sizeof(t));
                f.row = (int)p[1];                     // total rotations of the loop
                f.q[sizeof(TransformP) / 8] = (double)f.row;     // (RotxP of the specialised chains)
                fp.uses_aux = 1;
                break;
            }
            case PXF_OP_ZERNSURF: {
                const ZernP *tab;
                memcpy(&tab, &p[0], sizeof(tab));
                if (!tab || fp.zern) { set_error("program: PXF_OP_ZERNSURF needs a device table, and only one per program"); return PXF_ERR_INVALID; }
                if (!(p[2] >= 0. && p[2] <= 7.)) { set_error("program: PXF_OP_ZERNSURF supports radial orders <= 7 (use pxf_tracezern)"); return PXF_ERR_UNSUPPORTED; }
                fp.zern = tab;
                f.q[0] = 0.; f.q[1] = p[1] != 0. ? 1. : 0.;
                f.row = p[1] != 0. ? 1 : 0;            // opd flag: decides whether row 0 is touched
                break;
            }
            case PXF_OP_LLSURF: {
                const LLTab *tab;
                memcpy(&tab, &p[0], sizeof(tab));
                if (!tab) { set_error("program: PXF_OP_LLSURF needs a device table"); return PXF_ERR_INVALID; }
                if (!(p[1] >= 0. && p[1] <= PXF_LL_PROG_MAXN)) {
                    set_error("program: PXF_OP_LLSURF supports Legendre orders <= %d (use pxf_wolterprimll and the other "
                              "stand-alone routines)", PXF_LL_PROG_MAXN);
                    return PXF_ERR_UNSUPPORTED;
                }
                if (fp.nll == PXF_PROG_MAX_LL) {
                    set_error("program: at most %d PXF_OP_LLSURF ops per program", PXF_PROG_MAX_LL);
                    return PXF_ERR_UNSUPPORTED;
                }
                // q: the order N the specialised kernels evaluate (make_ll's rounding), the table slot
                const int top = (int)p[1];
                f.q[0] = top <= 3 ? 3. : top <= 5 ? 5. : 7.;
                f.q[1] = (double)fp.nll;
                f.row = fp.nll;
                fp.ll[fp.nll++] = tab;
                break;
            }
            default: set_error("program: unknown opcode %d", o.code); return PXF_ERR_INVALID;
        }
        if (o.code == PXF_OP_VIGNETTE_MAG || o.code == PXF_OP_VIGNETTE_BOX || o.code == PXF_OP_VIGNETTE_ABS ||
            o.code == PXF_OP_VIGNETTE_RHOGT)
            fp.has_vignette = 1;
        unsigned use, st, kill;
        op_masks(o.code, f.row, use, st, kill);
        store |= st;
        // forward constant tracking: whatever this op writes is no longer a known constant, except
        // the plane's own outputs z = 0, u = (0,0,1) (surfacesf.f95:17-23)
        fp.const_mask &= ~st;
        if (o.code == PXF_OP_FLAT || o.code == PXF_OP_FLATOPD) {
            fp.const_mask |= R_Z | R_NRM;
            fp.const_val[3] = 0.; fp.const_val[7] = 0.; fp.const_val[8] = 0.; fp.const_val[9] = 1.;
        }
    }
    if (fp.nll && (fp.zern || fp.uses_aux)) {
        set_error("program: Legendre-Legendre shells cannot share a program with a Zernike surface or a grating fan");
        return PXF_ERR_UNSUPPORTED;
    }
    if (fp.has_vignette) fp.const_mask = 0;
    // Backward liveness: a row is read from HBM only if some op consumes its incoming value
    // before an op overwrites it unconditionally (e.g. the normals entering a transform that is
    // followed by a surface are dead: never loaded, never rotated).  Every row any op may write
    // is live at the end (it is stored).
    unsigned live = store;
    for (int k = nops - 1; k >= 0; k--) {
        FusedOp &f = fp.ops[k];
        unsigned use, st, kill;
        op_masks(f.code, f.row, use, st, kill);
        if (f.code == PXF_OP_TRANSFORM || f.code == PXF_OP_ITRANSFORM) {
            // position / direction / normal triplets transform independently
            unsigned groups = 0, in = live & ~R_NINE;
            if (live & R_POS) { groups |= 1; in |= R_POS; }
            if (live & R_DIR) { groups |= 2; in |= R_DIR; }
            if (live & R_NRM) { groups |= 4; in |= R_NRM; }
            reinterpret_cast<TransformP *>(f.q)->groups = (int)groups;
            live = in;
        } else {
            const bool side_effect = (st == 0);   // vignette predicates
            unsigned in = live & ~kill;
            if ((st & live) || side_effect) in |= use;
            live = in;
        }
    }
    fp.load_mask = live;
    fp.store_mask = store;
    // A ray stopped by a vignette predicate is stored in the state it had AT the predicate (the contract for dead
    // rays: whatever the ops before the predicate made of them, nothing after).  Rows a later op would have
    // overwritten are dead for the survivors but not for the stopped rays, so they must be loaded as well.
    if (fp.has_vignette) fp.load_mask |= store;
    return PXF_OK;
}

// Register cap (resident CTAs per SM) of the interpreter of the remaining scalar surfaces, k_program<surf> and
// k_program_seg<surf>.  ptxas: 120 registers uncapped (1 and 2 CTAs/SM are the same kernel), 80 with 0.1 KB of spills at
// 3, 64 with 0.2 KB at 4.  Measured at 5e7 rays, out of place, on one B200 (1000 W), caps 2 / 3 / 4: tracesphere 5.55 /
// 4.88 / 5.39 ms, paraxial 4.73 / 4.23 / 4.59, wssecondaryback 7.74 / 6.93 / 7.18, torus 3.11 / 3.59 / 3.51, the
// 1000-segment lens 17.4 / 13.8 / 15.2 (profiles/surface_ops_bench_b200.json)
#define SURF_MINB 3
// ... and of the interpreters with the table surfaces (k_program<tabsurf>, the surface family plus conicplus / legsurf)
// and with the Zernike phase surface (k_program<zphase>), and their segmented forms.  Not swept: the cap of
// k_program<surf>, whose ops they hold, and of k_program<zernike> (ZERN_MINB), whose table staging they share.
// ptxas at 3: 80 registers and 128 / 112 B of spill stores.
#define TABSURF_MINB 3
#define ZPHASE_MINB 3
// ... of the Zernike interpreter, k_program<zernike> and k_program_seg<zernike>.  Measured on config 3's 14-op program at
// 5e7 rays, caps 1 / 2 / 3 / 4: 9.40 / 6.28 / 6.01 / 6.28 ms; the same work as three launches (transform, tracezern,
// 12-op tail) takes 7.0 ms
#define ZERN_MINB 3
// ... of the Legendre-Legendre interpreter, k_program<ll> and k_program_seg<ll>.  Measured on the LL pair (36 terms per
// mirror) at 5e7 rays, out of place, one B200 at 1000 W, caps 1 / 2 / 3 / 4: 11.6 / 13.7 / 20.2 / 28.2 ms (1: 212
// registers, no spills; 2-4 spill 0.4-0.8 KB); with 16 / 64 terms 11.9 / 12.7 ms at 1 CTA/SM
// (profiles/ll_program_bench_b200.json)
#define LL_MINB 1

int launch_program(double *const rays[10], int64_t num, const FusedProgram &fp, uint8_t *alive, cudaStream_t s,
                   double *const rays_out[10], double *partials, int *grid_out)
{
    if (num < 0 || !rays) { set_error("program: bad argument"); return PXF_ERR_INVALID; }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    if (fp.has_vignette && !alive) { set_error("program with a VIGNETTE op needs an alive array"); return PXF_ERR_INVALID; }
    if (num == 0) return PXF_OK;
    RowPtrs P, Q;
    bool aligned = true;
    for (int k = 0; k < 10; k++) {
        P.p[k] = rays[k];
        Q.p[k] = rays_out ? rays_out[k] : rays[k];
        if (fp.load_mask & (1u << k)) {
            if (!P.p[k]) { set_error("program: null input row pointer (row %d)", k); return PXF_ERR_INVALID; }
            if (reinterpret_cast<uintptr_t>(P.p[k]) & 15) aligned = false;
        }
        if (fp.store_mask & (1u << k)) {
            if (!Q.p[k]) { set_error("program: null output row pointer (row %d)", k); return PXF_ERR_INVALID; }
            if (reinterpret_cast<uintptr_t>(Q.p[k]) & 15) aligned = false;
        }
    }
    {
        // statically specialised kernel for the canonical chains, else the interpreter below
        int rc = launch_chain(P, Q, num, fp, alive, aligned, s, partials, grid_out);
        if (rc != PXF_ERR_UNSUPPORTED) return rc;
        // ... else a kernel specialised for this op list at run time (NVRTC, cached), else the interpreter
        rc = jit_launch_chain(P, Q, num, fp, alive, aligned, s, partials, grid_out);
        if (rc != PXF_ERR_UNSUPPORTED) return rc;
    }
    // every interpreter runs one ray per thread
    auto go = [&](auto kern) {
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, PXF_BLOCK, 0) != cudaSuccess || nb <= 0) { cudaGetLastError(); nb = 2; }
        const int grid = grid_for(num, PXF_BLOCK, nb);
        if (grid_out) *grid_out = grid;
        kern<<<grid, PXF_BLOCK, 0, s>>>(P, Q, num, alive, partials, fp);
    };
    bool zphase, tabsurf;
    new_table_kinds(fp.ops, fp.nops, zphase, tabsurf);
    const bool arrays = has_array_ops(fp.ops, fp.nops);
    if (fp.uses_aux || arrays) {
        if (fp.zern) { set_error("program: a Zernike surface and a grating fan in one program are not supported"); return PXF_ERR_UNSUPPORTED; }
        go(k_program<3, false, true>);
    }
    else if (zphase) go(k_program<ZPHASE_MINB, false, false, false, false, false, true>);
    else if (fp.zern) go(k_program<ZERN_MINB, true>);
    else if (fp.nll) go(k_program<LL_MINB, false, false, true>);
    else if (tabsurf) go(k_program<TABSURF_MINB, false, false, false, true, true>);
    else if (fp.surf) go(k_program<SURF_MINB, false, false, false, true>);
    // capped for 4 resident CTAs per SM.  Measured on config 3's 12-op tail at 5e7 rays (profiles/r01h_notes.md): two
    // rays per thread (double2 rows) 3.82 ms; one ray per thread capped for 1 / 3 / 4 CTAs/SM 3.75 / 3.27 / 3.00 ms (5
    // and 6 CTAs/SM spill: 4.6 / 5.7 ms)
    else go(k_program<4>);
    count_launch();
    note_kernel(zphase ? "k_program<zphase> (interpreter)" : fp.zern ? "k_program<zernike> (interpreter)" :
                (fp.uses_aux || arrays) ? "k_program<aux> (interpreter)" : fp.nll ? "k_program<ll> (interpreter)" :
                tabsurf ? "k_program<tabsurf> (interpreter)" : fp.surf ? "k_program<surf> (interpreter)" :
                "k_program (interpreter)");
    return check_launch("k_program");
}

}  // namespace pxf

using namespace pxf;
// pxf_analysis.cu
namespace pxf { int sums_finalize(const double *partial, int nblocks, int ns, double *out_dev, cudaStream_t s); }

extern "C" int pxf_trace_program(double *const rays[10], int64_t num, const pxf_op *ops, int32_t nops,
                                 uint8_t *alive, pxf_stream_t stream)
{
    FusedProgram fp;
    int rc = build_program(fp, ops, nops);
    if (rc) return rc;
    return launch_program(rays, num, fp, alive, reinterpret_cast<cudaStream_t>(stream), nullptr, nullptr, nullptr);
}

extern "C" int pxf_trace_program_to(double *const rays_in[10], double *const rays_out[10], int64_t num,
                                    const pxf_op *ops, int32_t nops, uint8_t *alive, pxf_stream_t stream)
{
    if (!rays_out) { set_error("pxf_trace_program_to: null output table"); return PXF_ERR_INVALID; }
    FusedProgram fp;
    int rc = build_program(fp, ops, nops);
    if (rc) return rc;
    // out of place: rows that are read but never written must still appear in the output
    // bundle, so every row the program touches is stored
    fp.store_mask |= fp.load_mask;
    return launch_program(rays_in, num, fp, alive, reinterpret_cast<cudaStream_t>(stream), rays_out, nullptr, nullptr);
}

extern "C" int pxf_trace_program_aux(double *const rays_in[10], double *const rays_out[10], int64_t num,
                                     const pxf_op *ops, int32_t nops, uint8_t *alive, const pxf_program_aux *aux,
                                     double *sums_dev, void *scratch, pxf_stream_t stream)
{
    FusedProgram fp;
    int rc = build_program(fp, ops, nops, aux);
    if (rc) return rc;
    if (rays_out) fp.store_mask |= fp.load_mask;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (!sums_dev) return launch_program(rays_in, num, fp, alive, s, rays_out, nullptr, nullptr);
    if (!scratch) { set_error("pxf_trace_program_aux: sums need scratch"); return PXF_ERR_INVALID; }
    fp.load_mask |= (R_X | R_Y) & ~fp.store_mask;
    if (num == 0) {
        PXF_CUDA(cudaMemsetAsync(sums_dev, 0, 4 * sizeof(double), s));
        return PXF_OK;
    }
    int grid = 0;
    rc = launch_program(rays_in, num, fp, alive, s, rays_out, static_cast<double *>(scratch), &grid);
    if (rc) return rc;
    return sums_finalize(static_cast<const double *>(scratch), grid, 4, sums_dev, s);
}

extern "C" size_t pxf_zern_table_bytes(void) { return sizeof(ZernP); }

extern "C" int32_t pxf_zern_table_fill(const double *coeff, const int32_t *rorder, const int32_t *aorder, int32_t arrsize,
                                       double rad, int32_t opd, double nr, void *table_host)
{
    if (!coeff || !rorder || !aorder || arrsize <= 0 || !table_host) { set_error("pxf_zern_table_fill: bad argument"); return -1; }
    ZernP z;
    const int n = make_zern(z, coeff, rorder, aorder, arrsize, rad, opd != 0, nr);
    if (n < 0) { set_error("pxf_zern_table_fill: invalid Zernike table"); return -1; }
    memcpy(table_host, &z, sizeof(z));
    return n;
}

extern "C" size_t pxf_ll_table_bytes(void) { return sizeof(LLTab); }

extern "C" int32_t pxf_ll_table_fill(int32_t kind, double r0, double z0, double psi, double S, double zmax, double zmin,
                                     double dphi, const double *coeff, const int32_t *axial, const int32_t *az,
                                     int32_t cnum, void *table_host)
{
    if (!coeff || !axial || !az || cnum <= 0 || !table_host || kind < 0 || kind > 2) {
        set_error("pxf_ll_table_fill: bad argument");
        return -1;
    }
    // folded by the routine of the stand-alone kernels, so every scalar and coefficient has the same bits
    LLP q;
    if (make_ll(q, kind, r0, z0, psi, S, zmax, zmin, dphi, coeff, axial, az, cnum) < 0) {
        set_error("pxf_ll_table_fill: invalid Legendre orders (need 0 <= order <= %d)", PXF_LL_MAXN);
        return -1;
    }
    const int top = q.s.nz > q.s.nt ? q.s.nz : q.s.nt;
    if (top > PXF_LL_PROG_MAXN) {
        set_error("pxf_ll_table_fill: programs hold Legendre orders <= %d (this list has %d; use the stand-alone routine)",
                  PXF_LL_PROG_MAXN, top);
        return -1;
    }
    LLTab t;
    memset(&t, 0, sizeof(t));
    t.s = q.s;
    const int N = q.s.stride - 1;
    for (int a = 0; a <= N; a++)
        for (int b = 0; b <= N; b++) t.C[a * (PXF_LL_PROG_MAXN + 1) + b] = q.C[a * q.s.stride + b];
    memcpy(table_host, &t, sizeof(t));
    return top;
}

// the two make_zern steps of pxf_tracezernrot, in that order
extern "C" int32_t pxf_zern_table_fill_rot(const double *coeff1, const int32_t *rorder1, const int32_t *aorder1,
                                           int32_t arrsize1, const double *coeff2, const int32_t *rorder2,
                                           const int32_t *aorder2, int32_t arrsize2, double rad, double rot,
                                           void *table_host)
{
    if (!coeff1 || !rorder1 || !aorder1 || arrsize1 <= 0 || !coeff2 || !rorder2 || !aorder2 || arrsize2 <= 0 || !table_host) {
        set_error("pxf_zern_table_fill_rot: bad argument");
        return -1;
    }
    ZernP z;
    if (make_zern(z, coeff1, rorder1, aorder1, arrsize1, rad, false, 0.) < 0 ||
        make_zern(z, coeff2, rorder2, aorder2, arrsize2, rad, false, 0., rot, true) < 0) {
        set_error("pxf_zern_table_fill_rot: invalid Zernike table");
        return -1;
    }
    memcpy(table_host, &z, sizeof(z));
    return z.nmax;
}

extern "C" size_t pxf_conicplus_table_bytes(void) { return sizeof(ConicPlusP); }

extern "C" int32_t pxf_conicplus_table_fill(double R, double K, const double *p, int32_t np, int32_t opd, double nr,
                                            void *table_host)
{
    ConicPlusP q;
    if (!table_host || (np > 0 && !p) || make_conicplus(q, R, K, p, np, opd != 0, opd != 0 ? nr : 0.) < 0) {
        set_error("pxf_conicplus_table_fill: need 0..%d polynomial terms", PXF_CONICPLUS_MAXP);
        return -1;
    }
    memcpy(table_host, &q, sizeof(q));
    return (int32_t)sizeof(q);
}

extern "C" size_t pxf_legsurf_table_bytes(void) { return sizeof(LegSurfP); }

extern "C" int32_t pxf_legsurf_table_fill(double xwidth, double ywidth, double order, const double *coeff,
                                          const int32_t *xo, const int32_t *yo, int32_t nc, void *table_host)
{
    LegSurfP q;
    if (!table_host || !coeff || !xo || !yo || make_legsurf(q, xwidth, ywidth, order, coeff, xo, yo, nc) < 0) {
        set_error("pxf_legsurf_table_fill: need 0..%d terms with orders 0..%d", PXF_LEGSURF_MAXC, PXF_LEGSURF_MAXN);
        return -1;
    }
    memcpy(table_host, &q, sizeof(q));
    return (int32_t)sizeof(q);
}

// ---- segmented programs -------------------------------------------------------------------------
static size_t seg_align(size_t v) { return (v + 15) & ~(size_t)15; }
static size_t seg_ops_offset(int nseg) { return seg_align(sizeof(SegHeader)) + seg_align((size_t)(nseg + 1) * 8); }

extern "C" size_t pxf_segmented_table_bytes(int32_t nops, int32_t nseg)
{
    if (nops < 1 || nseg < 1) return 0;
    size_t packs = seg_chain_bytes(nseg), jp = (size_t)nseg * jit_seg_pack_bytes(nops);
    return seg_align(seg_ops_offset(nseg) + (size_t)nseg * nops * sizeof(FusedOp)) + (packs > jp ? packs : jp);
}
static size_t seg_chain_offset(int nops, int nseg) { return seg_align(seg_ops_offset(nseg) + (size_t)nseg * nops * sizeof(FusedOp)); }

static bool is_vignette(int code)
{
    return code == PXF_OP_VIGNETTE_MAG || code == PXF_OP_VIGNETTE_BOX || code == PXF_OP_VIGNETTE_ABS ||
           code == PXF_OP_VIGNETTE_RHOGT;
}

// Zernike tables of a segmented program: behind everything pxf_segmented_table_bytes lays out, one per segment
static size_t seg_zern_offset(int nops, int nseg) { return seg_align(pxf_segmented_table_bytes(nops, nseg)); }

extern "C" size_t pxf_segmented_table_bytes_zern(int32_t nops, int32_t nseg)
{
    if (nops < 1 || nseg < 1) return 0;
    return seg_zern_offset(nops, nseg) + (size_t)nseg * sizeof(ZernP);
}

// LL tables of a segmented program: at the same place, room for PXF_PROG_MAX_LL per segment
extern "C" size_t pxf_segmented_table_bytes_ll(int32_t nops, int32_t nseg)
{
    if (nops < 1 || nseg < 1) return 0;
    return seg_zern_offset(nops, nseg) + (size_t)nseg * PXF_PROG_MAX_LL * sizeof(LLTab);
}

// Which per-segment tables a fill takes: none, one Zernike table, or one LL table per PXF_OP_LLSURF op
enum SegTables { SEG_PLAIN, SEG_ZERN, SEG_LL };

// tables: nseg tables of pxf_zern_table_fill (SEG_ZERN), nseg * nll tables of pxf_ll_table_fill (SEG_LL), segment-major;
// NULL: the program may not have such an op
static int seg_table_fill(const pxf_op *ops, int nops, int nseg, const int64_t *seg_start, const void *tables,
                          SegTables kind, void *table_host)
{
    const bool zern_ok = kind == SEG_ZERN, ll_ok = kind == SEG_LL;
    const void *zern_tables = zern_ok ? tables : nullptr;
    if (!ops || !seg_start || !table_host || nops < 1 || nops > PXF_MAX_OPS || nseg < 1) {
        set_error("pxf_segmented_table_fill: bad argument");
        return PXF_ERR_INVALID;
    }
    if (seg_start[0] != 0) { set_error("segmented program: seg_start[0] must be 0"); return PXF_ERR_INVALID; }
    for (int sgm = 0; sgm < nseg; sgm++)
        if (seg_start[sgm + 1] < seg_start[sgm]) { set_error("segmented program: seg_start must be non-decreasing"); return PXF_ERR_INVALID; }
    bool zern = false;
    if (zern_ok || ll_ok) {
        for (size_t k = 0; k < (size_t)nseg * nops; k++) {
            if (ops[k].code == PXF_OP_GRATFAN || ops[k].code == PXF_OP_ROTX_REMAINING) {
                set_error("segmented program: PXF_OP_GRATFAN / PXF_OP_ROTX_REMAINING are not supported");
                return PXF_ERR_UNSUPPORTED;
            }
            if ((ops[k].code == PXF_OP_ZERNSURF || ops[k].code == PXF_OP_ZERNPHASE) && zern_ok) zern = true;
        }
        if (zern && !zern_tables) { set_error("segmented program: PXF_OP_ZERNSURF / ZERNPHASE need one Zernike table per segment"); return PXF_ERR_INVALID; }
    }
    // LL ops: their positions in segment 0's list (the others must match, checked with the opcode sequence below)
    int llpos[PXF_PROG_MAX_LL], nll = 0;
    bool surf = false;
    for (size_t k = 0; k < (size_t)nseg * nops; k++) {
        if (ops[k].code == PXF_OP_LLSURF && !ll_ok) {
            set_error("segmented program: PXF_OP_LLSURF needs pxf_segmented_table_fill_ll");
            return PXF_ERR_UNSUPPORTED;
        }
        if (is_surface_op(ops[k].code)) {
            if (zern_ok || ll_ok) {
                set_error("segmented program: the sphere / cylinder / cylconic / paraxial / torus / W-S back-surface / "
                          "conicplus / legsurf ops need pxf_segmented_table_fill");
                return PXF_ERR_UNSUPPORTED;
            }
            surf = true;
        }
    }
    for (int k = 0; k < nops; k++)
        if (ops[k].code == PXF_OP_LLSURF) {
            if (nll == PXF_PROG_MAX_LL) { set_error("program: at most %d PXF_OP_LLSURF ops per program", PXF_PROG_MAX_LL); return PXF_ERR_UNSUPPORTED; }
            llpos[nll++] = k;
        }
    if (nll && !tables) { set_error("segmented program: PXF_OP_LLSURF needs one LL table per op and segment"); return PXF_ERR_INVALID; }
    char *base = static_cast<char *>(table_host);
    SegHeader *h = reinterpret_cast<SegHeader *>(base);
    memset(h, 0, seg_align(sizeof(SegHeader)));
    memcpy(base + seg_align(sizeof(SegHeader)), seg_start, (size_t)(nseg + 1) * 8);
    FusedOp *dst = reinterpret_cast<FusedOp *>(base + seg_ops_offset(nseg));
    ZernP *zdst = zern ? reinterpret_cast<ZernP *>(base + seg_zern_offset(nops, nseg)) : nullptr;
    LLTab *ldst = nll ? reinterpret_cast<LLTab *>(base + seg_zern_offset(nops, nseg)) : nullptr;
    h->nops = nops; h->nseg = nseg; h->surf = surf ? 1 : 0;
    // the segment's own LL tables, copied into this one; every segment evaluates position j at the largest order
    // any segment has there (the zero padding makes that the same bits)
    int lln[PXF_PROG_MAX_LL] = {0, 0};
    if (nll) {
        memcpy(ldst, tables, (size_t)nseg * nll * sizeof(LLTab));
        for (size_t t = 0; t < (size_t)nseg * nll; t++) {
            const LLS &ls = ldst[t].s;
            const int top = ls.nz > ls.nt ? ls.nz : ls.nt;
            if (ls.kind < 0 || ls.kind > 2 || ls.nz < 0 || ls.nt < 0 || top > PXF_LL_PROG_MAXN) {
                set_error("segmented program: segment %d: PXF_OP_LLSURF supports Legendre orders <= %d (table has %d)",
                          (int)(t / nll), PXF_LL_PROG_MAXN, top);
                return PXF_ERR_UNSUPPORTED;
            }
            if (top > lln[t % nll]) lln[t % nll] = top;
        }
    }
    for (int sgm = 0; sgm < nseg; sgm++) {
        pxf_op sops[PXF_MAX_OPS];
        memcpy(sops, ops + (size_t)sgm * nops, (size_t)nops * sizeof(pxf_op));
        if (zern) {
            // the segment's own table, copied into this one (the op's device address p[0] is not used)
            memcpy(zdst + sgm, static_cast<const char *>(zern_tables) + (size_t)sgm * sizeof(ZernP), sizeof(ZernP));
            const int nmax = zdst[sgm].nmax;
            if (nmax < 0 || nmax > 7) {
                set_error("segmented program: segment %d: PXF_OP_ZERNSURF / ZERNPHASE support radial orders <= 7 (table has %d)", sgm, nmax);
                return PXF_ERR_UNSUPPORTED;
            }
            for (int k = 0; k < nops; k++)
                if (sops[k].code == PXF_OP_ZERNSURF || sops[k].code == PXF_OP_ZERNPHASE) {
                    const ZernP *any = zdst + sgm;       // build_program only checks that a table is there
                    memcpy(&sops[k].p[0], &any, sizeof(any));
                    sops[k].p[2] = (double)nmax;
                }
        }
        for (int j = 0; j < nll; j++)
            if (sops[llpos[j]].code == PXF_OP_LLSURF) {
                const LLTab *any = ldst + (size_t)sgm * nll + j;
                memcpy(&sops[llpos[j]].p[0], &any, sizeof(any));
                sops[llpos[j]].p[1] = (double)lln[j];
            }
        FusedProgram fp;
        int rc = build_program(fp, sops, nops);
        if (rc) return rc;
        if ((fp.zern && !zern_ok) || fp.uses_aux) {
            set_error("segmented program: PXF_OP_ZERNSURF / ZERNPHASE need pxf_segmented_table_fill_zern; PXF_OP_GRATFAN is "
                      "not supported");
            return PXF_ERR_UNSUPPORTED;
        }
        if (sgm > 0)
            for (int k = 0; k < nops; k++)
                if (fp.ops[k].code != dst[k].code || fp.ops[k].row != dst[k].row) {   // dst[0..nops) = segment 0
                    set_error("segmented program: every segment must run the same opcode sequence (segment %d, op %d)", sgm, k);
                    return PXF_ERR_INVALID;
                }
        h->load_mask |= fp.load_mask;
        h->store_mask |= fp.store_mask;
        memcpy(dst + (size_t)sgm * nops, fp.ops, (size_t)nops * sizeof(FusedOp));
    }
    if (zern) h->zern_off = (long long)seg_zern_offset(nops, nseg);
    if (nll) { h->ll_off = (long long)seg_zern_offset(nops, nseg); h->nll = nll; }
    // a statically specialised kernel for the canonical chains: one parameter pack per segment behind the op table
    h->chain_id = seg_chain_fill(dst, nops, nseg, base + seg_chain_offset(nops, nseg));
    bool vig = false;
    for (int k = 0; k < nops; k++)
        if (is_vignette(dst[k].code)) vig = true;
    if (h->chain_id == 0 || vig) {
        // any other op list: parameter packs for a kernel specialised at run time (pxf_jit.cu)
        const size_t pb = jit_seg_fill(dst, nops, nseg, base + seg_chain_offset(nops, nseg));
        if (pb) { h->chain_id = 2; h->jit_pack_bytes = (int)pb; }
        else if (vig) h->chain_id = 0;
    }
    return PXF_OK;
}

extern "C" int pxf_segmented_table_fill(const pxf_op *ops, int32_t nops, int32_t nseg, const int64_t *seg_start,
                                        void *table_host)
{
    return seg_table_fill(ops, nops, nseg, seg_start, nullptr, SEG_PLAIN, table_host);
}

extern "C" int pxf_segmented_table_fill_zern(const pxf_op *ops, int32_t nops, int32_t nseg, const int64_t *seg_start,
                                             const void *zern_tables_host, void *table_host)
{
    return seg_table_fill(ops, nops, nseg, seg_start, zern_tables_host, SEG_ZERN, table_host);
}

extern "C" int pxf_segmented_table_fill_ll(const pxf_op *ops, int32_t nops, int32_t nseg, const int64_t *seg_start,
                                           const void *ll_tables_host, void *table_host)
{
    return seg_table_fill(ops, nops, nseg, seg_start, ll_tables_host, SEG_LL, table_host);
}

extern "C" int pxf_trace_program_segmented(double *const rays_in[10], double *const rays_out[10], int64_t num,
                                           const void *table_host, const void *table_dev, uint8_t *alive,
                                           pxf_stream_t stream)
{
    if (!rays_in || !table_host || !table_dev || num < 0) { set_error("pxf_trace_program_segmented: bad argument"); return PXF_ERR_INVALID; }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    const SegHeader *h = static_cast<const SegHeader *>(table_host);
    const int nops = h->nops, nseg = h->nseg;
    const int64_t *hs = reinterpret_cast<const int64_t *>(static_cast<const char *>(table_host) + seg_align(sizeof(SegHeader)));
    if (nops < 1 || nops > PXF_MAX_OPS || nseg < 1 || hs[nseg] != num) {
        set_error("segmented program: table does not describe a bundle of %lld rays", (long long)num);
        return PXF_ERR_INVALID;
    }
    if (num == 0) return PXF_OK;
    unsigned LM = h->load_mask, SM = h->store_mask;
    if (rays_out) SM |= LM;
    RowPtrs P, Q;
    for (int k = 0; k < 10; k++) {
        P.p[k] = rays_in[k];
        Q.p[k] = rays_out ? rays_out[k] : rays_in[k];
        if ((LM & (1u << k)) && !P.p[k]) { set_error("segmented program: null input row pointer (row %d)", k); return PXF_ERR_INVALID; }
        if ((SM & (1u << k)) && !Q.p[k]) { set_error("segmented program: null output row pointer (row %d)", k); return PXF_ERR_INVALID; }
    }
    const FusedOp *hops = reinterpret_cast<const FusedOp *>(static_cast<const char *>(table_host) + seg_ops_offset(nseg));
    bool vig = false, zph, tab;
    for (int k = 0; k < nops; k++)
        if (is_vignette(hops[k].code)) vig = true;
    new_table_kinds(hops, nops, zph, tab);
    if (vig && !alive) { set_error("program with a VIGNETTE op needs an alive array"); return PXF_ERR_INVALID; }
    const char *db = static_cast<const char *>(table_dev);
    const long long *dstart = reinterpret_cast<const long long *>(db + seg_align(sizeof(SegHeader)));
    const FusedOp *dops = reinterpret_cast<const FusedOp *>(db + seg_ops_offset(nseg));
    const ZernP *dzern = h->zern_off ? reinterpret_cast<const ZernP *>(db + h->zern_off) : nullptr;
    const LLTab *dll = h->ll_off ? reinterpret_cast<const LLTab *>(db + h->ll_off) : nullptr;
    const int nll = dll ? h->nll : 0;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (h->chain_id == 1 && !vig) {
        int rc = seg_chain_launch(h->chain_id, P, Q, num, alive, dstart, db + seg_chain_offset(nops, nseg), nseg, LM, SM, s);
        if (rc != PXF_ERR_UNSUPPORTED) return rc;
    }
    if (h->chain_id == 2) {
        int rc = jit_seg_launch(hops, nops, P, Q, num, alive, dstart, db + seg_chain_offset(nops, nseg), nseg, LM, SM,
                                dzern, dll, s);
        if (rc != PXF_ERR_UNSUPPORTED) return rc;
    }
    auto go = [&](auto kern, size_t smem) {
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, PXF_BLOCK, smem) != cudaSuccess || nb <= 0) { cudaGetLastError(); nb = 2; }
        const int grid = grid_for(num, SEG_TILE, nb);
        kern<<<grid, PXF_BLOCK, smem, s>>>(P, Q, num, alive, dstart, dops, nops, nseg, LM, SM, dzern, dll, nll);
    };
    if (dzern && zph) {
        // the segment's Zernike table is staged behind its op table; register cap as for k_program<zphase>
        go(k_program_seg<ZPHASE_MINB, false, false, false, false, true>, (size_t)seg_zern_smem_offset(nops) + sizeof(ZernP));
        count_launch();
        note_kernel("k_program_seg<zphase> (interpreter)");
        return check_launch("k_program_seg<zphase>");
    }
    if (dzern) {
        // the segment's Zernike table is staged behind its op table; register cap as for k_program<zernike>
        go(k_program_seg<ZERN_MINB, true>, (size_t)seg_zern_smem_offset(nops) + sizeof(ZernP));
        count_launch();
        note_kernel("k_program_seg<zernike> (interpreter)");
        return check_launch("k_program_seg<zernike>");
    }
    if (dll) {
        // the segment's LL tables are staged behind its op table; register cap as for k_program<ll>
        go(k_program_seg<LL_MINB, false, true>, (size_t)seg_zern_smem_offset(nops) + (size_t)nll * sizeof(LLTab));
        count_launch();
        note_kernel("k_program_seg<ll> (interpreter)");
        return check_launch("k_program_seg<ll>");
    }
    if (tab) {
        go(k_program_seg<TABSURF_MINB, false, false, true, true>, (size_t)nops * sizeof(FusedOp));
        count_launch();
        note_kernel("k_program_seg<tabsurf> (interpreter)");
        return check_launch("k_program_seg<tabsurf>");
    }
    if (has_array_ops(hops, nops)) {
        // the plain interpreter's ops and the gratings with per-ray arrays; register cap as for k_program_seg
        go(k_program_seg<4, false, false, false, false, false, true>, (size_t)nops * sizeof(FusedOp));
        count_launch();
        note_kernel("k_program_seg<grat> (interpreter)");
        return check_launch("k_program_seg<grat>");
    }
    if (h->surf) {
        go(k_program_seg<SURF_MINB, false, false, true>, (size_t)nops * sizeof(FusedOp));
        count_launch();
        note_kernel("k_program_seg<surf> (interpreter)");
        return check_launch("k_program_seg<surf>");
    }
    go(k_program_seg<4>, (size_t)nops * sizeof(FusedOp));
    count_launch();
    note_kernel("k_program_seg (interpreter)");
    return check_launch("k_program_seg");
}

extern "C" int pxf_trace_program_sums(double *const rays_in[10], double *const rays_out[10], int64_t num,
                                      const pxf_op *ops, int32_t nops, uint8_t *alive, double *sums_dev,
                                      void *scratch, pxf_stream_t stream)
{
    if (!sums_dev || !scratch) { set_error("pxf_trace_program_sums: null sums/scratch"); return PXF_ERR_INVALID; }
    FusedProgram fp;
    int rc = build_program(fp, ops, nops);
    if (rc) return rc;
    if (rays_out) fp.store_mask |= fp.load_mask;
    // the sums need the final x,y in registers: make sure they are loaded even if the program
    // itself never reads them
    fp.load_mask |= (R_X | R_Y) & ~fp.store_mask;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (num == 0) {
        PXF_CUDA(cudaMemsetAsync(sums_dev, 0, 4 * sizeof(double), s));
        return PXF_OK;
    }
    int grid = 0;
    rc = launch_program(rays_in, num, fp, alive, s, rays_out, static_cast<double *>(scratch), &grid);
    if (rc) return rc;
    return sums_finalize(static_cast<const double *>(scratch), grid, 4, sums_dev, s);
}
