// Per-routine kernels: one launch per f2py routine, one pass over the rows it touches.
// HBM-bound streaming kernels (SURVEY 8a "B/ray"): rows are read and written with double2
// accesses (two rays per thread) when every row is 16-byte aligned, by a persistent grid
// of SM-count x resident-CTA blocks striding over ray pairs.
#include <stdarg.h>
#include <atomic>
#include <type_traits>
#include "pxf_internal.h"
#include "pxf_params.h"

namespace pxf {

// ------------------------------------------------------------------ library state
static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};
static int g_sms = 0;

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
static std::atomic<int> g_ws_libm{0};
static std::atomic<int> g_ws_retrace{PXF_WS_RETRACE_DEFAULT};
int opt_ws_libm() { return g_ws_libm.load(std::memory_order_relaxed); }
int opt_ws_retrace() { return g_ws_retrace.load(std::memory_order_relaxed); }
static std::atomic<int> g_ws_graze_ppm{PXF_WS_GRAZE_PPM_DEFAULT};
int opt_ws_graze_ppm() { return g_ws_graze_ppm.load(std::memory_order_relaxed); }
int sm_count()
{
    if (g_sms == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
            cudaGetLastError();
            return 0;
        }
        g_sms = n;
    }
    return g_sms;
}
int grid_for(int64_t work_items, int per_block, int ctas_per_sm)
{
    int64_t need = (work_items + per_block - 1) / per_block;
    int64_t cap = (int64_t)sm_count() * ctas_per_sm;
    if (cap <= 0) cap = 1;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}
int Scratch::alloc(size_t bytes, cudaStream_t stream)
{
    s = stream;
    // The default pool gives its memory back to the driver at every synchronisation (release threshold 0), so
    // each convenience call would re-map its scratch: measured 3-30 ms per analysis call at 1e7 rays.  Keep it.
    static bool pooled[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64 && !pooled[dev]) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
        pooled[dev] = true;
    }
    cudaError_t e = cudaMallocAsync(&p, bytes ? bytes : 8, stream);
    if (e != cudaSuccess) {
        p = nullptr;
        set_error("cudaMallocAsync(%zu): %s", bytes, cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? PXF_ERR_NOMEM : PXF_ERR_CUDA;
    }
    return PXF_OK;
}
Scratch::~Scratch()
{
    if (p) cudaFreeAsync(p, s);
}

// ------------------------------------------------------------------ row access
struct RowPtrs { double *p[10]; };

template <unsigned M>
PXF_DEV void load1(Ray &r, const RowPtrs &P, int64_t i)
{
    if (M & R_OPD) r.opd = P.p[0][i];
    if (M & R_X) r.x = P.p[1][i];
    if (M & R_Y) r.y = P.p[2][i];
    if (M & R_Z) r.z = P.p[3][i];
    if (M & R_L) r.l = P.p[4][i];
    if (M & R_M) r.m = P.p[5][i];
    if (M & R_N) r.n = P.p[6][i];
    if (M & R_UX) r.ux = P.p[7][i];
    if (M & R_UY) r.uy = P.p[8][i];
    if (M & R_UZ) r.uz = P.p[9][i];
}
template <unsigned M>
PXF_DEV void store1(const Ray &r, const RowPtrs &P, int64_t i)
{
    if (M & R_OPD) P.p[0][i] = r.opd;
    if (M & R_X) P.p[1][i] = r.x;
    if (M & R_Y) P.p[2][i] = r.y;
    if (M & R_Z) P.p[3][i] = r.z;
    if (M & R_L) P.p[4][i] = r.l;
    if (M & R_M) P.p[5][i] = r.m;
    if (M & R_N) P.p[6][i] = r.n;
    if (M & R_UX) P.p[7][i] = r.ux;
    if (M & R_UY) P.p[8][i] = r.uy;
    if (M & R_UZ) P.p[9][i] = r.uz;
}
#define PXF_LD2(bit, k, f)                                                          \
    if (M & bit) {                                                                  \
        double2 v = *reinterpret_cast<const double2 *>(P.p[k] + i);                 \
        a.f = v.x; b.f = v.y;                                                       \
    }
#define PXF_ST2(bit, k, f)                                                          \
    if (M & bit) *reinterpret_cast<double2 *>(P.p[k] + i) = make_double2(a.f, b.f);
template <unsigned M>
PXF_DEV void load2(Ray &a, Ray &b, const RowPtrs &P, int64_t i)
{
    PXF_LD2(R_OPD, 0, opd) PXF_LD2(R_X, 1, x) PXF_LD2(R_Y, 2, y) PXF_LD2(R_Z, 3, z) PXF_LD2(R_L, 4, l)
    PXF_LD2(R_M, 5, m) PXF_LD2(R_N, 6, n) PXF_LD2(R_UX, 7, ux) PXF_LD2(R_UY, 8, uy) PXF_LD2(R_UZ, 9, uz)
}
template <unsigned M>
PXF_DEV void store2(const Ray &a, const Ray &b, const RowPtrs &P, int64_t i)
{
    PXF_ST2(R_OPD, 0, opd) PXF_ST2(R_X, 1, x) PXF_ST2(R_Y, 2, y) PXF_ST2(R_Z, 3, z) PXF_ST2(R_L, 4, l)
    PXF_ST2(R_M, 5, m) PXF_ST2(R_N, 6, n) PXF_ST2(R_UX, 7, ux) PXF_ST2(R_UY, 8, uy) PXF_ST2(R_UZ, 9, uz)
}

// ------------------------------------------------------------------ op functors
// LOAD: rows the loop body reads; STORE: rows it may write.  Rows that are written only
// conditionally are also in LOAD so that the unconditional row store is a no-op for them.
struct NoParams { int unused; };

struct OpTransform {
    using Params = TransformP;
    static constexpr unsigned LOAD = R_NINE, STORE = R_NINE;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_transform(r, p); }
};
struct OpITransform {
    using Params = TransformP;
    static constexpr unsigned LOAD = R_NINE, STORE = R_NINE;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_itransform(r, p); }
};
struct OpReflect {
    using Params = NoParams;
    static constexpr unsigned LOAD = R_DIR | R_NRM, STORE = R_DIR;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &, const double *, double, double) { op_reflect(r); }
};
// one ray per thread, 4 CTAs/SM (measured: 1.408 / 1.283 / 1.229 / 1.300 / 1.408 ms; shapes as listed at OpMinB)
struct OpRefract {
    static constexpr int MINB = 4;
    static constexpr bool SCALAR = true;
    using Params = RefractP;
    static constexpr unsigned LOAD = R_DIR | R_NRM, STORE = R_DIR | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_refract(r, p); }
};
struct OpRadgrat {
    using Params = RadgratP;
    static constexpr unsigned LOAD = R_X | R_Y | R_DIR, STORE = R_DIR;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double)
    {
        op_radgrat(r, p, p.wave, false);
    }
};
struct OpRadgratW {
    using Params = RadgratP;
    static constexpr unsigned LOAD = R_X | R_Y | R_DIR, STORE = R_DIR;
    static constexpr int AUX = 1, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double wave, double)
    {
        op_radgrat(r, p, wave, true);
    }
};
struct GratP { double d; };
struct OpGrat {
    using Params = GratP;
    static constexpr unsigned LOAD = R_DIR, STORE = R_DIR;
    static constexpr int AUX = 2, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double order, double wave)
    {
        op_grat(r, p.d, order, wave);
    }
};
// transformations.pointTo (transformations.py:91-100): direction cosines toward (reverse=-1) or away from a point
struct PointToP { double x0, y0, z0, reverse; };
struct OpPointTo {
    using Params = PointToP;
    static constexpr unsigned LOAD = R_POS, STORE = R_DIR;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double)
    {
        const double dx = r.x - p.x0, dy = r.y - p.y0, dz = r.z - p.z0;
        const double R = sqrt(dx * dx + dy * dy + dz * dz);
        r.l = p.reverse * dx / R;
        r.m = p.reverse * dy / R;
        r.n = p.reverse * dz / R;
    }
};
// transformations.applyT (transformations.py:257-280): positions through the 4x4 point matrix, direction cosines and
// normals through the 4x4 rotation matrix (the homogeneous coordinate is 1 for all three, as in the reference)
struct ApplyTP { double P[12], R[12]; };
struct OpApplyT {
    using Params = ApplyTP;
    static constexpr unsigned LOAD = R_NINE, STORE = R_NINE;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void mul(const double *M, double &a, double &b, double &c)
    {
        const double u = M[0] * a + M[1] * b + M[2] * c + M[3];
        const double v = M[4] * a + M[5] * b + M[6] * c + M[7];
        const double w = M[8] * a + M[9] * b + M[10] * c + M[11];
        a = u; b = v; c = w;
    }
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double)
    {
        mul(p.P, r.x, r.y, r.z);
        mul(p.R, r.l, r.m, r.n);
        mul(p.R, r.ux, r.uy, r.uz);
    }
};
// analyses.indAngle (analyses.py:164-182): arccos(l*ux + m*uy + n*uz), or arccos(normal . (l,m,n)) for a fixed
// normal; the angle is written to the row passed in the opd slot
struct IndAngleP { double nx, ny, nz; int fixed; };
struct OpIndAngle {
    using Params = IndAngleP;
    static constexpr unsigned LOAD = R_DIR | R_NRM, STORE = R_OPD;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double)
    {
        const double d = p.fixed ? p.nx * r.l + p.ny * r.m + p.nz * r.n : r.l * r.ux + r.m * r.uy + r.n * r.uz;
        r.opd = acos(d);
    }
};
// analyses.measureOPD (analyses.py:232-244): distance of every ray from a point, written to the row in the opd slot
struct OpDistance {
    using Params = PointToP;
    static constexpr unsigned LOAD = R_POS, STORE = R_OPD;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double)
    {
        const double dx = r.x - p.x0, dy = r.y - p.y0, dz = r.z - p.z0;
        r.opd = sqrt(dx * dx + dy * dy + dz * dz);
    }
};
struct OpIndAngleFixed {
    using Params = IndAngleP;
    static constexpr unsigned LOAD = R_DIR, STORE = R_OPD;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double)
    {
        r.opd = acos(p.nx * r.l + p.ny * r.m + p.nz * r.n);
    }
};
struct FlatP { double nr; };
struct OpFlat {
    using Params = FlatP;
    static constexpr unsigned LOAD = R_POS | R_DIR, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &, const double *, double, double) { op_flat(r, false, 0.); }
};
struct OpFlatOpd {
    using Params = FlatP;
    static constexpr unsigned LOAD = R_POS | R_DIR | R_OPD, STORE = R_POS | R_NRM | R_OPD;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_flat(r, true, p.nr); }
};
struct OpConic {
    using Params = ConicP;
    static constexpr unsigned LOAD = R_NINE, STORE = R_NINE;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_conic(r, p); }
};
struct OpConicOpd {
    using Params = ConicP;
    static constexpr unsigned LOAD = R_ALL, STORE = R_ALL;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_conic(r, p); }
};
struct OpWolterPrimary {
    using Params = WolterP;
    static constexpr unsigned LOAD = R_POS | R_DIR, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_wolterprimary(r, p); }
};
struct OpWolterPrimaryOpd {
    using Params = WolterP;
    static constexpr unsigned LOAD = R_POS | R_DIR | R_OPD, STORE = R_POS | R_NRM | R_OPD;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_wolterprimary(r, p); }
};
// one ray per thread, 5 CTAs/SM (measured: 0.893 / 0.900 / 0.900 / 0.865 / 0.897 ms; shapes as listed at OpMinB)
struct OpWolterSecondary {
    static constexpr int MINB = 5;
    static constexpr bool SCALAR = true;
    using Params = WolterP;
    static constexpr unsigned LOAD = R_POS | R_DIR, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_woltersecondary(r, p); }
};
struct OpWolterSine {
    using Params = WolterSineP;
    static constexpr unsigned LOAD = R_POS | R_DIR, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_woltersine(r, p); }
};
// One ray per thread, 3 CTAs/SM: the W-S Newton loops are latency bound at two rays per thread and 140 registers
// (8 warps per SM, fp64 pipe 30 %: profiles/r02d_k_op_wsprimary.txt).  Measured at 5e7 rays, primary / secondary: two
// rays per thread uncapped 2.60 / 5.70 ms, capped for 2 CTAs/SM 1.68 / 3.59 ms; one ray per thread capped for 3 / 4 / 2
// CTAs/SM 1.51 / 3.21, 1.76 / 3.21, 1.76 / 3.58 ms
struct OpWsPrimary {
    static constexpr int MINB = 3;
    static constexpr bool SCALAR = true;
    using Params = WSP;
    static constexpr unsigned LOAD = R_NINE, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_wsprimary(r, p); }
};
struct OpWsSecondary {
    static constexpr int MINB = 3;
    static constexpr bool SCALAR = true;
    using Params = WSP;
    static constexpr unsigned LOAD = R_NINE, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_wssecondary(r, p); }
};
struct OpWsPrimaryBack {
    using Params = WSP;
    static constexpr unsigned LOAD = R_NINE, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_wsprimary_t<true>(r, p); }
};
struct OpWsSecondaryBack {
    using Params = WSP;
    static constexpr unsigned LOAD = R_NINE, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_wssecondary_t<true>(r, p); }
};
template <bool OPD>
struct OpSphere {
    using Params = SphereP;
    static constexpr unsigned LOAD = R_POS | R_DIR | (OPD ? R_OPD : 0u), STORE = R_NINE | (OPD ? R_OPD : 0u);
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_tracesphere(r, p); }
};
template <bool OPD>
struct OpCyl {
    using Params = SphereP;
    static constexpr unsigned LOAD = R_POS | R_DIR | (OPD ? R_OPD : 0u), STORE = R_NINE | (OPD ? R_OPD : 0u);
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_tracecyl(r, p); }
};
struct OpCylConic {
    using Params = CylConicP;
    static constexpr unsigned LOAD = R_POS | R_DIR, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_cylconic(r, p); }
};
struct OpParaxial {
    using Params = ParaxialP;
    static constexpr unsigned LOAD = R_X | R_Y | R_L | R_M, STORE = R_L | R_M;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_paraxial(r, p); }
};
struct OpTorus {
    using Params = TorusP;
    static constexpr unsigned LOAD = R_POS | R_DIR, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_torus(r, p); }
};
template <bool OPD>
struct OpConicPlus {
    using Params = ConicPlusP;
    static constexpr unsigned LOAD = R_POS | R_DIR | (OPD ? R_OPD : 0u), STORE = R_POS | R_NRM | (OPD ? R_OPD : 0u);
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_conicplus(r, p); }
};
struct OpLegSurf {
    using Params = LegSurfP;
    static constexpr unsigned LOAD = R_X | R_Y | R_DIR, STORE = R_DIR;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_legsurf(r, p); }
};
// one ray per thread, 3 CTAs/SM (measured: 1.199 / 1.001 / 1.049 / 1.137 / 1.215 ms; shapes as listed at OpMinB)
struct OpSpoCone {
    static constexpr int MINB = 3;
    static constexpr bool SCALAR = true;
    using Params = SpoP;
    static constexpr unsigned LOAD = R_NINE, STORE = R_NINE;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_spocone(r, p); }
};
// nmax <= 7: one ray per thread even on aligned rows, 4 CTAs/SM (the unrolled Zernike evaluation needs ~200 registers
// per ray: two rays per thread leave 8 warps per SM to cover the fp64 latency).  The Cartesian Horner form needs far
// fewer live values than the polar one; measured, 36 terms at 5e7 rays: two rays per thread uncapped 1.81 ms, capped
// for 2 CTAs/SM 1.35 ms; one ray per thread capped for 3 / 4 / 2 CTAs/SM 1.46 / 1.35 / 1.50 ms (profiles/r02_notes.md).
// Higher orders: two rays per thread, uncapped (measured, profiles/r01h_notes.md: two rays per thread at ~240
// registers = 8 warps/SM runs 3.69 ms per 5e7 rays; one ray per thread capped for 1/2/3 CTAs per SM 4.12/3.99/4.03
// ms -- the evaluation is issue bound)
template <int NMAX, bool OPD>
struct OpZern {
    static constexpr int MINB = NMAX <= 7 ? 4 : 1;
    static constexpr bool SCALAR = NMAX <= 7;
    using Params = ZernP;
    static constexpr unsigned LOAD = R_POS | R_DIR | (OPD ? R_OPD : 0u);
    static constexpr unsigned STORE = R_POS | R_NRM | (OPD ? R_OPD : 0u);
    static constexpr int AUX = 0, SMEM = PXF_ZERN_SMEM_DOUBLES;
    PXF_DEV static const double *table(const Params &p) { return reinterpret_cast<const double *>(p.e); }
    PXF_DEV static void apply(Ray &r, const Params &p, const double *smem, double, double)
    {
        op_tracezern<NMAX>(r, p.rad, p.nr, p.tol, p.nmax, OPD ? 1 : 0, smem);
    }
};

struct ZernPhaseP { ZernP z; double wave; };
template <int NMAX>
struct OpZernPhase {
    using Params = ZernPhaseP;
    static constexpr unsigned LOAD = R_X | R_Y | R_DIR | R_OPD, STORE = R_DIR | R_OPD;
    static constexpr int AUX = 0, SMEM = PXF_ZERN_SMEM_DOUBLES;
    PXF_DEV static const double *table(const Params &p) { return reinterpret_cast<const double *>(p.z.e); }
    PXF_DEV static void apply(Ray &r, const Params &p, const double *smem, double, double)
    {
        op_zernphase<NMAX>(r, p.z.rad, p.wave, p.z.nmax, smem);
    }
};

// N = 5: one ray per thread, 4 CTAs/SM; the other orders: two rays per thread, 2 CTAs/SM.  Measured at N = 5, 36 terms
// at 5e7 rays: two rays per thread capped for 2 CTAs/SM 2.68 ms; one ray per thread capped for 3 / 4 CTAs/SM 2.58 /
// 2.55 ms; two rays per thread uncapped 3.74 ms
template <int N>
struct OpLL {
    static constexpr int MINB = N == 5 ? 4 : 2;
    static constexpr bool SCALAR = N == 5;
    using Params = LLP;
    static constexpr unsigned LOAD = R_POS | R_DIR, STORE = R_POS | R_NRM;
    static constexpr int AUX = 0, SMEM = 0;
    PXF_DEV static const double *table(const Params &p) { return p.C; }
    // the coefficient matrix is read straight from the kernel parameter (constant bank, static offsets)
    PXF_DEV static void apply(Ray &r, const Params &p, const double *, double, double) { op_ll<N>(r, p.s, p.C); }
};

// ------------------------------------------------------------------ the kernel
// Launch shape of a routine.  MINB: resident CTAs per SM the register allocation is capped for (default 1, uncapped);
// SCALAR: one ray per thread even on aligned rows (default: two rays per thread with double2 accesses).  The
// compute-bound routines were timed at 5e7 rays in five shapes, listed as "measured:" in this order: two rays per
// thread uncapped / one ray per thread capped for 3 / 4 / 5 CTAs per SM / two rays per thread capped for 2 CTAs per
// SM (profiles/r02l_op_variants.txt).  Where the fastest shape wins by less than 1 %, the routine keeps the default.
template <class Op, class = void> struct OpMinB { static constexpr int v = 1; };
template <class Op> struct OpMinB<Op, std::void_t<decltype(Op::MINB)>> { static constexpr int v = Op::MINB; };
template <class Op, class = void> struct OpScalar { static constexpr bool v = false; };
template <class Op> struct OpScalar<Op, std::void_t<decltype(Op::SCALAR)>> { static constexpr bool v = Op::SCALAR; };

template <class Op, bool MASKED, bool VEC2>
__global__ void __launch_bounds__(PXF_BLOCK, OpMinB<Op>::v)
k_op(const RowPtrs P, const int64_t num, const uint8_t *__restrict__ mask,
     const double *__restrict__ aux0, const double *__restrict__ aux1,
     const __grid_constant__ typename Op::Params prm)
{
    constexpr unsigned LD = MASKED ? (Op::LOAD | Op::STORE) : Op::LOAD;
    constexpr unsigned ST = Op::STORE;
    __shared__ double smem[Op::SMEM > 0 ? Op::SMEM : 1];
    if constexpr (Op::SMEM > 0) {
        // stage the coefficient table (Zernike) once per CTA
        const double *src = Op::table(prm);
        for (int t = threadIdx.x; t < Op::SMEM; t += blockDim.x) smem[t] = src[t];
        __syncthreads();
    }
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    if (VEC2) {
        const int64_t npair = num >> 1;
        for (int64_t q = tid; q < npair; q += nthr) {
            const int64_t i = q << 1;
            bool do0 = true, do1 = true;
            if (MASKED) {
                do0 = mask[i] != 0; do1 = mask[i + 1] != 0;
                if (!do0 && !do1) continue;
            }
            Ray a, b;
            load2<LD>(a, b, P, i);
            double w0a = 0., w0b = 0., w1a = 0., w1b = 0.;
            if (Op::AUX >= 1) { w0a = aux0[i]; w0b = aux0[i + 1]; }
            if (Op::AUX >= 2) { w1a = aux1[i]; w1b = aux1[i + 1]; }
            if (do0) Op::apply(a, prm, smem, w0a, w1a);
            if (do1) Op::apply(b, prm, smem, w0b, w1b);
            store2<ST>(a, b, P, i);
        }
        if ((num & 1) && tid == 0) {
            const int64_t i = num - 1;
            if (!MASKED || mask[i] != 0) {
                Ray a;
                load1<LD>(a, P, i);
                Op::apply(a, prm, smem, Op::AUX >= 1 ? aux0[i] : 0., Op::AUX >= 2 ? aux1[i] : 0.);
                store1<ST>(a, P, i);
            }
        }
    } else {
        for (int64_t i = tid; i < num; i += nthr) {
            if (MASKED && mask[i] == 0) continue;
            Ray a;
            load1<LD>(a, P, i);
            Op::apply(a, prm, smem, Op::AUX >= 1 ? aux0[i] : 0., Op::AUX >= 2 ? aux1[i] : 0.);
            store1<ST>(a, P, i);
        }
    }
}

template <class Op, bool MASKED, bool VEC2>
static int launch3(const RowPtrs &P, int64_t num, const uint8_t *mask, const double *aux0,
                   const double *aux1, const typename Op::Params &prm, cudaStream_t s)
{
    static int ctas = 0;
    if (ctas == 0) {
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_op<Op, MASKED, VEC2>, PXF_BLOCK, 0) !=
                cudaSuccess || nb <= 0) {
            cudaGetLastError();
            nb = 4;
        }
        ctas = nb;
    }
    int64_t items = VEC2 ? ((num + 1) >> 1) : num;
    int grid = grid_for(items, PXF_BLOCK, ctas);
    k_op<Op, MASKED, VEC2><<<grid, PXF_BLOCK, 0, s>>>(P, num, mask, aux0, aux1, prm);
    count_launch();
    return check_launch("k_op");
}

template <class Op>
static int launch_op(RowPtrs P, int64_t num, const uint8_t *mask, const double *aux0, const double *aux1,
                     const typename Op::Params &prm, pxf_stream_t stream)
{
    if (num < 0) { set_error("num < 0"); return PXF_ERR_INVALID; }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    if (num == 0) return PXF_OK;   // empty bundle: nothing to do (pointers may be NULL)
    const unsigned used = Op::LOAD | Op::STORE;
    bool aligned = true;
    for (int k = 0; k < 10; k++) {
        if (used & (1u << k)) {
            if (!P.p[k]) { set_error("null row pointer (row %d)", k); return PXF_ERR_INVALID; }
            if (reinterpret_cast<uintptr_t>(P.p[k]) & 15) aligned = false;
        } else {
            P.p[k] = nullptr;
        }
    }
    if (Op::AUX >= 1 && !aux0) { set_error("null per-ray argument"); return PXF_ERR_INVALID; }
    if (Op::AUX >= 2 && !aux1) { set_error("null per-ray argument"); return PXF_ERR_INVALID; }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if constexpr (OpScalar<Op>::v) {
        if (mask) return launch3<Op, true, false>(P, num, mask, aux0, aux1, prm, s);
        return launch3<Op, false, false>(P, num, mask, aux0, aux1, prm, s);
    } else {
        if (mask) {
            if (aligned) return launch3<Op, true, true>(P, num, mask, aux0, aux1, prm, s);
            return launch3<Op, true, false>(P, num, mask, aux0, aux1, prm, s);
        }
        if (aligned) return launch3<Op, false, true>(P, num, mask, aux0, aux1, prm, s);
        return launch3<Op, false, false>(P, num, mask, aux0, aux1, prm, s);
    }
}

static RowPtrs rows9(double *x, double *y, double *z, double *l, double *m, double *n,
                     double *ux, double *uy, double *uz, double *opd = nullptr)
{
    RowPtrs P;
    P.p[0] = opd; P.p[1] = x; P.p[2] = y; P.p[3] = z; P.p[4] = l; P.p[5] = m; P.p[6] = n;
    P.p[7] = ux; P.p[8] = uy; P.p[9] = uz;
    return P;
}

template <bool OPD>
static int launch_zern(RowPtrs P, int64_t num, const uint8_t *mask, const ZernP &z, pxf_stream_t stream)
{
    if (z.nmax <= 7) return launch_op<OpZern<7, OPD>>(P, num, mask, nullptr, nullptr, z, stream);
    if (z.nmax <= 11) return launch_op<OpZern<11, OPD>>(P, num, mask, nullptr, nullptr, z, stream);
    return launch_op<OpZern<15, OPD>>(P, num, mask, nullptr, nullptr, z, stream);
}

static int launch_ll(RowPtrs P, int64_t num, const uint8_t *mask, int kind, double r0, double z0, double psi, double S,
                     double zmax, double zmin, double dphi, const double *coeff, const int32_t *axial,
                     const int32_t *az, int32_t cnum, pxf_stream_t stream)
{
    if (!coeff || !axial || !az || cnum <= 0) { set_error("bad Legendre table"); return PXF_ERR_INVALID; }
    LLP q;
    if (make_ll(q, kind, r0, z0, psi, S, zmax, zmin, dphi, coeff, axial, az, cnum) < 0) {
        set_error("invalid Legendre orders (need 0 <= order <= %d)", PXF_LL_MAXN);
        return PXF_ERR_INVALID;
    }
    // one instantiation per padded order (the Horner scheme is fully unrolled, coefficients read with static offsets)
    switch (q.s.stride - 1) {
    case 3: return launch_op<OpLL<3>>(P, num, mask, nullptr, nullptr, q, stream);
    case 5: return launch_op<OpLL<5>>(P, num, mask, nullptr, nullptr, q, stream);
    case 7: return launch_op<OpLL<7>>(P, num, mask, nullptr, nullptr, q, stream);
    case 11: return launch_op<OpLL<11>>(P, num, mask, nullptr, nullptr, q, stream);
    default: return launch_op<OpLL<15>>(P, num, mask, nullptr, nullptr, q, stream);
    }
}

}  // namespace pxf

using namespace pxf;

// =================================================================== C ABI
extern "C" {

int pxf_version(void) { return 100; }
const char *pxf_last_error(void) { return g_err; }
int64_t pxf_launch_count(void) { return g_launches.load(); }
int pxf_set_option(int32_t option, int32_t value)
{
    if (option == PXF_OPT_WS_LIBM) { g_ws_libm.store(value ? 1 : 0); return PXF_OK; }
    if (option == PXF_OPT_WS_GRAZE_PPM) { g_ws_graze_ppm.store(value >= 0 ? value : PXF_WS_GRAZE_PPM_DEFAULT); return PXF_OK; }
    if (option == PXF_OPT_WS_RETRACE) { g_ws_retrace.store(value > 0 ? value : PXF_WS_RETRACE_DEFAULT); return PXF_OK; }
    set_error("pxf_set_option: unknown option %d", option);
    return PXF_ERR_INVALID;
}
int pxf_newton_cap(void) { return PXF_NEWTON_CAP; }

int pxf_transform(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num,
                  double tx, double ty, double tz, double rx, double ry, double rz,
                  const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpTransform>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                  make_transform(tx, ty, tz, rx, ry, rz), stream);
}

int pxf_itransform(double *x, double *y, double *z, double *l, double *m, double *n,
                   double *ux, double *uy, double *uz, int64_t num,
                   double tx, double ty, double tz, double rx, double ry, double rz,
                   const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpITransform>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                   make_itransform(tx, ty, tz, rx, ry, rz), stream);
}

int pxf_reflect(double *l, double *m, double *n, double *ux, double *uy, double *uz, int64_t num,
                const uint8_t *mask, pxf_stream_t stream)
{
    NoParams np{0};
    return launch_op<OpReflect>(rows9(nullptr, nullptr, nullptr, l, m, n, ux, uy, uz), num, mask, nullptr,
                                nullptr, np, stream);
}

int pxf_refract(double *l, double *m, double *n, double *ux, double *uy, double *uz, int64_t num,
                double n1, double n2, const uint8_t *mask, pxf_stream_t stream)
{
    RefractP p;
    p.ratio = n1 / n2;
    return launch_op<OpRefract>(rows9(nullptr, nullptr, nullptr, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr, p, stream);
}

int pxf_pointto(const double *x, const double *y, const double *z, double *l, double *m, double *n, int64_t num,
                double x0, double y0, double z0, double reverse, const uint8_t *mask, pxf_stream_t stream)
{
    PointToP p{x0, y0, z0, reverse};
    return launch_op<OpPointTo>(rows9(const_cast<double *>(x), const_cast<double *>(y), const_cast<double *>(z), l, m, n,
                                      nullptr, nullptr, nullptr), num, mask, nullptr, nullptr, p, stream);
}

int pxf_distance(const double *x, const double *y, const double *z, double *dist, int64_t num, double x0, double y0, double z0,
                 const uint8_t *mask, pxf_stream_t stream)
{
    PointToP p{x0, y0, z0, 0.};
    return launch_op<OpDistance>(rows9(const_cast<double *>(x), const_cast<double *>(y), const_cast<double *>(z), nullptr,
                                       nullptr, nullptr, nullptr, nullptr, nullptr, dist), num, mask, nullptr, nullptr, p, stream);
}

int pxf_applyt(double *x, double *y, double *z, double *l, double *m, double *n, double *ux, double *uy, double *uz,
               int64_t num, const double *point_matrix, const double *rotation_matrix, pxf_stream_t stream)
{
    if (!point_matrix || !rotation_matrix) { set_error("pxf_applyt: null matrix"); return PXF_ERR_INVALID; }
    ApplyTP p;
    for (int k = 0; k < 12; k++) { p.P[k] = point_matrix[k]; p.R[k] = rotation_matrix[k]; }
    return launch_op<OpApplyT>(rows9(x, y, z, l, m, n, ux, uy, uz), num, nullptr, nullptr, nullptr, p, stream);
}

int pxf_indangle(const double *l, const double *m, const double *n, const double *ux, const double *uy, const double *uz,
                 double *ang, int64_t num, const double *normal, const uint8_t *mask, pxf_stream_t stream)
{
    IndAngleP p{0., 0., 0., normal ? 1 : 0};
    if (normal) {
        p.nx = normal[0]; p.ny = normal[1]; p.nz = normal[2];
        return launch_op<OpIndAngleFixed>(rows9(nullptr, nullptr, nullptr, const_cast<double *>(l), const_cast<double *>(m),
                                                const_cast<double *>(n), nullptr, nullptr, nullptr, ang),
                                          num, mask, nullptr, nullptr, p, stream);
    }
    return launch_op<OpIndAngle>(rows9(nullptr, nullptr, nullptr, const_cast<double *>(l), const_cast<double *>(m),
                                       const_cast<double *>(n), const_cast<double *>(ux), const_cast<double *>(uy),
                                       const_cast<double *>(uz), ang),
                                 num, mask, nullptr, nullptr, p, stream);
}

int pxf_radgrat(const double *x, const double *y, double *l, double *m, double *n, double wave,
                int64_t num, double dpermm, double order, const uint8_t *mask, pxf_stream_t stream)
{
    // two rays per thread, uncapped (measured: 0.654 / 0.693 / 0.694 / 0.676 / 0.653 ms; shapes as listed at OpMinB)
    return launch_op<OpRadgrat>(rows9(const_cast<double *>(x), const_cast<double *>(y), nullptr, l, m, n,
                                      nullptr, nullptr, nullptr),
                                num, mask, nullptr, nullptr, make_radgrat(wave, dpermm, order), stream);
}

int pxf_radgratw(const double *x, const double *y, double *l, double *m, double *n, const double *wave,
                 int64_t num, double dpermm, double order, const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpRadgratW>(rows9(const_cast<double *>(x), const_cast<double *>(y), nullptr, l, m, n,
                                       nullptr, nullptr, nullptr),
                                 num, mask, wave, nullptr, make_radgrat(0., dpermm, order), stream);
}

int pxf_grat(const double *x, const double *y, double *l, double *m, double *n, int64_t num, double d,
             const double *order, const double *wave, const uint8_t *mask, pxf_stream_t stream)
{
    (void)x; (void)y;
    GratP p{d};
    return launch_op<OpGrat>(rows9(nullptr, nullptr, nullptr, l, m, n, nullptr, nullptr, nullptr), num, mask,
                             order, wave, p, stream);
}

int pxf_flat(double *x, double *y, double *z, const double *l, const double *m, const double *n,
             double *ux, double *uy, double *uz, int64_t num, const uint8_t *mask, pxf_stream_t stream)
{
    FlatP p{0.};
    return launch_op<OpFlat>(rows9(x, y, z, const_cast<double *>(l), const_cast<double *>(m),
                                   const_cast<double *>(n), ux, uy, uz),
                             num, mask, nullptr, nullptr, p, stream);
}

int pxf_flatopd(double *x, double *y, double *z, const double *l, const double *m, const double *n,
                double *ux, double *uy, double *uz, double *opd, int64_t num, double nr,
                const uint8_t *mask, pxf_stream_t stream)
{
    FlatP p{nr};
    return launch_op<OpFlatOpd>(rows9(x, y, z, const_cast<double *>(l), const_cast<double *>(m),
                                      const_cast<double *>(n), ux, uy, uz, opd),
                                num, mask, nullptr, nullptr, p, stream);
}

int pxf_conic(double *x, double *y, double *z, double *l, double *m, double *n,
              double *ux, double *uy, double *uz, int64_t num, double R, double K,
              const uint8_t *mask, pxf_stream_t stream)
{
    // two rays per thread, uncapped (measured: 1.165 / 1.163 / 1.281 / 1.422 / 1.160 ms; shapes as listed at OpMinB)
    return launch_op<OpConic>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr, make_conic(R, K, false, 0.),
                              stream);
}

int pxf_conicopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                 double *ux, double *uy, double *uz, int64_t num, double R, double K, double nr,
                 const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpConicOpd>(rows9(x, y, z, l, m, n, ux, uy, uz, opd), num, mask, nullptr, nullptr,
                                 make_conic(R, K, true, nr), stream);
}

int pxf_wolterprimary(double *x, double *y, double *z, double *l, double *m, double *n,
                      double *ux, double *uy, double *uz, int64_t num, double r0, double z0, double psi,
                      const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpWolterPrimary>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                      make_wolter(r0, z0, psi, false, 0.), stream);
}

int pxf_wolterprimaryopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                         double *ux, double *uy, double *uz, int64_t num,
                         double r0, double z0, double psi, double nr,
                         const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpWolterPrimaryOpd>(rows9(x, y, z, l, m, n, ux, uy, uz, opd), num, mask, nullptr,
                                         nullptr, make_wolter(r0, z0, psi, true, nr), stream);
}

int pxf_woltersecondary(double *x, double *y, double *z, double *l, double *m, double *n,
                        double *ux, double *uy, double *uz, int64_t num, double r0, double z0, double psi,
                        const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpWolterSecondary>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                        make_wolter(r0, z0, psi, false, 0.), stream);
}

int pxf_woltersine(double *x, double *y, double *z, double *l, double *m, double *n,
                   double *ux, double *uy, double *uz, int64_t num,
                   double r0, double z0, double amp, double freq,
                   const uint8_t *mask, pxf_stream_t stream)
{
    // two rays per thread, uncapped (measured: 1.596 / 1.610 / 1.613 / 1.636 / 1.597 ms; shapes as listed at OpMinB --
    // bound by the two sin/cos evaluations per Newton step)
    return launch_op<OpWolterSine>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                   make_woltersine(r0, z0, amp, freq), stream);
}

int pxf_wsprimary(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num, double alpha, double z0, double psi,
                  const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpWsPrimary>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                  make_ws(alpha, z0, psi), stream);
}

int pxf_wssecondary(double *x, double *y, double *z, double *l, double *m, double *n,
                    double *ux, double *uy, double *uz, int64_t num, double alpha, double z0, double psi,
                    const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpWsSecondary>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                    make_ws(alpha, z0, psi), stream);
}

int pxf_spocone(double *x, double *y, double *z, double *l, double *m, double *n,
                double *ux, double *uy, double *uz, int64_t num, double R0, double tg,
                const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpSpoCone>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr, make_spo(R0, tg), stream);
}

int pxf_wolterprimll(double *x, double *y, double *z, double *l, double *m, double *n,
                     double *ux, double *uy, double *uz, int64_t num, double r0, double z0,
                     double zmax, double zmin, double dphi, const double *coeff, const int32_t *axial,
                     const int32_t *az, int32_t cnum, const uint8_t *mask, pxf_stream_t stream)
{
    return launch_ll(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, 0, r0, z0, 1., 0., zmax, zmin, dphi, coeff, axial,
                     az, cnum, stream);
}

int pxf_woltersecll(double *x, double *y, double *z, double *l, double *m, double *n,
                    double *ux, double *uy, double *uz, int64_t num, double r0, double z0, double psi,
                    double zmax, double zmin, double dphi, const double *coeff, const int32_t *axial,
                    const int32_t *az, int32_t cnum, const uint8_t *mask, pxf_stream_t stream)
{
    return launch_ll(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, 1, r0, z0, psi, 0., zmax, zmin, dphi, coeff,
                     axial, az, cnum, stream);
}

int pxf_ellipsoidwoltll(double *x, double *y, double *z, double *l, double *m, double *n,
                        double *ux, double *uy, double *uz, int64_t num, double r0, double z0, double psi,
                        double S, double zmax, double zmin, double dphi, const double *coeff,
                        const int32_t *axial, const int32_t *az, int32_t cnum, const uint8_t *mask,
                        pxf_stream_t stream)
{
    return launch_ll(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, 2, r0, z0, psi, S, zmax, zmin, dphi, coeff,
                     axial, az, cnum, stream);
}

int pxf_tracezern(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num,
                  const double *coeff, const int32_t *rorder, const int32_t *aorder, int32_t arrsize,
                  double rad, const uint8_t *mask, pxf_stream_t stream)
{
    if (!coeff || !rorder || !aorder || arrsize <= 0) { set_error("bad Zernike table"); return PXF_ERR_INVALID; }
    ZernP zp;
    if (make_zern(zp, coeff, rorder, aorder, arrsize, rad, false, 0.) < 0) {
        set_error("invalid Zernike orders (need 0<=n<=15, |m|<=n, n-|m| even, n < radnum(arrsize))");
        return PXF_ERR_INVALID;
    }
    return launch_zern<false>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, zp, stream);
}

int pxf_tracezernopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                     double *ux, double *uy, double *uz, int64_t num,
                     const double *coeff, const int32_t *rorder, const int32_t *aorder, int32_t arrsize,
                     double rad, double nr, const uint8_t *mask, pxf_stream_t stream)
{
    if (!coeff || !rorder || !aorder || arrsize <= 0) { set_error("bad Zernike table"); return PXF_ERR_INVALID; }
    ZernP zp;
    if (make_zern(zp, coeff, rorder, aorder, arrsize, rad, true, nr) < 0) {
        set_error("invalid Zernike orders (need 0<=n<=15, |m|<=n, n-|m| even, n < radnum(arrsize))");
        return PXF_ERR_INVALID;
    }
    return launch_zern<true>(rows9(x, y, z, l, m, n, ux, uy, uz, opd), num, mask, zp, stream);
}


/* ---- surfacesf: remaining surfaces (SURVEY 8f rank 2) ---- */
int pxf_tracesphere(double *x, double *y, double *z, double *l, double *m, double *n,
                    double *ux, double *uy, double *uz, int64_t num, double rad,
                    const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpSphere<false>>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                      make_sphere(rad, false, 0.), stream);
}
int pxf_tracesphereopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                       double *ux, double *uy, double *uz, int64_t num, double rad, double nr,
                       const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpSphere<true>>(rows9(x, y, z, l, m, n, ux, uy, uz, opd), num, mask, nullptr, nullptr,
                                     make_sphere(rad, true, nr), stream);
}
int pxf_tracecyl(double *x, double *y, double *z, double *l, double *m, double *n,
                 double *ux, double *uy, double *uz, int64_t num, double rad,
                 const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpCyl<false>>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                   make_sphere(rad, false, 0.), stream);
}
int pxf_tracecylopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                    double *ux, double *uy, double *uz, int64_t num, double rad, double nr,
                    const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpCyl<true>>(rows9(x, y, z, l, m, n, ux, uy, uz, opd), num, mask, nullptr, nullptr,
                                  make_sphere(rad, true, nr), stream);
}
int pxf_cylconic(double *x, double *y, double *z, double *l, double *m, double *n,
                 double *ux, double *uy, double *uz, int64_t num, double rad, double k,
                 const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpCylConic>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                 make_cylconic(rad, k), stream);
}
int pxf_paraxial(double *x, double *y, double *z, double *l, double *m, double *n,
                 double *ux, double *uy, double *uz, int64_t num, double F,
                 const uint8_t *mask, pxf_stream_t stream)
{
    (void)z; (void)n; (void)ux; (void)uy; (void)uz;
    ParaxialP p{F, 0, 0};
    return launch_op<OpParaxial>(rows9(x, y, nullptr, l, m, nullptr, nullptr, nullptr, nullptr), num, mask, nullptr,
                                 nullptr, p, stream);
}
int pxf_paraxialy(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num, double F,
                  const uint8_t *mask, pxf_stream_t stream)
{
    (void)z; (void)n; (void)ux; (void)uy; (void)uz;
    ParaxialP p{F, 1, 0};
    return launch_op<OpParaxial>(rows9(x, y, nullptr, l, m, nullptr, nullptr, nullptr, nullptr), num, mask, nullptr,
                                 nullptr, p, stream);
}
int pxf_torus(double *x, double *y, double *z, double *l, double *m, double *n,
              double *ux, double *uy, double *uz, int64_t num, double rin, double rout,
              const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpTorus>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                              make_torus(rin, rout), stream);
}
int pxf_conicplus(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num, double R, double K,
                  const double *p, int32_t np, const uint8_t *mask, pxf_stream_t stream)
{
    ConicPlusP q;
    if ((np > 0 && !p) || make_conicplus(q, R, K, p, np, false, 0.) < 0) {
        set_error("conicplus: need 0..%d polynomial terms", PXF_CONICPLUS_MAXP);
        return PXF_ERR_INVALID;
    }
    return launch_op<OpConicPlus<false>>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr, q, stream);
}
int pxf_conicplusopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                     double *ux, double *uy, double *uz, int64_t num, double R, double K,
                     const double *p, int32_t np, double nr, const uint8_t *mask, pxf_stream_t stream)
{
    ConicPlusP q;
    if ((np > 0 && !p) || make_conicplus(q, R, K, p, np, true, nr) < 0) {
        set_error("conicplusopd: need 0..%d polynomial terms", PXF_CONICPLUS_MAXP);
        return PXF_ERR_INVALID;
    }
    return launch_op<OpConicPlus<true>>(rows9(x, y, z, l, m, n, ux, uy, uz, opd), num, mask, nullptr, nullptr, q, stream);
}
int pxf_legsurf(double *x, double *y, double *z, double *l, double *m, double *n,
                double *ux, double *uy, double *uz, int64_t num, double xwidth, double ywidth, double order,
                const double *coeff, const int32_t *xo, const int32_t *yo, int32_t nc,
                const uint8_t *mask, pxf_stream_t stream)
{
    (void)z; (void)ux; (void)uy; (void)uz;
    LegSurfP q;
    if (!coeff || !xo || !yo || make_legsurf(q, xwidth, ywidth, order, coeff, xo, yo, nc) < 0) {
        set_error("legsurf: need 1..%d terms with orders 0..%d", PXF_LEGSURF_MAXC, PXF_LEGSURF_MAXN);
        return PXF_ERR_INVALID;
    }
    return launch_op<OpLegSurf>(rows9(x, y, nullptr, l, m, n, nullptr, nullptr, nullptr), num, mask, nullptr, nullptr,
                                q, stream);
}

/* ---- woltsurf: Wolter-Schwarzschild back surfaces ---- */
int pxf_wsprimaryback(double *x, double *y, double *z, double *l, double *m, double *n,
                      double *ux, double *uy, double *uz, int64_t num, double alpha, double z0, double psi,
                      double thick, const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpWsPrimaryBack>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                      make_ws(alpha, z0, psi, thick), stream);
}
int pxf_wssecondaryback(double *x, double *y, double *z, double *l, double *m, double *n,
                        double *ux, double *uy, double *uz, int64_t num, double alpha, double z0, double psi,
                        double thick, const uint8_t *mask, pxf_stream_t stream)
{
    return launch_op<OpWsSecondaryBack>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, nullptr, nullptr,
                                        make_ws(alpha, z0, psi, thick), stream);
}

/* ---- zernsurf: phase surface and the two-set rotated surface ---- */
int pxf_zernphase(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num, const double *coeff,
                  const int32_t *rorder, const int32_t *aorder, int32_t arrsize, double rad, double wave,
                  const uint8_t *mask, pxf_stream_t stream)
{
    (void)z; (void)ux; (void)uy; (void)uz;
    ZernPhaseP q;
    if (!coeff || !rorder || !aorder || arrsize <= 0 || make_zern(q.z, coeff, rorder, aorder, arrsize, rad, false, 0.) < 0) {
        set_error("zernphase: invalid Zernike table");
        return PXF_ERR_INVALID;
    }
    q.wave = wave;
    RowPtrs P = rows9(x, y, nullptr, l, m, n, nullptr, nullptr, nullptr, opd);
    if (q.z.nmax <= 7) return launch_op<OpZernPhase<7>>(P, num, mask, nullptr, nullptr, q, stream);
    if (q.z.nmax <= 11) return launch_op<OpZernPhase<11>>(P, num, mask, nullptr, nullptr, q, stream);
    return launch_op<OpZernPhase<15>>(P, num, mask, nullptr, nullptr, q, stream);
}
int pxf_tracezernrot(double *x, double *y, double *z, double *l, double *m, double *n,
                     double *ux, double *uy, double *uz, int64_t num,
                     const double *coeff1, const int32_t *rorder1, const int32_t *aorder1, int32_t arrsize1,
                     const double *coeff2, const int32_t *rorder2, const int32_t *aorder2, int32_t arrsize2,
                     double rad, double rot, const uint8_t *mask, pxf_stream_t stream)
{
    ZernP q;
    if (!coeff1 || !rorder1 || !aorder1 || arrsize1 <= 0 || !coeff2 || !rorder2 || !aorder2 || arrsize2 <= 0 ||
        make_zern(q, coeff1, rorder1, aorder1, arrsize1, rad, false, 0.) < 0 ||
        make_zern(q, coeff2, rorder2, aorder2, arrsize2, rad, false, 0., rot, true) < 0) {
        set_error("tracezernrot: invalid Zernike table");
        return PXF_ERR_INVALID;
    }
    return launch_zern<false>(rows9(x, y, z, l, m, n, ux, uy, uz), num, mask, q, stream);
}

}  // extern "C"
