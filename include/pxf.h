/*
 * pxf.h -- C ABI of libpxf.so, the B200 (sm_100a) ray-trace engine that replaces
 * PyXFocus's four f2py Fortran extension modules (transformationsf, surfacesf,
 * woltsurf, zernsurf) plus the numpy analyses on the trace hot path.
 *
 * Conventions
 *   - Every ray array is a DEVICE pointer to `num` contiguous IEEE fp64 values
 *     (one row of the structure-of-arrays bundle [opd,x,y,z,l,m,n,ux,uy,uz],
 *     reference sources.py:1-15).  Arrays are mutated in place, exactly like the
 *     Fortran `intent(inout)` arguments they replace.  Rows may be independent
 *     allocations; when every row is 16-byte aligned the kernels use double2
 *     loads/stores.
 *   - Scalars have the meaning and order of the Fortran dummy arguments
 *     (file:line cited at each entry).  The array-length argument `num` that
 *     f2py hides is explicit here.
 *   - `mask` (nullable) is a device uint8 array of length num: ray i is
 *     processed iff mask[i] != 0.  It replaces the reference's ind= gather ->
 *     Fortran -> scatter idiom (transformations.py:20-27, surfaces.py:17-24).
 *   - `stream` is a cudaStream_t (CUstream); work is enqueued asynchronously.
 *     Entry points that return scalars to host memory synchronise the stream.
 *   - Return value: PXF_OK or an error code; pxf_last_error() gives text.
 *     Per-ray failures stay in-band exactly as in the reference (zeroed
 *     direction cosines, NaN, restored positions).
 *   - No CPU fallback exists: without a CUDA device every entry point that
 *     touches rays returns PXF_ERR_CUDA.
 */
#ifndef PXF_H
#define PXF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st *pxf_stream_t;

enum {
    PXF_OK = 0,
    PXF_ERR_INVALID = 1, /* bad argument (null pointer, negative size, bad table) */
    PXF_ERR_CUDA = 2,    /* CUDA runtime/launch failure                           */
    PXF_ERR_NOMEM = 3,   /* workspace allocation failed                           */
    PXF_ERR_UNSUPPORTED = 4
};

int pxf_version(void);
const char *pxf_last_error(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t pxf_launch_count(void);
/* Process-wide options.
 *   PXF_OPT_WS_LIBM (default 0): 1 = evaluate the Wolter-Schwarzschild surfaces (wsprimary/wssecondary and the back
 *   surfaces) with the reference's own libm call sequence (asin/atan2/sincos/tan/pow per Newton step, woltsurf.f95:
 *   420-449,513-551), every function CORRECTLY ROUNDED (double-double evaluation, one rounding), instead of the
 *   algebraically identical transcendental-free form.  Both agree with the reference to 1e-12 on every ray inside the
 *   field of view; the exact form is bit for bit against an oracle whose libm is correctly rounded at ANY field
 *   angle, including the chaotic rays around and beyond the graze angle whose discrete outcome (which root, restored
 *   or not) hangs on the last bit.  ~50x slower.
 *   PXF_OPT_WS_RETRACE (default off): n > 0 = rays that took >= n Newton steps in the default form, or that the
 *   iteration cap restored while still converging, are traced again with the exact form (the fringe of the
 *   restored set).  PXF_OPT_WS_GRAZE_PPM (default 0): also those whose sine of the graze angle is below value*1e-6. */
enum pxf_option { PXF_OPT_WS_LIBM = 1, PXF_OPT_WS_RETRACE = 2, PXF_OPT_WS_GRAZE_PPM = 3 };
int pxf_set_option(int32_t option, int32_t value);
/* Iteration cap applied to the reference's uncapped Newton loops (oracle uses the same). */
int pxf_newton_cap(void);

/* ======================= transformationsf =============================== */
/* transformationsf.f95:134-163  transform(x,y,z,l,m,n,ux,uy,uz,num,tx,ty,tz,rx,ry,rz) */
int pxf_transform(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num,
                  double tx, double ty, double tz, double rx, double ry, double rz,
                  const uint8_t *mask, pxf_stream_t stream);
/* transformationsf.f95:168-201 */
int pxf_itransform(double *x, double *y, double *z, double *l, double *m, double *n,
                   double *ux, double *uy, double *uz, int64_t num,
                   double tx, double ty, double tz, double rx, double ry, double rz,
                   const uint8_t *mask, pxf_stream_t stream);
/* transformationsf.f95:60-79 */
int pxf_reflect(double *l, double *m, double *n, double *ux, double *uy, double *uz, int64_t num,
                const uint8_t *mask, pxf_stream_t stream);
/* transformationsf.f95:82-130 */
int pxf_refract(double *l, double *m, double *n, double *ux, double *uy, double *uz, int64_t num,
                double n1, double n2, const uint8_t *mask, pxf_stream_t stream);
/* transformations.pointTo (transformations.py:91-100): l,m,n = reverse*(r - p0)/|r - p0|. */
int pxf_pointto(const double *x, const double *y, const double *z, double *l, double *m, double *n, int64_t num,
                double x0, double y0, double z0, double reverse, const uint8_t *mask, pxf_stream_t stream);
/* analyses.measureOPD (analyses.py:232-244): dist[i] = |r_i - p0|. */
int pxf_distance(const double *x, const double *y, const double *z, double *dist, int64_t num, double x0, double y0, double z0,
                 const uint8_t *mask, pxf_stream_t stream);
/* transformations.applyT (transformations.py:257-280), in place: positions through the first three rows of the 4x4
 * point matrix, direction cosines and normals through those of the 4x4 rotation matrix (HOST row-major double[>=12],
 * i.e. coords[i+1] and coords[i]). */
int pxf_applyt(double *x, double *y, double *z, double *l, double *m, double *n, double *ux, double *uy, double *uz,
               int64_t num, const double *point_matrix, const double *rotation_matrix, pxf_stream_t stream);
/* analyses.indAngle (analyses.py:164-182): ang[i] = arccos(l ux + m uy + n uz), or arccos(normal . (l,m,n)) when
 * `normal` (HOST double[3]) is given (ux,uy,uz may then be NULL).  Rays with mask[i]==0 leave ang[i] untouched. */
int pxf_indangle(const double *l, const double *m, const double *n, const double *ux, const double *uy, const double *uz,
                 double *ang, int64_t num, const double *normal, const uint8_t *mask, pxf_stream_t stream);
/* transformationsf.f95:205-238 (scalar wavelength; sign of n kept) */
int pxf_radgrat(const double *x, const double *y, double *l, double *m, double *n, double wave,
                int64_t num, double dpermm, double order, const uint8_t *mask, pxf_stream_t stream);
/* transformationsf.f95:242-272 (per-ray wavelength; sign taken from y) */
int pxf_radgratw(const double *x, const double *y, double *l, double *m, double *n, const double *wave,
                 int64_t num, double dpermm, double order, const uint8_t *mask, pxf_stream_t stream);
/* transformationsf.f95:277-305 (linear grating, per-ray order and wavelength) */
int pxf_grat(const double *x, const double *y, double *l, double *m, double *n, int64_t num, double d,
             const double *order, const double *wave, const uint8_t *mask, pxf_stream_t stream);

/* ======================= surfacesf ====================================== */
/* surfacesf.f95:4-29 (REAL*4 delta) */
int pxf_flat(double *x, double *y, double *z, const double *l, const double *m, const double *n,
             double *ux, double *uy, double *uz, int64_t num, const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:32-53 */
int pxf_flatopd(double *x, double *y, double *z, const double *l, const double *m, const double *n,
                double *ux, double *uy, double *uz, double *opd, int64_t num, double nr,
                const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:302-360 */
int pxf_conic(double *x, double *y, double *z, double *l, double *m, double *n,
              double *ux, double *uy, double *uz, int64_t num, double R, double K,
              const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:366-420 */
int pxf_conicopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                 double *ux, double *uy, double *uz, int64_t num, double R, double K, double nr,
                 const uint8_t *mask, pxf_stream_t stream);

/* ======================= woltsurf ======================================= */
/* woltsurf.f95:7-54 */
int pxf_wolterprimary(double *x, double *y, double *z, double *l, double *m, double *n,
                      double *ux, double *uy, double *uz, int64_t num, double r0, double z0, double psi,
                      const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:60-108 */
int pxf_wolterprimaryopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                         double *ux, double *uy, double *uz, int64_t num,
                         double r0, double z0, double psi, double nr,
                         const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:114-161 */
int pxf_woltersecondary(double *x, double *y, double *z, double *l, double *m, double *n,
                        double *ux, double *uy, double *uz, int64_t num, double r0, double z0, double psi,
                        const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:167-215 */
int pxf_woltersine(double *x, double *y, double *z, double *l, double *m, double *n,
                   double *ux, double *uy, double *uz, int64_t num,
                   double r0, double z0, double amp, double freq,
                   const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:387-476 */
int pxf_wsprimary(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num, double alpha, double z0, double psi,
                  const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:484-588 */
int pxf_wssecondary(double *x, double *y, double *z, double *l, double *m, double *n,
                    double *ux, double *uy, double *uz, int64_t num, double alpha, double z0, double psi,
                    const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:591-638 */
int pxf_spocone(double *x, double *y, double *z, double *l, double *m, double *n,
                double *ux, double *uy, double *uz, int64_t num, double R0, double tg,
                const uint8_t *mask, pxf_stream_t stream);

/* Legendre-Legendre deformed shells.  coeff/axial/az are HOST pointers (cnum terms, orders
 * 0..15), like the Zernike tables below. */
/* woltsurf.f95:219-288 */
int pxf_wolterprimll(double *x, double *y, double *z, double *l, double *m, double *n,
                     double *ux, double *uy, double *uz, int64_t num, double r0, double z0,
                     double zmax, double zmin, double dphi, const double *coeff, const int32_t *axial,
                     const int32_t *az, int32_t cnum, const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:293-379 */
int pxf_woltersecll(double *x, double *y, double *z, double *l, double *m, double *n,
                    double *ux, double *uy, double *uz, int64_t num, double r0, double z0, double psi,
                    double zmax, double zmin, double dphi, const double *coeff, const int32_t *axial,
                    const int32_t *az, int32_t cnum, const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:643-718 */
int pxf_ellipsoidwoltll(double *x, double *y, double *z, double *l, double *m, double *n,
                        double *ux, double *uy, double *uz, int64_t num, double r0, double z0, double psi,
                        double S, double zmax, double zmin, double dphi, const double *coeff,
                        const int32_t *axial, const int32_t *az, int32_t cnum, const uint8_t *mask,
                        pxf_stream_t stream);

/* ---- remaining surfacesf routines (one entry per Fortran subroutine) ---- */
/* surfacesf.f95:57-101 */
int pxf_tracesphere(double *x, double *y, double *z, double *l, double *m, double *n,
                    double *ux, double *uy, double *uz, int64_t num, double rad,
                    const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:104-149 */
int pxf_tracesphereopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                       double *ux, double *uy, double *uz, int64_t num, double rad, double nr,
                       const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:153-197 */
int pxf_tracecyl(double *x, double *y, double *z, double *l, double *m, double *n,
                 double *ux, double *uy, double *uz, int64_t num, double rad,
                 const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:201-246 */
int pxf_tracecylopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                    double *ux, double *uy, double *uz, int64_t num, double rad, double nr,
                    const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:251-296 (rad is the curvature) */
int pxf_cylconic(double *x, double *y, double *z, double *l, double *m, double *n,
                 double *ux, double *uy, double *uz, int64_t num, double rad, double k,
                 const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:423-440 */
int pxf_paraxial(double *x, double *y, double *z, double *l, double *m, double *n,
                 double *ux, double *uy, double *uz, int64_t num, double F,
                 const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:443-460 */
int pxf_paraxialy(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num, double F,
                  const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:468-508 */
int pxf_torus(double *x, double *y, double *z, double *l, double *m, double *n,
              double *ux, double *uy, double *uz, int64_t num, double rin, double rout,
              const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:514-572.  p: HOST pointer, np (<= 16) even-polynomial terms */
int pxf_conicplus(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num, double R, double K,
                  const double *p, int32_t np, const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:578-638 */
int pxf_conicplusopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                     double *ux, double *uy, double *uz, int64_t num, double R, double K,
                     const double *p, int32_t np, double nr, const uint8_t *mask, pxf_stream_t stream);
/* surfacesf.f95:642-668.  coeff/xo/yo: HOST pointers, nc (<= 48) terms, orders 0..15 */
int pxf_legsurf(double *x, double *y, double *z, double *l, double *m, double *n,
                double *ux, double *uy, double *uz, int64_t num, double xwidth, double ywidth, double order,
                const double *coeff, const int32_t *xo, const int32_t *yo, int32_t nc,
                const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:726-815 */
int pxf_wsprimaryback(double *x, double *y, double *z, double *l, double *m, double *n,
                      double *ux, double *uy, double *uz, int64_t num, double alpha, double z0, double psi,
                      double thick, const uint8_t *mask, pxf_stream_t stream);
/* woltsurf.f95:824-933 */
int pxf_wssecondaryback(double *x, double *y, double *z, double *l, double *m, double *n,
                        double *ux, double *uy, double *uz, int64_t num, double alpha, double z0, double psi,
                        double thick, const uint8_t *mask, pxf_stream_t stream);
/* zernsurf.f95:206-250 (tables are HOST pointers, as for pxf_tracezern) */
int pxf_zernphase(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num, const double *coeff,
                  const int32_t *rorder, const int32_t *aorder, int32_t arrsize, double rad, double wave,
                  const uint8_t *mask, pxf_stream_t stream);
/* zernsurf.f95:257-359: two Zernike sets, the second evaluated at theta+rot */
int pxf_tracezernrot(double *x, double *y, double *z, double *l, double *m, double *n,
                     double *ux, double *uy, double *uz, int64_t num,
                     const double *coeff1, const int32_t *rorder1, const int32_t *aorder1, int32_t arrsize1,
                     const double *coeff2, const int32_t *rorder2, const int32_t *aorder2, int32_t arrsize2,
                     double rad, double rot, const uint8_t *mask, pxf_stream_t stream);

/* ======================= zernsurf ======================================= */
/* zernsurf.f95:8-101.  coeff/rorder/aorder are HOST pointers (arrsize entries; the f2py
 * wrapper receives them as small numpy arrays, surfaces.py:39-43).  rorder[i] <= 15. */
int pxf_tracezern(double *x, double *y, double *z, double *l, double *m, double *n,
                  double *ux, double *uy, double *uz, int64_t num,
                  const double *coeff, const int32_t *rorder, const int32_t *aorder, int32_t arrsize,
                  double rad, const uint8_t *mask, pxf_stream_t stream);
/* zernsurf.f95:108-203 */
int pxf_tracezernopd(double *opd, double *x, double *y, double *z, double *l, double *m, double *n,
                     double *ux, double *uy, double *uz, int64_t num,
                     const double *coeff, const int32_t *rorder, const int32_t *aorder, int32_t arrsize,
                     double rad, double nr, const uint8_t *mask, pxf_stream_t stream);

/* ======================= fused per-ray program ========================== */
/* One kernel: load a ray once, run a list of the operations above in registers,
 * store once.  Arithmetic is the same device code as the per-op entry points, so
 * results are bit-identical to calling them one by one. */
enum {
    PXF_OP_TRANSFORM = 1,      /* p: tx,ty,tz,rx,ry,rz                 */
    PXF_OP_ITRANSFORM = 2,     /* p: tx,ty,tz,rx,ry,rz                 */
    PXF_OP_REFLECT = 3,
    PXF_OP_REFRACT = 4,        /* p: n1,n2                             */
    PXF_OP_RADGRAT = 5,        /* p: wave,dpermm,order                 */
    PXF_OP_FLAT = 6,
    PXF_OP_FLATOPD = 7,        /* p: nr                                */
    PXF_OP_CONIC = 8,          /* p: R,K                               */
    PXF_OP_CONICOPD = 9,       /* p: R,K,nr                            */
    PXF_OP_WOLTERPRIMARY = 10, /* p: r0,z0,psi                         */
    PXF_OP_WOLTERPRIMARYOPD = 11, /* p: r0,z0,psi,nr                   */
    PXF_OP_WOLTERSECONDARY = 12,  /* p: r0,z0,psi                      */
    PXF_OP_WOLTERSINE = 13,    /* p: r0,z0,amp,freq                    */
    PXF_OP_WSPRIMARY = 14,     /* p: alpha,z0,psi                      */
    PXF_OP_WSSECONDARY = 15,   /* p: alpha,z0,psi                      */
    PXF_OP_SPOCONE = 16,       /* p: R0,tg                             */
    PXF_OP_VIGNETTE_MAG = 17,  /* kill ray unless l^2+m^2+n^2 > .1 (transformations.py:220-223) */
    PXF_OP_VIGNETTE_BOX = 18,  /* p: row(1..9),lo,hi ; kill ray unless lo < row < hi             */
    PXF_OP_VIGNETTE_ABS = 19,  /* p: row(1..9),hi[,c] ; kill ray unless |row - c| < hi (c defaults to 0)   */
    PXF_OP_ZERNSURF = 21,      /* p: table (a DEVICE copy of what pxf_zern_table_fill wrote, its address bit-cast
                                  into the double), opd flag (0: tracezern, 1: tracezernOPD), nmax as returned by
                                  the fill.  Radial orders <= 7 only; at most one Zernike table per program.     */
    PXF_OP_KICK = 20,          /* p: dl,dm,sn ; l+=dl, m+=dm, n=sn*sqrt(1-l^2-m^2) (field angle,
                                  examples/axro/axialHeights.py:94-95 with dm=0 uses l only)   */
    PXF_OP_KICKN = 22,         /* p: dl,dm ; l+=dl, m+=dm, n=-sqrt(n^2-dl^2-dm^2): the pointing offsets of
                                  examples/arcus/cat.py:246-249                                 */
    PXF_OP_VIGNETTE_RHOGT = 23, /* p: rho0 ; kill ray unless sqrt(x^2+y^2) > rho0 (the back-of-previous-shell test,
                                  examples/axro/axialHeights.py:285-286)                        */
    PXF_OP_GRATFAN = 24,       /* p: ang,hubdist,l,dpermm,order,wave ; the fanned radial-grating array of
                                  examples/arcus/sector.py:636-700 as ONE per-ray loop (see pxf_trace_program_aux).
                                  wave = NaN: per-ray wavelengths from aux.wave (radgratW), else scalar (radgrat). */
    PXF_OP_ROTX_REMAINING = 25, /* p: ang,total ; apply transform(0,0,0,ang,0,0) (total - aux.count[i]) times: the
                                  whole-bundle rotations a ray still receives after it met its grating */
    PXF_OP_LLSURF = 26,        /* p: table (a DEVICE copy of what pxf_ll_table_fill wrote, its address bit-cast into
                                  the double), highest order as returned by the fill (it must be that value: the
                                  specialised kernels evaluate the terms up to the order p[1] rounds to -- 3, 5 or
                                  7 -- so a smaller p[1] drops terms on that path, silently, and not in the
                                  interpreter, which evaluates all 8x8).  A Legendre-Legendre shell
                                  (wolterprimLL / woltersecLL / ellipsoidWoltLL, the kind is in the table) with the
                                  bits of pxf_wolterprimll / pxf_woltersecll / pxf_ellipsoidwoltll.  Orders <= 7 only;
                                  at most two per program, and not in a program with PXF_OP_ZERNSURF or
                                  PXF_OP_GRATFAN (PXF_ERR_UNSUPPORTED).                                          */
    /* The remaining scalar surfaces of surfacesf / woltsurf, with the bits of the stand-alone entry point of the
     * same name (the scalars mean what they mean there).  A program that holds one of them together with
     * PXF_OP_ZERNSURF, PXF_OP_LLSURF, PXF_OP_GRATFAN or PXF_OP_ROTX_REMAINING is refused (PXF_ERR_UNSUPPORTED). */
    PXF_OP_TRACESPHERE = 27,   /* p: rad ; pxf_tracesphere (a ray that misses is zeroed and gets a NaN normal) */
    PXF_OP_TRACESPHEREOPD = 28, /* p: rad,nr ; pxf_tracesphereopd                                        */
    PXF_OP_TRACECYL = 29,      /* p: rad ; pxf_tracecyl (cylinder about y; misses as for the sphere)     */
    PXF_OP_TRACECYLOPD = 30,   /* p: rad,nr ; pxf_tracecylopd                                           */
    PXF_OP_CYLCONIC = 31,      /* p: rad,k ; pxf_cylconic                                               */
    PXF_OP_PARAXIAL = 32,      /* p: F ; pxf_paraxial                                                   */
    PXF_OP_PARAXIALY = 33,     /* p: F ; pxf_paraxialy (m only)                                         */
    PXF_OP_TORUS = 34,         /* p: rin,rout ; pxf_torus                                               */
    PXF_OP_WSPRIMARYBACK = 35, /* p: alpha,z0,psi,thick ; pxf_wsprimaryback (PXF_OPT_WS_* apply as to
                                  PXF_OP_WSPRIMARY)                                                    */
    PXF_OP_WSSECONDARYBACK = 36, /* p: alpha,z0,psi,thick ; pxf_wssecondaryback                        */
    PXF_OP_ZERNPHASE = 37,     /* p: table (a DEVICE copy of what pxf_zern_table_fill wrote with opd = 0, its address
                                  bit-cast into the double), wave, nmax as returned by the fill ; pxf_zernphase.
                                  Radial orders <= 7 only.  A program's single Zernike-table op: refused
                                  (PXF_ERR_UNSUPPORTED) next to PXF_OP_ZERNSURF, another PXF_OP_ZERNPHASE,
                                  PXF_OP_LLSURF, PXF_OP_GRATFAN, PXF_OP_ROTX_REMAINING or ops 27..40.           */
    /* Two more surfaces of the family of ops 27..36 (they may share a program with those, and are refused where those
     * are).  Their parameter block is a table in DEVICE memory, its address bit-cast into p[0]; the table must stay
     * alive as long as a program or segmented table refers to it. */
    PXF_OP_CONICPLUS = 38,     /* p: table (pxf_conicplus_table_fill, opd = 0) ; pxf_conicplus                    */
    PXF_OP_CONICPLUSOPD = 39,  /* p: table (pxf_conicplus_table_fill, opd = 1, nr) ; pxf_conicplusopd            */
    PXF_OP_LEGSURF = 40,       /* p: table (pxf_legsurf_table_fill) ; pxf_legsurf                                 */
    /* The gratings with per-ray arrays.  Each array is a DEVICE double[num], its address bit-cast into the double, and
     * indexed by the ray's index in the bundle the program runs on (in a segmented program: in the whole bundle, so
     * segment s reads entries seg_start[s] .. seg_start[s+1]-1).  A null address is PXF_ERR_INVALID.  The arrays
     * must stay alive as long as a program or segmented table refers to them.  These ops run in the side-array
     * interpreter: a program that also holds PXF_OP_ZERNSURF, PXF_OP_ZERNPHASE, PXF_OP_LLSURF or ops 27..40 is
     * refused (PXF_ERR_UNSUPPORTED), and so is pxf_host_trace_program, which has no device arrays to point at. */
    PXF_OP_RADGRATW = 41,      /* p: wave (array), dpermm, order ; pxf_radgratw (the sign of n comes from y)       */
    PXF_OP_GRAT = 42           /* p: d, order (array), wave (array) ; pxf_grat (l, m, n zeroed where
                                  l^2+m^2 > 1 after the kick)                                                      */
};
typedef struct pxf_op {
    int32_t code;
    int32_t reserved;
    double p[6];
} pxf_op;
#define PXF_MAX_OPS 24
/* rays[10] = device pointers in bundle order [opd,x,y,z,l,m,n,ux,uy,uz] (opd may be NULL when
 * no OPD op is in the program).  alive (nullable): device uint8[num], set to 0 for rays killed
 * by a VIGNETTE op (they stop executing at that op; their state at that point is stored), 1
 * otherwise.  Required when the program contains a VIGNETTE op. */
/* Table for a PXF_OP_ZERNSURF op: folds (coeff, rorder, aorder, rad, nr) exactly as pxf_tracezern[opd] does into
 * pxf_zern_table_bytes() bytes of HOST memory; the caller uploads them unchanged.  Returns the highest radial order
 * (>= 0) or -1 for an invalid term list. */
size_t pxf_zern_table_bytes(void);
int32_t pxf_zern_table_fill(const double *coeff, const int32_t *rorder, const int32_t *aorder, int32_t arrsize,
                            double rad, int32_t opd, double nr, void *table_host);
/* Table for a PXF_OP_LLSURF op: folds the term list exactly as pxf_wolterprimll (kind 0; psi and S unused),
 * pxf_woltersecll (kind 1; S unused) or pxf_ellipsoidwoltll (kind 2) do, into pxf_ll_table_bytes() bytes of HOST
 * memory: the scalars and the coefficient matrix as an 8x8 block, zero beyond the orders present.  The caller uploads
 * them unchanged.  Returns the highest axial / azimuthal order (0..7), or -1 for an invalid term list or an order
 * above 7 (those run through the stand-alone routines). */
size_t pxf_ll_table_bytes(void);
int32_t pxf_ll_table_fill(int32_t kind, double r0, double z0, double psi, double S, double zmax, double zmin,
                          double dphi, const double *coeff, const int32_t *axial, const int32_t *az, int32_t cnum,
                          void *table_host);
/* Table of the two Zernike sets of pxf_tracezernrot (the second evaluated at theta + rot), folded by the same two
 * steps, into pxf_zern_table_bytes() bytes of HOST memory.  It is a PXF_OP_ZERNSURF table (opd flag 0): a rotated
 * Zernike surface needs no opcode of its own.  Returns the highest radial order or -1. */
int32_t pxf_zern_table_fill_rot(const double *coeff1, const int32_t *rorder1, const int32_t *aorder1, int32_t arrsize1,
                                const double *coeff2, const int32_t *rorder2, const int32_t *aorder2, int32_t arrsize2,
                                double rad, double rot, void *table_host);
/* Table for a PXF_OP_CONICPLUS (opd = 0) / PXF_OP_CONICPLUSOPD (opd = 1) op: R, K and 0..16 polynomial terms folded
 * exactly as pxf_conicplus[opd] does, into pxf_conicplus_table_bytes() bytes of HOST memory; the caller uploads them
 * unchanged.  Returns the byte count, or -1 for more than 16 terms. */
size_t pxf_conicplus_table_bytes(void);
int32_t pxf_conicplus_table_fill(double R, double K, const double *p, int32_t np, int32_t opd, double nr,
                                 void *table_host);
/* Table for a PXF_OP_LEGSURF op: 0..48 terms with orders 0..15, folded exactly as pxf_legsurf does, into
 * pxf_legsurf_table_bytes() bytes of HOST memory.  Returns the byte count, or -1 for an invalid term list. */
size_t pxf_legsurf_table_bytes(void);
int32_t pxf_legsurf_table_fill(double xwidth, double ywidth, double order, const double *coeff, const int32_t *xo,
                               const int32_t *yo, int32_t nc, void *table_host);
int pxf_trace_program(double *const rays[10], int64_t num, const pxf_op *ops, int32_t nops,
                      uint8_t *alive, pxf_stream_t stream);
/* Per-ray side arrays of the ops that need them (all device pointers, each nullable unless an op uses it):
 *   wave       double[num]  per-ray wavelength of a PXF_OP_GRATFAN with p.wave = NaN
 *   count      int32[num]   PXF_OP_GRATFAN writes the number of fan rotations the ray received before it met a
 *                           grating (-1: it never did within `cap` gratings); PXF_OP_ROTX_REMAINING reads it
 *   count_max  int32[1]     PXF_OP_GRATFAN raises it (atomic max) to the largest count of the launch; the caller
 *                           zeroes it beforehand.  cap + 1 when some ray never met a grating.
 *   cap        most gratings a ray may pass (<= 0: 4096); the reference's loop would not terminate instead.
 * PXF_OP_GRATFAN, per ray (sector.py:681-707; each step is the masked whole-bundle call of the reference):
 *   repeat { if |asin(n)| > .001: flat ; rho = -sqrt(x^2+y^2)*sign(y) ; if hubdist < rho < l+hubdist: stop ;
 *            transform(0,0,0,ang,0,0) } ; reflect ; radgrat[W](dpermm, order, wave).
 * rays_out == NULL: in place. */
typedef struct pxf_program_aux {
    const double *wave;
    int32_t *count;
    int32_t *count_max;
    int32_t cap;
    int32_t reserved;
} pxf_program_aux;
int pxf_trace_program_aux(double *const rays_in[10], double *const rays_out[10], int64_t num,
                          const pxf_op *ops, int32_t nops, uint8_t *alive, const pxf_program_aux *aux,
                          double *sums_dev, void *scratch, pxf_stream_t stream);
/* Run-time specialisation.  Every op list that is not one of the chains built into the library is compiled once
 * (NVRTC, sm_100a, the library's arithmetic flags) into a straight-line kernel of the same per-op device functions
 * -- same bits as the interpreter -- and cached by signature in memory and under <libpxf dir>/_jit/ (PXF_JIT_CACHE
 * overrides).  Bundles below PXF_JIT_MIN_RAYS (default 262144) use a cached kernel when there is one and the
 * interpreter otherwise; PXF_JIT=0 turns it off.
 *   pxf_jit_compile      compile (no GPU needed) the kernels a program will want -- in place / out of place, with /
 *                        without the centroid sums; segmented != 0: the segmented form.  Returns the number of
 *                        kernels now available (0: NVRTC missing or the compilation failed), -1: invalid program.
 *                        Ops with a device table (PXF_OP_ZERNSURF, LLSURF, ZERNPHASE, CONICPLUS[OPD], LEGSURF): any
 *                        non-null table address will do; aux may be NULL.
 *   pxf_jit_status       "ok" or why the interpreter is being used, plus counters
 *   pxf_last_trace_kernel  name of the kernel the last trace on this process launched                          */
int32_t pxf_jit_compile(const pxf_op *ops, int32_t nops, int32_t segmented, const pxf_program_aux *aux);
const char *pxf_jit_status(void);
const char *pxf_last_trace_kernel(void);
/* Out-of-place variant: rows are read from rays_in and every row the program reads or writes
 * is stored to rays_out (rows it touches neither way are not copied).  rays_in is left
 * untouched, e.g. to trace one source bundle through several configurations. */
int pxf_trace_program_to(double *const rays_in[10], double *const rays_out[10], int64_t num,
                         const pxf_op *ops, int32_t nops, uint8_t *alive, pxf_stream_t stream);
/* As above (rays_out == NULL: in place) and, from the same kernel, the centroid sums of the
 * FINAL bundle over the surviving rays: sums_dev (device double[16]) = {count, sum x, sum y,
 * count}, i.e. what analyses.centroid / hpd (analyses.py:16-22,88-97) need next -- no extra
 * pass over x,y.  scratch: pxf_sums_scratch_bytes() device bytes. */
int pxf_trace_program_sums(double *const rays_in[10], double *const rays_out[10], int64_t num,
                           const pxf_op *ops, int32_t nops, uint8_t *alive, double *sums_dev,
                           void *scratch, pxf_stream_t stream);

/* Segmented programs (nested mirror assemblies, BASELINE config 5; the reference loops over shells in Python,
 * examples/axro/axialHeights.py:215-322): the bundle is the concatenation of nseg segments
 * [seg_start[s], seg_start[s+1]) and segment s runs ops[s*nops .. s*nops+nops) -- the same opcode sequence
 * for every segment, its own scalars.  ONE launch for the whole bundle.
 *   pxf_segmented_table_fill folds the scalars into a host table (pxf_segmented_table_bytes bytes; seg_start
 *   has nseg+1 entries, seg_start[0] == 0); the caller uploads it unchanged to device memory and passes both
 *   copies to pxf_trace_program_segmented (the host copy is read for the row masks only).
 *   The surface ops 27..36 (PXF_OP_TRACESPHERE .. PXF_OP_WSSECONDARYBACK) go through this pair; their scalars may
 *   differ between segments.  So do PXF_OP_CONICPLUS / CONICPLUSOPD / LEGSURF: each segment's op carries the device
 *   address of its own table, copied like any scalar, so those tables must outlive the segmented table.  The _zern
 *   and _ll fills refuse ops 27..36 and 38..40 (PXF_ERR_UNSUPPORTED).
 *   PXF_OP_RADGRATW / PXF_OP_GRAT go through this pair as well, with their scalars per segment.  Their arrays are
 *   indexed by the ray's index in the WHOLE bundle (segment s reads entries seg_start[s] .. seg_start[s+1]-1); the
 *   segments' ops may carry the same or different addresses, and the arrays must outlive the segmented table.  The
 *   _zern and _ll fills refuse them (PXF_ERR_UNSUPPORTED).
 *   rays_out == NULL: in place. */
size_t pxf_segmented_table_bytes(int32_t nops, int32_t nseg);
int pxf_segmented_table_fill(const pxf_op *ops, int32_t nops, int32_t nseg, const int64_t *seg_start,
                             void *table_host);
int pxf_trace_program_segmented(double *const rays_in[10], double *const rays_out[10], int64_t num,
                                const void *table_host, const void *table_dev, uint8_t *alive,
                                pxf_stream_t stream);
/* Segmented programs with one Zernike surface per segment (a figure-error Monte Carlo, or shells that each have a
 * measured figure): every segment's op list has its PXF_OP_ZERNSURF at the same position, with the same opd flag
 * (p[1]); the term count, radial order (<= 7), rad and nr may differ.  pxf_segmented_table_fill refuses such lists;
 * this pair takes them (and any list the plain pair takes, except one with ops 27..36 or 38..40).
 * PXF_OP_ZERNPHASE may take the place of PXF_OP_ZERNSURF: the same opcode in every segment, each with its own table
 * and wave (p[1]); segments whose Zernike op differs in kind are refused (PXF_ERR_INVALID).
 *   zern_tables_host: nseg consecutive tables of pxf_zern_table_bytes() bytes, table s filled by pxf_zern_table_fill
 *   for segment s (NULL is accepted when no op is a PXF_OP_ZERNSURF).  They are copied into the segmented table, so it
 *   stays self-contained: upload it unchanged and pass both copies to pxf_trace_program_segmented, which stages the
 *   segment's Zernike table next to its op table -- still ONE launch.  The op's p[0] (device table address) is not
 *   used; its nmax p[2] is taken from the table.
 *   Returns PXF_ERR_UNSUPPORTED for a table of radial order > 7 and for PXF_OP_GRATFAN / PXF_OP_ROTX_REMAINING,
 *   PXF_ERR_INVALID for segments that differ in opcode sequence or opd flag, or for missing tables. */
size_t pxf_segmented_table_bytes_zern(int32_t nops, int32_t nseg);
int pxf_segmented_table_fill_zern(const pxf_op *ops, int32_t nops, int32_t nseg, const int64_t *seg_start,
                                  const void *zern_tables_host, void *table_host);
/* Segmented programs with Legendre-Legendre shells (a figure-error Monte Carlo of a Wolter-I pair, or shells that each
 * have a measured figure): every segment's op list has its PXF_OP_LLSURF ops (one or two) at the same positions.
 * Kinds, term lists and orders (<= 7) may differ between segments.  pxf_segmented_table_fill and
 * pxf_segmented_table_fill_zern refuse such lists; this pair takes them (and any list the plain pair takes, except one
 * with ops 27..36 or 38..40).
 *   ll_tables_host: nseg * (LL ops per program) tables of pxf_ll_table_bytes() bytes, segment-major and in op order,
 *   each filled by pxf_ll_table_fill (NULL is accepted when no op is a PXF_OP_LLSURF).  They are copied into the
 *   segmented table (pxf_segmented_table_bytes_ll has room for two per segment), so it stays self-contained: upload
 *   it unchanged and pass both copies to pxf_trace_program_segmented -- still ONE launch.  The op's p[0] (device
 *   table address) is not used; at each LL position every segment is evaluated at the largest order of any segment
 *   there, which gives the same bits as its own order.
 *   Returns PXF_ERR_UNSUPPORTED for an order above 7, a third LL op and PXF_OP_GRATFAN / PXF_OP_ROTX_REMAINING,
 *   PXF_ERR_INVALID for segments that differ in opcode sequence, or for missing tables. */
size_t pxf_segmented_table_bytes_ll(int32_t nops, int32_t nseg);
int pxf_segmented_table_fill_ll(const pxf_op *ops, int32_t nops, int32_t nseg, const int64_t *seg_start,
                                const void *ll_tables_host, void *table_host);

/* ======================= vignetting / compaction ======================== */
/* flags[i] = (l^2+m^2+n^2 > .1), the default predicate of transformations.vignette
 * (transformations.py:220-223; NaN compares false). */
int pxf_vignette_flags(const double *l, const double *m, const double *n, int64_t num,
                       uint8_t *flags, pxf_stream_t stream);
/* Order-preserving stream compaction of nrows arrays by a uint8 flag array (replaces the
 * ten numpy fancy-index copies of transformations.py:225).  Step 1 counts survivors
 * (synchronises, returns the count in *count_host); step 2 scatters.  `scratch` is a device
 * buffer of pxf_compact_scratch_bytes(num) bytes shared by both steps. */
size_t pxf_compact_scratch_bytes(int64_t num);
int pxf_compact_count(const uint8_t *flags, int64_t num, void *scratch, int64_t *count_host,
                      pxf_stream_t stream);
int pxf_compact_scatter(const double *const *rows_in, double *const *rows_out, int32_t nrows,
                        const uint8_t *flags, int64_t num, const void *scratch, pxf_stream_t stream);
/* int64 indices of the surviving rays (np.where(flags)[0]); same scratch as above. */
int pxf_compact_indices(const uint8_t *flags, int64_t num, const void *scratch, int64_t *idx_out,
                        pxf_stream_t stream);

/* ======================= analyses ======================================= */
/* Weighted sums for analyses.centroid / rmsCentroid / analyticImagePlane
 * (analyses.py:16-30,118-133).  w may be NULL (unit weights).  out_dev: device double[16].
 *   PXF_SUMS_CENTROID   : [0]=sum w, [1]=sum w x, [2]=sum w y, [3]=count of rays
 *   PXF_SUMS_RMS        : [0]=sum w, [1]=sum w ((x-cx)^2+(y-cy)^2)        (a=cx, b=cy)
 *   PXF_SUMS_IMAGEPLANE : [0]=sum w, [1]=sum w x, [2]=sum w y, [3]=sum w l/n, [4]=sum w m/n,
 *                         [5]=sum w x l/n, [6]=sum w y m/n, [7]=sum w (l/n)^2, [8]=sum w (m/n)^2
 * Deterministic (fixed-shape tree, no atomics).  scratch: pxf_sums_scratch_bytes() bytes. */
enum { PXF_SUMS_CENTROID = 0, PXF_SUMS_RMS = 1, PXF_SUMS_IMAGEPLANE = 2, PXF_SUMS_IMAGEPLANE_Z = 3,
       PXF_SUMS_POINT = 4 /* internal to pxf_rmspoint: sum w, sum w |r - p|^2 */ };
size_t pxf_sums_scratch_bytes(void);
int pxf_sums(int32_t mode, const double *x, const double *y, const double *l, const double *m,
             const double *n, const double *w, int64_t num, double a, double b,
             double *out_dev, void *scratch, pxf_stream_t stream);

/* The PXF_SUMS_IMAGEPLANE sums taken at the rays' crossing of z = 0, (x - z l/n, y - z m/n): what a literal plane
 * scan (move the plane by dz, trace to it, rmsCentroid -- the legacy findimageplane the reference's examples call,
 * examples/axro/WSverify.py:161-164) needs when the rays are not on z = 0 (e.g. after transform(0,0,dz) without a
 * flat).  analyticImagePlane itself ignores z (analyses.py:122-131) and uses pxf_sums. */
int pxf_sums_z(const double *x, const double *y, const double *z, const double *l, const double *m,
               const double *n, const double *w, int64_t num, double *out_dev, void *scratch, pxf_stream_t stream);

/* rho[i] = sqrt((x-cx)^2+(y-cy)^2)  (analyses.py:60-71) */
int pxf_rho(const double *x, const double *y, int64_t num, double cx, double cy, double *rho_out,
            pxf_stream_t stream);

/* Exact radix select of the two middle order statistics of r = sqrt((x-cx)^2+(y-cy)^2)
 * (keys==NULL) or of keys[i] (keys!=NULL), i.e. np.median in analyses.hpd (analyses.py:96),
 * with DEVICE-RESIDENT state so no pass needs a host round trip and so that a sharded
 * bundle can all-reduce the per-pass histogram between pxf_select_hist and
 * pxf_select_narrow (SURVEY 8e).  `state` is a device buffer of pxf_select_state_bytes()
 * bytes laid out [chain state 48 B][nan count u64][pad][histogram u64 x 2*8192]; the two
 * accessors return device pointers into it (for the collective).
 *   pxf_select_begin   : ranks k0 <= k1 (0-based, over the GLOBAL ray count) to resolve
 *   pxf_select_hist    : add this shard's histogram of digit (key>>shift)&(2^bits-1) for the
 *                        keys that match the prefix of each still-unresolved chain; NaN
 *                        keys are counted separately.  cxy_dev = device double[2] centroid.
 *   pxf_select_narrow  : pick the bin holding each rank, extend the prefixes, clear hist
 *   pxf_select_finish  : out_dev (double[4]): [0] = 2*median (mean of the two order
 *                        statistics; NaN if any key is NaN or num_total == 0 -- numpy
 *                        semantics), [1], [2] = the two order statistics, [3] = 1 unless a
 *                        bracketed select missed (see below)
 *   pxf_select_schedule: digit schedule (shift,bits) of pass `pass`; returns #passes (5). */
size_t pxf_select_state_bytes(void);
int pxf_select_begin(void *state, int64_t k0, int64_t k1, pxf_stream_t stream);
int pxf_select_hist(const double *x, const double *y, const double *keys, int64_t num,
                    const double *cxy_dev, int32_t shift, int32_t bits, void *state,
                    pxf_stream_t stream);
uint64_t *pxf_select_hist_ptr(void *state);
uint64_t *pxf_select_nan_ptr(void *state);
int pxf_select_narrow(int32_t bits, void *state, pxf_stream_t stream);
int pxf_select_finish(void *state, int64_t num_total, double *out_dev, pxf_stream_t stream);
int pxf_select_schedule(int32_t pass, int32_t *shift, int32_t *bits);
/* cxy_dev[0] = sums[1]/sums[0], cxy_dev[1] = sums[2]/sums[0] (np.average) */
int pxf_centroid_from_sums(const double *sums_dev, double *cxy_dev, pxf_stream_t stream);
/* Bracketed select: the median of 1e8 radii without five full passes.  A strided sample of
 * pxf_bracket_samples() radii gives, by an exact select of the sample order statistics
 * pxf_bracket_sample_ranks(), a bracket [lo,hi] around the median; ONE pass
 * (pxf_bracket_collect) counts the radii below lo and appends those inside the bracket to a
 * candidate buffer (capacity pxf_bracket_capacity(num)); the exact select then runs on the
 * candidates (pxf_select_begin_bracket -> pxf_select_hist_keys/narrow x5 -> pxf_select_finish).
 * A miss (rank outside the bracket, buffer overflow) marks the state invalid -- out_dev[3]==0
 * from pxf_select_finish -- and the caller falls back to the five-pass select: the result is
 * exact either way.  counters: device uint64[5] = {#below, #inside, #NaN, #overflowed shards,
 * summed capacities}, zeroed by the caller; a sharded bundle all-reduces them (SURVEY 8e);
 * pxf_select_begin_bracket reads the capacity from counters[4] when cap_total < 0. */
int64_t pxf_bracket_min_num(void);
int32_t pxf_bracket_samples(void);
int64_t pxf_bracket_capacity(int64_t num);
void pxf_bracket_sample_ranks(int32_t nsamp, int64_t *a, int64_t *b);
int pxf_select_sample(const double *x, const double *y, int64_t num, const double *cxy_dev, int32_t nsamp,
                      double *keys_out, pxf_stream_t stream);
int pxf_bracket_collect(const double *x, const double *y, int64_t num, const double *cxy_dev,
                        const double *lohi_dev, double *cand, int64_t cap, uint64_t *counters,
                        pxf_stream_t stream);
int pxf_select_begin_bracket(void *state, int64_t k0, int64_t k1, const uint64_t *counters,
                             int64_t cap_total, pxf_stream_t stream);
int pxf_select_hist_keys(const double *keys, int64_t cap, const uint64_t *count_dev, int32_t shift,
                         int32_t bits, void *state, pxf_stream_t stream);
/* Building blocks of the fused bracketed select for callers that put a collective between them
 * (multi-GPU): sample -> all-gather -> pxf_small_select(npass 3) = bracket -> pxf_bracket_collect ->
 * all-reduce counters -> pxf_cand_hist -> all-reduce the bins -> pxf_cand_scan -> pxf_cand_gather ->
 * all-gather -> pxf_small_select(npass 5, fastsel) = the exact pair.
 * pxf_small_select: ONE-CTA radix select of order statistics ra, rb of nseg x seg_cap keys, the first
 * seg_counts[s] of each segment valid (NULL: all); npass 3 returns a bracket rounded outwards over the
 * 25 unresolved bits, npass 5 the exact values; with `fastsel` the ranks and the valid/NaN verdict come
 * from pxf_cand_scan.  out_dev = {a+b, a, b, valid}. */
/* pack_out[4 + 2*nsamp] = {count, sum x, sum y, count | x, y of nsamp strided rays}: one rank's share of
 * the single all-gather that replaces "all-reduce the centroid sums" + "all-gather the radius sample";
 * pxf_sample_radii turns the gathered packs into the global sums, the centroid and the sample radii. */
int pxf_sample_pack(const double *x, const double *y, int64_t num, const double *sums_dev, int32_t nsamp,
                    double *pack_out, pxf_stream_t stream);
int pxf_sample_radii(const double *gathered, int32_t world, int32_t nsamp, double *sums_out, double *cxy_out,
                     double *keys_out, pxf_stream_t stream);
size_t pxf_fastsel_bytes(void);
int32_t pxf_fast_nbins(void);
int32_t pxf_fast_fincap(void);
int pxf_small_select(const double *keys, const int32_t *seg_counts, int32_t nseg, int32_t seg_cap, int64_t ra,
                     int64_t rb, int32_t npass, const void *fastsel, double *out_dev, pxf_stream_t stream);
int pxf_cand_hist(const double *cand, int64_t cap, const uint64_t *count_dev, const double *lohi_dev,
                  uint32_t *fhist, pxf_stream_t stream);
int pxf_cand_scan(const uint32_t *fhist, const uint64_t *counters, int64_t k0, int64_t k1, void *fastsel,
                  pxf_stream_t stream);
int pxf_cand_gather(const double *cand, int64_t cap, const uint64_t *count_dev, const double *lohi_dev,
                    void *fastsel, double *fin, int32_t *fin_count, pxf_stream_t stream);
/* Unweighted HPD entirely on the device.  out_dev: double[4] = {2*median, lower middle, upper
 * middle, valid}.  mode 0 = automatic (bracketed select for bundles >= pxf_bracket_min_num(),
 * small selects fused into single kernels), 1 = force the five-pass select, 2 = bracketed select
 * through the pass-wise entry points above.  With mode 0/2 the caller checks out_dev[3]: 0 means
 * the bracket missed (probability ~1e-9) and the call must be repeated with mode 1.
 * workspace: pxf_hpd_workspace_bytes(num). */
size_t pxf_hpd_workspace_bytes(int64_t num);
int pxf_hpd_unweighted_dev(const double *x, const double *y, int64_t num, double *out_dev,
                           void *workspace, int32_t mode, pxf_stream_t stream);
/* Same with the centroid sums {count, sum x, sum y} already on the device (sums_dev, e.g. from
 * pxf_trace_program_sums); NULL computes them with one pass over x,y. */
int pxf_hpd_from_sums_dev(const double *x, const double *y, int64_t num, const double *sums_dev,
                          double *out_dev, void *workspace, int32_t mode, pxf_stream_t stream);
/* host-result convenience of the above (synchronises; falls back to the five-pass select itself) */
int pxf_hpd_with_sums(const double *x, const double *y, int64_t num, const double *sums_dev,
                      double *hpd_host, pxf_stream_t stream);
/* ---- per-segment analyses of a segmented bundle -------------------------------------------------
 * The bundle is a concatenation of nseg segments, segment s = rays [seg_start[s], seg_start[s+1]) with
 * seg_start_dev a device int64[nseg+1], seg_start[0] == 0 (the layout of pxf_trace_program_segmented).  Each call
 * does what the single-bundle call does, once per segment, in a number of launches that does not depend on nseg.
 *   pxf_segment_counts : counts_dev[s] = #(flags != 0) in segment s (device int64[nseg]); one pass over the flags.
 *                        The segments of the bundle pxf_compact_scatter makes are the exclusive scan of the counts.
 *   pxf_sums_segmented : the PXF_SUMS_* sums of every segment, out_dev = device double[nseg][16] (entries past the
 *                        mode's count are 0).  z is needed by PXF_SUMS_IMAGEPLANE_Z / PXF_SUMS_POINT; ab_dev is the
 *                        per-segment centre, double[nseg][2] for PXF_SUMS_RMS, (px,py,pz) double[nseg][3] for
 *                        PXF_SUMS_POINT.  The per-ray arithmetic is that of pxf_sums; each segment's sums are
 *                        folded in a fixed order (same bits on every run for the same bundle and layout, no
 *                        floating-point atomics).  scratch: pxf_sums_segmented_scratch_bytes(num, nseg).
 *   pxf_centroids_segmented : cxy_dev[s] = {sums[s][1] / sums[s][0], sums[s][2] / sums[s][0]}.
 *   pxf_hpd_segmented  : analyses.hpd (analyses.py:88-97) of every segment, out_dev = device double[nseg][4] =
 *                        {HPD, lower, upper, valid}.  sums_dev = pxf_sums_segmented(PXF_SUMS_CENTROID) output (with
 *                        the same weights); radii are taken about exactly that centroid.
 *                        Unweighted (w == NULL): 2*median of the radii (np.median: mean of the two middle values,
 *                        NaN if the segment is empty or has a NaN radius); lower/upper = the middle order statistics.
 *                        Segments of up to 8192 rays are sorted in shared memory; larger ones are bracketed from a
 *                        strided sample, ONE pass over the bundle collects the radii inside every bracket and the
 *                        exact pair is selected among them.  valid == 0 flags a segment whose bracket missed or whose
 *                        candidates overflowed: resolve it with pxf_hpd_from_sums_dev(mode 1) on its slice.
 *                        mode 1 runs that five-pass select for every segment (reads seg_start back; for tests).
 *                        Weighted: r[argmin|cdf-.75|] - r[argmin|cdf-.25|] with the cdf taken within the segment
 *                        (stable sort by (segment, radius), cumulative weights restarted per segment, first
 *                        minimisers); upper/lower = r75/r25.  A segment with no rays or zero total weight gives NaN.
 *                        workspace: pxf_hpd_segmented_workspace_bytes(num, nseg, w != NULL). */
int pxf_segment_counts(const uint8_t *flags, int64_t num, const int64_t *seg_start_dev, int32_t nseg,
                       int64_t *counts_dev, pxf_stream_t stream);
size_t pxf_sums_segmented_scratch_bytes(int64_t num, int32_t nseg);
int pxf_sums_segmented(int32_t mode, const double *x, const double *y, const double *z, const double *l,
                       const double *m, const double *n, const double *w, int64_t num, const int64_t *seg_start_dev,
                       int32_t nseg, const double *ab_dev, double *out_dev, void *scratch, pxf_stream_t stream);
int pxf_centroids_segmented(const double *sums_dev, int32_t nseg, double *cxy_dev, pxf_stream_t stream);
size_t pxf_hpd_segmented_workspace_bytes(int64_t num, int32_t nseg, int32_t weighted);
int pxf_hpd_segmented(const double *x, const double *y, const double *w, int64_t num, const int64_t *seg_start_dev,
                      int32_t nseg, const double *sums_dev, double *out_dev, void *workspace, int32_t mode,
                      pxf_stream_t stream);
/* rows_out[r][i] = rows_in[r][idx[i]] for nrows <= 16 rows (vignette with an index array,
 * transformations.py:225).  rows_in/rows_out are HOST arrays of device pointers;
 * table_scratch: >= 256 B device. */
int pxf_gather_rows(const double *const *rows_in, double *const *rows_out, int32_t nrows,
                    const int64_t *idx, int64_t count, void *table_scratch, pxf_stream_t stream);

/* Convenience, single GPU: analyses.hpd / rmsCentroid / centroid / analyticImagePlane end to
 * end, result in host memory (synchronises).  weights may be NULL.
 *   pxf_hpd unweighted: 2*median(r) (exact order statistics; mean of the two middle values for
 *   even num, NaN if any r is NaN -- numpy semantics).  Weighted: radix sort by r, cumulative
 *   weights, r[argmin|cdf-.75|]-r[argmin|cdf-.25|] (analyses.py:91-94). */
int pxf_centroid(const double *x, const double *y, const double *w, int64_t num,
                 double *cx_host, double *cy_host, pxf_stream_t stream);
int pxf_rmscentroid(const double *x, const double *y, const double *w, int64_t num,
                    double *rms_host, pxf_stream_t stream);
int pxf_hpd(const double *x, const double *y, const double *w, int64_t num, double *hpd_host,
            pxf_stream_t stream);
/* analyses.rmsPoint (analyses.py:33-45): sqrt(average((x-px)^2+(y-py)^2+(z-pz)^2, weights)); w may be NULL. */
int pxf_rmspoint(const double *x, const double *y, const double *z, const double *w, int64_t num,
                 double px, double py, double pz, double *rms_host, pxf_stream_t stream);
int pxf_analyticimageplane(const double *x, const double *y, const double *l, const double *m,
                           const double *n, const double *w, int64_t num, double *dz_host,
                           pxf_stream_t stream);

/* Weighted HPD (analyses.py:88-97, weighted branch).  pxf_hpd_weighted = what pxf_hpd calls when
 * w != NULL: the bracketed path for num >= pxf_wq_min_num(), the full sort otherwise or when the
 * bracketed path reports valid == 0 (bracket miss, candidate overflow, NaN radius, NaN/negative
 * weight).  pxf_hpd_weighted_sorted is the literal argsort -> cumsum -> argmin pipeline.
 * The pxf_wq_* pieces are the steps of the bracketed path (also used by the sharded driver):
 *   pxf_wq_sample    strided sample of (radius about cxy_dev, weight) pairs
 *   pxf_wq_brackets  sorted sample + prefix weights -> closed brackets around the .25 / .75 crossings
 *                    (state: pxf_wq_state_bytes(), layout double lohi[4], below[2], u64 count[2], nbad)
 *   pxf_wq_collect   one pass: weight strictly below each bracket (deterministic tree) and the
 *                    (radius, weight) pairs inside, appended to cand_r/w{0,1} (capacity cap each)
 *   pxf_wq_argmin    argmin |(below + cum[i]) / total - q| inside a sorted window;
 *                    out_dev[4] = {r, valid, cdf, index} */
int pxf_hpd_weighted(const double *x, const double *y, const double *w, int64_t num, double *hpd_host,
                     pxf_stream_t stream);
int pxf_hpd_weighted_sorted(const double *x, const double *y, const double *w, int64_t num, double *hpd_host,
                            pxf_stream_t stream);
int pxf_hpd_weighted_bracket(const double *x, const double *y, const double *w, int64_t num, double *hpd_host,
                             int32_t *valid_host, pxf_stream_t stream);
size_t pxf_wq_state_bytes(void);
int64_t pxf_wq_min_num(void);
int32_t pxf_wq_samples(int64_t num);
int64_t pxf_wq_capacity(int64_t num);
int pxf_wq_sample(const double *x, const double *y, const double *w, int64_t num, const double *cxy_dev,
                  int32_t nsamp, double *rs_out, double *ws_out, pxf_stream_t stream);
/* keybits: the sample is ordered by the top `keybits` bits of the radius patterns (64 = fully sorted; the
 * single-GPU driver sorts the sample on 32); the brackets are widened by the unordered low bits. */
int pxf_wq_brackets(const double *rs_sorted, const double *cum, int32_t nsamp, int32_t keybits, void *state,
                    pxf_stream_t stream);
size_t pxf_wq_collect_scratch_bytes(void);
int pxf_wq_collect(const double *x, const double *y, const double *w, int64_t num, const double *cxy_dev, void *state,
                   double *cand_r0, double *cand_w0, double *cand_r1, double *cand_w1, int64_t cap, void *scratch,
                   pxf_stream_t stream);
double *pxf_wq_below_ptr(void *state, int32_t b);
size_t pxf_wq_argmin_scratch_bytes(void);
int pxf_wq_argmin(const double *rs_sorted, const double *cum, int64_t n, const double *below_dev, const double *total_dev,
                  double q, double *out_dev, void *scratch, pxf_stream_t stream);
/* Sharded merge of sorted runs (two quantiles at once): each rank holds per quantile a sorted run of radius
 * patterns (int64) with prefix weights.  state (pxf_wq_merge_state_bytes): int64 lo[2], hi[2], klo[2];
 * double res[2], valid[2].  Per step: probe (this rank's weight at or below each of K pivots of [lo,hi] ->
 * out_dev[2*K]), the caller all-reduces out_dev (sum), narrow (shrinks [lo,hi] by K+1).  When lo == hi:
 * final_probe (out_dev[4] = weight at or below / strictly below hi per quantile; klo = largest local key
 * below hi), the caller all-reduces out_dev (sum) and klo (max), finish -> res[i] = r[argmin|cdf-q_i|],
 * valid[i].  offsets_dev (nullable): weight below the runs; total_dev: total weight. */
size_t pxf_wq_merge_state_bytes(void);
int64_t *pxf_wq_merge_klo_ptr(void *state);
double *pxf_wq_merge_result_ptr(void *state);
int pxf_wq_merge_begin(void *state, int64_t lo0, int64_t hi0, int64_t lo1, int64_t hi1, pxf_stream_t stream);
int pxf_wq_merge_probe(const int64_t *keys0, const double *cum0, int64_t n0, const int64_t *keys1, const double *cum1,
                       int64_t n1, const void *state, int32_t K, double *out_dev, pxf_stream_t stream);
int pxf_wq_merge_narrow(void *state, const double *sum_dev, const double *offsets_dev, const double *total_dev,
                        double q0, double q1, int32_t K, pxf_stream_t stream);
int pxf_wq_merge_final_probe(const int64_t *keys0, const double *cum0, int64_t n0, const int64_t *keys1,
                             const double *cum1, int64_t n1, void *state, double *out_dev, pxf_stream_t stream);
int pxf_wq_merge_finish(void *state, const double *sum_dev, const double *offsets_dev, const double *total_dev,
                        double q0, double q1, pxf_stream_t stream);

/* Stable LSD radix sort of fp64 keys with the permutation: np.argsort(keys, kind='stable') and np.sort (analyses.py:76).
 * Order: -inf < ... < -0 == +0 < ... < +inf < NaN; keys that compare equal (ties, -0/+0, all NaNs) keep their input
 * order, and the sorted keys carry the original bit patterns.  One-sweep passes (one kernel per non-constant key
 * byte, decoupled look-back); nothing is read back, the call is asynchronous on `stream`.  keys_out / idx_out:
 * device arrays of length num (either may be NULL); keys_out must not alias keys_in.
 * scratch: pxf_sort_scratch_bytes(num). */
size_t pxf_sort_scratch_bytes(int64_t num);
int pxf_argsort(const double *keys_in, int64_t num, double *keys_out, int64_t *idx_out,
                void *scratch, pxf_stream_t stream);
/* Same, sorting only on the bytes of the 64-bit key whose bit is set in `digits` (bit 0 = least significant
 * byte); 0 = skip the bytes that are constant over the array (decided on the device; what pxf_argsort does).
 * A mask is for keys from a known narrow range, or when a partial order is enough. */
int pxf_argsort_digits(const double *keys_in, int64_t num, double *keys_out, int64_t *idx_out,
                       void *scratch, int32_t digits, pxf_stream_t stream);
/* out[i] = inclusive prefix sum of (w ? w[idx[i]] : 1.0)  (np.cumsum(weights[ind]),
 * analyses.py:83-85).  scratch: pxf_scan_scratch_bytes(num). */
size_t pxf_scan_scratch_bytes(int64_t num);
int pxf_cumsum_gather(const double *w, const int64_t *idx, int64_t num, double *out,
                      void *scratch, pxf_stream_t stream);

/* ======================= reconstruct (SURVEY 8f rank 4) ================= */
/* reconstruct.f95:1-128  reconstruct(xang,yang,xdim,ydim,criteria,h,phase,phasec,maxiter): Southwell successive
 * over-relaxation in the reference's lexicographic Gauss-Seidel order, run as a diagonal-parity pipeline
 * (bit-identical, see pxf_reconstruct.cu).  Arrays: device, column-major [xdim][ydim], 100. = invalid lenslet;
 * xang, yang, phase are updated in place like the Fortran intent(inout) arguments, phasec receives the result.
 * *sweeps_host (nullable) = sweeps executed.  Synchronises the stream. */
int pxf_reconstruct(double *xang, double *yang, int32_t xdim, int32_t ydim, double criteria, double h, double *phase,
                    double *phasec, int32_t maxiter, int64_t *sweeps_host, pxf_stream_t stream);
/* reconstruct.f95:136-187  southwellbin(x,y,l,m,num,binsize,xang,yang,phase,xdim,ydim): mean direction cosines of
 * the rays in each lenslet -> slopes tan(asin(.)), 100. for empty lenslets.  Per-lenslet sums are taken in ray
 * order (stable sort by cell, one thread per cell), i.e. the single-thread semantics of the reference loop.
 * scratch: pxf_southwellbin_scratch_bytes(num, xdim, ydim). */
size_t pxf_southwellbin_scratch_bytes(int64_t num, int32_t xdim, int32_t ydim);
int pxf_southwellbin(const double *x, const double *y, const double *l, const double *m, int64_t num, double binsize,
                     double *xang, double *yang, double *phase, int32_t xdim, int32_t ydim, void *scratch,
                     pxf_stream_t stream);

/* ======================= scattered-data interpolation =================== */
/* scipy.interpolate.griddata((x, y), v, (qx, qy), method) as analyses.interpolateVec / wavefront call it
 * (analyses.py:189-230, 305-334; scipy is a third-party dependency of the reference).  method 0 = 'nearest', 1 = 'linear'
 * (barycentric interpolation inside the Delaunay triangle that contains the query; NaN outside the convex hull), 2 =
 * 'cubic' (scipy's CloughTocher2DInterpolator: Gauss-Seidel vertex gradients in input order to 1e-6, reproduced sweep for
 * sweep by level scheduling, then the Clough-Tocher patch of the containing triangle).  The triangle is found by pivoting
 * to the empty circumcircle over a uniform cell grid; no global triangulation is built.  All arrays on the device; out[nq].  *nfail_host (may be NULL; reading it synchronises)
 * receives the number of queries whose cell could not be resolved (degenerate input; they are NaN).
 * scratch: pxf_griddata_scratch_bytes(num) -- about 300 bytes per point (cell-ordered copies, sort scratch and, for 'cubic',
 * 48 neighbour slots, the level order and the gradient of every point). */
size_t pxf_griddata_scratch_bytes(int64_t num);
int pxf_griddata(const double *x, const double *y, const double *v, int64_t num, const double *qx, const double *qy,
                 double *out, int64_t nq, int32_t method, int64_t *nfail_host, void *scratch, pxf_stream_t stream);

/* The Delaunay neighbours of every point, counter-clockwise (the structure scipy's 'cubic' griddata takes its vertex
 * gradients over; gift wrapping about each point over the same cell grid, no triangulation stored).  ring_out:
 * device int32 [num][pxf_delaunay_max_degree()], unused slots -1; deg_out, open_out: device uint8 [num] (open = 1: a hull
 * vertex, its ring is the chain from the clockwise to the counter-clockwise hull neighbour).  scratch:
 * pxf_griddata_scratch_bytes(num). */
int pxf_delaunay_max_degree(void);
int pxf_delaunay_neighbors(const double *x, const double *y, int64_t num, int32_t *ring_out, uint8_t *deg_out,
                           uint8_t *open_out, void *scratch, pxf_stream_t stream);
/* Helpers of analyses.interpolateVec: the bounding box of the ray positions (xr = [x.min(), x.max()], analyses.py:206-208;
 * box_host[4] = xmin, xmax, ymin, ymax; scratch: pxf_bbox_scratch_bytes()), the polar coordinates of its polar=True
 * branch (rho, rho*arctan2(y,x), rho*arctan2(x,y); analyses.py:219-226) and np.nanmedian of two arrays (:227). */
size_t pxf_bbox_scratch_bytes(void);
int pxf_bbox(const double *x, const double *y, int64_t num, double *box_host, void *scratch, pxf_stream_t stream);
int pxf_polar_coords(const double *x, const double *y, int64_t num, double *rho, double *az1, double *az2, pxf_stream_t stream);
int pxf_nanmedian2(const double *a, const double *b, int64_t num, double *out, pxf_stream_t stream);

/* ======================= sources ======================================== */
/* Device-side ray generation for bundles too large for host MT19937 (SURVEY 7 "RNG parity").
 * Counter-based Philox4x32-10, key=(seed lo,hi), counter=(global ray index, stream id);
 * u1,u2 are 53-bit uniforms built as numpy does ((a>>5)*2^26+(b>>6))/2^53.  Same formulas as
 * sources.py:130-170 / :56-88 / :20-53 / :91-127.  `first` is the global index of ray 0 of
 * this shard so that sharded generation reproduces the single-GPU stream.
 * kind: 0=subannulus(a=rin,b=rout,c=dphi,d=zhat) 1=circularbeam(a=rad) 2=pointsource(a=ang)
 *       3=annulus(a=rin,b=rout,d=zhat) */
int pxf_source(int32_t kind, double *const rays[10], int64_t num, int64_t first, uint64_t seed,
               double a, double b, double c, double d, pxf_stream_t stream);
/* The same formulas applied to caller-supplied uniforms u1,u2 (device arrays, e.g. uploaded
 * from numpy's legacy MT19937 for bit-identical seeds). */
int pxf_source_from_uniform(int32_t kind, double *const rays[10], int64_t num, const double *u1,
                            const double *u2, double a, double b, double c, double d,
                            pxf_stream_t stream);
/* One launch for a nested assembly: segment s of the bundle is drawn from source `kind` (0 subannulus,
 * 1 circularbeam, 3 annulus) with params_dev[4*s..4*s+3] = (a,b,c,d); seg_start_dev: device int64[nseg+1].
 * Same Philox stream as per-segment pxf_source calls with first + seg_start[s]. */
int pxf_source_segmented(int32_t kind, double *const rays[10], int64_t num, int64_t first, uint64_t seed,
                         int32_t nseg, const int64_t *seg_start_dev, const double *params_dev, pxf_stream_t stream);

/* The reference's set-up sources (sources.py:173-471), generated on the device.
 * Grid sources are functions of the global ray index first+i alone (numpy.linspace / meshgrid arithmetic restated:
 * i*step + start, last point pinned to stop; meshgrid flattened row-major):
 *   PXF_SRC_XSLIT     (sources.py:173-207)  a=xin b=xout c=zhat, n1 = num
 *   PXF_SRC_RECTARRAY (sources.py:210-247)  a=xsize b=ysize,     n1 = num (n1*n1 rays)
 *   PXF_SRC_FANBEAM   (sources.py:418-442)  a=xang b=yang,       n1 = num (n1*n1 rays)
 *   PXF_SRC_CIRCFAN   (sources.py:444-471)  a=halfang,           n1 = rings, n2 = arms (n1*n2 rays)
 * `num` rays starting at global index `first` are written (a shard of the source). */
enum { PXF_SRC_XSLIT = 4, PXF_SRC_RECTARRAY = 5, PXF_SRC_CONVERGING = 6, PXF_SRC_CONVERGING2 = 7, PXF_SRC_RECTBEAM = 8,
       PXF_SRC_GAUSSIAN = 9, PXF_SRC_FANBEAM = 10, PXF_SRC_CIRCFAN = 11 };
int pxf_source_grid(int32_t kind, double *const rays[10], int64_t num, int64_t first, int64_t n1, int64_t n2,
                    double a, double b, double c, pxf_stream_t stream);
/* Beam sources: two or three random draws per ray.
 *   PXF_SRC_CONVERGING  (sources.py:250-296) par = (zset, rin, rout, tmin, tmax, lscat); draws: radius, angle, scatter
 *   PXF_SRC_CONVERGING2 (sources.py:299-345) par = (zset, xmin, xmax, ymin, ymax, lscat); draws: x, y, scatter
 *   PXF_SRC_RECTBEAM    (sources.py:348-379) par = (xhalfwidth, yhalfwidth);             draws: x, y
 *   PXF_SRC_GAUSSIAN    (sources.py:381-416) par = (ang);                                draws: two standard normals
 * pxf_source_beam draws on the device (Philox4x32-10 keyed like pxf_source; block 1 of a ray's counter feeds the
 * third draw, the normals are a Box-Muller pair); pxf_source_beam_from_draws applies the same formulas to
 * caller-supplied device arrays (numpy's stream in the reference's order of draws; d3 may be NULL for two-draw
 * kinds).  par is a HOST array. */
int pxf_source_beam(int32_t kind, double *const rays[10], int64_t num, int64_t first, uint64_t seed,
                    const double *par, pxf_stream_t stream);
int pxf_source_beam_from_draws(int32_t kind, double *const rays[10], int64_t num, const double *d1, const double *d2,
                               const double *d3, const double *par, pxf_stream_t stream);

/* ======================= host-buffer entry point ======================== */
/* The call an f2py user makes (the reference's extension modules take HOST numpy arrays and
 * mutate them in place, e.g. transformations.py:29, surfaces.py:224): HOST rows in, HOST rows
 * mutated in place, a whole op list per call.  The bundle streams through the device in chunks
 * on three internal streams (H2D of chunk c+1, fused program on chunk c, D2H of chunk c-1
 * overlap).  Only rows the program reads are uploaded, only rows it may write are downloaded;
 * rows_host[k] may be NULL for rows it touches neither way.  Pinned (page-locked) host rows
 * get full PCIe rate; pageable rows work but are staged by the driver.
 *   write_back       0 skips the D2H of the ray rows (analysis-only callers)
 *   hpd_host         nullable; receives the unweighted HPD (analyses.py:88-97) of the final
 *                    bundle -- of the surviving rays when the program has VIGNETTE ops
 *   alive_host       nullable uint8[num]; receives the survivor flags of VIGNETTE ops
 *   alive_count_host nullable; number of surviving rays (-1 if it was not computed because
 *                    neither hpd_host nor alive_host was given)
 *   x_dev_keep/y_dev_keep  nullable pair of caller-owned DEVICE rows (num doubles, 16-byte
 *                    aligned): the final x,y stay resident there for follow-up analyses (a
 *                    sharded bundle's global HPD, SURVEY.md 8e)
 * Synchronous: returns when every host row is final. */
int pxf_host_trace_program(double *const rows_host[10], int64_t num, const pxf_op *ops, int32_t nops,
                           int32_t write_back, double *hpd_host, uint8_t *alive_host,
                           int64_t *alive_count_host, double *x_dev_keep, double *y_dev_keep);
/* The same with a caller hint: const_rows_mask bit r set = the caller vouches that every entry of input row r
 * equals its first (z, l, m, n of every PyXFocus source, sources.py:20-170) -- the row is then filled on the device
 * without being scanned or uploaded.  Rows not vouched for are still scanned chunk by chunk. */
int pxf_host_trace_program_hint(double *const rows_host[10], int64_t num, const pxf_op *ops, int32_t nops,
                                int32_t write_back, double *hpd_host, uint8_t *alive_host,
                                int64_t *alive_count_host, double *x_dev_keep, double *y_dev_keep,
                                uint32_t const_rows_mask);
/* Frees the streams / device buffers the host entry point caches between calls. */
void pxf_host_release(void);

#ifdef __cplusplus
}
#endif
#endif /* PXF_H */
