// Host-side folding of the scalar arguments of each routine into the *P structs the
// device code consumes.  Every expression keeps the Fortran's evaluation order and is
// evaluated with the host libm, so the folded constants are the values the reference
// (and the CPU oracle) compute once per call or once per ray from the same scalars.
// Compiled with -ffp-contract=off.
#pragma once
#include <math.h>
#include <string.h>
#include "pxf_ray.cuh"
#include "pxf_internal.h"

namespace pxf {

inline double h_sq(double a) { return a * a; }
inline double h_pow4(double a) { double t = a * a; return t * t; }
inline double h_pi32() { return (double)acosf(-1.0f); }   // REAL*4 acos(-1.)
inline double h_tol8() { return (double)1.e-8f; }
inline double h_tol10() { return (double)1.e-10f; }

// transformationsf.f95:134-163: rotatevector(…,rx,1) etc.
inline TransformP make_transform(double tx, double ty, double tz, double rx, double ry, double rz)
{
    TransformP p;
    p.tx = tx; p.ty = ty; p.tz = tz;
    p.cx = cos(rx); p.sx = sin(rx);
    p.cy = cos(ry); p.sy = sin(ry);
    p.cz = cos(rz); p.sz = sin(rz);
    p.groups = 7;
    p.ident = ((p.cx == 1. && p.sx == 0.) ? 1 : 0) | ((p.cy == 1. && p.sy == 0.) ? 2 : 0) | ((p.cz == 1. && p.sz == 0.) ? 4 : 0);
    return p;
}
// transformationsf.f95:168-201: tmp = -rz; rotatevector(…,tmp,3) …
inline TransformP make_itransform(double tx, double ty, double tz, double rx, double ry, double rz)
{
    return make_transform(tx, ty, tz, -rx, -ry, -rz);
}

// woltsurf.f95:18-25
inline void vanspeybroeck(double r0, double z0, double psi, double &p, double &d, double &e)
{
    double alpha = .25 * atan(r0 / z0);
    double thetah = 2 * (1 + 2 * psi) / (1 + psi) * alpha;
    double thetap = 2 * psi / (1 + psi) * alpha;
    p = z0 * tan(4 * alpha) * tan(thetap);
    d = z0 * tan(4 * alpha) * tan(4 * alpha - thetah);
    e = cos(4 * alpha) * (1 + tan(4 * alpha) * tan(thetah));
}

inline WolterP make_wolter(double r0, double z0, double psi, bool opd, double nr)
{
    double p, d, e;
    vanspeybroeck(r0, z0, psi, p, d, e);
    WolterP w;
    w.twop = 2 * p;
    w.p2 = h_sq(p);
    w.c1 = 4 * h_sq(e) * p * d / (h_sq(e) - 1);
    w.e2 = h_sq(e);
    w.two_e2 = 2 * h_sq(e);
    w.d = d;
    w.tol = opd ? h_tol10() : h_tol8();
    w.nr = nr;
    w.opd = opd ? 1 : 0;
    return w;
}

// woltsurf.f95:178-183 (psi fixed: thetah = 3.*alpha, thetap = alpha)
inline WolterSineP make_woltersine(double r0, double z0, double amp, double freq)
{
    double alpha = .25 * atan(r0 / z0);
    double thetah = 3. * alpha;
    double thetap = alpha;
    double p = z0 * tan(4 * alpha) * tan(thetap);
    double d = z0 * tan(4 * alpha) * tan(4 * alpha - thetah);
    double e = cos(4 * alpha) * (1 + tan(4 * alpha) * tan(thetah));
    WolterSineP w;
    w.twop = 2 * p;            // also 2.*p at :194
    w.p2 = h_sq(p);
    w.c1 = 4 * h_sq(e) * p * d / (h_sq(e) - 1);
    w.amp = amp;
    w.freq = freq;
    w.twopi32 = (double)(2 * acosf(-1.0f));
    w.pi32 = h_pi32();
    w.tol = h_tol10();
    return w;
}

inline WSP make_ws(double alpha, double z0, double psi, double thick = 0.)
{
    WSP p;
    memset(&p, 0, sizeof(p));
    p.thick = thick;
    p.betas = 4 * alpha;
    p.ff = z0 / cos(p.betas);
    p.g = p.ff / psi;
    p.k = h_sq(tan(p.betas / 2));
    p.tol = h_tol8();
    const double betas = p.betas, ff = p.ff, g = p.g, k = p.k;
    p.invk = 1 / k;
    p.omk = 1 - k;
    p.opk = 1 + k;
    p.ff2 = h_sq(ff);
    const double sh2 = h_sq(sin(betas / 2));
    p.A0 = ff * sh2;
    p.denF = 4 * ff * sh2;
    p.denFb = 2 * ff * sh2;
    p.twog = 2 * g;
    p.gomk = g * (1 - k);
    p.Cs = h_sq(ff) * h_sq(sin(betas)) / (4 * ff * sh2);
    p.Ds = g * h_pow4(cos(betas / 2)) * pow(0., 1 - k);
    p.FbS = h_sq(ff) * sin(betas) * cos(betas) / (2 * ff * sh2) +
            g * (1 - k) * cos(betas / 2) * sin(betas / 2) * (1 / k);
    p.ffsinbs = ff * sin(betas);
    p.a_s = 1 / ff;
    p.F0s = cos(betas) / p.a_s;
    p.omcbs = 1 - cos(betas);
    p.sinbs2 = h_sq(sin(betas));
    double dadbs = sin(betas) / ff / (1 - cos(betas)) +
                   (k + 1) * (cos(betas) + 1) * tan(betas / 2) / h_sq(cos(betas / 2)) / 2 / g / k;
    p.gamA = -ff * sin(betas) - h_sq(ff) * cos(betas) * dadbs;
    p.tanbs = tan(betas);
    p.twootan = 2. / tan(betas);
    p.kp1 = k + 1;
    p.fast = (!opt_ws_libm() && k > 0. && k < .25) ? 1. : 0.;
    p.retrace = (double)opt_ws_retrace();
    p.graze_min = 1.e-6 * (double)opt_ws_graze_ppm();
    p.tanhbs = tan(betas / 2);
    p.iff = 1 / ff;
    p.idenF = 1 / p.denF;
    p.idenFb = 1 / p.denFb;
    p.c1 = 1 / (p.omcbs * ff);
    p.c2 = 1 / p.twog;
    p.c3 = p.kp1 / g / k;
    return p;
}

// ---- surfacesf.f95: remaining surfaces
inline SphereP make_sphere(double rad, bool opd, double nr)
{
    SphereP p;
    p.rad2 = h_sq(rad); p.nr = nr; p.opd = opd ? 1 : 0; p.pad = 0;
    return p;
}
inline CylConicP make_cylconic(double rad, double k)
{
    CylConicP p;
    p.A = (1 + k) * h_sq(rad);
    p.rad = rad;
    p.tworad = 2 * rad;
    p.tol = h_tol10();
    return p;
}
inline TorusP make_torus(double rin, double rout)
{
    TorusP p;
    p.rin = rin; p.rout = rout;
    p.rin2 = h_sq(rin); p.rout2 = h_sq(rout);
    p.four_rout2 = 4 * h_sq(rout);
    p.tworin = 2 * rin; p.tworout = 2 * rout;
    p.rpr = rin + rout;
    p.tol = h_tol10();
    return p;
}
inline int make_conicplus(ConicPlusP &q, double R, double K, const double *p, int np, bool opd, double nr)
{
    if (np < 0 || np > PXF_CONICPLUS_MAXP) return -1;
    memset(&q, 0, sizeof(q));
    q.c = 1 / R;
    q.twoc = 2 * q.c;
    q.c3 = (q.c * q.c) * q.c;
    q.Kp1 = K + 1;
    q.Kp1c2 = (K + 1) * h_sq(q.c);
    q.nr = nr; q.tol = h_tol10(); q.np = np; q.opd = opd ? 1 : 0;
    for (int j = 0; j < np; j++) q.p[j] = p[j];
    return 0;
}
inline double h_factorial(int n)
{
    double f = 1.;
    for (int i = 2; i <= n; i++) f = f * (double)i;
    return f;
}
inline int make_legsurf(LegSurfP &q, double xwidth, double ywidth, double order, const double *coeff,
                        const int32_t *xo, const int32_t *yo, int nc)
{
    if (nc < 0 || nc > PXF_LEGSURF_MAXC) return -1;
    memset(&q, 0, sizeof(q));
    q.xwidth = xwidth; q.ywidth = ywidth; q.order = order; q.nc = nc;
    for (int j = 0; j < nc; j++) {
        if (xo[j] < 0 || xo[j] > PXF_LEGSURF_MAXN || yo[j] < 0 || yo[j] > PXF_LEGSURF_MAXN) return -1;
        q.coeff[j] = coeff[j]; q.xo[j] = xo[j]; q.yo[j] = yo[j];
    }
    // specialFunctions.f95:337-388: (-1)**i*f(2n-2i)/f(i)/f(n-i)/f(n-2i)/2**n [*(n-2i)], 2**n INTEGER
    for (int n = 0; n <= PXF_LEGSURF_MAXN; n++)
        for (int i = 0; i <= n / 2; i++) {
            const double sign = (i % 2) ? -1. : 1.;
            const double c = sign * h_factorial(2 * n - 2 * i) / h_factorial(i) / h_factorial(n - i) /
                             h_factorial(n - 2 * i) / (double)(1 << n);
            q.lc[n][i] = c;
            q.lpc[n][i] = c * (double)(n - 2 * i);
        }
    return 0;
}

inline SpoP make_spo(double R0, double tg)
{
    SpoP p;
    p.R0 = R0;
    p.sl = tan(tg);
    p.sl2 = h_sq(p.sl);
    p.R02 = h_sq(R0);
    p.twoslR0 = 2 * p.sl * R0;
    p.ctg = cos(tg);
    p.stg = sin(tg);
    return p;
}

inline ConicP make_conic(double R, double K, bool opd, double nr)
{
    ConicP p;
    p.R = R; p.K = K;
    p.Kp1 = K + 1;
    p.twoR = 2 * R;
    p.R2 = h_sq(R);
    p.sgnR = -R / fabs(R);
    p.nr = nr;
    p.kis_m1 = (K == -1) ? 1 : 0;
    p.opd = opd ? 1 : 0;
    return p;
}

inline RadgratP make_radgrat(double wave, double dpermm, double order)
{
    RadgratP p;
    p.neg_half_pi32 = -h_pi32() / 2;
    p.dpermm = dpermm; p.order = order; p.wave = wave;
    return p;
}

inline double h_tol7() { return (double)1.e-7f; }

// Legendre-Legendre shells: fold the (coeff, axial, az) term list into the dense matrix of
// pxf_ray.cuh.  kind 0/1/2 = wolterprimLL / woltersecLL / ellipsoidWoltLL; S only for kind 2.
// Returns 0, or -1 for an invalid table (orders outside 0..15).
inline int make_ll(LLP &q, int kind, double r0, double z0, double psi, double S, double zmax, double zmin,
                   double dphi, const double *coeff, const int32_t *axial, const int32_t *az, int cnum)
{
    memset(&q, 0, sizeof(q));
    LLS &s = q.s;
    s.kind = kind;
    int nz = 0, nt = 0;
    for (int a = 0; a < cnum; a++) {
        if (axial[a] < 0 || axial[a] > PXF_LL_MAXN || az[a] < 0 || az[a] > PXF_LL_MAXN) return -1;
        if (axial[a] > nz) nz = axial[a];
        if (az[a] > nt) nt = az[a];
    }
    s.nz = nz; s.nt = nt;
    const int top = nz > nt ? nz : nt;
    const int N = top <= 3 ? 3 : top <= 5 ? 5 : top <= 7 ? 7 : top <= 11 ? 11 : 15;
    s.stride = N + 1;
    // power-basis coefficients of P_0..P_15 from (n+1) P_{n+1} = (2n+1) x P_n - n P_{n-1} (dyadic rationals with
    // numerators < 2**53: exact), then  M[a][b] = sum_t coeff_t * L[axial_t][a] * L[az_t][b]  accumulated in long double
    static long double L[PXF_LL_MAXN + 1][PXF_LL_MAXN + 1];
    static bool have_L = false;
    if (!have_L) {
        memset(L, 0, sizeof(L));
        L[0][0] = 1.L; L[1][1] = 1.L;
        for (int n = 1; n < PXF_LL_MAXN; n++)
            for (int k = 0; k <= n + 1; k++)
                L[n + 1][k] = ((2 * n + 1) * (k ? L[n][k - 1] : 0.L) - n * L[n - 1][k]) / (n + 1);
        have_L = true;
    }
    long double M[PXF_LL_MAXN + 1][PXF_LL_MAXN + 1];
    memset(M, 0, sizeof(M));
    for (int t = 0; t < cnum; t++)
        for (int a = 0; a <= axial[t]; a++)
            for (int b = 0; b <= az[t]; b++) M[a][b] += (long double)coeff[t] * L[axial[t]][a] * L[az[t]][b];
    for (int a = 0; a <= N; a++)
        for (int b = 0; b <= N; b++) q.C[a * s.stride + b] = (double)M[a][b];
    s.zmid = (zmax + zmin) / 2.;
    s.zhalf = (zmax - zmin) / 2.;
    s.dphi = dphi;
    s.twoodphi = 2 / dphi;
    s.zrange = zmax - zmin;
    s.izhalf = 1 / s.zhalf;
    s.twoozrange = 2 / s.zrange;
    if (kind == 0) {            // woltsurf.f95:235-241: thetah = 3.*alpha, thetap = alpha
        double alpha = .25 * atan(r0 / z0);
        double thetah = 3. * alpha, thetap = alpha;
        double p = z0 * tan(4 * alpha) * tan(thetap);
        double d = z0 * tan(4 * alpha) * tan(4 * alpha - thetah);
        double e = cos(4 * alpha) * (1 + tan(4 * alpha) * tan(thetah));
        s.g0 = h_sq(p); s.g1 = 2 * p; s.g2 = 4 * h_sq(e) * p * d / (h_sq(e) - 1);
        s.tol = h_tol10();
    } else if (kind == 1) {     // woltsurf.f95:307-312, tol 1.e-7 (:319)
        double p, d, e;
        vanspeybroeck(r0, z0, psi, p, d, e);
        s.g0 = h_sq(e); s.g1 = 2 * h_sq(e); s.g2 = d;
        s.tol = h_tol7();
    } else {                    // woltsurf.f95:657-666
        double P = r0 / sin((psi * asin(r0 / z0) - asin(r0 / S)) / (1 + psi));
        double ff = (S + P) / 2.;
        double bq = -(h_sq(r0) + h_sq(ff - P) + h_sq(ff));
        double cq = h_sq(ff) * h_sq(ff - P);
        double aa = sqrt((-bq + sqrt(h_sq(bq) - 4 * cq)) / 2.);
        double bb = sqrt(h_sq(aa) - h_sq(ff));
        s.g0 = ff - P + z0; s.g1 = h_sq(aa); s.g2 = h_sq(bb);
        s.ig1 = 1 / s.g1; s.ig2 = 1 / s.g2;
        s.tol = h_tol10();
    }
    return 0;
}

// Fold (coeff, rorder, aorder) into the (n,|m|) table of pxf_ray.cuh.  Returns the highest
// radial order, or -1 for an invalid table (n>15, |m|>n, n-|m| odd).
// rot: the set is evaluated at theta+rot (tracezernrot's second set, zernsurf.f95:311): cos/sin of
// m*(theta+rot) expanded by the angle-addition formulas rotate the (cosine, sine) coefficient pair of
// every (n,m).  accumulate: add the set to a table already built (same rad).
inline int make_zern(ZernP &z, const double *coeff, const int32_t *rorder, const int32_t *aorder,
                     int arrsize, double rad, bool opd, double nr, double rot = 0., bool accumulate = false)
{
    if (!accumulate) {
        memset(&z, 0, sizeof(z));
        z.rad = rad; z.nr = nr; z.tol = h_tol10(); z.opd = opd ? 1 : 0;
    }
    int nmax = 0;
    for (int i = 0; i < arrsize; i++) {
        int n = rorder[i], mm = aorder[i], m = mm < 0 ? -mm : mm;
        if (n < 0 || n > PXF_ZERN_MAXN || m > n || ((n - m) & 1)) return -1;
        if (n > nmax) nmax = n;
    }
    // the reference sizes its tables from znum (specialFunctions.f95:154-161); radial orders
    // beyond radnum-1 would index out of bounds there.  Mirror the table size.
    int tznum = 1, radnum = 1;
    while (tznum < arrsize) { tznum += radnum + 1; radnum += 1; }
    if (nmax > radnum - 1) return -1;
    if (!accumulate || nmax > z.nmax) z.nmax = nmax;
    const double sqrthalf32 = (double)sqrtf(0.5f);
    if (!accumulate) {
        int e = 0;
        for (int ni = 0; ni <= PXF_ZERN_MAXN; ni++) {
            for (int j = 0; j <= ni / 2; j++) {
                double n = ni, m = ni - 2 * j;
                ZernEntry &t = z.e[e + j];
                if (j >= 2) {
                    t.h3 = -4 * (m + 2) * (m + 1) / (n + m + 2) / (n - m);
                    t.h2 = t.h3 * (n + m + 4) * (n - m - 2) / 4. / (m + 3) + (m + 2);
                    t.h1 = .5 * (m + 4) * (m + 3) - (m + 4) * t.h2 + t.h3 * (n + m + 6) * (n - m - 4) / 8.;
                }
            }
            e += ni / 2 + 1;
        }
    }
    for (int i = 0; i < arrsize; i++) {
        int n = rorder[i], mm = aorder[i], m = mm < 0 ? -mm : mm;
        int base = 0;
        for (int q = 0; q < n; q++) base += q / 2 + 1;
        ZernEntry &t = z.e[base + (n - m) / 2];
        double norm = sqrt(2 * ((double)n + 1));
        if (rot == 0.) {
            if (mm < 0) t.as += coeff[i] * norm;
            else if (mm > 0) t.ac += coeff[i] * norm;
            else t.ac += coeff[i] * (norm * sqrthalf32);
        } else {
            const double cr = cos(m * rot), sr = sin(m * rot);
            if (mm < 0) { t.as += coeff[i] * norm * cr; t.ac += coeff[i] * norm * sr; }        // sin(m(theta+rot))
            else if (mm > 0) { t.ac += coeff[i] * norm * cr; t.as -= coeff[i] * norm * sr; }   // cos(m(theta+rot))
            else t.ac += coeff[i] * (norm * sqrthalf32);
        }
    }
    // power-basis table for the nmax <= 7 kernel, rebuilt from the folded (n,|m|) entries:
    //   R_n^m(rho) = sum_s (-1)**s (n-s)! / (s! ((n+m)/2-s)! ((n-m)/2-s)!) rho**(n-2s),  rho**(n-2s) = rho**m * u**((n-m)/2-s)
    memset(z.pc, 0, sizeof(z.pc));
    if (z.nmax <= 7) {
        double fact[16];
        fact[0] = 1.;
        for (int i = 1; i < 16; i++) fact[i] = fact[i - 1] * i;
        int e = 0;
        for (int n = 0; n <= 7; n++) {
            for (int j = 0; j <= n / 2; j++) {
                const int m = n - 2 * j;
                const ZernEntry &t = z.e[e + j];
                if (t.ac != 0. || t.as != 0.)
                    for (int sgn = 0; sgn <= (n - m) / 2; sgn++) {
                        const double c = ((sgn & 1) ? -1. : 1.) * fact[n - sgn] /
                                         (fact[sgn] * fact[(n + m) / 2 - sgn] * fact[(n - m) / 2 - sgn]);
                        const int jj = (n - m) / 2 - sgn;
                        z.pc[m][jj][0] += t.ac * c;
                        z.pc[m][jj][1] += t.as * c;
                    }
            }
            e += n / 2 + 1;
        }
    }
    // ... and the same polynomial in Cartesian form (ZernP::xy), expanded in long double
    memset(z.xy, 0, sizeof(z.xy));
    if (z.nmax <= 7) {
        long double K[8][8];
        memset(K, 0, sizeof(K));
        long double binom[8][8];
        memset(binom, 0, sizeof(binom));
        for (int n = 0; n < 8; n++) {
            binom[n][0] = 1.L;
            for (int k = 1; k <= n; k++) binom[n][k] = binom[n - 1][k - 1] + (k <= n - 1 ? binom[n - 1][k] : 0.L);
        }
        for (int m = 0; m < PXF_ZERN_PM; m++)
            for (int j = 0; j < PXF_ZERN_PJ; j++)
                for (int cs = 0; cs < 2; cs++) {
                    const long double c = z.pc[m][j][cs];
                    if (c == 0.L || m + 2 * j > 7) continue;
                    // Re / Im of (X+iY)**m: terms X**(m-k) Y**k with k even / odd, sign (-1)**(k div 2)
                    for (int k = cs; k <= m; k += 2) {
                        const long double w = c * binom[m][k] * (((k / 2) & 1) ? -1.L : 1.L);
                        for (int i = 0; i <= j; i++) K[m - k + 2 * i][k + 2 * (j - i)] += w * binom[j][i];
                    }
                }
        for (int a = 0; a < 8; a++)
            for (int b = 0; a + b <= 7; b++) z.xy[PXF_ZERN_XYOFF(a) + b] = (double)K[a][b];
    }
    return z.nmax;
}

}  // namespace pxf
