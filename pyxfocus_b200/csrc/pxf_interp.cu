// Scattered-data interpolation of a per-ray quantity onto query points: analyses.interpolateVec / wavefront
// (analyses.py:189-230, 305-334), which call scipy.interpolate.griddata (Delaunay triangulation + barycentric
// interpolation for 'linear', nearest neighbour for 'nearest').  SURVEY.md 8(f) rank 4.
//
// No global triangulation is built.  The Delaunay triangle that contains a query point q is the optimum of a
// three-variable linear programme (the facet of the lifted points' lower hull under q), reached by pivoting, one
// thread per query, with O(1) state:
//   1. the points are binned into a uniform cell grid (counting sort by cell through pxf_argsort);
//   2. a start triangle that contains q: the nearest point of each quadrant about q gives four points whose hull
//      holds q, and one of their triangles does.  If a quadrant is empty (q near or outside the hull) one pass over
//      all points finds the extreme directions on both sides of a first point: either they close a triangle
//      around q, or a half-plane through q holds every point and q is outside the convex hull -> NaN (griddata's
//      fill value);
//   3. while some point lies inside the triangle's circumcircle, the deepest such point replaces the vertex that
//      keeps q inside (q's height on the lifted plane falls monotonically, so this ends); only the cells under the
//      circumcircle are scanned.  The final triangle contains q and has an empty circumcircle: it is the triangle
//      of the Delaunay triangulation (unique in general position) that scipy/Qhull interpolates in;
//   4. barycentric interpolation inside that triangle.
#include <string.h>
#include <vector>
#include "pxf_internal.h"
#include "pxf_ray.cuh"

namespace pxf {

#define GI_THREADS 128
#define GI_COOP_THREADS 256    // threads of a CTA that share ONE deferred query / vertex
#define GI_MAX_PIVOTS 512
#define GI_ILP 8              // independent point loads in flight per lane in the all-points passes

#define GI_NDIR 256         // support directions of the outer hull approximation (the band between hull and polygon shrinks as 1/NDIR^2)
#define GI_DIR_SLICES 32
struct GridCells {
    double x0, y0, x1, y1, h;   // bounding box, cell size
    int gx, gy;
    // the points' support function in GI_NDIR directions: max_i p_i . u_k.  A query with q . u_k above it is outside
    // the convex hull (an exact certificate); only the thin band between this polygon and the hull pays for the
    // all-points pass of step 2
    double ux[GI_NDIR], uy[GI_NDIR], sup[GI_NDIR];
};

// ---------------------------------------------------------------- bounding box (two-stage, deterministic)
__global__ void __launch_bounds__(256)
k_bbox_partial(const double *__restrict__ x, const double *__restrict__ y, int64_t num, double *__restrict__ part /*[grid][4]*/)
{
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    double xl = inf, xh = -inf, yl = inf, yh = -inf;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < num; i += (int64_t)gridDim.x * blockDim.x) {
        const double a = x[i], b = y[i];
        xl = fmin(xl, a); xh = fmax(xh, a); yl = fmin(yl, b); yh = fmax(yh, b);
    }
    __shared__ double sh[4][8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        xl = fmin(xl, __shfl_down_sync(0xffffffffu, xl, o)); xh = fmax(xh, __shfl_down_sync(0xffffffffu, xh, o));
        yl = fmin(yl, __shfl_down_sync(0xffffffffu, yl, o)); yh = fmax(yh, __shfl_down_sync(0xffffffffu, yh, o));
    }
    if ((threadIdx.x & 31) == 0) { const int w = threadIdx.x >> 5; sh[0][w] = xl; sh[1][w] = xh; sh[2][w] = yl; sh[3][w] = yh; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) { xl = fmin(xl, sh[0][w]); xh = fmax(xh, sh[1][w]); yl = fmin(yl, sh[2][w]); yh = fmax(yh, sh[3][w]); }
        part[blockIdx.x * 4 + 0] = xl; part[blockIdx.x * 4 + 1] = xh; part[blockIdx.x * 4 + 2] = yl; part[blockIdx.x * 4 + 3] = yh;
    }
}

// block (k, s): max over slice s of the points of p . u_k
__global__ void __launch_bounds__(256)
k_support_partial(const double *__restrict__ x, const double *__restrict__ y, int64_t num, double *__restrict__ part /*[NDIR][SLICES]*/)
{
    const int k = blockIdx.x % GI_NDIR, sl = blockIdx.x / GI_NDIR;
    double sn, cs;
    sincospi(2. * k / GI_NDIR, &sn, &cs);
    double best = -__longlong_as_double(0x7ff0000000000000ll);
    for (int64_t i = (int64_t)sl * blockDim.x + threadIdx.x; i < num; i += (int64_t)GI_DIR_SLICES * blockDim.x)
        best = fmax(best, x[i] * cs + y[i] * sn);
    __shared__ double sh[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_down_sync(0xffffffffu, best, o));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) best = fmax(best, sh[w]);
        part[k * GI_DIR_SLICES + sl] = best;
    }
}

// one warp: fold the partial boxes and supports and lay out the cell grid (about two points per cell)
__global__ void k_grid_setup(const double *__restrict__ part, int nblk, int64_t num, int max_cells, GridCells *g,
                             const double *__restrict__ spart)
{
    if (blockIdx.x) return;
    for (int k = threadIdx.x; k < GI_NDIR; k += blockDim.x) {
        double sn, cs;
        sincospi(2. * k / GI_NDIR, &sn, &cs);
        double b = spart[k * GI_DIR_SLICES];
        for (int sl = 1; sl < GI_DIR_SLICES; sl++) b = fmax(b, spart[k * GI_DIR_SLICES + sl]);
        g->ux[k] = cs; g->uy[k] = sn; g->sup[k] = b;
    }
    if (threadIdx.x) return;
    double xl = part[0], xh = part[1], yl = part[2], yh = part[3];
    for (int b = 1; b < nblk; b++) {
        xl = fmin(xl, part[4 * b]); xh = fmax(xh, part[4 * b + 1]); yl = fmin(yl, part[4 * b + 2]); yh = fmax(yh, part[4 * b + 3]);
    }
    double W = xh - xl, H = yh - yl;
    const double diag = sqrt(W * W + H * H);
    if (!(W > 0.)) W = diag > 0. ? diag * 1e-6 : 1.;
    if (!(H > 0.)) H = diag > 0. ? diag * 1e-6 : 1.;
    double cells = (double)num / 2.;
    if (cells < 1.) cells = 1.;
    if (cells > (double)max_cells) cells = (double)max_cells;
    double h = sqrt(W * H / cells);
    // a very elongated box: never more than max_cells cells in total
    int gx = (int)ceil(W / h), gy = (int)ceil(H / h);
    while ((double)gx * (double)gy > (double)max_cells) { h *= 1.1; gx = (int)ceil(W / h); gy = (int)ceil(H / h); }
    if (gx < 1) gx = 1;
    if (gy < 1) gy = 1;
    g->x0 = xl; g->y0 = yl; g->x1 = xh; g->y1 = yh; g->h = h; g->gx = gx; g->gy = gy;
}

PXF_DEV int cell_of(const GridCells &g, double x, double y, int &cx, int &cy)
{
    cx = (int)floor((x - g.x0) / g.h);
    cy = (int)floor((y - g.y0) / g.h);
    cx = cx < 0 ? 0 : (cx >= g.gx ? g.gx - 1 : cx);
    cy = cy < 0 ? 0 : (cy >= g.gy ? g.gy - 1 : cy);
    return cy * g.gx + cx;
}

__global__ void __launch_bounds__(256)
k_cell_keys(const double *__restrict__ x, const double *__restrict__ y, int64_t num, const GridCells *__restrict__ gp,
            double *__restrict__ key)
{
    const GridCells &g = *gp;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < num; i += (int64_t)gridDim.x * blockDim.x) {
        int cx, cy;
        key[i] = (double)cell_of(g, x[i], y[i], cx, cy);
    }
}

// start[c] = first sorted position of cell c (start[ncell] = num); also the points in cell order
__global__ void __launch_bounds__(256)
k_cell_starts(const double *__restrict__ skey, const long long *__restrict__ perm, int64_t num, const GridCells *__restrict__ gp,
              const double *__restrict__ x, const double *__restrict__ y, const double *__restrict__ v,
              int *__restrict__ start, double *__restrict__ sx, double *__restrict__ sy, double *__restrict__ sv)
{
    const int ncell = gp->gx * gp->gy;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < num; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)skey[i];
        const int prev = i > 0 ? (int)skey[i - 1] : -1;
        for (int k = prev + 1; k <= c; k++) start[k] = (int)i;
        if (i == num - 1)
            for (int k = c + 1; k <= ncell; k++) start[k] = (int)num;
        const long long p = perm[i];
        sx[i] = x[p]; sy[i] = y[p]; sv[i] = v[p];
    }
}

// ---------------------------------------------------------------- the query kernel
// per row of cells: the next non-empty cell at or after each cell, and the previous one at or before it (-1: none).
// One thread per row.  (For the nearest-neighbour search of queries far from the data.)
__global__ void __launch_bounds__(128)
k_row_links(const int *__restrict__ start, const GridCells *__restrict__ gp, int *__restrict__ nxt, int *__restrict__ prv)
{
    const int gx = gp->gx, gy = gp->gy;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= gy) return;
    int last = -1;
    for (int i = gx - 1; i >= 0; i--) {
        const int c = j * gx + i;
        if (start[c + 1] > start[c]) last = c;
        nxt[c] = last;
    }
    last = -1;
    for (int i = 0; i < gx; i++) {
        const int c = j * gx + i;
        if (start[c + 1] > start[c]) last = c;
        prv[c] = last;
    }
}

// lower bound of the distance from q to any point in a cell outside the (2r+1)^2 block around cell (cx, cy);
// +inf when the block covers the whole grid
PXF_DEV double ring_clearance(const GridCells &g, double qx, double qy, int cx, int cy, int r)
{
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    double d = inf;
    if (cx - r > 0) d = fmin(d, fmax(0., qx - (g.x0 + (cx - r) * g.h)));
    if (cx + r < g.gx - 1) d = fmin(d, fmax(0., (g.x0 + (cx + r + 1) * g.h) - qx));
    if (cy - r > 0) d = fmin(d, fmax(0., qy - (g.y0 + (cy - r) * g.h)));
    if (cy + r < g.gy - 1) d = fmin(d, fmax(0., (g.y0 + (cy + r + 1) * g.h) - qy));
    return d;
}

// 2 x signed area: > 0 when a, b, c turn left
PXF_DEV double orient2(double ax, double ay, double bx, double by, double cx, double cy)
{
    return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax);
}

// > 0 when p is inside the circle through a, b, c (counter-clockwise)
PXF_DEV double incircle(double ax, double ay, double bx, double by, double cx, double cy, double px, double py)
{
    const double adx = ax - px, ady = ay - py, bdx = bx - px, bdy = by - py, cdx = cx - px, cdy = cy - py;
    const double ad = adx * adx + ady * ady, bd = bdx * bdx + bdy * bdy, cd = cdx * cdx + cdy * cdy;
    return adx * (bdy * cd - bd * cdy) - ady * (bdx * cd - bd * cdx) + ad * (bdx * cdy - bdy * cdx);
}

// ================================================================= 'cubic': scipy's CloughTocher2DInterpolator
// (what griddata(method='cubic') constructs for 2-D data; scipy/interpolate/interpnd.pyx).  Three ingredients:
//   (a) the Delaunay neighbours of every data point, in counter-clockwise order (k_dt_rings): gift wrapping about the
//       point -- the nearest neighbour is a Delaunay neighbour, and the apex of the Delaunay triangle on one side of an
//       edge p-n is the point of that side that minimises the centre offset t of the circle through p, n and it;
//   (b) the gradient at every data point from scipy's global estimate: Gauss-Seidel sweeps IN INPUT ORDER to a relative
//       change below tol (estimate_gradients_2d_global).  The sequential sweep is reproduced exactly in parallel by
//       level scheduling: a vertex's level is one more than the highest level among its neighbours that come earlier in
//       the input, vertices of one level are mutually non-adjacent, and levels run in order;
//   (c) the Clough-Tocher cubic on the triangle that holds the query (same triangle search as 'linear'), with the
//       cross-edge derivative taken towards the centroid of the neighbouring triangle (read off the rings).
#define GI_DEG 48              // Delaunay neighbours kept per point (a degenerate set -- a thin arc -- can exceed it)

struct Rings {
    int *ring;                 // [num][GI_DEG] neighbours, counter-clockwise
    unsigned char *deg;        // [num]
    unsigned char *open;       // [num] 1: hull vertex, the ring is a chain from its clockwise end to its counter-clockwise end
};

// Apex of the Delaunay triangle on one side (side = +1: left, -1: right) of the edge from point ip to point in_:
// the point x of that side with the smallest t = x.(x - e) / (2 side cross(e, x)) (positions relative to ip; the circle
// through ip, in_, x has its centre at e/2 + t * side-normal(e)).  -1: no point on that side (a hull edge); -2: not
// settled within GI_RQ_DT rings of cells (a hull edge or a sliver beside the hull: the warp kernel takes the vertex).
#define GI_RQ_DT 24
PXF_DEV int apex_of_edge(const GridCells &g, const double *__restrict__ sx, const double *__restrict__ sy,
                         const int *__restrict__ start, int ip, int in_, double side, int rq_dt)
{
    const double px = sx[ip], py = sy[ip];
    const double ex = sx[in_] - px, ey = sy[in_] - py;
    const double e2 = ex * ex + ey * ey;
    int cx, cy;
    cell_of(g, px, py, cx, cy);
    const int rcap = g.gx > g.gy ? g.gx : g.gy;
    double tbest = __longlong_as_double(0x7ff0000000000000ll), r2best = tbest;
    int best = -1;
    bool settled = false;
    for (int r = 0; r <= rcap && r <= rq_dt; r++) {
        for (int j = cy - r; j <= cy + r; j++) {
            if (j < 0 || j >= g.gy) continue;
            const bool edge_row = j == cy - r || j == cy + r;
            for (int i = cx - r; i <= cx + r; i += (edge_row ? 1 : 2 * r > 0 ? 2 * r : 1)) {
                if (i < 0 || i >= g.gx) continue;
                const int c = j * g.gx + i;
                for (int q = start[c]; q < start[c + 1]; q++) {
                    if (q == ip || q == in_) continue;
                    const double x = sx[q] - px, y = sy[q] - py;
                    const double cr = side * (ex * y - ey * x);
                    if (!(cr > 1e-14 * sqrt(e2 * (x * x + y * y)))) continue;
                    const double t = (x * (x - ex) + y * (y - ey)) / (2. * cr);
                    if (t < tbest || (t == tbest && q < best)) { tbest = t; best = q; r2best = e2 * (.25 + t * t); }
                }
            }
        }
        if (best >= 0) {
            // any better apex lies inside the best circle so far, i.e. within its diameter of ip
            const double clr = ring_clearance(g, px, py, cx, cy, r);
            if (clr * clr > 4. * r2best) { settled = true; break; }
        }
        if (r == rcap) settled = true;
    }
    return settled ? best : -2;
}

// the same by the 32 lanes of a warp over ALL points (every lane returns the result)
// one lane-strided pass over the points [p0, p1) of the apex search: keeps the smallest t
PXF_DEV void apex_scan_range(const double *__restrict__ sx, const double *__restrict__ sy, int p0, int p1, int lane, int ip, int in_,
                             double px, double py, double ex, double ey, double e2, double side, double &tbest, int &best)
{
    const int nco = (int)blockDim.x;                  // `lane`: position among the CTA's threads, which share the search
    for (int q0 = p0 + lane; q0 < p1; q0 += nco * GI_ILP) {
        double xs[GI_ILP], ys[GI_ILP];
#pragma unroll
        for (int u = 0; u < GI_ILP; u++) {
            const int q = q0 + nco * u;
            xs[u] = q < p1 ? sx[q] : px; ys[u] = q < p1 ? sy[q] : py;
        }
#pragma unroll
        for (int u = 0; u < GI_ILP; u++) {
            const int q = q0 + nco * u;
            if (q >= p1) break;
            if (q == ip || q == in_) continue;
            const double x = xs[u] - px, y = ys[u] - py;
            const double cr = side * (ex * y - ey * x);
            if (!(cr > 1e-14 * sqrt(e2 * (x * x + y * y)))) continue;
            const double t = (x * (x - ex) + y * (y - ey)) / (2. * cr);
            if (t < tbest || (t == tbest && q < best)) { tbest = t; best = q; }
        }
    }
}

// every thread of the CTA ends up with the same (smallest t, lowest index) pair
PXF_DEV void apex_agree(double &tbest, int &best)
{
    __shared__ double a_t[32];
    __shared__ int a_b[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ot = __shfl_xor_sync(0xffffffffu, tbest, o);
        const int ob = __shfl_xor_sync(0xffffffffu, best, o);
        if (ob >= 0 && (best < 0 || ot < tbest || (ot == tbest && ob < best))) { tbest = ot; best = ob; }
    }
    const int nw = blockDim.x >> 5;
    if (nw > 1) {
        if ((threadIdx.x & 31) == 0) { a_t[threadIdx.x >> 5] = tbest; a_b[threadIdx.x >> 5] = best; }
        __syncthreads();
        tbest = __longlong_as_double(0x7ff0000000000000ll); best = -1;
        for (int k = 0; k < nw; k++) {
            const double ot = a_t[k];
            const int ob = a_b[k];
            if (ob >= 0 && (best < 0 || ot < tbest || (ot == tbest && ob < best))) { tbest = ot; best = ob; }
        }
        __syncthreads();
    }
}

// the same by all threads of a CTA (every thread returns the result): a candidate from the block of cells the thread
// kernel gave up on, then every cell under the candidate's circle (any better apex lies inside it); only an edge
// with no candidate nearby -- a hull edge -- takes a pass over ALL points
PXF_DEV int apex_of_edge_warp(const GridCells &g, const double *__restrict__ sx, const double *__restrict__ sy,
                              const int *__restrict__ start, int np, int ip, int in_, double side)
{
    const int lane = threadIdx.x;
    const double px = sx[ip], py = sy[ip];
    const double ex = sx[in_] - px, ey = sy[in_] - py;
    const double e2 = ex * ex + ey * ey;
    double tbest = __longlong_as_double(0x7ff0000000000000ll);
    int best = -1;
    int cx, cy;
    cell_of(g, px, py, cx, cy);
    {
        const int i0 = cx - GI_RQ_DT < 0 ? 0 : cx - GI_RQ_DT, i1 = cx + GI_RQ_DT >= g.gx ? g.gx - 1 : cx + GI_RQ_DT;
        for (int j = cy - GI_RQ_DT; j <= cy + GI_RQ_DT; j++) {
            if (j < 0 || j >= g.gy) continue;
            apex_scan_range(sx, sy, start[j * g.gx + i0], start[j * g.gx + i1 + 1], lane, ip, in_, px, py, ex, ey, e2, side, tbest, best);
        }
        apex_agree(tbest, best);
    }
    if (best < 0) {
        apex_scan_range(sx, sy, 0, np, lane, ip, in_, px, py, ex, ey, e2, side, tbest, best);
        apex_agree(tbest, best);
        return best;
    }
    // centre of the candidate's circle: e/2 + t * side * (-ey, ex); radius^2 = e2 (1/4 + t^2)
    const double ox = px + .5 * ex - tbest * side * ey, oy = py + .5 * ey + tbest * side * ex;
    const double R = sqrt(e2 * (.25 + tbest * tbest));
    const double fi0 = (ox - R - g.x0) / g.h, fi1 = (ox + R - g.x0) / g.h, fj0 = (oy - R - g.y0) / g.h, fj1 = (oy + R - g.y0) / g.h;
    const int i0 = fi0 > 0. ? (fi0 < (double)g.gx ? (int)fi0 : g.gx - 1) : 0;
    const int i1 = fi1 < (double)g.gx ? (fi1 > 0. ? (int)fi1 : 0) : g.gx - 1;
    const int j0 = fj0 > 0. ? (fj0 < (double)g.gy ? (int)fj0 : g.gy - 1) : 0;
    const int j1 = fj1 < (double)g.gy ? (fj1 > 0. ? (int)fj1 : 0) : g.gy - 1;
    for (int j = j0; j <= j1; j++)
        apex_scan_range(sx, sy, start[j * g.gx + i0], start[j * g.gx + i1 + 1], lane, ip, in_, px, py, ex, ey, e2, side, tbest, best);
    apex_agree(tbest, best);
    return best;
}

__global__ void __launch_bounds__(GI_THREADS)
k_dt_rings(const double *__restrict__ sx, const double *__restrict__ sy, const int *__restrict__ start,
           const GridCells *__restrict__ gp, int num, Rings R, unsigned long long *__restrict__ nfail,
           unsigned *__restrict__ slow, int rq_dt)
{
    const int ip = blockIdx.x * blockDim.x + threadIdx.x;
    if (ip >= num) return;
    const GridCells &g = *gp;
    const double px = sx[ip], py = sy[ip];
    int cx, cy;
    cell_of(g, px, py, cx, cy);
    const int rcap = g.gx > g.gy ? g.gx : g.gy;
    // the nearest neighbour
    double best = __longlong_as_double(0x7ff0000000000000ll);
    int n0 = -1;
    for (int r = 0; r <= rcap; r++) {
        for (int j = cy - r; j <= cy + r; j++) {
            if (j < 0 || j >= g.gy) continue;
            const bool edge_row = j == cy - r || j == cy + r;
            for (int i = cx - r; i <= cx + r; i += (edge_row ? 1 : 2 * r > 0 ? 2 * r : 1)) {
                if (i < 0 || i >= g.gx) continue;
                const int c = j * g.gx + i;
                for (int q = start[c]; q < start[c + 1]; q++) {
                    if (q == ip) continue;
                    const double x = sx[q] - px, y = sy[q] - py, d2 = x * x + y * y;
                    if (d2 < best || (d2 == best && q < n0)) { best = d2; n0 = q; }
                }
            }
        }
        const double clr = ring_clearance(g, px, py, cx, cy, r);
        if (clr * clr > best) break;
    }
    int ccw[GI_DEG], cw[GI_DEG];
    int nccw = 0, ncw = 0;
    bool ok = n0 >= 0 && best > 0., open = false, defer = false;
    if (ok) {
        ccw[nccw++] = n0;
        for (int cur = n0;;) {
            const int d = apex_of_edge(g, sx, sy, start, ip, cur, 1., rq_dt);
            if (d == -2) { defer = true; break; }
            if (d < 0) { open = true; break; }
            if (d == n0) break;
            if (nccw >= GI_DEG) { ok = false; break; }
            ccw[nccw++] = d;
            cur = d;
        }
        if (ok && open && !defer)
            for (int cur = n0;;) {
                const int d = apex_of_edge(g, sx, sy, start, ip, cur, -1., rq_dt);
                if (d == -2) { defer = true; break; }
                if (d < 0) break;
                if (nccw + ncw >= GI_DEG) { ok = false; break; }
                cw[ncw++] = d;
                cur = d;
            }
    }
    if (!ok) { R.deg[ip] = 0; R.open[ip] = 1; atomicAdd(nfail, 1ull); atomicAdd(nfail + 2, 1ull); return; }
    if (defer) { R.deg[ip] = 0; slow[1 + atomicAdd(slow, 1u)] = (unsigned)ip; return; }
    int *out = R.ring + (size_t)ip * GI_DEG;
    for (int k = 0; k < ncw; k++) out[k] = cw[ncw - 1 - k];
    for (int k = 0; k < nccw; k++) out[ncw + k] = ccw[k];
    R.deg[ip] = (unsigned char)(ncw + nccw);
    R.open[ip] = open ? 1 : 0;
}

// One CTA per deferred vertex (beside the hull): the same gift wrapping with every apex searched by all threads.
__global__ void __launch_bounds__(GI_COOP_THREADS)
k_dt_rings_warp(const double *__restrict__ sx, const double *__restrict__ sy, const int *__restrict__ start,
                const GridCells *__restrict__ gp, int num, Rings R, unsigned long long *__restrict__ nfail,
                const unsigned *__restrict__ slow)
{
    const GridCells &g = *gp;
    const unsigned nslow = slow[0];
    const int tid = threadIdx.x;
    __shared__ double n_d[32];
    __shared__ int n_i[32];
    for (unsigned w = blockIdx.x; w < nslow; w += gridDim.x) {
        const int ip = (int)slow[1 + w];
        const double px = sx[ip], py = sy[ip];
        double best = __longlong_as_double(0x7ff0000000000000ll);
        int n0 = -1;
        for (int q0 = tid; q0 < num; q0 += (int)blockDim.x * GI_ILP) {
            double xs[GI_ILP], ys[GI_ILP];
#pragma unroll
            for (int u = 0; u < GI_ILP; u++) {
                const int q = q0 + (int)blockDim.x * u;
                xs[u] = q < num ? sx[q] : px; ys[u] = q < num ? sy[q] : py;
            }
#pragma unroll
            for (int u = 0; u < GI_ILP; u++) {
                const int q = q0 + (int)blockDim.x * u;
                if (q >= num || q == ip) continue;
                const double x = xs[u] - px, y = ys[u] - py, d2 = x * x + y * y;
                if (d2 < best || (d2 == best && q < n0)) { best = d2; n0 = q; }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double od = __shfl_xor_sync(0xffffffffu, best, o);
            const int on = __shfl_xor_sync(0xffffffffu, n0, o);
            if (on >= 0 && (n0 < 0 || od < best || (od == best && on < n0))) { best = od; n0 = on; }
        }
        if ((tid & 31) == 0) { n_d[tid >> 5] = best; n_i[tid >> 5] = n0; }
        __syncthreads();
        best = __longlong_as_double(0x7ff0000000000000ll); n0 = -1;
        for (int k = 0; k < (int)(blockDim.x >> 5); k++)
            if (n_i[k] >= 0 && (n0 < 0 || n_d[k] < best || (n_d[k] == best && n_i[k] < n0))) { best = n_d[k]; n0 = n_i[k]; }
        __syncthreads();
        int *out = R.ring + (size_t)ip * GI_DEG;       // assembled in place: clockwise part reversed at the end
        int nccw = 0, ncw = 0;
        bool ok = n0 >= 0 && best > 0., open = false;
        int cwbuf[GI_DEG];
        if (ok) {
            if (tid == 0) out[0] = n0;
            nccw = 1;
            for (int cur = n0;;) {
                const int d = apex_of_edge_warp(g, sx, sy, start, num, ip, cur, 1.);
                if (d < 0) { open = true; break; }
                if (d == n0) break;
                if (nccw >= GI_DEG) { ok = false; break; }
                if (tid == 0) out[nccw] = d;
                nccw++;
                cur = d;
            }
            if (ok && open)
                for (int cur = n0;;) {
                    const int d = apex_of_edge_warp(g, sx, sy, start, num, ip, cur, -1.);
                    if (d < 0) break;
                    if (nccw + ncw >= GI_DEG) { ok = false; break; }
                    cwbuf[ncw++] = d;
                    cur = d;
                }
        }
        if (tid == 0) {
            if (!ok) { R.deg[ip] = 0; R.open[ip] = 1; atomicAdd(nfail, 1ull); atomicAdd(nfail + 2, 1ull); }
            else {
                // shift the counter-clockwise part up and put the clockwise part, reversed, in front
                for (int k = nccw - 1; k >= 0; k--) out[ncw + k] = out[k];
                for (int k = 0; k < ncw; k++) out[k] = cwbuf[ncw - 1 - k];
                R.deg[ip] = (unsigned char)(ncw + nccw);
                R.open[ip] = open ? 1 : 0;
            }
        }
        __syncthreads();
    }
}

// rings in the caller's point numbering: row orig[i] of the output holds the neighbours of sorted point i
__global__ void __launch_bounds__(256)
k_rings_export(const Rings R, const long long *__restrict__ orig, int num, int *__restrict__ ring_out,
               unsigned char *__restrict__ deg_out, unsigned char *__restrict__ open_out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= num) return;
    const long long o = orig[i];
    const int *ring = R.ring + (size_t)i * GI_DEG;
    for (int k = 0; k < GI_DEG; k++) ring_out[o * GI_DEG + k] = k < R.deg[i] ? (int)orig[ring[k]] : -1;
    deg_out[o] = R.deg[i];
    open_out[o] = R.open[i];
}

// one relaxation of level[i] = 1 + max{ level[j] : j a neighbour that comes before i in the input }
__global__ void __launch_bounds__(256)
k_gs_levels(const Rings R, const long long *__restrict__ orig, int num, int *__restrict__ level, int *__restrict__ changed)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= num) return;
    const long long oi = orig[i];
    int L = 0;
    const int *ring = R.ring + (size_t)i * GI_DEG;
    for (int k = 0; k < R.deg[i]; k++) {
        const int j = ring[k];
        if (orig[j] < oi) { const int lj = level[j] + 1; L = lj > L ? lj : L; }
    }
    // (changed[1]: the highest level so far -- one launch can raise a chain of vertices by several levels)
    if (L > level[i]) { level[i] = L; changed[0] = 1; atomicMax(changed + 1, L); }
}

// level of every vertex as a sort key, and the first sorted position of every level (lstart[nlev + 1] = num)
__global__ void __launch_bounds__(256)
k_level_keys(const int *__restrict__ level, int num, double *__restrict__ key)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < num) key[i] = (double)level[i];
}
__global__ void __launch_bounds__(256)
k_level_starts(const double *__restrict__ skey, int num, int nlev, int *__restrict__ lstart)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= num) return;
    const int c = (int)skey[i];
    const int prev = i > 0 ? (int)skey[i - 1] : -1;
    for (int k = prev + 1; k <= c; k++) lstart[k] = i;
    if (i == num - 1)
        for (int k = c + 1; k <= nlev + 1; k++) lstart[k] = num;
}

// One Gauss-Seidel update of the vertices of one level (scipy _estimate_gradients_2d_global, the body of its loop over
// points).  err: the sweep's largest relative change, as the bits of a non-negative double.
__global__ void __launch_bounds__(256)
k_gs_update(const Rings R, const double *__restrict__ sx, const double *__restrict__ sy, const double *__restrict__ sv,
            const long long *__restrict__ members, int count, double *__restrict__ grad, unsigned long long *__restrict__ err)
{
    // members: the vertices of this level (the vertices sorted by level, cut at the level's range)
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const int i = (int)members[t];
    double Q0 = 0., Q1 = 0., Q3 = 0., s0 = 0., s1 = 0.;
    const int *ring = R.ring + (size_t)i * GI_DEG;
    const double f1 = sv[i], px = sx[i], py = sy[i];
    for (int k = 0; k < R.deg[i]; k++) {
        const int j = ring[k];
        const double ex = sx[j] - px, ey = sy[j] - py;
        const double L = sqrt(ex * ex + ey * ey), L3 = L * L * L;
        const double f2 = sv[j];
        const double df2 = -ex * grad[2 * j] - ey * grad[2 * j + 1];
        Q0 += 4 * ex * ex / L3; Q1 += 4 * ex * ey / L3; Q3 += 4 * ey * ey / L3;
        s0 += (6 * (f1 - f2) - 2 * df2) * ex / L3;
        s1 += (6 * (f1 - f2) - 2 * df2) * ey / L3;
    }
    const double det = Q0 * Q3 - Q1 * Q1;
    const double r0 = (Q3 * s0 - Q1 * s1) / det, r1 = (-Q1 * s0 + Q0 * s1) / det;
    double change = fmax(fabs(grad[2 * i] + r0), fabs(grad[2 * i + 1] + r1));
    grad[2 * i] = -r0; grad[2 * i + 1] = -r1;
    change /= fmax(1., fmax(fabs(r0), fabs(r1)));
    if (change == change) atomicMax(err, (unsigned long long)__double_as_longlong(change));
    else atomicMax(err, 0x7ff0000000000000ull);
}

// the third vertex of the triangle across the edge u -> v of a counter-clockwise triangle (u, v, w): the neighbour that
// precedes v counter-clockwise about u.  -1: a hull edge.
PXF_DEV int across_edge(const Rings &R, int u, int v)
{
    const int *ring = R.ring + (size_t)u * GI_DEG;
    const int deg = R.deg[u];
    for (int k = 0; k < deg; k++)
        if (ring[k] == v) {
            if (k > 0) return ring[k - 1];
            return R.open[u] ? -1 : ring[deg - 1];
        }
    return -2;      // v is not a neighbour of u: the rings and the triangle search disagree
}

// scipy _clough_tocher_2d_single on the counter-clockwise triangle (i0, i1, i2) holding the query; b: its barycentric
// coordinates.  Returns false when the rings do not know an edge of the triangle.
PXF_DEV bool clough_tocher(const double *__restrict__ sx, const double *__restrict__ sy, const double *__restrict__ sv,
                           const double *__restrict__ grad, const Rings &R, int i0, int i1, int i2, const double b[3],
                           double *res)
{
    const int v[3] = {i0, i1, i2};
    const double X0 = sx[i0], Y0 = sy[i0], X1 = sx[i1], Y1 = sy[i1], X2 = sx[i2], Y2 = sy[i2];
    const double e12x = X1 - X0, e12y = Y1 - Y0, e23x = X2 - X1, e23y = Y2 - Y1, e31x = X0 - X2, e31y = Y0 - Y2;
    const double f1 = sv[i0], f2 = sv[i1], f3 = sv[i2];
    const double df12 = +(grad[2 * i0] * e12x + grad[2 * i0 + 1] * e12y), df21 = -(grad[2 * i1] * e12x + grad[2 * i1 + 1] * e12y);
    const double df23 = +(grad[2 * i1] * e23x + grad[2 * i1 + 1] * e23y), df32 = -(grad[2 * i2] * e23x + grad[2 * i2 + 1] * e23y);
    const double df31 = +(grad[2 * i2] * e31x + grad[2 * i2 + 1] * e31y), df13 = -(grad[2 * i0] * e31x + grad[2 * i0 + 1] * e31y);
    const double c3000 = f1, c2100 = (df12 + 3 * c3000) / 3, c2010 = (df13 + 3 * c3000) / 3;
    const double c0300 = f2, c1200 = (df21 + 3 * c0300) / 3, c0210 = (df23 + 3 * c0300) / 3;
    const double c0030 = f3, c1020 = (df31 + 3 * c0030) / 3, c0120 = (df32 + 3 * c0030) / 3;
    const double c2001 = (c2100 + c2010 + c3000) / 3, c0201 = (c1200 + c0300 + c0210) / 3, c0021 = (c1020 + c0120 + c0030) / 3;
    // the gradient of the spline towards the neighbouring triangle's centroid is linear along each edge
    const double area = orient2(X0, Y0, X1, Y1, X2, Y2);
    double gk[3];
    for (int k = 0; k < 3; k++) {
        // neighbour opposite vertex k: across the edge v[k+1] -> v[k+2]
        const int u = v[(k + 1) % 3], w = v[(k + 2) % 3];
        const int d = across_edge(R, u, w);
        if (d == -2) return false;
        if (d < 0) { gk[k] = -.5; continue; }
        const double yx = (sx[u] + sx[w] + sx[d]) / 3, yy = (sy[u] + sy[w] + sy[d]) / 3;
        double c[3];
        c[0] = orient2(yx, yy, X1, Y1, X2, Y2) / area;
        c[1] = orient2(X0, Y0, yx, yy, X2, Y2) / area;
        c[2] = 1. - c[0] - c[1];
        if (k == 0) gk[k] = (2 * c[2] + c[1] - 1) / (2 - 3 * c[2] - 3 * c[1]);
        else if (k == 1) gk[k] = (2 * c[0] + c[2] - 1) / (2 - 3 * c[0] - 3 * c[2]);
        else gk[k] = (2 * c[1] + c[0] - 1) / (2 - 3 * c[1] - 3 * c[0]);
    }
    const double c0111 = (gk[0] * (-c0300 + 3 * c0210 - 3 * c0120 + c0030) + (-c0300 + 2 * c0210 - c0120 + c0021 + c0201)) / 2;
    const double c1011 = (gk[1] * (-c0030 + 3 * c1020 - 3 * c2010 + c3000) + (-c0030 + 2 * c1020 - c2010 + c2001 + c0021)) / 2;
    const double c1101 = (gk[2] * (-c3000 + 3 * c2100 - 3 * c1200 + c0300) + (-c3000 + 2 * c2100 - c1200 + c2001 + c0201)) / 2;
    const double c1002 = (c1101 + c1011 + c2001) / 3, c0102 = (c1101 + c0111 + c0201) / 3, c0012 = (c1011 + c0111 + c0021) / 3;
    const double c0003 = (c1002 + c0102 + c0012) / 3;
    // extended barycentric coordinates
    const double mn = fmin(b[0], fmin(b[1], b[2]));
    const double b1 = b[0] - mn, b2 = b[1] - mn, b3 = b[2] - mn, b4 = 3 * mn;
    *res = b1 * b1 * b1 * c3000 + 3 * b1 * b1 * b2 * c2100 + 3 * b1 * b1 * b3 * c2010 + 3 * b1 * b1 * b4 * c2001 +
           3 * b1 * b2 * b2 * c1200 + 6 * b1 * b2 * b4 * c1101 + 3 * b1 * b3 * b3 * c1020 + 6 * b1 * b3 * b4 * c1011 +
           3 * b1 * b4 * b4 * c1002 + b2 * b2 * b2 * c0300 + 3 * b2 * b2 * b3 * c0210 + 3 * b2 * b2 * b4 * c0201 +
           3 * b2 * b3 * b3 * c0120 + 6 * b2 * b3 * b4 * c0111 + 3 * b2 * b4 * b4 * c0102 + b3 * b3 * b3 * c0030 +
           3 * b3 * b3 * b4 * c0021 + 3 * b3 * b4 * b4 * c0012 + b4 * b4 * b4 * c0003;
    return true;
}

struct Cubic { const double *grad; Rings R; const int *nxt, *prv; };     // grad == nullptr: linear; nxt / prv: row links ('nearest')

#define GI_RQ 12               // rings searched for the quadrant points before a query is handed to the warp kernel
#define GI_CELL_BUDGET 4096    // cells under one circumcircle a single thread may scan

// Steps 3 and 4 for one query from a start triangle (ia, ib, ic: counter-clockwise, holds q).  COOP: ALL threads of the
// CTA work on the SAME query (identical control flow): the points of the cells under the circumcircle are dealt out to
// the threads and the deepest one is agreed on by shuffles and a shared-memory round.  Returns 0: *res holds the value
// (thread 0 when COOP), 1: over the single-thread budget (not COOP), 2: failed.
template <bool COOP>
PXF_DEV int settle_and_interpolate(const GridCells &g, const double *__restrict__ sx, const double *__restrict__ sy,
                                   const double *__restrict__ sv, const int *__restrict__ start, double qx, double qy,
                                   int ia, int ib, int ic, double *res, const Cubic &cub)
{
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    const int lane = COOP ? (int)threadIdx.x : 0;             // position among the cooperating threads
    const int nco = COOP ? (int)blockDim.x : 1;
    __shared__ double co_w[32];
    __shared__ int co_i[32];
    double ax = sx[ia] - qx, ay = sy[ia] - qy, bx = sx[ib] - qx, by = sy[ib] - qy, cx_ = sx[ic] - qx, cy_ = sy[ic] - qy;
    bool settled = false;
    for (int it = 0; it < GI_MAX_PIVOTS; it++) {
        const double area = orient2(ax, ay, bx, by, cx_, cy_);
        if (!(area > 0.)) break;
        // circumcentre (relative to q), radius
        const double ux_ = bx - ax, uy_ = by - ay, vx_ = cx_ - ax, vy_ = cy_ - ay;
        const double ul = ux_ * ux_ + uy_ * uy_, vl = vx_ * vx_ + vy_ * vy_;
        const double ox = ax + (vy_ * ul - uy_ * vl) / (2. * area), oy = ay + (ux_ * vl - vx_ * ul) / (2. * area);
        const double R = sqrt((ox - ax) * (ox - ax) + (oy - ay) * (oy - ay));
        const double tol = 1e-12 * area * R * R;
        // cells under the circle (a huge circle: clamp in floating point, floor() of a huge quotient saturates)
        const double fi0 = (qx + ox - R - g.x0) / g.h, fi1 = (qx + ox + R - g.x0) / g.h;
        const double fj0 = (qy + oy - R - g.y0) / g.h, fj1 = (qy + oy + R - g.y0) / g.h;
        const int i0 = fi0 > 0. ? (fi0 < (double)g.gx ? (int)fi0 : g.gx - 1) : 0;
        const int i1 = fi1 < (double)g.gx ? (fi1 > 0. ? (int)fi1 : 0) : g.gx - 1;
        const int j0 = fj0 > 0. ? (fj0 < (double)g.gy ? (int)fj0 : g.gy - 1) : 0;
        const int j1 = fj1 < (double)g.gy ? (fj1 > 0. ? (int)fj1 : 0) : g.gy - 1;
        if (!COOP && (int64_t)(i1 - i0 + 1) * (j1 - j0 + 1) > GI_CELL_BUDGET) return 1;
        double worst = tol;
        int iw = -1;
        if (COOP) {
            // the lanes share each row's point range, GI_ILP independent loads in flight per lane
            for (int j = j0; j <= j1; j++) {
                const int p0 = start[j * g.gx + i0], p1 = start[j * g.gx + i1 + 1];  // cells of one row are contiguous
                for (int pb = p0 + lane; pb < p1; pb += nco * GI_ILP) {
                    double xs[GI_ILP], ys[GI_ILP];
#pragma unroll
                    for (int u = 0; u < GI_ILP; u++) {
                        const int p = pb + nco * u;
                        xs[u] = p < p1 ? sx[p] : 0.; ys[u] = p < p1 ? sy[p] : 0.;
                    }
#pragma unroll
                    for (int u = 0; u < GI_ILP; u++) {
                        const int p = pb + nco * u;
                        if (p >= p1) break;
                        if (p == ia || p == ib || p == ic) continue;
                        const double v = incircle(ax, ay, bx, by, cx_, cy_, xs[u] - qx, ys[u] - qy);
                        if (v > worst) { worst = v; iw = p; }
                    }
                }
            }
        } else {
            for (int j = j0; j <= j1; j++) {
                const int p0 = start[j * g.gx + i0], p1 = start[j * g.gx + i1 + 1];  // cells of one row are contiguous
                for (int p = p0; p < p1; p++) {
                    if (p == ia || p == ib || p == ic) continue;
                    const double v = incircle(ax, ay, bx, by, cx_, cy_, sx[p] - qx, sy[p] - qy);
                    if (v > worst) { worst = v; iw = p; }
                }
            }
        }
        if (COOP) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, worst, o);
                const int oi = __shfl_xor_sync(0xffffffffu, iw, o);
                if (oi >= 0 && (iw < 0 || ov > worst || (ov == worst && oi < iw))) { worst = ov; iw = oi; }
            }
            if (nco > 32) {
                if ((lane & 31) == 0) { co_w[lane >> 5] = worst; co_i[lane >> 5] = iw; }
                __syncthreads();
                worst = tol; iw = -1;
                for (int k = 0; k < (nco >> 5); k++) {
                    const double ov = co_w[k];
                    const int oi = co_i[k];
                    if (oi >= 0 && (iw < 0 || ov > worst || (ov == worst && oi < iw))) { worst = ov; iw = oi; }
                }
                __syncthreads();
            }
        }
        if (iw < 0) { settled = true; break; }
        // the deepest point replaces the vertex that keeps q inside: of (p,b,c), (a,p,c), (a,b,p) the one that holds q best
        const double px = sx[iw] - qx, py = sy[iw] - qy;
        double bestm = -inf;
        int which = -1;
        for (int k = 0; k < 3; k++) {
            const double x0 = k == 0 ? px : ax, y0 = k == 0 ? py : ay, x1 = k == 1 ? px : bx, y1 = k == 1 ? py : by,
                         x2 = k == 2 ? px : cx_, y2 = k == 2 ? py : cy_;
            const double ar = orient2(x0, y0, x1, y1, x2, y2);
            if (!(ar > 0.)) continue;
            const double m = fmin(fmin(x0 * y1 - y0 * x1, x1 * y2 - y1 * x2), x2 * y0 - y2 * x0) / ar;
            if (m > bestm) { bestm = m; which = k; }
        }
        if (which < 0 || bestm < -1e-9) break;
        if (which == 0) { ax = px; ay = py; ia = iw; }
        else if (which == 1) { bx = px; by = py; ib = iw; }
        else { cx_ = px; cy_ = py; ic = iw; }
    }
    if (!settled) return 2;
    // 4. barycentric coordinates of q (the origin): areas of the sub-triangles
    const double area = orient2(ax, ay, bx, by, cx_, cy_);
    const double oab = ax * by - ay * bx, obc = bx * cy_ - by * cx_, oca = cx_ * ay - cy_ * ax;
    if (cub.grad) {
        const double bb[3] = {obc / area, oca / area, oab / area};
        if (COOP && lane != 0) return 0;                        // (thread 0 evaluates the patch)
        return clough_tocher(sx, sy, sv, cub.grad, cub.R, ia, ib, ic, bb, res) ? 0 : 2;
    }
    *res = obc / area * sv[ia] + oca / area * sv[ib] + oab / area * sv[ic];
    return 0;
}

// One thread per query.  Queries that need a pass over all points (an empty quadrant nearby: near or outside the hull)
// or a very large circumcircle are appended to `slow` for k_griddata_warp.
template <int METHOD>
__global__ void __launch_bounds__(GI_THREADS)
k_griddata(const double *__restrict__ sx, const double *__restrict__ sy, const double *__restrict__ sv,
           const int *__restrict__ start, const GridCells *__restrict__ gp, const double *__restrict__ qxs,
           const double *__restrict__ qys, int64_t nq, double *__restrict__ out, unsigned long long *__restrict__ nfail,
           unsigned *__restrict__ slow, const Cubic cub)
{
    const int64_t iq = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (iq >= nq) return;
    const GridCells &g = *gp;
    const double qx = qxs[iq], qy = qys[iq];
    const double nanv = __longlong_as_double(0x7ff8000000000000ll);
    if (!(qx == qx) || !(qy == qy)) { out[iq] = nanv; return; }
    int cx, cy;
    cell_of(g, qx, qy, cx, cy);
    const int rcap = g.gx > g.gy ? g.gx : g.gy;

    if (METHOD == 0) {
        // nearest neighbour, row by row of cells outwards from q's row: in each row the non-empty cells nearest to q's
        // column (per-row links: no walk over empty cells), as long as their lower bound can beat the best so far.  A
        // query in a corner of the grid, far outside a round aperture, costs O(rows) look-ups instead of O(cells).
        double best = __longlong_as_double(0x7ff0000000000000ll), val = nanv;
        const int *nxt = cub.nxt, *prv = cub.prv;
        for (int dj = 0; dj < g.gy; dj++) {
            bool any = false;
            for (int sgn = 0; sgn < (dj ? 2 : 1); sgn++) {
                const int j = sgn ? cy - dj : cy + dj;
                if (j < 0 || j >= g.gy) continue;
                // vertical distance from q to the band of row j
                const double ylo = g.y0 + j * g.h, yhi = ylo + g.h;
                const double dyb = qy < ylo ? ylo - qy : (qy > yhi ? qy - yhi : 0.);
                if (dyb * dyb > best) continue;
                any = true;
                for (int c = nxt[j * g.gx + cx]; c >= 0;) {            // q's column and to the right
                    const double xlo = g.x0 + (c - j * g.gx) * g.h;
                    const double dxb = qx < xlo ? xlo - qx : 0.;
                    if (dxb * dxb + dyb * dyb > best) break;
                    for (int p = start[c]; p < start[c + 1]; p++) {
                        const double dx = sx[p] - qx, dy = sy[p] - qy, d2 = dx * dx + dy * dy;
                        if (d2 < best) { best = d2; val = sv[p]; }
                    }
                    c = (c + 1 < (j + 1) * g.gx) ? nxt[c + 1] : -1;
                }
                for (int c = cx > 0 ? prv[j * g.gx + cx - 1] : -1; c >= 0;) {      // to the left
                    const double xhi = g.x0 + (c - j * g.gx + 1) * g.h;
                    const double dxb = qx > xhi ? qx - xhi : 0.;
                    if (dxb * dxb + dyb * dyb > best) break;
                    for (int p = start[c]; p < start[c + 1]; p++) {
                        const double dx = sx[p] - qx, dy = sy[p] - qy, d2 = dx * dx + dy * dy;
                        if (d2 < best) { best = d2; val = sv[p]; }
                    }
                    c = (c - 1 >= j * g.gx) ? prv[c - 1] : -1;
                }
            }
            // neither row at this distance is inside the grid and within reach; farther rows are farther still
            if (!any && dj > 0) break;
        }
        out[iq] = val;
        return;
    }

    // ---- linear
    // outside the points' bounding box or beyond their support in some direction: outside their convex hull
    if (qx < g.x0 || qx > g.x1 || qy < g.y0 || qy > g.y1) { out[iq] = nanv; return; }
    {
        const double slack = 1e-12 * (fabs(g.x0) + fabs(g.x1) + fabs(g.y0) + fabs(g.y1));
        bool outside = false;
        for (int k = 0; k < GI_NDIR; k++) outside = outside || (qx * g.ux[k] + qy * g.uy[k] > g.sup[k] + slack);
        if (outside) { out[iq] = nanv; return; }
    }
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    // 2. the nearest point of each half-open quadrant about q
    double qd[4] = {inf, inf, inf, inf};
    int qi[4] = {-1, -1, -1, -1};
    const int rq = rcap < GI_RQ ? rcap : GI_RQ;
    for (int r = 0; r <= rq; r++) {
        for (int j = cy - r; j <= cy + r; j++) {
            if (j < 0 || j >= g.gy) continue;
            const bool edge_row = j == cy - r || j == cy + r;
            for (int i = cx - r; i <= cx + r; i += (edge_row ? 1 : 2 * r > 0 ? 2 * r : 1)) {
                if (i < 0 || i >= g.gx) continue;
                const int c = j * g.gx + i;
                for (int p = start[c]; p < start[c + 1]; p++) {
                    const double dx = sx[p] - qx, dy = sy[p] - qy, d2 = dx * dx + dy * dy;
                    if (d2 == 0.) { out[iq] = sv[p]; return; }        // the query is a data point
                    const int quad = dx > 0. ? (dy >= 0. ? 0 : 3) : (dx < 0. ? (dy > 0. ? 1 : 2) : (dy > 0. ? 1 : 3));
                    if (d2 < qd[quad]) { qd[quad] = d2; qi[quad] = p; }
                }
            }
        }
        if (qi[0] >= 0 && qi[1] >= 0 && qi[2] >= 0 && qi[3] >= 0) break;
    }
    int ia = -1, ib = -1, ic = -1;
    if (qi[0] >= 0 && qi[1] >= 0 && qi[2] >= 0 && qi[3] >= 0) {
        // q is in the hull of the four points (no half-plane through q meets all four quadrants): take the triple
        // that holds it best
        double bestm = -inf;
        for (int skip = 0; skip < 4; skip++) {
            int t[3], n = 0;
            for (int k = 0; k < 4; k++) if (k != skip) t[n++] = qi[k];       // still in counter-clockwise quadrant order
            const double x0 = sx[t[0]] - qx, y0 = sy[t[0]] - qy, x1 = sx[t[1]] - qx, y1 = sy[t[1]] - qy,
                         x2 = sx[t[2]] - qx, y2 = sy[t[2]] - qy;
            const double area = orient2(x0, y0, x1, y1, x2, y2);
            if (!(area > 0.)) continue;
            const double m = fmin(fmin(x0 * y1 - y0 * x1, x1 * y2 - y1 * x2), x2 * y0 - y2 * x0) / area;
            if (m > bestm) { bestm = m; ia = t[0]; ib = t[1]; ic = t[2]; }
        }
        if (ia < 0 || bestm < -1e-12) ia = -1;        // (points exactly on the axes through q: let the warp kernel decide)
    }
    if (ia < 0) {
        // A quadrant is empty nearby (q beside the hull).  The same closure test the warp kernel applies to ALL points,
        // on the points of the rings just searched: a = the nearest one as the zero direction, b / c = the ones turned
        // farthest counter-clockwise / clockwise by less than pi; if c is counter-clockwise of b the triangle holds q.
        // (If it does not close q is outside the hull of the NEARBY points only: the warp kernel decides.)
        int na = -1;
        double nd = inf;
        for (int k = 0; k < 4; k++) if (qi[k] >= 0 && qd[k] < nd) { nd = qd[k]; na = qi[k]; }
        if (na >= 0) {
            const double a0x = sx[na] - qx, a0y = sy[na] - qy;
            int jb = -1, jc = -1;
            double bxx = 0., byy = 0., cxx = 0., cyy = 0.;
            for (int j = cy - rq; j <= cy + rq; j++) {
                if (j < 0 || j >= g.gy) continue;
                const int i0 = cx - rq < 0 ? 0 : cx - rq, i1 = cx + rq >= g.gx ? g.gx - 1 : cx + rq;
                for (int p = start[j * g.gx + i0]; p < start[j * g.gx + i1 + 1]; p++) {
                    if (p == na) continue;
                    const double dx = sx[p] - qx, dy = sy[p] - qy;
                    const double cr = a0x * dy - a0y * dx;
                    const bool opposite = cr == 0. && a0x * dx + a0y * dy < 0.;
                    if ((cr > 0. || opposite) && (jb < 0 || bxx * dy - byy * dx > 0.)) { jb = p; bxx = dx; byy = dy; }
                    if ((cr < 0. || opposite) && (jc < 0 || cxx * dy - cyy * dx < 0.)) { jc = p; cxx = dx; cyy = dy; }
                }
            }
            if (jb >= 0 && jc >= 0 && bxx * cyy - byy * cxx > 0.) { ia = na; ib = jb; ic = jc; }
        }
    }
    int rc = 1;
    double val = nanv;
    if (ia >= 0) rc = settle_and_interpolate<false>(g, sx, sy, sv, start, qx, qy, ia, ib, ic, &val, cub);
    if (rc == 1) {
        out[iq] = nanv;
        slow[1 + atomicAdd(slow, 1u)] = (unsigned)iq;
        return;
    }
    out[iq] = val;
    if (rc == 2) { atomicAdd(nfail, 1ull); atomicAdd(nfail + 3, 1ull); }
}

// One CTA per deferred query: a start triangle from a pass over ALL points -- with a = the first point as the zero
// direction, b = the point turned farthest counter-clockwise (by less than pi) and c = farthest clockwise: if b and c
// are less than pi apart on the far side the triangle a, b, c holds q, otherwise an empty half-plane through q exists
// and q is outside the hull -- then the same pivoting with the scans dealt out to the threads.  (The deferred queries
// are few, so what counts is the latency of ONE of them: 256 threads with eight loads in flight each.)
__global__ void __launch_bounds__(GI_COOP_THREADS)
k_griddata_warp(const double *__restrict__ sx, const double *__restrict__ sy, const double *__restrict__ sv,
                const int *__restrict__ start, const GridCells *__restrict__ gp, const double *__restrict__ qxs,
                const double *__restrict__ qys, double *__restrict__ out, unsigned long long *__restrict__ nfail,
                const unsigned *__restrict__ slow, const Cubic cub)
{
    const GridCells &g = *gp;
    const unsigned nslow = slow[0];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
    const double nanv = __longlong_as_double(0x7ff8000000000000ll);
    const int np = start[g.gx * g.gy];
    __shared__ int s_jb[32], s_jc[32], s_rc;
    __shared__ double s_bx[32], s_by[32], s_cx[32], s_cy[32];
    for (unsigned w = blockIdx.x; w < nslow; w += gridDim.x) {
        const int64_t iq = slow[1 + w];
        const double qx = qxs[iq], qy = qys[iq];
        const double a0x = sx[0] - qx, a0y = sy[0] - qy;
        int jb = -1, jc = -1;
        double bxx = 0., byy = 0., cxx = 0., cyy = 0.;
        for (int p0 = 1 + tid; p0 < np; p0 += (int)blockDim.x * GI_ILP) {
            double xs[GI_ILP], ys[GI_ILP];
#pragma unroll
            for (int u = 0; u < GI_ILP; u++) {
                const int p = p0 + (int)blockDim.x * u;
                xs[u] = p < np ? sx[p] : qx; ys[u] = p < np ? sy[p] : qy;
            }
#pragma unroll
            for (int u = 0; u < GI_ILP; u++) {
                const int p = p0 + (int)blockDim.x * u;
                if (p >= np) break;
                const double dx = xs[u] - qx, dy = ys[u] - qy;
                const double cr = a0x * dy - a0y * dx;                   // > 0: counter-clockwise of a
                const bool opposite = cr == 0. && a0x * dx + a0y * dy < 0.;   // (a point exactly opposite counts on both sides)
                if ((cr > 0. || opposite) && (jb < 0 || bxx * dy - byy * dx > 0.)) { jb = p; bxx = dx; byy = dy; }
                if ((cr < 0. || opposite) && (jc < 0 || cxx * dy - cyy * dx < 0.)) { jc = p; cxx = dx; cyy = dy; }
            }
        }
        // (the same direction from two threads: the lower index, so that all of them keep the same point)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const int ob = __shfl_xor_sync(0xffffffffu, jb, o), oc = __shfl_xor_sync(0xffffffffu, jc, o);
            const double obx = __shfl_xor_sync(0xffffffffu, bxx, o), oby = __shfl_xor_sync(0xffffffffu, byy, o);
            const double ocx = __shfl_xor_sync(0xffffffffu, cxx, o), ocy = __shfl_xor_sync(0xffffffffu, cyy, o);
            if (ob >= 0) {
                const double t = bxx * oby - byy * obx;
                if (jb < 0 || t > 0. || (t == 0. && ob < jb)) { jb = ob; bxx = obx; byy = oby; }
            }
            if (oc >= 0) {
                const double t = cxx * ocy - cyy * ocx;
                if (jc < 0 || t < 0. || (t == 0. && oc < jc)) { jc = oc; cxx = ocx; cyy = ocy; }
            }
        }
        if (lane == 0) { s_jb[warp] = jb; s_bx[warp] = bxx; s_by[warp] = byy; s_jc[warp] = jc; s_cx[warp] = cxx; s_cy[warp] = cyy; }
        __syncthreads();
        jb = -1; jc = -1;
        for (int k = 0; k < nwarp; k++) {
            if (s_jb[k] >= 0) {
                const double t = bxx * s_by[k] - byy * s_bx[k];
                if (jb < 0 || t > 0. || (t == 0. && s_jb[k] < jb)) { jb = s_jb[k]; bxx = s_bx[k]; byy = s_by[k]; }
            }
            if (s_jc[k] >= 0) {
                const double t = cxx * s_cy[k] - cyy * s_cx[k];
                if (jc < 0 || t < 0. || (t == 0. && s_jc[k] < jc)) { jc = s_jc[k]; cxx = s_cx[k]; cyy = s_cy[k]; }
            }
        }
        __syncthreads();
        // b counter-clockwise to c through the far side is less than pi  <=>  c is counter-clockwise of b
        if (jb < 0 || jc < 0 || !(bxx * cyy - byy * cxx > 0.)) { if (tid == 0) out[iq] = nanv; continue; }
        double val = nanv;
        const int rc = settle_and_interpolate<true>(g, sx, sy, sv, start, qx, qy, 0, jb, jc, &val, cub);
        if (tid == 0) s_rc = rc;
        __syncthreads();
        if (tid == 0) {
            out[iq] = val;
            if (s_rc) { atomicAdd(nfail, 1ull); atomicAdd(nfail + 3, 1ull); }
        }
        __syncthreads();
    }
}

// analyses.py:219-226 (polar=True): rho, rho*arctan2(y,x), rho*arctan2(x,y)
__global__ void __launch_bounds__(256)
k_polar_coords(const double *__restrict__ x, const double *__restrict__ y, int64_t num, double *__restrict__ rho,
               double *__restrict__ az1, double *__restrict__ az2)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < num; i += (int64_t)gridDim.x * blockDim.x) {
        const double a = x[i], b = y[i];
        const double r = sqrt(a * a + b * b);
        rho[i] = r;
        az1[i] = atan2(b, a) * r;
        az2[i] = atan2(a, b) * r;
    }
}

// np.nanmedian([a, b], axis=0): the mean of two numbers, the other one if one is NaN (analyses.py:227)
__global__ void __launch_bounds__(256)
k_nanmedian2(const double *__restrict__ a, const double *__restrict__ b, int64_t num, double *__restrict__ out)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < num; i += (int64_t)gridDim.x * blockDim.x) {
        const double u = a[i], v = b[i];
        out[i] = u != u ? v : (v != v ? u : (u + v) / 2.);      // numpy's mean of the two: (u+v)/2
    }
}

static size_t a256(size_t v) { return (v + 255) & ~(size_t)255; }
#define GI_QUERY_BATCH (1 << 22)                          // queries per launch pair (bounds the deferred list)
// the deferred list holds query indices of one batch or, for 'cubic', vertex indices: sized for the larger
static size_t slow_cap_bytes(size_t n) { return (((n > (size_t)GI_QUERY_BATCH ? n : (size_t)GI_QUERY_BATCH) + 64) * 4 + 255) & ~(size_t)255; }
#define GI_MAX_CELLS (1 << 24)
#define GI_BBOX_BLOCKS 512
#define GI_MAX_LEVELS 65536

// the scratch buffer of pxf_griddata / pxf_delaunay_neighbors, carved up
struct InterpScratch {
    double *key, *skey, *sx, *sy, *sv, *part, *spart, *grad;
    long long *perm, *lorder;   // lorder: the vertices sorted by Gauss-Seidel level
    int *start, *level, *flag, *nxt, *prv, *lstart;   // flag[0]: levels changed, flag[1]: highest level, flag[2..3]: the sweep's error
    GridCells *g;
    unsigned long long *nfail;
    unsigned *slow;
    Rings R;
    void *sort_scr;
    size_t cells;
};

static size_t interp_cells(size_t n)
{
    const size_t cells = n / 2 + 2;
    return cells > GI_MAX_CELLS ? GI_MAX_CELLS : cells;
}

static InterpScratch interp_carve(void *scratch, size_t n)
{
    InterpScratch w;
    w.cells = interp_cells(n);
    char *p = static_cast<char *>(scratch);
    w.key = (double *)p; p += a256(n * 8);
    w.skey = (double *)p; p += a256(n * 8);
    w.perm = (long long *)p; p += a256(n * 8);
    w.sx = (double *)p; p += a256(n * 8);
    w.sy = (double *)p; p += a256(n * 8);
    w.sv = (double *)p; p += a256(n * 8);
    w.start = (int *)p; p += a256((w.cells + 2) * 4);
    w.nxt = (int *)p; p += a256((w.cells + 2) * 4);
    w.prv = (int *)p; p += a256((w.cells + 2) * 4);
    w.part = (double *)p; p += a256(GI_BBOX_BLOCKS * 4 * 8);
    w.g = (GridCells *)p; p += a256(sizeof(GridCells));
    w.nfail = (unsigned long long *)p; p += 256;
    w.spart = (double *)p; p += a256(GI_NDIR * GI_DIR_SLICES * 8);
    w.slow = (unsigned *)p; p += slow_cap_bytes(n);
    w.R.ring = (int *)p; p += a256(n * GI_DEG * 4);
    w.R.deg = (unsigned char *)p; p += a256(n);
    w.R.open = (unsigned char *)p; p += a256(n);
    w.level = (int *)p; p += a256(n * 4);
    w.grad = (double *)p; p += a256(n * 16);
    w.flag = (int *)p; p += 256;
    w.lorder = (long long *)p; p += a256(n * 8);
    w.lstart = (int *)p; p += a256((GI_MAX_LEVELS + 4) * 4);
    w.sort_scr = p;
    return w;
}

// bounding box, support function and cell grid of the points; the points (and their values) in cell order
static int interp_bin(const InterpScratch &w, const double *x, const double *y, const double *v, int64_t num, pxf_stream_t stream)
{
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int nb = grid_for(num, 256 * 4, 4) < GI_BBOX_BLOCKS ? grid_for(num, 256 * 4, 4) : GI_BBOX_BLOCKS;
    PXF_CUDA(cudaMemsetAsync(w.nfail, 0, 32, s));
    k_bbox_partial<<<nb, 256, 0, s>>>(x, y, num, w.part);
    k_support_partial<<<GI_NDIR * GI_DIR_SLICES, 256, 0, s>>>(x, y, num, w.spart);
    k_grid_setup<<<1, 64, 0, s>>>(w.part, nb, num, (int)(w.cells - 2), w.g, w.spart);
    k_cell_keys<<<grid_for(num, 256, 8), 256, 0, s>>>(x, y, num, w.g, w.key);
    count_launch(4);
    const int rc = pxf_argsort(w.key, num, w.skey, reinterpret_cast<int64_t *>(w.perm), w.sort_scr, stream);
    if (rc) return rc;
    k_cell_starts<<<grid_for(num, 256, 8), 256, 0, s>>>(w.skey, w.perm, num, w.g, x, y, v, w.start, w.sx, w.sy, w.sv);
    count_launch();
    return check_launch("interp_bin");
}

// the Delaunay neighbour rings of the binned points
static int interp_rings(const InterpScratch &w, int64_t num, cudaStream_t s)
{
    PXF_CUDA(cudaMemsetAsync(w.slow, 0, 4, s));
    k_dt_rings<<<(unsigned)((num + GI_THREADS - 1) / GI_THREADS), GI_THREADS, 0, s>>>(w.sx, w.sy, w.start, w.g, (int)num, w.R, w.nfail,
                                                                                       w.slow, GI_RQ_DT);
    k_dt_rings_warp<<<grid_for(num, 1, 4), GI_COOP_THREADS, 0, s>>>(w.sx, w.sy, w.start, w.g, (int)num, w.R, w.nfail, w.slow);
    count_launch(2);
    unsigned long long hf[4] = {0, 0, 0, 0};
    PXF_CUDA(cudaMemcpyAsync(hf, w.nfail, 32, cudaMemcpyDeviceToHost, s));
    PXF_CUDA(cudaStreamSynchronize(s));
    if (hf[0]) {
        set_error("%llu points have no Delaunay neighbour ring (duplicate points, or more than %d neighbours)", hf[0], GI_DEG);
        return PXF_ERR_UNSUPPORTED;
    }
    return PXF_OK;
}

}  // namespace pxf

using namespace pxf;

extern "C" {

size_t pxf_griddata_scratch_bytes(int64_t num)
{
    const size_t n = (size_t)(num > 0 ? num : 1);
    char probe[1];                                           // (only the offsets are used)
    const InterpScratch w = interp_carve(probe, n);
    return (size_t)((char *)w.sort_scr - probe) + pxf_sort_scratch_bytes(num) + 1024;
}

int pxf_griddata(const double *x, const double *y, const double *v, int64_t num, const double *qx, const double *qy,
                 double *out, int64_t nq, int32_t method, int64_t *nfail_host, void *scratch, pxf_stream_t stream)
{
    if (num < 0 || nq < 0 || !x || !y || !v || !scratch || (nq > 0 && (!qx || !qy || !out)) || method < 0 || method > 2 ||
        num > 0x7fffffffll) {
        set_error("pxf_griddata: bad argument");
        return PXF_ERR_INVALID;
    }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    if (nfail_host) *nfail_host = 0;
    if (nq == 0) return PXF_OK;
    if (num < (method >= 1 ? 3 : 1)) { set_error("pxf_griddata: needs at least %d points", method >= 1 ? 3 : 1); return PXF_ERR_INVALID; }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const size_t n = (size_t)num;
    const InterpScratch w = interp_carve(scratch, n);
    int rc = interp_bin(w, x, y, v, num, stream);
    if (rc) return rc;
    double *const sx = w.sx, *const sy = w.sy, *const sv = w.sv, *const grad = w.grad;
    int *const start = w.start, *const level = w.level, *const flag = w.flag;
    GridCells *const g = w.g;
    unsigned long long *const nfail = w.nfail;
    unsigned *const slow = w.slow;
    const long long *const perm = w.perm;
    const Rings R = w.R;
    Cubic cub;
    cub.grad = nullptr; cub.R = R; cub.nxt = w.nxt; cub.prv = w.prv;
    if (method == 2) {
        // (a) the Delaunay neighbour rings
        if ((rc = interp_rings(w, num, s))) { if (nfail_host) *nfail_host = 1; return rc; }
        // (b) levels of the input-order Gauss-Seidel sweep, then the sweeps (scipy: maxiter 400, tol 1e-6)
        const unsigned vb = (unsigned)((num + 255) / 256);
        PXF_CUDA(cudaMemsetAsync(level, 0, n * 4, s));
        PXF_CUDA(cudaMemsetAsync(grad, 0, n * 16, s));
        int nlev = 0;
        PXF_CUDA(cudaMemsetAsync(flag, 0, 8, s));
        for (int it = 0;; it++) {
            if (it > 1 << 20) { set_error("pxf_griddata: the Gauss-Seidel levels did not settle"); return PXF_ERR_UNSUPPORTED; }
            int h[2] = {0, 0};
            PXF_CUDA(cudaMemsetAsync(flag, 0, 4, s));
            k_gs_levels<<<vb, 256, 0, s>>>(R, perm, (int)num, level, flag);
            count_launch();
            PXF_CUDA(cudaMemcpyAsync(h, flag, 8, cudaMemcpyDeviceToHost, s));
            PXF_CUDA(cudaStreamSynchronize(s));
            nlev = h[1];                       // the highest level assigned
            if (!h[0]) break;
        }
        if (nlev > GI_MAX_LEVELS) { set_error("pxf_griddata: the input order gives %d Gauss-Seidel levels", nlev); return PXF_ERR_UNSUPPORTED; }
        // the vertices bucketed by level (a sort by level: the binning's key / sorted-key / sort scratch are free again), so
        // that a level's launch touches its own vertices only
        k_level_keys<<<vb, 256, 0, s>>>(level, (int)num, w.key);
        count_launch();
        if ((rc = pxf_argsort(w.key, num, w.skey, reinterpret_cast<int64_t *>(w.lorder), w.sort_scr, stream))) return rc;
        k_level_starts<<<vb, 256, 0, s>>>(w.skey, (int)num, nlev, w.lstart);
        count_launch();
        std::vector<int> lstart((size_t)nlev + 2);
        PXF_CUDA(cudaMemcpyAsync(lstart.data(), w.lstart, lstart.size() * 4, cudaMemcpyDeviceToHost, s));
        PXF_CUDA(cudaStreamSynchronize(s));
        unsigned long long *err = reinterpret_cast<unsigned long long *>(flag + 2);
        for (int sweep = 0; sweep < 400; sweep++) {
            PXF_CUDA(cudaMemsetAsync(err, 0, 8, s));
            for (int lv = 0; lv <= nlev; lv++) {
                const int cnt = lstart[lv + 1] - lstart[lv];
                if (cnt <= 0) continue;
                k_gs_update<<<(unsigned)((cnt + 255) / 256), 256, 0, s>>>(R, sx, sy, sv, w.lorder + lstart[lv], cnt, grad, err);
            }
            count_launch(nlev + 1);
            unsigned long long he = 0;
            PXF_CUDA(cudaMemcpyAsync(&he, err, 8, cudaMemcpyDeviceToHost, s));
            PXF_CUDA(cudaStreamSynchronize(s));
            double e;
            memcpy(&e, &he, 8);
            if (e < 1e-6) break;
        }
        cub.grad = grad;
    }
    for (int64_t q0 = 0; q0 < nq; q0 += GI_QUERY_BATCH) {
        const int64_t nb_q = nq - q0 < GI_QUERY_BATCH ? nq - q0 : GI_QUERY_BATCH;
        const unsigned qb = (unsigned)((nb_q + GI_THREADS - 1) / GI_THREADS);
        if (method == 0) {
            if (q0 == 0) {
                k_row_links<<<(unsigned)(((int)(w.cells) + 127) / 128), 128, 0, s>>>(start, g, w.nxt, w.prv);     // (one thread per row; rows <= cells)
                count_launch();
            }
            k_griddata<0><<<qb, GI_THREADS, 0, s>>>(sx, sy, sv, start, g, qx + q0, qy + q0, nb_q, out + q0, nfail, slow, cub);
            count_launch();
            continue;
        }
        PXF_CUDA(cudaMemsetAsync(slow, 0, 4, s));
        k_griddata<1><<<qb, GI_THREADS, 0, s>>>(sx, sy, sv, start, g, qx + q0, qy + q0, nb_q, out + q0, nfail, slow, cub);
        k_griddata_warp<<<grid_for(nb_q, 1, 4), GI_COOP_THREADS, 0, s>>>(sx, sy, sv, start, g, qx + q0, qy + q0, out + q0, nfail, slow, cub);
        count_launch(2);
    }
    if ((rc = check_launch("pxf_griddata"))) return rc;
    if (nfail_host) {
        unsigned long long h[4] = {0, 0, 0, 0};
        PXF_CUDA(cudaMemcpyAsync(h, nfail, 32, cudaMemcpyDeviceToHost, s));
        PXF_CUDA(cudaStreamSynchronize(s));
        *nfail_host = (int64_t)h[0];
        if (h[0])
            set_error("pxf_griddata: %llu queries unresolved (%llu: no start triangle, %llu: pivoting did not settle)", h[0], h[1],
                      h[3]);
    }
    return PXF_OK;
}

int pxf_bbox(const double *x, const double *y, int64_t num, double *box_host /*[4]: xmin, xmax, ymin, ymax*/, void *scratch,
             pxf_stream_t stream)
{
    if (num <= 0 || !x || !y || !box_host || !scratch) { set_error("pxf_bbox: bad argument"); return PXF_ERR_INVALID; }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    double *part = static_cast<double *>(scratch);
    const int nb = grid_for(num, 256 * 4, 4) < GI_BBOX_BLOCKS ? grid_for(num, 256 * 4, 4) : GI_BBOX_BLOCKS;
    k_bbox_partial<<<nb, 256, 0, s>>>(x, y, num, part);
    count_launch();
    int rc = check_launch("k_bbox_partial");
    if (rc) return rc;
    std::vector<double> h((size_t)nb * 4);
    PXF_CUDA(cudaMemcpyAsync(h.data(), part, h.size() * 8, cudaMemcpyDeviceToHost, s));
    PXF_CUDA(cudaStreamSynchronize(s));
    box_host[0] = h[0]; box_host[1] = h[1]; box_host[2] = h[2]; box_host[3] = h[3];
    for (int b = 1; b < nb; b++) {
        box_host[0] = fmin(box_host[0], h[4 * b]); box_host[1] = fmax(box_host[1], h[4 * b + 1]);
        box_host[2] = fmin(box_host[2], h[4 * b + 2]); box_host[3] = fmax(box_host[3], h[4 * b + 3]);
    }
    return PXF_OK;
}

size_t pxf_bbox_scratch_bytes(void) { return (size_t)GI_BBOX_BLOCKS * 4 * 8; }

int pxf_polar_coords(const double *x, const double *y, int64_t num, double *rho, double *az1, double *az2, pxf_stream_t stream)
{
    if (num < 0 || (num > 0 && (!x || !y || !rho || !az1 || !az2))) { set_error("pxf_polar_coords: bad argument"); return PXF_ERR_INVALID; }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    if (num == 0) return PXF_OK;
    k_polar_coords<<<grid_for(num, 256, 8), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, y, num, rho, az1, az2);
    count_launch();
    return check_launch("k_polar_coords");
}

int pxf_nanmedian2(const double *a, const double *b, int64_t num, double *out, pxf_stream_t stream)
{
    if (num < 0 || (num > 0 && (!a || !b || !out))) { set_error("pxf_nanmedian2: bad argument"); return PXF_ERR_INVALID; }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    if (num == 0) return PXF_OK;
    k_nanmedian2<<<grid_for(num, 256, 8), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a, b, num, out);
    count_launch();
    return check_launch("k_nanmedian2");
}

int pxf_delaunay_max_degree(void) { return GI_DEG; }

int pxf_delaunay_neighbors(const double *x, const double *y, int64_t num, int32_t *ring_out, uint8_t *deg_out,
                           uint8_t *open_out, void *scratch, pxf_stream_t stream)
{
    if (num < 3 || !x || !y || !ring_out || !deg_out || !open_out || !scratch || num > 0x7fffffffll) {
        set_error("pxf_delaunay_neighbors: bad argument");
        return PXF_ERR_INVALID;
    }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const InterpScratch w = interp_carve(scratch, (size_t)num);
    int rc = interp_bin(w, x, y, x, num, stream);
    if (rc) return rc;
    if ((rc = interp_rings(w, num, s))) return rc;
    k_rings_export<<<(unsigned)((num + 255) / 256), 256, 0, s>>>(w.R, w.perm, (int)num, ring_out, deg_out, open_out);
    count_launch();
    if ((rc = check_launch("pxf_delaunay_neighbors"))) return rc;
    return PXF_OK;
}

}  // extern "C"
