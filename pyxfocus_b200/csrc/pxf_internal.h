// Internal helpers shared by the libpxf translation units (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/pxf.h"

#ifndef PXF_NEWTON_CAP
#define PXF_NEWTON_CAP 1000
#endif
#define PXF_BLOCK 256

namespace pxf {

void set_error(const char *fmt, ...);
void count_launch(int n = 1);
int sm_count();
int opt_ws_libm();      // PXF_OPT_WS_LIBM
int opt_ws_retrace();   // PXF_OPT_WS_RETRACE
int opt_ws_graze_ppm(); // PXF_OPT_WS_GRAZE_PPM

// Per-device one-time guard: function attributes (cudaFuncSetAttribute) belong to a device's primary context, so
// a process that works on cuda:0 and then on cuda:1 has to set them again there.  `seen` is a zero-initialised
// static array at the call site; true exactly once per device.
inline bool first_on_device(bool (&seen)[64])
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return true; }
    if (seen[dev]) return false;
    seen[dev] = true;
    return true;
}

// Persistent grid: SM count x resident CTAs, capped by the work available.
int grid_for(int64_t work_items, int per_block, int ctas_per_sm);

// Weighted HPD of every segment of a segmented bundle (pxf_sort.cu; the entry point is pxf_hpd_segmented).
size_t hpd_weighted_segmented_bytes(int64_t num);
int hpd_weighted_segmented(const double *x, const double *y, const double *w, int64_t num, const long long *seg_start,
                           int nseg, const double *sums, double *out, void *workspace, cudaStream_t s);

inline int check_launch(const char *what)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return PXF_ERR_CUDA;
    }
    return PXF_OK;
}

#define PXF_CUDA(call)                                                        \
    do {                                                                      \
        cudaError_t e__ = (call);                                             \
        if (e__ != cudaSuccess) {                                             \
            pxf::set_error("%s: %s", #call, cudaGetErrorString(e__));         \
            return PXF_ERR_CUDA;                                              \
        }                                                                     \
    } while (0)

// Stream-ordered scratch allocation for the convenience entry points.
struct Scratch {
    void *p = nullptr;
    cudaStream_t s = nullptr;
    int alloc(size_t bytes, cudaStream_t stream);
    ~Scratch();
};

}  // namespace pxf
