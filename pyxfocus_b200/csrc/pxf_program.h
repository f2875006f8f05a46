// Fused-program representation shared by pxf_fused.cu (kernel + builder) and pxf_host.cu
// (host-buffer streaming entry point).  Not part of the ABI.
#pragma once
#include "pxf_internal.h"
#include "pxf_params.h"
#include "pxf_rows.cuh"

namespace pxf {

#define FOP_PARAM_DOUBLES 38   // sizeof(WSP)/8 is the largest folded parameter block
#define PXF_PROG_MAX_LL 2      // Legendre-Legendre shells per program: a deformed primary and secondary

struct FusedOp {
    int code;
    int row;                 // VIGNETTE_BOX / ABS: bundle row index; LLSURF: table slot
    double q[FOP_PARAM_DOUBLES];
};
struct FusedProgram {
    int nops;
    unsigned load_mask, store_mask;
    int has_vignette;
    // rows whose final value is the same known constant for every ray (e.g. z = 0 and the normal
    // (0,0,1) after a closing `flat`): the host-buffer entry point fills them on the host instead
    // of downloading them.  Empty when the program can stop rays early (vignette predicates).
    unsigned const_mask;
    double const_val[10];
    const ZernP *zern;       // device table of the program's PXF_OP_ZERNSURF or ZERNPHASE op (NULL: none); staged in shared memory
    // per-ray side arrays (pxf_program_aux): wavelengths / grating counts of PXF_OP_GRATFAN, PXF_OP_ROTX_REMAINING
    const double *aux_wave;
    int *aux_count;
    int *aux_count_max;
    int uses_aux;            // some op reads or writes a side array (needs the ray index)
    FusedOp ops[PXF_MAX_OPS];
    // device tables of the program's PXF_OP_LLSURF ops in op order (FusedOp::row = slot); staged in shared memory
    const LLTab *ll[PXF_PROG_MAX_LL];
    int nll;
    int surf;                // some op is one of the remaining scalar surfaces (PXF_OP_TRACESPHERE .. WSSECONDARYBACK)
};

static_assert(sizeof(WSP) <= FOP_PARAM_DOUBLES * 8, "WSP does not fit a fused op slot");
static_assert(sizeof(GratFanP) <= FOP_PARAM_DOUBLES * 8, "GratFanP does not fit a fused op slot");
static_assert(sizeof(ConicP) <= FOP_PARAM_DOUBLES * 8, "ConicP does not fit");
static_assert(sizeof(WolterSineP) <= FOP_PARAM_DOUBLES * 8, "WolterSineP does not fit");

// pxf_fused.cu
int build_program(FusedProgram &fp, const pxf_op *ops, int nops, const pxf_program_aux *aux = nullptr);
// partials (nullable): device double[grid*9] receiving the per-CTA centroid sums; *grid_out = CTAs launched
int launch_program(double *const rays[10], int64_t num, const FusedProgram &fp, uint8_t *alive, cudaStream_t s,
                   double *const rays_out[10] = nullptr, double *partials = nullptr, int *grid_out = nullptr);
// pxf_chain.cu: statically specialised kernels for the reference's canonical chains.  Returns
// PXF_OK after launching, PXF_ERR_UNSUPPORTED when no specialisation matches the op list.
int launch_chain(const RowPtrs &P, const RowPtrs &Q, int64_t num, const FusedProgram &fp, uint8_t *alive,
                 bool aligned, cudaStream_t s, double *partials, int *grid_out);

// pxf_jit.cu: run-time specialisation (NVRTC) of any op list; PXF_ERR_UNSUPPORTED = not available, use the interpreter
int jit_launch_chain(const RowPtrs &P, const RowPtrs &Q, int64_t num, const FusedProgram &fp, uint8_t *alive,
                     bool aligned, cudaStream_t s, double *partials, int *grid_out);
size_t jit_seg_pack_bytes(int nops);
size_t jit_seg_fill(const FusedOp *ops, int nops, int nseg, void *dst);     // returns bytes per segment pack, 0 = none
int jit_seg_launch(const FusedOp *ops0, int nops, const RowPtrs &P, const RowPtrs &Q, int64_t num, uint8_t *alive,
                   const long long *seg_start_dev, const void *packs_dev, int nseg, unsigned LM, unsigned SM,
                   const ZernP *zern_dev, const LLTab *ll_dev, cudaStream_t s);
                   // zern_dev: one Zernike table per segment, ll_dev: the segment's LL tables, segment-major (NULL: none)
void note_kernel(const char *name);     // name of the last trace kernel launched (pxf_last_trace_kernel)

// segmented specialised chains (pxf_chain.cu)
size_t seg_chain_bytes(int nseg);
int seg_chain_fill(const FusedOp *ops, int nops, int nseg, void *dst);
int seg_chain_launch(int chain_id, const RowPtrs &P, const RowPtrs &Q, int64_t num, uint8_t *alive,
                     const long long *seg_start_dev, const void *table_dev, int nseg, unsigned LM, unsigned SM,
                     cudaStream_t s);

}  // namespace pxf
