// Run-time specialisation of fused programs.
//
// The interpreter (pxf_fused.cu) pays for its generality: an opcode switch per op and ray, parameters fetched
// through an op-indexed constant bank, a register allocation that is the maximum over every op in the library
// (i-cache misses dominate its stall profile, profiles/r01h_k_program_zern.txt).  pxf_chain.cu removes all of that
// for a handful of op lists known when the library is built.  This file does it for EVERY op list: the recorded
// list is turned into  Chain<COp1, COp2, ...>  (pxf_chain_ops.cuh -- the same per-op device functions, so the result
// is bit-identical to the interpreter and to the per-routine kernels), compiled with NVRTC for sm_100a with the
// library's own arithmetic flags (-fmad=false -prec-div -prec-sqrt), cached by signature in memory and as a cubin
// under <libpxf dir>/_jit/, loaded with cudaLibraryLoadData and launched with cudaLaunchKernel.
//
// libnvrtc is opened with dlopen at first use; when it is missing, or a compilation fails, the caller falls back to
// the interpreter (still on the GPU) and the reason is kept in pxf_jit_status().
#include <dlfcn.h>
#include <nvrtc.h>
#include <stdlib.h>
#include <sys/stat.h>
#include <unistd.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "pxf_program.h"
#include "pxf_chain_ops.cuh"

namespace pxf {

// ---------------------------------------------------------------- op table
struct OpDesc { int code; const char *name; size_t bytes; bool row; };
static const OpDesc OPS[] = {
    {PXF_OP_TRANSFORM, "CTransform", sizeof(CTransform::P), false},
    {PXF_OP_ITRANSFORM, "CITransform", sizeof(CITransform::P), false},
    {PXF_OP_REFLECT, "CReflect", sizeof(CReflect::P), false},
    {PXF_OP_REFRACT, "CRefract", sizeof(CRefract::P), false},
    {PXF_OP_RADGRAT, "CRadgrat", sizeof(CRadgrat::P), false},
    {PXF_OP_FLAT, "CFlat", sizeof(CFlat::P), false},
    {PXF_OP_FLATOPD, "CFlatOpd", sizeof(CFlatOpd::P), false},
    {PXF_OP_CONIC, "CConic", sizeof(CConic::P), false},
    {PXF_OP_CONICOPD, "CConicOpd", sizeof(CConicOpd::P), false},
    {PXF_OP_WOLTERPRIMARY, "CWolterPrimary", sizeof(CWolterPrimary::P), false},
    {PXF_OP_WOLTERPRIMARYOPD, "CWolterPrimaryOpd", sizeof(CWolterPrimaryOpd::P), false},
    {PXF_OP_WOLTERSECONDARY, "CWolterSecondary", sizeof(CWolterSecondary::P), false},
    {PXF_OP_WOLTERSINE, "CWolterSine", sizeof(CWolterSine::P), false},
    {PXF_OP_WSPRIMARY, "CWsPrimary", sizeof(CWsPrimary::P), false},
    {PXF_OP_WSSECONDARY, "CWsSecondary", sizeof(CWsSecondary::P), false},
    {PXF_OP_SPOCONE, "CSpoCone", sizeof(CSpoCone::P), false},
    {PXF_OP_VIGNETTE_MAG, "CVignetteMag", sizeof(CVignetteMag::P), false},
    {PXF_OP_VIGNETTE_BOX, "CVignetteBox", sizeof(VigBoxP), true},
    {PXF_OP_VIGNETTE_ABS, "CVignetteAbs", sizeof(VigAbsP), true},
    {PXF_OP_KICK, "CKick", sizeof(CKick::P), false},
    {PXF_OP_ZERNSURF, "CZernSurf", sizeof(CZernSurf::P), false},
    {PXF_OP_KICKN, "CKickN", sizeof(CKickN::P), false},
    {PXF_OP_VIGNETTE_RHOGT, "CVignetteRhoGt", sizeof(CVignetteRhoGt::P), false},
    {PXF_OP_GRATFAN, "CGratFan", sizeof(CGratFan::P), false},
    {PXF_OP_ROTX_REMAINING, "CRotxRemaining", sizeof(CRotxRemaining::P), false},
    {PXF_OP_LLSURF, "CLLSurf", sizeof(LLOpP), false},
    {PXF_OP_TRACESPHERE, "CTraceSphere", sizeof(CTraceSphere::P), false},
    {PXF_OP_TRACESPHEREOPD, "CTraceSphereOpd", sizeof(CTraceSphereOpd::P), false},
    {PXF_OP_TRACECYL, "CTraceCyl", sizeof(CTraceCyl::P), false},
    {PXF_OP_TRACECYLOPD, "CTraceCylOpd", sizeof(CTraceCylOpd::P), false},
    {PXF_OP_CYLCONIC, "CCylConic", sizeof(CCylConic::P), false},
    {PXF_OP_PARAXIAL, "CParaxial", sizeof(CParaxial::P), false},
    {PXF_OP_PARAXIALY, "CParaxialY", sizeof(CParaxialY::P), false},
    {PXF_OP_TORUS, "CTorus", sizeof(CTorus::P), false},
    {PXF_OP_WSPRIMARYBACK, "CWsPrimaryBack", sizeof(CWsPrimaryBack::P), false},
    {PXF_OP_WSSECONDARYBACK, "CWsSecondaryBack", sizeof(CWsSecondaryBack::P), false},
    {PXF_OP_ZERNPHASE, "CZernPhase", sizeof(CZernPhase::P), false},
    {PXF_OP_CONICPLUS, "CConicPlus", sizeof(CConicPlus::P), false},
    {PXF_OP_CONICPLUSOPD, "CConicPlusOpd", sizeof(CConicPlusOpd::P), false},
    {PXF_OP_LEGSURF, "CLegSurf", sizeof(CLegSurf::P), false},
    {PXF_OP_RADGRATW, "CRadgratW", sizeof(CRadgratW::P), false},
    {PXF_OP_GRAT, "CGrat", sizeof(CGrat::P), false},
};
static const OpDesc *op_desc(int code)
{
    for (const OpDesc &d : OPS)
        if (d.code == code) return &d;
    return nullptr;
}

// ---------------------------------------------------------------- small utilities
static uint64_t fnv1a(const void *data, size_t n, uint64_t h = 1469598103934665603ull)
{
    const unsigned char *p = static_cast<const unsigned char *>(data);
    for (size_t i = 0; i < n; i++) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}
static bool read_file(const std::string &path, std::vector<char> &out)
{
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) return false;
    fseek(f, 0, SEEK_END);
    long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    out.resize(n > 0 ? (size_t)n : 0);
    bool ok = n >= 0 && fread(out.data(), 1, out.size(), f) == out.size();
    fclose(f);
    return ok;
}
static std::string lib_dir()
{
    Dl_info info;
    if (dladdr(reinterpret_cast<const void *>(&op_desc), &info) && info.dli_fname) {
        std::string p(info.dli_fname);
        size_t k = p.rfind('/');
        return k == std::string::npos ? std::string(".") : p.substr(0, k);
    }
    return ".";
}

static std::mutex g_mu;
static std::string g_status = "not used yet";
static void set_status(const std::string &s) { g_status = s; }

// ---------------------------------------------------------------- NVRTC through dlopen
struct Nvrtc {
    void *h = nullptr;
    nvrtcResult (*CreateProgram)(nvrtcProgram *, const char *, const char *, int, const char *const *, const char *const *) = nullptr;
    nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char *const *) = nullptr;
    nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t *) = nullptr;
    nvrtcResult (*GetCUBIN)(nvrtcProgram, char *) = nullptr;
    nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t *) = nullptr;
    nvrtcResult (*GetProgramLog)(nvrtcProgram, char *) = nullptr;
    nvrtcResult (*DestroyProgram)(nvrtcProgram *) = nullptr;
    bool tried = false, ok = false;
    bool load()
    {
        if (tried) return ok;
        tried = true;
        const char *names[] = {"libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12", "libnvrtc.so",
                               "/usr/local/cuda/lib64/libnvrtc.so"};
        for (const char *n : names) {
            h = dlopen(n, RTLD_NOW | RTLD_LOCAL);
            if (h) break;
        }
        if (!h) { set_status("libnvrtc not found: interpreter only"); return false; }
#define PXF_SYM(field, name) field = reinterpret_cast<decltype(field)>(dlsym(h, name)); if (!field) { set_status(std::string("libnvrtc lacks ") + name); return false; }
        PXF_SYM(CreateProgram, "nvrtcCreateProgram")
        PXF_SYM(CompileProgram, "nvrtcCompileProgram")
        PXF_SYM(GetCUBINSize, "nvrtcGetCUBINSize")
        PXF_SYM(GetCUBIN, "nvrtcGetCUBIN")
        PXF_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
        PXF_SYM(GetProgramLog, "nvrtcGetProgramLog")
        PXF_SYM(DestroyProgram, "nvrtcDestroyProgram")
#undef PXF_SYM
        ok = true;
        return true;
    }
};
static Nvrtc g_nvrtc;

// ---------------------------------------------------------------- signatures and source text
struct JitSpec {
    std::vector<int> codes;
    std::vector<std::string> targs;     // template arguments of each functor ("" / "<row>" / "<N, slot>")
    unsigned LM = 0, SM = 0;
    int mode = 2, minb = 3, nll = 0;
    bool zern = false, seg = false;
    size_t cp_bytes = 8;
    std::string chain_type() const
    {
        std::string t;
        for (size_t k = 0; k < codes.size(); k++) {
            const OpDesc *d = op_desc(codes[k]);
            if (k) t += ", ";
            t += d->name;
            t += targs[k];
        }
        return t;
    }
    std::string signature() const
    {
        char buf[112];
        snprintf(buf, sizeof(buf), "v4;seg%d;m%d;b%d;z%d;l%d;L%u;S%u;", seg ? 1 : 0, mode, minb, zern ? 1 : 0, nll, LM, SM);
        return std::string(buf) + chain_type();
    }
    std::string source() const
    {
        const std::string t = chain_type();
        std::string s = "#include \"pxf_chain_ops.cuh\"\nusing namespace pxf;\n";
        s += "typedef Chain<" + t + "> C;\ntypedef ChainP<" + t + "> CP;\n";
        char buf[1024];
        if (!seg) {
            snprintf(buf, sizeof(buf),
                     "extern \"C\" __global__ void __launch_bounds__(PXF_BLOCK, %d)\n"
                     "pxf_jit_chain(const RowPtrs P, const RowPtrs Q, const long long num, unsigned char *alive, double *partials,\n"
                     "              const ZernP *zern, const double *aux_wave, int *aux_count, int *aux_count_max,\n"
                     "              const LLTab *ll0, const LLTab *ll1, const __grid_constant__ CP prm)\n"
                     "{\n    chain_body<C, CP, %d, %s, %d, %uu, %uu>(P, Q, num, alive, partials, prm, zern, aux_wave, aux_count,\n"
                     "                                          aux_count_max, ll0, ll1);\n}\n",
                     minb, mode, zern ? "true" : "false", nll, LM, SM);
        } else {
            snprintf(buf, sizeof(buf),
                     "extern \"C\" __global__ void __launch_bounds__(PXF_BLOCK, %d)\n"
                     "pxf_jit_chain(const RowPtrs P, const RowPtrs Q, const long long num, unsigned char *alive,\n"
                     "              const long long *seg_start, const CP *table, const int nseg, const unsigned LM, const unsigned SM,\n"
                     "              const ZernP *zern, const LLTab *ll)\n"
                     "{\n    chain_seg_body<C, CP, %s, %d, %uu, %uu>(P, Q, num, alive, seg_start, table, nseg, LM, SM, zern, ll);\n}\n",
                     minb, zern ? "true" : "false", nll, LM, SM);
        }
        return s + buf;
    }
};

static bool spec_from_ops(const FusedOp *ops, int nops, JitSpec &sp)
{
    sp.codes.clear(); sp.targs.clear();
    sp.cp_bytes = 8;
    sp.zern = false;
    sp.nll = 0;
    for (int k = 0; k < nops; k++) {
        const OpDesc *d = op_desc(ops[k].code);
        if (!d) return false;
        sp.codes.push_back(ops[k].code);
        std::string ta;
        if (d->row) ta = "<" + std::to_string(ops[k].row) + ">";
        if (ops[k].code == PXF_OP_LLSURF) {
            ta = "<" + std::to_string((int)ops[k].q[0]) + ", " + std::to_string(ops[k].row) + ">";
            sp.nll++;
        }
        sp.targs.push_back(ta);
        sp.cp_bytes += d->bytes;
        if (ops[k].code == PXF_OP_ZERNSURF || ops[k].code == PXF_OP_ZERNPHASE) sp.zern = true;
    }
    return true;
}
static void pack_params(const FusedOp *ops, int nops, unsigned char *dst)
{
    size_t off = 0;
    for (int k = 0; k < nops; k++) {
        const OpDesc *d = op_desc(ops[k].code);
        memcpy(dst + off, ops[k].q, d->bytes);
        off += d->bytes;
    }
    memset(dst + off, 0, 8);
}

// ---------------------------------------------------------------- compile, cache, load
struct JitEntry {
    bool failed = false, loaded = false;
    std::vector<char> cubin;
    cudaLibrary_t lib = nullptr;
    cudaKernel_t kern = nullptr;
};
static std::map<std::string, JitEntry> g_cache;
static uint64_t g_stamp = 0;
static std::string g_src_dir, g_cache_dir;
static int64_t g_compiles = 0, g_disk_hits = 0;

static void init_paths()
{
    if (!g_src_dir.empty()) return;
    const std::string base = lib_dir();
    g_src_dir = base + "/csrc";
    const char *e = getenv("PXF_JIT_CACHE");
    g_cache_dir = e ? std::string(e) : base + "/_jit";
    // the cache is keyed by the CONTENT of the device headers: editing one invalidates every cubin
    uint64_t h = 1469598103934665603ull;
    for (const char *f : {"pxf_chain_ops.cuh", "pxf_rows.cuh", "pxf_ray.cuh", "pxf_crmath.cuh"}) {
        std::vector<char> txt;
        if (read_file(g_src_dir + "/" + f, txt)) h = fnv1a(txt.data(), txt.size(), h);
    }
    g_stamp = h;
}
static std::string cache_path(const std::string &sig)
{
    uint64_t h = fnv1a(sig.data(), sig.size(), g_stamp);
    char buf[40];
    snprintf(buf, sizeof(buf), "/%016llx.cubin", (unsigned long long)h);
    return g_cache_dir + buf;
}

// the cubin of a spec: memory cache, then disk, then NVRTC (compile == false: do not compile, report a miss)
static JitEntry *get_cubin(const JitSpec &sp, bool compile)
{
    init_paths();
    const std::string sig = sp.signature();
    JitEntry &e = g_cache[sig];
    if (e.failed || !e.cubin.empty()) return e.failed ? nullptr : &e;
    const std::string path = cache_path(sig);
    if (read_file(path, e.cubin) && !e.cubin.empty()) { g_disk_hits++; return &e; }
    e.cubin.clear();
    if (!compile) { g_cache.erase(sig); return nullptr; }
    if (!g_nvrtc.load()) { e.failed = true; return nullptr; }
    const std::string src = sp.source();
    nvrtcProgram prog;
    if (g_nvrtc.CreateProgram(&prog, src.c_str(), "pxf_jit_chain.cu", 0, nullptr, nullptr) != NVRTC_SUCCESS) {
        e.failed = true; set_status("nvrtcCreateProgram failed"); return nullptr;
    }
    const std::string inc = "--include-path=" + g_src_dir;
    const char *opts[] = {"--gpu-architecture=sm_100a", "--fmad=false", "--prec-div=true", "--prec-sqrt=true",
                          "--std=c++17", "-lineinfo", inc.c_str(), "-DPXF_BLOCK=256"};
    nvrtcResult rc = g_nvrtc.CompileProgram(prog, (int)(sizeof(opts) / sizeof(opts[0])), opts);
    if (rc != NVRTC_SUCCESS) {
        size_t n = 0;
        g_nvrtc.GetProgramLogSize(prog, &n);
        std::string log(n, '\0');
        if (n) g_nvrtc.GetProgramLog(prog, &log[0]);
        g_nvrtc.DestroyProgram(&prog);
        e.failed = true;
        set_status("NVRTC failed for " + sig + ": " + log.substr(0, 1500));
        if (getenv("PXF_JIT_VERBOSE")) fprintf(stderr, "[pxf jit] %s\n", g_status.c_str());
        return nullptr;
    }
    size_t n = 0;
    g_nvrtc.GetCUBINSize(prog, &n);
    e.cubin.resize(n);
    g_nvrtc.GetCUBIN(prog, e.cubin.data());
    g_nvrtc.DestroyProgram(&prog);
    g_compiles++;
    // best effort: keep it for the next process (and for the GPU box: the cache directory travels with the tree)
    mkdir(g_cache_dir.c_str(), 0755);
    const std::string tmp = path + ".tmp" + std::to_string((long)getpid());
    FILE *f = fopen(tmp.c_str(), "wb");
    if (f) {
        bool ok = fwrite(e.cubin.data(), 1, e.cubin.size(), f) == e.cubin.size();
        fclose(f);
        if (!ok || rename(tmp.c_str(), path.c_str()) != 0) unlink(tmp.c_str());
    }
    set_status("ok");
    return &e;
}

static JitEntry *get_kernel(const JitSpec &sp, bool compile)
{
    JitEntry *e = get_cubin(sp, compile);
    if (!e) return nullptr;
    if (!e->loaded) {
        if (cudaLibraryLoadData(&e->lib, e->cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0) != cudaSuccess ||
            cudaLibraryGetKernel(&e->kern, e->lib, "pxf_jit_chain") != cudaSuccess) {
            set_status(std::string("loading a specialised cubin failed: ") + cudaGetErrorString(cudaGetLastError()));
            e->failed = true;
            return nullptr;
        }
        e->loaded = true;
    }
    return e;
}

// PXF_JIT=0 disables; PXF_JIT_MIN_RAYS: smallest bundle worth a compilation (cached kernels are used at any size)
static bool jit_enabled()
{
    static int on = -1;
    if (on < 0) {
        const char *e = getenv("PXF_JIT");
        const char *n = getenv("PXF_NO_SPECIALIZE");
        on = ((e && e[0] == '0') || (n && n[0] == '1')) ? 0 : 1;
    }
    return on != 0;
}
static int64_t jit_min_rays()
{
    static int64_t v = -1;
    if (v < 0) { const char *e = getenv("PXF_JIT_MIN_RAYS"); v = e ? atoll(e) : 262144; }
    return v;
}

static char g_last_kernel[512] = "";
void note_kernel(const char *name) { snprintf(g_last_kernel, sizeof(g_last_kernel), "%s", name); }

// LL chains: 2 resident CTAs per SM.  ptxas, the LL pair: N = 5 needs 154 registers uncapped and spills 100 B at
// 2 CTAs/SM (692 B at 3); N = 7 needs 216 and spills 772 B at 2.  Measured at 5e7 rays on one B200 (1000 W): 4.9 /
// 7.1 / 13.0 ms for N = 3 / 5 / 7 (profiles/ll_program_bench_b200.json)
static const int LL_MINB = 2;

// Chains with a conicplus run one ray per thread: its Newton loop over up to 16 powers does not gain from a second ray
// in flight, and the pair costs registers.  The aspheric singlet of profiles/table_surface_ops_bench.py (sphere,
// conicplus with 8 terms, 5e7 rays) on one B200 (1000 W): 11.80 ms with two rays per thread, 8.68 ms with one, at
// 3 CTAs/SM; reading the conicplus block from shared memory or from a register copy instead of through L1 changed
// either by less than 1 %.
static bool has_conicplus(const FusedProgram &fp)
{
    for (int k = 0; k < fp.nops; k++)
        if (fp.ops[k].code == PXF_OP_CONICPLUS || fp.ops[k].code == PXF_OP_CONICPLUSOPD) return true;
    return false;
}

static void fill_spec(JitSpec &sp, const FusedProgram &fp, bool aligned)
{
    sp.LM = fp.load_mask; sp.SM = fp.store_mask;
    sp.seg = false;
    sp.mode = (aligned && !sp.zern && !sp.nll && !fp.uses_aux && !has_conicplus(fp)) ? 2 : 1;
    sp.minb = sp.nll ? LL_MINB : 3;
}

int jit_launch_chain(const RowPtrs &P, const RowPtrs &Q, int64_t num, const FusedProgram &fp, uint8_t *alive,
                     bool aligned, cudaStream_t s, double *partials, int *grid_out)
{
    if (!jit_enabled()) return PXF_ERR_UNSUPPORTED;
    std::lock_guard<std::mutex> lock(g_mu);
    JitSpec sp;
    if (!spec_from_ops(fp.ops, fp.nops, sp)) return PXF_ERR_UNSUPPORTED;
    fill_spec(sp, fp, aligned);
    JitEntry *e = get_kernel(sp, num >= jit_min_rays());
    if (!e) return PXF_ERR_UNSUPPORTED;
    std::vector<unsigned char> cp(sp.cp_bytes);
    pack_params(fp.ops, fp.nops, cp.data());
    const int64_t items = sp.mode >= 2 ? ((num + 1) >> 1) : num;
    const int grid = grid_for(items, PXF_BLOCK, sp.minb);
    if (grid_out) *grid_out = grid;
    long long n = num;
    const ZernP *zern = fp.zern;
    const double *aw = fp.aux_wave;
    int *ac = fp.aux_count, *acm = fp.aux_count_max;
    const LLTab *ll0 = fp.ll[0], *ll1 = fp.ll[1];
    void *args[] = {(void *)&P, (void *)&Q, &n, &alive, &partials, &zern, &aw, &ac, &acm, &ll0, &ll1, cp.data()};
    cudaError_t rc = cudaLaunchKernel(reinterpret_cast<const void *>(e->kern), dim3(grid), dim3(PXF_BLOCK), args, 0, s);
    if (rc != cudaSuccess) { set_error("specialised chain launch: %s", cudaGetErrorString(rc)); return PXF_ERR_CUDA; }
    count_launch();
    note_kernel(("pxf_jit_chain<Chain<" + sp.chain_type() + ">>").c_str());
    return check_launch("pxf_jit_chain");
}

// ---- segmented form: the per-segment parameter packs are built when the table is filled
// register cap (resident CTAs per SM): the Zernike form needs the budget of the fused Zernike kernel, the LL form
// that of the specialised LL chains
static int seg_minb(const JitSpec &sp) { return sp.zern ? 3 : sp.nll ? LL_MINB : 4; }
size_t jit_seg_pack_bytes(int nops) { return (size_t)nops * FOP_PARAM_DOUBLES * 8 + 8; }
size_t jit_seg_fill(const FusedOp *ops, int nops, int nseg, void *dst)
{
    JitSpec sp;
    if (!jit_enabled() || !spec_from_ops(ops, nops, sp)) return 0;
    unsigned char *out = static_cast<unsigned char *>(dst);
    for (int sgm = 0; sgm < nseg; sgm++) pack_params(ops + (size_t)sgm * nops, nops, out + (size_t)sgm * sp.cp_bytes);
    return sp.cp_bytes;
}
int jit_seg_launch(const FusedOp *ops0, int nops, const RowPtrs &P, const RowPtrs &Q, int64_t num, uint8_t *alive,
                   const long long *seg_start_dev, const void *packs_dev, int nseg, unsigned LM, unsigned SM,
                   const ZernP *zern_dev, const LLTab *ll_dev, cudaStream_t s)
{
    if (!jit_enabled()) return PXF_ERR_UNSUPPORTED;
    std::lock_guard<std::mutex> lock(g_mu);
    JitSpec sp;
    if (!spec_from_ops(ops0, nops, sp) || sp.zern != (zern_dev != nullptr) || (sp.nll > 0) != (ll_dev != nullptr))
        return PXF_ERR_UNSUPPORTED;
    sp.LM = LM; sp.SM = SM; sp.seg = true; sp.mode = 1; sp.minb = seg_minb(sp);
    JitEntry *e = get_kernel(sp, num >= jit_min_rays());
    if (!e) return PXF_ERR_UNSUPPORTED;
    const int grid = grid_for(num, CHAIN_SEG_TILE, sp.minb);
    long long n = num;
    void *args[] = {(void *)&P, (void *)&Q, &n, &alive, &seg_start_dev, &packs_dev, &nseg, &LM, &SM, &zern_dev, &ll_dev};
    cudaError_t rc = cudaLaunchKernel(reinterpret_cast<const void *>(e->kern), dim3(grid), dim3(PXF_BLOCK), args, 0, s);
    if (rc != cudaSuccess) { set_error("specialised segmented chain launch: %s", cudaGetErrorString(rc)); return PXF_ERR_CUDA; }
    count_launch();
    note_kernel(("pxf_jit_chain_seg<Chain<" + sp.chain_type() + ">>").c_str());
    return check_launch("pxf_jit_chain_seg");
}

// compile (no GPU needed) the kernels a program will want: in place and out of place, aligned rows, with and
// without the centroid sums' extra x,y loads; returns how many cubins are now available
int jit_precompile(const FusedProgram &fp0, bool segmented)
{
    std::lock_guard<std::mutex> lock(g_mu);
    int have = 0;
    JitSpec sp;
    if (!spec_from_ops(fp0.ops, fp0.nops, sp)) return 0;
    if (segmented) {
        for (int oop = 0; oop < 2; oop++) {
            sp.LM = fp0.load_mask; sp.SM = fp0.store_mask | (oop ? fp0.load_mask : 0u);
            sp.seg = true; sp.mode = 1; sp.minb = seg_minb(sp);
            if (get_cubin(sp, true)) have++;
        }
        return have;
    }
    for (int oop = 0; oop < 2; oop++)
        for (int sums = 0; sums < 2; sums++) {
            FusedProgram fp = fp0;
            if (oop) fp.store_mask |= fp.load_mask;
            if (sums) fp.load_mask |= (R_X | R_Y) & ~fp.store_mask;
            fill_spec(sp, fp, true);
            if (get_cubin(sp, true)) have++;
        }
    return have;
}

}  // namespace pxf

using namespace pxf;

extern "C" const char *pxf_jit_status(void)
{
    std::lock_guard<std::mutex> lock(g_mu);
    static char buf[2048];
    snprintf(buf, sizeof(buf), "%s (compiled %lld, loaded from disk %lld, in memory %zu)", g_status.c_str(),
             (long long)g_compiles, (long long)g_disk_hits, g_cache.size());
    return buf;
}

extern "C" const char *pxf_last_trace_kernel(void) { return g_last_kernel; }

extern "C" int32_t pxf_jit_compile(const pxf_op *ops, int32_t nops, int32_t segmented, const pxf_program_aux *aux)
{
    FusedProgram fp;
    // (side-array pointers only decide validity here; nothing is launched)
    pxf_program_aux dummy;
    memset(&dummy, 0, sizeof(dummy));
    dummy.wave = reinterpret_cast<const double *>(8); dummy.count = reinterpret_cast<int32_t *>(8);
    dummy.count_max = reinterpret_cast<int32_t *>(8);
    if (build_program(fp, ops, nops, aux ? aux : &dummy)) return -1;
    return jit_precompile(fp, segmented != 0);
}
