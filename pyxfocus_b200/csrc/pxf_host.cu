// Host-buffer entry point: the call an f2py user makes.  HOST arrays in, HOST arrays mutated
// in place, the device in between.  The bundle is cut into chunks that stream through a ring
// of device slots on three streams -- H2D of chunk c+1, the fused per-ray program on chunk c
// and D2H of chunk c-1 overlap (PCIe is full duplex) -- so the transfer cost is
// max(H2D, D2H), not their sum, and device memory is bounded by the ring, not the bundle.
// Only the rows the program reads are uploaded and only the rows it writes are downloaded
// (the liveness masks of build_program).  When the caller also wants the HPD, final x,y stay
// resident in full-length device rows and the select-based HPD runs on them at the end.
// Rows the program leaves at a known constant for every ray (z = 0 and the normal (0,0,1) after a
// closing `flat`; FusedProgram::const_mask) are not downloaded at all: a few host threads fill
// them in place while the DMA engines move the other rows -- for the Wolter-I chain that is 4 of
// the 9 written rows, i.e. 40 instead of 72 B/ray over PCIe on the way back.  A constant row that
// is also an INPUT row (z) is filled chunk by chunk, each only after its upload has completed.
// The same holds on the way IN for data, not program, reasons: every PyXFocus source leaves at
// least four of the six live rows constant (z = 0, l = m = 0, n = +-1 for a collimated beam;
// x = y = z = 0 for a point source).  Host threads scan each 16 MiB chunk of each input row ahead
// of the upload (8-byte patterns against the chunk's first element, early exit on the first
// difference, so varying rows cost nothing); a chunk that is bitwise constant is not uploaded --
// a fill kernel writes the value into the device slot instead.  Exact for any data; for the
// Wolter-I chain from `subannulus` it takes the upload from 48 to 16 B/ray.
// Streams, events and device buffers are cached between calls (pxf_host_release frees them).
#include <atomic>
#include <memory>
#include <chrono>
#include <mutex>
#include <stdlib.h>
#include <thread>
#include <vector>
#include "pxf_program.h"

namespace pxf {

#define HOST_SLOTS 4
#define HOST_CHUNK (int64_t(1) << 21)   // rays per chunk: 16 MiB per row

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes)
    {
        if (bytes <= cap) return PXF_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("pxf_host_trace_program: cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
            return PXF_ERR_NOMEM;
        }
        cap = bytes;
        return PXF_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct HostRing {
    int device = -1;
    cudaStream_t s_in = nullptr, s_run = nullptr, s_out = nullptr;
    cudaEvent_t in_done[HOST_SLOTS] = {}, run_done[HOST_SLOTS] = {}, out_done[HOST_SLOTS] = {};
    DevBuf slot_rows[HOST_SLOTS][10];
    DevBuf slot_alive[HOST_SLOTS];
    DevBuf full_x, full_y, full_alive, misc, cx, cy, scr;

    int init()
    {
        int dev = 0;
        PXF_CUDA(cudaGetDevice(&dev));
        if (device == dev && s_in) return PXF_OK;
        release();
        device = dev;
        PXF_CUDA(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
        PXF_CUDA(cudaStreamCreateWithFlags(&s_run, cudaStreamNonBlocking));
        PXF_CUDA(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
        for (int k = 0; k < HOST_SLOTS; k++) {
            PXF_CUDA(cudaEventCreateWithFlags(&in_done[k], cudaEventDisableTiming));
            PXF_CUDA(cudaEventCreateWithFlags(&run_done[k], cudaEventDisableTiming));
            PXF_CUDA(cudaEventCreateWithFlags(&out_done[k], cudaEventDisableTiming));
        }
        return PXF_OK;
    }
    void release()
    {
        for (int k = 0; k < HOST_SLOTS; k++) {
            for (int r = 0; r < 10; r++) slot_rows[k][r].release();
            slot_alive[k].release();
            if (in_done[k]) cudaEventDestroy(in_done[k]);
            if (run_done[k]) cudaEventDestroy(run_done[k]);
            if (out_done[k]) cudaEventDestroy(out_done[k]);
            in_done[k] = run_done[k] = out_done[k] = nullptr;
        }
        full_x.release(); full_y.release(); full_alive.release(); misc.release(); cx.release(); cy.release(); scr.release();
        if (s_in) cudaStreamDestroy(s_in);
        if (s_run) cudaStreamDestroy(s_run);
        if (s_out) cudaStreamDestroy(s_out);
        s_in = s_run = s_out = nullptr;
        device = -1;
    }
};

static HostRing g_ring;
static std::mutex g_ring_mutex;

static int chunk_is_constant(const double *p, int64_t n);
static void fill_const(double *dst, int64_t n, double v)
{
    // a row that already holds the constant (the previous call left it there: a pipeline that traces bundle after
    // bundle into the same arrays) is only read -- half the memory traffic of writing it, and no dirty lines
    if (n > 0 && memcmp(dst, &v, 8) == 0 && chunk_is_constant(dst, n)) return;
    if (v == 0.) memset(dst, 0, (size_t)n * 8);      // +0.0 is all-zero bits
    else for (int64_t i = 0; i < n; i++) dst[i] = v;
}

// 1 if the n doubles at p all have the bit pattern of p[0]
static int chunk_is_constant(const double *p, int64_t n)
{
    const uint64_t *q = reinterpret_cast<const uint64_t *>(p);
    const uint64_t v = q[0];
    int64_t i = 0;
    for (; i + 512 <= n; i += 512) {
        uint64_t acc = 0;
        for (int k = 0; k < 512; k++) acc |= q[i + k] ^ v;
        if (acc) return 0;
    }
    for (; i < n; i++)
        if (q[i] != v) return 0;
    return 1;
}

__global__ void __launch_bounds__(256) k_fill(double *__restrict__ p, int64_t n, double v)
{
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nthr) p[i] = v;
}

static void CUDART_CB bump_counter(void *p) { static_cast<std::atomic<int64_t> *>(p)->fetch_add(1, std::memory_order_release); }

static double now_ms()
{
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

}  // namespace pxf

using namespace pxf;

extern "C" {

void pxf_host_release(void)
{
    std::lock_guard<std::mutex> lock(g_ring_mutex);
    g_ring.release();
}

int pxf_host_trace_program(double *const rows_host[10], int64_t num, const pxf_op *ops, int32_t nops,
                           int32_t write_back, double *hpd_host, uint8_t *alive_host,
                           int64_t *alive_count_host, double *x_dev_keep, double *y_dev_keep)
{
    return pxf_host_trace_program_hint(rows_host, num, ops, nops, write_back, hpd_host, alive_host, alive_count_host,
                                       x_dev_keep, y_dev_keep, 0u);
}

int pxf_host_trace_program_hint(double *const rows_host[10], int64_t num, const pxf_op *ops, int32_t nops,
                                int32_t write_back, double *hpd_host, uint8_t *alive_host,
                                int64_t *alive_count_host, double *x_dev_keep, double *y_dev_keep,
                                uint32_t const_rows_mask)
{
    if (!rows_host || num < 0) { set_error("pxf_host_trace_program: bad argument"); return PXF_ERR_INVALID; }
    FusedProgram fp;
    int rc = build_program(fp, ops, nops);
    if (rc) return rc;
    for (int k = 0; k < fp.nops; k++)
        if (fp.ops[k].code == PXF_OP_RADGRATW || fp.ops[k].code == PXF_OP_GRAT) {
            // their arrays live on the device, and this entry point streams host rows through device buffers
            set_error("pxf_host_trace_program: PXF_OP_RADGRATW / GRAT read device arrays; use pxf_trace_program");
            return PXF_ERR_UNSUPPORTED;
        }
    if (sm_count() <= 0) { set_error("no CUDA device available (libpxf has no CPU fallback)"); return PXF_ERR_CUDA; }
    const unsigned LM = fp.load_mask, SM = fp.store_mask, USED = LM | SM;
    for (int r = 0; r < 10; r++)
        if ((USED & (1u << r)) && !rows_host[r]) {
            set_error("pxf_host_trace_program: row %d is used by the program but NULL", r);
            return PXF_ERR_INVALID;
        }
    const bool want_alive = fp.has_vignette != 0;
    const bool want_hpd = hpd_host != nullptr;
    if (want_hpd && !rows_host[1]) { set_error("pxf_host_trace_program: hpd needs the x,y rows"); return PXF_ERR_INVALID; }
    if (num == 0) {
        if (alive_count_host) *alive_count_host = 0;
        if (hpd_host) *hpd_host = __builtin_nan("");
        return PXF_OK;
    }
    const bool keep_xy = x_dev_keep && y_dev_keep;      // caller-owned device rows of length num
    if (keep_xy && ((reinterpret_cast<uintptr_t>(x_dev_keep) | reinterpret_cast<uintptr_t>(y_dev_keep)) & 15)) {
        set_error("pxf_host_trace_program: x_dev_keep/y_dev_keep must be 16-byte aligned");
        return PXF_ERR_INVALID;
    }
    static int debug = -1;
    if (debug < 0) { const char *e = getenv("PXF_HOST_DEBUG"); debug = (e && e[0] == '1') ? 1 : 0; }
    const double t0 = now_ms();

    std::lock_guard<std::mutex> lock(g_ring_mutex);
    HostRing &R = g_ring;
    if ((rc = R.init())) return rc;
    const int64_t chunk = num < HOST_CHUNK ? ((num + 1) & ~int64_t(1)) : HOST_CHUNK;
    const int64_t nchunks = (num + chunk - 1) / chunk;
    const int nslots = nchunks < HOST_SLOTS ? (int)nchunks : HOST_SLOTS;
    // x,y of the final bundle stay resident when the HPD is wanted (rows 1,2 then live in
    // full-length arrays and the slots alias into them)
    const bool xy_full = want_hpd || keep_xy;
    double *fx = nullptr, *fy = nullptr;
    if (xy_full) {
        if (keep_xy) { fx = x_dev_keep; fy = y_dev_keep; }
        else {
            if ((rc = R.full_x.ensure((size_t)(nchunks * chunk) * 8))) return rc;
            if ((rc = R.full_y.ensure((size_t)(nchunks * chunk) * 8))) return rc;
            fx = static_cast<double *>(R.full_x.p); fy = static_cast<double *>(R.full_y.p);
        }
        if (want_alive && (rc = R.full_alive.ensure((size_t)(nchunks * chunk)))) return rc;
    }
    for (int k = 0; k < nslots; k++) {
        for (int r = 0; r < 10; r++) {
            if (!(USED & (1u << r))) continue;
            if (xy_full && (r == 1 || r == 2)) continue;
            if ((rc = R.slot_rows[k][r].ensure((size_t)chunk * 8))) return rc;
        }
        if (want_alive && !xy_full && (rc = R.slot_alive[k].ensure((size_t)chunk))) return rc;
    }
    const double t1 = now_ms();

    // constant output rows: filled on the host, never downloaded
    const unsigned CM = write_back ? (SM & fp.const_mask) : 0u;
    const unsigned CM_late = CM & LM;            // also inputs: chunk c may be overwritten only after its H2D
    const unsigned CM_now = CM & ~LM;
    std::atomic<int64_t> uploaded(0);
    std::atomic<bool> abort_fill(false);
    std::vector<std::thread> fillers;
    // input rows: verdict[ri * nchunks + c] = -1 not scanned yet, 0 varies, 1 constant
    int in_rows[10], n_in = 0;
    for (int r = 0; r < 10; r++)
        if (LM & (1u << r)) in_rows[n_in++] = r;
    static int scan_inputs = -1;
    if (scan_inputs < 0) { const char *e = getenv("PXF_HOST_NO_SCAN"); scan_inputs = (e && e[0] == '1') ? 0 : 1; }
    const bool scanning = scan_inputs && n_in > 0;
    const int64_t nverd = scanning ? (int64_t)n_in * nchunks : 0;
    std::unique_ptr<std::atomic<int>[]> verdict(new std::atomic<int>[nverd > 0 ? nverd : 1]);
    for (int64_t i = 0; i < nverd; i++) verdict[i].store(-1, std::memory_order_relaxed);
    // rows the caller vouches for (every entry equals the first, e.g. z, l, m, n of a PyXFocus source): no scan
    int64_t nscan = 0;
    if (scanning)
        for (int ri = 0; ri < n_in; ri++) {
            if (const_rows_mask & (1u << in_rows[ri]))
                for (int64_t c = 0; c < nchunks; c++) verdict[(int64_t)ri * nchunks + c].store(1, std::memory_order_relaxed);
            else nscan++;
        }
    if (CM || scanning) {
        unsigned hc = std::thread::hardware_concurrency();
        int T = (int)(hc >= 4 ? (hc * 3) / 4 : 2);      // measured on the 16-vCPU B200 host: 8 -> 141 ms, 12 -> 135 ms
        if (const char *e = getenv("LOCAL_WORLD_SIZE")) {  // one process per GPU: the ranks share the host cores
            const int lws = atoi(e);
            // every core, split evenly (the copies themselves are DMA): 32 cores / 8 ranks = 4 threads, not 3
            if (lws > 1) T = (int)hc / lws > 2 ? (int)hc / lws : 2;
        }
        if (T > 16) T = 16;
        if (const char *e = getenv("PXF_HOST_THREADS")) { const int v = atoi(e); if (v >= 1 && v <= 64) T = v; }
        for (int t = 0; t < T; t++)
            fillers.emplace_back([&, t, T]() {
                // scans first (they gate the upload pipeline), chunk-major so early chunks finish first
                for (int64_t job = t; job < nverd; job += T) {
                    if (abort_fill.load()) return;
                    const int64_t c = job / n_in;
                    const int ri = (int)(job % n_in);
                    std::atomic<int> &vd = verdict[(int64_t)ri * nchunks + c];
                    if (vd.load(std::memory_order_relaxed) >= 0) continue;          // vouched for by the caller
                    const int64_t lo = c * chunk, n = (lo + chunk <= num) ? chunk : (num - lo);
                    const int v = chunk_is_constant(rows_host[in_rows[ri]] + lo, n);
                    vd.store(v, std::memory_order_release);
                }
                for (int r = 0; r < 10; r++)
                    if (CM_now & (1u << r)) {
                        const int64_t a = num * t / T, b = num * (t + 1) / T;
                        fill_const(rows_host[r] + a, b - a, fp.const_val[r]);
                    }
                if (!CM_late) return;
                for (int64_t c = t; c < nchunks; c += T) {
                    while (uploaded.load(std::memory_order_acquire) <= c) {
                        if (abort_fill.load()) return;
                        std::this_thread::sleep_for(std::chrono::microseconds(50));
                    }
                    const int64_t lo = c * chunk, n = (lo + chunk <= num) ? chunk : (num - lo);
                    for (int r = 0; r < 10; r++)
                        if (CM_late & (1u << r)) {
                            // already that very constant (scan verdict + first element): nothing to write
                            bool same = false;
                            if (scanning)
                                for (int ri = 0; ri < n_in; ri++)
                                    if (in_rows[ri] == r && verdict[(int64_t)ri * nchunks + c].load(std::memory_order_acquire) == 1)
                                        same = memcmp(rows_host[r] + lo, &fp.const_val[r], 8) == 0;
                            if (!same) fill_const(rows_host[r] + lo, n, fp.const_val[r]);
                        }
                }
            });
    }
    struct Joiner {       // error paths: stop the fillers and drain the callbacks that point at `uploaded`
        std::vector<std::thread> &th; std::atomic<bool> &ab; cudaStream_t s, s2, s3; bool ok = false;
        // on failure nothing may still be writing into the caller's host rows after we return: drain all three streams
        ~Joiner() { if (!ok) { ab.store(true); cudaStreamSynchronize(s); cudaStreamSynchronize(s2); cudaStreamSynchronize(s3); }
                    for (auto &t : th) if (t.joinable()) t.join(); }
    } joiner{fillers, abort_fill, R.s_in, R.s_run, R.s_out};

    int64_t alive_total = 0;
    size_t h2d_skipped = 0;
    for (int64_t c = 0; c < nchunks; c++) {
        const int k = (int)(c % nslots);
        const int64_t lo = c * chunk;
        const int64_t n = (lo + chunk <= num) ? chunk : (num - lo);
        double *rows[10];
        for (int r = 0; r < 10; r++) rows[r] = static_cast<double *>(R.slot_rows[k][r].p);
        if (xy_full) { rows[1] = fx + lo; rows[2] = fy + lo; }
        uint8_t *alive = want_alive ? (xy_full ? static_cast<uint8_t *>(R.full_alive.p) + lo
                                               : static_cast<uint8_t *>(R.slot_alive[k].p)) : nullptr;
        // the slot is free once its previous D2H finished
        if (c >= nslots) PXF_CUDA(cudaStreamWaitEvent(R.s_in, R.out_done[k], 0));
        for (int ri = 0; ri < n_in; ri++) {
            const int r = in_rows[ri];
            int v = 0;
            if (scanning) {
                std::atomic<int> &vd = verdict[(int64_t)ri * nchunks + c];
                while ((v = vd.load(std::memory_order_acquire)) < 0) std::this_thread::yield();
            }
            if (v == 1) {
                k_fill<<<sm_count() * 2, 256, 0, R.s_in>>>(rows[r], n, rows_host[r][lo]);
                count_launch();
                h2d_skipped += (size_t)n * 8;
            } else {
                PXF_CUDA(cudaMemcpyAsync(rows[r], rows_host[r] + lo, (size_t)n * 8, cudaMemcpyHostToDevice, R.s_in));
            }
        }
        PXF_CUDA(cudaEventRecord(R.in_done[k], R.s_in));
        if (CM_late) PXF_CUDA(cudaLaunchHostFunc(R.s_in, bump_counter, &uploaded));
        PXF_CUDA(cudaStreamWaitEvent(R.s_run, R.in_done[k], 0));
        if ((rc = launch_program(rows, n, fp, alive, R.s_run))) return rc;
        PXF_CUDA(cudaEventRecord(R.run_done[k], R.s_run));
        PXF_CUDA(cudaStreamWaitEvent(R.s_out, R.run_done[k], 0));
        if (write_back)
            for (int r = 0; r < 10; r++)
                if ((SM & ~CM) & (1u << r))
                    PXF_CUDA(cudaMemcpyAsync(rows_host[r] + lo, rows[r], (size_t)n * 8, cudaMemcpyDeviceToHost, R.s_out));
        if (want_alive && alive_host)
            PXF_CUDA(cudaMemcpyAsync(alive_host + lo, alive, (size_t)n, cudaMemcpyDeviceToHost, R.s_out));
        PXF_CUDA(cudaEventRecord(R.out_done[k], R.s_out));
    }
    const double t2 = now_ms();
    PXF_CUDA(cudaStreamSynchronize(R.s_run));
    const double t3 = now_ms();

    if (want_hpd) {
        const double *hx = fx, *hy = fy;
        int64_t hn = num;
        pxf_stream_t ps = reinterpret_cast<pxf_stream_t>(R.s_run);
        if (want_alive) {
            // HPD over the surviving rays only: compact x,y by the alive flags first
            if ((rc = R.scr.ensure(pxf_compact_scratch_bytes(num)))) return rc;
            int64_t cnt = 0;
            const uint8_t *fa = static_cast<const uint8_t *>(R.full_alive.p);
            if ((rc = pxf_compact_count(fa, num, R.scr.p, &cnt, ps))) return rc;
            if (cnt > 0) {
                if ((rc = R.cx.ensure((size_t)(cnt + 1) * 8)) || (rc = R.cy.ensure((size_t)(cnt + 1) * 8))) return rc;
                const double *in2[2] = {fx, fy};
                double *out2[2] = {static_cast<double *>(R.cx.p), static_cast<double *>(R.cy.p)};
                if ((rc = pxf_compact_scatter(in2, out2, 2, fa, num, R.scr.p, ps))) return rc;
            }
            hx = static_cast<const double *>(R.cx.p); hy = static_cast<const double *>(R.cy.p); hn = cnt;
            alive_total = cnt;
        }
        if (hn > 0) {
            const size_t wb = pxf_hpd_workspace_bytes(hn);
            if ((rc = R.misc.ensure(wb + 64))) return rc;
            double *out = reinterpret_cast<double *>((char *)R.misc.p + wb);
            double h[4] = {0, 0, 0, 0};
            for (int mode = 0; mode < 2; mode++) {
                if ((rc = pxf_hpd_unweighted_dev(hx, hy, hn, out, R.misc.p, mode, ps))) return rc;
                PXF_CUDA(cudaMemcpyAsync(h, out, sizeof(h), cudaMemcpyDeviceToHost, R.s_run));
                PXF_CUDA(cudaStreamSynchronize(R.s_run));
                if (h[3] != 0.) break;
            }
            *hpd_host = h[0];
        } else {
            *hpd_host = __builtin_nan("");
        }
    }
    const double t4 = now_ms();
    PXF_CUDA(cudaStreamSynchronize(R.s_out));
    PXF_CUDA(cudaStreamSynchronize(R.s_in));
    joiner.ok = true;
    for (auto &t : fillers) t.join();
    const double t5 = now_ms();
    if (alive_count_host) {
        if (!want_alive) *alive_count_host = num;
        else if (want_hpd) *alive_count_host = alive_total;
        else if (alive_host) {
            int64_t t = 0;
            for (int64_t i = 0; i < num; i++) t += alive_host[i] != 0;
            *alive_count_host = t;
        } else {
            *alive_count_host = -1;   // flags were not requested anywhere
        }
    }
    if (debug)
        fprintf(stderr, "[pxf_host] num=%lld chunks=%lld: alloc %.1f ms, enqueue %.1f ms, wait-run %.1f ms, hpd %.1f ms, "
                        "wait-d2h %.1f ms, total %.1f ms; %.2f GB of constant input chunks not uploaded\n",
                (long long)num, (long long)nchunks, t1 - t0, t2 - t1, t3 - t2, t4 - t3, t5 - t4, t5 - t0, h2d_skipped * 1e-9);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("pxf_host_trace_program: %s", cudaGetErrorString(e)); return PXF_ERR_CUDA; }
    return PXF_OK;
}

}  // extern "C"
