#!/usr/bin/env python
"""Benchmark of the hot path: Wolter-I trace + HPD, rays/s (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this engine (one rank per GPU)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)

A STEP is one pass of the hot path over one synthetic bundle:
    transform -> wolterprimary -> reflect -> woltersecondary -> reflect -> flat  (ONE fused kernel)
    -> hpd (centroid reduction + exact radix select; all-reduced over ranks for N>1)
on ``--rays`` rays per GPU (default 1.25e8 = 10 GB of bundle; x8 GPUs = the 1e9-ray bundle of
BASELINE config 5, traced with config 1's chain).  The source bundle is generated on the
device once and stays resident; every step reads it and writes a second bundle, so each step
does the full Newton work on fresh rays.  Inputs (6 GB/GPU) are far larger than L2, so no L2
flush is needed between steps.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
``--dump-outputs DIR`` also writes what the last timed step computed as DIR/<name>.npy (see ``dump_outputs``).
The benchmark writes nothing into the repository tree, which may be read-only.
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "rays/sec (fp64, Wolter-I trace + HPD)"
R0, Z0, PSI = 220., 8400., 1.
RIN, ROUT = 220., 220.6
SURFACES_PER_RAY = 3                 # primary, secondary, focal plane
# algorithmic HBM bytes per ray of the fused trace kernel: read x,y,z,l,m,n + write x,y,z,l,m,n,ux,uy,uz
FP64_INSTR_PER_RAY = 283        # DADD+DMUL+DFMA+DSETP per ray, profiles/r01f_k_chain.txt (source page)
TRACE_BYTES_PER_RAY = 6 * 8 + 9 * 8
# per-routine API for comparison (SURVEY.md 8d): 144+96+72+96+72+96
PERCALL_BYTES_PER_RAY = 576


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--rays", type=float, default=1.25e8, help="rays per GPU")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-rays", type=float, default=2.0e7, help="rays per step of the reference arm")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs 1-5 sub-results")
    ap.add_argument("--configs-scale", type=float, default=1., help="scale the configs' ray counts (smoke runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's traced rows (a fixed sample of rays) and HPD "
                         "to DIR/<name>.npy, float64 (N > 1: rank 0's shard and the global HPD)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_ROWS = ("x", "y", "z", "l", "m", "n", "ux", "uy", "uz")
DUMP_RAYS = 1 << 18          # rays per dumped row: 9 rows x 2 MB


def dump_sample(n):
    """Indices of the rays --dump-outputs writes: all of a small bundle, else a fixed seeded sample in ascending
    order, so that two builds run with the same arguments dump the same rays."""
    import numpy as np
    if n <= DUMP_RAYS:
        return np.arange(n)
    return np.sort(np.random.default_rng(20261020).choice(n, DUMP_RAYS, replace=False))


def dump_outputs(path, rows, hpd):
    """What the timed path hands its caller after its last step: rows x..uz of the traced bundle at the
    ``dump_sample`` rays, and the HPD."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, row in zip(DUMP_ROWS, rows):
        np.save(os.path.join(path, name + ".npy"), np.asarray(row, dtype=np.float64))
    np.save(os.path.join(path, "hpd.npy"), np.array([hpd], dtype=np.float64))


def private_jit_cache():
    """Specialised kernels compiled at run time are cached in a temporary directory instead of the tree: the
    kernels build() cached under pyxfocus_b200/_jit are copied there and PXF_JIT_CACHE points at it."""
    if "PXF_JIT_CACHE" in os.environ:
        return
    tmp = tempfile.mkdtemp(prefix="pxf_jit_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    built = os.path.join(ROOT, "pyxfocus_b200", "_jit")
    if os.path.isdir(built):
        for f in os.listdir(built):
            if f.endswith(".cubin"):
                shutil.copy(os.path.join(built, f), tmp)
    os.environ["PXF_JIT_CACHE"] = tmp


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks line of /opt/skills/guides/B200_PROFILING.md, sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []          # (wall-clock time the line was read, line)
        self.proc = None
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # nvidia-smi is started BEFORE the warm-up (its start-up holds driver locks for ~100 ms and
        # must not land in the timed region); keep the samples read inside the timed region, or --
        # when the region is shorter than the sampling period -- those taken under load since the
        # warm-up began (the GPU runs the same step back to back from there on).
        inside = [ln for t, ln in self.lines if self.t0 is not None and self.t0 <= t <= (self.t1 or t)]
        window = "timed region"
        if not inside:
            inside = [ln for t, ln in self.lines]
            window = "warm-up + timed region"
        self.window = window
        for ln in inside:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power), "window": self.window}


# ------------------------------------------------------------------------------- CPU arm
def cpu_step_factory(n):
    """One step of the reference's CPU path on n rays: the six Fortran-routine calls (C oracle
    port, OpenMP over rays like the Fortran) under the reference's Python call pattern, then
    analyses.hpd (numpy).  Returns (fresh_inputs(), step(rays))."""
    import numpy as np
    from oracle import chains, pyref

    np.random.seed(0)
    src = pyref.subannulus(RIN, ROUT, 2 * np.pi, n, zhat=-1.)

    def fresh():
        return [r.copy() for r in src]

    def step(rays):
        chains.run_steps_cpu(rays, chains.wolter1_steps(R0, Z0, PSI))
        return pyref.hpd(rays)
    return fresh, step


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def use_all_host_cores():
    """The CPU arm runs on EVERY host core this process may use, whatever the launcher exported: torchrun sets
    OMP_NUM_THREADS=1 for its workers, which would time the reference on one core.  Must run before liboracle
    (libgomp) is loaded -- libgomp reads the variable once, at load time.  Returns the thread count the oracle's
    OpenMP runtime then reports (omp_get_max_threads), i.e. the count actually used."""
    n = host_cores()
    os.environ["OMP_NUM_THREADS"] = str(n)
    os.environ.pop("OMP_THREAD_LIMIT", None)
    from oracle import f2py as of
    lib = of.lib()
    try:
        import ctypes
        gomp = ctypes.CDLL("libgomp.so.1")
        gomp.omp_set_num_threads(n)
        got = int(gomp.omp_get_max_threads())
    except OSError:
        got = n
    return got


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  Its Fortran cannot
    be compiled in this image (no Fortran compiler), so this is the C oracle port (kind
    'port'), OpenMP on every host core, driven through the reference's call pattern."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = use_all_host_cores()
    n = int(args.ref_rays)
    fresh, step = cpu_step_factory(n)
    for _ in range(max(1, min(args.warmup, 2))):
        step(fresh())
    inputs = [fresh() for _ in range(args.steps)] if n * 80 * args.steps < 24e9 else None
    t = 0.
    hp = None
    for k in range(args.steps):
        rays = inputs[k] if inputs is not None else fresh()
        t0 = time.perf_counter()
        hp = step(rays)
        t += time.perf_counter() - t0
    if args.dump_outputs:
        idx = dump_sample(n)
        dump_outputs(args.dump_outputs, [rays[k][idx] for k in range(1, 10)], hp)
    val = n * args.steps / t
    sample = "%d steps x %.3g rays (same chain + hpd), C oracle port with OpenMP" % (args.steps, n)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "wolter1_trace_hpd", "rays_per_step": n, "surfaces_per_ray": SURFACES_PER_RAY,
                   "r0": R0, "z0": Z0, "psi": PSI, "hpd": hp},
        "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def cpu_baseline():
    """Bounded sample (~10-20 s) of the same step on the host cores."""
    cores = use_all_host_cores()
    n = 4_000_000
    fresh, step = cpu_step_factory(n)
    step(fresh())                                   # warm-up (page faults, thread pool)
    rays = fresh()
    t0 = time.perf_counter()
    step(rays)
    t1 = time.perf_counter() - t0
    reps = max(1, min(20, int(12. / max(t1, 1e-3))))
    ins = [fresh() for _ in range(reps)]
    t0 = time.perf_counter()
    for r in ins:
        step(r)
    t = time.perf_counter() - t0
    return {"value": n * reps / t, "unit": "rays/s", "cores": cores, "kind": "port",
            "sample": "%d x %.1e rays, six oracle-routine passes + numpy hpd, OpenMP on all host cores "
                      "(C restatement of the f2py Fortran; the Fortran itself cannot be built here)" % (reps, n)}


# ------------------------------------------------------------------------------- engine arm
def sharded_parity_check(pxf, pdist, prog, rank, world, dev, total=6_000_001):
    """N > 1, before anything is timed: trace a 6e6-ray bundle sharded over the ranks AND whole on every rank; the
    shard must be the slice of the whole bundle bit for bit and the all-reduced HPD / rms must equal the single-GPU
    ones (what tests/run_dist_nccl.py asserts, made visible in the bench line)."""
    import numpy as np
    import torch
    import torch.distributed as td
    lo, hi = pdist.shard_range(total, rank, world)
    shard = pxf.sources.subannulus(RIN, ROUT, 2 * np.pi, hi - lo, zhat=-1., rng="philox", seed=3, first=lo, device=dev)
    prog.run(shard)
    h = pdist.hpd(shard)
    r = pdist.rmsCentroid(shard)
    whole = pxf.sources.subannulus(RIN, ROUT, 2 * np.pi, total, zhat=-1., rng="philox", seed=3, first=0, device=dev)
    prog.run(whole)
    rows_equal = all(bool(torch.equal(whole[k][lo:hi], shard[k])) for k in range(1, 10))
    h1 = pxf.analyses.hpd(whole)
    r1 = pxf.analyses.rmsCentroid(whole)
    flags = torch.tensor([1 if rows_equal else 0, 1 if abs(h - h1) <= 1e-9 * abs(h1) else 0, 1 if abs(r - r1) <= 1e-9 * r1 else 0],
                         dtype=torch.int32, device=dev)
    td.all_reduce(flags, op=td.ReduceOp.MIN)
    f = flags.cpu().tolist()
    del shard, whole
    torch.cuda.empty_cache()
    return {"rays": total, "rows_equal": bool(f[0]), "hpd_equal": bool(f[1]), "rms_equal": bool(f[2]),
            "tolerance": "rows: same bits as the slice of the single-GPU bundle; hpd, rms: 1e-9 relative "
                         "(the all-reduced centroid may differ from the one-GPU tree sum in the last bit)",
            "hpd_sharded": h, "hpd_single_gpu": h1, "hpd_rel_diff": abs(h - h1) / abs(h1) if h1 else 0.}


def run_engine(args):
    import numpy as np
    import torch
    import torch.distributed as td

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    # nvidia-smi starts FIRST (before the process group, the library load and the source generation): its start-up
    # holds driver locks for ~100 ms, which must be over long before the timed region on every rank's GPU
    clk = ClockSampler(local)
    if rank == 0:
        clk.start()
    t_sampler = time.time()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        td.init_process_group("nccl", device_id=dev)
    private_jit_cache()
    import pyxfocus_b200 as pxf
    from pyxfocus_b200 import dist as pdist
    from pyxfocus_b200._call import bundle_alloc

    n = int(args.rays)
    total = n * world
    first = rank * n
    prog = (pxf.Program().transform(0., 0., Z0, 0., 0., 0.).wolterprimary(R0, Z0, PSI).reflect()
            .woltersecondary(R0, Z0, PSI).reflect().flat())

    def barrier():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()

    # ---- N > 1: the sharded path must reproduce the single-GPU result of the whole bundle before it is timed
    parity = sharded_parity_check(pxf, pdist, prog, rank, world, dev) if world > 1 else None

    # ---- resident inputs: source bundle generated on the device (counter-based, seed 0,
    # global ray index => identical stream for any sharding)
    src = pxf.sources.subannulus(RIN, ROUT, 2 * np.pi, n, zhat=-1., rng="philox", seed=0, first=first, device=dev)
    out = bundle_alloc(n, dev, zero=True)
    sums = torch.zeros(16, dtype=torch.float64, device=dev)
    ws = pxf.analyses.hpd_workspace(n, dev)

    def step(res_row):
        """One step: the fused trace (which also emits the centroid sums) + the HPD, result left on the device in
        res_row = [HPD, lower, upper, valid] -- nothing forces a host round trip between steps."""
        prog.run(src, out=out, sums=sums)
        if world > 1:
            pdist.hpd(out, sums=sums, total=total, min_shard=n, out=res_row)
        else:
            pxf.analyses.hpd_enqueue(out, res_row, ws, sums=sums)

    def step_readback():
        prog.run(src, out=out, sums=sums)
        return pdist.hpd(out, sums=sums, total=total, min_shard=n) if world > 1 else pxf.analyses.hpd(out, sums=sums)

    # ---- warm-up: the read-back path once (reference HPD value), then the path that is timed, at least W steps
    # and -- on every rank alike -- until the sampler has been up for a second and has delivered samples
    hp = step_readback()
    wres = torch.zeros(4, dtype=torch.float64, device=dev)
    nw = 0
    go = torch.ones(1, dtype=torch.int32, device=dev)
    while True:
        step(wres)
        nw += 1
        if nw < max(args.warmup, 3):
            continue
        more = (time.time() - t_sampler < 1.0 or (clk.proc is not None and len(clk.lines) < 2)) and nw < 400
        if world > 1:
            go[0] = 1 if (rank == 0 and more) else 0
            td.all_reduce(go, op=td.ReduceOp.MAX)        # rank 0 decides for everybody
            more = bool(int(go.item()))
        if not more:
            break
    barrier()

    # ---- timed region: K steps, CUDA events on the launching stream, clocks sampled alongside
    K = args.steps
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    bev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]       # step boundaries

    def timed_loop(deferred):
        res = torch.zeros(K, 4, dtype=torch.float64, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        last = None
        barrier()
        clk.mark_begin()
        e0.record()
        for k in range(K):
            bev[k].record()
            kev[k][0].record()
            prog.run(src, out=out, sums=sums)
            kev[k][1].record()
            if deferred:
                if world > 1:
                    pdist.hpd(out, sums=sums, total=total, min_shard=n, out=res[k])
                else:
                    pxf.analyses.hpd_enqueue(out, res[k], ws, sums=sums)
            else:
                last = pdist.hpd(out, sums=sums, total=total, min_shard=n) if world > 1 else pxf.analyses.hpd(out, sums=sums)
        bev[K].record()
        e1.record()
        barrier()
        clk.mark_end()
        if deferred:
            h = res.cpu().numpy()
            if not (h[:, 3] != 0.).all():
                return None, None          # a bracket missed (~1e-9): the caller re-times with read-backs
            last = float(h[-1, 0])
        return e0.elapsed_time(e1), last

    launches0 = pxf.launch_count()
    readback = "deferred: K results read after the timed region"
    ms, hp_t = timed_loop(True)
    if ms is None:
        launches0 = pxf.launch_count()
        readback = "per step"
        ms, hp_t = timed_loop(False)
    assert hp_t == hp or (hp_t != hp_t and hp != hp), "HPD changed between warm-up and timed steps"
    launches = pxf.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        idx = torch.from_numpy(dump_sample(n)).to(dev)
        dump_outputs(args.dump_outputs, [out[k].index_select(0, idx).cpu().numpy() for k in range(1, 10)], hp_t)
    kname = pxf.last_trace_kernel()             # the kernel the timed steps launched
    clocks = clk.stop() if rank == 0 else None
    trace_ms = sum(a.elapsed_time(b) for a, b in kev) / K
    per_step = sorted(bev[k].elapsed_time(bev[k + 1]) for k in range(K))
    step_med, step_max = per_step[K // 2], per_step[-1]
    # per-step latency WITH a host read-back of every result (what a caller that needs each HPD before going on sees)
    torch.cuda.synchronize()
    lat = []
    for _ in range(min(K, 10)):
        barrier()
        t0 = time.perf_counter()
        step_readback()
        lat.append((time.perf_counter() - t0) * 1e3)
    lat.sort()
    if world > 1:
        t = torch.tensor([ms, trace_ms, step_med, step_max, lat[len(lat) // 2]], dtype=torch.float64, device=dev)
        td.all_reduce(t, op=td.ReduceOp.MAX)
        ms, trace_ms, step_med, step_max = float(t[0]), float(t[1]), float(t[2]), float(t[3])
        lat_med = float(t[4])
    else:
        lat_med = lat[len(lat) // 2]
    value = total * args.steps / (ms * 1e-3)

    # ---- end to end through the host-array C ABI entry (pinned host rows -> device -> host)
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, pxf, pdist, src, prog, n, world, dev, barrier)
    # ---- the other BASELINE configurations (the headline's buffers are released first)
    configs = None
    if not args.no_configs:
        del src, out, ws
        torch.cuda.empty_cache()
        try:
            configs = run_configs(args, pxf, world, rank, dev, barrier)
        except Exception as e:                                    # noqa: BLE001  (sub-results never take the headline down)
            configs = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}

    if rank != 0:
        if world > 1:
            td.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = TRACE_BYTES_PER_RAY * n / (trace_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:
        # dram__bytes_read.sum + dram__bytes_write.sum of the fused kernel, one launch, from the committed
        # ncu --set full capture named in the file (per-ray figure x rays per launch: the kernel streams)
        tj = json.load(open(os.path.join(ROOT, "profiles", "trace_kernel_traffic.json")))
        traffic = float(tj["dram_bytes_per_ray"]) * n
        traffic_src = "static: %s (%s rays/launch, kernel %s)" % (tj.get("capture"), tj.get("rays_per_launch_measured"), tj.get("kernel"))
    except (OSError, ValueError, KeyError):
        pass
    fp64_frac = FP64_INSTR_PER_RAY * n / (trace_ms * 1e-3) / (148 * 64 * 1.965e9)
    line = {
        "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": nw, "ms_per_step": ms / args.steps, "ms_per_step_median": step_med, "ms_per_step_max": step_max,
        "ms_per_step_with_readback": lat_med, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "wolter1_trace_hpd (BASELINE configs[0] chain at configs[4] scale: "
                               "subannulus -> transform -> wolterprimary -> reflect -> woltersecondary -> reflect -> flat -> hpd)",
                   "rays_per_gpu": n, "total_rays": total, "surfaces_per_ray": SURFACES_PER_RAY,
                   "interactions_per_s": value * SURFACES_PER_RAY, "r0": R0, "z0": Z0, "psi": PSI,
                   "parallelism": "rays sharded %d-way, no trace-time communication; HPD = bracketed exact "
                                  "select, 3 small collectives (sums+sample all-gather, counters+bins "
                                  "all-reduce, key lists all-gather)" % world,
                   "l2": "inputs (%.1f GB/GPU) larger than L2, no flush needed" % (48e-9 * n),
                   "hpd": hp, "trace_kernel_ms": trace_ms, "hpd_readback": readback,
                   "latency_note": "ms_per_step: K steps enqueued back to back, results read after the region; "
                                   "ms_per_step_with_readback: median wall time of a step that reads its HPD back "
                                   "before the next one starts (what the CPU arm does every step)"},
        "roofline": {"bound": "fp64-issue", "kernel": kname, "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak,
                     "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback",
                     "algorithmic_bytes_per_ray": TRACE_BYTES_PER_RAY, "traffic": traffic, "traffic_source": traffic_src,
                     "note": "achieved/peak/frac are the HBM figures the contract asks for (algorithmic bytes / kernel "
                             "time vs the measured copy rate); the kernel itself is bound by fp64 instruction issue "
                             "along serial Newton/division chains (no FMA contraction, for bit parity with the "
                             "reference): a compute-only replay takes the same time (profiles/r01_trace_compute.txt)",
                     # second denominator: fp64 warp instructions per ray from the ncu capture (static),
                     # duration measured live; peak = 148 SMs x 64 lanes x sm_max clock, reached to 99 %
                     # by profiles/micro/fp64_peak.cu
                     "fp64": {"thread_instr_per_ray": FP64_INSTR_PER_RAY,
                              "achieved_Tinstr_s": FP64_INSTR_PER_RAY * n / (trace_ms * 1e-3) / 1e12,
                              "peak_Tinstr_s": 148 * 64 * 1.965e9 / 1e12, "frac": fp64_frac}},
        "clocks": clocks,
        "gpu_launches": launches,
    }
    if parity is not None:
        line["parity_check"] = parity
    if configs is not None:
        line["configs"] = configs
    if e2e is not None:
        line["e2e"] = e2e
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline()
    emit(line)
    if world > 1:
        td.destroy_process_group()


def run_configs(args, pxf, world, rank, dev, barrier):
    """BASELINE configs 1-5 as SURVEY.md 8(d) specifies them, through the public API (pyxfocus_b200/examples.py, the
    GPU-arranged forms of the reference's example scripts), each at its named size with the source drawn on the
    device every pass.  Per config: wall time of a whole pass (source -> trace -> vignette -> analyses, results read
    back as the scripts do), rays/s, ray-surface interactions/s, the headline result, and a parity field: the same
    code at the size of the committed golden (tests/golden/configs.npz, produced by the reference's own Python layer
    over the C oracle), numpy-seeded, compared with it.  Configs 1-4 run at N = 1 only; config 5 is the sharded one."""
    import numpy as np
    import torch
    ex = pxf.examples
    sc = args.configs_scale
    out = {}

    def timed(fn, reps=3):
        fn()                                  # warm-up (allocator, occupancy queries, tables)
        ts = []
        res = None
        for _ in range(reps):
            barrier()
            t0 = time.perf_counter()
            res = fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        del fn
        return min(ts), res

    def rel(a, b):
        return abs(a - b) / max(abs(b), 1e-300)

    gold = None
    try:
        gold = np.load(os.path.join(ROOT, "tests", "golden", "configs.npz"))
        sizes = {}
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
        from make_golden_configs import SIZES as sizes          # noqa: N811  (constants only; nothing is generated)
    except Exception as e:                                        # noqa: BLE001
        gold, sizes = None, {"error": str(e)[:80]}

    if world == 1:
        # ---- config 1 at its own size (1e5 rays: launch-latency territory), numpy-seeded like the reference script
        n1 = 100_000
        t, r = timed(lambda: {k: v for k, v in ex.config1_fast(n1, rng="numpy").items() if k != "rays"})
        out["config1"] = {"workload": "Wolter-I pair + hpd, 1e5 rays, np.random.seed(0) source (host MT19937 draws uploaded)",
                          "rays": n1, "ms": 1e3 * t, "rays_per_s": n1 / t, "interactions_per_s": 3 * n1 / t,
                          "hpd": r["hpd"], "parity": {"expected_hpd_mm": 1.278e-5, "source": "SURVEY.md 8d probe of the reference chain",
                                                      "ok": bool(rel(r["hpd"], 1.278e-5) < 2e-2)}}
        # ---- config 2: W-S field sweep, 31 field points x 1e7 rays
        n2 = max(1000, int(1e7 * sc))
        ap = ex.ws_aperture(ex.product_api(dev))
        arc = np.linspace(0., 30., 31)

        def c2():
            res = ex.config2_fast(n2, arc, ap, rng="philox", device=dev)
            return [{k: v for k, v in p.items() if k != "rays"} for p in res]
        t, r = timed(c2, reps=2)
        par = None
        if gold is not None:
            ok, worst = True, 0.
            for a in (0., 5., 10.):
                g = gold["c2_%02d_scalars" % int(a)]
                p = ex.config2_point_fast(sizes["c2_n"], a / 60. * np.pi / 180., tuple(gold["c2_aperture"]))
                for got, want in ((p["hpd"], g[3]), (p["rms"], g[4]), (p["hpd_scan"], g[5]), (p["rms_scan"], g[6])):
                    # 1e-9 relative, but no finer than the rays are determined: 4e-12 of the 1e4 mm system = 4e-8 mm
                    # (the on-axis 1e-5 mm spot is rounding noise of flat's REAL*4 step), i.e. a floor of 40 mm
                    e = abs(got - want) / max(abs(want), 40.)
                    worst = max(worst, e)
                ok = ok and p["d2"] == g[1] and p["d3"] == g[2]
            par = {"vs": "tests/golden/configs.npz (reference Python layer + C oracle), field points 0/5/10 arcmin, %d rays" % sizes["c2_n"],
                   "scan_offsets_equal": bool(ok), "worst_rel_err_hpd_rms": worst, "ok": bool(ok and worst <= 1e-9)}
        out["config2"] = {"workload": "W-S shell field sweep: 31 field points x (subannulus, wsPrimary, kick, reflect, wsSecondary, "
                                      "reflect, flat, findimageplane(20,100), findimageplane(1,100), flat, hpd, rms, focusI, hpd, rms)",
                          "rays_per_field_point": n2, "field_points": 31, "ms": 1e3 * t, "rays_per_s": 31 * n2 / t,
                          "interactions_per_s": 31 * n2 * 3 / t,
                          "hpd_mm_at_0_5_10_20_30_arcmin": [r[i]["hpd"] for i in (0, 5, 10, 20, 30)],
                          "rms_over_z0_at_5_arcmin": r[5]["rms"] / 1e4, "parity": par}
        # ---- config 3: Zernike figure error + Wolter-I pair + two vignettes, 1e8 rays
        n3 = max(1000, int(1e8 * sc))
        t, r = timed(lambda: {k: (v if k != "rays" else v[1].shape[0]) for k, v in
                              ex.config3_fast(n3, rng="philox", device=dev, want_idx=False).items()})
        par = None
        if gold is not None:
            p = ex.config3_fast(sizes["c3_n"])
            same_idx = bool(np.array_equal(p["idx"].cpu().numpy(), gold["c3_idx"]))
            e = rel(p["hpd"], gold["c3_scalars"][0])
            par = {"vs": "tests/golden/configs.npz, %d rays" % sizes["c3_n"], "surviving_index_set_equal": same_idx,
                   "hpd_rel_err": e, "ok": bool(same_idx and e <= 1e-9)}
        out["config3"] = {"workload": "subannulus -> transform -> zernsurf(36 terms, nr=1) -> reflect -> flat(nr=1) -> wolterprimary -> "
                                      "reflect -> vignette(z range & |y|) -> woltersecondary -> reflect -> vignette() -> flat -> hpd: "
                                      "ONE fused launch + compaction + hpd",
                          "rays": n3, "ms": 1e3 * t, "rays_per_s": n3 / t, "interactions_per_s": 4 * n3 / t,
                          "kept": r["rays"] / n3, "hpd": r["hpd"], "parity": par}
        # ---- config 4: Arcus SPO module row (72 shells) + fanned radial-grating array, 1e8 rays
        M = 72
        npsh = max(10, int(1e8 * sc) // M)

        def c4(order=-3, wave=2.4):
            res = ex.config4_fast(npsh, M, order=order, wave=wave, rng="philox", device=dev)
            return {k: v for k, v in res.items() if k not in ("rays", "surv")}
        t, r = timed(c4)
        tw, rw = timed(lambda: c4(-1, "uniform"), reps=2)
        par = None
        if gold is not None:
            ok, worst = True, 0.
            for order, wave in ((-1, 4.8), (-3, 2.4), (-8, .6)):
                g = gold["c4_o%d_s_scalars" % (-order)]
                p = ex.config4_fast(sizes["c4_n"], sizes["c4_M"], order=order, wave=wave)
                ok = ok and p["kept"] == g[0] and p["gratings"] == g[2]
                worst = max(worst, abs(p["dz"] - g[1]) / 1.2e4, abs(p["cy"] - g[4]) / 1.2e4)
            par = {"vs": "tests/golden/configs.npz, orders -1/-3/-8, %d rays" % (sizes["c4_n"] * sizes["c4_M"]),
                   "kept_and_grating_counts_equal": bool(ok), "worst_err_over_focal_length": worst, "ok": bool(ok and worst <= 1e-9)}
        out["config4"] = {"workload": "Arcus: 72 SPO shells (subannulus, transform, spoPrimary, reflect, spoSecondary, reflect, "
                                      "transform) in one segmented launch -> fanned radial-grating array (%d gratings; masked "
                                      "flat/reflect/radgrat loop of sector.py as ONE per-ray in-kernel loop + one host read of the "
                                      "grating count) -> flat -> focusY -> vignette(|y-<y>|<10) -> weighted centroid/rmsY/hpdY"
                                      % r["gratings"],
                          "rays": npsh * M, "shells": M, "order_wave_nm": [-3, 2.4], "ms": 1e3 * t, "rays_per_s": npsh * M / t,
                          "interactions_per_s": npsh * M * (2 + 1 + 1) / t, "kept": r["kept"] / (npsh * M), "dz": r["dz"],
                          "cy": r["cy"], "rmsY": r["rmsY"],
                          "radgratW_per_ray_wavelengths": {"order": -1, "wave": "uniform(3.6,7.2) nm", "ms": 1e3 * tw,
                                                           "rays_per_s": npsh * M / tw, "kept": rw["kept"] / (npsh * M)},
                          "parity": par}
    # ---- config 5: nested assembly, 260 shells; 1e9 rays over 8 GPUs = 1.25e8 per GPU (weak scaling)
    S = 260
    nps = max(10, int(1.25e8 * sc) // S)
    per_gpu = nps * S

    def c5():
        res = ex.config5_fast(nps, S, offaxis=0., rng="philox", device=dev, first=rank * per_gpu,
                              analyses=pxf.dist if world > 1 else None)
        return {k: v for k, v in res.items() if k not in ("rays", "weights")}
    t, r = timed(c5)
    if world > 1:
        import torch.distributed as td
        tt = torch.tensor([t, float(r["kept"])], dtype=torch.float64, device=dev)
        td.all_reduce(tt[:1], op=td.ReduceOp.MAX)
        td.all_reduce(tt[1:], op=td.ReduceOp.SUM)
        t, kept = float(tt[0]), float(tt[1])
    else:
        kept = float(r["kept"])
    par = None
    if gold is not None and world == 1:
        g = gold["c5_scalars"]
        p = ex.config5_fast(sizes["c5_n"], sizes["c5_shells"], offaxis=1. / 60. * np.pi / 180.)
        e = max(rel(p["hpd"], g[1]), rel(p["rms"], g[2]))
        par = {"vs": "tests/golden/configs.npz, %d shells x %d rays, 1 arcmin off axis" % (sizes["c5_shells"], sizes["c5_n"]),
               "kept_equal": bool(p["kept"] == g[0]), "worst_rel_err_hpd_rms": e, "ok": bool(p["kept"] == g[0] and e <= 1e-9)}
    out["config5"] = {"workload": "nested Wolter-I assembly, 260 shells: annulus, transform, wolterprimary, kick, reflect, "
                                  "woltersecondary, reflect, vignette(z range), transform, flat, vignette(rho > back of previous "
                                  "shell), transform, flat -- ONE segmented launch -- compaction of rays + area weights, weighted "
                                  "centroid / rms / hpd (all-reduced over ranks for N > 1)",
                      "rays_per_gpu": per_gpu, "total_rays": per_gpu * world, "shells": S, "ms": 1e3 * t,
                      "rays_per_s": per_gpu * world / t, "interactions_per_s": per_gpu * world * 4 / t,
                      "kept": kept / (per_gpu * world), "hpd_weighted": r["hpd"], "rms_weighted": r["rms"], "parity": par}
    return out


def run_e2e(args, pxf, pdist, src, prog, n, world, dev, barrier):
    """Same step through ``pxf_host_trace_program``: the bundle lives in pinned HOST memory,
    every step uploads the rows the chain reads, runs the fused kernel chunk by chunk, downloads
    every row it writes back into the host arrays (the f2py in-place contract) and returns the
    HPD.  For N>1 each rank keeps its final x,y on the device and the HPD is the global one."""
    import torch
    import torch.distributed as td
    rank = int(os.environ.get("RANK", "0"))
    try:
        host = [None] + [torch.empty(n, dtype=torch.float64).pin_memory() for _ in range(9)]
    except RuntimeError as e:
        return {"value": None, "unit": "rays/s", "error": "pinned allocation failed: %s" % str(e)[:80]}
    pristine = [None] + [src[k].cpu() for k in range(1, 7)]
    keep = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(2)] if world > 1 else None
    rays10 = [None] + [None] * 9

    def reset():
        for k in range(1, 7):
            host[k].copy_(pristine[k])

    def one():
        if world > 1:
            pxf.host.trace(host, prog, write_back=True, keep_xy=keep, const_rows=pxf.host.SOURCE_CONST_ROWS)
            rays10[1], rays10[2] = keep
            for k in range(3, 10):
                rays10[k] = keep[0]          # placeholders; dist.hpd reads rows 1,2 only
            return pdist.hpd(rays10)
        return pxf.host.trace(host, prog, write_back=True, hpd=True, const_rows=pxf.host.SOURCE_CONST_ROWS)["hpd"]

    reset()
    one()                                             # warm-up (allocator, page tables)
    t = 0.
    hp = None
    steps = max(1, args.e2e_steps)
    for _ in range(steps):
        reset()
        barrier()
        t0 = time.perf_counter()
        hp = one()
        torch.cuda.synchronize()
        t += time.perf_counter() - t0
    if world > 1:
        tt = torch.tensor([t], dtype=torch.float64, device=dev)
        td.all_reduce(tt, op=td.ReduceOp.MAX)
        t = float(tt[0])
    return {"value": n * world * steps / t, "unit": "rays/s", "steps": steps,
            # x, y uploaded; z, l, m, n of the subannulus source are constant over the bundle: the caller says so
            # (host.SOURCE_CONST_ROWS) and they are filled on the device instead of scanned and uploaded
            "h2d_bytes_per_step": 16 * n * world, "d2h_bytes_per_step": 40 * n * world + 8,
            "host_scanned_bytes_per_step": 0, "host_filled_bytes_per_step": 24 * n * world,
            "path": "pxf_host_trace_program: pinned host rows -> chunked H2D / fused kernel / D2H on 3 streams "
                    "-> all nine rows mutated in place (z,l,m,n of the source are constant rows the caller vouches for: "
                    "filled on the device, not uploaded; x,y,l,m,n downloaded; z=0 and the normal (0,0,1) left by flat "
                    "are written -- or, when the arrays already hold them, only verified -- by host threads instead of "
                    "crossing PCIe) + HPD", "hpd": hp}


def emit(line):
    """The one JSON line, on the real stdout."""
    sys.stdout.flush()
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


if __name__ == "__main__":
    a = parse()
    # rank 0 prints exactly ONE line on stdout: anything a library writes to fd 1 meanwhile (NCCL prints its
    # version banner there when NCCL_DEBUG is set) goes to stderr instead
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if a.impl == "reference":
        run_reference(a)
    else:
        run_engine(a)
