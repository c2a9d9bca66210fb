"""bench.py — eigsolve(Lanczos) iterations/sec on the 1e7 x 1e7 CSR 5-point Laplacian
(BASELINE.json configs[1]), Float64, krylovdim = 60, ClassicalGramSchmidt2, 5 restart cycles.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (N > 1)

A "step" is one whole eigsolve job: Lanczos factorization to krylovdim 60, then 4 thick
restarts (keep 36, re-expand 24) = 156 operator applications (`info.numops`), with the
convergence tolerance at 0 so the amount of work is fixed.  The metric is operator
applications per second (KrylovKit's numops/s, SURVEY §5 "iterations/sec").

  value    : inputs (A as CSR, x0) already resident in HBM when the timed region starts,
             timed with CUDA events on the library's stream, max over ranks.
  e2e      : the same job through the host-buffer API — kk.eigsolve(A_csr_host, x0_host, ...):
             context creation, H2D of A and x0 from pinned memory, the solve, D2H of the Ritz
             vectors into pinned memory, all inside the timed region (wall clock around
             device-synchronised calls).
  roofline : the fused Gram-Schmidt sweep (the dominant kernel): algorithmic bytes
             (2k+3)*8n per launch (SURVEY §8d "one CGS pass", k = basis size incl. the new
             vector) summed over the launches of the timed region / their summed device time
             (CUDA events around every launch, on the launching stream), vs the measured HBM
             peak in MEASURED_PEAKS.json.
  cpu_baseline : the restated reference path (oracle/krylov_oracle.py; its n-length loops run in the
             OpenMP kernels of oracle/csrc/kernels.c on all host cores, like KrylovKit's own
             multi-threaded Array fast path; no Julia in the image) on a bounded sample of the
             same workload at full n: initialize + 30 expand! steps (31 operator applications at
             basis sizes 1..31 — the cheap early part of a cycle, so the CPU figure is optimistic).
  --impl reference : the same CPU path on the WHOLE job (the oracle's eigsolve driver with the same restart
             cycles), as many whole jobs as fit a ~200 s budget (steps_timed); prints its Ritz values.
  parity   : every arm asserts its Ritz values against the oracle's committed full-size results
             (tests/golden/fullsize.json): <= 1e-10 relative (+ 4 ulp(||A||) floor), numops equal.
  other_configs : BASELINE.json configs 3, 4, 5 measured after the headline, with their own parity evidence.
  --dump-outputs DIR : what the last timed job returned (Ritz values, ConvergenceInfo, the Ritz and residual vectors
             at a fixed, seeded sample of rows) as float64 DIR/<name>.npy, about 38 MB in all: the inputs are
             seeded, so two builds run with the same arguments can be compared output for output.

N > 1: STRONG scaling — the same 1e7-row problem row-sharded over N ranks; halo rows, <v,Av>, the projection
coefficients and ||w||^2 are exchanged inside the two kernels of a step through the NVLink peer window
(DESIGN.md §4; B2K_PEER=0 falls back to NCCL calls between the sweeps).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os

# libgomp reads this once, when it is first loaded (torch loads it): idle OpenMP workers of the CPU baseline
# must sleep, not spin, on hosts whose logical CPUs are shared
os.environ.setdefault("OMP_WAIT_POLICY", "passive")
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 20260923
HOWMANY = 4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nx", type=int, default=4000)
    ap.add_argument("--ny", type=int, default=2500)
    ap.add_argument("--krylovdim", type=int, default=60)
    ap.add_argument("--cycles", type=int, default=5)
    ap.add_argument("--orth", default="cgs2", choices=["cgs2", "mgs2", "cgs", "mgs", "mgs2b"])
    ap.add_argument("--cpu-steps", type=int, default=30, help="expand! steps in the CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--extra", default=None,
                    help="other BASELINE.json configs measured after the headline (records under 'other_configs'); "
                         "'' = none.  Default: c2f,c2m,w,c3,c4,c5,c4o on one GPU (c4o = config 4 in the flagged one-pass "
                         "GKL mode, run LAST: its kernel had not run on a B200 when the round's GPU budget ended); c5 — the "
                         "configuration BASELINE.json names for 8 GPUs — under torchrun")
    ap.add_argument("--c4-rows", type=int, default=2_000_000, help="rows of config 4's dense matrix (tests use fewer)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed job returned to DIR/<name>.npy (float64, one GPU, --impl ours)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if a.extra is None:
        a.extra = "c2f,c2m,w,c3,c4,c5,c4o" if int(os.environ.get("WORLD_SIZE", "1")) == 1 else "c5"
    return a


# ---------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def json_safe(obj):
    """json.dumps writes NaN / Infinity for non-finite floats, which a strict JSON parser rejects: the one line this
    script prints must stay parseable whatever an (extra) configuration measured, so they become strings."""
    if isinstance(obj, dict):
        return {str(k): json_safe(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return [json_safe(v) for v in obj]
    if isinstance(obj, (np.floating, float)):
        f = float(obj)
        return f if np.isfinite(f) else repr(f)
    if isinstance(obj, np.integer):
        return int(obj)
    if isinstance(obj, np.bool_):
        return bool(obj)
    if isinstance(obj, np.ndarray):
        return json_safe(obj.tolist())
    return obj


def pinned_array(lib, count, dtype):
    dt = np.dtype(dtype)
    p = C.c_void_p()
    st = lib.b2k_pinned_alloc(count * dt.itemsize, C.byref(p))
    if st != 0:
        raise MemoryError("cudaHostAlloc failed")
    buf = (C.c_byte * (count * dt.itemsize)).from_address(p.value)
    return np.frombuffer(buf, dtype=dt, count=count), p


# --------------------------------------------------------------------------------------- CPU arm
def _cpu_backend():
    """The restated reference's n-length loops: OpenMP kernels (oracle/csrc/kernels.c — KrylovKit runs its
    Array fast path multi-threaded too, orthonormal.jl:66-73) when they can be loaded, else plain numpy."""
    import contextlib
    try:
        from oracle import native
        if native.available():
            return native, native.patched, native.num_threads(), "OpenMP kernels oracle/csrc/kernels.c"
    except Exception:
        pass
    return None, contextlib.nullcontext, 1, "numpy+OpenBLAS, scipy CSR matvec"


def _cpu_operator(nx, ny, native):
    """Host operator; with the OpenMP backend also settles the thread count by a short calibration
    (nproc threads are not always the fastest choice on a shared box) and logs the host's CPU limits."""
    from oracle import krylov_oracle as ko
    A = ko.stencil_matrix(nx, ny)
    if native is None:
        return A
    An = native.CSR(A)
    log = lambda m: print(m, file=sys.stderr, flush=True)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us", "/proc/loadavg"):
        try:
            log(f"host: {path} = {open(path).read().strip()}")
        except OSError:
            pass
    t = native.calibrate(An, ko.splitmix_vector(SEED, nx * ny), verbose=log)
    log(f"host: using {t} OpenMP threads of {os.cpu_count()} logical CPUs")
    return An


def _cpu_host_note():
    """'N threads; cgroup CPU quota Q of M logical CPUs' — what the CPU legs really had."""
    note = f"{os.cpu_count()} logical CPUs"
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            note += f", cgroup CPU quota {float(q) / float(per):g}"
    except (OSError, ValueError):
        pass
    return note


def cpu_sample(nx, ny, krylovdim, orth_name, nsteps, A=None):
    """Restated reference path on the host cores: initialize + nsteps expand! at full n."""
    from oracle import krylov_oracle as ko
    native, patched, _, _ = _cpu_backend()
    orth = {"cgs2": ko.Orth(ko.CGS2), "mgs2": ko.Orth(ko.MGS2), "cgs": ko.Orth(ko.CGS),
            "mgs": ko.Orth(ko.MGS), "mgs2b": ko.Orth(ko.MGS2)}[orth_name]       # mgs2b is OUR flagged mode of MGS2
    if A is None:
        A = _cpu_operator(nx, ny, native)
    x0 = ko.splitmix_vector(SEED, nx * ny)
    with patched():
        t0 = time.perf_counter()
        f = ko.lanczos_initialize(A, x0, orth)
        for _ in range(nsteps):
            f = ko.lanczos_expand(A, f, orth)
        dt = time.perf_counter() - t0
    numops = nsteps + 1
    return numops / dt, dt, numops


def cpu_full_job(a, A):
    """The whole workload on the host cores: the oracle's eigsolve driver, same restart cycles."""
    from oracle import krylov_oracle as ko
    _, patched, _, _ = _cpu_backend()
    orth = {"cgs2": ko.Orth(ko.CGS2), "mgs2": ko.Orth(ko.MGS2), "cgs": ko.Orth(ko.CGS), "mgs": ko.Orth(ko.MGS),
            "mgs2b": ko.Orth(ko.MGS2)}[a.orth]
    x0 = ko.splitmix_vector(SEED, a.nx * a.ny)
    with patched():
        t0 = time.perf_counter()
        vals, vecs, info = ko.eigsolve_lanczos(A, x0, HOWMANY, "SR", krylovdim=a.krylovdim, maxiter=a.cycles,
                                               tol=0.0, orth=orth)
        dt = time.perf_counter() - t0
    return info["numops"] / dt, dt, info["numops"], vals


def golden_case(a):
    """The oracle's committed full-size results for this workload (tests/golden/fullsize.json, written by
    tests/golden/make_fullsize_golden.py) or None when the command line asks for another workload."""
    p = os.path.join(ROOT, "tests", "golden", "fullsize.json")
    if not os.path.exists(p):
        return None
    g = json.load(open(p))
    for name in ("c2", "c2_mgs2", "c2_1e6"):
        c = g.get(name)
        if c and c["grid"] == [a.nx, a.ny, 1] and c["krylovdim"] == a.krylovdim \
                and c["orth"] == ("mgs2" if a.orth == "mgs2b" else a.orth) \
                and str(a.cycles) in c["after_cycles"]:
            return {"name": f"tests/golden/fullsize.json:{name}:after_cycles[{a.cycles}]", **c["after_cycles"][str(a.cycles)]}
    return None


def check_parity(a, vals, numops, what):
    """Ritz values of this run vs the oracle's on the same (A, x0): <= 1e-10 relative (north_star), numops equal."""
    g = golden_case(a)
    if g is None:
        return {"checked": False, "why": "no committed oracle result for this workload"}
    ref = np.array(g["ritz"])
    diff = np.abs(np.array(vals[:len(ref)]) - ref)
    rel = float(np.max(diff / np.abs(ref)))
    # 1e-10 relative (north_star), with the floor any Ritz value of this operator has: a few ulps of ||A|| = 8.
    # (lambda_1 ~ 1.3e-5 here, so 1e-10 relative IS 1.3e-15 absolute ~ 1.5 ulp of ||A||: two correct summation
    # orders of the same algorithm differ by that much — round 1's GPU run vs the oracle: 7.8e-11.)
    floor = 4 * 8.0 * np.finfo(np.float64).eps
    ok = bool(np.all(diff <= 1e-10 * np.abs(ref) + floor)) and int(numops) == int(g["numops"])
    out = {"checked": True, "against": g["name"] + " (oracle/krylov_oracle.py at full size)", "max_rel_diff_ritz": rel,
           "max_abs_diff_ritz": float(diff.max()), "tolerance": "1e-10 relative + 4 ulp(||A||) absolute",
           "numops": int(numops), "numops_oracle": int(g["numops"]), "ok": bool(ok)}
    if not ok:
        raise AssertionError(f"{what}: parity with the oracle lost: {out}; ritz = {list(vals[:len(ref)])}, oracle = {list(ref)}")
    return out


def run_reference(a):
    """The reference arm runs the SAME job as the GPU arm — the whole eigsolve (krylovdim expansion + restart
    cycles, `numops` operator applications) — through the restated reference on the host cores.  The number of
    timed jobs is capped (a whole job costs ~10-20 s of the box's CPU quota) independently of --steps, and is
    reported as steps_timed; the Ritz values of the last job are printed so both arms can be compared."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    native, _, cores, backend = _cpu_backend()
    A = _cpu_operator(a.nx, a.ny, native)
    if native is not None:
        cores = native.num_threads()                 # the calibrated thread count
    backend += f" with {cores} threads ({_cpu_host_note()})"
    # one short untimed sample (also the warm-up) sizes the run: whole jobs only, as many as fit ~200 s
    # (the cost of a step grows with the basis size: the job averages ~3x the cost of the first four steps)
    _, dt_w, ops_w = cpu_sample(a.nx, a.ny, a.krylovdim, a.orth, 4, A)
    budget_s = 200.0
    per_op = dt_w / ops_w
    job_ops = a.krylovdim + (a.cycles - 1) * (a.krylovdim - (3 * a.krylovdim) // 5)
    est_job = 3.0 * per_op * job_ops
    jobs = int(max(1, min(a.steps, budget_s // max(est_job, 1e-9))))
    t_tot, ops_tot, vals = 0.0, 0, None
    for _ in range(jobs):
        v, dt, ops, vals = cpu_full_job(a, A)
        t_tot += dt
        ops_tot += ops
        if t_tot > budget_s:
            jobs = _ + 1
            break
    sample = (f"the WHOLE job, {jobs} time(s) ({ops_tot // jobs} operator applications per job, {a.cycles} restart "
              f"cycles) through oracle/krylov_oracle.py eigsolve_lanczos; n-length loops: {backend}")
    value = ops_tot / t_tot
    parity = check_parity(a, vals, ops_tot // jobs, "reference arm (oracle on this host)")
    line = {
        "impl": "reference", "metric": "eigsolve_lanczos_operator_applications_per_sec", "value": value,
        "unit": "it/s", "n_gpus": a.gpus, "steps": a.steps, "steps_timed": jobs, "warmup": a.warmup,
        "ms_per_step": 1000.0 * t_tot / jobs, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(a), "numops_per_step": ops_tot // jobs,
        "ritz_values": [float(x) for x in vals[:HOWMANY]], "parity": parity,
        "cpu_baseline": {"value": value, "unit": "it/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(json_safe(line), allow_nan=False, default=str), flush=True)


DUMP_ROWS = 1 << 19      # rows of each Ritz / residual vector in a dump: 2 * HOWMANY * 4 MiB + the row list


def dump_outputs(out_dir, vals, vecs, info):
    """Write what an eigsolve call returned to out_dir as float64 .npy files: the Ritz values, the ConvergenceInfo
    numbers (normres; converged, numiter, numops) and the Ritz and residual vectors at DUMP_ROWS rows drawn with a
    fixed seed (sample_rows.npy; every row when n is smaller).  Whole vectors at n = 1e7 would be 640 MB."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(vecs[0])
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(SEED).choice(n, DUMP_ROWS, replace=False))
    arrays = {
        "ritz_values": np.asarray(vals, dtype=np.float64),
        "ritz_vectors": np.stack([v.to_host()[rows] for v in vecs]).astype(np.float64),
        "residuals": np.stack([r.to_host()[rows] for r in info.residual]).astype(np.float64),
        "normres": np.asarray(info.normres, dtype=np.float64),
        "counts": np.array([info.converged, info.numiter, info.numops], dtype=np.float64),
        "sample_rows": rows.astype(np.float64),
    }
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), arr)


def workload_config(a):
    return {"workload": f"eigsolve(Lanczos, :SR, {HOWMANY}) on the {a.nx * a.ny}x{a.nx * a.ny} CSR 5-point "
                        f"Laplacian ({a.nx}x{a.ny} grid, Dirichlet), Float64, krylovdim={a.krylovdim}, "
                        f"orth={a.orth}, {a.cycles} restart cycles (tol=0: fixed work)",
            "n": a.nx * a.ny, "krylovdim": a.krylovdim, "restart_cycles": a.cycles, "orth": a.orth,
            "l2": "inputs (4.9 GB basis, 0.8 GB matrix) >> 126 MB L2; no explicit flush",
            "parallelism": f"rows sharded over {a.gpus} GPU(s)" if a.gpus > 1 else "single GPU"}


# --------------------------------------------------------------------------------------- GPU arm
def run_ours(a):
    import krylovkit_jl_b200 as kk
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        if world == 1 and a.gpus > 1:
            raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    if a.dump_outputs and world > 1:
        raise SystemExit("bench.py --dump-outputs writes the outputs of a one-GPU run: use it with --gpus 1")
    dist = None
    n = a.nx * a.ny
    orth = {"cgs2": kk.cgs2, "mgs2": kk.mgs2, "cgs": kk.cgs, "mgs": kk.mgs, "mgs2b": kk.mgs2b}[a.orth]
    alg = kk.Lanczos(orth=orth, krylovdim=a.krylovdim, maxiter=a.cycles, tol=0.0, verbosity=0)
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        from krylovkit_jl_b200 import sharding
        uid_bytes = sharding.broadcast_nccl_uid(dist, kk._lib.load())
        shard = sharding.shard_grid_lines(a.nx, a.ny, rank, world)      # whole grid lines per rank
        ctx = kk.B200Context(shard.n_local, a.krylovdim + 2 * HOWMANY + 8, device=local_rank, rank=rank,
                             nranks=world, nccl_uid=uid_bytes, n_global=n, row_offset=shard.row_offset)
    else:
        ctx = kk.B200Context(n, a.krylovdim + 2 * HOWMANY + 8, device=local_rank)
    lib = ctx.lib
    op = kk.B200CSR.stencil(ctx, a.nx, a.ny)
    x0 = ctx.splitmix(SEED)

    def job():
        return kk.eigsolve(op, x0, HOWMANY, "SR", alg)

    def barrier():
        if dist is not None:
            dist.barrier()
        lib.b2k_device_sync()

    for _ in range(a.warmup):
        vals, vecs, info = job()
        del vecs
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    lib.b2k_prof_reset(ctx.h)
    lib.b2k_prof_enable(ctx.h, 1)
    import importlib
    _es = importlib.import_module("krylovkit_jl_b200.eigsolve")   # the module (kk.eigsolve is the function)
    _es.HOSTPROF = {}                      # wall seconds the host spends per driver section (incl. waiting)
    launches0 = ctx.launches
    barrier()
    lib.b2k_timer_start(ctx.h)
    t0 = time.perf_counter()
    numops = 0
    for i in range(a.steps):
        vals, vecs, info = job()
        numops += info.numops
        if i + 1 < a.steps or not a.dump_outputs:
            del vecs
    ms = C.c_double()
    lib.b2k_timer_stop(ctx.h, C.byref(ms))
    barrier()
    wall = time.perf_counter() - t0
    lib.b2k_prof_enable(ctx.h, 0)
    host_ms = {k: round(1000.0 * v / a.steps, 3) for k, v in _es.HOSTPROF.items()}
    _es.HOSTPROF = None
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launches - launches0
    t_dev = ms.value / 1000.0
    if dist is not None:
        import torch
        tt = torch.tensor([t_dev], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_dev = float(tt.item())
        ll = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(ll)
        launches = int(ll.item())
    value = numops / t_dev
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, vals, vecs, info)
        del vecs
    parity = check_parity(a, vals, numops // a.steps, "device-resident path")     # every rank: values are replicated

    # roofline of the dominant kernel (fused Gram-Schmidt sweep) + SpMV beside it
    def prof(cls):
        c, m, b = C.c_int64(), C.c_double(), C.c_double()
        lib.b2k_prof_read(ctx.h, cls, C.byref(c), C.byref(m), C.byref(b))
        return c.value, m.value, b.value
    pk, pk_kind = peak_hbm()
    kern = {}
    for cls, name in ((1, "gs_fused"), (0, "spmv_csr"), (2, "basis_transform")):
        c, m, b = prof(cls)
        if c:
            kern[name] = {"launches": c, "ms_total": round(m, 3), "avg_ms": round(m / c, 4),
                          "GBs": round(b / m / 1e6, 1), "frac": round(b / m / 1e6 / pk, 3),
                          "share_of_step": round(m / (ms.value), 3)}
    traffic, traffic_note = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        traffic = tj.get("gs_fused_bytes_per_launch")
        traffic_note = (f"dram__bytes_read+write of one ncu --set full capture ({tj.get('captured_launch')}); "
                        f"algorithmic bytes of that launch {tj.get('algorithmic_bytes_same_launch')}")
    gs = kern.get("gs_fused", {})
    roofline = {"kernel": "k_gs_fused<double> (3-term prologue + project, grid barrier, update + norm)",
                "bound": "hbm", "achieved": gs.get("GBs"), "peak": pk, "unit": "GB/s",
                "frac": gs.get("frac"), "peak_kind": pk_kind, "traffic": traffic, "traffic_note": traffic_note,
                "algorithmic_bytes": "(2k+3)*8n per launch, k = basis size incl. the new vector; summed over launches",
                "avg_launch_ms": gs.get("avg_ms"),
                "includes": ("kernel only" if world == 1 else
                             "kernel INCLUDING its in-kernel cross-GPU exchanges over the NVLink peer window (waiting for "
                             "<v,Av>, the coefficient sum at the phase boundary and ||w||^2 of the slowest rank): at "
                             "N > 1 this is kernel + collective time, not a pure HBM figure")}

    # ---- end to end through the host-buffer API: every rank uploads ITS rows of A (CSR with global
    # column indices) and its slice of x0 from pinned memory, solves, downloads its slice of the vectors
    e2e = None
    if not a.no_e2e:
        n_loc = op.n_rows
        rp, prp = pinned_array(lib, n_loc + 1, np.int32)
        ci, pci = pinned_array(lib, op.nnz, np.int32)
        va, pva = pinned_array(lib, op.nnz, np.float64)
        ctx.check(lib.b2k_op_csr_download(ctx.h, op.h, rp.ctypes.data, ci.ctypes.data, va.ctypes.data))
        shard, uid2 = None, None
        if world > 1:
            # the device stores localised columns ([local | lo halo | hi halo]); undo that to get
            # the global indices a user would hand over (5-point stencil: one grid line of halo)
            from krylovkit_jl_b200 import sharding
            shard = sharding.shard_grid_lines(a.nx, a.ny, rank, world)
            lo = a.nx if rank > 0 else 0
            loc = ci.astype(np.int64)
            glob = np.where(loc < n_loc, loc + shard.row_offset,
                            np.where(loc < n_loc + lo, loc - n_loc + shard.row_offset - lo,
                                     loc - n_loc - lo + shard.row_offset + n_loc))
            ci[:] = glob.astype(np.int32)
            import torch
            uid2 = sharding.broadcast_nccl_uid(dist, lib)
        xh, pxh = pinned_array(lib, n_loc, np.float64)
        x0.to_host(xh)
        # the resident context is no longer needed: closing it returns its slab to the library's
        # block cache and (N > 1) its NCCL communicator to the per-process cache, so the per-call
        # contexts of the host-buffer path reuse both instead of paying for new ones
        ctx.close()
        outs = [pinned_array(lib, n_loc, np.float64) for _ in range(HOWMANY)]
        out_arrs = [o[0] for o in outs]
        h2d = rp.nbytes + ci.nbytes + va.nbytes + xh.nbytes
        d2h = sum(o.nbytes for o in out_arrs) + 8 * HOWMANY

        def job_e2e():
            return kk.eigsolve((rp, ci, va), xh, HOWMANY, "SR", alg, out_vectors=out_arrs, shard=shard,
                               nccl_uid=uid2, device=local_rank)

        for _ in range(max(1, min(a.warmup, 2))):
            job_e2e()
        barrier()
        t0 = time.perf_counter()
        ops = 0
        for _ in range(a.steps):
            v2, vec2, info2 = job_e2e()
            ops += info2.numops
        barrier()
        te = time.perf_counter() - t0
        assert np.allclose(v2, vals, rtol=1e-10), (v2, vals)
        parity_e2e = check_parity(a, v2, ops // a.steps, "host-buffer (e2e) path")
        if dist is not None:
            import torch
            tt = torch.tensor([te, float(h2d), float(d2h)], dtype=torch.float64, device="cuda")
            tmax = tt.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(tt)
            te, h2d, d2h = float(tmax[0].item()), float(tt[1].item()), float(tt[2].item())
        e2e = {"value": ops / te, "unit": "it/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": 1000.0 * te / a.steps,
               "path": "kk.eigsolve(csr_host_arrays, x0_host, ...) on every rank: ctx create + H2D (pinned) + solve "
                       "+ D2H (pinned); wall clock, max over ranks; bytes summed over ranks.  Steady state: the "
                       "library's block cache (slab, CSR arrays) and the per-process NCCL communicator are warm "
                       "from the previous call, so cudaMalloc / ncclCommInitRank of a first call are not in it",
               "parity": parity_e2e}
        for p in (prp, pci, pva, pxh, *[o[1] for o in outs]):
            lib.b2k_pinned_free(p)

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        native, _, cores, backend = _cpu_backend()
        A_host = _cpu_operator(a.nx, a.ny, native)
        if native is not None:
            cores = native.num_threads()             # the calibrated thread count
        backend += f" with {cores} threads ({_cpu_host_note()})"
        v, dt, ops = cpu_sample(a.nx, a.ny, a.krylovdim, a.orth, a.cpu_steps, A_host)
        cpu = {"value": v, "unit": "it/s", "cores": cores, "kind": "port",
               "sample": f"initialize + {a.cpu_steps} expand! steps ({ops} operator applications, basis sizes "
                         f"1..{a.cpu_steps + 1}) of the same n={n} job in {dt:.1f} s; oracle/krylov_oracle.py "
                         f"(restated reference; n-length loops: {backend}); no Julia in the image"}

    extras = None
    if a.extra:
        if not a.no_e2e:
            pass                                   # the resident context was closed before the e2e leg
        else:
            ctx.close()
        lib.b2k_cache_release()                    # config 5 needs 31 GB on one GPU: start from a clean allocator
        extras = other_configs(kk, a, rank, world, local_rank, dist)

    if rank == 0:
        line = {
            "metric": "eigsolve_lanczos_operator_applications_per_sec", "value": value, "unit": "it/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1000.0 * t_dev / a.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(a),
            "numops_per_step": numops // a.steps, "wall_s": wall, "host_ms_per_step": host_ms,
            "ritz_values": [float(v) for v in vals[:HOWMANY]], "parity": parity,
            "roofline": roofline, "kernels": kern, "cpu_baseline": cpu, "e2e": e2e, "other_configs": extras,
            "gpu_launches": int(launches), "clocks": clocks,
        }
        print(json.dumps(json_safe(line), allow_nan=False, default=str), flush=True)
    ctx.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------- other configs
def other_configs(kk, a, rank, world, local_rank, dist):
    """BASELINE.json configs[2..4] on the same box, after the headline measurement: one warm-up + one timed job
    each (CUDA events on the library stream, max over ranks), with the parity evidence that exists at full size:
    the oracle's committed results (tests/golden/fullsize.json) for config 3, residual identities evaluated on the
    device for config 4, the closed-form lower bound + cross-N agreement for config 5."""
    from krylovkit_jl_b200 import sharding
    lib = kk._lib.load()
    want = [w for w in a.extra.split(",") if w]
    gold = {}
    gp = os.path.join(ROOT, "tests", "golden", "fullsize.json")
    if os.path.exists(gp):
        gold = json.load(open(gp))
    out = {}

    def c4_truth_err(sig, m, nn):
        """max relative distance of the leading singular values from the Float64 truth of the same matrix
        (tests/golden/fullsize.json:c4_truth, sqrt eig of the Float64 Gram matrix) or None at another shape"""
        g = gold.get("c4_truth")
        if not g or g.get("shape") != [m, nn]:
            return None
        ref = np.array(g["sigma_float64_truth"])
        k = min(len(ref), len(sig))
        return float(np.max(np.abs(np.array(sig[:k], dtype=np.float64) - ref[:k]) / ref[:k]))

    def config_failed(e, ctx):
        """an exception inside one of the extra configs (raised alike on every rank: the host logic is
        rank-replicated) becomes that config's record; its context is closed so the next one finds the memory"""
        import traceback
        sys.stderr.write(traceback.format_exc())
        try:
            if ctx is not None:
                ctx.close()
        except Exception:
            pass
        return {"ok": False, "error": f"{type(e).__name__}: {e}"[:600]}

    def make_ctx(n_lines, line, ncols, dtype=np.float64):
        n = n_lines * line
        if world == 1:
            return kk.B200Context(n, ncols, dtype=dtype, device=local_rank), n
        import torch
        u = sharding.broadcast_nccl_uid(dist, lib)
        sh = sharding.shard_grid_lines(line, n_lines, rank, world)
        return kk.B200Context(sh.n_local, ncols, dtype=dtype, device=local_rank, rank=rank, nranks=world, nccl_uid=u,
                              n_global=n, row_offset=sh.row_offset), n

    def timed(ctx, fn):
        fn()
        lib.b2k_device_sync()
        if dist is not None:
            dist.barrier()
        lib.b2k_timer_start(ctx.h)
        res = fn()
        ms = C.c_double()
        lib.b2k_timer_stop(ctx.h, C.byref(ms))
        t = ms.value / 1000.0
        if dist is not None:
            import torch
            tt = torch.tensor([t], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t = float(tt.item())
        return res, t

    if "c2f" in want:
        ctx = None
        try:
            # the headline job with the MATRIX-FREE stencil operator (KrylovKit takes any function as its linear map):
            # same arithmetic, same Ritz values, 16n instead of 12 nnz + 20n bytes per operator application
            ctx, n = make_ctx(a.ny, a.nx, a.krylovdim + 2 * HOWMANY + 8)
            op = kk.B200CSR.stencil_free(ctx, a.nx, a.ny)
            x0 = ctx.splitmix(SEED)
            orth = {"cgs2": kk.cgs2, "mgs2": kk.mgs2, "cgs": kk.cgs, "mgs": kk.mgs, "mgs2b": kk.mgs2b}[a.orth]
            alg = kk.Lanczos(orth=orth, krylovdim=a.krylovdim, maxiter=a.cycles, tol=0.0, verbosity=0)
            (vals, vecs, info), t = timed(ctx, lambda: kk.eigsolve(op, x0, HOWMANY, "SR", alg))
            del vecs
            out["c2_matrix_free"] = {
                "workload": workload_config(a)["workload"].replace("CSR 5-point", "matrix-free 5-point"),
                "numops": info.numops, "ms": 1000 * t, "value": info.numops / t, "unit": "it/s",
                "ritz": [float(v) for v in vals[:HOWMANY]], "parity": check_parity(a, vals, info.numops, "matrix-free operator")}
            ctx.close()
        except Exception as e:      # the headline line must still be printed: record the failure instead
            out["c2_matrix_free"] = config_failed(e, ctx)

    if "c2m" in want:
        # the headline job with the REFERENCE-DEFAULT orthogonalizer (KrylovDefaults.orth = ModifiedGramSchmidt2,
        # algorithms.jl:558): literal MGS2 and the flagged blocked form kk.mgs2b (DESIGN §3.7).  Timed on the same
        # restart cycles as the headline; parity on the 2-cycle job the oracle's full-size MGS2 result exists for.
        ctx = None
        try:
            ctx, n = make_ctx(a.ny, a.nx, a.krylovdim + 2 * HOWMANY + 8)
            op = kk.B200CSR.stencil(ctx, a.nx, a.ny)
            x0 = ctx.splitmix(SEED)
            gm = gold.get("c2_mgs2", {})
            g2 = gm.get("after_cycles", {}).get("2") if gm.get("grid") == [a.nx, a.ny, 1] and gm.get("krylovdim") == a.krylovdim else None
            rec = {"workload": workload_config(a)["workload"].replace(f"orth={a.orth}", "orth=mgs2 (reference default) / mgs2b (flagged blocked form)")}
            for name, orth in (("mgs2_reference_default", kk.mgs2), ("mgs2_blocked_flagged", kk.mgs2b)):
                alg = kk.Lanczos(orth=orth, krylovdim=a.krylovdim, maxiter=a.cycles, tol=0.0, verbosity=0)
                (vals, vecs, info), t = timed(ctx, lambda: kk.eigsolve(op, x0, HOWMANY, "SR", alg))
                r = {"numops": info.numops, "ms": 1000 * t, "value": info.numops / t, "unit": "it/s",
                     "ritz": [float(v) for v in vals[:HOWMANY]]}
                del vecs, info                    # Ritz vectors and residuals hold slab columns the next solve needs
                if g2:
                    alg2 = kk.Lanczos(orth=orth, krylovdim=a.krylovdim, maxiter=2, tol=0.0, verbosity=0)
                    v2, vecs2, info2 = kk.eigsolve(op, x0, HOWMANY, "SR", alg2)
                    numops2 = int(info2.numops)
                    del vecs2, info2
                    ref = np.array(g2["ritz"])
                    diff = np.abs(np.array(v2[:len(ref)]) - ref)
                    floor = 4 * 8.0 * np.finfo(np.float64).eps
                    r["parity"] = {"against": "tests/golden/fullsize.json:c2_mgs2:after_cycles[2] (the oracle's literal MGS2 at full size)",
                                   "max_rel_diff_ritz": float(np.max(diff / np.abs(ref))), "max_abs_diff_ritz": float(diff.max()),
                                   "numops": numops2, "numops_oracle": int(g2["numops"]),
                                   "ok": bool(np.all(diff <= 1e-10 * np.abs(ref) + floor) and numops2 == int(g2["numops"]))}
                rec[name] = r
            out["c2_reference_default_orth"] = rec
            ctx.close()
        except Exception as e:      # the headline line must still be printed: record the failure instead
            out["c2_reference_default_orth"] = config_failed(e, ctx)

    if "w" in want and world == 1:
        # the widened solvers (SURVEY §8f-2/3/4) at the 1e7 scale, as tools/run_configs.py measures them: CG (device-
        # chained / one call per iteration / literal), BiCGStab (chained vs literal), Arnoldi eigsolve, BlockLanczos
        # p = 4 in the reference mode and the flagged block mode, exponentiate — each with its residual identity
        ctx = None
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("_b2k_run_configs", os.path.join(ROOT, "tools", "run_configs.py"))
            rc = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(rc)
            rec = {"workload": "linsolve(CG, 200 iterations) / linsolve(BiCGStab, 40) / eigsolve(Arnoldi, krylovdim 30, 3 cycles) / "
                               "eigsolve(BlockLanczos p = 4, krylovdim 32, 3 cycles) / exponentiate(Lanczos 30) on the 1e7-row 5-point "
                               "operators (tools/run_configs.py cg, widened)",
                   "cg": rc.cg()}
            rec.update(rc.widened(lsmr=False))
            out["widened_solvers"] = rec
        except Exception as e:      # the headline line must still be printed: record the failure instead
            out["widened_solvers"] = config_failed(e, ctx)

    if "c3" in want:
        ctx = None
        try:
            nx, ny, kd = 4000, 2500, 40
            ctx, n = make_ctx(ny, nx, kd + 16)
            op = kk.B200CSR.stencil(ctx, nx, ny, 1, (4.0, -1.4, -0.6, -1.2, -0.8, 0.0, 0.0))
            ones = ctx.full(1.0)
            b = kk.apply(op, ones)
            rec = {"workload": f"linsolve(GMRES, krylovdim={kd}) on the {n}x{n} convection-diffusion CSR (5-point, "
                               "nonsymmetric), b = A*1, x0 = 0, 5 restart cycles (tol -> 0: fixed work)"}
            for name, orth, gname in (("cgs2", kk.cgs2, "c3"), ("mgs2_reference_default", kk.mgs2, None),
                                      ("mgs2_blocked_flagged", kk.mgs2b, None)):
                alg = kk.GMRES(orth=orth, krylovdim=kd, maxiter=5, tol=1e-300, verbosity=0)
                (x, info), t = timed(ctx, lambda: kk.linsolve(op, b, None, alg))
                chk = kk.apply(op, x)
                chk.add_(info.residual, 1.0).add_(b, -1.0)          # b = A x + r  (test/linsolve.jl:230)
                r = {"numops": info.numops, "numiter": info.numiter, "ms": 1000 * t, "value": info.numops / t,
                     "unit": "it/s", "normres": float(info.normres), "||A x + r - b||/||b||": chk.norm() / b.norm()}
                g = gold.get(gname, {}).get("after_cycles", {}).get("5") if gname else None
                if g:
                    rel = abs(info.normres - g["normres"]) / g["normres"]
                    xn = x.norm()
                    r["parity"] = {"against": f"tests/golden/fullsize.json:{gname}:after_cycles[5] (oracle at full size)",
                                   "numops_oracle": g["numops"], "normres_rel_diff": rel,
                                   "x_norm_rel_diff": abs(xn - g["x_norm"]) / g["x_norm"],
                                   "ok": bool(info.numops == g["numops"] and rel <= 1e-8 and abs(xn - g["x_norm"]) <= 1e-10 * g["x_norm"])}
                    if not r["parity"]["ok"]:
                        raise AssertionError(f"config 3: parity with the oracle lost: {r}")
                rec[name] = r
                del x, info, chk
            out["c3"] = rec
            ctx.close()
        except Exception as e:      # the headline line must still be printed: record the failure instead
            out["c3"] = config_failed(e, ctx)

    if "c4" in want and world == 1:
        ctx = None
        try:
            m, nn, kd = a.c4_rows, 512, 30
            ctx = kk.B200Context(m, kd + 24, dtype=np.float32, device=local_rank)
            sv = ctx.add_space(nn, kd + 24, sharded=False)
            op = kk.B200Dense.splitmix(ctx, m, nn, SEED, sv)
            u0 = ctx.splitmix(SEED + 1)
            rec = {"workload": f"svdsolve(GKL, krylovdim={kd}, tol=1e-5) on the dense {m}x{nn} Float32 matrix (splitmix "
                               "entries in (-0.5, 0.5)), 6 triplets :LR",
                   "note": "with ClassicalGramSchmidt2 the Float32 recurrence loses orthogonality on this clustered spectrum "
                           "(in the CPU oracle too) and the driver raises B200Error; reported with the reference's default "
                           "orthogonalizer and with the iterative-refinement one its Float32 tests use (test/runtests.jl:18)"}
            for name, orth in (("mgs2_reference_default", kk.mgs2), ("cgsr_eta0.75", kk.ClassicalGramSchmidtIR(eta=0.75)),
                               ("cgs2", kk.cgs2)):
                alg = kk.GKL(orth=orth, krylovdim=kd, maxiter=100, tol=1e-5, verbosity=0)
                try:
                    (S, Lv, Rv, info), t = timed(ctx, lambda: kk.svdsolve(op, u0, 6, "LR", alg))
                except kk.B200Error as e:
                    rec[name] = {"raised": "B200Error: " + str(e)[:160]}
                    continue
                res = []
                for i in range(3):                                  # A v = s u + r, A' u = s v on the device
                    w = kk.apply_normal(op, Rv[i])
                    w.add_(Lv[i], -float(S[i]))
                    z = kk.apply_adjoint(op, Lv[i])
                    z.add_(Rv[i], -float(S[i]))
                    res.append([float(w.norm() / S[i]), float(z.norm() / S[i])])
                rec[name] = {"numops": info.numops, "numiter": info.numiter, "converged": info.converged, "ms": 1000 * t,
                             "value": info.numops / t, "unit": "it/s", "sigma": [float(v) for v in S[:6]],
                             "rel_residuals(Av-su, A'u-sv)": res}
                err = c4_truth_err(S[:6], m, nn)
                if err is not None:
                    rec[name]["max_rel_err_sigma_vs_float64_truth"] = err
                    rec[name]["ok"] = bool(err <= 3e-5)          # the Float32 bar of DESIGN §1
                del Lv, Rv, info
            out["c4"] = rec
            ctx.close()
        except Exception as e:      # the headline line must still be printed: record the failure instead
            out["c4"] = config_failed(e, ctx)

    if "c5" in want:
        ctx = None
        try:
            nx, ny, nz, kd = 625, 500, 256, 30
            ctx, n = make_ctx(nz, nx * ny, kd + 14)
            op = kk.B200CSR.stencil(ctx, nx, ny, nz, (6.0, -1, -1, -1, -1, -1, -1))
            x0 = ctx.splitmix(SEED)
            alg = kk.Lanczos(orth=kk.cgs2, krylovdim=kd, maxiter=3, tol=0.0, verbosity=0)
            (vals, vecs, info), t = timed(ctx, lambda: kk.eigsolve(op, x0, 4, "SR", alg))
            del vecs
            lam_min = 6.0 - 2.0 * (np.cos(np.pi / (nx + 1)) + np.cos(np.pi / (ny + 1)) + np.cos(np.pi / (nz + 1)))
            rec = {"workload": f"eigsolve(Lanczos, :SR, 4) on the {n}x{n} 7-point Laplacian ({nx}x{ny}x{nz}), Float64, "
                               f"krylovdim={kd}, orth=cgs2, 3 restart cycles, rows sharded by z-planes over {world} GPU(s)",
                   "numops": info.numops, "ms": 1000 * t, "value": info.numops / t, "unit": "it/s",
                   "ritz": [float(v) for v in vals[:4]], "closed_form_lambda_min": float(lam_min),
                   "ritz_above_lambda_min": bool(vals[0] >= lam_min * (1 - 1e-12))}
            g = gold.get("c5", {}).get("after_cycles", {}).get("3")
            if g:
                ref = np.array(g["ritz"])
                rel = float(np.max(np.abs(np.array(vals[:4]) - ref) / np.abs(ref)))
                rec["parity"] = {"against": "tests/golden/fullsize.json:c5:after_cycles[3] (oracle at full size)",
                                 "max_rel_diff_ritz": rel, "numops_oracle": g["numops"],
                                 "ok": bool(rel <= 1e-10 and info.numops == g["numops"])}
                if not rec["parity"]["ok"]:
                    raise AssertionError(f"config 5: parity with the oracle lost: {rec}")
            out["c5"] = rec
            ctx.close()
        except Exception as e:      # the headline line must still be printed: record the failure instead
            out["c5"] = config_failed(e, ctx)

    if "c4o" in want and world == 1 and os.environ.get("B2K_BENCH_CHILD") != "1":
        # the one-pass kernel has not run on a B200 yet: its record is produced by a CHILD process (this script with
        # --extra c4o and B2K_BENCH_CHILD=1), so that nothing it does — a crash, a hang, a poisoned CUDA context — can
        # take the headline line of this process with it
        try:
            env = dict(os.environ, B2K_BENCH_CHILD="1")
            cmd = [sys.executable, os.path.abspath(__file__), "--extra", "c4o", "--c4-rows", str(a.c4_rows)]
            res = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
            lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
            if res.returncode == 0 and lines:
                out["c4_onepass"] = json.loads(lines[-1])
            else:
                out["c4_onepass"] = {"ok": False, "error": f"child exited with {res.returncode}: " + res.stderr[-500:]}
        except Exception as e:
            out["c4_onepass"] = {"ok": False, "error": f"{type(e).__name__}: {e}"[:600]}
    elif "c4o" in want and world == 1:
        # config 4 in the flagged ONE-PASS mode of the GKL step (SURVEY §8f-4, DESIGN §6): z = A'(A v) comes out of the
        # pass that forms A v (b2k_op_apply_normal_gram) and A'u_{k+1} is recovered from it, guarded by an error
        # estimate that falls back to a direct A'u.  Each orthogonalizer is run in the reference's two-pass form and in
        # the one-pass form in the same process: singular values side by side, passes over A counted, the SVD
        # residual identities evaluated on the device, the fused kernel's own event-timed bandwidth.
        ctx = None
        try:
            m, nn, kd = a.c4_rows, 512, 30
            ctx = kk.B200Context(m, kd + 24, dtype=np.float32, device=local_rank)
            sv = ctx.add_space(nn, 2 * kd + 40, sharded=False)
            op = kk.B200Dense.splitmix(ctx, m, nn, SEED, sv)
            u0 = ctx.splitmix(SEED + 1)
            pk, _ = peak_hbm()
            rec = {"workload": f"svdsolve(GKL, krylovdim={kd}, tol=1e-5) on the dense {m}x{nn} Float32 matrix, 6 triplets "
                               ":LR; reference two-pass step vs the flagged one-pass step (GKL(onepass=True))",
                   "note": "numops counts both products of a step in both modes (as the reference does); passes = what was "
                           "streamed from HBM: 2 per step in the reference's form, 1 per step in the one-pass form unless "
                           "the error estimate of the recycled A'u forces a direct product"}
            # 1) the fused kernel alone, both variants: 12 event-timed launches each (profile class 8); each variant's y
            #    and z against the library's two separate products (same arithmetic, different summation order).  The
            #    faster variant that passed its check is the one the solver legs below use.
            x = ctx.splitmix(SEED + 2, sv)
            y2 = kk.apply_normal(op, x)
            z2 = kk.apply_adjoint(op, y2)
            ref = (y2.to_host().astype(np.float64), z2.to_host().astype(np.float64))
            del y2, z2
            names = {0: "A_32row_tiles_3cta_per_sm", 1: "B_64row_tiles_register_pipelined"}
            best = None
            for vid in (0, 1):
                if lib.b2k_debug_set_onepass_variant(vid) != 0:
                    continue
                try:
                    lib.b2k_prof_reset(ctx.h)
                    lib.b2k_prof_enable(ctx.h, 1)
                    for _ in range(12):
                        y, z = kk.apply_normal_gram(op, x)
                        del y, z
                    c, ms, b = C.c_int64(), C.c_double(), C.c_double()
                    lib.b2k_prof_read(ctx.h, 8, C.byref(c), C.byref(ms), C.byref(b))
                    lib.b2k_prof_enable(ctx.h, 0)
                    y, z = kk.apply_normal_gram(op, x)
                    yh, zh = y.to_host().astype(np.float64), z.to_host().astype(np.float64)
                    del y, z
                    k = {"launches": c.value}
                    if c.value:
                        k.update({"avg_ms": ms.value / c.value, "GBs": b.value / ms.value / 1e6,
                                  "frac_of_hbm_peak": b.value / ms.value / 1e6 / pk,
                                  "algorithmic_bytes": "4 (m n + m + n) per launch: A read ONCE for A v and A'(A v)"})
                    k["max_rel_diff_y_vs_separate_products"] = float(np.abs(yh - ref[0]).max() / np.abs(ref[0]).max())
                    k["max_rel_diff_z_vs_separate_products"] = float(np.abs(zh - ref[1]).max() / np.abs(ref[1]).max())
                    k["ok"] = bool(k["max_rel_diff_y_vs_separate_products"] < 1e-4 and k["max_rel_diff_z_vs_separate_products"] < 1e-4)
                    rec["kernel:" + names[vid]] = k
                    if k["ok"] and (best is None or k.get("avg_ms", 1e30) < best[1]):
                        best = (vid, k.get("avg_ms", 1e30))
                except Exception as e:
                    rec["kernel:" + names[vid]] = {"ok": False, "error": f"{type(e).__name__}: {e}"[:300]}
                finally:
                    lib.b2k_debug_set_onepass_variant(0)
            del x
            use = best[0] if best is not None else 0
            rec["kernel_variant_used_by_the_solver"] = names[use] + ("" if best is not None else " (no variant passed its check)")
            # 2) the solver, two-pass reference step against the one-pass step, per orthogonalizer
            lib.b2k_debug_set_onepass_variant(use)
            for oname, orth in (("mgs2", kk.mgs2), ("cgsr_eta0.75", kk.ClassicalGramSchmidtIR(eta=0.75))):
                sig = {}
                for mode, onepass in (("two_pass_reference", False), ("one_pass_flagged", True)):
                    alg = kk.GKL(orth=orth, krylovdim=kd, maxiter=100, tol=1e-5, verbosity=0, onepass=onepass)
                    lib.b2k_prof_reset(ctx.h)
                    (S, Lv, Rv, info), t = timed(ctx, lambda: kk.svdsolve(op, u0, 6, "LR", alg))
                    res = []
                    for i in range(3):                                  # A v = s u + r, A' u = s v on the device
                        w = kk.apply_normal(op, Rv[i])
                        w.add_(Lv[i], -float(S[i]))
                        z = kk.apply_adjoint(op, Lv[i])
                        z.add_(Rv[i], -float(S[i]))
                        res.append([float(w.norm() / S[i]), float(z.norm() / S[i])])
                        del w, z
                    r = {"numops": info.numops, "numiter": info.numiter, "converged": info.converged,
                         "passes_over_A": int(info.passes), "ms": 1000 * t, "value": info.numops / t, "unit": "it/s",
                         "sigma": [float(v) for v in S[:6]], "rel_residuals(Av-su, A'u-sv)": res}
                    sig[mode] = np.array(S[:6], dtype=np.float64)
                    err = c4_truth_err(S[:6], m, nn)
                    if err is not None:
                        r["max_rel_err_sigma_vs_float64_truth"] = err
                    del Lv, Rv, info
                    if onepass:
                        r["max_rel_diff_sigma_vs_two_pass"] = float(np.max(np.abs(sig[mode] - sig["two_pass_reference"])
                                                                           / sig["two_pass_reference"]))
                        r["ok"] = bool(r["max_rel_diff_sigma_vs_two_pass"] <= 3e-5 and r["converged"] >= 6 and
                                       r.get("max_rel_err_sigma_vs_float64_truth", 0.0) <= 3e-5)
                    rec[f"{oname}:{mode}"] = r
            lib.b2k_debug_set_onepass_variant(0)
            out["c4_onepass"] = rec
            ctx.close()
        except Exception as e:      # the headline line must still be printed: record the failure instead
            out["c4_onepass"] = config_failed(e, ctx)

    return out


def main():
    # the tree this runs from may be read-only and stays as the build left it: the modules imported from it below
    # write no bytecode caches there (nor in the child process of the c4o leg, which runs main() too)
    sys.dont_write_bytecode = True
    a = parse()
    if os.environ.get("B2K_BENCH_CHILD") == "1":
        # child of other_configs' c4o leg: that one record, as one JSON line, nothing else
        import krylovkit_jl_b200 as kk
        rec = other_configs(kk, a, 0, 1, int(os.environ.get("LOCAL_RANK", "0")), None).get("c4_onepass")
        print(json.dumps(json_safe(rec), allow_nan=False, default=str), flush=True)
        return
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
