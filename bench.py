#!/usr/bin/env python
"""bench.py -- drawdown points/sec of the Laplace-Hankel hot path on B200.

Workload (BASELINE.json configs[4], SURVEY.md section 8(d) "C5a"): a synthetic dense
(r,z,t) contour grid with the Malama partial-penetration model (model 5) and the
numerics of malama-partpen-input.dat: nr=1024 r=linspace(1,500), nz=128 z=linspace(0,b),
nt=8 t=logspace(0,7,8)  =>  2^20 points per GPU.  One "step" = one pass of the whole hot
path (driver.f90:100-231 of the reference) over that grid.  Multi-GPU: every rank owns
its own 2^20-point grid (weak scaling; rank k shifts the 8 times by 10^(k/8) so the
work is distinct), no data-path collective, final gather of the results to rank 0.

  python bench.py --gpus N --steps K --warmup W            # our CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # CPU oracle port on host cores

`value`  : device-resident inputs, CUDA-event time of the kernel launches only.
`e2e`    : the same metric through the C-ABI call unc_eval_grid_ex with HOST (pinned)
           buffers: H2D of inputs + kernel + D2H of results inside the timed region.
`roofline`: FP64 CUDA-core bound (no tensor cores, HBM traffic ~16 B/point).  `achieved` =
           EXECUTED FP64 flops (2*DFMA + DMUL + DADD per launch, counted by the committed ncu
           capture profiles/r02_ncu_grid8_summary.json of this very build and workload -- the
           capture is refused, frac = null, when the SASS hash of the library or the grid
           differs) / the launch time measured live in this run; `peak` = DFMA-chain
           microbenchmark of this run (MEASURED_PEAKS.json has no FP64 entry).  The SURVEY 8(d)
           minimal-evaluation model is reported under `algorithmic`; it is a work model, not a
           fraction of the pipe (the kernel executes ~4x fewer flops than the model counts).
`strong` : (N > 1) ONE 2^20-point grid (rank 0's) split by time rows across the ranks.

  python bench.py ... --dump-outputs DIR   # also write s and ds of the last timed step as DIR/*.npy

The benchmark writes nothing into the tree: the CPU arm's native build goes to a temporary
directory and no bytecode is cached.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # no __pycache__ in the tree for the modules imported below


# ----------------------------------------------------------------------------- workload
def c5_deck():
    """Physical/numerical lines 2-14 of malama-partpen-input.dat (patched), SURVEY 8(d) C5."""
    return dict(model=5, Q=2.0189e-2, l=0.9548, d=4.428e-4, rw=2.54e-2, b=52.669, Kr=1.225e-3,
                kappa=0.5288, Ss=3.766e-6, Sy=0.2521, beta=2.0, M=26, alpha=1e-8, tol=1e-9,
                ts_k=7, ts_R=5, j0s=(2, 2), gl_nacc=12, gl_ord=50, rwobs=2.54e-2, sF=20.0,
                time_type=1, time_par=[0.0, 1.0])


def c5a_grid(rank=0, nr=1024, nz=128, nt=8, rmin=1.0, zfrac=1.0):
    d = c5_deck()
    r = np.linspace(rmin, 500.0, nr)
    z = np.linspace(0.0, d["b"] * zfrac, nz)
    t = 10.0 ** (np.linspace(0.0, 7.0, nt) + rank / 8.0)
    return d, t, r, z


def derive(d, t, r, z, tables):
    """driver_io.f90:531-567 non-dimensionalisation + set-up tables through `tables`
    (the product's own unc_j0_zeros/unc_split_index/unc_zlay, or the oracle's)."""
    Lc = d["b"]
    Tc = Lc ** 2 / (d["Kr"] / d["Ss"])
    sigma = d["Sy"] / (d["Ss"] * d["b"])
    p = dict(model=d["model"], M=d["M"], alpha=d["alpha"], tol=d["tol"], tee_mult=2.0,
             time_type=d["time_type"], time_par=d["time_par"], ts_k=d["ts_k"], ts_R=d["ts_R"],
             gl_nacc=d["gl_nacc"], gl_ord=d["gl_ord"], kappa=d["kappa"],
             alphaD=d["kappa"] / sigma, beta=d["beta"], moench_gamma=[],
             lD=d["l"] / Lc, dD=d["d"] / Lc, rDw=d["rw"] / Lc, l=d["l"], d=d["d"], Ss=d["Ss"],
             rDwobs=d["rwobs"] / Lc, sF=d["sF"])
    p["bD"] = p["lD"] - p["dD"]
    p["j0z"] = tables.j0_zeros(max(d["j0s"]) + d["gl_nacc"] + 1)
    tD, rD, zD = t / Tc, r / Lc, z / Lc
    sv = tables.split_index(tD, d["j0s"])
    lay = tables.zlay(zD, p["lD"], p["dD"])
    return p, tD, sv, rD, zD, lay


def flops_per_point(p, lay, nz_share):
    """SURVEY 8(d): F_point = N_a*np*(C_ap/z_share + C_apz) + np*(R^2*8 + nacc^2*45) + 2*(M^2*60+M*60)."""
    W = json.load(open(os.path.join(ROOT, "roofline_weights.json")))
    m = str(p["model"])
    C_ap = W["C_ap"][m] + (W["moench_per_alpha"] * (len(p["moench_gamma"]) - 1) if m == "3" else 0)
    capz = W["C_apz_by_layer"][m]
    C_apz = float(np.mean([capz[int(k) - 1] for k in lay]))
    Na = (2 ** p["ts_k"] - 1) + p["gl_nacc"] * (p["gl_ord"] - 2)
    npp = 2 * p["M"] + 1
    return (Na * npp * (C_ap / nz_share + C_apz) + npp * (p["ts_R"] ** 2 * 8 + p["gl_nacc"] ** 2 * 45)
            + 2 * (p["M"] ** 2 * 60 + p["M"] * 60))


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], False
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                   timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = []
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(r[3 + i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "samples": len(self.rows),
                "reasons": reasons}


# ----------------------------------------------------------------------------- arms
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_sample(p_dict, tD, sv, rD, zD, lay, ncols, nthreads=0, schedule="points"):
    """Oracle (CPU port) timed on a bounded sample of the grid: `ncols` (t,r) columns x all z,
    spread over four time levels (or all of them if fewer) and evenly over the radii.
    schedule "points": OpenMP over the (t,r) columns (the better CPU schedule);
    schedule "abscissae": the reference's own schedule -- columns in sequence, OpenMP over the
    quadrature abscissae inside each (driver.f90:129-133,195-199)."""
    from oracle import oracle
    prm = oracle.Params(p_dict)
    tsel = np.unique(np.linspace(0, len(tD) - 1, min(4, len(tD))).astype(int))
    per_t = max(1, ncols // len(tsel))
    idx = np.unique(np.linspace(0, len(rD) - 1, per_t).astype(int))
    t0 = time.perf_counter()
    s, ds, fl = oracle.eval_grid(prm, tD[tsel], sv[tsel], rD[idx], zD, lay, carry=(schedule == "abscissae"),
                                 nthreads=nthreads)
    dt = time.perf_counter() - t0
    n = len(tsel) * len(idx)
    return n * len(zD) / dt, dt, n


def cpu_build():
    """The CPU arm is timed on a build with the reference's release flags (-O3 -march=native
    -flto -fopenmp, /root/reference Makefile:32) made on this host; returns a description.
    A real gfortran build of the reference would be used instead if a Fortran compiler existed."""
    import shutil
    from oracle import oracle
    flags = oracle.use_native_build()
    fc = [c for c in ("gfortran", "flang", "nvfortran", "ifx") if shutil.which(c)]
    return {"flags": flags, "fortran_compiler": fc[0] if fc else None}


def sass_sha256(so=None):
    """Hash of the SASS of the library being timed (identifies the build an ncu capture was taken from).
    The dump's `identifier = <source path as passed to nvcc>` lines are left out: the same sources
    built under another directory are the same build."""
    import hashlib
    from unconfined_b200.build import _nvcc
    if so is None:
        import unconfined_b200.api as api
        so = api._SO
    try:
        cuobjdump = os.path.join(os.path.dirname(os.path.realpath(_nvcc())), "cuobjdump")  # the toolkit that built it
        out = subprocess.run([cuobjdump, "-sass", so], capture_output=True, timeout=120).stdout
        if not out:
            return None
        keep = [ln for ln in out.split(b"\n") if not ln.lstrip().startswith(b"identifier =")]
        return hashlib.sha256(b"\n".join(keep)).hexdigest()
    except Exception:  # noqa: BLE001
        return None


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port; no Fortran compiler exists
    in this image, so oracle/_ref cannot be built) on all host threads, rank 0 only."""
    if rank != 0:
        return
    from oracle import oracle
    d, t, r, z = c5a_grid(0)
    p, tD, sv, rD, zD, lay = derive(d, t, r, z, oracle)
    cores = host_cores()   # torchrun exports OMP_NUM_THREADS=1: ask for every host core explicitly
    build = cpu_build()
    ncols = 12 * cores   # ~10-15 s of wall time per step on the host cores
    cpu_sample(p, tD, sv, rD[:2], zD, lay, 2, cores)  # warm
    for _ in range(max(0, args.warmup - 1)):
        cpu_sample(p, tD, sv, rD, zD, lay, max(4, ncols // 4), cores)
    times, pts = [], 0
    for _ in range(args.steps):
        _, dt, n = cpu_sample(p, tD, sv, rD, zD, lay, ncols, cores)
        times.append(dt)
        pts = n * len(zD)
    ms = 1e3 * float(np.mean(times))
    val = pts / (ms * 1e-3)
    va, dta, na = cpu_sample(p, tD, sv, rD, zD, lay, max(4, ncols // 8), cores, schedule="abscissae")
    sample = (f"{pts // len(zD)} (t,r) columns (4 time levels) x {len(zD)} z = {pts} points of the C5a grid per step")
    line = {"impl": "reference", "metric": "drawdown points/sec (r,z,t)", "value": val,
            "unit": "points/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C5a Malama partial-penetration contour grid 1024r x 128z x 8t "
                                   "(2^20 points/GPU), M=26 k=7 R=5 nacc=12 ord=50", "sample": sample},
            "cpu_baseline": {"value": val, "unit": "points/s", "cores": cores, "kind": "port",
                             "sample": sample, "schedule": "points-parallel (OpenMP over (t,r) columns)",
                             "abscissa_parallel": {"value": va, "unit": "points/s",
                                                   "schedule": "the reference's: OpenMP over abscissae, driver.f90:129-133,195-199",
                                                   "sample": f"{na} columns x {len(zD)} z, {dta:.1f} s"},
                             **build},
            "e2e": {"value": val, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DUMP_BYTES = 60 * 2 ** 20      # data of all dumped arrays together (under 64 MB with the .npy headers)


def dump_outputs(out_dir, arrays, shape):
    """--dump-outputs: the float64 device arrays the timed call returned in its last step, as
    out_dir/<name>.npy with `shape` (nt, nr, nz).  A grid too large for DUMP_BYTES is written as
    a fixed sample instead: the same sorted flat indices (seed 0) of every array, 1-D."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = int(np.prod(shape))
    keep = DUMP_BYTES // (8 * len(arrays))
    idx = None
    if n > keep:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        idx = torch.from_numpy(idx).to(next(iter(arrays.values())).device)
    for name, a in arrays.items():
        out = a.index_select(0, idx) if idx is not None else a.view(shape)
        np.save(os.path.join(out_dir, name + ".npy"), out.cpu().numpy())


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import unconfined_b200 as ub

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    ub.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    d, t, r, z = c5a_grid(rank, args.nr, args.nz, args.nt, args.rmin, args.zfrac)
    p, tD, sv, rD, zD, lay = derive(d, t, r, z, ub)
    prm = ub.Params(p)
    nt, nr, nz = len(tD), len(rD), len(zD)
    npts = nt * nr * nz

    # device-resident inputs/outputs for `value`
    g = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dev, dtype=dt)  # noqa: E731
    d_tD, d_rD, d_zD = g(tD, torch.float64), g(rD, torch.float64), g(zD, torch.float64)
    d_sv, d_lay = g(sv, torch.int32), g(lay, torch.int32)
    d_s = torch.empty(npts, dtype=torch.float64, device=dev)
    d_ds = torch.empty_like(d_s)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # pinned host buffers for `e2e`
    def pin(a):
        tt = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return tt, tt.numpy()
    keep = [pin(a) for a in (tD, sv, rD, zD, lay)]
    h_tD, h_sv, h_rD, h_zD, h_lay = [k[1] for k in keep]
    hs_t = torch.empty(npts, dtype=torch.float64).pin_memory()
    hd_t = torch.empty(npts, dtype=torch.float64).pin_memory()
    h_s, h_ds = hs_t.numpy().reshape(nt, nr, nz), hd_t.numpy().reshape(nt, nr, nz)
    import ctypes as C
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))  # noqa: E731
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))  # noqa: E731
    gathered = [torch.empty(npts, dtype=torch.float64, device=dev) for _ in range(world)] \
        if (world > 1 and rank == 0) else None

    def step_device():
        ub.eval_grid_device(prm, d_tD, d_sv, d_rD, d_zD, d_lay, d_s, d_ds)

    def step_e2e():
        rc = ub.lib().unc_eval_grid_ex(C.byref(prm.s), nt, dp(h_tD), ip(h_sv), nr, dp(h_rD), nz,
                                       dp(h_zD), ip(h_lay), None, 1, dp(h_s), dp(h_ds), None)
        if rc != 0:
            raise RuntimeError(ub.last_error())
        if world > 1:  # final gather of the results to rank 0 (north_star); 8 MB per rank
            d_s.copy_(hs_t, non_blocking=True)
            dist.gather(d_s, gathered, dst=0)
            torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
    barrier()
    launches0 = ub.kernel_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    with ClockSampler(local_rank) as cs:
        barrier()
        for k in range(args.steps):
            flush.zero_()            # L2 flush between timed iterations (outside the event pair)
            ev[k][0].record()
            step_device()
            ev[k][1].record()
        barrier()
    launches = ub.kernel_launch_count() - launches0
    if args.dump_outputs and rank == 0:     # before the e2e leg, which reuses d_s for the gather
        dump_outputs(args.dump_outputs, {"s": d_s, "ds": d_ds}, (nt, nr, nz))
    step_ms = [a.elapsed_time(b) for a, b in ev]
    tot_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot_ms, op=dist.ReduceOp.MAX)
    tot_ms = float(tot_ms.item())
    clocks = cs.summary()

    # e2e through the C ABI with host buffers
    for _ in range(min(args.warmup, 3)):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())
    # sanity: device and host paths agree bit for bit on the same inputs
    same = bool(np.array_equal(d_s.cpu().numpy(), h_s.ravel(), equal_nan=True)) if world == 1 else None

    # strong scaling (N > 1): rank 0's grid, split by time rows across the ranks (device-resident,
    # CUDA events, max over ranks); the headline stays the weak number above
    strong = None
    if world > 1 and nt % world == 0:
        d0, t0_, r0, z0_ = c5a_grid(0, args.nr, args.nz, args.nt, args.rmin, args.zfrac)
        p0, tD0, sv0, rD0, zD0, lay0 = derive(d0, t0_, r0, z0_, ub)
        prm0 = ub.Params(p0)
        rows = nt // world
        sl = slice(rank * rows, (rank + 1) * rows)
        s_tD, s_sv, s_rD = g(tD0[sl], torch.float64), g(sv0[sl], torch.int32), g(rD0, torch.float64)
        s_out = torch.empty(rows * nr * nz, dtype=torch.float64, device=dev)
        s_dout = torch.empty_like(s_out)

        def step_strong():
            ub.eval_grid_device(prm0, s_tD, s_sv, s_rD, d_zD, d_lay, s_out, s_dout)
        for _ in range(2):
            step_strong()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a_, b_ in evs:
            flush.zero_()
            a_.record(); step_strong(); b_.record()
        barrier()
        st_ms = torch.tensor([sum(a_.elapsed_time(b_) for a_, b_ in evs) / args.steps], dtype=torch.float64, device=dev)
        dist.all_reduce(st_ms, op=dist.ReduceOp.MAX)
        strong = {"value": npts / (float(st_ms.item()) * 1e-3), "unit": "points/s", "ms_per_step": float(st_ms.item()),
                  "workload": f"ONE {nr}r x {nz}z x {nt}t grid (rank 0's), {rows} time row(s) per rank, no exchange"}

    if rank == 0:
        total_pts = npts * world
        ms_per_step = tot_ms / args.steps
        value = total_pts / (ms_per_step * 1e-3)
        F = flops_per_point(p, lay, nz)
        peak = ub.measure_fp64_peak()
        cores = 0
        cpu = None
        if world == 1 and not args.no_cpu:
            from oracle import oracle
            cores = host_cores()
            ncols = 12 * cores
            build = cpu_build()
            po, tDo, svo, rDo, zDo, layo = derive(d, t, r, z, oracle)
            cpu_sample(po, tDo, svo, rDo[:2], zDo, layo, 2, cores)
            v, dt, n = cpu_sample(po, tDo, svo, rDo, zDo, layo, ncols, cores)
            va, dta, na = cpu_sample(po, tDo, svo, rDo, zDo, layo, max(4, ncols // 8), cores, schedule="abscissae")
            cpu = {"value": v, "unit": "points/s", "cores": cores, "kind": "port",
                   "sample": f"{n} (t,r) columns (4 time levels) x {nz} z = {n * nz} points of the C5a grid, "
                             f"{dt:.1f} s of CPU work (C++ port of the reference's algorithm; no Fortran compiler "
                             "in the image)",
                   "schedule": "points-parallel (OpenMP over (t,r) columns)",
                   "abscissa_parallel": {"value": va, "unit": "points/s",
                                         "schedule": "the reference's: OpenMP over abscissae, driver.f90:129-133,195-199",
                                         "sample": f"{na} columns x {nz} z, {dta:.1f} s"},
                   **build}
        # Executed FP64 flops per launch come from the committed ncu capture of THIS build on THIS
        # workload; anything else (kernel changed since the capture, other grid) gives frac = null.
        ncu, why = None, None
        cap_path = os.path.join("profiles", "r02_ncu_grid8_summary.json")
        try:
            ncu = json.load(open(os.path.join(ROOT, cap_path)))
            sha = sass_sha256()
            if ncu.get("sass_sha256") != sha:
                why = f"{cap_path} was captured from another build (sass {str(ncu.get('sass_sha256'))[:12]} != {str(sha)[:12]})"
            elif int(ncu["points_per_launch"]) != npts:
                why = f"{cap_path} was captured on {ncu['points_per_launch']} points per launch, this run has {npts}"
        except Exception as e:  # noqa: BLE001
            why = f"no usable capture: {e}"
        ok = ncu is not None and why is None
        sec = ms_per_step * 1e-3
        alg_bytes = 16.0 * npts + 8.0 * (nt + nr + nz) + 4.0 * (nt + nz)
        roof = {"bound": "fp64",
                "achieved": (ncu["executed_fp64_flop"] / sec / 1e12) if ok else None,
                "peak": peak / 1e12, "unit": "TFLOP/s",
                "frac": (ncu["executed_fp64_flop"] / sec / peak) if ok else None,
                "traffic": (ncu["dram_bytes_read"] + ncu["dram_bytes_write"]) if ok else None,
                "traffic_ratio": ((ncu["dram_bytes_read"] + ncu["dram_bytes_write"]) / alg_bytes) if ok else None,
                "algorithmic_bytes": alg_bytes,
                "executed_flop_per_point": ncu["executed_fp64_flop_per_point"] if ok else None,
                "fp64_pipe_pct_ncu": ncu["fp64_pipe_pct_of_peak_active"] if ok else None,
                "capture": cap_path, "capture_rejected": why,
                "definition": "achieved = executed FP64 flops per launch (2*DFMA + DMUL + DADD, ncu) / launch time "
                              "measured in this run with CUDA events; frac = achieved / peak",
                "algorithmic": {"flops_per_point": F, "tflops": F * npts / sec / 1e12,
                                "note": "SURVEY 8(d) minimal-evaluation work model per point x points / time; a work "
                                        "rate for comparisons across implementations, NOT a fraction of the pipe"},
                "traffic_note": "DRAM bytes of the launch are L2-evicted thread-local memory (areas, q-d tables, spills); "
                                "algorithmic bytes are 16 B/point; the bound is the FP64 pipe, not HBM",
                "peak_source": "DFMA-chain microbenchmark measured in this run "
                               "(MEASURED_PEAKS.json has no FP64 entry); nominal 37.2"}
        line = {"metric": "drawdown points/sec (r,z,t)", "value": value, "unit": "points/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"C5a Malama partial-penetration (model 5) contour grid "
                                       f"{nr}r x {nz}z x {nt}t = {npts} points per GPU, M=26 k=7 R=5 "
                                       "j0s=2,2 nacc=12 ord=50 (703 abscissae x 53 p per point)",
                           "l2_flush": "256 MiB memset between timed steps",
                           "sharding": "one grid per rank, no data-path collective, gather to rank 0 in e2e"},
                "clocks": clocks,
                "e2e": {"value": total_pts * args.steps / e2e_s, "unit": "points/s",
                        "h2d_bytes_per_step": int(8 * (nt + nr + nz) + 4 * (nt + nz)),
                        "d2h_bytes_per_step": int(16 * npts), "device_equals_host_path": same},
                "gpu_launches": int(launches),
                "roofline": roof,
                "cpu_baseline": cpu}
        if strong:
            line["strong"] = strong
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nr", type=int, default=1024)
    ap.add_argument("--nz", type=int, default=128)
    ap.add_argument("--nt", type=int, default=8)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--zfrac", type=float, default=1.0, help="(experiments only) top of the z grid as a fraction of b")
    ap.add_argument("--rmin", type=float, default=1.0, help="(experiments only) smallest radius of the grid")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write s and ds of the last timed step as DIR/s.npy, DIR/ds.npy (float64, "
                         "(nt, nr, nz); rank 0's grid; a fixed seeded sample above 60 MiB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's outputs (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
