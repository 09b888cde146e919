#!/usr/bin/env python
"""bench.py -- sparse H.v throughput (nnz/s, achieved HBM GB/s) on B200, with the CPU baseline beside it.

Default workload (BASELINE.json configs[3]): C2 cc-pVDZ r=1.24253 (data/C2_v2z_curve), time_sym=f, an HCI run on the
GPU (heat-bath selection + H build + Davidson per iteration through this library) with eps_var lowered until the space
holds 10^7 determinants; then the matrix of the final space is rebuilt from scratch (timed) and K H.v products are timed
(the Davidson matvec, more_tools.f90:2188).  A "step" is one H.v over the whole matrix.  Under torchrun (N GPUs) rows
of H are sharded and every rank's block of the vector is stored into all GPUs over NVLink before each product (strong
scaling: the matrix is fixed).

  value : nnz_full / t  with x, y and H resident in HBM (CUDA events on the launching stream)
  e2e   : the same through the reference-facing call with HOST vectors, H2D + D2H inside the timed region:
          1 GPU : sqmc_b200_matvec (fast_sparse_matrix_multiply_upper_triangular, more_tools.f90:3622)
          N GPUs: sqmc_b200_matvec_local -- every rank passes / receives only the slice of the determinants it owns
                  (fast_sparse_matrix_multiply_local_band + MPI_REDUCE_SCATTER, do_walk.f90:2259-2260)
  roofline.achieved : algorithmic bytes (12*nnz_full + 20*n, SURVEY.md 8(d)) / event time
  parity : y = H x for the splitmix vector: 16 rows recomputed by the CPU oracle from brute-forced full rows, and
           (x.y, |y|^2) printed so that runs at different N can be compared; a mismatch exits non-zero.

--config hubbard | heg | sweep run BASELINE.json configs 2, 3 and 5 with the same timing code (one JSON line each).
--impl reference times the CPU restatement of the reference's own fast_sparse_matrix_multiply_upper_triangular
(oracle/, threads emulate the MPI rank decomposition of davidson_sparse_mpi2) on a bounded sample of the same workload.
--dump-outputs DIR writes y of the last timed step (caller row order, float64) as DIR/y.npy with the caller rows it holds
as DIR/y_rows.npy (a fixed seeded sample of at most 2^21 rows per run), so that two builds can be compared row for row.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True   # the tree may be read-only; nothing is written into it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
CURVE = os.path.join(ROOT, "data", "C2_v2z_curve")
FCIDUMP = os.path.join(CURVE, "r1.24253", "FCIDUMP")
METRIC = "sparse_Hv_nnz_per_s"
UNIT = "nnz/s"
GEOMETRIES = ("1.0", "1.1", "1.2", "1.24253", "1.3", "1.4", "1.6", "1.8", "2.0")


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [names[k] for k in range(4) if any(len(r) > 2 + k and r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
CPU_SAMPLE_SCHED = (1e-3, 3e-4, 1e-4)            # cpu_baseline leg of the default run: 171,060 determinants
CPU_REFERENCE_SCHED = (1e-3, 3e-4, 1e-4, 3e-5)   # --impl reference: 541,648 determinants (iteration 4 of the same run)


def fortran_toolchain():
    """BASELINE.md section 4 step 2: is there a Fortran compiler + MPI + LAPACK to build the reference itself?"""
    found = {k: shutil.which(k) for k in ("mpif90", "mpifort", "gfortran", "ifort", "nvfortran", "flang", "mpirun")}
    lapack = any(os.path.exists(os.path.join(d, "liblapack.so")) or os.path.exists(os.path.join(d, "liblapack.a"))
                 for d in ("/usr/lib/x86_64-linux-gnu", "/usr/lib64", "/usr/lib", "/usr/local/lib"))
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "sqmc")
    return {"compilers": {k: v for k, v in found.items() if v}, "lapack": lapack, "reference_binary": ref_bin if os.path.exists(ref_bin) else None}


def cpu_sample(space, sched, cpu_sample_dets, time_build=True):
    """The bounded CPU sample of the workload, built with the oracle only: the same HCI run stopped early (oracle
    perform_hci), or for --space lowest the cpu_sample_dets lowest-energy determinants."""
    import sqmc_b200 as sq
    from sqmc_b200 import spaces
    from oracle import oracle as O
    chem = sq.ChemSystem(FCIDUMP)
    S = O.System.chem(FCIDUMP, chem.norb, chem.nelec, chem.nup, chem.orbital_symmetries_fcidump)
    t0 = time.perf_counter()
    if space == "hci":
        r = S.hci(sched[-1], eps_var_sched=sched, max_iters=len(sched))
        up, dn = r["up"], r["dn"]
        desc = "the same HCI run stopped at eps_var=%.0e (oracle perform_hci, %d dets)" % (sched[-1], len(up))
    else:
        up, dn, _ = spaces.c2_lowest_energy_space(chem, cpu_sample_dets)
        desc = "the %d lowest-energy A_g dets" % len(up)
    t_space = time.perf_counter() - t0
    t0 = time.perf_counter()
    # time_build: a from-scratch build of the sample (the CPU build rate reported beside the GPU one); otherwise the matrix the
    # oracle's HCI run left behind is taken over (incremental call that finds nothing to add)
    cnt, idx, val = S.build_upper(up, dn, incremental=(not time_build and space == "hci"))
    t_build = time.perf_counter() - t0
    return cnt, idx, val, desc, t_space, t_build


def workload_name(n):
    return ("C2 cc-pVDZ r1.24253 (FCIDUMP), time_sym=f, %d determinants: HCI space (heat-bath selection + build + Davidson per "
            "iteration, eps_var lowered 1e-3 -> 5e-7); step = one H.v" % n)


def run_reference(args):
    """CPU arm: the oracle's restatement of fast_sparse_matrix_multiply_upper_triangular on a bounded sample, all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from sqmc_b200 import spaces
    from oracle import oracle as O
    tool = fortran_toolchain()
    cnt, idx, val, desc, t_space, t_build = cpu_sample(args.space, CPU_REFERENCE_SCHED, args.cpu_sample_dets, time_build=False)
    n = len(cnt)
    nnz_full = 2 * len(idx) - n
    cores = os.cpu_count() or 1
    x = spaces.splitmix_vector(n)
    for _ in range(args.warmup):
        O.matvec_upper_mt(cnt, idx, val, x, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y = O.matvec_upper_mt(cnt, idx, val, x, cores)
    t = (time.perf_counter() - t0) / args.steps
    dump_outputs(args, "", y)
    v = nnz_full / t
    sample = ("C2 cc-pVDZ r1.24253 time_sym=f, %s (nnz_full=%d); %d threads, rows dealt round-robin, private y + reduction; "
              "obtaining the sample (oracle HCI run incl. its H builds) took %.1f s on one core (untimed)" % (desc, nnz_full, cores, t_space + t_build))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.n_dets), "space": args.space, "n_dets": args.n_dets,
                       "sample_n_dets": n, "sample_nnz_full": nnz_full,
                       "note": "each step is one CPU H.v on the bounded sample described in cpu_baseline.sample"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "why_port": "the reference is Fortran 90 + MPI + LAPACK; probe of this host: %s" % json.dumps(tool)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


DUMP_ROWS = 1 << 21   # --dump-outputs: rows kept per run, shared by its workloads (y + row ids in float64: 33.6 MB in all)


def dump_outputs(args, tag, y):
    """--dump-outputs: y (caller row order) of the last timed step as DIR/<tag>y.npy, or a fixed seeded sample of its rows when
    it holds more than this workload's share of DUMP_ROWS; the caller rows kept go to DIR/<tag>y_rows.npy (float64, 0-based)"""
    if not args.dump_outputs:
        return
    n, m = len(y), DUMP_ROWS // args.dump_workloads
    rows = np.arange(n) if n <= m else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
    os.makedirs(args.dump_outputs, exist_ok=True)
    np.save(os.path.join(args.dump_outputs, tag + "y.npy"), np.ascontiguousarray(y[rows], dtype=np.float64))
    np.save(os.path.join(args.dump_outputs, tag + "y_rows.npy"), rows.astype(np.float64))


def cpu_baseline(args):
    """oracle (port of the reference algorithm) on a bounded sample, 1 core: ~10-30 s of CPU work."""
    from sqmc_b200 import spaces
    from oracle import oracle as O
    cnt, idx, val, desc, t_space, t_build = cpu_sample(args.space, CPU_SAMPLE_SCHED, args.cpu_sample_dets)
    n = len(cnt)
    nnz_full = 2 * len(idx) - n
    x = spaces.splitmix_vector(n)
    O.matvec_upper(cnt, idx, val, x)
    reps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < 5.0:
        O.matvec_upper(cnt, idx, val, x)
        reps += 1
    t = (time.perf_counter() - t0) / reps
    return {"value": nnz_full / t, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "oracle fast_sparse_matrix_multiply_upper_triangular on %s of the same C2 workload (nnz_full=%d), %d reps; "
                      "obtaining the sample's space took the oracle %.1f s, its from-scratch H build %.1f s" % (desc, nnz_full, reps, t_space, t_build),
            "build_nnz_upper_per_s": len(idx) / t_build}


# ----------------------------------------------------------------------------------------------- GPU arm
class Ctx:
    pass


def setup_dist():
    import torch
    import torch.distributed as dist
    from sqmc_b200 import _lib
    c = Ctx()
    c.rank = int(os.environ.get("RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this benchmark has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(c.local)
    uid = None
    if c.world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=c.rank, world_size=c.world, device_id=torch.device("cuda", c.local))
        obj = [_lib.get_unique_id() if c.rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        uid = obj[0]
    _lib.init(device=c.local, rank=c.rank, nranks=c.world, unique_id=uid)
    c.L = _lib.load()
    c.stream = torch.cuda.Stream()  # a real (non-default) stream: the library launches on the stream it is handed
    torch.cuda.set_stream(c.stream)
    return c


def max_over_ranks(c, v):
    import torch
    import torch.distributed as dist
    if c.world == 1:
        return v
    t = torch.tensor([v], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(c):
    import torch
    import torch.distributed as dist
    if c.world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def bench_owner(up, dn, world):
    """Ownership map for the distributed-slice e2e leg.  The reference hashes the determinant (djb_hash,
    mpi_routines.f90:354-379, restated in oracle/oracle.py for the parity tests); at 10^7 determinants the bench uses a
    vectorised 64-bit mix with the same purpose: a balanced pseudo-random deal of determinants to ranks."""
    z = up[:, 0] ^ ((dn[:, 0] << np.uint64(29)) | (dn[:, 0] >> np.uint64(35)))
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z % np.uint64(world)).astype(np.int32)


def time_hv(c, H, n, nloc, steps, warmup, x_host, projector=None):
    """device-resident H.v steps on x_host (internal row order): CUDA events on the launching stream, max over ranks
    -> (ms per step, per-step list, launches, y of the last step on the device)"""
    import ctypes as C
    import torch
    from sqmc_b200 import _lib
    x = torch.from_numpy(x_host).cuda()
    y = torch.zeros(max(nloc, 1), dtype=torch.float64, device="cuda")
    sptr = C.c_void_p(c.stream.cuda_stream)

    def step():
        _lib.check(c.L.sqmc_b200_matvec_dev(H._h, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), sptr))

    prof_range = os.environ.get("SQMC_BENCH_PROFILE_RANGE") == "1"   # ncu --profile-from-start off: only warm-up + timed steps
    if prof_range:
        torch.cuda.profiler.start()
    for _ in range(warmup):
        step()
    barrier(c)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    barrier(c)
    l0 = c.L.sqmc_b200_launch_count()
    ev[0].record(c.stream)
    for k in range(steps):
        step()
        ev[k + 1].record(c.stream)
    barrier(c)
    l1 = c.L.sqmc_b200_launch_count()
    if prof_range:
        torch.cuda.profiler.stop()
    per = [ev[k].elapsed_time(ev[k + 1]) for k in range(steps)]
    ms = max_over_ranks(c, ev[0].elapsed_time(ev[steps])) / steps
    return ms, per, int(l1 - l0), y


def time_e2e(c, H, n, up, dn, x_host, steps, projector=None):
    """host vectors through the reference-facing call; returns (seconds per step, h2d bytes, d2h bytes, full y on rank 0 or None, call name)"""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from sqmc_b200 import _lib
    L = c.L
    if c.world == 1:
        xh = torch.from_numpy(x_host.copy()).pin_memory()
        yh = torch.zeros(n, dtype=torch.float64).pin_memory()
        if projector:
            tau, e_trial = projector

            def step():
                _lib.check(L.sqmc_b200_projector(H._h, tau, e_trial, C.c_void_p(xh.data_ptr()), C.c_void_p(yh.data_ptr())))
            name = "sqmc_b200_projector (pinned host vectors)"
        else:
            def step():
                _lib.check(L.sqmc_b200_matvec(H._h, C.c_void_p(xh.data_ptr()), C.c_void_p(yh.data_ptr()), 1, n))
            name = "sqmc_b200_matvec (pinned host vectors)"
        nb = 8 * n
        owner = None
    else:
        owner = bench_owner(up, dn, c.world)
        mine = np.nonzero(owner == c.rank)[0]
        m = H.set_ownership(owner)
        assert m == len(mine)
        xh = torch.from_numpy(x_host[mine].copy()).pin_memory()
        yh = torch.zeros(max(m, 1), dtype=torch.float64).pin_memory()
        if projector:
            tau, e_trial = projector

            def step():
                _lib.check(L.sqmc_b200_projector_local(H._h, tau, e_trial, C.c_void_p(xh.data_ptr()), C.c_void_p(yh.data_ptr())))
            name = "sqmc_b200_projector_local (owned slices, pinned)"
        else:
            def step():
                _lib.check(L.sqmc_b200_matvec_local(H._h, C.c_void_p(xh.data_ptr()), C.c_void_p(yh.data_ptr()), 1, max(m, 1)))
            name = "sqmc_b200_matvec_local (owned slices, pinned)"
        nb = int(max_over_ranks(c, 8.0 * m))
    for _ in range(2):
        step()
    barrier(c)
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    barrier(c)
    t = max_over_ranks(c, (time.perf_counter() - t0) / steps)
    # the result of the last step, whole vector in caller order on rank 0 (for the parity block)
    y_full = None
    if c.world == 1:
        y_full = yh.numpy().copy()
    else:
        sizes = np.bincount(owner, minlength=c.world)
        mx = int(sizes.max())
        pad = torch.zeros(mx, dtype=torch.float64, device="cuda")
        pad[:len(mine)] = yh[:len(mine)].cuda()
        bufs = [torch.zeros(mx, dtype=torch.float64, device="cuda") for _ in range(c.world)]
        dist.all_gather(bufs, pad)
        if c.rank == 0:
            y_full = np.zeros(n)
            for r in range(c.world):
                y_full[owner == r] = bufs[r][:sizes[r]].cpu().numpy()
    return t, nb, nb, y_full, name


def parity_block(system_factory, up, dn, x_host, y_full, nrows=16, scale=1.0, shift=None):
    """rank 0: nrows rows of y recomputed by the CPU oracle from brute-forced full rows of H (oracle orc_row: every
    determinant of the list tested against the row's, element rule abs(H) > 1e-12) + order-independent sums of y."""
    n = len(up)
    S = system_factory()
    rows = sorted(set([0, n - 1] + [int(v) for v in np.linspace(0, n - 1, nrows)]))[:nrows]
    worst = 0.0
    ymax = float(np.max(np.abs(y_full)))
    t0 = time.perf_counter()
    for i in rows:
        cols, vals = S.row(up, dn, i, cap=1 << 20)
        ref = float(np.dot(vals * scale, x_host[cols - 1]))
        if shift is not None:
            ref += shift * x_host[i]
        worst = max(worst, abs(ref - y_full[i]) / ymax)
    return {"rows_checked": len(rows), "max_rel_err_vs_oracle_rows": worst, "tolerance": 1e-12, "ok": bool(worst <= 1e-12),
            "x_dot_y": float(np.dot(x_host, y_full)), "y_norm2": float(np.dot(y_full, y_full)), "oracle_seconds": time.perf_counter() - t0,
            "how": "y from the e2e call (host vectors); rows recomputed from oracle brute-force full rows; x_dot_y / y_norm2 must agree to 1e-12 relative across GPU counts"}


def emit(c, args, H, system_factory, up, dn, workload, config_extra, t_build, t_space, hci_log=None, projector=None, with_cpu=True,
         dump_tag=""):
    """time the resident matrix and print the JSON line (rank 0)"""
    import torch.distributed as dist
    from sqmc_b200 import spaces
    n = len(up)
    info = H.nnz()
    nnz_full, nnz_upper = info["nnz_full"], info["nnz_upper"]
    nloc, nnz_loc = H.local_rows()
    bt = H.build_times()
    nnz_max = max_over_ranks(c, float(nnz_loc))
    x_host = spaces.splitmix_vector(n)
    perm = H.perm()   # internal row p holds caller row perm[p]: the device leg gets the same x (caller order) as the e2e leg
    sampler = ClockSampler(c.local)
    if c.rank == 0:
        sampler.start()
    ms_step, per, launches, y = time_hv(c, H, n, nloc, args.steps, args.warmup, x_host[perm])
    clocks = sampler.stop() if c.rank == 0 else None
    if args.dump_outputs:   # one rank (main): y holds all n rows
        y_caller = np.empty(n)
        y_caller[perm] = y[:n].cpu().numpy()
        dump_outputs(args, dump_tag, y_caller)
    t_e2e, h2d, d2h, y_full, e2e_call = time_e2e(c, H, n, up, dn, x_host, args.steps, projector=projector)
    mode = H.exchange_mode()
    if c.rank != 0:
        return
    par = None
    if not args.no_parity:
        scale, shift = 1.0, None
        if projector:
            scale, shift = -projector[0], projector[0] * projector[1]   # stored matrix is -tau*H; deltaw = Hstored.w + e_trial*tau*w
        par = parity_block(system_factory, up, dn, x_host, y_full, scale=scale, shift=shift)
    peak, peak_src = measured_peak_gbs()
    # per-rank algorithmic bytes (the slowest rank bounds the step; rows are balanced by candidate count)
    alg_bytes = 12.0 * nnz_max + 20.0 * (n / c.world) if c.world > 1 else 12.0 * nnz_full + 20.0 * n
    achieved = alg_bytes / (ms_step * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "spmv_dram_bytes_per_launch.json")
    if os.path.exists(tp) and c.world == 1:  # only when the committed ncu capture is of this exact matrix
        try:
            tj = json.load(open(tp))
            if int(tj.get("nnz_full", -1)) == int(nnz_full):
                traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    cfg = {"workload": workload, "n_dets": n, "nnz_upper": nnz_upper, "nnz_full": nnz_full, "parallelism": "rows x%d" % c.world,
           "vector_exchange": mode, "l2": "inputs larger than L2 (matrix %.1f GB streamed per step)" % (12.0 * nnz_full / 1e9)}
    cfg.update(config_extra)
    line = {
        "metric": METRIC, "value": nnz_full / (ms_step * 1e-3), "unit": UNIT, "n_gpus": c.world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "peak_source": peak_src, "algorithmic_bytes_per_step": alg_bytes, "frac_of_nominal_8TBs": achieved / 8000.0},
        "e2e": {"value": nnz_full / t_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": t_e2e * 1e3,
                "call": e2e_call},
        "gpu_launches": launches,
        "clocks": clocks,
        "build": {"seconds_wall": t_build, "nnz_upper_per_s": nnz_upper / t_build, "phases_ms": bt, "alloc_stall_ms": LAST_BUILD_STALL_MS,
                  "space_seconds": t_space},
        "step_ms_min_max": [min(per), max(per)],
        "nnz_per_rank_max_over_mean": nnz_max / (nnz_full / c.world),
    }
    if par is not None:
        line["parity"] = par
    if hci_log:
        line["hci_iterations"] = hci_log
    if with_cpu and not args.no_cpu_baseline and c.world == 1:
        line["cpu_baseline"] = cpu_baseline(args)
    print(json.dumps(line), flush=True)
    if par is not None and not par["ok"]:
        raise SystemExit("bench.py: parity check failed: %s" % json.dumps(par))


LAST_BUILD_STALL_MS = 0.0


def timed_build(c, H, up, dn, **kw):
    """wall time of one build (max over ranks); the host time this rank spent blocked inside allocator / memory-mapping calls during it
    goes to LAST_BUILD_STALL_MS (printed as build.alloc_stall_ms: erratic on virtualised hosts, profiles/r02_alloc_trace.txt)"""
    global LAST_BUILD_STALL_MS
    from sqmc_b200 import _lib
    barrier(c)
    _lib.load().sqmc_b200_alloc_stall_ms(1)
    t0 = time.perf_counter()
    H.generate_sparse_ham_upper_triangular(up, dn, **kw)
    LAST_BUILD_STALL_MS = float(_lib.load().sqmc_b200_alloc_stall_ms(1))
    barrier(c)
    return max_over_ranks(c, time.perf_counter() - t0)


def run_c2(c, args):
    import sqmc_b200 as sq
    from sqmc_b200 import spaces
    from oracle import oracle as O
    t0 = time.perf_counter()
    chem = sq.ChemSystem(FCIDUMP)
    H = sq.SparseHamiltonian(chem, device=c.local)
    hci_log = []
    if args.space == "hci":
        up, dn, _, e_var = spaces.hci_space(H, chem, args.n_dets, log=hci_log)
        detail = "HCI space grown on the GPU (heat-bath selection + build + Davidson), eps_var lowered to %.0e, E_var = %.9f Ha" % (
            hci_log[-1]["eps_var"], e_var)
    else:
        up, dn, sector = spaces.c2_lowest_energy_space(chem, args.n_dets)
        detail = "%d lowest-diagonal-energy A_g determinants of %d" % (len(up), sector)
    t_space = time.perf_counter() - t0
    t_build = timed_build(c, H, up, dn)   # timed from-scratch build of the final space
    fac = lambda: O.System.chem(FCIDUMP, chem.norb, chem.nelec, chem.nup, chem.orbital_symmetries_fcidump)  # noqa: E731
    emit(c, args, H, fac, up, dn, workload_name(len(up)), {"space": args.space, "space_detail": detail}, t_build, t_space, hci_log=hci_log)
    if args.davidson:
        t0 = time.perf_counter()
        dv = H.davidson_sparse(n_states=1)
        if c.rank == 0:
            print(json.dumps({"davidson": {"seconds": time.perf_counter() - t0, "n_matvec": dv["n_matvec"], "energy": float(dv["evals"][0])}}))
    H.close()


def run_hubbard(c, args):
    """config 2: 2D Hubbard 4x4 half filling, k-space, momentum sector (0,0): deterministic-space projector matvec"""
    import sqmc_b200 as sq
    from sqmc_b200 import spaces
    from oracle import oracle as O
    hub = sq.HubbardKSystem(4, 4, 1.0, 4.0, 8, 8)
    t0 = time.perf_counter()
    nd = None if args.n_dets >= 10_000_000 else args.n_dets
    up, dn, total = spaces.hubbard_momentum_sector(hub, nd)
    t_space = time.perf_counter() - t0
    H = sq.SparseHamiltonian(hub, device=c.local)
    t_build = timed_build(c, H, up, dn)
    tau, e_trial = 0.01, -10.0
    H.scale_values(-tau)                      # the walk keeps -tau*H resident (semistoch.f90:657,880)
    fac = lambda: O.System.hubbardk(4, 4, 1.0, 4.0, 8, 8)  # noqa: E731
    wl = ("2D Hubbard 4x4 half filling (k-space, U/t=4), total-momentum (0,0) sector, %d of %d determinants; step = one deterministic "
          "projector H.v (do_walk.f90:2259-2290)" % (len(up), total))
    emit(c, args, H, fac, up, dn, wl, {"case": "hubbard", "tau": tau, "e_trial": e_trial}, t_build, t_space, projector=(tau, e_trial), with_cpu=False)
    H.close()


def run_heg(c, args):
    """config 3: HEG 14 electrons r_s = 0.5: H build + H.v on HCI spaces grown on the GPU at two basis sizes"""
    import sqmc_b200 as sq
    from sqmc_b200 import spaces
    from oracle import oracle as O
    for cutoff, eps_sched, target in ((2.0, (1e-3, 3e-4, 2e-4), 10**9), (2.5, (1e-3, 3e-4, 1e-4, 5e-5, 3e-5, 2e-5, 1e-5), args.heg_dets)):
        heg = sq.HegSystem(3, 0.5, 14, 7, cutoff)
        H = sq.SparseHamiltonian(heg, device=c.local)
        t0 = time.perf_counter()
        log = []
        up, dn, _, e = spaces.hci_space(H, heg, target, eps_schedule=eps_sched, log=log)
        t_space = time.perf_counter() - t0
        t_build = timed_build(c, H, up, dn)
        fac = lambda cutoff=cutoff: O.System.heg(3, 0.5, 14, 7, cutoff)  # noqa: E731
        wl = ("HEG 14 electrons r_s=0.5 cutoff %.1f (%d orbitals), %d determinants: HCI space grown on the GPU to eps_var=%.0e; "
              "step = one H.v" % (cutoff, heg.norb, len(up), log[-1]["eps_var"]))
        emit(c, args, H, fac, up, dn, wl, {"case": "heg", "cutoff": cutoff, "E_var": e}, t_build, t_space, hci_log=log, with_cpu=False,
             dump_tag="cutoff%.1f_" % cutoff)
        H.close()


def run_sweep(c, args):
    """config 5: C2 binding curve, 9 geometries: H build + H.v on the N lowest-diagonal-energy A_g determinants of each"""
    import sqmc_b200 as sq
    from sqmc_b200 import spaces
    from oracle import oracle as O
    for rr in (args.geometries.split(",") if args.geometries else GEOMETRIES):
        fd = os.path.join(CURVE, "r" + rr, "FCIDUMP")
        chem = sq.ChemSystem(fd)
        t0 = time.perf_counter()
        up, dn, sector = spaces.c2_lowest_energy_space(chem, args.sweep_dets)
        t_space = time.perf_counter() - t0
        H = sq.SparseHamiltonian(chem, device=c.local)
        t_build = timed_build(c, H, up, dn)
        fac = lambda fd=fd, chem=chem: O.System.chem(fd, chem.norb, chem.nelec, chem.nup, chem.orbital_symmetries_fcidump)  # noqa: E731
        wl = "C2 cc-pVDZ r%s (FCIDUMP), time_sym=f, the %d lowest-diagonal-energy A_g determinants of %d; step = one H.v" % (rr, len(up), sector)
        emit(c, args, H, fac, up, dn, wl, {"case": "sweep", "geometry": rr}, t_build, t_space, with_cpu=False, dump_tag="r%s_" % rr)
        H.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "hubbard", "heg", "sweep"],
                    help="c2 = BASELINE.json configs[3] (the headline metric); hubbard / heg / sweep = configs 2, 3, 5")
    ap.add_argument("--n-dets", type=int, default=int(os.environ.get("SQMC_BENCH_NDETS", 10_000_000)))
    ap.add_argument("--space", default=os.environ.get("SQMC_BENCH_SPACE", "hci"), choices=["hci", "lowest"],
                    help="hci (BASELINE.json configs[3] recipe): an HCI run on the GPU (selection + build + Davidson through the "
                         "library) with eps_var lowered until N determinants; lowest: the N lowest-diagonal-energy A_g "
                         "determinants (host generated, SURVEY.md S4 fallback)")
    ap.add_argument("--cpu-sample-dets", type=int, default=200_000)
    ap.add_argument("--sweep-dets", type=int, default=1_000_000)
    ap.add_argument("--heg-dets", type=int, default=1_000_000)
    ap.add_argument("--geometries", default="", help="--config sweep: comma-separated subset of " + ",".join(GEOMETRIES))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--davidson", action="store_true", help="also run a full device Davidson and print it on a second line")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write y of the last timed step (caller row order; a fixed seeded sample of rows above 2^21) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    args.dump_workloads = {"heg": 2, "sweep": len(args.geometries.split(",")) if args.geometries else len(GEOMETRIES)}.get(args.config, 1)
    if args.impl == "reference":
        return run_reference(args)
    c = setup_dist()
    if args.dump_outputs and c.world > 1:
        raise SystemExit("bench.py: --dump-outputs runs on one GPU (the device leg's y is sharded over ranks)")
    {"c2": run_c2, "hubbard": run_hubbard, "heg": run_heg, "sweep": run_sweep}[args.config](c, args)
    if c.world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
