#!/usr/bin/env python
"""Measure the orbital gradient and Hessian (sqmc_b200_orbital_derivatives) and the orbital optimiser, in one process:
  1. orbital_derivatives against two_rdm on the bench's C2 HCI space (26 orbitals, ~10^7 plain determinants grown by
     spaces.hci_space, its ground-state vector): median and range over --repeats, repeats must be bit-identical;
  2. a synthetic 64-orbital C1 FCIDUMP (random 8-fold symmetric integrals written with formats.write_fcidump) with --n-synth
     random determinants: the call, its phase split (SQMC_ORBD_PROFILE=1, read back from stderr), the host path it replaces
     (two_rdm download + the numpy reference of tests/orbopt_reference.py) and the FP64 rate of the Y contraction (its FMA
     count 2 norb^6 over the longest orb_gemm_kernel per call, from torch.profiler in a separate profiled call);
  3. scripts/orbopt.py on the shipped C2 input in both modes (a subprocess each; its JSON line).
Times are host wall clock around calls that end in a device synchronisation, after a warm-up.  Appends JSON lines to --out."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from rdm_gpu import gpu_info  # noqa: E402


def timed(f, repeats, same):
    out, ts = None, []
    for _ in range(repeats):
        t0 = time.perf_counter()
        r = f()
        ts.append(time.perf_counter() - t0)
        if out is None:
            out = r
        elif not same(out, r):
            raise AssertionError("repeats differ")
    ts = np.array(ts) * 1e3
    return out, dict(median_ms=float(np.median(ts)), min_ms=float(ts.min()), max_ms=float(ts.max()), repeats=repeats)


def same_derivatives(a, b):
    return np.array_equal(a["fock"], b["fock"]) and np.array_equal(a["hessian"], b["hessian"]) and a["energy"] == b["energy"]


def with_stderr_captured(f):
    """f() with file descriptor 2 redirected to a temporary file -> (result, captured text)"""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            r = f()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        tmp.seek(0)
        return r, tmp.read()


def synthetic_fcidump(path, norb, nelec, seed):
    from sqmc_b200 import formats
    rng = np.random.default_rng(seed)
    g = 0.01 * rng.standard_normal((norb,) * 4)
    g = g + g.transpose(1, 0, 2, 3)
    g = g + g.transpose(0, 1, 3, 2)
    g = g + g.transpose(2, 3, 0, 1)
    h = 0.01 * rng.standard_normal((norb, norb))
    h = h + h.T + np.diag(np.linspace(-2.0, 2.0, norb))
    formats.write_fcidump(path, h, g, 1.0, nelec, orbsym=[1] * norb)


def random_list(norb, nup, ndn, n, seed):
    rng = np.random.default_rng(seed)
    seen = set()
    while len(seen) < n:
        u = sum(1 << int(k) for k in rng.choice(norb, nup, replace=False))
        d = sum(1 << int(k) for k in rng.choice(norb, ndn, replace=False))
        seen.add((u, d))
    up, dn = zip(*sorted(seen))
    return list(up), list(dn)


def main():
    import sqmc_b200 as sq
    from sqmc_b200 import rdm, spaces
    from orbopt_reference import densities, orbital_derivatives_reference
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-dets", type=int, default=10_000_000)
    ap.add_argument("--n-synth", type=int, default=100_000)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--skip-scripts", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_orbopt.jsonl"))
    args = ap.parse_args()
    name, power = gpu_info()
    rows = []

    def emit(r):
        rows.append(r)
        print(json.dumps(r), flush=True)

    # 1. bench space
    chem = sq.ChemSystem(os.path.join(ROOT, "data", "C2_v2z_curve", "r1.24253", "FCIDUMP"))
    H = sq.SparseHamiltonian(chem)
    up, dn, wts, e = spaces.hci_space(H, chem, args.n_dets)
    w1 = np.ascontiguousarray(wts[:, 0])
    base = dict(gpu=name, power_limit_and_max_sm_clock=power, n_dets=len(up), norb=chem.norb)
    H.orbital_derivatives(up, dn, w1)
    od, t_od = timed(lambda: H.orbital_derivatives(up, dn, w1), args.repeats, same_derivatives)
    H.two_rdm(up, dn, w1)
    _, t_2 = timed(lambda: H.two_rdm(up, dn, w1), args.repeats, np.array_equal)
    emit(dict(base, what="orbital_derivatives (C2 bench space, ground state)", **t_od, energy=od["energy"], e_var=e,
              abs_energy_minus_e_var=abs(od["energy"] - e), max_abs_gradient=float(np.max(np.abs(od["gradient"]))), repeats_bit_identical=True))
    emit(dict(base, what="two_rdm (same list and vector)", **t_2, repeats_bit_identical=True))
    del H, up, dn, wts, w1

    # 2. synthetic 64-orbital C1 system
    norb, nup, ndn = 64, 5, 5
    with tempfile.TemporaryDirectory() as tmp:
        fd = os.path.join(tmp, "FCIDUMP")
        synthetic_fcidump(fd, norb, nup + ndn, 7)
        sysm = sq.ChemSystem(fd)
    Hs = sq.SparseHamiltonian(sysm)
    su, sd = random_list(norb, nup, ndn, args.n_synth, 8)
    su, sd = sq.dets_to_u64(su), sq.dets_to_u64(sd)
    ws = spaces.splitmix_vector(len(su))
    Hs.orbital_derivatives(su, sd, ws)
    a, t_call = timed(lambda: Hs.orbital_derivatives(su, sd, ws), args.repeats, same_derivatives)
    os.environ["SQMC_ORBD_PROFILE"] = "1"
    _, marks = with_stderr_captured(lambda: Hs.orbital_derivatives(su, sd, ws))
    del os.environ["SQMC_ORBD_PROFILE"]
    phases = {}
    for ln in marks.splitlines():
        if ln.startswith("[sqmc orbital_derivatives]"):
            body = ln[len("[sqmc orbital_derivatives]"):].split(" ms")[0].rsplit(None, 1)
            phases[body[0].strip()] = float(body[1])
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        Hs.orbital_derivatives(su, sd, ws)
        torch.cuda.synchronize()
    gemm_us = sorted(ev.time_range.elapsed_us() for ev in prof.events() if "orb_gemm_kernel" in ev.name)
    y_ms = gemm_us[-1] / 1e3 if gemm_us else float("nan")
    fma = 2.0 * norb ** 6
    sbase = dict(gpu=name, power_limit_and_max_sm_clock=power, n_dets=len(su), norb=norb, nup=nup, ndn=ndn, integrals="random 8-fold symmetric, C1")
    emit(dict(sbase, what="orbital_derivatives (synthetic 64 orbitals)", **t_call, repeats_bit_identical=True,
              phase_split_ms_synchronising=phases))
    emit(dict(sbase, what="Y contraction kernel (orb_gemm_kernel, torch.profiler)", kernel_ms=y_ms, fma=fma,
              fp64_tflops=2.0 * fma / (y_ms * 1e-3) / 1e12, gemm_kernels_us=gemm_us))
    t0 = time.perf_counter()
    g1 = Hs.one_rdm(su, sd, ws)
    g2 = Hs.two_rdm(su, sd, ws)
    t_dl = time.perf_counter() - t0
    t0 = time.perf_counter()
    D, d = densities(g1[None], g2[None], [float(ws @ ws)], [1.0])
    h, g, ec = rdm.integrals_library_order(sysm)
    ref = orbital_derivatives_reference(h, g, D, d)
    t_np = time.perf_counter() - t0
    err = float(np.max(np.abs(ref["hessian"] - a["hessian"])) / np.max(np.abs(ref["hessian"])))
    emit(dict(sbase, what="host path: one_rdm + two_rdm download, then the numpy reference", download_ms=t_dl * 1e3, numpy_ms=t_np * 1e3,
              total_ms=(t_dl + t_np) * 1e3, cpu_threads=os.cpu_count(), max_rel_hessian_difference=err))
    del Hs, g1, g2, D, d, g, ref

    # 3. the optimiser on the shipped input
    if not args.skip_scripts:
        inp = os.path.join(ROOT, "data", "C2_v2z_curve", "r1.24253", "i_1sigma_g")
        for mode in ([], ["--fixed-list"]):
            with tempfile.TemporaryDirectory() as tmp:
                p = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "orbopt.py"), inp, "--out", tmp] + mode,
                                   capture_output=True, text=True, check=True)
                emit(dict(gpu=name, power_limit_and_max_sm_clock=power, what="scripts/orbopt.py i_1sigma_g " + " ".join(mode),
                          **json.loads(p.stdout.strip().splitlines()[-1])))

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
