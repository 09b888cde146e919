#!/usr/bin/env python
"""Time the Green's function stages on the bench's C2 HCI space (spaces.hci_space on ChemSystem(FCIDUMP), plain
determinants, ~10^7 by default), for the two highest occupied and the two lowest empty orbitals of each spin:
  ladder       SparseHamiltonian.ladder of the two occupied orbitals (removal) and of the two empty ones (addition), and the
               sizes of the N-1 / N+1 lists;
  build        the H build of each N-1 / N+1 list on its own handle (the N-electron matrix is freed first);
  lanczos      lanczos_tridiagonal from the images, per step, split into H.v and orthogonalisation (SQMC_DAV_PROFILE phase
               timer, synchronised), next to the model 12 nnz_full bytes per pass over H plus 20 n per vector (one pass
               serves a pair) and 2 (j + 1) 8 n bytes of reorthogonalisation at step j = 0, 1, ...
Then the full scripts/greens.py run on the shipped C2 input.  Times are host wall clock around calls that end in a device
synchronisation.  The card name and power limit are read in the same run.  Appends JSON lines to --out."""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                            timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the number is reported as unknown rather than guessed
        pl = "unknown (%s)" % e
    return name, pl


def lanczos_profiled(HX, V, max_steps):
    """lanczos_tridiagonal with the library's phase timer on; its stderr line is read back through a temporary file"""
    os.environ["SQMC_DAV_PROFILE"] = "1"
    with tempfile.TemporaryFile(mode="w+") as f:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            t0 = time.perf_counter()
            r = HX.lanczos_tridiagonal(V, max_steps, 1e-12)
            t = time.perf_counter() - t0
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            os.environ.pop("SQMC_DAV_PROFILE")
        f.seek(0)
        text = f.read()
    m = re.search(r"H\.v ([\d.]+) ms \| orthogonalisation ([\d.]+) ms", text)
    return r, t, (float(m.group(1)), float(m.group(2))) if m else (None, None)


def main():
    import sqmc_b200 as sq
    from sqmc_b200 import greens, spaces
    from sqmc_b200._lib import SqmcError
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-dets", type=int, default=10_000_000)
    ap.add_argument("--max-steps", type=int, default=100)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_greens.jsonl"))
    ap.add_argument("--skip-script", action="store_true")
    args = ap.parse_args()
    name, power = gpu_info()
    fcidump = os.path.join(ROOT, "data", "C2_v2z_curve", "r1.24253", "FCIDUMP")
    chem = sq.ChemSystem(fcidump)
    H = sq.SparseHamiltonian(chem)
    t0 = time.perf_counter()
    up, dn, wts, e = spaces.hci_space(H, chem, args.n_dets)
    t_space = time.perf_counter() - t0
    w = np.ascontiguousarray(wts[:, 0]) / np.linalg.norm(wts[:, 0])
    H.close()   # the N-electron matrix is not needed any more; ladder needs no matrix
    H = sq.SparseHamiltonian(chem)
    base = dict(gpu=name, power_limit_and_max_sm_clock=power, n=len(up), hci_space_s=t_space)
    rows = []
    for spin in (0, 1):
        nocc = chem.ndn if spin else chem.nup
        for create, orbs in ((False, [nocc - 2, nocc - 1]), (True, [nocc, nocc + 1])):
            H.ladder(up, dn, w, orbs, spin, create)   # warm-up
            t0 = time.perf_counter()
            u2, d2, phi = H.ladder(up, dn, w, orbs, spin, create)
            t_lad = time.perf_counter() - t0
            row = dict(base, stage="sector", spin="ab"[spin], create=create, orbitals_library=orbs, ladder_ms=t_lad * 1e3, n_sector=len(u2))
            sx, flipped = greens.electron_space(chem, spin, create)
            if flipped:   # chem handles hold N_alpha >= N_beta: the spin-flipped space has the same H
                u2, d2 = d2, u2
            HX = sq.SparseHamiltonian(sx)
            try:
                t0 = time.perf_counter()
                nnz = HX.generate_sparse_ham_upper_triangular(u2, d2)
                row["build_ms"] = (time.perf_counter() - t0) * 1e3
                info = HX.nnz()
                row.update(nnz_upper=nnz, nnz_full=info["nnz_full"])
                r, t, (hv_ms, orth_ms) = lanczos_profiled(HX, phi, args.max_steps)
                steps = [int(s) for s in r["steps"]]
                nstep = max(steps)   # the two runs share one two-vector H.v per step
                n2 = len(u2)
                row.update(lanczos_ms=t * 1e3, steps=steps, hv_ms_per_step=hv_ms / nstep, orth_ms_per_step=orth_ms / nstep,
                           model_hv_bytes_per_pair_step=12 * info["nnz_full"] + 2 * 20 * n2,
                           model_orth_bytes_total=int(sum(8 * n2 * j * (j + 1) for j in steps)))   # sum over j < steps of 2 (j + 1) 8 n
                row["hv_GBps_model"] = row["model_hv_bytes_per_pair_step"] / (row["hv_ms_per_step"] * 1e-3) / 1e9
                row["orth_GBps_model"] = row["model_orth_bytes_total"] / (orth_ms * 1e-3) / 1e9
            except SqmcError as ex:
                row["error"] = str(ex)
            finally:
                HX.close()
            print(json.dumps(row), flush=True)
            rows.append(row)
    if not args.skip_script:
        with tempfile.TemporaryDirectory() as d:
            t0 = time.perf_counter()
            # run from the repository root with a relative input, so the recorded "input" does not depend on the checkout
            p = subprocess.run([sys.executable, os.path.join("scripts", "greens.py"), os.path.join("data", "C2_v2z_curve", "r1.24253", "i_1sigma_g"),
                                "--spin", "a", "--out", d], capture_output=True, text=True, cwd=ROOT)
            t = time.perf_counter() - t0
            row = dict(gpu=name, power_limit_and_max_sm_clock=power, stage="scripts/greens.py shipped C2 input", wall_s=t, returncode=p.returncode,
                       result=json.loads(p.stdout.strip().splitlines()[-1]) if p.returncode == 0 else p.stderr[-2000:])
            print(json.dumps(row), flush=True)
            rows.append(row)
    with open(args.out, "a") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
