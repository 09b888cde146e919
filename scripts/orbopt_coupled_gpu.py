#!/usr/bin/env python
"""Measure the sigma-vector (sqmc_b200_sigma), the orbital-gradient response (sqmc_b200_orbital_gradient_response) and the
one-step orbital optimiser, in one process:
  1. on the bench's C2 HCI space (26 orbitals, ~10^7 plain determinants grown by spaces.hci_space, its ground-state vector, H
     resident): sigma without and with kappa, orbital_gradient_response and two_rdm, median and range over --repeats (repeats
     must be bit-identical), and sigma without kappa against the resident H.v;
  2. the shipped C2 input (2 states, time_sym): optimize_orbitals in one-step and in two-step fixed-list mode, 10 macro
     iterations each (history, seconds per macro iteration), and the three calls of one micro-iteration (sigma with kappa,
     orbital_gradient_response, H.v) timed on the final list.
Times are host wall clock around calls that end in a device synchronisation, after a warm-up.  The card's name, power limit
and max SM clock are read in the same run.  Appends JSON lines to --out."""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from orbopt_gpu import timed  # noqa: E402
from rdm_gpu import gpu_info  # noqa: E402


def main():
    import sqmc_b200 as sq
    from sqmc_b200 import orbopt, spaces
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-dets", type=int, default=10_000_000)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--max-macro", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_orbopt_coupled.jsonl"))
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
    w1 = w1 / np.linalg.norm(w1)
    rng = np.random.default_rng(1)
    dw = rng.standard_normal(len(w1))
    dw -= (w1 @ dw) * w1
    sym = np.asarray(chem.orbital_symmetries)
    a = np.tril(rng.standard_normal((chem.norb, chem.norb)), -1) * (sym[:, None] == sym[None, :])
    K = 1e-2 * (a - a.T)
    base = dict(gpu=name, power_limit_and_max_sm_clock=power, n_dets=len(up), norb=chem.norb)
    hv = H.matvec(w1)
    for label, f in [("sigma, kappa None", lambda: H.sigma(up, dn, w1)), ("sigma, kappa within irreps", lambda: H.sigma(up, dn, w1, kappa=K)),
                     ("orbital_gradient_response", lambda: H.orbital_gradient_response(up, dn, w1, dw)),
                     ("two_rdm (same list and vector)", lambda: H.two_rdm(up, dn, w1))]:
        f()
        r, t = timed(f, args.repeats, np.array_equal)
        extra = {}
        if label == "sigma, kappa None":
            extra = dict(max_abs_minus_resident_hv_over_max=float(np.max(np.abs(r - hv)) / np.max(np.abs(hv))))
        emit(dict(base, what=label + " (C2 bench space, ground state)", **t, repeats_bit_identical=True, **extra))
        del r
    del H, up, dn, wts, w1, dw, hv

    # 2. the optimiser on the shipped input
    inp = os.path.join(ROOT, "data", "C2_v2z_curve", "r1.24253", "i_1sigma_g")
    for mode, kw in (("one_step", dict(one_step=True)), ("fixed_list (two-step)", dict(fixed_list=True))):
        with tempfile.TemporaryDirectory() as tmp:
            t0 = time.perf_counter()
            res = orbopt.optimize_orbitals(inp, tmp, max_macro=args.max_macro, **kw)
            emit(dict(gpu=name, power_limit_and_max_sm_clock=power, what="optimize_orbitals i_1sigma_g " + mode, converged=res["converged"],
                      seconds=time.perf_counter() - t0, history=res["history"]))
            if mode == "one_step":
                Hf, uf, df = res["hamiltonian"], res["up"], res["dn"]
                C = np.asarray(res["wts"]).reshape(len(uf), -1)
                Y = np.random.default_rng(2).standard_normal(C.shape)
                Y -= C @ (C.T @ Y)
                Kf = 1e-2 * (a - a.T)

                def micro():
                    Hf.sigma(uf, df, C, kappa=Kf)
                    Hf.orbital_gradient_response(uf, df, C, Y)
                    return Hf.matvec(Y)

                micro()
                _, t = timed(micro, args.repeats, np.array_equal)
                emit(dict(gpu=name, power_limit_and_max_sm_clock=power, what="one micro-iteration (sigma with kappa + response + H.v), shipped input",
                          n_dets=len(uf), n_states=C.shape[1], **t))

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
