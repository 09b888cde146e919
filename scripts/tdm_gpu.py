#!/usr/bin/env python
"""Time the transition density matrices (sqmc_b200_transition_one_rdm / transition_two_rdm) against two_rdm on the bench's
C2 HCI space with that run's H still resident, in one process: the space is grown on the GPU (spaces.hci_space on
ChemSystem(FCIDUMP), plain determinants, ~10^7 by default); bra = the ground state that run returns, ket = a fixed
pseudo-random vector (spaces.splitmix_vector).  Times are host wall clock around calls that end in a device synchronisation
(the call copies the result back), after a warm-up; median and spread over --repeats, and repeats must be bit-identical.
Also records max|transition_two_rdm(c, c) - two_rdm(c)| (must be 0) and |rdm_energy(T1(a,b), T2(a,b)) - a.(H b)| with the
resident matrix-vector product.  Appends JSON lines to --out."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from rdm_gpu import gpu_info  # noqa: E402


def timed(f, repeats, what):
    out, ts = None, []
    for _ in range(repeats):
        t0 = time.perf_counter()
        r = f()
        ts.append(time.perf_counter() - t0)
        if out is None:
            out = r
        elif not np.array_equal(out, r):
            raise AssertionError("%s repeats differ" % what)
    ts = np.array(ts) * 1e3
    return out, dict(median_ms=float(np.median(ts)), min_ms=float(ts.min()), max_ms=float(ts.max()), repeats=repeats)


def main():
    import sqmc_b200 as sq
    from sqmc_b200 import rdm, spaces
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-dets", type=int, default=10_000_000)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_transition_rdm_1e7.jsonl"))
    args = ap.parse_args()
    name, power = gpu_info()
    chem = sq.ChemSystem(os.path.join(ROOT, "data", "C2_v2z_curve", "r1.24253", "FCIDUMP"))
    H = sq.SparseHamiltonian(chem)
    t0 = time.perf_counter()
    up, dn, wts, e = spaces.hci_space(H, chem, args.n_dets)
    t_space = time.perf_counter() - t0
    n = len(up)
    a = np.ascontiguousarray(wts[:, 0])
    b = spaces.splitmix_vector(n)
    H.transition_one_rdm(up, dn, a, b)  # warm-up
    t1, r1 = timed(lambda: H.transition_one_rdm(up, dn, a, b), args.repeats, "transition_one_rdm")
    H.transition_two_rdm(up, dn, a, b)
    t2, r2 = timed(lambda: H.transition_two_rdm(up, dn, a, b), args.repeats, "transition_two_rdm")
    H.two_rdm(up, dn, a)
    g2, r2ref = timed(lambda: H.two_rdm(up, dn, a), args.repeats, "two_rdm")
    d_cc = float(np.max(np.abs(H.transition_two_rdm(up, dn, a, a) - g2)))
    e_tdm = rdm.rdm_energy(chem, t1, t2)
    e_mv = float(a @ H.matvec(b))
    base = dict(gpu=name, power_limit_and_max_sm_clock=power, n_dets=n, e_var=e, space_s=t_space)
    rows = [dict(base, what="transition_one_rdm", n_pairs=1, **r1),
            dict(base, what="transition_two_rdm", n_pairs=1, **r2),
            dict(base, what="two_rdm", n_states=1, **r2ref),
            dict(base, what="transition_two_rdm(c, c) vs two_rdm(c)", max_abs_diff=d_cc),
            dict(base, what="energy identity", rdm_energy_of_tdms=e_tdm, a_dot_H_b=e_mv, abs_diff=abs(e_tdm - e_mv),
                 norm_a_times_norm_b=float(np.linalg.norm(a) * np.linalg.norm(b)))]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
            print(json.dumps(r))


if __name__ == "__main__":
    main()
