#!/usr/bin/env python
"""Time the two-particle density matrix (sqmc_b200_two_rdm) on the bench's C2 HCI space with that run's H still resident,
against one from-scratch H build of the same list, in one process: the space is grown on the GPU (spaces.hci_space on
ChemSystem(FCIDUMP), plain determinants, ~10^7 by default) and its wavefunction is the one that run returns; the second state
of the two-state timing is a fixed pseudo-random vector.  Times are host wall clock around calls that end in a device
synchronisation (the call copies the result back), after a warm-up; median and spread over --repeats.  Repeats must be
bit-identical.  Also records |rdm_energy - e_var|, <S^2>, and one call's phase split (SQMC_RDM2_PROFILE=1, on stderr).
Appends JSON lines to --out."""
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


def timed(f, repeats):
    out, ts = None, []
    for _ in range(repeats):
        t0 = time.perf_counter()
        r = f()
        ts.append(time.perf_counter() - t0)
        if out is None:
            out = r
        elif not np.array_equal(out, r):
            raise AssertionError("two_rdm repeats differ")
    ts = np.array(ts) * 1e3
    return out, dict(median_ms=float(np.median(ts)), min_ms=float(ts.min()), max_ms=float(ts.max()), repeats=repeats)


def main():
    import sqmc_b200 as sq
    from sqmc_b200 import rdm, spaces
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-dets", type=int, default=10_000_000)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_two_rdm_1e7.jsonl"))
    args = ap.parse_args()
    name, power = gpu_info()
    chem = sq.ChemSystem(os.path.join(ROOT, "data", "C2_v2z_curve", "r1.24253", "FCIDUMP"))
    H = sq.SparseHamiltonian(chem)
    t0 = time.perf_counter()
    up, dn, wts, e = spaces.hci_space(H, chem, args.n_dets)
    t_space = time.perf_counter() - t0
    n = len(up)
    w1 = np.ascontiguousarray(wts[:, 0])
    w2 = np.asfortranarray(np.stack([w1, spaces.splitmix_vector(n)], axis=1))
    H.two_rdm(up, dn, w1)  # warm-up
    g1, t1 = timed(lambda: H.two_rdm(up, dn, w1), args.repeats)
    H.two_rdm(up, dn, w2)
    g2, t2 = timed(lambda: H.two_rdm(up, dn, w2), args.repeats)
    d = np.max(np.abs(g2[0] - g1))
    os.environ["SQMC_RDM2_PROFILE"] = "1"
    sys.stderr.flush()
    t0 = time.perf_counter()
    H.two_rdm(up, dn, w1)
    t_prof = (time.perf_counter() - t0) * 1e3
    del os.environ["SQMC_RDM2_PROFILE"]
    g1e = H.one_rdm(up, dn, w1)
    norm2 = float(w1 @ w1)
    e_rdm = rdm.rdm_energy(chem, g1e, g1)
    s2 = float(rdm.spin_squared(g1, chem.nup, chem.ndn, norm2)) / norm2
    t0 = time.perf_counter()
    nnz = H.generate_sparse_ham_upper_triangular(up, dn, ndet_old=0)
    t_build = (time.perf_counter() - t0) * 1e3
    base = dict(gpu=name, power_limit_and_max_sm_clock=power, n_dets=n, e_var=e, space_s=t_space, nnz_upper=int(nnz))
    rows = [dict(base, what="two_rdm", n_states=1, **t1, rdm_energy=e_rdm, abs_rdm_energy_minus_e_var=abs(e_rdm - e), s_squared=s2),
            dict(base, what="two_rdm", n_states=2, **t2, max_abs_state0_vs_one_state_call=float(d)),
            dict(base, what="two_rdm phase-split call (synchronising marks on stderr)", wall_ms=t_prof),
            dict(base, what="build_h from scratch", wall_ms=t_build, device_total_ms=H.build_times()["total_ms"])]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
            print(json.dumps(r))


if __name__ == "__main__":
    main()
