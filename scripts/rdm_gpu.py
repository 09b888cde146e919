#!/usr/bin/env python
"""Time the one-particle density matrix (sqmc_b200_one_rdm) on the bench's C2 HCI space against one from-scratch H build of
the same list, in one process: the space is grown on the GPU (spaces.hci_space on ChemSystem(FCIDUMP), plain
determinants, ~10^7 by default) and its wavefunction is the one that run returns; the second state of the two-state timing
is a fixed pseudo-random vector.  Times are host wall clock around calls that end in a device synchronisation (the call copies
the result back), after a warm-up; median and spread over --repeats.  Repeats must be bit-identical.  Appends JSON lines to --out."""
import argparse
import json
import os
import subprocess
import sys
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


def timed(f, repeats):
    out, ts = None, []
    for _ in range(repeats):
        t0 = time.perf_counter()
        r = f()
        ts.append(time.perf_counter() - t0)
        if out is None:
            out = r
        elif not np.array_equal(out, r):
            raise AssertionError("one_rdm repeats differ")
    ts = np.array(ts) * 1e3
    return out, dict(median_ms=float(np.median(ts)), min_ms=float(ts.min()), max_ms=float(ts.max()), repeats=repeats)


def main():
    import sqmc_b200 as sq
    from sqmc_b200 import spaces
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-dets", type=int, default=10_000_000)
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_one_rdm_1e7.jsonl"))
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
    rows = []
    H.one_rdm(up, dn, w1)  # warm-up
    g1, t1 = timed(lambda: H.one_rdm(up, dn, w1), args.repeats)
    H.one_rdm(up, dn, w2)
    g2, t2 = timed(lambda: H.one_rdm(up, dn, w2), args.repeats)
    assert np.array_equal(g2[0], g1)
    t0 = time.perf_counter()
    nnz = H.generate_sparse_ham_upper_triangular(up, dn, ndet_old=0)
    t_build = (time.perf_counter() - t0) * 1e3
    tr = [float(np.trace(g1[s])) for s in (0, 1)]
    base = dict(gpu=name, power_limit_and_max_sm_clock=power, n_dets=n, e_var=e, space_s=t_space, nnz_upper=int(nnz))
    rows.append(dict(base, what="one_rdm", n_states=1, **t1, trace_up_dn=tr))
    rows.append(dict(base, what="one_rdm", n_states=2, **t2))
    rows.append(dict(base, what="build_h from scratch", wall_ms=t_build, device_total_ms=H.build_times()["total_ms"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
            print(json.dumps(r))
    assert t1["median_ms"] < t_build, "one_rdm (one state) is not faster than one H build"


if __name__ == "__main__":
    main()
