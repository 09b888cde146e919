#!/usr/bin/env python
"""Davidson with n_states = 1 and 2 on a C2 space (time per run, matvecs): shows the two-vector H.v kernel at work."""
import os, sys, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import sqmc_b200 as sq
from sqmc_b200 import _lib, spaces
n = int(sys.argv[1]) if len(sys.argv) > 1 else 3_000_000
_lib.init(device=0)
chem = sq.ChemSystem("data/C2_v2z_curve/r1.24253/FCIDUMP")
up, dn, _ = spaces.c2_lowest_energy_space(chem, n)
H = sq.SparseHamiltonian(chem)
H.generate_sparse_ham_upper_triangular(up, dn)
for R in (4, 0):
    H.set_row_bundle(R)
    for ns in (1, 2):
        H.davidson_sparse(n_states=ns, max_vec_per_state=3)  # warm-up
        H.davidson_sparse(n_states=ns, max_vec_per_state=3)
        t0 = time.perf_counter()
        d = H.davidson_sparse(n_states=ns)
        t = time.perf_counter() - t0
        print(json.dumps({"rows_per_bundle": R, "n_states": ns, "seconds": t, "n_matvec": d["n_matvec"],
                          "ms_per_matvec_all_in": 1e3 * t / d["n_matvec"], "evals": [float(e) for e in d["evals"]]}), flush=True)
