#!/usr/bin/env python
"""In-process A/B of the H.v row layouts on ONE resident matrix (same box, same clocks).
usage: bundle_inproc.py [n_dets] [space: hci|lowest] [R,...]   R = rows per bundle (2 or 4), 0 = plain rows"""
import ctypes as C, json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import sqmc_b200 as sq
from sqmc_b200 import _lib, spaces

n_dets = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
space = sys.argv[2] if len(sys.argv) > 2 else "hci"
order = [int(a) for a in sys.argv[3].split(",")] if len(sys.argv) > 3 else [4, 2, 0, 4, 2, 0]
_lib.init(device=0)
L = _lib.load()
chem = sq.ChemSystem("data/C2_v2z_curve/r1.24253/FCIDUMP")
H = sq.SparseHamiltonian(chem)
if space == "hci":
    up, dn, _, _ = spaces.hci_space(H, chem, n_dets)
else:
    up, dn, _ = spaces.c2_lowest_energy_space(chem, n_dets)
H.generate_sparse_ham_upper_triangular(up, dn)
n = len(up); nnz = H.nnz()["nnz_full"]
stream = torch.cuda.Stream(); torch.cuda.set_stream(stream)
x = torch.from_numpy(spaces.splitmix_vector(n)).cuda(); y = torch.zeros(n, dtype=torch.float64, device="cuda")
sp = C.c_void_p(stream.cuda_stream)
ref = None
cur = 4
for R in order:
    t0 = time.perf_counter()
    if R != cur:
        H.set_row_bundle(R); cur = R
    t_set = time.perf_counter() - t0
    for _ in range(5):
        _lib.check(L.sqmc_b200_matvec_dev(H._h, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), sp))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(30):
        _lib.check(L.sqmc_b200_matvec_dev(H._h, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), sp))
    e1.record(stream); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 30
    yy = y.cpu().numpy().copy()
    if ref is None: ref = yy
    print(json.dumps({"n": n, "nnz_full": nnz, "R": R, "ms": ms, "GBs": (12.0 * nnz + 20.0 * n) / ms / 1e6, "frac_6455.6": (12.0 * nnz + 20.0 * n) / ms / 1e6 / 6455.6,
                      "set_layout_s": t_set, "max_rel_diff_vs_first": float(np.max(np.abs(yy - ref)) / np.max(np.abs(ref)))}), flush=True)
