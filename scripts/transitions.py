#!/usr/bin/env python
"""HCI -> state-to-state quantities: run a reference `hci` input with n_states >= 2 on the GPU, then the transition density
matrices of every pair (I, J) of its final states in one call each (sqmc_b200 transition_one_rdm / transition_two_rdm, on
the GPU), and from them:
  - the overlaps <I|J> (trace of gamma over N), <I|H|J> (rdm.rdm_energy) and <I|S^2|J> (rdm.spin_squared), as matrices;
  - for every (0, J), J > 0, the natural transition orbitals (natorb.natural_transition_orbitals): singular values and the
    participation ratio, and DIR/nto_0_J.txt with the hole and particle columns in FCIDUMP orbitals.  The spin coupling is
    singlet (spin_sign = +1) when states 0 and J have the same S, triplet (-1) otherwise.
Prints one JSON line with the matrices and each state's <S^2>, then one JSON line per (0, J).
  python scripts/transitions.py data/C2_v2z_curve/r1.24253/i_1sigma_g --out tdm"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sqmc_b200 import hci, natorb, rdm  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("input")
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--fcidump", default=None, help="FCIDUMP of the input (default: next to it)")
    args = ap.parse_args()
    cfg = hci.read_input(args.input)
    if cfg["hamiltonian_type"] != "chem":
        sys.exit("transitions.py: transition properties are for chem inputs")
    if cfg["n_states"] < 2:
        sys.exit("transitions.py: the input asks for n_states = %d; transitions need at least two states" % cfg["n_states"])
    fcidump = args.fcidump or os.path.join(os.path.dirname(os.path.abspath(args.input)), "FCIDUMP")
    res = hci.run_input(args.input, fcidump=fcidump, log=lambda *a: print(*a, file=sys.stderr))
    system, H = res["system"], res["hamiltonian"]
    wts = np.asarray(res["wts"])
    ns = wts.shape[1]
    I, J = np.meshgrid(np.arange(ns), np.arange(ns), indexing="ij")
    bra, ket = wts[:, I.ravel()], wts[:, J.ravel()]
    t1 = H.transition_one_rdm(res["up"], res["dn"], bra, ket)
    t2 = H.transition_two_rdm(res["up"], res["dn"], bra, ket)
    nel = system.nup + system.ndn
    ovl = np.array([np.trace(t1[k, 0] + t1[k, 1]) / nel for k in range(ns * ns)]).reshape(ns, ns)
    h = np.array([rdm.rdm_energy(system, t1[k], t2[k]) for k in range(ns * ns)]).reshape(ns, ns)
    s2 = np.array([rdm.spin_squared(t2[k], system.nup, system.ndn, ovl.ravel()[k]) for k in range(ns * ns)]).reshape(ns, ns)
    s2_state = np.diag(s2) / np.diag(ovl)
    spin = np.round((np.sqrt(1.0 + 4.0 * np.maximum(s2_state, 0.0)) - 1.0) / 2.0 * 2.0) / 2.0   # nearest S (half-integers allowed)
    off = ~np.eye(ns, dtype=bool)
    print(json.dumps({"input": args.input, "n_det": len(res["up"]), "energies": [float(e) for e in res["energy"]],
                      "overlap": ovl.tolist(), "H": h.tolist(), "S2": s2.tolist(), "state_S2": s2_state.tolist(),
                      "max_abs_offdiag_overlap": float(np.max(np.abs(ovl[off]))), "max_abs_offdiag_H": float(np.max(np.abs(h[off])))}))
    os.makedirs(args.out, exist_ok=True)
    norb = system.norb
    for j in range(1, ns):
        sign = 1 if spin[0] == spin[j] else -1
        nto = natorb.natural_transition_orbitals(system, t1[j], spin_sign=sign)
        path = os.path.join(args.out, "nto_0_%d.txt" % j)
        cols = np.hstack([nto["holes"], nto["particles"]])
        header = ("natural transition orbitals <0| . |%d>, spin_sign %+d, FCIDUMP orbitals 1..%d by row\n"
                  "columns 1..%d: holes (ket side), %d..%d: particles (bra side), ordered by singular value\n"
                  "singular values: %s") % (j, sign, norb, norb, norb + 1, 2 * norb, " ".join("%.10e" % x for x in nto["singular_values"]))
        np.savetxt(path, cols, fmt="%.12e", header=header)
        print(json.dumps({"pair": [0, j], "spin_sign": sign, "singular_values": [float(x) for x in nto["singular_values"]],
                          "participation_ratio": float(nto["participation_ratio"]), "file": path}))


if __name__ == "__main__":
    main()
