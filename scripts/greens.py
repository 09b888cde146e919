#!/usr/bin/env python
"""HCI -> single-particle Green's function: run a reference `hci` input (chem) on the GPU, then the removal and addition
Green's functions of its first state for the chosen orbitals of one spin (sqmc_b200.greens, every heavy step on the GPU):
  DIR/spectrum.txt   omega, the total A(omega) = sum_p A_pp and A_pp per orbital (FCIDUMP numbering and irrep in the header)
  DIR/poles.txt      every pole of every diagonal element: kind (removal / addition), orbital, omega, residue
and prints one JSON line with the first removal and addition poles (largest removal / smallest addition omega with a
residue above 1e-3): IP = -omega_removal and EA = -omega_addition.
  python scripts/greens.py data/C2_v2z_curve/r1.24253/i_1sigma_g --spin a --omega -1.5 1.0 501 --eta 0.01 --out gf
--orbitals takes FCIDUMP orbital numbers (1-based); the default is the two highest occupied and the two lowest empty orbitals
of that spin in the HF determinant."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sqmc_b200 import greens, hci  # noqa: E402

SIGNIFICANT = 1e-3   # residue of a pole reported as the IP / EA estimate


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("input")
    ap.add_argument("--orbitals", type=int, nargs="+", default=None, help="FCIDUMP orbital numbers (1-based)")
    ap.add_argument("--spin", choices=["a", "b"], default="a")
    ap.add_argument("--omega", type=float, nargs=3, metavar=("LO", "HI", "N"), default=[-1.5, 1.0, 501])
    ap.add_argument("--eta", type=float, default=0.01)
    ap.add_argument("--max-steps", type=int, default=100)
    ap.add_argument("--eps-select", type=float, default=None, help="widen the N-1 / N+1 spaces by heat-bath selection")
    ap.add_argument("--select-rounds", type=int, default=1)
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--fcidump", default=None, help="FCIDUMP of the input (default: next to it)")
    args = ap.parse_args()
    if hci.read_input(args.input)["hamiltonian_type"] != "chem":
        sys.exit("greens.py: the Green's function driver is for chem inputs")
    fcidump = args.fcidump or os.path.join(os.path.dirname(os.path.abspath(args.input)), "FCIDUMP")
    res = hci.run_input(args.input, fcidump=fcidump, log=lambda *a: print(*a, file=sys.stderr))
    system, H = res["system"], res["hamiltonian"]
    spin = 0 if args.spin == "a" else 1
    norb = system.norb
    if args.orbitals is None:
        nocc = system.ndn if spin else system.nup
        lib = [p for p in (nocc - 2, nocc - 1, nocc, nocc + 1) if 0 <= p < norb]
    else:
        if any(not 1 <= o <= norb for o in args.orbitals):
            sys.exit("greens.py: --orbitals must be FCIDUMP orbital numbers in 1..%d" % norb)
        lib = [int(system.orb_order_inv[o - 1]) - 1 for o in args.orbitals]
    fcid = [int(system.orb_order[p]) for p in lib]                 # FCIDUMP number of library orbital p
    irrep = [int(system.orbital_symmetries[p]) for p in lib]
    omega = np.linspace(args.omega[0], args.omega[1], int(args.omega[2]))
    wts = np.asarray(res["wts"])[:, 0]
    e0 = float(res["energy"][0])
    g = greens.greens_function(system, H, res["up"], res["dn"], wts, e0, lib, spin, omega, args.eta, max_steps=args.max_steps,
                               eps_select=args.eps_select, select_rounds=args.select_rounds)
    A = np.diagonal(greens.spectral_function(g["G_minus"] + g["G_plus"]), axis1=1, axis2=2)
    os.makedirs(args.out, exist_ok=True)
    labels = ["orb%d(irrep%d)" % (o, s) for o, s in zip(fcid, irrep)]
    np.savetxt(os.path.join(args.out, "spectrum.txt"), np.column_stack([omega, A.sum(axis=1), A]),
               header="spin %s, E0 = %.10f, eta = %g; columns: omega A_total %s" % (args.spin, e0, args.eta, " ".join(labels)))
    first = {}
    with open(os.path.join(args.out, "poles.txt"), "w") as f:
        f.write("# kind orbital(FCIDUMP) irrep omega residue\n")
        for kind in ("minus", "plus"):
            for k, p in enumerate(lib):
                for om, r in zip(g["poles_" + kind][k], g["residues_" + kind][k]):
                    f.write("%s %d %d %.10f %.3e\n" % ("removal" if kind == "minus" else "addition", fcid[k], irrep[k], om, r))
                    if r > SIGNIFICANT:
                        best = first.get(kind)
                        if best is None or (om > best[0] if kind == "minus" else om < best[0]):
                            first[kind] = (float(om), fcid[k])
    out = {"input": args.input, "spin": args.spin, "E0": e0, "orbitals_fcidump": fcid, "n_minus": g["n_minus"], "n_plus": g["n_plus"],
           "steps_minus": [int(s) for s in g["steps_minus"]], "steps_plus": [int(s) for s in g["steps_plus"]]}
    if "minus" in first:
        out.update(first_removal_pole=first["minus"][0], ip=-first["minus"][0], ip_orbital=first["minus"][1])
    if "plus" in first:
        out.update(first_addition_pole=first["plus"][0], ea=-first["plus"][0], ea_orbital=first["plus"][1])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
