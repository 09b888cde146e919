#!/usr/bin/env python
"""HCI -> natural orbitals: run a reference `hci` input (chem) on the GPU, compute the 1-RDM of its final wavefunction (all
states, on the GPU), and write the state-averaged natural-orbital basis for the next HCI run:
  DIR/FCIDUMP          the integrals rotated into the natural orbitals (descending occupation)
  DIR/<input name>     the input with only its orbital_symmetries line replaced by the natural orbitals' irreps
Prints one JSON line (occupations, variational energies, sum of the occupations).  The next run uses the existing tools:
  python scripts/natorb.py data/C2_v2z_curve/r1.24253/i_1sigma_g --out no
  python scripts/run_reference_input.py no/i_1sigma_g"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sqmc_b200 import hci, natorb  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("input")
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--fcidump", default=None, help="FCIDUMP of the input (default: next to it)")
    args = ap.parse_args()
    if hci.read_input(args.input)["hamiltonian_type"] != "chem":
        sys.exit("natorb.py: natural orbitals are for chem inputs (heg / hubbardk: gamma is the diagonal n(k))")
    fcidump = args.fcidump or os.path.join(os.path.dirname(os.path.abspath(args.input)), "FCIDUMP")
    res = hci.run_input(args.input, fcidump=fcidump, log=lambda *a: print(*a, file=sys.stderr))
    rdm = res["hamiltonian"].one_rdm(res["up"], res["dn"], res["wts"])
    no = natorb.natural_orbitals(res["system"], rdm)
    os.makedirs(args.out, exist_ok=True)
    natorb.rotate_fcidump(fcidump, no["coeffs"], no["irreps"], os.path.join(args.out, "FCIDUMP"))
    lines = open(args.input).read().splitlines(keepends=True)
    k = next(i for i, ln in enumerate(lines) if "orbital_symmetries" in ln)
    new = ",".join(str(int(x)) for x in no["irreps"]) + ","
    lines[k] = "%-34s orbital_symmetries(1:norb)\n" % new
    with open(os.path.join(args.out, os.path.basename(args.input)), "w") as f:
        f.write("".join(lines))
    occ = no["occupations"]
    print(json.dumps({"input": args.input, "n_det": len(res["up"]), "occupations": [float(x) for x in occ],
                      "energies": [float(e) for e in res["energy"]], "pt": [float(d) for d, _ in res["pt"]],
                      "sum_occupations": float(occ.sum())}))


if __name__ == "__main__":
    main()
