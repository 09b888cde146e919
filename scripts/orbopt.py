#!/usr/bin/env python
"""Orbital-optimised HCI: run a reference `hci` input (chem) and optimise its orbitals on the GPU's orbital gradient and
Hessian (sqmc_b200.orbopt), then write the optimised basis for the next HCI run:
  DIR/FCIDUMP          the integrals in the optimised orbitals (rotations within irreps, FCIDUMP column order kept)
  DIR/<input name>     a copy of the input (its orbital_symmetries line stays valid)
Prints one JSON line with the history of the macro iterations.  The next run uses the existing tools:
  python scripts/orbopt.py data/C2_v2z_curve/r1.24253/i_1sigma_g --out oo [--fixed-list | --one-step]
  python scripts/run_reference_input.py oo/i_1sigma_g
Natural orbitals first: run scripts/natorb.py and optimise its output."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sqmc_b200 import orbopt  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("input")
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--fixed-list", action="store_true", help="carry the first run's determinant list instead of re-selecting")
    ap.add_argument("--one-step", action="store_true", help="CI-orbital coupled Newton steps (implies --fixed-list)")
    ap.add_argument("--max-macro", type=int, default=10)
    ap.add_argument("--tol", type=float, default=1.0e-4, help="stop when max|gradient| < tol (Ha)")
    ap.add_argument("--fcidump", default=None, help="FCIDUMP of the input (default: next to it)")
    args = ap.parse_args()
    t0 = time.perf_counter()
    res = orbopt.optimize_orbitals(args.input, args.out, fixed_list=args.fixed_list, max_macro=args.max_macro, tol=args.tol,
                                   fcidump=args.fcidump, log=lambda *a: print(*a, file=sys.stderr), one_step=args.one_step)
    mode = "one_step" if args.one_step else "fixed_list" if args.fixed_list else "reselect"
    print(json.dumps({"input": args.input, "mode": mode, "converged": res["converged"],
                      "seconds": time.perf_counter() - t0, "history": res["history"]}))


if __name__ == "__main__":
    main()
