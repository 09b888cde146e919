"""Orbital-optimised HCI: a two-step optimiser (CI, then orbitals) on the GPU's orbital gradient and Hessian.

Every macro iteration solves the CI problem in the current orbitals, takes SparseHamiltonian.orbital_derivatives of the
state-averaged variational energy, and makes a Newton step in the rotations kappa_pq (p > q, same irrep) on the reduced
Hessian, level-shifted when its lowest eigenvalue is below a small positive floor and capped in size.  The orbitals are kept
as the total rotation C relative to the original FCIDUMP, and every iteration writes natorb.rotate_fcidump(original, C), so
the integral filter of the reader never compounds.  CI-orbital coupling is not included.

Two modes, both through hci.perform_hci:
  re-select (default)  every iteration runs the input's HCI schedule from the HF determinant in the current orbitals (no PT);
  fixed list           the determinant list of the first run is carried along (remap_determinants), each iteration rebuilds
                       H and runs Davidson from the previous vectors; a step that raises the weighted energy is halved and
                       retried, so the energy does not increase.
"""
import os
import time

import numpy as np
from scipy.linalg import expm

from . import hci, natorb


def library_to_library(old_system, new_system):
    """perm[p] = library orbital of new_system that is library orbital p of old_system (both number the same FCIDUMP columns)"""
    norb = old_system.norb
    col = np.asarray(old_system.orb_order[:norb]) - 1                 # old library orbital -> FCIDUMP column
    return np.asarray(new_system.orb_order_inv[:norb])[col] - 1       # FCIDUMP column -> new library orbital


def remap_strings(strings, perm):
    """strings (n,) python ints or uint64 words of one spin, orbital p renamed perm[p] -> (new words (n,) uint64, signs (n,))
    The sign is the parity of the permutation that sorts the renamed creation operators back into ascending order."""
    s = np.asarray(strings, dtype=np.uint64)
    perm = np.asarray(perm)
    norb = len(perm)
    bits = [((s >> np.uint64(p)) & np.uint64(1)).astype(bool) for p in range(norb)]
    out = np.zeros(len(s), dtype=np.uint64)
    for p in range(norb):
        out |= bits[p].astype(np.uint64) << np.uint64(perm[p])
    odd = np.zeros(len(s), dtype=bool)
    for a in range(norb):
        for b in range(a + 1, norb):
            if perm[a] > perm[b]:
                odd ^= bits[a] & bits[b]
    return out, np.where(odd, -1.0, 1.0)


def remap_determinants(up, dn, wts, perm, time_sym=False, z=1):
    """A wavefunction over (n, 2) uint64 determinants (norb <= 64) written in new orbital labels perm[p]: strings remapped,
    each coefficient times the parities of its alpha and beta strings; on time_sym lists a representative whose renamed
    strings come out with up > dn is swapped back to representative form and its coefficient multiplied by z."""
    up = np.asarray(up, dtype=np.uint64).reshape(-1, 2)
    dn = np.asarray(dn, dtype=np.uint64).reshape(-1, 2)
    if np.any(up[:, 1]) or np.any(dn[:, 1]):
        raise ValueError("remap_determinants: orbitals beyond 64 are not supported")
    u, su = remap_strings(up[:, 0], perm)
    d, sd = remap_strings(dn[:, 0], perm)
    w = np.array(wts, dtype=np.float64).reshape(len(up), -1) * (su * sd)[:, None]
    if time_sym:
        flip = u > d
        u, d = np.where(flip, d, u), np.where(flip, u, d)
        w[flip] *= z
    nu = np.zeros_like(up)
    nd = np.zeros_like(dn)
    nu[:, 0], nd[:, 0] = u, d
    return nu, nd, w.reshape(np.shape(wts))


def rotation_parameters(system):
    """(p, q) with p > q in library numbering and the same irrep"""
    sym = np.asarray(system.orbital_symmetries)
    return [(p, q) for p in range(system.norb) for q in range(p) if sym[p] == sym[q]]


def newton_step(grad, hess, max_step=0.5, floor=1.0e-4):
    """-(H + shift)^-1 g with shift = floor - lambda_min when the lowest eigenvalue lambda_min is below floor; the step is
    scaled down to norm max_step if longer.  -> (step, shift)"""
    ev, vec = np.linalg.eigh(0.5 * (hess + hess.T))
    shift = max(0.0, floor - ev[0])
    step = -vec @ ((vec.T @ grad) / (ev + shift))
    nrm = float(np.linalg.norm(step))
    if nrm > max_step:
        step *= max_step / nrm
    return step, shift


def kappa_in_fcidump_columns(system, pairs, step):
    """the antisymmetric kappa in FCIDUMP columns from the step over library pairs (p, q)"""
    norb = system.norb
    col = np.asarray(system.orb_order[:norb]) - 1
    K = np.zeros((norb, norb))
    for (p, q), k in zip(pairs, step):
        K[col[p], col[q]] = k
        K[col[q], col[p]] = -k
    return K


def _write_input(input_path, out_dir):
    dst = os.path.join(out_dir, os.path.basename(input_path))
    with open(input_path) as f, open(dst, "w") as g:
        g.write(f.read())
    return dst


def optimize_orbitals(input_path, out_dir, fixed_list=False, max_macro=10, tol=1.0e-4, max_step=0.5, shift_floor=1.0e-4, max_halvings=8,
                      state_weights=None, fcidump=None, log=None):
    """Optimise the orbitals of a chem `hci` input.  Writes out_dir/FCIDUMP (the orbitals of the last macro iteration that ran
    the CI, columns and irreps as in the original) and a copy of the input as out_dir/<input name>.
    -> dict(history=[{macro, n_det, energies, energy (weighted), max_grad, step_norm, shift, halvings, seconds}], converged,
    coeffs C (column k = orbital k in the original FCIDUMP orbitals), irreps, system, hamiltonian, up, dn, wts)"""
    from . import ChemSystem, SparseHamiltonian
    say = log or (lambda *_: None)
    cfg = hci.read_input(input_path)
    if cfg["hamiltonian_type"] != "chem":
        raise ValueError("optimize_orbitals: chem inputs only (heg / hubbardk orbitals are fixed by momentum)")
    src = fcidump or os.path.join(os.path.dirname(os.path.abspath(input_path)), "FCIDUMP")
    os.makedirs(out_dir, exist_ok=True)
    _write_input(input_path, out_dir)
    out_fcidump = os.path.join(out_dir, "FCIDUMP")
    orbsym = list(cfg["orbital_symmetries"])
    ns = cfg["n_states"]
    sw = np.full(ns, 1.0 / ns) if state_weights is None else np.asarray(state_weights, dtype=np.float64)
    norb = cfg["norb"]

    def setup(C):
        natorb.rotate_fcidump(src, C, orbsym, out_fcidump)
        system = ChemSystem(out_fcidump, nelec=cfg["nelec"], nup=cfg["nup"], orbital_symmetries=orbsym, time_sym=cfg["time_sym"], z=cfg["z"])
        return system, SparseHamiltonian(system)

    def solve_fixed(C, prev):
        """CI on the carried list in the orbitals C, from the previous vectors remapped"""
        system, H = setup(C)
        perm = library_to_library(prev["system"], system)
        up, dn, w = remap_determinants(prev["up"], prev["dn"], prev["wts"], perm, time_sym=system.time_sym, z=system.z)
        H.generate_sparse_ham_upper_triangular(up, dn)
        dv = H.davidson_sparse(n_states=ns, initial_vector=w)
        return dict(system=system, H=H, up=up, dn=dn, wts=np.asarray(dv["evecs"]), energy=np.asarray(dv["evals"], dtype=np.float64))

    C = np.eye(norb)
    history = []
    converged = False
    state = None
    for macro in range(max_macro):
        t0 = time.perf_counter()
        halvings = 0
        if state is None or not fixed_list:
            system, H = setup(C)
            res = hci.perform_hci(H, system, cfg["eps_var"], cfg["eps_var_sched"], n_states=ns, eps_pt=None)
            state = dict(system=system, H=H, up=res["up"], dn=res["dn"], wts=res["wts"], energy=np.asarray(res["energy"], dtype=np.float64))
        system, H = state["system"], state["H"]
        der = H.orbital_derivatives(state["up"], state["dn"], state["wts"], state_weights=sw)
        pairs = rotation_parameters(system)
        idx_p = np.array([p for p, _ in pairs], dtype=np.int64)
        idx_q = np.array([q for _, q in pairs], dtype=np.int64)
        grad = der["gradient"][idx_p, idx_q]
        max_g = float(np.max(np.abs(grad))) if len(grad) else 0.0
        entry = dict(macro=macro, n_det=int(len(state["up"])), energies=[float(e) for e in state["energy"]], energy=float(sw @ state["energy"]),
                     rdm_energy=der["energy"], max_grad=max_g, n_params=len(pairs), step_norm=0.0, shift=0.0, halvings=0)
        if max_g < tol or macro == max_macro - 1:
            converged = max_g < tol
            entry["seconds"] = time.perf_counter() - t0
            history.append(entry)
            say("orbopt %d: E=%.10f max|g|=%.3e n_det=%d" % (macro, entry["energy"], max_g, entry["n_det"]))
            break
        hess = der["hessian"][idx_p, idx_q][:, idx_p, idx_q]
        step, shift = newton_step(grad, hess, max_step=max_step, floor=shift_floor)
        if fixed_list:
            e_prev = entry["energy"]
            while True:
                U = expm(-kappa_in_fcidump_columns(system, pairs, step))
                trial = solve_fixed(C @ U, state)
                if float(sw @ trial["energy"]) <= e_prev or halvings >= max_halvings:
                    break
                step = 0.5 * step
                halvings += 1
            if float(sw @ trial["energy"]) > e_prev:   # no step lowered the energy: stay, and stop
                setup(C)
                entry.update(step_norm=0.0, shift=shift, halvings=halvings, seconds=time.perf_counter() - t0)
                history.append(entry)
                say("orbopt %d: no energy-lowering step after %d halvings" % (macro, halvings))
                break
            C = C @ U
            state = trial
        else:
            C = C @ expm(-kappa_in_fcidump_columns(system, pairs, step))
        entry.update(step_norm=float(np.linalg.norm(step)), shift=shift, halvings=halvings, seconds=time.perf_counter() - t0)
        history.append(entry)
        say("orbopt %d: E=%.10f max|g|=%.3e |step|=%.3e shift=%.2e halvings=%d n_det=%d"
            % (macro, entry["energy"], max_g, entry["step_norm"], shift, halvings, entry["n_det"]))
    return dict(history=history, converged=converged, coeffs=C, irreps=np.array(orbsym, dtype=np.int32), system=state["system"],
                hamiltonian=state["H"], up=state["up"], dn=state["dn"], wts=state["wts"], fcidump=out_fcidump)
