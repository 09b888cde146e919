"""Single-particle Green's function of a variational wavefunction (chem), with removal and addition spectra.

For one state Psi_0 of energy E_0 (library orbital numbering, real orbitals, z = omega + i eta, Hartree):
  removal   G-_pq(z) = <Psi_0| a+_q (z + H - E_0)^-1 a_p |Psi_0>,   poles at omega = E_0 - E_n(N-1)
  addition  G+_pq(z) = <Psi_0| a_p (z - H + E_0)^-1 a+_q |Psi_0>,   poles at omega = E_n(N+1) - E_0
  G = G+ + G-,  A_pp(omega) = -Im G_pp(omega) / pi.
Both spins are separate calls; the mixed-spin blocks are zero.

Every heavy step runs on the GPU: the images phi_p = a_p Psi_0 (chi_p = a+_p Psi_0) and the union of their determinants
(SparseHamiltonian.ladder), optional heat-bath widening of that space, the H build of the N-1 / N+1 space on a plain handle,
and one Lanczos run per image with full reorthogonalisation (SparseHamiltonian.lanczos_tridiagonal).  The host evaluates
the continued fractions from the tridiagonal matrices T: with T = U diag(e) U^T,
  <v_q| (z -+ (H - E_0))^-1 |v_p> = ||v_p|| sum_j <v_q|q_j> sum_k U_jk U_0k / (z - omega_k),
omega_k = E_0 - e_k (removal) or e_k - E_0 (addition), and the residue of the diagonal element at omega_k is ||v_p||^2 U_0k^2.
Off-diagonal elements come from the Krylov overlaps of each run, not from a block Lanczos: they are exact when the Krylov
spaces are complete.
"""
import copy

import numpy as np
from scipy.linalg import eigh_tridiagonal

from . import systems


def electron_space(system, spin, create):
    """The ChemSystem of the N-1 (create False) or N+1 (create True) electron space, one electron less / more of `spin`
    (0 up, 1 dn): the same integrals, orbital order and core energy as `system`, not time-reversal symmetrised.  Its HF
    determinant is that of `system` with the highest occupied orbital of that spin emptied or the lowest empty one filled.
    -> (system_x, flipped).  Chem handles hold N_alpha >= N_beta; when the new space has fewer alpha than beta electrons,
    system_x describes the spin-flipped space and flipped is True: its determinants are (dn, up) of the images.  H is spin
    free, and the swap changes the alpha-first phase of every determinant of the space by the same (-1)^(N_alpha N_beta),
    which the Green's function (bilinear in the images) does not see."""
    if not isinstance(system, systems.ChemSystem):
        raise ValueError("greens: the Green's function driver is for chem systems")
    s = copy.copy(system)
    d = 1 if create else -1
    hf = int(system.hf_dn if spin else system.hf_up)
    hf = (hf | ((~hf) & (hf + 1))) if create else (hf & ~(1 << (hf.bit_length() - 1)) if hf else 0)
    if spin:
        s.ndn, s.hf_dn = s.ndn + d, hf
    else:
        s.nup, s.hf_up = s.nup + d, hf
    s.nelec = system.nelec + d
    s.time_sym, s.z = False, 1
    flipped = s.nup < s.ndn
    if flipped:
        s.nup, s.ndn, s.hf_up, s.hf_dn = s.ndn, s.nup, s.hf_dn, s.hf_up
    return s, flipped


def krylov_resolvent(alpha, beta, overlaps, steps, norms, e0, z, addition):
    """M[w, a, b] = <v_b| R(z_w) |v_a> for the Lanczos runs of lanczos_tridiagonal started from v_a (norms[a] = ||v_a||;
    runs with norms[a] = 0 give zeros), R = (z + H - E_0)^-1 (addition False) or (z - H + E_0)^-1 (addition True).
    -> (M (n_z, P, P) complex, poles: list of P arrays, residues: list of P arrays of the diagonal elements)"""
    z = np.asarray(z, dtype=np.complex128).reshape(-1)
    P = len(norms)
    M = np.zeros((len(z), P, P), dtype=np.complex128)
    poles, residues = [], []
    for a in range(P):
        m = int(steps[a])
        if norms[a] == 0.0 or m == 0:
            poles.append(np.zeros(0))
            residues.append(np.zeros(0))
            continue
        ev, U = eigh_tridiagonal(alpha[a, :m], beta[a, :m - 1])
        om = ev - e0 if addition else e0 - ev
        W = U * U[0, :]                                    # W[j, k] = U_jk U_0k
        R = (1.0 / (z[:, None] - om[None, :])) @ W.T       # R[w, j] = [(z -+ (T - E_0))^-1]_j0
        M[:, a, :] = norms[a] * (R @ overlaps[a, :m, :])
        order = np.argsort(om)
        poles.append(om[order])
        residues.append(norms[a] ** 2 * U[0, order] ** 2)
    return M, poles, residues


def _first_order_amplitudes(HX, up, dn, phi, n_old):
    """max_j |(H phi_j)_i / (E_j - H_ii)| for the rows i >= n_old that a selection round added (phi is zero there): the
    first-order amplitudes of the new determinants, with E_j the Rayleigh quotient of phi_j, so the next round screens
    their excitations like those of the images.  Builds H over the current list."""
    HX.generate_sparse_ham_upper_triangular(up, dn)
    y = HX.matvec(phi).reshape(len(up), -1)
    n2 = np.sum(phi * phi, axis=0)
    e = np.divide(np.sum(phi * y, axis=0), n2, out=np.zeros_like(n2), where=n2 > 0.0)
    den = e[None, :] - HX.diagonal(up[n_old:], dn[n_old:])[:, None]
    den = np.where(np.abs(den) < 1e-8, 1e-8, den)   # the Davidson preconditioner's guard
    return np.max(np.abs(y[n_old:] / den), axis=1)


def _sector(system, H, up, dn, wts, state, e0, orbitals, spin, create, z, max_steps, eps_select, select_rounds, tol):
    from .api import SparseHamiltonian
    w = np.asarray(wts, dtype=np.float64)
    w = w.reshape(-1, 1) if w.ndim == 1 else w
    up2, dn2, phi = H.ladder(up, dn, w, orbitals, spin, create, state=state)
    phi = phi / np.sqrt(np.sum(np.sort(w[:, state] ** 2)))   # summed in sorted order: the same bits for any row order
    P = len(orbitals)
    if len(up2) == 0:
        return np.zeros((len(z), P, P), dtype=np.complex128), [np.zeros(0)] * P, [np.zeros(0)] * P, 0, np.zeros(P, dtype=np.int64)
    sysx, flipped = electron_space(system, spin, create)
    if flipped:
        up2, dn2 = dn2, up2
    HX = SparseHamiltonian(sysx)
    try:
        if eps_select is not None:
            coeff = np.max(np.abs(phi), axis=1)
            for r in range(int(select_rounds)):
                nu, nd, _ = HX.get_next_det_list(up2, dn2, coeff, np.full(len(up2), 9.0e99), float(eps_select))
                if len(nu) == 0:
                    break
                n_old = len(up2)
                up2, dn2 = np.concatenate([up2, nu]), np.concatenate([dn2, nd])
                phi = np.vstack([phi, np.zeros((len(nu), P))])
                if r + 1 < int(select_rounds):
                    coeff = np.concatenate([coeff, _first_order_amplitudes(HX, up2, dn2, phi, n_old)])
        HX.generate_sparse_ham_upper_triangular(up2, dn2)
        norms = np.linalg.norm(phi, axis=0)
        live = np.flatnonzero(norms > 0.0)
        alpha = np.zeros((P, max_steps))
        beta = np.zeros((P, max_steps))
        ovl = np.zeros((P, max_steps, P))
        steps = np.zeros(P, dtype=np.int64)
        if len(live):
            r = HX.lanczos_tridiagonal(phi[:, live], max_steps, tol)
            alpha[live], beta[live], steps[live] = r["alpha"], r["beta"], r["steps"]
            ovl[np.ix_(live, np.arange(max_steps), live)] = r["overlaps"]
    finally:
        HX.close()
    M, poles, residues = krylov_resolvent(alpha, beta, ovl, steps, norms, e0, z, create)
    return M, poles, residues, len(up2), steps


def greens_function(system, H, up, dn, wts, e0, orbitals, spin, omega, eta, max_steps=100, eps_select=None, select_rounds=1, state=0,
                    tol=1e-12):
    """Removal and addition Green's functions of Psi_0 = wts[:, state] / ||wts[:, state]|| over the list (up, dn) of the chem
    handle H of `system` (time_sym lists: the representatives), E_0 = e0, for the orbitals `orbitals` (library numbering) of
    one spin ("a" / 0 up, "b" / 1 dn), on the grid z = omega + i eta.

    The N-1 / N+1 space is the union of the images; with eps_select it is widened by up to select_rounds heat-bath selection
    rounds on the N-1 / N+1 handle (a round that adds nothing ends the widening).  The first round screens from
    max_j |phi_ij|; the determinants a round adds enter the next one with their first-order amplitudes
    max_j |(H phi_j)_i / (E_j - H_ii)|, E_j the Rayleigh quotient of phi_j.  Each image then starts
    one Lanczos run of at most max_steps steps (tol: lanczos_tridiagonal's invariance test).
    -> dict(G_minus, G_plus: (n_omega, P, P) complex; poles_minus, residues_minus, poles_plus, residues_plus: per orbital, the
    poles (ascending omega) and residues of the diagonal element; n_minus, n_plus: sizes of the N-1 / N+1 spaces;
    steps_minus, steps_plus: Lanczos steps per orbital)."""
    sp = {"a": 0, "b": 1}.get(spin, spin)
    if sp not in (0, 1):
        raise ValueError("greens_function: spin must be 'a' / 0 or 'b' / 1, got %r" % (spin,))
    if not isinstance(system, systems.ChemSystem):
        raise ValueError("greens: the Green's function driver is for chem systems")
    if int(max_steps) < 1:
        raise ValueError("greens_function: max_steps must be >= 1")
    orbitals = [int(p) for p in orbitals]
    z = np.asarray(omega, dtype=np.float64).reshape(-1) + 1j * float(eta)
    out = {}
    for key, create in (("minus", False), ("plus", True)):
        M, poles, res, nx, steps = _sector(system, H, up, dn, wts, int(state), float(e0), orbitals, sp, create, z, int(max_steps),
                                           eps_select, select_rounds, tol)
        # M[w, a, b] = <v_b|R|v_a>: G-_pq = <phi_q|R|phi_p> = M[p, q], G+_pq = <chi_p|R|chi_q> = M[q, p]
        out["G_" + key] = M if not create else np.ascontiguousarray(M.transpose(0, 2, 1))
        out["poles_" + key], out["residues_" + key], out["n_" + key], out["steps_" + key] = poles, res, nx, steps
    return out


def spectral_function(G):
    """A(omega) = -Im G(omega) / pi of a Green's function (n_omega, P, P) (or any array of G values)."""
    return -np.imag(np.asarray(G)) / np.pi
