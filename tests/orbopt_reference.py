"""numpy restatement of the orbital gradient and Hessian, for the tests only (the product never imports it).

Helgaker, Jorgensen, Olsen, Molecular Electronic-Structure Theory, 10.8.1, real orbitals; D and d are the spin-summed one- and
two-particle density matrices in chemists' order, d_pqrs = sum_st <a+_ps a+_rt a_st a_qs>.
"""
import numpy as np
from scipy.linalg import expm


def densities(rdm1, rdm2, norm2, state_weights):
    """one_rdm (n_states, 2, n, n) and two_rdm (n_states, 3, n, n, n, n) -> (D, d): spins summed, state k divided by
    norm2[k] = ||Psi_k||^2 and weighted with state_weights[k]"""
    w = np.asarray(state_weights, dtype=np.float64) / np.asarray(norm2, dtype=np.float64)
    D, d = 0.0, 0.0
    for k in range(len(w)):
        g1, g2 = rdm1[k], rdm2[k]
        D = D + w[k] * (g1[0] + g1[1])
        d = d + w[k] * (g2[0] + g2[2] + g2[1] + g2[1].transpose(2, 3, 0, 1))
    return D, d


def energy(h, g, ecore, D, d):
    return ecore + float(np.sum(h * D)) + 0.5 * float(np.sum(g * d))


def orbital_derivatives_reference(h, g, D, d):
    """-> dict(fock F_pq = sum_m D_pm h_qm + sum_mnt d_pmnt g_qmnt, gradient 2 (F - F^T),
    hessian E2_pq,rs = (1 - P_pq)(1 - P_rs)[2 D_pr h_qs - (F_pr + F_rp) delta_qs + 2 Y_pqrs],
    Y_pqrs = sum_mn [(d_pmrn + d_pmnr) g_qmsn + d_prmn g_qsmn])"""
    F = np.einsum("pm,qm->pq", D, h) + np.einsum("pmnt,qmnt->pq", d, g, optimize=True)
    Y = (np.einsum("pmrn,qmsn->pqrs", d + d.transpose(0, 1, 3, 2), g, optimize=True)
         + np.einsum("prmn,qsmn->pqrs", d, g, optimize=True))
    f = 2.0 * np.einsum("pr,qs->pqrs", D, h) - np.einsum("pr,qs->pqrs", F + F.T, np.eye(len(h))) + 2.0 * Y
    E2 = f - f.transpose(1, 0, 2, 3) - f.transpose(0, 1, 3, 2) + f.transpose(1, 0, 3, 2)
    return dict(fock=F, gradient=2.0 * (F - F.T), hessian=E2)


def rotation(kappa):
    """U = expm(-kappa) for the antisymmetric (n, n) matrix kappa[p,q] = k_pq = -kappa[q,p]: the sign for which the gradient
    with respect to k_pq (p > q) is 2 (F_pq - F_qp),"""
    return expm(-np.asarray(kappa, dtype=np.float64))


def rotated_energy(h, g, ecore, D, d, kappa):
    """E(kappa) with h' = U^T h U and (pq|rs)' = sum U_ap U_bq U_cr U_ds (ab|cd) (rotate_fcidump's rule, C = U), U = expm(-kappa)"""
    U = rotation(kappa)
    h2 = U.T @ h @ U
    g2 = g
    for _ in range(4):
        g2 = np.tensordot(g2, U, axes=([0], [0]))
    return energy(h2, g2, ecore, D, d)
