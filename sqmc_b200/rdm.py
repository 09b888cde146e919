"""Host quantities from the density matrices of SparseHamiltonian.one_rdm / two_rdm: <S^2> and the energy identity.

Both read the matrices in the library's numbering (the bits of the determinant words) and apply no normalisation: a
wavefunction of norm ||Psi||^2 gives ||Psi||^2 times the expectation value.
"""
import numpy as np


def spin_squared(rdm2, nup, ndn, norm2=1.0):
    """<Psi|S^2|Psi> = [S_z(S_z+1) + N_beta] ||Psi||^2 - sum_pq Gamma^{ab}_{pq,qp}, S_z = (N_alpha - N_beta)/2.

    rdm2: [b, p, q, r, s] of one state, or [k, b, p, q, r, s] (then norm2 may be one value per state)."""
    g = np.asarray(rdm2)
    sz = 0.5 * (nup - ndn)
    return (sz * (sz + 1.0) + ndn) * np.asarray(norm2, dtype=np.float64) - np.einsum("...pqqp->...", g[..., 1, :, :, :, :])


def integrals_library_order(chem_system):
    """(h, eri, enuc) of the library's chem Hamiltonian as it evaluates it: h[p,q], eri[p,q,r,s] = (pq|rs) and the core energy
    read from system.integrals through _index in the reordered numbering (so after the integral filter applied on reading)."""
    norb = chem_system.norb
    n1 = norb + 1
    c2 = np.asarray(chem_system._c2, dtype=np.int64)
    pq = c2[:norb, :norb]
    core = c2[n1 - 1, n1 - 1]

    def index(a, b):
        hi, lo = np.maximum(a, b), np.minimum(a, b)
        return hi * (hi - 1) // 2 + lo

    ints = np.asarray(chem_system.integrals, dtype=np.float64)
    h = ints[index(pq, core) - 1]
    eri = ints[index(pq[:, :, None, None], pq[None, None, :, :]) - 1]
    return h, eri, float(ints[index(core, core) - 1])   # the core energy the library puts on the diagonal


def rdm_energy(chem_system, rdm1, rdm2):
    """enuc ||Psi||^2 + sum_pq h_pq gamma_pq + 1/2 sum (pq|rs) Gamma_pq,rs of one state, spins summed (the alpha-beta block
    counts twice: beta-alpha is the same block).  rdm1: [sigma, p, q] from one_rdm; rdm2: [b, p, q, r, s] from two_rdm.
    ||Psi||^2 is the trace of gamma over the electron count."""
    h, eri, enuc = integrals_library_order(chem_system)
    g1 = np.asarray(rdm1)
    g2 = np.asarray(rdm2)
    norm2 = (np.trace(g1[0]) + np.trace(g1[1])) / (chem_system.nup + chem_system.ndn)
    e1 = float(np.sum(h * (g1[0] + g1[1])))
    e2 = 0.5 * float(np.sum(eri * (g2[0] + 2.0 * g2[1] + g2[2])))
    return enuc * norm2 + e1 + e2
