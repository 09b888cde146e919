"""numpy restatement of the CI-orbital coupled (one-step) Newton system, for the tests only (the product never imports it).

E(kappa, c) = sum_k w_k <c_k| H(U) |c_k> / ||c_k||^2,  U = expm(-kappa) with rotate_fcidump's rule (orbopt_reference.rotation).
At kappa = 0 and orthonormal c_k, for directions (x over the rotations, y_k orthogonal to every c_j; P = 1 - sum_j |c_j><c_j|):
  oo  the orbital Hessian E2 of orbital_derivatives
  co  (x -> y): 2 w_k P H^x c_k           H^x = d/dt H(expm(-t x)) at t = 0: the one-index transformed integrals
  oc  (y -> x): d/dt gradient(c + t y) = sum_k 2 w_k <y_k| H^{E_pq - E_qp} |c_k>
  cc  (y -> y): 2 w_k P (H - E_k) y_k
Determinants are plain (u, d) python ints; spin orbitals alpha first, as the library's signs.
"""
import numpy as np

from orbopt_reference import densities, orbital_derivatives_reference, rotation
from rdm2_reference import two_rdm
from rdm_reference import one_rdm


def one_index_transform(h, g, kappa):
    """(h^k, g^k) = d/dt at t = 0 of the integrals rotated by U = expm(-t kappa): h^k = kappa h - h kappa,
    g^k_pqrs = sum_m (k_pm g_mqrs + k_qm g_pmrs + k_rm g_pqms + k_sm g_pqrm)"""
    k = np.asarray(kappa, dtype=np.float64)
    hk = k @ h - h @ k
    gk = (np.einsum("pm,mqrs->pqrs", k, g) + np.einsum("qm,pmrs->pqrs", k, g) + np.einsum("rm,pqms->pqrs", k, g)
          + np.einsum("sm,pqrm->pqrs", k, g))
    return hk, gk


def _sign(word, ops):
    """<result| ops |word> for ops [(spin orbital, create?)] applied right to left -> (result, sign) or (None, 0)"""
    sign = 1
    for so, cr in reversed(ops):
        if bool((word >> so) & 1) == cr:
            return None, 0
        if bin(word & ((1 << so) - 1)).count("1") & 1:
            sign = -sign
        word ^= 1 << so
    return word, sign


class DenseH:
    """<i| H |j> over a fixed list of plain determinants for any integrals h, g = (pq|rs) and core energy: every connected pair
    of the list is classified once (Slater-Condon), so building the matrix for new integrals is a few array operations."""

    def __init__(self, up, dn, norb):
        self.n, self.norb = len(up), norb
        self.occ = np.array([[(u >> p) & 1 for p in range(norb)] + [(d >> p) & 1 for p in range(norb)] for u, d in zip(up, dn)], dtype=float)
        words = [int(u) | int(d) << norb for u, d in zip(up, dn)]
        bits = lambda x: [k for k in range(2 * norb) if (x >> k) & 1]
        s1, d2 = [], []
        for j, wj in enumerate(words):
            for i, wi in enumerate(words):
                x = wi ^ wj
                nx = bin(x).count("1")
                if i == j or nx > 4 or bin(x & wi).count("1") != bin(x & wj).count("1"):
                    continue
                cre, ann = bits(x & wi), bits(x & wj)   # created in i, annihilated from j
                if [c < norb for c in cre] != [a < norb for a in ann]:
                    continue   # spin not conserved
                if nx == 2:
                    p, q = cre[0], ann[0]
                    _, sg = _sign(wj, [(p, True), (q, False)])
                    spin = q // norb
                    same, opp = np.zeros(norb), np.zeros(norb)
                    for r in bits(wj):
                        if r != q:
                            (same if r // norb == spin else opp)[r % norb] = 1.0
                    s1.append((i, j, p % norb, q % norb, sg, same, opp))
                else:   # cre, ann ascending: an opposite-spin pair is (alpha, beta) on both sides
                    p, r = cre
                    q, s = ann
                    _, sg = _sign(wj, [(p, True), (r, True), (s, False), (q, False)])
                    d2.append((i, j, p % norb, q % norb, r % norb, s % norb, sg, (p < norb) == (r < norb)))
        self.s1 = s1
        self.d2 = d2

    def __call__(self, h, g, ecore=0.0):
        n, no = self.n, self.norb
        H = np.zeros((n, n))
        oa, ob = self.occ[:, :no], self.occ[:, no:]
        J = np.einsum("pprr->pr", g)
        K = np.einsum("prrp->pr", g)
        diag = (oa + ob) @ np.diag(h) + ecore
        diag += 0.5 * (np.einsum("ip,pr,ir->i", oa, J - K, oa) + np.einsum("ip,pr,ir->i", ob, J - K, ob)) + np.einsum("ip,pr,ir->i", oa, J, ob)
        H[np.arange(n), np.arange(n)] = diag
        for i, j, p, q, sg, same, opp in self.s1:
            H[i, j] += sg * (h[p, q] + (g[p, q].diagonal() - g[p, :, :, q].diagonal()) @ same + g[p, q].diagonal() @ opp)
        for i, j, p, q, r, s, sg, same_spin in self.d2:
            H[i, j] += sg * (g[p, q, r, s] - (g[p, s, r, q] if same_spin else 0.0))
        return H


def rotated_integrals(h, g, kappa):
    """h' = U^T h U and (pq|rs)' = sum U_ap U_bq U_cr U_ds (ab|cd), U = expm(-kappa)"""
    U = rotation(kappa)
    g2 = g
    for _ in range(4):
        g2 = np.tensordot(g2, U, axes=([0], [0]))
    return U.T @ h @ U, g2


def antisym(pairs, x, norb):
    K = np.zeros((norb, norb))
    for (p, q), v in zip(pairs, x):
        K[p, q], K[q, p] = v, -v
    return K


def projector(C):
    return np.eye(len(C)) - C @ C.T


def transition_response(h, g, up, dn, C, dC, w, norb):
    """d/dt of the orbital gradient 2 (F - F^T) at C + t dC, from symmetrised transition densities
    T(a, b) = [Gamma(a + b) - Gamma(a - b)] / 4 with the factor 2 w_k / ||c_k||^2 and dC made orthogonal to C per state"""
    D, d = 0.0, 0.0
    for k in range(C.shape[1]):
        a = C[:, k]
        b = dC[:, k] - (a @ dC[:, k]) / (a @ a) * a
        g1p, g1m = one_rdm(up, dn, a + b, norb)[0], one_rdm(up, dn, a - b, norb)[0]
        g2p, g2m = two_rdm(up, dn, a + b, norb)[0], two_rdm(up, dn, a - b, norb)[0]
        Dk, dk = densities([(g1p - g1m) / 4.0], [(g2p - g2m) / 4.0], [a @ a], [2.0 * w[k]])
        D, d = D + Dk, d + dk
    return orbital_derivatives_reference(h, g, D, d)["gradient"]


def coupled_hessian_vector(dense, h, g, ecore, C, w, E2red, pairs, x, Y):
    """the joint Hessian-vector product at orthonormal C (n x S) over the list of `dense` (a DenseH), E2red the orbital Hessian
    over pairs; (x over pairs, Y n x S orthogonal to C) -> (orbital part, CI part)"""
    norb = len(h)
    Hd = dense(h, g, ecore)
    P = projector(C)
    E = np.einsum("ik,ij,jk->k", C, Hd, C)
    Hx = dense(*one_index_transform(h, g, antisym(pairs, x, norb)))
    rc = np.zeros_like(Y)
    for k in range(C.shape[1]):
        rc[:, k] = 2.0 * w[k] * P @ (Hx @ C[:, k] + (Hd - E[k] * np.eye(len(Hd))) @ Y[:, k])
    resp = np.zeros(len(pairs))
    for t, (p, q) in enumerate(pairs):
        Hpq = dense(*one_index_transform(h, g, antisym([(p, q)], [1.0], norb)))
        resp[t] = sum(2.0 * w[k] * Y[:, k] @ Hpq @ C[:, k] for k in range(C.shape[1]))
    return E2red @ x + resp, rc
