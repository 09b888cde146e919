"""Natural orbitals of a variational wavefunction and the FCIDUMP rotated into them (host-side numpy).

The usual next step after an HCI run: the one-particle density matrix (SparseHamiltonian.one_rdm, computed on the GPU)
is diagonalised, and HCI is run again in the natural-orbital basis, where it converges with fewer determinants.
"""
import numpy as np

from . import formats, systems

MAX_DENSE_NORB = 64  # dense (pq|rs) holds norb^4 doubles: 134 MB at 64 orbitals


def natural_orbitals(system, rdm, state_weights=None):
    """Natural orbitals from one_rdm's output (n_states, 2, norb, norb) or (2, norb, norb).

    The two spins are summed and the states averaged (equal weights unless state_weights is given).
    chem: gamma is mapped from the library's reordered orbitals to FCIDUMP numbering (system.orb_order) and diagonalised
    block by block over the FCIDUMP irreps, so every natural orbital keeps a point-group label (the selection and the HF
    determinant's symmetry rely on it).  -> dict(occupations (descending), coeffs (norb, norb): column k = natural orbital k
    in FCIDUMP orbitals, irreps).  Equal occupations are ordered by irrep, then by position inside the irrep block; each
    column's largest component is made positive.
    heg / hubbardk: every determinant of a list has the same total momentum, so gamma is diagonal and its diagonal is the
    momentum distribution n(k) over the library's orbitals.  Nothing is rotated: -> dict(occupations = n(k) in orbital order,
    coeffs = identity, irreps = None)."""
    g = np.asarray(rdm, dtype=np.float64)
    if g.ndim == 3:
        g = g[None]
    ns, norb = g.shape[0], g.shape[-1]
    w = np.full(ns, 1.0 / ns) if state_weights is None else np.asarray(state_weights, dtype=np.float64) / np.sum(state_weights)
    gamma = np.tensordot(w, g.sum(axis=1), axes=1)
    if not isinstance(system, systems.ChemSystem):
        return dict(occupations=np.diag(gamma).copy(), coeffs=np.eye(norb), irreps=None)
    o = np.asarray(system.orb_order[:norb]) - 1          # library orbital p is FCIDUMP orbital o[p]
    gf = np.zeros_like(gamma)
    gf[np.ix_(o, o)] = gamma
    sym = np.asarray(system.orbital_symmetries_fcidump)
    occ, irr, pos = [], [], []
    cols = []
    for s in sorted(set(sym.tolist())):
        idx = np.flatnonzero(sym == s)
        ev, vec = np.linalg.eigh(gf[np.ix_(idx, idx)])
        for k in range(len(idx)):
            c = np.zeros(norb)
            c[idx] = vec[:, k]
            if c[np.argmax(np.abs(c))] < 0:
                c = -c
            occ.append(ev[k]); irr.append(s); pos.append(k); cols.append(c)
    order = np.lexsort((np.array(pos), np.array(irr), -np.array(occ)))
    return dict(occupations=np.array(occ)[order], coeffs=np.array(cols).T[:, order].copy(), irreps=np.array(irr, dtype=np.int32)[order])


def dense_integrals(path):
    """FCIDUMP -> (header, h (norb, norb), eri (norb,)*4 with the 8-fold symmetry filled in, core energy)."""
    header, body = systems._read_fcidump(path)
    norb = int(header["NORB"])
    if norb > MAX_DENSE_NORB:
        raise ValueError("FCIDUMP has %d orbitals: dense (pq|rs) is limited to %d" % (norb, MAX_DENSE_NORB))
    h = np.zeros((norb, norb))
    eri = np.zeros((norb,) * 4)
    ecore = 0.0
    for v, p, q, r, s in body:
        if p == 0:
            ecore = v
        elif r == 0:
            h[p - 1, q - 1] = h[q - 1, p - 1] = v
        else:
            p, q, r, s = p - 1, q - 1, r - 1, s - 1
            for a, b, c, d in ((p, q, r, s), (q, p, r, s), (p, q, s, r), (q, p, s, r)):
                eri[a, b, c, d] = eri[c, d, a, b] = v
    return header, h, eri, ecore


def rotate_fcidump(src_path, coeffs, orbsym, out_path):
    """Write the FCIDUMP of src_path in the orbitals coeffs (column k = new orbital k in the old orbitals):
    h' = C^T h C, (pq|rs)' by four successive contractions (O(norb^5)), the core energy unchanged; NORB, NELEC, MS2 and ISYM
    are kept and ORBSYM becomes orbsym.  Entries with |v| <= 1e-12 are not written (a reader may drop more: ChemSystem
    keeps only |v| > 1e-9)."""
    header, h, eri, ecore = dense_integrals(src_path)
    C = np.asarray(coeffs, dtype=np.float64)
    if C.shape != h.shape:
        raise ValueError("rotate_fcidump: coeffs must be (norb, norb) = %s" % (h.shape,))
    h2 = C.T @ h @ C
    for _ in range(4):          # contracts the leading index each time; the new index goes last
        eri = np.tensordot(eri, C, axes=([0], [0]))
    formats.write_fcidump(out_path, h2, eri, ecore, int(header["NELEC"]), ms2=int(header.get("MS2", 0)), orbsym=orbsym,
                          isym=int(header.get("ISYM", 1)))
