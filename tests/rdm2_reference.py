"""CPU restatement of the two-particle density matrix, for the tests only (the product never imports it).

It restates the definition, not the GPU algorithm: a_q, a_s, a+_r, a+_p applied in turn to every determinant, the result
looked up in a dictionary, every sign counted from the bits below the orbital acted on.  Time-reversal symmetrised
representatives are expanded as in rdm_reference.
"""
import numpy as np

from rdm_reference import expand_time_sym, u64_to_ints


def _apply(det, k, create):
    """a+_k (create) or a_k on the occupation word det -> (new word, sign), or (None, 0) when the result vanishes"""
    if ((det >> k) & 1) == create:
        return None, 0
    return det ^ (1 << k), (-1 if bin(det & ((1 << k) - 1)).count("1") & 1 else 1)


def two_rdm(up, dn, wts, norb, time_sym=False, z=1):
    """<Psi_k| a+_{p sigma} a+_{r tau} a_{s tau} a_{q sigma} |Psi_k> -> (n_states, 3, norb, norb, norb, norb), [k, b, p, q, r, s],
    b = 0 (alpha alpha), 1 (alpha beta), 2 (beta beta).  Spin orbital p of spin sigma is bit p + sigma*norb of u | d << norb
    (alpha string first); a_q, a_s, a+_r, a+_p are applied in turn to every determinant and the result is looked up."""
    if not isinstance(up, list):
        up, dn = u64_to_ints(up), u64_to_ints(dn)
    w = np.asarray(wts, dtype=np.float64).reshape(len(up), -1)
    if time_sym:
        up, dn, w = expand_time_sym(up, dn, w, z)
    full = [u | (d << norb) for u, d in zip(up, dn)]
    index = {f: i for i, f in enumerate(full)}
    if len(index) != len(full):
        raise ValueError("duplicated determinant")
    g = np.zeros((w.shape[1], 3, norb, norb, norb, norb))
    for j, det in enumerate(full):
        for b, sg, tau in ((0, 0, 0), (1, 0, 1), (2, 1, 1)):
            for q in range(norb):
                d1, s1 = _apply(det, q + sg * norb, 0)
                if d1 is None:
                    continue
                for s in range(norb):
                    d2, s2 = _apply(d1, s + tau * norb, 0)
                    if d2 is None:
                        continue
                    for r in range(norb):
                        d3, s3 = _apply(d2, r + tau * norb, 1)
                        if d3 is None:
                            continue
                        for p in range(norb):
                            d4, s4 = _apply(d3, p + sg * norb, 1)
                            i = index.get(d4) if d4 is not None else None
                            if i is not None:
                                g[:, b, p, q, r, s] += (s1 * s2 * s3 * s4) * w[i] * w[j]
    return g
