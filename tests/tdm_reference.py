"""CPU restatement of the one- and two-particle transition density matrices, for the tests only (the product never imports it).

It restates the definitions <bra| a+_p a_q |ket> and <bra| a+_p a+_r a_s a_q |ket> from second quantisation, as
rdm2_reference does for one state: the operators are applied in turn to every ket determinant, the result is looked up in a
dictionary, and every sign is counted from the bits below the orbital acted on (alpha string first).  Time-reversal
symmetrised representatives of both vectors are expanded with the same factors, as in rdm_reference.
"""
import numpy as np

from rdm2_reference import _apply
from rdm_reference import expand_time_sym, u64_to_ints


def _plain(up, dn, bra, ket, norb, time_sym, z):
    """-> spin-orbital words (alpha bits, then beta bits from norb), their index, bra (n2, n_pairs), ket (n2, n_pairs)"""
    if not isinstance(up, list):
        up, dn = u64_to_ints(up), u64_to_ints(dn)
    a = np.asarray(bra, dtype=np.float64).reshape(len(up), -1)
    b = np.asarray(ket, dtype=np.float64).reshape(len(up), -1)
    if a.shape != b.shape:
        raise ValueError("bra and ket differ in shape")
    k = a.shape[1]
    w = np.concatenate([a, b], axis=1)
    if time_sym:
        up, dn, w = expand_time_sym(up, dn, w, z)
    full = [u | (d << norb) for u, d in zip(up, dn)]
    index = {f: i for i, f in enumerate(full)}
    if len(index) != len(full):
        raise ValueError("duplicated determinant")
    return full, index, w[:, :k], w[:, k:]


def transition_one_rdm(up, dn, bra, ket, norb, time_sym=False, z=1):
    """<bra_k| a+_{p sigma} a_{q sigma} |ket_k> -> (n_pairs, 2, norb, norb), [k, sigma, p, q]"""
    full, index, a, b = _plain(up, dn, bra, ket, norb, time_sym, z)
    g = np.zeros((a.shape[1], 2, norb, norb))
    for j, det in enumerate(full):
        for sigma in (0, 1):
            for q in range(norb):
                d1, s1 = _apply(det, q + sigma * norb, 0)
                if d1 is None:
                    continue
                for p in range(norb):
                    d2, s2 = _apply(d1, p + sigma * norb, 1)
                    i = index.get(d2) if d2 is not None else None
                    if i is not None:
                        g[:, sigma, p, q] += (s1 * s2) * a[i] * b[j]
    return g


def transition_two_rdm(up, dn, bra, ket, norb, time_sym=False, z=1):
    """<bra_k| a+_{p sigma} a+_{r tau} a_{s tau} a_{q sigma} |ket_k> -> (n_pairs, 3, norb, norb, norb, norb), [k, b, p, q, r, s],
    b = 0 (alpha alpha), 1 (alpha beta), 2 (beta beta)"""
    full, index, a, b = _plain(up, dn, bra, ket, norb, time_sym, z)
    g = np.zeros((a.shape[1], 3, norb, norb, norb, norb))
    for j, det in enumerate(full):
        for blk, sg, tau in ((0, 0, 0), (1, 0, 1), (2, 1, 1)):
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
                                g[:, blk, p, q, r, s] += (s1 * s2 * s3 * s4) * a[i] * b[j]
    return g
