"""CPU restatement of the one-particle density matrix, for the tests only (the product never imports it).

It restates the definition, not the GPU algorithm: every determinant, every single excitation in both directions,
the partner looked up in a dictionary, the sign counted from the bits between the two orbitals.  Time-reversal
symmetrised representatives are expanded here on their own: (u,d), u != d -> c/sqrt2 on (u,d) and z c/sqrt2 on (d,u).
"""
import math

import numpy as np


def u64_to_ints(a):
    a = np.asarray(a, dtype=np.uint64).reshape(-1, 2)
    return [int(lo) | (int(hi) << 64) for lo, hi in a]


def expand_time_sym(up, dn, wts, z):
    """representatives -> plain determinants (python ints) and their coefficients (n2, n_states)"""
    w = np.asarray(wts, dtype=np.float64).reshape(len(up), -1)
    ou, od, ow = [], [], []
    r = 1.0 / math.sqrt(2.0)
    for u, d, c in zip(up, dn, w):
        if u == d:
            ou.append(u); od.append(d); ow.append(c)
        else:
            ou += [u, d]; od += [d, u]; ow += [c * r, z * c * r]
    return ou, od, np.array(ow)


def one_rdm(up, dn, wts, norb, time_sym=False, z=1):
    """up, dn: python ints or (n, 2) uint64; wts (n,) or (n, n_states) -> (n_states, 2, norb, norb), [s, sigma, p, q]"""
    if not isinstance(up, list):
        up, dn = u64_to_ints(up), u64_to_ints(dn)
    w = np.asarray(wts, dtype=np.float64).reshape(len(up), -1)
    if time_sym:
        up, dn, w = expand_time_sym(up, dn, w, z)
    index = {(u, d): i for i, (u, d) in enumerate(zip(up, dn))}
    if len(index) != len(up):
        raise ValueError("duplicated determinant")
    g = np.zeros((w.shape[1], 2, norb, norb))
    for i, (u, d) in enumerate(zip(up, dn)):
        c = w[i]
        for sigma in (0, 1):
            a = u if sigma == 0 else d
            for q in range(norb):
                if not (a >> q) & 1:
                    continue
                g[:, sigma, q, q] += c * c
                for p in range(norb):
                    if (a >> p) & 1:
                        continue
                    a2 = a ^ (1 << q) ^ (1 << p)
                    j = index.get((a2, d) if sigma == 0 else (u, a2))
                    if j is None:
                        continue
                    lo, hi = min(p, q), max(p, q)
                    between = bin(a & (((1 << hi) - 1) ^ ((1 << (lo + 1)) - 1))).count("1")
                    g[:, sigma, p, q] += (-1.0) ** between * w[j] * c
    return g
