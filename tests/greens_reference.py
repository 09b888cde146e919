"""numpy restatements for the Green's function tests (the product never imports this file).

ladder: the images a_{p sigma}|Psi> / a+_{p sigma}|Psi> over python-int determinants with the library's phase convention
(alpha string first, ascending creators); fock_ladder: the same from occupation lists of spin orbitals alpha_0 .. alpha_{n-1},
beta_0 .. beta_{n-1}; lanczos: Lanczos with full reorthogonalisation as lanczos_tridiagonal states it; sum_over_states:
<v_b| R(z) |v_a> from a dense diagonalisation.
"""
import numpy as np

from rdm_reference import expand_time_sym, u64_to_ints


def _popc(x):
    return bin(x).count("1")


def ladder(up, dn, wts, orbs, spin, create, time_sym=False, z=1, state=0):
    """-> (up', dn' python ints sorted by (up, dn), phi (m, len(orbs)))"""
    if not isinstance(up, list):
        up, dn = u64_to_ints(up), u64_to_ints(dn)
    w = np.asarray(wts, dtype=np.float64).reshape(len(up), -1)[:, state]
    if time_sym:
        up, dn, w = expand_time_sym(up, dn, w, z)
        w = np.asarray(w).reshape(-1)
    images = {}
    for u, d, c in zip(up, dn, w):
        for j, p in enumerate(orbs):
            x = d if spin else u
            if bool((x >> p) & 1) == bool(create):
                continue
            par = _popc(x & ((1 << p) - 1)) + (_popc(u) if spin else 0)
            x ^= 1 << p
            key = (u, x) if spin else (x, d)
            images.setdefault(key, {})[j] = -c if par & 1 else c
    keys = sorted(images)
    phi = np.zeros((len(keys), len(orbs)))
    for i, k in enumerate(keys):
        for j, v in images[k].items():
            phi[i, j] = v
    return [k[0] for k in keys], [k[1] for k in keys], phi


def fock_ladder(up, dn, wts, norb, orbs, spin, create, time_sym=False, z=1):
    """the images as dict {(up, dn): [coefficient per orbital]} from second quantisation on sorted occupation tuples"""
    r = 1.0 / np.sqrt(2.0)
    psi = {}
    occ = lambda a, b: tuple([k for k in range(norb) if (a >> k) & 1] + [norb + k for k in range(norb) if (b >> k) & 1])
    for u, d, c in zip(up, dn, wts):
        if time_sym and u != d:
            psi[occ(u, d)] = c * r
            psi[occ(d, u)] = z * c * r
        else:
            psi[occ(u, d)] = c
    out = {}
    for det, c in psi.items():
        for j, p in enumerate(orbs):
            so = spin * norb + p
            if create:
                if so in det:
                    continue
                k = sum(1 for x in det if x < so)
                new = det[:k] + (so,) + det[k:]
            else:
                if so not in det:
                    continue
                k = det.index(so)
                new = det[:k] + det[k + 1:]
            u = sum(1 << x for x in new if x < norb)
            d = sum(1 << (x - norb) for x in new if x >= norb)
            out.setdefault((u, d), [0.0] * len(orbs))[j] += (-1) ** k * c
    return out


def lanczos(H, v0, max_steps, tol):
    """H dense or scipy sparse; -> (alpha, beta, Q (n, steps)) with a second classical Gram-Schmidt pass per step"""
    q = v0 / np.linalg.norm(v0)
    Q = [q]
    alpha, beta = [], []
    for j in range(min(max_steps, len(v0))):
        w = H @ Q[j]
        a = Q[j] @ w
        w = w - a * Q[j] - (beta[-1] * Q[j - 1] if j > 0 else 0.0)
        Qm = np.array(Q).T
        w = w - Qm @ (Qm.T @ w)
        b = np.linalg.norm(w)
        alpha.append(a)
        beta.append(b)
        if b < tol * np.max(np.abs(alpha)) or b == 0.0 or j + 1 == max_steps:
            break
        Q.append(w / b)
    return np.array(alpha), np.array(beta), np.array(Q).T


def sum_over_states(Hd, V, e0, z, addition):
    """M[w, a, b] = <v_b| R(z_w) |v_a>, R = (z + H - E_0)^-1 or (z - H + E_0)^-1, V (n, P) the vectors v_a"""
    E, X = np.linalg.eigh(Hd)
    om = E - e0 if addition else e0 - E
    Y = X.T @ V                                            # Y[n, a] = <n|v_a>
    z = np.asarray(z).reshape(-1)
    f = 1.0 / (z[:, None] - om[None, :])
    return np.einsum("wn,na,nb->wab", f, Y, Y)
