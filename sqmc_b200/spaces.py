"""Synthetic determinant spaces for benchmarks and large-size tests (SURVEY.md section 8(d), S2/S4/S5).

These are INPUT GENERATORS (host, numpy): they produce determinant lists; nothing here
computes Hamiltonian elements or H.v.  The reference's own way to obtain such lists
(heat-bath selection inside an HCI run) is out of scope of this path.
"""
import itertools

import numpy as np


def _strings(norb, nel):
    """all nel-electron occupation strings of norb orbitals as python ints, ascending."""
    out = [sum(1 << o for o in c) for c in itertools.combinations(range(norb), nel)]
    out.sort()
    return out


def c2_lowest_energy_space(chem, n_dets, target_irrep=1, time_sym=False):
    """The n_dets lowest-diagonal-energy determinants of one spatial-symmetry sector
    (ties at the cut broken by label), returned sorted by label (up, dn).

    chem: systems.ChemSystem (orbitals already in the reference's reordered numbering).
    E_diag(u,d) = Ea(u) + Ea(d) + sum_{i in u, j in d} (ii|jj),
    Ea(s) = sum_i h_ii + sum_{i<j in s} [(ii|jj) - (ij|ji)]   (chemistry.f90:1297-1301,1410-1433,1777-1835).
    The ranking energy is evaluated in numpy (summation order differs from the device
    element routine in the last bits; it only ranks determinants).
    Returns (up, dn) as (n,2) uint64 arrays.
    """
    norb, nup, ndn = chem.norb, chem.nup, chem.ndn
    h, J, K = chem.jk_tables()
    sym = np.asarray(chem.orbital_symmetries, dtype=np.int64) - 1

    def table(nel):
        strs = _strings(norb, nel)
        occ = np.zeros((len(strs), norb), dtype=np.float64)
        for k, s in enumerate(strs):
            for o in range(norb):
                if (s >> o) & 1:
                    occ[k, o] = 1.0
        ea = occ @ h + 0.5 * np.einsum("ki,ij,kj->k", occ, J - K, occ) - 0.5 * occ @ np.diag(J - K)
        irr = np.zeros(len(strs), dtype=np.int64)
        for o in range(norb):
            irr ^= (occ[:, o].astype(np.int64) * sym[o])
        return np.array(strs, dtype=np.uint64), occ, ea, irr

    su, occ_u, ea_u, irr_u = table(nup)
    sd, occ_d, ea_d, irr_d = (su, occ_u, ea_u, irr_u) if ndn == nup else table(ndn)
    tgt = target_irrep - 1
    ups, dns, ens = [], [], []
    for g in range(8):
        iu = np.nonzero(irr_u == g)[0]
        id_ = np.nonzero(irr_d == (g ^ tgt))[0]
        if len(iu) == 0 or len(id_) == 0:
            continue
        E = ea_u[iu][:, None] + ea_d[id_][None, :] + (occ_u[iu] @ J) @ occ_d[id_].T
        U = np.broadcast_to(su[iu][:, None], E.shape)
        D = np.broadcast_to(sd[id_][None, :], E.shape)
        if time_sym:
            keep = U <= D
            ups.append(U[keep]); dns.append(D[keep]); ens.append(E[keep])
        else:
            ups.append(U.ravel()); dns.append(D.ravel()); ens.append(E.ravel())
    up = np.concatenate(ups); dn = np.concatenate(dns); en = np.concatenate(ens)
    total = len(en)
    n_dets = min(int(n_dets), total)
    if n_dets < total:
        part = np.argpartition(en, n_dets - 1)
        cut = en[part[n_dets - 1]]
        below = np.nonzero(en < cut)[0]
        at = np.nonzero(en == cut)[0]
        need = n_dets - len(below)
        if need < len(at):
            order = np.lexsort((dn[at], up[at]))
            at = at[order[:need]]
        sel = np.concatenate([below, at])
    else:
        sel = np.arange(total)
    up, dn = up[sel], dn[sel]
    order = np.lexsort((dn, up))
    up, dn = up[order], dn[order]
    z = np.zeros(len(up), dtype=np.uint64)
    return np.ascontiguousarray(np.stack([up, z], axis=1)), np.ascontiguousarray(np.stack([dn, z], axis=1)), total


def hci_space(H, system, n_dets, eps_schedule=(1e-3, 3e-4, 1e-4, 3e-5, 1e-5, 5e-6, 2e-6, 1e-6, 5e-7, 2e-7, 1e-7), log=None):
    """The determinant space of an HCI run (perform_hci, hci.f90:359-517) grown on the GPU through the library itself --
    heat-bath selection, H build and Davidson per iteration -- with eps_var lowered along `eps_schedule` until the space
    holds n_dets determinants (the last batch of new determinants, sorted by label, is cut to land exactly on n_dets).
    This is the BASELINE.json configs[3] recipe ("eps_var lowered to give ~10^7 determinants").  Under torchrun every
    rank runs the same loop (selection is replicated, build / Davidson are sharded collectives) and obtains identical lists.
    Returns (up, dn, wts, energy); H keeps the matrix of the final space resident."""
    import time
    from .api import dets_to_u64
    up = dets_to_u64([system.hf_up])
    dn = dets_to_u64([system.hf_dn])
    wts = np.ones((1, 1))
    min_h = np.full(1, 9e99)
    energy = None
    for it, eps in enumerate(eps_schedule, 1):
        n_old = len(up)
        t0 = time.perf_counter()
        nu, nd, min_h = H.get_next_det_list(up, dn, np.abs(wts[:, 0]), min_h, eps)
        t_sel = time.perf_counter() - t0
        if len(nu) == 0:
            continue
        if n_old + len(nu) > n_dets:
            nu, nd = nu[:n_dets - n_old], nd[:n_dets - n_old]
        up, dn = np.concatenate([up, nu]), np.concatenate([dn, nd])
        min_h = np.concatenate([min_h, np.full(len(nu), 9e99)])
        t0 = time.perf_counter()
        from . import _lib
        _lib.load().sqmc_b200_alloc_stall_ms(1)
        nnz = H.generate_sparse_ham_upper_triangular(up, dn, ndet_old=n_old)
        t_build = time.perf_counter() - t0
        stall_build = float(_lib.load().sqmc_b200_alloc_stall_ms(1))
        v0 = np.zeros((len(up), 1))
        v0[:n_old, 0] = wts[:, 0]
        t0 = time.perf_counter()
        d = H.davidson_sparse(n_states=1, initial_vector=v0)
        t_dav = time.perf_counter() - t0
        wts, energy = d["evecs"], float(d["evals"][0])
        if log is not None:
            log.append({"iter": it, "eps_var": eps, "n_dets": len(up), "nnz_upper": int(nnz), "energy": energy, "select_s": t_sel, "build_s": t_build,
                        "build_device_ms": H.build_times()["total_ms"], "build_alloc_stall_ms": stall_build,
                        "build_incremental": bool(H.last_build_incremental()),
                        "davidson_s": t_dav, "n_matvec": int(d["n_matvec"])})
        if len(up) >= n_dets:
            break
    return up, dn, wts, energy


def hubbard_momentum_sector(hub, n_dets=None, ktot=(0, 0)):
    """Determinants of one total-momentum sector of the k-space Hubbard model, ranked by
    ascending diagonal energy then label, truncated to n_dets, stored sorted by label
    (the order generate_sparse_ham_hubbardk_upper_triangular's binary search needs, hubbard.f90:9646).
    Strings are (n, 2) uint64 words, so lattices of more than 64 sites (up to 127) are enumerated too."""
    ns = hub.norb
    su = _words(_strings(ns, hub.nup))
    sd = _words(_strings(ns, hub.ndn))
    kx = hub.k_vectors[:, 0].astype(np.int64)
    ky = hub.k_vectors[:, 1].astype(np.int64)

    def props(strs):
        occ = np.stack([(strs[:, o >> 6] >> np.uint64(o & 63)) & np.uint64(1) for o in range(ns)], axis=1).astype(np.int64)
        return (occ @ kx) % (2 * hub.l_x), (occ @ ky) % (2 * hub.l_y), occ.astype(np.float64) @ hub.k_energies

    ux, uy, ue = props(su)
    dx, dy, de = props(sd)
    ups, dns, ens = [], [], []
    for mx in range(0, 2 * hub.l_x, 2):
        for my in range(0, 2 * hub.l_y, 2):
            iu = np.nonzero((ux == mx) & (uy == my))[0]
            id_ = np.nonzero((dx == (ktot[0] - mx) % (2 * hub.l_x)) & (dy == (ktot[1] - my) % (2 * hub.l_y)))[0]
            if len(iu) == 0 or len(id_) == 0:
                continue
            E = ue[iu][:, None] + de[id_][None, :]
            ups.append(np.broadcast_to(iu[:, None], E.shape).ravel())
            dns.append(np.broadcast_to(id_[None, :], E.shape).ravel())
            ens.append(E.ravel())
    up = su[np.concatenate(ups)]; dn = sd[np.concatenate(dns)]; en = np.concatenate(ens)
    total = len(en)
    if n_dets is not None and n_dets < total:
        order = np.lexsort((dn[:, 0], dn[:, 1], up[:, 0], up[:, 1], np.round(en, 12)))[:n_dets]
        up, dn = up[order], dn[order]
    order = np.lexsort((dn[:, 0], dn[:, 1], up[:, 0], up[:, 1]))   # 128-bit label: high word first
    return np.ascontiguousarray(up[order]), np.ascontiguousarray(dn[order]), total


def _words(strs):
    """python ints below 2^128 -> (n, 2) uint64, low word first"""
    return np.array([(s & 0xFFFFFFFFFFFFFFFF, s >> 64) for s in strs], dtype=np.uint64).reshape(-1, 2)


def splitmix_vector(n, seed=12345):
    """x_i = splitmix64(seed, i) mapped to U(-1,1), normalised (SURVEY.md 8(d)); identical for any GPU count."""
    i = np.arange(1, n + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = (np.uint64(seed) + i * np.uint64(0x9E3779B97F4A7C15))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    x = (z >> np.uint64(11)).astype(np.float64) * (2.0 / 9007199254740992.0) - 1.0
    return x / np.linalg.norm(x)
