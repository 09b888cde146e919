"""Host checks of the 1-RDM reference, the FCIDUMP writer and the orbital rotation (no GPU)."""
import itertools
import os

import numpy as np
import pytest

from conftest import C2_FCIDUMP, C2_ORBSYM
from rdm_reference import one_rdm
from sqmc_b200 import formats, natorb, systems


def _random_list(rng, norb, nup, ndn, n, time_sym=False):
    seen, up, dn = set(), [], []
    while len(up) < n:
        u = sum(1 << int(k) for k in rng.choice(norb, nup, replace=False))
        d = sum(1 << int(k) for k in rng.choice(norb, ndn, replace=False))
        if time_sym and d < u:
            u, d = d, u
        if (u, d) in seen or (time_sym and (d, u) in seen):
            continue
        seen.add((u, d)); up.append(u); dn.append(d)
    if time_sym:  # a few closed-shell representatives
        for k in range(5):
            u = sum(1 << int(x) for x in rng.choice(norb, nup, replace=False))
            if (u, u) not in seen:
                seen.add((u, u)); up.append(u); dn.append(u)
    return up, dn


def _brute_force(up, dn, wts, norb, time_sym=False, z=1):
    """<Psi| a+_{p sigma} a_{q sigma} |Psi> by applying the operators to occupation lists of spin orbitals
    (alpha orbital k = k, beta orbital k = norb + k, creation operators in ascending order)"""
    r = 1.0 / np.sqrt(2.0)
    psi = {}
    for u, d, c in zip(up, dn, wts):
        occ = lambda a, b: tuple([k for k in range(norb) if (a >> k) & 1] + [norb + k for k in range(norb) if (b >> k) & 1])
        if time_sym and u != d:
            psi[occ(u, d)] = c * r
            psi[occ(d, u)] = z * c * r
        else:
            psi[occ(u, d)] = c

    def annihilate(det, q):
        if q not in det:
            return None, 0
        k = det.index(q)
        return det[:k] + det[k + 1:], (-1) ** k

    def create(det, p):
        if p in det:
            return None, 0
        k = sum(1 for x in det if x < p)
        return det[:k] + (p,) + det[k:], (-1) ** k

    g = np.zeros((2, norb, norb))
    for det, c in psi.items():
        for sigma in (0, 1):
            for q in range(norb):
                d1, s1 = annihilate(det, sigma * norb + q)
                if d1 is None:
                    continue
                for p in range(norb):
                    d2, s2 = create(d1, sigma * norb + p)
                    if d2 is not None and d2 in psi:
                        g[sigma, p, q] += psi[d2] * s1 * s2 * c
    return g


@pytest.mark.parametrize("nup,ndn,time_sym,z", [(3, 3, False, 1), (4, 2, False, 1), (3, 3, True, 1), (3, 3, True, -1)])
def test_reference_rdm_matches_second_quantisation(nup, ndn, time_sym, z):
    rng = np.random.default_rng(7 + nup + 10 * ndn + 100 * time_sym + z)
    norb = 12
    up, dn = _random_list(rng, norb, nup, ndn, 300, time_sym=time_sym)
    w = rng.standard_normal(len(up))
    got = one_rdm(up, dn, w, norb, time_sym=time_sym, z=z)[0]
    ref = _brute_force(up, dn, w, norb, time_sym=time_sym, z=z)
    assert np.max(np.abs(got - ref)) <= 1e-12
    assert np.max(np.abs(got - ref.transpose(0, 2, 1))) <= 1e-12


def test_fcidump_identity_rotation_round_trip(tmp_path):
    _, h, _, _ = natorb.dense_integrals(C2_FCIDUMP)
    out = str(tmp_path / "FCIDUMP")
    natorb.rotate_fcidump(C2_FCIDUMP, np.eye(h.shape[0]), C2_ORBSYM, out)
    a = systems.ChemSystem(C2_FCIDUMP)
    b = systems.ChemSystem(out)
    assert np.array_equal(a.integrals, b.integrals)
    assert a.enuc == b.enuc
    assert np.array_equal(a.orb_order, b.orb_order)
    assert list(b.orbital_symmetries_fcidump) == C2_ORBSYM


def write_toy_fcidump(path, norb=10, nelec=4):
    """the first `norb` C2 orbitals with nelec electrons (MS2 = 0), written by the FCIDUMP writer"""
    _, h, eri, ecore = natorb.dense_integrals(C2_FCIDUMP)
    formats.write_fcidump(path, h[:norb, :norb], eri[:norb, :norb, :norb, :norb], ecore, nelec, orbsym=C2_ORBSYM[:norb])


def fci_dets(norb, nup, ndn):
    ups = [sum(1 << k for k in c) for c in itertools.combinations(range(norb), nup)]
    dns = [sum(1 << k for k in c) for c in itertools.combinations(range(norb), ndn)]
    return [u for u in ups for _ in dns], [d for _ in ups for d in dns]


def random_rotation_within_irreps(rng, orbsym):
    orbsym = np.asarray(orbsym)
    C = np.zeros((len(orbsym), len(orbsym)))
    for s in set(orbsym.tolist()):
        idx = np.flatnonzero(orbsym == s)
        q, _ = np.linalg.qr(rng.standard_normal((len(idx), len(idx))))
        C[np.ix_(idx, idx)] = q
    return C


def _oracle_fci(oracle, path, norb, orbsym):
    S = oracle.System.chem(path, norb, 4, 2, orbsym)
    up, dn = fci_dets(norb, 2, 2)
    cnt, idx, val = S.build_upper(oracle.dets_to_u64(up), oracle.dets_to_u64(dn))
    Hm = oracle.upper_to_scipy(cnt, idx, val).toarray()
    return np.linalg.eigvalsh(Hm)


def test_fci_energy_invariant_under_rotation_within_irreps(tmp_path, oracle):
    toy = str(tmp_path / "FCIDUMP_toy")
    write_toy_fcidump(toy)
    orbsym = C2_ORBSYM[:10]
    e0 = _oracle_fci(oracle, toy, 10, orbsym)
    assert len(e0) == 2025
    C = random_rotation_within_irreps(np.random.default_rng(3), orbsym)
    rot = str(tmp_path / "FCIDUMP_rot")
    natorb.rotate_fcidump(toy, C, orbsym, rot)
    e1 = _oracle_fci(oracle, rot, 10, orbsym)
    assert abs(e1[0] - e0[0]) <= 1e-10


def test_rotate_rejects_large_norb(tmp_path):
    p = str(tmp_path / "FCIDUMP_big")
    with open(p, "w") as f:
        f.write(" &FCI NORB=65,NELEC=2,MS2=0,\n &END\n0.0 0 0 0 0\n")
    with pytest.raises(ValueError, match="limited to 64"):
        natorb.rotate_fcidump(p, np.eye(65), [1] * 65, str(tmp_path / "out"))


def test_natural_orbitals_keep_irreps_and_order():
    sysm = systems.ChemSystem(C2_FCIDUMP)
    norb = sysm.norb
    rng = np.random.default_rng(5)
    # a gamma that is block diagonal over the irreps in FCIDUMP numbering, mapped to the library's numbering
    C = random_rotation_within_irreps(rng, C2_ORBSYM)
    occ = np.sort(rng.uniform(0, 1, norb))[::-1]
    gf = C @ np.diag(occ) @ C.T
    o = sysm.orb_order[:norb] - 1
    g = gf[np.ix_(o, o)]
    res = natorb.natural_orbitals(sysm, np.stack([g, g]))
    assert np.allclose(res["occupations"], 2 * occ, atol=1e-12)
    assert np.all(np.diff(res["occupations"]) <= 0)
    Cn = res["coeffs"]
    assert np.allclose(Cn.T @ Cn, np.eye(norb), atol=1e-12)
    for k in range(norb):  # every natural orbital lives in its irrep
        assert np.all(np.abs(Cn[np.asarray(C2_ORBSYM) != res["irreps"][k], k]) == 0)
    assert sorted(res["irreps"].tolist()) == sorted(C2_ORBSYM)
