"""Host checks of the 2-RDM reference (tests/rdm2_reference.two_rdm) and of sqmc_b200.rdm (no GPU)."""
import numpy as np
import pytest

from rdm2_reference import two_rdm
from rdm_reference import one_rdm
from sqmc_b200 import rdm, systems
from test_natorb_host import _random_list, fci_dets, write_toy_fcidump


def _brute_force(up, dn, wts, norb, time_sym=False, z=1):
    """Gamma by second quantisation on sorted tuples of spin orbitals (alpha orbital k = k, beta orbital k = norb + k)"""
    r = 1.0 / np.sqrt(2.0)
    psi = {}
    occ = lambda a, b: tuple([k for k in range(norb) if (a >> k) & 1] + [norb + k for k in range(norb) if (b >> k) & 1])
    for u, d, c in zip(up, dn, wts):
        if time_sym and u != d:
            psi[occ(u, d)] = c * r
            psi[occ(d, u)] = z * c * r
        else:
            psi[occ(u, d)] = c

    def annihilate(det, q):
        if det is None or q not in det:
            return None, 0
        k = det.index(q)
        return det[:k] + det[k + 1:], (-1) ** k

    def create(det, p):
        if det is None or p in det:
            return None, 0
        k = sum(1 for x in det if x < p)
        return det[:k] + (p,) + det[k:], (-1) ** k

    g = np.zeros((3, norb, norb, norb, norb))
    for det, c in psi.items():
        for b, sg, tau in ((0, 0, 0), (1, 0, 1), (2, 1, 1)):
            for q in range(norb):
                d1, s1 = annihilate(det, sg * norb + q)
                for s in range(norb if d1 is not None else 0):
                    d2, s2 = annihilate(d1, tau * norb + s)
                    for rr in range(norb if d2 is not None else 0):
                        d3, s3 = create(d2, tau * norb + rr)
                        for p in range(norb if d3 is not None else 0):
                            d4, s4 = create(d3, sg * norb + p)
                            if d4 in psi:
                                g[b, p, q, rr, s] += psi[d4] * s1 * s2 * s3 * s4 * c
    return g


@pytest.mark.parametrize("nup,ndn,time_sym,z", [(3, 3, False, 1), (4, 2, False, 1), (3, 3, True, 1), (3, 3, True, -1)])
def test_reference_two_rdm_matches_second_quantisation(nup, ndn, time_sym, z):
    rng = np.random.default_rng(17 + nup + 10 * ndn + 100 * time_sym + z)
    norb = 9
    up, dn = _random_list(rng, norb, nup, ndn, 250, time_sym=time_sym)
    w = rng.standard_normal(len(up))
    got = two_rdm(up, dn, w, norb, time_sym=time_sym, z=z)[0]
    ref = _brute_force(up, dn, w, norb, time_sym=time_sym, z=z)
    assert np.max(np.abs(got - ref)) <= 1e-12
    # partial trace against the 1-RDM: sum_r Gamma^{ab}_{pq,rr} = N_beta gamma^alpha
    g1 = one_rdm(up, dn, w, norb, time_sym=time_sym, z=z)[0]
    assert np.max(np.abs(np.einsum("pqrr->pq", got[1]) - ndn * g1[0])) <= 1e-12
    assert np.max(np.abs(np.einsum("pqrr->pq", got[0]) - (nup - 1) * g1[0])) <= 1e-12


def test_spin_squared_of_toy_fci_eigenvectors(tmp_path, oracle):
    """<S^2> of the lowest non-degenerate eigenvectors of the 10-orbital toy FCI (2 alpha, 2 beta) is S(S+1)"""
    toy = str(tmp_path / "FCIDUMP")
    write_toy_fcidump(toy)
    S = oracle.System.chem(toy, 10, 4, 2, [1, 5, 3, 2, 1, 7, 6, 5, 1, 2])
    up, dn = fci_dets(10, 2, 2)
    cnt, idx, val = S.build_upper(oracle.dets_to_u64(up), oracle.dets_to_u64(dn))
    ev, vec = np.linalg.eigh(oracle.upper_to_scipy(cnt, idx, val).toarray())
    keep = [k for k in range(12) if min(abs(ev[k] - ev[k - 1]) if k else 1.0, abs(ev[k + 1] - ev[k])) > 1e-6][:8]
    g = two_rdm(up, dn, vec[:, keep], 10)
    s2 = rdm.spin_squared(g, 2, 2)
    spins = np.round((np.sqrt(1.0 + 4.0 * s2) - 1.0) / 2.0)
    assert np.max(np.abs(s2 - spins * (spins + 1))) <= 1e-10
    assert 0 in spins and 1 in spins


def test_integrals_library_order_match_index():
    from conftest import C2_FCIDUMP
    sysm = systems.ChemSystem(C2_FCIDUMP)
    h, eri, enuc = rdm.integrals_library_order(sysm)
    n1 = sysm.norb + 1
    rng = np.random.default_rng(0)
    for _ in range(200):
        p, q, r, s = (int(x) for x in rng.integers(1, n1, 4))
        assert eri[p - 1, q - 1, r - 1, s - 1] == sysm.integral(p, q, r, s)
        assert h[p - 1, q - 1] == sysm.integral(p, q, n1, n1)
    assert enuc == sysm.integral(n1, n1, n1, n1)
    assert np.array_equal(eri, eri.transpose(2, 3, 0, 1)) and np.array_equal(eri, eri.transpose(1, 0, 2, 3))
