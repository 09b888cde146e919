"""Host checks of the orbital-derivative reference (tests/orbopt_reference.py) and of the determinant remap of
sqmc_b200.orbopt (no GPU)."""
import itertools

import numpy as np
import pytest

from orbopt_reference import densities, energy, orbital_derivatives_reference, rotated_energy
from rdm2_reference import two_rdm
from rdm_reference import one_rdm
from sqmc_b200 import orbopt, rdm, systems
from test_natorb_host import fci_dets, write_toy_fcidump


@pytest.fixture(scope="module")
def toy(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("toy") / "FCIDUMP")
    write_toy_fcidump(path)
    sysm = systems.ChemSystem(path)
    h, g, ec = rdm.integrals_library_order(sysm)
    return path, sysm, h, g, ec


def _random_state(sysm, n, seed):
    rng = np.random.default_rng(seed)
    up, dn = fci_dets(sysm.norb, sysm.nup, sysm.ndn)
    k = np.sort(rng.choice(len(up), n, replace=False))
    up, dn = [up[i] for i in k], [dn[i] for i in k]
    return up, dn, rng.standard_normal(len(up))


def _antisym(rng, n):
    a = np.tril(rng.standard_normal((n, n)), -1)
    return a - a.T


def _mixed_fd(E, A, B, t=1e-3):
    """d^2 E(a A + b B) / da db at 0: f(t) = [E(t(A+B)) - E(t(A-B)) + E(-t(A+B)) - E(-t(A-B))] / 4 = t^2 X + O(t^4), extrapolated"""
    f = lambda t: (E(t * (A + B)) - E(t * (A - B)) + E(-t * (A + B)) - E(-t * (A - B))) / 4.0
    return (16.0 * f(t) - f(2 * t)) / (12.0 * t * t)


def test_reference_matches_finite_differences(toy):
    _, sysm, h, g, ec = toy
    n = sysm.norb
    up, dn, w = _random_state(sysm, 150, 1)
    norm2 = float(w @ w)
    D, d = densities(one_rdm(up, dn, w, n), two_rdm(up, dn, w, n), [norm2], [1.0])
    r = orbital_derivatives_reference(h, g, D, d)
    E = lambda k: rotated_energy(h, g, ec, D, d, k)
    assert abs(E(np.zeros((n, n))) - (energy(h, g, ec, D, d))) == 0.0
    rng = np.random.default_rng(2)
    il = np.tril_indices(n, -1)
    H2 = r["hessian"][il[0], il[1]][:, il[0], il[1]]
    assert np.max(np.abs(H2 - H2.T)) <= 1e-10 * np.max(np.abs(H2))
    eps = 1e-4
    for _ in range(3):   # random antisymmetric directions
        A, B = _antisym(rng, n), _antisym(rng, n)
        fd1 = (E(eps * A) - E(-eps * A)) / (2 * eps)
        assert abs(fd1 - A[il] @ r["gradient"][il]) <= 1e-7
        an = A[il] @ H2 @ B[il]
        assert abs(_mixed_fd(E, A, B) - an) <= 1e-5 * max(1.0, abs(an))
    for (p, q), (r_, s) in [((3, 1), (3, 1)), ((5, 0), (9, 2)), ((7, 6), (4, 1)), ((8, 4), (8, 0))]:   # coordinate pairs
        A = np.zeros((n, n)); A[p, q], A[q, p] = 1.0, -1.0
        B = np.zeros((n, n)); B[r_, s], B[s, r_] = 1.0, -1.0
        assert abs((E(eps * A) - E(-eps * A)) / (2 * eps) - r["gradient"][p, q]) <= 1e-7
        an = r["hessian"][p, q, r_, s]
        assert abs(_mixed_fd(E, A, B) - an) <= 1e-5 * max(1.0, abs(an))


def test_fci_ground_state_is_stationary(toy, oracle):
    path, sysm, h, g, ec = toy
    n = sysm.norb
    up, dn = fci_dets(n, sysm.nup, sysm.ndn)
    S = oracle.System.chem(path, n, sysm.nelec, sysm.nup, list(sysm.orbital_symmetries_fcidump))
    cnt, idx, val = S.build_upper(oracle.dets_to_u64(up), oracle.dets_to_u64(dn))
    ev, vec = np.linalg.eigh(oracle.upper_to_scipy(cnt, idx, val).toarray())
    c = vec[:, 0]
    D, d = densities(one_rdm(up, dn, c, n), two_rdm(up, dn, c, n), [1.0], [1.0])
    assert abs(energy(h, g, ec, D, d) - ev[0]) <= 1e-10
    r = orbital_derivatives_reference(h, g, D, d)
    assert np.max(np.abs(r["gradient"])) <= 1e-9


def _brute_sign(occ, perm):
    """parity of the bubble sort of the renamed creation operators"""
    a = [int(perm[o]) for o in occ]
    sign = 1
    for i in range(len(a)):
        for j in range(len(a) - 1 - i):
            if a[j] > a[j + 1]:
                a[j], a[j + 1] = a[j + 1], a[j]
                sign = -sign
    return sign


def test_remap_strings_against_brute_force():
    rng = np.random.default_rng(4)
    norb = 9
    for _ in range(5):
        perm = rng.permutation(norb)
        strings = [sum(1 << k for k in c) for m in (2, 3, 4) for c in itertools.combinations(range(norb), m)]
        got, sg = orbopt.remap_strings(np.array(strings, dtype=np.uint64), perm)
        for s, gw, gs in zip(strings, got, sg):
            occ = [k for k in range(norb) if (s >> k) & 1]
            assert int(gw) == sum(1 << int(perm[o]) for o in occ)
            assert gs == _brute_sign(occ, perm)


@pytest.mark.parametrize("time_sym,z", [(False, 1), (True, 1), (True, -1)])
def test_remap_round_trip(time_sym, z):
    from test_natorb_host import _random_list
    rng = np.random.default_rng(5 + z)
    norb = 12
    up, dn = _random_list(rng, norb, 3, 3, 200, time_sym=time_sym)
    from sqmc_b200.api import dets_to_u64
    U, Dn = dets_to_u64(up), dets_to_u64(dn)
    w = rng.standard_normal((len(up), 2))
    perm = rng.permutation(norb)
    u2, d2, w2 = orbopt.remap_determinants(U, Dn, w, perm, time_sym=time_sym, z=z)
    if time_sym:
        assert np.all(u2[:, 0] <= d2[:, 0]) and np.any(u2[:, 0] != U[:, 0])
    u3, d3, w3 = orbopt.remap_determinants(u2, d2, w2, np.argsort(perm), time_sym=time_sym, z=z)
    assert np.array_equal(u3, U) and np.array_equal(d3, Dn) and np.array_equal(w3, w)


@pytest.mark.parametrize("z", [1, -1])
def test_remap_time_sym_matches_expanded_wavefunction(z):
    """the remapped representatives expand to the renamed plain wavefunction, signs included"""
    from rdm_reference import expand_time_sym
    from test_natorb_host import _random_list
    from sqmc_b200.api import dets_to_u64
    rng = np.random.default_rng(11 + z)
    norb = 8
    up, dn = _random_list(rng, norb, 3, 3, 60, time_sym=True)
    w = rng.standard_normal(len(up))
    perm = rng.permutation(norb)
    u2, d2, w2 = orbopt.remap_determinants(dets_to_u64(up), dets_to_u64(dn), w, perm, time_sym=True, z=z)
    eu, ed, ew = expand_time_sym(up, dn, w, z)
    ref = {}
    for u, d, c in zip(eu, ed, ew[:, 0]):
        ou = [k for k in range(norb) if (u >> k) & 1]
        od = [k for k in range(norb) if (d >> k) & 1]
        key = (sum(1 << int(perm[k]) for k in ou), sum(1 << int(perm[k]) for k in od))
        ref[key] = c * _brute_sign(ou, perm) * _brute_sign(od, perm)
    gu, gd, gw = expand_time_sym([int(x) for x in u2[:, 0]], [int(x) for x in d2[:, 0]], w2, z)
    got = {(u, d): c for u, d, c in zip(gu, gd, gw[:, 0])}
    assert got.keys() == ref.keys()
    assert all(abs(got[k] - ref[k]) <= 1e-15 for k in ref)
