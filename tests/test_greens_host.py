"""Host checks of the Green's function references and of the continued-fraction evaluation of sqmc_b200.greens (no GPU):
the ladder reference against second quantisation, and on the toy 10-orbital FCIDUMP (2 alpha + 2 beta electrons) the
Lanczos continued fraction of a complete Krylov space against the exact sum over states of each N-1 / N+1 sector."""
import numpy as np
import pytest

from greens_reference import fock_ladder, ladder, lanczos, sum_over_states
from rdm_reference import one_rdm
from sqmc_b200 import greens, systems
from test_natorb_host import _random_list, fci_dets, write_toy_fcidump


@pytest.mark.parametrize("time_sym,z", [(False, 1), (True, 1), (True, -1)])
@pytest.mark.parametrize("spin", [0, 1])
@pytest.mark.parametrize("create", [False, True])
def test_reference_ladder_matches_second_quantisation(time_sym, z, spin, create):
    rng = np.random.default_rng(11 + 2 * spin + create + 10 * time_sym + z)
    norb = 12
    up, dn = _random_list(rng, norb, 3, 3 if time_sym else 4, 200, time_sym=time_sym)
    w = rng.standard_normal(len(up))
    orbs = [5, 0, 11, 3]
    u2, d2, phi = ladder(up, dn, w, orbs, spin, create, time_sym=time_sym, z=z)
    ref = fock_ladder(up, dn, w, norb, orbs, spin, create, time_sym=time_sym, z=z)
    assert set(zip(u2, d2)) == set(ref)
    assert list(zip(u2, d2)) == sorted(zip(u2, d2))
    for i, k in enumerate(zip(u2, d2)):
        assert np.max(np.abs(phi[i] - np.array(ref[k]))) <= 1e-14


def _dense(oracle, path, nup, ndn):
    S = oracle.System.chem(path, 10, nup + ndn, nup, [1, 5, 3, 2, 1, 7, 6, 5, 1, 2])
    up, dn = fci_dets(10, nup, ndn)
    cnt, idx, val = S.build_upper(oracle.dets_to_u64(up), oracle.dets_to_u64(dn))
    return up, dn, oracle.upper_to_scipy(cnt, idx, val).toarray()


@pytest.fixture(scope="module")
def toy(tmp_path_factory, oracle):
    path = str(tmp_path_factory.mktemp("toy_greens") / "FCIDUMP")
    write_toy_fcidump(path)
    sysm = systems.ChemSystem(path)
    # the library's orbital order is the same in every electron sector of the toy space (the oracle's dense H uses its own)
    for nup, ndn in ((1, 2), (2, 1), (3, 2), (2, 3)):
        assert np.array_equal(systems.ChemSystem(path, nelec=nup + ndn, nup=nup).orb_order, sysm.orb_order)
    up, dn, H0 = _dense(oracle, path, 2, 2)
    assert len(up) == 2025
    c, e0 = clean_ground_state(H0)
    return dict(path=path, system=sysm, up=up, dn=dn, c=c, e0=e0, dense=lambda nu, nd: _dense(oracle, path, nu, nd))


def clean_ground_state(H0):
    """the lowest eigenvector of a dense H with its rounding noise (~1e-13) outside its symmetry block set to zero, and its
    energy: the images then lie in one block of each sector and their Krylov spaces close after at most that block's size"""
    E, X = np.linalg.eigh(H0)
    c = np.where(np.abs(X[:, 0]) > 1e-9, X[:, 0], 0.0)
    c /= np.linalg.norm(c)
    return c, float(c @ H0 @ c)


def _images_in_sector(toy, orbs, spin, create):
    """the images of the toy ground state embedded in the full N-1 / N+1 sector, and that sector's dense H"""
    nup, ndn = 2 + (0 if spin else (1 if create else -1)), 2 + ((1 if create else -1) if spin else 0)
    su, sd, Hs = toy["dense"](nup, ndn)
    u2, d2, phi = ladder(toy["up"], toy["dn"], toy["c"], orbs, spin, create)
    index = {k: i for i, k in enumerate(zip(su, sd))}
    V = np.zeros((len(su), len(orbs)))
    for i, k in enumerate(zip(u2, d2)):
        V[index[k]] = phi[i]
    return Hs, V


@pytest.mark.parametrize("spin,create,size", [(0, False, 450), (1, False, 450), (0, True, 5400)])
def test_complete_krylov_continued_fraction_equals_sum_over_states(toy, spin, create, size):
    orbs = [0, 1, 2, 5, 8]
    Hs, V = _images_in_sector(toy, orbs, spin, create)
    assert Hs.shape == (size, size)
    P = len(orbs)
    norms = np.linalg.norm(V, axis=0)
    m = size
    alpha, beta = np.zeros((P, m)), np.zeros((P, m))
    ovl = np.zeros((P, m, P))
    steps = np.zeros(P, dtype=int)
    for a in range(P):
        al, be, Q = lanczos(Hs, V[:, a], m, 1e-10)
        assert len(al) < m   # the Krylov space closed
        steps[a] = len(al)
        alpha[a, :len(al)], beta[a, :len(al)] = al, be
        ovl[a, :len(al)] = Q.T @ V
    z = np.linspace(-3.0, 3.0, 41) + 0.05j
    M, poles, res = greens.krylov_resolvent(alpha, beta, ovl, steps, norms, toy["e0"], z, create)
    ref = sum_over_states(Hs, V, toy["e0"], z, create)
    assert np.max(np.abs(M - ref)) <= 1e-10
    # residues of the diagonal elements: gamma_pp (removal), 1 - gamma_pp (addition)
    g = one_rdm(toy["up"], toy["dn"], toy["c"], 10)[0, spin]
    for a, p in enumerate(orbs):
        want = 1.0 - g[p, p] if create else g[p, p]
        assert abs(np.sum(res[a]) - want) <= 1e-12
        assert np.all(np.diff(poles[a]) >= 0)
    # the matrix of residues, summed over the exact poles: <v_b|v_a> = gamma_pq (removal) or delta_pq - gamma_qp (addition)
    R = V.T @ V
    want = np.eye(P) - g[np.ix_(orbs, orbs)].T if create else g[np.ix_(orbs, orbs)]
    assert np.max(np.abs(R - want)) <= 1e-12


def test_electron_space_keeps_the_orbitals(toy):
    s = toy["system"]
    for spin in (0, 1):
        for create in (False, True):
            x, flipped = greens.electron_space(s, spin, create)
            d = 1 if create else -1
            nup, ndn = s.nup + d * (spin == 0), s.ndn + d * (spin == 1)
            assert flipped == (nup < ndn)   # the 2 + 2 toy: removing alpha or adding beta flips the spins
            assert (x.nup, x.ndn, x.nelec) == ((ndn, nup) if flipped else (nup, ndn)) + (s.nelec + d,)
            assert x.nup >= x.ndn
            assert x.integrals is s.integrals and np.array_equal(x.orb_order, s.orb_order) and not x.time_sym
            assert bin(x.hf_up).count("1") == x.nup and bin(x.hf_dn).count("1") == x.ndn
    with pytest.raises(ValueError, match="chem systems"):
        greens.electron_space(systems.HubbardKSystem(2, 2, 1.0, 4.0, 2, 2), 0, False)


def test_spectral_function_is_minus_imag_over_pi():
    G = np.array([[1.0 - 2.0j, 0.5j]])
    assert np.array_equal(greens.spectral_function(G), np.array([[2.0, -0.5]]) / np.pi)
