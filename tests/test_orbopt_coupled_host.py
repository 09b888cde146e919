"""Host checks of the coupled (one-step) Newton reference (tests/orbopt_coupled_reference.py) against finite differences of
E(kappa, c) on the toy 10-orbital FCIDUMP (no GPU)."""
import numpy as np
import pytest

from orbopt_coupled_reference import (DenseH, antisym, coupled_hessian_vector, one_index_transform, projector, rotated_integrals,
                                      transition_response)
from orbopt_reference import densities, orbital_derivatives_reference
from rdm2_reference import two_rdm
from rdm_reference import one_rdm
from sqmc_b200 import rdm, systems
from test_natorb_host import fci_dets, write_toy_fcidump
from test_orbopt_host import _mixed_fd


@pytest.fixture(scope="module")
def toy(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("toy_coupled") / "FCIDUMP")
    write_toy_fcidump(path)
    sysm = systems.ChemSystem(path)
    h, g, ec = rdm.integrals_library_order(sysm)
    rng = np.random.default_rng(21)
    up, dn = fci_dets(sysm.norb, sysm.nup, sysm.ndn)
    k = np.sort(rng.choice(len(up), 120, replace=False))
    up, dn = [up[i] for i in k], [dn[i] for i in k]
    return sysm, h, g, ec, up, dn, DenseH(up, dn, sysm.norb)


def test_dense_h_is_symmetric_and_gives_the_rdm_energy(toy):
    sysm, h, g, ec, up, dn, dense = toy
    Hd = dense(h, g, ec)
    assert np.max(np.abs(Hd - Hd.T)) <= 1e-13
    c = np.random.default_rng(1).standard_normal(len(up))
    c /= np.linalg.norm(c)
    D, d = densities(one_rdm(up, dn, c, sysm.norb), two_rdm(up, dn, c, sysm.norb), [1.0], [1.0])
    assert abs(c @ Hd @ c - (ec + np.sum(h * D) + 0.5 * np.sum(g * d))) <= 1e-12


def test_h_kappa_is_the_derivative_of_the_rotated_h(toy):
    sysm, h, g, ec, up, dn, dense = toy
    n = sysm.norb
    rng = np.random.default_rng(2)
    a = np.tril(rng.standard_normal((n, n)), -1)
    K = a - a.T
    hk, gk = one_index_transform(h, g, K)
    assert np.array_equal(hk, hk.T)
    for perm in [(1, 0, 2, 3), (0, 1, 3, 2), (2, 3, 0, 1)]:
        assert np.max(np.abs(gk - gk.transpose(perm))) <= 1e-13
    t = 1e-4
    fd = lambda t: (dense(*rotated_integrals(h, g, t * K)) - dense(*rotated_integrals(h, g, -t * K))) / (2 * t)
    ext = (4.0 * fd(t) - fd(2 * t)) / 3.0
    Hk = dense(hk, gk)
    assert np.max(np.abs(ext - Hk)) <= 1e-9 * np.max(np.abs(Hk))
    # a rotation changes no energy to first order when it is a symmetry: <c|H^k c> = kappa . gradient
    c = rng.standard_normal(len(up))
    c /= np.linalg.norm(c)
    D, d = densities(one_rdm(up, dn, c, n), two_rdm(up, dn, c, n), [1.0], [1.0])
    grad = orbital_derivatives_reference(h, g, D, d)["gradient"]
    il = np.tril_indices(n, -1)
    assert abs(c @ Hk @ c - K[il] @ grad[il]) <= 1e-11


@pytest.mark.parametrize("n_states", [1, 2])
def test_joint_hessian_vector_matches_finite_differences(toy, n_states):
    sysm, h, g, ec, up, dn, dense = toy
    n = sysm.norb
    rng = np.random.default_rng(3 + n_states)
    C, _ = np.linalg.qr(rng.standard_normal((len(up), n_states)))
    w = np.array([1.0]) if n_states == 1 else np.array([0.6, 0.4])
    pairs = [(p, q) for p in range(n) for q in range(p)]
    g1 = one_rdm(up, dn, C, n)
    g2 = two_rdm(up, dn, C, n)
    D, d = densities(g1, g2, [1.0] * n_states, w)
    ref = orbital_derivatives_reference(h, g, D, d)
    ip = np.array([p for p, _ in pairs])
    iq = np.array([q for _, q in pairs])
    E2red = ref["hessian"][ip, iq][:, ip, iq]
    P = projector(C)
    m = len(pairs)

    def split(v):
        return v[:m], v[m:].reshape(len(up), n_states)

    def E(v):
        x, Y = split(v)
        hr, gr = rotated_integrals(h, g, antisym(pairs, x, n))
        Hr = dense(hr, gr, ec)
        Cv = C + Y
        return sum(w[k] * (Cv[:, k] @ Hr @ Cv[:, k]) / (Cv[:, k] @ Cv[:, k]) for k in range(n_states))

    def direction():
        return np.concatenate([rng.standard_normal(m), (P @ rng.standard_normal((len(up), n_states))).ravel()])

    # the gradient: orbital part from orbital_derivatives, CI part 2 w_k (H - E_k) c_k
    Hd = dense(h, g, ec)
    Ek = np.einsum("ik,ij,jk->k", C, Hd, C)
    gc = np.stack([2.0 * w[k] * (Hd @ C[:, k] - Ek[k] * C[:, k]) for k in range(n_states)], axis=1)
    eps = 1e-4
    for _ in range(2):
        A, B = direction(), direction()
        c1 = lambda t: (E(t * A) - E(-t * A)) / (2 * t)
        fd1 = (4.0 * c1(eps) - c1(2 * eps)) / 3.0
        xa, Ya = split(A)
        assert abs(fd1 - (xa @ ref["gradient"][ip, iq] + np.sum(Ya * gc))) <= 1e-9
        xb, Yb = split(B)
        ho, hc = coupled_hessian_vector(dense, h, g, ec, C, w, E2red, pairs, xb, Yb)
        an = xa @ ho + np.sum(Ya * hc)
        assert abs(_mixed_fd(E, A, B) - an) <= 1e-5 * max(1.0, abs(an))
        # the orbital-CI block is the response of the gradient, and symmetric with the CI-orbital block
        resp = transition_response(h, g, up, dn, C, Yb, w, n)
        ho0, _ = coupled_hessian_vector(dense, h, g, ec, C, w, 0.0 * E2red, pairs, np.zeros(m), Yb)
        assert np.max(np.abs(resp[ip, iq] - ho0)) <= 1e-11 * max(1.0, np.max(np.abs(ho0)))
        _, hc0 = coupled_hessian_vector(dense, h, g, ec, C, w, E2red, pairs, xa, 0.0 * Yb)
        assert abs(np.sum(Yb * hc0) - xa @ ho0) <= 1e-11 * max(1.0, abs(xa @ ho0))
