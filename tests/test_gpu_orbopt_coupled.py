"""sigma-vectors with and without a one-index transformation (SparseHamiltonian.sigma), the orbital-gradient response
(SparseHamiltonian.orbital_gradient_response) and the one-step orbital optimiser (sqmc_b200.orbopt, one_step=True)."""
import os

import numpy as np
import pytest

from conftest import C2_FCIDUMP, ROOT
from orbopt_coupled_reference import DenseH, one_index_transform
from orbopt_reference import densities, orbital_derivatives_reference
from rdm_reference import expand_time_sym, u64_to_ints
from test_gpu_rdm2 import _list53, _random_eri_system, _subset

pytestmark = pytest.mark.gpu
C2_INPUT = os.path.join(ROOT, "data", "C2_v2z_curve", "r1.24253", "i_1sigma_g")


def _sq():
    import sqmc_b200 as sq
    return sq


def _kappa(rng, sysm, within_irreps=True):
    n = sysm.norb
    a = np.tril(rng.standard_normal((n, n)), -1)
    if within_irreps:
        sym = np.asarray(sysm.orbital_symmetries)
        a *= sym[:, None] == sym[None, :]
    return a - a.T


def _lists(sq, c2_space, c2_space_ts):
    """(label, handle, up, dn, x) for the C2 lists of the issue: plain, time_sym, 5 alpha / 3 beta, two vectors, random (pq|rs)"""
    rng = np.random.default_rng(31)
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = _subset(c2_space[1], 250, 1)
    out = [("plain", H, up, dn, rng.standard_normal(len(up))), ("two vectors", H, up, dn, rng.standard_normal((len(up), 2)))]
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    up, dn = _subset(c2_space_ts[1], 250, 2)
    out.append(("time_sym", Hts, up, dn, rng.standard_normal(len(up))))
    H53 = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, nelec=8, nup=5, time_sym=False, z=1))
    up, dn = _list53(sq, 300, 3)
    out.append(("5a3b", H53, up, dn, rng.standard_normal(len(up))))
    sysm, _ = _random_eri_system(sq, rng, time_sym=False, z=1)
    up, dn = _subset(c2_space[1], 250, 5)
    out.append(("random eri", sq.SparseHamiltonian(sysm), up, dn, rng.standard_normal(len(up))))
    return out


def _dense_apply(H, up, dn, x, kappa):
    """y = H x (kappa None) or H^kappa x over the list from the numpy Slater-Condon reference, time_sym through the plain
    expansion -> (y, dense matrix over the plain list, plain up, plain dn)"""
    from sqmc_b200 import rdm
    sysm = H.system
    h, g, ec = rdm.integrals_library_order(sysm)
    ui, di = u64_to_ints(up), u64_to_ints(dn)
    x2 = np.asarray(x, dtype=np.float64).reshape(len(ui), -1)
    ts = bool(sysm.time_sym)
    eu, ed, ex = expand_time_sym(ui, di, x2, sysm.z) if ts else (ui, di, x2)
    dense = DenseH(eu, ed, sysm.norb)
    M = dense(h, g, ec) if kappa is None else dense(*one_index_transform(h, g, kappa))
    ye = M @ ex
    if not ts:
        return ye.reshape(np.shape(x)), M, eu, ed
    pos = {(u, d): k for k, (u, d) in enumerate(zip(eu, ed))}
    y = np.zeros_like(x2)
    for i, (u, d) in enumerate(zip(ui, di)):
        y[i] = ye[pos[(u, d)]] if u == d else (ye[pos[(u, d)]] + sysm.z * ye[pos[(d, u)]]) / np.sqrt(2.0)
    return y.reshape(np.shape(x)), M, eu, ed


def test_sigma_without_kappa_matches_the_resident_matrix(c2_space, c2_space_ts):
    sq = _sq()
    for label, H, up, dn, x in _lists(sq, c2_space, c2_space_ts):
        H.generate_sparse_ham_upper_triangular(up, dn)
        ref = H.matvec(x)
        got = H.sigma(up, dn, x)
        assert got.shape == np.shape(x)
        assert np.max(np.abs(got - ref)) <= 1e-12 * np.max(np.abs(ref)), label


def test_sigma_with_kappa_matches_the_dense_reference(c2_space, c2_space_ts):
    sq = _sq()
    rng = np.random.default_rng(32)
    covered_zero = False
    for label, H, up, dn, x in _lists(sq, c2_space, c2_space_ts):
        K = _kappa(rng, H.system)
        ref, Mk, eu, ed = _dense_apply(H, up, dn, x, K)
        got = H.sigma(up, dn, x, kappa=K)
        assert np.max(np.abs(got - ref)) <= 1e-10 * np.max(np.abs(ref)), label
        if not H.system.time_sym and label != "random eri":
            # a pair whose element of H is exactly 0 and whose element of H^kappa is not: sigma must reach it
            M0 = _dense_apply(H, up, dn, x, None)[1]
            cand = np.argwhere((M0 == 0.0) & (np.abs(Mk) > 1e-6))
            if len(cand):
                i, j = cand[0]
                e = np.zeros(len(up))
                e[j] = 1.0
                yj = H.sigma(up, dn, e, kappa=K)
                assert abs(yj[i] - Mk[i, j]) <= 1e-10 * abs(Mk[i, j]) and yj[i] != 0.0
                covered_zero = True
    assert covered_zero


def test_sigma_kappa_and_response_identities(c2_space, c2_space_ts):
    """<c|H^k c> / |c|^2 = sum_{p>q} k_pq gradient_pq and sum_{p>q} k_pq response_pq = 2 <dc|H^k c> for dc orthogonal to c"""
    sq = _sq()
    rng = np.random.default_rng(33)
    for label, H, up, dn, x in _lists(sq, c2_space, c2_space_ts):
        if np.ndim(x) != 1:
            continue
        n = H.system.norb
        il = np.tril_indices(n, -1)
        K = _kappa(rng, H.system, within_irreps=False)
        sk = H.sigma(up, dn, x, kappa=K)
        grad = H.orbital_derivatives(up, dn, x)["gradient"]
        lhs = float(x @ sk) / float(x @ x)
        assert abs(lhs - K[il] @ grad[il]) <= 1e-10 * max(1.0, abs(lhs)), label
        c = x / np.linalg.norm(x)
        dc = rng.standard_normal(len(c))
        dc -= (c @ dc) * c
        resp = H.orbital_gradient_response(up, dn, c, dc)
        assert np.max(np.abs(resp + resp.T)) == 0.0
        rhs = 2.0 * float(dc @ H.sigma(up, dn, c, kappa=K))
        assert abs(K[il] @ resp[il] - rhs) <= 1e-10 * max(1.0, abs(rhs)), label


def _response_reference(H, up, dn, C, dC, sw):
    """numpy: the gradient of orbital_derivatives_reference at the densities 2 w_k / |c_k|^2 T(c_k, dc_k'), T from one_rdm / two_rdm
    of c +- dc' by polarisation"""
    from sqmc_b200 import rdm
    h, g, _ = rdm.integrals_library_order(H.system)
    C2 = np.asarray(C).reshape(len(up), -1)
    dC2 = np.asarray(dC).reshape(C2.shape)
    D, d = 0.0, 0.0
    for k in range(C2.shape[1]):
        a = C2[:, k]
        b = dC2[:, k] - (a @ dC2[:, k]) / (a @ a) * a
        g1 = (H.one_rdm(up, dn, a + b) - H.one_rdm(up, dn, a - b)) / 4.0
        g2 = (H.two_rdm(up, dn, a + b) - H.two_rdm(up, dn, a - b)) / 4.0
        Dk, dk = densities([g1], [g2], [a @ a], [2.0 * sw[k]])
        D, d = D + Dk, d + dk
    return orbital_derivatives_reference(h, g, D, d)["gradient"]


def test_response_against_finite_differences_and_reference(c2_space, c2_space_ts):
    sq = _sq()
    rng = np.random.default_rng(34)
    for label, H, up, dn, x in _lists(sq, c2_space, c2_space_ts):
        ns = 1 if np.ndim(x) == 1 else np.shape(x)[1]
        sw = np.full(ns, 1.0 / ns) if ns == 1 else np.array([0.7, 0.3])
        dx = rng.standard_normal(np.shape(x))   # not orthogonal: the normalisation term counts
        got = H.orbital_gradient_response(up, dn, x, dx, state_weights=sw)
        ref = _response_reference(H, up, dn, x, dx, sw)
        assert np.max(np.abs(got - ref)) <= 1e-10 * max(1.0, np.max(np.abs(ref))), label
        t = 1e-4
        gr = lambda s: H.orbital_derivatives(up, dn, x + s * dx, state_weights=sw)["gradient"]
        c1 = lambda t: (gr(t) - gr(-t)) / (2 * t)
        fd = (4.0 * c1(t) - c1(2 * t)) / 3.0
        assert np.max(np.abs(got - fd)) <= 1e-7 * max(1.0, np.max(np.abs(got))), label


def test_determinism(c2_space):
    sq = _sq()
    _, r = c2_space
    up, dn = r["up"], r["dn"]
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    rng = np.random.default_rng(35)
    x, dx = rng.standard_normal((len(up), 2)), rng.standard_normal((len(up), 2))
    K = _kappa(rng, H.system)
    p = rng.permutation(len(up))
    for kap in (None, K):
        a = H.sigma(up, dn, x, kappa=kap)
        assert np.array_equal(a, H.sigma(up, dn, x, kappa=kap))
        assert np.array_equal(a[p], H.sigma(up[p], dn[p], x[p], kappa=kap))
    a = H.orbital_gradient_response(up, dn, x, dx, state_weights=[0.25, 0.75])
    assert np.array_equal(a, H.orbital_gradient_response(up, dn, x, dx, state_weights=[0.25, 0.75]))
    assert np.array_equal(a, H.orbital_gradient_response(up[p], dn[p], x[p], dx[p], state_weights=[0.25, 0.75]))


def test_input_errors(c2_space, c2_space_ts, tmp_path):
    sq = _sq()
    _, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = r["up"][:50], r["dn"][:50]
    w = np.ones(len(up))
    n = H.system.norb
    with pytest.raises(sq.SqmcError, match="not antisymmetric"):
        H.sigma(up, dn, w, kappa=np.eye(n))
    with pytest.raises(ValueError, match="kappa must have shape"):
        H.sigma(up, dn, w, kappa=np.zeros((3, 3)))
    with pytest.raises(ValueError, match="dwts has shape"):
        H.orbital_gradient_response(up, dn, w, np.ones(len(up) + 1))
    with pytest.raises(sq.SqmcError, match="negative"):
        H.orbital_gradient_response(up, dn, np.ones((len(up), 2)), np.ones((len(up), 2)), state_weights=[1.5, -0.5])
    with pytest.raises(sq.SqmcError, match="sum to"):
        H.orbital_gradient_response(up, dn, np.ones((len(up), 2)), np.ones((len(up), 2)), state_weights=[0.5, 0.6])
    for call in (lambda u, d, v: H.sigma(u, d, v), lambda u, d, v: H.orbital_gradient_response(u, d, v, v)):
        with pytest.raises(sq.SqmcError, match="twice"):
            call(np.concatenate([up, up[:1]]), np.concatenate([dn, dn[:1]]), np.ones(len(up) + 1))
        with pytest.raises(sq.SqmcError, match="n must be positive"):
            call(up[:0], dn[:0], w[:0])
        with pytest.raises(sq.SqmcError, match="electrons"):
            call(np.concatenate([up, sq.dets_to_u64([0b111])]), np.concatenate([dn, sq.dets_to_u64([0b1111])]), np.ones(len(up) + 1))
    with pytest.raises(sq.SqmcError, match="n_states"):
        H.sigma(up, dn, np.zeros((len(up), 0)))
    _, rt = c2_space_ts
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    k = next(i for i in range(len(rt["up"])) if not np.array_equal(rt["up"][i], rt["dn"][i]))
    with pytest.raises(sq.SqmcError, match="time-reversed partner"):
        Hts.sigma(np.concatenate([rt["up"], rt["dn"][k:k + 1]]), np.concatenate([rt["dn"], rt["up"][k:k + 1]]), np.ones(len(rt["up"]) + 1))
    hs = sq.HegSystem(3, 0.5, 14, 7, 1.49)
    with pytest.raises(sq.SqmcError, match="sigma: .*fixed by momentum"):
        sq.SparseHamiltonian(hs).sigma(sq.dets_to_u64([hs.hf_up]), sq.dets_to_u64([hs.hf_dn]), np.ones(1))
    hub = sq.HubbardKSystem(4, 2, 1.0, 4.0, 3, 2)
    with pytest.raises(sq.SqmcError, match="orbital_gradient_response: .*fixed by momentum"):
        sq.SparseHamiltonian(hub).orbital_gradient_response(sq.dets_to_u64([0b111]), sq.dets_to_u64([0b11]), np.ones(1), np.ones(1))
    big = str(tmp_path / "FCIDUMP65")
    with open(big, "w") as f:
        f.write(" &FCI NORB=65,NELEC=2,MS2=0,\n &END\n" + "".join("-1.0 %d %d 0 0\n" % (p, p) for p in range(1, 66)) + "0.0 0 0 0 0\n")
    Hb = sq.SparseHamiltonian(sq.ChemSystem(big))
    with pytest.raises(sq.SqmcError, match="norb = 65 > 64"):
        Hb.sigma(sq.dets_to_u64([1]), sq.dets_to_u64([1]), np.ones(1))
    with pytest.raises(sq.SqmcError, match="norb = 65 > 64"):
        Hb.orbital_gradient_response(sq.dets_to_u64([1]), sq.dets_to_u64([1]), np.ones(1), np.ones(1))


def test_existing_density_paths_unchanged_by_the_two_vector_mode(c2_space):
    """two_rdm and orbital_derivatives give the same bits before and after a two-vector (response) call on the handle"""
    sq = _sq()
    _, r = c2_space
    up, dn = _subset(r, 300, 7)
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    w = np.random.default_rng(36).standard_normal((len(up), 2))
    g2 = H.two_rdm(up, dn, w)
    od = H.orbital_derivatives(up, dn, w, state_weights=[0.4, 0.6])
    H.orbital_gradient_response(up, dn, w, w[::-1].copy(), state_weights=[0.4, 0.6])
    H.sigma(up, dn, w, kappa=_kappa(np.random.default_rng(37), H.system))
    assert np.array_equal(g2, H.two_rdm(up, dn, w))
    od2 = H.orbital_derivatives(up, dn, w, state_weights=[0.4, 0.6])
    for key in ("fock", "hessian"):
        assert np.array_equal(od[key], od2[key])


def test_one_step_c2_converges(tmp_path):
    from sqmc_b200 import hci, orbopt
    res = orbopt.optimize_orbitals(C2_INPUT, str(tmp_path / "one"), one_step=True, max_macro=10)
    hist = res["history"]
    e = [h["energy"] for h in hist]
    print("one step: converged=%s after %d macro iterations; max|g| %s; E %s; micro %s"
          % (res["converged"], len(hist), ["%.2e" % h["max_grad"] for h in hist], ["%.10f" % x for x in e], [h["micro"] for h in hist]))
    assert all(b <= a for a, b in zip(e, e[1:]))
    assert res["converged"] and hist[-1]["max_grad"] < 1e-4
    two = orbopt.optimize_orbitals(C2_INPUT, str(tmp_path / "two"), fixed_list=True, max_macro=10)
    print("two step: max|g| %.2e E %.10f" % (two["history"][-1]["max_grad"], two["history"][-1]["energy"]))
    assert not two["converged"]
    assert e[-1] <= two["history"][-1]["energy"]
    rerun = hci.run_input(os.path.join(str(tmp_path / "one"), "i_1sigma_g"), log=lambda *a: None)
    assert np.isfinite(rerun["energy"]).all()
