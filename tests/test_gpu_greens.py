"""Single-particle Green's function on the device: ladder images (csrc/rdm.cu), tridiagonal Lanczos (csrc/davidson.cu) and
sqmc_b200.greens end to end."""
import ctypes as C
import itertools

import numpy as np
import pytest

from conftest import C2_FCIDUMP
from greens_reference import ladder as ref_ladder, lanczos as ref_lanczos, sum_over_states
from rdm_reference import expand_time_sym, u64_to_ints
from test_greens_host import _dense, clean_ground_state
from test_natorb_host import write_toy_fcidump

pytestmark = pytest.mark.gpu


def _sq():
    import sqmc_b200 as sq
    return sq


def _norm(w):
    w = np.asarray(w, dtype=np.float64)
    return w / np.linalg.norm(w, axis=0)


def _check_ladder(H, up, dn, w, orbs, spin, create, time_sym=False, z=1):
    u2, d2, phi = H.ladder(up, dn, w, orbs, spin, create)
    ru, rd, rphi = ref_ladder(up, dn, w, orbs, spin, create, time_sym=time_sym, z=z)
    assert u64_to_ints(u2) == ru and u64_to_ints(d2) == rd
    assert phi.shape == rphi.shape
    assert np.max(np.abs(phi - rphi)) <= 1e-15
    return u2, d2, phi


def _c2_53(rng, n=3000):
    ups = [sum(1 << k for k in c) for c in itertools.combinations(range(10), 5)]
    dns = [sum(1 << k for k in c) for c in itertools.combinations(range(9), 3)]
    pairs = [(u, d) for u in ups for d in dns]
    sel = rng.choice(len(pairs), n, replace=False)
    return [pairs[k][0] for k in sel], [pairs[k][1] for k in sel]


def test_ladder_c2_plain_and_53(c2_space):
    sq = _sq()
    _, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    w = _norm(np.random.default_rng(1).standard_normal(len(r["up"])))
    for spin in (0, 1):
        for create in (False, True):
            _check_ladder(H, r["up"], r["dn"], w, [3, 0, 7, 25, 4], spin, create)
    rng = np.random.default_rng(2)
    up, dn = _c2_53(rng)
    H53 = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, nelec=8, nup=5, time_sym=False, z=1))
    w = _norm(rng.standard_normal((len(up), 2)))
    for spin in (0, 1):
        for create in (False, True):
            u2, d2, phi = H53.ladder(sq.dets_to_u64(up), sq.dets_to_u64(dn), w, [4, 2, 9, 11], spin, create, state=1)
            ru, rd, rphi = ref_ladder(up, dn, w, [4, 2, 9, 11], spin, create, state=1)
            assert u64_to_ints(u2) == ru and u64_to_ints(d2) == rd and np.max(np.abs(phi - rphi)) <= 1e-15


@pytest.mark.parametrize("z", [1, -1])
def test_ladder_c2_time_sym(c2_space_ts, z):
    sq = _sq()
    _, r = c2_space_ts
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=z))
    w = _norm(np.random.default_rng(3).standard_normal(len(r["up"])))
    for spin in (0, 1):
        for create in (False, True):
            _check_ladder(H, r["up"], r["dn"], w, [3, 2, 8], spin, create, time_sym=True, z=z)


def test_ladder_heg_two_word_strings():
    sq = _sq()
    from sqmc_b200 import spaces
    hs = sq.HegSystem(3, 0.5, 14, 7, 2.5)
    assert hs.norb == 81
    H = sq.SparseHamiltonian(hs)
    up, dn, wts, _ = spaces.hci_space(H, hs, 4000, eps_schedule=(1e-2, 3e-3))
    w = _norm(wts[:, 0])
    for spin in (0, 1):
        for create in (False, True):
            _check_ladder(H, up, dn, w, [6, 0, 70, 80, 64, 63], spin, create)


@pytest.mark.parametrize("ts", [False, True])
def test_phase_identity_with_one_rdm(c2_space, c2_space_ts, ts):
    """<phi_p|phi_q> = gamma_pq and <chi_p|chi_q> = delta_pq - gamma_qp against one_rdm, all orbitals, both spins"""
    sq = _sq()
    _, r = c2_space_ts if ts else c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=ts, z=1))
    w = _norm(np.random.default_rng(4).standard_normal(len(r["up"])))
    g = H.one_rdm(r["up"], r["dn"], w)
    orbs = list(range(26))
    for spin in (0, 1):
        _, _, phi = H.ladder(r["up"], r["dn"], w, orbs, spin, False)
        assert np.max(np.abs(phi.T @ phi - g[spin])) <= 1e-13
        _, _, chi = H.ladder(r["up"], r["dn"], w, orbs, spin, True)
        assert np.max(np.abs(chi.T @ chi - (np.eye(26) - g[spin].T))) <= 1e-13


@pytest.fixture(scope="module")
def c2_minus(c2_space):
    """H of the N-1 (alpha removed) space spanned by the images of the shipped C2 list, built on the device"""
    sq = _sq()
    from sqmc_b200 import greens
    _, r = c2_space
    sysm = sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1)
    H = sq.SparseHamiltonian(sysm)
    u2, d2, phi = H.ladder(r["up"], r["dn"], _norm(r["wts"][:, 0]), [3, 2, 1, 0], 0, False)
    sx, flipped = greens.electron_space(sysm, 0, False)
    assert flipped   # 3 alpha + 4 beta: the handle holds the spin-flipped space
    HX = sq.SparseHamiltonian(sx)
    HX.generate_sparse_ham_upper_triangular(d2, u2)
    return HX, phi


def test_lanczos_tridiagonal_matches_numpy(c2_minus, oracle):
    HX, phi = c2_minus
    cnt, idx, val = HX.export_upper()
    Hs = oracle.upper_to_scipy(cnt, idx, val)
    r = HX.lanczos_tridiagonal(phi[:, :3], 30, 0.0)
    for a in range(3):
        al, be, Q = ref_lanczos(Hs, phi[:, a], 30, 0.0)
        assert r["steps"][a] == 30 == len(al)
        assert np.max(np.abs(r["alpha"][a] - al)) <= 1e-10 * np.max(np.abs(al))
        assert np.max(np.abs(r["beta"][a] - be)) <= 1e-10 * np.max(np.abs(al))
        assert np.max(np.abs(r["overlaps"][a] - Q.T @ phi[:, :3])) <= 1e-10


def test_lanczos_tridiagonal_pairs_and_repeats_are_bit_identical(c2_minus):
    HX, phi = c2_minus
    both = HX.lanczos_tridiagonal(phi[:, :3], 25, 1e-12)
    again = HX.lanczos_tridiagonal(phi[:, :3], 25, 1e-12)
    for k in ("alpha", "beta", "overlaps", "steps"):
        assert np.array_equal(both[k], again[k])
    for a in range(3):
        alone = HX.lanczos_tridiagonal(phi[:, a], 25, 1e-12)
        assert np.array_equal(alone["alpha"][0], both["alpha"][a])
        assert np.array_equal(alone["beta"][0], both["beta"][a])
        assert alone["steps"][0] == both["steps"][a]


def test_lanczos_tridiagonal_stops_in_an_invariant_subspace(c2_minus, oracle):
    HX, _ = c2_minus
    cnt, idx, val = HX.export_upper()
    Hd = oracle.upper_to_scipy(cnt, idx, val).toarray()
    E, X = np.linalg.eigh(Hd)
    v = X[:, 0] + 0.5 * X[:, 3] - 0.25 * X[:, 7]
    r = HX.lanczos_tridiagonal(v, 40, 1e-8)
    assert r["steps"][0] == 3
    T = np.diag(r["alpha"][0, :3]) + np.diag(r["beta"][0, :2], 1) + np.diag(r["beta"][0, :2], -1)
    assert np.max(np.abs(np.linalg.eigvalsh(T) - E[[0, 3, 7]])) <= 1e-9


@pytest.fixture(scope="module")
def toy(tmp_path_factory, oracle):
    sq = _sq()
    path = str(tmp_path_factory.mktemp("toy_greens_gpu") / "FCIDUMP")
    write_toy_fcidump(path)
    sysm = sq.ChemSystem(path)
    up, dn, H0 = _dense(oracle, path, 2, 2)
    c, e0 = clean_ground_state(H0)
    return dict(path=path, system=sysm, H=sq.SparseHamiltonian(sysm), up=sq.dets_to_u64(up), dn=sq.dets_to_u64(dn), c=c, e0=e0,
                dense=lambda nu, nd: _dense(oracle, path, nu, nd))


def test_end_to_end_toy_fci_equals_sum_over_states(toy):
    from sqmc_b200 import greens
    orbs = [0, 1, 2, 5, 8]
    omega = np.linspace(-3.0, 3.0, 61)
    z = omega + 0.05j
    for spin in (0, 1):
        res = greens.greens_function(toy["system"], toy["H"], toy["up"], toy["dn"], toy["c"], toy["e0"], orbs, spin, omega, 0.05,
                                     max_steps=1000, eps_select=1e-12, select_rounds=10, tol=1e-10)
        for key, create in (("G_minus", False), ("G_plus", True)):
            nup = 2 + (0 if spin else (1 if create else -1))
            ndn = 2 + ((1 if create else -1) if spin else 0)
            su, sd, Hs = toy["dense"](nup, ndn)
            ru, rd, rphi = ref_ladder(u64_to_ints(toy["up"]), u64_to_ints(toy["dn"]), toy["c"], orbs, spin, create)
            index = {k: i for i, k in enumerate(zip(su, sd))}
            V = np.zeros((len(su), len(orbs)))
            for i, k in enumerate(zip(ru, rd)):
                V[index[k]] = rphi[i]
            M = sum_over_states(Hs, V, toy["e0"], z, create)
            want = M if not create else M.transpose(0, 2, 1)
            assert res[key].shape == (len(omega), len(orbs), len(orbs))
            assert np.max(np.abs(res[key] - want)) <= 1e-8
            assert np.all(res["steps_" + key[2:]] < 1000)
        A = greens.spectral_function(res["G_minus"] + res["G_plus"])
        assert np.all(np.diagonal(A, axis1=1, axis2=2) >= -1e-12)


def test_later_selection_rounds_widen_the_space(c2_space):
    """a round screens the determinants the previous one added, seeded with their first-order amplitudes"""
    sq = _sq()
    from sqmc_b200 import greens
    _, r = c2_space
    sysm = sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1)
    H = sq.SparseHamiltonian(sysm)
    w = _norm(r["wts"][:, 0])
    omega = np.linspace(-1.0, 0.5, 11)
    n = {}
    for rounds in (0, 1, 2):
        g = greens.greens_function(sysm, H, r["up"], r["dn"], w, -75.7, [3, 2], "b", omega, 0.1, max_steps=10,
                                   eps_select=None if rounds == 0 else 1e-5, select_rounds=max(rounds, 1))
        n[rounds] = (g["n_minus"], g["n_plus"])
        assert np.all(np.isfinite(g["G_minus"])) and np.all(np.isfinite(g["G_plus"]))
    assert n[0][0] < n[1][0] < n[2][0] and n[0][1] < n[1][1] < n[2][1]


def test_invariance_under_row_order_and_time_sym(c2_space_ts):
    sq = _sq()
    from sqmc_b200 import greens
    _, r = c2_space_ts
    w = _norm(np.random.default_rng(5).standard_normal(len(r["up"])))
    omega = np.linspace(-2.0, 1.0, 31)
    orbs = [3, 2, 8]
    sts = sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1)
    Hts = sq.SparseHamiltonian(sts)
    a = greens.greens_function(sts, Hts, r["up"], r["dn"], w, -75.6, orbs, "a", omega, 0.1, max_steps=40)
    perm = np.random.default_rng(6).permutation(len(w))
    b = greens.greens_function(sts, Hts, r["up"][perm], r["dn"][perm], w[perm], -75.6, orbs, "a", omega, 0.1, max_steps=40)
    for k in ("G_minus", "G_plus"):
        assert np.array_equal(a[k], b[k])
    eu, ed, ew = expand_time_sym(u64_to_ints(r["up"]), u64_to_ints(r["dn"]), w, 1)
    spl = sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1)
    c = greens.greens_function(spl, sq.SparseHamiltonian(spl), sq.dets_to_u64(eu), sq.dets_to_u64(ed), np.asarray(ew).reshape(-1), -75.6,
                               orbs, "a", omega, 0.1, max_steps=40)
    for k in ("G_minus", "G_plus"):
        assert np.max(np.abs(a[k] - c[k])) <= 1e-10 * max(1.0, np.max(np.abs(c[k])))
    assert a["n_minus"] == c["n_minus"] and a["n_plus"] == c["n_plus"]


def test_errors(c2_space, c2_space_ts, c2_minus):
    sq = _sq()
    from sqmc_b200 import greens
    from sqmc_b200._lib import SqmcError
    _, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = r["up"], r["dn"]
    w = r["wts"][:, 0].copy()
    L, h = H._L, H._h
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    orbs = np.array([1, 2], dtype=np.int32)
    nn = C.c_int64()

    def lad(n=len(up), ns=1, ldw=len(up), state=0, spin=0, create=0, norbs=2, o=orbs):
        from sqmc_b200._lib import check
        check(L.sqmc_b200_ladder(h, n, p(up), p(dn), ns, p(w), ldw, state, spin, create, norbs, p(o), C.byref(nn)))

    cases = [(dict(n=0), "n must be positive"), (dict(ns=0), "n_states must be >= 1"), (dict(ldw=5), r"ldw \(5\) must be >= n"),
             (dict(state=1), r"state 1 is not in \[0, 1\)"), (dict(spin=2), "spin must be 0"), (dict(norbs=0), "n_orbs must be >= 1"),
             (dict(o=np.array([1, 26], dtype=np.int32)), r"orbital 26 is not in \[0, 26\)"),
             (dict(o=np.array([3, 3], dtype=np.int32)), "orbital 3 is listed twice")]
    for kw, msg in cases:
        with pytest.raises(SqmcError, match=msg):
            lad(**kw)
    with pytest.raises(SqmcError, match="ladder: null argument"):
        _sq()._lib.check(L.sqmc_b200_ladder(h, len(up), None, p(dn), 1, p(w), len(up), 0, 0, 0, 2, p(orbs), C.byref(nn)))
    lad()
    buf = np.zeros((nn.value, 2), dtype=np.uint64)
    with pytest.raises(SqmcError, match="ldc .* must be >= the number of images"):
        _sq()._lib.check(L.sqmc_b200_ladder_result(h, p(buf), p(buf), p(np.zeros(2 * nn.value)), nn.value - 1))
    with pytest.raises(SqmcError, match="ladder_result: null argument"):
        _sq()._lib.check(L.sqmc_b200_ladder_result(h, None, p(buf), p(np.zeros(2 * nn.value)), nn.value))
    with pytest.raises(SqmcError, match="holds a determinant twice"):
        H.ladder(np.concatenate([up, up[:1]]), np.concatenate([dn, dn[:1]]), np.concatenate([w, w[:1]]), [1], 0, False)
    _, rt = c2_space_ts
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    k = int(np.flatnonzero(np.any(rt["up"] != rt["dn"], axis=1))[0])
    with pytest.raises(SqmcError, match="time-reversed partner"):
        Hts.ladder(np.concatenate([rt["up"], rt["dn"][k:k + 1]]), np.concatenate([rt["dn"], rt["up"][k:k + 1]]),
                   np.ones(len(rt["up"]) + 1), [1], 0, False)
    # empty / full spin strings: 4 alpha electrons and no beta on C2; all 4 orbitals filled on a 2x2 Hubbard lattice
    H40 = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, nelec=4, nup=4, time_sym=False, z=1))
    with pytest.raises(SqmcError, match="cannot annihilate from an empty dn string"):
        H40.ladder(sq.dets_to_u64([15]), sq.dets_to_u64([0]), [1.0], [0], 1, False)
    Hh = sq.SparseHamiltonian(sq.HubbardKSystem(2, 2, 1.0, 4.0, 4, 1))
    with pytest.raises(SqmcError, match="cannot create into a full up string"):
        Hh.ladder(sq.dets_to_u64([15]), sq.dets_to_u64([1]), [1.0], [0], 0, True)
    # tridiagonal Lanczos
    HX, phi = c2_minus
    with pytest.raises(SqmcError, match="no matrix on this handle"):   # H has never built a matrix
        _sq()._lib.check(L.sqmc_b200_lanczos_tridiagonal(h, 1, p(np.ones(4)), 4, 5, 0.0, p(np.zeros(5)), p(np.zeros(5)), p(np.zeros(5)),
                                                         p(np.zeros(1, dtype=np.int32))))
    v = np.ascontiguousarray(phi[:, 0])
    out = [np.zeros(64), np.zeros(64), np.zeros(64), np.zeros(2, dtype=np.int32)]

    def lz(nv=1, ldv=HX.n, ms=5, tol=0.0, vec=v):
        _sq()._lib.check(L.sqmc_b200_lanczos_tridiagonal(HX._h, nv, p(vec), ldv, ms, tol, *[p(o) for o in out]))

    for kw, msg in [(dict(nv=0), "nvec must be >= 1"), (dict(ldv=HX.n - 1), r"ldv \(\d+\) must be >= n"), (dict(ms=0), "max_steps must be >= 1"),
                    (dict(tol=-1.0), "tol must be >= 0"), (dict(vec=np.zeros(HX.n)), "start vector 0 has zero norm")]:
        with pytest.raises(SqmcError, match=msg):
            lz(**kw)
    with pytest.raises(SqmcError, match="lanczos_tridiagonal: null argument"):
        _sq()._lib.check(L.sqmc_b200_lanczos_tridiagonal(HX._h, 1, None, HX.n, 5, 0.0, *[p(o) for o in out]))
    with pytest.raises(ValueError, match="V0 has"):
        HX.lanczos_tridiagonal(np.ones(HX.n + 1), 5)
    # a basis that cannot fit: a diagonal matrix of 200000 rows and a Krylov basis of 200000 vectors (640 GB)
    Hbig = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    nbig = 200000
    Hbig.import_upper(np.ones(nbig, dtype=np.int64), np.arange(1, nbig + 1, dtype=np.int64), np.linspace(1.0, 2.0, nbig))
    with pytest.raises(SqmcError, match="the Krylov basis needs .* GB .* lower max_steps"):
        Hbig.lanczos_tridiagonal(np.ones((nbig, 3)), nbig)
    # Python-side arguments of the driver
    with pytest.raises(ValueError, match="spin must be"):
        greens.greens_function(H.system, H, up, dn, w, 0.0, [1], "c", [0.0], 0.1)
    with pytest.raises(ValueError, match="chem systems"):
        greens.greens_function(Hh.system, Hh, sq.dets_to_u64([3]), sq.dets_to_u64([1]), [1.0], 0.0, [1], 0, [0.0], 0.1)
    with pytest.raises(ValueError, match="max_steps must be >= 1"):
        greens.greens_function(H.system, H, up, dn, w, 0.0, [1], 0, [0.0], 0.1, max_steps=0)
