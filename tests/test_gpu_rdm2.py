"""Two-particle density matrix on the device (csrc/rdm.cu, SparseHamiltonian.two_rdm), <S^2> and the RDM energy."""
import ctypes as C
import itertools

import numpy as np
import pytest

from conftest import C2_FCIDUMP
from rdm2_reference import two_rdm as ref_two_rdm
from test_natorb_host import fci_dets, write_toy_fcidump

pytestmark = pytest.mark.gpu


def _sq():
    import sqmc_b200 as sq
    return sq


def _norm(w):
    w = np.asarray(w, dtype=np.float64)
    return w / np.linalg.norm(w, axis=0)


def _structure(g, same_spin_zero=True):
    """exact index symmetries of [.., b, p, q, r, s]"""
    g = g.reshape((-1, 3) + g.shape[-4:])
    assert np.array_equal(g, g.transpose(0, 1, 3, 2, 5, 4))          # Gamma_pq,rs = Gamma_qp,sr
    for b in (0, 2):
        x = g[:, b]
        assert np.array_equal(x, x.transpose(0, 3, 4, 1, 2))         # Gamma_pq,rs = Gamma_rs,pq
        assert np.array_equal(x, -x.transpose(0, 1, 4, 3, 2))        # Gamma_pq,rs = -Gamma_ps,rq
        n = x.shape[-1]
        e = np.eye(n, dtype=bool)
        assert np.all(x[:, e[:, None, :, None] * np.ones((n, n, n, n), bool)] == 0)   # p = r
        assert np.all(x[:, e[None, :, None, :] * np.ones((n, n, n, n), bool)] == 0)   # q = s


def _check(H, up, dn, w, norb, time_sym=False, z=1, zeros_exact=False):
    got = H.two_rdm(up, dn, w)
    ref = ref_two_rdm(up, dn, w, norb, time_sym=time_sym, z=z)
    ref = ref[0] if np.ndim(w) == 1 else ref
    assert got.shape == ref.shape
    assert np.max(np.abs(got - ref)) <= 1e-13
    _structure(got)
    if zeros_exact:   # no term reaches these slots (momentum conservation in heg / hubbardk): exactly 0 on the device too
        assert np.all(got[ref == 0] == 0)
    return got


def _subset(r, m, seed):
    rng = np.random.default_rng(seed)
    k = np.sort(rng.choice(len(r["up"]), m, replace=False))
    return r["up"][k], r["dn"][k]


def _list53(sq, n, seed):
    rng = np.random.default_rng(seed)
    ups = [sum(1 << k for k in c) for c in itertools.combinations(range(10), 5)]
    dns = [sum(1 << k for k in c) for c in itertools.combinations(range(9), 3)]
    pairs = [(u, d) for u in ups for d in dns]
    sel = rng.choice(len(pairs), n, replace=False)
    return sq.dets_to_u64([pairs[k][0] for k in sel]), sq.dets_to_u64([pairs[k][1] for k in sel])


def test_c2_plain_time_sym_and_two_states(c2_space, c2_space_ts):
    sq = _sq()
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = _subset(c2_space[1], 300, 1)
    rng = np.random.default_rng(1)
    _check(H, up, dn, _norm(rng.standard_normal(len(up))), 26)
    g2 = _check(H, up, dn, _norm(rng.standard_normal((len(up), 2))), 26)
    assert g2.shape == (2, 3, 26, 26, 26, 26)
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    up, dn = _subset(c2_space_ts[1], 300, 2)
    _check(Hts, up, dn, _norm(rng.standard_normal(len(up))), 26, time_sym=True, z=1)


def test_c2_nup_ne_ndn():
    sq = _sq()
    H53 = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, nelec=8, nup=5, time_sym=False, z=1))
    up, dn = _list53(sq, 400, 3)
    _check(H53, up, dn, _norm(np.random.default_rng(3).standard_normal(len(up))), 26)


def test_heg_subset_and_hubbardk_sector(heg_space):
    sq = _sq()
    from sqmc_b200 import spaces
    S, r = heg_space
    H = sq.SparseHamiltonian(sq.HegSystem(3, 0.5, 14, 7, 1.49))
    up, dn = _subset(r, 250, 4)
    _check(H, up, dn, _norm(np.random.default_rng(4).standard_normal(len(up))), S.norb, zeros_exact=True)
    hub = sq.HubbardKSystem(4, 2, 1.0, 4.0, 3, 2)
    up, dn, _ = spaces.hubbard_momentum_sector(hub)
    Hh = sq.SparseHamiltonian(hub)
    _check(Hh, up, dn, _norm(np.random.default_rng(5).standard_normal(len(up))), 8, zeros_exact=True)


@pytest.mark.parametrize("case", ["c2", "c2_ts", "heg"])
def test_partial_traces_against_one_rdm(c2_space, c2_space_ts, heg_space, case):
    sq = _sq()
    if case == "heg":
        S, r = heg_space
        system, nup, ndn = sq.HegSystem(3, 0.5, 14, 7, 1.49), 7, 7
    else:
        r = (c2_space_ts if case == "c2_ts" else c2_space)[1]
        system, nup, ndn = sq.ChemSystem(C2_FCIDUMP, time_sym=case == "c2_ts", z=1), 4, 4
    H = sq.SparseHamiltonian(system)
    w = _norm(np.random.default_rng(6).standard_normal(len(r["up"])))
    g1 = H.one_rdm(r["up"], r["dn"], w)
    g2 = H.two_rdm(r["up"], r["dn"], w)
    tol = 1e-11
    assert np.max(np.abs(np.einsum("pqrr->pq", g2[0]) - (nup - 1) * g1[0])) <= tol
    assert np.max(np.abs(np.einsum("pqrr->pq", g2[2]) - (ndn - 1) * g1[1])) <= tol
    assert np.max(np.abs(np.einsum("pqrr->pq", g2[1]) - ndn * g1[0])) <= tol
    assert np.max(np.abs(np.einsum("pprs->rs", g2[1]) - nup * g1[1])) <= tol


def _random_eri_system(sq, rng, **kw):
    """ChemSystem whose integrals are random 8-fold symmetric (pq|rs) in library numbering, h = 0 and enuc = 0"""
    from sqmc_b200 import rdm
    sysm = sq.ChemSystem(C2_FCIDUMP, **kw)
    n = sysm.norb
    g = rng.standard_normal((n, n, n, n))
    g = g + g.transpose(1, 0, 2, 3)
    g = g + g.transpose(0, 1, 3, 2)
    g = g + g.transpose(2, 3, 0, 1)
    c2 = np.asarray(sysm._c2, dtype=np.int64)[:n, :n]
    a, b = c2[:, :, None, None], c2[None, None, :, :]
    idx = np.maximum(a, b) * (np.maximum(a, b) - 1) // 2 + np.minimum(a, b)
    ints = np.zeros_like(sysm.integrals)
    ints[idx - 1] = g
    sysm.integrals = ints
    h, eri, enuc = rdm.integrals_library_order(sysm)
    assert np.array_equal(eri, g) and not h.any() and enuc == 0.0
    return sysm, g


@pytest.mark.parametrize("case", ["plain", "time_sym", "nup5_ndn3"])
def test_energy_identity_random_integrals(c2_space, c2_space_ts, case):
    """w.Hw of the library's own build with random (pq|rs) equals 1/2 sum g Gamma"""
    sq = _sq()
    rng = np.random.default_rng(21 + len(case))
    if case == "nup5_ndn3":
        kw = dict(nelec=8, nup=5, time_sym=False, z=1)
        up, dn = _list53(sq, 2000, 7)
    else:
        kw = dict(time_sym=case == "time_sym", z=1)
        up, dn = _subset((c2_space_ts if case == "time_sym" else c2_space)[1], 2000, 8)
    sysm, g = _random_eri_system(sq, rng, **kw)
    H = sq.SparseHamiltonian(sysm)
    w = _norm(rng.standard_normal(len(up)))
    H.generate_sparse_ham_upper_triangular(up, dn)
    e = float(w @ H.matvec(w))
    G = H.two_rdm(up, dn, w)
    e2 = 0.5 * float(np.sum(g * (G[0] + 2.0 * G[1] + G[2])))
    assert abs(e - e2) <= 1e-10 * max(1.0, abs(e))


def test_rdm_energy_of_ground_state(c2_space):
    sq = _sq()
    from sqmc_b200 import rdm
    _, r = c2_space
    sysm = sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1)
    H = sq.SparseHamiltonian(sysm)
    H.generate_sparse_ham_upper_triangular(r["up"], r["dn"])
    d = H.davidson_sparse(n_states=1)
    c, e0 = d["evecs"][:, 0], d["evals"][0]
    e = rdm.rdm_energy(sysm, H.one_rdm(r["up"], r["dn"], c), H.two_rdm(r["up"], r["dn"], c))
    assert abs(e - e0) <= 1e-9


def test_spin_squared_toy_fci(tmp_path):
    sq = _sq()
    from sqmc_b200 import rdm
    toy = str(tmp_path / "FCIDUMP")
    write_toy_fcidump(toy)
    sysm = sq.ChemSystem(toy)
    H = sq.SparseHamiltonian(sysm)
    up, dn = fci_dets(sysm.norb, sysm.nup, sysm.ndn)
    up, dn = sq.dets_to_u64(up), sq.dets_to_u64(dn)
    H.generate_sparse_ham_upper_triangular(up, dn)
    cnt, idx, val = H.export_upper()
    M = np.zeros((len(cnt), len(cnt)))
    M[np.repeat(np.arange(len(cnt)), cnt), idx - 1] = val
    M = M + np.triu(M, 1).T
    ev, vec = np.linalg.eigh(M)
    keep = [k for k in range(12) if min(abs(ev[k] - ev[k - 1]) if k else 1.0, abs(ev[k + 1] - ev[k])) > 1e-6][:8]
    s2 = rdm.spin_squared(H.two_rdm(up, dn, vec[:, keep]), sysm.nup, sysm.ndn)
    spins = np.round((np.sqrt(1.0 + 4.0 * s2) - 1.0) / 2.0)
    assert np.max(np.abs(s2 - spins * (spins + 1))) <= 1e-9
    assert 0 in spins and 1 in spins


def test_determinism_scaling_and_resident_matrix(c2_space):
    sq = _sq()
    _, r = c2_space
    up, dn = r["up"], r["dn"]
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    H.generate_sparse_ham_upper_triangular(up, dn)
    rng = np.random.default_rng(9)
    x = rng.standard_normal(len(up))
    y0 = H.matvec(x)
    w = rng.standard_normal((len(up), 2))
    a = H.two_rdm(up, dn, w)
    assert np.array_equal(a, H.two_rdm(up, dn, w))
    p = rng.permutation(len(up))
    assert np.array_equal(a, H.two_rdm(up[p], dn[p], w[p]))
    b = H.two_rdm(up, dn, w[:, 0] * 1e6)
    assert np.max(np.abs(b - 1e12 * a[0])) <= 1e-15 * np.max(np.abs(b))
    assert np.array_equal(H.matvec(x), y0)


def test_input_errors(c2_space, c2_space_ts):
    sq = _sq()
    from sqmc_b200 import _lib
    _, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = r["up"][:50], r["dn"][:50]
    w = np.ones(len(up))
    with pytest.raises(sq.SqmcError, match="twice"):
        H.two_rdm(np.concatenate([up, up[:1]]), np.concatenate([dn, dn[:1]]), np.ones(len(up) + 1))
    with pytest.raises(sq.SqmcError, match="n_states"):
        H.two_rdm(up, dn, np.zeros((len(up), 0)))
    with pytest.raises(sq.SqmcError, match="n must be positive"):
        H.two_rdm(up[:0], dn[:0], w[:0])
    out = np.zeros((1, 3) + (26,) * 4)
    with pytest.raises(sq.SqmcError, match="ldw"):
        _lib.check(H._L.sqmc_b200_two_rdm(H._h, len(up), up.ctypes.data_as(C.c_void_p), dn.ctypes.data_as(C.c_void_p), 1,
                                        w.ctypes.data_as(C.c_void_p), len(up) - 1, out.ctypes.data_as(C.c_void_p)))
    with pytest.raises(sq.SqmcError, match="electrons"):
        H.two_rdm(np.concatenate([up, sq.dets_to_u64([0b111])]), np.concatenate([dn, sq.dets_to_u64([0b1111])]), np.ones(len(up) + 1))
    _, rt = c2_space_ts
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    k = next(i for i in range(len(rt["up"])) if not np.array_equal(rt["up"][i], rt["dn"][i]))
    with pytest.raises(sq.SqmcError, match="time-reversed partner"):
        Hts.two_rdm(np.concatenate([rt["up"], rt["dn"][k:k + 1]]), np.concatenate([rt["dn"], rt["up"][k:k + 1]]), np.ones(len(rt["up"]) + 1))
    hs = sq.HegSystem(3, 0.5, 14, 7, 2.5)
    assert hs.norb == 81
    Hh = sq.SparseHamiltonian(hs)
    with pytest.raises(sq.SqmcError, match=r"3\*norb\^4"):
        Hh.two_rdm(sq.dets_to_u64([hs.hf_up]), sq.dets_to_u64([hs.hf_dn]), np.ones(1))
