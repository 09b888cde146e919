"""Transition density matrices on the device (csrc/rdm.cu, SparseHamiltonian.transition_one_rdm / transition_two_rdm)."""
import ctypes as C
import itertools

import numpy as np
import pytest

from conftest import C2_FCIDUMP
from tdm_reference import transition_one_rdm as ref_t1, transition_two_rdm as ref_t2
from test_natorb_host import fci_dets, write_toy_fcidump

pytestmark = pytest.mark.gpu


def _sq():
    import sqmc_b200 as sq
    return sq


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


def _same_spin_structure(g):
    """the index symmetries a transition 2-RDM keeps, exactly: same spin Gamma_pq,rs = Gamma_rs,pq = -Gamma_ps,rq, 0 at p = r, q = s"""
    g = g.reshape((-1, 3) + g.shape[-4:])
    for b in (0, 2):
        x = g[:, b]
        assert np.array_equal(x, x.transpose(0, 3, 4, 1, 2))
        assert np.array_equal(x, -x.transpose(0, 1, 4, 3, 2))
        n = x.shape[-1]
        e = np.eye(n, dtype=bool)
        assert np.all(x[:, e[:, None, :, None] * np.ones((n, n, n, n), bool)] == 0)
        assert np.all(x[:, e[None, :, None, :] * np.ones((n, n, n, n), bool)] == 0)


def _check(H, up, dn, a, b, norb, time_sym=False, z=1, zeros_exact=False):
    t1 = H.transition_one_rdm(up, dn, a, b)
    t2 = H.transition_two_rdm(up, dn, a, b)
    r1 = ref_t1(up, dn, a, b, norb, time_sym=time_sym, z=z)
    r2 = ref_t2(up, dn, a, b, norb, time_sym=time_sym, z=z)
    if np.ndim(a) == 1:
        r1, r2 = r1[0], r2[0]
    assert t1.shape == r1.shape and t2.shape == r2.shape
    assert np.max(np.abs(t1 - r1)) <= 1e-13
    assert np.max(np.abs(t2 - r2)) <= 1e-13
    n0 = r2.ndim - 4
    assert np.max(np.abs(r2 - r2.transpose(tuple(range(n0)) + (n0 + 1, n0, n0 + 3, n0 + 2)))) > 1e-6   # not Hermitian: a real test
    _same_spin_structure(t2)
    if zeros_exact:   # no term reaches these slots (momentum conservation): exactly 0 on the device too
        assert np.all(t1[r1 == 0] == 0)
        assert np.all(t2[r2 == 0] == 0)


def _vectors(rng, n, k):
    """random, unnormalised, not orthogonal: b shares a component with a"""
    shape = (n,) if k == 1 else (n, k)
    a = rng.standard_normal(shape)
    return a, 0.5 * a + rng.standard_normal(shape)


@pytest.mark.parametrize("k", [1, 3])
def test_c2_against_definition(c2_space, c2_space_ts, k):
    sq = _sq()
    rng = np.random.default_rng(30 + k)
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = _subset(c2_space[1], 200, 31)
    _check(H, up, dn, *_vectors(rng, len(up), k), 26)
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    up, dn = _subset(c2_space_ts[1], 200, 32)
    _check(Hts, up, dn, *_vectors(rng, len(up), k), 26, time_sym=True, z=1)


def test_c2_nup_ne_ndn():
    sq = _sq()
    H53 = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, nelec=8, nup=5, time_sym=False, z=1))
    up, dn = _list53(sq, 300, 33)
    rng = np.random.default_rng(33)
    _check(H53, up, dn, *_vectors(rng, len(up), 1), 26)
    _check(H53, up, dn, *_vectors(rng, len(up), 3), 26)


def test_heg_subset_and_hubbardk_sector(heg_space):
    sq = _sq()
    from sqmc_b200 import spaces
    S, r = heg_space
    rng = np.random.default_rng(34)
    H = sq.SparseHamiltonian(sq.HegSystem(3, 0.5, 14, 7, 1.49))
    up, dn = _subset(r, 150, 34)
    _check(H, up, dn, *_vectors(rng, len(up), 1), S.norb, zeros_exact=True)
    hub = sq.HubbardKSystem(4, 2, 1.0, 4.0, 3, 2)
    up, dn, _ = spaces.hubbard_momentum_sector(hub)
    Hh = sq.SparseHamiltonian(hub)
    _check(Hh, up, dn, *_vectors(rng, len(up), 3), 8, zeros_exact=True)


@pytest.mark.parametrize("time_sym", [False, True])
def test_reduces_to_one_and_two_rdm(c2_space, c2_space_ts, time_sym):
    sq = _sq()
    r = (c2_space_ts if time_sym else c2_space)[1]
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=time_sym, z=1))
    rng = np.random.default_rng(35 + time_sym)
    for c in (rng.standard_normal(len(r["up"])), rng.standard_normal((len(r["up"]), 2))):
        assert np.array_equal(H.transition_one_rdm(r["up"], r["dn"], c, c), H.one_rdm(r["up"], r["dn"], c))
        assert np.array_equal(H.transition_two_rdm(r["up"], r["dn"], c, c), H.two_rdm(r["up"], r["dn"], c))


def test_one_tdm_beyond_64_orbitals():
    """the 1-TDM has no orbital limit: two-word strings (HEG, 81 orbitals) against the definition and one_rdm"""
    sq = _sq()
    hs = sq.HegSystem(3, 0.5, 14, 7, 2.5)
    assert hs.norb == 81
    H = sq.SparseHamiltonian(hs)
    r = H.get_next_det_list(sq.dets_to_u64([hs.hf_up]), sq.dets_to_u64([hs.hf_dn]), np.ones(1), np.full(1, 9e99), 1e-3)
    up = np.concatenate([sq.dets_to_u64([hs.hf_up]), r[0][:150]])
    dn = np.concatenate([sq.dets_to_u64([hs.hf_dn]), r[1][:150]])
    rng = np.random.default_rng(36)
    a, b = _vectors(rng, len(up), 2)
    t1 = H.transition_one_rdm(up, dn, a, b)
    assert np.max(np.abs(t1 - ref_t1(up, dn, a, b, 81))) <= 1e-13
    assert np.array_equal(H.transition_one_rdm(up, dn, a, a), H.one_rdm(up, dn, a))


def test_hermiticity_and_determinism(c2_space, c2_space_ts):
    sq = _sq()
    for time_sym, r in ((False, c2_space[1]), (True, c2_space_ts[1])):
        up, dn = r["up"], r["dn"]
        H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=time_sym, z=1))
        rng = np.random.default_rng(37 + time_sym)
        a, b = _vectors(rng, len(up), 2)
        t1, t2 = H.transition_one_rdm(up, dn, a, b), H.transition_two_rdm(up, dn, a, b)
        assert np.array_equal(H.transition_one_rdm(up, dn, b, a), t1.transpose(0, 1, 3, 2))
        assert np.array_equal(H.transition_two_rdm(up, dn, b, a), t2.transpose(0, 1, 3, 2, 5, 4))
        assert np.array_equal(H.transition_one_rdm(up, dn, a, b), t1)
        assert np.array_equal(H.transition_two_rdm(up, dn, a, b), t2)
        p = rng.permutation(len(up))
        assert np.array_equal(H.transition_one_rdm(up[p], dn[p], a[p], b[p]), t1)
        assert np.array_equal(H.transition_two_rdm(up[p], dn[p], a[p], b[p]), t2)
        _same_spin_structure(t2)


@pytest.mark.parametrize("time_sym", [False, True])
def test_energy_identity(c2_space, c2_space_ts, time_sym):
    """<a|H|b> from the transition matrices equals a . (H b) from the resident matrix"""
    sq = _sq()
    from sqmc_b200 import rdm
    r = (c2_space_ts if time_sym else c2_space)[1]
    up, dn = r["up"], r["dn"]
    chem = sq.ChemSystem(C2_FCIDUMP, time_sym=time_sym, z=1)
    H = sq.SparseHamiltonian(chem)
    H.generate_sparse_ham_upper_triangular(up, dn)
    rng = np.random.default_rng(39 + time_sym)
    a, b = _vectors(rng, len(up), 1)
    e = rdm.rdm_energy(chem, H.transition_one_rdm(up, dn, a, b), H.transition_two_rdm(up, dn, a, b))
    assert abs(e - float(a @ H.matvec(b))) <= 1e-10 * np.linalg.norm(a) * np.linalg.norm(b)
    ovl = np.trace(H.transition_one_rdm(up, dn, a, b).sum(axis=0)) / (chem.nup + chem.ndn)
    assert abs(ovl - float(a @ b)) <= 1e-12 * np.linalg.norm(a) * np.linalg.norm(b)


def test_spin_and_hamiltonian_over_toy_fci_states(tmp_path):
    sq = _sq()
    from sqmc_b200 import rdm
    toy = str(tmp_path / "FCIDUMP")
    write_toy_fcidump(toy)
    sysm = sq.ChemSystem(toy)
    H = sq.SparseHamiltonian(sysm)
    up, dn = fci_dets(sysm.norb, sysm.nup, sysm.ndn)
    up, dn = sq.dets_to_u64(up), sq.dets_to_u64(dn)
    assert len(up) == 2025
    H.generate_sparse_ham_upper_triangular(up, dn)
    cnt, idx, val = H.export_upper()
    M = np.zeros((len(cnt), len(cnt)))
    M[np.repeat(np.arange(len(cnt)), cnt), idx - 1] = val
    M = M + np.triu(M, 1).T
    ev, vec = np.linalg.eigh(M)
    ns = 6
    I, J = np.meshgrid(np.arange(ns), np.arange(ns), indexing="ij")
    bra, ket = vec[:, I.ravel()], vec[:, J.ravel()]
    t1 = H.transition_one_rdm(up, dn, bra, ket)
    t2 = H.transition_two_rdm(up, dn, bra, ket)
    nel = sysm.nup + sysm.ndn
    ovl = np.array([np.trace(t1[k, 0] + t1[k, 1]) / nel for k in range(ns * ns)]).reshape(ns, ns)
    h = np.array([rdm.rdm_energy(sysm, t1[k], t2[k]) for k in range(ns * ns)]).reshape(ns, ns)
    s2 = np.array([rdm.spin_squared(t2[k], sysm.nup, sysm.ndn, ovl.ravel()[k]) for k in range(ns * ns)]).reshape(ns, ns)
    assert np.max(np.abs(ovl - np.eye(ns))) <= 1e-12
    assert np.max(np.abs(h - np.diag(ev[:ns]))) <= 1e-9
    assert np.max(np.abs(s2 - np.diag(np.diag(s2)))) <= 1e-9
    d = np.diag(s2)
    assert np.max(np.min(np.abs(d[:, None] - np.array([0.0, 2.0, 6.0])[None, :]), axis=1)) <= 1e-9


def test_input_errors(c2_space, c2_space_ts):
    sq = _sq()
    from sqmc_b200 import _lib
    _, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = r["up"][:50], r["dn"][:50]
    w = np.ones(len(up))
    for f in (H.transition_one_rdm, H.transition_two_rdm):
        with pytest.raises(ValueError, match="same shape"):
            f(up, dn, w, np.ones((len(up), 2)))
        with pytest.raises(sq.SqmcError, match="n_pairs"):
            f(up, dn, np.zeros((len(up), 0)), np.zeros((len(up), 0)))
        with pytest.raises(sq.SqmcError, match="twice"):
            f(np.concatenate([up, up[:1]]), np.concatenate([dn, dn[:1]]), np.ones(len(up) + 1), np.ones(len(up) + 1))
    for fn, size in ((H._L.sqmc_b200_transition_one_rdm, 2 * 26 * 26), (H._L.sqmc_b200_transition_two_rdm, 3 * 26 ** 4)):
        out = np.zeros(size)
        with pytest.raises(sq.SqmcError, match="ldw"):
            _lib.check(fn(H._h, len(up), up.ctypes.data_as(C.c_void_p), dn.ctypes.data_as(C.c_void_p), 1, w.ctypes.data_as(C.c_void_p),
                          w.ctypes.data_as(C.c_void_p), len(up) - 1, out.ctypes.data_as(C.c_void_p)))
    _, rt = c2_space_ts
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    k = next(i for i in range(len(rt["up"])) if not np.array_equal(rt["up"][i], rt["dn"][i]))
    upt, dnt = np.concatenate([rt["up"], rt["dn"][k:k + 1]]), np.concatenate([rt["dn"], rt["up"][k:k + 1]])
    wt = np.ones(len(upt))
    for f in (Hts.transition_one_rdm, Hts.transition_two_rdm):
        with pytest.raises(sq.SqmcError, match="time-reversed partner"):
            f(upt, dnt, wt, wt)
    hs = sq.HegSystem(3, 0.5, 14, 7, 2.5)
    Hh = sq.SparseHamiltonian(hs)
    with pytest.raises(sq.SqmcError, match=r"3\*norb\^4"):
        Hh.transition_two_rdm(sq.dets_to_u64([hs.hf_up]), sq.dets_to_u64([hs.hf_dn]), np.ones(1), np.ones(1))
