"""One-particle density matrix on the device (csrc/rdm.cu, SparseHamiltonian.one_rdm) and natural orbitals end to end."""
import itertools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import C2_FCIDUMP, ROOT
from rdm_reference import expand_time_sym, one_rdm as ref_rdm, u64_to_ints
from test_natorb_host import fci_dets, write_toy_fcidump

pytestmark = pytest.mark.gpu


def _sq():
    import sqmc_b200 as sq
    return sq


def _norm(w):
    w = np.asarray(w, dtype=np.float64)
    return w / np.linalg.norm(w, axis=0)


def _check(H, up, dn, w, norb, time_sym=False, z=1):
    got = H.one_rdm(up, dn, w)
    ref = ref_rdm(up, dn, w, norb, time_sym=time_sym, z=z)
    ref = ref[0] if np.ndim(w) == 1 else ref
    assert got.shape == ref.shape
    assert np.max(np.abs(got - ref)) <= 1e-12
    return got


def _invariants(g, nup, ndn, norm2, offdiag_zero=False, time_sym=False):
    g = g.reshape(-1, 2, g.shape[-2], g.shape[-1])
    for s in range(g.shape[0]):
        assert abs(np.trace(g[s, 0]) - nup * norm2[s]) <= 1e-11
        assert abs(np.trace(g[s, 1]) - ndn * norm2[s]) <= 1e-11
        for sig in (0, 1):
            assert np.array_equal(g[s, sig], g[s, sig].T)
            ev = np.linalg.eigvalsh(g[s, sig] / norm2[s])
            assert ev.min() >= -1e-12 and ev.max() <= 1 + 1e-12
            if offdiag_zero:
                assert np.array_equal(g[s, sig], np.diag(np.diag(g[s, sig])))
        if time_sym:
            assert np.max(np.abs(g[s, 0] - g[s, 1])) <= 1e-13


def test_c2_plain_and_nup_ne_ndn(c2_space):
    sq = _sq()
    _, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    rng = np.random.default_rng(1)
    w = _norm(rng.standard_normal(len(r["up"])))
    g = _check(H, r["up"], r["dn"], w, 26)
    _invariants(g, 4, 4, [1.0])
    g = _check(H, r["up"], r["dn"], r["wts"][:, 0], 26)
    # nup != ndn: 5 alpha + 3 beta electrons, random list
    H53 = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, nelec=8, nup=5, time_sym=False, z=1))
    ups = [sum(1 << k for k in c) for c in itertools.combinations(range(10), 5)]
    dns = [sum(1 << k for k in c) for c in itertools.combinations(range(9), 3)]
    pairs = [(u, d) for u in ups for d in dns]
    sel = rng.choice(len(pairs), 3000, replace=False)
    up = sq.dets_to_u64([pairs[k][0] for k in sel])
    dn = sq.dets_to_u64([pairs[k][1] for k in sel])
    w = _norm(rng.standard_normal(len(up)))
    g = _check(H53, up, dn, w, 26)
    _invariants(g, 5, 3, [1.0])


def test_c2_time_sym(c2_space_ts):
    sq = _sq()
    _, r = c2_space_ts
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    w = _norm(np.random.default_rng(2).standard_normal(len(r["up"])))
    g = _check(H, r["up"], r["dn"], w, 26, time_sym=True, z=1)
    _invariants(g, 4, 4, [1.0], time_sym=True)


def test_c2_two_states(oracle):
    sq = _sq()
    S = oracle.System.chem(C2_FCIDUMP, 26, 8, 4, [1, 5, 3, 2, 1, 7, 6, 5, 1, 2, 3, 1, 6, 7, 5, 4, 1, 5, 3, 2, 8, 5, 1, 7, 6, 5], hf_symmetry=1)
    r = S.hci(2e-3, n_states=2, max_iters=3)
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    w = _norm(r["wts"][:, :2])
    g = _check(H, r["up"], r["dn"], w, 26)
    assert g.shape == (2, 2, 26, 26)
    _invariants(g, 4, 4, [1.0, 1.0])
    # each state equals its own one-state call
    for s in range(2):
        assert np.max(np.abs(H.one_rdm(r["up"], r["dn"], w[:, s]) - g[s])) <= 1e-13


def test_heg_9475(heg_space):
    sq = _sq()
    S, r = heg_space
    H = sq.SparseHamiltonian(sq.HegSystem(3, 0.5, 14, 7, 1.49))
    w = _norm(r["wts"][:, 0])
    g = _check(H, r["up"], r["dn"], w, S.norb)
    _invariants(g, 7, 7, [1.0], offdiag_zero=True)


def test_heg_two_word_strings():
    sq = _sq()
    from sqmc_b200 import spaces
    hs = sq.HegSystem(3, 0.5, 14, 7, 2.5)
    assert hs.norb == 81
    H = sq.SparseHamiltonian(hs)
    up, dn, wts, _ = spaces.hci_space(H, hs, 4000, eps_schedule=(1e-2, 3e-3))
    assert len(up) > 1   # norb > 64: the strings are two words whatever orbitals are occupied
    w = _norm(wts[:, 0])
    g = _check(H, up, dn, w, 81)
    _invariants(g, 7, 7, [1.0], offdiag_zero=True)


def test_hubbardk_nup_ne_ndn():
    sq = _sq()
    from sqmc_b200 import spaces
    hub = sq.HubbardKSystem(4, 2, 1.0, 4.0, 3, 2)
    up, dn, _ = spaces.hubbard_momentum_sector(hub)
    H = sq.SparseHamiltonian(hub)
    w = _norm(np.random.default_rng(3).standard_normal(len(up)))
    g = _check(H, up, dn, w, 8)
    _invariants(g, 3, 2, [1.0], offdiag_zero=True)


@pytest.mark.parametrize("time_sym", [False, True])
def test_one_body_energy_through_build(c2_space, c2_space_ts, time_sym):
    """E1 = c^T H1 c with H1 the library's own Hamiltonian of a random one-body operator equals sum h gamma"""
    sq = _sq()
    _, r = c2_space_ts if time_sym else c2_space
    rng = np.random.default_rng(11 + time_sym)
    base = sq.ChemSystem(C2_FCIDUMP, time_sym=time_sym, z=1)
    norb, n1 = base.norb, base.norb + 1
    w = _norm(rng.standard_normal(len(r["up"])))
    g = sq.SparseHamiltonian(base).one_rdm(r["up"], r["dn"], w).sum(axis=0)   # spins summed, library numbering
    o = base.orb_order[:norb] - 1
    gf = np.zeros_like(g)
    gf[np.ix_(o, o)] = g
    for _ in range(3):
        h = rng.standard_normal((norb, norb))
        h = h + h.T   # FCIDUMP numbering
        sysm = sq.ChemSystem(C2_FCIDUMP, time_sym=time_sym, z=1)
        ints = np.zeros_like(sysm.integrals)
        for p in range(1, norb + 1):   # _index takes the reordered orbitals: library orbital p is FCIDUMP orbital o[p - 1] + 1
            for q in range(1, p + 1):
                ints[sysm._index(p, q, n1, n1) - 1] = h[o[p - 1], o[q - 1]]
        sysm.integrals = ints   # two-electron integrals and the core energy are 0
        H1 = sq.SparseHamiltonian(sysm)
        H1.generate_sparse_ham_upper_triangular(r["up"], r["dn"])
        e1 = float(w @ H1.matvec(w))
        assert abs(e1 - float(np.sum(h * gf))) <= 1e-10 * max(1.0, abs(e1))


def test_time_sym_expansion(c2_space_ts):
    sq = _sq()
    _, r = c2_space_ts
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    Hts.generate_sparse_ham_upper_triangular(r["up"], r["dn"])
    d = Hts.davidson_sparse(n_states=1)
    c, e_ts = d["evecs"][:, 0], d["evals"][0]
    eu, ed, ew = expand_time_sym(u64_to_ints(r["up"]), u64_to_ints(r["dn"]), c, 1)
    up, dn = sq.dets_to_u64(eu), sq.dets_to_u64(ed)
    Hp = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    Hp.generate_sparse_ham_upper_triangular(up, dn)
    x = ew[:, 0]
    assert abs(float(x @ Hp.matvec(x)) / float(x @ x) - e_ts) <= 1e-10
    a = Hp.one_rdm(up, dn, x)
    b = Hts.one_rdm(r["up"], r["dn"], c)
    assert np.max(np.abs(a - b)) <= 1e-13


def test_determinism(c2_space):
    sq = _sq()
    _, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    rng = np.random.default_rng(4)
    w = rng.standard_normal((len(r["up"]), 2))
    a = H.one_rdm(r["up"], r["dn"], w)
    assert np.array_equal(a, H.one_rdm(r["up"], r["dn"], w))
    p = rng.permutation(len(r["up"]))
    assert np.array_equal(a, H.one_rdm(r["up"][p], r["dn"][p], w[p]))


def test_input_errors(c2_space, c2_space_ts):
    sq = _sq()
    import ctypes as C
    from sqmc_b200 import _lib
    _, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = r["up"], r["dn"]
    w = np.ones(len(up))
    with pytest.raises(sq.SqmcError, match="twice"):
        H.one_rdm(np.concatenate([up, up[:1]]), np.concatenate([dn, dn[:1]]), np.ones(len(up) + 1))
    with pytest.raises(sq.SqmcError, match="n_states"):
        H.one_rdm(up, dn, np.zeros((len(up), 0)))
    out = np.zeros((1, 2, 26, 26))
    with pytest.raises(sq.SqmcError, match="ldw"):
        _lib.check(H._L.sqmc_b200_one_rdm(H._h, len(up), up.ctypes.data_as(C.c_void_p), dn.ctypes.data_as(C.c_void_p), 1,
                                        w.ctypes.data_as(C.c_void_p), len(up) - 1, out.ctypes.data_as(C.c_void_p)))
    _, rt = c2_space_ts
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    k = next(i for i in range(len(rt["up"])) if not np.array_equal(rt["up"][i], rt["dn"][i]))
    with pytest.raises(sq.SqmcError, match="time-reversed partner"):
        Hts.one_rdm(np.concatenate([rt["up"], rt["dn"][k:k + 1]]), np.concatenate([rt["dn"], rt["up"][k:k + 1]]), np.ones(len(rt["up"]) + 1))


def _fci_ground(sq, path):
    sysm = sq.ChemSystem(path)
    H = sq.SparseHamiltonian(sysm)
    up, dn = fci_dets(sysm.norb, sysm.nup, sysm.ndn)
    up, dn = sq.dets_to_u64(up), sq.dets_to_u64(dn)
    H.generate_sparse_ham_upper_triangular(up, dn)
    cnt, idx, val = H.export_upper()
    M = np.zeros((len(cnt), len(cnt)))
    row = np.repeat(np.arange(len(cnt)), cnt)
    M[row, idx - 1] = val
    M = M + np.triu(M, 1).T
    ev, vec = np.linalg.eigh(M)
    return sysm, H, up, dn, ev, vec[:, 0]


def test_natural_orbitals_end_to_end(tmp_path):
    sq = _sq()
    from sqmc_b200 import natorb
    toy = str(tmp_path / "FCIDUMP")
    write_toy_fcidump(toy)
    sysm, H, up, dn, ev, c = _fci_ground(sq, toy)
    assert ev[1] - ev[0] > 1e-3
    res = natorb.natural_orbitals(sysm, H.one_rdm(up, dn, c))
    rot = str(tmp_path / "FCIDUMP_no")
    natorb.rotate_fcidump(toy, res["coeffs"], res["irreps"], rot)
    sys2, H2, up2, dn2, ev2, c2 = _fci_ground(sq, rot)
    assert abs(ev2[0] - ev[0]) <= 1e-10
    g = H2.one_rdm(up2, dn2, c2).sum(axis=0)
    o = sys2.orb_order[:sys2.norb] - 1
    gf = np.zeros_like(g)
    gf[np.ix_(o, o)] = g
    assert np.max(np.abs(gf - np.diag(np.diag(gf)))) <= 1e-9
    assert np.max(np.abs(np.diag(gf) - res["occupations"])) <= 1e-9


def test_natorb_script_on_shipped_input(tmp_path):
    from sqmc_b200 import hci
    inp = os.path.join(ROOT, "data", "C2_v2z_curve", "r1.24253", "i_1sigma_g")
    out = str(tmp_path / "no")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "natorb.py"), inp, "--out", out], capture_output=True, text=True, check=True)
    res = json.loads(p.stdout.strip().splitlines()[-1])
    occ = np.array(res["occupations"])
    assert abs(occ.sum() - 8) <= 1e-10 and abs(res["sum_occupations"] - 8) <= 1e-10
    assert occ.min() >= -1e-12 and occ.max() <= 2 + 1e-12
    orig = hci.read_input(inp)["orbital_symmetries"]
    new = hci.read_input(os.path.join(out, "i_1sigma_g"))["orbital_symmetries"]
    assert sorted(new) == sorted(orig)
    r2 = hci.run_input(os.path.join(out, "i_1sigma_g"), log=lambda *_: None)
    assert len(r2["up"]) > 0 and len(r2["pt"]) == len(res["energies"])
