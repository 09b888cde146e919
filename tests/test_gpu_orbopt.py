"""Orbital gradient and Hessian on the device (SparseHamiltonian.orbital_derivatives) and the orbital optimiser
(sqmc_b200.orbopt, scripts/orbopt.py)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import C2_FCIDUMP, C2_ORBSYM, ROOT
from orbopt_reference import densities, energy, orbital_derivatives_reference
from test_gpu_rdm2 import _list53, _random_eri_system, _subset
from test_natorb_host import fci_dets, write_toy_fcidump

pytestmark = pytest.mark.gpu
C2_INPUT = os.path.join(ROOT, "data", "C2_v2z_curve", "r1.24253", "i_1sigma_g")


def _sq():
    import sqmc_b200 as sq
    return sq


def _reference(H, up, dn, w, sw):
    from sqmc_b200 import rdm
    w2 = np.asarray(w).reshape(len(up), -1)
    g1 = H.one_rdm(up, dn, w2)
    g2 = H.two_rdm(up, dn, w2)
    D, d = densities(g1, g2, np.sum(w2 * w2, axis=0), sw)
    h, g, ec = rdm.integrals_library_order(H.system)
    r = orbital_derivatives_reference(h, g, D, d)
    r["energy"] = energy(h, g, ec, D, d)
    return r, D


def _check(H, up, dn, w, sw=None):
    got = H.orbital_derivatives(up, dn, w, state_weights=sw)
    ns = 1 if np.ndim(w) == 1 else np.shape(w)[1]
    ref, _ = _reference(H, up, dn, w, np.full(ns, 1.0 / ns) if sw is None else sw)
    for key in ("fock", "gradient", "hessian"):
        assert np.max(np.abs(got[key] - ref[key])) <= 1e-10 * np.max(np.abs(ref[key])), key
    assert abs(got["energy"] - ref["energy"]) <= 1e-10 * abs(ref["energy"])
    return got


def test_c2_lists_against_reference(c2_space, c2_space_ts):
    sq = _sq()
    rng = np.random.default_rng(1)
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = _subset(c2_space[1], 300, 1)
    _check(H, up, dn, rng.standard_normal(len(up)))                                   # plain, unnormalised
    _check(H, up, dn, rng.standard_normal((len(up), 2)), sw=[0.7, 0.3])               # two states
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    up, dn = _subset(c2_space_ts[1], 300, 2)
    _check(Hts, up, dn, rng.standard_normal(len(up)))                                 # time_sym
    H53 = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, nelec=8, nup=5, time_sym=False, z=1))
    up, dn = _list53(sq, 400, 3)
    _check(H53, up, dn, rng.standard_normal(len(up)))                                 # 5 alpha / 3 beta


def test_random_integrals_against_reference(c2_space):
    sq = _sq()
    rng = np.random.default_rng(4)
    sysm, _ = _random_eri_system(sq, rng, time_sym=False, z=1)
    H = sq.SparseHamiltonian(sysm)
    up, dn = _subset(c2_space[1], 300, 5)
    _check(H, up, dn, rng.standard_normal(len(up)))


def test_energy_and_density(c2_space):
    """energy = weighted Davidson energies; with h = 1 and g = 0, F is D, which equals one_rdm's spin sum"""
    sq = _sq()
    from sqmc_b200 import rdm
    _, r = c2_space
    sysm = sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1)
    H = sq.SparseHamiltonian(sysm)
    H.generate_sparse_ham_upper_triangular(r["up"], r["dn"])
    dv = H.davidson_sparse(n_states=2)
    got = H.orbital_derivatives(r["up"], r["dn"], dv["evecs"], state_weights=[0.7, 0.3])
    assert abs(got["energy"] - (0.7 * dv["evals"][0] + 0.3 * dv["evals"][1])) <= 1e-9
    # the spatially symmetric ground state: rotations between irreps have zero gradient
    g0 = H.orbital_derivatives(r["up"], r["dn"], dv["evecs"][:, 0])["gradient"]
    sym = np.asarray(sysm.orbital_symmetries)
    cross = sym[:, None] != sym[None, :]
    assert np.max(np.abs(g0[cross])) <= 1e-12 and np.max(np.abs(g0[~cross])) > 1e-6
    unit = sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1)
    n, n1 = unit.norb, unit.norb + 1
    ints = np.zeros_like(unit.integrals)
    c2 = np.asarray(unit._c2, dtype=np.int64)
    core = c2[n1 - 1, n1 - 1]
    for p in range(n):
        a = c2[p, p]
        ints[max(a, core) * (max(a, core) - 1) // 2 + min(a, core) - 1] = 1.0
    unit.integrals = ints
    assert np.array_equal(rdm.integrals_library_order(unit)[0], np.eye(n))
    Hu = sq.SparseHamiltonian(unit)
    w = np.random.default_rng(6).standard_normal(len(r["up"]))
    g1 = Hu.one_rdm(r["up"], r["dn"], w)
    F = Hu.orbital_derivatives(r["up"], r["dn"], w)["fock"]
    assert np.max(np.abs(F - (g1[0] + g1[1]) / float(w @ w))) <= 1e-13


def test_toy_fci_is_stationary(tmp_path):
    sq = _sq()
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
    got = H.orbital_derivatives(up, dn, vec[:, 0])
    assert abs(got["energy"] - ev[0]) <= 1e-10
    assert np.max(np.abs(got["gradient"])) <= 1e-9


def test_determinism(c2_space):
    sq = _sq()
    _, r = c2_space
    up, dn = r["up"], r["dn"]
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    w = np.random.default_rng(9).standard_normal((len(up), 2))
    a = H.orbital_derivatives(up, dn, w, state_weights=[0.25, 0.75])
    b = H.orbital_derivatives(up, dn, w, state_weights=[0.25, 0.75])
    p = np.random.default_rng(10).permutation(len(up))
    c = H.orbital_derivatives(up[p], dn[p], w[p], state_weights=[0.25, 0.75])
    for x in (b, c):
        for key in ("fock", "hessian"):
            assert np.array_equal(a[key], x[key])
        assert a["energy"] == x["energy"]


def test_input_errors(c2_space, c2_space_ts, tmp_path):
    sq = _sq()
    _, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    up, dn = r["up"][:50], r["dn"][:50]
    w = np.ones(len(up))
    with pytest.raises(ValueError, match="state_weights"):
        H.orbital_derivatives(up, dn, w, state_weights=[0.5, 0.5])
    with pytest.raises(sq.SqmcError, match="negative"):
        H.orbital_derivatives(up, dn, np.ones((len(up), 2)), state_weights=[1.5, -0.5])
    with pytest.raises(sq.SqmcError, match="sum to"):
        H.orbital_derivatives(up, dn, np.ones((len(up), 2)), state_weights=[0.5, 0.6])
    with pytest.raises(sq.SqmcError, match="twice"):
        H.orbital_derivatives(np.concatenate([up, up[:1]]), np.concatenate([dn, dn[:1]]), np.ones(len(up) + 1))
    with pytest.raises(sq.SqmcError, match="n_states"):
        H.orbital_derivatives(up, dn, np.zeros((len(up), 0)), state_weights=np.zeros(0))
    with pytest.raises(sq.SqmcError, match="n must be positive"):
        H.orbital_derivatives(up[:0], dn[:0], w[:0])
    with pytest.raises(sq.SqmcError, match="electrons"):
        H.orbital_derivatives(np.concatenate([up, sq.dets_to_u64([0b111])]), np.concatenate([dn, sq.dets_to_u64([0b1111])]), np.ones(len(up) + 1))
    _, rt = c2_space_ts
    Hts = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    k = next(i for i in range(len(rt["up"])) if not np.array_equal(rt["up"][i], rt["dn"][i]))
    with pytest.raises(sq.SqmcError, match="time-reversed partner"):
        Hts.orbital_derivatives(np.concatenate([rt["up"], rt["dn"][k:k + 1]]), np.concatenate([rt["dn"], rt["up"][k:k + 1]]), np.ones(len(rt["up"]) + 1))
    hs = sq.HegSystem(3, 0.5, 14, 7, 1.49)
    with pytest.raises(sq.SqmcError, match="fixed by momentum"):
        sq.SparseHamiltonian(hs).orbital_derivatives(sq.dets_to_u64([hs.hf_up]), sq.dets_to_u64([hs.hf_dn]), np.ones(1))
    hub = sq.HubbardKSystem(4, 2, 1.0, 4.0, 3, 2)
    with pytest.raises(sq.SqmcError, match="fixed by momentum"):
        sq.SparseHamiltonian(hub).orbital_derivatives(sq.dets_to_u64([0b111]), sq.dets_to_u64([0b11]), np.ones(1))
    big = str(tmp_path / "FCIDUMP65")
    with open(big, "w") as f:
        f.write(" &FCI NORB=65,NELEC=2,MS2=0,\n &END\n" + "".join("-1.0 %d %d 0 0\n" % (p, p) for p in range(1, 66)) + "0.0 0 0 0 0\n")
    Hb = sq.SparseHamiltonian(sq.ChemSystem(big))
    with pytest.raises(sq.SqmcError, match="norb = 65 > 64"):
        Hb.orbital_derivatives(sq.dets_to_u64([1]), sq.dets_to_u64([1]), np.ones(1))


@pytest.mark.parametrize("time_sym", [False, True])
def test_remap_on_device_keeps_energy(c2_space, c2_space_ts, tmp_path, time_sym):
    """permuting the FCIDUMP orbitals within irreps and remapping list and vector leaves w.Hw unchanged"""
    sq = _sq()
    from sqmc_b200 import natorb, orbopt
    norb = len(C2_ORBSYM)
    sym = np.asarray(C2_ORBSYM)
    rng = np.random.default_rng(12)
    col = np.arange(norb)                       # new column k holds old column col[k]
    for s in set(C2_ORBSYM):
        idx = np.flatnonzero(sym == s)
        col[idx] = idx[rng.permutation(len(idx))]
    P = np.zeros((norb, norb))
    P[col, np.arange(norb)] = 1.0
    a, b = str(tmp_path / "FCIDUMP_a"), str(tmp_path / "FCIDUMP_b")
    natorb.rotate_fcidump(C2_FCIDUMP, np.eye(norb), C2_ORBSYM, a)
    natorb.rotate_fcidump(C2_FCIDUMP, P, C2_ORBSYM, b)
    sa = sq.ChemSystem(a, time_sym=time_sym, z=1)
    sb = sq.ChemSystem(b, time_sym=time_sym, z=1)
    old_col = np.asarray(sa.orb_order[:norb]) - 1
    new_col = np.argsort(col)[old_col]          # old column c is new column k with col[k] = c
    perm = np.asarray(sb.orb_order_inv[:norb])[new_col] - 1
    r = (c2_space_ts if time_sym else c2_space)[1]
    up, dn = r["up"], r["dn"]
    w = np.random.default_rng(13).standard_normal(len(up))
    Ha = sq.SparseHamiltonian(sa)
    Ha.generate_sparse_ham_upper_triangular(up, dn)
    ea = float(w @ Ha.matvec(w))
    u2, d2, w2 = orbopt.remap_determinants(up, dn, w, perm, time_sym=time_sym, z=1)
    Hb = sq.SparseHamiltonian(sb)
    Hb.generate_sparse_ham_upper_triangular(u2, d2)
    eb = float(w2 @ Hb.matvec(w2))
    assert abs(ea - eb) <= 1e-12 * abs(ea)


def test_orbopt_fixed_list_c2(tmp_path):
    from sqmc_b200 import orbopt
    res = orbopt.optimize_orbitals(C2_INPUT, str(tmp_path / "fixed"), fixed_list=True, max_macro=15)
    hist = res["history"]
    e = [h["energy"] for h in hist]
    assert all(b <= a for a, b in zip(e, e[1:]))
    assert e[-1] < e[0] - 1e-4
    # two-step (no CI-orbital coupling): the gradient falls linearly on this list, it does not reach 1e-4 in 15 iterations
    assert hist[-1]["max_grad"] < 0.8 * hist[0]["max_grad"]
    assert res["converged"] == (hist[-1]["max_grad"] < 1e-4)
    print("fixed list: converged=%s after %d macro iterations, max|g| %.2e -> %.2e"
          % (res["converged"], len(hist), hist[0]["max_grad"], hist[-1]["max_grad"]))
    assert res["history"][0]["n_params"] == 42
    C = res["coeffs"]
    assert np.max(np.abs(C.T @ C - np.eye(len(C)))) <= 1e-12
    assert np.all(np.abs(C[np.asarray(C2_ORBSYM)[:, None] != np.asarray(C2_ORBSYM)[None, :]]) == 0)


def test_orbopt_reselect_script_and_rerun(tmp_path):
    from sqmc_b200 import hci
    out = str(tmp_path / "reselect")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "orbopt.py"), C2_INPUT, "--out", out, "--max-macro", "6"],
                       capture_output=True, text=True, check=True)
    res = json.loads(p.stdout.strip().splitlines()[-1])
    hist = res["history"]
    assert res["converged"] == (hist[-1]["max_grad"] < 1e-4)
    assert res["converged"] or len(hist) == 6
    print("reselect: converged=%s after %d macro iterations, max|g| %.2e" % (res["converged"], len(hist), hist[-1]["max_grad"]))
    rerun = hci.run_input(os.path.join(out, "i_1sigma_g"), log=lambda *a: None)
    assert np.max(np.abs(np.asarray(rerun["energy"]) - np.asarray(hist[-1]["energies"]))) <= 1e-8
