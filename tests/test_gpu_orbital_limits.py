"""The orbital-count limits of every GPU entry point: 64 orbitals (bit 63 of a one-word string, the largest size of the
heat-bath tables and of the two-body family) and 65..127 orbitals (two-word strings).

1. Embedded C2: the shipped C2 FCIDUMP with padding orbitals that carry no two-electron integrals.  Each result must
   equal the 26-orbital one mapped by phi, the orbital relabelling, exactly or to rounding.
2. A fully coupled random Hamiltonian at 64, 65 and 96 orbitals against the oracle.
3. The k-space Hubbard model on 8x8 and 9x8 lattices against the oracle and the density references.
4. The edges themselves: the orbital beyond norb, norb = 128, and the 64-orbital limit of the two-body family.

The tests without the gpu mark check the inputs: the embedding, the orbital placement, the oracle's own invariance
under padding, and the momentum-sector enumeration beyond 64 sites."""
import itertools
import json
import os
import time

import numpy as np
import pytest

from conftest import C2_FCIDUMP, C2_ORBSYM, label_sorted
from oracle.oracle import dets_to_u64
from rdm_reference import one_rdm as ref_one_rdm, u64_to_ints
from rdm2_reference import two_rdm as ref_two_rdm

HERE = os.path.dirname(os.path.abspath(__file__))
C2_NORB, C2_NELEC, C2_NOCC = 26, 8, 4
EMBED_NORBS = [64, 65, 80, 108, 127]   # 108: combine_2 fits in 48 KiB but not beside the kernels' static shared memory
gpu = pytest.mark.gpu


# ----------------------------------------------------------------------------------------------------------- helpers
def embed_c2_fcidump(path, norb):
    """Write the shipped C2 FCIDUMP with norb - 26 padding orbitals appended after FCIDUMP orbital 26, line by line (the
    dense integral table of 127 orbitals would take 2 GB).  The C2 lines keep their labels and their value text, so they
    parse to the same doubles.  Padding orbital 27 + k gets h = -10 - 0.01 k (distinct, below the C2 LUMO), irrep
    1 + k % 8 and no two-electron integral: it couples to nothing."""
    with open(C2_FCIDUMP) as f:
        lines = f.read().splitlines()
    end = next(k for k, ln in enumerate(lines) if "&END" in ln.upper())
    pad = norb - C2_NORB
    sym = C2_ORBSYM + [1 + k % 8 for k in range(pad)]
    with open(path, "w") as f:
        f.write(" &FCI NORB=%d,NELEC=%d,MS2=0,\n  ORBSYM=%s,\n  ISYM=1,\n &END\n" % (norb, C2_NELEC, ",".join(map(str, sym))))
        for ln in lines[end + 1:]:
            t = ln.split()
            if len(t) >= 5:
                f.write("%s %d %d %d %d\n" % (t[0], int(t[1]), int(t[2]), int(t[3]), int(t[4])))
        for k in range(pad):
            f.write("%.17g %d %d 0 0\n" % (-10.0 - 0.01 * k, C2_NORB + 1 + k, C2_NORB + 1 + k))
    return sym


def phi_positions(sys26, sysn):
    """library position of each of the 26 C2 orbitals in the padded system (orbitals matched by FCIDUMP label)"""
    where = {int(f): i for i, f in enumerate(sysn.orb_order[:sysn.norb])}
    return np.array([where[int(f)] for f in sys26.orb_order[:C2_NORB]])


def phi_dets(dets, pos):
    """(n, 2) uint64 strings of the 26-orbital system -> the same determinants in the padded numbering"""
    out = []
    for s in u64_to_ints(dets):
        t = 0
        for i in range(C2_NORB):
            if (s >> i) & 1:
                t |= 1 << int(pos[i])
        out.append(t)
    return dets_to_u64(out)


def embed(a, pos, norb, axes):
    """a with its last `axes` orbital axes (26 long) scattered to pos in zero arrays of norb"""
    out = np.zeros(a.shape[:a.ndim - axes] + (norb,) * axes)
    out[(Ellipsis,) + np.ix_(*([pos] * axes))] = a
    return out


@pytest.fixture(scope="module")
def embedded(tmp_path_factory):
    """norb -> (FCIDUMP path, orbital symmetries) of the embedded C2 input"""
    d = tmp_path_factory.mktemp("embedded_c2")
    out = {}
    for norb in EMBED_NORBS:
        p = str(d / ("FCIDUMP_%d" % norb))
        out[norb] = (p, embed_c2_fcidump(p, norb))
    return out


def _c2_lowest(n):
    from sqmc_b200 import spaces, systems
    up, dn, _ = spaces.c2_lowest_energy_space(systems.ChemSystem(C2_FCIDUMP), n)
    return up, dn


# ------------------------------------------------------------------------------------------ 1. embedded C2 (host side)
@pytest.mark.parametrize("norb", EMBED_NORBS)
def test_embedding_places_c2_virtuals_at_the_top(embedded, norb):
    """occupied orbitals first, then the padding, then the 22 C2 virtuals in their own order at norb-22..norb-1"""
    from sqmc_b200 import systems
    path, sym = embedded[norb]
    s26 = systems.ChemSystem(C2_FCIDUMP)
    sn = systems.ChemSystem(path)
    assert sn.norb == norb and list(sn.orbital_symmetries_fcidump) == sym
    assert sn.hf_up == s26.hf_up == sn.hf_dn == (1 << C2_NOCC) - 1
    pos = phi_positions(s26, sn)
    assert list(pos) == list(range(C2_NOCC)) + list(range(norb - (C2_NORB - C2_NOCC), norb))
    assert sorted(int(f) for f in sn.orb_order[C2_NOCC:norb - 22]) == list(range(C2_NORB + 1, norb + 1))
    assert np.array_equal(sn.orbital_energies[pos], s26.orbital_energies)
    assert np.array_equal(sn.orbital_symmetries[pos], s26.orbital_symmetries)
    h, J, K = s26.jk_tables()
    hn, Jn, Kn = sn.jk_tables()
    assert np.array_equal(hn[pos], h) and np.array_equal(Jn[np.ix_(pos, pos)], J) and np.array_equal(Kn[np.ix_(pos, pos)], K)
    pad = np.setdiff1d(np.arange(norb), pos)
    assert np.all(Jn[pad] == 0) and np.all(Kn[pad] == 0)


@pytest.mark.parametrize("norb", EMBED_NORBS)
def test_oracle_build_is_invariant_under_padding(oracle, embedded, norb):
    """the oracle's matrix over phi of a C2 list is bit for bit its 26-orbital matrix (both numberings from the oracle)"""
    from sqmc_b200 import systems
    path, sym = embedded[norb]
    S26 = oracle.System.chem(C2_FCIDUMP, C2_NORB, C2_NELEC, 4, C2_ORBSYM)
    Sn = oracle.System.chem(path, norb, C2_NELEC, 4, sym)
    on = Sn.chem_tables()["orb_order"]
    assert np.array_equal(on[:norb], systems.ChemSystem(path).orb_order[:norb])
    up, dn = _c2_lowest(1500)
    pos = phi_positions(systems.ChemSystem(C2_FCIDUMP), systems.ChemSystem(path))
    ref = S26.build_upper(up, dn)
    got = Sn.build_upper(phi_dets(up, pos), phi_dets(dn, pos))
    assert all(np.array_equal(a, b) for a, b in zip(got, ref)) and len(ref[1]) > 10 * len(up)


# ------------------------------------------------------------------------------------------- 1. embedded C2 (device)
class Embedded:
    """padded and 26-orbital handles of one setting (time_sym, z) and the map phi between them"""

    def __init__(self, path, time_sym=False):
        import sqmc_b200 as sq
        self.s26 = sq.ChemSystem(C2_FCIDUMP, time_sym=time_sym, z=1)
        self.sn = sq.ChemSystem(path, time_sym=time_sym, z=1)
        self.H26 = sq.SparseHamiltonian(self.s26)
        self.Hn = sq.SparseHamiltonian(self.sn)
        self.pos = phi_positions(self.s26, self.sn)
        self.norb = self.sn.norb

    def phi(self, dets):
        return phi_dets(dets, self.pos)


@gpu
@pytest.mark.parametrize("norb", EMBED_NORBS)
def test_embedded_build_matvec_projector(oracle, c2_space, c2_space_ts, embedded, norb):
    for ts, (s, r) in ((False, c2_space), (True, c2_space_ts)):
        E = Embedded(embedded[norb][0], time_sym=ts)
        up, dn = r["up"], r["dn"]
        ref = s.build_upper(up, dn)
        nnz = E.Hn.generate_sparse_ham_upper_triangular(E.phi(up), E.phi(dn))
        assert nnz == len(ref[1])
        got = E.Hn.export_upper()
        assert all(np.array_equal(a, b) for a, b in zip(got, ref)), (norb, ts)
        E.H26.generate_sparse_ham_upper_triangular(up, dn)
        x = np.random.default_rng(norb).uniform(-1, 1, (len(up), 2))
        assert np.array_equal(E.Hn.matvec(x), E.H26.matvec(x))
        yref = oracle.matvec_upper(*ref, x[:, 0])
        assert np.max(np.abs(E.Hn.matvec(x[:, 0]) - yref)) <= 1e-12 * np.max(np.abs(yref))
        for H in (E.Hn, E.H26):
            H.scale_values(-0.01)
        assert np.array_equal(E.Hn.projector_step(0.01, -75.7, x[:, 0]), E.H26.projector_step(0.01, -75.7, x[:, 0]))


@pytest.fixture(scope="module")
def c2_gpu_hci():
    """the three runs of tests/golden/c2_s1_hci.json on the 26-orbital handles, with the selection trace of each"""
    import sqmc_b200 as sq
    from test_gpu_select import _hci_on_gpu
    out = {}
    for name, ts, ns in (("n_states=1", True, 1), ("n_states=2", True, 2), ("time_sym=f n_states=1", False, 1)):
        cs = sq.ChemSystem(C2_FCIDUMP, time_sym=ts, z=1)
        trace = []
        res = _hci_on_gpu(sq.SparseHamiltonian(cs), cs.hf_up, cs.hf_dn, [2e-3, 2e-3] + [1e-3] * 28, n_states=ns, trace=trace)
        out[name] = (ts, ns, res, trace)
    return out


@gpu
@pytest.mark.parametrize("norb", EMBED_NORBS)
def test_embedded_hci_loop_reproduces_golden_runs(c2_gpu_hci, embedded, norb):
    """selection (heat-bath tables at 64 orbitals, enumeration above), incremental build and Davidson on the GPU"""
    import sqmc_b200 as sq
    from test_gpu_select import _hci_on_gpu
    gold = json.load(open(os.path.join(HERE, "golden", "c2_s1_hci.json")))["runs"]
    for name, (ts, ns, (up0, dn0, _, _), trace0) in c2_gpu_hci.items():
        E = Embedded(embedded[norb][0], time_sym=ts)
        trace = []
        up, dn, wts, log = _hci_on_gpu(E.Hn, E.sn.hf_up, E.sn.hf_dn, [2e-3, 2e-3] + [1e-3] * 28, n_states=ns, trace=trace)
        g = gold[name]
        assert [l[0] for l in log] == g["n_det"], (norb, name)
        assert [l[1] for l in log] == g["nnz"], (norb, name)
        assert np.max(np.abs(np.array([l[2] for l in log]) - np.array(g["iter_energy"]))) < 1e-8
        assert np.array_equal(up, E.phi(up0)) and np.array_equal(dn, E.phi(dn0))
        assert len(trace) == len(trace0)
        for (nu, nd, mh), (nu0, nd0, mh0) in zip(trace, trace0):
            assert np.array_equal(nu, E.phi(nu0)) and np.array_equal(nd, E.phi(nd0)) and np.array_equal(mh, mh0)


@gpu
@pytest.mark.parametrize("norb", EMBED_NORBS)
def test_embedded_pt(c2_space, c2_space_ts, embedded, norb):
    """deterministic and stochastic PT: the padded list connects to the same determinants with the same elements"""
    for ts, (s, r) in ((False, c2_space), (True, c2_space_ts)):
        E = Embedded(embedded[norb][0], time_sym=ts)
        up, dn, w = label_sorted(r)
        e0 = r["energy"][0]
        de0, nc0 = E.H26.second_order_pt(up, dn, w, e0, 1e-5)
        de, nc = E.Hn.second_order_pt(E.phi(up), E.phi(dn), w, e0, 1e-5)
        assert nc == nc0 and abs(de - de0) <= 1e-10 * abs(de0), (norb, ts)
        seed = [11, 22, 33, 45]
        a0 = E.H26.second_order_pt_alias(up, dn, w, e0, 1e-5, 2e-4, 50, 1e-9, seed, max_samples=4)
        a = E.Hn.second_order_pt_alias(E.phi(up), E.phi(dn), w, e0, 1e-5, 2e-4, 50, 1e-9, seed, max_samples=4)
        assert a["n_samples"] == a0["n_samples"] == 4 and a["ndets_connected"] == a0["ndets_connected"]
        assert np.max(np.abs(a["e_2pt_samples"] - a0["e_2pt_samples"])) <= 1e-10 * np.max(np.abs(a0["e_2pt_samples"]))
        assert np.array_equal(a["rannyu_state"], a0["rannyu_state"])


@gpu
@pytest.mark.parametrize("norb", EMBED_NORBS)
def test_embedded_densities_ladder_lanczos(c2_space, c2_space_ts, embedded, norb):
    rng = np.random.default_rng(100 + norb)
    for ts, (s, r) in ((False, c2_space), (True, c2_space_ts)):
        E = Embedded(embedded[norb][0], time_sym=ts)
        up, dn = r["up"], r["dn"]
        pu, pd = E.phi(up), E.phi(dn)
        w = rng.standard_normal((len(up), 2))
        pad = np.setdiff1d(np.arange(norb), E.pos)
        for got, ref in ((E.Hn.one_rdm(pu, pd, w), E.H26.one_rdm(up, dn, w)),
                         (E.Hn.transition_one_rdm(pu, pd, w[:, 0], w[:, 1]), E.H26.transition_one_rdm(up, dn, w[:, 0], w[:, 1]))):
            emb = embed(ref, E.pos, norb, 2)
            assert np.max(np.abs(got - emb)) <= 1e-14 * np.max(np.abs(emb)), (norb, ts)
            assert np.all(got[..., pad, :] == 0) and np.all(got[..., :, pad] == 0)
        orbs = [0, 3, 4, 11, 25]
        for spin, create in ((0, False), (1, False), (0, True), (1, True)):
            u0, d0, f0 = E.H26.ladder(up, dn, w, orbs, spin, create, state=1)
            u1, d1, f1 = E.Hn.ladder(pu, pd, w, E.pos[orbs], spin, create, state=1)
            assert np.array_equal(u1, E.phi(u0)) and np.array_equal(d1, E.phi(d0)) and np.array_equal(f1, f0), (norb, ts, spin, create)
        E.H26.generate_sparse_ham_upper_triangular(up, dn)
        E.Hn.generate_sparse_ham_upper_triangular(pu, pd)
        v0 = rng.standard_normal((len(up), 2))
        l0 = E.H26.lanczos_tridiagonal(v0, 12)
        l1 = E.Hn.lanczos_tridiagonal(v0, 12)
        for key in ("alpha", "beta"):
            assert np.max(np.abs(l1[key] - l0[key])) <= 1e-12 * np.max(np.abs(l0[key])), (norb, ts, key)


@gpu
def test_embedded_two_body_family_at_64(c2_space, c2_space_ts, embedded):
    from test_gpu_orbopt import _check as check_orbital_derivatives
    from test_gpu_orbopt_coupled import _dense_apply, _response_reference
    from test_gpu_rdm2 import _subset
    norb = 64
    rng = np.random.default_rng(64)
    for ts, (s, r) in ((False, c2_space), (True, c2_space_ts)):
        E = Embedded(embedded[norb][0], time_sym=ts)
        up, dn = _subset(r, 120, 7)
        pu, pd = E.phi(up), E.phi(dn)
        a, b = rng.standard_normal(len(up)), rng.standard_normal(len(up))
        pad = np.setdiff1d(np.arange(norb), E.pos)
        # two_rdm / transition_two_rdm: fixed-point accumulation, so the embedding is exact, zeros included
        for got, ref in ((E.Hn.two_rdm(pu, pd, a), E.H26.two_rdm(up, dn, a)),
                         (E.Hn.transition_two_rdm(pu, pd, a, b), E.H26.transition_two_rdm(up, dn, a, b))):
            assert np.array_equal(got, embed(ref, E.pos, norb, 4)), ts
            del got, ref
        # orbital gradient and Hessian against the dense numpy reference at 64 orbitals; the active block is the 26-orbital one
        got = check_orbital_derivatives(E.Hn, pu, pd, a)
        g26 = E.H26.orbital_derivatives(up, dn, a)
        m = E.pos
        assert np.max(np.abs(got["fock"][np.ix_(m, m)] - g26["fock"])) <= 1e-12 * np.max(np.abs(g26["fock"]))
        assert np.max(np.abs(got["hessian"][np.ix_(m, m, m, m)] - g26["hessian"])) <= 1e-12 * np.max(np.abs(g26["hessian"]))
        assert abs(got["energy"] - g26["energy"]) <= 1e-12 * abs(g26["energy"])
        assert np.all(got["fock"][pad] == 0)
        del got, g26
        # sigma with a kappa that rotates C2 orbitals into the padding, and the gradient response
        K = np.tril(rng.standard_normal((norb, norb)), -1)
        K = K - K.T
        ref, _, _, _ = _dense_apply(E.Hn, pu, pd, a, K)
        y = E.Hn.sigma(pu, pd, a, kappa=K)
        assert np.max(np.abs(y - ref)) <= 1e-10 * np.max(np.abs(ref)), ts
        y0 = E.H26.sigma(up, dn, a)
        assert np.max(np.abs(E.Hn.sigma(pu, pd, a) - y0)) <= 1e-13 * np.max(np.abs(y0))
        resp = E.Hn.orbital_gradient_response(pu, pd, a, b)
        rref = _response_reference(E.Hn, pu, pd, a, b, [1.0])
        assert np.max(np.abs(resp - rref)) <= 1e-10 * max(1.0, np.max(np.abs(rref))), ts


# -------------------------------------------------------------------------- 2. fully coupled random Hamiltonian vs oracle
RANDOM_CASES = [(norb, ts, z, nup) for norb in (64, 65, 96) for ts, z, nup in ((False, 1, 4), (True, 1, 4), (True, -1, 4), (False, 1, 5))]


def write_random_fcidump(path, norb, nelec, seed):
    """8-fold symmetric integrals, allowed by the symmetry of irreps 1..4: a diagonal-dominant one-body part rising with
    the orbital label (so the Hartree-Fock determinant of the first orbitals is lowest), Coulomb and exchange integrals,
    and ~20000 random (pq|rs) of size ~0.05 that couple every orbital, 63..norb included."""
    rng = np.random.default_rng(seed)
    sym = [1 + k % 4 for k in range(norb)]
    ints = {}

    def put(v, p, q, r, s):
        a, b = max(p, q), min(p, q)
        c, d = max(r, s), min(r, s)
        key = max((a, b), (c, d)) + min((a, b), (c, d))
        ints[key] = v

    for p in range(1, norb + 1):
        for q in range(1, p):
            if sym[p - 1] == sym[q - 1] and rng.random() < 0.2:
                put(rng.uniform(-0.02, 0.02), p, q, 0, 0)
            put(0.3 + 0.1 * rng.random(), p, p, q, q)
            if rng.random() < 0.3:
                put(0.02 * rng.random(), p, q, q, p)
        put(0.5 + 0.1 * rng.random(), p, p, p, p)
    for _ in range(20000):
        p, q, r, s = (int(x) for x in rng.integers(1, norb + 1, 4))
        if ((sym[p - 1] - 1) ^ (sym[q - 1] - 1) ^ (sym[r - 1] - 1) ^ (sym[s - 1] - 1)) == 0 and len({(p, q), (q, p)} & {(r, s), (s, r)}) == 0:
            put(rng.uniform(-0.05, 0.05), p, q, r, s)
    with open(path, "w") as f:
        f.write(" &FCI NORB=%d,NELEC=%d,MS2=0,\n  ORBSYM=%s,\n  ISYM=1,\n &END\n" % (norb, nelec, ",".join(map(str, sym))))
        for (p, q, r, s), v in sorted(ints.items()):
            f.write("%.17e %d %d %d %d\n" % (v, p, q, r, s))
        for p in range(1, norb + 1):
            f.write("%.17e %d %d 0 0\n" % (-3.0 + 0.05 * p, p, p))
        f.write("1.25 0 0 0 0\n")
    return sym


def _random_case(oracle, tmp_path, norb, ts, z, nup):
    """(library system, oracle system, det list, coefficients, variational energy): the oracle's first HCI iteration from
    Hartree-Fock plus hand-placed determinants with electrons on orbitals 63, 64, 65 and norb (bits 62, 63, 64, norb-1)"""
    import sqmc_b200 as sq
    path = str(tmp_path / ("FCIDUMP_%d" % norb))
    sym = write_random_fcidump(path, norb, 8, 1000 + norb)
    cs = sq.ChemSystem(path, nup=nup, time_sym=ts, z=z)
    S = oracle.System.chem(path, norb, 8, nup, sym, time_sym=ts, z=z)
    t = S.chem_tables()
    assert np.array_equal(cs.integrals, t["integrals"]) and np.array_equal(cs.orb_order[:norb], t["orb_order"][:norb])
    r = S.hci(2e-3, n_states=1, max_iters=1)
    keep = np.sort(np.argsort(-np.abs(r["wts"][:, 0]), kind="stable")[:80 if norb <= 65 else 30])   # bounds the oracle's time
    have = set(zip(u64_to_ints(r["up"][keep]), u64_to_ints(r["dn"][keep])))
    hu, hd, ndn = cs.hf_up, cs.hf_dn, 8 - nup
    his = sorted({b for b in (62, 63, 64) if b < norb} | {norb - 1})
    b0, b1 = (63, 64) if norb > 64 else (62, 63)
    cand = [(hu & ~3 | 1 << b0 | 1 << b1, hd), (hu, hd & ~3 | 1 << his[0] | 1 << his[-1])]   # pairs at the top, across the word boundary
    for hi in his:
        for lo in (nup - 1, 0):
            u1, d1 = hu & ~(1 << lo) | 1 << hi, hd & ~(1 << ((lo + 1) % ndn)) | 1 << hi
            cand += [(u1, hd), (hu, d1), (u1, d1)]
    extra = []
    for u, d in cand:
        if ts:
            u, d = min(u, d), max(u, d)
            if u == d and z == -1:
                continue
        if (u, d) not in have:
            have.add((u, d))
            extra.append((u, d))
    up = np.concatenate([r["up"][keep], dets_to_u64([u for u, d in extra])])
    dn = np.concatenate([r["dn"][keep], dets_to_u64([d for u, d in extra])])
    w = np.concatenate([r["wts"][keep, 0], np.random.default_rng(norb).uniform(-1e-3, 1e-3, len(extra))])
    assert all(bin(u).count("1") == nup and bin(d).count("1") == 8 - nup for u, d in extra)
    top = max(int(v).bit_length() for v in u64_to_ints(up) + u64_to_ints(dn))
    assert top == norb and len(extra) >= 10
    return cs, S, up, dn, w, r["energy"][0]


@gpu
@pytest.mark.parametrize("norb,ts,z,nup", RANDOM_CASES)
def test_random_hamiltonian_against_oracle(oracle, tmp_path, norb, ts, z, nup):
    """build (bit-exact), selection (up, dn, min_H exact), deterministic PT and single PT samples; the CPU time of the oracle's
    build, selection and PT calls is printed (-s)"""
    import sqmc_b200 as sq
    from test_gpu_pt2 import _draw_sample
    cs, S, up, dn, w, e0 = _random_case(oracle, tmp_path, norb, ts, z, nup)
    H = sq.SparseHamiltonian(cs)
    t0 = time.perf_counter()
    ref = S.build_upper(up, dn)
    t_oracle = time.perf_counter() - t0
    assert H.generate_sparse_ham_upper_triangular(up, dn) == len(ref[1])
    got = H.export_upper()
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))
    assert np.array_equal(H.diagonal(up, dn), S.elements(up, dn, up, dn))
    rng = np.random.default_rng(norb + nup)
    coeffs = np.abs(w)
    for eps, mh in ((1e-3, np.full(len(up), 9e99)), (5e-4, 10.0 ** rng.uniform(-3, 0, len(up)))):
        t1 = time.perf_counter()
        ru, rd, rm = S.select(up, dn, coeffs, mh, eps)
        t_oracle += time.perf_counter() - t1
        gu, gd, gm = H.get_next_det_list(up, dn, coeffs, mh, eps)
        assert len(ru) > 0 and np.array_equal(gu, ru) and np.array_equal(gd, rd) and np.array_equal(gm, rm), eps
    lu, ld, lw = label_sorted(dict(up=up, dn=dn, wts=w.reshape(-1, 1)))
    t1 = time.perf_counter()
    ode, onc = S.pt2(lu, ld, lw, e0, 1e-4)
    t_oracle += time.perf_counter() - t1
    de, nc = H.second_order_pt(lu, ld, lw, e0, 1e-4)
    assert nc == onc and nc > len(up) and abs(de - ode) <= 1e-10 * abs(ode)
    for n_mc, eps_big, seed in ((20, 1e-3, 1), (3, 5e-3, 2)):
        idx, wop = _draw_sample(lw, n_mc, seed)
        t1 = time.perf_counter()
        oe, onc = S.pt2_sample(lu, ld, lu[idx], ld[idx], lw[idx], wop, n_mc, e0, 1e-4, eps_big)
        t_oracle += time.perf_counter() - t1
        e, nc = H.second_order_pt_sample(lu, ld, lu[idx], ld[idx], lw[idx], wop, n_mc, e0, 1e-4, eps_big)
        assert nc == onc and abs(e - oe) <= 1e-12 * max(1.0, abs(oe) / 1e-3) and e != 0.0
    print("random Hamiltonian norb=%d time_sym=%s z=%d nup=%d: %d dets, oracle %.1f s" % (norb, ts, z, nup, len(up), t_oracle))


# ------------------------------------------------------------------------------------------------ 3. Hubbard k-space
def _brute_sector(hub, ktot=(0, 0)):
    """every (up, dn) pair of python ints with the total momentum ktot, in label order, with its kinetic energy"""
    def strings(k):
        out = []
        for c in itertools.combinations(range(hub.norb), k):
            s = sum(1 << o for o in c)
            kx = sum(int(hub.k_vectors[o, 0]) for o in c)
            ky = sum(int(hub.k_vectors[o, 1]) for o in c)
            out.append((s, kx, ky, sum(float(hub.k_energies[o]) for o in c)))
        return out
    su, sd = strings(hub.nup), strings(hub.ndn)
    out = []
    for u, ux, uy, ue in su:
        for d, dx, dy, de in sd:
            if (ux + dx - ktot[0]) % (2 * hub.l_x) == 0 and (uy + dy - ktot[1]) % (2 * hub.l_y) == 0:
                out.append((u, d, ue + de))
    return sorted(out)


def test_hubbard_sector_beyond_64_sites_matches_brute_force():
    """9x8 lattice, 2 up and 2 down electrons: two-word strings, the whole (0,0) sector and a truncated one"""
    from sqmc_b200 import spaces, systems
    hub = systems.HubbardKSystem(9, 8, 1.0, 4.0, 2, 2)
    assert hub.norb == 72
    ref = _brute_sector(hub)
    up, dn, total = spaces.hubbard_momentum_sector(hub)
    assert total == len(ref) == len(up)
    assert list(zip(u64_to_ints(up), u64_to_ints(dn))) == [(u, d) for u, d, _ in ref]
    assert max(u for u, _, _ in ref).bit_length() == 72
    n = 5000
    keep = sorted(ref, key=lambda t: (round(t[2], 12), t[0], t[1]))[:n]
    up, dn, _ = spaces.hubbard_momentum_sector(hub, n_dets=n)
    assert list(zip(u64_to_ints(up), u64_to_ints(dn))) == sorted((u, d) for u, d, _ in keep)


@gpu
@pytest.mark.parametrize("l_x,l_y", [(8, 8), (9, 8)])
def test_hubbard_64_and_72_sites_against_oracle(oracle, l_x, l_y):
    import sqmc_b200 as sq
    from sqmc_b200 import spaces
    hub = sq.HubbardKSystem(l_x, l_y, 1.0, 4.0, 2, 2)
    S = oracle.System.hubbardk(l_x, l_y, 1.0, 4.0, 2, 2)
    t = S.hubbardk_tables()
    assert np.array_equal(t["k_vectors"], hub.k_vectors) and np.array_equal(t["k_energies"], hub.k_energies)
    up, dn, total = spaces.hubbard_momentum_sector(hub)
    assert len(up) == total > 60000
    ref = S.build_upper(up, dn)
    H = sq.SparseHamiltonian(hub)
    assert H.generate_sparse_ham_upper_triangular(up, dn) == len(ref[1])
    got = H.export_upper()
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))
    x = np.random.default_rng(l_x).uniform(-1, 1, len(up))
    yref = oracle.matvec_upper(*ref, x)
    assert np.max(np.abs(H.matvec(x) - yref)) <= 1e-12 * np.max(np.abs(yref))
    d = H.davidson_sparse(n_states=1)
    od = oracle.davidson(*ref, n_states=1)
    assert abs(d["evals"][0] - od["evals"][0]) < 1e-9
    # densities over a low-energy part of the sector (the references loop in python)
    rng = np.random.default_rng(7)
    su, sd, _ = spaces.hubbard_momentum_sector(hub, n_dets=3000)
    w = rng.standard_normal(len(su))
    g = H.one_rdm(su, sd, w)
    assert np.max(np.abs(g - ref_one_rdm(su, sd, w, hub.norb)[0])) <= 1e-12
    if hub.norb <= 64:
        su, sd, _ = spaces.hubbard_momentum_sector(hub, n_dets=120)
        w = rng.standard_normal(len(su))
        g2 = H.two_rdm(su, sd, w)
        assert np.max(np.abs(g2 - ref_two_rdm(su, sd, w, hub.norb)[0])) <= 1e-13


# ------------------------------------------------------------------------------------------------------ 4. the edges
@gpu
@pytest.mark.parametrize("norb,bit", [(64, 64), (127, 127)])
def test_orbital_beyond_norb_is_refused(embedded, norb, bit):
    import sqmc_b200 as sq
    cs = sq.ChemSystem(embedded[norb][0])
    H = sq.SparseHamiltonian(cs)
    ok = sq.dets_to_u64([cs.hf_up, cs.hf_up])
    bad = sq.dets_to_u64([cs.hf_dn, (cs.hf_dn & ~1) | (1 << bit)])
    with pytest.raises(sq.SqmcError, match="beyond norb"):
        H.generate_sparse_ham_upper_triangular(ok, bad)
    with pytest.raises(sq.SqmcError, match="beyond norb"):
        H.generate_sparse_ham_upper_triangular(bad, ok)
    good = sq.dets_to_u64([cs.hf_dn, (cs.hf_dn & ~1) | (1 << (bit - 1))])
    assert H.generate_sparse_ham_upper_triangular(ok, good) >= 2


def test_128_orbitals_are_refused_by_the_host_systems(tmp_path):
    from sqmc_b200 import systems
    with pytest.raises(ValueError, match="outside 1..127"):
        systems.HubbardKSystem(16, 8, 1.0, 4.0, 2, 2)
    path = str(tmp_path / "FCIDUMP_128")
    embed_c2_fcidump(path, 128)
    with pytest.raises(ValueError, match="outside 1..127"):
        systems.ChemSystem(path)
    with pytest.raises(ValueError, match="outside 1..127"):
        systems.HegSystem(3, 0.5, 14, 7, 3.2)           # 147 plane waves inside the cutoff
    assert systems.HegSystem(3, 0.5, 14, 7, 3.0).norb == 123


@gpu
def test_128_orbitals_are_refused_by_the_library():
    """the C ABI checks the orbital count itself, before it reads any table"""
    import ctypes as C
    import sqmc_b200 as sq
    from sqmc_b200 import _lib
    _lib.init(device=0)
    L, h = _lib.load(), C.c_void_p()
    with pytest.raises(sq.SqmcError, match="norb=128 outside 1..127"):
        _lib.check(L.sqmc_b200_system_chem(C.byref(h), 128, 4, 4, None, 0, None, 0, 1))
    with pytest.raises(sq.SqmcError, match="bad lattice"):
        _lib.check(L.sqmc_b200_system_hubbardk(C.byref(h), 16, 8, None, None, C.c_double(0.03125), 2, 2))
    with pytest.raises(sq.SqmcError, match="bad norb"):
        _lib.check(L.sqmc_b200_system_heg(C.byref(h), 128, 3, None, C.c_double(1.0), 7, 7))


@gpu
def test_two_body_family_accepts_64_and_refuses_65(c2_space, embedded):
    import sqmc_b200 as sq
    from test_gpu_rdm2 import _subset
    up, dn = _subset(c2_space[1], 20, 3)
    s26 = sq.ChemSystem(C2_FCIDUMP)
    w = np.random.default_rng(5).standard_normal(len(up))
    for norb in (64, 65):
        sn = sq.ChemSystem(embedded[norb][0])
        H = sq.SparseHamiltonian(sn)
        pos = phi_positions(s26, sn)
        pu, pd = phi_dets(up, pos), phi_dets(dn, pos)
        calls = {"sigma": lambda: H.sigma(pu, pd, w),
                 "orbital_derivatives": lambda: H.orbital_derivatives(pu, pd, w),
                 "orbital_gradient_response": lambda: H.orbital_gradient_response(pu, pd, w, w[::-1].copy()),
                 "transition_two_rdm": lambda: H.transition_two_rdm(pu, pd, w, w[::-1].copy())}
        for name, call in calls.items():
            if norb == 64:
                call()
            else:
                with pytest.raises(sq.SqmcError, match="%s: norb = 65 > 64 is not supported" % name):
                    call()
