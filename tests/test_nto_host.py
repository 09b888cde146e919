"""Host checks of natural transition orbitals and of the transition-density reference (no GPU)."""
import numpy as np
import pytest

from conftest import C2_FCIDUMP
from rdm2_reference import two_rdm
from rdm_reference import one_rdm
from sqmc_b200 import natorb, systems
from tdm_reference import transition_one_rdm, transition_two_rdm
from test_natorb_host import _random_list


@pytest.mark.parametrize("nup,ndn,time_sym,z", [(3, 2, False, 1), (2, 2, True, -1)])
def test_reference_reduces_to_the_one_state_references(nup, ndn, time_sym, z):
    rng = np.random.default_rng(3 + nup + ndn + time_sym)
    norb = 7
    up, dn = _random_list(rng, norb, nup, ndn, 40, time_sym=time_sym)
    c = rng.standard_normal((len(up), 2))
    assert np.max(np.abs(transition_one_rdm(up, dn, c, c, norb, time_sym, z) - one_rdm(up, dn, c, norb, time_sym, z))) <= 1e-13
    assert np.max(np.abs(transition_two_rdm(up, dn, c, c, norb, time_sym, z) - two_rdm(up, dn, c, norb, time_sym, z))) <= 1e-13
    a, b = rng.standard_normal(len(up)), rng.standard_normal(len(up))
    ab = transition_two_rdm(up, dn, a, b, norb, time_sym, z)
    assert np.max(np.abs(transition_two_rdm(up, dn, b, a, norb, time_sym, z) - ab.transpose(0, 1, 3, 2, 5, 4))) <= 1e-13
    # the polarisation identity: T(a,b) + T(b,a) = Gamma(a + b) - Gamma(a) - Gamma(b)
    ba = transition_one_rdm(up, dn, b, a, norb, time_sym, z)
    pol = one_rdm(up, dn, a + b, norb, time_sym, z) - one_rdm(up, dn, a, norb, time_sym, z) - one_rdm(up, dn, b, norb, time_sym, z)
    assert np.max(np.abs(transition_one_rdm(up, dn, a, b, norb, time_sym, z) + ba - pol)) <= 1e-12


def _single_excitation_tdm(norb, i, a, spin_sign):
    """gamma^sigma of bra = (a+_{a alpha} a_{i alpha} + spin_sign a+_{a beta} a_{i beta}) |HF> / sqrt2, ket = |HF>"""
    g = np.zeros((2, norb, norb))
    g[0, a, i] = 1.0 / np.sqrt(2.0)
    g[1, a, i] = spin_sign / np.sqrt(2.0)
    return g


def test_singlet_single_excitation():
    chem = systems.ChemSystem(C2_FCIDUMP)
    norb = chem.norb
    o = np.asarray(chem.orb_order[:norb]) - 1      # library orbital p is FCIDUMP orbital o[p]
    assert not np.array_equal(o, np.arange(norb))  # the mapping is exercised
    i, a = chem.nup - 1, chem.nup + 2
    res = natorb.natural_transition_orbitals(chem, _single_excitation_tdm(norb, i, a, +1), spin_sign=+1)
    sv = res["singular_values"]
    assert abs(sv[0] - np.sqrt(2.0)) <= 1e-14 and np.all(sv[1:] <= 1e-14)
    assert np.all(np.diff(sv) <= 0)
    assert res["participation_ratio"] == pytest.approx(1.0, abs=1e-14)
    assert res["weights"][0] == pytest.approx(1.0, abs=1e-14)
    assert np.max(np.abs(res["holes"][:, 0] - np.eye(norb)[o[i]])) <= 1e-14
    assert np.max(np.abs(res["particles"][:, 0] - np.eye(norb)[o[a]])) <= 1e-14
    # the same excitation read as triplet-coupled vanishes; a triplet-coupled one is seen with spin_sign = -1
    assert np.max(natorb.natural_transition_orbitals(chem, _single_excitation_tdm(norb, i, a, +1), spin_sign=-1)["singular_values"]) == 0
    trip = natorb.natural_transition_orbitals(chem, _single_excitation_tdm(norb, i, a, -1), spin_sign=-1)
    assert abs(trip["singular_values"][0] - np.sqrt(2.0)) <= 1e-14


@pytest.mark.parametrize("spin_sign", [1, -1])
def test_random_tdm_reconstructs(spin_sign):
    chem = systems.ChemSystem(C2_FCIDUMP)
    norb = chem.norb
    rng = np.random.default_rng(11 + spin_sign)
    g = rng.standard_normal((2, norb, norb))
    res = natorb.natural_transition_orbitals(chem, g, spin_sign=spin_sign)
    o = np.asarray(chem.orb_order[:norb]) - 1
    gf = np.zeros((norb, norb))
    gf[np.ix_(o, o)] = g[0] + spin_sign * g[1]
    P, Hh, sv = res["particles"], res["holes"], res["singular_values"]
    assert np.max(np.abs(P @ np.diag(sv) @ Hh.T - gf)) <= 1e-12
    assert np.max(np.abs(Hh.T @ Hh - np.eye(norb))) <= 1e-12 and np.max(np.abs(P.T @ P - np.eye(norb))) <= 1e-12
    for k in range(norb):
        assert Hh[np.argmax(np.abs(Hh[:, k])), k] > 0
    s2 = sv ** 2
    assert res["participation_ratio"] == pytest.approx(s2.sum() ** 2 / (s2 ** 2).sum(), rel=1e-14)
    assert np.sum(res["weights"]) == pytest.approx(1.0, abs=1e-14)


def test_bad_arguments():
    chem = systems.ChemSystem(C2_FCIDUMP)
    with pytest.raises(ValueError, match="spin_sign"):
        natorb.natural_transition_orbitals(chem, np.zeros((2, 26, 26)), spin_sign=0)
    with pytest.raises(ValueError, match="one pair"):
        natorb.natural_transition_orbitals(chem, np.zeros((3, 2, 26, 26)))
