"""Heat-bath determinant selection on the GPU (csrc/select.cu, SURVEY 8(f) item 1) against the oracle's restatement of
get_next_det_list, and the whole HCI variational loop (selection -> H build -> Davidson) on the GPU against the
reference's golden HEG log and the committed C2 fixture."""
import json
import os

import numpy as np
import pytest

from conftest import C2_FCIDUMP, C2_ORBSYM

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("time_sym", [False, True])
def test_select_step_matches_oracle(oracle, c2_space, c2_space_ts, time_sym):
    import sqmc_b200 as sq
    s, r = c2_space_ts if time_sym else c2_space
    up, dn = r["up"], r["dn"]
    n = len(up)
    coeffs = np.abs(r["wts"][:, 0])
    rng = np.random.default_rng(8)
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=time_sym, z=1))
    for eps, min_h in ((1e-3, np.full(n, 9e99)), (5e-4, 10.0 ** rng.uniform(-3, 0, n))):
        ref_up, ref_dn, ref_mh = s.select(up, dn, coeffs, min_h, eps)
        got_up, got_dn, got_mh = H.get_next_det_list(up, dn, coeffs, min_h, eps)
        assert len(ref_up) > 0
        assert np.array_equal(got_up, ref_up) and np.array_equal(got_dn, ref_dn)
        assert np.array_equal(got_mh, ref_mh)


def test_select_step_heg(oracle, heg_space):
    import sqmc_b200 as sq
    s, r = heg_space
    n = 277
    up, dn = r["up"][:n], r["dn"][:n]
    S2 = oracle.System.heg(3, 0.5, 14, 7, 1.49)
    r1 = S2.hci(1e-3, n_states=1, max_iters=1)
    coeffs = np.abs(r1["wts"][:, 0])
    ref_up, ref_dn, ref_mh = S2.select(up, dn, coeffs, np.full(n, 9e99), 1e-3)
    assert n + len(ref_up) == 9475  # golden: src/e2e_tests/heg/o_det_ref:330
    H = sq.SparseHamiltonian(sq.HegSystem(3, 0.5, 14, 7, 1.49))
    got_up, got_dn, got_mh = H.get_next_det_list(up, dn, coeffs, np.full(n, 9e99), 1e-3)
    assert np.array_equal(got_up, ref_up) and np.array_equal(got_dn, ref_dn) and np.array_equal(got_mh, ref_mh)


def _hci_on_gpu(H, hf_up, hf_dn, sched, n_states=1, max_iters=50, trace=None):
    """perform_hci (hci.f90:359-517) with selection, build and Davidson all on the GPU; trace, a list, receives the
    (new up, new dn, updated min_H) of every selection step."""
    import sqmc_b200 as sq
    up = sq.dets_to_u64([hf_up])
    dn = sq.dets_to_u64([hf_dn])
    wts = np.ones((1, n_states))
    min_h = np.full(1, 9e99)
    energy = np.array([H.diagonal(up, dn)[0]] + [0.0] * (n_states - 1))
    log = []
    eps_last = sched[-1]
    for it in range(1, max_iters + 1):
        eps = sched[min(it, len(sched)) - 1]
        n_old = len(up)
        coeffs = np.abs(wts).max(axis=1) if it > 1 else wts[:, 0].copy()
        nu, nd, min_h = H.get_next_det_list(up, dn, coeffs, min_h, eps)
        if trace is not None:
            trace.append((nu, nd, min_h.copy()))
        n_new = n_old + len(nu)
        min_h = np.concatenate([min_h, np.full(len(nu), 9e99)])
        if n_new == n_old:
            continue
        if n_new <= int(1.00001 * n_old) and eps == eps_last:
            break
        up, dn = np.concatenate([up, nu]), np.concatenate([dn, nd])
        nnz = H.generate_sparse_ham_upper_triangular(up, dn, ndet_old=n_old)
        v0 = np.zeros((n_new, n_states))
        if it == 1:
            for k in range(n_states):
                v0[k, k] = 1.0
        else:
            v0[:n_old] = wts
        d = H.davidson_sparse(n_states=n_states, initial_vector=v0)
        wts, old_energy, energy = d["evecs"], energy, d["evals"].copy()
        log.append((n_new, nnz, energy.copy()))
        if np.max(np.abs(energy - old_energy)) < 1e-5 and eps == eps_last:
            break
    return up, dn, wts, log


def test_heg_hci_loop_fully_on_gpu_reproduces_reference_log():
    import sqmc_b200 as sq
    gold = json.load(open(os.path.join(HERE, "golden", "heg_o_det_ref.json")))
    hs = sq.HegSystem(3, 0.5, 14, 7, 1.49)
    H = sq.SparseHamiltonian(hs)
    up, dn, wts, log = _hci_on_gpu(H, hs.hf_up, hs.hf_dn, [1e-3] * 30, max_iters=2)
    assert [l[0] for l in log] == gold["n_det"]          # 277, 9475
    assert [l[1] for l in log] == gold["nnz"]            # 3511, 165193
    for k in range(2):
        assert abs(log[k][2][0] - gold["davidson_final"][k]["energy"]) < 2e-9   # 58.2825967049, 58.2769060846
    where = {(int(u[0]), int(d[0])): i for i, (u, d) in enumerate(zip(up, dn))}
    sign = np.sign(wts[0, 0])
    for c in gold["final_coefficients"]:                 # CI coefficients incl. signs, o_det_ref:394-413
        assert abs(sign * wts[where[(c["up"], c["dn"])], 0] - c["coef"]) < 1e-8


def test_c2_hci_loop_fully_on_gpu_matches_fixture():
    import sqmc_b200 as sq
    gold = json.load(open(os.path.join(HERE, "golden", "c2_s1_hci.json")))["runs"]["n_states=1"]
    cs = sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1)
    H = sq.SparseHamiltonian(cs)
    sched = [2e-3, 2e-3] + [1e-3] * 28
    up, dn, wts, log = _hci_on_gpu(H, cs.hf_up, cs.hf_dn, sched)
    assert [l[0] for l in log] == gold["n_det"]
    assert [l[1] for l in log] == gold["nnz"]
    assert np.max(np.abs(np.array([l[2][0] for l in log]) - np.array(gold["iter_energy"])[:, 0])) < 1e-8
    assert abs(log[-1][2][0] - gold["energy"][0]) < 1e-8   # C2 cc-pVDZ HCI variational energy, eps_var = 1e-3


def test_c2_eps_scheduled_hci_space_matches_oracle_golden():
    """spaces.hci_space (the bench workload's recipe) stopped at eps_var = 1e-4: sizes, nnz, energies and the exact
    determinant list (SHA-256 over the label-sorted list) equal the oracle's perform_hci run (tests/golden/c2_hci_sched.json)."""
    import hashlib
    import sqmc_b200 as sq
    from sqmc_b200 import spaces
    gold = json.load(open(os.path.join(HERE, "golden", "c2_hci_sched.json")))
    cs = sq.ChemSystem(C2_FCIDUMP)
    H = sq.SparseHamiltonian(cs)
    log = []
    up, dn, wts, e = spaces.hci_space(H, cs, 10**9, eps_schedule=gold["eps_var_sched"], log=log)
    assert [l["n_dets"] for l in log] == gold["n_det"]
    assert [l["nnz_upper"] for l in log] == gold["nnz"]
    assert np.max(np.abs(np.array([l["energy"] for l in log]) - np.array(gold["iter_energy"]))) < 1e-8
    order = np.lexsort((dn[:, 0], up[:, 0]))
    dig = hashlib.sha256(np.ascontiguousarray(np.stack([up[order, 0], dn[order, 0]], axis=1)).tobytes()).hexdigest()
    assert dig == gold["sha256_sorted_up_dn_u64"]
