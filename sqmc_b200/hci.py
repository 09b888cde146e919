"""Host-side mirror of perform_hci (hci.f90:66-862): the variational HCI loop and the deterministic second-order
correction, every heavy step through the GPU library (selection -> H build -> Davidson -> PT), plus a reader for the
reference's positional input files so its shipped inputs can be run as they are.

Loop rules restated from the reference (hci.f90:359-517; do_walk.f90:418-533):
  * eps_var schedule: 30 entries, eps_var_sched padded with eps_var, each entry max(entry, eps_var) (do_walk.f90:425);
  * iteration 1 selects with the signed coefficient of state 1, later iterations with max_state |c_i| (hci.f90:369-382);
  * stop when the list grew by <= 0.001 % or max|dE| < 1e-5, both only once eps_var reached its last value (:420,502),
    or after 50 iterations (:89);
  * Davidson starts from the previous vectors padded with zeros, from unit vectors in iteration 1 (:453-485);
  * PT per state: second_order_pt with eps_pt on the final wavefunction (do_pt, :4220-4243).
Out of scope here: active spaces, stochastic PT (n_mc > 0, eps_pt_big).  Natural orbitals of the final wavefunction:
natorb.py and scripts/natorb.py; its single-particle Green's function: greens.py and scripts/greens.py.
"""
import re

import numpy as np


def eps_schedule(eps_var, eps_var_sched=()):
    sched = np.full(30, float(eps_var))
    for k, e in enumerate(list(eps_var_sched)[:30]):
        sched[k] = e
    return np.maximum(sched, eps_var)


def sort_by_label(up, dn, wts):
    """the variational wavefunction sorted by (up, dn) as 128-bit integers: what the reference does before the checkpoint
    dump and the PT (hci.f90:569-596, merge_sort2_up_dn)"""
    order = np.lexsort((dn[:, 0], dn[:, 1], up[:, 0], up[:, 1]))
    return up[order], dn[order], wts[order]


def perform_hci(H, system, eps_var, eps_var_sched=(), n_states=1, max_iters=50, eps_pt=None, log=None, wf_dir=None, dump_wf_var=False):
    """-> dict(up, dn, wts (n, n_states), energy (n_states,), iterations=[{n_det, nnz, energy}], pt=[(delta_e, ndets_connected)]).
    H: SparseHamiltonian of `system` (chem / heg).  log: optional callable receiving one line of text per event.
    wf_dir: directory of the `wf_eps_var=...` checkpoint: if the file of this eps_var exists the variational stage is
    skipped and the wavefunction is read from it (hci.f90:194-231); with dump_wf_var it is written after the stage
    (:601-625).  The returned wavefunction is sorted by label like the reference's."""
    import os
    from . import formats
    from .api import dets_to_u64
    say = log or (lambda *_: None)
    sched = eps_schedule(eps_var, eps_var_sched)
    eps_last = sched[29]
    wf_path = os.path.join(wf_dir, formats.wf_filename(float(np.min(sched)))) if wf_dir else None
    if wf_path and os.path.exists(wf_path):
        say("Reading variational wavefn from %s" % wf_path)
        ck = formats.read_wf(wf_path)
        if ck["wts"].shape[1] != n_states:
            raise ValueError("perform_hci: checkpoint holds %d states, run asks for %d" % (ck["wts"].shape[1], n_states))
        out = dict(up=ck["up"], dn=ck["dn"], wts=ck["wts"], energy=np.array(ck["energies"]), iterations=[], pt=[], from_checkpoint=True)
        return _pt_stage(H, out, n_states, eps_pt, say)
    hf_up, hf_dn = int(system.hf_up), int(system.hf_dn)
    if getattr(system, "time_sym", False) and hf_dn < hf_up:
        hf_up, hf_dn = hf_dn, hf_up
    up, dn = dets_to_u64([hf_up]), dets_to_u64([hf_dn])
    wts = np.zeros((1, n_states))
    wts[0, 0] = 1.0
    energy = np.zeros(n_states)
    energy[0] = H.diagonal(up, dn)[0]
    old_energy = energy.copy()
    min_h = np.full(1, 9.0e99)
    iterations = []
    eps = sched[0]
    for it in range(1, max_iters + 1):
        if it <= 30:
            eps = sched[it - 1]
        n_old = len(up)
        coeffs = np.max(np.abs(wts), axis=1) if it > 1 else wts[:, 0].copy()
        nu, nd, min_h_new = H.get_next_det_list(up, dn, coeffs, min_h, eps)
        n_new = n_old + len(nu)
        if n_new == n_old:
            # hci.f90:413-417 "Cycling hci iteration because ndets_global_new==ndets_global_old": no rebuild, no Davidson;
            # min_H_already_done was already updated inside get_next_det_list (hci.f90:1014-1016)
            min_h = min_h_new
            say("Cycling hci iteration because ndets_global_new==ndets_global_old")
            continue
        if n_new <= int(1.00001 * n_old) and eps == eps_last:
            break
        up, dn = np.concatenate([up, nu]), np.concatenate([dn, nd])
        min_h = np.concatenate([min_h_new, np.full(len(nu), 9.0e99)])
        v0 = np.zeros((n_new, n_states))
        if it == 1:
            for s in range(min(n_states, n_new)):
                v0[s, s] = 1.0
        else:
            v0[:n_old, :] = wts
        nnz = H.generate_sparse_ham_upper_triangular(up, dn, ndet_old=n_old)
        d = H.davidson_sparse(n_states=n_states, initial_vector=v0)
        wts, energy = d["evecs"], np.array(d["evals"], dtype=np.float64)
        iterations.append({"n_det": int(n_new), "nnz": int(nnz), "energy": [float(e) for e in energy], "eps_var": float(eps)})
        say("HCI iteration %d: eps_var=%.3e n_det=%d nnz=%d E=%s" % (it, eps, n_new, nnz, " ".join("%.9f" % e for e in energy)))
        md = float(np.max(np.abs(energy - old_energy)))
        old_energy = energy.copy()
        if md < 1.0e-5 and eps == eps_last:
            break
    up, dn, wts = sort_by_label(up, dn, wts)
    out = dict(up=up, dn=dn, wts=wts, energy=energy, iterations=iterations, pt=[], from_checkpoint=False)
    if wf_path and dump_wf_var:
        say("Writing variational wavefn to %s" % wf_path)
        formats.write_wf(wf_path, up, dn, wts, energy)
    return _pt_stage(H, out, n_states, eps_pt, say)


def _pt_stage(H, out, n_states, eps_pt, say):
    if eps_pt is not None and eps_pt > 0:
        up, dn, wts, energy = out["up"], out["dn"], out["wts"], out["energy"]
        for s in range(n_states):
            de, nconn = H.second_order_pt(up, dn, wts[:, s], energy[s], eps_pt)
            out["pt"].append((de, nconn))
            say("state %d: ndets, ndets_connected, Variational, PT, Total Energies= %d %d %.9f %.9f %.9f"
                % (s + 1, len(up), nconn, energy[s], de, energy[s] + de))
            # the two lines the reference's own end-to-end checker greps (src/e2e_tests/e2e_check.py; hci.f90 log format)
            say("Variational energy=%31.9f" % energy[s])
            say("Second-order PT energy lowering=%18.9f" % de)
    return out


# ----------------------------------------------------------------------------- reference input files
def _namelist(text, name):
    m = re.search(r"&" + name + r"\b(.*?)/", text, flags=re.S | re.I)
    out = {}
    if not m:
        return out
    for key, val in re.findall(r"(\w+)\s*=\s*([^=]*?)(?=\s+\w+\s*=|\s*$)", m.group(1).strip(), flags=re.S):
        items = []
        for tok in re.split(r"[,\s]+", val.strip()):
            if not tok:
                continue
            rep = re.match(r"(\d+)\*(.+)", tok)          # Fortran repeat count, e.g. 2*2e-3
            items += [rep.group(2)] * int(rep.group(1)) if rep else [tok]
        out[key.lower()] = items
    return out


def _logical(tok):
    return tok.strip().strip(".").lower() in ("t", "true")


def read_input(path):
    """The positional input of an `hci` run (SURVEY.md appendix A; do_walk.f90:231-533, chemistry.f90:136-248, heg.f90:119-166).
    Handles the two layouts the reference ships: the short HCI layout (C2_v2z_curve/*/i_*) and the full layout whose
    QMC lines precede run_type (src/e2e_tests/heg/i_det).  -> dict"""
    text = "\n".join(ln for ln in open(path).read().splitlines() if not ln.lstrip().startswith("!"))   # '!' lines are comments
    lines = [ln for ln in text.splitlines() if ln.strip() and not ln.lstrip().startswith("&")]
    k = next(i for i, ln in enumerate(lines) if ln.split()[0].strip("'\"").lower() == "hci")
    t = lines[k + 1].split()
    cfg = {"run_type": "hci", "eps_var": float(t[0]), "eps_pt": float(t[1]), "target_error": float(t[2]), "n_states": int(t[3]) if len(t) > 3 and re.fullmatch(r"\d+", t[3]) else 1,
           "dump_wf_var": _logical(lines[k + 2].split()[0])}
    j = next(i for i in range(k + 2, len(lines)) if lines[i].lstrip().startswith(("'", '"')))
    cfg["hamiltonian_type"] = lines[j].split()[0].strip("'\"").lower()
    body = lines[j + 1:]
    if cfg["hamiltonian_type"] == "chem":
        cfg["nelec"], cfg["nup"] = int(body[0].split()[0]), int(body[0].split()[1])
        cfg["point_group"] = body[1].split()[0].lower()
        cfg["time_sym"] = _logical(body[2].split()[0])
        p = 3
        cfg["z"] = 1
        if cfg["time_sym"]:
            cfg["z"] = int(body[p].split()[0]); p += 1
        cfg["norb"] = int(body[p].split()[0]); p += 1
        cfg["orbital_symmetries"] = [int(x) for x in re.split(r"[,\s]+", body[p].split("orbital")[0].strip().rstrip(",")) if x][:cfg["norb"]]
        p += 1
        cfg["spatial_symmetry_wf"] = int(body[p].split()[0])
    elif cfg["hamiltonian_type"] == "heg":
        cfg["n_dim"] = int(body[0].split()[0])
        cfg["r_s"] = float(body[1].split()[0])
        cfg["nelec"], cfg["nup"] = int(body[2].split()[0]), int(body[2].split()[1])
        cfg["cutoff_radius"] = float(body[3].split()[0])
    else:
        raise ValueError("read_input: hamiltonian_type %r is not an HCI system of this path" % cfg["hamiltonian_type"])
    sel = _namelist(text, "selected_ci")
    cfg["eps_var_sched"] = [float(x) for x in sel.get("eps_var_sched", [])]
    if "n_states" in sel:
        cfg["n_states"] = int(sel["n_states"][0])
    cfg["n_mc"] = int(sel["n_mc"][0]) if "n_mc" in sel else None
    hf = _namelist(text, "hf_det")
    cfg["hf_symmetry"] = int(hf["hf_symmetry"][0]) if "hf_symmetry" in hf else None
    return cfg


def run_input(path, fcidump=None, device=0, log=print, wf_dir=None):
    """Run a reference `hci` input file on the GPU path: system set-up, variational loop, deterministic PT.
    wf_dir: where the `wf_eps_var=...` checkpoint is looked for / dumped (the reference uses the working directory)."""
    import os
    from . import ChemSystem, HegSystem, SparseHamiltonian
    cfg = read_input(path)
    if cfg["hamiltonian_type"] == "chem":
        fcidump = fcidump or os.path.join(os.path.dirname(os.path.abspath(path)), "FCIDUMP")
        system = ChemSystem(fcidump, nelec=cfg["nelec"], nup=cfg["nup"], orbital_symmetries=cfg["orbital_symmetries"],
                            time_sym=cfg["time_sym"], z=cfg["z"])
    else:
        system = HegSystem(cfg["n_dim"], cfg["r_s"], cfg["nelec"], cfg["nup"], cfg["cutoff_radius"])
    H = SparseHamiltonian(system, device=device)
    res = perform_hci(H, system, cfg["eps_var"], cfg["eps_var_sched"], n_states=cfg["n_states"], eps_pt=cfg["eps_pt"], log=log,
                      wf_dir=wf_dir, dump_wf_var=cfg["dump_wf_var"])
    res["config"] = cfg
    res["system"], res["hamiltonian"] = system, H
    return res
