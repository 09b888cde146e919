"""Host-side mirror of the reference's interface for the hot path.

Names follow the Fortran entry points they stand in for (paths relative to
/root/reference/src):

  SparseHamiltonian.generate_sparse_ham_upper_triangular
        generate_sparse_ham_chem_upper_triangular   chemistry.f90:7639
        generate_sparse_ham_heg_upper_triangular    heg.f90:3553
        generate_sparse_ham_hubbardk_upper_triangular hubbard.f90:9435
  SparseHamiltonian.fast_sparse_matrix_multiply_upper_triangular
        more_tools.f90:3622 (and _mpi :3674, _local_band :3562)
  SparseHamiltonian.davidson_sparse                 more_tools.f90:2018 / :2525
  SparseHamiltonian.projector_step                  do_walk.f90:2255-2325

Everything is a thin call into the C ABI of libsqmc_b200.so; there is no Python
or CPU implementation of any of it here.  Determinants are python ints or
(n,2) uint64 arrays (little-endian 128-bit = Fortran integer(16)).
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import SqmcError, check


def dets_to_u64(dets):
    a = np.asarray(dets)
    if a.dtype == np.uint64 and a.ndim == 2 and a.shape[1] == 2:
        return np.ascontiguousarray(a)
    out = np.zeros((len(dets), 2), dtype=np.uint64)
    for k, d in enumerate(dets):
        d = int(d)
        out[k, 0] = d & 0xFFFFFFFFFFFFFFFF
        out[k, 1] = d >> 64
    return out


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class SparseHamiltonian:
    """Opaque device-resident H for one system (chem / heg / hubbardk)."""

    def __init__(self, system, device=0):
        from . import systems
        _lib.init(device=device)
        self._L = _lib.load()
        self._h = C.c_void_p()
        self.system = system
        self.n = 0
        self.n_owned = 0
        L = self._L
        if isinstance(system, systems.ChemSystem):
            integrals = np.ascontiguousarray(system.integrals, dtype=np.float64)
            c2 = np.asfortranarray(system.combine_2, dtype=np.int32)
            check(L.sqmc_b200_system_chem(C.byref(self._h), system.norb, system.nup, system.ndn, _p(integrals), len(integrals),
                                          c2.ctypes.data_as(C.c_void_p), int(system.time_sym), int(system.z)))
            sym = np.ascontiguousarray(system.orbital_symmetries, dtype=np.int32)
            check(L.sqmc_b200_system_orbital_symmetries(self._h, _p(sym)))
        elif isinstance(system, systems.HegSystem):
            kv = np.ascontiguousarray(system.k_vectors, dtype=np.float64)
            check(L.sqmc_b200_system_heg(C.byref(self._h), system.norb, system.n_dim, _p(kv), float(system.length_cell),
                                         system.nup, system.ndn))
        elif isinstance(system, systems.HubbardKSystem):
            kv = np.ascontiguousarray(system.k_vectors, dtype=np.int32)
            ke = np.ascontiguousarray(system.k_energies, dtype=np.float64)
            check(L.sqmc_b200_system_hubbardk(C.byref(self._h), system.l_x, system.l_y, _p(kv), _p(ke), float(system.ubyn),
                                              system.nup, system.ndn))
        else:
            raise SqmcError("unknown system type %r" % type(system))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.sqmc_b200_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- selection -----------------------------------------------------
    def get_next_det_list(self, dets_up, dets_dn, coeffs, min_H_already_done, eps_var):
        """hci.f90:865 get_next_det_list: returns (new_up, new_dn) = the determinants to append (sorted by label, not yet in
        the list) and the updated min_H_already_done of the old determinants."""
        up, dn = dets_to_u64(dets_up), dets_to_u64(dets_dn)
        c = np.ascontiguousarray(coeffs, dtype=np.float64)
        mh = np.array(min_H_already_done, dtype=np.float64)
        nn = C.c_int64()
        check(self._L.sqmc_b200_hci_select(self._h, len(up), _p(up), _p(dn), _p(c), _p(mh), float(eps_var), C.byref(nn)))
        nu = np.zeros((nn.value, 2), dtype=np.uint64)
        nd = np.zeros((nn.value, 2), dtype=np.uint64)
        check(self._L.sqmc_b200_hci_new_dets(self._h, _p(nu), _p(nd)))
        return nu, nd, mh

    # ---- build ---------------------------------------------------------
    def generate_sparse_ham_upper_triangular(self, dets_up, dets_dn, ndet_old=0, hf_to_psit=False):
        """Build H over the determinant list (caller order). Returns nnz of the
        reference's upper-triangular format (its "# of nonzero elem in H")."""
        up, dn = dets_to_u64(dets_up), dets_to_u64(dets_dn)
        if len(up) != len(dn):
            raise SqmcError("dets_up / dets_dn length mismatch")
        check(self._L.sqmc_b200_set_hf_to_psit(self._h, int(bool(hf_to_psit))))
        nnz = C.c_int64()
        check(self._L.sqmc_b200_build_h(self._h, len(up), _p(up), _p(dn), int(ndet_old), C.byref(nnz)))
        self.n = len(up)
        return nnz.value

    def last_build_incremental(self):
        """True when the last build extended the previous matrix (sparse_ham%ndet reuse, chemistry.f90:7769-7843)."""
        return self._L.sqmc_b200_last_build_incremental(self._h) == 1

    def import_upper(self, H_nonzero_elements, H_indices, H_values):
        cnt = np.ascontiguousarray(H_nonzero_elements, dtype=np.int64)
        idx = np.ascontiguousarray(H_indices, dtype=np.int64)
        val = np.ascontiguousarray(H_values, dtype=np.float64)
        check(self._L.sqmc_b200_import_upper(self._h, len(cnt), _p(cnt), _p(idx), _p(val)))
        self.n = len(cnt)

    def dump_dtm_projector(self, path, dets_up, dets_dn, dtm_energy=0.0, tau=None, n_core_orb=0):
        """Write the resident matrix as the reference's deterministic-projector text file (do_walk.f90:964-1013).
        The file holds H itself; pass tau when the handle currently stores -tau*H (after scale_values(-tau))."""
        from . import formats
        cnt, idx, val = self.export_upper()
        if tau is not None:
            val = -val / tau          # do_walk.f90:1007
        formats.write_dtm_projector(path, dets_up, dets_dn, cnt, idx, val, dtm_energy=dtm_energy, n_core_orb=n_core_orb)

    def load_dtm_projector(self, path, tau, nup, ndn, n_core_orb=0):
        """Read a deterministic-projector file and keep -tau*H resident (do_walk.f90:883-945: the values are multiplied
        by -tau right after the read).  -> (imp_up, imp_dn) of the file."""
        from . import formats
        d = formats.read_dtm_projector(path, nup, ndn, n_core_orb=n_core_orb)
        self.import_upper(d["counts"], d["indices"], d["values"])
        self.scale_values(-tau)
        return d["up"], d["dn"]

    def nnz(self):
        n, u, f = C.c_int64(), C.c_int64(), C.c_int64()
        check(self._L.sqmc_b200_nnz(self._h, C.byref(n), C.byref(u), C.byref(f)))
        return dict(n=n.value, nnz_upper=u.value, nnz_full=f.value)

    def local_rows(self):
        r, z = C.c_int64(), C.c_int64()
        check(self._L.sqmc_b200_local_rows(self._h, C.byref(r), C.byref(z)))
        return r.value, z.value

    def export_upper(self):
        """-> (H_nonzero_elements int64[n], H_indices int64[nnz] 1-based, H_values f64[nnz])"""
        info = self.nnz()
        nloc, _ = self.local_rows()
        cnt = np.zeros(nloc, dtype=np.int64)
        idx = np.zeros(info["nnz_upper"], dtype=np.int64)
        val = np.zeros(info["nnz_upper"], dtype=np.float64)
        check(self._L.sqmc_b200_export_upper(self._h, _p(cnt), _p(idx), _p(val)))
        tot = int(cnt.sum())
        return cnt, idx[:tot], val[:tot]

    def get_row(self, caller_row, cap=1 << 16):
        """full row `caller_row` (1-based): (columns 1-based ascending, values); None if another rank owns it."""
        cols = np.zeros(cap, dtype=np.int64)
        vals = np.zeros(cap)
        ln = C.c_int64()
        check(self._L.sqmc_b200_get_row(self._h, int(caller_row), cap, _p(cols), _p(vals), C.byref(ln)))
        if ln.value < 0:
            return None
        return cols[:ln.value].copy(), vals[:ln.value].copy()

    def diagonal(self, dets_up, dets_dn):
        up, dn = dets_to_u64(dets_up), dets_to_u64(dets_dn)
        out = np.zeros(len(up))
        check(self._L.sqmc_b200_diagonal(self._h, len(up), _p(up), _p(dn), _p(out)))
        return out

    def build_times(self):
        t = np.zeros(8)
        check(self._L.sqmc_b200_build_times(self._h, _p(t)))
        return dict(prep_ms=t[0], count_ms=t[1], fill_sort_ms=t[2], eval_compact_ms=t[3], total_ms=t[4],
                    candidates=int(t[5]), alpha_strings=int(t[6]), beta_strings=int(t[7]))

    def perm(self):
        p = np.zeros(self.n, dtype=np.int64)
        check(self._L.sqmc_b200_get_perm(self._h, _p(p)))
        return p

    # ---- H.v -------------------------------------------------------------
    def fast_sparse_matrix_multiply_upper_triangular(self, vector):
        """answer = H . vector; vector (n,) or (n, nvec) in caller row order."""
        x = np.asarray(vector, dtype=np.float64)
        one = x.ndim == 1
        xf = np.asfortranarray(x.reshape(self.n, -1))
        y = np.zeros_like(xf, order="F")
        check(self._L.sqmc_b200_matvec(self._h, _p(xf), _p(y), xf.shape[1], self.n))
        return y[:, 0].copy() if one else np.ascontiguousarray(y)

    matvec = fast_sparse_matrix_multiply_upper_triangular

    def scale_values(self, ratio):
        check(self._L.sqmc_b200_scale_values(self._h, float(ratio)))

    def set_row_bundle(self, rows_per_bundle):
        """storage-order hint for H.v: 0 = plain CSR rows, 2/4/8 = column-merged bundles of that many rows (csrc/bundle.cu)."""
        check(self._L.sqmc_b200_set_row_bundle(self._h, int(rows_per_bundle)))

    def projector_step(self, tau, e_trial, w):
        """deltaw = Hstored.w + e_trial*tau*w (do_walk.f90:2259-2290)."""
        w = np.ascontiguousarray(w, dtype=np.float64)
        dw = np.zeros_like(w)
        check(self._L.sqmc_b200_projector(self._h, float(tau), float(e_trial), _p(w), _p(dw)))
        return dw

    # ---- the caller's data distribution (MPI ranks own hashed subsets of the determinants) ----
    def set_ownership(self, owner_of_row):
        """owner_of_row[i] = rank owning determinant i of the list last built (get_det_owner, mpi_routines.f90:419).
        -> number of determinants this rank owns (my_nimp).  Repeat after every build."""
        o = np.ascontiguousarray(owner_of_row, dtype=np.int32)
        if len(o) != self.n:
            raise SqmcError("set_ownership: owner_of_row must have n entries")
        m = C.c_int64()
        check(self._L.sqmc_b200_set_ownership(self._h, _p(o), C.byref(m)))
        self.n_owned = m.value
        return m.value

    def matvec_local(self, x_local, out=None):
        """fast_sparse_matrix_multiply_local_band + mpi_redscatt_real_dparray (do_walk.f90:2259-2260): owned slice in, owned slice out."""
        x = np.ascontiguousarray(x_local, dtype=np.float64)
        y = np.zeros_like(x) if out is None else out
        check(self._L.sqmc_b200_matvec_local(self._h, _p(x), _p(y), 1, max(self.n_owned, 1)))
        return y

    def projector_step_local(self, tau, e_trial, w_local, out=None):
        w = np.ascontiguousarray(w_local, dtype=np.float64)
        dw = np.zeros_like(w) if out is None else out
        check(self._L.sqmc_b200_projector_local(self._h, float(tau), float(e_trial), _p(w), _p(dw)))
        return dw

    def davidson_sparse_local(self, n_states=1, initial_vector_local=None, tol=1.0e-10, max_vec_per_state=50):
        """davidson_sparse_mpi2 (more_tools.f90:2525): vectors are the owned slices (n_owned x n_states)."""
        m = self.n_owned
        v0 = None
        if initial_vector_local is not None:
            v0 = np.asfortranarray(np.asarray(initial_vector_local, dtype=np.float64).reshape(m, n_states))
        evecs = np.zeros((max(m, 1), n_states), order="F")
        evals = np.zeros(n_states)
        cap = 1024
        ritz = np.zeros(cap * n_states)
        nmv, nlog = C.c_int(), C.c_int()
        check(self._L.sqmc_b200_davidson_local(self._h, n_states, _p(v0), _p(evecs), _p(evals), float(tol), int(max_vec_per_state),
                                               C.byref(nmv), _p(ritz), cap, C.byref(nlog)))
        k = min(nlog.value, cap)
        return dict(evals=evals, evecs=np.ascontiguousarray(evecs[:m]), ritz=ritz[:k * n_states].reshape(k, n_states), n_matvec=nmv.value)

    def register_host(self, array):
        check(self._L.sqmc_b200_register_host(_p(array), array.nbytes))

    def unregister_host(self, array):
        check(self._L.sqmc_b200_unregister_host(_p(array)))

    def exchange_mode(self):
        return {0: "single", 1: "nvlink-peer-stores", 2: "nccl"}[self._L.sqmc_b200_exchange_mode(self._h)]

    # ---- Davidson ----------------------------------------------------------
    def davidson_sparse(self, n_states=1, initial_vector=None, tol=1.0e-10, max_vec_per_state=50):
        n = self.n
        v0 = None
        if initial_vector is not None:
            v0 = np.asfortranarray(np.asarray(initial_vector, dtype=np.float64).reshape(n, n_states))
        evecs = np.zeros((n, n_states), order="F")
        evals = np.zeros(n_states)
        cap = 1024
        ritz = np.zeros(cap * n_states)
        nmv, nlog = C.c_int(), C.c_int()
        check(self._L.sqmc_b200_davidson(self._h, n_states, _p(v0), _p(evecs), _p(evals), float(tol), int(max_vec_per_state),
                                         C.byref(nmv), _p(ritz), cap, C.byref(nlog)))
        k = min(nlog.value, cap)
        return dict(evals=evals, evecs=np.ascontiguousarray(evecs), ritz=ritz[:k * n_states].reshape(k, n_states),
                    n_matvec=nmv.value)

    def matrix_lanczos_sparse(self, initial_vector=None, tol=1.0e-10, max_iter=50):
        """matrix_lanczos_sparse (more_tools.f90:1742-1883) on the resident matrix ->
        dict(lowest_eigenvalue, highest_eigenvalue, second_lowest_eigenvalue, lowest_eigenvector, ritz, n_iter)."""
        n = self.n
        evec = np.zeros(n)
        eig3 = np.zeros(3)
        ritz = np.zeros(max_iter + 2)
        nit, nlog = C.c_int(), C.c_int()
        v0p = None
        if initial_vector is not None:
            v0 = np.ascontiguousarray(initial_vector, dtype=np.float64).reshape(-1)
            if len(v0) != n:
                raise ValueError("initial_vector must have n entries")
            v0p = _p(v0)
        check(self._L.sqmc_b200_lanczos(self._h, v0p, _p(evec), _p(eig3), float(tol), int(max_iter), C.byref(nit), _p(ritz), len(ritz), C.byref(nlog)))
        return dict(lowest_eigenvalue=eig3[0], highest_eigenvalue=eig3[1], second_lowest_eigenvalue=eig3[2], lowest_eigenvector=evec,
                    ritz=ritz[:nlog.value].copy(), n_iter=nit.value)

    def one_rdm(self, dets_up, dets_dn, wts):
        """One-particle density matrices <Psi_s| a+_{p sigma} a_{q sigma} |Psi_s> of the wavefunctions wts (n,) or (n, n_states)
        over the determinant list (any order, no built matrix needed; on time_sym systems the representatives).  Orbitals are
        the bits of the determinant words (chem: the reordered numbering, see natorb.natural_orbitals).  No normalisation.
        -> float64 array [s, sigma, p, q] of shape (n_states, 2, norb, norb), sigma 0 = up, 1 = dn; (2, norb, norb) for 1-D wts."""
        up = np.ascontiguousarray(dets_up, dtype=np.uint64).reshape(-1, 2)
        dn = np.ascontiguousarray(dets_dn, dtype=np.uint64).reshape(-1, 2)
        w = np.asarray(wts, dtype=np.float64)
        one = w.ndim == 1
        w = np.asfortranarray(w.reshape(-1, 1) if one else w)
        if len(dn) != len(up) or w.shape[0] != len(up):
            raise ValueError("one_rdm: dets_up, dets_dn and wts must have the same number of rows")
        norb, ns = self.system.norb, w.shape[1]
        out = np.zeros((ns, 2, norb, norb))
        check(self._L.sqmc_b200_one_rdm(self._h, len(up), _p(up), _p(dn), ns, _p(w), max(w.shape[0], 1), _p(out)))
        # the library stores (p,q) at p + norb*q: the [s, sigma] block read in C order is gamma transposed
        out = np.ascontiguousarray(out.transpose(0, 1, 3, 2))
        return out[0] if one else out

    def two_rdm(self, dets_up, dets_dn, wts):
        """Two-particle density matrices Gamma^{st}_{pq,rs} = <Psi_k| a+_{p s} a+_{r t} a_{s t} a_{q s} |Psi_k> (chemists' order:
        1/2 sum (pq|rs) Gamma over aa, ab, ba = ab and bb is the two-body energy) of the wavefunctions wts (n,) or (n, n_states),
        with the determinant list, orbital numbering and normalisation of one_rdm; norb <= 64.
        -> float64 array [k, b, p, q, r, s] of shape (n_states, 3, norb, norb, norb, norb), b = 0 (alpha alpha), 1 (alpha beta),
        2 (beta beta); (3, norb, norb, norb, norb) for 1-D wts."""
        up = np.ascontiguousarray(dets_up, dtype=np.uint64).reshape(-1, 2)
        dn = np.ascontiguousarray(dets_dn, dtype=np.uint64).reshape(-1, 2)
        w = np.asarray(wts, dtype=np.float64)
        one = w.ndim == 1
        w = np.asfortranarray(w.reshape(-1, 1) if one else w)
        if len(dn) != len(up) or w.shape[0] != len(up):
            raise ValueError("two_rdm: dets_up, dets_dn and wts must have the same number of rows")
        norb, ns = self.system.norb, w.shape[1]
        out = np.zeros((ns, 3) + (norb,) * 4) if norb <= 64 else np.zeros(1)   # the library rejects norb > 64
        check(self._L.sqmc_b200_two_rdm(self._h, len(up), _p(up), _p(dn), ns, _p(w), max(w.shape[0], 1), _p(out)))
        # the library stores (p,q,r,s) at p + norb*(q + norb*(r + norb*s)): the [k, b] block read in C order is [s, r, q, p]
        out = np.ascontiguousarray(out.transpose(0, 1, 5, 4, 3, 2))
        return out[0] if one else out

    def orbital_derivatives(self, dets_up, dets_dn, wts, state_weights=None):
        """Orbital gradient and Hessian at kappa = 0 of the state-averaged variational energy
        E(kappa) = E_core + sum h'D + 1/2 sum g'd, h' = U^T h U and (pq|rs)' rotated alike (natorb.rotate_fcidump with C = U),
        U = expm(-kappa), kappa[p,q] = k_pq = -kappa[q,p] (p > q), in the library's orbital numbering (chem only, norb <= 64).  D and d are the
        spin-summed density matrices of every state normalised to ||Psi_k|| = 1 and averaged with state_weights (default equal).
        The determinant list, wts and time_sym handling are those of two_rdm.
        -> dict(fock [p, q] = F_pq, gradient = 2 (F - F^T), hessian [p, q, r, s] = d^2 E / dk_pq dk_rs (extended
        antisymmetrically to p < q, r < s), energy = sum_k w_k E_k)."""
        up = np.ascontiguousarray(dets_up, dtype=np.uint64).reshape(-1, 2)
        dn = np.ascontiguousarray(dets_dn, dtype=np.uint64).reshape(-1, 2)
        w = np.asarray(wts, dtype=np.float64)
        w = np.asfortranarray(w.reshape(-1, 1) if w.ndim == 1 else w)
        if len(dn) != len(up) or w.shape[0] != len(up):
            raise ValueError("orbital_derivatives: dets_up, dets_dn and wts must have the same number of rows")
        norb, ns = self.system.norb, w.shape[1]
        sw = np.full(max(ns, 1), 1.0 / max(ns, 1)) if state_weights is None else np.ascontiguousarray(state_weights, dtype=np.float64).reshape(-1)
        if len(sw) != ns:
            raise ValueError("orbital_derivatives: state_weights holds %d values for %d states" % (len(sw), ns))
        small = norb <= 64   # the library rejects norb > 64
        fock = np.zeros((norb, norb) if small else 1)
        hess = np.zeros((norb,) * 4 if small else 1)
        e = np.zeros(1)
        check(self._L.sqmc_b200_orbital_derivatives(self._h, len(up), _p(up), _p(dn), ns, _p(w), max(w.shape[0], 1), _p(sw), _p(fock),
                                                    _p(hess), _p(e)))
        # (p,q) at p + norb*q and (p,q,r,s) at p + norb*(q + norb*(r + norb*s)): read in C order they come out reversed
        fock = np.ascontiguousarray(fock.T)
        return dict(fock=fock, gradient=2.0 * (fock - fock.T), hessian=np.ascontiguousarray(hess.transpose(3, 2, 1, 0)), energy=float(e[0]))

    def second_order_pt(self, dets_up, dets_dn, wts, var_energy, eps_pt):
        """Deterministic second-order PT with the HCI screened sum (second_order_pt, hci.f90:1100-1182) -> (delta_e_2pt, ndets_connected)."""
        up = np.ascontiguousarray(dets_up, dtype=np.uint64).reshape(-1, 2)
        dn = np.ascontiguousarray(dets_dn, dtype=np.uint64).reshape(-1, 2)
        w = np.ascontiguousarray(wts, dtype=np.float64).reshape(-1)
        if len(dn) != len(up) or len(w) != len(up):
            raise ValueError("second_order_pt: dets_up, dets_dn and wts must have the same length")
        de, nc = C.c_double(), C.c_int64()
        check(self._L.sqmc_b200_pt2(self._h, len(up), _p(up), _p(dn), _p(w), float(var_energy), float(eps_pt), C.byref(de), C.byref(nc)))
        return de.value, nc.value

    def second_order_pt_sample(self, dets_up, dets_dn, sampled_up, sampled_dn, sampled_coeffs, w_over_p, n_mc, var_energy, eps_pt, eps_pt_big):
        """One sample of second_order_pt_alias (hci.f90:1563-1654): the find_doubly_excited call with n_mc / w_over_p / eps_var_pt_big
        and the k loop behind it -> (e_2pt_this_sample, ndets_connected)."""
        up = np.ascontiguousarray(dets_up, dtype=np.uint64).reshape(-1, 2)
        dn = np.ascontiguousarray(dets_dn, dtype=np.uint64).reshape(-1, 2)
        su = np.ascontiguousarray(sampled_up, dtype=np.uint64).reshape(-1, 2)
        sd = np.ascontiguousarray(sampled_dn, dtype=np.uint64).reshape(-1, 2)
        sc = np.ascontiguousarray(sampled_coeffs, dtype=np.float64).reshape(-1)
        sw = np.ascontiguousarray(w_over_p, dtype=np.float64).reshape(-1)
        if len(dn) != len(up) or not (len(su) == len(sd) == len(sc) == len(sw)):
            raise ValueError("second_order_pt_sample: inconsistent array lengths")
        e, nc = C.c_double(), C.c_int64()
        check(self._L.sqmc_b200_pt2_sample(self._h, len(up), _p(up), _p(dn), len(su), _p(su), _p(sd), _p(sc), _p(sw), int(n_mc), float(var_energy),
                                           float(eps_pt), float(eps_pt_big), C.byref(e), C.byref(nc)))
        return e.value, nc.value

    def second_order_pt_alias(self, dets_up, dets_dn, wts, var_energy, eps_pt, eps_pt_big, n_mc, target_error, rannyu_state, max_samples=1000000):
        """second_order_pt_alias (hci.f90:1314-1684) for n_mc > 0: the label-sorted variational wavefunction, the reference's rannyu
        state (4 twelve-bit digits; the advanced state is returned) -> dict(pt_energy, pt_energy_std_dev, n_samples, e_2pt_samples,
        ndets_connected, rannyu_state)."""
        up = np.ascontiguousarray(dets_up, dtype=np.uint64).reshape(-1, 2)
        dn = np.ascontiguousarray(dets_dn, dtype=np.uint64).reshape(-1, 2)
        w = np.ascontiguousarray(wts, dtype=np.float64).reshape(-1)
        if len(dn) != len(up) or len(w) != len(up):
            raise ValueError("second_order_pt_alias: dets_up, dets_dn and wts must have the same length")
        st = np.array(rannyu_state, dtype=np.int32).reshape(4).copy()
        cap = int(min(max_samples, 1000000))
        es = np.zeros(cap)
        pe, sd, ns, nc = C.c_double(), C.c_double(), C.c_int(), C.c_int64()
        check(self._L.sqmc_b200_pt2_alias(self._h, len(up), _p(up), _p(dn), _p(w), float(var_energy), float(eps_pt), float(eps_pt_big), int(n_mc),
                                          float(target_error), _p(st), cap, C.byref(pe), C.byref(sd), C.byref(ns), _p(es), C.byref(nc)))
        return dict(pt_energy=pe.value, pt_energy_std_dev=sd.value, n_samples=ns.value, e_2pt_samples=es[:ns.value].copy(),
                    ndets_connected=nc.value, rannyu_state=st)

    def davidson_sparse_single(self, initial_vector=None, tol=1.0e-10, max_iter=50):
        """davidson_sparse_single (more_tools.f90:3055-3233) on the resident matrix ->
        dict(lowest_eigenvalue, highest_eigenvalue, lowest_eigenvector, ritz, n_iter)."""
        n = self.n
        evec = np.zeros(n)
        eig2 = np.zeros(2)
        ritz = np.zeros(max_iter + 2)
        nit, nlog = C.c_int(), C.c_int()
        v0p = None
        if initial_vector is not None:
            v0 = np.ascontiguousarray(initial_vector, dtype=np.float64).reshape(-1)
            if len(v0) != n:
                raise ValueError("initial_vector must have n entries")
            v0p = _p(v0)
        check(self._L.sqmc_b200_davidson_single(self._h, v0p, _p(evec), _p(eig2), float(tol), int(max_iter), C.byref(nit), _p(ritz), len(ritz),
                                                C.byref(nlog)))
        return dict(lowest_eigenvalue=eig2[0], highest_eigenvalue=eig2[1], lowest_eigenvector=evec, ritz=ritz[:nlog.value].copy(), n_iter=nit.value)
