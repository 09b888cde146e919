/*
 * sqmc_b200.h -- C ABI of libsqmc_b200.so, the B200-native (sm_100a) replacement
 * of ONE hot path of QMC-Cornell/sqmc: sparse Hamiltonian construction over a
 * determinant list + the repeated sparse H.v (Davidson matvec / deterministic
 * projector).  Everything else of the reference (driver, input, selection,
 * PT, stochastic walk) stays Fortran and calls in through ISO_C_BINDING
 * (fortran/sqmc_b200_iface.f90; see INTEGRATION.md).
 *
 * Conventions
 *  - all functions return int status, 0 = ok; sqmc_b200_last_error() gives the
 *    message (the reference's error style is `stop`/mpi_stop, mpi_routines.f90:5137;
 *    the Fortran shim maps non-zero to mpi_stop).
 *  - all pointers are HOST pointers owned by the caller unless the name ends in
 *    _dev; the library owns all device memory behind the opaque handle.
 *  - determinants are arrays of 16-byte little-endian integers = Fortran
 *    integer(ik), ik = 16 bytes (types.f90:26); bit k-1 set <=> orbital k occupied.
 *  - row / column indices exchanged with the caller are 1-based int64 (i8b,
 *    types.f90:18), exactly the reference's H_indices / H_nonzero_elements.
 *  - one host thread per process calls in (the reference is single threaded per
 *    MPI rank); one process drives one GPU.
 *  - there is NO CPU fallback: every entry point fails (non-zero) when no
 *    sm_100 device is usable.
 *
 * File:line citations are relative to /root/reference/src.
 */
#ifndef SQMC_B200_H
#define SQMC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sqmc_b200_handle sqmc_b200_handle;

/* ---- process / device / communicator -------------------------------------
 * Replaces cluster_init's MPI_INIT + communicators for this path
 * (mpi_routines.f90:766-915).  nccl_unique_id: 128 opaque bytes (ncclUniqueId)
 * produced by sqmc_b200_get_unique_id on rank 0 and broadcast by the caller
 * (e.g. with MPI_Bcast); ignored when nranks == 1. */
int sqmc_b200_get_unique_id(void *nccl_unique_id_128B);
int sqmc_b200_init(int device, int rank, int nranks, const void *nccl_unique_id_128B);
int sqmc_b200_finalize(void);
const char *sqmc_b200_last_error(void);

/* ---- system set-up (once) -------------------------------------------------
 * chem: module globals integrals / combine_2 / norb,nup,ndn / time_sym,z
 *       (chemistry.f90:24,104,396-398,855-867; nuclear energy is
 *       integrals(integral_index(norb+1,...)), :398).
 *       integrals: nint doubles, 1-based Fortran array passed as is.
 *       combine_2: (norb+1)x(norb+1) int32, column-major. */
int sqmc_b200_system_chem(sqmc_b200_handle **h, int norb, int nup, int ndn, const double *integrals, int64_t nint,
                          const int32_t *combine_2, int time_sym, int z);
/* heg: k_vectors(n_dim,norb) column-major doubles, length_cell (heg.f90:208,643-749) */
int sqmc_b200_system_heg(sqmc_b200_handle **h, int norb, int n_dim, const double *k_vectors, double length_cell, int nup,
                         int ndn);
/* hubbardk: k_vectors(2,nsites) int32 column-major, k_energies(nsites), ubyn=U/nsites
 * (hubbard.f90:2179-2324); l_x,l_y give the momentum period. */
int sqmc_b200_system_hubbardk(sqmc_b200_handle **h, int l_x, int l_y, const int32_t *k_vectors, const double *k_energies,
                              double ubyn, int nup, int ndn);
/* hf_to_psit argument of generate_sparse_ham_hubbardk_upper_triangular (hubbard.f90:9435,9636-9643): when set, the next
 * builds store row 1 as a single zero diagonal entry and no other row links to column 1.  Ignored for chem / heg, whose
 * partial-connection builders ignore the flag too (chemistry.f90:7721). */
int sqmc_b200_set_hf_to_psit(sqmc_b200_handle *h, int flag);
int sqmc_b200_free(sqmc_b200_handle *h);

/* ---- heat-bath determinant selection (SURVEY 8(f) item 1: the step before the H build in every HCI iteration)
 * Replaces get_next_det_list (hci.f90:865-1039): for the current list (n dets, caller order) with coefficients
 * coeffs(i) = max_state |c_i| (hci.f90:369-382) generate every excitation with |H| |c_i| above eps_var
 * (find_important_connected_dets_chem chemistry.f90:6819 / _heg heg.f90:2475), drop the ones already in the list and
 * return the rest sorted by label: the reference appends exactly these after the old dets (hci.f90:945-991).
 * min_H_already_done (n, in/out) follows hci.f90:1014-1016 for the old dets; the caller sets 9e99 for the new ones.
 * chem needs the (reordered) orbital irreps first: orbital_symmetries(1:norb) of chemistry.f90:27. */
int sqmc_b200_system_orbital_symmetries(sqmc_b200_handle *h, const int32_t *orbital_symmetries);
int sqmc_b200_hci_select(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *coeffs,
                         double *min_H_already_done, double eps_var, int64_t *n_new_out);
int sqmc_b200_hci_new_dets(sqmc_b200_handle *h, void *new_up /* n_new x 16 B */, void *new_dn);
/* Deterministic second-order Epstein-Nesbet correction with the HCI screened sum (SURVEY.md 8(f) item 4):
 * replaces second_order_pt (hci.f90:1100-1182) = find_doubly_excited(..., eps_var_pt = eps_pt, e_mix_num)
 * (semistoch.f90:1579-2231) + the sum over the determinants outside the variational space (:1160-1170):
 *   delta_e = sum_a (sum_i H_ai c_i)^2 / (var_energy - H_aa),  |H_ai c_i| above eps_pt by the selection rules.
 * wts: the n variational coefficients of the state; n_connected: distinct determinants generated, variational ones
 * included (the "ndets_connected" the reference prints, e2e_tests/heg/o_det_ref:431).  chem (plain and time-reversal
 * symmetrised determinants) and heg. */
int sqmc_b200_pt2(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy,
                  double eps_pt, double *delta_e, int64_t *n_connected);
/* Stochastic second-order correction, the semistochastic PT of do_pt (hci.f90:4245-4300): replaces second_order_pt_alias
 * (hci.f90:1314-1684).
 * sqmc_b200_pt2_sample = ONE sample, for a caller that keeps the sampling (rannyu, alias tables) on its side: replaces the call
 *   find_doubly_excited(..., ref = the distinct sampled determinants, ref_coeffs, n_mc, w_over_p = counts/probs,
 *   eps_var_pt = eps_pt, eps_var_pt_big = eps_pt_big, term1, term2, term1_big, term2_big) (hci.f90:1563-1566,
 *   semistoch.f90:2044-2060) and the k loop behind it (hci.f90:1616-1632):
 *     e = 1/(n_mc (n_mc-1)) * sum over k outside the variational list (dets_up/dn, n entries, any order) of
 *         (term1(k)^2 + term2(k) - term1_big(k)^2 - term2_big(k)) / (var_energy - H_kk)
 *   = the "E_2pt_now" the reference prints per sample (e2e_tests/heg/o_st_ref:442).  n_connected = ndets_connected of the call.
 * sqmc_b200_pt2_alias = the whole routine: probabilities |c_i| / sum |c|, setup_alias / sample_alias (more_tools.f90:5603-5752),
 *   n_mc draws per sample merged with counts (tools.f90:1574), Welford mean and variance (tools.f90:1761), stop when
 *   sample >= 10 and the variance of the mean < target_error^2 (hci.f90:1670) or after max_samples; the variational list stays
 *   on the device for all samples.  rannyu_state (4 x 12-bit digits, in/out) is the generator state the caller reads with savern
 *   and writes back with setrn (rannyu.f90:11,76), so the reference's random stream continues unchanged: seeded like the
 *   reference's HEG test the call reproduces all 143 samples of e2e_tests/heg/o_st_ref.  dets/wts must be sorted by label as in
 *   the reference (hci.f90:1372-1378); e_2pt_samples (optional, max_samples entries) receives the per-sample values.
 *   n_mc > 0 only (the reference's memory-based choice of n_mc, hci.f90:1570-1612, is host policy and stays with the caller). */
int sqmc_b200_pt2_sample(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int64_t n_sampled, const void *sampled_up,
                         const void *sampled_dn, const double *sampled_coeffs, const double *w_over_p, int n_mc, double var_energy, double eps_pt,
                         double eps_pt_big, double *e_2pt_this_sample, int64_t *n_connected);
int sqmc_b200_pt2_alias(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy, double eps_pt,
                        double eps_pt_big, int n_mc, double target_error, int32_t *rannyu_state, int max_samples, double *pt_energy,
                        double *pt_energy_std_dev, int *n_samples, double *e_2pt_samples, int64_t *n_connected);

/* ---- one-particle density matrix (the step before natural orbitals, hci.f90:3198,3400,3554) ----------------
 * One-particle density matrices of (variational) wavefunctions, spin resolved:
 *   rdm[s][sigma](p,q) = <Psi_s| a+_{p sigma} a_{q sigma} |Psi_s>,   Psi_s = sum_i wts(i,s) |D_i>,   sigma = 0 (up), 1 (dn)
 * p,q = 0..norb-1 index the bits of the determinant words (for chem: the reference's reordered orbital numbering).
 * wts: n x n_states column-major, leading dimension ldw >= n; no normalisation is applied.
 * rdm: n_states * 2 * norb * norb doubles, matrix (s, sigma) at offset (s*2 + sigma)*norb*norb, element (p,q) at p + norb*q.
 * time_sym handles: D_i are the representatives, each standing for (|u,d> + z|d,u>)/sqrt2 (u != d) or |u,u>.
 * The sign of a+_p a_q is permutation_factor's (alpha string first), so sum_pq h_pq gamma_pq is the one-body energy of the
 * library's Hamiltonian.  The result is exactly symmetric and bit-identical across calls and across permutations of the rows.
 * Errors: n <= 0, n_states < 1, ldw < n, a determinant listed twice, on time_sym handles a representative whose partner
 * (d,u) is listed too.  No communication: on a multi-rank handle the call works on this rank's GPU over the list given. */
int sqmc_b200_one_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states,
                      const double *wts, int64_t ldw, double *rdm);

/* ---- two-particle density matrix ------------------------------------------------------------------------------------
 * Spin-resolved two-particle density matrices in chemists' order (they pair with (pq|rs)):
 *   rdm2[s][b](p,q,r,s') = <Psi_s| a+_{p sigma} a+_{r tau} a_{s' tau} a_{q sigma} |Psi_s>,   b = 0 (sigma tau = alpha alpha),
 *   1 (alpha beta), 2 (beta beta); beta alpha is alpha beta with the index pairs swapped and is not stored.
 * 1/2 sum_b' sum (pq|rs') Gamma is the two-body energy, with b' running over aa, ab, ba (= ab) and bb.
 * Arguments, orbital numbering, time_sym handling and errors are those of sqmc_b200_one_rdm; in addition norb must be <= 64.
 * rdm2: n_states * 3 * norb^4 doubles, element (p,q,r,s') of block b, state s at p + norb*(q + norb*(r + norb*(s' + norb*(b + 3*s)))).
 * Signs are those of the library's Hamiltonian (alpha string first), so the energy identity holds with its own integrals.
 * Every element is written from one accumulated representative of its symmetry orbit, so Gamma_{pq,rs} = Gamma_{qp,sr}, and in
 * the same-spin blocks Gamma_{pq,rs} = Gamma_{rs,pq} = -Gamma_{ps,rq} and Gamma = 0 for p = r or q = s, hold bit for bit.  The
 * representatives are summed as 128-bit fixed-point integers, so the result is bit-identical across calls and row permutations. */
int sqmc_b200_two_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states,
                      const double *wts, int64_t ldw, double *rdm2);

/* ---- transition density matrices -----------------------------------------------------------------------------------
 * One- and two-particle transition density matrices between pairs of vectors over one determinant list:
 *   tdm[k][sigma](p,q)        = <bra_k| a+_{p sigma} a_{q sigma} |ket_k>
 *   tdm2[k][b](p,q,r,s')      = <bra_k| a+_{p sigma} a+_{r tau} a_{s' tau} a_{q sigma} |ket_k>,   b = 0 (aa), 1 (ab), 2 (bb)
 * bra, ket: n x n_pairs each, column-major with leading dimension ldw >= n; pair k is (column k of bra, column k of ket).  The
 * vectors are arbitrary (not normalised, not made orthogonal); pass state I as bra and state J as ket for <I| . |J>.
 * The output layouts are those of sqmc_b200_one_rdm / sqmc_b200_two_rdm with "state" read as "pair"; so are the orbital
 * numbering, the phase convention (alpha string first), time_sym handling (both vectors over the representatives, expanded
 * with the same factors), the duplicate and partner checks, the errors (n_pairs in place of n_states), the models covered and
 * "no communication on a multi-rank handle".  The 2-TDM needs norb <= 64, the 1-TDM has no such limit.
 * Bit-for-bit properties: T(ket, bra) is the Hermitian transpose of T(bra, ket) ((p,q) -> (q,p) for the 1-TDM,
 * (p,q,r,s') -> (q,p,s',r) for the 2-TDM); T(c, c) equals sqmc_b200_one_rdm / sqmc_b200_two_rdm of c; the result is identical
 * across calls and across permutations of the rows.  In the same-spin blocks Gamma_{pq,rs} = Gamma_{rs,pq} = -Gamma_{ps,rq} and
 * Gamma = 0 for p = r or q = s still hold exactly; Gamma_{pq,rs} = Gamma_{qp,sr} does not hold for a transition density.
 * With them, <bra|H|ket> = E_core <bra|ket> + sum h tdm + 1/2 sum (pq|rs) tdm2 and <bra|ket> = trace(tdm) / N. */
int sqmc_b200_transition_one_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_pairs,
                                 const double *bra, const double *ket, int64_t ldw, double *tdm);
int sqmc_b200_transition_two_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_pairs,
                                 const double *bra, const double *ket, int64_t ldw, double *tdm2);

/* ---- orbital gradient and Hessian (orbital optimisation) ------------------------------------------------------------
 * Derivatives at kappa = 0 of the state-averaged variational energy E(kappa) = E_core + sum h'D + 1/2 sum g'd under a real orbital
 * rotation kappa = sum_{p>q} k_pq (E_pq - E_qp) (Helgaker, Jorgensen, Olsen, 10.8.1), chem handles only, norb <= 64:
 *   D_pq = sum_k w_k (gamma^a + gamma^b)_pq / ||Psi_k||^2,  d_pqrs = sum_k w_k (G^aa + G^bb + G^ab_pq,rs + G^ab_rs,pq) / ||Psi_k||^2,
 *   with h_pq, g_pqrs = (pq|rs) read from the handle's integral table in the library's orbital numbering.
 * fock:    norb^2 doubles, F_pq = sum_m D_pm h_qm + sum_mnt d_pmnt g_qmnt at p + norb*q; the gradient is 2 (F_pq - F_qp).
 * hessian: norb^4 doubles, E2_pq,rs = (1 - P_pq)(1 - P_rs)[2 D_pr h_qs - (F_pr + F_rp) delta_qs + 2 Y_pqrs],
 *          Y_pqrs = sum_mn [(d_pmrn + d_pmnr) g_qmsn + d_prmn g_qsmn], at p + norb*(q + norb*(r + norb*s)).
 * energy:  1 double, E_core + sum h D + 1/2 sum g d = sum_k w_k E_k.
 * Arguments, orbital numbering, time_sym handling and errors are those of sqmc_b200_two_rdm; in addition the handle must be
 * chem, hold at least two electrons, and state_weights (n_states values) must be >= 0 and sum to 1 within 1e-12.
 * The density matrices and integrals stay on the device; every output is summed in a fixed order, so the result is
 * bit-identical across calls and row permutations. */
int sqmc_b200_orbital_derivatives(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states,
                                  const double *wts, int64_t ldw, const double *state_weights,
                                  double *fock, double *hessian, double *energy);

/* ---- sigma-vector over a determinant list (orbital optimisation) ----------------------------------------------------
 * y = H x (kappa == NULL: the handle's own integrals, core energy included) or y = H^kappa x (kappa != NULL: the Hamiltonian
 * with one-index-transformed integrals h^k = kappa h - h kappa, g^k_pqrs = sum_m (k_pm g_mqrs + k_qm g_pmrs + k_rm g_pqms +
 * k_sm g_pqrm), no core term), i.e. d/dt H(U(t)) at t = 0 for U(t) = expm(-t kappa) with rotate_fcidump's rule.
 * kappa: norb^2 doubles, antisymmetric, kappa_pq at p + norb*q in the library's orbital numbering.  x: n_states columns of
 * leading dimension ldx; y: n x n_states, column-major with leading dimension n, in the caller's row order.
 * No built matrix is needed or used: every pair of the list connected by a single or double excitation is visited, whatever
 * its matrix element.  Arguments, orbital numbering, time_sym handling (x and y over the representatives) and errors are
 * those of sqmc_b200_orbital_derivatives without state weights.  y is summed as 128-bit fixed-point integers, so it is
 * bit-identical across calls and row permutations. */
int sqmc_b200_sigma(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states,
                    const double *x, int64_t ldx, const double *kappa, double *y);

/* ---- orbital-gradient response (orbital optimisation) ---------------------------------------------------------------
 * response (norb^2 doubles, (p,q) at p + norb*q, antisymmetric) = d/dt at t = 0 of the gradient 2 (F - F^T) that
 * sqmc_b200_orbital_derivatives returns for the vectors wts + t dwts (both n_states columns of leading dimension ldw),
 * normalisation term included.  It is 2 (F' - F'^T) with F' built from the symmetrised transition densities of (c_k, dc_k');
 * the O(norb^6) Hessian product is not formed.  Arguments and errors are those of sqmc_b200_orbital_derivatives; the result is
 * bit-identical across calls and row permutations. */
int sqmc_b200_orbital_gradient_response(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states,
                                        const double *wts, const double *dwts, int64_t ldw, const double *state_weights,
                                        double *response);

/* ---- ladder images (single-particle Green's function) --------------------------------------------------------------
 * Images a_{p sigma}|Psi> (create = 0) or a+_{p sigma}|Psi> (create != 0) of state `state` (0-based column of wts, n_states
 * columns of leading dimension ldw) for every p of orbs[0 .. n_orbs) (library orbital numbering), sigma = spin (0 up, 1 dn).
 * Phase convention: alpha string first, each string with ascending creators (that of chem_single, permutation_factor and
 * sqmc_b200_one_rdm): a_{p alpha} carries (-1)^(alpha electrons below p), a_{p beta} (-1)^(N_alpha + beta electrons below p).
 * time_sym handles: the representatives are expanded first (c/sqrt2 on (u,d), z c/sqrt2 on (d,u)); the images are plain
 * determinants of the N-1 / N+1 electron space.  *n_out receives the number of determinants of the union of the images;
 * sqmc_b200_ladder_result then copies that list (16 bytes per determinant, sorted by (up, dn) as unsigned 128-bit labels, no
 * duplicates) and the n_out x n_orbs coefficient matrix (column j = the image of orbs[j], leading dimension ldc >= n_out).
 * Every coefficient is written once, so the result is bit-identical across calls and row permutations.  The model tables
 * are not read: one- and two-word strings of any model work.
 * Errors: n <= 0, n_states < 1, ldw < n, state outside [0, n_states), spin not 0 / 1, an orbital outside [0, norb) or listed
 * twice, annihilation from an empty spin string or creation into a full one, the duplicate / time_sym partner checks of
 * sqmc_b200_one_rdm, nranks > 1. */
int sqmc_b200_ladder(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw,
                     int state, int spin, int create, int n_orbs, const int32_t *orbs, int64_t *n_out);
int sqmc_b200_ladder_result(sqmc_b200_handle *h, void *up_out, void *dn_out, double *coeffs, int64_t ldc);

/* ---- sparse H build --------------------------------------------------------
 * Replaces generate_sparse_ham_chem_upper_triangular (chemistry.f90:7639),
 * its _mpi twin (:8012), generate_sparse_ham_heg_upper_triangular
 * (heg.f90:3553) and generate_sparse_ham_hubbardk_upper_triangular
 * (hubbard.f90:9435).  dets_up/dn: n x 16 B in the CALLER's row order (the
 * global list under MPI; the library shards rows itself).  ndet_old mirrors
 * sparse_ham%ndet (incremental reuse, chemistry.f90:7769-7843): rows
 * 1..ndet_old are promised unchanged since the previous call on this handle.
 * When the previous matrix is still resident and unscaled (one rank, chem without time-reversal symmetry or heg) it is
 * kept and only pairs involving a new determinant are generated and evaluated; otherwise the matrix is rebuilt.
 * Either way the result is identical to a from-scratch build (see DESIGN.md);
 * sqmc_b200_last_build_incremental tells which path the last call took (1 = extended, 0 = rebuilt).
 * nnz_upper_out: stored entries of the reference's upper-triangular format
 * (what its log prints as "# of nonzero elem in H"), summed over ranks. */
int sqmc_b200_build_h(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int64_t ndet_old,
                      int64_t *nnz_upper_out);
/* Fill the reference's arrays (sparse_mat, commons/common_selected_ci.f90:26-31):
 * H_nonzero_elements(n) per-row counts, H_indices(nnz_upper) 1-based int64
 * columns ascending with the diagonal first, H_values(nnz_upper).  Single-rank
 * handles only (under nranks>1 each rank exports its own rows: row_first/row_count
 * from sqmc_b200_local_rows; counts are for those rows). */
int sqmc_b200_export_upper(sqmc_b200_handle *h, int64_t *H_nonzero_elements, int64_t *H_indices, double *H_values);
/* Import an existing reference-format matrix instead of building (dtm_projector
 * read path, do_walk.f90:883-951): n rows, upper triangular, 1-based. */
int sqmc_b200_import_upper(sqmc_b200_handle *h, int64_t n, const int64_t *H_nonzero_elements, const int64_t *H_indices,
                           const double *H_values);
int sqmc_b200_last_build_incremental(sqmc_b200_handle *h);
int sqmc_b200_nnz(sqmc_b200_handle *h, int64_t *n, int64_t *nnz_upper, int64_t *nnz_full);
int sqmc_b200_local_rows(sqmc_b200_handle *h, int64_t *n_local_rows, int64_t *nnz_full_local);
/* One FULL row (both triangles) of the resident matrix in the caller's numbering: 1-based row in,
 * 1-based ascending columns out.  len = -1 when another rank owns the row.  Inspection / test aid
 * (the reference can only do this by scanning its upper-triangular arrays). */
int sqmc_b200_get_row(sqmc_b200_handle *h, int64_t caller_row, int64_t cap, int64_t *cols, double *vals, int64_t *len);
/* diagonal elements H_ii for a det list (hci.f90:664-676 "quick hack" loops) */
int sqmc_b200_diagonal(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, double *diag);

/* ---- sparse H.v -------------------------------------------------------------
 * Replaces fast_sparse_matrix_multiply_upper_triangular (more_tools.f90:3622),
 * _mpi (:3674) and _local_band (:3562).  x, y: nvec vectors of length n in
 * caller row order, leading dimension ldx (column-major, like v(:,i)).
 * Host<->device copies are inside the call. */
int sqmc_b200_matvec(sqmc_b200_handle *h, const double *x, double *y, int nvec, int64_t ldx);
/* Deterministic projector step of walk (do_walk.f90:2255-2325):
 *   deltaw = Hstored.w + e_trial*tau*w      (Hstored = -tau*H after scale_values(-tau),
 *                                            semistoch.f90:657,880)
 * The caller then does walk_wt(imp) += deltaw (:2321-2323). */
int sqmc_b200_projector(sqmc_b200_handle *h, double tau, double e_trial, const double *w, double *deltaw);
/* values *= ratio: the tau rescaling of do_walk.f90:2179,2919 */
int sqmc_b200_scale_values(sqmc_b200_handle *h, double ratio);
/* Storage-order hint for H.v (no reference counterpart; results of every other call are unchanged):
 * rows_per_bundle = 0 keeps plain CSR rows; 2 or 4 re-orders the entries of that many consecutive
 * rows by column in place (csrc/bundle.cu) so that the gathers of x coalesce.  The environment variable
 * SQMC_BUNDLE sets the default applied after every build / import. */
int sqmc_b200_set_row_bundle(sqmc_b200_handle *h, int rows_per_bundle);

/* ---- Davidson ------------------------------------------------------------------
 * Replaces davidson_sparse (more_tools.f90:2018) / davidson_sparse_mpi2 (:2525):
 * diagonal preconditioner with the 1e-8 guard, <= max_vec_per_state (50) Krylov
 * vectors per state then restart, stop when max|dE| < tol (1e-10, :73,2213).
 * v0: n x n_states column-major initial vectors (NULL => unit vectors on the
 * first n_states rows, :2085-2088).  evecs: n x n_states, evals: n_states.
 * ritz_log (may be NULL): receives up to ritz_log_cap*n_states doubles, the
 * values the reference prints as "Iteration, Eigenvalues=" (:2130,2219). */
int sqmc_b200_davidson(sqmc_b200_handle *h, int n_states, const double *v0, double *evecs, double *evals, double tol,
                       int max_vec_per_state, int *n_matvec_out, double *ritz_log, int ritz_log_cap, int *n_ritz_logged);

/* Replaces davidson_sparse_single (more_tools.f90:3055-3233; call sites chemistry.f90:6286,6290): one state, <= max_iter (50)
 * vectors, no restart, the zero-denominator guard on the first element only (:3143).  v0: n-vector or NULL (unit vector
 * on the first row).  eig2: lowest eigenvalue, and max(largest diagonal element, largest Ritz value) (the optional
 * highest_eigenvalue of the reference).  ritz_log: the printed "Iteration, Eigenvalue=" values. */
int sqmc_b200_davidson_single(sqmc_b200_handle *h, const double *v0, double *evec, double *eig2, double tol, int max_iter,
                              int *n_iter_out, double *ritz_log, int ritz_log_cap, int *n_ritz_logged);

/* ---- the caller's data distribution under MPI ----------------------------------------
 * The reference deals determinants to MPI ranks by hash (get_det_owner, mpi_routines.f90:419-445; do_walk.f90:1760-1807)
 * and every rank passes / receives only ITS slice of a vector, in ascending caller index:
 *   walk:      fast_sparse_matrix_multiply_local_band(..., vector = walk_wt(my_locations_of_imp_dets(1:my_nimp)), answer = deltaw)
 *              + mpi_redscatt_real_dparray(deltaw(1:n_imp), imp_core_mask)         (do_walk.f90:2259-2260, mpi_routines.f90:1592)
 *   Davidson:  davidson_sparse_mpi2 on local_det_map%ndets-long vectors             (more_tools.f90:2525, 2842-2861)
 * set_ownership: owner_of_row(1:n) = rank (0-based) owning each determinant of the list last passed to build_h /
 *   import_upper (every rank passes the same map; the library keeps its own row sharding and moves data between the two
 *   distributions over NVLink).  n_owned_out = my_nimp.  Must be repeated after every build_h.
 * matvec_local / projector_local: x_local, y_local = the owned slices (n_owned entries per vector, leading dimension
 *   ld_local); only those bytes cross PCIe.  Collective: every rank calls with its own slice.
 * davidson_local: v0_local / evecs_local are n_owned x n_states, leading dimension n_owned.
 * With one rank the slice is the whole vector.  register_host page-locks a caller buffer once (the projector runs every
 * Monte Carlo step on the same arrays). */
int sqmc_b200_set_ownership(sqmc_b200_handle *h, const int32_t *owner_of_row, int64_t *n_owned_out);
int sqmc_b200_matvec_local(sqmc_b200_handle *h, const double *x_local, double *y_local, int nvec, int64_t ld_local);
int sqmc_b200_projector_local(sqmc_b200_handle *h, double tau, double e_trial, const double *w_local, double *deltaw_local);
int sqmc_b200_davidson_local(sqmc_b200_handle *h, int n_states, const double *v0_local, double *evecs_local, double *evals, double tol,
                             int max_vec_per_state, int *n_matvec_out, double *ritz_log, int ritz_log_cap, int *n_ritz_logged);
int sqmc_b200_register_host(void *ptr, int64_t bytes);
int sqmc_b200_unregister_host(void *ptr);
/* how vectors travel between GPUs on this handle: 0 = single rank, 1 = NVLink peer-memory stores, 2 = NCCL (fallback) */
int sqmc_b200_exchange_mode(sqmc_b200_handle *h);

/* ---- Lanczos -------------------------------------------------------------------
 * Replaces matrix_lanczos_sparse (more_tools.f90:1742-1883), the eigensolver of the
 * k-space Hubbard path: <= min(n, max_iter = 50) vectors, full Gram-Schmidt pass per
 * step, stop when |dE| < tol (1e-10, :73,1847).  v0: n-vector or NULL (unit vector on
 * the first row, :1788-1790).  evec: n.  eig3: lowest, highest and second-lowest
 * eigenvalue of the tridiagonal matrix (the optional outputs of the reference).
 * ritz_log (may be NULL): the values printed as "Iteration, Eigenvalue=" (:1852). */
int sqmc_b200_lanczos(sqmc_b200_handle *h, const double *v0, double *evec, double *eig3, double tol, int max_iter,
                      int *n_iter_out, double *ritz_log, int ritz_log_cap, int *n_ritz_logged);

/* ---- tridiagonal Lanczos (single-particle Green's function) ---------------------------------------------------------
 * One Lanczos run on the resident matrix per start vector r (v0: nvec columns of leading dimension ldv >= n, caller row
 * order): q_0 = v0_r / ||v0_r||, w = H q_j - alpha_j q_j - beta_{j-1} q_{j-1}, then one classical Gram-Schmidt pass of w
 * against q_0 .. q_j (full reorthogonalisation), beta_j = ||w||, q_{j+1} = w / beta_j.  A run stops after max_steps steps (at
 * most n) or when beta_j < tol * max|alpha| (the Krylov space is invariant).
 * alpha, beta: nvec x max_steps (run r at r * max_steps); entries past the run's steps are 0.  beta[j] couples q_j and q_{j+1};
 * the last one is the norm of the final residual.  overlaps: nvec x max_steps x nvec, <v0_k | q_j> of run r at
 * (r * max_steps + j) * nvec + k (v0_k as given, not normalised).  steps_out: nvec steps taken.
 * Start vectors go through the two-vector H.v in pairs; a run's alpha / beta are bit-identical whether it runs alone or in a
 * pair, and across calls.  Errors: no matrix, nvec < 1, ldv < n, max_steps < 1, tol < 0, a zero start vector, a basis that
 * does not fit in device memory, nranks > 1. */
int sqmc_b200_lanczos_tridiagonal(sqmc_b200_handle *h, int nvec, const double *v0, int64_t ldv, int max_steps, double tol, double *alpha,
                                  double *beta, double *overlaps, int *steps_out);

/* ---- device-resident entry points (used by bench.py for the HBM-resident leg)
 * x_dev/y_dev are device pointers in the library's INTERNAL row order (length n for x,
 * n_local_rows for y).  Under nranks>1 only this rank's row block of x_dev is read: the call first
 * gathers every rank's block into the library's exchange buffer over NVLink (what Davidson does with
 * every new basis vector; the reference: zero-padded MPI_ALLREDUCE, more_tools.f90:2647), then
 * multiplies; x_dev itself is not written.  stream is a cudaStream_t (NULL = the library's own stream). */
int sqmc_b200_matvec_dev(sqmc_b200_handle *h, double *x_dev, double *y_dev, void *stream);
/* average device time (ms) of the last sqmc_b200_matvec_dev launches is measured by the caller with events */
int sqmc_b200_device_malloc(void **p, int64_t bytes);
int sqmc_b200_device_free(void *p);
int sqmc_b200_memcpy_h2d(void *dst_dev, const void *src, int64_t bytes);
int sqmc_b200_memcpy_d2h(void *dst, const void *src_dev, int64_t bytes);
int sqmc_b200_device_sync(void);
/* permutation between caller order and internal order: internal row p holds caller row perm[p] (0-based) */
int sqmc_b200_get_perm(sqmc_b200_handle *h, int64_t *perm);
/* statistics of the last build: ms (device events) [0] sort/prep [1] count [2] fill+sort [3] eval+compact [4] total;
 * [5] candidate pairs generated on this rank [6] unique alpha strings [7] unique beta strings */
int sqmc_b200_build_times(sqmc_b200_handle *h, double *stats8);
/* Row sharding rule (pure host code, usable without a GPU): contiguous row blocks balanced by a
 * work measure.  work_prefix: n+1 exclusive prefix sums; row_starts: nranks+1 outputs.  This is what
 * build_h uses to shard rows of H over ranks (the reference deals dets out by hash ownership,
 * mpi_routines.f90:419-445). */
int sqmc_b200_partition_rows(const int64_t *work_prefix, int64_t n, int nranks, int64_t *row_starts);
/* number of kernels launched by the library since init (for gpu_launches accounting) */
int64_t sqmc_b200_launch_count(void);
/* Host milliseconds this process has spent inside device allocator / memory-mapping calls since start (or since the last call with
 * reset != 0).  On virtualised GPU hosts these driver calls block for 0.01-1.2 s at random; the bench prints the number next to every
 * build so that its wall time can be read (profiles/r02_alloc_trace.txt). */
double sqmc_b200_alloc_stall_ms(int reset);

#ifdef __cplusplus
}
#endif
#endif
