// handle.h -- opaque handle behind the C ABI (include/sqmc_b200.h) and the
// process-wide device / communicator state.
#pragma once
#include <nccl.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "elements.cuh"

struct sqmc_b200_handle;
namespace sqmc {

struct Global {
  bool inited = false;
  int device = 0, rank = 0, nranks = 1;
  int sm_count = 148;
  ncclComm_t comm = nullptr;
  cudaStream_t stream = nullptr;  // all library work is issued on this stream unless a stream is passed in
};
extern Global G;
extern std::vector<struct ::sqmc_b200_handle *> g_handles;  // live handles (their growable arrays can give memory back)

// RAII device buffer for temporaries.  Stream-ordered allocation from the device's default memory pool on the library
// stream (the pool keeps up to kPoolKeepBytes cached, sqmc_b200_init): the selection / build / conversion paths allocate
// and free dozens of temporaries per call and cudaMalloc / cudaFree cost milliseconds each next to a ~100 GB matrix.
// SQMC_POOL=0 falls back to cudaMalloc / cudaFree.
int devbuf_alloc(void **p, size_t bytes);
void devbuf_free(void *p);
int big_malloc(void **p, size_t bytes);  // cudaMalloc that first releases the pool's cache when memory is short
template <typename T>
struct DevBuf {
  T *p = nullptr;
  int64_t n = 0;
  int alloc(int64_t count) {
    release();
    n = count;
    if (count <= 0) return 0;
    if (devbuf_alloc((void **)&p, (size_t)count * sizeof(T))) {
      p = nullptr;
      return 1;
    }
    return 0;
  }
  void release() {
    if (p) devbuf_free(p);
    p = nullptr;
    n = 0;
  }
  T *take() {
    T *q = p;
    p = nullptr;
    n = 0;
    return q;
  }
  ~DevBuf() { release(); }
};

// host wall-clock marks of one build (SQMC_BUILD_PROFILE=1 prints them): finds time spent outside kernels
// (allocation of the ~100 GB arrays, host loops, synchronisation) that the CUDA-event phases do not see
struct HostMarks {
  int level;  // 0 off, 1: synchronise + print at every mark, 2: record the host clock without synchronising and print at the end
  const char *tag;
  std::chrono::steady_clock::time_point t0, last;
  std::vector<std::pair<const char *, double>> log;
  explicit HostMarks(const char *env = "SQMC_BUILD_PROFILE", const char *tag_ = "build") : tag(tag_) {
    const char *e = getenv(env);
    level = e ? atoi(e) : 0;
    t0 = last = std::chrono::steady_clock::now();
  }
  void mark(const char *what) {
    if (level <= 0) return;
    if (level == 1) cudaDeviceSynchronize();
    auto t = std::chrono::steady_clock::now();
    if (level == 1) {
      fprintf(stderr, "[sqmc %s] %-28s %9.1f ms  (t = %9.1f ms)\n", tag, what, std::chrono::duration<double, std::milli>(t - last).count(),
              std::chrono::duration<double, std::milli>(t - t0).count());
    } else {
      log.push_back({what, std::chrono::duration<double, std::milli>(t - last).count()});
    }
    last = t;
  }
  ~HostMarks() {
    if (level != 2) return;
    for (auto &e : log) fprintf(stderr, "[sqmc %s host, no sync] %-28s %9.1f ms\n", tag, e.first, e.second);
  }
};

// ---- peer-memory vector exchange (csrc/p2p.cu) ----
static const int kMaxRanks = 16;
struct P2P {
  bool on = false;            // peers' slabs are mapped: exchanges use NVLink stores; otherwise NCCL
  void *slab = nullptr;       // this rank's slab: flags | x[2] (two interleaved vectors each) | xs[2] | y
  void *peer[kMaxRanks] = {nullptr};
  int64_t cap = 0;            // doubles per vector slot
  size_t bytes = 0;
  unsigned long long epoch_x = 0, epoch_y = 0, epoch_bar = 0;
  cudaStream_t last_stream = nullptr;
};

// ---- device array that grows in place (csrc/growbuf.cu: CUDA virtual memory management) ----
struct GrowBuf {
  unsigned long long base = 0;  // device address of the reserved range
  size_t reserved = 0, mapped = 0, chunk = 0;
  std::vector<unsigned long long> handles;  // physical chunks mapped behind [base, base + mapped)
};
int grow_reserve(GrowBuf &b, size_t max_bytes);
int grow_ensure(GrowBuf &b, size_t bytes);
void grow_trim(GrowBuf &b, size_t bytes);
void grow_release(GrowBuf &b);

// arguments of the fused H.v + owner exchange kernel (csrc/bundle.cu)
struct OwnerScatter {
  double *dst[kMaxRanks];               // every rank's result buffer (this rank's own: device memory)
  unsigned long long *flag[kMaxRanks];  // the calling rank's word in every rank's flag array (null entries: single rank)
  unsigned long long *counter;          // local CTA counter
  const int32_t *owner, *pos;           // per local row: owning rank, position inside the owner's slice
  const double *w;                      // projector: deltaw = H.w + c*w (null: plain product)
  double c;
  unsigned long long epoch;
  int nranks;
};

// number of degree bins for the SpMV (sub-warp vector sizes 2,4,8,16,32 + CTA-per-row)
static const int kNumBins = 6;

}  // namespace sqmc

struct sqmc_b200_handle {
  sqmc::ModelTables T;  // device pointers inside
  int NW = 1;
  // owned device tables
  double *d_integrals = nullptr;
  int32_t *d_combine_2 = nullptr;
  double *d_kvec = nullptr;
  int32_t *d_hkvec = nullptr;
  double *d_kenergies = nullptr;

  // ---- determinant list (internal = alpha-major sorted order) ----
  int64_t n = 0;
  uint64_t *d_up = nullptr, *d_dn = nullptr;  // n*NW words each, internal order
  int32_t *d_perm = nullptr;                  // internal row -> caller row (0-based)
  int32_t *d_iperm = nullptr;                 // caller row -> internal row

  // ---- row sharding (contiguous internal row blocks, balanced by nnz) ----
  std::vector<int64_t> row_starts;  // nranks+1
  int64_t row0 = 0, row1 = 0;       // this rank's rows [row0,row1)

  // ---- full symmetric CSR of the local rows, columns in internal numbering ----
  int64_t *d_rowptr = nullptr;  // (row1-row0+1) offsets into cols/vals
  int32_t *d_cols = nullptr;    // = g_cols.base: the two entry arrays keep their address and memory across builds
  double *d_vals = nullptr;     // = g_vals.base
  sqmc::GrowBuf g_cols, g_vals;
  int last_build_incremental = 0;  // 1 when the last build_h extended the previous matrix instead of rebuilding it
  int64_t nnz_local = 0, capacity = 0;
  int64_t nnz_full = 0, nnz_upper = 0;  // global
  double scale = 1.0;                   // product of scale_values() ratios applied to d_vals

  // ---- SpMV degree bins: row lists (local row ids) ----
  int32_t *d_bin_rows = nullptr;  // concatenated lists
  int64_t bin_off[sqmc::kNumBins + 1] = {0};
  bool bins_ready = false;  // built lazily by the first plain-row H.v

  // ---- row-bundle ordering (csrc/bundle.cu; active when bundle_R > 0: d_cols holds column << 4 | 1 << row-in-bundle) ----
  int bundle_R = 0, bundle_cap = 0;
  double *d_diag = nullptr;        // [nloc] diagonal of the local rows (copied out before the entries are re-ordered)

  // ---- peer-memory exchange + the caller's data distribution (sqmc_b200_set_ownership) ----
  sqmc::P2P p2p;
  bool own_set = false;
  std::vector<int64_t> own_count, own_off;  // per rank: determinants owned / offset of its slice in the slice-concatenated order
  int64_t my_n = 0;                         // determinants this rank owns
  int32_t *d_shuf_of_internal = nullptr;    // [n] internal row -> position in the slice-concatenated order
  int32_t *d_dest_rank = nullptr;           // [nloc] owner rank of the local row's determinant
  int32_t *d_dest_pos = nullptr;            // [nloc] its position inside the owner's slice
  int32_t *d_my_internal = nullptr;         // [my_n] internal row of the k-th determinant this rank owns
  struct XTex { const double *ptr; int64_t n; int nv; cudaTextureObject_t tex; };
  std::vector<XTex> xtex;  // linear textures over gathered vectors (texture-path gathers of the H.v kernels)
  unsigned long long *d_scat_counter = nullptr;  // CTA counter of the fused H.v + owner exchange kernel on a single rank
  // ---- work buffers ----
  double *d_x = nullptr;   // n (global length, internal order)
  double *d_y = nullptr;   // local rows
  double *d_tmp = nullptr; // n (caller order staging)
  double *d_x2 = nullptr;  // 2n: two vectors interleaved (global length; NCCL fallback of the two-vector H.v only)
  double *d_xi2 = nullptr; // 2*local rows: this rank's block of two interleaved vectors
  double *d_y2 = nullptr;  // 2*local rows
  // ---- heat-bath selection (select.cu) ----
  int32_t *d_orbsym = nullptr;        // [norb] orbital irreps (chem), set by sqmc_b200_system_orbital_symmetries
  std::vector<uint64_t> sel_new_up, sel_new_dn;  // result of the last hci_select (host, 16 B per det)
  // ---- ladder images (rdm.cu): result of the last sqmc_b200_ladder (host; 16 B per det, coefficients n x lad_norbs column-major)
  std::vector<uint64_t> lad_up, lad_dn;
  std::vector<double> lad_coef;
  int lad_norbs = 0;
  // heat-bath tables of the chem double excitations (norb <= 64): per hole pair (p,q) -- row p*norb+q -- the particle
  // pairs (r,s) packed r | s<<8, sorted by decreasing |H|; [0] same spin (p<q, r<s), [1] opposite spin (p,r up; q,s dn)
  double *d_hb_val[2] = {nullptr, nullptr};
  uint16_t *d_hb_rs[2] = {nullptr, nullptr};
  int hb_norb = 0;
  double build_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // [5] candidates (local) [6] alpha groups [7] beta groups
};

namespace sqmc {
// build.cu
int build_h(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int64_t ndet_old);
int diagonal(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, double *diag);
int export_upper(sqmc_b200_handle *h, int64_t *counts, int64_t *indices, double *values);
int import_upper(sqmc_b200_handle *h, int64_t n, const int64_t *counts, const int64_t *indices, const double *values);
void free_matrix(sqmc_b200_handle *h);
int matrix_arrays_ensure(sqmc_b200_handle *h, int64_t entries);  // (re)map the growable cols / vals arrays
void matrix_arrays_release(sqmc_b200_handle *h);
void matrix_arrays_release_surplus();  // all handles: unmap the part of the entry arrays no matrix uses (out-of-memory path)
void partition_rows(const int64_t *prefix, int64_t n, int nranks, int64_t *starts);
int upload_dets(int NW, int norb, const void *host16, uint64_t *out, int64_t n, cudaStream_t s);
int sort_pairs_index(int NW, int norb, const uint64_t *a, const uint64_t *b, int32_t *idx, int64_t n, cudaStream_t s);
int gather_strings(int NW, const uint64_t *src, const int32_t *idx, uint64_t *out, int64_t n, cudaStream_t s);
// select.cu
int hci_select(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *coeffs, double *min_H, double eps_var,
               int64_t *n_new_out);
int pt2(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy, double eps_pt,
        double *delta_out, int64_t *nconn_out);
int pt2_sample(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int64_t m, const void *s_up, const void *s_dn, const double *s_c,
               const double *s_wop, int n_mc, double var_energy, double eps_pt, double eps_pt_big, double *e_out, int64_t *nconn_out);
int pt2_alias(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy, double eps_pt, double eps_pt_big,
              int n_mc, double target_error, int *rng4, int max_samples, double *pt_out, double *sd_out, int *ns_out, double *e_now, int64_t *nconn_out);
// spmv.cu
int spmv_setup_bins(sqmc_b200_handle *h);
int spmv_launch(sqmc_b200_handle *h, const double *x_dev, double *y_dev, cudaStream_t s);
int permute_gather(const double *src, const int32_t *idx, double *dst, int64_t n, cudaStream_t s);   // dst[i] = src[idx[i]]
int permute_scatter(const double *src, const int32_t *idx, double *dst, int64_t n, cudaStream_t s);  // dst[idx[i]] = src[i]
int gather_i32(const int32_t *src, const int32_t *idx, int32_t *dst, int64_t n, cudaStream_t s);         // dst[i] = src[idx[i]]
int scale_array(double *a, int64_t n, double r, cudaStream_t s);
int projector_epilogue(double *deltaw, const double *w, double c, int64_t n, cudaStream_t s);  // deltaw += c*w
int allgather_rows(sqmc_b200_handle *h, double *x_full, cudaStream_t s);  // in-place allgather of row blocks
int allgather_rows_k(sqmc_b200_handle *h, double *x_full, int k, cudaStream_t s);  // same for k interleaved vectors
// HVa = H Va, HVb = H Vb (local blocks) with ONE pass over the matrix when it is in row-bundle order
int spmv_pair(sqmc_b200_handle *h, const double *Va, const double *Vb, double *HVa, double *HVb, cudaStream_t s);
// whole vector (k interleaved vectors) on this rank from every rank's row block: NVLink peer stores, else NCCL
int gather_vector(sqmc_b200_handle *h, const double *block, int k, cudaStream_t s, const double **full);
// y = H x, x given as this rank's row block (gathered first under nranks > 1)
int spmv_block(sqmc_b200_handle *h, const double *block, double *y_dev, cudaStream_t s);
// p2p.cu
int p2p_setup(sqmc_b200_handle *h, int64_t n);
void p2p_release(sqmc_b200_handle *h);
int p2p_gather(sqmc_b200_handle *h, const double *src, int64_t count, int64_t off, int which, cudaStream_t s, double **full_out);
int p2p_to_owners(sqmc_b200_handle *h, const double *src, const int32_t *owner, const int32_t *pos, int64_t count, cudaStream_t s, double **y_out);
int p2p_barrier(sqmc_b200_handle *h, cudaStream_t s);
// owner exchange done by the producing kernel itself: fills the peer tables / epoch of O (after the barrier that makes the
// peers' result buffers writable), then p2p_owner_wait queues the wait for everybody's rows
int p2p_owner_begin(sqmc_b200_handle *h, OwnerScatter &O, cudaStream_t s);
int p2p_owner_wait(sqmc_b200_handle *h, const OwnerScatter &O, cudaStream_t s, double **y_out);
int p2p_check(sqmc_b200_handle *h, cudaStream_t s);
double *p2p_x(sqmc_b200_handle *h, int r, int b);
// local.cu: the caller's data distribution (owned slices in / out)
int set_ownership(sqmc_b200_handle *h, const int32_t *owner_host, int64_t *n_owned_out);
int load_local_vector(sqmc_b200_handle *h, const double *host_slice, cudaStream_t s);                       // -> whole vector, internal order, in h->d_x
int store_local_vector(sqmc_b200_handle *h, const double *block, double *host_slice, cudaStream_t s);       // this rank's row block -> owners -> host
int matvec_local(sqmc_b200_handle *h, const double *x_local, double *y_local);
int projector_local(sqmc_b200_handle *h, double tau, double e_trial, const double *w_local, double *deltaw_local);
// convert.cu
int export_upper_device(sqmc_b200_handle *h, int64_t *counts, int64_t *indices, double *values);
int import_upper_device(sqmc_b200_handle *h, int64_t n, const int64_t *counts, const int64_t *indices, const double *values);
int extract_diag(sqmc_b200_handle *h, double *diag_dev, cudaStream_t s);  // diagonal of the local rows (spmv.cu)
// bundle.cu
int bundle_encode(sqmc_b200_handle *h);  // plain CSR -> row bundles in place (SQMC_BUNDLE=2|4, default 4), no-op otherwise
int bundle_encode_r(sqmc_b200_handle *h, int R);  // same with an explicit bundle size
int bundle_decode(sqmc_b200_handle *h);  // exact inverse
int bundle_spmv(sqmc_b200_handle *h, const double *x_dev, double *y_dev, cudaStream_t s);
int bundle_spmm2(sqmc_b200_handle *h, const double *x2_dev, double *y2_dev, cudaStream_t s);  // two interleaved vectors
void x_textures_release(sqmc_b200_handle *h);
int bundle_spmv_scatter(sqmc_b200_handle *h, const double *x_dev, const OwnerScatter &O, cudaStream_t s);  // H.v fused with the owner exchange
int bundle_get_row(sqmc_b200_handle *h, int64_t internal_row, std::vector<int32_t> &cols, std::vector<double> &vals);
// davidson.cu
// local_io: v0 / evecs are this rank's owned slices (my_n x n_states, leading dimension my_n) instead of full vectors
int davidson(sqmc_b200_handle *h, int n_states, const double *v0, double *evecs, double *evals, double tol, int max_vec,
             int *n_matvec_out, double *ritz_log, int ritz_log_cap, int *n_ritz_logged, bool local_io);
int davidson_single(sqmc_b200_handle *h, const double *v0, double *evec, double *eig2, double tol, int max_iter, int *n_iter_out, double *ritz_log,
                    int ritz_log_cap, int *n_ritz_logged);
int lanczos(sqmc_b200_handle *h, const double *v0, double *evec, double *eig3, double tol, int max_iter, int *n_iter_out, double *ritz_log,
            int ritz_log_cap, int *n_ritz_logged);
int lanczos_tridiagonal(sqmc_b200_handle *h, int nvec, const double *v0, int64_t ldv, int max_steps, double tol, double *alpha, double *beta,
                        double *overlaps, int *steps_out);
// rdm.cu
int one_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw, double *rdm);
int two_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw, double *rdm2);
int transition_one_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_pairs, const double *bra, const double *ket,
                       int64_t ldw, double *tdm);
int transition_two_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_pairs, const double *bra, const double *ket,
                       int64_t ldw, double *tdm2);
int orbital_derivatives(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw,
                        const double *state_weights, double *fock, double *hessian, double *energy);
int sigma(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *x, int64_t ldx,
          const double *kappa, double *y);
int orbital_gradient_response(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts,
                              const double *dwts, int64_t ldw, const double *state_weights, double *response);
int ladder(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw, int state, int spin,
           int create, int n_orbs, const int32_t *orbs, int64_t *n_out);
int ladder_result(sqmc_b200_handle *h, void *up_out, void *dn_out, double *coeffs, int64_t ldc);
}  // namespace sqmc
