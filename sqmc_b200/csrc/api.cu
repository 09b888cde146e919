// api.cu -- the C ABI of libsqmc_b200.so (include/sqmc_b200.h): handle management,
// device / NCCL set-up and the host-pointer entry points (H2D / D2H inside the call).
#include <algorithm>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/sqmc_b200.h"
#include "handle.h"

namespace sqmc {
std::string g_last_error;
int64_t g_launch_count = 0;
Global G;
std::vector<sqmc_b200_handle *> g_handles;
void set_error(const char *fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_last_error = buf;
}
static int require_init() {
  if (!G.inited) {
    set_error("sqmc_b200_init has not been called (or failed): no CUDA device, no CPU fallback");
    return 1;
  }
  return 0;
}
}  // namespace sqmc

using namespace sqmc;

namespace sqmc {
// The stream-ordered pool never gives memory back on its own: with a finite release threshold every synchronisation trimmed
// the pool and the next selection / build phase mapped the memory again (0.3-1.5 s stalls at random places of an HCI loop, unmapping
// costs ~40 ms per GB).  Memory is returned explicitly when some allocation fails (devbuf_alloc, big_malloc, grow_ensure).
static const uint64_t kPoolKeepBytes = ~0ull;
static bool g_use_pool = true;
// Host time spent inside allocator / mapping calls is accumulated (g_alloc_stall_ms, sqmc_b200_alloc_stall_ms): on the measurement
// boxes these calls block for 0.01-1.2 s at random, and a build's wall time is only readable next to this number.
// SQMC_ALLOC_TRACE=1 additionally reports every call that blocks the host for more than 10 ms.
double g_alloc_stall_ms = 0.0;
struct AllocTrace {
  const char *what;
  size_t bytes;
  std::chrono::steady_clock::time_point t0;
  static bool on() {
    static int v = -1;
    if (v < 0) { const char *e = getenv("SQMC_ALLOC_TRACE"); v = (e && atoi(e) > 0) ? 1 : 0; }
    return v == 1;
  }
  AllocTrace(const char *w, size_t b) : what(w), bytes(b) { t0 = std::chrono::steady_clock::now(); }
  ~AllocTrace() {
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    g_alloc_stall_ms += ms;
    if (on() && ms > 10.0) fprintf(stderr, "[sqmc alloc] %s of %.3f GB blocked the host for %.1f ms\n", what, bytes / 1e9, ms);
  }
};
int devbuf_alloc(void **p, size_t bytes) {
  AllocTrace tr("devbuf_alloc", bytes);
  cudaError_t e = g_use_pool ? cudaMallocAsync(p, bytes, G.stream) : cudaMalloc(p, bytes);
  if (e != cudaSuccess && g_use_pool) {  // pool exhausted next to a large matrix: give the cache back and retry
    cudaGetLastError();
    cudaStreamSynchronize(G.stream);
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, G.device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
    e = cudaMallocAsync(p, bytes, G.stream);
    if (e != cudaSuccess) {  // still short: the matrices give back the surplus of their growable arrays
      cudaGetLastError();
      matrix_arrays_release_surplus();
      e = cudaMallocAsync(p, bytes, G.stream);
    }
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("device allocation of %lld bytes failed: %s", (long long)bytes, cudaGetErrorString(e));
    *p = nullptr;
    return 1;
  }
  return 0;
}
void devbuf_free(void *p) {
  if (!p) return;
  AllocTrace tr("devbuf_free", 0);
  if (g_use_pool && G.stream) cudaFreeAsync(p, G.stream);
  else cudaFree(p);
}
// cudaMalloc for the long-lived large arrays: when it fails, the temporaries cached by the pool are released first
int big_malloc(void **p, size_t bytes) {
  cudaError_t e = cudaMalloc(p, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    cudaStreamSynchronize(G.stream);
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, G.device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
    e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      matrix_arrays_release_surplus();
      e = cudaMalloc(p, bytes);
    }
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaMalloc of %lld bytes failed: %s", (long long)bytes, cudaGetErrorString(e));
    *p = nullptr;
    return 1;
  }
  return 0;
}
}  // namespace sqmc

extern "C" {

const char *sqmc_b200_last_error(void) { return g_last_error.c_str(); }
int64_t sqmc_b200_launch_count(void) { return g_launch_count; }
double sqmc_b200_alloc_stall_ms(int reset) {
  const double v = sqmc::g_alloc_stall_ms;
  if (reset) sqmc::g_alloc_stall_ms = 0.0;
  return v;
}

int sqmc_b200_get_unique_id(void *id128) {
  ncclUniqueId id;
  ncclResult_t r = ncclGetUniqueId(&id);
  if (r != ncclSuccess) { set_error("ncclGetUniqueId: %s", ncclGetErrorString(r)); return 3; }
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  memcpy(id128, &id, 128);
  return 0;
}

int sqmc_b200_init(int device, int rank, int nranks, const void *id128) {
  if (G.inited) { set_error("sqmc_b200_init: already initialised"); return 1; }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error("sqmc_b200_init: no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(e));
    return 1;
  }
  if (device < 0 || device >= ndev) { set_error("sqmc_b200_init: device %d out of range (%d devices)", device, ndev); return 1; }
  SQ_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SQ_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    set_error("sqmc_b200_init: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    return 1;
  }
  G.device = device;
  G.rank = rank;
  G.nranks = nranks < 1 ? 1 : nranks;
  G.sm_count = prop.multiProcessorCount;
  SQ_CUDA(cudaStreamCreateWithFlags(&G.stream, cudaStreamNonBlocking));
  {
    const char *pe = getenv("SQMC_POOL");
    sqmc::g_use_pool = !(pe && atoi(pe) == 0);
    cudaMemPool_t pool;
    if (sqmc::g_use_pool && cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      uint64_t keep = sqmc::kPoolKeepBytes;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
      // grow the pool once, up front: on the measurement boxes a cudaMallocAsync that needs fresh physical memory blocks the
      // host for 0.01-1.2 s at random (SQMC_ALLOC_TRACE=1 shows it, profiles/r02_alloc_trace.txt), whatever its size; with the
      // memory already in the pool the per-call temporaries of selection / build / Davidson are served without the driver.
      // SQMC_POOL_PREWARM_GB overrides the size (default: 1/12 of the device, at most 16 GB; 0 disables).
      size_t fr = 0, tot = 0;
      cudaMemGetInfo(&fr, &tot);
      const char *pw = getenv("SQMC_POOL_PREWARM_GB");
      size_t warm = pw ? (size_t)(atof(pw) * 1e9) : std::min<size_t>(tot / 12, (size_t)16 << 30);
      if (warm > fr / 2) warm = fr / 2;
      if (warm > 0) {
        void *w = nullptr;
        if (cudaMallocAsync(&w, warm, G.stream) == cudaSuccess) cudaFreeAsync(w, G.stream);
        else cudaGetLastError();
        cudaStreamSynchronize(G.stream);
      }
    } else {
      sqmc::g_use_pool = false;
      cudaGetLastError();
    }
  }
  if (G.nranks > 1) {
    if (!id128) { set_error("sqmc_b200_init: nranks>1 needs an ncclUniqueId"); return 1; }
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclResult_t r = ncclCommInitRank(&G.comm, G.nranks, id, G.rank);
    if (r != ncclSuccess) { set_error("ncclCommInitRank: %s", ncclGetErrorString(r)); return 3; }
  }
  G.inited = true;
  return 0;
}

int sqmc_b200_finalize(void) {
  if (!G.inited) return 0;
  if (G.comm) ncclCommDestroy(G.comm);
  G.comm = nullptr;
  if (G.stream) cudaStreamDestroy(G.stream);
  G.stream = nullptr;
  G.inited = false;
  return 0;
}

// frees a partially constructed handle (and its device tables) when a system_* constructor fails half way
struct HandleGuard {
  sqmc_b200_handle *h;
  ~HandleGuard() { if (h) sqmc_b200_free(h); }
  sqmc_b200_handle *release() { sqmc_b200_handle *q = h; h = nullptr; return q; }
};
static sqmc_b200_handle *new_handle(int model, int norb, int nup, int ndn) {
  sqmc_b200_handle *h = new sqmc_b200_handle();
  memset(&h->T, 0, sizeof(h->T));
  h->T.model = model;
  h->T.norb = norb;
  h->T.nup = nup;
  h->T.ndn = ndn;
  h->T.z = 1;
  h->NW = norb <= 64 ? 1 : 2;
  g_handles.push_back(h);
  return h;
}

int sqmc_b200_system_chem(sqmc_b200_handle **out, int norb, int nup, int ndn, const double *integrals, int64_t nint,
                          const int32_t *combine_2, int time_sym, int z) {
  SQ_CHECK(require_init());
  if (norb < 1 || norb > 127) { set_error("system_chem: norb=%d outside 1..127 (types.f90:44)", norb); return 2; }
  if (nup < ndn) { set_error("system_chem: nup < ndn (chemistry.f90:158)"); return 2; }
  if (time_sym && nup != ndn) { set_error("system_chem: time_sym needs nup == ndn (chemistry.f90:186)"); return 2; }
  if (time_sym && z != 1 && z != -1) { set_error("system_chem: z must be +1 or -1 (chemistry.f90:190)"); return 2; }
  sqmc_b200_handle *h = new_handle(MODEL_CHEM, norb, nup, ndn);
  HandleGuard guard{h};
  int n1 = norb + 1;
  SQ_CUDA(cudaMalloc(&h->d_integrals, nint * sizeof(double)));
  SQ_CUDA(cudaMalloc(&h->d_combine_2, (size_t)n1 * n1 * sizeof(int32_t)));
  SQ_CUDA(cudaMemcpy(h->d_integrals, integrals, nint * sizeof(double), cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(h->d_combine_2, combine_2, (size_t)n1 * n1 * sizeof(int32_t), cudaMemcpyHostToDevice));
  h->T.integrals = h->d_integrals;
  h->T.combine_2 = h->d_combine_2;
  h->T.nint = nint;
  h->T.time_sym = time_sym ? 1 : 0;
  h->T.z = z;
  h->T.sqrt2 = sqrt(2.0);            // chemistry.f90:360-361
  h->T.sqrt2inv = 1.0 / h->T.sqrt2;
  // nuclear_nuclear_energy = integrals(integral_index(norb+1,norb+1,norb+1,norb+1)) (chemistry.f90:398)
  int64_t a = combine_2[(size_t)(n1 - 1) * n1 + (n1 - 1)];
  int64_t idx = (a * (a - 1)) / 2 + a;
  if (idx < 1 || idx > nint) { set_error("system_chem: integrals array shorter than the nuclear-energy index"); return 2; }
  h->T.enuc = integrals[idx - 1];
  *out = guard.release();
  return 0;
}

int sqmc_b200_system_heg(sqmc_b200_handle **out, int norb, int n_dim, const double *k_vectors, double length_cell, int nup,
                         int ndn) {
  SQ_CHECK(require_init());
  if (norb < 1 || norb > 127 || (n_dim != 2 && n_dim != 3)) { set_error("system_heg: bad norb/n_dim"); return 2; }
  sqmc_b200_handle *h = new_handle(MODEL_HEG, norb, nup, ndn);
  HandleGuard guard{h};
  SQ_CUDA(cudaMalloc(&h->d_kvec, (size_t)norb * n_dim * sizeof(double)));
  SQ_CUDA(cudaMemcpy(h->d_kvec, k_vectors, (size_t)norb * n_dim * sizeof(double), cudaMemcpyHostToDevice));
  h->T.k_vectors = h->d_kvec;
  h->T.n_dim = n_dim;
  h->T.length_cell = length_cell;
  *out = guard.release();
  return 0;
}

int sqmc_b200_system_hubbardk(sqmc_b200_handle **out, int l_x, int l_y, const int32_t *k_vectors, const double *k_energies,
                              double ubyn, int nup, int ndn) {
  SQ_CHECK(require_init());
  int ns = l_x * l_y;
  if (ns < 1 || ns > 127) { set_error("system_hubbardk: bad lattice"); return 2; }
  sqmc_b200_handle *h = new_handle(MODEL_HUBBARDK, ns, nup, ndn);
  HandleGuard guard{h};
  SQ_CUDA(cudaMalloc(&h->d_hkvec, (size_t)2 * ns * sizeof(int32_t)));
  SQ_CUDA(cudaMalloc(&h->d_kenergies, (size_t)ns * sizeof(double)));
  SQ_CUDA(cudaMemcpy(h->d_hkvec, k_vectors, (size_t)2 * ns * sizeof(int32_t), cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(h->d_kenergies, k_energies, (size_t)ns * sizeof(double), cudaMemcpyHostToDevice));
  h->T.hk_vectors = h->d_hkvec;
  h->T.k_energies = h->d_kenergies;
  h->T.ubyn = ubyn;
  h->T.l_x = l_x;
  h->T.l_y = l_y;
  *out = guard.release();
  return 0;
}

int sqmc_b200_free(sqmc_b200_handle *h) {
  if (!h) return 0;
  free_matrix(h);
  matrix_arrays_release(h);
  p2p_release(h);
  if (h->d_orbsym) cudaFree(h->d_orbsym);
  if (h->d_scat_counter) cudaFree(h->d_scat_counter);
  for (int k = 0; k < 2; k++) {
    if (h->d_hb_val[k]) cudaFree(h->d_hb_val[k]);
    if (h->d_hb_rs[k]) cudaFree(h->d_hb_rs[k]);
  }
  if (h->d_integrals) cudaFree(h->d_integrals);
  if (h->d_combine_2) cudaFree(h->d_combine_2);
  if (h->d_kvec) cudaFree(h->d_kvec);
  if (h->d_hkvec) cudaFree(h->d_hkvec);
  if (h->d_kenergies) cudaFree(h->d_kenergies);
  g_handles.erase(std::remove(g_handles.begin(), g_handles.end(), h), g_handles.end());
  delete h;
  return 0;
}

int sqmc_b200_set_hf_to_psit(sqmc_b200_handle *h, int flag) {
  if (!h) { set_error("set_hf_to_psit: null handle"); return 2; }
  // honoured by the Hubbard builder only: the chem/heg partial-connection builders ignore it (chemistry.f90:7721,7885)
  h->T.hf_to_psit = (flag && h->T.model == MODEL_HUBBARDK) ? 1 : 0;
  return 0;
}
int sqmc_b200_system_orbital_symmetries(sqmc_b200_handle *h, const int32_t *orbital_symmetries) {
  SQ_CHECK(require_init());
  if (!h) { set_error("orbital_symmetries: null handle"); return 2; }
  if (!h->d_orbsym) SQ_CUDA(cudaMalloc(&h->d_orbsym, h->T.norb * sizeof(int32_t)));
  SQ_CUDA(cudaMemcpy(h->d_orbsym, orbital_symmetries, h->T.norb * sizeof(int32_t), cudaMemcpyHostToDevice));
  return 0;
}
int sqmc_b200_hci_select(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *coeffs, double *min_H_already_done,
                         double eps_var, int64_t *n_new_out) {
  SQ_CHECK(require_init());
  if (!h) { set_error("hci_select: null handle"); return 2; }
  return hci_select(h, n, dets_up, dets_dn, coeffs, min_H_already_done, eps_var, n_new_out);
}
int sqmc_b200_hci_new_dets(sqmc_b200_handle *h, void *new_up, void *new_dn) {
  if (!h) { set_error("hci_new_dets: null handle"); return 2; }
  if (!h->sel_new_up.empty()) {
    memcpy(new_up, h->sel_new_up.data(), h->sel_new_up.size() * sizeof(uint64_t));
    memcpy(new_dn, h->sel_new_dn.data(), h->sel_new_dn.size() * sizeof(uint64_t));
  }
  return 0;
}
int sqmc_b200_build_h(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int64_t ndet_old,
                      int64_t *nnz_upper_out) {
  SQ_CHECK(require_init());
  if (!h) { set_error("build_h: null handle"); return 2; }
  SQ_CHECK(build_h(h, n, dets_up, dets_dn, ndet_old));
  if (nnz_upper_out) *nnz_upper_out = h->nnz_upper;
  return 0;
}
int sqmc_b200_export_upper(sqmc_b200_handle *h, int64_t *counts, int64_t *indices, double *values) {
  SQ_CHECK(require_init());
  if (!h) { set_error("export_upper: null handle"); return 2; }
  return export_upper(h, counts, indices, values);
}
int sqmc_b200_import_upper(sqmc_b200_handle *h, int64_t n, const int64_t *counts, const int64_t *indices, const double *values) {
  SQ_CHECK(require_init());
  if (!h) { set_error("import_upper: null handle"); return 2; }
  return import_upper(h, n, counts, indices, values);
}
int sqmc_b200_nnz(sqmc_b200_handle *h, int64_t *n, int64_t *nnz_upper, int64_t *nnz_full) {
  if (!h) { set_error("nnz: null handle"); return 2; }
  if (n) *n = h->n;
  if (nnz_upper) *nnz_upper = h->nnz_upper;
  if (nnz_full) *nnz_full = h->nnz_full;
  return 0;
}
int sqmc_b200_local_rows(sqmc_b200_handle *h, int64_t *n_local_rows, int64_t *nnz_full_local) {
  if (!h) { set_error("local_rows: null handle"); return 2; }
  if (n_local_rows) *n_local_rows = h->row1 - h->row0;
  if (nnz_full_local) *nnz_full_local = h->nnz_local;
  return 0;
}
int sqmc_b200_diagonal(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, double *diag) {
  SQ_CHECK(require_init());
  if (!h) { set_error("diagonal: null handle"); return 2; }
  return diagonal(h, n, dets_up, dets_dn, diag);
}

// x (caller order, host) -> d_x (internal order, device, full length)
static int upload_vector(sqmc_b200_handle *h, const double *x) {
  cudaStream_t s = G.stream;
  SQ_CUDA(cudaMemcpyAsync(h->d_tmp, x, h->n * sizeof(double), cudaMemcpyHostToDevice, s));
  return permute_gather(h->d_tmp, h->d_perm, h->d_x, h->n, s);
}
// d_y (local rows, internal order) -> y (caller order, host, full length; all ranks get the full vector)
static int download_result(sqmc_b200_handle *h, double *y) {
  cudaStream_t s = G.stream;
  const int64_t nloc = h->row1 - h->row0;
  // reuse d_x as the gather buffer
  if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(h->d_x + h->row0, h->d_y, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
  SQ_CHECK(allgather_rows(h, h->d_x, s));
  SQ_CHECK(permute_scatter(h->d_x, h->d_perm, h->d_tmp, h->n, s));
  SQ_CUDA(cudaMemcpyAsync(y, h->d_tmp, h->n * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

int sqmc_b200_matvec(sqmc_b200_handle *h, const double *x, double *y, int nvec, int64_t ldx) {
  SQ_CHECK(require_init());
  if (!h || !h->d_rowptr) { set_error("matvec: no matrix on this handle"); return 2; }
  if (ldx < h->n) { set_error("matvec: ldx < n"); return 2; }
  int v = 0;
  // pairs of vectors share one pass over the matrix when it is in row-bundle order (two-vector kernel, csrc/bundle.cu)
  if (h->bundle_R && nvec >= 2) {
    cudaStream_t s = G.stream;
    const int64_t n = h->n, nloc = h->row1 - h->row0;
    DevBuf<double> xa, xb, ya, yb;
    SQ_CHECK(xa.alloc(std::max<int64_t>(nloc, 1)));
    SQ_CHECK(xb.alloc(std::max<int64_t>(nloc, 1)));
    SQ_CHECK(ya.alloc(std::max<int64_t>(nloc, 1)));
    SQ_CHECK(yb.alloc(std::max<int64_t>(nloc, 1)));
    for (; v + 1 < nvec; v += 2) {
      SQ_CHECK(upload_vector(h, x + (size_t)v * ldx));   // caller order -> internal order in d_x
      if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(xa.p, h->d_x + h->row0, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
      SQ_CHECK(upload_vector(h, x + (size_t)(v + 1) * ldx));
      if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(xb.p, h->d_x + h->row0, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
      SQ_CHECK(spmv_pair(h, xa.p, xb.p, ya.p, yb.p, s));
      if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(h->d_y, ya.p, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
      SQ_CHECK(download_result(h, y + (size_t)v * ldx));
      if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(h->d_y, yb.p, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
      SQ_CHECK(download_result(h, y + (size_t)(v + 1) * ldx));
    }
    (void)n;
  }
  for (; v < nvec; v++) {
    SQ_CHECK(upload_vector(h, x + (size_t)v * ldx));
    SQ_CHECK(spmv_launch(h, h->d_x, h->d_y, G.stream));
    SQ_CHECK(download_result(h, y + (size_t)v * ldx));
  }
  return 0;
}

int sqmc_b200_projector(sqmc_b200_handle *h, double tau, double e_trial, const double *w, double *deltaw) {
  SQ_CHECK(require_init());
  if (!h || !h->d_rowptr) { set_error("projector: no matrix on this handle"); return 2; }
  cudaStream_t s = G.stream;
  SQ_CHECK(upload_vector(h, w));
  SQ_CHECK(spmv_launch(h, h->d_x, h->d_y, s));                                               // deltaw = Hstored . w  (do_walk.f90:2262)
  SQ_CHECK(projector_epilogue(h->d_y, h->d_x + h->row0, e_trial * tau, h->row1 - h->row0, s));  // += e_trial*tau*w (:2290)
  return download_result(h, deltaw);
}

int sqmc_b200_scale_values(sqmc_b200_handle *h, double ratio) {
  SQ_CHECK(require_init());
  if (!h || !h->d_rowptr) { set_error("scale_values: no matrix on this handle"); return 2; }
  SQ_CHECK(scale_array(h->d_vals, h->nnz_local, ratio, G.stream));
  if (h->d_diag) SQ_CHECK(scale_array(h->d_diag, h->row1 - h->row0, ratio, G.stream));
  SQ_CUDA(cudaStreamSynchronize(G.stream));
  h->scale *= ratio;
  return 0;
}

int sqmc_b200_one_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw,
                      double *rdm) {
  SQ_CHECK(require_init());
  if (!h || !dets_up || !dets_dn || !wts || !rdm) { set_error("one_rdm: null argument"); return 2; }
  return one_rdm(h, n, dets_up, dets_dn, n_states, wts, ldw, rdm);
}

int sqmc_b200_two_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw,
                      double *rdm2) {
  SQ_CHECK(require_init());
  if (!h || !dets_up || !dets_dn || !wts || !rdm2) { set_error("two_rdm: null argument"); return 2; }
  return two_rdm(h, n, dets_up, dets_dn, n_states, wts, ldw, rdm2);
}

int sqmc_b200_orbital_derivatives(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts,
                                  int64_t ldw, const double *state_weights, double *fock, double *hessian, double *energy) {
  SQ_CHECK(require_init());
  if (!h || !dets_up || !dets_dn || !wts || !state_weights || !fock || !hessian || !energy) {
    set_error("orbital_derivatives: null argument");
    return 2;
  }
  return orbital_derivatives(h, n, dets_up, dets_dn, n_states, wts, ldw, state_weights, fock, hessian, energy);
}

int sqmc_b200_pt2(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy, double eps_pt,
                  double *delta_e, int64_t *n_connected) {
  SQ_CHECK(require_init());
  if (!h || !delta_e || !n_connected) { set_error("pt2: null argument"); return 2; }
  return pt2(h, n, dets_up, dets_dn, wts, var_energy, eps_pt, delta_e, n_connected);
}

int sqmc_b200_pt2_sample(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int64_t n_sampled, const void *sampled_up,
                         const void *sampled_dn, const double *sampled_coeffs, const double *w_over_p, int n_mc, double var_energy, double eps_pt,
                         double eps_pt_big, double *e_2pt_this_sample, int64_t *n_connected) {
  SQ_CHECK(require_init());
  if (!h || !dets_up || !dets_dn || !sampled_up || !sampled_dn || !sampled_coeffs || !w_over_p || !e_2pt_this_sample || !n_connected) {
    set_error("pt2_sample: null argument");
    return 2;
  }
  return pt2_sample(h, n, dets_up, dets_dn, n_sampled, sampled_up, sampled_dn, sampled_coeffs, w_over_p, n_mc, var_energy, eps_pt, eps_pt_big,
                    e_2pt_this_sample, n_connected);
}

int sqmc_b200_pt2_alias(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy, double eps_pt,
                        double eps_pt_big, int n_mc, double target_error, int32_t *rannyu_state, int max_samples, double *pt_energy,
                        double *pt_energy_std_dev, int *n_samples, double *e_2pt_samples, int64_t *n_connected) {
  SQ_CHECK(require_init());
  if (!h || !dets_up || !dets_dn || !wts || !rannyu_state || !pt_energy || !pt_energy_std_dev || !n_samples || !n_connected) {
    set_error("pt2_alias: null argument");
    return 2;
  }
  return pt2_alias(h, n, dets_up, dets_dn, wts, var_energy, eps_pt, eps_pt_big, n_mc, target_error, rannyu_state, max_samples, pt_energy,
                   pt_energy_std_dev, n_samples, e_2pt_samples, n_connected);
}

int sqmc_b200_davidson_single(sqmc_b200_handle *h, const double *v0, double *evec, double *eig2, double tol, int max_iter, int *n_iter_out,
                              double *ritz_log, int ritz_log_cap, int *n_ritz_logged) {
  SQ_CHECK(require_init());
  if (!h) { set_error("davidson_single: null handle"); return 2; }
  if (max_iter < 1) { set_error("davidson_single: max_iter must be positive"); return 2; }
  return davidson_single(h, v0, evec, eig2, tol, max_iter, n_iter_out, ritz_log, ritz_log_cap, n_ritz_logged);
}

int sqmc_b200_lanczos(sqmc_b200_handle *h, const double *v0, double *evec, double *eig3, double tol, int max_iter, int *n_iter_out,
                      double *ritz_log, int ritz_log_cap, int *n_ritz_logged) {
  SQ_CHECK(require_init());
  if (!h) { set_error("lanczos: null handle"); return 2; }
  if (max_iter < 1) { set_error("lanczos: max_iter must be positive"); return 2; }
  return lanczos(h, v0, evec, eig3, tol, max_iter, n_iter_out, ritz_log, ritz_log_cap, n_ritz_logged);
}

int sqmc_b200_set_row_bundle(sqmc_b200_handle *h, int rows_per_bundle) {
  SQ_CHECK(require_init());
  if (!h || !h->d_rowptr) { set_error("set_row_bundle: no matrix on this handle"); return 2; }
  if (rows_per_bundle != 0 && rows_per_bundle != 2 && rows_per_bundle != 4) {
    set_error("set_row_bundle: rows_per_bundle must be 0, 2 or 4");
    return 2;
  }
  SQ_CHECK(bundle_decode(h));
  if (rows_per_bundle) SQ_CHECK(bundle_encode_r(h, rows_per_bundle));
  SQ_CUDA(cudaStreamSynchronize(G.stream));
  return 0;
}

int sqmc_b200_davidson(sqmc_b200_handle *h, int n_states, const double *v0, double *evecs, double *evals, double tol,
                       int max_vec_per_state, int *n_matvec_out, double *ritz_log, int ritz_log_cap, int *n_ritz_logged) {
  SQ_CHECK(require_init());
  if (!h) { set_error("davidson: null handle"); return 2; }
  return davidson(h, n_states, v0, evecs, evals, tol, max_vec_per_state, n_matvec_out, ritz_log, ritz_log_cap, n_ritz_logged, false);
}

// ---- the caller's data distribution (owned slices in, owned slices out)
int sqmc_b200_set_ownership(sqmc_b200_handle *h, const int32_t *owner_of_row, int64_t *n_owned_out) {
  SQ_CHECK(require_init());
  if (!h || !owner_of_row) { set_error("set_ownership: null argument"); return 2; }
  return set_ownership(h, owner_of_row, n_owned_out);
}
int sqmc_b200_matvec_local(sqmc_b200_handle *h, const double *x_local, double *y_local, int nvec, int64_t ld_local) {
  SQ_CHECK(require_init());
  if (!h || !h->d_rowptr) { set_error("matvec_local: no matrix on this handle"); return 2; }
  if (!h->own_set) { set_error("matvec_local: call sqmc_b200_set_ownership first"); return 2; }
  if (ld_local < h->my_n) { set_error("matvec_local: ld_local < number of owned determinants"); return 2; }
  for (int v = 0; v < nvec; v++) SQ_CHECK(matvec_local(h, x_local + (size_t)v * ld_local, y_local + (size_t)v * ld_local));
  return 0;
}
int sqmc_b200_projector_local(sqmc_b200_handle *h, double tau, double e_trial, const double *w_local, double *deltaw_local) {
  SQ_CHECK(require_init());
  if (!h || !h->d_rowptr) { set_error("projector_local: no matrix on this handle"); return 2; }
  if (!h->own_set) { set_error("projector_local: call sqmc_b200_set_ownership first"); return 2; }
  return projector_local(h, tau, e_trial, w_local, deltaw_local);
}
int sqmc_b200_davidson_local(sqmc_b200_handle *h, int n_states, const double *v0_local, double *evecs_local, double *evals, double tol,
                             int max_vec_per_state, int *n_matvec_out, double *ritz_log, int ritz_log_cap, int *n_ritz_logged) {
  SQ_CHECK(require_init());
  if (!h) { set_error("davidson_local: null handle"); return 2; }
  return davidson(h, n_states, v0_local, evecs_local, evals, tol, max_vec_per_state, n_matvec_out, ritz_log, ritz_log_cap, n_ritz_logged, true);
}
// page-lock a caller buffer once so that the per-step H2D / D2H of the projector run at PCIe speed
int sqmc_b200_register_host(void *ptr, int64_t bytes) {
  SQ_CHECK(require_init());
  if (!ptr || bytes <= 0) { set_error("register_host: bad arguments"); return 2; }
  cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault);
  if (e == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return 0; }
  if (e != cudaSuccess) { cudaGetLastError(); set_error("register_host: %s", cudaGetErrorString(e)); return 1; }
  return 0;
}
int sqmc_b200_unregister_host(void *ptr) {
  if (!ptr) return 0;
  cudaError_t e = cudaHostUnregister(ptr);
  if (e != cudaSuccess) { cudaGetLastError(); set_error("unregister_host: %s", cudaGetErrorString(e)); return 1; }
  return 0;
}
int sqmc_b200_last_build_incremental(sqmc_b200_handle *h) { return h ? h->last_build_incremental : -1; }
int sqmc_b200_exchange_mode(sqmc_b200_handle *h) {  // 0 single rank, 1 NVLink peer stores, 2 NCCL
  if (!h || G.nranks == 1) return 0;
  return h->p2p.on ? 1 : 2;
}

int sqmc_b200_matvec_dev(sqmc_b200_handle *h, double *x_dev, double *y_dev, void *stream) {
  SQ_CHECK(require_init());
  if (!h || !h->d_rowptr) { set_error("matvec_dev: no matrix on this handle"); return 2; }
  cudaStream_t s = stream ? (cudaStream_t)stream : G.stream;
  return spmv_block(h, x_dev + h->row0, y_dev, s);
}
int sqmc_b200_device_malloc(void **p, int64_t bytes) {
  SQ_CHECK(require_init());
  SQ_CUDA(cudaMalloc(p, (size_t)bytes));
  return 0;
}
int sqmc_b200_device_free(void *p) {
  if (p) cudaFree(p);
  return 0;
}
int sqmc_b200_memcpy_h2d(void *dst, const void *src, int64_t bytes) {
  SQ_CUDA(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, G.stream));
  SQ_CUDA(cudaStreamSynchronize(G.stream));
  return 0;
}
int sqmc_b200_memcpy_d2h(void *dst, const void *src, int64_t bytes) {
  SQ_CUDA(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost, G.stream));
  SQ_CUDA(cudaStreamSynchronize(G.stream));
  return 0;
}
int sqmc_b200_device_sync(void) {
  SQ_CUDA(cudaDeviceSynchronize());
  return 0;
}
int sqmc_b200_get_perm(sqmc_b200_handle *h, int64_t *perm) {
  if (!h || !h->d_perm) { set_error("get_perm: no determinant list"); return 2; }
  std::vector<int32_t> p(h->n);
  SQ_CUDA(cudaMemcpy(p.data(), h->d_perm, h->n * sizeof(int32_t), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < h->n; i++) perm[i] = p[i];
  return 0;
}
int sqmc_b200_get_row(sqmc_b200_handle *h, int64_t caller_row, int64_t cap, int64_t *cols, double *vals, int64_t *len) {
  SQ_CHECK(require_init());
  if (!h || !h->d_rowptr) { set_error("get_row: no matrix on this handle"); return 2; }
  if (caller_row < 1 || caller_row > h->n) { set_error("get_row: row out of range"); return 2; }
  int32_t p = 0;
  SQ_CUDA(cudaMemcpy(&p, h->d_iperm + (caller_row - 1), sizeof(int32_t), cudaMemcpyDeviceToHost));
  if (p < h->row0 || p >= h->row1) { *len = -1; return 0; }  // another rank owns this row
  std::vector<int32_t> c;
  std::vector<double> v;
  int64_t L = 0;
  if (h->bundle_R) {
    SQ_CHECK(bundle_get_row(h, p, c, v));
    L = (int64_t)c.size();
  } else {
    int64_t rp[2];
    SQ_CUDA(cudaMemcpy(rp, h->d_rowptr + (p - h->row0), 2 * sizeof(int64_t), cudaMemcpyDeviceToHost));
    L = rp[1] - rp[0];
    c.resize(L);
    v.resize(L);
    SQ_CUDA(cudaMemcpy(c.data(), h->d_cols + rp[0], L * sizeof(int32_t), cudaMemcpyDeviceToHost));
    SQ_CUDA(cudaMemcpy(v.data(), h->d_vals + rp[0], L * sizeof(double), cudaMemcpyDeviceToHost));
  }
  *len = L;
  if (L > cap) { set_error("get_row: row has %lld entries, capacity %lld", (long long)L, (long long)cap); return 2; }
  // internal columns -> caller columns in one device gather (perm lives on the device)
  std::vector<int32_t> cc(L);
  if (L > 0) {
    DevBuf<int32_t> d_in, d_out;
    SQ_CHECK(d_in.alloc(L));
    SQ_CHECK(d_out.alloc(L));
    SQ_CUDA(cudaMemcpyAsync(d_in.p, c.data(), L * sizeof(int32_t), cudaMemcpyHostToDevice, G.stream));
    SQ_CHECK(gather_i32(h->d_perm, d_in.p, d_out.p, L, G.stream));
    SQ_CUDA(cudaMemcpyAsync(cc.data(), d_out.p, L * sizeof(int32_t), cudaMemcpyDeviceToHost, G.stream));
    SQ_CUDA(cudaStreamSynchronize(G.stream));
  }
  std::vector<std::pair<int64_t, double>> e(L);
  for (int64_t k = 0; k < L; k++) e[k] = {(int64_t)cc[k] + 1, v[k]};
  std::sort(e.begin(), e.end(), [](const std::pair<int64_t, double> &a, const std::pair<int64_t, double> &b) { return a.first < b.first; });
  for (int64_t k = 0; k < L; k++) { cols[k] = e[k].first; vals[k] = e[k].second; }
  return 0;
}
int sqmc_b200_partition_rows(const int64_t *work_prefix, int64_t n, int nranks, int64_t *row_starts) {
  if (n < 0 || nranks < 1) { set_error("partition_rows: bad arguments"); return 2; }
  partition_rows(work_prefix, n, nranks, row_starts);
  return 0;
}
int sqmc_b200_build_times(sqmc_b200_handle *h, double *ms8) {
  if (!h || !ms8) { set_error("build_times: null argument"); return 2; }
  for (int i = 0; i < 8; i++) ms8[i] = h->build_ms[i];
  return 0;
}

}  // extern "C"
