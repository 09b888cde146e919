// davidson.cu -- diagonally preconditioned Davidson with all Krylov vectors resident in HBM.
//
// Replaces davidson_sparse (more_tools.f90:2018-2244) and davidson_sparse_mpi2
// (:2525-2865).  The control flow (circular column index, restart after
// min(n, 50*n_states) vectors, residual/(E-H_ii) preconditioner with the 1e-8
// guard, modified Gram-Schmidt, subspace diagonalisation every n_states vectors,
// stop on max|dE| < tol) follows the reference statement by statement so that the
// printed Ritz values agree; the <= (50 n_states)^2 subspace problem (LAPACK dsyev
// in the reference, :2204) is solved on the host with a cyclic Jacobi sweep.
// Vectors are sharded by rows under nranks>1: dots are completed with a small
// ncclAllReduce, the new basis vector is all-gathered before the SpMV
// (the reference does both with n-long MPI_ALLREDUCEs, :2647,2658).
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "handle.h"

namespace sqmc {

static const int kDotBlocks = 592;  // 148 SMs x 4

// partial[c*gridDim.x + b] = sum over this block's rows of A[c*ld + j] * bvec[j]
__global__ void __launch_bounds__(256) multi_dot_kernel(const double *__restrict__ A, int64_t ld, int k, const double *__restrict__ bvec,
                                                        int64_t n, double *__restrict__ partial) {
  __shared__ double sm[8];
  const int64_t per = (n + gridDim.x - 1) / gridDim.x;
  const int64_t j0 = blockIdx.x * per, j1 = min(n, j0 + per);
  for (int c = 0; c < k; c++) {
    const double *a = A + (int64_t)c * ld;
    double acc = 0.0;
    for (int64_t j = j0 + threadIdx.x; j < j1; j += blockDim.x) acc += a[j] * bvec[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < 8; w++) t += sm[w];
      partial[(int64_t)c * gridDim.x + blockIdx.x] = t;
    }
    __syncthreads();
  }
}
__global__ void reduce_partials_kernel(const double *partial, int nblk, int k, double *out) {
  int c = blockIdx.x;
  if (c >= k) return;
  __shared__ double sm[256];
  double acc = 0.0;
  for (int b = threadIdx.x; b < nblk; b += blockDim.x) acc += partial[(int64_t)c * nblk + b];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[c] = sm[0];
}
// v = (Hw - E w) / (E - diag), guarded (more_tools.f90:2166-2169)
__global__ void resid_precond_kernel(const double *Hw, const double *w, const double *diag, double E, double *v, int64_t n) {
  int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= n) return;
  double r = (Hw[j] - E * w[j]) / (E - diag[j]);
  if (fabs(E - diag[j]) < 1e-8) r = -1.0;
  v[j] = r;
}
// y -= (*s) * x
__global__ void axpy_neg_dev_kernel(double *y, const double *x, const double *s, int64_t n) {
  int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j < n) y[j] = y[j] - (*s) * x[j];
}
// y *= 1/sqrt(*s)
__global__ void normalize_dev_kernel(double *y, const double *s, int64_t n) {
  int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j < n) {
    double ninv = 1.0 / sqrt(*s);
    y[j] = y[j] * ninv;
  }
}
// out[s*ld + j] = sum_k V[k*ld + j] * coef[s*dim + k]
__global__ void combine_kernel(const double *__restrict__ V, int64_t ld, int dim, const double *__restrict__ coef, int ns,
                               double *__restrict__ out, int64_t n) {
  int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= n) return;
  for (int s = 0; s < ns; s++) {
    double acc = 0.0;
    for (int k = 0; k < dim; k++) acc += V[(int64_t)k * ld + j] * coef[s * dim + k];
    out[(int64_t)s * ld + j] = acc;
  }
}
static void jacobi_eigh(int n, std::vector<double> a, std::vector<double> &evals, std::vector<double> &evecs) {
  // cyclic Jacobi, column-major; eigenvalues ascending, eigenvectors in columns
  evecs.assign((size_t)n * n, 0.0);
  for (int i = 0; i < n; i++) evecs[(size_t)i * n + i] = 1.0;
  auto A = [&](int i, int j) -> double & { return a[(size_t)j * n + i]; };
  auto V = [&](int i, int j) -> double & { return evecs[(size_t)j * n + i]; };
  double frob = 0.0;
  for (int p = 0; p < n; p++)
    for (int q = 0; q < n; q++) frob += A(p, q) * A(p, q);
  // stop when the off-diagonal part is below rounding relative to the matrix (an absolute test sweeps until underflow)
  const double stop = std::max(frob * 1e-34, 1e-300);
  for (int sweep = 0; sweep < 100; sweep++) {
    double off = 0.0;
    for (int p = 0; p < n; p++)
      for (int q = p + 1; q < n; q++) off += A(p, q) * A(p, q);
    if (off <= stop) break;
    for (int p = 0; p < n; p++)
      for (int q = p + 1; q < n; q++) {
        double apq = A(p, q);
        if (fabs(apq) < 1e-300) continue;
        double theta = (A(q, q) - A(p, p)) / (2.0 * apq);
        double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < n; k++) {
          double akp = A(k, p), akq = A(k, q);
          A(k, p) = c * akp - s * akq;
          A(k, q) = s * akp + c * akq;
        }
        for (int k = 0; k < n; k++) {
          double apk = A(p, k), aqk = A(q, k);
          A(p, k) = c * apk - s * aqk;
          A(q, k) = s * apk + c * aqk;
        }
        for (int k = 0; k < n; k++) {
          double vkp = V(k, p), vkq = V(k, q);
          V(k, p) = c * vkp - s * vkq;
          V(k, q) = s * vkp + c * vkq;
        }
      }
  }
  std::vector<int> order(n);
  for (int i = 0; i < n; i++) order[i] = i;
  std::sort(order.begin(), order.end(), [&](int x, int y) { return A(x, x) < A(y, y); });
  evals.resize(n);
  std::vector<double> v2((size_t)n * n);
  for (int j = 0; j < n; j++) {
    evals[j] = A(order[j], order[j]);
    for (int i = 0; i < n; i++) v2[(size_t)j * n + i] = V(i, order[j]);
  }
  evecs.swap(v2);
}

__global__ void set_unit_kernel(double *v, const int32_t *iperm, int32_t caller_row, int64_t row0, int64_t row1) {
  const int32_t p = iperm[caller_row];
  if (p >= row0 && p < row1) v[p - row0] = 1.0;
}
// H(1,1) of a one-determinant space: the rank that owns the row holds it (more_tools.f90:2235-2238)
static int single_element(sqmc_b200_handle *h, double *out) {
  cudaStream_t s = G.stream;
  DevBuf<double> t;
  SQ_CHECK(t.alloc(1));
  if (h->row1 - h->row0 > 0) SQ_CUDA(cudaMemcpyAsync(t.p, h->d_vals, sizeof(double), cudaMemcpyDeviceToDevice, s));
  else SQ_CUDA(cudaMemsetAsync(t.p, 0, sizeof(double), s));
  if (G.nranks > 1) {
    ncclResult_t r = ncclAllReduce(t.p, t.p, 1, ncclDouble, ncclSum, G.comm, s);
    if (r != ncclSuccess) { set_error("davidson: ncclAllReduce failed: %s", ncclGetErrorString(r)); return 3; }
  }
  SQ_CUDA(cudaMemcpyAsync(out, t.p, sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}
// host vector (whole vector in caller order, or the owned slice when local_io) -> this rank's row block
static int load_block(sqmc_b200_handle *h, const double *host, bool local_io, double *block, cudaStream_t s) {
  const int64_t n = h->n, nloc = h->row1 - h->row0;
  if (local_io) {
    SQ_CHECK(load_local_vector(h, host, s));
  } else {
    SQ_CUDA(cudaMemcpyAsync(h->d_tmp, host, n * sizeof(double), cudaMemcpyHostToDevice, s));
    SQ_CHECK(permute_gather(h->d_tmp, h->d_perm, h->d_x, n, s));
  }
  if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(block, h->d_x + h->row0, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
  return 0;
}
// this rank's row block -> host (whole vector in caller order on every rank, or the owned slice when local_io)
static int store_block(sqmc_b200_handle *h, const double *block, bool local_io, double *host, cudaStream_t s) {
  const int64_t n = h->n, nloc = h->row1 - h->row0;
  if (local_io) return store_local_vector(h, block, host, s);
  if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(h->d_x + h->row0, block, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
  SQ_CHECK(allgather_rows(h, h->d_x, s));  // the reference publishes final vectors with an n-long allreduce (:2856)
  SQ_CHECK(permute_scatter(h->d_x, h->d_perm, h->d_tmp, n, s));
  SQ_CUDA(cudaMemcpyAsync(host, h->d_tmp, n * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// optional phase timing (SQMC_DAV_PROFILE=1): host clock around synchronised phases, printed to stderr
struct PhaseTimer {
  bool on;
  cudaStream_t s;
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::chrono::steady_clock::time_point t0;
  PhaseTimer(cudaStream_t st) : s(st) {
    const char *e = getenv("SQMC_DAV_PROFILE");
    on = e && atoi(e) > 0;
  }
  void start() {
    if (!on) return;
    cudaStreamSynchronize(s);
    t0 = std::chrono::steady_clock::now();
  }
  void stop(int i) {
    if (!on) return;
    cudaStreamSynchronize(s);
    acc[i] += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  }
};

// pinned host scratch for the few doubles fetched per iteration: allocated once per process (cudaMallocHost per solver call
// costs up to milliseconds and synchronises the device)
static int pinned_scratch(double **out, size_t bytes) {
  static double *buf = nullptr;
  static size_t cap = 0;
  if (bytes > cap) {
    if (buf) cudaFreeHost(buf);
    buf = nullptr;
    cap = std::max<size_t>(bytes, 1 << 16);
    SQ_CUDA(cudaMallocHost(&buf, cap));
  }
  *out = buf;
  return 0;
}

struct Dav {
  sqmc_b200_handle *h;
  cudaStream_t s;
  int64_t n, nloc, ld;
  double *V = nullptr, *HV = nullptr, *W = nullptr, *HW = nullptr, *diag = nullptr, *partial = nullptr, *scal = nullptr, *coef = nullptr;
  double *resid = nullptr;  // n_states residual norms kept on the device until their Krylov columns are fetched
  double *h_scal = nullptr;  // pinned
  int nmv = 0;
  ~Dav() {
    for (double *p : {V, HV, W, HW, diag, partial, scal, coef, resid})
      if (p) devbuf_free(p);  // stream-ordered, back into the pool cache: the next HCI iteration reuses it
    // h_scal is the process-wide pinned scratch (pinned_scratch): not freed here
  }
  unsigned blocks(int64_t cnt) const { return (unsigned)std::max<int64_t>(1, div_up(cnt, 256)); }
  // out_dev[0..k) = A(:,0..k)^T b  (summed over ranks)
  int dots(const double *A, int k, const double *b, double *out_dev) {
    if (nloc > 0) {
      multi_dot_kernel<<<kDotBlocks, 256, 0, s>>>(A, ld, k, b, nloc, partial);
      SQ_LAUNCH_CHECK();
      reduce_partials_kernel<<<k, 256, 0, s>>>(partial, kDotBlocks, k, out_dev);
      SQ_LAUNCH_CHECK();
    } else {
      SQ_CUDA(cudaMemsetAsync(out_dev, 0, k * sizeof(double), s));
    }
    if (G.nranks > 1) {
      ncclResult_t r = ncclAllReduce(out_dev, out_dev, k, ncclDouble, ncclSum, G.comm, s);
      if (r != ncclSuccess) { set_error("davidson: ncclAllReduce failed: %s", ncclGetErrorString(r)); return 3; }
    }
    return 0;
  }
  int fetch(const double *dev, int k, double *host) {
    SQ_CUDA(cudaMemcpyAsync(h_scal, dev, k * sizeof(double), cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < k; i++) host[i] = h_scal[i];
    return 0;
  }
  int axpy_neg(double *y, const double *x, const double *s_dev) {
    if (nloc == 0) return 0;
    axpy_neg_dev_kernel<<<blocks(nloc), 256, 0, s>>>(y, x, s_dev, nloc);
    SQ_LAUNCH_CHECK();
    return 0;
  }
  int normalize(double *y, const double *s_dev) {
    if (nloc == 0) return 0;
    normalize_dev_kernel<<<blocks(nloc), 256, 0, s>>>(y, s_dev, nloc);
    SQ_LAUNCH_CHECK();
    return 0;
  }
  // HVc = H * Vc (Vc is the local block; the other ranks' blocks are gathered first)
  int apply_h(const double *Vc, double *HVc) {
    SQ_CHECK(spmv_block(h, Vc, HVc, s));
    nmv++;
    return 0;
  }
  // the same for a list of basis columns: pairs share one pass over the matrix (two-vector kernel, csrc/bundle.cu)
  int apply_h_block(const std::vector<int> &cols_) {
    size_t k = 0;
    for (; k + 1 < cols_.size(); k += 2) {
      SQ_CHECK(spmv_pair(h, V + (int64_t)cols_[k] * ld, V + (int64_t)cols_[k + 1] * ld, HV + (int64_t)cols_[k] * ld, HV + (int64_t)cols_[k + 1] * ld, s));
      nmv += 2;
    }
    if (k < cols_.size()) SQ_CHECK(apply_h(V + (int64_t)cols_[k] * ld, HV + (int64_t)cols_[k] * ld));
    return 0;
  }
};

int davidson(sqmc_b200_handle *h, int n_states, const double *v0, double *evecs, double *evals, double tol, int max_vec,
             int *n_matvec_out, double *ritz_log, int ritz_log_cap, int *n_ritz_logged, bool local_io) {
  if (!h->d_rowptr) { set_error("davidson: no matrix on this handle"); return 2; }
  const int64_t n = h->n;
  if (n_states < 1 || n_states > n) { set_error("davidson: bad n_states"); return 2; }
  if (local_io && !h->own_set) { set_error("davidson_local: call sqmc_b200_set_ownership first"); return 2; }
  if (max_vec <= 0) max_vec = 50;
  const int64_t host_ld = local_io ? h->my_n : n;  // leading dimension of v0 / evecs
  if (n == 1) {  // more_tools.f90:2235-2238
    double d = 0;
    SQ_CHECK(single_element(h, &d));
    evals[0] = d;
    if (!local_io || h->my_n > 0) evecs[0] = 1.0;
    if (n_matvec_out) *n_matvec_out = 0;
    if (n_ritz_logged) *n_ritz_logged = 0;
    return 0;
  }
  int nlogged = 0;
  auto log_ritz = [&](const double *e) {
    if (ritz_log && nlogged < ritz_log_cap)
      for (int s = 0; s < n_states; s++) ritz_log[(size_t)nlogged * n_states + s] = e[s];
    nlogged++;
  };
  Dav D;
  D.h = h;
  D.s = G.stream;
  PhaseTimer PT(G.stream);
  PT.start();
  D.n = n;
  D.nloc = h->row1 - h->row0;
  D.ld = (std::max<int64_t>(D.nloc, 1) + 63) / 64 * 64;  // columns start on 512-byte boundaries (texture-path gathers)
  const int64_t nloc = D.nloc, ld = D.ld;
  cudaStream_t s = D.s;
  int iterations = (int)std::min<int64_t>(n, max_vec);
  const int m = n_states * iterations;
  SQ_CHECK(devbuf_alloc((void **)&D.V, (size_t)ld * m * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.HV, (size_t)ld * m * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.W, (size_t)ld * n_states * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.HW, (size_t)ld * n_states * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.diag, (size_t)ld * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.partial, (size_t)kDotBlocks * (m + 2) * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.scal, (size_t)(m + 8) * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.coef, (size_t)m * n_states * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.resid, (size_t)n_states * sizeof(double)));
  SQ_CHECK(pinned_scratch(&D.h_scal, (size_t)(m + 8) * sizeof(double)));
  SQ_CUDA(cudaMemsetAsync(D.V, 0, (size_t)ld * m * sizeof(double), s));
  auto Vc = [&](int c) { return D.V + (int64_t)c * ld; };
  auto HVc = [&](int c) { return D.HV + (int64_t)c * ld; };

  // ---- initial vectors (more_tools.f90:2067-2089)
  if (v0) {
    for (int i = 0; i < n_states; i++) {
      // caller order -> internal order, local block
      SQ_CHECK(load_block(h, v0 + (size_t)i * host_ld, local_io, Vc(i), s));
      SQ_CHECK(D.dots(Vc(i), 1, Vc(i), D.scal));
      SQ_CHECK(D.normalize(Vc(i), D.scal));
      if (i > 0) {
        for (int j = 0; j < i; j++) {
          SQ_CHECK(D.dots(Vc(i), 1, Vc(j), D.scal));
          SQ_CHECK(D.axpy_neg(Vc(i), Vc(j), D.scal));
        }
        SQ_CHECK(D.dots(Vc(i), 1, Vc(i), D.scal));
        SQ_CHECK(D.normalize(Vc(i), D.scal));
      }
    }
  } else {
    // unit vectors on the first n_states CALLER rows (v(i,i)=1); V is zeroed above
    for (int i = 0; i < n_states; i++) {
      set_unit_kernel<<<1, 1, 0, s>>>(Vc(i), h->d_iperm, i, h->row0, h->row1);
      SQ_LAUNCH_CHECK();
    }
  }

  PT.stop(0);  // allocation + initial vectors
  std::vector<double> lowest(n_states, 0.0), prev(n_states, 1e300), residual_norm(n_states, 1.0);
  std::vector<double> h_krylov((size_t)m * m, 0.0), col(m + 8);
  auto HK = [&](int i, int j) -> double & { return h_krylov[(size_t)j * m + i]; };

  SQ_CHECK(extract_diag(h, D.diag, s));
  {
    std::vector<int> first(n_states);
    for (int i = 0; i < n_states; i++) first[i] = i;
    SQ_CHECK(D.apply_h_block(first));
  }
  for (int j = 0; j < n_states; j++) {
    SQ_CHECK(D.dots(D.V, n_states, HVc(j), D.scal));
    SQ_CHECK(D.fetch(D.scal, n_states, col.data()));
    for (int i = 0; i <= j; i++) { HK(i, j) = col[i]; HK(j, i) = col[i]; }
  }
  for (int i = 0; i < n_states; i++) lowest[i] = HK(i, i);
  log_ritz(lowest.data());
  SQ_CUDA(cudaMemcpyAsync(D.W, D.V, (size_t)ld * n_states * sizeof(double), cudaMemcpyDeviceToDevice, s));
  SQ_CUDA(cudaMemcpyAsync(D.HW, D.HV, (size_t)ld * n_states * sizeof(double), cudaMemcpyDeviceToDevice, s));

  const int64_t niter = std::min<int64_t>(n, (int64_t)n_states * iterations);
  bool converged = false;
  std::vector<int> pending;  // basis columns of the current block whose H.v is still to be applied
  for (int64_t it = n_states + 1; it <= niter * 10; it++) {
    const int it_circ = (int)((it - 1) % niter) + 1;
    if (it > niter && it_circ == 1) {  // restart with the current Ritz vectors (:2144-2163)
      SQ_CUDA(cudaMemcpyAsync(D.V, D.W, (size_t)ld * n_states * sizeof(double), cudaMemcpyDeviceToDevice, s));
      SQ_CUDA(cudaMemcpyAsync(D.HV, D.HW, (size_t)ld * n_states * sizeof(double), cudaMemcpyDeviceToDevice, s));
      for (int j = 0; j < n_states; j++) {
        SQ_CHECK(D.dots(D.V, n_states, HVc(j), D.scal));
        SQ_CHECK(D.fetch(D.scal, n_states, col.data()));
        for (int i = 0; i <= j; i++) { HK(i, j) = col[i]; HK(j, i) = col[i]; }
      }
      for (int i = 0; i < n_states; i++) lowest[i] = HK(i, i);
      continue;
    }
    const int i = (it_circ - 1) % n_states;
    const int c = it_circ - 1;
    PT.start();
    if (nloc > 0) {
      resid_precond_kernel<<<D.blocks(nloc), 256, 0, s>>>(D.HW + (int64_t)i * ld, D.W + (int64_t)i * ld, D.diag, lowest[i], Vc(c), nloc);
      SQ_LAUNCH_CHECK();
    }
    double *d_resid = D.resid + i;  // kept on the device until this column's Krylov entries are fetched
    SQ_CHECK(D.dots(Vc(c), 1, Vc(c), d_resid));
    for (int k = 0; k < c; k++) {  // modified Gram-Schmidt (:2176-2179)
      SQ_CHECK(D.dots(Vc(c), 1, Vc(k), D.scal + m + 2));
      SQ_CHECK(D.axpy_neg(Vc(c), Vc(k), D.scal + m + 2));
    }
    SQ_CHECK(D.dots(Vc(c), 1, Vc(c), D.scal + m + 2));
    SQ_CHECK(D.normalize(Vc(c), D.scal + m + 2));
    PT.stop(1);  // residual + Gram-Schmidt
    // The new vector of state i+1 does not depend on H times the vector of state i (only on the Ritz pairs of the last
    // subspace diagonalisation and on the basis itself), so the H.v of one block of n_states vectors are applied
    // together -- identical arithmetic per vector, one pass over the matrix per pair of vectors.
    pending.push_back(c);
    if (i != n_states - 1 && it_circ != niter) continue;
    PT.start();
    SQ_CHECK(D.apply_h_block(pending));
    PT.stop(2);  // H.v
    PT.start();
    for (int cc : pending) {
      const int ii = cc % n_states;
      SQ_CHECK(D.dots(D.V, cc + 1, HVc(cc), D.scal));  // Krylov column (:2194-2197)
      SQ_CUDA(cudaMemcpyAsync(D.scal + cc + 1, D.resid + ii, sizeof(double), cudaMemcpyDeviceToDevice, s));
      SQ_CHECK(D.fetch(D.scal, cc + 2, col.data()));
      for (int k = 0; k <= cc; k++) { HK(k, cc) = col[k]; HK(cc, k) = col[k]; }
      residual_norm[ii] = col[cc + 1];
      double rs = 0;
      for (int q = 0; q < n_states; q++) rs += residual_norm[q];
      if (rs < 1.e-12) converged = true;
    }
    pending.clear();
    PT.stop(3);  // Krylov column

    if (it_circ % n_states == 0) {
      const int dim = it_circ;
      PT.start();
      std::vector<double> hsub((size_t)dim * dim), ev, evec;
      for (int a = 0; a < dim; a++)
        for (int b = 0; b < dim; b++) hsub[(size_t)b * dim + a] = HK(a, b);
      jacobi_eigh(dim, hsub, ev, evec);
      for (int q = 0; q < n_states; q++) lowest[q] = ev[q];
      SQ_CUDA(cudaMemcpyAsync(D.coef, evec.data(), (size_t)dim * n_states * sizeof(double), cudaMemcpyHostToDevice, s));
      if (nloc > 0) {
        combine_kernel<<<D.blocks(nloc), 256, 0, s>>>(D.V, ld, dim, D.coef, n_states, D.W, nloc);
        SQ_LAUNCH_CHECK();
        combine_kernel<<<D.blocks(nloc), 256, 0, s>>>(D.HV, ld, dim, D.coef, n_states, D.HW, nloc);
        SQ_LAUNCH_CHECK();
      }
      SQ_CUDA(cudaStreamSynchronize(s));  // evec goes out of scope
      PT.stop(4);  // subspace diagonalisation + Ritz vectors
      double md = 0;
      for (int q = 0; q < n_states; q++) md = std::max(md, fabs(lowest[q] - prev[q]));
      if (md < tol) { converged = true; break; }
      for (int q = 0; q < n_states; q++) prev[q] = lowest[q];
      log_ritz(lowest.data());
      if (converged) break;
    }
  }
  // ---- results: evals + eigenvectors in caller order
  PT.start();
  for (int q = 0; q < n_states; q++) evals[q] = lowest[q];
  for (int q = 0; q < n_states; q++) SQ_CHECK(store_block(h, D.W + (int64_t)q * ld, local_io, evecs + (size_t)q * host_ld, s));
  PT.stop(5);  // eigenvector download
  if (PT.on)
    fprintf(stderr, "[sqmc_b200 davidson] n=%lld matvecs=%d  setup %.1f ms | residual+GS %.1f | H.v %.1f | krylov %.1f | ritz %.1f | download %.1f\n",
            (long long)n, D.nmv, PT.acc[0] * 1e3, PT.acc[1] * 1e3, PT.acc[2] * 1e3, PT.acc[3] * 1e3, PT.acc[4] * 1e3, PT.acc[5] * 1e3);
  if (n_matvec_out) *n_matvec_out = D.nmv;
  if (n_ritz_logged) *n_ritz_logged = nlogged;
  return 0;
}

// y += c * x with a host scalar
__global__ void axpy_host_kernel(double *y, const double *x, double c, int64_t n) {
  int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j < n) y[j] = y[j] + c * x[j];
}
__global__ void scale_copy_kernel(double *dst, const double *src, double c, int64_t n) {
  int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j < n) dst[j] = src[j] * c;
}

// v = (Hw - E w) / (E - diag) with the zero-denominator guard on ONE element only (davidson_sparse_single, :3140-3144)
__global__ void resid_precond_single_kernel(const double *Hw, const double *w, const double *diag, double E, double *v, int64_t n, int64_t guard) {
  int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= n) return;
  double r = (Hw[j] - E * w[j]) / (E - diag[j]);
  if (j == guard && fabs(E - diag[j]) < 1e-8) r = -1.0;
  v[j] = r;
}

// ------------------------------------------------------------------ single-state Davidson
// Statement-by-statement device version of davidson_sparse_single (more_tools.f90:3055-3233; called from
// chemistry.f90:6286-6290): one state, <= min(n, max_iter = 50) vectors, no restart, the preconditioner guard on the first
// (caller) element only, Ritz vector rebuilt from the whole basis every step, stop at |dE| < tol (1e-10).
// eig2 = {lowest eigenvalue, max(largest diagonal element, largest Ritz value)}.
int davidson_single(sqmc_b200_handle *h, const double *v0, double *evec, double *eig2, double tol, int max_iter, int *n_iter_out, double *ritz_log,
                    int ritz_log_cap, int *n_ritz_logged) {
  if (!h->d_rowptr) { set_error("davidson_single: no matrix on this handle"); return 2; }
  const int64_t n = h->n;
  if (n_ritz_logged) *n_ritz_logged = 0;
  if (n_iter_out) *n_iter_out = 0;
  if (n == 1) {  // :3215-3218
    double d = 0;
    SQ_CHECK(single_element(h, &d));
    eig2[0] = eig2[1] = d;
    evec[0] = 0.0;   // the reference returns its unset work vector here
    return 0;
  }
  Dav D;
  D.h = h;
  D.s = G.stream;
  D.n = n;
  D.nloc = h->row1 - h->row0;
  D.ld = (std::max<int64_t>(D.nloc, 1) + 63) / 64 * 64;  // columns start on 512-byte boundaries (texture-path gathers)
  const int64_t nloc = D.nloc, ld = D.ld;
  cudaStream_t s = D.s;
  const int iterations = (int)std::min<int64_t>(n, max_iter);
  SQ_CHECK(devbuf_alloc((void **)&D.V, (size_t)ld * iterations * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.HV, (size_t)ld * iterations * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.W, (size_t)ld * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.HW, (size_t)ld * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.diag, (size_t)ld * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.partial, (size_t)kDotBlocks * (iterations + 2) * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.scal, (size_t)(iterations + 8) * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.coef, (size_t)(iterations + 8) * sizeof(double)));
  SQ_CHECK(pinned_scratch(&D.h_scal, (size_t)(iterations + 8) * sizeof(double)));
  SQ_CUDA(cudaMemsetAsync(D.V, 0, (size_t)ld * iterations * sizeof(double), s));
  auto Vc = [&](int c) { return D.V + (int64_t)c * ld; };
  auto HVc = [&](int c) { return D.HV + (int64_t)c * ld; };
  SQ_CHECK(extract_diag(h, D.diag, s));
  // largest diagonal element (:3109-3114) and the internal position of the first caller row (the guarded element)
  double highest = -1e300;
  int32_t first_internal = 0;
  {
    std::vector<double> hd(std::max<int64_t>(nloc, 1));
    if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(hd.data(), D.diag, nloc * sizeof(double), cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaMemcpyAsync(&first_internal, h->d_iperm, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
    for (int64_t j = 0; j < nloc; j++) highest = std::max(highest, hd[j]);
    if (G.nranks > 1) {
      SQ_CUDA(cudaMemcpyAsync(D.scal, &highest, sizeof(double), cudaMemcpyHostToDevice, s));
      ncclResult_t r = ncclAllReduce(D.scal, D.scal, 1, ncclDouble, ncclMax, G.comm, s);
      if (r != ncclSuccess) { set_error("davidson_single: ncclAllReduce failed: %s", ncclGetErrorString(r)); return 3; }
      SQ_CHECK(D.fetch(D.scal, 1, &highest));
    }
  }
  const int64_t guard = (first_internal >= h->row0 && first_internal < h->row1) ? first_internal - h->row0 : -1;
  // initial vector (:3099-3105)
  {
    std::vector<double> e;
    const double *src = v0;
    if (!v0) { e.assign(n, 0.0); e[0] = 1.0; src = e.data(); }
    SQ_CUDA(cudaMemcpyAsync(h->d_tmp, src, n * sizeof(double), cudaMemcpyHostToDevice, s));
    SQ_CHECK(permute_gather(h->d_tmp, h->d_perm, h->d_x, n, s));
    if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(Vc(0), h->d_x + h->row0, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
    SQ_CUDA(cudaStreamSynchronize(s));
    if (v0) {
      SQ_CHECK(D.dots(Vc(0), 1, Vc(0), D.scal));
      SQ_CHECK(D.normalize(Vc(0), D.scal));
    }
  }
  std::vector<double> hk((size_t)iterations * iterations, 0.0), col(iterations + 8), evals, evecs;
  SQ_CHECK(D.apply_h(Vc(0), HVc(0)));
  SQ_CHECK(D.dots(Vc(0), 1, HVc(0), D.scal));
  double lowest = 0, prev = 0;
  SQ_CHECK(D.fetch(D.scal, 1, &lowest));
  prev = lowest;
  int nlogged = 0;
  if (ritz_log && nlogged < ritz_log_cap) ritz_log[nlogged] = lowest;
  nlogged++;
  if (nloc > 0) {
    SQ_CUDA(cudaMemcpyAsync(D.W, Vc(0), nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
    SQ_CUDA(cudaMemcpyAsync(D.HW, HVc(0), nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
  }
  hk[0] = lowest;
  bool converged = false;
  int it = 2;
  for (; it <= iterations; it++) {
    const int c = it - 1;
    if (nloc > 0) {
      resid_precond_single_kernel<<<D.blocks(nloc), 256, 0, s>>>(D.HW, D.W, D.diag, lowest, Vc(c), nloc, guard);
      SQ_LAUNCH_CHECK();
    }
    SQ_CHECK(D.dots(Vc(c), 1, Vc(c), D.scal + iterations + 1));
    for (int k = 0; k < c; k++) {  // Gram-Schmidt, each coefficient from the partly orthogonalised vector (:3150-3153)
      SQ_CHECK(D.dots(Vc(c), 1, Vc(k), D.scal + iterations + 2));
      SQ_CHECK(D.axpy_neg(Vc(c), Vc(k), D.scal + iterations + 2));
    }
    SQ_CHECK(D.dots(Vc(c), 1, Vc(c), D.scal + iterations + 2));
    SQ_CHECK(D.normalize(Vc(c), D.scal + iterations + 2));
    SQ_CHECK(D.apply_h(Vc(c), HVc(c)));
    SQ_CHECK(D.dots(D.V, it, HVc(c), D.scal));
    SQ_CUDA(cudaMemcpyAsync(D.scal + it, D.scal + iterations + 1, sizeof(double), cudaMemcpyDeviceToDevice, s));
    SQ_CHECK(D.fetch(D.scal, it + 1, col.data()));
    if (col[it] < 1.e-12) converged = true;  // norm of the new direction before orthogonalisation (:3147-3148)
    for (int k = 0; k < it; k++) { hk[(size_t)c * iterations + k] = col[k]; hk[(size_t)k * iterations + c] = col[k]; }
    std::vector<double> sub((size_t)it * it);
    for (int a = 0; a < it; a++)
      for (int b = 0; b < it; b++) sub[(size_t)b * it + a] = hk[(size_t)b * iterations + a];
    jacobi_eigh(it, sub, evals, evecs);
    lowest = evals[0];
    SQ_CUDA(cudaMemcpyAsync(D.coef, evecs.data(), it * sizeof(double), cudaMemcpyHostToDevice, s));
    if (nloc > 0) {
      combine_kernel<<<D.blocks(nloc), 256, 0, s>>>(D.V, ld, it, D.coef, 1, D.W, nloc);
      SQ_LAUNCH_CHECK();
      combine_kernel<<<D.blocks(nloc), 256, 0, s>>>(D.HV, ld, it, D.coef, 1, D.HW, nloc);
      SQ_LAUNCH_CHECK();
    }
    SQ_CUDA(cudaStreamSynchronize(s));  // evecs is reused next step
    highest = std::max(highest, evals[it - 1]);
    if (fabs(lowest - prev) < tol) { converged = true; break; }
    prev = lowest;
    if (ritz_log && nlogged < ritz_log_cap) ritz_log[nlogged] = lowest;
    nlogged++;
    if (converged) break;
  }
  it = std::min(it, iterations);
  if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(h->d_x + h->row0, D.W, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
  SQ_CHECK(allgather_rows(h, h->d_x, s));
  SQ_CHECK(permute_scatter(h->d_x, h->d_perm, h->d_tmp, n, s));
  SQ_CUDA(cudaMemcpyAsync(evec, h->d_tmp, n * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  eig2[0] = lowest;
  eig2[1] = highest;
  if (n_iter_out) *n_iter_out = it;
  if (n_ritz_logged) *n_ritz_logged = std::min(nlogged, ritz_log_cap);
  return 0;
}

// ------------------------------------------------------------------ Lanczos
// Statement-by-statement device version of matrix_lanczos_sparse (more_tools.f90:1742-1883), the eigensolver the k-space
// Hubbard path uses: <= min(n, max_iter = 50) vectors, w = H v - beta v_prev - alpha v, one Gram-Schmidt pass of the new
// vector against all previous ones (coefficients taken from v_{it+1}, :1820-1826), the tridiagonal matrix diagonalised on
// the host every step (cyclic Jacobi for dsyev), stop at |E - E_prev| < tol (1e-10, :1847) or when the new vector
// vanishes (:1816).  eig3 = {lowest, highest, second lowest}; ritz_log receives the "Iteration, Eigenvalue=" values.
int lanczos(sqmc_b200_handle *h, const double *v0, double *evec, double *eig3, double tol, int max_iter, int *n_iter_out, double *ritz_log,
            int ritz_log_cap, int *n_ritz_logged) {
  if (!h->d_rowptr) { set_error("lanczos: no matrix on this handle"); return 2; }
  const int64_t n = h->n;
  if (n_ritz_logged) *n_ritz_logged = 0;
  if (n_iter_out) *n_iter_out = 0;
  if (n == 1) {  // :1874-1876
    double d = 0;
    SQ_CHECK(single_element(h, &d));
    eig3[0] = eig3[1] = eig3[2] = d;
    evec[0] = 1.0;
    return 0;
  }
  Dav D;
  D.h = h;
  D.s = G.stream;
  D.n = n;
  D.nloc = h->row1 - h->row0;
  D.ld = (std::max<int64_t>(D.nloc, 1) + 63) / 64 * 64;  // columns start on 512-byte boundaries (texture-path gathers)
  const int64_t nloc = D.nloc, ld = D.ld;
  cudaStream_t s = D.s;
  const int iterations = (int)std::min<int64_t>(n, max_iter);
  SQ_CHECK(devbuf_alloc((void **)&D.V, (size_t)ld * (iterations + 1) * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.W, (size_t)ld * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.partial, (size_t)kDotBlocks * (iterations + 2) * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.scal, (size_t)(iterations + 8) * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&D.coef, (size_t)(iterations + 8) * sizeof(double)));
  SQ_CHECK(pinned_scratch(&D.h_scal, (size_t)(iterations + 8) * sizeof(double)));
  SQ_CUDA(cudaMemsetAsync(D.V, 0, (size_t)ld * (iterations + 1) * sizeof(double), s));
  auto Vc = [&](int c) { return D.V + (int64_t)c * ld; };
  double *w = D.W;
  // initial vector: normalised input, or the unit vector on the first CALLER row (:1785-1791)
  {
    std::vector<double> e;
    const double *src = v0;
    if (!v0) { e.assign(n, 0.0); e[0] = 1.0; src = e.data(); }
    SQ_CUDA(cudaMemcpyAsync(h->d_tmp, src, n * sizeof(double), cudaMemcpyHostToDevice, s));
    SQ_CHECK(permute_gather(h->d_tmp, h->d_perm, h->d_x, n, s));
    if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(Vc(0), h->d_x + h->row0, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
    SQ_CUDA(cudaStreamSynchronize(s));
    if (v0) {
      SQ_CHECK(D.dots(Vc(0), 1, Vc(0), D.scal));
      SQ_CHECK(D.normalize(Vc(0), D.scal));
    }
  }
  std::vector<double> alphas(iterations + 1, 0.0), betas(iterations + 2, 0.0), evals, evecs;
  double lowest = 0, highest = 0, second = 0, prev = 0, sc[2];
  bool converged = false;
  int it = 1, nlogged = 0;
  for (; it <= iterations; it++) {
    SQ_CHECK(D.apply_h(Vc(it - 1), w));
    if (it > 1 && nloc > 0) {
      axpy_host_kernel<<<D.blocks(nloc), 256, 0, s>>>(w, Vc(it - 2), -betas[it - 1], nloc);
      SQ_LAUNCH_CHECK();
    }
    SQ_CHECK(D.dots(w, 1, Vc(it - 1), D.scal));
    SQ_CHECK(D.fetch(D.scal, 1, sc));
    alphas[it - 1] = sc[0];
    if (nloc > 0) {
      axpy_host_kernel<<<D.blocks(nloc), 256, 0, s>>>(w, Vc(it - 1), -alphas[it - 1], nloc);
      SQ_LAUNCH_CHECK();
    }
    SQ_CHECK(D.dots(w, 1, w, D.scal));
    SQ_CHECK(D.fetch(D.scal, 1, sc));
    if (sc[0] < 1.e-12) converged = true;
    betas[it] = sqrt(sc[0]);
    if (nloc > 0) {
      scale_copy_kernel<<<D.blocks(nloc), 256, 0, s>>>(Vc(it), w, 1.0 / betas[it], nloc);
      SQ_LAUNCH_CHECK();
      SQ_CUDA(cudaMemcpyAsync(w, Vc(it), nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
    }
    SQ_CHECK(D.dots(D.V, it, Vc(it), D.coef));  // all coefficients v_{it+1}.v_i at once, as the reference computes them
    for (int k = 0; k < it; k++) SQ_CHECK(D.axpy_neg(w, Vc(k), D.coef + k));
    if (nloc > 0) SQ_CUDA(cudaMemcpyAsync(Vc(it), w, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
    SQ_CHECK(D.dots(Vc(it), 1, Vc(it), D.scal));
    SQ_CHECK(D.normalize(Vc(it), D.scal));
    std::vector<double> tri((size_t)it * it, 0.0);
    for (int k = 0; k < it; k++) {
      tri[(size_t)k * it + k] = alphas[k];
      if (k < it - 1) { tri[(size_t)(k + 1) * it + k] = betas[k + 1]; tri[(size_t)k * it + k + 1] = betas[k + 1]; }
    }
    jacobi_eigh(it, tri, evals, evecs);
    lowest = evals[0];
    highest = evals[it - 1];
    if (it > 1) second = evals[1];
    if (it > 1 && fabs(lowest - prev) < tol) { converged = true; break; }
    prev = lowest;
    if (ritz_log && nlogged < ritz_log_cap) ritz_log[nlogged] = lowest;
    nlogged++;
    if (converged) break;
  }
  it = std::min(it, iterations);
  // lowest eigenvector = V(:,1:it) * tridiagonal eigenvector 1 (:1868), published in caller order on every rank
  SQ_CUDA(cudaMemcpyAsync(D.coef, evecs.data(), it * sizeof(double), cudaMemcpyHostToDevice, s));
  if (nloc > 0) {
    combine_kernel<<<D.blocks(nloc), 256, 0, s>>>(D.V, ld, it, D.coef, 1, w, nloc);
    SQ_LAUNCH_CHECK();
    SQ_CUDA(cudaMemcpyAsync(h->d_x + h->row0, w, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
  }
  SQ_CHECK(allgather_rows(h, h->d_x, s));
  SQ_CHECK(permute_scatter(h->d_x, h->d_perm, h->d_tmp, n, s));
  SQ_CUDA(cudaMemcpyAsync(evec, h->d_tmp, n * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  eig3[0] = lowest; eig3[1] = highest; eig3[2] = second;
  if (n_iter_out) *n_iter_out = it;
  if (n_ritz_logged) *n_ritz_logged = std::min(nlogged, ritz_log_cap);
  return 0;
}

// ------------------------------------------------------------------ tridiagonal Lanczos (Green's functions)
// For every start vector v0_r: q_0 = v0_r / ||v0_r||, and for j = 0, 1, ...
//   w = H q_j,  alpha_j = q_j . w,  w -= alpha_j q_j + beta_{j-1} q_{j-1},  w -= Q_j (Q_j^T w)  (one classical Gram-Schmidt pass
//   against q_0 .. q_j: full reorthogonalisation),  beta_j = ||w||,  q_{j+1} = w / beta_j,
// until j + 1 = max_steps or beta_j < tol max|alpha| (beta_j = 0 included): the Krylov space is then invariant.
// Runs go in pairs through the two-vector H.v (one pass over the matrix); every other operation of a run reads only its own
// vectors, in the fixed order of the two-stage dot products, so a run's alpha / beta do not depend on its partner.  The
// scalars of the three-term step and of the projection stay on the device; alpha_j and beta_j^2 are fetched once per step
// for the stopping test.  SQMC_DAV_PROFILE=1 prints the H.v / orthogonalisation split to stderr.

// The two update kernels below subtract in place in one pass over w.  axpy_neg_dev_kernel would take one launch and one read
// and write of w per basis column (j + 1 passes at step j), and combine_kernel writes a fresh output rather than updating w;
// the three-term kernel reads beta^2, the value the dot product leaves on the device, so beta never goes through the host.
// w -= alpha q + sqrt(beta2) q_prev (q_prev null: first step)
__global__ void lanczos_three_term_kernel(double *w, const double *q, const double *q_prev, const double *alpha, const double *beta2, int64_t n) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= n) return;
  double v = w[j] - (*alpha) * q[j];
  if (q_prev) v -= sqrt(*beta2) * q_prev[j];
  w[j] = v;
}
// w -= sum_k Q[k*ld + j] c[k], k ascending
__global__ void project_out_columns_kernel(double *w, const double *__restrict__ Q, int64_t ld, int k, const double *__restrict__ c, int64_t n) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= n) return;
  double acc = 0.0;
  for (int i = 0; i < k; i++) acc += Q[(int64_t)i * ld + j] * c[i];
  w[j] -= acc;
}

int lanczos_tridiagonal(sqmc_b200_handle *h, int nvec, const double *v0, int64_t ldv, int max_steps, double tol, double *alpha, double *beta,
                        double *overlaps, int *steps_out) {
  if (G.nranks > 1) { set_error("lanczos_tridiagonal: runs on a single process only (nranks = %d)", G.nranks); return 2; }
  if (!h->d_rowptr) { set_error("lanczos_tridiagonal: no matrix on this handle"); return 2; }
  const int64_t n = h->n;
  if (nvec < 1) { set_error("lanczos_tridiagonal: nvec must be >= 1"); return 2; }
  if (ldv < n) { set_error("lanczos_tridiagonal: ldv (%lld) must be >= n (%lld)", (long long)ldv, (long long)n); return 2; }
  if (max_steps < 1) { set_error("lanczos_tridiagonal: max_steps must be >= 1"); return 2; }
  if (!(tol >= 0.0)) { set_error("lanczos_tridiagonal: tol must be >= 0"); return 2; }
  const int m = (int)std::min<int64_t>(max_steps, n);  // a Krylov space has at most n dimensions
  Dav D;
  D.h = h;
  D.s = G.stream;
  D.n = n;
  D.nloc = n;
  D.ld = (std::max<int64_t>(n, 1) + 63) / 64 * 64;  // columns start on 512-byte boundaries (texture-path gathers)
  const int64_t ld = D.ld;
  cudaStream_t s = D.s;
  const int npair = std::min(nvec, 2);
  // every device buffer of the call: V0 (nvec columns), (m + 1) Lanczos columns and 3m + 8 scalars per run of a pair, the
  // overlaps, the dot partials, and the two interleaved-vector buffers spmv_pair allocates on its first use
  const bool pair_buffers = nvec >= 2 && h->bundle_R && !h->d_y2;
  const size_t need = sizeof(double) * ((size_t)ld * ((size_t)nvec + (size_t)npair * (m + 1)) + (size_t)npair * (3 * m + 8) +
                                        (size_t)m * nvec + (size_t)kDotBlocks * (std::max(m, nvec) + 2) +
                                        (pair_buffers ? (size_t)4 * std::max<int64_t>(n, 1) : 0));
  {
    size_t fr = 0, tot = 0;
    SQ_CUDA(cudaMemGetInfo(&fr, &tot));
    size_t cached = 0;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, G.device) == cudaSuccess) {
      uint64_t res = 0, used = 0;
      if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &res) == cudaSuccess &&
          cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && res > used)
        cached = (size_t)(res - used);
    }
    if (need > fr + cached) {
      set_error("lanczos_tridiagonal: the Krylov basis needs %.2f GB (%d start vectors + %d runs x %d vectors of %lld doubles, with work buffers) but "
                "%.2f GB of device memory is free; lower max_steps",
                need / 1e9, nvec, npair, m + 1, (long long)n, (fr + cached) / 1e9);
      return 2;
    }
  }
  double *V0 = nullptr, *Q[2] = {nullptr, nullptr}, *sc[2] = {nullptr, nullptr}, *ov = nullptr;
  struct Free {
    std::vector<double *> p;
    ~Free() {
      for (double *q : p)
        if (q) devbuf_free(q);
    }
  } fr;
  SQ_CHECK(devbuf_alloc((void **)&V0, (size_t)ld * nvec * sizeof(double)));
  fr.p.push_back(V0);
  for (int r = 0; r < npair; r++) {
    SQ_CHECK(devbuf_alloc((void **)&Q[r], (size_t)ld * (m + 1) * sizeof(double)));
    fr.p.push_back(Q[r]);
    SQ_CHECK(devbuf_alloc((void **)&sc[r], (size_t)(3 * m + 8) * sizeof(double)));  // [alpha_j, beta_j^2] pairs | projection coefficients
    fr.p.push_back(sc[r]);
  }
  SQ_CHECK(devbuf_alloc((void **)&ov, (size_t)m * nvec * sizeof(double)));
  fr.p.push_back(ov);
  SQ_CHECK(devbuf_alloc((void **)&D.partial, (size_t)kDotBlocks * (std::max(m, nvec) + 2) * sizeof(double)));
  SQ_CHECK(pinned_scratch(&D.h_scal, (size_t)((int64_t)m * nvec + 8) * sizeof(double)));
  SQ_CUDA(cudaMemsetAsync(V0, 0, (size_t)ld * nvec * sizeof(double), s));
  std::vector<double> norm2(nvec);
  for (int r = 0; r < nvec; r++) {
    SQ_CHECK(load_block(h, v0 + (int64_t)r * ldv, false, V0 + (int64_t)r * ld, s));
    SQ_CHECK(D.dots(V0 + (int64_t)r * ld, 1, V0 + (int64_t)r * ld, sc[0]));
    SQ_CHECK(D.fetch(sc[0], 1, &norm2[r]));
    if (!(norm2[r] > 0.0)) { set_error("lanczos_tridiagonal: start vector %d has zero norm", r); return 2; }
  }
  for (int r = 0; r < nvec; r++)
    for (int j = 0; j < max_steps; j++) {
      alpha[(int64_t)r * max_steps + j] = 0.0;
      beta[(int64_t)r * max_steps + j] = 0.0;
    }
  PhaseTimer PT(s);
  for (int r0 = 0; r0 < nvec; r0 += 2) {
    const int nr = std::min(2, nvec - r0);
    int steps[2] = {0, 0};
    bool active[2] = {false, false};
    double amax[2] = {0.0, 0.0};
    auto q = [&](int r, int j) { return Q[r] + (int64_t)j * ld; };
    for (int r = 0; r < nr; r++) {
      SQ_CUDA(cudaMemcpyAsync(q(r, 0), V0 + (int64_t)(r0 + r) * ld, n * sizeof(double), cudaMemcpyDeviceToDevice, s));
      SQ_CHECK(D.dots(q(r, 0), 1, q(r, 0), sc[r]));
      SQ_CHECK(D.normalize(q(r, 0), sc[r]));
      active[r] = true;
    }
    for (int j = 0; j < m && (active[0] || active[1]); j++) {
      PT.start();
      if (active[0] && active[1]) {
        SQ_CHECK(spmv_pair(h, q(0, j), q(1, j), q(0, j + 1), q(1, j + 1), s));
      } else {
        const int r = active[0] ? 0 : 1;
        SQ_CHECK(spmv_block(h, q(r, j), q(r, j + 1), s));
      }
      PT.stop(0);
      PT.start();
      for (int r = 0; r < nr; r++) {
        if (!active[r]) continue;
        double *w = q(r, j + 1), *a = sc[r] + 2 * j, *b2 = a + 1, *c = sc[r] + 2 * m + 4;
        SQ_CHECK(D.dots(q(r, j), 1, w, a));
        lanczos_three_term_kernel<<<D.blocks(n), 256, 0, s>>>(w, q(r, j), j > 0 ? q(r, j - 1) : nullptr, a, j > 0 ? a - 1 : nullptr, n);
        SQ_LAUNCH_CHECK();
        SQ_CHECK(D.dots(Q[r], j + 1, w, c));
        project_out_columns_kernel<<<D.blocks(n), 256, 0, s>>>(w, Q[r], ld, j + 1, c, n);
        SQ_LAUNCH_CHECK();
        SQ_CHECK(D.dots(w, 1, w, b2));
        double ab[2];
        SQ_CHECK(D.fetch(a, 2, ab));
        const int64_t o = (int64_t)(r0 + r) * max_steps + j;
        alpha[o] = ab[0];
        beta[o] = sqrt(ab[1]);
        amax[r] = std::max(amax[r], fabs(ab[0]));
        steps[r] = j + 1;
        if (beta[o] < tol * amax[r] || beta[o] == 0.0 || j + 1 == m) active[r] = false;
        else SQ_CHECK(D.normalize(w, b2));
      }
      PT.stop(1);
    }
    // overlaps <v0_k | q_j> of every start vector with this pair's Lanczos vectors
    for (int r = 0; r < nr; r++) {
      for (int j = 0; j < steps[r]; j++) SQ_CHECK(D.dots(V0, nvec, q(r, j), ov + (int64_t)j * nvec));
      SQ_CHECK(D.fetch(ov, steps[r] * nvec, overlaps + (int64_t)(r0 + r) * max_steps * nvec));
      for (int64_t k = (int64_t)steps[r] * nvec; k < (int64_t)max_steps * nvec; k++) overlaps[(int64_t)(r0 + r) * max_steps * nvec + k] = 0.0;
      steps_out[r0 + r] = steps[r];
    }
  }
  if (PT.on)
    fprintf(stderr, "[sqmc_b200 lanczos_tridiagonal] n=%lld runs=%d  H.v %.3f ms | orthogonalisation %.3f ms\n", (long long)n, nvec, PT.acc[0] * 1e3,
            PT.acc[1] * 1e3);
  return 0;
}

}  // namespace sqmc
