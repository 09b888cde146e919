// rdm.cu -- one-particle density matrices of variational wavefunctions (sqmc_b200_one_rdm).
//
//   rdm[s][sigma](p,q) = <Psi_s| a+_{p sigma} a_{q sigma} |Psi_s>,   Psi_s = sum_i wts(i,s) |D_i>
//
// The list is sorted twice: by (up, dn) and by (dn, up).  In the first view a beta single excitation keeps the alpha
// string, so its partner lies inside the determinant's alpha group, a contiguous range of the view; in the second view the
// same holds for alpha singles and the beta group.  One kernel serves both views with the roles of the two strings swapped:
// for every determinant it adds c^2 to the diagonal of the occupied orbitals of the "minor" string and looks up every single
// excitation q -> p with p > q of the minor string inside the group.  Each unordered pair of determinants is met once, and its
// value sign * c_i * c_j goes to (p,q) and (q,p), so gamma is exactly symmetric.  The sign is permutation_factor's (the one
// chem_single uses), which makes sum_pq h_pq gamma_pq the one-body energy of the library's own Hamiltonian; with the alpha
// string first, neither spin picks up a sign from the other string.
//
// Determinism: warp w walks the fixed contiguous range [w*chunk, (w+1)*chunk) of a view (chunk depends on n only), one
// determinant at a time.  Within one determinant every accumulator slot is touched by at most one lane, so the warp's private
// accumulators need no atomics; the partial matrices of all warps are then summed in warp order by a fixed tree.  The sorted
// views do not depend on the caller's row order, so neither does the result.
//
// Time-reversal symmetrised lists are first expanded to plain determinants on the device: a representative (u,d), u != d,
// becomes c/sqrt2 on (u,d) and z c/sqrt2 on (d,u); (u,u) keeps c (the norm factors of chem_hamiltonian_time_sym).
#include <thrust/iterator/counting_iterator.h>

#include <cub/cub.cuh>

#include "handle.h"

namespace sqmc {

static const int kRdmThreads = 256;               // 8 warps per block
static const int kRdmMaxWarps = 2048;             // per view: both views stay resident in one wave on a B200 (56 registers, 4 blocks / SM)
static const size_t kRdmSharedMax = 160 * 1024;   // larger accumulator sets stay in global memory (still warp-private)

// position of the k-th (0-based) set bit of b; k < popc(b)
template <int NW>
__device__ __forceinline__ int nth_set_bit(const Bits<NW> &b, int k) {
  int base = 0;
  uint64_t w = b.w[0];
  if constexpr (NW == 2) {
    const int c0 = __popcll(b.w[0]);
    if (k >= c0) {
      k -= c0;
      w = b.w[1];
      base = 64;
    }
  }
#pragma unroll
  for (int sh = 32; sh > 0; sh >>= 1) {
    const uint64_t lo = w & ((1ull << sh) - 1ull);
    const int c = __popcll(lo);
    if (k >= c) {
      k -= c;
      w >>= sh;
      base += sh;
    } else {
      w = lo;
    }
  }
  return base;
}

// [begin, end) of the run of strings equal to m around position i of the sorted array a (galloping, then bisection)
template <int NW>
__device__ __forceinline__ int64_t run_end(const uint64_t *a, int64_t i, int64_t n, const Bits<NW> &m) {
  int64_t lo = i, step = 1;
  while (lo + step < n && b_eq(b_load<NW>(a, lo + step), m)) {
    lo += step;
    step <<= 1;
  }
  int64_t hi = min(lo + step, n);
  while (hi - lo > 1) {
    const int64_t mid = lo + (hi - lo) / 2;
    if (b_eq(b_load<NW>(a, mid), m)) lo = mid;
    else hi = mid;
  }
  return hi;
}
template <int NW>
__device__ __forceinline__ int64_t run_begin(const uint64_t *a, int64_t i, const Bits<NW> &m) {
  int64_t hi = i, step = 1;
  while (hi - step >= 0 && b_eq(b_load<NW>(a, hi - step), m)) {
    hi -= step;
    step <<= 1;
  }
  int64_t lo = max(hi - step, (int64_t)-1);
  while (hi - lo > 1) {
    const int64_t mid = lo + (hi - lo) / 2;
    if (b_eq(b_load<NW>(a, mid), m)) hi = mid;
    else lo = mid;
  }
  return hi;
}

struct RdmView {
  const uint64_t *major, *minor;  // n*NW words each, sorted by (major, minor)
  const double *c;                // c[i*S + s], same order
  double *part;                   // [nwarps][S][tri] per-warp partial sums of the minor spin's matrix
};

// slot of (p,q), p >= q, in a packed lower triangle
__device__ __forceinline__ int tri_slot(int p, int q) { return p * (p + 1) / 2 + q; }

template <int NW>
__global__ void one_rdm_kernel(RdmView v0, RdmView v1, int64_t n, int norb, int S, int tri, int64_t chunk, int nwarps, int shared_acc) {
  extern __shared__ double sacc[];
  // field by field: selecting the whole struct by a run-time index would copy it to local memory
  const bool y = blockIdx.y != 0;
  const uint64_t *major = y ? v1.major : v0.major, *minor = y ? v1.minor : v0.minor;
  const double *coef = y ? v1.c : v0.c;
  double *part = y ? v1.part : v0.part;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warp = blockIdx.x * (kRdmThreads / 32) + wib;
  if (warp >= nwarps) return;
  const int64_t per = (int64_t)S * tri;
  double *acc = shared_acc ? sacc + wib * per : part + warp * per;
  for (int64_t k = lane; k < per; k += 32) acc[k] = 0.0;
  __syncwarp();
  const int64_t i0 = min(n, warp * chunk), i1 = min(n, i0 + chunk);
  const Bits<NW> all = b_maskr<NW>(norb);
  int64_t g0 = i0, g1 = i0;  // group of the current major string: [g0, g1)
  for (int64_t i = i0; i < i1; i++) {
    if (i >= g1) {
      const Bits<NW> ma = b_load<NW>(major, i);
      g0 = (i == i0) ? run_begin<NW>(major, i, ma) : i;
      g1 = run_end<NW>(major, i, n, ma);
    }
    const Bits<NW> mi = b_load<NW>(minor, i);
    const double *ci = coef + i * S;
    for (int p = lane; p < norb; p += 32) {
      if (b_test(mi, p)) {
        const int t = tri_slot(p, p);
        for (int s = 0; s < S; s++) acc[s * tri + t] += ci[s] * ci[s];
      }
    }
    const Bits<NW> emp = b_andnot(all, mi);
    const int nocc = b_popc(mi), nemp = norb - nocc;
    const int npair = nocc * nemp;
    for (int k = lane; k < npair; k += 32) {
      const int q = nth_set_bit(mi, k / nemp), p = nth_set_bit(emp, k % nemp);
      if (p < q) continue;  // the pair is met from the other determinant
      Bits<NW> mj = mi;
      b_clear(mj, q);
      b_set(mj, p);
      int64_t lo = g0, hi = g1;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (b_lt(b_load<NW>(minor, mid), mj)) lo = mid + 1;
        else hi = mid;
      }
      if (lo >= g1 || !b_eq(b_load<NW>(minor, lo), mj)) continue;
      const double sg = (double)permutation_factor(mi, mj);
      const double *cj = coef + lo * S;
      const int t = tri_slot(p, q);
      for (int s = 0; s < S; s++) acc[s * tri + t] += (sg * ci[s]) * cj[s];
    }
    __syncwarp();
  }
  if (shared_acc) {
    double *dst = part + warp * per;
    for (int64_t k = lane; k < per; k += 32) dst[k] = acc[k];
  }
}

// one block per (slot, view): thread k sums warps k, k + 256, ... in order, then a fixed tree; writes (p,q) and (q,p)
__global__ void __launch_bounds__(kRdmThreads) one_rdm_reduce_kernel(const double *part0, const double *part1, int nwarps, int S, int tri, int norb,
                                                                       double *out) {
  __shared__ double red[kRdmThreads];
  const int64_t slot = blockIdx.x, per = (int64_t)S * tri;
  const double *part = blockIdx.y ? part1 : part0;
  double a = 0.0;
  for (int w = threadIdx.x; w < nwarps; w += kRdmThreads) a += part[w * per + slot];
  red[threadIdx.x] = a;
  __syncthreads();
  for (int h = kRdmThreads / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  const int s = (int)(slot / tri), t = (int)(slot % tri);
  int p = 0;
  while ((p + 1) * (p + 2) / 2 <= t) p++;
  const int q = t - p * (p + 1) / 2;
  const int sigma = blockIdx.y ? 0 : 1;  // view 0 is (up, dn) order: its minor string is beta
  double *m = out + ((int64_t)s * 2 + sigma) * norb * norb;
  m[p + (int64_t)norb * q] = red[0];
  m[q + (int64_t)norb * p] = red[0];
}

template <int NW>
__global__ void off_diagonal_flag_kernel(const uint64_t *u, const uint64_t *d, int32_t *flag, int64_t n) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) flag[i] = b_eq(b_load<NW>(u, i), b_load<NW>(d, i)) ? 0 : 1;
}

// time_sym -> plain determinants: entries [0, n) the representatives, [n, n + m) the partners (d,u) of the m reps sel[] with u != d
template <int NW>
__global__ void ts_expand_kernel(const uint64_t *u, const uint64_t *d, const double *w, int64_t n, const int32_t *sel, int64_t m, int S,
                                 double r, double zr, uint64_t *eu, uint64_t *ed, double *ew) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t n2 = n + m;
  if (t >= n2) return;
  if (t < n) {
    const Bits<NW> U = b_load<NW>(u, t), D = b_load<NW>(d, t);
    b_store(eu, t, U);
    b_store(ed, t, D);
    const double f = b_eq(U, D) ? 1.0 : r;
    for (int s = 0; s < S; s++) ew[s * n2 + t] = w[s * n + t] * f;
  } else {
    const int64_t i = sel[t - n];
    b_store(eu, t, b_load<NW>(d, i));
    b_store(ed, t, b_load<NW>(u, i));
    for (int s = 0; s < S; s++) ew[s * n2 + t] = w[s * n + i] * zr;
  }
}

__global__ void gather_coeffs_kernel(const double *w, int64_t n, const int32_t *idx, int S, double *c) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n * S) return;
  const int64_t k = t / S;
  const int s = (int)(t % S);
  c[t] = w[s * n + idx[k]];
}

// bit 0: two equal entries that come from the same side of the expansion (a duplicated determinant); bit 1: a representative
// equal to another one's time-reversed partner
template <int NW>
__global__ void duplicate_kernel(const uint64_t *a, const uint64_t *b, const int32_t *idx, int64_t n, int64_t n_rep, int *flag) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x + 1;
  if (k >= n) return;
  if (b_eq(b_load<NW>(a, k), b_load<NW>(a, k - 1)) && b_eq(b_load<NW>(b, k), b_load<NW>(b, k - 1)))
    atomicOr(flag, ((idx[k] < n_rep) == (idx[k - 1] < n_rep)) ? 1 : 2);
}

// one sorted view: (major, minor) strings and the interleaved coefficients in (major, minor) order
template <int NW>
static int make_view(int norb, const uint64_t *major, const uint64_t *minor, const double *w, int64_t n, int S, DevBuf<int32_t> &idx,
                     DevBuf<uint64_t> &sma, DevBuf<uint64_t> &smi, DevBuf<double> &c, cudaStream_t s) {
  SQ_CHECK(idx.alloc(n));
  SQ_CHECK(sort_pairs_index(NW, norb, major, minor, idx.p, n, s));
  SQ_CHECK(sma.alloc(n * NW));
  SQ_CHECK(smi.alloc(n * NW));
  SQ_CHECK(gather_strings(NW, major, idx.p, sma.p, n, s));
  SQ_CHECK(gather_strings(NW, minor, idx.p, smi.p, n, s));
  SQ_CHECK(c.alloc(n * S));
  gather_coeffs_kernel<<<(unsigned)div_up(n * S, 256), 256, 0, s>>>(w, n, idx.p, S, c.p);
  SQ_LAUNCH_CHECK();
  return 0;
}

template <int NW>
static int one_rdm_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts, int64_t ldw, double *rdm) {
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  const int norb = T.norb;
  const bool ts = T.model == MODEL_CHEM && T.time_sym;
  DevBuf<uint64_t> up, dn;
  DevBuf<double> w;
  SQ_CHECK(up.alloc(n * NW));
  SQ_CHECK(dn.alloc(n * NW));
  SQ_CHECK(upload_dets(NW, norb, dets_up, up.p, n, s));
  SQ_CHECK(upload_dets(NW, norb, dets_dn, dn.p, n, s));
  SQ_CHECK(w.alloc(n * S));
  SQ_CUDA(cudaMemcpy2DAsync(w.p, n * sizeof(double), wts, ldw * sizeof(double), n * sizeof(double), S, cudaMemcpyHostToDevice, s));
  int64_t n2 = n;
  if (ts) {
    DevBuf<int32_t> flag, sel, nsel;
    SQ_CHECK(flag.alloc(n));
    SQ_CHECK(sel.alloc(n));
    SQ_CHECK(nsel.alloc(1));
    off_diagonal_flag_kernel<NW><<<(unsigned)div_up(n, 256), 256, 0, s>>>(up.p, dn.p, flag.p, n);
    SQ_LAUNCH_CHECK();
    thrust::counting_iterator<int32_t> rows(0);
    size_t tb = 0;
    cub::DeviceSelect::Flagged(nullptr, tb, rows, flag.p, sel.p, nsel.p, (int)n, s);
    DevBuf<char> tmp;
    SQ_CHECK(tmp.alloc((int64_t)tb + 16));
    SQ_CUDA(cub::DeviceSelect::Flagged(tmp.p, tb, rows, flag.p, sel.p, nsel.p, (int)n, s));
    g_launch_count += 1;
    int m = 0;
    SQ_CUDA(cudaMemcpyAsync(&m, nsel.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
    n2 = n + m;
    if (n2 > INT32_MAX) { set_error("one_rdm: %lld plain determinants after the time-reversal expansion exceed the 32-bit row index", (long long)n2); return 2; }
    DevBuf<uint64_t> eu, ed;
    DevBuf<double> ew;
    SQ_CHECK(eu.alloc(n2 * NW));
    SQ_CHECK(ed.alloc(n2 * NW));
    SQ_CHECK(ew.alloc(n2 * S));
    ts_expand_kernel<NW><<<(unsigned)div_up(n2, 256), 256, 0, s>>>(up.p, dn.p, w.p, n, sel.p, m, S, T.sqrt2inv, T.z * T.sqrt2inv, eu.p, ed.p, ew.p);
    SQ_LAUNCH_CHECK();
    up.release(); dn.release(); w.release();
    up.p = eu.take(); dn.p = ed.take(); w.p = ew.take();
    up.n = dn.n = n2 * NW;
    w.n = n2 * S;
  }
  // view 0: (up, dn) order, beta singles; view 1: (dn, up) order, alpha singles
  DevBuf<int32_t> idx0, idx1;
  DevBuf<uint64_t> ma0, mi0, ma1, mi1;
  DevBuf<double> c0, c1;
  SQ_CHECK(make_view<NW>(norb, up.p, dn.p, w.p, n2, S, idx0, ma0, mi0, c0, s));
  {
    DevBuf<int> flag;
    SQ_CHECK(flag.alloc(1));
    SQ_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), s));
    if (n2 > 1) {
      duplicate_kernel<NW><<<(unsigned)div_up(n2 - 1, 256), 256, 0, s>>>(ma0.p, mi0.p, idx0.p, n2, n, flag.p);
      SQ_LAUNCH_CHECK();
    }
    int hf = 0;
    SQ_CUDA(cudaMemcpyAsync(&hf, flag.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
    if (hf & 1) { set_error("one_rdm: the determinant list holds a determinant twice"); return 2; }
    if (hf & 2) { set_error("one_rdm: the list holds both (u,d) and its time-reversed partner (d,u); pass one representative per pair"); return 2; }
  }
  SQ_CHECK(make_view<NW>(norb, dn.p, up.p, w.p, n2, S, idx1, ma1, mi1, c1, s));
  up.release(); dn.release(); w.release(); idx0.release(); idx1.release();

  const int tri = norb * (norb + 1) / 2;
  const int64_t per = (int64_t)S * tri;
  const int nwarps = (int)std::min<int64_t>(kRdmMaxWarps, div_up(n2, 32));
  const int64_t chunk = div_up(n2, nwarps);
  const int wpb = kRdmThreads / 32;
  const size_t shmem = (size_t)wpb * per * sizeof(double);
  const int shared_acc = shmem <= kRdmSharedMax ? 1 : 0;
  DevBuf<double> part0, part1, out;
  SQ_CHECK(part0.alloc(nwarps * per));
  SQ_CHECK(part1.alloc(nwarps * per));
  SQ_CHECK(out.alloc((int64_t)S * 2 * norb * norb));
  auto kern = one_rdm_kernel<NW>;
  const size_t dyn = shared_acc ? shmem : 0;
  SQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  RdmView v0{ma0.p, mi0.p, c0.p, part0.p}, v1{ma1.p, mi1.p, c1.p, part1.p};
  kern<<<dim3((unsigned)div_up(nwarps, wpb), 2), kRdmThreads, dyn, s>>>(v0, v1, n2, norb, S, tri, chunk, nwarps, shared_acc);
  SQ_LAUNCH_CHECK();
  one_rdm_reduce_kernel<<<dim3((unsigned)per, 2), kRdmThreads, 0, s>>>(part0.p, part1.p, nwarps, S, tri, norb, out.p);
  SQ_LAUNCH_CHECK();
  SQ_CUDA(cudaMemcpyAsync(rdm, out.p, (size_t)S * 2 * norb * norb * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

int one_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw, double *rdm) {
  if (n <= 0) { set_error("one_rdm: n must be positive"); return 2; }
  if (n_states < 1) { set_error("one_rdm: n_states must be >= 1"); return 2; }
  if (ldw < n) { set_error("one_rdm: ldw (%lld) must be >= n (%lld)", (long long)ldw, (long long)n); return 2; }
  if (n > INT32_MAX) { set_error("one_rdm: n exceeds the 32-bit row index"); return 2; }
  return h->NW == 1 ? one_rdm_impl<1>(h, n, dets_up, dets_dn, n_states, wts, ldw, rdm)
                    : one_rdm_impl<2>(h, n, dets_up, dets_dn, n_states, wts, ldw, rdm);
}

}  // namespace sqmc
