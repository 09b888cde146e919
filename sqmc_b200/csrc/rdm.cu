// rdm.cu -- one- and two-particle density matrices of variational wavefunctions (sqmc_b200_one_rdm, sqmc_b200_two_rdm).
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
#include <vector>

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

// The part both density matrices share: upload, the time_sym expansion to n2 plain determinants (up, dn, w column-major
// n2 x S), and view 0 (sorted by (up, dn): idx0, ma0 = up, mi0 = dn, c0 interleaved) with the duplicate and partner check.
template <int NW>
static int prepare_dets(sqmc_b200_handle *h, const char *who, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts,
                        int64_t ldw, DevBuf<uint64_t> &up, DevBuf<uint64_t> &dn, DevBuf<double> &w, int64_t &n2, DevBuf<int32_t> &idx0,
                        DevBuf<uint64_t> &ma0, DevBuf<uint64_t> &mi0, DevBuf<double> &c0) {
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  const int norb = T.norb;
  const bool ts = T.model == MODEL_CHEM && T.time_sym;
  SQ_CHECK(up.alloc(n * NW));
  SQ_CHECK(dn.alloc(n * NW));
  SQ_CHECK(upload_dets(NW, norb, dets_up, up.p, n, s));
  SQ_CHECK(upload_dets(NW, norb, dets_dn, dn.p, n, s));
  SQ_CHECK(w.alloc(n * S));
  SQ_CUDA(cudaMemcpy2DAsync(w.p, n * sizeof(double), wts, ldw * sizeof(double), n * sizeof(double), S, cudaMemcpyHostToDevice, s));
  n2 = n;
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
    if (n2 > INT32_MAX) { set_error("%s: %lld plain determinants after the time-reversal expansion exceed the 32-bit row index", who, (long long)n2); return 2; }
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
  SQ_CHECK(make_view<NW>(norb, up.p, dn.p, w.p, n2, S, idx0, ma0, mi0, c0, s));
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
  if (hf & 1) { set_error("%s: the determinant list holds a determinant twice", who); return 2; }
  if (hf & 2) { set_error("%s: the list holds both (u,d) and its time-reversed partner (d,u); pass one representative per pair", who); return 2; }
  return 0;
}

template <int NW>
static int one_rdm_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts, int64_t ldw, double *rdm) {
  cudaStream_t s = G.stream;
  const int norb = h->T.norb;
  // view 0: (up, dn) order, beta singles; view 1: (dn, up) order, alpha singles
  DevBuf<uint64_t> up, dn;
  DevBuf<double> w;
  int64_t n2 = 0;
  DevBuf<int32_t> idx0, idx1;
  DevBuf<uint64_t> ma0, mi0, ma1, mi1;
  DevBuf<double> c0, c1;
  SQ_CHECK(prepare_dets<NW>(h, "one_rdm", n, dets_up, dets_dn, S, wts, ldw, up, dn, w, n2, idx0, ma0, mi0, c0));
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

// ---------------------------------------------------------------------------------------------------------------------
// two-particle density matrix (sqmc_b200_two_rdm), one-word strings
//
//   Gamma^{st}_{pq,rs} = <Psi| a+_{p s} a+_{r t} a_{s t} a_{q s} |Psi>,   blocks b = 0 (alpha alpha), 1 (alpha beta), 2 (beta beta)
//
// Pairs of determinants: every determinant emits hole keys of three classes, each class is sorted by key, and every pair of
// entries inside a run of equal keys (a bucket) is a connected pair met exactly once in that class:
//   same spin (alpha; beta mirrored): key (u \ {a,b}, d).  A pair whose removed sets are disjoint is an alpha double and has
//     exactly this one bucket.  A pair sharing one removed orbital r is an alpha single j -> i; it lies in N_alpha - 1 buckets,
//     one per r in u_i & u_j, and in each adds its one term Gamma^{aa}_{x_i x_j, r r}.
//   alpha beta: key (u \ {a}, d \ {b}).  Both removed orbitals differ: an alpha-beta double, one bucket.  Only a differs: an
//     alpha single, met once per beta orbital b, adding Gamma^{ab}_{x_i x_j, b b}; only b differs: the beta mirror.
// The diagonal terms c^2 of each determinant are added by a separate kernel that pre-reduces them per block in shared memory.
// Signs are the products of single-excitation permutation factors (alpha string first: beta operators pass every alpha
// electron twice), as in chem_single / chem_double.
//
// Only one representative per symmetry orbit is accumulated, and a fill kernel writes every element from its representative:
//   Gamma_{pq,rs} = Gamma_{qp,sr};  same spin also Gamma_{pq,rs} = -Gamma_{rq,ps} = -Gamma_{ps,rq}, and 0 when p = r or q = s.
// Same-spin representatives are indexed by the creator pair A = {p < r} and the annihilator pair B = {q < s}, A <= B; alpha-beta
// ones by (p + norb q, r + norb s) or its Hermitian image, whichever is smaller.
//
// Determinism: each representative is a 128-bit two's-complement fixed-point integer per state k, in units of 2^(e_k - 120)
// with 2^e_k >= sum_i c_ik^2 (by Cauchy-Schwarz no element exceeds that).  A term sign * c_i * c_j is rounded once to that grid
// and added with a 64-bit atomic on the low word plus the carry and sign extension on the high word.  Integer addition does not
// depend on order, so repeated calls and permuted rows give the same bits.
static const int kFixBits = 120;

__device__ __forceinline__ int par_between(uint64_t x, int a, int b) {  // parity of the electrons of x strictly between a and b
  const int lo = min(a, b), hi = max(a, b);
  return __popcll(x & ((1ull << hi) - 1ull) & ~((2ull << lo) - 1ull)) & 1;
}

// x (already on the fixed-point grid, |x| < 2^126) rounded to a 128-bit two's-complement integer (lo, hi)
__device__ __forceinline__ void fix_to_i128(double x, uint64_t &lo, uint64_t &hi) {
  if (fabs(x) < 9.0e18) {
    const long long v = __double2ll_rn(x);
    lo = (uint64_t)v;
    hi = v < 0 ? ~0ull : 0ull;
  } else {  // already an integer: the 53-bit mantissa shifted into place
    int e;
    const double m = frexp(x, &e);
    const __int128 v = (__int128)(long long)ldexp(m, 53) << (e - 53);
    lo = (uint64_t)v;
    hi = (uint64_t)(v >> 64);
  }
}
// adds (lo, hi) to the 128-bit value at slot[0] (low word), slot[1] (high word), global or shared memory
__device__ __forceinline__ void i128_add(unsigned long long *slot, uint64_t lo, uint64_t hi) {
  if ((lo | hi) == 0) return;
  const unsigned long long old = atomicAdd(slot, (unsigned long long)lo);
  const uint64_t h = hi + ((old + lo < old) ? 1ull : 0ull);
  if (h) atomicAdd(slot + 1, (unsigned long long)h);
}

__device__ __forceinline__ int pair_index(int p, int r) { return r * (r - 1) / 2 + p; }  // p < r
// representative of the same-spin element (p,q,r,s), p != r, q != s, inside an M x M block; sg: element = sg * representative
__device__ __forceinline__ int64_t ss_slot(int p, int q, int r, int s, int M, int &sg) {
  sg = 1;
  if (p > r) { const int t = p; p = r; r = t; sg = -sg; }
  if (q > s) { const int t = q; q = s; s = t; sg = -sg; }
  const int64_t A = pair_index(p, r), B = pair_index(q, s);
  return A <= B ? A + M * B : B + M * A;
}
__device__ __forceinline__ int64_t ab_slot(int p, int q, int r, int s, int norb) {
  int64_t X = p + (int64_t)norb * q, Y = r + (int64_t)norb * s;
  const int64_t X2 = q + (int64_t)norb * p, Y2 = s + (int64_t)norb * r;
  if (X2 < X || (X2 == X && Y2 < Y)) { X = X2; Y = Y2; }
  return X + (int64_t)norb * norb * Y;
}

struct Rdm2Acc {
  unsigned long long *a;  // [S][per] slots of two words
  const double *scale;    // [S] 2^(120 - e_k)
  int64_t per, off_bb, off_ab;
  int M, norb, S;
};

__global__ void electron_count_kernel(const uint64_t *u, const uint64_t *d, int64_t n, int nup, int ndn, int *bad) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n && (__popcll(u[i]) != nup || __popcll(d[i]) != ndn)) atomicOr(bad, 1);
}

// same-spin keys: (x \ {a, b}, y) for every pair a < b of x; payload row << 16 | a | b << 8
__global__ void rdm2_keys_same_kernel(const uint64_t *x, const uint64_t *y, int64_t n, int K, uint64_t *ku, uint64_t *kd, uint64_t *pay) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t X = x[i], Y = y[i];
  int64_t e = i * K;
  for (uint64_t as = X; as; as &= as - 1) {
    const int a = __ffsll((long long)as) - 1;
    for (uint64_t bs = as & (as - 1); bs; bs &= bs - 1) {
      const int b = __ffsll((long long)bs) - 1;
      ku[e] = X & ~(1ull << a) & ~(1ull << b);
      kd[e] = Y;
      pay[e] = (uint64_t)i << 16 | (uint64_t)a | (uint64_t)b << 8;
      e++;
    }
  }
}
// alpha-beta keys: (u \ {a}, d \ {b}); payload row << 16 | a | b << 8
__global__ void rdm2_keys_ab_kernel(const uint64_t *u, const uint64_t *d, int64_t n, int K, uint64_t *ku, uint64_t *kd, uint64_t *pay) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t U = u[i], D = d[i];
  int64_t e = i * K;
  for (uint64_t as = U; as; as &= as - 1) {
    const int a = __ffsll((long long)as) - 1;
    for (uint64_t bs = D; bs; bs &= bs - 1) {
      const int b = __ffsll((long long)bs) - 1;
      ku[e] = U & ~(1ull << a);
      kd[e] = D & ~(1ull << b);
      pay[e] = (uint64_t)i << 16 | (uint64_t)a | (uint64_t)b << 8;
      e++;
    }
  }
}

// one thread per sorted entry i: every later entry j of the same bucket; boff: block offset of a same-spin class, -1: alpha beta
__global__ void __launch_bounds__(256) rdm2_pair_kernel(const uint64_t *ku, const uint64_t *kd, const uint64_t *pay, int64_t m, int64_t boff,
                                                        const double *coef, Rdm2Acc R) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const uint64_t ki = ku[i], kdi = kd[i], pi = pay[i];
  const int ai = (int)(pi & 0xff), bi = (int)((pi >> 8) & 0xff);
  const double *ci = coef + (int64_t)(pi >> 16) * R.S;
  for (int64_t j = i + 1; j < m && ku[j] == ki && kd[j] == kdi; j++) {
    const uint64_t pj = pay[j];
    const int aj = (int)(pj & 0xff), bj = (int)((pj >> 8) & 0xff);
    int neg, sg = 1;
    int64_t slot;
    if (boff >= 0) {
      int p, q, r, s;
      if (ai != aj && ai != bj && bi != aj && bi != bj) {  // double: <i| a+_ai a+_bi a_bj a_aj |j> = <i| a+_ai a_aj a+_bi a_bj |j>
        const uint64_t uj = ki | 1ull << aj | 1ull << bj;
        neg = par_between(uj, bi, bj) ^ par_between(uj ^ (1ull << bj) ^ (1ull << bi), ai, aj);
        p = ai; q = aj; r = bi; s = bj;
      } else {  // single x_j -> x_i; the shared removed orbital r stays occupied in both
        const int r0 = (ai == aj || ai == bj) ? ai : bi;
        const int xi = ai == r0 ? bi : ai, xj = aj == r0 ? bj : aj;
        neg = par_between(ki | 1ull << r0, xi, xj);
        p = xi; q = xj; r = r0; s = r0;
      }
      slot = boff + ss_slot(p, q, r, s, R.M, sg);
    } else if (ai != aj && bi != bj) {
      neg = par_between(ki, ai, aj) ^ par_between(kdi, bi, bj);
      slot = R.off_ab + ab_slot(ai, aj, bi, bj, R.norb);
    } else if (ai != aj) {
      neg = par_between(ki, ai, aj);
      slot = R.off_ab + ab_slot(ai, aj, bi, bi, R.norb);
    } else {
      neg = par_between(kdi, bi, bj);
      slot = R.off_ab + ab_slot(ai, ai, bi, bj, R.norb);
    }
    const double f = (neg ? -1.0 : 1.0) * sg;
    const double *cj = coef + (int64_t)(pj >> 16) * R.S;
    for (int k = 0; k < R.S; k++) {
      uint64_t lo, hi;
      fix_to_i128(f * (ci[k] * cj[k]) * R.scale[k], lo, hi);
      i128_add(R.a + 2 * (k * R.per + slot), lo, hi);
    }
  }
}

// diagonal terms c_i^2: Gamma^{ss}_{pp,rr} (p < r occupied in the same string) and Gamma^{ab}_{pp,rr}, one state at a time,
// summed per block in shared memory ([3][norb][norb] 128-bit values) and then added to the representatives
__global__ void __launch_bounds__(256) rdm2_diag_kernel(const uint64_t *u, const uint64_t *d, int64_t n, const double *coef, Rdm2Acc R) {
  extern __shared__ unsigned long long sd[];
  const int norb = R.norb, nn = norb * norb;
  for (int k = 0; k < R.S; k++) {
    for (int t = threadIdx.x; t < 6 * nn; t += blockDim.x) sd[t] = 0ull;
    __syncthreads();
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
      const double c = coef[i * R.S + k];
      uint64_t lo, hi;
      fix_to_i128((c * c) * R.scale[k], lo, hi);
      if ((lo | hi) == 0) continue;
      const uint64_t U = u[i], D = d[i];
      for (uint64_t ps = U; ps; ps &= ps - 1) {
        const int p = __ffsll((long long)ps) - 1;
        for (uint64_t rs = ps & (ps - 1); rs; rs &= rs - 1) i128_add(sd + 2 * (p * norb + __ffsll((long long)rs) - 1), lo, hi);
        for (uint64_t rs = D; rs; rs &= rs - 1) i128_add(sd + 2 * (2 * nn + p * norb + __ffsll((long long)rs) - 1), lo, hi);
      }
      for (uint64_t ps = D; ps; ps &= ps - 1) {
        const int p = __ffsll((long long)ps) - 1;
        for (uint64_t rs = ps & (ps - 1); rs; rs &= rs - 1) i128_add(sd + 2 * (nn + p * norb + __ffsll((long long)rs) - 1), lo, hi);
      }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 3 * nn; t += blockDim.x) {
      const uint64_t lo = sd[2 * t], hi = sd[2 * t + 1];
      if ((lo | hi) == 0) continue;
      const int b = t / nn, p = (t % nn) / norb, r = t % norb;
      int64_t slot;
      if (b == 2) {
        slot = R.off_ab + ab_slot(p, p, r, r, norb);
      } else {
        const int64_t A = pair_index(p, r);
        slot = (b ? R.off_bb : 0) + A + R.M * A;
      }
      i128_add(R.a + 2 * (k * R.per + slot), lo, hi);
    }
    __syncthreads();
  }
}

// every element of the output (column-major p, q, r, s, block, state) from its representative
__global__ void rdm2_fill_kernel(Rdm2Acc R, const double *unscale, double *out) {
  const int norb = R.norb;
  const int64_t n4 = (int64_t)norb * norb * norb * norb, total = n4 * 3 * R.S;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t x = t;
    const int p = (int)(x % norb); x /= norb;
    const int q = (int)(x % norb); x /= norb;
    const int r = (int)(x % norb); x /= norb;
    const int s = (int)(x % norb); x /= norb;
    const int b = (int)(x % 3);
    const int k = (int)(x / 3);
    int sg = 1;
    int64_t slot;
    if (b == 1) {
      slot = R.off_ab + ab_slot(p, q, r, s, norb);
    } else if (p == r || q == s) {
      out[t] = 0.0;
      continue;
    } else {
      slot = (b ? R.off_bb : 0) + ss_slot(p, q, r, s, R.M, sg);
    }
    const unsigned long long *v = R.a + 2 * (k * R.per + slot);
    const double a = (ldexp((double)(long long)v[1], 64) + (double)v[0]) * unscale[k];
    out[t] = sg < 0 ? -a : a;
  }
}

// sum_i c_ik^2 per state over the sorted view (its order does not depend on the caller's rows): thread t sums rows t, t + 256,
// ... in order, then a fixed tree
__global__ void __launch_bounds__(256) norm2_kernel(const double *c, int64_t n, int S, double *norm2) {
  __shared__ double red[256];
  const int k = blockIdx.x;
  double a = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += 256) a += c[i * S + k] * c[i * S + k];
  red[threadIdx.x] = a;
  __syncthreads();
  for (int hh = 128; hh > 0; hh >>= 1) {
    if (threadIdx.x < hh) red[threadIdx.x] += red[threadIdx.x + hh];
    __syncthreads();
  }
  if (threadIdx.x == 0) norm2[k] = red[0];
}

// The accumulation both two-particle entry points share: upload, time_sym expansion, checks, the diagonal and the three key
// classes with their pairs.  On return acc / scale hold the representatives of R (scale[S + k]: the factor back to doubles);
// norm2 (device, S doubles, may be null) receives ||Psi_k||^2 summed in a fixed order.
static int rdm2_accumulate(sqmc_b200_handle *h, const char *who, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts,
                           int64_t ldw, HostMarks &marks, DevBuf<unsigned long long> &acc, DevBuf<double> &scale, Rdm2Acc &R, double *norm2) {
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  const int norb = T.norb;
  DevBuf<uint64_t> up, dn, U, D;
  DevBuf<double> w, c;
  DevBuf<int32_t> idx0;
  int64_t n2 = 0;
  SQ_CHECK(prepare_dets<1>(h, who, n, dets_up, dets_dn, S, wts, ldw, up, dn, w, n2, idx0, U, D, c));
  up.release(); dn.release(); w.release(); idx0.release();
  marks.mark("upload, expansion, checks");
  {
    DevBuf<int> bad;
    SQ_CHECK(bad.alloc(1));
    SQ_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), s));
    electron_count_kernel<<<(unsigned)div_up(n2, 256), 256, 0, s>>>(U.p, D.p, n2, T.nup, T.ndn, bad.p);
    SQ_LAUNCH_CHECK();
    int hb = 0;
    SQ_CUDA(cudaMemcpyAsync(&hb, bad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
    if (hb) { set_error("%s: a determinant does not hold %d alpha and %d beta electrons", who, T.nup, T.ndn); return 2; }
  }
  if (norm2) {
    norm2_kernel<<<S, 256, 0, s>>>(c.p, n2, S, norm2);
    SQ_LAUNCH_CHECK();
  }
  // grid exponent per state from sum_i w_ik^2 (the time_sym expansion keeps it); the margin keeps e_k the same whatever order
  // the sum was taken in, unless the norm lies within a few ulps of 2^e / (1 + 2^-20)
  std::vector<double> hs(2 * S);
  for (int k = 0; k < S; k++) {
    double n2k = 0.0;
    for (int64_t i = 0; i < n; i++) n2k += wts[k * ldw + i] * wts[k * ldw + i];
    int e = 0;
    if (n2k > 0.0) frexp(n2k * (1.0 + 0x1p-20), &e);
    hs[k] = ldexp(1.0, kFixBits - e);
    hs[S + k] = ldexp(1.0, e - kFixBits);
  }
  const int M = norb * (norb - 1) / 2;
  const int64_t n4 = (int64_t)norb * norb * norb * norb;
  R.M = M; R.norb = norb; R.S = S;
  R.off_bb = (int64_t)M * M;
  R.off_ab = 2 * R.off_bb;
  R.per = R.off_ab + n4;
  SQ_CHECK(acc.alloc(2 * S * R.per));
  SQ_CHECK(scale.alloc(2 * S));
  SQ_CUDA(cudaMemsetAsync(acc.p, 0, (size_t)acc.n * sizeof(unsigned long long), s));
  SQ_CUDA(cudaMemcpyAsync(scale.p, hs.data(), 2 * S * sizeof(double), cudaMemcpyHostToDevice, s));
  R.a = acc.p;
  R.scale = scale.p;

  const size_t dsh = (size_t)6 * norb * norb * sizeof(unsigned long long);
  SQ_CUDA(cudaFuncSetAttribute(rdm2_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsh));
  rdm2_diag_kernel<<<(unsigned)std::min<int64_t>(div_up(n2, 256), 2 * G.sm_count), 256, dsh, s>>>(U.p, D.p, n2, c.p, R);
  SQ_LAUNCH_CHECK();
  marks.mark("diagonal");

  // class 0: alpha holes (block 0), 1: beta holes (block 2), 2: one hole of each spin (block 1)
  for (int cls = 0; cls < 3; cls++) {
    const int K = cls == 0 ? T.nup * (T.nup - 1) / 2 : cls == 1 ? T.ndn * (T.ndn - 1) / 2 : T.nup * T.ndn;
    if (K == 0 || n2 < 2) continue;
    const int64_t m = n2 * K;
    if (m > INT32_MAX) { set_error("%s: %lld hole keys (%lld determinants x %d) exceed the 32-bit sort index", who, (long long)m, (long long)n2, K); return 2; }
    DevBuf<uint64_t> ku, kd, pay, sku, skd, spay;
    DevBuf<int32_t> idx;
    SQ_CHECK(ku.alloc(m));
    SQ_CHECK(kd.alloc(m));
    SQ_CHECK(pay.alloc(m));
    if (cls == 2) rdm2_keys_ab_kernel<<<(unsigned)div_up(n2, 256), 256, 0, s>>>(U.p, D.p, n2, K, ku.p, kd.p, pay.p);
    else rdm2_keys_same_kernel<<<(unsigned)div_up(n2, 256), 256, 0, s>>>(cls ? D.p : U.p, cls ? U.p : D.p, n2, K, ku.p, kd.p, pay.p);
    SQ_LAUNCH_CHECK();
    SQ_CHECK(idx.alloc(m));
    SQ_CHECK(sort_pairs_index(1, norb, ku.p, kd.p, idx.p, m, s));
    SQ_CHECK(sku.alloc(m));
    SQ_CHECK(gather_strings(1, ku.p, idx.p, sku.p, m, s));
    ku.release();
    SQ_CHECK(skd.alloc(m));
    SQ_CHECK(gather_strings(1, kd.p, idx.p, skd.p, m, s));
    kd.release();
    SQ_CHECK(spay.alloc(m));
    SQ_CHECK(gather_strings(1, pay.p, idx.p, spay.p, m, s));
    pay.release(); idx.release();
    marks.mark(cls == 0 ? "alpha alpha keys + sort" : cls == 1 ? "beta beta keys + sort" : "alpha beta keys + sort");
    rdm2_pair_kernel<<<(unsigned)div_up(m, 256), 256, 0, s>>>(sku.p, skd.p, spay.p, m, cls == 2 ? -1 : cls == 0 ? 0 : R.off_bb, c.p, R);
    SQ_LAUNCH_CHECK();
    marks.mark(cls == 0 ? "alpha alpha pairs" : cls == 1 ? "beta beta pairs" : "alpha beta pairs");
  }
  return 0;
}

static int two_rdm_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts, int64_t ldw, double *rdm) {
  cudaStream_t s = G.stream;
  const int norb = h->T.norb;
  HostMarks marks("SQMC_RDM2_PROFILE", "two_rdm");  // =1: phase split (synchronising) on stderr
  DevBuf<unsigned long long> acc;
  DevBuf<double> scale;
  Rdm2Acc R;
  SQ_CHECK(rdm2_accumulate(h, "two_rdm", n, dets_up, dets_dn, S, wts, ldw, marks, acc, scale, R, nullptr));
  const int64_t n4 = (int64_t)norb * norb * norb * norb;
  DevBuf<double> out;
  SQ_CHECK(out.alloc(3 * S * n4));
  rdm2_fill_kernel<<<(unsigned)std::min<int64_t>(div_up(3 * S * n4, 256), 64 * G.sm_count), 256, 0, s>>>(R, scale.p + S, out.p);
  SQ_LAUNCH_CHECK();
  SQ_CUDA(cudaMemcpyAsync(rdm, out.p, (size_t)out.n * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  marks.mark("fill + copy out");
  return 0;
}

// argument checks both two-particle entry points share
static int rdm2_check_args(sqmc_b200_handle *h, const char *who, int64_t n, int n_states, int64_t ldw) {
  if (n <= 0) { set_error("%s: n must be positive", who); return 2; }
  if (n_states < 1) { set_error("%s: n_states must be >= 1", who); return 2; }
  if (ldw < n) { set_error("%s: ldw (%lld) must be >= n (%lld)", who, (long long)ldw, (long long)n); return 2; }
  if (n > INT32_MAX) { set_error("%s: n exceeds the 32-bit row index", who); return 2; }
  if (h->T.norb > 64) {
    set_error("%s: norb = %d > 64 is not supported (the dense output holds 3*norb^4 doubles per state, and strings of more than one word are not handled)",
              who, h->T.norb);
    return 2;
  }
  return 0;
}

int two_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw, double *rdm) {
  SQ_CHECK(rdm2_check_args(h, "two_rdm", n, n_states, ldw));
  return two_rdm_impl(h, n, dets_up, dets_dn, n_states, wts, ldw, rdm);
}

// ---------------------------------------------------------------------------------------------------------------------
// orbital gradient and Hessian of the variational energy (sqmc_b200_orbital_derivatives), chem, norb <= 64
//
// Helgaker, Jorgensen, Olsen, Molecular Electronic-Structure Theory, 10.8.1 (real orbitals, kappa = sum_{p>q} k_pq E-_pq):
//   D_pq   = sum_k w_k (gamma^a + gamma^b)_pq / ||Psi_k||^2,   d_pqrs = sum_k w_k (G^aa + G^bb + G^ab_pq,rs + G^ab_rs,pq) / ||Psi_k||^2
//   F_pq   = sum_m D_pm h_qm + sum_mnt d_pmnt g_qmnt                                 (gradient 2 (F_pq - F_qp))
//   Y_pqrs = sum_mn [(d_pmrn + d_pmnr) g_qmsn + d_prmn g_qsmn]
//   E2_pq,rs = (1 - P_pq)(1 - P_rs) [2 D_pr h_qs - (F_pr + F_rp) delta_qs + 2 Y_pqrs]
// d is filled from the two_rdm representatives and never leaves the device; D is its partial trace sum_r d_pqrr / (N - 1).
// F and Y are both products C = A B^T of column-major matrices in FP64 (orb_gemm_kernel): F with A = [D | d] (norb x
// (norb + norb^3)) and B = [h | g]; Y with rows (p + norb r), columns (q + norb s) and A = [X | d], B = [G | g] over
// (m + norb n), X = d_pmrn + d_pmnr, G = g_qmsn (the d_prmn g_qsmn term reads d and g as they are stored).  Every output is
// summed by one thread in k order, and split-K partials are added in a fixed order: no atomics anywhere.

// d (p,q,r,s at p + norb (q + norb (r + norb s))) from the representatives, spin summed and state averaged; f[k] = w_k / ||Psi_k||^2
__global__ void orbd_fill_kernel(Rdm2Acc R, const double *unscale, const double *state_w, const double *norm2, double *d) {
  const int norb = R.norb;
  const int64_t n4 = (int64_t)norb * norb * norb * norb;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n4; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t x = t;
    const int p = (int)(x % norb); x /= norb;
    const int q = (int)(x % norb); x /= norb;
    const int r = (int)(x % norb);
    const int s = (int)(x / norb);
    double v = 0.0;
    for (int k = 0; k < R.S; k++) {
      const unsigned long long *a = R.a + 2 * (int64_t)k * R.per;
      auto val = [&](int64_t slot) { return (ldexp((double)(long long)a[2 * slot + 1], 64) + (double)a[2 * slot]) * unscale[k]; };
      double e = val(R.off_ab + ab_slot(p, q, r, s, norb)) + val(R.off_ab + ab_slot(r, s, p, q, norb));
      if (p != r && q != s) {
        int sg;
        const int64_t slot = ss_slot(p, q, r, s, R.M, sg);
        const double ss = val(slot) + val(R.off_bb + slot);
        e += sg < 0 ? -ss : ss;
      }
      v += (state_w[k] / norm2[k]) * e;
    }
    d[t] = v;
  }
}

// D_pq = sum_r d_pqrr / (N - 1), r in order
__global__ void orbd_trace_kernel(const double *d, int norb, double inv_nm1, double *D) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int nn = norb * norb;
  if (t >= nn) return;
  double a = 0.0;
  for (int r = 0; r < norb; r++) a += d[t + (int64_t)nn * (r + (int64_t)norb * r)];
  D[t] = a * inv_nm1;
}

// dense h (p + norb q) and g (p + norb (q + norb (r + norb s))) from the handle's integral table, as ChemCtx::I reads it
__global__ void orbd_integrals_kernel(const double *ints, const int32_t *c2, int norb, double *hd, double *gd) {
  const int n1 = norb + 1;
  const int64_t nn = (int64_t)norb * norb, n4 = nn * nn;
  const long long core = c2[norb * n1 + norb];
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n4 + nn; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t u = t < n4 ? t : t - n4;
    const long long a = c2[(u / norb % norb) * n1 + u % norb];
    const long long b = t < n4 ? c2[(u / nn / norb) * n1 + u / nn % norb] : core;
    const long long idx = a > b ? a * (a - 1) / 2 + b : b * (b - 1) / 2 + a;
    (t < n4 ? gd : hd)[u] = ints[idx - 1];
  }
}

// X[(p + norb r) + norb^2 (m + norb n)] = d_pmrn + d_pmnr and G[(q + norb s) + norb^2 (m + norb n)] = g_qmsn
__global__ void orbd_y_operands_kernel(const double *d, const double *g, int norb, double *X, double *Gq) {
  const int64_t nn = (int64_t)norb * norb, n4 = nn * nn;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n4; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t x = t;
    const int64_t p = x % norb; x /= norb;
    const int64_t r = x % norb; x /= norb;
    const int64_t m = x % norb;
    const int64_t n = x / norb;
    X[t] = d[p + norb * (m + norb * (r + norb * n))] + d[p + norb * (m + norb * (n + norb * r))];
    Gq[t] = g[p + norb * (m + norb * (r + norb * n))];
  }
}

static const int kGemmTile = 64, kGemmK = 16, kGemmThreads = 256;
struct GemmSeg {  // A(i, k) = a[i + M k], B(j, k) = b[j + N k] for k < K
  const double *a, *b;
  int64_t K;
};

// part[z][i + M j] = sum over the k of chunk z of A(i,k) B(j,k), k running over segment 0 then segment 1.  64 x 64 tile per
// block, 4 x 4 outputs per thread (rows tx + 16 x, columns ty + 16 y), 16-deep k slices staged in shared memory.
__global__ void __launch_bounds__(kGemmThreads) orb_gemm_kernel(GemmSeg s0, GemmSeg s1, int M, int N, int64_t kchunk, double *part) {
  __shared__ double As[kGemmK][kGemmTile], Bs[kGemmK][kGemmTile];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int i0 = blockIdx.x * kGemmTile, j0 = blockIdx.y * kGemmTile;
  const int64_t K = s0.K + s1.K;
  const int64_t kb = blockIdx.z * kchunk, ke = min(K, kb + kchunk);
  double acc[4][4];
#pragma unroll
  for (int x = 0; x < 4; x++)
#pragma unroll
    for (int y = 0; y < 4; y++) acc[x][y] = 0.0;
  for (int64_t k0 = kb; k0 < ke; k0 += kGemmK) {
#pragma unroll
    for (int e = threadIdx.x; e < kGemmK * kGemmTile; e += kGemmThreads) {
      const int kk = e / kGemmTile, ii = e % kGemmTile;
      const int64_t k = k0 + kk;
      double av = 0.0, bv = 0.0;
      if (k < ke) {
        const bool first = k < s0.K;
        const int64_t kl = first ? k : k - s0.K;
        if (i0 + ii < M) av = (first ? s0.a : s1.a)[i0 + ii + (int64_t)M * kl];
        if (j0 + ii < N) bv = (first ? s0.b : s1.b)[j0 + ii + (int64_t)N * kl];
      }
      As[kk][ii] = av;
      Bs[kk][ii] = bv;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kGemmK; kk++) {
      double a[4], b[4];
#pragma unroll
      for (int x = 0; x < 4; x++) a[x] = As[kk][tx + 16 * x];
#pragma unroll
      for (int y = 0; y < 4; y++) b[y] = Bs[kk][ty + 16 * y];
#pragma unroll
      for (int x = 0; x < 4; x++)
#pragma unroll
        for (int y = 0; y < 4; y++) acc[x][y] = fma(a[x], b[y], acc[x][y]);
    }
    __syncthreads();
  }
  double *c = part + (int64_t)blockIdx.z * M * N;
#pragma unroll
  for (int x = 0; x < 4; x++)
#pragma unroll
    for (int y = 0; y < 4; y++) {
      const int i = i0 + tx + 16 * x, j = j0 + ty + 16 * y;
      if (i < M && j < N) c[i + (int64_t)M * j] = acc[x][y];
    }
}

// out[t] = sum_z part[z][t], z in order
__global__ void orb_splitk_reduce_kernel(const double *part, int64_t mn, int nz, double *out) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < mn; t += (int64_t)gridDim.x * blockDim.x) {
    double a = 0.0;
    for (int z = 0; z < nz; z++) a += part[z * mn + t];
    out[t] = a;
  }
}

// C = A B^T (M x N, column-major) over the two segments; split-K when the output has too few tiles to fill the GPU
static int orb_gemm(GemmSeg s0, GemmSeg s1, int M, int N, double *C, cudaStream_t s) {
  const int64_t K = s0.K + s1.K;
  const int64_t tiles = div_up(M, kGemmTile) * div_up(N, kGemmTile);
  const int64_t kslices = div_up(K, kGemmK);
  const int nz = (int)std::max<int64_t>(1, std::min<int64_t>(kslices, div_up(2 * G.sm_count, tiles)));
  const int64_t kchunk = div_up(kslices, nz) * kGemmK;
  const int nzu = (int)div_up(K, kchunk);
  DevBuf<double> part;
  if (nzu > 1) SQ_CHECK(part.alloc((int64_t)nzu * M * N));
  dim3 grid((unsigned)div_up(M, kGemmTile), (unsigned)div_up(N, kGemmTile), (unsigned)nzu);
  orb_gemm_kernel<<<grid, kGemmThreads, 0, s>>>(s0, s1, M, N, kchunk, nzu > 1 ? part.p : C);
  SQ_LAUNCH_CHECK();
  if (nzu > 1) {
    const int64_t mn = (int64_t)M * N;
    orb_splitk_reduce_kernel<<<(unsigned)std::min<int64_t>(div_up(mn, 256), 8 * G.sm_count), 256, 0, s>>>(part.p, mn, nzu, C);
    SQ_LAUNCH_CHECK();
  }
  return 0;
}

// E2 from D, h, F and Y (Y[(p + norb r) + norb^2 (q + norb s)]); the four permuted terms added in a fixed order
__global__ void orbd_hessian_kernel(const double *D, const double *hd, const double *F, const double *Y, int norb, double *E2) {
  const int64_t nn = (int64_t)norb * norb, n4 = nn * nn;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n4; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t x = t;
    const int p = (int)(x % norb); x /= norb;
    const int q = (int)(x % norb); x /= norb;
    const int r = (int)(x % norb);
    const int s = (int)(x / norb);
    auto f = [&](int a, int b, int c, int e) {
      double v = 2.0 * D[a + (int64_t)norb * c] * hd[b + (int64_t)norb * e];
      if (b == e) v -= F[a + (int64_t)norb * c] + F[c + (int64_t)norb * a];
      return v + 2.0 * Y[(a + (int64_t)norb * c) + nn * (b + (int64_t)norb * e)];
    };
    E2[t] = ((f(p, q, r, s) - f(q, p, r, s)) - f(p, q, s, r)) + f(q, p, s, r);
  }
}

// energy = E_core + 1/2 (sum_pq h_pq D_pq + sum_p F_pp), one block, fixed order
__global__ void __launch_bounds__(256) orbd_energy_kernel(const double *D, const double *hd, const double *F, int norb, double ecore, double *e) {
  __shared__ double red[256];
  const int nn = norb * norb;
  double a = 0.0;
  for (int t = threadIdx.x; t < nn; t += 256) a += hd[t] * D[t];
  for (int p = threadIdx.x; p < norb; p += 256) a += F[p + norb * p];
  red[threadIdx.x] = a;
  __syncthreads();
  for (int hh = 128; hh > 0; hh >>= 1) {
    if (threadIdx.x < hh) red[threadIdx.x] += red[threadIdx.x + hh];
    __syncthreads();
  }
  if (threadIdx.x == 0) *e = ecore + 0.5 * red[0];
}

static int orbital_derivatives_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts,
                                    int64_t ldw, const double *state_weights, double *fock, double *hessian, double *energy) {
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  const int norb = T.norb;
  const int64_t nn = (int64_t)norb * norb, n4 = nn * nn;
  HostMarks marks("SQMC_ORBD_PROFILE", "orbital_derivatives");  // =1: phase split (synchronising) on stderr
  DevBuf<double> norm2, sw;
  SQ_CHECK(norm2.alloc(S));
  SQ_CHECK(sw.alloc(S));
  SQ_CUDA(cudaMemcpyAsync(sw.p, state_weights, S * sizeof(double), cudaMemcpyHostToDevice, s));
  DevBuf<double> d, D;
  {
    DevBuf<unsigned long long> acc;
    DevBuf<double> scale;
    Rdm2Acc R;
    SQ_CHECK(rdm2_accumulate(h, "orbital_derivatives", n, dets_up, dets_dn, S, wts, ldw, marks, acc, scale, R, norm2.p));
    SQ_CHECK(d.alloc(n4));
    orbd_fill_kernel<<<(unsigned)std::min<int64_t>(div_up(n4, 256), 64 * G.sm_count), 256, 0, s>>>(R, scale.p + S, sw.p, norm2.p, d.p);
    SQ_LAUNCH_CHECK();
  }
  SQ_CHECK(D.alloc(nn));
  orbd_trace_kernel<<<(unsigned)div_up(nn, 256), 256, 0, s>>>(d.p, norb, 1.0 / (T.nup + T.ndn - 1), D.p);
  SQ_LAUNCH_CHECK();
  DevBuf<double> hd, gd;
  SQ_CHECK(hd.alloc(nn));
  SQ_CHECK(gd.alloc(n4));
  orbd_integrals_kernel<<<(unsigned)std::min<int64_t>(div_up(n4 + nn, 256), 64 * G.sm_count), 256, 0, s>>>(T.integrals, T.combine_2, norb, hd.p, gd.p);
  SQ_LAUNCH_CHECK();
  marks.mark("d, D, dense integrals");
  DevBuf<double> F, X, Gq, Y, E2, e;
  SQ_CHECK(F.alloc(nn));
  SQ_CHECK(orb_gemm(GemmSeg{D.p, hd.p, norb}, GemmSeg{d.p, gd.p, nn * norb}, norb, norb, F.p, s));
  SQ_CHECK(X.alloc(n4));
  SQ_CHECK(Gq.alloc(n4));
  orbd_y_operands_kernel<<<(unsigned)std::min<int64_t>(div_up(n4, 256), 64 * G.sm_count), 256, 0, s>>>(d.p, gd.p, norb, X.p, Gq.p);
  SQ_LAUNCH_CHECK();
  SQ_CHECK(Y.alloc(n4));
  SQ_CHECK(orb_gemm(GemmSeg{X.p, Gq.p, nn}, GemmSeg{d.p, gd.p, nn}, (int)nn, (int)nn, Y.p, s));
  X.release(); Gq.release(); d.release(); gd.release();
  SQ_CHECK(E2.alloc(n4));
  orbd_hessian_kernel<<<(unsigned)std::min<int64_t>(div_up(n4, 256), 64 * G.sm_count), 256, 0, s>>>(D.p, hd.p, F.p, Y.p, norb, E2.p);
  SQ_LAUNCH_CHECK();
  SQ_CHECK(e.alloc(1));
  orbd_energy_kernel<<<1, 256, 0, s>>>(D.p, hd.p, F.p, norb, T.enuc, e.p);  // T.enuc: table entry _index(n1, n1, n1, n1)
  SQ_LAUNCH_CHECK();
  marks.mark("contractions");
  SQ_CUDA(cudaMemcpyAsync(fock, F.p, nn * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaMemcpyAsync(hessian, E2.p, n4 * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaMemcpyAsync(energy, e.p, sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  marks.mark("copy out");
  return 0;
}

int orbital_derivatives(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw,
                        const double *state_weights, double *fock, double *hessian, double *energy) {
  if (h->T.model != MODEL_CHEM) {
    set_error("orbital_derivatives: only chem handles have orbitals to optimise (heg and hubbardk orbitals are fixed by momentum)");
    return 2;
  }
  SQ_CHECK(rdm2_check_args(h, "orbital_derivatives", n, n_states, ldw));
  if (h->T.nup + h->T.ndn < 2) { set_error("orbital_derivatives: needs at least two electrons"); return 2; }
  double sum = 0.0;
  for (int k = 0; k < n_states; k++) {
    if (!(state_weights[k] >= 0.0)) { set_error("orbital_derivatives: state_weights[%d] = %g is negative", k, state_weights[k]); return 2; }
    sum += state_weights[k];
  }
  if (!(fabs(sum - 1.0) <= 1e-12)) { set_error("orbital_derivatives: state_weights sum to %.17g, not 1", sum); return 2; }
  return orbital_derivatives_impl(h, n, dets_up, dets_dn, n_states, wts, ldw, state_weights, fock, hessian, energy);
}

}  // namespace sqmc
