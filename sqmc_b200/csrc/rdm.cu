// rdm.cu -- one- and two-particle density matrices of variational wavefunctions (sqmc_b200_one_rdm, sqmc_b200_two_rdm), the
// orbital-optimisation quantities built on them, and the ladder images a_p|Psi>, a+_p|Psi> of the Green's function (sqmc_b200_ladder).
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
//
// Transition mode (sqmc_b200_transition_one_rdm, TR = true): every row holds 2S coefficients, bra a_k at k and ket b_k at
// S + k, and gamma^{ab}_pq = <a| a+_p a_q |b> is accumulated as the full norb x norb matrix.  The pair D_j = sg a+_p a_q D_i
// (p > q) adds (sg a_i) b_j to (q,p) and (sg a_j) b_i to (p,q), the diagonal a_i b_i.  Both slots of a pair belong to one
// lane, so the warp-private accumulation and the reduction tree are those of one_rdm; for a = b every product has the bits
// of its one_rdm counterpart (IEEE products commute), so the result is one_rdm's bit for bit.
#include <thrust/iterator/counting_iterator.h>

#include <cub/cub.cuh>
#include <cstring>
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

// tri: accumulator slots per state, the packed triangle (TR = false) or norb^2 (TR = true, (p,q) at p + norb q)
template <int NW, bool TR>
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
    const int cs = TR ? 2 * S : S;
    const double *ci = coef + i * cs;
    for (int p = lane; p < norb; p += 32) {
      if (b_test(mi, p)) {
        if constexpr (TR) {
          for (int s = 0; s < S; s++) acc[s * tri + p + norb * p] += ci[s] * ci[S + s];
        } else {
          const int t = tri_slot(p, p);
          for (int s = 0; s < S; s++) acc[s * tri + t] += ci[s] * ci[s];
        }
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
      const double *cj = coef + lo * cs;
      if constexpr (TR) {
        for (int s = 0; s < S; s++) {
          acc[s * tri + q + norb * p] += (sg * ci[s]) * cj[S + s];
          acc[s * tri + p + norb * q] += (sg * cj[s]) * ci[S + s];
        }
      } else {
        const int t = tri_slot(p, q);
        for (int s = 0; s < S; s++) acc[s * tri + t] += (sg * ci[s]) * cj[s];
      }
    }
    __syncwarp();
  }
  if (shared_acc) {
    double *dst = part + warp * per;
    for (int64_t k = lane; k < per; k += 32) dst[k] = acc[k];
  }
}

// one block per (slot, view): thread k sums warps k, k + 256, ... in order, then a fixed tree; writes (p,q) and (q,p) of the
// packed triangle, or (full: tri = norb^2 slots) the one element (p,q) the slot holds
__global__ void __launch_bounds__(kRdmThreads) one_rdm_reduce_kernel(const double *part0, const double *part1, int nwarps, int S, int tri, int norb,
                                                                       int full, double *out) {
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
  const int sigma = blockIdx.y ? 0 : 1;  // view 0 is (up, dn) order: its minor string is beta
  double *m = out + ((int64_t)s * 2 + sigma) * norb * norb;
  if (full) {
    m[t] = red[0];
    return;
  }
  int p = 0;
  while ((p + 1) * (p + 2) / 2 <= t) p++;
  const int q = t - p * (p + 1) / 2;
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
// sel_out (time_sym, optional): the representatives whose partner (d,u) is expanded entry n + j, j < n2 - n.
template <int NW>
static int prepare_dets(sqmc_b200_handle *h, const char *who, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts,
                        int64_t ldw, DevBuf<uint64_t> &up, DevBuf<uint64_t> &dn, DevBuf<double> &w, int64_t &n2, DevBuf<int32_t> &idx0,
                        DevBuf<uint64_t> &ma0, DevBuf<uint64_t> &mi0, DevBuf<double> &c0, DevBuf<int32_t> *sel_out = nullptr) {
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
    if (sel_out) {
      sel_out->release();
      sel_out->n = sel.n;
      sel_out->p = sel.take();
    }
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

// TR: wts holds 2S columns, the bras a_k = column k and the kets b_k = column S + k (one_rdm_kernel's transition mode)
template <int NW, bool TR>
static int one_rdm_impl(sqmc_b200_handle *h, const char *who, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts,
                        int64_t ldw, double *rdm) {
  cudaStream_t s = G.stream;
  const int norb = h->T.norb;
  const int cs = TR ? 2 * S : S;
  // view 0: (up, dn) order, beta singles; view 1: (dn, up) order, alpha singles
  DevBuf<uint64_t> up, dn;
  DevBuf<double> w;
  int64_t n2 = 0;
  DevBuf<int32_t> idx0, idx1;
  DevBuf<uint64_t> ma0, mi0, ma1, mi1;
  DevBuf<double> c0, c1;
  SQ_CHECK(prepare_dets<NW>(h, who, n, dets_up, dets_dn, cs, wts, ldw, up, dn, w, n2, idx0, ma0, mi0, c0));
  SQ_CHECK(make_view<NW>(norb, dn.p, up.p, w.p, n2, cs, idx1, ma1, mi1, c1, s));
  up.release(); dn.release(); w.release(); idx0.release(); idx1.release();

  const int tri = TR ? norb * norb : norb * (norb + 1) / 2;
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
  auto kern = one_rdm_kernel<NW, TR>;
  const size_t dyn = shared_acc ? shmem : 0;
  SQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  RdmView v0{ma0.p, mi0.p, c0.p, part0.p}, v1{ma1.p, mi1.p, c1.p, part1.p};
  kern<<<dim3((unsigned)div_up(nwarps, wpb), 2), kRdmThreads, dyn, s>>>(v0, v1, n2, norb, S, tri, chunk, nwarps, shared_acc);
  SQ_LAUNCH_CHECK();
  one_rdm_reduce_kernel<<<dim3((unsigned)per, 2), kRdmThreads, 0, s>>>(part0.p, part1.p, nwarps, S, tri, norb, TR ? 1 : 0, out.p);
  SQ_LAUNCH_CHECK();
  SQ_CUDA(cudaMemcpyAsync(rdm, out.p, (size_t)S * 2 * norb * norb * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// argument checks both one-particle entry points share; count: "n_states" or "n_pairs"
static int rdm1_check_args(const char *who, const char *count, int64_t n, int S, int64_t ldw) {
  if (n <= 0) { set_error("%s: n must be positive", who); return 2; }
  if (S < 1) { set_error("%s: %s must be >= 1", who, count); return 2; }
  if (ldw < n) { set_error("%s: ldw (%lld) must be >= n (%lld)", who, (long long)ldw, (long long)n); return 2; }
  if (n > INT32_MAX) { set_error("%s: n exceeds the 32-bit row index", who); return 2; }
  return 0;
}

int one_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw, double *rdm) {
  SQ_CHECK(rdm1_check_args("one_rdm", "n_states", n, n_states, ldw));
  return h->NW == 1 ? one_rdm_impl<1, false>(h, "one_rdm", n, dets_up, dets_dn, n_states, wts, ldw, rdm)
                    : one_rdm_impl<2, false>(h, "one_rdm", n, dets_up, dets_dn, n_states, wts, ldw, rdm);
}

// [a_1 .. a_S | b_1 .. b_S], leading dimension n: the 2S-column layout of the transition modes
static std::vector<double> stack_columns(int64_t n, int S, const double *a, const double *b, int64_t ldw) {
  std::vector<double> ab((size_t)2 * S * n);
  for (int k = 0; k < S; k++) {
    memcpy(ab.data() + (size_t)k * n, a + k * ldw, n * sizeof(double));
    memcpy(ab.data() + (size_t)(S + k) * n, b + k * ldw, n * sizeof(double));
  }
  return ab;
}

int transition_one_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_pairs, const double *bra, const double *ket,
                       int64_t ldw, double *tdm) {
  SQ_CHECK(rdm1_check_args("transition_one_rdm", "n_pairs", n, n_pairs, ldw));
  const std::vector<double> ab = stack_columns(n, n_pairs, bra, ket, ldw);
  return h->NW == 1 ? one_rdm_impl<1, true>(h, "transition_one_rdm", n, dets_up, dets_dn, n_pairs, ab.data(), n, tdm)
                    : one_rdm_impl<2, true>(h, "transition_one_rdm", n, dets_up, dets_dn, n_pairs, ab.data(), n, tdm);
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
//
// Transition mode (sqmc_b200_transition_two_rdm): Gamma^{ab} = <a| ... |b> is not Hermitian, so Gamma_{pq,rs} = Gamma_{qp,sr}
// no longer holds and the two orientations of a representative are kept apart.  Each slot has two accumulators: F =
// <a| E_c |b> and B = <a| E_c^+ |b>, E_c the canonical orientation ss_slot / ab_slot pick (flip: they took the Hermitian image
// of the element asked for).  A pair (i, j) with f = <i| E |j> adds f a_i b_j to the orientation of E and f a_j b_i to the
// other one.  Diagonal terms a_i b_i fall only on self-adjoint slots (A = B, or p = q and r = s), where F = B; they go to F
// once and the fill reads F there.  The grid is set from ||a|| ||b||.  For a = b every term has the bits of its two_rdm
// counterpart, sqrt(fl(na na)) = na, and F = B = two_rdm's representative; T(b, a) holds in F what T(a, b) holds in B.
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
// representative of the same-spin element (p,q,r,s), p != r, q != s, inside an M x M block; sg: element = sg * representative;
// flip: the representative is the Hermitian image of the element (creator pair A > annihilator pair B)
__device__ __forceinline__ int64_t ss_slot(int p, int q, int r, int s, int M, int &sg, bool &flip) {
  sg = 1;
  if (p > r) { const int t = p; p = r; r = t; sg = -sg; }
  if (q > s) { const int t = q; q = s; s = t; sg = -sg; }
  const int64_t A = pair_index(p, r), B = pair_index(q, s);
  flip = A > B;
  return flip ? B + M * A : A + M * B;
}
__device__ __forceinline__ int64_t ss_slot(int p, int q, int r, int s, int M, int &sg) {
  bool flip;
  return ss_slot(p, q, r, s, M, sg, flip);
}
__device__ __forceinline__ int64_t ab_slot(int p, int q, int r, int s, int norb, bool &flip) {
  int64_t X = p + (int64_t)norb * q, Y = r + (int64_t)norb * s;
  const int64_t X2 = q + (int64_t)norb * p, Y2 = s + (int64_t)norb * r;
  flip = X2 < X || (X2 == X && Y2 < Y);
  if (flip) { X = X2; Y = Y2; }
  return X + (int64_t)norb * norb * Y;
}
__device__ __forceinline__ int64_t ab_slot(int p, int q, int r, int s, int norb) {
  bool flip;
  return ab_slot(p, q, r, s, norb, flip);
}

struct Rdm2Acc {
  unsigned long long *a;  // [S][per] slots of two words
  unsigned long long *b;  // transition mode: [S][per] accumulators of the Hermitian-image orientation B (a holds F); else null
  const double *scale;    // [S] 2^(120 - e_k)
  int64_t per, off_bb, off_ab;
  int M, norb, S;
  int cs;                 // coefficients per row: S, or 2S in the two-vector modes (a_k at k, b_k at S + k)
};

// rdm2_accumulate modes: one state, the symmetrised two-vector density (orbital-gradient response), the transition density
enum Rdm2Mode { RDM2_ONE = 0, RDM2_SYM = 1, RDM2_TRANS = 2 };

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

// The representative slot of the pair (i, j) of one bucket (entries ki / kdi / ai / bi of i and aj / bj of j) and the sign f
// of <i| operator |j> on it; boff: block offset of a same-spin class, -1: alpha beta; flip: the slot's canonical orientation
// is the Hermitian image of the <i| . |j> one, f = <j| E_c |i>
__device__ __forceinline__ int64_t rdm2_pair_slot(uint64_t ki, uint64_t kdi, int ai, int bi, int aj, int bj, int64_t boff, int M, int norb,
                                                  int64_t off_ab, double &f, bool &flip) {
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
    slot = boff + ss_slot(p, q, r, s, M, sg, flip);
  } else if (ai != aj && bi != bj) {
    neg = par_between(ki, ai, aj) ^ par_between(kdi, bi, bj);
    slot = off_ab + ab_slot(ai, aj, bi, bj, norb, flip);
  } else if (ai != aj) {
    neg = par_between(ki, ai, aj);
    slot = off_ab + ab_slot(ai, aj, bi, bi, norb, flip);
  } else {
    neg = par_between(kdi, bi, bj);
    slot = off_ab + ab_slot(ai, ai, bi, bj, norb, flip);
  }
  f = (neg ? -1.0 : 1.0) * sg;
  return slot;
}

// one thread per sorted entry i: every later entry j of the same bucket; boff: block offset of a same-spin class, -1: alpha beta.
// RDM2_ONE: the term f c_i c_j of each state; RDM2_SYM: the symmetrised transition term f (a_i b_j + b_i a_j) / 2; RDM2_TRANS:
// f a_i b_j to the orientation of <i| . |j> and f a_j b_i to the other one (F in R.a, B in R.b).
template <int MODE>
__global__ void __launch_bounds__(256) rdm2_pair_kernel(const uint64_t *ku, const uint64_t *kd, const uint64_t *pay, int64_t m, int64_t boff,
                                                        const double *coef, Rdm2Acc R) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const uint64_t ki = ku[i], kdi = kd[i], pi = pay[i];
  const int ai = (int)(pi & 0xff), bi = (int)((pi >> 8) & 0xff);
  const double *ci = coef + (int64_t)(pi >> 16) * R.cs;
  for (int64_t j = i + 1; j < m && ku[j] == ki && kd[j] == kdi; j++) {
    const uint64_t pj = pay[j];
    double f;
    bool flip;
    const int64_t slot = rdm2_pair_slot(ki, kdi, ai, bi, (int)(pj & 0xff), (int)((pj >> 8) & 0xff), boff, R.M, R.norb, R.off_ab, f, flip);
    const double *cj = coef + (int64_t)(pj >> 16) * R.cs;
    for (int k = 0; k < R.S; k++) {
      uint64_t lo, hi;
      if constexpr (MODE == RDM2_TRANS) {
        const double fw = f * (ci[k] * cj[R.S + k]), bw = f * (cj[k] * ci[R.S + k]);
        fix_to_i128((flip ? bw : fw) * R.scale[k], lo, hi);
        i128_add(R.a + 2 * (k * R.per + slot), lo, hi);
        fix_to_i128((flip ? fw : bw) * R.scale[k], lo, hi);
        i128_add(R.b + 2 * (k * R.per + slot), lo, hi);
      } else {
        if constexpr (MODE == RDM2_SYM) fix_to_i128(f * (0.5 * (ci[k] * cj[R.S + k] + ci[R.S + k] * cj[k])) * R.scale[k], lo, hi);
        else fix_to_i128(f * (ci[k] * cj[k]) * R.scale[k], lo, hi);
        i128_add(R.a + 2 * (k * R.per + slot), lo, hi);
      }
    }
  }
}

// diagonal terms c_i^2 (TWO: a_i b_i): Gamma^{ss}_{pp,rr} (p < r occupied in the same string) and Gamma^{ab}_{pp,rr}, one state
// at a time, summed per block in shared memory ([3][norb][norb] 128-bit values) and then added to the representatives
template <bool TWO>
__global__ void __launch_bounds__(256) rdm2_diag_kernel(const uint64_t *u, const uint64_t *d, int64_t n, const double *coef, Rdm2Acc R) {
  extern __shared__ unsigned long long sd[];
  const int norb = R.norb, nn = norb * norb;
  for (int k = 0; k < R.S; k++) {
    for (int t = threadIdx.x; t < 6 * nn; t += blockDim.x) sd[t] = 0ull;
    __syncthreads();
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
      const double c = coef[i * R.cs + k];
      uint64_t lo, hi;
      fix_to_i128((TWO ? c * coef[i * R.cs + R.S + k] : c * c) * R.scale[k], lo, hi);
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

// every element of the output (column-major p, q, r, s, block, state) from its representative; transition mode (R.b set):
// from F or B by the element's orientation (self-adjoint slots never flip and read F)
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
    bool flip;
    int64_t slot;
    if (b == 1) {
      slot = R.off_ab + ab_slot(p, q, r, s, norb, flip);
    } else if (p == r || q == s) {
      out[t] = 0.0;
      continue;
    } else {
      slot = (b ? R.off_bb : 0) + ss_slot(p, q, r, s, R.M, sg, flip);
    }
    const unsigned long long *v = (flip && R.b ? R.b : R.a) + 2 * (k * R.per + slot);
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

// every determinant of the sorted view holds T.nup alpha and T.ndn beta electrons
static int rdm2_electron_check(const ModelTables &T, const char *who, const uint64_t *U, const uint64_t *D, int64_t n2, cudaStream_t s) {
  DevBuf<int> bad;
  SQ_CHECK(bad.alloc(1));
  SQ_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), s));
  electron_count_kernel<<<(unsigned)div_up(n2, 256), 256, 0, s>>>(U, D, n2, T.nup, T.ndn, bad.p);
  SQ_LAUNCH_CHECK();
  int hb = 0;
  SQ_CUDA(cudaMemcpyAsync(&hb, bad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  if (hb) { set_error("%s: a determinant does not hold %d alpha and %d beta electrons", who, T.nup, T.ndn); return 2; }
  return 0;
}

// per state k over the sorted view (two-vector layout, 2S coefficients per row): out[k] = sum_i a_ik^2, out[S + k] =
// sum_i a_ik b_ik; thread t sums rows t, t + 256, ... in order, then a fixed tree
__global__ void __launch_bounds__(256) dots_kernel(const double *c, int64_t n, int S, double *out) {
  __shared__ double red[2][256];
  const int k = blockIdx.x;
  double aa = 0.0, ab = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += 256) {
    const double a = c[i * 2 * S + k];
    aa += a * a;
    ab += a * c[i * 2 * S + S + k];
  }
  red[0][threadIdx.x] = aa;
  red[1][threadIdx.x] = ab;
  __syncthreads();
  for (int hh = 128; hh > 0; hh >>= 1) {
    if (threadIdx.x < hh) {
      red[0][threadIdx.x] += red[0][threadIdx.x + hh];
      red[1][threadIdx.x] += red[1][threadIdx.x + hh];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[k] = red[0][0];
    out[S + k] = red[1][0];
  }
}

// b_k -= (<a_k|b_k> / ||a_k||^2) a_k: the change of a_k along itself only rescales it and leaves the normalised densities alone
__global__ void project_out_kernel(double *c, int64_t n, int S, const double *dots) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n * S) return;
  const int64_t i = t / S;
  const int k = (int)(t % S);
  const double aa = dots[k];
  if (aa > 0.0) c[i * 2 * S + S + k] -= (dots[S + k] / aa) * c[i * 2 * S + k];
}

// The pair enumeration the two-particle entry points share: the three hole-key classes of the sorted view (U, D: n2 one-word
// strings), each sorted by key; visit(sku, skd, spay, m, boff) is called once per class with the sorted keys and payloads
// (boff: block offset of a same-spin class, -1: alpha beta).
template <class Visit>
static int rdm2_for_each_class(const ModelTables &T, const char *who, const uint64_t *U, const uint64_t *D, int64_t n2, const Rdm2Acc &R,
                               HostMarks &marks, Visit visit) {
  cudaStream_t s = G.stream;
  const int norb = T.norb;
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
    if (cls == 2) rdm2_keys_ab_kernel<<<(unsigned)div_up(n2, 256), 256, 0, s>>>(U, D, n2, K, ku.p, kd.p, pay.p);
    else rdm2_keys_same_kernel<<<(unsigned)div_up(n2, 256), 256, 0, s>>>(cls ? D : U, cls ? U : D, n2, K, ku.p, kd.p, pay.p);
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
    SQ_CHECK(visit(sku.p, skd.p, spay.p, m, cls == 2 ? (int64_t)-1 : cls == 0 ? (int64_t)0 : R.off_bb));
    marks.mark(cls == 0 ? "alpha alpha pairs" : cls == 1 ? "beta beta pairs" : "alpha beta pairs");
  }
  return 0;
}

// slot layout of the representatives (aa, bb, ab) for norb orbitals and S states
static void rdm2_layout(Rdm2Acc &R, int norb, int S) {
  const int M = norb * (norb - 1) / 2;
  R.M = M; R.norb = norb; R.S = S; R.cs = S;
  R.b = nullptr;
  R.off_bb = (int64_t)M * M;
  R.off_ab = 2 * R.off_bb;
  R.per = R.off_ab + (int64_t)norb * norb * norb * norb;
}

// The accumulation both two-particle entry points share: upload, time_sym expansion, checks, the diagonal and the three key
// classes with their pairs.  On return acc / scale hold the representatives of R (scale[S + k]: the factor back to doubles);
// norm2 (device, S doubles, may be null) receives ||Psi_k||^2 summed in a fixed order.
// mode RDM2_SYM: wts holds 2S columns, a_k = column k and b_k = column S + k; b_k is first made orthogonal to a_k on the device,
// and the representatives are those of the symmetrised transition density (<a_k| E |b_k> + <b_k| E |a_k>) / 2, on a grid from
// ||a_k|| ||b_k|| (Cauchy-Schwarz again); norm2 receives ||a_k||^2.
// mode RDM2_TRANS: the same 2S columns, no projection; R.a / R.b hold F = <a_k| E_c |b_k> and B = <a_k| E_c^+ |b_k> on the grid
// from ||a_k|| ||b_k||; norm2 must be null.
static int rdm2_accumulate(sqmc_b200_handle *h, const char *who, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts,
                           int64_t ldw, HostMarks &marks, DevBuf<unsigned long long> &acc, DevBuf<double> &scale, Rdm2Acc &R, double *norm2,
                           int mode = RDM2_ONE) {
  const bool two = mode != RDM2_ONE;
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  const int norb = T.norb;
  DevBuf<uint64_t> up, dn, U, D;
  DevBuf<double> w, c;
  DevBuf<int32_t> idx0;
  int64_t n2 = 0;
  SQ_CHECK(prepare_dets<1>(h, who, n, dets_up, dets_dn, two ? 2 * S : S, wts, ldw, up, dn, w, n2, idx0, U, D, c));
  up.release(); dn.release(); w.release(); idx0.release();
  marks.mark("upload, expansion, checks");
  SQ_CHECK(rdm2_electron_check(T, who, U.p, D.p, n2, s));
  if (mode == RDM2_SYM) {
    DevBuf<double> dots;
    SQ_CHECK(dots.alloc(2 * S));
    dots_kernel<<<S, 256, 0, s>>>(c.p, n2, S, dots.p);
    SQ_LAUNCH_CHECK();
    project_out_kernel<<<(unsigned)div_up(n2 * S, 256), 256, 0, s>>>(c.p, n2, S, dots.p);
    SQ_LAUNCH_CHECK();
    if (norm2) SQ_CUDA(cudaMemcpyAsync(norm2, dots.p, S * sizeof(double), cudaMemcpyDeviceToDevice, s));
  } else if (norm2) {
    norm2_kernel<<<S, 256, 0, s>>>(c.p, n2, S, norm2);
    SQ_LAUNCH_CHECK();
  }
  // grid exponent per state from sum_i w_ik^2 (the time_sym expansion keeps it); the margin keeps e_k the same whatever order
  // the sum was taken in, unless the norm lies within a few ulps of 2^e / (1 + 2^-20)
  std::vector<double> hs(2 * S);
  for (int k = 0; k < S; k++) {
    double n2k = 0.0;
    if (two) {
      double na = 0.0, nb = 0.0;
      for (int64_t i = 0; i < n; i++) na += wts[k * ldw + i] * wts[k * ldw + i];
      for (int64_t i = 0; i < n; i++) nb += wts[(S + k) * ldw + i] * wts[(S + k) * ldw + i];
      n2k = sqrt(na * nb);
    } else {
      for (int64_t i = 0; i < n; i++) n2k += wts[k * ldw + i] * wts[k * ldw + i];
    }
    int e = 0;
    if (n2k > 0.0) frexp(n2k * (1.0 + 0x1p-20), &e);
    hs[k] = ldexp(1.0, kFixBits - e);
    hs[S + k] = ldexp(1.0, e - kFixBits);
  }
  rdm2_layout(R, norb, S);
  if (two) R.cs = 2 * S;
  const int nacc = mode == RDM2_TRANS ? 2 : 1;  // F, and B in the transition mode
  SQ_CHECK(acc.alloc(2 * nacc * S * R.per));
  SQ_CHECK(scale.alloc(2 * S));
  SQ_CUDA(cudaMemsetAsync(acc.p, 0, (size_t)acc.n * sizeof(unsigned long long), s));
  SQ_CUDA(cudaMemcpyAsync(scale.p, hs.data(), 2 * S * sizeof(double), cudaMemcpyHostToDevice, s));
  R.a = acc.p;
  R.b = mode == RDM2_TRANS ? acc.p + 2 * S * R.per : nullptr;
  R.scale = scale.p;

  const size_t dsh = (size_t)6 * norb * norb * sizeof(unsigned long long);
  auto diag = two ? rdm2_diag_kernel<true> : rdm2_diag_kernel<false>;
  SQ_CUDA(cudaFuncSetAttribute(diag, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsh));
  diag<<<(unsigned)std::min<int64_t>(div_up(n2, 256), 2 * G.sm_count), 256, dsh, s>>>(U.p, D.p, n2, c.p, R);
  SQ_LAUNCH_CHECK();
  marks.mark("diagonal");

  const Rdm2Acc Rc = R;
  const double *cp = c.p;
  return rdm2_for_each_class(T, who, U.p, D.p, n2, R, marks, [&](const uint64_t *sku, const uint64_t *skd, const uint64_t *spay, int64_t m, int64_t boff) {
    if (mode == RDM2_TRANS) rdm2_pair_kernel<RDM2_TRANS><<<(unsigned)div_up(m, 256), 256, 0, s>>>(sku, skd, spay, m, boff, cp, Rc);
    else if (two) rdm2_pair_kernel<RDM2_SYM><<<(unsigned)div_up(m, 256), 256, 0, s>>>(sku, skd, spay, m, boff, cp, Rc);
    else rdm2_pair_kernel<RDM2_ONE><<<(unsigned)div_up(m, 256), 256, 0, s>>>(sku, skd, spay, m, boff, cp, Rc);
    SQ_LAUNCH_CHECK();
    return 0;
  });
}

// mode RDM2_ONE (two_rdm) or RDM2_TRANS (transition_two_rdm: wts holds the 2S columns [bras | kets])
static int two_rdm_impl(sqmc_b200_handle *h, const char *who, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts,
                        int64_t ldw, double *rdm, int mode) {
  cudaStream_t s = G.stream;
  const int norb = h->T.norb;
  HostMarks marks("SQMC_RDM2_PROFILE", who);  // =1: phase split (synchronising) on stderr
  DevBuf<unsigned long long> acc;
  DevBuf<double> scale;
  Rdm2Acc R;
  SQ_CHECK(rdm2_accumulate(h, who, n, dets_up, dets_dn, S, wts, ldw, marks, acc, scale, R, nullptr, mode));
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

// argument checks the two-particle entry points share; count: the name of n_states in the caller's interface
static int rdm2_check_args(sqmc_b200_handle *h, const char *who, int64_t n, int n_states, int64_t ldw, const char *count = "n_states") {
  if (n <= 0) { set_error("%s: n must be positive", who); return 2; }
  if (n_states < 1) { set_error("%s: %s must be >= 1", who, count); return 2; }
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
  return two_rdm_impl(h, "two_rdm", n, dets_up, dets_dn, n_states, wts, ldw, rdm, RDM2_ONE);
}

int transition_two_rdm(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_pairs, const double *bra, const double *ket,
                       int64_t ldw, double *tdm2) {
  SQ_CHECK(rdm2_check_args(h, "transition_two_rdm", n, n_pairs, ldw, "n_pairs"));
  const std::vector<double> ab = stack_columns(n, n_pairs, bra, ket, ldw);
  return two_rdm_impl(h, "transition_two_rdm", n, dets_up, dets_dn, n_pairs, ab.data(), n, tdm2, RDM2_TRANS);
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

// argument checks of the entry points that work on the orbitals of a chem handle
static int orbital_check_args(sqmc_b200_handle *h, const char *who, int64_t n, int n_states, int64_t ldw) {
  if (h->T.model != MODEL_CHEM) {
    set_error("%s: only chem handles have orbitals to optimise (heg and hubbardk orbitals are fixed by momentum)", who);
    return 2;
  }
  SQ_CHECK(rdm2_check_args(h, who, n, n_states, ldw));
  if (h->T.nup + h->T.ndn < 2) { set_error("%s: needs at least two electrons", who); return 2; }
  return 0;
}

static int state_weights_check(const char *who, int n_states, const double *state_weights) {
  double sum = 0.0;
  for (int k = 0; k < n_states; k++) {
    if (!(state_weights[k] >= 0.0)) { set_error("%s: state_weights[%d] = %g is negative", who, k, state_weights[k]); return 2; }
    sum += state_weights[k];
  }
  if (!(fabs(sum - 1.0) <= 1e-12)) { set_error("%s: state_weights sum to %.17g, not 1", who, sum); return 2; }
  return 0;
}

int orbital_derivatives(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw,
                        const double *state_weights, double *fock, double *hessian, double *energy) {
  SQ_CHECK(orbital_check_args(h, "orbital_derivatives", n, n_states, ldw));
  SQ_CHECK(state_weights_check("orbital_derivatives", n_states, state_weights));
  return orbital_derivatives_impl(h, n, dets_up, dets_dn, n_states, wts, ldw, state_weights, fock, hessian, energy);
}

// ---------------------------------------------------------------------------------------------------------------------
// sigma-vector y = H x over a determinant list (sqmc_b200_sigma), chem, norb <= 64
//
// The two-body contraction of rdm_energy, E(c) = E_core ||c||^2 + 1/2 sum g'_pqrs d_pqrs with the one-body part folded into
//   g'_pqrs = g_pqrs + (h_pq delta_rs + delta_pq h_rs) / (N - 1)        (sum_r d_pqrr = (N - 1) gamma_pq),
// is a sum over the representatives of two_rdm, E = E_core ||c||^2 + sum_slot G[slot] rep[slot], G[slot] = dE / drep[slot]
// (sigma_table_kernel: same spin (g'_pqrs - g'_psrq) x (2 if A != B), alpha beta g'_pqrs x (1 if p = q and r = s, else 2)).
// rep is quadratic in c: each pair visit of rdm2_for_each_class adds f c_i c_j, each determinant's diagonal slots c_i^2.  So
// H x = 1/2 grad E(x): a visit adds f G[slot] x_j / 2 to y_i and f G[slot] x_i / 2 to y_j (a single is met once per spectator
// orbital and each visit adds its own share), the diagonal adds x_i sum G over the determinant's diagonal slots.  Every pair of
// the list connected by a single or double excitation is visited, whatever its matrix element: no stored pattern is used.
// With kappa, h and g are replaced by their derivatives along the rotation U(t) = expm(-t kappa) (rotate_fcidump's rule):
//   h^k = kappa h - h kappa,   g^k_pqrs = sum_m (k_pm g_mqrs + k_qm g_pmrs + k_rm g_pqms + k_sm g_pqrm),
// and the core term is left out.  g^k is one FP64 product T1(p; x y z) = sum_m k_pm g_mxyz (orb_gemm_kernel, O(norb^5)) and
// its four index placements.
//
// Determinism: y is accumulated per (row of the sorted view, state) as a 128-bit fixed-point integer in units of 2^(e_k - 120),
// 2^e_k > B_k = max|G| max|x_k| (n_diag + V / 2): n_diag diagonal slots per determinant, and at most V = (N - 1) x
// min(n2 - 1, singles + doubles of one determinant) visits per row (a single is met N - 1 times, a double once).  B_k bounds
// every partial sum of a row, so the integers stay below 2^120, and integer addition does not depend on the order of the
// atomics: repeated calls and row permutations give the same bits.  time_sym lists are expanded as for two_rdm and y is folded
// back onto the representatives, (y_(u,d) + z y_(d,u)) / sqrt2 and y_(u,u) as it is.

// T1(i; x y z) = C[i + norb (z + norb (y + norb x))] (the product of kappa with g read as B(j, m) = g_{j, m}); g^k and h^k
__global__ void sigma_kappa_ints_kernel(const double *kap, const double *hd, const double *T1, int norb, double *hk, double *gk) {
  const int64_t n = norb, nn = n * n, n4 = nn * nn;
  auto t1 = [&](int64_t i, int64_t x, int64_t y, int64_t z) { return T1[i + n * (z + n * (y + n * x))]; };
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n4 + nn; t += (int64_t)gridDim.x * blockDim.x) {
    if (t < n4) {
      int64_t x = t;
      const int64_t p = x % n; x /= n;
      const int64_t q = x % n; x /= n;
      const int64_t r = x % n;
      const int64_t s = x / n;
      gk[t] = (t1(p, q, r, s) + t1(q, p, r, s)) + (t1(r, s, p, q) + t1(s, r, p, q));  // symmetric under p<->q, r<->s, pq<->rs
    } else {
      const int64_t u = t - n4, p = u % n, q = u / n;
      double a = 0.0, b = 0.0;
      for (int64_t m = 0; m < n; m++) {
        a += kap[p + n * m] * hd[m + n * q];
        b += hd[p + n * m] * kap[m + n * q];
      }
      hk[u] = a - b;
    }
  }
}

// G[slot] = dE / drep[slot] for every representative slot of R's layout (slots no pair reaches get values nobody reads)
__global__ void sigma_table_kernel(const double *hd, const double *gd, Rdm2Acc R, double inv_nm1, double *G) {
  const int64_t n = R.norb, nn = n * n, M = R.M;
  auto gp = [&](int64_t p, int64_t q, int64_t r, int64_t s) {
    double a = gd[p + n * (q + n * (r + n * s))];
    double one = 0.0;
    if (r == s) one += hd[p + n * q];
    if (p == q) one += hd[r + n * s];
    return a + one * inv_nm1;
  };
  auto unpair = [](int64_t A, int64_t &p, int64_t &r) {  // A = r (r - 1) / 2 + p, p < r
    r = (int64_t)((1.0 + sqrt(1.0 + 8.0 * (double)A)) * 0.5);
    while (r * (r - 1) / 2 > A) r--;
    while ((r + 1) * r / 2 <= A) r++;
    p = A - r * (r - 1) / 2;
  };
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < R.per; t += (int64_t)gridDim.x * blockDim.x) {
    double v;
    if (t < R.off_ab) {
      const int64_t u = t < R.off_bb ? t : t - R.off_bb;
      const int64_t A = u % M, B = u / M;
      if (A > B) {
        v = 0.0;
      } else {
        int64_t p, q, r, s;
        unpair(A, p, r);
        unpair(B, q, s);
        v = (gp(p, q, r, s) - gp(p, s, r, q)) * (A != B ? 2.0 : 1.0);
      }
    } else {
      const int64_t u = t - R.off_ab, X = u % nn, Y = u / nn;
      const int64_t p = X % n, q = X / n, r = Y % n, s = Y / n;
      v = gp(p, q, r, s) * ((p == q && r == s) ? 1.0 : 2.0);
    }
    G[t] = v;
  }
}

// *out = max |a| (the bit patterns of non-negative doubles order as the values: an integer max, independent of order)
__global__ void absmax_kernel(const double *a, int64_t n, unsigned long long *out) {
  unsigned long long m = 0ull;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
    m = max(m, (unsigned long long)__double_as_longlong(fabs(a[t])));
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// y of row i starts at x_i times the sum of G over its diagonal slots (summed in bit order), stored, not added
__global__ void sigma_diag_kernel(const uint64_t *u, const uint64_t *d, int64_t n, const double *x, const double *G, Rdm2Acc R,
                                  const double *scale, unsigned long long *Y) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t U = u[i], D = d[i];
  double a = 0.0;
  for (uint64_t ps = U; ps; ps &= ps - 1) {
    const int p = __ffsll((long long)ps) - 1;
    for (uint64_t rs = ps & (ps - 1); rs; rs &= rs - 1) a += G[(int64_t)pair_index(p, __ffsll((long long)rs) - 1) * (1 + R.M)];
    for (uint64_t rs = D; rs; rs &= rs - 1) {
      const int r = __ffsll((long long)rs) - 1;
      a += G[R.off_ab + ab_slot(p, p, r, r, R.norb)];
    }
  }
  for (uint64_t ps = D; ps; ps &= ps - 1) {
    const int p = __ffsll((long long)ps) - 1;
    for (uint64_t rs = ps & (ps - 1); rs; rs &= rs - 1) a += G[R.off_bb + (int64_t)pair_index(p, __ffsll((long long)rs) - 1) * (1 + R.M)];
  }
  for (int k = 0; k < R.S; k++) {
    uint64_t lo, hi;
    fix_to_i128(a * x[i * R.S + k] * scale[k], lo, hi);
    Y[2 * (i * R.S + k)] = lo;
    Y[2 * (i * R.S + k) + 1] = hi;
  }
}

// one thread per sorted entry i, every later entry j of its bucket: f G[slot] / 2 times x_j into y_i and times x_i into y_j
__global__ void __launch_bounds__(256) sigma_pair_kernel(const uint64_t *ku, const uint64_t *kd, const uint64_t *pay, int64_t m, int64_t boff,
                                                         const double *x, const double *G, Rdm2Acc R, const double *scale,
                                                         unsigned long long *Y) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const uint64_t ki = ku[i], kdi = kd[i], pi = pay[i];
  const int ai = (int)(pi & 0xff), bi = (int)((pi >> 8) & 0xff);
  const int64_t ri = (int64_t)(pi >> 16);
  const double *xi = x + ri * R.S;
  for (int64_t j = i + 1; j < m && ku[j] == ki && kd[j] == kdi; j++) {
    const uint64_t pj = pay[j];
    double f;
    bool flip;
    const int64_t slot = rdm2_pair_slot(ki, kdi, ai, bi, (int)(pj & 0xff), (int)((pj >> 8) & 0xff), boff, R.M, R.norb, R.off_ab, f, flip);
    const double gs = 0.5 * f * G[slot];
    if (gs == 0.0) continue;
    const int64_t rj = (int64_t)(pj >> 16);
    const double *xj = x + rj * R.S;
    for (int k = 0; k < R.S; k++) {
      uint64_t lo, hi;
      fix_to_i128(gs * xj[k] * scale[k], lo, hi);
      i128_add(Y + 2 * (ri * R.S + k), lo, hi);
      fix_to_i128(gs * xi[k] * scale[k], lo, hi);
      i128_add(Y + 2 * (rj * R.S + k), lo, hi);
    }
  }
}

// y back to doubles, plus the core term, scattered from the sorted view to the expanded order (column-major n2 x S)
__global__ void sigma_finish_kernel(const unsigned long long *Y, const double *x, const int32_t *idx, int64_t n2, int S, const double *unscale,
                                    double ecore, double *ye) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n2 * S) return;
  const int64_t v = t / S;
  const int k = (int)(t % S);
  const double a = (ldexp((double)(long long)Y[2 * t + 1], 64) + (double)Y[2 * t]) * unscale[k];
  ye[k * n2 + idx[v]] = a + ecore * x[t];
}

__global__ void partner_index_kernel(const int32_t *sel, int64_t m, int64_t n, int32_t *partner) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j < m) partner[sel[j]] = (int32_t)(n + j);
}

// time_sym: y of each representative from its plain determinants, (y_(u,d) + z y_(d,u)) / sqrt2, or y_(u,u)
__global__ void ts_fold_kernel(const double *ye, int64_t n, int64_t n2, int S, const int32_t *partner, double z, double r, double *y) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n * S) return;
  const int64_t i = t % n, k = t / n;
  const double a = ye[k * n2 + i];
  y[t] = partner[i] < 0 ? a : (a + z * ye[k * n2 + partner[i]]) * r;
}

// dense h and g from the handle's table, or their kappa derivatives (kappa: host, norb^2, kappa_pq at p + norb q)
static int orbital_integrals(sqmc_b200_handle *h, const double *kappa, DevBuf<double> &hd, DevBuf<double> &gd, cudaStream_t s) {
  const ModelTables &T = h->T;
  const int norb = T.norb;
  const int64_t nn = (int64_t)norb * norb, n4 = nn * nn;
  SQ_CHECK(hd.alloc(nn));
  SQ_CHECK(gd.alloc(n4));
  orbd_integrals_kernel<<<(unsigned)std::min<int64_t>(div_up(n4 + nn, 256), 64 * G.sm_count), 256, 0, s>>>(T.integrals, T.combine_2, norb, hd.p, gd.p);
  SQ_LAUNCH_CHECK();
  if (!kappa) return 0;
  DevBuf<double> kap, T1, hk, gk;
  SQ_CHECK(kap.alloc(nn));
  SQ_CUDA(cudaMemcpyAsync(kap.p, kappa, nn * sizeof(double), cudaMemcpyHostToDevice, s));
  SQ_CHECK(T1.alloc(n4));
  SQ_CHECK(orb_gemm(GemmSeg{kap.p, gd.p, norb}, GemmSeg{nullptr, nullptr, 0}, norb, (int)(nn * norb), T1.p, s));
  SQ_CHECK(hk.alloc(nn));
  SQ_CHECK(gk.alloc(n4));
  sigma_kappa_ints_kernel<<<(unsigned)std::min<int64_t>(div_up(n4 + nn, 256), 64 * G.sm_count), 256, 0, s>>>(kap.p, hd.p, T1.p, norb, hk.p, gk.p);
  SQ_LAUNCH_CHECK();
  hd.release(); gd.release();
  hd.n = nn; hd.p = hk.take();
  gd.n = n4; gd.p = gk.take();
  return 0;
}

static int sigma_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *x, int64_t ldx,
                      const double *kappa, double *y) {
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  const int norb = T.norb;
  const bool ts = T.time_sym;
  HostMarks marks("SQMC_SIGMA_PROFILE", "sigma");  // =1: phase split (synchronising) on stderr
  DevBuf<uint64_t> up, dn, U, D;
  DevBuf<double> w, c;
  DevBuf<int32_t> idx0, sel;
  int64_t n2 = 0;
  SQ_CHECK(prepare_dets<1>(h, "sigma", n, dets_up, dets_dn, S, x, ldx, up, dn, w, n2, idx0, U, D, c, &sel));
  up.release(); dn.release(); w.release();
  marks.mark("upload, expansion, checks");
  SQ_CHECK(rdm2_electron_check(T, "sigma", U.p, D.p, n2, s));

  Rdm2Acc R;
  rdm2_layout(R, norb, S);
  DevBuf<double> Gt, scale;
  DevBuf<unsigned long long> gmax;
  {
    DevBuf<double> hd, gd;
    SQ_CHECK(orbital_integrals(h, kappa, hd, gd, s));
    SQ_CHECK(Gt.alloc(R.per));
    sigma_table_kernel<<<(unsigned)std::min<int64_t>(div_up(R.per, 256), 64 * G.sm_count), 256, 0, s>>>(hd.p, gd.p, R, 1.0 / (T.nup + T.ndn - 1), Gt.p);
    SQ_LAUNCH_CHECK();
  }
  SQ_CHECK(gmax.alloc(1));
  SQ_CUDA(cudaMemsetAsync(gmax.p, 0, sizeof(unsigned long long), s));
  absmax_kernel<<<(unsigned)std::min<int64_t>(div_up(R.per, 256), 8 * G.sm_count), 256, 0, s>>>(Gt.p, R.per, gmax.p);
  SQ_LAUNCH_CHECK();
  unsigned long long gbits = 0;
  SQ_CUDA(cudaMemcpyAsync(&gbits, gmax.p, sizeof(gbits), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  double gm;
  memcpy(&gm, &gbits, sizeof(gm));
  marks.mark("integrals, G table");

  // the grid exponent per state (see above); every input of the bound is independent of the row order
  const double na = T.nup, nb = T.ndn, no = norb;
  const double ndiag = na * (na - 1) / 2 + nb * (nb - 1) / 2 + na * nb;
  const double sa = na * (no - na), sb = nb * (no - nb);
  const double nexc = sa + sb + (na * (na - 1) / 2) * ((no - na) * (no - na - 1) / 2) + (nb * (nb - 1) / 2) * ((no - nb) * (no - nb - 1) / 2) + sa * sb;
  const double visits = (na + nb - 1) * std::min((double)(n2 - 1), nexc);
  std::vector<double> hs(2 * S);
  for (int k = 0; k < S; k++) {
    double xm = 0.0;
    for (int64_t i = 0; i < n; i++) xm = std::max(xm, fabs(x[k * ldx + i]));
    const double B = gm * xm * (ndiag + 0.5 * visits);
    int e = 0;
    if (B > 0.0) frexp(B, &e);
    hs[k] = ldexp(1.0, kFixBits - e);
    hs[S + k] = ldexp(1.0, e - kFixBits);
  }
  SQ_CHECK(scale.alloc(2 * S));
  SQ_CUDA(cudaMemcpyAsync(scale.p, hs.data(), 2 * S * sizeof(double), cudaMemcpyHostToDevice, s));

  DevBuf<unsigned long long> Y;
  SQ_CHECK(Y.alloc(2 * n2 * S));
  sigma_diag_kernel<<<(unsigned)div_up(n2, 256), 256, 0, s>>>(U.p, D.p, n2, c.p, Gt.p, R, scale.p, Y.p);
  SQ_LAUNCH_CHECK();
  marks.mark("diagonal");
  const double *cp = c.p, *gp = Gt.p, *sp = scale.p;
  unsigned long long *yp = Y.p;
  SQ_CHECK(rdm2_for_each_class(T, "sigma", U.p, D.p, n2, R, marks, [&](const uint64_t *sku, const uint64_t *skd, const uint64_t *spay, int64_t m, int64_t boff) {
    sigma_pair_kernel<<<(unsigned)div_up(m, 256), 256, 0, s>>>(sku, skd, spay, m, boff, cp, gp, R, sp, yp);
    SQ_LAUNCH_CHECK();
    return 0;
  }));

  DevBuf<double> ye, yo;
  SQ_CHECK(ye.alloc(n2 * S));
  sigma_finish_kernel<<<(unsigned)div_up(n2 * S, 256), 256, 0, s>>>(Y.p, c.p, idx0.p, n2, S, scale.p + S, kappa ? 0.0 : T.enuc, ye.p);
  SQ_LAUNCH_CHECK();
  const double *out = ye.p;
  if (ts) {
    DevBuf<int32_t> partner;
    SQ_CHECK(partner.alloc(n));
    SQ_CUDA(cudaMemsetAsync(partner.p, 0xff, n * sizeof(int32_t), s));  // -1: no partner
    if (n2 > n) {
      partner_index_kernel<<<(unsigned)div_up(n2 - n, 256), 256, 0, s>>>(sel.p, n2 - n, n, partner.p);
      SQ_LAUNCH_CHECK();
    }
    SQ_CHECK(yo.alloc(n * S));
    ts_fold_kernel<<<(unsigned)div_up(n * S, 256), 256, 0, s>>>(ye.p, n, n2, S, partner.p, T.z, T.sqrt2inv, yo.p);
    SQ_LAUNCH_CHECK();
    out = yo.p;
  }
  SQ_CUDA(cudaMemcpyAsync(y, out, (size_t)n * S * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  marks.mark("fold + copy out");
  return 0;
}

int sigma(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *x, int64_t ldx,
          const double *kappa, double *y) {
  SQ_CHECK(orbital_check_args(h, "sigma", n, n_states, ldx));
  if (kappa) {
    const int norb = h->T.norb;
    for (int p = 0; p < norb; p++)
      for (int q = 0; q <= p; q++)
        if (kappa[p + norb * q] != -kappa[q + norb * p]) {
          set_error("sigma: kappa is not antisymmetric (kappa[%d,%d] = %g, kappa[%d,%d] = %g)", p, q, kappa[p + norb * q], q, p, kappa[q + norb * p]);
          return 2;
        }
  }
  return sigma_impl(h, n, dets_up, dets_dn, n_states, x, ldx, kappa, y);
}

// ---------------------------------------------------------------------------------------------------------------------
// orbital-gradient response (sqmc_b200_orbital_gradient_response): d/dt of the orbital gradient 2 (F - F^T) of
// orbital_derivatives at the vectors c_k + t dc_k, t = 0.  F is linear in the state-averaged normalised densities, and
//   d/dt [w_k d(c_k + t dc_k) / ||c_k + t dc_k||^2] = (2 w_k / ||c_k||^2) T(c_k, dc_k')
// with T the symmetrised transition density and dc_k' = dc_k - (<c_k|dc_k> / ||c_k||^2) c_k (the normalisation term).  So the
// two-vector mode of rdm2_accumulate gives the representatives of T(c_k, dc_k'), orbd_fill_kernel the spin-summed d with the
// factors 2 w_k / ||c_k||^2, and one F product (no Y term) the response 2 (F - F^T).
static int orbital_gradient_response_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int S, const double *wts,
                                          const double *dwts, int64_t ldw, const double *state_weights, double *response) {
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  const int norb = T.norb;
  const int64_t nn = (int64_t)norb * norb, n4 = nn * nn;
  HostMarks marks("SQMC_ORBD_PROFILE", "orbital_gradient_response");  // =1: phase split (synchronising) on stderr
  const std::vector<double> ab = stack_columns(n, S, wts, dwts, ldw);  // [c_1 .. c_S | dc_1 .. dc_S]
  std::vector<double> w2(S);
  for (int k = 0; k < S; k++) w2[k] = 2.0 * state_weights[k];
  DevBuf<double> norm2, sw, d, D;
  SQ_CHECK(norm2.alloc(S));
  SQ_CHECK(sw.alloc(S));
  SQ_CUDA(cudaMemcpyAsync(sw.p, w2.data(), S * sizeof(double), cudaMemcpyHostToDevice, s));
  {
    DevBuf<unsigned long long> acc;
    DevBuf<double> scale;
    Rdm2Acc R;
    SQ_CHECK(rdm2_accumulate(h, "orbital_gradient_response", n, dets_up, dets_dn, S, ab.data(), n, marks, acc, scale, R, norm2.p, RDM2_SYM));
    SQ_CHECK(d.alloc(n4));
    orbd_fill_kernel<<<(unsigned)std::min<int64_t>(div_up(n4, 256), 64 * G.sm_count), 256, 0, s>>>(R, scale.p + S, sw.p, norm2.p, d.p);
    SQ_LAUNCH_CHECK();
  }
  SQ_CHECK(D.alloc(nn));
  orbd_trace_kernel<<<(unsigned)div_up(nn, 256), 256, 0, s>>>(d.p, norb, 1.0 / (T.nup + T.ndn - 1), D.p);
  SQ_LAUNCH_CHECK();
  DevBuf<double> hd, gd, F;
  SQ_CHECK(orbital_integrals(h, nullptr, hd, gd, s));
  SQ_CHECK(F.alloc(nn));
  SQ_CHECK(orb_gemm(GemmSeg{D.p, hd.p, norb}, GemmSeg{d.p, gd.p, nn * norb}, norb, norb, F.p, s));
  std::vector<double> Fh(nn);
  SQ_CUDA(cudaMemcpyAsync(Fh.data(), F.p, nn * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  marks.mark("d, F, copy out");
  for (int q = 0; q < norb; q++)
    for (int p = 0; p < norb; p++) response[p + (int64_t)norb * q] = 2.0 * (Fh[p + norb * q] - Fh[q + norb * p]);
  return 0;
}

int orbital_gradient_response(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts,
                              const double *dwts, int64_t ldw, const double *state_weights, double *response) {
  SQ_CHECK(orbital_check_args(h, "orbital_gradient_response", n, n_states, ldw));
  SQ_CHECK(state_weights_check("orbital_gradient_response", n_states, state_weights));
  return orbital_gradient_response_impl(h, n, dets_up, dets_dn, n_states, wts, dwts, ldw, state_weights, response);
}

// ---------------------------------------------------------------------------------------------------------------------
// ladder images (sqmc_b200_ladder / sqmc_b200_ladder_result): a_{p sigma}|Psi> or a+_{p sigma}|Psi> for every p of a list
//
// Determinant phase convention: the alpha string first, each string with ascending creators (chem_single,
// permutation_factor, one_rdm).  a_{p alpha} and a+_{p alpha} carry (-1)^(alpha electrons below p); the beta operators carry
// (-1)^(N_alpha + beta electrons below p).
//
// Every determinant of the sorted view 0 of prepare_dets (time_sym lists expanded) emits one candidate per orbital into slot
// i * P + j.  For a fixed orbital the map D -> a_p D is injective, so a column never receives two values; the same image
// reached from several orbitals is one row of the union.  The valid candidates are compacted in slot order, sorted by
// (up, dn) with the stable radix sort of sort_pairs_index, and the first entry of each run of equal determinants opens a
// row.  Each coefficient is then written to (row, column) exactly once: no sums, so the result does not depend on the
// caller's row order or on scheduling.
template <int NW>
__global__ void ladder_candidates_kernel(const uint64_t *up, const uint64_t *dn, const double *c, int64_t n, const int32_t *orbs, int P, int spin,
                                         int create, uint64_t *iu, uint64_t *id, double *iv, int32_t *ok) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n * P) return;
  const int64_t i = t / P;
  const int p = orbs[t - i * P];
  const Bits<NW> U = b_load<NW>(up, i), D = b_load<NW>(dn, i);
  Bits<NW> x = spin ? D : U;
  const bool occ = b_test(x, p);
  ok[t] = occ != (create != 0);
  const int par = b_popc(b_and(x, b_maskr<NW>(p))) + (spin ? b_popc(U) : 0);
  if (create) b_set(x, p);
  else b_clear(x, p);
  b_store(iu, t, spin ? U : x);
  b_store(id, t, spin ? x : D);
  iv[t] = (par & 1) ? -c[i] : c[i];
}

// first entry of each run of equal (up, dn) in a sorted list
template <int NW>
__global__ void run_head_kernel(const uint64_t *u, const uint64_t *d, int64_t m, int32_t *head) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= m) return;
  head[k] = (k == 0 || !b_eq(b_load<NW>(u, k), b_load<NW>(u, k - 1)) || !b_eq(b_load<NW>(d, k), b_load<NW>(d, k - 1))) ? 1 : 0;
}

// coef[row(k) + nout * col(k)] = value of sorted candidate k; row(k) = inclusive head count - 1
__global__ void ladder_scatter_kernel(const int32_t *sel, const int32_t *order, const int32_t *row_incl, const double *iv, int64_t m, int P, int64_t nout,
                                      double *coef) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= m) return;
  const int32_t slot = sel[order[k]];
  coef[(int64_t)(row_incl[k] - 1) + nout * (slot % P)] = iv[slot];
}

// strings of NW words -> the 16-byte host layout (two words per determinant)
template <int NW>
__global__ void widen_strings_kernel(const uint64_t *src, int64_t n, uint64_t *dst) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  dst[2 * k] = src[k * NW];
  dst[2 * k + 1] = NW == 2 ? src[k * NW + 1] : 0ull;
}

// indices k < n with flag[k] != 0, in ascending order -> sel (device), count (host)
static int select_flagged(const int32_t *flag, int64_t n, DevBuf<int32_t> &sel, int64_t &count, cudaStream_t s) {
  SQ_CHECK(sel.alloc(std::max<int64_t>(n, 1)));
  DevBuf<int> nsel;
  SQ_CHECK(nsel.alloc(1));
  thrust::counting_iterator<int32_t> rows(0);
  size_t tb = 0;
  cub::DeviceSelect::Flagged(nullptr, tb, rows, flag, sel.p, nsel.p, (int)n, s);
  DevBuf<char> tmp;
  SQ_CHECK(tmp.alloc((int64_t)tb + 16));
  SQ_CUDA(cub::DeviceSelect::Flagged(tmp.p, tb, rows, flag, sel.p, nsel.p, (int)n, s));
  g_launch_count += 1;
  int m = 0;
  SQ_CUDA(cudaMemcpyAsync(&m, nsel.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  count = m;
  return 0;
}

template <int NW>
static int ladder_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *w_state, int64_t ldw, int spin, int create,
                       int P, const int32_t *orbs, int64_t *n_out) {
  cudaStream_t s = G.stream;
  const int norb = h->T.norb;
  DevBuf<uint64_t> up, dn, ma0, mi0;
  DevBuf<double> w, c0;
  DevBuf<int32_t> idx0;
  int64_t n2 = 0;
  SQ_CHECK(prepare_dets<NW>(h, "ladder", n, dets_up, dets_dn, 1, w_state, ldw, up, dn, w, n2, idx0, ma0, mi0, c0));
  up.release(); dn.release(); w.release(); idx0.release();
  const int64_t nc = n2 * P;
  if (nc > INT32_MAX) { set_error("ladder: %lld determinants x %d orbitals exceed the 32-bit candidate index", (long long)n2, P); return 2; }
  DevBuf<int32_t> d_orbs, ok, sel;
  DevBuf<uint64_t> iu, id;
  DevBuf<double> iv;
  SQ_CHECK(d_orbs.alloc(P));
  SQ_CUDA(cudaMemcpyAsync(d_orbs.p, orbs, P * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  SQ_CHECK(iu.alloc(nc * NW));
  SQ_CHECK(id.alloc(nc * NW));
  SQ_CHECK(iv.alloc(nc));
  SQ_CHECK(ok.alloc(nc));
  ladder_candidates_kernel<NW><<<(unsigned)div_up(nc, 256), 256, 0, s>>>(ma0.p, mi0.p, c0.p, n2, d_orbs.p, P, spin, create, iu.p, id.p, iv.p, ok.p);
  SQ_LAUNCH_CHECK();
  ma0.release(); mi0.release(); c0.release();
  int64_t m = 0;
  SQ_CHECK(select_flagged(ok.p, nc, sel, m, s));
  ok.release();
  h->lad_up.clear();
  h->lad_dn.clear();
  h->lad_coef.clear();
  h->lad_norbs = P;
  *n_out = 0;
  if (m == 0) return 0;
  // valid candidates in slot order, then sorted by (up, dn)
  DevBuf<uint64_t> cu, cd, su, sd;
  DevBuf<int32_t> order;
  SQ_CHECK(cu.alloc(m * NW));
  SQ_CHECK(cd.alloc(m * NW));
  SQ_CHECK(gather_strings(NW, iu.p, sel.p, cu.p, m, s));
  SQ_CHECK(gather_strings(NW, id.p, sel.p, cd.p, m, s));
  iu.release(); id.release();
  SQ_CHECK(order.alloc(m));
  SQ_CHECK(sort_pairs_index(NW, norb, cu.p, cd.p, order.p, m, s));
  SQ_CHECK(su.alloc(m * NW));
  SQ_CHECK(sd.alloc(m * NW));
  SQ_CHECK(gather_strings(NW, cu.p, order.p, su.p, m, s));
  SQ_CHECK(gather_strings(NW, cd.p, order.p, sd.p, m, s));
  cu.release(); cd.release();
  DevBuf<int32_t> head, row;
  SQ_CHECK(head.alloc(m));
  SQ_CHECK(row.alloc(m));
  run_head_kernel<NW><<<(unsigned)div_up(m, 256), 256, 0, s>>>(su.p, sd.p, m, head.p);
  SQ_LAUNCH_CHECK();
  {
    size_t tb = 0;
    cub::DeviceScan::InclusiveSum(nullptr, tb, head.p, row.p, (int)m, s);
    DevBuf<char> tmp;
    SQ_CHECK(tmp.alloc((int64_t)tb + 16));
    SQ_CUDA(cub::DeviceScan::InclusiveSum(tmp.p, tb, head.p, row.p, (int)m, s));
    g_launch_count += 1;
  }
  int32_t nout32 = 0;
  SQ_CUDA(cudaMemcpyAsync(&nout32, row.p + (m - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  const int64_t nout = nout32;
  DevBuf<double> coef;
  SQ_CHECK(coef.alloc(nout * P));
  SQ_CUDA(cudaMemsetAsync(coef.p, 0, nout * P * sizeof(double), s));
  ladder_scatter_kernel<<<(unsigned)div_up(m, 256), 256, 0, s>>>(sel.p, order.p, row.p, iv.p, m, P, nout, coef.p);
  SQ_LAUNCH_CHECK();
  // the union: the head of every run, widened to the 16-byte layout
  DevBuf<int32_t> heads;
  int64_t nh = 0;
  SQ_CHECK(select_flagged(head.p, m, heads, nh, s));
  DevBuf<uint64_t> ou, od, wide;
  SQ_CHECK(ou.alloc(nout * NW));
  SQ_CHECK(od.alloc(nout * NW));
  SQ_CHECK(gather_strings(NW, su.p, heads.p, ou.p, nout, s));
  SQ_CHECK(gather_strings(NW, sd.p, heads.p, od.p, nout, s));
  SQ_CHECK(wide.alloc(2 * nout));
  h->lad_up.resize(2 * nout);
  h->lad_dn.resize(2 * nout);
  h->lad_coef.resize(nout * P);
  widen_strings_kernel<NW><<<(unsigned)div_up(nout, 256), 256, 0, s>>>(ou.p, nout, wide.p);
  SQ_LAUNCH_CHECK();
  SQ_CUDA(cudaMemcpyAsync(h->lad_up.data(), wide.p, 2 * nout * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  widen_strings_kernel<NW><<<(unsigned)div_up(nout, 256), 256, 0, s>>>(od.p, nout, wide.p);
  SQ_LAUNCH_CHECK();
  SQ_CUDA(cudaMemcpyAsync(h->lad_dn.data(), wide.p, 2 * nout * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaMemcpyAsync(h->lad_coef.data(), coef.p, nout * P * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  *n_out = nout;
  return 0;
}

int ladder(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int n_states, const double *wts, int64_t ldw, int state, int spin,
           int create, int n_orbs, const int32_t *orbs, int64_t *n_out) {
  h->lad_up.clear();
  h->lad_dn.clear();
  h->lad_coef.clear();
  h->lad_norbs = 0;
  if (G.nranks > 1) { set_error("ladder: runs on a single process only (nranks = %d)", G.nranks); return 2; }
  if (n <= 0) { set_error("ladder: n must be positive"); return 2; }
  if (n > INT32_MAX) { set_error("ladder: n exceeds the 32-bit row index"); return 2; }
  if (n_states < 1) { set_error("ladder: n_states must be >= 1"); return 2; }
  if (ldw < n) { set_error("ladder: ldw (%lld) must be >= n (%lld)", (long long)ldw, (long long)n); return 2; }
  if (state < 0 || state >= n_states) { set_error("ladder: state %d is not in [0, %d)", state, n_states); return 2; }
  if (spin != 0 && spin != 1) { set_error("ladder: spin must be 0 (up) or 1 (dn), got %d", spin); return 2; }
  if (n_orbs < 1) { set_error("ladder: n_orbs must be >= 1"); return 2; }
  const int norb = h->T.norb;
  std::vector<char> seen(norb, 0);
  for (int j = 0; j < n_orbs; j++) {
    if (orbs[j] < 0 || orbs[j] >= norb) { set_error("ladder: orbital %d is not in [0, %d)", orbs[j], norb); return 2; }
    if (seen[orbs[j]]) { set_error("ladder: orbital %d is listed twice", orbs[j]); return 2; }
    seen[orbs[j]] = 1;
  }
  const int nspin = spin ? h->T.ndn : h->T.nup;
  if (!create && nspin == 0) { set_error("ladder: cannot annihilate from an empty %s string", spin ? "dn" : "up"); return 2; }
  if (create && nspin == norb) { set_error("ladder: cannot create into a full %s string", spin ? "dn" : "up"); return 2; }
  const double *w_state = wts + (int64_t)state * ldw;
  return h->NW == 1 ? ladder_impl<1>(h, n, dets_up, dets_dn, w_state, ldw, spin, create, n_orbs, orbs, n_out)
                    : ladder_impl<2>(h, n, dets_up, dets_dn, w_state, ldw, spin, create, n_orbs, orbs, n_out);
}

int ladder_result(sqmc_b200_handle *h, void *up_out, void *dn_out, double *coeffs, int64_t ldc) {
  const int64_t nout = (int64_t)h->lad_up.size() / 2, P = h->lad_norbs;
  if (ldc < nout) { set_error("ladder_result: ldc (%lld) must be >= the number of images (%lld)", (long long)ldc, (long long)nout); return 2; }
  if (nout == 0) return 0;
  memcpy(up_out, h->lad_up.data(), h->lad_up.size() * sizeof(uint64_t));
  memcpy(dn_out, h->lad_dn.data(), h->lad_dn.size() * sizeof(uint64_t));
  for (int64_t j = 0; j < P; j++) memcpy(coeffs + j * ldc, h->lad_coef.data() + j * nout, nout * sizeof(double));
  return 0;
}

}  // namespace sqmc
