// select.cu -- heat-bath determinant selection on the device: SURVEY.md section 8(f) item 1, the step
// immediately before the H build in every HCI iteration.
//
// Replaces get_next_det_list (hci.f90:865-1039) + find_doubly_excited (semistoch.f90:1579-2231) with
// find_important_connected_dets_chem (chemistry.f90:6819-7159) / find_important_connected_dets_heg
// (heg.f90:2475-2727).  For every determinant i of the current list with coefficient c_i and
// |c_i| * min_H_already_done(i) > eps_var the excitations with |H| * |c_i| above eps_var are generated:
//   chem singles  (same irrep only): eps' <= |H| <= min_H_already_done(i)       (:6956-6959)
//   chem doubles                   : eps' <  |H| <= min_H_already_done(i)       (:7042-7046)
//   heg  doubles (momentum conserving): eps' < |H|                              (heg.f90:2609,2625)
// with eps' = eps_var/|c_i|; the reference walks per-pair tables sorted by |H| (dtm_hb) only to prune the
// search -- the selected set is defined by these inequalities, so the kernel enumerates all excitations of a
// determinant (one warp per determinant) and evaluates the same element arithmetic (elements.cuh, no FMA).
// Time-reversal symmetry: new_up == new_dn dropped for z<0, the time-reversed partner of det i dropped, results
// mapped to the representative up <= dn (:6949-6952,6966-6971,7110-7132).
// Chem doubles (norb <= 64) use heat-bath tables like the reference's dtm_hb (chemistry.f90:872-994): |H| of a double
// excitation depends on the four orbitals only, so per hole pair the particle pairs are stored sorted by decreasing |H|
// (built on the device with the same chem_double arithmetic on two-electron determinants -> bit-identical magnitudes);
// a determinant then visits only the table range eps' < |H| <= min_H_already_done of each of its hole pairs instead of
// all ~10^4 double excitations.  Singles, HEG and norb > 64 enumerate and evaluate every excitation.
// The generated determinants are sorted by label, made unique, and those already in the list removed: what
// remains is exactly the tail the reference appends to its list (hci.f90:945-991).
#include <cub/cub.cuh>

#include <algorithm>
#include <cstdlib>

#include "handle.h"

namespace sqmc {

static const int kSelMaxOrb = 128;

template <int NW>
struct SelCtx {
  ModelTables T;
  const int32_t *orbsym;
  const uint64_t *up, *dn;
  const double *coeffs, *min_H;
  double eps_var;
  int64_t n;
  const double *hb_val[2];   // heat-bath tables (null: enumerate all doubles)
  const uint16_t *hb_rs[2];
  // stochastic PT (VALS = 4, second_order_pt_alias): count/probability ratio of every sampled determinant, n_mc - 1, eps_pt_big
  const double *wop;
  double nmc1, eps_big;
};

// ---- heat-bath tables
struct RowOffset {
  int n2;
  __host__ __device__ __forceinline__ int operator()(const int &row) const { return row * n2; }
};
__global__ void hb_fill_kernel(ModelTables T, int os, double *val, uint16_t *rs) {
  extern __shared__ int32_t c2s[];
  const int norb = T.norb, n1 = norb + 1;
  for (int k = threadIdx.x; k < n1 * n1; k += blockDim.x) c2s[k] = T.combine_2[k];
  __syncthreads();
  const int64_t n2 = (int64_t)norb * norb, tot = n2 * n2;
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= tot) return;
  const int row = (int)(t / n2), col = (int)(t % n2);
  const int p = row / norb, q = row % norb, r = col / norb, s = col % norb;
  double v = 0.0;
  ChemCtx C{T.integrals, c2s, n1, T.enuc, T.sqrt2, T.sqrt2inv, T.z};
  Bits<1> iu = b_zero<1>(), id = b_zero<1>(), ju = b_zero<1>(), jd = b_zero<1>();
  if (!os) {
    if (p < q && r < s && r != p && r != q && s != p && s != q) {
      b_set(iu, p); b_set(iu, q); b_set(ju, r); b_set(ju, s);
      v = fabs(chem_double(C, iu, id, ju, jd));
    }
  } else {
    if (r != p && s != q) {
      b_set(iu, p); b_set(id, q); b_set(ju, r); b_set(jd, s);
      v = fabs(chem_double(C, iu, id, ju, jd));
    }
  }
  val[t] = v;
  rs[t] = (uint16_t)(r | (s << 8));
}
static int hb_build(sqmc_b200_handle *h) {
  const ModelTables &T = h->T;
  if (h->hb_norb == T.norb && h->d_hb_val[0]) return 0;
  cudaStream_t s = G.stream;
  const int norb = T.norb;
  const int64_t n2 = (int64_t)norb * norb, tot = n2 * n2;
  const int c2bytes = (norb + 1) * (norb + 1) * 4;
  DevBuf<double> kin;
  DevBuf<uint16_t> vin;
  SQ_CHECK(kin.alloc(tot));
  SQ_CHECK(vin.alloc(tot));
  cub::CountingInputIterator<int> cnt0(0), cnt1(1);
  cub::TransformInputIterator<int, RowOffset, cub::CountingInputIterator<int>> beg(cnt0, RowOffset{(int)n2}), end(cnt1, RowOffset{(int)n2});
  for (int os = 0; os < 2; os++) {
    if (h->d_hb_val[os]) { cudaFree(h->d_hb_val[os]); h->d_hb_val[os] = nullptr; }
    if (h->d_hb_rs[os]) { cudaFree(h->d_hb_rs[os]); h->d_hb_rs[os] = nullptr; }
    SQ_CUDA(cudaMalloc(&h->d_hb_val[os], tot * sizeof(double)));
    SQ_CUDA(cudaMalloc(&h->d_hb_rs[os], tot * sizeof(uint16_t)));
    hb_fill_kernel<<<(unsigned)div_up(tot, 256), 256, c2bytes, s>>>(T, os, kin.p, vin.p);
    SQ_LAUNCH_CHECK();
    size_t tb = 0;
    cub::DeviceSegmentedRadixSort::SortPairsDescending(nullptr, tb, kin.p, h->d_hb_val[os], vin.p, h->d_hb_rs[os], (int)tot, (int)n2, beg, end, 0, 64, s);
    DevBuf<char> tmp;
    SQ_CHECK(tmp.alloc((int64_t)tb + 16));
    SQ_CUDA(cub::DeviceSegmentedRadixSort::SortPairsDescending(tmp.p, tb, kin.p, h->d_hb_val[os], vin.p, h->d_hb_rs[os], (int)tot, (int)n2, beg, end, 0, 64, s));
    g_launch_count += 1;
    SQ_CUDA(cudaStreamSynchronize(s));
  }
  h->hb_norb = norb;
  return 0;
}
// number of leading entries of a row (sorted by decreasing value) that are > x
__device__ __forceinline__ int hb_count_gt(const double *row, int n, double x) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (row[mid] > x) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ int nth_set(const uint8_t *list, int k) { return list[k]; }

// one warp per determinant; FILL=false counts, FILL=true writes (up,dn) of the selected determinants at out_ptr[i];
// VALS = 1 additionally writes H(selected, i) * c_i, the numerator contributions of the second-order correction (pt2 below);
// VALS = 4 writes the four sums of one stochastic-PT sample per connection k of sampled determinant i (semistoch.f90:2044-2060):
//   H_ki c_i w_i/p_i,  (H_ki c_i)^2 ((n_mc-1) w_i/p_i - (w_i/p_i)^2),  and the same two with H_ki replaced by 0 unless
//   |H_ki| > eps_pt_big/|c_i| (chemistry.f90:6977-6983,7134-7140), interleaved out_val[4*q + 0..3]
template <int NW, bool FILL, int VALS, int MODEL, bool TS>
__global__ void __launch_bounds__(128) select_kernel(SelCtx<NW> S, int64_t i_begin, int64_t i_end, int32_t *counts, const int64_t *out_ptr,
                                                     uint64_t *out_up, uint64_t *out_dn, double *out_val) {
  __shared__ uint8_t s_occ[4][2][kSelMaxOrb], s_virt[4][2][kSelMaxOrb];
  extern __shared__ int32_t c2s[];
  const ModelTables &T = S.T;
  const int32_t *c2 = T.combine_2;
  if (MODEL == MODEL_CHEM) {
    const int n1 = T.norb + 1;
    for (int k = threadIdx.x; k < n1 * n1; k += blockDim.x) c2s[k] = T.combine_2[k];
    __syncthreads();
    c2 = c2s;
  }
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t i = i_begin + ((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
  if (i >= i_end) return;
  const unsigned full = 0xffffffffu, lt = (1u << lane) - 1u;
  const Bits<NW> u = b_load<NW>(S.up, i), d = b_load<NW>(S.dn, i);
  const double cs = S.coeffs[i], c = fabs(cs), minH = S.min_H[i];
  const double wop = VALS == 4 ? S.wop[i] : 0.0, wfac = S.nmc1 * wop - wop * wop, eps_big = S.eps_big / c;
  const int norb = T.norb;
  constexpr bool ts = TS;  // time-reversal symmetrised determinants (chem only)
  int64_t base = FILL ? out_ptr[i - i_begin] : 0;
  int cnt = 0;
  // val = determinant-level element (VALS only): under time-reversal symmetry only this contribution to the symmetrised
  // element is kept -- norm factors (chemistry.f90:6961-6964, 7121-7124), z when mapped to the representative
  // (:6966-6971, 7127-7134) -- and the coefficient of the generating determinant is multiplied in last (semistoch.f90:2048)
  auto emit = [&](bool keep, Bits<NW> nu, Bits<NW> nd, double val) {
    if (VALS && keep && ts) {
      if (b_eq(u, d) && !b_eq(nu, nd)) val = T.sqrt2inv * val;
      if (b_eq(nu, nd) && !b_eq(u, d)) val = T.sqrt2 * val;
    }
    if (keep && ts && b_lt(nd, nu)) {  // representative up <= dn
      Bits<NW> t = nu; nu = nd; nd = t;
      if (VALS) val = T.z * val;
    }
    unsigned m = __ballot_sync(full, keep);
    if (FILL && keep) {
      int64_t q = base + cnt + __popc(m & lt);
      b_store<NW>(out_up, q, nu);
      b_store<NW>(out_dn, q, nd);
      if (VALS == 1) out_val[q] = val * cs;
      if (VALS == 4) {
        const double hc = val * cs, t1 = hc * wop, t2 = (hc * hc) * wfac;
        const bool big = fabs(val) > eps_big;
        out_val[4 * q] = t1;
        out_val[4 * q + 1] = t2;
        out_val[4 * q + 2] = big ? t1 : 0.0;
        out_val[4 * q + 3] = big ? t2 : 0.0;
      }
    }
    cnt += __popc(m);
  };
  emit(lane == 0, u, d, 0.0);  // the determinant itself comes first (chemistry.f90:6893-6895), with element 0 (heg.f90:2525-2529)
  const bool expand = c * minH > S.eps_var;  // semistoch.f90:1825
  if (expand) {  // warp-uniform
    const double eps = S.eps_var / c;
    // occupied / virtual orbital lists of both spins (lane 0 of the warp fills them)
    uint8_t *occ_u = s_occ[wib][0], *occ_d = s_occ[wib][1], *vir_u = s_virt[wib][0], *vir_d = s_virt[wib][1];
    int nu_ = 0, nd_ = 0, nvu = 0, nvd = 0;
    if (lane == 0) {
      for (int o = 0; o < norb; o++) {
        if (b_test(u, o)) occ_u[nu_++] = (uint8_t)o; else vir_u[nvu++] = (uint8_t)o;
        if (b_test(d, o)) occ_d[nd_++] = (uint8_t)o; else vir_d[nvd++] = (uint8_t)o;
      }
    }
    nu_ = __shfl_sync(full, nu_, 0); nd_ = __shfl_sync(full, nd_, 0); nvu = __shfl_sync(full, nvu, 0); nvd = __shfl_sync(full, nvd, 0);
    __syncwarp();
    ChemCtx C{T.integrals, c2, T.norb + 1, T.enuc, T.sqrt2, T.sqrt2inv, T.z};
    HegCtx Hg{T.k_vectors, T.n_dim, T.length_cell};
    auto ts_excluded = [&](const Bits<NW> &nu, const Bits<NW> &nd) {
      if (!ts) return false;
      if (b_eq(nu, nd) && T.z < 0) return true;
      return b_eq(u, nd) && b_eq(d, nu);
    };
    // ---- singles (chem only)
    if constexpr (MODEL == MODEL_CHEM) {
      for (int spin = 0; spin < 2; spin++) {
        const uint8_t *occ = spin == 0 ? occ_u : occ_d, *vir = spin == 0 ? vir_u : vir_d;
        const int no = spin == 0 ? nu_ : nd_, nv = spin == 0 ? nvu : nvd;
        const int tot = no * nv;
        for (int b0 = 0; b0 < tot; b0 += 32) {
          const int f = b0 + lane;
          bool keep = false;
          double val = 0.0;
          Bits<NW> nu = u, nd = d;
          if (f < tot) {
            const int p = occ[f / nv], r = vir[f % nv];
            if (S.orbsym[p] == S.orbsym[r]) {
              if (spin == 0) { b_clear(nu, p); b_set(nu, r); } else { b_clear(nd, p); b_set(nd, r); }
              if (!ts_excluded(nu, nd)) {
                val = chem_hamiltonian_level(C, u, d, nu, nd, 1);
                const double me = fabs(val);
                keep = !(me < eps) && !(me > minH);
              }
            }
          }
          emit(keep, nu, nd, val);
        }
      }
    }
    const bool use_hb = (MODEL == MODEL_CHEM) && S.hb_val[0] != nullptr;
    if (use_hb) {
      // ---- doubles from the heat-bath tables: one lane per hole pair finds its table range, then the warp walks it
      const int nss_u = nu_ * (nu_ - 1) / 2, nss_d = nd_ * (nd_ - 1) / 2, nos = nu_ * nd_;
      const int npairs = nss_u + nss_d + nos;
      const int n2 = norb * norb;
      for (int pb0 = 0; pb0 < npairs; pb0 += 32) {
        int kind = 0, p = 0, q = 0, lo = 0, hi = 0;  // kind 0: up-up, 1: dn-dn, 2: up-dn
        const int pi = pb0 + lane;
        if (pi < npairs) {
          int t = pi;
          if (t < nss_u + nss_d) {
            kind = t < nss_u ? 0 : 1;
            if (kind == 1) t -= nss_u;
            const uint8_t *occ = kind == 0 ? occ_u : occ_d;
            const int no = kind == 0 ? nu_ : nd_;
            int a = 0;
            while (t >= no - 1 - a) { t -= no - 1 - a; a++; }
            p = occ[a]; q = occ[a + 1 + t];
          } else {
            kind = 2;
            t -= nss_u + nss_d;
            p = occ_u[t / nd_]; q = occ_d[t % nd_];
          }
          const double *row = S.hb_val[kind == 2] + (int64_t)(p * norb + q) * n2;
          lo = hb_count_gt(row, n2, minH);  // |H| > min_H_already_done: handled in an earlier iteration
          hi = hb_count_gt(row, n2, eps);   // |H| > eps'
        }
        const int npb = min(32, npairs - pb0);
        for (int j = 0; j < npb; j++) {
          const int kj = __shfl_sync(full, kind, j), pj = __shfl_sync(full, p, j), qj = __shfl_sync(full, q, j);
          const int loj = __shfl_sync(full, lo, j), hij = __shfl_sync(full, hi, j);
          const uint16_t *rsrow = S.hb_rs[kj == 2] + (int64_t)(pj * norb + qj) * n2;
          for (int f0 = loj; f0 < hij; f0 += 32) {
            const int f = f0 + lane;
            bool keep = false;
            Bits<NW> nu = u, nd = d;
            if (f < hij) {
              const int rs = rsrow[f], r = rs & 255, sx = rs >> 8;
              if (kj == 0) {
                keep = !b_test(u, r) && !b_test(u, sx);
                b_clear(nu, pj); b_clear(nu, qj); b_set(nu, r); b_set(nu, sx);
              } else if (kj == 1) {
                keep = !b_test(d, r) && !b_test(d, sx);
                b_clear(nd, pj); b_clear(nd, qj); b_set(nd, r); b_set(nd, sx);
              } else {
                keep = !b_test(u, r) && !b_test(d, sx);
                b_clear(nu, pj); b_set(nu, r); b_clear(nd, qj); b_set(nd, sx);
              }
              if (keep && ts_excluded(nu, nd)) keep = false;
            }
            double val = 0.0;
            if (VALS && keep) val = chem_double(C, u, d, nu, nd);  // the table holds |H|; the sign needs the determinant
            emit(keep, nu, nd, val);
          }
        }
      }
    }
    // ---- same-spin doubles
    for (int spin = 0; spin < 2 && !use_hb; spin++) {
      const uint8_t *occ = spin == 0 ? occ_u : occ_d, *vir = spin == 0 ? vir_u : vir_d;
      const int no = spin == 0 ? nu_ : nd_, nv = spin == 0 ? nvu : nvd;
      const int npo = no * (no - 1) / 2, npv = nv * (nv - 1) / 2;
      const int tot = npo * npv;
      for (int b0 = 0; b0 < tot; b0 += 32) {
        const int f = b0 + lane;
        bool keep = false;
        double val = 0.0;
        Bits<NW> nu = u, nd = d;
        if (f < tot) {
          int po = f / npv, pv = f % npv;
          // unrank pairs (a<b): pair index -> (a,b)
          int a = 0;
          while (po >= no - 1 - a) { po -= no - 1 - a; a++; }
          const int bq = a + 1 + po;
          int r = 0;
          while (pv >= nv - 1 - r) { pv -= nv - 1 - r; r++; }
          const int sq = r + 1 + pv;
          Bits<NW> &tgt = spin == 0 ? nu : nd;
          b_clear(tgt, occ[a]); b_clear(tgt, occ[bq]); b_set(tgt, vir[r]); b_set(tgt, vir[sq]);
          if (!ts_excluded(nu, nd)) {
            if constexpr (MODEL == MODEL_CHEM) val = chem_hamiltonian_level(C, u, d, nu, nd, 2);
            else val = heg_hamiltonian(Hg, u, d, nu, nd);
            const double me = fabs(val);
            keep = (me > eps) && (MODEL != MODEL_CHEM || !(me > minH));
          }
        }
        emit(keep, nu, nd, val);
      }
    }
    // ---- opposite-spin doubles
    if (!use_hb) {
      const int tu = nu_ * nvu, td = nd_ * nvd;
      const int64_t tot = (int64_t)tu * td;
      for (int64_t b0 = 0; b0 < tot; b0 += 32) {
        const int64_t f = b0 + lane;
        bool keep = false;
        double val = 0.0;
        Bits<NW> nu = u, nd = d;
        if (f < tot) {
          const int fu = (int)(f / td), fd = (int)(f % td);
          b_clear(nu, occ_u[fu / nvu]); b_set(nu, vir_u[fu % nvu]);
          b_clear(nd, occ_d[fd / nvd]); b_set(nd, vir_d[fd % nvd]);
          if (!ts_excluded(nu, nd)) {
            if constexpr (MODEL == MODEL_CHEM) val = chem_hamiltonian_level(C, u, d, nu, nd, 2);
            else val = heg_hamiltonian(Hg, u, d, nu, nd);
            const double me = fabs(val);
            keep = (me > eps) && (MODEL != MODEL_CHEM || !(me > minH));
          }
        }
        emit(keep, nu, nd, val);
      }
    }
  }
  if (!FILL && lane == 0) counts[i - i_begin] = cnt;
}

__global__ void stride_index_kernel(int32_t *idx, int64_t m, int first, int stride) {
  int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < m) idx[k] = (int32_t)(first + k * stride);
}

template <int NW>
__global__ void uniq_flag_kernel(const uint64_t *a, const uint64_t *b, int32_t *flag, int64_t m) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= m) return;
  flag[t] = (t == 0) ? 1 : ((b_eq(b_load<NW>(a, t), b_load<NW>(a, t - 1)) && b_eq(b_load<NW>(b, t), b_load<NW>(b, t - 1))) ? 0 : 1);
}
// flag[t] &= (a[t], b[t]) not in the sorted list (oa, ob)
template <int NW>
__global__ void not_in_list_kernel(const uint64_t *a, const uint64_t *b, const uint64_t *oa, const uint64_t *ob, int64_t nold, int32_t *flag, int64_t m) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= m || !flag[t]) return;
  const Bits<NW> x = b_load<NW>(a, t), y = b_load<NW>(b, t);
  int64_t lo = 0, hi = nold;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    const Bits<NW> ma = b_load<NW>(oa, mid), mb = b_load<NW>(ob, mid);
    const bool less = b_lt(ma, x) || (b_eq(ma, x) && b_lt(mb, y));
    if (less) lo = mid + 1;
    else hi = mid;
  }
  if (lo < nold && b_eq(b_load<NW>(oa, lo), x) && b_eq(b_load<NW>(ob, lo), y)) flag[t] = 0;
}

// sort (a,b) pairs by label, keep the unique ones that are not in the sorted old list; returns them compacted in (ra, rb)
template <int NW>
static int sort_unique_new(int norb, DevBuf<uint64_t> &a, DevBuf<uint64_t> &b, int64_t m, const uint64_t *oa, const uint64_t *ob, int64_t nold,
                           DevBuf<uint64_t> &ra, DevBuf<uint64_t> &rb, int64_t &mout, cudaStream_t s) {
  mout = 0;
  if (m == 0) return 0;
  DevBuf<int32_t> idx, flag, sel;
  DevBuf<uint64_t> sa, sb;
  SQ_CHECK(idx.alloc(m));
  SQ_CHECK(sort_pairs_index(NW, norb, a.p, b.p, idx.p, m, s));
  SQ_CHECK(sa.alloc(m * NW));
  SQ_CHECK(sb.alloc(m * NW));
  SQ_CHECK(gather_strings(NW, a.p, idx.p, sa.p, m, s));
  SQ_CHECK(gather_strings(NW, b.p, idx.p, sb.p, m, s));
  SQ_CHECK(flag.alloc(m));
  const unsigned g = (unsigned)div_up(m, 256);
  uniq_flag_kernel<NW><<<g, 256, 0, s>>>(sa.p, sb.p, flag.p, m);
  SQ_LAUNCH_CHECK();
  if (nold > 0) {
    not_in_list_kernel<NW><<<g, 256, 0, s>>>(sa.p, sb.p, oa, ob, nold, flag.p, m);
    SQ_LAUNCH_CHECK();
  }
  SQ_CHECK(sel.alloc(m));
  DevBuf<int32_t> num;
  SQ_CHECK(num.alloc(1));
  cub::CountingInputIterator<int32_t> it(0);
  size_t tb = 0;
  cub::DeviceSelect::Flagged(nullptr, tb, it, flag.p, sel.p, num.p, (int)m, s);
  DevBuf<char> tmp;
  SQ_CHECK(tmp.alloc((int64_t)tb + 16));
  SQ_CUDA(cub::DeviceSelect::Flagged(tmp.p, tb, it, flag.p, sel.p, num.p, (int)m, s));
  g_launch_count += 2;
  int32_t k = 0;
  SQ_CUDA(cudaMemcpyAsync(&k, num.p, 4, cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  mout = k;
  SQ_CHECK(ra.alloc(std::max<int64_t>(mout, 1) * NW));
  SQ_CHECK(rb.alloc(std::max<int64_t>(mout, 1) * NW));
  SQ_CHECK(gather_strings(NW, sa.p, sel.p, ra.p, mout, s));
  SQ_CHECK(gather_strings(NW, sb.p, sel.p, rb.p, mout, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// nranks > 1: deal the determinants round-robin to the ranks (the early, large-coefficient determinants of an HCI list
// generate most of the connections, so contiguous slices would be unbalanced).  Replaces (up, dn, c, m) by this rank's
// share and returns its size.
template <int NW>
static int shard_round_robin(DevBuf<uint64_t> &up, DevBuf<uint64_t> &dn, DevBuf<double> &c, DevBuf<double> &m, int64_t n, int64_t &n_local,
                             cudaStream_t s) {
  n_local = n;
  if (G.nranks == 1) return 0;
  const int64_t nd = n > G.rank ? (n - G.rank + G.nranks - 1) / G.nranks : 0;
  DevBuf<int32_t> sidx;
  DevBuf<uint64_t> lu, ld_;
  DevBuf<double> lc, lm;
  SQ_CHECK(sidx.alloc(std::max<int64_t>(nd, 1)));
  SQ_CHECK(lu.alloc(std::max<int64_t>(nd, 1) * NW));
  SQ_CHECK(ld_.alloc(std::max<int64_t>(nd, 1) * NW));
  SQ_CHECK(lc.alloc(std::max<int64_t>(nd, 1)));
  SQ_CHECK(lm.alloc(std::max<int64_t>(nd, 1)));
  if (nd > 0) {
    stride_index_kernel<<<(unsigned)div_up(nd, 256), 256, 0, s>>>(sidx.p, nd, G.rank, G.nranks);
    SQ_LAUNCH_CHECK();
    SQ_CHECK(gather_strings(NW, up.p, sidx.p, lu.p, nd, s));
    SQ_CHECK(gather_strings(NW, dn.p, sidx.p, ld_.p, nd, s));
    SQ_CHECK(permute_gather(c.p, sidx.p, lc.p, nd, s));
    SQ_CHECK(permute_gather(m.p, sidx.p, lm.p, nd, s));
    SQ_CUDA(cudaStreamSynchronize(s));
  }
  up.release(); dn.release(); c.release(); m.release();
  up.p = lu.take(); dn.p = ld_.take(); c.p = lc.take(); m.p = lm.take();
  n_local = nd;
  return 0;
}

// nranks > 1: concatenate the rank-local lists (a, b[, v]) of nf entries on every rank (sizes all-gathered, payload padded to the
// largest list for a plain ncclAllGather).  v may be null.  Returns the concatenation in (ca, cb, cv) with tot entries.
template <int NW>
static int allgather_lists(const uint64_t *a, const uint64_t *b, const double *v, int64_t nf, DevBuf<uint64_t> &ca, DevBuf<uint64_t> &cb,
                           DevBuf<double> &cv, int64_t &tot, cudaStream_t s, int nch = 1) {
  DevBuf<int64_t> cnt_dev;
  SQ_CHECK(cnt_dev.alloc(G.nranks));
  SQ_CUDA(cudaMemcpyAsync(cnt_dev.p + G.rank, &nf, sizeof(int64_t), cudaMemcpyHostToDevice, s));
  ncclResult_t rc = ncclAllGather(cnt_dev.p + G.rank, cnt_dev.p, 1, ncclInt64, G.comm, s);
  if (rc != ncclSuccess) { set_error("ncclAllGather(list sizes) failed: %s", ncclGetErrorString(rc)); return 3; }
  std::vector<int64_t> cnts(G.nranks);
  SQ_CUDA(cudaMemcpyAsync(cnts.data(), cnt_dev.p, G.nranks * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  int64_t mx = 0;
  tot = 0;
  for (int64_t c : cnts) { mx = std::max(mx, c); tot += c; }
  if (mx == 0) return 0;
  DevBuf<uint64_t> ga, gb;
  DevBuf<double> gv;
  SQ_CHECK(ga.alloc(mx * NW * G.nranks));
  SQ_CHECK(gb.alloc(mx * NW * G.nranks));
  if (v) SQ_CHECK(gv.alloc(mx * nch * G.nranks));
  if (nf > 0) {
    SQ_CUDA(cudaMemcpyAsync(ga.p + (int64_t)G.rank * mx * NW, a, nf * NW * 8, cudaMemcpyDeviceToDevice, s));
    SQ_CUDA(cudaMemcpyAsync(gb.p + (int64_t)G.rank * mx * NW, b, nf * NW * 8, cudaMemcpyDeviceToDevice, s));
    if (v) SQ_CUDA(cudaMemcpyAsync(gv.p + (int64_t)G.rank * mx * nch, v, nf * nch * 8, cudaMemcpyDeviceToDevice, s));
  }
  rc = ncclAllGather(ga.p + (int64_t)G.rank * mx * NW, ga.p, mx * NW, ncclUint64, G.comm, s);
  if (rc == ncclSuccess) rc = ncclAllGather(gb.p + (int64_t)G.rank * mx * NW, gb.p, mx * NW, ncclUint64, G.comm, s);
  if (rc == ncclSuccess && v) rc = ncclAllGather(gv.p + (int64_t)G.rank * mx * nch, gv.p, mx * nch, ncclDouble, G.comm, s);
  if (rc != ncclSuccess) { set_error("ncclAllGather(lists) failed: %s", ncclGetErrorString(rc)); return 3; }
  SQ_CHECK(ca.alloc(std::max<int64_t>(tot, 1) * NW));
  SQ_CHECK(cb.alloc(std::max<int64_t>(tot, 1) * NW));
  if (v) SQ_CHECK(cv.alloc(std::max<int64_t>(tot, 1) * nch));
  int64_t off = 0;
  for (int r = 0; r < G.nranks; r++) {
    if (cnts[r] == 0) continue;
    SQ_CUDA(cudaMemcpyAsync(ca.p + off * NW, ga.p + (int64_t)r * mx * NW, cnts[r] * NW * 8, cudaMemcpyDeviceToDevice, s));
    SQ_CUDA(cudaMemcpyAsync(cb.p + off * NW, gb.p + (int64_t)r * mx * NW, cnts[r] * NW * 8, cudaMemcpyDeviceToDevice, s));
    if (v) SQ_CUDA(cudaMemcpyAsync(cv.p + off * nch, gv.p + (int64_t)r * mx * nch, cnts[r] * nch * 8, cudaMemcpyDeviceToDevice, s));
    off += cnts[r];
  }
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

template <int NW>
static int select_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *coeffs, double *min_H, double eps_var,
                       int64_t *n_new_out) {
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  HostMarks HM("SQMC_SELECT_PROFILE", "select");
  DevBuf<uint64_t> up, dn, sup, sdn;
  DevBuf<double> dc, dm;
  SQ_CHECK(up.alloc(n * NW));
  SQ_CHECK(dn.alloc(n * NW));
  SQ_CHECK(upload_dets(NW, T.norb, dets_up, up.p, n, s));
  SQ_CHECK(upload_dets(NW, T.norb, dets_dn, dn.p, n, s));
  SQ_CHECK(dc.alloc(n));
  SQ_CHECK(dm.alloc(n));
  SQ_CUDA(cudaMemcpyAsync(dc.p, coeffs, n * sizeof(double), cudaMemcpyHostToDevice, s));
  SQ_CUDA(cudaMemcpyAsync(dm.p, min_H, n * sizeof(double), cudaMemcpyHostToDevice, s));
  // sorted copy of the current list for the membership test
  {
    DevBuf<int32_t> idx;
    SQ_CHECK(idx.alloc(n));
    SQ_CHECK(sort_pairs_index(NW, T.norb, up.p, dn.p, idx.p, n, s));
    SQ_CHECK(sup.alloc(n * NW));
    SQ_CHECK(sdn.alloc(n * NW));
    SQ_CHECK(gather_strings(NW, up.p, idx.p, sup.p, n, s));
    SQ_CHECK(gather_strings(NW, dn.p, idx.p, sdn.p, n, s));
  }
  HM.mark("upload + sorted copy of the list");
  const bool use_hb = T.model == MODEL_CHEM && NW == 1 && T.norb <= 64;
  if (use_hb) SQ_CHECK(hb_build(h));
  int64_t nd = n;  // determinants this rank expands (all of them on one rank)
  SQ_CHECK(shard_round_robin<NW>(up, dn, dc, dm, n, nd, s));
  SelCtx<NW> S{T, h->d_orbsym, up.p, dn.p, dc.p, dm.p, eps_var, nd,
               {use_hb ? h->d_hb_val[0] : nullptr, use_hb ? h->d_hb_val[1] : nullptr}, {use_hb ? h->d_hb_rs[0] : nullptr, use_hb ? h->d_hb_rs[1] : nullptr}};
  const int c2bytes = (T.model == MODEL_CHEM) ? (T.norb + 1) * (T.norb + 1) * 4 : 0;
  // count pass over all determinants
  DevBuf<int32_t> counts;
  SQ_CHECK(counts.alloc(nd + 1));
  SQ_CUDA(cudaMemsetAsync(counts.p, 0, (nd + 1) * sizeof(int32_t), s));
  if (nd > 0) {
    SQ_MODEL_DISPATCH(T, SQ_CUDA((allow_dynamic_smem(select_kernel<NW, false, 0, kModel, kTS>, c2bytes))));
    SQ_MODEL_DISPATCH(T, (select_kernel<NW, false, 0, kModel, kTS><<<(unsigned)div_up(nd * 32, 128), 128, c2bytes, s>>>(S, 0, nd, counts.p, nullptr, nullptr, nullptr, nullptr)));
    SQ_LAUNCH_CHECK();
  }
  std::vector<int32_t> hc(nd + 1);
  SQ_CUDA(cudaMemcpyAsync(hc.data(), counts.p, (nd + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  std::vector<int64_t> prefix(nd + 1, 0);
  for (int64_t i = 0; i < nd; i++) prefix[i + 1] = prefix[i] + hc[i];
  HM.mark("count pass + prefix");
  // chunks of determinants bounded by generated candidates; per chunk: fill, sort, unique, drop members of the list
  const int64_t kChunk = 1ll << 27;
  DevBuf<uint64_t> acc_a, acc_b;  // unique new determinants found so far (unsorted union of the chunk results)
  int64_t acc_n = 0;
  int64_t i0 = 0;
  while (i0 < nd) {
    int64_t i1 = std::upper_bound(prefix.begin() + i0 + 1, prefix.end(), prefix[i0] + kChunk) - prefix.begin() - 1;
    if (i1 <= i0) i1 = i0 + 1;
    if (i1 > nd) i1 = nd;
    const int64_t m = prefix[i1] - prefix[i0];
    if (m >= (1ll << 31)) { set_error("hci_select: one determinant generates too many connections"); return 2; }
    DevBuf<uint64_t> ca, cb, ra, rb;
    DevBuf<int64_t> optr;
    SQ_CHECK(ca.alloc(std::max<int64_t>(m, 1) * NW));
    SQ_CHECK(cb.alloc(std::max<int64_t>(m, 1) * NW));
    SQ_CHECK(optr.alloc(i1 - i0 + 1));
    std::vector<int64_t> hp(prefix.begin() + i0, prefix.begin() + i1 + 1);
    for (auto &v : hp) v -= prefix[i0];
    SQ_CUDA(cudaMemcpyAsync(optr.p, hp.data(), hp.size() * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    SQ_MODEL_DISPATCH(T, SQ_CUDA((allow_dynamic_smem(select_kernel<NW, true, 0, kModel, kTS>, c2bytes))));
    SQ_MODEL_DISPATCH(T, (select_kernel<NW, true, 0, kModel, kTS><<<(unsigned)div_up((i1 - i0) * 32, 128), 128, c2bytes, s>>>(S, i0, i1, nullptr, optr.p, ca.p, cb.p, nullptr)));
    SQ_LAUNCH_CHECK();
    SQ_CUDA(cudaStreamSynchronize(s));
    int64_t mu = 0;
    SQ_CHECK(sort_unique_new<NW>(T.norb, ca, cb, m, sup.p, sdn.p, n, ra, rb, mu, s));
    if (mu > 0) {  // append to the accumulator
      DevBuf<uint64_t> na, nb;
      SQ_CHECK(na.alloc((acc_n + mu) * NW));
      SQ_CHECK(nb.alloc((acc_n + mu) * NW));
      if (acc_n) {
        SQ_CUDA(cudaMemcpyAsync(na.p, acc_a.p, acc_n * NW * 8, cudaMemcpyDeviceToDevice, s));
        SQ_CUDA(cudaMemcpyAsync(nb.p, acc_b.p, acc_n * NW * 8, cudaMemcpyDeviceToDevice, s));
      }
      SQ_CUDA(cudaMemcpyAsync(na.p + acc_n * NW, ra.p, mu * NW * 8, cudaMemcpyDeviceToDevice, s));
      SQ_CUDA(cudaMemcpyAsync(nb.p + acc_n * NW, rb.p, mu * NW * 8, cudaMemcpyDeviceToDevice, s));
      SQ_CUDA(cudaStreamSynchronize(s));
      acc_a.release(); acc_b.release();
      acc_a.p = na.take(); acc_b.p = nb.take();
      acc_n += mu;
    }
    i0 = i1;
  }
  HM.mark("fill + sort/unique chunks");
  // final sort + unique across chunks (members of the list are already gone)
  DevBuf<uint64_t> fa, fb;
  int64_t nf = 0;
  SQ_CHECK(sort_unique_new<NW>(T.norb, acc_a, acc_b, acc_n, nullptr, nullptr, 0, fa, fb, nf, s));
  if (G.nranks > 1) {  // merge the rank-local results: all-gather, sort + unique once more (identical on every rank)
    DevBuf<uint64_t> ca, cb, ma, mb;
    DevBuf<double> none;
    int64_t tot = 0, nm = 0;
    SQ_CHECK(allgather_lists<NW>(fa.p, fb.p, nullptr, nf, ca, cb, none, tot, s));
    if (tot > 0) SQ_CHECK(sort_unique_new<NW>(T.norb, ca, cb, tot, nullptr, nullptr, 0, ma, mb, nm, s));
    fa.release(); fb.release();
    fa.p = ma.take(); fb.p = mb.take();
    nf = nm;
  }
  HM.mark("final merge");
  h->sel_new_up.assign((size_t)nf * 2, 0);
  h->sel_new_dn.assign((size_t)nf * 2, 0);
  if (nf > 0) {
    std::vector<uint64_t> ha(nf * NW), hb(nf * NW);
    SQ_CUDA(cudaMemcpy(ha.data(), fa.p, nf * NW * 8, cudaMemcpyDeviceToHost));
    SQ_CUDA(cudaMemcpy(hb.data(), fb.p, nf * NW * 8, cudaMemcpyDeviceToHost));
    for (int64_t k = 0; k < nf; k++)
      for (int w = 0; w < NW; w++) {
        h->sel_new_up[2 * k + w] = ha[k * NW + w];
        h->sel_new_dn[2 * k + w] = hb[k * NW + w];
      }
  }
  // min_H_already_done of the current dets (hci.f90:1015); new dets start at 9e99 on the caller's side (:1016)
  for (int64_t i = 0; i < n; i++) min_H[i] = std::min(min_H[i], eps_var / fabs(coeffs[i]) - 1.e-14);
  HM.mark("download + min_H");
  *n_new_out = nf;
  return 0;
}

// ------------------------------------------------------------------ deterministic second-order correction
// second_order_pt (hci.f90:1100-1182) over find_doubly_excited(..., eps_var_pt = eps_pt, e_mix_num) (semistoch.f90:1579-2231):
// every variational determinant i contributes H_ai c_i to each important connection a (the same screened enumeration as the
// selection, without the min_H_already_done bound); contributions are summed per determinant after a sort by label;
// delta_E = sum over a outside the variational space of (sum_i H_ai c_i)^2 / (E_var - H_aa).  n_connected = number of
// distinct determinants generated (variational ones included), the "ndets_connected" of the reference's log.
__global__ void fill_double_kernel(double *a, int64_t n, double v) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) a[i] = v;
}
__global__ void set_i32_kernel(int32_t *p, int32_t v) { *p = v; }
// NCH = 1: (sum_i H_ai c_i)^2 / (E_var - H_aa) (hci.f90:1167); NCH = 4: one stochastic sample,
// (term1^2 + term2 - term1_big^2 - term2_big) / (E_var - H_aa) (hci.f90:1626)
template <int NW, int MODEL, bool TS, int NCH>
__global__ void pt_term_kernel(ModelTables T, const uint64_t *a, const uint64_t *b, const double *num, const int32_t *external, double e_var,
                               double *term, int64_t m) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= m) return;
  double r = 0.0;
  if (external[t]) {
    const Bits<NW> u = b_load<NW>(a, t), d = b_load<NW>(b, t);
    const double haa = model_hamiltonian<NW, MODEL, TS>(T, T.combine_2, u, d, u, d);
    if (NCH == 1) {
      r = num[t] * num[t] / (e_var - haa);
    } else {
      const double t1 = num[4 * t], t2 = num[4 * t + 1], b1 = num[4 * t + 2], b2 = num[4 * t + 3];
      r = 1.0 / (e_var - haa) * (t1 * t1 + t2 - b1 * b1 - b2);
    }
  }
  term[t] = r;
}
// out[t] = sum of v[off[t] .. off[t+1]) per channel (nch interleaved values per entry): the segments (contributions to one
// determinant) hold a handful of entries on average, so one thread per (segment, channel) in entry order -- deterministic, and
// 50x faster here than cub's block-per-segment DeviceSegmentedReduce (profiles/r01_launches_pt2_summary.txt)
__global__ void segment_sum_kernel(const double *v, const int32_t *off, int64_t nseg, double *out, int nch) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= nseg * nch) return;
  const int64_t g = t / nch;
  const int c = (int)(t % nch);
  double acc = 0.0;
  for (int32_t k = off[g]; k < off[g + 1]; k++) acc += v[(int64_t)k * nch + c];
  out[t] = acc;
}
__global__ void gather_rows_kernel(const double *src, const int32_t *idx, double *dst, int64_t m, int nch) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= m * nch) return;
  dst[t] = src[(int64_t)idx[t / nch] * nch + t % nch];
}
// sort (a,b,v) by label and sum the values of equal determinants -> (ra, rb, rv), mout distinct determinants; v holds nch
// interleaved values per entry
template <int NW>
static int reduce_by_det(int norb, DevBuf<uint64_t> &a, DevBuf<uint64_t> &b, DevBuf<double> &v, int64_t m, DevBuf<uint64_t> &ra, DevBuf<uint64_t> &rb,
                         DevBuf<double> &rv, int64_t &mout, cudaStream_t s, int nch = 1) {
  mout = 0;
  if (m == 0) return 0;
  if (m >= ((1ll << 31) - 1) / nch) { set_error("pt2: %lld (determinant, contribution) pairs exceed the 32-bit segment offsets; lower the work per call (larger eps_pt)", (long long)m); return 2; }
  DevBuf<int32_t> idx, flag, sel, num;
  DevBuf<uint64_t> sa, sb;
  DevBuf<double> sv;
  SQ_CHECK(idx.alloc(m));
  SQ_CHECK(sort_pairs_index(NW, norb, a.p, b.p, idx.p, m, s));
  SQ_CHECK(sa.alloc(m * NW));
  SQ_CHECK(sb.alloc(m * NW));
  SQ_CHECK(sv.alloc(m * nch));
  SQ_CHECK(gather_strings(NW, a.p, idx.p, sa.p, m, s));
  SQ_CHECK(gather_strings(NW, b.p, idx.p, sb.p, m, s));
  gather_rows_kernel<<<(unsigned)div_up(m * nch, 256), 256, 0, s>>>(v.p, idx.p, sv.p, m, nch);
  SQ_LAUNCH_CHECK();
  SQ_CHECK(flag.alloc(m));
  uniq_flag_kernel<NW><<<(unsigned)div_up(m, 256), 256, 0, s>>>(sa.p, sb.p, flag.p, m);
  SQ_LAUNCH_CHECK();
  SQ_CHECK(sel.alloc(m + 1));
  SQ_CHECK(num.alloc(1));
  cub::CountingInputIterator<int32_t> it(0);
  size_t tb = 0;
  cub::DeviceSelect::Flagged(nullptr, tb, it, flag.p, sel.p, num.p, (int)m, s);
  DevBuf<char> tmp;
  SQ_CHECK(tmp.alloc((int64_t)tb + 16));
  SQ_CUDA(cub::DeviceSelect::Flagged(tmp.p, tb, it, flag.p, sel.p, num.p, (int)m, s));
  g_launch_count += 2;
  int32_t k = 0;
  SQ_CUDA(cudaMemcpyAsync(&k, num.p, 4, cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  mout = k;
  set_i32_kernel<<<1, 1, 0, s>>>(sel.p + mout, (int32_t)m);  // closing offset of the last segment
  SQ_LAUNCH_CHECK();
  SQ_CHECK(rv.alloc(mout * nch));
  segment_sum_kernel<<<(unsigned)div_up(mout * nch, 256), 256, 0, s>>>(sv.p, sel.p, mout, rv.p, nch);
  SQ_LAUNCH_CHECK();
  SQ_CHECK(ra.alloc(mout * NW));
  SQ_CHECK(rb.alloc(mout * NW));
  SQ_CHECK(gather_strings(NW, sa.p, sel.p, ra.p, mout, s));
  SQ_CHECK(gather_strings(NW, sb.p, sel.p, rb.p, mout, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// The screened sum over the connections of a GENERATING set (gu, gd, gc[, gw]: all determinants of the variational list for the
// deterministic correction, the distinct sampled determinants with their count/probability ratios for one stochastic sample),
// with membership tested against the label-sorted variational list (sup, sdn), both resident on the device.  The generating
// arrays are consumed (replaced by this rank's round-robin share under N > 1 ranks).
template <int NW>
static int pt2_core(sqmc_b200_handle *h, int64_t n_var, const uint64_t *sup, const uint64_t *sdn, int64_t n, DevBuf<uint64_t> &up, DevBuf<uint64_t> &dn,
                    DevBuf<double> &dc, DevBuf<double> &dw, int nch, int n_mc, double var_energy, double eps_pt, double eps_pt_big, double *delta_out,
                    int64_t *nconn_out) {
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  const bool use_hb = T.model == MODEL_CHEM && NW == 1 && T.norb <= 64;
  if (use_hb) SQ_CHECK(hb_build(h));
  if (nch == 1) {  // no upper bound on |H| in the PT sum; the fourth array of the round-robin deal doubles as min_H
    SQ_CHECK(dw.alloc(std::max<int64_t>(n, 1)));
    fill_double_kernel<<<(unsigned)div_up(std::max<int64_t>(n, 1), 256), 256, 0, s>>>(dw.p, n, 9.e99);
    SQ_LAUNCH_CHECK();
  }
  SQ_CHECK(shard_round_robin<NW>(up, dn, dc, dw, n, n, s));  // n = this rank's share; partial sums are merged below
  DevBuf<double> dm;
  if (nch == 4) {
    SQ_CHECK(dm.alloc(std::max<int64_t>(n, 1)));
    fill_double_kernel<<<(unsigned)div_up(std::max<int64_t>(n, 1), 256), 256, 0, s>>>(dm.p, n, 9.e99);
    SQ_LAUNCH_CHECK();
  }
  SelCtx<NW> S{T, h->d_orbsym, up.p, dn.p, dc.p, nch == 4 ? dm.p : dw.p, eps_pt, n,
               {use_hb ? h->d_hb_val[0] : nullptr, use_hb ? h->d_hb_val[1] : nullptr}, {use_hb ? h->d_hb_rs[0] : nullptr, use_hb ? h->d_hb_rs[1] : nullptr},
               nch == 4 ? dw.p : nullptr, (double)(n_mc - 1), eps_pt_big};
  const int c2bytes = (T.model == MODEL_CHEM) ? (T.norb + 1) * (T.norb + 1) * 4 : 0;
  DevBuf<int32_t> counts;
  SQ_CHECK(counts.alloc(n + 1));
  SQ_CUDA(cudaMemsetAsync(counts.p, 0, (n + 1) * sizeof(int32_t), s));
  if (n > 0) {
    SQ_MODEL_DISPATCH(T, SQ_CUDA((allow_dynamic_smem(select_kernel<NW, false, 0, kModel, kTS>, c2bytes))));
    SQ_MODEL_DISPATCH(T, (select_kernel<NW, false, 0, kModel, kTS><<<(unsigned)div_up(n * 32, 128), 128, c2bytes, s>>>(S, 0, n, counts.p, nullptr, nullptr, nullptr, nullptr)));
    SQ_LAUNCH_CHECK();
  }
  std::vector<int32_t> hc(n + 1);
  SQ_CUDA(cudaMemcpyAsync(hc.data(), counts.p, (n + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  std::vector<int64_t> prefix(n + 1, 0);
  for (int64_t i = 0; i < n; i++) prefix[i + 1] = prefix[i] + hc[i];
  // chunks of determinants bounded by generated connections; per chunk: fill, sort, sum per determinant; the partial sums
  // of all chunks are concatenated and reduced once more at the end
  const int64_t kChunk = (1ll << 27) / nch;
  DevBuf<uint64_t> acc_a, acc_b;
  DevBuf<double> acc_v;
  int64_t acc_n = 0, acc_cap = 0;
  int64_t i0 = 0;
  while (i0 < n) {
    int64_t i1 = std::upper_bound(prefix.begin() + i0 + 1, prefix.end(), prefix[i0] + kChunk) - prefix.begin() - 1;
    if (i1 <= i0) i1 = i0 + 1;
    if (i1 > n) i1 = n;
    const int64_t m = prefix[i1] - prefix[i0];
    if (m >= (1ll << 31) / nch) { set_error("pt2: one determinant generates too many connections"); return 2; }
    DevBuf<uint64_t> ca, cb, ra, rb;
    DevBuf<double> cv, rv;
    DevBuf<int64_t> optr;
    SQ_CHECK(ca.alloc(std::max<int64_t>(m, 1) * NW));
    SQ_CHECK(cb.alloc(std::max<int64_t>(m, 1) * NW));
    SQ_CHECK(cv.alloc(std::max<int64_t>(m, 1) * nch));
    SQ_CHECK(optr.alloc(i1 - i0 + 1));
    std::vector<int64_t> hp(prefix.begin() + i0, prefix.begin() + i1 + 1);
    for (auto &x : hp) x -= prefix[i0];
    SQ_CUDA(cudaMemcpyAsync(optr.p, hp.data(), hp.size() * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    const unsigned g = (unsigned)div_up((i1 - i0) * 32, 128);
    if (nch == 1) {
      SQ_MODEL_DISPATCH(T, SQ_CUDA((allow_dynamic_smem(select_kernel<NW, true, 1, kModel, kTS>, c2bytes))));
      SQ_MODEL_DISPATCH(T, (select_kernel<NW, true, 1, kModel, kTS><<<g, 128, c2bytes, s>>>(S, i0, i1, nullptr, optr.p, ca.p, cb.p, cv.p)));
    } else {
      SQ_MODEL_DISPATCH(T, SQ_CUDA((allow_dynamic_smem(select_kernel<NW, true, 4, kModel, kTS>, c2bytes))));
      SQ_MODEL_DISPATCH(T, (select_kernel<NW, true, 4, kModel, kTS><<<g, 128, c2bytes, s>>>(S, i0, i1, nullptr, optr.p, ca.p, cb.p, cv.p)));
    }
    SQ_LAUNCH_CHECK();
    SQ_CUDA(cudaStreamSynchronize(s));
    int64_t mu = 0;
    SQ_CHECK(reduce_by_det<NW>(T.norb, ca, cb, cv, m, ra, rb, rv, mu, s, nch));
    if (mu > 0) {
      // the accumulated partial sums are reduced again whenever they pass kAccReduce entries (the reference batches its PT
      // for the same reason), and the buffers grow geometrically instead of being re-allocated for every chunk
      const int64_t kAccReduce = (1ll << 28) / nch;
      if (acc_n > 0 && acc_n + mu > kAccReduce) {
        DevBuf<uint64_t> qa, qb;
        DevBuf<double> qv;
        int64_t qn = 0;
        SQ_CHECK(reduce_by_det<NW>(T.norb, acc_a, acc_b, acc_v, acc_n, qa, qb, qv, qn, s, nch));
        acc_a.release(); acc_b.release(); acc_v.release();
        acc_a.p = qa.take(); acc_b.p = qb.take(); acc_v.p = qv.take();
        acc_n = qn;
        acc_cap = qn;
      }
      if (acc_n + mu >= ((1ll << 31) - 1) / nch) { set_error("pt2: more than 2^31 distinct connected determinants"); return 2; }
      if (acc_n + mu > acc_cap) {
        const int64_t cap = std::max<int64_t>(acc_n + mu, 2 * acc_cap);
        DevBuf<uint64_t> na, nb;
        DevBuf<double> nv;
        SQ_CHECK(na.alloc(cap * NW));
        SQ_CHECK(nb.alloc(cap * NW));
        SQ_CHECK(nv.alloc(cap * nch));
        if (acc_n) {
          SQ_CUDA(cudaMemcpyAsync(na.p, acc_a.p, acc_n * NW * 8, cudaMemcpyDeviceToDevice, s));
          SQ_CUDA(cudaMemcpyAsync(nb.p, acc_b.p, acc_n * NW * 8, cudaMemcpyDeviceToDevice, s));
          SQ_CUDA(cudaMemcpyAsync(nv.p, acc_v.p, acc_n * nch * 8, cudaMemcpyDeviceToDevice, s));
        }
        SQ_CUDA(cudaStreamSynchronize(s));
        acc_a.release(); acc_b.release(); acc_v.release();
        acc_a.p = na.take(); acc_b.p = nb.take(); acc_v.p = nv.take();
        acc_cap = cap;
      }
      SQ_CUDA(cudaMemcpyAsync(acc_a.p + acc_n * NW, ra.p, mu * NW * 8, cudaMemcpyDeviceToDevice, s));
      SQ_CUDA(cudaMemcpyAsync(acc_b.p + acc_n * NW, rb.p, mu * NW * 8, cudaMemcpyDeviceToDevice, s));
      SQ_CUDA(cudaMemcpyAsync(acc_v.p + acc_n * nch, rv.p, mu * nch * 8, cudaMemcpyDeviceToDevice, s));
      SQ_CUDA(cudaStreamSynchronize(s));
      acc_n += mu;
    }
    i0 = i1;
  }
  DevBuf<uint64_t> fa, fb;
  DevBuf<double> fv;
  int64_t nf = 0;
  SQ_CHECK(reduce_by_det<NW>(T.norb, acc_a, acc_b, acc_v, acc_n, fa, fb, fv, nf, s, nch));
  if (G.nranks > 1) {  // all-gather of (determinant, partial sums), one more reduction: identical on every rank
    DevBuf<uint64_t> ca, cb, ma, mb;
    DevBuf<double> cv, mv;
    int64_t tot = 0, nm = 0;
    SQ_CHECK(allgather_lists<NW>(fa.p, fb.p, fv.p, nf, ca, cb, cv, tot, s, nch));
    if (tot > 0) SQ_CHECK(reduce_by_det<NW>(T.norb, ca, cb, cv, tot, ma, mb, mv, nm, s, nch));
    fa.release(); fb.release(); fv.release();
    fa.p = ma.take(); fb.p = mb.take(); fv.p = mv.take();
    nf = nm;
  }
  double delta = 0.0;
  if (nf > 0) {
    DevBuf<int32_t> ext;
    DevBuf<double> term, total;
    SQ_CHECK(ext.alloc(nf));
    SQ_CHECK(term.alloc(nf));
    SQ_CHECK(total.alloc(1));
    const unsigned g = (unsigned)div_up(nf, 256);
    uniq_flag_kernel<NW><<<g, 256, 0, s>>>(fa.p, fb.p, ext.p, nf);   // all ones: the list is already unique
    SQ_LAUNCH_CHECK();
    not_in_list_kernel<NW><<<g, 256, 0, s>>>(fa.p, fb.p, sup, sdn, n_var, ext.p, nf);  // 0 for variational determinants
    SQ_LAUNCH_CHECK();
    if (nch == 1) {
      SQ_MODEL_DISPATCH(T, (pt_term_kernel<NW, kModel, kTS, 1><<<g, 256, 0, s>>>(T, fa.p, fb.p, fv.p, ext.p, var_energy, term.p, nf)));
    } else {
      SQ_MODEL_DISPATCH(T, (pt_term_kernel<NW, kModel, kTS, 4><<<g, 256, 0, s>>>(T, fa.p, fb.p, fv.p, ext.p, var_energy, term.p, nf)));
    }
    SQ_LAUNCH_CHECK();
    size_t tb = 0;
    cub::DeviceReduce::Sum(nullptr, tb, term.p, total.p, (int)nf, s);
    DevBuf<char> tmp;
    SQ_CHECK(tmp.alloc((int64_t)tb + 16));
    SQ_CUDA(cub::DeviceReduce::Sum(tmp.p, tb, term.p, total.p, (int)nf, s));
    g_launch_count += 1;
    SQ_CUDA(cudaMemcpyAsync(&delta, total.p, sizeof(double), cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
  }
  *delta_out = delta;
  *nconn_out = nf;
  return 0;
}

// upload a determinant list and keep a label-sorted copy (the membership test's search list)
template <int NW>
static int upload_sorted(int norb, int64_t n, const void *dets_up, const void *dets_dn, DevBuf<uint64_t> &up, DevBuf<uint64_t> &dn, DevBuf<uint64_t> &sup,
                         DevBuf<uint64_t> &sdn, cudaStream_t s) {
  SQ_CHECK(up.alloc(n * NW));
  SQ_CHECK(dn.alloc(n * NW));
  SQ_CHECK(upload_dets(NW, norb, dets_up, up.p, n, s));
  SQ_CHECK(upload_dets(NW, norb, dets_dn, dn.p, n, s));
  DevBuf<int32_t> idx;
  SQ_CHECK(idx.alloc(n));
  SQ_CHECK(sort_pairs_index(NW, norb, up.p, dn.p, idx.p, n, s));
  SQ_CHECK(sup.alloc(n * NW));
  SQ_CHECK(sdn.alloc(n * NW));
  SQ_CHECK(gather_strings(NW, up.p, idx.p, sup.p, n, s));
  SQ_CHECK(gather_strings(NW, dn.p, idx.p, sdn.p, n, s));
  return 0;
}

template <int NW>
static int pt2_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy, double eps_pt,
                    double *delta_out, int64_t *nconn_out) {
  cudaStream_t s = G.stream;
  DevBuf<uint64_t> up, dn, sup, sdn;
  DevBuf<double> dc, dw;
  SQ_CHECK(upload_sorted<NW>(h->T.norb, n, dets_up, dets_dn, up, dn, sup, sdn, s));
  SQ_CHECK(dc.alloc(n));
  SQ_CUDA(cudaMemcpyAsync(dc.p, wts, n * sizeof(double), cudaMemcpyHostToDevice, s));
  return pt2_core<NW>(h, n, sup.p, sdn.p, n, up, dn, dc, dw, 1, 0, var_energy, eps_pt, 0.0, delta_out, nconn_out);
}

static int pt2_check(sqmc_b200_handle *h, int64_t n, double eps_pt, const char *who) {
  if (n <= 0) { set_error("%s: n must be positive", who); return 2; }
  if (h->T.model == MODEL_HUBBARDK) { set_error("%s: only chem and heg", who); return 2; }
  if (h->T.model == MODEL_CHEM && !h->d_orbsym) { set_error("%s: call sqmc_b200_system_orbital_symmetries first", who); return 2; }
  if (!(eps_pt > 0.0)) { set_error("%s: eps_pt must be > 0 (the screened sum, hci.f90:1143)", who); return 2; }
  return 0;
}

int pt2(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy, double eps_pt,
        double *delta_out, int64_t *nconn_out) {
  SQ_CHECK(pt2_check(h, n, eps_pt, "pt2"));
  return h->NW == 1 ? pt2_impl<1>(h, n, dets_up, dets_dn, wts, var_energy, eps_pt, delta_out, nconn_out)
                    : pt2_impl<2>(h, n, dets_up, dets_dn, wts, var_energy, eps_pt, delta_out, nconn_out);
}

// ------------------------------------------------------------------ stochastic second-order correction (second_order_pt_alias, hci.f90:1314-1684)
// One sample = find_doubly_excited(sampled determinants, n_mc, w_over_p, eps_var_pt = eps_pt, eps_var_pt_big = eps_pt_big)
// (semistoch.f90:1579-2231, the term1/term2 forms at :2044-2060) + the k loop of hci.f90:1616-1632, divided by n_mc (n_mc - 1)
// (:1654).  The variational list stays on the device for all samples of one call of pt2_alias.
template <int NW>
static int pt2_sample_dev(sqmc_b200_handle *h, int64_t n_var, const uint64_t *sup, const uint64_t *sdn, int64_t m, const void *s_up, const void *s_dn,
                          const double *s_c, const double *s_wop, int n_mc, double var_energy, double eps_pt, double eps_pt_big, double *e_out,
                          int64_t *nconn_out) {
  cudaStream_t s = G.stream;
  DevBuf<uint64_t> up, dn;
  DevBuf<double> dc, dw;
  SQ_CHECK(up.alloc(m * NW));
  SQ_CHECK(dn.alloc(m * NW));
  SQ_CHECK(upload_dets(NW, h->T.norb, s_up, up.p, m, s));
  SQ_CHECK(upload_dets(NW, h->T.norb, s_dn, dn.p, m, s));
  SQ_CHECK(dc.alloc(m));
  SQ_CHECK(dw.alloc(m));
  SQ_CUDA(cudaMemcpyAsync(dc.p, s_c, m * sizeof(double), cudaMemcpyHostToDevice, s));
  SQ_CUDA(cudaMemcpyAsync(dw.p, s_wop, m * sizeof(double), cudaMemcpyHostToDevice, s));
  double sum = 0.0;
  SQ_CHECK(pt2_core<NW>(h, n_var, sup, sdn, m, up, dn, dc, dw, 4, n_mc, var_energy, eps_pt, eps_pt_big, &sum, nconn_out));
  *e_out = sum / (n_mc * (double)(n_mc - 1));
  return 0;
}

template <int NW>
static int pt2_sample_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int64_t m, const void *s_up, const void *s_dn,
                           const double *s_c, const double *s_wop, int n_mc, double var_energy, double eps_pt, double eps_pt_big, double *e_out,
                           int64_t *nconn_out) {
  DevBuf<uint64_t> up, dn, sup, sdn;
  SQ_CHECK(upload_sorted<NW>(h->T.norb, n, dets_up, dets_dn, up, dn, sup, sdn, G.stream));
  up.release(); dn.release();
  return pt2_sample_dev<NW>(h, n, sup.p, sdn.p, m, s_up, s_dn, s_c, s_wop, n_mc, var_energy, eps_pt, eps_pt_big, e_out, nconn_out);
}

int pt2_sample(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int64_t m, const void *s_up, const void *s_dn, const double *s_c,
               const double *s_wop, int n_mc, double var_energy, double eps_pt, double eps_pt_big, double *e_out, int64_t *nconn_out) {
  SQ_CHECK(pt2_check(h, n, eps_pt, "pt2_sample"));
  if (m <= 0) { set_error("pt2_sample: the sample must hold at least one determinant"); return 2; }
  if (n_mc < 2) { set_error("pt2_sample: n_mc must be >= 2 (the estimator divides by n_mc (n_mc - 1), hci.f90:1654)"); return 2; }
  for (int64_t i = 0; i < m; i++)
    if (s_c[i] == 0.0) { set_error("pt2_sample: sampled determinants must have non-zero coefficients (they are drawn with probability |c|)"); return 2; }
  return h->NW == 1 ? pt2_sample_impl<1>(h, n, dets_up, dets_dn, m, s_up, s_dn, s_c, s_wop, n_mc, var_energy, eps_pt, eps_pt_big, e_out, nconn_out)
                    : pt2_sample_impl<2>(h, n, dets_up, dets_dn, m, s_up, s_dn, s_c, s_wop, n_mc, var_energy, eps_pt, eps_pt_big, e_out, nconn_out);
}

// rannyu (rannyu.f90:53-74): the reference's 48-bit multiplicative congruential generator on four 12-bit digits.  The caller
// hands its current state in (savern) and gets the advanced state back (setrn), so the Fortran driver's random stream continues
// exactly as if second_order_pt_alias had run on the host.
namespace {
struct Rannyu {
  long long l[4];
  double next() {
    const long long m1 = 502, m2 = 1521, m3 = 4071, m4 = 2107, t12 = 4096;
    long long i1 = l[0] * m4 + l[1] * m3 + l[2] * m2 + l[3] * m1;
    long long i2 = l[1] * m4 + l[2] * m3 + l[3] * m2;
    long long i3 = l[2] * m4 + l[3] * m3;
    long long i4 = l[3] * m4;
    l[3] = i4 % t12;
    i3 += i4 / t12;
    l[2] = i3 % t12;
    i2 += i3 / t12;
    l[1] = i2 % t12;
    l[0] = (i1 + i2 / t12) % t12;
    const double s = 2.44140625e-4;
    return s * ((double)l[0] + s * ((double)l[1] + s * ((double)l[2] + s * ((double)l[3]))));
  }
  int random_int(int n) { return (int)(n * next()) + 1; }  // tools.f90:130-149
};
}  // namespace

template <int NW>
static int pt2_alias_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy, double eps_pt,
                          double eps_pt_big, int n_mc, double target_error, int *rng4, int max_samples, double *pt_out, double *sd_out, int *ns_out,
                          double *e_now, int64_t *nconn_out) {
  DevBuf<uint64_t> up, dn, sup, sdn;
  SQ_CHECK(upload_sorted<NW>(h->T.norb, n, dets_up, dets_dn, up, dn, sup, sdn, G.stream));
  up.release(); dn.release();
  // probabilities |c_i| / sum |c| and the alias tables (setup_alias, more_tools.f90:5603-5662); 1-based as in the reference
  const int K = (int)n;
  double norm = 0.0;
  for (int64_t i = 0; i < n; i++) norm += fabs(wts[i]);
  std::vector<double> prob(n), q(K + 1, 0.0);
  std::vector<int> J(K + 1, 0), smaller(K + 1, 0), larger(K + 1, 0);
  int n_s = 0, n_l = 0;
  for (int i = 1; i <= K; i++) {
    prob[i - 1] = fabs(wts[i - 1]) / norm;
    J[i] = i;
    q[i] = K * prob[i - 1];
    if (q[i] < 1.0) smaller[++n_s] = i; else larger[++n_l] = i;
  }
  while (n_s > 0 && n_l > 0) {
    const int small = smaller[n_s], large = larger[n_l];
    J[small] = large;
    q[large] = q[large] + q[small] - 1.0;
    if (q[large] < 1.0) { smaller[n_s] = large; n_l--; } else n_s--;
  }
  Rannyu R;
  for (int k = 0; k < 4; k++) R.l[k] = rng4[k];
  const unsigned char *hu = (const unsigned char *)dets_up, *hd = (const unsigned char *)dets_dn;
  double mean = 0.0, S2 = 0.0, var = 0.0;
  int sample = 1;
  std::vector<int> samples(n_mc);
  std::vector<unsigned char> su, sd;
  std::vector<double> sc, sw;
  for (; sample <= max_samples; sample++) {
    for (int i = 0; i < n_mc; i++) {  // sample_alias (more_tools.f90:5727-5752)
      const int k = R.random_int(K);
      samples[i] = R.next() < q[k] ? k : J[k];
    }
    std::sort(samples.begin(), samples.end());  // sort_and_merge_count_repeats (tools.f90:1574-1602)
    su.clear(); sd.clear(); sc.clear(); sw.clear();
    for (size_t i = 0; i < samples.size();) {
      size_t j = i;
      while (j < samples.size() && samples[j] == samples[i]) j++;
      const int64_t d = samples[i] - 1;
      su.insert(su.end(), hu + 16 * d, hu + 16 * d + 16);
      sd.insert(sd.end(), hd + 16 * d, hd + 16 * d + 16);
      sc.push_back(wts[d]);
      sw.push_back((double)(j - i) / prob[d]);
      i = j;
    }
    double e = 0.0;
    SQ_CHECK(pt2_sample_dev<NW>(h, n, sup.p, sdn.p, (int64_t)sc.size(), su.data(), sd.data(), sc.data(), sw.data(), n_mc, var_energy, eps_pt, eps_pt_big, &e,
                                nconn_out));
    if (e_now) e_now[sample - 1] = e;
    const double oldM = mean;  // welford (tools.f90:1761-1778)
    mean = mean + (e - mean) / sample;
    S2 = S2 + (e - mean) * (e - oldM);
    var = S2 / (double)(sample - 1) / sample;
    if (sample >= 10 && var < target_error * target_error) break;  // hci.f90:1670
  }
  if (sample > max_samples) sample = max_samples;
  for (int k = 0; k < 4; k++) rng4[k] = (int)R.l[k];
  *pt_out = mean;
  *sd_out = sqrt(var);
  *ns_out = sample;
  return 0;
}

int pt2_alias(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *wts, double var_energy, double eps_pt, double eps_pt_big,
              int n_mc, double target_error, int *rng4, int max_samples, double *pt_out, double *sd_out, int *ns_out, double *e_now, int64_t *nconn_out) {
  SQ_CHECK(pt2_check(h, n, eps_pt, "pt2_alias"));
  if (n >= (1ll << 31) - 1) { set_error("pt2_alias: the reference samples with 32-bit indices (hci.f90:1365)"); return 2; }
  if (n_mc < 2) { set_error("pt2_alias: n_mc must be >= 2"); return 2; }
  if (max_samples < 1) { set_error("pt2_alias: max_samples must be >= 1"); return 2; }
  if (!(rng4[3] & 1)) { set_error("pt2_alias: the last digit of the rannyu state must be odd (setrn, rannyu.f90:19)"); return 2; }
  double norm = 0.0;
  for (int64_t i = 0; i < n; i++) norm += fabs(wts[i]);
  if (!(norm > 0.0)) { set_error("pt2_alias: all coefficients are zero"); return 2; }
  return h->NW == 1 ? pt2_alias_impl<1>(h, n, dets_up, dets_dn, wts, var_energy, eps_pt, eps_pt_big, n_mc, target_error, rng4, max_samples, pt_out, sd_out,
                                        ns_out, e_now, nconn_out)
                    : pt2_alias_impl<2>(h, n, dets_up, dets_dn, wts, var_energy, eps_pt, eps_pt_big, n_mc, target_error, rng4, max_samples, pt_out, sd_out,
                                        ns_out, e_now, nconn_out);
}

int hci_select(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, const double *coeffs, double *min_H, double eps_var,
               int64_t *n_new_out) {
  if (n <= 0) { set_error("hci_select: n must be positive"); return 2; }
  if (h->T.model == MODEL_HUBBARDK) { set_error("hci_select: only chem and heg (hci.f90:1073-1075)"); return 2; }
  if (h->T.model == MODEL_CHEM && !h->d_orbsym) { set_error("hci_select: call sqmc_b200_system_orbital_symmetries first"); return 2; }
  if (!(eps_var >= 0.0)) { set_error("hci_select: eps_var must be >= 0 (hci.f90:932)"); return 2; }
  return h->NW == 1 ? select_impl<1>(h, n, dets_up, dets_dn, coeffs, min_H, eps_var, n_new_out)
                    : select_impl<2>(h, n, dets_up, dets_dn, coeffs, min_H, eps_var, n_new_out);
}

}  // namespace sqmc
