// elements.cuh -- Hamiltonian matrix elements between bit-packed determinants.
//
// Device restatement of the reference's element routines; the order of every
// floating-point operation is kept so that values (and therefore the
// abs(H) > 1e-12 pattern test, chemistry.f90:9901) are bit-identical to the
// reference's CPU build.  This translation unit MUST be compiled with
// --fmad=false (the reference is gfortran -O3 on baseline x86-64: no FMA).
//
//   chem   : chemistry.f90:1260-2001 (hamiltonian_chem, one_body, two_body,
//            one_body_single, two_body_single, two_body_double), :1323-1377
//            (hamiltonian_chem_time_sym), :7162-7227 (excitation_level),
//            :9106-9134 (integral_index); tools.f90:1294-1396 (permutation factors)
//   heg    : heg.f90:775-1010 (find_set_bits, get_gamma_exp, hamiltonian_heg)
//   hubbard: hubbard.f90:2866-2924 (hamiltonian_hubbard_k), :9676-9722
#pragma once
#include "common.cuh"

namespace sqmc {

enum ModelKind { MODEL_CHEM = 0, MODEL_HEG = 1, MODEL_HUBBARDK = 2 };

struct ModelTables {
  int model;
  int norb, nup, ndn;
  int time_sym, z;
  int hf_to_psit;  // Hubbard builder: row/column 1 reduced to a zero diagonal (hubbard.f90:9636-9643)
  // chem
  const double *integrals;   // device; Fortran integrals(1:nint) stored 0-based
  const int32_t *combine_2;  // device; (norb+1)x(norb+1) column-major, values as in Fortran
  int64_t nint;
  double enuc, sqrt2, sqrt2inv;
  // heg
  int n_dim;
  const double *k_vectors;  // device; (n_dim, norb) column-major
  double length_cell;
  // hubbard k-space
  int l_x, l_y;
  const int32_t *hk_vectors;  // device; (2, nsites)
  const double *k_energies;   // device
  double ubyn;
};

// ---------------------------------------------------------------------------
// fermionic phases (tools.f90:1294-1396)
// ---------------------------------------------------------------------------
// electrons of `det` strictly between bit positions lo < hi
template <int NW>
__device__ __forceinline__ int count_between(const Bits<NW> &det, int lo, int hi) {
  Bits<NW> m = b_xor(b_maskr<NW>(hi), b_maskr<NW>(lo + 1));  // bits lo+1 .. hi-1
  return b_popc(b_and(det, m));
}
// permutation_factor for two strings one excitation apart
template <int NW>
__device__ __forceinline__ int permutation_factor(const Bits<NW> &d1, const Bits<NW> &d2) {
  int a = b_ctz(b_andnot(d1, d2)), b = b_ctz(b_andnot(d2, d1));
  int lo = min(a, b), hi = max(a, b);
  return (count_between(d1, lo, hi) & 1) ? -1 : 1;
}
template <int NW>
__device__ __forceinline__ void permutation_factor2(const Bits<NW> &di, const Bits<NW> &dj, int &gamma, int &fi, int &si,
                                                    int &fj, int &sj) {
  Bits<NW> diff = b_andnot(di, dj);
  fi = b_ctz(diff);
  b_clear(diff, fi);
  si = b_ctz(diff);
  diff = b_andnot(dj, di);
  fj = b_ctz(diff);
  b_clear(diff, fj);
  sj = b_ctz(diff);
  Bits<NW> m = b_xor(b_xor(b_maskr<NW>(fi), b_maskr<NW>(fj)), b_xor(b_maskr<NW>(si), b_maskr<NW>(sj)));
  gamma = (b_popc(b_and(b_and(di, dj), m)) & 1) ? -1 : 1;
}
// excitation_level (chemistry.f90:7162): 0,1,2 or -1
template <int NW>
__device__ __forceinline__ int excitation_level(const Bits<NW> &iu, const Bits<NW> &id, const Bits<NW> &ju, const Bits<NW> &jd) {
  int l = b_popc(b_andnot(iu, ju)) + b_popc(b_andnot(id, jd));
  return l > 2 ? -1 : l;
}

// ---------------------------------------------------------------------------
// chem
// ---------------------------------------------------------------------------
struct ChemCtx {
  const double *ints;
  const int32_t *c2;  // may point to shared memory
  int n1;             // norb + 1
  double enuc, sqrt2, sqrt2inv;
  int z;
  __device__ __forceinline__ double I(int p, int q, int r, int s) const {  // 1-based orbital numbers
    long long a = c2[(q - 1) * n1 + (p - 1)], b = c2[(s - 1) * n1 + (r - 1)];
    long long idx = (a > b) ? (a * (a - 1)) / 2 + b : (b * (b - 1)) / 2 + a;
    return __ldg(ints + (idx - 1));
  }
};

template <int NW>
__device__ __forceinline__ double chem_one_body(const ChemCtx &C, const Bits<NW> &up, const Bits<NW> &dn) {
  double energy = 0.0;
  Bits<NW> det = up;
  while (!b_is_zero(det)) {
    int i = b_ctz(det) + 1;
    energy = energy + C.I(i, i, C.n1, C.n1);
    b_clear_lowest(det);
  }
  if (b_eq(dn, up)) {
    energy = energy * 2.0;
  } else {
    det = dn;
    while (!b_is_zero(det)) {
      int i = b_ctz(det) + 1;
      energy = energy + C.I(i, i, C.n1, C.n1);
      b_clear_lowest(det);
    }
  }
  return energy;
}

template <int NW>
__device__ __forceinline__ double chem_two_body(const ChemCtx &C, const Bits<NW> &up, const Bits<NW> &dn) {
  double exchange = 0.0, direct = 0.0;
  // exchange: up pairs i<j ascending
  Bits<NW> di = up;
  while (!b_is_zero(di)) {
    int i = b_ctz(di) + 1;
    b_clear_lowest(di);
    Bits<NW> dj = di;
    while (!b_is_zero(dj)) {
      int j = b_ctz(dj) + 1;
      b_clear_lowest(dj);
      exchange = exchange - C.I(i, j, j, i);
    }
  }
  if (b_eq(dn, up)) {
    exchange = exchange * 2.0;
  } else {
    di = dn;
    while (!b_is_zero(di)) {
      int i = b_ctz(di) + 1;
      b_clear_lowest(di);
      Bits<NW> dj = di;
      while (!b_is_zero(dj)) {
        int j = b_ctz(dj) + 1;
        b_clear_lowest(dj);
        exchange = exchange - C.I(i, j, j, i);
      }
    }
  }
  // direct: i ascending over all orbitals; for up(i): up j>i then all dn j; for dn(i): dn j>i
  Bits<NW> uni;
#pragma unroll
  for (int k = 0; k < NW; k++) uni.w[k] = up.w[k] | dn.w[k];
  while (!b_is_zero(uni)) {
    int i0 = b_ctz(uni);
    b_clear_lowest(uni);
    int i = i0 + 1;
    if (b_test(up, i0)) {
      Bits<NW> dj = b_andnot(up, b_maskr<NW>(i));  // up orbitals j > i
      while (!b_is_zero(dj)) {
        int j = b_ctz(dj) + 1;
        b_clear_lowest(dj);
        direct = direct + C.I(i, i, j, j);
      }
      dj = dn;
      while (!b_is_zero(dj)) {
        int j = b_ctz(dj) + 1;
        b_clear_lowest(dj);
        direct = direct + C.I(i, i, j, j);
      }
    }
    if (b_test(dn, i0)) {
      Bits<NW> dj = b_andnot(dn, b_maskr<NW>(i));
      while (!b_is_zero(dj)) {
        int j = b_ctz(dj) + 1;
        b_clear_lowest(dj);
        direct = direct + C.I(i, i, j, j);
      }
    }
  }
  return exchange + direct;
}

template <int NW>
__device__ __forceinline__ double chem_single(const ChemCtx &C, const Bits<NW> &iu, const Bits<NW> &id, const Bits<NW> &ju, const Bits<NW> &jd) {
  // one_body_single + two_body_single (chemistry.f90:1439-1480,1845-1930)
  bool up_moves = !b_eq(iu, ju);
  // selected by value (word-wise selects): a reference picked at run time would force the strings into local memory
  Bits<NW> same_i, same_j, other;
#pragma unroll
  for (int k = 0; k < NW; k++) {
    same_i.w[k] = up_moves ? iu.w[k] : id.w[k];
    same_j.w[k] = up_moves ? ju.w[k] : jd.w[k];
    other.w[k] = up_moves ? id.w[k] : iu.w[k];
  }
  int i_bit = b_ctz(b_andnot(same_i, same_j)) + 1, j_bit = b_ctz(b_andnot(same_j, same_i)) + 1;
  int pf = permutation_factor(same_i, same_j);
  double one_body = pf * C.I(i_bit, j_bit, C.n1, C.n1);
  double energy = 0.0;
  Bits<NW> det = same_i;
  while (!b_is_zero(det)) {
    int i = b_ctz(det) + 1;
    b_clear_lowest(det);
    if (i != i_bit && i != j_bit) energy = energy - C.I(i_bit, i, i, j_bit) + C.I(i_bit, j_bit, i, i);
  }
  det = other;
  while (!b_is_zero(det)) {
    int i = b_ctz(det) + 1;
    b_clear_lowest(det);
    energy = energy + C.I(i_bit, j_bit, i, i);
  }
  double two_body = pf * energy;
  return one_body + two_body;
}

template <int NW>
__device__ __forceinline__ double chem_double(const ChemCtx &C, const Bits<NW> &iu, const Bits<NW> &id, const Bits<NW> &ju, const Bits<NW> &jd) {
  int gamma, fi, si, fj, sj;
  if (b_eq(iu, ju)) {
    permutation_factor2(id, jd, gamma, fi, si, fj, sj);
    return gamma * (C.I(fi + 1, fj + 1, si + 1, sj + 1) - C.I(fi + 1, sj + 1, si + 1, fj + 1));
  } else if (b_eq(id, jd)) {
    permutation_factor2(iu, ju, gamma, fi, si, fj, sj);
    return gamma * (C.I(fi + 1, fj + 1, si + 1, sj + 1) - C.I(fi + 1, sj + 1, si + 1, fj + 1));
  } else {
    fi = b_ctz(b_andnot(iu, ju));
    fj = b_ctz(b_andnot(ju, iu));
    si = b_ctz(b_andnot(id, jd));
    sj = b_ctz(b_andnot(jd, id));
    return (permutation_factor(iu, ju) * permutation_factor(id, jd)) * C.I(fi + 1, fj + 1, si + 1, sj + 1);
  }
}

template <int NW>
__device__ __forceinline__ double chem_hamiltonian_level(const ChemCtx &C, const Bits<NW> &iu, const Bits<NW> &id, const Bits<NW> &ju,
                                         const Bits<NW> &jd, int level) {
  if (level == 0) {
    double e1 = chem_one_body(C, iu, id);
    double e2 = chem_two_body(C, iu, id);
    return e1 + e2 + C.enuc;
  } else if (level == 1) {
    return chem_single(C, iu, id, ju, jd);
  } else if (level == 2) {
    return chem_double(C, iu, id, ju, jd);
  }
  return 0.0;
}

template <int NW>
__device__ __forceinline__ double chem_hamiltonian_time_sym(const ChemCtx &C, const Bits<NW> &iu, const Bits<NW> &id, const Bits<NW> &ju,
                                            const Bits<NW> &jd) {
  double m1 = 0.0, m2 = 0.0, norm_ketinv = 1.0, norm_bra = 1.0;
  bool check = true;
  if (b_eq(ju, jd)) norm_ketinv = C.sqrt2inv;
  if (b_eq(iu, id)) {
    norm_bra = C.sqrt2;
    check = false;
  }
  int lvl = excitation_level(iu, id, ju, jd);
  if (lvl >= 0) m1 = chem_hamiltonian_level(C, iu, id, ju, jd, lvl);
  if (check) {
    if (!b_eq(ju, jd)) {
      lvl = excitation_level(id, iu, ju, jd);
      if (lvl >= 0) m2 = chem_hamiltonian_level(C, id, iu, ju, jd, lvl);
    } else {
      m2 = m1;
    }
  }
  return (norm_bra * norm_ketinv) * (m1 + (C.z * m2));
}

// ---------------------------------------------------------------------------
// heg
// ---------------------------------------------------------------------------
struct HegCtx {
  const double *kv;  // (n_dim, norb)
  int n_dim;
  double length_cell;
  __device__ __forceinline__ double k(int orb1, int d) const { return kv[(orb1 - 1) * n_dim + d]; }
  // n_dim is 2 or 3: loops are written over 3 fixed components with the third one guarded, so nothing is indexed dynamically
  __device__ __forceinline__ double ksum2(int p) const {
    double s = 0.0;
#pragma unroll
    for (int d = 0; d < 3; d++)
      if (d < n_dim) s += k(p, d) * k(p, d);
    return s;
  }
  __device__ __forceinline__ double kdiff2(int p, int q) const {
    double s = 0.0;
#pragma unroll
    for (int d = 0; d < 3; d++)
      if (d < n_dim) {
        double t = k(p, d) - k(q, d);
        s += t * t;
      }
    return s;
  }
};

// get_gamma_exp (heg.f90:811-842): for each eor bit that is set in det, the number of
// electrons of det below it
template <int NW>
__device__ __forceinline__ int heg_gamma_exp(const Bits<NW> &det, const Bits<NW> &eor) {
  int g = 0;
  Bits<NW> e = b_and(eor, det);
  while (!b_is_zero(e)) {
    int o = b_ctz(e);
    b_clear_lowest(e);
    g += b_popc(b_and(det, b_maskr<NW>(o)));
  }
  return g;
}

template <int NW>
__device__ __forceinline__ double heg_hamiltonian(const HegCtx &H, const Bits<NW> &iu, const Bits<NW> &id, const Bits<NW> &ju, const Bits<NW> &jd) {
  const double FOUR_PI = 4.0 * 3.14159265358979323846264338327950288;
  const double EPSILON = 1.0e-15;
  double L3 = H.length_cell * H.length_cell * H.length_cell;
  if (b_eq(iu, ju) && b_eq(id, jd)) {
    double me = 0.0;
    Bits<NW> d = iu;
    while (!b_is_zero(d)) {
      int p = b_ctz(d) + 1;
      b_clear_lowest(d);
      me = me + H.ksum2(p) * 0.5;
    }
    d = id;
    while (!b_is_zero(d)) {
      int p = b_ctz(d) + 1;
      b_clear_lowest(d);
      me = me + H.ksum2(p) * 0.5;
    }
    double pot = 0.0;
    for (int spin = 0; spin < 2; spin++) {
      Bits<NW> di = spin == 0 ? iu : id;
      while (!b_is_zero(di)) {
        int p = b_ctz(di) + 1;
        b_clear_lowest(di);
        Bits<NW> dj = di;
        while (!b_is_zero(dj)) {
          int q = b_ctz(dj) + 1;
          b_clear_lowest(dj);
          pot = pot + FOUR_PI / H.kdiff2(p, q);
        }
      }
    }
    return me - pot / L3;
  }
  Bits<NW> eu = b_xor(iu, ju), ed = b_xor(id, jd);
  int n_eu = b_popc(eu), n_ed = b_popc(ed);
  if (n_eu + n_ed != 4) return 0.0;
  double mom[3] = {0.0, 0.0, 0.0};
  bool pset = false, qset = false, sset = false;
  int orb_p = 0, orb_q = 0, orb_s = 0;
  for (int spin = 0; spin < 2; spin++) {
    Bits<NW> e, di;
#pragma unroll
    for (int k = 0; k < NW; k++) {
      e.w[k] = spin == 0 ? eu.w[k] : ed.w[k];
      di.w[k] = spin == 0 ? iu.w[k] : id.w[k];
    }
    while (!b_is_zero(e)) {
      int o = b_ctz(e);
      b_clear_lowest(e);
      int orb = o + 1;
      if (b_test(di, o)) {
#pragma unroll
        for (int d = 0; d < 3; d++)
          if (d < H.n_dim) mom[d] = mom[d] - H.k(orb, d);
        if (!pset) { orb_p = orb; pset = true; }
      } else {
#pragma unroll
        for (int d = 0; d < 3; d++)
          if (d < H.n_dim) mom[d] = mom[d] + H.k(orb, d);
        if (!qset) { orb_q = orb; qset = true; }
        else if (!sset) { orb_s = orb; sset = true; }
      }
    }
  }
  double m2 = 0.0;
#pragma unroll
  for (int d = 0; d < 3; d++)
    if (d < H.n_dim) m2 += mom[d] * mom[d];
  if (m2 * (H.length_cell * H.length_cell) > EPSILON) return 0.0;
  double pot = FOUR_PI / H.kdiff2(orb_p, orb_q);
  if (n_eu != 2) pot = pot - FOUR_PI / H.kdiff2(orb_p, orb_s);
  int g = heg_gamma_exp(iu, eu) + heg_gamma_exp(ju, eu) + heg_gamma_exp(id, ed) + heg_gamma_exp(jd, ed);
  if (g & 1) pot = -pot;
  return pot / L3;
}

// ---------------------------------------------------------------------------
// hubbard k-space
// ---------------------------------------------------------------------------
struct HubCtx {
  const int32_t *kv;  // (2, nsites)
  const double *ke;
  double ubyn;
  int l_x, l_y, nup, ndn;
};
template <int NW>
__device__ __forceinline__ double hub_hamiltonian(const HubCtx &H, const Bits<NW> &ub, const Bits<NW> &db, const Bits<NW> &uk, const Bits<NW> &dk) {
  if (b_eq(ub, uk) && b_eq(db, dk)) {
    double me = H.ubyn * H.nup * H.ndn;
    Bits<NW> d = ub;
    while (!b_is_zero(d)) {
      int i = b_ctz(d);
      b_clear_lowest(d);
      me = me + H.ke[i];
    }
    d = db;
    while (!b_is_zero(d)) {
      int i = b_ctz(d);
      b_clear_lowest(d);
      me = me + H.ke[i];
    }
    return me;
  }
  if (b_popc(b_andnot(ub, uk)) != 1 || b_popc(b_andnot(db, dk)) != 1) return 0.0;
  int p = b_ctz(b_andnot(ub, uk)), r = b_ctz(b_andnot(uk, ub)), q = b_ctz(b_andnot(db, dk)), s = b_ctz(b_andnot(dk, db));
  int dx = H.kv[2 * p] + H.kv[2 * q] - H.kv[2 * r] - H.kv[2 * s];
  int dy = H.kv[2 * p + 1] + H.kv[2 * q + 1] - H.kv[2 * r + 1] - H.kv[2 * s + 1];
  int px = 2 * H.l_x, py = 2 * H.l_y;
  if ((((dx % px) + px) % px) != 0 || (((dy % py) + py) % py) != 0) return 0.0;
  return H.ubyn * permutation_factor(ub, uk) * permutation_factor(db, dk);
}

// ---------------------------------------------------------------------------
// hamiltonian(up1,dn1,up2,dn2) of chemistry.f90:10273, heg.f90:3968, semistoch.f90:2234, specialised at COMPILE time on
// the model and on time-reversal symmetry: every kernel that evaluates elements is instantiated per <NW, MODEL, TS> and
// carries only its own model's code (no runtime switch inside a kernel; the host picks the instantiation once per call
// with SQ_MODEL_DISPATCH).  c2: combine_2, normally the shared-memory copy.
// ---------------------------------------------------------------------------
template <int NW, int MODEL, bool TS>
__device__ __forceinline__ double model_hamiltonian(const ModelTables &T, const int32_t *c2, const Bits<NW> &iu, const Bits<NW> &id, const Bits<NW> &ju,
                                                    const Bits<NW> &jd) {
  if constexpr (MODEL == MODEL_CHEM) {
    ChemCtx C{T.integrals, c2, T.norb + 1, T.enuc, T.sqrt2, T.sqrt2inv, T.z};
    if constexpr (TS) {
      return chem_hamiltonian_time_sym(C, iu, id, ju, jd);
    } else {
      int lvl = excitation_level(iu, id, ju, jd);
      return lvl >= 0 ? chem_hamiltonian_level(C, iu, id, ju, jd, lvl) : 0.0;
    }
  } else if constexpr (MODEL == MODEL_HEG) {
    HegCtx H{T.k_vectors, T.n_dim, T.length_cell};
    int lvl = excitation_level(iu, id, ju, jd);
    return lvl >= 0 ? heg_hamiltonian(H, iu, id, ju, jd) : 0.0;
  } else {
    HubCtx H{T.hk_vectors, T.k_energies, T.ubyn, T.l_x, T.l_y, T.nup, T.ndn};
    return hub_hamiltonian(H, iu, id, ju, jd);
  }
}

// host: a kernel may take 48 KiB of static plus dynamic shared memory unless it opts into more, so its default dynamic
// budget is 48 KiB minus its own static shared memory.  Chem kernels stage combine_2, (norb + 1)^2 * 4 bytes: 64 KiB at
// 127 orbitals, and already above the default budget of eval_kernel / select_kernel (3 KiB static) from 107 orbitals on.
template <typename Kernel>
inline cudaError_t allow_dynamic_smem(Kernel kernel, int bytes) {
  cudaFuncAttributes a;
  cudaError_t e = cudaFuncGetAttributes(&a, kernel);
  if (e != cudaSuccess || bytes <= a.maxDynamicSharedSizeBytes) return e;
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

// host: run `call` with the compile-time constants kModel / kTS of the system described by T
#define SQ_MODEL_DISPATCH(T, call)                                                          \
  do {                                                                                      \
    if ((T).model == sqmc::MODEL_CHEM && (T).time_sym) {                                    \
      constexpr int kModel = sqmc::MODEL_CHEM; constexpr bool kTS = true; call;             \
    } else if ((T).model == sqmc::MODEL_CHEM) {                                             \
      constexpr int kModel = sqmc::MODEL_CHEM; constexpr bool kTS = false; call;            \
    } else if ((T).model == sqmc::MODEL_HEG) {                                              \
      constexpr int kModel = sqmc::MODEL_HEG; constexpr bool kTS = false; call;             \
    } else {                                                                                \
      constexpr int kModel = sqmc::MODEL_HUBBARDK; constexpr bool kTS = false; call;        \
    }                                                                                       \
  } while (0)

}  // namespace sqmc
