// bundle.cu -- "row bundle" ordering of the local CSR for H.v (sm_100a).
//
// Why: the plain warp-per-row H.v is bound by the L1TEX data pipe, not by HBM (profiles/r01_spmv_vec32_hci1e7_ncu_full.txt):
// a 32-lane gather of x touches ~30 distinct 32-byte sectors because one row's columns are spread over the whole vector.
// Neighbouring rows of the alpha-major order (same alpha string, adjacent beta strings) connect to NEIGHBOURING columns,
// so the entries of R consecutive rows, merged in column order, gather from far fewer sectors per 32 entries
// (measured on C2: 28 -> 21 (R=2) -> 16.5 (R=4) sectors).
//
// Layout (format 2): a bundle = R consecutive local rows (R = 2 or 4); its entries keep their place in cols/vals (the
// bundle's segment is [rowptr[bR], rowptr[bR+R])) but
//   * are re-ordered by (column, row) -- the "merged order";
//   * the column word carries the row-in-bundle ONE-HOT in its low 4 bits (stored = column << 4 | 1 << r), so the
//     kernel routes a product to its row sum with a 0.0 / 1.0 multiplier built from one bit (LOP3 + IMAD + DFMA per row
//     sum) instead of compare + add + two selects;
//   * inside every 16-byte-aligned block of 128 entries the merged order is stored TRANSPOSED (storage slot 4*l + u holds
//     merged entry 32*u + l): one 128-bit load hands lane l the entries l, l+32, l+64, l+96 of the block, i.e. the four
//     column words (and two such loads the four values) it needs, while each gather of x still covers 32 CONSECUTIVE
//     merged entries (the coalescing the bundles exist for).  Entries in front of the first aligned block (<= 3) and
//     after the last full block (<= 127) stay in merged order and are read with scalar loads.
// The byte count is unchanged (12 B per entry) and the encoding is an in-place permutation inside each segment, so it is
// undone exactly (bundle_decode) whenever a consumer wants plain CSR rows (export_upper, incremental build); get_row
// reads one bundle and filters.  One warp multiplies one bundle; the block loop is software pipelined with two named
// register sets (next block's 128-bit loads are issued between the current block's gathers and its arithmetic).
#include <cub/cub.cuh>

#include <algorithm>
#include <cstdlib>

#include "handle.h"
#include "stream_loads.cuh"

namespace sqmc {

static const int kBShift = 4;       // low bits of the stored column word = one-hot row within the bundle
static const int kBCapMax = 16384;  // entries of one bundle staged in shared memory by encode/decode (12 B each)

static inline unsigned bblocks(int64_t n, int t = 256) { return (unsigned)std::max<int64_t>(1, std::min<int64_t>(div_up(n, t), 0x7fffffff)); }

// storage slot of merged entry i of a segment that starts at global entry index e0 and holds L entries
struct Sigma {
  int h;          // entries in front of the first 4-aligned index
  int64_t nblk;   // full 128-entry blocks
  __host__ __device__ Sigma(int64_t e0, int64_t L) {
    h = (int)((4 - (e0 & 3)) & 3);
    if (h > L) h = (int)L;
    nblk = (L - h) / 128;
  }
  __host__ __device__ int64_t operator()(int64_t i) const {
    const int64_t q = i - h;
    if (q < 0 || q >= nblk * 128) return i;
    const int64_t j = q >> 7;
    const int t = (int)(q & 127);
    return h + (j << 7) + 4 * (t & 31) + (t >> 5);
  }
};

__global__ void bundle_len_kernel(const int64_t *rowptr, int64_t nloc, int R, int64_t nb, int64_t *len) {
  int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= nb) return;
  const int64_t r1 = min(b * R + R, nloc);
  len[b] = rowptr[r1] - rowptr[b * R];
}

// ------------------------------------------------------------------ encode: plain rows -> (column,row)-merged, tagged, block-transposed
template <int R>
__global__ void __launch_bounds__(512) bundle_encode_kernel(const int64_t *__restrict__ rowptr, int64_t nloc, int64_t nb, int32_t *cols, double *vals, int cap,
                                                            int len_lo, bool take_longer) {
  extern __shared__ __align__(8) unsigned char bsm[];
  double *sv = reinterpret_cast<double *>(bsm);
  int32_t *sc = reinterpret_cast<int32_t *>(sv + cap);
  __shared__ int64_t rp[R + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  for (int64_t b = blockIdx.x; b < nb; b += gridDim.x) {
    if (threadIdx.x <= R) rp[threadIdx.x] = rowptr[min(b * R + (int64_t)threadIdx.x, nloc)];
    __syncthreads();
    const int64_t base = rp[0];
    const int64_t Ltot = rp[R] - base;
    // this launch handles bundles with len_lo < length <= cap (and the longer ones when take_longer):
    // short bundles run with a small shared-memory footprint, i.e. several CTAs per SM
    if (Ltot <= len_lo || (Ltot > cap && !take_longer)) { __syncthreads(); continue; }
    const Sigma S(base, Ltot);
    if (Ltot > cap) {
      // too long to stage: rows stay contiguous (merged order = natural order), tags + block transposition only.
      // pass 1: tags; pass 2: one warp transposes one 128-entry block through registers (reads precede writes)
      for (int64_t i = threadIdx.x; i < Ltot; i += blockDim.x) {
        int r = 0;
#pragma unroll
        for (int q = 1; q < R; q++) r += (base + i >= rp[q]);
        cols[base + i] = (cols[base + i] << kBShift) | (1 << r);
      }
      __syncthreads();
      for (int64_t j = warp; j < S.nblk; j += nwarp) {
        const int64_t o = base + S.h + (j << 7);
        int32_t c[4];
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) { c[u] = cols[o + 32 * u + lane]; v[u] = vals[o + 32 * u + lane]; }
        __syncwarp();
#pragma unroll
        for (int u = 0; u < 4; u++) { cols[o + 4 * lane + u] = c[u]; vals[o + 4 * lane + u] = v[u]; }
      }
    } else {
      const int L = (int)Ltot;
      int off[R + 1];
#pragma unroll
      for (int r = 0; r <= R; r++) off[r] = (int)(rp[r] - base);
      for (int i = threadIdx.x; i < L; i += blockDim.x) { sc[i] = cols[base + i]; sv[i] = vals[base + i]; }
      __syncthreads();
      for (int i = threadIdx.x; i < L; i += blockDim.x) {
        int r = 0;
#pragma unroll
        for (int q = 1; q < R; q++) r += (i >= off[q]);
        const int32_t c = sc[i];
        int pos = 0;
#pragma unroll
        for (int q = 0; q < R; q++) {
          if (q == r) { pos += i - off[q]; continue; }
          // entries of row q that sort before (c, r): columns < c, plus an equal column when q < r
          const int32_t key = q < r ? c + 1 : c;
          int lo = off[q], hi = off[q + 1];
          while (lo < hi) {
            int mid = (lo + hi) >> 1;
            if (sc[mid] < key) lo = mid + 1;
            else hi = mid;
          }
          pos += lo - off[q];
        }
        const int64_t st = S(pos);
        cols[base + st] = (c << kBShift) | (1 << r);
        vals[base + st] = sv[i];
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ decode: exact inverse (stable partition of the merged order by row tag)
template <int R>
__global__ void __launch_bounds__(256) bundle_decode_kernel(const int64_t *__restrict__ rowptr, int64_t nloc, int64_t nb, int32_t *cols, double *vals, int cap) {
  extern __shared__ __align__(8) unsigned char bsm[];
  double *sv = reinterpret_cast<double *>(bsm);
  int32_t *sc = reinterpret_cast<int32_t *>(sv + cap);
  __shared__ int64_t rp[R + 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int64_t b = blockIdx.x; b < nb; b += gridDim.x) {
    if (threadIdx.x <= R) rp[threadIdx.x] = rowptr[min(b * R + (int64_t)threadIdx.x, nloc)];
    __syncthreads();
    const int64_t base = rp[0];
    const int64_t Ltot = rp[R] - base;
    const Sigma S(base, Ltot);
    if (Ltot > cap) {
      for (int64_t j = w; j < S.nblk; j += nw) {  // undo the block transposition, then drop the tags
        const int64_t o = base + S.h + (j << 7);
        int32_t c[4];
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) { c[u] = cols[o + 4 * lane + u]; v[u] = vals[o + 4 * lane + u]; }
        __syncwarp();
#pragma unroll
        for (int u = 0; u < 4; u++) { cols[o + 32 * u + lane] = c[u]; vals[o + 32 * u + lane] = v[u]; }
      }
      __syncthreads();
      for (int64_t i = threadIdx.x; i < Ltot; i += blockDim.x) cols[base + i] = cols[base + i] >> kBShift;
    } else {
      const int L = (int)Ltot;
      for (int i = threadIdx.x; i < L; i += blockDim.x) { sc[i] = cols[base + i]; sv[i] = vals[base + i]; }
      __syncthreads();
      for (int r = w; r < R; r += nw) {
        int64_t out = rp[r];
        for (int i0 = 0; i0 < L; i0 += 32) {
          const int i = i0 + lane;
          const int st = i < L ? (int)S(i) : 0;
          const int32_t word = i < L ? sc[st] : 0;
          const bool m = i < L && ((word >> r) & 1);
          const unsigned bal = __ballot_sync(0xffffffffu, m);
          if (m) {
            const int64_t p = out + __popc(bal & ((1u << lane) - 1));
            cols[p] = word >> kBShift;
            vals[p] = sv[st];
          }
          out += __popc(bal);
        }
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ H.v on bundles: one warp per bundle, R sums per lane
// A product is routed to its row sum with a 0.0 / 1.0 multiplier built from the one-hot bit (exact: p*1+a and p*0+a round like
// a+p and a).
template <int R, int Q = 0>
__device__ __forceinline__ void badd(double (&acc)[R], int32_t word, double p) {
  if constexpr (Q < R) {
    const int hi = (word & (1 << Q)) * (0x3FF00000 >> Q);  // 0x3FF00000 = high word of 1.0
    acc[Q] = fma(p, __hiloint2double(hi, 0), acc[Q]);
    badd<R, Q + 1>(acc, word, p);
  }
}

__device__ __forceinline__ int4 ld_col4(const int32_t *p, const Policies &P) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.b32 {%0, %1, %2, %3}, [%4], %5;" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(P.stream));
  return r;
}
__device__ __forceinline__ double2 ld_val2(const double *p, const Policies &P) {
  double2 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(r.x), "=d"(r.y) : "l"(p), "l"(P.stream));
  return r;
}
__device__ __forceinline__ double2 bld_x2(const double *p, const Policies &P) {
  double2 r;
  asm volatile("ld.global.nc.L1::evict_last.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(r.x), "=d"(r.y) : "l"(p), "l"(P.x));
  return r;
}

struct Blk {  // one lane's share of a 128-entry block: merged entries lane, lane+32, lane+64, lane+96
  int4 c;
  double2 v01, v23;
};
__device__ __forceinline__ void blk_load(Blk &B, const int32_t *cols, const double *vals, int64_t o, int lane, const Policies &P) {
  B.c = ld_col4(cols + o + 4 * lane, P);
  B.v01 = ld_val2(vals + o + 4 * lane, P);
  B.v23 = ld_val2(vals + o + 4 * lane + 2, P);
}

// XT: the gathers of x go through the texture path (tex1Dfetch on a linear texture over x) instead of LSU loads: the LSU data
// pipe of L1TEX is the busiest unit of this kernel (90 % under ncu, half of its wavefronts are the gathers) and the texture
// pipe is idle otherwise.  A linear texture needs a 512-byte aligned base; other vectors are gathered with LSU loads.
//
// SCAT (distributed-slice entry points): the kernel does not write y but sends every finished row sum -- plus c*w[row] for the
// projector, do_walk.f90:2290 -- straight to the rank that owns the determinant (a store into that rank's exchange buffer
// over NVLink, p2p.cu), and the last CTA publishes the epoch to every peer: H.v and the reduce-scatter of
// mpi_redscatt_real_dparray (mpi_routines.f90:1592) are one kernel, the transfers overlap the arithmetic bundle by bundle.
//
// The start of a bundle is ordered for latency.  ncu's stall samples and the shared-bundle / several-bundles-per-warp experiments
// (profiles/r02_bundle_kernel_ab.txt) showed that the per-bundle prologue -- row pointers -> head / tail entries (up to five scalar
// load -> gather -> add rounds, one after the other) -> first block -> first gathers -- is a chain of serial memory latencies during
// which the warp has nothing else in flight.  Here the first block's three 128-bit stream loads are issued FIRST, and the (up to
// five) scalar load pairs of the head / tail entries are all issued before their gathers, so these latencies overlap: 2 % on the
// 26-block bundles of the bench matrix, 6 % on 9-block bundles.
//
// x is the last parameter: placed in front of O it would move OwnerScatter in parameter space and change how the SCAT
// instantiations load it.
template <int R, bool SCAT, bool XT>
__global__ void __launch_bounds__(256, 4) bundle_hv_kernel(const int64_t *__restrict__ rowptr, int64_t nloc, int64_t nb, const int32_t *__restrict__ cols,
                                                           const double *__restrict__ vals, double *__restrict__ y, OwnerScatter O,
                                                           cudaTextureObject_t xtex, const double *__restrict__ x) {
  const Policies P;
  auto gx = [&](int32_t col) -> double {
    if constexpr (XT) {
      const int2 t = tex1Dfetch<int2>(xtex, col);
      return __hiloint2double(t.y, t.x);
    } else {
      return ld_x(x + col, P);
    }
  };
  const int lane = threadIdx.x & 31;
  const int64_t b = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (b < nb) {
    const int64_t e0 = rowptr[b * R], e1 = rowptr[min(b * R + R, nloc)];
    const Sigma S(e0, e1 - e0);
    const int64_t nblk = S.nblk, o0 = e0 + S.h;
    Blk A, B;
    double xa[4], acc[R];
    if (nblk > 0) blk_load(A, cols, vals, o0, lane, P);
#pragma unroll
    for (int r = 0; r < R; r++) acc[r] = 0.0;
    {
      // head entry of this lane (slot 0) and its tail entries (slots 1..4); absent entries get column word 0 / value 0.0: a product
      // 0.0 * x[0] that is routed nowhere (the one-hot bits of the word are 0)
      const int64_t t0 = o0 + (nblk << 7) + lane;
      int32_t cw[5];
      double vv[5], xx[5];
      cw[0] = 0; vv[0] = 0.0;
      if (lane < S.h) { cw[0] = ld_col(cols + e0 + lane, P); vv[0] = ld_val(vals + e0 + lane, P); }
#pragma unroll
      for (int q = 0; q < 4; q++) {
        cw[q + 1] = 0; vv[q + 1] = 0.0;
        if (t0 + 32 * q < e1) { cw[q + 1] = ld_col(cols + t0 + 32 * q, P); vv[q + 1] = ld_val(vals + t0 + 32 * q, P); }
      }
#pragma unroll
      for (int q = 0; q < 5; q++) xx[q] = gx(cw[q] >> kBShift);
#pragma unroll
      for (int q = 0; q < 5; q++) badd<R>(acc, cw[q], vv[q] * xx[q]);
    }
    auto gather = [&](const Blk &K) {
      xa[0] = gx(K.c.x >> kBShift);
      xa[1] = gx(K.c.y >> kBShift);
      xa[2] = gx(K.c.z >> kBShift);
      xa[3] = gx(K.c.w >> kBShift);
    };
    auto work = [&](const Blk &K) {
      badd<R>(acc, K.c.x, K.v01.x * xa[0]);
      badd<R>(acc, K.c.y, K.v01.y * xa[1]);
      badd<R>(acc, K.c.z, K.v23.x * xa[2]);
      badd<R>(acc, K.c.w, K.v23.y * xa[3]);
    };
    // software pipeline over the full blocks with two named register sets: gathers of the current block, then the next block's
    // 128-bit stream loads, then the current block's arithmetic (the loads are asm volatile: their order is kept)
    int64_t j = 0;
    for (; j + 2 <= nblk; j += 2) {
      gather(A);
      blk_load(B, cols, vals, o0 + ((j + 1) << 7), lane, P);
      work(A);
      gather(B);
      if (j + 2 < nblk) blk_load(A, cols, vals, o0 + ((j + 2) << 7), lane, P);
      work(B);
    }
    if (j < nblk) {
      gather(A);
      work(A);
    }
    double m0 = 0.0;
#pragma unroll
    for (int r = 0; r < R; r++) {
      double a0 = acc[r];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) a0 += __shfl_xor_sync(0xffffffffu, a0, o);
      if (lane == r) m0 = a0;
    }
    const int64_t row = b * R + lane;
    if (lane < R && row < nloc) {
      if (SCAT) {
        double v = m0;
        if (O.w) v = v + O.c * O.w[row];
        O.dst[O.owner[row]][O.pos[row]] = v;
      } else {
        y[row] = m0;
      }
    }
  }
  if (SCAT) {  // all rows of this CTA are on their way: the last CTA publishes the epoch to every peer
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned long long prev = atomicAdd(O.counter, 1ull);
      if (prev == gridDim.x - 1) {
        *O.counter = 0ull;
        __threadfence_system();
        for (int p = 0; p < O.nranks; p++)
          if (O.flag[p]) asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(O.flag[p]), "l"(O.epoch) : "memory");
      }
    }
  }
}

// Two right-hand sides at once (Davidson with n_states >= 2, SURVEY.md 8(d) "SpMM"): x / y hold the two vectors interleaved
// (x[2*col + k]), one 16-byte gather serves both and the matrix is streamed once (algorithmic bytes 12*nnz_full + 36*n for two
// vectors instead of 2*(12*nnz_full + 20*n)).  2 R row sums are live, so the head / tail entries are taken one round at a time.
template <int R, bool XT>
__global__ void __launch_bounds__(256, 4) bundle_hv2_kernel(const int64_t *__restrict__ rowptr, int64_t nloc, int64_t nb, const int32_t *__restrict__ cols,
                                                            const double *__restrict__ vals, const double *__restrict__ x, double *__restrict__ y,
                                                            cudaTextureObject_t xtex) {
  const Policies P;
  auto gx2 = [&](int32_t col) -> double2 {
    if constexpr (XT) {
      const int4 t = tex1Dfetch<int4>(xtex, col);
      return make_double2(__hiloint2double(t.y, t.x), __hiloint2double(t.w, t.z));
    } else {
      return bld_x2(x + 2 * (int64_t)col, P);
    }
  };
  const int64_t b = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= nb) return;
  const int64_t r0 = b * R;
  const int64_t e0 = rowptr[r0], e1 = rowptr[min(r0 + R, nloc)];
  const Sigma S(e0, e1 - e0);
  double acc[R], acc2[R];
#pragma unroll
  for (int r = 0; r < R; r++) acc[r] = 0.0;
#pragma unroll
  for (int r = 0; r < R; r++) acc2[r] = 0.0;

  const int64_t o0 = e0 + S.h;
  auto work = [&](const Blk &K, double (&xa)[4], double (&xb)[4]) {
    badd<R>(acc, K.c.x, K.v01.x * xa[0]);
    badd<R>(acc, K.c.y, K.v01.y * xa[1]);
    badd<R>(acc, K.c.z, K.v23.x * xa[2]);
    badd<R>(acc, K.c.w, K.v23.y * xa[3]);
    badd<R>(acc2, K.c.x, K.v01.x * xb[0]);
    badd<R>(acc2, K.c.y, K.v01.y * xb[1]);
    badd<R>(acc2, K.c.z, K.v23.x * xb[2]);
    badd<R>(acc2, K.c.w, K.v23.y * xb[3]);
  };
  auto gather = [&](const Blk &K, double (&xa)[4], double (&xb)[4]) {
    double2 t;
    t = gx2(K.c.x >> kBShift); xa[0] = t.x; xb[0] = t.y;
    t = gx2(K.c.y >> kBShift); xa[1] = t.x; xb[1] = t.y;
    t = gx2(K.c.z >> kBShift); xa[2] = t.x; xb[2] = t.y;
    t = gx2(K.c.w >> kBShift); xa[3] = t.x; xb[3] = t.y;
  };
  // software pipeline over the full blocks as in bundle_hv_kernel
  Blk A, B;
  double xa[4], xb[4];
  const int64_t nblk = S.nblk;
  if (nblk > 0) blk_load(A, cols, vals, o0, lane, P);
  // entries in front of the first aligned block (<= 3) and behind the last full block (<= 127), merged order, scalar loads -- after the
  // first block's stream loads are on their way
  auto one = [&](int32_t cw, double v) {
    const double2 xv = gx2(cw >> kBShift);
    badd<R>(acc, cw, v * xv.x);
    badd<R>(acc2, cw, v * xv.y);
  };
  if (lane < S.h) one(ld_col(cols + e0 + lane, P), ld_val(vals + e0 + lane, P));
  for (int64_t k = o0 + (nblk << 7) + lane; k < e1; k += 32) one(ld_col(cols + k, P), ld_val(vals + k, P));
  int64_t j = 0;
  for (; j + 2 <= nblk; j += 2) {
    gather(A, xa, xb);
    blk_load(B, cols, vals, o0 + ((j + 1) << 7), lane, P);
    work(A, xa, xb);
    gather(B, xa, xb);
    if (j + 2 < nblk) blk_load(A, cols, vals, o0 + ((j + 2) << 7), lane, P);
    work(B, xa, xb);
  }
  if (j < nblk) {
    gather(A, xa, xb);
    work(A, xa, xb);
  }

  double m0 = 0.0, m1 = 0.0;
#pragma unroll
  for (int r = 0; r < R; r++) {
    double a0 = acc[r], a1 = acc2[r];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a0 += __shfl_xor_sync(0xffffffffu, a0, o);
      a1 += __shfl_xor_sync(0xffffffffu, a1, o);
    }
    if (lane == r) { m0 = a0; m1 = a1; }
  }
  if (lane < R && r0 + lane < nloc) {
    const int64_t row = r0 + lane;
    y[2 * row] = m0;
    y[2 * row + 1] = m1;
  }
}

// ------------------------------------------------------------------ host side
// default: bundles of 4 rows (measured best on B200, profiles/r01_bundle_experiment.txt); SQMC_BUNDLE=0|2|4 overrides.
// Read per call (a getenv is ~100 ns) so that one process can A/B layouts on one resident matrix.
static int bundle_want() {
  const char *e = getenv("SQMC_BUNDLE");
  const int v = e ? atoi(e) : 4;
  return (v == 2 || v == 4) ? v : 0;
}
template <int R>
static int encode_t(sqmc_b200_handle *h, int cap, cudaStream_t s) {
  const int64_t nloc = h->row1 - h->row0, nb = div_up(nloc, (int64_t)R);
  SQ_CUDA(cudaFuncSetAttribute(bundle_encode_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap * 12));
  // two passes: bundles up to kSmall entries with 4 CTAs per SM, the rest with the full staging capacity
  const int kSmall = 4096;
  int lo = 0;
  if (cap > kSmall) {
    bundle_encode_kernel<R><<<(unsigned)std::min<int64_t>(nb, (int64_t)G.sm_count * 4), 512, kSmall * 12, s>>>(h->d_rowptr, nloc, nb, h->d_cols, h->d_vals, kSmall, 0, false);
    SQ_LAUNCH_CHECK();
    lo = kSmall;
  }
  const int smem = cap * 12;
  const int per_sm = std::max(1, std::min(4, (220 * 1024) / std::max(smem, 1)));
  bundle_encode_kernel<R><<<(unsigned)std::min<int64_t>(nb, (int64_t)G.sm_count * per_sm), 512, smem, s>>>(h->d_rowptr, nloc, nb, h->d_cols, h->d_vals, cap, lo, true);
  SQ_LAUNCH_CHECK();
  return 0;
}
template <int R>
static int decode_t(sqmc_b200_handle *h, int cap, cudaStream_t s) {
  const int64_t nloc = h->row1 - h->row0, nb = div_up(nloc, (int64_t)R);
  const int smem = cap * 12;
  SQ_CUDA(cudaFuncSetAttribute(bundle_decode_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const int per_sm = std::max(1, std::min(8, (220 * 1024) / std::max(smem, 1)));
  bundle_decode_kernel<R><<<(unsigned)std::min<int64_t>(nb, (int64_t)G.sm_count * per_sm), 256, smem, s>>>(h->d_rowptr, nloc, nb, h->d_cols, h->d_vals, cap);
  SQ_LAUNCH_CHECK();
  return 0;
}

// plain CSR -> bundles (no-op when disabled, already bundled or the column word has no room for the tag)
int bundle_encode(sqmc_b200_handle *h) { return bundle_encode_r(h, bundle_want()); }
int bundle_encode_r(sqmc_b200_handle *h, int R) {
  const int64_t nloc = h->row1 - h->row0;
  if (!R || h->bundle_R || !h->d_rowptr) return 0;
  if (R != 2 && R != 4) { set_error("bundle_encode: rows per bundle must be 2 or 4"); return 2; }
  if (h->n >= (1ll << (31 - kBShift))) return 0;
  cudaStream_t s = G.stream;
  if (!h->d_diag && nloc > 0) {  // Davidson's preconditioner and the projector read the diagonal: keep a copy
    double *dst = nullptr;
    SQ_CHECK(devbuf_alloc((void **)&dst, nloc * sizeof(double)));
    int rc = extract_diag(h, dst, s);  // reads the plain rows (d_diag is still unset)
    if (rc) { devbuf_free(dst); return rc; }
    h->d_diag = dst;
  }
  if (nloc == 0 || h->nnz_local == 0) {
    // a rank without rows still switches layout: every rank must take the same (collective) code path in the two-vector H.v
    h->bundle_R = R;
    h->bundle_cap = 1024;
    return 0;
  }
  // staging capacity = longest bundle (rounded up), capped
  const int64_t nb = div_up(nloc, (int64_t)R);
  DevBuf<int64_t> len, mx;
  SQ_CHECK(len.alloc(nb));
  SQ_CHECK(mx.alloc(1));
  bundle_len_kernel<<<bblocks(nb), 256, 0, s>>>(h->d_rowptr, nloc, R, nb, len.p);
  SQ_LAUNCH_CHECK();
  size_t tb = 0;
  cub::DeviceReduce::Max(nullptr, tb, len.p, mx.p, (int)std::min<int64_t>(nb, 0x7fffffff), s);
  DevBuf<unsigned char> tmp;
  SQ_CHECK(tmp.alloc((int64_t)tb + 16));
  SQ_CUDA(cub::DeviceReduce::Max(tmp.p, tb, len.p, mx.p, (int)std::min<int64_t>(nb, 0x7fffffff), s));
  g_launch_count += 1;
  int64_t maxlen = 0;
  SQ_CUDA(cudaMemcpyAsync(&maxlen, mx.p, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  int cap = (int)std::min<int64_t>(kBCapMax, std::max<int64_t>(1024, (maxlen + 1023) / 1024 * 1024));
  if (const char *ce = getenv("SQMC_BUNDLE_CAP")) cap = std::max(64, std::min(cap, atoi(ce)));  // test hook: force the tag-only path
  h->bundle_cap = cap;
  int rc = R == 2 ? encode_t<2>(h, cap, s) : encode_t<4>(h, cap, s);
  if (rc) return rc;
  h->bundle_R = R;
  return 0;
}

// bundles -> plain CSR (exact inverse)
int bundle_decode(sqmc_b200_handle *h) {
  if (!h->bundle_R) return 0;
  cudaStream_t s = G.stream;
  const int R = h->bundle_R, cap = h->bundle_cap;
  if (h->row1 - h->row0 > 0 && h->nnz_local > 0) {
    int rc = R == 2 ? decode_t<2>(h, cap, s) : decode_t<4>(h, cap, s);
    if (rc) return rc;
  }
  SQ_CUDA(cudaStreamSynchronize(s));
  h->bundle_R = 0;
  return 0;
}

// linear texture over x (nv interleaved vectors per element), cached per (pointer, length, nv) on the handle
static int x_texture(sqmc_b200_handle *h, const double *x, int nv, cudaTextureObject_t *out) {
  for (auto &t : h->xtex)
    if (t.ptr == x && t.n == h->n && t.nv == nv) { *out = t.tex; return 0; }
  cudaResourceDesc rd = {};
  rd.resType = cudaResourceTypeLinear;
  rd.res.linear.devPtr = const_cast<double *>(x);
  rd.res.linear.desc = nv == 1 ? cudaCreateChannelDesc<int2>() : cudaCreateChannelDesc<int4>();
  rd.res.linear.sizeInBytes = (size_t)h->n * nv * sizeof(double);
  cudaTextureDesc td = {};
  td.readMode = cudaReadModeElementType;
  cudaTextureObject_t tex = 0;
  SQ_CUDA(cudaCreateTextureObject(&tex, &rd, &td, nullptr));
  if (h->xtex.size() >= 16) {  // bounded cache
    cudaDestroyTextureObject(h->xtex.front().tex);
    h->xtex.erase(h->xtex.begin());
  }
  h->xtex.push_back({x, h->n, nv, tex});
  *out = tex;
  return 0;
}
void x_textures_release(sqmc_b200_handle *h) {
  for (auto &t : h->xtex) cudaDestroyTextureObject(t.tex);
  h->xtex.clear();
}

template <int R, bool XT>
static void hv_launch(const sqmc_b200_handle *h, int nv, const OwnerScatter *O, unsigned grid, int64_t nloc, int64_t nb, const double *x, double *y,
                      cudaTextureObject_t tex, cudaStream_t s) {
  if (nv == 2) bundle_hv2_kernel<R, XT><<<grid, 256, 0, s>>>(h->d_rowptr, nloc, nb, h->d_cols, h->d_vals, x, y, tex);
  else if (O) bundle_hv_kernel<R, true, XT><<<grid, 256, 0, s>>>(h->d_rowptr, nloc, nb, h->d_cols, h->d_vals, y, *O, tex, x);
  else bundle_hv_kernel<R, false, XT><<<grid, 256, 0, s>>>(h->d_rowptr, nloc, nb, h->d_cols, h->d_vals, y, OwnerScatter{}, tex, x);
}

// y = H x on bundles for nv (1 or 2) interleaved vectors; with O (one vector) every row sum goes to its owner instead of y.
// R is the matrix's bundle size; x is gathered through a texture when its base is 512-byte aligned, with LSU loads otherwise.
static int launch_hv(sqmc_b200_handle *h, int nv, const double *x, double *y, const OwnerScatter *O, cudaStream_t s) {
  const int64_t nloc = h->row1 - h->row0;
  const int R = h->bundle_R;
  const int64_t nb = div_up(nloc, (int64_t)R);
  if (nb == 0 && !O) return 0;  // the scatter grid keeps one CTA so that a rank without rows still publishes its epoch
  const unsigned grid = (unsigned)std::max<int64_t>(1, div_up(nb * 32, (int64_t)256));
  cudaTextureObject_t tex = 0;
  const bool xt = ((uintptr_t)x & 511) == 0;
  if (xt) SQ_CHECK(x_texture(h, x, nv, &tex));
  if (R == 4) (xt ? hv_launch<4, true> : hv_launch<4, false>)(h, nv, O, grid, nloc, nb, x, y, tex, s);
  else (xt ? hv_launch<2, true> : hv_launch<2, false>)(h, nv, O, grid, nloc, nb, x, y, tex, s);
  SQ_LAUNCH_CHECK();
  return 0;
}
int bundle_spmv(sqmc_b200_handle *h, const double *x, double *y, cudaStream_t s) { return launch_hv(h, 1, x, y, nullptr, s); }

// y = H x (+ c*w) with every row sum sent to its owner from inside the kernel (see OwnerScatter)
int bundle_spmv_scatter(sqmc_b200_handle *h, const double *x, const OwnerScatter &O, cudaStream_t s) { return launch_hv(h, 1, x, nullptr, &O, s); }

// y2 = H x2 for two interleaved vectors; only on bundled matrices (the caller falls back to two H.v otherwise)
int bundle_spmm2(sqmc_b200_handle *h, const double *x2, double *y2, cudaStream_t s) {
  if (!h->bundle_R) { set_error("bundle_spmm2: matrix is not in row-bundle order"); return 2; }
  return launch_hv(h, 2, x2, y2, nullptr, s);
}

// one row out of a bundled matrix (get_row): read the bundle's segment and keep the entries tagged with this row
int bundle_get_row(sqmc_b200_handle *h, int64_t internal_row, std::vector<int32_t> &cols, std::vector<double> &vals) {
  const int R = h->bundle_R;
  const int64_t nloc = h->row1 - h->row0, q = internal_row - h->row0;
  const int64_t b = q / R, r = q % R;
  const int64_t ra = b * R, rb = std::min(ra + R, nloc);
  std::vector<int64_t> rp(rb - ra + 1);
  SQ_CUDA(cudaMemcpy(rp.data(), h->d_rowptr + ra, rp.size() * sizeof(int64_t), cudaMemcpyDeviceToHost));
  const int64_t L = rp.back() - rp[0];
  std::vector<int32_t> c(L);
  std::vector<double> v(L);
  if (L) {
    SQ_CUDA(cudaMemcpy(c.data(), h->d_cols + rp[0], L * sizeof(int32_t), cudaMemcpyDeviceToHost));
    SQ_CUDA(cudaMemcpy(v.data(), h->d_vals + rp[0], L * sizeof(double), cudaMemcpyDeviceToHost));
  }
  cols.clear();
  vals.clear();
  const Sigma S(rp[0], L);
  for (int64_t i = 0; i < L; i++) {  // merged order: ascending columns within the row
    const int64_t st = S(i);
    if ((c[st] >> r) & 1) { cols.push_back(c[st] >> kBShift); vals.push_back(v[st]); }
  }
  return 0;
}

}  // namespace sqmc
