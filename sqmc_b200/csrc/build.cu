// build.cu -- sparse Hamiltonian construction over a determinant list (sm_100a).
//
// Replaces generate_sparse_ham_chem_upper_triangular (chemistry.f90:7639-8009,
// MPI twin :8012-8546), generate_sparse_ham_heg_upper_triangular
// (heg.f90:3553-3809), generate_sparse_ham_hubbardk_upper_triangular
// (hubbard.f90:9435-9672) and their helper get_connected_dets_in_list
// (chemistry.f90:9851-9991, heg.f90:3846-3964).
//
// GPU-first formulation (not the reference's per-row binary searches):
//   1. determinants are sorted alpha-major (up, dn) -> INTERNAL row order; equal up
//      strings form alpha-groups, equal dn strings beta-groups (second sorted view).
//   2. unique alpha strings are linked through their (N-1)-electron keys (the
//      reference's alpha_m1 idea, chemistry.f90:9819, applied to unique strings,
//      not to determinants): the run of a key lists every alpha string one
//      excitation away.
//   3. candidate generation is pure XOR/popcount work, one CTA per tile of <= 256 rows of one alpha-group, the beta
//      strings of each candidate group staged once in shared memory (connect_tile_kernel):
//        same alpha-group      : popc(dn^dn') in {2,4}   (dn single / double)
//        neighbour alpha-groups : popc(dn^dn') in {0,2}   (up single, up+dn double)
//        same beta-group        : popc(up^up') == 4       (up double)
//      Every pair within two excitations is found exactly once per orientation.
//   4. candidates are sorted per row, duplicates (time-reversed partners) dropped,
//      elements evaluated with the reference's arithmetic (elements.cuh) and the
//      abs(H) > 1e-12 filter applied (chemistry.f90:9901); the diagonal is always kept.
//   5. FULL rows (both triangles) are produced directly; H(i,j) is always evaluated
//      with the lower CALLER index as bra, exactly the element the reference stores
//      in its upper triangle, so the matrix is bit-symmetric and export is a filter.
// Compile with --fmad=false (see elements.cuh).
#include <cub/cub.cuh>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>

#include "handle.h"

namespace sqmc {



// ------------------------------------------------------------------ helpers
static const int kThreads = 256;
static const int64_t kSlack = 1024;
static inline int nblocks(int64_t n, int t = kThreads) { return (int)std::min<int64_t>(div_up(n, t), 0x7fffffff); }

// 16-byte caller dets -> NW-word strings
template <int NW>
__global__ void split_dets_kernel(const uint64_t *raw /*n x 2*/, uint64_t *out, int64_t n, int *bad, uint64_t hi_mask0, uint64_t hi_mask1) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t lo = raw[2 * i], hi = raw[2 * i + 1];
  if ((lo & hi_mask0) || (hi & hi_mask1)) atomicExch(bad, 1);  // occupied orbital beyond norb
  out[i * NW] = lo;
  if (NW == 2) out[i * NW + 1] = hi;
}

__global__ void iota_kernel(int32_t *a, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) a[i] = (int32_t)i;
}
__global__ void gather_word_kernel(const uint64_t *src, int nw, int w, const int32_t *idx, uint64_t *out, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = src[(int64_t)idx[i] * nw + w];
}
template <int NW>
__global__ void gather_bits_kernel(const uint64_t *src, const int32_t *idx, uint64_t *out, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) b_store<NW>(out, i, b_load<NW>(src, idx[i]));
}
__global__ void invert_perm_kernel(const int32_t *perm, int32_t *iperm, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) iperm[perm[i]] = (int32_t)i;
}

// Stable LSD radix sort of records by a multi-word key given as a list of (array, nw, word)
// from least to most significant; idx (in/out) carries the permutation.
struct KeyWord {
  const uint64_t *src;
  int nw, w, bits;
};
static int sort_by_words(const std::vector<KeyWord> &words, int32_t *d_idx, int64_t n, cudaStream_t s) {
  if (n <= 1) return 0;
  DevBuf<uint64_t> k_in, k_out;
  DevBuf<int32_t> i_out;
  SQ_CHECK(k_in.alloc(n));
  SQ_CHECK(k_out.alloc(n));
  SQ_CHECK(i_out.alloc(n));
  size_t tmp_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in.p, k_out.p, d_idx, i_out.p, (int)n, 0, 64, s);
  DevBuf<char> tmp;
  SQ_CHECK(tmp.alloc((int64_t)tmp_bytes + 16));
  for (const KeyWord &kw : words) {
    if (kw.bits <= 0) continue;
    gather_word_kernel<<<nblocks(n), kThreads, 0, s>>>(kw.src, kw.nw, kw.w, d_idx, k_in.p, n);
    SQ_LAUNCH_CHECK();
    SQ_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, k_in.p, k_out.p, d_idx, i_out.p, (int)n, 0, kw.bits, s));
    g_launch_count += 3;
    SQ_CUDA(cudaMemcpyAsync(d_idx, i_out.p, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
  }
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// group boundaries of a sorted key array: flag[t] = key[t] != key[t-1]
template <int NW>
__global__ void group_flag_kernel(const uint64_t *keys, int32_t *flag, int64_t m) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= m) return;
  flag[t] = (t == 0) ? 1 : (b_eq(b_load<NW>(keys, t), b_load<NW>(keys, t - 1)) ? 0 : 1);
}
// gid = inclusive_scan(flag) - 1 ; offsets[gid] = t at flagged positions
__global__ void group_offsets_kernel(const int32_t *flag, const int32_t *gid_incl, int32_t *gid, int64_t *off, int64_t m) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= m) return;
  int32_t g = gid_incl[t] - 1;
  gid[t] = g;
  if (flag[t]) off[g] = t;
}

// build the groups of a sorted key array; returns number of groups; gid[m], off[ng+1]
template <int NW>
static int make_groups(const uint64_t *keys, int64_t m, DevBuf<int32_t> &gid, DevBuf<int64_t> &off, int64_t &ng, cudaStream_t s) {
  DevBuf<int32_t> flag, incl;
  SQ_CHECK(flag.alloc(m));
  SQ_CHECK(incl.alloc(m));
  SQ_CHECK(gid.alloc(m));
  group_flag_kernel<NW><<<nblocks(m), kThreads, 0, s>>>(keys, flag.p, m);
  SQ_LAUNCH_CHECK();
  size_t tb = 0;
  cub::DeviceScan::InclusiveSum(nullptr, tb, flag.p, incl.p, (int)m, s);
  DevBuf<char> tmp;
  SQ_CHECK(tmp.alloc((int64_t)tb + 16));
  SQ_CUDA(cub::DeviceScan::InclusiveSum(tmp.p, tb, flag.p, incl.p, (int)m, s));
  g_launch_count += 2;
  int32_t last = 0;
  SQ_CUDA(cudaMemcpyAsync(&last, incl.p + (m - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  ng = last;
  SQ_CHECK(off.alloc(ng + 1));
  group_offsets_kernel<<<nblocks(m), kThreads, 0, s>>>(flag.p, incl.p, gid.p, off.p, m);
  SQ_LAUNCH_CHECK();
  SQ_CUDA(cudaMemcpyAsync(off.p + ng, &m, sizeof(int64_t), cudaMemcpyHostToDevice, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// time-reversal expansion (chemistry.f90:9934-9979 searches with spins flipped):
// entry t<n : (a=up, b=dn, rep=t) ; entries for rows with up != dn: (a=dn, b=up, rep=row|SWAP)
static const uint32_t kSwapBit = 0x80000000u;
template <int NW>
__global__ void ts_flag_kernel(const uint64_t *up, const uint64_t *dn, int32_t *flag, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) flag[i] = b_eq(b_load<NW>(up, i), b_load<NW>(dn, i)) ? 0 : 1;
}
template <int NW>
__global__ void ts_expand_kernel(const uint64_t *up, const uint64_t *dn, const int32_t *flag, const int32_t *excl, uint64_t *Ea,
                                 uint64_t *Eb, uint32_t *Erep, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  Bits<NW> u = b_load<NW>(up, i), d = b_load<NW>(dn, i);
  b_store<NW>(Ea, i, u);
  b_store<NW>(Eb, i, d);
  Erep[i] = (uint32_t)i;
  if (flag[i]) {
    int64_t t = n + excl[i];
    b_store<NW>(Ea, t, d);
    b_store<NW>(Eb, t, u);
    Erep[t] = (uint32_t)i | kSwapBit;
  }
}
__global__ void gather_u32_kernel(const uint32_t *src, const int32_t *idx, uint32_t *out, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = src[idx[i]];
}
__global__ void row_entry_kernel(const uint32_t *Erep, int32_t *rowE, int64_t m) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < m && !(Erep[t] & kSwapBit)) rowE[Erep[t]] = (int32_t)t;
}
__global__ void scatter_gid_kernel(const int32_t *gid_sorted, const int32_t *entry_of_sorted, int32_t *gid_of_entry, int64_t m) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < m) gid_of_entry[entry_of_sorted[t]] = gid_sorted[t];
}

// (N-1)-electron keys of the unique alpha strings
template <int NW>
__global__ void nm1_keys_kernel(const uint64_t *Ea, const int64_t *gA_off, int64_t nA, int nel, uint64_t *keys, int32_t *grp) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= nA) return;
  Bits<NW> s = b_load<NW>(Ea, gA_off[g]);
  Bits<NW> t = s;
  for (int e = 0; e < nel; e++) {
    int o = b_ctz(t);
    b_clear_lowest(t);
    Bits<NW> k = s;
    b_clear(k, o);
    b_store<NW>(keys, g * nel + e, k);
    grp[g * nel + e] = (int32_t)g;
  }
}
// for every (group, electron) the run [lo,hi) of its key in the sorted key list
template <int NW>
__global__ void nm1_runs_kernel(const uint64_t *Ea, const int64_t *gA_off, int64_t nA, int nel, const uint64_t *skeys, int64_t m2,
                                int32_t *run_lo, int32_t *run_hi) {
  int64_t id = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (id >= nA * nel) return;
  int64_t g = id / nel;
  int e = (int)(id % nel);
  Bits<NW> s = b_load<NW>(Ea, gA_off[g]);
  Bits<NW> t = s;
  int o = 0;
  for (int k = 0; k <= e; k++) {
    o = b_ctz(t);
    b_clear_lowest(t);
  }
  Bits<NW> key = s;
  b_clear(key, o);
  int64_t lo = 0, hi = m2;
  while (lo < hi) {  // lower bound
    int64_t mid = (lo + hi) >> 1;
    if (b_lt(b_load<NW>(skeys, mid), key)) lo = mid + 1;
    else hi = mid;
  }
  int64_t first = lo;
  hi = m2;
  while (lo < hi) {  // upper bound
    int64_t mid = (lo + hi) >> 1;
    if (b_lt(key, b_load<NW>(skeys, mid))) hi = mid;
    else lo = mid + 1;
  }
  run_lo[id] = (int32_t)first;
  run_hi[id] = (int32_t)lo;
}

// neighbour groups of every alpha group = the members of the runs of its (N-1)-electron keys, plus the group itself
__global__ void nbr_count_kernel(const int32_t *run_lo, const int32_t *run_hi, int64_t nA, int nel, int32_t *cnt) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= nA) return;
  int c = 1;
  for (int e = 0; e < nel; e++) c += run_hi[g * nel + e] - run_lo[g * nel + e] - 1;  // every run contains the group itself once
  cnt[g] = c;
}
__global__ void nbr_fill_kernel(const int32_t *run_lo, const int32_t *run_hi, const int32_t *K_grp, int64_t nA, int nel, const int64_t *off, int32_t *nbr) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g >= nA) return;
  int64_t o = off[g];
  nbr[o++] = (int32_t)g;
  for (int e = 0; e < nel; e++)
    for (int32_t r = run_lo[g * nel + e]; r < run_hi[g * nel + e]; r++) {
      const int32_t g2 = K_grp[r];
      if (g2 != (int32_t)g) nbr[o++] = g2;
    }
}

// ------------------------------------------------------------------ candidate generation
struct ConnView {
  // expanded entries in alpha-major order
  const uint64_t *Ea, *Eb;
  const uint32_t *Erep;
  const int32_t *eA;       // alpha group of entry
  const int64_t *gA_off;   // alpha group offsets
  const int32_t *eB;       // beta group of entry
  const int64_t *gB_off;   // beta group offsets (into the beta-major view)
  const uint64_t *EBa;     // a-string in beta-major order
  const uint32_t *EBrep;   // rep in beta-major order
  const int32_t *rowE;     // row -> its unswapped entry
  // per alpha group: its own index and the groups of the strings one excitation away, ascending
  const int64_t *nbr_off;
  const int32_t *nbr;
  // incremental build (null otherwise): inside every alpha group the determinants of the previous list first, then the new
  // ones, each part in beta order.  Pidx = internal row at a view position, Pb = its beta string, gNew_off = first new position.
  const int32_t *Pidx;
  const uint64_t *Pb;
  const int64_t *gNew_off;
};

// Tiled candidate generation: one CTA per tile of <= 256 consecutive entries of ONE alpha-group, one thread per entry
// (= row, when the entry is not a time-reversed partner).  All rows of the tile share their candidate alpha-groups
// (own group + the groups of the strings one excitation away), so the beta strings of a candidate group are staged
// ONCE in shared memory and every thread tests them against its own beta string with XOR/popcount (broadcast
// shared-memory reads, no divergence in the test).  The same-beta up-doubles are found afterwards, one warp per row.
// FILL=false counts, FILL=true writes candidate rep indices (order inside a row is arbitrary; rows are sorted later).
struct TileDesc {
  int64_t e0;    // first entry (position in the row view)
  int16_t n;     // entries (<= kConnTile)
  int16_t kind;  // 0: candidates = every entry of a group; 1 (incremental build, rows of the previous list): only the new entries
  int32_t g;     // alpha group
};
static const int kConnTile = 256;
static const int kConnStage = 1024;  // beta strings staged per step
static const int kBmpStage = 256;    // the same in connect_bitmap_kernel (own group only): with the probe lists in shared memory a small
                                     // stage lets four CTAs share an SM (54 KB each for C2) instead of three

// W32: norb <= 32 -> strings are compared as 32-bit words (POPC is a quarter-rate instruction: one instead of two per test)
// SORTED (no time-reversal expansion: entries == rows): the candidate groups are visited in ascending order and the row
// itself is emitted in its place inside its own group, so the "alpha part" of a row comes out in ascending column order;
// the same-beta up-doubles follow as a second ascending run (alen = length of the first run).  The two runs are merged
// when the evaluated row is copied to its final place -- no per-row sort.  Otherwise (time-reversed partners in the
// entry list) the diagonal comes first, the order is arbitrary and the rows are sorted afterwards.
template <int NW, bool FILL, bool W32, bool SORTED>
__global__ void __launch_bounds__(kConnTile) connect_tile_kernel(ConnView V, const TileDesc *tiles, int64_t ntiles, int64_t row_begin,
                                                                 int32_t *counts, const int64_t *cand_ptr, int32_t *cand, int32_t *alen,
                                                                 const int32_t *old_of_new, const int32_t *olen) {
  __shared__ uint64_t sEb[W32 ? 1 : kConnStage * NW];
  __shared__ uint32_t sEb32[W32 ? kConnStage : 1];
  __shared__ uint32_t sErep[FILL ? kConnStage : 1];
  __shared__ int32_t s_cnt[kConnTile];
  __shared__ int32_t s_row[kConnTile];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    const TileDesc T = tiles[t];
    const int64_t e = T.e0 + threadIdx.x;
    const bool have = threadIdx.x < T.n;
    const bool part = SORTED && V.Pidx != nullptr;  // rows come from the partitioned view
    const uint32_t rep = have ? (part ? (uint32_t)V.Pidx[e] : V.Erep[e]) : kSwapBit;
    const bool active = have && !(rep & kSwapBit);  // rows are the unswapped entries
    const int64_t p = active ? (int64_t)rep : -1;
    Bits<NW> b = b_zero<NW>();
    if (active) b = b_load<NW>(part ? V.Pb : V.Eb, e);
    // incremental build: a pair of two determinants of the previous list is already stored in the previous matrix -- only
    // pairs with at least one new determinant are generated (tiles of kind 1 stage just the new entries of every candidate
    // group); the row's old entries sit in front of its candidates (olen of them)
    const bool only_new = part && T.kind == 1;
    int64_t base = 0;
    if (FILL && active) base = cand_ptr[p - row_begin] + (olen ? olen[p] : 0);
    int cnt = 0;
    if (!SORTED && active) {
      if (FILL) cand[base] = (int32_t)p;  // diagonal
      cnt = 1;
    }
    const int g = T.g;
    // candidate groups: the group itself and the groups of the strings one excitation away, in ascending order
    for (int64_t q = V.nbr_off[g]; q < V.nbr_off[g + 1]; q++) {
      const int32_t g2 = V.nbr[q];
      const bool own = g2 == g;
      const int64_t lo = only_new ? V.gNew_off[g2] : V.gA_off[g2], hi = V.gA_off[g2 + 1];
      const uint64_t *cEb = only_new ? V.Pb : V.Eb;
      for (int64_t s0 = lo; s0 < hi; s0 += kConnStage) {
        const int ns = (int)min((int64_t)kConnStage, hi - s0);
        __syncthreads();  // previous stage fully consumed
        for (int i = threadIdx.x; i < ns; i += blockDim.x) {
          if (W32) {
            sEb32[i] = (uint32_t)cEb[s0 + i];
          } else {
#pragma unroll
            for (int w = 0; w < NW; w++) sEb[i * NW + w] = cEb[(s0 + i) * NW + w];
          }
          if (FILL) sErep[i] = only_new ? (uint32_t)V.Pidx[s0 + i] : V.Erep[s0 + i];
        }
        __syncthreads();
        if (active) {
          const uint32_t b32 = (uint32_t)b.w[0];
#pragma unroll 8
          for (int i = 0; i < ns; i++) {
            int pc = 0;
            if (W32) {
              pc = __popc(b32 ^ sEb32[i]);
            } else {
#pragma unroll
              for (int w = 0; w < NW; w++) pc += __popcll(b.w[w] ^ sEb[i * NW + w]);
            }
            const bool hit = own ? (pc == 2 || pc == 4 || (SORTED && pc == 0)) : (pc == 0 || pc == 2);
            if (hit) {
              if (FILL) cand[base + cnt] = (int32_t)(sErep[i] & ~kSwapBit);
              cnt++;
            }
          }
        }
      }
    }
    // same beta-group, up doubles: one warp per row (coalesced scan of the beta-major view)
    __syncthreads();
    s_cnt[threadIdx.x] = cnt;
    s_row[threadIdx.x] = active ? (int32_t)threadIdx.x : -1;
    __syncthreads();
    const unsigned lt_mask = (1u << lane) - 1u;
    for (int rr = warp; rr < T.n; rr += kConnTile / 32) {
      if (s_row[rr] < 0) continue;
      const int64_t e2 = part ? (int64_t)V.Pidx[T.e0 + rr] : T.e0 + rr;  // entry == row when the view is partitioned (no time-reversal expansion)
      const Bits<NW> a2 = b_load<NW>(V.Ea, e2);
      const int64_t p2 = part ? e2 : (int64_t)V.Erep[e2];
      const bool new2 = !old_of_new || old_of_new[p2] < 0;
      const int64_t base2 = FILL ? cand_ptr[p2 - row_begin] + (olen ? olen[p2] : 0) : 0;
      int c2 = s_cnt[rr];
      if (FILL && SORTED && lane == 0) alen[p2 - row_begin] = c2;
      const int32_t gb = V.eB[e2];
      const int64_t lo = V.gB_off[gb], hi = V.gB_off[gb + 1];
      for (int64_t tb = lo; tb < hi; tb += 32) {
        const int64_t k = tb + lane;
        const bool in = k < hi;
        const int pc = in ? b_popc_xor(a2, b_load<NW>(V.EBa, k)) : 0;
        const bool hit = in && pc == 4 && (new2 || old_of_new[V.EBrep[k] & ~kSwapBit] < 0);
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (FILL && hit) cand[base2 + c2 + __popc(m & lt_mask)] = (int32_t)(V.EBrep[k] & ~kSwapBit);
        c2 += __popc(m);
      }
      if (!FILL && lane == 0) counts[p2 - row_begin] = c2;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ candidate generation by bitmap probes
// The tiled XOR/popcount join above tests a row's beta string against EVERY entry of EVERY neighbour alpha group (~670 tests per
// (row, group) at n = 10^7, ~1.5 % hits).  For a neighbour group (alpha' one excitation from alpha) the hits are exactly the
// entries (alpha', beta') with beta' in {beta} U singles(beta).  So with
//   * the unique beta strings numbered in sorted order (beta ids = beta groups), their single-excitation adjacency lists
//     (ascending ids, the string itself included; same (N-1)-key construction as for the alpha groups), and
//   * per alpha group a bitmap over beta ids ("is (alpha, beta) in the list?") with the popcount prefix of every word
//     (entries of a group are beta-sorted, so rank in the bitmap = position inside the group),
// a row probes ~89 bits per neighbour group instead of scanning it, and the hits still come out in ascending order.
// The row's own group (beta doubles count too) is still scanned, as are the same-beta up-doubles.
struct BmpView {
  const uint32_t *bm, *rk;    // [nA][W] membership bits over beta ids / set bits in front of each word
  const uint32_t *bmN, *rkN;  // incremental build: the same over the NEW entries only (rank inside the group's new part)
  int W;
  const int64_t *nbrB_off;    // [nB+1]
  const int32_t *nbrB;        // beta ids one excitation away (+ itself), ascending
};
__global__ void bitmap_set_kernel(const int32_t *eA, const int32_t *eB, const int32_t *old_of_new /* null: all entries */, int64_t n, int W, uint32_t *bm) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n) return;
  if (old_of_new && old_of_new[e] >= 0) return;
  const int32_t b = eB[e];
  atomicOr(bm + (int64_t)eA[e] * W + (b >> 5), 1u << (b & 31));
}
// one warp per alpha group: exclusive prefix of the popcounts of its bitmap words
__global__ void __launch_bounds__(256) bitmap_rank_kernel(const uint32_t *bm, int64_t nA, int W, uint32_t *rk) {
  const int lane = threadIdx.x & 31;
  const int64_t g = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (g >= nA) return;
  uint32_t run = 0;
  for (int w0 = 0; w0 < W; w0 += 32) {
    const int w = w0 + lane;
    const uint32_t c = w < W ? __popc(bm[g * W + w]) : 0;
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (w < W) rk[g * W + w] = run + incl - c;
    run += __shfl_sync(0xffffffffu, incl, 31);
  }
}

// STG: every thread's probe list (the ids of {beta} U singles(beta), <= lmax of them, ids < 65536) is staged ONCE per tile in shared
// memory, transposed ([k][thread]: conflict-free), instead of being re-read from global memory for each of the ~89 neighbour groups --
// those reads are uncoalesced (one cache line per lane: 32 L1 wavefronts per warp instruction) and made the probe loop L1-bound.
template <int NW, bool FILL, bool STG>
__global__ void __launch_bounds__(kConnTile) connect_bitmap_kernel(ConnView V, BmpView B, const TileDesc *tiles, int64_t ntiles, int64_t row_begin,
                                                                   int32_t *counts, const int64_t *cand_ptr, int32_t *cand, int32_t *alen,
                                                                   const int32_t *old_of_new, const int32_t *olen) {
  extern __shared__ uint32_t s_words[];  // bitmap row [W], rank row [W], (STG) probe lists [lmax][kConnTile] as 16-bit ids
  __shared__ uint64_t sEb[kBmpStage * NW];
  __shared__ uint32_t sErep[FILL ? kBmpStage : 1];
  __shared__ int32_t s_cnt[kConnTile];
  __shared__ int32_t s_row[kConnTile];
  uint32_t *s_bm = s_words, *s_rk = s_words + B.W;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    const TileDesc T = tiles[t];
    const int64_t e = T.e0 + threadIdx.x;
    const bool active = threadIdx.x < T.n;
    const bool part = V.Pidx != nullptr;  // rows come from the partitioned view (incremental build)
    const int64_t p = active ? (part ? (int64_t)V.Pidx[e] : e) : -1;  // entry == row: no time-reversal expansion on this path
    Bits<NW> b = b_zero<NW>();
    if (active) b = b_load<NW>(part ? V.Pb : V.Eb, e);
    const bool only_new = part && T.kind == 1;  // a row of the previous list: pairs with new determinants only
    int64_t base = 0;
    if (FILL && active) base = cand_ptr[p - row_begin] + (olen ? olen[p] : 0);
    int cnt = 0;
    int64_t nb0 = 0, nb1 = 0;
    if (active) {
      const int32_t bid = V.eB[p];
      nb0 = B.nbrB_off[bid];
      nb1 = B.nbrB_off[bid + 1];
    }
    uint16_t *s_ids = reinterpret_cast<uint16_t *>(s_words + 2 * B.W);
    if (STG) {  // every thread fills and reads only its own column: no barrier needed
      for (int64_t k = nb0; k < nb1; k++) s_ids[(k - nb0) * kConnTile + threadIdx.x] = (uint16_t)__ldg(B.nbrB + k);
    }
    const int g = T.g;
    for (int64_t q = V.nbr_off[g]; q < V.nbr_off[g + 1]; q++) {
      const int32_t g2 = V.nbr[q];
      if (g2 == g) {
        // own group: beta singles and doubles (and the row itself) -> scan the staged strings
        const int64_t lo = only_new ? V.gNew_off[g2] : V.gA_off[g2], hi = V.gA_off[g2 + 1];
        const uint64_t *cEb = only_new ? V.Pb : V.Eb;
        for (int64_t s0 = lo; s0 < hi; s0 += kBmpStage) {
          const int ns = (int)min((int64_t)kBmpStage, hi - s0);
          __syncthreads();
          for (int i = threadIdx.x; i < ns; i += blockDim.x) {
#pragma unroll
            for (int w = 0; w < NW; w++) sEb[i * NW + w] = cEb[(s0 + i) * NW + w];
            if (FILL) sErep[i] = only_new ? (uint32_t)V.Pidx[s0 + i] : (uint32_t)(s0 + i);
          }
          __syncthreads();
          if (active) {
            if (!FILL) {
#pragma unroll 8
              for (int i = 0; i < ns; i++) {
                int pc = 0;
#pragma unroll
                for (int w = 0; w < NW; w++) pc += __popcll(b.w[w] ^ sEb[i * NW + w]);
                cnt += (pc == 0 || pc == 2 || pc == 4);
              }
            } else {  // tests of 32 staged strings collected in a mask, then only the hits are walked (see the probes below)
              for (int i0 = 0; i0 < ns; i0 += 32) {
                const int ni = min(32, ns - i0);
                uint32_t hm = 0;
#pragma unroll 8
                for (int j = 0; j < ni; j++) {
                  int pc = 0;
#pragma unroll
                  for (int w = 0; w < NW; w++) pc += __popcll(b.w[w] ^ sEb[(i0 + j) * NW + w]);
                  hm |= (uint32_t)(pc == 0 || pc == 2 || pc == 4) << j;
                }
                while (hm) {
                  const int j = __ffs(hm) - 1;
                  hm &= hm - 1;
                  cand[base + cnt] = (int32_t)sErep[i0 + j];
                  cnt++;
                }
              }
            }
          }
        }
      } else {
        // neighbour group: probe the bits of {beta} U singles(beta)
        const uint32_t *bmrow = (only_new ? B.bmN : B.bm) + (int64_t)g2 * B.W;
        const uint32_t *rkrow = (only_new ? B.rkN : B.rk) + (int64_t)g2 * B.W;
        __syncthreads();
        for (int i = threadIdx.x; i < B.W; i += blockDim.x) { s_bm[i] = bmrow[i]; s_rk[i] = rkrow[i]; }
        __syncthreads();
        const int64_t pos0 = only_new ? V.gNew_off[g2] : V.gA_off[g2];
        auto probe_id = [&](int64_t k) -> int32_t { return STG ? (int32_t)s_ids[(k - nb0) * kConnTile + threadIdx.x] : __ldg(B.nbrB + k); };
        if (!FILL) {
          for (int64_t k = nb0; k < nb1; k++) {
            const int32_t id = probe_id(k);
            cnt += (int)((s_bm[id >> 5] >> (id & 31)) & 1u);
          }
        } else if (!STG) {  // ids come from global memory: one pass, test and emit together
          for (int64_t k = nb0; k < nb1; k++) {
            const int32_t id = __ldg(B.nbrB + k);
            const uint32_t w = s_bm[id >> 5];
            const int bit = id & 31;
            if ((w >> bit) & 1u) {
              const int64_t pos = pos0 + s_rk[id >> 5] + __popc(w & ((1u << bit) - 1u));
              cand[base + cnt] = only_new ? V.Pidx[pos] : (int32_t)pos;
              cnt++;
            }
          }
        } else {
          // ~9 % of the probes hit, so almost every probe has SOME lane of the warp on the hit path: the tests of 32 probes are
          // collected in a mask first (branch-free) and only the set bits are walked -- ~7 instead of ~30 divergent hit-path
          // executions per 32 probes; hits still come out in ascending order
          for (int64_t k0 = nb0; k0 < nb1; k0 += 32) {
            const int nk = (int)min((int64_t)32, nb1 - k0);
            uint32_t hm = 0;
#pragma unroll 4
            for (int j = 0; j < nk; j++) {
              const int32_t id = probe_id(k0 + j);
              hm |= ((s_bm[id >> 5] >> (id & 31)) & 1u) << j;
            }
            while (hm) {
              const int j = __ffs(hm) - 1;
              hm &= hm - 1;
              const int32_t id = probe_id(k0 + j);
              const uint32_t w = s_bm[id >> 5];
              const int64_t pos = pos0 + s_rk[id >> 5] + __popc(w & ((1u << (id & 31)) - 1u));
              cand[base + cnt] = only_new ? V.Pidx[pos] : (int32_t)pos;
              cnt++;
            }
          }
        }
      }
    }
    // same beta-group, up doubles: one warp per row (coalesced scan of the beta-major view)
    __syncthreads();
    s_cnt[threadIdx.x] = cnt;
    s_row[threadIdx.x] = active ? (int32_t)threadIdx.x : -1;
    __syncthreads();
    const unsigned lt_mask = (1u << lane) - 1u;
    for (int rr = warp; rr < T.n; rr += kConnTile / 32) {
      if (s_row[rr] < 0) continue;
      const int64_t p2 = part ? (int64_t)V.Pidx[T.e0 + rr] : T.e0 + rr;
      const Bits<NW> a2 = b_load<NW>(V.Ea, p2);
      const bool new2 = !old_of_new || old_of_new[p2] < 0;
      const int64_t base2 = FILL ? cand_ptr[p2 - row_begin] + (olen ? olen[p2] : 0) : 0;
      int c2 = s_cnt[rr];
      if (FILL && lane == 0) alen[p2 - row_begin] = c2;
      const int32_t gb = V.eB[p2];
      const int64_t lo = V.gB_off[gb], hi = V.gB_off[gb + 1];
      for (int64_t tb = lo; tb < hi; tb += 32) {
        const int64_t k = tb + lane;
        const bool in = k < hi;
        const int pc = in ? b_popc_xor(a2, b_load<NW>(V.EBa, k)) : 0;
        const bool hit = in && pc == 4 && (new2 || old_of_new[V.EBrep[k] & ~kSwapBit] < 0);
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (FILL && hit) cand[base2 + c2 + __popc(m & lt_mask)] = (int32_t)(V.EBrep[k] & ~kSwapBit);
        c2 += __popc(m);
      }
      if (!FILL && lane == 0) counts[p2 - row_begin] = c2;
    }
    __syncthreads();
  }
}

// tiles covering the entries [e_lo, e_hi) (host; gA is the host copy of the alpha-group offsets)
static void make_conn_tiles(const std::vector<int64_t> &gA, int64_t e_lo, int64_t e_hi, std::vector<TileDesc> &tiles) {
  tiles.clear();
  if (e_hi <= e_lo) return;
  int64_t g = std::upper_bound(gA.begin(), gA.end(), e_lo) - gA.begin() - 1;
  for (; g + 1 < (int64_t)gA.size() && gA[g] < e_hi; g++) {
    int64_t a = std::max(gA[g], e_lo), b = std::min(gA[g + 1], e_hi);
    for (int64_t x = a; x < b; x += kConnTile) tiles.push_back({x, (int16_t)std::min<int64_t>(kConnTile, b - x), (int16_t)0, (int32_t)g});
  }
}
// incremental build: the rows of whole alpha groups [g_lo, g_hi) in the partitioned view (inside a group: the determinants of
// the previous list, then the new ones; gNew = first new position of every group): old rows meet only new candidates
static void make_conn_tiles_split(const std::vector<int64_t> &gA, const std::vector<int64_t> &gNew, int64_t g_lo, int64_t g_hi, std::vector<TileDesc> &tiles) {
  tiles.clear();
  for (int64_t g = g_lo; g < g_hi; g++) {
    for (int64_t x = gA[g]; x < gNew[g]; x += kConnTile) tiles.push_back({x, (int16_t)std::min<int64_t>(kConnTile, gNew[g] - x), (int16_t)1, (int32_t)g});
    for (int64_t x = gNew[g]; x < gA[g + 1]; x += kConnTile) tiles.push_back({x, (int16_t)std::min<int64_t>(kConnTile, gA[g + 1] - x), (int16_t)0, (int32_t)g});
  }
}

// ------------------------------------------------------------------ per-row sort of candidate columns
// all-ascending ("flip") bitonic network: correct for arbitrary length, see DESIGN.md
__device__ __forceinline__ void bitonic_sort_i32(int32_t *a, int len, int tid, int nthr, bool block_sync) {
  int np2 = 1;
  while (np2 < len) np2 <<= 1;
  for (int k = 2; k <= np2; k <<= 1) {
    // flip step
    for (int i = tid; i < np2; i += nthr) {
      int partner = i ^ (k - 1);
      if (partner > i && partner < len) {
        int32_t x = a[i], y = a[partner];
        if (x > y) { a[i] = y; a[partner] = x; }
      }
    }
    if (block_sync) __syncthreads(); else __syncwarp();
    for (int j = k >> 2; j > 0; j >>= 1) {
      for (int i = tid; i < np2; i += nthr) {
        int partner = i ^ j;
        if (partner > i && partner < len) {
          int32_t x = a[i], y = a[partner];
          if (x > y) { a[i] = y; a[partner] = x; }
        }
      }
      if (block_sync) __syncthreads(); else __syncwarp();
    }
  }
}
static const int kWarpSortMax = 256;    // rows up to this length: one warp, smem
static const int kBlockSortMax = 32768; // rows up to this length: one CTA, smem; longer: CTA in global memory

__global__ void __launch_bounds__(256) sort_rows_warp_kernel(const int64_t *ptr, const int32_t *len, int64_t nrows, int32_t *cand) {
  __shared__ int32_t sm[8][kWarpSortMax];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t row = blockIdx.x * 8ll + w;
  if (row >= nrows) return;
  int L = len[row];
  if (L <= 1 || L > kWarpSortMax) return;
  int32_t *src = cand + ptr[row];
  for (int i = lane; i < L; i += 32) sm[w][i] = src[i];
  __syncwarp();
  bitonic_sort_i32(sm[w], L, lane, 32, false);
  for (int i = lane; i < L; i += 32) src[i] = sm[w][i];
}
__global__ void __launch_bounds__(256) sort_rows_block_kernel(const int64_t *ptr, const int32_t *len, int64_t nrows, int32_t *cand) {
  extern __shared__ int32_t smb[];
  for (int64_t row = blockIdx.x; row < nrows; row += gridDim.x) {
    int L = len[row];
    if (L <= kWarpSortMax) continue;
    int32_t *src = cand + ptr[row];
    if (L <= kBlockSortMax) {
      for (int i = threadIdx.x; i < L; i += blockDim.x) smb[i] = src[i];
      __syncthreads();
      bitonic_sort_i32(smb, L, threadIdx.x, blockDim.x, true);
      for (int i = threadIdx.x; i < L; i += blockDim.x) src[i] = smb[i];
      __syncthreads();
    } else {
      bitonic_sort_i32(src, L, threadIdx.x, blockDim.x, true);
    }
  }
}

// ------------------------------------------------------------------ element evaluation + in-row compaction
// chem: does the element of this pair take the long path (a single excitation: ~nelec integral look-ups per spin, or a
// diagonal-like term of the symmetrised element) instead of the 1-2 look-ups of a double?
template <int NW, bool TS>
__device__ __forceinline__ bool chem_is_heavy(const Bits<NW> &iu, const Bits<NW> &id, const Bits<NW> &ju, const Bits<NW> &jd) {
  const int l1 = excitation_level(iu, id, ju, jd);
  if (!TS) return l1 == 1;
  bool heavy = l1 == 1 || l1 == 0;
  if (!b_eq(iu, id) && !b_eq(ju, jd)) {  // second term of hamiltonian_chem_time_sym (chemistry.f90:1355-1364)
    const int l2 = excitation_level(id, iu, ju, jd);
    heavy = heavy || l2 == 1 || l2 == 0;
  }
  return heavy;
}

// diagonal elements of the rows [row0, row0 + nloc) (internal order), one thread per row; kept in the handle (Davidson's
// preconditioner, the projector) and read by eval_kernel, whose body then holds no diagonal code at all
template <int NW, int MODEL, bool TS>
__global__ void diag_rows_kernel(ModelTables T, const uint64_t *up, const uint64_t *dn, const int32_t *perm, int64_t row0, int64_t nloc, double *out) {
  int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q >= nloc) return;
  const Bits<NW> u = b_load<NW>(up, row0 + q), d = b_load<NW>(dn, row0 + q);
  double v = model_hamiltonian<NW, MODEL, TS>(T, T.combine_2, u, d, u, d);
  if (MODEL == MODEL_HUBBARDK && T.hf_to_psit && perm[row0 + q] == 0) v = 0.0;  // first row = single zero diagonal entry (hubbard.f90:9636-9643)
  out[q] = v;
}

// One warp per row, specialised per model.  Pass 1 evaluates the element of every (sorted) candidate into vals[]:
// doubles at once; chem singles -- ten times the work -- are queued per warp and evaluated 32 at a time, so a warp never
// idles 31 lanes behind one single.  Pass 2 applies abs(H) > 1e-12 (chemistry.f90:9901; the diagonal is always kept,
// :9887-9890), drops duplicate candidates (time-reversed partners) and compacts cand / vals in place, in order.
template <int NW, int MODEL, bool TS>
__global__ void __launch_bounds__(256) eval_kernel(ModelTables T, const uint64_t *__restrict__ up, const uint64_t *__restrict__ dn, const int32_t *__restrict__ perm,
                                                   const double *__restrict__ diag, int64_t diag_row0, int64_t row_begin, int64_t row_end,
                                                   const int64_t *__restrict__ cand_ptr, const int32_t *__restrict__ cand_len, int32_t *cand, double *vals,
                                                   int32_t *row_nnz, int32_t *alen /* in: candidates of the first sorted run, out: kept ones; may be null */,
                                                   const int32_t *olen /* incremental build: entries of the previous matrix in front of the candidates */) {
  extern __shared__ int32_t c2s[];
  __shared__ int32_t s_q[8][64];
  const int32_t *c2 = T.combine_2;
  if (MODEL == MODEL_CHEM) {
    const int n1 = T.norb + 1;
    for (int i = threadIdx.x; i < n1 * n1; i += blockDim.x) c2s[i] = T.combine_2[i];
    __syncthreads();
    c2 = c2s;
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t p = row_begin + warp;
  if (p >= row_end) return;
  const unsigned full = 0xffffffffu, lt_mask = (1u << lane) - 1u;
  const Bits<NW> pu = b_load<NW>(up, p), pd = b_load<NW>(dn, p);
  const int32_t cp = perm[p];
  const int ol = olen ? olen[p] : 0;
  const int64_t base = cand_ptr[warp] + ol;
  const int L = cand_len[warp];
  // ---- pass 1: values.  Every trip of the loop gives each lane at most one job (a candidate position to evaluate): a
  // scan trip classifies the next 32 candidates -- light ones become the lane's job, chem singles go to the warp's queue --
  // and a drain trip hands out 32 queued singles.  The element code is instantiated once, at the single job site below.
  int qn = 0;  // queued singles (warp-uniform)
  int kb = 0;
  while (true) {
    int job = -1;
    // a light job found by the scan trip keeps its candidate (row index, strings, orientation) in registers; a queued single is
    // loaded at the job site
    int32_t j = -1;
    Bits<NW> ku = b_zero<NW>(), kd = b_zero<NW>();
    bool fwd = true, loaded = false;
    if (MODEL == MODEL_CHEM && (qn >= 32 || (kb >= L && qn > 0))) {
      const int take = min(qn, 32);
      if (lane < take) job = s_q[w][lane];
      const int rest = (32 + lane < qn) ? s_q[w][32 + lane] : 0;
      __syncwarp();
      s_q[w][lane] = rest;
      qn -= take;
      __syncwarp();
    } else if (kb < L) {
      const int k = kb + lane;
      const bool in = k < L;
      j = in ? cand[base + k] : -1;
      const int32_t jprev = (TS && in && k > 0) ? cand[base + k - 1] : -2;
      const bool todo = in && j != (int32_t)p && j != jprev;
      bool heavy = false;
      if (todo) {
        ku = b_load<NW>(up, j);
        kd = b_load<NW>(dn, j);
        fwd = cp < perm[j];  // the reference stores H(i,j) for caller index i<j with det_i as bra: evaluate in that orientation
        loaded = true;
        if (MODEL == MODEL_CHEM) heavy = fwd ? chem_is_heavy<NW, TS>(pu, pd, ku, kd) : chem_is_heavy<NW, TS>(ku, kd, pu, pd);
      }
      if (todo && !heavy) job = k;
      if (MODEL == MODEL_CHEM) {
        const unsigned hm = __ballot_sync(full, heavy);
        if (heavy) s_q[w][qn + __popc(hm & lt_mask)] = k;
        qn += __popc(hm);
        __syncwarp();
      }
      kb += 32;
    } else {
      break;
    }
    if (job >= 0) {
      if (!loaded) {
        j = cand[base + job];
        ku = b_load<NW>(up, j);
        kd = b_load<NW>(dn, j);
        fwd = cp < perm[j];
      }
      Bits<NW> bu = pu, bd = pd;
      if (!fwd) {
        Bits<NW> t = bu; bu = ku; ku = t;
        t = bd; bd = kd; kd = t;
      }
      vals[base + job] = model_hamiltonian<NW, MODEL, TS>(T, c2, bu, bd, ku, kd);
    }
  }
  __syncwarp();
  // ---- pass 2: filter + ordered in-place compaction
  const int asplit = alen ? alen[warp] : L;
  int kept = 0, kept_a = 0;
  for (int kb = 0; kb < L; kb += 32) {
    const int k = kb + lane;
    const bool in = k < L;
    const int32_t j = in ? cand[base + k] : -1;
    const int32_t jprev = (TS && in && k > 0) ? cand[base + k - 1] : -2;
    bool keep = false;
    double v = 0.0;
    if (in && j != jprev) {
      if (j == (int32_t)p) {
        v = diag[p - diag_row0];
        keep = true;
      } else {
        v = vals[base + k];
        keep = fabs(v) > 1.e-12;
        if (MODEL == MODEL_HUBBARDK && T.hf_to_psit && (cp == 0 || perm[j] == 0)) keep = false;  // no row links to the first state
      }
    }
    __syncwarp();
    const unsigned m = __ballot_sync(full, keep);
    if (keep) {
      const int pos = kept + __popc(m & lt_mask);
      cand[base + pos] = j;
      vals[base + pos] = v;
    }
    kept += __popc(m);
    if (alen) kept_a += __popc(__ballot_sync(full, keep && k < asplit));
    __syncwarp();
  }
  if (lane == 0) {
    row_nnz[warp] = kept + ol;
    if (alen) alen[warp] = kept_a;
  }
}

// copy compacted rows to their final place.  A row is up to three ascending runs that share no column: the entries taken
// over from the previous matrix (olen, incremental build), the candidates of the alpha part (alen) and the same-beta
// up-doubles (the rest).  They are merged on the way: an entry's final position = its index in its own run + the entries
// of the other runs that sort before it (binary searches).  alen == null: one run (rows were sorted), plain copy.
__device__ __forceinline__ int lower_bound_i32(const int32_t *a, int n, int32_t c) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < c) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}
__global__ void __launch_bounds__(256) compact_copy_kernel(const int64_t *cand_ptr, const int32_t *row_nnz, const int32_t *alen, const int32_t *olen,
                                                           int64_t row_begin, const int64_t *rowptr_chunk, int64_t nrows, const int32_t *cand,
                                                           const double *vals, int32_t *cols_out, double *vals_out) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (row >= nrows) return;
  const int64_t src = cand_ptr[row], dst = rowptr_chunk[row];
  const int L = row_nnz[row];
  const int KO = olen ? olen[row_begin + row] : 0;
  const int KA = alen ? alen[row] : L - KO;
  const int KB = L - KO - KA;
  if ((KO == L) || (KO == 0 && KB == 0) ) {
    for (int k = lane; k < L; k += 32) {
      cols_out[dst + k] = cand[src + k];
      vals_out[dst + k] = vals[src + k];
    }
    return;
  }
  const int32_t *O = cand + src, *A = O + KO, *B = A + KA;
  for (int k = lane; k < L; k += 32) {
    const int32_t c = cand[src + k];
    int pos;
    if (k < KO) pos = k + lower_bound_i32(A, KA, c) + lower_bound_i32(B, KB, c);
    else if (k < KO + KA) pos = (k - KO) + lower_bound_i32(O, KO, c) + lower_bound_i32(B, KB, c);
    else pos = (k - KO - KA) + lower_bound_i32(O, KO, c) + lower_bound_i32(A, KA, c);
    cols_out[dst + pos] = c;
    vals_out[dst + pos] = vals[src + k];
  }
}

// ---- incremental build helpers (chemistry.f90:7769-7843: rows 1..ndet_old are kept and only extended)
// old_of_new[p] = row of the previous matrix that holds determinant p of the new internal order, -1 for a new determinant
__global__ void old_of_new_kernel(const int32_t *perm_new, const int32_t *iperm_old, int64_t n, int64_t n_old, int32_t *old_of_new) {
  int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int32_t cr = perm_new[p];
  old_of_new[p] = cr < n_old ? iperm_old[cr] : -1;
}
__global__ void new_of_old_kernel(const int32_t *perm_old, const int32_t *iperm_new, int64_t n_old, int32_t *new_of_old) {
  int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q < n_old) new_of_old[q] = iperm_new[perm_old[q]];
}
__global__ void old_len_kernel(const int32_t *old_of_new, const int64_t *rowptr_old, int64_t n, int32_t *olen) {
  int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int32_t q = old_of_new[p];
  olen[p] = q >= 0 ? (int32_t)(rowptr_old[q + 1] - rowptr_old[q]) : 0;
}
__global__ void is_new_kernel(const int32_t *old_of_new, int64_t n, int32_t *flag) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e <= n) flag[e] = (e < n && old_of_new[e] < 0) ? 1 : 0;
}
// stable partition inside every alpha group: previous determinants first, new ones after (newrank = exclusive scan of is_new)
template <int NW>
__global__ void partition_view_kernel(const int32_t *old_of_new, const int32_t *newrank, const int32_t *eA, const int64_t *gA_off, const uint64_t *Eb, int64_t n,
                                      int32_t *Pidx, uint64_t *Pb) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n) return;
  const int32_t g = eA[e];
  const int64_t s = gA_off[g], e1 = gA_off[g + 1];
  const int64_t nn_before = newrank[e] - newrank[s];
  const int64_t nold_g = (e1 - s) - (newrank[e1] - newrank[s]);
  const int64_t pos = old_of_new[e] < 0 ? s + nold_g + nn_before : s + (e - s) - nn_before;
  Pidx[pos] = (int32_t)e;
  b_store<NW>(Pb, pos, b_load<NW>(Eb, e));
}
__global__ void group_new_off_kernel(const int32_t *newrank, const int64_t *gA_off, int64_t nA, int64_t *gNew_off) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g > nA) return;
  if (g == nA) { gNew_off[g] = gA_off[nA]; return; }
  const int64_t s = gA_off[g], e1 = gA_off[g + 1];
  gNew_off[g] = e1 - (newrank[e1] - newrank[s]);
}
__global__ void gather_i64_kernel(const int64_t *src, const int64_t *idx, int64_t *dst, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[idx[i]];
}
__global__ void add_i32_kernel(const int32_t *a, const int32_t *b, int32_t *out, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] + b[i];
}
// rows [row_begin, row_begin + nrows): copy the row's old entries (columns renumbered; the map is monotone, so they stay
// ascending) in front of its candidates in the chunk's temporaries.  One warp per row.
__global__ void __launch_bounds__(256) copy_old_rows_kernel(const int32_t *old_of_new, const int64_t *rowptr_old, const int32_t *cols_old, const double *vals_old,
                                                            const int32_t *new_of_old, int64_t row_begin, int64_t nrows, const int64_t *cand_ptr,
                                                            int32_t *cand, double *vals) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (row >= nrows) return;
  const int32_t q = old_of_new[row_begin + row];
  if (q < 0) return;
  const int64_t b = rowptr_old[q], e = rowptr_old[q + 1], dst = cand_ptr[row];
  for (int64_t k = b + lane; k < e; k += 32) {
    cand[dst + (k - b)] = new_of_old[cols_old[k]];
    vals[dst + (k - b)] = vals_old[k];
  }
}

__global__ void add_offset_kernel(int64_t *a, int64_t n, int64_t off) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) a[i] += off;
}

template <int NW, int MODEL, bool TS>
__global__ void diag_kernel(ModelTables T, const uint64_t *up, const uint64_t *dn, int64_t n, double *out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  Bits<NW> u = b_load<NW>(up, i), d = b_load<NW>(dn, i);
  out[i] = model_hamiltonian<NW, MODEL, TS>(T, T.combine_2, u, d, u, d);
}

// exclusive scan int32 -> int64 offsets (n+1 outputs)
static int exclusive_scan_i32_to_i64(const int32_t *in, int64_t *out, int64_t n, cudaStream_t s) {
  size_t tb = 0;
  auto it = cub::TransformInputIterator<int64_t, cub::CastOp<int64_t>, const int32_t *>(in, cub::CastOp<int64_t>());
  cub::DeviceScan::ExclusiveSum(nullptr, tb, it, out, (int)(n + 1), s);
  DevBuf<char> tmp;
  SQ_CHECK(tmp.alloc((int64_t)tb + 16));
  // scanning n+1 items reads in[n]: callers allocate counts with one spare zeroed slot
  SQ_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb, it, out, (int)(n + 1), s));
  g_launch_count += 2;
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// same scan with caller-provided temporary storage and no synchronisation (the chunk loop of the build stays asynchronous)
static int exclusive_scan_i32_to_i64_async(const int32_t *in, int64_t *out, int64_t n, void *tmp, size_t tmp_bytes, cudaStream_t s) {
  auto it = cub::TransformInputIterator<int64_t, cub::CastOp<int64_t>, const int32_t *>(in, cub::CastOp<int64_t>());
  size_t tb = tmp_bytes;
  SQ_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, it, out, (int)(n + 1), s));
  g_launch_count += 2;
  return 0;
}
static size_t exclusive_scan_tmp_bytes(int64_t n) {
  size_t tb = 0;
  auto it = cub::TransformInputIterator<int64_t, cub::CastOp<int64_t>, const int32_t *>((const int32_t *)nullptr, cub::CastOp<int64_t>());
  cub::DeviceScan::ExclusiveSum(nullptr, tb, it, (int64_t *)nullptr, (int)(n + 1));
  return tb;
}
__global__ void add_offset_dev_kernel(int64_t *a, int64_t n, const int64_t *off) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) a[i] += *off;
}
__global__ void set_scalar_kernel(int64_t *dst, const int64_t *src) { *dst = *src; }

// ---- helpers shared with select.cu
// upload n 16-byte determinants (host) and split them into NW-word strings (device, caller allocates n*NW words)
int upload_dets(int NW, int norb, const void *host16, uint64_t *out, int64_t n, cudaStream_t s) {
  DevBuf<uint64_t> raw;
  DevBuf<int> bad;
  SQ_CHECK(raw.alloc(2 * n));
  SQ_CHECK(bad.alloc(1));
  SQ_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), s));
  uint64_t m0 = 0, m1 = 0;
  if (norb < 64) { m0 = ~((1ull << norb) - 1ull); m1 = ~0ull; }
  else if (norb == 64) { m0 = 0; m1 = ~0ull; }
  else { m0 = 0; m1 = (norb >= 128) ? 0ull : ~((1ull << (norb - 64)) - 1ull); }
  SQ_CUDA(cudaMemcpyAsync(raw.p, host16, (size_t)n * 16, cudaMemcpyHostToDevice, s));
  if (NW == 1) split_dets_kernel<1><<<nblocks(n), kThreads, 0, s>>>(raw.p, out, n, bad.p, m0, m1);
  else split_dets_kernel<2><<<nblocks(n), kThreads, 0, s>>>(raw.p, out, n, bad.p, m0, m1);
  SQ_LAUNCH_CHECK();
  int hbad = 0;
  SQ_CUDA(cudaMemcpyAsync(&hbad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  if (hbad) { set_error("a determinant occupies an orbital beyond norb=%d", norb); return 2; }
  return 0;
}
// idx (device, n entries, initialised here) := permutation sorting the pairs (a, b) ascending, a most significant
int sort_pairs_index(int NW, int norb, const uint64_t *a, const uint64_t *b, int32_t *idx, int64_t n, cudaStream_t s) {
  if (n == 0) return 0;
  iota_kernel<<<nblocks(n), kThreads, 0, s>>>(idx, n);
  SQ_LAUNCH_CHECK();
  std::vector<KeyWord> words;
  for (int w = 0; w < NW; w++) words.push_back({b, NW, w, std::min(64, norb - 64 * w)});
  for (int w = 0; w < NW; w++) words.push_back({a, NW, w, std::min(64, norb - 64 * w)});
  return sort_by_words(words, idx, n, s);
}
int gather_strings(int NW, const uint64_t *src, const int32_t *idx, uint64_t *out, int64_t n, cudaStream_t s) {
  if (n == 0) return 0;
  if (NW == 1) gather_bits_kernel<1><<<nblocks(n), kThreads, 0, s>>>(src, idx, out, n);
  else gather_bits_kernel<2><<<nblocks(n), kThreads, 0, s>>>(src, idx, out, n);
  SQ_LAUNCH_CHECK();
  return 0;
}

void free_matrix(sqmc_b200_handle *h) {
  // per-build arrays come from the stream-ordered pool (devbuf_alloc): freeing and re-allocating them costs no unmapping
  auto F = [](auto *&p) {
    if (p) devbuf_free(p);
    p = nullptr;
  };
  F(h->d_up); F(h->d_dn); F(h->d_perm); F(h->d_iperm); F(h->d_rowptr);
  // d_cols / d_vals live in the growable arrays: they keep their memory for the next build (released by matrix_arrays_release)
  F(h->d_bin_rows); F(h->d_x); F(h->d_y); F(h->d_tmp); F(h->d_x2); F(h->d_xi2); F(h->d_y2);
  F(h->d_shuf_of_internal); F(h->d_dest_rank); F(h->d_dest_pos); F(h->d_my_internal);
  h->own_set = false; h->my_n = 0; h->own_count.clear(); h->own_off.clear();
  F(h->d_diag);
  x_textures_release(h);
  h->bins_ready = false;
  h->bundle_R = 0;
  h->n = 0; h->nnz_local = 0; h->nnz_full = 0; h->nnz_upper = 0; h->capacity = 0; h->scale = 1.0;
  h->row_starts.clear();
}

// reserve (once) and map the two entry arrays for `entries` stored entries
int matrix_arrays_ensure(sqmc_b200_handle *h, int64_t entries) {
  if (!h->g_cols.base) {
    size_t fr = 0, tot = 0;
    SQ_CUDA(cudaMemGetInfo(&fr, &tot));
    const size_t max_entries = tot / 12 + (1 << 20);  // the device cannot hold more than this
    SQ_CHECK(grow_reserve(h->g_cols, max_entries * sizeof(int32_t)));
    SQ_CHECK(grow_reserve(h->g_vals, max_entries * sizeof(double)));
  }
  SQ_CHECK(grow_ensure(h->g_cols, (size_t)(entries + kSlack) * sizeof(int32_t)));
  SQ_CHECK(grow_ensure(h->g_vals, (size_t)(entries + kSlack) * sizeof(double)));
  h->d_cols = reinterpret_cast<int32_t *>(h->g_cols.base);
  h->d_vals = reinterpret_cast<double *>(h->g_vals.base);
  return 0;
}
// called when a device allocation failed: unmap what the matrices do not use
void matrix_arrays_release_surplus() {
  for (sqmc_b200_handle *h : g_handles) {
    if (!h->g_cols.base) continue;
    const int64_t keep = h->d_rowptr ? h->capacity + kSlack : 0;
    grow_trim(h->g_cols, (size_t)keep * sizeof(int32_t));
    grow_trim(h->g_vals, (size_t)keep * sizeof(double));
  }
}
void matrix_arrays_release(sqmc_b200_handle *h) {
  grow_release(h->g_cols);
  grow_release(h->g_vals);
  h->d_cols = nullptr;
  h->d_vals = nullptr;
}

// the previous matrix, detached from the handle while an incremental build extends it
struct OldMatrix {
  int64_t n = 0, nnz = 0;
  int32_t *d_perm = nullptr, *d_iperm = nullptr;
  int64_t *d_rowptr = nullptr;
  ~OldMatrix() {
    if (d_perm) devbuf_free(d_perm);
    if (d_iperm) devbuf_free(d_iperm);
    if (d_rowptr) devbuf_free(d_rowptr);
  }
};
struct EventSet {  // timing events of one build, destroyed on every exit path
  cudaEvent_t e[5];
  EventSet() { for (auto &x : e) cudaEventCreate(&x); }
  ~EventSet() { for (auto &x : e) cudaEventDestroy(x); }
};

static int alloc_work_vectors(sqmc_b200_handle *h) {
  SQ_CHECK(p2p_setup(h, h->n));  // collective: (re)maps the peers' exchange buffers when the vectors outgrew them
  SQ_CHECK(devbuf_alloc((void **)&h->d_x, std::max<int64_t>(h->n, 1) * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&h->d_y, std::max<int64_t>(h->row1 - h->row0, 1) * sizeof(double)));
  SQ_CHECK(devbuf_alloc((void **)&h->d_tmp, std::max<int64_t>(h->n, 1) * sizeof(double)));
  return 0;
}

// Contiguous row blocks balanced by work: rank r gets rows [starts[r], starts[r+1]) such that the
// exclusive prefix `prefix` (n+1 entries, prefix[n] = total) is split as evenly as possible.
void partition_rows(const int64_t *prefix, int64_t n, int nranks, int64_t *starts) {
  const int64_t total = prefix[n];
  starts[0] = 0;
  for (int r = 1; r < nranks; r++) {
    int64_t target = (total / nranks) * r + ((total % nranks) * r) / nranks;
    int64_t pos = std::lower_bound(prefix, prefix + n + 1, target) - prefix;
    if (pos > n) pos = n;
    if (pos < starts[r - 1]) pos = starts[r - 1];
    starts[r] = pos;
  }
  starts[nranks] = n;
}

// Sorted single-excitation neighbour lists of a set of unique strings: string g is str[g_off[g]] (first member of group g of a
// sorted array).  Two strings are one excitation apart iff they share an (N-1)-electron key (the alpha_m1 idea of
// chemistry.f90:9819 applied to unique strings): keys are sorted, the run of a key lists the strings that contain it.
// nbr[nbr_off[g] .. nbr_off[g+1]) = g itself and its neighbours, ascending.
template <int NW>
static int neighbour_lists(const uint64_t *str, const int64_t *g_off, int64_t ng, int nel, int norb, DevBuf<int64_t> &nbr_off, DevBuf<int32_t> &nbr,
                           cudaStream_t s) {
  const int64_t m2 = ng * nel;
  DevBuf<uint64_t> K_keys_u, K_keys;
  DevBuf<int32_t> K_grp_u, K_grp, kidx, run_lo, run_hi, nbr_cnt;
  SQ_CHECK(K_keys_u.alloc(std::max<int64_t>(m2, 1) * NW));
  SQ_CHECK(K_grp_u.alloc(std::max<int64_t>(m2, 1)));
  SQ_CHECK(K_keys.alloc(std::max<int64_t>(m2, 1) * NW));
  SQ_CHECK(K_grp.alloc(std::max<int64_t>(m2, 1)));
  SQ_CHECK(kidx.alloc(std::max<int64_t>(m2, 1)));
  SQ_CHECK(run_lo.alloc(std::max<int64_t>(m2, 1)));
  SQ_CHECK(run_hi.alloc(std::max<int64_t>(m2, 1)));
  if (m2 > 0) {
    nm1_keys_kernel<NW><<<nblocks(ng), kThreads, 0, s>>>(str, g_off, ng, nel, K_keys_u.p, K_grp_u.p);
    SQ_LAUNCH_CHECK();
    iota_kernel<<<nblocks(m2), kThreads, 0, s>>>(kidx.p, m2);
    SQ_LAUNCH_CHECK();
    std::vector<KeyWord> words;
    for (int w = 0; w < NW; w++) words.push_back({K_keys_u.p, NW, w, std::min(64, norb - 64 * w)});
    SQ_CHECK(sort_by_words(words, kidx.p, m2, s));
    gather_bits_kernel<NW><<<nblocks(m2), kThreads, 0, s>>>(K_keys_u.p, kidx.p, K_keys.p, m2);
    SQ_LAUNCH_CHECK();
    gather_u32_kernel<<<nblocks(m2), kThreads, 0, s>>>((const uint32_t *)K_grp_u.p, kidx.p, (uint32_t *)K_grp.p, m2);
    SQ_LAUNCH_CHECK();
    nm1_runs_kernel<NW><<<nblocks(m2), kThreads, 0, s>>>(str, g_off, ng, nel, K_keys.p, m2, run_lo.p, run_hi.p);
    SQ_LAUNCH_CHECK();
  }
  SQ_CHECK(nbr_cnt.alloc(ng + 1));
  SQ_CHECK(nbr_off.alloc(ng + 1));
  SQ_CUDA(cudaMemsetAsync(nbr_cnt.p, 0, (ng + 1) * sizeof(int32_t), s));
  nbr_count_kernel<<<nblocks(ng), kThreads, 0, s>>>(run_lo.p, run_hi.p, ng, nel, nbr_cnt.p);
  SQ_LAUNCH_CHECK();
  SQ_CHECK(exclusive_scan_i32_to_i64(nbr_cnt.p, nbr_off.p, ng, s));
  int64_t nbr_total = 0;
  SQ_CUDA(cudaMemcpy(&nbr_total, nbr_off.p + ng, sizeof(int64_t), cudaMemcpyDeviceToHost));
  SQ_CHECK(nbr.alloc(std::max<int64_t>(nbr_total, 1)));
  nbr_fill_kernel<<<nblocks(ng), kThreads, 0, s>>>(run_lo.p, run_hi.p, K_grp.p, ng, nel, nbr_off.p, nbr.p);
  SQ_LAUNCH_CHECK();
  sort_rows_warp_kernel<<<nblocks(ng, 8), 256, 0, s>>>(nbr_off.p, nbr_cnt.p, ng, nbr.p);
  SQ_LAUNCH_CHECK();
  if ((int64_t)nel * (norb - nel) + 1 > kWarpSortMax) {  // more neighbours than the warp sort handles (large basis sets)
    SQ_CUDA(cudaFuncSetAttribute(sort_rows_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBlockSortMax * 4));
    sort_rows_block_kernel<<<(int)std::min<int64_t>(ng, 148 * 16), 256, kBlockSortMax * 4, s>>>(nbr_off.p, nbr_cnt.p, ng, nbr.p);
    SQ_LAUNCH_CHECK();
  }
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// ------------------------------------------------------------------ the build
template <int NW>
static int build_impl(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, OldMatrix *old) {
  cudaStream_t s = G.stream;
  const ModelTables &T = h->T;
  EventSet evset;
  cudaEvent_t *ev = evset.e;
  HostMarks HM;
  cudaEventRecord(ev[0], s);

  // ---- upload + split
  DevBuf<uint64_t> raw, up_c, dn_c;
  DevBuf<int> bad;
  SQ_CHECK(raw.alloc(2 * n));
  SQ_CHECK(up_c.alloc(n * NW));
  SQ_CHECK(dn_c.alloc(n * NW));
  SQ_CHECK(bad.alloc(1));
  SQ_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), s));
  uint64_t m0 = 0, m1 = 0;  // bits that must be zero
  if (T.norb < 64) { m0 = ~((1ull << T.norb) - 1ull); m1 = ~0ull; }
  else if (T.norb == 64) { m0 = 0; m1 = ~0ull; }
  else { m0 = 0; m1 = (T.norb >= 128) ? 0ull : ~((1ull << (T.norb - 64)) - 1ull); }
  for (int which = 0; which < 2; which++) {
    SQ_CUDA(cudaMemcpyAsync(raw.p, which == 0 ? dets_up : dets_dn, (size_t)n * 16, cudaMemcpyHostToDevice, s));
    split_dets_kernel<NW><<<nblocks(n), kThreads, 0, s>>>(raw.p, which == 0 ? up_c.p : dn_c.p, n, bad.p, m0, m1);
    SQ_LAUNCH_CHECK();
  }
  int hbad = 0;
  SQ_CUDA(cudaMemcpyAsync(&hbad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  raw.release();
  if (hbad) {
    set_error("build_h: a determinant occupies an orbital beyond norb=%d", T.norb);
    return 2;
  }

  // ---- internal (alpha-major) order
  SQ_CHECK(devbuf_alloc((void **)&h->d_perm, n * sizeof(int32_t)));
  SQ_CHECK(devbuf_alloc((void **)&h->d_iperm, n * sizeof(int32_t)));
  iota_kernel<<<nblocks(n), kThreads, 0, s>>>(h->d_perm, n);
  SQ_LAUNCH_CHECK();
  {
    std::vector<KeyWord> words;
    for (int w = 0; w < NW; w++) words.push_back({dn_c.p, NW, w, std::min(64, T.norb - 64 * w)});
    for (int w = 0; w < NW; w++) words.push_back({up_c.p, NW, w, std::min(64, T.norb - 64 * w)});
    SQ_CHECK(sort_by_words(words, h->d_perm, n, s));
  }
  invert_perm_kernel<<<nblocks(n), kThreads, 0, s>>>(h->d_perm, h->d_iperm, n);
  SQ_LAUNCH_CHECK();
  SQ_CHECK(devbuf_alloc((void **)&h->d_up, n * NW * sizeof(uint64_t)));
  SQ_CHECK(devbuf_alloc((void **)&h->d_dn, n * NW * sizeof(uint64_t)));
  gather_bits_kernel<NW><<<nblocks(n), kThreads, 0, s>>>(up_c.p, h->d_perm, h->d_up, n);
  SQ_LAUNCH_CHECK();
  gather_bits_kernel<NW><<<nblocks(n), kThreads, 0, s>>>(dn_c.p, h->d_perm, h->d_dn, n);
  SQ_LAUNCH_CHECK();
  SQ_CUDA(cudaStreamSynchronize(s));
  up_c.release();
  dn_c.release();
  h->n = n;
  // ---- incremental build: where the determinants of the previous list went
  DevBuf<int32_t> old_of_new, new_of_old, olen;
  if (old) {
    SQ_CHECK(old_of_new.alloc(n));
    SQ_CHECK(new_of_old.alloc(old->n));
    SQ_CHECK(olen.alloc(n + 1));
    old_of_new_kernel<<<nblocks(n), kThreads, 0, s>>>(h->d_perm, old->d_iperm, n, old->n, old_of_new.p);
    SQ_LAUNCH_CHECK();
    new_of_old_kernel<<<nblocks(old->n), kThreads, 0, s>>>(old->d_perm, h->d_iperm, old->n, new_of_old.p);
    SQ_LAUNCH_CHECK();
    SQ_CUDA(cudaMemsetAsync(olen.p + n, 0, sizeof(int32_t), s));
    old_len_kernel<<<nblocks(n), kThreads, 0, s>>>(old_of_new.p, old->d_rowptr, n, olen.p);
    SQ_LAUNCH_CHECK();
  }
  const int32_t *d_oon = old ? old_of_new.p : nullptr;
  const int32_t *d_olen = old ? olen.p : nullptr;

  // ---- expanded entry list E (alpha-major)
  const bool ts = (T.model == MODEL_CHEM) && T.time_sym;
  int64_t m = n;
  DevBuf<uint64_t> Ea_buf, Eb_buf;
  DevBuf<uint32_t> Erep_buf;
  DevBuf<int32_t> rowE_buf;
  const uint64_t *Ea = h->d_up, *Eb = h->d_dn;
  SQ_CHECK(Erep_buf.alloc(1));
  SQ_CHECK(rowE_buf.alloc(n));
  if (ts) {
    DevBuf<int32_t> flag, excl;
    SQ_CHECK(flag.alloc(n));
    SQ_CHECK(excl.alloc(n));
    ts_flag_kernel<NW><<<nblocks(n), kThreads, 0, s>>>(h->d_up, h->d_dn, flag.p, n);
    SQ_LAUNCH_CHECK();
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, flag.p, excl.p, (int)n, s);
    DevBuf<char> tmp;
    SQ_CHECK(tmp.alloc((int64_t)tb + 16));
    SQ_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb, flag.p, excl.p, (int)n, s));
    g_launch_count += 2;
    int32_t le = 0, lf = 0;
    SQ_CUDA(cudaMemcpyAsync(&le, excl.p + (n - 1), 4, cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaMemcpyAsync(&lf, flag.p + (n - 1), 4, cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
    m = n + le + lf;
    DevBuf<uint64_t> Ua, Ub;
    DevBuf<uint32_t> Urep;
    SQ_CHECK(Ua.alloc(m * NW));
    SQ_CHECK(Ub.alloc(m * NW));
    SQ_CHECK(Urep.alloc(m));
    ts_expand_kernel<NW><<<nblocks(n), kThreads, 0, s>>>(h->d_up, h->d_dn, flag.p, excl.p, Ua.p, Ub.p, Urep.p, n);
    SQ_LAUNCH_CHECK();
    DevBuf<int32_t> idx;
    SQ_CHECK(idx.alloc(m));
    iota_kernel<<<nblocks(m), kThreads, 0, s>>>(idx.p, m);
    SQ_LAUNCH_CHECK();
    std::vector<KeyWord> words;
    for (int w = 0; w < NW; w++) words.push_back({Ub.p, NW, w, std::min(64, T.norb - 64 * w)});
    for (int w = 0; w < NW; w++) words.push_back({Ua.p, NW, w, std::min(64, T.norb - 64 * w)});
    SQ_CHECK(sort_by_words(words, idx.p, m, s));
    SQ_CHECK(Ea_buf.alloc(m * NW));
    SQ_CHECK(Eb_buf.alloc(m * NW));
    SQ_CHECK(Erep_buf.alloc(m));
    gather_bits_kernel<NW><<<nblocks(m), kThreads, 0, s>>>(Ua.p, idx.p, Ea_buf.p, m);
    SQ_LAUNCH_CHECK();
    gather_bits_kernel<NW><<<nblocks(m), kThreads, 0, s>>>(Ub.p, idx.p, Eb_buf.p, m);
    SQ_LAUNCH_CHECK();
    gather_u32_kernel<<<nblocks(m), kThreads, 0, s>>>(Urep.p, idx.p, Erep_buf.p, m);
    SQ_LAUNCH_CHECK();
    SQ_CUDA(cudaStreamSynchronize(s));
    Ea = Ea_buf.p;
    Eb = Eb_buf.p;
  } else {
    SQ_CHECK(Erep_buf.alloc(m));
    iota_kernel<<<nblocks(m), kThreads, 0, s>>>((int32_t *)Erep_buf.p, m);
    SQ_LAUNCH_CHECK();
  }
  row_entry_kernel<<<nblocks(m), kThreads, 0, s>>>(Erep_buf.p, rowE_buf.p, m);
  SQ_LAUNCH_CHECK();

  // ---- alpha groups
  DevBuf<int32_t> eA;
  DevBuf<int64_t> gA_off;
  int64_t nA = 0;
  SQ_CHECK(make_groups<NW>(Ea, m, eA, gA_off, nA, s));

  // ---- beta-major view
  DevBuf<int32_t> bidx;
  SQ_CHECK(bidx.alloc(m));
  iota_kernel<<<nblocks(m), kThreads, 0, s>>>(bidx.p, m);
  SQ_LAUNCH_CHECK();
  {
    std::vector<KeyWord> words;  // entries are alpha-major already: a stable sort by b gives (b, a) order
    for (int w = 0; w < NW; w++) words.push_back({Eb, NW, w, std::min(64, T.norb - 64 * w)});
    SQ_CHECK(sort_by_words(words, bidx.p, m, s));
  }
  DevBuf<uint64_t> EBa, EBb;
  DevBuf<uint32_t> EBrep;
  SQ_CHECK(EBa.alloc(m * NW));
  SQ_CHECK(EBb.alloc(m * NW));
  SQ_CHECK(EBrep.alloc(m));
  gather_bits_kernel<NW><<<nblocks(m), kThreads, 0, s>>>(Ea, bidx.p, EBa.p, m);
  SQ_LAUNCH_CHECK();
  gather_bits_kernel<NW><<<nblocks(m), kThreads, 0, s>>>(Eb, bidx.p, EBb.p, m);
  SQ_LAUNCH_CHECK();
  gather_u32_kernel<<<nblocks(m), kThreads, 0, s>>>(Erep_buf.p, bidx.p, EBrep.p, m);
  SQ_LAUNCH_CHECK();
  DevBuf<int32_t> eB_sorted, eB;
  DevBuf<int64_t> gB_off;
  int64_t nB = 0;
  SQ_CHECK(make_groups<NW>(EBb.p, m, eB_sorted, gB_off, nB, s));
  SQ_CHECK(eB.alloc(m));
  scatter_gid_kernel<<<nblocks(m), kThreads, 0, s>>>(eB_sorted.p, bidx.p, eB.p, m);
  SQ_LAUNCH_CHECK();
  SQ_CUDA(cudaStreamSynchronize(s));
  eB_sorted.release();
  bidx.release();

  // ---- sorted neighbour-group list of every alpha group (itself + the groups of the strings one excitation away)
  const int nel = T.nup;  // time_sym requires nup == ndn (chemistry.f90:186)
  DevBuf<int64_t> nbr_off;
  DevBuf<int32_t> nbr;
  SQ_CHECK(neighbour_lists<NW>(Ea, gA_off.p, nA, nel, T.norb, nbr_off, nbr, s));
  // ---- bitmap-probe structures (connect_bitmap_kernel): beta adjacency over the unique beta strings, membership bitmaps
  // + ranks per alpha group.  Not with time-reversal expansion (entries != rows) and only while the bitmaps stay small.
  DevBuf<int64_t> nbrB_off;
  DevBuf<int32_t> nbrB;
  DevBuf<uint32_t> bm, rk, bmN, rkN;
  const int W = (int)div_up(nB, 32);
  // Probing pays when the alpha groups are large: the scanning join costs a row ~n/nA tests per neighbour group, a probe pass ~lmax
  // probes plus the staging of 2 W words per (tile, group).  HEG spaces have ~10 determinants per alpha string (137 220 / 15 024,
  // 10^6 / 73 111): there the scan is 3-4x faster (build of the 10^6-determinant HEG space: 0.10 s vs 0.47 s), so probes need
  // n >= 64 nA (C2 10^7: 669 per group, C2 10^6 lowest-energy: 96, Hubbard full sector: 804).
  const bool use_bmp = !ts && W <= 8192 && nA * (int64_t)W <= (1ll << 28) && n >= 64 * nA;
  if (use_bmp) {
    SQ_CHECK(neighbour_lists<NW>(EBb.p, gB_off.p, nB, T.ndn, T.norb, nbrB_off, nbrB, s));
    for (int pass = 0; pass < (old ? 2 : 1); pass++) {
      DevBuf<uint32_t> &bits = pass == 0 ? bm : bmN, &rank = pass == 0 ? rk : rkN;
      SQ_CHECK(bits.alloc(nA * W));
      SQ_CHECK(rank.alloc(nA * W));
      SQ_CUDA(cudaMemsetAsync(bits.p, 0, (size_t)nA * W * sizeof(uint32_t), s));
      bitmap_set_kernel<<<nblocks(n), kThreads, 0, s>>>(eA.p, eB.p, pass == 0 ? nullptr : old_of_new.p, n, W, bits.p);
      SQ_LAUNCH_CHECK();
      bitmap_rank_kernel<<<nblocks(nA * 32), 256, 0, s>>>(bits.p, nA, W, rank.p);
      SQ_LAUNCH_CHECK();
    }
  }
  // probe lists staged in shared memory when they are short enough (lmax = ndn (norb - ndn) + 1 ids per string) and the ids fit 16 bits
  const int probe_lmax = T.ndn * (T.norb - T.ndn) + 1;
  const bool stage_ids = use_bmp && nB <= 65535 && 2 * W * 4 + probe_lmax * kConnTile * 2 <= 160 * 1024;
  const int bmp_smem = 2 * W * 4 + (stage_ids ? probe_lmax * kConnTile * 2 : 0);
  if (use_bmp && bmp_smem > 24 * 1024) {
    SQ_CUDA(cudaFuncSetAttribute(connect_bitmap_kernel<NW, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bmp_smem));
    SQ_CUDA(cudaFuncSetAttribute(connect_bitmap_kernel<NW, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bmp_smem));
    SQ_CUDA(cudaFuncSetAttribute(connect_bitmap_kernel<NW, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bmp_smem));
    SQ_CUDA(cudaFuncSetAttribute(connect_bitmap_kernel<NW, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bmp_smem));
  }
  EBb.release();
  const BmpView BV{bm.p, rk.p, bmN.p, rkN.p, W, nbrB_off.p, nbrB.p};
  // incremental build: the partitioned row / candidate view
  DevBuf<int32_t> Pidx;
  DevBuf<uint64_t> Pb;
  DevBuf<int64_t> gNew_off;
  std::vector<int64_t> gNew_host;
  if (old) {
    DevBuf<int32_t> isnew, newrank;
    SQ_CHECK(isnew.alloc(n + 1));
    SQ_CHECK(newrank.alloc(n + 1));
    SQ_CHECK(Pidx.alloc(n));
    SQ_CHECK(Pb.alloc(n * NW));
    SQ_CHECK(gNew_off.alloc(nA + 1));
    is_new_kernel<<<nblocks(n + 1), kThreads, 0, s>>>(old_of_new.p, n, isnew.p);
    SQ_LAUNCH_CHECK();
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, isnew.p, newrank.p, (int)(n + 1), s);
    DevBuf<char> tmp;
    SQ_CHECK(tmp.alloc((int64_t)tb + 16));
    SQ_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb, isnew.p, newrank.p, (int)(n + 1), s));
    g_launch_count += 2;
    partition_view_kernel<NW><<<nblocks(n), kThreads, 0, s>>>(old_of_new.p, newrank.p, eA.p, gA_off.p, Eb, n, Pidx.p, Pb.p);
    SQ_LAUNCH_CHECK();
    group_new_off_kernel<<<nblocks(nA + 1), kThreads, 0, s>>>(newrank.p, gA_off.p, nA, gNew_off.p);
    SQ_LAUNCH_CHECK();
    gNew_host.resize(nA + 1);
    SQ_CUDA(cudaMemcpyAsync(gNew_host.data(), gNew_off.p, (nA + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
  }
  ConnView V{Ea, Eb, Erep_buf.p, eA.p, gA_off.p, eB.p, gB_off.p, EBa.p, EBrep.p, rowE_buf.p, nbr_off.p, nbr.p,
             old ? Pidx.p : nullptr, old ? Pb.p : nullptr, old ? gNew_off.p : nullptr};
  // host copies for the tile lists: alpha-group offsets and (time-reversal only) the row -> entry map
  std::vector<int64_t> gA_host(nA + 1);
  SQ_CUDA(cudaMemcpy(gA_host.data(), gA_off.p, (nA + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost));
  std::vector<int32_t> rowE_host;
  if (ts) {
    rowE_host.resize(n);
    SQ_CUDA(cudaMemcpy(rowE_host.data(), rowE_buf.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost));
  }
  auto row_entry = [&](int64_t p) -> int64_t { return ts ? (int64_t)rowE_host[p] : p; };
  std::vector<TileDesc> fill_tiles;
  DevBuf<TileDesc> fill_tiles_dev;
  HM.mark("prep (sort, groups, keys)");
  cudaEventRecord(ev[1], s);

  // ---- P1: candidate counts.  Under sharding every rank counts an equal slice of rows,
  // the counts are all-gathered and the final row blocks are balanced by candidate count.
  DevBuf<int32_t> cand_count;  // all n rows (+1 spare zero for the scan)
  SQ_CHECK(cand_count.alloc(n + 1));
  SQ_CUDA(cudaMemsetAsync(cand_count.p, 0, (n + 1) * sizeof(int32_t), s));
  {
    int64_t per = div_up(n, G.nranks);
    int64_t c0 = std::min<int64_t>(n, per * G.rank), c1 = std::min<int64_t>(n, c0 + per);
    if (c1 > c0) {
      std::vector<TileDesc> tiles;
      if (old) make_conn_tiles_split(gA_host, gNew_host, 0, nA, tiles);  // single rank: all rows
      else make_conn_tiles(gA_host, row_entry(c0), row_entry(c1 - 1) + 1, tiles);
      DevBuf<TileDesc> dt;
      SQ_CHECK(dt.alloc((int64_t)tiles.size()));
      SQ_CUDA(cudaMemcpyAsync(dt.p, tiles.data(), tiles.size() * sizeof(TileDesc), cudaMemcpyHostToDevice, s));
      const unsigned cgrid = (unsigned)std::min<int64_t>((int64_t)tiles.size(), G.sm_count * 16);
      const bool w32 = NW == 1 && T.norb <= 32;
#define SQ_CONN(FILL, ...)                                                                               \
  do {                                                                                                   \
    if (w32 && !ts) connect_tile_kernel<NW, FILL, true, true><<<cgrid, kConnTile, 0, s>>>(__VA_ARGS__);       \
    else if (w32) connect_tile_kernel<NW, FILL, true, false><<<cgrid, kConnTile, 0, s>>>(__VA_ARGS__);        \
    else if (!ts) connect_tile_kernel<NW, FILL, false, true><<<cgrid, kConnTile, 0, s>>>(__VA_ARGS__);        \
    else connect_tile_kernel<NW, FILL, false, false><<<cgrid, kConnTile, 0, s>>>(__VA_ARGS__);                \
  } while (0)
      if (use_bmp && stage_ids) connect_bitmap_kernel<NW, false, true><<<cgrid, kConnTile, bmp_smem, s>>>(V, BV, dt.p, (int64_t)tiles.size(), c0, cand_count.p + c0, nullptr, nullptr, nullptr, d_oon, nullptr);
      else if (use_bmp) connect_bitmap_kernel<NW, false, false><<<cgrid, kConnTile, bmp_smem, s>>>(V, BV, dt.p, (int64_t)tiles.size(), c0, cand_count.p + c0, nullptr, nullptr, nullptr, d_oon, nullptr);
      else SQ_CONN(false, V, dt.p, (int64_t)tiles.size(), c0, cand_count.p + c0, nullptr, nullptr, nullptr, d_oon, nullptr);
      SQ_LAUNCH_CHECK();
      SQ_CUDA(cudaStreamSynchronize(s));
    }
    if (G.nranks > 1) {
      // equal-sized padded slices so that a plain allgather works
      DevBuf<int32_t> padded;
      SQ_CHECK(padded.alloc(per * G.nranks));
      SQ_CUDA(cudaMemsetAsync(padded.p, 0, per * G.nranks * sizeof(int32_t), s));
      SQ_CUDA(cudaMemcpyAsync(padded.p + per * G.rank, cand_count.p + c0, (c1 - c0) * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
      ncclResult_t r = ncclAllGather(padded.p + per * G.rank, padded.p, per, ncclInt32, G.comm, s);
      if (r != ncclSuccess) { set_error("ncclAllGather(counts) failed: %s", ncclGetErrorString(r)); return 3; }
      SQ_CUDA(cudaMemcpyAsync(cand_count.p, padded.p, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
      SQ_CUDA(cudaStreamSynchronize(s));
    }
  }
  HM.mark("count pass");
  // per-row length of the chunk temporaries: the candidates, and in an incremental build the row's old entries in front
  DevBuf<int32_t> seg_buf;
  int32_t *seg_count = cand_count.p;
  if (old) {
    SQ_CHECK(seg_buf.alloc(n + 1));
    add_i32_kernel<<<nblocks(n + 1), kThreads, 0, s>>>(cand_count.p, olen.p, seg_buf.p, n + 1);
    SQ_LAUNCH_CHECK();
    seg_count = seg_buf.p;
  }
  DevBuf<int64_t> cand_prefix;  // n+1 exclusive prefix of the segment lengths over ALL rows
  SQ_CHECK(cand_prefix.alloc(n + 1));
  SQ_CHECK(exclusive_scan_i32_to_i64(seg_count, cand_prefix.p, n, s));
  // The host plans with the prefix SAMPLED at a few thousand rows (row blocks of the ranks and chunk boundaries fall on sample
  // rows): every 256th row for large lists, every row for small ones, and the alpha-group boundaries in an incremental
  // build (whose tiles cover whole groups).  Downloading and walking the full n-long prefix cost tens of ms of host time.
  std::vector<int64_t> srow;
  if (old) {
    srow = gA_host;
  } else {
    const int64_t S = n > (1ll << 20) ? 256 : 1;
    srow.reserve(n / S + 2);
    for (int64_t q = 0; q < n; q += S) srow.push_back(q);
    srow.push_back(n);
  }
  const int64_t ns = (int64_t)srow.size() - 1;  // sample intervals
  std::vector<int64_t> spre(ns + 1);
  int64_t max_seg = 0;
  {
    DevBuf<int64_t> d_srow, d_spre;
    SQ_CHECK(d_srow.alloc(ns + 1));
    SQ_CHECK(d_spre.alloc(ns + 1));
    SQ_CUDA(cudaMemcpyAsync(d_srow.p, srow.data(), (ns + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    gather_i64_kernel<<<nblocks(ns + 1), kThreads, 0, s>>>(cand_prefix.p, d_srow.p, d_spre.p, ns + 1);
    SQ_LAUNCH_CHECK();
    SQ_CUDA(cudaMemcpyAsync(spre.data(), d_spre.p, (ns + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    // longest row segment (selects the sort kernel of the time-reversal path)
    DevBuf<int32_t> mx;
    SQ_CHECK(mx.alloc(1));
    size_t tb = 0;
    cub::DeviceReduce::Max(nullptr, tb, seg_count, mx.p, (int)n, s);
    DevBuf<char> tmp;
    SQ_CHECK(tmp.alloc((int64_t)tb + 16));
    SQ_CUDA(cub::DeviceReduce::Max(tmp.p, tb, seg_count, mx.p, (int)n, s));
    g_launch_count += 1;
    int32_t m32 = 0;
    SQ_CUDA(cudaMemcpyAsync(&m32, mx.p, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
    max_seg = m32;
  }
  cand_prefix.release();
  const int64_t Ttot = spre[ns];
  std::vector<int64_t> sstart(G.nranks + 1, 0);
  partition_rows(spre.data(), ns, G.nranks, sstart.data());  // balance the candidates over the ranks, boundaries on sample rows
  h->row_starts.assign(G.nranks + 1, 0);
  for (int rk = 0; rk <= G.nranks; rk++) h->row_starts[rk] = srow[sstart[rk]];
  h->row0 = h->row_starts[G.rank];
  h->row1 = h->row_starts[G.rank + 1];
  const int64_t nloc = h->row1 - h->row0;
  const int64_t Tloc = spre[sstart[G.rank + 1]] - spre[sstart[G.rank]];
  HM.mark("prefix + partition");
  cudaEventRecord(ev[2], s);

  // ---- final arrays (capacity = candidate upper bound)
  h->capacity = std::max<int64_t>(Tloc, 1);
  // + kSlack entries: the 128-bit stream loads of the H.v kernels may touch a few entries past the last one
  SQ_CHECK(matrix_arrays_ensure(h, h->capacity));
  SQ_CUDA(cudaMemsetAsync(h->d_cols + h->capacity, 0, kSlack * sizeof(int32_t), s));
  SQ_CUDA(cudaMemsetAsync(h->d_vals + h->capacity, 0, kSlack * sizeof(double), s));
  SQ_CHECK(devbuf_alloc((void **)&h->d_rowptr, (nloc + 1) * sizeof(int64_t)));
  // incremental build: the previous entries move to the END of the arrays.  New rows are written from the front in
  // ascending row order and old rows are consumed in the same order, so the write position never overtakes the unread
  // old entries (at most capacity - nnz_old new entries are ever added).  The move goes through a bounded staging buffer,
  // back to front, because source and destination overlap.
  const int32_t *old_cols = nullptr;
  const double *old_vals = nullptr;
  HM.mark("map entry arrays");
  if (old) {
    const int64_t shift = h->capacity - old->nnz;
    old_cols = h->d_cols + shift;
    old_vals = h->d_vals + shift;
    if (shift > 0 && old->nnz > 0) {
      const int64_t step = std::min<int64_t>(old->nnz, 1ll << 26);
      DevBuf<double> stage;
      SQ_CHECK(stage.alloc(step));
      for (int64_t e1 = old->nnz; e1 > 0; e1 -= step) {
        const int64_t e0 = std::max<int64_t>(0, e1 - step), len = e1 - e0;
        if (shift >= len) {  // disjoint: direct copy
          SQ_CUDA(cudaMemcpyAsync(h->d_cols + e0 + shift, h->d_cols + e0, len * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
          SQ_CUDA(cudaMemcpyAsync(h->d_vals + e0 + shift, h->d_vals + e0, len * sizeof(double), cudaMemcpyDeviceToDevice, s));
        } else {
          SQ_CUDA(cudaMemcpyAsync(stage.p, h->d_cols + e0, len * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
          SQ_CUDA(cudaMemcpyAsync(h->d_cols + e0 + shift, stage.p, len * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
          SQ_CUDA(cudaMemcpyAsync(stage.p, h->d_vals + e0, len * sizeof(double), cudaMemcpyDeviceToDevice, s));
          SQ_CUDA(cudaMemcpyAsync(h->d_vals + e0 + shift, stage.p, len * sizeof(double), cudaMemcpyDeviceToDevice, s));
        }
      }
    }
  }

  HM.mark("move old entries to the end");
  // diagonal of the local rows: read by eval_kernel, kept for Davidson's preconditioner and the projector
  SQ_CHECK(devbuf_alloc((void **)&h->d_diag, std::max<int64_t>(nloc, 1) * sizeof(double)));
  if (nloc > 0) {
    SQ_MODEL_DISPATCH(T, (diag_rows_kernel<NW, kModel, kTS><<<nblocks(nloc), kThreads, 0, s>>>(T, h->d_up, h->d_dn, h->d_perm, h->row0, nloc, h->d_diag)));
    SQ_LAUNCH_CHECK();
  }
  HM.mark("alloc cols/vals/rowptr");
  // ---- chunks of rows bounded by temp candidates
  // candidates per chunk of rows: 2^28 (3.2 GB of temporaries) gives the per-chunk kernels ~2000 tiles / ~300k rows -- with 2^27 the
  // candidate-generation launches were a single partial wave of CTAs (ncu: 975 CTAs for 1184 slots); SQMC_BUILD_CHUNK_LOG2 overrides
  int chunk_log2 = 28;
  if (const char *ce = getenv("SQMC_BUILD_CHUNK_LOG2")) chunk_log2 = std::max(20, std::min(30, atoi(ce)));
  const int64_t kChunkCand = 1ll << chunk_log2;
  int64_t maxlen = 0;
  double ms_fill = 0, ms_eval = 0;
  int64_t base_nnz = 0;
  DevBuf<int32_t> cand_tmp, row_nnz, alen;
  DevBuf<double> vals_tmp;
  DevBuf<int64_t> cptr, rptr;
  int64_t r = h->row0;
  int64_t tmp_cap = 0, rows_cap = 0;
  (void)Ttot;
  // the chunk loop is asynchronous: the running entry count lives on the device, the scans use one preallocated
  // workspace, and the per-chunk timing events are read after the loop; the host prepares the next chunk's tiles meanwhile
  DevBuf<int64_t> base_dev;
  SQ_CHECK(base_dev.alloc(1));
  SQ_CUDA(cudaMemsetAsync(base_dev.p, 0, sizeof(int64_t), s));
  const size_t scan_bytes = exclusive_scan_tmp_bytes(std::max<int64_t>(nloc, 1)) + 256;
  DevBuf<char> scan_tmp;
  SQ_CHECK(scan_tmp.alloc((int64_t)scan_bytes));
  // plan: chunk boundaries, the connection tiles of every chunk (uploaded once) and the temporary sizes
  struct ChunkPlan { int64_t r, r_end, tile_off, ntiles, ml; };
  std::vector<ChunkPlan> plan;
  std::vector<TileDesc> all_tiles;
  maxlen = max_seg;
  for (int64_t i = sstart[G.rank], i_end = sstart[G.rank + 1]; i < i_end;) {
    // largest sample j with prefix[j] - prefix[i] <= kChunkCand
    int64_t j = std::upper_bound(spre.begin() + i + 1, spre.begin() + i_end + 1, spre[i] + kChunkCand) - spre.begin() - 1;
    if (j <= i) j = i + 1;
    r = srow[i];
    const int64_t r_end = srow[j];
    tmp_cap = std::max(tmp_cap, spre[j] - spre[i]);
    rows_cap = std::max(rows_cap, r_end - r);
    if (old) make_conn_tiles_split(gA_host, gNew_host, i, j, fill_tiles);  // samples = alpha-group boundaries
    else make_conn_tiles(gA_host, row_entry(r), row_entry(r_end - 1) + 1, fill_tiles);
    plan.push_back({r, r_end, (int64_t)all_tiles.size(), (int64_t)fill_tiles.size(), max_seg});
    all_tiles.insert(all_tiles.end(), fill_tiles.begin(), fill_tiles.end());
    i = j;
  }
  if (!plan.empty()) {
    SQ_CHECK(cand_tmp.alloc(tmp_cap));
    SQ_CHECK(vals_tmp.alloc(tmp_cap));
    SQ_CHECK(row_nnz.alloc(rows_cap + 1));
    SQ_CHECK(alen.alloc(rows_cap + 1));
    SQ_CHECK(cptr.alloc(rows_cap + 1));
    SQ_CHECK(rptr.alloc(rows_cap + 1));
    SQ_CHECK(fill_tiles_dev.alloc(std::max<int64_t>((int64_t)all_tiles.size(), 1)));
    SQ_CUDA(cudaMemcpyAsync(fill_tiles_dev.p, all_tiles.data(), all_tiles.size() * sizeof(TileDesc), cudaMemcpyHostToDevice, s));
  }
  std::vector<cudaEvent_t> evs;
  for (const ChunkPlan &cp : plan) {
    cudaEvent_t e0, e1, e2;
    cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventCreate(&e2);
    evs.push_back(e0); evs.push_back(e1); evs.push_back(e2);
    r = cp.r;
    const int64_t r_end = cp.r_end, nr = r_end - r;
    cudaEventRecord(e0, s);
    // chunk-local candidate offsets
    SQ_CHECK(exclusive_scan_i32_to_i64_async(seg_count + r, cptr.p, nr, scan_tmp.p, scan_bytes, s));
    // the scan above read seg_count[r+nr] as its spare slot; offsets beyond nr are unused
    if (old) {
      copy_old_rows_kernel<<<nblocks(nr * 32), 256, 0, s>>>(old_of_new.p, old->d_rowptr, old_cols, old_vals, new_of_old.p, r, nr, cptr.p, cand_tmp.p, vals_tmp.p);
      SQ_LAUNCH_CHECK();
    }
    {
      const TileDesc *td = fill_tiles_dev.p + cp.tile_off;
      const unsigned cgrid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(cp.ntiles, G.sm_count * 16));
      const bool w32 = NW == 1 && T.norb <= 32;
      if (use_bmp && stage_ids) connect_bitmap_kernel<NW, true, true><<<cgrid, kConnTile, bmp_smem, s>>>(V, BV, td, cp.ntiles, r, nullptr, cptr.p, cand_tmp.p, alen.p, d_oon, d_olen);
      else if (use_bmp) connect_bitmap_kernel<NW, true, false><<<cgrid, kConnTile, bmp_smem, s>>>(V, BV, td, cp.ntiles, r, nullptr, cptr.p, cand_tmp.p, alen.p, d_oon, d_olen);
      else SQ_CONN(true, V, td, cp.ntiles, r, nullptr, cptr.p, cand_tmp.p, ts ? nullptr : alen.p, d_oon, d_olen);
      SQ_LAUNCH_CHECK();
    }
    if (ts) {  // time-reversed partners in the entry list: arbitrary candidate order, duplicates -> sort the rows
      sort_rows_warp_kernel<<<nblocks(nr, 8), 256, 0, s>>>(cptr.p, cand_count.p + r, nr, cand_tmp.p);
      SQ_LAUNCH_CHECK();
      if (cp.ml > kWarpSortMax) {
        int smem = (int)std::min<int64_t>(cp.ml, kBlockSortMax) * 4;
        SQ_CUDA(cudaFuncSetAttribute(sort_rows_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBlockSortMax * 4));
        sort_rows_block_kernel<<<(int)std::min<int64_t>(nr, 148 * 16), 256, smem, s>>>(cptr.p, cand_count.p + r, nr, cand_tmp.p);
        SQ_LAUNCH_CHECK();
      }
    }
    cudaEventRecord(e1, s);
    SQ_CUDA(cudaMemsetAsync(row_nnz.p, 0, (nr + 1) * sizeof(int32_t), s));
    int c2bytes = (T.model == MODEL_CHEM) ? (T.norb + 1) * (T.norb + 1) * 4 : 0;
    SQ_MODEL_DISPATCH(T, (eval_kernel<NW, kModel, kTS><<<nblocks(nr * 32), 256, c2bytes, s>>>(T, h->d_up, h->d_dn, h->d_perm, h->d_diag, h->row0, r, r_end, cptr.p,
                                                                                              cand_count.p + r, cand_tmp.p, vals_tmp.p, row_nnz.p, ts ? nullptr : alen.p, d_olen)));
    SQ_LAUNCH_CHECK();
    SQ_CHECK(exclusive_scan_i32_to_i64_async(row_nnz.p, rptr.p, nr, scan_tmp.p, scan_bytes, s));
    add_offset_dev_kernel<<<nblocks(nr + 1), kThreads, 0, s>>>(rptr.p, nr + 1, base_dev.p);
    SQ_LAUNCH_CHECK();
    compact_copy_kernel<<<nblocks(nr * 32), 256, 0, s>>>(cptr.p, row_nnz.p, ts ? nullptr : alen.p, d_olen, r, rptr.p, nr, cand_tmp.p, vals_tmp.p, h->d_cols, h->d_vals);
    SQ_LAUNCH_CHECK();
    SQ_CUDA(cudaMemcpyAsync(h->d_rowptr + (r - h->row0), rptr.p, (nr + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
    set_scalar_kernel<<<1, 1, 0, s>>>(base_dev.p, rptr.p + nr);
    SQ_LAUNCH_CHECK();
    cudaEventRecord(e2, s);
  }
  SQ_CUDA(cudaMemcpyAsync(&base_nnz, base_dev.p, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  for (size_t q = 0; q + 2 < evs.size(); q += 3) {
    float f1 = 0, f2 = 0;
    cudaEventElapsedTime(&f1, evs[q], evs[q + 1]);
    cudaEventElapsedTime(&f2, evs[q + 1], evs[q + 2]);
    ms_fill += f1;
    ms_eval += f2;
  }
  for (cudaEvent_t e : evs) cudaEventDestroy(e);
  HM.mark("fill/sort/eval/compact chunks");
  if (nloc == 0) SQ_CUDA(cudaMemsetAsync(h->d_rowptr, 0, sizeof(int64_t), s));
  h->nnz_local = base_nnz;
  cudaEventRecord(ev[3], s);

  // ---- global counts
  int64_t tot = h->nnz_local;
  if (G.nranks > 1) {
    DevBuf<int64_t> t;
    SQ_CHECK(t.alloc(1));
    SQ_CUDA(cudaMemcpyAsync(t.p, &tot, 8, cudaMemcpyHostToDevice, s));
    ncclResult_t rr = ncclAllReduce(t.p, t.p, 1, ncclInt64, ncclSum, G.comm, s);
    if (rr != ncclSuccess) { set_error("ncclAllReduce(nnz) failed: %s", ncclGetErrorString(rr)); return 3; }
    SQ_CUDA(cudaMemcpyAsync(&tot, t.p, 8, cudaMemcpyDeviceToHost, s));
    SQ_CUDA(cudaStreamSynchronize(s));
  }
  h->nnz_full = tot;
  h->nnz_upper = (tot + n) / 2;
  h->scale = 1.0;

  // the surplus above the stored entries (candidate bound vs kept entries) stays mapped: unmapping costs ~10 ms per 256 MB and
  // the next build needs the room again; it is given back only when some other allocation runs out of memory (release_surplus)
  h->capacity = std::max<int64_t>(h->nnz_local, 1);
  HM.mark("nnz reduce + shrink");
  SQ_CHECK(alloc_work_vectors(h));
  HM.mark("work vectors");
  SQ_CHECK(bundle_encode(h));
  HM.mark("bundle encode");
  cudaEventRecord(ev[4], s);
  SQ_CUDA(cudaStreamSynchronize(s));
  float f;
  cudaEventElapsedTime(&f, ev[0], ev[1]); h->build_ms[0] = f;
  cudaEventElapsedTime(&f, ev[1], ev[2]); h->build_ms[1] = f;
  h->build_ms[2] = ms_fill;
  h->build_ms[3] = ms_eval;
  cudaEventElapsedTime(&f, ev[0], ev[4]); h->build_ms[4] = f;
  h->build_ms[5] = (double)Tloc;
  h->build_ms[6] = (double)nA;
  h->build_ms[7] = (double)nB;
  (void)maxlen;
  return 0;
}

int build_h(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, int64_t ndet_old) {
  if (n <= 0) { set_error("build_h: n must be positive"); return 2; }
  if (n >= (1ll << 31) - 2) { set_error("build_h: n=%lld exceeds 32-bit row indices", (long long)n); return 2; }
  if (ndet_old < 0 || ndet_old > n) { set_error("build_h: ndet_old out of range"); return 2; }
  // Incremental build (sparse_ham%ndet, chemistry.f90:7769-7843): the caller promises that rows 1..ndet_old are the list of
  // the previous call on this handle.  Then the previous matrix is kept and only pairs with a new determinant are generated
  // and evaluated -- the result is identical to a from-scratch build (an entry depends only on its two determinants).
  // Taken when the previous matrix is resident, unscaled, built (not imported) on one rank, without time-reversal
  // expansion and by a partial-connection builder (chem / heg); otherwise the matrix is rebuilt.  A caller that wants a rebuild
  // passes ndet_old = 0.
  const ModelTables &T = h->T;
  bool inc = ndet_old > 0 && ndet_old < n && h->d_rowptr && h->d_up && h->n == ndet_old && G.nranks == 1 && h->scale == 1.0 &&
             !(T.model == MODEL_CHEM && T.time_sym) && T.model != MODEL_HUBBARDK && h->row0 == 0 && h->row1 == h->n;
  OldMatrix old;
  if (inc) {
    if (bundle_decode(h)) inc = false;  // the merge reads plain rows
  }
  if (inc) {
    old.n = h->n;
    old.nnz = h->nnz_local;
    old.d_perm = h->d_perm; h->d_perm = nullptr;
    old.d_iperm = h->d_iperm; h->d_iperm = nullptr;
    old.d_rowptr = h->d_rowptr; h->d_rowptr = nullptr;
  }
  {
    HostMarks FM;
    free_matrix(h);
    FM.mark("free previous matrix");
  }
  if (inc) h->capacity = old.nnz;  // the entries of the previous matrix stay in the arrays until the merge has consumed them
  h->last_build_incremental = inc ? 1 : 0;
  int rc = h->NW == 1 ? build_impl<1>(h, n, dets_up, dets_dn, inc ? &old : nullptr) : build_impl<2>(h, n, dets_up, dets_dn, inc ? &old : nullptr);
  if (rc) {  // leave no half-built matrix behind
    cudaStreamSynchronize(G.stream);
    free_matrix(h);
  }
  return rc;
}

int diagonal(sqmc_b200_handle *h, int64_t n, const void *dets_up, const void *dets_dn, double *diag) {
  cudaStream_t s = G.stream;
  if (n <= 0) return 0;
  DevBuf<uint64_t> raw, up, dn;
  DevBuf<int> bad;
  DevBuf<double> out;
  int NW = h->NW;
  SQ_CHECK(raw.alloc(2 * n));
  SQ_CHECK(up.alloc(n * NW));
  SQ_CHECK(dn.alloc(n * NW));
  SQ_CHECK(bad.alloc(1));
  SQ_CHECK(out.alloc(n));
  SQ_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), s));
  for (int which = 0; which < 2; which++) {
    SQ_CUDA(cudaMemcpyAsync(raw.p, which == 0 ? dets_up : dets_dn, (size_t)n * 16, cudaMemcpyHostToDevice, s));
    if (NW == 1) split_dets_kernel<1><<<nblocks(n), kThreads, 0, s>>>(raw.p, which == 0 ? up.p : dn.p, n, bad.p, 0, 0);
    else split_dets_kernel<2><<<nblocks(n), kThreads, 0, s>>>(raw.p, which == 0 ? up.p : dn.p, n, bad.p, 0, 0);
    SQ_LAUNCH_CHECK();
  }
  if (NW == 1) SQ_MODEL_DISPATCH(h->T, (diag_kernel<1, kModel, kTS><<<nblocks(n), kThreads, 0, s>>>(h->T, up.p, dn.p, n, out.p)));
  else SQ_MODEL_DISPATCH(h->T, (diag_kernel<2, kModel, kTS><<<nblocks(n), kThreads, 0, s>>>(h->T, up.p, dn.p, n, out.p)));
  SQ_LAUNCH_CHECK();
  SQ_CUDA(cudaMemcpyAsync(diag, out.p, n * sizeof(double), cudaMemcpyDeviceToHost, s));
  SQ_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// ------------------------------------------------------------------ export / import (compatibility paths, host side)
int export_upper(sqmc_b200_handle *h, int64_t *counts, int64_t *indices, double *values) {
  if (!h->d_rowptr) { set_error("export_upper: no matrix"); return 2; }
  const int was_bundled = h->bundle_R;
  SQ_CHECK(bundle_decode(h));  // the exporter walks plain rows; re-ordered again afterwards
  int rc = export_upper_device(h, counts, indices, values);
  if (rc) return rc;
  if (was_bundled) {
    SQ_CHECK(bundle_encode_r(h, was_bundled));
    SQ_CUDA(cudaStreamSynchronize(G.stream));
  }
  return 0;
}

int import_upper(sqmc_b200_handle *h, int64_t n, const int64_t *counts, const int64_t *indices, const double *values) {
  if (G.nranks != 1) { set_error("import_upper: single-rank handles only"); return 2; }
  if (n <= 0 || n >= (1ll << 31) - 2) { set_error("import_upper: bad n"); return 2; }
  free_matrix(h);
  cudaStream_t s = G.stream;
  h->n = n;
  h->row_starts = {0, n};
  h->row0 = 0;
  h->row1 = n;
  SQ_CHECK(devbuf_alloc((void **)&h->d_perm, n * 4));
  SQ_CHECK(devbuf_alloc((void **)&h->d_iperm, n * 4));
  iota_kernel<<<nblocks(n), kThreads, 0, s>>>(h->d_perm, n);
  SQ_LAUNCH_CHECK();
  iota_kernel<<<nblocks(n), kThreads, 0, s>>>(h->d_iperm, n);
  SQ_LAUNCH_CHECK();
  SQ_CHECK(import_upper_device(h, n, counts, indices, values));
  SQ_CHECK(alloc_work_vectors(h));
  return bundle_encode(h);
}

}  // namespace sqmc
