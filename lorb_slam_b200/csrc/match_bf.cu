// match_bf.cu — brute-force Hamming matching on sm_100a.
//
// Replaces the arithmetic behind Matcher::SearchByProjection(Frame*,Frame*)
// (reference src/matcher.cpp:13-62) and Matcher::SearchLocalPoints (:319-366):
// cv::BFMatcher(NORM_HAMMING, crossCheck=true).match + minDist scan +
// `distance > max(2*minDist, 30.0)` rejection; plus the kNN-2/ratio variant and
// the keyframe-pair sweep (BASELINE config 5).
//
// Kernel plan (DESIGN.md §3):
//   hamming_tile_kernel   one CTA = 128*QPT queries (register-resident, 8 words
//                         each) x a contiguous range of trains streamed through
//                         shared memory in TMA-bulk-copied chunks; row minima in
//                         registers, column minima by REDUX + shared atomics;
//                         packed (dist<<20 | idx) keys give OpenCV's
//                         lowest-index tie-break for free.
//   crosscheck_finalize   one CTA: mutual test, minDist, filter, ordered compaction.
//   knn2_finalize         merges per-split best/second keys, ratio + threshold.
//   sweep_kernel          persistent, one CTA per SM, one keyframe pair at a
//                         time: A-side descriptors in registers, B-side double
//                         buffered in shared memory by cp.async.bulk (TMA).
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace lorb {

constexpr int TILE_THREADS = 128;
constexpr int TILE_CHUNK = 256;  // trains per shared-memory stage (8 KB)

// Scan `nt` train descriptors held in shared memory (`Bs`, 2 x uint4 each)
// against the QPT register-resident queries of this thread.
//   rowkey[k]   running min of (dist<<20 | train index)          [MODE 0, 1]
//   rowkey2[k]  running second min                               [MODE 1]
//   colkey      shared array, entry j = min over queries of
//               (dist<<20 | query index) for train j             [MODE 0]
template <int QPT, int MODE>
__device__ __forceinline__ void scan_trains(const uint4* __restrict__ Bs, int nt, uint32_t t_base,
                                            const uint32_t (&q)[QPT][8], const uint32_t (&qidx)[QPT],
                                            uint32_t (&rowkey)[QPT], uint32_t (&rowkey2)[QPT],
                                            uint32_t* colkey, int lane) {
  for (int t0 = 0; t0 < nt; t0 += 32) {
    uint32_t colacc = KEY_NONE;
    const int jn = min(32, nt - t0);
#pragma unroll 2
    for (int j = 0; j < jn; j++) {
      const int t = t0 + j;
      const uint4 lo = Bs[2 * t], hi = Bs[2 * t + 1];  // broadcast LDS.128 x2
      const uint32_t tw[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
      uint32_t ck = KEY_NONE;
#pragma unroll
      for (int k = 0; k < QPT; k++) {
        const uint32_t d = hamming256_csa(q[k], tw);
        const uint32_t rk = make_key(d, t_base + (uint32_t)t);
        if (MODE == 1) {
          rowkey2[k] = min(rowkey2[k], max(rowkey[k], rk));
        }
        rowkey[k] = min(rowkey[k], rk);
        if (MODE == 0) ck = min(ck, make_key(d, qidx[k]));
      }
      if (MODE == 0) {
        const uint32_t wmin = __reduce_min_sync(0xffffffffu, ck);
        if (lane == j) colacc = wmin;
      }
    }
    if (MODE == 0) {
      if (lane < jn) atomicMin(&colkey[t0 + lane], colacc);
    }
  }
}

// Load the QPT queries of this thread.  Slots past the end replicate the last
// valid descriptor with the largest index, so they can never win a column
// minimum (same distance, higher index) and their row results are discarded.
template <int QPT>
__device__ __forceinline__ void load_queries(const uint4* __restrict__ Q, int nq, int q_first,
                                             int stride, uint32_t (&q)[QPT][8],
                                             uint32_t (&qidx)[QPT]) {
#pragma unroll
  for (int k = 0; k < QPT; k++) {
    int qi = q_first + k * stride;
    const bool valid = qi < nq;
    qidx[k] = valid ? (uint32_t)qi : KEY_IDX_MASK;
    qi = valid ? qi : nq - 1;
    const uint4 lo = Q[2 * qi], hi = Q[2 * qi + 1];
    q[k][0] = lo.x; q[k][1] = lo.y; q[k][2] = lo.z; q[k][3] = lo.w;
    q[k][4] = hi.x; q[k][5] = hi.y; q[k][6] = hi.z; q[k][7] = hi.w;
  }
}

// grid = (query tiles, train splits).  MODE 0: cross-check keys into
// fwd_key[nq] / bwd_key[nt] (global atomicMin).  MODE 1: per split best/second
// row keys into part[split][nq][2].
template <int QPT, int MODE>
__global__ void __launch_bounds__(TILE_THREADS)
    hamming_tile_kernel(const uint4* __restrict__ Q, int nq, const uint4* __restrict__ T, int nt,
                        int trains_per_split, uint32_t* __restrict__ fwd_key,
                        uint32_t* __restrict__ bwd_key, uint32_t* __restrict__ part) {
  __shared__ __align__(128) uint4 Bs[2][TILE_CHUNK * 2];
  __shared__ uint32_t colkey[TILE_CHUNK];
  __shared__ __align__(8) uint64_t bar[2];
  const int tid = threadIdx.x, lane = tid & 31;
  const int q_first = blockIdx.x * (TILE_THREADS * QPT) + tid;
  const int t_begin = blockIdx.y * trains_per_split;
  const int t_end = min(nt, t_begin + trains_per_split);
  const int n_chunks = (t_end - t_begin + TILE_CHUNK - 1) / TILE_CHUNK;

  if (tid == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  auto issue = [&](int c) {
    const int c0 = t_begin + c * TILE_CHUNK;
    const uint32_t bytes = (uint32_t)(min(TILE_CHUNK, t_end - c0) * 32);
    mbar_arrive_expect_tx(&bar[c & 1], bytes);
    tma_load_1d(&Bs[c & 1][0], T + 2 * (size_t)c0, bytes, &bar[c & 1]);
  };
  if (tid == 0 && n_chunks > 0) issue(0);

  uint32_t q[QPT][8], qidx[QPT], rowkey[QPT], rowkey2[QPT];
  load_queries<QPT>(Q, nq, q_first, TILE_THREADS, q, qidx);
#pragma unroll
  for (int k = 0; k < QPT; k++) rowkey[k] = rowkey2[k] = KEY_NONE;

  for (int c = 0; c < n_chunks; c++) {
    const int c0 = t_begin + c * TILE_CHUNK;
    const int len = min(TILE_CHUNK, t_end - c0);
    if (tid == 0 && c + 1 < n_chunks) issue(c + 1);  // buffer (c+1)&1 was released by the sync below
    if (MODE == 0) {
      for (int j = tid; j < len; j += TILE_THREADS) colkey[j] = KEY_NONE;
      __syncthreads();
    }
    mbar_wait(&bar[c & 1], (uint32_t)((c >> 1) & 1));
    scan_trains<QPT, MODE>(&Bs[c & 1][0], len, (uint32_t)c0, q, qidx, rowkey, rowkey2, colkey, lane);
    __syncthreads();
    if (MODE == 0) {
      for (int j = tid; j < len; j += TILE_THREADS)
        if (colkey[j] != KEY_NONE) atomicMin(&bwd_key[c0 + j], colkey[j]);
    }
  }
#pragma unroll
  for (int k = 0; k < QPT; k++) {
    const int qi = q_first + k * TILE_THREADS;
    if (qi < nq) {
      if (MODE == 0) {
        if (rowkey[k] != KEY_NONE) atomicMin(&fwd_key[qi], rowkey[k]);
      } else {
        part[((size_t)blockIdx.y * nq + qi) * 2 + 0] = rowkey[k];
        part[((size_t)blockIdx.y * nq + qi) * 2 + 1] = rowkey2[k];
      }
    }
  }
}

// Result block of a cross-check call (device and pinned-host mirror):
//   int hdr[4] = {n_matches, n_kept, min_dist, 0}; int q[cap]; int t[cap];
//   int d[cap]; uint8 keep[cap]
__device__ __forceinline__ bool cc_match(const uint32_t* fwd_key, const uint32_t* bwd_key,
                                         const uint32_t* leg_key, int mode, int qi, int& t, int& d) {
  if (mode == LORB_CROSSCHECK_MUTUAL) {
    const uint32_t fk = fwd_key[qi];
    if (fk == KEY_NONE) return false;
    t = (int)(fk & KEY_IDX_MASK);
    d = (int)(fk >> KEY_IDX_BITS);
    return (bwd_key[t] & KEY_IDX_MASK) == (uint32_t)qi;
  }
  const uint32_t lk = leg_key[qi];
  if (lk == KEY_NONE) return false;
  t = (int)(lk & KEY_IDX_MASK);
  d = (int)(lk >> KEY_IDX_BITS);
  return true;
}

__global__ void __launch_bounds__(1024)
    crosscheck_finalize_kernel(const uint32_t* __restrict__ fwd_key,
                               const uint32_t* __restrict__ bwd_key, uint32_t* __restrict__ leg_key,
                               int nq, int nt, int mode, int cap, int* __restrict__ res) {
  __shared__ int s_red[32];
  __shared__ int s_min, s_base, s_kept;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int* out_q = res + 4;
  int* out_t = out_q + cap;
  int* out_d = out_t + cap;
  uint8_t* out_keep = reinterpret_cast<uint8_t*>(out_d + cap);

  if (mode == LORB_CROSSCHECK_LEGACY) {
    // OpenCV 3.1 batchDistance cross-check (recalled): train t votes for its
    // nearest query; the query keeps the vote of smallest (dist, t).
    for (int t = tid; t < nt; t += blockDim.x) {
      const uint32_t bk = bwd_key[t];
      if (bk != KEY_NONE)
        atomicMin(&leg_key[bk & KEY_IDX_MASK], (bk & ~KEY_IDX_MASK) | (uint32_t)t);
    }
    __syncthreads();
  }
  // pass 1: minDist over the matches (reference src/matcher.cpp:42-47)
  int lmin = 1 << 30;
  for (int qi = tid; qi < nq; qi += blockDim.x) {
    int t, d;
    if (cc_match(fwd_key, bwd_key, leg_key, mode, qi, t, d)) lmin = min(lmin, d);
  }
  lmin = __reduce_min_sync(0xffffffffu, lmin);
  if (lane == 0) s_red[warp] = lmin;
  if (tid == 0) {
    s_base = 0;
    s_kept = 0;
  }
  __syncthreads();
  if (warp == 0) {
    int v = s_red[lane];
    v = __reduce_min_sync(0xffffffffu, v);
    if (lane == 0) s_min = v;
  }
  __syncthreads();
  const int min_dist = s_min;
  // `distance > max(2*minDist, 30.0)` (:52) — exact in integers
  const int thr = max(2 * min_dist, 30);
  // pass 2: ordered compaction in ascending query index
  int kept_local = 0;
  for (int base = 0; base < nq; base += blockDim.x) {
    const int qi = base + tid;
    int t = 0, d = 0;
    const bool m = qi < nq && cc_match(fwd_key, bwd_key, leg_key, mode, qi, t, d);
    const uint32_t bal = __ballot_sync(0xffffffffu, m);
    if (lane == 0) s_red[warp] = __popc(bal);
    __syncthreads();
    int woff = 0, total = 0;
    for (int w = 0; w < 32; w++) {
      const int cnt = s_red[w];
      if (w < warp) woff += cnt;
      total += cnt;
    }
    const int pos = s_base + woff + __popc(bal & ((1u << lane) - 1u));
    if (m) {
      const int k = !(d > thr);
      out_q[pos] = qi;
      out_t[pos] = t;
      out_d[pos] = d;
      out_keep[pos] = (uint8_t)k;
      kept_local += k;
    }
    __syncthreads();
    if (tid == 0) s_base += total;
    __syncthreads();
  }
  kept_local = __reduce_add_sync(0xffffffffu, kept_local);
  if (lane == 0 && kept_local) atomicAdd(&s_kept, kept_local);
  __syncthreads();
  if (tid == 0) {
    res[0] = s_base;
    res[1] = s_kept;
    res[2] = s_base > 0 ? min_dist : -1;
    res[3] = 0;
  }
}

// Merge per-split (best, second) keys; Lowe ratio + absolute threshold.
__global__ void knn2_finalize_kernel(const uint32_t* __restrict__ part, int nq, int n_splits,
                                     float ratio, int max_dist, int* __restrict__ out_idx,
                                     int* __restrict__ out_dist, uint8_t* __restrict__ out_pass) {
  const int qi = blockIdx.x * blockDim.x + threadIdx.x;
  if (qi >= nq) return;
  uint32_t k0 = KEY_NONE, k1 = KEY_NONE;
  for (int s = 0; s < n_splits; s++) {
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const uint32_t k = part[((size_t)s * nq + qi) * 2 + j];
      k1 = min(k1, max(k0, k));
      k0 = min(k0, k);
    }
  }
  const int i0 = k0 == KEY_NONE ? -1 : (int)(k0 & KEY_IDX_MASK);
  const int d0 = k0 == KEY_NONE ? 256 : (int)(k0 >> KEY_IDX_BITS);
  const int i1 = k1 == KEY_NONE ? -1 : (int)(k1 & KEY_IDX_MASK);
  const int d1 = k1 == KEY_NONE ? 256 : (int)(k1 >> KEY_IDX_BITS);
  out_idx[2 * qi] = i0;
  out_idx[2 * qi + 1] = i1;
  out_dist[2 * qi] = d0;
  out_dist[2 * qi + 1] = d1;
  bool pass = i0 >= 0 && d0 <= max_dist;
  if (pass && i1 >= 0) pass = (float)d0 < ratio * (float)d1;
  out_pass[qi] = pass ? 1 : 0;
}

// ---- MapPoint::ComputeDescriptor (reference src/map_point.cpp:69-129), one CTA per map point
constexpr int CD_MAX = 128;
__global__ void __launch_bounds__(128)
    compute_descriptor_kernel(int n_points, const int* __restrict__ offsets,
                              const uint4* __restrict__ desc, int* __restrict__ out_best,
                              int* __restrict__ out_median) {
  extern __shared__ __align__(16) unsigned char cd_raw[];
  __shared__ uint32_t s_key[4];
  const int k = blockIdx.x;
  if (k >= n_points) return;
  const int s0 = offsets[k], m = offsets[k + 1] - s0, tid = threadIdx.x;
  if (m <= 0) {
    if (tid == 0) {
      out_best[k] = -1;
      if (out_median) out_median[k] = -1;
    }
    return;
  }
  uint4* D = reinterpret_cast<uint4*>(cd_raw);                       // m x 2 uint4
  uint16_t* dist = reinterpret_cast<uint16_t*>(cd_raw + CD_MAX * 32);  // m x m
  for (int e = tid; e < 2 * m; e += 128) D[e] = desc[2 * (size_t)s0 + e];
  __syncthreads();
  for (int e = tid; e < m * m; e += 128) {
    const int i = e / m, j = e % m;
    const uint4 a0 = D[2 * i], a1 = D[2 * i + 1], b0 = D[2 * j], b1 = D[2 * j + 1];
    const uint32_t q[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const uint32_t t[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
    dist[e] = (uint16_t)hamming256_popc8(q, t);
  }
  __syncthreads();
  // row i: element (int)(0.5*(m-1)) of the sorted row, by counting selection
  const int kth = (int)(0.5 * (double)(m - 1));
  uint32_t key = KEY_NONE;
  if (tid < m) {
    const uint16_t* row = dist + (size_t)tid * m;
    int median = 0;
    for (int j = 0; j < m; j++) {
      const int v = row[j];
      int less = 0, eq = 0;
      for (int j2 = 0; j2 < m; j2++) {
        less += row[j2] < v;
        eq += row[j2] == v;
      }
      if (less <= kth && kth < less + eq) {
        median = v;
        break;
      }
    }
    key = ((uint32_t)median << KEY_IDX_BITS) | (uint32_t)tid;  // min = smallest median, first row
  }
  key = __reduce_min_sync(0xffffffffu, key);
  if ((tid & 31) == 0) s_key[tid >> 5] = key;
  __syncthreads();
  if (tid == 0) {
    const uint32_t best = min(min(s_key[0], s_key[1]), min(s_key[2], s_key[3]));
    out_best[k] = (int)(best & KEY_IDX_MASK);
    if (out_median) out_median[k] = (int)(best >> KEY_IDX_BITS);
  }
}

// ------------------------------------------------------------------ sweep
constexpr int SWEEP_THREADS = 512;

template <int QPT>
__global__ void __launch_bounds__(SWEEP_THREADS, 1)
    sweep_kernel(const uint4* __restrict__ bank, const uint4* __restrict__ bank_b, int n_desc,
                 const int2* __restrict__ pairs, int n_pairs,
                 int* __restrict__ out /* [n_pairs][3] kept, matches, min */) {
  // `bank` / `bank_b` already point at the base keyframes of the a / b side
  // (lorb_sweep_plan_run_at, lorb_sweep_plan_run_at2)
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int desc_bytes = n_desc * 32;
  const int buf_bytes = (desc_bytes + 127) & ~127;
  uint4* As = reinterpret_cast<uint4*>(smem_raw);
  uint4* Bs0 = reinterpret_cast<uint4*>(smem_raw + buf_bytes);
  uint4* Bs1 = reinterpret_cast<uint4*>(smem_raw + 2 * (size_t)buf_bytes);
  uint32_t* colkey = reinterpret_cast<uint32_t*>(smem_raw + 3 * (size_t)buf_bytes);
  uint64_t* bar = reinterpret_cast<uint64_t*>(colkey + ((n_desc + 31) & ~31));
  int* s_red = reinterpret_cast<int*>(bar + 4);  // [16] mins, [16] sums, [2] results

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // contiguous slice of the (a-sorted) pair list for this CTA
  const int p_begin = (int)(((long long)n_pairs * blockIdx.x) / gridDim.x);
  const int p_end = (int)(((long long)n_pairs * (blockIdx.x + 1)) / gridDim.x);
  if (p_begin >= p_end) return;

  if (tid == 0) {
    mbar_init(&bar[0], 1);  // A
    mbar_init(&bar[1], 1);  // B buffer 0
    mbar_init(&bar[2], 1);  // B buffer 1
    fence_barrier_init();
  }
  __syncthreads();
  const size_t kf_u4 = (size_t)n_desc * 2;  // uint4 per keyframe
  if (tid == 0) {
    const int2 p0 = pairs[p_begin];
    mbar_arrive_expect_tx(&bar[0], (uint32_t)desc_bytes);
    tma_load_1d(As, bank + kf_u4 * p0.x, (uint32_t)desc_bytes, &bar[0]);
    mbar_arrive_expect_tx(&bar[1], (uint32_t)desc_bytes);
    tma_load_1d(Bs0, bank_b + kf_u4 * p0.y, (uint32_t)desc_bytes, &bar[1]);
  }
  uint32_t q[QPT][8], qidx[QPT], rowkey[QPT], rowkey2[QPT];
  int cur_a = -1;
  uint32_t a_phase = 0;
  for (int p = p_begin; p < p_end; p++) {
    const int i = p - p_begin;
    const int2 pr = pairs[p];
    uint4* Bs = (i & 1) ? Bs1 : Bs0;
    // prefetch the next pair's B side into the other buffer (released by the
    // trailing __syncthreads of the previous iteration)
    if (tid == 0 && p + 1 < p_end) {
      const int2 pn = pairs[p + 1];
      uint64_t* nb = &bar[1 + ((i + 1) & 1)];
      mbar_arrive_expect_tx(nb, (uint32_t)desc_bytes);
      tma_load_1d((i & 1) ? Bs0 : Bs1, bank_b + kf_u4 * pn.y, (uint32_t)desc_bytes, nb);
    }
    for (int j = tid; j < n_desc; j += SWEEP_THREADS) colkey[j] = KEY_NONE;
    if (pr.x != cur_a) {
      mbar_wait(&bar[0], a_phase);
      a_phase ^= 1u;
      load_queries<QPT>(As, n_desc, tid, SWEEP_THREADS, q, qidx);
      cur_a = pr.x;
    }
    __syncthreads();  // colkey initialised; everyone holds its A rows in registers
    if (tid == 0 && p + 1 < p_end) {
      const int2 pn = pairs[p + 1];
      if (pn.x != cur_a) {  // A buffer is free again: fetch the next A side early
        mbar_arrive_expect_tx(&bar[0], (uint32_t)desc_bytes);
        tma_load_1d(As, bank + kf_u4 * pn.x, (uint32_t)desc_bytes, &bar[0]);
      }
    }
#pragma unroll
    for (int k = 0; k < QPT; k++) rowkey[k] = rowkey2[k] = KEY_NONE;
    mbar_wait(&bar[1 + (i & 1)], (uint32_t)((i >> 1) & 1));
    scan_trains<QPT, 0>(Bs, n_desc, 0u, q, qidx, rowkey, rowkey2, colkey, lane);
    __syncthreads();  // all column keys final
    // mutual test + minDist + max(2*minDist,30) filter (reference :42-56)
    int cnt = 0, lmin = 1 << 30;
    int dd[QPT];
#pragma unroll
    for (int k = 0; k < QPT; k++) {
      dd[k] = -1;
      if (qidx[k] != KEY_IDX_MASK) {
        const uint32_t t = rowkey[k] & KEY_IDX_MASK;
        if ((colkey[t] & KEY_IDX_MASK) == qidx[k]) {
          dd[k] = (int)(rowkey[k] >> KEY_IDX_BITS);
          cnt++;
          lmin = min(lmin, dd[k]);
        }
      }
    }
    lmin = __reduce_min_sync(0xffffffffu, lmin);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) {
      s_red[warp] = lmin;
      s_red[16 + warp] = cnt;
    }
    __syncthreads();
    if (warp == 0) {
      int v = lane < 16 ? s_red[lane] : (1 << 30);
      int c = lane < 16 ? s_red[16 + lane] : 0;
      v = __reduce_min_sync(0xffffffffu, v);
      c = __reduce_add_sync(0xffffffffu, c);
      if (lane == 0) {
        s_red[32] = v;
        s_red[33] = c;
      }
    }
    __syncthreads();
    const int min_dist = s_red[32], n_match = s_red[33];
    const int thr = max(2 * min_dist, 30);
    int kept = 0;
#pragma unroll
    for (int k = 0; k < QPT; k++) kept += (dd[k] >= 0 && !(dd[k] > thr)) ? 1 : 0;
    kept = __reduce_add_sync(0xffffffffu, kept);
    __syncthreads();  // s_red[0..31] reads done before reuse
    if (lane == 0) s_red[warp] = kept;
    __syncthreads();
    if (tid == 0) {
      int ksum = 0;
      for (int w = 0; w < SWEEP_THREADS / 32; w++) ksum += s_red[w];
      out[3 * (size_t)p + 0] = ksum;
      out[3 * (size_t)p + 1] = n_match;
      out[3 * (size_t)p + 2] = n_match > 0 ? min_dist : -1;
    }
    __syncthreads();  // colkey / B buffer / s_red free for the next pair
  }
}

static size_t sweep_smem_bytes(int n_desc) {
  const size_t buf = ((size_t)n_desc * 32 + 127) & ~(size_t)127;
  return 3 * buf + (size_t)((n_desc + 31) & ~31) * 4 + 4 * 8 + 40 * 4;
}

template <int QPT>
static int launch_sweep_qpt(lorb_ctx* c, const uint4* bank, const uint4* bank_b, int n_desc,
                            const int2* pairs, int n_pairs, int* out) {
  const size_t smem = sweep_smem_bytes(n_desc);
  const int grid = std::min(n_pairs, c->sm_count);
  LORB_CUDA_TRY(cudaFuncSetAttribute(sweep_kernel<QPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  LORB_LAUNCH(c, sweep_kernel<QPT>, grid, SWEEP_THREADS, smem, bank, bank_b, n_desc, pairs, n_pairs, out);
  return LORB_OK;
}

static int launch_sweep(lorb_ctx* c, const uint4* bank, const uint4* bank_b, int n_desc,
                        const int2* pairs, int n_pairs, int* out) {
  if (n_pairs == 0) return LORB_OK;
  const int qpt = (n_desc + SWEEP_THREADS - 1) / SWEEP_THREADS;
  switch (qpt) {
    case 1: return launch_sweep_qpt<1>(c, bank, bank_b, n_desc, pairs, n_pairs, out);
    case 2: return launch_sweep_qpt<2>(c, bank, bank_b, n_desc, pairs, n_pairs, out);
    case 3: return launch_sweep_qpt<3>(c, bank, bank_b, n_desc, pairs, n_pairs, out);
    case 4: return launch_sweep_qpt<4>(c, bank, bank_b, n_desc, pairs, n_pairs, out);
  }
  set_error("sweep: n_desc=%d exceeds the shared-memory resident limit (2048)", n_desc);
  return LORB_ERR_ARG;
}

// Launch the tile kernel over (query tiles x train splits).
template <int MODE>
static int launch_tiles(lorb_ctx* c, const uint4* dq, int nq, const uint4* dt, int nt,
                        uint32_t* fwd, uint32_t* bwd, uint32_t* part, int* n_splits_out) {
  // wide tiles once there is enough work to fill the GPU with them
  const bool wide = (long long)nq * nt >= (long long)c->sm_count * 512 * 512;
  const int qpt = wide ? 4 : 1;
  const int q_tiles = (nq + TILE_THREADS * qpt - 1) / (TILE_THREADS * qpt);
  int splits = (2 * c->sm_count + q_tiles - 1) / q_tiles;
  splits = std::max(1, std::min(splits, (nt + 31) / 32));
  if (MODE == 1) splits = std::min(splits, 64);
  int per = (nt + splits - 1) / splits;
  per = (per + 31) & ~31;
  splits = (nt + per - 1) / per;
  if (n_splits_out) *n_splits_out = splits;
  dim3 grid(q_tiles, splits);
  if (wide)
    LORB_LAUNCH(c, (hamming_tile_kernel<4, MODE>), grid, TILE_THREADS, 0, dq, nq, dt, nt, per, fwd, bwd, part);
  else
    LORB_LAUNCH(c, (hamming_tile_kernel<1, MODE>), grid, TILE_THREADS, 0, dq, nq, dt, nt, per, fwd, bwd, part);
  return LORB_OK;
}

}  // namespace lorb

using namespace lorb;

extern "C" {

int lorb_match_bf_crosscheck(lorb_ctx* c, const uint8_t* q, int nq, const uint8_t* t, int nt,
                             int mode, int* out_q, int* out_t, int* out_dist, uint8_t* out_keep,
                             int* n_matches, int* n_kept, int* min_dist) {
  LORB_REQUIRE(c, "ctx");
  LORB_REQUIRE(nq >= 0 && nt >= 0, "negative size");
  LORB_REQUIRE(nq == 0 || q, "q");
  LORB_REQUIRE(nt == 0 || t, "t");
  LORB_REQUIRE(n_matches && n_kept && min_dist, "scalar outputs");
  LORB_REQUIRE(mode == LORB_CROSSCHECK_MUTUAL || mode == LORB_CROSSCHECK_LEGACY, "mode");
  LORB_REQUIRE((unsigned)nq < KEY_IDX_MASK && (unsigned)nt < KEY_IDX_MASK,
               "more than 2^20-2 descriptors per side");
  *n_matches = 0;
  *n_kept = 0;
  *min_dist = -1;
  if (nq == 0 || nt == 0) {  // cv::BFMatcher returns no matches for an empty side
    LORB_CUDA_TRY(cudaSetDevice(c->device));
    return LORB_OK;
  }
  LORB_REQUIRE(out_q && out_t && out_dist && out_keep, "output arrays");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  const int cap = std::min(nq, nt);
  const size_t qb = (size_t)nq * 32, tb = (size_t)nt * 32;
  const size_t qb_al = (qb + 255) & ~(size_t)255;
  const size_t res_bytes = 16 + (size_t)cap * 13;
  // pinned staging: [q | t] up, result block down
  LORB_TRY(pin_reserve(c, 0, qb_al + tb));
  LORB_TRY(pin_reserve(c, 1, res_bytes));
  LORB_TRY(dev_reserve(c, 0, qb_al + tb));
  LORB_TRY(dev_reserve(c, 1, (size_t)(2 * nq + nt) * 4));
  LORB_TRY(dev_reserve(c, 2, res_bytes));
  uint8_t* hs = c->h[0].as<uint8_t>();
  memcpy(hs, q, qb);
  memcpy(hs + qb_al, t, tb);
  uint8_t* dq = c->d[0].as<uint8_t>();
  LORB_CUDA_TRY(cudaMemcpyAsync(dq, hs, qb_al + tb, cudaMemcpyHostToDevice, c->stream));
  uint32_t* fwd = c->d[1].as<uint32_t>();
  uint32_t* bwd = fwd + nq;
  uint32_t* leg = bwd + nt;
  LORB_CUDA_TRY(cudaMemsetAsync(fwd, 0xFF, (size_t)(2 * nq + nt) * 4, c->stream));
  LORB_TRY(launch_tiles<0>(c, (const uint4*)dq, nq, (const uint4*)(dq + qb_al), nt, fwd, bwd,
                           nullptr, nullptr));
  LORB_LAUNCH(c, crosscheck_finalize_kernel, 1, 1024, 0, fwd, bwd, leg, nq, nt, mode, cap,
              c->d[2].as<int>());
  LORB_CUDA_TRY(cudaMemcpyAsync(c->h[1].p, c->d[2].p, res_bytes, cudaMemcpyDeviceToHost, c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  const int* res = c->h[1].as<int>();
  const int n = res[0];
  *n_matches = n;
  *n_kept = res[1];
  *min_dist = res[2];
  memcpy(out_q, res + 4, (size_t)n * 4);
  memcpy(out_t, res + 4 + cap, (size_t)n * 4);
  memcpy(out_dist, res + 4 + 2 * (size_t)cap, (size_t)n * 4);
  memcpy(out_keep, reinterpret_cast<const uint8_t*>(res + 4 + 3 * (size_t)cap), (size_t)n);
  return LORB_OK;
}

int lorb_match_knn2(lorb_ctx* c, const uint8_t* q, int nq, const uint8_t* t, int nt, float ratio,
                    int max_dist, int* out_idx, int* out_dist, uint8_t* out_pass) {
  LORB_REQUIRE(c, "ctx");
  LORB_REQUIRE(nq >= 0 && nt >= 0, "negative size");
  LORB_REQUIRE(nq == 0 || (q && out_idx && out_dist && out_pass), "q / outputs");
  LORB_REQUIRE(nt == 0 || t, "t");
  LORB_REQUIRE((unsigned)nq < KEY_IDX_MASK && (unsigned)nt < KEY_IDX_MASK,
               "more than 2^20-2 descriptors per side");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  if (nq == 0) return LORB_OK;
  if (nt == 0) {
    for (int i = 0; i < nq; i++) {
      out_idx[2 * i] = out_idx[2 * i + 1] = -1;
      out_dist[2 * i] = out_dist[2 * i + 1] = 256;
      out_pass[i] = 0;
    }
    return LORB_OK;
  }
  const size_t qb = (size_t)nq * 32, tb = (size_t)nt * 32;
  const size_t qb_al = (qb + 255) & ~(size_t)255;
  const size_t res_bytes = (size_t)nq * 17;
  LORB_TRY(pin_reserve(c, 0, qb_al + tb));
  LORB_TRY(pin_reserve(c, 1, res_bytes));
  LORB_TRY(dev_reserve(c, 0, qb_al + tb));
  LORB_TRY(dev_reserve(c, 1, (size_t)nq * 2 * 64 * 4));
  LORB_TRY(dev_reserve(c, 2, res_bytes));
  uint8_t* hs = c->h[0].as<uint8_t>();
  memcpy(hs, q, qb);
  memcpy(hs + qb_al, t, tb);
  uint8_t* dq = c->d[0].as<uint8_t>();
  LORB_CUDA_TRY(cudaMemcpyAsync(dq, hs, qb_al + tb, cudaMemcpyHostToDevice, c->stream));
  int splits = 1;
  LORB_TRY(launch_tiles<1>(c, (const uint4*)dq, nq, (const uint4*)(dq + qb_al), nt, nullptr,
                           nullptr, c->d[1].as<uint32_t>(), &splits));
  int* d_idx = c->d[2].as<int>();
  int* d_dist = d_idx + 2 * (size_t)nq;
  uint8_t* d_pass = reinterpret_cast<uint8_t*>(d_dist + 2 * (size_t)nq);
  LORB_LAUNCH(c, knn2_finalize_kernel, (nq + 255) / 256, 256, 0, c->d[1].as<uint32_t>(), nq, splits,
              ratio, max_dist, d_idx, d_dist, d_pass);
  LORB_CUDA_TRY(cudaMemcpyAsync(c->h[1].p, c->d[2].p, res_bytes, cudaMemcpyDeviceToHost, c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  const int* res = c->h[1].as<int>();
  memcpy(out_idx, res, (size_t)nq * 8);
  memcpy(out_dist, res + 2 * (size_t)nq, (size_t)nq * 8);
  memcpy(out_pass, reinterpret_cast<const uint8_t*>(res + 4 * (size_t)nq), (size_t)nq);
  return LORB_OK;
}

int lorb_compute_descriptors(lorb_ctx* c, int n_points, const int* offsets, const uint8_t* desc,
                             int* out_best, int* out_median) {
  LORB_REQUIRE(c, "ctx");
  LORB_REQUIRE(n_points >= 0, "n_points");
  if (n_points == 0) return LORB_OK;
  LORB_REQUIRE(offsets && out_best, "offsets / out_best");
  LORB_REQUIRE(offsets[0] == 0, "offsets[0] must be 0");
  int mmax = 0;
  for (int k = 0; k < n_points; k++) {
    const int m = offsets[k + 1] - offsets[k];
    LORB_REQUIRE(m >= 0, "offsets must be non-decreasing");
    LORB_REQUIRE(m <= CD_MAX, "more than 128 observations for one map point");
    mmax = std::max(mmax, m);
  }
  const int total = offsets[n_points];
  LORB_REQUIRE(total == 0 || desc, "desc");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  const size_t b_off = ((size_t)(n_points + 1) * 4 + 255) & ~(size_t)255;
  const size_t up = b_off + (size_t)total * 32, down = (size_t)n_points * 8;
  LORB_TRY(pin_reserve(c, 0, up));
  LORB_TRY(pin_reserve(c, 1, down));
  LORB_TRY(dev_reserve(c, 0, up));
  LORB_TRY(dev_reserve(c, 2, down));
  uint8_t* h = c->h[0].as<uint8_t>();
  memcpy(h, offsets, (size_t)(n_points + 1) * 4);
  if (total) memcpy(h + b_off, desc, (size_t)total * 32);
  uint8_t* d = c->d[0].as<uint8_t>();
  LORB_CUDA_TRY(cudaMemcpyAsync(d, h, up, cudaMemcpyHostToDevice, c->stream));
  const size_t smem = (size_t)CD_MAX * 32 + (size_t)mmax * mmax * 2 + 16;
  LORB_CUDA_TRY(cudaFuncSetAttribute(compute_descriptor_kernel,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int* d_best = c->d[2].as<int>();
  LORB_LAUNCH(c, compute_descriptor_kernel, n_points, 128, smem, n_points, (const int*)d,
              (const uint4*)(d + b_off), d_best, d_best + n_points);
  LORB_CUDA_TRY(cudaMemcpyAsync(c->h[1].p, c->d[2].p, down, cudaMemcpyDeviceToHost, c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  memcpy(out_best, c->h[1].p, (size_t)n_points * 4);
  if (out_median) memcpy(out_median, c->h[1].as<int>() + n_points, (size_t)n_points * 4);
  return LORB_OK;
}

// Which kernel runs the sweep: the popc kernel above or the tensor-core kernel of match_tc.cu.
// Both return identical results; LORB_SWEEP_IMPL=popc|tensor overrides the default.
static int sweep_impl(lorb_ctx* c) {
  if (c->sweep_impl >= 0) return c->sweep_impl;
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("LORB_SWEEP_IMPL");
    v = (e && !strcmp(e, "popc")) ? LORB_SWEEP_POPC : LORB_SWEEP_TENSOR;
  }
  return v;
}

int lorb_sweep_set_impl(lorb_ctx* c, int impl) {
  LORB_REQUIRE(c, "ctx");
  LORB_REQUIRE(impl == LORB_SWEEP_POPC || impl == LORB_SWEEP_TENSOR || impl == -1, "impl");
  c->sweep_impl = impl;
  c->tc_img_n_kf = 0;  // operand images are rebuilt on the next plan upload if needed
  return LORB_OK;
}

int lorb_bank_upload(lorb_ctx* c, const uint8_t* bank, int n_kf, int n_desc) {
  LORB_REQUIRE(c && bank, "ctx/bank");
  LORB_REQUIRE(n_kf > 0 && n_desc > 0 && n_desc <= 2048, "bank shape (n_desc <= 2048)");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  const size_t bytes = (size_t)n_kf * n_desc * 32;
  LORB_TRY(c->bank.reserve(bytes));
  LORB_CUDA_TRY(cudaMemcpyAsync(c->bank.p, bank, bytes, cudaMemcpyHostToDevice, c->stream));
  c->bank_n_kf = n_kf;
  c->bank_n_desc = n_desc;
  c->tc_img_n_kf = 0;
  if (sweep_impl(c) == LORB_SWEEP_TENSOR) LORB_TRY(tc::bank_expand(c));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  return LORB_OK;
}

static int check_pairs(lorb_ctx* c, const int* pa, const int* pb, int n_pairs) {
  LORB_REQUIRE(c->bank_n_kf > 0, "no bank uploaded");
  LORB_REQUIRE(n_pairs >= 0 && (n_pairs == 0 || (pa && pb)), "pair list");
  for (int i = 0; i < n_pairs; i++)
    LORB_REQUIRE(pa[i] >= 0 && pa[i] < c->bank_n_kf && pb[i] >= 0 && pb[i] < c->bank_n_kf,
                 "pair index out of range");
  return LORB_OK;
}

// The kernel keeps the A side in registers while `a` does not change, so the
// plan is executed in a-sorted order and scattered back to caller order.
int lorb_sweep_plan_upload(lorb_ctx* c, const int* pa, const int* pb, int n_pairs) {
  LORB_REQUIRE(c, "ctx");
  LORB_TRY(check_pairs(c, pa, pb, n_pairs));
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  c->plan_n_pairs = n_pairs;
  c->plan_max_a = c->plan_max_b = 0;
  for (int i = 0; i < n_pairs; i++) {
    c->plan_max_a = std::max(c->plan_max_a, pa[i]);
    c->plan_max_b = std::max(c->plan_max_b, pb[i]);
  }
  if (n_pairs == 0) return LORB_OK;
  LORB_TRY(c->plan_pairs.reserve((size_t)n_pairs * 8));
  LORB_TRY(c->plan_out.reserve((size_t)n_pairs * 12));
  LORB_TRY(pin_reserve(c, 2, (size_t)n_pairs * 12));
  int2* hp = c->h[2].as<int2>();
  for (int i = 0; i < n_pairs; i++) hp[i] = make_int2(pa[i], pb[i]);
  LORB_CUDA_TRY(cudaMemcpyAsync(c->plan_pairs.p, hp, (size_t)n_pairs * 8, cudaMemcpyHostToDevice,
                                c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  if (sweep_impl(c) == LORB_SWEEP_TENSOR) {
    if (c->tc_img_n_kf != c->bank_n_kf || c->tc_img_n_desc != c->bank_n_desc) LORB_TRY(tc::bank_expand(c));
    LORB_TRY(tc::plan_build(c, pa, pb, n_pairs));
  } else {
    c->tc_n_units = 0;
  }
  return LORB_OK;
}

int lorb_sweep_plan_run_at2(lorb_ctx* c, int kf_base_a, int kf_base_b) {
  LORB_REQUIRE(c, "ctx");
  LORB_REQUIRE(c->bank_n_kf > 0, "no bank uploaded");
  LORB_REQUIRE(kf_base_a >= 0 && kf_base_a + c->plan_max_a < c->bank_n_kf, "kf_base_a out of range");
  LORB_REQUIRE(kf_base_b >= 0 && kf_base_b + c->plan_max_b < c->bank_n_kf, "kf_base_b out of range");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  if (sweep_impl(c) == LORB_SWEEP_TENSOR) {
    LORB_REQUIRE(c->plan_n_pairs == 0 || c->tc_n_units > 0, "plan was uploaded for the popc kernel");
    return tc::launch_sweep(c, kf_base_a, kf_base_b, c->plan_n_pairs, c->plan_out.as<int>());
  }
  const size_t kf_u4 = (size_t)c->bank_n_desc * 2;
  return launch_sweep(c, c->bank.as<uint4>() + kf_u4 * kf_base_a, c->bank.as<uint4>() + kf_u4 * kf_base_b,
                      c->bank_n_desc, c->plan_pairs.as<int2>(), c->plan_n_pairs, c->plan_out.as<int>());
}

int lorb_sweep_plan_run_at(lorb_ctx* c, int kf_base) { return lorb_sweep_plan_run_at2(c, kf_base, kf_base); }

int lorb_sweep_plan_run(lorb_ctx* c) { return lorb_sweep_plan_run_at(c, 0); }

int lorb_sweep_plan_download(lorb_ctx* c, int* out_kept, int* out_matches, int* out_min) {
  LORB_REQUIRE(c, "ctx");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  const int n = c->plan_n_pairs;
  if (n == 0) return LORB_OK;
  LORB_TRY(pin_reserve(c, 2, (size_t)n * 12));
  LORB_CUDA_TRY(cudaMemcpyAsync(c->h[2].p, c->plan_out.p, (size_t)n * 12, cudaMemcpyDeviceToHost,
                                c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  const int* r = c->h[2].as<int>();
  for (int i = 0; i < n; i++) {
    if (out_kept) out_kept[i] = r[3 * i];
    if (out_matches) out_matches[i] = r[3 * i + 1];
    if (out_min) out_min[i] = r[3 * i + 2];
  }
  return LORB_OK;
}

int lorb_match_sweep_resident(lorb_ctx* c, const int* pa, const int* pb, int n_pairs, int* out_kept,
                              int* out_matches, int* out_min) {
  LORB_REQUIRE(c, "ctx");
  LORB_REQUIRE(n_pairs == 0 || out_kept, "out_kept");
  LORB_TRY(lorb_sweep_plan_upload(c, pa, pb, n_pairs));
  LORB_TRY(lorb_sweep_plan_run(c));
  return lorb_sweep_plan_download(c, out_kept, out_matches, out_min);
}

// ---- the whole sweep as a tile grid (SURVEY 8(e) row 1): blocks of block_kf keyframes, the
// upper-triangular grid of (block, block) tiles dealt round-robin to the ranks.
long long lorb_sweep_tile_count(int n_kf, int block_kf) {
  if (n_kf <= 0 || block_kf <= 0) return 0;
  const long long T = (n_kf + block_kf - 1) / block_kf;
  return T * (T + 1) / 2;
}

long long lorb_sweep_pair_index(int n_kf, int a, int b) {
  if (a > b) std::swap(a, b);
  return (long long)a * n_kf - (long long)a * (a + 1) / 2 + (b - a - 1);
}

int lorb_sweep_rank_tiles(int n_kf, int block_kf, int rank, int world, int cap, int* tile_bi,
                          int* tile_bj, int* n_out) {
  LORB_REQUIRE(n_kf > 0 && block_kf > 0 && world >= 1 && rank >= 0 && rank < world && n_out, "arguments");
  const int T = (n_kf + block_kf - 1) / block_kf;
  long long t = 0;
  int n = 0;
  for (int bi = 0; bi < T; bi++)
    for (int bj = bi; bj < T; bj++, t++) {
      if (t % world != rank) continue;
      // a one-keyframe diagonal block has no pair
      if (bi == bj && std::min(block_kf, n_kf - bi * block_kf) < 2) continue;
      if (n < cap && tile_bi && tile_bj) {
        tile_bi[n] = bi;
        tile_bj[n] = bj;
      }
      n++;
    }
  *n_out = n;
  return LORB_OK;
}

int lorb_match_sweep_all(lorb_ctx* c, int block_kf, int rank, int world, int* out_kept,
                         long long* n_pairs_done) {
  LORB_REQUIRE(c && out_kept, "ctx / out_kept");
  LORB_REQUIRE(c->bank_n_kf > 0, "no bank uploaded");
  LORB_REQUIRE(block_kf >= 1, "block_kf");
  const int n_kf = c->bank_n_kf;
  int n_tiles = 0;
  LORB_TRY(lorb_sweep_rank_tiles(n_kf, block_kf, rank, world, 0, nullptr, nullptr, &n_tiles));
  std::vector<int> bi(std::max(1, n_tiles)), bj(std::max(1, n_tiles));
  LORB_TRY(lorb_sweep_rank_tiles(n_kf, block_kf, rank, world, n_tiles, bi.data(), bj.data(), &n_tiles));
  // tiles of one shape (rows, columns, diagonal?) share a plan: go shape by shape
  std::vector<int> order(n_tiles);
  auto shape = [&](int t) {
    const int na = std::min(block_kf, n_kf - bi[t] * block_kf), nb = std::min(block_kf, n_kf - bj[t] * block_kf);
    return ((long long)na << 33) | ((long long)nb << 1) | (bi[t] == bj[t] ? 1 : 0);
  };
  for (int t = 0; t < n_tiles; t++) order[t] = t;
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return shape(x) > shape(y); });
  long long done = 0, cur_shape = -1;
  std::vector<int> pa, pb;
  // Results come back through two pinned buffers: the copy of tile k is queued behind its kernels, the
  // kernels of tile k+1 behind the copy, and the host scatters tile k while the GPU runs tile k+1.
  cudaEvent_t ev[2] = {nullptr, nullptr};
  for (auto& e : ev) LORB_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  struct Pending {
    int base_a, base_b, n;
    std::vector<int> pa, pb;
  } pend[2];
  pend[0].n = pend[1].n = 0;
  auto scatter = [&](int slot) -> int {
    Pending& P = pend[slot];
    if (P.n == 0) return LORB_OK;
    LORB_CUDA_TRY(cudaEventSynchronize(ev[slot]));
    const int* r = c->h[5 + slot].as<int>();
    for (int i = 0; i < P.n; i++)
      out_kept[lorb_sweep_pair_index(n_kf, P.base_a + P.pa[i], P.base_b + P.pb[i])] = r[3 * (size_t)i];
    done += P.n;
    P.n = 0;
    return LORB_OK;
  };
  int rc = LORB_OK;
  for (int k = 0; k < n_tiles && rc == LORB_OK; k++) {
    const int t = order[k], slot = k & 1;
    const int na = std::min(block_kf, n_kf - bi[t] * block_kf), nb = std::min(block_kf, n_kf - bj[t] * block_kf);
    const bool diag = bi[t] == bj[t];
    if (shape(t) != cur_shape) {
      // a new plan overwrites the device pair list: drain what is in flight first
      if ((rc = scatter(0)) != LORB_OK || (rc = scatter(1)) != LORB_OK) break;
      pa.clear();
      pb.clear();
      for (int a = 0; a < na; a++)
        for (int b = diag ? a + 1 : 0; b < nb; b++) {
          pa.push_back(a);
          pb.push_back(b);
        }
      if ((rc = lorb_sweep_plan_upload(c, pa.data(), pb.data(), (int)pa.size())) != LORB_OK) break;
      cur_shape = shape(t);
    }
    if ((rc = scatter(slot)) != LORB_OK) break;  // the buffer of tile k-2
    const int base_a = bi[t] * block_kf, base_b = bj[t] * block_kf, n = (int)pa.size();
    if ((rc = lorb_sweep_plan_run_at2(c, base_a, base_b)) != LORB_OK) break;
    if ((rc = pin_reserve(c, 5 + slot, (size_t)n * 12)) != LORB_OK) break;
    if (cudaMemcpyAsync(c->h[5 + slot].p, c->plan_out.p, (size_t)n * 12, cudaMemcpyDeviceToHost, c->stream) !=
            cudaSuccess ||
        cudaEventRecord(ev[slot], c->stream) != cudaSuccess) {
      set_error("sweep: result copy failed");
      rc = LORB_ERR_CUDA;
      break;
    }
    pend[slot].base_a = base_a;
    pend[slot].base_b = base_b;
    pend[slot].n = n;
    pend[slot].pa = pa;
    pend[slot].pb = pb;
  }
  if (rc == LORB_OK) rc = scatter(0);
  if (rc == LORB_OK) rc = scatter(1);
  cudaStreamSynchronize(c->stream);
  for (auto& e : ev) cudaEventDestroy(e);
  if (rc != LORB_OK) return rc;
  if (n_pairs_done) *n_pairs_done = done;
  return LORB_OK;
}

int lorb_match_sweep(lorb_ctx* c, const uint8_t* bank, int n_kf, int n_desc, const int* pa,
                     const int* pb, int n_pairs, int* out_kept, int* out_matches, int* out_min) {
  LORB_TRY(lorb_bank_upload(c, bank, n_kf, n_desc));
  return lorb_match_sweep_resident(c, pa, pb, n_pairs, out_kept, out_matches, out_min);
}

}  // extern "C"
