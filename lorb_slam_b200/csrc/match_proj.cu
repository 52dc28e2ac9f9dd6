// match_proj.cu — projection-guided descriptor search on sm_100a.
//
// Replaces Matcher::SearchByProjection(Frame*, const set<MapPoint*>&, th)
// (reference src/matcher.cpp:220-316) and
// Matcher::SearchByProjection(Frame* Cur, Frame* Last, th) (:64-218), including
// Frame::GetFeaturesInArea / PosInGrid (src/frame.cpp:370-423, :105-115).
//
// The reference is a sequential greedy loop: a keypoint claimed by an earlier
// point whose mnObs>0 is skipped by later points (:149-151, :273-275).  The GPU
// version splits it into
//   1. grid_build_kernel     64x48 cell CSR, items ascending inside a cell
//   2. candidates_kernel     one warp per point: window query in the
//                            reference's iteration order (cell column major),
//                            level / window / stereo gates, Hamming distance;
//                            ordered candidate lists (kp | dist<<20) in a CSR
//   3. resolve_coop_kernel   one cooperative launch: the claim semantics as a monotone
//                            fixpoint — fp[kp] = order index of the first
//                            protecting point that took kp; point k ignores
//                            candidates with fp[kp] < k.  Every fixpoint equals
//                            the sequential result (induction over k) and is
//                            reached in <= n+1 sweeps, in practice 3-6.
// Float arithmetic that decides candidate sets uses explicit _rn intrinsics so
// nothing is contracted into FMA (the reference is -O0 x86-64 code).
#include <cooperative_groups.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"

namespace lorb {

constexpr int NCELL = LORB_GRID_COLS * LORB_GRID_ROWS;

struct FrameDev {
  int n_kp;
  const float* x;
  const float* y;
  const int* octave;
  const float* angle;
  const float* uright;
  const uint4* desc;
  const int* claim_obs;
  const float* sf;
  float min_x, max_x, min_y, max_y, inv_w, inv_h;
  const int* cell_start;  // NCELL+1, cell id = ix*ROWS + iy
  const int* cell_items;
};

// ---- 1. grid (reference src/frame.cpp:87-115)
__global__ void __launch_bounds__(1024)
    grid_build_kernel(int n_kp, const float* __restrict__ x, const float* __restrict__ y,
                      float min_x, float min_y, float inv_w, float inv_h, int* __restrict__ cell_of,
                      int* __restrict__ cell_start, int* __restrict__ cell_items) {
  __shared__ int cnt[NCELL + 1];
  __shared__ int s_part[32];
  const int tid = threadIdx.x;
  for (int c = tid; c <= NCELL; c += blockDim.x) cnt[c] = 0;
  __syncthreads();
  for (int i = tid; i < n_kp; i += blockDim.x) {
    // PosInGrid: round(), not floor; cells 64 / 48 fall outside and the keypoint is dropped
    const int px = (int)roundf(__fmul_rn(__fsub_rn(x[i], min_x), inv_w));
    const int py = (int)roundf(__fmul_rn(__fsub_rn(y[i], min_y), inv_h));
    int c = -1;
    if (!(px < 0 || px >= LORB_GRID_COLS || py < 0 || py >= LORB_GRID_ROWS)) {
      c = px * LORB_GRID_ROWS + py;
      atomicAdd(&cnt[c], 1);
    }
    cell_of[i] = c;
  }
  __syncthreads();
  // exclusive scan of cnt[0..NCELL): 3 cells per thread + block scan
  const int per = (NCELL + 1023) / 1024;  // 3
  int local[4];
  int sum = 0;
  for (int k = 0; k < per; k++) {
    const int c = tid * per + k;
    local[k] = c < NCELL ? cnt[c] : 0;
    sum += local[k];
  }
  int incl = sum;
  const int lane = tid & 31, warp = tid >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_part[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int v = s_part[lane];
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += u;
    }
    s_part[lane] = v;
  }
  __syncthreads();
  int run = incl - sum + (warp > 0 ? s_part[warp - 1] : 0);
  __syncthreads();
  for (int k = 0; k < per; k++) {
    const int c = tid * per + k;
    if (c < NCELL) {
      cell_start[c] = run;
      cnt[c] = run;  // becomes the fill cursor
      run += local[k];
    }
  }
  if (tid == 1023) cell_start[NCELL] = run;
  __syncthreads();
  for (int i = tid; i < n_kp; i += blockDim.x) {
    const int c = cell_of[i];
    if (c >= 0) cell_items[atomicAdd(&cnt[c], 1)] = i;
  }
  __syncthreads();
  // cells are filled in ascending keypoint index in the reference (:95-102):
  // sort each (tiny) cell
  for (int c = tid; c < NCELL; c += blockDim.x) {
    const int s = cell_start[c], e = cnt[c];
    for (int a = s + 1; a < e; a++) {
      const int v = cell_items[a];
      int b = a - 1;
      while (b >= s && cell_items[b] > v) {
        cell_items[b + 1] = cell_items[b];
        b--;
      }
      cell_items[b + 1] = v;
    }
  }
}

// ---- window query shared by both searches (reference src/frame.cpp:370-423)
struct Window {
  float x, y, r;
  int min_level, max_level;
  int cx0, cx1, cy0, cy1;  // inclusive cell ranges; cx0 > cx1 means empty
};

__device__ __forceinline__ Window make_window(const FrameDev& f, float x, float y, float r,
                                              int min_level, int max_level) {
  Window w;
  w.x = x;
  w.y = y;
  w.r = r;
  w.min_level = min_level;
  w.max_level = max_level;
  w.cx0 = 1;
  w.cx1 = 0;
  w.cy0 = w.cy1 = 0;
  const float dx = __fsub_rn(x, f.min_x), dy = __fsub_rn(y, f.min_y);
  const int minx = max(0, (int)floorf(__fmul_rn(__fsub_rn(dx, r), f.inv_w)));
  if (minx >= LORB_GRID_COLS) return w;
  const int maxx = min(LORB_GRID_COLS - 1, (int)ceilf(__fmul_rn(__fadd_rn(dx, r), f.inv_w)));
  if (maxx < 0) return w;
  const int miny = max(0, (int)floorf(__fmul_rn(__fsub_rn(dy, r), f.inv_h)));
  if (miny >= LORB_GRID_ROWS) return w;
  const int maxy = min(LORB_GRID_ROWS - 1, (int)ceilf(__fmul_rn(__fadd_rn(dy, r), f.inv_h)));
  if (maxy < 0) return w;
  w.cx0 = minx;
  w.cx1 = maxx;
  w.cy0 = miny;
  w.cy1 = maxy;
  return w;
}

__device__ __forceinline__ bool in_window(const FrameDev& f, const Window& w, int k) {
  const bool check_levels = (w.min_level > 0) || (w.max_level >= 0);
  if (check_levels) {
    const int o = f.octave[k];
    if (o < w.min_level) return false;
    if (w.max_level >= 0 && o > w.max_level) return false;
  }
  const float distx = __fsub_rn(f.x[k], w.x), disty = __fsub_rn(f.y[k], w.y);
  return fabsf(distx) < w.r && fabsf(disty) < w.r;
}

__device__ __forceinline__ uint32_t hamming_gmem(const uint32_t (&q)[8], const uint4* __restrict__ d) {
  const uint4 lo = d[0], hi = d[1];
  const uint32_t t[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
  return hamming256_popc8(q, t);
}

// Per-point parameters produced by the mode-specific front end.
struct PointQuery {
  bool active;
  float x, y, r;       // window centre and half-size
  int min_level, max_level;
  float stereo_ref;    // value compared with mvuRight[idx]
  float stereo_tol;    // gate: |stereo_ref - uRight| > stereo_tol -> skip
};

// One warp per point.  Walks the window column by column (each column is one
// contiguous item range of the CSR), keeps the reference's order through
// ballot compaction.  Pass 0 counts, pass 1 writes (kp | dist<<20).
template <typename F>
__device__ __forceinline__ void warp_candidates(const FrameDev& f, const PointQuery& pq,
                                                const uint4* __restrict__ mp_desc, int lane,
                                                int* __restrict__ seg_start, int* __restrict__ seg_len,
                                                uint32_t* __restrict__ cand, int cand_cap,
                                                unsigned long long* __restrict__ counter, int k,
                                                F&& unused) {
  (void)unused;
  if (!pq.active) {
    if (lane == 0) {
      seg_start[k] = 0;
      seg_len[k] = 0;
    }
    return;
  }
  const Window w = make_window(f, pq.x, pq.y, pq.r, pq.min_level, pq.max_level);
  uint32_t q[8];
  {
    const uint4 lo = mp_desc[0], hi = mp_desc[1];
    q[0] = lo.x; q[1] = lo.y; q[2] = lo.z; q[3] = lo.w;
    q[4] = hi.x; q[5] = hi.y; q[6] = hi.z; q[7] = hi.w;
  }
  int total = 0, base = 0, in_win = 0;
  for (int pass = 0; pass < 2; pass++) {
    int written = 0;
    for (int ix = w.cx0; ix <= w.cx1; ix++) {
      const int s = f.cell_start[ix * LORB_GRID_ROWS + w.cy0];
      const int e = f.cell_start[ix * LORB_GRID_ROWS + w.cy1 + 1];
      for (int j0 = s; j0 < e; j0 += 32) {
        const int j = j0 + lane;
        bool ok = false;
        int kp = 0;
        if (j < e) {
          kp = f.cell_items[j];
          ok = in_window(f, w, kp);
          if (pass == 0) in_win += ok ? 1 : 0;
          if (ok) {
            const float ur = f.uright[kp];
            if (ur > 0.0f) {
              const float er = fabsf(__fsub_rn(pq.stereo_ref, ur));
              if (er > pq.stereo_tol) ok = false;
            }
          }
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, ok);
        if (pass == 1 && ok) {
          const int pos = base + written + __popc(bal & ((1u << lane) - 1u));
          if (pos < cand_cap) {
            const uint32_t d = hamming_gmem(q, f.desc + 2 * (size_t)kp);
            cand[pos] = (uint32_t)kp | (d << KEY_IDX_BITS);
          }
        }
        written += __popc(bal);
      }
    }
    if (pass == 0) {
      total = written;
      // counter[1]: sum of GetFeaturesInArea result sizes (before the stereo gate)
      in_win = __reduce_add_sync(0xffffffffu, in_win);
      if (lane == 0 && in_win > 0) atomicAdd(counter + 1, (unsigned long long)in_win);
      unsigned long long b = 0;
      if (lane == 0 && total > 0) b = atomicAdd(counter, (unsigned long long)total);
      b = __shfl_sync(0xffffffffu, b, 0);
      base = (int)min(b, (unsigned long long)0x7fffffff);
      if (lane == 0) {
        seg_start[k] = base;
        seg_len[k] = total;
      }
      if (total == 0) return;
    }
  }
}

// ---- 2a. candidates for SearchByProjection(F, set<MapPoint*>, th) (:226-253, :277-282)
__global__ void __launch_bounds__(256)
    candidates_points_kernel(FrameDev f, int n_pts, const float* __restrict__ proj_x,
                             const float* __restrict__ proj_y, const float* __restrict__ proj_xr,
                             const int* __restrict__ level, const float* __restrict__ view_cos,
                             const uint8_t* __restrict__ active, const uint4* __restrict__ mp_desc,
                             float th, int* __restrict__ seg_start, int* __restrict__ seg_len,
                             uint32_t* __restrict__ cand, int cand_cap,
                             unsigned long long* __restrict__ counter) {
  const int lane = threadIdx.x & 31;
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (k >= n_pts) return;
  PointQuery pq;
  pq.active = active[k] != 0;
  if (pq.active) {
    const int lvl = level[k];
    float r = ((double)view_cos[k] > 0.998) ? 2.5f : 4.0f;  // RadiusByViewingCos :430-436
    if (th != 1.0f) r = __fmul_rn(r, th);                     // bFactor :224, :244
    const float rs = __fmul_rn(r, f.sf[lvl]);
    pq.x = proj_x[k];
    pq.y = proj_y[k];
    pq.r = rs;
    pq.min_level = lvl - 1;
    pq.max_level = lvl;
    pq.stereo_ref = proj_xr[k];
    pq.stereo_tol = rs;
  }
  warp_candidates(f, pq, mp_desc + 2 * (size_t)k, lane, seg_start, seg_len, cand, cand_cap, counter,
                  k, 0);
}

struct PoseDev {
  float tcw[16];
  float fx, fy, cx, cy, mbf, mb;
  int forward, backward;
};

// ---- 2b. candidates for SearchByProjection(Cur, Last, th) (:89-160)
__global__ void __launch_bounds__(256)
    candidates_frame_kernel(FrameDev f, PoseDev P, int n_last, const uint8_t* __restrict__ valid,
                            const float* __restrict__ xw, const int* __restrict__ last_octave,
                            const uint4* __restrict__ mp_desc, float th,
                            int* __restrict__ seg_start, int* __restrict__ seg_len,
                            uint32_t* __restrict__ cand, int cand_cap,
                            unsigned long long* __restrict__ counter) {
  const int lane = threadIdx.x & 31;
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= n_last) return;
  PointQuery pq;
  pq.active = valid[i] != 0;
  if (pq.active) {
    const float X0 = xw[3 * i], X1 = xw[3 * i + 1], X2 = xw[3 * i + 2];
    // x3Dc = Rcw*x3Dw + tcw: OpenCV small-matrix gemm = sequential fp32, then + t
    float c[3];
#pragma unroll
    for (int r = 0; r < 3; r++) {
      float t = __fmul_rn(P.tcw[4 * r], X0);
      t = __fadd_rn(t, __fmul_rn(P.tcw[4 * r + 1], X1));
      t = __fadd_rn(t, __fmul_rn(P.tcw[4 * r + 2], X2));
      c[r] = __fadd_rn(t, P.tcw[4 * r + 3]);
    }
    const float invzc = (float)(1.0 / (double)c[2]);  // :105 double divide
    if (invzc < 0) {
      pq.active = false;  // :107
    } else {
      const float u = __fadd_rn(__fmul_rn(__fmul_rn(P.fx, c[0]), invzc), P.cx);  // :110
      const float v = __fadd_rn(__fmul_rn(__fmul_rn(P.fy, c[1]), invzc), P.cy);  // :111
      if (u < f.min_x || u > f.max_x || v < f.min_y || v > f.max_y) {
        pq.active = false;  // :113-116
      } else {
        const int oct = last_octave[i];
        const float radius = __fmul_rn(th, f.sf[oct]);  // :121
        pq.x = u;
        pq.y = v;
        pq.r = radius;
        if (P.forward) {  // :129-134
          pq.min_level = oct;
          pq.max_level = -1;
        } else if (P.backward) {
          pq.min_level = 0;
          pq.max_level = oct;
        } else {
          pq.min_level = oct - 1;
          pq.max_level = oct + 1;
        }
        pq.stereo_ref = __fsub_rn(u, __fmul_rn(P.mbf, invzc));  // :156
        pq.stereo_tol = radius;
      }
    }
  }
  warp_candidates(f, pq, mp_desc + 2 * (size_t)i, lane, seg_start, seg_len, cand, cand_cap, counter,
                  i, 0);
}

// ---- 3. claim resolution.  MODE 0: points (best/second + ratio, :265-312);
// MODE 1: frame (best only + rotation histogram, :139-215).
//
// One warp evaluates one point: lanes read consecutive candidates (coalesced),
// keys (dist << 32 | position) are min-reduced over the warp.  The reference's
// sequential best/second bookkeeping (:289-301) is reproduced exactly from
// three order statistics.  Let c* be the FIRST position of the minimum distance
// (strict '<' keeps the first).  When c* arrived it demoted the best of the
// prefix A = [0,c*) into the "second" slot; afterwards only a strictly smaller
// distance from the suffix Z = (c*,m) can replace it.  Hence
//     second = first-min(Z) if dist(first-min(Z)) < dist(first-min(A)) else first-min(A)
// (with (256, level -1) for an empty A), and bestLevel2 is that element's octave.
constexpr int RG = 8;  // lanes per point in the claim resolution (4 points per warp in flight)
__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
#pragma unroll
  for (int o = RG / 2; o > 0; o >>= 1) {
    const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o);
    v = u < v ? u : v;
  }
  return v;
}

template <int MODE>
__device__ __forceinline__ int choose_warp(const uint32_t* __restrict__ cand, int s, int n,
                                           const int* fp /* rewritten between sweeps: no .nc loads */, int k,
                                           const int* __restrict__ kp_octave, int lane) {
  const unsigned long long NONE = ~0ull;
  unsigned long long kbest = NONE;
  for (int c = lane; c < n; c += RG) {
    const uint32_t rec = cand[s + c];
    if (fp[rec & KEY_IDX_MASK] < k) continue;  // held by a map point with mnObs>0 at this point's turn
    if ((rec >> KEY_IDX_BITS) >= 256u) continue;  // 256 never beats the initial bestDist / bestDist2
    const unsigned long long key = ((unsigned long long)(rec >> KEY_IDX_BITS) << 32) | (unsigned)c;
    kbest = key < kbest ? key : kbest;
  }
  kbest = warp_min_u64(kbest);
  // (no early return before the last shuffle: the other groups of the warp still need this one)
  const bool none = kbest == NONE || (int)(kbest >> 32) > LORB_TH_HIGH;
  const int bestDist = none ? 256 : (int)(kbest >> 32);
  const int cstar = none ? -1 : (int)(kbest & 0xffffffffu);
  const int bestIdx = none ? -1 : (int)(cand[s + cstar] & KEY_IDX_MASK);
  if (MODE == 1) return bestIdx;
  unsigned long long ka = NONE, kz = NONE;
  for (int c = lane; c < n; c += RG) {
    if (c == cstar) continue;
    const uint32_t rec = cand[s + c];
    if (fp[rec & KEY_IDX_MASK] < k) continue;
    if ((rec >> KEY_IDX_BITS) >= 256u) continue;
    const unsigned long long key = ((unsigned long long)(rec >> KEY_IDX_BITS) << 32) | (unsigned)c;
    if (c < cstar) ka = key < ka ? key : ka;
    else kz = key < kz ? key : kz;
  }
  ka = warp_min_u64(ka);
  kz = warp_min_u64(kz);
  if (none) return -1;
  int bestDist2 = 256, bestLevel2 = -1;
  if (ka != NONE) {
    bestDist2 = (int)(ka >> 32);
    bestLevel2 = kp_octave[cand[s + (int)(ka & 0xffffffffu)] & KEY_IDX_MASK];
  }
  if (kz != NONE && (int)(kz >> 32) < bestDist2) {
    bestDist2 = (int)(kz >> 32);
    bestLevel2 = kp_octave[cand[s + (int)(kz & 0xffffffffu)] & KEY_IDX_MASK];
  }
  const int bestLevel = kp_octave[bestIdx];
  if (bestLevel == bestLevel2 && (double)bestDist > 0.8 * (double)bestDist2) return -1;  // :307
  return bestIdx;
}

// ---- Frame::IsInFrustum + MapPoint::PredictScale, one thread per map point
struct FrustumDev {
  float tcw[16];
  float ow[3];
  float fx, fy, cx, cy, mbf;
  float min_x, max_x, min_y, max_y;
  float cos_limit, log_sf;
  int n_levels;
};

__global__ void frustum_kernel(FrustumDev F, int n, const float* __restrict__ xw,
                               const float* __restrict__ nrm, const float* __restrict__ dmin,
                               const float* __restrict__ dmax, uint8_t* __restrict__ in_view,
                               float* __restrict__ px, float* __restrict__ py, float* __restrict__ pxr,
                               int* __restrict__ level, float* __restrict__ vcos) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  in_view[i] = 0;
  const float P0 = xw[3 * i], P1 = xw[3 * i + 1], P2 = xw[3 * i + 2];
  // Pc = mTcw * (P,1): OpenCV small gemm = sequential fp32 multiply-add, no FMA (frame.cpp:434-440)
  float c[3];
#pragma unroll
  for (int r = 0; r < 3; r++) {
    float t = __fmul_rn(F.tcw[4 * r], P0);
    t = __fadd_rn(t, __fmul_rn(F.tcw[4 * r + 1], P1));
    t = __fadd_rn(t, __fmul_rn(F.tcw[4 * r + 2], P2));
    c[r] = __fadd_rn(t, __fmul_rn(F.tcw[4 * r + 3], 1.0f));
  }
  if (c[2] < 0.0f) return;                                                        // :443
  const float invz = __fdiv_rn(1.0f, c[2]);                                       // :446
  const float u = __fadd_rn(__fmul_rn(__fmul_rn(F.fx, c[0]), invz), F.cx);        // :447
  const float v = __fadd_rn(__fmul_rn(__fmul_rn(F.fy, c[1]), invz), F.cy);        // :448
  if (u < F.min_x || u > F.max_x) return;                                         // :450
  if (v < F.min_y || v > F.max_y) return;                                         // :452
  const float maxd = __fmul_rn(1.2f, dmax[i]), mind = __fmul_rn(0.8f, dmin[i]);   // map_point.cpp:209-217
  const float o0 = __fsub_rn(P0, F.ow[0]), o1 = __fsub_rn(P1, F.ow[1]), o2 = __fsub_rn(P2, F.ow[2]);
  // cv::norm(Point3f) accumulates in double (:462)
  const float dist = (float)sqrt((double)o0 * o0 + (double)o1 * o1 + (double)o2 * o2);
  if (dist < mind || dist > maxd) return;                                         // :464
  const float dot = __fadd_rn(__fadd_rn(__fmul_rn(o0, nrm[3 * i]), __fmul_rn(o1, nrm[3 * i + 1])),
                              __fmul_rn(o2, nrm[3 * i + 2]));
  const float vc = __fdiv_rn(dot, dist);                                          // :472
  if (vc < F.cos_limit) return;                                                   // :474
  // PredictScale (map_point.cpp:267-284): ceil(log(mfMaxDistance/dist) / mfLogScaleFactor)
  const float ratio = __fdiv_rn(dmax[i], dist);
  const float lg = (float)log((double)ratio);  // logf; double log rounded = correctly rounded float
  int ns = (int)ceilf(__fdiv_rn(lg, F.log_sf));
  if (ns < 0) ns = 0;
  else if (ns >= F.n_levels) ns = F.n_levels - 1;
  in_view[i] = 1;
  px[i] = u;
  pxr[i] = __fsub_rn(u, __fmul_rn(F.mbf, invz));                                  // :487
  py[i] = v;
  level[i] = ns;
  vcos[i] = vc;
}

// ---- 3b. the claim resolution runs as one COOPERATIVE multi-CTA launch: the
// per-sweep evaluation is latency-bound (a handful of dependent loads per
// point), so it is spread over all SMs (8 lanes per point, every point in
// flight at once) with a grid-wide barrier between the phases of a sweep.
// scratch: int[8] = {changed[3], count, ind1, ind2, ind3, sweeps} + int hist[30]
template <int MODE>
__global__ void __launch_bounds__(256)
    resolve_coop_kernel(int n_kp, int n_pts, const int* __restrict__ claim_obs,
                        const int* __restrict__ kp_octave, const float* __restrict__ kp_angle,
                        const int* __restrict__ mp_nobs, const float* __restrict__ last_angle,
                        const int* __restrict__ seg_start, const int* __restrict__ seg_len,
                        const uint32_t* __restrict__ cand, int* fp_a, int* fp_b, int* choice,
                        int* out_for_kp, int* res, int* scratch,
                        const unsigned long long* __restrict__ cand_total, unsigned long long cand_cap) {
  namespace cg = cooperative_groups;
  // the candidate arena overflowed: the segments point past its end and the host repeats the search
  // with the exact size -- nothing to resolve in this attempt; every CTA leaves, before any grid barrier
  if (*cand_total > cand_cap) return;
  cg::grid_group grid = cg::this_grid();
  const int INF = 0x7fffffff;
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsize = gridDim.x * blockDim.x;
  int* changed = scratch;       // [3]
  int* count = scratch + 3;
  int* ind = scratch + 4;       // [3]
  int* hist = scratch + 8;      // [30]
  for (int i = gtid; i < n_kp; i += gsize) {
    fp_a[i] = claim_obs[i] > 0 ? -1 : INF;
    out_for_kp[i] = -1;
  }
  for (int k = gtid; k < n_pts; k += gsize) choice[k] = -2;
  if (gtid < 8 + LORB_HISTO_LENGTH) scratch[gtid] = 0;
  int* fp_cur = fp_a;
  int* fp_new = fp_b;
  int sweeps = 0;
  for (;;) {
    for (int i = gtid; i < n_kp; i += gsize) fp_new[i] = claim_obs[i] > 0 ? -1 : INF;
    if (gtid == 0) changed[(sweeps + 1) % 3] = 0;
    grid.sync();
    {
      const int lane = gtid & (RG - 1), ngroups = gsize / RG, per_warp = 32 / RG;
      for (int base = (gtid >> 5) * per_warp; base < n_pts; base += ngroups) {
        const int k = base + ((gtid & 31) / RG);
        const int n = k < n_pts ? seg_len[k] : 0;
        const int c = choose_warp<MODE>(cand, n > 0 ? seg_start[k] : 0, n, fp_cur, k, kp_octave, lane);
        if (lane == 0 && k < n_pts) {
          if (c != choice[k]) {
            choice[k] = c;
            changed[sweeps % 3] = 1;
          }
          if (c >= 0 && mp_nobs[k] > 0) atomicMin(&fp_new[c], k);
        }
      }
    }
    grid.sync();
    const int any = *reinterpret_cast<volatile int*>(&changed[sweeps % 3]);
    sweeps++;
    int* t = fp_cur;
    fp_cur = fp_new;
    fp_new = t;
    if (!any) break;
  }
  // final holder of a keypoint = last point that took it
  auto bin_of = [&](int k, int c) {
    float rot = __fsub_rn(last_angle[k], kp_angle[c]);  // :181-188
    if (rot < 0.0f) rot = __fadd_rn(rot, 360.0f);
    int bin = (int)roundf(__fmul_rn(rot, (float)LORB_HISTO_LENGTH / 360.0f));
    if (bin == LORB_HISTO_LENGTH) bin = 0;
    return bin;
  };
  int cnt = 0;
  for (int k = gtid; k < n_pts; k += gsize) {
    const int c = choice[k];
    if (c >= 0) {
      cnt++;
      atomicMax(&out_for_kp[c], k);
      if (MODE == 1) atomicAdd(&hist[bin_of(k, c)], 1);
    }
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(count, cnt);
  grid.sync();
  if (MODE == 1) {
    if (gtid == 0) {  // ComputeThreeMaxima :387-428
      int max1 = 0, max2 = 0, max3 = 0, i1 = -1, i2 = -1, i3 = -1;
      for (int i = 0; i < LORB_HISTO_LENGTH; i++) {
        const int sz = hist[i];
        if (sz > max1) {
          max3 = max2; max2 = max1; max1 = sz;
          i3 = i2; i2 = i1; i1 = i;
        } else if (sz > max2) {
          max3 = max2; max2 = sz;
          i3 = i2; i2 = i;
        } else if (sz > max3) {
          max3 = sz;
          i3 = i;
        }
      }
      if ((float)max2 < __fmul_rn(0.1f, (float)max1)) {
        i2 = -1;
        i3 = -1;
      } else if ((float)max3 < __fmul_rn(0.1f, (float)max1)) {
        i3 = -1;
      }
      ind[0] = i1; ind[1] = i2; ind[2] = i3;
    }
    grid.sync();
    const int i1 = *reinterpret_cast<volatile int*>(&ind[0]), i2 = *reinterpret_cast<volatile int*>(&ind[1]),
              i3 = *reinterpret_cast<volatile int*>(&ind[2]);
    int dropped = 0;
    for (int k = gtid; k < n_pts; k += gsize) {
      const int c = choice[k];
      if (c >= 0) {
        const int bin = bin_of(k, c);
        if (bin != i1 && bin != i2 && bin != i3) {
          out_for_kp[c] = -2;  // :204-214
          dropped++;
        }
      }
    }
    dropped = __reduce_add_sync(0xffffffffu, dropped);
    if ((threadIdx.x & 31) == 0 && dropped) atomicSub(count, dropped);
    grid.sync();
  }
  if (gtid == 0) {
    res[0] = *reinterpret_cast<volatile int*>(count);
    res[1] = sweeps;
  }
}

// ------------------------------------------------------------------ host side
struct Packer {  // lays host arrays out in one pinned block / one device block
  size_t off = 0;
  size_t add(size_t bytes) {
    const size_t o = off;
    off = (off + bytes + 255) & ~(size_t)255;
    return o;
  }
};

static int check_frame(const lorb_frame_view* f) {
  LORB_REQUIRE(f, "frame view");
  LORB_REQUIRE(f->n_kp >= 0 && (unsigned)f->n_kp < KEY_IDX_MASK, "n_kp");
  LORB_REQUIRE(f->n_levels > 0 && f->scale_factors, "scale factors");
  LORB_REQUIRE(f->max_x > f->min_x && f->max_y > f->min_y, "image bounds");
  if (f->n_kp > 0)
    LORB_REQUIRE(f->kp_x && f->kp_y && f->kp_octave && f->kp_angle && f->kp_uright && f->desc &&
                     f->kp_claim_obs,
                 "frame arrays");
  return LORB_OK;
}

struct Upload {
  uint8_t* h;
  uint8_t* d;
  template <typename T>
  const T* put(size_t off, const void* src, size_t bytes) const {
    if (bytes) memcpy(h + off, src, bytes);
    return reinterpret_cast<const T*>(d + off);
  }
};

// Shared driver: uploads, builds the grid, runs `launch_cand`, resolves, downloads.
template <int MODE, typename LaunchCand>
static int run_search(lorb_ctx* c, const lorb_frame_view* fv, int n_pts, const uint8_t* mp_desc,
                      const int* mp_nobs, const float* last_angle, size_t extra_bytes,
                      LaunchCand&& launch_cand, int* out_for_point, int* out_for_kp, int* n_matches,
                      long long* n_candidates) {
  const int n_kp = fv->n_kp;
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  Packer pk;
  const size_t o_x = pk.add((size_t)n_kp * 4), o_y = pk.add((size_t)n_kp * 4),
               o_oct = pk.add((size_t)n_kp * 4), o_ang = pk.add((size_t)n_kp * 4),
               o_ur = pk.add((size_t)n_kp * 4), o_desc = pk.add((size_t)n_kp * 32),
               o_claim = pk.add((size_t)n_kp * 4), o_sf = pk.add((size_t)fv->n_levels * 4),
               o_mpd = pk.add((size_t)n_pts * 32), o_nobs = pk.add((size_t)n_pts * 4),
               o_lang = pk.add(last_angle ? (size_t)n_pts * 4 : 0), o_extra = pk.add(extra_bytes);
  const size_t up_bytes = pk.off;
  // device-only scratch
  Packer ws;
  const size_t w_cellof = ws.add((size_t)n_kp * 4), w_cstart = ws.add((size_t)(NCELL + 1) * 4),
               w_citems = ws.add((size_t)n_kp * 4), w_segs = ws.add((size_t)n_pts * 4),
               w_segl = ws.add((size_t)n_pts * 4), w_fpa = ws.add((size_t)n_kp * 4),
               w_fpb = ws.add((size_t)n_kp * 4), w_counter = ws.add(16), w_scratch = ws.add(256);
  // outputs (one D2H): res[4] | choice[n_pts] | out_for_kp[n_kp] | counter
  Packer op;
  const size_t r_res = op.add(16), r_choice = op.add((size_t)n_pts * 4),
               r_forkp = op.add((size_t)n_kp * 4), r_cnt = op.add(16);
  LORB_TRY(pin_reserve(c, 0, up_bytes));
  LORB_TRY(pin_reserve(c, 1, op.off));
  LORB_TRY(dev_reserve(c, 0, up_bytes));
  LORB_TRY(dev_reserve(c, 1, ws.off));
  LORB_TRY(dev_reserve(c, 2, op.off));
  size_t cand_cap = std::max<size_t>((size_t)n_pts * 128, (size_t)1 << 18);
  for (int attempt = 0; attempt < 2; attempt++) {
    LORB_TRY(dev_reserve(c, 3, cand_cap * 4));
    Upload up{c->h[0].as<uint8_t>(), c->d[0].as<uint8_t>()};
    FrameDev f;
    f.n_kp = n_kp;
    f.x = up.put<float>(o_x, fv->kp_x, (size_t)n_kp * 4);
    f.y = up.put<float>(o_y, fv->kp_y, (size_t)n_kp * 4);
    f.octave = up.put<int>(o_oct, fv->kp_octave, (size_t)n_kp * 4);
    f.angle = up.put<float>(o_ang, fv->kp_angle, (size_t)n_kp * 4);
    f.uright = up.put<float>(o_ur, fv->kp_uright, (size_t)n_kp * 4);
    f.desc = up.put<uint4>(o_desc, fv->desc, (size_t)n_kp * 32);
    f.claim_obs = up.put<int>(o_claim, fv->kp_claim_obs, (size_t)n_kp * 4);
    f.sf = up.put<float>(o_sf, fv->scale_factors, (size_t)fv->n_levels * 4);
    const uint4* d_mpd = up.put<uint4>(o_mpd, mp_desc, (size_t)n_pts * 32);
    const int* d_nobs = up.put<int>(o_nobs, mp_nobs, (size_t)n_pts * 4);
    const float* d_lang = up.put<float>(o_lang, last_angle, last_angle ? (size_t)n_pts * 4 : 0);
    f.min_x = fv->min_x;
    f.max_x = fv->max_x;
    f.min_y = fv->min_y;
    f.max_y = fv->max_y;
    // ComputeImageBounds src/frame.cpp:83-84 (float division)
    f.inv_w = (float)LORB_GRID_COLS / (fv->max_x - fv->min_x);
    f.inv_h = (float)LORB_GRID_ROWS / (fv->max_y - fv->min_y);
    uint8_t* wsd = c->d[1].as<uint8_t>();
    int* d_cellof = reinterpret_cast<int*>(wsd + w_cellof);
    int* d_cstart = reinterpret_cast<int*>(wsd + w_cstart);
    int* d_citems = reinterpret_cast<int*>(wsd + w_citems);
    int* d_segs = reinterpret_cast<int*>(wsd + w_segs);
    int* d_segl = reinterpret_cast<int*>(wsd + w_segl);
    int* d_fpa = reinterpret_cast<int*>(wsd + w_fpa);
    int* d_fpb = reinterpret_cast<int*>(wsd + w_fpb);
    unsigned long long* d_counter = reinterpret_cast<unsigned long long*>(wsd + w_counter);
    f.cell_start = d_cstart;
    f.cell_items = d_citems;
    uint8_t* outd = c->d[2].as<uint8_t>();
    int* d_res = reinterpret_cast<int*>(outd + r_res);
    int* d_choice = reinterpret_cast<int*>(outd + r_choice);
    int* d_forkp = reinterpret_cast<int*>(outd + r_forkp);
    uint32_t* d_cand = c->d[3].as<uint32_t>();

    launch_cand.fill(up.h + o_extra);  // mode-specific host arrays into the staging block
    LORB_CUDA_TRY(cudaMemcpyAsync(up.d, up.h, up_bytes, cudaMemcpyHostToDevice, c->stream));
    LORB_CUDA_TRY(cudaMemsetAsync(d_counter, 0, 16, c->stream));
    LORB_LAUNCH(c, grid_build_kernel, 1, 1024, 0, n_kp, f.x, f.y, f.min_x, f.min_y, f.inv_w,
                f.inv_h, d_cellof, d_cstart, d_citems);
    if (n_pts > 0) {
      LORB_TRY(launch_cand.launch(c, f, up.d + o_extra, d_mpd, d_segs, d_segl, d_cand,
                                  (int)std::min<size_t>(cand_cap, 0x7fffffff), d_counter));
    }
    // per context (= per device and calling thread): co-resident CTAs of the cooperative kernel
    int* coop_blocks = c->proj_coop_blocks;
    if (coop_blocks[MODE] < 0) {
      int per_sm = 0;
      LORB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, resolve_coop_kernel<MODE>, 256, 0));
      if (per_sm == 0) {
        set_error("projection search: the claim resolution kernel cannot be resident on this device");
        return LORB_ERR_STATE;
      }
      coop_blocks[MODE] = per_sm * c->sm_count;
    }
    int* d_scratch = reinterpret_cast<int*>(wsd + w_scratch);
    const int want = std::max(1, (int)(((size_t)std::max(n_pts, 1) * RG + 255) / 256));
    const int grid = std::min(want, coop_blocks[MODE]);
    int a_nkp = n_kp, a_npts = n_pts;
    const int* a_claim = f.claim_obs;
    const int* a_oct = f.octave;
    const float* a_ang = f.angle;
    const uint32_t* a_cand = d_cand;
    const int* a_segs = d_segs;
    const int* a_segl = d_segl;
    const unsigned long long* a_total = d_counter;
    unsigned long long a_cap = cand_cap;
    void* args[] = {&a_nkp, &a_npts, &a_claim, &a_oct, &a_ang, (void*)&d_nobs, (void*)&d_lang,
                    &a_segs, &a_segl, &a_cand, &d_fpa, &d_fpb, &d_choice, &d_forkp, &d_res,
                    &d_scratch, &a_total, &a_cap};
    LORB_CUDA_TRY(cudaLaunchCooperativeKernel((void*)resolve_coop_kernel<MODE>, dim3(grid),
                                              dim3(256), args, 0, c->stream));
    c->launches++;
    LORB_CUDA_TRY(cudaMemcpyAsync(outd + r_cnt, d_counter, 16, cudaMemcpyDeviceToDevice, c->stream));
    LORB_CUDA_TRY(cudaMemcpyAsync(c->h[1].p, outd, op.off, cudaMemcpyDeviceToHost, c->stream));
    LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
    const uint8_t* ho = c->h[1].as<uint8_t>();
    const unsigned long long total = *reinterpret_cast<const unsigned long long*>(ho + r_cnt);
    if (total > cand_cap) {  // candidate arena too small: retry once with the exact size
      cand_cap = (size_t)total;
      continue;
    }
    const int* res = reinterpret_cast<const int*>(ho + r_res);
    *n_matches = res[0];
    if (getenv("LORB_DEBUG")) fprintf(stderr, "[lorb] projection search: %d claim sweeps\n", res[1]);
    if (n_candidates)
      *n_candidates = (long long)reinterpret_cast<const unsigned long long*>(ho + r_cnt)[1];
    if (n_pts) memcpy(out_for_point, ho + r_choice, (size_t)n_pts * 4);
    if (n_kp) memcpy(out_for_kp, ho + r_forkp, (size_t)n_kp * 4);
    return LORB_OK;
  }
  set_error("candidate arena overflow persisted");
  return LORB_ERR_STATE;
}

}  // namespace lorb

using namespace lorb;

extern "C" {

int lorb_frustum_project(lorb_ctx* c, const float* tcw, const float* ow, const lorb_intrinsics* K,
                         float min_x, float max_x, float min_y, float max_y, int n, const float* xw,
                         const float* normal, const float* min_dist, const float* max_dist,
                         float viewing_cos_limit, float log_scale_factor, int n_levels,
                         uint8_t* in_view, float* proj_x, float* proj_y, float* proj_xr, int* level,
                         float* view_cos) {
  LORB_REQUIRE(c && tcw && ow && K, "ctx / pose / intrinsics");
  LORB_REQUIRE(n >= 0 && n_levels > 0, "sizes");
  if (n == 0) return LORB_OK;
  LORB_REQUIRE(xw && normal && min_dist && max_dist, "point arrays");
  LORB_REQUIRE(in_view && proj_x && proj_y && proj_xr && level && view_cos, "outputs");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  Packer in, out;
  const size_t i_xw = in.add((size_t)n * 12), i_n = in.add((size_t)n * 12), i_dmin = in.add((size_t)n * 4),
               i_dmax = in.add((size_t)n * 4);
  const size_t o_px = out.add((size_t)n * 4), o_py = out.add((size_t)n * 4), o_pxr = out.add((size_t)n * 4),
               o_lvl = out.add((size_t)n * 4), o_vc = out.add((size_t)n * 4), o_in = out.add((size_t)n);
  LORB_TRY(pin_reserve(c, 0, in.off));
  LORB_TRY(pin_reserve(c, 1, out.off));
  LORB_TRY(dev_reserve(c, 0, in.off));
  LORB_TRY(dev_reserve(c, 2, out.off));
  uint8_t* h = c->h[0].as<uint8_t>();
  memcpy(h + i_xw, xw, (size_t)n * 12);
  memcpy(h + i_n, normal, (size_t)n * 12);
  memcpy(h + i_dmin, min_dist, (size_t)n * 4);
  memcpy(h + i_dmax, max_dist, (size_t)n * 4);
  // outputs of points that fail a test keep the caller's values: stage them too
  uint8_t* ho = c->h[1].as<uint8_t>();
  memcpy(ho + o_px, proj_x, (size_t)n * 4);
  memcpy(ho + o_py, proj_y, (size_t)n * 4);
  memcpy(ho + o_pxr, proj_xr, (size_t)n * 4);
  memcpy(ho + o_lvl, level, (size_t)n * 4);
  memcpy(ho + o_vc, view_cos, (size_t)n * 4);
  uint8_t* d = c->d[0].as<uint8_t>();
  uint8_t* dout = c->d[2].as<uint8_t>();
  LORB_CUDA_TRY(cudaMemcpyAsync(d, h, in.off, cudaMemcpyHostToDevice, c->stream));
  LORB_CUDA_TRY(cudaMemcpyAsync(dout, ho, out.off, cudaMemcpyHostToDevice, c->stream));
  FrustumDev F;
  memcpy(F.tcw, tcw, sizeof(F.tcw));
  memcpy(F.ow, ow, sizeof(F.ow));
  F.fx = K->fx; F.fy = K->fy; F.cx = K->cx; F.cy = K->cy; F.mbf = K->mbf;
  F.min_x = min_x; F.max_x = max_x; F.min_y = min_y; F.max_y = max_y;
  F.cos_limit = viewing_cos_limit;
  F.log_sf = log_scale_factor;
  F.n_levels = n_levels;
  LORB_LAUNCH(c, frustum_kernel, (n + 255) / 256, 256, 0, F, n, (const float*)(d + i_xw),
              (const float*)(d + i_n), (const float*)(d + i_dmin), (const float*)(d + i_dmax),
              dout + o_in, (float*)(dout + o_px), (float*)(dout + o_py), (float*)(dout + o_pxr),
              (int*)(dout + o_lvl), (float*)(dout + o_vc));
  LORB_CUDA_TRY(cudaMemcpyAsync(ho, dout, out.off, cudaMemcpyDeviceToHost, c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  memcpy(proj_x, ho + o_px, (size_t)n * 4);
  memcpy(proj_y, ho + o_py, (size_t)n * 4);
  memcpy(proj_xr, ho + o_pxr, (size_t)n * 4);
  memcpy(level, ho + o_lvl, (size_t)n * 4);
  memcpy(view_cos, ho + o_vc, (size_t)n * 4);
  memcpy(in_view, ho + o_in, (size_t)n);
  return LORB_OK;
}

int lorb_search_proj_points(lorb_ctx* c, const lorb_frame_view* frame, int n_pts,
                            const float* proj_x, const float* proj_y, const float* proj_xr,
                            const int* level, const float* view_cos, const uint8_t* active,
                            const uint8_t* mp_desc, const int* mp_nobs, float th,
                            int* out_kp_for_point, int* out_point_for_kp, int* n_matches,
                            long long* n_candidates) {
  LORB_REQUIRE(c, "ctx");
  LORB_TRY(check_frame(frame));
  LORB_REQUIRE(n_pts >= 0 && n_matches, "n_pts / n_matches");
  if (n_pts > 0) {
    LORB_REQUIRE(proj_x && proj_y && proj_xr && level && view_cos && active && mp_desc && mp_nobs &&
                     out_kp_for_point,
                 "point arrays");
    for (int k = 0; k < n_pts; k++)
      if (active[k]) LORB_REQUIRE(level[k] >= 0 && level[k] < frame->n_levels, "level out of range");
  }
  LORB_REQUIRE(frame->n_kp == 0 || out_point_for_kp, "out_point_for_kp");
  struct L {
    int n;
    const float *px, *py, *pxr, *vc;
    const int* lvl;
    const uint8_t* act;
    float th;
    size_t o1, o2, o3, o4, o5, o6;
    void fill(uint8_t* h) const {
      if (!n) return;
      memcpy(h + o1, px, (size_t)n * 4);
      memcpy(h + o2, py, (size_t)n * 4);
      memcpy(h + o3, pxr, (size_t)n * 4);
      memcpy(h + o4, lvl, (size_t)n * 4);
      memcpy(h + o5, vc, (size_t)n * 4);
      memcpy(h + o6, act, (size_t)n);
    }
    int launch(lorb_ctx* c, const FrameDev& f, const uint8_t* d, const uint4* d_mpd, int* segs,
               int* segl, uint32_t* cand, int cap, unsigned long long* counter) const {
      LORB_LAUNCH(c, candidates_points_kernel, (n * 32 + 255) / 256, 256, 0, f, n,
                  (const float*)(d + o1), (const float*)(d + o2), (const float*)(d + o3),
                  (const int*)(d + o4), (const float*)(d + o5), d + o6, d_mpd, th, segs, segl, cand,
                  cap, counter);
      return LORB_OK;
    }
  } l;
  Packer pk;
  l.n = n_pts;
  l.px = proj_x; l.py = proj_y; l.pxr = proj_xr; l.vc = view_cos; l.lvl = level; l.act = active;
  l.th = th;
  l.o1 = pk.add((size_t)n_pts * 4); l.o2 = pk.add((size_t)n_pts * 4); l.o3 = pk.add((size_t)n_pts * 4);
  l.o4 = pk.add((size_t)n_pts * 4); l.o5 = pk.add((size_t)n_pts * 4); l.o6 = pk.add((size_t)n_pts);
  return run_search<0>(c, frame, n_pts, mp_desc, mp_nobs, nullptr, pk.off, l, out_kp_for_point,
                       out_point_for_kp, n_matches, n_candidates);
}

int lorb_search_proj_frame(lorb_ctx* c, const lorb_frame_view* cur, const float* tcw_cur,
                           const float* tcw_last, const lorb_intrinsics* K, int n_last,
                           const uint8_t* last_valid, const float* last_xw, const int* last_octave,
                           const float* last_angle, const uint8_t* mp_desc, const int* mp_nobs,
                           float th, int* out_kp_for_item, int* out_state_for_kp, int* n_matches,
                           long long* n_candidates) {
  LORB_REQUIRE(c, "ctx");
  LORB_TRY(check_frame(cur));
  LORB_REQUIRE(tcw_cur && tcw_last && K && n_matches, "poses / intrinsics");
  LORB_REQUIRE(n_last >= 0, "n_last");
  if (n_last > 0) {
    LORB_REQUIRE(last_valid && last_xw && last_octave && last_angle && mp_desc && mp_nobs &&
                     out_kp_for_item,
                 "last-frame arrays");
    for (int i = 0; i < n_last; i++)
      if (last_valid[i])
        LORB_REQUIRE(last_octave[i] >= 0 && last_octave[i] < cur->n_levels, "octave out of range");
  }
  LORB_REQUIRE(cur->n_kp == 0 || out_state_for_kp, "out_state_for_kp");
  PoseDev P;
  memcpy(P.tcw, tcw_cur, sizeof(P.tcw));
  P.fx = K->fx; P.fy = K->fy; P.cx = K->cx; P.cy = K->cy; P.mbf = K->mbf; P.mb = K->mb;
  {
    // tlc of reference src/matcher.cpp:74-83 — three 3x3 float products per call, done on the
    // host with the rounding OpenCV's small-matrix gemm uses (sequential fp32, no FMA;
    // pinned against cv2.gemm in tests/golden/gemm_golden.npz)
    volatile float twc[3], tlc2;
    for (int i = 0; i < 3; i++) {
      volatile float t = tcw_cur[i] * tcw_cur[3];
      volatile float m1 = tcw_cur[4 + i] * tcw_cur[7];
      t = t + m1;
      volatile float m2 = tcw_cur[8 + i] * tcw_cur[11];
      t = t + m2;
      twc[i] = -t;
    }
    volatile float t = tcw_last[8] * twc[0];
    volatile float m1 = tcw_last[9] * twc[1];
    t = t + m1;
    volatile float m2 = tcw_last[10] * twc[2];
    t = t + m2;
    tlc2 = t + tcw_last[11];
    P.forward = tlc2 > K->mb;    // :86
    P.backward = -tlc2 > K->mb;  // :87
  }
  struct L {
    int n;
    PoseDev P;
    const uint8_t* valid;
    const float* xw;
    const int* oct;
    float th;
    size_t o1, o2, o3;
    void fill(uint8_t* h) const {
      if (!n) return;
      memcpy(h + o1, valid, (size_t)n);
      memcpy(h + o2, xw, (size_t)n * 12);
      memcpy(h + o3, oct, (size_t)n * 4);
    }
    int launch(lorb_ctx* c, const FrameDev& f, const uint8_t* d, const uint4* d_mpd, int* segs,
               int* segl, uint32_t* cand, int cap, unsigned long long* counter) const {
      LORB_LAUNCH(c, candidates_frame_kernel, (n * 32 + 255) / 256, 256, 0, f, P, n, d + o1,
                  (const float*)(d + o2), (const int*)(d + o3), d_mpd, th, segs, segl, cand, cap,
                  counter);
      return LORB_OK;
    }
  } l;
  Packer pk;
  l.n = n_last;
  l.P = P;
  l.valid = last_valid; l.xw = last_xw; l.oct = last_octave; l.th = th;
  l.o1 = pk.add((size_t)n_last); l.o2 = pk.add((size_t)n_last * 12); l.o3 = pk.add((size_t)n_last * 4);
  return run_search<1>(c, cur, n_last, mp_desc, mp_nobs, last_angle, pk.off, l, out_kp_for_item,
                       out_state_for_kp, n_matches, n_candidates);
}

}  // extern "C"
