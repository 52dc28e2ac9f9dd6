/*
 * lorb_cuda.h — C ABI of the B200 (sm_100a) hot-path library for LORB-SLAM.
 *
 * This is the drop-in boundary: the bodies of the reference's two stateless
 * operator classes,
 *     Matcher  (reference include/matcher.h:15-36, src/matcher.cpp)
 *     BA       (reference include/bundle_adjust.h:12-21, src/bundle_adjust.cpp)
 * flatten their Frame/MapPoint objects into the plain arrays below and call
 * these entry points.  Nothing here knows about cv::Mat, Frame or MapPoint.
 *
 * Conventions
 *  - every pointer is a HOST pointer owned by the caller for the duration of
 *    the call, unless the parameter name ends in `_dev` or the function name in
 *    `_resident` (then it refers to memory previously uploaded into the ctx);
 *  - every function returns an int status: 0 = LORB_OK, <0 = error (see enum);
 *    nothing throws or unwinds across the boundary; lorb_last_error() gives text;
 *  - one lorb_ctx per calling thread (stream + device/pinned scratch live in it);
 *    a ctx is not thread-safe, different ctxs are independent (re-entrant library);
 *  - there is NO CPU fallback: without a usable CUDA device every compute entry
 *    point returns LORB_ERR_CUDA.
 *  - descriptors are 256-bit ORB strings, 32 bytes each, row-major contiguous
 *    (reference src/ORBextractor.cpp:1114: N x 32 CV_8U).
 */
#ifndef LORB_CUDA_H
#define LORB_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LORB_DESC_BYTES 32
#define LORB_GRID_COLS 64 /* reference include/frame.h:14 FRAME_GRID_COLS */
#define LORB_GRID_ROWS 48 /* reference include/frame.h:13 FRAME_GRID_ROWS */
#define LORB_TH_HIGH 100  /* reference src/matcher.cpp:6 */
#define LORB_TH_LOW 50    /* reference src/matcher.cpp:7 */
#define LORB_HISTO_LENGTH 30 /* reference src/matcher.cpp:8 */

enum {
  LORB_OK = 0,
  LORB_ERR_ARG = -1,     /* bad argument (null pointer, negative size, index out of range) */
  LORB_ERR_CUDA = -2,    /* CUDA runtime error / no device */
  LORB_ERR_NCCL = -3,    /* NCCL error / libnccl not loadable */
  LORB_ERR_NOMEM = -4,   /* allocation failure */
  LORB_ERR_STATE = -5,   /* call sequence error (e.g. sharded call without lorb_dist_init) */
  LORB_ERR_NUMERIC = -6  /* solver broke down (non-finite step, Cholesky pivot <= 0 repeatedly) */
};

typedef struct lorb_ctx lorb_ctx; /* opaque */

/* ------------------------------------------------------------------ context */

/* Create a context bound to CUDA device `device` (cudaSetDevice ordinal). */
int lorb_ctx_create(int device, lorb_ctx** out);
int lorb_ctx_destroy(lorb_ctx* ctx);
/* Block until all work queued on the ctx stream has finished. */
int lorb_ctx_sync(lorb_ctx* ctx);
/* Raw cudaStream_t of the ctx (as void*), for callers that time with CUDA events. */
void* lorb_ctx_stream(lorb_ctx* ctx);
/* Number of kernels this ctx has launched since creation (bench "gpu_launches"). */
long long lorb_ctx_launch_count(lorb_ctx* ctx);
/* Thread-local text of the last error raised by any entry point on this thread. */
const char* lorb_last_error(void);
/* Library version string. */
const char* lorb_version(void);

/* ------------------------------------------------- brute-force Hamming match */

/* Cross-check mode.  MUTUAL is what OpenCV >= 3.4 / 4.x does (executable pin:
 * cv2 4.13 in this image): keep (q,t) iff t = argmin_t' d(q,t') and
 * q = argmin_q' d(q',t), lowest index winning ties on both sides.  It is the
 * only mode the drop-in Matcher uses and the only one with a reference behind it.
 *
 * LEGACY is EXPERIMENTAL and UNPINNED: a restatement of OpenCV 3.1's
 * batchDistance cross-check as recalled from its source (the version the
 * reference's CMakeLists.txt:10 names; not executable here, so nothing pins it):
 * for every train t take q = argmin_q' d(q',t); query q keeps the t of smallest
 * d among those (lowest t on ties).  Kept for experiments against a real 3.1
 * build; no product path selects it and no parity claim covers it. */
enum { LORB_CROSSCHECK_MUTUAL = 0, LORB_CROSSCHECK_LEGACY = 1 };

/*
 * Replaces the arithmetic of Matcher::SearchByProjection(Frame*,Frame*)
 * (reference src/matcher.cpp:13-62) and Matcher::SearchLocalPoints
 * (src/matcher.cpp:319-366): cv::BFMatcher(NORM_HAMMING, crossCheck=true)
 * .match(query, train) followed by the minDist scan (:42-47) and the
 * `distance > max(2*minDist, 30.0)` rejection (:49-56).
 *
 *   q [nq x 32], t [nt x 32]  descriptors
 *   out_q/out_t/out_dist      cross-check matches in ascending query index,
 *                             capacity >= min(nq,nt) each; dist is the integer
 *                             Hamming distance (cv::DMatch::distance is that
 *                             value as float)
 *   out_keep                  1 iff the match survives the max(2*minDist,30) test
 *   n_matches                 number of cross-check matches written
 *   n_kept                    number with out_keep==1  (the reference's return value)
 *   min_dist                  smallest distance over the matches, -1 if none
 */
int lorb_match_bf_crosscheck(lorb_ctx* ctx, const uint8_t* q, int nq, const uint8_t* t, int nt,
                             int mode, int* out_q, int* out_t, int* out_dist, uint8_t* out_keep,
                             int* n_matches, int* n_kept, int* min_dist);

/*
 * kNN-2 Hamming search with Lowe ratio + absolute threshold (north_star asks
 * for it; the reference has no caller — cv::BFMatcher::knnMatch(k=2) is the
 * oracle: neighbours ordered by (distance, train index)).
 *   out_idx/out_dist [nq x 2]  best and second best (-1 / 256 when nt < 2 or 1)
 *   out_pass [nq]              1 iff dist0 <= max_dist && dist0 < ratio * dist1
 *                              (float compare, a missing second neighbour passes)
 */
int lorb_match_knn2(lorb_ctx* ctx, const uint8_t* q, int nq, const uint8_t* t, int nt, float ratio,
                    int max_dist, int* out_idx, int* out_dist, uint8_t* out_pass);

/*
 * Keyframe-pair matching sweep (BASELINE config 5): a bank of n_kf keyframes,
 * each with n_desc descriptors, and a list of (a,b) keyframe pairs.  For every
 * pair the kernel runs the same cross-check + max(2*minDist,30) rule as
 * lorb_match_bf_crosscheck(query = bank[a], train = bank[b]) and returns
 *   out_kept[p]    number of kept matches
 *   out_matches[p] number of cross-check matches  (may be NULL)
 *   out_min[p]     minDist (-1 if no match)       (may be NULL)
 * Host-buffer form: uploads bank, runs, downloads (the e2e path).
 */
int lorb_match_sweep(lorb_ctx* ctx, const uint8_t* bank, int n_kf, int n_desc, const int* pair_a,
                     const int* pair_b, int n_pairs, int* out_kept, int* out_matches, int* out_min);

/* Two kernels compute the sweep, with identical results: LORB_SWEEP_POPC (XOR / POPC on the
 * integer pipes, operands in registers / shared memory) and LORB_SWEEP_TENSOR (tcgen05.mma
 * kind::i8 on +-32 expansions of the bit strings, distance and both tie-breaks read off the
 * int32 accumulator).  Default: tensor (environment LORB_SWEEP_IMPL=popc|tensor overrides);
 * impl = -1 restores the default.  Takes effect at the next bank / plan upload. */
enum { LORB_SWEEP_POPC = 0, LORB_SWEEP_TENSOR = 1 };
int lorb_sweep_set_impl(lorb_ctx* ctx, int impl);

/* Resident form: upload the bank once, then sweep pair lists against it. */
int lorb_bank_upload(lorb_ctx* ctx, const uint8_t* bank, int n_kf, int n_desc);
/* Pair lists / outputs are host pointers; only the bank stays in HBM. */
int lorb_match_sweep_resident(lorb_ctx* ctx, const int* pair_a, const int* pair_b, int n_pairs,
                              int* out_kept, int* out_matches, int* out_min);
/* Fully device-resident variant used to time the kernel alone: pair list is
 * uploaded once with lorb_sweep_plan_upload, each call only launches kernels;
 * results stay on the device until lorb_sweep_plan_download. */
int lorb_sweep_plan_upload(lorb_ctx* ctx, const int* pair_a, const int* pair_b, int n_pairs);
int lorb_sweep_plan_run(lorb_ctx* ctx);
/* Same plan, keyframe indices shifted by kf_base (sweeps block after block of a
 * resident bank with one uploaded pair pattern). */
int lorb_sweep_plan_run_at(lorb_ctx* ctx, int kf_base);
/* Same plan with separate bases for the two sides: pair (a, b) of the plan is keyframe pair
 * (kf_base_a + a, kf_base_b + b) of the bank (off-diagonal tiles of the keyframe grid). */
int lorb_sweep_plan_run_at2(lorb_ctx* ctx, int kf_base_a, int kf_base_b);
int lorb_sweep_plan_download(lorb_ctx* ctx, int* out_kept, int* out_matches, int* out_min);

/*
 * The whole sweep of BASELINE config 5 -- every unordered keyframe pair of the resident bank -- as
 * the reference would do it one BFMatcher call at a time (src/matcher.cpp:36-56 per pair), split
 * over the GPUs of a box the way SURVEY 8(e) row 1 says: the keyframes are cut into blocks of
 * block_kf, the upper-triangular grid of (block, block) tiles is enumerated row-major and tile t
 * belongs to rank t % world; no collective during compute.
 *   lorb_sweep_tile_count   tiles of the grid
 *   lorb_sweep_rank_tiles   the (block row, block column) of the tiles of `rank` (cap = capacity of
 *                           the two arrays, which may be NULL to query *n_out)
 *   lorb_sweep_pair_index   position of pair (a, b), a != b, in the result array: row-major upper
 *                           triangle, a * n_kf - a (a + 1) / 2 + (b - a - 1) for a < b
 *   lorb_match_sweep_all    runs the tiles of `rank` and writes out_kept[pair index] = number of kept
 *                           matches of that pair (host array of n_kf (n_kf - 1) / 2 ints); entries of
 *                           other ranks' tiles are left untouched, so a sum / gather over ranks of
 *                           zero-initialised arrays is the complete result (33.5 MB for 4096 keyframes).
 *                           *n_pairs_done = keyframe pairs this rank processed (may be NULL).
 */
long long lorb_sweep_tile_count(int n_kf, int block_kf);
int lorb_sweep_rank_tiles(int n_kf, int block_kf, int rank, int world, int cap, int* tile_bi,
                          int* tile_bj, int* n_out);
long long lorb_sweep_pair_index(int n_kf, int a, int b);
int lorb_match_sweep_all(lorb_ctx* ctx, int block_kf, int rank, int world, int* out_kept,
                         long long* n_pairs_done);

/* ------------------------------------------- projection-guided search (a5/a6) */

/* Current-frame view: what Matcher reads from a Frame through public members
 * (reference include/frame.h:76-110) plus the descriptor matrix. */
typedef struct lorb_frame_view {
  int n_kp;
  const float* kp_x;      /* mvKeysUn[i].pt.x */
  const float* kp_y;      /* mvKeysUn[i].pt.y */
  const int* kp_octave;   /* mvKeysUn[i].octave */
  const float* kp_angle;  /* mvKeysUn[i].angle (degrees) */
  const float* kp_uright; /* mvuRight[i]; <= 0 means "no stereo" */
  const uint8_t* desc;    /* [n_kp x 32] */
  /* claim state of mvpMapPoints[i] on entry: -1 = NULL, otherwise the mnObs of
   * the map point currently held (0 = held but unprotected, >0 = protected:
   * reference src/matcher.cpp:149-151, 273-275) */
  const int* kp_claim_obs;
  float min_x, max_x, min_y, max_y; /* mnMinX..mnMaxY (src/frame.cpp:79-82) */
  int n_levels;
  const float* scale_factors; /* mvScaleFactors[n_levels] */
} lorb_frame_view;

/*
 * Matcher::SearchByProjection(Frame* F, const std::set<MapPoint*>&, float th)
 * (reference src/matcher.cpp:220-316).  Points are given in the set's
 * iteration order (that order IS the semantics: earlier points claim first).
 *   active[k]    mbTrackInView && !IsBad()
 *   level[k]     mnTrackScaleLevel (must index scale_factors)
 *   mp_nobs[k]   the map point's mnObs (decides whether its claim protects)
 * Outputs:
 *   out_kp_for_point[n_pts]  keypoint assigned at that point's turn, -1 if none
 *   out_point_for_kp[n_kp]   index of the point that finally holds the keypoint
 *                            (last writer), -1 if this call did not touch it
 *   n_matches                the reference's return value (assignments made)
 *   n_candidates             optional (may be NULL): sum over points of the
 *                            GetFeaturesInArea window sizes (work measure)
 */
int lorb_search_proj_points(lorb_ctx* ctx, const lorb_frame_view* frame, int n_pts,
                            const float* proj_x, const float* proj_y, const float* proj_xr,
                            const int* level, const float* view_cos, const uint8_t* active,
                            const uint8_t* mp_desc, const int* mp_nobs, float th,
                            int* out_kp_for_point, int* out_point_for_kp, int* n_matches,
                            long long* n_candidates);

typedef struct lorb_intrinsics {
  float fx, fy, cx, cy, mbf, mb; /* Frame::fx.. (src/frame.cpp:70-77); mb = mbf/fx */
} lorb_intrinsics;

/*
 * Matcher::SearchByProjection(Frame* Cur, Frame* Last, float th)
 * (reference src/matcher.cpp:64-218): project Last's map points with Cur's
 * pose, octave-dependent window, best Hamming <= TH_HIGH, rotation histogram.
 *   tcw_cur/tcw_last [16]  row-major 4x4 float mTcw
 *   last_valid[i]          mvpMapPoints[i] != NULL && !mvbOutlier[i]
 *   last_xw [n_last x 3]   MapPoint::GetPos()
 *   last_octave[i]         LastFrame->mvKeys[i].octave
 *   last_angle[i]          LastFrame->mvKeysUn[i].angle
 * Outputs:
 *   out_kp_for_item[n_last]  keypoint chosen at that item's turn (-1 none)
 *   out_state_for_kp[n_kp]   -1 untouched, -2 set to NULL by the rotation
 *                            check, >=0 index of the Last item finally held
 *   n_matches                the reference's return value
 */
int lorb_search_proj_frame(lorb_ctx* ctx, const lorb_frame_view* cur, const float* tcw_cur,
                           const float* tcw_last, const lorb_intrinsics* K, int n_last,
                           const uint8_t* last_valid, const float* last_xw, const int* last_octave,
                           const float* last_angle, const uint8_t* mp_desc, const int* mp_nobs,
                           float th, int* out_kp_for_item, int* out_state_for_kp, int* n_matches,
                           long long* n_candidates);

/*
 * Frame::IsInFrustum (reference src/frame.cpp:425-494) with
 * MapPoint::PredictScale (src/map_point.cpp:267-284) for n map points at once —
 * the step that fills MapPoint::mTrack* before the local-map search
 * (src/visual_odometry.cpp:176-195; SURVEY 8(f) rank 1).
 *   tcw [16]      row-major float mTcw
 *   ow [3]        camera centre = translation column of mTcw.inv() (the caller
 *                 computes it with the same cv::Mat::inv() the reference uses)
 *   xw, normal    [n x 3] GetPos() / GetNormal()
 *   min_dist/max_dist [n]  mfMinDistance / mfMaxDistance (0.8 / 1.2 applied inside)
 *   log_scale_factor       Frame::mfLogScaleFactor, n_levels = mnScaleLevels
 * Outputs (what IsInFrustum leaves in the MapPoint): in_view (mbTrackInView),
 * proj_x/proj_y/proj_xr, level (mnTrackScaleLevel), view_cos.  Entries of
 * points that are not in view are left untouched except in_view = 0.
 */
int lorb_frustum_project(lorb_ctx* ctx, const float* tcw, const float* ow, const lorb_intrinsics* K,
                         float min_x, float max_x, float min_y, float max_y, int n, const float* xw,
                         const float* normal, const float* min_dist, const float* max_dist,
                         float viewing_cos_limit, float log_scale_factor, int n_levels,
                         uint8_t* in_view, float* proj_x, float* proj_y, float* proj_xr, int* level,
                         float* view_cos);

/*
 * Frame::ComputeStereoMatches (reference src/frame.cpp:125-333; SURVEY 8(f) rank 2): for every
 * left keypoint, the best right keypoint in its row band by Hamming distance (octave within
 * +-1, disparity in [0, mbf/mb]), 11x11 SAD refinement over 11 shifts at the keypoint's pyramid
 * level with a parabola fit, then removal of matches whose SAD is >= 1.5*1.4*median.
 *   left / right       image pyramids as ORBextractor::mvImagePyramid holds them
 *                      (reference include/ORBextractor.h:85): 8-bit, data[l] -> pixel (0,0),
 *                      step[l] bytes between rows, width[l] x height[l]
 *   scale_factors / inv_scale_factors [n_levels]   Frame::mvScaleFactors / mvInvScaleFactors
 *   mbf, mb            Frame::mbf, Frame::mb
 *   lx, ly, loct, ldesc   left  mvKeys[i].pt.x / .pt.y / .octave, mDescriptors rows
 *   rx, ry, roct, rdesc   right mvKeysRight / mDescriptorsRight
 * Outputs: out_uright[n_left] (mvuRight), out_depth[n_left] (mvDepth), -1 where unmatched;
 * n_matched = matches left after the outlier step (may be NULL).
 * A keypoint whose correlation patch would leave its level image is left unmatched (in the
 * reference cv::Mat::rowRange/colRange would throw there).
 */
typedef struct lorb_pyramid_view {
  int n_levels;
  const int* width;          /* [n_levels] */
  const int* height;         /* [n_levels] */
  const int* step;           /* [n_levels] bytes per row */
  const uint8_t* const* data;/* [n_levels] host pointers */
} lorb_pyramid_view;

int lorb_stereo_matches(lorb_ctx* ctx, const lorb_pyramid_view* left, const lorb_pyramid_view* right,
                        int n_levels, const float* scale_factors, const float* inv_scale_factors,
                        float mbf, float mb, int n_left, const float* lx, const float* ly,
                        const int* loct, const uint8_t* ldesc, int n_right, const float* rx,
                        const float* ry, const int* roct, const uint8_t* rdesc, float* out_uright,
                        float* out_depth, int* n_matched);

/*
 * Orientation and steered-BRIEF stages of ORBextractor (reference src/ORBextractor.cpp:79-149 =
 * IC_Angle + computeOrbDescriptor, driven by computeOrientation :487-494 and computeDescriptors
 * :1078-1085; SURVEY 8(f) rank 5) for keypoints given in the coordinates of their pyramid level.
 *   raw        the image pyramid (ORBextractor::mvImagePyramid): orientation reads it (:1105)
 *   blurred    the same levels after cv::GaussianBlur(7x7, sigma 2) (:1131-1132): the descriptor
 *              reads it
 *   pattern    [512 x 2] int, the sampling pattern the ORBextractor constructor holds
 *              (ORBextractor::pattern, :464-467); every point inside radius 19
 *   kx, ky     keypoint position in level coordinates (before the scale-back of :1142-1147),
 *              klevel its pyramid level; each keypoint at least EDGE_THRESHOLD = 19 px inside its
 *              level, which the extractor guarantees (:76, :820-823) -- LORB_ERR_ARG otherwise
 *   angle_in   NULL: compute the orientation (out_angle receives KeyPoint::angle, degrees);
 *              non-NULL: describe with these angles (raw may then be NULL)
 *   out_desc   [n_kp x 32] descriptor rows (Frame::mDescriptors layout, row a1 of SURVEY 8(a))
 * cos/sin of the angle carry the bits of the host libm the reference links (glibc >= 2.28 on an
 * FMA-capable x86-64), see lorb_slam_b200/csrc/libm_sincosf.cuh.
 */
int lorb_orb_describe(lorb_ctx* ctx, const lorb_pyramid_view* raw, const lorb_pyramid_view* blurred,
                      int n_levels, const int* pattern, int n_kp, const float* kx, const float* ky,
                      const int* klevel, const float* angle_in, float* out_angle, uint8_t* out_desc);

/*
 * ORBextractor::operator() (reference src/ORBextractor.cpp:1087-1151; SURVEY 8(f) rank 5): scale
 * pyramid (ComputePyramid :1157-1184, cv::resize INTER_LINEAR level from level), FAST-9 with
 * non-maximum suppression per ~30x30 cell at iniThFAST, else minThFAST (ComputeKeyPointsOctTree
 * :799-880), quadtree selection of about nfeatures keypoints (DistributeOctTree :554-797),
 * orientation, cv::GaussianBlur(7x7, 2) and the steered-BRIEF descriptors, keypoints scaled back
 * to level-0 coordinates.  The OpenCV operations follow OpenCV 4.x (pinned to cv2 4.13; the
 * reference's CMakeLists.txt:10 names 3.1).  The quadtree's tie-break among equally filled nodes
 * (the reference compares node addresses, :695) is creation order: last created first.
 *   params       the ORBextractor constructor arguments (:412-415)
 *   pattern      as lorb_orb_describe
 *   cap          capacity of the output arrays (lorb_orb_max_keypoints gives the bound; the extractor
 *                usually returns slightly more than nfeatures); LORB_ERR_ARG if it is too small
 * Outputs in the reference's order (level by level, nodes in list order): KeyPoint pt.x, pt.y,
 * octave, angle, response (may be NULL), size (may be NULL), descriptor rows; *n_out keypoints.
 * raw_levels (may be NULL): [nlevels] host buffers of level_w*level_h bytes (lorb_orb_level_sizes)
 * that receive ORBextractor::mvImagePyramid, which Frame::ComputeStereoMatches reads.
 */
typedef struct lorb_orb_params {
  int nfeatures;
  float scale_factor;
  int nlevels;
  int ini_th_fast;
  int min_th_fast;
} lorb_orb_params;

int lorb_orb_extract(lorb_ctx* ctx, const uint8_t* image, int width, int height, int step,
                     const lorb_orb_params* params, const int* pattern, int cap, float* kp_x,
                     float* kp_y, int* kp_octave, float* kp_angle, float* kp_response, float* kp_size,
                     uint8_t* desc, int* n_out, uint8_t* const* raw_levels);

/*
 * The device work of Frame::Frame(imgLeft, imgRight, camera) (reference src/frame.cpp:17-68) in one
 * call: ORBextractor::operator() on both images (:42-46) and Frame::ComputeStereoMatches (:49) on
 * the pyramids, keypoints and descriptors left on the device by the two extractions.  Results are
 * those of lorb_orb_extract(left), lorb_orb_extract(right) and lorb_stereo_matches on their outputs.
 *   out_left / out_right  keypoint arrays of capacity cap (response, size, raw_levels may be NULL);
 *                         n receives the keypoint count
 *   mbf, mb               Frame::mbf, Frame::mb
 *   out_uright, out_depth [cap] mvuRight / mvDepth of the left keypoints (-1 where unmatched)
 */
typedef struct lorb_orb_keypoints {
  int n;
  float* x;
  float* y;
  int* octave;
  float* angle;
  float* response;
  float* size;
  uint8_t* desc;              /* [cap x 32] */
  uint8_t* const* raw_levels; /* [nlevels] host buffers for mvImagePyramid, or NULL */
} lorb_orb_keypoints;

int lorb_stereo_frame(lorb_ctx* ctx, const uint8_t* left, const uint8_t* right, int width, int height,
                      int step_left, int step_right, const lorb_orb_params* params, const int* pattern,
                      float mbf, float mb, int cap, lorb_orb_keypoints* out_left,
                      lorb_orb_keypoints* out_right, float* out_uright, float* out_depth, int* n_matched);

/*
 * ORBextractor::DistributeOctTree (:554-797) on its own (one CTA on the device: what lorb_orb_extract
 * runs per level between the FAST and the descriptor kernels): from the candidate keypoints of one
 * level (coordinates relative to min_x / min_y, in the order the detection loop produced them) pick
 * about n_features of them, spread over the image by a quadtree.  out_index [lorb_orb_max_keypoints or
 * n_keys] receives the indices of the chosen keypoints in the reference's output order, *n_out their
 * number.  Equal-size tie-break: see lorb_orb_extract.  Keys must be integer pixels below 4096 with
 * integer responses below 256, which is what the FAST stage produces.
 */
int lorb_orb_distribute(lorb_ctx* ctx, int n_keys, const float* x, const float* y,
                            const float* response, int min_x, int max_x, int min_y, int max_y,
                            int n_features, int* out_index, int* n_out);

/* Upper bound of the number of keypoints the extractor can return for this frame size: usually a few
 * more than nfeatures (each level stops at >= its share), but a wide level with a small share keeps
 * 4 nodes per initial quadtree column whatever its budget (src/ORBextractor.cpp:566-594, 610-672).
 * Size the output arrays of lorb_orb_extract / lorb_stereo_frame with it. */
int lorb_orb_max_keypoints(const lorb_orb_params* params, int width, int height, int* max_keypoints);

/* Level geometry of the extractor: sizes of the pyramid levels (:1161-1163), mnFeaturesPerLevel
 * (:448-461, may be NULL) and mvScaleFactor (:428-436, may be NULL). */
int lorb_orb_level_sizes(const lorb_orb_params* params, int width, int height, int* level_w,
                         int* level_h, int* n_features_per_level, float* scale_factors);

/*
 * The intermediate products of the extractor, any of them optional (NULL):
 *   raw_levels / blur_levels  [nlevels] host buffers of level_w*level_h bytes: mvImagePyramid and
 *                             its blurred copy (what Frame::ComputeStereoMatches and
 *                             lorb_orb_describe take)
 *   cand_*                    the keypoints handed to DistributeOctTree (vToDistributeKeys :813),
 *                             level after level in the reference's order (cell row, cell column,
 *                             row-major inside the cell), coordinates relative to the 16-px
 *                             margin; cand_level_start [nlevels + 1]
 */
int lorb_orb_stages(lorb_ctx* ctx, const uint8_t* image, int width, int height, int step,
                    const lorb_orb_params* params, uint8_t* const* raw_levels,
                    uint8_t* const* blur_levels, int cand_cap, float* cand_x, float* cand_y,
                    float* cand_response, int* cand_level_start);

/* ORBextractor::umax (:469-482): half widths of the rows 0..15 of the orientation disc. */
void lorb_orb_umax(int* umax16);

/* Arithmetic pins for the tests: the device's sinf / cosf (host-libm bits) of a[i] and
 * cv::fastAtan2(a[i], b[i]). */
int lorb_orb_selftest(lorb_ctx* ctx, int n, const float* a, const float* b, float* out_sin,
                      float* out_cos, float* out_atan2);

/*
 * MapPoint::ComputeDescriptor (reference src/map_point.cpp:69-129) for a batch
 * of map points (SURVEY 8(f) rank 4): point k owns the observation descriptors
 * desc[offsets[k] .. offsets[k+1]) (in the iteration order of its observation
 * map, bad frames already dropped); all pairwise Hamming distances, per row the
 * element (int)(0.5*(m-1)) of the sorted row, the row with the smallest such
 * median wins (first one on ties).  At most 128 observations per point.
 *   out_best[k]    index (0-based inside the point's slice) of the chosen
 *                  descriptor, -1 for a point without observations
 *   out_median[k]  its median distance (may be NULL)
 */
int lorb_compute_descriptors(lorb_ctx* ctx, int n_points, const int* offsets, const uint8_t* desc,
                             int* out_best, int* out_median);

/* ------------------------------------------------------- bundle adjustment */

/* Solver options: the Ceres Solver::Options fields that shape the LM
 * trajectory (SURVEY §8(a) row a12).  lorb_ba_default_options fills Ceres'
 * defaults; the reference sets nothing but DENSE_SCHUR
 * (src/bundle_adjust.cpp:189-191, 308-310). */
typedef struct lorb_ba_options {
  int max_num_iterations;           /* 50 */
  int jacobi_scaling;               /* 1 */
  int max_consecutive_invalid_steps;/* 5 */
  int reserved0;
  double function_tolerance;        /* 1e-6 */
  double gradient_tolerance;        /* 1e-10 */
  double parameter_tolerance;       /* 1e-8 */
  double initial_trust_region_radius; /* 1e4 */
  double max_trust_region_radius;   /* 1e16 */
  double min_trust_region_radius;   /* 1e-32 */
  double min_relative_decrease;     /* 1e-3 */
  double min_lm_diagonal;           /* 1e-6 */
  double max_lm_diagonal;           /* 1e32 */
} lorb_ba_options;

enum {
  LORB_BA_NO_CONVERGENCE = 0,   /* iteration budget exhausted */
  LORB_BA_CONV_FUNCTION = 1,
  LORB_BA_CONV_GRADIENT = 2,
  LORB_BA_CONV_PARAMETER = 3,
  LORB_BA_CONV_RADIUS = 4,      /* trust region radius below minimum */
  LORB_BA_FAILURE = 5           /* too many consecutive invalid steps */
};

typedef struct lorb_ba_summary {
  double initial_cost;  /* 1/2 sum rho(|r|^2) at the input (rho = identity unless a loss is set) */
  double final_cost;
  double final_radius;
  double final_gradient_max_norm;
  int iterations;       /* LM steps attempted (Ceres' iteration index at exit) */
  int num_successful_steps;
  int num_unsuccessful_steps;
  int termination;      /* LORB_BA_* */
} lorb_ba_summary;

void lorb_ba_default_options(lorb_ba_options* opt);

/*
 * Robust loss of every BA solve on a ctx (beyond the reference, which passes no loss to
 * AddResidualBlock; Ceres LossFunction semantics).  With s = |r|^2 of one observation's 2-vector
 * residual, a = scale, b = a^2, c = 1/b:
 *   LORB_LOSS_TRIVIAL   rho(s) = s                      (default: plain least squares, the reference)
 *   LORB_LOSS_HUBER     rho(s) = s (s <= b), 2 a sqrt(s) - b (s > b)        (ceres::HuberLoss)
 *   LORB_LOSS_SOFTLONE  rho(s) = 2 b (sqrt(1 + s c) - 1)                    (ceres::SoftLOneLoss)
 *   LORB_LOSS_CAUCHY    rho(s) = b log(1 + s c)                             (ceres::CauchyLoss)
 * The solvers minimise 1/2 sum rho(s); residuals and Jacobians are scaled by sqrt(rho'(s)) at the
 * point of linearisation (Ceres' Corrector, whose curvature term vanishes for these losses), so the
 * gradient, the normal equations, the Jacobi scaling and the model decrease are those of the
 * corrected problem.  Summary costs and gradient norms are those of the robust problem.
 * lorb_ba_set_loss(ctx, NULL) restores the trivial loss.  It returns < 0 and leaves the ctx as it
 * was for an unknown kind, or for a scale that is not finite and > 0 when the kind is not trivial
 * (the trivial loss ignores the scale).  The setting holds until the next call on that ctx.
 */
enum { LORB_LOSS_TRIVIAL = 0, LORB_LOSS_HUBER = 1, LORB_LOSS_SOFTLONE = 2, LORB_LOSS_CAUCHY = 3 };
typedef struct lorb_ba_loss {
  int kind;     /* LORB_LOSS_* */
  int reserved;
  double scale; /* a > 0, in pixels */
} lorb_ba_loss;
int lorb_ba_set_loss(lorb_ctx* ctx, const lorb_ba_loss* loss);
int lorb_ba_get_loss(lorb_ctx* ctx, lorb_ba_loss* loss);

/*
 * BA::ProjectPoseOptimization (reference src/bundle_adjust.cpp:158-202):
 * 6-dof pose (angle-axis R, translation T) of one frame against fixed 3-D
 * points, PoseCost residuals (src/bundle_adjust.cpp:22-64 — including its use
 * of fx for the v coordinate, :51).
 *   xw [n x 3] float   MapPoint::GetPos()
 *   uv [n x 2] float   Frame::GetKp2d(i)
 *   K = {fx, fy, cx, cy} float (fy is unused by PoseCost; kept for symmetry)
 *   rt [6] double in/out: (R0,R1,R2,T0,T1,T2)
 * Minimises with the ctx's robust loss (lorb_ba_set_loss).
 */
int lorb_ba_pose_only(lorb_ctx* ctx, int n, const float* xw, const float* uv, const float* K,
                      double* rt, const lorb_ba_options* opt, lorb_ba_summary* summary);

/*
 * Pose-only BA with outlier rounds (beyond the reference; ORB-SLAM2's Optimizer::PoseOptimization),
 * for a batch of frames.  Frame f owns observations [obs_off[f], obs_off[f+1]) of xw / uv / info
 * and the pose rt[6f .. 6f+6).
 *   obs_off [n_frames+1] int, obs_off[0] = 0, non-decreasing; O = obs_off[n_frames]
 *   xw [O x 3], uv [O x 2] float    as lorb_ba_pose_only
 *   info [O] float or NULL          per-observation weight w (NULL = 1), e.g. 1 / sigma^2 of the octave
 *   K = {fx, fy, cx, cy} float      shared by every frame
 *   rt [n_frames x 6] double in/out
 *   out_inlier [O]                  1 = inlier, 0 = outlier
 *   out_chi2 [O] or NULL            w |r|^2 of each observation
 *   n_inliers [n_frames]            number of inliers of each frame
 *   rounds_run [n_frames] or NULL   rounds each frame ran
 *   summaries [n_frames x n_rounds] or NULL   LM summary of every round of every frame
 * Semantics:
 * - The residual is PoseCost, with its fx-for-v quirk (ba_math.cuh::obs_eval, as lorb_ba_pose_only).
 * - A weighted observation is the residual sqrt(w) r.  The ctx's robust loss (lorb_ba_set_loss)
 *   applies to s = w |r|^2, as in Ceres with a scaled cost function and a LossFunction.  With a loss
 *   set, its scale is therefore in whitened units.
 * - Each round is one full solve under the Ceres contract of lorb_ba_pose_only, with opt as its budget:
 *   - it starts from the input pose, as ORB-SLAM2 resets to pFrame->mTcw every round;
 *   - it has a fresh trust region and Jacobi scaling;
 *   - it runs over the observations flagged inlier at its start.  Round 0 starts with all of them.
 * - After a round, every observation of the frame is classified at that round's pose: inlier iff
 *   w |r|^2 <= chi2.  This chi^2 is the unrobustified one.
 * - If fewer than 3 observations are inliers at the start of a round, that round and the rest are
 *   skipped.
 * - rt, out_inlier, out_chi2 and n_inliers always describe the returned pose.  That is the pose after
 *   the last round that ran, or the input pose with its classification if no round ran.
 * - Summary slots of rounds that did not run are zero-filled.
 * - Refused with LORB_ERR_ARG, before any device work: bad offsets, a weight that is not finite and
 *   > 0, or an out-of-range rounds field.
 * - n_frames = 0 is a no-op.
 * One CTA per frame, all rounds of all frames in one launch; a frame's result is bit-identical whether
 * it is solved alone or in a batch.
 */
typedef struct lorb_ba_pose_rounds {
  int n_rounds;       /* 4     (1..16) */
  int robust_rounds;  /* 3     rounds [0, robust_rounds) use the ctx's loss, later rounds plain least squares (0..n_rounds) */
  double chi2;        /* 5.991 chi-square threshold on w*|r|^2 (finite, > 0) */
} lorb_ba_pose_rounds;
void lorb_ba_default_pose_rounds(lorb_ba_pose_rounds* r);

int lorb_ba_pose_rounds_batched(lorb_ctx* ctx, int n_frames, const int* obs_off /* [n_frames+1] */,
    const float* xw /* [O x 3] */, const float* uv /* [O x 2] */, const float* info /* [O] or NULL = 1 */,
    const float* K /* fx fy cx cy, shared */, double* rt /* [n_frames x 6] in/out */,
    const lorb_ba_pose_rounds* rounds, const lorb_ba_options* opt /* per round */,
    uint8_t* out_inlier /* [O] */, double* out_chi2 /* [O] or NULL */, int* n_inliers /* [n_frames] */,
    int* rounds_run /* [n_frames] or NULL */, lorb_ba_summary* summaries /* [n_frames x n_rounds] or NULL */);

/*
 * BA::LocalPoseOptimization (reference src/bundle_adjust.cpp:207-330).
 *   cams [C x 6] double in/out   (w0,w1,w2,t0,t1,t2) per window frame (:250-255)
 *   pts  [P x 3] double in/out   (:262-264)
 *   obs_*  [O]   PoseMPCost residuals (point, pose) (:116-151, :299-300)
 *   fix_*  [F]   MPCost residuals: point seen from an out-of-window frame whose
 *                float pose fix_rt[f] = (r0,r1,r2,t0,t1,t2) stays constant
 *                (:68-113, :288-289)
 *   K = {fx, fy, cx, cy} of pCurrFrame->mpCamera
 * No parameter block is held constant (the reference holds none).
 * Minimises with the ctx's robust loss (lorb_ba_set_loss), in-window and fixed
 * observations alike.
 */
int lorb_ba_local(lorb_ctx* ctx, int C, double* cams, int P, double* pts, int O, const int* obs_cam,
                  const int* obs_pt, const float* obs_uv, int F, const int* fix_pt,
                  const float* fix_uv, const float* fix_rt, const float* K,
                  const lorb_ba_options* opt, lorb_ba_summary* summary);

/*
 * lorb_ba_local for one rank of a point-sharded problem (BASELINE config 5 on several GPUs): the
 * arrays hold THIS RANK'S points with all their observations (lorb_shard_range / the natural layout
 * of a distributed map) and every camera; a collective call over the communicator of lorb_dist_init.
 * On return cams holds all C cameras (identical on every rank), pts this rank's points.
 * Every rank must have set the same robust loss (lorb_ba_set_loss) on its ctx.
 */
int lorb_ba_local_shard(lorb_ctx* ctx, int C, double* cams, int P, double* pts, int O, const int* obs_cam,
                        const int* obs_pt, const float* obs_uv, int F, const int* fix_pt,
                        const float* fix_uv, const float* fix_rt, const float* K,
                        const lorb_ba_options* opt, lorb_ba_summary* summary);

/*
 * Batched independent windows (BASELINE config 4).  Window w owns
 *   cams[cam_off[w] .. cam_off[w+1]), pts[pt_off[w] .. pt_off[w+1]),
 *   obs[obs_off[w] .. obs_off[w+1])  with obs_cam / obs_pt LOCAL to the window,
 *   fixed observations [fix_off[w] .. fix_off[w+1]) likewise (fix_off may be
 *   NULL when there are none).
 * Every window runs its own LM loop (own trust region, own termination), all
 * with the ctx's robust loss (lorb_ba_set_loss).
 */
int lorb_ba_local_batched(lorb_ctx* ctx, int n_windows, const int* cam_off, double* cams,
                          const int* pt_off, double* pts, const int* obs_off, const int* obs_cam,
                          const int* obs_pt, const float* obs_uv, const int* fix_off,
                          const int* fix_pt, const float* fix_uv, const float* fix_rt,
                          const float* K, const lorb_ba_options* opt, lorb_ba_summary* summaries);

/*
 * Local BA with outlier rounds (beyond the reference; ORB-SLAM2's Optimizer::LocalBundleAdjustment),
 * for a batch of windows in the layout of lorb_ba_local_batched.
 *   obs_w [O] float or NULL         per-observation weight w of the in-window observations (NULL = 1),
 *                                   e.g. 1 / sigma^2 of the keypoint's octave; indexed like obs_cam
 *   fix_w [F] float or NULL         the same for the fixed observations; indexed like fix_pt
 *   rounds, opt [n_rounds]          round r runs under opt[r]
 *   obs_inlier [O], fix_inlier [F]  1 = inlier, 0 = outlier
 *   obs_chi2 [O], fix_chi2 [F]      w |r|^2 of each observation (either may be NULL)
 *   n_inliers [n_windows]           in-window + fixed inliers of each window
 *   summaries [n_windows x n_rounds] or NULL   LM summary of every round of every window
 * Semantics:
 * - Residuals: PoseMPCost for in-window observations, MPCost with the float pose for fixed observers,
 *   as lorb_ba_local.
 * - A weighted observation is the residual sqrt(w) r.  The ctx's robust loss (lorb_ba_set_loss)
 *   applies to s = w |r|^2, so its scale is in whitened units.
 * - Each round is one full LM solve under opt[r], with a fresh trust region and Jacobi scaling taken
 *   at the round's start from the weighted Jacobian of its inliers:
 *   - it runs over the observations flagged inlier at its start.  Round 0 runs over all of them;
 *   - rounds [0, robust_rounds) use the ctx's loss, later rounds plain least squares;
 *   - it starts from the previous round's result, not from the input, as ORB-SLAM2's
 *     LocalBundleAdjustment continues where its first optimisation stopped.
 * - A camera or point with no inlier observation keeps its value bit for bit through the round.  It
 *   stays in |x| of the parameter-tolerance test (Ceres would drop such a block from its program;
 *   only that test differs).
 * - After each round, every observation of the window (in-window and fixed, inlier or not) is
 *   classified at that round's parameters: inlier iff w |r|^2 <= chi2 and, with depth_check, the
 *   point's depth in the observing camera is > 0.  This chi^2 is the unrobustified one.
 * - A window with no inliers still runs its round: it stops at its first gradient test
 *   (LORB_BA_CONV_GRADIENT, 0 iterations).
 * - cams, pts, the flags, chi^2 values and counts describe the returned parameters, i.e. the
 *   classification after the last round.  Flags and chi^2 are in the caller's order.
 * - Every window runs its own LM loop in every round; the rounds run in lockstep across the batch.
 * - Refused with LORB_ERR_ARG, before any device work and with the outputs untouched: whatever
 *   lorb_ba_local_batched refuses, a weight that is not finite and > 0, an out-of-range rounds field,
 *   opt NULL, or a NULL inlier array for a side (in-window / fixed) with observations.
 * - n_windows = 0 is a no-op.
 * Not sharded: the rounds run on one GPU.
 */
typedef struct lorb_ba_local_rounds {
  int n_rounds;       /* 2     (1..16) */
  int robust_rounds;  /* 1     rounds [0, robust_rounds) use the ctx's loss, later rounds plain least squares (0..n_rounds) */
  double chi2;        /* 5.991 threshold on w*|r|^2 (finite, > 0) */
  int depth_check;    /* 1     0/1: an observation whose point is not in front of its camera (z <= 0) is an outlier */
  int reserved;
} lorb_ba_local_rounds;
/* ORB-SLAM2's LocalBundleAdjustment settings; opt2 (may be NULL) receives two lorb_ba_default_options
 * with max_num_iterations 5 and 10. */
void lorb_ba_default_local_rounds(lorb_ba_local_rounds* r, lorb_ba_options* opt2);

int lorb_ba_local_rounds_batched(lorb_ctx* ctx, int n_windows, const int* cam_off, double* cams,
    const int* pt_off, double* pts, const int* obs_off, const int* obs_cam, const int* obs_pt,
    const float* obs_uv, const float* obs_w /* [O] or NULL = 1 */,
    const int* fix_off /* or NULL */, const int* fix_pt, const float* fix_uv, const float* fix_rt,
    const float* fix_w /* [F] or NULL = 1 */, const float* K,
    const lorb_ba_local_rounds* rounds, const lorb_ba_options* opt /* [n_rounds], round r runs under opt[r] */,
    uint8_t* obs_inlier /* [O] */, double* obs_chi2 /* [O] or NULL */,
    uint8_t* fix_inlier /* [F] */, double* fix_chi2 /* [F] or NULL */,
    int* n_inliers /* [n_windows], in-window + fixed */, lorb_ba_summary* summaries /* [n_windows x n_rounds] or NULL */);
/* The same for one window, in the argument layout of lorb_ba_local (the name lorb_ba_local_rounds is
 * the settings type). */
int lorb_ba_local_rounds_single(lorb_ctx* ctx, int C, double* cams, int P, double* pts, int O,
    const int* obs_cam, const int* obs_pt, const float* obs_uv, const float* obs_w, int F,
    const int* fix_pt, const float* fix_uv, const float* fix_rt, const float* fix_w, const float* K,
    const lorb_ba_local_rounds* rounds, const lorb_ba_options* opt,
    uint8_t* obs_inlier, double* obs_chi2, uint8_t* fix_inlier, double* fix_chi2,
    int* n_inliers /* [1] */, lorb_ba_summary* summaries /* [n_rounds] or NULL */);

/*
 * Pose from 2D-3D matches without a prior: batched P3P RANSAC (beyond the reference: the pose half of
 * VisualOdometry::EstimatePosePnP, and of ORB-SLAM2's per-candidate relocalisation before PoseOptimization).
 * Problem b owns correspondences [corr_off[b], corr_off[b+1]) of xw / uv / info.  Problems are independent;
 * no input pose is read.
 *   corr_off [n_problems+1] int, corr_off[0] = 0, non-decreasing; O = corr_off[n_problems]
 *   xw [O x 3], uv [O x 2] float    world point and its keypoint
 *   info [O] float or NULL          per-correspondence weight w (NULL = 1), e.g. 1 / sigma^2 of the octave
 *   K = {fx, fy, cx, cy} float      shared by every problem
 *   seeds [n_problems] or NULL      sampler seed of each problem (NULL: the seed of problem b is b)
 *   out_rt [n_problems x 6] double  (w0, w1, w2, t0, t1, t2): angle-axis R(w) as ba_math.cuh::cam_rotation,
 *                                   x_c = R(w) X + t, so it feeds lorb_ba_pose_rounds_batched directly
 *   best_hyp [n_problems]           the selected hypothesis h, or -1
 *   n_inliers [n_problems]          its inlier count
 *   out_inlier [O]                  1 = inlier of the selected hypothesis, 0 otherwise
 *   out_chi2 [O] or NULL            w |r|^2 at the selected hypothesis (+inf behind the camera)
 * Semantics:
 * - Camera model: the true pinhole, u = fx x/z + cx, v = fy y/z + cy with (x, y, z) = R(w) X + t.  This is
 *   not PoseCost's fx-for-v quirk (reference src/bundle_adjust.cpp:51); the two agree when fx = fy.
 * - Sampler (counter-based): with sm(x) = SplitMix64 (x += 0x9E3779B97F4A7C15;
 *   z = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9; z = (z ^ (z >> 27)) * 0x94D049BB133111EB; return z ^ (z >> 31)),
 *   draw k of hypothesis h is r = sm(seed ^ sm(((uint64)h << 8) | k)) and names correspondence
 *   ((r >> 32) * n) >> 32 of the problem's n.  Draws k = 0, 1, ... that repeat an index already taken are
 *   skipped until 4 distinct indices are taken; if k passes 255 first, the hypothesis is invalid.  The first
 *   three indices are the P3P triple, the fourth the check point.
 * - Hypothesis: a closed-form P3P solve (Lambda Twist, Persson & Nordberg 2018) in fp64 on the triple's
 *   unit bearings normalise((u - cx) / fx, (v - cy) / fy, 1).  Solutions that put any of the three sample
 *   points at depth <= 0 are dropped.  Of the rest, the hypothesis is the solution with the smallest squared
 *   pixel error at the check point, among those that put the check point at depth > 0; ties keep the
 *   earlier solution in solver order.  A degenerate triple (collinear world points or coincident bearings,
 *   tolerances in csrc/pnp_math.cuh) has no solution; no solution makes the hypothesis invalid.
 * - Score: the inlier count, z > 0 and w |r|^2 <= chi2 over all of the problem's correspondences.  The best
 *   hypothesis has the largest count among the valid ones; ties go to the lowest h.  best_hyp[b] = -1 if the
 *   problem has fewer than 4 correspondences or no valid hypothesis: then rt is zeros, flags are 0, chi^2
 *   is +inf and the count is 0.
 * - out_rt, out_inlier, out_chi2 and n_inliers describe the best hypothesis.  The sampler-to-score arithmetic
 *   is IEEE correctly rounded (no contraction), so a problem's result depends only on its correspondences,
 *   its seed and params, and is bit-identical alone or in a batch when seeds are given.
 * - Refused with LORB_ERR_ARG, before any device work and with every output untouched: bad offsets, a weight
 *   that is not finite and > 0, fx or fy not finite and > 0, an out-of-range params field, or a NULL
 *   required pointer (out_inlier may be NULL only when O = 0).
 * - n_problems = 0 is a no-op.
 * Two launches on the ctx stream (scoring, then the finalize pass), one upload and one download.
 */
typedef struct lorb_pnp_ransac {
  int n_hypotheses;   /* 300   (1..65536) hypotheses drawn and scored per problem */
  int reserved;
  double chi2;        /* 5.991 inlier iff w*|r|^2 <= chi2 (finite, > 0) */
} lorb_pnp_ransac;
void lorb_default_pnp_ransac(lorb_pnp_ransac* p);

int lorb_pnp_ransac_batched(lorb_ctx* ctx, int n_problems, const int* corr_off /* [n_problems+1] */,
    const float* xw /* [O x 3] */, const float* uv /* [O x 2] */, const float* info /* [O] or NULL = 1 */,
    const float* K /* fx fy cx cy, shared */, const uint64_t* seeds /* [n_problems] or NULL: seed of b = b */,
    const lorb_pnp_ransac* params,
    double* out_rt /* [n_problems x 6] */, int* best_hyp /* [n_problems] */, int* n_inliers /* [n_problems] */,
    uint8_t* out_inlier /* [O] */, double* out_chi2 /* [O] or NULL */);

/* Team size of the library's host-side staging loops (OpenMP) for the calling thread.  Launchers
 * such as torchrun export OMP_NUM_THREADS=1 to every rank; a host that knows how many ranks share
 * the box hands each its share of the cores here.  (omp_set_num_threads on the process's OpenMP
 * runtime: host code that changes the team size for its own loops changes it for the library.) */
int lorb_set_host_threads(int n);

/* Device-resident local BA problem, for timing the solver without the
 * host<->device copies and for the multi-GPU sharded solve. */
typedef struct lorb_ba_problem lorb_ba_problem; /* opaque */
int lorb_ba_problem_create(lorb_ctx* ctx, int C, const double* cams, int P, const double* pts, int O,
                           const int* obs_cam, const int* obs_pt, const float* obs_uv, int F,
                           const int* fix_pt, const float* fix_uv, const float* fix_rt,
                           const float* K, lorb_ba_problem** out);
/* Batched form of the above: n_windows independent windows in the offset-array
 * layout of lorb_ba_local_batched; lorb_ba_problem_solve then fills
 * summary[0..n_windows) and lorb_ba_problem_download returns the concatenated
 * cameras / points. */
int lorb_ba_problem_create_batched(lorb_ctx* ctx, int n_windows, const int* cam_off,
                                   const double* cams, const int* pt_off, const double* pts,
                                   const int* obs_off, const int* obs_cam, const int* obs_pt,
                                   const float* obs_uv, const int* fix_off, const int* fix_pt,
                                   const float* fix_uv, const float* fix_rt, const float* K,
                                   lorb_ba_problem** out);
/*
 * Sharding helpers of the multi-GPU paths (SURVEY 8(e)), so that a C++ host need not restate them:
 *   lorb_shard_range   contiguous [lo, hi) slice of n units (batched windows) owned by `rank`: sizes
 *                      differ by at most one, the first n % world ranks take the extra unit
 *   lorb_ba_shard_points
 *                      the points of `rank` in the large BA.  Any partition of the points, each with
 *                      all its observations, is a valid shard; this one orders the points by the lowest
 *                      window camera observing them and cuts that order into `world` runs of equal
 *                      observation count, so that a rank meets a band of cameras (its camera-pair work
 *                      lists shrink with world) and the ranks carry the same work.  out_point_ids
 *                      (capacity P, may be NULL to query *n_out) receives the point indices.
 *   lorb_ba_problem_create_sharded
 *                      that shard of a WHOLE problem given in the arrays of lorb_ba_problem_create:
 *                      the points lorb_ba_shard_points names (renumbered in that order) with all their
 *                      observations, every camera replicated.  Solve with
 *                      lorb_ba_problem_solve(..., sharded = 1); lorb_ba_problem_download then returns
 *                      all C cameras (identical on every rank) and this rank's *n_points points, point
 *                      i of the result being point out_point_ids[i] of the whole problem.
 */
int lorb_shard_range(long long n, int rank, int world, long long* lo, long long* hi);
int lorb_ba_shard_points(int P, int O, const int* obs_cam, const int* obs_pt, int rank, int world,
                         int* out_point_ids, int* n_out);
int lorb_ba_problem_create_sharded(lorb_ctx* ctx, int C, const double* cams, int P, const double* pts,
                                   int O, const int* obs_cam, const int* obs_pt, const float* obs_uv,
                                   int F, const int* fix_pt, const float* fix_uv, const float* fix_rt,
                                   const float* K, int rank, int world, lorb_ba_problem** out,
                                   int* out_point_ids, int* n_points);
/* Restore the parameters uploaded at creation (so a bench can re-solve). */
int lorb_ba_problem_reset(lorb_ba_problem* p);
/* Run LM on the resident problem.  If the ctx has a distributed group
 * (lorb_dist_init) and `sharded` != 0, the points/observations given to this
 * rank are its shard, cameras are replicated, and the reduced camera system is
 * all-reduced over NCCL every iteration (SURVEY §8(e)).  The robust loss is the
 * one set on the problem's ctx when this is called, not at creation, so one
 * resident problem can be re-solved under different losses. */
int lorb_ba_problem_solve(lorb_ba_problem* p, const lorb_ba_options* opt, int sharded,
                          lorb_ba_summary* summary);
int lorb_ba_problem_download(lorb_ba_problem* p, double* cams, double* pts);
int lorb_ba_problem_destroy(lorb_ba_problem* p);

/* ------------------------------------------------------------- multi-GPU */

#define LORB_NCCL_UNIQUE_ID_BYTES 128
/* Rank 0 calls this and broadcasts the 128 bytes by any host channel
 * (torch.distributed, MPI, a file). */
int lorb_dist_get_unique_id(uint8_t id[LORB_NCCL_UNIQUE_ID_BYTES]);
/* Create the NCCL communicator of this ctx (one ctx = one rank = one GPU). */
int lorb_dist_init(lorb_ctx* ctx, const uint8_t id[LORB_NCCL_UNIQUE_ID_BYTES], int rank, int world);
int lorb_dist_finalize(lorb_ctx* ctx);
/* Sum-allreduce `n` doubles in place on the host through the ctx communicator
 * (used by tests and to gather tiny per-rank results). */
int lorb_dist_allreduce_f64(lorb_ctx* ctx, double* data, int n);

/* ------------------------------------------------------------ diagnostics */

/* Integer-pipe micro-benchmark used for the matching roofline denominator
 * (SURVEY §8(d)): runs `iters` dependent-free popc/xor word operations per
 * thread on the whole GPU and returns 32-bit words processed per second.
 * kind 0 = xor+popc+add per word; kind 1 = the carry-save (4 popc / 8 words)
 * distance kernel body on register operands. */
int lorb_microbench_popc(lorb_ctx* ctx, int kind, int iters, double* words_per_s);

/* Tensor-pipe micro-benchmark for the tensor-core sweep's roofline denominator: the sweep's own
 * MMA stream (tcgen05.mma kind::i8, 128 x 256 x 32, `tiles` x 9 per SM) on zeroed operands with
 * no TMA traffic and no epilogue.  Returns int8 operations (2 per multiply-add) per second. */
int lorb_microbench_tensor_i8(lorb_ctx* ctx, int tiles, double* ops_per_s);

/* fp64 micro-benchmark for the BA roofline denominator (SURVEY 8(d): "a measured fp64 FMA
 * peak"): independent DFMA chains on register operands over the whole GPU.  kind 0 = scalar
 * DFMA (2 flop each), kind 1 = DMMA m8n8k4 on the tensor cores (512 flop per warp instruction).
 * Returns floating-point operations per second. */
int lorb_microbench_fp64(lorb_ctx* ctx, int kind, int iters, double* flop_per_s);

/* Device-side timing of the library's own kernels, for bench.py's roofline: while enabled,
 * the BA solver brackets its dominant kernels with CUDA events on the ctx stream
 * (slot 0 = build pass of an LM attempt, 1 = back-substitution, 2 = reduced-system solve),
 * the tensor-core sweep its main kernel (slot 3), the sharded BA its collectives (slot 4: the
 * all-reduce after the build pass and the one after the back-substitution of every attempt, as
 * seen by this rank, i.e. including the wait for the slowest rank).
 * lorb_ctx_profile_read synchronises the stream and returns the accumulated milliseconds and
 * the number of bracketed launches of a slot since the last lorb_ctx_profile(ctx, 1). */
#define LORB_PROF_SLOTS 5
int lorb_ctx_profile(lorb_ctx* ctx, int enable);
int lorb_ctx_profile_read(lorb_ctx* ctx, int slot, double* total_ms, long long* count);

#ifdef __cplusplus
}
#endif
#endif /* LORB_CUDA_H */
