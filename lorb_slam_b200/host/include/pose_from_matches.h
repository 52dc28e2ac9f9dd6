// pose_from_matches.h — pose of a frame from its 2D-3D matches without a prior, for the drop-in layer (beyond
// the reference: the pose half of VisualOdometry::EstimatePosePnP, declared and never called there, and of
// ORB-SLAM2's per-candidate relocalisation step).  It runs after the brute-force
// Matcher::SearchByProjection(curr, refer) has filled the frame's mvpMapPoints.
#ifndef LORB_POSE_FROM_MATCHES_H
#define LORB_POSE_FROM_MATCHES_H

#include "common.h"
#include "frame.h"
#include "camera.h"

namespace lorb_host
{

// P3P RANSAC (lorb_pnp_ransac_batched, default parameters: 300 hypotheses, chi-square 5.991) over the frame's
// non-NULL map points, each weighted by 1 / sigma^2 of its octave.  Below min_inliers RANSAC inliers it returns
// that count and leaves the frame untouched.  Otherwise it sets mvpMapPoints[i] = NULL for the RANSAC outliers
// (as ORB-SLAM2's Relocalization does), sets the RANSAC pose and returns lorb_host::PoseOptimization(pF): the
// pose-only rounds from that pose, which set the final pose and mvbOutlier.
int PoseFromMatches(Simple_ORB_SLAM::Frame* pF, int min_inliers = 10);

}

#endif
