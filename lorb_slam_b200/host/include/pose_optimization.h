// pose_optimization.h — pose-only BA with outlier rounds for the drop-in layer (beyond the reference:
// ORB-SLAM2's Optimizer::PoseOptimization).  A caller that wants outlier rejection calls it in place
// of BA::ProjectPoseOptimization; it sets the frame's pose and its mvbOutlier flags, which the next
// Matcher::SearchByProjection(Cur, Last, th) reads.  BA and bundle_adjust.h are unchanged.
#ifndef LORB_POSE_OPTIMIZATION_H
#define LORB_POSE_OPTIMIZATION_H

#include "common.h"
#include "frame.h"
#include "camera.h"

namespace lorb_host
{

// Four rounds of at most 10 LM iterations over the frame's non-NULL map points, each observation
// weighted by 1 / sigma^2 of its octave (mvScaleFactors[mvKeysUn[i].octave]^-2), Huber with
// delta = sqrt(5.991) in the first three rounds, chi-square 5.991 classification after each round
// (lorb_ba_pose_rounds_batched).  Sets the pose (SetPose) and mvbOutlier[i] of every non-NULL map
// point; returns the number of inliers.  The calling thread's ctx keeps its own robust loss.
int PoseOptimization(Simple_ORB_SLAM::Frame* pFrame);

}

#endif
