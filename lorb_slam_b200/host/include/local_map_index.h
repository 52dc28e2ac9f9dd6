// local_map_index.h — the hand-off between the mapper and lorb_ba_local (SURVEY 8(f) rank 3).
//
// The reference assembles the local-BA problem from scratch on every call
// (src/bundle_adjust.cpp:207-303): it copies one std::map<Frame*, size_t> per map point
// (GetObservations()), searches the window with std::find per observation (:280) and the point
// list with std::find per map point (:235).  LocalMapping is where that information is born --
// ProcessNewFrames (src/local_mapping.cpp:48-78) adds the new keyframe's observations one by one
// -- so this index is maintained THERE, once per keyframe insert, with dense integer ids:
//
//   frame id  -> its (map point id, keypoint) slots in mvpMapPoints order
//   point id  -> its observations (frame id, keypoint index), kept in Frame* address order,
//                which is the iteration order of the reference's std::map<Frame*, size_t>
//
// Assemble() then produces the flat SoA of lorb_ba_local (the on-wire format between mapper and
// solver) by integer walks only: window = current frame + its non-bad covisible frames (:210-220),
// points in first-occurrence order (:224-241), one PoseMPCost record per in-window observation and
// one MPCost record (with the observer's fixed float pose) per out-of-window one (:270-303), in
// exactly the order the reference adds its residual blocks.  Optimize() = Assemble + lorb_ba_local
// + the float write-back (:317-329): what local_mapping.cpp:32 would call.
//
// Contract: a keyframe's map-point slots are read when it is inserted (call UpdateKeyFrame after
// changing them); observations added to a map point behind the index's back are picked up when
// the point is first seen (its whole observation map is imported) and by AddObservation().
#ifndef LORB_LOCAL_MAP_INDEX_H
#define LORB_LOCAL_MAP_INDEX_H
#include <unordered_map>
#include <vector>

#include "frame.h"
#include "map_point.h"

namespace lorb_host
{

// Flat problem of one local-BA call: the argument arrays of lorb_ba_local (include/lorb_cuda.h).
struct LocalBAWindow
{
	std::vector<Simple_ORB_SLAM::Frame*> frames;      // [C] window, current frame first
	std::vector<Simple_ORB_SLAM::MapPoint*> points;   // [P]
	std::vector<double> cams;                         // [C][6] (w, t) from float mRvec / mTvec
	std::vector<double> pts;                          // [P][3]
	std::vector<int> obs_cam, obs_pt;                 // [O] window-local indices
	std::vector<float> obs_uv;                        // [O][2]
	std::vector<int> fix_pt;                          // [F]
	std::vector<float> fix_uv, fix_rt;                // [F][2], [F][6]
	// the keypoint behind each record: in-window observation i is keypoint obs_kp[i] of
	// frames[obs_cam[i]]; fixed observation i is keypoint fix_kp[i] of fix_frame[i]
	std::vector<int> obs_kp;                          // [O]
	std::vector<Simple_ORB_SLAM::Frame*> fix_frame;   // [F]
	std::vector<int> fix_kp;                          // [F]
	void clear();
};

class LocalMapIndex
{
public:
	// LocalMapping::ProcessNewFrames step 1 (src/local_mapping.cpp:55-69) for one keyframe: every
	// non-bad map point it holds gains the observation (pF, slot) unless it already has it, and
	// the keyframe's slots enter the index.  Returns the keyframe's dense id.
	int InsertKeyFrame(Simple_ORB_SLAM::Frame* pF);
	// Re-read a keyframe's mvpMapPoints after the mapper changed them.
	void UpdateKeyFrame(Simple_ORB_SLAM::Frame* pF);
	// MapPoint::AddObservation through the index (keeps both in step).
	void AddObservation(Simple_ORB_SLAM::MapPoint* pMP, Simple_ORB_SLAM::Frame* pF, size_t idx);

	void Assemble(Simple_ORB_SLAM::Frame* pCurrFrame, LocalBAWindow& w);
	// BA::LocalPoseOptimization(pCurrFrame) with the problem taken from the index.
	void Optimize(Simple_ORB_SLAM::Frame* pCurrFrame);
	// ORB-SLAM2's Optimizer::LocalBundleAdjustment over the same problem (lorb_ba_local_rounds_single
	// with lorb_ba_default_local_rounds: 5 iterations under Huber sqrt(chi2), then 10 plain ones over the
	// inliers; every observation weighted by 1 / sigma^2 of its keypoint's octave, read from the
	// observing frame's mvScaleFactors / mvKeysUn).  The ctx's loss is put back afterwards.  Writes the
	// floats back as Optimize does, then erases every observation flagged outlier (chi^2 > 5.991 or
	// not in front of its camera): the frame's mvpMapPoints[kp] becomes NULL, the point's mnObs drops
	// by one and the index forgets the observation, so no later Assemble sees it.  The map point's own
	// observation map is private in the reference and is left alone.  Returns the number of erased
	// observations.
	int OptimizeRejectingOutliers(Simple_ORB_SLAM::Frame* pCurrFrame);

	size_t NumFrames() const { return mFrames.size(); }
	size_t NumPoints() const { return mPoints.size(); }
	size_t NumObservations() const { return mnObservations; }

private:
	struct Obs { int frame; int kp; };
	int FrameId(Simple_ORB_SLAM::Frame* pF);
	int PointId(Simple_ORB_SLAM::MapPoint* pMP);
	void Record(int pid, int fid, int kp);
	void Forget(int pid, int fid);

	std::unordered_map<Simple_ORB_SLAM::Frame*, int> mFrameIds;
	std::unordered_map<Simple_ORB_SLAM::MapPoint*, int> mPointIds;
	std::vector<Simple_ORB_SLAM::Frame*> mFrames;
	std::vector<Simple_ORB_SLAM::MapPoint*> mPoints;
	std::vector<std::vector<int> > mFramePoints;  // per frame: point id per non-NULL slot, slot order
	std::vector<std::vector<Obs> > mPointObs;     // per point: observations in Frame* address order
	std::vector<int> mFrameStamp, mFrameWindowIdx, mPointStamp;
	int mnEpoch = 0;
	size_t mnObservations = 0;
	LocalBAWindow mWindow;  // reused between calls: steady state allocates nothing
};

}
#endif
