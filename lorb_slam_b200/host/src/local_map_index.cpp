// local_map_index.cpp — see include/local_map_index.h.  Host-side only: the incremental
// (window, points, observations) index of the mapper and the SoA it hands to lorb_ba_local.
#include "../include/local_map_index.h"

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <functional>

#include "lorb_host.h"

using namespace Simple_ORB_SLAM;

namespace lorb_host
{

void LocalBAWindow::clear()
{
	frames.clear(); points.clear(); cams.clear(); pts.clear();
	obs_cam.clear(); obs_pt.clear(); obs_uv.clear();
	fix_pt.clear(); fix_uv.clear(); fix_rt.clear();
	obs_kp.clear(); fix_frame.clear(); fix_kp.clear();
}

int LocalMapIndex::FrameId(Frame* pF)
{
	std::unordered_map<Frame*, int>::const_iterator it = mFrameIds.find(pF);
	if(it != mFrameIds.end())
		return it->second;
	const int id = (int)mFrames.size();
	mFrameIds[pF] = id;
	mFrames.push_back(pF);
	mFramePoints.push_back(std::vector<int>());
	mFrameStamp.push_back(0);
	mFrameWindowIdx.push_back(-1);
	return id;
}

void LocalMapIndex::Record(int pid, int fid, int kp)
{
	// std::map<Frame*, size_t> semantics: one entry per frame (a second AddObservation overwrites
	// the slot), iteration in key order
	std::vector<Obs>& v = mPointObs[pid];
	std::less<Frame*> before;
	size_t k = 0;
	while(k < v.size() && before(mFrames[v[k].frame], mFrames[fid]))
		k++;
	if(k < v.size() && v[k].frame == fid)
	{
		v[k].kp = kp;
		return;
	}
	Obs o; o.frame = fid; o.kp = kp;
	v.insert(v.begin() + k, o);
	mnObservations++;
}

// The observation of point pid by frame fid leaves the index: its per-point record and the frame's
// slot entry of that point.
void LocalMapIndex::Forget(int pid, int fid)
{
	std::vector<Obs>& v = mPointObs[pid];
	for(size_t k=0; k<v.size(); k++)
		if(v[k].frame == fid)
		{
			v.erase(v.begin() + k);
			mnObservations--;
			break;
		}
	std::vector<int>& slots = mFramePoints[fid];
	std::vector<int>::iterator it = std::find(slots.begin(), slots.end(), pid);
	if(it != slots.end())
		slots.erase(it);
}

int LocalMapIndex::PointId(MapPoint* pMP)
{
	std::unordered_map<MapPoint*, int>::const_iterator it = mPointIds.find(pMP);
	if(it != mPointIds.end())
		return it->second;
	const int id = (int)mPoints.size();
	mPointIds[pMP] = id;
	mPoints.push_back(pMP);
	mPointObs.push_back(std::vector<Obs>());
	mPointStamp.push_back(0);
	// first sight: import what the map point already knows (e.g. the observations
	// VisualOdometry::Initialize added, src/visual_odometry.cpp:93)
	const std::map<Frame*, size_t> observations = pMP->GetObservations();
	for(std::map<Frame*, size_t>::const_iterator o = observations.begin(); o != observations.end(); o++)
		Record(id, FrameId(o->first), (int)o->second);
	return id;
}

void LocalMapIndex::AddObservation(MapPoint* pMP, Frame* pF, size_t idx)
{
	const int pid = PointId(pMP);
	pMP->AddObservation(pF, idx);
	Record(pid, FrameId(pF), (int)idx);
}

void LocalMapIndex::UpdateKeyFrame(Frame* pF)
{
	const int fid = FrameId(pF);
	std::vector<int>& slots = mFramePoints[fid];
	slots.clear();
	for(size_t i=0; i<pF->mvpMapPoints.size(); i++)
	{
		MapPoint* pMP = pF->mvpMapPoints[i];
		if(pMP == NULL)
			continue;
		slots.push_back(PointId(pMP));
	}
}

int LocalMapIndex::InsertKeyFrame(Frame* pF)
{
	const int fid = FrameId(pF);
	for(size_t i=0; i<pF->mvpMapPoints.size(); i++)
	{
		MapPoint* pMP = pF->mvpMapPoints[i];
		if(pMP == NULL || pMP->IsBad())
			continue;
		const int pid = PointId(pMP);
		// the reference's `IsInFrame(mpCurrFrame) == false` test (src/local_mapping.cpp:62)
		bool has = false;
		const std::vector<Obs>& v = mPointObs[pid];
		for(size_t k=0; k<v.size() && !has; k++)
			has = v[k].frame == fid;
		if(!has)
			AddObservation(pMP, pF, i);
	}
	UpdateKeyFrame(pF);
	return fid;
}

void LocalMapIndex::Assemble(Frame* pCurrFrame, LocalBAWindow& w)
{
	w.clear();
	mnEpoch++;
	// window (src/bundle_adjust.cpp:210-220); std::find returns the first occurrence of a frame
	w.frames.push_back(pCurrFrame);
	const std::vector<Frame*> vpCovisibleFrames = pCurrFrame->GetCovisibleFrames();
	for(size_t i=0; i<vpCovisibleFrames.size(); i++)
		if(!vpCovisibleFrames[i]->IsBad())
			w.frames.push_back(vpCovisibleFrames[i]);
	std::vector<int> fids(w.frames.size());
	for(size_t i=0; i<w.frames.size(); i++)
	{
		const int fid = FrameId(w.frames[i]);
		fids[i] = fid;
		if(mFrameStamp[fid] != mnEpoch)
		{
			mFrameStamp[fid] = mnEpoch;
			mFrameWindowIdx[fid] = (int)i;
		}
	}
	// points in first-occurrence order (:224-241)
	std::vector<int> pids;
	for(size_t i=0; i<w.frames.size(); i++)
	{
		const std::vector<int>& slots = mFramePoints[fids[i]];
		for(size_t j=0; j<slots.size(); j++)
		{
			const int pid = slots[j];
			if(mPointStamp[pid] == mnEpoch || mPoints[pid]->IsBad())
				continue;
			mPointStamp[pid] = mnEpoch;
			pids.push_back(pid);
			w.points.push_back(mPoints[pid]);
		}
	}
	// float state widened to double (:244-265)
	w.cams.resize(w.frames.size()*6);
	w.pts.resize(w.points.size()*3);
	for(size_t i=0; i<w.frames.size(); i++)
		for(int k=0; k<3; k++)
		{
			w.cams[6*i+k] = w.frames[i]->mRvec.at<float>(k);
			w.cams[6*i+3+k] = w.frames[i]->mTvec.at<float>(k);
		}
	for(size_t i=0; i<w.points.size(); i++)
	{
		const cv::Point3f p = w.points[i]->GetPos();
		w.pts[3*i] = p.x; w.pts[3*i+1] = p.y; w.pts[3*i+2] = p.z;
	}
	// residual records (:270-303), point by point, observers in Frame* order
	for(size_t i=0; i<pids.size(); i++)
	{
		const std::vector<Obs>& v = mPointObs[pids[i]];
		for(size_t k=0; k<v.size(); k++)
		{
			Frame* pF = mFrames[v[k].frame];
			if(pF->IsBad())
				continue;
			const cv::Point2f kp2d = pF->GetKp2d(v[k].kp);
			if(mFrameStamp[v[k].frame] == mnEpoch)
			{
				w.obs_cam.push_back(mFrameWindowIdx[v[k].frame]);
				w.obs_pt.push_back((int)i);
				w.obs_uv.push_back(kp2d.x); w.obs_uv.push_back(kp2d.y);
				w.obs_kp.push_back(v[k].kp);
			}
			else
			{
				w.fix_pt.push_back((int)i);
				w.fix_uv.push_back(kp2d.x); w.fix_uv.push_back(kp2d.y);
				for(int a=0; a<3; a++) w.fix_rt.push_back(pF->mRvec.at<float>(a));
				for(int a=0; a<3; a++) w.fix_rt.push_back(pF->mTvec.at<float>(a));
				w.fix_frame.push_back(pF);
				w.fix_kp.push_back(v[k].kp);
			}
		}
	}
}

// float write-back of a solved window (src/bundle_adjust.cpp:317-329)
static void WriteBack(const LocalBAWindow& w)
{
	for(size_t i=0; i<w.frames.size(); i++)
	{
		cv::Mat R(3, 1, CV_32F), T(3, 1, CV_32F);
		for(int k=0; k<3; k++)
		{
			R.at<float>(k) = (float)w.cams[6*i+k];
			T.at<float>(k) = (float)w.cams[6*i+3+k];
		}
		w.frames[i]->SetPose(T, R);
	}
	for(size_t i=0; i<w.points.size(); i++)
		w.points[i]->SetWorldPos(cv::Point3f((float)w.pts[3*i], (float)w.pts[3*i+1], (float)w.pts[3*i+2]));
}

static float InvSigma2(Frame* pF, int kp)
{
	const float s = pF->mvScaleFactors[pF->mvKeysUn[kp].octave];
	return 1.0f / (s * s);
}

void LocalMapIndex::Optimize(Frame* pCurrFrame)
{
	LocalBAWindow& w = mWindow;
	Assemble(pCurrFrame, w);
	const Camera* cam = pCurrFrame->mpCamera;
	const float K[4] = {cam->fx, cam->fy, cam->cx, cam->cy};
	lorb_ba_options opt;
	lorb_ba_default_options(&opt);
	lorb_ba_summary summary;
	LORB_HOST_CALL(lorb_ba_local(lorb_host::ctx(), (int)w.frames.size(), w.cams.data(), (int)w.points.size(),
	                             w.pts.data(), (int)w.obs_cam.size(), w.obs_cam.data(), w.obs_pt.data(),
	                             w.obs_uv.data(), (int)w.fix_pt.size(), w.fix_pt.data(), w.fix_uv.data(),
	                             w.fix_rt.data(), K, &opt, &summary));
	WriteBack(w);
}

int LocalMapIndex::OptimizeRejectingOutliers(Frame* pCurrFrame)
{
	LocalBAWindow& w = mWindow;
	Assemble(pCurrFrame, w);
	const Camera* cam = pCurrFrame->mpCamera;
	const float K[4] = {cam->fx, cam->fy, cam->cx, cam->cy};
	const int O = (int)w.obs_cam.size(), F = (int)w.fix_pt.size();
	std::vector<float> obs_w(O), fix_w(F);
	for(int i=0; i<O; i++)
		obs_w[i] = InvSigma2(w.frames[w.obs_cam[i]], w.obs_kp[i]);
	for(int i=0; i<F; i++)
		fix_w[i] = InvSigma2(w.fix_frame[i], w.fix_kp[i]);
	lorb_ba_local_rounds rounds;
	lorb_ba_options opt[2];
	lorb_ba_default_local_rounds(&rounds, opt);
	std::vector<uint8_t> obs_in(O), fix_in(F);
	int n_in = 0;
	lorb_ctx* c = ctx();
	lorb_ba_loss prev, huber = {LORB_LOSS_HUBER, 0, std::sqrt(rounds.chi2)};
	LORB_HOST_CALL(lorb_ba_get_loss(c, &prev));
	LORB_HOST_CALL(lorb_ba_set_loss(c, &huber));
	const int rc = lorb_ba_local_rounds_single(c, (int)w.frames.size(), w.cams.data(), (int)w.points.size(),
	                                           w.pts.data(), O, w.obs_cam.data(), w.obs_pt.data(), w.obs_uv.data(),
	                                           obs_w.data(), F, w.fix_pt.data(), w.fix_uv.data(), w.fix_rt.data(),
	                                           fix_w.data(), K, &rounds, opt, obs_in.data(), NULL, fix_in.data(),
	                                           NULL, &n_in, NULL);
	LORB_HOST_CALL(lorb_ba_set_loss(c, &prev));
	if(rc != LORB_OK) die("lorb_ba_local_rounds_single", rc);
	WriteBack(w);
	int n_erased = 0;
	for(int i=0; i<O+F; i++)
	{
		if(i < O ? obs_in[i] : fix_in[i-O])
			continue;
		Frame* pF = i < O ? w.frames[w.obs_cam[i]] : w.fix_frame[i-O];
		const int kp = i < O ? w.obs_kp[i] : w.fix_kp[i-O];
		MapPoint* pMP = w.points[i < O ? w.obs_pt[i] : w.fix_pt[i-O]];
		pF->mvpMapPoints[kp] = NULL;
		pMP->mnObs--;
		Forget(PointId(pMP), FrameId(pF));
		n_erased++;
	}
	return n_erased;
}

}
