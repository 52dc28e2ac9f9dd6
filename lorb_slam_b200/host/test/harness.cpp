// harness.cpp — test-only C entry points that build Frame / MapPoint objects
// (shim versions here, the real ones in a LORB-SLAM checkout) from flat arrays,
// call the drop-in Matcher / BA classes exactly as VisualOdometry / LocalMapping
// do, and hand the mutated object state back as arrays.  tests/test_host_dropin_gpu.py
// compares those with the oracle.
#include <cstring>
#include <deque>
#include <thread>

#include "../include/ORBextractor.h"
#include "../src/lorb_host.h"
#include "../include/bundle_adjust.h"
#include "../include/matcher.h"
#include "../include/local_map_index.h"
#include "../include/pose_optimization.h"
#include "../include/pose_from_matches.h"

#include <algorithm>
#include <chrono>

using namespace Simple_ORB_SLAM;

namespace
{
cv::Mat DescMat(const uint8_t* d, int n)
{
	cv::Mat m(n, 32, CV_8U);
	if(n) std::memcpy(m.ptr<uint8_t>(), d, (size_t)n*32);
	return m;
}

void FillFrame(Frame& F, int n, const float* x, const float* y, const int* oct, const float* ang,
               const float* ur, const uint8_t* desc, float minx, float maxx, float miny, float maxy,
               int nlev, const float* sf)
{
	F.mnMapPoints = n;
	F.mvpMapPoints.assign(n, static_cast<MapPoint*>(NULL));
	F.mvKeysUn.resize(n);
	for(int i=0;i<n;i++)
	{
		F.mvKeysUn[i].pt = cv::Point2f(x[i], y[i]);
		F.mvKeysUn[i].octave = oct[i];
		F.mvKeysUn[i].angle = ang[i];
	}
	F.mvKeys = F.mvKeysUn;
	F.mvuRight.assign(ur, ur+n);
	F.mvbOutlier.assign(n, false);
	F.mDescriptors = DescMat(desc, n);
	F.mnMinX = minx; F.mnMaxX = maxx; F.mnMinY = miny; F.mnMaxY = maxy;
	F.mvScaleFactors.assign(sf, sf+nlev);
	F.mnScaleLevels = nlev;
}
}

extern "C" {

// Matcher::SearchByProjection(curr, prev) [which=0] / Matcher::SearchLocalPoints [which=1]
// prev_has[j] == 0 leaves a NULL slot in prev->mvpMapPoints.  out_assign[i] = index j of the
// map point now held by curr keypoint i, -1 if none.
int harness_bf(int which, int nq, const uint8_t* qdesc, int nt, const uint8_t* tdesc,
               const uint8_t* prev_has, int* out_assign)
{
	Frame curr, prev;
	std::vector<float> z(nq, 0.f);
	std::vector<int> zi(nq, 0);
	float sf = 1.f;
	FillFrame(curr, nq, z.data(), z.data(), zi.data(), z.data(), z.data(), qdesc, 0, 640, 0, 480, 1, &sf);
	std::vector<MapPoint> mps(nt);  // contiguous: pointer order == index order (std::set iteration)
	prev.mnMapPoints = nt;
	prev.mvpMapPoints.assign(nt, static_cast<MapPoint*>(NULL));
	std::set<MapPoint*> local;
	for(int j=0;j<nt;j++)
	{
		mps[j].mDescriptor = DescMat(tdesc + (size_t)j*32, 1);
		if(prev_has[j]) { prev.mvpMapPoints[j] = &mps[j]; local.insert(&mps[j]); }
	}
	const size_t n = which == 0 ? Matcher::SearchByProjection(&curr, &prev)
	                            : Matcher::SearchLocalPoints(&curr, local);
	for(int i=0;i<nq;i++)
		out_assign[i] = curr.mvpMapPoints[i] ? (int)(curr.mvpMapPoints[i] - &mps[0]) : -1;
	return (int)n;
}

// Matcher::SearchByProjection(F, set<MapPoint*>, th)
int harness_proj_points(int n_kp, const float* x, const float* y, const int* oct, const float* ang,
                        const float* ur, const uint8_t* desc, const int* claim_obs, float minx,
                        float maxx, float miny, float maxy, int nlev, const float* sf, int n_pts,
                        const float* px, const float* py, const float* pxr, const int* level,
                        const float* vcos, const uint8_t* active, const uint8_t* mpdesc,
                        const int* nobs, float th, int* out_assign)
{
	Frame F;
	FillFrame(F, n_kp, x, y, oct, ang, ur, desc, minx, maxx, miny, maxy, nlev, sf);
	std::deque<MapPoint> holders;  // pre-existing claims
	for(int i=0;i<n_kp;i++)
		if(claim_obs[i] >= 0)
		{
			holders.emplace_back();
			holders.back().mnObs = (size_t)claim_obs[i];
			F.mvpMapPoints[i] = &holders.back();
		}
	std::vector<MapPoint> mps(n_pts);
	std::set<MapPoint*> local;
	for(int k=0;k<n_pts;k++)
	{
		MapPoint& m = mps[k];
		m.mDescriptor = DescMat(mpdesc + (size_t)k*32, 1);
		m.mnObs = (size_t)nobs[k];
		m.mbTrackInView = active[k] != 0;
		m.mTrackProjX = px[k]; m.mTrackProjY = py[k]; m.mTrackProjXR = pxr[k];
		m.mnTrackScaleLevel = level[k]; m.mTrackViewCos = vcos[k];
		local.insert(&m);
	}
	const size_t n = Matcher::SearchByProjection(&F, local, th);
	for(int i=0;i<n_kp;i++)
	{
		MapPoint* h = F.mvpMapPoints[i];
		out_assign[i] = (h && n_pts && h >= &mps[0] && h <= &mps[n_pts-1]) ? (int)(h - &mps[0]) : -1;
	}
	return (int)n;
}

// Matcher::SearchByProjection(Cur, Last, th).  out_state: >=0 last item held, -2 NULL (was
// touched and cleared or never held), -1 still holding its pre-existing claim.
int harness_proj_frame(int n_kp, const float* x, const float* y, const int* oct, const float* ang,
                       const float* ur, const uint8_t* desc, const int* claim_obs, float minx,
                       float maxx, float miny, float maxy, int nlev, const float* sf,
                       const float* tcw_cur, const float* tcw_last, const float* K6, int n_last,
                       const uint8_t* valid, const float* xw, const int* loct, const float* lang,
                       const uint8_t* mpdesc, const int* nobs, float th, int* out_state)
{
	Frame Cur, Last;
	FillFrame(Cur, n_kp, x, y, oct, ang, ur, desc, minx, maxx, miny, maxy, nlev, sf);
	Cur.fx = K6[0]; Cur.fy = K6[1]; Cur.cx = K6[2]; Cur.cy = K6[3]; Cur.mbf = K6[4]; Cur.mb = K6[5];
	for(int r=0;r<4;r++) for(int c=0;c<4;c++)
	{
		Cur.mTcw.at<float>(r,c) = tcw_cur[4*r+c];
		Last.mTcw.at<float>(r,c) = tcw_last[4*r+c];
	}
	std::deque<MapPoint> holders;
	for(int i=0;i<n_kp;i++)
		if(claim_obs[i] >= 0)
		{
			holders.emplace_back();
			holders.back().mnObs = (size_t)claim_obs[i];
			Cur.mvpMapPoints[i] = &holders.back();
		}
	std::vector<MapPoint> mps(n_last);
	Last.mnMapPoints = n_last;
	Last.mvpMapPoints.assign(n_last, static_cast<MapPoint*>(NULL));
	Last.mvbOutlier.assign(n_last, false);
	Last.mvKeys.resize(n_last);
	Last.mvKeysUn.resize(n_last);
	for(int i=0;i<n_last;i++)
	{
		Last.mvKeys[i].octave = loct[i];
		Last.mvKeysUn[i].octave = loct[i];
		Last.mvKeysUn[i].angle = lang[i];
		if(valid[i])
		{
			mps[i].mWorldPos = cv::Point3f(xw[3*i], xw[3*i+1], xw[3*i+2]);
			mps[i].mDescriptor = DescMat(mpdesc + (size_t)i*32, 1);
			mps[i].mnObs = (size_t)nobs[i];
			Last.mvpMapPoints[i] = &mps[i];
		}
	}
	const size_t n = Matcher::SearchByProjection(&Cur, &Last, th);
	for(int i=0;i<n_kp;i++)
	{
		MapPoint* h = Cur.mvpMapPoints[i];
		if(h == NULL) out_state[i] = -2;
		else if(n_last && h >= &mps[0] && h <= &mps[n_last-1]) out_state[i] = (int)(h - &mps[0]);
		else out_state[i] = -1;
	}
	return (int)n;
}

// The tracking loop with outlier rounds: lorb_host::PoseOptimization on Last (keypoints luv, octaves
// loct, valid map points xw; rt float[6] R then T in/out), then Matcher::SearchByProjection(Cur, Last, th)
// on the same Last object, which reads the mvbOutlier flags PoseOptimization set.  Out: Last's
// mvbOutlier (1 = outlier, 0 otherwise), its mTcw after SetPose, Cur's state as harness_proj_frame,
// the number of matches in *n_matches.  Returns PoseOptimization's inlier count.
int harness_pose_rounds_search(int n_kp, const float* x, const float* y, const int* oct, const float* ang,
                               const float* ur, const uint8_t* desc, float minx, float maxx, float miny,
                               float maxy, int nlev, const float* sf, const float* tcw_cur, const float* K6,
                               int n_last, const uint8_t* valid, const float* xw, const int* loct,
                               const float* lang, const float* luv, const uint8_t* mpdesc, const int* nobs,
                               float* rt, float th, uint8_t* out_outlier, float* out_tcw_last, int* out_state,
                               int* n_matches)
{
	Camera cam;
	cam.fx = K6[0]; cam.fy = K6[1]; cam.cx = K6[2]; cam.cy = K6[3];
	Frame Cur, Last;
	std::vector<float> lz(n_last, 0.0f), lur(n_last, -1.0f);
	std::vector<uint8_t> ldesc((size_t)n_last*32, 0);
	FillFrame(Last, n_last, lz.data(), lz.data(), loct, lang, lur.data(), ldesc.data(), minx, maxx, miny, maxy,
	          nlev, sf);
	Last.mpCamera = &cam;
	std::vector<MapPoint> mps(n_last);
	for(int i=0;i<n_last;i++)
	{
		Last.mvKeysUn[i].pt = cv::Point2f(luv[2*i], luv[2*i+1]);
		if(valid[i])
		{
			mps[i].mWorldPos = cv::Point3f(xw[3*i], xw[3*i+1], xw[3*i+2]);
			mps[i].mDescriptor = DescMat(mpdesc + (size_t)i*32, 1);
			mps[i].mnObs = (size_t)nobs[i];
			Last.mvpMapPoints[i] = &mps[i];
		}
	}
	for(int k=0;k<3;k++) { Last.mRvec.at<float>(k) = rt[k]; Last.mTvec.at<float>(k) = rt[3+k]; }
	const int n_in = lorb_host::PoseOptimization(&Last);
	for(int k=0;k<3;k++) { rt[k] = Last.mRvec.at<float>(k); rt[3+k] = Last.mTvec.at<float>(k); }
	for(int i=0;i<n_last;i++) out_outlier[i] = Last.mvbOutlier[i] ? 1 : 0;
	for(int r=0;r<4;r++) for(int c=0;c<4;c++) out_tcw_last[4*r+c] = Last.mTcw.at<float>(r,c);

	FillFrame(Cur, n_kp, x, y, oct, ang, ur, desc, minx, maxx, miny, maxy, nlev, sf);
	Cur.fx = K6[0]; Cur.fy = K6[1]; Cur.cx = K6[2]; Cur.cy = K6[3]; Cur.mbf = K6[4]; Cur.mb = K6[5];
	for(int r=0;r<4;r++) for(int c=0;c<4;c++) Cur.mTcw.at<float>(r,c) = tcw_cur[4*r+c];
	*n_matches = (int)Matcher::SearchByProjection(&Cur, &Last, th);
	for(int i=0;i<n_kp;i++)
	{
		MapPoint* h = Cur.mvpMapPoints[i];
		if(h == NULL) out_state[i] = -2;
		else if(n_last && h >= &mps[0] && h <= &mps[n_last-1]) out_state[i] = (int)(h - &mps[0]);
		else out_state[i] = -1;
	}
	return n_in;
}

// lorb_host::PoseFromMatches on a frame of n keypoints (uv, octaves oct, scale factors sf) whose
// mvpMapPoints[i] holds a map point at xw[i] iff has_mp[i]; rt (float[6]: R then T) in/out.  Out: which slots
// still hold their map point, and mvbOutlier.  Returns PoseFromMatches' result.
int harness_pose_from_matches(int n, const float* xw, const float* uv, const int* oct, const uint8_t* has_mp,
                              int nlev, const float* sf, const float* K4, int min_inliers, float* rt,
                              uint8_t* out_has_mp, uint8_t* out_outlier)
{
	Camera cam;
	cam.fx = K4[0]; cam.fy = K4[1]; cam.cx = K4[2]; cam.cy = K4[3];
	Frame F;
	F.mpCamera = &cam;
	F.mnMapPoints = n;
	F.mvKeysUn.resize(n);
	F.mvbOutlier.assign(n, false);
	F.mvScaleFactors.assign(sf, sf+nlev);
	F.mnScaleLevels = nlev;
	std::vector<MapPoint> mps(n);
	F.mvpMapPoints.assign(n, static_cast<MapPoint*>(NULL));
	for(int i=0;i<n;i++)
	{
		F.mvKeysUn[i].pt = cv::Point2f(uv[2*i], uv[2*i+1]);
		F.mvKeysUn[i].octave = oct[i];
		mps[i].mWorldPos = cv::Point3f(xw[3*i], xw[3*i+1], xw[3*i+2]);
		if(has_mp[i]) F.mvpMapPoints[i] = &mps[i];
	}
	for(int k=0;k<3;k++) { F.mRvec.at<float>(k) = rt[k]; F.mTvec.at<float>(k) = rt[3+k]; }
	const int r = lorb_host::PoseFromMatches(&F, min_inliers);
	for(int k=0;k<3;k++) { rt[k] = F.mRvec.at<float>(k); rt[3+k] = F.mTvec.at<float>(k); }
	for(int i=0;i<n;i++)
	{
		out_has_mp[i] = F.mvpMapPoints[i] ? 1 : 0;
		out_outlier[i] = F.mvbOutlier[i] ? 1 : 0;
	}
	return r;
}

// BA::ProjectPoseOptimization: rt (float[6]: R then T) in/out
void harness_pose_opt(int n, const float* xw, const float* uv, const float* K4, float* rt)
{
	Camera cam;
	cam.fx = K4[0]; cam.fy = K4[1]; cam.cx = K4[2]; cam.cy = K4[3];
	Frame F;
	F.mpCamera = &cam;
	F.mnMapPoints = n;
	F.mvKeysUn.resize(n);
	std::vector<MapPoint> mps(n);
	F.mvpMapPoints.assign(n, static_cast<MapPoint*>(NULL));
	for(int i=0;i<n;i++)
	{
		F.mvKeysUn[i].pt = cv::Point2f(uv[2*i], uv[2*i+1]);
		mps[i].mWorldPos = cv::Point3f(xw[3*i], xw[3*i+1], xw[3*i+2]);
		F.mvpMapPoints[i] = &mps[i];
	}
	for(int k=0;k<3;k++) { F.mRvec.at<float>(k) = rt[k]; F.mTvec.at<float>(k) = rt[3+k]; }
	BA::ProjectPoseOptimization(&F);
	for(int k=0;k<3;k++) { rt[k] = F.mRvec.at<float>(k); rt[3+k] = F.mTvec.at<float>(k); }
}

// BA::LocalPoseOptimization on a window of C frames (frame 0 = current, the rest covisible)
// plus n_fix out-of-window observers.  cams / fix_rt are float (R then T); points float.
void harness_local_ba(int C, float* cams, int P, float* pts, int O, const int* obs_cam,
                      const int* obs_pt, const float* obs_uv, int n_fix, const int* fix_pt,
                      const float* fix_uv, const float* fix_rt, const float* K4)
{
	Camera cam;
	cam.fx = K4[0]; cam.fy = K4[1]; cam.cx = K4[2]; cam.cy = K4[3];
	// frames live in one array so that std::map<Frame*,...> iterates window frames by index and
	// the fixed observers (allocated after them) last — the order the flat arrays are given in
	std::vector<Frame> frames(C + n_fix);
	std::vector<MapPoint> mps(P);
	for(int p=0;p<P;p++) mps[p].mWorldPos = cv::Point3f(pts[3*p], pts[3*p+1], pts[3*p+2]);
	for(int c=0;c<C+n_fix;c++)
	{
		Frame& F = frames[c];
		F.mpCamera = &cam;
		const float* rt = c < C ? cams + 6*c : fix_rt + 6*(c-C);
		cv::Mat R(3,1,CV_32F), T(3,1,CV_32F);
		for(int k=0;k<3;k++) { R.at<float>(k) = rt[k]; T.at<float>(k) = rt[3+k]; }
		F.SetPose(T, R);
	}
	auto add_obs = [&](Frame& F, int p, float u, float v)
	{
		cv::KeyPoint kp;
		kp.pt = cv::Point2f(u, v);
		F.mvKeysUn.push_back(kp);
		F.mvpMapPoints.push_back(&mps[p]);
		F.mnMapPoints = F.mvKeysUn.size();
		mps[p].AddObservation(&F, F.mvKeysUn.size()-1);
	};
	for(int i=0;i<O;i++) add_obs(frames[obs_cam[i]], obs_pt[i], obs_uv[2*i], obs_uv[2*i+1]);
	for(int i=0;i<n_fix;i++) add_obs(frames[C+i], fix_pt[i], fix_uv[2*i], fix_uv[2*i+1]);
	for(int c=1;c<C;c++) frames[0].mvpOrderedKeyFrames.push_back(&frames[c]);
	BA::LocalPoseOptimization(&frames[0]);
	for(int c=0;c<C;c++)
		for(int k=0;k<3;k++)
		{
			cams[6*c+k] = frames[c].mRvec.at<float>(k);
			cams[6*c+3+k] = frames[c].mTvec.at<float>(k);
		}
	for(int p=0;p<P;p++)
	{
		const cv::Point3f q = mps[p].GetPos();
		pts[3*p] = q.x; pts[3*p+1] = q.y; pts[3*p+2] = q.z;
	}
}


// The mapper's hand-off (SURVEY 8(f) rank 3): keyframes are inserted one by one, as
// LocalMapping::ProcessNewFrames would (reference src/local_mapping.cpp:48-78), and after every
// insert from keyframe `first_ba` on the local BA of the new keyframe runs (the call the reference
// has at src/local_mapping.cpp:32).  Two identical worlds are driven side by side:
//   A: lorb_host::LocalMapIndex::InsertKeyFrame + Optimize (index maintained per insert)
//   B: MapPoint::AddObservation per slot + BA::LocalPoseOptimization (re-walks the std::maps)
// Keyframe k holds the slots [kf_off[k], kf_off[k+1]) = (point, u, v); its covisible list is
// cov_idx[cov_off[k] .. cov_off[k+1]) (earlier keyframes).  Outputs: final float poses / points of
// both worlds, the number of BA calls, and the host microseconds spent assembling in each world
// (B: a dry run of the reference's own walks, :207-303).
int harness_local_mapping(int n_kf, const float* kf_rt, const int* kf_off, const int* slot_pt,
                          const float* slot_uv, const int* cov_off, const int* cov_idx, int P,
                          const float* pts, const float* K4, int first_ba, float* out_cams_a,
                          float* out_pts_a, float* out_cams_b, float* out_pts_b, double* us_assemble)
{
	Camera cam;
	cam.fx = K4[0]; cam.fy = K4[1]; cam.cx = K4[2]; cam.cy = K4[3];
	struct World
	{
		std::vector<Frame> frames;
		std::vector<MapPoint> mps;
	};
	World W[2];
	for(int w=0; w<2; w++)
	{
		W[w].frames.resize(n_kf);
		W[w].mps.resize(P);
		for(int p=0;p<P;p++) W[w].mps[p].mWorldPos = cv::Point3f(pts[3*p], pts[3*p+1], pts[3*p+2]);
	}
	lorb_host::LocalMapIndex index;
	lorb_host::LocalBAWindow probe;
	int n_ba = 0;
	us_assemble[0] = us_assemble[1] = 0;
	for(int k=0; k<n_kf; k++)
	{
		for(int w=0; w<2; w++)
		{
			Frame& F = W[w].frames[k];
			F.mpCamera = &cam;
			cv::Mat R(3,1,CV_32F), T(3,1,CV_32F);
			for(int a=0;a<3;a++) { R.at<float>(a) = kf_rt[6*k+a]; T.at<float>(a) = kf_rt[6*k+3+a]; }
			F.SetPose(T, R);
			for(int s=kf_off[k]; s<kf_off[k+1]; s++)
			{
				cv::KeyPoint kp;
				kp.pt = cv::Point2f(slot_uv[2*s], slot_uv[2*s+1]);
				F.mvKeysUn.push_back(kp);
				F.mvpMapPoints.push_back(slot_pt[s] >= 0 ? &W[w].mps[slot_pt[s]] : static_cast<MapPoint*>(NULL));
			}
			F.mnMapPoints = F.mvKeysUn.size();
			for(int c=cov_off[k]; c<cov_off[k+1]; c++) F.mvpOrderedKeyFrames.push_back(&W[w].frames[cov_idx[c]]);
		}
		// world A: through the index
		index.InsertKeyFrame(&W[0].frames[k]);
		// world B: the reference's step 1 by hand
		for(size_t i=0; i<W[1].frames[k].mvpMapPoints.size(); i++)
		{
			MapPoint* pMP = W[1].frames[k].mvpMapPoints[i];
			if(pMP != NULL && !pMP->IsBad() && !pMP->mObservations.count(&W[1].frames[k]))
				pMP->AddObservation(&W[1].frames[k], i);
		}
		if(k < first_ba)
			continue;
		{
			const auto t0 = std::chrono::steady_clock::now();
			index.Assemble(&W[0].frames[k], probe);
			const auto t1 = std::chrono::steady_clock::now();
			us_assemble[0] += std::chrono::duration<double, std::micro>(t1 - t0).count();
			// dry run of the reference's walks (window, dedup by std::find, one std::map copy per point)
			Frame* pCurr = &W[1].frames[k];
			std::vector<Frame*> local;
			local.push_back(pCurr);
			std::vector<Frame*> cov = pCurr->GetCovisibleFrames();
			for(size_t i=0;i<cov.size();i++) if(!cov[i]->IsBad()) local.push_back(cov[i]);
			std::vector<MapPoint*> lmp;
			for(size_t i=0;i<local.size();i++)
			{
				std::vector<MapPoint*> v = local[i]->GetMapPoints();
				for(size_t j=0;j<v.size();j++)
				{
					if(v[j] == NULL || v[j]->IsBad()) continue;
					if(std::find(lmp.begin(), lmp.end(), v[j]) != lmp.end()) continue;
					lmp.push_back(v[j]);
				}
			}
			size_t n_res = 0;
			for(size_t i=0;i<lmp.size();i++)
			{
				std::map<Frame*, size_t> obs = lmp[i]->GetObservations();
				for(std::map<Frame*, size_t>::const_iterator it = obs.begin(); it != obs.end(); it++)
					if(!it->first->IsBad())
						n_res += std::find(local.begin(), local.end(), it->first) != local.end() ? 2 : 1;
			}
			const auto t2 = std::chrono::steady_clock::now();
			us_assemble[1] += std::chrono::duration<double, std::micro>(t2 - t1).count();
			if(n_res == 0) return -1;
		}
		index.Optimize(&W[0].frames[k]);
		BA::LocalPoseOptimization(&W[1].frames[k]);
		n_ba++;
	}
	for(int w=0; w<2; w++)
	{
		float* oc = w == 0 ? out_cams_a : out_cams_b;
		float* op = w == 0 ? out_pts_a : out_pts_b;
		for(int k=0;k<n_kf;k++)
			for(int a=0;a<3;a++)
			{
				oc[6*k+a] = W[w].frames[k].mRvec.at<float>(a);
				oc[6*k+3+a] = W[w].frames[k].mTvec.at<float>(a);
			}
		for(int p=0;p<P;p++)
		{
			const cv::Point3f q = W[w].mps[p].GetPos();
			op[3*p] = q.x; op[3*p+1] = q.y; op[3*p+2] = q.z;
		}
	}
	return n_ba;
}

// The mapper's loop with outlier removal: as harness_local_mapping's world A, but the local BA of every
// new keyframe from `first_ba` on is LocalMapIndex::OptimizeRejectingOutliers (reject = 1) or Optimize
// (reject = 0).  Slot s carries the ORB octave slot_oct[s]; every frame has the 8-level 1.2 pyramid.
// Outputs: final float poses / points, per slot whether mvpMapPoints ended NULL (slot_null) and whether
// the final Assemble of the last keyframe still holds that observation (slot_assembled), mnObs per point.
// Returns the number of erased observations.
int harness_local_mapping_rejecting(int n_kf, const float* kf_rt, const int* kf_off, const int* slot_pt,
                                    const float* slot_uv, const int* slot_oct, const int* cov_off,
                                    const int* cov_idx, int P, const float* pts, const float* K4, int first_ba,
                                    int reject, float* out_cams, float* out_pts, uint8_t* slot_null,
                                    uint8_t* slot_assembled, int* mnobs)
{
	Camera cam;
	cam.fx = K4[0]; cam.fy = K4[1]; cam.cx = K4[2]; cam.cy = K4[3];
	std::vector<Frame> frames(n_kf);
	std::vector<MapPoint> mps(P);
	for(int p=0;p<P;p++) mps[p].mWorldPos = cv::Point3f(pts[3*p], pts[3*p+1], pts[3*p+2]);
	lorb_host::LocalMapIndex index;
	int n_erased = 0;
	for(int k=0; k<n_kf; k++)
	{
		Frame& F = frames[k];
		F.mpCamera = &cam;
		for(int l=0; l<8; l++) F.mvScaleFactors.push_back(std::pow(1.2f, (float)l));
		cv::Mat R(3,1,CV_32F), T(3,1,CV_32F);
		for(int a=0;a<3;a++) { R.at<float>(a) = kf_rt[6*k+a]; T.at<float>(a) = kf_rt[6*k+3+a]; }
		F.SetPose(T, R);
		for(int s=kf_off[k]; s<kf_off[k+1]; s++)
		{
			cv::KeyPoint kp;
			kp.pt = cv::Point2f(slot_uv[2*s], slot_uv[2*s+1]);
			kp.octave = slot_oct[s];
			F.mvKeysUn.push_back(kp);
			F.mvpMapPoints.push_back(slot_pt[s] >= 0 ? &mps[slot_pt[s]] : static_cast<MapPoint*>(NULL));
		}
		F.mnMapPoints = F.mvKeysUn.size();
		for(int c=cov_off[k]; c<cov_off[k+1]; c++) F.mvpOrderedKeyFrames.push_back(&frames[cov_idx[c]]);
		index.InsertKeyFrame(&F);
		if(k < first_ba)
			continue;
		if(reject)
			n_erased += index.OptimizeRejectingOutliers(&F);
		else
			index.Optimize(&F);
	}
	for(int k=0;k<n_kf;k++)
	{
		for(int a=0;a<3;a++)
		{
			out_cams[6*k+a] = frames[k].mRvec.at<float>(a);
			out_cams[6*k+3+a] = frames[k].mTvec.at<float>(a);
		}
		for(int s=kf_off[k]; s<kf_off[k+1]; s++)
		{
			slot_null[s] = slot_pt[s] >= 0 && frames[k].mvpMapPoints[s - kf_off[k]] == NULL;
			slot_assembled[s] = 0;
		}
	}
	for(int p=0;p<P;p++)
	{
		const cv::Point3f q = mps[p].GetPos();
		out_pts[3*p] = q.x; out_pts[3*p+1] = q.y; out_pts[3*p+2] = q.z;
		mnobs[p] = (int)mps[p].mnObs;
	}
	lorb_host::LocalBAWindow w;
	index.Assemble(&frames[n_kf-1], w);
	for(size_t i=0; i<w.obs_kp.size(); i++)
		slot_assembled[kf_off[w.frames[w.obs_cam[i]] - &frames[0]] + w.obs_kp[i]] = 1;
	for(size_t i=0; i<w.fix_kp.size(); i++)
		slot_assembled[kf_off[w.fix_frame[i] - &frames[0]] + w.fix_kp[i]] = 1;
	return n_erased;
}

// LocalMapIndex on its own (host logic only, no device call): insert the keyframes, then assemble the
// local-BA problem of keyframe `k_ba` and hand its index arrays back.  Same inputs as
// harness_local_mapping; bad_kf / bad_pt flag frames / points whose IsBad() is true.
// out_sizes = {C, P, O, F, frames in index, points in index, observations in index}.
int harness_local_map_assemble(int n_kf, const float* kf_rt, const int* kf_off, const int* slot_pt,
                               const float* slot_uv, const int* cov_off, const int* cov_idx, int P,
                               const float* pts, const uint8_t* bad_kf, const uint8_t* bad_pt, int k_ba,
                               int cap, int* out_window, int* out_points, int* out_obs_cam, int* out_obs_pt,
                               float* out_obs_uv, int* out_fix_pt, float* out_fix_uv, float* out_fix_rt,
                               int* out_sizes)
{
	std::vector<Frame> frames(n_kf);
	std::vector<MapPoint> mps(P);
	for(int p=0;p<P;p++)
	{
		mps[p].mWorldPos = cv::Point3f(pts[3*p], pts[3*p+1], pts[3*p+2]);
		mps[p].mbBadFlag = bad_pt && bad_pt[p];
	}
	lorb_host::LocalMapIndex index;
	for(int k=0; k<n_kf; k++)
	{
		Frame& F = frames[k];
		cv::Mat R(3,1,CV_32F), T(3,1,CV_32F);
		for(int a=0;a<3;a++) { R.at<float>(a) = kf_rt[6*k+a]; T.at<float>(a) = kf_rt[6*k+3+a]; }
		F.SetPose(T, R);
		for(int s=kf_off[k]; s<kf_off[k+1]; s++)
		{
			cv::KeyPoint kp;
			kp.pt = cv::Point2f(slot_uv[2*s], slot_uv[2*s+1]);
			F.mvKeysUn.push_back(kp);
			F.mvpMapPoints.push_back(slot_pt[s] >= 0 ? &mps[slot_pt[s]] : static_cast<MapPoint*>(NULL));
		}
		F.mnMapPoints = F.mvKeysUn.size();
		for(int c=cov_off[k]; c<cov_off[k+1]; c++) F.mvpOrderedKeyFrames.push_back(&frames[cov_idx[c]]);
		index.InsertKeyFrame(&F);
	}
	for(int k=0; k<n_kf; k++) frames[k].mbBadFlag = bad_kf && bad_kf[k];  // culled after insertion
	lorb_host::LocalBAWindow w;
	index.Assemble(&frames[k_ba], w);
	const int C = (int)w.frames.size(), Pw = (int)w.points.size(), O = (int)w.obs_cam.size(), Fx = (int)w.fix_pt.size();
	if(C > cap || Pw > cap || O > cap || Fx > cap) return -1;
	for(int i=0;i<C;i++) out_window[i] = (int)(w.frames[i] - &frames[0]);
	for(int i=0;i<Pw;i++) out_points[i] = (int)(w.points[i] - &mps[0]);
	for(int i=0;i<O;i++)
	{
		out_obs_cam[i] = w.obs_cam[i]; out_obs_pt[i] = w.obs_pt[i];
		out_obs_uv[2*i] = w.obs_uv[2*i]; out_obs_uv[2*i+1] = w.obs_uv[2*i+1];
	}
	for(int i=0;i<Fx;i++)
	{
		out_fix_pt[i] = w.fix_pt[i];
		out_fix_uv[2*i] = w.fix_uv[2*i]; out_fix_uv[2*i+1] = w.fix_uv[2*i+1];
		for(int a=0;a<6;a++) out_fix_rt[6*i+a] = w.fix_rt[6*i+a];
	}
	out_sizes[0] = C; out_sizes[1] = Pw; out_sizes[2] = O; out_sizes[3] = Fx;
	out_sizes[4] = (int)index.NumFrames(); out_sizes[5] = (int)index.NumPoints(); out_sizes[6] = (int)index.NumObservations();
	return 0;
}

// ORBextractor(nfeatures, 1.2, 8, 20, 7)(image, Mat(), keypoints, descriptors) as Frame's
// constructor calls it (reference src/frame.cpp:34-56, 132-133); returns the keypoint count.
// out_pyr_sum[l] = byte sum of mvImagePyramid[l] (the member ComputeStereoMatches reads).
int harness_orb_extract(const uint8_t* img, int w, int h, int nfeatures, int cap, float* kx, float* ky, int* koct,
                        float* kangle, float* kresp, float* ksize, uint8_t* desc, long long* out_pyr_sum)
{
	cv::Mat image(h, w, CV_8U);
	std::memcpy(image.ptr<uint8_t>(), img, (size_t)w*h);
	ORBextractor ex(nfeatures, 1.2f, 8, 20, 7);
	std::vector<cv::KeyPoint> kps;
	cv::Mat d;
	ex(image, cv::Mat(), kps, d);
	const int n = (int)kps.size();
	for(int i = 0; i < n && i < cap; i++)
	{
		kx[i] = kps[i].pt.x; ky[i] = kps[i].pt.y; koct[i] = kps[i].octave; kangle[i] = kps[i].angle;
		kresp[i] = kps[i].response; ksize[i] = kps[i].size;
		std::memcpy(desc + 32*(size_t)i, d.ptr<uint8_t>(i), 32);
	}
	for(int l = 0; l < ex.GetLevels(); l++)
	{
		long long s = 0;
		const cv::Mat& m = ex.mvImagePyramid[l];
		for(int r = 0; r < m.rows; r++)
			for(int c = 0; c < m.cols; c++) s += m.ptr<uint8_t>(r)[c];
		out_pyr_sum[l] = s;
	}
	return n;
}

// Frame::Frame(imgLeft, imgRight, camera) extracts the two images on two freshly started threads
// (reference src/frame.cpp:42-45) with two ORBextractor objects, every frame.  Runs that pattern
// n_frames times; returns the number of GPU contexts the drop-in layer had to create (the pool
// hands the same two back to the new threads) and the last frame's keypoint counts / descriptors.
int harness_stereo_extract_threads(const uint8_t* left, const uint8_t* right, int w, int h, int nfeatures,
                                   int n_frames, int cap, int* n_left, int* n_right, uint8_t* desc_left,
                                   uint8_t* desc_right)
{
	cv::Mat imL(h, w, CV_8U), imR(h, w, CV_8U);
	std::memcpy(imL.ptr<uint8_t>(), left, (size_t)w*h);
	std::memcpy(imR.ptr<uint8_t>(), right, (size_t)w*h);
	const int before = lorb_host::pool().created();
	for(int f = 0; f < n_frames; f++)
	{
		ORBextractor exL(nfeatures, 1.2f, 8, 20, 7), exR(nfeatures, 1.2f, 8, 20, 7);
		std::vector<cv::KeyPoint> kL, kR;
		cv::Mat dL, dR;
		std::thread tl([&]{ exL(imL, cv::Mat(), kL, dL); });
		std::thread tr([&]{ exR(imR, cv::Mat(), kR, dR); });
		tl.join();
		tr.join();
		*n_left = (int)kL.size();
		*n_right = (int)kR.size();
		for(int i = 0; i < *n_left && i < cap; i++) std::memcpy(desc_left + 32*(size_t)i, dL.ptr<uint8_t>(i), 32);
		for(int i = 0; i < *n_right && i < cap; i++) std::memcpy(desc_right + 32*(size_t)i, dR.ptr<uint8_t>(i), 32);
	}
	return lorb_host::pool().created() - before;
}

}  // extern "C"
