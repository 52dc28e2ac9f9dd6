// pose_optimization.cpp — lorb_host::PoseOptimization (include/pose_optimization.h) over
// lorb_ba_pose_rounds_batched with one frame.  The problem is gathered as BA::ProjectPoseOptimization
// gathers it (non-NULL map points in index order, float pose in and out).
#include "../include/pose_optimization.h"

#include <cmath>

#include "lorb_host.h"

namespace lorb_host
{

int PoseOptimization(Simple_ORB_SLAM::Frame* pFrame)
{
	double rt[6];
	for(int i=0; i<3; i++)
	{
		rt[i] = pFrame->mRvec.at<float>(i);
		rt[3+i] = pFrame->mTvec.at<float>(i);
	}
	std::vector<float> xw, uv, info;
	std::vector<size_t> idx;
	for(size_t i=0; i<pFrame->mnMapPoints; i++)
	{
		Simple_ORB_SLAM::MapPoint* pMP = pFrame->mvpMapPoints[i];
		if(pMP == NULL)
			continue;
		const cv::Point2f kp2d = pFrame->GetKp2d(i);
		const cv::Point3f kp3d = pMP->GetPos();
		xw.push_back(kp3d.x); xw.push_back(kp3d.y); xw.push_back(kp3d.z);
		uv.push_back(kp2d.x); uv.push_back(kp2d.y);
		const float s = pFrame->mvScaleFactors[pFrame->mvKeysUn[i].octave];
		info.push_back(1.0f / (s * s));
		idx.push_back(i);
	}
	const int n = (int)idx.size();
	const Simple_ORB_SLAM::Camera* cam = pFrame->mpCamera;
	const float K[4] = {cam->fx, cam->fy, cam->cx, cam->cy};
	lorb_ba_options opt;
	lorb_ba_default_options(&opt);
	opt.max_num_iterations = 10;
	lorb_ba_pose_rounds rounds;
	lorb_ba_default_pose_rounds(&rounds);
	lorb_ctx* c = ctx();
	lorb_ba_loss prev, huber = {LORB_LOSS_HUBER, 0, std::sqrt(rounds.chi2)};
	LORB_HOST_CALL(lorb_ba_get_loss(c, &prev));
	LORB_HOST_CALL(lorb_ba_set_loss(c, &huber));
	const int off[2] = {0, n};
	std::vector<uint8_t> inlier(n);
	int n_inliers = 0;
	const int rc = lorb_ba_pose_rounds_batched(c, 1, off, xw.data(), uv.data(), info.data(), K, rt, &rounds,
	                                           &opt, inlier.data(), NULL, &n_inliers, NULL, NULL);
	LORB_HOST_CALL(lorb_ba_set_loss(c, &prev));
	if(rc != LORB_OK) die("lorb_ba_pose_rounds_batched", rc);
	cv::Mat T(3, 1, CV_32F), R(3, 1, CV_32F);
	for(int k=0; k<3; k++)
	{
		R.at<float>(k) = (float)rt[k];
		T.at<float>(k) = (float)rt[3+k];
	}
	pFrame->SetPose(T, R);
	if(pFrame->mvbOutlier.size() < pFrame->mnMapPoints)
		pFrame->mvbOutlier.resize(pFrame->mnMapPoints, false);
	for(int j=0; j<n; j++)
		pFrame->mvbOutlier[idx[j]] = !inlier[j];
	return n_inliers;
}

}
