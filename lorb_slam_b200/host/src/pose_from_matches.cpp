// pose_from_matches.cpp — lorb_host::PoseFromMatches (include/pose_from_matches.h): one-problem
// lorb_pnp_ransac_batched, then lorb_host::PoseOptimization on the surviving matches.  The problem is gathered
// as PoseOptimization gathers it (non-NULL map points in index order, octave weights).
#include "../include/pose_from_matches.h"

#include "../include/pose_optimization.h"
#include "lorb_host.h"

namespace lorb_host
{

int PoseFromMatches(Simple_ORB_SLAM::Frame* pF, int min_inliers)
{
	std::vector<float> xw, uv, info;
	std::vector<size_t> idx;
	for(size_t i=0; i<pF->mnMapPoints; i++)
	{
		Simple_ORB_SLAM::MapPoint* pMP = pF->mvpMapPoints[i];
		if(pMP == NULL)
			continue;
		const cv::Point2f kp2d = pF->GetKp2d(i);
		const cv::Point3f kp3d = pMP->GetPos();
		xw.push_back(kp3d.x); xw.push_back(kp3d.y); xw.push_back(kp3d.z);
		uv.push_back(kp2d.x); uv.push_back(kp2d.y);
		const float s = pF->mvScaleFactors[pF->mvKeysUn[i].octave];
		info.push_back(1.0f / (s * s));
		idx.push_back(i);
	}
	const int n = (int)idx.size();
	const Simple_ORB_SLAM::Camera* cam = pF->mpCamera;
	const float K[4] = {cam->fx, cam->fy, cam->cx, cam->cy};
	lorb_pnp_ransac params;
	lorb_default_pnp_ransac(&params);
	const int off[2] = {0, n};
	double rt[6];
	int best = -1, n_inliers = 0;
	std::vector<uint8_t> inlier(n);
	LORB_HOST_CALL(lorb_pnp_ransac_batched(ctx(), 1, off, xw.data(), uv.data(), info.data(), K, NULL, &params, rt,
	                                       &best, &n_inliers, inlier.data(), NULL));
	if(n_inliers < min_inliers)
		return n_inliers;
	for(int j=0; j<n; j++)
		if(!inlier[j])
			pF->mvpMapPoints[idx[j]] = NULL;
	cv::Mat T(3, 1, CV_32F), R(3, 1, CV_32F);
	for(int k=0; k<3; k++)
	{
		R.at<float>(k) = (float)rt[k];
		T.at<float>(k) = (float)rt[3+k];
	}
	pF->SetPose(T, R);
	return PoseOptimization(pF);
}

}
