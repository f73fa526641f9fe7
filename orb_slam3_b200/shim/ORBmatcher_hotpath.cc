// Replacements for the hot-path ORBmatcher methods (reference src/ORBmatcher.cc) that
// flatten Frame / KeyFrame / MapPoint state into the views of orb_b200.h and
// forward to liborbb200.so.  Build inside the ORB_SLAM3 tree: delete the bodies
// of these methods from src/ORBmatcher.cc (or compile that file with
// -DORB_B200_HOTPATH and guard them) and add this file; signatures are the
// reference's own (include/ORBmatcher.h:43-76).  Syntax-checked against the reference's headers over stand-ins for its third-party libraries
// (tests/test_shim_syntax.py); not linked here -- see INTEGRATION.md.  Pinhole, single camera only (orbb200_gate.h): KannalaBrandt8 rigs
// (monocular too) and the fisheye-stereo branches call the reference bodies kept
// under *_Reference names.
#include <cstring>
#include <memory>
#include <stdexcept>

#include "Frame.h"
#include "KeyFrame.h"
#include "MapPoint.h"
#include "ORBmatcher.h"
#include "orb_b200.h"
#include "orbb200_gate.h"

namespace ORB_SLAM3 {

namespace {

orb_matcher* matcher_for_this_thread() {
  // Tracking and LocalMapping call the matchers from different threads; a handle is not thread-safe
  thread_local std::unique_ptr<orb_matcher, void (*)(orb_matcher*)> m(nullptr, match_destroy);
  if (!m) {
    orb_matcher* h = nullptr;
    if (match_create(0, &h) != ORB_OK) throw std::runtime_error(orb_last_error());
    m.reset(h);
  }
  return m.get();
}

struct FrameArrays {  // storage the view points into
  std::vector<orb_keypoint> keys;
  std::vector<uint8_t> taken;
  orb_frame_view v;
};

template <class F>  // F = Frame or KeyFrame
void fill_common(const F& f, const std::vector<cv::KeyPoint>& keysUn, const std::vector<float>& uRight,
                 const cv::Mat& desc, FrameArrays& a) {
  static_assert(sizeof(cv::KeyPoint) == sizeof(orb_keypoint), "layout");
  a.v.n = (int)keysUn.size();
  a.v.keys = reinterpret_cast<const orb_keypoint*>(keysUn.data());
  a.v.u_right = uRight.empty() ? nullptr : uRight.data();
  a.v.desc = desc.data;  // N x 32, continuous (Frame.cc:222 / ORBextractor _descriptors.create)
  a.v.n_levels = (int)f.mvScaleFactors.size();
  a.v.scale_factors = f.mvScaleFactors.data();
  a.v.level_sigma2 = f.mvLevelSigma2.data();
  a.v.fx = f.fx; a.v.fy = f.fy; a.v.cx = f.cx; a.v.cy = f.cy; a.v.bf = f.mbf; a.v.b = f.mb;
  a.v.kp_taken = a.taken.data();
}

void frame_view(Frame& F, FrameArrays& a) {
  a.taken.assign(F.N, 0);
  for (int i = 0; i < F.N; i++)  // ORBmatcher.cc:88-90 / :1747-1749
    if (F.mvpMapPoints[i] && F.mvpMapPoints[i]->Observations() > 0) a.taken[i] = 1;
  fill_common(F, F.mvKeysUn, F.mvuRight, F.mDescriptors, a);
  a.v.min_x = Frame::mnMinX; a.v.min_y = Frame::mnMinY; a.v.max_x = Frame::mnMaxX; a.v.max_y = Frame::mnMaxY;
  a.v.grid_w_inv = Frame::mfGridElementWidthInv; a.v.grid_h_inv = Frame::mfGridElementHeightInv;
}

struct FeatVecArrays {  // DBoW2::FeatureVector as the CSR of orb_featvec_view
  std::vector<uint32_t> ids;
  std::vector<int32_t> ptr, idx;
  orb_featvec_view v;
};

void featvec_view(const DBoW2::FeatureVector& fv, FeatVecArrays& a) {
  a.ptr.push_back(0);
  for (const auto& kv : fv) {  // std::map: ascending node id
    a.ids.push_back(kv.first);
    for (unsigned int i : kv.second) a.idx.push_back((int32_t)i);
    a.ptr.push_back((int32_t)a.idx.size());
  }
  a.v = orb_featvec_view{(int32_t)a.ids.size(), a.ids.data(), a.ptr.data(), a.idx.data()};
}

// pMP && !pMP->isBad() for every entry of one GetMapPointMatches() snapshot
std::vector<uint8_t> mappoint_ok(const std::vector<MapPoint*>& mps) {
  std::vector<uint8_t> ok(mps.size(), 0);
  for (size_t i = 0; i < mps.size(); i++) ok[i] = mps[i] && !mps[i]->isBad();
  return ok;
}

}  // namespace

// ORBmatcher.cc:2058-2074
int ORBmatcher::DescriptorDistance(const cv::Mat& a, const cv::Mat& b) { return ham_distance(a.data, b.data); }

// ORBmatcher.cc:43-141
int ORBmatcher::SearchByProjection(Frame& F, const vector<MapPoint*>& vpMapPoints, const float th,
                                   const bool bFarPoints, const float thFarPoints) {
  if (!orbb200_gate::gpu_path(F)) return SearchByProjection_Reference(F, vpMapPoints, th, bFarPoints, thFarPoints);
  FrameArrays fa;
  frame_view(F, fa);
  const int n = (int)vpMapPoints.size();
  std::vector<uint8_t> in_view(n), bad(n), has_obs(n), desc((size_t)n * 32);
  std::vector<float> px(n), py(n), pxr(n), vcos(n), depth(n);
  std::vector<int32_t> lvl(n);
  for (int i = 0; i < n; i++) {
    MapPoint* p = vpMapPoints[i];
    in_view[i] = p->mbTrackInView; bad[i] = p->isBad(); has_obs[i] = p->Observations() > 0;
    px[i] = p->mTrackProjX; py[i] = p->mTrackProjY; pxr[i] = p->mTrackProjXR;
    lvl[i] = p->mnTrackScaleLevel; vcos[i] = p->mTrackViewCos; depth[i] = p->mTrackDepth;
    if (in_view[i] && !bad[i]) memcpy(&desc[(size_t)i * 32], p->GetDescriptor().data, 32);
  }
  orb_mappoint_view mv{n, in_view.data(), bad.data(), has_obs.data(), px.data(), py.data(), pxr.data(),
                       lvl.data(), vcos.data(), depth.data(), desc.data()};
  std::vector<int32_t> assign(F.N);
  const int nmatches = match_project_local(matcher_for_this_thread(), &fa.v, &mv, th, mfNNratio, bFarPoints,
                                           thFarPoints, assign.data());
  if (nmatches < 0) throw std::runtime_error(orb_last_error());
  for (int i = 0; i < F.N; i++)
    if (assign[i] >= 0) F.mvpMapPoints[i] = vpMapPoints[assign[i]];  // :129
  return nmatches;
}

// ORBmatcher.cc:1676-1887
int ORBmatcher::SearchByProjection(Frame& CurrentFrame, const Frame& LastFrame, const float th, const bool bMono) {
  if (!orbb200_gate::gpu_path(CurrentFrame)) return SearchByProjection_Reference(CurrentFrame, LastFrame, th, bMono);
  const Sophus::SE3f Tcw = CurrentFrame.GetPose();
  const Eigen::Vector3f twc = Tcw.inverse().translation();
  const Eigen::Vector3f tlc = LastFrame.GetPose() * twc;
  const bool bForward = tlc(2) > CurrentFrame.mb && !bMono;    // :1692
  const bool bBackward = -tlc(2) > CurrentFrame.mb && !bMono;  // :1693
  FrameArrays fa;
  frame_view(CurrentFrame, fa);
  const int n = LastFrame.N;
  std::vector<uint8_t> has_mp(n, 0), has_obs(n, 0), desc((size_t)n * 32);
  std::vector<float> wpos((size_t)n * 3), angle(n);
  std::vector<int32_t> octave(n);
  for (int i = 0; i < n; i++) {
    MapPoint* p = LastFrame.mvpMapPoints[i];
    octave[i] = LastFrame.mvKeys[i].octave;
    angle[i] = LastFrame.mvKeysUn[i].angle;
    if (!p || LastFrame.mvbOutlier[i]) continue;
    has_mp[i] = 1; has_obs[i] = p->Observations() > 0;
    const Eigen::Vector3f x = p->GetWorldPos();
    wpos[3 * i] = x(0); wpos[3 * i + 1] = x(1); wpos[3 * i + 2] = x(2);
    memcpy(&desc[(size_t)i * 32], p->GetDescriptor().data, 32);
  }
  orb_lastframe_view lv{n, has_mp.data(), has_obs.data(), wpos.data(), desc.data(), octave.data(), angle.data()};
  const Eigen::Quaternionf q = Tcw.unit_quaternion();
  const float T[7] = {q.x(), q.y(), q.z(), q.w(), Tcw.translation()(0), Tcw.translation()(1), Tcw.translation()(2)};
  std::vector<int32_t> assign(CurrentFrame.N);
  const int nmatches = match_project_last(matcher_for_this_thread(), &fa.v, &lv, T, bForward, bBackward, th,
                                          mbCheckOrientation, assign.data());
  if (nmatches < 0) throw std::runtime_error(orb_last_error());
  for (int i = 0; i < CurrentFrame.N; i++) {
    if (assign[i] >= 0) CurrentFrame.mvpMapPoints[i] = LastFrame.mvpMapPoints[assign[i]];   // :1772
    else if (assign[i] == -2) CurrentFrame.mvpMapPoints[i] = static_cast<MapPoint*>(NULL);  // :1880
  }
  return nmatches;
}

// ORBmatcher.cc:907-1146
int ORBmatcher::SearchForTriangulation(KeyFrame* pKF1, KeyFrame* pKF2, vector<pair<size_t, size_t> >& vMatchedPairs,
                                       const bool bOnlyStereo, const bool bCoarse) {
  if (!orbb200_gate::gpu_path(pKF1) || !orbb200_gate::gpu_path(pKF2))
    return SearchForTriangulation_Reference(pKF1, pKF2, vMatchedPairs, bOnlyStereo, bCoarse);
  auto kf_view = [](KeyFrame* kf, FrameArrays& a) {
    a.taken.assign(kf->N, 0);
    for (int i = 0; i < kf->N; i++)
      if (kf->GetMapPoint(i)) a.taken[i] = 1;  // :972-977, :1003-1005
    fill_common(*kf, kf->mvKeysUn, kf->mvuRight, kf->mDescriptors, a);
  };
  FrameArrays a1, a2;
  kf_view(pKF1, a1);
  kf_view(pKF2, a2);
  FeatVecArrays f1, f2;
  featvec_view(pKF1->mFeatVec, f1);
  featvec_view(pKF2->mFeatVec, f2);
  // epipole and fundamental matrix exactly as the reference computes them (:914-920, Pinhole.cpp:107-112)
  const Sophus::SE3f T1w = pKF1->GetPose(), T2w = pKF2->GetPose(), Tw2 = pKF2->GetPoseInverse();
  const Eigen::Vector2f ep = pKF2->mpCamera->project(T2w * pKF1->GetCameraCenter());
  const Sophus::SE3f T12 = T1w * Tw2;
  const Eigen::Matrix3f K1 = pKF1->mpCamera->toK_(), K2 = pKF2->mpCamera->toK_();
  const Eigen::Matrix3f F12 = K1.transpose().inverse() * Sophus::SO3f::hat(T12.translation()) *
                              T12.rotationMatrix() * K2.inverse();
  float Frm[9];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) Frm[3 * r + c] = F12(r, c);
  const float epv[2] = {ep(0), ep(1)};
  std::vector<int32_t> pairs(2 * (size_t)pKF1->N + 2);
  const int n = match_triangulate(matcher_for_this_thread(), &a1.v, &a2.v, &f1.v, &f2.v, Frm, epv, bOnlyStereo, bCoarse,
                                  mbCheckOrientation, pairs.data(), pKF1->N + 1);
  if (n < 0) throw std::runtime_error(orb_last_error());
  vMatchedPairs.clear();
  vMatchedPairs.reserve(n);
  for (int i = 0; i < n; i++) vMatchedPairs.push_back(make_pair((size_t)pairs[2 * i], (size_t)pairs[2 * i + 1]));
  return n;
}

// ORBmatcher.cc:223-…  (Tracking::TrackReferenceKeyFrame, Tracking::Relocalization)
int ORBmatcher::SearchByBoW(KeyFrame* pKF, Frame& F, vector<MapPoint*>& vpMapPointMatches) {
  if (!orbb200_gate::gpu_path(pKF) || !orbb200_gate::gpu_path(F))
    return SearchByBoW_Reference(pKF, F, vpMapPointMatches);
  const vector<MapPoint*> vpMapPointsKF = pKF->GetMapPointMatches();  // one snapshot: flags and write-back agree
  const std::vector<uint8_t> ok = mappoint_ok(vpMapPointsKF);
  vpMapPointMatches = vector<MapPoint*>(F.N, static_cast<MapPoint*>(NULL));
  FrameArrays ka, fa;
  fill_common(*pKF, pKF->mvKeysUn, pKF->mvuRight, pKF->mDescriptors, ka);
  fill_common(F, F.mvKeysUn, F.mvuRight, F.mDescriptors, fa);
  FeatVecArrays fk, ff;
  featvec_view(pKF->mFeatVec, fk);
  featvec_view(F.mFeatVec, ff);
  std::vector<int32_t> assign(F.N);
  const int nmatches = match_bow_frame(matcher_for_this_thread(), &ka.v, ok.data(), &fk.v, &fa.v, &ff.v, mfNNratio,
                                       mbCheckOrientation, assign.data());
  if (nmatches < 0) throw std::runtime_error(orb_last_error());
  for (int i = 0; i < F.N; i++)
    if (assign[i] >= 0) vpMapPointMatches[i] = vpMapPointsKF[assign[i]];  // -2: cleared by the rotation check
  return nmatches;
}

// ORBmatcher.cc:765-…  (LoopClosing: loop and merge detection)
int ORBmatcher::SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, vector<MapPoint*>& vpMatches12) {
  if (!orbb200_gate::gpu_path(pKF1) || !orbb200_gate::gpu_path(pKF2))
    return SearchByBoW_Reference(pKF1, pKF2, vpMatches12);
  const vector<MapPoint*> vpMapPoints1 = pKF1->GetMapPointMatches();
  const vector<MapPoint*> vpMapPoints2 = pKF2->GetMapPointMatches();
  const std::vector<uint8_t> ok1 = mappoint_ok(vpMapPoints1), ok2 = mappoint_ok(vpMapPoints2);
  vpMatches12 = vector<MapPoint*>(vpMapPoints1.size(), static_cast<MapPoint*>(NULL));
  FrameArrays a1, a2;
  fill_common(*pKF1, pKF1->mvKeysUn, pKF1->mvuRight, pKF1->mDescriptors, a1);
  fill_common(*pKF2, pKF2->mvKeysUn, pKF2->mvuRight, pKF2->mDescriptors, a2);
  FeatVecArrays f1, f2;
  featvec_view(pKF1->mFeatVec, f1);
  featvec_view(pKF2->mFeatVec, f2);
  std::vector<int32_t> match12(pKF1->N);
  const int nmatches = match_bow_keyframes(matcher_for_this_thread(), &a1.v, ok1.data(), &f1.v, &a2.v, ok2.data(),
                                           &f2.v, mfNNratio, mbCheckOrientation, match12.data());
  if (nmatches < 0) throw std::runtime_error(orb_last_error());
  for (int i = 0; i < pKF1->N; i++)
    if (match12[i] >= 0) vpMatches12[i] = vpMapPoints2[match12[i]];
  return nmatches;
}

}  // namespace ORB_SLAM3
