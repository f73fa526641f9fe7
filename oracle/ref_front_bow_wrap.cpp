// TEST INFRASTRUCTURE ONLY -- the reference's own ORBmatcher::SearchByBoW, both overloads (ORBmatcher.cc:223-…, :765-…), on
// real KeyFrame / Frame / MapPoint objects, as object code (oracle/_ref/libref_front_bow.so, built by ref_front_bow.mk with
// libref_front.so's recipe).  The objects are filled by ref_front_wrap.cpp's helpers: that translation unit is included
// here, so this library also carries its entry points.  tests/test_ref_bow_match.py holds the oracle (orc_bow_match.cpp)
// against these.  Nothing in the product links this.
#include "ref_front_wrap.cpp"

namespace {
// KeyFrame map points from per-keypoint flags: ok -> a good MapPoint; not ok -> alternately no MapPoint and a bad one
void fill_mappoints(KeyFrame& K, const uint8_t* ok, World& W, std::map<MapPoint*, int>& index) {
  for (int i = 0, miss = 0; i < K.N; i++) {
    if (!ok[i] && (miss++ & 1) == 0) { K.mvpMapPoints[i] = static_cast<MapPoint*>(NULL); continue; }
    MapPoint* p = W.point();
    p->mbBad = !ok[i];
    K.mvpMapPoints[i] = p;
    index[p] = i;
  }
}
const float kIdentity[7] = {0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f};
}  // namespace

extern "C" {

// ORBmatcher(nn_ratio, check_orientation).SearchByBoW(pKF, F, vpMapPointMatches) on a real KeyFrame and Frame.
// assign_out as match_bow_frame, except that a match cleared by the rotation check reads -1 (the vector holds NULL).
int ref_front_bow_frame(const orb_frame_view* kf, const uint8_t* kf_mp_ok, const orb_featvec_view* fv_kf, const orb_frame_view* fv,
                        const orb_featvec_view* fv_f, float nn_ratio, int check_orientation, int32_t* assign_out) {
  World W;
  KeyFrame K;
  Frame F;
  fill_keyframe(K, kf, fv_kf, kIdentity, W);
  std::map<MapPoint*, int> index;
  fill_mappoints(K, kf_mp_ok, W, index);
  fill_frame(F, fv, W);
  for (int k = 0; k < fv_f->n_nodes; k++) {
    std::vector<unsigned int>& f = F.mFeatVec[fv_f->node_ids[k]];
    for (int p = fv_f->ptr[k]; p < fv_f->ptr[k + 1]; p++) f.push_back((unsigned int)fv_f->idx[p]);
  }
  ORBmatcher matcher(nn_ratio, check_orientation != 0);
  std::vector<MapPoint*> matches;
  const int n = matcher.SearchByBoW(&K, F, matches);
  for (int i = 0; i < fv->n; i++) {
    auto it = index.find(matches[i]);
    assign_out[i] = it == index.end() ? -1 : it->second;
  }
  return n;
}

// ORBmatcher(nn_ratio, check_orientation).SearchByBoW(pKF1, pKF2, vpMatches12) on two real KeyFrames; match12_out as
// match_bow_keyframes with -1 in place of -2.
int ref_front_bow_keyframes(const orb_frame_view* kf1, const uint8_t* mp_ok1, const orb_featvec_view* fv1, const orb_frame_view* kf2,
                            const uint8_t* mp_ok2, const orb_featvec_view* fv2, float nn_ratio, int check_orientation,
                            int32_t* match12_out) {
  World W;
  KeyFrame K1, K2;
  fill_keyframe(K1, kf1, fv1, kIdentity, W);
  fill_keyframe(K2, kf2, fv2, kIdentity, W);
  std::map<MapPoint*, int> index1, index2;
  fill_mappoints(K1, mp_ok1, W, index1);
  fill_mappoints(K2, mp_ok2, W, index2);
  ORBmatcher matcher(nn_ratio, check_orientation != 0);
  std::vector<MapPoint*> matches;
  const int n = matcher.SearchByBoW(&K1, &K2, matches);
  for (int i = 0; i < kf1->n; i++) {
    auto it = index2.find(matches[i]);
    match12_out[i] = it == index2.end() ? -1 : it->second;
  }
  return n;
}

}  // extern "C"
