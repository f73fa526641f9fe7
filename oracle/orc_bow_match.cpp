// TEST INFRASTRUCTURE ONLY (see orc_common.h).  CPU restatement of the reference's SearchByBoW, both overloads, on
// the flat views of include/orb_b200.h (interface types only; no product code is used).
//
// Restates (paths relative to the reference tree; the end lines are not verified here):
//   src/ORBmatcher.cc:223-…   SearchByBoW(KeyFrame* pKF, Frame& F, vector<MapPoint*>&)         (Nleft == -1, no mpCamera2)
//   src/ORBmatcher.cc:765-…   SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, vector<MapPoint*>&)  (NLeft == -1, no mpCamera2)
// DescriptorDistance and ComputeThreeMaxima are orc_match.cpp's (orc_ham_distance / orc_three_maxima, the same library).
// Float semantics: strict IEEE single, no FMA (-ffp-contract=off).
#include <cmath>
#include <cstdint>
#include <vector>

#include "../include/orb_b200.h"

extern "C" int orc_ham_distance(const uint8_t* a, const uint8_t* b);
extern "C" void orc_three_maxima(const int* sizes, int L, int* ind);

namespace {

const int TH_LOW = 50, HISTO_LENGTH = 30;

// kind 0: (KeyFrame* pKF = Q, Frame& F = Cand), out[F.n] = KF index whose map point lands in vpMapPointMatches[i];
// kind 1: (pKF1 = Q, pKF2 = Cand), out[Q.n] = KF2 index whose map point lands in vpMatches12[i].  -1 untouched,
// -2 cleared by the rotation check.  ok_q / ok_c = GetMapPointMatches()[i] && !isBad() (ok_c: kind 1 only).
int bow_match(int kind, const orb_frame_view* Q, const uint8_t* ok_q, const orb_featvec_view* fvq,
              const orb_frame_view* Cand, const uint8_t* ok_c, const orb_featvec_view* fvc, float nnratio,
              int check_ori, int32_t* out) {
  const int n_out = kind == 0 ? Cand->n : Q->n;
  for (int i = 0; i < n_out; i++) out[i] = -1;                 // vpMapPointMatches / vpMatches12 all NULL
  std::vector<uint8_t> taken(Cand->n, 0);                      // kind 0: vpMapPointMatches[i] != NULL; kind 1: vbMatched2
  std::vector<int> rotHist[HISTO_LENGTH];
  const float factor = 1.0f / HISTO_LENGTH;
  int nmatches = 0;
  int a = 0, b = 0;                                            // KFit / Fit (kind 0), f1it / f2it (kind 1)
  while (a < fvq->n_nodes && b < fvc->n_nodes) {
    if (fvq->node_ids[a] == fvc->node_ids[b]) {
      for (int p1 = fvq->ptr[a]; p1 < fvq->ptr[a + 1]; p1++) {
        const int idx1 = fvq->idx[p1];
        if (!ok_q[idx1]) continue;                             // if(!pMP) continue; if(pMP->isBad()) continue;
        const uint8_t* d1 = Q->desc + (size_t)idx1 * 32;
        int bestDist1 = 256, bestIdx2 = -1, bestDist2 = 256;
        for (int p2 = fvc->ptr[b]; p2 < fvc->ptr[b + 1]; p2++) {
          const int idx2 = fvc->idx[p2];
          if (taken[idx2]) continue;                           // if(vpMapPointMatches[realIdxF]) / if(vbMatched2[idx2] ...
          if (kind == 1 && !ok_c[idx2]) continue;              // ... || !pMP2) continue; if(pMP2->isBad()) continue;
          const int dist = orc_ham_distance(d1, Cand->desc + (size_t)idx2 * 32);
          if (dist < bestDist1) { bestDist2 = bestDist1; bestDist1 = dist; bestIdx2 = idx2; }
          else if (dist < bestDist2) { bestDist2 = dist; }
        }
        const bool pass = kind == 0 ? bestDist1 <= TH_LOW : bestDist1 < TH_LOW;
        if (pass && static_cast<float>(bestDist1) < nnratio * static_cast<float>(bestDist2)) {
          const int rec = kind == 0 ? bestIdx2 : idx1;         // rotHist holds bestIdxF (kind 0) / idx1 (kind 1)
          out[rec] = kind == 0 ? idx1 : bestIdx2;
          taken[bestIdx2] = 1;
          if (check_ori) {
            float rot = Q->keys[idx1].angle - Cand->keys[bestIdx2].angle;
            if (rot < 0.0) rot += 360.0f;
            int bin = (int)std::round(rot * factor);
            if (bin == HISTO_LENGTH) bin = 0;
            rotHist[bin].push_back(rec);
          }
          nmatches++;
        }
      }
      a++; b++;
    } else if (fvq->node_ids[a] < fvc->node_ids[b]) {
      while (a < fvq->n_nodes && fvq->node_ids[a] < fvc->node_ids[b]) a++;  // KFit = vFeatVecKF.lower_bound(Fit->first)
    } else {
      while (b < fvc->n_nodes && fvc->node_ids[b] < fvq->node_ids[a]) b++;  // Fit = F.mFeatVec.lower_bound(KFit->first)
    }
  }
  if (check_ori) {
    int ind[3] = {-1, -1, -1}, sizes[HISTO_LENGTH];
    for (int i = 0; i < HISTO_LENGTH; i++) sizes[i] = (int)rotHist[i].size();
    orc_three_maxima(sizes, HISTO_LENGTH, ind);
    for (int i = 0; i < HISTO_LENGTH; i++) {
      if (i == ind[0] || i == ind[1] || i == ind[2]) continue;
      for (int rec : rotHist[i]) { out[rec] = -2; nmatches--; }
    }
  }
  return nmatches;
}

}  // namespace

extern "C" {

int orc_match_bow_frame(const orb_frame_view* kf, const uint8_t* kf_mp_ok, const orb_featvec_view* fv_kf,
                        const orb_frame_view* F, const orb_featvec_view* fv_f, float nn_ratio, int check_ori,
                        int32_t* assign) {
  return bow_match(0, kf, kf_mp_ok, fv_kf, F, nullptr, fv_f, nn_ratio, check_ori, assign);
}

int orc_match_bow_keyframes(const orb_frame_view* kf1, const uint8_t* mp_ok1, const orb_featvec_view* fv1,
                            const orb_frame_view* kf2, const uint8_t* mp_ok2, const orb_featvec_view* fv2,
                            float nn_ratio, int check_ori, int32_t* match12) {
  return bow_match(1, kf1, mp_ok1, fv1, kf2, mp_ok2, fv2, nn_ratio, check_ori, match12);
}

}  // extern "C"
