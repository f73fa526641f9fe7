#!/usr/bin/env python3
"""Writes the reference's include/ tree, WITH the one-line header additions INTEGRATION.md asks a maintainer to make,
into a scratch directory (never into this repo: no reference source is copied here).  tests/test_shim_syntax.py compiles
the shims against the result, so the list of additions in INTEGRATION.md is exercised by a compiler.
usage: apply_header_additions.py <reference root> <out dir>"""
import os
import re
import shutil
import sys


def patch(text, anchor_regex, addition, what):
    m = re.search(anchor_regex, text, flags=re.S)
    if not m:
        raise SystemExit("anchor not found for " + what)
    return text[:m.end()] + "\n" + addition + "\n" + text[m.end():]


def main(ref, out):
    src = os.path.join(ref, "include")
    if os.path.exists(out):
        shutil.rmtree(out)
    shutil.copytree(src, out)
    P = lambda name: os.path.join(out, name)  # noqa: E731

    t = open(P("Optimizer.h")).read()
    t = patch(t, r"void static LocalBundleAdjustment\(KeyFrame\* pKF,[^;]*;",
              "    void static LocalBundleAdjustment_Reference(KeyFrame* pKF, bool *pbStopFlag, Map *pMap, int& num_fixedKF, int &num_OptKF, int &num_MPs, int &num_edges);",
              "LocalBundleAdjustment_Reference")
    t = patch(t, r"int static PoseOptimization\(Frame\* pFrame\);", "    int static PoseOptimization_Reference(Frame* pFrame);",
              "PoseOptimization_Reference")
    t = patch(t, r"void static LocalInertialBA\(KeyFrame\* pKF,[^;]*;",
              "    void static LocalInertialBA_Reference(KeyFrame* pKF, bool *pbStopFlag, Map *pMap, int& num_fixedKF, int& num_OptKF, int& num_MPs, int& num_edges, bool bLarge, bool bRecInit);",
              "LocalInertialBA_Reference")
    open(P("Optimizer.h"), "w").write(t)

    t = open(P("ORBmatcher.h")).read()
    t = patch(t, r"int SearchByProjection\(Frame &F, const std::vector<MapPoint\*> &vpMapPoints,[^;]*;",
              "    int SearchByProjection_Reference(Frame &F, const std::vector<MapPoint*> &vpMapPoints, const float th, const bool bFarPoints, const float thFarPoints);",
              "SearchByProjection_Reference (local map)")
    t = patch(t, r"int SearchByProjection\(Frame &CurrentFrame, const Frame &LastFrame,[^;]*;",
              "    int SearchByProjection_Reference(Frame &CurrentFrame, const Frame &LastFrame, const float th, const bool bMono);",
              "SearchByProjection_Reference (last frame)")
    t = patch(t, r"int SearchForTriangulation\(KeyFrame \*pKF1, KeyFrame\* pKF2,\s*std::vector<pair<size_t, size_t> > &vMatchedPairs, const bool bOnlyStereo, const bool bCoarse[^;]*;",
              "    int SearchForTriangulation_Reference(KeyFrame *pKF1, KeyFrame* pKF2, std::vector<pair<size_t, size_t> > &vMatchedPairs, const bool bOnlyStereo, const bool bCoarse);",
              "SearchForTriangulation_Reference")
    t = patch(t, r"int SearchByBoW\(KeyFrame\s*\*\s*pKF,\s*Frame\s*&\s*F,[^;]*;",
              "    int SearchByBoW_Reference(KeyFrame *pKF, Frame &F, std::vector<MapPoint*> &vpMapPointMatches);",
              "SearchByBoW_Reference (keyframe-frame)")
    t = patch(t, r"int SearchByBoW\(KeyFrame\s*\*\s*pKF1,\s*KeyFrame\s*\*\s*pKF2,[^;]*;",
              "    int SearchByBoW_Reference(KeyFrame *pKF1, KeyFrame* pKF2, std::vector<MapPoint*> &vpMatches12);",
              "SearchByBoW_Reference (keyframe-keyframe)")
    open(P("ORBmatcher.h"), "w").write(t)

    t = open(P("Tracking.h")).read()
    t = patch(t, r"void SearchLocalPoints\(\);", "    void SearchLocalPoints_Reference();", "SearchLocalPoints_Reference")
    open(P("Tracking.h"), "w").write(t)

    t = open(P("MapPoint.h")).read()
    t = patch(t, r"float GetMaxDistanceInvariance\(\);",
              "    float GetMinDistanceRaw() { unique_lock<mutex> lock(mMutexPos); return mfMinDistance; }\n"
              "    float GetMaxDistanceRaw() { unique_lock<mutex> lock(mMutexPos); return mfMaxDistance; }", "GetMin/MaxDistanceRaw")
    open(P("MapPoint.h"), "w").write(t)

    # ORBVocabulary::flatten: TemplatedVocabulary's m_nodes is protected, so the typedef becomes a two-line subclass
    t = open(P("ORBVocabulary.h")).read()
    m = re.search(r"typedef DBoW2::TemplatedVocabulary<DBoW2::FORB::TDescriptor, DBoW2::FORB>\s*ORBVocabulary;", t)
    if not m:
        raise SystemExit("anchor not found for ORBVocabulary")
    t = t[:m.start()] + (
        "struct ORBVocabulary : DBoW2::TemplatedVocabulary<DBoW2::FORB::TDescriptor, DBoW2::FORB> {\n"
        "  using DBoW2::TemplatedVocabulary<DBoW2::FORB::TDescriptor, DBoW2::FORB>::TemplatedVocabulary;\n"
        "  void flatten(int& L, std::vector<int32_t>& child_ptr, std::vector<int32_t>& child_ids, std::vector<uint8_t>& desc,\n"
        "               std::vector<double>& weight, std::vector<int32_t>& word_id) const;\n"
        "};") + t[m.end():]
    open(P("ORBVocabulary.h"), "w").write(t)

    t = open(P("ORBextractor.h")).read()
    t = patch(t, r"class ORBextractor\s*\{.*?\n\};", "void orbb200_release(const ORBextractor* self);", "orbb200_release")
    open(P("ORBextractor.h"), "w").write(t)
    print("patched headers in", out)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
