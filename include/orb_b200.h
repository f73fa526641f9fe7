/* orb_b200.h -- C ABI of liborbb200.so, the B200 (sm_100a) replacement for the
 * hot path of UZ-SLAMLab/ORB_SLAM3.  Plain pointers and sizes only; every entry
 * point cites the reference interface it stands in for (paths relative to the
 * reference tree).  The C++ shims in orb_slam3_b200/shim/ keep the reference's
 * class signatures on top of these calls; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - return value: >= 0 success (often a count), < 0 error (ORB_E_*).  There is
 *     no CPU fallback: without a usable CUDA device every compute call fails.
 *   - all buffers are owned by the caller unless stated otherwise.
 *   - a handle owns its CUDA stream and device memory and is NOT thread-safe;
 *     distinct handles may be used concurrently from distinct threads (the
 *     reference runs the left/right extractors on two threads, Frame.cc:122-125).
 */
#ifndef ORB_B200_H_
#define ORB_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORB_OK 0
#define ORB_E_EMPTY (-1)      /* empty image: ORBextractor::operator() returns -1 (ORBextractor.cc:1090) */
#define ORB_E_ARG (-2)        /* bad argument */
#define ORB_E_CUDA (-3)       /* CUDA runtime error, see orb_last_error() */
#define ORB_E_CAPACITY (-4)   /* caller buffer too small (*n tells the need) */
#define ORB_E_NODEVICE (-5)   /* no CUDA device: the engine has no CPU path */
#define ORB_E_NCCL (-6)

/* Same 28-byte layout as cv::KeyPoint. */
typedef struct orb_keypoint {
  float x, y;      /* pt, level-0 pixel coordinates */
  float size;      /* 31 * scale[octave], truncated (ORBextractor.cc:880) */
  float angle;     /* degrees [0,360), IC_Angle (ORBextractor.cc:76-103) */
  float response;  /* FAST score */
  int32_t octave;
  int32_t class_id; /* -1 */
} orb_keypoint;

typedef struct orb_extractor orb_extractor;

const char* orb_version(void);
/* Last error text of the calling thread (also set when a handle call fails). */
const char* orb_last_error(void);
/* Number of CUDA devices visible; 0 when there is none (then every compute call
 * returns ORB_E_NODEVICE). */
int orb_device_count(void);

/* ---- ORBextractor (include/ORBextractor.h:49-83, src/ORBextractor.cc) ---- */

/* ORBextractor::ORBextractor(nfeatures, scaleFactor, nlevels, iniThFAST,
 * minThFAST) (ORBextractor.cc:409-469).  `device` = CUDA ordinal.  Tables are
 * computed on the host exactly as the reference does; no device work happens
 * until the first extract, so creation succeeds without a GPU. */
int orb_create(int nfeatures, float scale_factor, int nlevels, int ini_th_fast, int min_th_fast,
               int device, orb_extractor** out);
void orb_destroy(orb_extractor* h);

/* Getters of ORBextractor.h:61-81.  `out` has nlevels entries. */
int orb_get_levels(const orb_extractor* h);
float orb_get_scale_factor(const orb_extractor* h);
int orb_get_scale_factors(const orb_extractor* h, float* out);
int orb_get_inverse_scale_factors(const orb_extractor* h, float* out);
int orb_get_scale_sigma_squares(const orb_extractor* h, float* out);
int orb_get_inverse_scale_sigma_squares(const orb_extractor* h, float* out);
int orb_get_features_per_level(const orb_extractor* h, int* out);

/* int ORBextractor::operator()(image, mask (ignored), keypoints, descriptors,
 * vLappingArea) (ORBextractor.cc:1086-1168) for one CV_8UC1 image.
 *   img/rows/cols/step : host image (step in bytes)
 *   lap0, lap1         : vLappingArea[0], [1]
 *   kps, desc          : caller buffers for `cap` keypoints / cap*32 bytes
 *   *n                 : total keypoints written (the size of _keypoints)
 * Returns monoIndex (>= 0) like the reference, ORB_E_EMPTY for an empty image. */
int orb_extract(orb_extractor* h, const uint8_t* img, int rows, int cols, size_t step, int lap0,
                int lap1, orb_keypoint* kps, uint8_t* desc, int cap, int* n);

/* The same for `batch` equally sized frames in one submission (a camera stream
 * or the eyes of stereo rigs).  imgs[b] are host pointers (pinned memory makes
 * the copies asynchronous).  Frame b writes kps[b*cap ..], desc[b*cap*32 ..],
 * n[b], mono_index[b].  lap = NULL or 2*batch ints.  Returns batch or < 0. */
int orb_extract_batch(orb_extractor* h, int batch, const uint8_t* const* imgs, int rows, int cols,
                      size_t step, const int* lap, orb_keypoint* kps, uint8_t* desc, int cap, int* n,
                      int* mono_index);

/* Device-resident variant: d_imgs = batch frames already in HBM (frame b at
 * d_imgs + b*frame_stride, row pitch `step`), results stay in HBM.  Runs on the
 * handle's stream, or on `cuda_stream` (a cudaStream_t) when non-NULL.  The results are
 * double-buffered: orb_device_results after call i returns pointers that stay valid (and
 * untouched) until call i + 2 on the handle, so a consumer on another stream may still be
 * reading them while the next batch is extracted. */
int orb_extract_batch_device(orb_extractor* h, int batch, const uint8_t* d_imgs, size_t frame_stride,
                             int rows, int cols, size_t step, const int* lap, void* cuda_stream);
int orb_device_results(orb_extractor* h, const orb_keypoint** d_kps, const uint8_t** d_desc,
                       const int** d_n, const int** d_mono_index, int* cap_per_frame);
/* Copy frame `frame`'s results of the last device-resident batch to host buffers
 * (synchronises the stream).  Returns monoIndex, *n = keypoint count. */
int orb_download_results(orb_extractor* h, int frame, orb_keypoint* kps, uint8_t* desc, int cap, int* n);
/* Block until the work submitted by orb_extract_batch_device has finished. */
int orb_synchronize(orb_extractor* h);

/* Host mirror of ORBextractor::mvImagePyramid (ORBextractor.h:83) for frame
 * `frame` of the last batch: *ptr points at the unpadded level (rows x cols,
 * pitch *step) in engine-owned pinned memory, valid until the next extract.
 * The device->host copy happens on first request per extract. */
int orb_pyramid(orb_extractor* h, int frame, int level, const uint8_t** ptr, int* rows, int* cols,
                size_t* step);

/* ------------------------------------------------------------------------
 * ORBmatcher (include/ORBmatcher.h:43-76, src/ORBmatcher.cc) on flat views.
 * Only the Pinhole single-camera layout (Frame::Nleft == -1) is covered; the
 * fisheye-stereo branches (ORBmatcher.cc:144-210, 1797-1857) are out of scope.
 * TH_HIGH=100, TH_LOW=50, HISTO_LENGTH=30 (ORBmatcher.cc:35-37) are built in.
 * ---------------------------------------------------------------------- */

/* static int ORBmatcher::DescriptorDistance(const cv::Mat&, const cv::Mat&)
 * (ORBmatcher.cc:2058-2074): Hamming distance of two 32-byte descriptors.
 * Host helper (the device kernels use __popc on the same 8 words). */
int ham_distance(const uint8_t* a, const uint8_t* b);

/* The Frame / KeyFrame fields the matchers read (include/Frame.h, KeyFrame.h). */
typedef struct orb_frame_view {
  int32_t n;                    /* N */
  const orb_keypoint* keys;     /* mvKeysUn: pt, octave, angle are read */
  const float* u_right;         /* mvuRight; NULL = monocular (all -1) */
  const uint8_t* desc;          /* mDescriptors, n x 32 */
  float min_x, min_y, max_x, max_y;   /* mnMinX, mnMinY, mnMaxX, mnMaxY */
  float grid_w_inv, grid_h_inv;       /* mfGridElementWidthInv / HeightInv (64 x 48 grid) */
  int32_t n_levels;
  const float* scale_factors;   /* mvScaleFactors */
  const float* level_sigma2;    /* mvLevelSigma2 */
  float fx, fy, cx, cy, bf, b;  /* Pinhole parameters, mbf, mb */
  const uint8_t* kp_taken;      /* per keypoint: mvpMapPoints[i] != NULL && ->Observations() > 0
                                   (SearchByProjection) / GetMapPoint(i) != NULL (SearchForTriangulation); NULL = none */
} orb_frame_view;

/* The MapPoint tracking fields SearchByProjection(Frame&, vector<MapPoint*>&) reads
 * (ORBmatcher.cc:43-141), one entry per element of vpMapPoints. */
typedef struct orb_mappoint_view {
  int32_t n;
  const uint8_t* track_in_view; /* mbTrackInView */
  const uint8_t* is_bad;        /* isBad() */
  const uint8_t* has_obs;       /* Observations() > 0 */
  const float* proj_x;          /* mTrackProjX */
  const float* proj_y;          /* mTrackProjY */
  const float* proj_xr;         /* mTrackProjXR */
  const int32_t* scale_level;   /* mnTrackScaleLevel */
  const float* view_cos;        /* mTrackViewCos */
  const float* depth;           /* mTrackDepth */
  const uint8_t* desc;          /* GetDescriptor(), n x 32 */
} orb_mappoint_view;

/* What SearchByProjection(Frame& Cur, const Frame& Last, ...) reads of LastFrame
 * (ORBmatcher.cc:1695-1733), one entry per last-frame keypoint. */
typedef struct orb_lastframe_view {
  int32_t n;                    /* LastFrame.N */
  const uint8_t* has_mp;        /* mvpMapPoints[i] != NULL && !mvbOutlier[i] */
  const uint8_t* has_obs;       /* that MapPoint's Observations() > 0 */
  const float* world_pos;       /* GetWorldPos(), n x 3 */
  const uint8_t* desc;          /* pMP->GetDescriptor(), n x 32 */
  const int32_t* octave;        /* mvKeys[i].octave */
  const float* angle;           /* mvKeysUn[i].angle */
} orb_lastframe_view;

/* DBoW2::FeatureVector as CSR: node_ids ascending (std::map order),
 * feature indices of node k are idx[ptr[k] .. ptr[k+1]). */
typedef struct orb_featvec_view {
  int32_t n_nodes;
  const uint32_t* node_ids;
  const int32_t* ptr;
  const int32_t* idx;
} orb_featvec_view;

typedef struct orb_matcher orb_matcher;
int match_create(int device, orb_matcher** out);
void match_destroy(orb_matcher* m);

/* int ORBmatcher(nnratio).SearchByProjection(Frame& F, const vector<MapPoint*>&, th,
 * bFarPoints, thFarPoints) (ORBmatcher.cc:43-141).  assign_out[i] (F.n entries) =
 * index into `mps` written to F.mvpMapPoints[i] by this call, or -1 when the
 * call leaves the slot untouched.  Returns nmatches. */
int match_project_local(orb_matcher* m, const orb_frame_view* F, const orb_mappoint_view* mps, float th,
                        float nn_ratio, int far_points, float th_far, int32_t* assign_out);

/* int ORBmatcher(nnratio, checkOri).SearchByProjection(Frame& Cur, const Frame& Last, th,
 * bMono) (ORBmatcher.cc:1676-1887).  Tcw = Cur.GetPose() as Sophus stores it:
 * unit quaternion (x,y,z,w) then translation.  forward/backward are the
 * reference's bForward/bBackward (:1692-1693, computed by the shim).
 * assign_out[i] (Cur.n entries) = index of the last-frame keypoint whose
 * MapPoint ends up in Cur.mvpMapPoints[i]; -1 = untouched; -2 = written and then
 * cleared by the rotation-consistency check (:1875-1884).  Returns nmatches. */
int match_project_last(orb_matcher* m, const orb_frame_view* cur, const orb_lastframe_view* last,
                       const float* Tcw_qt7, int forward, int backward, float th, int check_orientation,
                       int32_t* assign_out);

/* int ORBmatcher(nnratio, checkOri).SearchForTriangulation(KF1, KF2, vMatchedPairs,
 * bOnlyStereo, bCoarse) (ORBmatcher.cc:907-1146), both KFs Pinhole without a
 * second camera.  F12 = K1^-T [t12]x R12 K2^-1 (Pinhole.cpp:107-112, computed by the
 * shim with Eigen), ep = epipole of KF1 in KF2 (:919-920).  pairs_out receives
 * (idx1, idx2) pairs in increasing idx1; returns the pair count (>cap: ORB_E_CAPACITY). */
int match_triangulate(orb_matcher* m, const orb_frame_view* kf1, const orb_frame_view* kf2,
                      const orb_featvec_view* fv1, const orb_featvec_view* fv2, const float* F12_rowmajor9,
                      const float* ep2, int only_stereo, int coarse, int check_orientation,
                      int32_t* pairs_out, int cap);

/* int ORBmatcher(nnratio, checkOri).SearchByBoW(KeyFrame* pKF, Frame& F, vector<MapPoint*>& vpMapPointMatches)
 * (ORBmatcher.cc:223-…), Pinhole without a second camera.  kf_mp_ok[i] (kf.n entries) = pKF->GetMapPointMatches()[i]
 * is non-NULL and !isBad().  Reads keys[].angle and desc of both views; F.kp_taken is not read (the call starts
 * from an all-NULL vpMapPointMatches).  fv_kf / fv_f = pKF->mFeatVec / F.mFeatVec; every feature index must occur in
 * at most one node, as DBoW2::transform makes them.  assign_out[i] (F.n entries) = KF keypoint index whose map point
 * lands in vpMapPointMatches[i], -1 = untouched, -2 = written and then cleared by the rotation check.
 * Returns nmatches (the number of entries >= 0).  Malformed FeatureVectors (node ids not ascending, ptr
 * decreasing, an index outside [0, n) or in two places) are rejected with ORB_E_ARG before any device work. */
int match_bow_frame(orb_matcher* m, const orb_frame_view* kf, const uint8_t* kf_mp_ok, const orb_featvec_view* fv_kf,
                    const orb_frame_view* F, const orb_featvec_view* fv_f, float nn_ratio, int check_orientation,
                    int32_t* assign_out);

/* int ORBmatcher(nnratio, checkOri).SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, vector<MapPoint*>& vpMatches12)
 * (ORBmatcher.cc:765-…), both Pinhole without a second camera.  mp_ok1 / mp_ok2 as kf_mp_ok above, for
 * GetMapPointMatches() of either keyframe.  match12_out[i] (kf1.n entries) = KF2 keypoint index whose map point lands
 * in vpMatches12[i], -1 / -2 as above.  Returns nmatches. */
int match_bow_keyframes(orb_matcher* m, const orb_frame_view* kf1, const uint8_t* mp_ok1, const orb_featvec_view* fv1,
                        const orb_frame_view* kf2, const uint8_t* mp_ok2, const orb_featvec_view* fv2, float nn_ratio,
                        int check_orientation, int32_t* match12_out);

/* Batched forms: `count` independent problems in one submission (frames of a
 * stream, keyframe pairs).  on_device = 0: all views are host memory.  on_device = 1: every pointer inside the
 * views (and the outputs) is a device pointer and nothing is copied.  on_device = 2 (projection matchers):
 * only keys / u_right / desc of the frame views are device pointers -- the device results of an extractor
 * (orb_device_results), so the keypoints and descriptors of a frame that was just extracted are not uploaded
 * again -- everything else, assign_out included, is host memory.  results[k] = per-problem return value. */
int match_project_last_batch(orb_matcher* m, int count, const orb_frame_view* cur, const orb_lastframe_view* last,
                             const float* Tcw_qt7, const int32_t* forward, const int32_t* backward, float th,
                             int check_orientation, int32_t* const* assign_out, int32_t* results, int on_device);
int match_project_local_batch(orb_matcher* m, int count, const orb_frame_view* F, const orb_mappoint_view* mps,
                              float th, float nn_ratio, int far_points, float th_far, int32_t* const* assign_out,
                              int32_t* results, int on_device);
int match_triangulate_batch(orb_matcher* m, int count, const orb_frame_view* kf1, const orb_frame_view* kf2,
                            const orb_featvec_view* fv1, const orb_featvec_view* fv2, const float* F12_rowmajor9,
                            const float* ep2, int only_stereo, int coarse, int check_orientation,
                            int32_t* const* pairs_out, int cap, int32_t* results, int on_device);
/* SearchByBoW batches: Relocalization (one frame against each candidate keyframe) and loop / merge detection (one
 * keyframe pair per covisible keyframe).  Problem k reads kf_mp_ok[k] / mp_ok1[k] / mp_ok2[k] and writes
 * assign_out[k] / match12_out[k]; results[k] = its nmatches.  on_device = 1: every array, the FeatureVectors' and the
 * outputs included, is device memory (the FeatureVectors are then not checked: they must be well formed).
 * on_device = 2 (match_bow_frame_batch only): the frames' keys / desc are an extractor's device results, everything
 * else is host memory.  Repeating one frame view in several problems stages it once.  Returns count or ORB_E_*. */
int match_bow_frame_batch(orb_matcher* m, int count, const orb_frame_view* kf, const uint8_t* const* kf_mp_ok,
                          const orb_featvec_view* fv_kf, const orb_frame_view* F, const orb_featvec_view* fv_f,
                          float nn_ratio, int check_orientation, int32_t* const* assign_out, int32_t* results,
                          int on_device);
int match_bow_keyframes_batch(orb_matcher* m, int count, const orb_frame_view* kf1, const uint8_t* const* mp_ok1,
                              const orb_featvec_view* fv1, const orb_frame_view* kf2, const uint8_t* const* mp_ok2,
                              const orb_featvec_view* fv2, float nn_ratio, int check_orientation,
                              int32_t* const* match12_out, int32_t* results, int on_device);
/* Submit subsequent batches on `cuda_stream` (a cudaStream_t) instead of the
 * matcher's own stream, e.g. the stream an extractor ran on; NULL restores it. */
int match_set_stream(orb_matcher* m, void* cuda_stream);
/* Asynchronous mode for device-resident batches (on_device = 1): the *_batch call returns after
 * enqueueing; `results` (which must stay valid) and the device outputs are complete after
 * match_synchronize() or the next batch on the same handle.  A candidate-buffer overflow is handled inside
 * that call: the budget is grown and the batch is run again from the inputs still staged on the device. */
int match_set_async(orb_matcher* m, int enabled);
int match_synchronize(orb_matcher* m);
long long match_kernel_launches(const orb_matcher* m);
/* Device time of the last batch (CUDA events on the matcher's stream), ms. */
double match_last_ms(orb_matcher* m);

/* ------------------------------------------------------------------------
 * Optimizer::LocalBundleAdjustment (src/Optimizer.cc:1116-1498): the g2o
 * Levenberg-Marquardt loop `optimizer.optimize(10)` (:1410-1411) on a flat graph.
 * The shim keeps steps 1-4 (collecting KFs/MPs/edges, :1119-1400) and 6-7
 * (outlier erase, write-back under Map::mMutexMapUpdate, :1413-1497).
 * Mono (EdgeSE3ProjectXYZ, Pinhole or KannalaBrandt8 camera), stereo
 * (g2o::EdgeStereoSE3ProjectXYZ) and second-camera (EdgeSE3ProjectXYZToBody,
 * src/OptimizableTypes.cpp:192-213, edges of :1366-1400) edges.
 * ---------------------------------------------------------------------- */
#define ORB_CAM_PINHOLE 0 /* GeometricCamera::CAM_PINHOLE */
#define ORB_CAM_KB8 1     /* GeometricCamera::CAM_FISHEYE (KannalaBrandt8) */
#define LBA_EDGE_MONO 0   /* EdgeSE3ProjectXYZ, obs = kpUn.pt (:1305-1331) */
#define LBA_EDGE_STEREO 1 /* g2o::EdgeStereoSE3ProjectXYZ, obs = kpUn.pt, mvuRight (:1332-1364) */
#define LBA_EDGE_BODY 2   /* EdgeSE3ProjectXYZToBody, obs = mvKeysRight[rightIndex].pt (:1366-1400) */
typedef struct lba_graph_view {
  int32_t n_kf;               /* local + fixed keyframes */
  const double* kf_pose;      /* n_kf x 7: g2o::SE3Quat(Tcw): quaternion x,y,z,w then translation (:1217, :1236) */
  const uint8_t* kf_fixed;    /* vSE3->setFixed() (:1219, :1238) */
  const float* kf_cam;        /* n_kf x 5: fx, fy, cx, cy, mbf of the KF's Pinhole camera */
  int32_t n_mp;
  const double* mp_pos;       /* n_mp x 3, VertexSBAPointXYZ estimates (:1285) */
  int32_t n_edges;
  const int32_t* e_kf;        /* index into kf arrays */
  const int32_t* e_mp;        /* index into mp arrays */
  const uint8_t* e_stereo;    /* LBA_EDGE_MONO / LBA_EDGE_STEREO / LBA_EDGE_BODY */
  const double* e_obs;        /* n_edges x 3: pt.x, pt.y, mvuRight (third entry ignored unless LBA_EDGE_STEREO) */
  const float* e_inv_sigma2;  /* mvInvLevelSigma2[octave] */
  /* Rig extension; every pointer may be NULL (= all keyframes carry one Pinhole camera, as above). */
  const uint8_t* kf_cam_model;  /* n_kf: ORB_CAM_* of pKFi->mpCamera (e->pCamera of the mono edges, :1326) */
  const float* kf_cam_dist;     /* n_kf x 4: KannalaBrandt8 k0..k3 = mvParameters[4..7]; read for ORB_CAM_KB8 only */
  const uint8_t* kf_cam2_model; /* n_kf: ORB_CAM_* of pKFi->mpCamera2 (e->pCamera of the body edges, :1387) */
  const float* kf_cam2;         /* n_kf x 8: fx, fy, cx, cy, k0..k3 of mpCamera2 */
  const double* kf_trl;         /* n_kf x 7: g2o::SE3Quat(GetRelativePoseTrl()) = quaternion x,y,z,w + translation (:1384-1385);
                                 * required when any edge is LBA_EDGE_BODY */
} lba_graph_view;

typedef struct lba_stats {
  int32_t iterations;         /* outer LM iterations executed (return value of optimize()) */
  int32_t trials;             /* total lambda trials (linear solves), incl. rejected ones */
  int32_t stopped;            /* 1 when *stop ended the loop */
  double chi2_initial, chi2_final, lambda_final;
  double ms_total;            /* device time of the whole solve (CUDA events) */
  double ms_linearize, ms_schur, ms_solve, ms_update;   /* accumulated per stage */
  int32_t n_free_kf, n_pairs;
  double schur_flops;         /* block-sparse useful flops per trial (SURVEY.md 8d) */
  int32_t solver_kind;        /* reduced solve: 0 = dense cooperative LDL^T (all SMs), 1 = envelope LDL^T, 32-column panels
                               * (one CTA), 2 = window-resident envelope LDL^T, 8-column panels (one CTA, shared memory),
                               * 3 = the same from both ends at once (two CTAs + a dense separator block) */
  int32_t envelope_rows_max;  /* tallest panel window of the row envelope of S (rows) */
  double ms_host_prep;        /* host wall time before the first kernel: edge sort, CSRs, pair lists, ordering, uploads queued */
  double ms_wall;             /* host wall time of the whole call (prep + H2D + kernels + D2H + un-sort) */
  double allreduce_bytes_per_trial; /* bytes each rank contributes to the per-trial ncclAllReduce (0 on one GPU) */
} lba_stats;

typedef struct lba_solver lba_solver;
int lba_create(int device, lba_solver** out);
void lba_destroy(lba_solver* s);
/* Multi-GPU: landmarks (with their edges) are sharded over `world` ranks, poses
 * replicated; one ncclAllReduce(sum, fp64) of [S, b_schur, chi2] per trial.
 * unique_id = the 128 bytes of ncclGetUniqueId from rank 0 (lba_nccl_unique_id). */
int lba_nccl_unique_id(void* out128);
int lba_comm_init(lba_solver* s, int rank, int world, const void* unique_id128);

/* Runs optimize(max_iters) (reference: 10).  lambda_init <= 0 selects g2o's
 * tau*max(diag H) (tau = 1e-5); > 0 is setUserLambdaInit (100 for inertial maps,
 * Optimizer.cc:1197-1198).  `stop` is polled between trials like
 * SparseOptimizer::terminate(); NULL = never.  Outputs (caller buffers):
 *   kf_pose_out n_kf x 7, mp_pos_out n_mp x 3,
 *   chi2_out n_edges      e->chi2() as the reference reads it after optimize()
 *                          (errors of the last evaluated trial, :1423-1460),
 *   depth_pos_out n_edges  e->isDepthPositive() at the final estimates.
 * With a communicator, the graph view holds this rank's landmark shard and all
 * keyframes; outputs cover the shard.  Returns iterations or < 0. */
int lba_solve(lba_solver* s, const lba_graph_view* g, const volatile uint8_t* stop, int max_iters,
              double lambda_init, double* kf_pose_out, double* mp_pos_out, double* chi2_out,
              uint8_t* depth_pos_out, lba_stats* stats);
long long lba_kernel_launches(const lba_solver* s);
/* Measurement helper: dense fp64 tensor-pipe peak (DMMA m8n8k4 issued from registers by a full grid, best of
 * `reps` launches, CUDA events) in TFLOP/s -- the denominator of the Schur roofline in bench.py. */
int lba_measure_fp64_mma_peak(int device, int reps, double* tflops_out);
/* Host-only test hook: the plan of the two-sided reduced solve (solver_kind 3) for a row envelope -- env_reach[c] =
 * last row whose envelope holds a column <= c.  out9 = ok, m, e2, p0, p1, w, R0, R1, WIN_ROWS; first1 / reach1
 * (n ints each, may be NULL) = side 1's tables.  No device needed. */
int lba_debug_two_sided_plan(int n, const int* env_reach, int* out9, int* first1_out, int* reach1_out);

/* ------------------------------------------------------------------------
 * void Frame::ComputeStereoMatches() (src/Frame.cc:811-981), SURVEY.md 8(f-1).
 * Works on what the two extractor handles left on the device after their last
 * extract (mvKeys / mDescriptors / mvImagePyramid of mpORBextractorLeft and
 * mpORBextractorRight): frame i of the left batch is matched against frame i of
 * the right batch.  bf = Frame::mbf, b = Frame::mb.  Outputs per frame:
 * u_right[cap] = mvuRight, depth[cap] = mvDepth (-1 where there is no stereo
 * match), for the left handle's keypoints in their output order.
 * Where the reference is undefined (no left keypoint survives to the median
 * test, Frame.cc:969) every output is -1.
 * ---------------------------------------------------------------------- */
typedef struct orb_stereo orb_stereo;
int stereo_create(int device, orb_stereo** out);
void stereo_destroy(orb_stereo* h);
/* One stereo pair (frame 0 of both handles), host outputs.  Returns the number of
 * keypoints with a stereo match, or ORB_E_*. */
int stereo_match(orb_stereo* h, orb_extractor* left, orb_extractor* right, float bf, float b, float* u_right,
                 float* depth, int cap);
/* `batch` pairs.  on_device = 0: u_right / depth are host arrays of batch x cap floats, kept[batch]
 * (optional) receives the match counts, the call returns after the copy.  on_device = 1: results stay
 * on the device (stereo_device_results), the call only enqueues work on cuda_stream (NULL = the left
 * handle's stream) after both extractions.  Returns batch or ORB_E_*. */
int stereo_match_batch(orb_stereo* h, orb_extractor* left, orb_extractor* right, int batch, float bf, float b,
                       float* u_right, float* depth, int cap, int* kept, int on_device, void* cuda_stream);
int stereo_device_results(orb_stereo* h, const float** d_u_right, const float** d_depth, const int** d_kept,
                          int* stride);
long long stereo_kernel_launches(const orb_stereo* h);
float stereo_last_ms(orb_stereo* h); /* device time of the last call (CUDA events), waits for it */

/* ------------------------------------------------------------------------
 * int Optimizer::PoseOptimization(Frame* pFrame) (src/Optimizer.cc:814-1115),
 * SURVEY.md 8(f-2): motion-only bundle adjustment of one frame pose against its
 * matched MapPoints -- 4 rounds of g2o Levenberg-Marquardt optimize(10), each
 * restarted from the frame pose, with chi2 re-classification (5.991 / 7.815)
 * between rounds and the Huber kernel dropped for the last round.  fp64.
 * Only the Pinhole single-camera layout (!pFrame->mpCamera2) is covered.
 * One edge per keypoint i with mvpMapPoints[i] != NULL, in keypoint order.
 * ---------------------------------------------------------------------- */
typedef struct pose_opt_view {
  int32_t n;               /* number of edges (nInitialCorrespondences) */
  const float* xw;         /* n x 3: pMP->GetWorldPos() */
  const float* obs;        /* n x 3: mvKeysUn[i].pt.x, .pt.y, mvuRight[i] (< 0: monocular edge) */
  const float* inv_sigma2; /* n: mvInvLevelSigma2[mvKeysUn[i].octave] */
  float fx, fy, cx, cy, bf;/* Frame::fx, fy, cx, cy, mbf */
  double pose[7];          /* pFrame->GetPose(): unit quaternion (x,y,z,w) + translation */
} pose_opt_view;

typedef struct orb_poseopt orb_poseopt;
int poseopt_create(int device, orb_poseopt** out);
void poseopt_destroy(orb_poseopt* h);
/* pose_out[7]: optimised Tcw (quaternion xyzw + translation; the shim casts to float for
 * Frame::SetPose); outlier_out[n] = mvbOutlier of the edges.  Returns
 * nInitialCorrespondences - nBad (0 and an untouched pose when n < 3), or ORB_E_*. */
int pose_optimize(orb_poseopt* h, const pose_opt_view* v, double* pose_out, uint8_t* outlier_out);
/* `batch` independent frames, one CTA each, one kernel launch.  pose_out: batch x 7;
 * outlier_out[k]: n_k flags; inliers_out[batch].  stats_out (optional): batch x 3 ints =
 * rounds run, LM iterations, LM trials.  Returns batch or ORB_E_*. */
int pose_optimize_batch(orb_poseopt* h, int batch, const pose_opt_view* views, double* pose_out,
                        uint8_t* const* outlier_out, int* inliers_out, int* stats_out);
long long poseopt_kernel_launches(const orb_poseopt* h);
float poseopt_last_ms(orb_poseopt* h); /* device time of the last call (CUDA events) */

/* ------------------------------------------------------------------------
 * bool Frame::isInFrustum(MapPoint* pMP, float viewingCosLimit) (src/Frame.cc:512-570,
 * the Nleft == -1 branch) with MapPoint::PredictScale (src/MapPoint.cc:531-546),
 * SURVEY.md 8(f-3): the producer of the mbTrackInView / mTrackProj* / mnTrackScaleLevel /
 * mTrackViewCos / mTrackDepth fields that SearchByProjection(Frame&, vector<MapPoint*>&)
 * consumes (orb_mappoint_view above).  One call tests all local map points of a frame
 * (Tracking::SearchLocalPoints, src/Tracking.cc:3367-3390).
 * ---------------------------------------------------------------------- */
typedef struct orb_frustum_view {
  int32_t n;               /* map points */
  const float* world_pos;  /* n x 3: GetWorldPos() */
  const float* normal;     /* n x 3: GetNormal() */
  const float* min_dist;   /* n: mfMinDistance (GetMinDistanceInvariance() = 0.8f * this) */
  const float* max_dist;   /* n: mfMaxDistance (GetMaxDistanceInvariance() = 1.2f * this) */
  float Rcw[9];            /* Frame::mRcw, row-major */
  float tcw[3];            /* Frame::mtcw */
  float Ow[3];             /* Frame::mOw */
  float fx, fy, cx, cy, bf;
  float min_x, max_x, min_y, max_y; /* Frame::mnMinX .. mnMaxY */
  float log_scale_factor;  /* Frame::mfLogScaleFactor = log(mfScaleFactor) as float */
  int32_t n_levels;        /* Frame::mnScaleLevels */
} orb_frustum_view;

typedef struct orb_frustum orb_frustum;
int frustum_create(int device, orb_frustum** out);
void frustum_destroy(orb_frustum* h);
/* Host outputs, n entries each.  track_in_view, proj_x, proj_y are always written (the reference
 * resets mTrackProjX/Y to -1 and overwrites them once the projection is inside the image);
 * proj_xr, scale_level, view_cos, depth are written only where track_in_view = 1 -- elsewhere the
 * caller's values stay, like the stale MapPoint members of the reference.  Returns the number of
 * points in view, or ORB_E_*. */
int frame_is_in_frustum(orb_frustum* h, const orb_frustum_view* v, float viewing_cos_limit, uint8_t* track_in_view,
                        float* proj_x, float* proj_y, float* proj_xr, int32_t* scale_level, float* view_cos,
                        float* depth);
/* Enqueue-only variant for device-resident chaining: the SoA results stay on the device in the layout
 * of orb_mappoint_view's fields (frustum_device_results), on cuda_stream (NULL = the handle's). */
int frame_is_in_frustum_device(orb_frustum* h, const orb_frustum_view* v, float viewing_cos_limit, void* cuda_stream);
int frustum_device_results(orb_frustum* h, const uint8_t** d_track_in_view, const float** d_proj_x,
                           const float** d_proj_y, const float** d_proj_xr, const int32_t** d_scale_level,
                           const float** d_view_cos, const float** d_depth, const int32_t** d_count);
long long frustum_kernel_launches(const orb_frustum* h);
float frustum_last_ms(orb_frustum* h);
/* The kernel's per-point body executed on the host (same source, csrc/frustum_core.h) -- a debug hook
 * for the CPU tests, not a product path: needs no device and is not used by any caller of this library. */
int frustum_debug_host(const orb_frustum_view* v, float viewing_cos_limit, uint8_t* track_in_view, float* proj_x,
                       float* proj_y, float* proj_xr, int32_t* scale_level, float* view_cos, float* depth);

/* ------------------------------------------------------------------------
 * void Frame::ComputeBoW() / KeyFrame::ComputeBoW() (src/Frame.cc:738-745): DBoW2's
 * TemplatedVocabulary<FORB::TDescriptor, FORB>::transform(features, BowVector&, FeatureVector&,
 * levelsup = 4) (Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1127-1195, :1218-1258; FORB::distance
 * FORB.cpp:81-101; BowVector.cpp:34-84; FeatureVector.cpp:31-45), SURVEY.md 8(f-4).
 * Covered: the ORB vocabulary's configuration -- TF_IDF (or TF) weighting with L1 scoring.
 * The vocabulary is uploaded once and stays resident.  Outputs are the two std::maps flattened in
 * key order; the FeatureVector comes out as the CSR that match_triangulate reads (orb_featvec_view).
 * ---------------------------------------------------------------------- */
typedef struct orb_vocab_view {
  int32_t n_nodes;          /* m_nodes.size(); node 0 is the root */
  int32_t L;                /* m_L, depth levels */
  const int32_t* child_ptr; /* n_nodes + 1: CSR over m_nodes[i].children, in that vector's order */
  const int32_t* child_ids; /* child node ids */
  const uint8_t* desc;      /* n_nodes x 32: m_nodes[i].descriptor (the root's row is unused) */
  const double* weight;     /* n_nodes: m_nodes[i].weight */
  const int32_t* word_id;   /* n_nodes: m_nodes[i].word_id for leaves (nodes without children) */
} orb_vocab_view;

typedef struct orb_vocab orb_vocab;
int vocab_create(int device, const orb_vocab_view* v, orb_vocab** out);
void vocab_destroy(orb_vocab* h);
/* desc: n x 32 host descriptors (Converter::toDescriptorVector(mDescriptors)).
 * BowVector:     bow_ids[cap_words] ascending WordId, bow_vals[cap_words] (L1-normalised), *n_words.
 * FeatureVector: fv_node_ids[cap_words] ascending NodeId, fv_ptr[cap_words + 1], fv_idx[n] feature indices
 *                (ascending inside a node), *n_fv_nodes.  cap_words >= n is always enough.
 * Any n: up to 8192 features the per-frame sort runs in one CTA's shared memory, larger frames (monocular
 * initialisation: 5 x nFeatures) sort in global-memory scratch.
 * Returns the number of features that contributed (weight > 0), or ORB_E_*. */
int bow_transform(orb_vocab* h, const uint8_t* desc, int n, int levelsup, int32_t* bow_ids, double* bow_vals,
                  int32_t* n_words, int32_t* fv_node_ids, int32_t* fv_ptr, int32_t* fv_idx, int32_t* n_fv_nodes,
                  int cap_words);
/* Same, for frame `frame` of what an extractor handle left on the device after its last extract
 * (no descriptor upload). */
int bow_transform_extracted(orb_vocab* h, orb_extractor* ex, int frame, int levelsup, int32_t* bow_ids,
                            double* bow_vals, int32_t* n_words, int32_t* fv_node_ids, int32_t* fv_ptr,
                            int32_t* fv_idx, int32_t* n_fv_nodes, int cap_words);
long long bow_kernel_launches(const orb_vocab* h);
float bow_last_ms(orb_vocab* h);
/* The kernels' source (csrc/bow_core.h) executed single-threaded on the host -- a debug hook for the
 * CPU tests, not a product path. */
int bow_debug_host(const orb_vocab_view* v, const uint8_t* desc, int n, int levelsup, int32_t* bow_ids,
                   double* bow_vals, int32_t* n_words, int32_t* fv_node_ids, int32_t* fv_ptr, int32_t* fv_idx,
                   int32_t* n_fv_nodes, int cap_words);

/* ------------------------------------------------------------------------
 * void Optimizer::LocalInertialBA(KeyFrame*, bool* pbStopFlag, Map*, ..., bool bLarge, bool bRecInit)
 * (src/Optimizer.cc:2383-2958), SURVEY.md 8(f-4b): the optimizer.optimize(opt_it) in the middle --
 * g2o Levenberg-Marquardt (user lambda) over VertexPose (ImuCamPose) / VertexVelocity / VertexGyroBias /
 * VertexAccBias and marginalised map points with EdgeMono / EdgeStereo / EdgeInertial / EdgeGyroRW /
 * EdgeAccRW (src/G2oTypes.cc).  Graph set-up, outlier erasure and write-back stay in the shim, like for
 * LocalBundleAdjustment.  One camera per keyframe (no mpCamera2).  fp64.
 * STATUS: the per-window source (csrc/lia_core.h) is held against the oracle on the host
 * (lia_debug_host); the single-launch device path is validated against the oracle on the B200.
 * ---------------------------------------------------------------------- */
typedef struct lia_graph_view {
  /* keyframes: vpOptimizableKFs (newest first), then lFixedKeyFrames */
  int32_t n_kf;
  const double* kf_Rwb;      /* n_kf x 9 row-major: GetImuRotation().cast<double>() */
  const double* kf_twb;      /* n_kf x 3: GetImuPosition() */
  const double* kf_Rcw;      /* n_kf x 9: GetRotation() (left camera) */
  const double* kf_tcw;      /* n_kf x 3: GetTranslation() */
  const uint8_t* kf_fixed;   /* VertexPose (and the IMU vertices) fixed */
  const uint8_t* kf_has_imu; /* KeyFrame::bImu: velocity / gyro-bias / acc-bias vertices exist */
  const double* kf_vel;      /* n_kf x 3: GetVelocity() */
  const double* kf_bg;       /* n_kf x 3: GetGyroBias() */
  const double* kf_ba;       /* n_kf x 3: GetAccBias() */
  double Rcb[9], tcb[3], tbc[3]; /* mImuCalib.mTcb / mTbc (one rig) */
  float fx, fy, cx, cy, bf;
  /* map points and visual edges (EdgeMono / EdgeStereo, left camera) */
  int32_t n_mp;
  const double* mp_pos;      /* n_mp x 3 */
  int32_t n_edges;
  const int32_t* e_kf;
  const int32_t* e_mp;
  const uint8_t* e_stereo;
  const double* e_obs;       /* n_edges x 3: u, v, uRight */
  const float* e_inv_sigma2; /* mvInvLevelSigma2[octave] / uncertainty2 */
  /* inertial edges: EdgeInertial + EdgeGyroRW + EdgeAccRW between kf1 (previous) and kf2 */
  int32_t n_inertial;
  const int32_t* i_kf1;
  const int32_t* i_kf2;
  const float* i_dR;         /* x 9: IMU::Preintegrated::dR, then dV, dP (x 3 each) */
  const float* i_dV;
  const float* i_dP;
  const float* i_JRg;        /* x 9 each: bias Jacobians of the preintegration */
  const float* i_JVg;
  const float* i_JVa;
  const float* i_JPg;
  const float* i_JPa;
  const float* i_bias;       /* x 6: linearisation bias b = (bax, bay, baz, bwx, bwy, bwz) */
  const float* i_dT;         /* integrated time */
  const float* i_C;          /* x 225: 15x15 covariance, row-major */
  const uint8_t* i_last;     /* i == N-1: Huber(sqrt(16.92)) and information * 1e-2 (:2585-2596) */
  double lambda_init;        /* setUserLambdaInit: 1e0, or 1e-2 when bLarge */
  int32_t iterations;        /* opt_it: 10, or 4 when bLarge */
} lia_graph_view;

typedef struct orb_lia orb_lia;
int lia_create(int device, orb_lia** out);
void lia_destroy(orb_lia* h);
/* kf_out: n_kf x 21 doubles (Rcw 9 row-major, tcw 3, velocity 3, gyro bias 3, acc bias 3); mp_out: n_mp x 3;
 * chi2_out / depth_pos_out: per visual edge (e->chi2(), isDepthPositive()); stats[8]: iterations, trials,
 * activeRobustChi2 before (err) and after (err_end), final lambda, pose-side dimension, 2 reserved.
 * Returns the number of LM iterations or ORB_E_*. */
int lia_solve(orb_lia* h, const lia_graph_view* g, double* kf_out, double* mp_out, double* chi2_out,
              uint8_t* depth_pos_out, double* stats);
long long lia_kernel_launches(const orb_lia* h);
float lia_last_ms(orb_lia* h);
/* csrc/lia_core.h executed single-threaded on the host -- a debug hook for the CPU tests, not a product path. */
int lia_debug_host(const lia_graph_view* g, double* kf_out, double* mp_out, double* chi2_out,
                   uint8_t* depth_pos_out, double* stats);

/* Per-stage device timing (CUDA events on the launching stream).  Stages:
 * 0 h2d, 1 pyramid, 2 fast, 3 octree, 4 blur, 5 layout, 6 orient+describe,
 * 7 d2h.  orb_stage_times fills ms[8] (accumulated) and launches[8]. */
#define ORB_NUM_STAGES 8
int orb_set_profiling(orb_extractor* h, int enabled);
int orb_stage_times(orb_extractor* h, double* ms, long long* launches, int reset);
const char* orb_stage_name(int stage);
/* Kernel launches issued by the handle since creation (the gpu_launches claim of bench.py). */
long long orb_kernel_launches(const orb_extractor* h);

/* Intermediate results of the last batch, for the parity tests: raw FAST
 * candidates handed to the octree for (frame, level): x,y relative to the
 * 16-px border (ORBextractor.cc:863-868) and score; returns the count. */
int orb_debug_candidates(orb_extractor* h, int frame, int level, int* xys, int cap);
/* Host execution of the array octree formulation (no GPU needed). */
int orb_debug_octree_host(const int* xys, int n, int band_w, int band_h, int n_features, int w_cell,
                          int h_cell, int n_cols, int* out_xys, int out_cap);
/* Host execution of the libstdc++ introsort emulation: perm_out[i] = input index. */
int orb_debug_introsort(const int* count, const int* ulx, int n, int* perm_out);
/* the same permutation from the level-synchronous form the octree CTA runs (csrc/introsort_emul.h) */
int orb_debug_introsort_levels(const int* count, const int* ulx, int n, int* perm_out);
/* cosf / sinf exactly as glibc 2.39 rounds them (csrc/glibc_sincosf.h; the reference's `(float)cos(angle)`
 * in computeOrbDescriptor, ORBextractor.cc:111-112), evaluated by a kernel on `device` (x, outputs: host
 * arrays of n floats) and by the same source on the host (fused = 1: the -mfma build of libm, 0: SSE2). */
int orb_debug_sincos_device(int device, const float* x, size_t n, float* cos_out, float* sin_out);
int orb_debug_sincos_host(const float* x, size_t n, float* cos_out, float* sin_out, int fused);

#ifdef __cplusplus
}
#endif
#endif /* ORB_B200_H_ */
