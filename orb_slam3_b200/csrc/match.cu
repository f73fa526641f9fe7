// Hamming / projection matchers for B200 (sm_100a) behind include/orb_b200.h:
//   match_project_local  <- ORBmatcher::SearchByProjection(Frame&, vector<MapPoint*>&)  ORBmatcher.cc:43-141
//   match_project_last   <- ORBmatcher::SearchByProjection(Frame&, const Frame&)        ORBmatcher.cc:1676-1887
//   match_triangulate    <- ORBmatcher::SearchForTriangulation                           ORBmatcher.cc:907-1146
//   match_bow_frame      <- ORBmatcher::SearchByBoW(KeyFrame*, Frame&, vector<MapPoint*>&)     ORBmatcher.cc:223-…
//   match_bow_keyframes  <- ORBmatcher::SearchByBoW(KeyFrame*, KeyFrame*, vector<MapPoint*>&)  ORBmatcher.cc:765-…
//
// The reference loops are greedy and order dependent: a keypoint already held by
// a MapPoint with observations is skipped *before* its distance is looked at, and
// assignments are made inside the same loop (SURVEY.md H3).  The GPU path keeps
// the exact result with three phases per problem:
//   1. static phase, fully parallel: the 64x48 grid (Frame.cc:385-416), the window
//      query of every map point in GetFeaturesInArea order (Frame.cc:657-723), and
//      the Hamming distance (__popc over 8 words) of every (point, candidate) pair;
//   2. resolution rounds inside one CTA per problem.  A point can only ever TAKE a candidate whose distance is
//      <= TH_HIGH, so an unresolved point claims exactly those (atomicMin of its index per keypoint); a point may
//      finalise iff none of its still-free candidates is claimed by a lower-index unresolved point.  It then replays
//      the reference's scan (best / second best / ratio, or best only); `takenby[c]` records WHICH point took a
//      keypoint, and a point ignores takes by higher indices (those happen later in the reference's loop).  Takes
//      of a round are applied after the round's barrier.  With real descriptors almost every point finalises in
//      the first one or two rounds (the previous rule -- own ALL free candidates -- needed tens of rounds);
//   3. rotation histogram, ComputeThreeMaxima (ORBmatcher.cc:2012-2053) and the
//      clearing pass, preserving the 1/30 bin quirk (SURVEY.md 0.11).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/orb_b200.h"
#include "orb_engine.h"

namespace orbb200 {

constexpr int GRID_COLS = 64, GRID_ROWS = 48, GRID_CELLS = GRID_COLS * GRID_ROWS;
constexpr int TH_HIGH = 100, TH_LOW = 50, HISTO_LENGTH = 30;

#define CUDA_TRYM(expr)                                                                \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      set_last_error(std::string(#expr) + ": " + cudaGetErrorString(_e));              \
      return ORB_E_CUDA;                                                               \
    }                                                                                  \
  } while (0)

struct DevFrame {
  int n;
  const orb_keypoint* keys;
  const float* u_right;
  const uint8_t* desc;
  const uint8_t* kp_taken;
  float min_x, min_y, max_x, max_y, gwi, ghi;
  int n_levels;
  const float* scale;
  const float* sigma2;
  float fx, fy, cx, cy, bf, b;
  int* cell_start;  // [GRID_CELLS+1]
  int* cell_items;  // [n]
  uint4* cell_rec;  // [n] (x, y, octave, index) of the keypoints in cell_items order: the window scans read these
};

// One projection-match problem (local-map or last-frame flavour).
struct ProjProblem {
  DevFrame F;
  int kind;  // 0: SearchByProjection(F, MapPoints)   1: SearchByProjection(Cur, Last)
  int nq;    // number of query points (map points / last-frame keypoints)
  // kind 0 inputs
  const uint8_t *in_view, *is_bad;
  const float *px, *py, *pxr, *vcos, *depth;
  const int* lvl;
  // kind 1 inputs
  const uint8_t* has_mp;
  const float* wpos;
  const int* octave;
  const float* angle;
  float T[7];
  int forward, backward, check_ori;
  // common
  const uint8_t* has_obs;
  const uint8_t* qdesc;
  float th, ratio, th_far;
  int far_points;
  // scratch
  int* q_cnt;          // candidate list of point j: cand_*[j * cand_slot .. + q_cnt[j])
  uint8_t* q_state;    // 0 inactive/resolved, 1 unresolved, 2 finalised this round with a take to apply
  int* cand_idx;
  unsigned short* cand_dist;
  int cand_slot;       // entries per point
  int* ulist;          // [2 * nq] points blocked in the current / next round
  int* minidx;
  int* takenby;        // [F.n] index of the point that took the keypoint; -1 taken on entry; INT_MAX free
  int *acc_kp, *acc_bin;
  // outputs
  int* assign;   // [F.n]
  int* result;   // [3]: nmatches, overflow flag, resolution rounds
};

struct TriProblem {
  DevFrame K1, K2;
  int n_nodes1, n_nodes2;
  const uint32_t *nid1, *nid2;
  const int *ptr1, *idx1, *ptr2, *idx2;
  int n_feat1;  // ptr1[n_nodes1]
  float F12[9], ep[2];
  int only_stereo, coarse, check_ori;
  int* match12;  // [K1.n]
  int* bins;     // [K1.n]
  int* pairs;    // [2*cap]
  int cap;
  int* result;   // [2]
};

__device__ const DevFrame& frame_of(const ProjProblem* probs, int k) { return probs[k].F; }

__device__ __forceinline__ int popc256(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b) {
  const uint4* pa = reinterpret_cast<const uint4*>(a);
  const uint4* pb = reinterpret_cast<const uint4*>(b);
  const uint4 a0 = pa[0], a1 = pa[1], b0 = pb[0], b1 = pb[1];
  return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
         __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// ---- Frame::AssignFeaturesToGrid (Frame.cc:385-416): CSR over 64x48 cells,
// ascending keypoint index inside a cell.  One CTA per frame.
struct ProjProblem;
__device__ const DevFrame& frame_of(const ProjProblem* probs, int k);
__device__ void init_problem(const ProjProblem* probs, int k);
__global__ void __launch_bounds__(256) grid_build_kernel(const ProjProblem* probs) {
  __shared__ int cnt[GRID_CELLS + 1];
  __shared__ int wsum[8];
  const DevFrame F = frame_of(probs, blockIdx.x);
  for (int c = threadIdx.x; c <= GRID_CELLS; c += 256) cnt[c] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < F.n; i += 256) {
    const orb_keypoint kp = F.keys[i];
    const int px = (int)roundf(__fmul_rn(__fsub_rn(kp.x, F.min_x), F.gwi));
    const int py = (int)roundf(__fmul_rn(__fsub_rn(kp.y, F.min_y), F.ghi));
    if (px < 0 || px >= GRID_COLS || py < 0 || py >= GRID_ROWS) continue;
    atomicAdd(&cnt[px * GRID_ROWS + py], 1);
  }
  __syncthreads();
  // exclusive scan of 3072 counts: 12 per thread
  const int per = GRID_CELLS / 256;
  int local[per];
  int sum = 0;
  for (int k = 0; k < per; k++) { local[k] = cnt[threadIdx.x * per + k]; sum += local[k]; }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = sum;
  for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  int base = incl - sum;
  for (int w = 0; w < warp; w++) base += wsum[w];
  __syncthreads();
  for (int k = 0; k < per; k++) { cnt[threadIdx.x * per + k] = base; F.cell_start[threadIdx.x * per + k] = base; base += local[k]; }
  if (threadIdx.x == 255) F.cell_start[GRID_CELLS] = base;
  __syncthreads();
  for (int i = threadIdx.x; i < F.n; i += 256) {
    const orb_keypoint kp = F.keys[i];
    const int px = (int)roundf(__fmul_rn(__fsub_rn(kp.x, F.min_x), F.gwi));
    const int py = (int)roundf(__fmul_rn(__fsub_rn(kp.y, F.min_y), F.ghi));
    if (px < 0 || px >= GRID_COLS || py < 0 || py >= GRID_ROWS) continue;
    F.cell_items[atomicAdd(&cnt[px * GRID_ROWS + py], 1)] = i;
  }
  __syncthreads();
  // restore insertion (ascending index) order inside each cell
  for (int c = threadIdx.x; c < GRID_CELLS; c += 256) {
    const int s = F.cell_start[c], e = cnt[c];
    for (int i = s + 1; i < e; i++) {
      const int v = F.cell_items[i];
      int j = i - 1;
      while (j >= s && F.cell_items[j] > v) { F.cell_items[j + 1] = F.cell_items[j]; j--; }
      F.cell_items[j + 1] = v;
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < cnt[GRID_CELLS - 1]; k += 256) {  // cnt[c] = end of cell c by now
    const int i = F.cell_items[k];
    const orb_keypoint kp = F.keys[i];
    F.cell_rec[k] = make_uint4(__float_as_uint(kp.x), __float_as_uint(kp.y), (unsigned)kp.octave, (unsigned)i);
  }
  init_problem(probs, blockIdx.x);
}

// Outputs / per-keypoint state of one problem, reset by the CTA that builds its grid.
__device__ void init_problem(const ProjProblem* probs, int k) {
  const ProjProblem& P = probs[k];
  for (int i = threadIdx.x; i < P.F.n; i += blockDim.x) {
    P.assign[i] = -1;
    P.takenby[i] = (P.F.kp_taken && P.F.kp_taken[i]) ? -1 : 0x7fffffff;
  }
  if (threadIdx.x == 0) { P.result[0] = 0; P.result[1] = 0; }
}

// Phase 1: one WARP per query point, four points per warp.  The window parameters (ORBmatcher.cc:51-70 /
// :1701-1733) of the warp's four points are computed by four lanes at once (one round of global-memory latency
// instead of four); then, point by point, the window query of Frame::GetFeaturesInArea (Frame.cc:657-723) with the
// per-candidate gate on mvuRight (ORBmatcher.cc:92-97 / :1752-1758) is spread over the lanes: the cells
// (ix, minY..maxY) of one grid column are one contiguous CSR range, lanes 0..ncol-1 fetch the ranges, a warp scan
// concatenates them, and lane t of a chunk tests the t-th keypoint of the concatenation -- one 16-byte record of
// cell_rec, contiguous within a column (the scattered 28-byte orb_keypoint gathers of a thread-per-point version
// were bound by L2 sector traffic).  A ballot keeps the candidates in the reference's order.  Candidates that can
// never influence the point's outcome are dropped here: beyond TH_HIGH a keypoint cannot be taken, and it matters
// as SECOND best only while ratio * dist < TH_HIGH (ORBmatcher.cc:123-128); SearchByProjection(Cur, Last) has no
// second best at all.  Every point owns a fixed slot of `cand_slot` entries (no counting pass, no atomics); a
// point that needs more raises the overflow flag and the host runs the batch again with larger slots.
constexpr int PC_WARPS = 4, PC_Q_PER_WARP = 4;
__global__ void __launch_bounds__(PC_WARPS * 32, 7) proj_candidates_kernel(ProjProblem* probs) {
  __shared__ ProjProblem P;
  {
    const int* src = reinterpret_cast<const int*>(probs + blockIdx.y);
    int* dst = reinterpret_cast<int*>(&P);
    for (int i = threadIdx.x; i < (int)(sizeof(ProjProblem) / 4); i += PC_WARPS * 32) dst[i] = src[i];
  }
  __syncthreads();
  const DevFrame& F = P.F;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned full = 0xffffffffu, lt = (1u << lane) - 1u;
  const int j0 = (blockIdx.x * PC_WARPS + warp) * PC_Q_PER_WARP;
  if (j0 >= P.nq) return;
  // ---- parameters of points j0 .. j0+3 on lanes 0..3
  bool my_active = false;
  float my_u = 0, my_v = 0, my_r = 0, my_aux = 0;
  int my_minl = 0, my_maxl = 0;
  if (lane < PC_Q_PER_WARP && j0 + lane < P.nq) {
    const int j = j0 + lane;
    if (P.kind == 0) {
      // ORBmatcher.cc:51-70 (all inputs fetched up front: one round trip)
      const uint8_t in_view = P.in_view[j], bad = P.is_bad[j];
      const float depth = P.depth[j], vcos = P.vcos[j], px = P.px[j], py = P.py[j], pxr = P.pxr ? P.pxr[j] : 0.f;
      const int lvl = P.lvl[j];
      my_active = in_view && !(P.far_points && depth > P.th_far) && !bad;
      if (my_active) {
        float rr = ((double)vcos > 0.998) ? 2.5f : 4.0f;
        if (P.th != 1.0f) rr = __fmul_rn(rr, P.th);
        my_r = __fmul_rn(rr, F.scale[lvl]);
        my_u = px; my_v = py; my_aux = pxr;
        my_minl = lvl - 1; my_maxl = lvl;
      }
    } else {
      // ORBmatcher.cc:1701-1733; Tcw * x3Dw as Sophus/Eigen evaluate it
      const uint8_t has_mp = P.has_mp[j];
      const float vx = P.wpos[3 * j], vy = P.wpos[3 * j + 1], vz = P.wpos[3 * j + 2];
      const int o = P.octave[j];
      if (has_mp) {
        const float qx = P.T[0], qy = P.T[1], qz = P.T[2], qw = P.T[3];
        float ux = __fsub_rn(__fmul_rn(qy, vz), __fmul_rn(qz, vy));
        float uy = __fsub_rn(__fmul_rn(qz, vx), __fmul_rn(qx, vz));
        float uz = __fsub_rn(__fmul_rn(qx, vy), __fmul_rn(qy, vx));
        ux = __fadd_rn(ux, ux); uy = __fadd_rn(uy, uy); uz = __fadd_rn(uz, uz);
        const float c0 = __fsub_rn(__fmul_rn(qy, uz), __fmul_rn(qz, uy));
        const float c1 = __fsub_rn(__fmul_rn(qz, ux), __fmul_rn(qx, uz));
        const float c2 = __fsub_rn(__fmul_rn(qx, uy), __fmul_rn(qy, ux));
        const float xc = __fadd_rn(__fadd_rn(__fadd_rn(vx, __fmul_rn(qw, ux)), c0), P.T[4]);
        const float yc = __fadd_rn(__fadd_rn(__fadd_rn(vy, __fmul_rn(qw, uy)), c1), P.T[5]);
        const float zc = __fadd_rn(__fadd_rn(__fadd_rn(vz, __fmul_rn(qw, uz)), c2), P.T[6]);
        const float invzc = (float)(1.0 / (double)zc);
        if (!(invzc < 0)) {
          const float u = __fadd_rn(__fdiv_rn(__fmul_rn(F.fx, xc), zc), F.cx);
          const float v = __fadd_rn(__fdiv_rn(__fmul_rn(F.fy, yc), zc), F.cy);
          if (!(u < F.min_x || u > F.max_x) && !(v < F.min_y || v > F.max_y)) {
            my_active = true;
            my_u = u; my_v = v;
            my_r = __fmul_rn(P.th, F.scale[o]);
            my_aux = __fsub_rn(u, __fmul_rn(F.bf, invzc));  // ur (:1754)
            if (P.forward) { my_minl = o; my_maxl = -1; }
            else if (P.backward) { my_minl = 0; my_maxl = o; }
            else { my_minl = o - 1; my_maxl = o + 1; }
          }
        }
      }
    }
  }
  const int slot = P.cand_slot;
  for (int q = 0; q < PC_Q_PER_WARP && j0 + q < P.nq; q++) {
    const int j = j0 + q;
    const bool active = __shfl_sync(full, (int)my_active, q) != 0;
    const float u = __shfl_sync(full, my_u, q), v = __shfl_sync(full, my_v, q), r = __shfl_sync(full, my_r, q),
                aux = __shfl_sync(full, my_aux, q);
    const int minl = __shfl_sync(full, my_minl, q), maxl = __shfl_sync(full, my_maxl, q);
    // Frame::GetFeaturesInArea's cell rectangle (Frame.cc:664-686)
    int cx0 = 0, cx1 = -1, cy0 = 0, cy1 = -1;
    if (active) {
      cx0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(u, F.min_x), r), F.gwi)));
      cx1 = min(GRID_COLS - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(u, F.min_x), r), F.gwi)));
      cy0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(v, F.min_y), r), F.ghi)));
      cy1 = min(GRID_ROWS - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(v, F.min_y), r), F.ghi)));
      if (cx0 >= GRID_COLS || cx1 < 0 || cy0 >= GRID_ROWS || cy1 < 0) cx1 = cx0 - 1;
    }
    const bool check_levels = (minl > 0) || (maxl >= 0);
    uint4 qa = make_uint4(0, 0, 0, 0), qb = qa;
    if (cx0 <= cx1) {
      const uint4* pq = reinterpret_cast<const uint4*>(P.qdesc + (size_t)j * 32);
      qa = pq[0]; qb = pq[1];
    }
    const size_t base = (size_t)j * slot;
    int written = 0;
    bool overflow = false;
    for (int g0 = cx0; g0 <= cx1; g0 += 32) {
      const int ix = g0 + lane;
      int s = 0, len = 0;
      if (ix <= cx1) {
        s = F.cell_start[ix * GRID_ROWS + cy0];
        len = F.cell_start[ix * GRID_ROWS + cy1 + 1] - s;
      }
      int incl = len;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(full, incl, o); if (lane >= o) incl += t; }
      const int total = __shfl_sync(full, incl, 31);
      for (int t0 = 0; t0 < total; t0 += 32) {
        const int t = t0 + lane;
        int col = 0;  // first column whose inclusive prefix exceeds t
#pragma unroll
        for (int step = 16; step; step >>= 1) {
          const int pv = __shfl_sync(full, incl, col + step - 1);
          if (pv <= t) col += step;
        }
        const int cs = __shfl_sync(full, s, col), cex = __shfl_sync(full, incl - len, col);
        int pick = -1, dist = 0;
        if (t < total) {
          const uint4 rec = F.cell_rec[cs + (t - cex)];
          const int oc = (int)rec.z, idx = (int)rec.w;
          bool ok = true;
          if (check_levels) ok = oc >= minl && !(maxl >= 0 && oc > maxl);
          if (ok) ok = fabsf(__fsub_rn(__uint_as_float(rec.x), u)) < r && fabsf(__fsub_rn(__uint_as_float(rec.y), v)) < r;
          if (ok && F.u_right) {
            const float ur = F.u_right[idx];
            if (ur > 0 && fabsf(__fsub_rn(aux, ur)) > r) ok = false;
          }
          if (ok) {
            const uint4* pd = reinterpret_cast<const uint4*>(F.desc + (size_t)idx * 32);
            const uint4 d0 = pd[0], d1 = pd[1];
            dist = __popc(qa.x ^ d0.x) + __popc(qa.y ^ d0.y) + __popc(qa.z ^ d0.z) + __popc(qa.w ^ d0.w) +
                   __popc(qb.x ^ d1.x) + __popc(qb.y ^ d1.y) + __popc(qb.z ^ d1.z) + __popc(qb.w ^ d1.w);
            if (dist <= TH_HIGH || (P.kind == 0 && __fmul_rn(P.ratio, (float)dist) < (float)TH_HIGH)) pick = idx;
          }
        }
        const unsigned m = __ballot_sync(full, pick >= 0);
        const int o = written + __popc(m & lt);
        if (pick >= 0) {
          if (o < slot) { P.cand_idx[base + o] = pick; P.cand_dist[base + o] = (unsigned short)dist; }
          else overflow = true;
        }
        written += __popc(m);
      }
    }
    if (__any_sync(full, overflow)) {  // the host grows the slots and runs the batch again
      if (lane == 0) P.result[1] = 1;
      written = 0;
    }
    if (lane == 0) { P.q_cnt[j] = written; P.q_state[j] = written > 0 ? 1 : 0; }
  }
}

// ORBmatcher::ComputeThreeMaxima (ORBmatcher.cc:2012-2053) on bin sizes.
__device__ void three_maxima(const int* size, int& ind1, int& ind2, int& ind3) {
  int max1 = 0, max2 = 0, max3 = 0;
  ind1 = ind2 = ind3 = -1;
  for (int i = 0; i < HISTO_LENGTH; i++) {
    const int s = size[i];
    if (s > max1) { max3 = max2; max2 = max1; max1 = s; ind3 = ind2; ind2 = ind1; ind1 = i; }
    else if (s > max2) { max3 = max2; max2 = s; ind3 = ind2; ind2 = i; }
    else if (s > max3) { max3 = s; ind3 = i; }
  }
  if ((float)max2 < __fmul_rn(0.1f, (float)max1)) { ind2 = -1; ind3 = -1; }
  else if ((float)max3 < __fmul_rn(0.1f, (float)max1)) { ind3 = -1; }
}

__device__ __forceinline__ int rot_bin(float a1, float a2) {
  float rot = __fsub_rn(a1, a2);
  if (rot < 0.0f) rot = __fadd_rn(rot, 360.0f);
  int bin = (int)roundf(__fmul_rn(rot, 1.0f / HISTO_LENGTH));
  if (bin == HISTO_LENGTH) bin = 0;
  return bin;
}

// Phase 2+3: resolution rounds, one CTA per problem, one thread per unresolved point (the lists are short after
// the filtering of phase 1; a warp per point was measured slower: too few chains in flight).  Round 1 visits every
// point, later rounds only the list of points that were blocked.
__global__ void __launch_bounds__(1024, 1) proj_resolve_kernel(ProjProblem* probs, int smem_nk) {
  extern __shared__ int rs_dyn[];
  __shared__ ProjProblem P;
  __shared__ int s_nmatch, s_nlist[2];
  __shared__ int s_hist[HISTO_LENGTH];
  __shared__ int s_ind[3];
  {
    const int* src = reinterpret_cast<const int*>(probs + blockIdx.x);
    int* dst = reinterpret_cast<int*>(&P);
    for (int i = threadIdx.x; i < (int)(sizeof(ProjProblem) / 4); i += 1024) dst[i] = src[i];
  }
  __syncthreads();
  if (P.result[1]) return;  // a candidate slot overflowed: host re-runs with larger ones
  const DevFrame& F = P.F;
  const int nq = P.nq, nk = F.n, slot = P.cand_slot;
  // per-keypoint state of the rounds (lowest claiming point, taker, octave) in shared memory when it fits: every
  // round is a chain of dependent look-ups into these arrays
  const bool in_smem = nk <= smem_nk;
  int* minidx = in_smem ? rs_dyn : P.minidx;
  int* takenby = in_smem ? rs_dyn + smem_nk : P.takenby;
  uint8_t* oct8 = reinterpret_cast<uint8_t*>(rs_dyn + 2 * smem_nk);
  if (in_smem)
    for (int i = threadIdx.x; i < nk; i += 1024) { takenby[i] = P.takenby[i]; oct8[i] = (uint8_t)F.keys[i].octave; }
  if (threadIdx.x == 0) { s_nmatch = 0; s_nlist[0] = 0; s_nlist[1] = 0; }
  for (int b = threadIdx.x; b < HISTO_LENGTH; b += 1024) s_hist[b] = 0;
  for (int j = threadIdx.x; j < nq; j += 1024) P.acc_kp[j] = -1;
  __syncthreads();
  int* ulist[2] = {P.ulist, P.ulist + nq};
  int rounds = 0, n_cur = nq;  // round 1: the "list" is 0..nq-1
  while (true) {
    const int cur = rounds & 1;
    const bool first = rounds == 0;
    rounds++;
    for (int i = threadIdx.x; i < nk; i += 1024) minidx[i] = 0x7fffffff;
    // takes of the previous round (one taker per keypoint: see the claim rule)
    if (!first)
      for (int j = threadIdx.x; j < nq; j += 1024)
        if (P.q_state[j] == 2) { takenby[P.acc_kp[j]] = j; P.q_state[j] = 0; }
    if (threadIdx.x == 0) s_nlist[cur ^ 1] = 0;
    __syncthreads();
    // claims: only a candidate within TH_HIGH can be taken by j; free for j = not taken by a lower index
    for (int i = threadIdx.x; i < n_cur; i += 1024) {
      const int j = first ? i : ulist[cur][i];
      if (first && P.q_state[j] != 1) continue;
      const size_t e0 = (size_t)j * slot;
      const int cnt = P.q_cnt[j];
      for (int t = 0; t < cnt; t++) {
        if (P.cand_dist[e0 + t] > TH_HIGH) continue;
        const int c = P.cand_idx[e0 + t];
        if (takenby[c] > j) atomicMin(&minidx[c], j);
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_cur; i += 1024) {
      const int j = first ? i : ulist[cur][i];
      if (first && P.q_state[j] != 1) continue;
      const size_t e0 = (size_t)j * slot;
      const int cnt = P.q_cnt[j];
      // one pass: blocked? and the reference's scan over the candidates that are free for j (a keypoint is skipped
      // iff it was taken on entry or by a lower-index point)
      bool blocked = false;
      int bestDist = 256, bestLevel = -1, bestDist2 = 256, bestLevel2 = -1, bestIdx = -1;
      for (int t = 0; t < cnt; t++) {
        const int c = P.cand_idx[e0 + t];
        if (takenby[c] < j) continue;
        if (minidx[c] < j) { blocked = true; break; }  // a lower unresolved point may still take it
        const int dist = P.cand_dist[e0 + t];
        if (dist < bestDist) {
          bestDist2 = bestDist; bestDist = dist; bestLevel2 = bestLevel;
          bestLevel = in_smem ? (int)oct8[c] : F.keys[c].octave; bestIdx = c;
        } else if (P.kind == 0 && dist < bestDist2) {
          bestLevel2 = in_smem ? (int)oct8[c] : F.keys[c].octave; bestDist2 = dist;
        }
      }
      if (blocked) { ulist[cur ^ 1][atomicAdd(&s_nlist[cur ^ 1], 1)] = j; continue; }
      bool accept = bestDist <= TH_HIGH;
      // ratio only when best and second best share the level (:123-128)
      if (accept && P.kind == 0 && bestLevel == bestLevel2 && (float)bestDist > __fmul_rn(P.ratio, (float)bestDist2))
        accept = false;
      int state = 0;
      if (accept) {
        P.assign[bestIdx] = j;
        P.acc_kp[j] = bestIdx;
        if (P.has_obs[j]) state = 2;  // the keypoint is closed to later points (ORBmatcher.cc:88-90 / :1748-1750)
        atomicAdd(&s_nmatch, 1);
        if (P.kind == 1 && P.check_ori) {
          const int bin = rot_bin(P.angle[j], F.keys[bestIdx].angle);
          P.acc_bin[j] = bin;
          atomicAdd(&s_hist[bin], 1);
        }
      }
      P.q_state[j] = (uint8_t)state;
    }
    __syncthreads();
    n_cur = s_nlist[cur ^ 1];
    if (n_cur == 0) break;
  }
  if (P.kind == 1 && P.check_ori) {
    if (threadIdx.x == 0) {
      int a, b, c;
      three_maxima(s_hist, a, b, c);
      s_ind[0] = a; s_ind[1] = b; s_ind[2] = c;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < nq; j += 1024) {
      const int kp = P.acc_kp[j];
      if (kp < 0) continue;
      const int bin = P.acc_bin[j];
      if (bin != s_ind[0] && bin != s_ind[1] && bin != s_ind[2]) {
        P.assign[kp] = -2;  // cleared by the rotation check (:1875-1884)
        atomicSub(&s_nmatch, 1);
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { P.result[0] = s_nmatch; P.result[2] = rounds; }
}

// ---- SearchForTriangulation: one thread per KF1 feature-vector entry.
__device__ __forceinline__ int find_node(const uint32_t* ids, int n, uint32_t key) {
  int lo = 0, hi = n;
  while (lo < hi) { int mid = (lo + hi) >> 1; if (ids[mid] < key) lo = mid + 1; else hi = mid; }
  return (lo < n && ids[lo] == key) ? lo : -1;
}

__global__ void __launch_bounds__(128) tri_match_kernel(TriProblem* probs) {
  TriProblem& T = probs[blockIdx.y];
  const int p1 = blockIdx.x * 128 + threadIdx.x;
  if (p1 >= T.n_feat1) return;
  // owner node of entry p1: last a with ptr1[a] <= p1
  int lo = 0, hi = T.n_nodes1;
  while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (T.ptr1[mid] <= p1) lo = mid; else hi = mid; }
  const int a = lo;
  const int idx1 = T.idx1[p1];
  int best = -1;
  const int b = find_node(T.nid2, T.n_nodes2, T.nid1[a]);
  const DevFrame& K1 = T.K1;
  const DevFrame& K2 = T.K2;
  const bool skip1 = (K1.kp_taken && K1.kp_taken[idx1]);
  const bool bStereo1 = K1.u_right && K1.u_right[idx1] >= 0;
  if (b >= 0 && !skip1 && !(T.only_stereo && !bStereo1)) {
    const orb_keypoint kp1 = K1.keys[idx1];
    const uint8_t* d1 = K1.desc + (size_t)idx1 * 32;
    // epipolar line of kp1 in image 2 (Pinhole.cpp:114-117)
    const float la = __fadd_rn(__fadd_rn(__fmul_rn(kp1.x, T.F12[0]), __fmul_rn(kp1.y, T.F12[3])), T.F12[6]);
    const float lb = __fadd_rn(__fadd_rn(__fmul_rn(kp1.x, T.F12[1]), __fmul_rn(kp1.y, T.F12[4])), T.F12[7]);
    const float lc = __fadd_rn(__fadd_rn(__fmul_rn(kp1.x, T.F12[2]), __fmul_rn(kp1.y, T.F12[5])), T.F12[8]);
    const float den = __fadd_rn(__fmul_rn(la, la), __fmul_rn(lb, lb));
    int bestDist = TH_LOW;
    for (int p2 = T.ptr2[b]; p2 < T.ptr2[b + 1]; p2++) {
      const int idx2 = T.idx2[p2];
      if (K2.kp_taken && K2.kp_taken[idx2]) continue;
      const bool bStereo2 = K2.u_right && K2.u_right[idx2] >= 0;
      if (T.only_stereo && !bStereo2) continue;
      const int dist = popc256(d1, K2.desc + (size_t)idx2 * 32);
      if (dist > TH_LOW || dist > bestDist) continue;
      const orb_keypoint kp2 = K2.keys[idx2];
      if (!bStereo1 && !bStereo2) {
        const float ex = __fsub_rn(T.ep[0], kp2.x), ey = __fsub_rn(T.ep[1], kp2.y);
        if (__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)) < __fmul_rn(100.f, K2.scale[kp2.octave])) continue;
      }
      bool ok = T.coarse != 0;
      if (!ok && den != 0) {
        const float num = __fadd_rn(__fadd_rn(__fmul_rn(la, kp2.x), __fmul_rn(lb, kp2.y)), lc);
        const float dsqr = __fdiv_rn(__fmul_rn(num, num), den);
        ok = (double)dsqr < 3.84 * (double)K2.sigma2[kp2.octave];
      }
      if (ok) { best = idx2; bestDist = dist; }
    }
  }
  T.match12[idx1] = best;
  if (best >= 0 && T.check_ori) T.bins[idx1] = rot_bin(K1.keys[idx1].angle, K2.keys[best].angle);
}

// Rotation-consistency check of SearchForTriangulation and SearchByBoW, run by a whole CTA after the matching loop:
// histogram of bins[i] over the entries with out[i] >= 0, ComputeThreeMaxima (ORBmatcher.cc:2012-2053), and every
// such entry whose bin is not among the (at most three) maxima is set to `cleared`.  Ends with a barrier.
__device__ void rot_filter_cta(int* out, const int* bins, int n, int cleared) {
  __shared__ int s_hist[HISTO_LENGTH], s_ind[3];
  for (int b = threadIdx.x; b < HISTO_LENGTH; b += blockDim.x) s_hist[b] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (out[i] >= 0) atomicAdd(&s_hist[bins[i]], 1);
  __syncthreads();
  if (threadIdx.x == 0) { int a, b, c; three_maxima(s_hist, a, b, c); s_ind[0] = a; s_ind[1] = b; s_ind[2] = c; }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (out[i] >= 0) {
      const int bin = bins[i];
      if (bin != s_ind[0] && bin != s_ind[1] && bin != s_ind[2]) out[i] = cleared;
    }
  __syncthreads();
}

__global__ void __launch_bounds__(1024) tri_finish_kernel(TriProblem* probs) {
  __shared__ int wsum[32], carry;
  TriProblem& T = probs[blockIdx.x];
  const int n = T.K1.n;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  if (T.check_ori) rot_filter_cta(T.match12, T.bins, n, -1);
  // compaction in increasing idx1 (:1138-1143)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < n; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = (i < n && T.match12[i] >= 0) ? 1 : 0;
    int incl = v;
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      int w = wsum[lane], wi = w;
      for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
      wsum[lane] = wi - w;
    }
    __syncthreads();
    const int pos = carry + wsum[warp] + incl - v;
    if (v && pos < T.cap) { T.pairs[2 * pos] = i; T.pairs[2 * pos + 1] = T.match12[i]; }
    __syncthreads();
    if (threadIdx.x == 1023) carry = pos + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) { T.result[0] = carry; T.result[1] = carry > T.cap ? 1 : 0; }
}

// ---- SearchByBoW, both overloads (ORBmatcher.cc:223-… KeyFrame-Frame, :765-… KeyFrame-KeyFrame).
// The query side is the (first) keyframe, the candidate side the frame / second keyframe.  Features of different
// vocabulary nodes never compete (every feature index is in at most one node of a FeatureVector), so the shared nodes
// are independent work items; inside a node the reference's scan is sequential over the queries, because a match takes
// its candidate for the rest of the call.
struct BowProblem {
  int kind;                       // 0: SearchByBoW(KeyFrame*, Frame&)   1: SearchByBoW(KeyFrame*, KeyFrame*)
  int nq, nc;                     // keypoints of the query side (KF / KF1) and of the candidate side (F / KF2)
  const orb_keypoint *kq, *kc;    // angle only
  const uint8_t *dq, *dc;
  const uint8_t *okq, *okc;       // map point present and !isBad(); okc: kind 1 only
  int nodes_q, nodes_c;
  const uint32_t *nid_q, *nid_c;
  const int *ptr_q, *idx_q, *ptr_c, *idx_c;
  float ratio;
  int check_ori;
  int n_out;                      // kind 0: nc (vpMapPointMatches), kind 1: nq (vpMatches12)
  int* out;                       // [n_out] matched index on the other side, -1 untouched, -2 cleared by the rotation check
  int* bins;                      // [n_out] rotation bin of a match
  uint8_t* free_c;                // [nc] candidate still available, for nodes too large for the shared-memory copy
  int* result;                    // [1] nmatches
};

constexpr int BOW_WARPS = 4;           // one warp per shared node
constexpr int BOW_SMEM_CAND = 256;     // candidates of a node staged in shared memory (8 KB of descriptors per warp)
constexpr unsigned BOW_POS_BITS = 23;  // key = dist << 23 | position in the node; the host rejects n >= 2^23
constexpr unsigned BOW_POS_MASK = (1u << BOW_POS_BITS) - 1;

__global__ void __launch_bounds__(256) bow_init_kernel(const BowProblem* probs) {
  const BowProblem& P = probs[blockIdx.x];
  for (int i = threadIdx.x; i < P.n_out; i += 256) P.out[i] = -1;
}

// One warp per (problem, query-side node).  For each query in the node's order, lane l scans the candidates at
// positions l, l+32, ... that are still free and keeps (min key, second-smallest distance); the butterfly merge of two
// such pairs (a1, a2), (b1, b2) is (min(a1, b1), min(dist(max(a1, b1)), a2, b2)).  The result is the reference's
// bestDist1 with the FIRST position reaching it (`dist < bestDist1` only moves on a strictly smaller distance) and its
// bestDist2, the second smallest value of the distance multiset (a tie at the minimum gives bestDist2 == bestDist1).
// Nodes up to BOW_SMEM_CAND candidates are copied to shared memory with their free flags; larger ones (levelsup >= L
// makes the whole frame one node) read descriptors from global memory and keep the flags in P.free_c.  The scan order,
// and hence every result, is the same on both paths.
__global__ void __launch_bounds__(BOW_WARPS * 32) bow_match_kernel(const BowProblem* probs) {
  __shared__ uint4 s_desc[BOW_WARPS][BOW_SMEM_CAND][2];
  __shared__ uint8_t s_free[BOW_WARPS][BOW_SMEM_CAND];
  const BowProblem& P = probs[blockIdx.y];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int a = blockIdx.x * BOW_WARPS + warp;
  if (a >= P.nodes_q) return;
  const int b = find_node(P.nid_c, P.nodes_c, P.nid_q[a]);
  if (b < 0) return;
  const int q0 = P.ptr_q[a], q1 = P.ptr_q[a + 1], c0 = P.ptr_c[b], m = P.ptr_c[b + 1] - c0;
  const bool staged = m <= BOW_SMEM_CAND;
  uint4 (*sd)[2] = s_desc[warp];
  uint8_t* sf = s_free[warp];
  for (int pos = lane; pos < m; pos += 32) {
    const int idx = P.idx_c[c0 + pos];
    const uint8_t ok = P.kind == 1 ? P.okc[idx] : 1;  // KF2: pMP2 && !isBad(); F: vpMapPointMatches starts all NULL
    if (staged) {
      const uint4* pd = reinterpret_cast<const uint4*>(P.dc + (size_t)idx * 32);
      sd[pos][0] = pd[0]; sd[pos][1] = pd[1];
      sf[pos] = ok;
    } else {
      P.free_c[idx] = ok;
    }
  }
  __syncwarp();
  for (int p = q0; p < q1; p++) {
    const int i1 = P.idx_q[p];
    if (!P.okq[i1]) continue;  // pMP && !pMP->isBad()
    const uint4* pq = reinterpret_cast<const uint4*>(P.dq + (size_t)i1 * 32);
    const uint4 qa = pq[0], qb = pq[1];
    unsigned k1 = (256u << BOW_POS_BITS) | BOW_POS_MASK;  // bestDist1 = 256, no position
    int d2 = 256;                                          // bestDist2
    for (int pos = lane; pos < m; pos += 32) {
      uint4 ca, cb;
      if (staged) {
        if (!sf[pos]) continue;
        ca = sd[pos][0]; cb = sd[pos][1];
      } else {
        const int idx = P.idx_c[c0 + pos];
        if (!P.free_c[idx]) continue;
        const uint4* pd = reinterpret_cast<const uint4*>(P.dc + (size_t)idx * 32);
        ca = pd[0]; cb = pd[1];
      }
      const int dist = __popc(qa.x ^ ca.x) + __popc(qa.y ^ ca.y) + __popc(qa.z ^ ca.z) + __popc(qa.w ^ ca.w) +
                       __popc(qb.x ^ cb.x) + __popc(qb.y ^ cb.y) + __popc(qb.z ^ cb.z) + __popc(qb.w ^ cb.w);
      const unsigned key = ((unsigned)dist << BOW_POS_BITS) | (unsigned)pos;
      if (key < k1) { d2 = min(d2, (int)(k1 >> BOW_POS_BITS)); k1 = key; }
      else d2 = min(d2, dist);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const unsigned ok1 = __shfl_xor_sync(0xffffffffu, k1, o);
      const int od2 = __shfl_xor_sync(0xffffffffu, d2, o);
      d2 = min(min(d2, od2), (int)(max(k1, ok1) >> BOW_POS_BITS));
      k1 = min(k1, ok1);
    }
    const int best = (int)(k1 >> BOW_POS_BITS);
    // keyframe-frame accepts bestDist1 <= TH_LOW, keyframe-keyframe bestDist1 < TH_LOW
    const bool pass = P.kind == 0 ? best <= TH_LOW : best < TH_LOW;
    if (pass && (float)best < __fmul_rn(P.ratio, (float)d2)) {
      const int pos = (int)(k1 & BOW_POS_MASK);
      if (lane == 0) {
        const int i2 = P.idx_c[c0 + pos];
        if (staged) sf[pos] = 0; else P.free_c[i2] = 0;
        const int r = P.kind == 0 ? i2 : i1;
        P.out[r] = P.kind == 0 ? i1 : i2;
        if (P.check_ori) P.bins[r] = rot_bin(P.kq[i1].angle, P.kc[i2].angle);
      }
    }
    __syncwarp();  // the take is visible to every lane before the next query
  }
}

// One CTA per problem: the rotation check over the recorded matches, then nmatches = entries still >= 0.
__global__ void __launch_bounds__(1024) bow_finish_kernel(const BowProblem* probs) {
  __shared__ int s_count;
  const BowProblem& P = probs[blockIdx.x];
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  if (P.check_ori) rot_filter_cta(P.out, P.bins, P.n_out, -2);
  int c = 0;
  for (int i = threadIdx.x; i < P.n_out; i += blockDim.x) c += P.out[i] >= 0;
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_count, c);
  __syncthreads();
  if (threadIdx.x == 0) P.result[0] = s_count;
}

// ------------------------------------------------------------------ host side
// Growable device arena + pinned staging blob: one H2D and one D2H per batch.
struct Arena {
  uint8_t* d = nullptr;
  size_t cap = 0, used = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return 0;
    if (d) cudaFree(d);
    cap = bytes + bytes / 4;
    d = nullptr;
    CUDA_TRYM(cudaMalloc((void**)&d, cap));
    return 0;
  }
  size_t take(size_t bytes) { size_t o = used; used = (used + bytes + 255) & ~(size_t)255; return o; }
};
struct Pinned {
  uint8_t* h = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return 0;
    if (h) cudaFreeHost(h);
    cap = bytes + bytes / 4;
    h = nullptr;
    CUDA_TRYM(cudaHostAlloc((void**)&h, cap, cudaHostAllocDefault));
    return 0;
  }
};

struct Matcher {
  int device = 0;
  bool initialized = false;
  cudaStream_t stream = nullptr, user_stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  Arena in_arena, scratch, out_arena;
  Pinned h_in, h_out;
  long long launches = 0;
  double last_ms = 0;
  // initial candidate budget per query, grows on overflow (ORB_B200_MATCH_BUDGET: tests start it small to take
  // the overflow paths)
  size_t cand_per_query = getenv("ORB_B200_MATCH_BUDGET") ? std::max(1, atoi(getenv("ORB_B200_MATCH_BUDGET"))) : 24;
  // asynchronous mode (device-resident problems only): one batch may be in flight per handle
  bool async_mode = false, pending = false;
  int pending_count = 0;
  std::vector<size_t> pending_off;
  int32_t* pending_results = nullptr;
  std::vector<ProjProblem> pending_P;  // the staged problems of the batch in flight (inputs stay in in_arena)
  size_t pending_in_bytes = 0;
  int finish_pending();

  int init() {
    if (initialized) return 0;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
      set_last_error("no CUDA device: orb_slam3_b200 has no CPU path");
      return ORB_E_NODEVICE;
    }
    CUDA_TRYM(cudaSetDevice(device));
    CUDA_TRYM(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    CUDA_TRYM(cudaEventCreate(&ev0));
    CUDA_TRYM(cudaEventCreate(&ev1));
    initialized = true;
    return 0;
  }
  ~Matcher() {
    if (!initialized) return;
    cudaSetDevice(device);
    if (in_arena.d) cudaFree(in_arena.d);
    if (scratch.d) cudaFree(scratch.d);
    if (out_arena.d) cudaFree(out_arena.d);
    if (h_in.h) cudaFreeHost(h_in.h);
    if (h_out.h) cudaFreeHost(h_out.h);
    cudaEventDestroy(ev0);
    cudaEventDestroy(ev1);
    cudaStreamDestroy(stream);
  }
};

// Lays out host arrays in the staging blob (two passes: size, then copy).
struct Stager {
  bool on_device;          // every array of the views already lives on the device
  bool frame_dev = false;  // only the frame's keys / u_right / desc do (an extractor's device results)
  uint8_t* h_base = nullptr;
  uint8_t* d_base = nullptr;
  size_t off = 0;
  template <class T>
  const T* put(const T* src, size_t count) {
    if (!src) return nullptr;
    if (on_device) return src;
    const size_t bytes = count * sizeof(T);
    const size_t o = off;
    off = (off + bytes + 15) & ~(size_t)15;
    if (h_base) memcpy(h_base + o, src, bytes);
    return (const T*)(d_base + o);
  }
};

static void stage_frame(Stager& st, const orb_frame_view& v, DevFrame& d) {
  d.n = v.n;
  if (st.frame_dev) {
    d.keys = v.keys; d.u_right = v.u_right; d.desc = v.desc;
  } else {
    d.keys = st.put(v.keys, v.n);
    d.u_right = st.put(v.u_right, v.n);
    d.desc = st.put(v.desc, (size_t)v.n * 32);
  }
  d.kp_taken = st.put(v.kp_taken, v.n);
  d.min_x = v.min_x; d.min_y = v.min_y; d.max_x = v.max_x; d.max_y = v.max_y;
  d.gwi = v.grid_w_inv; d.ghi = v.grid_h_inv;
  d.n_levels = v.n_levels;
  // scale tables are tiny and always host-side
  Stager hs = st; hs.on_device = false;
  d.scale = hs.put(v.scale_factors, v.n_levels);
  d.sigma2 = hs.put(v.level_sigma2, v.n_levels);
  st.off = hs.off;
  d.fx = v.fx; d.fy = v.fy; d.cx = v.cx; d.cy = v.cy; d.bf = v.bf; d.b = v.b;
}

template <class T>
static T* carve_dev(Arena& a, size_t count) { return (T*)(a.d + a.take(count * sizeof(T))); }

static int launch_projection(Matcher& M, std::vector<ProjProblem>& P, size_t in_bytes, bool all_on_device,
                             int32_t* const* assign_out, int32_t* results, bool allow_async);

// ORB_B200_MATCH_DEBUG: resolution rounds and event time of the batch that just completed, on stderr
static void debug_rounds(const Matcher& M, int kind, int count, const std::vector<size_t>& out_off) {
  static const bool dbg = getenv("ORB_B200_MATCH_DEBUG") != nullptr;
  if (!dbg) return;
  long long rs = 0;
  int rmax = 0;
  for (int k = 0; k < count; k++) {
    const int r = ((const int*)(M.h_out.h + out_off[k]))[2];
    rs += r; rmax = std::max(rmax, r);
  }
  fprintf(stderr, "[orbb200 match] kind %d: %d problems, resolution rounds mean %.1f max %d, %.3f ms\n", kind, count,
          (double)rs / count, rmax, M.last_ms);
}

int Matcher::finish_pending() {
  if (!pending) return 0;
  pending = false;
  cudaStream_t s = user_stream ? user_stream : stream;
  CUDA_TRYM(cudaStreamSynchronize(s));
  float ms = 0;
  cudaEventElapsedTime(&ms, ev0, ev1);
  last_ms = ms;
  bool overflow = false;
  for (int k = 0; k < pending_count; k++)
    if (((const int*)(h_out.h + pending_off[k]))[1]) overflow = true;
  if (overflow) {
    // the candidate lists of some problem did not fit: grow the budget and run the batch again, synchronously,
    // from the inputs that are still staged on the device (the caller never sees the overflow)
    cand_per_query *= 4;
    return launch_projection(*this, pending_P, pending_in_bytes, true, nullptr, pending_results, false) < 0
               ? ORB_E_CAPACITY : 0;
  }
  debug_rounds(*this, pending_P.empty() ? -1 : pending_P[0].kind, pending_count, pending_off);
  for (int k = 0; k < pending_count; k++) pending_results[k] = ((const int*)(h_out.h + pending_off[k]))[0];
  return 0;
}

static int run_projection(Matcher& M, int count, int kind, const orb_frame_view* F, const orb_mappoint_view* mps,
                          const orb_lastframe_view* last, const float* Tcw, const int32_t* forward,
                          const int32_t* backward, float th, float ratio, int far_points, float th_far,
                          int check_ori, int32_t* const* assign_out, int32_t* results, int on_device) {
  if (count <= 0 || !F || !assign_out || !results) { set_last_error("bad argument"); return ORB_E_ARG; }
  int rc = M.init();
  if (rc) return rc;
  CUDA_TRYM(cudaSetDevice(M.device));
  if ((rc = M.finish_pending())) return rc;  // the arenas are about to be reused
  // on_device: 0 = host views, 1 = every array of the views is device memory (assign_out too),
  //            2 = only the frames' keys / u_right / desc are device memory (an extractor's results)
  const bool all_dev = on_device == 1;
  std::vector<ProjProblem> P(count);
  // ---- stage inputs (sizing pass, then copy pass)
  Stager st{all_dev};
  st.frame_dev = on_device == 2;
  for (int pass = 0; pass < 2; pass++) {
    st.off = 0;
    for (int k = 0; k < count; k++) {
      ProjProblem& p = P[k];
      memset(&p, 0, sizeof(p));
      stage_frame(st, F[k], p.F);
      p.kind = kind;
      if (kind == 0) {
        const orb_mappoint_view& m = mps[k];
        p.nq = m.n;
        p.in_view = st.put(m.track_in_view, m.n); p.is_bad = st.put(m.is_bad, m.n);
        p.has_obs = st.put(m.has_obs, m.n);
        p.px = st.put(m.proj_x, m.n); p.py = st.put(m.proj_y, m.n); p.pxr = st.put(m.proj_xr, m.n);
        p.lvl = st.put(m.scale_level, m.n); p.vcos = st.put(m.view_cos, m.n); p.depth = st.put(m.depth, m.n);
        p.qdesc = st.put(m.desc, (size_t)m.n * 32);
      } else {
        const orb_lastframe_view& l = last[k];
        p.nq = l.n;
        p.has_mp = st.put(l.has_mp, l.n); p.has_obs = st.put(l.has_obs, l.n);
        p.wpos = st.put(l.world_pos, (size_t)l.n * 3); p.qdesc = st.put(l.desc, (size_t)l.n * 32);
        p.octave = st.put(l.octave, l.n); p.angle = st.put(l.angle, l.n);
        memcpy(p.T, Tcw + 7 * k, sizeof(float) * 7);
        p.forward = forward ? forward[k] : 0; p.backward = backward ? backward[k] : 0;
        p.check_ori = check_ori;
      }
      p.th = th; p.ratio = ratio; p.far_points = far_points; p.th_far = th_far;
    }
    if (pass == 0) {
      const size_t need = st.off;
      if (M.h_in.reserve(std::max<size_t>(need, 16))) return ORB_E_CUDA;
      if (M.in_arena.reserve(std::max<size_t>(need, 16))) return ORB_E_CUDA;
      st.h_base = M.h_in.h;
      st.d_base = M.in_arena.d;
    }
  }
  return launch_projection(M, P, st.off, all_dev, assign_out, results, true);
}

// Scratch / output carving, the three kernels and the result read-back of a staged batch.  A candidate-buffer
// overflow grows the budget and runs the batch again from the staged inputs.
static int launch_projection(Matcher& M, std::vector<ProjProblem>& P, size_t in_bytes, bool on_device,
                             int32_t* const* assign_out, int32_t* results, bool allow_async) {
  const int count = (int)P.size();
  for (int attempt = 0; attempt < 6; attempt++) {
    // ---- scratch + outputs
    size_t sbytes = 0, obytes = 0;
    for (int k = 0; k < count; k++) {
      const size_t nq = P[k].nq, nk = P[k].F.n, cc = std::max<size_t>(nq * M.cand_per_query, 16);
      sbytes += 256 * 16 + (GRID_CELLS + 1 + nk) * 4 + nk * 16 + nq * (4 * 4 + 1 + 8) + 4 + cc * 6 + nk * 8;
      obytes += 256 * 2 + nk * 4 + 8;
    }
    sbytes += sizeof(ProjProblem) * count + 4096;
    if (M.scratch.reserve(sbytes)) return ORB_E_CUDA;
    if (M.out_arena.reserve(obytes)) return ORB_E_CUDA;
    if (M.h_out.reserve(obytes)) return ORB_E_CUDA;
    M.scratch.used = 0; M.out_arena.used = 0;
    ProjProblem* d_probs = carve_dev<ProjProblem>(M.scratch, count);
    int max_nq = 0;
    std::vector<size_t> out_off(count);
    for (int k = 0; k < count; k++) {
      ProjProblem& p = P[k];
      const size_t nq = p.nq, nk = p.F.n, cc = std::max<size_t>(nq * M.cand_per_query, 16);
      max_nq = std::max(max_nq, p.nq);
      p.F.cell_start = carve_dev<int>(M.scratch, GRID_CELLS + 1);
      p.F.cell_items = carve_dev<int>(M.scratch, nk);
      p.F.cell_rec = carve_dev<uint4>(M.scratch, nk);
      p.q_cnt = carve_dev<int>(M.scratch, nq); p.ulist = carve_dev<int>(M.scratch, 2 * nq);
      p.q_state = carve_dev<uint8_t>(M.scratch, nq);
      p.acc_kp = carve_dev<int>(M.scratch, nq); p.acc_bin = carve_dev<int>(M.scratch, nq);
      p.cand_idx = carve_dev<int>(M.scratch, cc); p.cand_dist = carve_dev<unsigned short>(M.scratch, cc);
      p.cand_slot = (int)M.cand_per_query;
      p.minidx = carve_dev<int>(M.scratch, nk); p.takenby = carve_dev<int>(M.scratch, nk);
      if (on_device) {
        if (assign_out) p.assign = assign_out[k];  // (a retry keeps the pointer staged by the first launch)
        p.result = carve_dev<int>(M.out_arena, 3);
        out_off[k] = (uint8_t*)p.result - M.out_arena.d;
      } else {
        out_off[k] = M.out_arena.used;
        p.result = carve_dev<int>(M.out_arena, 3);
        p.assign = carve_dev<int>(M.out_arena, nk);
      }
    }
    cudaStream_t s = M.user_stream ? M.user_stream : M.stream;
    CUDA_TRYM(cudaEventRecord(M.ev0, s));
    if (in_bytes)  // host views: everything; device views: only the scale tables were staged
      CUDA_TRYM(cudaMemcpyAsync(M.in_arena.d, M.h_in.h, in_bytes, cudaMemcpyHostToDevice, s));
    CUDA_TRYM(cudaMemcpyAsync(d_probs, P.data(), sizeof(ProjProblem) * count, cudaMemcpyHostToDevice, s));
    grid_build_kernel<<<count, 256, 0, s>>>(d_probs);
    const int q_per_cta = PC_WARPS * PC_Q_PER_WARP;
    if (max_nq > 0) proj_candidates_kernel<<<dim3((max_nq + q_per_cta - 1) / q_per_cta, count), PC_WARPS * 32, 0, s>>>(d_probs);
    {
      int max_nk = 0;
      for (int k = 0; k < count; k++) max_nk = std::max(max_nk, P[k].F.n);
      int smem_nk = (max_nk + 3) & ~3;
      size_t smem_bytes = (size_t)smem_nk * 9;
      if (smem_bytes > 160 * 1024) { smem_nk = 0; smem_bytes = 0; }
      CUDA_TRYM(raise_dynamic_smem((const void*)proj_resolve_kernel, smem_bytes, M.device));
      proj_resolve_kernel<<<count, 1024, smem_bytes, s>>>(d_probs, smem_nk);
    }
    M.launches += 3;
    const size_t out_bytes = M.out_arena.used;
    CUDA_TRYM(cudaMemcpyAsync(M.h_out.h, M.out_arena.d, out_bytes, cudaMemcpyDeviceToHost, s));
    CUDA_TRYM(cudaEventRecord(M.ev1, s));
    if (allow_async && M.async_mode && on_device) {
      // results land in `results` at match_synchronize() / the next batch on this handle
      M.pending = true; M.pending_count = count; M.pending_off = out_off; M.pending_results = results;
      M.pending_P = P; M.pending_in_bytes = in_bytes;
      return count;
    }
    CUDA_TRYM(cudaStreamSynchronize(s));
    float ms = 0;
    cudaEventElapsedTime(&ms, M.ev0, M.ev1);
    M.last_ms = ms;
    bool overflow = false;
    for (int k = 0; k < count; k++) {
      const int* r = (const int*)(M.h_out.h + out_off[k]);
      if (r[1]) overflow = true;
    }
    if (overflow) { M.cand_per_query *= 4; continue; }
    debug_rounds(M, P[0].kind, count, out_off);
    for (int k = 0; k < count; k++) {
      const int* r = (const int*)(M.h_out.h + out_off[k]);
      results[k] = r[0];
      if (!on_device) {
        const uint8_t* a = M.h_out.h + ((uint8_t*)P[k].assign - M.out_arena.d);
        memcpy(assign_out[k], a, sizeof(int) * P[k].F.n);
      }
    }
    return count;
  }
  set_last_error("candidate buffer overflow");
  return ORB_E_CAPACITY;
}

static int run_triangulate(Matcher& M, int count, const orb_frame_view* kf1, const orb_frame_view* kf2,
                           const orb_featvec_view* fv1, const orb_featvec_view* fv2, const float* F12,
                           const float* ep, int only_stereo, int coarse, int check_ori, int32_t* const* pairs_out,
                           int cap, int32_t* results, int on_device) {
  if (count <= 0 || !kf1 || !kf2 || !fv1 || !fv2 || !F12 || !ep || !pairs_out || !results || cap <= 0) {
    set_last_error("bad argument");
    return ORB_E_ARG;
  }
  int rc = M.init();
  if (rc) return rc;
  CUDA_TRYM(cudaSetDevice(M.device));
  if ((rc = M.finish_pending())) return rc;
  std::vector<TriProblem> P(count);
  Stager st{on_device != 0};
  std::vector<int> nfeat(count);
  for (int k = 0; k < count; k++) {
    if (on_device) { set_last_error("match_triangulate_batch: on_device needs host-visible ptr arrays"); }
  }
  for (int pass = 0; pass < 2; pass++) {
    st.off = 0;
    for (int k = 0; k < count; k++) {
      TriProblem& p = P[k];
      memset(&p, 0, sizeof(p));
      stage_frame(st, kf1[k], p.K1);
      stage_frame(st, kf2[k], p.K2);
      // the CSR row pointers are read on the host for sizing: always host memory
      Stager hs = st; hs.on_device = false;
      p.n_nodes1 = fv1[k].n_nodes; p.n_nodes2 = fv2[k].n_nodes;
      p.nid1 = hs.put(fv1[k].node_ids, fv1[k].n_nodes); p.nid2 = hs.put(fv2[k].node_ids, fv2[k].n_nodes);
      p.ptr1 = hs.put(fv1[k].ptr, fv1[k].n_nodes + 1); p.ptr2 = hs.put(fv2[k].ptr, fv2[k].n_nodes + 1);
      p.n_feat1 = fv1[k].n_nodes ? fv1[k].ptr[fv1[k].n_nodes] : 0;
      const int n_feat2 = fv2[k].n_nodes ? fv2[k].ptr[fv2[k].n_nodes] : 0;
      p.idx1 = hs.put(fv1[k].idx, p.n_feat1); p.idx2 = hs.put(fv2[k].idx, n_feat2);
      st.off = hs.off;
      memcpy(p.F12, F12 + 9 * k, sizeof(float) * 9);
      p.ep[0] = ep[2 * k]; p.ep[1] = ep[2 * k + 1];
      p.only_stereo = only_stereo; p.coarse = coarse; p.check_ori = check_ori; p.cap = cap;
    }
    if (pass == 0) {
      if (M.h_in.reserve(std::max<size_t>(st.off, 16))) return ORB_E_CUDA;
      if (M.in_arena.reserve(std::max<size_t>(st.off, 16))) return ORB_E_CUDA;
      st.h_base = M.h_in.h;
      st.d_base = M.in_arena.d;
    }
  }
  const size_t in_bytes = st.off;
  size_t sbytes = sizeof(TriProblem) * count + 4096, obytes = 0;
  for (int k = 0; k < count; k++) {
    sbytes += 256 * 4 + (size_t)P[k].K1.n * 8;
    obytes += 256 * 2 + 8 + (size_t)cap * 8;
  }
  if (M.scratch.reserve(sbytes) || M.out_arena.reserve(obytes) || M.h_out.reserve(obytes)) return ORB_E_CUDA;
  M.scratch.used = 0; M.out_arena.used = 0;
  TriProblem* d_probs = carve_dev<TriProblem>(M.scratch, count);
  int max_feat = 0;
  std::vector<size_t> res_off(count), pair_off(count);
  for (int k = 0; k < count; k++) {
    TriProblem& p = P[k];
    max_feat = std::max(max_feat, p.n_feat1);
    p.match12 = carve_dev<int>(M.scratch, p.K1.n);
    p.bins = carve_dev<int>(M.scratch, p.K1.n);
    res_off[k] = M.out_arena.used;
    p.result = carve_dev<int>(M.out_arena, 3);
    if (on_device) p.pairs = pairs_out[k];
    else { pair_off[k] = M.out_arena.used; p.pairs = carve_dev<int>(M.out_arena, 2 * (size_t)cap); }
  }
  cudaStream_t s = M.user_stream ? M.user_stream : M.stream;
  CUDA_TRYM(cudaEventRecord(M.ev0, s));
  if (in_bytes) CUDA_TRYM(cudaMemcpyAsync(M.in_arena.d, M.h_in.h, in_bytes, cudaMemcpyHostToDevice, s));
  CUDA_TRYM(cudaMemcpyAsync(d_probs, P.data(), sizeof(TriProblem) * count, cudaMemcpyHostToDevice, s));
  for (int k = 0; k < count; k++)
    CUDA_TRYM(cudaMemsetAsync(P[k].match12, 0xff, sizeof(int) * P[k].K1.n, s));
  if (max_feat > 0) tri_match_kernel<<<dim3((max_feat + 127) / 128, count), 128, 0, s>>>(d_probs);
  tri_finish_kernel<<<count, 1024, 0, s>>>(d_probs);
  M.launches += 2;
  CUDA_TRYM(cudaMemcpyAsync(M.h_out.h, M.out_arena.d, M.out_arena.used, cudaMemcpyDeviceToHost, s));
  CUDA_TRYM(cudaEventRecord(M.ev1, s));
  CUDA_TRYM(cudaStreamSynchronize(s));
  float ms = 0;
  cudaEventElapsedTime(&ms, M.ev0, M.ev1);
  M.last_ms = ms;
  int worst = 0;
  for (int k = 0; k < count; k++) {
    const int* r = (const int*)(M.h_out.h + res_off[k]);
    results[k] = r[0];
    if (r[1]) worst = ORB_E_CAPACITY;
    if (!on_device) memcpy(pairs_out[k], M.h_out.h + pair_off[k], sizeof(int) * 2 * (size_t)std::min(r[0], cap));
  }
  if (worst) { set_last_error("pair buffer too small"); return worst; }
  return count;
}

// A FeatureVector over n keypoints as bow_match_kernel needs it: node ids strictly ascending, ptr non-decreasing
// from >= 0, every index inside [0, n) and in at most one node (DBoW2::transform files each feature once).  A bad
// index would be read out of bounds on the device, so host views are checked before anything is launched.
static bool featvec_ok(const orb_featvec_view& f, int n, std::vector<uint8_t>& seen) {
  if (f.n_nodes < 0) return false;
  if (f.n_nodes == 0) return true;
  if (!f.node_ids || !f.ptr || f.ptr[0] < 0) return false;
  for (int k = 0; k < f.n_nodes; k++) {
    if (f.ptr[k + 1] < f.ptr[k]) return false;
    if (k > 0 && f.node_ids[k] <= f.node_ids[k - 1]) return false;
  }
  if (f.ptr[f.n_nodes] > f.ptr[0] && !f.idx) return false;
  seen.assign(std::max(n, 0), 0);
  for (int p = f.ptr[0]; p < f.ptr[f.n_nodes]; p++) {
    const int i = f.idx[p];
    if (i < 0 || i >= n || seen[i]) return false;
    seen[i] = 1;
  }
  return true;
}

static bool bow_view_ok(const orb_frame_view& v, bool dev) {
  return v.n >= 0 && v.n < (1 << BOW_POS_BITS) && (v.n == 0 || dev || (v.keys && v.desc));
}

// kind 0: q = keyframes, c = frames (on_device 2: the frames' keys / desc are an extractor's device results);
// kind 1: q = KF1, c = KF2.  outs[k] has c[k].n (kind 0) or q[k].n (kind 1) entries.
static int run_bow(Matcher& M, int count, int kind, const orb_frame_view* q, const uint8_t* const* okq,
                   const orb_featvec_view* fvq, const orb_frame_view* c, const uint8_t* const* okc,
                   const orb_featvec_view* fvc, float ratio, int check_ori, int32_t* const* outs, int32_t* results,
                   int on_device) {
  if (count <= 0 || !q || !okq || !fvq || !c || !fvc || (kind == 1 && !okc) || !outs || !results ||
      on_device < 0 || on_device > (kind == 0 ? 2 : 1)) {
    set_last_error("bad argument");
    return ORB_E_ARG;
  }
  const bool all_dev = on_device == 1;
  std::vector<uint8_t> seen;
  for (int k = 0; k < count; k++) {
    if (!bow_view_ok(q[k], all_dev) || !bow_view_ok(c[k], on_device != 0) || !outs[k] ||
        (q[k].n > 0 && !okq[k]) || (kind == 1 && c[k].n > 0 && !okc[k])) {
      set_last_error("bad argument: view, map point flags or output");
      return ORB_E_ARG;
    }
    if (!all_dev && (!featvec_ok(fvq[k], q[k].n, seen) || !featvec_ok(fvc[k], c[k].n, seen))) {
      set_last_error("malformed FeatureVector: node ids must ascend, ptr must not decrease, every index must lie in "
                     "[0, n) and occur once");
      return ORB_E_ARG;
    }
  }
  int rc = M.init();
  if (rc) return rc;
  CUDA_TRYM(cudaSetDevice(M.device));
  if ((rc = M.finish_pending())) return rc;
  std::vector<BowProblem> P(count);
  Stager st{all_dev};
  for (int pass = 0; pass < 2; pass++) {
    st.off = 0;
    for (int k = 0; k < count; k++) {
      BowProblem& p = P[k];
      memset(&p, 0, sizeof(p));
      p.kind = kind;
      p.nq = q[k].n; p.nc = c[k].n;
      p.kq = st.put(q[k].keys, q[k].n); p.dq = st.put(q[k].desc, (size_t)q[k].n * 32);
      p.okq = st.put(okq[k], q[k].n);
      if (on_device == 2) {
        p.kc = c[k].keys; p.dc = c[k].desc;
      } else {  // Relocalization matches one frame against many keyframes: the frame is staged once
        int j = 0;
        while (j < k && !(c[j].keys == c[k].keys && c[j].desc == c[k].desc && c[j].n == c[k].n)) j++;
        if (j < k) { p.kc = P[j].kc; p.dc = P[j].dc; }
        else { p.kc = st.put(c[k].keys, c[k].n); p.dc = st.put(c[k].desc, (size_t)c[k].n * 32); }
      }
      if (kind == 1) p.okc = st.put(okc[k], c[k].n);
      // device views (on_device 1): the CSR arrays are the caller's device memory; only n_nodes is read here
      p.nodes_q = fvq[k].n_nodes; p.nodes_c = fvc[k].n_nodes;
      const size_t fq = (all_dev || !fvq[k].n_nodes) ? 0 : (size_t)fvq[k].ptr[fvq[k].n_nodes];
      const size_t fc = (all_dev || !fvc[k].n_nodes) ? 0 : (size_t)fvc[k].ptr[fvc[k].n_nodes];
      p.nid_q = st.put(fvq[k].node_ids, fvq[k].n_nodes); p.nid_c = st.put(fvc[k].node_ids, fvc[k].n_nodes);
      p.ptr_q = st.put(fvq[k].ptr, fvq[k].n_nodes + 1); p.ptr_c = st.put(fvc[k].ptr, fvc[k].n_nodes + 1);
      p.idx_q = st.put(fvq[k].idx, fq); p.idx_c = st.put(fvc[k].idx, fc);
      p.ratio = ratio; p.check_ori = check_ori;
      p.n_out = kind == 0 ? c[k].n : q[k].n;
    }
    if (pass == 0) {
      if (M.h_in.reserve(std::max<size_t>(st.off, 16))) return ORB_E_CUDA;
      if (M.in_arena.reserve(std::max<size_t>(st.off, 16))) return ORB_E_CUDA;
      st.h_base = M.h_in.h;
      st.d_base = M.in_arena.d;
    }
  }
  const size_t in_bytes = st.off;
  size_t sbytes = sizeof(BowProblem) * count + 4096, obytes = 0;
  for (int k = 0; k < count; k++) {
    sbytes += 512 + (size_t)P[k].n_out * 4 + (size_t)P[k].nc;
    obytes += 512 + (all_dev ? 0 : (size_t)P[k].n_out * 4);
  }
  if (M.scratch.reserve(sbytes) || M.out_arena.reserve(obytes) || M.h_out.reserve(obytes)) return ORB_E_CUDA;
  M.scratch.used = 0; M.out_arena.used = 0;
  BowProblem* d_probs = carve_dev<BowProblem>(M.scratch, count);
  int max_nodes = 0;
  std::vector<size_t> res_off(count), out_off(count);
  for (int k = 0; k < count; k++) {
    BowProblem& p = P[k];
    max_nodes = std::max(max_nodes, p.nodes_q);
    p.bins = carve_dev<int>(M.scratch, p.n_out);
    p.free_c = carve_dev<uint8_t>(M.scratch, p.nc);
    res_off[k] = M.out_arena.used;
    p.result = carve_dev<int>(M.out_arena, 1);
    if (all_dev) p.out = outs[k];
    else { out_off[k] = M.out_arena.used; p.out = carve_dev<int>(M.out_arena, p.n_out); }
  }
  cudaStream_t s = M.user_stream ? M.user_stream : M.stream;
  CUDA_TRYM(cudaEventRecord(M.ev0, s));
  if (in_bytes) CUDA_TRYM(cudaMemcpyAsync(M.in_arena.d, M.h_in.h, in_bytes, cudaMemcpyHostToDevice, s));
  CUDA_TRYM(cudaMemcpyAsync(d_probs, P.data(), sizeof(BowProblem) * count, cudaMemcpyHostToDevice, s));
  bow_init_kernel<<<count, 256, 0, s>>>(d_probs);
  if (max_nodes > 0) bow_match_kernel<<<dim3((max_nodes + BOW_WARPS - 1) / BOW_WARPS, count), BOW_WARPS * 32, 0, s>>>(d_probs);
  bow_finish_kernel<<<count, 1024, 0, s>>>(d_probs);
  M.launches += 2 + (max_nodes > 0);
  CUDA_TRYM(cudaGetLastError());
  CUDA_TRYM(cudaMemcpyAsync(M.h_out.h, M.out_arena.d, M.out_arena.used, cudaMemcpyDeviceToHost, s));
  CUDA_TRYM(cudaEventRecord(M.ev1, s));
  CUDA_TRYM(cudaStreamSynchronize(s));
  float ms = 0;
  cudaEventElapsedTime(&ms, M.ev0, M.ev1);
  M.last_ms = ms;
  for (int k = 0; k < count; k++) {
    results[k] = *(const int*)(M.h_out.h + res_off[k]);
    if (!all_dev && P[k].n_out) memcpy(outs[k], M.h_out.h + out_off[k], sizeof(int) * (size_t)P[k].n_out);
  }
  return count;
}

}  // namespace orbb200

using orbb200::Matcher;
struct orb_matcher { Matcher m; };

extern "C" {

int ham_distance(const uint8_t* a, const uint8_t* b) {
  int d = 0;
  for (int i = 0; i < 32; i += 8) {
    unsigned long long x, y;
    memcpy(&x, a + i, 8);
    memcpy(&y, b + i, 8);
    d += __builtin_popcountll(x ^ y);
  }
  return d;
}

int match_create(int device, orb_matcher** out) {
  if (!out || device < 0) return ORB_E_ARG;
  *out = new orb_matcher();
  (*out)->m.device = device;
  return ORB_OK;
}
void match_destroy(orb_matcher* m) { delete m; }

int match_project_local(orb_matcher* m, const orb_frame_view* F, const orb_mappoint_view* mps, float th,
                        float nn_ratio, int far_points, float th_far, int32_t* assign_out) {
  if (!m) return ORB_E_ARG;
  int32_t res = 0;
  int32_t* outs[1] = {assign_out};
  int rc = orbb200::run_projection(m->m, 1, 0, F, mps, nullptr, nullptr, nullptr, nullptr, th, nn_ratio, far_points,
                                   th_far, 0, outs, &res, 0);
  return rc < 0 ? rc : res;
}

int match_project_last(orb_matcher* m, const orb_frame_view* cur, const orb_lastframe_view* last,
                       const float* Tcw_qt7, int forward, int backward, float th, int check_orientation,
                       int32_t* assign_out) {
  if (!m) return ORB_E_ARG;
  int32_t res = 0, f = forward, b = backward;
  int32_t* outs[1] = {assign_out};
  int rc = orbb200::run_projection(m->m, 1, 1, cur, nullptr, last, Tcw_qt7, &f, &b, th, 0.f, 0, 0.f,
                                   check_orientation, outs, &res, 0);
  return rc < 0 ? rc : res;
}

int match_triangulate(orb_matcher* m, const orb_frame_view* kf1, const orb_frame_view* kf2,
                      const orb_featvec_view* fv1, const orb_featvec_view* fv2, const float* F12_rowmajor9,
                      const float* ep2, int only_stereo, int coarse, int check_orientation, int32_t* pairs_out,
                      int cap) {
  if (!m) return ORB_E_ARG;
  int32_t res = 0;
  int32_t* outs[1] = {pairs_out};
  int rc = orbb200::run_triangulate(m->m, 1, kf1, kf2, fv1, fv2, F12_rowmajor9, ep2, only_stereo, coarse,
                                    check_orientation, outs, cap, &res, 0);
  return rc < 0 ? rc : res;
}

int match_project_last_batch(orb_matcher* m, int count, const orb_frame_view* cur, const orb_lastframe_view* last,
                             const float* Tcw_qt7, const int32_t* forward, const int32_t* backward, float th,
                             int check_orientation, int32_t* const* assign_out, int32_t* results, int on_device) {
  if (!m) return ORB_E_ARG;
  return orbb200::run_projection(m->m, count, 1, cur, nullptr, last, Tcw_qt7, forward, backward, th, 0.f, 0, 0.f,
                                 check_orientation, assign_out, results, on_device);
}

int match_project_local_batch(orb_matcher* m, int count, const orb_frame_view* F, const orb_mappoint_view* mps,
                              float th, float nn_ratio, int far_points, float th_far, int32_t* const* assign_out,
                              int32_t* results, int on_device) {
  if (!m) return ORB_E_ARG;
  return orbb200::run_projection(m->m, count, 0, F, mps, nullptr, nullptr, nullptr, nullptr, th, nn_ratio, far_points,
                                 th_far, 0, assign_out, results, on_device);
}

int match_triangulate_batch(orb_matcher* m, int count, const orb_frame_view* kf1, const orb_frame_view* kf2,
                            const orb_featvec_view* fv1, const orb_featvec_view* fv2, const float* F12_rowmajor9,
                            const float* ep2, int only_stereo, int coarse, int check_orientation,
                            int32_t* const* pairs_out, int cap, int32_t* results, int on_device) {
  if (!m) return ORB_E_ARG;
  return orbb200::run_triangulate(m->m, count, kf1, kf2, fv1, fv2, F12_rowmajor9, ep2, only_stereo, coarse,
                                  check_orientation, pairs_out, cap, results, on_device);
}

int match_bow_frame(orb_matcher* m, const orb_frame_view* kf, const uint8_t* kf_mp_ok, const orb_featvec_view* fv_kf,
                    const orb_frame_view* F, const orb_featvec_view* fv_f, float nn_ratio, int check_orientation,
                    int32_t* assign_out) {
  if (!m) return ORB_E_ARG;
  int32_t res = 0;
  int32_t* outs[1] = {assign_out};
  const uint8_t* ok[1] = {kf_mp_ok};
  int rc = orbb200::run_bow(m->m, 1, 0, kf, ok, fv_kf, F, nullptr, fv_f, nn_ratio, check_orientation, outs, &res, 0);
  return rc < 0 ? rc : res;
}

int match_bow_keyframes(orb_matcher* m, const orb_frame_view* kf1, const uint8_t* mp_ok1, const orb_featvec_view* fv1,
                        const orb_frame_view* kf2, const uint8_t* mp_ok2, const orb_featvec_view* fv2, float nn_ratio,
                        int check_orientation, int32_t* match12_out) {
  if (!m) return ORB_E_ARG;
  int32_t res = 0;
  int32_t* outs[1] = {match12_out};
  const uint8_t* ok1[1] = {mp_ok1};
  const uint8_t* ok2[1] = {mp_ok2};
  int rc = orbb200::run_bow(m->m, 1, 1, kf1, ok1, fv1, kf2, ok2, fv2, nn_ratio, check_orientation, outs, &res, 0);
  return rc < 0 ? rc : res;
}

int match_bow_frame_batch(orb_matcher* m, int count, const orb_frame_view* kf, const uint8_t* const* kf_mp_ok,
                          const orb_featvec_view* fv_kf, const orb_frame_view* F, const orb_featvec_view* fv_f,
                          float nn_ratio, int check_orientation, int32_t* const* assign_out, int32_t* results,
                          int on_device) {
  if (!m) return ORB_E_ARG;
  return orbb200::run_bow(m->m, count, 0, kf, kf_mp_ok, fv_kf, F, nullptr, fv_f, nn_ratio, check_orientation,
                          assign_out, results, on_device);
}

int match_bow_keyframes_batch(orb_matcher* m, int count, const orb_frame_view* kf1, const uint8_t* const* mp_ok1,
                              const orb_featvec_view* fv1, const orb_frame_view* kf2, const uint8_t* const* mp_ok2,
                              const orb_featvec_view* fv2, float nn_ratio, int check_orientation,
                              int32_t* const* match12_out, int32_t* results, int on_device) {
  if (!m) return ORB_E_ARG;
  return orbb200::run_bow(m->m, count, 1, kf1, mp_ok1, fv1, kf2, mp_ok2, fv2, nn_ratio, check_orientation,
                          match12_out, results, on_device);
}

int match_set_stream(orb_matcher* m, void* cuda_stream) {
  if (!m) return ORB_E_ARG;
  m->m.user_stream = (cudaStream_t)cuda_stream;
  return ORB_OK;
}

int match_set_async(orb_matcher* m, int enabled) {
  if (!m) return ORB_E_ARG;
  m->m.async_mode = enabled != 0;
  return ORB_OK;
}

int match_synchronize(orb_matcher* m) {
  if (!m || !m->m.initialized) return ORB_E_ARG;
  cudaSetDevice(m->m.device);
  if (m->m.pending) return m->m.finish_pending();
  return cudaStreamSynchronize(m->m.user_stream ? m->m.user_stream : m->m.stream) == cudaSuccess ? ORB_OK : ORB_E_CUDA;
}
long long match_kernel_launches(const orb_matcher* m) { return m ? m->m.launches : 0; }
double match_last_ms(orb_matcher* m) { return m ? m->m.last_ms : 0.0; }

}  // extern "C"
