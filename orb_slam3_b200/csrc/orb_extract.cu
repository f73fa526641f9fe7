// ORB front-end for B200 (sm_100a): pyramid -> per-cell FAST-9/16 + NMS ->
// octree cull -> intensity-centroid angle -> 7x7 blur -> steered rBRIEF-256,
// batched over frames.  Replaces ORBextractor::operator() (reference
// src/ORBextractor.cc:1086-1168) behind the C ABI of include/orb_b200.h.
//
// All integer/float semantics follow SURVEY.md Appendix A (bit-exact with the
// CPU oracle): fixed-point bilinear resize, FAST score = max arc threshold - 1,
// per-cell NMS band + minTh fallback, libstdc++-ordered octree, strict-IEEE
// fastAtan2 and rBRIEF rotation (no FMA contraction: built with -fmad=false and
// explicit _rn intrinsics).
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/orb_b200.h"
#include "octree_core.h"
#include "orb_engine.h"
#include "cta_backend.cuh"
#include "glibc_sincosf.h"

namespace orbb200 {

// ----------------------------------------------------------------- constants
__constant__ int c_pattern[1024];  // (kept for reference; the kernels read the lane-transposed copy below)
__constant__ int c_umax[16];
static const int h_pattern[1024] = {
#include "pattern_31.inc"
};

static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }
const char* last_error() { return g_last_error.c_str(); }

#define CUDA_TRY(expr)                                                                  \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      set_last_error(std::string(#expr) + ": " + cudaGetErrorString(_e));               \
      return ORB_E_CUDA;                                                                \
    }                                                                                   \
  } while (0)

static inline int h_cv_round(float v) { return (int)lrintf(v); }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------- kernels

// cv::resize INTER_LINEAR 8UC1, fixed-point (SURVEY.md A.1); one launch per
// level over the whole batch, 4 output pixels per thread.
__global__ void __launch_bounds__(256)
resize_level_kernel(uint8_t* __restrict__ pyr, size_t frame_stride, size_t src_off, int sw, int sh,
                    int spitch, size_t dst_off, int dw, int dh, int dpitch,
                    const int* __restrict__ xofs, const short2* __restrict__ alpha,
                    const int* __restrict__ yofs, const short2* __restrict__ beta) {
  const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int y = blockIdx.y;
  if (x4 >= dw) return;
  uint8_t* base = pyr + (size_t)blockIdx.z * frame_stride;
  const uint8_t* S = base + src_off;
  const int sy = yofs[y];
  const int sy0 = min(max(sy, 0), sh - 1), sy1 = min(max(sy + 1, 0), sh - 1);
  const uint8_t* S0 = S + (size_t)sy0 * spitch;
  const uint8_t* S1 = S + (size_t)sy1 * spitch;
  const short2 b = beta[y];
  uint32_t packed = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const int x = x4 + k;
    int v = 0;
    if (x < dw) {
      const int sx = xofs[x];
      const int sx1 = min(sx + 1, sw - 1);
      const short2 a = alpha[x];
      const int h0 = S0[sx] * a.x + S0[sx1] * a.y;
      const int h1 = S1[sx] * a.x + S1[sx1] * a.y;
      v = (((b.x * (h0 >> 4)) >> 16) + ((b.y * (h1 >> 4)) >> 16) + 2) >> 2;
    }
    packed |= (uint32_t)(v & 0xff) << (8 * k);
  }
  *reinterpret_cast<uint32_t*>(base + dst_off + (size_t)y * dpitch + x4) = packed;
}

// Same arithmetic, staged: one CTA produces RS_ROWS consecutive output rows of one frame.  The (<= RS_SRC) source
// rows they touch are copied to shared memory with coalesced 16-byte loads; the four byte gathers per output
// pixel then hit shared memory instead of issuing four global loads each, and the per-column tables
// (xofs, alpha) are read once per thread and reused for every row of the CTA.
constexpr int RS_ROWS = 4, RS_SRC = 8, RS_THREADS = 256;

__global__ void __launch_bounds__(RS_THREADS)
resize_rows_kernel(uint8_t* __restrict__ pyr, size_t frame_stride, size_t src_off, int sw, int sh, int spitch,
                   size_t dst_off, int dw, int dh, int dpitch, const int* __restrict__ xofs,
                   const short2* __restrict__ alpha, const int* __restrict__ yofs, const short2* __restrict__ beta) {
  extern __shared__ __align__(16) uint8_t rs_rows[];  // [RS_SRC][spitch]
  __shared__ int s_y[RS_ROWS];
  uint8_t* base = pyr + (size_t)blockIdx.y * frame_stride;
  const uint8_t* S = base + src_off;
  const int y0 = blockIdx.x * RS_ROWS, ny = min(RS_ROWS, dh - y0);
  // source rows [lo, hi]: yofs is non-decreasing, rows are clamped like the reference clamps sy and sy + 1
  const int lo = min(max(yofs[y0], 0), sh - 1), hi = min(max(yofs[y0 + ny - 1] + 1, 0), sh - 1);
  const int nsrc = hi - lo + 1;  // <= RS_SRC for down-scaling factors up to 2 (host-checked)
  const int vec = spitch >> 4;   // the slab pitch is a multiple of 64
  for (int i = threadIdx.x; i < nsrc * vec; i += RS_THREADS) {
    const int r = i / vec, c = i - r * vec;
    reinterpret_cast<uint4*>(rs_rows + (size_t)r * spitch)[c] =
        reinterpret_cast<const uint4*>(S + (size_t)(lo + r) * spitch)[c];
  }
  if (threadIdx.x < ny) s_y[threadIdx.x] = yofs[y0 + threadIdx.x];
  __syncthreads();
  for (int x4 = threadIdx.x * 4; x4 < dw; x4 += RS_THREADS * 4) {
    int sx[4], sx1[4];
    short2 a[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int x = min(x4 + k, dw - 1);
      sx[k] = xofs[x];
      sx1[k] = min(sx[k] + 1, sw - 1);
      a[k] = alpha[x];
    }
    for (int r = 0; r < ny; r++) {
      const int y = y0 + r, sy = s_y[r];
      const uint8_t* S0 = rs_rows + (size_t)(min(max(sy, 0), sh - 1) - lo) * spitch;
      const uint8_t* S1 = rs_rows + (size_t)(min(max(sy + 1, 0), sh - 1) - lo) * spitch;
      const short2 b = beta[y];
      uint32_t packed = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int h0 = S0[sx[k]] * a[k].x + S0[sx1[k]] * a[k].y;
        const int h1 = S1[sx[k]] * a[k].x + S1[sx1[k]] * a[k].y;
        const int v = (((b.x * (h0 >> 4)) >> 16) + ((b.y * (h1 >> 4)) >> 16) + 2) >> 2;
        if (x4 + k < dw) packed |= (uint32_t)(v & 0xff) << (8 * k);
      }
      *reinterpret_cast<uint32_t*>(base + dst_off + (size_t)y * dpitch + x4) = packed;
    }
  }
}

// Third form of the same arithmetic (default): the four output pixels of a thread read a span of at most eight
// consecutive source bytes, so instead of eight byte loads per source row pair the thread loads three aligned words
// per row, shifts them to the span's start (2 SHF) and picks each pixel's byte pair with one PRMT whose selector is
// fixed for the thread; the horizontal pass h = S[sx] * a.x + S[sx1] * a.y is then ONE integer dot product
// (IDP.2A: two signed 16-bit coefficients x two unsigned bytes).  ncu on resize_rows_kernel: LSU-bound on the byte
// gathers from shared memory (issue 67 %, DRAM 7 %).  Requires the span sx1[3] - sx[0] <= 7 (host-checked: any
// down-scaling factor up to 2; ORB-SLAM3's is 1.2).
__global__ void __launch_bounds__(RS_THREADS)
resize_words_kernel(uint8_t* __restrict__ pyr, size_t frame_stride, size_t src_off, int sw, int sh, int spitch,
                    size_t dst_off, int dw, int dh, int dpitch, const int* __restrict__ xofs,
                    const short2* __restrict__ alpha, const int* __restrict__ yofs, const short2* __restrict__ beta) {
  extern __shared__ __align__(16) uint8_t rs_rows[];  // [RS_SRC][spitch] + 16 bytes of slack for the last word loads
  __shared__ int s_y[RS_ROWS];
  uint8_t* base = pyr + (size_t)blockIdx.y * frame_stride;
  const uint8_t* S = base + src_off;
  const int y0 = blockIdx.x * RS_ROWS, ny = min(RS_ROWS, dh - y0);
  const int lo = min(max(yofs[y0], 0), sh - 1), hi = min(max(yofs[y0 + ny - 1] + 1, 0), sh - 1);
  const int nsrc = hi - lo + 1;
  const int vec = spitch >> 4;
  for (int i = threadIdx.x; i < nsrc * vec; i += RS_THREADS) {
    const int r = i / vec, c = i - r * vec;
    reinterpret_cast<uint4*>(rs_rows + (size_t)r * spitch)[c] =
        reinterpret_cast<const uint4*>(S + (size_t)(lo + r) * spitch)[c];
  }
  if (threadIdx.x < ny) s_y[threadIdx.x] = yofs[y0 + threadIdx.x];
  __syncthreads();
  for (int x4 = threadIdx.x * 4; x4 < dw; x4 += RS_THREADS * 4) {
    uint32_t selp[4], ab[4];
    int sx0 = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int x = min(x4 + k, dw - 1);
      const int sx = xofs[x], sx1 = min(sx + 1, sw - 1);
      if (k == 0) sx0 = sx;
      // PRMT selector: byte 0 <- span[sx - sx0], byte 1 <- span[sx1 - sx0], bytes 2, 3 <- (don't care)
      selp[k] = (uint32_t)(sx - sx0) | ((uint32_t)(sx1 - sx0) << 4);
      const short2 a = alpha[x];
      ab[k] = (uint32_t)(uint16_t)a.x | ((uint32_t)(uint16_t)a.y << 16);
    }
    const int w0 = sx0 >> 2, sh8 = (sx0 & 3) * 8;
    for (int r = 0; r < ny; r++) {
      const int y = y0 + r, sy = s_y[r];
      const uint32_t* R0 = reinterpret_cast<const uint32_t*>(rs_rows + (size_t)(min(max(sy, 0), sh - 1) - lo) * spitch) + w0;
      const uint32_t* R1 = reinterpret_cast<const uint32_t*>(rs_rows + (size_t)(min(max(sy + 1, 0), sh - 1) - lo) * spitch) + w0;
      const uint32_t a0 = R0[0], a1 = R0[1], a2 = R0[2], c0 = R1[0], c1 = R1[1], c2 = R1[2];
      // the eight bytes that start at sx0, of both rows
      const uint32_t p0 = __funnelshift_r(a0, a1, sh8), p1 = __funnelshift_r(a1, a2, sh8);
      const uint32_t q0 = __funnelshift_r(c0, c1, sh8), q1 = __funnelshift_r(c1, c2, sh8);
      const short2 b = beta[y];
      uint32_t packed = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        // unsigned overload: unsigned 16-bit coefficients (<= 2048) x unsigned bytes, lo16 * byte 0 + hi16 * byte 1
        const int h0 = (int)__dp2a_lo(ab[k], __byte_perm(p0, p1, selp[k]), 0u);
        const int h1 = (int)__dp2a_lo(ab[k], __byte_perm(q0, q1, selp[k]), 0u);
        const int v = (((b.x * (h0 >> 4)) >> 16) + ((b.y * (h1 >> 4)) >> 16) + 2) >> 2;
        if (x4 + k < dw) packed |= (uint32_t)(v & 0xff) << (8 * k);
      }
      *reinterpret_cast<uint32_t*>(base + dst_off + (size_t)y * dpitch + x4) = packed;
    }
  }
}

// Copy the caller's level-0 images (arbitrary pitch / frame stride, device memory) into the
// pyramid slabs: one launch for the whole batch, 16-byte accesses when the layout allows.
__global__ void __launch_bounds__(256)
copy_level0_kernel(const uint8_t* __restrict__ src, size_t src_frame_stride, size_t src_step,
                   uint8_t* __restrict__ pyr, size_t frame_stride, int w, int h, int pitch, int vec16) {
  const int y = blockIdx.y;
  const uint8_t* s = src + (size_t)blockIdx.z * src_frame_stride + (size_t)y * src_step;
  uint8_t* d = pyr + (size_t)blockIdx.z * frame_stride + (size_t)y * pitch;
  if (vec16) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i * 16 < w) reinterpret_cast<uint4*>(d)[i] = reinterpret_cast<const uint4*>(s)[i];
  } else {
    for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < w; x += gridDim.x * blockDim.x) d[x] = s[x];
  }
}

// FAST-9/16 score of the centre pixel from its ring; returns best (=score+1) or
// 0 when the pixel is not a corner at threshold t.
__device__ __forceinline__ int fast_best(const uint8_t* __restrict__ c, int pitch, int t) {
  const int v = c[0];
  const int hi = v + t, lo = v - t;
  // a 9-arc contains one end of every diameter: test 2 diameters first
  const int r0 = c[3 * pitch], r8 = c[-3 * pitch];
  bool bp = (r0 > hi) | (r8 > hi), dp = (r0 < lo) | (r8 < lo);
  if (!(bp | dp)) return 0;
  const int r4 = c[3], r12 = c[-3];
  bp = bp & ((r4 > hi) | (r12 > hi));
  dp = dp & ((r4 < lo) | (r12 < lo));
  if (!(bp | dp)) return 0;
  int r[16];
  r[0] = r0; r[8] = r8; r[4] = r4; r[12] = r12;
  r[1] = c[3 * pitch + 1];  r[2] = c[2 * pitch + 2];   r[3] = c[pitch + 3];
  r[5] = c[-pitch + 3];     r[6] = c[-2 * pitch + 2];  r[7] = c[-3 * pitch + 1];
  r[9] = c[-3 * pitch - 1]; r[10] = c[-2 * pitch - 2]; r[11] = c[-pitch - 3];
  r[13] = c[pitch - 3];     r[14] = c[2 * pitch - 2];  r[15] = c[3 * pitch - 1];
  // bright arcs: v - max(window9 of r); dark arcs: min(window9 of r) - v
  int mx2[16], mn2[16];
#pragma unroll
  for (int k = 0; k < 16; k++) { mx2[k] = max(r[k], r[(k + 1) & 15]); mn2[k] = min(r[k], r[(k + 1) & 15]); }
  int mx4[16], mn4[16];
#pragma unroll
  for (int k = 0; k < 16; k++) { mx4[k] = max(mx2[k], mx2[(k + 2) & 15]); mn4[k] = min(mn2[k], mn2[(k + 2) & 15]); }
  int best = 0;
#pragma unroll
  for (int k = 0; k < 16; k++) {
    const int mx9 = max(max(mx4[k], mx4[(k + 4) & 15]), r[(k + 8) & 15]);
    const int mn9 = min(min(mn4[k], mn4[(k + 4) & 15]), r[(k + 8) & 15]);
    best = max(best, max(v - mx9, mn9 - v));
  }
  return best > t ? best : 0;
}

// The same score on packed 16-bit halves: the 9-arcs starting at ring positions k and k+8 are evaluated together
// in the two halves of one register (VIMNMX.U16x2 / VIMNMX3.U16x2 are native on sm_100a), and
// max_k max(v - mx9[k], mn9[k] - v) = max(v - min_k mx9[k], max_k mn9[k] - v) moves the subtraction out of
// the loop.  P[k] = (r[k], r[k+8]); every array index k+8 is the half-swapped entry k.  No early exit: the callers
// only pass pixels that already survived the packed 4-diameter test.
__device__ __forceinline__ int fast_best_packed(const uint8_t* __restrict__ c, int pitch, int t) {
  const int v = c[0];
  uint32_t r[16];
  r[0] = c[3 * pitch];      r[8] = c[-3 * pitch];      r[4] = c[3];               r[12] = c[-3];
  r[1] = c[3 * pitch + 1];  r[2] = c[2 * pitch + 2];   r[3] = c[pitch + 3];
  r[5] = c[-pitch + 3];     r[6] = c[-2 * pitch + 2];  r[7] = c[-3 * pitch + 1];
  r[9] = c[-3 * pitch - 1]; r[10] = c[-2 * pitch - 2]; r[11] = c[-pitch - 3];
  r[13] = c[pitch - 3];     r[14] = c[2 * pitch - 2];  r[15] = c[3 * pitch - 1];
  uint32_t P[12];
#pragma unroll
  for (int k = 0; k < 8; k++) P[k] = r[k] | (r[k + 8] << 16);
#pragma unroll
  for (int k = 8; k < 12; k++) P[k] = __byte_perm(P[k - 8], 0, 0x1032);
  uint32_t X2[10], N2[10];  // max / min over ring positions [k, k+1]
#pragma unroll
  for (int k = 0; k < 8; k++) { X2[k] = __vmaxu2(P[k], P[k + 1]); N2[k] = __vminu2(P[k], P[k + 1]); }
#pragma unroll
  for (int k = 8; k < 10; k++) { X2[k] = __byte_perm(X2[k - 8], 0, 0x1032); N2[k] = __byte_perm(N2[k - 8], 0, 0x1032); }
  uint32_t X4[12], N4[12];  // [k, k+3]
#pragma unroll
  for (int k = 0; k < 8; k++) { X4[k] = __vmaxu2(X2[k], X2[k + 2]); N4[k] = __vminu2(N2[k], N2[k + 2]); }
#pragma unroll
  for (int k = 8; k < 12; k++) { X4[k] = __byte_perm(X4[k - 8], 0, 0x1032); N4[k] = __byte_perm(N4[k - 8], 0, 0x1032); }
  uint32_t minmx = 0xffffffffu, maxmn = 0u;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const uint32_t last = k + 8 < 12 ? P[k + 8] : __byte_perm(P[k], 0, 0x1032);  // ring position k+8 | k
    const uint32_t mx9 = __vimax3_u16x2(X4[k], X4[k + 4], last);   // arcs [k, k+8] | [k+8, k+16]
    const uint32_t mn9 = __vimin3_u16x2(N4[k], N4[k + 4], last);
    minmx = __vminu2(minmx, mx9);
    maxmn = __vmaxu2(maxmn, mn9);
  }
  const int m1 = (int)min(minmx & 0xffffu, minmx >> 16), m2 = (int)max(maxmn & 0xffffu, maxmn >> 16);
  const int best = max(v - m1, m2 - v);
  return best > t ? best : 0;
}

// One CTA per FAST cell of ComputeKeyPointsOctTree (ORBextractor.cc:805-872):
// score map at minTh in shared memory, 3x3 strict NMS inside the cell's band,
// keep score>=iniTh survivors, or all survivors when there is none.
//   1. the cell tile comes in as aligned 32-bit words (one warp per row);
//   2. every band pixel takes the cheap two-diameter rejection test; the few that
//      pass are compacted into a shared-memory queue (ballot + popc), so
//   3. the full 16-ring score and 4. the NMS / emission only ever run on dense
//      queues -- no warp drags 31 rejected lanes through the expensive path.
constexpr int FAST_THREADS = 128;
constexpr int FAST_TILE_MAX = 76;    // TMA box rows: hCell+6 <= 76
constexpr int FAST_TILE_PITCH = 96;  // TMA box columns (bytes): (x0 & 15) + wCell+6 <= 91, multiple of 16
constexpr int FAST_BAND_MAX = 70;

struct LevelTensorMaps {
  CUtensorMap m[64];  // one 3-D (x, y, frame) uint8 map per pyramid level: [0,16) box of fast_cells_kernel,
                      // [16,32) box of fast_warp_kernel, [32,48) raw patch box of describe_tma_kernel,
                      // [48,64) its blurred patch box (over the blurred slab)
};

__global__ void __launch_bounds__(FAST_THREADS)
fast_cells_kernel(const CUtensorMap* __restrict__ maps, int frame0,
                  const CellDesc* __restrict__ cells, const LevelDev* __restrict__ lv, int ini_th,
                  int min_th, Cand* __restrict__ cand, size_t cand_frame_stride,
                  int* __restrict__ cand_count, int nlevels) {
  __shared__ __align__(128) uint8_t tile[FAST_TILE_MAX * FAST_TILE_PITCH];
  __shared__ __align__(8) unsigned long long tma_bar;
  __shared__ __align__(16) uint8_t smap[(FAST_BAND_MAX + 2) * (FAST_BAND_MAX + 2) + 8];
  __shared__ unsigned short queue[FAST_BAND_MAX * FAST_BAND_MAX];
  __shared__ int s_qn, s_cnt_all, s_base;
  __shared__ int s_warp_tot[FAST_THREADS / 32];
  const CellDesc cd = cells[blockIdx.x];
  const LevelDev L = lv[cd.level];
  const int f = blockIdx.y;
  const int tw = cd.x1 - cd.x0, th = cd.y1 - cd.y0;
  const int bw = tw - 6, bh = th - 6;
  if (bw <= 0 || bh <= 0) return;
  const int sw = bw + 2;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // 1. the cell tile arrives through TMA: one 96x76 box of the (x, y, frame) tensor of this level,
  //    issued by one thread, completion signalled on an mbarrier (out-of-image bytes are zero-filled
  //    and never read by a band pixel)
  const unsigned bar_addr = (unsigned)__cvta_generic_to_shared(&tma_bar);
  if (threadIdx.x == 0) {
    s_qn = 0; s_cnt_all = 0;
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_addr));
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(tile);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_addr),
                 "r"(FAST_TILE_MAX * FAST_TILE_PITCH)
                 : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(maps + cd.level), "r"(bar_addr), "r"(cd.x0 & ~15), "r"(cd.y0), "r"(frame0 + f)
        : "memory");
  }
  {
    const int nz = ((bw + 2) * (bh + 2) + 3) >> 2;
    for (int i = threadIdx.x; i < nz; i += FAST_THREADS) reinterpret_cast<uint32_t*>(smap)[i] = 0;
  }
  {
    unsigned done = 0;
    while (!done) {
      asm volatile(
          "{\n.reg .pred p;\n"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n"
          "selp.u32 %0, 1, 0, p;\n}"
          : "=r"(done)
          : "r"(bar_addr)
          : "memory");
    }
  }
  __syncthreads();
  const int ox = cd.x0 & 15;  // the box starts at the 16-byte aligned column left of the cell (TMA needs
                              // 16-byte aligned global row starts)
  // The reference calls cv::FAST(cell, iniThFAST) and only when that returns nothing
  // cv::FAST(cell, minThFAST) (:826-846).  Same here: pass 0 at iniTh (few pixels survive the
  // cheap test), pass 1 at minTh only for the rare cells that came out empty.
  // 4-pixel groups = aligned words of a tile row that overlap the band columns [ox+3, ox+3+bw)
  const int g0 = (ox + 3) >> 2, ng = ((ox + 3 + bw + 3) >> 2) - g0;
  const int nitems = bh * ng;                           // <= 70 * 19
  const unsigned magic_g = ((1u << 20) + ng - 1) / ng;  // idx / ng for idx < 70*19
  unsigned long long keep_bits = 0;
  int qn = 0;
  for (int pass = 0; pass < 2; pass++) {
    const int th_fast = pass == 0 ? ini_th : min_th;
    if (pass == 1) {
      const int nz = ((bw + 2) * (bh + 2) + 3) >> 2;
      for (int i = threadIdx.x; i < nz; i += FAST_THREADS) reinterpret_cast<uint32_t*>(smap)[i] = 0;
    }
    // 2. cheap rejection, 4 pixels per thread on packed bytes: a 9-arc contains one end of every
    //    diameter, so a corner needs |ring - centre| > t at one end of each of the 8 diameters; 4
    //    diameters are tested with VABSDIFF4 + a SWAR compare on aligned 32-bit shared-memory
    //    words (sign consistency is left to the exact test: the filter only has to be a superset).
    //    Survivors stay as one bit per (visit, byte): <= 11 visits x 4.
    unsigned long long pass_bits = 0;
    {
      const uint32_t* tw32 = reinterpret_cast<const uint32_t*>(tile);
      constexpr int PWD = FAST_TILE_PITCH / 4;
      const uint32_t t4 = 0x01010101u * (uint32_t)th_fast;
      int it = 0;
      for (int idx = threadIdx.x; idx < nitems; idx += FAST_THREADS, it++) {
        const int y = (int)(((unsigned)idx * magic_g) >> 20), g = g0 + (idx - y * ng);
        const uint32_t* rc = tw32 + (y + 3) * PWD + g;  // centre row, word g
        const uint32_t v = rc[0];
        const uint32_t r0 = rc[3 * PWD], r8 = rc[-3 * PWD];
        const uint32_t r4 = __funnelshift_r(rc[0], rc[1], 24), r12 = __funnelshift_r(rc[-1], rc[0], 8);
        const uint32_t* rp = rc + 2 * PWD;
        const uint32_t* rm = rc - 2 * PWD;
        const uint32_t r2 = __funnelshift_r(rp[0], rp[1], 16), r14 = __funnelshift_r(rp[-1], rp[0], 16);
        const uint32_t r6 = __funnelshift_r(rm[0], rm[1], 16), r10 = __funnelshift_r(rm[-1], rm[0], 16);
        uint32_t m = __vcmpgtu4(__vabsdiffu4(r0, v), t4) | __vcmpgtu4(__vabsdiffu4(r8, v), t4);
        m &= __vcmpgtu4(__vabsdiffu4(r4, v), t4) | __vcmpgtu4(__vabsdiffu4(r12, v), t4);
        m &= __vcmpgtu4(__vabsdiffu4(r2, v), t4) | __vcmpgtu4(__vabsdiffu4(r10, v), t4);
        m &= __vcmpgtu4(__vabsdiffu4(r6, v), t4) | __vcmpgtu4(__vabsdiffu4(r14, v), t4);
        if (m) {
          // keep bytes whose column lies inside the band [ox+3, ox+3+bw)
          unsigned nib = ((m >> 7) & 1u) | ((m >> 14) & 2u) | ((m >> 21) & 4u) | ((m >> 28) & 8u);
          const int c0 = 4 * g - (ox + 3);  // band x of byte 0
#pragma unroll
          for (int k = 0; k < 4; k++)
            if ((unsigned)(c0 + k) >= (unsigned)bw) nib &= ~(1u << k);
          pass_bits |= (unsigned long long)nib << (4 * it);
        }
      }
    }
    // compaction of the survivors into the queue: one block-wide exclusive scan
    {
      const int cnt = __popcll(pass_bits);
      int incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      __syncthreads();  // previous pass is done with s_warp_tot / queue / smap zeroing is visible
      if (lane == 31) s_warp_tot[warp] = incl;
      if (threadIdx.x == 0) { s_cnt_all = 0; }
      __syncthreads();
      int base = incl - cnt;
      for (int w = 0; w < warp; w++) base += s_warp_tot[w];
      if (threadIdx.x == FAST_THREADS - 1) s_qn = base + cnt;
      while (pass_bits) {
        const int bit = __ffsll((long long)pass_bits) - 1;
        pass_bits &= pass_bits - 1;
        const int idx = threadIdx.x + (bit >> 2) * FAST_THREADS;
        const int y = (int)(((unsigned)idx * magic_g) >> 20), g = g0 + (idx - y * ng);
        const int x = 4 * g + (bit & 3) - (ox + 3);
        queue[base++] = (unsigned short)((y << 8) | x);
      }
    }
    __syncthreads();
    qn = s_qn;
    // 3. exact segment test + score (max arc threshold) of the queued pixels, dense lanes
    for (int q = threadIdx.x; q < qn; q += FAST_THREADS) {
      const int e = queue[q], y = e >> 8, x = e & 255;
      const int best = fast_best(&tile[(y + 3) * FAST_TILE_PITCH + ox + x + 3], FAST_TILE_PITCH, th_fast);
      smap[(y + 1) * sw + x + 1] = (uint8_t)best;
    }
    __syncthreads();
    // 4. strict 3x3 NMS on the queue; a thread remembers its survivors as one bit per visit
    keep_bits = 0;
    int it = 0;
    for (int q = threadIdx.x; q < qn; q += FAST_THREADS, it++) {
      const int e = queue[q], y = e >> 8, x = e & 255;
      const uint8_t* p = &smap[(y + 1) * sw + x + 1];
      const int s = p[0];
      if (s && s > p[-1] && s > p[1] && s > p[-sw - 1] && s > p[-sw] && s > p[-sw + 1] &&
          s > p[sw - 1] && s > p[sw] && s > p[sw + 1])
        keep_bits |= 1ull << it;
    }
    if (keep_bits) atomicAdd(&s_cnt_all, __popcll(keep_bits));
    __syncthreads();
    if (s_cnt_all > 0 || ini_th == min_th) break;
  }
  const int total = s_cnt_all;
  if (total == 0) return;
  if (threadIdx.x == 0) s_base = atomicAdd(&cand_count[f * nlevels + cd.level], total);
  __syncthreads();
  if (!keep_bits) return;
  // the order inside the level's list is irrelevant (the octree uses order keys)
  Cand* out = cand + (size_t)f * cand_frame_stride + L.cand_off;
  int it = 0;
  for (int q = threadIdx.x; q < qn; q += FAST_THREADS, it++) {
    if (!(keep_bits & (1ull << it))) continue;
    const int e = queue[q], y = e >> 8, x = e & 255;
    const int pos = atomicAdd(&s_base, 1);
    if (pos < L.cand_cap) {
      Cand c;
      c.xy = (uint32_t)(x + 3 + cd.shift_x) | ((uint32_t)(y + 3 + cd.shift_y) << 16);
      c.score = (uint32_t)(smap[(y + 1) * sw + x + 1] - 1);
      out[pos] = c;
    }
  }
}

// ---- FAST, second formulation: ONE WARP PER CELL, persistent, TMA ring ----------------------------------------
// Same per-cell semantics as fast_cells_kernel above, reorganised around what the profile of that kernel showed
// (profiles/r1_fast_breakdown.md): a quarter of its stall samples sat in a prologue that waits for the CTA's own
// tile, a fifth of its instructions were a block-wide scan with two barriers per pass, and its packed `d > t`
// compare cost five instructions.  Here every warp owns a cell at a time and walks the (cell, frame) list with
// stride = warps in the grid; the tile of its NEXT cell is already in flight (cp.async.bulk.tensor into the other
// half of a two-slot ring, one mbarrier per slot) while it works on the current one; all hand-offs inside the
// cell are warp-synchronous (ballot / shuffle prefix sums, __syncwarp) -- there is no __syncthreads in the
// kernel; the packed threshold test is ((d & 0x7f..) + K | d) on the byte MSBs (3 instructions per sample).
// The box starts at the 16-byte aligned column left of the cell (TMA needs that) and is only as large as the
// largest cell of the image size needs: 64 x 48 bytes at 1280x720 (3 KB per cell instead of 7.3 KB through L2).
struct FastGeom {
  int tile_pitch, tile_rows, tile_bytes;  // TMA box = tile_pitch x tile_rows bytes (pitch multiple of 16)
  int smap_pitch, smap_bytes;             // score map with a one-pixel zero frame
  int queue_cap;                          // pre-test survivors of one cell (<= band pixels)
  int gq_off;                             // byte offset (from the end of the score map) of the 4-pixel group queue
  int per_warp_bytes;
};
constexpr int FASTW_WARPS = 8;

template <bool HI>
__device__ __forceinline__ uint32_t fast_gt4_msb(uint32_t d, uint32_t K) {
  // byte-wise d > t, result in bit 7 of every byte (other bits are garbage): t < 128: ((d & 0x7f) + 127 - t) | d,
  // t >= 128: ((d & 0x7f) + 255 - t) & d
  const uint32_t s = (d & 0x7f7f7f7fu) + K;
  return HI ? (s & d) : (s | d);
}

// Packed 4-diameter rejection test of one cell at threshold K (fast_gt4_msb) and compaction of the survivors into
// `queue`.  PWD = tile pitch in words (compile-time for the common 64-byte box).  Two steps, because per-pixel
// compaction inside the scan cost more than the test itself (four ballots per visit): the scan only appends the
// 4-pixel GROUPS that have a survivor (one ballot per visit, entry = first band column | row << 7 | nibble << 16)
// to `gq`; the groups are expanded to pixels afterwards, 32 at a time, with one warp prefix sum per 32 groups.
template <bool HI, int PWD_C>
__device__ __forceinline__ int fast_pretest(const uint32_t* __restrict__ tw32, int pwd_rt, unsigned short* queue,
                                            uint32_t* __restrict__ gq, int nitems, int ng, int g0, unsigned magic_g,
                                            int ox, int bw, uint32_t K, int lane) {
  const int PWD = PWD_C ? PWD_C : pwd_rt;
  const unsigned lt = (1u << lane) - 1u;
  int gn = 0;
  for (int base = 0; base < nitems; base += 32) {
    const int idx = base + lane;
    uint32_t m = 0;
    int y = 0, c0 = 0;
    if (idx < nitems) {
      y = (int)(((unsigned)idx * magic_g) >> 20);
      const int g = g0 + (idx - y * ng);
      const uint32_t* rc = tw32 + (y + 3) * PWD + g;
      const uint32_t v = rc[0];
      const uint32_t r0 = rc[3 * PWD], r8 = rc[-3 * PWD];
      const uint32_t r4 = __funnelshift_r(rc[0], rc[1], 24), r12 = __funnelshift_r(rc[-1], rc[0], 8);
      const uint32_t* rp = rc + 2 * PWD;
      const uint32_t* rm = rc - 2 * PWD;
      const uint32_t r2 = __funnelshift_r(rp[0], rp[1], 16), r14 = __funnelshift_r(rp[-1], rp[0], 16);
      const uint32_t r6 = __funnelshift_r(rm[0], rm[1], 16), r10 = __funnelshift_r(rm[-1], rm[0], 16);
      m = fast_gt4_msb<HI>(__vabsdiffu4(r0, v), K) | fast_gt4_msb<HI>(__vabsdiffu4(r8, v), K);
      m &= fast_gt4_msb<HI>(__vabsdiffu4(r4, v), K) | fast_gt4_msb<HI>(__vabsdiffu4(r12, v), K);
      m &= fast_gt4_msb<HI>(__vabsdiffu4(r2, v), K) | fast_gt4_msb<HI>(__vabsdiffu4(r10, v), K);
      m &= fast_gt4_msb<HI>(__vabsdiffu4(r6, v), K) | fast_gt4_msb<HI>(__vabsdiffu4(r14, v), K);
      m &= 0x80808080u;
      c0 = 4 * g - (ox + 3);  // band x of byte 0; only bytes whose column lies in [0, bw) count
      if (c0 < 0) m &= 0xffffffffu << (8 * -c0);
      if (c0 + 3 >= bw) m &= 0xffffffffu >> (8 * (c0 + 4 - bw));
    }
    const unsigned bal = __ballot_sync(0xffffffffu, m != 0);
    if (m) {
      const uint32_t nib = ((((m >> 7) & 0x01010101u) * 0x01020408u) >> 24) & 0xfu;  // byte MSBs -> bits 0..3
      gq[gn + __popc(bal & lt)] = (uint32_t)((y << 7) + c0 + 4) | (nib << 16);       // +4 keeps the low half >= 0
    }
    gn += __popc(bal);
  }
  __syncwarp();
  int qn = 0;
  for (int gb = 0; gb < gn; gb += 32) {
    const int gi = gb + lane;
    const uint32_t ent = gi < gn ? gq[gi] : 0u;
    const uint32_t nib = ent >> 16;
    const int cnt = __popc(nib);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    int pos = qn + incl - cnt;
    const int e0 = (int)(ent & 0xffffu) - 4;
#pragma unroll
    for (int k = 0; k < 4; k++)
      if ((nib >> k) & 1u) queue[pos++] = (unsigned short)(e0 + k);
    qn += __shfl_sync(0xffffffffu, incl, 31);
  }
  return qn;
}

template <int TP_C>
__global__ void __launch_bounds__(FASTW_WARPS * 32)
fast_warp_kernel(const CUtensorMap* __restrict__ maps, int frame0, int nframes, const CellDesc* __restrict__ cells,
                 int num_cells, const LevelDev* __restrict__ lv, int ini_th, int min_th, Cand* __restrict__ cand,
                 size_t cand_frame_stride, int* __restrict__ cand_count, int nlevels, FastGeom G) {
  extern __shared__ __align__(128) uint8_t fw_dyn[];
  __shared__ __align__(8) unsigned long long bars[FASTW_WARPS][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* wbase = fw_dyn + (size_t)warp * G.per_warp_bytes;
  uint8_t* smap = wbase + 2 * G.tile_bytes;
  unsigned short* queue = reinterpret_cast<unsigned short*>(smap + G.smap_bytes);
  uint32_t* gq = reinterpret_cast<uint32_t*>(smap + G.smap_bytes + G.gq_off);
  const unsigned bar0 = (unsigned)__cvta_generic_to_shared(&bars[warp][0]);
  const unsigned tile0 = (unsigned)__cvta_generic_to_shared(wbase);
  const int SW = G.smap_pitch, TP = TP_C ? TP_C : G.tile_pitch;
  const int total = num_cells * nframes;  // host-checked < 2^31
  const int gw = blockIdx.x * FASTW_WARPS + warp, NW = gridDim.x * FASTW_WARPS;
  // all mbarriers are initialised by one thread at CTA-uniform addresses; the only block-wide barrier of the kernel
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 0; w < FASTW_WARPS; w++) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(&bars[w][0])));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(&bars[w][1])));
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  for (int i = lane; i < G.smap_bytes / 4; i += 32) reinterpret_cast<uint32_t*>(smap)[i] = 0;
  __syncthreads();
  auto issue = [&](int item, int slot) {  // lane 0 only
    const int f = item / num_cells, c = item - f * num_cells;
    const CellDesc cd = cells[c];
    const unsigned bar = bar0 + 8 * slot, dst = tile0 + slot * G.tile_bytes;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(G.tile_bytes) : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(maps + cd.level), "r"(bar), "r"(cd.x0 & ~15), "r"(cd.y0), "r"(frame0 + f)
        : "memory");
  };
  if (gw < total && lane == 0) issue(gw, 0);
  const bool hi_ini = ini_th >= 128, hi_min = min_th >= 128;
  const uint32_t K_ini = 0x01010101u * (uint32_t)(hi_ini ? 255 - ini_th : 127 - ini_th);
  const uint32_t K_min = 0x01010101u * (uint32_t)(hi_min ? 255 - min_th : 127 - min_th);
  int n = 0;
  for (int item = gw; item < total; item += NW, n++) {
    const int slot = n & 1;
    // the other slot was read during the previous iteration; every lane is past it (the __syncwarp that ends
    // an iteration), so its refill can start now and overlaps this whole cell
    if (item + NW < total && lane == 0) issue(item + NW, slot ^ 1);
    {
      const unsigned bar = bar0 + 8 * slot, parity = (unsigned)(n >> 1) & 1u;
      unsigned done = 0;
      while (!done) {
        asm volatile(
            "{\n.reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
      }
    }
    const int f = item / num_cells, ci = item - f * num_cells;
    const CellDesc cd = cells[ci];
    const uint8_t* tile = wbase + slot * G.tile_bytes;
    const int bw = cd.x1 - cd.x0 - 6, bh = cd.y1 - cd.y0 - 6;
    if (bw > 0 && bh > 0) {
      const int ox = cd.x0 & 15;
      // 4-pixel groups = aligned words of a tile row that overlap the band columns [ox+3, ox+3+bw)
      const int g0 = (ox + 3) >> 2, ng = ((ox + 3 + bw + 3) >> 2) - g0;
      const int nitems = bh * ng;
      const unsigned magic_g = ((1u << 20) + ng - 1) / ng;  // idx / ng for idx < 2^20 / ng
      const uint32_t* tw32 = reinterpret_cast<const uint32_t*>(tile);
      int qn = 0, total_keep = 0;
      for (int pass = 0; pass < 2; pass++) {
        const int th_fast = pass == 0 ? ini_th : min_th;
        const uint32_t K = pass == 0 ? K_ini : K_min;
        // 2. packed 4-diameter rejection test; survivors go to the queue (order inside a cell is irrelevant)
        if (pass == 0 ? hi_ini : hi_min)
          qn = fast_pretest<true, TP_C / 4>(tw32, TP >> 2, queue, gq, nitems, ng, g0, magic_g, ox, bw, K, lane);
        else
          qn = fast_pretest<false, TP_C / 4>(tw32, TP >> 2, queue, gq, nitems, ng, g0, magic_g, ox, bw, K, lane);
        __syncwarp();
        // 3. exact segment test + score of the queued pixels on dense lanes
        for (int q = lane; q < qn; q += 32) {
          const int e = queue[q], y = e >> 7, x = e & 127;
          const int best = fast_best_packed(&tile[(y + 3) * TP + ox + x + 3], TP, th_fast);
          smap[(y + 1) * SW + x + 1] = (uint8_t)best;
        }
        __syncwarp();
        // 4. strict 3x3 NMS; survivors are marked in bit 15 of their queue entry
        total_keep = 0;
        for (int q0 = 0; q0 < qn; q0 += 32) {
          const int q = q0 + lane;
          bool keep = false;
          if (q < qn) {
            const int e = queue[q], y = e >> 7, x = e & 127;
            const uint8_t* p = &smap[(y + 1) * SW + x + 1];
            const int sc = p[0];
            keep = sc && sc > p[-1] && sc > p[1] && sc > p[-SW - 1] && sc > p[-SW] && sc > p[-SW + 1] &&
                   sc > p[SW - 1] && sc > p[SW] && sc > p[SW + 1];
            if (keep) queue[q] = (unsigned short)(e | 0x8000);
          }
          total_keep += __popc(__ballot_sync(0xffffffffu, keep));
        }
        if (total_keep > 0 || ini_th == min_th || pass == 1) break;
        // empty at iniTh (ORBextractor.cc:843-846): forget this pass' scores, try again at minTh
        for (int q = lane; q < qn; q += 32) {
          const int e = queue[q];
          smap[((e >> 7) + 1) * SW + (e & 127) + 1] = 0;
        }
        __syncwarp();
      }
      if (total_keep > 0) {
        const LevelDev L = lv[cd.level];
        int base = 0;
        if (lane == 0) base = atomicAdd(&cand_count[f * nlevels + cd.level], total_keep);
        base = __shfl_sync(0xffffffffu, base, 0);
        Cand* out = cand + (size_t)f * cand_frame_stride + L.cand_off;
        for (int q0 = 0; q0 < qn; q0 += 32) {
          const int q = q0 + lane;
          const int e = q < qn ? queue[q] : 0;
          const bool keep = (e & 0x8000) != 0;
          const unsigned bal = __ballot_sync(0xffffffffu, keep);
          if (keep) {
            const int y = (e >> 7) & 127, x = e & 127;
            const int pos = base + __popc(bal & ((1u << lane) - 1u));
            if (pos < L.cand_cap) {
              Cand c;
              c.xy = (uint32_t)(x + 3 + cd.shift_x) | ((uint32_t)(y + 3 + cd.shift_y) << 16);
              c.score = (uint32_t)(smap[(y + 1) * SW + x + 1] - 1);
              out[pos] = c;
            }
          }
          base += __popc(bal);
        }
      }
      // the score map goes back to all-zero for the next cell: only the entries this cell wrote
      __syncwarp();
      for (int q = lane; q < qn; q += 32) {
        const int e = queue[q];
        smap[(((e >> 7) & 127) + 1) * SW + (e & 127) + 1] = 0;
      }
    }
    __syncwarp();
  }
}

// One CTA per (level, frame): DistributeOctTree (octree_core.h).
constexpr int OCT_THREADS = 512;

__host__ __device__ inline size_t carve(size_t& off, size_t bytes) {
  size_t o = off;
  off = (off + bytes + 15) & ~(size_t)15;
  return o;
}

__host__ __device__ inline size_t octree_scratch_layout(uint8_t* base, int cand_cap, int node_cap,
                                                        OctreeScratch* s) {
  size_t off = 0;
  size_t o;
  o = carve(off, sizeof(int) * (size_t)cand_cap); if (s) s->pt_node = (int*)(base + o);
  o = carve(off, (size_t)cand_cap);               if (s) s->pt_q = base + o;
  for (int b = 0; b < 2; b++)
    for (int f = 0; f < 5; f++) {
      o = carve(off, sizeof(int) * (size_t)node_cap);
      if (s) s->nd[b][f] = (int*)(base + o);
    }
  o = carve(off, sizeof(int) * 4 * (size_t)node_cap); if (s) s->childcnt = (int*)(base + o);
  o = carve(off, sizeof(int) * 4 * (size_t)node_cap); if (s) s->cidx = (int*)(base + o);
  o = carve(off, sizeof(int) * 4 * (size_t)node_cap); if (s) s->eidx = (int*)(base + o);
  o = carve(off, sizeof(int) * 4 * (size_t)node_cap); if (s) s->remap = (int*)(base + o);
  o = carve(off, sizeof(int) * (size_t)node_cap); if (s) s->rank = (int*)(base + o);
  o = carve(off, sizeof(int) * (size_t)node_cap); if (s) s->proc = (int*)(base + o);
  o = carve(off, sizeof(int) * (size_t)node_cap); if (s) s->surv = (int*)(base + o);
  o = carve(off, sizeof(int) * (size_t)node_cap); if (s) s->tmp = (int*)(base + o);
  o = carve(off, sizeof(int) * (size_t)node_cap); if (s) s->expand_pos = (int*)(base + o);
  o = carve(off, sizeof(SortNode) * (size_t)node_cap); if (s) s->sortbuf = (SortNode*)(base + o);
  o = carve(off, sizeof(int) * 6 * (size_t)node_cap); if (s) s->sortwork = (int*)(base + o);
  o = carve(off, sizeof(unsigned long long) * (size_t)node_cap);
  if (s) s->best = (unsigned long long*)(base + o);
  return off;
}

__global__ void __launch_bounds__(OCT_THREADS)
octree_kernel(const Cand* __restrict__ cand, size_t cand_frame_stride, const int* __restrict__ cand_count,
              const LevelDev* __restrict__ lv, uint8_t* __restrict__ scratch, size_t scratch_frame_stride,
              int* __restrict__ sel, size_t sel_frame_stride, int* __restrict__ sel_count, int nlevels,
              int smem_node_cap, int smem_node_cap_full) {
  __shared__ int smem_ints[48];
  extern __shared__ __align__(16) int oct_dyn[];
  // level-major launch order (blockIdx.x = frame): all the heavy level-0 CTAs start in the first
  // wave and the light high levels back-fill the SMs as they drain
  const int level = blockIdx.y, f = blockIdx.x;
  const LevelDev L = lv[level];
  CtaBackend be;
  be.smem_ints = smem_ints;
  OctreeScratch s;
  octree_scratch_layout(scratch + (size_t)f * scratch_frame_stride + L.scratch_off, L.cand_cap,
                        L.oct.node_cap, &s);
  if (smem_node_cap >= L.oct.node_cap) {
    // the per-node arrays every point loop dereferences (bounds, counts, child counts, remap)
    // live in shared memory: ~30-cycle instead of ~300-cycle dependent loads
    int* q = oct_dyn;
    const int nc = L.oct.node_cap;
    for (int b = 0; b < 2; b++)
      for (int k = 0; k < 5; k++) { s.nd[b][k] = q; q += nc; }
    s.childcnt = q; q += 4 * nc;
    s.remap = q; q += 4 * nc;
    s.rank = q; q += nc;
    if (smem_node_cap_full >= L.oct.node_cap) {
      // second tier: everything the block scans walk and -- above all -- the buffer that ONE thread sorts with the
      // libstdc++-order introsort in the overshoot phase (a few thousand dependent accesses: ~30 cycles each here
      // instead of a trip to L1 / L2 per access)
      s.cidx = q; q += 4 * nc;
      s.eidx = q; q += 4 * nc;
      s.surv = q; q += nc;
      s.tmp = q; q += nc;
      s.proc = q; q += nc;
      s.expand_pos = q; q += nc;
      s.sortbuf = reinterpret_cast<SortNode*>(q + (nc & 1)); q += 2 * nc + 2;  // 8-byte aligned
      s.sortwork = q; q += 6 * nc;
    }
  }
  const int n = min(cand_count[f * nlevels + level], L.cand_cap);
  const Cand* c = cand + (size_t)f * cand_frame_stride + L.cand_off;
  int* out = sel + (size_t)f * sel_frame_stride + 3 * (size_t)L.sel_off;
  const int m = octree_select(be, c, n, L.oct, s, out);
  if (threadIdx.x == 0) sel_count[f * nlevels + level] = m;
}

// GaussianBlur 7x7 sigma 2 (SURVEY.md A.5) over every level of every frame.
// 128x32 output tile per CTA; aligned 32-bit loads, 4 pixels per thread in both
// passes, one coalesced 32-bit store per thread.
constexpr int BLUR_TW = 128, BLUR_TH = 58;  // TH + 6 staged rows = 32 row pairs
constexpr int BLUR_IW = BLUR_TW + 8;          // bytes per staged input row: [x0-4, x0+TW+4)
constexpr int BLUR_PAIRS = (BLUR_TH + 6) / 2;
static_assert(BLUR_TH % 2 == 0 && BLUR_TW % 4 == 0, "row pairs / 4-pixel groups");

__device__ __forceinline__ int reflect101(int p, int n) {
  if (p < 0) p = -p;
  if (p >= n) p = 2 * n - 2 - p;
  return min(max(p, 0), n - 1);
}

// 8.8 fixed-point taps of cv::GaussianBlur(7x7, sigma 2) (oracle orc_extract.cpp, reference call
// ORBextractor.cc:1110) as byte vectors for the integer dot-product instructions:
// horizontal: 7 u8 taps = IDP.4A over bytes [c-3, c] and [c+1, c+4) (8th weight 0);
// vertical:   rows are stored in pairs (row 2j | row 2j+1 << 16), 7 u16 taps = 4 IDP.2A.
constexpr uint32_t BLUR_K_LO = 18u | (34u << 8) | (48u << 16) | (56u << 24);
constexpr uint32_t BLUR_K_HI = 48u | (34u << 8) | (18u << 16);
constexpr uint32_t BLUR_K_ODD_A = (18u << 8) | (34u << 16) | (48u << 24);             // (0,18 | 34,48)
constexpr uint32_t BLUR_K_ODD_B = 56u | (48u << 8) | (34u << 16) | (18u << 24);      // (56,48 | 34,18)

__device__ __forceinline__ void blur_h4(const uint32_t* __restrict__ row, uint32_t o[4]) {
  const uint32_t w0 = row[0], w1 = row[1], w2 = row[2];
  // output k is centred on staged byte 4q+k+4: taps cover bytes 4q+k+1 .. 4q+k+7
  o[0] = __dp4a(__funnelshift_r(w0, w1, 8), BLUR_K_LO, __dp4a(__funnelshift_r(w1, w2, 8), BLUR_K_HI, 0u));
  o[1] = __dp4a(__funnelshift_r(w0, w1, 16), BLUR_K_LO, __dp4a(__funnelshift_r(w1, w2, 16), BLUR_K_HI, 0u));
  o[2] = __dp4a(__funnelshift_r(w0, w1, 24), BLUR_K_LO, __dp4a(__funnelshift_r(w1, w2, 24), BLUR_K_HI, 0u));
  o[3] = __dp4a(w1, BLUR_K_LO, __dp4a(w2, BLUR_K_HI, 0u));
}

__global__ void __launch_bounds__(256)
blur_kernel(const uint8_t* __restrict__ pyr, uint8_t* __restrict__ blr, size_t frame_stride,
            const BlurTile* __restrict__ tiles, const LevelDev* __restrict__ lv) {
  __shared__ __align__(16) uint8_t in[(BLUR_TH + 6) * BLUR_IW];
  __shared__ __align__(16) uint32_t hp[BLUR_PAIRS * BLUR_TW];  // horizontal sums, two rows per word
  const BlurTile t = tiles[blockIdx.x];
  const LevelDev L = lv[t.level];
  const uint8_t* src = pyr + (size_t)blockIdx.y * frame_stride + L.img_off;
  uint8_t* dst = blr + (size_t)blockIdx.y * frame_stride + L.img_off;
  const int w = L.w, h = L.h;
  const int out_rows = min(BLUR_TH, h - t.y0);           // rows of this tile inside the image
  const int in_rows = out_rows + 6;
  // stage [y0-3, y0+out_rows+3) x [x0-4, x0+TW+4) word by word; BORDER_REFLECT_101 at the true image
  // edge (bytes past the right edge feed only outputs that are never stored)
  for (int i = threadIdx.x; i < in_rows * (BLUR_IW / 4); i += 256) {
    const int r = i / (BLUR_IW / 4), c = i - r * (BLUR_IW / 4);
    const int gy = reflect101(t.y0 - 3 + r, h), gx = t.x0 - 4 + 4 * c;
    const uint8_t* rowp = src + (size_t)gy * L.pitch;
    uint32_t v;
    if (gx >= 0 && gx + 3 < w) {
      v = *reinterpret_cast<const uint32_t*>(rowp + gx);
    } else {
      v = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) v |= (uint32_t)rowp[reflect101(gx + k, w)] << (8 * k);
    }
    reinterpret_cast<uint32_t*>(in)[i] = v;
  }
  __syncthreads();
  // horizontal pass: one thread = 4 columns of one row pair, stored as (even row | odd row << 16)
  const int in_pairs = (in_rows + 1) >> 1;
  for (int i = threadIdx.x; i < in_pairs * (BLUR_TW / 4); i += 256) {
    const int j = i / (BLUR_TW / 4), q = i - j * (BLUR_TW / 4);
    uint32_t a[4], b[4];
    blur_h4(reinterpret_cast<const uint32_t*>(in + (2 * j) * BLUR_IW) + q, a);
    blur_h4(reinterpret_cast<const uint32_t*>(in + (2 * j + 1) * BLUR_IW) + q, b);  // row in_rows (odd count) is unused slack
    uint4 pk;
    pk.x = a[0] | (b[0] << 16); pk.y = a[1] | (b[1] << 16); pk.z = a[2] | (b[2] << 16); pk.w = a[3] | (b[3] << 16);
    reinterpret_cast<uint4*>(hp + j * BLUR_TW)[q] = pk;
  }
  __syncthreads();
  // vertical pass + rounding: one thread = 4 columns x 2 output rows (2jo, 2jo+1) from pairs jo..jo+3
  const int out_pairs = (out_rows + 1) >> 1;
  for (int i = threadIdx.x; i < out_pairs * (BLUR_TW / 4); i += 256) {
    const int jo = i / (BLUR_TW / 4), q = i - jo * (BLUR_TW / 4);
    const int gy = t.y0 + 2 * jo, gx = t.x0 + 4 * q;
    if (gx >= w) continue;
    const uint4 p0 = reinterpret_cast<const uint4*>(hp + (jo + 0) * BLUR_TW)[q];
    const uint4 p1 = reinterpret_cast<const uint4*>(hp + (jo + 1) * BLUR_TW)[q];
    const uint4 p2 = reinterpret_cast<const uint4*>(hp + (jo + 2) * BLUR_TW)[q];
    const uint4 p3 = reinterpret_cast<const uint4*>(hp + (jo + 3) * BLUR_TW)[q];
    uint32_t e[4], o[4];
#define BLUR_V(c, k)                                                                                       \
    e[k] = __dp2a_hi(p3.c, BLUR_K_HI, __dp2a_lo(p2.c, BLUR_K_HI, __dp2a_hi(p1.c, BLUR_K_LO,               \
             __dp2a_lo(p0.c, BLUR_K_LO, 1u << 15))));                                                      \
    o[k] = __dp2a_hi(p3.c, BLUR_K_ODD_B, __dp2a_lo(p2.c, BLUR_K_ODD_B, __dp2a_hi(p1.c, BLUR_K_ODD_A,      \
             __dp2a_lo(p0.c, BLUR_K_ODD_A, 1u << 15))));
    BLUR_V(x, 0) BLUR_V(y, 1) BLUR_V(z, 2) BLUR_V(w, 3)
#undef BLUR_V
    // (acc + 2^15) >> 16 < 256: the result is byte 2 of each accumulator
    const uint32_t oe = __byte_perm(__byte_perm(e[0], e[1], 0x0062), __byte_perm(e[2], e[3], 0x0062), 0x5410);
    const uint32_t oo = __byte_perm(__byte_perm(o[0], o[1], 0x0062), __byte_perm(o[2], o[3], 0x0062), 0x5410);
    // the pitch is a multiple of 64, so the (rare) partial last word stays inside the row
    *reinterpret_cast<uint32_t*>(dst + (size_t)gy * L.pitch + gx) = oe;
    if (gy + 1 < h) *reinterpret_cast<uint32_t*>(dst + (size_t)(gy + 1) * L.pitch + gx) = oo;
  }
}

// Output slot of every selected keypoint: operator() walks levels and list
// order, lapping-area points fill the array from the back (ORBextractor.cc
// :1122-1163).  One CTA per frame.
__global__ void __launch_bounds__(256)
layout_kernel(const int* __restrict__ sel, size_t sel_frame_stride, const int* __restrict__ sel_count,
              const LevelDev* __restrict__ lv, int nlevels, const int* __restrict__ lap,
              int* __restrict__ slot, int* __restrict__ n_out, int* __restrict__ mono_out, int out_cap) {
  __shared__ int smem_ints[48];
  __shared__ int s_total;
  CtaBackend be;
  be.smem_ints = smem_ints;
  const int f = blockIdx.x;
  const float lap0 = lap ? (float)lap[2 * f] : 0.f, lap1 = lap ? (float)lap[2 * f + 1] : 0.f;
  const int* fsel = sel + (size_t)f * sel_frame_stride;
  int* fslot = slot + (size_t)f * sel_frame_stride / 3;
  if (threadIdx.x == 0) {
    int t = 0;
    for (int l = 0; l < nlevels; l++) t += sel_count[f * nlevels + l];
    s_total = t;
  }
  __syncthreads();
  const int total = s_total;
  int mono = 0, stereo = total - 1;
  for (int l = 0; l < nlevels; l++) {
    const LevelDev L = lv[l];
    const int m = sel_count[f * nlevels + l];
    int* ls = fslot + L.sel_off;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      float x = (float)(fsel[3 * (L.sel_off + i)] + 16);  // minBorder added back (:884)
      if (l != 0) x = __fmul_rn(x, L.scale);
      ls[i] = (x >= lap0 && x <= lap1) ? 1 : 0;
    }
    __syncthreads();
    // ls[i] <- number of lapped points before i; then slot
    const int nlap = be.exclusive_scan(ls, m);
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      float x = (float)(fsel[3 * (L.sel_off + i)] + 16);  // minBorder added back (:884)
      if (l != 0) x = __fmul_rn(x, L.scale);
      const bool lapped = (x >= lap0 && x <= lap1);
      const int before = ls[i];
      const int pos = lapped ? (stereo - before) : (mono + (i - before));
      ls[i] = pos < out_cap ? pos : -1;
    }
    __syncthreads();
    mono += m - nlap;
    stereo -= nlap;
  }
  if (threadIdx.x == 0) { n_out[f] = total; mono_out[f] = mono; }
}

// cv::fastAtan2 (SURVEY.md A.4), every operation rounded to float.
__device__ __forceinline__ float fast_atan2_deg(float y, float x) {
  const float s180 = 57.29577951308232f;  // (float)(180/pi)
  const float p1 = __fmul_rn(0.9997878412794807f, s180), p3 = __fmul_rn(-0.3258083974640975f, s180);
  const float p5 = __fmul_rn(0.1555786518463281f, s180), p7 = __fmul_rn(-0.04432655554792128f, s180);
  const float ax = fabsf(x), ay = fabsf(y);
  const float eps = 2.220446049250313e-16f;
  float a;
  if (ax >= ay) {
    const float c = __fdiv_rn(ay, __fadd_rn(ax, eps));
    const float c2 = __fmul_rn(c, c);
    a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
  } else {
    const float c = __fdiv_rn(ax, __fadd_rn(ay, eps));
    const float c2 = __fmul_rn(c, c);
    a = __fsub_rn(90.f, __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c));
  }
  if (x < 0) a = __fsub_rn(180.f, a);
  if (y < 0) a = __fsub_rn(360.f, a);
  return a;
}

// One warp per selected keypoint: IC_Angle (ORBextractor.cc:76-103) on the raw level, computeOrbDescriptor
// (:107-146) on the blurred level, final KeyPoint fields (:880-890, :1149-1151), written to its output slot.  The two
// patches arrive as 2-D tiles through the tensor-memory accelerator -- the 31x31 raw patch of IC_Angle (box 48 x 32
// bytes of the level's raw tensor) and the 37x37 blurred patch of the steered pattern (box 64 x 38 bytes of the
// blurred tensor), both issued by lane 0 before any arithmetic and awaited on the warp's own mbarrier; the orientation
// moments and the 512 pattern samples then read shared memory only.  Boxes start at the 16-byte aligned column left
// of the patch.
constexpr int DT_WARPS = 8;
constexpr int DT_RAW_P = 48, DT_RAW_R = 32, DT_BLR_P = 64, DT_BLR_R = 38;
constexpr int DT_RAW_BYTES = DT_RAW_P * DT_RAW_R, DT_BLR_BYTES = DT_BLR_P * DT_BLR_R;  // 1536 + 2432: 128-byte multiples

__global__ void __launch_bounds__(DT_WARPS * 32)
describe_tma_kernel(const CUtensorMap* __restrict__ raw_maps, const CUtensorMap* __restrict__ blr_maps, int frame0,
                    const int* __restrict__ sel, size_t sel_frame_stride, const int* __restrict__ sel_count,
                    const int* __restrict__ slot, const LevelDev* __restrict__ lv, int nlevels,
                    const int* __restrict__ warp_level, const int* __restrict__ pattern_t,
                    orb_keypoint* __restrict__ kps, uint8_t* __restrict__ desc, int out_cap) {
  __shared__ __align__(128) uint8_t s_raw[DT_WARPS][DT_RAW_BYTES];
  __shared__ __align__(128) uint8_t s_blr[DT_WARPS][DT_BLR_BYTES];
  __shared__ __align__(8) unsigned long long s_bar[DT_WARPS];
  // rBRIEF pattern, lane-transposed ([word j][lane]): lane-dependent indexing of __constant__
  // memory would serialise into 32 replays per load
  __shared__ int s_pat[1024];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 0; w < DT_WARPS; w++)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(&s_bar[w])));
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  for (int i = threadIdx.x; i < 1024; i += blockDim.x) s_pat[i] = pattern_t[i];
  __syncthreads();
  const int gw = blockIdx.x * DT_WARPS + warp;  // index in the sel slab
  const int f = blockIdx.y;
  const int level = warp_level[gw];
  if (level < 0) return;
  const LevelDev L = lv[level];
  const int i = gw - L.sel_off;
  if (i >= sel_count[f * nlevels + level]) return;
  const int* rec = sel + (size_t)f * sel_frame_stride + 3 * (size_t)gw;
  const int x = rec[0] + 16, y = rec[1] + 16, score = rec[2];  // add minBorder back (:884-885)
  const int pos = slot[(size_t)f * sel_frame_stride / 3 + gw];
  if (pos < 0) return;
  const int ax = (x - 15) & ~15, bx = (x - 18) & ~15;
  if (lane == 0) {
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&s_bar[warp]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(DT_RAW_BYTES + DT_BLR_BYTES) : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"((unsigned)__cvta_generic_to_shared(s_raw[warp])), "l"(raw_maps + level), "r"(bar), "r"(ax), "r"(y - 15), "r"(frame0 + f)
        : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"((unsigned)__cvta_generic_to_shared(s_blr[warp])), "l"(blr_maps + level), "r"(bar), "r"(bx), "r"(y - 18), "r"(frame0 + f)
        : "memory");
  }
  {
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&s_bar[warp]);
    unsigned done = 0;
    while (!done) {
      asm volatile(
          "{\n.reg .pred p;\n"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n"
          "selp.u32 %0, 1, 0, p;\n}"
          : "=r"(done)
          : "r"(bar)
          : "memory");
    }
  }
  // ---- IC_Angle on the raw patch: lane <-> u = lane-15
  int m10 = 0, m01 = 0;
  if (lane < 31) {
    const int u = lane - 15, au = abs(u);
    const uint8_t* c = s_raw[warp] + 15 * DT_RAW_P + (x - ax) + u;
    int colsum = 0;
#pragma unroll
    for (int v = -15; v <= 15; v++) {
      const int val = (au <= c_umax[v < 0 ? -v : v]) ? (int)c[v * DT_RAW_P] : 0;
      colsum += val;
      m01 += v * val;
    }
    m10 = u * colsum;
  }
  m10 = __reduce_add_sync(0xffffffffu, m10);
  m01 = __reduce_add_sync(0xffffffffu, m01);
  const float angle = fast_atan2_deg((float)m01, (float)m10);
  // ---- steered BRIEF: lane <-> descriptor byte
  const float factorPI = 0.017453292519943295f;  // (float)(CV_PI/180.f)
  const float ang = __fmul_rn(angle, factorPI);
  // glibc's cosf / sinf bit for bit (csrc/glibc_sincosf.h): the reference's `(float)cos(angle)` resolves to
  // std::cos(float) = cosf (ORBextractor.cc:111-112); (float)cos((double)x) differs for 0.13 % of the floats
  const float a = glibc_sincosf::cosf_exact<true>(ang), b = glibc_sincosf::sinf_exact<true>(ang);
  const uint8_t* bc = s_blr[warp] + 18 * DT_BLR_P + (x - bx);
  int val = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const float x0 = (float)s_pat[(4 * k) * 32 + lane], y0 = (float)s_pat[(4 * k + 1) * 32 + lane];
    const float x1 = (float)s_pat[(4 * k + 2) * 32 + lane], y1 = (float)s_pat[(4 * k + 3) * 32 + lane];
    const int ry0 = __float2int_rn(__fadd_rn(__fmul_rn(x0, b), __fmul_rn(y0, a)));
    const int rx0 = __float2int_rn(__fsub_rn(__fmul_rn(x0, a), __fmul_rn(y0, b)));
    const int ry1 = __float2int_rn(__fadd_rn(__fmul_rn(x1, b), __fmul_rn(y1, a)));
    const int rx1 = __float2int_rn(__fsub_rn(__fmul_rn(x1, a), __fmul_rn(y1, b)));
    const int t0 = bc[ry0 * DT_BLR_P + rx0], t1 = bc[ry1 * DT_BLR_P + rx1];
    val |= (t0 < t1) << k;
  }
  desc[((size_t)f * out_cap + pos) * 32 + lane] = (uint8_t)val;
  if (lane == 0) {
    orb_keypoint kp;
    float fx = (float)x, fy = (float)y;
    if (level != 0) { fx = __fmul_rn(fx, L.scale); fy = __fmul_rn(fy, L.scale); }
    kp.x = fx; kp.y = fy;
    kp.size = (float)L.patch_size;
    kp.angle = angle;
    kp.response = (float)score;
    kp.octave = level;
    kp.class_id = -1;
    kps[(size_t)f * out_cap + pos] = kp;
  }
}

// cosf / sinf of csrc/glibc_sincosf.h on the device (debug hook of the parity tests)
__global__ void sincos_debug_kernel(const float* __restrict__ x, float* __restrict__ c, float* __restrict__ s, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    c[i] = glibc_sincosf::cosf_exact<true>(x[i]);
    s[i] = glibc_sincosf::sinf_exact<true>(x[i]);
  }
}

int debug_sincos_device(int device, const float* x, size_t n, float* c, float* s) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_last_error("no CUDA device: orb_slam3_b200 has no CPU path");
    return ORB_E_NODEVICE;
  }
  CUDA_TRY(cudaSetDevice(device));
  float *dx = nullptr, *dc = nullptr, *ds = nullptr;
  CUDA_TRY(cudaMalloc(&dx, n * 4));
  CUDA_TRY(cudaMalloc(&dc, n * 4));
  CUDA_TRY(cudaMalloc(&ds, n * 4));
  cudaError_t e = cudaMemcpy(dx, x, n * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    sincos_debug_kernel<<<148 * 8, 256>>>(dx, dc, ds, n);
    e = cudaMemcpy(c, dc, n * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(s, ds, n * 4, cudaMemcpyDeviceToHost);
  }
  cudaFree(dx); cudaFree(dc); cudaFree(ds);
  if (e != cudaSuccess) { set_last_error(cudaGetErrorString(e)); return ORB_E_CUDA; }
  return 0;
}

void debug_sincos_host(const float* x, size_t n, float* c, float* s, int fused) {
  for (size_t i = 0; i < n; i++) {
    c[i] = fused ? glibc_sincosf::cosf_exact<true>(x[i]) : glibc_sincosf::cosf_exact<false>(x[i]);
    s[i] = fused ? glibc_sincosf::sinf_exact<true>(x[i]) : glibc_sincosf::sinf_exact<false>(x[i]);
  }
}

// ------------------------------------------------------------------- engine
Engine::Engine(int nf, float sf, int nl, int ini, int mn, int dev)
    : nfeatures(nf), nlevels(nl), ini_th(ini), min_th(mn), device(dev), scale_factor(sf) {
  // ORBextractor.cc:409-469
  scale.resize(nl); sigma2.resize(nl); inv_scale.resize(nl); inv_sigma2.resize(nl); quota.resize(nl);
  scale[0] = 1.0f; sigma2[0] = 1.0f;
  for (int i = 1; i < nl; i++) {
    scale[i] = (float)(scale[i - 1] * scale_factor);
    sigma2[i] = scale[i] * scale[i];
  }
  for (int i = 0; i < nl; i++) {
    inv_scale[i] = 1.0f / scale[i];
    inv_sigma2[i] = 1.0f / sigma2[i];
  }
  float factor = (float)(1.0f / scale_factor);
  float nDesired = nfeatures * (1 - factor) / (1 - (float)pow((double)factor, (double)nlevels));
  int sum = 0;
  for (int l = 0; l < nl - 1; l++) {
    quota[l] = h_cv_round(nDesired);
    sum += quota[l];
    nDesired *= factor;
  }
  quota[nl - 1] = std::max(nfeatures - sum, 0);
  int um[17];
  memset(um, 0, sizeof(um));
  const int HP = 15;
  int vmax = (int)floorf(HP * sqrtf(2.f) / 2 + 1);
  int vmin = (int)ceilf(HP * sqrtf(2.f) / 2);
  const double hp2 = HP * HP;
  for (int v = 0; v <= vmax; ++v) um[v] = (int)lrint(sqrt(hp2 - v * v));
  for (int v = HP, v0 = 0; v >= vmin; --v) {
    while (um[v0] == um[v0 + 1]) ++v0;
    um[v] = v0;
    ++v0;
  }
  for (int i = 0; i < 16; i++) umax[i] = um[i];
}

Engine::~Engine() { release(); }

void Engine::release() {
  if (!initialized) return;
  cudaSetDevice(device);
  for (void* p : dev_allocs) cudaFree(p);
  dev_allocs.clear();
  for (void* p : host_allocs) cudaFreeHost(p);
  host_allocs.clear();
  for (int i = 0; i < ORB_NUM_STAGES + 1; i++)
    for (auto& e : ev_pool[i]) cudaEventDestroy(e);
  for (auto& e : chunk_events) cudaEventDestroy(e);
  chunk_events.clear();
  if (stream) cudaStreamDestroy(stream);
  if (stream_in) cudaStreamDestroy(stream_in);
  if (stream_out) cudaStreamDestroy(stream_out);
  for (int l = 0; l < MAX_LANES; l++) {
    if (stream_side[l]) cudaStreamDestroy(stream_side[l]);
    if (stream_lane[l]) cudaStreamDestroy(stream_lane[l]);
    if (ev_pyr_done[l]) cudaEventDestroy(ev_pyr_done[l]);
    if (ev_blur_done[l]) cudaEventDestroy(ev_blur_done[l]);
    if (ev_lane_done[l]) cudaEventDestroy(ev_lane_done[l]);
    stream_side[l] = stream_lane[l] = nullptr;
    ev_pyr_done[l] = ev_blur_done[l] = ev_lane_done[l] = nullptr;
  }
  if (ev_lane_go) cudaEventDestroy(ev_lane_go);
  ev_lane_go = nullptr;
  stream = stream_in = stream_out = nullptr;
  initialized = false;
  cap_rows = cap_cols = cap_batch = 0;
}

template <class T>
int Engine::dalloc(T** p, size_t count) {
  void* q = nullptr;
  CUDA_TRY(cudaMalloc(&q, std::max<size_t>(count * sizeof(T), 16)));
  dev_allocs.push_back(q);
  *p = (T*)q;
  return 0;
}

int Engine::ensure(int rows, int cols, int batch) {
  if (rows == cap_rows && cols == cap_cols && batch <= cap_batch) return 0;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_last_error("no CUDA device: orb_slam3_b200 has no CPU path");
    return ORB_E_NODEVICE;
  }
  release();
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&stream_in, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&stream_out, cudaStreamNonBlocking));
  for (int l = 0; l < MAX_LANES; l++) {
    CUDA_TRY(cudaStreamCreateWithFlags(&stream_side[l], cudaStreamNonBlocking));
    if (l) CUDA_TRY(cudaStreamCreateWithFlags(&stream_lane[l], cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&ev_pyr_done[l], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&ev_blur_done[l], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&ev_lane_done[l], cudaEventDisableTiming));
  }
  CUDA_TRY(cudaEventCreateWithFlags(&ev_lane_go, cudaEventDisableTiming));
  {
    // measured on the B200 (profiles/r2_summary.md): 3 lanes give +3 % on 128-frame device-resident batches
    const char* env = getenv("ORB_B200_LANES");
    lanes = env ? std::min(std::max(atoi(env), 1), (int)MAX_LANES) : 3;
  }
  initialized = true;
  CUDA_TRY(cudaMemcpyToSymbol(c_pattern, h_pattern, sizeof(h_pattern)));
  CUDA_TRY(cudaMemcpyToSymbol(c_umax, umax, sizeof(umax)));

  // ---- geometry (ComputePyramid :1170-1195, ComputeKeyPointsOctTree :781-822)
  levels.assign(nlevels, LevelDev());
  std::vector<CellDesc> cells;
  std::vector<BlurTile> tiles;
  std::vector<int> h_xofs, h_yofs;
  std::vector<short2> h_alpha, h_beta;
  size_t img_off = 0, cand_off = 0, scratch_off = 0;
  int sel_off = 0;
  rs.assign(nlevels, ResizeTab());
  for (int l = 0; l < nlevels; l++) {
    LevelDev& L = levels[l];
    L.w = h_cv_round((float)cols * inv_scale[l]);
    L.h = h_cv_round((float)rows * inv_scale[l]);
    if (L.w < 40 || L.h < 40) {
      set_last_error("image too small for the pyramid (level < 40 px)");
      return ORB_E_ARG;
    }
    L.pitch = (int)align_up(L.w, 64);
    L.img_off = img_off;
    img_off += align_up((size_t)L.pitch * L.h, 256);
    L.scale = scale[l];
    L.patch_size = (int)(31 * scale[l]);
    const int minB = 16, maxBX = L.w - 16, maxBY = L.h - 16;
    const float width = (float)(maxBX - minB), height = (float)(maxBY - minB);
    const int nCols = (int)(width / 35.f), nRows = (int)(height / 35.f);
    const int wCell = (int)ceilf(width / nCols), hCell = (int)ceilf(height / nRows);
    if (wCell > FAST_BAND_MAX || hCell > FAST_BAND_MAX || wCell + 6 + 15 > FAST_TILE_PITCH || hCell + 6 > FAST_TILE_MAX) {
      set_last_error("unsupported FAST cell size");
      return ORB_E_ARG;
    }
    for (int i = 0; i < nRows; i++) {
      const float iniY = (float)(minB + i * hCell);
      float maxY = iniY + hCell + 6;
      if (iniY >= maxBY - 3) continue;
      if (maxY > maxBY) maxY = (float)maxBY;
      for (int j = 0; j < nCols; j++) {
        const float iniX = (float)(minB + j * wCell);
        float maxX = iniX + wCell + 6;
        if (iniX >= maxBX - 6) continue;
        if (maxX > maxBX) maxX = (float)maxBX;
        CellDesc c;
        c.level = l; c.x0 = (int)iniX; c.y0 = (int)iniY; c.x1 = (int)maxX; c.y1 = (int)maxY;
        c.shift_x = j * wCell; c.shift_y = i * hCell;
        cells.push_back(c);
      }
    }
    OctreeLevelParams& o = L.oct;
    o.bandW = maxBX - minB; o.bandH = maxBY - minB;
    o.N = quota[l];
    o.nIni = (int)roundf((float)o.bandW / (float)o.bandH);
    if (o.nIni < 1) {
      set_last_error("aspect ratio < 0.5 is undefined in the reference (nIni == 0)");
      return ORB_E_ARG;
    }
    o.hX = (float)o.bandW / o.nIni;
    if (o.bandW >= 4096) {
      set_last_error("image wider than 4127 px: the octree sort key packs UL.x into 12 bits");
      return ORB_E_ARG;
    }
    o.wCell = wCell; o.hCell = hCell; o.nCols = nCols;
    o.node_cap = o.N + 4 * o.nIni + 16;
    L.cand_cap = (o.bandW / 2 + nCols + 2) * (o.bandH / 2 + nRows + 2);
    L.cand_off = cand_off;
    cand_off += align_up(L.cand_cap, 4);
    L.sel_off = sel_off;
    sel_off += o.node_cap;
    L.scratch_off = scratch_off;
    scratch_off += align_up(octree_scratch_layout(nullptr, L.cand_cap, o.node_cap, nullptr), 256);
    for (int ty = 0; ty < L.h; ty += BLUR_TH)
      for (int tx = 0; tx < L.w; tx += BLUR_TW) tiles.push_back(BlurTile{l, tx, ty});
    if (l > 0) {
      // cv::resize coefficient tables (SURVEY.md A.1)
      const LevelDev& S = levels[l - 1];
      ResizeTab& R = rs[l];
      R.x_off = (int)h_xofs.size(); R.y_off = (int)h_yofs.size();
      const double scale_x = 1. / ((double)L.w / S.w), scale_y = 1. / ((double)L.h / S.h);
      auto sat = [](int v) { return (short)std::min(32767, std::max(-32768, v)); };
      for (int dx = 0; dx < L.w; dx++) {
        float fx = (float)((dx + 0.5) * scale_x - 0.5);
        int sx = (int)floorf(fx);
        fx -= sx;
        if (sx < 0) { fx = 0; sx = 0; }
        if (sx >= S.w - 1) { fx = 0; sx = S.w - 1; }
        h_xofs.push_back(sx);
        h_alpha.push_back(make_short2(sat(h_cv_round((1.f - fx) * 2048.f)), sat(h_cv_round(fx * 2048.f))));
      }
      for (int dy = 0; dy < L.h; dy++) {
        float fy = (float)((dy + 0.5) * scale_y - 0.5);
        int sy = (int)floorf(fy);
        fy -= sy;
        h_yofs.push_back(sy);
        h_beta.push_back(make_short2(sat(h_cv_round((1.f - fy) * 2048.f)), sat(h_cv_round(fy * 2048.f))));
      }
    }
  }
  {
    int max_nc = 0;
    for (int l = 0; l < nlevels; l++) max_nc = std::max(max_nc, levels[l].oct.node_cap);
    const size_t need = (size_t)19 * max_nc * sizeof(int), need_full = ((size_t)39 * max_nc + 2) * sizeof(int);
    oct_smem_node_cap_full = 0;
    if (need_full <= 100 * 1024 && !getenv("ORB_B200_OCTREE_SMEM_BASE")) {
      oct_smem_node_cap = oct_smem_node_cap_full = max_nc;
      oct_smem_bytes = need_full;
      CUDA_TRY(raise_dynamic_smem((const void*)octree_kernel, need_full, device));
    } else if (need <= 96 * 1024) {
      oct_smem_node_cap = max_nc;
      oct_smem_bytes = need;
      CUDA_TRY(raise_dynamic_smem((const void*)octree_kernel, need, device));
    } else {
      oct_smem_node_cap = 0;  // huge quotas: keep the node arrays in global memory
      oct_smem_bytes = 0;
    }
  }
  {
    // resize_rows_kernel: RS_ROWS output rows must span <= RS_SRC source rows, and the staged rows must fit
    resize_rows_ok = !(getenv("ORB_B200_RESIZE") && !strcmp(getenv("ORB_B200_RESIZE"), "level"));
    size_t smem = 0;
    for (int l = 1; l < nlevels && resize_rows_ok; l++) {
      const LevelDev& S = levels[l - 1];
      const LevelDev& D = levels[l];
      smem = std::max(smem, (size_t)RS_SRC * S.pitch);
      for (int y0 = 0; y0 < D.h; y0 += RS_ROWS) {
        const int y1 = std::min(y0 + RS_ROWS, D.h) - 1;
        const int lo = std::min(std::max(h_yofs[rs[l].y_off + y0], 0), S.h - 1);
        const int hi = std::min(std::max(h_yofs[rs[l].y_off + y1] + 1, 0), S.h - 1);
        if (hi - lo + 1 > RS_SRC) resize_rows_ok = false;
      }
    }
    if (smem > 200 * 1024) resize_rows_ok = false;
    if (resize_rows_ok) CUDA_TRY(raise_dynamic_smem((const void*)resize_rows_kernel, smem, device));
    // resize_words_kernel: the source bytes of four consecutive output pixels must lie within eight bytes, and the
    // horizontal coefficients must be non-negative (they are: 2048 (1 - fx), 2048 fx); ORB_B200_RESIZE=rows pins the
    // byte-gather kernel
    resize_words_ok = resize_rows_ok && !(getenv("ORB_B200_RESIZE") && !strcmp(getenv("ORB_B200_RESIZE"), "rows"));
    for (int l = 1; l < nlevels && resize_words_ok; l++) {
      const LevelDev& S = levels[l - 1];
      const LevelDev& D = levels[l];
      for (int x4 = 0; x4 < D.w; x4 += 4) {
        const int xa = h_xofs[rs[l].x_off + x4], xb = h_xofs[rs[l].x_off + std::min(x4 + 3, D.w - 1)];
        if (std::min(xb + 1, S.w - 1) - xa > 7 || xb < xa) resize_words_ok = false;
      }
      for (int x = 0; x < D.w; x++)
        if (h_alpha[rs[l].x_off + x].x < 0 || h_alpha[rs[l].x_off + x].y < 0) resize_words_ok = false;
    }
    if (resize_words_ok) CUDA_TRY(raise_dynamic_smem((const void*)resize_words_kernel, smem + 16, device));
  }
  pyr_frame_bytes = align_up(img_off, 256);
  cand_frame_elems = cand_off;
  scratch_frame_bytes = scratch_off;
  sel_frame_elems = align_up(sel_off, 32);
  out_cap = sel_off;  // >= any possible keypoint count
  num_cells = (int)cells.size();
  num_tiles = (int)tiles.size();
  std::vector<int> warp_level(sel_frame_elems, -1);
  for (int l = 0; l < nlevels; l++)
    for (int i = 0; i < levels[l].oct.node_cap; i++) warp_level[levels[l].sel_off + i] = l;

  {
    // warp-per-cell FAST geometry: box = (3 + widest cell + 6, rounded to 16) x (tallest cell + 6)
    int max_tw = 0, max_th = 0;
    for (const CellDesc& c : cells) { max_tw = std::max(max_tw, c.x1 - c.x0); max_th = std::max(max_th, c.y1 - c.y0); }
    // the box must start at a 16-byte aligned column: a TMA tile load whose innermost coordinate is not a
    // multiple of 16 bytes faults as an illegal instruction (compute-sanitizer, round 2)
    fw_align_mask = 15;
    fw_tile_pitch = (int)align_up(fw_align_mask + max_tw, 16);
    fw_tile_rows = (int)align_up(max_th, 8);  // pitch % 16 == 0 and rows % 8 == 0: every slot is 128-byte aligned for TMA
    fw_smap_pitch = max_tw - 6 + 2;
    fw_smap_bytes = (int)align_up((size_t)fw_smap_pitch * (max_th - 6 + 2) + 4, 16);
    fw_queue_cap = (max_tw - 6) * (max_th - 6);
    const int tile_bytes = (int)align_up((size_t)fw_tile_pitch * fw_tile_rows, 128);
    int max_groups = 0;  // 4-pixel groups of the largest band, with the box starting at x0 & ~15
    for (const CellDesc& c : cells) {
      const int ox = c.x0 & 15, bw = c.x1 - c.x0 - 6, bh = c.y1 - c.y0 - 6;
      if (bw > 0 && bh > 0) max_groups = std::max(max_groups, bh * (((ox + 3 + bw + 3) >> 2) - ((ox + 3) >> 2)));
    }
    fw_gq_off = (int)align_up(2 * (size_t)fw_queue_cap, 16);
    fw_per_warp = (int)align_up((size_t)2 * tile_bytes + fw_smap_bytes + fw_gq_off + 4 * (size_t)max_groups, 128);
    const size_t smem = (size_t)fw_per_warp * FASTW_WARPS;
    const char* env = getenv("ORB_B200_FAST");  // "cta": the CTA-per-cell kernel
    fw_enabled = !(env && !strcmp(env, "cta")) && fw_tile_pitch <= 256 && fw_tile_rows <= 256 && smem <= 200 * 1024 &&
                 max_tw - 6 <= 127 && max_th - 6 <= 127 && (size_t)fw_tile_pitch * fw_tile_rows == (size_t)tile_bytes &&
                 (long long)cells.size() * batch < (1ll << 30);
    if (fw_enabled) {
      const void* kfn = fw_tile_pitch == 64 ? (const void*)fast_warp_kernel<64> : (const void*)fast_warp_kernel<0>;
      CUDA_TRY(raise_dynamic_smem(kfn, smem, device));
      int per_sm = 0, sms = 0;
      if (fw_tile_pitch == 64)
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fast_warp_kernel<64>, FASTW_WARPS * 32, smem));
      else
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fast_warp_kernel<0>, FASTW_WARPS * 32, smem));
      CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
      fw_grid = sms * std::max(per_sm, 1);
    }
  }
  const size_t B = batch;
  if (dalloc(&d_pyr, pyr_frame_bytes * B)) return ORB_E_CUDA;
  if (dalloc(&d_blur, pyr_frame_bytes * B + 256)) return ORB_E_CUDA;
  if (encode_tensor_maps((int)B)) return ORB_E_CUDA;
  if (dalloc(&d_cand, cand_frame_elems * B)) return ORB_E_CUDA;
  if (dalloc(&d_scratch, scratch_frame_bytes * B)) return ORB_E_CUDA;
  if (dalloc(&d_sel, 3 * sel_frame_elems * B)) return ORB_E_CUDA;
  if (dalloc(&d_slot, sel_frame_elems * B)) return ORB_E_CUDA;
  if (dalloc(&d_cand_count, (size_t)nlevels * B)) return ORB_E_CUDA;
  if (dalloc(&d_sel_count, (size_t)nlevels * B)) return ORB_E_CUDA;
  for (int k = 0; k < 2; k++) {
    if (dalloc(&d_n_buf[k], B)) return ORB_E_CUDA;
    if (dalloc(&d_mono_buf[k], B)) return ORB_E_CUDA;
    if (dalloc(&d_kps_buf[k], (size_t)out_cap * B)) return ORB_E_CUDA;
    if (dalloc(&d_desc_buf[k], (size_t)out_cap * 32 * B)) return ORB_E_CUDA;
  }
  out_idx = 1;
  flip_outputs();
  if (dalloc(&d_lap, 2 * B)) return ORB_E_CUDA;
  if (dalloc(&d_levels, (size_t)nlevels)) return ORB_E_CUDA;
  if (dalloc(&d_cells, cells.size())) return ORB_E_CUDA;
  if (dalloc(&d_tiles, tiles.size())) return ORB_E_CUDA;
  if (dalloc(&d_warp_level, warp_level.size())) return ORB_E_CUDA;
  if (dalloc(&d_pattern_t, (size_t)1024)) return ORB_E_CUDA;
  {
    std::vector<int> pt(1024);
    for (int lane = 0; lane < 32; lane++)
      for (int j = 0; j < 32; j++) pt[j * 32 + lane] = h_pattern[32 * lane + j];
    CUDA_TRY(cudaMemcpy(d_pattern_t, pt.data(), sizeof(int) * 1024, cudaMemcpyHostToDevice));
  }
  if (dalloc(&d_xofs, h_xofs.size())) return ORB_E_CUDA;
  if (dalloc(&d_yofs, h_yofs.size())) return ORB_E_CUDA;
  if (dalloc(&d_alpha, h_alpha.size())) return ORB_E_CUDA;
  if (dalloc(&d_beta, h_beta.size())) return ORB_E_CUDA;
  if (dalloc(&d_stage, (size_t)rows * cols * B)) return ORB_E_CUDA;
  CUDA_TRY(cudaMemcpy(d_levels, levels.data(), sizeof(LevelDev) * nlevels, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_cells, cells.data(), sizeof(CellDesc) * cells.size(), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_tiles, tiles.data(), sizeof(BlurTile) * tiles.size(), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_warp_level, warp_level.data(), sizeof(int) * warp_level.size(), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_xofs, h_xofs.data(), sizeof(int) * h_xofs.size(), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_yofs, h_yofs.data(), sizeof(int) * h_yofs.size(), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_alpha, h_alpha.data(), sizeof(short2) * h_alpha.size(), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_beta, h_beta.data(), sizeof(short2) * h_beta.size(), cudaMemcpyHostToDevice));
  void* hp = nullptr;
  CUDA_TRY(cudaHostAlloc(&hp, sizeof(int) * 2 * B, cudaHostAllocDefault));
  host_allocs.push_back(hp);
  h_counts = (int*)hp;
  CUDA_TRY(cudaHostAlloc(&hp, pyr_frame_bytes * B, cudaHostAllocDefault));
  host_allocs.push_back(hp);
  h_pyr = (uint8_t*)hp;
  cap_rows = rows; cap_cols = cols; cap_batch = batch;
  return 0;
}

void Engine::stage_begin(int st, cudaStream_t s) {
  if (!profiling) return;
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  ev_pool[st].push_back(a);
  ev_pool[st].push_back(b);
  cudaEventRecord(a, s);
}
void Engine::stage_end(int st, cudaStream_t s, int launches) {
  stage_launches[st] += launches;
  total_launches += launches;
  if (!profiling) return;
  cudaEventRecord(ev_pool[st].back(), s);
}

int Engine::collect_times(double* ms, long long* launches, bool reset) {
  for (int st = 0; st < ORB_NUM_STAGES; st++) {
    for (size_t i = 0; i + 1 < ev_pool[st].size(); i += 2) {
      float t = 0;
      cudaEventSynchronize(ev_pool[st][i + 1]);
      if (cudaEventElapsedTime(&t, ev_pool[st][i], ev_pool[st][i + 1]) == cudaSuccess) stage_ms[st] += t;
      cudaEventDestroy(ev_pool[st][i]);
      cudaEventDestroy(ev_pool[st][i + 1]);
    }
    ev_pool[st].clear();
    if (ms) ms[st] = stage_ms[st];
    if (launches) launches[st] = stage_launches[st];
    if (reset) { stage_ms[st] = 0; stage_launches[st] = 0; }
  }
  return 0;
}

// Everything between "level 0 is in the pyramid slab" and "results are in
// d_kps/d_desc/d_n/d_mono" for frames [f0, f0+batch) of the slabs, on stream s.
int Engine::run_device(int f0, int batch, const int* lap_host, cudaStream_t s, int lane) {
  const int B = batch;
  pyramid_fetched = false;
  uint8_t* pyr = d_pyr + (size_t)f0 * pyr_frame_bytes;
  uint8_t* blr = d_blur + (size_t)f0 * pyr_frame_bytes;
  Cand* cand = d_cand + (size_t)f0 * cand_frame_elems;
  uint8_t* scratch = d_scratch + (size_t)f0 * scratch_frame_bytes;
  int* sel = d_sel + 3 * (size_t)f0 * sel_frame_elems;
  int* slot = d_slot + (size_t)f0 * sel_frame_elems;
  int* cand_count = d_cand_count + (size_t)f0 * nlevels;
  int* sel_count = d_sel_count + (size_t)f0 * nlevels;
  if (lap_host) {
    CUDA_TRY(cudaMemcpyAsync(d_lap + 2 * f0, lap_host + 2 * f0, sizeof(int) * 2 * B, cudaMemcpyHostToDevice, s));
  }
  // 1. pyramid
  stage_begin(1, s);
  for (int l = 1; l < nlevels; l++) {
    const LevelDev& S = levels[l - 1];
    const LevelDev& D = levels[l];
    if (resize_rows_ok && resize_words_ok) {
      resize_words_kernel<<<dim3((D.h + RS_ROWS - 1) / RS_ROWS, B), RS_THREADS, (size_t)RS_SRC * S.pitch + 16, s>>>(
          pyr, pyr_frame_bytes, S.img_off, S.w, S.h, S.pitch, D.img_off, D.w, D.h, D.pitch, d_xofs + rs[l].x_off,
          d_alpha + rs[l].x_off, d_yofs + rs[l].y_off, d_beta + rs[l].y_off);
    } else if (resize_rows_ok) {
      resize_rows_kernel<<<dim3((D.h + RS_ROWS - 1) / RS_ROWS, B), RS_THREADS, (size_t)RS_SRC * S.pitch, s>>>(
          pyr, pyr_frame_bytes, S.img_off, S.w, S.h, S.pitch, D.img_off, D.w, D.h, D.pitch, d_xofs + rs[l].x_off,
          d_alpha + rs[l].x_off, d_yofs + rs[l].y_off, d_beta + rs[l].y_off);
    } else {
      dim3 grid((D.w + 4 * 256 - 1) / (4 * 256), D.h, B);
      resize_level_kernel<<<grid, 256, 0, s>>>(pyr, pyr_frame_bytes, S.img_off, S.w, S.h, S.pitch, D.img_off,
                                              D.w, D.h, D.pitch, d_xofs + rs[l].x_off, d_alpha + rs[l].x_off,
                                              d_yofs + rs[l].y_off, d_beta + rs[l].y_off);
    }
  }
  stage_end(1, s, nlevels - 1);
  // 4. blur: needs only the pyramid, so it runs on a side stream next to FAST + octree (the
  //    octree is a latency-bound 8-CTA-per-frame kernel that leaves most SMs idle)
  const bool side_stream_used = !profiling;
  if (side_stream_used) {
    CUDA_TRY(cudaEventRecord(ev_pyr_done[lane], s));
    CUDA_TRY(cudaStreamWaitEvent(stream_side[lane], ev_pyr_done[lane], 0));
    blur_kernel<<<dim3(num_tiles, B), 256, 0, stream_side[lane]>>>(pyr, blr, pyr_frame_bytes, d_tiles, d_levels);
    CUDA_TRY(cudaEventRecord(ev_blur_done[lane], stream_side[lane]));
    stage_launches[4] += 1; total_launches += 1;
  } else {
    stage_begin(4, s);
    blur_kernel<<<dim3(num_tiles, B), 256, 0, s>>>(pyr, blr, pyr_frame_bytes, d_tiles, d_levels);
    stage_end(4, s, 1);
  }
  // 2. FAST cells
  stage_begin(2, s);
  CUDA_TRY(cudaMemsetAsync(cand_count, 0, sizeof(int) * nlevels * B, s));
  if (fw_enabled) {
    FastGeom G;
    G.tile_pitch = fw_tile_pitch; G.tile_rows = fw_tile_rows; G.tile_bytes = fw_tile_pitch * fw_tile_rows;
    G.smap_pitch = fw_smap_pitch; G.smap_bytes = fw_smap_bytes; G.queue_cap = fw_queue_cap; G.gq_off = fw_gq_off; G.per_warp_bytes = fw_per_warp;
    const long long items = (long long)num_cells * B;
    const int grid = (int)std::min<long long>(fw_grid, (items + FASTW_WARPS - 1) / FASTW_WARPS);
    if (fw_tile_pitch == 64)
      fast_warp_kernel<64><<<grid, FASTW_WARPS * 32, (size_t)fw_per_warp * FASTW_WARPS, s>>>(
          (const CUtensorMap*)d_tmaps_raw + 16, f0, B, d_cells, num_cells, d_levels, ini_th, min_th, cand, cand_frame_elems,
          cand_count, nlevels, G);
    else
      fast_warp_kernel<0><<<grid, FASTW_WARPS * 32, (size_t)fw_per_warp * FASTW_WARPS, s>>>(
          (const CUtensorMap*)d_tmaps_raw + 16, f0, B, d_cells, num_cells, d_levels, ini_th, min_th, cand, cand_frame_elems,
          cand_count, nlevels, G);
  } else {
    fast_cells_kernel<<<dim3(num_cells, B), FAST_THREADS, 0, s>>>((const CUtensorMap*)d_tmaps_raw, f0, d_cells, d_levels, ini_th, min_th, cand,
                                                                  cand_frame_elems, cand_count, nlevels);
  }
  stage_end(2, s, 1);
  // 3. octree
  stage_begin(3, s);
  octree_kernel<<<dim3(B, nlevels), OCT_THREADS, oct_smem_bytes, s>>>(cand, cand_frame_elems, cand_count, d_levels,
                                                                      scratch, scratch_frame_bytes, sel,
                                                                      3 * sel_frame_elems, sel_count, nlevels,
                                                                      oct_smem_node_cap, oct_smem_node_cap_full);
  stage_end(3, s, 1);
  // 5. output layout
  stage_begin(5, s);
  layout_kernel<<<B, 256, 0, s>>>(sel, 3 * sel_frame_elems, sel_count, d_levels, nlevels,
                                  lap_host ? d_lap + 2 * f0 : nullptr, slot, d_n + f0, d_mono + f0, out_cap);
  stage_end(5, s, 1);
  // 6. orientation + descriptors (one fused kernel measured faster than an orient/brief split)
  stage_begin(6, s);
  if (side_stream_used) CUDA_TRY(cudaStreamWaitEvent(s, ev_blur_done[lane], 0));
  describe_tma_kernel<<<dim3((unsigned)(sel_frame_elems / DT_WARPS), B), DT_WARPS * 32, 0, s>>>(
      (const CUtensorMap*)d_tmaps_raw + 32, (const CUtensorMap*)d_tmaps_raw + 48, f0, sel, 3 * sel_frame_elems, sel_count,
      slot, d_levels, nlevels, d_warp_level, d_pattern_t, d_kps + (size_t)f0 * out_cap,
      d_desc + (size_t)f0 * out_cap * 32, out_cap);
  stage_end(6, s, 1);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// Host-buffer path.  The batch is cut into chunks that flow through three
// streams (H2D | kernels | D2H) so the PCIe copies overlap the compute of the
// neighbouring chunks.
int Engine::extract_batch_host(int batch, const uint8_t* const* imgs, int rows, int cols, size_t step,
                               const int* lap, orb_keypoint* kps, uint8_t* desc, int cap, int* n, int* mono) {
  if (batch <= 0 || !imgs || !kps || !desc || !n || !mono) { set_last_error("bad argument"); return ORB_E_ARG; }
  if (rows <= 0 || cols <= 0) return ORB_E_EMPTY;
  for (int b = 0; b < batch; b++)
    if (!imgs[b]) return ORB_E_EMPTY;
  int rc = ensure(rows, cols, std::max(batch, cap_batch_hint));
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(device));
  flip_outputs();
  last_batch = batch;
  last_stream = stream;
  cudaStream_t s = stream;
  const LevelDev& L0 = levels[0];
  const int chunk = batch <= 8 ? batch : std::max(8, (batch + 3) / 4);
  const int nchunks = (batch + chunk - 1) / chunk;
  if ((int)chunk_events.size() < 2 * nchunks) {
    const size_t old = chunk_events.size();
    chunk_events.resize(2 * nchunks);
    for (size_t i = old; i < chunk_events.size(); i++)
      CUDA_TRY(cudaEventCreateWithFlags(&chunk_events[i], cudaEventDisableTiming));
  }
  // keypoints are dense from slot 0; copy the quota-sized prefix as each chunk finishes,
  // the rare overshoot (<= 3 per level) after the counts are known
  const int guess = std::min(std::min(cap, out_cap), nfeatures + 4 * nlevels);
  stage_begin(0, s);
  for (int c = 0; c < nchunks; c++) {
    const int f0 = c * chunk, fb = std::min(chunk, batch - f0);
    // frames that lie back to back in host memory with dense rows (a pinned [B][H][W] block) go up as ONE copy
    // per chunk: a "2-D" copy whose rows are whole level-0 images and whose destination pitch is the slab stride
    bool dense = step == (size_t)cols && L0.pitch == cols;
    for (int b = f0 + 1; b < f0 + fb && dense; b++) dense = imgs[b] == imgs[b - 1] + (size_t)rows * step;
    if (dense) {
      CUDA_TRY(cudaMemcpy2DAsync(d_pyr + (size_t)f0 * pyr_frame_bytes, pyr_frame_bytes, imgs[f0], (size_t)rows * cols,
                                 (size_t)rows * cols, fb, cudaMemcpyHostToDevice, nchunks > 1 ? stream_in : s));
    } else {
      for (int b = f0; b < f0 + fb; b++)
        CUDA_TRY(cudaMemcpy2DAsync(d_pyr + (size_t)b * pyr_frame_bytes, L0.pitch, imgs[b], step, cols, rows,
                                   cudaMemcpyHostToDevice, nchunks > 1 ? stream_in : s));
    }
    if (nchunks > 1) CUDA_TRY(cudaEventRecord(chunk_events[2 * c], stream_in));
  }
  stage_end(0, s, 0);
  for (int c = 0; c < nchunks; c++) {
    const int f0 = c * chunk, fb = std::min(chunk, batch - f0);
    if (nchunks > 1) CUDA_TRY(cudaStreamWaitEvent(s, chunk_events[2 * c], 0));
    rc = run_device(f0, fb, lap, s);
    if (rc) return rc;
    cudaStream_t so = nchunks > 1 ? stream_out : s;
    if (nchunks > 1) {
      CUDA_TRY(cudaEventRecord(chunk_events[2 * c + 1], s));
      CUDA_TRY(cudaStreamWaitEvent(so, chunk_events[2 * c + 1], 0));
    }
    CUDA_TRY(cudaMemcpyAsync(h_counts + f0, d_n + f0, sizeof(int) * fb, cudaMemcpyDeviceToHost, so));
    CUDA_TRY(cudaMemcpyAsync(h_counts + cap_batch + f0, d_mono + f0, sizeof(int) * fb, cudaMemcpyDeviceToHost, so));
    for (int b = f0; b < f0 + fb; b++) {
      CUDA_TRY(cudaMemcpyAsync(kps + (size_t)b * cap, d_kps + (size_t)b * out_cap, sizeof(orb_keypoint) * guess,
                               cudaMemcpyDeviceToHost, so));
      CUDA_TRY(cudaMemcpyAsync(desc + (size_t)b * cap * 32, d_desc + (size_t)b * out_cap * 32, (size_t)32 * guess,
                               cudaMemcpyDeviceToHost, so));
    }
  }
  stage_begin(7, s);
  if (nchunks > 1) CUDA_TRY(cudaStreamSynchronize(stream_out));
  CUDA_TRY(cudaStreamSynchronize(s));
  int worst = 0;
  for (int b = 0; b < batch; b++) {
    n[b] = h_counts[b];
    mono[b] = h_counts[cap_batch + b];
    worst = std::max(worst, n[b]);
  }
  if (worst > cap) { set_last_error("keypoint buffer too small"); return ORB_E_CAPACITY; }
  if (worst > guess) {
    for (int b = 0; b < batch; b++) {
      if (n[b] <= guess) continue;
      CUDA_TRY(cudaMemcpyAsync(kps + (size_t)b * cap + guess, d_kps + (size_t)b * out_cap + guess,
                               sizeof(orb_keypoint) * (n[b] - guess), cudaMemcpyDeviceToHost, s));
      CUDA_TRY(cudaMemcpyAsync(desc + ((size_t)b * cap + guess) * 32, d_desc + ((size_t)b * out_cap + guess) * 32,
                               (size_t)32 * (n[b] - guess), cudaMemcpyDeviceToHost, s));
    }
    CUDA_TRY(cudaStreamSynchronize(s));
  }
  stage_end(7, s, 0);
  return batch;
}

int Engine::extract_batch_device(int batch, const uint8_t* d_imgs, size_t frame_stride, int rows, int cols,
                                 size_t step, const int* lap, cudaStream_t user) {
  if (batch <= 0 || !d_imgs) { set_last_error("bad argument"); return ORB_E_ARG; }
  if (rows <= 0 || cols <= 0) return ORB_E_EMPTY;
  int rc = ensure(rows, cols, std::max(batch, cap_batch_hint));
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(device));
  flip_outputs();
  cudaStream_t s = user ? user : stream;
  last_stream = s;
  const LevelDev& L0 = levels[0];
  stage_begin(0, s);
  {
    // rows are 16-byte copyable when pointers/pitches are 16-aligned (the slab pitch is a multiple
    // of 64, so the tail of the last vector stays inside the destination row)
    const int vec16 = ((uintptr_t)d_imgs % 16 == 0) && (step % 16 == 0) && (frame_stride % 16 == 0) &&
                      ((size_t)((cols + 15) / 16) * 16 <= step);
    const int per_row = vec16 ? (cols + 15) / 16 : cols;
    dim3 grid((per_row + 255) / 256, rows, batch);
    if (!vec16) grid.x = std::min<unsigned>(grid.x, 8);
    copy_level0_kernel<<<grid, 256, 0, s>>>(d_imgs, frame_stride, step, d_pyr, pyr_frame_bytes, cols, rows, L0.pitch,
                                            vec16);
  }
  stage_end(0, s, 1);
  last_batch = batch;
  const int nl = (profiling || batch < 32) ? 1 : std::min(lanes, batch);
  if (nl > 1) {
    // sub-batches on their own streams; lane 0 is the caller's stream, the others branch off after the level-0
    // copy and are joined back before the call returns control of `s`
    CUDA_TRY(cudaEventRecord(ev_lane_go, s));
    const int per = (batch + nl - 1) / nl;
    for (int l = 0; l < nl; l++) {
      const int f0 = l * per, fb = std::min(per, batch - f0);
      if (fb <= 0) break;
      cudaStream_t ls = l ? stream_lane[l] : s;
      if (l) CUDA_TRY(cudaStreamWaitEvent(ls, ev_lane_go, 0));
      if (run_device(f0, fb, lap, ls, l)) return ORB_E_CUDA;
      if (l) CUDA_TRY(cudaEventRecord(ev_lane_done[l], ls));
    }
    for (int l = 1; l < nl; l++)
      if (l * per < batch) CUDA_TRY(cudaStreamWaitEvent(s, ev_lane_done[l], 0));
    return batch;
  }
  // one lane: the whole batch in one pass.  Cutting it into L2-sized chunks measured no faster on B200
  // (profiles/r1_summary.md) -- no stage is HBM bound and the latency-bound octree wants as many (frame, level) CTAs
  // in flight as possible
  if (run_device(0, batch, lap, s)) return ORB_E_CUDA;
  return batch;
}

// TMA descriptors of the pyramid levels: uint8 tensor (x = level width, y = level height, z = frame)
// with byte strides (pitch, slab stride); box = the FAST tile.  cuTensorMapEncodeTiled is taken from
// the driver through the runtime so the library does not link libcuda.
int Engine::encode_tensor_maps(int batch) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) { set_last_error("cuTensorMapEncodeTiled not available"); return ORB_E_CUDA; }
  if (!tmaps) tmaps = new LevelTensorMaps();
  memset(tmaps, 0, sizeof(LevelTensorMaps));
  if (nlevels > 16) { set_last_error("more than 16 pyramid levels"); return ORB_E_ARG; }
  for (int l = 0; l < nlevels; l++) {
    const LevelDev& L = levels[l];
    const cuuint64_t dims[3] = {(cuuint64_t)L.w, (cuuint64_t)L.h, (cuuint64_t)batch};
    const cuuint64_t strides[2] = {(cuuint64_t)L.pitch, (cuuint64_t)pyr_frame_bytes};
    const cuuint32_t box[3] = {(cuuint32_t)FAST_TILE_PITCH, (cuuint32_t)FAST_TILE_MAX, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = ((EncodeFn)fn)(&tmaps->m[l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, d_pyr + L.img_off, dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_last_error("cuTensorMapEncodeTiled failed, level " + std::to_string(l) + " rc " + std::to_string((int)r)); return ORB_E_CUDA; }
    {
      const cuuint32_t box3[3] = {(cuuint32_t)DT_RAW_P, (cuuint32_t)DT_RAW_R, 1};
      r = ((EncodeFn)fn)(&tmaps->m[32 + l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, d_pyr + L.img_off, dims, strides, box3, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) { set_last_error("cuTensorMapEncodeTiled (raw patch box) failed, rc " + std::to_string((int)r)); return ORB_E_CUDA; }
      const cuuint32_t box4[3] = {(cuuint32_t)DT_BLR_P, (cuuint32_t)DT_BLR_R, 1};
      r = ((EncodeFn)fn)(&tmaps->m[48 + l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, d_blur + L.img_off, dims, strides, box4, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) { set_last_error("cuTensorMapEncodeTiled (blurred patch box) failed, rc " + std::to_string((int)r)); return ORB_E_CUDA; }
    }
    if (fw_enabled) {
      const cuuint32_t box2[3] = {(cuuint32_t)fw_tile_pitch, (cuuint32_t)fw_tile_rows, 1};
      r = ((EncodeFn)fn)(&tmaps->m[16 + l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, d_pyr + L.img_off, dims, strides, box2, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) { set_last_error("cuTensorMapEncodeTiled (warp box) failed, level " + std::to_string(l) + " rc " + std::to_string((int)r)); return ORB_E_CUDA; }
    }
  }
  // the descriptors live in global memory (cudaMalloc is 256-byte aligned; TMA needs 64)
  {
    void* q = nullptr;  // (re)allocated with the other slabs: release() frees dev_allocs
    CUDA_TRY(cudaMalloc(&q, sizeof(LevelTensorMaps)));
    dev_allocs.push_back(q);
    d_tmaps_raw = q;
  }
  CUDA_TRY(cudaMemcpy(d_tmaps_raw, tmaps, sizeof(LevelTensorMaps), cudaMemcpyHostToDevice));
  return 0;
}

int Engine::fetch_pyramid() {
  if (pyramid_fetched) return 0;
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaMemcpyAsync(h_pyr, d_pyr, pyr_frame_bytes * last_batch, cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  pyramid_fetched = true;
  return 0;
}

int Engine::debug_candidates(int frame, int level, int* xys, int cap) {
  if (!initialized || frame < 0 || frame >= last_batch || level < 0 || level >= nlevels) return ORB_E_ARG;
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaStreamSynchronize(stream));
  int cnt = 0;
  CUDA_TRY(cudaMemcpy(&cnt, d_cand_count + frame * nlevels + level, sizeof(int), cudaMemcpyDeviceToHost));
  const int m = std::min(std::min(cnt, levels[level].cand_cap), cap);
  std::vector<Cand> tmp(std::max(m, 1));
  CUDA_TRY(cudaMemcpy(tmp.data(), d_cand + (size_t)frame * cand_frame_elems + levels[level].cand_off,
                      sizeof(Cand) * m, cudaMemcpyDeviceToHost));
  for (int i = 0; i < m; i++) {
    xys[3 * i] = tmp[i].xy & 0xffff;
    xys[3 * i + 1] = tmp[i].xy >> 16;
    xys[3 * i + 2] = tmp[i].score;
  }
  return cnt;
}

}  // namespace orbb200
