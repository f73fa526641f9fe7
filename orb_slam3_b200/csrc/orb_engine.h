// Host-side state of one ORB extractor handle (see orb_extract.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/orb_b200.h"
#include "octree_core.h"

namespace orbb200 {

void set_last_error(const std::string& s);
const char* last_error();

// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the kernel (per device), not to a handle:
// several handles with different sizes share it, so it is only ever raised, process-wide.
inline cudaError_t raise_dynamic_smem(const void* kernel, size_t bytes, int device) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> cur;
  std::lock_guard<std::mutex> lk(mu);
  size_t& c = cur[std::make_pair(kernel, device)];
  if (c == 0) c = 48 * 1024;  // what every kernel may use without the attribute
  if (bytes <= c) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) c = bytes;
  return e;
}

// Per pyramid level; lives in host and device memory.
struct LevelDev {
  int w, h, pitch;
  size_t img_off;        // byte offset inside a frame's pyramid slab
  float scale;           // mvScaleFactor[level]
  int patch_size;        // (int)(31 * scale)
  OctreeLevelParams oct;
  int cand_cap;
  size_t cand_off;       // element offset inside a frame's candidate slab
  int sel_off;           // element offset inside a frame's selected-keypoint slab
  size_t scratch_off;    // byte offset inside a frame's octree scratch slab
};

// One FAST cell (ORBextractor.cc:805-822): image rectangle and the shift the
// reference adds to cell-local keypoint coordinates (:863-868).
struct CellDesc {
  int level, x0, y0, x1, y1, shift_x, shift_y;
};

struct BlurTile {
  int level, x0, y0;
};

struct ResizeTab {
  int x_off = 0, y_off = 0;
};

struct LevelTensorMaps;

struct Engine {
  // parameters and tables (ORBextractor.cc:409-469)
  int nfeatures, nlevels, ini_th, min_th, device;
  double scale_factor;
  std::vector<float> scale, inv_scale, sigma2, inv_sigma2;
  std::vector<int> quota;
  int umax[16];

  // geometry for the current image size
  std::vector<LevelDev> levels;
  std::vector<ResizeTab> rs;
  size_t pyr_frame_bytes = 0, cand_frame_elems = 0, scratch_frame_bytes = 0, sel_frame_elems = 0;
  int out_cap = 0, num_cells = 0, num_tiles = 0, oct_smem_node_cap = 0, oct_smem_node_cap_full = 0;
  size_t oct_smem_bytes = 0;
  int cap_rows = 0, cap_cols = 0, cap_batch = 0, cap_batch_hint = 1;

  // device state
  bool initialized = false;
  cudaStream_t stream = nullptr, last_stream = nullptr, stream_in = nullptr, stream_out = nullptr;
  // lanes: a device-resident batch can be cut into up to MAX_LANES sub-batches that run the whole kernel chain on
  // their own streams (lane 0 = the caller's stream), so the latency-bound kernels of one sub-batch (octree) share
  // the SMs with the issue-bound ones of another (FAST); every lane has its own blur side stream
  static constexpr int MAX_LANES = 4;
  cudaStream_t stream_side[MAX_LANES] = {nullptr, nullptr, nullptr, nullptr};
  cudaStream_t stream_lane[MAX_LANES] = {nullptr, nullptr, nullptr, nullptr};   // [0] unused
  cudaEvent_t ev_pyr_done[MAX_LANES] = {nullptr, nullptr, nullptr, nullptr}, ev_blur_done[MAX_LANES] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_lane_go = nullptr, ev_lane_done[MAX_LANES] = {nullptr, nullptr, nullptr, nullptr};
  int lanes = 1;
  std::vector<cudaEvent_t> chunk_events;
  std::vector<void*> dev_allocs, host_allocs;
  uint8_t *d_pyr = nullptr, *d_blur = nullptr, *d_scratch = nullptr, *d_desc = nullptr, *d_stage = nullptr;
  Cand* d_cand = nullptr;
  int *d_sel = nullptr, *d_slot = nullptr, *d_cand_count = nullptr, *d_sel_count = nullptr;
  int *d_n = nullptr, *d_mono = nullptr, *d_lap = nullptr, *d_warp_level = nullptr;
  int *d_xofs = nullptr, *d_yofs = nullptr, *d_pattern_t = nullptr;
  short2 *d_alpha = nullptr, *d_beta = nullptr;
  orb_keypoint* d_kps = nullptr;
  // Results are double-buffered: every extract_batch_* call writes the set the previous call did not use, so the
  // keypoints / descriptors / counts of call i stay valid (for matchers still reading them on another stream)
  // until call i + 2.  d_kps / d_desc / d_n / d_mono always point at the set of the latest call.
  orb_keypoint* d_kps_buf[2] = {nullptr, nullptr};
  uint8_t* d_desc_buf[2] = {nullptr, nullptr};
  int* d_n_buf[2] = {nullptr, nullptr};
  int* d_mono_buf[2] = {nullptr, nullptr};
  int out_idx = 0;
  void flip_outputs() {
    out_idx ^= 1;
    d_kps = d_kps_buf[out_idx]; d_desc = d_desc_buf[out_idx]; d_n = d_n_buf[out_idx]; d_mono = d_mono_buf[out_idx];
  }
  LevelDev* d_levels = nullptr;
  CellDesc* d_cells = nullptr;
  BlurTile* d_tiles = nullptr;
  int* h_counts = nullptr;
  uint8_t* h_pyr = nullptr;
  bool pyramid_fetched = false;
  int last_batch = 0;

  // profiling
  bool profiling = false;
  std::vector<cudaEvent_t> ev_pool[ORB_NUM_STAGES + 1];
  double stage_ms[ORB_NUM_STAGES] = {0};
  long long stage_launches[ORB_NUM_STAGES] = {0};
  long long total_launches = 0;

  Engine(int nfeatures, float scale_factor, int nlevels, int ini_th, int min_th, int device);
  ~Engine();
  void release();
  template <class T> int dalloc(T** p, size_t count);
  int ensure(int rows, int cols, int batch);
  void stage_begin(int st, cudaStream_t s);
  void stage_end(int st, cudaStream_t s, int launches);
  int collect_times(double* ms, long long* launches, bool reset);
  int run_device(int f0, int batch, const int* lap_host, cudaStream_t s, int lane = 0);
  int extract_batch_host(int batch, const uint8_t* const* imgs, int rows, int cols, size_t step, const int* lap,
                         orb_keypoint* kps, uint8_t* desc, int cap, int* n, int* mono);
  int extract_batch_device(int batch, const uint8_t* d_imgs, size_t frame_stride, int rows, int cols, size_t step,
                           const int* lap, cudaStream_t user);
  LevelTensorMaps* tmaps = nullptr;  // host copy of the per-level TMA descriptors
  void* d_tmaps_raw = nullptr;       // device copy read by cp.async.bulk.tensor (first 16: CTA-per-cell boxes,
                                     // next 16: the warp-per-cell boxes)
  // warp-per-cell FAST (fast_warp_kernel): tile / score map / queue geometry, persistent grid size
  int fw_tile_pitch = 0, fw_tile_rows = 0, fw_smap_pitch = 0, fw_smap_bytes = 0, fw_queue_cap = 0, fw_per_warp = 0;
  int fw_grid = 0, fw_align_mask = 15, fw_gq_off = 0;
  bool fw_enabled = false;
  bool resize_words_ok = false;  // resize_words_kernel (word loads + PRMT + IDP.2A) applies as well
  bool resize_rows_ok = false;  // resize_rows_kernel (shared-memory staged) applies to this pyramid geometry
  int encode_tensor_maps(int batch);
  int fetch_pyramid();
  int debug_candidates(int frame, int level, int* xys, int cap);
};

int debug_sincos_device(int device, const float* x, size_t n, float* c, float* s);
void debug_sincos_host(const float* x, size_t n, float* c, float* s, int fused);

}  // namespace orbb200

// The opaque handle of include/orb_b200.h.
struct orb_extractor {
  orbb200::Engine e;
  orb_extractor(int nf, float sf, int nl, int ini, int mn, int dev) : e(nf, sf, nl, ini, mn, dev) {}
};
