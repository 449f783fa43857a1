// common.cuh -- host/device data model shared by the pyramid and tracker translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/dvo_b200.h"
#include "se3.cuh"

namespace dvo_b200 {

constexpr int kMaxLevels = DVO_B200_MAX_LEVELS;

// ---- device image layout --------------------------------------------------------------------
// Per image, per level l: two float2 planes of h_l rows, row pitch = w_l rounded up to even (every row
// starts 16-byte aligned, which the bulk-copy engine requires of its sources), for the role of CURRENT image:
//   P0 = (I, Z')   P2 = (I, Z)
// and the REFERENCE TILE RECORDS (below) for the role of reference image: (I, Zsel), tx and (Ix, Iy) per tile.
// Z' is the depth with NaN wherever ANY of the six channels is NaN at that pixel: a bilinear tap
// on such a pixel makes the reference reject the point (cmpunord over the 8-vector,
// dense_tracking_impl.cpp:261) and a reference point there fails isPointOk (point_selection.h:63-66),
// so one NaN test on the interpolated Z' replaces the reference's test on all lanes.
// The 8-channel AoS "acceleration" image of the reference (rgbd_image.cpp:534-543) exists only to
// make CPU gathers contiguous.  The tracker stages rectangular windows of ONE float2 plane of the
// current image in shared memory: P0 for the residual/weight/scale stage, P2 (true depth) for the
// linearisation stage, which forms the four gradient channels of every bilinear tap from the staged
// (I, Z) neighbours with the very operations of calculateDerivativeX/Y (rgbd_image.cpp:419-472), so
// gradient planes of the current image are never read (the depth gradients are not even stored).
// Zsel is the depth where the pixel belongs to the reference point list of PointSelection::select
// (point_selection.cpp:89-152; the odd last point that computeResidualsSse skips excluded) and NaN
// elsewhere: the reference side of an alignment reads the tile records and needs no mask lookup -- an
// unselected point projects to NaN and fails the bounds test like any other rejected point.
struct LevelInfo {
  int w, h, n, words;          // n = w*h pixels, words = ceil(n/32) selection-mask words (linear index y*w+x)
  int pitch;                   // row pitch of the planes in float2 elements (w rounded up to even)
  int nbands, nstrips;         // tiles of kTileW x kTileH reference pixels: nbands x nstrips
  float fx, fy, ox, oy;        // IntrinsicMatrix of this level (intrinsic_matrix.cpp:90-93: whole K * 0.5)
  size_t plane_off;            // float2 offset of P0 = (I, Z') inside dvo_b200_pyramid::planes; P2 = (I, Z) follows at + pitch*h
  size_t rec_off;              // float2 offset of the reference tile records (kRecF2 each, tile = strip * nbands + band)
  size_t mask_off;             // uint32 offset inside sel_mask
  size_t tmpl_off;             // float offset of tx[w] then ty[h] inside tmpl
  size_t range_off;            // float2 offset of the per-tile depth range {zmin, zmax} inside tile_range
};

// tile geometry of the level kernel (tracker.cu) and of the per-tile depth ranges (pyramid.cu)
constexpr int kTileW = 128;    // reference pixels per tile row: 4 warp rounds
#ifndef DVO_TILE_H
#define DVO_TILE_H 7
#endif
constexpr int kTileH = DVO_TILE_H;      // tile rows = consumer warps of a CTA (warp q walks row q of every tile of a strip); 7 consumers +
                               // 1 producer warp = 256 threads, two CTAs per SM at 128 registers per thread

// Reference tile record: everything the level kernel reads of the REFERENCE image for one tile, contiguous in HBM so that
// one bulk copy stages it (row-major planes cost one copy per tile row and plane: 14 of the ~29 copies of a stage-B tile):
//   kTileH rows x kTileW of (I, Zsel)   Zsel = depth where the pixel is a selected reference point, NaN elsewhere
//   kTileW floats tx                     point-cloud template of the tile's columns
//   kTileH rows x kTileW of (Ix, Iy)     only stage B copies this part
// Cells outside the image hold (0, NaN) / 0 / (0, 0).
constexpr int kRecTx = kTileH * kTileW;              // float2 offset of tx[]
constexpr int kRecP1 = kRecTx + kTileW / 2;          // float2 offset of the gradient rows
constexpr int kRecF2 = kRecP1 + kTileH * kTileW;     // float2 elements per record (14 848 bytes)
__host__ __device__ __forceinline__ size_t rec_cell(int x, int y, int nbands) {   // (I, Zsel) of pixel (x, y) relative to the level's records
  return (size_t)((y / kTileH) * nbands + x / kTileW) * kRecF2 + (size_t)(y % kTileH) * kTileW + (x % kTileW);
}

struct Slab;
// Pool of released slabs of one context, keyed by size (release -> reuse instead of cudaFree).  Pyramids are
// independent objects in the reference (boost::shared_ptr<RgbdImagePyramid>) and routinely outlive the tracker that
// first used them, and they may be released from another host thread than the one that built them: the pool is
// shared-owned by the context and by every slab, and guarded by its own mutex.
struct SlabPool {
  std::mutex mu;
  std::multimap<size_t, Slab*> free;
  bool closed = false;           // the context is gone: released slabs are freed instead of pooled
  int device = 0;
};

struct Slab {                  // one cudaMalloc shared by a batch of pyramids
  void* base = nullptr;
  size_t bytes = 0;
  int refs = 0;
  cudaEvent_t ready = nullptr;   // recorded on the creating stream after the build kernels
  std::shared_ptr<SlabPool> pool;
};

}  // namespace dvo_b200

// opaque handle types of the C ABI
struct dvo_b200_pyramid {
  dvo_b200_ctx* ctx = nullptr;   // the context that built it (may be gone by the time the pyramid is read: never dereferenced for that)
  int device = 0;                // CUDA ordinal the planes live on
  std::atomic<int> refcount{1};   // retain/release may come from any host thread (boost::shared_ptr semantics)
  int levels = 0;
  dvo_b200::LevelInfo L[dvo_b200::kMaxLevels];
  dvo_b200::Slab* slab = nullptr;
  float2* planes = nullptr;      // device
  uint32_t* sel_mask = nullptr;  // device: selection bitmasks of all levels (default thresholds)
  int* sel_info = nullptr;       // device: per level {S, last selected linear pixel index}
  float* tmpl = nullptr;         // device: per level tx[w], ty[h] point-cloud template (rgbd_image.cpp:197-198)
  float2* tile_range = nullptr;  // device: per level, per tile {min, max} of the non-NaN Z' (min > max: none)
  float sel_ti = 0.f, sel_td = 0.f;  // thresholds the masks were built with
  std::mutex sel_mu;                 // guards sel_ti / sel_td and the enqueueing of a re-selection
  uint64_t id = 0;
};

// A reference point selection of one pyramid (dvo::core::PointSelection with its own predicate and an optional per-pixel
// mask), separate from the pyramid's built-in selection: its own copy of the reference tile records of every level (only
// the Zsel channel differs from the pyramid's), its own mask words and {S, last}.  The level kernel reads nothing else of
// the selection, so an alignment against it runs the same kernel over the same bytes.  The template and the per-tile depth
// ranges are borrowed from the pyramid, which the selection retains.
struct dvo_b200_selection {
  int device = 0;
  std::atomic<int> refcount{1};
  dvo_b200_pyramid* pyr = nullptr;   // retained
  dvo_b200::Slab* slab = nullptr;    // shared by the selections of one build; slab->ready = build finished
  float2* rec = nullptr;             // device: tile records of every level (rec_off[l] float2 into it)
  uint32_t* mask = nullptr;          // device: mask words of every level, at the pyramid's mask_off
  int* sel_info = nullptr;           // device: per level {S, last selected linear pixel index}
  size_t rec_off[dvo_b200::kMaxLevels] = {};
  int predicate = 0;
  float ti = 0.f, td = 0.f;
};

namespace dvo_b200 {

// ---- per-pair device state ---------------------------------------------------------------------
struct PairLevel {              // what one alignment reads at the current level (uploaded per level)
  const float2* r0; const float2* r1;  // reference tile records of the level (r1: unused, kept for layout)
  const uint32_t* rmask;               // reference selection mask
  const int* rsel;                     // {S, last selected pixel}
  const float* rtmpl;                  // tx[w], ty[h]
  const float2* rrange;                // per-tile depth range of the reference
  const float2* c0; const float2* c3;  // current P0 (I, Z') and P2 (I, Z)
  float cfx, cfy, cox, coy;            // current-image intrinsics (dense_tracking.cpp:212)
  long long max_valid_pixels;          // PointSelection::getMaximumNumberOfPoints
};

struct LevelSummary {           // device mirror of dvo_b200_level_stats
  int id, termination;
  long long max_valid_pixels, valid_pixels;
  int num_iterations, has_inc;
  long long last_n, last_inc_n;
  double last_inc_nll;
};

struct PairState {
  SE3d estimate, estimate_old, initial, initial_old, inc;   // Revertable<SE3d> (util/revertable.h:45-55)
  double x[6];                  // current increment
  double error, last_error;     // IterationContext::Error / LastError
  double A[36], b[6];           // last linearisation (A without mu)
  double A_done[36];            // EstimateInformation of the last completed iteration on this level (incl. mu)
  double nll_done, prior_done;  // its TDistributionLogLikelihood / PriorLogLikelihood
  double nll_cur, prior_cur;
  int have_done;
  float precision[4];           // P_k (row-major), also P_{k-1} on entry of an iteration
  float precision_prev[4];      // P_{k-1}: what the weights of the current iteration were computed with
  float ll;
  float kt[12];                 // K * float(estimate)[0:3,:]  (dense_tracking_impl.cpp:142-152)
  long long n;                  // valid constraints of the current iteration
  long long n_keep;             // 50*floor(n/50): log-likelihood terms kept (dense_tracking_impl.cpp:413-422)
  int iteration;                // IterationContext::Iteration
  int level_active;             // 1 while this pair still iterates on the current level
  int phase_ok;                 // 1 if the residual stage produced >= 6 constraints (normal stage runs)
  int termination;
  int num_levels;
  int num_iterations_total;
  int iter_log_count;
  int pad_;
  LevelSummary levels[kMaxLevels];
  double result_T[16], result_info[36], result_ll;
};

struct Workspace {              // per-ctx scratch of the level kernel
  PairLevel* d_pair_level = nullptr;
  PairState* d_state = nullptr;
  float* d_row_exports = nullptr;    // per squad: one scale summary per image row (kSegExportFloats)
  int* d_row_base = nullptr;         // per squad, per row: valid points before the row inside its CTA
  double* d_strip_exports = nullptr; // per squad, per strip: scale summary of the strip's rows (fp64, kStripExportDoubles)
  int* d_strip_base = nullptr;       // per squad: nstrips + 1 exclusive prefixes of the strips' valid counts
  float* d_row_partial = nullptr;    // per squad, per image row: log-likelihood sum, 21 upper-triangular A, 6 b of the row
  double* d_strip_partial = nullptr; // per squad, per strip: the same, summed over the strip's rows in fp64
  float* d_dump = nullptr;           // test hook: seven residual-record planes of one level
  double* d_tinit = nullptr;         // per pair initial estimate (4x4)
  dvo_b200_iteration_stats* d_iter_log = nullptr;
  int* h_active = nullptr;           // pinned: per level, the kernel's error flag
  int* h_flag_accum = nullptr;       // pinned: a timeout code not yet reported (enqueued launches fold their flag in here)
  char* d_squads = nullptr;          // persistent kernel: SquadState[nsquads] + {queue head, error flag}
  size_t cap_pairs = 0, cap_row_exports = 0, cap_row_base = 0, cap_strip_exports = 0, cap_strip_base = 0, cap_row_partial = 0, cap_strip_partial = 0,
         cap_squads = 0, cap_iter_log = 0, cap_dump = 0, cap_tinit = 0;
};

}  // namespace dvo_b200

struct dvo_b200_ctx {
  int device = 0;
  int num_sms = 0, ctas_per_sm = 0;   // persistent-kernel grid geometry (queried once)
  unsigned long long* d_dbg = nullptr;   // DVO_B200_TIMING=1: per-level phase timers of the persistent kernel (64 slots)
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string last_error;
  int64_t launches = 0, h2d_bytes = 0, d2h_bytes = 0;
  int pending_level_flags = 0;          // levels whose error flag has been copied to pinned memory but not yet checked
  // pinned pair-descriptor slots of dvo_b200_match_batch_enqueue, used round robin: a slot is rewritten only once the event
  // recorded after the k_stage_words that read it has completed, so the host waits only when the ring wraps onto a slot
  // still in flight
  static constexpr int kDescSlots = 4;
  void* h_desc[kDescSlots] = {};
  cudaEvent_t desc_staged[kDescSlots] = {};
  size_t desc_slot_bytes = 0;
  int desc_next = 0;
  uint64_t next_pyramid_id = 1;
  dvo_b200::Workspace ws;
  std::shared_ptr<dvo_b200::SlabPool> pool;   // pooled device slabs (see SlabPool)
  // staging for uploads
  void* d_stage = nullptr; size_t d_stage_bytes = 0;
  void* h_stage = nullptr; size_t h_stage_bytes = 0;   // pinned bounce buffer for pageable sources
  void* h_results = nullptr; size_t h_results_bytes = 0;  // pinned
  // profiling
  bool profile = false;
  double prof_ms[16] = {0};           // classes 0..7 (dvo_b200_profile_read); 8 + i: level kernel of the i-th level of a match
  int64_t prof_launches[16] = {0};
  std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> prof_pending;
  std::vector<cudaEvent_t> event_pool;
  std::mutex mu;
};

namespace dvo_b200 {

int set_error(dvo_b200_ctx* ctx, int code, const std::string& msg);
int check_cuda(dvo_b200_ctx* ctx, cudaError_t e, const char* what);

#define DVO_CUDA(ctx, call)                                              \
  do {                                                                   \
    int rc__ = ::dvo_b200::check_cuda((ctx), (call), #call);             \
    if (rc__ != 0) return rc__;                                          \
  } while (0)

// profiling scope: records start/stop events around a kernel class when enabled
struct ProfScope {
  dvo_b200_ctx* ctx; int cls; cudaEvent_t a = nullptr, b = nullptr;
  ProfScope(dvo_b200_ctx* c, int cls_, int nlaunch = 1);
  ~ProfScope();
};

// Level-0 input frames of a pyramid build, in device memory, addressed in bytes: pixel (x, y) of image i of the intensity
// lies at I + i * i_img + y * i_row + x * (pixel size), likewise for the depth.  raw == 0: float32 intensity / float32 depth
// in metres (NaN = invalid); raw == 1: 8-bit grey / 16-bit raw depth (depth = raw * zscale, 0 -> NaN).  The host entry
// points stage dense images (dense_frames); device-input callers pass their own pitches.
struct FrameInput {
  const void* I = nullptr;
  const void* Z = nullptr;
  size_t i_row = 0, i_img = 0, z_row = 0, z_img = 0;
  int raw = 0;
  float zscale = 0.f;
};

// pyramid.cu
FrameInput dense_frames(const void* d_I, const void* d_Z, int raw, float zscale, int w, int h);
int pyramid_build_batch(dvo_b200_ctx* ctx, int n, const float* d_I, const float* d_Z, int w, int h, float fx, float fy,
                        float ox, float oy, int levels, float ti, float td, dvo_b200_pyramid** out);
int pyramid_build_batch_input(dvo_b200_ctx* ctx, int n, const FrameInput& in, int w, int h, float fx, float fy, float ox, float oy,
                              int levels, float ti, float td, dvo_b200_pyramid** out);
int pyramid_reselect(dvo_b200_ctx* ctx, dvo_b200_pyramid* p, float ti, float td);
void pyramid_free(dvo_b200_pyramid* p);
// Selection masks of a build: level-0 masks read at byte strides and subsampled (shift = level, the depth chain), or one
// host-staged mask per level (dense rows, shift 0; a null level allows every pixel).  mask == null everywhere: no mask.
struct SelMaskInput {
  const uint8_t* level0 = nullptr; size_t row = 0, img = 0;   // device level-0 masks of n images
  const uint8_t* per_level[kMaxLevels] = {};                  // n == 1: dense h_l x w_l bytes per level, or null
};
// n selections of n pyramids with identical geometry, one slab; out[i] retains pyrs[i].
int selection_build_batch(dvo_b200_ctx* ctx, int n, dvo_b200_pyramid* const* pyrs, int predicate, float ti, float td,
                          const SelMaskInput& masks, dvo_b200_selection** out);
void selection_free(dvo_b200_selection* s);
void pool_close(dvo_b200_ctx* ctx);
int ensure_stage(dvo_b200_ctx* ctx, size_t dev_bytes, size_t host_bytes);

// tracker.cu
// enqueue = false: T_init is host memory (staged with the descriptors); the call waits for the previous use of the pinned
// stage and, with h_results, for the results.  enqueue = true (dvo_b200_match_batch_enqueue): T_init and d_results are
// device memory, the descriptors go through the slot ring and the host does not wait for the GPU.
int tracker_match_batch(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int n, dvo_b200_pyramid* const* refs,
                        dvo_b200_pyramid* const* curs, const double* T_init, dvo_b200_result* h_results,
                        void* d_results, dvo_b200_iteration_stats* iter_stats, int max_iter_stats, bool enqueue = false,
                        dvo_b200_selection* const* sels = nullptr);
// sels != null: pair i aligns against selection sels[i] of refs[i] (= sels[i]->pyr) instead of the pyramid's own selection,
// and cfg's derivative thresholds are not read.
int check_level_flags(dvo_b200_ctx* ctx);   // after a stream synchronisation: did a level kernel report a timeout?
void fold_level_flags(dvo_b200_ctx* ctx);   // after a stream synchronisation: keep reported timeouts for check_level_flags
void tracker_release(dvo_b200_ctx* ctx);    // frees the tracker's pinned buffers and events (stream synchronised)
int tracker_linearize(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* ref, dvo_b200_pyramid* cur,
                      int level, const double* T, int use_weights, const float* prev_precision, int64_t* count,
                      float* precision_out, float* ll_out, double* A_out, double* b_out, float* planes7);

}  // namespace dvo_b200
