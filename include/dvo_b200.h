/*
 * dvo_b200.h -- C ABI of the B200-native dense RGB-D alignment engine.
 *
 * This is the drop-in boundary for ONE hot path of tum-vision/dvo_slam: dvo::DenseTracker::match()
 * (dvo_core/src/dense_tracking.cpp:123-376) and the image model it consumes
 * (dvo_core/src/core/rgbd_image.cpp, point_selection.cpp).  The reference has no FFI today: the
 * boundary there is the C++ class API of libdvo_core.so (dvo_core/include/dvo/dense_tracking.h:39-170,
 * dvo_core/include/dvo/core/rgbd_image.h:127-262).  The C++ adapter in include/dvo_b200/ keeps those
 * class signatures and forwards to the entry points below; INTEGRATION.md shows the binding.
 *
 * Plain C types only (no torch / Eigen / OpenCV types).  All functions return 0 on success and a
 * negative dvo_b200_status on failure; numerical failure is reported exactly like the reference
 * (NaN Result + TerminationCriterion), never as an error code (dense_tracking.cpp:135,375: match()
 * always returns true).  Nothing here falls back to a CPU implementation: without a CUDA device
 * dvo_b200_create fails with DVO_B200_ERR_CUDA.
 */
#ifndef DVO_B200_H_
#define DVO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVO_B200_MAX_LEVELS 8
#define DVO_B200_ABI_VERSION 1

typedef enum dvo_b200_status {
  DVO_B200_OK = 0,
  DVO_B200_ERR_INVALID_ARGUMENT = -1,
  DVO_B200_ERR_CUDA = -2,
  DVO_B200_ERR_OUT_OF_MEMORY = -3,
  DVO_B200_ERR_SHAPE_MISMATCH = -4
} dvo_b200_status;

/* dvo::DenseTracker::TerminationCriteria::Enum (dense_tracking.h:71-81) -- same numeric values */
typedef enum dvo_b200_termination {
  DVO_B200_TERM_ITERATIONS_EXCEEDED = 0,
  DVO_B200_TERM_INCREMENT_TOO_SMALL = 1,
  DVO_B200_TERM_LOG_LIKELIHOOD_DECREASED = 2,
  DVO_B200_TERM_TOO_FEW_CONSTRAINTS = 3
} dvo_b200_termination;

/* The fields of dvo::DenseTracker::Config that match() reads (dense_tracking.h:42-69; defaults
 * dense_tracking_config.cpp:27-42).  UseWeighting / InfluenceFunction* / ScaleEstimator* /
 * UseParallel are accepted by the C++ adapter for API compatibility but never reach match() in the
 * reference either (dense_tracking.cpp:81-97 vs 286-295), so they are not part of the ABI. */
typedef struct dvo_b200_config {
  int32_t first_level;                  /* FirstLevel (coarsest), default 3 */
  int32_t last_level;                   /* LastLevel (finest), default 1 */
  int32_t max_iterations_per_level;     /* default 100 */
  int32_t use_initial_estimate;         /* default 0 */
  double precision;                     /* default 5e-7 */
  double mu;                            /* default 0 */
  float intensity_derivative_threshold; /* default 0 */
  float depth_derivative_threshold;     /* default 0 */
} dvo_b200_config;

/* dvo::DenseTracker::IterationStats (dense_tracking.h:83-101) */
typedef struct dvo_b200_iteration_stats {
  int32_t level;
  int32_t id;
  int64_t valid_constraints;
  double tdist_log_likelihood;          /* TDistributionLogLikelihood (= -ll, dense_tracking.cpp:299) */
  double tdist_precision[4];            /* row-major 2x2 */
  double prior_log_likelihood;
  double increment[6];                  /* EstimateIncrement; NaN if the iteration was rejected */
  double information[36];               /* EstimateInformation (A + mu*I), row-major; NaN if rejected */
} dvo_b200_iteration_stats;

/* dvo::DenseTracker::LevelStats (dense_tracking.h:104-117) plus what its helpers expose */
typedef struct dvo_b200_level_stats {
  int32_t id;
  int32_t termination;                  /* dvo_b200_termination */
  int64_t max_valid_pixels;             /* PointSelection::getMaximumNumberOfPoints (point_selection.cpp:68-71) */
  int64_t valid_pixels;                 /* number of selected reference points S */
  int32_t num_iterations;               /* Iterations.size() */
  int32_t has_iteration_with_increment; /* LevelStats::HasIterationWithIncrement (dense_tracking_config.cpp:138-143) */
  int64_t last_valid_constraints;       /* Iterations.back().ValidConstraints */
  int64_t last_increment_valid_constraints; /* LastIterationWithIncrement().ValidConstraints, -1 if none */
  double last_increment_log_likelihood; /* LastIterationWithIncrement().TDistributionLogLikelihood, NaN if none */
} dvo_b200_level_stats;

/* dvo::DenseTracker::Result (dense_tracking.h:125-140) */
typedef struct dvo_b200_result {
  double transformation[16];            /* row-major 4x4; = estimate^-1 (dense_tracking.cpp:371) */
  double information[36];               /* row-major 6x6; = A_last * 0.008^2 (dense_tracking.cpp:372) */
  double log_likelihood;
  int32_t num_levels;
  int32_t num_iterations_total;
  dvo_b200_level_stats levels[DVO_B200_MAX_LEVELS];
} dvo_b200_result;

typedef struct dvo_b200_ctx dvo_b200_ctx;          /* one per host thread / CUDA stream */
typedef struct dvo_b200_pyramid dvo_b200_pyramid;  /* device mirror of dvo::core::RgbdImagePyramid */
typedef struct dvo_b200_selection dvo_b200_selection;  /* dvo::core::PointSelection of one pyramid (see below) */

/* ---- context ------------------------------------------------------------------------------ */
int dvo_b200_abi_version(void);
/* device: CUDA ordinal.  stream: a cudaStream_t to run on, or NULL to create a private stream. */
int dvo_b200_create(int device, void* stream, dvo_b200_ctx** out);
int dvo_b200_destroy(dvo_b200_ctx* ctx);
void* dvo_b200_stream(dvo_b200_ctx* ctx);             /* the cudaStream_t all work is enqueued on */
int dvo_b200_synchronize(dvo_b200_ctx* ctx);
const char* dvo_b200_last_error(dvo_b200_ctx* ctx);   /* human readable, valid until next call */
void dvo_b200_config_default(dvo_b200_config* cfg);   /* DenseTracker::getDefaultConfig() */
/* counters for the bench harness: kernels launched / bytes copied through this ctx so far */
int64_t dvo_b200_kernel_launches(dvo_b200_ctx* ctx);
int64_t dvo_b200_h2d_bytes(dvo_b200_ctx* ctx);
int64_t dvo_b200_d2h_bytes(dvo_b200_ctx* ctx);

/* ---- image pyramid (replaces RgbdCameraPyramid::create + RgbdImagePyramid::build +
 *      RgbdImage::buildAccelerationStructure, rgbd_image.cpp:156-172,283-296,534-543) ---------- */
/* intensity/depth: HOST pointers to height*width float32, row-major; depth in metres, NaN = invalid
 * (what benchmark_slam.cpp:46-93 produces).  K = fx, fy, ox, oy of level 0.  levels >= 1.
 * Uploads, builds all levels (2x2 mean / subsample / central differences) and the default
 * point-selection masks on the device.  Asynchronous on the ctx stream; host buffers must stay
 * valid until dvo_b200_synchronize() unless they are not pinned (then the copy is staged). */
int dvo_b200_pyramid_create(dvo_b200_ctx* ctx, const float* intensity, const float* depth, int32_t width,
                            int32_t height, float fx, float fy, float ox, float oy, int32_t levels,
                            dvo_b200_pyramid** out);
/* n images with identical geometry; intensity/depth point to n consecutive images. */
int dvo_b200_pyramid_create_batch(dvo_b200_ctx* ctx, int32_t n, const float* intensity, const float* depth,
                                  int32_t width, int32_t height, float fx, float fy, float ox, float oy,
                                  int32_t levels, dvo_b200_pyramid** out /* n handles */);
/* N2 row (surface_pyramid.cpp:65-105, benchmark_slam.cpp:58-77): 8-bit grey + 16-bit raw depth in,
 * conversion (u16*scale, 0 -> NaN; u8 -> f32) fused into the upload. */
int dvo_b200_pyramid_create_raw(dvo_b200_ctx* ctx, const uint8_t* grey, const uint16_t* raw_depth, float depth_scale,
                                int32_t width, int32_t height, float fx, float fy, float ox, float oy,
                                int32_t levels, dvo_b200_pyramid** out);
/* n images with identical geometry; grey / raw_depth point to n consecutive images. */
int dvo_b200_pyramid_create_raw_batch(dvo_b200_ctx* ctx, int32_t n, const uint8_t* grey, const uint16_t* raw_depth,
                                      float depth_scale, int32_t width, int32_t height, float fx, float fy, float ox,
                                      float oy, int32_t levels, dvo_b200_pyramid** out /* n handles */);
/* 8-bit BGR (interleaved, the order cv::imread(file, 1) returns) + 16-bit raw depth in: cv::cvtColor(rgb, grey,
 * CV_BGR2GRAY) + convertTo(CV_32F) of the loader (benchmark_slam.cpp:50-68) and convertRawDepthImageSse run on the
 * device.  Grey = (1868 B + 9617 G + 4899 R + 8192) >> 14, OpenCV's 8-bit fixed-point BGR2GRAY. */
int dvo_b200_pyramid_create_bgr_batch(dvo_b200_ctx* ctx, int32_t n, const uint8_t* bgr, const uint16_t* raw_depth,
                                      float depth_scale, int32_t width, int32_t height, float fx, float fy, float ox,
                                      float oy, int32_t levels, dvo_b200_pyramid** out /* n handles */);
/* ---- frames already in GPU memory ---------------------------------------------------------------------------------
 * The three pixel formats of the host entry points above, read in place from DEVICE memory (a decoder surface, a
 * rendered frame, a tensor): the pyramids equal bit for bit those the matching host entry point builds from the same
 * pixels (dvo_b200_pyramid_create_batch / _raw_batch / _bgr_batch). */
typedef enum dvo_b200_frame_format {
  DVO_B200_FRAME_F32 = 0,          /* float32 intensity (0..255 units) + float32 depth in metres, NaN = invalid */
  DVO_B200_FRAME_GREY8_RAW16 = 1,  /* 8-bit grey + 16-bit raw depth: depth = raw * depth_scale, 0 -> NaN       */
  DVO_B200_FRAME_BGR8_RAW16 = 2    /* interleaved 8-bit BGR (OpenCV order) + 16-bit raw depth                  */
} dvo_b200_frame_format;

/* n images of width x height.  Pixel (x, y) of image i of the colour plane lies at
 *   colour + i * colour_image_bytes + y * colour_row_bytes + x * (4 bytes F32, 1 GREY8, 3 BGR8)
 * and likewise for depth (4 bytes F32, 2 RAW16): pitched buffers, slices of wider tensors and every k-th image of a batch
 * need no copy.  Row strides are at least width x pixel size, image strides (read only for n > 1) at least height x row
 * stride; pointers and strides are multiples of the element size (4 for float32, 2 for 16-bit). */
typedef struct dvo_b200_device_frames {
  int32_t format, width, height, reserved;                             /* dvo_b200_frame_format; reserved = 0 */
  const void* colour;  int64_t colour_row_bytes, colour_image_bytes;   /* DEVICE pointer to image 0 + strides in bytes */
  const void* depth;   int64_t depth_row_bytes,  depth_image_bytes;
  float depth_scale;                                                   /* raw formats only */
} dvo_b200_device_frames;

/* Both pointers must be device (or managed) memory of the context's device; host memory is refused with
 * DVO_B200_ERR_INVALID_ARGUMENT and nothing is copied.  The frames are read on the context's stream: a caller that writes
 * them on another stream makes the context's stream wait for that work first (cudaStreamWaitEvent).  The pyramids keep no
 * reference to the frames, so work enqueued later on the context's stream may overwrite them.  Moves no frame over the bus
 * and does not synchronise. */
int dvo_b200_pyramid_create_device_batch(dvo_b200_ctx* ctx, int32_t n, const dvo_b200_device_frames* frames,
                                         float fx, float fy, float ox, float oy, int32_t levels, dvo_b200_pyramid** out);

int dvo_b200_pyramid_device(const dvo_b200_pyramid* p);   /* CUDA ordinal the pyramid lives on (-1: null handle) */
int dvo_b200_pyramid_retain(dvo_b200_pyramid* p);   /* boost::shared_ptr semantics of RgbdImagePyramidPtr */
int dvo_b200_pyramid_release(dvo_b200_pyramid* p);
int dvo_b200_pyramid_num_levels(const dvo_b200_pyramid* p);
int dvo_b200_pyramid_level_info(const dvo_b200_pyramid* p, int32_t level, int32_t* width, int32_t* height, float K[4]);
/* Debug/test read-back of one level: 6 planes (I, Z, Ix, Iy, Zx, Zy) of h*w floats into host memory.
 * Z is the tracker's masked depth: NaN wherever the reference would reject the pixel as a bilinear
 * tap or as a reference point (any of I,Z,Ix,Iy,Zx,Zy NaN).  Synchronises.  ctx may be NULL: pyramids are shared objects
 * that can outlive the context that built them (boost::shared_ptr<RgbdImagePyramid>); the read then waits for the
 * pyramid's own build to finish and uses no context at all. */
int dvo_b200_pyramid_download(dvo_b200_ctx* ctx, const dvo_b200_pyramid* p, int32_t level, float* planes6);
/* PointSelection::select result (point_selection.cpp:89-152) for the given thresholds: number of
 * selected points S and (optional) h*w byte mask.  Synchronises. */
int dvo_b200_pyramid_select(dvo_b200_ctx* ctx, dvo_b200_pyramid* p, int32_t level, float intensity_threshold,
                            float depth_threshold, int64_t* count, uint8_t* mask);

/* ---- alignment ---------------------------------------------------------------------------- */
/* DenseTracker::match(RgbdImagePyramid& reference, RgbdImagePyramid& current, Result&)
 * (dense_tracking.cpp:123-129).  T_init: row-major 4x4 Result.Transformation on entry (read iff
 * cfg->use_initial_estimate), may be NULL.  Blocks until the result is on the host. */
int dvo_b200_match(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* reference,
                   dvo_b200_pyramid* current, const double* T_init, dvo_b200_result* result);
/* n independent alignments (the TBB fan-outs of local_tracker.cpp:180-184 and
 * keyframe_graph.cpp:587-590 as one call).  T_init: n*16 doubles or NULL.  iteration_stats: optional
 * n*max_iteration_stats entries, pair p's iterations start at p*max_iteration_stats, in order. */
int dvo_b200_match_batch(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n,
                         dvo_b200_pyramid* const* references, dvo_b200_pyramid* const* currents,
                         const double* T_init, dvo_b200_result* results,
                         dvo_b200_iteration_stats* iteration_stats, int32_t max_iteration_stats);
/* Asynchronous variant: enqueues the batch and leaves the n results in DEVICE memory
 * (d_results: device pointer to n dvo_b200_result) so they can be gathered with NCCL without a
 * host round trip.  No synchronisation. */
int dvo_b200_match_batch_device(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n,
                                dvo_b200_pyramid* const* references, dvo_b200_pyramid* const* currents,
                                const double* T_init, void* d_results);

/* Enqueue-only batch alignment: d_T_init (DEVICE, n*16 doubles, row-major Result.Transformation on entry, read iff
 * cfg->use_initial_estimate; may be NULL) and d_results (DEVICE, n dvo_b200_result) live on the context's device and are
 * read / written on its stream, so steps can be chained on a stream without the host waiting.  Once the context is warm
 * (an earlier call with at least as many pairs and levels), the call does not block on the GPU: the pair descriptors --
 * the only host-to-device traffic -- go up through a ring of pinned slots, and the host waits only when the ring wraps
 * onto a slot the GPU has not read yet.  A kernel timeout in any call enqueued since the last synchronisation is
 * reported by the next dvo_b200_synchronize.  Pyramids built by another context must stay referenced until then. */
int dvo_b200_match_batch_enqueue(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n,
                                 dvo_b200_pyramid* const* references, dvo_b200_pyramid* const* currents,
                                 const double* d_T_init, void* d_results);

/* ---- reference point selections (dvo::core::PointSelection with its own predicate, point_selection.h:39-124) -----------
 * A selection is a device object of its own, separate from the pyramid's built-in selection (the one cfg's thresholds and
 * dvo_b200_pyramid_select set): the reference points of every level of one pyramid, chosen by a predicate and optionally
 * restricted by a per-pixel mask (exclude dynamic objects, the robot's body, saturated regions).  It retains its pyramid
 * and may outlive the caller's pyramid handle and the context that built it.  Any number of selections of one pyramid can
 * be aligned against at the same time, from any context.  Memory: its own copy of the reference tile records (about
 * 7.4 MB at 640x480, 5 levels) from the context's slab pool. */
typedef enum dvo_b200_predicate {
  DVO_B200_PREDICATE_GRADIENT_THRESHOLD = 0,  /* ValidPointAndGradientThresholdPredicate(ti, td) (point_selection.h:52-67)  */
  DVO_B200_PREDICATE_VALID_POINT = 1,         /* ValidPointPredicate: z, zdx, zdy not NaN (point_selection.h:39-47)        */
  DVO_B200_PREDICATE_MASK_ONLY = 2            /* the mask alone decides; a pixel without valid depth still counts in S     */
} dvo_b200_predicate;

/* One selection of p.  level_masks: NULL (no mask), or p's number of levels entries, each NULL (every pixel allowed) or
 * h_l*w_l HOST bytes of level l, nonzero = allowed.  The selected pixels are those where the predicate holds and the
 * mask allows; the odd last one is dropped as computeResidualsSse does (dense_tracking_impl.cpp:169).  ti / td are read
 * for GRADIENT_THRESHOLD only.  Asynchronous on the ctx stream; the masks are copied before the call returns. */
int dvo_b200_selection_create(dvo_b200_ctx* ctx, dvo_b200_pyramid* p, int32_t predicate, float ti, float td,
                              const uint8_t* const* level_masks, dvo_b200_selection** out);
/* n selections of n pyramids of identical geometry in one build.  d_masks: NULL (no mask) or n level-0 masks of 8 bits per
 * pixel in DEVICE memory, nonzero = allowed: pixel (x, y) of mask i at d_masks + i * image_bytes + y * row_bytes + x, row
 * stride at least the width, image stride (read for n > 1) at least height x row stride.  Level l reads
 * M_0(y << l, x << l), the subsample chain of the depth.  Host pointers, memory of another device and short strides are
 * refused with DVO_B200_ERR_INVALID_ARGUMENT and build nothing.  Does not synchronise; the masks are read on the ctx
 * stream (a caller that writes them on another stream makes the ctx stream wait first). */
int dvo_b200_selection_create_device_batch(dvo_b200_ctx* ctx, int32_t n, dvo_b200_pyramid* const* pyramids, int32_t predicate,
                                           float ti, float td, const void* d_masks, int64_t row_bytes, int64_t image_bytes,
                                           dvo_b200_selection** out /* n handles */);
int dvo_b200_selection_retain(dvo_b200_selection* s);
int dvo_b200_selection_release(dvo_b200_selection* s);
dvo_b200_pyramid* dvo_b200_selection_pyramid(dvo_b200_selection* s);   /* borrowed: the selection holds the reference */
/* Number of selected points S of a level (PointSelection::select's point count) and, optionally, the h*w byte mask of the
 * selected points (the odd last one included, as dvo_b200_pyramid_select reports it).  Synchronises; ctx may be NULL: the
 * read then waits for the selection's build only. */
int dvo_b200_selection_download(dvo_b200_ctx* ctx, const dvo_b200_selection* s, int32_t level, int64_t* count, uint8_t* mask);
/* dvo_b200_match_batch / dvo_b200_match_batch_enqueue with pair i aligned against selection references[i] of its pyramid:
 * DenseTracker::match(PointSelection& reference, current, result) (dense_tracking.cpp:131-376).  cfg's derivative
 * thresholds are not read: the selection's predicate decides.  A selection equal to the pyramid's own selection gives
 * the same result records byte for byte. */
int dvo_b200_match_batch_selected(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n,
                                  dvo_b200_selection* const* references, dvo_b200_pyramid* const* currents,
                                  const double* T_init, dvo_b200_result* results,
                                  dvo_b200_iteration_stats* iteration_stats, int32_t max_iteration_stats);
int dvo_b200_match_batch_selected_enqueue(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n,
                                          dvo_b200_selection* const* references, dvo_b200_pyramid* const* currents,
                                          const double* d_T_init, void* d_results);

/* ---- one process, several GPUs (SURVEY.md 8e) ----------------------------------------------------
 * The reference's batch producers are single-process C++ loops over independent match() calls
 * (constraint_proposal_validator.cpp:141-146, keyframe_graph.cpp:587-590).  A dvo_b200_sharded owns one context per
 * device; a batch of n pairs is cut into contiguous shards of pair indices (dvo_b200_shard_range: the remainder goes to
 * the first shards -- the same partition the multi-process path dvo_slam_b200/distributed.py uses), each shard runs on
 * its own host thread and device, and every shard writes its results into its range of the caller's host array.  The
 * alignments exchange nothing, so a one-process caller needs no communicator; across processes the gather is one NCCL
 * all-gather of the records left in device memory by dvo_b200_match_batch_device. */
typedef struct dvo_b200_sharded dvo_b200_sharded;
/* devices: n_devices CUDA ordinals, or NULL for 0..n_devices-1 (an ordinal may repeat: two shards on one GPU). */
int dvo_b200_sharded_create(int32_t n_devices, const int32_t* devices, dvo_b200_sharded** out);
int dvo_b200_sharded_destroy(dvo_b200_sharded* s);
int32_t dvo_b200_sharded_num_shards(const dvo_b200_sharded* s);
dvo_b200_ctx* dvo_b200_sharded_ctx(dvo_b200_sharded* s, int32_t shard);     /* the shard's context (owned by s) */
const char* dvo_b200_sharded_last_error(dvo_b200_sharded* s);
int dvo_b200_shard_range(int64_t total, int32_t n_shards, int32_t shard, int64_t* begin, int64_t* end);
/* n images -> n pyramids, image i on the device of the shard that owns index i of n; blocks until the uploads are done */
int dvo_b200_sharded_pyramid_create_batch(dvo_b200_sharded* s, int32_t n, const float* intensity, const float* depth,
                                          int32_t width, int32_t height, float fx, float fy, float ox, float oy,
                                          int32_t levels, dvo_b200_pyramid** out /* n handles */);
int dvo_b200_sharded_pyramid_create_raw_batch(dvo_b200_sharded* s, int32_t n, const uint8_t* grey, const uint16_t* raw_depth,
                                              float depth_scale, int32_t width, int32_t height, float fx, float fy,
                                              float ox, float oy, int32_t levels, dvo_b200_pyramid** out);
/* dvo_b200_match_batch over all shards: pair i must live on the device of the shard that owns index i of n (as the two
 * calls above place them), else DVO_B200_ERR_INVALID_ARGUMENT.  Same result layout as dvo_b200_match_batch. */
int dvo_b200_match_batch_sharded(dvo_b200_sharded* s, const dvo_b200_config* cfg, int32_t n,
                                 dvo_b200_pyramid* const* references, dvo_b200_pyramid* const* currents,
                                 const double* T_init, dvo_b200_result* results,
                                 dvo_b200_iteration_stats* iteration_stats, int32_t max_iteration_stats);

/* One evaluation of the residual stage at a fixed transform (test / debug; also the basis of
 * DenseTracker::computeIntensityErrorImage, dense_tracking.cpp:378-444): 7 planes
 * {e.i, e.z, e.idx, e.idy, e.zdx, e.zdy, z_ref} of h*w floats, NaN where invalid.  T: row-major
 * 4x4 double "estimate" (reference -> current).  Returns n (valid constraints) in *count. */
int dvo_b200_residual_image(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* reference,
                            dvo_b200_pyramid* current, int32_t level, const double* T, float* planes7,
                            int64_t* count);
/* DenseTracker::computeIntensityErrorImage (dense_tracking.cpp:378-444): image = h*w floats on the host,
 * |intensity residual| at every selected reference pixel whose warped residual is valid, 0 elsewhere (the odd
 * last selected point included: the reference's SSE residual loop never visits it).  T as above; the selection
 * thresholds come from cfg.  *count (optional) = residuals written. */
int dvo_b200_intensity_error_image(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* reference,
                                   dvo_b200_pyramid* current, int32_t level, const double* T, float* image,
                                   int64_t* count);
/* One linearisation at a fixed transform (test hook mirroring dense_tracking.cpp:271-343):
 * use_weights=0 -> w=1 (first iteration on a level), else Student-t weights from prev_precision. */
int dvo_b200_linearize(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* reference,
                       dvo_b200_pyramid* current, int32_t level, const double* T, int32_t use_weights,
                       const float* prev_precision, int64_t* count, float* precision_out, float* ll_out,
                       double* A_out, double* b_out);

/* ---- profiling hooks (bench.py roofline): per-kernel-class accumulated device time measured with
 *      CUDA events on the ctx stream.  classes: 0 residual/scale stage, 1 normal-equation stage,
 *      2 per-pair step kernels, 3 pyramid build, 4 selection. -------------------------------- */
int dvo_b200_profile_enable(dvo_b200_ctx* ctx, int32_t enable);
int dvo_b200_profile_read(dvo_b200_ctx* ctx, double ms_out[8], int64_t launches_out[8], int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* DVO_B200_H_ */
