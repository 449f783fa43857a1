// capi.cu -- the extern "C" surface declared in include/dvo_b200.h.
#include "common.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <vector>

namespace dvo_b200 {

int set_error(dvo_b200_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->last_error = msg;
  return code;
}

int check_cuda(dvo_b200_ctx* ctx, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  std::string msg = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
  cudaGetLastError();
  return set_error(ctx, e == cudaErrorMemoryAllocation ? DVO_B200_ERR_OUT_OF_MEMORY : DVO_B200_ERR_CUDA, msg);
}

static cudaEvent_t get_event(dvo_b200_ctx* ctx) {
  if (!ctx->event_pool.empty()) { cudaEvent_t e = ctx->event_pool.back(); ctx->event_pool.pop_back(); return e; }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}

ProfScope::ProfScope(dvo_b200_ctx* c, int cls_, int nlaunch) : ctx(c), cls(cls_) {
  if (!ctx->profile) return;
  a = get_event(ctx); b = get_event(ctx);
  cudaEventRecord(a, ctx->stream);
  ctx->prof_launches[cls] += nlaunch;
}
ProfScope::~ProfScope() {
  if (!a) return;
  cudaEventRecord(b, ctx->stream);
  ctx->prof_pending.push_back({cls, {a, b}});
}

static void drain_profile(dvo_b200_ctx* ctx) {
  for (auto& e : ctx->prof_pending) {
    float ms = 0.f;
    cudaEventSynchronize(e.second.second);
    cudaEventElapsedTime(&ms, e.second.first, e.second.second);
    ctx->prof_ms[e.first] += ms;
    ctx->event_pool.push_back(e.second.first);
    ctx->event_pool.push_back(e.second.second);
  }
  ctx->prof_pending.clear();
}

namespace {

__global__ void k_convert_bgr(const uint8_t* __restrict__ bgr, size_t row_bytes, size_t image_bytes, uint8_t* __restrict__ grey,
                              int w, int h) {
  // benchmark_slam.cpp:58-68: cv::cvtColor(rgb, grey, CV_BGR2GRAY) on CV_8UC3 (convertTo(CV_32F) happens in the pyramid
  // kernels' loads).  OpenCV's 8-bit path is fixed point: (B*1868 + G*9617 + R*4899 + (1 << 13)) >> 14.  The BGR frames
  // are read at their byte strides; the grey images are written dense.
  const int img = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= w * h) return;
  const int y = i / w, x = i - y * w;
  const uint8_t* p = bgr + img * image_bytes + (size_t)y * row_bytes + 3 * (size_t)x;
  grey[(size_t)img * w * h + i] = (uint8_t)((1868 * (int)p[0] + 9617 * (int)p[1] + 4899 * (int)p[2] + 8192) >> 14);
}

void convert_bgr(dvo_b200_ctx* ctx, const uint8_t* bgr, size_t row_bytes, size_t image_bytes, uint8_t* grey, int n, int w, int h) {
  k_convert_bgr<<<dim3((unsigned)(((size_t)w * h + 255) / 256), n), 256, 0, ctx->stream>>>(bgr, row_bytes, image_bytes, grey, w, h);
  ctx->launches++;
}

// device frames: device or managed memory of the context's device (no host memory, no silent copy)
int check_device_pointer(dvo_b200_ctx* ctx, const void* p, const std::string& what) {
  cudaPointerAttributes a;
  const cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, what + ": not a CUDA pointer (" + cudaGetErrorString(e) + ")");
  }
  if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, what + ": host memory; device or managed memory of the context's device required");
  if (a.device != ctx->device)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, what + ": memory of device " + std::to_string(a.device) +
                                                             ", the context runs on device " + std::to_string(ctx->device));
  return 0;
}

// one plane of dvo_b200_device_frames: minimum strides and element alignment
int check_plane(dvo_b200_ctx* ctx, const char* name, const void* p, int64_t row_bytes, int64_t image_bytes, int n, int width,
                int height, int pixel_bytes, int elem_bytes) {
  const std::string f = std::string("pyramid_create_device_batch: frames->") + name;
  if (!p) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + " is null");
  if (row_bytes < (int64_t)width * pixel_bytes)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + "_row_bytes " + std::to_string(row_bytes) + " < width x " +
                                                             std::to_string(pixel_bytes) + " bytes");
  if (n > 1 && image_bytes < (int64_t)height * row_bytes)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + "_image_bytes " + std::to_string(image_bytes) + " < height x " + name +
                                                             "_row_bytes");
  if ((uintptr_t)p % elem_bytes) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + " is not " + std::to_string(elem_bytes) + "-byte aligned");
  if (row_bytes % elem_bytes)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + "_row_bytes is not a multiple of " + std::to_string(elem_bytes));
  if (n > 1 && image_bytes % elem_bytes)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + "_image_bytes is not a multiple of " + std::to_string(elem_bytes));
  return check_device_pointer(ctx, p, f);
}

// device result records and initial estimates of the enqueue entry points
int check_enqueue_buffers(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, const double* d_T_init, void* d_results, const std::string& f) {
  if ((uintptr_t)d_results % 8) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + ": d_results is not 8-byte aligned");
  int rc = check_device_pointer(ctx, d_results, f + ": d_results");
  if (rc) return rc;
  if (cfg && cfg->use_initial_estimate && d_T_init) {
    if ((uintptr_t)d_T_init % 8) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + ": d_T_init is not 8-byte aligned");
    if ((rc = check_device_pointer(ctx, d_T_init, f + ": d_T_init"))) return rc;
  }
  return 0;
}

}  // namespace
}  // namespace dvo_b200

using namespace dvo_b200;

extern "C" {

int dvo_b200_abi_version(void) { return DVO_B200_ABI_VERSION; }

int dvo_b200_create(int device, void* stream, dvo_b200_ctx** out) {
  if (!out) return DVO_B200_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
    cudaGetLastError();
    return DVO_B200_ERR_CUDA;   // no CPU fallback: without a CUDA device there is no engine
  }
  if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return DVO_B200_ERR_CUDA; }
  dvo_b200_ctx* ctx = new dvo_b200_ctx;
  ctx->device = device;
  ctx->pool = std::make_shared<SlabPool>();
  ctx->pool->device = device;
  if (stream) { ctx->stream = (cudaStream_t)stream; ctx->own_stream = false; }
  else {
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); delete ctx; return DVO_B200_ERR_CUDA; }
    ctx->own_stream = true;
  }
  if (getenv("DVO_B200_TIMING")) {
    cudaMalloc((void**)&ctx->d_dbg, sizeof(unsigned long long) * 256);
    cudaMemset(ctx->d_dbg, 0, sizeof(unsigned long long) * 256);
    for (int l = 0; l < 8; ++l) { unsigned long long big = ~0ull; cudaMemcpy(ctx->d_dbg + 128 + 8 * l + 6, &big, 8, cudaMemcpyHostToDevice); }
  }
  *out = ctx;
  return 0;
}

int dvo_b200_destroy(dvo_b200_ctx* ctx) {
  if (!ctx) return DVO_B200_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  drain_profile(ctx);
  for (cudaEvent_t e : ctx->event_pool) cudaEventDestroy(e);
  Workspace& ws = ctx->ws;
  cudaFree(ws.d_pair_level); cudaFree(ws.d_state); cudaFree(ws.d_row_exports); cudaFree(ws.d_row_base);
  cudaFree(ws.d_strip_exports); cudaFree(ws.d_strip_base); cudaFree(ws.d_row_partial); cudaFree(ws.d_strip_partial); cudaFree(ws.d_dump); cudaFree(ws.d_tinit);
  cudaFree(ws.d_iter_log); cudaFree(ws.d_squads);
  if (ws.h_active) cudaFreeHost(ws.h_active);
  pool_close(ctx);
  tracker_release(ctx);
  cudaFree(ctx->d_stage);
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  if (ctx->h_results) cudaFreeHost(ctx->h_results);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  cudaGetLastError();
  delete ctx;
  return 0;
}

void* dvo_b200_stream(dvo_b200_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int dvo_b200_synchronize(dvo_b200_ctx* ctx) {
  if (!ctx) return DVO_B200_ERR_INVALID_ARGUMENT;
  DVO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return check_level_flags(ctx);   // a timeout inside dvo_b200_match_batch_device surfaces here
}

const char* dvo_b200_last_error(dvo_b200_ctx* ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }

void dvo_b200_config_default(dvo_b200_config* cfg) {
  if (!cfg) return;
  // dense_tracking_config.cpp:27-42
  cfg->first_level = 3; cfg->last_level = 1; cfg->max_iterations_per_level = 100; cfg->use_initial_estimate = 0;
  cfg->precision = 5e-7; cfg->mu = 0.0; cfg->intensity_derivative_threshold = 0.0f; cfg->depth_derivative_threshold = 0.0f;
}

int64_t dvo_b200_kernel_launches(dvo_b200_ctx* ctx) { return ctx ? ctx->launches : 0; }
int64_t dvo_b200_h2d_bytes(dvo_b200_ctx* ctx) { return ctx ? ctx->h2d_bytes : 0; }
int64_t dvo_b200_d2h_bytes(dvo_b200_ctx* ctx) { return ctx ? ctx->d2h_bytes : 0; }

int dvo_b200_pyramid_create_batch(dvo_b200_ctx* ctx, int32_t n, const float* intensity, const float* depth, int32_t width,
                                  int32_t height, float fx, float fy, float ox, float oy, int32_t levels,
                                  dvo_b200_pyramid** out) {
  if (!ctx || !intensity || !depth || !out || n <= 0 || width <= 0 || height <= 0)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid_create: null/invalid argument");
  cudaSetDevice(ctx->device);
  size_t img = (size_t)width * height * sizeof(float);
  int rc = ensure_stage(ctx, 2 * img * n, 0);
  if (rc) return rc;
  float* dI = (float*)ctx->d_stage;
  float* dZ = dI + (size_t)n * width * height;
  DVO_CUDA(ctx, cudaMemcpyAsync(dI, intensity, img * n, cudaMemcpyHostToDevice, ctx->stream));
  DVO_CUDA(ctx, cudaMemcpyAsync(dZ, depth, img * n, cudaMemcpyHostToDevice, ctx->stream));
  ctx->h2d_bytes += 2 * img * n;
  return pyramid_build_batch(ctx, n, dI, dZ, width, height, fx, fy, ox, oy, levels, 0.f, 0.f, out);
}

int dvo_b200_pyramid_create(dvo_b200_ctx* ctx, const float* intensity, const float* depth, int32_t width, int32_t height,
                            float fx, float fy, float ox, float oy, int32_t levels, dvo_b200_pyramid** out) {
  return dvo_b200_pyramid_create_batch(ctx, 1, intensity, depth, width, height, fx, fy, ox, oy, levels, out);
}

int dvo_b200_pyramid_create_raw_batch(dvo_b200_ctx* ctx, int32_t n, const uint8_t* grey, const uint16_t* raw_depth,
                                      float depth_scale, int32_t width, int32_t height, float fx, float fy, float ox,
                                      float oy, int32_t levels, dvo_b200_pyramid** out) {
  if (!ctx || !grey || !raw_depth || !out || n <= 0 || width <= 0 || height <= 0)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid_create_raw: null/invalid argument");
  cudaSetDevice(ctx->device);
  // the frames stay in their file representation (3 bytes per pixel) in the device staging area; the pyramid kernels
  // convert in their loads (no float32 copy of the frame is written, no conversion kernel)
  size_t npx = (size_t)width * height * n;
  const size_t grey_off = (npx * 2 + 255) / 256 * 256;
  int rc = ensure_stage(ctx, grey_off + npx + 64, 0);
  if (rc) return rc;
  uint16_t* dR = (uint16_t*)ctx->d_stage;
  uint8_t* dG = (uint8_t*)((char*)ctx->d_stage + grey_off);
  DVO_CUDA(ctx, cudaMemcpyAsync(dR, raw_depth, npx * 2, cudaMemcpyHostToDevice, ctx->stream));
  DVO_CUDA(ctx, cudaMemcpyAsync(dG, grey, npx, cudaMemcpyHostToDevice, ctx->stream));
  ctx->h2d_bytes += npx * 3;
  return pyramid_build_batch_input(ctx, n, dense_frames(dG, dR, 1, depth_scale, width, height), width, height, fx, fy, ox, oy, levels,
                                   0.f, 0.f, out);
}

int dvo_b200_pyramid_create_bgr_batch(dvo_b200_ctx* ctx, int32_t n, const uint8_t* bgr, const uint16_t* raw_depth,
                                      float depth_scale, int32_t width, int32_t height, float fx, float fy, float ox,
                                      float oy, int32_t levels, dvo_b200_pyramid** out) {
  if (!ctx || !bgr || !raw_depth || !out || n <= 0 || width <= 0 || height <= 0)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid_create_bgr: null/invalid argument");
  cudaSetDevice(ctx->device);
  size_t npx = (size_t)width * height * n;
  const size_t grey_off = (npx * 2 + 255) / 256 * 256, bgr_off = grey_off + (npx + 255) / 256 * 256;
  int rc = ensure_stage(ctx, bgr_off + npx * 3 + 64, 0);
  if (rc) return rc;
  uint16_t* dR = (uint16_t*)ctx->d_stage;
  uint8_t* dG = (uint8_t*)((char*)ctx->d_stage + grey_off);
  uint8_t* dC = (uint8_t*)((char*)ctx->d_stage + bgr_off);
  DVO_CUDA(ctx, cudaMemcpyAsync(dR, raw_depth, npx * 2, cudaMemcpyHostToDevice, ctx->stream));
  DVO_CUDA(ctx, cudaMemcpyAsync(dC, bgr, npx * 3, cudaMemcpyHostToDevice, ctx->stream));
  ctx->h2d_bytes += npx * 5;
  convert_bgr(ctx, dC, (size_t)width * 3, (size_t)width * height * 3, dG, n, width, height);   // 8-bit grey, as cv::cvtColor leaves it
  return pyramid_build_batch_input(ctx, n, dense_frames(dG, dR, 1, depth_scale, width, height), width, height, fx, fy, ox, oy, levels,
                                   0.f, 0.f, out);
}

int dvo_b200_pyramid_create_raw(dvo_b200_ctx* ctx, const uint8_t* grey, const uint16_t* raw_depth, float depth_scale,
                                int32_t width, int32_t height, float fx, float fy, float ox, float oy, int32_t levels,
                                dvo_b200_pyramid** out) {
  return dvo_b200_pyramid_create_raw_batch(ctx, 1, grey, raw_depth, depth_scale, width, height, fx, fy, ox, oy, levels, out);
}

int dvo_b200_pyramid_create_device_batch(dvo_b200_ctx* ctx, int32_t n, const dvo_b200_device_frames* frames, float fx, float fy,
                                         float ox, float oy, int32_t levels, dvo_b200_pyramid** out) {
  if (!ctx || !frames || !out || n <= 0)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid_create_device_batch: null/invalid argument");
  const dvo_b200_device_frames& f = *frames;
  if (f.format < DVO_B200_FRAME_F32 || f.format > DVO_B200_FRAME_BGR8_RAW16)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid_create_device_batch: frames->format " + std::to_string(f.format) + " is unknown");
  if (f.width <= 0 || f.height <= 0)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid_create_device_batch: frames->width / height must be positive");
  cudaSetDevice(ctx->device);
  const bool f32 = f.format == DVO_B200_FRAME_F32;
  const int colour_px = f32 ? 4 : (f.format == DVO_B200_FRAME_GREY8_RAW16 ? 1 : 3), colour_elem = f32 ? 4 : 1;
  const int depth_px = f32 ? 4 : 2;
  int rc = check_plane(ctx, "colour", f.colour, f.colour_row_bytes, f.colour_image_bytes, n, f.width, f.height, colour_px, colour_elem);
  if (!rc) rc = check_plane(ctx, "depth", f.depth, f.depth_row_bytes, f.depth_image_bytes, n, f.width, f.height, depth_px, depth_px);
  if (rc) return rc;
  FrameInput in;
  in.I = f.colour; in.i_row = (size_t)f.colour_row_bytes; in.i_img = n > 1 ? (size_t)f.colour_image_bytes : 0;
  in.Z = f.depth; in.z_row = (size_t)f.depth_row_bytes; in.z_img = n > 1 ? (size_t)f.depth_image_bytes : 0;
  in.raw = f32 ? 0 : 1; in.zscale = f32 ? 0.f : f.depth_scale;
  if (f.format == DVO_B200_FRAME_BGR8_RAW16) {
    // grey into the staging area, as the host path leaves it; then the raw path reads it dense
    const size_t npx = (size_t)f.width * f.height * n;
    if ((rc = ensure_stage(ctx, npx + 64, 0))) return rc;
    uint8_t* dG = (uint8_t*)ctx->d_stage;
    convert_bgr(ctx, (const uint8_t*)f.colour, in.i_row, in.i_img, dG, n, f.width, f.height);
    in.I = dG; in.i_row = (size_t)f.width; in.i_img = (size_t)f.width * f.height;
  }
  return pyramid_build_batch_input(ctx, n, in, f.width, f.height, fx, fy, ox, oy, levels, 0.f, 0.f, out);
}

int dvo_b200_pyramid_device(const dvo_b200_pyramid* p) { return p ? p->device : -1; }

int dvo_b200_pyramid_retain(dvo_b200_pyramid* p) {
  if (!p) return DVO_B200_ERR_INVALID_ARGUMENT;
  p->refcount.fetch_add(1, std::memory_order_relaxed);
  return 0;
}

int dvo_b200_pyramid_release(dvo_b200_pyramid* p) {
  if (!p) return DVO_B200_ERR_INVALID_ARGUMENT;
  if (p->refcount.fetch_sub(1, std::memory_order_acq_rel) == 1) {
    // No synchronisation: the slab returns to the owning ctx's pool and is only ever rewritten by
    // work enqueued later on that ctx's stream (stream order protects queued readers).  A second
    // ctx that uses this pyramid holds a reference until its (blocking) match call has returned.
    pyramid_free(p);
  }
  return 0;
}

int dvo_b200_pyramid_num_levels(const dvo_b200_pyramid* p) { return p ? p->levels : DVO_B200_ERR_INVALID_ARGUMENT; }

int dvo_b200_pyramid_level_info(const dvo_b200_pyramid* p, int32_t level, int32_t* width, int32_t* height, float K[4]) {
  if (!p || level < 0 || level >= p->levels) return DVO_B200_ERR_INVALID_ARGUMENT;
  const LevelInfo& L = p->L[level];
  if (width) *width = L.w;
  if (height) *height = L.h;
  if (K) { K[0] = L.fx; K[1] = L.fy; K[2] = L.ox; K[3] = L.oy; }
  return 0;
}

int dvo_b200_pyramid_download(dvo_b200_ctx* ctx, const dvo_b200_pyramid* p, int32_t level, float* planes6) {
  if (!p || !planes6 || level < 0 || level >= p->levels)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid_download: invalid argument");
  cudaSetDevice(ctx ? ctx->device : (p->slab && p->slab->pool ? p->slab->pool->device : 0));
  const LevelInfo& L = p->L[level];
  size_t N = L.n;
  const size_t plane = (size_t)L.pitch * L.h;      // float2 elements per plane, rows padded to the pitch
  const size_t nrec = (size_t)L.nbands * L.nstrips * dvo_b200::kRecF2;
  std::vector<float> tmp(4 * plane), rec(2 * nrec);
  if (ctx) DVO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (p->slab && p->slab->ready) DVO_CUDA(ctx, cudaEventSynchronize(p->slab->ready));   // the pyramid's own build has finished
  DVO_CUDA(ctx, cudaMemcpy(tmp.data(), p->planes + L.plane_off, sizeof(float) * 4 * plane, cudaMemcpyDeviceToHost));
  DVO_CUDA(ctx, cudaMemcpy(rec.data(), p->planes + L.rec_off, sizeof(float) * 2 * nrec, cudaMemcpyDeviceToHost));
  if (ctx) ctx->d2h_bytes += sizeof(float) * (4 * plane + 2 * nrec);
  // device layout: P0 = (I, Z'), P2 = (I, Z) row-major; (Ix, Iy) in the reference tile records.  The depth gradients are not
  // stored (the tracker forms them from P2 on the fly): restate calculateDerivativeX/Y<float> on the true depth
  // (rgbd_image.cpp:419-472).
  auto Zt = [&](int y, int x) { return tmp[2 * plane + 2 * ((size_t)y * L.pitch + x) + 1]; };
  for (int y = 0; y < L.h; ++y)
    for (int x = 0; x < L.w; ++x) {
      const size_t o = 2 * ((size_t)y * L.pitch + x), i = (size_t)y * L.w + x;
      const size_t g = 2 * (dvo_b200::rec_cell(x, y, L.nbands) + dvo_b200::kRecP1);
      planes6[0 * N + i] = tmp[o]; planes6[1 * N + i] = tmp[o + 1];
      planes6[2 * N + i] = rec[g]; planes6[3 * N + i] = rec[g + 1];
      const int xp = x > 0 ? x - 1 : 0, xn = x < L.w - 1 ? x + 1 : L.w - 1, yp = y > 0 ? y - 1 : 0, yn = y < L.h - 1 ? y + 1 : L.h - 1;
      const float dzx = Zt(y, xn) - Zt(y, xp), dzy = Zt(yn, x) - Zt(yp, x);
      planes6[4 * N + i] = dzx * 0.5f; planes6[5 * N + i] = dzy * 0.5f;
    }
  return 0;
}

int dvo_b200_pyramid_select(dvo_b200_ctx* ctx, dvo_b200_pyramid* p, int32_t level, float intensity_threshold,
                            float depth_threshold, int64_t* count, uint8_t* mask) {
  if (!ctx || !p || level < 0 || level >= p->levels)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid_select: invalid argument");
  cudaSetDevice(ctx->device);
  int rc = pyramid_reselect(ctx, p, intensity_threshold, depth_threshold);
  if (rc) return rc;
  const LevelInfo& L = p->L[level];
  DVO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  int info[2];
  DVO_CUDA(ctx, cudaMemcpy(info, p->sel_info + 2 * level, sizeof(info), cudaMemcpyDeviceToHost));
  if (count) *count = info[0];
  if (mask) {
    std::vector<uint32_t> words(L.words);
    DVO_CUDA(ctx, cudaMemcpy(words.data(), p->sel_mask + L.mask_off, sizeof(uint32_t) * L.words, cudaMemcpyDeviceToHost));
    for (int i = 0; i < L.n; ++i) mask[i] = (words[i >> 5] >> (i & 31)) & 1u;
  }
  return 0;
}

int dvo_b200_match_batch(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n, dvo_b200_pyramid* const* references,
                         dvo_b200_pyramid* const* currents, const double* T_init, dvo_b200_result* results,
                         dvo_b200_iteration_stats* iteration_stats, int32_t max_iteration_stats) {
  if (!ctx || !results) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match_batch: null argument");
  cudaSetDevice(ctx->device);
  return tracker_match_batch(ctx, cfg, n, references, currents, T_init, results, nullptr, iteration_stats,
                             iteration_stats ? max_iteration_stats : 0);
}

int dvo_b200_match(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* reference, dvo_b200_pyramid* current,
                   const double* T_init, dvo_b200_result* result) {
  dvo_b200_pyramid* r[1] = {reference};
  dvo_b200_pyramid* c[1] = {current};
  return dvo_b200_match_batch(ctx, cfg, 1, r, c, T_init, result, nullptr, 0);
}

int dvo_b200_match_batch_device(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n,
                                dvo_b200_pyramid* const* references, dvo_b200_pyramid* const* currents,
                                const double* T_init, void* d_results) {
  if (!ctx || !d_results) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match_batch_device: null argument");
  cudaSetDevice(ctx->device);
  return tracker_match_batch(ctx, cfg, n, references, currents, T_init, nullptr, d_results, nullptr, 0);
}

int dvo_b200_match_batch_enqueue(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n, dvo_b200_pyramid* const* references,
                                 dvo_b200_pyramid* const* currents, const double* d_T_init, void* d_results) {
  if (!ctx || !d_results) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match_batch_enqueue: null argument");
  cudaSetDevice(ctx->device);
  int rc = check_enqueue_buffers(ctx, cfg, d_T_init, d_results, "match_batch_enqueue");
  if (rc) return rc;
  return tracker_match_batch(ctx, cfg, n, references, currents, d_T_init, nullptr, d_results, nullptr, 0, true);
}

int dvo_b200_selection_create(dvo_b200_ctx* ctx, dvo_b200_pyramid* p, int32_t predicate, float ti, float td,
                              const uint8_t* const* level_masks, dvo_b200_selection** out) {
  if (!ctx || !p || !out) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "selection_create: null argument");
  if (predicate < DVO_B200_PREDICATE_GRADIENT_THRESHOLD || predicate > DVO_B200_PREDICATE_MASK_ONLY)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "selection_create: predicate " + std::to_string(predicate) + " is unknown");
  if (p->device != ctx->device) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "selection_create: pyramid lives on another device");
  cudaSetDevice(ctx->device);
  SelMaskInput mi;
  if (level_masks)
    for (int l = 0; l < p->levels; ++l) mi.per_level[l] = level_masks[l];
  dvo_b200_pyramid* pyrs[1] = {p};
  return selection_build_batch(ctx, 1, pyrs, predicate, ti, td, mi, out);
}

int dvo_b200_selection_create_device_batch(dvo_b200_ctx* ctx, int32_t n, dvo_b200_pyramid* const* pyramids, int32_t predicate,
                                           float ti, float td, const void* d_masks, int64_t row_bytes, int64_t image_bytes,
                                           dvo_b200_selection** out) {
  const char* f = "selection_create_device_batch: ";
  if (!ctx || !pyramids || !out || n <= 0) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, std::string(f) + "null/invalid argument");
  if (predicate < DVO_B200_PREDICATE_GRADIENT_THRESHOLD || predicate > DVO_B200_PREDICATE_MASK_ONLY)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + std::string("predicate ") + std::to_string(predicate) + " is unknown");
  for (int i = 0; i < n; ++i) {
    const dvo_b200_pyramid* p = pyramids[i];
    if (!p) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, std::string(f) + "null pyramid");
    if (p->device != ctx->device) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, std::string(f) + "pyramid lives on another device");
    if (p->levels != pyramids[0]->levels || p->L[0].w != pyramids[0]->L[0].w || p->L[0].h != pyramids[0]->L[0].h)
      return set_error(ctx, DVO_B200_ERR_SHAPE_MISMATCH, std::string(f) + "all pyramids must share width, height and levels");
  }
  cudaSetDevice(ctx->device);
  SelMaskInput mi;
  if (d_masks) {
    const int w = pyramids[0]->L[0].w, h = pyramids[0]->L[0].h;
    if (row_bytes < w)
      return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + std::string("row_bytes ") + std::to_string(row_bytes) + " < width");
    if (n > 1 && image_bytes < (int64_t)h * row_bytes)
      return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, f + std::string("image_bytes ") + std::to_string(image_bytes) + " < height x row_bytes");
    int rc = check_device_pointer(ctx, d_masks, std::string(f) + "d_masks");
    if (rc) return rc;
    mi.level0 = (const uint8_t*)d_masks; mi.row = (size_t)row_bytes; mi.img = n > 1 ? (size_t)image_bytes : 0;
  }
  return selection_build_batch(ctx, n, pyramids, predicate, ti, td, mi, out);
}

int dvo_b200_selection_retain(dvo_b200_selection* s) {
  if (!s) return DVO_B200_ERR_INVALID_ARGUMENT;
  s->refcount.fetch_add(1, std::memory_order_relaxed);
  return 0;
}

int dvo_b200_selection_release(dvo_b200_selection* s) {
  if (!s) return DVO_B200_ERR_INVALID_ARGUMENT;
  // as dvo_b200_pyramid_release: the slab returns to the building ctx's pool and is rewritten only by work enqueued later
  // on that ctx's stream
  if (s->refcount.fetch_sub(1, std::memory_order_acq_rel) == 1) selection_free(s);
  return 0;
}

dvo_b200_pyramid* dvo_b200_selection_pyramid(dvo_b200_selection* s) { return s ? s->pyr : nullptr; }

int dvo_b200_selection_download(dvo_b200_ctx* ctx, const dvo_b200_selection* s, int32_t level, int64_t* count, uint8_t* mask) {
  if (!s || level < 0 || level >= s->pyr->levels) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "selection_download: invalid argument");
  cudaSetDevice(s->device);
  const LevelInfo& L = s->pyr->L[level];
  if (ctx) DVO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (s->slab && s->slab->ready) DVO_CUDA(ctx, cudaEventSynchronize(s->slab->ready));   // the selection's build has finished
  int info[2];
  DVO_CUDA(ctx, cudaMemcpy(info, s->sel_info + 2 * level, sizeof(info), cudaMemcpyDeviceToHost));
  if (count) *count = info[0];
  if (mask) {
    std::vector<uint32_t> words(L.words);
    DVO_CUDA(ctx, cudaMemcpy(words.data(), s->mask + L.mask_off, sizeof(uint32_t) * L.words, cudaMemcpyDeviceToHost));
    for (int i = 0; i < L.n; ++i) mask[i] = (words[i >> 5] >> (i & 31)) & 1u;
  }
  if (ctx) ctx->d2h_bytes += sizeof(info) + (mask ? sizeof(uint32_t) * L.words : 0);
  return 0;
}

}  // extern "C"

// the pyramids of n selections, for the shared match path
static int selection_refs(dvo_b200_ctx* ctx, int n, dvo_b200_selection* const* sels, std::vector<dvo_b200_pyramid*>& refs) {
  if (!sels || n <= 0) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match_batch_selected: null argument");
  refs.resize(n);
  for (int i = 0; i < n; ++i) {
    if (!sels[i]) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match_batch_selected: null selection");
    refs[i] = sels[i]->pyr;
  }
  return 0;
}

extern "C" {

int dvo_b200_match_batch_selected(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n, dvo_b200_selection* const* references,
                                  dvo_b200_pyramid* const* currents, const double* T_init, dvo_b200_result* results,
                                  dvo_b200_iteration_stats* iteration_stats, int32_t max_iteration_stats) {
  if (!ctx || !results) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match_batch_selected: null argument");
  cudaSetDevice(ctx->device);
  std::vector<dvo_b200_pyramid*> refs;
  int rc = selection_refs(ctx, n, references, refs);
  if (rc) return rc;
  return tracker_match_batch(ctx, cfg, n, refs.data(), currents, T_init, results, nullptr, iteration_stats,
                             iteration_stats ? max_iteration_stats : 0, false, references);
}

int dvo_b200_match_batch_selected_enqueue(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int32_t n, dvo_b200_selection* const* references,
                                          dvo_b200_pyramid* const* currents, const double* d_T_init, void* d_results) {
  if (!ctx || !d_results) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match_batch_selected_enqueue: null argument");
  cudaSetDevice(ctx->device);
  int rc = check_enqueue_buffers(ctx, cfg, d_T_init, d_results, "match_batch_selected_enqueue");
  if (rc) return rc;
  std::vector<dvo_b200_pyramid*> refs;
  if ((rc = selection_refs(ctx, n, references, refs))) return rc;
  return tracker_match_batch(ctx, cfg, n, refs.data(), currents, d_T_init, nullptr, d_results, nullptr, 0, true, references);
}

int dvo_b200_residual_image(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* reference,
                            dvo_b200_pyramid* current, int32_t level, const double* T, float* planes7, int64_t* count) {
  if (!ctx || !cfg || !planes7) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "residual_image: null argument");
  cudaSetDevice(ctx->device);
  return tracker_linearize(ctx, cfg, reference, current, level, T, 0, nullptr, count, nullptr, nullptr, nullptr, nullptr, planes7);
}

int dvo_b200_intensity_error_image(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* reference,
                                   dvo_b200_pyramid* current, int32_t level, const double* T, float* image, int64_t* count) {
  if (!ctx || !cfg || !image || !reference || !current) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "intensity_error_image: null argument");
  if (level < 0 || level >= reference->levels) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "intensity_error_image: level out of range");
  const size_t n = size_t(reference->L[level].w) * reference->L[level].h;
  std::vector<float> planes(7 * n);
  int64_t valid = 0;
  int rc = dvo_b200_residual_image(ctx, cfg, reference, current, level, T, planes.data(), &valid);
  if (rc != 0) return rc;
  // the residual stage leaves NaN at pixels that are unselected, dropped (odd last point) or invalid after the warp:
  // exactly the pixels the reference's raster walk leaves at the zero initialisation (dense_tracking.cpp:415-439)
  for (size_t i = 0; i < n; ++i) image[i] = planes[i] == planes[i] ? fabsf(planes[i]) : 0.0f;
  if (count) *count = valid;
  return 0;
}

int dvo_b200_linearize(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* reference, dvo_b200_pyramid* current,
                       int32_t level, const double* T, int32_t use_weights, const float* prev_precision, int64_t* count,
                       float* precision_out, float* ll_out, double* A_out, double* b_out) {
  if (!ctx || !cfg) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "linearize: null argument");
  cudaSetDevice(ctx->device);
  return tracker_linearize(ctx, cfg, reference, current, level, T, use_weights, prev_precision, count, precision_out, ll_out,
                           A_out, b_out, nullptr);
}

int dvo_b200_profile_enable(dvo_b200_ctx* ctx, int32_t enable) {
  if (!ctx) return DVO_B200_ERR_INVALID_ARGUMENT;
  ctx->profile = enable != 0;
  return 0;
}

int dvo_b200_profile_read(dvo_b200_ctx* ctx, double ms_out[8], int64_t launches_out[8], int32_t reset) {
  if (!ctx) return DVO_B200_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  drain_profile(ctx);
  if (ctx->d_dbg) {   // developer timing dump (DVO_B200_TIMING=1)
    unsigned long long h[256];
    cudaStreamSynchronize(ctx->stream);
    cudaMemcpy(h, ctx->d_dbg, sizeof(h), cudaMemcpyDeviceToHost);
    static const char* names[8] = {"stageA", "stageB", "waitA", "waitB", "mid", "end", "queue", "total"};
    for (int l = 0; l < 8; ++l) {
      const unsigned long long* v = h + 16 * l;
      if (!v[7]) continue;
      fprintf(stderr, "[dvo_b200 timing] level-slot %d:", l);
      for (int i = 0; i < 8; ++i) fprintf(stderr, " %s=%.1f%%", names[i], 100.0 * (double)v[i] / (double)v[7]);
      fprintf(stderr, " (cta-ms total %.1f)\n", (double)v[7] * 1e-6);
      fprintf(stderr, "[dvo_b200 timing]   consumer warp 0: wait-full %.1f%% of stage A, %.1f%% of stage B; producer: descriptor %.1f%%, "
                      "wait-empty %.1f%% of its stage time\n", 100.0 * (double)v[9] / (double)(v[8] + 1), 100.0 * (double)v[11] / (double)(v[10] + 1),
              100.0 * (double)v[12] / (double)(v[14] + v[15] + 1), 100.0 * (double)v[13] / (double)(v[14] + v[15] + 1));
      const unsigned long long* u = h + 128 + 8 * l;
      if (u[0]) fprintf(stderr, "[dvo_b200 timing]   tiles %llu (inexact %.2f%%, skipped %.2f%%), stage-B rounds of inexact tiles %.2f%%; CTA lifetime of the last launch-set: "
                                "max %.3f ms, min %.3f ms\n", u[0], 100.0 * (double)u[1] / (double)u[0], 100.0 * (double)u[2] / (double)u[0],
                        100.0 * (double)u[4] / (double)(u[3] + 1), (double)u[5] * 1e-6, (double)u[6] * 1e-6);
      const unsigned long long* e = h + 192 + 8 * l;   // e[7]: critical ns; e[0..5]: sub-phases
      if (e[7]) {
        double tot = 0;
        for (int i = 0; i < 6; ++i) tot += (double)e[i];
        fprintf(stderr, "[dvo_b200 timing]   end step: critical part %.1f%% of the end time; of the end thread's time: partial sums %.1f%%, state+log %.1f%%, "
                        "LDLT %.1f%%, exp+K*T %.1f%%, release %.1f%%, deferred %.1f%% (total %.1f cta-ms)\n", 100.0 * (double)e[7] / (double)(v[5] + 1),
                100.0 * e[0] / tot, 100.0 * e[1] / tot, 100.0 * e[2] / tot, 100.0 * e[3] / tot, 100.0 * e[4] / tot, 100.0 * e[5] / tot, tot * 1e-6);
      }
    }
    if (reset) {
      cudaMemset(ctx->d_dbg, 0, sizeof(h));
      for (int l = 0; l < 8; ++l) { unsigned long long big = ~0ull; cudaMemcpy(ctx->d_dbg + 128 + 8 * l + 6, &big, 8, cudaMemcpyHostToDevice); }
    }
  }
  if (getenv("DVO_B200_TIMING")) {   // developer: device time of the level kernels, per level of the match (coarse -> fine)
    fprintf(stderr, "[dvo_b200 timing] level kernels, ms per launch:");
    for (int i = 8; i < 16; ++i)
      if (ctx->prof_launches[i]) fprintf(stderr, " %.3f", ctx->prof_ms[i] / (double)ctx->prof_launches[i]);
    fprintf(stderr, "\n");
  }
  for (int i = 0; i < 16; ++i) {
    if (i < 8 && ms_out) ms_out[i] = ctx->prof_ms[i];
    if (i < 8 && launches_out) launches_out[i] = ctx->prof_launches[i];
    if (reset) { ctx->prof_ms[i] = 0; ctx->prof_launches[i] = 0; }
  }
  return 0;
}

}  // extern "C"
