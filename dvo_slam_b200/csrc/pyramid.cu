// pyramid.cu -- device image pyramid: replaces RgbdImagePyramid::build (rgbd_image.cpp:156-172),
// pyrDownMeanSmooth / pyrDownSubsample (rgbd_image.cpp:38-55,127-139), RgbdCameraPyramid::build
// (rgbd_image.cpp:283-296), calculateDerivativeX/Y (rgbd_image.cpp:419-472, rgbd_image_sse.cpp:241-284),
// the RgbdCamera point-cloud template (rgbd_image.cpp:186-204) and PointSelection::select with the
// default predicate (point_selection.cpp:89-152, point_selection.h:63-66).
#include "common.cuh"

#include <algorithm>
#include <cstdio>
#include <cstring>

namespace dvo_b200 {

namespace {

__device__ __forceinline__ bool is_nan(float v) { return v != v; }

// Level-0 pixels as they were uploaded.  kRaw = false: float32 intensity and float32 depth in metres (NaN = invalid), what
// benchmark_slam.cpp:46-93 hands to RgbdCameraPyramid::create.  kRaw = true: 8-bit grey and 16-bit raw depth straight from
// the image files; the loader's conversions -- convertTo(CV_32F) and SurfacePyramid::convertRawDepthImageSse
// (surface_pyramid.cpp:65-105: u16 * scale, 0 -> NaN) -- happen in the load, no float32 copy of the frame is ever written.
// The input images are addressed in bytes (FrameInput: row and image strides), so a pitched or sliced frame is read in
// place; `off` is the byte offset of the pixel from `base`.
template <bool kRaw>
__device__ __forceinline__ float load_intensity(const char* base, size_t off) {
  if (kRaw) return (float)__ldg(reinterpret_cast<const uint8_t*>(base + off));
  return __ldg(reinterpret_cast<const float*>(base + off));
}
template <bool kRaw>
__device__ __forceinline__ float load_depth(const char* base, size_t off, float scale) {
  if (kRaw) {
    const uint16_t r = __ldg(reinterpret_cast<const uint16_t*>(base + off));
    return r == 0 ? __int_as_float(0x7fc00000) : __fmul_rn((float)r, scale);
  }
  return __ldg(reinterpret_cast<const float*>(base + off));
}
template <bool kRaw> constexpr int intensity_bytes() { return kRaw ? 1 : 4; }
template <bool kRaw> constexpr int depth_bytes() { return kRaw ? 2 : 4; }

// level l intensity = ((a+b)+c)+d)/4 of the 2x2 block of level l-1 (rgbd_image.cpp:38-55), into P0.x (the Z slot is
// filled by the finish pass).  kFromInput: level 1 reads the input image, which is level 0's intensity, at byte strides
// in_row / in_img.  sp / dp: row pitch of the source / destination planes (float2 elements).
template <bool kFromInput, bool kRaw>
__global__ void k_pyr_intensity_down(const void* __restrict__ I0, size_t in_row, size_t in_img, int aligned, float2* __restrict__ planes,
                                     size_t planes_per_image, size_t src_off, int sp, size_t dst_off, int dw, int dh, int dp) {
  int img = blockIdx.y;
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= dw * dh) return;
  int y = idx / dw, x = idx - y * dw;
  float2* D = planes + img * planes_per_image + dst_off;
  float a, b, c, d;
  if (kFromInput) {
    const char* r0 = reinterpret_cast<const char*>(I0) + img * in_img + (size_t)(2 * y) * in_row + (size_t)(2 * x) * intensity_bytes<kRaw>();
    const char* r1 = r0 + in_row;
    if (kRaw) {
      if (aligned) {   // base, row and image strides even: every 2x2 block starts 2-byte aligned
        const uchar2 u = __ldg(reinterpret_cast<const uchar2*>(r0)), v = __ldg(reinterpret_cast<const uchar2*>(r1));
        a = (float)u.x; b = (float)u.y; c = (float)v.x; d = (float)v.y;
      } else {
        a = load_intensity<true>(r0, 0); b = load_intensity<true>(r0, 1); c = load_intensity<true>(r1, 0); d = load_intensity<true>(r1, 1);
      }
    } else {
      if (aligned) {   // base, row and image strides multiples of 8 bytes: every 2x2 block starts 8-byte aligned
        const float2 u = __ldg(reinterpret_cast<const float2*>(r0)), v = __ldg(reinterpret_cast<const float2*>(r1));
        a = u.x; b = u.y; c = v.x; d = v.y;
      } else {
        a = load_intensity<false>(r0, 0); b = load_intensity<false>(r0, 4); c = load_intensity<false>(r1, 0); d = load_intensity<false>(r1, 4);
      }
    }
  } else {
    const float2* S = planes + img * planes_per_image + src_off;
    const float2* r0 = S + (size_t)(2 * y) * sp + 2 * x;
    const float2* r1 = r0 + sp;
    a = r0[0].x; b = r0[1].x; c = r1[0].x; d = r1[1].x;
  }
  float s = __fadd_rn(a, b);
  s = __fadd_rn(s, c);
  s = __fadd_rn(s, d);
  D[(size_t)y * dp + x] = make_float2(s * 0.25f, 0.f);
}

// gradients (clamped central differences), masked and true depth, default selection mask and reference plane
// (I, Zsel: depth where the pixel is selected, NaN elsewhere) for one level.
// Depth of level l is the pure subsample chain of level 0 (rgbd_image.cpp:127-139): Z_l(y,x) = Z_0(y<<l, x<<l).
// Level 0 reads its intensity straight from the input image (no intermediate copy); the other levels read the
// intensity that k_pyr_intensity_down left in P0.x.  Input taps are addressed with the byte strides of `src`.  The
// selection count / last selected index are derived from the masks afterwards (k_sel_info): no atomics here.  Threads walk the linear pixel index y*w+x (the order of the
// selection mask); the planes are addressed with the row pitch.
template <bool kLevel0, bool kRaw>
__global__ void __launch_bounds__(256)
k_pyr_finish(const FrameInput src, float2* __restrict__ planes,
             size_t planes_per_image, size_t plane_off, size_t rec_off, int nbands, int w, int h, int pitch, int level,
             uint32_t* __restrict__ masks, size_t mask_words_per_image, size_t mask_off, float ti, float td) {
  const int img = blockIdx.y;
  const int n = w * h;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = idx < n;
  bool sel = false;
  if (in) {
    const int y = idx / w, x = idx - y * w;
    const size_t plane = (size_t)pitch * h;
    float2* P0 = planes + img * planes_per_image + plane_off;
    float2* P2 = P0 + plane;   // P2 = (I, Z); the depth gradients are not stored
    float2* rec = planes + img * planes_per_image + rec_off;   // reference tile records: (I, Zsel) and (Ix, Iy)
    const char* Ib = reinterpret_cast<const char*>(src.I) + img * src.i_img;
    const char* Zb = reinterpret_cast<const char*>(src.Z) + img * src.z_img;
    const int xp = max(x - 1, 0), xn = min(x + 1, w - 1), yp = max(y - 1, 0), yn = min(y + 1, h - 1);
    float I, ixp, ixn, iyp, iyn;
    if (kLevel0) {
      constexpr int E = intensity_bytes<kRaw>();
      const char* row = Ib + (size_t)y * src.i_row;
      I = load_intensity<kRaw>(row, (size_t)x * E); ixp = load_intensity<kRaw>(row, (size_t)xp * E); ixn = load_intensity<kRaw>(row, (size_t)xn * E);
      iyp = load_intensity<kRaw>(Ib + (size_t)yp * src.i_row, (size_t)x * E); iyn = load_intensity<kRaw>(Ib + (size_t)yn * src.i_row, (size_t)x * E);
    } else {
      const size_t row = (size_t)y * pitch;
      I = P0[row + x].x; ixp = P0[row + xp].x; ixn = P0[row + xn].x;
      iyp = P0[(size_t)yp * pitch + x].x; iyn = P0[(size_t)yn * pitch + x].x;
    }
    const float ix = (ixn - ixp) * 0.5f;
    const float iy = (iyn - iyp) * 0.5f;
    constexpr int EZ = depth_bytes<kRaw>();
    const float zscale = src.zscale;
    const char* zr = Zb + (size_t)(y << level) * src.z_row;
    const size_t zc = (size_t)(x << level) * EZ;
    const float z = load_depth<kRaw>(zr, zc, zscale);
    const float zx = (load_depth<kRaw>(zr, (size_t)(xn << level) * EZ, zscale) - load_depth<kRaw>(zr, (size_t)(xp << level) * EZ, zscale)) * 0.5f;
    const float zy = (load_depth<kRaw>(Zb + (size_t)(yn << level) * src.z_row, zc, zscale) -
                      load_depth<kRaw>(Zb + (size_t)(yp << level) * src.z_row, zc, zscale)) * 0.5f;
    const bool bad = is_nan(I) || is_nan(ix) || is_nan(iy) || is_nan(z) || is_nan(zx) || is_nan(zy);
    const float zm = bad ? __int_as_float(0x7fc00000) : z;
    const size_t o = (size_t)y * pitch + x;
    // ValidPointAndGradientThresholdPredicate::isPointOk (point_selection.h:63-66)
    sel = !bad && (fabsf(ix) > ti || fabsf(iy) > ti || fabsf(zx) > td || fabsf(zy) > td);
    const float nanv = __int_as_float(0x7fc00000);
    const size_t rc = rec_cell(x, y, nbands);
    P0[o] = make_float2(I, zm);
    P2[o] = make_float2(I, z);
    rec[rc] = make_float2(I, sel ? z : nanv);
    rec[rc + kRecP1] = make_float2(ix, iy);
    if (x == w - 1 && pitch > w) {   // the pad column of an odd width: never a valid tap
      P0[o + 1] = make_float2(0.f, nanv);
      P2[o + 1] = make_float2(0.f, nanv);
    }
  }
  const unsigned m = __ballot_sync(0xffffffffu, sel);
  if ((threadIdx.x & 31) == 0 && idx < ((n + 31) / 32) * 32) masks[img * mask_words_per_image + mask_off + (idx >> 5)] = m;
}

// The parts of the reference tile records that no pixel owns: the tx[] slice of every tile and, in border tiles, the cells
// outside the image (never selected).  One thread per tile column; runs after k_template.
__global__ void k_rec_fill(float2* __restrict__ planes, size_t planes_per_image, size_t rec_off, int nbands, int ntiles, int w, int h,
                           const float* __restrict__ tmpl, size_t tmpl_per_image, size_t tmpl_off) {
  const int img = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ntiles * kTileW) return;
  const int tile = t / kTileW, cx = t - tile * kTileW;
  const int s = tile / nbands, b = tile - s * nbands;
  const int x = b * kTileW + cx, y0 = s * kTileH;
  float2* rec = planes + img * planes_per_image + rec_off + (size_t)tile * kRecF2;
  reinterpret_cast<float*>(rec + kRecTx)[cx] = x < w ? tmpl[img * tmpl_per_image + tmpl_off + x] : 0.f;
  const int r0 = x >= w ? 0 : min(max(h - y0, 0), kTileH);      // first row of this column that lies outside the image
  for (int r = r0; r < kTileH; ++r) {
    rec[r * kTileW + cx] = make_float2(0.f, __int_as_float(0x7fc00000));
    rec[kRecP1 + r * kTileW + cx] = make_float2(0.f, 0.f);
  }
}

// {min, max} of the non-NaN Z' of every tile of kTileW x kTileH pixels (one warp per tile).  The level kernel
// projects the tile's corner rays at both depths to bound the window of the current image its taps fall into.
__global__ void k_tile_range(const float2* __restrict__ planes, size_t planes_per_image, size_t plane_off, int w, int h,
                             int pitch, int nbands, int ntiles, float2* __restrict__ ranges, size_t ranges_per_image,
                             size_t range_off) {
  const int img = blockIdx.y;
  const int tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (tile >= ntiles) return;
  const int lane = threadIdx.x & 31;
  const int s = tile / nbands, b = tile - s * nbands;
  const float2* P0 = planes + img * planes_per_image + plane_off;
  float lo = 3.0e38f, hi = -3.0e38f;
  const int x0 = b * kTileW, x1 = min(x0 + kTileW, w), y0 = s * kTileH, y1 = min(y0 + kTileH, h);
  for (int y = y0; y < y1; ++y)
    for (int x = x0 + lane; x < x1; x += 32) {
      const float z = P0[(size_t)y * pitch + x].y;
      if (z == z) { lo = fminf(lo, z); hi = fmaxf(hi, z); }
    }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, off));
    hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, off));
  }
  if (lane == 0) ranges[img * ranges_per_image + range_off + tile] = make_float2(lo, hi);
}

// {S, last selected linear index} of one (image, level) from its selection mask: one warp each
__global__ void k_sel_info(const uint32_t* __restrict__ masks, size_t mask_words_per_image, size_t mask_off, int words,
                           int* __restrict__ sel_info, int sel_info_per_image, int level) {
  const int img = blockIdx.x, lane = threadIdx.x;
  const uint32_t* m = masks + img * mask_words_per_image + mask_off;
  int cnt = 0, last = -1;
  for (int i = lane; i < words; i += 32) {
    const uint32_t v = m[i];
    cnt += __popc(v);
    if (v) last = i * 32 + 31 - __clz(v);     // i increases: the lane's last non-empty word wins
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    last = max(last, __shfl_xor_sync(0xffffffffu, last, off));
  }
  if (lane == 0) {
    sel_info[img * sel_info_per_image + 2 * level] = cnt;
    sel_info[img * sel_info_per_image + 2 * level + 1] = last;
  }
}

// computeResidualsSse walks the point list two at a time and skips the last point of an odd list
// (dense_tracking_impl.cpp:169): that point is unselected in the reference plane.  Runs after k_sel_info.
__global__ void k_drop_odd_last(float2* __restrict__ planes, size_t planes_per_image, size_t rec_off, int nbands, int w,
                                const int* __restrict__ sel_info, int sel_info_per_image, int level, int nimg) {
  const int img = blockIdx.x * blockDim.x + threadIdx.x;
  if (img >= nimg) return;
  const int S = sel_info[img * sel_info_per_image + 2 * level], last = sel_info[img * sel_info_per_image + 2 * level + 1];
  if ((S & 1) && last >= 0) {
    const int y = last / w, x = last - y * w;
    float2* rec = planes + img * planes_per_image + rec_off;
    rec[rec_cell(x, y, nbands)].y = __int_as_float(0x7fc00000);
  }
}

// recompute the selection mask and the reference plane of one level for non-default thresholds
__global__ void k_reselect(const float2* __restrict__ P0, float2* __restrict__ rec, int nbands, int w, int h, int pitch,
                           uint32_t* __restrict__ mask, float ti, float td) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = w * h;
  bool sel = false;
  if (idx < n) {
    const int y = idx / w, x = idx - y * w;
    const size_t plane = (size_t)pitch * h, o = (size_t)y * pitch + x;
    const float2* P2 = P0 + plane;
    const size_t rc = rec_cell(x, y, nbands);
    const int xp = max(x - 1, 0), xn = min(x + 1, w - 1), yp = max(y - 1, 0), yn = min(y + 1, h - 1);
    const float2 a = P0[o], b = rec[rc + kRecP1];
    const float zx = (P2[(size_t)y * pitch + xn].y - P2[(size_t)y * pitch + xp].y) * 0.5f;
    const float zy = (P2[(size_t)yn * pitch + x].y - P2[(size_t)yp * pitch + x].y) * 0.5f;
    sel = !is_nan(a.y) && (fabsf(b.x) > ti || fabsf(b.y) > ti || fabsf(zx) > td || fabsf(zy) > td);
    rec[rc] = make_float2(a.x, sel ? a.y : __int_as_float(0x7fc00000));
  }
  unsigned m = __ballot_sync(0xffffffffu, sel);
  if ((threadIdx.x & 31) == 0 && idx < ((n + 31) / 32) * 32) mask[idx >> 5] = m;
}

// One level of n point selections (blockIdx.y = selection), each over its own pyramid (src[img]: that pyramid's planes).
// Per pixel: the predicate from the pyramid's P0 / P2 planes and the gradient rows of its records, AND the mask, then the
// (I, Zsel) cell (Zsel = Z' where selected, NaN elsewhere, as k_reselect writes it), the gradient cell and the mask word
// (ballot).  Threads below ntiles x kTileW also copy one tile column of what no pixel owns: the tx slice and the cells
// outside the image.  The mask, if any, is read at m[img * m_img + (y << m_shift) * m_row + (x << m_shift)], nonzero =
// allowed: m_shift = level subsamples a level-0 mask like the depth chain, m_shift = 0 reads a mask of this level.
__global__ void __launch_bounds__(256)
k_sel_build(const float2* const* __restrict__ src, size_t plane_off, size_t src_rec_off, int nbands, int ntiles, int w, int h,
            int pitch, const uint8_t* __restrict__ m, size_t m_row, size_t m_img, int m_shift, float2* __restrict__ rec,
            size_t rec_per_image, size_t rec_off, uint32_t* __restrict__ masks, size_t mask_words_per_image, size_t mask_off,
            int words, int predicate, float ti, float td) {
  const int img = blockIdx.y;
  const int n = w * h;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const float2* P0 = src[img] + plane_off;
  const float2* srec = src[img] + src_rec_off;
  float2* drec = rec + img * rec_per_image + rec_off;
  const float nanv = __int_as_float(0x7fc00000);
  bool sel = false;
  if (idx < n) {
    const int y = idx / w, x = idx - y * w;
    const size_t o = (size_t)y * pitch + x;
    const float2* P2 = P0 + (size_t)pitch * h;
    const size_t rc = rec_cell(x, y, nbands);
    const int xp = max(x - 1, 0), xn = min(x + 1, w - 1), yp = max(y - 1, 0), yn = min(y + 1, h - 1);
    const float2 a = P0[o], g = srec[rc + kRecP1];
    const float zx = (P2[(size_t)y * pitch + xn].y - P2[(size_t)y * pitch + xp].y) * 0.5f;
    const float zy = (P2[(size_t)yn * pitch + x].y - P2[(size_t)yp * pitch + x].y) * 0.5f;
    if (predicate == DVO_B200_PREDICATE_GRADIENT_THRESHOLD)   // ValidPointAndGradientThresholdPredicate (point_selection.h:52-67)
      sel = !is_nan(a.y) && (fabsf(g.x) > ti || fabsf(g.y) > ti || fabsf(zx) > td || fabsf(zy) > td);
    else if (predicate == DVO_B200_PREDICATE_VALID_POINT)     // ValidPointPredicate (point_selection.h:39-47): true depth
      sel = !is_nan(P2[o].y) && !is_nan(zx) && !is_nan(zy);
    else                                                      // MASK_ONLY
      sel = true;
    if (m) sel = sel && __ldg(m + img * m_img + (size_t)(y << m_shift) * m_row + ((size_t)x << m_shift)) != 0;
    drec[rc] = make_float2(a.x, sel ? a.y : nanv);
    drec[rc + kRecP1] = g;
  }
  const unsigned bits = __ballot_sync(0xffffffffu, sel);
  if ((threadIdx.x & 31) == 0 && idx < words * 32) masks[img * mask_words_per_image + mask_off + (idx >> 5)] = bits;
  if (idx < ntiles * kTileW) {
    const int tile = idx / kTileW, cx = idx - tile * kTileW;
    const int s = tile / nbands, b = tile - s * nbands;
    const int x = b * kTileW + cx, y0 = s * kTileH;
    const float2* st = srec + (size_t)tile * kRecF2;
    float2* dt = drec + (size_t)tile * kRecF2;
    reinterpret_cast<float*>(dt + kRecTx)[cx] = reinterpret_cast<const float*>(st + kRecTx)[cx];
    const int r0 = x >= w ? 0 : min(max(h - y0, 0), kTileH);
    for (int r = r0; r < kTileH; ++r) {
      dt[r * kTileW + cx] = st[r * kTileW + cx];
      dt[kRecP1 + r * kTileW + cx] = st[kRecP1 + r * kTileW + cx];
    }
  }
}

// point-cloud template tx[x] = (x - ox)/fx, ty[y] = (y - oy)/fy (IEEE division, rgbd_image.cpp:197-198)
__global__ void k_template(float* __restrict__ tmpl, size_t tmpl_per_image, size_t off, int w, int h, float fx,
                           float fy, float ox, float oy) {
  int img = blockIdx.y;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  float* t = tmpl + img * tmpl_per_image + off;
  if (i < w) t[i] = __fdiv_rn((float)i - ox, fx);
  else if (i < w + h) t[i] = __fdiv_rn((float)(i - w) - oy, fy);
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

int ensure_stage(dvo_b200_ctx* ctx, size_t dev_bytes, size_t host_bytes) {
  if (dev_bytes > ctx->d_stage_bytes) {
    if (ctx->d_stage) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->d_stage); ctx->d_stage = nullptr; ctx->d_stage_bytes = 0; }
    DVO_CUDA(ctx, cudaMalloc(&ctx->d_stage, dev_bytes));
    ctx->d_stage_bytes = dev_bytes;
  }
  if (host_bytes > ctx->h_stage_bytes) {
    if (ctx->h_stage) { cudaStreamSynchronize(ctx->stream); cudaFreeHost(ctx->h_stage); ctx->h_stage = nullptr; ctx->h_stage_bytes = 0; }
    DVO_CUDA(ctx, cudaMallocHost(&ctx->h_stage, host_bytes));
    ctx->h_stage_bytes = host_bytes;
  }
  return 0;
}

static void destroy_slab(Slab* s) {
  cudaFree(s->base);
  if (s->ready) cudaEventDestroy(s->ready);
  delete s;
}

static Slab* acquire_slab(dvo_b200_ctx* ctx, size_t bytes) {
  SlabPool& pool = *ctx->pool;
  std::lock_guard<std::mutex> lock(pool.mu);   // pyramids may be released by another host thread (see pyramid_free)
  auto it = pool.free.find(bytes);
  if (it != pool.free.end()) {
    Slab* s = it->second;
    pool.free.erase(it);
    s->refs = 0;
    return s;
  }
  void* p = nullptr;
  if (cudaMalloc(&p, bytes) != cudaSuccess) {
    // drop the pool and retry once
    for (auto& kv : pool.free) destroy_slab(kv.second);
    pool.free.clear();
    cudaGetLastError();
    if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  }
  Slab* s = new Slab;
  s->base = p; s->bytes = bytes; s->refs = 0; s->pool = ctx->pool;
  return s;
}

// Drops one reference to a slab: back to its context's pool, or freed if that context is gone.  Called from any host
// thread, possibly after the owning context has been destroyed.
static void slab_unref(Slab* s) {
  if (!s) return;
  std::shared_ptr<SlabPool> pool = s->pool;    // keeps the pool alive while its mutex is held
  std::lock_guard<std::mutex> lock(pool->mu);
  if (--s->refs == 0) {
    if (pool->closed) { cudaSetDevice(pool->device); destroy_slab(s); }
    else pool->free.insert({s->bytes, s});
  }
}

void pyramid_free(dvo_b200_pyramid* p) {
  Slab* s = p->slab;
  delete p;
  slab_unref(s);
}

void selection_free(dvo_b200_selection* s) {
  dvo_b200_pyramid* p = s->pyr;
  Slab* slab = s->slab;
  delete s;
  slab_unref(slab);
  if (p && p->refcount.fetch_sub(1, std::memory_order_acq_rel) == 1) pyramid_free(p);
}

// The context goes away: free what is pooled, and have slabs still referenced by live pyramids freed on release.
void pool_close(dvo_b200_ctx* ctx) {
  if (!ctx->pool) return;
  std::lock_guard<std::mutex> lock(ctx->pool->mu);
  for (auto& kv : ctx->pool->free) destroy_slab(kv.second);
  ctx->pool->free.clear();
  ctx->pool->closed = true;
}

FrameInput dense_frames(const void* d_I, const void* d_Z, int raw, float zscale, int w, int h) {
  FrameInput f;
  f.I = d_I; f.Z = d_Z; f.raw = raw; f.zscale = zscale;
  f.i_row = (size_t)w * (raw ? 1 : 4); f.i_img = f.i_row * h;
  f.z_row = (size_t)w * (raw ? 2 : 4); f.z_img = f.z_row * h;
  return f;
}

int pyramid_build_batch(dvo_b200_ctx* ctx, int n, const float* d_I, const float* d_Z, int w, int h, float fx, float fy,
                        float ox, float oy, int levels, float ti, float td, dvo_b200_pyramid** out) {
  return pyramid_build_batch_input(ctx, n, dense_frames(d_I, d_Z, 0, 0.f, w, h), w, h, fx, fy, ox, oy, levels, ti, td, out);
}

int pyramid_build_batch_input(dvo_b200_ctx* ctx, int n, const FrameInput& in, int w, int h, float fx, float fy, float ox, float oy,
                              int levels, float ti, float td, dvo_b200_pyramid** out) {
  if (n <= 0 || levels < 1 || levels > kMaxLevels || w < 32 || h < 2)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid: bad geometry");
  LevelInfo L[kMaxLevels];
  size_t plane_f2 = 0, mask_words = 0, tmpl_floats = 0, range_f2 = 0;
  for (int l = 0; l < levels; ++l) {
    LevelInfo& q = L[l];
    if (l == 0) { q.w = w; q.h = h; q.fx = fx; q.fy = fy; q.ox = ox; q.oy = oy; }
    else {
      q.w = L[l - 1].w / 2; q.h = L[l - 1].h / 2;
      q.fx = L[l - 1].fx * 0.5f; q.fy = L[l - 1].fy * 0.5f; q.ox = L[l - 1].ox * 0.5f; q.oy = L[l - 1].oy * 0.5f;
    }
    // odd sizes: the last column / row is dropped by the 2x2 mean exactly as in pyrDownMeanSmooth (rgbd_image.cpp:41)
    if (q.w < 8 || q.h < 2) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid: level too small");
    // the level kernel splits a linear pixel index with one multiply-high (tracker.cu): exact only below this bound
    if ((uint64_t)q.w * q.h >= (1ull << 30)) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "pyramid: image too large");
    q.n = q.w * q.h;
    q.words = (q.n + 31) / 32;
    q.pitch = (q.w + 1) & ~1;
    q.nbands = (q.w + kTileW - 1) / kTileW;
    q.nstrips = (q.h + kTileH - 1) / kTileH;
    q.plane_off = plane_f2; plane_f2 += 2 * (size_t)q.pitch * q.h;                       // P0, P2 (row-major, even pitch)
    q.rec_off = plane_f2; plane_f2 += (size_t)q.nbands * q.nstrips * kRecF2;               // reference tile records
    q.mask_off = mask_words; mask_words += q.words;
    q.tmpl_off = tmpl_floats; tmpl_floats += (size_t)((q.w + q.h + 3) & ~3);   // every level's tx[] starts 16-byte aligned (bulk copies)
    q.range_off = range_f2; range_f2 += (size_t)q.nbands * q.nstrips;
  }
  plane_f2 = align_up(plane_f2, 32);          // keep every image 256-byte aligned
  mask_words = align_up(mask_words, 64);
  tmpl_floats = align_up(tmpl_floats + kTileW, 64);   // lanes past a partial band read (and discard) up to kTileW floats beyond tx[w]
  range_f2 = align_up(range_f2, 32);
  const int sel_ints = 2 * kMaxLevels;
  size_t bytes_planes = (size_t)n * plane_f2 * sizeof(float2);
  size_t bytes_masks = (size_t)n * mask_words * sizeof(uint32_t);
  size_t bytes_tmpl = (size_t)n * tmpl_floats * sizeof(float);
  size_t bytes_sel = align_up((size_t)n * sel_ints * sizeof(int), 256);
  size_t bytes_range = (size_t)n * range_f2 * sizeof(float2);
  size_t total = bytes_planes + bytes_masks + bytes_tmpl + bytes_sel + bytes_range;
  Slab* slab = acquire_slab(ctx, total);
  if (!slab) return set_error(ctx, DVO_B200_ERR_OUT_OF_MEMORY, "pyramid: cudaMalloc failed");
  char* base = (char*)slab->base;
  float2* planes = (float2*)base;
  uint32_t* masks = (uint32_t*)(base + bytes_planes);
  float* tmpl = (float*)(base + bytes_planes + bytes_masks);
  int* sel = (int*)(base + bytes_planes + bytes_masks + bytes_tmpl);
  float2* ranges = (float2*)(base + bytes_planes + bytes_masks + bytes_tmpl + bytes_sel);

  cudaStream_t st = ctx->stream;
  {
    ProfScope prof(ctx, 3, 6 * levels - 1);
    const int T = 256;
    for (int l = 0; l < levels; ++l) {
      const LevelInfo& q = L[l];
      dim3 gt((q.w + q.h + T - 1) / T, n);
      k_template<<<gt, T, 0, st>>>(tmpl, tmpl_floats, q.tmpl_off, q.w, q.h, q.fx, q.fy, q.ox, q.oy);
      ctx->launches += 1;
      if (l == 0) continue;   // level 0 takes its intensity from the input image
      dim3 g((q.n + T - 1) / T, n);
      // the vector 2x2 loads need every block to start on a multiple of two pixels: base, row stride and (for a batch) image
      // stride all even multiples of the pixel size
      const size_t pair_bytes = in.raw ? 2 : 8;
      const int aligned = (((uintptr_t)in.I | in.i_row | (n > 1 ? in.i_img : 0)) % pair_bytes) == 0 ? 1 : 0;
      if (l == 1 && in.raw) k_pyr_intensity_down<true, true><<<g, T, 0, st>>>(in.I, in.i_row, in.i_img, aligned, planes, plane_f2, 0, L[0].pitch, q.plane_off, q.w, q.h, q.pitch);
      else if (l == 1) k_pyr_intensity_down<true, false><<<g, T, 0, st>>>(in.I, in.i_row, in.i_img, aligned, planes, plane_f2, 0, L[0].pitch, q.plane_off, q.w, q.h, q.pitch);
      else k_pyr_intensity_down<false, false><<<g, T, 0, st>>>(nullptr, 0, 0, 0, planes, plane_f2, L[l - 1].plane_off, L[l - 1].pitch, q.plane_off, q.w, q.h, q.pitch);
      ctx->launches += 1;
    }
    for (int l = 0; l < levels; ++l) {
      const LevelInfo& q = L[l];
      dim3 g((q.words * 32 + T - 1) / T, n);
      if (l == 0 && in.raw) k_pyr_finish<true, true><<<g, T, 0, st>>>(in, planes, plane_f2, q.plane_off, q.rec_off, q.nbands, q.w, q.h, q.pitch, l, masks, mask_words, q.mask_off, ti, td);
      else if (l == 0) k_pyr_finish<true, false><<<g, T, 0, st>>>(in, planes, plane_f2, q.plane_off, q.rec_off, q.nbands, q.w, q.h, q.pitch, l, masks, mask_words, q.mask_off, ti, td);
      else if (in.raw) k_pyr_finish<false, true><<<g, T, 0, st>>>(in, planes, plane_f2, q.plane_off, q.rec_off, q.nbands, q.w, q.h, q.pitch, l, masks, mask_words, q.mask_off, ti, td);
      else k_pyr_finish<false, false><<<g, T, 0, st>>>(in, planes, plane_f2, q.plane_off, q.rec_off, q.nbands, q.w, q.h, q.pitch, l, masks, mask_words, q.mask_off, ti, td);
      k_sel_info<<<n, 32, 0, st>>>(masks, mask_words, q.mask_off, q.words, sel, sel_ints, l);
      k_drop_odd_last<<<(n + 127) / 128, 128, 0, st>>>(planes, plane_f2, q.rec_off, q.nbands, q.w, sel, sel_ints, l, n);
      const int ntiles = q.nbands * q.nstrips;
      k_rec_fill<<<dim3((ntiles * kTileW + T - 1) / T, n), T, 0, st>>>(planes, plane_f2, q.rec_off, q.nbands, ntiles, q.w, q.h,
                                                                              tmpl, tmpl_floats, q.tmpl_off);
      ctx->launches += 1;
      k_tile_range<<<dim3((ntiles + 7) / 8, n), 256, 0, st>>>(planes, plane_f2, q.plane_off, q.w, q.h, q.pitch, q.nbands, ntiles,
                                                              ranges, range_f2, q.range_off);
      ctx->launches += 4;
    }
  }
  DVO_CUDA(ctx, cudaGetLastError());
  if (!slab->ready) DVO_CUDA(ctx, cudaEventCreateWithFlags(&slab->ready, cudaEventDisableTiming));
  DVO_CUDA(ctx, cudaEventRecord(slab->ready, st));
  for (int i = 0; i < n; ++i) {
    dvo_b200_pyramid* p = new dvo_b200_pyramid;
    p->ctx = ctx; p->device = ctx->device; p->refcount.store(1); p->levels = levels;
    std::memcpy(p->L, L, sizeof(LevelInfo) * levels);
    p->slab = slab; slab->refs++;
    p->planes = planes + (size_t)i * plane_f2;
    p->sel_mask = masks + (size_t)i * mask_words;
    p->sel_info = sel + (size_t)i * sel_ints;
    p->tmpl = tmpl + (size_t)i * tmpl_floats;
    p->tile_range = ranges + (size_t)i * range_f2;
    p->sel_ti = ti; p->sel_td = td;
    p->id = ctx->next_pyramid_id++;
    out[i] = p;
  }
  return 0;
}

// The selection (mask, {S, last}, the Zsel channel of the reference tile records) is state of the PYRAMID, shared by every context that aligns
// against it, while the reference keeps it per tracker (PointSelection, point_selection.cpp:100-113).  Contexts that use
// the same thresholds -- every caller in dvo_slam: one configuration per tracker family -- never get here twice.  A context
// that asks for other thresholds rewrites the selection on its stream; the host-side state is guarded by sel_mu and the
// slab's ready event is re-recorded, so a context that enqueues work on this pyramid LATER waits for the rewrite.  What is
// not supported: two contexts aligning against one reference pyramid with different thresholds at the same time
// (INTEGRATION.md, limits).
int pyramid_reselect(dvo_b200_ctx* ctx, dvo_b200_pyramid* p, float ti, float td) {
  std::lock_guard<std::mutex> lock(p->sel_mu);
  if (p->sel_ti == ti && p->sel_td == td) return 0;
  cudaStream_t st = ctx->stream;
  ProfScope prof(ctx, 4, 3 * p->levels);
  for (int l = 0; l < p->levels; ++l) {
    const LevelInfo& q = p->L[l];
    const int T = 256;
    k_reselect<<<(q.words * 32 + T - 1) / T, T, 0, st>>>(p->planes + q.plane_off, p->planes + q.rec_off, q.nbands, q.w, q.h, q.pitch,
                                                         p->sel_mask + q.mask_off, ti, td);
    k_sel_info<<<1, 32, 0, st>>>(p->sel_mask, 0, q.mask_off, q.words, p->sel_info, 0, l);
    k_drop_odd_last<<<1, 32, 0, st>>>(p->planes, 0, q.rec_off, q.nbands, q.w, p->sel_info, 0, l, 1);
    ctx->launches += 3;
  }
  DVO_CUDA(ctx, cudaGetLastError());
  if (p->slab && p->slab->ready) DVO_CUDA(ctx, cudaEventRecord(p->slab->ready, st));
  p->sel_ti = ti; p->sel_td = td;
  return 0;
}

// Layout of one selection inside its slab: the tile records of every level, then the mask words (at the pyramid's
// mask_off), then {S, last} per level.  The only part that differs from the pyramid is the Zsel channel and the masks.
int selection_build_batch(dvo_b200_ctx* ctx, int n, dvo_b200_pyramid* const* pyrs, int predicate, float ti, float td,
                          const SelMaskInput& mi, dvo_b200_selection** out) {
  const dvo_b200_pyramid* p0 = pyrs[0];
  const int levels = p0->levels;
  size_t rec_off[kMaxLevels], rec_f2 = 0;
  for (int l = 0; l < levels; ++l) {
    rec_off[l] = rec_f2;
    rec_f2 += (size_t)p0->L[l].nbands * p0->L[l].nstrips * kRecF2;
  }
  rec_f2 = align_up(rec_f2, 32);
  const size_t mask_words = align_up(p0->L[levels - 1].mask_off + p0->L[levels - 1].words, 64);
  const int sel_ints = 2 * kMaxLevels;
  const size_t bytes_rec = (size_t)n * rec_f2 * sizeof(float2);
  const size_t bytes_mask = (size_t)n * mask_words * sizeof(uint32_t);
  const size_t bytes_sel = align_up((size_t)n * sel_ints * sizeof(int), 256);
  const size_t bytes_tab = (size_t)n * sizeof(const float2*);
  Slab* slab = acquire_slab(ctx, bytes_rec + bytes_mask + bytes_sel + bytes_tab);
  if (!slab) return set_error(ctx, DVO_B200_ERR_OUT_OF_MEMORY, "selection: cudaMalloc failed");
  char* base = (char*)slab->base;
  float2* rec = (float2*)base;
  uint32_t* masks = (uint32_t*)(base + bytes_rec);
  int* sel = (int*)(base + bytes_rec + bytes_mask);
  const float2** tab = (const float2**)(base + bytes_rec + bytes_mask + bytes_sel);
  cudaStream_t st = ctx->stream;

  // host per-level masks go up through the device staging area (a pageable source is copied before the call returns)
  const uint8_t* staged[kMaxLevels] = {};
  size_t stage_bytes = 0, stage_off[kMaxLevels] = {};
  for (int l = 0; l < levels; ++l)
    if (mi.per_level[l]) { stage_off[l] = stage_bytes; stage_bytes += align_up((size_t)p0->L[l].n, 256); }
  if (stage_bytes) {
    int rc = ensure_stage(ctx, stage_bytes, 0);
    if (rc) { slab->refs = 1; slab_unref(slab); return rc; }
    for (int l = 0; l < levels; ++l)
      if (mi.per_level[l]) {
        staged[l] = (const uint8_t*)ctx->d_stage + stage_off[l];
        DVO_CUDA(ctx, cudaMemcpyAsync((void*)staged[l], mi.per_level[l], (size_t)p0->L[l].n, cudaMemcpyHostToDevice, st));
        ctx->h2d_bytes += p0->L[l].n;
      }
  }
  std::vector<const float2*> h_tab(n);
  for (int i = 0; i < n; ++i) {
    h_tab[i] = pyrs[i]->planes;
    // a pyramid built on another ctx's stream: order this stream after its build
    if (pyrs[i]->slab && pyrs[i]->slab->pool != ctx->pool && pyrs[i]->slab->ready) cudaStreamWaitEvent(st, pyrs[i]->slab->ready, 0);
  }
  DVO_CUDA(ctx, cudaMemcpyAsync(tab, h_tab.data(), bytes_tab, cudaMemcpyHostToDevice, st));
  ctx->h2d_bytes += bytes_tab;
  {
    ProfScope prof(ctx, 4, 3 * levels);
    const int T = 256;
    for (int l = 0; l < levels; ++l) {
      const LevelInfo& q = p0->L[l];
      const uint8_t* m = nullptr;
      size_t m_row = 0, m_img = 0;
      int m_shift = 0;
      if (mi.level0) { m = mi.level0; m_row = mi.row; m_img = mi.img; m_shift = l; }
      else if (staged[l]) { m = staged[l]; m_row = (size_t)q.w; }
      const int ntiles = q.nbands * q.nstrips;
      const int threads = std::max(q.words * 32, ntiles * kTileW);
      k_sel_build<<<dim3((threads + T - 1) / T, n), T, 0, st>>>(tab, q.plane_off, q.rec_off, q.nbands, ntiles, q.w, q.h, q.pitch, m, m_row,
                                                                  m_img, m_shift, rec, rec_f2, rec_off[l], masks, mask_words, q.mask_off,
                                                                  q.words, predicate, ti, td);
      k_sel_info<<<n, 32, 0, st>>>(masks, mask_words, q.mask_off, q.words, sel, sel_ints, l);
      k_drop_odd_last<<<(n + 127) / 128, 128, 0, st>>>(rec, rec_f2, rec_off[l], q.nbands, q.w, sel, sel_ints, l, n);
      ctx->launches += 3;
    }
  }
  DVO_CUDA(ctx, cudaGetLastError());
  if (!slab->ready) DVO_CUDA(ctx, cudaEventCreateWithFlags(&slab->ready, cudaEventDisableTiming));
  DVO_CUDA(ctx, cudaEventRecord(slab->ready, st));
  for (int i = 0; i < n; ++i) {
    dvo_b200_selection* s = new dvo_b200_selection;
    s->device = ctx->device;
    s->pyr = pyrs[i];
    pyrs[i]->refcount.fetch_add(1, std::memory_order_relaxed);
    s->slab = slab; slab->refs++;
    s->rec = rec + (size_t)i * rec_f2;
    s->mask = masks + (size_t)i * mask_words;
    s->sel_info = sel + (size_t)i * sel_ints;
    std::memcpy(s->rec_off, rec_off, sizeof(size_t) * levels);
    s->predicate = predicate; s->ti = ti; s->td = td;
    out[i] = s;
  }
  return 0;
}

}  // namespace dvo_b200
