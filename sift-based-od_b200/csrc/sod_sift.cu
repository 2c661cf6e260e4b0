// SIFT keypoints and descriptors on the device, reproducing cv2.SIFT_create() with its default parameters
// (3 layers per octave, contrast threshold 0.04, edge threshold 10, sigma 1.6, image doubled first, all
// features kept).  It replaces the host OpenCV call of Main.get_query_features (main.py:43-46) and of
// stream.sift_features; the conventions below follow OpenCV's sift.simd.hpp and were checked against cv2
// as a black box (GaussianBlur = sepFilter2D with getGaussianKernel CV_32F and BORDER_REFLECT_101,
// resize INTER_LINEAR with half-pixel centres, fastAtan2, the output sort and duplicate rule).
//
//   pyramid     u8 -> f32, bilinear x2, Gaussian chain per octave (one fused two-pass launch per level,
//               the horizontal pass kept in shared memory), octave o+1 starts from every other pixel of
//               level 3 of octave o.  DoG levels are never stored: every reader takes G[l+1] - G[l].
//   extrema     one thread per pixel and layer: 26-neighbour test, then OpenCV's Newton refinement,
//               contrast and edge tests in the same thread; survivors go to a candidate list.
//   orientation one warp per candidate: 36-bin histogram (per-lane partial histograms summed in a fixed
//               order, so the result does not depend on scheduling), smoothing, one keypoint per peak.
//   order       cub radix sort by (x, y), short runs of equal (x, y) ordered by (size, angle, response,
//               octave), entries equal in (pt, size, angle) dropped: cv2's KeyPointsFilter order.
//   descriptor  one block per keypoint, 4x4x8 histogram with trilinear spreading, clip 0.2, x512, u8.
//
// Every kernel has a frame dimension: a batch of B same-size images is one launch per pyramid level and one per
// stage.  Frame f has its own pyramid (at f x the pyramid of one frame in the workspace), its own counters and
// its own candidate / keypoint slabs of cap entries.  The order is per frame: the (x, y) sort over all slabs is
// followed, for B > 1, by a stable sort by frame, so each frame's slab ends up in the order one frame alone
// gets.  sod_sift_extract is the batch of one.  sod_sift_extract_mixed runs frames of different sizes through the
// same kernels: each reads a frame's geometry through the layout it is instantiated for (Pyramid or Mixed, below).
#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cfloat>
#include <climits>
#include <cstdio>
#include <cmath>

#include "sod_common.cuh"

namespace sod {
namespace {

constexpr int kLayers = 3;             // nOctaveLayers
constexpr int kLevels = kLayers + 3;   // Gaussian levels per octave
constexpr float kSigma = 1.6f;
constexpr float kContrast = 0.04f;
constexpr float kEdge = 10.f;
constexpr int kBorder = 5;             // SIFT_IMG_BORDER
constexpr int kMaxInterp = 5;          // SIFT_MAX_INTERP_STEPS
constexpr int kOriBins = 36;
constexpr int kD = 4, kN = 8;          // descriptor: kD x kD cells of kN orientation bins
constexpr int kHistLen = (kD + 2) * (kD + 2) * (kN + 2);
constexpr int kMaxOct = SOD_SIFT_MAX_OCTAVES;
constexpr int kMaxSide = 32768;        // input side limit: the doubled image stays below 2^16 pixels a side
constexpr int kTile = 32;              // blur output tile
constexpr int kMaxRadius = 13;         // largest blur radius of the default parameters (sigma 3.09, 27 taps)
constexpr int kOriWarps = 4;

// The kernels read a frame's geometry through one accessor, templated on the layout: Pyramid (frames of one size,
// fstride elements apart) or Mixed (a per-frame table, frames of any size).  Both give level(o, l, f), the size
// width / height(o, f) of octave o of frame f and octaves(f); the pyramid kernels take a step view of either
// (UniformUpsample / UniformStep or MixedStep: where frame f reads and writes one level).
struct Pyramid {
  float* base;
  int64_t off[kMaxOct];                // element offset of octave o's first level
  int64_t fstride;                     // elements from one frame's pyramid to the next
  int w[kMaxOct], h[kMaxOct];
  int n_oct;
  __host__ __device__ float* level(int o, int l, int f = 0) const {
    return base + f * fstride + off[o] + (int64_t)l * w[o] * h[o];
  }
  __device__ int width(int o, int) const { return w[o]; }
  __device__ int height(int o, int) const { return h[o]; }
  __device__ int octaves(int) const { return n_oct; }
};

// One frame of a mixed batch, written into the workspace by sift_mixed_setup_kernel.  Octave o of the frame is
// (2 width) >> o by (2 height) >> o pixels for o < n_oct, its first level at element off[o] of the workspace.
struct FrameGeom {
  const uint8_t* img;
  int64_t pitch;
  int64_t off[kMaxOct];
  int32_t width, height, n_oct, pad;
};

struct MixedTable {                    // the kernel parameter that carries the table to the device
  FrameGeom f[SOD_SIFT_MAX_MIXED_FRAMES];
};

struct Mixed {
  float* base;
  const FrameGeom* g;
  int frames;
  __device__ int octaves(int f) const {
    SOD_DCHECK(f >= 0 && f < frames);
    return g[f].n_oct;
  }
  __device__ int width(int o, int f) const { return o < octaves(f) ? (2 * g[f].width) >> o : 0; }
  __device__ int height(int o, int f) const { return o < octaves(f) ? (2 * g[f].height) >> o : 0; }
  __device__ float* level(int o, int l, int f) const {
    SOD_DCHECK(f >= 0 && f < frames && o >= 0 && o < g[f].n_oct && l >= 0 && l < kLevels);
    return base + g[f].off[o] + (int64_t)l * width(o, f) * height(o, f);
  }
};

struct Plane {                         // one level of one frame; w = h = 0 when the frame has no such octave
  float* p;
  int w, h;
};

struct Image {
  const uint8_t* p;
  int w, h;
  int64_t pitch;
};

// Frames of one size: every pointer is frame 0's, frame f's lies f strides further on.
struct UniformUpsample {
  const uint8_t* src;
  int sw, sh;
  int64_t pitch, frame_stride;
  float* dst;
  int64_t dst_stride;
  __device__ Image image(int f) const { return {src + f * frame_stride, sw, sh, pitch}; }
  __device__ Plane out(int f) const { return {dst + f * dst_stride, 2 * sw, 2 * sh}; }
};

struct UniformStep {
  static constexpr bool kRagged = false;
  const float* src;
  float* dst;
  int sw, sh, dw, dh;
  int64_t fstride;
  __device__ Plane in(int f) const { return {const_cast<float*>(src) + f * fstride, sw, sh}; }
  __device__ Plane out(int f) const { return {dst + f * fstride, dw, dh}; }
};

// Frames of any size: level (oi, li) -> level (oo, lo) of each frame (oi = -1: its u8 image).  Grids cover the
// largest frame; blocks outside their frame's level return at once.
struct MixedStep {
  static constexpr bool kRagged = true;
  Mixed P;
  int oi, li, oo, lo;
  __device__ Image image(int f) const {
    SOD_DCHECK(f >= 0 && f < P.frames);
    const FrameGeom& g = P.g[f];
    return {g.img, g.width, g.height, g.pitch};
  }
  __device__ Plane plane(int o, int l, int f) const {
    const int w = P.width(o, f), h = P.height(o, f);
    return {w ? P.level(o, l, f) : nullptr, w, h};
  }
  __device__ Plane in(int f) const { return plane(oi, li, f); }
  __device__ Plane out(int f) const { return plane(oo, lo, f); }
};

struct Taps {
  float k[2 * kMaxRadius + 1];
  int r;
};

struct Cand {                          // a refined extremum, before orientation (octave index o is 0-based)
  float x, y, size, response;
  int32_t octave, o, layer, r, c, frame;
};

struct Kp {                            // a finished keypoint in cv2's conventions (first octave -1)
  float x, y, size, angle, response;
  int32_t octave;
};

// Per-frame counters: candidates, keypoints, overflow flag, unused.  After them, kBatchInts ints of the batch:
// [0] rows written (the descriptor count).
constexpr int kFrameInts = 4;
constexpr int kBatchInts = 4;

// Workspace layout (byte offsets from the workspace start, every block 256-byte aligned).  The pyramids come
// first so that sod_sift_level_offset (frame 0) does not depend on the keypoint capacity or the batch.  Slabs
// hold frames x cap entries, frame f's at f x cap.
struct Plan {
  Pyramid pyr;
  int frames;
  int64_t cap;
  size_t cand, raw, keys_in, keys_out, vals_in, vals_out, keep, pos, counters, offset, cub_tmp, cub_bytes, total;
  size_t geom = 0;                     // mixed batches: the FrameGeom table
};

size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

int octave_count(int width, int height) {
  // cvRound(log2(min side of the doubled image) - 2) - firstOctave, firstOctave = -1
  const double m = 2.0 * (width < height ? width : height);
  return (int)std::lrint(std::log(m) / std::log(2.0) - 2.0) + 1;
}

// The pyramid of one image of this size (base and fstride left to the caller) and its bytes, 256-byte aligned;
// false if it has too many octaves.
bool plan_pyramid(int width, int height, Pyramid* P, size_t* bytes) {
  int n_oct = octave_count(width, height);
  if (n_oct < 0) n_oct = 0;
  if (n_oct > kMaxOct) return false;
  P->base = nullptr;
  P->n_oct = n_oct;
  int64_t off = 0;
  int w = 2 * width, h = 2 * height;
  for (int o = 0; o < kMaxOct; ++o) {
    P->off[o] = off;
    P->w[o] = o < n_oct ? w : 0;
    P->h[o] = o < n_oct ? h : 0;
    if (o < n_oct) {
      off += (int64_t)kLevels * w * h;
      w /= 2;
      h /= 2;
    }
  }
  *bytes = align256((size_t)off * sizeof(float));
  return true;
}

// The slabs of `frames` x cap keypoints from byte `at` of the workspace on, and the total.
void plan_slabs(int frames, int64_t cap, size_t at, Plan* p);

// Pyramid geometry and workspace offsets for `frames` images and cap keypoints a frame; cap = 0 plans the
// pyramids alone (sod_sift_describe).  frames x cap <= SOD_SIFT_MAX_CAP is the caller's check.
bool make_plan(int width, int height, int frames, int64_t cap, Plan* p) {
  size_t pyr_bytes;
  if (!plan_pyramid(width, height, &p->pyr, &pyr_bytes)) return false;
  p->pyr.fstride = (int64_t)(pyr_bytes / sizeof(float));
  plan_slabs(frames, cap, pyr_bytes * frames, p);
  return true;
}

void plan_slabs(int frames, int64_t cap, size_t at, Plan* p) {
  p->frames = frames;
  p->cap = cap;
  const int64_t slots = frames * cap;
  auto take = [&](size_t bytes) { size_t r = at; at += align256(bytes); return r; };
  p->cand = take(sizeof(Cand) * slots);
  p->raw = take(sizeof(Kp) * slots);
  p->keys_in = take(sizeof(uint64_t) * slots);      // for B > 1 also the frame keys of the second sort (2 x u32)
  p->keys_out = take(sizeof(uint64_t) * slots);
  p->vals_in = take(sizeof(int32_t) * slots);
  p->vals_out = take(sizeof(int32_t) * slots);
  p->keep = take(sizeof(int32_t) * slots);
  p->pos = take(sizeof(int32_t) * slots);
  p->counters = take(slots > 0 ? sizeof(int32_t) * (kFrameInts * frames + kBatchInts) : 0);
  p->offset = take(slots > 0 ? sizeof(int32_t) * frames : 0);
  size_t sort_bytes = 0, frame_sort_bytes = 0, scan_bytes = 0;
  if (slots > 0) {
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                    (const int32_t*)nullptr, (int32_t*)nullptr, (int)slots);
    if (frames > 1)
      cub::DeviceRadixSort::SortPairs(nullptr, frame_sort_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                      (const int32_t*)nullptr, (int32_t*)nullptr, (int)slots);
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, (int)slots);
  }
  p->cub_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
  if (frame_sort_bytes > p->cub_bytes) p->cub_bytes = frame_sort_bytes;
  p->cub_tmp = take(p->cub_bytes);
  p->total = at;
}

// A mixed batch: frame f's pyramid at the sum of the pyramids of frames 0..f-1 (each as plan_pyramid sizes it),
// then the slabs as for a uniform batch, then the geometry table (p->geom, frames x FrameGeom).  p->pyr holds the
// launch grids: per octave the largest size any frame has, and the largest octave count.  Sizes are the caller's
// check (1..kMaxSide a side).
bool make_mixed_plan(const int32_t* wh, int frames, int64_t cap, Plan* p, MixedTable* t) {
  Pyramid& grid = p->pyr;
  grid = Pyramid{};
  size_t at = 0;
  for (int f = 0; f < frames; ++f) {
    Pyramid one;
    size_t bytes;
    if (!plan_pyramid(wh[2 * f], wh[2 * f + 1], &one, &bytes)) return false;
    FrameGeom& g = t->f[f];
    g = FrameGeom{};
    g.width = wh[2 * f];
    g.height = wh[2 * f + 1];
    g.n_oct = one.n_oct;
    for (int o = 0; o < kMaxOct; ++o) {
      g.off[o] = (int64_t)(at / sizeof(float)) + one.off[o];
      grid.w[o] = std::max(grid.w[o], one.w[o]);
      grid.h[o] = std::max(grid.h[o], one.h[o]);
    }
    grid.n_oct = std::max(grid.n_oct, one.n_oct);
    at += bytes;
  }
  plan_slabs(frames, cap, at, p);
  p->geom = p->total;
  p->total += align256(sizeof(FrameGeom) * frames);
  return true;
}

// cv::getGaussianKernel(round(8 sigma + 1) | 1, sigma, CV_32F): exp in double, stored as float, normalised
// by the double sum of the stored values.
bool gaussian_taps(double sigma, Taps* t) {
  const int n = (int)std::lrint(sigma * 8 + 1) | 1;
  t->r = n / 2;
  if (t->r > kMaxRadius) return false;
  const double scale2 = -0.5 / (sigma * sigma);
  double sum = 0;
  for (int i = 0; i < n; ++i) {
    const double x = i - (n - 1) * 0.5;
    t->k[i] = (float)std::exp(scale2 * x * x);
    sum += t->k[i];
  }
  sum = 1. / sum;
  for (int i = 0; i < n; ++i) t->k[i] = (float)(t->k[i] * sum);
  return true;
}

// ---------------------------------------------------------------------------------------------- device

__device__ __forceinline__ int reflect101(int p, int len) {   // cv::borderInterpolate, BORDER_REFLECT_101
  if (len == 1) return 0;
  while ((unsigned)p >= (unsigned)len) p = p < 0 ? -p : 2 * len - 2 - p;
  return p;
}

// cv::fastAtan2 (degrees in [0, 360)), the polynomial OpenCV uses in its SIFT, not atan2.
__device__ __forceinline__ float fast_atan2(float y, float x) {
  constexpr float s = (float)(180 / 3.14159265358979323846);
  const float p1 = 0.9997878412794807f * s, p3 = -0.3258083974640975f * s, p5 = 0.1555786518463281f * s,
              p7 = -0.04432655554792128f * s;
  const float ax = fabsf(x), ay = fabsf(y);
  float a, c, c2;
  if (ax >= ay) {
    c = ay / (ax + (float)DBL_EPSILON);
    c2 = c * c;
    a = (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
  } else {
    c = ax / (ay + (float)DBL_EPSILON);
    c2 = c * c;
    a = 90.f - (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
  }
  if (x < 0) a = 180.f - a;
  if (y < 0) a = 360.f - a;
  return a;
}

// cv::resize(INTER_LINEAR) to exactly twice the size: source coordinate (d + 0.5) / 2 - 0.5, clamped.
// blockIdx.z = frame.
template <class S>
__global__ void sift_upsample_kernel(S s) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  const Image im = s.image(blockIdx.z);
  const Plane d = s.out(blockIdx.z);
  const int sw = im.w, sh = im.h, dw = d.w, dh = d.h;
  const int64_t pitch = im.pitch;
  if (x >= dw || y >= dh) return;
  const uint8_t* __restrict__ src = im.p;
  float* __restrict__ dst = d.p;
  float fx = (float)((x + 0.5) * 0.5 - 0.5), fy = (float)((y + 0.5) * 0.5 - 0.5);
  int sx = (int)floorf(fx), sy = (int)floorf(fy);
  fx -= sx;
  fy -= sy;
  if (sx < 0) fx = 0.f, sx = 0;
  if (sy < 0) fy = 0.f, sy = 0;
  if (sx >= sw - 1) fx = 0.f, sx = sw - 1;
  if (sy >= sh - 1) fy = 0.f, sy = sh - 1;
  const int sx1 = min(sx + 1, sw - 1), sy1 = min(sy + 1, sh - 1);
  const uint8_t* r0 = src + (int64_t)sy * pitch;
  const uint8_t* r1 = src + (int64_t)sy1 * pitch;
  const float a0 = (float)r0[sx] * (1.f - fx) + (float)r0[sx1] * fx;
  const float a1 = (float)r1[sx] * (1.f - fx) + (float)r1[sx1] * fx;
  dst[(int64_t)y * dw + x] = a0 * (1.f - fy) + a1 * fy;
}

// cv::GaussianBlur on a float image: horizontal pass into shared memory, then the vertical pass, both in the
// symmetric form of OpenCV's row / column filters (centre tap, then pairs outwards), BORDER_REFLECT_101.
// blockIdx.z = frame; source and destination have the same size.
template <class S>
__global__ void __launch_bounds__(256) sift_blur_kernel(S s, Taps t) {
  __shared__ float in[kTile + 2 * kMaxRadius][kTile + 2 * kMaxRadius + 1];
  __shared__ float mid[kTile + 2 * kMaxRadius][kTile + 1];
  __shared__ float k[2 * kMaxRadius + 1];
  const Plane a = s.in(blockIdx.z);
  const int w = a.w, h = a.h, r = t.r, x0 = blockIdx.x * kTile, y0 = blockIdx.y * kTile, span = kTile + 2 * r;
  if (S::kRagged && (x0 >= w || y0 >= h)) return;
  const float* __restrict__ src = a.p;
  float* __restrict__ dst = s.out(blockIdx.z).p;
  if (threadIdx.x < 2 * r + 1) k[threadIdx.x] = t.k[threadIdx.x];
  for (int i = threadIdx.x; i < span * span; i += blockDim.x) {
    const int ty = i / span, tx = i - ty * span;
    const int gy = reflect101(y0 - r + ty, h), gx = reflect101(x0 - r + tx, w);
    SOD_DCHECK(gy >= 0 && gy < h && gx >= 0 && gx < w);
    in[ty][tx] = src[(int64_t)gy * w + gx];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < span * kTile; i += blockDim.x) {
    const int ty = i / kTile, tx = i - ty * kTile;
    const float* s = &in[ty][tx + r];
    float acc = k[r] * s[0];
    for (int j = 1; j <= r; ++j) acc += k[r + j] * (s[j] + s[-j]);
    mid[ty][tx] = acc;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kTile * kTile; i += blockDim.x) {
    const int ty = i / kTile, tx = i - ty * kTile, gx = x0 + tx, gy = y0 + ty;
    if (gx >= w || gy >= h) continue;
    float acc = k[r] * mid[ty + r][tx];
    for (int j = 1; j <= r; ++j) acc += k[r + j] * (mid[ty + r + j][tx] + mid[ty + r - j][tx]);
    dst[(int64_t)gy * w + gx] = acc;
  }
}

// cv::resize(INTER_NEAREST) to half size: every other pixel.  blockIdx.z = frame.
template <class S>
__global__ void sift_halve_kernel(S s) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  const Plane d = s.out(blockIdx.z);
  if (x >= d.w || y >= d.h) return;
  const Plane a = s.in(blockIdx.z);
  d.p[(int64_t)y * d.w + x] = a.p[(int64_t)(2 * y) * a.w + 2 * x];
}

// DoG level l of octave o of frame f at (r, c): G[l+1] - G[l], the value cv::subtract stores.
template <class L>
__device__ __forceinline__ float dog(const L& P, int f, int o, int l, int r, int c) {
  const int64_t i = (int64_t)r * P.width(o, f) + c;
  return P.level(o, l + 1, f)[i] - P.level(o, l, f)[i];
}

// OpenCV's adjustLocalExtrema: Newton steps on the 3x3 Hessian of the DoG (derivatives scaled by 1/255),
// contrast and edge tests, keypoint fields in the octave numbering of the doubled image.
template <class L>
__device__ bool refine(const L& P, int f, int o, int& layer, int& r, int& c, Cand* kp) {
  constexpr float img_scale = 1.f / 255.f, deriv_scale = img_scale * 0.5f, second_scale = img_scale,
                  cross_scale = img_scale * 0.25f;
  const int w = P.width(o, f), h = P.height(o, f);
  float xi = 0, xr = 0, xc = 0;
  int i = 0;
  for (; i < kMaxInterp; ++i) {
    auto D = [&](int dl, int dr, int dc) { return dog(P, f, o, layer + dl, r + dr, c + dc); };
    const float dx = (D(0, 0, 1) - D(0, 0, -1)) * deriv_scale, dy = (D(0, 1, 0) - D(0, -1, 0)) * deriv_scale,
                ds = (D(1, 0, 0) - D(-1, 0, 0)) * deriv_scale;
    const float v2 = D(0, 0, 0) * 2;
    const float dxx = (D(0, 0, 1) + D(0, 0, -1) - v2) * second_scale;
    const float dyy = (D(0, 1, 0) + D(0, -1, 0) - v2) * second_scale;
    const float dss = (D(1, 0, 0) + D(-1, 0, 0) - v2) * second_scale;
    const float dxy = (D(0, 1, 1) - D(0, 1, -1) - D(0, -1, 1) + D(0, -1, -1)) * cross_scale;
    const float dxs = (D(1, 0, 1) - D(1, 0, -1) - D(-1, 0, 1) + D(-1, 0, -1)) * cross_scale;
    const float dys = (D(1, 1, 0) - D(1, -1, 0) - D(-1, 1, 0) + D(-1, -1, 0)) * cross_scale;
    // Matx33f::solve(DECOMP_LU) of a 3x3 system: Cramer's rule; a singular matrix leaves X = 0
    const float a00 = dxx, a01 = dxy, a02 = dxs, a10 = dxy, a11 = dyy, a12 = dys, a20 = dxs, a21 = dys, a22 = dss;
    float det = a00 * (a11 * a22 - a21 * a12) - a01 * (a10 * a22 - a20 * a12) + a02 * (a10 * a21 - a20 * a11);
    float X0 = 0, X1 = 0, X2 = 0;
    if (det != 0) {
      det = 1 / det;
      X0 = det * (dx * (a11 * a22 - a12 * a21) - a01 * (dy * a22 - a12 * ds) + a02 * (dy * a21 - a11 * ds));
      X1 = det * (a00 * (dy * a22 - a12 * ds) - dx * (a10 * a22 - a12 * a20) + a02 * (a10 * ds - dy * a20));
      X2 = det * (a00 * (a11 * ds - dy * a21) - a01 * (a10 * ds - dy * a20) + dx * (a10 * a21 - a11 * a20));
    }
    xi = -X2;
    xr = -X1;
    xc = -X0;
    if (fabsf(xi) < 0.5f && fabsf(xr) < 0.5f && fabsf(xc) < 0.5f) break;
    constexpr float far = (float)(INT_MAX / 3);
    if (fabsf(xi) > far || fabsf(xr) > far || fabsf(xc) > far) return false;
    c += __float2int_rn(xc);
    r += __float2int_rn(xr);
    layer += __float2int_rn(xi);
    if (layer < 1 || layer > kLayers || c < kBorder || c >= w - kBorder || r < kBorder || r >= h - kBorder)
      return false;
  }
  if (i >= kMaxInterp) return false;
  auto D = [&](int dl, int dr, int dc) { return dog(P, f, o, layer + dl, r + dr, c + dc); };
  const float dx = (D(0, 0, 1) - D(0, 0, -1)) * deriv_scale, dy = (D(0, 1, 0) - D(0, -1, 0)) * deriv_scale,
              ds = (D(1, 0, 0) - D(-1, 0, 0)) * deriv_scale;
  const float t = dx * xc + dy * xr + ds * xi;
  const float contr = D(0, 0, 0) * img_scale + t * 0.5f;
  if (fabsf(contr) * kLayers < kContrast) return false;
  const float v2 = D(0, 0, 0) * 2.f;
  const float dxx = (D(0, 0, 1) + D(0, 0, -1) - v2) * second_scale;
  const float dyy = (D(0, 1, 0) + D(0, -1, 0) - v2) * second_scale;
  const float dxy = (D(0, 1, 1) - D(0, 1, -1) - D(0, -1, 1) + D(0, -1, -1)) * cross_scale;
  const float tr = dxx + dyy, det = dxx * dyy - dxy * dxy;
  if (det <= 0 || tr * tr * kEdge >= (kEdge + 1) * (kEdge + 1) * det) return false;
  const float scale = (float)(1 << o);
  kp->x = ((float)c + xc) * scale;
  kp->y = ((float)r + xr) * scale;
  kp->octave = o + (layer << 8) + (__double2int_rn(((double)xi + 0.5) * 255) << 16);
  kp->size = kSigma * powf(2.f, ((float)layer + xi) / kLayers) * scale * 2;
  kp->response = fabsf(contr);
  return true;
}

// Scale-space extrema of octave o: |DoG| > floor(0.5 * 0.04 / 3 * 255) = 1, not smaller (or not larger)
// than all 26 neighbours, outside the 5-pixel border; refined survivors are appended to their frame's slab of
// cand.  blockIdx.z = frame * kLayers + layer - 1.
template <class L>
__global__ void sift_extrema_kernel(L P, int o, Cand* __restrict__ cand, int cap, int* __restrict__ counters) {
  const int c = kBorder + blockIdx.x * blockDim.x + threadIdx.x;
  const int r = kBorder + blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z / kLayers, layer = 1 + blockIdx.z % kLayers;
  if (c >= P.width(o, f) - kBorder || r >= P.height(o, f) - kBorder) return;
  const float val = dog(P, f, o, layer, r, c);
  if (!(fabsf(val) > 1.f)) return;
  bool ext = true;
  if (val > 0) {
    for (int dl = -1; dl <= 1 && ext; ++dl)
      for (int dr = -1; dr <= 1 && ext; ++dr)
        for (int dc = -1; dc <= 1; ++dc)
          if ((dl | dr | dc) && !(val >= dog(P, f, o, layer + dl, r + dr, c + dc))) { ext = false; break; }
  } else {
    for (int dl = -1; dl <= 1 && ext; ++dl)
      for (int dr = -1; dr <= 1 && ext; ++dr)
        for (int dc = -1; dc <= 1; ++dc)
          if ((dl | dr | dc) && !(val <= dog(P, f, o, layer + dl, r + dr, c + dc))) { ext = false; break; }
  }
  if (!ext) return;
  int l1 = layer, r1 = r, c1 = c;
  Cand kp;
  if (!refine(P, f, o, l1, r1, c1, &kp)) return;
  kp.o = o;
  kp.layer = l1;
  kp.r = r1;
  kp.c = c1;
  kp.frame = f;
  int* fc = counters + f * kFrameInts;
  const int slot = atomicAdd(&fc[0], 1);
  if (slot >= cap) {
    atomicExch(&fc[2], 1);
    return;
  }
  SOD_DCHECK(slot >= 0 && slot < cap);
  cand[(int64_t)f * cap + slot] = kp;
}

// OpenCV's calcOrientationHist + the peak loop of findScaleSpaceExtrema, one warp per candidate; blockIdx.y is
// the frame whose slab the blocks walk.  Every keypoint is written to its frame's raw slab already moved to the
// first octave -1 (octave byte - 1, pt and size halved).
template <class L>
__global__ void __launch_bounds__(32 * kOriWarps) sift_orient_kernel(L P, const Cand* __restrict__ cand,
                                                                     int cap, int* __restrict__ counters,
                                                                     Kp* __restrict__ raw) {
  __shared__ float part[kOriWarps][32][kOriBins + 1];
  __shared__ float hist[kOriWarps][kOriBins + 4];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  int* fc = counters + blockIdx.y * kFrameInts;
  const int n = min(fc[0], cap);
  for (int ci = blockIdx.x * kOriWarps + wib; ci < n; ci += gridDim.x * kOriWarps) {
    const Cand k = cand[(int64_t)blockIdx.y * cap + ci];
    SOD_DCHECK(k.o >= 0 && k.o < P.octaves(k.frame) && k.layer >= 1 && k.layer <= kLayers &&
               k.frame == (int)blockIdx.y);
    const float* img = P.level(k.o, k.layer, k.frame);
    const int w = P.width(k.o, k.frame), h = P.height(k.o, k.frame);
    const float scl = k.size * 0.5f / (float)(1 << k.o);
    const int radius = __float2int_rn(4.5f * scl);
    const float sigma = 1.5f * scl, expf_scale = -1.f / (2.f * sigma * sigma);
    for (int b = 0; b < kOriBins; ++b) part[wib][lane][b] = 0.f;
    const int side = 2 * radius + 1;
    for (int s = lane; s < side * side; s += 32) {
      const int i = s / side - radius, j = s % side - radius;
      const int y = k.r + i, x = k.c + j;
      if (y <= 0 || y >= h - 1 || x <= 0 || x >= w - 1) continue;
      const float dx = img[(int64_t)y * w + x + 1] - img[(int64_t)y * w + x - 1];
      const float dy = img[(int64_t)(y - 1) * w + x] - img[(int64_t)(y + 1) * w + x];
      const float wt = expf((float)(i * i + j * j) * expf_scale);
      const float ori = fast_atan2(dy, dx), mag = sqrtf(dx * dx + dy * dy);
      int bin = __float2int_rn((kOriBins / 360.f) * ori);
      if (bin >= kOriBins) bin -= kOriBins;
      if (bin < 0) bin += kOriBins;
      SOD_DCHECK(bin >= 0 && bin < kOriBins);
      part[wib][lane][bin] += wt * mag;
    }
    __syncwarp();
    for (int b = lane; b < kOriBins; b += 32) {
      float acc = 0.f;
      for (int l = 0; l < 32; ++l) acc += part[wib][l][b];
      hist[wib][b + 2] = acc;
    }
    __syncwarp();
    if (lane == 0) {
      float* t = &hist[wib][2];
      t[-1] = t[kOriBins - 1];
      t[-2] = t[kOriBins - 2];
      t[kOriBins] = t[0];
      t[kOriBins + 1] = t[1];
      float sm[kOriBins];
      float omax = 0.f;
      for (int b = 0; b < kOriBins; ++b) {
        sm[b] = (t[b - 2] + t[b + 2]) * (1.f / 16.f) + (t[b - 1] + t[b + 1]) * (4.f / 16.f) + t[b] * (6.f / 16.f);
        omax = b ? fmaxf(omax, sm[b]) : sm[b];
      }
      const float mag_thr = omax * 0.8f;
      for (int j = 0; j < kOriBins; ++j) {
        const int l = j > 0 ? j - 1 : kOriBins - 1, r2 = j < kOriBins - 1 ? j + 1 : 0;
        if (sm[j] > sm[l] && sm[j] > sm[r2] && sm[j] >= mag_thr) {
          float bin = j + 0.5f * (sm[l] - sm[r2]) / (sm[l] - 2 * sm[j] + sm[r2]);
          bin = bin < 0 ? kOriBins + bin : bin >= kOriBins ? bin - kOriBins : bin;
          float angle = 360.f - (float)((360.f / kOriBins) * bin);
          if (fabsf(angle - 360.f) < FLT_EPSILON) angle = 0.f;
          const int slot = atomicAdd(&fc[1], 1);
          if (slot >= cap) {
            atomicExch(&fc[2], 1);
            continue;
          }
          SOD_DCHECK(slot >= 0 && slot < cap);
          Kp& o = raw[(int64_t)k.frame * cap + slot];
          o.x = k.x * 0.5f;
          o.y = k.y * 0.5f;
          o.size = k.size * 0.5f;
          o.angle = angle;
          o.response = k.response;
          o.octave = (k.octave & ~255) | ((k.octave - 1) & 255);
        }
      }
    }
    __syncwarp();
  }
}

// Sort key: (x bits, y bits) of the non-negative coordinates order as (x, y).
__device__ __forceinline__ uint64_t xy_key(const Kp& k) {
  return ((uint64_t)__float_as_uint(k.x) << 32) | __float_as_uint(k.y);
}

// Keys of every slot of every frame's raw slab; unused slots sort last.
__global__ void sift_sort_keys_kernel(const Kp* __restrict__ raw, const int* __restrict__ counters, int cap,
                                      int slots, uint64_t* __restrict__ keys, int32_t* __restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= slots) return;
  const int f = i / cap, n = min(counters[f * kFrameInts + 1], cap);
  keys[i] = i - f * cap < n ? xy_key(raw[i]) : ~0ull;
  vals[i] = i;
}

// B > 1: the frame of each slot in (x, y) order, the key of the stable sort that gathers each frame's slots
// into its slab again (in (x, y) order, unused slots last).
__global__ void sift_frame_keys_kernel(const int32_t* __restrict__ vals, int cap, int slots,
                                       uint32_t* __restrict__ fkeys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= slots) return;
  SOD_DCHECK(vals[i] >= 0 && vals[i] < slots);
  fkeys[i] = (uint32_t)(vals[i] / cap);
}

__device__ __forceinline__ bool kp_less(const Kp& a, const Kp& b) {   // cv2's order after equal (x, y)
  if (a.size != b.size) return a.size < b.size;
  if (a.angle != b.angle) return a.angle < b.angle;
  if (a.response != b.response) return a.response < b.response;
  return a.octave < b.octave;
}

// Orders every run of equal (x, y) inside a frame's slab by (size, angle, response, octave); runs are a few
// keypoints long (the orientations of one location), so the first thread of a run sorts it by insertion.  The
// other threads of a run only compare keys, which every entry of the run shares.
__global__ void sift_sort_runs_kernel(const Kp* __restrict__ raw, const int* __restrict__ counters, int cap,
                                      int slots, int32_t* __restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= slots) return;
  const int f = i / cap, j = i - f * cap, n = min(counters[f * kFrameInts + 1], cap);
  if (j + 1 >= n) return;
  const uint64_t key = xy_key(raw[vals[i]]);
  if ((j > 0 && xy_key(raw[vals[i - 1]]) == key) || xy_key(raw[vals[i + 1]]) != key) return;
  const int end = f * cap + n;
  int e = i + 1;
  while (e < end && xy_key(raw[vals[e]]) == key) ++e;
  for (int a = i + 1; a < e; ++a) {
    const int v = vals[a];
    SOD_DCHECK(v >= f * cap && v < end);
    int b = a - 1;
    while (b >= i && kp_less(raw[v], raw[vals[b]])) {
      vals[b + 1] = vals[b];
      --b;
    }
    vals[b + 1] = v;
  }
}

// KeyPointsFilter::removeDuplicatedSorted: keep an entry unless it equals its predecessor in pt, size and
// angle (equal entries are adjacent in this order).
__global__ void sift_keep_kernel(const Kp* __restrict__ raw, const int* __restrict__ counters, int cap, int slots,
                                 const int32_t* __restrict__ vals, int32_t* __restrict__ keep) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= slots) return;
  const int f = i / cap, j = i - f * cap, n = min(counters[f * kFrameInts + 1], cap);
  int k = 0;
  if (j < n) {
    k = 1;
    if (j > 0) {
      SOD_DCHECK(vals[i] >= 0 && vals[i] < slots && vals[i - 1] >= 0 && vals[i - 1] < slots);
      const Kp a = raw[vals[i - 1]], b = raw[vals[i]];
      k = !(a.x == b.x && a.y == b.y && a.size == b.size && a.angle == b.angle);
    }
  }
  keep[i] = k;
}

// Where the rows go.  count / offset / overflow have one entry per frame; frame and rows_overflow may be NULL.
struct Rows {
  float *xy, *size, *angle, *response;
  int32_t* octave;
  uint8_t* des;
  int32_t *frame, *count, *offset, *overflow, *rows_overflow;
  int64_t cap_rows;
};

// Per frame: the keypoints left after duplicate removal, capped at max_per_frame (0 = all), and where they start
// when the frames are packed in batch order; the overflow flags; batch[0] = rows written.  One block.
__global__ void __launch_bounds__(256) sift_frame_rows_kernel(const int32_t* __restrict__ keep,
                                                              const int32_t* __restrict__ pos,
                                                              const int* __restrict__ counters, int cap, int frames,
                                                              int64_t max_per_frame, Rows out,
                                                              int* __restrict__ batch) {
  using Scan = cub::BlockScan<int, 256>;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int f0 = 0; f0 < frames; f0 += 256) {
    const int f = f0 + threadIdx.x;
    int n = 0;
    if (f < frames) {
      const int last = (f + 1) * cap - 1;
      n = pos[last] + keep[last] - pos[f * cap];
      if (max_per_frame > 0 && n > max_per_frame) n = (int)max_per_frame;
    }
    int excl, total;
    Scan(tmp).ExclusiveSum(n, excl, total);
    if (f < frames) {
      out.count[f] = n;
      out.offset[f] = carry + excl;
      out.overflow[f] = counters[f * kFrameInts + 2];
    }
    __syncthreads();
    if (threadIdx.x == 0) carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    batch[0] = (int)min((int64_t)carry, out.cap_rows);
    if (out.rows_overflow) out.rows_overflow[0] = carry > out.cap_rows;
  }
}

// The first count[f] kept entries of each frame, at rows offset[f].. (rows past cap_rows are dropped and flagged).
__global__ void sift_emit_kernel(const Kp* __restrict__ raw, int cap, int slots, const int32_t* __restrict__ vals,
                                 const int32_t* __restrict__ keep, const int32_t* __restrict__ pos, Rows out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= slots || !keep[i]) return;
  const int f = i / cap, local = pos[i] - pos[f * cap];
  if (local >= out.count[f]) return;
  const int64_t p = (int64_t)out.offset[f] + local;
  if (p >= out.cap_rows) return;
  const int v = vals[i];
  SOD_DCHECK(p >= 0 && v >= f * cap && v < (f + 1) * cap);
  const Kp k = raw[v];
  out.xy[2 * p] = k.x;
  out.xy[2 * p + 1] = k.y;
  out.size[p] = k.size;
  out.angle[p] = k.angle;
  out.response[p] = k.response;
  out.octave[p] = k.octave;
  if (out.frame) out.frame[p] = f;
}

// OpenCV's calcDescriptors + calcSIFTDescriptor, one 128-thread block per keypoint.  n_dev (device, may be
// NULL) overrides n; frame (may be NULL = all 0) names each keypoint's pyramid.  A keypoint whose octave / layer
// names no level of the pyramid gets a zero row and is counted in n_invalid (cv2 refuses such a keypoint).
// 16 blocks an SM (32 registers): the grid below is 16 blocks an SM, one wave.
template <class L>
__global__ void __launch_bounds__(128, 16) sift_descriptor_kernel(L P, const float* __restrict__ xy,
                                                              const float* __restrict__ size,
                                                              const float* __restrict__ angle,
                                                              const int32_t* __restrict__ octave,
                                                              const int32_t* __restrict__ frame, int64_t n,
                                                              const int32_t* __restrict__ n_dev,
                                                              uint8_t* __restrict__ des, int32_t* n_invalid) {
  __shared__ float hist[kHistLen];
  __shared__ float red[4];
  const int tid = threadIdx.x;
  if (n_dev && n_dev[0] < n) n = n_dev[0];
  for (int64_t q = blockIdx.x; q < n; q += gridDim.x) {
    const int packed = octave[q];
    int oct = packed & 255;
    const int layer = (packed >> 8) & 255;
    oct = oct < 128 ? oct : (-128 | oct);
    const int o = oct + 1;
    const int f = frame ? frame[q] : 0;
    SOD_DCHECK(f >= 0);
    if (o < 0 || o >= P.octaves(f) || layer > kLayers + 2) {
      des[q * 128 + tid] = 0;
      if (tid == 0 && n_invalid) atomicAdd(n_invalid, 1);
      continue;
    }
    const float scale = oct >= 0 ? 1.f / (float)(1 << oct) : (float)(1 << -oct);
    const float scl = size[q] * scale * 0.5f;
    const float ptx = xy[2 * q] * scale, pty = xy[2 * q + 1] * scale;
    float ori = 360.f - angle[q];
    if (fabsf(ori - 360.f) < FLT_EPSILON) ori = 0.f;
    const float* img = P.level(o, layer, f);
    const int cols = P.width(o, f), rows = P.height(o, f);
    const int px = __float2int_rn(ptx), py = __float2int_rn(pty);
    float cos_t = cosf(ori * (float)(3.14159265358979323846 / 180)),
          sin_t = sinf(ori * (float)(3.14159265358979323846 / 180));
    const float bins_per_deg = kN / 360.f, exp_scale = -1.f / (kD * kD * 0.5f);
    const float hist_width = 3.f * scl;
    int radius = __float2int_rn(hist_width * 1.4142135623730951f * (kD + 1) * 0.5f);
    radius = min(radius, (int)sqrt((double)cols * cols + (double)rows * rows));
    cos_t /= hist_width;
    sin_t /= hist_width;
    for (int i = tid; i < kHistLen; i += blockDim.x) hist[i] = 0.f;
    __syncthreads();
    const int side = 2 * radius + 1;
    for (int s = tid; s < side * side; s += blockDim.x) {
      const int i = s / side - radius, j = s % side - radius;
      const float c_rot = j * cos_t - i * sin_t, r_rot = j * sin_t + i * cos_t;
      float rbin = r_rot + kD / 2 - 0.5f, cbin = c_rot + kD / 2 - 0.5f;
      const int r = py + i, c = px + j;
      if (!(rbin > -1 && rbin < kD && cbin > -1 && cbin < kD && r > 0 && r < rows - 1 && c > 0 && c < cols - 1))
        continue;
      const float dx = img[(int64_t)r * cols + c + 1] - img[(int64_t)r * cols + c - 1];
      const float dy = img[(int64_t)(r - 1) * cols + c] - img[(int64_t)(r + 1) * cols + c];
      const float wt = expf((c_rot * c_rot + r_rot * r_rot) * exp_scale);
      float obin = (fast_atan2(dy, dx) - ori) * bins_per_deg;
      const float mag = sqrtf(dx * dx + dy * dy) * wt;
      const int r0 = (int)floorf(rbin), c0 = (int)floorf(cbin);
      int o0 = (int)floorf(obin);
      rbin -= r0;
      cbin -= c0;
      obin -= o0;
      if (o0 < 0) o0 += kN;
      if (o0 >= kN) o0 -= kN;
      const float v_r1 = mag * rbin, v_r0 = mag - v_r1;
      const float v_rc11 = v_r1 * cbin, v_rc10 = v_r1 - v_rc11;
      const float v_rc01 = v_r0 * cbin, v_rc00 = v_r0 - v_rc01;
      const float v_rco111 = v_rc11 * obin, v_rco110 = v_rc11 - v_rco111;
      const float v_rco101 = v_rc10 * obin, v_rco100 = v_rc10 - v_rco101;
      const float v_rco011 = v_rc01 * obin, v_rco010 = v_rc01 - v_rco011;
      const float v_rco001 = v_rc00 * obin, v_rco000 = v_rc00 - v_rco001;
      const int idx = ((r0 + 1) * (kD + 2) + c0 + 1) * (kN + 2) + o0;
      SOD_DCHECK(idx >= 0 && idx + (kD + 3) * (kN + 2) + 1 < kHistLen);
      atomicAdd(&hist[idx], v_rco000);
      atomicAdd(&hist[idx + 1], v_rco001);
      atomicAdd(&hist[idx + (kN + 2)], v_rco010);
      atomicAdd(&hist[idx + (kN + 3)], v_rco011);
      atomicAdd(&hist[idx + (kD + 2) * (kN + 2)], v_rco100);
      atomicAdd(&hist[idx + (kD + 2) * (kN + 2) + 1], v_rco101);
      atomicAdd(&hist[idx + (kD + 3) * (kN + 2)], v_rco110);
      atomicAdd(&hist[idx + (kD + 3) * (kN + 2) + 1], v_rco111);
    }
    __syncthreads();
    // the orientation histograms are circular: bins n and n+1 fold onto 0 and 1
    const int cell = tid / kN, k = tid % kN;
    const int hidx = ((cell / kD + 1) * (kD + 2) + (cell % kD + 1)) * (kN + 2);
    float v = hist[hidx + k] + (k < 2 ? hist[hidx + kN + k] : 0.f);
    auto block_sum = [&](float x) {
      for (int m = 16; m; m >>= 1) x += __shfl_xor_sync(0xffffffffu, x, m);
      if ((tid & 31) == 0) red[tid >> 5] = x;
      __syncthreads();
      const float s = red[0] + red[1] + red[2] + red[3];
      __syncthreads();
      return s;
    };
    const float thr = sqrtf(block_sum(v * v)) * 0.2f;
    v = fminf(v, thr);
    const float nrm = 512.f / fmaxf(sqrtf(block_sum(v * v)), FLT_EPSILON);
    des[q * 128 + tid] = (uint8_t)min(255, max(0, __float2int_rn(v * nrm)));
  }
}

// The Gaussian pyramids of `frames` images (frame_stride bytes apart) into the workspace, one launch per level.
// The arguments of each pyramid launch, for frames of one size (UniformSteps) or of any size (MixedSteps).
struct UniformSteps {
  const uint8_t* gray;
  int width, height;
  int64_t pitch, frame_stride;
  Pyramid P;
  UniformUpsample upsample() const {
    return {gray, width, height, pitch, frame_stride, P.level(0, 1), P.fstride};
  }
  UniformStep step(int oi, int li, int oo, int lo) const {
    return {P.level(oi, li), P.level(oo, lo), P.w[oi], P.h[oi], P.w[oo], P.h[oo], P.fstride};
  }
};

struct MixedSteps {
  Mixed M;
  MixedStep upsample() const { return {M, -1, 0, 0, 1}; }
  MixedStep step(int oi, int li, int oo, int lo) const { return {M, oi, li, oo, lo}; }
};

// The Gaussian pyramids of `frames` images into the workspace, one launch per level for all frames; grid holds
// the launch sizes (per octave the largest frame's).
template <class Steps>
int build_pyramid(const Steps& s, const Pyramid& grid, int frames, cudaStream_t st) {
  double sig[kLevels];
  const double k = std::pow(2., 1. / kLayers);
  for (int i = 1; i < kLevels; ++i) {
    const double prev = std::pow(k, (double)(i - 1)) * kSigma, total = prev * k;
    sig[i] = std::sqrt(total * total - prev * prev);
  }
  Taps taps[kLevels];
  const float sig_diff = sqrtf(fmaxf(kSigma * kSigma - 0.5f * 0.5f * 4, 0.01f));
  if (!gaussian_taps(sig_diff, &taps[0])) return SOD_ERR_UNSUPPORTED;
  for (int i = 1; i < kLevels; ++i)
    if (!gaussian_taps(sig[i], &taps[i])) return SOD_ERR_UNSUPPORTED;
  const dim3 pb(32, 8);
  auto pgrid = [&](int w, int h) { return dim3((w + 31) / 32, (h + 7) / 8, frames); };
  auto tgrid = [&](int w, int h) { return dim3((w + kTile - 1) / kTile, (h + kTile - 1) / kTile, frames); };
  const Pyramid& P = grid;
  // the doubled image goes to level 1's slot, blurred into level 0, and level 1 is then computed over it
  sift_upsample_kernel<<<pgrid(P.w[0], P.h[0]), pb, 0, st>>>(s.upsample());
  sift_blur_kernel<<<tgrid(P.w[0], P.h[0]), 256, 0, st>>>(s.step(0, 1, 0, 0), taps[0]);
  for (int o = 0; o < P.n_oct; ++o) {
    if (o > 0) sift_halve_kernel<<<pgrid(P.w[o], P.h[o]), pb, 0, st>>>(s.step(o - 1, kLayers, o, 0));
    for (int l = 1; l < kLevels; ++l)
      sift_blur_kernel<<<tgrid(P.w[o], P.h[o]), 256, 0, st>>>(s.step(o, l - 1, o, l), taps[l]);
  }
  SOD_CHECK_LAUNCH("sift pyramid");
  return SOD_OK;
}

// Pyramids, detection, order, duplicate removal, rows and descriptors of p.frames images: the whole of
// sod_sift_extract, sod_sift_extract_batch and sod_sift_extract_mixed after their argument checks (and, for a mixed
// batch, its geometry table).  lay reads the pyramids, steps builds them, p.pyr sizes the launches.  Never
// synchronises.
template <class L, class Steps>
int extract_frames(const L& lay, const Steps& steps, const Plan& p, int64_t max_per_frame, const Rows& out,
                   void* workspace, cudaStream_t st) {
  char* ws = (char*)workspace;
  const int cap = (int)p.cap, frames = p.frames, slots = frames * cap;
  int32_t* counters = (int32_t*)(ws + p.counters);
  int32_t* batch = counters + kFrameInts * frames;
  Cand* cand = (Cand*)(ws + p.cand);
  Kp* raw = (Kp*)(ws + p.raw);
  uint64_t* keys_in = (uint64_t*)(ws + p.keys_in);
  uint64_t* keys_out = (uint64_t*)(ws + p.keys_out);
  int32_t* vals_in = (int32_t*)(ws + p.vals_in);
  int32_t* vals_out = (int32_t*)(ws + p.vals_out);
  int32_t* keep = (int32_t*)(ws + p.keep);
  int32_t* pos = (int32_t*)(ws + p.pos);
  SOD_CHECK_CUDA(cudaMemsetAsync(counters, 0, (kFrameInts * frames + kBatchInts) * sizeof(int32_t), st));
  const int sms = device_sm_count();
  if (sms < 0) return SOD_ERR_CUDA;
  if (p.pyr.n_oct > 0) {
    if (int rc = build_pyramid(steps, p.pyr, frames, st)) return rc;
    for (int o = 0; o < p.pyr.n_oct; ++o) {
      const int iw = p.pyr.w[o] - 2 * kBorder, ih = p.pyr.h[o] - 2 * kBorder;
      if (iw <= 0 || ih <= 0) continue;
      sift_extrema_kernel<<<dim3((iw + 31) / 32, (ih + 7) / 8, kLayers * frames), dim3(32, 8), 0, st>>>(
          lay, o, cand, cap, counters);
    }
    SOD_CHECK_LAUNCH("sift_extrema_kernel");
    // sms * 8 blocks in all, as for one frame, split over the frames' slabs
    sift_orient_kernel<<<dim3((sms * 8 + frames - 1) / frames, frames), 32 * kOriWarps, 0, st>>>(lay, cand, cap,
                                                                                             counters, raw);
    SOD_CHECK_LAUNCH("sift_orient_kernel");
  }
  const int blocks = (slots + 255) / 256;
  sift_sort_keys_kernel<<<blocks, 256, 0, st>>>(raw, counters, cap, slots, keys_in, vals_in);
  SOD_CHECK_LAUNCH("sift_sort_keys_kernel");
  size_t tmp = p.cub_bytes;
  SOD_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(ws + p.cub_tmp, tmp, keys_in, keys_out, vals_in, vals_out, slots, 0,
                                                 64, st));
  int32_t* vals = vals_out;
  if (frames > 1) {
    uint32_t* fkeys_in = (uint32_t*)keys_in;      // keys_in is free after the first sort: 2 x slots u32
    uint32_t* fkeys_out = fkeys_in + slots;
    sift_frame_keys_kernel<<<blocks, 256, 0, st>>>(vals_out, cap, slots, fkeys_in);
    SOD_CHECK_LAUNCH("sift_frame_keys_kernel");
    int bits = 0;
    while ((1 << bits) < frames) ++bits;
    tmp = p.cub_bytes;
    SOD_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(ws + p.cub_tmp, tmp, fkeys_in, fkeys_out, vals_out, vals_in, slots,
                                                   0, bits, st));
    vals = vals_in;
  }
  sift_sort_runs_kernel<<<blocks, 256, 0, st>>>(raw, counters, cap, slots, vals);
  sift_keep_kernel<<<blocks, 256, 0, st>>>(raw, counters, cap, slots, vals, keep);
  SOD_CHECK_LAUNCH("sift_keep_kernel");
  tmp = p.cub_bytes;
  SOD_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(ws + p.cub_tmp, tmp, keep, pos, slots, st));
  sift_frame_rows_kernel<<<1, 256, 0, st>>>(keep, pos, counters, cap, frames, max_per_frame, out, batch);
  sift_emit_kernel<<<blocks, 256, 0, st>>>(raw, cap, slots, vals, keep, pos, out);
  SOD_CHECK_LAUNCH("sift_emit_kernel");
  if (p.pyr.n_oct > 0) {
    sift_descriptor_kernel<<<sms * 16, 128, 0, st>>>(lay, out.xy, out.size, out.angle, out.octave, out.frame,
                                                     out.cap_rows, batch, out.des, nullptr);
    SOD_CHECK_LAUNCH("sift_descriptor_kernel");
  }
  return SOD_OK;
}

// extract_frames of `frames` images of one size, image f at gray + f x frame_stride.
int extract_uniform(const uint8_t* gray, int width, int height, int64_t pitch, int64_t frame_stride, Plan& p,
                    int64_t max_per_frame, const Rows& out, void* workspace, cudaStream_t st) {
  p.pyr.base = (float*)workspace;
  return extract_frames(p.pyr, UniformSteps{gray, width, height, pitch, frame_stride, p.pyr}, p, max_per_frame, out,
                        workspace, st);
}

// Copies the geometry table of a mixed batch from the kernel parameter into the workspace, so that the call
// needs no host-to-device copy and stays capturable.  One block.
__global__ void sift_mixed_setup_kernel(const __grid_constant__ MixedTable t, int frames, FrameGeom* __restrict__ g) {
  static_assert(sizeof(FrameGeom) % sizeof(int) == 0, "FrameGeom is copied as ints");
  const int n = frames * (int)(sizeof(FrameGeom) / sizeof(int));
  const int* src = (const int*)t.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) ((int*)g)[i] = src[i];
}

int check_image(const uint8_t* gray, int32_t width, int32_t height, int64_t pitch, const char* fn) {
  SOD_CHECK_ARG(width >= 1 && height >= 1 && width <= kMaxSide && height <= kMaxSide,
                "%s: image size %dx%d out of range (1..%d a side)", fn, width, height, kMaxSide);
  SOD_CHECK_ARG(pitch >= width, "%s: pitch %lld < width %d", fn, (long long)pitch, width);
  SOD_CHECK_ARG(gray != nullptr, "%s: null image", fn);
  return SOD_OK;
}

int check_batch_out(const sod_sift_batch_out* out, int32_t frames, const char* fn) {
  SOD_CHECK_ARG(out != nullptr, "%s: null out", fn);
  SOD_CHECK_ARG(out->cap_per_frame >= 1 && out->cap_per_frame <= SOD_SIFT_MAX_CAP &&
                    frames * out->cap_per_frame <= SOD_SIFT_MAX_CAP,
                "%s: cap_per_frame %lld out of range (1..%d / frames)", fn, (long long)out->cap_per_frame,
                SOD_SIFT_MAX_CAP);
  SOD_CHECK_ARG(out->cap_rows >= 1 && out->cap_rows <= SOD_SIFT_MAX_CAP, "%s: cap_rows %lld out of range (1..%d)",
                fn, (long long)out->cap_rows, SOD_SIFT_MAX_CAP);
  SOD_CHECK_ARG(out->xy && out->size && out->angle && out->response && out->octave && out->des && out->frame &&
                    out->count && out->offset && out->overflow && out->rows_overflow,
                "%s: null output array", fn);
  return SOD_OK;
}

Rows batch_rows(const sod_sift_batch_out* out) {
  return Rows{out->xy,    out->size,  out->angle,  out->response,   out->octave, out->des,
              out->frame, out->count, out->offset, out->overflow, out->rows_overflow, out->cap_rows};
}

}  // namespace
}  // namespace sod

using namespace sod;

extern "C" {

size_t sod_sift_batch_workspace_bytes(int32_t width, int32_t height, int32_t frames, int64_t cap_per_frame) {
  Plan p;
  if (width < 1 || height < 1 || width > kMaxSide || height > kMaxSide || frames < 1 ||
      frames > SOD_SIFT_MAX_FRAMES || cap_per_frame < 0 || cap_per_frame > SOD_SIFT_MAX_CAP ||
      frames * cap_per_frame > SOD_SIFT_MAX_CAP || !make_plan(width, height, frames, cap_per_frame, &p))
    return 0;
  return p.total;
}

size_t sod_sift_workspace_bytes(int32_t width, int32_t height, int64_t max_keypoints) {
  return sod_sift_batch_workspace_bytes(width, height, 1, max_keypoints);
}

int64_t sod_sift_level_offset(int32_t width, int32_t height, int32_t octave, int32_t level, int32_t* wh_host) {
  Plan p;
  if (width < 1 || height < 1 || width > kMaxSide || height > kMaxSide || !make_plan(width, height, 1, 0, &p) ||
      octave < -1 || octave + 1 >= p.pyr.n_oct || level < 0 || level >= kLevels) {
    set_error("sod_sift_level_offset: no level %d of octave %d for a %dx%d image", level, octave, width, height);
    return -1;
  }
  if (wh_host) {
    wh_host[0] = p.pyr.w[octave + 1];
    wh_host[1] = p.pyr.h[octave + 1];
  }
  const int o = octave + 1;
  return (p.pyr.off[o] + (int64_t)level * p.pyr.w[o] * p.pyr.h[o]) * (int64_t)sizeof(float);
}

int sod_sift_extract(const uint8_t* gray, int32_t width, int32_t height, int64_t pitch, const sod_sift_out* out,
                     void* workspace, size_t workspace_bytes, sod_stream_t stream) {
  if (int rc = check_image(gray, width, height, pitch, "sod_sift_extract")) return rc;
  SOD_CHECK_ARG(out != nullptr, "sod_sift_extract: null out");
  SOD_CHECK_ARG(out->cap >= 1 && out->cap <= SOD_SIFT_MAX_CAP, "sod_sift_extract: cap %lld out of range (1..%d)",
                (long long)out->cap, SOD_SIFT_MAX_CAP);
  SOD_CHECK_ARG(out->xy && out->size && out->angle && out->response && out->octave && out->des && out->counters,
                "sod_sift_extract: null output array");
  Plan p;
  SOD_CHECK_ARG(make_plan(width, height, 1, out->cap, &p), "sod_sift_extract: too many octaves");
  SOD_CHECK_ARG(workspace != nullptr && workspace_bytes >= p.total && ((uintptr_t)workspace & 255) == 0,
                "sod_sift_extract: workspace of %zu bytes at %p; need %zu bytes, 256-byte aligned", workspace_bytes,
                workspace, p.total);
  // the batch of one: count and overflow land in out->counters, the frame's offset (0) in the workspace
  const Rows rows{out->xy,       out->size,         out->angle,  out->response,
                  out->octave,   out->des,          nullptr,     out->counters,
                  (int32_t*)((char*)workspace + p.offset), out->counters + 1, nullptr, out->cap};
  return extract_uniform(gray, width, height, pitch, (int64_t)pitch * height, p, 0, rows, workspace,
                        (cudaStream_t)stream);
}

int sod_sift_extract_batch(const uint8_t* gray, int32_t width, int32_t height, int64_t pitch, int64_t frame_stride,
                           int32_t frames, int64_t max_per_frame, const sod_sift_batch_out* out, void* workspace,
                           size_t workspace_bytes, sod_stream_t stream) {
  const char* fn = "sod_sift_extract_batch";
  if (int rc = check_image(gray, width, height, pitch, fn)) return rc;
  SOD_CHECK_ARG(frames >= 1 && frames <= SOD_SIFT_MAX_FRAMES, "%s: frames %d out of range (1..%d)", fn, frames,
                SOD_SIFT_MAX_FRAMES);
  SOD_CHECK_ARG(frame_stride >= pitch * height, "%s: frame_stride %lld < pitch x height %lld", fn,
                (long long)frame_stride, (long long)(pitch * height));
  SOD_CHECK_ARG(max_per_frame >= 0, "%s: max_per_frame %lld < 0", fn, (long long)max_per_frame);
  if (int rc = check_batch_out(out, frames, fn)) return rc;
  Plan p;
  SOD_CHECK_ARG(make_plan(width, height, frames, out->cap_per_frame, &p), "%s: too many octaves", fn);
  SOD_CHECK_ARG(workspace != nullptr && workspace_bytes >= p.total && ((uintptr_t)workspace & 255) == 0,
                "%s: workspace of %zu bytes at %p; need %zu bytes, 256-byte aligned", fn, workspace_bytes, workspace,
                p.total);
  return extract_uniform(gray, width, height, pitch, frame_stride, p, max_per_frame, batch_rows(out), workspace,
                        (cudaStream_t)stream);
}

int sod_sift_describe(const uint8_t* gray, int32_t width, int32_t height, int64_t pitch, const float* xy,
                      const float* size, const float* angle, const int32_t* octave, int64_t n, uint8_t* des,
                      int32_t* n_invalid, void* workspace, size_t workspace_bytes, sod_stream_t stream) {
  if (int rc = check_image(gray, width, height, pitch, "sod_sift_describe")) return rc;
  SOD_CHECK_ARG(n >= 0 && n <= SOD_SIFT_MAX_CAP, "sod_sift_describe: n %lld out of range (0..%d)", (long long)n,
                SOD_SIFT_MAX_CAP);
  if (n == 0) return SOD_OK;
  SOD_CHECK_ARG(xy && size && angle && octave && des, "sod_sift_describe: null keypoint or descriptor array");
  Plan p;
  SOD_CHECK_ARG(make_plan(width, height, 1, 0, &p), "sod_sift_describe: too many octaves");
  SOD_CHECK_ARG(workspace != nullptr && workspace_bytes >= p.total && ((uintptr_t)workspace & 255) == 0,
                "sod_sift_describe: workspace of %zu bytes at %p; need %zu bytes, 256-byte aligned", workspace_bytes,
                workspace, p.total);
  cudaStream_t st = (cudaStream_t)stream;
  p.pyr.base = (float*)workspace;
  if (p.pyr.n_oct > 0)
    if (int rc = build_pyramid(UniformSteps{gray, width, height, pitch, (int64_t)pitch * height, p.pyr}, p.pyr, 1, st))
      return rc;
  const int sms = device_sm_count();
  if (sms < 0) return SOD_ERR_CUDA;
  sift_descriptor_kernel<<<sms * 16, 128, 0, st>>>(p.pyr, xy, size, angle, octave, nullptr, n, nullptr, des,
                                                   n_invalid);
  SOD_CHECK_LAUNCH("sift_descriptor_kernel");
  return SOD_OK;
}

size_t sod_sift_mixed_workspace_bytes(const int32_t* wh_host, int32_t frames, int64_t cap_per_frame) {
  if (wh_host == nullptr || frames < 1 || frames > SOD_SIFT_MAX_MIXED_FRAMES || cap_per_frame < 0 ||
      cap_per_frame > SOD_SIFT_MAX_CAP || frames * cap_per_frame > SOD_SIFT_MAX_CAP)
    return 0;
  for (int f = 0; f < frames; ++f)
    if (wh_host[2 * f] < 1 || wh_host[2 * f + 1] < 1 || wh_host[2 * f] > kMaxSide || wh_host[2 * f + 1] > kMaxSide)
      return 0;
  Plan p;
  MixedTable t;
  return make_mixed_plan(wh_host, frames, cap_per_frame, &p, &t) ? p.total : 0;
}

int sod_sift_extract_mixed(const uint8_t* const* images_host, const int32_t* wh_host, const int64_t* pitch_host,
                           int32_t frames, int64_t max_per_frame, const sod_sift_batch_out* out, void* workspace,
                           size_t workspace_bytes, sod_stream_t stream) {
  const char* fn = "sod_sift_extract_mixed";
  SOD_CHECK_ARG(images_host && wh_host && pitch_host, "%s: null image, size or pitch array", fn);
  SOD_CHECK_ARG(frames >= 1 && frames <= SOD_SIFT_MAX_MIXED_FRAMES, "%s: frames %d out of range (1..%d)", fn, frames,
                SOD_SIFT_MAX_MIXED_FRAMES);
  char what[64];
  for (int f = 0; f < frames; ++f) {
    snprintf(what, sizeof what, "%s: frame %d", fn, f);
    if (int rc = check_image(images_host[f], wh_host[2 * f], wh_host[2 * f + 1], pitch_host[f], what)) return rc;
  }
  SOD_CHECK_ARG(max_per_frame >= 0, "%s: max_per_frame %lld < 0", fn, (long long)max_per_frame);
  if (int rc = check_batch_out(out, frames, fn)) return rc;
  Plan p;
  MixedTable t;
  SOD_CHECK_ARG(make_mixed_plan(wh_host, frames, out->cap_per_frame, &p, &t), "%s: too many octaves", fn);
  SOD_CHECK_ARG(workspace != nullptr && workspace_bytes >= p.total && ((uintptr_t)workspace & 255) == 0,
                "%s: workspace of %zu bytes at %p; need %zu bytes, 256-byte aligned", fn, workspace_bytes, workspace,
                p.total);
  for (int f = 0; f < frames; ++f) {
    t.f[f].img = images_host[f];
    t.f[f].pitch = pitch_host[f];
  }
  cudaStream_t st = (cudaStream_t)stream;
  FrameGeom* g = (FrameGeom*)((char*)workspace + p.geom);
  sift_mixed_setup_kernel<<<1, 256, 0, st>>>(t, frames, g);
  SOD_CHECK_LAUNCH("sift_mixed_setup_kernel");
  const Mixed M{(float*)workspace, g, frames};
  return extract_frames(M, MixedSteps{M}, p, max_per_frame, batch_rows(out), workspace, st);
}

}  // extern "C"
