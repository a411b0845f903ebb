// The steps either side of the path on the device (SURVEY.md 8(f) rows 1-2):
//   * cdn_warp_affine_u8_batch -- the image transform of BaseDetector.pre_process (lib/detectors/base_detector.py:48-76):
//     cv2.warpAffine(resized, trans_input, (inp_w, inp_h), flags=cv2.INTER_LINEAR) on raw uint8 HWC images, bit for bit
//     (OpenCV's fixed-point scheme: coordinates in 1/1024 pixel rounded to 1/32, 15-bit bilinear weights, constant border 0),
//     optionally with the mirrored copy --flip_test appends (:69-70), for a ragged batch: source frames of different sizes
//     back to back in one byte pool, one descriptor per output image.  cdn_warp_affine_u8 is its one-descriptor case.  At
//     test scale 1 the cv2.resize in front of it is the identity, so the raw frame goes to the device as it is and the
//     normalisation happens in the stem kernel's 3 x 256 table.
//   * cdn_warp_affine_u8_f32_batch -- the same warp for the unquantised model, whose network takes normalised fp32 NCHW: every
//     warped byte goes through a 3 x 256 fp32 table (the normalisation of BaseDetector.pre_process, :66-68, is a function of
//     the byte and its channel) and is written in planes.  Both kernels call one interpolation function, so the fp32 output is
//     the u8 kernel's output looked up, by construction.
//   * cdn_warp_affine_src_u8_batch / cdn_warp_affine_src_u8_f32_batch -- the same two warps from frames anywhere in device memory
//     (absolute plane addresses, row pitches): BGR, or YUV 4:2:0 (I420, YV12, NV12, NV21) converted to BGR tap by tap with
//     OpenCV's COLOR_YUV2BGR_* arithmetic, so that each output is cv2.warpAffine(cv2.cvtColor(frame, COLOR_YUV2BGR_*), ...).
//   * cdn_ctdet_group_by_class -- the per-class grouping of ctdet_post_process (lib/utils/post_process.py:86-103): detections
//     [B][K][6] reordered by class (stable, i.e. by descending score inside a class) + per-class counts, so the host only
//     slices views.
#include "common.cuh"
#include <algorithm>
#include <cstddef>

// one output image: its source frame in the pool and the INVERSE (destination -> source) matrix
struct WarpDesc { long long off; int H, W; double m[6]; int dst, mirror; };
static_assert(sizeof(WarpDesc) == 72, "WarpDesc layout");

constexpr int WARP_THREADS = 128;
constexpr int WARP_PX = 4;                          // output pixels per thread: 12 bytes = three 32-bit words
// descriptors per launch: the kernel parameter space holds 32764 bytes (CUDA 12.1+), the rest of the struct is 24
constexpr int WARP_MAX_DESC = (32764 - 32) / (int)sizeof(WarpDesc);
static_assert(WARP_MAX_DESC == CDN_WARP_DESC_PER_LAUNCH, "include/codenet_b200.h states the descriptors per launch");
static_assert(sizeof(cdn_warp_desc) == 72, "cdn_warp_desc layout (codenet_b200._lib.WARP_DESC)");
struct WarpBatchParams { const uint8_t* pool; uint8_t* dst; int dh, dw, groups, pad; WarpDesc d[WARP_MAX_DESC]; };
static_assert(sizeof(WarpBatchParams) <= 32764, "kernel parameters exceed 32764 bytes");
// the fp32 variant: 40 bytes of header, then per descriptor its WarpDesc and the one-byte index of its normalisation table
constexpr int WARP_F32_MAX_DESC = (32764 - 40) / (int)(sizeof(WarpDesc) + sizeof(uint8_t));
static_assert(WARP_F32_MAX_DESC == CDN_WARP_F32_DESC_PER_LAUNCH, "include/codenet_b200.h states the descriptors per launch");
struct WarpF32Params {
  const uint8_t* pool; float* dst; const float* tables; int dh, dw, groups, vec;
  WarpDesc d[WARP_F32_MAX_DESC]; uint8_t table[WARP_F32_MAX_DESC];
};
static_assert(offsetof(WarpF32Params, d) == 40, "WarpF32Params header");
static_assert(sizeof(WarpF32Params) <= 32764, "kernel parameters exceed 32764 bytes");
// cdn_warp_src_desc on the device: absolute plane addresses, row pitches, the INVERSE matrix
struct WarpSrcDesc { const uint8_t* p[3]; long long pitch[2]; double m[6]; int H, W, kind, step, dst, mirror; };
static_assert(sizeof(WarpSrcDesc) == 112, "WarpSrcDesc layout");
static_assert(sizeof(cdn_warp_src_desc) == 112, "cdn_warp_src_desc layout (codenet_b200._lib.WARP_SRC_DESC)");
// the general-source variants: 24 (u8) and 32 (fp32: 289 table bytes follow the descriptors) bytes of header
constexpr int WARP_SRC_MAX_DESC = (32764 - 24) / (int)sizeof(WarpSrcDesc);
static_assert(WARP_SRC_MAX_DESC == CDN_WARP_SRC_DESC_PER_LAUNCH, "include/codenet_b200.h states the descriptors per launch");
struct WarpSrcParams { uint8_t* dst; int dh, dw, groups, pad; WarpSrcDesc d[WARP_SRC_MAX_DESC]; };
static_assert(offsetof(WarpSrcParams, d) == 24 && sizeof(WarpSrcParams) <= 32764, "WarpSrcParams");
constexpr int WARP_SRC_F32_MAX_DESC = (32764 - 32) / (int)(sizeof(WarpSrcDesc) + sizeof(uint8_t));
static_assert(WARP_SRC_F32_MAX_DESC == CDN_WARP_SRC_F32_DESC_PER_LAUNCH, "include/codenet_b200.h states the descriptors per launch");
struct WarpSrcF32Params {
  float* dst; const float* tables; int dh, dw, groups, vec;
  WarpSrcDesc d[WARP_SRC_F32_MAX_DESC]; uint8_t table[WARP_SRC_F32_MAX_DESC];
};
static_assert(offsetof(WarpSrcF32Params, d) == 32 && sizeof(WarpSrcF32Params) <= 32764, "WarpSrcF32Params");
// cdn_warp_rs_desc on the device: the warp sees an H x W image (the resized size), read from an FH x FW frame
struct WarpRsDesc { const uint8_t* p[3]; long long pitch[2]; double m[6]; double scale[2]; int H, W, FH, FW, kind, step, dst, mirror; };
static_assert(sizeof(WarpRsDesc) == 136, "WarpRsDesc layout");
static_assert(sizeof(cdn_warp_rs_desc) == 136, "cdn_warp_rs_desc layout (codenet_b200._lib.WARP_RS_DESC)");
constexpr int WARP_RS_MAX_DESC = (32764 - 24) / (int)sizeof(WarpRsDesc);
static_assert(WARP_RS_MAX_DESC == CDN_WARP_RS_DESC_PER_LAUNCH, "include/codenet_b200.h states the descriptors per launch");
struct WarpRsParams { uint8_t* dst; int dh, dw, groups, pad; WarpRsDesc d[WARP_RS_MAX_DESC]; };
static_assert(offsetof(WarpRsParams, d) == 24 && sizeof(WarpRsParams) <= 32764, "WarpRsParams");
constexpr int WARP_RS_F32_MAX_DESC = (32764 - 32) / (int)(sizeof(WarpRsDesc) + sizeof(uint8_t));
static_assert(WARP_RS_F32_MAX_DESC == CDN_WARP_RS_F32_DESC_PER_LAUNCH, "include/codenet_b200.h states the descriptors per launch");
struct WarpRsF32Params {
  float* dst; const float* tables; int dh, dw, groups, vec;
  WarpRsDesc d[WARP_RS_F32_MAX_DESC]; uint8_t table[WARP_RS_F32_MAX_DESC];
};
static_assert(offsetof(WarpRsF32Params, d) == 32 && sizeof(WarpRsF32Params) <= 32764, "WarpRsF32Params");

// cv::warpAffine's inversion of the 2 x 3 matrix (imgwarp.cpp), in double on the host: the same expressions on the device
// would be contracted into FMAs and could round differently
static void warp_invert(const double* M6, double* m) {
  for (int i = 0; i < 6; ++i) m[i] = M6[i];
  double D = m[0] * m[4] - m[1] * m[3];
  D = D != 0 ? 1. / D : 0;
  const double A11 = m[4] * D, A22 = m[0] * D;
  m[0] = A11; m[1] *= -D; m[3] *= -D; m[4] = A22;
  const double b1 = -m[0] * m[2] - m[1] * m[5], b2 = -m[3] * m[2] - m[4] * m[5];
  m[2] = b1; m[5] = b2;
}

__device__ __forceinline__ void warp_store(uint8_t* d, const uint8_t (&v)[WARP_PX * 3], int n) {
  if (n == WARP_PX && ((uintptr_t)d & 3) == 0) {
    uint32_t w[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) w[i] = v[4 * i] | (v[4 * i + 1] << 8) | (v[4 * i + 2] << 16) | ((uint32_t)v[4 * i + 3] << 24);
    uint32_t* d32 = reinterpret_cast<uint32_t*>(d);
    d32[0] = w[0]; d32[1] = w[1]; d32[2] = w[2];
  } else {
#pragma unroll
    for (int i = 0; i < WARP_PX * 3; ++i)
      if (i < n * 3) d[i] = v[i];
  }
}

// How warp_pixels reads a tap: tap(yy, xx, w, acc) adds w x channel c (B, G, R) of source pixel (yy, xx), which lies inside the
// frame, to acc[c].  PoolBgr: a uint8 BGR HWC frame of rows exactly 3W bytes long (cdn_warp_desc); PitchedBgr: the same with any row pitch;
// Yuv420: Y, U and V planes of 4:2:0 video, converted per tap by OpenCV's COLOR_YUV2BGR_* (color_yuv.simd.hpp: BT.601 video
// range, 20-bit fixed point), so that interpolating the converted taps is cv2.warpAffine(cv2.cvtColor(frame), ...) exactly.
struct PoolBgr {
  const uint8_t* src; const WarpDesc& q;
  __device__ __forceinline__ void operator()(int yy, int xx, int w, int (&acc)[3]) const {
    const uint8_t* s = src + ((size_t)yy * q.W + xx) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) acc[c] += (int)__ldg(s + c) * w;
  }
};
struct PitchedBgr {
  const uint8_t* src; long long pitch;
  __device__ __forceinline__ void operator()(int yy, int xx, int w, int (&acc)[3]) const {
    const uint8_t* s = src + (size_t)yy * pitch + (size_t)xx * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) acc[c] += (int)__ldg(s + c) * w;
  }
};
constexpr int YUV_CY = 1220542, YUV_CUB = 2116026, YUV_CUG = -409993, YUV_CVG = -852492, YUV_CVR = 1673527, YUV_SHIFT = 20;
struct Yuv420 {
  const uint8_t *y, *u, *v; long long pitch, chroma_pitch; int step;
  __device__ __forceinline__ void operator()(int yy, int xx, int w, int (&acc)[3]) const {
    const size_t c = (size_t)(yy >> 1) * chroma_pitch + (size_t)(xx >> 1) * step;
    const int U = (int)__ldg(u + c) - 128, V = (int)__ldg(v + c) - 128;
    // |each sum| < 2^30: int32 is exact, and >> is the arithmetic shift OpenCV's int arithmetic uses
    const int l = max((int)__ldg(y + (size_t)yy * pitch + xx) - 16, 0) * YUV_CY + (1 << (YUV_SHIFT - 1));
    acc[0] += min(max((l + YUV_CUB * U) >> YUV_SHIFT, 0), 255) * w;
    acc[1] += min(max((l + YUV_CVG * V + YUV_CUG * U) >> YUV_SHIFT, 0), 255) * w;
    acc[2] += min(max((l + YUV_CVR * V) >> YUV_SHIFT, 0), 255) * w;
  }
};

// cv2.resize's INTER_LINEAR coefficients of destination index d for 8-bit images (resize.cpp): the two source indices s0, s1
// (clipped into [0, n)) and their 11-bit weights c0, c1.  fx = float((d + 0.5) * scale - 0.5) in OpenCV's rounding order (the
// intrinsics keep nvcc from contracting into FMAs), floor, the fraction, then saturate_cast<short>, which rounds half to even.
// Columns (clamp) left of the frame or past its last pixel take that pixel at full weight; rows keep their fraction even there,
// so an upscale's first and last rows read one row twice with two truncating products (DESIGN.md section 9).
__device__ __forceinline__ void resize_coef(int d, double scale, int n, bool clamp, int& s0, int& s1, int& c0, int& c1) {
  float f = __double2float_rn(__dadd_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), -0.5));
  const float fl = floorf(f);
  int s = (int)fl;
  f = __fsub_rn(f, fl);
  if (clamp && (s < 0 || s >= n - 1)) {
    s = min(max(s, 0), n - 1);
    f = 0.f;
  }
  c0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
  c1 = __float2int_rn(__fmul_rn(f, 2048.f));
  s0 = min(max(s, 0), n - 1);
  s1 = min(max(s + 1, 0), n - 1);
}

// A tap of the resized image: pixel (yy, xx) of cv2.resize(frame, (rs_w, rs_h)) from four frame pixels read by Src, with
// OpenCV's passes: exact horizontal sums S = p0 * a0 + p1 * a1 (< 2^20), then (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >>
// 16) + 2) >> 2 (every product < 2^27).  Each frame pixel goes through Src as it is, so a YUV frame is converted before it is
// resized, as cv2.resize(cv2.cvtColor(frame, ...)) sees it.
template <class Src>
struct Resized {
  Src src; int H, W; double sx, sy;                  // the frame's size; 1 / (rs_w / W), 1 / (rs_h / H)
  __device__ __forceinline__ void operator()(int yy, int xx, int w, int (&acc)[3]) const {
    int x0, x1, a0, a1, y0, y1, b0, b1;
    resize_coef(xx, sx, W, true, x0, x1, a0, a1);
    resize_coef(yy, sy, H, false, y0, y1, b0, b1);
    int s0[3] = {0, 0, 0}, s1[3] = {0, 0, 0};
    src(y0, x0, a0, s0); src(y0, x1, a1, s0);
    src(y1, x0, a0, s1); src(y1, x1, a1, s1);
#pragma unroll
    for (int c = 0; c < 3; ++c) acc[c] += min((((b0 * (s0[c] >> 4)) >> 16) + ((b1 * (s1[c] >> 4)) >> 16) + 2) >> 2, 255) * w;
  }
};

// OpenCV's fixed-point bilinear interpolation of WARP_PX consecutive destination pixels (y, x0 .. x0 + WARP_PX - 1) of one
// H x W source through the inverse matrix m, the one every warp kernel calls: v[i * 3 + c] = channel c of pixel x0 + i (a pixel
// past the row's end is computed like the others and left unstored by the caller).  Tap reads a source pixel (PoolBgr, ...).
template <class Desc, class Tap>
__device__ __forceinline__ void warp_pixels(const Desc& q, const Tap& tap3, int y, int x0, uint8_t (&v)[WARP_PX * 3]) {
  // dst -> src map in 1/1024 pixel, as OpenCV forms it: per-column and per-row terms are rounded SEPARATELY, then summed;
  // the row term is m1 * y + m2 in two roundings (no FMA), like OpenCV's and numpy's double arithmetic
  const int X0 = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(q.m[1], (double)y), q.m[2]), 1024.0)) + 16;
  const int Y0 = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(q.m[4], (double)y), q.m[5]), 1024.0)) + 16;
#pragma unroll
  for (int i = 0; i < WARP_PX; ++i) {
    const int x = x0 + i;
    const int adelta = __double2int_rn(__dmul_rn(__dmul_rn(q.m[0], (double)x), 1024.0));
    const int bdelta = __double2int_rn(__dmul_rn(__dmul_rn(q.m[3], (double)x), 1024.0));
    const int X = (X0 + adelta) >> 5, Y = (Y0 + bdelta) >> 5;
    const int sx = min(max(X >> 5, -32768), 32767), sy = min(max(Y >> 5, -32768), 32767);
    const int fx = X & 31, fy = Y & 31;
    const int w00 = (32 - fy) * (32 - fx) * 32, w01 = (32 - fy) * fx * 32, w10 = fy * (32 - fx) * 32, w11 = fy * fx * 32;
    int acc[3] = {0, 0, 0};
    auto tap = [&](int yy, int xx, int w) {
      if ((unsigned)yy < (unsigned)q.H && (unsigned)xx < (unsigned)q.W) tap3(yy, xx, w, acc);
    };
    tap(sy, sx, w00); tap(sy, sx + 1, w01); tap(sy + 1, sx, w10); tap(sy + 1, sx + 1, w11);
#pragma unroll
    for (int c = 0; c < 3; ++c) v[i * 3 + c] = (uint8_t)min(max((acc[c] + (1 << 14)) >> 15, 0), 255);
  }
}

// grid (tiles of WARP_THREADS x WARP_PX pixels over the flattened dst_h x dst_w image, descriptors of this launch)
__global__ void __launch_bounds__(WARP_THREADS) warp_affine_u8_kernel(const __grid_constant__ WarpBatchParams p) {
  const WarpDesc& q = p.d[blockIdx.y];
  const int t = blockIdx.x * WARP_THREADS + threadIdx.x;
  const int y = t / p.groups, x0 = (t - y * p.groups) * WARP_PX;
  if (y >= p.dh) return;
  const int n = min(WARP_PX, p.dw - x0);
  uint8_t v[WARP_PX * 3];
  warp_pixels(q, PoolBgr{p.pool + q.off, q}, y, x0, v);
  const size_t plane = (size_t)p.dh * p.dw * 3, row = (size_t)y * p.dw * 3;
  warp_store(p.dst + (size_t)q.dst * plane + row + (size_t)x0 * 3, v, n);
  if (q.mirror >= 0) {                               // the n pixels reversed, ending at column dw - 1 - x0
    uint8_t f[WARP_PX * 3];
#pragma unroll
    for (int i = 0; i < WARP_PX; ++i)
#pragma unroll
      for (int c = 0; c < 3; ++c) f[i * 3 + c] = v[(WARP_PX - 1 - i) * 3 + c];
    uint8_t* m = p.dst + (size_t)q.mirror * plane + row + (size_t)(p.dw - x0 - n) * 3;
    if (n == WARP_PX) {
      warp_store(m, f, n);
    } else {
      const int skip = (WARP_PX - n) * 3;
#pragma unroll
      for (int i = 0; i < WARP_PX * 3; ++i)
        if (i >= skip) m[i - skip] = f[i];
    }
  }
}

// The same pixels through a 3 x 256 table into fp32 NCHW: element (slot, c, y, x) = table[c][byte the u8 kernel writes at
// (slot, y, x, c)].  The descriptor's table is staged in shared memory; with vec (dst_w % 4 == 0, 16-byte-aligned dst) a thread
// stores one float4 per channel plane, and one per plane of the mirror.
__global__ void __launch_bounds__(WARP_THREADS) warp_affine_u8_f32_kernel(const __grid_constant__ WarpF32Params p) {
  __shared__ float s_tab[3 * 256];
  const WarpDesc& q = p.d[blockIdx.y];
  const float* tab = p.tables + (size_t)p.table[blockIdx.y] * (3 * 256);
  for (int i = threadIdx.x; i < 3 * 256; i += WARP_THREADS) s_tab[i] = __ldg(tab + i);
  __syncthreads();
  const int t = blockIdx.x * WARP_THREADS + threadIdx.x;
  const int y = t / p.groups, x0 = (t - y * p.groups) * WARP_PX;
  if (y >= p.dh) return;
  const int n = min(WARP_PX, p.dw - x0);
  uint8_t v[WARP_PX * 3];
  warp_pixels(q, PoolBgr{p.pool + q.off, q}, y, x0, v);
  const size_t plane = (size_t)p.dh * p.dw, row = (size_t)y * p.dw;
  float* d = p.dst + (size_t)q.dst * 3 * plane + row + x0;
  float* m = q.mirror >= 0 ? p.dst + (size_t)q.mirror * 3 * plane + row + (p.dw - x0 - n) : nullptr;   // ends at dw - 1 - x0
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float f[WARP_PX];
#pragma unroll
    for (int i = 0; i < WARP_PX; ++i) f[i] = s_tab[c * 256 + v[i * 3 + c]];
    if (p.vec) {
      *reinterpret_cast<float4*>(d + c * plane) = make_float4(f[0], f[1], f[2], f[3]);
      if (m) *reinterpret_cast<float4*>(m + c * plane) = make_float4(f[3], f[2], f[1], f[0]);
    } else {
#pragma unroll
      for (int i = 0; i < WARP_PX; ++i)
        if (i < n) {
          d[c * plane + i] = f[i];
          if (m) m[c * plane + n - 1 - i] = f[i];
        }
    }
  }
}

// The general-source kernels: the kernels above with each descriptor's frame read through its own tap, BGR at any row pitch or
// YUV 4:2:0 (the source kind is uniform per CTA: blockIdx.y selects the descriptor).  The stores are those of the kernels above,
// which keep their own code so that their SASS stays as it is.
__device__ __forceinline__ void warp_src_pixels(const WarpSrcDesc& q, int y, int x0, uint8_t (&v)[WARP_PX * 3]) {
  if (q.kind == CDN_WARP_SRC_YUV420)
    warp_pixels(q, Yuv420{q.p[0], q.p[1], q.p[2], q.pitch[0], q.pitch[1], q.step}, y, x0, v);
  else
    warp_pixels(q, PitchedBgr{q.p[0], q.pitch[0]}, y, x0, v);
}

__global__ void __launch_bounds__(WARP_THREADS) warp_affine_src_u8_kernel(const __grid_constant__ WarpSrcParams p) {
  const WarpSrcDesc& q = p.d[blockIdx.y];
  const int t = blockIdx.x * WARP_THREADS + threadIdx.x;
  const int y = t / p.groups, x0 = (t - y * p.groups) * WARP_PX;
  if (y >= p.dh) return;
  const int n = min(WARP_PX, p.dw - x0);
  uint8_t v[WARP_PX * 3];
  warp_src_pixels(q, y, x0, v);
  const size_t plane = (size_t)p.dh * p.dw * 3, row = (size_t)y * p.dw * 3;
  warp_store(p.dst + (size_t)q.dst * plane + row + (size_t)x0 * 3, v, n);
  if (q.mirror >= 0) {
    uint8_t f[WARP_PX * 3];
#pragma unroll
    for (int i = 0; i < WARP_PX; ++i)
#pragma unroll
      for (int c = 0; c < 3; ++c) f[i * 3 + c] = v[(WARP_PX - 1 - i) * 3 + c];
    uint8_t* m = p.dst + (size_t)q.mirror * plane + row + (size_t)(p.dw - x0 - n) * 3;
    if (n == WARP_PX) {
      warp_store(m, f, n);
    } else {
      const int skip = (WARP_PX - n) * 3;
#pragma unroll
      for (int i = 0; i < WARP_PX * 3; ++i)
        if (i >= skip) m[i - skip] = f[i];
    }
  }
}

__global__ void __launch_bounds__(WARP_THREADS) warp_affine_src_u8_f32_kernel(const __grid_constant__ WarpSrcF32Params p) {
  __shared__ float s_tab[3 * 256];
  const WarpSrcDesc& q = p.d[blockIdx.y];
  const float* tab = p.tables + (size_t)p.table[blockIdx.y] * (3 * 256);
  for (int i = threadIdx.x; i < 3 * 256; i += WARP_THREADS) s_tab[i] = __ldg(tab + i);
  __syncthreads();
  const int t = blockIdx.x * WARP_THREADS + threadIdx.x;
  const int y = t / p.groups, x0 = (t - y * p.groups) * WARP_PX;
  if (y >= p.dh) return;
  const int n = min(WARP_PX, p.dw - x0);
  uint8_t v[WARP_PX * 3];
  warp_src_pixels(q, y, x0, v);
  const size_t plane = (size_t)p.dh * p.dw, row = (size_t)y * p.dw;
  float* d = p.dst + (size_t)q.dst * 3 * plane + row + x0;
  float* m = q.mirror >= 0 ? p.dst + (size_t)q.mirror * 3 * plane + row + (p.dw - x0 - n) : nullptr;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float f[WARP_PX];
#pragma unroll
    for (int i = 0; i < WARP_PX; ++i) f[i] = s_tab[c * 256 + v[i * 3 + c]];
    if (p.vec) {
      *reinterpret_cast<float4*>(d + c * plane) = make_float4(f[0], f[1], f[2], f[3]);
      if (m) *reinterpret_cast<float4*>(m + c * plane) = make_float4(f[3], f[2], f[1], f[0]);
    } else {
#pragma unroll
      for (int i = 0; i < WARP_PX; ++i)
        if (i < n) {
          d[c * plane + i] = f[i];
          if (m) m[c * plane + n - 1 - i] = f[i];
        }
    }
  }
}

// The resize-and-warp kernels: the general-source kernels with every tap of the warp a pixel of the resized frame (Resized), or
// of the frame itself where the descriptor's resized size is the frame's (the branch is uniform per CTA).
template <class Src>
__device__ __forceinline__ void warp_rs_pixels_of(const WarpRsDesc& q, const Src& src, int y, int x0, uint8_t (&v)[WARP_PX * 3]) {
  if (q.FH == q.H && q.FW == q.W)
    warp_pixels(q, src, y, x0, v);
  else
    warp_pixels(q, Resized<Src>{src, q.FH, q.FW, q.scale[0], q.scale[1]}, y, x0, v);
}

__device__ __forceinline__ void warp_rs_pixels(const WarpRsDesc& q, int y, int x0, uint8_t (&v)[WARP_PX * 3]) {
  if (q.kind == CDN_WARP_SRC_YUV420)
    warp_rs_pixels_of(q, Yuv420{q.p[0], q.p[1], q.p[2], q.pitch[0], q.pitch[1], q.step}, y, x0, v);
  else
    warp_rs_pixels_of(q, PitchedBgr{q.p[0], q.pitch[0]}, y, x0, v);
}

__global__ void __launch_bounds__(WARP_THREADS) warp_affine_resize_u8_kernel(const __grid_constant__ WarpRsParams p) {
  const WarpRsDesc& q = p.d[blockIdx.y];
  const int t = blockIdx.x * WARP_THREADS + threadIdx.x;
  const int y = t / p.groups, x0 = (t - y * p.groups) * WARP_PX;
  if (y >= p.dh) return;
  const int n = min(WARP_PX, p.dw - x0);
  uint8_t v[WARP_PX * 3];
  warp_rs_pixels(q, y, x0, v);
  const size_t plane = (size_t)p.dh * p.dw * 3, row = (size_t)y * p.dw * 3;
  warp_store(p.dst + (size_t)q.dst * plane + row + (size_t)x0 * 3, v, n);
  if (q.mirror >= 0) {
    uint8_t f[WARP_PX * 3];
#pragma unroll
    for (int i = 0; i < WARP_PX; ++i)
#pragma unroll
      for (int c = 0; c < 3; ++c) f[i * 3 + c] = v[(WARP_PX - 1 - i) * 3 + c];
    uint8_t* m = p.dst + (size_t)q.mirror * plane + row + (size_t)(p.dw - x0 - n) * 3;
    if (n == WARP_PX) {
      warp_store(m, f, n);
    } else {
      const int skip = (WARP_PX - n) * 3;
#pragma unroll
      for (int i = 0; i < WARP_PX * 3; ++i)
        if (i >= skip) m[i - skip] = f[i];
    }
  }
}

__global__ void __launch_bounds__(WARP_THREADS) warp_affine_resize_u8_f32_kernel(const __grid_constant__ WarpRsF32Params p) {
  __shared__ float s_tab[3 * 256];
  const WarpRsDesc& q = p.d[blockIdx.y];
  const float* tab = p.tables + (size_t)p.table[blockIdx.y] * (3 * 256);
  for (int i = threadIdx.x; i < 3 * 256; i += WARP_THREADS) s_tab[i] = __ldg(tab + i);
  __syncthreads();
  const int t = blockIdx.x * WARP_THREADS + threadIdx.x;
  const int y = t / p.groups, x0 = (t - y * p.groups) * WARP_PX;
  if (y >= p.dh) return;
  const int n = min(WARP_PX, p.dw - x0);
  uint8_t v[WARP_PX * 3];
  warp_rs_pixels(q, y, x0, v);
  const size_t plane = (size_t)p.dh * p.dw, row = (size_t)y * p.dw;
  float* d = p.dst + (size_t)q.dst * 3 * plane + row + x0;
  float* m = q.mirror >= 0 ? p.dst + (size_t)q.mirror * 3 * plane + row + (p.dw - x0 - n) : nullptr;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float f[WARP_PX];
#pragma unroll
    for (int i = 0; i < WARP_PX; ++i) f[i] = s_tab[c * 256 + v[i * 3 + c]];
    if (p.vec) {
      *reinterpret_cast<float4*>(d + c * plane) = make_float4(f[0], f[1], f[2], f[3]);
      if (m) *reinterpret_cast<float4*>(m + c * plane) = make_float4(f[3], f[2], f[1], f[0]);
    } else {
#pragma unroll
      for (int i = 0; i < WARP_PX; ++i)
        if (i < n) {
          d[c * plane + i] = f[i];
          if (m) m[c * plane + n - 1 - i] = f[i];
        }
    }
  }
}

// the destination checks of every batch entry point
static int warp_dst_check(const char* who, int n, int dst_slots, int dst_h, int dst_w) {
  CDN_CHECK(n >= 0, CDN_ERR_INVALID, "%s: n = %d", who, n);
  CDN_CHECK(dst_slots > 0 && dst_h > 0 && dst_w > 0, CDN_ERR_INVALID, "%s: bad destination %d x %d x %d", who, dst_slots, dst_h,
            dst_w);
  const long long groups = ((long long)dst_w + WARP_PX - 1) / WARP_PX;
  const long long tiles = ((long long)dst_h * groups + WARP_THREADS - 1) / WARP_THREADS;
  CDN_CHECK(tiles <= 0x7fffffffLL && (long long)dst_h * groups <= 0x7fffffffLL, CDN_ERR_INVALID,
            "%s: destination %d x %d too large", who, dst_h, dst_w);
  return 0;
}

// the checks both pool batch entry points make before anything is launched
static int warp_batch_check(const char* who, const cdn_warp_desc* h_desc, int n, int dst_slots, int dst_h, int dst_w) {
  if (int rc = warp_dst_check(who, n, dst_slots, dst_h, dst_w)) return rc;
  for (int i = 0; i < n; ++i) {
    const cdn_warp_desc& d = h_desc[i];
    CDN_CHECK(d.src_offset >= 0 && d.src_h > 0 && d.src_w > 0, CDN_ERR_INVALID,
              "%s: descriptor %d: bad source (offset %lld, %d x %d)", who, i, d.src_offset, d.src_h, d.src_w);
    CDN_CHECK(d.dst_slot >= 0 && d.dst_slot < dst_slots && d.mirror_slot >= -1 && d.mirror_slot < dst_slots, CDN_ERR_INVALID,
              "%s: descriptor %d: slot %d / mirror %d outside [0, %d)", who, i, d.dst_slot, d.mirror_slot, dst_slots);
  }
  return 0;
}

// the checks the general-source and the resize entry points make on a descriptor before anything is launched: what every plane
// must hold, per source kind
template <class Desc>
static int warp_frame_check(const char* who, const Desc& d, int i, int dst_slots) {
  CDN_CHECK(d.kind == CDN_WARP_SRC_BGR || d.kind == CDN_WARP_SRC_YUV420, CDN_ERR_INVALID, "%s: descriptor %d: unknown source kind %d",
          who, i, d.kind);
  CDN_CHECK(d.src_h > 0 && d.src_w > 0, CDN_ERR_INVALID, "%s: descriptor %d: bad source size %d x %d", who, i, d.src_h, d.src_w);
  if (d.kind == CDN_WARP_SRC_BGR) {
    CDN_CHECK(d.plane[0], CDN_ERR_INVALID, "%s: descriptor %d: null plane", who, i);
    CDN_CHECK(d.pitch[0] >= 3LL * d.src_w, CDN_ERR_INVALID, "%s: descriptor %d: pitch %lld below the row's %lld bytes", who, i,
              d.pitch[0], 3LL * d.src_w);
  } else {
    CDN_CHECK(d.plane[0] && d.plane[1] && d.plane[2], CDN_ERR_INVALID, "%s: descriptor %d: null plane", who, i);
    CDN_CHECK(d.src_h % 2 == 0 && d.src_w % 2 == 0, CDN_ERR_INVALID, "%s: descriptor %d: odd YUV 4:2:0 size %d x %d", who, i,
              d.src_h, d.src_w);
    CDN_CHECK(d.chroma_step == 1 || d.chroma_step == 2, CDN_ERR_INVALID, "%s: descriptor %d: chroma step %d not 1 or 2", who, i,
              d.chroma_step);
    const long long chroma_row = (long long)(d.src_w / 2 - 1) * d.chroma_step + 1;
    CDN_CHECK(d.pitch[0] >= d.src_w && d.pitch[1] >= chroma_row, CDN_ERR_INVALID,
              "%s: descriptor %d: pitch %lld / %lld below the rows' %d / %lld bytes", who, i, d.pitch[0], d.pitch[1], d.src_w,
              chroma_row);
  }
  CDN_CHECK(d.dst_slot >= 0 && d.dst_slot < dst_slots && d.mirror_slot >= -1 && d.mirror_slot < dst_slots, CDN_ERR_INVALID,
            "%s: descriptor %d: slot %d / mirror %d outside [0, %d)", who, i, d.dst_slot, d.mirror_slot, dst_slots);
  return 0;
}

static int warp_src_check(const char* who, const cdn_warp_src_desc* h_desc, int n, int dst_slots, int dst_h, int dst_w) {
  if (int rc = warp_dst_check(who, n, dst_slots, dst_h, dst_w)) return rc;
  for (int i = 0; i < n; ++i)
    if (int rc = warp_frame_check(who, h_desc[i], i, dst_slots)) return rc;
  return 0;
}

// the resize entry points: the frame checks plus a resized size of at least 1 x 1 whose scales are the descriptor's, bit for bit
static int warp_rs_check(const char* who, const cdn_warp_rs_desc* h_desc, int n, int dst_slots, int dst_h, int dst_w) {
  if (int rc = warp_dst_check(who, n, dst_slots, dst_h, dst_w)) return rc;
  for (int i = 0; i < n; ++i) {
    const cdn_warp_rs_desc& d = h_desc[i];
    if (int rc = warp_frame_check(who, d, i, dst_slots)) return rc;
    CDN_CHECK(d.rs_h > 0 && d.rs_w > 0, CDN_ERR_INVALID, "%s: descriptor %d: bad resized size %d x %d", who, i, d.rs_h, d.rs_w);
    CDN_CHECK(d.inv_scale[0] == 1. / ((double)d.rs_w / d.src_w) && d.inv_scale[1] == 1. / ((double)d.rs_h / d.src_h), CDN_ERR_INVALID,
              "%s: descriptor %d: scales %.17g, %.17g are not those of %d x %d -> %d x %d", who, i, d.inv_scale[0], d.inv_scale[1],
              d.src_h, d.src_w, d.rs_h, d.rs_w);
  }
  return 0;
}

static void warp_fill(const cdn_warp_desc& d, WarpDesc& q) {
  q.off = d.src_offset; q.H = d.src_h; q.W = d.src_w; q.dst = d.dst_slot; q.mirror = d.mirror_slot;
  warp_invert(d.M, q.m);
}

static void warp_src_fill(const cdn_warp_src_desc& d, WarpSrcDesc& q) {
  for (int k = 0; k < 3; ++k) q.p[k] = d.plane[k];
  q.pitch[0] = d.pitch[0]; q.pitch[1] = d.pitch[1];
  q.H = d.src_h; q.W = d.src_w; q.kind = d.kind; q.step = d.chroma_step; q.dst = d.dst_slot; q.mirror = d.mirror_slot;
  warp_invert(d.M, q.m);
}

extern "C" int cdn_warp_affine_u8_batch(const uint8_t* d_pool, const cdn_warp_desc* h_desc, int n, uint8_t* d_dst, int dst_slots,
                                        int dst_h, int dst_w, cdn_stream_t stream) {
  CDN_CHECK(d_pool && h_desc && d_dst, CDN_ERR_INVALID, "warp_affine_batch: null pointer");
  if (int rc = warp_batch_check("warp_affine_batch", h_desc, n, dst_slots, dst_h, dst_w)) return rc;
  const int groups = (dst_w + WARP_PX - 1) / WARP_PX;
  const long long tiles = ((long long)dst_h * groups + WARP_THREADS - 1) / WARP_THREADS;
  WarpBatchParams p;
  p.pool = d_pool; p.dst = d_dst; p.dh = dst_h; p.dw = dst_w; p.groups = groups; p.pad = 0;
  for (int base = 0; base < n; base += WARP_MAX_DESC) {
    const int m = std::min(WARP_MAX_DESC, n - base);
    for (int i = 0; i < m; ++i) warp_fill(h_desc[base + i], p.d[i]);
    warp_affine_u8_kernel<<<dim3((unsigned)tiles, (unsigned)m), WARP_THREADS, 0, (cudaStream_t)stream>>>(p);
    CDN_LAUNCH_CHECK("warp_affine_u8_kernel");
  }
  return 0;
}

extern "C" int cdn_warp_affine_u8_f32_batch(const uint8_t* d_pool, const cdn_warp_desc* h_desc, const int32_t* h_table, int n,
                                            const float* d_tables, int n_tables, float* d_dst, int dst_slots, int dst_h, int dst_w,
                                            cdn_stream_t stream) {
  CDN_CHECK(d_pool && h_desc && h_table && d_tables && d_dst, CDN_ERR_INVALID, "warp_affine_f32_batch: null pointer");
  CDN_CHECK(((uintptr_t)d_tables & 3) == 0 && ((uintptr_t)d_dst & 3) == 0, CDN_ERR_INVALID,
            "warp_affine_f32_batch: tables and destination must be 4-byte aligned");
  CDN_CHECK(n_tables >= 1 && n_tables <= 2, CDN_ERR_INVALID, "warp_affine_f32_batch: n_tables = %d outside [1, 2]", n_tables);
  if (int rc = warp_batch_check("warp_affine_f32_batch", h_desc, n, dst_slots, dst_h, dst_w)) return rc;
  for (int i = 0; i < n; ++i)
    CDN_CHECK(h_table[i] >= 0 && h_table[i] < n_tables, CDN_ERR_INVALID, "warp_affine_f32_batch: descriptor %d: table %d outside [0, %d)",
              i, h_table[i], n_tables);
  const int groups = (dst_w + WARP_PX - 1) / WARP_PX;
  const long long tiles = ((long long)dst_h * groups + WARP_THREADS - 1) / WARP_THREADS;
  WarpF32Params p;
  p.pool = d_pool; p.dst = d_dst; p.tables = d_tables; p.dh = dst_h; p.dw = dst_w; p.groups = groups;
  p.vec = dst_w % WARP_PX == 0 && ((uintptr_t)d_dst & 15) == 0;
  for (int base = 0; base < n; base += WARP_F32_MAX_DESC) {
    const int m = std::min(WARP_F32_MAX_DESC, n - base);
    for (int i = 0; i < m; ++i) {
      warp_fill(h_desc[base + i], p.d[i]);
      p.table[i] = (uint8_t)h_table[base + i];
    }
    warp_affine_u8_f32_kernel<<<dim3((unsigned)tiles, (unsigned)m), WARP_THREADS, 0, (cudaStream_t)stream>>>(p);
    CDN_LAUNCH_CHECK("warp_affine_u8_f32_kernel");
  }
  return 0;
}

extern "C" int cdn_warp_affine_src_u8_batch(const cdn_warp_src_desc* h_desc, int n, uint8_t* d_dst, int dst_slots, int dst_h,
                                            int dst_w, cdn_stream_t stream) {
  CDN_CHECK(h_desc && d_dst, CDN_ERR_INVALID, "warp_affine_src_batch: null pointer");
  if (int rc = warp_src_check("warp_affine_src_batch", h_desc, n, dst_slots, dst_h, dst_w)) return rc;
  const int groups = (dst_w + WARP_PX - 1) / WARP_PX;
  const long long tiles = ((long long)dst_h * groups + WARP_THREADS - 1) / WARP_THREADS;
  WarpSrcParams p;
  p.dst = d_dst; p.dh = dst_h; p.dw = dst_w; p.groups = groups; p.pad = 0;
  for (int base = 0; base < n; base += WARP_SRC_MAX_DESC) {
    const int m = std::min(WARP_SRC_MAX_DESC, n - base);
    for (int i = 0; i < m; ++i) warp_src_fill(h_desc[base + i], p.d[i]);
    warp_affine_src_u8_kernel<<<dim3((unsigned)tiles, (unsigned)m), WARP_THREADS, 0, (cudaStream_t)stream>>>(p);
    CDN_LAUNCH_CHECK("warp_affine_src_u8_kernel");
  }
  return 0;
}

extern "C" int cdn_warp_affine_src_u8_f32_batch(const cdn_warp_src_desc* h_desc, const int32_t* h_table, int n, const float* d_tables,
                                                int n_tables, float* d_dst, int dst_slots, int dst_h, int dst_w, cdn_stream_t stream) {
  CDN_CHECK(h_desc && h_table && d_tables && d_dst, CDN_ERR_INVALID, "warp_affine_src_f32_batch: null pointer");
  CDN_CHECK(((uintptr_t)d_tables & 3) == 0 && ((uintptr_t)d_dst & 3) == 0, CDN_ERR_INVALID,
            "warp_affine_src_f32_batch: tables and destination must be 4-byte aligned");
  CDN_CHECK(n_tables >= 1 && n_tables <= 2, CDN_ERR_INVALID, "warp_affine_src_f32_batch: n_tables = %d outside [1, 2]", n_tables);
  if (int rc = warp_src_check("warp_affine_src_f32_batch", h_desc, n, dst_slots, dst_h, dst_w)) return rc;
  for (int i = 0; i < n; ++i)
    CDN_CHECK(h_table[i] >= 0 && h_table[i] < n_tables, CDN_ERR_INVALID,
              "warp_affine_src_f32_batch: descriptor %d: table %d outside [0, %d)", i, h_table[i], n_tables);
  const int groups = (dst_w + WARP_PX - 1) / WARP_PX;
  const long long tiles = ((long long)dst_h * groups + WARP_THREADS - 1) / WARP_THREADS;
  WarpSrcF32Params p;
  p.dst = d_dst; p.tables = d_tables; p.dh = dst_h; p.dw = dst_w; p.groups = groups;
  p.vec = dst_w % WARP_PX == 0 && ((uintptr_t)d_dst & 15) == 0;
  for (int base = 0; base < n; base += WARP_SRC_F32_MAX_DESC) {
    const int m = std::min(WARP_SRC_F32_MAX_DESC, n - base);
    for (int i = 0; i < m; ++i) {
      warp_src_fill(h_desc[base + i], p.d[i]);
      p.table[i] = (uint8_t)h_table[base + i];
    }
    warp_affine_src_u8_f32_kernel<<<dim3((unsigned)tiles, (unsigned)m), WARP_THREADS, 0, (cudaStream_t)stream>>>(p);
    CDN_LAUNCH_CHECK("warp_affine_src_u8_f32_kernel");
  }
  return 0;
}

static void warp_rs_fill(const cdn_warp_rs_desc& d, WarpRsDesc& q) {
  for (int k = 0; k < 3; ++k) q.p[k] = d.plane[k];
  q.pitch[0] = d.pitch[0]; q.pitch[1] = d.pitch[1];
  q.scale[0] = d.inv_scale[0]; q.scale[1] = d.inv_scale[1];
  q.H = d.rs_h; q.W = d.rs_w; q.FH = d.src_h; q.FW = d.src_w;
  q.kind = d.kind; q.step = d.chroma_step; q.dst = d.dst_slot; q.mirror = d.mirror_slot;
  warp_invert(d.M, q.m);
}

extern "C" int cdn_warp_affine_resize_u8_batch(const cdn_warp_rs_desc* h_desc, int n, uint8_t* d_dst, int dst_slots, int dst_h,
                                               int dst_w, cdn_stream_t stream) {
  CDN_CHECK(h_desc && d_dst, CDN_ERR_INVALID, "warp_affine_resize_batch: null pointer");
  if (int rc = warp_rs_check("warp_affine_resize_batch", h_desc, n, dst_slots, dst_h, dst_w)) return rc;
  const int groups = (dst_w + WARP_PX - 1) / WARP_PX;
  const long long tiles = ((long long)dst_h * groups + WARP_THREADS - 1) / WARP_THREADS;
  WarpRsParams p;
  p.dst = d_dst; p.dh = dst_h; p.dw = dst_w; p.groups = groups; p.pad = 0;
  for (int base = 0; base < n; base += WARP_RS_MAX_DESC) {
    const int m = std::min(WARP_RS_MAX_DESC, n - base);
    for (int i = 0; i < m; ++i) warp_rs_fill(h_desc[base + i], p.d[i]);
    warp_affine_resize_u8_kernel<<<dim3((unsigned)tiles, (unsigned)m), WARP_THREADS, 0, (cudaStream_t)stream>>>(p);
    CDN_LAUNCH_CHECK("warp_affine_resize_u8_kernel");
  }
  return 0;
}

extern "C" int cdn_warp_affine_resize_u8_f32_batch(const cdn_warp_rs_desc* h_desc, const int32_t* h_table, int n,
                                                   const float* d_tables, int n_tables, float* d_dst, int dst_slots, int dst_h,
                                                   int dst_w, cdn_stream_t stream) {
  CDN_CHECK(h_desc && h_table && d_tables && d_dst, CDN_ERR_INVALID, "warp_affine_resize_f32_batch: null pointer");
  CDN_CHECK(((uintptr_t)d_tables & 3) == 0 && ((uintptr_t)d_dst & 3) == 0, CDN_ERR_INVALID,
            "warp_affine_resize_f32_batch: tables and destination must be 4-byte aligned");
  CDN_CHECK(n_tables >= 1 && n_tables <= 2, CDN_ERR_INVALID, "warp_affine_resize_f32_batch: n_tables = %d outside [1, 2]", n_tables);
  if (int rc = warp_rs_check("warp_affine_resize_f32_batch", h_desc, n, dst_slots, dst_h, dst_w)) return rc;
  for (int i = 0; i < n; ++i)
    CDN_CHECK(h_table[i] >= 0 && h_table[i] < n_tables, CDN_ERR_INVALID,
              "warp_affine_resize_f32_batch: descriptor %d: table %d outside [0, %d)", i, h_table[i], n_tables);
  const int groups = (dst_w + WARP_PX - 1) / WARP_PX;
  const long long tiles = ((long long)dst_h * groups + WARP_THREADS - 1) / WARP_THREADS;
  WarpRsF32Params p;
  p.dst = d_dst; p.tables = d_tables; p.dh = dst_h; p.dw = dst_w; p.groups = groups;
  p.vec = dst_w % WARP_PX == 0 && ((uintptr_t)d_dst & 15) == 0;
  for (int base = 0; base < n; base += WARP_RS_F32_MAX_DESC) {
    const int m = std::min(WARP_RS_F32_MAX_DESC, n - base);
    for (int i = 0; i < m; ++i) {
      warp_rs_fill(h_desc[base + i], p.d[i]);
      p.table[i] = (uint8_t)h_table[base + i];
    }
    warp_affine_resize_u8_f32_kernel<<<dim3((unsigned)tiles, (unsigned)m), WARP_THREADS, 0, (cudaStream_t)stream>>>(p);
    CDN_LAUNCH_CHECK("warp_affine_resize_u8_f32_kernel");
  }
  return 0;
}

extern "C" int cdn_warp_affine_u8(const uint8_t* d_src, int H, int W, const double* M6, uint8_t* d_dst, int dst_h, int dst_w,
                                  int flip_copy, cdn_stream_t stream) {
  CDN_CHECK(d_src && d_dst && M6 && H > 0 && W > 0 && dst_h > 0 && dst_w > 0, CDN_ERR_INVALID, "warp_affine: bad arguments");
  cdn_warp_desc d;
  d.src_offset = 0; d.src_h = H; d.src_w = W; d.dst_slot = 0; d.mirror_slot = flip_copy ? 1 : -1;
  for (int i = 0; i < 6; ++i) d.M[i] = M6[i];
  return cdn_warp_affine_u8_batch(d_src, &d, 1, d_dst, flip_copy ? 2 : 1, dst_h, dst_w, stream);
}

// one CTA per image; K <= 1024.  out[b][rank] = dets[b][t] with rank = (detections of smaller classes) + (earlier ones of
// the same class); counts[b][c] = detections of class c.  Classes outside [0, num_classes) go last and are not counted.
__global__ void ctdet_group_by_class_kernel(const float* __restrict__ dets, int K, int num_classes, float* __restrict__ out,
                                            int* __restrict__ counts) {
  extern __shared__ int s_cls[];                 // [K] classes, then [num_classes + 1] histogram / offsets
  int* s_hist = s_cls + K;
  const int b = blockIdx.x, t = threadIdx.x;
  const float* d = dets + (size_t)b * K * 6;
  for (int c = t; c <= num_classes; c += blockDim.x) s_hist[c] = 0;
  __syncthreads();
  int cls = num_classes;
  if (t < K) {
    const float cf = d[t * 6 + 5];
    const int ci = (int)cf;
    if (cf >= 0.f && ci < num_classes) cls = ci;
    s_cls[t] = cls;
    atomicAdd(&s_hist[cls], 1);
  }
  __syncthreads();
  if (t < K) {
    int rank = 0;
    for (int c = 0; c < cls; ++c) rank += s_hist[c];
    for (int j = 0; j < t; ++j) rank += s_cls[j] == cls;
    float* o = out + ((size_t)b * K + rank) * 6;
#pragma unroll
    for (int i = 0; i < 6; ++i) o[i] = d[t * 6 + i];
  }
  for (int c = t; c < num_classes; c += blockDim.x) counts[(size_t)b * num_classes + c] = s_hist[c];
}

extern "C" int cdn_ctdet_group_by_class(const float* d_dets, int batch, int K, int num_classes, float* d_out, int32_t* d_counts,
                                        cdn_stream_t stream) {
  CDN_CHECK(d_dets && d_out && d_counts && batch >= 0 && K >= 1 && K <= 1024 && num_classes >= 1 && num_classes <= 4096, CDN_ERR_INVALID,
            "group_by_class: bad arguments (K <= 1024)");
  CDN_CHECK(d_dets != d_out, CDN_ERR_INVALID, "group_by_class: in-place operation is not supported");
  if (batch == 0) return 0;
  const int threads = (std::max(K, 32) + 31) / 32 * 32;
  ctdet_group_by_class_kernel<<<batch, threads, (size_t)(K + num_classes + 1) * sizeof(int), (cudaStream_t)stream>>>(
      d_dets, K, num_classes, d_out, d_counts);
  CDN_LAUNCH_CHECK("ctdet_group_by_class_kernel");
  return 0;
}
