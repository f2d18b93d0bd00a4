// ingest.cuh -- device-side image ingest: cv2.resize(orig_img, (input_w, input_h)) of
// pose_detector.py:493 (default INTER_LINEAR on uint8 BGR), bit-exact.
//
// OpenCV's 8-bit path (imgproc/resize.cpp) is fixed point: per axis
//   f = float((d + 0.5) * scale - 0.5), s = floor(f), f -= s        (scale = 1 / (dst/src) in double)
//   columns clamp (s < 0 -> s = 0, f = 0;  s >= w-1 -> s = w-1, f = 0); rows keep f and clip the two
//   source rows separately;  coefficients = rint((1-f)*2048), rint(f*2048)  (int16)
//   horizontal   D = S[s]*a0 + S[s+1]*a1                                   (int32)
//   vertical     dst = (((b0*(D0>>4))>>16) + ((b1*(D1>>4))>>16) + 2) >> 2
// Every float/double step below is a single IEEE operation, so the device reproduces the host bits.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace opb {

__device__ __forceinline__ void cv_linear_axis(int d, double scale, int src_n, bool clamp, int& s0, int& s1, int& c0,
                                               int& c1) {
  float f = __double2float_rn(__dsub_rn(__dmul_rn(__dadd_rn(static_cast<double>(d), 0.5), scale), 0.5));
  int s = static_cast<int>(floorf(f));
  f = __fsub_rn(f, static_cast<float>(s));
  if (clamp) {
    if (s < 0) { s = 0; f = 0.f; }
    if (s >= src_n - 1) { s = src_n - 1; f = 0.f; }
  }
  c0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
  c1 = __float2int_rn(__fmul_rn(f, 2048.f));
  s0 = min(max(s, 0), src_n - 1);
  s1 = min(max(s + 1, 0), src_n - 1);
}

// One output pixel (x, y) of the INTER_LINEAR resize of the image img [h0][w0][3] into o[0..2].  With h0 == h and
// w0 == w the arithmetic is the identity (f = 0: coefficients 2048 / 0), so no size needs a separate copy path.
__device__ __forceinline__ void resize_linear_u8_pixel(const uint8_t* __restrict__ img, int h0, int w0, int x, int y,
                                                       double scale_x, double scale_y, uint8_t* __restrict__ o) {
  int sx0, sx1, a0, a1, sy0, sy1, b0, b1;
  cv_linear_axis(x, scale_x, w0, true, sx0, sx1, a0, a1);
  cv_linear_axis(y, scale_y, h0, false, sy0, sy1, b0, b1);
  const uint8_t* r0 = img + static_cast<size_t>(sy0) * w0 * 3;
  const uint8_t* r1 = img + static_cast<size_t>(sy1) * w0 * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int d0 = r0[sx0 * 3 + c] * a0 + r0[sx1 * 3 + c] * a1;
    const int d1 = r1[sx0 * 3 + c] * a0 + r1[sx1 * 3 + c] * a1;
    o[c] = static_cast<uint8_t>((((b0 * (d0 >> 4)) >> 16) + ((b1 * (d1 >> 4)) >> 16) + 2) >> 2);
  }
}

// src [n][h0][w0][3] uint8 -> dst [n][h][w][3] uint8; grid (ceil(w/32), ceil(h/8), n), block (32, 8)
__global__ void __launch_bounds__(256)
resize_linear_u8_kernel(const uint8_t* __restrict__ src, int h0, int w0, uint8_t* __restrict__ dst, int h, int w,
                        double scale_x, double scale_y) {
  const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y, n = blockIdx.z;
  if (x >= w || y >= h) return;
  resize_linear_u8_pixel(src + static_cast<size_t>(n) * h0 * w0 * 3, h0, w0, x, y, scale_x, scale_y,
                         dst + ((static_cast<size_t>(n) * h + y) * w + x) * 3);
}

// One crop of a ragged batch: crop i = h0 x w0 x 3 uint8 at byte offset `src_off` of the packed source.
struct RaggedCrop {
  long long src_off;
  int h0, w0;
  double scale_x, scale_y;   // 1 / (dst / src) in double, as cv2::resize forms them
};

// Crops of different sizes packed back to back -> dst [n][h][w][3] (one network-input slot per crop);
// grid (ceil(w/32), ceil(h/8), n), block (32, 8).
__global__ void __launch_bounds__(256)
resize_linear_u8_ragged_kernel(const uint8_t* __restrict__ src, const RaggedCrop* __restrict__ crops,
                               uint8_t* __restrict__ dst, int h, int w) {
  const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y, n = blockIdx.z;
  if (x >= w || y >= h) return;
  const RaggedCrop c = crops[n];
  resize_linear_u8_pixel(src + c.src_off, c.h0, c.w0, x, y, c.scale_x, c.scale_y,
                         dst + ((static_cast<size_t>(n) * h + y) * w + x) * 3);
}

// ---- cv2.resize(orig_img, ..., interpolation=cv2.INTER_CUBIC) on uint8 BGR (detect_precise, pose_detector.py:443) ----
// OpenCV's own 8-bit cubic path (imgproc/resize.cpp, the code that runs when the build has no IPP or cv2.ipp.setUseIPP(False)):
//   per axis   f = float((d + 0.5) * scale - 0.5), s = floor(f), f -= s;   Keys taps (A = -0.75) in float32,
//              coefficients = rint(tap * 2048) (int16, no renormalisation); source index s-1+k clamped (replicate)
//   horizontal D = sum_k S[s-1+k] * a[k]                                   (int32, exact)
//   vertical   elements e = x*3 + c < (3*w & ~7)  (the 8-lane SIMD body of VResizeCubicVec_32s8u):
//                  float32, b[k] = beta[k] / 2^22:  ((D3*b3 + D2*b2) + D1*b1) + D0*b0, each product and sum rounded
//                  (SSE baseline: no FMA), rint (half-even), saturate to [0, 255]
//              the last (3*w) % 8 elements of a row (scalar tail, FixedPtCast<int, uchar, 22>):
//                  (D0*beta0 + D1*beta1 + D2*beta2 + D3*beta3 + 2^21) >> 22, saturated
// Pinned by tests against cv2 4.13 with IPP disabled; IPP builds (ippiResizeCubic, arithmetic unpublished) differ
// from this path by 1 LSB in 4-8 % of the pixels (DESIGN.md 4.3), which is why the host cv2 call stays the default.
__device__ __forceinline__ void cv_cubic_axis(int d, double scale, int& s, int (&c)[4]) {
  float f = __double2float_rn(__dsub_rn(__dmul_rn(__dadd_rn(static_cast<double>(d), 0.5), scale), 0.5));
  s = static_cast<int>(floorf(f));
  f = __fsub_rn(f, static_cast<float>(s));
  const float A = -0.75f;
  const float t = __fadd_rn(f, 1.f), u = __fsub_rn(1.f, f);
  // ((A*(x+1) - 5A)*(x+1) + 8A)*(x+1) - 4A
  const float k0 = __fsub_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(A, t), 5.f * A), t), 8.f * A), t), 4.f * A);
  // ((A+2)*x - (A+3))*x*x + 1
  const float k1 = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(A + 2.f, f), A + 3.f), f), f), 1.f);
  const float k2 = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(A + 2.f, u), A + 3.f), u), u), 1.f);
  const float k3 = __fsub_rn(__fsub_rn(__fsub_rn(1.f, k0), k1), k2);
  c[0] = __float2int_rn(__fmul_rn(k0, 2048.f));
  c[1] = __float2int_rn(__fmul_rn(k1, 2048.f));
  c[2] = __float2int_rn(__fmul_rn(k2, 2048.f));
  c[3] = __float2int_rn(__fmul_rn(k3, 2048.f));
}

// src [n][h0][w0][3] uint8 -> dst [n][h][w][3] uint8; grid (ceil(w/32), ceil(h/8), n), block (32, 8)
__global__ void __launch_bounds__(256)
resize_cubic_u8_kernel(const uint8_t* __restrict__ src, int h0, int w0, uint8_t* __restrict__ dst, int h, int w,
                       double scale_x, double scale_y) {
  const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y, n = blockIdx.z;
  if (x >= w || y >= h) return;
  int sx, sy, a[4], b[4];
  cv_cubic_axis(x, scale_x, sx, a);
  cv_cubic_axis(y, scale_y, sy, b);
  int xi[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) xi[k] = min(max(sx - 1 + k, 0), w0 - 1) * 3;
  int D[4][3];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const uint8_t* row = src + (static_cast<size_t>(n) * h0 + min(max(sy - 1 + r, 0), h0 - 1)) * w0 * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c)
      D[r][c] = row[xi[0] + c] * a[0] + row[xi[1] + c] * a[1] + row[xi[2] + c] * a[2] + row[xi[3] + c] * a[3];
  }
  const int simd_end = (w * 3) & ~7;
  const float inv = 1.f / 4194304.f;
  const float fb0 = __fmul_rn(static_cast<float>(b[0]), inv), fb1 = __fmul_rn(static_cast<float>(b[1]), inv);
  const float fb2 = __fmul_rn(static_cast<float>(b[2]), inv), fb3 = __fmul_rn(static_cast<float>(b[3]), inv);
  uint8_t* o = dst + ((static_cast<size_t>(n) * h + y) * w + x) * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    int v;
    if (x * 3 + c < simd_end) {
      float acc = __fmul_rn(static_cast<float>(D[3][c]), fb3);
      acc = __fadd_rn(__fmul_rn(static_cast<float>(D[2][c]), fb2), acc);
      acc = __fadd_rn(__fmul_rn(static_cast<float>(D[1][c]), fb1), acc);
      acc = __fadd_rn(__fmul_rn(static_cast<float>(D[0][c]), fb0), acc);
      v = __float2int_rn(acc);
    } else {
      v = (D[0][c] * b[0] + D[1][c] * b[1] + D[2][c] * b[2] + D[3][c] * b[3] + (1 << 21)) >> 22;
    }
    o[c] = static_cast<uint8_t>(min(max(v, 0), 255));
  }
}

// pad_image (pose_detector.py:46-55): copy src [h][w][3] into the top-left corner of dst [ph][pw][3] and fill the
// bottom / right margin with the per-channel pad value (104, 117, 123 in detect_precise, :445).
__global__ void __launch_bounds__(256)
pad_image_u8_kernel(const uint8_t* __restrict__ src, int h, int w, uint8_t* __restrict__ dst, int ph, int pw, int v0,
                    int v1, int v2) {
  const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
  if (x >= pw || y >= ph) return;
  uint8_t* o = dst + (static_cast<size_t>(y) * pw + x) * 3;
  if (x < w && y < h) {
    const uint8_t* i = src + (static_cast<size_t>(y) * w + x) * 3;
    o[0] = i[0]; o[1] = i[1]; o[2] = i[2];
  } else {
    o[0] = static_cast<uint8_t>(v0); o[1] = static_cast<uint8_t>(v1); o[2] = static_cast<uint8_t>(v2);
  }
}

}  // namespace opb
