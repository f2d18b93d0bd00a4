// upsample.cuh -- map upsampling.
//   upsample_bilinear_ac_kernel : F.resize_images (Chainer, align-corners bilinear) of
//       pose_detector.py:501-502.  Restates Chainer's published ResizeImages.forward: sample
//       grid u = linspace(0, w-1, W) in float64, u0 = clip(floor(u), 0, w-2), the four tap
//       weights formed in float64 and cast to float32, y = w1*x00; y += w2*x01; y += w3*x10;
//       y += w4*x11 in float32 (no FMA contraction) -> bit-exact vs the oracle.
//   resize_cubic_kernel : cv2.resize(..., INTER_CUBIC) for float32 maps (pose_detector.py
//       :461-467): Keys cubic A=-0.75, half-pixel centres, replicate border, float32 taps.
#pragma once
#include <cuda_runtime.h>

namespace opb {

__device__ __forceinline__ void ac_axis(int i, int n_in, int n_out, int& i0, double& f) {
  // numpy.linspace(0, n_in-1, n_out)[i]: i*step (+0), last element exactly n_in-1
  double u;
  if (n_out == 1) {
    u = 0.0;
  } else if (i == n_out - 1) {
    u = static_cast<double>(n_in - 1);
  } else {
    const double step = __ddiv_rn(static_cast<double>(n_in - 1), static_cast<double>(n_out - 1));
    u = __dmul_rn(static_cast<double>(i), step);
  }
  int k = static_cast<int>(floor(u));
  k = max(0, min(k, n_in - 2));
  i0 = k;
  f = u;
}

// in [planes][h][w] -> out [planes][H][W]; grid (ceil(W/32), ceil(H/8), plane_groups).
// The float64 grid values depend on x or y only: one warp computes them per block into shared
// memory; each thread then forms its four float32 weights (4 DMUL) once and streams
// `planes_per_block` output planes.
__global__ void __launch_bounds__(256)
upsample_bilinear_ac_kernel(const float* __restrict__ in, int planes, int h, int w, float* __restrict__ out, int H,
                            int W, int planes_per_block) {
  __shared__ double s_du0[32], s_du1[32], s_dv0[8], s_dv1[8];
  __shared__ int s_u0[32], s_v0[8];
  const int tid = threadIdx.y * 32 + threadIdx.x;
  if (tid < 32) {
    const int xx = min(blockIdx.x * 32 + tid, W - 1);
    int u0; double u;
    ac_axis(xx, w, W, u0, u);
    s_u0[tid] = u0;
    s_du1[tid] = __dsub_rn(static_cast<double>(u0 + 1), u);
    s_du0[tid] = __dsub_rn(u, static_cast<double>(u0));
  } else if (tid < 40) {
    const int yy = min(blockIdx.y * 8 + (tid - 32), H - 1);
    int v0; double v;
    ac_axis(yy, h, H, v0, v);
    s_v0[tid - 32] = v0;
    s_dv1[tid - 32] = __dsub_rn(static_cast<double>(v0 + 1), v);
    s_dv0[tid - 32] = __dsub_rn(v, static_cast<double>(v0));
  }
  __syncthreads();
  const int x = blockIdx.x * 32 + threadIdx.x;
  const int y = blockIdx.y * 8 + threadIdx.y;
  if (x >= W || y >= H) return;
  const int u0 = s_u0[threadIdx.x], v0 = s_v0[threadIdx.y];
  const double du1 = s_du1[threadIdx.x], du0 = s_du0[threadIdx.x];
  const double dv1 = s_dv1[threadIdx.y], dv0 = s_dv0[threadIdx.y];
  const float w1 = static_cast<float>(__dmul_rn(du1, dv1));
  const float w2 = static_cast<float>(__dmul_rn(du0, dv1));
  const float w3 = static_cast<float>(__dmul_rn(du1, dv0));
  const float w4 = static_cast<float>(__dmul_rn(du0, dv0));
  const int o00 = v0 * w + u0, o01 = o00 + 1, o10 = o00 + w, o11 = o10 + 1;
  const int p_begin = blockIdx.z * planes_per_block;
  const int p_end = min(planes, p_begin + planes_per_block);
  const size_t in_plane = static_cast<size_t>(h) * w, out_plane = static_cast<size_t>(H) * W;
  const float* src = in + p_begin * in_plane;
  float* dst = out + p_begin * out_plane + static_cast<size_t>(y) * W + x;
#pragma unroll 4
  for (int p = p_begin; p < p_end; ++p) {
    float r = __fmul_rn(w1, __ldg(src + o00));
    r = __fadd_rn(r, __fmul_rn(w2, __ldg(src + o01)));
    r = __fadd_rn(r, __fmul_rn(w3, __ldg(src + o10)));
    r = __fadd_rn(r, __fmul_rn(w4, __ldg(src + o11)));
    __stcs(dst, r);   // streaming store: the full-resolution map is written once
    src += in_plane;
    dst += out_plane;
  }
}

// Vectorised variant: one thread = 4 consecutive output columns of one row -> one 16-byte
// streaming store per plane.  When the horizontal scale is >= 3 the four outputs read at most
// three source columns (u0, u0+1, u0+2), so 6 loads replace 16.  Same arithmetic (and therefore
// the same bits) as upsample_bilinear_ac_kernel.  Requires W % 4 == 0.
__global__ void __launch_bounds__(256)
upsample_bilinear_ac_v4_kernel(const float* __restrict__ in, int planes, int h, int w, float* __restrict__ out, int H,
                               int W, int planes_per_block) {
  __shared__ double s_du0[128], s_du1[128], s_dv0[8], s_dv1[8];
  __shared__ int s_u0[128], s_v0[8];
  const int tid = threadIdx.y * 32 + threadIdx.x;
  if (tid < 128) {
    const int xx = min(blockIdx.x * 128 + tid, W - 1);
    int u0; double u;
    ac_axis(xx, w, W, u0, u);
    s_u0[tid] = u0;
    s_du1[tid] = __dsub_rn(static_cast<double>(u0 + 1), u);
    s_du0[tid] = __dsub_rn(u, static_cast<double>(u0));
  } else if (tid < 136) {
    const int yy = min(blockIdx.y * 8 + (tid - 128), H - 1);
    int v0; double v;
    ac_axis(yy, h, H, v0, v);
    s_v0[tid - 128] = v0;
    s_dv1[tid - 128] = __dsub_rn(static_cast<double>(v0 + 1), v);
    s_dv0[tid - 128] = __dsub_rn(v, static_cast<double>(v0));
  }
  __syncthreads();
  const int x = blockIdx.x * 128 + threadIdx.x * 4;
  const int y = blockIdx.y * 8 + threadIdx.y;
  if (x >= W || y >= H) return;
  const int v0 = s_v0[threadIdx.y];
  const double dv1 = s_dv1[threadIdx.y], dv0 = s_dv0[threadIdx.y];
  float w1[4], w2[4], w3[4], w4[4];
  int du[4];
  const int ub = s_u0[threadIdx.x * 4];
  bool compact = true;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int t = threadIdx.x * 4 + k;
    du[k] = s_u0[t] - ub;
    compact = compact && (du[k] <= 1);
    w1[k] = static_cast<float>(__dmul_rn(s_du1[t], dv1));
    w2[k] = static_cast<float>(__dmul_rn(s_du0[t], dv1));
    w3[k] = static_cast<float>(__dmul_rn(s_du1[t], dv0));
    w4[k] = static_cast<float>(__dmul_rn(s_du0[t], dv0));
  }
  const int base = v0 * w + ub;
  const int p_begin = blockIdx.z * planes_per_block;
  const int p_end = min(planes, p_begin + planes_per_block);
  const size_t in_plane = static_cast<size_t>(h) * w, out_plane = static_cast<size_t>(H) * W;
  const float* src = in + p_begin * in_plane + base;
  float* dst = out + p_begin * out_plane + static_cast<size_t>(y) * W + x;
  const bool c2 = (ub + 2 < w);   // third source column exists
  if (compact) {
#pragma unroll 2
    for (int p = p_begin; p < p_end; ++p) {
      const float a0 = __ldg(src), a1 = __ldg(src + 1), a2 = c2 ? __ldg(src + 2) : 0.f;
      const float b0 = __ldg(src + w), b1 = __ldg(src + w + 1), b2 = c2 ? __ldg(src + w + 2) : 0.f;
      float r[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float x00 = du[k] ? a1 : a0, x01 = du[k] ? a2 : a1, x10 = du[k] ? b1 : b0, x11 = du[k] ? b2 : b1;
        float t = __fmul_rn(w1[k], x00);
        t = __fadd_rn(t, __fmul_rn(w2[k], x01));
        t = __fadd_rn(t, __fmul_rn(w3[k], x10));
        t = __fadd_rn(t, __fmul_rn(w4[k], x11));
        r[k] = t;
      }
      __stcs(reinterpret_cast<float4*>(dst), make_float4(r[0], r[1], r[2], r[3]));
      src += in_plane;
      dst += out_plane;
    }
  } else {
    for (int p = p_begin; p < p_end; ++p) {
      float r[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float* q = src + du[k];
        float t = __fmul_rn(w1[k], __ldg(q));
        t = __fadd_rn(t, __fmul_rn(w2[k], __ldg(q + 1)));
        t = __fadd_rn(t, __fmul_rn(w3[k], __ldg(q + w)));
        t = __fadd_rn(t, __fmul_rn(w4[k], __ldg(q + w + 1)));
        r[k] = t;
      }
      __stcs(reinterpret_cast<float4*>(dst), make_float4(r[0], r[1], r[2], r[3]));
      src += in_plane;
      dst += out_plane;
    }
  }
}

// ---- point sampling of the align-corners bilinear map ------------------------------------------
// The value upsample_bilinear_ac_kernel writes at output position (Y, X), computed on demand from the
// low-resolution plane with the same operations in the same order (bit-identical): consumers that
// touch only a few full-resolution positions (PAF line integrals) or that stage a tile anyway (the
// peak kernel) can then skip the materialised full-resolution map and its HBM round trip.
struct AcAxis {
  int i0;          // left / upper source index
  double f0, f1;   // u - i0, (i0 + 1) - u
};

__device__ __forceinline__ double ac_step(int n_in, int n_out) {
  return (n_out > 1) ? __ddiv_rn(static_cast<double>(n_in - 1), static_cast<double>(n_out - 1)) : 0.0;
}

// ac_axis with the (loop-invariant) linspace step hoisted
__device__ __forceinline__ AcAxis ac_axis_frac(int i, int n_in, int n_out, double step) {
  double u;
  if (n_out == 1) u = 0.0;
  else if (i == n_out - 1) u = static_cast<double>(n_in - 1);
  else u = __dmul_rn(static_cast<double>(i), step);
  int k = static_cast<int>(floor(u));
  k = max(0, min(k, n_in - 2));
  AcAxis a;
  a.i0 = k;
  a.f1 = __dsub_rn(static_cast<double>(k + 1), u);
  a.f0 = __dsub_rn(u, static_cast<double>(k));
  return a;
}

struct AcTap {
  int o00;                 // offset of the upper-left source sample in the plane
  float w1, w2, w3, w4;    // weights of x00, x01, x10, x11
};

__device__ __forceinline__ AcTap ac_tap(const AcAxis& ax, const AcAxis& ay, int w) {
  AcTap t;
  t.o00 = ay.i0 * w + ax.i0;
  t.w1 = static_cast<float>(__dmul_rn(ax.f1, ay.f1));
  t.w2 = static_cast<float>(__dmul_rn(ax.f0, ay.f1));
  t.w3 = static_cast<float>(__dmul_rn(ax.f1, ay.f0));
  t.w4 = static_cast<float>(__dmul_rn(ax.f0, ay.f0));
  return t;
}

__device__ __forceinline__ float ac_sample(const float* __restrict__ plane, int w, const AcTap& t) {
  const float* q = plane + t.o00;
  float r = __fmul_rn(t.w1, __ldg(q));
  r = __fadd_rn(r, __fmul_rn(t.w2, __ldg(q + 1)));
  r = __fadd_rn(r, __fmul_rn(t.w3, __ldg(q + w)));
  r = __fadd_rn(r, __fmul_rn(t.w4, __ldg(q + w + 1)));
  return r;
}

// ---- ragged batches: crops of different sizes in one launch -------------------------------------
// Crop i's full-resolution maps are [planes][h][w] floats at `off` of one packed buffer.  A launch covers every crop
// with a flat block index: the crop's blocks start at blk_up (upsample: plane groups x 32x8 tiles) or at blk_plane
// (one block per plane and 32x8 tile: the Gaussian passes); ragged_crop_of finds the crop of a block.
struct RaggedMaps {
  long long off;      // float offset of the crop's first plane in the packed buffer
  int h, w;
  int tiles_x, tiles; // ceil(w/32), ceil(w/32) * ceil(h/8)
  int blk_up;         // first block of the crop in upsample_bilinear_ac_ragged_kernel
  int blk_plane;      // first block of the crop in the per-plane-tile launches
  int mirror;         // keypoints: report positions in the horizontally flipped maps
  int pad_;
};

// the last crop whose first block (blk_up or blk_plane) is <= b
__device__ __forceinline__ int ragged_crop_of(const RaggedMaps* __restrict__ c, int n, int b, bool up) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((up ? c[mid].blk_up : c[mid].blk_plane) <= b) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

// F.resize_images of every crop's low-resolution maps: in = slot i at in + i * in_stride ([planes][h][w] of it are
// read), out = crop i's [planes][crops[i].h][crops[i].w] at crops[i].off.  Same operations in the same order as
// upsample_bilinear_ac_kernel (ac_axis_frac / ac_tap / ac_sample), so the same bits.  Block (32, 8); one block =
// one 32x8 tile of `planes_per_block` planes.
__global__ void __launch_bounds__(256)
upsample_bilinear_ac_ragged_kernel(const float* __restrict__ in, long long in_stride, int planes, int h, int w,
                                   const RaggedMaps* __restrict__ crops, int n, float* __restrict__ out,
                                   int planes_per_block) {
  const int i = ragged_crop_of(crops, n, blockIdx.x, true);
  const RaggedMaps c = crops[i];
  const int local = blockIdx.x - c.blk_up, group = local / c.tiles, tile = local - group * c.tiles;
  const int ty = tile / c.tiles_x, tx = tile - ty * c.tiles_x;
  const int x = tx * 32 + threadIdx.x, y = ty * 8 + threadIdx.y;
  if (x >= c.w || y >= c.h) return;
  const AcTap t = ac_tap(ac_axis_frac(x, w, c.w, ac_step(w, c.w)), ac_axis_frac(y, h, c.h, ac_step(h, c.h)), w);
  const int p_begin = group * planes_per_block, p_end = min(planes, p_begin + planes_per_block);
  const size_t in_plane = static_cast<size_t>(h) * w, out_plane = static_cast<size_t>(c.h) * c.w;
  const float* src = in + i * in_stride + p_begin * in_plane;
  float* dst = out + c.off + p_begin * out_plane + static_cast<size_t>(y) * c.w + x;
  for (int p = p_begin; p < p_end; ++p) {
    __stcs(dst, ac_sample(src, w, t));
    src += in_plane;
    dst += out_plane;
  }
}

// ---- cv2 INTER_CUBIC for float32 (A = -0.75), separable, replicate border ------------------
__device__ __forceinline__ void cubic_taps(float t, float (&c)[4]) {
  const float A = -0.75f;
  c[0] = ((A * (t + 1) - 5 * A) * (t + 1) + 8 * A) * (t + 1) - 4 * A;
  c[1] = ((A + 2) * t - (A + 3)) * t * t + 1;
  c[2] = ((A + 2) * (1 - t) - (A + 3)) * (1 - t) * (1 - t) + 1;
  c[3] = 1.f - c[0] - c[1] - c[2];
}

// in: HWC float32 [h][w][C] (cv2 layout) or planar [C][h][w] selected by in_planar;
// out planar [C][H][W] (cropped region [crop_h, crop_w] of the (H_full, W_full) resize),
// out = ((accumulate ? out : 0) + value) * scale.
__global__ void __launch_bounds__(256)
resize_cubic_kernel(const float* __restrict__ in, int C, int h, int w, float* __restrict__ out, int H_full,
                    int W_full, int crop_h, int crop_w, int accumulate, float divisor) {
  const int x = blockIdx.x * 32 + threadIdx.x;
  const int y = blockIdx.y * 8 + threadIdx.y;
  if (x >= crop_w || y >= crop_h) return;
  // cv2: fx = (x + 0.5) * (w / W_full) - 0.5 with scale computed in double, cast to float
  // cv2::resize: inv_scale = dsize/ssize (double); scale = 1./inv_scale
  const double sx = 1.0 / (static_cast<double>(W_full) / w), sy = 1.0 / (static_cast<double>(H_full) / h);
  float fx = static_cast<float>((x + 0.5) * sx - 0.5);
  float fy = static_cast<float>((y + 0.5) * sy - 0.5);
  int ix = static_cast<int>(floorf(fx)), iy = static_cast<int>(floorf(fy));
  fx -= ix;
  fy -= iy;
  float cx[4], cy[4];
  cubic_taps(fx, cx);
  cubic_taps(fy, cy);
  int xs[4], ys[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    xs[k] = min(max(ix - 1 + k, 0), w - 1);
    ys[k] = min(max(iy - 1 + k, 0), h - 1);
  }
  const size_t in_plane = static_cast<size_t>(h) * w, out_plane = static_cast<size_t>(crop_h) * crop_w;
  for (int c = blockIdx.z; c < C; c += gridDim.z) {
    const float* src = in + c * in_plane;
    float acc = 0.f;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const float* row = src + static_cast<size_t>(ys[r]) * w;
      const float hsum = __ldg(row + xs[0]) * cx[0] + __ldg(row + xs[1]) * cx[1] + __ldg(row + xs[2]) * cx[2] +
                         __ldg(row + xs[3]) * cx[3];
      acc += hsum * cy[r];
    }
    float* o = out + c * out_plane + static_cast<size_t>(y) * crop_w + x;
    const float sum = __fadd_rn(accumulate ? *o : 0.f, acc);
    *o = divisor > 0.f ? __fdiv_rn(sum, divisor) : sum;   // `/ len(scales)` (pose_detector.py:471-472) on the last pass, a true division
  }
}

}  // namespace opb
