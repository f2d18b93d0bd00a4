// keypoints.cuh -- post-process of the face / hand nets: FaceDetector.compute_peaks_from_heatmaps
// (face_detector.py:55-67) == HandDetector.compute_peaks_from_heatmaps (hand_detector.py:65-77), CPU branch:
//   per channel (background excluded)  g = scipy.ndimage.gaussian_filter(map, sigma = 2.5);  m = g.max();
//   m > thresh  ->  [x, y, m]  at  np.where(g == m)
// The smoothing restates scipy's arithmetic exactly (see peaks.cuh): 21 taps, 'reflect' boundary, axis-0 pass then
// axis-1 pass, each  acc = x0*w0;  for j = -R..-1: acc += (x[j] + x[-j]) * w[j]  in float64, stored as float32.
// HBM-bound (two 4-byte streams per pass); the maps are crops of at most a few hundred pixels a side.
// Every kernel covers a ragged batch of crops (RaggedMaps, upsample.cuh) in one launch; one crop is the batch of one.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "peaks.cuh"
#include "upsample.cuh"

namespace opb {

// One separable pass over every plane of every crop. AXIS 0: along y (first), AXIS 1: along x (second).
// grid (sum over crops of planes * tiles), block (32, 8).
template <int AXIS>
__global__ void __launch_bounds__(256)
gauss_pass_ragged_kernel(const float* __restrict__ in, float* __restrict__ out, const RaggedMaps* __restrict__ crops,
                         int n, GaussTaps taps) {
  const RaggedMaps c = crops[ragged_crop_of(crops, n, blockIdx.x, false)];
  const int local = blockIdx.x - c.blk_plane, p = local / c.tiles, tile = local - p * c.tiles;
  const int ty = tile / c.tiles_x, tx = tile - ty * c.tiles_x;
  const int H = c.h, W = c.w;
  const int x = tx * 32 + threadIdx.x, y = ty * 8 + threadIdx.y;
  if (x >= W || y >= H) return;
  const size_t plane = c.off + static_cast<size_t>(p) * H * W;
  const float* src = in + plane;
  const int R = taps.radius;
  const int n_ax = AXIS == 0 ? H : W, i0 = AXIS == 0 ? y : x;
  const size_t stride = AXIS == 0 ? W : 1;
  const float* line = AXIS == 0 ? src + x : src + static_cast<size_t>(y) * W;
  double acc = __dmul_rn(static_cast<double>(line[i0 * stride]), taps.w[R]);
  for (int j = -R; j < 0; ++j) {
    const double a = static_cast<double>(line[reflect_index(i0 + j, n_ax) * stride]);
    const double b = static_cast<double>(line[reflect_index(i0 - j, n_ax) * stride]);
    acc = __dadd_rn(acc, __dmul_rn(__dadd_rn(a, b), taps.w[R + j]));
  }
  out[plane + static_cast<size_t>(y) * W + x] = static_cast<float>(acc);
}

struct ChannelMax {
  float value;      // maximum of the smoothed map
  int32_t count;    // number of pixels equal to it (np.where(g == m) length)
  int32_t key0;     // row-major index y*W + x of the first such pixel (in the possibly mirrored map)
  int32_t key1;     // ... of the second one (count >= 2), else -1
};

// One block per (crop, plane): block b = crop b / planes, plane b % planes; out[b].  The crop's `mirror`: report
// positions of the horizontally flipped map (cv2.flip(maps, 1), hand_detector.py:46-47); the Gaussian commutes
// exactly with the flip (a + b is commutative), only the row-major order of exact ties changes.
__global__ void __launch_bounds__(256)
channel_argmax_ragged_kernel(const float* __restrict__ maps, const RaggedMaps* __restrict__ crops, int planes,
                             ChannelMax* __restrict__ out) {
  const RaggedMaps c = crops[blockIdx.x / planes];
  const int H = c.h, W = c.w, mirror = c.mirror;
  const float* m = maps + c.off + static_cast<size_t>(blockIdx.x % planes) * H * W;
  const int n = H * W;
  __shared__ float s_max[8];
  __shared__ int s_cnt, s_k0, s_k1;
  float best = -INFINITY;
  for (int i = threadIdx.x; i < n; i += 256) best = fmaxf(best, m[i]);
  for (int o = 16; o; o >>= 1) best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = best;
  if (threadIdx.x == 0) { s_cnt = 0; s_k0 = n; s_k1 = n; }
  __syncthreads();
  best = s_max[0];
  for (int w = 1; w < 8; ++w) best = fmaxf(best, s_max[w]);
  auto key_of = [&](int i) { const int y = i / W, x = i - y * W; return mirror ? y * W + (W - 1 - x) : i; };
  for (int i = threadIdx.x; i < n; i += 256)
    if (m[i] == best) { atomicAdd(&s_cnt, 1); atomicMin(&s_k0, key_of(i)); }
  __syncthreads();
  if (s_cnt > 1)
    for (int i = threadIdx.x; i < n; i += 256)
      if (m[i] == best) { const int k = key_of(i); if (k != s_k0) atomicMin(&s_k1, k); }
  __syncthreads();
  if (threadIdx.x == 0) {
    ChannelMax r;
    r.value = best; r.count = s_cnt; r.key0 = s_k0; r.key1 = (s_cnt > 1) ? s_k1 : -1;
    out[blockIdx.x] = r;
  }
}

}  // namespace opb
