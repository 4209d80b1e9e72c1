// adaptive.cuh -- adaptive sampling in sum mode (fspt_set_adaptive): before each wave, the pixels of a band whose mean
// has not converged yet are listed, and the wave renders only those.  No counterpart in the reference.
//
// A pixel's samples depend only on the pixel and the tick's rand bases (slot = j * S + s, path_to_pixel), so rendering
// a subset of the pixels changes none of their values.  A pixel that is not rendered keeps its sum, count and moment,
// so under a fixed threshold it never becomes active again: the ticks a pixel received are always a prefix of the
// render's ticks, and the pixel equals the uniform sum-mode render after that many ticks, bit for bit.
#pragma once
#include "device_common.cuh"
#include "shade.cuh"

// Floor of the mean in the relative-error test: a near-black pixel would otherwise need an absolute error of zero and
// could never stop.
#define FSPT_ADAPTIVE_MEAN_FLOOR 1e-3f

// The rule, every step in f32 in this order (lumaCoefs of draw.fs; n = the pixel's sample count, m2 = its sum of
// squared sample luminances):
//   mean = ((r*Lr + g*Lg) + b*Lb) / n,  var = (m2/n - mean*mean) * (n / (n-1)),
//   active = n < min_samples  ||  sqrt(max(var, 0) / n) > max_rel_error * max(mean, FLOOR)
__device__ __forceinline__ bool pixel_active(float4 acc, float m2, float max_rel_error, int min_samples) {
  const float n = acc.w;
  if (n < (float)min_samples) return true;
  const float mean = ((acc.x * 0.2126f + acc.y * 0.7152f) + acc.z * 0.0722f) / n;
  const float var = (m2 / n - mean * mean) * (n / (n - 1.0f));
  return sqrtf(fmaxf(var, 0.0f) / n) > max_rel_error * fmaxf(mean, FSPT_ADAPTIVE_MEAN_FLOOR);
}

// One thread per slot j of the rectangle f (in its slot order: 8x4 tiles or row-major, as set_rect chose).  The j of
// every active pixel goes to `list` (NULL: only counted), their number is added to *n_active, and S samples per active
// pixel to *samples (NULL: not counted).  Order across blocks is free -- no result depends on it -- but inside a block
// the active slots keep their order (warp ballot + block prefix, one atomicAdd per block), so the warps of the wave
// stay spatially coherent.
__global__ void __launch_bounds__(256) k_select_active(const FrameParams f, const float4* __restrict__ fb,
                                                       const float* __restrict__ m2, float max_rel_error, int min_samples,
                                                       int* list, int* n_active, unsigned long long* samples, int S) {
  __shared__ int s_warp[8];
  __shared__ int s_base;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  bool active = false;
  if (j < f.rw * f.rh) {
    int x, y;
    path_to_pixel(f, j, x, y);
    const size_t p = (size_t)(f.ry0 + y) * f.width + (size_t)(f.rx0 + x);
    active = pixel_active(fb[p], m2[p], max_rel_error, min_samples);
  }
  const unsigned m = __ballot_sync(0xffffffffu, active);
  if (lane == 0) s_warp[warp] = __popc(m);
  __syncthreads();
  if (threadIdx.x == 0) {
    int total = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { const int v = s_warp[w]; s_warp[w] = total; total += v; }
    s_base = total ? atomicAdd(n_active, total) : 0;
    if (samples && total) atomicAdd(samples, (unsigned long long)total * (unsigned long long)S);
  }
  __syncthreads();
  if (active && list) list[s_base + s_warp[warp] + __popc(m & ((1u << lane) - 1u))] = j;
}

// k_accumulate over the wave's list (sum mode): thread t accumulates the pixel of slot list[t] of the band's rectangle
// f, t < *n_active, and adds the squared luminance of each of its samples to its moment m2.
__global__ void __launch_bounds__(256) k_accumulate_active(const FrameParams f, const int* __restrict__ list,
                                                           const int* __restrict__ n_active,
                                                           const float4* __restrict__ sample_color, float4* fb,
                                                           float4* last_color, float* m2, int n_samples, int sanitize) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= *n_active) return;
  int x, y;
  path_to_pixel(f, list[t], x, y);
  const size_t p = (size_t)(f.ry0 + y) * f.width + (size_t)(f.rx0 + x);
  accumulate_pixel<true>(sample_color, fb, last_color, y * f.rw + x, p, n_samples, 0u, 1, sanitize, m2);
}
