// Gradient clipping on the device, ahead of the fused Adam step (Lightning's Trainer(gradient_clip_val=...,
// gradient_clip_algorithm="norm" | "value"), i.e. torch.nn.utils.clip_grad_norm_ / clip_grad_value_ on the averaged
// gradient, once per optimizer step):
//   * grad_norm_partial_kernel + grad_norm_finalize_kernel: the global L2 norm of one flat fp32 buffer times
//     grad_scale, and clip_grad_norm_'s coefficient, written to a device buffer -- no host round trip;
//   * adam_clip_kernel: adam_kernel (edge_kernels.cuh) with the gradient scaled by that coefficient, or clamped.
#pragma once
#include <cstdint>

namespace xmm {

// ------------------------------------------------------------------------------ global L2 norm
// Squares are formed and added in fp64: an fp32 square under- or overflows for |g| < ~1e-23 or > ~1.8e19, and the
// sum of 38 M of them must not lose the small ones.  The order of every addition is fixed by n alone: CTA b owns
// float4s [b * kNormChunk4, (b + 1) * kNormChunk4) (the last CTA also the n % 4 scalar tail), each thread adds its
// kNormVec float4s in order, the warp adds by a fixed xor tree, the CTA in warp order, and the finalize kernel adds
// the per-CTA partials (one double per CTA, slot b) in slot order.  Same bits on every run, whatever the SM count.
constexpr int kNormThreads = 256;
constexpr int kNormVec = 8;                                  // float4 loads in flight per thread
constexpr size_t kNormChunk4 = size_t(kNormThreads) * kNormVec;  // float4s per CTA (32 KB)

__host__ __device__ inline size_t grad_norm_blocks(size_t n) { return (n + 4 * kNormChunk4 - 1) / (4 * kNormChunk4); }

__device__ __forceinline__ double block_sum_fixed(double s, double* red) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) red[warp] = s;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < int(blockDim.x >> 5); ++w) t += red[w];
  return t;  // valid in thread 0
}

__global__ void __launch_bounds__(kNormThreads) grad_norm_partial_kernel(const float* __restrict__ g, size_t n,
                                                                        double* __restrict__ partials) {
  __shared__ double red[kNormThreads / 32];
  const size_t n4 = n / 4;
  const size_t base = size_t(blockIdx.x) * kNormChunk4 + threadIdx.x;
  const float4* g4 = reinterpret_cast<const float4*>(g);
  float4 v[kNormVec];
#pragma unroll
  for (int j = 0; j < kNormVec; ++j) {
    const size_t i = base + size_t(j) * kNormThreads;
    v[j] = i < n4 ? __ldg(g4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < kNormVec; ++j) {
    s = fma(double(v[j].x), double(v[j].x), s);
    s = fma(double(v[j].y), double(v[j].y), s);
    s = fma(double(v[j].z), double(v[j].z), s);
    s = fma(double(v[j].w), double(v[j].w), s);
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x < n - 4 * n4) {
    const double x = g[4 * n4 + threadIdx.x];
    s = fma(x, x, s);
  }
  s = block_sum_fixed(s, red);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

// out[0] = ||g||_2 * |grad_scale| (rounded once to fp32), out[1] = clip_grad_norm_'s coefficient computed as torch
// computes it in fp32: min(max_norm * (1 / (total + 1e-6)), 1) -- `max_norm / t` on a tensor is
// t.reciprocal() * max_norm -- with NaN kept (torch.clamp propagates it).  An inf norm gives 0, a NaN norm NaN.
__global__ void __launch_bounds__(kNormThreads) grad_norm_finalize_kernel(const double* __restrict__ partials,
                                                                         size_t count, float grad_scale,
                                                                         float max_norm, float* __restrict__ out) {
  __shared__ double red[kNormThreads / 32];
  double s = 0.0;
  for (size_t i = threadIdx.x; i < count; i += kNormThreads) s += partials[i];
  s = block_sum_fixed(s, red);
  if (threadIdx.x == 0) {
    const float total = float(sqrt(s) * fabs(double(grad_scale)));
    const float r = 1.0f / (total + 1e-6f);
    const float c = r * max_norm;
    out[0] = total;
    out[1] = c > 1.0f ? 1.0f : c;
  }
}

// ------------------------------------------------------------------------------ Adam on a clipped gradient
// adam_kernel with gv = g * (grad_scale * coef[0]) (coef != nullptr: clip by norm) or
// gv = clamp(g * grad_scale, -clip_value, clip_value) (clip by value; NaN stays NaN, as torch.clamp keeps it).
// The moment updates spell out the roundings nvcc gives adam_kernel's expressions when it contracts them to FMAs
// (fma(b1, m, (1 - b1) * g) and fma(b2, v, (1 - b2) * g * g); left to contraction here, the same source compiles to
// the other pairing), so a coefficient of 1 at grad_scale 1 gives adam_kernel's bits.
__global__ void adam_clip_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                 float* __restrict__ v, size_t n, float lr, float b1, float b2, float eps, float bc1,
                                 float bc2_sqrt, float grad_scale, const float* __restrict__ coef,
                                 float clip_value) {
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float gv;
  if (coef != nullptr) {
    gv = g[i] * (grad_scale * coef[0]);
  } else {
    gv = g[i] * grad_scale;
    gv = gv < -clip_value ? -clip_value : (gv > clip_value ? clip_value : gv);
  }
  const float mv = __fmaf_rn(b1, m[i], __fmul_rn(1.0f - b1, gv));
  const float vv = __fmaf_rn(b2, v[i], __fmul_rn(__fmul_rn(1.0f - b2, gv), gv));
  m[i] = mv;
  v[i] = vv;
  const float denom = sqrtf(vv) / bc2_sqrt + eps;
  p[i] -= (lr / bc1) * (mv / denom);
}

}  // namespace xmm
