// HBM-bound kernels at the two ends of the generator:
//   * normalize / denormalize  (transforms/normalize.py:66-92, data/dataset.py:41-42)
//   * conv_first  (1..4 -> F channels, generator_rrdb.py:31-37,67): K = 9*Cin is far too small
//     for an MMA, so it is a CUDA-core stencil that writes the NHWC bf16 feature map;
//   * conv_last   (F -> 1..4 channels, generator_rrdb.py:48-54,107-108,132-135): a per-pixel
//     9*F dot product fused with the DN input residual and both clamps (model.py:49).
#pragma once
#include <cuda_bf16.h>
#include <cstdint>

#include "conv3x3_tc.cuh"  // unpack8 / pack8

namespace xmm {

enum StretchMode : int { kLinear = 0, kSqrt = 1, kAsinh = 2, kLog = 3 };

__device__ __forceinline__ float stretch_fwd(float x, int mode) {
  switch (mode) {
    case kSqrt: return sqrtf(x);
    case kAsinh: return asinhf(x / 0.02f) / asinhf(50.0f);   // normalize.py:4-10
    case kLog: return logf(1000.0f * x + 1.0f) / logf(1000.0f);  // normalize.py:23-26
    default: return x;
  }
}
__device__ __forceinline__ float stretch_inv(float x, int mode) {
  switch (mode) {
    case kSqrt: return x * x;
    case kAsinh: return 0.02f * sinhf(x * asinhf(50.0f));    // normalize.py:13-19
    case kLog: return (powf(1000.0f, x) - 1.0f) / 1000.0f;  // normalize.py:29-32
    default: return x;
  }
}

struct NormalizeArgs {
  const void* in;        // fp32 or int32 [n]
  const uint8_t* mask;   // optional detector mask, broadcast over the batch: [mask_n]
  float* out;            // fp32 [n]
  size_t n;
  size_t mask_n;         // pixels per image (mask period)
  int in_is_int32;
  float pre_scale;       // multiplies the raw value first (1/exposure: counts -> rate)
  float max_val;         // > 0 ; (the max_val <= 0 branch divides by *dyn_max instead)
  const float* dyn_max;  // device scalar, used when max_val <= 0
  int mode;
};

// 4 elements per thread, 16-byte loads/stores; tail handled by the last threads scalar-wise.
__global__ void normalize_kernel(const NormalizeArgs a) {
  const size_t i4 = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i4 >= a.n) return;
  const bool clamp_in = a.max_val > 0.0f;
  const float mx = clamp_in ? a.max_val : *a.dyn_max;
  float v[4];
  const int cnt = (a.n - i4 >= 4) ? 4 : int(a.n - i4);
  if (cnt == 4) {
    if (a.in_is_int32) {
      const int4 q = *reinterpret_cast<const int4*>(static_cast<const int*>(a.in) + i4);
      v[0] = float(q.x); v[1] = float(q.y); v[2] = float(q.z); v[3] = float(q.w);
    } else {
      const float4 q = *reinterpret_cast<const float4*>(static_cast<const float*>(a.in) + i4);
      v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    }
  } else {
    for (int j = 0; j < cnt; ++j)
      v[j] = a.in_is_int32 ? float(static_cast<const int*>(a.in)[i4 + j]) : static_cast<const float*>(a.in)[i4 + j];
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (j < cnt) {
      float x = v[j] * a.pre_scale;
      if (a.mask != nullptr) x *= float(a.mask[(i4 + j) % a.mask_n]);
      // image / max_val is a true division in the reference; keep it a division so results are
      // bit-identical to torch (x * (1/max) differs in the last ulp).
      if (clamp_in) x = fminf(fmaxf(x, 0.0f), mx);
      x = x / mx;
      x = stretch_fwd(x, a.mode);
      v[j] = fminf(fmaxf(x, 0.0f), 1.0f);
    }
  }
  if (cnt == 4) {
    *reinterpret_cast<float4*>(a.out + i4) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
    for (int j = 0; j < cnt; ++j) a.out[i4 + j] = v[j];
  }
}

// out = clamp(max * denorm(x), 0, max); max_vals has max_n entries (1 = scalar, else one per image)
__global__ void denormalize_kernel(const float* __restrict__ in, float* __restrict__ out, size_t n, size_t per_image,
                                   const float* __restrict__ max_vals, int max_n, int mode) {
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float mx = max_vals[max_n == 1 ? 0 : (i / per_image)];
  float v = mx * stretch_inv(in[i], mode);
  out[i] = fminf(fmaxf(v, 0.0f), mx);
}

// out = norm_to(denorm_from(x)): the validation metric collection evaluates every metric under several
// normalisers (metrics/xmm_metric_collection.py:135-143: dataset_normalizer.denorm, then normalizer.norm) --
// one pass, 8 B per pixel, instead of two.
__global__ void restretch_kernel(const float* __restrict__ in, float* __restrict__ out, size_t n, int mode_from,
                                 int mode_to) {
  const size_t i4 = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i4 >= n) return;
  if (n - i4 >= 4) {
    float4 q = *reinterpret_cast<const float4*>(in + i4);
    q.x = stretch_fwd(stretch_inv(q.x, mode_from), mode_to);
    q.y = stretch_fwd(stretch_inv(q.y, mode_from), mode_to);
    q.z = stretch_fwd(stretch_inv(q.z, mode_from), mode_to);
    q.w = stretch_fwd(stretch_inv(q.w, mode_from), mode_to);
    *reinterpret_cast<float4*>(out + i4) = q;
  } else {
    for (size_t i = i4; i < n; ++i) out[i] = stretch_fwd(stretch_inv(in[i], mode_from), mode_to);
  }
}

// The data feed of one batch (data/dataset.py:24-49 _load_and_combine_simulations, data/tools.py:103-126
// reshape_img_to_res, data/dataset.py:258-270 normalisation), from raw FITS planes already in device memory:
//   v = (img + agn + bkg) * det_mask            int32 or fp32 counts, [B][h][w]; mask [h][w], broadcast
//   v = nearest-upsample(v, up) / up^2           optional ImageUpsample (real-SR targets)
//   zero-pad (or crop) to res_h x res_w with floor(diff/2) before, the rest after
//   out = clamp(stretch(clamp(v * pre_scale, 0, max) / max), 0, 1)       pre_scale = 1/exposure (SURVEY I4)
// One thread per output pixel: 4..12 B read (+1 mask) and 4 B written.
struct PrepareCountsArgs {
  const void* src[3];
  int nsrc, src_is_int32;
  const uint8_t* mask;
  int batch, h, w, up, res_h, res_w;
  float pre_scale;
  const float* pre_scale_dev;  // optional per-image scale (B floats), multiplied with pre_scale
  float max_val;
  int mode;
  float* out;
};

__global__ void prepare_counts_kernel(const PrepareCountsArgs a) {
  const size_t n = size_t(a.batch) * a.res_h * a.res_w;
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int X = int(i % a.res_w);
  const size_t t = i / a.res_w;
  const int Y = int(t % a.res_h);
  const int b = int(t / a.res_h);
  const int uh = a.h * a.up, uw = a.w * a.up;
  // floor division (a negative difference crops, as torch.nn.functional.pad with negative pads does)
  const int dyv = a.res_h - uh, dxv = a.res_w - uw;
  const int top = (dyv >= 0) ? dyv / 2 : -((-dyv + 1) / 2);
  const int left = (dxv >= 0) ? dxv / 2 : -((-dxv + 1) / 2);
  const int y = Y - top, x = X - left;
  float v = 0.0f;
  if (y >= 0 && y < uh && x >= 0 && x < uw) {
    const size_t sidx = (size_t(b) * a.h + y / a.up) * a.w + x / a.up;
    for (int k = 0; k < a.nsrc; ++k)
      v += a.src_is_int32 ? float(static_cast<const int*>(a.src[k])[sidx]) : static_cast<const float*>(a.src[k])[sidx];
    if (a.mask != nullptr) v *= float(a.mask[size_t(y / a.up) * a.w + x / a.up]);
    if (a.up > 1) v /= float(a.up * a.up);
  }
  float sc = a.pre_scale;
  if (a.pre_scale_dev != nullptr) sc *= a.pre_scale_dev[b];
  v *= sc;
  v = fminf(fmaxf(v, 0.0f), a.max_val);
  v = stretch_fwd(v / a.max_val, a.mode);
  a.out[i] = fminf(fmaxf(v, 0.0f), 1.0f);
}

// max over a float array (normalize's max_val <= 0 branch): atomicMax on the int view is valid for
// non-negative floats; negative inputs clamp to 0 which matches a counts image.
__global__ void max_kernel(const float* __restrict__ in, size_t n, float pre_scale, float* __restrict__ out) {
  float m = 0.0f;
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x)
    m = fmaxf(m, in[i] * pre_scale);
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(out), __float_as_int(m));
}

// nearest-neighbour upsample by an integer factor, divided by factor^2 (brightness preserving)
// -- transforms/imageupsample.py:10-26.  in [n_img][h][w] -> out [n_img][h*s][w*s]
__global__ void image_upsample_kernel(const float* __restrict__ in, float* __restrict__ out, size_t n_out, int h,
                                      int w, int s) {
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  const int ow = w * s, oh = h * s;
  const int ox = int(i % ow);
  const size_t t = i / ow;
  const int oy = int(t % oh);
  const size_t img = t / oh;
  out[i] = in[(img * h + oy / s) * w + ox / s] / float(s * s);
}

// ------------------------------------------------------------------------------ conv_first
struct ConvFirstArgs {
  const float* in;   // fp32 NCHW [B][cin][H][W]
  const float* w;    // fp32 OIHW [F][cin][3][3]
  const float* bias; // fp32 [F]
  __nv_bfloat16* out; int out_ctot, out_coff;
  __nv_bfloat16* out2; int out2_ctot, out2_coff;  // optional second copy (the trunk skip `fea`)
  int batch, cin, height, width;
  // backward use (data gradient of conv_last): the input image is a gradient that only passes
  // where the forward clamp did not saturate, and the result is multiplied by LeakyReLU'(act).
  const float* gate;          // optional, same shape as `in`: v = (0 <= gate <= 1) ? in : 0
  const __nv_bfloat16* mask;  // optional NHWC bf16 window: out *= (mask > 0 ? 1 : mask_slope)
  int mask_ctot, mask_coff;
  float mask_slope;
};

template <int F>
__global__ void __launch_bounds__(128) conv_first_kernel(const ConvFirstArgs a) {
  extern __shared__ float wsm[];  // [cin*9][F] + bias[F]
  const int kw = a.cin * 9;
  for (int i = threadIdx.x; i < kw * F; i += blockDim.x) {
    const int f = i % F, k = i / F;  // k = c*9 + tap
    wsm[i] = a.w[size_t(f) * kw + k];
  }
  for (int i = threadIdx.x; i < F; i += blockDim.x) wsm[kw * F + i] = a.bias ? a.bias[i] : 0.0f;
  __syncthreads();
  const size_t hw = size_t(a.height) * a.width;
  const size_t pix = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (pix >= hw * a.batch) return;
  const int b = int(pix / hw);
  const int rem = int(pix - size_t(b) * hw);
  const int y = rem / a.width, x = rem - y * a.width;
  float acc[F];
#pragma unroll
  for (int f = 0; f < F; ++f) acc[f] = wsm[kw * F + f];
  for (int c = 0; c < a.cin; ++c) {
    const float* ip = a.in + (size_t(b) * a.cin + c) * hw;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
      const int yy = y + dy - 1;
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const int xx = x + dx - 1;
        float v = 0.0f;
        if (yy >= 0 && yy < a.height && xx >= 0 && xx < a.width) {
          v = __ldg(ip + size_t(yy) * a.width + xx);
          if (a.gate != nullptr) {
            const float gt = __ldg(a.gate + (size_t(b) * a.cin + c) * hw + size_t(yy) * a.width + xx);
            if (!(gt >= 0.0f && gt <= 1.0f)) v = 0.0f;
          }
        }
        const float* wp = wsm + (c * 9 + dy * 3 + dx) * F;
#pragma unroll
        for (int f = 0; f < F; ++f) acc[f] = fmaf(v, wp[f], acc[f]);
      }
    }
  }
  if (a.mask != nullptr) {
    const uint4* mp = reinterpret_cast<const uint4*>(a.mask + pix * a.mask_ctot + a.mask_coff);
#pragma unroll
    for (int q = 0; q < F / 8; ++q) {
      float m[8];
      unpack8(__ldg(mp + q), m);
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[q * 8 + i] *= (m[i] > 0.0f ? 1.0f : a.mask_slope);
    }
  }
  uint4* op = reinterpret_cast<uint4*>(a.out + pix * a.out_ctot + a.out_coff);
#pragma unroll
  for (int q = 0; q < F / 8; ++q) op[q] = pack8(acc + q * 8);
  if (a.out2 != nullptr) {
    uint4* op2 = reinterpret_cast<uint4*>(a.out2 + pix * a.out2_ctot + a.out2_coff);
#pragma unroll
    for (int q = 0; q < F / 8; ++q) op2[q] = pack8(acc + q * 8);
  }
}

// ------------------------------------------------------------------------------ conv_last
struct ConvLastArgs {
  const __nv_bfloat16* in; int in_ctot, in_coff;  // NHWC bf16 window of F channels
  const float* w;     // fp32 OIHW [cout][F][3][3]
  const float* bias;  // fp32 [cout]
  const float* residual;  // optional fp32 NCHW [B][cout][H][W] (DN: the network input)
  float* out;         // fp32 NCHW [B][cout][H][W], clamped to [0,1] when clamp != 0
  float* pre;         // optional: un-clamped value (needed by the backward clamp mask)
  int batch, cout, height, width;
  int clamp;
};

template <int F>
__global__ void __launch_bounds__(128) conv_last_kernel(const ConvLastArgs a) {
  extern __shared__ float wsm[];  // [cout][9][F]
  for (int i = threadIdx.x; i < a.cout * 9 * F; i += blockDim.x) {
    const int f = i % F, t = (i / F) % 9, o = i / (9 * F);
    wsm[i] = a.w[(size_t(o) * F + f) * 9 + t];
  }
  __syncthreads();
  const size_t hw = size_t(a.height) * a.width;
  const size_t pix = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (pix >= hw * a.batch) return;
  const int b = int(pix / hw);
  const int rem = int(pix - size_t(b) * hw);
  const int y = rem / a.width, x = rem - y * a.width;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int dy = 0; dy < 3; ++dy) {
    const int yy = y + dy - 1;
    if (yy < 0 || yy >= a.height) continue;
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
      const int xx = x + dx - 1;
      if (xx < 0 || xx >= a.width) continue;
      const uint4* ip = reinterpret_cast<const uint4*>(a.in + ((size_t(b) * a.height + yy) * a.width + xx) * a.in_ctot + a.in_coff);
#pragma unroll
      for (int q = 0; q < F / 8; ++q) {
        float v[8];
        unpack8(__ldg(ip + q), v);
        for (int o = 0; o < a.cout; ++o) {
          const float* wp = wsm + (o * 9 + dy * 3 + dx) * F + q * 8;
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[o] = fmaf(v[i], wp[i], acc[o]);
        }
      }
    }
  }
  for (int o = 0; o < a.cout; ++o) {
    const size_t oi = (size_t(b) * a.cout + o) * hw + rem;
    float v = acc[o] + (a.bias ? a.bias[o] : 0.0f);
    if (a.residual != nullptr) v += a.residual[oi];
    if (a.pre != nullptr) a.pre[oi] = v;
    a.out[oi] = a.clamp ? fminf(fmaxf(v, 0.0f), 1.0f) : v;
  }
}

// ------------------------------------------------------------------------------ fused Adam
// torch.optim.Adam (models/model.py:239-247; no weight decay, no amsgrad) over ONE flat fp32 buffer
// holding every parameter of the generator: a single launch instead of ~130 per-tensor updates.
//   g = grad * grad_scale (1/world_size after the all-reduce)
//   m = b1*m + (1-b1)*g ; v = b2*v + (1-b2)*g*g ; p -= (lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps)
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, size_t n, float lr, float b1, float b2, float eps, float bc1,
                            float bc2_sqrt, float grad_scale) {
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gv = g[i] * grad_scale;
  const float mv = b1 * m[i] + (1.0f - b1) * gv;
  const float vv = b2 * v[i] + (1.0f - b2) * gv * gv;
  m[i] = mv;
  v[i] = vv;
  const float denom = sqrtf(vv) / bc2_sqrt + eps;
  p[i] -= (lr / bc1) * (mv / denom);
}

// ------------------------------------------------------------------------------ edge weight grads
// R[o][c][tap] (+)= sum_p s[o][p] * (V[p + off(tap)][c] + V2[p + off(tap)][c]),   S[o] (+)= sum_p s[o][p]
// with s an fp32 NCHW image (optionally gated by the forward clamp) and V a bf16 NHWC window.
//   conv_last:  s = dL/d(out), V = its input features          -> dW[o][c][tap] = R, db[o] = S
//   conv_first: s = the input image x, V = dL/d(fea)           -> dW[f][o][8-tap] = R[o][f][tap]
// One CTA (256 threads) owns `rows` image rows of one image.  The (gated) s rows, with a one-pixel zero halo, are
// staged in shared memory; V is then streamed ONCE, 16 bytes (8 channels) per thread and pixel, and every thread
// keeps an 8-channel x 9-tap accumulator block in registers: R[c][tap] += s[q - off(tap)] * V[q][c].  Warp
// shuffles, a shared-memory pass and one atomicAdd per (channel, tap) and CTA finish the sum.
// Deterministic form (ws != nullptr): the per-warp s sums are added in warp order instead of through a shared-memory
// atomic, and CTA (x, y) stores its sums to its own slot ws[(y * gridDim.x + x) * (ns * C * 9 + ns) + ...]
// (R[o][c][tap] at o * C * 9 + c * 9 + tap, S[o] at ns * C * 9 + o) instead of adding them to r / ssum; the slots are
// added in slot order by xmm_det_finalize.
// HBM-bound: C*2 (+C*2) + 4 (+4) bytes per pixel.
struct EdgeWgradArgs {
  const float* s;     // [B][ns][H][W]
  const float* gate;  // optional clamp gate for s
  const __nv_bfloat16* v; int v_ctot, v_coff;
  const __nv_bfloat16* v2; int v2_ctot, v2_coff;  // optional second addend
  float* r;           // [ns][C][9]
  float* ssum;        // [ns] or nullptr
  int batch, ns, height, width;
  int rows;           // image rows per CTA
  float* ws;          // deterministic form: per-CTA slots (r and ssum are then not written; ssum != nullptr still
                      // selects whether S is computed)
};

constexpr int kEdgeWgradThreads = 256;

template <int C>
__global__ void __launch_bounds__(kEdgeWgradThreads) edge_wgrad_kernel(const EdgeWgradArgs a) {
  constexpr int LP = C / 8;                       // lanes per pixel
  constexpr int PPI = kEdgeWgradThreads / LP;     // pixels per CTA iteration
  extern __shared__ float sm[];
  const int W = a.width, H = a.height;
  const int pitch = W + 2;
  float* s_tile = sm;                                        // [rows + 2][W + 2]
  float* red = sm + size_t(a.rows + 2) * pitch;              // [8 warps][C * 9]
  __shared__ float ssum_s;
  __shared__ float ssum_w[kEdgeWgradThreads / 32];
  const int b = blockIdx.y;
  const int y0 = blockIdx.x * a.rows;
  const int nrows = (y0 + a.rows <= H) ? a.rows : H - y0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slot = tid / LP, cg = tid % LP;
  const size_t hw = size_t(H) * W;
  float* ws_slot = a.ws == nullptr ? nullptr
                   : a.ws + (size_t(blockIdx.y) * gridDim.x + blockIdx.x) * (size_t(a.ns) * C * 9 + a.ns);

  for (int o = 0; o < a.ns; ++o) {
    if (tid == 0) ssum_s = 0.f;
    __syncthreads();  // previous plane's readers are done with s_tile / red
    // ---- stage s rows y0-1 .. y0+rows with a zero halo; sum the owned rows
    const float* sp = a.s + (size_t(b) * a.ns + o) * hw;
    const float* gp = a.gate != nullptr ? a.gate + (size_t(b) * a.ns + o) * hw : nullptr;
    float ss = 0.f;
    for (int i = tid; i < (a.rows + 2) * pitch; i += kEdgeWgradThreads) {
      const int r = i / pitch, cx = i - r * pitch;
      const int y = y0 - 1 + r, x = cx - 1;
      float sv = 0.f;
      if (y >= 0 && y < H && x >= 0 && x < W) {
        sv = __ldg(sp + size_t(y) * W + x);
        if (gp != nullptr) {
          const float gt = __ldg(gp + size_t(y) * W + x);
          if (!(gt >= 0.0f && gt <= 1.0f)) sv = 0.0f;
        }
        if (r >= 1 && r <= nrows) ss += sv;
      }
      s_tile[i] = sv;
    }
    if (a.ssum != nullptr) {
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, d);
      if (lane == 0) {
        if (a.ws != nullptr)
          ssum_w[warp] = ss;
        else
          atomicAdd(&ssum_s, ss);
      }
    }
    __syncthreads();
    // ---- stream V
    float acc[8][9];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int t = 0; t < 9; ++t) acc[i][t] = 0.f;
    const int npx = nrows * W;
    for (int idx = slot; idx < npx; idx += PPI) {
      const int y = idx / W, x = idx - y * W;
      const size_t q = (size_t(b) * H + (y0 + y)) * W + x;
      float v[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(a.v + q * a.v_ctot + a.v_coff + cg * 8)), v);
      if (a.v2 != nullptr) {
        float w2[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(a.v2 + q * a.v2_ctot + a.v2_coff + cg * 8)), w2);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] += w2[i];
      }
      const float* st = s_tile + (y + 1) * pitch + (x + 1);
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int dy = t / 3 - 1, dx = t % 3 - 1;
        const float sv = st[-dy * pitch - dx];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i][t] = fmaf(sv, v[i], acc[i][t]);
      }
    }
    // ---- reduce: lanes of a warp with the same channel group, then the 8 warps, then one atomic per value
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        float x = acc[i][t];
#pragma unroll
        for (int d = LP; d < 32; d <<= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
        if (lane < LP) red[warp * (C * 9) + (cg * 8 + i) * 9 + t] = x;
      }
    __syncthreads();
    for (int i = tid; i < C * 9; i += kEdgeWgradThreads) {
      float x = 0.f;
#pragma unroll
      for (int w = 0; w < kEdgeWgradThreads / 32; ++w) x += red[w * (C * 9) + i];
      if (ws_slot != nullptr)
        ws_slot[size_t(o) * C * 9 + i] = x;
      else
        atomicAdd(a.r + size_t(o) * C * 9 + i, x);
    }
    if (a.ssum != nullptr && tid == 0) {
      if (ws_slot != nullptr) {
        float x = 0.f;
#pragma unroll
        for (int w = 0; w < kEdgeWgradThreads / 32; ++w) x += ssum_w[w];
        ws_slot[size_t(a.ns) * C * 9 + o] = x;
      } else {
        atomicAdd(a.ssum + o, ssum_s);
      }
    }
  }
}

}  // namespace xmm
