// Weight gradient of the 3x3 convolutions on the sm_100a tensor cores
// (what autograd's cuDNN bwd-filter computes for rrdb_blocks.py:27-31 / generator_rrdb.py:39-45,93-101).
//
//   dW[tap][c][n] = sum over pixels p of  X[p + off(tap)][c] * dY[p][n]
//
// is a GEMM whose contraction dimension K is the PIXEL index, so both operands are "MN-major"
// for the UMMA (channels are the contiguous dimension of NHWC): the A tile is the haloed
// activation patch [pixels][64*xb channels], viewed once per tap exactly like the forward
// kernel does, the B tile is the un-shifted dY patch [pixels][n channels].  One accumulator
// D_tap[c][n] per tap lives in TMEM for the whole life of the persistent CTA (split-K over
// pixel tiles), so a CTA can only own tap_count * n <= 512 columns: the launch is split into
// ROLES (e.g. one role per filter row dy) and every role streams all pixel tiles.
// At the end each CTA dumps its partial sums; wgrad_reduce_kernel adds them up per role and
// scatters into the fp32 OIHW gradient tensors.
//
// Dense-block use (F = 32): X = the 5F-channel activation buffer, dY = the 5F-channel
// gradient buffer (slot k-1 = dY_k).  Role "main(dy)": X channels 0..127 (x0..x3) against all
// 160 dY columns, 3 taps -> 480 TMEM columns; role "tail": X channels 128..159 (x4) against
// dY_5.  Blocks (x_j, dY_k) with j >= k are computed but unused.
//
// The tail is a 32 x 32 product per tap -- nine N = 32 MMAs at the ~47-cycle floor of an M = 128 instruction would
// cost more than half of the main roles' 3 x 3 N = 160 MMAs for 1/15 of the work.  Role mode 1 ("stacked") swaps the
// operands and puts the three dx taps of a filter row into ONE instruction: A = the dY box (M = output channels),
// B = a 32-channel SWIZZLE_64B patch of X whose N = 96 columns are three swizzle atoms placed ONE PIXEL (64 bytes)
// apart (LBO = 64: the atoms overlap; the UMMA address generator is linear and the swizzle is a function of the
// absolute shared-memory address, so atom j simply reads the patch shifted by j pixels).  3 MMAs instead of 9.
#pragma once
#include <cuda_bf16.h>

#include "../../include/xmm_b200.h"
#include "conv3x3_tc.cuh"

namespace xmm {

constexpr int kWgThreads = 192;
// Pixel tile of one pipeline stage: 8 rows x 8 columns (4 MMAs of K = 16 pixels per tap), which lets 4 stages fit
// (a 16-row tile is 95 KB per stage: only two).  Measured on B200 (ncu, dense block at batch 16): 1.15 ms, tensor
// pipe 59 % active, DRAM 30 %, L2 28 % with EITHER tile height -- the limiter is not the pipeline depth but the
// per-instruction cost of the MN-major tap views (A starts at arbitrary 128-byte rows of the swizzle atom).
constexpr int kWgTileH = 8;
constexpr int kWgMaxStages = 6;
constexpr int kWgBoxXBytes = 13312;   // (8+2)*10 pixels * 128 B = 12800, padded to a 1024-B multiple
constexpr int kWgBoxYBytes = 8192;    // 8*8 pixels * 128 B
constexpr int kWgBoxX8Bytes = 10240;   // roles whose taps share one filter row: 8 patch rows * 10 pixels * 128 B
constexpr int kWgBoxX32Bytes = 7168;  // mode 1: (8+2)*10 pixels * 64 B = 6400, padded to a 1024-B multiple
constexpr int kWgMaxRoles = 4;
constexpr int kWgWsFloatsPerCta = 128 * 512;

struct WgradRole {
  int cta_begin, cta_count;
  int tap_begin, tap_count;
  int x_c0;      // first X channel of the M tile (box of 64 channels; beyond-ctot channels read as 0)
  int x_boxes;   // boxes of the M operand: 1 (M rows 64..127 alias rows 0..63) or 2
  int y_c0;      // first dY channel of the N tile
  int y_boxes;   // ceil(n / 64)
  int n;         // N of the MMA (multiple of 16, <= 192)
  int rows8;     // mode 0, all taps in one filter row dy0 = tap_begin / 3: the patch box holds only the 8 rows
                 //    [ty*8 - 1 + dy0, +8) that those taps read (20 % less X traffic and shared-memory fill)
  int mode;      // 0: A = X taps, B = dY.  1: stacked -- A = dY channels [y_c0, y_c0 + 64 * x_boxes),
                 //    B = X channels [x_c0, x_c0+32) at dx = 0,1,2 (n = 96); tap_count = 3 filter rows, accumulator
                 //    column = dy * 96 + dx * 32 + (x channel - x_c0), lane = dY channel - y_c0
};

struct WgradArgs {
  WgradRole roles[kWgMaxRoles];
  int nroles;
  int batch, height, width;
  int tiles_x, tiles_y, num_tiles;
  int stages;    // pipeline depth (<= kWgMaxStages)
  float* ws;     // [gridDim.x][128 lanes][512 columns] fp32 partial sums
};

__global__ void __launch_bounds__(kWgThreads, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_y,
                const __grid_constant__ CUtensorMap tmap_x32, const __grid_constant__ CUtensorMap tmap_x8,
                const WgradArgs args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full_bar[kWgMaxStages], empty_bar[kWgMaxStages], done_bar;
  __shared__ uint32_t tmem_ptr_s;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // role lookup (uniform per CTA)
  int ri = 0;
  for (int r = 0; r < args.nroles; ++r)
    if (int(blockIdx.x) >= args.roles[r].cta_begin && int(blockIdx.x) < args.roles[r].cta_begin + args.roles[r].cta_count) ri = r;
  const WgradRole role = args.roles[ri];
  const int x_box_bytes = role.rows8 ? kWgBoxX8Bytes : kWgBoxXBytes;
  const int stage_bytes = role.mode == 1 ? role.x_boxes * kWgBoxYBytes + kWgBoxX32Bytes
                                         : role.x_boxes * x_box_bytes + role.y_boxes * kWgBoxYBytes;
  const int dy0 = role.rows8 ? role.tap_begin / 3 : 0;
  const int first_tile = int(blockIdx.x) - role.cta_begin;
  const bool has_work = first_tile < args.num_tiles;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_x);
    ptx::prefetch_tmap(&tmap_y);
    ptx::prefetch_tmap(&tmap_x32);
    ptx::prefetch_tmap(&tmap_x8);
    for (int s = 0; s < args.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    ptx::mbar_init(&done_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc<512>(&tmem_ptr_s);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = tmem_ptr_s;
  const int tiles_per_img = args.tiles_x * args.tiles_y;

  if (warp == 0) {
    if (has_work && ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = first_tile; tile < args.num_tiles; tile += role.cta_count) {
        const int b = tile / tiles_per_img;
        const int r = tile - b * tiles_per_img;
        const int ty = r / args.tiles_x;
        const int tx = r - ty * args.tiles_x;
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1u);
        uint8_t* dst = smem + size_t(stage) * stage_bytes;
        if (role.mode == 1) {
          ptx::mbar_expect_tx(&full_bar[stage],
                              uint32_t(role.x_boxes * kWgBoxYBytes + (kWgTileH + 2) * (kTileW + 2) * 64));
          for (int yb = 0; yb < role.x_boxes; ++yb)
            ptx::tma_load_4d(dst + yb * kWgBoxYBytes, &tmap_y, &full_bar[stage], role.y_c0 + 64 * yb, tx * kTileW,
                             ty * kWgTileH, b);
          ptx::tma_load_4d(dst + role.x_boxes * kWgBoxYBytes, &tmap_x32, &full_bar[stage], role.x_c0, tx * kTileW - 1,
                           ty * kWgTileH - 1, b);
          if (++stage == args.stages) {
            stage = 0;
            phase ^= 1u;
          }
          continue;
        }
        ptx::mbar_expect_tx(&full_bar[stage], uint32_t(role.x_boxes * (role.rows8 ? kWgTileH : kWgTileH + 2) * (kTileW + 2) * 128 +
                                                       role.y_boxes * kWgBoxYBytes));
        for (int xb = 0; xb < role.x_boxes; ++xb)
          ptx::tma_load_4d(dst + xb * x_box_bytes, role.rows8 ? &tmap_x8 : &tmap_x, &full_bar[stage], role.x_c0 + 64 * xb,
                           tx * kTileW - 1, ty * kWgTileH - 1 + dy0, b);
        uint8_t* ydst = dst + role.x_boxes * x_box_bytes;
        for (int yb = 0; yb < role.y_boxes; ++yb)
          ptx::tma_load_4d(ydst + yb * kWgBoxYBytes, &tmap_y, &full_bar[stage], role.y_c0 + 64 * yb, tx * kTileW,
                           ty * kWgTileH, b);
        if (++stage == args.stages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    if (has_work && ptx::elect_one()) {
      const uint32_t idesc = ptx::umma_idesc_bf16_f32(128, role.n, 1, 1);
      const uint32_t a_lbo = role.x_boxes > 1 ? uint32_t(x_box_bytes) : 0u;
      int stage = 0;
      uint32_t phase = 0;
      bool first = true;
      for (int tile = first_tile; tile < args.num_tiles; tile += role.cta_count) {
        ptx::mbar_wait(&full_bar[stage], phase);
        ptx::tc_fence_after();
        const uint32_t x_addr = ptx::smem_u32(smem + size_t(stage) * stage_bytes);
        const uint32_t y_addr = x_addr + uint32_t(role.x_boxes * x_box_bytes);
        if (role.mode == 1) {  // stage = [dY box(es)][X32 patch]
          const uint32_t p_addr = x_addr + uint32_t(role.x_boxes * kWgBoxYBytes);
          const uint32_t m_lbo = role.x_boxes > 1 ? uint32_t(kWgBoxYBytes) : 0u;
#pragma unroll 1
          for (int s = 0; s < kWgTileH / 2; ++s) {
            const uint64_t adesc =
                ptx::umma_smem_desc(x_addr + uint32_t(s * 2 * kTileW * 128), m_lbo, kTileW * 128, ptx::UMMA_SW128);
#pragma unroll 1
            for (int dy = 0; dy < 3; ++dy) {
              const uint64_t bdesc = ptx::umma_smem_desc(p_addr + uint32_t((2 * s + dy) * (kTileW + 2) * 64), 64,
                                                         (kTileW + 2) * 64, ptx::UMMA_SW64);
              ptx::umma_ss(tmem_base + uint32_t(dy * role.n), adesc, bdesc, idesc, (first && s == 0) ? 0u : 1u);
            }
          }
        } else {
#pragma unroll 1
          for (int s = 0; s < kWgTileH / 2; ++s) {  // 16 pixels (two tile rows) per MMA
            const uint64_t bdesc = ptx::umma_smem_desc(y_addr + uint32_t(s * 2 * kTileW * 128), kWgBoxYBytes,
                                                       kTileW * 128, ptx::UMMA_SW128);
#pragma unroll 1
            for (int t = 0; t < role.tap_count; ++t) {
              const int tap = role.tap_begin + t;
              const int dy = tap / 3, dx = tap - dy * 3;
              const uint32_t a_addr = x_addr + uint32_t(((2 * s + dy - dy0) * (kTileW + 2) + dx) * 128);
              const uint64_t adesc = ptx::umma_smem_desc(a_addr, a_lbo, (kTileW + 2) * 128, ptx::UMMA_SW128);
              ptx::umma_ss(tmem_base + uint32_t(t * role.n), adesc, bdesc, idesc, (first && s == 0) ? 0u : 1u);
            }
          }
        }
        first = false;
        ptx::umma_commit(&empty_bar[stage]);
        if (++stage == args.stages) {
          stage = 0;
          phase ^= 1u;
        }
      }
      ptx::umma_commit(&done_bar);
    }
  } else if (has_work) {
    // epilogue: dump this CTA's accumulators  ws[cta][lane][col]
    const int q = warp & 3;
    ptx::mbar_wait(&done_bar, 0);
    ptx::tc_fence_after();
    const int cols = role.tap_count * role.n;
    float* dst = args.ws + size_t(blockIdx.x) * kWgWsFloatsPerCta + size_t(q * 32 + lane) * 512;
    for (int c0 = 0; c0 < cols; c0 += 32) {
      uint32_t r[32];
      ptx::tmem_ld_32x32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(c0), r);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; i += 4)
        *reinterpret_cast<uint4*>(dst + c0 + i) = make_uint4(r[i], r[i + 1], r[i + 2], r[i + 3]);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

// One destination tensor of the reduction: dW (fp32 OIHW [o_count][i_total][3][3]) gathers
//   dW[o][i][tap] (+)= scale * sum over the role's CTAs of ws[cta][lane = i - x_c0][(tap - tap_begin) * n + y_col0 + o]
// for i in [i_begin, i_end), from the role that owns (tap, i).  For a stacked role (mode 1) lanes are output channels:
//   ws[cta][lane0 + o][(tap / 3) * 96 + (tap % 3) * 32 + col0 + (i - i_begin)],  all 9 taps.
struct WgradDst {
  float* dw;
  int o_count, i_total;
  int i_begin, i_end;   // input channels taken from this role
  int role;             // index into WgradArgs::roles (for taps in that role's range)
  int lane0;            // ws lane of input channel i_begin
  int col0;             // column (within one tap's n columns) of output channel 0
  float scale;
  int accumulate;       // 0: overwrite, 1: add to the existing gradient
  int perm;             // 1: output channel o is the PixelShuffle-packed index (see shuffle_perm)
  int o_begin, o_total; // this destination covers output channels [o_begin, o_begin + o_count) of o_total
};

struct WgradReduceArgs {
  WgradRole roles[kWgMaxRoles];
  int nroles;
  const float* ws;
  int ndst;
  WgradDst dst[16];
};

__global__ void wgrad_reduce_kernel(const WgradReduceArgs a, int num_tiles) {
  const WgradDst d = a.dst[blockIdx.y];
  const WgradRole role = a.roles[d.role];
  const int ni = d.i_end - d.i_begin;
  const int ntap = role.mode == 1 ? 9 : role.tap_count;
  const int total = d.o_count * ni * ntap;
  int active = role.cta_count < num_tiles ? role.cta_count : num_tiles;  // CTAs beyond num_tiles wrote nothing
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int o = e % d.o_count;
    const int rest = e / d.o_count;
    const int i = rest % ni;
    const int t = rest / ni;
    const size_t off = role.mode == 1 ? size_t(d.lane0 + o) * 512 + size_t((t / 3) * role.n + (t % 3) * 32 + d.col0 + i)
                                      : size_t(d.lane0 + i) * 512 + size_t(t * role.n + d.col0 + o);
    float s = 0.f;
    for (int c = 0; c < active; ++c) s += a.ws[size_t(role.cta_begin + c) * kWgWsFloatsPerCta + off];
    const int oo = d.perm ? shuffle_perm(d.o_begin + o, d.o_total / 4) : d.o_begin + o;
    float* p = d.dw + (size_t(oo) * d.i_total + (d.i_begin + i)) * 9 + (role.mode == 1 ? t : role.tap_begin + t);
    *p = d.accumulate ? (*p + d.scale * s) : d.scale * s;
  }
}

// Column sums of bf16 NHWC channel windows: bias gradients  db[n] = scale * sum_p dY[p][c0 + n], for up to
// kColsumMaxSeg windows of one buffer in ONE pass (a dense block's five bias gradients are five windows of its
// gradient buffer).  Thread -> (pixel lane, 8-channel group); 4 independent 16-byte loads in flight per thread.
constexpr int kColsumMaxSeg = 8;
constexpr int kColsumThreads = 256;
struct ColsumSeg {
  int c0, n, group0;
  float scale;
  float* out;
};
struct ColsumArgs {
  const __nv_bfloat16* in;
  int ctot, nseg, ngroups;
  size_t npix;
  ColsumSeg seg[kColsumMaxSeg];
  float* ws;  // deterministic form: CTA b stores its unscaled sums to ws[b * ngroups * 8 + channel] (no atomics, outs unused)
};

__global__ void __launch_bounds__(kColsumThreads) colsum_multi_kernel(const ColsumArgs a) {
  __shared__ float red[kColsumThreads * 8];
  const int ppb = kColsumThreads / a.ngroups;  // pixel lanes per block
  const int g = threadIdx.x % a.ngroups, pl = threadIdx.x / a.ngroups;
  int si = 0;
#pragma unroll
  for (int i = 1; i < kColsumMaxSeg; ++i)
    if (i < a.nseg && g >= a.seg[i].group0) si = i;
  const int ch = a.seg[si].c0 + (g - a.seg[si].group0) * 8;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (pl < ppb) {
    const size_t stride = size_t(gridDim.x) * ppb;
    size_t p = size_t(blockIdx.x) * ppb + pl;
    const __nv_bfloat16* base = a.in + ch;
    for (; p + 3 * stride < a.npix; p += 4 * stride) {
      uint4 q[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) q[u] = __ldg(reinterpret_cast<const uint4*>(base + (p + u * stride) * a.ctot));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float v[8];
        unpack8(q[u], v);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] += v[i];
      }
    }
    for (; p < a.npix; p += stride) {
      float v[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(base + p * a.ctot)), v);
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] += v[i];
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) red[threadIdx.x * 8 + i] = (pl < ppb) ? acc[i] : 0.f;
  __syncthreads();
  // thread t < ngroups * 8: channel t of the concatenated windows; sum over the pixel lanes
  for (int t = threadIdx.x; t < a.ngroups * 8; t += kColsumThreads) {
    const int gg = t / 8, i = t % 8;
    float x = 0.f;
    for (int l = 0; l < ppb; ++l) x += red[(l * a.ngroups + gg) * 8 + i];
    if (a.ws != nullptr) {
      a.ws[size_t(blockIdx.x) * (a.ngroups * 8) + t] = x;
      continue;
    }
    int sj = 0;
#pragma unroll
    for (int k = 1; k < kColsumMaxSeg; ++k)
      if (k < a.nseg && gg >= a.seg[k].group0) sj = k;
    atomicAdd(a.seg[sj].out + (gg - a.seg[sj].group0) * 8 + i, a.seg[sj].scale * x);
  }
}

// Deterministic reductions (xmm_det_finalize): job blockIdx.y, element i of it:
//   dst[i] = (accumulate ? dst[i] : 0) + scale * sum_{k = 0, 1, .., count-1} slots[k * stride + i]
// with k in increasing order, so the bits depend only on the slot contents.  Each slot is cleared after it is read: a
// producer that leaves some of its slots unwritten (a smaller grid, a warp without some of the columns) adds exact
// zeros the next time, and needs no clearing launch of its own.  One thread per element; eight independent loads in
// flight per thread (a conv3x3 job reads ~1200 slots).
constexpr int kDetFinalizeThreads = 128;
__global__ void __launch_bounds__(kDetFinalizeThreads) det_finalize_kernel(const xmm_det_job* __restrict__ jobs,
                                                                          float* __restrict__ dst_base) {
  const xmm_det_job& j = jobs[blockIdx.y];
  for (int i = blockIdx.x * kDetFinalizeThreads + threadIdx.x; i < j.n; i += gridDim.x * kDetFinalizeThreads) {
    float* p = j.slots + i;
    const size_t st = size_t(j.stride);
    float s = 0.f;
    int k = 0;
    for (; k + 8 <= j.count; k += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = p[(k + u) * st];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        s += v[u];
        p[(k + u) * st] = 0.f;
      }
    }
    for (; k < j.count; ++k) {
      s += p[k * st];
      p[k * st] = 0.f;
    }
    float* d = dst_base + j.dst + i;
    *d = (j.accumulate ? *d : 0.f) + j.scale * s;
  }
}

}  // namespace xmm
