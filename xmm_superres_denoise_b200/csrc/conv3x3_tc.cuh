// 3x3 / stride 1 / pad 1 convolution as an implicit GEMM on the sm_100a tensor cores.
//
// Replaces the nn.Conv2d calls of the reference's dense blocks
// (xmm_superres_denoise/models/modules/rrdb_blocks.py:27-31,49-52 and
// generator_rrdb.py:39-45,93-101) *and* the torch.cat that feeds them: the input is a
// channel window [coff, coff+cin) of one NHWC bf16 buffer, the output a channel window of
// another (or the same) buffer, so the dense connection is pointer arithmetic.
//
// GEMM mapping (per CTA tile): M = 128 output pixels (16 rows x 8 cols), N = Cout,
// K = 9 taps x Cin.  One TMA box per K-chunk brings the (16+2)x(8+2) haloed pixel patch
// x KC channels into shared memory once; the 9 taps are 9 *views* of that patch (UMMA
// descriptor start address + stride), so activations cross L2->SMEM 1.4x, not 9x.
// Weights for the whole layer stay resident in shared memory for the life of the
// persistent CTA.  Accumulators live in TMEM (double buffered) and the epilogue warps
// apply bias / LeakyReLU / mask / scaled residuals and store bf16 while the next tile's
// MMAs run.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM owner),
// warps 2..5 = epilogue (TMEM lane quarter = warp_id % 4).
#pragma once
#include <cuda_bf16.h>

#include "ptx_sm100.cuh"

#ifdef XMM_CONV_PROFILE
#define XMM_PROF_T0() prof_t0_ = clock64()
#define XMM_PROF_ADD(i) prof_acc_[i] += clock64() - prof_t0_
#define XMM_PROF_START(i) long long prof_s_ = clock64()
#define XMM_PROF_STOP(i) prof_acc_[i] += clock64() - prof_s_
#define XMM_PROF_FLUSH(i) args.prof[size_t(blockIdx.x) * 8 + (i)] = prof_acc_[i]
// finer phases inside the column-scatter epilogue (one warp reports): slots [148*8 + cta*8 + i]
#define XMM_EPI_T0() long long epi_t_ = clock64()
#define XMM_EPI_ADD(w, i) { const long long n_ = clock64(); (w).phase[i] += n_ - epi_t_; epi_t_ = n_; }
#else
#define XMM_EPI_T0()
#define XMM_EPI_ADD(w, i)
#define XMM_PROF_T0()
#define XMM_PROF_ADD(i)
#define XMM_PROF_START(i)
#define XMM_PROF_STOP(i)
#define XMM_PROF_FLUSH(i)
#endif

namespace xmm {

constexpr int kTileH = 16;
constexpr int kTileW = 8;
constexpr int kHaloH = kTileH + 2;
constexpr int kMaxStages = 8;  // activation stages (16 measured no faster: the TMA feed is not bytes-in-flight bound)
constexpr int kConvThreads = 192;

// How the 9 tap views are formed from shared memory (probe-selectable; see DESIGN.md):
//   kTapHalo : one haloed [18][10] patch; tap = start-address offset, SBO = 10 rows.
//   kTapHaloBaseOff : same, plus the descriptor's base_offset field = (start>>7)&7.
//   kTapDx3  : three dx-shifted dense [18][8] patches; tap dy = 8-row aligned offset.
enum TapMode : int { kTapHalo = 0, kTapHaloBaseOff = 1, kTapDx3 = 2 };

struct ConvEpilogue {
  // v = acc + bias[n];  v = v > 0 ? v : lrelu_slope * v;
  // v *= (mask[p][n] > 0 ? 1 : mask_slope)            (mask == nullptr: skipped)
  // out[p][n] = s0 * v + s1 * r1[p][n] + s2 * r2[p][n] (r == nullptr: term skipped)
  float lrelu_slope;
  float mask_slope;
  float s0, s1, s2;
  const __nv_bfloat16* mask;
  int mask_ctot, mask_coff;
  const __nv_bfloat16* r1;
  int r1_ctot, r1_coff;
  const __nv_bfloat16* r2;
  int r2_ctot, r2_coff;
  __nv_bfloat16* out;
  int out_ctot, out_coff;
  // 0: out is [B][H][W][out_ctot]
  // 1: PixelShuffle(2) store: out is [B][2H][2W][out_ctot]; column group g=(i,j) -> pixel (2y+i,2x+j)
  // 2: inverse (backward of 1): out is [B][H/2][W/2][out_ctot]; pixel (y,x) -> (y/2,x/2), channel block g=(y&1,x&1)
  int pixel_shuffle;
  int shuffle_stride;  // mode 2: channel distance between the four (y&1, x&1) blocks (the full layer's cout)
  // Image mode (conv_last, generator_rrdb.py:48-54,107-108,132-135, on the tensor cores): img_out != nullptr.
  // The packed layer holds bf16(w) in rows [0, img_cout) and the low-order halves bf16(w - bf16(w)) in rows
  // [16, 16 + img_cout); out[b][o][y][x] = clamp?(acc[o] + acc[16+o] + bias[o] + img_res[...]) in fp32 NCHW.
  // Optional fused bias gradient: colsum[n] += colsum_scale * sum over the launch's pixels of the value written to
  // channel n (the data gradient dY a layer produces is also the bias gradient's integrand).  Cout = 32 kernels.
  float* colsum;
  float colsum_scale;
  // Deterministic form of the same sums (colsum_ws != nullptr): every epilogue warp stores its unscaled column sums to
  // its own slot, colsum_ws[(blockIdx.x * kCsumWarpSlots + warp - 2) * 32 + n], instead of adding them to colsum; a
  // later xmm_det_finalize adds the slots in slot order.  The result depends only on which tiles each warp summed, so
  // every kernel that flushes here hands its tiles to CTAs by a static schedule (a function of blockIdx.x and
  // gridDim.x: conv3x3_tc, conv3x3_dx's DxRuns, conv3x3_row's RowSched, conv3x3_chain's item0 / item_step).
  float* colsum_ws;
  float* img_out;
  const float* img_res;
  float* img_pre;   // optional copy of the un-clamped value (backward clamp gate)
  int img_cout, img_clamp;
};

struct ConvArgs {
  const void* wblob;  // packed weights image + bias (see pack_weights.cuh)
  uint32_t w_bytes;   // bytes of the weight image (multiple of 1024)
  int nchunks;        // Cin / KC
  int cin_off;        // first input channel inside the input buffer
  int batch, height, width;
  int tiles_x, tiles_y, num_tiles;
  int stages;
  int strip_rr;  // conv3x3_dx: 1 = whole strips dealt round-robin to the CTAs, 0 = equal contiguous tile ranges
  int tma_store; // conv3x3_tc: 1 = epilogue warps stage their [4 rows][8 px] x NT result and TMA-store it
  int side_mask; // conv3x3_dx: bit k set = side input k (0 mask, 1 r1, 2 r2) is staged through shared memory by TMA
  ConvEpilogue epi;
#ifdef XMM_CONV_PROFILE
  long long* prof;  // [gridDim.x][8] cycle counters (tools/probe.cu only)
#endif
};

// EG = epilogue groups (1 or 2): groups of four epilogue warps take alternate tiles of the CTA's sequence (the tiles
// are independent here: haloed patches, no carries), with 2 * EG accumulator stages in TMEM.
template <int KC, int NT, int MODE, int EG = 1>
struct ConvCfg {
  static_assert(EG == 1 || EG == 2, "one or two epilogue groups");
  static constexpr int kThreads = 64 + 128 * EG;
  static constexpr int kAccStages = 2 * EG;
  static_assert(KC == 32 || KC == 64, "K chunk is 32 (SWIZZLE_64B) or 64 (SWIZZLE_128B) channels");
  static_assert(NT % 32 == 0 && NT >= 32 && NT <= 256, "Cout tile");
  static constexpr int kRowB = KC * 2;  // bytes of one pixel's K-chunk in shared memory
  static constexpr uint32_t kLayout = (KC == 64) ? ptx::UMMA_SW128 : ptx::UMMA_SW64;
  static constexpr int kPitchPx = (MODE == kTapDx3) ? kTileW : kTileW + 2;
  static constexpr int kSubBytes = kHaloH * kPitchPx * kRowB;
  static constexpr int kSubStride = (kSubBytes + 1023) / 1024 * 1024;
  static constexpr int kNumSub = (MODE == kTapDx3) ? 3 : 1;
  static constexpr int kStageBytes = kNumSub * kSubStride;
  static constexpr int kStageTx = kNumSub * kSubBytes;
  static constexpr int kKSteps = KC / 16;
  static constexpr int kTapBytes = NT * kRowB;  // one (chunk, tap) weight block
  static_assert(2 * EG * NT <= 512, "accumulator stages exceed the 512 TMEM columns");
  static constexpr int kTmemCols = (2 * EG * NT <= 32) ? 32 : (2 * EG * NT <= 64) ? 64 : (2 * EG * NT <= 128) ? 128
                                   : (2 * EG * NT <= 256) ? 256 : 512;
  static constexpr uint32_t kIdesc = ptx::umma_idesc_bf16_f32(128, NT, 0, 0);
  static constexpr int kBiasBytes = NT * 4;
  // barriers: full[8] empty[8] tmem_full[4] tmem_empty[4] wbar + tmem ptr
  static constexpr int kBarBytes = (2 * kMaxStages + 9) * 8 + 16;
  // per-warp output staging for the TMA store ([4 rows][8 px] x NT bf16, swizzled; 4 warps, double buffered)
  static constexpr int kWarpOutBytes = (NT <= 64) ? 32 * NT * 2 : 0;
  static constexpr int kOutBytes = 4 * EG * 2 * kWarpOutBytes;
  // with_out: the per-warp staging tiles of the TMA-store path (ConvArgs::tma_store) are part of the layout
  static size_t smem_bytes(uint32_t w_bytes, int stages, bool with_out = true) {
    return 1024 /*align slack*/ + w_bytes + kBiasBytes + 1024 + size_t(stages) * kStageBytes + (with_out ? kOutBytes : 0) +
           kBarBytes;
  }
};

__host__ __device__ __forceinline__ int shuffle_perm(int idx, int group) {
  // packed index g*group + c  ->  PixelShuffle channel 4*c + g   (g = 2*i + j)
  const int g = idx / group, c = idx - g * group;
  return 4 * c + g;
}

__device__ __forceinline__ void unpack8(const uint4& q, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  uint4 q;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&q);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return q;
}

// Fused epilogue arithmetic for NC accumulator columns [col0, col0+NC) of one pixel, in place on v (raw fp32 sums):
// bias (bias_s == nullptr: already added), LeakyReLU, LeakyReLU' mask, scale, residuals.
// Side inputs (mask, r1, r2) are read from global memory, or -- when `staged` is given -- from shared-memory copies
// a TMA load placed there: staged[k] points at this lane's NC channels of side input k (nullptr: not staged), with
// consecutive 16-byte chunks at staged_xor-swizzled positions (see conv3x3_dx.cuh).
struct StagedSides {
  const uint8_t* base[3];  // tile base per side input (mask, r1, r2) or nullptr
  uint32_t row_off;        // byte offset of this lane's pixel row inside the tile
  uint32_t chunk0;         // first 16-byte chunk index of this lane's channels
  uint32_t xor_mask;       // swizzle: chunk ^= xor_mask
};
__device__ __forceinline__ uint4 staged_chunk(const StagedSides& s, int k, int q) {
  return *reinterpret_cast<const uint4*>(s.base[k] + s.row_off + (((s.chunk0 + uint32_t(q)) ^ s.xor_mask) << 4));
}

template <int NT, int NC>
__device__ __forceinline__ void conv_epilogue_math(const ConvEpilogue& e, const float* __restrict__ bias_s,
                                                   float (&v)[NC], int col0, int b, int y, int x, int H, int W,
                                                   const StagedSides* staged = nullptr) {
  static_assert(NC % 8 == 0, "whole 16-byte accesses");
#pragma unroll
  for (int i = 0; i < NC; ++i) {
    const float t = bias_s != nullptr ? v[i] + bias_s[col0 + i] : v[i];
    v[i] = t > 0.f ? t : t * e.lrelu_slope;
  }
  const size_t pix = (size_t(b) * H + y) * W + x;
  if (e.mask != nullptr) {
    const uint4* mp = reinterpret_cast<const uint4*>(e.mask + pix * e.mask_ctot + e.mask_coff + col0);
#pragma unroll
    for (int q = 0; q < NC / 8; ++q) {
      float m[8];
      unpack8((staged != nullptr && staged->base[0] != nullptr) ? staged_chunk(*staged, 0, q) : __ldg(mp + q), m);
#pragma unroll
      for (int i = 0; i < 8; ++i) v[q * 8 + i] *= (m[i] > 0.f ? 1.f : e.mask_slope);
    }
  }
  if (e.s0 != 1.f) {
#pragma unroll
    for (int i = 0; i < NC; ++i) v[i] *= e.s0;
  }
  if (e.r1 != nullptr) {
    const uint4* rp = reinterpret_cast<const uint4*>(e.r1 + pix * e.r1_ctot + e.r1_coff + col0);
#pragma unroll
    for (int q = 0; q < NC / 8; ++q) {
      float m[8];
      unpack8((staged != nullptr && staged->base[1] != nullptr) ? staged_chunk(*staged, 1, q) : __ldg(rp + q), m);
#pragma unroll
      for (int i = 0; i < 8; ++i) v[q * 8 + i] = fmaf(e.s1, m[i], v[q * 8 + i]);
    }
  }
  if (e.r2 != nullptr) {
    const uint4* rp = reinterpret_cast<const uint4*>(e.r2 + pix * e.r2_ctot + e.r2_coff + col0);
#pragma unroll
    for (int q = 0; q < NC / 8; ++q) {
      float m[8];
      unpack8((staged != nullptr && staged->base[2] != nullptr) ? staged_chunk(*staged, 2, q) : __ldg(rp + q), m);
#pragma unroll
      for (int i = 0; i < 8; ++i) v[q * 8 + i] = fmaf(e.s2, m[i], v[q * 8 + i]);
    }
  }
}

// Epilogue for NC accumulator columns [col0, col0+NC) of one pixel: arithmetic + direct bf16 store.
template <int NT, int NC>
__device__ __forceinline__ void conv_epilogue_cols(const ConvEpilogue& e, const float* __restrict__ bias_s,
                                                   float (&v)[NC], int col0, int b, int y, int x, int H, int W,
                                                   float* csum = nullptr) {
  conv_epilogue_math<NT, NC>(e, bias_s, v, col0, b, y, x, H, W);
  if (csum != nullptr) {
#pragma unroll
    for (int i = 0; i < NC; ++i) csum[i] += v[i];
  }
  const size_t pix = (size_t(b) * H + y) * W + x;
  uint4* op;
  if (e.pixel_shuffle == 2) {
    const int g = ((y & 1) << 1) | (x & 1);
    const size_t lp = (size_t(b) * (H >> 1) + (y >> 1)) * (W >> 1) + (x >> 1);
    op = reinterpret_cast<uint4*>(e.out + lp * e.out_ctot + e.out_coff + g * e.shuffle_stride + col0);
  } else if (e.pixel_shuffle == 1) {
    constexpr int kGroup = NT / 4;  // channels of the shuffled (HR) tensor
    const int g = col0 / kGroup, c = col0 % kGroup;
    const size_t hp = (size_t(b) * (2 * H) + (2 * y + (g >> 1))) * (2 * W) + (2 * x + (g & 1));
    op = reinterpret_cast<uint4*>(e.out + hp * e.out_ctot + e.out_coff + c);
  } else {
    op = reinterpret_cast<uint4*>(e.out + pix * e.out_ctot + e.out_coff + col0);
  }
#ifdef XMM_EXP_NOSTORE
  if (v[0] == 123.456f)
#endif
#pragma unroll
  for (int q = 0; q < NC / 8; ++q) op[q] = pack8(v + q * 8);
}

// 32 raw accumulator registers (tcgen05.ld bit pattern) -> epilogue.
template <int NT>
__device__ __forceinline__ void conv_epilogue_32(const ConvEpilogue& e, const float* __restrict__ bias_s,
                                                 uint32_t (&acc)[32], int col0, int b, int y, int x,
                                                 int H, int W, float* csum = nullptr) {
  float v[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(acc[i]);
  conv_epilogue_cols<NT, 32>(e, bias_s, v, col0, b, y, x, H, W, csum);
}

// Deterministic column sums: slots per CTA, one per epilogue warp.  The epilogue warps of every kernel that calls
// colsum_flush are warps 2 .. 2 + kCsumWarpSlots - 1; a warp that owns only some columns leaves the rest of its slot
// as it found it (zero: xmm_det_finalize clears the slots it reads).
constexpr int kCsumWarpSlots = 8;

// End of a warp's life: add its lanes' column sums and publish them (one atomic per column and warp, or one store to
// the warp's slot in the deterministic form).
template <int NC>
__device__ __forceinline__ void colsum_flush(const ConvEpilogue& e, float (&csum)[NC], int col0, int lane) {
  static_assert(NC <= 32, "fused column sums are for cout = 32");
  float* slot = e.colsum_ws == nullptr ? nullptr
                : e.colsum_ws + (size_t(blockIdx.x) * kCsumWarpSlots + ((threadIdx.x >> 5) - 2)) * 32 + col0;
#pragma unroll
  for (int i = 0; i < NC; ++i) {
    float x = csum[i];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
    if (lane == 0) {
      if (slot != nullptr)
        slot[i] = x;
      else
        atomicAdd(e.colsum + col0 + i, e.colsum_scale * x);
    }
  }
}

template <int KC, int NT, int MODE, int EG = 1>
__global__ void __launch_bounds__(64 + 128 * EG, 1)
conv3x3_tc_kernel(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_out,
                  const ConvArgs args) {
  using Cfg = ConvCfg<KC, NT, MODE, EG>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w_s = smem;                                                   // weights image
  float* bias_s = reinterpret_cast<float*>(smem + args.w_bytes);         // NT floats (same bulk copy)
  uint8_t* stage_s = smem + ((args.w_bytes + Cfg::kBiasBytes + 1023) & ~1023u);
  uint8_t* out_s = stage_s + size_t(args.stages) * Cfg::kStageBytes;  // 1 KB aligned (stage sizes are)
  uint64_t* bars = reinterpret_cast<uint64_t*>(out_s + (args.tma_store != 0 ? Cfg::kOutBytes : 0));
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kMaxStages;
  uint64_t* tfull_bar = bars + 2 * kMaxStages;
  uint64_t* tempty_bar = tfull_bar + 4;
  uint64_t* w_bar = tempty_bar + 4;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(w_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
#ifdef XMM_CONV_PROFILE
  long long prof_t0_ = 0;
  long long prof_acc_[6] = {0, 0, 0, 0, 0, 0};
  const long long prof_k0_ = clock64();
  unsigned long long prof_g0_;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(prof_g0_));
#endif

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_in);
    for (int s = 0; s < args.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < Cfg::kAccStages; ++a) {
      ptx::mbar_init(&tfull_bar[a], 1);
      ptx::mbar_init(&tempty_bar[a], 4);
    }
    ptx::mbar_init(w_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc<Cfg::kTmemCols>(tmem_ptr_s);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;

  const int tiles_per_img = args.tiles_x * args.tiles_y;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (ptx::elect_one()) {
      const uint32_t wtot = args.w_bytes + Cfg::kBiasBytes;
      ptx::mbar_expect_tx(w_bar, wtot);
      const uint8_t* gsrc = static_cast<const uint8_t*>(args.wblob);
      for (uint32_t off = 0; off < wtot; off += 32768u) {
        const uint32_t n = (wtot - off < 32768u) ? (wtot - off) : 32768u;
        ptx::bulk_load(w_s + off, gsrc + off, n, w_bar);
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < args.num_tiles; tile += gridDim.x) {
        const int b = tile / tiles_per_img;
        const int r = tile - b * tiles_per_img;
        const int ty = r / args.tiles_x;
        const int tx = r - ty * args.tiles_x;
        const int y0 = ty * kTileH - 1, x0 = tx * kTileW - 1;
        for (int ch = 0; ch < args.nchunks; ++ch) {
          XMM_PROF_T0();
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1u);
          XMM_PROF_ADD(0);
          ptx::mbar_expect_tx(&full_bar[stage], Cfg::kStageTx);
          uint8_t* dst = stage_s + size_t(stage) * Cfg::kStageBytes;
          const int c0 = args.cin_off + ch * KC;
#pragma unroll
          for (int sub = 0; sub < Cfg::kNumSub; ++sub)
            ptx::tma_load_4d(dst + sub * Cfg::kSubStride, &tmap_in, &full_bar[stage], c0, x0 + sub, y0, b);
          if (++stage == args.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
      XMM_PROF_FLUSH(0);
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (ptx::elect_one()) {
      ptx::mbar_wait(w_bar, 0);
      ptx::tc_fence_after();
      const uint32_t w_addr = ptx::smem_u32(w_s);
      const uint32_t st_addr = ptx::smem_u32(stage_s);
      const uint64_t bdesc0 = ptx::umma_smem_desc(w_addr, 16, 8 * Cfg::kRowB, Cfg::kLayout);
      const uint64_t adesc0 = ptx::umma_smem_desc(0, 16, Cfg::kPitchPx * Cfg::kRowB, Cfg::kLayout);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      XMM_PROF_START(3);
      for (int tile = blockIdx.x; tile < args.num_tiles; tile += gridDim.x) {
        XMM_PROF_T0();
        ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
        XMM_PROF_ADD(1);
        ptx::tc_fence_after();
        const uint32_t d_addr = tmem_base + uint32_t(acc * NT);
        for (int ch = 0; ch < args.nchunks; ++ch) {
          XMM_PROF_T0();
          ptx::mbar_wait(&full_bar[stage], phase);
          XMM_PROF_ADD(2);
          ptx::tc_fence_after();
          const uint32_t a_stage = st_addr + uint32_t(stage) * Cfg::kStageBytes;
          const uint64_t bdesc_ch = bdesc0 + uint64_t((uint32_t(ch) * 9u * Cfg::kTapBytes) >> 4);
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            const int dy = tap / 3, dx = tap % 3;
            uint32_t a_off;
            if (MODE == kTapDx3)
              a_off = uint32_t(dx * Cfg::kSubStride + dy * kTileW * Cfg::kRowB);
            else
              a_off = uint32_t((dy * Cfg::kPitchPx + dx) * Cfg::kRowB);
#pragma unroll
            for (int ks = 0; ks < Cfg::kKSteps; ++ks) {
              const uint32_t a_addr = a_stage + a_off + uint32_t(ks * 32);
              uint64_t adesc = adesc0 | uint64_t((a_addr & 0x3FFFFu) >> 4);
              if (MODE == kTapHaloBaseOff) adesc |= uint64_t((a_addr >> 7) & 7u) << 49;
              const uint64_t bdesc = bdesc_ch + uint64_t((uint32_t(tap) * Cfg::kTapBytes + uint32_t(ks * 32)) >> 4);
              ptx::umma_ss(d_addr, adesc, bdesc, Cfg::kIdesc, (ch | tap | ks) != 0 ? 1u : 0u);
            }
          }
          ptx::umma_commit(&empty_bar[stage]);
          if (++stage == args.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        ptx::umma_commit(&tfull_bar[acc]);
        if (++acc == Cfg::kAccStages) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
      XMM_PROF_STOP(3);
      XMM_PROF_FLUSH(1); XMM_PROF_FLUSH(2); XMM_PROF_FLUSH(3);
    }
  } else {
    // ------------------------------------------------------------ epilogue
    const int q = warp & 3;  // TMEM lane quarter this warp may read
    const int m = q * 32 + lane;
    const int py = m >> 3, px = m & 7;
    ptx::mbar_wait(w_bar, 0);  // bias rides with the weights
    // TMA-store path: this warp's [4 rows][8 px] x NT result goes through its own swizzled staging tile (rows of
    // NT*2 = 64 B: SWIZZLE_64B, 128 B: SWIZZLE_128B) -- per-lane 16-byte global stores at a 64..640-byte pitch cost
    // ~512 L1 transactions per tile on the datapath the MMA operand reads share.
    const bool use_tma = Cfg::kOutBytes > 0 && args.tma_store != 0;
    uint8_t* my_out = out_s + (warp - 2) * 2 * Cfg::kWarpOutBytes;
    const uint32_t sw_xor = NT == 32 ? uint32_t((lane >> 1) & 3) : uint32_t(lane & 7);
    int obuf = 0;
    const int group = (warp - 2) >> 2;  // which tiles of the sequence this warp's group takes
    int seq = 0;                        // position in this CTA's tile sequence
    const bool do_csum = NT == 32 && args.epi.colsum != nullptr;
    float csum[NT == 32 ? 32 : 1];
#pragma unroll
    for (int i = 0; i < (NT == 32 ? 32 : 1); ++i) csum[i] = 0.f;
    for (int tile = blockIdx.x; tile < args.num_tiles; tile += gridDim.x, ++seq) {
      if (EG > 1 && (seq & (EG - 1)) != group) continue;
      const int acc = seq & (Cfg::kAccStages - 1);
      const uint32_t acc_phase = uint32_t(seq / Cfg::kAccStages) & 1u;
      const int b = tile / tiles_per_img;
      const int r = tile - b * tiles_per_img;
      const int ty = r / args.tiles_x;
      const int tx = r - ty * args.tiles_x;
      const int y = ty * kTileH + py, x = tx * kTileW + px;
      const bool valid = (y < args.height) && (x < args.width);
      XMM_PROF_T0();
      ptx::mbar_wait(&tfull_bar[acc], acc_phase);
      XMM_PROF_ADD(4);
      XMM_PROF_T0();
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(acc * NT);
      uint8_t* stage = my_out + obuf * Cfg::kWarpOutBytes;
      if (use_tma) {  // the store issued two tiles ago has finished reading this staging tile
        if (ptx::elect_one()) ptx::bulk_wait_read<1>();
        __syncwarp();
      }
#pragma unroll 1
      for (int cc = 0; cc < NT / 32; ++cc) {
        uint32_t accr[32];
        ptx::tmem_ld_32x32(t_addr + uint32_t(cc * 32), accr);
        ptx::tmem_ld_wait();
        if (cc == NT / 32 - 1) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tempty_bar[acc]);
        }
#ifdef XMM_EXP_NOEPI
        if (__uint_as_float(accr[0]) == 123.456f)
#endif
        if (valid) {
          if (NT == 32 && args.epi.img_out != nullptr) {
            const size_t hw = size_t(args.height) * args.width;
            const size_t o0 = size_t(b) * args.epi.img_cout * hw + size_t(y) * args.width + x;
#pragma unroll
            for (int o = 0; o < 4; ++o) {
              if (o < args.epi.img_cout) {
                float v = __uint_as_float(accr[o]) + __uint_as_float(accr[16 + o]) + bias_s[o];
                if (args.epi.img_res != nullptr) v += args.epi.img_res[o0 + o * hw];
                if (args.epi.img_pre != nullptr) args.epi.img_pre[o0 + o * hw] = v;
                args.epi.img_out[o0 + o * hw] = args.epi.img_clamp ? fminf(fmaxf(v, 0.0f), 1.0f) : v;
              }
            }
          } else if (use_tma) {
            float v[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(accr[i]);
            conv_epilogue_math<NT, 32>(args.epi, bias_s, v, cc * 32, b, y, x, args.height, args.width);
            if (NT == 32 && do_csum) {
#pragma unroll
              for (int i = 0; i < 32; ++i) csum[NT == 32 ? i : 0] += v[i];
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
              *reinterpret_cast<uint4*>(stage + lane * (NT * 2) + (((uint32_t(cc * 4 + j)) ^ sw_xor) << 4)) = pack8(v + j * 8);
          } else {
            if (NT == 32) {
              float (&cs32)[32] = reinterpret_cast<float (&)[32]>(csum);
              conv_epilogue_32<NT>(args.epi, bias_s, accr, cc * 32, b, y, x, args.height, args.width,
                                   do_csum ? &cs32[0] : nullptr);
            } else {
              conv_epilogue_32<NT>(args.epi, bias_s, accr, cc * 32, b, y, x, args.height, args.width);
            }
          }
        }
      }
      if (use_tma) {
        ptx::fence_proxy_async();
        __syncwarp();
        if (ptx::elect_one()) {
          ptx::tma_store_4d(&tmap_out, stage, args.epi.out_coff, tx * kTileW, ty * kTileH + 4 * q, b);
          ptx::bulk_commit();
        }
        obuf ^= 1;
      }
      XMM_PROF_ADD(5);
    }
    if (use_tma && ptx::elect_one()) ptx::bulk_wait<0>();  // stores complete before the CTA (and its smem) goes away
    if (NT == 32 && do_csum) {
      float (&cs32)[32] = reinterpret_cast<float (&)[32]>(csum);
      colsum_flush<32>(args.epi, cs32, 0, lane);
    }
    if (warp == 2 && lane == 0) { XMM_PROF_FLUSH(4); XMM_PROF_FLUSH(5); }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
#ifdef XMM_CONV_PROFILE
  if (threadIdx.x == 0) {
    unsigned long long g1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
    args.prof[size_t(blockIdx.x) * 8 + 6] = clock64() - prof_k0_;
    args.prof[size_t(blockIdx.x) * 8 + 7] = (long long)(g1 - prof_g0_);
  }
#endif
}

}  // namespace xmm
