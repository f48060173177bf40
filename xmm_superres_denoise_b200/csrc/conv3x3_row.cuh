// 3x3 / stride 1 / pad 1 convolution, "row-hop" form, for the narrow layers (Cout = 32 or 64) of the reference's
// dense blocks (rrdb_blocks.py:27-31,37-54), trunk_conv / HRconv (generator_rrdb.py:39-45,101) and their data
// gradients.
//
// Why a third form.  The column-scatter form (conv3x3_dx.cuh) made one N = 3*Cout MMA out of the three dx taps of a
// filter row, but has to add the three partial sums one pixel apart along the M (= TMEM lane) dimension: 64
// shuffles, a carry mailbox and ~320 instructions per warp and tile on a 136 KB kernel body.  ncu's source page put
// 55 % of its stall samples on branch resolution, fixed-latency waits and instruction fetch; its tile period was
// 1900-2400 cycles whatever Cin, for 670-1700 cycles of MMA.
//
// Here the shift that is summed in the epilogue is replaced by a shift BETWEEN ACCUMULATORS.  A tile is ONE image row
// of each of 16 horizontal bands of the image, 8 pixels wide: M = 128 = [16 bands][8 px].  The dx taps are
// descriptor views of the [16][10]-pixel patch (start address + one pixel, SBO = 10 pixels: conv3x3_tc.cuh's proven
// haloed-tap-view operand), and the three dy taps are the N = 3*Cout columns of one MMA:
//
//     step r (input row r of every band):   D[:, (2 - dy) * Cout + co] += X[r][x + dx - 1][:] . W[dy][dx][co][:]
//
// whose three Cout-column blocks belong to output rows r-1 (dy = 2), r (dy = 1) and r+1 (dy = 0).  Output row j lives
// in TMEM accumulator slot j mod S (S = 512 / Cout slots of Cout columns), so the MMA of step r simply targets the
// CONTIGUOUS slot window (r-1, r, r+1): every partial sum lands in the accumulator of the pixel it belongs to, with
// the same lane mapping.  After step j+1 output row j is complete.  The epilogue is a plain GEMM epilogue: one
// tcgen05.ld of Cout columns, bias / LeakyReLU / mask / residuals, one TMA store.  No shuffles, no carries, a third
// of the TMEM reads.
//
// Accumulator bookkeeping.  The first MMA that touches a slot must overwrite it: the first instruction of a step is
// split into [blocks already started: accumulate][new block: overwrite]; a window that straddles the end of the slot
// ring is split in two.  A CTA walks a column of the image ((image, 8-px column), rows top to bottom); the input rows
// above / below a band are the neighbouring bands' rows (TMA band coordinate -1 / +1; outside the image = the zero
// padding).  Pieces that start or end mid-column only pay one extra input row at each end.
//
// Layout.  The banded view is a 5-D tensor map (c, x, row-in-band, band, image) of the NHWC buffer (H = nbands *
// band_h, nbands <= 16: lanes of missing bands compute on zero-filled rows and are clipped by the store).
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM owner), warps 2..9 = two epilogue
// groups of four (TMEM lane quarter = warp % 4) that take alternate output rows.
#pragma once
#include "conv3x3_tc.cuh"

namespace xmm {

constexpr int kRowBands = 16;
constexpr int kRowPx = 8;
constexpr int kRowPitch = kRowPx + 2;
constexpr int kRowEpiWarps = 8;
constexpr int kRowThreads = 64 + 32 * kRowEpiWarps;
static_assert(kRowEpiWarps <= kCsumWarpSlots, "one deterministic column-sum slot per epilogue warp");
// EVEN, like the accumulator slots: output rows alternate between the two epilogue groups, so with an even ring every
// stage is always waited for by the SAME group, which therefore sees each of the barrier's phases.  (With 3 stages a
// group saw every other phase of a stage's "landed" barrier: a parity wait two phases ahead passes at once, the
// group read the side tile before it had landed and released it early -- wrong residuals / masks or a wedged
// pipeline, depending on timing; found with the protocol simulator of the fused kernels, tools/rdb_protocol_sim.py.)
constexpr int kRowSideStages = 4;  // NT = 32; the 64-filter instantiation takes 2 (RowCfg::kSideStages)
constexpr int kRowMaxSlots = 16;

// compile-time epilogue variants (the launcher picks the instantiation; see row_epilogue_math)
enum RowEpi : int { kRowLrelu = 1, kRowMask = 2, kRowR1 = 4, kRowR2 = 8, kRowCsum = 16 };

template <int KC, int NT>
struct RowCfg {
  static_assert(KC == 32 || KC == 64, "K chunk is 32 (SWIZZLE_64B) or 64 (SWIZZLE_128B) channels");
  static_assert(NT == 32 || NT == 64, "row-hop form is for Cout 32 / 64");
  static constexpr int kRowB = KC * 2;
  static constexpr uint32_t kLayout = (KC == 64) ? ptx::UMMA_SW128 : ptx::UMMA_SW64;
  static constexpr int kStageBytes = kRowBands * kRowPitch * kRowB;  // 10 KB / 20 KB
  static constexpr int kKSteps = KC / 16;
  static constexpr int kTapBytes = NT * kRowB;
  static constexpr int kSlots = 512 / NT;  // accumulator slots (one output row each)
  static constexpr int kSideStages = NT == 32 ? kRowSideStages : 2;  // even (see kRowSideStages); 16 KB tiles at NT = 64
  static constexpr int kBiasBytes = NT * 4;
  static constexpr int kWarpOutBytes = 32 * NT * 2;  // [4 bands][8 px] x NT bf16, swizzled
  static constexpr int kOutBytes = kRowEpiWarps * kWarpOutBytes;
  static constexpr int kSideTileBytes = kRowBands * kRowPx * NT * 2;  // one side input of one output row
  // full[8] empty[8] tfull[16] tempty[16] w sfull[3] sempty[3] + tmem pointer
  static constexpr int kBarBytes = (2 * kMaxStages + 2 * kRowMaxSlots + 1 + 2 * kRowSideStages) * 8 + 16;
  static size_t smem_bytes(uint32_t w_bytes, int stages, int nside) {
    return 1024 + ((size_t(w_bytes) + kBiasBytes + 1023) & ~size_t(1023)) + size_t(stages) * kStageBytes + kOutBytes +
           size_t(kSideStages * nside) * kSideTileBytes + kBarBytes;
  }
};

struct RowArgs {
  const void* wblob;  // packed weights, row-hop tap order [chunk][dx][2 - dy][Cout][KC] + bias
  uint32_t w_bytes;
  int nchunks;
  int cin_off;
  int batch, height, width;
  int band_h, nbands;  // height == band_h * nbands
  int tiles_x;         // ceil(width / 8)
  int ncols;           // batch * tiles_x columns of band_h output rows
  int rr_rounds;       // whole columns dealt round-robin before the tail is cut into equal row ranges
  int stages;
  int side_mask;       // bit k: side input k (0 mask, 1 r1, 2 r2) present
  ConvEpilogue epi;
};

struct RowSideMaps {
  CUtensorMap m[3];
};

// This CTA's work as PIECES (column, first output row, end row).  Round-robin part: column blockIdx.x + i * gridDim.x
// (neighbouring CTAs walk neighbouring columns at the same pace: the two halo pixels they share meet in L2).  Tail:
// the rows of the columns that do not fill a round are cut into gridDim.x equal contiguous ranges.
struct RowSched {
  int rr_rounds, grid, cta, band_h, tiles_x;
  int tail_col0, tail_c0;  // first tail column, first column (relative) of this CTA's tail range
  long long t0, t1;
  int npieces;
  __device__ __forceinline__ void init(const RowArgs& a) {
    grid = int(gridDim.x);
    cta = int(blockIdx.x);
    band_h = a.band_h;
    tiles_x = a.tiles_x;
    rr_rounds = a.rr_rounds;
    tail_col0 = rr_rounds * grid;
    const long long total = (long long)(a.ncols - tail_col0) * band_h;
    t0 = total * cta / grid;
    t1 = total * (cta + 1) / grid;
    tail_c0 = int(t0 / band_h);
    const int ntail = t1 > t0 ? int((t1 - 1) / band_h) - tail_c0 + 1 : 0;
    npieces = rr_rounds + ntail;
  }
  __device__ __forceinline__ void get(int i, int& b, int& xt, int& ra, int& rb) const {
    int col;
    if (i < rr_rounds) {
      col = cta + i * grid;
      ra = 0;
      rb = band_h;
    } else {
      const int c = tail_c0 + (i - rr_rounds);
      col = tail_col0 + c;
      const long long base = (long long)c * band_h;
      ra = t0 > base ? int(t0 - base) : 0;
      rb = t1 < base + band_h ? int(t1 - base) : band_h;
    }
    b = col / tiles_x;
    xt = col - b * tiles_x;
  }
};

struct RowSeg {
  uint32_t boff16;  // weight-operand offset of the segment's first block (16-byte units)
  uint32_t dcol;    // TMEM column of its first slot
  uint32_t idesc;
  uint32_t acc;
};

// Fused epilogue arithmetic on 32 accumulator columns [col0, col0 + 32) of one pixel (ConvEpilogue's definition):
//   t = acc + bias; v = t > 0 ? t : slope * t; v *= mask > 0 ? 1 : mask_slope; v = s0 * v + s1 * r1 + s2 * r2
// Side inputs come from the TMA-staged tiles of this output row (16-byte chunks at swizzled positions).
template <int NT, int EPI>
__device__ __forceinline__ void row_epilogue_math(const ConvEpilogue& e, const float* __restrict__ bias_s, float (&v)[32],
                                                  int col0, const uint8_t* const (&side)[3], uint32_t row_off,
                                                  uint32_t xor_mask) {
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 b4 = *reinterpret_cast<const float4*>(bias_s + col0 + 4 * q);
    v[4 * q] += b4.x;
    v[4 * q + 1] += b4.y;
    v[4 * q + 2] += b4.z;
    v[4 * q + 3] += b4.w;
  }
  if (EPI & kRowLrelu) {
    const float slope = e.lrelu_slope;
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = v[i] > 0.f ? v[i] : v[i] * slope;
  }
  const uint32_t chunk0 = uint32_t(col0 >> 3);
  if (EPI & kRowMask) {
    const float ms = e.mask_slope;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float m[8];
      unpack8(*reinterpret_cast<const uint4*>(side[0] + row_off + (((chunk0 + uint32_t(q)) ^ xor_mask) << 4)), m);
#pragma unroll
      for (int i = 0; i < 8; ++i) v[q * 8 + i] *= (m[i] > 0.f ? 1.f : ms);
    }
  }
  if (e.s0 != 1.f) {
    const float s0 = e.s0;
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] *= s0;
  }
  if (EPI & kRowR1) {
    const float s1 = e.s1;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float m[8];
      unpack8(*reinterpret_cast<const uint4*>(side[1] + row_off + (((chunk0 + uint32_t(q)) ^ xor_mask) << 4)), m);
#pragma unroll
      for (int i = 0; i < 8; ++i) v[q * 8 + i] = fmaf(s1, m[i], v[q * 8 + i]);
    }
  }
  if (EPI & kRowR2) {
    const float s2 = e.s2;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float m[8];
      unpack8(*reinterpret_cast<const uint4*>(side[2] + row_off + (((chunk0 + uint32_t(q)) ^ xor_mask) << 4)), m);
#pragma unroll
      for (int i = 0; i < 8; ++i) v[q * 8 + i] = fmaf(s2, m[i], v[q * 8 + i]);
    }
  }
}

template <int KC, int NT, int EPI>
__global__ void __launch_bounds__(kRowThreads, 1)
conv3x3_row_kernel(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_out,
                   const __grid_constant__ RowSideMaps side_maps, const RowArgs args) {
  using Cfg = RowCfg<KC, NT>;
  constexpr int kSlots = Cfg::kSlots;
  constexpr int kSlotShift = kSlots == 16 ? 4 : 3;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w_s = smem;
  float* bias_s = reinterpret_cast<float*>(smem + args.w_bytes);
  uint8_t* stage_s = smem + ((args.w_bytes + Cfg::kBiasBytes + 1023) & ~1023u);
  uint8_t* out_s = stage_s + size_t(args.stages) * Cfg::kStageBytes;
  uint8_t* side_s = out_s + Cfg::kOutBytes;
  const int nside = __popc(args.side_mask);
  uint64_t* bars = reinterpret_cast<uint64_t*>(side_s + size_t(Cfg::kSideStages * nside) * Cfg::kSideTileBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kMaxStages;
  uint64_t* tfull_bar = bars + 2 * kMaxStages;
  uint64_t* tempty_bar = tfull_bar + kRowMaxSlots;
  uint64_t* w_bar = tempty_bar + kRowMaxSlots;
  uint64_t* sfull_bar = w_bar + 1;
  uint64_t* sempty_bar = sfull_bar + kRowSideStages;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(sempty_bar + kRowSideStages);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_in);
    ptx::prefetch_tmap(&tmap_out);
    for (int s = 0; s < args.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < kSlots; ++a) {
      ptx::mbar_init(&tfull_bar[a], 1);
      ptx::mbar_init(&tempty_bar[a], 4);  // the four warps of the group that drains this slot
    }
    ptx::mbar_init(w_bar, 1);
    for (int a = 0; a < Cfg::kSideStages; ++a) {
      ptx::mbar_init(&sfull_bar[a], 1);
      ptx::mbar_init(&sempty_bar[a], 4);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc<512>(tmem_ptr_s);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;

  RowSched sched;
  sched.init(args);

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (ptx::elect_one()) {
      const uint8_t* gsrc = static_cast<const uint8_t*>(args.wblob);
      const uint32_t wtot = args.w_bytes + Cfg::kBiasBytes;
      ptx::mbar_expect_tx(w_bar, wtot);
      for (uint32_t off = 0; off < wtot; off += 32768u) {
        const uint32_t n = (wtot - off < 32768u) ? (wtot - off) : 32768u;
        ptx::bulk_load(w_s + off, gsrc + off, n, w_bar);
      }
      int stage = 0;
      uint32_t phase = 0;
      int sst = 0;
      uint32_t sphase = 0;
      const int coff[3] = {args.epi.mask_coff, args.epi.r1_coff, args.epi.r2_coff};
      for (int i = 0; i < sched.npieces; ++i) {
        int b, xt, ra, rb;
        sched.get(i, b, xt, ra, rb);
        const int x0 = xt * kRowPx - 1;
        for (int r = ra - 1; r <= rb; ++r) {
          // input row r of every band; above / below a band: the neighbouring band's last / first row
          int row = r, band0 = 0;
          if (r < 0) {
            row = args.band_h - 1;
            band0 = -1;
          } else if (r >= args.band_h) {
            row = 0;
            band0 = 1;
          }
          for (int ch = 0; ch < args.nchunks; ++ch) {
            ptx::mbar_wait(&empty_bar[stage], phase ^ 1u);
            ptx::mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
            ptx::tma_load_5d(stage_s + size_t(stage) * Cfg::kStageBytes, &tmap_in, &full_bar[stage],
                             args.cin_off + ch * KC, x0, row, band0, b);
            if (++stage == args.stages) {
              stage = 0;
              phase ^= 1u;
            }
          }
          if (nside > 0 && r - 1 >= ra) {  // side inputs of output row r-1, which this step completes
            ptx::mbar_wait(&sempty_bar[sst], sphase ^ 1u);
            ptx::mbar_expect_tx(&sfull_bar[sst], uint32_t(nside) * Cfg::kSideTileBytes);
            uint8_t* dst = side_s + size_t(sst * nside) * Cfg::kSideTileBytes;
#pragma unroll
            for (int k = 0; k < 3; ++k)
              if (args.side_mask & (1 << k)) {
                ptx::tma_load_5d(dst, &side_maps.m[k], &sfull_bar[sst], coff[k], xt * kRowPx, r - 1, 0, b);
                dst += Cfg::kSideTileBytes;
              }
            if (++sst == Cfg::kSideStages) {
              sst = 0;
              sphase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (ptx::elect_one()) {
      ptx::mbar_wait(w_bar, 0);
      ptx::tc_fence_after();
      const uint64_t bdesc0 = ptx::umma_smem_desc(ptx::smem_u32(w_s), 16, 8 * Cfg::kRowB, Cfg::kLayout);
      const uint64_t adesc0 = ptx::umma_smem_desc(ptx::smem_u32(stage_s), 16, kRowPitch * Cfg::kRowB, Cfg::kLayout);
      // descriptors as (low, high) words: every offset below is a 32-bit add on the low word (16-byte units)
      const uint32_t a_hi = uint32_t(adesc0 >> 32), b_hi = uint32_t(bdesc0 >> 32);
      const uint32_t a_lo0 = uint32_t(adesc0), b_lo0 = uint32_t(bdesc0);
      constexpr uint32_t kTap16 = uint32_t(Cfg::kTapBytes) >> 4;
      constexpr uint32_t kIdesc0 = ptx::umma_idesc_bf16_f32(128, 0, 0, 0);  // + (N >> 3) << 17
      constexpr uint32_t kIdescBlk = uint32_t(NT >> 3) << 17;
      int stage = 0;
      uint32_t phase = 0;
      int v = 0;  // output rows before the current piece (slot = row counter mod kSlots)
      for (int i = 0; i < sched.npieces; ++i) {
        int b, xt, ra, rb;
        sched.get(i, b, xt, ra, rb);
        for (int r = ra - 1; r <= rb; ++r) {
          const int j0 = r - 1 > ra ? r - 1 : ra;
          const int j1 = r + 1 < rb - 1 ? r + 1 : rb - 1;
          const int nblk = j1 - j0 + 1;       // 1..3 output rows take a contribution from input row r
          const int jb = j0 - (r - 1);        // first weight block (block k <-> output row r-1+k <-> dy = 2-k)
          const int vj0 = v + (j0 - ra);
          const bool has_new = r + 1 <= rb - 1;  // output row r+1 is touched for the first time
          // MMA segments of this step.  A window that straddles the end of the slot ring is split there (the second
          // part starts at slot 0); in the step's FIRST instruction the new block is an overwriting instruction of
          // its own.
          const int s0 = vj0 & (kSlots - 1);
          const int wrap = kSlots - s0;                // blocks before the ring end
          const int nold = has_new ? nblk - 1 : nblk;  // blocks that already hold partial sums
          const int a0_len = nold < wrap ? nold : wrap, a1_len = nold - a0_len;
          const int b0_len = nblk < wrap ? nblk : wrap, b1_len = nblk - b0_len;
          const uint32_t d0 = tmem_base + uint32_t(s0 * NT);
          const uint32_t d_new = tmem_base + uint32_t(((vj0 + nblk - 1) & (kSlots - 1)) * NT);
          const uint32_t bw0 = b_lo0 + uint32_t(jb) * kTap16;           // first block of the window
          const uint32_t bw1a = bw0 + uint32_t(a0_len) * kTap16;        // second part (after the ring end), first MMA
          const uint32_t bw1b = bw0 + uint32_t(b0_len) * kTap16;        // second part, other MMAs
          const uint32_t bw_new = bw0 + uint32_t(nblk - 1) * kTap16;
          const uint32_t id_a0 = kIdesc0 + uint32_t(a0_len) * kIdescBlk, id_a1 = kIdesc0 + uint32_t(a1_len) * kIdescBlk;
          const uint32_t id_b0 = kIdesc0 + uint32_t(b0_len) * kIdescBlk, id_b1 = kIdesc0 + uint32_t(b1_len) * kIdescBlk;
          constexpr uint32_t id_new = kIdesc0 + kIdescBlk;
          if (has_new) {  // the slot's previous occupant (kSlots rows ago) has been drained
            const int vnew = v + (r + 1 - ra);
            ptx::mbar_wait(&tempty_bar[vnew & (kSlots - 1)], (uint32_t(vnew >> kSlotShift) & 1u) ^ 1u);
            ptx::tc_fence_after();
          }
          for (int ch = 0; ch < args.nchunks; ++ch) {
            ptx::mbar_wait(&full_bar[stage], phase);
            ptx::tc_fence_after();
            const uint32_t a_st = a_lo0 + uint32_t(stage) * (uint32_t(Cfg::kStageBytes) >> 4);
            const uint32_t b_ch = uint32_t(ch) * 9u * kTap16;
            if (ch == 0) {  // first instruction of the step
              if (a0_len > 0) ptx::umma_ss_lh<true>(d0, a_st, a_hi, bw0 + b_ch, b_hi, id_a0);
              if (a1_len > 0) ptx::umma_ss_lh<true>(tmem_base, a_st, a_hi, bw1a + b_ch, b_hi, id_a1);
              if (has_new) ptx::umma_ss_lh<false>(d_new, a_st, a_hi, bw_new + b_ch, b_hi, id_new);
            }
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
              for (int ks = 0; ks < Cfg::kKSteps; ++ks) {
                if (dx == 0 && ks == 0) {
                  if (ch == 0) continue;
                }
                const uint32_t a_off = uint32_t(dx * Cfg::kRowB + ks * 32) >> 4;
                const uint32_t b_off = (uint32_t(dx * 3) * uint32_t(Cfg::kTapBytes) + uint32_t(ks * 32)) >> 4;
                ptx::umma_ss_lh<true>(d0, a_st + a_off, a_hi, bw0 + b_ch + b_off, b_hi, id_b0);
                if (b1_len > 0) ptx::umma_ss_lh<true>(tmem_base, a_st + a_off, a_hi, bw1b + b_ch + b_off, b_hi, id_b1);
              }
            }
            ptx::umma_commit(&empty_bar[stage]);
            if (++stage == args.stages) {
              stage = 0;
              phase ^= 1u;
            }
          }
          if (r - 1 >= ra) ptx::umma_commit(&tfull_bar[(v + (r - 1 - ra)) & (kSlots - 1)]);  // row r-1 is complete
        }
        v += rb - ra;
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue
    ptx::mbar_wait(w_bar, 0);  // bias rides with the weights
    const int q = warp & 3;             // TMEM lane quarter this warp may read
    const int group = (warp - 2) >> 2;  // output rows v with (v & 1) == group
    const int m = q * 32 + lane;        // MMA row: band m / 8, pixel m % 8
    const int band = m >> 3, px = m & 7;
    uint8_t* stage = out_s + (warp - 2) * Cfg::kWarpOutBytes;
    const uint32_t out_xor = NT == 32 ? uint32_t((lane >> 1) & 3) : uint32_t(lane & 7);
    const uint32_t side_row = uint32_t(m * NT * 2);
    const uint32_t side_xor = NT == 32 ? uint32_t((m >> 1) & 3) : uint32_t(m & 7);
    float csum[(EPI & kRowCsum) ? NT : 1];
#pragma unroll
    for (int k = 0; k < ((EPI & kRowCsum) ? NT : 1); ++k) csum[k] = 0.f;
    int v = 0;
    for (int i = 0; i < sched.npieces; ++i) {
      int b, xt, ra, rb;
      sched.get(i, b, xt, ra, rb);
      const bool valid = band < args.nbands && xt * kRowPx + px < args.width;
      for (int j = ra; j < rb; ++j, ++v) {
        if ((v & 1) != group) continue;
        const int slot = v & (kSlots - 1);
        ptx::mbar_wait(&tfull_bar[slot], uint32_t(v >> kSlotShift) & 1u);
        ptx::tc_fence_after();
        const uint32_t t_addr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(slot * NT);
        const int sst = v % Cfg::kSideStages;
        const uint8_t* side[3] = {nullptr, nullptr, nullptr};
        if (EPI & (kRowMask | kRowR1 | kRowR2)) {
          ptx::mbar_wait(&sfull_bar[sst], uint32_t(v / Cfg::kSideStages) & 1u);
          const uint8_t* src = side_s + size_t(sst * nside) * Cfg::kSideTileBytes;
#pragma unroll
          for (int k = 0; k < 3; ++k)
            if (args.side_mask & (1 << k)) {
              side[k] = src;
              src += Cfg::kSideTileBytes;
            }
        }
        // the TMA store of this warp's previous row has finished reading the staging tile
        if (ptx::elect_one()) ptx::bulk_wait_read<0>();
        __syncwarp();
#pragma unroll
        for (int cc = 0; cc < NT / 32; ++cc) {
          uint32_t accr[32];
          ptx::tmem_ld_32x32(t_addr + uint32_t(cc * 32), accr);
          ptx::tmem_ld_wait();
          if (cc == NT / 32 - 1) {
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&tempty_bar[slot]);
          }
          float val[32];
#pragma unroll
          for (int k = 0; k < 32; ++k) val[k] = __uint_as_float(accr[k]);
          row_epilogue_math<NT, EPI>(args.epi, bias_s, val, cc * 32, side, side_row, side_xor);
          if (EPI & kRowCsum) {
            if (valid) {
#pragma unroll
              for (int k = 0; k < 32; ++k) csum[(EPI & kRowCsum) ? cc * 32 + k : 0] += val[k];
            }
          }
#pragma unroll
          for (int k = 0; k < 4; ++k)
            *reinterpret_cast<uint4*>(stage + lane * (NT * 2) + ((uint32_t(cc * 4 + k) ^ out_xor) << 4)) = pack8(val + k * 8);
        }
        if (EPI & (kRowMask | kRowR1 | kRowR2)) {
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&sempty_bar[sst]);
        }
        ptx::fence_proxy_async();  // this thread's st.shared -> visible to the async proxy
        __syncwarp();
        if (ptx::elect_one()) {
          ptx::tma_store_5d(&tmap_out, stage, args.epi.out_coff, xt * kRowPx, j, 4 * q, b);
          ptx::bulk_commit();
        }
      }
    }
    if (ptx::elect_one()) ptx::bulk_wait<0>();  // stores complete before the CTA (and its shared memory) goes away
    if (EPI & kRowCsum) {
      constexpr int kN = (EPI & kRowCsum) ? NT : 1;
      float (&cs)[kN] = csum;
      if (kN > 1) colsum_flush<kN>(args.epi, cs, 0, lane);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace xmm
