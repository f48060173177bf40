// 3x3 / stride 1 / pad 1 convolution, "row-gather / column-scatter" form, for narrow layers
// (Cout = 32 or 64: every conv of the reference's dense blocks, rrdb_blocks.py:27-31, and their
// data gradients).
//
// Why a second form.  With pixels on M and Cout on N (conv3x3_tc.cuh) one tcgen05.mma reads a
// 128-row A slice (4 KB) from shared memory to feed only N = 32 columns; the instruction is
// shared-memory bound at 32 + N/4 = 40 cycles for 16 cycles of math (measured, tools/probe.cu).
// Here the three taps of one filter ROW share one A read:
//
//     D_dx[y][x'] = sum_dy sum_ci X[y + dy - 1][x'][ci] * W[dy][dx][co][ci]        (N = 3 * Cout)
//     out[y][x]   = D_0[y][x - 1] + D_1[y][x] + D_2[y][x + 1]
//
// so a (dy, k-step) pair is ONE MMA with N = 96 (56 cycles for 48 of math) instead of three.
// dy stays a gather: the M = 128 rows are an [8 rows][16 columns] pixel block of the [10][16]
// row-haloed patch, and a row shift is a 1 KB-aligned start address (canonical K-major layout).
//
// The +-1 column shift is applied in the epilogue.  Neighbouring columns are neighbouring TMEM lanes =
// neighbouring threads of an epilogue warp (two image rows of 16 columns per warp): two warp shuffles per
// output value.  Across the 16-column tile boundary the sums are CARRIED: a CTA walks a strip of 8 image
// rows left to right; lane 15 of each row leaves D_0[15] (the left term of the next tile's column 0) and the
// unfinished sum D_0[14] + D_1[15] of its own column in a per-warp shared-memory mailbox and completes -- and
// stores -- that column one tile later, when lane 0 holds D_2[16].  No column halo is ever loaded or multiplied:
// every MMA row is a useful pixel (D_0[-1] and D_2[W] are products with the zero padding).  The mailbox moves
// are predicated 16-byte shared-memory accesses of the two boundary lanes, so the common path has no selects.
//
// Work split.  Large problems (>= 4 strips per CTA): whole strips are dealt round-robin, so that at any moment the
// CTAs work on a band of ADJACENT strips at about the same column -- the two halo rows a strip shares with its
// neighbours are then read from L2 instead of HBM (measured: with contiguous ranges the halo was re-read from
// DRAM, 1.25x the algorithmic traffic, and the kernel is DRAM-bound for cin >= 96).  Small problems: the
// B * ceil(H/8) * ceil(W/16) tiles, strip-major, are cut into gridDim.x equal contiguous ranges; a range that
// starts mid-strip first runs the tile before it as a "pre-tile" (outputs suppressed) to establish the carry, a
// range that ends mid-strip leaves its last column to the next CTA's pre-tile.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM owner), warps 2..9 = epilogue:
// TMEM lane quarter = warp_id % 4, and the two warps of a quarter take half of the Cout columns each.  Every
// epilogue warp stages its [2 rows][16 px][Cout/2] result in its own swizzled shared-memory tile and issues its
// own TMA store (box x = 16*tx - 1: the carried column comes first; rows / columns outside the image are clipped
// by the tensor map), so the epilogue warps never synchronise with each other.  A TMA store may not start at a
// negative coordinate (illegal instruction on B200), so tile 0 of a strip stores directly.
//
// CTA pairs (template PAIR, round-robin mode only).  An N = 96 MMA reads 4 KB of A + 3 KB of B from shared memory:
// 56 cycles at 128 B/clk for 48 cycles of math -- and the TMA fills and the epilogue use the same port.  Two CTAs
// of a cluster run as a tcgen05 cta_group::2 pair: each walks its OWN strips exactly as above (own activation
// stages, TMEM accumulators, epilogue, stores), but the leader's MMA warp issues ONE M = 256 instruction for both
// (rows 0..127 = the leader's pixel block, 128..255 = the peer's) and each CTA supplies only HALF of the weight
// rows: 5.5 KB per CTA and instruction, 49 cycles measured (tools/probe_pair.cu).  The peer's resident weight image
// is loaded 48 rows "early" so that the same descriptor offsets address rows 48..95 of every (chunk, filter row)
// group.  The pair runs in lock step: the peer's TMA loads complete on the LEADER's full barriers, the peer's
// epilogue warps release accumulators on the leader's barriers, the leader's commits are multicast to both CTAs.
// When the peer has one strip fewer it repeats its first strip with all outputs suppressed.
//
// Everything else -- resident weights, TMA pipeline, TMEM accumulator ring, fused bias / LeakyReLU / mask /
// residual / inverse-pixel-shuffle arithmetic -- is conv3x3_tc.cuh's.  The packed weight image is the same one
// ([chunk][tap][Cout][KC]: the three dx taps of a row are adjacent, so they are one N = 3*Cout operand).
#pragma once
#include "conv3x3_tc.cuh"

namespace xmm {

constexpr int kDxTileH = 8;
constexpr int kDxTileW = 16;
constexpr int kDxPatchH = kDxTileH + 2;
constexpr int kDxEpiWarps = 8;
constexpr int kDxThreads = 64 + 32 * kDxEpiWarps;
static_assert(kDxEpiWarps <= kCsumWarpSlots, "one deterministic column-sum slot per epilogue warp");

// G2: the eight epilogue warps form TWO GROUPS of four (one warp per TMEM lane quarter, all Cout columns each) that
// work on DIFFERENT strips; the MMA warp alternates tiles between the two strips.  An epilogue pass costs a warp
// ~1800 cycles per tile whatever the layer (about a quarter of it per-tile fixed cost), and with all eight warps on
// every tile that pass -- not the MMA stream -- is the tile period for Cin <= 128.
template <int KC, int NT, bool G2 = false>
struct DxCfg {
  static_assert(KC == 32 || KC == 64, "K chunk is 32 (SWIZZLE_64B) or 64 (SWIZZLE_128B) channels");
  static_assert(NT == 32 || NT == 64, "column-scatter form is for Cout 32 / 64");
  static constexpr int kRowB = KC * 2;
  static constexpr uint32_t kLayout = (KC == 64) ? ptx::UMMA_SW128 : ptx::UMMA_SW64;
  static constexpr int kStageBytes = kDxPatchH * kDxTileW * kRowB;  // 10 KB / 20 KB: a multiple of 1024
  static constexpr int kKSteps = KC / 16;
  static constexpr int kTapBytes = NT * kRowB;
  static constexpr int kAccCols = 3 * NT;
  static constexpr int kAccStages = 512 / kAccCols >= 4 ? 4 : 2;  // accumulator ring in TMEM (4 x 96 or 2 x 192 columns)
  static constexpr int kTmemCols = 512;
  static constexpr uint32_t kIdesc = ptx::umma_idesc_bf16_f32(128, 3 * NT, 0, 0);
  static constexpr int kBiasBytes = NT * 4;
  static constexpr int kBarBytes = (2 * kMaxStages + 2 * 4 + 1) * 8 + 16;
  static constexpr int kGroups = G2 ? 2 : 1;
  static constexpr int kTileWarps = kDxEpiWarps / kGroups;  // epilogue warps that share one tile
  static constexpr int kWarpCols = G2 ? NT : NT / 2;  // Cout columns owned by one epilogue warp
  static constexpr int kWarpChunks = kWarpCols / 16;  // 16-column groups per tcgen05.ld / arithmetic pass
  // per-warp output staging tile for the TMA store: [2 rows][16 px] x kWarpCols bf16, swizzled (32 B / 64 B rows)
  static constexpr int kWarpOutBytes = 32 * kWarpCols * 2;
  static constexpr int kOutBytes = kDxEpiWarps * 2 * kWarpOutBytes;  // double buffered
  // per-warp carry mailboxes: [parity][A = D_0 of column 15 | B = unfinished column 15][half-warp row][kWarpCols] fp32
  static constexpr int kWarpMailBytes = 2 * 2 * 2 * kWarpCols * 4;
  static constexpr int kMailBytes = kDxEpiWarps * kWarpMailBytes;
  // side-input tile (mask / residual of the output pixels): [8 rows][16 px] x NT bf16, TMA swizzled, double buffered
  static constexpr int kSideTileBytes = kDxTileH * kDxTileW * NT * 2;
  static size_t smem_bytes(uint32_t w_bytes, int stages, int nside = 0) {
    return 1024 + w_bytes + kBiasBytes + 1024 + size_t(stages) * kStageBytes + kOutBytes + kMailBytes +
           size_t(2 * nside) * kSideTileBytes + kBarBytes + 4 * 8;
  }
};

// Byte offset of 16-byte chunk k16 of warp-local pixel p (0..31) inside a warp's staging tile: rows of 32 B
// (SWIZZLE_32B: chunk bit 4 ^= address bit 7) or 64 B (SWIZZLE_64B: chunk bits [4,6) ^= address bits [7,9)) --
// the layout the output tensor map expects, and conflict-free for the warp's 16-byte stores.
template <int WC>  // WC = columns per warp: 16 -> 32-byte rows, 32 -> 64-byte rows
__device__ __forceinline__ uint32_t dx_out_offset(int p, int k16) {
  if (WC == 16) return uint32_t(p * 32 + ((k16 ^ ((p >> 2) & 1)) << 4));
  return uint32_t(p * 64 + ((k16 ^ ((p >> 1) & 3)) << 4));
}

// Predicated 16-byte shared-memory moves IN PLACE (the boundary lanes' mailbox traffic must not turn into a
// select per value on the other 30 lanes).
__device__ __forceinline__ void lds4_if(bool p, float& a, float& b, float& c, float& d, uint32_t addr) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %4, 0;\n\t"
      "@q ld.shared.v4.f32 {%0, %1, %2, %3}, [%5];\n\t"
      "}\n"
      : "+f"(a), "+f"(b), "+f"(c), "+f"(d)
      : "r"(int(p)), "r"(addr)
      : "memory");
}
__device__ __forceinline__ void sts4_if(bool p, float a, float b, float c, float d, uint32_t addr) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %4, 0;\n\t"
      "@q st.shared.v4.f32 [%5], {%0, %1, %2, %3};\n\t"
      "}\n" ::"f"(a),
      "f"(b), "f"(c), "f"(d), "r"(int(p)), "r"(addr)
      : "memory");
}

// Tile g of the strip-major order -> image, strip row, tile column.
struct DxTile {
  int b, ty, tx;
  __device__ __forceinline__ DxTile(int g, int tiles_x, int tiles_y) {
    const int strip = g / tiles_x;
    tx = g - strip * tiles_x;
    b = strip / tiles_y;
    ty = strip - b * tiles_y;
  }
  __device__ __forceinline__ void next(int tiles_x, int tiles_y) {
    if (++tx == tiles_x) {
      tx = 0;
      if (++ty == tiles_y) {
        ty = 0;
        ++b;
      }
    }
  }
};

// The MMAs of one K-chunk (KC channels) of one tile: per filter row dy, KC/16 instructions of N = 3*NT.
template <int KC, int NT, bool PAIR = false>
__device__ __forceinline__ void dx_issue_chunk(uint32_t d_addr, uint64_t adesc_st, uint64_t bdesc_ch, bool first_chunk) {
  using Cfg = DxCfg<KC, NT>;
  constexpr uint32_t kIdescPair = ptx::umma_idesc_bf16_f32(256, 3 * NT, 0, 0);
#pragma unroll
  for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
    for (int ks = 0; ks < Cfg::kKSteps; ++ks) {
      const uint64_t adesc = adesc_st + uint64_t((uint32_t(dy * kDxTileW * Cfg::kRowB) + uint32_t(ks * 32)) >> 4);
      const uint64_t bdesc = bdesc_ch + uint64_t((uint32_t(dy * 3 * Cfg::kTapBytes) + uint32_t(ks * 32)) >> 4);
      if (PAIR)
        ptx::umma_ss_pair(d_addr, adesc, bdesc, kIdescPair, (first_chunk && dy == 0 && ks == 0) ? 0u : 1u);
      else
        ptx::umma_ss(d_addr, adesc, bdesc, Cfg::kIdesc, (first_chunk && dy == 0 && ks == 0) ? 0u : 1u);
    }
  }
}

// Per-warp constants of the epilogue.
template <int KC, int NT, bool G2 = false>
struct DxEpiWarp {
  using Cfg = DxCfg<KC, NT, G2>;
  int lane, q, half, group, prow, pcol, col_w;
  bool first_col, last_col;
  int src_l, src_r;
  uint32_t mail;       // shared-memory address of this warp's mailboxes (+ this lane's half-warp row)
  uint8_t* out_tile;   // this warp's two staging tiles
  float bias[Cfg::kWarpCols];
  float csum[Cfg::kWarpCols];  // fused bias gradient: this lane's running column sums (ConvEpilogue::colsum)
  int par;             // tile parity (mailbox / staging double buffering)
#ifdef XMM_CONV_PROFILE
  long long phase[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
  __device__ __forceinline__ void init(int warp, int lane_, const float* bias_s, uint8_t* out_s, uint8_t* mail_s) {
    lane = lane_;
    q = warp & 3;
    half = G2 ? 0 : (warp - 2) >> 2;   // which half of the Cout columns
    group = G2 ? (warp - 2) >> 2 : 0;  // which of the two strips in flight
    prow = 2 * q + (lane >> 4);
    pcol = lane & 15;
    first_col = pcol == 0;
    last_col = pcol == 15;
    src_l = (lane & 16) | ((lane + 15) & 15);
    src_r = (lane & 16) | ((lane + 1) & 15);
    col_w = half * Cfg::kWarpCols;
    const int ew = warp - 2;
    mail = ptx::smem_u32(mail_s + ew * Cfg::kWarpMailBytes) + uint32_t((lane >> 4) * Cfg::kWarpCols * 4);
    out_tile = out_s + ew * 2 * Cfg::kWarpOutBytes;
    par = 0;
#pragma unroll
    for (int i = 0; i < Cfg::kWarpCols; ++i) {
      bias[i] = bias_s[col_w + i];
      csum[i] = 0.f;
    }
  }
  // mailbox slot: kind 0 = D_0 of column 15, kind 1 = unfinished column 15
  __device__ __forceinline__ uint32_t slot(int parity, int kind) const {
    return mail + uint32_t((parity * 2 + kind) * 2 * Cfg::kWarpCols * 4);
  }
};

// Epilogue of one tile for one warp.  Reads this warp's columns of the three partial sums, forms
// out[c] = D_0[c-1] + D_1[c] + D_2[c+1] with two shuffles per value (tile-boundary terms through the mailbox),
// releases the accumulator, applies the fused arithmetic and stores (TMA store through the warp's staging tile, or
// directly when `direct`).  Lanes 0..14 own columns 16*tx + lane of the current tile, lane 15 the previous
// tile's column 15.
//   tx          tile column inside the strip (0: no left neighbour; the mailbox is not read)
//   pre         pre-tile: only the carry is produced
//   has_pend    lane 15 holds an unfinished column from the previous tile of this CTA
//   PAIR        `tempty` is the LEADER CTA's barrier: released through its shared::cluster address
template <int KC, int NT, bool PAIR = false, bool G2 = false>
__device__ __forceinline__ void dx_epilogue_tile(DxEpiWarp<KC, NT, G2>& w, const ConvEpilogue& epi,
                                                 const CUtensorMap* tmap_out, uint32_t t_addr, uint64_t* tempty, int b,
                                                 int ty, int tx, int tiles_x, bool pre, bool has_pend, bool direct, int H,
                                                 int W, const uint8_t* const* side_tiles = nullptr) {
  using Cfg = DxCfg<KC, NT, G2>;
  const int y = ty * kDxTileH + w.prow;
  const int x = w.last_col ? tx * kDxTileW - 1 : tx * kDxTileW + w.pcol;
  const bool valid = (y < H) && (w.last_col ? has_pend : (!pre && x < W));
  const bool strip_end = (tx == tiles_x - 1) && !pre;
  const bool use_tma = !direct && !pre && tx > 0;
  uint8_t* stage = w.out_tile + w.par * Cfg::kWarpOutBytes;
  XMM_EPI_T0();
  if (use_tma) {  // the TMA store issued two tiles ago has finished reading this staging tile
    if (ptx::elect_one()) ptx::bulk_wait_read<1>();
    __syncwarp();
  }
  XMM_EPI_ADD(w, 0);
#pragma unroll
  for (int cc = 0; cc < Cfg::kWarpChunks; ++cc) {
    uint32_t d0[16], d1[16], d2[16];
    const uint32_t ta = t_addr + uint32_t(w.col_w + cc * 16);
    ptx::tmem_ld_32x16(ta, d0);
    ptx::tmem_ld_32x16(ta + uint32_t(NT), d1);
    ptx::tmem_ld_32x16(ta + uint32_t(2 * NT), d2);
    ptx::tmem_ld_wait();
    if (cc == Cfg::kWarpChunks - 1) {
      ptx::tc_fence_before();
      __syncwarp();
      if (w.lane == 0) {
        if (PAIR)
          ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(tempty), 0));
        else
          ptx::mbar_arrive(tempty);
      }
    }
    XMM_EPI_ADD(w, 1);
    const uint32_t a_w = w.slot(w.par, 0) + uint32_t(cc * 64), a_r = w.slot(w.par ^ 1, 0) + uint32_t(cc * 64);
    const uint32_t b_w = w.slot(w.par, 1) + uint32_t(cc * 64), b_r = w.slot(w.par ^ 1, 1) + uint32_t(cc * 64);
    // lane 15 publishes D_0[15] for the next tile's lane 0
#pragma unroll
    for (int j = 0; j < 4; ++j)
      sts4_if(w.last_col, __uint_as_float(d0[4 * j]), __uint_as_float(d0[4 * j + 1]), __uint_as_float(d0[4 * j + 2]),
              __uint_as_float(d0[4 * j + 3]), a_w + uint32_t(j * 16));
    float left[16], right[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
#ifdef XMM_EXP_NOSHFL
      left[i] = __uint_as_float(d0[i]);
      right[i] = __uint_as_float(d2[i]);
#else
      left[i] = __shfl_sync(0xffffffffu, __uint_as_float(d0[i]), w.src_l);
      right[i] = __shfl_sync(0xffffffffu, __uint_as_float(d2[i]), w.src_r);
#endif
    }
    // lane 0: its left neighbour is the previous tile's column 15 (strip start: the zero padding)
    if (tx == 0) {
#pragma unroll
      for (int i = 0; i < 16; ++i) left[i] = w.first_col ? 0.f : left[i];
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        lds4_if(w.first_col, left[4 * j], left[4 * j + 1], left[4 * j + 2], left[4 * j + 3], a_r + uint32_t(j * 16));
    }
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = left[i] + (__uint_as_float(d1[i]) + w.bias[cc * 16 + i]);
    // lane 15: park D_0[14] + D_1[15] (+ bias) of this tile, take over the previous tile's parked column
#pragma unroll
    for (int j = 0; j < 4; ++j) sts4_if(w.last_col, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3], b_w + uint32_t(j * 16));
#pragma unroll
    for (int j = 0; j < 4; ++j) lds4_if(w.last_col, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3], b_r + uint32_t(j * 16));
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += right[i];
    XMM_EPI_ADD(w, 2);
    const int col = w.col_w + cc * 16;
    if (valid) {
      if (use_tma) {
        StagedSides st;
        const int ps = w.prow * kDxTileW + ((w.pcol + 1) & 15);  // this lane's pixel inside the CTA-wide side tile
        st.base[0] = side_tiles ? side_tiles[0] : nullptr;
        st.base[1] = side_tiles ? side_tiles[1] : nullptr;
        st.base[2] = side_tiles ? side_tiles[2] : nullptr;
        st.row_off = uint32_t(ps * NT * 2);
        st.chunk0 = uint32_t(col / 8);
        st.xor_mask = NT == 32 ? uint32_t((ps >> 1) & 3) : uint32_t(ps & 7);
        conv_epilogue_math<NT, 16>(epi, nullptr, v, col, b, y, x, H, W, side_tiles ? &st : nullptr);
        if (epi.colsum != nullptr) {
#pragma unroll
          for (int i = 0; i < 16; ++i) w.csum[cc * 16 + i] += v[i];
        }
        const int p = (w.lane >> 4) * kDxTileW + ((w.pcol + 1) & 15);  // box pixel: lane 15 is the box's column 0
        *reinterpret_cast<uint4*>(stage + dx_out_offset<Cfg::kWarpCols>(p, cc * 2)) = pack8(v);
        *reinterpret_cast<uint4*>(stage + dx_out_offset<Cfg::kWarpCols>(p, cc * 2 + 1)) = pack8(v + 8);
      } else {
        conv_epilogue_cols<NT, 16>(epi, nullptr, v, col, b, y, x, H, W, epi.colsum != nullptr ? &w.csum[cc * 16] : nullptr);
      }
    }
    XMM_EPI_ADD(w, 3);
    // End of the strip: column 15 of the last tile has no right neighbour (D_2[W] = 0).
    if (strip_end && w.last_col && y < H && tx * kDxTileW + 15 < W) {
      float f[16];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 t4 = *reinterpret_cast<const float4*>(__cvta_shared_to_generic(size_t(b_w) + size_t(j * 16)));
        f[4 * j] = t4.x; f[4 * j + 1] = t4.y; f[4 * j + 2] = t4.z; f[4 * j + 3] = t4.w;
      }
      conv_epilogue_cols<NT, 16>(epi, nullptr, f, col, b, y, tx * kDxTileW + 15, H, W,
                                 epi.colsum != nullptr ? &w.csum[cc * 16] : nullptr);
    }
  }
  if (use_tma) {
    ptx::fence_proxy_async();  // this thread's st.shared -> visible to the async proxy
    __syncwarp();
    if (ptx::elect_one()) {
      ptx::tma_store_4d(tmap_out, stage, epi.out_coff + w.col_w, tx * kDxTileW - 1, ty * kDxTileH + 2 * w.q, b);
      ptx::bulk_commit();
    }
  }
  XMM_EPI_ADD(w, 4);
  w.par ^= 1;
}

// This CTA's tiles as RUNS of consecutive tiles of the strip-major order.
//   round-robin part: while a full round of gridDim.x strips is left, run r = strip blockIdx.x + r * gridDim.x;
//   tail: the tiles that are left (all of them for small problems) are cut into gridDim.x equal contiguous ranges; a
//         range that starts mid-strip begins one tile early with a "pre-tile" (outputs suppressed, carry established).
// (With whole strips only, 832 strips on 148 CTAs -- batch 16 -- make 92 CTAs walk 6 strips and 56 walk 5.)
// CTA pairs run in lock step and keep whole strips: both CTAs take the leader's count, a missing strip is a dummy.
struct DxRuns {
  int rr_runs, nruns;
  int rr_r0, rr_step, rr_len;      // round-robin runs
  int tail_g0, tail_t0, tail_len;  // tail run (tail_len > 0)
  int dummy_from;                  // pair mode: runs >= dummy_from repeat run 0 with nothing stored
  template <bool PAIR>
  __device__ __forceinline__ void init(const ConvArgs& args) {
    const int grid = int(gridDim.x), b = int(blockIdx.x);
    const int nstrips = args.num_tiles / args.tiles_x;
    rr_step = grid * args.tiles_x;
    rr_len = args.tiles_x;
    rr_r0 = b * args.tiles_x;
    tail_len = 0;
    tail_g0 = tail_t0 = 0;
    if (PAIR) {
      const int lead = b & ~1;
      rr_runs = nstrips > lead ? (nstrips - lead + grid - 1) / grid : 0;
      dummy_from = nstrips > b ? (nstrips - b + grid - 1) / grid : 0;
      nruns = rr_runs;
      return;
    }
    rr_runs = args.strip_rr ? nstrips / grid : 0;
    dummy_from = 1 << 30;
    const long long done = (long long)rr_runs * rr_step;
    const long long rem = (long long)args.num_tiles - done;
    const int t0 = int(done + rem * b / grid), t1 = int(done + rem * (b + 1) / grid);
    if (t1 > t0) {
      tail_t0 = t0;
      tail_g0 = (t0 % args.tiles_x != 0) ? t0 - 1 : t0;
      tail_len = t1 - tail_g0;
    }
    nruns = rr_runs + (tail_len > 0 ? 1 : 0);
  }
  // run -> first tile, tile count, first tile whose outputs are stored (tiles before it are pre-tiles), dummy?
  __device__ __forceinline__ void get(int run, int& r0, int& len, int& tvalid, bool& dummy) const {
    dummy = run >= dummy_from;
    if (run < rr_runs) {
      r0 = dummy ? rr_r0 : rr_r0 + run * rr_step;
      len = rr_len;
      tvalid = r0;
    } else {
      r0 = tail_g0;
      len = tail_len;
      tvalid = tail_t0;
    }
  }
  __device__ __forceinline__ int total_tiles() const { return rr_runs * rr_len + tail_len; }
};

// Tensor maps of the side inputs (mask, r1, r2) that are staged through shared memory (ConvArgs::side_mask).
struct DxSideMaps {
  CUtensorMap m[3];
};

template <int KC, int NT, bool PAIR = false, bool G2 = false>
__global__ void __launch_bounds__(kDxThreads, 1)
conv3x3_dx_kernel(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_out,
                  const __grid_constant__ DxSideMaps side_maps, const ConvArgs args) {
  using Cfg = DxCfg<KC, NT, G2>;
  static_assert(!(PAIR && G2), "CTA pairs and epilogue groups are separate experiments");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w_s = smem;
  float* bias_s = reinterpret_cast<float*>(smem + args.w_bytes);
  uint8_t* stage_s = smem + ((args.w_bytes + Cfg::kBiasBytes + 1023) & ~1023u);
  uint8_t* out_s = stage_s + size_t(args.stages) * Cfg::kStageBytes;  // per-warp staging tiles for the TMA stores
  uint8_t* mail_s = out_s + Cfg::kOutBytes;
  const int nside = __popc(args.side_mask);
  uint8_t* side_s = mail_s + Cfg::kMailBytes;  // [2 buffers][nside] side-input tiles (1 KB aligned)
  uint64_t* bars = reinterpret_cast<uint64_t*>(side_s + size_t(2 * nside) * Cfg::kSideTileBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kMaxStages;
  uint64_t* tfull_bar = bars + 2 * kMaxStages;
  uint64_t* tempty_bar = tfull_bar + 4;
  uint64_t* w_bar = tempty_bar + 4;
  uint64_t* sfull_bar = w_bar + 1;   // [2]
  uint64_t* sempty_bar = sfull_bar + 2;  // [2]
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(sempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
#ifdef XMM_CONV_PROFILE
  long long prof_t0_ = 0;
  long long prof_acc_[6] = {0, 0, 0, 0, 0, 0};
  const long long prof_k0_ = clock64();
  unsigned long long prof_g0_;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(prof_g0_));
#endif

  const uint32_t pair_rank = PAIR ? ptx::cluster_ctarank() : 0u;
  const bool leader = pair_rank == 0;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_in);
    ptx::prefetch_tmap(&tmap_out);
    for (int s = 0; s < args.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < Cfg::kAccStages; ++a) {
      ptx::mbar_init(&tfull_bar[a], 1);
      ptx::mbar_init(&tempty_bar[a], PAIR ? 2 * kDxEpiWarps : Cfg::kTileWarps);
    }
    ptx::mbar_init(w_bar, 1);
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&sfull_bar[a], 1);
      ptx::mbar_init(&sempty_bar[a], Cfg::kTileWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    if (PAIR)
      ptx::tmem_alloc_pair<Cfg::kTmemCols>(tmem_ptr_s);
    else
      ptx::tmem_alloc<Cfg::kTmemCols>(tmem_ptr_s);
  }
  ptx::tc_fence_before();
  if (PAIR)
    ptx::cluster_sync();  // the peer's barriers are initialised before anything arrives on them
  else
    __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;

  DxRuns runs{};
  runs.template init<PAIR>(args);
  // Issue order.  A UNIT is one run -- or, with two epilogue groups, two consecutive round-robin runs (strips) whose
  // tiles alternate A0 B0 A1 B1 ...: group 0 takes A, group 1 takes B.  The tail run is never paired.
  const int npairs = G2 ? runs.rr_runs / 2 : 0;
  const int nunits = runs.nruns - npairs;
  // tile counter c -> accumulator stage c % kAccStages, side-tile counter sc -> buffer sc & 1

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (ptx::elect_one()) {
      const uint8_t* gsrc = static_cast<const uint8_t*>(args.wblob);
      if (PAIR && !leader) {
        // the peer supplies rows [3*NT/2, 3*NT) of every (chunk, filter row) group: load the image half a group early
        constexpr uint32_t kShift = uint32_t(3 * NT / 2) * Cfg::kRowB;
        const uint32_t wpart = args.w_bytes - kShift;
        ptx::mbar_expect_tx(w_bar, wpart + Cfg::kBiasBytes);
        for (uint32_t off = 0; off < wpart; off += 32768u) {
          const uint32_t n = (wpart - off < 32768u) ? (wpart - off) : 32768u;
          ptx::bulk_load(w_s + off, gsrc + kShift + off, n, w_bar);
        }
        ptx::bulk_load(w_s + args.w_bytes, gsrc + args.w_bytes, Cfg::kBiasBytes, w_bar);
        ptx::mbar_wait(w_bar, 0);  // the leader's MMAs read these weights once this CTA's first stage has landed
      } else {
        const uint32_t wtot = args.w_bytes + Cfg::kBiasBytes;
        ptx::mbar_expect_tx(w_bar, wtot);
        for (uint32_t off = 0; off < wtot; off += 32768u) {
          const uint32_t n = (wtot - off < 32768u) ? (wtot - off) : 32768u;
          ptx::bulk_load(w_s + off, gsrc + off, n, w_bar);
        }
      }
      int stage = 0;
      uint32_t phase = 0;
      int sbuf = 0;
      uint32_t sphase = 0;
      auto load_tile = [&](const DxTile& t, bool with_sides) {
        const int y0 = t.ty * kDxTileH - 1, x0 = t.tx * kDxTileW;
        for (int ch = 0; ch < args.nchunks; ++ch) {
          XMM_PROF_T0();
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1u);
          XMM_PROF_ADD(0);
          if (PAIR) {  // both CTAs' stages complete on the leader's barrier
            if (leader) ptx::mbar_expect_tx(&full_bar[stage], 2 * Cfg::kStageBytes);
            ptx::tma_load_4d_pair(stage_s + size_t(stage) * Cfg::kStageBytes, &tmap_in,
                                  ptx::mapa(ptx::smem_u32(&full_bar[stage]), 0), args.cin_off + ch * KC, x0, y0, t.b);
          } else {
            ptx::mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
            ptx::tma_load_4d(stage_s + size_t(stage) * Cfg::kStageBytes, &tmap_in, &full_bar[stage],
                             args.cin_off + ch * KC, x0, y0, t.b);
          }
          if (++stage == args.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if (with_sides) {  // the output pixels' mask / residual tiles (not for pre-tiles)
          ptx::mbar_wait(&sempty_bar[sbuf], sphase ^ 1u);
          ptx::mbar_expect_tx(&sfull_bar[sbuf], uint32_t(nside) * Cfg::kSideTileBytes);
          uint8_t* dst = side_s + size_t(sbuf * nside) * Cfg::kSideTileBytes;
          const int coff[3] = {args.epi.mask_coff, args.epi.r1_coff, args.epi.r2_coff};
#pragma unroll
          for (int k = 0; k < 3; ++k)
            if (args.side_mask & (1 << k)) {
              ptx::tma_load_4d(dst, &side_maps.m[k], &sfull_bar[sbuf], coff[k], t.tx * kDxTileW - 1, t.ty * kDxTileH,
                               t.b);
              dst += Cfg::kSideTileBytes;
            }
          if (++sbuf == 2) {
            sbuf = 0;
            sphase ^= 1u;
          }
        }
      };
      for (int u = 0; u < nunits; ++u) {
        const bool paired = u < npairs;
        const int run_a = paired ? 2 * u : u + npairs;
        int r0, run_len, t0, r0b = 0, len_b, t0b;
        bool dummy, dummy_b;
        runs.get(run_a, r0, run_len, t0, dummy);
        if (paired) runs.get(run_a + 1, r0b, len_b, t0b, dummy_b);
        DxTile t(r0, args.tiles_x, args.tiles_y), tb(r0b, args.tiles_x, args.tiles_y);
        for (int g = r0; g < r0 + run_len; ++g) {
          load_tile(t, nside > 0 && g >= t0 && !dummy);
          t.next(args.tiles_x, args.tiles_y);
          if (paired) {
            load_tile(tb, nside > 0);
            tb.next(args.tiles_x, args.tiles_y);
          }
        }
      }
      XMM_PROF_FLUSH(0);
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (leader && ptx::elect_one()) {
      ptx::mbar_wait(w_bar, 0);
      ptx::tc_fence_after();
      const uint32_t w_addr = ptx::smem_u32(w_s);
      const uint32_t st_addr = ptx::smem_u32(stage_s);
      const uint64_t bdesc0 = ptx::umma_smem_desc(w_addr, 16, 8 * Cfg::kRowB, Cfg::kLayout);
      const uint64_t adesc0 = ptx::umma_smem_desc(st_addr, 16, 8 * Cfg::kRowB, Cfg::kLayout);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      XMM_PROF_START(3);
      const int my_tiles = runs.total_tiles();
      for (int g = 0; g < my_tiles; ++g) {
        XMM_PROF_T0();
        ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
        XMM_PROF_ADD(1);
        ptx::tc_fence_after();
        const uint32_t d_addr = tmem_base + uint32_t(acc * Cfg::kAccCols);
        for (int ch = 0; ch < args.nchunks; ++ch) {
          XMM_PROF_T0();
          ptx::mbar_wait(&full_bar[stage], phase);
          XMM_PROF_ADD(2);
          ptx::tc_fence_after();
          const uint64_t adesc_st = adesc0 + uint64_t((uint32_t(stage) * Cfg::kStageBytes) >> 4);
          const uint64_t bdesc_ch = bdesc0 + uint64_t((uint32_t(ch) * 9u * Cfg::kTapBytes) >> 4);
          dx_issue_chunk<KC, NT, PAIR>(d_addr, adesc_st, bdesc_ch, ch == 0);
          if (PAIR)
            ptx::umma_commit_pair(&empty_bar[stage]);
          else
            ptx::umma_commit(&empty_bar[stage]);
          if (++stage == args.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if (PAIR)
          ptx::umma_commit_pair(&tfull_bar[acc]);
        else
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
    ptx::mbar_wait(w_bar, 0);
    DxEpiWarp<KC, NT, G2> w;
    w.init(warp, lane, bias_s, out_s, mail_s);
    const bool direct = args.epi.pixel_shuffle != 0;  // (inverse) pixel shuffle scatters: direct stores
    constexpr int kAccShift = Cfg::kAccStages == 4 ? 2 : 1;
    // one tile: c = its position in the issue order, sc = position among the tiles with side inputs
    auto process = [&](const DxTile& t, int g, int r0, int t0, bool dummy, int c, int sc) {
      const int acc = c & (Cfg::kAccStages - 1);
      const uint32_t acc_phase = uint32_t(c >> kAccShift) & 1u;
      XMM_PROF_T0();
      ptx::mbar_wait(&tfull_bar[acc], acc_phase);
      XMM_PROF_ADD(4);
      XMM_PROF_T0();
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + (uint32_t(w.q * 32) << 16) + uint32_t(acc * Cfg::kAccCols);
      const bool sides = nside > 0 && g >= t0 && !dummy;
      const int sbuf = sc & 1;
      const uint8_t* side_tiles[3] = {nullptr, nullptr, nullptr};
      if (sides) {
        ptx::mbar_wait(&sfull_bar[sbuf], uint32_t(sc >> 1) & 1u);
        const uint8_t* src = side_s + size_t(sbuf * nside) * Cfg::kSideTileBytes;
#pragma unroll
        for (int k = 0; k < 3; ++k)
          if (args.side_mask & (1 << k)) {
            // tile 0 of a strip stores (and reads its side inputs) directly: see dx_epilogue_tile
            side_tiles[k] = src;
            src += Cfg::kSideTileBytes;
          }
      }
      dx_epilogue_tile<KC, NT, PAIR, G2>(w, args.epi, &tmap_out, t_addr, &tempty_bar[acc], t.b, t.ty, t.tx, args.tiles_x,
                                         /*pre=*/g < t0 || dummy, /*has_pend=*/(t.tx > 0) && (g != r0) && !dummy,
                                         direct, args.height, args.width, sides ? side_tiles : nullptr);
      if (sides) {
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&sempty_bar[sbuf]);
      }
      XMM_PROF_ADD(5);
    };
    int c = 0, sc = 0;
    for (int u = 0; u < nunits; ++u) {
      const bool paired = u < npairs;
      const int run_a = paired ? 2 * u : u + npairs;
      int r0, run_len, t0;
      bool dummy;
      runs.get(paired ? run_a + w.group : run_a, r0, run_len, t0, dummy);
      DxTile t(r0, args.tiles_x, args.tiles_y);  // advanced incrementally: no divisions in the tile loop
      if (paired) {  // this group's strip: every second tile of the issue order
        for (int g = r0; g < r0 + run_len; ++g) {
          process(t, g, r0, t0, dummy, c + w.group, sc + w.group);
          c += 2;
          sc += nside > 0 ? 2 : 0;
          t.next(args.tiles_x, args.tiles_y);
        }
      } else {       // a single run: group 0 (group 1 only keeps count)
        for (int g = r0; g < r0 + run_len; ++g) {
          if (w.group == 0) process(t, g, r0, t0, dummy, c, sc);
          c += 1;
          sc += (nside > 0 && g >= t0 && !dummy) ? 1 : 0;
          t.next(args.tiles_x, args.tiles_y);
        }
      }
    }
    if (ptx::elect_one()) ptx::bulk_wait<0>();  // this warp's stores complete before the CTA (and its smem) goes away
    if constexpr (NT == 32)  // (column sums are for cout = 32: xmm_conv3x3_bf16 rejects them elsewhere)
      if (args.epi.colsum != nullptr) colsum_flush<Cfg::kWarpCols>(args.epi, w.csum, w.col_w, lane);
    if (warp == 2 && lane == 0) { XMM_PROF_FLUSH(4); XMM_PROF_FLUSH(5); }
#ifdef XMM_CONV_PROFILE
    if (warp == 2 && lane == 0)
      for (int i = 0; i < 8; ++i) args.prof[size_t(148 + blockIdx.x) * 8 + i] = w.phase[i];
#endif
  }

  ptx::tc_fence_before();
  if (PAIR)
    ptx::cluster_sync();  // neither CTA's shared memory / TMEM may go away while the other still uses it
  else
    __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    if (PAIR)
      ptx::tmem_dealloc_pair<Cfg::kTmemCols>(tmem_base);
    else
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
