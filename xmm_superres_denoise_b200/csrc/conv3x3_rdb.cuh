// Fused dense-block convolutions: conv1..conv3 (or conv4..conv5) of one ResidualDenseBlock_5C.forward
// (rrdb_blocks.py:37-54) in ONE kernel, the intermediate feature maps handed from layer to layer through shared memory.
//
// Why.  Layer by layer a dense block moves 1280 B per pixel through HBM (conv_k re-reads x0..x_{k-1}) for 135*F^2 MAC:
// at batch 64 that is 2.2 ms of pure HBM time per block against 1.8 ms of tensor time, and every per-layer kernel of
// round 1 / the row-hop kernel sits on that wall (3.75-4.6 TB/s whatever Cin, tools/row_probe.py).  Fusing 1-2-3 and
// 4-5 leaves 64 + 192 B (read x0, write x1..x3) and 256 + 64 B (read x0..x3, write the block output): 576 B per pixel,
// and the kernel becomes tensor-bound.
//
// Form.  The row-hop form of conv3x3_row.cuh (the three dy taps are the N = 96 columns of one MMA and land in the
// accumulators of output rows r-1, r, r+1), on a tile that makes halo recompute cheap: M = 128 lanes = one image row of
// TWO horizontal bands x 63 pixels.  In shared memory a row tile is 130 consecutive 64-byte pixel positions
//     [halo | 63 px of band 0 | halo][halo | 63 px of band 1 | halo]
// written by one 5-D TMA box (c, 65 px, 1 row, 2 bands); the dx taps are descriptor views one position apart, lane i
// is centred on position i + 1 (lanes 63 / 64 are centred on the two inner halo positions and compute nothing useful).
// A CTA walks a 63-pixel column of both bands top to bottom.  Layer l+1 consumes the rows layer l produced two steps
// earlier: the epilogue writes them as bf16 into a ring of row tiles with the same swizzled layout a TMA load would
// have produced, so they are MMA A operands as they are -- they never leave the SM unless a later kernel needs them
// (then the epilogue also stores the lanes this tile owns).
//
// Halo recompute instead of halo exchange: with NL fused layers the lanes within NL-1-l pixels of a tile edge that
// is not an image edge are wrong after layer l (their neighbours belong to another tile), so tile t+1 starts
// 2*(NL-1) pixels before tile t ends and each tile stores only the pixels it owns (416 px = 7 tiles: 61 + 5*59 + 61
// for three layers, 93 % of the lanes useful).  The same in y: a piece of rows [ra, rb) computes layer l on
// [ra-e, rb+e), e = NL-1-l, from input rows of the neighbouring piece / band (recomputed, not stored).  Rows and
// pixels outside the image are ZERO in every intermediate map (Conv2d's padding is per layer), so the epilogue
// writes zeros there.
//
// Accumulators.  Layer l owns 5 TMEM slots of 32 columns.  The step on input row r targets the window
// (c, c+1, c+2), c = (r-1) mod 3, i.e. slots are a function of the ROW INDEX, not of a running counter: the result
// does not depend on how the work is split (batch invariance is bit-exact).  A row whose window position is 0 or 1
// collected its first partial sums in slots 3 / 4 (the window slid over the ring end); the epilogue adds the two
// slots.  Every MMA accumulates: the epilogue zeroes a slot after draining it, and the issuer starts the step on
// row r only after row r-2 has been drained (one barrier pair per layer, strictly alternating).
//
// Schedule and roles (512 threads).  One deterministic walk (rdb_walk) interleaves the layers -- L0 step, L1 step,
// L2 step, L0 step ...; layer l takes its step on row r when layer l-1 took its step on row r+1 in an EARLIER round;
// after the last row of a piece a layer takes two flush steps (no MMAs) that complete and re-initialise the two
// trailing partial rows.  Only the TMA producer (warp 0) follows the walk: it decides the order in which rows are
// loaded into the ONE stage ring all layers share (the stage id travels next to a per-layer "landed" barrier ring).
// Layer l's MMA issuer (one thread of warp 1 + l) and its epilogue group (warps 4 + 4 l .. 7 + 4 l, one per TMEM lane
// quarter) iterate their own layer only -- pieces in order, rows top to bottom -- and meet the other roles through
// mbarriers.  Rule for every barrier here: its waiter observes EVERY phase (a parity wait two phases ahead passes at
// once) -- hence per-layer barriers and per-layer roles; tools/rdb_protocol_sim.py models the whole protocol.
//
// CTA pairs (template PAIR; both kernels).  Single CTAs hold all the weights (164 KB for conv4 + conv5, 111 KB for
// conv1..conv3), which leaves five TMA stages, and the issuers wait for chunks to land.  Two CTAs of a cluster run as
// a tcgen05 cta_group::2 pair: the leader's issuers issue M = 256 MMAs (rows 0..127 = the leader's row tile,
// 128..255 = the peer's) and each CTA holds a compacted HALF of every (chunk, dx) group of the weight image (rank 0
// rows 0..47, rank 1 rows 48..95, 3 KB per group).  Each CTA keeps its own producer, stage ring, map rings, epilogue
// groups and TMEM lanes, and walks its own column of the same pair-column (RdbSched<NL, true>): both CTAs take the
// same walk over the same stage count, so the stage and ring-slot ids are the same in both and the leader's
// descriptors address both.  Both producers' loads complete on the leader's full barriers; the peer's epilogue warps
// arrive on the leader's `tdrain` / `mfull` (count 8); the leader's commits (`empty`, `mempty`, `tfull`) are
// multicast to both CTAs.
//   conv4 + conv5 (G = 4): 14 stages of the shared walk-order ring fit.
//   conv1..conv3 (G = 1, the x0 ring, kRdbXRing): every input chunk is an x0 row, and the walk-order ring loads each
// of them three times (once per layer).  The pair instead loads each x0 row of a piece ONCE, in row order, into a ring
// of 11 row tiles that all three issuers read the way they read map rows: the slot comes from the row's sequence
// number, `lfull[slot]` is the TMA transaction barrier and `empty[slot]` is released by the commit of the last layer
// that reads the row (conv3 for [ra-1, rb], conv2 for ra-2 and rb+1, conv1 for ra-3 and rb+2).  For that release to
// come after the earlier layers' reads, the first step of a piece of conv2 / conv3 waits for its map rows before it
// reads x0.  The issuers that skip a piece's edge rows skip phases of their slots; tools/rdb_protocol_sim.py checks
// that no wait can land in the wrong phase.  The K order of every layer (x0 first, then its maps) is that of the
// single CTA, so the bits are the same.
#pragma once
#include <cstdio>

#include "conv3x3_tc.cuh"

namespace xmm {

constexpr int kRdbP = 63;                         // pixels of one band segment (lanes per band, minus the junk lane)
constexpr int kRdbBoxPx = kRdbP + 2;              // segment + both halo pixels
constexpr int kRdbTileData = 2 * kRdbBoxPx * 64;  // bytes one TMA box writes (32 bf16 channels per pixel)
constexpr int kRdbTileBytes = 17 * 512;           // tile pitch: whole SWIZZLE_64B atoms
constexpr int kRdbThreads = 512;                  // producer warp, one issuer warp + four epilogue warps per layer (<= 3)
constexpr int kRdbSlots = 5;                      // accumulator slots per layer
constexpr int kRdbSlotCols = kRdbSlots * 32;
constexpr int kRdbMaxRing = 8;
constexpr int kRdbMaxStages = 16;
// Length of the per-layer landed rings (lfull / lstage) = capacity of the stage ring.  Issuer l waits on slot
// k = chunk mod kRdbLRing; the producer is at most `stages` chunks ahead of the last chunk consumed, so with
// stages <= kRdbLRing no parity wait can pass a phase early.  A single CTA fits <= 8 stages next to its weights.
template <bool PAIR>
constexpr int kRdbLRing = PAIR ? kRdbMaxStages : 8;
// conv1..conv3 as a CTA pair: the stage ring is the x0 row ring (see the top of this file), `lfull` / `empty` are its
// [stages] full / empty barriers and there is no `lstage`.
template <int G, bool PAIR>
constexpr bool kRdbXRing = PAIR && G == 1;
constexpr int kRdbTapBytes = 32 * 64;             // one (dx, dy) block of a chunk: 32 output channels x 32 inputs
constexpr int kRdbGroupBytes = 3 * kRdbTapBytes;  // one (chunk, dx) group of the row-hop image: 96 rows of 64 B
constexpr int kRdbProfSlots = 24;                 // XMM_RDB_PROFILE counters per CTA

struct RdbLayerArgs {
  const void* wblob;   // row-hop order [chunk][dx][2 - dy][32][32] bf16 (SWIZZLE_64B applied) + 32 fp32 biases
  uint32_t w_bytes;    // of the image in shared memory, without the biases (CTA pair: half of the blob's)
  uint32_t smem_off;   // where this layer's image starts in the weight region (1024-aligned)
  float lrelu_slope;   // 1 = none
  int store;           // the output is needed outside the kernel
  __nv_bfloat16* out;
  int out_ctot, out_coff;
};

struct RdbArgs {
  RdbLayerArgs layer[3];
  int cin_off;                 // channel of x0 in the input buffer (x_j at cin_off + 32 j)
  int batch, height, width, band_h, tiles_x;
  long long total_rows;        // batch * tiles_x * band_h (rows of all columns; CTA pairs: of all pair-columns)
  int stages, ring0, ring1;    // TMA stages; row tiles of the first / second in-CTA map
  uint32_t w_total;            // bytes of the weight region
  // residuals of the LAST layer (conv5: out = s0 * v + s1 * r1 + s2 * r2, rrdb_blocks.py:54,70)
  float s0, s1, s2;
  const __nv_bfloat16* r1;
  int r1_ctot, r1_coff;
  const __nv_bfloat16* r2;
  int r2_ctot, r2_coff;
  int backoff_ns;   // nanosleep between polls of the producer / epilogue waits (0: none)
  int prefetch_rows;  // the producer asks L2 for the global maps of the row this many steps ahead (0: off)
  int split_producers;  // two fused layers: one TMA producer thread and stage-ring slice per layer
  long long* prof;  // optional (XMM_RDB_PROF=1): kRdbProfSlots cycle counters per CTA, see launch_rdb
};

template <int NL>
__host__ __device__ inline int rdb_tile_origin(int t) {  // first owned pixel of tile t
  return t == 0 ? 0 : (kRdbP - (NL - 1)) + (t - 1) * (kRdbP - 2 * (NL - 1));
}
template <int NL>
__host__ __device__ inline int rdb_tiles_x(int width) {
  int n = 1;
  while ((n == 1 ? 0 : rdb_tile_origin<NL>(n - 1) - (NL - 1)) + kRdbP < width) ++n;
  return n;
}

struct RdbPiece {
  int b, x0;            // image, pixel of lane 0 of each band
  int own_lo, own_hi;   // pixels this tile stores
  int ra, rb;           // rows (band-local) this piece stores
};

// The CTA's share of the work: the rows of all (image, tile) columns, in column order, cut into gridDim.x equal
// contiguous ranges; a range touches a few columns = pieces.
// PAIR: pair-column p is column 2p on cluster rank 0 and 2p + 1 on rank 1; the rows of the pair-columns are cut into
// gridDim.x / 2 ranges, so both CTAs of a pair take the same pieces, rows and flush steps (the same walk) and differ
// only in b, x0 and the owned pixels.  With an odd column count rank 1's last column is a phantom: it repeats the
// last real column (in-bounds loads) and owns no pixel, so it stores nothing.
template <int NL, bool PAIR = false>
struct RdbSched {
  int band_h, tiles_x, width, c0, npieces;
  int ncols, rank;  // PAIR: columns, cluster rank
  long long t0, t1;
  __device__ __forceinline__ void init(const RdbArgs& a) {
    band_h = a.band_h;
    tiles_x = a.tiles_x;
    width = a.width;
    if (PAIR) {
      ncols = a.batch * a.tiles_x;
      rank = int(ptx::cluster_ctarank());
      const long long unit = blockIdx.x >> 1, nunits = gridDim.x >> 1;
      t0 = a.total_rows * unit / nunits;
      t1 = a.total_rows * (unit + 1) / nunits;
    } else {
      t0 = a.total_rows * blockIdx.x / gridDim.x;
      t1 = a.total_rows * (blockIdx.x + 1) / gridDim.x;
    }
    c0 = int(t0 / band_h);
    npieces = t1 > t0 ? int((t1 - 1) / band_h) - c0 + 1 : 0;
  }
  __device__ __forceinline__ RdbPiece get(int i) const {
    RdbPiece p;
    int col = c0 + i;
    const long long base = (long long)col * band_h;
    p.ra = t0 > base ? int(t0 - base) : 0;
    p.rb = t1 < base + band_h ? int(t1 - base) : band_h;
    bool phantom = false;
    if (PAIR) {
      col = 2 * col + rank;
      phantom = col >= ncols;
      if (phantom) col = ncols - 1;
    }
    p.b = col / tiles_x;
    const int t = col - p.b * tiles_x;
    p.own_lo = rdb_tile_origin<NL>(t);
    p.x0 = t == 0 ? 0 : p.own_lo - (NL - 1);
    p.own_hi = phantom ? p.own_lo : t == tiles_x - 1 ? width : rdb_tile_origin<NL>(t + 1);
    return p;
  }
};

// The step sequence.  f(l, piece, r, flush, n, seq): layer l takes its step on input row r of `piece` (flush: one of
// the two MMA-less steps after the piece's last row); n = how many steps layer l took before; seq[m] = sequence
// number, among all rows of in-CTA map m, of the piece's first row ra - (NL-1-m).
template <int NL, class S, class F>
__device__ __forceinline__ void rdb_walk(const S& s, F&& f) {
  int piece[NL], r[NL], hi[NL], n[NL], seq[NL][NL];
  RdbPiece pc[NL];
  bool done[NL];
#pragma unroll
  for (int l = 0; l < NL; ++l) {
    piece[l] = 0;
    n[l] = 0;
    done[l] = s.npieces == 0;
#pragma unroll
    for (int m = 0; m < NL; ++m) seq[l][m] = 0;
    pc[l] = s.get(0);
    r[l] = pc[l].ra - (NL - 1 - l) - 1;
    hi[l] = pc[l].rb + (NL - 1 - l) + 2;
  }
  while (!done[NL - 1]) {
    // Which layers step in this round, decided on the state at the START of the round: layer l steps when layer l-1
    // took its step on row r+1 in an earlier round.  Steady state (the bulk of the walk): every layer is inside the
    // same piece, two rows behind the layer before it, so all of them step once per round until the first one runs
    // out of real rows -- `reps` rounds without a decision.
    uint32_t go = done[0] ? 0u : 1u;
    bool steady = !done[0];
    int reps = pc[0].rb + (NL - 1) - r[0] + 1;  // real steps layer 0 has left in this piece
#pragma unroll
    for (int l = 1; l < NL; ++l) {
      const bool ready = !done[l] && (done[l - 1] || piece[l - 1] > piece[l] || (piece[l - 1] == piece[l] && r[l - 1] > r[l] + 1));
      go |= ready ? (1u << l) : 0u;
      steady = steady && ready && piece[l] == piece[0];
      const int kl = pc[l].rb + (NL - 1 - l) - r[l] + 1;
      reps = kl < reps ? kl : reps;
    }
    if (!steady || reps < 1) reps = 1;
    for (int i = 0; i < reps; ++i) {
#pragma unroll
      for (int l = 0; l < NL; ++l) {
        if ((go >> l) & 1u) {
          const int e = NL - 1 - l;
          f(l, pc[l], r[l], r[l] > pc[l].rb + e, n[l], seq[l]);
          ++n[l];
          if (++r[l] > hi[l]) {
#pragma unroll
            for (int m = 0; m < NL; ++m) seq[l][m] += (pc[l].rb - pc[l].ra) + 2 * (NL - 1 - m);
            if (++piece[l] >= s.npieces) {
              done[l] = true;
            } else {
              pc[l] = s.get(piece[l]);
              r[l] = pc[l].ra - e - 1;
              hi[l] = pc[l].rb + e + 2;
            }
          }
        }
      }
    }
  }
}

// mbarrier wait with a watchdog: a wait that spins for ~seconds reports who waits for what and traps (a wedged
// schedule must fail loudly instead of hanging the process).
__device__ __noinline__ void rdb_wait_timeout(int tag, int a, int b2, int c) {
  printf("conv3x3_rdb: CTA %d thread %d stuck in wait %d (layer/map %d, index %d, parity %d)\n", int(blockIdx.x),
         int(threadIdx.x), tag, a, b2, c);
  __trap();
}
__device__ __forceinline__ void rdb_wait(uint64_t* bar, uint32_t parity, int tag, int a, int b2) {
  uint32_t spins = 0;
  while (!ptx::mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) rdb_wait_timeout(tag, a, b2, int(parity));
  }
}

// for the warps that are not on the critical path of the tensor pipe (producer, epilogue): back off between polls so
// that the polling itself (a shared-memory access per try_wait, an issue slot per loop turn) does not compete with
// the MMA operand reads and the working warps of the same scheduler
__device__ __forceinline__ void rdb_wait_backoff(uint64_t* bar, uint32_t parity, int tag, int a, int b2, uint32_t ns) {
  uint32_t spins = 0;
  while (!ptx::mbar_try_wait(bar, parity)) {
    if (ns) __nanosleep(ns);
    if (++spins > (1u << 24)) rdb_wait_timeout(tag, a, b2, int(parity));
  }
}
// the same, adding the cycles spent waiting to `acc` when profiling
#ifndef XMM_RDB_PROFILE
#define XMM_RDB_PROFILE 0  // 1: cycle counters of the issuer (XMM_RDB_PROF=1 prints them per launch)
#endif
__device__ __forceinline__ void rdb_wait_p(uint64_t* bar, uint32_t parity, int tag, int a, int b2, bool prof, long long& acc) {
  if (XMM_RDB_PROFILE && prof) {
    const long long t0 = clock64();
    rdb_wait(bar, parity, tag, a, b2);
    acc += clock64() - t0;
  } else {
    rdb_wait(bar, parity, tag, a, b2);
  }
}

__device__ __forceinline__ int rdb_phi(int row) { return (row + 30) % 3; }  // window position of a row (row >= -30)

__device__ __forceinline__ void tmem_st_zero32(uint32_t taddr) {
  const uint32_t z = 0;
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
      "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr),
      "r"(z)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns <- 32 registers per thread
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
      "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
      "r"(r[31])
      : "memory");
}
// 32-byte global accesses (LDG.256 / STG.256 on sm_100): a lane's 64-byte pixel row in two instructions
__device__ __forceinline__ void st_global_256(void* p, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w),
               "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}
__device__ __forceinline__ void ld_global_nc_256(const void* p, uint4& a, uint4& b) {
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
               : "l"(p));
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Shared-memory carve-up, identical in every thread.
struct RdbCtx {
  uint8_t* w_s;        // weights + biases of every layer
  uint8_t* stage_s;    // TMA stages (one ring shared by all layers, handed out in walk order; x0 ring: in row order)
  uint8_t* map_s[2];   // row tiles of the in-CTA maps
  uint64_t* lfull;     // [3][R] chunk k (mod R = kRdbLRing) of layer l has landed (waiter: issuer l)
                       // (x0 ring: [R] the row in slot s has landed                (waiters: all issuers))
  uint64_t* empty;     // [stages] the MMAs that read the stage are done        (waiter: producer)
                       // (x0 ring: ... the row's last reader is done)
  uint64_t* tfull;     // [NL] the row a step completes is in TMEM              (waiter: epilogue group l)
  uint64_t* tdrain;    // [NL] ... has been drained and its slot re-initialised (waiter: issuer l)
  uint64_t* mfull;     // [2][8] row tile of map m written                       (waiters: issuers m+1 ..)
  uint64_t* mempty;    // [2][8] ... read by its last reader                     (waiter: epilogue group m)
  uint64_t* w_bar;
  volatile int* lstage;  // [3][R] which stage holds chunk k (mod R) of layer l (written by the producer)
  uint32_t tmem_base;
};

// ---------------------------------------------------------------------------------------------------- MMA issuer
// One thread per layer: the bookkeeping of one layer's step (~60 instructions of a single thread) overlaps the MMAs
// of the other layers.  The thread walks its OWN layer only: pieces in order, rows top to bottom.
// PAIR: runs in the leader only and issues for both CTAs; its commits reach both.
template <int G, int NL, int L, bool PAIR>
__device__ __forceinline__ void rdb_issuer(const RdbArgs& args, const RdbCtx& c, const RdbSched<NL, PAIR>& sched) {
  constexpr int NM = NL - 1;
  constexpr int e = NL - 1 - L;
  constexpr int ring[2] = {NL == 3 ? 5 : 2, 3};
  constexpr uint32_t kR = kRdbLRing<PAIR>;
  rdb_wait(c.w_bar, 0, 7, L, 0);
  ptx::tc_fence_after();
  const uint64_t bdesc0 = ptx::umma_smem_desc(ptx::smem_u32(c.w_s), 16, 512, ptx::UMMA_SW64);
  const uint64_t adesc0 = ptx::umma_smem_desc(ptx::smem_u32(c.stage_s), 16, 512, ptx::UMMA_SW64);
  const uint32_t a_hi = uint32_t(adesc0 >> 32), b_hi = uint32_t(bdesc0 >> 32);
  const uint32_t a_lo0 = uint32_t(adesc0);
  const uint32_t b_l = uint32_t(bdesc0) + (args.layer[L].smem_off >> 4);
  const uint32_t a_map0[2] = {a_lo0 + uint32_t((c.map_s[0] - c.stage_s) >> 4), a_lo0 + uint32_t((c.map_s[1] - c.stage_s) >> 4)};
  constexpr uint32_t kTile16 = uint32_t(kRdbTileBytes) >> 4;
  // a (chunk, dx) group of B: 96 rows (3 dy x 32 couts) in one CTA, the CTA's 48 of them in a pair
  constexpr uint32_t kGroup16 = uint32_t(PAIR ? kRdbGroupBytes / 2 : kRdbGroupBytes) >> 4;
  constexpr uint32_t kChunk16 = 3 * kGroup16;
  constexpr uint32_t kIdesc = ptx::umma_idesc_bf16_f32(PAIR ? 256 : 128, 96, 0, 0);
  auto issue6 = [&](uint32_t d, uint32_t a, uint32_t b) {
#pragma unroll
    for (int dx = 0; dx < 3; ++dx)
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        const uint32_t a_lo = a + uint32_t((dx * 64 + ks * 32) >> 4), b_lo = b + uint32_t(dx) * kGroup16 + uint32_t((ks * 32) >> 4);
        if constexpr (PAIR)
          ptx::umma_ss_lh_pair<true>(d, a_lo, a_hi, b_lo, b_hi, kIdesc);
        else
          ptx::umma_ss_lh<true>(d, a_lo, a_hi, b_lo, b_hi, kIdesc);
      }
  };
  auto commit = [](uint64_t* bar) {
    if constexpr (PAIR)
      ptx::umma_commit_pair(bar);
    else
      ptx::umma_commit(bar);
  };
  const bool prof = XMM_RDB_PROFILE && args.prof != nullptr && L == 0;
  long long pw[3] = {0, 0, 0};
  const long long t_begin = XMM_RDB_PROFILE ? clock64() : 0;
  uint32_t fills = 0;  // chunks consumed so far
  uint32_t n = 0;      // steps taken so far
  int seq[2] = {0, 0}; // sequence number, in map m, of the current piece's first row
  int xseq = 0;        // x0 ring: sequence number of the current piece's first x0 row, ra - NL
  for (int pi = 0; pi < sched.npieces; ++pi) {
    const RdbPiece pc = sched.get(pi);
    const int r_last = pc.rb + e;  // last step with MMAs; two flush steps follow
    for (int r = pc.ra - e - 1; r <= r_last + 2; ++r, ++n) {
      // the row completed by the previous step is out of its accumulator slots (and they are re-initialised)
      if (n > 0) rdb_wait_p(&c.tdrain[L], (n - 1u) & 1u, 2, L, int(n), prof, pw[0]);
      ptx::tc_fence_after();
      if (r <= r_last) {
        const uint32_t d = c.tmem_base + uint32_t(L * kRdbSlotCols + rdb_phi(r - 1) * 32);
        auto global_chunks = [&]() {
          if constexpr (kRdbXRing<G, PAIR>) {
            // x0 row r of this piece, loaded once for all layers; the last layer that reads it gives the slot back.
            // Every later step of a piece follows a step that waited for the map rows r - 1 (the earlier layers' steps
            // on r, which read x0 row r), but the first one follows flush steps: it waits for its map rows r (the
            // earlier layers' steps on r + 1) before it can release row r.
            if (L > 0 && r == pc.ra - e - 1) {
#pragma unroll
              for (int m = 0; m < NM; ++m)
                if (m < L) {
                  const int sq = seq[m] + (r - (pc.ra - (NL - 1 - m)));
                  rdb_wait_p(&c.mfull[m * 8 + sq % ring[m]], uint32_t(sq / ring[m]) & 1u, 4, L * 10 + m, sq, prof, pw[2]);
                }
            }
            const int sq = xseq + (r - (pc.ra - NL));
            const int slot = sq % args.stages;
            rdb_wait_p(&c.lfull[slot], uint32_t(sq / args.stages) & 1u, 3, L, sq, prof, pw[1]);
            ptx::tc_fence_after();
            issue6(d, a_lo0 + uint32_t(slot) * kTile16, b_l);
            if (L == NL - 1 || r < pc.ra - e || r > pc.rb + e - 1) commit(&c.empty[slot]);
          } else {
#pragma unroll
            for (int g = 0; g < G; ++g) {
              const int k = int(fills % kR);
              rdb_wait_p(&c.lfull[L * kR + k], (fills / kR) & 1u, 3, L, k, prof, pw[1]);
              const int stage = c.lstage[L * kR + k];
              ++fills;
              ptx::tc_fence_after();
              issue6(d, a_lo0 + uint32_t(stage) * kTile16, b_l + uint32_t(g) * kChunk16);
              commit(&c.empty[stage]);
            }
          }
        };
        auto map_chunks = [&]() {
#pragma unroll
          for (int m = 0; m < NM; ++m)
            if (m < L) {
              const int sq = seq[m] + (r - (pc.ra - (NL - 1 - m)));
              const int slot = sq % ring[m];
              rdb_wait_p(&c.mfull[m * 8 + slot], uint32_t(sq / ring[m]) & 1u, 4, L * 10 + m, sq, prof, pw[2]);
              ptx::tc_fence_after();
              issue6(d, a_map0[m] + uint32_t(slot) * kTile16, b_l + uint32_t(G + m) * kChunk16);
              // the last layer that reads this row gives the tile back: layer L+1 reads rows [ra-e, rb+e-1]
              if (L == NL - 1 || r < pc.ra - e || r > pc.rb + e - 1) commit(&c.mempty[m * 8 + slot]);
            }
        };
        // Two fused layers: the in-CTA map first -- x4 was written a round ago, while the four global chunks of this
        // step may still be landing in the few stages the weights leave room for.  (The order of the K chunks only
        // changes the order of the fp32 sums.)
        if (NL == 2) {
          map_chunks();
          global_chunks();
        } else {
          global_chunks();
          map_chunks();
        }
      }
      commit(&c.tfull[L]);  // row r-1 is complete
    }
#pragma unroll
    for (int m = 0; m < NM; ++m) seq[m] += (pc.rb - pc.ra) + 2 * (NL - 1 - m);
    xseq += (pc.rb - pc.ra) + 2 * NL;
  }
  if (XMM_RDB_PROFILE && prof) {
    long long* o = args.prof + size_t(blockIdx.x) * kRdbProfSlots;
    o[0] = clock64() - t_begin;
    o[1] = pw[0];
    o[2] = pw[1];
    o[3] = pw[2];
  }
}

// ---------------------------------------------------------------------------------------------------- epilogue
// Four warps per layer (one per TMEM lane quarter) drain that layer's rows in order.
// PAIR: the peer's warps arrive on the LEADER's tdrain / mfull (relaxed: a release.cluster arrive would wait for this
// warp's global stores as well and stall the epilogue).
template <int G, int NL, int L, bool PAIR, bool FIRST_ONLY = false>
__device__ __forceinline__ void rdb_epilogue(const RdbArgs& args, const RdbCtx& c, const RdbSched<NL, PAIR>& sched, int q,
                                             int lane) {
  const bool remote = PAIR && sched.rank != 0;
  auto arrive = [&](uint64_t* bar) {
    if (remote)
      ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(bar), 0));
    else
      ptx::mbar_arrive(bar);
  };
  constexpr int e = NL - 1 - L;
  constexpr int ring[2] = {NL == 3 ? 5 : 2, 3};
  constexpr bool last = L == NL - 1;
  const int pos = q * 32 + lane + 1;  // pixel position of this lane in a row tile
  const int band = pos >= kRdbBoxPx ? 1 : 0;
  const int pl = band ? pos - (kRdbBoxPx + 1) : pos - 1;  // pixel within the band segment
  const bool lane_ok = band ? pl >= 0 : pl < kRdbP;
  const uint32_t lane_base = c.tmem_base + (uint32_t(q * 32) << 16) + uint32_t(L * kRdbSlotCols);
  const uint32_t pos_off = uint32_t(pos) * 64u;
  const uint32_t pos_xor = uint32_t(pos >> 1) & 3u;
  const uint32_t bias_a = ptx::smem_u32(c.w_s + args.layer[L].smem_off + args.layer[L].w_bytes);
  const float slope = args.layer[L].lrelu_slope;
  const bool has_r1 = last && args.r1 != nullptr, has_r2 = last && args.r2 != nullptr;
  const bool prof = XMM_RDB_PROFILE && args.prof != nullptr;
  long long pw[2] = {0, 0};
  long long ph[4] = {0, 0, 0, 0};
  long long tph = 0;
  const long long t_begin = XMM_RDB_PROFILE ? clock64() : 0;
  uint32_t n = 0;  // rows drained so far
  int seq = 0;     // sequence number, in map L, of the current piece's first row
  for (int pi = 0; pi < sched.npieces; ++pi) {
    const RdbPiece pc = sched.get(pi);
    const int px = pc.x0 + pl;
    const bool px_ok = lane_ok && px < args.width;
    const bool px_own = px_ok && px >= pc.own_lo && px < pc.own_hi;
    for (int r = pc.ra - e - 1; r <= pc.rb + e + 2; ++r, ++n) {
      const int j = r - 1;  // the row this step completed
      const bool real = j >= pc.ra - e && j < pc.rb + e;
      const int y = band * args.band_h + j;
      const bool inimg = px_ok && y >= 0 && y < args.height;
      const bool owned = real && px_own && inimg && j >= pc.ra && j < pc.rb;
      const size_t pix = size_t((pc.b * args.height + (y < 0 ? 0 : y)) * args.width + (px_ok ? px : 0));
      // residuals of the last layer: requested before the accumulator is waited for
      uint4 res1[4], res2[4];
      if (has_r1 && owned) {
        const __nv_bfloat16* p = args.r1 + pix * args.r1_ctot + args.r1_coff;
        ld_global_nc_256(p, res1[0], res1[1]);
        ld_global_nc_256(p + 16, res1[2], res1[3]);
      }
      if (has_r2 && owned) {
        const __nv_bfloat16* p = args.r2 + pix * args.r2_ctot + args.r2_coff;
        ld_global_nc_256(p, res2[0], res2[1]);
        ld_global_nc_256(p + 16, res2[2], res2[3]);
      }
      if (XMM_RDB_PROFILE)
        rdb_wait_p(&c.tfull[L], n & 1u, 5, L, int(n), prof, pw[0]);
      else
        rdb_wait_backoff(&c.tfull[L], n & 1u, 5, L, int(n), uint32_t(args.backoff_ns));
      if (XMM_RDB_PROFILE) tph = clock64();
      ptx::tc_fence_after();
      const int phi = rdb_phi(j);
      const uint32_t t_main = lane_base + uint32_t(phi * 32);
      const uint32_t t_carry = lane_base + uint32_t((3 + phi) * 32);
      float v[32];
      {
        uint32_t accr[32];
        ptx::tmem_ld_32x32(t_main, accr);
        if (phi < 2) {  // the row's first partial sums were collected in a carry slot
          uint32_t car[32];
          ptx::tmem_ld_32x32(t_carry, car);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(car[k]) + __uint_as_float(accr[k]);
          tmem_st_zero32(t_carry);
        } else {
          ptx::tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(accr[k]);
        }
      }
      {  // the slot's next row starts from the bias
        uint32_t b32[32];
#pragma unroll
        for (int k = 0; k < 8; ++k)
          asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                       : "=r"(b32[4 * k]), "=r"(b32[4 * k + 1]), "=r"(b32[4 * k + 2]), "=r"(b32[4 * k + 3])
                       : "r"(bias_a + 16u * k));
        tmem_st_32x32(t_main, b32);
      }
      tmem_st_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) arrive(&c.tdrain[L]);
      if (XMM_RDB_PROFILE) {
        const long long t = clock64();
        ph[0] += t - tph;
        tph = t;
      }
      if (!real) continue;

      if (slope != 1.f) {  // LeakyReLU, 0 < slope < 1: max(v, slope * v)
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] = fmaxf(v[k], v[k] * slope);
      }
      if (last) {
        const float s0 = args.s0;
        if (s0 != 1.f) {
#pragma unroll
          for (int k = 0; k < 32; ++k) v[k] *= s0;
        }
        if (has_r1 && owned) {
          const float s1 = args.s1;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float m8[8];
            unpack8(res1[k], m8);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[8 * k + i] = fmaf(s1, m8[i], v[8 * k + i]);
          }
        }
        if (has_r2 && owned) {
          const float s2 = args.s2;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float m8[8];
            unpack8(res2[k], m8);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[8 * k + i] = fmaf(s2, m8[i], v[8 * k + i]);
          }
        }
      }
      uint4 o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) o[k] = pack8(v + 8 * k);
      if (XMM_RDB_PROFILE) {
        const long long t = clock64();
        ph[1] += t - tph;
        tph = t;
      }
      if (args.layer[L].store && owned) {  // (before the map write: the stores drain while the fence below waits)
        __nv_bfloat16* gp = args.layer[L].out + pix * args.layer[L].out_ctot + args.layer[L].out_coff;
        st_global_256(gp, o[0], o[1]);
        st_global_256(gp + 16, o[2], o[3]);
      }
      if (!last && !FIRST_ONLY) {
        // the next layers' A operand: row j of map L, swizzled as a TMA load would have written it; zeros outside
        // the image (padding) and on the junk lanes
        const int sq = seq + (j - (pc.ra - e));
        const int slot = sq % ring[L];
        rdb_wait_p(&c.mempty[L * 8 + slot], (uint32_t(sq / ring[L]) & 1u) ^ 1u, 6, L, sq, prof, pw[1]);
        if (XMM_RDB_PROFILE) tph = clock64();
        uint8_t* dst = c.map_s[L] + size_t(slot) * kRdbTileBytes + pos_off;
        const uint4 zero = make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int k = 0; k < 4; ++k) *reinterpret_cast<uint4*>(dst + ((uint32_t(k) ^ pos_xor) << 4)) = inimg ? o[k] : zero;
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) arrive(&c.mfull[L * 8 + slot]);
        if (XMM_RDB_PROFILE) {
          const long long t = clock64();
          ph[2] += t - tph;
          tph = t;
        }
      }
      if (XMM_RDB_PROFILE) {
        const long long t = clock64();
        ph[3] += t - tph;
        tph = t;
      }
    }
    seq += (pc.rb - pc.ra) + 2 * e;
  }
  if (XMM_RDB_PROFILE && prof && q == 0 && lane == 0 && L < 2) {
    long long* o = args.prof + size_t(blockIdx.x) * kRdbProfSlots + 4 + 4 * L;
    o[0] = clock64() - t_begin;
    o[1] = pw[0];
    o[2] = pw[1];
    o[3] = (long long)n;
    long long* o2 = args.prof + size_t(blockIdx.x) * kRdbProfSlots + 12 + 4 * L;  // the phases of one row
    o2[0] = ph[0];
    o2[1] = ph[1];
    o2[2] = ph[2];
    o2[3] = ph[3];
  }
}

// ---------------------------------------------------------------------------------------------------- TMA producer
// (two fused layers) One producer thread PER LAYER, each with its own slice [s0, s0 + ns) of the stage ring: with the
// 166 KB of weights of conv4 + conv5 only five stages fit, and one thread walking both layers' steps in one shared ring
// could not keep them full (the issuer of conv4 waited 31 % of its time for chunks).  A layer's thread only follows
// its own layer -- pieces in order, rows top to bottom -- and only waits for its own layer's MMAs.
template <int G, int NL, int L>
__device__ __forceinline__ void rdb_layer_producer(const CUtensorMap* tmap_in, const RdbArgs& args, const RdbCtx& c,
                                                   const RdbSched<NL>& sched, int s0, int ns) {
  constexpr int e = NL - 1 - L;
  int idx = 0;
  uint32_t phase = 0;
  uint32_t fills = 0;
  for (int pi = 0; pi < sched.npieces; ++pi) {
    const RdbPiece pc = sched.get(pi);
    for (int r = pc.ra - e - 1; r <= pc.rb + e; ++r) {
      int row = r, band0 = 0;
      if (r < 0) {
        row = r + args.band_h;
        band0 = -1;
      } else if (r >= args.band_h) {
        row = r - args.band_h;
        band0 = 1;
      }
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const int stage = s0 + idx;
        rdb_wait_backoff(&c.empty[stage], phase ^ 1u, 1, L, stage, uint32_t(args.backoff_ns));
        const int k = int(fills++ & 7u);
        c.lstage[L * 8 + k] = stage;
        uint64_t* fb = &c.lfull[L * 8 + k];
        ptx::mbar_expect_tx(fb, kRdbTileData);
        ptx::tma_load_5d(c.stage_s + size_t(stage) * kRdbTileBytes, tmap_in, fb, args.cin_off + 32 * g, pc.x0 - 1, row, band0, pc.b);
        if (++idx == ns) {
          idx = 0;
          phase ^= 1u;
        }
      }
      if (L == 0 && args.prefetch_rows > 0) {  // the first layer's rows come from HBM: ask L2 for them ahead of time
        const int rp = r + args.prefetch_rows;
        if (rp <= pc.rb + e) {
          int prow = rp, pband = 0;
          if (rp < 0) {
            prow = rp + args.band_h;
            pband = -1;
          } else if (rp >= args.band_h) {
            prow = rp - args.band_h;
            pband = 1;
          }
#pragma unroll
          for (int g = 0; g < G; ++g)
            asm volatile("cp.async.bulk.prefetch.tensor.5d.L2.global.tile [%0, {%1, %2, %3, %4, %5}];" ::"l"(
                             reinterpret_cast<uint64_t>(tmap_in)),
                         "r"(args.cin_off + 32 * g), "r"(pc.x0 - 1), "r"(prow), "r"(pband), "r"(pc.b)
                         : "memory");
        }
      }
    }
  }
}

// (conv1..conv3 as a CTA pair) The x0 ring: every x0 row of a piece once, in row order, over the first layer's rows
// [ra - NL, rb + NL - 1]; no walk.  No L2 prefetch: the ring runs 11 rows ahead by itself, and a dense block took
// 2.73 ms with a prefetch three rows ahead against 2.66 ms without (profiles/r05_rdb_probe_ring_prefetch.log).  Slot and phase follow the row's sequence number, as in the issuers.  Both CTAs'
// loads complete on the leader's lfull[slot], which the leader arms for both; each CTA waits for its own empty[slot]
// (the multicast commit of the row's last reader).
template <int NL>
__device__ __forceinline__ void rdb_x0_producer(const CUtensorMap* tmap_in, const RdbArgs& args, const RdbCtx& c,
                                                const RdbSched<NL, true>& sched) {
  int slot = 0;
  uint32_t phase = 0;
  for (int pi = 0; pi < sched.npieces; ++pi) {
    const RdbPiece pc = sched.get(pi);
    for (int r = pc.ra - NL; r <= pc.rb + NL - 1; ++r) {
      int row = r, band0 = 0;
      if (r < 0) {
        row = r + args.band_h;
        band0 = -1;
      } else if (r >= args.band_h) {
        row = r - args.band_h;
        band0 = 1;
      }
      rdb_wait_backoff(&c.empty[slot], phase ^ 1u, 1, 0, slot, uint32_t(args.backoff_ns));
      uint64_t* fb = &c.lfull[slot];
      if (sched.rank == 0) ptx::mbar_expect_tx(fb, 2 * kRdbTileData);
      ptx::tma_load_5d_pair(c.stage_s + size_t(slot) * kRdbTileBytes, tmap_in, ptx::mapa(ptx::smem_u32(fb), 0),
                            args.cin_off, pc.x0 - 1, row, band0, pc.b);
      if (++slot == args.stages) {
        slot = 0;
        phase ^= 1u;
      }
    }
  }
}

// G: feature maps read from global memory (x0 .. x_{G-1}); NL: fused layers.  Layer l (0-based) is conv_{G+l}: its K
// chunks are the G global maps then the l maps produced in this CTA.
// Warp roles (512 threads): warp 0 = TMA producer (the only role that follows the interleaved walk: it decides the
// order in which the layers' rows are loaded), warp 1 + l = MMA issuer of layer l, warps 4 + 4 l .. 7 + 4 l = epilogue
// of layer l.  Issuers and epilogue groups only know their own layer; everything between roles is an mbarrier.
// PAIR: launched as clusters of 2 (see the top of this file).
// FIRST_ONLY (conv4 + conv5 only): the conv4-only form that recomputes x4 for a backward pass.  It keeps the two-layer
// work split, walk and conv4 accumulator rule, so x4 is bit-equal to what the full kernel stores; conv5's issuer and
// epilogue group do nothing, the producer loads conv4's chunks only and conv4's epilogue writes no map rows.
template <int G, int NL, bool PAIR = false, bool FIRST_ONLY = false>
__global__ void __launch_bounds__(kRdbThreads, 1)
conv3x3_rdb_kernel(const __grid_constant__ CUtensorMap tmap_in, const RdbArgs args) {
  static_assert(NL == 2 || NL == 3, "two or three fused layers");
  static_assert(!FIRST_ONLY || NL == 2, "the conv4-only form is a form of conv4 + conv5");
  constexpr int NA = FIRST_ONLY ? 1 : NL;  // layers that run
  static_assert(NL * kRdbSlotCols <= 512, "accumulators exceed TMEM");
  constexpr int NM = NL - 1;  // in-CTA maps
  constexpr int kR = kRdbLRing<PAIR>;
  constexpr bool XR = kRdbXRing<G, PAIR>;
  constexpr int kFull = XR ? kR : 3 * kR;   // lfull: per-layer landed rings, or the x0 ring's full barriers
  constexpr int kStageIds = XR ? 0 : 3 * kR;  // lstage
  // lfull, empty, tfull, tdrain, mfull, mempty, w_bar; lstage; the TMEM address: the 1024 B the launcher reserves
  static_assert((kFull + kR + 3 + 3 + 16 + 16 + 1) * 8 + kStageIds * 4 + 4 <= 1024, "barrier block exceeds 1024 B");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  RdbCtx c;
  c.w_s = smem;
  c.stage_s = smem + args.w_total;
  c.map_s[0] = c.stage_s + size_t(args.stages) * kRdbTileBytes;
  c.map_s[1] = c.map_s[0] + size_t(args.ring0) * kRdbTileBytes;
  uint8_t* after = c.map_s[1] + size_t(NM > 1 ? args.ring1 : 0) * kRdbTileBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(after);
  c.lfull = bars;              // 3 R (x0 ring: R)
  c.empty = c.lfull + kFull;   // R
  c.tfull = c.empty + kR;      // 3
  c.tdrain = c.tfull + 3;      // 3
  c.mfull = c.tdrain + 3;      // 16
  c.mempty = c.mfull + 16;     // 16
  c.w_bar = c.mempty + 16;     // 1
  c.lstage = reinterpret_cast<volatile int*>(c.w_bar + 1);  // 3 R ints (x0 ring: none)
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(const_cast<int*>(c.lstage) + kStageIds);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? ptx::cluster_ctarank() : 0u;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_in);
    for (int s = 0; s < (XR ? kFull : NL * kR); ++s) ptx::mbar_init(&c.lfull[s], 1);
    for (int s = 0; s < args.stages; ++s) ptx::mbar_init(&c.empty[s], 1);
    for (int l = 0; l < NL; ++l) {
      ptx::mbar_init(&c.tfull[l], 1);
      ptx::mbar_init(&c.tdrain[l], PAIR ? 8 : 4);  // the four warps of the layer's epilogue group (pair: in both CTAs)
    }
    for (int s = 0; s < 16; ++s) {
      ptx::mbar_init(&c.mfull[s], PAIR ? 8 : 4);
      ptx::mbar_init(&c.mempty[s], 1);  // the commit of the row's last reader
    }
    ptx::mbar_init(c.w_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (PAIR)
      ptx::tmem_alloc_pair<512>(tmem_ptr_s);
    else
      ptx::tmem_alloc<512>(tmem_ptr_s);
  }
  ptx::tc_fence_before();
  if constexpr (PAIR)
    ptx::cluster_sync();  // the peer's barriers are initialised before anything arrives on them
  else
    __syncthreads();
  ptx::tc_fence_after();
  c.tmem_base = *tmem_ptr_s;

  if (warp == 0 && ptx::elect_one()) {  // weights + biases of every layer (the accumulators are initialised from them)
    uint32_t wtot = 0;
    for (int l = 0; l < NA; ++l) wtot += args.layer[l].w_bytes + 128u;
    ptx::mbar_expect_tx(c.w_bar, wtot);
    for (int l = 0; l < NA; ++l) {
      const uint8_t* gsrc = static_cast<const uint8_t*>(args.layer[l].wblob);
      uint8_t* dst = c.w_s + args.layer[l].smem_off;
      const uint32_t wb = args.layer[l].w_bytes;
      if constexpr (PAIR) {
        // this CTA's half of every (chunk, dx) group: rows [48 rank, 48 rank + 48), six whole SWIZZLE_64B atoms
        constexpr uint32_t kHalf = kRdbGroupBytes / 2;
        for (uint32_t grp = 0; grp < wb / kHalf; ++grp)
          ptx::bulk_load(dst + grp * kHalf, gsrc + grp * kRdbGroupBytes + rank * kHalf, kHalf, c.w_bar);
        ptx::bulk_load(dst + wb, gsrc + 2 * wb, 128u, c.w_bar);
      } else {
        const uint32_t n_l = wb + 128u;
        for (uint32_t off = 0; off < n_l; off += 32768u)
          ptx::bulk_load(dst + off, gsrc + off, n_l - off < 32768u ? n_l - off : 32768u, c.w_bar);
      }
    }
  }
  const int egroup = (warp - 4) >> 2;  // epilogue group = layer (warps 4..)
  if (warp >= 4) {
    // halo positions of the map tiles stay zero for ever
    uint4* z = reinterpret_cast<uint4*>(c.map_s[0]);
    const int nz = (args.ring0 + (NM > 1 ? args.ring1 : 0)) * (kRdbTileBytes / 16);
    for (int i = int(threadIdx.x) - 128; i < nz; i += kRdbThreads - 128) z[i] = make_uint4(0, 0, 0, 0);
    ptx::fence_proxy_async();
    // Every MMA accumulates.  A row's accumulator (window slots 0..2) starts as the layer's BIAS, its carry slot
    // (3, 4) as zero: the epilogue re-initialises a slot right after draining it and never adds the bias itself.
    if (egroup < NA) {
      rdb_wait(c.w_bar, 0, 9, 0, 0);
      const uint32_t lane_base = c.tmem_base + (uint32_t((warp & 3) * 32) << 16) + uint32_t(egroup * kRdbSlotCols);
      const float* bias_s = reinterpret_cast<const float*>(c.w_s + args.layer[egroup].smem_off + args.layer[egroup].w_bytes);
      uint32_t b32[32];
#pragma unroll
      for (int k = 0; k < 32; ++k) b32[k] = __float_as_uint(bias_s[k]);
      for (int sl = 0; sl < 3; ++sl) tmem_st_32x32(lane_base + uint32_t(sl * 32), b32);
      for (int sl = 3; sl < kRdbSlots; ++sl) tmem_st_zero32(lane_base + uint32_t(sl * 32));
      tmem_st_wait();
    }
  }
  ptx::tc_fence_before();
  if constexpr (PAIR)
    ptx::cluster_sync();  // the leader's first MMAs read the peer's weights and accumulate into the peer's TMEM
  else
    __syncthreads();
  ptx::tc_fence_after();

  RdbSched<NL, PAIR> sched;
  sched.init(args);

  if (!PAIR && NL == 2 && !FIRST_ONLY && args.split_producers && (warp == 0 || warp == 3)) {
    // ------------------------------------------------------------ TMA producers, one per layer (warps 0 and 3)
    if constexpr (!PAIR) {
      if (ptx::elect_one()) {
        const int ns0 = (args.stages + 1) / 2;  // conv4 (whose rows come from HBM) gets the larger half
        if (warp == 0) rdb_layer_producer<G, NL, 0>(&tmap_in, args, c, sched, 0, ns0);
        if (warp == 3) rdb_layer_producer<G, NL, 1>(&tmap_in, args, c, sched, ns0, args.stages - ns0);
      }
    }
  } else if (XR && warp == 0) {
    // ------------------------------------------------------------ TMA producer of the x0 ring (conv1..conv3 pair)
    if constexpr (XR) {
      if (ptx::elect_one()) rdb_x0_producer<NL>(&tmap_in, args, c, sched);
    }
  } else if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    // PAIR: both CTAs' producers take the same walk over the same stage count, so they write the same stage ids into
    // lstage -- the leader's issuers address the peer's stages with the leader's ids.  Both loads of a chunk complete
    // on the leader's lfull, which the leader's producer arms for both.
    if (!XR && ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t fills[NL];  // chunks loaded for layer l so far
#pragma unroll
      for (int l = 0; l < NL; ++l) fills[l] = 0;
      rdb_walk<NL>(sched, [&](int l, const RdbPiece& pc, int r, bool flush, int, const int*) {
        if (flush || (FIRST_ONLY && l > 0)) return;
        // input row r of both bands; above / below a band: the neighbouring band's rows (outside the image: zeros)
        int row = r, band0 = 0;
        if (r < 0) {
          row = r + args.band_h;
          band0 = -1;
        } else if (r >= args.band_h) {
          row = r - args.band_h;
          band0 = 1;
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
          rdb_wait_backoff(&c.empty[stage], phase ^ 1u, 1, l, stage, uint32_t(args.backoff_ns));
          const int k = int(fills[l]++ % uint32_t(kR));
          c.lstage[l * kR + k] = stage;  // (made visible to the issuer by the release of the arrive below)
          uint64_t* fb = &c.lfull[l * kR + k];
          if constexpr (PAIR) {
            if (rank == 0) ptx::mbar_expect_tx(fb, 2 * kRdbTileData);
            ptx::tma_load_5d_pair(c.stage_s + size_t(stage) * kRdbTileBytes, &tmap_in, ptx::mapa(ptx::smem_u32(fb), 0),
                                  args.cin_off + 32 * g, pc.x0 - 1, row, band0, pc.b);
          } else {
            ptx::mbar_expect_tx(fb, kRdbTileData);
            ptx::tma_load_5d(c.stage_s + size_t(stage) * kRdbTileBytes, &tmap_in, fb, args.cin_off + 32 * g, pc.x0 - 1, row,
                             band0, pc.b);
          }
          if (++stage == args.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        // the first layer streams the global maps from HBM (the others re-read them out of L2 a few rows later): with
        // few stages the TMA latency is exposed, so its rows can be requested into L2 ahead of time
        if (l == 0 && args.prefetch_rows > 0) {
          const int rp = r + args.prefetch_rows;
          if (rp <= pc.rb + (NL - 1)) {
            int prow = rp, pband = 0;
            if (rp < 0) {
              prow = rp + args.band_h;
              pband = -1;
            } else if (rp >= args.band_h) {
              prow = rp - args.band_h;
              pband = 1;
            }
#pragma unroll
            for (int g = 0; g < G; ++g)
              asm volatile("cp.async.bulk.prefetch.tensor.5d.L2.global.tile [%0, {%1, %2, %3, %4, %5}];" ::"l"(
                               reinterpret_cast<uint64_t>(&tmap_in)),
                           "r"(args.cin_off + 32 * g), "r"(pc.x0 - 1), "r"(prow), "r"(pband), "r"(pc.b)
                           : "memory");
          }
        }
      });
    }
  } else if (warp <= 3) {
    // (warp 3 of a two-layer kernel: idle, or the second producer above; PAIR: the peer issues nothing)
    if (warp - 1 < NA && rank == 0 && ptx::elect_one()) {
      if (warp == 1) rdb_issuer<G, NL, 0, PAIR>(args, c, sched);
      if (warp == 2) rdb_issuer<G, NL, 1, PAIR>(args, c, sched);
      if constexpr (NL == 3) {
        if (warp == 3) rdb_issuer<G, NL, 2, PAIR>(args, c, sched);
      }
    }
  } else if (egroup < NA) {
    const int q = warp & 3;  // TMEM lane quarter this warp may read
    if (egroup == 0) rdb_epilogue<G, NL, 0, PAIR, FIRST_ONLY>(args, c, sched, q, lane);
    if (egroup == 1) rdb_epilogue<G, NL, 1, PAIR>(args, c, sched, q, lane);
    if constexpr (NL == 3) {
      if (egroup == 2) rdb_epilogue<G, NL, 2, PAIR>(args, c, sched, q, lane);
    }
  }

  ptx::tc_fence_before();
  if constexpr (PAIR)
    ptx::cluster_sync();  // neither CTA may exit while the other can still multicast to it or arrive on it
  else
    __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    if constexpr (PAIR)
      ptx::tmem_dealloc_pair<512>(c.tmem_base);
    else
      ptx::tmem_dealloc<512>(c.tmem_base);
  }
}

}  // namespace xmm
