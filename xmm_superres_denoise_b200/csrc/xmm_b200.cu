// libxmm_b200.so -- C ABI launchers (see include/xmm_b200.h for the contract).
#include "../../include/xmm_b200.h"

#include <unordered_map>
#include <vector>

#include "conv3x3_chain.cuh"
#include "conv3x3_dx.cuh"
#include "conv3x3_row.cuh"
#include "conv3x3_rdb.cuh"
#include "conv3x3_tc.cuh"
#include "edge_kernels.cuh"
#include "host_common.cuh"
#include "loss_kernels.cuh"
#include "pack_weights.cuh"
#include "wgrad_tc.cuh"

#ifndef XMM_DEFAULT_TAP_MODE
#define XMM_DEFAULT_TAP_MODE 0
#endif

using namespace xmm;

extern "C" const char* xmm_last_error(void) { return last_error_ref().c_str(); }
extern "C" int xmm_version(void) { return 101; }
extern "C" int xmm_check_device(void) {
  DeviceInfo d;
  return require_sm100(&d);
}

// ----------------------------------------------------------------------------- packing
extern "C" size_t xmm_pack_blob_bytes(int nt, int kc, int nchunks) {
  return size_t(nchunks) * 9 * nt * kc * 2 + size_t(nt) * 4;
}

extern "C" int xmm_pack_weights(const xmm_pack_job* jobs_dev, int njobs, void* stream) {
  DeviceInfo d;
  int rc = require_sm100(&d);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(jobs_dev != nullptr && njobs > 0, "xmm_pack_weights: empty job table");
  dim3 grid(45, njobs);
  pack_jobs_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(jobs_dev);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

// ----------------------------------------------------------------------------- conv3x3
namespace {

struct TmapKey {
  const void* base;
  int batch, height, width, ctot, box_c, box_w, box_h;
  bool operator==(const TmapKey& o) const {
    return base == o.base && batch == o.batch && height == o.height && width == o.width && ctot == o.ctot &&
           box_c == o.box_c && box_w == o.box_w && box_h == o.box_h;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.base);
    auto mix = [&h](size_t v) { h ^= v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2); };
    mix(k.batch); mix(k.height); mix(k.width); mix(k.ctot); mix(k.box_c); mix(k.box_w); mix(k.box_h);
    return h;
  }
};


// cudaFuncSetAttribute is per DEVICE: remember (kernel, device) pairs, not just kernels (a second GPU driven from
// the same process would otherwise never get the > 48 KB dynamic shared-memory opt-in).
int ensure_max_smem(const void* kernel, const DeviceInfo& dev, int reserve = 0) {
  static std::mutex mu;
  static std::unordered_map<const void*, unsigned long long> done;
  {
    std::lock_guard<std::mutex> lk(mu);
    unsigned long long& bits = done[kernel];
    if (bits & (1ull << dev.device)) return XMM_OK;
    bits |= 1ull << dev.device;
  }
  XMM_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin - reserve));
  return XMM_OK;
}

// Descriptors are pure functions of (pointer, shape); caching only saves the encode call.
int cached_tmap(CUtensorMap* out, const void* base, int batch, int height, int width, int ctot, int box_c,
                int box_w, int box_h) {
  static std::mutex mu;
  static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  TmapKey key{base, batch, height, width, ctot, box_c, box_w, box_h};
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(key);
  if (it != cache.end()) {
    *out = it->second;
    return XMM_OK;
  }
  int rc = make_nhwc_tmap(out, base, batch, height, width, ctot, box_c, box_w, box_h, false);
  if (rc != XMM_OK) return rc;
  if (cache.size() > 4096) cache.clear();
  cache.emplace(key, *out);
  return XMM_OK;
}

void fill_epilogue(ConvEpilogue& e, const xmm_conv3x3_params& p) {
  e.lrelu_slope = p.lrelu_slope;
  e.mask_slope = p.mask_slope;
  e.s0 = p.s0; e.s1 = p.s1; e.s2 = p.s2;
  e.mask = static_cast<const __nv_bfloat16*>(p.mask); e.mask_ctot = p.mask_ctot; e.mask_coff = p.mask_coff;
  e.r1 = static_cast<const __nv_bfloat16*>(p.r1); e.r1_ctot = p.r1_ctot; e.r1_coff = p.r1_coff;
  e.r2 = static_cast<const __nv_bfloat16*>(p.r2); e.r2_ctot = p.r2_ctot; e.r2_coff = p.r2_coff;
  e.out = static_cast<__nv_bfloat16*>(p.out); e.out_ctot = p.out_ctot; e.out_coff = p.out_coff;
  e.pixel_shuffle = p.pixel_shuffle;
  e.shuffle_stride = p.shuffle_stride > 0 ? p.shuffle_stride : p.cout;
  e.img_out = nullptr; e.img_res = nullptr; e.img_pre = nullptr; e.img_cout = 0; e.img_clamp = 0;
  e.colsum = p.colsum; e.colsum_scale = p.colsum_scale;
  e.colsum_ws = p.colsum ? p.colsum_ws : nullptr;
}

struct ImageOut {
  float* out;
  const float* res;
  float* pre;
  int cout, clamp;
};

constexpr bool kTcTwoGroupsDefault = true;  // measured: Cin=32 layer 0.129 -> 0.114 ms, F->4F conv 0.346 -> 0.315 ms (batch 16)
template <int KC, int NT, int MODE, int EG>
int launch_conv_impl(const xmm_conv3x3_params& p, const DeviceInfo& dev, cudaStream_t stream, const ImageOut* img) {
  using Cfg = ConvCfg<KC, NT, MODE, EG>;
  ConvArgs a{};
  a.wblob = p.wblob;
  a.nchunks = p.cin / KC;
  a.w_bytes = uint32_t(a.nchunks) * 9u * Cfg::kTapBytes;
  a.cin_off = p.in_coff;
  a.batch = p.batch;
  a.height = p.height;
  a.width = p.width;
  a.tiles_x = (p.width + kTileW - 1) / kTileW;
  a.tiles_y = (p.height + kTileH - 1) / kTileH;
  a.num_tiles = a.tiles_x * a.tiles_y * p.batch;
  // Plain NHWC outputs of narrow layers leave through per-warp TMA stores (XMM_TC_TMA_STORE=0: direct stores, 2: always) -- as
  // long as their staging tiles (16 / 32 KB) do not cost the layer a pipeline stage it needs: the 64-filter layers with
  // 74..147 KB of resident weights keep their stages instead (measured: F=64 inference 146 -> 160 img/s).
  static const int tma_env = [] { const char* e = getenv("XMM_TC_TMA_STORE"); return e ? atoi(e) : 1; }();
  const size_t fixed_plain = Cfg::smem_bytes(a.w_bytes, 0, false), fixed_out = Cfg::smem_bytes(a.w_bytes, 0, true);
  if (fixed_plain + 2 * size_t(Cfg::kStageBytes) > size_t(dev.max_smem_optin))
    return fail(XMM_ERR_UNSUPPORTED_SHAPE,
                "conv3x3: weights of cin=%d cout=%d (%u B) do not fit in shared memory next to 2 pipeline stages",
                p.cin, p.cout, a.w_bytes);
  auto stages_for = [&](size_t fixed) {
    const int st = size_t(dev.max_smem_optin) > fixed ? int((size_t(dev.max_smem_optin) - fixed) / Cfg::kStageBytes) : 0;
    return st > kMaxStages ? kMaxStages : st;
  };
  const int st_plain = stages_for(fixed_plain), st_out = stages_for(fixed_out);
  a.tma_store = (Cfg::kOutBytes > 0 && p.pixel_shuffle == 0 && img == nullptr && st_out >= 2 &&
                 (tma_env == 2 || (tma_env == 1 && (st_out >= 6 || st_out == st_plain))))
                    ? 1 : 0;
  const int stages = a.tma_store ? st_out : st_plain;
  a.stages = stages;
  const size_t smem = Cfg::smem_bytes(a.w_bytes, stages, a.tma_store != 0);

  fill_epilogue(a.epi, p);
  if (img != nullptr) {
    a.epi.img_out = img->out; a.epi.img_res = img->res; a.epi.img_pre = img->pre;
    a.epi.img_cout = img->cout; a.epi.img_clamp = img->clamp;
  }

  CUtensorMap tmap;
  int rc = cached_tmap(&tmap, p.in, p.batch, p.height, p.width, p.in_ctot, KC, Cfg::kPitchPx, kHaloH);
  if (rc != XMM_OK) return rc;
  CUtensorMap tmap_out = tmap;
  if (a.tma_store) {
    rc = cached_tmap(&tmap_out, p.out, p.batch, p.height, p.width, p.out_ctot, NT, kTileW, 4);
    if (rc != XMM_OK) return rc;
  }

  rc = ensure_max_smem(reinterpret_cast<const void*>(conv3x3_tc_kernel<KC, NT, MODE, EG>), dev);
  if (rc != XMM_OK) return rc;
  const int grid = a.num_tiles < dev.sm_count ? a.num_tiles : dev.sm_count;
  conv3x3_tc_kernel<KC, NT, MODE, EG><<<grid, Cfg::kThreads, smem, stream>>>(tmap, tmap_out, a);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

// Two epilogue groups (alternate tiles, 4 accumulator stages) where TMEM holds them: XMM_TC_EG=1 / 2 forces.
template <int KC, int NT, int MODE>
int launch_conv(const xmm_conv3x3_params& p, const DeviceInfo& dev, cudaStream_t stream, const ImageOut* img = nullptr) {
  static const int eg_env = [] { const char* e = getenv("XMM_TC_EG"); return e ? atoi(e) : 0; }();
  if constexpr (4 * NT <= 512) {
    const long long ntiles = (long long)((p.width + kTileW - 1) / kTileW) * ((p.height + kTileH - 1) / kTileH) * p.batch;
    if (eg_env == 2 || (eg_env == 0 && kTcTwoGroupsDefault && ntiles >= 4LL * dev.sm_count))
      return launch_conv_impl<KC, NT, MODE, 2>(p, dev, stream, img);
  }
  return launch_conv_impl<KC, NT, MODE, 1>(p, dev, stream, img);
}

// Row-gather / column-scatter form (conv3x3_dx.cuh): the default for Cout = 32 / 64.
template <int KC, int NT, bool G2>
int launch_conv_dx_impl(const xmm_conv3x3_params& p, const DeviceInfo& dev, cudaStream_t stream) {
  using Cfg = DxCfg<KC, NT, G2>;
  ConvArgs a{};
  a.wblob = p.wblob;
  a.nchunks = p.cin / KC;
  a.w_bytes = uint32_t(a.nchunks) * 9u * Cfg::kTapBytes;
  a.cin_off = p.in_coff;
  a.batch = p.batch;
  a.height = p.height;
  a.width = p.width;
  a.tiles_x = (p.width + kDxTileW - 1) / kDxTileW;
  a.tiles_y = (p.height + kDxTileH - 1) / kDxTileH;
  a.num_tiles = a.tiles_x * a.tiles_y * p.batch;
  // side inputs (LeakyReLU' mask, residuals) travel through shared memory by TMA unless the output is pixel-shuffled
  // (XMM_DX_SIDES=0 keeps the per-lane global loads, for experiments)
  static const int sides_env = [] { const char* e = getenv("XMM_DX_SIDES"); return e ? atoi(e) : 1; }();
  const void* side_ptr[3] = {p.mask, p.r1, p.r2};
  const int side_ctot[3] = {p.mask_ctot, p.r1_ctot, p.r2_ctot};
  int nside = 0;
  if (p.pixel_shuffle == 0 && sides_env)
    for (int k = 0; k < 3; ++k)
      if (side_ptr[k] != nullptr) { a.side_mask |= 1 << k; ++nside; }
  size_t fixed = Cfg::smem_bytes(a.w_bytes, 0, nside);
  if (nside > 0 && fixed + 4 * size_t(Cfg::kStageBytes) > size_t(dev.max_smem_optin)) {  // keep >= 4 pipeline stages
    a.side_mask = 0;
    nside = 0;
    fixed = Cfg::smem_bytes(a.w_bytes, 0, 0);
  }
  if (fixed + 2 * size_t(Cfg::kStageBytes) > size_t(dev.max_smem_optin))
    return fail(XMM_ERR_UNSUPPORTED_SHAPE,
                "conv3x3: weights of cin=%d cout=%d (%u B) do not fit in shared memory next to 2 pipeline stages",
                p.cin, p.cout, a.w_bytes);
  int stages = int((size_t(dev.max_smem_optin) - fixed) / Cfg::kStageBytes);
  if (stages > kMaxStages) stages = kMaxStages;
  a.stages = stages;
  const size_t smem = Cfg::smem_bytes(a.w_bytes, stages, nside);
  fill_epilogue(a.epi, p);
  CUtensorMap tmap;
  int rc = cached_tmap(&tmap, p.in, p.batch, p.height, p.width, p.in_ctot, KC, kDxTileW, kDxPatchH);
  if (rc != XMM_OK) return rc;
  CUtensorMap tmap_out = tmap;  // unused (direct stores) when the output is pixel-shuffled
  if (p.pixel_shuffle == 0) {
    rc = cached_tmap(&tmap_out, p.out, p.batch, p.height, p.width, p.out_ctot, Cfg::kWarpCols, kDxTileW, 2);
    if (rc != XMM_OK) return rc;
  }
  DxSideMaps sides;
  for (int k = 0; k < 3; ++k) {
    sides.m[k] = tmap;
    if (a.side_mask & (1 << k)) {
      rc = cached_tmap(&sides.m[k], side_ptr[k], p.batch, p.height, p.width, side_ctot[k], NT, kDxTileW, kDxTileH);
      if (rc != XMM_OK) return rc;
    }
  }
  rc = ensure_max_smem(reinterpret_cast<const void*>(conv3x3_dx_kernel<KC, NT, false, G2>), dev);
  if (rc != XMM_OK) return rc;
  const int grid = a.num_tiles < dev.sm_count ? a.num_tiles : dev.sm_count;
  // >= 4 strips per CTA: deal whole strips round-robin (halo rows of adjacent strips meet in L2); XMM_DX_RR=0/1 forces
  static const int rr_env = [] { const char* e = getenv("XMM_DX_RR"); return e ? atoi(e) : -1; }();
  const long long nstrips = (long long)a.tiles_y * p.batch;
  // (cin <= 64 is not DRAM-bound: there the round-robin's wave quantisation only pays off with many strips)
  a.strip_rr = rr_env >= 0 ? (rr_env != 0) : (nstrips >= 4LL * grid && (a.nchunks >= 3 || nstrips >= 16LL * grid));
  // Round-robin strips on an even grid: CTA pairs (cta_group::2, the weight operand split between the two SMs of a
  // TPC).  Opt-in (XMM_DX_PAIR=1): bit-identical and the MMA stream gets cheaper (49 vs 56 cycles), but the layers are
  // epilogue- (cin <= 96) or HBM-bound (cin >= 128), so the launch is not faster (profiles/r01_conv_prof_pair.log).
  static const int pair_env = [] { const char* e = getenv("XMM_DX_PAIR"); return e ? atoi(e) : 0; }();
  if constexpr (!G2)
  if (KC == 32 && NT == 32 && (pair_env || p.tap_mode == 6) && p.tap_mode != 5 && a.strip_rr && grid % 2 == 0 &&
      nstrips >= grid) {
    rc = ensure_max_smem(reinterpret_cast<const void*>(conv3x3_dx_kernel<KC, NT, true>), dev);
    if (rc != XMM_OK) return rc;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(unsigned(grid));
    cfg.blockDim = dim3(kDxThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    XMM_CUDA_OK(cudaLaunchKernelEx(&cfg, conv3x3_dx_kernel<KC, NT, true>, tmap, tmap_out, sides, a));
    return XMM_OK;
  }
  conv3x3_dx_kernel<KC, NT, false, G2><<<grid, kDxThreads, smem, stream>>>(tmap, tmap_out, sides, a);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

// Many round-robin strips per CTA (>= 16: inference batches), Cout = 32: two epilogue groups, two strips in flight per
// CTA (DxCfg::G2): +2.5 % at batch 64; with few strips the unpaired ones run at half the epilogue capacity (batch 16:
// -5 %), so those keep the single group (profiles/r01_dx_two_group_epilogue.log).  XMM_DX_G2=0 / tap_mode 5..7: off.
template <int KC, int NT>
int launch_conv_dx(const xmm_conv3x3_params& p, const DeviceInfo& dev, cudaStream_t stream) {
  if constexpr (NT == 32) {
    static const int g2_env = [] { const char* e = getenv("XMM_DX_G2"); return e ? atoi(e) : 1; }();
    static const int rr_env = [] { const char* e = getenv("XMM_DX_RR"); return e ? atoi(e) : -1; }();
    const int tiles_x = (p.width + kDxTileW - 1) / kDxTileW, tiles_y = (p.height + kDxTileH - 1) / kDxTileH;
    const long long ntiles = (long long)tiles_x * tiles_y * p.batch, nstrips = (long long)tiles_y * p.batch;
    const long long grid = ntiles < dev.sm_count ? ntiles : dev.sm_count;
    const int nchunks = p.cin / KC;
    const bool rr = rr_env >= 0 ? (rr_env != 0) : (nstrips >= 4LL * grid && (nchunks >= 3 || nstrips >= 16LL * grid));
    const bool g2 = (p.tap_mode == 8) || (g2_env && rr && nstrips >= 16LL * grid && (p.tap_mode <= 0 || p.tap_mode == 4));
    // (the second group's staging tiles cost 20 KB of shared memory: only where >= 6 activation stages remain)
    if (g2 && DxCfg<KC, NT, true>::smem_bytes(uint32_t(nchunks) * 9u * DxCfg<KC, NT, true>::kTapBytes,
                                               p.tap_mode == 8 ? 2 : 6,
                                               (p.mask != nullptr) + (p.r1 != nullptr) + (p.r2 != nullptr)) <=
                  size_t(dev.max_smem_optin))
      return launch_conv_dx_impl<KC, NT, true>(p, dev, stream);
  }
  return launch_conv_dx_impl<KC, NT, false>(p, dev, stream);
}


// ----------------------------------------------------------------------------- row-hop form (conv3x3_row.cuh)
struct BandTmapKey {
  const void* base;
  int batch, height, width, ctot, band_h, nbands, box_c, box_w, box_bands;
  bool operator==(const BandTmapKey& o) const {
    return base == o.base && batch == o.batch && height == o.height && width == o.width && ctot == o.ctot &&
           band_h == o.band_h && nbands == o.nbands && box_c == o.box_c && box_w == o.box_w && box_bands == o.box_bands;
  }
};
struct BandTmapKeyHash {
  size_t operator()(const BandTmapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.base);
    auto mix = [&h](size_t v) { h ^= v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2); };
    mix(k.batch); mix(k.height); mix(k.width); mix(k.ctot); mix(k.band_h); mix(k.nbands); mix(k.box_c); mix(k.box_w);
    mix(k.box_bands);
    return h;
  }
};
int cached_band_tmap(CUtensorMap* out, const void* base, int batch, int height, int width, int ctot, int band_h,
                     int nbands, int box_c, int box_w, int box_bands) {
  static std::mutex mu;
  static std::unordered_map<BandTmapKey, CUtensorMap, BandTmapKeyHash> cache;
  BandTmapKey key{base, batch, height, width, ctot, band_h, nbands, box_c, box_w, box_bands};
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(key);
  if (it != cache.end()) {
    *out = it->second;
    return XMM_OK;
  }
  int rc = make_band_tmap(out, base, batch, height, width, ctot, band_h, nbands, box_c, box_w, box_bands);
  if (rc != XMM_OK) return rc;
  if (cache.size() > 4096) cache.clear();
  cache.emplace(key, *out);
  return XMM_OK;
}

// height = nbands * band_h with the largest nbands <= 16 (lanes of missing bands idle: at least half must work)
bool row_bands(int height, int* nbands, int* band_h) {
  for (int n = kRowBands; n >= kRowBands / 2; --n)
    if (height % n == 0) {
      *nbands = n;
      *band_h = height / n;
      return true;
    }
  return false;
}

int row_epi_flags(const xmm_conv3x3_params& p) {
  return (p.lrelu_slope != 1.0f ? kRowLrelu : 0) | (p.mask ? kRowMask : 0) | (p.r1 ? kRowR1 : 0) | (p.r2 ? kRowR2 : 0) |
         (p.colsum ? kRowCsum : 0);
}
bool row_epi_built(int f) {
  switch (f) {
    case 0: case kRowLrelu: case kRowR1: case kRowR1 | kRowR2: case kRowMask: case kRowMask | kRowCsum: case kRowCsum:
    case kRowR1 | kRowCsum: case kRowR1 | kRowR2 | kRowCsum:
      return true;
    default:
      return false;
  }
}

// Why (if at all) this launch cannot take the row-hop form; nullptr = it can.  stages_out: activation stages.
template <int KC, int NT>
const char* row_blocker(const xmm_conv3x3_params& p, const DeviceInfo& dev, int* stages_out) {
  using Cfg = RowCfg<KC, NT>;
  if (p.wblob_row == nullptr) return "no row-hop weight image (wblob_row)";
  if (p.pixel_shuffle != 0) return "pixel shuffle";
  int nbands, band_h;
  if (!row_bands(p.height, &nbands, &band_h)) return "height has no divisor in 8..16";
  const int flags = row_epi_flags(p);
  if (!row_epi_built(flags)) return "epilogue combination not instantiated";
  if ((flags & kRowCsum) && NT != 32) return "fused column sums need cout = 32";
  const int nside = (p.mask != nullptr) + (p.r1 != nullptr) + (p.r2 != nullptr);
  const uint32_t w_bytes = uint32_t(p.cin / KC) * 9u * Cfg::kTapBytes;
  const size_t fixed = Cfg::smem_bytes(w_bytes, 0, nside);
  if (fixed + 3 * size_t(Cfg::kStageBytes) > size_t(dev.max_smem_optin)) return "weights do not fit next to 3 pipeline stages";
  int stages = int((size_t(dev.max_smem_optin) - fixed) / Cfg::kStageBytes);
  if (stages > kMaxStages) stages = kMaxStages;
  *stages_out = stages;
  return nullptr;
}

template <int KC, int NT, int EPI>
int launch_conv_row_epi(const xmm_conv3x3_params& p, const DeviceInfo& dev, cudaStream_t stream, int stages) {
  using Cfg = RowCfg<KC, NT>;
  RowArgs a{};
  a.wblob = p.wblob_row;
  a.nchunks = p.cin / KC;
  a.w_bytes = uint32_t(a.nchunks) * 9u * Cfg::kTapBytes;
  a.cin_off = p.in_coff;
  a.batch = p.batch;
  a.height = p.height;
  a.width = p.width;
  row_bands(p.height, &a.nbands, &a.band_h);
  a.tiles_x = (p.width + kRowPx - 1) / kRowPx;
  a.ncols = a.tiles_x * p.batch;
  a.stages = stages;
  const void* side_ptr[3] = {p.mask, p.r1, p.r2};
  const int side_ctot[3] = {p.mask_ctot, p.r1_ctot, p.r2_ctot};
  int nside = 0;
  for (int k = 0; k < 3; ++k)
    if (side_ptr[k] != nullptr) { a.side_mask |= 1 << k; ++nside; }
  fill_epilogue(a.epi, p);
  const long long total_rows = (long long)a.ncols * a.band_h;
  const int grid = total_rows < dev.sm_count ? int(total_rows) : dev.sm_count;
  // whole columns round-robin while they fill rounds (neighbouring columns run side by side: shared halo pixels meet
  // in L2), the rest as equal row ranges; XMM_ROW_RR=0 forces contiguous ranges only (experiments)
  static const int rr_env = [] { const char* e = getenv("XMM_ROW_RR"); return e ? atoi(e) : 1; }();
  a.rr_rounds = (rr_env && a.ncols >= 2 * grid) ? a.ncols / grid : 0;
  CUtensorMap tmap, tmap_out;
  int rc = cached_band_tmap(&tmap, p.in, p.batch, p.height, p.width, p.in_ctot, a.band_h, a.nbands, KC, kRowPitch, kRowBands);
  if (rc != XMM_OK) return rc;
  rc = cached_band_tmap(&tmap_out, p.out, p.batch, p.height, p.width, p.out_ctot, a.band_h, a.nbands, NT, kRowPx, 4);
  if (rc != XMM_OK) return rc;
  RowSideMaps sides;
  for (int k = 0; k < 3; ++k) {
    sides.m[k] = tmap;
    if (a.side_mask & (1 << k)) {
      rc = cached_band_tmap(&sides.m[k], side_ptr[k], p.batch, p.height, p.width, side_ctot[k], a.band_h, a.nbands, NT,
                            kRowPx, kRowBands);
      if (rc != XMM_OK) return rc;
    }
  }
  rc = ensure_max_smem(reinterpret_cast<const void*>(conv3x3_row_kernel<KC, NT, EPI>), dev);
  if (rc != XMM_OK) return rc;
  const size_t smem = Cfg::smem_bytes(a.w_bytes, stages, nside);
  conv3x3_row_kernel<KC, NT, EPI><<<grid, kRowThreads, smem, stream>>>(tmap, tmap_out, sides, a);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

template <int KC, int NT>
int launch_conv_row(const xmm_conv3x3_params& p, const DeviceInfo& dev, cudaStream_t stream, int stages) {
  switch (row_epi_flags(p)) {
#define XMM_ROW_CASE(F_) case (F_): return launch_conv_row_epi<KC, NT, (F_)>(p, dev, stream, stages);
    XMM_ROW_CASE(0)
    XMM_ROW_CASE(kRowLrelu)
    XMM_ROW_CASE(kRowR1)
    XMM_ROW_CASE(kRowR1 | kRowR2)
    XMM_ROW_CASE(kRowMask)
    default: break;
  }
  if constexpr (NT == 32) {
    switch (row_epi_flags(p)) {
      XMM_ROW_CASE(kRowCsum)
      XMM_ROW_CASE(kRowMask | kRowCsum)
      XMM_ROW_CASE(kRowR1 | kRowCsum)
      XMM_ROW_CASE(kRowR1 | kRowR2 | kRowCsum)
#undef XMM_ROW_CASE
      default: break;
    }
  }
  return fail(XMM_ERR_INVALID_ARGUMENT, "conv3x3 (row-hop): epilogue combination %d is not instantiated", row_epi_flags(p));
}

template <int KC, int NT>
int launch_conv_mode(const xmm_conv3x3_params& p, const DeviceInfo& dev, cudaStream_t stream) {
  const int mode = p.tap_mode <= 0 ? XMM_DEFAULT_TAP_MODE : p.tap_mode - 1;
  switch (mode) {
    case kTapHalo: return launch_conv<KC, NT, kTapHalo>(p, dev, stream);
    case kTapHaloBaseOff: return launch_conv<KC, NT, kTapHaloBaseOff>(p, dev, stream);
    case kTapDx3: return launch_conv<KC, NT, kTapDx3>(p, dev, stream);
    default: return fail(XMM_ERR_INVALID_ARGUMENT, "conv3x3: unknown tap_mode %d", mode);
  }
}

}  // namespace

namespace {
int check_conv_params(const xmm_conv3x3_params& p, const DeviceInfo& dev) {
  XMM_REQUIRE(p.in && p.out && p.wblob, "conv3x3: null tensor pointer");
  XMM_REQUIRE(p.batch > 0 && p.height > 0 && p.width > 0, "conv3x3: bad shape %dx%dx%d", p.batch, p.height, p.width);
  XMM_REQUIRE(p.kc == 32 || p.kc == 64, "conv3x3: kc must be 32 or 64 (got %d)", p.kc);
  XMM_REQUIRE(p.cin > 0 && p.cin % p.kc == 0, "conv3x3: cin=%d is not a multiple of kc=%d", p.cin, p.kc);
  XMM_REQUIRE(p.in_ctot % 8 == 0 && p.in_coff % 8 == 0 && p.in_coff + p.cin <= p.in_ctot,
              "conv3x3: input channel window [%d,%d) of %d", p.in_coff, p.in_coff + p.cin, p.in_ctot);
  XMM_REQUIRE(p.shuffle_stride == 0 || (p.pixel_shuffle == 2 && p.shuffle_stride >= p.cout && p.shuffle_stride % 8 == 0),
              "conv3x3: shuffle_stride is the inverse pixel shuffle's block distance (>= cout)");
  const int out_c = p.pixel_shuffle == 1 ? p.cout / 4
                    : (p.pixel_shuffle == 2 ? 3 * (p.shuffle_stride > 0 ? p.shuffle_stride : p.cout) + p.cout : p.cout);
  XMM_REQUIRE(p.pixel_shuffle >= 0 && p.pixel_shuffle <= 2, "conv3x3: pixel_shuffle must be 0, 1 or 2");
  XMM_REQUIRE(p.pixel_shuffle != 2 || (p.height % 2 == 0 && p.width % 2 == 0 && !p.r1 && !p.r2),
              "conv3x3: inverse pixel shuffle needs even height/width and no residual");
  XMM_REQUIRE(p.out_ctot % 8 == 0 && p.out_coff % 8 == 0 && p.out_coff + out_c <= p.out_ctot,
              "conv3x3: output channel window [%d,%d) of %d", p.out_coff, p.out_coff + out_c, p.out_ctot);
  XMM_REQUIRE(!p.mask || (p.mask_ctot % 8 == 0 && p.mask_coff % 8 == 0), "conv3x3: mask window alignment");
  XMM_REQUIRE(!p.r1 || (p.r1_ctot % 8 == 0 && p.r1_coff % 8 == 0), "conv3x3: r1 window alignment");
  XMM_REQUIRE(!p.r2 || (p.r2_ctot % 8 == 0 && p.r2_coff % 8 == 0), "conv3x3: r2 window alignment");
  XMM_REQUIRE(!p.colsum || (p.cout == 32 && p.pixel_shuffle == 0), "conv3x3: fused column sums need cout = 32");
  // every form that takes column sums launches at most dev.sm_count CTAs (the pipelined chain: all of its layers)
  XMM_REQUIRE(!p.colsum_ws || (p.colsum && p.colsum_ws_slots >= size_t(dev.sm_count) * kCsumWarpSlots &&
                               (reinterpret_cast<uintptr_t>(p.colsum_ws) & 3) == 0),
              "conv3x3: colsum_ws needs colsum and %zu slots (got %zu)", size_t(dev.sm_count) * kCsumWarpSlots,
              p.colsum_ws_slots);
  XMM_REQUIRE(p.pixel_shuffle != 1 || (!p.mask && !p.r1 && !p.r2 && p.cout % 128 == 0),
              "conv3x3: pixel_shuffle needs cout %% 128 == 0 and no mask/residual");
  XMM_REQUIRE((reinterpret_cast<uintptr_t>(p.in) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(p.wblob) & 15) == 0,
              "conv3x3: pointers must be 16-byte aligned");
  return XMM_OK;
}
}  // namespace

extern "C" int xmm_conv3x3_bf16(const xmm_conv3x3_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "conv3x3: null params");
  const xmm_conv3x3_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  rc = check_conv_params(p, dev);
  if (rc != XMM_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // Row-hop form (conv3x3_row.cuh): the default for the NARROW layers it qualifies for (tap_mode 0 with a row-hop
  // weight image and cin <= 64 * kc / 32).  Measured at batch 64, 416x416 (tools/row_probe.py, profiles/
  // r02_row_probe.log): cin 32 0.378 vs 0.426 ms (tap views), cin 64 0.565 vs 0.592 ms (column scatter); from cin 96
  // on its 10/8 column halo costs more HBM traffic than its cheap epilogue saves (cin 160: 1.12 vs 0.92 ms).
  // tap_mode 9 forces it; XMM_ROW=0 switches it off, XMM_ROW=2 lifts the cin limit (A/B runs).
  static const int row_env = [] { const char* e = getenv("XMM_ROW"); return e ? atoi(e) : 1; }();
  const bool row_narrow = p.cin <= 2 * p.kc || row_env == 2;
  if ((p.tap_mode <= 0 && row_env && row_narrow && p.wblob_row != nullptr) || p.tap_mode == 9) {
    const char* why = "cout must equal kc (32 or 64)";
    int stages = 0;
    if (p.kc == 32 && p.cout == 32) {
      why = row_blocker<32, 32>(p, dev, &stages);
      if (why == nullptr) return launch_conv_row<32, 32>(p, dev, s, stages);
    } else if (p.kc == 64 && p.cout == 64) {
      why = row_blocker<64, 64>(p, dev, &stages);
      if (why == nullptr) return launch_conv_row<64, 64>(p, dev, s, stages);
    }
    if (p.tap_mode == 9) return fail(XMM_ERR_UNSUPPORTED_SHAPE, "conv3x3: the row-hop form does not qualify (%s)", why);
  }
  // tap_mode 0 = auto: the column-scatter form (conv3x3_dx.cuh) wherever it is faster than the haloed tap views
  // (measured on B200, 16x416x416, F=32: cin 64..160 -> 1.13x..1.37x; cin = 32 ties; F=64 layers are faster on the
  // tap views, whose N=64 MMAs are less shared-memory bound).  4 forces it.
  const bool dx_auto = p.tap_mode <= 0 && p.kc == 32 && p.cout == 32 && p.cin >= 64 &&
                       DxCfg<32, 32>::smem_bytes(uint32_t(p.cin / 32) * 9u * DxCfg<32, 32>::kTapBytes, 4) <=
                           size_t(dev.max_smem_optin);  // >= 4 pipeline stages next to the resident weights
  if ((p.tap_mode >= 4 && p.tap_mode <= 8) || dx_auto) {  // 5 / 6: without / with CTA pairs, 7 / 8: one / two epilogue groups
    if (p.kc == 32 && p.cout == 32) return launch_conv_dx<32, 32>(p, dev, s);
    if (p.kc == 64 && p.cout == 64) return launch_conv_dx<64, 64>(p, dev, s);
    return fail(XMM_ERR_INVALID_ARGUMENT, "conv3x3: the column-scatter form is built for cout = kc = 32 or 64");
  }
#define XMM_CONV_CASE(KC_, NT_) \
  if (p.kc == KC_ && p.cout == NT_) return launch_conv_mode<KC_, NT_>(p, dev, s);
  XMM_CONV_CASE(32, 32)
  XMM_CONV_CASE(32, 128)
  XMM_CONV_CASE(64, 64)
  XMM_CONV_CASE(64, 256)
#undef XMM_CONV_CASE
  return fail(XMM_ERR_UNSUPPORTED_SHAPE, "conv3x3: no kernel for kc=%d cout=%d", p.kc, p.cout);
}

// ----------------------------------------------------------------------------- conv chain (dense block)
namespace {

struct Window {
  const void* base;
  int ctot, c0, c1;
};
bool overlaps(const Window& a, const Window& b) {
  return a.base && b.base && a.base == b.base && a.ctot == b.ctot && a.c0 < b.c1 && b.c0 < a.c1;
}
bool same(const Window& a, const Window& b) { return a.base == b.base && a.ctot == b.ctot && a.c0 == b.c0 && a.c1 == b.c1; }

// Can layers[0..n) run as one pipelined launch?  (Same image geometry, the column-scatter kernel's layer shape,
// and no hazard the strip-level dependency tracking does not cover.)
const char* chain_blocker(const xmm_conv3x3_params* L, int n) {
  if (n < 2 || n > kChainMaxLayers) return "2..5 layers";
  for (int l = 0; l < n; ++l) {
    const xmm_conv3x3_params& p = L[l];
    if (p.kc != 32 || p.cout != 32) return "kc = cout = 32 layers only";
    if (p.pixel_shuffle != 0) return "no pixel shuffle inside a chain";
    if (p.batch != L[0].batch || p.height != L[0].height || p.width != L[0].width) return "one image geometry";
    if (uint32_t(p.cin / 32) * 9u * DxCfg<32, 32>::kTapBytes > 160u * 1024u) return "weights must stay resident";
  }
  for (int l = 0; l < n; ++l) {
    const Window in{L[l].in, L[l].in_ctot, L[l].in_coff, L[l].in_coff + L[l].cin};
    const Window out{L[l].out, L[l].out_ctot, L[l].out_coff, L[l].out_coff + L[l].cout};
    const Window side[3] = {{L[l].mask, L[l].mask_ctot, L[l].mask_coff, L[l].mask_coff + L[l].cout},
                            {L[l].r1, L[l].r1_ctot, L[l].r1_coff, L[l].r1_coff + L[l].cout},
                            {L[l].r2, L[l].r2_ctot, L[l].r2_coff, L[l].r2_coff + L[l].cout}};
    if (overlaps(in, out)) return "a layer may not write its own input window";
    for (int m = 0; m < n; ++m) {
      const Window om{L[m].out, L[m].out_ctot, L[m].out_coff, L[m].out_coff + L[m].cout};
      if (m > l && overlaps(in, om)) return "a later layer overwrites an earlier layer's input";
      if (m != l && overlaps(out, om)) return "two layers write the same window";
      for (const Window& sd : side) {
        if (!sd.base) continue;
        if (m == l ? (overlaps(sd, om) && !same(sd, om)) : overlaps(sd, om))
          return "an epilogue input (mask / residual) is produced inside the chain";
      }
    }
  }
  return nullptr;
}

int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e && *e ? atoi(e) : dflt;
}

int launch_chain(const xmm_conv3x3_params* L, int n, const DeviceInfo& dev, int* done, cudaStream_t stream) {
  using Cfg = DxCfg<32, 32>;
  ChainArgs a{};
  ChainTmaps tm{};
  a.nlayers = n;
  a.batch = L[0].batch;
  a.height = L[0].height;
  a.width = L[0].width;
  a.tiles_x = (a.width + kDxTileW - 1) / kDxTileW;
  a.tiles_y = (a.height + kDxTileH - 1) / kDxTileH;
  int segs = env_int("XMM_CHAIN_SEGS", 2);
  if (segs < 1) segs = 1;
  if (segs > a.tiles_x) segs = a.tiles_x;
  a.segs = segs;
  a.done = done;
  const int nstrips = a.batch * a.tiles_y;
  const int grid = dev.sm_count;

  // CTAs per layer in proportion to the layer's per-tile cost: 6 MMAs of 56 cycles per 32 input channels, but
  // never less than the epilogue's three TMEM reads (48 KB at 64 B/clk).
  double cost[kChainMaxLayers], total = 0;
  for (int l = 0; l < n; ++l) {
    const int nch = L[l].cin / 32;
    cost[l] = 60.0 + 340.0 * nch;
    if (cost[l] < 850.0) cost[l] = 850.0;
    total += cost[l];
  }
  int cnt[kChainMaxLayers], used = 0;
  for (int l = 0; l < n; ++l) {
    cnt[l] = int(grid * cost[l] / total);
    if (cnt[l] < 1) cnt[l] = 1;
    used += cnt[l];
  }
  for (int l = n - 1; used < grid; l = (l + n - 1) % n) { ++cnt[l]; ++used; }   // leftovers to the heaviest layers
  for (int l = 0; used > grid; l = (l + 1) % n) if (cnt[l] > 1) { --cnt[l]; --used; }
  if (const char* e = getenv("XMM_CHAIN_SPLIT")) {  // "n0,n1,..." (experiments)
    int v[kChainMaxLayers], k = 0, sum = 0;
    for (const char* q = e; *q && k < n; ++k) {
      v[k] = atoi(q);
      sum += v[k];
      while (*q && *q != ',') ++q;
      if (*q == ',') ++q;
    }
    if (k == n && sum <= grid) {
      bool ok = true;
      for (int l = 0; l < n; ++l) ok = ok && v[l] >= 1;
      if (ok) for (int l = 0; l < n; ++l) cnt[l] = v[l];
    }
  }
  size_t smem = 0;
  int begin = 0;
  for (int l = 0; l < n; ++l) {
    ChainLayer& c = a.layer[l];
    c.wblob = L[l].wblob;
    c.nchunks = L[l].cin / 32;
    c.w_bytes = uint32_t(c.nchunks) * 9u * Cfg::kTapBytes;
    c.cin_off = L[l].in_coff;
    c.cta_begin = begin;
    c.cta_count = cnt[l];
    begin += cnt[l];
    const size_t fixed = Cfg::smem_bytes(c.w_bytes, 0);
    int stages = int((size_t(dev.max_smem_optin) - fixed) / Cfg::kStageBytes);
    if (stages > kMaxStages) stages = kMaxStages;
    c.stages = stages;
    const size_t need = Cfg::smem_bytes(c.w_bytes, stages);
    if (need > smem) smem = need;
    fill_epilogue(c.epi, L[l]);
    int rc = cached_tmap(&tm.m[l], L[l].in, a.batch, a.height, a.width, L[l].in_ctot, 32, kDxTileW, kDxPatchH);
    if (rc != XMM_OK) return rc;
    rc = cached_tmap(&tm.out[l], L[l].out, a.batch, a.height, a.width, L[l].out_ctot, Cfg::kWarpCols, kDxTileW, 2);
    if (rc != XMM_OK) return rc;
  }
  const int total_ctas = begin;
  XMM_CUDA_OK(cudaMemsetAsync(done, 0, size_t(n) * nstrips * sizeof(int), stream));
  {
    const int rc_attr = ensure_max_smem(reinterpret_cast<const void*>(conv3x3_chain_kernel<32, 32>), dev);
    if (rc_attr != XMM_OK) return rc_attr;
  }
  // XMM_CHAIN_PROF=1 (developer): per-layer-group cycle counters of this launch, printed after a device sync
  static const bool prof_on = env_int("XMM_CHAIN_PROF", 0) != 0;
  long long* prof_d = nullptr;
  if (prof_on) {
    XMM_CUDA_OK(cudaMalloc(&prof_d, size_t(total_ctas) * 4 * sizeof(long long)));
    XMM_CUDA_OK(cudaMemsetAsync(prof_d, 0, size_t(total_ctas) * 4 * sizeof(long long), stream));
    a.prof = prof_d;
  }
  void* kargs[2] = {&tm, &a};
  // cooperative: every CTA must be resident, later layers spin on earlier layers' progress
  XMM_CUDA_OK(cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(conv3x3_chain_kernel<32, 32>), dim3(total_ctas),
                                          dim3(kDxThreads), kargs, smem, stream));
  if (prof_on) {
    XMM_CUDA_OK(cudaStreamSynchronize(stream));
    std::vector<long long> h(size_t(total_ctas) * 4);
    XMM_CUDA_OK(cudaMemcpy(h.data(), prof_d, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    cudaFree(prof_d);
    for (int l = 0; l < n; ++l) {
      double tot = 0, dep = 0, idle = 0, tiles = 0;
      for (int c = a.layer[l].cta_begin; c < a.layer[l].cta_begin + a.layer[l].cta_count; ++c) {
        tot += double(h[size_t(c) * 4]); dep += double(h[size_t(c) * 4 + 1]);
        idle += double(h[size_t(c) * 4 + 2]); tiles += double(h[size_t(c) * 4 + 3]);
      }
      const double nc = a.layer[l].cta_count;
      fprintf(stderr, "chain layer %d: %3d CTAs, nchunks %d, stages %d | per CTA: total %.0f cyc, dependency wait %.0f, "
              "epilogue idle %.0f, tiles %.1f -> %.0f cyc/tile all-in, %.0f cyc/tile busy\n", l, a.layer[l].cta_count,
              a.layer[l].nchunks, a.layer[l].stages, tot / nc, dep / nc, idle / nc, tiles / nc, tot / tiles,
              (tot - idle) / tiles);
    }
  }
  return XMM_OK;
}

}  // namespace

extern "C" size_t xmm_conv3x3_chain_workspace_bytes(int nlayers, int batch, int height) {
  if (nlayers < 1 || batch < 1 || height < 1) return 0;
  return size_t(nlayers) * size_t(batch) * size_t((height + kDxTileH - 1) / kDxTileH) * sizeof(int);
}

// ----------------------------------------------------------------------------- fused dense block (conv3x3_rdb.cuh)
// Why (if at all) the five layers are not one ResidualDenseBlock_5C.forward the fused kernels can take; nullptr = ok.
const char* rdb_blocker(const xmm_conv3x3_params* L, int n, const DeviceInfo& dev) {
  if (n != 5) return "five layers";
  const xmm_conv3x3_params& p0 = L[0];
  if (p0.height < 8 || (p0.height & 1)) return "image height must be even (two bands) and >= 8";
  for (int k = 0; k < 5; ++k) {
    const xmm_conv3x3_params& p = L[k];
    if (p.kc != 32 || p.cout != 32) return "kc = cout = 32 layers only";
    if (p.pixel_shuffle != 0 || p.mask != nullptr || p.colsum != nullptr) return "no pixel shuffle / mask / column sums";
    if (p.wblob_row == nullptr) return "no row-hop weight image (wblob_row)";
    if (p.tap_mode > 0) return "a kernel form is forced (tap_mode)";
    if (p.batch != p0.batch || p.height != p0.height || p.width != p0.width) return "one image geometry";
    if (p.in != p0.in || p.in_ctot != p0.in_ctot || p.in_coff != p0.in_coff || p.cin != 32 * (k + 1))
      return "layer k must read channels [c0, c0 + 32 (k+1)) of one buffer";
    if (k < 4) {
      if (p.out != p0.in || p.out_ctot != p0.in_ctot || p.out_coff != p0.in_coff + 32 * (k + 1))
        return "layer k < 5 must write channels [c0 + 32 k, c0 + 32 (k+1)) of the same buffer";
      if (p.r1 != nullptr || p.r2 != nullptr || p.s0 != 1.0f) return "residuals only on the last layer";
    } else {
      if (p.out == p0.in && p.out_coff < p0.in_coff + 160 && p.out_coff + 32 > p0.in_coff)
        return "the last layer may not overwrite the block's own feature maps";
    }
  }
  if ((long long)p0.batch * p0.height * p0.width >= (1LL << 31)) return "more than 2^31 pixels";
  if (size_t(dev.max_smem_optin) < 232448) return "needs 227 KB of shared memory per CTA";
  return nullptr;
}

// PAIR: clusters of two CTAs that share every MMA (conv3x3_rdb.cuh): each holds half of the weights, so 14 instead of
// 5 TMA stages fit next to conv4 + conv5's, and an x0 ring of 11 rows next to conv1..conv3's.
template <int G, int NL, bool PAIR>
int launch_rdb(const xmm_conv3x3_params* L, const bool* store, const DeviceInfo& dev, cudaStream_t stream) {
  RdbArgs a{};
  uint32_t off = 0;
  for (int l = 0; l < NL; ++l) {
    const xmm_conv3x3_params& p = L[l];
    a.layer[l].wblob = p.wblob_row;
    a.layer[l].w_bytes = uint32_t(p.cin / 32) * 9u * uint32_t(kRdbTapBytes) / (PAIR ? 2u : 1u);
    a.layer[l].smem_off = off;
    off += (a.layer[l].w_bytes + 128u + 1023u) & ~1023u;
    a.layer[l].lrelu_slope = p.lrelu_slope;
    a.layer[l].store = store[l] ? 1 : 0;
    a.layer[l].out = static_cast<__nv_bfloat16*>(p.out);
    a.layer[l].out_ctot = p.out_ctot;
    a.layer[l].out_coff = p.out_coff;
  }
  a.w_total = off;
  const xmm_conv3x3_params& pl = L[NL - 1];
  a.cin_off = L[0].in_coff;
  a.batch = L[0].batch;
  a.height = L[0].height;
  a.width = L[0].width;
  a.band_h = a.height / 2;
  a.tiles_x = rdb_tiles_x<NL>(a.width);
  const long long ncols = (long long)a.batch * a.tiles_x;
  a.total_rows = (PAIR ? (ncols + 1) / 2 : ncols) * a.band_h;  // (pairs: rows of the pair-columns)
  a.s0 = pl.s0; a.s1 = pl.s1; a.s2 = pl.s2;
  a.r1 = static_cast<const __nv_bfloat16*>(pl.r1); a.r1_ctot = pl.r1_ctot; a.r1_coff = pl.r1_coff;
  a.r2 = static_cast<const __nv_bfloat16*>(pl.r2); a.r2_ctot = pl.r2_ctot; a.r2_coff = pl.r2_coff;
  static const int backoff_env = env_int("XMM_RDB_BACKOFF_NS", 0);
  static const int prefetch_env = env_int("XMM_RDB_PREFETCH_ROWS", 3);  // measured: 3.13 -> 3.06 ms per block at batch 64
  a.backoff_ns = backoff_env;
  a.prefetch_rows = prefetch_env;
  constexpr int kBarBytes = 1024;
  const long long room = (long long)dev.max_smem_optin - 1024 - kBarBytes - (long long)a.w_total;
  int tiles = int(room / kRdbTileBytes);
  a.ring0 = NL == 3 ? 5 : 2;  // (two fused layers: x4 is read one row behind its producer -- two tiles, one more TMA stage)
  a.ring1 = NL == 3 ? 3 : 0;
  a.stages = tiles - a.ring0 - a.ring1;
  if (a.stages > kRdbLRing<PAIR>) a.stages = kRdbLRing<PAIR>;
  static const int stages_env = env_int("XMM_RDB_STAGES", 0);
  if (stages_env > 0 && stages_env < a.stages) a.stages = stages_env;
  // (the x0 ring holds the rows between the last layer's and the first layer's step: tools/rdb_protocol_sim.py)
  const int min_stages = kRdbXRing<G, PAIR> ? 4 : 3;
  if (a.stages < min_stages)
    return fail(XMM_ERR_UNSUPPORTED_SHAPE, "conv3x3 (fused dense block): %d pipeline stages fit", a.stages);
  // measured (profiles/r02_rdb_v8_split_producers.log): 3.08 ms per block against 2.87 ms with one producer and one shared
  // ring -- rings of 3 + 2 stages are less elastic than one of 5 -- so it is off (and not built for pairs)
  static const int split_env = env_int("XMM_RDB_SPLIT_PRODUCERS", 0);
  a.split_producers = (!PAIR && NL == 2 && split_env && a.stages >= 4) ? 1 : 0;
  CUtensorMap tmap;
  int rc = cached_band_tmap(&tmap, L[0].in, a.batch, a.height, a.width, L[0].in_ctot, a.band_h, 2, 32, kRdbBoxPx, 2);
  if (rc != XMM_OK) return rc;
  const void* kernel = reinterpret_cast<const void*>(conv3x3_rdb_kernel<G, NL, PAIR>);
  rc = ensure_max_smem(kernel, dev);
  if (rc != XMM_OK) return rc;
  const size_t smem = 1024 + size_t(a.w_total) + size_t(a.stages + a.ring0 + a.ring1) * kRdbTileBytes + kBarBytes;
  static const int max_ctas = env_int("XMM_RDB_MAX_CTAS", 0);
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute attr[1];
  cfg.blockDim = dim3(kRdbThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  long long grid;
  if constexpr (PAIR) {
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // persistent: every pair must be resident at once (a second wave would double the time), so the grid is what the
    // device can co-schedule as clusters, not the SM count
    static int max_clusters = 0;
    if (max_clusters == 0) {
      cfg.gridDim = dim3(unsigned(2 * dev.sm_count));
      XMM_CUDA_OK(cudaOccupancyMaxActiveClusters(&max_clusters, conv3x3_rdb_kernel<G, NL, PAIR>, &cfg));
      if (max_clusters < 1) return fail(XMM_ERR_UNSUPPORTED_SHAPE, "conv3x3 (fused dense block): no CTA pair fits an SM pair");
    }
    long long pairs = a.total_rows < max_clusters ? a.total_rows : max_clusters;
    if (max_ctas > 0 && pairs > max_ctas / 2) pairs = max_ctas / 2 > 0 ? max_ctas / 2 : 1;
    grid = 2 * pairs;
  } else {
    grid = a.total_rows < dev.sm_count ? a.total_rows : dev.sm_count;
    if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  }
  cfg.gridDim = dim3(unsigned(grid));
  // XMM_RDB_PROF=1 (developer): per-CTA cycle counters of the issuer and the two epilogue groups, printed per launch
  static const int prof_env = XMM_RDB_PROFILE ? env_int("XMM_RDB_PROF", 0) : 0;
  static long long* prof_dev = nullptr;
  constexpr size_t kProfBytes = kRdbProfSlots * sizeof(long long) * 1024;
  if (prof_env) {
    if (prof_dev == nullptr) XMM_CUDA_OK(cudaMalloc(&prof_dev, kProfBytes));
    XMM_CUDA_OK(cudaMemsetAsync(prof_dev, 0, kProfBytes, stream));
    a.prof = prof_dev;
  }
  if constexpr (PAIR) {
    XMM_CUDA_OK(cudaLaunchKernelEx(&cfg, conv3x3_rdb_kernel<G, NL, PAIR>, tmap, a));
  } else {
    conv3x3_rdb_kernel<G, NL, PAIR><<<cfg.gridDim, kRdbThreads, smem, stream>>>(tmap, a);
    XMM_CUDA_OK(cudaGetLastError());
  }
  if (prof_env) {
    XMM_CUDA_OK(cudaStreamSynchronize(stream));
    std::vector<long long> h(size_t(grid) * kRdbProfSlots);
    XMM_CUDA_OK(cudaMemcpy(h.data(), prof_dev, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    static const char* names[kRdbProfSlots] = {
        "issuer total", "issuer wait drained", "issuer wait TMA", "issuer wait map row",
        "epi0 total", "epi0 wait row complete", "epi0 wait map slot", "epi0 rows",
        "epi1 total", "epi1 wait row complete", "epi1 wait map slot", "epi1 rows",
        "epi0 drain (ld+st+arrive)", "epi0 math+pack", "epi0 map write+fence+arrive", "epi0 global store",
        "epi1 drain (ld+st+arrive)", "epi1 math+residuals+pack", "epi1 map write (none)", "epi1 global store",
        "", "", "", ""};
    fprintf(stderr, "conv3x3_rdb<%d,%d%s> grid %lld stages %d:", G, NL, PAIR ? ",pair" : "", grid, a.stages);
    for (int k = 0; k < 20; ++k) {
      // (the issuer counters: of the CTAs that issue -- in pairs, the leaders)
      double sum = 0;
      int n = 0;
      for (long long c = 0; c < grid; ++c)
        if (k >= 4 || !PAIR || c % 2 == 0) {
          sum += double(h[size_t(c) * kRdbProfSlots + k]);
          ++n;
        }
      fprintf(stderr, " %s %.0f;", names[k], sum / n);
    }
    fprintf(stderr, "\n");
  }
  return XMM_OK;
}

// Which fused kernels run as CTA pairs, a bit mask: bit 0 conv1..conv3, bit 1 conv4..conv5.  XMM_RDB_PAIR (default 3,
// measured: DESIGN 4.3c), or per call the XMM_CHAIN_RDB_PAIR (both) / XMM_CHAIN_RDB_SINGLE (neither) flags.
int rdb_pair(int mode_flags) {
  if (mode_flags & XMM_CHAIN_RDB_PAIR) return 3;
  if (mode_flags & XMM_CHAIN_RDB_SINGLE) return 0;
  static const int pair_env = env_int("XMM_RDB_PAIR", 3);
  return pair_env & 3;
}

// conv1..conv3 in one launch, conv4..conv5 in a second one.  skip_dead: x4 is read by nobody after this block
// (inference), so it is never written.  pair: rdb_pair's mask.
int launch_rdb_block(const xmm_conv3x3_params* L, bool skip_dead, int pair, const DeviceInfo& dev, cudaStream_t stream) {
  const bool store_a[3] = {true, true, true};
  int rc = (pair & 1) ? launch_rdb<1, 3, true>(L, store_a, dev, stream) : launch_rdb<1, 3, false>(L, store_a, dev, stream);
  if (rc != XMM_OK) return rc;
  const bool store_b[2] = {!skip_dead, true};
  return (pair & 2) ? launch_rdb<4, 2, true>(L + 3, store_b, dev, stream) : launch_rdb<4, 2, false>(L + 3, store_b, dev, stream);
}

extern "C" int xmm_set_sm_reserve(int sms) {
  if (sms < 0) sms = 0;
  return sm_reserve().exchange(sms);
}

namespace {
thread_local int g_last_chain_launches = 0;
}
extern "C" int xmm_last_chain_launches(void) { return g_last_chain_launches; }

extern "C" int xmm_conv3x3_chain_bf16(const xmm_conv3x3_params* layers, int nlayers, int mode_flags, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  XMM_REQUIRE(layers != nullptr && nlayers >= 1, "conv3x3_chain: no layers");
  g_last_chain_launches = 0;
  const int mode = mode_flags & 0xff;
  const bool skip_dead = (mode_flags & XMM_CHAIN_SKIP_DEAD_STORES) != 0;
  constexpr int kFlags = XMM_CHAIN_SKIP_DEAD_STORES | XMM_CHAIN_RDB_PAIR | XMM_CHAIN_RDB_SINGLE;
  XMM_REQUIRE(mode >= 0 && mode <= 3 && (mode_flags & ~(0xff | kFlags)) == 0 &&
                  (mode_flags & (XMM_CHAIN_RDB_PAIR | XMM_CHAIN_RDB_SINGLE)) != (XMM_CHAIN_RDB_PAIR | XMM_CHAIN_RDB_SINGLE),
              "conv3x3_chain: mode must be 0 (auto), 1 (pipelined), 2 (layer by layer) or 3 (fused dense block), with at most "
              "one of the pair / single flags");
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  for (int l = 0; l < nlayers; ++l) {
    rc = check_conv_params(layers[l], dev);
    if (rc != XMM_OK) return rc;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // fused dense block (conv3x3_rdb.cuh): the default wherever the five layers are one ResidualDenseBlock_5C.forward
  static const int rdb_env = env_int("XMM_RDB", 1);
  if (mode == 3 || (mode == 0 && rdb_env)) {
    const char* why_not = rdb_blocker(layers, nlayers, dev);
    if (why_not == nullptr) {
      g_last_chain_launches = 2;
      return launch_rdb_block(layers, skip_dead, rdb_pair(mode_flags), dev, s);
    }
    if (mode == 3) return fail(XMM_ERR_UNSUPPORTED_SHAPE, "conv3x3_chain: cannot fuse the dense block (%s)", why_not);
  }
  const char* why = chain_blocker(layers, nlayers);
  bool pipelined = mode == 1 && why == nullptr;
  if (mode == 1 && why != nullptr) return fail(XMM_ERR_UNSUPPORTED_SHAPE, "conv3x3_chain: cannot pipeline (%s)", why);
  if (pipelined) {
    const size_t need = xmm_conv3x3_chain_workspace_bytes(nlayers, layers[0].batch, layers[0].height);
    XMM_REQUIRE(workspace != nullptr && workspace_bytes >= need && (reinterpret_cast<uintptr_t>(workspace) & 3) == 0,
                "conv3x3_chain: workspace of %zu bytes needed (got %zu)", need, workspace_bytes);
    g_last_chain_launches = 1;
    return launch_chain(layers, nlayers, dev, static_cast<int*>(workspace), s);
  }
  for (int l = 0; l < nlayers; ++l) {
    rc = xmm_conv3x3_bf16(&layers[l], stream);
    if (rc != XMM_OK) return rc;
  }
  g_last_chain_launches = nlayers;
  return XMM_OK;
}

// ----------------------------------------------------------------------------- transforms
extern "C" int xmm_normalize(const xmm_normalize_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "normalize: null params");
  const xmm_normalize_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  if (p.n == 0) return XMM_OK;
  XMM_REQUIRE(p.in && p.out, "normalize: null tensor pointer");
  XMM_REQUIRE(p.stretch_mode >= 0 && p.stretch_mode <= 3, "normalize: Stretching function %d is not implemented",
              p.stretch_mode);
  XMM_REQUIRE((reinterpret_cast<uintptr_t>(p.in) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0,
              "normalize: pointers must be 16-byte aligned");
  XMM_REQUIRE(!p.mask || p.mask_n > 0, "normalize: mask_n must be > 0 with a mask");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  NormalizeArgs a{};
  a.in = p.in; a.mask = p.mask; a.out = p.out; a.n = p.n; a.mask_n = p.mask_n; a.in_is_int32 = p.in_is_int32;
  a.pre_scale = p.pre_scale; a.max_val = p.max_val; a.mode = p.stretch_mode; a.dyn_max = p.scratch;
  if (!(p.max_val > 0.0f)) {
    XMM_REQUIRE(p.scratch != nullptr && !p.in_is_int32 && p.mask == nullptr,
                "normalize: the max_val <= 0 branch needs fp32 input, no mask and a scratch float");
    XMM_CUDA_OK(cudaMemsetAsync(p.scratch, 0, sizeof(float), s));
    max_kernel<<<dev.sm_count * 4, 256, 0, s>>>(static_cast<const float*>(p.in), p.n, p.pre_scale, p.scratch);
    XMM_CUDA_OK(cudaGetLastError());
  }
  const size_t threads = (p.n + 3) / 4;
  normalize_kernel<<<unsigned((threads + 255) / 256), 256, 0, s>>>(a);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_denormalize(const float* in, float* out, size_t n, size_t per_image, const float* max_vals_dev,
                               int max_n, int stretch_mode, void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  if (n == 0) return XMM_OK;
  XMM_REQUIRE(in && out && max_vals_dev, "denormalize: null tensor pointer");
  XMM_REQUIRE(stretch_mode >= 0 && stretch_mode <= 3, "denormalize: Stretching function %d is not implemented",
              stretch_mode);
  XMM_REQUIRE(max_n == 1 || (per_image > 0 && size_t(max_n) * per_image == n),
              "denormalize: %d max values do not match %zu elements of %zu per image", max_n, n, per_image);
  denormalize_kernel<<<unsigned((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in, out, n, per_image ? per_image : n, max_vals_dev, max_n, stretch_mode);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_restretch(const float* in, float* out, size_t n, int from_mode, int to_mode, void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  if (n == 0) return XMM_OK;
  XMM_REQUIRE(in && out, "restretch: null tensor pointer");
  XMM_REQUIRE(from_mode >= 0 && from_mode <= 3 && to_mode >= 0 && to_mode <= 3,
              "restretch: Stretching function %d -> %d is not implemented", from_mode, to_mode);
  XMM_REQUIRE((reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
              "restretch: pointers must be 16-byte aligned");
  const size_t threads = (n + 3) / 4;
  restretch_kernel<<<unsigned((threads + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, out, n, from_mode,
                                                                                                  to_mode);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_prepare_counts(const xmm_prepare_counts_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "prepare_counts: null params");
  const xmm_prepare_counts_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(p.nsrc >= 1 && p.nsrc <= 3 && p.src[0] && p.out, "prepare_counts: 1..3 source planes and an output");
  for (int k = 0; k < p.nsrc; ++k) XMM_REQUIRE(p.src[k] != nullptr, "prepare_counts: source plane %d is null", k);
  XMM_REQUIRE(p.batch > 0 && p.h > 0 && p.w > 0 && p.res_h > 0 && p.res_w > 0 && p.up >= 1,
              "prepare_counts: bad shape %dx%dx%d (x%d) -> %dx%d", p.batch, p.h, p.w, p.up, p.res_h, p.res_w);
  XMM_REQUIRE(p.max_val > 0.0f, "prepare_counts: max_val must be positive");
  XMM_REQUIRE(p.stretch_mode >= 0 && p.stretch_mode <= 3, "prepare_counts: Stretching function %d is not implemented",
              p.stretch_mode);
  PrepareCountsArgs a{};
  for (int k = 0; k < 3; ++k) a.src[k] = k < p.nsrc ? p.src[k] : nullptr;
  a.nsrc = p.nsrc; a.src_is_int32 = p.src_is_int32; a.mask = p.mask;
  a.batch = p.batch; a.h = p.h; a.w = p.w; a.up = p.up; a.res_h = p.res_h; a.res_w = p.res_w;
  a.pre_scale = p.pre_scale; a.pre_scale_dev = p.pre_scale_dev; a.max_val = p.max_val; a.mode = p.stretch_mode;
  a.out = p.out;
  const size_t n = size_t(p.batch) * p.res_h * p.res_w;
  prepare_counts_kernel<<<unsigned((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_image_upsample(const float* in, float* out, int n_img, int h, int w, int scale, void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(scale >= 1, "image_upsample: scale factor %d must be a positive integer", scale);
  const size_t n_out = size_t(n_img) * h * w * scale * scale;
  if (n_out == 0) return XMM_OK;
  XMM_REQUIRE(in && out, "image_upsample: null tensor pointer");
  image_upsample_kernel<<<unsigned((n_out + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, out, n_out,
                                                                                                   h, w, scale);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

// ----------------------------------------------------------------------------- first / last conv
extern "C" int xmm_conv_first(const xmm_conv_first_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "conv_first: null params");
  const xmm_conv_first_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(p.in && p.weight && p.out, "conv_first: null tensor pointer");
  XMM_REQUIRE(p.cin >= 1 && p.cin <= 4, "conv_first: in_channels=%d not in 1..4", p.cin);
  XMM_REQUIRE(p.batch > 0 && p.height > 0 && p.width > 0, "conv_first: bad shape");
  XMM_REQUIRE(p.out_ctot % 8 == 0 && p.out_coff % 8 == 0 && p.out_coff + p.filters <= p.out_ctot,
              "conv_first: output channel window");
  XMM_REQUIRE(!p.out2 || (p.out2_ctot % 8 == 0 && p.out2_coff % 8 == 0 && p.out2_coff + p.filters <= p.out2_ctot),
              "conv_first: second output channel window");
  ConvFirstArgs a{};
  a.in = p.in; a.w = p.weight; a.bias = p.bias;
  a.out = static_cast<__nv_bfloat16*>(p.out); a.out_ctot = p.out_ctot; a.out_coff = p.out_coff;
  a.out2 = static_cast<__nv_bfloat16*>(p.out2); a.out2_ctot = p.out2_ctot; a.out2_coff = p.out2_coff;
  a.batch = p.batch; a.cin = p.cin; a.height = p.height; a.width = p.width;
  a.gate = p.gate;
  a.mask = static_cast<const __nv_bfloat16*>(p.mask); a.mask_ctot = p.mask_ctot; a.mask_coff = p.mask_coff;
  a.mask_slope = p.mask_slope;
  XMM_REQUIRE(!p.mask || (p.mask_ctot % 8 == 0 && p.mask_coff % 8 == 0), "conv_first: mask window alignment");
  const size_t npix = size_t(p.batch) * p.height * p.width;
  const unsigned grid = unsigned((npix + 127) / 128);
  const size_t smem = (size_t(p.cin) * 9 + 1) * p.filters * sizeof(float);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (p.filters == 32) conv_first_kernel<32><<<grid, 128, smem, s>>>(a);
  else if (p.filters == 64) conv_first_kernel<64><<<grid, 128, smem, s>>>(a);
  else return fail(XMM_ERR_UNSUPPORTED_SHAPE, "conv_first: filters=%d (supported: 32, 64)", p.filters);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_conv_last(const xmm_conv_last_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "conv_last: null params");
  const xmm_conv_last_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(p.in && p.weight && p.out, "conv_last: null tensor pointer");
  XMM_REQUIRE(p.cout >= 1 && p.cout <= 4, "conv_last: out_channels=%d not in 1..4", p.cout);
  XMM_REQUIRE(p.batch > 0 && p.height > 0 && p.width > 0, "conv_last: bad shape");
  XMM_REQUIRE(p.in_ctot % 8 == 0 && p.in_coff % 8 == 0 && p.in_coff + p.filters <= p.in_ctot,
              "conv_last: input channel window");
  if (p.wblob != nullptr) {  // tensor-core path: an F -> 32-row split-precision layer with the image epilogue
    XMM_REQUIRE(p.filters % 32 == 0 && p.in_ctot % 8 == 0 && p.in_coff % 8 == 0 &&
                    (reinterpret_cast<uintptr_t>(p.wblob) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.in) & 15) == 0,
                "conv_last: tensor-core path needs filters %% 32 == 0 and 16-byte aligned buffers");
    xmm_conv3x3_params c{};
    c.in = p.in; c.in_ctot = p.in_ctot; c.in_coff = p.in_coff; c.cin = p.filters;
    c.wblob = p.wblob; c.kc = 32; c.cout = 32;
    c.batch = p.batch; c.height = p.height; c.width = p.width;
    c.lrelu_slope = 1.0f; c.s0 = 1.0f;
    c.out = p.out; c.out_ctot = 32; c.out_coff = 0;  // unused in image mode
    ImageOut img{p.out, p.residual, p.pre, p.cout, p.clamp};
    return launch_conv<32, 32, kTapHalo>(c, dev, static_cast<cudaStream_t>(stream), &img);
  }
  ConvLastArgs a{};
  a.in = static_cast<const __nv_bfloat16*>(p.in); a.in_ctot = p.in_ctot; a.in_coff = p.in_coff;
  a.w = p.weight; a.bias = p.bias; a.residual = p.residual; a.out = p.out; a.pre = p.pre;
  a.batch = p.batch; a.cout = p.cout; a.height = p.height; a.width = p.width; a.clamp = p.clamp;
  const size_t npix = size_t(p.batch) * p.height * p.width;
  const unsigned grid = unsigned((npix + 127) / 128);
  const size_t smem = size_t(p.cout) * 9 * p.filters * sizeof(float);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (p.filters == 32) conv_last_kernel<32><<<grid, 128, smem, s>>>(a);
  else if (p.filters == 64) conv_last_kernel<64><<<grid, 128, smem, s>>>(a);
  else return fail(XMM_ERR_UNSUPPORTED_SHAPE, "conv_last: filters=%d (supported: 32, 64)", p.filters);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

// ----------------------------------------------------------------------------- weight gradients
extern "C" size_t xmm_wgrad_workspace_bytes(void) {
  DeviceInfo d;
  int sms = 160;
  if (device_info(&d) == XMM_OK && d.sm_count > 0) sms = d.sm_count;
  return size_t(sms) * kWgWsFloatsPerCta * sizeof(float);
}

// CTA share of a stacked role relative to the max(n/2, 47)-cycles-per-MMA model (XMM_WG_STACKED_COST overrides).
static double wg_stacked_cost_scale() {
  static const double v = [] {
    const char* e = getenv("XMM_WG_STACKED_COST");
    return e ? atof(e) : 1.3;
  }();
  return v;
}

extern "C" int xmm_conv3x3_wgrad(const xmm_wgrad_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "wgrad: null params");
  const xmm_wgrad_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(p.x && p.dy && p.workspace, "wgrad: null tensor pointer");
  XMM_REQUIRE(p.batch > 0 && p.height > 0 && p.width > 0, "wgrad: bad shape");
  XMM_REQUIRE(p.x_ctot % 8 == 0 && p.dy_ctot % 8 == 0, "wgrad: channel counts must be multiples of 8");
  XMM_REQUIRE(p.nroles >= 1 && p.nroles <= kWgMaxRoles && p.ndst >= 1 && p.ndst <= 16, "wgrad: %d roles / %d dsts",
              p.nroles, p.ndst);
  XMM_REQUIRE(dev.sm_count >= p.nroles, "wgrad: fewer SMs than roles");
  static const int max_ctas_env = [] {  // experiments only: leave SMs idle to separate per-SM from chip-wide limits
    const char* e = getenv("XMM_WG_MAX_CTAS");
    return e ? atoi(e) : 0;
  }();
  if (max_ctas_env >= p.nroles && max_ctas_env < dev.sm_count) dev.sm_count = max_ctas_env;
  WgradArgs a{};
  WgradReduceArgs ra{};
  a.nroles = ra.nroles = p.nroles;
  double cost[kWgMaxRoles], total = 0;
  size_t max_stage = 0;
  for (int r = 0; r < p.nroles; ++r) {
    const xmm_wgrad_role& q = p.roles[r];
    XMM_REQUIRE(q.tap_begin >= 0 && q.tap_count >= 1 && q.tap_begin + q.tap_count <= 9, "wgrad: role %d taps", r);
    XMM_REQUIRE(q.n >= 16 && q.n % 16 == 0 && q.n <= 192 && q.tap_count * q.n <= 512,
                "wgrad: role %d needs %d x %d TMEM columns (max 512)", r, q.tap_count, q.n);
    XMM_REQUIRE(q.mode == 0 || q.mode == 1, "wgrad: role %d mode %d", r, q.mode);
    if (q.mode == 1)
      XMM_REQUIRE(q.tap_begin == 0 && q.tap_count == 3 && q.n == 96 && q.x_c0 + 32 <= p.x_ctot && q.y_c0 < p.dy_ctot,
                  "wgrad: stacked role %d must be 3 filter rows x (3 dx x 32 X channels)", r);
    XMM_REQUIRE((q.x_boxes == 1 || q.x_boxes == 2) && q.x_c0 % 8 == 0 && q.y_c0 % 8 == 0 && q.x_c0 < p.x_ctot &&
                    (q.mode == 1 || q.y_c0 + q.n <= ((p.dy_ctot + 63) / 64) * 64 + 64),
                "wgrad: role %d channel windows", r);
    WgradRole& w = a.roles[r];
    w.tap_begin = q.tap_begin; w.tap_count = q.tap_count; w.x_c0 = q.x_c0; w.x_boxes = q.x_boxes;
    w.y_c0 = q.y_c0; w.n = q.n; w.y_boxes = (q.n + 63) / 64; w.mode = q.mode;
    static const int rows8_env = [] { const char* e = getenv("XMM_WG_ROWS8"); return e ? atoi(e) : 1; }();
    w.rows8 = (q.mode == 0 && rows8_env && q.tap_begin / 3 == (q.tap_begin + q.tap_count - 1) / 3) ? 1 : 0;
    const double per_mma = q.n / 2.0 > 47.0 ? q.n / 2.0 : 47.0;  // measured tcgen05 floor, profiles/r01_probe1
    cost[r] = q.tap_count * per_mma * (q.mode == 1 ? wg_stacked_cost_scale() : 1.0);
    total += cost[r];
    const size_t st = q.mode == 1 ? size_t(w.x_boxes) * kWgBoxYBytes + size_t(kWgBoxX32Bytes)
                                  : size_t(w.x_boxes) * (w.rows8 ? kWgBoxX8Bytes : kWgBoxXBytes) +
                                        size_t(w.y_boxes) * kWgBoxYBytes;
    if (st > max_stage) max_stage = st;
  }
  int assigned = 0;
  for (int r = 0; r < p.nroles; ++r) {
    int c = int(dev.sm_count * cost[r] / total);
    if (c < 1) c = 1;
    a.roles[r].cta_count = c;
    assigned += c;
  }
  for (int r = 0; assigned != dev.sm_count; r = (r + 1) % p.nroles) {  // distribute the rounding remainder
    if (assigned < dev.sm_count) { ++a.roles[r].cta_count; ++assigned; }
    else if (a.roles[r].cta_count > 1) { --a.roles[r].cta_count; --assigned; }
  }
  int begin = 0;
  for (int r = 0; r < p.nroles; ++r) {
    a.roles[r].cta_begin = begin;
    begin += a.roles[r].cta_count;
    ra.roles[r] = a.roles[r];
  }
  a.batch = p.batch; a.height = p.height; a.width = p.width;
  a.tiles_x = (p.width + kTileW - 1) / kTileW;
  a.tiles_y = (p.height + kWgTileH - 1) / kWgTileH;
  a.num_tiles = a.tiles_x * a.tiles_y * p.batch;
  a.ws = p.workspace;
  int wg_stages = int((size_t(dev.max_smem_optin) - 2048) / max_stage);
  if (wg_stages > kWgMaxStages) wg_stages = kWgMaxStages;
  XMM_REQUIRE(wg_stages >= 2, "wgrad: stage of %zu B does not fit twice in shared memory", max_stage);
  a.stages = wg_stages;
  const size_t smem = 1024 + size_t(wg_stages) * max_stage;

  ra.ws = p.workspace;
  ra.ndst = p.ndst;
  for (int i = 0; i < p.ndst; ++i) {
    const xmm_wgrad_dst& q = p.dst[i];
    XMM_REQUIRE(q.dw && q.role >= 0 && q.role < p.nroles && q.i_begin >= 0 && q.i_end > q.i_begin &&
                    q.i_end <= q.i_total && q.lane0 >= 0 && q.col0 >= 0,
                "wgrad: destination %d is inconsistent with its role", i);
    if (p.roles[q.role].mode == 1)
      XMM_REQUIRE(q.lane0 + q.o_count <= 64 * p.roles[q.role].x_boxes && q.col0 + (q.i_end - q.i_begin) <= 32,
                  "wgrad: destination %d does not fit its stacked role", i);
    else
      XMM_REQUIRE(q.lane0 + (q.i_end - q.i_begin) <= 128 && q.col0 + q.o_count <= p.roles[q.role].n,
                  "wgrad: destination %d is inconsistent with its role", i);
    WgradDst& d = ra.dst[i];
    d.dw = q.dw; d.o_count = q.o_count; d.i_total = q.i_total; d.i_begin = q.i_begin; d.i_end = q.i_end;
    d.role = q.role; d.lane0 = q.lane0; d.col0 = q.col0; d.scale = q.scale; d.accumulate = q.accumulate; d.perm = q.perm;
    d.o_begin = q.o_begin; d.o_total = q.o_total > 0 ? q.o_total : q.o_count;
    XMM_REQUIRE(q.o_begin >= 0 && q.o_begin + q.o_count <= d.o_total, "wgrad: destination %d output-channel window", i);
  }

  CUtensorMap tx, ty, tx32, tx8;
  rc = cached_tmap(&tx, p.x, p.batch, p.height, p.width, p.x_ctot, 64, kTileW + 2, kWgTileH + 2);
  if (rc != XMM_OK) return rc;
  rc = cached_tmap(&tx32, p.x, p.batch, p.height, p.width, p.x_ctot, 32, kTileW + 2, kWgTileH + 2);  // SWIZZLE_64B
  if (rc != XMM_OK) return rc;
  rc = cached_tmap(&tx8, p.x, p.batch, p.height, p.width, p.x_ctot, 64, kTileW + 2, kWgTileH);  // single-filter-row roles
  if (rc != XMM_OK) return rc;
  rc = cached_tmap(&ty, p.dy, p.batch, p.height, p.width, p.dy_ctot, 64, kTileW, kWgTileH);
  if (rc != XMM_OK) return rc;
  rc = ensure_max_smem(reinterpret_cast<const void*>(wgrad_tc_kernel), dev, 1024);  // the kernel also has static shared memory
  if (rc != XMM_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  wgrad_tc_kernel<<<dev.sm_count, kWgThreads, smem, s>>>(tx, ty, tx32, tx8, a);
  XMM_CUDA_OK(cudaGetLastError());
  wgrad_reduce_kernel<<<dim3(24, p.ndst), 256, 0, s>>>(ra, a.num_tiles);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

namespace {
// Grid of one colsum launch: >= 8 pixels per thread, at most 8 CTAs per SM.
unsigned colsum_grid(size_t npix, int groups, const DeviceInfo& dev) {
  const int ppb = kColsumThreads / groups;
  const size_t want = (npix + size_t(ppb) * 8 - 1) / (size_t(ppb) * 8);
  const size_t cap = size_t(dev.sm_count) * 8;
  return unsigned(want < 1 ? 1 : (want > cap ? cap : want));
}

int colsum_launch(const void* in, int ctot, size_t npix, const xmm_colsum_segment* segs, int nseg, float* ws,
                  size_t ws_slots, void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(in && segs && nseg >= 1 && nseg <= kColsumMaxSeg, "colsum: 1..%d segments", kColsumMaxSeg);
  XMM_REQUIRE(ctot % 8 == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0, "colsum: input alignment");
  ColsumArgs a{};
  a.in = static_cast<const __nv_bfloat16*>(in);
  a.ctot = ctot;
  a.npix = npix;
  a.nseg = nseg;
  a.ws = ws;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int groups = 0;
  for (int i = 0; i < nseg; ++i) {
    const xmm_colsum_segment& g = segs[i];
    XMM_REQUIRE((ws != nullptr || g.out != nullptr) && g.n > 0 && g.n % 8 == 0 && g.c0 % 8 == 0 && g.c0 >= 0 &&
                    g.c0 + g.n <= ctot,
                "colsum: channel window [%d,%d) of %d", g.c0, g.c0 + g.n, ctot);
    a.seg[i].c0 = g.c0; a.seg[i].n = g.n; a.seg[i].out = g.out; a.seg[i].scale = g.scale;
    a.seg[i].group0 = groups;
    groups += g.n / 8;
    if (ws == nullptr && !g.accumulate) XMM_CUDA_OK(cudaMemsetAsync(g.out, 0, size_t(g.n) * sizeof(float), s));
  }
  XMM_REQUIRE(groups <= kColsumThreads, "colsum: %d channels in one call (max %d)", groups * 8, kColsumThreads * 8);
  a.ngroups = groups;
  if (npix == 0) return XMM_OK;
  const unsigned grid = colsum_grid(npix, groups, dev);
  XMM_REQUIRE(ws == nullptr || (ws_slots >= grid && (reinterpret_cast<uintptr_t>(ws) & 3) == 0),
              "colsum: %u workspace slots needed (got %zu)", grid, ws_slots);
  colsum_multi_kernel<<<grid, kColsumThreads, 0, s>>>(a);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

// Rows of one image per edge_wgrad CTA: as many as fit 40 KB of staged s rows (+ halo), at most 8 (0: too wide).
int edge_rows(int height, int width) {
  int rows = int((40 * 1024) / (size_t(width + 2) * sizeof(float))) - 2;
  if (rows > 8) rows = 8;
  if (rows > height) rows = height;
  return rows;
}
}  // namespace

extern "C" int xmm_colsum_multi_bf16(const void* in, int ctot, size_t npix, const xmm_colsum_segment* segs, int nseg,
                                     void* stream) {
  return colsum_launch(in, ctot, npix, segs, nseg, nullptr, 0, stream);
}

extern "C" int xmm_colsum_multi_det_bf16(const void* in, int ctot, size_t npix, const xmm_colsum_segment* segs,
                                         int nseg, float* ws, size_t ws_slots, void* stream) {
  XMM_REQUIRE(ws != nullptr, "colsum (deterministic): null workspace");
  return colsum_launch(in, ctot, npix, segs, nseg, ws, ws_slots, stream);
}

extern "C" int xmm_colsum_bf16(const void* in, int ctot, int c0, int n, size_t npix, float* out, float scale,
                               int accumulate, void* stream) {
  xmm_colsum_segment g{c0, n, out, scale, accumulate};
  return xmm_colsum_multi_bf16(in, ctot, npix, &g, 1, stream);
}

extern "C" size_t xmm_det_slots(int site, int batch, int height, int width, int channels) {
  DeviceInfo dev;
  if (require_sm100(&dev) != XMM_OK || batch < 1 || height < 1 || width < 1 || channels < 8) return 0;
  switch (site) {
    case XMM_DET_CONV3X3: return size_t(dev.sm_count) * kCsumWarpSlots;
    case XMM_DET_COLSUM:
      return channels / 8 > kColsumThreads ? 0 : colsum_grid(size_t(batch) * height * width, channels / 8, dev);
    case XMM_DET_EDGE_WGRAD: {
      const int rows = edge_rows(height, width);
      return rows < 1 ? 0 : size_t((height + rows - 1) / rows) * size_t(batch);
    }
    default: return 0;
  }
}

extern "C" int xmm_det_finalize(const xmm_det_job* jobs_dev, int njobs, int max_n, float* dst_base, void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(jobs_dev != nullptr && dst_base != nullptr && njobs >= 1 && njobs <= 65535 && max_n >= 1,
              "det_finalize: %d jobs (1..65535), max_n %d", njobs, max_n);
  const dim3 grid(unsigned((max_n + kDetFinalizeThreads - 1) / kDetFinalizeThreads), unsigned(njobs));
  det_finalize_kernel<<<grid, kDetFinalizeThreads, 0, static_cast<cudaStream_t>(stream)>>>(jobs_dev, dst_base);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_edge_wgrad(const xmm_edge_wgrad_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "edge_wgrad: null params");
  const xmm_edge_wgrad_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(p.s && p.v && (p.r || p.ws), "edge_wgrad: null tensor pointer");
  XMM_REQUIRE(p.ns >= 1 && p.ns <= 4 && p.batch > 0 && p.height > 0 && p.width > 0, "edge_wgrad: bad shape");
  EdgeWgradArgs a{};
  a.s = p.s; a.gate = p.gate;
  a.v = static_cast<const __nv_bfloat16*>(p.v); a.v_ctot = p.v_ctot; a.v_coff = p.v_coff;
  a.v2 = static_cast<const __nv_bfloat16*>(p.v2); a.v2_ctot = p.v2_ctot; a.v2_coff = p.v2_coff;
  a.r = p.r; a.ssum = p.ssum; a.batch = p.batch; a.ns = p.ns; a.height = p.height; a.width = p.width;
  a.ws = p.ws;
  XMM_REQUIRE(p.v_ctot % 8 == 0 && p.v_coff % 8 == 0 && (!p.v2 || (p.v2_ctot % 8 == 0 && p.v2_coff % 8 == 0)),
              "edge_wgrad: channel windows must be 8-channel aligned");
  XMM_REQUIRE(p.channels == 32 || p.channels == 64, "edge_wgrad: channels=%d (supported: 32, 64)", p.channels);
  const size_t red_bytes = size_t(kEdgeWgradThreads / 32) * p.channels * 9 * sizeof(float);
  const int rows = edge_rows(p.height, p.width);
  XMM_REQUIRE(rows >= 1, "edge_wgrad: image width %d too large for the shared-memory row staging", p.width);
  a.rows = rows;
  const size_t smem = size_t(rows + 2) * (p.width + 2) * sizeof(float) + red_bytes;
  const dim3 grid(unsigned((p.height + rows - 1) / rows), unsigned(p.batch));
  XMM_REQUIRE(!p.ws || (p.ws_slots >= size_t(grid.x) * grid.y && (reinterpret_cast<uintptr_t>(p.ws) & 3) == 0),
              "edge_wgrad: %zu workspace slots needed (got %zu)", size_t(grid.x) * grid.y, p.ws_slots);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (p.channels == 32) {
    static bool attr32 = false;
    if (!attr32) {
      XMM_CUDA_OK(cudaFuncSetAttribute(edge_wgrad_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
      attr32 = true;
    }
    edge_wgrad_kernel<32><<<grid, kEdgeWgradThreads, smem, s>>>(a);
  } else {
    static bool attr64 = false;
    if (!attr64) {
      XMM_CUDA_OK(cudaFuncSetAttribute(edge_wgrad_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
      attr64 = true;
    }
    edge_wgrad_kernel<64><<<grid, kEdgeWgradThreads, smem, s>>>(a);
  }
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

// ----------------------------------------------------------------------------- losses
static_assert(sizeof(xmm_scale_stats) == sizeof(ScaleStats), "xmm_scale_stats mirrors ScaleStats");
static const int kLossBlocks = 592;  // 4 x 148

extern "C" size_t xmm_loss_workspace_floats(void) { return size_t(kLossBlocks) * 8; }

extern "C" int xmm_loss_reduce(const float* preds, const float* target, size_t n, float* sums_dev,
                               xmm_scale_stats* stats_dev, float* workspace, void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(preds && target && workspace && n > 0, "loss_reduce: null pointer or empty input");
  XMM_REQUIRE((reinterpret_cast<uintptr_t>(preds) & 15) == 0 && (reinterpret_cast<uintptr_t>(target) & 15) == 0,
              "loss_reduce: pointers must be 16-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  size_t need = (n + 1023) / 1024;
  const int blocks = int(need < size_t(kLossBlocks) ? need : size_t(kLossBlocks));
  loss_reduce_kernel<<<blocks, 256, 0, s>>>(preds, target, n, workspace);
  XMM_CUDA_OK(cudaGetLastError());
  loss_reduce_finalize_kernel<<<1, 32, 0, s>>>(workspace, blocks, sums_dev, reinterpret_cast<ScaleStats*>(stats_dev));
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_loss_grad(const float* preds, const float* target, size_t n, const float* coef_dev,
                             const float* gl_dev, float* grad, int accumulate, void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(preds && target && coef_dev && grad, "loss_grad: null pointer");
  if (n == 0) return XMM_OK;
  loss_grad_kernel<<<unsigned((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(preds, target, n, coef_dev,
                                                                                            gl_dev, grad, accumulate);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_avgpool2_pair(const float* preds, const float* target, float* preds_out, float* target_out,
                                 int nimg, int h, int w, void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(preds && target && preds_out && target_out, "avgpool2: null pointer");
  const size_t n = size_t(nimg) * (h / 2) * (w / 2);
  if (n == 0) return XMM_OK;
  avgpool2_pair_kernel<<<unsigned((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      preds, target, preds_out, target_out, nimg, h, w);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_ssim_prepare(const float* preds, size_t n, xmm_scale_stats* stats_dev, float k1, float k2,
                                void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(preds && stats_dev && n > 0, "ssim_prepare: null pointer or empty input");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  ssim_constants_kernel<<<1, 32, 0, s>>>(reinterpret_cast<ScaleStats*>(stats_dev), k1, k2);
  XMM_CUDA_OK(cudaGetLastError());
  size_t need = (n + 255) / 256;
  const int blocks = int(need < size_t(kLossBlocks) ? need : size_t(kLossBlocks));
  count_ties_kernel<<<blocks, 256, 0, s>>>(preds, n, reinterpret_cast<ScaleStats*>(stats_dev));
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_ssim_tiles(int h, int w) {
  const int vh = h - 2 * kSsimPad, vw = w - 2 * kSsimPad;
  if (vh <= 0 || vw <= 0) return 0;
  return ((vh + kSsimTileH - 1) / kSsimTileH) * ((vw + kSsimTileW - 1) / kSsimTileW);
}

extern "C" int xmm_ssim_stats(const xmm_ssim_stats_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "ssim_stats: null params");
  const xmm_ssim_stats_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(p.preds && p.target && p.stats_dev, "ssim_stats: null pointer");
  XMM_REQUIRE(p.h > 2 * kSsimPad && p.w > 2 * kSsimPad && p.nimg > 0 && p.nimg <= 65535,
              "ssim_stats: image %dx%d is not larger than the %d-tap Gaussian window", p.h, p.w, kSsimTaps);
  XMM_REQUIRE((p.kimg == nullptr) == (p.acc != nullptr), "ssim_stats: give acc (forward) or kimg+ga/gb/gc (backward)");
  XMM_REQUIRE(p.kimg == nullptr || (p.ga && p.gb && p.gc), "ssim_stats: backward needs ga, gb, gc");
  SsimArgs a{};
  a.p = p.preds; a.t = p.target; a.nimg = p.nimg; a.h = p.h; a.w = p.w;
  a.st = reinterpret_cast<const ScaleStats*>(p.stats_dev);
  for (int i = 0; i < kSsimTaps; ++i) a.win.w[i] = p.window[i];
  a.acc = p.acc; a.use_sim = p.use_sim; a.kimg = p.kimg; a.ga = p.ga; a.gb = p.gb; a.gc = p.gc;
  const int vh = p.h - 2 * kSsimPad, vw = p.w - 2 * kSsimPad;
  dim3 grid((vw + kSsimTileW - 1) / kSsimTileW, (vh + kSsimTileH - 1) / kSsimTileH, p.nimg);
  ssim_stats_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_ssim_grad(const xmm_ssim_grad_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "ssim_grad: null params");
  const xmm_ssim_grad_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(p.preds && p.target && p.stats_dev && p.ga && p.gb && p.gc && p.grad, "ssim_grad: null pointer");
  XMM_REQUIRE(p.h > 2 * kSsimPad && p.w > 2 * kSsimPad && p.nimg > 0 && p.nimg <= 65535, "ssim_grad: bad shape");
  SsimGradArgs a{};
  a.p = p.preds; a.t = p.target; a.nimg = p.nimg; a.h = p.h; a.w = p.w;
  a.st = reinterpret_cast<const ScaleStats*>(p.stats_dev);
  for (int i = 0; i < kSsimTaps; ++i) a.win.w[i] = p.window[i];
  a.ga = p.ga; a.gb = p.gb; a.gc = p.gc; a.coarse = p.coarse; a.grad = p.grad; a.accumulate = p.accumulate;
  dim3 grid((p.w + kSsimTileW - 1) / kSsimTileW, (p.h + kSsimTileH - 1) / kSsimTileH, p.nimg);
  ssim_grad_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

extern "C" int xmm_msssim_finalize(const xmm_msssim_finalize_params* pp, void* stream) {
  XMM_REQUIRE(pp != nullptr, "msssim_finalize: null params");
  const xmm_msssim_finalize_params& p = *pp;
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(p.nscales >= 1 && p.nscales <= kMaxScales && p.batch >= 1 && p.batch <= 1024 && p.channels >= 1,
              "msssim_finalize: %d scales, batch %d", p.nscales, p.batch);
  XMM_REQUIRE(p.stats_dev && p.value && p.img_val && p.kimg, "msssim_finalize: null pointer");
  MsFinalizeArgs a{};
  for (int s = 0; s < p.nscales; ++s) {
    XMM_REQUIRE(p.acc[s] && p.tiles[s] > 0 && p.nvalid[s] > 0, "msssim_finalize: scale %d is empty", s);
    a.acc[s] = p.acc[s]; a.tiles[s] = p.tiles[s]; a.nvalid[s] = p.nvalid[s]; a.betas[s] = p.betas[s];
  }
  a.nscales = p.nscales; a.batch = p.batch; a.channels = p.channels; a.k1 = p.k1; a.k2 = p.k2;
  a.st = reinterpret_cast<ScaleStats*>(p.stats_dev);
  a.value = p.value; a.img_val = p.img_val; a.kimg = p.kimg; a.gl = p.gl_dev; a.weight = p.weight;
  const size_t fin_smem = size_t(3) * p.nscales * p.batch * p.channels * sizeof(float);
  XMM_REQUIRE(fin_smem <= 40 * 1024, "msssim_finalize: batch*channels=%d too large for the single-block reduction",
              p.batch * p.channels);
  msssim_finalize_kernel<<<1, 256, fin_smem, static_cast<cudaStream_t>(stream)>>>(a);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}

// ----------------------------------------------------------------------------- optimizer
extern "C" int xmm_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                             float beta1, float beta2, float eps, int step, float grad_scale, void* stream) {
  DeviceInfo dev;
  int rc = require_sm100(&dev);
  if (rc != XMM_OK) return rc;
  XMM_REQUIRE(params && grads && exp_avg && exp_avg_sq, "adam: null pointer");
  XMM_REQUIRE(step >= 1, "adam: step count starts at 1 (got %d)", step);
  if (n == 0) return XMM_OK;
  const double bc1 = 1.0 - pow(double(beta1), double(step));
  const double bc2 = 1.0 - pow(double(beta2), double(step));
  adam_kernel<<<unsigned((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, float(bc1), float(sqrt(bc2)), grad_scale);
  XMM_CUDA_OK(cudaGetLastError());
  return XMM_OK;
}
