/* xmm_b200.h -- C ABI of libxmm_b200.so: the B200 (sm_100a) kernels behind the RRDB hot
 * path of SamSweere/xmm-superres-denoise.
 *
 * The reference is pure Python; it has no FFI of its own.  Each entry point below names
 * the reference code (path:line under xmm_superres_denoise/) whose arithmetic it
 * replaces.  The Python host layer (xmm_superres_denoise_b200/) binds these with ctypes
 * and keeps the reference's class/function names; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless a name ends in _host.  Buffers are owned
 *     by the caller and only borrowed for the duration of the call; the library keeps no
 *     pointer except cached TMA descriptors keyed by (pointer, shape).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *     Every call is asynchronous with respect to the host.
 *   - Return value: 0 on success, otherwise an XMM_ERR_* code; xmm_last_error() returns a
 *     thread-local human-readable message.  There is no CPU fallback anywhere.
 *   - Activations are NHWC bf16 "channel-window" tensors: a base pointer, the number of
 *     channels per pixel of the underlying buffer (ctot) and the first channel (coff).
 *     This is how the dense-block torch.cat (rrdb_blocks.py:49-52) disappears.
 */
#ifndef XMM_B200_H_
#define XMM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XMM_OK 0
#define XMM_ERR_INVALID_ARGUMENT 1
#define XMM_ERR_UNSUPPORTED_DEVICE 2
#define XMM_ERR_CUDA 3
#define XMM_ERR_UNSUPPORTED_SHAPE 4

/* Library / device ------------------------------------------------------------------ */
const char* xmm_last_error(void);
int xmm_version(void);
/* 0 iff the current device is compute capability 10.x (sm_100a image present). */
int xmm_check_device(void);
/* Persistent kernels launch on (SM count - sms) CTAs from now on; returns the previous value.  Used by the data-parallel
 * training step (training.TrainStep, replacing Lightning's DDP of train.py:148-155) while NCCL's all-reduce kernels
 * share the GPU with the backward pass: a 148-CTA grid whose work was divided for 148 resident CTAs would otherwise
 * run its last CTAs as a second wave.  0 restores the full GPU. */
int xmm_set_sm_reserve(int sms);

/* Weight repacking ------------------------------------------------------------------- */
/* One source tensor contributing a run of K (input-channel) positions of a packed layer.
 * src is an nn.Conv2d weight, fp32 OIHW [O][src_cin][3][3].
 *   transpose == 0 (forward):  packed row n = O index o_off+n, packed k = I index i_off+c
 *   transpose == 1 (data grad): packed row n = I index i_off+n, packed k = O index o_off+c,
 *                               taps flipped (dL/dx of a correlation is a convolution)   */
typedef struct {
  const float* src;
  int src_cin;
  int o_off, i_off;
  int transpose;
  int k_off, k_count;  /* K positions [k_off, k_off+k_count) of the packed layer                */
  float scale;
  int n_off, n_count;  /* rows [n_off, n_off+n_count) of the packed layer; the segment's own row
                          index is n - n_off                                                    */
  int part;            /* 0: bf16(w); 1: bf16(w - bf16(w)), the low-order half of a split-precision
                          layer (conv_last on the tensor cores keeps fp32-accurate weights)      */
} xmm_pack_segment;

typedef struct {
  void* dst;          /* blob: nchunks*9*nt*kc bf16 (swizzled) then nt fp32 biases        */
  const float* bias;  /* fp32 [O] or NULL; only used when seg[0].transpose == 0           */
  int nt;             /* rows (output channels of the packed GEMM), multiple of 32        */
  int kc;             /* K chunk: 32 or 64 channels                                        */
  int nchunks;        /* K / kc                                                            */
  int nseg;           /* 1..5                                                              */
  int perm;           /* 1: PixelShuffle(2) channel permutation on the O index             */
  int n_valid;        /* rows >= n_valid are zero                                          */
  int bias_n;         /* rows < bias_n take bias[seg[0].o_off + row]; the rest get 0               */
  xmm_pack_segment seg[5];
  int tap_order;      /* order of the nine (chunk, tap) blocks: 0 = dy*3 + dx (tap views / column scatter),
                         1 = dx*3 + (2 - dy): the three filter rows of one dx are one N = 3*nt operand whose
                         blocks belong to output rows r-1, r, r+1 of input row r (row-hop form, wblob_row)  */
} xmm_pack_job;

/* Bytes of one packed blob. */
size_t xmm_pack_blob_bytes(int nt, int kc, int nchunks);
/* jobs_dev: device array of njobs jobs.  Replaces nothing in the reference -- it is the
 * OIHW fp32 -> tensor-core image conversion run after every optimizer step.              */
int xmm_pack_weights(const xmm_pack_job* jobs_dev, int njobs, void* stream);

/* 3x3 convolution on tensor cores ---------------------------------------------------- */
/* Replaces nn.Conv2d(k=3,s=1,p=1) + torch.cat + LeakyReLU + residual arithmetic of
 * rrdb_blocks.py:37-54,66-70 and generator_rrdb.py:66-69,93-107; with `mask` it is also
 * the data-gradient of the same layers (autograd's conv backward + LeakyReLU backward).
 *   v      = acc + bias
 *   v      = v > 0 ? v : lrelu_slope * v
 *   v     *= (mask[p][n] > 0 ? 1 : mask_slope)           if mask
 *   out    = s0*v + s1*r1[p][n] + s2*r2[p][n]                                            */
typedef struct {
  const void* in;     /* bf16 NHWC [batch][height][width][in_ctot]                         */
  int in_ctot, in_coff, cin; /* cin multiple of kc                                         */
  const void* wblob;  /* from xmm_pack_weights, nt == cout                                 */
  int kc;
  int cout;           /* 32, 64, 128 or 256                                                */
  int batch, height, width;
  float lrelu_slope;  /* 1.0f = no activation                                              */
  const void* mask; int mask_ctot, mask_coff; float mask_slope;
  float s0;
  const void* r1; int r1_ctot, r1_coff; float s1;
  const void* r2; int r2_ctot, r2_coff; float s2;
  void* out; int out_ctot, out_coff;
  int pixel_shuffle;  /* 1: out is [batch][2*height][2*width][out_ctot], cout/4 channels;
                         2: inverse -- out is [batch][height/2][width/2][out_ctot], 4*cout ch. */
  int tap_mode;       /* 0 = library default; 1..3 force a haloed-tap-view layout, 4 the column-scatter form, 5 / 6 the same without / with CTA pairs, 7 / 8 with one / two epilogue groups (tests / probes) */
  float* colsum;      /* optional (cout == 32): colsum[n] += colsum_scale * sum over all pixels of the value written
                         to channel n -- the bias gradient whose integrand this data-gradient layer produces       */
  float colsum_scale;
  int shuffle_stride; /* pixel_shuffle == 2 only: channel distance between the four (y&1, x&1) blocks of the output
                         (0 = cout).  A layer split along its output channels writes part n0 with out_coff + n0 and
                         the full layer's cout here.                                                              */
  const void* wblob_row; /* optional: the same layer packed with tap_order = 1.  When given, and the shape qualifies
                         (cout == kc in {32, 64}, no pixel shuffle, height = nbands * band_h with 8 <= nbands <= 16,
                         weights resident next to >= 3 pipeline stages), the launch takes the row-hop form
                         (conv3x3_row.cuh); tap_mode 9 forces it (error if it does not qualify), 1..8 never use it. */
  float* colsum_ws;   /* optional, with colsum: the deterministic form of the column sums.  colsum is then NOT written;
                         the launch stores unscaled partial sums to colsum_ws_slots slots of 32 floats
                         (xmm_det_slots(XMM_DET_CONV3X3, ...) of them at least), which must be zero on entry, and
                         xmm_det_finalize adds them.  Not taken by the fused dense-block form of xmm_conv3x3_chain_bf16
                         (column sums never are).                                                                 */
  size_t colsum_ws_slots;
} xmm_conv3x3_params;

int xmm_conv3x3_bf16(const xmm_conv3x3_params* p, void* stream);

/* A chain of dependent 3x3 convolutions -- the five convs of one ResidualDenseBlock_5C.forward
 * (rrdb_blocks.py:37-54: each reads what the previous ones wrote) or the five data gradients of its backward --
 * with the SAME result (up to fp32 summation order) as calling xmm_conv3x3_bf16 on layers[0], layers[1], ... in order.
 * mode_flags = mode | flags.
 * mode 0: library chooses (the fused dense block where the layers qualify, else layer by layer);
 *      1: one pipelined launch (layer k runs on its own group of SMs two image strips behind layer k-1, so
 *         intermediate activations are consumed from L2; error if the layers do not qualify; needs `workspace`,
 *         xmm_conv3x3_chain_workspace_bytes);
 *      2: layer by layer;
 *      3: fused dense block (conv3x3_rdb.cuh): conv1..conv3 in one launch and conv4..conv5 in a second, the feature
 *         maps in between handed over in shared memory (576 instead of 1280 bytes per pixel through HBM); error if
 *         the layers are not exactly a dense block: five kc = cout = 32 layers with a row-hop weight image
 *         (wblob_row), layer k reading channels [c0, c0 + 32 (k+1)) of ONE buffer and, for k < 5, writing channels
 *         [c0 + 32 k, c0 + 32 (k+1)) of it; LeakyReLU / residuals (last layer only) as usual; even image height.
 * XMM_CHAIN_SKIP_DEAD_STORES: the caller will not read the outputs of layers 1..n-1 after this call (inference);
 *         outputs that no later launch of the chain reads need not be written (the fused form never writes x4).   */
#define XMM_CHAIN_SKIP_DEAD_STORES 0x100
/* XMM_CHAIN_SKIP_LAST: compute and store the outputs of layers 1..n-1 only; the last layer's output is never written
 *         (recomputing a dense block's x1..x4 from its input for a backward pass).  The launch form is chosen as
 *         without the flag; the fused form then runs conv1..conv3 as usual and conv4 in a conv4-only form of the
 *         second kernel, every other form runs layers 1..n-1 one by one.  The fused and layer-by-layer forms store
 *         the bits the same call without the flag stores (mode 1: the same values up to fp32 summation order).
 *         Not with XMM_CHAIN_SKIP_DEAD_STORES (XMM_ERR_INVALID_ARGUMENT); nlayers >= 2.                            */
#define XMM_CHAIN_SKIP_LAST 0x800
/* XMM_CHAIN_RDB_PAIR / XMM_CHAIN_RDB_SINGLE (mode 0 / 3, at most one): run both kernels of the fused dense block
 *         (conv1..conv3, conv4..conv5) as CTA pairs (two SMs share every MMA, each holding half of the weights) / as
 *         single CTAs, for this call, whatever XMM_RDB_PAIR selects.  Both forms compute the same bits.            */
#define XMM_CHAIN_RDB_PAIR 0x200
#define XMM_CHAIN_RDB_SINGLE 0x400
size_t xmm_conv3x3_chain_workspace_bytes(int nlayers, int batch, int height);
int xmm_conv3x3_chain_bf16(const xmm_conv3x3_params* layers, int nlayers, int mode_flags, void* workspace,
                           size_t workspace_bytes, void* stream);
/* Kernels the calling thread's last xmm_conv3x3_chain_bf16 launched (2 fused, 1 pipelined, nlayers layer by layer). */
int xmm_last_chain_launches(void);

/* Input transforms ------------------------------------------------------------------- */
#define XMM_STRETCH_LINEAR 0
#define XMM_STRETCH_SQRT 1
#define XMM_STRETCH_ASINH 2
#define XMM_STRETCH_LOG 3

/* Replaces Normalize.normalize_image (transforms/normalize.py:66-82) fused with the detector
 * mask multiply (data/dataset.py:41-42) and the counts -> rate division the refactor lost
 * (SURVEY I4): v = in * pre_scale * mask; v = clamp(v, 0, max_val) / max_val; stretch;
 * clamp(0,1).  max_val <= 0 selects the reference's "divide by the image maximum" branch
 * (fp32 input only; `scratch` = one device float).                                        */
typedef struct {
  const void* in;       /* fp32 or int32, n elements                                       */
  int in_is_int32;
  const uint8_t* mask;  /* optional, mask_n elements, repeated every mask_n                */
  size_t mask_n;
  float* out;           /* fp32, n elements (may alias `in` when in is fp32)               */
  size_t n;
  float pre_scale;
  float max_val;
  int stretch_mode;
  float* scratch;
} xmm_normalize_params;
int xmm_normalize(const xmm_normalize_params* p, void* stream);

/* Replaces Normalize.denormalize_image (transforms/normalize.py:84-92):
 * out = clamp(max * denorm(in), 0, max); max_vals_dev holds 1 value or one per image.     */
int xmm_denormalize(const float* in, float* out, size_t n, size_t per_image, const float* max_vals_dev,
                    int max_n, int stretch_mode, void* stream);

/* out = norm_to(denorm_from(in)), element-wise: the re-normalisation XMMMetricCollection.update applies
 * before every metric (metrics/xmm_metric_collection.py:135-143), as one pass.                           */
int xmm_restretch(const float* in, float* out, size_t n, int from_mode, int to_mode, void* stream);

/* The per-batch data feed (data/dataset.py:24-49,258-270; data/tools.py:103-126) on raw count planes that are
 * already in device memory: sum of up to 3 planes (image, AGN, background) x detector mask, optional
 * ImageUpsample, zero-pad / crop to res_h x res_w (floor(diff/2) before), counts -> rate, Normalize.       */
typedef struct {
  const void* src[3];  /* [batch][h][w] int32 or fp32; src[0] required                                    */
  int nsrc;
  int src_is_int32;
  const unsigned char* mask; /* [h][w] or NULL                                                              */
  int batch, h, w;
  int up;              /* integer ImageUpsample factor (1 = none)                                          */
  int res_h, res_w;    /* output image size                                                                */
  float pre_scale;     /* 1/exposure                                                                       */
  const float* pre_scale_dev; /* optional per-image factor [batch] (multiplied with pre_scale)            */
  float max_val;       /* > 0                                                                              */
  int stretch_mode;
  float* out;          /* [batch][res_h][res_w] fp32                                                       */
} xmm_prepare_counts_params;
int xmm_prepare_counts(const xmm_prepare_counts_params* p, void* stream);

/* Replaces ImageUpsample.__call__ (transforms/imageupsample.py:10-26): nearest upsample by an
 * integer factor then divide by factor^2.  in [n_img][h][w] fp32 -> out [n_img][h*s][w*s].  */
int xmm_image_upsample(const float* in, float* out, int n_img, int h, int w, int scale, void* stream);

/* First / last convolution ------------------------------------------------------------ */
/* conv_first (generator_rrdb.py:31-37,67): fp32 NCHW image -> bf16 NHWC features.          */
typedef struct {
  const float* in;    /* [batch][cin][height][width]                                       */
  const float* weight; /* fp32 OIHW [filters][cin][3][3]                                   */
  const float* bias;  /* fp32 [filters] or NULL                                            */
  int batch, cin, height, width, filters;  /* cin 1..4, filters 32 or 64                    */
  void* out; int out_ctot, out_coff;
  void* out2; int out2_ctot, out2_coff;    /* optional second copy (trunk skip), or NULL     */
  /* Backward use -- the data gradient of conv_last is this same stencil on the loss gradient: */
  const float* gate;  /* optional, shape of `in`: in is used only where 0 <= gate <= 1 (clamp)   */
  const void* mask; int mask_ctot, mask_coff; float mask_slope; /* optional LeakyReLU' on out  */
} xmm_conv_first_params;
int xmm_conv_first(const xmm_conv_first_params* p, void* stream);

/* conv_last (generator_rrdb.py:48-54,107-108,132-135) + DN input residual + clamp[0,1]
 * (also covers Model.forward's second clamp, models/model.py:49).                          */
typedef struct {
  const void* in; int in_ctot, in_coff;  /* bf16 NHWC, `filters` channels                   */
  const float* weight; /* fp32 OIHW [cout][filters][3][3]                                  */
  const float* bias;   /* fp32 [cout] or NULL                                              */
  const float* residual; /* optional fp32 NCHW [batch][cout][height][width]                */
  float* out;          /* fp32 NCHW [batch][cout][height][width]                           */
  float* pre;          /* optional un-clamped copy (training)                              */
  int batch, cout, height, width, filters;  /* cout 1..4                                    */
  int clamp;
  const void* wblob;  /* optional: packed split-precision layer (nt = 32, kc = 32, rows [0,cout) = bf16(w),
                         rows [16,16+cout) = low-order halves, bias in the blob) -> tensor-core path;
                         NULL -> CUDA-core path reading `weight` / `bias`                           */
} xmm_conv_last_params;
int xmm_conv_last(const xmm_conv_last_params* p, void* stream);

/* Weight gradients -------------------------------------------------------------------- */
/* dW[tap][c][n] = sum_p X[p+off(tap)][c] * dY[p][n] on the tensor cores (autograd's conv
 * bwd-filter for rrdb_blocks.py:27-31, generator_rrdb.py:39-45,93-101).  The launch is split
 * into roles (a CTA keeps tap_count*n <= 512 TMEM columns of accumulators for its whole life);
 * every role streams all pixel tiles; a second kernel reduces the per-CTA partial sums into
 * the fp32 OIHW gradient tensors listed in dst[].                                           */
typedef struct {
  int tap_begin, tap_count; /* taps [tap_begin, tap_begin+tap_count) of the 9, tap = 3*dy+dx   */
  int x_c0, x_boxes;        /* M tile: X channels [x_c0, x_c0 + 64*x_boxes) (x_boxes 1 or 2)    */
  int y_c0, n;              /* N tile: dY channels [y_c0, y_c0 + n), n multiple of 16, <= 192   */
  int mode;                 /* 0: as above.  1: "stacked" 32-channel role -- M = dY channels [y_c0, y_c0 + 64*x_boxes),
                               N = 96 = X channels [x_c0, x_c0+32) at dx = 0,1,2; tap_begin 0, tap_count 3 (filter
                               rows).  Destinations of such a role: lane0 = first dY channel - y_c0,
                               col0 = i_begin - x_c0; all 9 taps are written.                                  */
} xmm_wgrad_role;

typedef struct {
  float* dw;                /* fp32 OIHW [o_count][i_total][3][3]                               */
  int o_count, i_total;
  int i_begin, i_end;       /* input channels taken from role `role`                            */
  int role;
  int lane0;                /* accumulator row of input channel i_begin ( = i_begin - x_c0 )    */
  int col0;                 /* accumulator column (within one tap) of output channel 0         */
  float scale;
  int accumulate;           /* 0: overwrite dw, 1: add                                          */
  int perm;                 /* 1: columns are in PixelShuffle-packed order                      */
  int o_begin, o_total;     /* the role covers output channels [o_begin, o_begin + o_count) of o_total
                               (o_total 0 = o_count, o_begin 0): layers with more output channels than lanes */
} xmm_wgrad_dst;

typedef struct {
  const void* x; int x_ctot;   /* bf16 NHWC activations                                        */
  const void* dy; int dy_ctot; /* bf16 NHWC gradients                                          */
  int batch, height, width;
  int nroles; xmm_wgrad_role roles[4];
  int ndst; xmm_wgrad_dst dst[16];
  float* workspace;            /* xmm_wgrad_workspace_bytes() bytes                            */
} xmm_wgrad_params;

size_t xmm_wgrad_workspace_bytes(void);
int xmm_conv3x3_wgrad(const xmm_wgrad_params* p, void* stream);

/* out[i] (+)= scale * sum over pixels of in[p][c0 + i]  (bias gradients), n multiple of 8.  */
int xmm_colsum_bf16(const void* in, int ctot, int c0, int n, size_t npix, float* out, float scale,
                    int accumulate, void* stream);

/* dst[p][dst_coff + i] = src[p][src_coff + i] for every pixel p < npix and i < channels: a channel window between two
 * bf16 NHWC buffers of different channel pitch (a dense block's input into and out of its 5F-channel buffer).
 * 16-byte accesses: channels, both pitches and both offsets multiples of 8, pointers 16-byte aligned.            */
int xmm_copy_channels_bf16(const void* src, int src_ctot, int src_coff, void* dst, int dst_ctot, int dst_coff,
                           int channels, size_t npix, void* stream);

/* Several channel windows of one buffer in a single pass (a dense block's five bias gradients).           */
typedef struct {
  int c0, n;          /* window [c0, c0+n), multiples of 8                                                */
  float* out;         /* n floats                                                                         */
  float scale;
  int accumulate;     /* 0: out is zeroed first                                                           */
} xmm_colsum_segment;
int xmm_colsum_multi_bf16(const void* in, int ctot, size_t npix, const xmm_colsum_segment* segs, int nseg,
                          void* stream);
/* Deterministic form of xmm_colsum_multi_bf16: the segments' out / accumulate are not used; each CTA stores the
 * unscaled sums of all segments' channels, concatenated in segment order, to its own slot of ws (ws_slots slots of
 * sum(n) floats, xmm_det_slots(XMM_DET_COLSUM, ...) at least, zero on entry).  xmm_det_finalize applies the
 * segments' scale and destination.                                                                                */
int xmm_colsum_multi_det_bf16(const void* in, int ctot, size_t npix, const xmm_colsum_segment* segs, int nseg,
                              float* ws, size_t ws_slots, void* stream);

/* Weight/bias gradients of the two CUDA-core convolutions:
 *   R[o][c][tap] += sum_p s[o][p] * (V[p+off(tap)][c] + V2[p+off(tap)][c]);  S[o] += sum_p s[o][p]
 * conv_last: s = dL/dout (gated by the clamp), V = input features.  conv_first: s = input
 * image, V (+V2) = dL/dfea; then dW_first[f][o][8-tap] = R[o][f][tap].                        */
typedef struct {
  const float* s; const float* gate;  /* fp32 NCHW [batch][ns][height][width]                  */
  const void* v; int v_ctot, v_coff;  /* bf16 NHWC, `channels` channels                        */
  const void* v2; int v2_ctot, v2_coff; /* optional                                            */
  float* r;                           /* fp32 [ns][channels][9], accumulated into              */
  float* ssum;                        /* fp32 [ns] or NULL, accumulated into                   */
  int batch, ns, height, width, channels; /* channels 32 or 64                                 */
  float* ws;                          /* optional: deterministic form.  r / ssum are then NOT written; each CTA
                                         stores R (ns*channels*9 floats) then S (ns floats, if ssum != NULL) to its
                                         own slot of ns*channels*9 + ns floats (ws_slots slots,
                                         xmm_det_slots(XMM_DET_EDGE_WGRAD, ...) at least, zero on entry)        */
  size_t ws_slots;
} xmm_edge_wgrad_params;
int xmm_edge_wgrad(const xmm_edge_wgrad_params* p, void* stream);

/* Deterministic gradient reductions ------------------------------------------------------ */
/* The three reductions above (fused conv3x3 column sums, colsum, edge_wgrad) add per-warp / per-CTA partial sums with
 * float atomics, in an order that depends on CTA timing.  Their deterministic forms store the partial sums to slots of
 * a caller-owned workspace instead; one xmm_det_finalize launch then reduces any number of slot ranges, each in a
 * fixed order, so the result is the same bits on every run (same device, same SM count and reserve, same shapes).
 * Slots per call of a site, for xmm_set_sm_reserve's current value (the row length is the caller's: 32 floats for
 * XMM_DET_CONV3X3, the segments' channels for XMM_DET_COLSUM, ns*channels*9 + ns for XMM_DET_EDGE_WGRAD);
 * `channels` is the total channel count of the call (conv3x3: 32; edge_wgrad: its `channels`).                        */
#define XMM_DET_CONV3X3 0
#define XMM_DET_COLSUM 1
#define XMM_DET_EDGE_WGRAD 2
size_t xmm_det_slots(int site, int batch, int height, int width, int channels);

/* dst_base[dst + i] = (accumulate ? dst_base[dst + i] : 0) + scale * sum_{k = 0..count-1} slots[k*stride + i], k in
 * increasing order, for i < n; every slot read is left zero.  Jobs of one call must not share destinations.       */
typedef struct {
  float* slots;       /* count slots, stride floats apart                                                        */
  int count, stride;
  size_t dst;         /* destination: element offset from the call's dst_base                                    */
  int n;
  float scale;
  int accumulate;
} xmm_det_job;
/* jobs_dev: device array of njobs jobs; max_n: the largest n among them.                                          */
int xmm_det_finalize(const xmm_det_job* jobs_dev, int njobs, int max_n, float* dst_base, void* stream);

/* Loss terms ------------------------------------------------------------------------- */
/* Per-scale record kept on the device by the (MS-)SSIM kernels (12 floats). */
typedef struct {
  float minp, maxp, mint, maxt;  /* ranges of preds / target                                */
  float nmaxp, nminp;            /* #pixels of preds equal to its max / min                  */
  float dr, c1, c2;              /* data range, (k1*dr)^2, (k2*dr)^2                         */
  float use_p;                   /* 1 if dr is preds' range (gradient flows into arg-max/min) */
  float d_dr;                    /* dL/d(dr), written by xmm_msssim_finalize                  */
  float pad;
} xmm_scale_stats;

/* One pass over preds/target (fp32, n elements): sums[0..6] = { sum|p-t|, sum(p - t*log(p+1e-8)),
 * sum (p-t)^2, min p, max p, min t, max t } (deterministic two-stage reduction), and, if `stats`
 * is given, the range fields of that record.  Replaces torchmetrics MeanAbsoluteError /
 * PeakSignalNoiseRatio updates and F.poisson_nll_loss (utils/loss_functions.py:15-21,
 * metrics/metrics.py:36-38).  workspace: xmm_loss_workspace_floats() floats.               */
size_t xmm_loss_workspace_floats(void);
int xmm_loss_reduce(const float* preds, const float* target, size_t n, float* sums_dev,
                    xmm_scale_stats* stats_dev, float* workspace, void* stream);
/* grad (=|+=) gl * ( coef[0]*sign(p-t) + coef[1]*(1 - t/(p+1e-8)) + coef[2]*(p-t) ); coef_dev and
 * gl_dev (may be NULL = 1) live on the device, so no host synchronisation is needed.          */
int xmm_loss_grad(const float* preds, const float* target, size_t n, const float* coef_dev,
                  const float* gl_dev, float* grad, int accumulate, void* stream);
/* 2x2 average pooling of preds and target at once (next MS-SSIM scale).                      */
int xmm_avgpool2_pair(const float* preds, const float* target, float* preds_out, float* target_out,
                      int nimg, int h, int w, void* stream);
/* After xmm_loss_reduce filled the ranges: SSIM constants c1,c2 and the arg-max/arg-min counts. */
int xmm_ssim_prepare(const float* preds, size_t n, xmm_scale_stats* stats_dev, float k1, float k2,
                     void* stream);

/* SSIM statistics of one scale (19-tap Gaussian, sigma from the window the caller passes).
 * Forward (kimg == NULL): acc[img][tile][4] partial sums {ssim, cs, d sel/dc1, d sel/dc2}.
 * Backward (kimg != NULL): ga/gb/gc[img][h-18][w-18] = kimg[img] * d sel/d{mu_p, E[pp], E[pt]}. */
typedef struct {
  const float* preds; const float* target;
  int nimg, h, w;
  const xmm_scale_stats* stats_dev;
  float window[19];
  int use_sim;          /* 1: the ssim map feeds this scale's value, 0: the contrast-structure map */
  float* acc;           /* forward output, xmm_ssim_tiles(h,w)*nimg*4 floats                      */
  const float* kimg;    /* backward: per-image coefficients                                       */
  float* ga; float* gb; float* gc;
} xmm_ssim_stats_params;
int xmm_ssim_tiles(int h, int w);
int xmm_ssim_stats(const xmm_ssim_stats_params* p, void* stream);

/* Gradient w.r.t. preds of one scale: transposed Gaussian of ga/gb/gc combined with p and t,
 * plus 1/4 of the coarser scale's gradient (avg-pool backward) and the data-range term.      */
typedef struct {
  const float* preds; const float* target;
  int nimg, h, w;
  const xmm_scale_stats* stats_dev;
  float window[19];
  const float* ga; const float* gb; const float* gc;
  const float* coarse;  /* [nimg][h/2][w/2] or NULL                                            */
  float* grad;          /* [nimg][h][w]                                                        */
  int accumulate;
} xmm_ssim_grad_params;
int xmm_ssim_grad(const xmm_ssim_grad_params* p, void* stream);

/* Combine the per-scale sums: value = mean_b prod_s relu(v_{b,s})^beta_s (nscales == 1: plain SSIM
 * mean), img_val[b], backward coefficients kimg[s][img] (including gl * weight / batch) and
 * stats[s].d_dr.  MultiScaleStructuralSimilarityIndexMeasure / StructuralSimilarityIndexMeasure
 * batch values (utils/loss_functions.py:19-20,33).                                            */
typedef struct {
  const float* acc[5];
  int tiles[5];
  int nvalid[5];
  int nscales;
  int batch, channels;
  float betas[5];
  float k1, k2;
  xmm_scale_stats* stats_dev;
  float* value;
  float* img_val;
  float* kimg;
  const float* gl_dev;
  float weight;
} xmm_msssim_finalize_params;
int xmm_msssim_finalize(const xmm_msssim_finalize_params* p, void* stream);

/* Optimizer -------------------------------------------------------------------------- */
/* One Adam step (torch.optim.Adam semantics: models/model.py:239-247, res/configs/models.toml:7-8)
 * over a flat fp32 parameter buffer; `step` is the 1-based step count; grad is multiplied by
 * grad_scale first (1/world_size after a sum all-reduce).                                     */
int xmm_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                  float beta1, float beta2, float eps, int step, float grad_scale, void* stream);

/* Gradient clipping (Lightning's Trainer(gradient_clip_val, gradient_clip_algorithm), applied once per optimizer step
 * to the averaged gradient g = grads * grad_scale).
 * xmm_grad_clip_coef: out[0] = ||g||_2 (squares added in fp64, rounded once to fp32), out[1] = the coefficient of
 * torch.nn.utils.clip_grad_norm_(max_norm=max_norm), in fp32 as torch computes it: min(max_norm / (out[0] + 1e-6), 1)
 * (an inf norm gives 0, a NaN norm NaN).  Two launches, no host synchronisation; the order of every addition depends
 * on n only, so the result is the same bits on every run.  grads 16-byte aligned; grad_scale > 0; max_norm >= 0;
 * workspace: xmm_grad_norm_workspace_bytes(n) bytes (per-CTA partial sums, overwritten).                          */
size_t xmm_grad_norm_workspace_bytes(size_t n);
int xmm_grad_clip_coef(const float* grads, size_t n, float grad_scale, float max_norm, float* out, void* workspace,
                       size_t workspace_bytes, void* stream);
/* xmm_adam_step on a clipped gradient: Adam sees grads * (grad_scale * clip_coef[0]) when clip_coef (a device float,
 * e.g. out + 1 of xmm_grad_clip_coef) is given -- clip by norm -- or clamp(grads * grad_scale, -clip_value,
 * clip_value) when clip_value > 0 -- clip by value, torch.nn.utils.clip_grad_value_.  Exactly one of the two.  With
 * clip_coef[0] == 1 and grad_scale == 1 the step is xmm_adam_step's, bit for bit.                                 */
int xmm_adam_step_clip(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                       float beta1, float beta2, float eps, int step, float grad_scale, const float* clip_coef,
                       float clip_value, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* XMM_B200_H_ */
