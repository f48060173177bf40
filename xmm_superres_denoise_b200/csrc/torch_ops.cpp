// TORCH_LIBRARY(xmm_b200, m): the torch custom-op face of the C ABI (SURVEY.md section 8b).
//
// Thin shims and nothing else: every op checks its tensors (CUDA, dtype, contiguity, one device), fills the
// extern "C" parameter struct of include/xmm_b200.h from tensor metadata, makes the tensors' device current and calls
// the launcher in libxmm_b200.so on torch's current stream of that device.  No arithmetic, no allocation (outputs
// are passed in and mutated), no fallback: a non-zero return code becomes a c10::Error carrying xmm_last_error().
//
// Why it exists next to the ctypes binding (_lib.py): registered ops are visible to the dispatcher -- they can be
// called from TorchScript / torch.compile graphs as opaque nodes, show up in the profiler under their own names, and
// cost ~2 us of dispatch per call where ctypes costs ~8-10 us of Python struct filling.  The reference has no
// operator layer of its own (it calls nn.Conv2d / F.leaky_relu / torch.cat: rrdb_blocks.py:37-54); each op below
// cites the reference lines its launcher replaces.
//
// Built by __graft_entry__.build() with g++ (no nvcc: this file holds no device code) into
// xmm_superres_denoise_b200/libxmm_b200_torch.so; load with xmm_superres_denoise_b200.torch_ops.load().
#include <ATen/ATen.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include "../../include/xmm_b200.h"

namespace {

using at::Tensor;
using OptTensor = std::optional<Tensor>;

void check_rc(int rc, const char* what) {
  if (rc != 0) {
    const char* msg = xmm_last_error();
    TORCH_CHECK(false, "xmm_b200::", what, ": libxmm_b200 error ", rc, ": ", msg ? msg : "?");
  }
}

void need(const Tensor& t, at::ScalarType dtype, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, ": expected a CUDA tensor (xmm_b200 has no CPU path)");
  TORCH_CHECK(t.scalar_type() == dtype, name, ": expected dtype ", dtype, ", got ", t.scalar_type());
  TORCH_CHECK(t.is_contiguous(), name, ": expected a contiguous tensor");
}

void same_device(const Tensor& a, const OptTensor& b, const char* name) {
  if (b.has_value()) TORCH_CHECK(b->device() == a.device(), name, ": tensors live on different devices");
}

void* stream_of(const Tensor& t) { return c10::cuda::getCurrentCUDAStream(t.device().index()).stream(); }

int stretch_mode(const std::string& s) {
  if (s == "linear") return XMM_STRETCH_LINEAR;
  if (s == "sqrt") return XMM_STRETCH_SQRT;
  if (s == "asinh") return XMM_STRETCH_ASINH;
  if (s == "log") return XMM_STRETCH_LOG;
  TORCH_CHECK(false, "unknown stretch mode '", s, "' (transforms/normalize.py:44-63 knows linear, sqrt, asinh, log)");
}

// rrdb_blocks.py:37-54,66-70 / generator_rrdb.py:66-69,93-107: one 3x3 conv of the generator with its fused epilogue
//   out[..., out_coff:out_coff+cout] = s0 * lrelu(conv(inp[..., in_coff:in_coff+cin]) + bias) + s1 * r1 + s2 * r2
// on NHWC bf16 buffers.  `wblob` / `wblob_row` are device addresses of weight images made by xmm_pack_weights
// (engine.WeightArena.ptr); wblob_row == 0: none.
void conv3x3_fwd(const Tensor& inp, int64_t in_coff, int64_t cin, int64_t wblob, int64_t kc, int64_t cout, Tensor out,
                 int64_t out_coff, double lrelu, double s0, const OptTensor& r1, int64_t r1_coff, double s1,
                 const OptTensor& r2, int64_t r2_coff, double s2, int64_t wblob_row, int64_t tap_mode) {
  need(inp, at::kBFloat16, "conv3x3_fwd input");
  need(out, at::kBFloat16, "conv3x3_fwd output");
  TORCH_CHECK(inp.dim() == 4 && out.dim() == 4, "conv3x3_fwd: NHWC [B,H,W,C] buffers expected");
  TORCH_CHECK(out.device() == inp.device(), "conv3x3_fwd: tensors live on different devices");
  same_device(inp, r1, "conv3x3_fwd r1");
  same_device(inp, r2, "conv3x3_fwd r2");
  TORCH_CHECK(out.size(0) == inp.size(0) && out.size(1) == inp.size(1) && out.size(2) == inp.size(2),
              "conv3x3_fwd: input and output geometry differ");
  xmm_conv3x3_params p{};
  p.in = inp.data_ptr();
  p.in_ctot = int(inp.size(3));
  p.in_coff = int(in_coff);
  p.cin = int(cin);
  p.wblob = reinterpret_cast<const void*>(wblob);
  p.wblob_row = reinterpret_cast<const void*>(wblob_row);
  p.kc = int(kc);
  p.cout = int(cout);
  p.batch = int(inp.size(0));
  p.height = int(inp.size(1));
  p.width = int(inp.size(2));
  p.lrelu_slope = float(lrelu);
  p.mask_slope = 1.f;
  p.s0 = float(s0);
  if (r1.has_value()) {
    need(*r1, at::kBFloat16, "conv3x3_fwd r1");
    p.r1 = r1->data_ptr();
    p.r1_ctot = int(r1->size(3));
    p.r1_coff = int(r1_coff);
    p.s1 = float(s1);
  }
  if (r2.has_value()) {
    need(*r2, at::kBFloat16, "conv3x3_fwd r2");
    p.r2 = r2->data_ptr();
    p.r2_ctot = int(r2->size(3));
    p.r2_coff = int(r2_coff);
    p.s2 = float(s2);
  }
  p.out = out.data_ptr();
  p.out_ctot = int(out.size(3));
  p.out_coff = int(out_coff);
  p.tap_mode = int(tap_mode);
  c10::cuda::CUDAGuard guard(inp.device());
  check_rc(xmm_conv3x3_bf16(&p, stream_of(inp)), "conv3x3_fwd");
}

// The data gradient of the same layers: autograd's conv backward-data + LeakyReLU backward (the mask is the
// forward activation the gradient passes through; wblob is the transposed / tap-flipped image).
void conv3x3_dgrad(const Tensor& dy, int64_t in_coff, int64_t cin, int64_t wblob, int64_t kc, int64_t cout, Tensor out,
                   int64_t out_coff, const Tensor& mask, int64_t mask_coff, double mask_slope, const OptTensor& r1,
                   int64_t r1_coff, double s1, int64_t wblob_row) {
  need(dy, at::kBFloat16, "conv3x3_dgrad dy");
  need(out, at::kBFloat16, "conv3x3_dgrad output");
  need(mask, at::kBFloat16, "conv3x3_dgrad mask");
  TORCH_CHECK(dy.dim() == 4 && out.dim() == 4 && mask.dim() == 4, "conv3x3_dgrad: NHWC [B,H,W,C] buffers expected");
  TORCH_CHECK(out.device() == dy.device() && mask.device() == dy.device(), "conv3x3_dgrad: tensors live on different devices");
  same_device(dy, r1, "conv3x3_dgrad r1");
  xmm_conv3x3_params p{};
  p.in = dy.data_ptr();
  p.in_ctot = int(dy.size(3));
  p.in_coff = int(in_coff);
  p.cin = int(cin);
  p.wblob = reinterpret_cast<const void*>(wblob);
  p.wblob_row = reinterpret_cast<const void*>(wblob_row);
  p.kc = int(kc);
  p.cout = int(cout);
  p.batch = int(dy.size(0));
  p.height = int(dy.size(1));
  p.width = int(dy.size(2));
  p.lrelu_slope = 1.f;
  p.mask = mask.data_ptr();
  p.mask_ctot = int(mask.size(3));
  p.mask_coff = int(mask_coff);
  p.mask_slope = float(mask_slope);
  p.s0 = 1.f;
  if (r1.has_value()) {
    need(*r1, at::kBFloat16, "conv3x3_dgrad r1");
    p.r1 = r1->data_ptr();
    p.r1_ctot = int(r1->size(3));
    p.r1_coff = int(r1_coff);
    p.s1 = float(s1);
  }
  p.out = out.data_ptr();
  p.out_ctot = int(out.size(3));
  p.out_coff = int(out_coff);
  c10::cuda::CUDAGuard guard(dy.device());
  check_rc(xmm_conv3x3_bf16(&p, stream_of(dy)), "conv3x3_dgrad");
}

// transforms/normalize.py:66-82 (+ the detector-mask multiply of data/dataset.py:41-42 and the counts -> rate
// division): out = stretch(clamp(inp * pre_scale * mask, 0, max_val) / max_val).  inp fp32 or int32.
void normalize(const Tensor& inp, Tensor out, double pre_scale, double max_val, const std::string& mode,
               const OptTensor& mask) {
  TORCH_CHECK(inp.is_cuda() && inp.is_contiguous(), "normalize input: expected a contiguous CUDA tensor");
  TORCH_CHECK(inp.scalar_type() == at::kFloat || inp.scalar_type() == at::kInt, "normalize input: fp32 or int32");
  need(out, at::kFloat, "normalize output");
  TORCH_CHECK(out.numel() == inp.numel() && out.device() == inp.device(), "normalize: input / output mismatch");
  TORCH_CHECK(max_val > 0, "normalize: the torch op takes max_val > 0 (the image-maximum branch needs a scratch buffer: "
                           "use xmm_superres_denoise_b200.transforms.Normalize)");
  same_device(inp, mask, "normalize mask");
  xmm_normalize_params p{};
  p.in = inp.data_ptr();
  p.in_is_int32 = inp.scalar_type() == at::kInt ? 1 : 0;
  if (mask.has_value()) {
    need(*mask, at::kByte, "normalize mask");
    TORCH_CHECK(mask->numel() > 0 && inp.numel() % mask->numel() == 0, "normalize: mask does not tile the input");
    p.mask = mask->data_ptr<uint8_t>();
    p.mask_n = size_t(mask->numel());
  }
  p.out = out.data_ptr<float>();
  p.n = size_t(inp.numel());
  p.pre_scale = float(pre_scale);
  p.max_val = float(max_val);
  p.stretch_mode = stretch_mode(mode);
  c10::cuda::CUDAGuard guard(inp.device());
  check_rc(xmm_normalize(&p, stream_of(inp)), "normalize");
}

// transforms/normalize.py:84-92: out = clamp(max * denorm(inp), 0, max); max_vals: 1 value or one per image.
void denormalize(const Tensor& inp, Tensor out, const Tensor& max_vals, const std::string& mode) {
  need(inp, at::kFloat, "denormalize input");
  need(out, at::kFloat, "denormalize output");
  need(max_vals, at::kFloat, "denormalize max_vals");
  TORCH_CHECK(out.numel() == inp.numel() && out.device() == inp.device() && max_vals.device() == inp.device(),
              "denormalize: input / output / max_vals mismatch");
  const int64_t nmax = max_vals.numel();
  TORCH_CHECK(nmax == 1 || (inp.dim() >= 1 && nmax == inp.size(0)), "denormalize: max_vals holds 1 value or one per image");
  const size_t per_image = nmax > 1 ? size_t(inp.numel() / nmax) : size_t(inp.numel());
  c10::cuda::CUDAGuard guard(inp.device());
  check_rc(xmm_denormalize(inp.data_ptr<float>(), out.data_ptr<float>(), size_t(inp.numel()), per_image,
                           max_vals.data_ptr<float>(), int(nmax), stretch_mode(mode), stream_of(inp)),
           "denormalize");
}

// transforms/imageupsample.py:10-26: nearest upsample by an integer factor, divided by factor^2.
void image_upsample(const Tensor& inp, Tensor out, int64_t scale) {
  need(inp, at::kFloat, "image_upsample input");
  need(out, at::kFloat, "image_upsample output");
  TORCH_CHECK(inp.dim() >= 2, "image_upsample: [..., H, W] expected");
  const int64_t h = inp.size(-2), w = inp.size(-1);
  TORCH_CHECK(out.device() == inp.device() && out.numel() == inp.numel() * scale * scale, "image_upsample: output size");
  c10::cuda::CUDAGuard guard(inp.device());
  check_rc(xmm_image_upsample(inp.data_ptr<float>(), out.data_ptr<float>(), int(inp.numel() / (h * w)), int(h), int(w),
                              int(scale), stream_of(inp)),
           "image_upsample");
}

// models/model.py:239-247 (torch.optim.Adam) on flat fp32 buffers, one launch; grads are multiplied by grad_scale
// first (1 / world size after a summing all-reduce).
void adam_step(Tensor params, const Tensor& grads, Tensor exp_avg, Tensor exp_avg_sq, double lr, double beta1,
               double beta2, double eps, int64_t step, double grad_scale) {
  need(params, at::kFloat, "adam_step params");
  need(grads, at::kFloat, "adam_step grads");
  need(exp_avg, at::kFloat, "adam_step exp_avg");
  need(exp_avg_sq, at::kFloat, "adam_step exp_avg_sq");
  const int64_t n = params.numel();
  TORCH_CHECK(grads.numel() == n && exp_avg.numel() == n && exp_avg_sq.numel() == n, "adam_step: buffer sizes differ");
  TORCH_CHECK(grads.device() == params.device() && exp_avg.device() == params.device() &&
                  exp_avg_sq.device() == params.device(), "adam_step: tensors live on different devices");
  c10::cuda::CUDAGuard guard(params.device());
  check_rc(xmm_adam_step(params.data_ptr<float>(), grads.data_ptr<float>(), exp_avg.data_ptr<float>(),
                         exp_avg_sq.data_ptr<float>(), size_t(n), float(lr), float(beta1), float(beta2), float(eps),
                         int(step), float(grad_scale), stream_of(params)),
           "adam_step");
}

// torch.nn.utils.clip_grad_norm_(max_norm) without the multiply: out = {||grads * grad_scale||_2, min(max_norm /
// (norm + 1e-6), 1)} (fp32, on the device); workspace: any contiguous CUDA tensor of
// xmm_grad_norm_workspace_bytes(grads.numel()) bytes or more.
void grad_clip_coef(const Tensor& grads, double grad_scale, double max_norm, Tensor out, Tensor workspace) {
  need(grads, at::kFloat, "grad_clip_coef grads");
  need(out, at::kFloat, "grad_clip_coef out");
  TORCH_CHECK(workspace.is_cuda() && workspace.is_contiguous(), "grad_clip_coef workspace: expected a contiguous CUDA tensor");
  TORCH_CHECK(out.numel() >= 2, "grad_clip_coef: out holds {norm, coef}");
  TORCH_CHECK(out.device() == grads.device() && workspace.device() == grads.device(),
              "grad_clip_coef: tensors live on different devices");
  c10::cuda::CUDAGuard guard(grads.device());
  check_rc(xmm_grad_clip_coef(grads.data_ptr<float>(), size_t(grads.numel()), float(grad_scale), float(max_norm),
                              out.data_ptr<float>(), workspace.data_ptr(), size_t(workspace.nbytes()), stream_of(grads)),
           "grad_clip_coef");
}

// adam_step on a clipped gradient: grads * (grad_scale * clip_coef[0]) (clip_coef: one float on the device, e.g.
// out[1:] of grad_clip_coef) or clamp(grads * grad_scale, -clip_value, clip_value) (clip_value > 0); exactly one.
void adam_step_clip(Tensor params, const Tensor& grads, Tensor exp_avg, Tensor exp_avg_sq, double lr, double beta1,
                    double beta2, double eps, int64_t step, double grad_scale, const OptTensor& clip_coef,
                    double clip_value) {
  need(params, at::kFloat, "adam_step_clip params");
  need(grads, at::kFloat, "adam_step_clip grads");
  need(exp_avg, at::kFloat, "adam_step_clip exp_avg");
  need(exp_avg_sq, at::kFloat, "adam_step_clip exp_avg_sq");
  const int64_t n = params.numel();
  TORCH_CHECK(grads.numel() == n && exp_avg.numel() == n && exp_avg_sq.numel() == n,
              "adam_step_clip: buffer sizes differ");
  TORCH_CHECK(grads.device() == params.device() && exp_avg.device() == params.device() &&
                  exp_avg_sq.device() == params.device(), "adam_step_clip: tensors live on different devices");
  same_device(params, clip_coef, "adam_step_clip clip_coef");
  const float* coef = nullptr;
  if (clip_coef.has_value()) {
    need(*clip_coef, at::kFloat, "adam_step_clip clip_coef");
    TORCH_CHECK(clip_coef->numel() >= 1, "adam_step_clip: clip_coef is empty");
    coef = clip_coef->data_ptr<float>();
  }
  c10::cuda::CUDAGuard guard(params.device());
  check_rc(xmm_adam_step_clip(params.data_ptr<float>(), grads.data_ptr<float>(), exp_avg.data_ptr<float>(),
                              exp_avg_sq.data_ptr<float>(), size_t(n), float(lr), float(beta1), float(beta2),
                              float(eps), int(step), float(grad_scale), coef, float(clip_value), stream_of(params)),
           "adam_step_clip");
}

int64_t abi_version() { return xmm_version(); }

}  // namespace

TORCH_LIBRARY(xmm_b200, m) {
  m.def("conv3x3_fwd(Tensor inp, int in_coff, int cin, int wblob, int kc, int cout, Tensor(a!) out, int out_coff, "
        "float lrelu=1.0, float s0=1.0, Tensor? r1=None, int r1_coff=0, float s1=0.0, Tensor? r2=None, int r2_coff=0, "
        "float s2=0.0, int wblob_row=0, int tap_mode=0) -> ()");
  m.def("conv3x3_dgrad(Tensor dy, int in_coff, int cin, int wblob, int kc, int cout, Tensor(a!) out, int out_coff, "
        "Tensor mask, int mask_coff, float mask_slope, Tensor? r1=None, int r1_coff=0, float s1=0.0, int wblob_row=0) -> ()");
  m.def("normalize(Tensor inp, Tensor(a!) out, float pre_scale, float max_val, str mode, Tensor? mask=None) -> ()");
  m.def("denormalize(Tensor inp, Tensor(a!) out, Tensor max_vals, str mode) -> ()");
  m.def("image_upsample(Tensor inp, Tensor(a!) out, int scale) -> ()");
  m.def("adam_step(Tensor(a!) params, Tensor grads, Tensor(b!) exp_avg, Tensor(c!) exp_avg_sq, float lr, float beta1, "
        "float beta2, float eps, int step, float grad_scale=1.0) -> ()");
  m.def("grad_clip_coef(Tensor grads, float grad_scale, float max_norm, Tensor(a!) out, Tensor(b!) workspace) -> ()");
  m.def("adam_step_clip(Tensor(a!) params, Tensor grads, Tensor(b!) exp_avg, Tensor(c!) exp_avg_sq, float lr, "
        "float beta1, float beta2, float eps, int step, float grad_scale=1.0, Tensor? clip_coef=None, "
        "float clip_value=0.0) -> ()");
  m.def("abi_version() -> int", &abi_version);
}

TORCH_LIBRARY_IMPL(xmm_b200, CUDA, m) {
  m.impl("conv3x3_fwd", &conv3x3_fwd);
  m.impl("conv3x3_dgrad", &conv3x3_dgrad);
  m.impl("normalize", &normalize);
  m.impl("denormalize", &denormalize);
  m.impl("image_upsample", &image_upsample);
  m.impl("adam_step", &adam_step);
  m.impl("grad_clip_coef", &grad_clip_coef);
  m.impl("adam_step_clip", &adam_step_clip);
}
