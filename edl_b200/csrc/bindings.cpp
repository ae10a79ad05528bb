// torch <-> edl_b200 kernel bindings.  Only this file includes torch headers; the kernels are in
// torch-free .cu files (see kernels.h).  Every entry point launches on the current CUDA stream so
// the ops are capturable into CUDA graphs.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include "gemm.h"
#include "kernels.h"
#include "launch.h"

namespace {

using torch::Tensor;

inline cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

inline void check_bf16(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
  TORCH_CHECK(t.scalar_type() == at::kBFloat16, name, " must be bf16");
  TORCH_CHECK(t.is_contiguous(), name, " must be contiguous");
}
inline void check_f32(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
  TORCH_CHECK(t.scalar_type() == at::kFloat, name, " must be fp32");
  TORCH_CHECK(t.is_contiguous(), name, " must be contiguous");
}
template <typename T>
inline T* opt_ptr(const c10::optional<Tensor>& t) {
  return t.has_value() && t->defined() ? reinterpret_cast<T*>(t->data_ptr()) : nullptr;
}

// ------------------------------------------------------------------ batch norm (NHWC, [M, C])
void bn_stats(const Tensor& x, Tensor& sums) {
  check_bf16(x, "x");
  check_f32(sums, "sums");
  const int C = x.size(-1);
  const int64_t M = x.numel() / C;
  TORCH_CHECK(C % 8 == 0 && sums.numel() == 2 * C);
  c10::cuda::CUDAGuard g(x.device());
  edl::bn_stats(x.data_ptr(), sums.data_ptr<float>(), M, C, cur_stream());
}

void bn_apply(const Tensor& x, const c10::optional<Tensor>& res, Tensor& y, const Tensor& sums,
              const Tensor& gamma, const Tensor& beta, const c10::optional<Tensor>& running_mean,
              const c10::optional<Tensor>& running_var, Tensor& saved_mean, Tensor& saved_rstd,
              double eps, double momentum, bool relu) {
  check_bf16(x, "x");
  check_bf16(y, "y");
  check_f32(gamma, "gamma");
  check_f32(beta, "beta");
  const int C = x.size(-1);
  const int64_t M = x.numel() / C;
  c10::cuda::CUDAGuard g(x.device());
  edl::bn_apply(x.data_ptr(), opt_ptr<void>(res), y.data_ptr(), sums.data_ptr<float>(),
                gamma.data_ptr<float>(), beta.data_ptr<float>(), opt_ptr<float>(running_mean),
                opt_ptr<float>(running_var), saved_mean.data_ptr<float>(),
                saved_rstd.data_ptr<float>(), M, C, (float)eps, (float)momentum, relu,
                cur_stream());
}

void scale_shift_act(const Tensor& x, const c10::optional<Tensor>& res, Tensor& y,
                     const Tensor& scale, const Tensor& shift, bool relu) {
  check_bf16(x, "x");
  check_bf16(y, "y");
  check_f32(scale, "scale");
  check_f32(shift, "shift");
  const int C = x.size(-1);
  const int64_t M = x.numel() / C;
  c10::cuda::CUDAGuard g(x.device());
  edl::scale_shift_act(x.data_ptr(), opt_ptr<void>(res), y.data_ptr(), scale.data_ptr<float>(),
                       shift.data_ptr<float>(), M, C, relu, cur_stream());
}

void bn_bwd_reduce(const Tensor& dy, const Tensor& x, const c10::optional<Tensor>& y,
                   const Tensor& gamma, const Tensor& beta, const Tensor& saved_mean,
                   const Tensor& saved_rstd, Tensor& dsums, bool relu) {
  check_bf16(dy, "dy");
  check_bf16(x, "x");
  const int C = x.size(-1);
  const int64_t M = x.numel() / C;
  c10::cuda::CUDAGuard g(x.device());
  edl::bn_bwd_reduce(dy.data_ptr(), x.data_ptr(), opt_ptr<void>(y), gamma.data_ptr<float>(),
                     beta.data_ptr<float>(), saved_mean.data_ptr<float>(),
                     saved_rstd.data_ptr<float>(), dsums.data_ptr<float>(), M, C, relu,
                     cur_stream());
}

void bn_bwd_apply(const Tensor& dy, const Tensor& x, const c10::optional<Tensor>& y,
                  const Tensor& gamma, const Tensor& beta, const Tensor& saved_mean,
                  const Tensor& saved_rstd,
                  const Tensor& dsums, Tensor& dx, const c10::optional<Tensor>& dres,
                  const c10::optional<Tensor>& dgamma, const c10::optional<Tensor>& dbeta,
                  bool relu, bool accumulate) {
  check_bf16(dy, "dy");
  check_bf16(x, "x");
  check_bf16(dx, "dx");
  const int C = x.size(-1);
  const int64_t M = x.numel() / C;
  c10::cuda::CUDAGuard g(x.device());
  edl::bn_bwd_apply(dy.data_ptr(), x.data_ptr(), opt_ptr<void>(y), gamma.data_ptr<float>(),
                    beta.data_ptr<float>(), saved_mean.data_ptr<float>(),
                    saved_rstd.data_ptr<float>(),
                    dsums.data_ptr<float>(), dx.data_ptr(), opt_ptr<void>(dres),
                    opt_ptr<float>(dgamma), opt_ptr<float>(dbeta), M, C, relu, accumulate,
                    cur_stream());
}

bool bn_fused_fits(int64_t M, int64_t C, int64_t num_operands) {
  return edl::bn_fused_fits(M, (int)C, (int)num_operands);
}

void bn_fwd_fused(const Tensor& x, const c10::optional<Tensor>& res, Tensor& y, Tensor& sums,
                  const Tensor& gamma, const Tensor& beta, const c10::optional<Tensor>& running_mean,
                  const c10::optional<Tensor>& running_var, Tensor& saved_mean, Tensor& saved_rstd,
                  double eps, double momentum, bool relu, Tensor& sync_counter) {
  check_bf16(x, "x");
  check_bf16(y, "y");
  check_f32(sums, "sums");
  TORCH_CHECK(sync_counter.scalar_type() == at::kInt && sync_counter.is_cuda());
  const int C = x.size(-1);
  const int64_t M = x.numel() / C;
  c10::cuda::CUDAGuard g(x.device());
  const char* err = edl::bn_fwd_fused(
      x.data_ptr(), opt_ptr<void>(res), y.data_ptr(), sums.data_ptr<float>(), gamma.data_ptr<float>(),
      beta.data_ptr<float>(), opt_ptr<float>(running_mean), opt_ptr<float>(running_var),
      saved_mean.data_ptr<float>(), saved_rstd.data_ptr<float>(), M, C, (float)eps, (float)momentum, relu,
      reinterpret_cast<unsigned int*>(sync_counter.data_ptr<int>()), cur_stream());
  TORCH_CHECK(err == nullptr, "bn_fwd_fused: ", err);
}

void bn_bwd_fused(const Tensor& dy, const Tensor& x, const c10::optional<Tensor>& y, const Tensor& gamma,
                  const Tensor& beta, const Tensor& saved_mean, const Tensor& saved_rstd, Tensor& dsums,
                  Tensor& dx, const c10::optional<Tensor>& dres, const c10::optional<Tensor>& dgamma,
                  const c10::optional<Tensor>& dbeta, bool relu, bool accumulate, Tensor& sync_counter) {
  check_bf16(dy, "dy");
  check_bf16(x, "x");
  check_bf16(dx, "dx");
  TORCH_CHECK(sync_counter.scalar_type() == at::kInt && sync_counter.is_cuda());
  const int C = x.size(-1);
  const int64_t M = x.numel() / C;
  c10::cuda::CUDAGuard g(x.device());
  const char* err = edl::bn_bwd_fused(
      dy.data_ptr(), x.data_ptr(), opt_ptr<void>(y), gamma.data_ptr<float>(), beta.data_ptr<float>(),
      saved_mean.data_ptr<float>(), saved_rstd.data_ptr<float>(), dsums.data_ptr<float>(), dx.data_ptr(),
      opt_ptr<void>(dres), opt_ptr<float>(dgamma), opt_ptr<float>(dbeta), M, C, relu, accumulate,
      reinterpret_cast<unsigned int*>(sync_counter.data_ptr<int>()), cur_stream());
  TORCH_CHECK(err == nullptr, "bn_bwd_fused: ", err);
}

// ------------------------------------------------------------------ optimizers
void sgd_momentum(const c10::optional<Tensor>& param_lp, Tensor& master, Tensor& mom,
                  const Tensor& grad, const c10::optional<Tensor>& wd_mask, const Tensor& lr,
                  const c10::optional<Tensor>& grad_scale, const c10::optional<Tensor>& found_inf,
                  double momentum, double wd, bool nesterov) {
  check_f32(master, "master");
  check_f32(mom, "mom");
  check_f32(lr, "lr");
  TORCH_CHECK(grad.is_cuda() && grad.is_contiguous());
  const bool gbf = grad.scalar_type() == at::kBFloat16;
  TORCH_CHECK(gbf || grad.scalar_type() == at::kFloat);
  const int64_t n = master.numel();
  TORCH_CHECK(grad.numel() == n && mom.numel() == n);
  c10::cuda::CUDAGuard g(master.device());
  edl::sgd_momentum(opt_ptr<void>(param_lp), master.data_ptr<float>(), mom.data_ptr<float>(),
                    grad.data_ptr(), gbf, opt_ptr<float>(wd_mask), n, lr.data_ptr<float>(),
                    opt_ptr<float>(grad_scale), opt_ptr<int>(found_inf), (float)momentum,
                    (float)wd, nesterov, cur_stream());
}

void adam_step(const c10::optional<Tensor>& param_lp, Tensor& master, Tensor& m, Tensor& v,
               const Tensor& grad, const Tensor& lr, const c10::optional<Tensor>& grad_scale,
               const c10::optional<Tensor>& found_inf, const Tensor& step, double beta1,
               double beta2, double eps, double wd, bool decoupled) {
  check_f32(master, "master");
  const bool gbf = grad.scalar_type() == at::kBFloat16;
  const int64_t n = master.numel();
  c10::cuda::CUDAGuard g(master.device());
  edl::adam_step(opt_ptr<void>(param_lp), master.data_ptr<float>(), m.data_ptr<float>(),
                 v.data_ptr<float>(), grad.data_ptr(), gbf, n, lr.data_ptr<float>(),
                 opt_ptr<float>(grad_scale), opt_ptr<int>(found_inf), step.data_ptr<float>(),
                 (float)beta1, (float)beta2, (float)eps, (float)wd, decoupled, cur_stream());
}

// LARS / LAMB: `chunks` is the int64 [nchunks, 5] table of optim_layerwise.cu with offsets into these (window)
// tensors, `partials` fp32 scratch of >= 2 * nchunks floats.  Every chunk start must be a multiple of 8 elements.
bool check_layerwise(const c10::optional<Tensor>& param_lp, const Tensor& master, const Tensor& grad,
                            const Tensor& chunks, const Tensor& partials, const Tensor& lr) {
  check_f32(master, "master");
  check_f32(partials, "partials");
  check_f32(lr, "lr");
  TORCH_CHECK(grad.is_cuda() && grad.is_contiguous(), "grad must be a contiguous CUDA tensor");
  const bool gbf = grad.scalar_type() == at::kBFloat16;
  TORCH_CHECK(gbf || grad.scalar_type() == at::kFloat, "grad must be bf16 or fp32");
  TORCH_CHECK(grad.numel() == master.numel(), "grad / master size mismatch");
  TORCH_CHECK(chunks.is_cuda() && chunks.scalar_type() == at::kLong && chunks.is_contiguous() && chunks.dim() == 2 &&
                  chunks.size(1) == 5, "chunks must be a contiguous CUDA int64 [n, 5] table");
  TORCH_CHECK(partials.numel() >= 2 * chunks.size(0), "partials too small");
  TORCH_CHECK(reinterpret_cast<uintptr_t>(master.data_ptr()) % 16 == 0 &&
                  reinterpret_cast<uintptr_t>(grad.data_ptr()) % 16 == 0, "master / grad must be 16-byte aligned");
  if (param_lp.has_value() && param_lp->defined()) {
    check_bf16(*param_lp, "param_lp");
    TORCH_CHECK(param_lp->numel() == master.numel(), "param_lp / master size mismatch");
    TORCH_CHECK(reinterpret_cast<uintptr_t>(param_lp->data_ptr()) % 16 == 0, "param_lp must be 16-byte aligned");
  }
  return gbf;
}

void lars_step(const c10::optional<Tensor>& param_lp, Tensor& master, Tensor& mom, const Tensor& grad,
               const Tensor& chunks, Tensor& partials, const Tensor& lr, const c10::optional<Tensor>& grad_scale,
               const c10::optional<Tensor>& found_inf, double momentum, double lars_coeff, double wd, double eps) {
  const bool gbf = check_layerwise(param_lp, master, grad, chunks, partials, lr);
  check_f32(mom, "mom");
  TORCH_CHECK(mom.numel() == master.numel() && reinterpret_cast<uintptr_t>(mom.data_ptr()) % 16 == 0);
  c10::cuda::CUDAGuard g(master.device());
  edl::lars_step(opt_ptr<void>(param_lp), master.data_ptr<float>(), mom.data_ptr<float>(), grad.data_ptr(), gbf,
                 chunks.data_ptr<int64_t>(), (int)chunks.size(0), partials.data_ptr<float>(), lr.data_ptr<float>(),
                 opt_ptr<float>(grad_scale), opt_ptr<int>(found_inf), (float)momentum, (float)lars_coeff, (float)wd,
                 (float)eps, cur_stream());
}

void lamb_step(const c10::optional<Tensor>& param_lp, Tensor& master, Tensor& m, Tensor& v, const Tensor& grad,
               const Tensor& chunks, Tensor& partials, const Tensor& lr, const c10::optional<Tensor>& grad_scale,
               const c10::optional<Tensor>& found_inf, const Tensor& step, double beta1, double beta2, double eps,
               double wd) {
  const bool gbf = check_layerwise(param_lp, master, grad, chunks, partials, lr);
  check_f32(m, "m");
  check_f32(v, "v");
  check_f32(step, "step");
  TORCH_CHECK(m.numel() == master.numel() && v.numel() == master.numel());
  TORCH_CHECK(reinterpret_cast<uintptr_t>(m.data_ptr()) % 16 == 0 && reinterpret_cast<uintptr_t>(v.data_ptr()) % 16 == 0);
  c10::cuda::CUDAGuard g(master.device());
  edl::lamb_step(opt_ptr<void>(param_lp), master.data_ptr<float>(), m.data_ptr<float>(), v.data_ptr<float>(),
                 grad.data_ptr(), gbf, chunks.data_ptr<int64_t>(), (int)chunks.size(0), partials.data_ptr<float>(),
                 lr.data_ptr<float>(), opt_ptr<float>(grad_scale), opt_ptr<int>(found_inf), step.data_ptr<float>(),
                 (float)beta1, (float)beta2, (float)eps, (float)wd, cur_stream());
}

// ------------------------------------------------------------------ losses
void soft_ce_fwd(const Tensor& logits, const c10::optional<Tensor>& target,
                 const c10::optional<Tensor>& labels, Tensor& loss_out, Tensor& row_stats,
                 int64_t mode, double s_temp, double t_temp, double label_smooth, bool kl,
                 double loss_scale) {
  TORCH_CHECK(logits.is_cuda() && logits.is_contiguous() && logits.dim() == 2);
  const int N = logits.size(0), C = logits.size(1);
  const bool lbf = logits.scalar_type() == at::kBFloat16;
  bool tbf = false;
  if (mode != 2) {
    TORCH_CHECK(target.has_value() && target->is_contiguous() && target->numel() == logits.numel());
    tbf = target->scalar_type() == at::kBFloat16;
    TORCH_CHECK(tbf || target->scalar_type() == at::kFloat);
  } else {
    TORCH_CHECK(labels.has_value() && labels->scalar_type() == at::kLong);
  }
  c10::cuda::CUDAGuard g(logits.device());
  edl::soft_ce_fwd(logits.data_ptr(), lbf, opt_ptr<void>(target), tbf, opt_ptr<int64_t>(labels),
                   loss_out.data_ptr<float>(), row_stats.data_ptr<float>(), N, C, (int)mode,
                   (float)s_temp, (float)t_temp, (float)label_smooth, kl, (float)loss_scale,
                   cur_stream());
}

void soft_ce_bwd(const Tensor& logits, const c10::optional<Tensor>& target,
                 const c10::optional<Tensor>& labels, const Tensor& row_stats,
                 const c10::optional<Tensor>& grad_out, Tensor& dlogits, int64_t mode,
                 double s_temp, double t_temp, double label_smooth, double loss_scale) {
  const int N = logits.size(0), C = logits.size(1);
  const bool lbf = logits.scalar_type() == at::kBFloat16;
  const bool tbf = mode != 2 && target->scalar_type() == at::kBFloat16;
  c10::cuda::CUDAGuard g(logits.device());
  edl::soft_ce_bwd(logits.data_ptr(), lbf, opt_ptr<void>(target), tbf, opt_ptr<int64_t>(labels),
                   row_stats.data_ptr<float>(), opt_ptr<float>(grad_out), dlogits.data_ptr(), N, C,
                   (int)mode, (float)s_temp, (float)t_temp, (float)label_smooth,
                   (float)loss_scale, cur_stream());
}

void topk_acc(const Tensor& logits, const Tensor& labels, Tensor& counts) {
  const int N = logits.size(0), C = logits.size(1);
  c10::cuda::CUDAGuard g(logits.device());
  edl::topk_acc(logits.data_ptr(), logits.scalar_type() == at::kBFloat16,
                labels.data_ptr<int64_t>(), counts.data_ptr<float>(), N, C, cur_stream());
}

// ------------------------------------------------------------------ pooling (NHWC)
void maxpool3x3s2_fwd(const Tensor& x, Tensor& y, Tensor& idx) {
  check_bf16(x, "x");
  c10::cuda::CUDAGuard g(x.device());
  edl::maxpool3x3s2_fwd(x.data_ptr(), y.data_ptr(), idx.data_ptr<uint8_t>(), x.size(0), x.size(1),
                        x.size(2), x.size(3), cur_stream());
}
void maxpool3x3s2_bwd(const Tensor& dy, const Tensor& idx, Tensor& dx) {
  check_bf16(dy, "dy");
  c10::cuda::CUDAGuard g(dy.device());
  edl::maxpool3x3s2_bwd(dy.data_ptr(), idx.data_ptr<uint8_t>(), dx.data_ptr(), dx.size(0),
                        dx.size(1), dx.size(2), dx.size(3), cur_stream());
}
void avgpool2x2_fwd(const Tensor& x, Tensor& y) {
  check_bf16(x, "x");
  c10::cuda::CUDAGuard g(x.device());
  edl::avgpool2x2_fwd(x.data_ptr(), y.data_ptr(), x.size(0), x.size(1), x.size(2), x.size(3),
                      cur_stream());
}
void avgpool2x2_bwd(const Tensor& dy, Tensor& dx) {
  check_bf16(dy, "dy");
  c10::cuda::CUDAGuard g(dy.device());
  edl::avgpool2x2_bwd(dy.data_ptr(), dx.data_ptr(), dx.size(0), dx.size(1), dx.size(2),
                      dx.size(3), cur_stream());
}
void gap_fwd(const Tensor& x, Tensor& y) {
  check_bf16(x, "x");
  c10::cuda::CUDAGuard g(x.device());
  edl::gap_fwd(x.data_ptr(), y.data_ptr(), x.size(0), x.size(1) * x.size(2), x.size(3),
               cur_stream());
}
void dilate2(const Tensor& x, Tensor& y) {
  TORCH_CHECK(x.is_cuda() && x.dim() == 4 && x.scalar_type() == at::kBFloat16 &&
              x.is_contiguous(at::MemoryFormat::ChannelsLast), "dilate2: x must be a channels_last bf16 NCHW tensor");
  TORCH_CHECK(y.is_cuda() && y.scalar_type() == at::kBFloat16 && y.is_contiguous(at::MemoryFormat::ChannelsLast));
  TORCH_CHECK(y.size(0) == x.size(0) && y.size(1) == x.size(1) && y.size(2) == 2 * x.size(2) && y.size(3) == 2 * x.size(3));
  TORCH_CHECK(x.size(1) % 8 == 0);
  c10::cuda::CUDAGuard g(x.device());
  edl::dilate2(x.data_ptr(), y.data_ptr(), x.size(0), x.size(2), x.size(3), x.size(1), cur_stream());
}
void gap_bwd(const Tensor& dy, Tensor& dx) {
  check_bf16(dy, "dy");
  c10::cuda::CUDAGuard g(dy.device());
  edl::gap_bwd(dy.data_ptr(), dx.data_ptr(), dx.size(0), dx.size(1) * dx.size(2), dx.size(3),
               cur_stream());
}

// ------------------------------------------------------------------ collectives
edl::CommHandles make_handles(const std::vector<int64_t>& data_ptrs,
                              const std::vector<int64_t>& sig_ptrs, int64_t mc_ptr, int64_t rank,
                              double timeout_s) {
  edl::CommHandles h{};
  const int world = (int)data_ptrs.size();
  TORCH_CHECK(world >= 1 && world <= edl::comm_max_world(), "unsupported world size ", world);
  TORCH_CHECK(sig_ptrs.size() == data_ptrs.size());
  for (int i = 0; i < world; ++i) {
    h.data[i] = reinterpret_cast<void*>(data_ptrs[i]);
    h.sig[i] = reinterpret_cast<void*>(sig_ptrs[i]);
  }
  h.mc_data = reinterpret_cast<void*>(mc_ptr);
  h.rank = (int)rank;
  h.world = world;
  h.timeout_ns = (unsigned long long)(timeout_s * 1e9);
  return h;
}

void allreduce_oneshot(const std::vector<int64_t>& data_ptrs, const std::vector<int64_t>& sig_ptrs,
                       int64_t rank, Tensor& out, int64_t n, double scale,
                       const c10::optional<Tensor>& found_inf, const c10::optional<Tensor>& sqnorm,
                       int64_t nblocks, double timeout_s) {
  auto h = make_handles(data_ptrs, sig_ptrs, 0, rank, timeout_s);
  c10::cuda::CUDAGuard g(out.device());
  edl::allreduce_oneshot(h, out.data_ptr(), out.scalar_type() == at::kBFloat16, n, (float)scale,
                         opt_ptr<int>(found_inf), opt_ptr<float>(sqnorm), (int)nblocks,
                         cur_stream());
}

void allreduce_twoshot(const std::vector<int64_t>& data_ptrs, const std::vector<int64_t>& sig_ptrs,
                       int64_t mc_ptr, int64_t rank, const Tensor& local, int64_t n, double scale,
                       const c10::optional<Tensor>& found_inf, const c10::optional<Tensor>& sqnorm,
                       bool multimem, int64_t nblocks, double timeout_s) {
  auto h = make_handles(data_ptrs, sig_ptrs, mc_ptr, rank, timeout_s);
  const bool bf = local.scalar_type() == at::kBFloat16;
  const int ve = bf ? 8 : 4;
  TORCH_CHECK(n % ve == 0, "two-shot needs n to be a multiple of 16 bytes");
  c10::cuda::CUDAGuard g(local.device());
  edl::allreduce_twoshot(h, bf, n, (float)scale, opt_ptr<int>(found_inf), opt_ptr<float>(sqnorm),
                         multimem, (int)nblocks, cur_stream());
}

// one bf16 bucket: gradient reduce-scatter -> SGD-momentum on the owned slice -> parameter all-gather
void allreduce_sgd(const std::vector<int64_t>& grad_ptrs, const std::vector<int64_t>& sig_ptrs, int64_t mc_grad,
                   const std::vector<int64_t>& param_ptrs, int64_t mc_param, int64_t rank, Tensor& master,
                   Tensor& mom, const c10::optional<Tensor>& wd_mask, const Tensor& lr, double scale,
                   const c10::optional<Tensor>& found_inf_out, const c10::optional<Tensor>& sqnorm,
                   const c10::optional<Tensor>& skip_flag, double momentum, double wd, bool nesterov,
                   bool multimem, int64_t nblocks, double timeout_s) {
  auto h = make_handles(grad_ptrs, sig_ptrs, mc_grad, rank, timeout_s);
  check_f32(master, "master");
  check_f32(mom, "mom");
  check_f32(lr, "lr");
  const int64_t n = master.numel();
  TORCH_CHECK(n % 8 == 0 && mom.numel() == n, "fused bucket must be a multiple of 8 elements");
  TORCH_CHECK(param_ptrs.size() == grad_ptrs.size());
  TORCH_CHECK(reinterpret_cast<uintptr_t>(master.data_ptr()) % 16 == 0 && reinterpret_cast<uintptr_t>(mom.data_ptr()) % 16 == 0);
  void* pp[16] = {};
  for (size_t i = 0; i < param_ptrs.size(); ++i) pp[i] = reinterpret_cast<void*>(param_ptrs[i]);
  c10::cuda::CUDAGuard g(master.device());
  edl::allreduce_sgd(h, pp, reinterpret_cast<void*>(mc_param), master.data_ptr<float>(), mom.data_ptr<float>(),
                     opt_ptr<float>(wd_mask), n, (float)scale, opt_ptr<int>(found_inf_out), opt_ptr<float>(sqnorm),
                     lr.data_ptr<float>(), opt_ptr<int>(skip_flag), (float)momentum, (float)wd, nesterov, multimem,
                     (int)nblocks, cur_stream());
}

void grad_sqnorm(const Tensor& grad, Tensor& out) {
  TORCH_CHECK(grad.is_cuda() && grad.is_contiguous());
  check_f32(out, "out");
  const bool gbf = grad.scalar_type() == at::kBFloat16;
  TORCH_CHECK(gbf || grad.scalar_type() == at::kFloat);
  c10::cuda::CUDAGuard g(grad.device());
  edl::grad_sqnorm(grad.data_ptr(), gbf, grad.numel(), out.data_ptr<float>(), cur_stream());
}

void clip_scale(const Tensor& parts, int64_t nparts, int64_t stride, double max_norm, Tensor& grad_scale,
                const c10::optional<Tensor>& norm_out) {
  check_f32(parts, "parts");
  check_f32(grad_scale, "grad_scale");
  TORCH_CHECK(nparts >= 1 && (nparts - 1) * stride < parts.numel());
  c10::cuda::CUDAGuard g(parts.device());
  edl::clip_scale(parts.data_ptr<float>(), (int)nparts, (int)stride, (float)max_norm, grad_scale.data_ptr<float>(),
                  opt_ptr<float>(norm_out), cur_stream());
}

void comm_broadcast(const std::vector<int64_t>& data_ptrs, const std::vector<int64_t>& sig_ptrs,
                    int64_t rank, int64_t root, int64_t nbytes, int64_t nblocks, double timeout_s,
                    const Tensor& local) {
  auto h = make_handles(data_ptrs, sig_ptrs, 0, rank, timeout_s);
  c10::cuda::CUDAGuard g(local.device());
  edl::comm_broadcast(h, (int)root, nbytes, (int)nblocks, cur_stream());
}

void comm_allgather_scalars(const std::vector<int64_t>& data_ptrs,
                            const std::vector<int64_t>& sig_ptrs, int64_t rank, const Tensor& in,
                            Tensor& out, double timeout_s) {
  auto h = make_handles(data_ptrs, sig_ptrs, 0, rank, timeout_s);
  TORCH_CHECK(in.numel() <= 8);
  c10::cuda::CUDAGuard g(in.device());
  edl::comm_allgather_scalars(h, in.data_ptr<float>(), out.data_ptr<float>(), (int)in.numel(),
                              cur_stream());
}

// ------------------------------------------------------------------ misc fused ops
void rope(const Tensor& x, const Tensor& cosv, const Tensor& sinv, Tensor& y, bool inverse) {
  check_bf16(x, "x");
  check_f32(cosv, "cos");
  check_f32(sinv, "sin");
  TORCH_CHECK(x.dim() == 3 && x.size(2) % 2 == 0 && cosv.size(0) == x.size(0) && cosv.size(1) == x.size(2) / 2);
  c10::cuda::CUDAGuard g(x.device());
  edl::rope(x.data_ptr(), cosv.data_ptr<float>(), sinv.data_ptr<float>(), y.data_ptr(), x.size(0), x.size(1),
            x.size(2), inverse, cur_stream());
}

// y [N,32,Ho,Wo] = conv3x3/s2/p1(x [N,3,H,W], w KRSC [32,3,3,3]), channels_last bf16; stats fp32 [64] += (sum, sum^2) of y
void stem_conv3x3s2(const Tensor& x, const Tensor& w, Tensor& y, const c10::optional<Tensor>& stats) {
  TORCH_CHECK(x.is_cuda() && x.dim() == 4 && x.size(1) == 3 && x.scalar_type() == at::kBFloat16);
  TORCH_CHECK(x.is_contiguous(at::MemoryFormat::ChannelsLast) && y.is_contiguous(at::MemoryFormat::ChannelsLast));
  TORCH_CHECK(w.scalar_type() == at::kBFloat16 && w.is_contiguous() && w.dim() == 4 && w.size(0) == 32 && w.size(1) == 3 &&
              w.size(2) == 3 && w.size(3) == 3, "stem weight must be KRSC [32,3,3,3] bf16");
  const int64_t H = x.size(2), W = x.size(3);
  TORCH_CHECK(y.scalar_type() == at::kBFloat16 && y.size(0) == x.size(0) && y.size(1) == 32 &&
              y.size(2) == (H - 1) / 2 + 1 && y.size(3) == (W - 1) / 2 + 1);
  float* st = nullptr;
  if (stats.has_value() && stats->defined()) {
    TORCH_CHECK(stats->scalar_type() == at::kFloat && stats->numel() >= 64 && stats->is_contiguous() &&
                reinterpret_cast<uintptr_t>(stats->data_ptr()) % 16 == 0);
    st = stats->data_ptr<float>();
  }
  c10::cuda::CUDAGuard guard(x.device());
  edl::stem_conv3x3s2(x.data_ptr(), w.data_ptr(), y.data_ptr(), st, (int)x.size(0), (int)H, (int)W,
                      at::cuda::getCurrentCUDAStream().stream());
}

// a [N * Ho * Wo, 160] = im2col of the 7x7 / stride 2 / pad 3 stem convolution of x [N,3,H,W] channels_last bf16
void stem7_im2col(const Tensor& x, Tensor& a) {
  TORCH_CHECK(x.is_cuda() && x.dim() == 4 && x.size(1) == 3 && x.scalar_type() == at::kBFloat16 &&
              x.is_contiguous(at::MemoryFormat::ChannelsLast), "stem7_im2col: x must be [N,3,H,W] channels_last bf16");
  const int64_t H = x.size(2), W = x.size(3), Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  TORCH_CHECK(a.is_cuda() && a.scalar_type() == at::kBFloat16 && a.is_contiguous() && a.dim() == 2 &&
              a.size(0) == x.size(0) * Ho * Wo && a.size(1) == 160, "stem7_im2col: a must be [N*Ho*Wo, 160] bf16");
  c10::cuda::CUDAGuard guard(x.device());
  const char* err = edl::stem7_im2col(x.data_ptr(), a.data_ptr(), (int)x.size(0), (int)H, (int)W,
                                      at::cuda::getCurrentCUDAStream().stream());
  TORCH_CHECK(err == nullptr, err);
}

// dw KRSC [32,3,3,3] bf16 (+)= wgrad of the stem convolution; x [N,3,H,W], dy [N,32,H/2,W/2] channels_last bf16
void stem_wgrad(const Tensor& x, const Tensor& dy, Tensor& dw, Tensor& ws, Tensor& counter, bool accumulate) {
  TORCH_CHECK(x.is_cuda() && x.dim() == 4 && x.size(1) == 3 && x.scalar_type() == at::kBFloat16 &&
              x.is_contiguous(at::MemoryFormat::ChannelsLast));
  TORCH_CHECK(dy.dim() == 4 && dy.size(1) == 32 && dy.scalar_type() == at::kBFloat16 &&
              dy.is_contiguous(at::MemoryFormat::ChannelsLast) && dy.size(0) == x.size(0) &&
              dy.size(2) * 2 == x.size(2) && dy.size(3) * 2 == x.size(3));
  TORCH_CHECK(dw.scalar_type() == at::kBFloat16 && dw.is_contiguous() && dw.numel() == 864);
  TORCH_CHECK(ws.scalar_type() == at::kFloat && ws.is_contiguous() && ws.numel() >= 864 &&
              reinterpret_cast<uintptr_t>(ws.data_ptr()) % 16 == 0);
  TORCH_CHECK(counter.scalar_type() == at::kInt && counter.numel() >= 1);
  c10::cuda::CUDAGuard guard(x.device());
  const char* err = edl::stem_wgrad(x.data_ptr(), dy.data_ptr(), ws.data_ptr<float>(), counter.data_ptr<int>(),
                                    dw.data_ptr(), accumulate, (int)x.size(0), (int)x.size(2), (int)x.size(3),
                                    at::cuda::getCurrentCUDAStream().stream());
  TORCH_CHECK(err == nullptr, "stem_wgrad: ", err);
}

void pair_weight_expand(const Tensor& w, Tensor& w2) {
  check_bf16(w, "w");
  check_bf16(w2, "w2");
  TORCH_CHECK(w.dim() == 4 && w.size(1) == 3 && w.size(2) == 3 && w.size(3) == 32 && w2.numel() == 4 * w.numel());
  c10::cuda::CUDAGuard g(w.device());
  edl::pair_weight_expand(w.data_ptr(), w2.data_ptr(), (int)w.size(0), cur_stream());
}
void pair_weight_fold(const Tensor& dw2, Tensor& dw, bool accumulate) {
  check_bf16(dw2, "dw2");
  check_bf16(dw, "dw");
  TORCH_CHECK(dw.numel() % (9 * 32) == 0 && dw2.numel() == 4 * dw.numel());
  c10::cuda::CUDAGuard g(dw.device());
  edl::pair_weight_fold(dw2.data_ptr(), dw.data_ptr(), (int)(dw.numel() / (9 * 32)), accumulate, cur_stream());
}
void fold_pair_stats(const Tensor& s2, Tensor& stats) {
  check_f32(s2, "s2");
  check_f32(stats, "stats");
  TORCH_CHECK(s2.numel() == 2 * stats.numel() && stats.numel() % 2 == 0);
  c10::cuda::CUDAGuard g(stats.device());
  edl::fold_pair_stats(s2.data_ptr<float>(), stats.data_ptr<float>(), (int)(stats.numel() / 2), cur_stream());
}

void embedding_bag_fwd(const Tensor& table, const Tensor& ids, Tensor& out) {
  TORCH_CHECK(table.is_cuda() && table.is_contiguous() && ids.is_contiguous() && ids.scalar_type() == at::kLong);
  c10::cuda::CUDAGuard g(table.device());
  edl::embedding_bag_fwd(table.data_ptr(), table.scalar_type() == at::kBFloat16, ids.data_ptr<int64_t>(),
                         out.data_ptr(), ids.size(0), ids.size(1), table.size(1), cur_stream());
}

void embedding_bag_bwd(const Tensor& dout, const Tensor& ids, Tensor& dtable) {
  check_f32(dtable, "dtable");
  c10::cuda::CUDAGuard g(dout.device());
  edl::embedding_bag_bwd(dout.data_ptr(), dout.scalar_type() == at::kBFloat16, ids.data_ptr<int64_t>(),
                         dtable.data_ptr<float>(), ids.size(0), ids.size(1), dtable.size(1), cur_stream());
}

void normalize_u8(const Tensor& x, Tensor& y, std::vector<double> mean, std::vector<double> stdv,
                  const c10::optional<Tensor>& flip) {
  TORCH_CHECK(x.is_cuda() && x.scalar_type() == at::kByte && x.is_contiguous() && x.dim() == 4 && x.size(3) == 3);
  check_bf16(y, "y");
  const float m[3] = {(float)mean[0], (float)mean[1], (float)mean[2]};
  const float sd[3] = {(float)stdv[0], (float)stdv[1], (float)stdv[2]};
  c10::cuda::CUDAGuard g(x.device());
  edl::normalize_u8(x.data_ptr<uint8_t>(), y.data_ptr(), x.size(0), x.size(1), x.size(2), m, sd,
                    opt_ptr<uint8_t>(flip), cur_stream());
}

// ------------------------------------------------------------------ logit ship / device distill feed
// Raw peer addresses (ints) come from parallel.symm.SymmSlice; local tensors are torch tensors.
void peer_ship(const Tensor& src, int64_t dst_peer, int64_t nbytes, int64_t flag_peer,
               const c10::optional<Tensor>& seq, int64_t seq_imm, Tensor& done) {
  TORCH_CHECK(src.is_cuda() && src.is_contiguous() && nbytes % 16 == 0);
  c10::cuda::CUDAGuard g(src.device());
  edl::peer_ship(src.data_ptr(), reinterpret_cast<void*>(dst_peer), nbytes, reinterpret_cast<void*>(flag_peer),
                 opt_ptr<void>(seq), (uint32_t)seq_imm, done.data_ptr(), cur_stream());
}

void logit_ship(const Tensor& logits, int64_t slot_peer, int64_t stats_peer, double temperature,
                int64_t flag_peer, const c10::optional<Tensor>& seq, int64_t seq_imm, Tensor& done) {
  check_bf16(logits, "logits");
  TORCH_CHECK(logits.dim() == 2);
  c10::cuda::CUDAGuard g(logits.device());
  edl::logit_ship(logits.data_ptr(), reinterpret_cast<void*>(slot_peer), reinterpret_cast<float*>(stats_peer),
                  logits.size(0), logits.size(1), (float)temperature, reinterpret_cast<void*>(flag_peer),
                  opt_ptr<void>(seq), (uint32_t)seq_imm, done.data_ptr(), cur_stream());
}

void soft_ce_recv(const Tensor& logits, const Tensor& slot, const c10::optional<Tensor>& slot_stats, const Tensor& flag,
                  const c10::optional<Tensor>& seq, int64_t seq_imm, Tensor& loss_out, Tensor& row_stats,
                  double s_temp, double t_temp, bool kl, double loss_scale, double timeout_s,
                  const c10::optional<Tensor>& err) {
  TORCH_CHECK(logits.is_cuda() && logits.is_contiguous() && logits.dim() == 2);
  c10::cuda::CUDAGuard g(logits.device());
  edl::soft_ce_recv(logits.data_ptr(), logits.scalar_type() == at::kBFloat16, slot.data_ptr(),
                    opt_ptr<float>(slot_stats), flag.data_ptr(), opt_ptr<void>(seq), (uint32_t)seq_imm,
                    loss_out.data_ptr<float>(), row_stats.data_ptr<float>(), logits.size(0), logits.size(1),
                    (float)s_temp, (float)t_temp, kl, (float)loss_scale, timeout_s, opt_ptr<void>(err),
                    cur_stream());
}

void slot_ack(int64_t ack_peer, const c10::optional<Tensor>& seq, int64_t seq_imm, const Tensor& any_local) {
  c10::cuda::CUDAGuard g(any_local.device());
  edl::slot_ack(reinterpret_cast<void*>(ack_peer), opt_ptr<void>(seq), (uint32_t)seq_imm, cur_stream());
}

void wait_flag_async(const Tensor& flag, const c10::optional<Tensor>& seq, int64_t seq_imm, double timeout_s,
                     const c10::optional<Tensor>& err) {
  c10::cuda::CUDAGuard g(flag.device());
  edl::wait_flag_async(flag.data_ptr(), opt_ptr<void>(seq), (uint32_t)seq_imm, timeout_s, opt_ptr<void>(err),
                       cur_stream());
}

}  // namespace

void register_gemm_bindings(pybind11::module_& m);  // gemm_bindings.cpp
void register_jpeg_bindings(pybind11::module_& m);  // jpeg_decode.cpp
void register_vmm_bindings(pybind11::module_& m);   // vmm.cpp

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "edl_b200 sm_100a kernels";
  m.def("bn_set_stream_kernels", &edl::bn_set_stream_kernels);
  m.def("set_pdl", &edl::set_pdl, "programmatic dependent launch for the hot kernels (EDL_PDL=1)");
  m.def("pdl_enabled", &edl::pdl_enabled);
  m.def("set_smem_carveout_policy", &edl::set_smem_carveout_policy);
  m.def("bn_fused_fits", &bn_fused_fits);
  m.def("bn_fwd_fused", &bn_fwd_fused);
  m.def("bn_bwd_fused", &bn_bwd_fused);
  m.def("bn_stats", &bn_stats);
  m.def("bn_apply", &bn_apply);
  m.def("scale_shift_act", &scale_shift_act);
  m.def("bn_bwd_reduce", &bn_bwd_reduce);
  m.def("bn_bwd_apply", &bn_bwd_apply);
  m.def("sgd_momentum", &sgd_momentum);
  m.def("adam_step", &adam_step);
  m.def("lars_step", &lars_step);
  m.def("lamb_step", &lamb_step);
  m.def("soft_ce_fwd", &soft_ce_fwd);
  m.def("soft_ce_bwd", &soft_ce_bwd);
  m.def("topk_acc", &topk_acc);
  m.def("maxpool3x3s2_fwd", &maxpool3x3s2_fwd);
  m.def("maxpool3x3s2_bwd", &maxpool3x3s2_bwd);
  m.def("avgpool2x2_fwd", &avgpool2x2_fwd);
  m.def("avgpool2x2_bwd", &avgpool2x2_bwd);
  m.def("dilate2", &dilate2);
  m.def("gap_fwd", &gap_fwd);
  m.def("gap_bwd", &gap_bwd);
  m.def("allreduce_oneshot", &allreduce_oneshot);
  m.def("allreduce_twoshot", &allreduce_twoshot);
  m.def("allreduce_sgd", &allreduce_sgd);
  m.def("grad_sqnorm", &grad_sqnorm);
  m.def("clip_scale", &clip_scale);
  m.def("comm_broadcast", &comm_broadcast);
  m.def("comm_allgather_scalars", &comm_allgather_scalars);
  m.def("comm_sig_words", &edl::comm_sig_words);
  m.def("comm_error_word_offset", &edl::comm_error_word_offset);
  m.def("rope", &rope);
  m.def("embedding_bag_fwd", &embedding_bag_fwd);
  m.def("stem_conv3x3s2", &stem_conv3x3s2);
  m.def("stem_wgrad", &stem_wgrad);
  m.def("stem7_im2col", &stem7_im2col);
  m.def("pair_weight_expand", &pair_weight_expand);
  m.def("pair_weight_fold", &pair_weight_fold);
  m.def("fold_pair_stats", &fold_pair_stats);
  m.def("embedding_bag_bwd", &embedding_bag_bwd);
  m.def("normalize_u8", &normalize_u8);
  m.def("peer_ship", &peer_ship);
  m.def("logit_ship", &logit_ship);
  m.def("soft_ce_recv", &soft_ce_recv);
  m.def("slot_ack", &slot_ack);
  m.def("wait_flag_async", &wait_flag_async);
  register_gemm_bindings(m);
  register_jpeg_bindings(m);
  register_vmm_bindings(m);
}
