// Host-side launcher declarations for the edl_b200 sm_100a kernels.
// Kernels live in torch-free .cu files; bindings.cpp adapts torch tensors to these entry points.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace edl {

// ---- bn.cu ----
void bn_stats(const void* x, float* sums, int64_t M, int C, cudaStream_t stream);
void bn_apply(const void* x, const void* res, void* y, const float* sums, const float* gamma,
              const float* beta, float* running_mean, float* running_var, float* saved_mean,
              float* saved_rstd, int64_t M, int C, float eps, float momentum, bool relu,
              cudaStream_t stream);
void scale_shift_act(const void* x, const void* res, void* y, const float* scale,
                     const float* shift, int64_t M, int C, bool relu, cudaStream_t stream);
// y == nullptr with relu: the ReLU mask is recomputed from x (no residual case)
void bn_bwd_reduce(const void* dy, const void* x, const void* y, const float* gamma,
                   const float* beta, const float* saved_mean, const float* saved_rstd,
                   float* dsums, int64_t M, int C, bool relu, cudaStream_t stream);
void bn_bwd_apply(const void* dy, const void* x, const void* y, const float* gamma,
                  const float* beta, const float* saved_mean, const float* saved_rstd,
                  const float* dsums, void* dx, void* dres, float* dgamma, float* dbeta, int64_t M,
                  int C, bool relu, bool accumulate, cudaStream_t stream);

// ---- bn_stream.cu (cp.async.bulk + mbarrier streaming variants; used when supported) ----
bool bn_stream_supported(int64_t M, int C);
void bn_stats_stream(const void* x, float* sums, int64_t M, int C, cudaStream_t s);
void bn_apply_stream(const void* x, const void* res, void* y, const float* sums, const float* gamma,
                     const float* beta, float* running_mean, float* running_var, float* saved_mean,
                     float* saved_rstd, int64_t M, int C, float eps, float momentum, bool relu,
                     cudaStream_t s);
void bn_bwd_reduce_stream(const void* dy, const void* x, const void* y, const float* gamma,
                          const float* beta, const float* saved_mean, const float* saved_rstd,
                          float* dsums, int64_t M, int C, bool relu, cudaStream_t s);
void bn_bwd_apply_stream(const void* dy, const void* x, const void* y, const float* gamma,
                         const float* beta, const float* saved_mean, const float* saved_rstd,
                         const float* dsums, void* dx, void* dres, float* dgamma, float* dbeta,
                         int64_t M, int C, bool relu, bool accumulate, cudaStream_t s);
void bn_set_stream_kernels(bool enabled);

// ---- bn_fused.cu (SM-resident single-launch BN forward / backward with a grid barrier) ----
bool bn_fused_fits(int64_t M, int C, int num_operands);
const char* bn_fwd_fused(const void* x, const void* res, void* y, float* sums, const float* gamma,
                         const float* beta, float* running_mean, float* running_var,
                         float* saved_mean, float* saved_rstd, int64_t M, int C, float eps,
                         float momentum, bool relu, unsigned int* sync_counter, cudaStream_t s);
const char* bn_bwd_fused(const void* dy, const void* x, const void* y, const float* gamma,
                         const float* beta, const float* saved_mean, const float* saved_rstd,
                         float* dsums, void* dx, void* dres, float* dgamma, float* dbeta, int64_t M,
                         int C, bool relu, bool accumulate, unsigned int* sync_counter,
                         cudaStream_t s);  // runtime switch (A/B measurements); default on

// ---- runtime policy (bn.cu): keep every SM in the max-shared-memory carveout so that kernels with
// large dynamic smem (TMA rings, GEMM stages) never force an L1/smem re-partition between launches ----
void set_smem_carveout_policy(bool prefer_max_shared);
bool smem_carveout_policy();
void apply_carveout(const void* kernel);   // call after cudaFuncSetAttribute(MaxDynamicSharedMemorySize)

// ---- optim.cu ----
void sgd_momentum(void* param_lp, float* master, float* mom, const void* grad, bool grad_is_bf16,
                  const float* wd_mask, int64_t n, const float* lr, const float* grad_scale,
                  const int* found_inf, float momentum, float wd, bool nesterov,
                  cudaStream_t stream);
void adam_step(void* param_lp, float* master, float* m, float* v, const void* grad,
               bool grad_is_bf16, int64_t n, const float* lr, const float* grad_scale,
               const int* found_inf, const float* step, float beta1, float beta2, float eps,
               float wd, bool decoupled, cudaStream_t stream);

// ---- optim_layerwise.cu ----
// LARS / LAMB over a chunk table (int64 [nchunks, 5]: start, len, first chunk of the entry, chunk count of the
// entry, decay flag); partials: fp32 [nchunks, 2] scratch.  Two launches each (norm pass, update pass).
void lars_step(void* param_lp, float* master, float* mom, const void* grad, bool grad_is_bf16,
               const int64_t* chunks, int nchunks, float* partials, const float* lr, const float* grad_scale,
               const int* found_inf, float momentum, float lars_coeff, float wd, float eps, cudaStream_t stream);
void lamb_step(void* param_lp, float* master, float* m, float* v, const void* grad, bool grad_is_bf16,
               const int64_t* chunks, int nchunks, float* partials, const float* lr, const float* grad_scale,
               const int* found_inf, const float* step, float beta1, float beta2, float eps, float wd,
               cudaStream_t stream);

// sum(g^2) of a flat gradient buffer into *out (+=), and the global-norm clip factor
//   grad_scale = min(1, max_norm / (sqrt(sum of parts) + 1e-6))   (parts: one squared-norm partial per rank)
void grad_sqnorm(const void* grad, bool grad_is_bf16, int64_t n, float* out, cudaStream_t stream);
void clip_scale(const float* parts, int nparts, int stride, float max_norm, float* grad_scale, float* norm_out,
                cudaStream_t stream);

// ---- loss.cu ----
void soft_ce_fwd(const void* logits, bool logits_bf16, const void* target, bool target_bf16,
                 const int64_t* labels, float* loss_out, float* row_stats, int N, int C, int mode,
                 float s_temp, float t_temp, float label_smooth, bool kl, float loss_scale,
                 cudaStream_t stream);
void soft_ce_bwd(const void* logits, bool logits_bf16, const void* target, bool target_bf16,
                 const int64_t* labels, const float* row_stats, const float* grad_out,
                 void* dlogits, int N, int C, int mode, float s_temp, float t_temp,
                 float label_smooth, float loss_scale, cudaStream_t stream);
void topk_acc(const void* logits, bool logits_bf16, const int64_t* labels, float* counts, int N,
              int C, cudaStream_t stream);

// ---- pool.cu ----
void maxpool3x3s2_fwd(const void* x, void* y, uint8_t* idx, int N, int H, int W, int C,
                      cudaStream_t s);
void maxpool3x3s2_bwd(const void* dy, const uint8_t* idx, void* dx, int N, int H, int W, int C,
                      cudaStream_t s);
void avgpool2x2_fwd(const void* x, void* y, int N, int H, int W, int C, cudaStream_t s);
void avgpool2x2_bwd(const void* dy, void* dx, int N, int H, int W, int C, cudaStream_t s);
void dilate2(const void* x, void* y, int N, int H, int W, int C, cudaStream_t s);   // zero-insertion by 2 (NHWC bf16)
void gap_fwd(const void* x, void* y, int N, int HW, int C, cudaStream_t s);
void gap_bwd(const void* dy, void* dx, int N, int HW, int C, cudaStream_t s);

// ---- allreduce.cu ----
struct CommHandles {
  void* data[16];
  void* sig[16];
  void* mc_data;
  int rank;
  int world;
  unsigned long long timeout_ns;
};
int comm_sig_words();
int comm_max_world();
int comm_error_word_offset();
void allreduce_oneshot(const CommHandles& h, void* out, bool is_bf16, int64_t n, float scale,
                       int* found_inf, float* sqnorm, int nblocks, cudaStream_t stream);
void allreduce_twoshot(const CommHandles& h, bool is_bf16, int64_t n, float scale, int* found_inf,
                       float* sqnorm, bool multimem, int nblocks, cudaStream_t stream);
// fused reduce-scatter -> SGD-momentum -> parameter all-gather of one bf16 bucket (allreduce.cu)
void allreduce_sgd(const CommHandles& h, void* const* param_ptrs, void* mc_param, float* master, float* mom,
                   const float* wd_mask, int64_t n, float scale, int* found_inf_out, float* sqnorm,
                   const float* lr, const int* skip_flag, float momentum, float wd, bool nesterov, bool multimem,
                   int nblocks, cudaStream_t stream);
void comm_broadcast(const CommHandles& h, int root, int64_t nbytes, int nblocks,
                    cudaStream_t stream);
void comm_allgather_scalars(const CommHandles& h, const float* in, float* out, int count,
                            cudaStream_t stream);

// ---- misc.cu ----
void rope(const void* x, const float* cosv, const float* sinv, void* y, int64_t T, int H, int D,
          bool inverse, cudaStream_t s);
// pixel-pair form of the 32-channel 3x3 stem convolutions (misc.cu): W [cout,3,3,32] <-> W2 [2*cout,3,3,64]
void pair_weight_expand(const void* w, void* w2, int cout, cudaStream_t s);
void pair_weight_fold(const void* dw2, void* dw, int cout, bool accumulate, cudaStream_t s);
void fold_pair_stats(const float* s2, float* stats, int cout, cudaStream_t s);
// ---- stem.cu: first stem convolution (3 -> 32, 3x3 / stride 2 / pad 1, NHWC bf16) + BN statistics of its output ----
void stem_conv3x3s2(const void* x, const void* w, void* y, float* stats, int N, int H, int W, cudaStream_t s);
// its weight gradient: dw KRSC [32,3,3,3] bf16 (+)= ; ws: >= 864 zero floats (left zero), counter: one zero int (left zero)
// A [N * Ho * Wo, 160] bf16 = im2col of the 7x7 / stride 2 / pad 3 convolution of x [N, H, W, 3] ((r, s, c) order, zero-padded)
const char* stem7_im2col(const void* x, void* a, int N, int H, int W, cudaStream_t s);
const char* stem_wgrad(const void* x, const void* dy, float* ws, int* counter, void* dw, bool accumulate, int N, int H,
                       int W, cudaStream_t s);

void embedding_bag_fwd(const void* table, bool bf16, const int64_t* ids, void* out, int64_t B, int L,
                       int D, cudaStream_t s);
void embedding_bag_bwd(const void* dout, bool bf16, const int64_t* ids, float* dtable, int64_t B, int L,
                       int D, cudaStream_t s);
void normalize_u8(const uint8_t* x, void* y, int64_t N, int H, int W, const float* mean,
                  const float* stdv, const uint8_t* flip, cudaStream_t s);

// ---- augment.cu: random-resized crop + flip + normalise from decoded uint8 RGB images of different sizes ----
struct AugmentItem {   // one per output image; 32 bytes = 8 x int32 (the Python side fills an int32 [N, 8] tensor)
  int64_t offset;      // byte offset of the decoded image (interleaved RGB) inside the pool buffer
  int pitch;           // bytes per source row
  int y, x, ch, cw;    // crop box inside the source image
  int flip;            // mirror horizontally
};
void crop_resize_normalize(const uint8_t* pool, const AugmentItem* items, void* y, int N, int S, const float* mean,
                           const float* stdv, cudaStream_t s);

// ---- logit_ship.cu (teacher -> student over NVSwitch peer memory, fused with the loss) ----
void peer_ship(const void* src, void* dst_peer, int64_t nbytes, void* flag_peer, const void* seq_ptr,
               uint32_t seq_imm, void* done_counter, cudaStream_t s);
void logit_ship(const void* logits, void* slot_peer, float* stats_peer, int B, int C, float temperature,
                void* flag_peer, const void* seq_ptr, uint32_t seq_imm, void* done_counter,
                cudaStream_t s);
void soft_ce_recv(const void* logits, bool logits_bf16, const void* slot, const float* slot_stats,
                  const void* flag, const void* seq_ptr, uint32_t seq_imm, float* loss_out,
                  float* row_stats, int B, int C, float s_temp, float t_temp, bool kl, float loss_scale,
                  double timeout_s, void* err, cudaStream_t s);
void slot_ack(void* ack_peer, const void* seq_ptr, uint32_t seq_imm, cudaStream_t s);
void wait_flag_async(const void* flag, const void* seq_ptr, uint32_t seq_imm, double timeout_s, void* err,
                     cudaStream_t s);

}  // namespace edl
