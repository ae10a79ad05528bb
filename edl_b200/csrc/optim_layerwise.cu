// Layer-wise adaptive optimizers on the flat buffers: LARS (Paddle's LarsMomentum) and LAMB.
//
// Both rules scale each parameter tensor's update by a ratio of per-tensor L2 norms, so the flat layout
// (one buffer per dtype, no per-tensor launches) needs a segmented reduction.  It is done in two passes
// over a host-built chunk table; every chunk lies inside ONE tensor ("entry") and has at most a few K
// elements, so one CTA owns one chunk:
//
//   pass 1  CTA c reduces its chunk to partial sums of squares  partials[c] = (sum w^2, sum x^2)
//           (x = g for LARS; LAMB first updates m / v and takes x = r, the unscaled update)
//   pass 2  CTA c sums the partials of its entry's chunks in chunk order, derives the entry's
//           local_lr (LARS) / trust ratio (LAMB) and applies the update to its chunk
//
// No atomics anywhere: every sum has a fixed shape (thread -> element map, warp shuffles, chunk order), so
// the result is bitwise identical from run to run, and applying the optimizer bucket by bucket (tables
// over sub-ranges of the buffer) gives the same bits as one whole-model pass.
//
// Chunk table: int64 [nchunks, 5] = (start, len, first chunk of the entry, chunk count of the entry,
// decay flag).  Entries start on 128-element boundaries (parallel/flat.py ALIGN_ELEMS), so chunks are
// 16-byte aligned for 8-wide vector loads; only the last chunk of an entry can end in a scalar tail.
// lr / grad_scale / found_inf / step are read from device memory: a captured graph replays with
// whatever set_lr() wrote last.
#include "common.cuh"
#include "kernels.h"

namespace edl {
namespace {

constexpr int kThreads = 256;
constexpr int kChunkCols = 5;

struct Chunk {
  int64_t start;
  int len, first, count;
  bool decay;
};

EDL_DEVICE Chunk load_chunk(const int64_t* __restrict__ table, int c) {
  const int64_t* t = table + (int64_t)c * kChunkCols;
  return Chunk{t[0], (int)t[1], (int)t[2], (int)t[3], t[4] != 0};
}

EDL_DEVICE void ld8(const float* p, float (&f)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p);
  const float4 b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
  f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

EDL_DEVICE void st8(float* p, const float (&f)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(f[4], f[5], f[6], f[7]);
}

template <typename GradT>
EDL_DEVICE void ld_grad8(const GradT* p, float (&f)[8]) {
  if constexpr (sizeof(GradT) == 2) unpack8(ld_stream(p), f);
  else ld8(reinterpret_cast<const float*>(p), f);
}

template <typename GradT>
EDL_DEVICE float ld_grad1(const GradT* p) {
  if constexpr (sizeof(GradT) == 2) return __bfloat162float(*p);
  else return *p;
}

// Sum of two per-thread values over the CTA in a fixed order; the result is returned to EVERY thread.
EDL_DEVICE float2 block_sum2(float a, float b) {
  __shared__ float2 sh[kThreads / 32];
  __syncthreads();                      // sh may still be read by a previous call
  a = warp_sum(a);
  b = warp_sum(b);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = make_float2(a, b);
  __syncthreads();
  float2 s = threadIdx.x < 32 && threadIdx.x < kThreads / 32 ? sh[threadIdx.x] : make_float2(0.f, 0.f);
  s.x = warp_sum(s.x);
  s.y = warp_sum(s.y);
  __shared__ float2 total;
  if (threadIdx.x == 0) total = s;
  __syncthreads();
  return total;
}

// The entry's squared norms: its chunks' partials summed in chunk order by every CTA of the entry alike.
EDL_DEVICE float2 entry_sqnorms(const float2* __restrict__ partials, const Chunk& ck) {
  float a = 0.f, b = 0.f;
  for (int i = threadIdx.x; i < ck.count; i += kThreads) {
    const float2 p = partials[ck.first + i];
    a += p.x;
    b += p.y;
  }
  return block_sum2(a, b);
}

struct LarsArgs {
  const float* lr;
  const float* grad_scale;  // nullptr: 1
  const int* found_inf;     // nullptr or flag: non-zero => the step is a no-op
  float momentum, coeff, wd, eps;
};

template <typename GradT>
__global__ void __launch_bounds__(kThreads)
lars_norms_kernel(const float* __restrict__ master, const GradT* __restrict__ grad,
                  const int64_t* __restrict__ table, float2* __restrict__ partials, LarsArgs a) {
  if (a.found_inf != nullptr && *a.found_inf != 0) return;
  const Chunk ck = load_chunk(table, blockIdx.x);
  const float gs = a.grad_scale ? *a.grad_scale : 1.f;
  const float* w = master + ck.start;
  const GradT* g = grad + ck.start;
  const int nvec = ck.len / 8;
  float sw = 0.f, sg = 0.f;
#pragma unroll 2
  for (int i = threadIdx.x; i < nvec; i += kThreads) {
    float wf[8], gf[8];
    ld8(w + i * 8, wf);
    ld_grad8(g + i * 8, gf);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float gk = gf[k] * gs;
      sw = fmaf(wf[k], wf[k], sw);
      sg = fmaf(gk, gk, sg);
    }
  }
  for (int i = nvec * 8 + threadIdx.x; i < ck.len; i += kThreads) {
    const float wk = w[i], gk = ld_grad1(g + i) * gs;
    sw = fmaf(wk, wk, sw);
    sg = fmaf(gk, gk, sg);
  }
  const float2 s = block_sum2(sw, sg);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

template <typename GradT>
__global__ void __launch_bounds__(kThreads)
lars_update_kernel(__nv_bfloat16* __restrict__ param_lp, float* __restrict__ master, float* __restrict__ mom,
                   const GradT* __restrict__ grad, const int64_t* __restrict__ table,
                   const float2* __restrict__ partials, LarsArgs a) {
  if (a.found_inf != nullptr && *a.found_inf != 0) return;
  const Chunk ck = load_chunk(table, blockIdx.x);
  const float2 sq = entry_sqnorms(partials, ck);
  const float lr = *a.lr;
  const float gs = a.grad_scale ? *a.grad_scale : 1.f;
  const float wd = ck.decay ? a.wd : 0.f;
  const float wn = sqrtf(sq.x), gn = sqrtf(sq.y);
  const float local_lr = (wd > 0.f && wn > 0.f && gn > 0.f) ? lr * a.coeff * wn / (gn + wd * wn + a.eps) : lr;
  float* w = master + ck.start;
  float* v = mom + ck.start;
  const GradT* g = grad + ck.start;
  __nv_bfloat16* lp = param_lp != nullptr ? param_lp + ck.start : nullptr;
  const int nvec = ck.len / 8;
  for (int i = threadIdx.x; i < nvec; i += kThreads) {
    float wf[8], vf[8], gf[8];
    ld_grad8(g + i * 8, gf);
    ld8(w + i * 8, wf);
    ld8(v + i * 8, vf);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      vf[k] = fmaf(a.momentum, vf[k], local_lr * fmaf(wd, wf[k], gf[k] * gs));
      wf[k] -= vf[k];
    }
    st8(w + i * 8, wf);
    st8(v + i * 8, vf);
    if (lp != nullptr) st_vec(lp + i * 8, pack8(wf));
  }
  for (int i = nvec * 8 + threadIdx.x; i < ck.len; i += kThreads) {
    float wk = w[i];
    const float vk = fmaf(a.momentum, v[i], local_lr * fmaf(wd, wk, ld_grad1(g + i) * gs));
    wk -= vk;
    w[i] = wk;
    v[i] = vk;
    if (lp != nullptr) lp[i] = __float2bfloat16(wk);
  }
}

struct LambArgs {
  const float* lr;
  const float* grad_scale;
  const int* found_inf;
  const float* step;  // applied steps BEFORE this one; this step is *step + 1
  float beta1, beta2, eps, wd;
};

struct LambCoef {
  float inv_bc1, inv_bc2;
};

EDL_DEVICE LambCoef lamb_coef(const LambArgs& a) {
  const float t = *a.step + 1.f;
  return LambCoef{1.f / (1.f - powf(a.beta1, t)), 1.f / (1.f - powf(a.beta2, t))};
}

// r = m_hat / (sqrt(v_hat) + eps) + wd * w: one function for both passes so they agree on every bit
EDL_DEVICE float lamb_r(float m, float v, float w, float wd, const LambCoef& c, float eps) {
  return fmaf(wd, w, (m * c.inv_bc1) / (sqrtf(v * c.inv_bc2) + eps));
}

template <typename GradT>
__global__ void __launch_bounds__(kThreads)
lamb_moments_kernel(const float* __restrict__ master, float* __restrict__ m, float* __restrict__ v,
                    const GradT* __restrict__ grad, const int64_t* __restrict__ table,
                    float2* __restrict__ partials, LambArgs a) {
  if (a.found_inf != nullptr && *a.found_inf != 0) return;
  const Chunk ck = load_chunk(table, blockIdx.x);
  const float gs = a.grad_scale ? *a.grad_scale : 1.f;
  const LambCoef c = lamb_coef(a);
  const float wd = ck.decay ? a.wd : 0.f;
  const float b1 = a.beta1, b2 = a.beta2, nb1 = 1.f - a.beta1, nb2 = 1.f - a.beta2;
  const float* w = master + ck.start;
  float* mp = m + ck.start;
  float* vp = v + ck.start;
  const GradT* g = grad + ck.start;
  const int nvec = ck.len / 8;
  float sw = 0.f, sr = 0.f;
  for (int i = threadIdx.x; i < nvec; i += kThreads) {
    float wf[8], mf[8], vf[8], gf[8];
    ld_grad8(g + i * 8, gf);
    ld8(w + i * 8, wf);
    ld8(mp + i * 8, mf);
    ld8(vp + i * 8, vf);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float gk = gf[k] * gs;
      mf[k] = fmaf(b1, mf[k], nb1 * gk);
      vf[k] = fmaf(b2, vf[k], nb2 * gk * gk);
      const float r = lamb_r(mf[k], vf[k], wf[k], wd, c, a.eps);
      sw = fmaf(wf[k], wf[k], sw);
      sr = fmaf(r, r, sr);
    }
    st8(mp + i * 8, mf);
    st8(vp + i * 8, vf);
  }
  for (int i = nvec * 8 + threadIdx.x; i < ck.len; i += kThreads) {
    const float gk = ld_grad1(g + i) * gs, wk = w[i];
    const float mk = fmaf(b1, mp[i], nb1 * gk);
    const float vk = fmaf(b2, vp[i], nb2 * gk * gk);
    const float r = lamb_r(mk, vk, wk, wd, c, a.eps);
    mp[i] = mk;
    vp[i] = vk;
    sw = fmaf(wk, wk, sw);
    sr = fmaf(r, r, sr);
  }
  const float2 s = block_sum2(sw, sr);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kThreads)
lamb_update_kernel(__nv_bfloat16* __restrict__ param_lp, float* __restrict__ master, const float* __restrict__ m,
                   const float* __restrict__ v, const int64_t* __restrict__ table,
                   const float2* __restrict__ partials, LambArgs a) {
  if (a.found_inf != nullptr && *a.found_inf != 0) return;
  const Chunk ck = load_chunk(table, blockIdx.x);
  const float2 sq = entry_sqnorms(partials, ck);
  const LambCoef c = lamb_coef(a);
  const float wd = ck.decay ? a.wd : 0.f;
  const float wn = sqrtf(sq.x), rn = sqrtf(sq.y);
  const float step = -*a.lr * ((wn > 0.f && rn > 0.f) ? wn / rn : 1.f);
  float* w = master + ck.start;
  const float* mp = m + ck.start;
  const float* vp = v + ck.start;
  __nv_bfloat16* lp = param_lp != nullptr ? param_lp + ck.start : nullptr;
  const int nvec = ck.len / 8;
  for (int i = threadIdx.x; i < nvec; i += kThreads) {
    float wf[8], mf[8], vf[8];
    ld8(w + i * 8, wf);
    ld8(mp + i * 8, mf);
    ld8(vp + i * 8, vf);
#pragma unroll
    for (int k = 0; k < 8; ++k) wf[k] = fmaf(step, lamb_r(mf[k], vf[k], wf[k], wd, c, a.eps), wf[k]);
    st8(w + i * 8, wf);
    if (lp != nullptr) st_vec(lp + i * 8, pack8(wf));
  }
  for (int i = nvec * 8 + threadIdx.x; i < ck.len; i += kThreads) {
    const float wk = fmaf(step, lamb_r(mp[i], vp[i], w[i], wd, c, a.eps), w[i]);
    w[i] = wk;
    if (lp != nullptr) lp[i] = __float2bfloat16(wk);
  }
}

}  // namespace

void lars_step(void* param_lp, float* master, float* mom, const void* grad, bool grad_is_bf16,
               const int64_t* chunks, int nchunks, float* partials, const float* lr, const float* grad_scale,
               const int* found_inf, float momentum, float lars_coeff, float wd, float eps, cudaStream_t stream) {
  if (nchunks <= 0) return;
  LarsArgs a{lr, grad_scale, found_inf, momentum, lars_coeff, wd, eps};
  auto* lp = reinterpret_cast<__nv_bfloat16*>(param_lp);
  auto* parts = reinterpret_cast<float2*>(partials);
  if (grad_is_bf16) {
    auto* g = reinterpret_cast<const __nv_bfloat16*>(grad);
    lars_norms_kernel<<<nchunks, kThreads, 0, stream>>>(master, g, chunks, parts, a);
    lars_update_kernel<<<nchunks, kThreads, 0, stream>>>(lp, master, mom, g, chunks, parts, a);
  } else {
    auto* g = reinterpret_cast<const float*>(grad);
    lars_norms_kernel<<<nchunks, kThreads, 0, stream>>>(master, g, chunks, parts, a);
    lars_update_kernel<<<nchunks, kThreads, 0, stream>>>(lp, master, mom, g, chunks, parts, a);
  }
}

void lamb_step(void* param_lp, float* master, float* m, float* v, const void* grad, bool grad_is_bf16,
               const int64_t* chunks, int nchunks, float* partials, const float* lr, const float* grad_scale,
               const int* found_inf, const float* step, float beta1, float beta2, float eps, float wd,
               cudaStream_t stream) {
  if (nchunks <= 0) return;
  LambArgs a{lr, grad_scale, found_inf, step, beta1, beta2, eps, wd};
  auto* parts = reinterpret_cast<float2*>(partials);
  if (grad_is_bf16)
    lamb_moments_kernel<<<nchunks, kThreads, 0, stream>>>(master, m, v, reinterpret_cast<const __nv_bfloat16*>(grad),
                                                          chunks, parts, a);
  else
    lamb_moments_kernel<<<nchunks, kThreads, 0, stream>>>(master, m, v, reinterpret_cast<const float*>(grad), chunks,
                                                          parts, a);
  lamb_update_kernel<<<nchunks, kThreads, 0, stream>>>(reinterpret_cast<__nv_bfloat16*>(param_lp), master, m, v,
                                                       chunks, parts, a);
}

}  // namespace edl
