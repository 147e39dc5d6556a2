// Fused optimizer step over a flat fp32 parameter arena (one launch for the whole model):
// L2 term folded into the gradient, moments, update, and the bf16 shadow copy the conv kernels
// read next step -- all in one pass over HBM.
//   tf.train.AdamOptimizer(lr, beta1=0.9, beta2=0.99) / ApplyAdam       <- /root/reference/core/solver.py:204-207
//   tf.train.MomentumOptimizer(lr, 0.9[, use_nesterov]) / ApplyMomentum <- /root/reference/core/solver.py:208-210
//   tf.contrib.opt.AdamWOptimizer(weight_decay, lr, 0.9, 0.99)          <- /root/reference/core/solver.py:211-216
//   (--adam_beta1/2, --adam_eps, --mm_mm, --mm_nesterov replace the defaults, solver.py:86-97)
//   slim.l2_regularizer(rate): loss += rate*sum(w^2)/2, grad += rate*w   <- /root/reference/NetworksV2/base.py:128-135
#include <cuda_bf16.h>
#include "reduce.cuh"

using namespace bsl;

namespace {

__global__ void adam_kernel(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, __nv_bfloat16* __restrict__ shadow, size_t n, float lr_t,
                            float beta1, float beta2, float eps, float l2, float gscale, float decay,
                            double* __restrict__ sq_part) {
  bsl::pdl_wait();
  __shared__ double sm[32];
  double sq = 0.0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float wi = w[i];
    sq += (double)wi * (double)wi;
    const float gi = fmaf(l2, wi, g[i] * gscale);
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    const float wd = decay != 0.f ? wi - decay * wi : wi;   // AdamW: decay first, Adam update on the decayed value
    const float wn = wd - lr_t * mi / (sqrtf(vi) + eps);
    m[i] = mi;
    v[i] = vi;
    w[i] = wn;
    if (shadow) shadow[i] = __float2bfloat16_rn(wn);
  }
  if (sq_part) {
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int k = 0; k < (int)(blockDim.x >> 5); ++k) s += sm[k];
      sq_part[blockIdx.x] = s;
    }
  }
}

__global__ void momentum_kernel(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ acc,
                                __nv_bfloat16* __restrict__ shadow, size_t n, float lr, float mom, int nesterov,
                                float l2, float gscale, double* __restrict__ sq_part) {
  bsl::pdl_wait();
  __shared__ double sm[32];
  double sq = 0.0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float wi = w[i];
    sq += (double)wi * (double)wi;
    const float gi = fmaf(l2, wi, g[i] * gscale);
    const float a = mom * acc[i] + gi;
    const float wn = nesterov ? wi - (gi * lr + a * mom * lr) : wi - lr * a;
    acc[i] = a;
    w[i] = wn;
    if (shadow) shadow[i] = __float2bfloat16_rn(wn);
  }
  if (sq_part) {
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int k = 0; k < (int)(blockDim.x >> 5); ++k) s += sm[k];
      sq_part[blockIdx.x] = s;
    }
  }
}

__global__ void sumsq_final_kernel(const double* __restrict__ part, int blocks, double* __restrict__ out) {
  bsl::pdl_wait();
  if (blockIdx.x || threadIdx.x >= 32) return;   // one warp: lane i adds partials i, i + 32, ..., then a fixed xor tree
  double s = 0.0;
  for (int b = threadIdx.x; b < blocks; b += 32) s += part[b];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (threadIdx.x == 0) *out = s;
}

int opt_blocks(bsl_ctx* ctx, size_t n) {
  size_t b = (n + 255) / 256;
  const size_t cap = 8 * (size_t)ctx->sm_count;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

extern "C" {

int bsl_adam_step(bsl_ctx* ctx, const bsl_adam_desc* d, float* w, const float* g, float* m, float* v,
                  void* w_bf16, size_t n, double* sumsq_out, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!d || !w || !g || !m || !v) return bsl_fail(ctx, BSL_EINVAL, "adam_step: null argument");
  if (d->step < 1) return bsl_fail(ctx, BSL_EINVAL, "adam_step: step must be >= 1 (TF global_step + 1)");
  if (n == 0) return BSL_OK;
  const double lr_t = (double)d->lr * sqrt(1.0 - pow((double)d->beta2, d->step)) / (1.0 - pow((double)d->beta1, d->step));
  const int blocks = opt_blocks(ctx, n);
  double* part = nullptr;
  if (sumsq_out) {
    float* base = nullptr;
    int rc = bsl_scratch(ctx, (size_t)blocks * sizeof(double), &base, as_stream(stream));
    if (rc) return rc;
    part = reinterpret_cast<double*>(base);
  }
  cudaStream_t s = as_stream(stream);
  bsl_launch(adam_kernel, dim3(blocks), dim3(256), 0, s, w, g, m, v, reinterpret_cast<__nv_bfloat16*>(w_bf16), n, (float)lr_t, d->beta1,
                                     d->beta2, d->eps, d->l2_rate, d->grad_scale, d->decoupled_decay, part);
  BSL_LAUNCH_CHECK(ctx, "adam_kernel");
  if (sumsq_out) {
    bsl_launch(sumsq_final_kernel, dim3(1), dim3(32), 0, s, part, blocks, sumsq_out);
    BSL_LAUNCH_CHECK(ctx, "sumsq_final_kernel");
  }
  return BSL_OK;
}

int bsl_momentum_step(bsl_ctx* ctx, float lr, float momentum, int use_nesterov, float l2_rate, float grad_scale,
                      float* w, const float* g, float* acc, void* w_bf16, size_t n, double* sumsq_out, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!w || !g || !acc) return bsl_fail(ctx, BSL_EINVAL, "momentum_step: null argument");
  if (n == 0) return BSL_OK;
  const int blocks = opt_blocks(ctx, n);
  double* part = nullptr;
  if (sumsq_out) {
    float* base = nullptr;
    int rc = bsl_scratch(ctx, (size_t)blocks * sizeof(double), &base, as_stream(stream));
    if (rc) return rc;
    part = reinterpret_cast<double*>(base);
  }
  cudaStream_t s = as_stream(stream);
  bsl_launch(momentum_kernel, dim3(blocks), dim3(256), 0, s, w, g, acc, reinterpret_cast<__nv_bfloat16*>(w_bf16), n, lr, momentum,
                                         use_nesterov, l2_rate, grad_scale, part);
  BSL_LAUNCH_CHECK(ctx, "momentum_kernel");
  if (sumsq_out) {
    bsl_launch(sumsq_final_kernel, dim3(1), dim3(32), 0, s, part, blocks, sumsq_out);
    BSL_LAUNCH_CHECK(ctx, "sumsq_final_kernel");
  }
  return BSL_OK;
}

}  // extern "C"
