// Losses, probabilities, threshold masks and integer Dice counts (all HBM-bound, one pixel per
// thread, warp-shuffle + fixed-order second-level reductions; counts are exact integers).
//   _compute_weights                      <- /root/reference/loss_metrics.py:115-165
//   weighted_sparse_softmax_cross_entropy <- /root/reference/loss_metrics.py:172-177
//   sparse_dice_loss                      <- /root/reference/loss_metrics.py:180-226
//   softmax + (p > 0.5) uint8 masks       <- /root/reference/NetworksV2/UNet.py:107-117
//   metric_dice/voe/vd I, L, R sums       <- /root/reference/loss_metrics.py:261-339
#include <cstdint>
#include "reduce.cuh"

using namespace bsl;

namespace {

constexpr int MAXC = 4;

__device__ __forceinline__ double block_sum(double v, double* sm) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) sm[warp] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sm[w];
  return s;  // valid in thread 0
}

// counts[n][c] = #pixels of image n with label c (labels outside [0, classes) are ignored)
__global__ void label_counts_kernel(const int* __restrict__ labels, int hw, int classes, int* __restrict__ counts) {
  bsl::pdl_wait();
  __shared__ int sc[MAXC];
  if (threadIdx.x < MAXC) sc[threadIdx.x] = 0;
  __syncthreads();
  const int img = blockIdx.y;
  int loc[MAXC] = {0, 0, 0, 0};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += gridDim.x * blockDim.x) {
    const int l = labels[(long long)img * hw + i];
#pragma unroll
    for (int c = 0; c < MAXC; ++c) loc[c] += (l == c);
  }
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    int v = loc[c];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&sc[c], v);
  }
  __syncthreads();
  if (threadIdx.x < classes && sc[threadIdx.x]) atomicAdd(&counts[img * classes + threadIdx.x], sc[threadIdx.x]);
}

// Per-image class weights after the reference's per-image renormalisation, and the number of
// pixels with non-zero weight (denominator of SUM_BY_NONZERO_WEIGHTS). One thread; n*classes is tiny.
// One warp: lane i takes images i, i + 32, ...; the count of weighted pixels is a sum of integers, exact in any order.
__global__ void weight_table_kernel(bsl_loss_desc d, const int* __restrict__ counts, float* __restrict__ wtab,
                                    double* __restrict__ nz_out) {
  bsl::pdl_wait();
  if (blockIdx.x || threadIdx.x >= 32) return;
  double nz = 0.0;
  for (int img = threadIdx.x; img < d.n; img += 32) {
    float w[MAXC];
    if (d.weight_type == 0) {
      for (int c = 0; c < d.classes; ++c) w[c] = 1.f;  // constant 1.0, no renormalisation (:123-124)
    } else {
      if (d.weight_type == 1) {
        for (int c = 0; c < d.classes; ++c) w[c] = d.numeric_w[c];
      } else {
        float prop[MAXC], s = 0.f;
        for (int c = 0; c < d.classes; ++c) {
          float num = (float)counts[img * d.classes + c];
          if (d.proportion_decay > 0.f) num += d.proportion_decay;
          prop[c] = 1.f / num;
          s += prop[c];
        }
        for (int c = 0; c < d.classes; ++c) w[c] = prop[c] / s;
      }
      double tot = 0.0;
      for (int c = 0; c < d.classes; ++c) tot += (double)w[c] * counts[img * d.classes + c];
      for (int c = 0; c < d.classes; ++c) w[c] = (float)((double)w[c] / tot * (double)d.hw);
    }
    for (int c = 0; c < d.classes; ++c) {
      wtab[img * d.classes + c] = w[c];
      if (w[c] != 0.f) nz += counts[img * d.classes + c];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nz += __shfl_xor_sync(0xffffffffu, nz, o);
  if (threadIdx.x == 0) *nz_out = nz;
}

template <int C>
__device__ __forceinline__ void softmax_c(const float* __restrict__ lg, float (&p)[C], float& lse_minus_max,
                                          float& mx) {
  mx = lg[0];
#pragma unroll
  for (int c = 1; c < C; ++c) mx = fmaxf(mx, lg[c]);
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    p[c] = expf(lg[c] - mx);
    s += p[c];
  }
  const float inv = 1.f / s;
#pragma unroll
  for (int c = 0; c < C; ++c) p[c] *= inv;
  lse_minus_max = logf(s);
}

// One pixel of the weighted cross entropy: returns w * ce and writes the C gradient entries to g.
template <int C>
__device__ __forceinline__ float wxent_pixel(const float* lg, int l, const float* __restrict__ wrow, float loss_scale,
                                             float inv_nz, float* g) {
  float pr[C], lse, mx;
  softmax_c<C>(lg, pr, lse, mx);
  const bool ok = l >= 0 && l < C;
  const float w = ok ? wrow[l] : 0.f;
  float ce = 0.f;
#pragma unroll
  for (int c = 0; c < C; ++c) ce = (c == l) ? -(lg[c] - mx - lse) : ce;
#pragma unroll
  for (int c = 0; c < C; ++c) g[c] = loss_scale * w * (pr[c] - (c == l ? 1.f : 0.f)) * inv_nz;
  return w * ce;
}

// VEC: a thread takes 4 consecutive pixels of one image (hw % 4 == 0): C 16-byte loads of logits, one of labels,
// C 16-byte stores of the gradient, one image-index division per quad. Otherwise one pixel per thread.
template <int C, bool VEC>
__global__ void wxent_kernel(const float* __restrict__ logits, const int* __restrict__ labels, int hw,
                             long long pixels, const float* __restrict__ wtab, const double* __restrict__ nz_p,
                             float loss_scale, float* __restrict__ dlogits, double* __restrict__ part) {
  bsl::pdl_wait();
  __shared__ double sm[32];
  const double nz = *nz_p;
  const float inv_nz = nz > 0.0 ? (float)(1.0 / nz) : 0.f;
  double acc = 0.0;
  const long long t0 = blockIdx.x * (long long)blockDim.x + threadIdx.x, nt = (long long)gridDim.x * blockDim.x;
  if (VEC) {
    const bool small = pixels <= 0xffffffffLL;
    for (long long q = t0; q < (pixels >> 2); q += nt) {
      float lg[4 * C], g[4 * C];
      const float4* src = reinterpret_cast<const float4*>(logits + q * 4 * C);
#pragma unroll
      for (int i = 0; i < C; ++i) {
        const float4 t = src[i];
        lg[4 * i] = t.x, lg[4 * i + 1] = t.y, lg[4 * i + 2] = t.z, lg[4 * i + 3] = t.w;
      }
      const int4 lb = *reinterpret_cast<const int4*>(labels + q * 4);
      const int img = small ? (int)((unsigned)(q << 2) / (unsigned)hw) : (int)((q << 2) / hw);
      const float* wrow = wtab + img * C;
      acc += (double)wxent_pixel<C>(lg, lb.x, wrow, loss_scale, inv_nz, g);
      acc += (double)wxent_pixel<C>(lg + C, lb.y, wrow, loss_scale, inv_nz, g + C);
      acc += (double)wxent_pixel<C>(lg + 2 * C, lb.z, wrow, loss_scale, inv_nz, g + 2 * C);
      acc += (double)wxent_pixel<C>(lg + 3 * C, lb.w, wrow, loss_scale, inv_nz, g + 3 * C);
      if (dlogits) {
        float4* dst = reinterpret_cast<float4*>(dlogits + q * 4 * C);
#pragma unroll
        for (int i = 0; i < C; ++i) dst[i] = make_float4(g[4 * i], g[4 * i + 1], g[4 * i + 2], g[4 * i + 3]);
      }
    }
  } else {
    for (long long p = t0; p < pixels; p += nt) {
      float lg[C], g[C];
#pragma unroll
      for (int c = 0; c < C; ++c) lg[c] = logits[p * C + c];
      acc += (double)wxent_pixel<C>(lg, labels[p], wtab + (int)(p / hw) * C, loss_scale, inv_nz, g);
      if (dlogits) {
#pragma unroll
        for (int c = 0; c < C; ++c) dlogits[p * C + c] = g[c];
      }
    }
  }
  const double s = block_sum(acc, sm);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}

// One warp: lane i adds partials i, i + 32, ... in order, then a fixed xor tree over the lanes.
__global__ void wxent_final_kernel(const double* __restrict__ part, int blocks, const double* __restrict__ nz_p,
                                   float* __restrict__ loss) {
  bsl::pdl_wait();
  if (blockIdx.x || threadIdx.x >= 32) return;
  double s = 0.0;
  for (int b = threadIdx.x; b < blocks; b += 32) s += part[b];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const double nz = *nz_p;
  if (threadIdx.x == 0) *loss = nz > 0.0 ? (float)(s / nz) : 0.f;
}

template <int C>
__global__ void softmax_threshold_kernel(const float* __restrict__ logits, const int* __restrict__ labels, int hw,
                                         long long pixels, float* __restrict__ prob, uint8_t* __restrict__ masks,
                                         uint8_t* __restrict__ argmax, unsigned int* __restrict__ ilr) {
  bsl::pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long p0 = blockIdx.x * (long long)blockDim.x; p0 < pixels; p0 += stride) {
    const long long p = p0 + threadIdx.x;
    const bool live = p < pixels;
    float lg[C], pr[C], lse, mx;
#pragma unroll
    for (int c = 0; c < C; ++c) lg[c] = live ? logits[p * C + c] : 0.f;
    softmax_c<C>(lg, pr, lse, mx);
    const int l = (live && labels) ? labels[p] : -1;
    const int img = live ? (int)(p / hw) : -1;
    if (live) {
      if (prob) {
#pragma unroll
        for (int c = 0; c < C; ++c) prob[p * C + c] = pr[c];
      }
      if (argmax) {  // np.argmax: first maximum
        int best = 0;
#pragma unroll
        for (int c = 1; c < C; ++c) best = pr[c] > pr[best] ? c : best;
        argmax[p] = (uint8_t)best;
      }
    }
    const int img0 = __shfl_sync(0xffffffffu, img, 0);
    const bool uniform = __all_sync(0xffffffffu, img == img0);
#pragma unroll
    for (int c = 1; c < C; ++c) {
      const bool m = live && pr[c] > 0.5f;
      if (live && masks) masks[(long long)(c - 1) * pixels + p] = m ? 1 : 0;
      if (ilr) {
        const bool lab = (l == c);
        if (uniform) {
          const unsigned bi = __ballot_sync(0xffffffffu, m && lab);
          const unsigned bl = __ballot_sync(0xffffffffu, m);
          const unsigned br = __ballot_sync(0xffffffffu, lab);
          if ((threadIdx.x & 31) == 0 && img0 >= 0) {
            unsigned int* o = ilr + ((long long)img0 * (C - 1) + (c - 1)) * 3;
            if (bi) atomicAdd(o + 0, __popc(bi));
            if (bl) atomicAdd(o + 1, __popc(bl));
            if (br) atomicAdd(o + 2, __popc(br));
          }
        } else if (live) {
          unsigned int* o = ilr + ((long long)img * (C - 1) + (c - 1)) * 3;
          if (m && lab) atomicAdd(o + 0, 1u);
          if (m) atomicAdd(o + 1, 1u);
          if (lab) atomicAdd(o + 2, 1u);
        }
      }
    }
  }
}

// Dice pass 1: per image, I = sum_{c>=1} onehot*p, U = sum_{c>=1} (onehot + p). grid = (blocks, n).
template <int C>
__global__ void dice_reduce_kernel(const float* __restrict__ logits, const int* __restrict__ labels, int hw,
                                   double* __restrict__ part) {
  bsl::pdl_wait();
  __shared__ double sm[32];
  const int img = blockIdx.y;
  double ai = 0.0, au = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += gridDim.x * blockDim.x) {
    const long long p = (long long)img * hw + i;
    float lg[C], pr[C], lse, mx;
#pragma unroll
    for (int c = 0; c < C; ++c) lg[c] = logits[p * C + c];
    softmax_c<C>(lg, pr, lse, mx);
    const int l = labels[p];
#pragma unroll
    for (int c = 1; c < C; ++c) {
      const float oh = (l == c) ? 1.f : 0.f;
      ai += (double)(oh * pr[c]);
      au += (double)(oh + pr[c]);
    }
  }
  const double si = block_sum(ai, sm);
  const double su = block_sum(au, sm);
  if (threadIdx.x == 0) {
    part[((long long)img * gridDim.x + blockIdx.x) * 2 + 0] = si;
    part[((long long)img * gridDim.x + blockIdx.x) * 2 + 1] = su;
  }
}

// One warp per image sums that image's per-block partials (lane-strided, then a fixed shuffle tree: deterministic);
// thread 0 then averages the per-image terms in image order. (A single thread walking n x blocks dependent fp64 loads
// took 0.24 ms at batch 32 -- profiles/r02_ncu_launches_cfg3.txt.)
__global__ void dice_final_kernel(const double* __restrict__ part, int blocks, int n, float eps,
                                  double* __restrict__ iu, float* __restrict__ loss) {
  bsl::pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int img = warp; img < n; img += nwarps) {
    double si = 0.0, su = 0.0;
    for (int b = lane; b < blocks; b += 32) {
      si += part[((long long)img * blocks + b) * 2];
      su += part[((long long)img * blocks + b) * 2 + 1];
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      si += __shfl_down_sync(0xffffffffu, si, o);
      su += __shfl_down_sync(0xffffffffu, su, o);
    }
    if (lane == 0) {
      iu[img * 2] = si;
      iu[img * 2 + 1] = su;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double mean = 0.0;
    for (int img = 0; img < n; ++img) mean += 2.0 * iu[img * 2] / (iu[img * 2 + 1] + (double)eps);
    *loss = (float)(1.0 - mean / n);
  }
}

template <int C>
__global__ void dice_bwd_kernel(const float* __restrict__ logits, const int* __restrict__ labels, int hw,
                                long long pixels, int n, float eps, const double* __restrict__ iu, float loss_scale,
                                int accumulate, float* __restrict__ dlogits) {
  bsl::pdl_wait();
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < pixels;
       p += (long long)gridDim.x * blockDim.x) {
    float lg[C], pr[C], lse, mx;
#pragma unroll
    for (int c = 0; c < C; ++c) lg[c] = logits[p * C + c];
    softmax_c<C>(lg, pr, lse, mx);
    const int l = labels[p];
    const int img = (int)(p / hw);
    const float ie = (float)iu[img * 2];
    const float ue = (float)(iu[img * 2 + 1] + (double)eps);
    float dp[C];
    dp[0] = 0.f;
    float dot = 0.f;
#pragma unroll
    for (int c = 1; c < C; ++c) {
      const float oh = (l == c) ? 1.f : 0.f;
      dp[c] = -(2.f / n) * (oh * ue - ie) / (ue * ue);
      dot += dp[c] * pr[c];
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const float g = loss_scale * pr[c] * (dp[c] - dot);
      dlogits[p * C + c] = accumulate ? dlogits[p * C + c] + g : g;
    }
  }
}

int check_loss(bsl_ctx* ctx, const bsl_loss_desc* d) {
  if (!ctx) return BSL_EINVAL;
  if (!d) return bsl_fail(ctx, BSL_EINVAL, "loss: null descriptor");
  if (d->n <= 0 || d->hw <= 0) return bsl_fail(ctx, BSL_EINVAL, "loss: non-positive size");
  if (d->classes < 2 || d->classes > MAXC)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "loss: classes=%d (2..%d)", d->classes, MAXC);
  if (d->weight_type < 0 || d->weight_type > 2)
    return bsl_fail(ctx, BSL_EUNSUPPORTED,
                    "loss: weight_type=%d (0 none, 1 numerical, 2 proportion; 'boundary' is a host scipy op in "
                    "the reference and is out of scope)", d->weight_type);
  return BSL_OK;
}

unsigned px_grid(bsl_ctx* ctx, long long pixels) {
  long long b = (pixels + 255) / 256;
  const long long cap = 8LL * ctx->sm_count;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

#define CLASS_SWITCH(C_, CALL)                       \
  switch (C_) {                                      \
    case 2: { constexpr int C = 2; CALL; } break;    \
    case 3: { constexpr int C = 3; CALL; } break;    \
    case 4: { constexpr int C = 4; CALL; } break;    \
  }

}  // namespace

extern "C" {

int bsl_label_counts(bsl_ctx* ctx, const bsl_loss_desc* d, const int* labels, int* counts, void* stream) {
  int rc = check_loss(ctx, d);
  if (rc) return rc;
  if (!labels || !counts) return bsl_fail(ctx, BSL_EINVAL, "label_counts: null buffer");
  cudaStream_t s = as_stream(stream);
  BSL_CUDA(ctx, cudaMemsetAsync(counts, 0, sizeof(int) * d->n * d->classes, s));
  int bx = (d->hw + 255) / 256;
  if (bx > 64) bx = 64;
  bsl_launch(label_counts_kernel, dim3(dim3(bx, d->n)), dim3(256), 0, s, labels, d->hw, d->classes, counts);
  BSL_LAUNCH_CHECK(ctx, "label_counts_kernel");
  return BSL_OK;
}

size_t bsl_loss_workspace(bsl_ctx* ctx, const bsl_loss_desc* d) {
  if (!ctx || !d) return 0;
  // [nz double][wtab float n*MAXC (padded)][partials double 8*SMs][dice iu double 2n][dice partials]
  return 64 + (size_t)d->n * MAXC * 4 + 64 + (size_t)8 * ctx->sm_count * 8 + (size_t)d->n * 2 * 8 +
         (size_t)d->n * 64 * 2 * 8 + 256;
}

struct LossWs {
  double* nz;
  float* wtab;
  double* part;
  double* iu;
  double* dpart;
};

static LossWs carve(bsl_ctx* ctx, const bsl_loss_desc* d, void* ws) {
  char* p = reinterpret_cast<char*>(ws);
  LossWs w;
  w.nz = reinterpret_cast<double*>(p); p += 64;
  w.wtab = reinterpret_cast<float*>(p); p += (((size_t)d->n * MAXC * 4 + 63) / 64) * 64;
  w.part = reinterpret_cast<double*>(p); p += (size_t)8 * ctx->sm_count * 8;
  w.iu = reinterpret_cast<double*>(p); p += (size_t)d->n * 2 * 8;
  w.dpart = reinterpret_cast<double*>(p);
  return w;
}

int bsl_wxent_fwd_bwd(bsl_ctx* ctx, const bsl_loss_desc* d, const float* logits, const int* labels,
                      const int* counts, float* loss, float* dlogits, void* workspace, size_t workspace_bytes,
                      void* stream) {
  int rc = check_loss(ctx, d);
  if (rc) return rc;
  if (!logits || !labels || !counts || !loss || !workspace)
    return bsl_fail(ctx, BSL_EINVAL, "wxent: null buffer");
  if (workspace_bytes < bsl_loss_workspace(ctx, d)) return bsl_fail(ctx, BSL_EWORKSPACE, "wxent: workspace too small");
  cudaStream_t s = as_stream(stream);
  LossWs w = carve(ctx, d, workspace);
  bsl_launch(weight_table_kernel, dim3(1), dim3(32), 0, s, *d, counts, w.wtab, w.nz);
  BSL_LAUNCH_CHECK(ctx, "weight_table_kernel");
  const long long pixels = (long long)d->n * d->hw;
  const unsigned blocks = px_grid(ctx, pixels);
  const bool vec = d->hw % 4 == 0 && ((uintptr_t)logits | (uintptr_t)labels | (uintptr_t)dlogits) % 16 == 0;
  if (vec) {
    CLASS_SWITCH(d->classes, (bsl_launch(wxent_kernel<C, true>, dim3(blocks), dim3(256), 0, s, logits, labels, d->hw, pixels,
                                         w.wtab, w.nz, d->loss_scale, dlogits, w.part)));
  } else {
    CLASS_SWITCH(d->classes, (bsl_launch(wxent_kernel<C, false>, dim3(blocks), dim3(256), 0, s, logits, labels, d->hw, pixels,
                                         w.wtab, w.nz, d->loss_scale, dlogits, w.part)));
  }
  BSL_LAUNCH_CHECK(ctx, "wxent_kernel");
  bsl_launch(wxent_final_kernel, dim3(1), dim3(32), 0, s, w.part, (int)blocks, w.nz, loss);
  BSL_LAUNCH_CHECK(ctx, "wxent_final_kernel");
  return BSL_OK;
}

int bsl_dice_fwd_bwd(bsl_ctx* ctx, const bsl_loss_desc* d, const float* logits, const int* labels, float* loss,
                     float* dlogits, int accumulate, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_loss(ctx, d);
  if (rc) return rc;
  if (!logits || !labels || !loss || !workspace) return bsl_fail(ctx, BSL_EINVAL, "dice: null buffer");
  if (workspace_bytes < bsl_loss_workspace(ctx, d)) return bsl_fail(ctx, BSL_EWORKSPACE, "dice: workspace too small");
  cudaStream_t s = as_stream(stream);
  LossWs w = carve(ctx, d, workspace);
  int bx = (d->hw + 255) / 256;
  if (bx > 64) bx = 64;
  const float eps = 1e-8f;
  CLASS_SWITCH(d->classes, (bsl_launch(dice_reduce_kernel<C>, dim3(dim3(bx, d->n)), dim3(256), 0, s, logits, labels, d->hw, w.dpart)));
  BSL_LAUNCH_CHECK(ctx, "dice_reduce_kernel");
  bsl_launch(dice_final_kernel, dim3(1), dim3(d->n >= 32 ? 1024 : (d->n >= 8 ? 256 : 32)), 0, s, w.dpart, bx, d->n, eps, w.iu, loss);
  BSL_LAUNCH_CHECK(ctx, "dice_final_kernel");
  if (dlogits) {
    const long long pixels = (long long)d->n * d->hw;
    CLASS_SWITCH(d->classes, (bsl_launch(dice_bwd_kernel<C>, dim3(px_grid(ctx, pixels)), dim3(256), 0, s, 
                                 logits, labels, d->hw, pixels, d->n, eps, w.iu, d->loss_scale, accumulate, dlogits)));
    BSL_LAUNCH_CHECK(ctx, "dice_bwd_kernel");
  }
  return BSL_OK;
}

int bsl_softmax_threshold(bsl_ctx* ctx, const bsl_loss_desc* d, const float* logits, const int* labels, float* prob,
                          uint8_t* masks, uint8_t* argmax, unsigned int* ilr, void* stream) {
  int rc = check_loss(ctx, d);
  if (rc) return rc;
  if (!logits) return bsl_fail(ctx, BSL_EINVAL, "softmax_threshold: null logits");
  if (ilr && !labels) return bsl_fail(ctx, BSL_EINVAL, "softmax_threshold: counts need labels");
  cudaStream_t s = as_stream(stream);
  if (ilr) BSL_CUDA(ctx, cudaMemsetAsync(ilr, 0, sizeof(unsigned int) * d->n * (d->classes - 1) * 3, s));
  const long long pixels = (long long)d->n * d->hw;
  CLASS_SWITCH(d->classes, (bsl_launch(softmax_threshold_kernel<C>, dim3(px_grid(ctx, pixels)), dim3(256), 0, s, 
                               logits, labels, d->hw, pixels, prob, masks, argmax, ilr)));
  BSL_LAUNCH_CHECK(ctx, "softmax_threshold_kernel");
  return BSL_OK;
}

}  // extern "C"
