// GUNet guide sub-networks (small, fp32, CUDA-core): the context MLP that produces the per-(sample, channel)
// modulation vector and the average-pooled pyramid of the spatial guide.
//   slim_nets.fc / mlp (fully_connected + dropout)   <- NetworksV2/Backbone/slim_nets.py:34-57, GUNet.py:31-59
//   slim.avg_pool2d(gs, 2) pyramid                   <- NetworksV2/GUNet.py:136-159
// The 1x1 guide convolutions themselves are never materialised: norm.cu evaluates guide[p] . w[:, c] inside the
// normalisation passes of the layer they modulate.
#include "internal.h"
#include "philox.cuh"
#include <cuda_bf16.h>

namespace {
using bsl::philox4x32_10;

__device__ __forceinline__ float dropout_scale(const bsl_dropout_desc& dd, unsigned long long idx) {
  // tf.nn.dropout: binary = floor(keep_prob + uniform[0,1)); y = x / keep_prob * binary
  const uint4 r = philox4x32_10(make_uint4((unsigned)(idx >> 2), (unsigned)(idx >> 34), (unsigned)dd.offset,
                                           (unsigned)(dd.offset >> 32)),
                                make_uint2((unsigned)dd.seed, (unsigned)(dd.seed >> 32)));
  const unsigned lane = (unsigned)(idx & 3);
  const unsigned bits = lane == 0 ? r.x : lane == 1 ? r.y : lane == 2 ? r.z : r.w;
  const float u = __uint_as_float((bits & 0x7fffffu) | 0x3f800000u) - 1.0f;
  return floorf(dd.keep_prob + u) >= 1.0f ? 1.0f / dd.keep_prob : 0.0f;
}

__global__ void fc_fwd_kernel(int n, int cin, int cout, const float* __restrict__ x, const float* __restrict__ w,
                              const float* __restrict__ b, int relu, bsl_dropout_desc dd, int use_dropout,
                              float* __restrict__ y) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * cout) return;
  const int s = i / cout, co = i - s * cout;
  float acc = b ? b[co] : 0.f;
  const float* xr = x + (long long)s * cin;
  for (int ci = 0; ci < cin; ++ci) acc = fmaf(xr[ci], w[(long long)ci * cout + co], acc);
  if (relu) acc = fmaxf(acc, 0.f);
  if (use_dropout) acc *= dropout_scale(dd, (unsigned long long)i);
  y[i] = acc;
}

// dpre = dy * d(out)/d(pre): out = relu(pre) * mask / keep, so out > 0 <=> (pre > 0 and kept).
__global__ void fc_dpre_kernel(int total, const float* __restrict__ y, const float* __restrict__ dy, int relu,
                               float inv_keep, float* __restrict__ dpre) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  float g = dy[i];
  if (relu) g = y[i] > 0.f ? g * inv_keep : 0.f;
  dpre[i] = g;
}

__global__ void fc_dw_kernel(int n, int cin, int cout, const float* __restrict__ x, const float* __restrict__ dpre,
                             float* __restrict__ dw, float* __restrict__ db) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (cin + 1) * cout) return;
  const int ci = i / cout, co = i - ci * cout;
  float acc = 0.f;
  if (ci < cin) {
    for (int s = 0; s < n; ++s) acc = fmaf(x[(long long)s * cin + ci], dpre[(long long)s * cout + co], acc);
    dw[i] = acc;
  } else if (db) {
    for (int s = 0; s < n; ++s) acc += dpre[(long long)s * cout + co];
    db[co] = acc;
  }
}

// one warp per (sample, input feature): lanes stride over cout (coalesced rows of w), shuffle tree at the end
__global__ void fc_dx_kernel(int n, int cin, int cout, const float* __restrict__ dpre, const float* __restrict__ w,
                             float* __restrict__ dx) {
  bsl::pdl_wait();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n * cin) return;
  const int s = warp / cin, ci = warp - s * cin;
  float acc = 0.f;
  for (int co = lane; co < cout; co += 32) acc = fmaf(dpre[(long long)s * cout + co], w[(long long)ci * cout + co], acc);
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) dx[warp] = acc;
}

__global__ void avgpool2x2_f32_kernel(int n, int h, int w, int c, const float* __restrict__ x, float* __restrict__ y) {
  bsl::pdl_wait();
  const int ho = h / 2, wo = w / 2;
  const long long total = (long long)n * ho * wo * c;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int ch = (int)(t % c); t /= c;
    const int xo = (int)(t % wo); t /= wo;
    const int yo = (int)(t % ho);
    const int s = (int)(t / ho);
    const float* p = x + (((long long)s * h + 2 * yo) * w + 2 * xo) * c + ch;
    y[i] = ((p[0] + p[c]) + (p[(long long)w * c] + p[(long long)w * c + c])) * 0.25f;
  }
}

// UNetInter --mid_cat (NetworksV2/UNetInter.py:124-125): max_pool2d(concat(net, sp_guide), 2) -- the guide's share of the
// pooled tensor, written as bf16 lanes [0, c) of y rows with stride y_ld (the activation lanes are written by the fused
// norm + ReLU + pool pass). bf16 rounding is monotonic, so round(max) == max(round).
__global__ void maxpool2x2_f32_bf16_kernel(int n, int h, int w, int c, const float* __restrict__ x,
                                           __nv_bfloat16* __restrict__ y, int y_ld) {
  bsl::pdl_wait();
  const int ho = h / 2, wo = w / 2;
  const long long total = (long long)n * ho * wo * c;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int ch = (int)(t % c); t /= c;
    const int xo = (int)(t % wo); t /= wo;
    const int yo = (int)(t % ho);
    const int s = (int)(t / ho);
    const float* p = x + (((long long)s * h + 2 * yo) * w + 2 * xo) * c + ch;
    const float m = fmaxf(fmaxf(p[0], p[c]), fmaxf(p[(long long)w * c], p[(long long)w * c + c]));
    y[(((long long)s * ho + yo) * wo + xo) * y_ld + ch] = __float2bfloat16_rn(m);
  }
}

// --img_grad (NetworksV2/GUNet.py:333-337): concat(images, dy, dx) with (dy, dx) = tf.image.image_gradients(images) --
// forward differences along H and W, zero in the last row / column -- written as bf16 lanes [0, 3c) of rows with stride
// y_ld (the remaining lanes of the zero-initialised buffer pad the first conv's input to a 64-channel block).
__global__ void image_gradients_pack_kernel(int n, int h, int w, int c, const float* __restrict__ x,
                                            __nv_bfloat16* __restrict__ y, int y_ld) {
  bsl::pdl_wait();
  const long long total = (long long)n * h * w * c;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int ch = (int)(t % c); t /= c;
    const int xx = (int)(t % w); t /= w;
    const int yy = (int)(t % h);
    const float v = x[i];
    const float dy = yy + 1 < h ? x[i + (long long)w * c] - v : 0.f;
    const float dx = xx + 1 < w ? x[i + c] - v : 0.f;
    __nv_bfloat16* o = y + (i / c) * y_ld;
    o[ch] = __float2bfloat16_rn(v);
    o[c + ch] = __float2bfloat16_rn(dy);
    o[2 * c + ch] = __float2bfloat16_rn(dx);
  }
}

// Backbone --dropout of GUNet (slim.dropout between normaliser and modulation, NetworksV2/GUNet.py:189-190) and its
// gradient (the same multiplication): out[p][ch] = bf16(x[p][ch] * multiplier(p * c + ch)), 8 channels per thread = two
// Philox counters (flat element index over the dense [pixels, c] tensor, as bsl_dropout_mask enumerates it).
__global__ void dropout_bf16_kernel(long long pixels, int c, bsl_dropout_desc dd, const __nv_bfloat16* __restrict__ x,
                                    int x_ld, __nv_bfloat16* __restrict__ out, int o_ld) {
  bsl::pdl_wait();
  const int cg = c / 8;
  const long long total = pixels * cg;
  const float inv = 1.0f / dd.keep_prob;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long p = i / cg;
    const int ch0 = (int)(i - p * cg) * 8;
    const unsigned long long idx = (unsigned long long)p * c + ch0;      // multiple of 8
    const uint4 raw = *reinterpret_cast<const uint4*>(x + p * x_ld + ch0);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
    uint4 res;
    __nv_bfloat162* o = reinterpret_cast<__nv_bfloat162*>(&res);
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const unsigned long long blk = (idx >> 2) + q;
      const uint4 r = philox4x32_10(make_uint4((unsigned)blk, (unsigned)(blk >> 32), (unsigned)dd.offset,
                                               (unsigned)(dd.offset >> 32)),
                                    make_uint2((unsigned)dd.seed, (unsigned)(dd.seed >> 32)));
      const unsigned bits[4] = {r.x, r.y, r.z, r.w};
      float m[4];
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        const float u = __uint_as_float((bits[l] & 0x7fffffu) | 0x3f800000u) - 1.0f;
        m[l] = floorf(dd.keep_prob + u) >= 1.0f ? inv : 0.0f;
      }
      const float2 a = __bfloat1622float2(h[2 * q]), b = __bfloat1622float2(h[2 * q + 1]);
      o[2 * q] = __floats2bfloat162_rn(a.x * m[0], a.y * m[1]);
      o[2 * q + 1] = __floats2bfloat162_rn(b.x * m[2], b.y * m[3]);
    }
    *reinterpret_cast<uint4*>(out + p * o_ld + ch0) = res;
  }
}

__global__ void dropout_mask_kernel(int total, bsl_dropout_desc dd, float* __restrict__ out) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) out[i] = dropout_scale(dd, (unsigned long long)i);
}

int check_fc(bsl_ctx* ctx, const bsl_fc_desc* d) {
  if (!ctx) return BSL_EINVAL;
  if (!d) return bsl_fail(ctx, BSL_EINVAL, "fc: null descriptor");
  if (d->n <= 0 || d->cin <= 0 || d->cout <= 0) return bsl_fail(ctx, BSL_EINVAL, "fc: non-positive size");
  if (d->use_dropout && !(d->dropout.keep_prob > 0.f && d->dropout.keep_prob <= 1.f))
    return bsl_fail(ctx, BSL_EINVAL, "fc: keep_prob %f outside (0, 1]", d->dropout.keep_prob);
  if (d->use_dropout && !d->relu)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "fc: dropout is only defined after the ReLU layers of slim_nets.mlp");
  return BSL_OK;
}

}  // namespace

extern "C" {

int bsl_fc_fwd(bsl_ctx* ctx, const bsl_fc_desc* d, const float* x, const float* w, const float* bias, float* y,
               void* stream) {
  int rc = check_fc(ctx, d);
  if (rc) return rc;
  if (!x || !w || !y) return bsl_fail(ctx, BSL_EINVAL, "fc_fwd: null buffer");
  const int total = d->n * d->cout;
  bsl_launch(fc_fwd_kernel, dim3((total + 127) / 128), dim3(128), 0, as_stream(stream), d->n, d->cin, d->cout, x, w, bias, d->relu,
                                                                   d->dropout, d->use_dropout, y);
  BSL_LAUNCH_CHECK(ctx, "fc_fwd_kernel");
  return BSL_OK;
}

size_t bsl_fc_bwd_workspace(bsl_ctx* ctx, const bsl_fc_desc* d) {
  if (!ctx || !d || check_fc(ctx, d)) return 0;
  return (size_t)d->n * d->cout * sizeof(float);
}

int bsl_fc_bwd(bsl_ctx* ctx, const bsl_fc_desc* d, const float* x, const float* w, const float* y, const float* dy,
               float* dx, float* dw, float* dbias, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_fc(ctx, d);
  if (rc) return rc;
  if (!x || !w || !y || !dy || !dw) return bsl_fail(ctx, BSL_EINVAL, "fc_bwd: null buffer");
  const size_t need = (size_t)d->n * d->cout * sizeof(float);
  if (!workspace || workspace_bytes < need)
    return bsl_fail(ctx, BSL_EWORKSPACE, "fc_bwd: workspace %zu < %zu", workspace_bytes, need);
  float* dpre = reinterpret_cast<float*>(workspace);
  cudaStream_t s = as_stream(stream);
  const int total = d->n * d->cout;
  bsl_launch(fc_dpre_kernel, dim3((total + 255) / 256), dim3(256), 0, s, total, y, dy, d->relu,
                                                     d->use_dropout ? 1.0f / d->dropout.keep_prob : 1.0f, dpre);
  BSL_LAUNCH_CHECK(ctx, "fc_dpre_kernel");
  const int nw = (d->cin + 1) * d->cout;
  bsl_launch(fc_dw_kernel, dim3((nw + 127) / 128), dim3(128), 0, s, d->n, d->cin, d->cout, x, dpre, dw, dbias);
  BSL_LAUNCH_CHECK(ctx, "fc_dw_kernel");
  if (dx) {
    const long long threads = (long long)d->n * d->cin * 32;
    bsl_launch(fc_dx_kernel, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, s, d->n, d->cin, d->cout, dpre, w, dx);
    BSL_LAUNCH_CHECK(ctx, "fc_dx_kernel");
  }
  return BSL_OK;
}

int bsl_dropout_mask(bsl_ctx* ctx, const bsl_dropout_desc* d, size_t n, float* out, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!d || !out || !(d->keep_prob > 0.f && d->keep_prob <= 1.f) || n > 0x7fffffffu)
    return bsl_fail(ctx, BSL_EINVAL, "dropout_mask: bad argument");
  bsl_launch(dropout_mask_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, as_stream(stream), (int)n, *d, out);
  BSL_LAUNCH_CHECK(ctx, "dropout_mask_kernel");
  return BSL_OK;
}

int bsl_avgpool2x2_f32(bsl_ctx* ctx, int n, int h, int w, int c, const float* x, float* y, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!x || !y) return bsl_fail(ctx, BSL_EINVAL, "avgpool2x2: null buffer");
  if (n <= 0 || c <= 0 || h <= 0 || w <= 0 || (h & 1) || (w & 1))
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "avgpool2x2: h=%d w=%d must be even (SAME == VALID then)", h, w);
  const long long total = (long long)n * (h / 2) * (w / 2) * c;
  long long blocks = (total + 255) / 256;
  const long long cap = 16LL * ctx->sm_count;
  if (blocks > cap) blocks = cap;
  bsl_launch(avgpool2x2_f32_kernel, dim3((unsigned)blocks), dim3(256), 0, as_stream(stream), n, h, w, c, x, y);
  BSL_LAUNCH_CHECK(ctx, "avgpool2x2_f32_kernel");
  return BSL_OK;
}

int bsl_image_gradients_pack(bsl_ctx* ctx, int n, int h, int w, int c, const float* x, void* y_bf16, int y_ld,
                             void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!x || !y_bf16) return bsl_fail(ctx, BSL_EINVAL, "image_gradients_pack: null buffer");
  if (n <= 0 || h <= 0 || w <= 0 || c <= 0 || y_ld < 3 * c)
    return bsl_fail(ctx, BSL_EINVAL, "image_gradients_pack: y_ld=%d must hold 3 * c = %d lanes", y_ld, 3 * c);
  const long long total = (long long)n * h * w * c;
  long long blocks = (total + 255) / 256;
  const long long cap = 16LL * ctx->sm_count;
  if (blocks > cap) blocks = cap;
  bsl_launch(image_gradients_pack_kernel, dim3((unsigned)blocks), dim3(256), 0, as_stream(stream), n, h, w, c, x,
             reinterpret_cast<__nv_bfloat16*>(y_bf16), y_ld);
  BSL_LAUNCH_CHECK(ctx, "image_gradients_pack_kernel");
  return BSL_OK;
}

int bsl_dropout_bf16(bsl_ctx* ctx, const bsl_dropout_desc* d, long long pixels, int c, const void* x_bf16, int x_ld,
                     void* out_bf16, int out_ld, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!d || !x_bf16 || !out_bf16) return bsl_fail(ctx, BSL_EINVAL, "dropout_bf16: null argument");
  if (!(d->keep_prob > 0.f && d->keep_prob <= 1.f)) return bsl_fail(ctx, BSL_EINVAL, "dropout_bf16: keep_prob %f outside (0, 1]", d->keep_prob);
  if (pixels <= 0 || c <= 0 || c % 8 || x_ld < c || out_ld < c || x_ld % 8 || out_ld % 8)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "dropout_bf16: c=%d (multiple of 8), strides %d / %d", c, x_ld, out_ld);
  const long long total = pixels * (c / 8);
  long long blocks = (total + 255) / 256;
  const long long cap = 16LL * ctx->sm_count;
  if (blocks > cap) blocks = cap;
  bsl_launch(dropout_bf16_kernel, dim3((unsigned)blocks), dim3(256), 0, as_stream(stream), pixels, c, *d,
             reinterpret_cast<const __nv_bfloat16*>(x_bf16), x_ld, reinterpret_cast<__nv_bfloat16*>(out_bf16), out_ld);
  BSL_LAUNCH_CHECK(ctx, "dropout_bf16_kernel");
  return BSL_OK;
}

int bsl_maxpool2x2_f32_bf16(bsl_ctx* ctx, int n, int h, int w, int c, const float* x, void* y_bf16, int y_ld,
                            void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!x || !y_bf16) return bsl_fail(ctx, BSL_EINVAL, "maxpool2x2_f32_bf16: null buffer");
  if (n <= 0 || c <= 0 || h <= 0 || w <= 0 || (h & 1) || (w & 1) || y_ld < c)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "maxpool2x2_f32_bf16: h=%d w=%d must be even, y_ld=%d >= c=%d", h, w, y_ld, c);
  const long long total = (long long)n * (h / 2) * (w / 2) * c;
  long long blocks = (total + 255) / 256;
  const long long cap = 16LL * ctx->sm_count;
  if (blocks > cap) blocks = cap;
  bsl_launch(maxpool2x2_f32_bf16_kernel, dim3((unsigned)blocks), dim3(256), 0, as_stream(stream), n, h, w, c, x,
             reinterpret_cast<__nv_bfloat16*>(y_bf16), y_ld);
  BSL_LAUNCH_CHECK(ctx, "maxpool2x2_f32_bf16_kernel");
  return BSL_OK;
}

}  // extern "C"
