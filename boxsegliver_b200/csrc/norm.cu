// Normalisation (+ReLU, +2x2 max-pool) forward and backward, HBM-bound passes.
//   slim.batch_norm  (FusedBatchNorm / FusedBatchNormGrad)  <- NetworksV2/base.py:154-162
//   slim.instance_norm (moments + batch_normalization)      <- NetworksV2/base.py:163-165
//   slim.max_pool2d 2x2 s2 (MaxPool / MaxPoolGrad)          <- NetworksV2/UNet.py:81
//   ReluGrad                                                <- slim default activation_fn
// Statistics are two-level deterministic reductions (reduce.cuh); the apply passes move 16 B per
// thread per access along the NHWC channel axis.
#include "reduce.cuh"
#include <mutex>
#include <unordered_map>

using namespace bsl;

namespace bsl {
// Block = 32 consecutive outputs x 32 partial lanes (1024 threads): lane q sums partials q, q + 32, ... in order
// (coalesced across outputs, 4 independent loads in flight), then the 32 lane sums are added in a fixed order.
// With up to 1184 partial blocks per output the 8-lane version spent ~10 us per launch on its chain of dependent
// L2 round trips, 41 launches per training step.
__global__ void __launch_bounds__(1024) pixel_reduce_final_kernel(const float* __restrict__ part, int blocks, int kc,
                                                                  double* __restrict__ out) {
  bsl::pdl_wait();
  __shared__ double sm[32][33];
  const int il = threadIdx.x & 31, q = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + il;
  double s = 0.0;
  if (i < kc) {
    const float* p = part + (long long)blockIdx.y * blocks * kc + i;
    int b = q;
    for (; b + 96 < blocks; b += 128) {
      const float v0 = p[(long long)b * kc], v1 = p[(long long)(b + 32) * kc], v2 = p[(long long)(b + 64) * kc],
                  v3 = p[(long long)(b + 96) * kc];
      s += (double)v0;
      s += (double)v1;
      s += (double)v2;
      s += (double)v3;
    }
    for (; b < blocks; b += 32) s += (double)p[(long long)b * kc];
  }
  sm[q][il] = s;
  __syncthreads();
  if (q == 0 && i < kc) {
    double t = sm[0][il];
#pragma unroll
    for (int k = 1; k < 32; ++k) t += sm[k][il];
    out[(long long)blockIdx.y * kc + i] = t;
  }
}

// Scratch arena for the two-level reductions: one per (context, stream), so reductions enqueued on the side streams
// (filter gradients, all-reduce tails) never share partials with the ones on the compute stream. Grows on demand;
// growth frees the old arena with cudaFree (which synchronises the device first) and is refused while the stream is
// being captured into a CUDA graph: the pointer would be baked into the graph and cudaMalloc is illegal there.
int bsl_scratch(bsl_ctx* ctx, size_t bytes, float** out, cudaStream_t stream) {
  std::lock_guard<std::mutex> g(ctx->scratch_mu);
  bsl_ctx::Scratch& a = ctx->scratch[stream];
  if (bytes > a.bytes) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone)
      return bsl_fail(ctx, BSL_EINVAL,
                      "scratch arena of this stream must grow (%zu > %zu bytes) while the stream is capturing: run the "
                      "sequence once outside capture first", bytes, a.bytes);
    if (a.ptr) cudaFree(a.ptr);
    size_t want = bytes < (16u << 20) ? (16u << 20) : bytes;
    a.ptr = nullptr;
    a.bytes = 0;
    BSL_CUDA(ctx, cudaMalloc(&a.ptr, want));
    a.bytes = want;
  }
  *out = a.ptr;
  return BSL_OK;
}

// A second, small arena per (context, stream) for filters re-laid-out in front of a convolution (the K-major copy the
// CTA-pair kernels read): separate from the reduction arena, which the same call may use for its statistics partials.
int bsl_scratch_w(bsl_ctx* ctx, size_t bytes, void** out, cudaStream_t stream) {
  std::lock_guard<std::mutex> g(ctx->scratch_mu);
  bsl_ctx::Scratch& a = ctx->scratch_w[stream];
  if (bytes > a.bytes) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone)
      return bsl_fail(ctx, BSL_EINVAL, "filter scratch of this stream must grow while the stream is capturing");
    if (a.ptr) cudaFree(a.ptr);
    const size_t want = bytes < (1u << 20) ? (1u << 20) : bytes;
    a.ptr = nullptr;
    a.bytes = 0;
    BSL_CUDA(ctx, cudaMalloc(&a.ptr, want));
    a.bytes = want;
  }
  *out = a.ptr;
  return BSL_OK;
}
}  // namespace bsl

void bsl_scratch_release(bsl_ctx* ctx, cudaStream_t stream, bool all) {
  std::lock_guard<std::mutex> g(ctx->scratch_mu);
  for (auto* m : {&ctx->scratch, &ctx->scratch_w})
    for (auto it = m->begin(); it != m->end();) {
      if (all || it->first == stream) {
        if (it->second.ptr) cudaFree(it->second.ptr);
        it = m->erase(it);
      } else {
        ++it;
      }
    }
}

namespace {

struct StatsF {
  static constexpr int K = 2, NIN = 1, UNROLL = 8;
  struct State {};
  const __nv_bfloat16* y;
  int ld;
  __device__ void init(State&, int, int) const {}
  __device__ void load(long long p, int ch0, uint4 (&raw)[1]) const { raw[0] = ld16(y + p * ld + ch0); }
  __device__ void accum(const State&, long long, const uint4 (&raw)[1], float (&acc)[2][8]) const {
    float v[8];
    unpack8(raw[0], v);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc[0][j] += v[j];
      acc[1][j] = fmaf(v[j], v[j], acc[1][j]);
    }
  }
};

// G = channels of the additive spatial-guide map (GUNet modulated_conv_block, NetworksV2/GUNet.py:205-210):
// z += sum_g guide[p][g] * wsp[g][c]; the extra K rows are sum(dz * guide_g) (gradient of the 1x1 guide conv).
template <int G>
struct BwdFG {
  static constexpr int K = 2 + G, NIN = 2, UNROLL = 4;
  struct State {
    float scale[8], shift[8], rstd[8], mrstd[8];
    float wsp[G ? G : 1][8];
  };
  const float* guide;
  const float* wsp;
  int wsp_ld;
  const __nv_bfloat16* y;
  const __nv_bfloat16* da;
  const float* mean;
  const float* rstd;
  const float* scale;
  const float* shift;
  int y_ld, da_ld, c, relu;
  __device__ void init(State& st, int group, int ch0) const {
    const int o = group * c + ch0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      st.scale[j] = scale[o + j];
      st.shift[j] = shift[o + j];
      st.rstd[j] = rstd[o + j];
      st.mrstd[j] = mean[o + j] * rstd[o + j];
#pragma unroll
      for (int q = 0; q < G; ++q) st.wsp[q][j] = wsp[q * wsp_ld + ch0 + j];
    }
  }
  __device__ void load(long long p, int ch0, uint4 (&raw)[2]) const {
    raw[0] = ld16(y + p * y_ld + ch0);
    raw[1] = ld16(da + p * da_ld + ch0);
  }
  __device__ void accum(const State& st, long long p, const uint4 (&raw)[2], float (&acc)[2 + G][8]) const {
    float v[8], g[8], gm[G ? G : 1];
    unpack8(raw[0], v);
    unpack8(raw[1], g);
#pragma unroll
    for (int q = 0; q < G; ++q) gm[q] = __ldg(guide + p * G + q);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float z = fmaf(v[j], st.scale[j], st.shift[j]);
#pragma unroll
      for (int q = 0; q < G; ++q) z = fmaf(gm[q], st.wsp[q][j], z);
      const float dz = (!relu || z > 0.f) ? g[j] : 0.f;
      const float xh = fmaf(v[j], st.rstd[j], -st.mrstd[j]);
      acc[0][j] += dz;
      acc[1][j] = fmaf(dz, xh, acc[1][j]);
#pragma unroll
      for (int q = 0; q < G; ++q) acc[2 + q][j] = fmaf(dz, gm[q], acc[2 + q][j]);
    }
  }
};
using BwdF = BwdFG<0>;

__global__ void norm_finalize_kernel(int groups, int c, double m, float eps, float decay, int bn_training,
                                     int use_moving, int center, int scale_flag, const double* __restrict__ sums,
                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                     float* __restrict__ moving_mean, float* __restrict__ moving_var,
                                     float* __restrict__ mean_o, float* __restrict__ rstd_o,
                                     float* __restrict__ scale_o, float* __restrict__ shift_o) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= groups * c) return;
  const int g = i / c, ch = i - g * c;
  double mean, var;
  if (use_moving) {
    mean = moving_mean[ch];
    var = moving_var[ch];
  } else {
    const double s0 = sums[(long long)g * 2 * c + ch];
    const double s1 = sums[(long long)g * 2 * c + c + ch];
    mean = s0 / m;
    var = s1 / m - mean * mean;
    if (var < 0.0) var = 0.0;
    if (bn_training) {  // FusedBatchNorm: moving variance is fed the Bessel-corrected estimate
      const double unb = var * (m / (m > 1.0 ? m - 1.0 : 1.0));
      moving_mean[ch] = (float)((double)moving_mean[ch] * decay + mean * (1.0 - (double)decay));
      moving_var[ch] = (float)((double)moving_var[ch] * decay + unb * (1.0 - (double)decay));
    }
  }
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  const float sc = (scale_flag ? gamma[ch] : 1.f) * rstd;
  mean_o[i] = (float)mean;
  rstd_o[i] = rstd;
  scale_o[i] = sc;
  shift_o[i] = (center ? beta[ch] : 0.f) - (float)mean * sc;
}

// Elementwise passes share one thread layout: block = (rows x c/8 channel groups), a thread owns ONE
// 8-channel group for the whole launch, so its per-channel parameters live in registers, and it
// keeps 4 independent 16 B loads in flight. grid.y = sample index when parameters are per sample.
constexpr int EW_UNROLL = 4;

template <int G>
__global__ void norm_apply_kernel(const __nv_bfloat16* __restrict__ y, int y_ld, __nv_bfloat16* __restrict__ a,
                                  int a_ld, long long pixels_per_group, int c, int relu,
                                  const float* __restrict__ scale, const float* __restrict__ shift,
                                  const float* __restrict__ guide, const float* __restrict__ wsp, int wsp_ld,
                                  int gstride) {
  bsl::pdl_wait();
  // blockIdx.y = group (instance norm: gstride = c) or image slice of the batch (batch norm, gstride = 0)
  const int cg = c / 8;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  const int ch0 = g * 8;
  const int o = blockIdx.y * gstride + ch0;
  float sc[8], sh[8], ws[G ? G : 1][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = scale[o + j];
    sh[j] = shift[o + j];
#pragma unroll
    for (int q = 0; q < G; ++q) ws[q][j] = wsp[q * wsp_ld + ch0 + j];
  }
  const long long base = (long long)blockIdx.y * pixels_per_group;
  const long long stride = (long long)gridDim.x * rows;
  long long p = (long long)blockIdx.x * rows + r;
  for (; p + (EW_UNROLL - 1) * stride < pixels_per_group; p += EW_UNROLL * stride) {
    uint4 raw[EW_UNROLL];
    float gm[EW_UNROLL][G ? G : 1];
#pragma unroll
    for (int u = 0; u < EW_UNROLL; ++u) {
      raw[u] = ld16(y + (base + p + u * stride) * y_ld + ch0);
#pragma unroll
      for (int q = 0; q < G; ++q) gm[u][q] = __ldg(guide + (base + p + u * stride) * G + q);
    }
#pragma unroll
    for (int u = 0; u < EW_UNROLL; ++u) {
      float v[8];
      unpack8(raw[u], v);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float z = fmaf(v[j], sc[j], sh[j]);
#pragma unroll
        for (int q = 0; q < G; ++q) z = fmaf(gm[u][q], ws[q][j], z);
        v[j] = relu ? fmaxf(z, 0.f) : z;
      }
      st16(a + (base + p + u * stride) * a_ld + ch0, pack8(v));
    }
  }
  for (; p < pixels_per_group; p += stride) {
    float v[8];
    unpack8(ld16(y + (base + p) * y_ld + ch0), v);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float z = fmaf(v[j], sc[j], sh[j]);
#pragma unroll
      for (int q = 0; q < G; ++q) z = fmaf(__ldg(guide + (base + p) * G + q), ws[q][j], z);
      v[j] = relu ? fmaxf(z, 0.f) : z;
    }
    st16(a + (base + p) * a_ld + ch0, pack8(v));
  }
}

// norm_apply_kernel (no guide) that also evaluates the 1x1 logits convolution on the activation it has just produced
// (slim.conv2d(net, num_classes, 1, activation_fn=None), NetworksV2/UNet.py:100): the last normalised layer feeds
// only that conv, so its 128 bytes per pixel need not be read back. Same arithmetic and summation order as
// head_fprop_kernel (small_conv.cu): bf16-rounded activations, 8 channels per lane in ascending order, xor-shuffle
// over the lanes of a pixel, + bias -- the logits are bit-identical to the two-pass path.
// Registers: the per-channel parameters (scale, shift, COUT filter taps) sit in shared memory, one conflict-free
// strip per 8-channel lane, and are fetched per channel pair (3 x LDS.128 serve 4 pixels), so a thread holds only
// 4 packed pixels + 4 x COUT accumulators: 4 blocks of 256 threads per SM instead of 2 (91 registers before).
template <int COUT>
struct HeadSmem {
  static constexpr int PAIR = 4 + ((2 * COUT + 3) / 4) * 4;   // [sc0 sc1 sh0 sh1][w0[COUT] w1[COUT] pad]
  static constexpr int LANE = 4 * PAIR + 4;                   // +4 floats: strips of the 8 lanes hit distinct banks
};
template <int COUT, int UNR, int MINB>
__global__ void __launch_bounds__(256, MINB)
norm_apply_head_kernel(const __nv_bfloat16* __restrict__ y, int y_ld, __nv_bfloat16* __restrict__ a,
                       int a_ld, long long pixels_per_group, int c, int relu,
                       const float* __restrict__ scale, const float* __restrict__ shift, int gstride,
                       const float* __restrict__ wh, const float* __restrict__ bh,
                       float* __restrict__ logits) {
  bsl::pdl_wait();
  using HS = HeadSmem<COUT>;
  __shared__ __align__(16) float s_par[32 * HS::LANE];
  const int cg = c / 8;                    // power of two <= 32: the lanes of a pixel sit in one warp
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  const int ch0 = g * 8;
  for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
    float* q = s_par + (ch >> 3) * HS::LANE + ((ch & 7) >> 1) * HS::PAIR;
    const int odd = ch & 1;
    q[odd] = scale[blockIdx.y * gstride + ch];
    q[2 + odd] = shift[blockIdx.y * gstride + ch];
#pragma unroll
    for (int k = 0; k < COUT; ++k) q[4 + odd * COUT + k] = wh[ch * COUT + k];
  }
  __syncthreads();
  const float* par = s_par + g * HS::LANE;
  const long long base = (long long)blockIdx.y * pixels_per_group;
  const long long stride = (long long)gridDim.x * rows;
  // block-uniform loop (every lane takes part in the shuffles); lanes past the end are masked
  for (long long pb = (long long)blockIdx.x * rows; pb < pixels_per_group; pb += UNR * stride) {
    uint32_t raw[UNR][4];
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const long long p = pb + u * stride + r;
      const uint4 t = p < pixels_per_group ? ld16(y + (base + p) * y_ld + ch0) : make_uint4(0, 0, 0, 0);
      raw[u][0] = t.x, raw[u][1] = t.y, raw[u][2] = t.z, raw[u][3] = t.w;
    }
    float acc[UNR][COUT];
#pragma unroll
    for (int u = 0; u < UNR; ++u)
#pragma unroll
      for (int k = 0; k < COUT; ++k) acc[u][k] = 0.f;
#pragma unroll
    for (int pr = 0; pr < 4; ++pr) {       // channel pairs in ascending order: the summation order of head_fprop_kernel
      float prm[HS::PAIR];
#pragma unroll
      for (int i = 0; i < HS::PAIR / 4; ++i) {
        const float4 t = *reinterpret_cast<const float4*>(par + pr * HS::PAIR + 4 * i);
        prm[4 * i] = t.x, prm[4 * i + 1] = t.y, prm[4 * i + 2] = t.z, prm[4 * i + 3] = t.w;
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const uint32_t w = raw[u][pr];                           // bf16 pair: low half = even channel
        float z0 = fmaf(__uint_as_float(w << 16), prm[0], prm[2]);
        float z1 = fmaf(__uint_as_float(w & 0xffff0000u), prm[1], prm[3]);
        if (relu) {
          z0 = fmaxf(z0, 0.f);
          z1 = fmaxf(z1, 0.f);
        }
        const __nv_bfloat162 hb = __floats2bfloat162_rn(z0, z1);
        uint32_t o;
        memcpy(&o, &hb, 4);
        raw[u][pr] = o;
        const float v0 = __uint_as_float(o << 16), v1 = __uint_as_float(o & 0xffff0000u);   // what the logits layer reads
#pragma unroll
        for (int k = 0; k < COUT; ++k) acc[u][k] = fmaf(v0, prm[4 + k], acc[u][k]);
#pragma unroll
        for (int k = 0; k < COUT; ++k) acc[u][k] = fmaf(v1, prm[4 + COUT + k], acc[u][k]);
      }
    }
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const long long p = pb + u * stride + r;
      const bool valid = p < pixels_per_group;
      if (valid) st16(a + (base + p) * a_ld + ch0, make_uint4(raw[u][0], raw[u][1], raw[u][2], raw[u][3]));
#pragma unroll
      for (int k = 0; k < COUT; ++k)
        for (int s = cg >> 1; s > 0; s >>= 1) acc[u][k] += __shfl_xor_sync(0xffffffffu, acc[u][k], s);
      if (valid && g == 0) {
#pragma unroll
        for (int k = 0; k < COUT; ++k) logits[(base + p) * COUT + k] = acc[u][k] + (bh ? bh[k] : 0.f);
      }
    }
  }
}

// Same as norm_apply_kernel, and also emits the 2x2/s2 max-pooled tensor from the same read.
// "pixels" here are pooled pixels of one sample (grid.y = sample).
template <int G>
__global__ void norm_apply_pool_kernel(const __nv_bfloat16* __restrict__ y, int y_ld, __nv_bfloat16* __restrict__ a,
                                       int a_ld, __nv_bfloat16* __restrict__ pooled, int p_ld, int h, int w, int c,
                                       int per_sample, int relu, const float* __restrict__ scale,
                                       const float* __restrict__ shift, const float* __restrict__ guide,
                                       const float* __restrict__ wsp, int wsp_ld) {
  bsl::pdl_wait();
  const int cg = c / 8, ho = h / 2, wo = w / 2;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  const int ch0 = g * 8;
  const int img = blockIdx.y;
  const int o = (per_sample ? img * c : 0) + ch0;
  float sc[8], sh[8], ws[G ? G : 1][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = scale[o + j];
    sh[j] = shift[o + j];
#pragma unroll
    for (int q = 0; q < G; ++q) ws[q][j] = wsp[q * wsp_ld + ch0 + j];
  }
  const long long in0 = (long long)img * h * w, out0 = (long long)img * ho * wo;
  for (int q = blockIdx.x * rows + r; q < ho * wo; q += gridDim.x * rows) {
    const int yo = q / wo, xo = q - yo * wo;
    long long pix[4];
    uint4 raw[4];
    float gm[4][G ? G : 1];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      pix[k] = in0 + (long long)(2 * yo + (k >> 1)) * w + (2 * xo + (k & 1));
      raw[k] = ld16(y + pix[k] * y_ld + ch0);
#pragma unroll
      for (int q = 0; q < G; ++q) gm[k][q] = __ldg(guide + pix[k] * G + q);
    }
    float mx[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) mx[j] = -INFINITY;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float v[8];
      unpack8(raw[k], v);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float z = fmaf(v[j], sc[j], sh[j]);
#pragma unroll
        for (int q = 0; q < G; ++q) z = fmaf(gm[k][q], ws[q][j], z);
        v[j] = relu ? fmaxf(z, 0.f) : z;
      }
      const uint4 packed = pack8(v);
      st16(a + pix[k] * a_ld + ch0, packed);
      float rr[8];
      unpack8(packed, rr);  // pool the bf16-rounded values: what the next layer actually sees
#pragma unroll
      for (int j = 0; j < 8; ++j) mx[j] = fmaxf(mx[j], rr[j]);
    }
    st16(pooled + (out0 + q) * p_ld + ch0, pack8(mx));
  }
}

// Block = 32 channels x 32 group lanes (instance norm: one group per sample): c1 / c2 per (group, channel) are
// independent; dgamma / dbeta sum over the groups through shared memory in ascending lane order (fixed order; identical
// to a serial loop when groups <= 32, and batch norm has a single group).
__global__ void __launch_bounds__(1024)
norm_bwd_finalize_kernel(int groups, int c, double m, const double* __restrict__ sums,
                         const float* __restrict__ rstd_unused, float* __restrict__ c1,
                         float* __restrict__ c2, float* __restrict__ dgamma,
                         float* __restrict__ dbeta) {
  bsl::pdl_wait();
  __shared__ double red[2][32][33];
  const int chl = threadIdx.x & 31, gl = threadIdx.x >> 5;
  const int ch = blockIdx.x * 32 + chl;
  double sg = 0.0, sb = 0.0;
  if (ch < c) {
    for (int g = gl; g < groups; g += (int)(blockDim.x >> 5)) {
      const double s0 = sums[(long long)g * 2 * c + ch];
      const double s1 = sums[(long long)g * 2 * c + c + ch];
      c1[g * c + ch] = (float)(s0 / m);
      c2[g * c + ch] = (float)(s1 / m);
      sb += s0;
      sg += s1;
    }
  }
  red[0][gl][chl] = sg;
  red[1][gl][chl] = sb;
  __syncthreads();
  if (gl == 0 && ch < c) {
    double tg = 0.0, tb = 0.0;
    const int lanes = blockDim.x >> 5;
    for (int j = 0; j < lanes; ++j) {
      tg += red[0][j][chl];
      tb += red[1][j][chl];
    }
    if (dgamma) dgamma[ch] = (float)tg;
    if (dbeta) dbeta[ch] = (float)tb;
  }
  (void)rstd_unused;
}

template <int G>
__global__ void norm_bwd_apply_kernel(const __nv_bfloat16* __restrict__ y, int y_ld,
                                      const __nv_bfloat16* __restrict__ da, int da_ld,
                                      __nv_bfloat16* __restrict__ dy, int dy_ld, long long pixels_per_group, int c,
                                      int relu, const float* __restrict__ mean, const float* __restrict__ rstd,
                                      const float* __restrict__ scale, const float* __restrict__ shift,
                                      const float* __restrict__ c1, const float* __restrict__ c2,
                                      const float* __restrict__ guide, const float* __restrict__ wsp, int wsp_ld,
                                      int gstride, int premul) {
  bsl::pdl_wait();
  const int cg = c / 8;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  const int ch0 = g * 8;
  const int o = blockIdx.y * gstride + ch0;
  // dy = scale*(dz - c1 - xhat*c2), xhat = (v - mean)*rstd  ==  scale*dz + k1*v + k0
  // premul (batch statistics with a per-sample scale, bsl_norm_bwd_finalize_bnmod): c1, c2 arrive multiplied by rstd
  // and already summed over the samples with their scales: dy = scale*dz - c1 - xhat*c2
  float sc[8], sh[8], k1[8], k0[8], ws[G ? G : 1][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = scale[o + j];
    sh[j] = shift[o + j];
#pragma unroll
    for (int q = 0; q < G; ++q) ws[q][j] = wsp[q * wsp_ld + ch0 + j];
    const float t = premul ? c2[o + j] * rstd[o + j] : sc[j] * c2[o + j] * rstd[o + j];
    k1[j] = -t;
    k0[j] = fmaf(t, mean[o + j], premul ? -c1[o + j] : -sc[j] * c1[o + j]);
  }
  const long long base = (long long)blockIdx.y * pixels_per_group;
  const long long stride = (long long)gridDim.x * rows;
  long long p = (long long)blockIdx.x * rows + r;
  constexpr int U = 4;
  for (; p + (U - 1) * stride < pixels_per_group; p += U * stride) {
    uint4 ry[U], rg[U];
    float gm[U][G ? G : 1];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      ry[u] = ld16(y + (base + p + u * stride) * y_ld + ch0);
      rg[u] = ld16(da + (base + p + u * stride) * da_ld + ch0);
#pragma unroll
      for (int q = 0; q < G; ++q) gm[u][q] = __ldg(guide + (base + p + u * stride) * G + q);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float v[8], gg[8];
      unpack8(ry[u], v);
      unpack8(rg[u], gg);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float z = fmaf(v[j], sc[j], sh[j]);
#pragma unroll
        for (int q = 0; q < G; ++q) z = fmaf(gm[u][q], ws[q][j], z);
        const float dz = (!relu || z > 0.f) ? gg[j] : 0.f;
        v[j] = fmaf(sc[j], dz, fmaf(k1[j], v[j], k0[j]));
      }
      st16(dy + (base + p + u * stride) * dy_ld + ch0, pack8(v));
    }
  }
  for (; p < pixels_per_group; p += stride) {
    float v[8], gg[8];
    unpack8(ld16(y + (base + p) * y_ld + ch0), v);
    unpack8(ld16(da + (base + p) * da_ld + ch0), gg);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float z = fmaf(v[j], sc[j], sh[j]);
#pragma unroll
      for (int q = 0; q < G; ++q) z = fmaf(__ldg(guide + (base + p) * G + q), ws[q][j], z);
      const float dz = (!relu || z > 0.f) ? gg[j] : 0.f;
      v[j] = fmaf(sc[j], dz, fmaf(k1[j], v[j], k0[j]));
    }
    st16(dy + (base + p) * dy_ld + ch0, pack8(v));
  }
}

// GUNet density modulation folded into the per-(sample, channel) affine of an instance-norm layer
// (conditional_normalization, NetworksV2/GUNet.py:119-133,193-204): z*gm + bias_sp == y*(sc*gm) + (sh*gm + bias_sp).
__global__ void norm_modulate_kernel(int n, int c, const float* __restrict__ gamma_mod, int gm_ld,
                                     const float* __restrict__ sp_bias, float* __restrict__ scale,
                                     float* __restrict__ shift) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * c) return;
  const int s = i / c, ch = i - s * c;
  const float gm = gamma_mod ? gamma_mod[(long long)s * gm_ld + ch] : 1.f;
  scale[i] *= gm;
  shift[i] = fmaf(shift[i], gm, sp_bias ? sp_bias[ch] : 0.f);
}

// Backward scalars of a modulated instance-norm layer. sums[n][K][c]: S0 = sum dz, S1 = sum dz*xhat, T_g = sum dz*guide_g.
// Block = 32 channels x FM_S sample lanes: the per-sample outputs are independent; the sums over samples are combined
// through shared memory in ascending sample-lane order (fixed order: bit-reproducible; identical to a serial loop over
// the samples when n <= FM_S). One thread per channel walking all n samples took 57 us per launch at batch 32.
constexpr int FM_S = 32;
__global__ void __launch_bounds__(32 * FM_S)
norm_bwd_finalize_mod_kernel(int n, int c, int K, double m, const double* __restrict__ sums,
                             const float* __restrict__ gamma_mod, int gm_ld,
                             const float* __restrict__ gamma, const float* __restrict__ beta,
                             float* __restrict__ c1, float* __restrict__ c2, float* __restrict__ dgamma,
                             float* __restrict__ dbeta, float* __restrict__ dgamma_mod,
                             float* __restrict__ dw_guide, int dw_ld, float* __restrict__ dbias_guide) {
  bsl::pdl_wait();
  __shared__ double red[5][FM_S][33];
  const int chl = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int ch = blockIdx.x * 32 + chl;
  double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};   // sg, sb, s0all, t0, t1
  if (ch < c) {
    const double ga = gamma ? (double)gamma[ch] : 1.0, be = beta ? (double)beta[ch] : 0.0;
    for (int s = sl; s < n; s += FM_S) {
      const double* q = sums + (long long)s * K * c + ch;
      const double s0 = q[0], s1 = q[c];
      c1[s * c + ch] = (float)(s0 / m);
      c2[s * c + ch] = (float)(s1 / m);
      const double gm = gamma_mod ? (double)gamma_mod[(long long)s * gm_ld + ch] : 1.0;
      if (dgamma_mod) dgamma_mod[(long long)s * gm_ld + ch] = (float)(ga * s1 + be * s0);
      acc[0] += gm * s1;
      acc[1] += gm * s0;
      acc[2] += s0;
      for (int g = 0; g < K - 2; ++g) acc[3 + g] += q[(long long)(2 + g) * c];
    }
  }
#pragma unroll
  for (int k = 0; k < 5; ++k) red[k][sl][chl] = acc[k];
  __syncthreads();
  if (sl == 0 && ch < c) {
    double tot[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int j = 0; j < FM_S; ++j)
#pragma unroll
      for (int k = 0; k < 5; ++k) tot[k] += red[k][j][chl];
    if (dgamma) dgamma[ch] = (float)tot[0];
    if (dbeta) dbeta[ch] = (float)tot[1];
    for (int g = 0; g < K - 2; ++g) dw_guide[g * dw_ld + ch] = (float)tot[3 + g];
    if (dbias_guide) dbias_guide[ch] = (float)tot[2];
  }
}

// after_affine fold (GUNet.py:213-214): z = ga*(y*sc + sh + guide.w) + ba = y*(sc*ga) + (sh*ga + ba) + guide.(w*ga)
__global__ void norm_affine_fold_kernel(int n, int c, int G, const float* __restrict__ ga, const float* __restrict__ ba,
                                        float* __restrict__ scale, float* __restrict__ shift,
                                        float* __restrict__ scale_pre, float* __restrict__ shift_pre,
                                        const float* __restrict__ w, int w_ld, float* __restrict__ w_eff) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n * c) {
    const int ch = i % c;
    const float sc = scale[i], sh = shift[i];
    scale_pre[i] = sc;
    shift_pre[i] = sh;
    scale[i] = sc * ga[ch];
    shift[i] = fmaf(sh, ga[ch], ba[ch]);
  }
  if (i < G * c) {
    const int g = i / c, ch = i - g * c;
    w_eff[i] = w[g * w_ld + ch] * ga[ch];
  }
}

// norm_bwd_finalize_mod_kernel with the folded channel-wise affine. S0 = sum dz, S1 = sum dz*xhat, T_g = sum dz*guide_g
// are sums of the gradient AFTER the affine, one row per group (a sample, or the whole batch in mode 0);
// u = xhat*(scale_pre/rstd) + (shift_pre + mean*scale_pre) + guide.w. `jac` selects what c1 / c2 hold:
//   BSL_NORM_JAC_GROUP   c1 = S0/m, c2 = S1/m per group (instance norm; batch norm on its single group)
//   BSL_NORM_JAC_BATCH   the per-sample view of a batch-norm layer: c1r = rstd*gamma*ga*sum_n gm[n]*S0_n / m,
//                        c2r likewise with S1 (m = n*hw), the same value for every sample (bsl_norm_bwd_apply_bnmod)
//   BSL_NORM_JAC_NONE    identity normaliser: c1 = c2 = 0
__global__ void norm_bwd_finalize_affine_kernel(int n, int c, int K, double m, int jac, const double* __restrict__ sums,
                                                const float* __restrict__ gamma_mod, int gm_ld,
                                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                                const float* __restrict__ ga, const float* __restrict__ mean,
                                                const float* __restrict__ rstd, const float* __restrict__ scale_pre,
                                                const float* __restrict__ shift_pre, const float* __restrict__ w,
                                                int w_ld, float* __restrict__ c1, float* __restrict__ c2,
                                                float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                float* __restrict__ dgamma_mod, float* __restrict__ dw_guide, int dw_ld,
                                                float* __restrict__ dbias_guide, float* __restrict__ dga,
                                                float* __restrict__ dba) {
  bsl::pdl_wait();
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  const double gam = gamma ? (double)gamma[ch] : 1.0, be = beta ? (double)beta[ch] : 0.0, a = (double)ga[ch];
  double sg = 0.0, sb = 0.0, s0all = 0.0, t[2] = {0.0, 0.0}, acc_ga = 0.0;
  for (int s = 0; s < n; ++s) {  // fixed order
    const double* q = sums + (long long)s * K * c + ch;
    const double s0 = q[0], s1 = q[c];
    const int o = s * c + ch;
    if (jac != BSL_NORM_JAC_BATCH) {
      c1[o] = jac == BSL_NORM_JAC_GROUP ? (float)(s0 / m) : 0.f;
      c2[o] = jac == BSL_NORM_JAC_GROUP ? (float)(s1 / m) : 0.f;
    }
    const double sp = (double)scale_pre[o], hp = (double)shift_pre[o];
    double du = sp / (double)rstd[o] * s1 + (hp + (double)mean[o] * sp) * s0;
    for (int g = 0; g < K - 2; ++g) du += (double)w[g * w_ld + ch] * q[(long long)(2 + g) * c];
    acc_ga += du;
    const double gm = gamma_mod ? (double)gamma_mod[(long long)s * gm_ld + ch] : 1.0;
    if (dgamma_mod) dgamma_mod[(long long)s * gm_ld + ch] = (float)(a * (gam * s1 + be * s0));
    sg += gm * s1;
    sb += gm * s0;
    s0all += s0;
    for (int g = 0; g < K - 2; ++g) t[g] += q[(long long)(2 + g) * c];
  }
  if (jac == BSL_NORM_JAC_BATCH) {
    const double r = (double)rstd[ch] * gam * a / m;
    const float k1 = (float)(r * sb), k2 = (float)(r * sg);
    for (int s = 0; s < n; ++s) {
      c1[s * c + ch] = k1;
      c2[s * c + ch] = k2;
    }
  }
  if (dgamma) dgamma[ch] = (float)(a * sg);
  if (dbeta) dbeta[ch] = (float)(a * sb);
  for (int g = 0; g < K - 2; ++g) dw_guide[g * dw_ld + ch] = (float)(a * t[g]);
  if (dbias_guide) dbias_guide[ch] = (float)(a * s0all);
  dga[ch] = (float)acc_ga;
  dba[ch] = (float)s0all;
}

// Batch-norm layer with per-sample modulation (GUNet --normalizer batch_norm, GUNet.py:301,321-325): bsl_norm_finalize
// (batch mode) left mean / rstd / scale / shift of the BATCH statistics in the first c entries; expand them to the
// per-(sample, channel) arrays the instance-mode passes index, folding gamma_mod and the guide-conv bias in:
//   z = (y*sc + sh) * gm[n] + b_sp  ==  y * (sc*gm[n]) + (sh*gm[n] + b_sp)
__global__ void norm_modulate_bn_kernel(int n, int c, const float* __restrict__ gamma_mod, int gm_ld,
                                        const float* __restrict__ sp_bias, float* __restrict__ mean,
                                        float* __restrict__ rstd, float* __restrict__ scale, float* __restrict__ shift) {
  bsl::pdl_wait();
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  const float mu = mean[ch], rs = rstd[ch], sc = scale[ch], sh = shift[ch], b = sp_bias ? sp_bias[ch] : 0.f;
  for (int s = n - 1; s >= 0; --s) {     // entry [0][ch] (the input) is overwritten last
    const float gm = gamma_mod ? gamma_mod[(long long)s * gm_ld + ch] : 1.f;
    mean[s * c + ch] = mu;
    rstd[s * c + ch] = rs;
    scale[s * c + ch] = sc * gm;
    shift[s * c + ch] = fmaf(sh, gm, b);
  }
}

// Backward scalars of such a layer from the per-sample sums S0 = sum dz, S1 = sum dz*xhat, T_g = sum dz*guide_g:
// dxhat = dz * s_n with s_n = gamma * gm[n], so FusedBatchNormGrad's two means run over ALL samples weighted by s_n:
//   dy = rstd * (s_n*dz - C1 - xhat*C2),  C1 = sum_n s_n*S0_n / M,  C2 = sum_n s_n*S1_n / M,  M = n * hw.
// c1r / c2r (per (sample, channel), equal for all samples) = rstd*C1, rstd*C2 for bsl_norm_bwd_apply_bnmod.
__global__ void norm_bwd_finalize_bnmod_kernel(int n, int c, int K, double m_all, const double* __restrict__ sums,
                                               const float* __restrict__ gamma_mod, int gm_ld,
                                               const float* __restrict__ gamma, const float* __restrict__ beta,
                                               const float* __restrict__ rstd, float* __restrict__ c1r,
                                               float* __restrict__ c2r, float* __restrict__ dgamma,
                                               float* __restrict__ dbeta, float* __restrict__ dgamma_mod,
                                               float* __restrict__ dw_guide, int dw_ld, float* __restrict__ dbias_guide) {
  bsl::pdl_wait();
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  const double ga = gamma ? (double)gamma[ch] : 1.0, be = beta ? (double)beta[ch] : 0.0;
  double sg = 0.0, sb = 0.0, s0all = 0.0, t[2] = {0.0, 0.0};
  for (int s = 0; s < n; ++s) {  // fixed order
    const double* q = sums + (long long)s * K * c + ch;
    const double s0 = q[0], s1 = q[c];
    const double gm = gamma_mod ? (double)gamma_mod[(long long)s * gm_ld + ch] : 1.0;
    if (dgamma_mod) dgamma_mod[(long long)s * gm_ld + ch] = (float)(ga * s1 + be * s0);
    sg += gm * s1;
    sb += gm * s0;
    s0all += s0;
    for (int g = 0; g < K - 2; ++g) t[g] += q[(long long)(2 + g) * c];
  }
  const double r = (double)rstd[ch];
  const float k1 = (float)(r * ga * sb / m_all), k2 = (float)(r * ga * sg / m_all);
  for (int s = 0; s < n; ++s) {
    c1r[s * c + ch] = k1;
    c2r[s * c + ch] = k2;
  }
  if (dgamma) dgamma[ch] = (float)sg;
  if (dbeta) dbeta[ch] = (float)sb;
  for (int g = 0; g < K - 2; ++g) dw_guide[g * dw_ld + ch] = (float)t[g];
  if (dbias_guide) dbias_guide[ch] = (float)s0all;
}

// da[n,2i+a,2j+b,:] = dskip (optional) + (first max of the window in scan order ? dpool[n,i,j,:] : 0)
__global__ void maxpool_bwd_add_kernel(const __nv_bfloat16* __restrict__ act, int a_ld,
                                       const __nv_bfloat16* __restrict__ dpool, int p_ld,
                                       const __nv_bfloat16* __restrict__ dskip, int s_ld,
                                       __nv_bfloat16* __restrict__ out, int o_ld, int n, int h, int w, int c) {
  bsl::pdl_wait();
  const int cg = c / 8, ho = h / 2, wo = w / 2;
  const long long total = (long long)n * ho * wo * cg;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int ch0 = (int)(t % cg) * 8; t /= cg;
    const int xo = (int)(t % wo); t /= wo;
    const int yo = (int)(t % ho);
    const int img = (int)(t / ho);
    float v[4][8], g[8];
    long long pix[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      pix[k] = ((long long)img * h + (2 * yo + (k >> 1))) * w + (2 * xo + (k & 1));
      unpack8(ld16(act + pix[k] * a_ld + ch0), v[k]);
    }
    unpack8(ld16(dpool + (((long long)img * ho + yo) * wo + xo) * p_ld + ch0), g);
    int arg[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int best = 0;
      float bv = v[0][j];
#pragma unroll
      for (int k = 1; k < 4; ++k)
        if (v[k][j] > bv) { bv = v[k][j]; best = k; }  // strict '>' keeps the FIRST maximum
      arg[j] = best;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float o[8];
      if (dskip) unpack8(ld16(dskip + pix[k] * s_ld + ch0), o);
      else {
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] += (arg[j] == k) ? g[j] : 0.f;
      st16(out + pix[k] * o_ld + ch0, pack8(o));
    }
  }
}

// y[n,i,j,:] = max of the 2x2 window x[n,2i..2i+1,2j..2j+1,:] (--without_norm encoder blocks: the pooled half of what
// bsl_norm_apply_pool writes), 8 channels per thread; the comparison is the one maxpool_bwd_add_kernel makes.
__global__ void maxpool2x2_bf16_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, __nv_bfloat16* __restrict__ y, int y_ld,
                                       int n, int h, int w, int c) {
  bsl::pdl_wait();
  const int cg = c / 8, ho = h / 2, wo = w / 2;
  const long long total = (long long)n * ho * wo * cg;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int ch0 = (int)(t % cg) * 8; t /= cg;
    const int xo = (int)(t % wo); t /= wo;
    const int yo = (int)(t % ho);
    const int img = (int)(t / ho);
    uint4 r[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      r[k] = ld16(x + (((long long)img * h + (2 * yo + (k >> 1))) * w + (2 * xo + (k & 1))) * x_ld + ch0);
    float m[8];
    unpack8(r[0], m);
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      float v[8];
      unpack8(r[k], v);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (v[j] > m[j]) m[j] = v[j];
    }
    st16(y + (((long long)img * ho + yo) * wo + xo) * y_ld + ch0, pack8(m));
  }
}

__global__ void relu_bwd_kernel(const __nv_bfloat16* __restrict__ y, int y_ld, const __nv_bfloat16* __restrict__ dy,
                                int dy_ld, __nv_bfloat16* __restrict__ out, int o_ld, long long pixels, int c) {
  bsl::pdl_wait();
  const int cg = c / 8;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  if (r >= rows) return;
  const int ch0 = g * 8;
  const long long stride = (long long)gridDim.x * rows;
  long long p = (long long)blockIdx.x * rows + r;
  for (; p + (EW_UNROLL - 1) * stride < pixels; p += EW_UNROLL * stride) {
    uint4 ry[EW_UNROLL], rg[EW_UNROLL];
#pragma unroll
    for (int u = 0; u < EW_UNROLL; ++u) {
      ry[u] = ld16(y + (p + u * stride) * y_ld + ch0);
      rg[u] = ld16(dy + (p + u * stride) * dy_ld + ch0);
    }
#pragma unroll
    for (int u = 0; u < EW_UNROLL; ++u) {
      float v[8], gg[8];
      unpack8(ry[u], v);
      unpack8(rg[u], gg);
#pragma unroll
      for (int j = 0; j < 8; ++j) gg[j] = v[j] > 0.f ? gg[j] : 0.f;
      st16(out + (p + u * stride) * o_ld + ch0, pack8(gg));
    }
  }
  for (; p < pixels; p += stride) {
    float v[8], gg[8];
    unpack8(ld16(y + p * y_ld + ch0), v);
    unpack8(ld16(dy + p * dy_ld + ch0), gg);
#pragma unroll
    for (int j = 0; j < 8; ++j) gg[j] = v[j] > 0.f ? gg[j] : 0.f;
    st16(out + p * o_ld + ch0, pack8(gg));
  }
}

__global__ void add_bf16_kernel(const __nv_bfloat16* __restrict__ a, int a_ld, const __nv_bfloat16* __restrict__ b,
                                int b_ld, __nv_bfloat16* __restrict__ out, int o_ld, long long pixels, int c) {
  bsl::pdl_wait();
  const int cg = c / 8;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  if (r >= rows) return;
  const int ch0 = g * 8;
  const long long stride = (long long)gridDim.x * rows;
  for (long long p = (long long)blockIdx.x * rows + r; p < pixels; p += stride) {
    float u[8], v[8];
    unpack8(ld16(a + p * a_ld + ch0), u);
    unpack8(ld16(b + p * b_ld + ch0), v);
#pragma unroll
    for (int j = 0; j < 8; ++j) u[j] += v[j];
    st16(out + p * o_ld + ch0, pack8(u));
  }
}

// Launch shape for the (rows x channel-group) elementwise kernels.
struct EwPlan {
  int threads, rows;
  unsigned blocks;
};
EwPlan ew_plan(bsl_ctx* ctx, long long pixels_per_group, int groups, int c, int unroll) {
  EwPlan p;
  const int cg = c / 8;
  p.threads = cg > 256 ? cg : 256;
  p.rows = p.threads / cg;
  p.threads = p.rows * cg;
  long long want = (pixels_per_group + (long long)p.rows * unroll - 1) / ((long long)p.rows * unroll);
  long long cap = (16LL * ctx->sm_count + groups - 1) / groups;
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  p.blocks = (unsigned)want;
  return p;
}

unsigned ew_grid(bsl_ctx* ctx, long long items) {
  long long b = (items + 255) / 256;
  const long long cap = 16LL * ctx->sm_count;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

int check_norm(bsl_ctx* ctx, const bsl_norm_desc* d) {
  if (!ctx) return BSL_EINVAL;
  if (!d) return bsl_fail(ctx, BSL_EINVAL, "norm: null descriptor");
  if (d->mode != 0 && d->mode != 1) return bsl_fail(ctx, BSL_EINVAL, "norm: mode %d", d->mode);
  if (d->n <= 0 || d->hw <= 0 || d->c <= 0 || d->c % 8)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "norm: n=%d hw=%d c=%d (c must be a multiple of 8)", d->n, d->hw, d->c);
  if (d->x_ld < d->c || d->y_ld < d->c || d->x_ld % 8 || d->y_ld % 8)
    return bsl_fail(ctx, BSL_EINVAL, "norm: bad channel strides");
  return BSL_OK;
}

}  // namespace

int bsl_stats_bf16(bsl_ctx* ctx, const void* x, long long pixels_per_group, int groups, int c, int ld, double* sums,
                   cudaStream_t stream) {
  StatsF f{reinterpret_cast<const __nv_bfloat16*>(x), ld};
  return run_pixel_reduce(ctx, f, pixels_per_group, groups, c, sums, stream);
}

extern "C" {

int bsl_norm_stats(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, double* sums, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!x || !sums) return bsl_fail(ctx, BSL_EINVAL, "norm_stats: null buffer");
  StatsF f{reinterpret_cast<const __nv_bfloat16*>(x), d->x_ld};
  const int groups = d->mode ? d->n : 1;
  const long long ppg = d->mode ? d->hw : (long long)d->n * d->hw;
  return run_pixel_reduce(ctx, f, ppg, groups, d->c, sums, as_stream(stream));
}

int bsl_norm_finalize(bsl_ctx* ctx, const bsl_norm_desc* d, int is_training, const double* sums,
                      const float* gamma, const float* beta, float* moving_mean, float* moving_var,
                      float* mean, float* rstd, float* scale, float* shift, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  const int groups = d->mode ? d->n : 1;
  const int bn = d->mode == 0;
  const int use_moving = bn && !is_training;
  if ((!use_moving && !sums) || !mean || !rstd || !scale || !shift || (d->scale && !gamma) || (d->center && !beta))
    return bsl_fail(ctx, BSL_EINVAL, "norm_finalize: null buffer");
  if (bn && (!moving_mean || !moving_var)) return bsl_fail(ctx, BSL_EINVAL, "norm_finalize: moving stats required");
  const double m = d->mode ? (double)d->hw : (double)d->n * d->hw;
  const int total = groups * d->c;
  bsl_launch(norm_finalize_kernel, dim3((total + 127) / 128), dim3(128), 0, as_stream(stream), 
      groups, d->c, m, d->eps, d->decay, bn && is_training, use_moving, d->center, d->scale, sums, gamma, beta,
      moving_mean, moving_var, mean, rstd, scale, shift);
  BSL_LAUNCH_CHECK(ctx, "norm_finalize_kernel");
  return BSL_OK;
}

static int check_guide(bsl_ctx* ctx, const bsl_norm_desc* d, const bsl_guide* g, int* G) {
  *G = 0;
  if (!g || !g->map) return BSL_OK;
  if (d->mode != 1) return bsl_fail(ctx, BSL_EUNSUPPORTED, "guide modulation is implemented for instance_norm layers");
  if (g->channels < 1 || g->channels > 2 || !g->w || g->w_ld < d->c)
    return bsl_fail(ctx, BSL_EINVAL, "guide: channels=%d (1 or 2), w_ld=%d >= c", g->channels, g->w_ld);
  *G = g->channels;
  return BSL_OK;
}

int bsl_norm_apply_mod(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const float* scale, const float* shift,
                       const bsl_guide* guide, void* y, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!x || !scale || !shift || !y) return bsl_fail(ctx, BSL_EINVAL, "norm_apply: null buffer");
  int G;
  if ((rc = check_guide(ctx, d, guide, &G))) return rc;
  const int groups = d->mode ? d->n : 1;
  const long long ppg = d->mode ? d->hw : (long long)d->n * d->hw;
  const EwPlan pl = ew_plan(ctx, ppg, groups, d->c, EW_UNROLL);
  const int gstride = d->mode ? d->c : 0;
  const dim3 grid(pl.blocks, groups);
  auto xb = reinterpret_cast<const __nv_bfloat16*>(x);
  auto yb = reinterpret_cast<__nv_bfloat16*>(y);
  cudaStream_t s = as_stream(stream);
  if (G == 0)
    bsl_launch(norm_apply_kernel<0>, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, yb, d->y_ld, ppg, d->c, d->relu, scale, shift,
                                                     nullptr, nullptr, 0, gstride);
  else if (G == 1)
    bsl_launch(norm_apply_kernel<1>, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, yb, d->y_ld, ppg, d->c, d->relu, scale, shift,
                                                     guide->map, guide->w, guide->w_ld, gstride);
  else
    bsl_launch(norm_apply_kernel<2>, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, yb, d->y_ld, ppg, d->c, d->relu, scale, shift,
                                                     guide->map, guide->w, guide->w_ld, gstride);
  BSL_LAUNCH_CHECK(ctx, "norm_apply_kernel");
  return BSL_OK;
}

int bsl_norm_apply_head(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const float* scale, const float* shift,
                        void* y, const float* w_head, const float* b_head, int classes, float* logits, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!x || !scale || !shift || !y || !w_head || !logits) return bsl_fail(ctx, BSL_EINVAL, "norm_apply_head: null buffer");
  const int cg = d->c / 8;
  if (cg > 32 || (cg & (cg - 1)) || classes < 2 || classes > 4)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "norm_apply_head: c=%d in {8,..,256}, classes=%d in 2..4", d->c, classes);
  const int groups = d->mode ? d->n : 1;
  const long long ppg = d->mode ? d->hw : (long long)d->n * d->hw;
  const EwPlan pl = ew_plan(ctx, ppg, groups, d->c, EW_UNROLL);
  const dim3 grid(pl.blocks, groups);
  auto xb = reinterpret_cast<const __nv_bfloat16*>(x);
  auto yb = reinterpret_cast<__nv_bfloat16*>(y);
  cudaStream_t s = as_stream(stream);
  const int gstride = d->mode ? d->c : 0;
  auto go = [&](auto kern) {
    bsl_launch(kern, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, yb, d->y_ld, ppg, d->c, d->relu, scale, shift,
               gstride, w_head, b_head, logits);
  };
  // 2 pixels per thread and iteration, 4 blocks per SM: 0.384 -> 0.310 ms at cfg2 (4 pixels x 3 blocks: 0.329 ms)
  switch (classes) {
    case 2: go(norm_apply_head_kernel<2, 2, 4>); break;
    case 3: go(norm_apply_head_kernel<3, 2, 4>); break;
    default: go(norm_apply_head_kernel<4, 2, 4>); break;
  }
  BSL_LAUNCH_CHECK(ctx, "norm_apply_head_kernel");
  return BSL_OK;
}

int bsl_norm_apply(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const float* scale, const float* shift,
                   void* y, void* stream) {
  return bsl_norm_apply_mod(ctx, d, x, scale, shift, nullptr, y, stream);
}

int bsl_norm_apply_pool_mod(bsl_ctx* ctx, const bsl_norm_desc* d, int h, int w, const void* x, const float* scale,
                            const float* shift, const bsl_guide* guide, void* y, void* pooled, int pooled_ld,
                            void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!x || !scale || !shift || !y || !pooled) return bsl_fail(ctx, BSL_EINVAL, "norm_apply_pool: null buffer");
  if (h * w != d->hw || (h & 1) || (w & 1) || pooled_ld < d->c || pooled_ld % 8)
    return bsl_fail(ctx, BSL_EINVAL, "norm_apply_pool: h=%d w=%d must be even and match hw=%d", h, w, d->hw);
  int G;
  if ((rc = check_guide(ctx, d, guide, &G))) return rc;
  const EwPlan pl = ew_plan(ctx, (long long)(h / 2) * (w / 2), d->n, d->c, 1);
  const dim3 grid(pl.blocks, d->n);
  auto xb = reinterpret_cast<const __nv_bfloat16*>(x);
  auto yb = reinterpret_cast<__nv_bfloat16*>(y);
  auto pb = reinterpret_cast<__nv_bfloat16*>(pooled);
  cudaStream_t s = as_stream(stream);
  if (G == 0)
    bsl_launch(norm_apply_pool_kernel<0>, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, yb, d->y_ld, pb, pooled_ld, h, w, d->c, d->mode,
                                                          d->relu, scale, shift, nullptr, nullptr, 0);
  else if (G == 1)
    bsl_launch(norm_apply_pool_kernel<1>, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, yb, d->y_ld, pb, pooled_ld, h, w, d->c, d->mode,
                                                          d->relu, scale, shift, guide->map, guide->w, guide->w_ld);
  else
    bsl_launch(norm_apply_pool_kernel<2>, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, yb, d->y_ld, pb, pooled_ld, h, w, d->c, d->mode,
                                                          d->relu, scale, shift, guide->map, guide->w, guide->w_ld);
  BSL_LAUNCH_CHECK(ctx, "norm_apply_pool_kernel");
  return BSL_OK;
}

int bsl_norm_apply_pool(bsl_ctx* ctx, const bsl_norm_desc* d, int h, int w, const void* x, const float* scale,
                        const float* shift, void* y, void* pooled, int pooled_ld, void* stream) {
  return bsl_norm_apply_pool_mod(ctx, d, h, w, x, scale, shift, nullptr, y, pooled, pooled_ld, stream);
}

}  // extern "C"

namespace {
// The un-guided backward sums with 4 channels (8 bytes per tensor) per thread instead of 8: the 16-byte version
// needs 126 registers (512 threads per SM) and reads at 4.1-4.8 TB/s; a read-only stream reaches 7.1 TB/s
// (profiles/r01_hbm_read_probe.log). Same partial layout as pixel_reduce_kernel with K = 2 ([group][block][2][c]),
// finished by pixel_reduce_final_kernel in block order: deterministic, no atomics.
// HEAD > 0 (last normalised layer, followed only by the 1x1 logits conv with HEAD classes): the gradient w.r.t. the
// activation is not read from memory but recomputed per pixel from the HEAD fp32 logit gradients,
//   da[ch] = bf16(sum_k dl[k] * w_head[ch][k])    (same FMA order and rounding as head_dgrad_kernel, small_conv.cu),
// so Conv2DBackpropInput of the logits layer never writes its 128 bytes per pixel and the two backward passes of
// this layer read 12 instead of 128 bytes per pixel for it. Bit-identical to the three-kernel path.
template <int HEAD>
__device__ __forceinline__ uint2 head_grad4(const float (&dl)[HEAD ? HEAD : 1], const float (&wq)[4][HEAD ? HEAD : 1]) {
  float s[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    s[j] = 0.f;
#pragma unroll
    for (int k = 0; k < HEAD; ++k) s[j] = fmaf(dl[k], wq[j][k], s[j]);
  }
  uint2 out;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&out);
  h[0] = __floats2bfloat162_rn(s[0], s[1]);
  h[1] = __floats2bfloat162_rn(s[2], s[3]);
  return out;
}

template <int U, int HEAD>
__global__ void __launch_bounds__(256, 4)
norm_bwd_reduce4_kernel(const __nv_bfloat16* __restrict__ y, int y_ld, const __nv_bfloat16* __restrict__ da, int da_ld,
                        const float* __restrict__ mean, const float* __restrict__ rstd,
                        const float* __restrict__ scale, const float* __restrict__ shift, int c, int relu,
                        long long pixels_per_group, long long ppb, float* __restrict__ part,
                        const float* __restrict__ dl, const float* __restrict__ wh) {
  bsl::pdl_wait();
  extern __shared__ float sm[];   // [rows][2][c]
  constexpr int HK = HEAD ? HEAD : 1;
  const int cg = c / 4;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  const int group = blockIdx.y;
  const int ch0 = g * 4;
  float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
  // filter of the logits layer in shared memory, re-read per batch of U pixels (volatile: kept out of registers,
  // the kernel stays at 4 resident blocks per SM)
  __shared__ float s_wh[HEAD ? 256 * HK : 1];
  if (HEAD) {
    for (int i = threadIdx.x; i < c * HK; i += blockDim.x) s_wh[i] = wh[i];
    __syncthreads();
  }
  const volatile float* wv = s_wh + ch0 * HK;
  if (r < rows) {
    float sc[4], sh[4], rs[4], mr[4];
    const int o = group * c + ch0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      sc[j] = scale[o + j];
      sh[j] = shift[o + j];
      rs[j] = rstd[o + j];
      mr[j] = mean[o + j] * rstd[o + j];
    }
    const long long p0 = blockIdx.x * ppb, p1 = min(pixels_per_group, p0 + ppb);
    const long long base = (long long)group * pixels_per_group;
    auto one = [&](const uint2& ry, const uint2& rd) {
      const __nv_bfloat162* hy = reinterpret_cast<const __nv_bfloat162*>(&ry);
      const __nv_bfloat162* hd = reinterpret_cast<const __nv_bfloat162*>(&rd);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float2 v = __bfloat1622float2(hy[h]), d2 = __bfloat1622float2(hd[h]);
        const float vv[2] = {v.x, v.y}, dd[2] = {d2.x, d2.y};
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const int j = 2 * h + t;
          const float z = fmaf(vv[t], sc[j], sh[j]);
          const float dz = (!relu || z > 0.f) ? dd[t] : 0.f;
          const float xh = fmaf(vv[t], rs[j], -mr[j]);
          a0[j] += dz;
          a1[j] = fmaf(dz, xh, a1[j]);
        }
      }
    };
    long long p = p0 + r;
    if (HEAD) {
      for (; p + (long long)(U - 1) * rows < p1; p += (long long)U * rows) {
        uint2 ry[U];
        float dv[U][HK];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          ry[u] = *reinterpret_cast<const uint2*>(y + (base + p + (long long)u * rows) * y_ld + ch0);
#pragma unroll
          for (int k = 0; k < HK; ++k) dv[u][k] = __ldg(dl + (base + p + (long long)u * rows) * HK + k);
        }
        float wq[4][HK];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int k = 0; k < HK; ++k) wq[j][k] = wv[j * HK + k];
#pragma unroll
        for (int u = 0; u < U; ++u) one(ry[u], head_grad4<HEAD>(dv[u], wq));
      }
      for (; p < p1; p += rows) {
        float dv[HK], wq[4][HK];
#pragma unroll
        for (int k = 0; k < HK; ++k) dv[k] = __ldg(dl + (base + p) * HK + k);
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int k = 0; k < HK; ++k) wq[j][k] = wv[j * HK + k];
        one(*reinterpret_cast<const uint2*>(y + (base + p) * y_ld + ch0), head_grad4<HEAD>(dv, wq));
      }
    } else {
      for (; p + (long long)(U - 1) * rows < p1; p += (long long)U * rows) {
        uint2 ry[U], rd[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          ry[u] = *reinterpret_cast<const uint2*>(y + (base + p + (long long)u * rows) * y_ld + ch0);
          rd[u] = *reinterpret_cast<const uint2*>(da + (base + p + (long long)u * rows) * da_ld + ch0);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) one(ry[u], rd[u]);
      }
      for (; p < p1; p += rows)
        one(*reinterpret_cast<const uint2*>(y + (base + p) * y_ld + ch0),
            *reinterpret_cast<const uint2*>(da + (base + p) * da_ld + ch0));
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      sm[(r * 2 + 0) * c + ch0 + j] = a0[j];
      sm[(r * 2 + 1) * c + ch0 + j] = a1[j];
    }
  }
  __syncthreads();
  float* out = part + ((long long)group * gridDim.x + blockIdx.x) * 2 * c;
  for (int i = threadIdx.x; i < 2 * c; i += blockDim.x) {
    float s = 0.f;
    for (int rr = 0; rr < rows; ++rr) s += sm[rr * 2 * c + i];
    out[i] = s;
  }
}

// The un-guided backward apply with 4 channels per thread (8-byte loads / stores): ~48 registers instead of 80.
//   dy = scale * dz + k1 * v + k0,  k1 = -scale * c2 * rstd,  k0 = scale * (c2 * rstd * mean - c1)
template <int U, int HEAD>
__global__ void __launch_bounds__(256, 4)
norm_bwd_apply4_kernel(const __nv_bfloat16* __restrict__ y, int y_ld, const __nv_bfloat16* __restrict__ da, int da_ld,
                       __nv_bfloat16* __restrict__ dy, int dy_ld, long long pixels_per_group, int c, int relu,
                       const float* __restrict__ mean, const float* __restrict__ rstd,
                       const float* __restrict__ scale, const float* __restrict__ shift,
                       const float* __restrict__ c1, const float* __restrict__ c2, int gstride,
                       const float* __restrict__ dl, const float* __restrict__ wh) {
  bsl::pdl_wait();
  constexpr int HK = HEAD ? HEAD : 1;
  const int cg = c / 4;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  const int ch0 = g * 4;
  const int o = blockIdx.y * gstride + ch0;
  float sc[4], sh[4], k1[4], k0[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    sc[j] = scale[o + j];
    sh[j] = shift[o + j];
    const float t = sc[j] * c2[o + j] * rstd[o + j];
    k1[j] = -t;
    k0[j] = fmaf(t, mean[o + j], -sc[j] * c1[o + j]);
  }
  const long long base = (long long)blockIdx.y * pixels_per_group;
  const long long stride = (long long)gridDim.x * rows;
  auto one = [&](const uint2& ry, const uint2& rd) -> uint2 {
    const __nv_bfloat162* hy = reinterpret_cast<const __nv_bfloat162*>(&ry);
    const __nv_bfloat162* hd = reinterpret_cast<const __nv_bfloat162*>(&rd);
    uint2 outv;
    __nv_bfloat162* ho = reinterpret_cast<__nv_bfloat162*>(&outv);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float2 v = __bfloat1622float2(hy[h]), d2 = __bfloat1622float2(hd[h]);
      const float vv[2] = {v.x, v.y}, dd[2] = {d2.x, d2.y};
      float res[2];
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int j = 2 * h + t;
        const float z = fmaf(vv[t], sc[j], sh[j]);
        const float dz = (!relu || z > 0.f) ? dd[t] : 0.f;
        res[t] = fmaf(sc[j], dz, fmaf(k1[j], vv[t], k0[j]));
      }
      ho[h] = __floats2bfloat162_rn(res[0], res[1]);
    }
    return outv;
  };
  __shared__ float s_wh[HEAD ? 256 * HK : 1];   // see norm_bwd_reduce4_kernel
  if (HEAD) {
    for (int i = threadIdx.x; i < c * HK; i += blockDim.x) s_wh[i] = wh[i];
    __syncthreads();
  }
  const volatile float* wv = s_wh + ch0 * HK;
  if (r < rows && HEAD) {
    long long p = (long long)blockIdx.x * rows + r;
    for (; p + (U - 1) * stride < pixels_per_group; p += U * stride) {
      uint2 ry[U];
      float dv[U][HK];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        ry[u] = *reinterpret_cast<const uint2*>(y + (base + p + u * stride) * y_ld + ch0);
#pragma unroll
        for (int k = 0; k < HK; ++k) dv[u][k] = __ldg(dl + (base + p + u * stride) * HK + k);
      }
      float wq[4][HK];
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < HK; ++k) wq[j][k] = wv[j * HK + k];
#pragma unroll
      for (int u = 0; u < U; ++u)
        *reinterpret_cast<uint2*>(dy + (base + p + u * stride) * dy_ld + ch0) = one(ry[u], head_grad4<HEAD>(dv[u], wq));
    }
    for (; p < pixels_per_group; p += stride) {
      float dv[HK], wq[4][HK];
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < HK; ++k) wq[j][k] = wv[j * HK + k];
#pragma unroll
      for (int k = 0; k < HK; ++k) dv[k] = __ldg(dl + (base + p) * HK + k);
      *reinterpret_cast<uint2*>(dy + (base + p) * dy_ld + ch0) =
          one(*reinterpret_cast<const uint2*>(y + (base + p) * y_ld + ch0), head_grad4<HEAD>(dv, wq));
    }
  } else if (r < rows) {
    long long p = (long long)blockIdx.x * rows + r;
    for (; p + (U - 1) * stride < pixels_per_group; p += U * stride) {
      uint2 ry[U], rd[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        ry[u] = *reinterpret_cast<const uint2*>(y + (base + p + u * stride) * y_ld + ch0);
        rd[u] = *reinterpret_cast<const uint2*>(da + (base + p + u * stride) * da_ld + ch0);
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
        *reinterpret_cast<uint2*>(dy + (base + p + u * stride) * dy_ld + ch0) = one(ry[u], rd[u]);
    }
    for (; p < pixels_per_group; p += stride)
      *reinterpret_cast<uint2*>(dy + (base + p) * dy_ld + ch0) =
          one(*reinterpret_cast<const uint2*>(y + (base + p) * y_ld + ch0),
              *reinterpret_cast<const uint2*>(da + (base + p) * da_ld + ch0));
  }
}

// Guided variant of the 4-channels-per-thread backward apply (GUNet's modulated layers, G = 1 or 2 guide channels):
// z = y * scale + shift + sum_g guide[p][g] * wsp[g][c]. Same thread layout as the un-guided kernel; 8-byte accesses,
// <= 64 registers.
template <int U, int G>
__global__ void __launch_bounds__(256, 4)
norm_bwd_apply4g_kernel(const __nv_bfloat16* __restrict__ y, int y_ld, const __nv_bfloat16* __restrict__ da, int da_ld,
                        __nv_bfloat16* __restrict__ dy, int dy_ld, long long pixels_per_group, int c, int relu,
                        const float* __restrict__ mean, const float* __restrict__ rstd,
                        const float* __restrict__ scale, const float* __restrict__ shift,
                        const float* __restrict__ c1, const float* __restrict__ c2, int gstride,
                        const float* __restrict__ guide, const float* __restrict__ wsp, int wsp_ld) {
  bsl::pdl_wait();
  const int cg = c / 4;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  const int ch0 = g * 4;
  const int o = blockIdx.y * gstride + ch0;
  float sc[4], sh[4], k1[4], k0[4], ws[G][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    sc[j] = scale[o + j];
    sh[j] = shift[o + j];
    const float t = sc[j] * c2[o + j] * rstd[o + j];
    k1[j] = -t;
    k0[j] = fmaf(t, mean[o + j], -sc[j] * c1[o + j]);
#pragma unroll
    for (int q = 0; q < G; ++q) ws[q][j] = wsp[q * wsp_ld + ch0 + j];
  }
  const long long base = (long long)blockIdx.y * pixels_per_group;
  const long long stride = (long long)gridDim.x * rows;
  auto one = [&](const uint2& ry, const uint2& rd, const float (&gm)[G]) -> uint2 {
    const __nv_bfloat162* hy = reinterpret_cast<const __nv_bfloat162*>(&ry);
    const __nv_bfloat162* hd = reinterpret_cast<const __nv_bfloat162*>(&rd);
    uint2 outv;
    __nv_bfloat162* ho = reinterpret_cast<__nv_bfloat162*>(&outv);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float2 v = __bfloat1622float2(hy[h]), d2 = __bfloat1622float2(hd[h]);
      const float vv[2] = {v.x, v.y}, dd[2] = {d2.x, d2.y};
      float res[2];
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int j = 2 * h + t;
        float z = fmaf(vv[t], sc[j], sh[j]);
#pragma unroll
        for (int q = 0; q < G; ++q) z = fmaf(gm[q], ws[q][j], z);
        const float dz = (!relu || z > 0.f) ? dd[t] : 0.f;
        res[t] = fmaf(sc[j], dz, fmaf(k1[j], vv[t], k0[j]));
      }
      ho[h] = __floats2bfloat162_rn(res[0], res[1]);
    }
    return outv;
  };
  if (r < rows) {
    long long p = (long long)blockIdx.x * rows + r;
    for (; p + (U - 1) * stride < pixels_per_group; p += U * stride) {
      uint2 ry[U], rd[U];
      float gm[U][G];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long px = base + p + u * stride;
        ry[u] = *reinterpret_cast<const uint2*>(y + px * y_ld + ch0);
        rd[u] = *reinterpret_cast<const uint2*>(da + px * da_ld + ch0);
#pragma unroll
        for (int q = 0; q < G; ++q) gm[u][q] = __ldg(guide + px * G + q);
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
        *reinterpret_cast<uint2*>(dy + (base + p + u * stride) * dy_ld + ch0) = one(ry[u], rd[u], gm[u]);
    }
    for (; p < pixels_per_group; p += stride) {
      float gm[G];
#pragma unroll
      for (int q = 0; q < G; ++q) gm[q] = __ldg(guide + (base + p) * G + q);
      *reinterpret_cast<uint2*>(dy + (base + p) * dy_ld + ch0) =
          one(*reinterpret_cast<const uint2*>(y + (base + p) * y_ld + ch0),
              *reinterpret_cast<const uint2*>(da + (base + p) * da_ld + ch0), gm);
    }
  }
}

int run_bwd_reduce4(bsl_ctx* ctx, const bsl_norm_desc* d, const __nv_bfloat16* xb, const __nv_bfloat16* db, int dy_ld,
                    const float* mean, const float* rstd, const float* scale, const float* shift, long long ppg,
                    int groups, double* sums, cudaStream_t stream, const float* dl = nullptr,
                    const float* wh = nullptr, int classes = 0) {
  const int c = d->c, cg = c / 4;
  const int rows = 256 / cg;
  const int threads = rows * cg;
  long long want = (ppg * c + 32767) / 32768;
  long long cap = (8LL * ctx->sm_count + groups - 1) / groups;   // two waves of four resident blocks
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  const int blocks = (int)want;
  const long long ppb = (ppg + blocks - 1) / blocks;
  float* part = nullptr;
  int rc = bsl_scratch(ctx, (size_t)groups * blocks * 2 * c * sizeof(float), &part, stream);
  if (rc) return rc;
  const size_t smem = (size_t)rows * 2 * c * sizeof(float);
  auto go = [&](auto kern) {
    bsl_launch(kern, dim3(blocks, groups), dim3(threads), smem, stream, xb, d->x_ld, db, dy_ld, mean, rstd, scale, shift, c,
               d->relu, ppg, ppb, part, dl, wh);
  };
  switch (classes) {
    case 0: go(norm_bwd_reduce4_kernel<4, 0>); break;
    case 2: go(norm_bwd_reduce4_kernel<4, 2>); break;
    case 3: go(norm_bwd_reduce4_kernel<4, 3>); break;
    default: go(norm_bwd_reduce4_kernel<4, 4>); break;
  }
  BSL_LAUNCH_CHECK(ctx, "norm_bwd_reduce4_kernel");
  bsl_launch(pixel_reduce_final_kernel, dim3(dim3((2 * c + 31) / 32, groups)), dim3(1024), 0, stream, part, blocks, 2 * c, sums);
  BSL_LAUNCH_CHECK(ctx, "pixel_reduce_final_kernel");
  return BSL_OK;
}
}  // namespace

extern "C" {

int bsl_norm_bwd_reduce_mod(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const void* dy, int dy_ld,
                            const float* mean, const float* rstd, const float* scale, const float* shift,
                            const bsl_guide* guide, double* sums, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!x || !dy || !mean || !rstd || !scale || !shift || !sums)
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_reduce: null buffer");
  int G;
  if ((rc = check_guide(ctx, d, guide, &G))) return rc;
  const int groups = d->mode ? d->n : 1;
  const long long ppg = d->mode ? d->hw : (long long)d->n * d->hw;
  auto xb = reinterpret_cast<const __nv_bfloat16*>(x);
  auto db = reinterpret_cast<const __nv_bfloat16*>(dy);
  if (G == 0) {
    if (d->c % 4 == 0 && d->c <= 1024 && 256 % (d->c / 4) == 0 && d->x_ld % 4 == 0 && dy_ld % 4 == 0)
      return run_bwd_reduce4(ctx, d, xb, db, dy_ld, mean, rstd, scale, shift, ppg, groups, sums, as_stream(stream));
    BwdFG<0> f{nullptr, nullptr, 0, xb, db, mean, rstd, scale, shift, d->x_ld, dy_ld, d->c, d->relu};
    return run_pixel_reduce(ctx, f, ppg, groups, d->c, sums, as_stream(stream));
  }
  // guided layers stay on the 8-channel functor: a 4-channel guided reduce measured 1.50 ms against 1.28 ms on cfg3
  // (8 guided layers per step); the guided APPLY, norm_bwd_apply4g_kernel, is the one that pays (3.80 -> 3.45 ms)
  if (G == 1) {
    BwdFG<1> f{guide->map, guide->w, guide->w_ld, xb, db, mean, rstd, scale, shift, d->x_ld, dy_ld, d->c, d->relu};
    return run_pixel_reduce(ctx, f, ppg, groups, d->c, sums, as_stream(stream));
  }
  BwdFG<2> f{guide->map, guide->w, guide->w_ld, xb, db, mean, rstd, scale, shift, d->x_ld, dy_ld, d->c, d->relu};
  return run_pixel_reduce(ctx, f, ppg, groups, d->c, sums, as_stream(stream));
}

int bsl_norm_bwd_reduce(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const void* dy, int dy_ld,
                        const float* mean, const float* rstd, const float* scale, const float* shift,
                        double* sums, void* stream) {
  return bsl_norm_bwd_reduce_mod(ctx, d, x, dy, dy_ld, mean, rstd, scale, shift, nullptr, sums, stream);
}

// ---- last normalised layer + logits layer: backward passes that recompute the activation gradient from dlogits
static bool bwd_head_ok(const bsl_norm_desc* d, int classes, int dx_ld) {
  return d->c % 4 == 0 && d->c <= 256 && 256 % (d->c / 4) == 0 && d->x_ld % 4 == 0 && dx_ld % 4 == 0 && classes >= 2 &&
         classes <= 4;
}

int bsl_norm_bwd_head_ok(bsl_ctx* ctx, const bsl_norm_desc* d, int classes) {
  return ctx && d && check_norm(ctx, d) == BSL_OK && bwd_head_ok(d, classes, 4) ? 1 : 0;
}

int bsl_norm_bwd_reduce_head(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const float* dlogits,
                             const float* w_head, int classes, const float* mean, const float* rstd,
                             const float* scale, const float* shift, double* sums, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!x || !dlogits || !w_head || !mean || !rstd || !scale || !shift || !sums)
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_reduce_head: null buffer");
  if (!bwd_head_ok(d, classes, 4))
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "norm_bwd_reduce_head: c=%d (multiple of 4 dividing 1024, <= 256), classes=%d (2..4)",
                    d->c, classes);
  const int groups = d->mode ? d->n : 1;
  const long long ppg = d->mode ? d->hw : (long long)d->n * d->hw;
  return run_bwd_reduce4(ctx, d, reinterpret_cast<const __nv_bfloat16*>(x), nullptr, 0, mean, rstd, scale, shift, ppg,
                         groups, sums, as_stream(stream), dlogits, w_head, classes);
}

int bsl_norm_bwd_apply_head(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const float* dlogits,
                            const float* w_head, int classes, const float* mean, const float* rstd,
                            const float* scale, const float* shift, const float* c1, const float* c2, void* dx,
                            int dx_ld, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!x || !dlogits || !w_head || !mean || !rstd || !scale || !shift || !c1 || !c2 || !dx)
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_apply_head: null buffer");
  if (!bwd_head_ok(d, classes, dx_ld))
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "norm_bwd_apply_head: c=%d (multiple of 4 dividing 1024, <= 256), classes=%d (2..4)",
                    d->c, classes);
  const int groups = d->mode ? d->n : 1;
  const long long ppg = d->mode ? d->hw : (long long)d->n * d->hw;
  const int cg4 = d->c / 4, rows4 = 256 / cg4;
  long long want = (ppg + (long long)rows4 * 4 - 1) / ((long long)rows4 * 4);
  const long long cap = (16LL * ctx->sm_count + groups - 1) / groups;
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  auto go = [&](auto kern) {
    bsl_launch(kern, dim3((unsigned)want, groups), dim3(rows4 * cg4), 0, as_stream(stream),
               reinterpret_cast<const __nv_bfloat16*>(x), d->x_ld, (const __nv_bfloat16*)nullptr, 0,
               reinterpret_cast<__nv_bfloat16*>(dx), dx_ld, ppg, d->c, d->relu, mean, rstd, scale, shift, c1, c2,
               d->mode ? d->c : 0, dlogits, w_head);
  };
  switch (classes) {
    case 2: go(norm_bwd_apply4_kernel<4, 2>); break;
    case 3: go(norm_bwd_apply4_kernel<4, 3>); break;
    default: go(norm_bwd_apply4_kernel<4, 4>); break;
  }
  BSL_LAUNCH_CHECK(ctx, "norm_bwd_apply4_kernel (logits gradient recomputed)");
  return BSL_OK;
}

int bsl_norm_bwd_finalize(bsl_ctx* ctx, const bsl_norm_desc* d, const double* sums, float* c1, float* c2,
                          float* dgamma, float* dbeta, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!sums || !c1 || !c2) return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_finalize: null buffer");
  const int groups = d->mode ? d->n : 1;
  const double m = d->mode ? (double)d->hw : (double)d->n * d->hw;
  const int glanes = groups >= 32 ? 32 : (groups >= 8 ? 8 : (groups >= 4 ? 4 : 1));
  bsl_launch(norm_bwd_finalize_kernel, dim3((d->c + 31) / 32), dim3(32 * glanes), 0, as_stream(stream), groups, d->c, m, sums, nullptr, c1, c2,
                                                                             dgamma, dbeta);
  BSL_LAUNCH_CHECK(ctx, "norm_bwd_finalize_kernel");
  return BSL_OK;
}

int bsl_norm_modulate(bsl_ctx* ctx, const bsl_norm_desc* d, const float* gamma_mod, int gm_ld, const float* sp_bias,
                      float* scale, float* shift, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (d->mode != 1) return bsl_fail(ctx, BSL_EUNSUPPORTED, "norm_modulate: instance_norm layers only");
  if (!scale || !shift || (gamma_mod && gm_ld < d->c)) return bsl_fail(ctx, BSL_EINVAL, "norm_modulate: bad argument");
  const int total = d->n * d->c;
  bsl_launch(norm_modulate_kernel, dim3((total + 127) / 128), dim3(128), 0, as_stream(stream), d->n, d->c, gamma_mod, gm_ld, sp_bias, scale,
                                                                         shift);
  BSL_LAUNCH_CHECK(ctx, "norm_modulate_kernel");
  return BSL_OK;
}

int bsl_norm_bwd_finalize_mod(bsl_ctx* ctx, const bsl_norm_desc* d, const double* sums, int guide_channels,
                              const float* gamma_mod, int gm_ld, const float* gamma, const float* beta, float* c1,
                              float* c2, float* dgamma, float* dbeta, float* dgamma_mod, float* dw_guide, int dw_ld,
                              float* dbias_guide, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (d->mode != 1) return bsl_fail(ctx, BSL_EUNSUPPORTED, "norm_bwd_finalize_mod: instance_norm layers only");
  if (!sums || !c1 || !c2 || guide_channels < 0 || guide_channels > 2 || (gamma_mod && !dgamma_mod) ||
      (guide_channels && (!dw_guide || dw_ld < d->c)))
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_finalize_mod: bad argument");
  bsl_launch(norm_bwd_finalize_mod_kernel, dim3((d->c + 31) / 32), dim3(32 * FM_S), 0, as_stream(stream), 
      d->n, d->c, 2 + guide_channels, (double)d->hw, sums, gamma_mod, gm_ld, d->scale ? gamma : nullptr,
      d->center ? beta : nullptr, c1, c2, dgamma, dbeta, dgamma_mod, dw_guide, dw_ld, dbias_guide);
  BSL_LAUNCH_CHECK(ctx, "norm_bwd_finalize_mod_kernel");
  return BSL_OK;
}

int bsl_norm_modulate_bn(bsl_ctx* ctx, const bsl_norm_desc* d, const float* gamma_mod, int gm_ld, const float* sp_bias,
                         float* mean, float* rstd, float* scale, float* shift, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!mean || !rstd || !scale || !shift || (gamma_mod && gm_ld < d->c))
    return bsl_fail(ctx, BSL_EINVAL, "norm_modulate_bn: bad argument");
  bsl_launch(norm_modulate_bn_kernel, dim3((d->c + 127) / 128), dim3(128), 0, as_stream(stream), d->n, d->c, gamma_mod, gm_ld,
             sp_bias, mean, rstd, scale, shift);
  BSL_LAUNCH_CHECK(ctx, "norm_modulate_bn_kernel");
  return BSL_OK;
}

int bsl_norm_bwd_finalize_bnmod(bsl_ctx* ctx, const bsl_norm_desc* d, const double* sums, int guide_channels,
                                const float* gamma_mod, int gm_ld, const float* gamma, const float* beta,
                                const float* rstd, float* c1r, float* c2r, float* dgamma, float* dbeta,
                                float* dgamma_mod, float* dw_guide, int dw_ld, float* dbias_guide, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!sums || !c1r || !c2r || !rstd || guide_channels < 0 || guide_channels > 2 || (gamma_mod && !dgamma_mod) ||
      (guide_channels && (!dw_guide || dw_ld < d->c)))
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_finalize_bnmod: bad argument");
  bsl_launch(norm_bwd_finalize_bnmod_kernel, dim3((d->c + 127) / 128), dim3(128), 0, as_stream(stream), d->n, d->c,
             2 + guide_channels, (double)d->n * d->hw, sums, gamma_mod, gm_ld, d->scale ? gamma : nullptr,
             d->center ? beta : nullptr, rstd, c1r, c2r, dgamma, dbeta, dgamma_mod, dw_guide, dw_ld, dbias_guide);
  BSL_LAUNCH_CHECK(ctx, "norm_bwd_finalize_bnmod_kernel");
  return BSL_OK;
}

int bsl_norm_affine_fold(bsl_ctx* ctx, const bsl_norm_desc* d, const float* gamma_a, const float* beta_a, float* scale,
                         float* shift, float* scale_pre, float* shift_pre, const float* w_guide, int w_ld,
                         int guide_channels, float* w_eff, void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!gamma_a || !beta_a || !scale || !shift || !scale_pre || !shift_pre || guide_channels < 0 || guide_channels > 2 ||
      (guide_channels && (!w_guide || !w_eff || w_ld < d->c)))
    return bsl_fail(ctx, BSL_EINVAL, "norm_affine_fold: bad argument");
  const int groups = d->mode ? d->n : 1;
  const int total = groups > guide_channels ? groups * d->c : guide_channels * d->c;
  bsl_launch(norm_affine_fold_kernel, dim3((total + 127) / 128), dim3(128), 0, as_stream(stream), groups, d->c,
             guide_channels, gamma_a, beta_a, scale, shift, scale_pre, shift_pre, w_guide, w_ld, w_eff);
  BSL_LAUNCH_CHECK(ctx, "norm_affine_fold_kernel");
  return BSL_OK;
}

int bsl_norm_bwd_finalize_affine_jac(bsl_ctx* ctx, const bsl_norm_desc* d, int jacobian, const double* sums,
                                     int guide_channels, const float* gamma_mod, int gm_ld, const float* gamma,
                                     const float* beta, const float* gamma_a, const float* mean, const float* rstd,
                                     const float* scale_pre, const float* shift_pre, const float* w_guide, int w_ld,
                                     float* c1, float* c2, float* dgamma, float* dbeta, float* dgamma_mod,
                                     float* dw_guide, int dw_ld, float* dbias_guide, float* dgamma_a, float* dbeta_a,
                                     void* stream) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (jacobian != BSL_NORM_JAC_GROUP && jacobian != BSL_NORM_JAC_BATCH && jacobian != BSL_NORM_JAC_NONE)
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_finalize_affine: jacobian %d", jacobian);
  if (jacobian == BSL_NORM_JAC_BATCH && d->mode != 1)
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_finalize_affine: BSL_NORM_JAC_BATCH takes the per-sample (mode 1) view");
  const int groups = d->mode ? d->n : 1;
  if (!sums || !c1 || !c2 || !gamma_a || !mean || !rstd || !scale_pre || !shift_pre || !dgamma_a || !dbeta_a ||
      guide_channels < 0 || guide_channels > 2 || (gamma_mod && (!dgamma_mod || groups != d->n)) ||
      (guide_channels && (!dw_guide || dw_ld < d->c || !w_guide || w_ld < d->c)))
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_finalize_affine: bad argument");
  const double m = d->mode && jacobian != BSL_NORM_JAC_BATCH ? (double)d->hw : (double)d->n * d->hw;
  bsl_launch(norm_bwd_finalize_affine_kernel, dim3((d->c + 127) / 128), dim3(128), 0, as_stream(stream), groups, d->c,
             2 + guide_channels, m, jacobian, sums, gamma_mod, gm_ld, d->scale ? gamma : nullptr,
             d->center ? beta : nullptr, gamma_a, mean, rstd, scale_pre, shift_pre, w_guide, w_ld, c1, c2, dgamma, dbeta,
             dgamma_mod, dw_guide, dw_ld, dbias_guide, dgamma_a, dbeta_a);
  BSL_LAUNCH_CHECK(ctx, "norm_bwd_finalize_affine_kernel");
  return BSL_OK;
}

int bsl_norm_bwd_finalize_affine(bsl_ctx* ctx, const bsl_norm_desc* d, const double* sums, int guide_channels,
                                 const float* gamma_mod, int gm_ld, const float* gamma, const float* beta,
                                 const float* gamma_a, const float* mean, const float* rstd, const float* scale_pre,
                                 const float* shift_pre, const float* w_guide, int w_ld, float* c1, float* c2,
                                 float* dgamma, float* dbeta, float* dgamma_mod, float* dw_guide, int dw_ld,
                                 float* dbias_guide, float* dgamma_a, float* dbeta_a, void* stream) {
  return bsl_norm_bwd_finalize_affine_jac(ctx, d, BSL_NORM_JAC_GROUP, sums, guide_channels, gamma_mod, gm_ld, gamma,
                                          beta, gamma_a, mean, rstd, scale_pre, shift_pre, w_guide, w_ld, c1, c2, dgamma,
                                          dbeta, dgamma_mod, dw_guide, dw_ld, dbias_guide, dgamma_a, dbeta_a, stream);
}

static int norm_bwd_apply_impl(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const void* dy, int dy_ld,
                               const float* mean, const float* rstd, const float* scale, const float* shift,
                               const float* c1, const float* c2, const bsl_guide* guide, void* dx, int dx_ld,
                               void* stream, int premul);

int bsl_norm_bwd_apply_mod(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const void* dy, int dy_ld,
                           const float* mean, const float* rstd, const float* scale, const float* shift,
                           const float* c1, const float* c2, const bsl_guide* guide, void* dx, int dx_ld,
                           void* stream) {
  return norm_bwd_apply_impl(ctx, d, x, dy, dy_ld, mean, rstd, scale, shift, c1, c2, guide, dx, dx_ld, stream, 0);
}

int bsl_norm_bwd_apply_bnmod(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const void* dy, int dy_ld,
                             const float* mean, const float* rstd, const float* scale, const float* shift,
                             const float* c1r, const float* c2r, const bsl_guide* guide, void* dx, int dx_ld,
                             void* stream) {
  if (d && d->mode != 1)
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_apply_bnmod: pass the per-sample (mode 1) view of the layer");
  return norm_bwd_apply_impl(ctx, d, x, dy, dy_ld, mean, rstd, scale, shift, c1r, c2r, guide, dx, dx_ld, stream, 1);
}

static int norm_bwd_apply_impl(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const void* dy, int dy_ld,
                               const float* mean, const float* rstd, const float* scale, const float* shift,
                               const float* c1, const float* c2, const bsl_guide* guide, void* dx, int dx_ld,
                               void* stream, int premul) {
  int rc = check_norm(ctx, d);
  if (rc) return rc;
  if (!x || !dy || !mean || !rstd || !scale || !shift || !c1 || !c2 || !dx)
    return bsl_fail(ctx, BSL_EINVAL, "norm_bwd_apply: null buffer");
  int G;
  if ((rc = check_guide(ctx, d, guide, &G))) return rc;
  const int groups = d->mode ? d->n : 1;
  const long long ppg = d->mode ? d->hw : (long long)d->n * d->hw;
  const EwPlan pl = ew_plan(ctx, ppg, groups, d->c, 4);
  const int gstride = d->mode ? d->c : 0;
  const dim3 grid(pl.blocks, groups);
  auto xb = reinterpret_cast<const __nv_bfloat16*>(x);
  auto db = reinterpret_cast<const __nv_bfloat16*>(dy);
  auto ob = reinterpret_cast<__nv_bfloat16*>(dx);
  cudaStream_t s = as_stream(stream);
  if (!premul && G == 0 && d->c % 4 == 0 && d->c <= 1024 && 256 % (d->c / 4) == 0 && d->x_ld % 4 == 0 &&
      dy_ld % 4 == 0 && dx_ld % 4 == 0) {
    const int cg4 = d->c / 4, rows4 = 256 / cg4;
    long long want = (ppg + (long long)rows4 * 4 - 1) / ((long long)rows4 * 4);
    const long long cap = (16LL * ctx->sm_count + groups - 1) / groups;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    bsl_launch(norm_bwd_apply4_kernel<4, 0>, dim3((unsigned)want, groups), dim3(rows4 * cg4), 0, s,
               xb, d->x_ld, db, dy_ld, ob, dx_ld, ppg, d->c, d->relu, mean, rstd, scale, shift, c1, c2, gstride,
               (const float*)nullptr, (const float*)nullptr);
    BSL_LAUNCH_CHECK(ctx, "norm_bwd_apply4_kernel");
    return BSL_OK;
  }
  if (!premul && G > 0 && d->c % 4 == 0 && d->c <= 1024 && 256 % (d->c / 4) == 0 && d->x_ld % 4 == 0 &&
      dy_ld % 4 == 0 && dx_ld % 4 == 0) {
    const int cg4 = d->c / 4, rows4 = 256 / cg4;
    long long want = (ppg + (long long)rows4 * 4 - 1) / ((long long)rows4 * 4);
    const long long cap = (16LL * ctx->sm_count + groups - 1) / groups;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    if (G == 1)   // (G == 2 unrolls two pixels instead of four: 64 registers without spills)
      bsl_launch(norm_bwd_apply4g_kernel<4, 1>, dim3((unsigned)want, groups), dim3(rows4 * cg4), 0, s, xb, d->x_ld, db, dy_ld,
                 ob, dx_ld, ppg, d->c, d->relu, mean, rstd, scale, shift, c1, c2, gstride, guide->map, guide->w, guide->w_ld);
    else
      bsl_launch(norm_bwd_apply4g_kernel<2, 2>, dim3((unsigned)want, groups), dim3(rows4 * cg4), 0, s, xb, d->x_ld, db, dy_ld,
                 ob, dx_ld, ppg, d->c, d->relu, mean, rstd, scale, shift, c1, c2, gstride, guide->map, guide->w, guide->w_ld);
    BSL_LAUNCH_CHECK(ctx, "norm_bwd_apply4g_kernel");
    return BSL_OK;
  }
  if (G == 0)
    bsl_launch(norm_bwd_apply_kernel<0>, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, db, dy_ld, ob, dx_ld, ppg, d->c, d->relu, mean,
                                                         rstd, scale, shift, c1, c2, nullptr, nullptr, 0, gstride, premul);
  else if (G == 1)
    bsl_launch(norm_bwd_apply_kernel<1>, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, db, dy_ld, ob, dx_ld, ppg, d->c, d->relu, mean,
                                                         rstd, scale, shift, c1, c2, guide->map, guide->w, guide->w_ld,
                                                         gstride, premul);
  else
    bsl_launch(norm_bwd_apply_kernel<2>, dim3(grid), dim3(pl.threads), 0, s, xb, d->x_ld, db, dy_ld, ob, dx_ld, ppg, d->c, d->relu, mean,
                                                         rstd, scale, shift, c1, c2, guide->map, guide->w, guide->w_ld,
                                                         gstride, premul);
  BSL_LAUNCH_CHECK(ctx, "norm_bwd_apply_kernel");
  return BSL_OK;
}

int bsl_norm_bwd_apply(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x, const void* dy, int dy_ld,
                       const float* mean, const float* rstd, const float* scale, const float* shift,
                       const float* c1, const float* c2, void* dx, int dx_ld, void* stream) {
  return bsl_norm_bwd_apply_mod(ctx, d, x, dy, dy_ld, mean, rstd, scale, shift, c1, c2, nullptr, dx, dx_ld, stream);
}

int bsl_maxpool2x2_bwd_add(bsl_ctx* ctx, int n, int h, int w, int c, const void* act, int act_ld,
                           const void* dpool, int dpool_ld, const void* dskip, int dskip_ld, void* dact,
                           int dact_ld, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!act || !dpool || !dact) return bsl_fail(ctx, BSL_EINVAL, "maxpool_bwd: null buffer");
  if ((h & 1) || (w & 1) || c % 8) return bsl_fail(ctx, BSL_EUNSUPPORTED, "maxpool_bwd: h,w even, c%%8==0");
  const long long items = (long long)n * (h / 2) * (w / 2) * (c / 8);
  bsl_launch(maxpool_bwd_add_kernel, dim3(ew_grid(ctx, items)), dim3(256), 0, as_stream(stream), 
      reinterpret_cast<const __nv_bfloat16*>(act), act_ld, reinterpret_cast<const __nv_bfloat16*>(dpool), dpool_ld,
      reinterpret_cast<const __nv_bfloat16*>(dskip), dskip_ld, reinterpret_cast<__nv_bfloat16*>(dact), dact_ld, n, h,
      w, c);
  BSL_LAUNCH_CHECK(ctx, "maxpool_bwd_add_kernel");
  return BSL_OK;
}

int bsl_maxpool2x2_bf16(bsl_ctx* ctx, int n, int h, int w, int c, const void* x, int x_ld, void* y, int y_ld,
                        void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!x || !y) return bsl_fail(ctx, BSL_EINVAL, "maxpool2x2_bf16: null buffer");
  if (n <= 0 || h <= 0 || w <= 0 || c <= 0) return bsl_fail(ctx, BSL_EINVAL, "maxpool2x2_bf16: non-positive size");
  if ((h & 1) || (w & 1) || c % 8 || x_ld < c || y_ld < c || x_ld % 8 || y_ld % 8 ||
      (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(y) & 15))
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "maxpool2x2_bf16: h=%d w=%d even, c=%d, x_ld=%d, y_ld=%d multiples of 8 >= c, "
                    "16-byte aligned buffers", h, w, c, x_ld, y_ld);
  const long long items = (long long)n * (h / 2) * (w / 2) * (c / 8);
  bsl_launch(maxpool2x2_bf16_kernel, dim3(ew_grid(ctx, items)), dim3(256), 0, as_stream(stream),
             reinterpret_cast<const __nv_bfloat16*>(x), x_ld, reinterpret_cast<__nv_bfloat16*>(y), y_ld, n, h, w, c);
  BSL_LAUNCH_CHECK(ctx, "maxpool2x2_bf16_kernel");
  return BSL_OK;
}

int bsl_add_bf16(bsl_ctx* ctx, long long pixels, int c, const void* a, int a_ld, const void* b, int b_ld, void* out,
                 int out_ld, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!a || !b || !out) return bsl_fail(ctx, BSL_EINVAL, "add_bf16: null buffer");
  if (c % 8 || a_ld % 8 || b_ld % 8 || out_ld % 8) return bsl_fail(ctx, BSL_EUNSUPPORTED, "add_bf16: c, ld %% 8");
  const EwPlan pl = ew_plan(ctx, pixels, 1, c, 2);
  bsl_launch(add_bf16_kernel, dim3(pl.blocks), dim3(pl.threads), 0, as_stream(stream), 
      reinterpret_cast<const __nv_bfloat16*>(a), a_ld, reinterpret_cast<const __nv_bfloat16*>(b), b_ld,
      reinterpret_cast<__nv_bfloat16*>(out), out_ld, pixels, c);
  BSL_LAUNCH_CHECK(ctx, "add_bf16_kernel");
  return BSL_OK;
}

int bsl_relu_bwd(bsl_ctx* ctx, long long pixels, int c, const void* y, int y_ld, const void* dy, int dy_ld,
                 void* out, int out_ld, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!y || !dy || !out) return bsl_fail(ctx, BSL_EINVAL, "relu_bwd: null buffer");
  if (c % 8) return bsl_fail(ctx, BSL_EUNSUPPORTED, "relu_bwd: c%%8");
  const EwPlan pl = ew_plan(ctx, pixels, 1, c, EW_UNROLL);
  bsl_launch(relu_bwd_kernel, dim3(pl.blocks), dim3(pl.threads), 0, as_stream(stream), 
      reinterpret_cast<const __nv_bfloat16*>(y), y_ld, reinterpret_cast<const __nv_bfloat16*>(dy), dy_ld,
      reinterpret_cast<__nv_bfloat16*>(out), out_ld, pixels, c);
  BSL_LAUNCH_CHECK(ctx, "relu_bwd_kernel");
  return BSL_OK;
}

}  // extern "C"
