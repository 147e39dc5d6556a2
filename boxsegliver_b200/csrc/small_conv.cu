// CUDA-core convolutions for the two layers that are HBM-bound and would waste MMA tiles
// (SURVEY.md section 7 "tiny-K / skinny-N layers"):
//   stem    : slim.conv2d(images, 64, 3), cin = im_channel (1 or 3)  -- NetworksV2/UNet.py:79 (first call)
//   logits  : slim.conv2d(x, num_classes, 1) + bias, no activation    -- NetworksV2/UNet.py:100
// Together they are 0.26 % of the FLOPs; both read/write full-resolution tensors exactly once.
#include "reduce.cuh"

using namespace bsl;

namespace {

// ------------------------------------------------------------------------------------ stem fprop
// Thread = (pixel, 16-channel slice). Filter [kh*kw*CIN][cout] sits in shared memory.
template <int CIN>
__global__ void stem_fprop_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                  __nv_bfloat16* __restrict__ y, int y_ld, int n, int h, int wd, int cout, int kh,
                                  int kw) {
  bsl::pdl_wait();
  extern __shared__ float sw[];  // [taps*CIN][cout]
  const int taps = kh * kw;
  for (int i = threadIdx.x; i < taps * CIN * cout; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const int slices = cout / 16;
  const long long total = (long long)n * h * wd * slices;
  const int ph = (kh - 1) / 2, pw = (kw - 1) / 2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int sl = (int)(i % slices);
    const long long p = i / slices;
    const int xw = (int)(p % wd);
    const int yh = (int)((p / wd) % h);
    const long long img = p / ((long long)wd * h);
    float acc[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[j] = 0.f;
    for (int r = 0; r < kh; ++r) {
      const int yy = yh + r - ph;
      if (yy < 0 || yy >= h) continue;
      for (int s = 0; s < kw; ++s) {
        const int xx = xw + s - pw;
        if (xx < 0 || xx >= wd) continue;
        const float* xp = x + ((img * h + yy) * wd + xx) * CIN;
        const float* wp = sw + ((r * kw + s) * CIN) * cout + sl * 16;
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) {
          const float xv = __ldg(xp + ci);
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[j] = fmaf(xv, wp[ci * cout + j], acc[j]);
        }
      }
    }
    float lo[8], hi[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { lo[j] = acc[j]; hi[j] = acc[8 + j]; }
    __nv_bfloat16* o = y + p * y_ld + sl * 16;
    st16(o, pack8(lo));
    st16(o + 8, pack8(hi));
  }
}

// ------------------------------------------------------------------------------------ stem im2col
// col[p][t*CIN + ci] = x[p + tap t][ci] (zero outside the image, zero for columns >= taps*CIN), bf16,
// 64 columns per pixel. With this matrix the stem becomes a 1x1 conv with cin = 64 on the tcgen05
// path (fprop and wgrad), instead of a CUDA-core kernel. Thread = (pixel, 8-column group).
// Block = one strip of IM2COL_STRIP pixels of one image row. The (kh x (strip + kw - 1) x cin) input patch is
// staged in shared memory with coalesced loads (zero outside the image = SAME padding); thread
// (pixel lane, 8-column group g) then gathers its 8 columns through offsets that depend only on g
// (held in registers) and writes one 16-byte chunk: a warp writes 512 contiguous bytes.
constexpr int IM2COL_STRIP = 256;
__global__ void stem_im2col_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ col, int n, int h, int wd,
                                   int cin, int kh, int kw, int cols) {
  bsl::pdl_wait();
  extern __shared__ float patch[];  // [kh][strip + kw - 1][cin]
  const int strips = (wd + IM2COL_STRIP - 1) / IM2COL_STRIP;
  const int ph = (kh - 1) / 2, pw = (kw - 1) / 2;
  const int kcols = kh * kw * cin;
  const int pitch = (IM2COL_STRIP + kw - 1) * cin;
  const int ngrp = cols >> 3;                 // 8-column groups per row: 8 (64 columns) or 4 (32 columns)
  const int g = threadIdx.x & (ngrp - 1);
  const int px0 = threadIdx.x / ngrp, pxs = blockDim.x / ngrp;
  int off[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = g * 8 + j;
    const int t = c / cin, ci = c - t * cin;
    off[j] = c < kcols ? (t / kw) * pitch + (t % kw) * cin + ci : -1;
  }
  for (long long b = blockIdx.x; b < (long long)n * h * strips; b += gridDim.x) {
    const int sx = (int)(b % strips) * IM2COL_STRIP;
    const int yh = (int)((b / strips) % h);
    const long long img = b / ((long long)strips * h);
    __syncthreads();
    for (int i = threadIdx.x; i < kh * pitch; i += blockDim.x) {
      const int r = i / pitch, rem = i - r * pitch;
      const int xx = sx - pw + rem / cin, yy = yh - ph + r;
      patch[i] = (yy >= 0 && yy < h && xx >= 0 && xx < wd) ? __ldg(x + ((img * h + yy) * wd + xx) * cin + rem % cin) : 0.f;
    }
    __syncthreads();
    for (int px = px0; px < IM2COL_STRIP && sx + px < wd; px += pxs) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = off[j] >= 0 ? patch[off[j] + px * cin] : 0.f;
      st16(col + ((img * h + yh) * wd + sx + px) * cols + g * 8, pack8(v));
    }
  }
}

// The same kernel for 3x3 stems with the channel count known at compile time: the patch loader's index arithmetic
// (three integer divisions per element by cin / the patch pitch) becomes multiply-shift sequences -- with run-time
// divisors it was the bottleneck of the pass (16 us per 256-pixel strip and block).
template <int CIN>
__global__ void stem_im2col3_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ col, int n, int h, int wd,
                                    int cols) {
  bsl::pdl_wait();
  constexpr int KW = 3, KH = 3, KCOLS = KH * KW * CIN;
  constexpr int PITCH = (IM2COL_STRIP + KW - 1) * CIN;
  __shared__ float patch[KH * PITCH];
  const unsigned strips = (wd + IM2COL_STRIP - 1) / IM2COL_STRIP;
  const int ngrp = cols >> 3;
  const int g = threadIdx.x & (ngrp - 1);
  const int px0 = threadIdx.x / ngrp, pxs = blockDim.x / ngrp;
  int off[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = g * 8 + j;
    const int t = c / CIN, ci = c - t * CIN;
    off[j] = c < KCOLS ? (t / KW) * PITCH + (t % KW) * CIN + ci : -1;
  }
  const unsigned total = (unsigned)n * h * strips;
  for (unsigned b = blockIdx.x; b < total; b += gridDim.x) {
    const int sx = (int)(b % strips) * IM2COL_STRIP;
    const unsigned row = b / strips;
    const int yh = (int)(row % (unsigned)h);
    const long long img = row / (unsigned)h;
    __syncthreads();
    for (int i = threadIdx.x; i < KH * PITCH; i += blockDim.x) {
      const int r = i / PITCH, rem = i - r * PITCH;
      const int xo = rem / CIN;
      const int xx = sx - 1 + xo, yy = yh - 1 + r;
      patch[i] = (yy >= 0 && yy < h && xx >= 0 && xx < wd) ? __ldg(x + ((img * h + yy) * wd + xx) * CIN + (rem - xo * CIN)) : 0.f;
    }
    __syncthreads();
    for (int px = px0; px < IM2COL_STRIP && sx + px < wd; px += pxs) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = off[j] >= 0 ? patch[off[j] + px * CIN] : 0.f;
      st16(col + ((img * h + yh) * wd + sx + px) * cols + g * 8, pack8(v));
    }
  }
}

// ------------------------------------------------------------------------------------ stem wgrad
// grid = (pixel chunks, kh). Warp = one 8-channel group of dy, lane = pixel lane; each thread keeps
// kw*CIN*8 accumulators for filter row r, reduced across the warp with shuffles, then one fp32
// partial per chunk; a second kernel sums the chunks in order.
template <int CIN, int KW>
__global__ void stem_wgrad_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ dy, int dy_ld, int n,
                                  int h, int wd, int cout, int kh, long long ppb, float* __restrict__ part) {
  bsl::pdl_wait();
  const int lane = threadIdx.x & 31;
  const int cg = threadIdx.x >> 5;  // 8-channel group handled by this warp
  const int groups = cout / 8;
  const int r = blockIdx.y;
  const int ph = (kh - 1) / 2, pw = (KW - 1) / 2;
  const long long pixels = (long long)n * h * wd;
  const long long p0 = blockIdx.x * ppb, p1 = min(pixels, p0 + ppb);
  float acc[KW * CIN][8];
#pragma unroll
  for (int t = 0; t < KW * CIN; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[t][j] = 0.f;
  if (cg < groups) {
    for (long long p = p0 + lane; p < p1; p += 32) {
      const int xw = (int)(p % wd);
      const int yh = (int)((p / wd) % h);
      const int yy = yh + r - ph;
      if (yy < 0 || yy >= h) continue;
      float g[8];
      unpack8(ld16(dy + p * dy_ld + cg * 8), g);
      const float* xrow = x + (p + (long long)(r - ph) * wd - xw) * CIN;
#pragma unroll
      for (int s = 0; s < KW; ++s) {
        const int xx = xw + s - pw;
        if (xx < 0 || xx >= wd) continue;
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) {
          const float xv = __ldg(xrow + xx * CIN + ci);
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[s * CIN + ci][j] = fmaf(xv, g[j], acc[s * CIN + ci][j]);
        }
      }
    }
  }
#pragma unroll
  for (int t = 0; t < KW * CIN; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = acc[t][j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      acc[t][j] = v;
    }
  if (lane == 0 && cg < groups) {
    // part[chunk][r][s][ci][co]
    float* o = part + (((long long)blockIdx.x * kh + r) * KW * CIN) * cout + cg * 8;
#pragma unroll
    for (int t = 0; t < KW * CIN; ++t)
#pragma unroll
      for (int j = 0; j < 8; ++j) o[(long long)t * cout + j] = acc[t][j];
  }
}

// One warp per output: lane l adds chunks l, l + 32, ... in order (fp64), then a fixed xor tree over the lanes.
__global__ void sum_chunks_kernel(const float* __restrict__ part, int chunks, int n, float* __restrict__ out) {
  bsl::pdl_wait();
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= n) return;   // warp-uniform
  double s = 0.0;
  for (int b = lane; b < chunks; b += 32) s += (double)part[(long long)b * n + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[i] = (float)s;
}

// ---------------------------------------------------------------------------------- logits (1x1)
// cin/8 lanes per pixel: 16 B coalesced loads, partial dot products, shuffle-reduce over the lanes.
template <int COUT>
__global__ void head_fprop_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, const float* __restrict__ w,
                                  const float* __restrict__ bias, float* __restrict__ y, long long pixels, int cin) {
  bsl::pdl_wait();
  extern __shared__ float sw[];  // [cin][COUT]
  for (int i = threadIdx.x; i < cin * COUT; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const int cg = cin / 8;  // power of two <= 32
  const int g = threadIdx.x % cg;
  float wr[8][COUT];       // this lane's 8 input channels: constant for the whole launch (blockDim % cg == 0)
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int k = 0; k < COUT; ++k) wr[j][k] = sw[(g * 8 + j) * COUT + k];
  const long long ppb = blockDim.x / cg;                  // pixels per block per iteration
  const long long stride = (long long)gridDim.x * ppb;
  constexpr int U = 4;                                    // independent 16 B loads in flight per thread
  for (long long p0 = blockIdx.x * ppb + threadIdx.x / cg; p0 < pixels; p0 += U * stride) {
    uint4 raw[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long p = p0 + u * stride;
      raw[u] = p < pixels ? ld16(x + p * x_ld + g * 8) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long p = p0 + u * stride;
      float v[8], acc[COUT];
      unpack8(raw[u], v);
#pragma unroll
      for (int k = 0; k < COUT; ++k) acc[k] = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int k = 0; k < COUT; ++k) acc[k] = fmaf(v[j], wr[j][k], acc[k]);
#pragma unroll
      for (int k = 0; k < COUT; ++k)
        for (int o = cg >> 1; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
      if (p < pixels && g == 0) {
#pragma unroll
        for (int k = 0; k < COUT; ++k) y[p * COUT + k] = acc[k] + (bias ? bias[k] : 0.f);
      }
    }
  }
}

template <int COUT>
__global__ void head_dgrad_kernel(const float* __restrict__ dl, const float* __restrict__ w,
                                  __nv_bfloat16* __restrict__ dx, int dx_ld, long long pixels, int cin) {
  bsl::pdl_wait();
  extern __shared__ float sw[];
  for (int i = threadIdx.x; i < cin * COUT; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const int cg = cin / 8;
  const int g = threadIdx.x % cg;
  float wr[8][COUT];
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int k = 0; k < COUT; ++k) wr[j][k] = sw[(g * 8 + j) * COUT + k];
  const long long ppb = blockDim.x / cg;
  const long long stride = (long long)gridDim.x * ppb;
  constexpr int U = 4;
  for (long long p0 = blockIdx.x * ppb + threadIdx.x / cg; p0 < pixels; p0 += U * stride) {
    float d[U][COUT];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long p = p0 + u * stride;
#pragma unroll
      for (int k = 0; k < COUT; ++k) d[u][k] = p < pixels ? __ldg(dl + p * COUT + k) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long p = p0 + u * stride;
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < COUT; ++k) s = fmaf(d[u][k], wr[j][k], s);
        o[j] = s;
      }
      if (p < pixels) st16(dx + p * dx_ld + g * 8, pack8(o));
    }
  }
}

template <int COUT>
struct HeadWgradF {
  static constexpr int K = COUT, NIN = 2, UNROLL = 4;
  struct State {};
  const __nv_bfloat16* x;
  const float* dl;
  int ld;
  __device__ void init(State&, int, int) const {}
  // raw[1] carries the COUT (<= 4) fp32 dlogits of the pixel
  __device__ void load(long long p, int ch0, uint4 (&raw)[2]) const {
    raw[0] = ld16(x + p * ld + ch0);
    float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < COUT; ++k) d[k] = __ldg(dl + p * COUT + k);
    raw[1] = make_uint4(__float_as_uint(d[0]), __float_as_uint(d[1]), __float_as_uint(d[2]), __float_as_uint(d[3]));
  }
  __device__ void accum(const State&, long long, const uint4 (&raw)[2], float (&acc)[COUT][8]) const {
    float v[8];
    unpack8(raw[0], v);
    const float d[4] = {__uint_as_float(raw[1].x), __uint_as_float(raw[1].y), __uint_as_float(raw[1].z),
                        __uint_as_float(raw[1].w)};
#pragma unroll
    for (int k = 0; k < COUT; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[k][j] = fmaf(v[j], d[k], acc[k][j]);
  }
};

// sums[k*cin + c] (fp64) -> dw[c*COUT + k] (fp32, [1,1,cin,cout] = HWIO)
__global__ void head_wgrad_finish_kernel(const double* __restrict__ sums, float* __restrict__ dw, int cin, int cout) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cin * cout) return;
  const int c = i / cout, k = i - c * cout;
  dw[i] = (float)sums[(long long)k * cin + c];
}

// column sums of a dense fp32 [rows][cols] matrix, cols <= 8 (bias gradient of the logits layer)
__global__ void colsum_partial_kernel(const float* __restrict__ a, long long rows, int cols, long long rpb,
                                      float* __restrict__ part) {
  bsl::pdl_wait();
  __shared__ float sm[8][8];  // [warp][col]
  const long long r0 = blockIdx.x * rpb, r1 = min(rows, r0 + rpb);
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (long long r = r0 + threadIdx.x; r < r1; r += blockDim.x)
    for (int k = 0; k < cols; ++k) acc[k] += a[r * cols + k];
  for (int k = 0; k < 8; ++k)
    for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0)
    for (int k = 0; k < 8; ++k) sm[warp][k] = acc[k];
  __syncthreads();
  if (threadIdx.x < cols) {
    float s = 0.f;
    for (int wv = 0; wv < (int)(blockDim.x >> 5); ++wv) s += sm[wv][threadIdx.x];
    part[(long long)blockIdx.x * cols + threadIdx.x] = s;
  }
}

unsigned ew_grid(bsl_ctx* ctx, long long items) {
  long long b = (items + 255) / 256;
  const long long cap = 16LL * ctx->sm_count;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

int check_small(bsl_ctx* ctx, const bsl_conv2d_desc* d) {
  if (!ctx) return BSL_EINVAL;
  if (!d) return bsl_fail(ctx, BSL_EINVAL, "small conv: null descriptor");
  if (d->n <= 0 || d->h <= 0 || d->w <= 0) return bsl_fail(ctx, BSL_EINVAL, "small conv: non-positive size");
  return BSL_OK;
}

}  // namespace

extern "C" {

int bsl_conv2d_stem_fprop(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* x, const float* w, void* y,
                          void* stream) {
  int rc = check_small(ctx, d);
  if (rc) return rc;
  if (!x || !w || !y) return bsl_fail(ctx, BSL_EINVAL, "stem_fprop: null buffer");
  if (d->cout % 16 || d->y_ld < d->cout || d->y_ld % 8 || d->kh != d->kw || (d->kh != 3 && d->kh != 1))
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "stem_fprop: cout=%d k=%dx%d", d->cout, d->kh, d->kw);
  const size_t smem = (size_t)d->kh * d->kw * d->cin * d->cout * sizeof(float);
  const long long items = (long long)d->n * d->h * d->w * (d->cout / 16);
  auto go = [&](auto kern) {
    bsl_launch(kern, dim3(ew_grid(ctx, items)), dim3(256), smem, as_stream(stream), x, w, reinterpret_cast<__nv_bfloat16*>(y), d->y_ld,
                                                                d->n, d->h, d->w, d->cout, d->kh, d->kw);
  };
  switch (d->cin) {
    case 1: go(stem_fprop_kernel<1>); break;
    case 2: go(stem_fprop_kernel<2>); break;
    case 3: go(stem_fprop_kernel<3>); break;
    case 4: go(stem_fprop_kernel<4>); break;
    case 5: go(stem_fprop_kernel<5>); break;
    default: return bsl_fail(ctx, BSL_EUNSUPPORTED, "stem_fprop: cin=%d (1..5)", d->cin);
  }
  BSL_LAUNCH_CHECK(ctx, "stem_fprop_kernel");
  return BSL_OK;
}

int bsl_stem_im2col_ld(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* x, void* col, int col_ld, void* stream) {
  int rc = check_small(ctx, d);
  if (rc) return rc;
  if (!x || !col) return bsl_fail(ctx, BSL_EINVAL, "stem_im2col: null buffer");
  if (d->kh * d->kw * d->cin > 64 || d->cin < 1)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "stem_im2col: kh*kw*cin = %d must be <= 64", d->kh * d->kw * d->cin);
  if ((col_ld != 32 && col_ld != 64) || d->kh * d->kw * d->cin > col_ld)
    return bsl_fail(ctx, BSL_EINVAL, "stem_im2col: col_ld = %d must be 32 or 64 and >= kh*kw*cin = %d", col_ld,
                    d->kh * d->kw * d->cin);
  const long long blocks = (long long)d->n * d->h * ((d->w + IM2COL_STRIP - 1) / IM2COL_STRIP);
  const size_t smem = (size_t)d->kh * (IM2COL_STRIP + d->kw - 1) * d->cin * sizeof(float);
  const long long cap = 16LL * ctx->sm_count;
  const dim3 grid((unsigned)(blocks < cap ? blocks : cap));
  auto colb = reinterpret_cast<__nv_bfloat16*>(col);
  auto go = [&](auto kern) { bsl_launch(kern, grid, dim3(256), 0, as_stream(stream), x, colb, d->n, d->h, d->w, col_ld); };
  if (d->kh == 3 && d->kw == 3 && blocks < 0x7fffffffLL) {
    switch (d->cin) {
      case 1: go(stem_im2col3_kernel<1>); break;
      case 2: go(stem_im2col3_kernel<2>); break;
      case 3: go(stem_im2col3_kernel<3>); break;
      case 4: go(stem_im2col3_kernel<4>); break;
      case 5: go(stem_im2col3_kernel<5>); break;
      case 6: go(stem_im2col3_kernel<6>); break;
      default: go(stem_im2col3_kernel<7>); break;
    }
  } else {
    bsl_launch(stem_im2col_kernel, grid, dim3(256), smem, as_stream(stream), x, colb, d->n, d->h, d->w, d->cin, d->kh,
               d->kw, col_ld);
  }
  BSL_LAUNCH_CHECK(ctx, "stem_im2col_kernel");
  return BSL_OK;
}

int bsl_stem_im2col(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* x, void* col, void* stream) {
  return bsl_stem_im2col_ld(ctx, d, x, col, 64, stream);
}

int bsl_conv2d_stem_wgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* x, const void* dy, float* dw,
                          void* stream) {
  int rc = check_small(ctx, d);
  if (rc) return rc;
  if (!x || !dy || !dw) return bsl_fail(ctx, BSL_EINVAL, "stem_wgrad: null buffer");
  if (d->cout % 8 || d->cout > 64 || d->kh != 3 || d->kw != 3)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "stem_wgrad: cout=%d (<=64) k=%dx%d (3x3)", d->cout, d->kh, d->kw);
  const long long pixels = (long long)d->n * d->h * d->w;
  long long chunks = (pixels + 4095) / 4096;
  const long long cap = 4LL * ctx->sm_count;
  if (chunks > cap) chunks = cap;
  const long long ppb = (pixels + chunks - 1) / chunks;
  const int nout = d->kh * d->kw * d->cin * d->cout;
  float* part = nullptr;
  rc = bsl_scratch(ctx, (size_t)chunks * nout * sizeof(float), &part, as_stream(stream));
  if (rc) return rc;
  const int threads = 32 * (d->cout / 8);
  auto go = [&](auto kern) {
    bsl_launch(kern, dim3(dim3((unsigned)chunks, d->kh)), dim3(threads), 0, as_stream(stream), 
        x, reinterpret_cast<const __nv_bfloat16*>(dy), d->y_ld, d->n, d->h, d->w, d->cout, d->kh, ppb, part);
  };
  switch (d->cin) {
    case 1: go(stem_wgrad_kernel<1, 3>); break;
    case 2: go(stem_wgrad_kernel<2, 3>); break;
    case 3: go(stem_wgrad_kernel<3, 3>); break;
    case 4: go(stem_wgrad_kernel<4, 3>); break;
    case 5: go(stem_wgrad_kernel<5, 3>); break;
    default: return bsl_fail(ctx, BSL_EUNSUPPORTED, "stem_wgrad: cin=%d (1..5)", d->cin);
  }
  BSL_LAUNCH_CHECK(ctx, "stem_wgrad_kernel");
  bsl_launch(sum_chunks_kernel, dim3((nout + 3) / 4), dim3(128), 0, as_stream(stream), part, (int)chunks, nout, dw);
  BSL_LAUNCH_CHECK(ctx, "sum_chunks_kernel");
  return BSL_OK;
}

#define HEAD_SWITCH(COUT_, CALL)                                   \
  switch (COUT_) {                                                 \
    case 2: { constexpr int CO = 2; CALL; } break;                 \
    case 3: { constexpr int CO = 3; CALL; } break;                 \
    case 4: { constexpr int CO = 4; CALL; } break;                 \
    default: return bsl_fail(ctx, BSL_EUNSUPPORTED, "head conv: classes=%d (2..4)", COUT_); \
  }

static int check_head(bsl_ctx* ctx, const bsl_conv2d_desc* d) {
  int rc = check_small(ctx, d);
  if (rc) return rc;
  const int cg = d->cin / 8;
  if (d->kh != 1 || d->kw != 1 || d->cin % 8 || cg > 32 || (cg & (cg - 1)) || d->x_ld < d->cin || d->x_ld % 8)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "head conv: 1x1 with cin in {8,16,...,256} (got k=%d cin=%d)", d->kh,
                    d->cin);
  return BSL_OK;
}

int bsl_conv2d_head_fprop(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const float* w, const float* bias,
                          float* logits, void* stream) {
  int rc = check_head(ctx, d);
  if (rc) return rc;
  if (!x || !w || !logits) return bsl_fail(ctx, BSL_EINVAL, "head_fprop: null buffer");
  const long long pixels = (long long)d->n * d->h * d->w;
  const size_t smem = (size_t)d->cin * d->cout * sizeof(float);
  HEAD_SWITCH(d->cout, (bsl_launch(head_fprop_kernel<CO>, dim3(ew_grid(ctx, pixels * (d->cin / 8))), dim3(256), smem, as_stream(stream), 
                           reinterpret_cast<const __nv_bfloat16*>(x), d->x_ld, w, bias, logits, pixels, d->cin)));
  BSL_LAUNCH_CHECK(ctx, "head_fprop_kernel");
  return BSL_OK;
}

int bsl_conv2d_head_dgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* dlogits, const float* w, void* dx,
                          void* stream) {
  int rc = check_head(ctx, d);
  if (rc) return rc;
  if (!dlogits || !w || !dx) return bsl_fail(ctx, BSL_EINVAL, "head_dgrad: null buffer");
  const long long pixels = (long long)d->n * d->h * d->w;
  const size_t smem = (size_t)d->cin * d->cout * sizeof(float);
  HEAD_SWITCH(d->cout, (bsl_launch(head_dgrad_kernel<CO>, dim3(ew_grid(ctx, pixels * (d->cin / 8))), dim3(256), smem, as_stream(stream), 
                           dlogits, w, reinterpret_cast<__nv_bfloat16*>(dx), d->x_ld, pixels, d->cin)));
  BSL_LAUNCH_CHECK(ctx, "head_dgrad_kernel");
  return BSL_OK;
}

int bsl_conv2d_head_wgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const float* dlogits, float* dw,
                          float* dbias, void* stream) {
  int rc = check_head(ctx, d);
  if (rc) return rc;
  if (!x || !dlogits || !dw) return bsl_fail(ctx, BSL_EINVAL, "head_wgrad: null buffer");
  const long long pixels = (long long)d->n * d->h * d->w;
  cudaStream_t s = as_stream(stream);
  // scratch layout: [level-1 partials | fp64 sums | colsum partials]
  ReducePlan p = plan_reduce(ctx, pixels, 1, d->cin, d->cout);
  const size_t off_sums = (p.scratch_bytes + 15) & ~(size_t)15;
  const size_t off_cols = off_sums + (size_t)d->cin * d->cout * sizeof(double);
  const int cblocks = 2 * ctx->sm_count;
  float* base = nullptr;
  rc = bsl_scratch(ctx, off_cols + (size_t)cblocks * d->cout * sizeof(float), &base, s);
  if (rc) return rc;
  double* sums = reinterpret_cast<double*>(reinterpret_cast<char*>(base) + off_sums);
  float* cpart = reinterpret_cast<float*>(reinterpret_cast<char*>(base) + off_cols);
  const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(x);
  HEAD_SWITCH(d->cout, (rc = run_pixel_reduce(ctx, HeadWgradF<CO>{xb, dlogits, d->x_ld}, pixels, 1, d->cin, sums, s)));
  if (rc) return rc;
  bsl_launch(head_wgrad_finish_kernel, dim3((d->cin * d->cout + 127) / 128), dim3(128), 0, s, sums, dw, d->cin, d->cout);
  BSL_LAUNCH_CHECK(ctx, "head_wgrad_finish_kernel");
  if (dbias) {
    const long long rpb = (pixels + cblocks - 1) / cblocks;
    bsl_launch(colsum_partial_kernel, dim3(cblocks), dim3(256), 0, s, dlogits, pixels, d->cout, rpb, cpart);
    BSL_LAUNCH_CHECK(ctx, "colsum_partial_kernel");
    bsl_launch(sum_chunks_kernel, dim3((d->cout + 3) / 4), dim3(128), 0, s, cpart, cblocks, d->cout, dbias);
    BSL_LAUNCH_CHECK(ctx, "sum_chunks_kernel");
  }
  return BSL_OK;
}

}  // extern "C"
