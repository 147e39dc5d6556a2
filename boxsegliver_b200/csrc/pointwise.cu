// Small HBM-bound helpers: dtype casts, in-place scaling, per-channel sums (bias gradients).
// Vectorised and coalesced along the NHWC channel axis; reductions are two-level with a fixed
// order (reduce.cuh), so results are bit-reproducible run to run.
#include <cuda_bf16.h>
#include "reduce.cuh"

namespace {

constexpr int kThreads = 256;

inline unsigned grid_for(long long work, int per_block, int cap) {
  long long b = (work + per_block - 1) / per_block;
  if (b < 1) b = 1;
  if (b > cap) b = cap;
  return (unsigned)b;
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                     size_t n) {
  bsl::pdl_wait();
  size_t i = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) * 4;
  const size_t stride = (size_t)gridDim.x * blockDim.x * 4;
  for (; i + 3 < n; i += stride) {
    float4 v = *reinterpret_cast<const float4*>(src + i);
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 o = make_uint2(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b));
    *reinterpret_cast<uint2*>(dst + i) = o;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (size_t j = n & ~(size_t)3; j < n; ++j) dst[j] = __float2bfloat16_rn(src[j]);
}

__global__ void cast_bf16_f32_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst,
                                     size_t n) {
  bsl::pdl_wait();
  size_t i = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) * 4;
  const size_t stride = (size_t)gridDim.x * blockDim.x * 4;
  for (; i + 3 < n; i += stride) {
    uint2 v = *reinterpret_cast<const uint2*>(src + i);
    __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&v.x), b = *reinterpret_cast<__nv_bfloat162*>(&v.y);
    float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
    *reinterpret_cast<float4*>(dst + i) = make_float4(fa.x, fa.y, fb.x, fb.y);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (size_t j = n & ~(size_t)3; j < n; ++j) dst[j] = __bfloat162float(src[j]);
}

__global__ void scale_f32_kernel(float* __restrict__ x, size_t n, float a) {
  bsl::pdl_wait();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    x[i] *= a;
}

// Filter re-layout by index table (UNet3D pixel-pair packing, unet3d_engine.py): dst[i] = bf16(src[idx[i]]) or 0.
__global__ void gather_f32_bf16_kernel(const float* __restrict__ src, const int* __restrict__ idx, size_t n,
                                       __nv_bfloat16* __restrict__ dst) {
  bsl::pdl_wait();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int j = idx[i];
    dst[i] = __float2bfloat16_rn(j >= 0 ? src[j] : 0.f);
  }
}

// ... and its adjoint for the gradient: dst[j] = src[idx2[j][0]] + src[idx2[j][1]] (negative index: no term).
__global__ void gather_add2_f32_kernel(const float* __restrict__ src, const int* __restrict__ idx2, size_t n,
                                       float* __restrict__ dst) {
  bsl::pdl_wait();
  for (size_t j = blockIdx.x * (size_t)blockDim.x + threadIdx.x; j < n; j += (size_t)gridDim.x * blockDim.x) {
    const int a = idx2[2 * j], b = idx2[2 * j + 1];
    dst[j] = (a >= 0 ? src[a] : 0.f) + (b >= 0 ? src[b] : 0.f);
  }
}

// Statistics of a pixel-pair packed tensor: the conv epilogue sums over 2 * c "super" channels (voxel parity, lane);
// the real channel's moments are the sum of its two halves. src [groups][2][2c] -> dst [groups][2][c].
__global__ void fold_pair_sums_kernel(const double* __restrict__ src, int total, int c, double* __restrict__ dst) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int row = i / c, ch = i - row * c;
  dst[i] = src[(long long)row * 2 * c + ch] + src[(long long)row * 2 * c + c + ch];
}

struct SumF {
  static constexpr int K = 1, NIN = 1, UNROLL = 8;
  struct State {};
  const __nv_bfloat16* x;
  int ld;
  __device__ void init(State&, int, int) const {}
  __device__ void load(long long p, int ch0, uint4 (&raw)[1]) const { raw[0] = bsl::ld16(x + p * ld + ch0); }
  __device__ void accum(const State&, long long, const uint4 (&raw)[1], float (&acc)[1][8]) const {
    float v[8];
    bsl::unpack8(raw[0], v);
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[0][j] += v[j];
  }
};

// ReluGrad fused with the BiasAddGrad that follows it (transposed conv: y = relu(convT(x) + b)): one pass writes
// dy * (y > 0) and accumulates its per-channel sum; same reduction plan and order as SumF over the written tensor.
struct ReluBiasF {
  static constexpr int K = 1, NIN = 2, UNROLL = 4;
  struct State {};
  const __nv_bfloat16* y;
  const __nv_bfloat16* dy;
  __nv_bfloat16* out;
  int y_ld, dy_ld, o_ld;
  __device__ void init(State&, int, int) const {}
  __device__ void load(long long p, int ch0, uint4 (&raw)[2]) const {
    raw[0] = bsl::ld16(y + p * y_ld + ch0);
    raw[1] = bsl::ld16(dy + p * dy_ld + ch0);
  }
  __device__ void accum(const State&, long long p, const uint4 (&raw)[2], float (&acc)[1][8]) const {
    float v[8], g[8];
    bsl::unpack8(raw[0], v);
    bsl::unpack8(raw[1], g);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      g[j] = v[j] > 0.f ? g[j] : 0.f;
      acc[0][j] += g[j];
    }
    // this thread's channel group, as pixel_reduce_kernel assigns it (threadIdx.x % (c / 8))
    bsl::st16(out + p * o_ld + (threadIdx.x % cg) * 8, bsl::pack8(g));
  }
  int cg;
};

__global__ void f64_to_f32_kernel(const double* __restrict__ src, float* __restrict__ dst, int n) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (float)src[i];
}

}  // namespace

int bsl_channel_sum_bf16(bsl_ctx* ctx, const void* x, long long pixels, int c, int ld, float* out,
                         cudaStream_t stream) {
  // fp64 second level lands in the tail of the scratch arena, then narrows to fp32.
  SumF f{reinterpret_cast<const __nv_bfloat16*>(x), ld};
  bsl::ReducePlan p = bsl::plan_reduce(ctx, pixels, 1, c, 1);
  float* base = nullptr;
  int rc = bsl::bsl_scratch(ctx, p.scratch_bytes + (size_t)c * sizeof(double) + 16, &base, stream);
  if (rc) return rc;
  double* tmp = reinterpret_cast<double*>(reinterpret_cast<char*>(base) + ((p.scratch_bytes + 15) & ~(size_t)15));
  rc = bsl::run_pixel_reduce(ctx, f, pixels, 1, c, tmp, stream);
  if (rc) return rc;
  bsl_launch(f64_to_f32_kernel, dim3((c + 127) / 128), dim3(128), 0, stream, tmp, out, c);
  BSL_LAUNCH_CHECK(ctx, "f64_to_f32_kernel");
  return BSL_OK;
}

namespace {
// ReluBiasF with 4 channels (8 bytes) per thread: 3 streams need the extra resident threads (norm.cu, the
// normalisation-backward kernels). Partials [block][c] -> pixel_reduce_final_kernel (fixed order) -> fp32.
template <int U>
__global__ void __launch_bounds__(256, 4)
relu_bwd_bias4_kernel(const __nv_bfloat16* __restrict__ y, int y_ld, const __nv_bfloat16* __restrict__ dy, int dy_ld,
                      __nv_bfloat16* __restrict__ out, int o_ld, int c, long long pixels, long long ppb,
                      float* __restrict__ part) {
  bsl::pdl_wait();
  extern __shared__ float sm[];   // [rows][c]
  const int cg = c / 4;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg, r = threadIdx.x / cg;
  const int ch0 = g * 4;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  auto one = [&](const uint2& ry, const uint2& rd, long long p) {
    const __nv_bfloat162* hy = reinterpret_cast<const __nv_bfloat162*>(&ry);
    const __nv_bfloat162* hd = reinterpret_cast<const __nv_bfloat162*>(&rd);
    uint2 o2;
    __nv_bfloat162* ho = reinterpret_cast<__nv_bfloat162*>(&o2);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float2 v = __bfloat1622float2(hy[h]);
      float2 d = __bfloat1622float2(hd[h]);
      d.x = v.x > 0.f ? d.x : 0.f;
      d.y = v.y > 0.f ? d.y : 0.f;
      acc[2 * h] += d.x;
      acc[2 * h + 1] += d.y;
      ho[h] = __floats2bfloat162_rn(d.x, d.y);
    }
    *reinterpret_cast<uint2*>(out + p * o_ld + ch0) = o2;
  };
  if (r < rows) {
    const long long p0 = blockIdx.x * ppb, p1 = min(pixels, p0 + ppb);
    long long p = p0 + r;
    for (; p + (long long)(U - 1) * rows < p1; p += (long long)U * rows) {
      uint2 ry[U], rd[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        ry[u] = *reinterpret_cast<const uint2*>(y + (p + (long long)u * rows) * y_ld + ch0);
        rd[u] = *reinterpret_cast<const uint2*>(dy + (p + (long long)u * rows) * dy_ld + ch0);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) one(ry[u], rd[u], p + (long long)u * rows);
    }
    for (; p < p1; p += rows)
      one(*reinterpret_cast<const uint2*>(y + p * y_ld + ch0), *reinterpret_cast<const uint2*>(dy + p * dy_ld + ch0), p);
#pragma unroll
    for (int j = 0; j < 4; ++j) sm[r * c + ch0 + j] = acc[j];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < c; i += blockDim.x) {
    float t = 0.f;
    for (int rr = 0; rr < rows; ++rr) t += sm[rr * c + i];
    part[(long long)blockIdx.x * c + i] = t;
  }
}
}  // namespace

namespace bsl {
__global__ void __launch_bounds__(1024) pixel_reduce_final_kernel(const float* __restrict__ part, int blocks, int kc,
                                                                  double* __restrict__ out);
}

extern "C" int bsl_relu_bwd_bias(bsl_ctx* ctx, long long pixels, int c, const void* y, int y_ld, const void* dy,
                                 int dy_ld, void* out, int out_ld, float* dbias, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!y || !dy || !out || !dbias) return bsl_fail(ctx, BSL_EINVAL, "relu_bwd_bias: null buffer");
  if (c % 8 || y_ld % 8 || dy_ld % 8 || out_ld % 8) return bsl_fail(ctx, BSL_EUNSUPPORTED, "relu_bwd_bias: c%%8");
  cudaStream_t s = as_stream(stream);
  if (c <= 1024 && 256 % (c / 4) == 0) {
    const int cg = c / 4, rows = 256 / cg;
    long long want = (pixels * c + 32767) / 32768;
    const long long cap = 8LL * ctx->sm_count;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    const int blocks = (int)want;
    const long long ppb = (pixels + blocks - 1) / blocks;
    float* base = nullptr;
    const size_t pbytes = ((size_t)blocks * c * sizeof(float) + 15) & ~(size_t)15;
    int rc = bsl::bsl_scratch(ctx, pbytes + (size_t)c * sizeof(double) + 16, &base, s);
    if (rc) return rc;
    double* tmp = reinterpret_cast<double*>(reinterpret_cast<char*>(base) + pbytes);
    bsl_launch(relu_bwd_bias4_kernel<4>, dim3(blocks), dim3(rows * cg), (size_t)rows * c * sizeof(float), s, 
        reinterpret_cast<const __nv_bfloat16*>(y), y_ld, reinterpret_cast<const __nv_bfloat16*>(dy), dy_ld,
        reinterpret_cast<__nv_bfloat16*>(out), out_ld, c, pixels, ppb, base);
    BSL_LAUNCH_CHECK(ctx, "relu_bwd_bias4_kernel");
    bsl_launch(bsl::pixel_reduce_final_kernel, dim3(dim3((c + 31) / 32, 1)), dim3(1024), 0, s, base, blocks, c, tmp);
    BSL_LAUNCH_CHECK(ctx, "pixel_reduce_final_kernel");
    bsl_launch(f64_to_f32_kernel, dim3((c + 127) / 128), dim3(128), 0, s, tmp, dbias, c);
    BSL_LAUNCH_CHECK(ctx, "f64_to_f32_kernel");
    return BSL_OK;
  }
  ReluBiasF f{reinterpret_cast<const __nv_bfloat16*>(y), reinterpret_cast<const __nv_bfloat16*>(dy),
              reinterpret_cast<__nv_bfloat16*>(out), y_ld, dy_ld, out_ld, c / 8};
  bsl::ReducePlan p = bsl::plan_reduce(ctx, pixels, 1, c, 1);
  float* base = nullptr;
  int rc = bsl::bsl_scratch(ctx, p.scratch_bytes + (size_t)c * sizeof(double) + 16, &base, s);
  if (rc) return rc;
  double* tmp = reinterpret_cast<double*>(reinterpret_cast<char*>(base) + ((p.scratch_bytes + 15) & ~(size_t)15));
  rc = bsl::run_pixel_reduce(ctx, f, pixels, 1, c, tmp, s);
  if (rc) return rc;
  bsl_launch(f64_to_f32_kernel, dim3((c + 127) / 128), dim3(128), 0, s, tmp, dbias, c);
  BSL_LAUNCH_CHECK(ctx, "f64_to_f32_kernel");
  return BSL_OK;
}

extern "C" {

int bsl_scale_f32(bsl_ctx* ctx, float* x, size_t n, float a, void* stream) {
  if (!ctx || !x) return BSL_EINVAL;
  if (n == 0) return BSL_OK;
  bsl_launch(scale_f32_kernel, dim3(grid_for((long long)n, kThreads, 8 * ctx->sm_count)), dim3(kThreads), 0, as_stream(stream), x, n, a);
  BSL_LAUNCH_CHECK(ctx, "scale_f32_kernel");
  return BSL_OK;
}

int bsl_gather_f32_bf16(bsl_ctx* ctx, const float* src, const int* idx, size_t n, void* dst_bf16, void* stream) {
  if (!ctx || !src || !idx || !dst_bf16) return BSL_EINVAL;
  if (n == 0) return BSL_OK;
  bsl_launch(gather_f32_bf16_kernel, dim3(grid_for((long long)n, kThreads, 8 * ctx->sm_count)), dim3(kThreads), 0,
             as_stream(stream), src, idx, n, reinterpret_cast<__nv_bfloat16*>(dst_bf16));
  BSL_LAUNCH_CHECK(ctx, "gather_f32_bf16_kernel");
  return BSL_OK;
}

int bsl_gather_add2_f32(bsl_ctx* ctx, const float* src, const int* idx2, size_t n, float* dst, void* stream) {
  if (!ctx || !src || !idx2 || !dst) return BSL_EINVAL;
  if (n == 0) return BSL_OK;
  bsl_launch(gather_add2_f32_kernel, dim3(grid_for((long long)n, kThreads, 8 * ctx->sm_count)), dim3(kThreads), 0,
             as_stream(stream), src, idx2, n, dst);
  BSL_LAUNCH_CHECK(ctx, "gather_add2_f32_kernel");
  return BSL_OK;
}

int bsl_fold_pair_sums(bsl_ctx* ctx, const double* src, int groups, int c, double* dst, void* stream) {
  if (!ctx || !src || !dst || groups < 1 || c < 1) return BSL_EINVAL;
  const int total = groups * 2 * c;
  bsl_launch(fold_pair_sums_kernel, dim3((total + 127) / 128), dim3(128), 0, as_stream(stream), src, total, c, dst);
  BSL_LAUNCH_CHECK(ctx, "fold_pair_sums_kernel");
  return BSL_OK;
}

int bsl_cast_f32_to_bf16(bsl_ctx* ctx, const float* src, void* dst, size_t n, void* stream) {
  if (!ctx || !src || !dst) return BSL_EINVAL;
  bsl_launch(cast_f32_bf16_kernel, dim3(grid_for((long long)n, kThreads * 4, 8 * ctx->sm_count)), dim3(kThreads), 0, as_stream(stream), src, reinterpret_cast<__nv_bfloat16*>(dst), n);
  BSL_LAUNCH_CHECK(ctx, "cast_f32_bf16_kernel");
  return BSL_OK;
}

int bsl_cast_bf16_to_f32(bsl_ctx* ctx, const void* src, float* dst, size_t n, void* stream) {
  if (!ctx || !src || !dst) return BSL_EINVAL;
  bsl_launch(cast_bf16_f32_kernel, dim3(grid_for((long long)n, kThreads * 4, 8 * ctx->sm_count)), dim3(kThreads), 0, as_stream(stream), reinterpret_cast<const __nv_bfloat16*>(src), dst, n);
  BSL_LAUNCH_CHECK(ctx, "cast_bf16_f32_kernel");
  return BSL_OK;
}

}  // extern "C"
