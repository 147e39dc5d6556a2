// Deterministic per-channel reductions over the pixels of an NHWC bf16 tensor.
//
// Thread layout inside a block: (pixel row r, 8-channel group g) with g fastest, so a warp reads
// whole 128 B+ runs of consecutive channels (16 B per thread). Level 1 leaves one fp32 partial per
// (group, block, k, channel) in scratch; level 2 sums the blocks in a fixed order in fp64.
// No float atomics anywhere: results are bit-reproducible.
#pragma once
#include <cuda_bf16.h>
#include <cstdlib>
#include "internal.h"

namespace bsl {

constexpr int kReduceThreads = 256;

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float2 t = __bfloat1622float2(h[j]);
    f[2 * j] = t.x;
    f[2 * j + 1] = t.y;
  }
}

__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 v;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
  return v;
}

__device__ __forceinline__ uint4 ld16(const __nv_bfloat16* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void st16(__nv_bfloat16* p, const uint4& v) { *reinterpret_cast<uint4*>(p) = v; }

// F must provide: static constexpr int K; a nested `struct State` of per-thread registers;
//   __device__ void init(State&, int group, int ch0) const          -- hoists per-channel parameters
//   __device__ void load(long long pixel, int ch0, uint4 (&raw)[NIN]) const, with static constexpr int NIN
//   __device__ void accum(const State&, long long pixel, const uint4 (&raw)[NIN], float (&acc)[K][8]) const
// Loads of UNROLL pixels are issued before any is consumed (memory-level parallelism).
template <class F, int UNROLL>
__global__ void pixel_reduce_kernel(F f, long long pixels_per_group, long long ppb, int c,
                                    float* __restrict__ part) {
  bsl::pdl_wait();
  extern __shared__ float sm[];  // [rows][K][c]
  constexpr int K = F::K;
  constexpr int NIN = F::NIN;
  const int cg = c / 8;
  const int rows = blockDim.x / cg;
  const int g = threadIdx.x % cg;
  const int r = threadIdx.x / cg;
  const int group = blockIdx.y;
  float acc[K][8];
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[k][j] = 0.f;
  if (r < rows) {
    typename F::State st;
    f.init(st, group, g * 8);
    const long long p0 = blockIdx.x * ppb;
    const long long p1 = min(pixels_per_group, p0 + ppb);
    const long long base = (long long)group * pixels_per_group;
    long long p = p0 + r;
    for (; p + (long long)(UNROLL - 1) * rows < p1; p += (long long)UNROLL * rows) {
      uint4 raw[UNROLL][NIN];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) f.load(base + p + (long long)u * rows, g * 8, raw[u]);
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) f.accum(st, base + p + (long long)u * rows, raw[u], acc);
    }
    for (; p < p1; p += rows) {
      uint4 raw[NIN];
      f.load(base + p, g * 8, raw);
      f.accum(st, base + p, raw, acc);
    }
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) sm[(r * K + k) * c + g * 8 + j] = acc[k][j];
  }
  __syncthreads();
  float* out = part + ((long long)group * gridDim.x + blockIdx.x) * K * c;
  for (int i = threadIdx.x; i < K * c; i += blockDim.x) {
    float s = 0.f;
    for (int rr = 0; rr < rows; ++rr) s += sm[rr * K * c + i];
    out[i] = s;
  }
}

// out[group][i] = sum_b part[group][b][i], i in [0, kc), fp64 accumulation in block order.
__global__ void __launch_bounds__(1024) pixel_reduce_final_kernel(const float* __restrict__ part, int blocks, int kc,
                                          double* __restrict__ out);

struct ReducePlan {
  int threads, rows, blocks;
  long long ppb;
  size_t smem, scratch_bytes;
};

inline ReducePlan plan_reduce(bsl_ctx* ctx, long long pixels_per_group, int groups, int c, int K) {
  ReducePlan p;
  const int cg = c / 8;
  p.threads = kReduceThreads;   // c <= 2048 (checked by run_pixel_reduce): cg <= 256 channel groups
  p.rows = p.threads / cg;
  // keep K*c*rows*4 bytes of smem under 48 KB
  while ((size_t)p.rows * K * c * 4 > 48 * 1024 && p.rows > 1) p.rows /= 2;
  p.threads = p.rows * cg;
  // ~32 KB of every input per block (512 pixels at 64 channels), so wide layers with few pixels still fill the GPU
  long long want = (pixels_per_group * c + 32767) / 32768;
  long long cap = (4LL * ctx->sm_count + groups - 1) / groups;
  if (cap < 1) cap = 1;
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  p.blocks = (int)want;
  p.ppb = (pixels_per_group + p.blocks - 1) / p.blocks;
  p.smem = (size_t)p.rows * K * c * 4;
  p.scratch_bytes = (size_t)groups * p.blocks * K * c * 4;
  return p;
}

int bsl_scratch(bsl_ctx* ctx, size_t bytes, float** out, cudaStream_t stream);
int bsl_scratch_w(bsl_ctx* ctx, size_t bytes, void** out, cudaStream_t stream);

template <class F>
int run_pixel_reduce(bsl_ctx* ctx, const F& f, long long pixels_per_group, int groups, int c, double* out,
                     cudaStream_t stream) {
  if (c % 8 || c <= 0 || c > 2048) return bsl_fail(ctx, BSL_EUNSUPPORTED, "pixel reduce: c=%d (multiple of 8, <= 2048)", c);
  ReducePlan p = plan_reduce(ctx, pixels_per_group, groups, c, F::K);
  float* part = nullptr;
  int rc = bsl_scratch(ctx, p.scratch_bytes, &part, stream);
  if (rc) return rc;
  bsl_launch(pixel_reduce_kernel<F, F::UNROLL>, dim3(dim3(p.blocks, groups)), dim3(p.threads), p.smem, stream, f, pixels_per_group,
                                                                                          p.ppb, c, part);
  BSL_LAUNCH_CHECK(ctx, "pixel_reduce_kernel");
  const int kc = F::K * c;
  bsl_launch(pixel_reduce_final_kernel, dim3(dim3((kc + 31) / 32, groups)), dim3(1024), 0, stream, part, p.blocks, kc, out);
  BSL_LAUNCH_CHECK(ctx, "pixel_reduce_final_kernel");
  return BSL_OK;
}

}  // namespace bsl
