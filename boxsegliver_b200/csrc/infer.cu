// Forward-only consumers of the probabilities (SURVEY.md section 8 row a13), kept on the device:
//   test-time mirroring   <- run_TTA, entry/main_eval_3d.py:246-287 and entry/infer_2d.py:60-78
//                            (probs += flip(prob of the flipped input); avg = probs / count; argmax)
//   np.argmax(...).astype(uint8) <- evaluators/evaluator_liver.py:663
//   ConfusionMatrix.compute (integer tp / fp / tn / fn) <- loss_metrics.py:542-556
// fp32 adds and the division happen in the reference's order, so argmax of the average is bit-identical to numpy's
// given the same probabilities; counts are exact integers.
#include "internal.h"

namespace {

struct Dims {
  long long n;
  int d, h, w, c;
};

__device__ __forceinline__ long long flipped_index(const Dims& s, long long i, int axes) {
  long long t = i;
  const int ch = (int)(t % s.c); t /= s.c;
  int x = (int)(t % s.w); t /= s.w;
  int y = (int)(t % s.h); t /= s.h;
  int z = (int)(t % s.d);
  const long long img = t / s.d;
  if (axes & 1) x = s.w - 1 - x;
  if (axes & 2) y = s.h - 1 - y;
  if (axes & 4) z = s.d - 1 - z;
  return (((img * s.d + z) * s.h + y) * s.w + x) * s.c + ch;
}

// dst[i] = (accumulate ? dst[i] : 0) + src[flip(i)]
__global__ void flip_f32_kernel(Dims s, int axes, int accumulate, const float* __restrict__ src, float* __restrict__ dst) {
  bsl::pdl_wait();
  const long long total = s.n * s.d * s.h * s.w * s.c;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const float v = src[flipped_index(s, i, axes)];
    dst[i] = accumulate ? dst[i] + v : v;
  }
}

template <int C>
__global__ void tta_finalize_kernel(long long pixels, float count, const float* __restrict__ acc, float* __restrict__ avg,
                                    uint8_t* __restrict__ pred) {
  bsl::pdl_wait();
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < pixels; p += (long long)gridDim.x * blockDim.x) {
    float best = 0.f;
    int arg = 0;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const float v = acc[p * C + c] / count;
      if (avg) avg[p * C + c] = v;
      if (c == 0 || v > best) { best = v; arg = c; }   // strict '>' keeps the first maximum (numpy argmax)
    }
    pred[p] = (uint8_t)arg;
  }
}

// out[0..3] += tp, fp, tn, fn of test = (t == test_value, or t != 0 when test_value < 0) vs ref = (label == ref_value)
__global__ void confusion_kernel(long long n, const uint8_t* __restrict__ t, int test_value, const int* __restrict__ labels,
                                 int ref_value, unsigned long long* __restrict__ out) {
  bsl::pdl_wait();
  unsigned long long tp = 0, fp = 0, tn = 0, fn = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const bool a = test_value < 0 ? t[i] != 0 : t[i] == test_value;
    const bool b = labels[i] == ref_value;
    tp += a && b;
    fp += a && !b;
    tn += !a && !b;
    fn += !a && b;
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    tp += __shfl_xor_sync(0xffffffffu, tp, o);
    fp += __shfl_xor_sync(0xffffffffu, fp, o);
    tn += __shfl_xor_sync(0xffffffffu, tn, o);
    fn += __shfl_xor_sync(0xffffffffu, fn, o);
  }
  if ((threadIdx.x & 31) == 0) {   // integer atomics: the result does not depend on the order
    atomicAdd(out + 0, tp);
    atomicAdd(out + 1, fp);
    atomicAdd(out + 2, tn);
    atomicAdd(out + 3, fn);
  }
}

unsigned grid_for(bsl_ctx* ctx, long long items) {
  long long b = (items + 255) / 256;
  const long long cap = 16LL * ctx->sm_count;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

extern "C" {

int bsl_flip_f32(bsl_ctx* ctx, long long n, int d, int h, int w, int c, int axes, int accumulate, const float* src,
                 float* dst, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!src || !dst || src == dst) return bsl_fail(ctx, BSL_EINVAL, "flip_f32: null or aliased buffer");
  if (n <= 0 || d <= 0 || h <= 0 || w <= 0 || c <= 0 || axes < 0 || axes > 7)
    return bsl_fail(ctx, BSL_EINVAL, "flip_f32: bad shape or axes mask %d", axes);
  const Dims s{n, d, h, w, c};
  bsl_launch(flip_f32_kernel, dim3(grid_for(ctx, n * d * h * w * c)), dim3(256), 0, as_stream(stream), s, axes, accumulate, src, dst);
  BSL_LAUNCH_CHECK(ctx, "flip_f32_kernel");
  return BSL_OK;
}

int bsl_tta_finalize(bsl_ctx* ctx, long long pixels, int classes, int count, const float* acc, float* avg_prob,
                     uint8_t* pred, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!acc || !pred || pixels <= 0 || count <= 0) return bsl_fail(ctx, BSL_EINVAL, "tta_finalize: bad argument");
  const unsigned g = grid_for(ctx, pixels);
  cudaStream_t s = as_stream(stream);
  switch (classes) {
    case 2: bsl_launch(tta_finalize_kernel<2>, dim3(g), dim3(256), 0, s, pixels, (float)count, acc, avg_prob, pred); break;
    case 3: bsl_launch(tta_finalize_kernel<3>, dim3(g), dim3(256), 0, s, pixels, (float)count, acc, avg_prob, pred); break;
    case 4: bsl_launch(tta_finalize_kernel<4>, dim3(g), dim3(256), 0, s, pixels, (float)count, acc, avg_prob, pred); break;
    default: return bsl_fail(ctx, BSL_EUNSUPPORTED, "tta_finalize: classes=%d (2..4)", classes);
  }
  BSL_LAUNCH_CHECK(ctx, "tta_finalize_kernel");
  return BSL_OK;
}

int bsl_confusion_counts(bsl_ctx* ctx, long long n, const uint8_t* test, int test_value, const int* labels, int ref_value,
                         unsigned long long* counts4, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!test || !labels || !counts4 || n <= 0) return bsl_fail(ctx, BSL_EINVAL, "confusion_counts: bad argument");
  bsl_launch(confusion_kernel, dim3(grid_for(ctx, n)), dim3(256), 0, as_stream(stream), n, test, test_value, labels, ref_value, counts4);
  BSL_LAUNCH_CHECK(ctx, "confusion_kernel");
  return BSL_OK;
}

}  // extern "C"
