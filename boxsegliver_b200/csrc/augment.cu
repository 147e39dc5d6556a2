// Device-side input stage (SURVEY.md 8f rank 4): what the reference's tf.data map function does per training sample
// on the host CPU, as one HBM-bound pass over the decoded slices.
//   data_processing_train                              <- DataLoader/Liver/input_pipeline.py:243-284
//   guide variant (Gaussian sp_guide, flips of guide)  <- DataLoader/Liver/input_pipeline_g.py:357-412
//   random_noise / random_flip                         <- utils/image_ops.py:209-238,245-320
//   create_spatial_guide_2d                            <- utils/image_ops.py:396-434
// TF-1.13 kernel semantics restated (not visible in the repo): resize_bilinear(align_corners=True) computes
// in = i * (in_size - 1) / (out_size - 1) in fp32, lower = (int)in, upper = min(lower + 1, in_size - 1),
// top + (bottom - top) * y_lerp with top = tl + (tr - tl) * x_lerp; resize_nearest_neighbor(align_corners=True) takes
// min(roundf(i * scale), in_size - 1). Every fp32 operation below is a single rounded IEEE operation (no FMA
// contraction), so the oracle (oracle/input_ref.py, numpy float32) reproduces images and labels bit for bit.
// One thread per output pixel: reads the 4 neighbours of each slice, writes `channels` contiguous floats.
#include "internal.h"
#include "philox.cuh"

namespace {

struct Interp {
  int lo, hi;
  float lerp;
};

__device__ __forceinline__ Interp interp_axis(int i, int in_size, int out_size) {
  const float scale = out_size > 1 ? __fdiv_rn((float)(in_size - 1), (float)(out_size - 1)) : 0.f;
  const float in = __fmul_rn((float)i, scale);
  Interp r;
  r.lo = (int)in;
  r.hi = min(r.lo + 1, in_size - 1);
  r.lerp = __fsub_rn(in, (float)r.lo);
  return r;
}

__device__ __forceinline__ float lerp2(float tl, float tr, float bl, float br, float xl, float yl) {
  const float top = __fadd_rn(tl, __fmul_rn(__fsub_rn(tr, tl), xl));
  const float bot = __fadd_rn(bl, __fmul_rn(__fsub_rn(br, bl), xl));
  return __fadd_rn(top, __fmul_rn(__fsub_rn(bot, top), yl));
}

__device__ __forceinline__ int nearest_axis(int i, int in_size, int out_size) {
  const float scale = out_size > 1 ? __fdiv_rn((float)(in_size - 1), (float)(out_size - 1)) : 0.f;
  return min((int)roundf(__fmul_rn((float)i, scale)), in_size - 1);
}

__device__ __forceinline__ float guide_at(int yy, int xx, const float* ctr, const float* sd, int k, float min_std) {
  float best = 0.f;   // exp(.) > 0; the reference's reduce_max runs over k >= 1 centres
  for (int j = 0; j < k; ++j) {
    const float sy = fmaxf(sd[2 * j], min_std), sx = fmaxf(sd[2 * j + 1], min_std);
    const float dy = __fsub_rn((float)yy, ctr[2 * j]), dx = __fsub_rn((float)xx, ctr[2 * j + 1]);
    const float ty = __fdiv_rn(__fmul_rn(dy, dy), __fmul_rn(__fmul_rn(2.f, sy), sy));
    const float tx = __fdiv_rn(__fmul_rn(dx, dx), __fmul_rn(__fmul_rn(2.f, sx), sx));
    const float g = expf(-__fadd_rn(ty, tx));
    best = j == 0 ? g : fmaxf(best, g);
  }
  return best;
}

__global__ void input_stage_kernel(bsl_input_desc d, bsl_input_params p, const unsigned short* __restrict__ slices,
                                   const unsigned char* __restrict__ seg, float* __restrict__ images,
                                   int* __restrict__ labels, float* __restrict__ sp_guide) {
  bsl::pdl_wait();
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per = (long long)d.out_h * d.out_w;
  if (t >= per * d.n) return;
  const int i = (int)(t / per);
  const int rem = (int)(t - (long long)i * per);
  const int y = rem / d.out_w, x = rem - y * d.out_w;
  const int flip = p.flips ? p.flips[i] : 0;
  // the value written at (y, x) is the un-flipped result at (ys, xs)
  const int ys = (flip & 2) ? d.out_h - 1 - y : y;
  const int xs = (flip & 1) ? d.out_w - 1 - x : x;
  const int off_r = p.bbox[4 * i], off_c = p.bbox[4 * i + 1], ch = p.bbox[4 * i + 2], cw = p.bbox[4 * i + 3];
  const Interp iy = interp_axis(ys, ch, d.out_h), ix = interp_axis(xs, cw, d.out_w);
  const float cmin = p.clip[2 * i], cmax = p.clip[2 * i + 1];
  const float range = __fsub_rn(cmax, cmin);
  float* out = images + t * d.channels;
  for (int c = 0; c < d.channels; ++c) {
    const unsigned short* pl = slices + ((long long)i * d.channels + c) * d.src_h * d.src_w;
    const long long r0 = (long long)(off_r + iy.lo) * d.src_w + off_c, r1 = (long long)(off_r + iy.hi) * d.src_w + off_c;
    float v = lerp2((float)pl[r0 + ix.lo], (float)pl[r0 + ix.hi], (float)pl[r1 + ix.lo], (float)pl[r1 + ix.hi], ix.lerp,
                    iy.lerp);
    v = __fdiv_rn(__fsub_rn(fminf(fmaxf(v, cmin), cmax), cmin), range);
    if (d.noise_scale != 0.f) {
      const float s = fabsf(d.noise_scale);
      const unsigned long long e = (((unsigned long long)i * d.out_h + ys) * d.out_w + xs) * d.channels + c;
      const float u = bsl::philox_uniform(d.seed, d.offset, e);
      v = __fadd_rn(v, __fadd_rn(__fmul_rn(u, __fmul_rn(2.f, s)), -s));
      v = __fmul_rn(v, p.present ? (float)p.present[i * d.channels + c] : 1.f);   // no noise in empty slices
    }
    out[c] = v;
  }
  if (labels != nullptr) {
    const int ny = nearest_axis(ys, ch, d.out_h), nx = nearest_axis(xs, cw, d.out_w);
    const float sv = (float)seg[((long long)i * d.src_h + off_r + ny) * d.src_w + off_c + nx];
    labels[t] = (int)__fdiv_rn(sv, (float)p.lab_scale[i]);
  }
  if (sp_guide != nullptr) {
    const int k = p.n_centers ? p.n_centers[i] : 0;
    float g = 0.5f;   // no tumour in the slice: constant 0.5 (input_pipeline_g.py:388-389)
    if (k > 0) {
      const float* ctr = p.centers + (long long)i * d.max_centers * 2;
      const float* sd = p.stddevs + (long long)i * d.max_centers * 2;
      const float v = lerp2(guide_at(iy.lo, ix.lo, ctr, sd, k, d.min_std), guide_at(iy.lo, ix.hi, ctr, sd, k, d.min_std),
                            guide_at(iy.hi, ix.lo, ctr, sd, k, d.min_std), guide_at(iy.hi, ix.hi, ctr, sd, k, d.min_std),
                            ix.lerp, iy.lerp);
      g = __fadd_rn(__fdiv_rn(v, 2.f), 0.5f);
    }
    sp_guide[t] = g;
  }
}

}  // namespace

extern "C" int bsl_input_stage(bsl_ctx* ctx, const bsl_input_desc* d, const bsl_input_params* p, const void* slices_u16,
                               const void* seg_u8, float* images, int* labels, float* sp_guide, void* stream) {
  if (!ctx) return BSL_EINVAL;
  if (!d || !p) return bsl_fail(ctx, BSL_EINVAL, "input_stage: null descriptor");
  if (d->n <= 0 || d->channels <= 0 || d->channels > 8 || d->src_h <= 0 || d->src_w <= 0 || d->out_h <= 0 || d->out_w <= 0)
    return bsl_fail(ctx, BSL_EINVAL, "input_stage: n=%d channels=%d src=%dx%d out=%dx%d", d->n, d->channels, d->src_h,
                    d->src_w, d->out_h, d->out_w);
  if (!slices_u16 || !images || !p->bbox || !p->clip) return bsl_fail(ctx, BSL_EINVAL, "input_stage: null buffer");
  if (labels && (!seg_u8 || !p->lab_scale)) return bsl_fail(ctx, BSL_EINVAL, "input_stage: labels need seg and lab_scale");
  if (sp_guide && (!p->n_centers || !p->centers || !p->stddevs || d->max_centers <= 0))
    return bsl_fail(ctx, BSL_EINVAL, "input_stage: sp_guide needs centers, stddevs, n_centers");
  const long long total = (long long)d->n * d->out_h * d->out_w;
  const unsigned blocks = (unsigned)((total + 255) / 256);
  bsl_launch(input_stage_kernel, dim3(blocks), dim3(256), 0, as_stream(stream), *d, *p, reinterpret_cast<const unsigned short*>(slices_u16),
                                                            reinterpret_cast<const unsigned char*>(seg_u8), images, labels,
                                                            sp_guide);
  BSL_LAUNCH_CHECK(ctx, "input_stage_kernel");
  return BSL_OK;
}
