// Host side of the tcgen05 implicit-GEMM convolutions: builds the TMA tensor maps and the
// IgemmArgs for each reference op and launches igemm_kernel (igemm.cuh).
//   conv2d fprop / dgrad / wgrad  <- slim.conv2d, NetworksV2/UNet.py:79,85,94 (+ tf.gradients)
//   convT2d fwd / bwd             <- slim.conv2d_transpose, NetworksV2/UNet.py:91
#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>
#include "igemm.cuh"
#include "igemm_halo.cuh"
#include "internal.h"
#include "reduce.cuh"

using namespace bsl;

namespace {

int g_mn_lbo = 8192, g_mn_sbo = 1024, g_mn_kadv = 2048;
long long* g_dbg_waits = nullptr;   // device [1024][4], allocated by bsl_debug_set(ctx, 3, 1)

template <int MODE, bool B_MN, int BN, int STAGES>
int launch_one(bsl_ctx* ctx, const CUtensorMap& a, const CUtensorMap& b, const IgemmArgs& args_in, dim3 grid,
               cudaStream_t stream) {
  IgemmArgs args = args_in;
  args.mn_lbo = g_mn_lbo;
  args.mn_sbo = g_mn_sbo;
  args.mn_kadv = g_mn_kadv;
  auto kern = igemm_kernel<MODE, B_MN, BN, STAGES>;
  constexpr int smem = igemm_smem_bytes<BN, STAGES>();
  static bool configured = false;
  if (!configured) {
    BSL_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  bsl_launch(kern, dim3(grid), dim3(IGEMM_THREADS), smem, stream, a, b, args);
  BSL_LAUNCH_CHECK(ctx, "igemm_kernel launch");
  return BSL_OK;
}

// Stage counts keep two CTAs resident per SM for BN <= 128 (96 KB each) so one CTA's epilogue
// overlaps the other's main loop; BN = 256 takes the SM alone with a 4-deep ring.
template <int MODE, bool B_MN>
int launch_igemm(bsl_ctx* ctx, int bn, const CUtensorMap& a, const CUtensorMap& b, const IgemmArgs& args,
                 dim3 grid, cudaStream_t stream) {
  switch (bn) {
    case 64: return launch_one<MODE, B_MN, 64, 4>(ctx, a, b, args, grid, stream);
    case 128: return launch_one<MODE, B_MN, 128, 3>(ctx, a, b, args, grid, stream);
    case 256: return launch_one<MODE, B_MN, 256, 4>(ctx, a, b, args, grid, stream);
  }
  return bsl_fail(ctx, BSL_EUNSUPPORTED, "igemm: column tile %d", bn);
}

int pick_bn(int n) { return n % 256 == 0 ? 256 : (n % 128 == 0 ? 128 : 64); }

// Pixel box (w, h, n) with w*h*n == prod, widest along W first (coalesced 128 B rows either way).
void pick_box(int prod, int W, int H, int N, int* tw, int* th, int* tn) {
  int w = 1;
  while (w < 16 && w < W && w < prod) w <<= 1;
  int h = 1;
  while (w * h < prod && h < H) h <<= 1;
  *tw = w;
  *th = h;
  *tn = prod / (w * h);
  (void)N;
}

int cdiv(int a, int b) { return (a + b - 1) / b; }

void set_tiles(IgemmArgs& a, const int tdim[4], const int tbox[4]) {
  for (int d = 0; d < 4; ++d) {
    a.tdim[d] = tdim[d];
    a.tbox[d] = tbox[d];
    a.ntile[d] = cdiv(tdim[d], tbox[d]);
    a.istride[d] = 1;
  }
}

int nhwc_map(bsl_ctx* ctx, const void* base, int c, int w, int h, int n, int ld, const int box[4],
             CUtensorMap* out) {
  // ld < c: the rows hold only ld channels (narrow im2col matrix of the stem); the 64-wide box then reaches past
  // the innermost extent and TMA zero-fills channels >= ld in shared memory
  uint64_t dims[5] = {(uint64_t)(ld < c ? ld : c), (uint64_t)w, (uint64_t)h, (uint64_t)n, 1};
  uint64_t str[5] = {2, (uint64_t)ld * 2, (uint64_t)w * ld * 2, (uint64_t)h * w * ld * 2,
                     (uint64_t)n * h * w * ld * 2};
  uint32_t bx[5] = {64, (uint32_t)box[0], (uint32_t)box[1], (uint32_t)box[2], 1};
  return bsl_get_tmap(ctx, base, 5, dims, str, bx, out);
}

// [n, 2h, 2w, c] seen as (c, b:2, w, a:2, n*h): taps of a k2 s2 transposed conv become coordinates.
// c == 32 (UNet3D's 30-channel level stored with 32 lanes; the gradient tensor must be DENSE, ld == 32): the two column
// parities b of an input pixel are 64 contiguous values -- (b, c) pairs -- so the view is (64, 1, w, a:2, n*h) and a
// 64-wide reduction / row block is one row parity `a` of the filter. (A 32-wide box over a strided tensor does not work:
// with the 128-byte swizzle TMA does not pack two 64-byte inner rows into one 128-byte shared-memory row.)
int upsampled_map(bsl_ctx* ctx, const void* base, int c, int w, int h, int n, int ld, int tw, int th,
                  CUtensorMap* out) {
  uint64_t dims[5] = {(uint64_t)c, 2, (uint64_t)w, 2, (uint64_t)n * h};
  uint64_t str[5] = {2, (uint64_t)ld * 2, (uint64_t)2 * ld * 2, (uint64_t)2 * w * ld * 2,
                     (uint64_t)4 * w * ld * 2};
  uint32_t bx[5] = {64, 1, (uint32_t)tw, 1, (uint32_t)th};
  if (c == 32) {
    if (ld != 32) return bsl_fail(ctx, BSL_EUNSUPPORTED, "convT2d backward with cout = 32 needs a dense gradient (y_ld = 32, got %d)", ld);
    dims[0] = 64;
    dims[1] = 1;
  }
  return bsl_get_tmap(ctx, base, 5, dims, str, bx, out);
}

// [n, h, w, c] seen as (c, 1, w, 1, n*h) so it shares pixel coordinates with upsampled_map.
int rows_map(bsl_ctx* ctx, const void* base, int c, int w, int h, int n, int ld, int tw, int th,
             CUtensorMap* out) {
  uint64_t dims[5] = {(uint64_t)c, 1, (uint64_t)w, 1, (uint64_t)n * h};
  uint64_t str[5] = {2, (uint64_t)ld * 2, (uint64_t)ld * 2, (uint64_t)w * ld * 2, (uint64_t)w * ld * 2};
  uint32_t bx[5] = {64, 1, (uint32_t)tw, 1, (uint32_t)th};
  return bsl_get_tmap(ctx, base, 5, dims, str, bx, out);
}

int matrix_map(bsl_ctx* ctx, const void* base, int inner, int rows, int box_inner, int box_rows,
               CUtensorMap* out) {
  uint64_t dims[2] = {(uint64_t)inner, (uint64_t)rows};
  uint64_t str[2] = {2, (uint64_t)inner * 2};
  uint32_t bx[2] = {(uint32_t)box_inner, (uint32_t)box_rows};
  return bsl_get_tmap(ctx, base, 2, dims, str, bx, out);
}

int check_conv(bsl_ctx* ctx, const bsl_conv2d_desc* d, bool narrow_x_ok = false) {
  if (!ctx) return BSL_EINVAL;
  if (!d) return bsl_fail(ctx, BSL_EINVAL, "conv2d: null descriptor");
  if (d->n <= 0 || d->h <= 0 || d->w <= 0 || d->cin <= 0 || d->cout <= 0)
    return bsl_fail(ctx, BSL_EINVAL, "conv2d: non-positive size");
  if (!((d->kh == 3 && d->kw == 3) || (d->kh == 1 && d->kw == 1)))
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv2d: kernel %dx%d (3x3 or 1x1 only)", d->kh, d->kw);
  if (d->cin % 64 || d->cout % 64)
    return bsl_fail(ctx, BSL_EUNSUPPORTED,
                    "conv2d tcgen05 path needs cin,cout multiples of 64 (got %d,%d); use "
                    "bsl_conv2d_small_* for the stem / logits layers", d->cin, d->cout);
  const bool narrow = narrow_x_ok && d->kh == 1 && d->cin == 64 && d->x_ld >= 8;   // x_ld < cin: see bsl_conv2d_desc
  if ((d->x_ld < d->cin && !narrow) || d->y_ld < d->cout || d->x_ld % 8 || d->y_ld % 8)
    return bsl_fail(ctx, BSL_EINVAL, "conv2d: channel strides must be >= channels and multiples of 8");
  return BSL_OK;
}

void conv_taps(IgemmArgs& a, int kh, int kw) {
  a.ntaps = kh * kw;
  for (int r = 0; r < kh; ++r)
    for (int s = 0; s < kw; ++s) {
      signed char* o = a.tapoff[r * kw + s];
      o[0] = (signed char)(s - (kw - 1) / 2);  // TF SAME, stride 1: pad_before = (k-1)/2
      o[1] = (signed char)(r - (kh - 1) / 2);
      o[2] = 0;
      o[3] = 0;
    }
}

struct SplitPlan {
  int k_tiles, per, splits;
};

SplitPlan plan_split(bsl_ctx* ctx, int mn_tiles, int k_tiles) {
  // Aim for ~2 CTAs per SM in flight, but never fewer than 8 pixel tiles per split.
  int want = std::max(1, (2 * ctx->sm_count + mn_tiles - 1) / mn_tiles);
  int splits = std::max(1, std::min(want, k_tiles / 8));
  int per = cdiv(k_tiles, splits);
  splits = cdiv(k_tiles, per);
  return {k_tiles, per, splits};
}

__global__ void reduce_splits_kernel(const float* __restrict__ part, float* __restrict__ out, long long n,
                                     int splits) {
  bsl::pdl_wait();
  long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  float4 acc = *reinterpret_cast<const float4*>(part + i);
  for (int s = 1; s < splits; ++s) {  // fixed order => bit-reproducible
    float4 v = *reinterpret_cast<const float4*>(part + s * n + i);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  *reinterpret_cast<float4*>(out + i) = acc;
}

__global__ void reduce_splits_strided_kernel(const float* __restrict__ part, float* __restrict__ out, long long n,
                                             int splits, long long stride) {
  bsl::pdl_wait();
  long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  float4 acc = *reinterpret_cast<const float4*>(part + i);
  for (int s = 1; s < splits; ++s) {  // fixed order => bit-reproducible
    float4 v = *reinterpret_cast<const float4*>(part + s * stride + i);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  *reinterpret_cast<float4*>(out + i) = acc;
}

int reduce_splits_strided(bsl_ctx* ctx, const float* part, float* out, long long n, int splits, long long stride,
                          cudaStream_t s) {
  const int threads = 256;
  const long long blocks = (n / 4 + threads - 1) / threads;
  bsl_launch(reduce_splits_strided_kernel, dim3((unsigned)blocks), dim3(threads), 0, s, part, out, n, splits, stride);
  BSL_LAUNCH_CHECK(ctx, "reduce_splits_strided_kernel");
  return BSL_OK;
}

int reduce_splits(bsl_ctx* ctx, const float* part, float* out, long long n, int splits, cudaStream_t s) {
  int threads = 256;
  long long blocks = (n / 4 + threads - 1) / threads;
  bsl_launch(reduce_splits_kernel, dim3((unsigned)blocks), dim3(threads), 0, s, part, out, n, splits);
  BSL_LAUNCH_CHECK(ctx, "reduce_splits_kernel");
  return BSL_OK;
}


// ------------------------------------------------------------------ second-generation (halo-tile) kernels

template <int BN, int NSUB, bool B_MN, bool STATS, bool SCATTER, bool TMA_ST = false, bool BR = false>
int launch_halo_one(bsl_ctx* ctx, const CUtensorMap& a, const CUtensorMap& b, const ConvHaloArgs& args, int grid,
                    cudaStream_t stream, const CUtensorMap* o = nullptr) {
  auto kern = conv_halo_kernel<BN, NSUB, B_MN, STATS, SCATTER, false, TMA_ST, false, BR>;
  constexpr int smem = ConvHaloCfg<BN, NSUB, TMA_ST>::SMEM_BYTES;
  static bool configured = false;
  if (!configured) {
    BSL_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  bsl_launch(kern, dim3(grid), dim3(CH_THREADS), smem, stream, a, b, o ? *o : a, args);
  BSL_LAUNCH_CHECK(ctx, "conv_halo_kernel launch");
  return BSL_OK;
}

struct HaloPlan {
  int bn, nsub, n_ntiles, n_sub_total, n_units, grid, slots;
  int pair;   // planned for CTA pairs (pair_replan): 128-wide tiles over sub-tile pairs, plain epilogue
};

template <int BN, int NSUB, bool B_MN, bool STATS, bool SCATTER, bool BR = false>
int launch_halo_res_one(bsl_ctx* ctx, const CUtensorMap& a, const CUtensorMap& b, const ConvHaloArgs& args, int grid,
                        int smem, cudaStream_t stream) {
  auto kern = conv_halo_kernel<BN, NSUB, B_MN, STATS, SCATTER, true, false, false, BR>;
  static int configured = 0;
  if (configured < smem) {
    BSL_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = smem;
  }
  bsl_launch(kern, dim3(grid), dim3(CH_THREADS), smem, stream, a, b, a, args);
  BSL_LAUNCH_CHECK(ctx, "conv_halo_kernel (resident filter) launch");
  return BSL_OK;
}

// Resident-filter plan: returns false when the filter slice of one column tile does not fit beside >= 2
// activation stages. May lower nsub to 1 (the filter is no longer re-read per unit, so sharing it matters less).
constexpr int CH_DYN_BUDGET = 232448 - 10 * 1024;   // 227 KB minus static shared memory (barriers, statistics)
bool plan_resident(int bn, int ntaps, int cblocks, int* nsub, int* a_stages, int* smem) {
  if (bn > 128) return false;
  const int res = ntaps * cblocks * bn * 128;
  const int left = CH_DYN_BUDGET - 1024 - res;
  if (left <= 0) return false;
  const int s2 = std::min(CH_MAX_A_STAGES, left / (2 * CH_SUB_BYTES)), s1 = std::min(CH_MAX_A_STAGES, left / CH_SUB_BYTES);
  int ns, st;
  if (*nsub == 2 && s2 >= 3) { ns = 2; st = s2; }
  else if (s1 >= 3) { ns = 1; st = s1; }
  else if (*nsub == 2 && s2 >= 2) { ns = 2; st = s2; }
  else return false;
  *nsub = ns;
  *a_stages = st;
  *smem = st * ns * CH_SUB_BYTES + res + 1024;
  return true;
}

template <bool B_MN, bool STATS, bool SCATTER, bool BR = false>
int launch_halo_res(bsl_ctx* ctx, int bn, int nsub, const CUtensorMap& a, const CUtensorMap& b, const ConvHaloArgs& args,
                    int grid, int smem, cudaStream_t stream) {
  if (bn == 64 && nsub == 2) return launch_halo_res_one<64, 2, B_MN, STATS, SCATTER, BR>(ctx, a, b, args, grid, smem, stream);
  if (bn == 64 && nsub == 1) return launch_halo_res_one<64, 1, B_MN, STATS, SCATTER, BR>(ctx, a, b, args, grid, smem, stream);
  if (bn == 128 && nsub == 2) return launch_halo_res_one<128, 2, B_MN, STATS, SCATTER, BR>(ctx, a, b, args, grid, smem, stream);
  if (bn == 128 && nsub == 1) return launch_halo_res_one<128, 1, B_MN, STATS, SCATTER, BR>(ctx, a, b, args, grid, smem, stream);
  return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv_halo (resident): tile %d x %d", bn, nsub);
}

// Re-derives the unit count / grid of a plan after nsub or bn changed.
void replan_units(bsl_ctx* ctx, HaloPlan& p) {
  p.n_units = cdiv(p.n_sub_total, p.nsub) * p.n_ntiles;
  int g = std::min(p.n_units, ctx->sm_count);
  if (g >= p.n_ntiles) g -= g % p.n_ntiles;
  p.grid = std::max(g, 1);
  p.slots = cdiv(p.grid, p.n_ntiles);
}

// How many CTA pairs of the (one-CTA-per-SM) pair kernels the device holds AT ONCE. The kernels are persistent with a
// static schedule, so a pair that had to wait for a second round would double the launch's time: a GPC with an odd number
// of usable SMs hosts one pair fewer than sm_count / 2 suggests. Asked from the driver once (the widest configuration).
int max_pairs(bsl_ctx* ctx) {
  static std::mutex mu;
  static int cached = -1;
  std::lock_guard<std::mutex> g(mu);
  if (cached >= 0) return cached;
  auto kern = conv_halo_kernel<128, 2, true, false, false, false, true, true>;
  constexpr int smem = ConvHaloCfg<128, 2, true, true>::SMEM_BYTES;
  int n = 0;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * (ctx->sm_count / 2));
    cfg.blockDim = dim3(CH_THREADS);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) n = 0;
  }
  (void)cudaGetLastError();
  cached = std::max(0, std::min(n, ctx->sm_count / 2));
  return cached;
}
// CTA pairs run 128-wide tiles: per CTA a pair takes in half of every filter slice, so the narrower tile costs no more
// filter traffic than a 256-wide tile of a single CTA, and twice as many units fill the 148 SMs evenly (512 units of a
// 512-channel layer at 32 x 32 are 3.46 per SM -- the last of 4 rounds is half empty; 1024 are 6.92) with the accumulators
// double-buffered. Measured on the wide cfg2 layers: -10 % against single CTAs with 256-wide tiles
// (profiles/r02_ab_experiments.md). min_cols: fprop keeps its fused statistics for 128-column layers.
bool pair_replan(bsl_ctx* ctx, HaloPlan& p, int ncols, int min_cols, int ntaps) {
  if (ntaps != 9 || ncols % 128 || ncols < min_cols || p.n_sub_total % 4) return false;
  if (max_pairs(ctx) < 1) return false;
  p.bn = 128;
  p.nsub = 2;
  p.n_ntiles = ncols / 128;
  replan_units(ctx, p);
  p.pair = 1;
  return true;
}

// Output tensor map of the TMA-store epilogue: (c, x, y, image) with a 64-channel x 8 x 16 pixel box.
int out_map(bsl_ctx* ctx, const ConvHaloArgs& a, int w, int h, CUtensorMap* out) {
  if (a.ostride_y != (long long)w * a.ostride_x || (a.n > 1 && a.ostride_n != (long long)h * a.ostride_y) ||
      (reinterpret_cast<uintptr_t>(a.out) & 15) || a.ostride_x % 8)
    return 1;   // not a plain NHWC window: keep the direct stores
  uint64_t dims[4] = {(uint64_t)a.n_total, (uint64_t)w, (uint64_t)h, (uint64_t)a.n};
  uint64_t str[4] = {2, (uint64_t)a.ostride_x * 2, (uint64_t)a.ostride_y * 2,
                     (uint64_t)(a.n > 1 ? a.ostride_n : (long long)h * a.ostride_y) * 2};
  uint32_t bx[4] = {64, 8, 16, 1};
  return bsl_get_tmap(ctx, a.out, 4, dims, str, bx, out);
}

// CTA pairs (conv_halo_kernel<..., PAIR>): 256-wide tiles of 3x3 windows whose sub-tile count is a multiple of 4 (a pair
// works on two units of two sub-tiles and the same column tile). `b_half`: for a K-major filter (dgrad) the tensor map
// whose box holds HALF the tile's rows; an MN-major filter (fprop) is loaded in 64-column blocks either way.
bool pair_eligible(bsl_ctx* ctx, const ConvHaloArgs& a, int bn, int nsub) {
  return max_pairs(ctx) >= 1 && (bn == 256 || bn == 128) && nsub == 2 && a.n_sub_total % 4 == 0 && a.ntaps == 9 && a.halo == 1 &&
         !a.tap_table && a.up_cpb == 0;
}
template <int BN, bool B_MN, bool BR = false>
int launch_halo_pair(bsl_ctx* ctx, const CUtensorMap& a, const CUtensorMap& b, const ConvHaloArgs& args, cudaStream_t stream,
                     const CUtensorMap& o) {
  auto kern = conv_halo_kernel<BN, 2, B_MN, false, false, false, true, true, BR>;
  constexpr int smem = ConvHaloCfg<BN, 2, true, true>::SMEM_BYTES;
  static bool configured = false;
  if (!configured) {
    BSL_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  const int pairs = std::min(args.n_units / 2, max_pairs(ctx));
  if (pairs < 1) return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv_halo (CTA pairs): the device holds no cluster of two CTAs");
  bsl_launch_cluster(kern, dim3(2 * pairs), dim3(CH_THREADS), smem, stream, 2, a, b, o, args);
  BSL_LAUNCH_CHECK(ctx, "conv_halo_kernel (CTA pairs) launch");
  return BSL_OK;
}

// ---- CTA pairs with a RESIDENT filter: the layers whose whole column range is one tile (N == 64 or 128) and whose
// filter slice fits in shared memory. Each CTA keeps half of the slice (rows [rank * N / 2, ...) of a K-MAJOR filter),
// which also frees room for activation stages. dgrad reads the HWIO filter K-major as it is; fprop gets a K-major copy
// ([tap][cout][cin], a few hundred KB at most) written into the per-stream filter scratch right before the launch --
// an MN-major filter would have to be split into 32-column halves, which the 128-byte swizzle cannot express.
bool plan_resident_pair(bsl_ctx* ctx, int bn, int ntaps, int cblocks, int n_sub_total, int* nsub, int* a_stages, int* smem) {
  // one-block reductions (K = 64) stay with single CTAs: their units are so short that the epilogue, not the tensor pipe,
  // sets the pace once the MMAs get faster (measured: 64 -> 64 fprop 0.298 -> 0.314 ms, dgrad unchanged), while
  // 128 -> 64 fprop gained 19 % and 128 -> 64 dgrad 25 % (profiles/r02_ab_experiments.md)
  if ((bn != 64 && bn != 128) || ntaps != 9 || cblocks < 2 || max_pairs(ctx) < 1) return false;
  const int res = ntaps * cblocks * (bn / 2) * 128;
  const int left = CH_DYN_BUDGET - 1024 - res;
  if (left <= 0) return false;
  const int s2 = std::min(CH_MAX_A_STAGES, left / (2 * CH_SUB_BYTES)), s1 = std::min(CH_MAX_A_STAGES, left / CH_SUB_BYTES);
  int ns, st;
  if (n_sub_total % 4 == 0 && s2 >= 3) { ns = 2; st = s2; }
  else if (n_sub_total % 2 == 0 && s1 >= 3) { ns = 1; st = s1; }
  else if (n_sub_total % 4 == 0 && s2 >= 2) { ns = 2; st = s2; }
  else return false;
  *nsub = ns;
  *a_stages = st;
  *smem = st * ns * CH_SUB_BYTES + res + 1024;
  return true;
}
void replan_pair_units(bsl_ctx* ctx, HaloPlan& p) {   // one column tile; both CTAs of a pair always work
  p.n_ntiles = 1;
  p.n_units = p.n_sub_total / p.nsub;
  p.grid = 2 * std::min(p.n_units / 2, max_pairs(ctx));
  p.slots = p.grid;
  p.pair = 1;
}

template <int BN, int NSUB, bool STATS, bool BR = false>
int launch_halo_res_pair_one(bsl_ctx* ctx, const CUtensorMap& a, const CUtensorMap& b, const ConvHaloArgs& args, int grid,
                             int smem, cudaStream_t stream) {
  auto kern = conv_halo_kernel<BN, NSUB, false, STATS, false, true, false, true, BR>;
  static int configured = 0;
  if (configured < smem) {
    BSL_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = smem;
  }
  bsl_launch_cluster(kern, dim3(grid), dim3(CH_THREADS), smem, stream, 2, a, b, a, args);
  BSL_LAUNCH_CHECK(ctx, "conv_halo_kernel (CTA pairs, resident filter) launch");
  return BSL_OK;
}
template <bool STATS, bool BR = false>
int launch_halo_res_pair(bsl_ctx* ctx, int bn, int nsub, const CUtensorMap& a, const CUtensorMap& b, const ConvHaloArgs& args,
                         int grid, int smem, cudaStream_t stream) {
  if (bn == 64 && nsub == 2) return launch_halo_res_pair_one<64, 2, STATS, BR>(ctx, a, b, args, grid, smem, stream);
  if (bn == 64 && nsub == 1) return launch_halo_res_pair_one<64, 1, STATS, BR>(ctx, a, b, args, grid, smem, stream);
  if (bn == 128 && nsub == 2) return launch_halo_res_pair_one<128, 2, STATS, BR>(ctx, a, b, args, grid, smem, stream);
  if (bn == 128 && nsub == 1) return launch_halo_res_pair_one<128, 1, STATS, BR>(ctx, a, b, args, grid, smem, stream);
  return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv_halo (CTA pairs, resident): tile %d x %d", bn, nsub);
}

// HWIO [taps][cin][cout] -> [taps][cout][cin] (bf16), the K-major filter of the forward pass of a CTA pair.
__global__ void filter_kmajor_kernel(const __nv_bfloat16* __restrict__ w, __nv_bfloat16* __restrict__ o, int cin, int cout,
                                     int total) {
  bsl::pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // output index: (tap, co, ci)
  if (i >= total) return;
  const int ci = i % cin, t = i / cin;
  const int co = t % cout, tap = t / cout;
  o[i] = w[((long long)tap * cin + ci) * cout + co];
}

// BR: the bias + ReLU epilogue (args.bias, bsl_conv2d_fprop_bias_relu) on the same schedules as the plain one.
template <bool B_MN, bool STATS, bool SCATTER, bool BR = false>
int launch_halo(bsl_ctx* ctx, int bn, int nsub, const CUtensorMap& a, const CUtensorMap& b, const ConvHaloArgs& args,
                int grid, cudaStream_t stream, const CUtensorMap* b_half = nullptr) {
  if constexpr (!STATS && !SCATTER) {
    if (pair_eligible(ctx, args, bn, nsub) && (B_MN || b_half != nullptr)) {
      CUtensorMap o;
      if (out_map(ctx, args, args.vw, args.vh, &o) == 0)
        return bn == 256 ? launch_halo_pair<256, B_MN, BR>(ctx, a, B_MN ? b : *b_half, args, stream, o)
                         : launch_halo_pair<128, B_MN, BR>(ctx, a, B_MN ? b : *b_half, args, stream, o);
    }
    if (bn == 256) {   // TMA-store epilogue of the 256-wide tiles (DESIGN.md 3.6)
      CUtensorMap o;
      if (out_map(ctx, args, args.vw, args.vh, &o) == 0) {
        if (nsub == 2) return launch_halo_one<256, 2, B_MN, false, false, true, BR>(ctx, a, b, args, grid, stream, &o);
        if (nsub == 1) return launch_halo_one<256, 1, B_MN, false, false, true, BR>(ctx, a, b, args, grid, stream, &o);
      }
    }
  }
  if (bn == 64 && nsub == 2) return launch_halo_one<64, 2, B_MN, STATS, SCATTER, false, BR>(ctx, a, b, args, grid, stream);
  if (bn == 64 && nsub == 1) return launch_halo_one<64, 1, B_MN, STATS, SCATTER, false, BR>(ctx, a, b, args, grid, stream);
  if (bn == 128 && nsub == 2) return launch_halo_one<128, 2, B_MN, STATS, SCATTER, false, BR>(ctx, a, b, args, grid, stream);
  if (bn == 128 && nsub == 1) return launch_halo_one<128, 1, B_MN, STATS, SCATTER, false, BR>(ctx, a, b, args, grid, stream);
  if (!STATS) {  // the widest tile has no spare TMEM for an overlapped epilogue: statistics stay a separate pass
    if (bn == 256 && nsub == 2) return launch_halo_one<256, 2, B_MN, false, SCATTER, false, BR>(ctx, a, b, args, grid, stream);
    if (bn == 256 && nsub == 1) return launch_halo_one<256, 1, B_MN, false, SCATTER, false, BR>(ctx, a, b, args, grid, stream);
  }
  return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv_halo: tile %d x %d", bn, nsub);
}

// Pixel sub-tiles are 8 (w) x 16 (h); `ncols` is the GEMM N extent (a multiple of 64).
// Ragged extents: a grid that the tile does not divide runs with ceil(extent / tile) tiles -- TMA zero-fills the reads
// past the edge (SAME padding already relies on it), the epilogue masks the stores and the statistics of pixels outside
// the image (ConvHaloArgs::vw / vh), the filter-gradient kernels need nothing (zero dy rows contribute zero). Taken when
// the padded grid holds at most 2x the pixels.
bool tiles_ok(int w, int h, int tw, int th) {
  if (w % tw == 0 && h % th == 0) return true;
  if (w < 1 || h < 1) return false;
  return (long long)cdiv(w, tw) * tw * cdiv(h, th) * th <= 2LL * w * h;
}
bool halo_eligible(int w, int h) { return tiles_ok(w, h, 8, 16); }

HaloPlan plan_halo(bsl_ctx* ctx, int w, int h, int n, int ncols) {
  HaloPlan p = {};
  p.n_sub_total = cdiv(w, 8) * cdiv(h, 16) * n;
  p.bn = ncols % 256 == 0 ? 256 : (ncols % 128 == 0 ? 128 : 64);
  p.nsub = p.n_sub_total % 2 == 0 ? 2 : 1;
  p.n_ntiles = ncols / p.bn;
  p.n_units = cdiv(p.n_sub_total, p.nsub) * p.n_ntiles;
  int g = std::min(p.n_units, ctx->sm_count);
  if (g >= p.n_ntiles) g -= g % p.n_ntiles;  // a CTA then always owns the same column tile (statistics)
  p.grid = std::max(g, 1);
  p.slots = cdiv(p.grid, p.n_ntiles);
  return p;
}

void halo_common(ConvHaloArgs& a, const HaloPlan& p, int w, int h, int n) {
  a.ntile_w = cdiv(w, 8);
  a.ntile_h = cdiv(h, 16);
  a.vw = w;
  a.vh = h;
  a.n = n;
  a.n_sub_total = p.n_sub_total;
  a.n_units = p.n_units;
  a.n_ntiles = p.n_ntiles;
  a.dbg = g_dbg_waits;
  a.kd = 1;        // 2-D: every image is its own one-slice "volume" (tensor map dims (c, w, h, n, 1))
  a.depth = n;
}

struct WgradPlan {
  int k_tiles, per, splits;
};

bool wgrad_halo_eligible(const bsl_conv2d_desc* d) {
  return d->kh == 3 && d->kw == 3 && tiles_ok(d->w, d->h, WG_TW, WG_TH);
}

// ---- wide wgrad (wgrad_halo3_kernel): 3x3 layers whose output channels come in 128-wide blocks. Split counts for the
// two CTA classes are chosen by simulating the hardware's in-order block dispatch onto the SMs.
struct WideWgradPlan {
  int k_tiles, splits_a, per_a, splits_b, per_b;
};

bool wgrad_wide_eligible(const bsl_conv2d_desc* d) {
  return d->kh == 3 && d->kw == 3 && tiles_ok(d->w, d->h, WG_TW, WG_TH) && d->cout % 128 == 0;
}

// Every CTA fills two accumulators per pixel tile. Costs per pixel tile in units of 384 tensor cycles, from the per-CTA
// cycle counters (tools/gpu_conv_bench.py --ops wgrad --waits).
WideWgradPlan plan_wgrad3_core(bsl_ctx* ctx, int k, int ncb, int nnbk) {
  const double cost_a = 2.0;
  const double cost_b2 = 2.1;   // two input blocks
  const double cost_b1 = 1.4;   // lone last input block
  WideWgradPlan best = {};
  const int sms = ctx->sm_count;
  const double fixed = 6.0;   // prologue + epilogue of a CTA
  const int ncb_b = cdiv(ncb, 2);
  const long long mn_a = (long long)ncb * nnbk, mn_b = (long long)ncb_b * nnbk;
  double best_t = 1e300;
  const int max_a = std::max(1, std::min(k / 2, (int)((2 * sms) / mn_a) + 2));
  std::vector<double> heap;
  for (int na = 1; na <= max_a; ++na) {
    const int per_a = cdiv(k, na), sa = cdiv(k, per_a);
    if (sa != na) continue;
    const int mid = std::max(1, (int)(na * (ncb >= 2 ? cost_b2 : cost_b1) / cost_a + 0.5));
    for (int nb2 = std::max(1, mid - 2); nb2 <= mid + 2; ++nb2) {
      if (nb2 > k) break;
      const int per_b = cdiv(k, nb2), sb = cdiv(k, per_b);
      if (sb != nb2) continue;
      // in-order dispatch: all class-a CTAs, then class b, each to the SM that frees up first (min-heap of free times)
      heap.assign(sms, 0.0);
      double makespan = 0;
      auto run = [&](double t) {
        std::pop_heap(heap.begin(), heap.end(), std::greater<double>());
        heap.back() += t;
        makespan = std::max(makespan, heap.back());
        std::push_heap(heap.begin(), heap.end(), std::greater<double>());
      };
      const double ta = cost_a * per_a + fixed;
      for (long long j = 0; j < mn_a * sa; ++j) run(ta);
      for (long long j = 0; j < mn_b * sb; ++j) {
        const int col = (int)(j % ncb_b);
        run((2 * col + 1 < ncb ? cost_b2 : cost_b1) * per_b + fixed);
      }
      makespan += 0.02 * (sa + sb);   // a little pressure towards fewer partials to reduce afterwards
      if (makespan < best_t) {
        best_t = makespan;
        best = {k, sa, per_a, sb, per_b};
      }
    }
  }
  return best;
}

// Launch + reduction of the partials; shared by the 2-D layers (kd = 1, depth = n) and UNet3D's stride-1 layers.
// Partials are [split][kd][taps][cin][cout]; a class with a single split writes its rows of dW directly when kd == 1.
size_t wgrad3_ws_bytes(const WideWgradPlan& q, int kd, size_t per_tap) {
  const bool direct_a = q.splits_a == 1 && kd == 1, direct_b = q.splits_b == 1 && kd == 1;
  return ((direct_a ? 0 : (size_t)q.splits_a * 6) + (direct_b ? 0 : (size_t)q.splits_b * 3)) * kd * per_tap * sizeof(float);
}

int launch_wgrad3(bsl_ctx* ctx, const WideWgradPlan& q, const CUtensorMap& txa, const CUtensorMap& txb, const CUtensorMap& ty,
                  int w, int h, int n_imgs, int cin, int cout, int kd, int depth, float* dw, void* workspace,
                  size_t workspace_bytes, cudaStream_t stream) {
  const long long per_tap = (long long)cin * cout;
  const size_t need = wgrad3_ws_bytes(q, kd, per_tap);
  if (need > workspace_bytes || (need && !workspace))
    return bsl_fail(ctx, BSL_EWORKSPACE, "conv wgrad: workspace %zu < %zu", workspace_bytes, need);
  float* ws = reinterpret_cast<float*>(workspace);
  const bool direct_a = q.splits_a == 1 && kd == 1, direct_b = q.splits_b == 1 && kd == 1;
  WgradHalo3Args a = {};
  a.ntile_w = cdiv(w, WG_TW);
  a.ntile_h = cdiv(h, WG_TH);
  a.n = n_imgs;
  a.k_tiles_total = q.k_tiles;
  a.ncb = cin / 64;
  a.nnb = cout / 128;
  a.ncb_b = cdiv(a.ncb, 2);
  a.splits_a = q.splits_a;
  a.per_a = q.per_a;
  a.splits_b = q.splits_b;
  a.per_b = q.per_b;
  a.n_cta_a = a.ncb * a.nnb * kd * q.splits_a;
  a.cin = cin;
  a.cout = cout;
  a.out_a = direct_a ? dw : ws;
  a.out_b = direct_b ? dw + 6 * per_tap : ws + (direct_a ? 0 : (long long)q.splits_a * kd * 6 * per_tap);
  a.kd = kd;
  a.depth = depth;
  a.dbg = g_dbg_waits;
  a.status = ctx->d_status;
  a.stages_a = WG3_STAGES_A;
  a.stages_b = WG3_STAGES_B;
  constexpr int smem = wg3_smem_bytes(WG3_STAGES_A, WG3_STAGES_B);
  static bool configured = false;
  if (!configured) {
    BSL_CUDA(ctx, cudaFuncSetAttribute(wgrad_halo3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  const int grid = a.n_cta_a + a.ncb_b * a.nnb * kd * q.splits_b;
  bsl_launch(wgrad_halo3_kernel, dim3(grid), dim3(WG_THREADS), smem, stream, txa, txb, ty, a);
  BSL_LAUNCH_CHECK(ctx, "wgrad_halo3_kernel launch");
  int rc;
  for (int k = 0; k < kd; ++k) {   // partial[split][kd][taps] -> dW[kd][9]: split stride = kd * taps * per_tap
    if (!direct_a && (rc = reduce_splits_strided(ctx, a.out_a + (long long)k * 6 * per_tap, dw + (long long)k * 9 * per_tap,
                                                 6 * per_tap, q.splits_a, (long long)kd * 6 * per_tap, stream)))
      return rc;
    if (!direct_b && (rc = reduce_splits_strided(ctx, a.out_b + (long long)k * 3 * per_tap, dw + ((long long)k * 9 + 6) * per_tap,
                                                 3 * per_tap, q.splits_b, (long long)kd * 3 * per_tap, stream)))
      return rc;
  }
  return BSL_OK;
}

const WideWgradPlan& cached_wgrad3(bsl_ctx* ctx, const bsl_conv2d_desc* d) {
  static std::mutex mu;
  static std::unordered_map<unsigned long long, WideWgradPlan> cache;
  const unsigned long long key = ((unsigned long long)d->n << 48) ^ ((unsigned long long)d->h << 36) ^
                                 ((unsigned long long)d->w << 24) ^ ((unsigned long long)d->cin << 12) ^ d->cout;
  std::lock_guard<std::mutex> g(mu);
  auto it = cache.find(key);
  if (it == cache.end())
    it = cache.emplace(key, plan_wgrad3_core(ctx, cdiv(d->w, WG_TW) * cdiv(d->h, WG_TH) * d->n, d->cin / 64, d->cout / 128)).first;
  return it->second;
}

int conv2d_wgrad3(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const void* dy, float* dw, void* workspace,
                  size_t workspace_bytes, cudaStream_t stream) {
  const WideWgradPlan& p = cached_wgrad3(ctx, d);
  const int xbox_a[4] = {WG_TW + 2, WG_TH + 1, 1, 1}, xbox_b[4] = {WG_TW + 2, WG_TH, 1, 1}, ybox[4] = {WG_TW, WG_TH, 1, 1};
  CUtensorMap txa, txb, ty;
  int rc;
  if ((rc = nhwc_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, xbox_a, &txa))) return rc;
  if ((rc = nhwc_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, xbox_b, &txb))) return rc;
  if ((rc = nhwc_map(ctx, dy, d->cout, d->w, d->h, d->n, d->y_ld, ybox, &ty))) return rc;
  return launch_wgrad3(ctx, p, txa, txb, ty, d->w, d->h, d->n, d->cin, d->cout, 1, d->n, dw, workspace, workspace_bytes, stream);
}

WgradPlan plan_wgrad_halo(bsl_ctx* ctx, const bsl_conv2d_desc* d) {
  WgradPlan p;
  p.k_tiles = cdiv(d->w, WG_TW) * cdiv(d->h, WG_TH) * d->n;
  const int mn = (d->cin / 64) * (d->cout / 64);
  int splits = std::max(1, ctx->sm_count / mn);
  splits = std::max(1, std::min(splits, p.k_tiles / 4));
  p.per = cdiv(p.k_tiles, splits);
  p.splits = cdiv(p.k_tiles, p.per);
  return p;
}
}  // namespace

extern "C" {

int bsl_debug_set(bsl_ctx* ctx, int key, int value) {
  switch (key) {
    case 0: g_mn_lbo = value; return BSL_OK;
    case 1: g_mn_sbo = value; return BSL_OK;
    case 2: g_mn_kadv = value; return BSL_OK;
    case 3:
      if (value && !g_dbg_waits) {
        BSL_CUDA(ctx, cudaMalloc(&g_dbg_waits, 1024 * 4 * sizeof(long long)));
        BSL_CUDA(ctx, cudaMemset(g_dbg_waits, 0, 1024 * 4 * sizeof(long long)));
      } else if (!value && g_dbg_waits) {
        cudaFree(g_dbg_waits);
        g_dbg_waits = nullptr;
      }
      return BSL_OK;
  }
  return bsl_fail(ctx, BSL_EINVAL, "debug_set: unknown key %d", key);
}

int bsl_debug_read_waits(bsl_ctx* ctx, long long* out, int ctas) {
  if (!ctx || !out || ctas < 1 || ctas > 1024) return BSL_EINVAL;
  if (!g_dbg_waits) return bsl_fail(ctx, BSL_EINVAL, "debug waits are off (bsl_debug_set(ctx, 3, 1))");
  BSL_CUDA(ctx, cudaMemcpy(out, g_dbg_waits, (size_t)ctas * 4 * sizeof(long long), cudaMemcpyDeviceToHost));
  return BSL_OK;
}

// Launch of an fprop on the halo-tile kernel with optional fused statistics of its bf16 outputs (shared by the 2-D
// layers and the stride-1 3-D layers, whose "images" are the n * d slices and whose statistics group is one volume).
static int launch_fprop_halo_stats(bsl_ctx* ctx, const HaloPlan& pl, bool res, int res_smem, const CUtensorMap& ta,
                                   const CUtensorMap& tb, ConvHaloArgs& a, double* sums, int group_imgs, int n_imgs, int h,
                                   int w, int cout, void* y, int y_ld, cudaStream_t stream) {
  int rc;
  const bool res_pair = res && pl.pair;   // resident filter of a CTA pair: tb is the K-major copy (conv2d_fprop_halo)
  auto run = [&](bool stats) -> int {
    if (res_pair)
      return stats ? launch_halo_res_pair<true>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, stream)
                   : launch_halo_res_pair<false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, stream);
    if (res)
      return stats ? launch_halo_res<true, true, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, stream)
                   : launch_halo_res<true, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, stream);
    return stats ? launch_halo<true, true, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, stream)
                 : launch_halo<true, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, stream);
  };
  if (!sums) return run(false);
  const int groups = group_imgs > 0 ? n_imgs / group_imgs : 1;
  const long long ppg = group_imgs > 0 ? (long long)group_imgs * h * w : (long long)n_imgs * h * w;
  if (pl.bn == 256 || (pl.pair && !res) || (group_imgs > 0 && pl.grid % pl.n_ntiles != 0)) {
    // long-reduction layers: small, L2-resident outputs; a separate statistics pass is cheaper than an
    // un-overlapped epilogue butterfly
    if ((rc = run(false))) return rc;
    return bsl_stats_bf16(ctx, y, ppg, groups, cout, y_ld, sums, stream);
  }
  float* part = nullptr;
  if (group_imgs > 0) {
    // [group][slot * 4 + lane quarter][2][cout], zero-filled: a CTA only writes the groups its units fall into
    const size_t bytes = (size_t)groups * pl.slots * 4 * 2 * cout * sizeof(float);
    if ((rc = bsl_scratch(ctx, bytes, &part, stream))) return rc;
    BSL_CUDA(ctx, cudaMemsetAsync(part, 0, bytes, stream));
    a.stats_part = part;
    a.stats_group_imgs = group_imgs;
    a.stats_blocks = pl.slots * 4;
    if ((rc = run(true))) return rc;
    const int kc2 = 2 * cout;
    bsl_launch(pixel_reduce_final_kernel, dim3((kc2 + 31) / 32, groups), dim3(1024), 0, stream, part, pl.slots * 4, kc2, sums);
    BSL_LAUNCH_CHECK(ctx, "pixel_reduce_final_kernel (conv instance statistics)");
    return BSL_OK;
  }
  if ((rc = bsl_scratch(ctx, (size_t)pl.slots * 2 * cout * sizeof(float), &part, stream))) return rc;
  a.stats_part = part;
  if ((rc = run(true))) return rc;
  const int kc = 2 * cout;
  bsl_launch(pixel_reduce_final_kernel, dim3(dim3((kc + 31) / 32, 1)), dim3(1024), 0, stream, part, pl.slots, kc, sums);
  BSL_LAUNCH_CHECK(ctx, "pixel_reduce_final_kernel (conv statistics)");
  return BSL_OK;
}

// fprop on the halo-tile kernel; `sums` (fp64 [2][cout], nullable) receives the per-channel sum and
// sum of squares of the bf16 outputs, reduced deterministically from per-CTA partials.
// group_imgs > 0: instance statistics, sums is [n / group_imgs][2][cout] (one group = group_imgs consecutive images).
// bias != nullptr (no sums): the bias + ReLU epilogue, y = bf16(relu(conv + bias)), on the schedule the plain fprop takes.
static int conv2d_fprop_halo(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const void* w, void* y,
                             double* sums, cudaStream_t stream, int group_imgs = 0, const float* bias = nullptr) {
  const int halo = d->kh == 3 ? 1 : 0;
  HaloPlan pl = plan_halo(ctx, d->w, d->h, d->n, d->cout);
  int res_stages = 0, res_smem = 0;
  bool res = false;
  const void* w_k = nullptr;   // K-major copy of the filter (resident CTA pairs)
  if (d->cout == pl.bn && d->cin % 64 == 0 && d->x_ld >= d->cin &&
      plan_resident_pair(ctx, pl.bn, d->kh * d->kw, d->cin / 64, pl.n_sub_total, &pl.nsub, &res_stages, &res_smem)) {
    void* wk = nullptr;
    const int total = 9 * d->cin * d->cout;
    int rc0;
    if ((rc0 = bsl_scratch_w(ctx, (size_t)total * 2, &wk, stream))) return rc0;
    bsl_launch(filter_kmajor_kernel, dim3(cdiv(total, 256)), dim3(256), 0, stream, reinterpret_cast<const __nv_bfloat16*>(w),
               reinterpret_cast<__nv_bfloat16*>(wk), d->cin, d->cout, total);
    BSL_LAUNCH_CHECK(ctx, "filter_kmajor_kernel");
    w_k = wk;
    res = true;
    replan_pair_units(ctx, pl);
  } else {
    res = plan_resident(pl.bn, d->kh * d->kw, d->cin / 64, &pl.nsub, &res_stages, &res_smem);
    if (res) replan_units(ctx, pl);
    else pair_replan(ctx, pl, d->cout, 256, d->kh * d->kw);
  }
  const int box[4] = {8 + 2 * halo, 16 + 2 * halo, 1, 1};
  CUtensorMap ta, tb;
  int rc;
  if ((rc = nhwc_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, box, &ta))) return rc;
  if (w_k) {   // [9 * cout rows][cin]: 64 consecutive input channels = the K block, half the tile's rows per CTA
    if ((rc = matrix_map(ctx, w_k, d->cin, 9 * d->cout, 64, pl.bn / 2, &tb))) return rc;
  } else if ((rc = matrix_map(ctx, w, d->cout, d->kh * d->kw * d->cin, 64, 64, &tb))) {
    return rc;
  }
  ConvHaloArgs a = {};
  halo_common(a, pl, d->w, d->h, d->n);
  a.ntaps = d->kh * d->kw;
  a.halo = halo;
  a.cblocks = d->cin / 64;
  a.out = y;
  a.ostride_x = d->y_ld;
  a.ostride_y = (long long)d->w * d->y_ld;
  a.ostride_n = (long long)d->h * d->w * d->y_ld;
  a.n_group = d->cout;
  a.n_total = d->cout;
  a.a_stages = res_stages;
  a.b_rows_per_tap = d->cout;   // (K-major copy of a resident CTA pair; unused otherwise)
  a.status = ctx->d_status;
  if (bias) {
    a.bias = bias;
    a.relu = 1;
    if (res && pl.pair) return launch_halo_res_pair<false, true>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, stream);
    if (res) return launch_halo_res<true, false, false, true>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, stream);
    return launch_halo<true, false, false, true>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, stream);
  }
  return launch_fprop_halo_stats(ctx, pl, res, res_smem, ta, tb, a, sums, group_imgs, d->n, d->h, d->w, d->cout, y,
                                 d->y_ld, stream);
}

int bsl_conv2d_fprop_stats(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const void* w, void* y,
                           double* sums, void* stream) {
  int rc = check_conv(ctx, d, true);
  if (rc) return rc;
  if (!x || !w || !y || !sums) return bsl_fail(ctx, BSL_EINVAL, "conv2d_fprop_stats: null buffer");
  if (halo_eligible(d->w, d->h)) return conv2d_fprop_halo(ctx, d, x, w, y, sums, as_stream(stream));
  if ((rc = bsl_conv2d_fprop(ctx, d, x, w, y, stream))) return rc;
  return bsl_stats_bf16(ctx, y, (long long)d->n * d->h * d->w, 1, d->cout, d->y_ld, sums, as_stream(stream));
}

int bsl_conv2d_fprop_group_stats(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const void* w, void* y,
                                 int imgs_per_group, double* sums, void* stream) {
  int rc = check_conv(ctx, d, true);
  if (rc) return rc;
  if (!x || !w || !y || !sums) return bsl_fail(ctx, BSL_EINVAL, "conv2d_fprop_group_stats: null buffer");
  if (imgs_per_group < 1 || d->n % imgs_per_group)
    return bsl_fail(ctx, BSL_EINVAL, "conv2d_fprop_group_stats: imgs_per_group=%d must divide n=%d", imgs_per_group, d->n);
  if (halo_eligible(d->w, d->h)) return conv2d_fprop_halo(ctx, d, x, w, y, sums, as_stream(stream), imgs_per_group);
  if ((rc = bsl_conv2d_fprop(ctx, d, x, w, y, stream))) return rc;
  return bsl_stats_bf16(ctx, y, (long long)imgs_per_group * d->h * d->w, d->n / imgs_per_group, d->cout, d->y_ld, sums,
                        as_stream(stream));
}

// fprop with the plain (bias == nullptr) or the bias + ReLU epilogue; both take the same schedule for a shape.
static int conv2d_fprop(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const void* w, const float* bias, void* y,
                        void* stream) {
  int rc;
  if (halo_eligible(d->w, d->h)) return conv2d_fprop_halo(ctx, d, x, w, y, nullptr, as_stream(stream), 0, bias);
  int box[4] = {0, 0, 0, 1};
  pick_box(128, d->w, d->h, d->n, &box[0], &box[1], &box[2]);
  const int bn = pick_bn(d->cout);
  CUtensorMap ta, tb;
  if ((rc = nhwc_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, box, &ta))) return rc;
  if ((rc = matrix_map(ctx, w, d->cout, d->kh * d->kw * d->cin, 64, 64, &tb))) return rc;
  IgemmArgs a = {};
  const int tdim[4] = {d->w, d->h, d->n, 1};
  set_tiles(a, tdim, box);
  conv_taps(a, d->kh, d->kw);
  a.cblocks = d->cin / 64;
  a.out = y;
  a.ostride[0] = d->y_ld;
  a.ostride[1] = (long long)d->w * d->y_ld;
  a.ostride[2] = (long long)d->h * d->w * d->y_ld;
  a.n_group = d->cout;
  a.n_total = d->cout;
  a.bias = bias;
  a.relu = bias != nullptr;
  a.status = ctx->d_status;
  dim3 grid(a.ntile[0] * a.ntile[1] * a.ntile[2], d->cout / bn, 1);
  return launch_igemm<MODE_PIX_M, true>(ctx, bn, ta, tb, a, grid, as_stream(stream));
}

int bsl_conv2d_fprop(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const void* w, void* y,
                     void* stream) {
  int rc = check_conv(ctx, d, true);
  if (rc) return rc;
  if (!x || !w || !y) return bsl_fail(ctx, BSL_EINVAL, "conv2d_fprop: null buffer");
  return conv2d_fprop(ctx, d, x, w, nullptr, y, stream);
}

int bsl_conv2d_fprop_bias_relu(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const void* w, const float* bias,
                               void* y, void* stream) {
  int rc = check_conv(ctx, d, true);
  if (rc) return rc;
  if (!x || !w || !bias || !y) return bsl_fail(ctx, BSL_EINVAL, "conv2d_fprop_bias_relu: null buffer");
  return conv2d_fprop(ctx, d, x, w, bias, y, stream);
}

int bsl_conv2d_dgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* dy, const void* w, void* dx,
                     void* stream) {
  int rc = check_conv(ctx, d);
  if (rc) return rc;
  if (!dy || !w || !dx) return bsl_fail(ctx, BSL_EINVAL, "conv2d_dgrad: null buffer");
  if (halo_eligible(d->w, d->h)) {
    const int halo = d->kh == 3 ? 1 : 0;
    HaloPlan pl = plan_halo(ctx, d->w, d->h, d->n, d->cin);
    int res_stages = 0, res_smem = 0;
    bool res = false, res_pair = false;
    if (d->cin == pl.bn &&
        plan_resident_pair(ctx, pl.bn, d->kh * d->kw, d->cout / 64, pl.n_sub_total, &pl.nsub, &res_stages, &res_smem)) {
      res = res_pair = true;
      replan_pair_units(ctx, pl);
    } else {
      res = plan_resident(pl.bn, d->kh * d->kw, d->cout / 64, &pl.nsub, &res_stages, &res_smem);
      if (res) replan_units(ctx, pl);
      else pair_replan(ctx, pl, d->cin, 128, d->kh * d->kw);
    }
    const int hbox[4] = {8 + 2 * halo, 16 + 2 * halo, 1, 1};
    CUtensorMap ta, tb;
    if ((rc = nhwc_map(ctx, dy, d->cout, d->w, d->h, d->n, d->y_ld, hbox, &ta))) return rc;
    if ((rc = matrix_map(ctx, w, d->cout, d->kh * d->kw * d->cin, 64, res_pair ? pl.bn / 2 : pl.bn, &tb))) return rc;
    ConvHaloArgs a = {};
    halo_common(a, pl, d->w, d->h, d->n);
    a.ntaps = d->kh * d->kw;
    a.halo = halo;
    a.cblocks = d->cout / 64;
    a.b_flip = 1;
    a.b_rows_per_tap = d->cin;
    a.out = dx;
    a.ostride_x = d->x_ld;
    a.ostride_y = (long long)d->w * d->x_ld;
    a.ostride_n = (long long)d->h * d->w * d->x_ld;
    a.n_group = d->cin;
    a.n_total = d->cin;
    a.a_stages = res_stages;
    a.status = ctx->d_status;
    if (res_pair) return launch_halo_res_pair<false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, as_stream(stream));
    if (res) return launch_halo_res<false, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, as_stream(stream));
    CUtensorMap tbh;
    const bool pair = pair_eligible(ctx, a, pl.bn, pl.nsub) &&
                      matrix_map(ctx, w, d->cout, d->kh * d->kw * d->cin, 64, pl.bn / 2, &tbh) == 0;
    return launch_halo<false, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, as_stream(stream), pair ? &tbh : nullptr);
  }
  int box[4] = {0, 0, 0, 1};
  pick_box(128, d->w, d->h, d->n, &box[0], &box[1], &box[2]);
  const int bn = pick_bn(d->cin);
  CUtensorMap ta, tb;
  if ((rc = nhwc_map(ctx, dy, d->cout, d->w, d->h, d->n, d->y_ld, box, &ta))) return rc;
  // HWIO read as a K-major B: row = tap*cin + ci (GEMM column), 64 consecutive cout = GEMM K.
  if ((rc = matrix_map(ctx, w, d->cout, d->kh * d->kw * d->cin, 64, bn, &tb))) return rc;
  IgemmArgs a = {};
  const int tdim[4] = {d->w, d->h, d->n, 1};
  set_tiles(a, tdim, box);
  conv_taps(a, d->kh, d->kw);
  a.cblocks = d->cout / 64;
  a.b_flip = 1;
  a.b_rows_per_tap = d->cin;
  a.out = dx;
  a.ostride[0] = d->x_ld;
  a.ostride[1] = (long long)d->w * d->x_ld;
  a.ostride[2] = (long long)d->h * d->w * d->x_ld;
  a.n_group = d->cin;
  a.n_total = d->cin;
  a.status = ctx->d_status;
  dim3 grid(a.ntile[0] * a.ntile[1] * a.ntile[2], d->cin / bn, 1);
  return launch_igemm<MODE_PIX_M, false>(ctx, bn, ta, tb, a, grid, as_stream(stream));
}

size_t bsl_conv2d_wgrad_workspace(bsl_ctx* ctx, const bsl_conv2d_desc* d) {
  if (!ctx || !d || check_conv(ctx, d, true)) return 0;
  if (wgrad_wide_eligible(d)) return wgrad3_ws_bytes(cached_wgrad3(ctx, d), 1, (size_t)d->cin * d->cout);
  if (wgrad_halo_eligible(d)) {
    const WgradPlan p = plan_wgrad_halo(ctx, d);
    return p.splits > 1 ? (size_t)p.splits * 9 * d->cin * d->cout * sizeof(float) : 0;
  }
  int box[4] = {0, 0, 0, 1};
  pick_box(64, d->w, d->h, d->n, &box[0], &box[1], &box[2]);
  const int k_tiles = cdiv(d->w, box[0]) * cdiv(d->h, box[1]) * cdiv(d->n, box[2]);
  const int taps = d->kh * d->kw;
  const int bn = pick_bn(d->cout);
  const int mn = cdiv(taps * d->cin / 64, 2) * (d->cout / bn);
  SplitPlan p = plan_split(ctx, mn, k_tiles);
  return p.splits > 1 ? (size_t)p.splits * taps * d->cin * d->cout * sizeof(float) : 0;
}

int bsl_conv2d_wgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x, const void* dy, float* dw,
                     void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_conv(ctx, d, true);
  if (rc) return rc;
  if (!x || !dy || !dw) return bsl_fail(ctx, BSL_EINVAL, "conv2d_wgrad: null buffer");
  if (wgrad_wide_eligible(d)) return conv2d_wgrad3(ctx, d, x, dy, dw, workspace, workspace_bytes, as_stream(stream));
  if (wgrad_halo_eligible(d)) {
    const WgradPlan p = plan_wgrad_halo(ctx, d);
    const size_t need = p.splits > 1 ? (size_t)p.splits * 9 * d->cin * d->cout * sizeof(float) : 0;
    if (need > workspace_bytes || (need && !workspace))
      return bsl_fail(ctx, BSL_EWORKSPACE, "conv2d_wgrad: workspace %zu < %zu", workspace_bytes, need);
    const int xbox[4] = {WG_TW + 2, WG_TH + 2, 1, 1}, ybox[4] = {WG_TW, WG_TH, 1, 1};
    CUtensorMap tx, ty;
    if ((rc = nhwc_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, xbox, &tx))) return rc;
    if ((rc = nhwc_map(ctx, dy, d->cout, d->w, d->h, d->n, d->y_ld, ybox, &ty))) return rc;
    WgradHaloArgs a = {};
    a.ntile_w = cdiv(d->w, WG_TW);
    a.ntile_h = cdiv(d->h, WG_TH);
    a.n = d->n;
    a.k_tiles_total = p.k_tiles;
    a.k_tiles_per_split = p.per;
    a.cin = d->cin;
    a.cout = d->cout;
    a.out = p.splits > 1 ? reinterpret_cast<float*>(workspace) : dw;
    a.kd = 1;
    a.depth = d->n;
    a.splits = p.splits;
    a.status = ctx->d_status;
    static bool configured = false;
    if (!configured) {
      BSL_CUDA(ctx, cudaFuncSetAttribute(wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         WG_SMEM_BYTES));
      configured = true;
    }
    bsl_launch(wgrad_halo_kernel, dim3(dim3(d->cin / 64, d->cout / 64, p.splits)), dim3(WG_THREADS), WG_SMEM_BYTES, as_stream(stream), 
        tx, ty, a);
    BSL_LAUNCH_CHECK(ctx, "wgrad_halo_kernel launch");
    if (p.splits > 1)
      return reduce_splits(ctx, reinterpret_cast<const float*>(workspace), dw, (long long)9 * d->cin * d->cout,
                           p.splits, as_stream(stream));
    return BSL_OK;
  }
  int box[4] = {0, 0, 0, 1};
  pick_box(64, d->w, d->h, d->n, &box[0], &box[1], &box[2]);
  const int taps = d->kh * d->kw;
  const int bn = pick_bn(d->cout);
  CUtensorMap ta, tb;
  if ((rc = nhwc_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, box, &ta))) return rc;
  if ((rc = nhwc_map(ctx, dy, d->cout, d->w, d->h, d->n, d->y_ld, box, &tb))) return rc;
  IgemmArgs a = {};
  const int tdim[4] = {d->w, d->h, d->n, 1};
  set_tiles(a, tdim, box);
  conv_taps(a, d->kh, d->kw);
  a.cblocks = d->cin / 64;
  a.m_total = taps * d->cin;
  a.n_total = d->cout;
  a.k_tiles_total = a.ntile[0] * a.ntile[1] * a.ntile[2];
  const int m_tiles = cdiv(taps * a.cblocks, 2);
  SplitPlan p = plan_split(ctx, m_tiles * (d->cout / bn), a.k_tiles_total);
  a.k_tiles_per_split = p.per;
  const size_t need = p.splits > 1 ? (size_t)p.splits * a.m_total * a.n_total * sizeof(float) : 0;
  if (need > workspace_bytes || (need && !workspace))
    return bsl_fail(ctx, BSL_EWORKSPACE, "conv2d_wgrad: workspace %zu < %zu", workspace_bytes, need);
  a.out = p.splits > 1 ? workspace : (void*)dw;
  a.status = ctx->d_status;
  dim3 grid(m_tiles, d->cout / bn, p.splits);
  rc = launch_igemm<MODE_PIX_K, true>(ctx, bn, ta, tb, a, grid, as_stream(stream));
  if (rc) return rc;
  if (p.splits > 1)
    return reduce_splits(ctx, (const float*)workspace, dw, (long long)a.m_total * a.n_total, p.splits,
                         as_stream(stream));
  return BSL_OK;
}

// ------------------------------------------------------------------ transposed conv k2 s2

static int check_convT(bsl_ctx* ctx, const bsl_convT2d_desc* d) {
  if (!ctx) return BSL_EINVAL;
  if (!d) return bsl_fail(ctx, BSL_EINVAL, "convT2d: null descriptor");
  if (d->n <= 0 || d->h <= 0 || d->w <= 0) return bsl_fail(ctx, BSL_EINVAL, "convT2d: non-positive size");
  // cout == 32: the half-block form (see upsampled_map), halo-tile shapes only
  const bool half = d->cout == 32 && halo_eligible(d->w, d->h) && halo_eligible(d->w, d->n * d->h);
  if (d->cin % 64 || (d->cout % 64 && !half))
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "convT2d needs cin,cout multiples of 64, or cout = 32 on 8x16-tileable "
                    "shapes (got %d,%d at %dx%d)", d->cin, d->cout, d->h, d->w);
  if (d->x_ld < d->cin || d->y_ld < d->cout || d->x_ld % 8 || d->y_ld % 8)
    return bsl_fail(ctx, BSL_EINVAL, "convT2d: bad channel strides");
  return BSL_OK;
}

// cout = 32 into a pixel-pair packed tensor: output voxel (2y + a, 2x + b) lane co lives at
// y[((n * 2h + 2y + a) * w + x) * y_ld + b * 32 + co], y_ld = lanes per voxel PAIR. The GEMM columns (a, b, co) are
// the filter's own row order, so this is a transposed conv with 2 "taps" (a) of 64 columns each.
int bsl_convT2d_fwd_pairs(bsl_ctx* ctx, const bsl_convT2d_desc* d, const void* x, const void* w, void* y, void* stream) {
  int rc = check_convT(ctx, d);
  if (rc) return rc;
  if (!x || !w || !y) return bsl_fail(ctx, BSL_EINVAL, "convT2d_fwd_pairs: null buffer");
  if (d->cout != 32 || d->y_ld < 64) return bsl_fail(ctx, BSL_EUNSUPPORTED, "convT2d_fwd_pairs: cout = 32, y_ld >= 64 (lanes per voxel pair)");
  HaloPlan pl = plan_halo(ctx, d->w, d->h, d->n, 128);
  if (pl.bn == 256) return bsl_fail(ctx, BSL_EUNSUPPORTED, "convT2d_fwd_pairs: column tile");
  int res_stages = 0, res_smem = 0;
  const bool res = plan_resident(pl.bn, 1, d->cin / 64, &pl.nsub, &res_stages, &res_smem);
  if (res) replan_units(ctx, pl);
  const int hbox[4] = {8, 16, 1, 1};
  CUtensorMap ta, tb;
  if ((rc = nhwc_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, hbox, &ta))) return rc;
  if ((rc = matrix_map(ctx, w, d->cin, 128, 64, pl.bn, &tb))) return rc;
  ConvHaloArgs a = {};
  halo_common(a, pl, d->w, d->h, d->n);
  a.ntaps = 1;
  a.halo = 0;
  a.cblocks = d->cin / 64;
  a.b_rows_per_tap = 0;
  a.out = y;
  const long long row = (long long)d->w * d->y_ld;   // one output row of voxel pairs
  a.ostride_x = d->y_ld;
  a.ostride_y = 2 * row;
  a.ostride_n = (long long)2 * d->h * row;
  a.n_group = 64;
  a.group_off[0] = 0;
  a.group_off[1] = row;
  a.bias = nullptr;
  a.relu = d->relu;
  a.n_total = 128;
  a.a_stages = res_stages;
  a.status = ctx->d_status;
  return res ? launch_halo_res<false, false, true>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, as_stream(stream))
             : launch_halo<false, false, true>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, as_stream(stream));
}

int bsl_convT2d_fwd(bsl_ctx* ctx, const bsl_convT2d_desc* d, const void* x, const void* w,
                    const float* bias, void* y, void* stream) {
  int rc = check_convT(ctx, d);
  if (rc) return rc;
  if (!x || !w || !y) return bsl_fail(ctx, BSL_EINVAL, "convT2d_fwd: null buffer");
  if (halo_eligible(d->w, d->h)) {
    HaloPlan pl = plan_halo(ctx, d->w, d->h, d->n, 4 * d->cout);
    if (pl.bn == 256 && d->cin <= 256) {
      // short reductions: the un-overlapped epilogue of the 256-wide tile would cost as much as its MMAs
      pl.bn = 128;
      pl.n_ntiles = 4 * d->cout / 128;
      pl.n_units = cdiv(pl.n_sub_total, pl.nsub) * pl.n_ntiles;
      pl.grid = std::max(1, std::min(pl.n_units, ctx->sm_count));
    }
    int res_stages = 0, res_smem = 0;
    const bool res = plan_resident(pl.bn, 1, d->cin / 64, &pl.nsub, &res_stages, &res_smem);
    if (res) replan_units(ctx, pl);   // also makes the grid a multiple of the column-tile count
    const int hbox[4] = {8, 16, 1, 1};
    CUtensorMap ta, tb;
    if ((rc = nhwc_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, hbox, &ta))) return rc;
    if ((rc = matrix_map(ctx, w, d->cin, 4 * d->cout, 64, pl.bn, &tb))) return rc;
    ConvHaloArgs a = {};
    halo_common(a, pl, d->w, d->h, d->n);
    a.ntaps = 1;
    a.halo = 0;
    a.cblocks = d->cin / 64;
    a.b_rows_per_tap = 0;
    a.out = y;
    const long long row = (long long)2 * d->w * d->y_ld;
    a.ostride_x = 2 * d->y_ld;
    a.ostride_y = 2 * row;
    a.ostride_n = (long long)2 * d->h * row;
    a.n_group = d->cout;
    for (int ta_ = 0; ta_ < 2; ++ta_)
      for (int tb_ = 0; tb_ < 2; ++tb_) a.group_off[ta_ * 2 + tb_] = ta_ * row + (long long)tb_ * d->y_ld;
    a.bias = bias;
    a.relu = d->relu;
    a.n_total = 4 * d->cout;
    a.a_stages = res_stages;
    a.status = ctx->d_status;
    return res ? launch_halo_res<false, false, true>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, as_stream(stream))
               : launch_halo<false, false, true>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, as_stream(stream));
  }
  int box[4] = {0, 0, 0, 1};
  pick_box(128, d->w, d->h, d->n, &box[0], &box[1], &box[2]);
  const int bn = pick_bn(d->cout);
  CUtensorMap ta, tb;
  if ((rc = nhwc_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, box, &ta))) return rc;
  // [2,2,cout,cin]: row = tap*cout + co (GEMM column), cin contiguous (GEMM K) => K-major B.
  if ((rc = matrix_map(ctx, w, d->cin, 4 * d->cout, 64, bn, &tb))) return rc;
  IgemmArgs a = {};
  const int tdim[4] = {d->w, d->h, d->n, 1};
  set_tiles(a, tdim, box);
  a.ntaps = 1;
  a.cblocks = d->cin / 64;
  a.out = y;
  const long long row = (long long)2 * d->w * d->y_ld;  // one output row
  a.ostride[0] = 2 * d->y_ld;
  a.ostride[1] = 2 * row;
  a.ostride[2] = (long long)2 * d->h * row;
  a.n_group = d->cout;
  for (int ta_ = 0; ta_ < 2; ++ta_)
    for (int tb_ = 0; tb_ < 2; ++tb_) a.group_off[ta_ * 2 + tb_] = ta_ * row + (long long)tb_ * d->y_ld;
  a.bias = bias;
  a.relu = d->relu;
  a.n_total = 4 * d->cout;
  a.status = ctx->d_status;
  dim3 grid(a.ntile[0] * a.ntile[1] * a.ntile[2], 4 * d->cout / bn, 1);
  return launch_igemm<MODE_PIX_M, false>(ctx, bn, ta, tb, a, grid, as_stream(stream));
}

int bsl_convT2d_bwd_data(bsl_ctx* ctx, const bsl_convT2d_desc* d, const void* dyr, const void* w, void* dx,
                         void* stream) {
  int rc = check_convT(ctx, d);
  if (rc) return rc;
  if (!dyr || !w || !dx) return bsl_fail(ctx, BSL_EINVAL, "convT2d_bwd_data: null buffer");
  if (halo_eligible(d->w, d->n * d->h)) {
    // Persistent halo-tile kernel as a 1-tap GEMM: dx[p, ci] = sum over (a, b, co) of dy[2y+a, 2x+b, co] w[a,b,co,ci].
    // For a fixed row parity a the pair (b, co) is the channel axis of a row-strided view of dy, so the reduction is
    // 2 "depth" steps (a) x 2 (b) x co/64 dense TMA boxes, no element-strided gather; the rows of all images form one
    // tall image (a 1x1 conv has no halo, tiles may straddle images).
    const int rows = d->n * d->h;
    HaloPlan pl = plan_halo(ctx, d->w, rows, 1, d->cin);
    const int kblocks = 4 * d->cout / 64;
    int res_stages = 0, res_smem = 0;
    const bool res = plan_resident(pl.bn, 1, kblocks, &pl.nsub, &res_stages, &res_smem);
    if (res) replan_units(ctx, pl);
    CUtensorMap ta, tb;
    if ((rc = upsampled_map(ctx, dyr, d->cout, d->w, d->h, d->n, d->y_ld, 8, 16, &ta))) return rc;
    if ((rc = matrix_map(ctx, w, d->cin, 4 * d->cout, 64, 64, &tb))) return rc;
    ConvHaloArgs a = {};
    halo_common(a, pl, d->w, rows, 1);
    a.ntaps = 1;
    a.halo = 0;
    a.kd = 2;
    a.depth = 1;
    a.cblocks = std::max(1, 2 * d->cout / 64);   // cout = 32: one 64-wide block per row parity holds both column parities
    a.up_cpb = std::max(1, d->cout / 64);
    a.out = dx;
    a.ostride_x = d->x_ld;
    a.ostride_y = (long long)d->w * d->x_ld;
    a.ostride_n = 0;
    a.n_group = d->cin;
    a.n_total = d->cin;
    a.a_stages = res_stages;
    a.status = ctx->d_status;
    return res ? launch_halo_res<true, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, as_stream(stream))
               : launch_halo<true, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, as_stream(stream));
  }
  int tw, th, tn;
  pick_box(128, d->w, d->n * d->h, 1, &tw, &th, &tn);
  if (tn != 1) th *= tn;  // rows absorb the remainder (boxes may overhang; OOB rows are masked)
  const int bn = pick_bn(d->cin);
  CUtensorMap ta, tb;
  if ((rc = upsampled_map(ctx, dyr, d->cout, d->w, d->h, d->n, d->y_ld, tw, th, &ta))) return rc;
  if ((rc = matrix_map(ctx, w, d->cin, 4 * d->cout, 64, 64, &tb))) return rc;
  IgemmArgs a = {};
  const int tdim[4] = {1, d->w, 1, d->n * d->h};
  const int tbox[4] = {1, tw, 1, th};
  set_tiles(a, tdim, tbox);
  a.ntaps = 4;
  for (int ta_ = 0; ta_ < 2; ++ta_)
    for (int tb_ = 0; tb_ < 2; ++tb_) {
      signed char* o = a.tapoff[ta_ * 2 + tb_];
      o[0] = (signed char)tb_;
      o[1] = 0;
      o[2] = (signed char)ta_;
      o[3] = 0;
    }
  a.cblocks = d->cout / 64;
  a.out = dx;
  a.ostride[1] = d->x_ld;
  a.ostride[3] = (long long)d->w * d->x_ld;
  a.n_group = d->cin;
  a.n_total = d->cin;
  a.status = ctx->d_status;
  dim3 grid(a.ntile[1] * a.ntile[3], d->cin / bn, 1);
  return launch_igemm<MODE_PIX_M, true>(ctx, bn, ta, tb, a, grid, as_stream(stream));
}

static void convT_wgrad_plan(bsl_ctx* ctx, const bsl_convT2d_desc* d, int* tw, int* th, int* bn, int* m_tiles,
                             SplitPlan* p) {
  int tn;
  pick_box(64, d->w, d->n * d->h, 1, tw, th, &tn);
  if (tn != 1) *th *= tn;
  *bn = pick_bn(d->cin);
  *m_tiles = cdiv(4 * d->cout / 64, 2);
  const int k_tiles = cdiv(d->w, *tw) * cdiv(d->n * d->h, *th);
  *p = plan_split(ctx, *m_tiles * (d->cin / *bn), k_tiles);
}

size_t bsl_convT2d_bwd_filter_workspace(bsl_ctx* ctx, const bsl_convT2d_desc* d) {
  if (!ctx || !d || check_convT(ctx, d)) return 0;
  int tw, th, bn, m_tiles;
  SplitPlan p;
  convT_wgrad_plan(ctx, d, &tw, &th, &bn, &m_tiles, &p);
  return p.splits > 1 ? (size_t)p.splits * 4 * d->cout * d->cin * sizeof(float) : 0;
}

int bsl_convT2d_bwd_filter(bsl_ctx* ctx, const bsl_convT2d_desc* d, const void* x, const void* dyr,
                           float* dw, float* dbias, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_convT(ctx, d);
  if (rc) return rc;
  if (!x || !dyr || !dw) return bsl_fail(ctx, BSL_EINVAL, "convT2d_bwd_filter: null buffer");
  int tw, th, bn, m_tiles;
  SplitPlan p;
  convT_wgrad_plan(ctx, d, &tw, &th, &bn, &m_tiles, &p);
  CUtensorMap ta, tb;
  if ((rc = upsampled_map(ctx, dyr, d->cout, d->w, d->h, d->n, d->y_ld, tw, th, &ta))) return rc;
  if ((rc = rows_map(ctx, x, d->cin, d->w, d->h, d->n, d->x_ld, tw, th, &tb))) return rc;
  IgemmArgs a = {};
  const int tdim[4] = {1, d->w, 1, d->n * d->h};
  const int tbox[4] = {1, tw, 1, th};
  set_tiles(a, tdim, tbox);
  a.ntaps = 4;
  for (int ta_ = 0; ta_ < 2; ++ta_)
    for (int tb_ = 0; tb_ < 2; ++tb_) {
      signed char* o = a.tapoff[ta_ * 2 + tb_];
      o[0] = (signed char)tb_;
      o[1] = 0;
      o[2] = (signed char)ta_;
      o[3] = 0;
    }
  a.cblocks = d->cout / 64;
  if (d->cout == 32) {   // half-block form: a 64-row block = (b, co) of one row parity a
    a.ntaps = 2;
    a.cblocks = 1;
    for (int ta_ = 0; ta_ < 2; ++ta_) {
      signed char* o = a.tapoff[ta_];
      o[0] = 0;
      o[1] = 0;
      o[2] = (signed char)ta_;
      o[3] = 0;
    }
  }
  a.m_total = 4 * d->cout;
  a.n_total = d->cin;
  a.k_tiles_total = p.k_tiles;
  a.k_tiles_per_split = p.per;
  const size_t need = p.splits > 1 ? (size_t)p.splits * a.m_total * a.n_total * sizeof(float) : 0;
  if (need > workspace_bytes || (need && !workspace))
    return bsl_fail(ctx, BSL_EWORKSPACE, "convT2d_bwd_filter: workspace %zu < %zu", workspace_bytes, need);
  a.out = p.splits > 1 ? workspace : (void*)dw;
  a.status = ctx->d_status;
  dim3 grid(m_tiles, d->cin / bn, p.splits);
  rc = launch_igemm<MODE_PIX_K, true>(ctx, bn, ta, tb, a, grid, as_stream(stream));
  if (rc) return rc;
  if (p.splits > 1) {
    rc = reduce_splits(ctx, (const float*)workspace, dw, (long long)a.m_total * a.n_total, p.splits,
                       as_stream(stream));
    if (rc) return rc;
  }
  if (dbias)
    return bsl_channel_sum_bf16(ctx, dyr, (long long)d->n * 4 * d->h * d->w, d->cout, d->y_ld, dbias,
                                as_stream(stream));
  return BSL_OK;
}

}  // extern "C"

// ------------------------------------------------------------------ 3-D layers on the halo-tile kernels
// (3,3,3) and (1,3,3) stride-1 convolutions of UNet3D (NetworksV2/UNet3D.py:31-91): the reduction of the 2-D kernels
// gains an outer loop over the filter depth, each step reading the slice z + kd - 1 through a 5-D (c, w, h, d, n)
// tensor map (out-of-volume slices are zero-filled = SAME padding). Called from conv3d.cu.
namespace {
int ndhwc_halo_map(bsl_ctx* ctx, const void* base, int c, int w, int h, int dd, int n, int ld, int bw, int bh,
                   CUtensorMap* out) {
  uint64_t dims[5] = {(uint64_t)c, (uint64_t)w, (uint64_t)h, (uint64_t)dd, (uint64_t)n};
  uint64_t str[5] = {2, (uint64_t)ld * 2, (uint64_t)w * ld * 2, (uint64_t)h * w * ld * 2, (uint64_t)dd * h * w * ld * 2};
  uint32_t bx[5] = {64, (uint32_t)bw, (uint32_t)bh, 1, 1};
  return bsl_get_tmap(ctx, base, 5, dims, str, bx, out);
}
bool d3_stride1(const bsl_conv3d_desc* d) {
  return d->kh == 3 && d->kw == 3 && (d->kd == 1 || d->kd == 3) && d->sd == 1 && d->sh == 1 && d->sw == 1;
}
}  // namespace

bool bsl_conv3d_halo_ok(const bsl_conv3d_desc* d) { return d3_stride1(d) && halo_eligible(d->w, d->h); }

int bsl_conv3d_halo_fprop(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x, const void* w, void* y,
                          cudaStream_t stream, double* sums, bool per_volume) {
  HaloPlan pl = plan_halo(ctx, d->w, d->h, d->n * d->d, d->cout);
  int res_stages = 0, res_smem = 0;
  const bool res = plan_resident(pl.bn, 9 * d->kd, d->cin / 64, &pl.nsub, &res_stages, &res_smem);
  if (res) replan_units(ctx, pl);
  else pair_replan(ctx, pl, d->cout, 256, 9);
  CUtensorMap ta, tb;
  int rc;
  if ((rc = ndhwc_halo_map(ctx, x, d->cin, d->w, d->h, d->d, d->n, d->x_ld, 10, 18, &ta))) return rc;
  if ((rc = matrix_map(ctx, w, d->cout, d->kd * 9 * d->cin, 64, 64, &tb))) return rc;
  ConvHaloArgs a = {};
  halo_common(a, pl, d->w, d->h, d->n * d->d);
  a.ntaps = 9;
  a.halo = 1;
  a.cblocks = d->cin / 64;
  a.kd = d->kd;
  a.depth = d->d;
  a.out = y;
  a.ostride_x = d->y_ld;
  a.ostride_y = (long long)d->w * d->y_ld;
  a.ostride_n = (long long)d->h * d->w * d->y_ld;
  a.n_group = d->cout;
  a.n_total = d->cout;
  a.a_stages = res_stages;
  a.status = ctx->d_status;
  // per_volume: instance statistics per (volume, channel), a statistics group is the d slices of one volume;
  // otherwise batch statistics per channel over all n * d slices
  return launch_fprop_halo_stats(ctx, pl, res, res_smem, ta, tb, a, sums, per_volume ? d->d : 0, d->n * d->d, d->h, d->w,
                                 d->cout, y, d->y_ld, stream);
}

int bsl_conv3d_halo_dgrad(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* dy, const void* w, void* dx,
                          cudaStream_t stream) {
  HaloPlan pl = plan_halo(ctx, d->w, d->h, d->n * d->d, d->cin);
  int res_stages = 0, res_smem = 0;
  const bool res = plan_resident(pl.bn, 9 * d->kd, d->cout / 64, &pl.nsub, &res_stages, &res_smem);
  if (res) replan_units(ctx, pl);
  else pair_replan(ctx, pl, d->cin, 128, 9);
  CUtensorMap ta, tb;
  int rc;
  if ((rc = ndhwc_halo_map(ctx, dy, d->cout, d->w, d->h, d->d, d->n, d->y_ld, 10, 18, &ta))) return rc;
  if ((rc = matrix_map(ctx, w, d->cout, d->kd * 9 * d->cin, 64, pl.bn, &tb))) return rc;
  ConvHaloArgs a = {};
  halo_common(a, pl, d->w, d->h, d->n * d->d);
  a.ntaps = 9;
  a.halo = 1;
  a.cblocks = d->cout / 64;
  a.kd = d->kd;
  a.depth = d->d;
  a.b_flip = 1;
  a.b_rows_per_tap = d->cin;
  a.out = dx;
  a.ostride_x = d->x_ld;
  a.ostride_y = (long long)d->w * d->x_ld;
  a.ostride_n = (long long)d->h * d->w * d->x_ld;
  a.n_group = d->cin;
  a.n_total = d->cin;
  a.a_stages = res_stages;
  a.status = ctx->d_status;
  if (res) return launch_halo_res<false, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, stream);
  CUtensorMap tbh;
  const bool pair = pair_eligible(ctx, a, pl.bn, pl.nsub) &&
                    matrix_map(ctx, w, d->cout, d->kd * 9 * d->cin, 64, pl.bn / 2, &tbh) == 0;
  return launch_halo<false, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, stream, pair ? &tbh : nullptr);
}

// dgrad of a layer with stride 2 along H and / or W (stride 1 along D): one launch of the halo-tile kernel per output
// phase (parity class of the input coordinate). Within a phase, dx[s * u' + phase] = sum over the taps r with
// (phase + pad - r) % s == 0 of dy[u' + (phase + pad - r) / s] w[r]: a stride-1 correlation over dy whose offsets lie in
// {-1, 0, +1}, i.e. inside the 1-pixel halo of the box the kernel loads anyway, written to the strided positions of dx.
namespace {
struct PhaseTaps {
  int cnt, r[3], off[3];
};
PhaseTaps phase_taps(int in, int k, int s, int phase) {
  const int out = (in + s - 1) / s;
  const int pad = std::max((out - 1) * s + k - in, 0) / 2;
  PhaseTaps t = {};
  for (int r = 0; r < k; ++r) {
    const int v = phase + pad - r;
    if (((v % s) + s) % s) continue;
    t.r[t.cnt] = r;
    t.off[t.cnt] = (v >= 0 ? v : v - (s - 1)) / s;
    ++t.cnt;
  }
  return t;
}
}  // namespace

bool bsl_conv3d_halo_dgrad_strided_ok(const bsl_conv3d_desc* d) {
  if (d->sd != 1 || !(d->kd == 1 || d->kd == 3) || (d->sh == 1 && d->sw == 1)) return false;
  if (d->kh < 2 || d->kh > 3 || d->kw < 2 || d->kw > 3 || d->h % d->sh || d->w % d->sw) return false;
  if (!halo_eligible(d->w / d->sw, d->h / d->sh)) return false;
  for (int ph = 0; ph < d->sh; ++ph)
    for (int pw = 0; pw < d->sw; ++pw) {
      const PhaseTaps th = phase_taps(d->h, d->kh, d->sh, ph), tw = phase_taps(d->w, d->kw, d->sw, pw);
      if (th.cnt == 0 || tw.cnt == 0) return false;
      for (int i = 0; i < th.cnt; ++i)
        if (th.off[i] < -1 || th.off[i] > 1) return false;
      for (int i = 0; i < tw.cnt; ++i)
        if (tw.off[i] < -1 || tw.off[i] > 1) return false;
    }
  return true;
}

int bsl_conv3d_halo_dgrad_strided(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* dy, const void* w, void* dx,
                                  cudaStream_t stream) {
  const int pw_ = d->w / d->sw, ph_ = d->h / d->sh;          // phase grid = output grid (extents divide the strides)
  int rc;
  CUtensorMap ta;
  if ((rc = ndhwc_halo_map(ctx, dy, d->cout, pw_, ph_, d->d, d->n, d->y_ld, 10, 18, &ta))) return rc;
  for (int ph = 0; ph < d->sh; ++ph)
    for (int pw = 0; pw < d->sw; ++pw) {
      const PhaseTaps th = phase_taps(d->h, d->kh, d->sh, ph), tw = phase_taps(d->w, d->kw, d->sw, pw);
      HaloPlan pl = plan_halo(ctx, pw_, ph_, d->n * d->d, d->cin);
      const int ntaps = th.cnt * tw.cnt;
      int res_stages = 0, res_smem = 0;
      const bool res = plan_resident(pl.bn, ntaps * d->kd, d->cout / 64, &pl.nsub, &res_stages, &res_smem);
      if (res) replan_units(ctx, pl);
      CUtensorMap tb;
      if ((rc = matrix_map(ctx, w, d->cout, d->kd * d->kh * d->kw * d->cin, 64, pl.bn, &tb))) return rc;
      ConvHaloArgs a = {};
      halo_common(a, pl, pw_, ph_, d->n * d->d);
      a.ntaps = ntaps;
      a.halo = 1;
      a.cblocks = d->cout / 64;
      a.kd = d->kd;
      a.depth = d->d;
      a.b_rows_per_tap = d->cin;
      a.tap_table = 1;
      for (int i = 0; i < th.cnt; ++i)
        for (int j = 0; j < tw.cnt; ++j) {
          const int t = i * tw.cnt + j;
          a.tap_off[t] = ((th.off[i] + 1) * 10 + (tw.off[j] + 1)) * 128;
          // slice z + kdi - (kd >> 1) of dy meets filter depth tap q = kd - 1 - kdi (stride 1, SAME)
          for (int kdi = 0; kdi < d->kd; ++kdi)
            a.tap_b[kdi * ntaps + t] = (signed char)(((d->kd - 1 - kdi) * d->kh + th.r[i]) * d->kw + tw.r[j]);
        }
      a.out = reinterpret_cast<__nv_bfloat16*>(dx) + (long long)pw * d->x_ld + (long long)ph * d->w * d->x_ld;
      a.ostride_x = (long long)d->sw * d->x_ld;
      a.ostride_y = (long long)d->sh * d->w * d->x_ld;
      a.ostride_n = (long long)d->h * d->w * d->x_ld;
      a.n_group = d->cin;
      a.n_total = d->cin;
      a.a_stages = res_stages;
      a.status = ctx->d_status;
      rc = res ? launch_halo_res<false, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, res_smem, stream)
               : launch_halo<false, false, false>(ctx, pl.bn, pl.nsub, ta, tb, a, pl.grid, stream);
      if (rc) return rc;
    }
  return BSL_OK;
}

bool bsl_conv3d_halo_wgrad_ok(const bsl_conv3d_desc* d) {
  return d3_stride1(d) && tiles_ok(d->w, d->h, WG_TW, WG_TH);
}

namespace {
struct Wgrad3Plan {
  bool wide;
  WideWgradPlan w2;
  int k_tiles, per, splits;
  size_t ws_bytes;
};
Wgrad3Plan plan_wgrad3_halo_uncached(bsl_ctx* ctx, const bsl_conv3d_desc* d);

// The split search simulates block dispatch (~1 ms on the host): once per shape.
Wgrad3Plan plan_wgrad3_halo(bsl_ctx* ctx, const bsl_conv3d_desc* d) {
  static std::mutex mu;
  static std::unordered_map<std::string, Wgrad3Plan> cache;
  char key[96];
  snprintf(key, sizeof(key), "%d.%d.%d.%d.%d.%d.%d", d->n, d->d, d->h, d->w, d->cin, d->cout, d->kd);
  std::lock_guard<std::mutex> g(mu);
  auto it = cache.find(key);
  if (it == cache.end()) it = cache.emplace(key, plan_wgrad3_halo_uncached(ctx, d)).first;
  return it->second;
}

Wgrad3Plan plan_wgrad3_halo_uncached(bsl_ctx* ctx, const bsl_conv3d_desc* d) {
  Wgrad3Plan p = {};
  p.k_tiles = cdiv(d->w, WG_TW) * cdiv(d->h, WG_TH) * d->n * d->d;
  const size_t per_tap = (size_t)d->cin * d->cout;
  p.wide = d->cout % 128 == 0;
  if (p.wide) {
    p.w2 = plan_wgrad3_core(ctx, p.k_tiles, d->cin / 64, (d->cout / 128) * d->kd);
    p.ws_bytes = wgrad3_ws_bytes(p.w2, d->kd, per_tap);
  } else {
    const int mn = (d->cin / 64) * (d->cout / 64) * d->kd;
    int splits = std::max(1, ctx->sm_count / mn);
    splits = std::max(1, std::min(splits, p.k_tiles / 4));
    p.per = cdiv(p.k_tiles, splits);
    p.splits = cdiv(p.k_tiles, p.per);
    p.ws_bytes = p.splits > 1 ? (size_t)p.splits * d->kd * 9 * per_tap * sizeof(float) : 0;
  }
  return p;
}
}  // namespace

size_t bsl_conv3d_halo_wgrad_ws(bsl_ctx* ctx, const bsl_conv3d_desc* d) { return plan_wgrad3_halo(ctx, d).ws_bytes; }

int bsl_conv3d_halo_wgrad(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x, const void* dy, float* dw,
                          void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  const Wgrad3Plan p = plan_wgrad3_halo(ctx, d);
  if (p.ws_bytes > workspace_bytes || (p.ws_bytes && !workspace))
    return bsl_fail(ctx, BSL_EWORKSPACE, "conv3d_wgrad: workspace %zu < %zu", workspace_bytes, p.ws_bytes);
  CUtensorMap tx, ty;
  int rc;
  if ((rc = ndhwc_halo_map(ctx, x, d->cin, d->w, d->h, d->d, d->n, d->x_ld, WG_TW + 2, WG_TH + 2, &tx))) return rc;
  if ((rc = ndhwc_halo_map(ctx, dy, d->cout, d->w, d->h, d->d, d->n, d->y_ld, WG_TW, WG_TH, &ty))) return rc;
  const long long per_tap = (long long)d->cin * d->cout;
  float* ws = reinterpret_cast<float*>(workspace);
  if (p.wide) {
    CUtensorMap txa, txb;
    if ((rc = ndhwc_halo_map(ctx, x, d->cin, d->w, d->h, d->d, d->n, d->x_ld, WG_TW + 2, WG_TH + 1, &txa))) return rc;
    if ((rc = ndhwc_halo_map(ctx, x, d->cin, d->w, d->h, d->d, d->n, d->x_ld, WG_TW + 2, WG_TH, &txb))) return rc;
    return launch_wgrad3(ctx, p.w2, txa, txb, ty, d->w, d->h, d->n * d->d, d->cin, d->cout, d->kd, d->d, dw, workspace,
                         workspace_bytes, stream);
  }
  WgradHaloArgs a = {};
  a.ntile_w = cdiv(d->w, WG_TW);
  a.ntile_h = cdiv(d->h, WG_TH);
  a.n = d->n * d->d;
  a.k_tiles_total = p.k_tiles;
  a.k_tiles_per_split = p.per;
  a.cin = d->cin;
  a.cout = d->cout;
  a.out = p.splits > 1 ? ws : dw;
  a.kd = d->kd;
  a.depth = d->d;
  a.splits = p.splits;
  a.status = ctx->d_status;
  static bool configured1 = false;
  if (!configured1) {
    BSL_CUDA(ctx, cudaFuncSetAttribute(wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM_BYTES));
    configured1 = true;
  }
  bsl_launch(wgrad_halo_kernel, dim3(dim3(d->cin / 64, d->cout / 64, d->kd * p.splits)), dim3(WG_THREADS), WG_SMEM_BYTES, stream, tx, ty, a);
  BSL_LAUNCH_CHECK(ctx, "wgrad_halo_kernel launch (3-D)");
  if (p.splits > 1) return reduce_splits(ctx, ws, dw, (long long)d->kd * 9 * per_tap, p.splits, stream);
  return BSL_OK;
}
