// 3-D and strided convolutions of the UNet3D path on the tcgen05 implicit-GEMM kernel (igemm.cuh).
//   slim.conv3d(x, c, kernel (1|3,3,3), stride (1|2, 1|2, 1|2))   <- NetworksV2/UNet3D.py:31-91,151-168
//   slim.conv3d_transpose(x, c, kernel == stride (1|2,2,2), biases_initializer=None) + ReLU <- UNet3D.py:160-163
// Tensors are NDHWC bf16 seen by TMA as (c, w, h, d, n). Strided layers use TMA traversal strides
// (cuTensorMapEncodeTiled elementStrides): one box still lands 128 consecutive OUTPUT voxels in shared memory, at
// input coordinates out * stride + tap - pad_before, zero-filled out of bounds (TF "SAME": pad_before = pad_total / 2,
// the extra voxel goes to the far side). dgrad of a strided layer is decomposed into one launch per output phase
// (parity class of the input coordinate), each a small stride-1 correlation over dy with its own tap list.
// (1,3,3) stride-1 layers need none of this: they are bsl_conv2d_* over n * d images.
#include <algorithm>
#include "igemm.cuh"
#include "internal.h"

using namespace bsl;

namespace {

int cdiv(int a, int b) { return (a + b - 1) / b; }

template <int MODE, bool B_MN, int BN, int STAGES>
int launch3_one(bsl_ctx* ctx, const CUtensorMap& a, const CUtensorMap& b, const IgemmArgs& args_in, dim3 grid,
                cudaStream_t stream) {
  IgemmArgs args = args_in;
  args.mn_lbo = 8192;
  args.mn_sbo = 1024;
  args.mn_kadv = 2048;
  auto kern = igemm_kernel<MODE, B_MN, BN, STAGES>;
  constexpr int smem = igemm_smem_bytes<BN, STAGES>();
  static bool configured = false;
  if (!configured) {
    BSL_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  bsl_launch(kern, dim3(grid), dim3(IGEMM_THREADS), smem, stream, a, b, args);
  BSL_LAUNCH_CHECK(ctx, "igemm_kernel launch (3-D)");
  return BSL_OK;
}

template <int MODE, bool B_MN>
int launch3(bsl_ctx* ctx, int bn, const CUtensorMap& a, const CUtensorMap& b, const IgemmArgs& args, dim3 grid,
            cudaStream_t stream) {
  switch (bn) {
    case 64: return launch3_one<MODE, B_MN, 64, 4>(ctx, a, b, args, grid, stream);
    case 128: return launch3_one<MODE, B_MN, 128, 3>(ctx, a, b, args, grid, stream);
    case 256: return launch3_one<MODE, B_MN, 256, 4>(ctx, a, b, args, grid, stream);
  }
  return bsl_fail(ctx, BSL_EUNSUPPORTED, "igemm: column tile %d", bn);
}

int pick_bn(int n) { return n % 256 == 0 ? 256 : (n % 128 == 0 ? 128 : 64); }

// Box of `prod` voxels over (w, h, d, n), filled innermost first with powers of two.
void pick_box4(int prod, const int dim[4], int box[4]) {
  int left = prod;
  for (int i = 0; i < 4; ++i) {
    int b = 1;
    const int cap = i == 0 ? 16 : 128;
    while (b < cap && b < dim[i] && b < left) b <<= 1;
    box[i] = b;
    left = std::max(1, left / b);
  }
  // if the extents ran out before the product was reached, let the outermost dimension overhang (masked rows)
  int have = box[0] * box[1] * box[2] * box[3];
  while (have < prod) {
    box[3] <<= 1;
    have <<= 1;
  }
}

struct Geo {
  int in[3], out[3], k[3], s[3], pad[3];  // order: w, h, d
};

int geometry(bsl_ctx* ctx, const bsl_conv3d_desc* d, Geo* g) {
  if (!ctx) return BSL_EINVAL;
  if (!d) return bsl_fail(ctx, BSL_EINVAL, "conv3d: null descriptor");
  if (d->n <= 0 || d->d <= 0 || d->h <= 0 || d->w <= 0 || d->cin <= 0 || d->cout <= 0)
    return bsl_fail(ctx, BSL_EINVAL, "conv3d: non-positive size");
  const int in[3] = {d->w, d->h, d->d}, k[3] = {d->kw, d->kh, d->kd}, s[3] = {d->sw, d->sh, d->sd};
  for (int i = 0; i < 3; ++i) {
    // extent 2 (SAME: one voxel of padding on the far side): the strided conv that leaves UNet3D's pixel-pair packed
    // level reads super voxels X and X + 1
    if (k[i] < 1 || k[i] > 3 || !(s[i] == 1 || s[i] == 2))
      return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv3d: kernel extents 1..3 and strides 1|2 only");
    g->in[i] = in[i];
    g->k[i] = k[i];
    g->s[i] = s[i];
    g->out[i] = cdiv(in[i], s[i]);
    const int total = std::max((g->out[i] - 1) * s[i] + k[i] - in[i], 0);
    g->pad[i] = total / 2;
  }
  if (d->cin % 64 || d->cout % 64)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv3d tcgen05 path needs cin, cout multiples of 64 (got %d, %d): the "
                    "UNet3D engine stores 30/60/120/240 channels zero-padded to 64/64/128/256", d->cin, d->cout);
  if (d->x_ld < d->cin || d->y_ld < d->cout || d->x_ld % 8 || d->y_ld % 8)
    return bsl_fail(ctx, BSL_EINVAL, "conv3d: channel strides must be >= channels and multiples of 8");
  if (k[0] * k[1] * k[2] > 27) return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv3d: more than 27 taps");
  return BSL_OK;
}

// (c, w, h, d, n) map of an NDHWC tensor with pixel box `box` (w, h, d, n) and traversal strides es (w, h, d).
int ndhwc_map(bsl_ctx* ctx, const void* base, int c, const int dim[3], int n, int ld, const int box[4], const int es[3],
              CUtensorMap* out) {
  uint64_t dims[5] = {(uint64_t)c, (uint64_t)dim[0], (uint64_t)dim[1], (uint64_t)dim[2], (uint64_t)n};
  uint64_t str[5] = {2, (uint64_t)ld * 2, (uint64_t)dim[0] * ld * 2, (uint64_t)dim[1] * dim[0] * ld * 2,
                     (uint64_t)dim[2] * dim[1] * dim[0] * ld * 2};
  uint32_t bx[5] = {64, (uint32_t)(box[0] * es[0]), (uint32_t)(box[1] * es[1]), (uint32_t)(box[2] * es[2]),
                    (uint32_t)box[3]};
  uint32_t e[5] = {1, (uint32_t)es[0], (uint32_t)es[1], (uint32_t)es[2], 1};
  for (int i = 1; i < 5; ++i)
    if (bx[i] > 256) return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv3d: TMA box extent %u > 256", bx[i]);
  return bsl_get_tmap_es(ctx, base, 5, dims, str, bx, e, out);
}

int matrix_map(bsl_ctx* ctx, const void* base, int inner, int rows, int box_inner, int box_rows, CUtensorMap* out) {
  uint64_t dims[2] = {(uint64_t)inner, (uint64_t)rows};
  uint64_t str[2] = {2, (uint64_t)inner * 2};
  uint32_t bx[2] = {(uint32_t)box_inner, (uint32_t)box_rows};
  return bsl_get_tmap(ctx, base, 2, dims, str, bx, out);
}

void set_tiles4(IgemmArgs& a, const int dim[4], const int box[4], const int istride[4]) {
  for (int i = 0; i < 4; ++i) {
    a.tdim[i] = dim[i];
    a.tbox[i] = box[i];
    a.ntile[i] = cdiv(dim[i], box[i]);
    a.istride[i] = istride[i];
  }
}

struct SplitPlan {
  int k_tiles, per, splits;
};
SplitPlan plan_split(bsl_ctx* ctx, int mn_tiles, int k_tiles) {
  int want = std::max(1, (2 * ctx->sm_count + mn_tiles - 1) / mn_tiles);
  int splits = std::max(1, std::min(want, k_tiles / 8));
  int per = cdiv(k_tiles, splits);
  splits = cdiv(k_tiles, per);
  return {k_tiles, per, splits};
}

__global__ void reduce_splits3_kernel(const float* __restrict__ part, float* __restrict__ out, long long n, int splits) {
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

int reduce_splits3(bsl_ctx* ctx, const float* part, float* out, long long n, int splits, cudaStream_t s) {
  const int threads = 256;
  const long long blocks = (n / 4 + threads - 1) / threads;
  bsl_launch(reduce_splits3_kernel, dim3((unsigned)blocks), dim3(threads), 0, s, part, out, n, splits);
  BSL_LAUNCH_CHECK(ctx, "reduce_splits3_kernel");
  return BSL_OK;
}

struct WgradPlan3 {
  int box[4], bn, m_tiles, taps;
  SplitPlan sp;
};
WgradPlan3 plan_wgrad3(bsl_ctx* ctx, const bsl_conv3d_desc* d, const Geo& g) {
  WgradPlan3 p;
  const int odim[4] = {g.out[0], g.out[1], g.out[2], d->n};
  pick_box4(64, odim, p.box);
  p.taps = g.k[0] * g.k[1] * g.k[2];
  p.bn = pick_bn(d->cout);
  p.m_tiles = cdiv(p.taps * (d->cin / 64), 2);
  const int k_tiles = cdiv(odim[0], p.box[0]) * cdiv(odim[1], p.box[1]) * cdiv(odim[2], p.box[2]) * cdiv(odim[3], p.box[3]);
  p.sp = plan_split(ctx, p.m_tiles * (d->cout / p.bn), k_tiles);
  return p;
}

int check_convT3(bsl_ctx* ctx, const bsl_convT3d_desc* d) {
  if (!ctx) return BSL_EINVAL;
  if (!d) return bsl_fail(ctx, BSL_EINVAL, "convT3d: null descriptor");
  if (d->n <= 0 || d->d <= 0 || d->h <= 0 || d->w <= 0) return bsl_fail(ctx, BSL_EINVAL, "convT3d: non-positive size");
  if (d->sd != 1 && d->sd != 2) return bsl_fail(ctx, BSL_EUNSUPPORTED, "convT3d: kernel == stride (1|2, 2, 2) only");
  if (d->cin % 64 || d->cout % 64)
    return bsl_fail(ctx, BSL_EUNSUPPORTED, "convT3d needs cin, cout multiples of 64 (got %d, %d)", d->cin, d->cout);
  if (d->x_ld < d->cin || d->y_ld < d->cout || d->x_ld % 8 || d->y_ld % 8)
    return bsl_fail(ctx, BSL_EINVAL, "convT3d: bad channel strides");
  return BSL_OK;
}

// taps of the transposed conv in filter order [kd][2][2]: offsets (b, a, c) into the (2w, 2h, sd*d) output grid
void convT3_taps(IgemmArgs& a, int sd) {
  a.ntaps = sd * 4;
  for (int c = 0; c < sd; ++c)
    for (int ta = 0; ta < 2; ++ta)
      for (int tb = 0; tb < 2; ++tb) {
        signed char* o = a.tapoff[(c * 2 + ta) * 2 + tb];
        o[0] = (signed char)tb;
        o[1] = (signed char)ta;
        o[2] = (signed char)c;
        o[3] = 0;
      }
}

}  // namespace

extern "C" {

int bsl_conv3d_fprop(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x, const void* w, void* y, void* stream) {
  Geo g;
  int rc = geometry(ctx, d, &g);
  if (rc) return rc;
  if (!x || !w || !y) return bsl_fail(ctx, BSL_EINVAL, "conv3d_fprop: null buffer");
  if (bsl_conv3d_halo_ok(d)) return bsl_conv3d_halo_fprop(ctx, d, x, w, y, as_stream(stream));
  const int odim[4] = {g.out[0], g.out[1], g.out[2], d->n};
  int box[4];
  pick_box4(128, odim, box);
  const int bn = pick_bn(d->cout);
  const int taps = g.k[0] * g.k[1] * g.k[2];
  CUtensorMap ta, tb;
  if ((rc = ndhwc_map(ctx, x, d->cin, g.in, d->n, d->x_ld, box, g.s, &ta))) return rc;
  if ((rc = matrix_map(ctx, w, d->cout, taps * d->cin, 64, 64, &tb))) return rc;
  IgemmArgs a = {};
  const int istride[4] = {g.s[0], g.s[1], g.s[2], 1};
  set_tiles4(a, odim, box, istride);
  a.ntaps = taps;
  for (int q = 0; q < g.k[2]; ++q)
    for (int r = 0; r < g.k[1]; ++r)
      for (int s = 0; s < g.k[0]; ++s) {
        signed char* o = a.tapoff[(q * g.k[1] + r) * g.k[0] + s];
        o[0] = (signed char)(s - g.pad[0]);
        o[1] = (signed char)(r - g.pad[1]);
        o[2] = (signed char)(q - g.pad[2]);
        o[3] = 0;
      }
  a.cblocks = d->cin / 64;
  a.out = y;
  a.ostride[0] = d->y_ld;
  a.ostride[1] = (long long)g.out[0] * d->y_ld;
  a.ostride[2] = (long long)g.out[1] * g.out[0] * d->y_ld;
  a.ostride[3] = (long long)g.out[2] * g.out[1] * g.out[0] * d->y_ld;
  a.n_group = d->cout;
  a.n_total = d->cout;
  a.status = ctx->d_status;
  dim3 grid(a.ntile[0] * a.ntile[1] * a.ntile[2] * a.ntile[3], d->cout / bn, 1);
  return launch3<MODE_PIX_M, true>(ctx, bn, ta, tb, a, grid, as_stream(stream));
}

// fprop + per-(volume, channel) sum and sum of squares of the bf16 outputs (instance norm over a volume): fused into
// the epilogue where the layer runs on the halo-tile kernel, else a separate pass over y.
int bsl_conv3d_fprop_group_stats(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x, const void* w, void* y,
                                 double* sums, void* stream) {
  Geo g;
  int rc = geometry(ctx, d, &g);
  if (rc) return rc;
  if (!x || !w || !y || !sums) return bsl_fail(ctx, BSL_EINVAL, "conv3d_fprop_group_stats: null buffer");
  if (bsl_conv3d_halo_ok(d)) return bsl_conv3d_halo_fprop(ctx, d, x, w, y, as_stream(stream), sums);
  if ((rc = bsl_conv3d_fprop(ctx, d, x, w, y, stream))) return rc;
  return bsl_stats_bf16(ctx, y, (long long)g.out[0] * g.out[1] * g.out[2], d->n, d->cout, d->y_ld, sums,
                        as_stream(stream));
}

// fprop + per-channel sum and sum of squares of the bf16 outputs over the whole batch (batch norm): the same two paths,
// with one statistics group.
int bsl_conv3d_fprop_stats(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x, const void* w, void* y, double* sums,
                           void* stream) {
  Geo g;
  int rc = geometry(ctx, d, &g);
  if (rc) return rc;
  if (!x || !w || !y || !sums) return bsl_fail(ctx, BSL_EINVAL, "conv3d_fprop_stats: null buffer");
  if (bsl_conv3d_halo_ok(d)) return bsl_conv3d_halo_fprop(ctx, d, x, w, y, as_stream(stream), sums, false);
  if ((rc = bsl_conv3d_fprop(ctx, d, x, w, y, stream))) return rc;
  return bsl_stats_bf16(ctx, y, (long long)d->n * g.out[0] * g.out[1] * g.out[2], 1, d->cout, d->y_ld, sums,
                        as_stream(stream));
}

int bsl_conv3d_dgrad(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* dy, const void* w, void* dx, void* stream) {
  Geo g;
  int rc = geometry(ctx, d, &g);
  if (rc) return rc;
  if (!dy || !w || !dx) return bsl_fail(ctx, BSL_EINVAL, "conv3d_dgrad: null buffer");
  if (bsl_conv3d_halo_ok(d)) return bsl_conv3d_halo_dgrad(ctx, d, dy, w, dx, as_stream(stream));
  if (bsl_conv3d_halo_dgrad_strided_ok(d))
    return bsl_conv3d_halo_dgrad_strided(ctx, d, dy, w, dx, as_stream(stream));
  for (int i = 0; i < 3; ++i)
    if (g.in[i] % g.s[i]) return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv3d_dgrad: extents must be multiples of the stride");
  const int bn = pick_bn(d->cin);
  const int taps = g.k[0] * g.k[1] * g.k[2];
  const int es1[3] = {1, 1, 1};
  CUtensorMap tb;
  // DHWIO read as a K-major B: row = tap * cin + ci (GEMM column), 64 consecutive cout = GEMM K
  if ((rc = matrix_map(ctx, w, d->cout, taps * d->cin, 64, bn, &tb))) return rc;
  const long long xs[3] = {d->x_ld, (long long)g.in[0] * d->x_ld, (long long)g.in[1] * g.in[0] * d->x_ld};
  const long long xn = (long long)g.in[2] * g.in[1] * g.in[0] * d->x_ld;
  // one launch per phase (ph[i] = input coordinate mod stride); stride-1 dimensions have a single phase
  for (int pd = 0; pd < g.s[2]; ++pd)
    for (int ph = 0; ph < g.s[1]; ++ph)
      for (int pw = 0; pw < g.s[0]; ++pw) {
        const int phase[3] = {pw, ph, pd};
        // dx[u] = sum_r dy[(u + pad - r) / s] w[r] over r with (u + pad - r) % s == 0; u = s * i + phase
        int cnt[3], rr[3][3], off[3][3];
        for (int i = 0; i < 3; ++i) {
          cnt[i] = 0;
          for (int r = 0; r < g.k[i]; ++r) {
            const int t = phase[i] + g.pad[i] - r;
            if (((t % g.s[i]) + g.s[i]) % g.s[i]) continue;
            rr[i][cnt[i]] = r;
            off[i][cnt[i]] = (t >= 0 ? t : t - (g.s[i] - 1)) / g.s[i];  // floor division
            ++cnt[i];
          }
        }
        const int pdim[4] = {g.in[0] / g.s[0], g.in[1] / g.s[1], g.in[2] / g.s[2], d->n};
        __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(dx) + pw * xs[0] + ph * xs[1] + pd * xs[2];
        int box[4];
        pick_box4(128, pdim, box);
        IgemmArgs a = {};
        const int one[4] = {1, 1, 1, 1};
        set_tiles4(a, pdim, box, one);
        a.ntaps = cnt[0] * cnt[1] * cnt[2];
        a.cblocks = d->cout / 64;
        a.b_flip = 2;
        a.b_rows_per_tap = d->cin;
        int t = 0;
        for (int q = 0; q < cnt[2]; ++q)
          for (int r = 0; r < cnt[1]; ++r)
            for (int s = 0; s < cnt[0]; ++s, ++t) {
              a.tapoff[t][0] = (signed char)off[0][s];
              a.tapoff[t][1] = (signed char)off[1][r];
              a.tapoff[t][2] = (signed char)off[2][q];
              a.tapoff[t][3] = 0;
              a.tapb[t] = (signed char)((rr[2][q] * g.k[1] + rr[1][r]) * g.k[0] + rr[0][s]);
            }
        a.out = out;
        a.ostride[0] = g.s[0] * xs[0];
        a.ostride[1] = g.s[1] * xs[1];
        a.ostride[2] = g.s[2] * xs[2];
        a.ostride[3] = xn;
        a.n_group = d->cin;
        a.n_total = d->cin;
        a.status = ctx->d_status;
        CUtensorMap ta;
        if ((rc = ndhwc_map(ctx, dy, d->cout, g.out, d->n, d->y_ld, box, es1, &ta))) return rc;
        dim3 grid(a.ntile[0] * a.ntile[1] * a.ntile[2] * a.ntile[3], d->cin / bn, 1);
        if (a.ntaps == 0) return bsl_fail(ctx, BSL_EUNSUPPORTED, "conv3d_dgrad: empty phase");
        if ((rc = launch3<MODE_PIX_M, false>(ctx, bn, ta, tb, a, grid, as_stream(stream)))) return rc;
      }
  return BSL_OK;
}

size_t bsl_conv3d_wgrad_workspace(bsl_ctx* ctx, const bsl_conv3d_desc* d) {
  Geo g;
  if (!ctx || !d || geometry(ctx, d, &g)) return 0;
  if (bsl_conv3d_halo_wgrad_ok(d)) return bsl_conv3d_halo_wgrad_ws(ctx, d);
  const WgradPlan3 p = plan_wgrad3(ctx, d, g);
  return p.sp.splits > 1 ? (size_t)p.sp.splits * p.taps * d->cin * d->cout * sizeof(float) : 0;
}

int bsl_conv3d_wgrad(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x, const void* dy, float* dw, void* workspace,
                     size_t workspace_bytes, void* stream) {
  Geo g;
  int rc = geometry(ctx, d, &g);
  if (rc) return rc;
  if (!x || !dy || !dw) return bsl_fail(ctx, BSL_EINVAL, "conv3d_wgrad: null buffer");
  if (bsl_conv3d_halo_wgrad_ok(d))
    return bsl_conv3d_halo_wgrad(ctx, d, x, dy, dw, workspace, workspace_bytes, as_stream(stream));
  const WgradPlan3 p = plan_wgrad3(ctx, d, g);
  const int odim[4] = {g.out[0], g.out[1], g.out[2], d->n};
  const int es1[3] = {1, 1, 1};
  CUtensorMap ta, tb;
  if ((rc = ndhwc_map(ctx, x, d->cin, g.in, d->n, d->x_ld, p.box, g.s, &ta))) return rc;
  if ((rc = ndhwc_map(ctx, dy, d->cout, g.out, d->n, d->y_ld, p.box, es1, &tb))) return rc;
  IgemmArgs a = {};
  const int istride[4] = {g.s[0], g.s[1], g.s[2], 1};
  set_tiles4(a, odim, p.box, istride);
  a.ntaps = p.taps;
  for (int q = 0; q < g.k[2]; ++q)
    for (int r = 0; r < g.k[1]; ++r)
      for (int s = 0; s < g.k[0]; ++s) {
        signed char* o = a.tapoff[(q * g.k[1] + r) * g.k[0] + s];
        o[0] = (signed char)(s - g.pad[0]);
        o[1] = (signed char)(r - g.pad[1]);
        o[2] = (signed char)(q - g.pad[2]);
        o[3] = 0;
      }
  a.cblocks = d->cin / 64;
  a.m_total = p.taps * d->cin;
  a.n_total = d->cout;
  a.k_tiles_total = p.sp.k_tiles;
  a.k_tiles_per_split = p.sp.per;
  const size_t need = p.sp.splits > 1 ? (size_t)p.sp.splits * a.m_total * a.n_total * sizeof(float) : 0;
  if (need > workspace_bytes || (need && !workspace))
    return bsl_fail(ctx, BSL_EWORKSPACE, "conv3d_wgrad: workspace %zu < %zu", workspace_bytes, need);
  a.out = p.sp.splits > 1 ? workspace : (void*)dw;
  a.status = ctx->d_status;
  dim3 grid(p.m_tiles, d->cout / p.bn, p.sp.splits);
  if ((rc = launch3<MODE_PIX_K, true>(ctx, p.bn, ta, tb, a, grid, as_stream(stream)))) return rc;
  if (p.sp.splits > 1)
    return reduce_splits3(ctx, (const float*)workspace, dw, (long long)a.m_total * a.n_total, p.sp.splits,
                          as_stream(stream));
  return BSL_OK;
}

// ------------------------------------------------------------------ transposed conv, kernel == stride (sd, 2, 2)

int bsl_convT3d_fwd(bsl_ctx* ctx, const bsl_convT3d_desc* d, const void* x, const void* w, const float* bias, void* y,
                    void* stream) {
  int rc = check_convT3(ctx, d);
  if (rc) return rc;
  if (!x || !w || !y) return bsl_fail(ctx, BSL_EINVAL, "convT3d_fwd: null buffer");
  const int taps = 4 * d->sd;
  const int dim3_[3] = {d->w, d->h, d->d};
  const int pdim[4] = {d->w, d->h, d->d, d->n};
  int box[4];
  pick_box4(128, pdim, box);
  const int bn = pick_bn(d->cout);
  const int es1[3] = {1, 1, 1};
  CUtensorMap ta, tb;
  if ((rc = ndhwc_map(ctx, x, d->cin, dim3_, d->n, d->x_ld, box, es1, &ta))) return rc;
  // [kd,2,2,cout,cin]: row = tap * cout + co (GEMM column), cin contiguous (GEMM K) => K-major B
  if ((rc = matrix_map(ctx, w, d->cin, taps * d->cout, 64, bn, &tb))) return rc;
  IgemmArgs a = {};
  const int one[4] = {1, 1, 1, 1};
  set_tiles4(a, pdim, box, one);
  a.ntaps = 1;
  a.cblocks = d->cin / 64;
  a.out = y;
  const long long row = (long long)2 * d->w * d->y_ld, plane = (long long)2 * d->h * row;
  a.ostride[0] = 2 * d->y_ld;
  a.ostride[1] = 2 * row;
  a.ostride[2] = d->sd * plane;
  a.ostride[3] = (long long)d->sd * d->d * plane;
  a.n_group = d->cout;
  for (int c = 0; c < d->sd; ++c)
    for (int ta_ = 0; ta_ < 2; ++ta_)
      for (int tb_ = 0; tb_ < 2; ++tb_)
        a.group_off[(c * 2 + ta_) * 2 + tb_] = c * plane + ta_ * row + (long long)tb_ * d->y_ld;
  a.bias = bias;
  a.relu = d->relu;
  a.n_total = taps * d->cout;
  a.status = ctx->d_status;
  dim3 grid(a.ntile[0] * a.ntile[1] * a.ntile[2] * a.ntile[3], taps * d->cout / bn, 1);
  return launch3<MODE_PIX_M, false>(ctx, bn, ta, tb, a, grid, as_stream(stream));
}

int bsl_convT3d_bwd_data(bsl_ctx* ctx, const bsl_convT3d_desc* d, const void* dyr, const void* w, void* dx,
                         void* stream) {
  int rc = check_convT3(ctx, d);
  if (rc) return rc;
  if (!dyr || !w || !dx) return bsl_fail(ctx, BSL_EINVAL, "convT3d_bwd_data: null buffer");
  const int taps = 4 * d->sd;
  const int odim3[3] = {2 * d->w, 2 * d->h, d->sd * d->d};
  const int pdim[4] = {d->w, d->h, d->d, d->n};
  int box[4];
  pick_box4(128, pdim, box);
  const int bn = pick_bn(d->cin);
  const int es[3] = {2, 2, d->sd};
  CUtensorMap ta, tb;
  if ((rc = ndhwc_map(ctx, dyr, d->cout, odim3, d->n, d->y_ld, box, es, &ta))) return rc;
  if ((rc = matrix_map(ctx, w, d->cin, taps * d->cout, 64, 64, &tb))) return rc;
  IgemmArgs a = {};
  const int istride[4] = {2, 2, d->sd, 1};
  set_tiles4(a, pdim, box, istride);
  convT3_taps(a, d->sd);
  a.cblocks = d->cout / 64;
  a.out = dx;
  a.ostride[0] = d->x_ld;
  a.ostride[1] = (long long)d->w * d->x_ld;
  a.ostride[2] = (long long)d->h * d->w * d->x_ld;
  a.ostride[3] = (long long)d->d * d->h * d->w * d->x_ld;
  a.n_group = d->cin;
  a.n_total = d->cin;
  a.status = ctx->d_status;
  dim3 grid(a.ntile[0] * a.ntile[1] * a.ntile[2] * a.ntile[3], d->cin / bn, 1);
  return launch3<MODE_PIX_M, true>(ctx, bn, ta, tb, a, grid, as_stream(stream));
}

static void convT3_wgrad_plan(bsl_ctx* ctx, const bsl_convT3d_desc* d, int box[4], int* bn, int* m_tiles, SplitPlan* p) {
  const int pdim[4] = {d->w, d->h, d->d, d->n};
  pick_box4(64, pdim, box);
  *bn = pick_bn(d->cin);
  *m_tiles = cdiv(4 * d->sd * d->cout / 64, 2);
  const int k_tiles = cdiv(pdim[0], box[0]) * cdiv(pdim[1], box[1]) * cdiv(pdim[2], box[2]) * cdiv(pdim[3], box[3]);
  *p = plan_split(ctx, *m_tiles * (d->cin / *bn), k_tiles);
}

size_t bsl_convT3d_bwd_filter_workspace(bsl_ctx* ctx, const bsl_convT3d_desc* d) {
  if (!ctx || !d || check_convT3(ctx, d)) return 0;
  int box[4], bn, m_tiles;
  SplitPlan p;
  convT3_wgrad_plan(ctx, d, box, &bn, &m_tiles, &p);
  return p.splits > 1 ? (size_t)p.splits * 4 * d->sd * d->cout * d->cin * sizeof(float) : 0;
}

int bsl_convT3d_bwd_filter(bsl_ctx* ctx, const bsl_convT3d_desc* d, const void* x, const void* dyr, float* dw,
                           float* dbias, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_convT3(ctx, d);
  if (rc) return rc;
  if (!x || !dyr || !dw) return bsl_fail(ctx, BSL_EINVAL, "convT3d_bwd_filter: null buffer");
  int box[4], bn, m_tiles;
  SplitPlan p;
  convT3_wgrad_plan(ctx, d, box, &bn, &m_tiles, &p);
  const int taps = 4 * d->sd;
  const int odim3[3] = {2 * d->w, 2 * d->h, d->sd * d->d}, idim3[3] = {d->w, d->h, d->d};
  const int pdim[4] = {d->w, d->h, d->d, d->n};
  const int es[3] = {2, 2, d->sd}, es1[3] = {1, 1, 1};
  CUtensorMap ta, tb;
  if ((rc = ndhwc_map(ctx, dyr, d->cout, odim3, d->n, d->y_ld, box, es, &ta))) return rc;
  if ((rc = ndhwc_map(ctx, x, d->cin, idim3, d->n, d->x_ld, box, es1, &tb))) return rc;
  IgemmArgs a = {};
  const int istride[4] = {2, 2, d->sd, 1};
  set_tiles4(a, pdim, box, istride);
  convT3_taps(a, d->sd);
  a.cblocks = d->cout / 64;
  a.m_total = taps * d->cout;
  a.n_total = d->cin;
  a.k_tiles_total = p.k_tiles;
  a.k_tiles_per_split = p.per;
  const size_t need = p.splits > 1 ? (size_t)p.splits * a.m_total * a.n_total * sizeof(float) : 0;
  if (need > workspace_bytes || (need && !workspace))
    return bsl_fail(ctx, BSL_EWORKSPACE, "convT3d_bwd_filter: workspace %zu < %zu", workspace_bytes, need);
  a.out = p.splits > 1 ? workspace : (void*)dw;
  a.status = ctx->d_status;
  dim3 grid(m_tiles, d->cin / bn, p.splits);
  if ((rc = launch3<MODE_PIX_K, true>(ctx, bn, ta, tb, a, grid, as_stream(stream)))) return rc;
  if (p.splits > 1) {
    rc = reduce_splits3(ctx, (const float*)workspace, dw, (long long)a.m_total * a.n_total, p.splits, as_stream(stream));
    if (rc) return rc;
  }
  if (dbias)
    return bsl_channel_sum_bf16(ctx, dyr, (long long)d->n * taps * d->d * d->h * d->w, d->cout, d->y_ld, dbias,
                                as_stream(stream));
  return BSL_OK;
}

}  // extern "C"
