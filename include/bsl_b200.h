/* bsl_b200.h -- C ABI of the B200-native U-Net hot path for BoxSegLiver.
 *
 * The reference (Jarvis73/BoxSegLiver) has no FFI of its own: its model code calls TF-slim layer
 * functions and TF 1.13 dispatches registered op kernels below them (SURVEY.md section 8b). Each
 * entry point here is the enqueue-only body of the TF op kernel it replaces; the citation on every
 * function names the reference call site whose op it stands in for. Rules of the boundary:
 *
 *   - plain pointers and sizes only; device buffers are owned by the caller (TF allocator, or
 *     bsl_malloc for the ctypes host in boxsegliver_b200/), the library owns only its context;
 *   - every compute call only ENQUEUES on `stream` (a cudaStream_t passed as void*), never
 *     synchronises and never touches the default stream;
 *   - return 0 on success, a negative BSL_E* code otherwise; bsl_last_error(ctx) has the text;
 *   - activations / gradients are NHWC bf16 with an explicit channel stride `*_ld` (elements) so a
 *     skip-concat (UNet.py:93) is two views of one buffer, never a copy;
 *   - conv filters are HWIO (TF variable layout, `weights`), transposed-conv filters are
 *     [kh,kw,Cout,Cin] (slim.conv2d_transpose variable layout); fp32 masters, bf16 shadows.
 */
#ifndef BSL_B200_H_
#define BSL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bsl_ctx bsl_ctx;

enum {
  BSL_OK = 0,
  BSL_EINVAL = -1,       /* malformed descriptor / null pointer */
  BSL_EUNSUPPORTED = -2, /* shape outside what the sm_100a kernels cover */
  BSL_EWORKSPACE = -3,   /* workspace too small */
  BSL_ECUDA = -4,        /* CUDA runtime / driver error */
  BSL_EDEVICE = -5,      /* device-side pipeline watchdog fired (see bsl_device_status) */
  BSL_ENCCL = -6
};

/* ------------------------------------------------------------------ context, memory, streams */
int bsl_init(int device, bsl_ctx** out);
void bsl_destroy(bsl_ctx* ctx);
const char* bsl_last_error(bsl_ctx* ctx);
const char* bsl_version(void);
/* Host-only helper: running CRC-32C (Castagnoli) as used by TF's Saver V2 bundles (core/estimator.py:694-703 saves
 * and restores through tf.train.Saver; boxsegliver_b200/checkpoint.py reads / writes that wire format). */
unsigned bsl_crc32c(unsigned crc, const void* data, size_t n);
/* Reads back (synchronously) and clears the device-side watchdog word. 0 = healthy. */
int bsl_device_status(bsl_ctx* ctx, int* block, int* site);

/* Number of kernels enqueued through this context since bsl_init (host-side counter). */
int bsl_launch_count(bsl_ctx* ctx, unsigned long long* out);

/* Probe hook: overrides a layout constant of the UMMA descriptors (tools/gpu_conv_probe.py). */
int bsl_debug_set(bsl_ctx* ctx, int key, int value);
/* Tuning aid: with bsl_debug_set(ctx, 3, 1) the UMMA issuer thread of every conv_halo CTA records {total cycles,
 * cycles waiting for a free accumulator, for an activation stage, for a filter stage} of its last launch. */
int bsl_debug_read_waits(bsl_ctx* ctx, long long* out /*[ctas][4]*/, int ctas);

/* cudaMemGetInfo of the context's device (bench.py sizes the strong-scaling points with it). */
int bsl_mem_info(bsl_ctx* ctx, size_t* free_bytes, size_t* total_bytes);
int bsl_malloc(bsl_ctx* ctx, size_t bytes, void** out);
int bsl_free(bsl_ctx* ctx, void* ptr);
int bsl_memset(bsl_ctx* ctx, void* dst, int value, size_t bytes, void* stream);
int bsl_memcpy_h2d(bsl_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream);
int bsl_memcpy_d2h(bsl_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream);
int bsl_memcpy_d2d(bsl_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream);
int bsl_host_alloc(bsl_ctx* ctx, size_t bytes, void** out); /* pinned */
int bsl_host_free(bsl_ctx* ctx, void* ptr);
int bsl_stream_create(bsl_ctx* ctx, void** out);
int bsl_stream_destroy(bsl_ctx* ctx, void* stream);
int bsl_stream_sync(bsl_ctx* ctx, void* stream);
int bsl_event_create(bsl_ctx* ctx, void** out);
int bsl_event_destroy(bsl_ctx* ctx, void* ev);
int bsl_event_record(bsl_ctx* ctx, void* ev, void* stream);
int bsl_event_sync(bsl_ctx* ctx, void* ev);
int bsl_stream_wait_event(bsl_ctx* ctx, void* stream, void* ev);
int bsl_event_elapsed_ms(bsl_ctx* ctx, void* start, void* stop, float* ms);
/* CUDA-graph capture of an enqueue sequence (the training step is launch-bound at small batch). */
int bsl_graph_begin(bsl_ctx* ctx, void* stream);
int bsl_graph_end(bsl_ctx* ctx, void* stream, void** graph_exec);
int bsl_graph_launch(bsl_ctx* ctx, void* graph_exec, void* stream);
int bsl_graph_destroy(bsl_ctx* ctx, void* graph_exec);

/* ------------------------------------------------------------------ dtype casts (fp32 <-> bf16) */
int bsl_cast_f32_to_bf16(bsl_ctx* ctx, const float* src, void* dst, size_t n, void* stream);
int bsl_cast_bf16_to_f32(bsl_ctx* ctx, const void* src, float* dst, size_t n, void* stream);
/* x *= a in place (cross-replica MEAN of the batch-norm moving statistics after a SUM all-reduce). */
int bsl_scale_f32(bsl_ctx* ctx, float* x, size_t n, float a, void* stream);
/* Filter re-layout by index table and its adjoint (the UNet3D engine's pixel-pair packing: the 30-channel full-resolution
 * layers of NetworksV2/UNet3D.py:31-91 run as 64-channel convolutions over PAIRS of horizontally adjacent voxels, whose
 * "super" filter is a fixed re-arrangement of the slim variable): dst[i] = bf16(src[idx[i]]) (0 where idx[i] < 0), and
 * dst[j] = src[idx2[2j]] + src[idx2[2j+1]] (terms with a negative index dropped) for the filter gradient. */
int bsl_gather_f32_bf16(bsl_ctx* ctx, const float* src, const int* idx, size_t n, void* dst_bf16, void* stream);
int bsl_gather_add2_f32(bsl_ctx* ctx, const float* src, const int* idx2, size_t n, float* dst, void* stream);
/* Moments of a pixel-pair packed tensor from the statistics of its 2c "super" channels (voxel parity, lane):
 * src fp64 [groups][2][2c] -> dst fp64 [groups][2][c], dst[g][k][ch] = src[g][k][ch] + src[g][k][c + ch]. */
int bsl_fold_pair_sums(bsl_ctx* ctx, const double* src, int groups, int c, double* dst, void* stream);

/* ------------------------------------------------------------------ conv2d, stride 1, SAME
 * Replaces TF ops Conv2D / Conv2DBackpropInput / Conv2DBackpropFilter behind
 * slim.conv2d(x, C, 3) -- NetworksV2/UNet.py:79,85,94 -- and their gradients created by
 * optimizer.minimize, core/solver.py:239. tcgen05 implicit GEMM when cin % 64 == 0 and
 * cout % 64 == 0; a direct CUDA-core kernel for the stem (cin < 64, UNet.py:79 first call). */
typedef struct {
  int n, h, w;     /* batch and spatial size (output == input size: stride 1, SAME) */
  int cin, cout;
  int kh, kw;      /* 3x3 or 1x1 */
  int x_ld;        /* channel stride of the input buffer (elements), >= cin. fprop / wgrad also take x_ld < cin
                    * (multiple of 8): rows then hold only x_ld channels and channels >= x_ld read as zero */
  int y_ld;        /* channel stride of the output buffer (elements), >= cout */
} bsl_conv2d_desc;

int bsl_conv2d_fprop(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x_bf16,
                     const void* w_hwio_bf16, void* y_bf16, void* stream);
/* Conv2D fused with the reduction half of FusedBatchNorm (NetworksV2/base.py:154-162): also returns
 * sums[0][c] = sum over (n,h,w) of y, sums[1][c] = sum of y^2 (of the bf16-rounded outputs, fp64), which is
 * exactly what bsl_norm_stats(mode = batch) computes from y in a separate pass. */
int bsl_conv2d_fprop_stats(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x_bf16,
                           const void* w_hwio_bf16, void* y_bf16, double* sums, void* stream);
/* Same fusion for slim.instance_norm (and UNet3D's (1,3,3) layers, whose depth slices run as images): sums is
 * fp64 [n / imgs_per_group][2][cout], one statistics group per `imgs_per_group` consecutive images (1 for a 2-D
 * instance norm, the volume depth for NDHWC tensors viewed as n*d images). Equals bsl_conv2d_fprop followed by
 * bsl_norm_stats in instance mode; the bf16 outputs are bit-identical. */
int bsl_conv2d_fprop_group_stats(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x_bf16, const void* w_bf16,
                                 void* y_bf16, int imgs_per_group, double* sums, void* stream);
/* slim.conv2d with normalizer_fn=None (--without_norm): y = bf16(relu(conv(x, w) + bias[c])), one rounding after the
 * ReLU. bias is fp32 [cout] (the master copy of the `biases` variable). Same descriptor rules, strides and kernel
 * schedules as bsl_conv2d_fprop; with a zero bias the output equals relu(bsl_conv2d_fprop) bit for bit. */
int bsl_conv2d_fprop_bias_relu(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x_bf16, const void* w_hwio_bf16,
                               const float* bias_f32, void* y_bf16, void* stream);
/* dx = dgrad(dy, w); dy has stride y_ld, dx has stride x_ld. */
int bsl_conv2d_dgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* dy_bf16,
                     const void* w_hwio_bf16, void* dx_bf16, void* stream);
size_t bsl_conv2d_wgrad_workspace(bsl_ctx* ctx, const bsl_conv2d_desc* d);
/* dw (fp32, HWIO) = wgrad(x, dy). Split-K partials go to `workspace` and are reduced in a fixed
 * order (bit-reproducible). */
int bsl_conv2d_wgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x_bf16, const void* dy_bf16,
                     float* dw_hwio_f32, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ conv2d_transpose k2 s2
 * Replaces Conv2DBackpropInput-as-forward + BiasAdd + Relu behind
 * slim.conv2d_transpose(x, C/2, 2, 2) -- NetworksV2/UNet.py:91 -- and its gradients.
 * x: [n,h,w,cin]; y: [n,2h,2w,cout] written with stride y_ld (the upper half of a concat buffer).
 * cin, cout multiples of 64; cout = 32 is accepted on 8x16-tileable shapes (UNet3D's 30-channel level stored with 32
 * lanes), where the two backward entry points need the gradient dense (y_ld = 32). */
typedef struct {
  int n, h, w;  /* INPUT spatial size */
  int cin, cout;
  int x_ld, y_ld;
  int relu;     /* slim default activation_fn=relu */
} bsl_convT2d_desc;

int bsl_convT2d_fwd(bsl_ctx* ctx, const bsl_convT2d_desc* d, const void* x_bf16,
                    const void* w_kkoi_bf16, const float* bias_f32, void* y_bf16, void* stream);
/* cout = 32 written into a pixel-pair packed tensor (UNet3D's full-resolution level, unet3d_engine.py): output voxel
 * (2y + a, 2x + b), lane co -> y[((n * 2h + 2y + a) * w + x) * y_ld + b * 32 + co]; y_ld = lanes per voxel pair. No bias
 * (slim.conv3d_transpose(..., biases_initializer=None), NetworksV2/UNet3D.py:160-163). */
int bsl_convT2d_fwd_pairs(bsl_ctx* ctx, const bsl_convT2d_desc* d, const void* x_bf16, const void* w_kkoi_bf16,
                          void* y_bf16, void* stream);
/* dyr must already carry the ReLU mask (dy * (y > 0)); see bsl_relu_bwd. */
int bsl_convT2d_bwd_data(bsl_ctx* ctx, const bsl_convT2d_desc* d, const void* dyr_bf16,
                         const void* w_kkoi_bf16, void* dx_bf16, void* stream);
size_t bsl_convT2d_bwd_filter_workspace(bsl_ctx* ctx, const bsl_convT2d_desc* d);
int bsl_convT2d_bwd_filter(bsl_ctx* ctx, const bsl_convT2d_desc* d, const void* x_bf16,
                           const void* dyr_bf16, float* dw_kkoi_f32, float* dbias_f32, void* workspace,
                           size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ conv3d / conv3d_transpose (UNet3D)
 * Replaces Conv3D / Conv3DBackpropInputV2 / Conv3DBackpropFilterV2 behind slim.conv3d(x, c, kernel, stride) and
 * slim.conv3d_transpose(x, c, kernel == stride, biases_initializer=None) -- NetworksV2/UNet3D.py:31-91,151-168.
 * Tensors are NDHWC bf16; filters DHWIO ([kd,kh,kw,Cin,Cout]) and [kd,kh,kw,Cout,Cin] for the transposed conv.
 * SAME padding as TF: out = ceil(in / stride), pad_before = max((out-1)*stride + k - in, 0) / 2.
 * Kernel extents 1 or 3, strides 1 or 2 per axis. (1,3,3)/stride-1 layers can equally be run as bsl_conv2d_* over
 * n*d images. cin and cout must be multiples of 64: the engine stores UNet3D's 30/60/120/240 channels zero-padded. */
typedef struct {
  int n, d, h, w; /* INPUT spatial size */
  int cin, cout;
  int kd, kh, kw;
  int sd, sh, sw;
  int x_ld, y_ld;
} bsl_conv3d_desc;

int bsl_conv3d_fprop(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x_bf16, const void* w_dhwio_bf16,
                     void* y_bf16, void* stream);
/* fprop + instance statistics: sums is fp64 [n][2][cout] (sum, sum of squares of the bf16 outputs per volume and
 * channel), what slim.instance_norm's moments need (NetworksV2/UNet3D.py:151-158). */
int bsl_conv3d_fprop_group_stats(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x_bf16, const void* w_dhwio_bf16,
                                 void* y_bf16, double* sums, void* stream);
/* fprop + batch statistics: sums is fp64 [2][cout] (sum, sum of squares of the bf16 outputs over all n*d*h*w output
 * voxels), the moments of slim.batch_norm after slim.conv3d (NetworksV2/UNet3D.py:151-158 with --normalizer batch_norm).
 * The 3-D counterpart of bsl_conv2d_fprop_stats; the bf16 outputs are bit-identical to bsl_conv3d_fprop's. */
int bsl_conv3d_fprop_stats(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x_bf16, const void* w_dhwio_bf16,
                           void* y_bf16, double* sums, void* stream);
int bsl_conv3d_dgrad(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* dy_bf16, const void* w_dhwio_bf16,
                     void* dx_bf16, void* stream);
size_t bsl_conv3d_wgrad_workspace(bsl_ctx* ctx, const bsl_conv3d_desc* d);
int bsl_conv3d_wgrad(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x_bf16, const void* dy_bf16,
                     float* dw_dhwio_f32, void* workspace, size_t workspace_bytes, void* stream);

typedef struct {
  int n, d, h, w; /* INPUT spatial size; output is [n, sd*d, 2h, 2w, cout] */
  int cin, cout;
  int sd;         /* kernel == stride == (sd, 2, 2), sd in {1, 2} */
  int x_ld, y_ld;
  int relu;
} bsl_convT3d_desc;

int bsl_convT3d_fwd(bsl_ctx* ctx, const bsl_convT3d_desc* d, const void* x_bf16, const void* w_bf16,
                    const float* bias_f32 /*nullable: UNet3D has none*/, void* y_bf16, void* stream);
int bsl_convT3d_bwd_data(bsl_ctx* ctx, const bsl_convT3d_desc* d, const void* dyr_bf16, const void* w_bf16,
                         void* dx_bf16, void* stream);
size_t bsl_convT3d_bwd_filter_workspace(bsl_ctx* ctx, const bsl_convT3d_desc* d);
int bsl_convT3d_bwd_filter(bsl_ctx* ctx, const bsl_convT3d_desc* d, const void* x_bf16, const void* dyr_bf16,
                           float* dw_f32, float* dbias_f32 /*nullable*/, void* workspace, size_t workspace_bytes,
                           void* stream);
/* out = a + b (bf16, channel-strided views): AddN of the skip gradient and the strided-conv gradient in UNet3D. */
int bsl_add_bf16(bsl_ctx* ctx, long long pixels, int c, const void* a_bf16, int a_ld, const void* b_bf16, int b_ld,
                 void* out_bf16, int out_ld, void* stream);

/* ------------------------------------------------------------------ stem + logits convolutions
 * CUDA-core kernels for the two HBM-bound layers (0.26 % of the FLOPs).
 * Stem:   slim.conv2d(images, 64, 3) on the fp32 input images -- NetworksV2/UNet.py:79 (first call);
 *         x fp32 [n,h,w,cin], w fp32 HWIO, y bf16 (pre-norm), dw fp32. No dgrad (inputs have none).
 * Logits: slim.conv2d(x, num_classes, 1, activation_fn=None) + bias -- NetworksV2/UNet.py:100;
 *         x bf16, w fp32 [cin][classes], logits / dlogits fp32 [n,h,w,classes] dense. */
/* col[n,h,w,64] (bf16) = im2col of the fp32 images: column t*cin+ci holds tap t, channel ci; columns
 * >= kh*kw*cin are zero. The stem then runs as bsl_conv2d_fprop / bsl_conv2d_wgrad with k = 1,
 * cin = 64 on the tensor cores (filter rows >= kh*kw*cin are zero padding). */
int bsl_stem_im2col(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* x_f32, void* col_bf16, void* stream);
/* Same with a row pitch of col_ld = 32 or 64 columns (>= kh*kw*cin). A 32-column matrix is handed to
 * bsl_conv2d_fprop / bsl_conv2d_wgrad as cin = 64, x_ld = 32: the TMA box is wider than the tensor and its upper
 * half is zero-filled on chip, so the K = 64 GEMM reads half the bytes (see x_ld in bsl_conv2d_desc). */
int bsl_stem_im2col_ld(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* x_f32, void* col_bf16, int col_ld,
                       void* stream);
int bsl_conv2d_stem_fprop(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* x_f32, const float* w_hwio_f32,
                          void* y_bf16, void* stream);
int bsl_conv2d_stem_wgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* x_f32, const void* dy_bf16,
                          float* dw_hwio_f32, void* stream);
int bsl_conv2d_head_fprop(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x_bf16, const float* w_f32,
                          const float* bias_f32, float* logits_f32, void* stream);
int bsl_conv2d_head_dgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const float* dlogits_f32, const float* w_f32,
                          void* dx_bf16, void* stream);
int bsl_conv2d_head_wgrad(bsl_ctx* ctx, const bsl_conv2d_desc* d, const void* x_bf16, const float* dlogits_f32,
                          float* dw_f32, float* dbias_f32, void* stream);

/* ------------------------------------------------------------------ normalisation (+ReLU, +pool)
 * slim.batch_norm (scale=True, runtime is_training, eps 1e-3, decay .999) and slim.instance_norm
 * (eps 1e-6) as selected by BaseNet._get_normalization -- NetworksV2/base.py:153-169; the ReLU is
 * slim.conv2d's default activation_fn and the 2x2/s2 max-pool is NetworksV2/UNet.py:81.
 * Pipeline per layer: stats -> finalize -> apply[_pool]; backward: bwd_reduce -> bwd_finalize ->
 * bwd_apply. `sums` are fp64 [groups][2][c] with groups = 1 (batch) or n (instance); mean / rstd /
 * scale / shift / c1 / c2 are fp32 [groups][c]. is_training is a RUNTIME argument (base.py:77). */
typedef struct {
  int mode;          /* 0 = batch_norm, 1 = instance_norm */
  int n, hw, c;      /* hw = product of the spatial dims (2-D or 3-D) */
  int x_ld, y_ld;    /* channel strides of the pre-norm tensor and of the activation output */
  float eps;
  float decay;       /* moving-average decay (batch_norm) */
  int relu;          /* fuse ReLU after the affine transform */
  int center, scale; /* beta / gamma present */
} bsl_norm_desc;

int bsl_norm_stats(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x_bf16, double* sums, void* stream);
int bsl_norm_finalize(bsl_ctx* ctx, const bsl_norm_desc* d, int is_training, const double* sums,
                      const float* gamma, const float* beta, float* moving_mean, float* moving_var,
                      float* mean, float* rstd, float* scale, float* shift, void* stream);
int bsl_norm_apply(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x_bf16, const float* scale,
                   const float* shift, void* y_bf16, void* stream);
int bsl_norm_apply_pool(bsl_ctx* ctx, const bsl_norm_desc* d, int h, int w, const void* x_bf16,
                        const float* scale, const float* shift, void* y_bf16, void* pooled_bf16,
                        int pooled_ld, void* stream);
/* dy is the gradient w.r.t. the (post-ReLU) activation, with channel stride dy_ld. */
int bsl_norm_bwd_reduce(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x_bf16, const void* dy_bf16, int dy_ld,
                        const float* mean, const float* rstd, const float* scale, const float* shift,
                        double* sums, void* stream);
int bsl_norm_bwd_finalize(bsl_ctx* ctx, const bsl_norm_desc* d, const double* sums, float* c1, float* c2,
                          float* dgamma, float* dbeta, void* stream);
int bsl_norm_bwd_apply(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x_bf16, const void* dy_bf16, int dy_ld,
                       const float* mean, const float* rstd, const float* scale, const float* shift,
                       const float* c1, const float* c2, void* dx_bf16, int dx_ld, void* stream);
/* Backward of the LAST normalised layer when only the 1x1 logits conv reads its activation (NetworksV2/UNet.py:94,100):
 * the gradient w.r.t. the activation, da[p][ch] = bf16(sum_k dlogits[p][k] * w_head[ch][k]), is recomputed per pixel
 * inside the two passes instead of being written by bsl_conv2d_head_dgrad and read back twice (12 instead of 128
 * bytes per pixel and pass). Bit-identical to head_dgrad -> norm_bwd_reduce -> norm_bwd_apply. classes in 2..4,
 * c <= 256 (bsl_norm_bwd_head_ok). */
int bsl_norm_bwd_head_ok(bsl_ctx* ctx, const bsl_norm_desc* d, int classes);
int bsl_norm_bwd_reduce_head(bsl_ctx* ctx, const bsl_norm_desc* d, const void* y_bf16, const float* dlogits,
                             const float* w_head /*[c][classes]*/, int classes, const float* mean, const float* rstd,
                             const float* scale, const float* shift, double* sums, void* stream);
int bsl_norm_bwd_apply_head(bsl_ctx* ctx, const bsl_norm_desc* d, const void* y_bf16, const float* dlogits,
                            const float* w_head, int classes, const float* mean, const float* rstd, const float* scale,
                            const float* shift, const float* c1, const float* c2, void* dx_bf16, int dx_ld,
                            void* stream);
/* ---- GUNet guide modulation of an instance-norm layer (NetworksV2/GUNet.py:162-217, modulated_conv_block):
 *   conv -> norm(center, scale per YAML) -> * gamma_mod[n, c] -> + (sp_guide[n, p, :] . w[:, c] + b[c]) -> ReLU
 * gamma_mod is this layer's slice of the context MLP output (conditional_normalization, GUNet.py:119-133); the
 * additive map is the 1x1 guide convolution of _spatial_subnets (GUNet.py:136-159), evaluated on the fly from the
 * 1- or 2-channel guide at this layer's resolution and never materialised. bsl_norm_modulate folds gamma_mod and the
 * guide-conv bias into the per-(sample, channel) scale / shift that bsl_norm_finalize produced; the *_mod passes are
 * the plain passes plus the guide term (guide == NULL or guide->map == NULL: identical to the plain pass). */
typedef struct {
  const float* map; /* fp32 [n][hw][channels]; NULL = no spatial guide */
  int channels;     /* 1 or 2 (--guide_channel) */
  const float* w;   /* this layer's columns of the guide conv filter: w[g * w_ld + c] */
  int w_ld;
} bsl_guide;

int bsl_norm_modulate(bsl_ctx* ctx, const bsl_norm_desc* d, const float* gamma_mod /*[n][gm_ld], nullable*/, int gm_ld,
                      const float* sp_bias /*[c], nullable*/, float* scale, float* shift, void* stream);
int bsl_norm_apply_mod(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x_bf16, const float* scale,
                       const float* shift, const bsl_guide* guide, void* y_bf16, void* stream);
int bsl_norm_apply_pool_mod(bsl_ctx* ctx, const bsl_norm_desc* d, int h, int w, const void* x_bf16,
                            const float* scale, const float* shift, const bsl_guide* guide, void* y_bf16,
                            void* pooled_bf16, int pooled_ld, void* stream);
/* bsl_norm_apply (no guide) that also produces the logits of the 1x1 class convolution that follows the last
 * normalised layer (NetworksV2/UNet.py:100): logits[p][k] = sum_c act[p][c] * w_head[c][k] + b_head[k], fp32
 * [n,h,w,classes], bit-identical to bsl_conv2d_head_fprop on the stored activation. c in {8,16,..,256}. */
int bsl_norm_apply_head(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x_bf16, const float* scale,
                        const float* shift, void* y_bf16, const float* w_head_f32, const float* b_head_f32,
                        int classes, float* logits_f32, void* stream);
/* sums: fp64 [n][2 + guide channels][c] = sum dz, sum dz * xhat, sum dz * guide_g. */
int bsl_norm_bwd_reduce_mod(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x_bf16, const void* dy_bf16, int dy_ld,
                            const float* mean, const float* rstd, const float* scale, const float* shift,
                            const bsl_guide* guide, double* sums, void* stream);
/* c1, c2 as bsl_norm_bwd_finalize; dgamma / dbeta (nullable) of the norm's own affine; dgamma_mod [n][gm_ld] is the
 * gradient w.r.t. the context MLP output slice; dw_guide [g * dw_ld + c] and dbias_guide [c] the guide conv's. */
int bsl_norm_bwd_finalize_mod(bsl_ctx* ctx, const bsl_norm_desc* d, const double* sums, int guide_channels,
                              const float* gamma_mod, int gm_ld, const float* gamma, const float* beta, float* c1,
                              float* c2, float* dgamma, float* dbeta, float* dgamma_mod, float* dw_guide, int dw_ld,
                              float* dbias_guide, void* stream);
/* ---- GUNet / UNetInter with --normalizer batch_norm (GUNet.py:301,321-325: decay 0.99 on the modulated blocks): the
 * statistics are per channel over the whole batch while the modulation is per sample. bsl_norm_finalize (mode 0) leaves
 * the batch statistics in the first c entries; bsl_norm_modulate_bn expands them in place to per-(sample, channel)
 * mean / rstd / scale / shift with gamma_mod and the guide bias folded in, so that the apply and backward-reduce passes
 * run on the per-sample (mode 1) view of the layer. bsl_norm_bwd_finalize_bnmod combines the per-sample sums with their
 * scales (FusedBatchNormGrad means over all samples) into c1r = rstd*C1, c2r = rstd*C2, which bsl_norm_bwd_apply_bnmod
 * consumes: dy = scale[n]*dz - c1r - xhat*c2r. The descriptor passed to all three is the mode-1 view. */
int bsl_norm_modulate_bn(bsl_ctx* ctx, const bsl_norm_desc* d, const float* gamma_mod /*nullable*/, int gm_ld,
                         const float* sp_bias /*nullable*/, float* mean, float* rstd, float* scale, float* shift,
                         void* stream);
int bsl_norm_bwd_finalize_bnmod(bsl_ctx* ctx, const bsl_norm_desc* d, const double* sums, int guide_channels,
                                const float* gamma_mod, int gm_ld, const float* gamma, const float* beta,
                                const float* rstd, float* c1r, float* c2r, float* dgamma, float* dbeta,
                                float* dgamma_mod, float* dw_guide, int dw_ld, float* dbias_guide, void* stream);
int bsl_norm_bwd_apply_bnmod(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x_bf16, const void* dy_bf16, int dy_ld,
                             const float* mean, const float* rstd, const float* scale, const float* shift,
                             const float* c1r, const float* c2r, const bsl_guide* guide, void* dx_bf16, int dx_ld,
                             void* stream);
/* ---- GUNet `after_affine` (NetworksV2/GUNet.py:213-214, Backbone/slim_nets.py:152-212 channel_wise_affine): a per-channel
 * gamma_a * u + beta_a between the modulation and the ReLU of every encoder block. With u = y*scale + shift + guide.w
 * the affine folds into the same three quantities, so no pass changes: bsl_norm_affine_fold rewrites scale *= gamma_a,
 * shift = shift*gamma_a + beta_a in place (keeping the un-folded values in scale_pre / shift_pre for the backward
 * finaliser) and writes the gamma_a-scaled guide filter w_eff[g * c + ch] the *_mod passes then read.
 * Representation: scale / shift / mean / rstd are [groups][c] in the view the descriptor describes, groups = n in
 * mode 1 and 1 in mode 0. An instance-norm layer and a modulated batch-norm layer (after bsl_norm_modulate_bn) pass the
 * per-sample mode-1 view; an un-modulated batch-norm layer passes its mode-0 descriptor and folds its per-channel
 * scale / shift (no guide there). scale_pre / shift_pre have the same [groups][c] shape. */
int bsl_norm_affine_fold(bsl_ctx* ctx, const bsl_norm_desc* d, const float* gamma_a, const float* beta_a, float* scale,
                         float* shift, float* scale_pre, float* shift_pre, const float* w_guide /*nullable*/, int w_ld,
                         int guide_channels, float* w_eff /*[guide_channels][c], nullable*/, void* stream);
/* bsl_norm_bwd_finalize_mod for a layer with the folded affine. `sums` were reduced with the FOLDED scale / shift /
 * w_eff (they are sums of dz, the gradient after the affine, one row per group of the descriptor's view); scale_pre /
 * shift_pre / w_guide are the un-folded ones. Emits dgamma_a[c] = sum_groups (scale_pre/rstd * S1 +
 * (shift_pre + mean*scale_pre) * S0 + sum_g w_g * T_g) (= sum dz * u, u the pre-affine value) and dbeta_a[c] = sum S0,
 * and every other gradient with the sums scaled by gamma_a (du = gamma_a * dz). `jacobian` selects c1 / c2:
 *   BSL_NORM_JAC_GROUP  c1 = S0/m, c2 = S1/m per group, m the values per group, for bsl_norm_bwd_apply[_mod]: instance
 *                       norm (mode 1) and an un-modulated batch-norm layer (mode 0, one group);
 *   BSL_NORM_JAC_BATCH  a modulated batch-norm layer on its per-sample view (mode 1): c1r / c2r of
 *                       bsl_norm_bwd_finalize_bnmod with gamma_a in the chain, for bsl_norm_bwd_apply_bnmod;
 *   BSL_NORM_JAC_NONE   identity normaliser (mean 0, rstd 1: the modulation stage of a GUNet --dropout layer, gamma /
 *                       beta NULL): c1 = c2 = 0.
 * bsl_norm_bwd_finalize_affine is the BSL_NORM_JAC_GROUP call. */
#define BSL_NORM_JAC_GROUP 0
#define BSL_NORM_JAC_BATCH 1
#define BSL_NORM_JAC_NONE 2
int bsl_norm_bwd_finalize_affine_jac(bsl_ctx* ctx, const bsl_norm_desc* d, int jacobian, const double* sums,
                                     int guide_channels, const float* gamma_mod, int gm_ld, const float* gamma,
                                     const float* beta, const float* gamma_a, const float* mean, const float* rstd,
                                     const float* scale_pre, const float* shift_pre, const float* w_guide, int w_ld,
                                     float* c1, float* c2, float* dgamma, float* dbeta, float* dgamma_mod,
                                     float* dw_guide, int dw_ld, float* dbias_guide, float* dgamma_a, float* dbeta_a,
                                     void* stream);
int bsl_norm_bwd_finalize_affine(bsl_ctx* ctx, const bsl_norm_desc* d, const double* sums, int guide_channels,
                                 const float* gamma_mod, int gm_ld, const float* gamma, const float* beta,
                                 const float* gamma_a, const float* mean, const float* rstd, const float* scale_pre,
                                 const float* shift_pre, const float* w_guide, int w_ld, float* c1, float* c2,
                                 float* dgamma, float* dbeta, float* dgamma_mod, float* dw_guide, int dw_ld,
                                 float* dbias_guide, float* dgamma_a, float* dbeta_a, void* stream);
int bsl_norm_bwd_apply_mod(bsl_ctx* ctx, const bsl_norm_desc* d, const void* x_bf16, const void* dy_bf16, int dy_ld,
                           const float* mean, const float* rstd, const float* scale, const float* shift,
                           const float* c1, const float* c2, const bsl_guide* guide, void* dx_bf16, int dx_ld,
                           void* stream);

/* ---- GUNet context MLP and guide pyramid (fp32, tiny): slim_nets.fc = fully_connected (+ ReLU) (+ dropout) --
 * NetworksV2/Backbone/slim_nets.py:34-57 called from GUNet._context_subnets (GUNet.py:31-59); slim.avg_pool2d(gs, 2)
 * -- GUNet.py:155-156. Dropout follows tf.nn.dropout (x / keep_prob * floor(keep_prob + u)) with u drawn from
 * Philox4x32-10 keyed by (seed, offset): element i uses counter i / 4, lane i % 4, so the oracle reproduces the mask
 * bit for bit. */
typedef struct {
  float keep_prob;
  unsigned long long seed, offset;
} bsl_dropout_desc;
typedef struct {
  int n, cin, cout;
  int relu;        /* slim.fully_connected default activation_fn */
  int use_dropout; /* only when is_training and side_dropout > 0 */
  bsl_dropout_desc dropout;
} bsl_fc_desc;

int bsl_fc_fwd(bsl_ctx* ctx, const bsl_fc_desc* d, const float* x, const float* w /*[cin][cout]*/, const float* bias,
               float* y, void* stream);
size_t bsl_fc_bwd_workspace(bsl_ctx* ctx, const bsl_fc_desc* d);
/* y is the forward OUTPUT (post ReLU / dropout); dx nullable (first layer). */
int bsl_fc_bwd(bsl_ctx* ctx, const bsl_fc_desc* d, const float* x, const float* w, const float* y, const float* dy,
               float* dx, float* dw, float* dbias, void* workspace, size_t workspace_bytes, void* stream);
/* out[i] = 1 / keep_prob or 0: the dropout multipliers themselves (tests, and backbone --dropout). */
int bsl_dropout_mask(bsl_ctx* ctx, const bsl_dropout_desc* d, size_t n, float* out, void* stream);
/* slim.dropout on a bf16 NHWC tensor (GUNet backbone --dropout, NetworksV2/GUNet.py:189-190) and, with the same
 * descriptor, its gradient: out[p][ch] = bf16(x[p][ch] * multiplier(p * c + ch)); in place when out == x. */
int bsl_dropout_bf16(bsl_ctx* ctx, const bsl_dropout_desc* d, long long pixels, int c, const void* x_bf16, int x_ld,
                     void* out_bf16, int out_ld, void* stream);
int bsl_avgpool2x2_f32(bsl_ctx* ctx, int n, int h, int w, int c, const float* x, float* y, void* stream);
/* --img_grad (NetworksV2/GUNet.py:333-337, UNet.py:69-71): tf.concat((images, dy, dx), -1) with tf.image.image_gradients
 * (forward differences, last row / column zero) as bf16 lanes [0, 3c) of y_bf16 rows with stride y_ld. */
int bsl_image_gradients_pack(bsl_ctx* ctx, int n, int h, int w, int c, const float* x, void* y_bf16, int y_ld,
                             void* stream);
/* UNetInter --mid_cat (NetworksV2/UNetInter.py:124-125, slim.max_pool2d(concat(net, sp_guide), 2)): the guide's share of
 * the pooled tensor, y_bf16[pixel * y_ld + ch] = bf16(max of the 2x2 window of x[n,h,w,c]), ch < c. */
int bsl_maxpool2x2_f32_bf16(bsl_ctx* ctx, int n, int h, int w, int c, const float* x, void* y_bf16, int y_ld,
                            void* stream);

/* slim.max_pool2d(x, 2) of a bf16 activation: y[n,i,j,ch] = max of x[n,2i..2i+1,2j..2j+1,ch]; h, w are the INPUT size
 * (even), x and y are read / written with channel strides x_ld, y_ld (c, x_ld, y_ld multiples of 8). Exact (no rounding).
 * The backward pass is bsl_maxpool2x2_bwd_add. */
int bsl_maxpool2x2_bf16(bsl_ctx* ctx, int n, int h, int w, int c, const void* x_bf16, int x_ld, void* y_bf16, int y_ld,
                        void* stream);
/* MaxPoolGrad (first maximum in scan order wins ties) fused with the skip-connection add:
 * dact = dskip (nullable) + unpool(dpool). */
int bsl_maxpool2x2_bwd_add(bsl_ctx* ctx, int n, int h, int w, int c, const void* act_bf16, int act_ld,
                           const void* dpool_bf16, int dpool_ld, const void* dskip_bf16, int dskip_ld,
                           void* dact_bf16, int dact_ld, void* stream);
/* ReluGrad: out = dy * (y > 0). */
int bsl_relu_bwd(bsl_ctx* ctx, long long pixels, int c, const void* y_bf16, int y_ld, const void* dy_bf16,
                 int dy_ld, void* out_bf16, int out_ld, void* stream);
/* ReluGrad + BiasAddGrad of slim.conv2d_transpose (UNet.py:91) in one pass: out = dy * (y > 0) and
 * dbias[c] = sum over pixels of out (the same fixed-order reduction bsl_convT2d_bwd_filter runs when it is given
 * dbias; pass dbias = NULL there afterwards). */
int bsl_relu_bwd_bias(bsl_ctx* ctx, long long pixels, int c, const void* y_bf16, int y_ld, const void* dy_bf16,
                      int dy_ld, void* out_bf16, int out_ld, float* dbias_f32, void* stream);

/* ------------------------------------------------------------------ losses, masks, Dice counts
 * loss_metrics._compute_weights / weighted_sparse_softmax_cross_entropy / sparse_dice_loss
 * (/root/reference/loss_metrics.py:115-226), slim.softmax + (p > 0.5) uint8 masks
 * (NetworksV2/UNet.py:107-117) and the integer sums behind metric_dice/voe/vd (loss_metrics.py:261-339).
 * logits / dlogits / prob are dense fp32 [n*hw][classes]; labels int32 [n*hw]. */
typedef struct {
  int n, hw, classes;      /* classes in 2..4 */
  int weight_type;         /* 0 none, 1 numerical, 2 proportion */
  float numeric_w[8];
  float proportion_decay;  /* <= 0: not applied */
  float loss_scale;        /* multiplies dlogits: 1/R under R-way data parallelism */
} bsl_loss_desc;

size_t bsl_loss_workspace(bsl_ctx* ctx, const bsl_loss_desc* d);
int bsl_label_counts(bsl_ctx* ctx, const bsl_loss_desc* d, const int* labels, int* counts /*[n][classes]*/,
                     void* stream);
int bsl_wxent_fwd_bwd(bsl_ctx* ctx, const bsl_loss_desc* d, const float* logits, const int* labels,
                      const int* counts, float* loss, float* dlogits /*nullable*/, void* workspace,
                      size_t workspace_bytes, void* stream);
int bsl_dice_fwd_bwd(bsl_ctx* ctx, const bsl_loss_desc* d, const float* logits, const int* labels, float* loss,
                     float* dlogits /*nullable*/, int accumulate, void* workspace, size_t workspace_bytes,
                     void* stream);
/* Any of prob [n*hw][classes], masks uint8 [classes-1][n*hw], argmax uint8 [n*hw] and
 * ilr uint32 [n][classes-1][3] = (intersection, left=pred, right=label) may be null. */
int bsl_softmax_threshold(bsl_ctx* ctx, const bsl_loss_desc* d, const float* logits, const int* labels,
                          float* prob, uint8_t* masks, uint8_t* argmax, unsigned int* ilr, void* stream);

/* ------------------------------------------------------------------ forward-only consumers (inference / evaluation)
 * Test-time mirroring as run_TTA does it on the host (/root/reference/entry/main_eval_3d.py:246-287,
 * entry/infer_2d.py:60-78): probs += np.flip(prob of the flipped input); avg = probs / count; np.argmax -> uint8;
 * and ConfusionMatrix.compute (/root/reference/loss_metrics.py:542-556) as exact integer counts.
 * Tensors are dense fp32 [n][d][h][w][c] (d = 1 for 2-D); `axes` is a bit mask: 1 = W, 2 = H, 4 = D. */
int bsl_flip_f32(bsl_ctx* ctx, long long n, int d, int h, int w, int c, int axes, int accumulate, const float* src,
                 float* dst, void* stream); /* dst = (accumulate ? dst : 0) + flip(src); src != dst */
int bsl_tta_finalize(bsl_ctx* ctx, long long pixels, int classes, int count, const float* acc,
                     float* avg_prob /*nullable*/, uint8_t* pred, void* stream);
/* counts4 += {tp, fp, tn, fn}; test = (test_u8 == test_value), or (test_u8 != 0) when test_value < 0;
 * reference = (labels == ref_value). The caller zeroes counts4 (accumulation over batches is the point). */
int bsl_confusion_counts(bsl_ctx* ctx, long long n, const uint8_t* test_u8, int test_value, const int* labels,
                         int ref_value, unsigned long long* counts4, void* stream);

/* ------------------------------------------------------------------ fused optimizer step
 * tf.train.AdamOptimizer(lr, beta1, beta2, epsilon) / MomentumOptimizer(lr, momentum, use_nesterov) /
 * tf.contrib.opt.AdamWOptimizer(weight_decay, lr, ...) -- /root/reference/core/solver.py:86-97,204-219,
 * with slim.l2_regularizer folded in (grad += l2_rate * w) -- NetworksV2/base.py:128-135.
 * Works on flat arenas; also emits the bf16 shadow weights and (optionally) sum(w^2) of the
 * pre-update weights for the reported regularisation loss. */
typedef struct {
  float lr, beta1, beta2, eps;
  float l2_rate;     /* 0 for parameters without a regulariser (norm gamma / beta) */
  float grad_scale;  /* applied to g before use */
  int step;          /* t >= 1 */
  float decoupled_decay; /* AdamW (DecoupledWeightDecayExtension): w <- w - decoupled_decay * w, THEN the Adam
                          * update on the decayed value with the gradient taken at the old w; 0 = plain Adam */
} bsl_adam_desc;

int bsl_adam_step(bsl_ctx* ctx, const bsl_adam_desc* d, float* w, const float* g, float* m, float* v,
                  void* w_bf16 /*nullable*/, size_t n, double* sumsq_out /*nullable*/, void* stream);
/* ApplyMomentum: acc = momentum * acc + g; w -= lr * acc, or with use_nesterov: w -= lr * g + lr * momentum * acc */
int bsl_momentum_step(bsl_ctx* ctx, float lr, float momentum, int use_nesterov, float l2_rate, float grad_scale,
                      float* w, const float* g, float* acc, void* w_bf16, size_t n, double* sumsq_out, void* stream);

/* ------------------------------------------------------------------ data-parallel gradient exchange
 * Replaces MirroredStrategy's NCCL all-reduce -- /root/reference/utils/distribution_utils.py:85-98.
 * One process per GPU; rank 0 creates the 128-byte id, the host distributes it (any side channel). */
int bsl_comm_unique_id(bsl_ctx* ctx, void* id128);
int bsl_comm_init(bsl_ctx* ctx, const void* id128, int rank, int world);
int bsl_allreduce_sum_f32(bsl_ctx* ctx, float* buf, size_t n, void* stream);
int bsl_comm_destroy(bsl_ctx* ctx);

/* ------------------------------------------------------------------ device-side input stage (SURVEY 8f rank 4)
 * One pass over the decoded PNG slices of a batch that does what the reference's tf.data map function does per
 * sample on the host: crop_to_bounding_box -> resize_bilinear(align_corners=True) -> [H,W,C] -> window clip and
 * normalise -> uniform noise (not in empty slices) -> random left/right and up/down flips of image, label and guide
 * (DataLoader/Liver/input_pipeline.py:243-284, utils/image_ops.py:209-238,245-320); labels go through
 * resize_nearest_neighbor(align_corners=True) and trunc(seg / lab_scale); the optional sp_guide is
 * create_spatial_guide_2d on the crop grid, resized, / 2 + 0.5 (input_pipeline_g.py:380-391, image_ops.py:396-434).
 * The random DECISIONS (bbox, flips) are inputs, drawn by the caller as the reference's generator does; the noise
 * stream is Philox4x32-10 keyed by (seed, offset), element ((i*H + y)*W + x)*C + c of the UN-flipped image.
 * Outputs are the engines' input buffers: images fp32 [n,H,W,C], labels int32 [n,H,W], sp_guide fp32 [n,H,W,1]. */
typedef struct {
  int n, channels;   /* samples, adjacent slices per sample (--im_channel) */
  int src_h, src_w;  /* decoded slice size (512 x 512) */
  int out_h, out_w;  /* --im_height, --im_width */
  int max_centers;   /* padded centre count per sample (sp_guide only) */
  float noise_scale; /* --noise_scale; 0 = no noise */
  float min_std;     /* lower bound of the guide stddevs (kwargs min_std, default 1) */
  unsigned long long seed, offset;
} bsl_input_desc;

typedef struct {          /* device pointers, one row per sample */
  const int* bbox;        /* [n][4] offset_row, offset_col, height, width (crop_to_bounding_box order) */
  const float* clip;      /* [n][2] window min, max */
  const int* lab_scale;   /* [n] */
  const unsigned char* present; /* [n][channels] 0 for a missing neighbour slice (nullable: all present) */
  const int* flips;       /* [n] bit 0: left/right, bit 1: up/down (nullable) */
  const float* centers;   /* [n][max_centers][2] (y, x) on the crop grid */
  const float* stddevs;   /* [n][max_centers][2] */
  const int* n_centers;   /* [n]; 0 = constant 0.5 guide */
} bsl_input_params;

int bsl_input_stage(bsl_ctx* ctx, const bsl_input_desc* d, const bsl_input_params* p, const void* slices_u16,
                    const void* seg_u8 /*nullable*/, float* images, int* labels /*nullable*/,
                    float* sp_guide /*nullable*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BSL_B200_H_ */
