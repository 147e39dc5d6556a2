// Library-private context shared by the translation units of libbsl_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <mutex>
#include <string>
#include <utility>
#include <unordered_map>
#include <vector>
#include "../../include/bsl_b200.h"
#include "ptx.cuh"

typedef CUresult (*bsl_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                        const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                        const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct bsl_ctx {
  int device = 0;
  int sm_count = 148;
  std::string err;
  std::mutex mu;
  bsl::DeviceStatus* d_status = nullptr;
  bsl_encode_tiled_fn encode_tiled = nullptr;
  std::unordered_map<std::string, CUtensorMap> tmaps;  // keyed by (ptr, dims, strides, box)
  void* nccl_lib = nullptr;                            // dlopen handle (comm.cu)
  void* nccl_comm = nullptr;
  int rank = 0, world = 1;
  unsigned long long launches = 0;  // kernels enqueued through this context (bench.py gpu_launches)
  // Scratch arenas of the two-level reductions, one per stream of THIS context (reduce.cuh bsl_scratch): released by
  // bsl_stream_destroy / bsl_destroy, never shared between contexts or devices.
  struct Scratch {
    float* ptr = nullptr;
    size_t bytes = 0;
  };
  std::mutex scratch_mu;
  std::unordered_map<cudaStream_t, Scratch> scratch;
  std::unordered_map<cudaStream_t, Scratch> scratch_w;   // re-laid-out filters of the CTA-pair kernels (conv.cu)
};

// Frees the scratch arena attached to `stream` (all of them when stream_or_all is true).
void bsl_scratch_release(bsl_ctx* ctx, cudaStream_t stream, bool all);

int bsl_fail(bsl_ctx* ctx, int code, const char* fmt, ...);
int bsl_check_cuda(bsl_ctx* ctx, cudaError_t e, const char* what);

#define BSL_CUDA(ctx, expr)                                        \
  do {                                                             \
    cudaError_t _e = (expr);                                       \
    if (_e != cudaSuccess) return bsl_check_cuda(ctx, _e, #expr);  \
  } while (0)

#define BSL_LAUNCH_CHECK(ctx, what)                                \
  do {                                                             \
    cudaError_t _e = cudaGetLastError();                           \
    if (_e != cudaSuccess) return bsl_check_cuda(ctx, _e, what);   \
    ++(ctx)->launches;                                             \
  } while (0)

// Kernel launch with the programmatic-stream-serialization attribute (on by default, BSL_PDL=0 turns it off): the grid may be
// scheduled while the previous kernel of the stream drains. Every kernel launched through here calls
// bsl::pdl_wait() before its first access to global data (ptx.cuh).
bool bsl_pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t bsl_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = bsl_pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}

// Same for a kernel that runs as thread-block clusters of `cluster_x` CTAs along x (grid.x a multiple of it).
template <typename... KArgs, typename... Args>
inline cudaError_t bsl_launch_cluster(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                      int cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster_x;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = bsl_pdl_enabled() ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}

// Encodes (or fetches from the cache) a bf16 tensor map with 128-byte swizzle and zero OOB fill.
// dims/strides are innermost-first; strides[0] is implied (2 bytes) and ignored.
int bsl_get_tmap(bsl_ctx* ctx, const void* base, int rank, const uint64_t* dims,
                 const uint64_t* strides_bytes, const uint32_t* box, CUtensorMap* out);

// Same, with a traversal stride per dimension (TMA elementStrides): a box of box[i] elements then holds
// ceil(box[i] / elem_strides[i]) loaded elements, taken every elem_strides[i]-th from the start coordinate.
int bsl_get_tmap_es(bsl_ctx* ctx, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, const uint32_t* elem_strides, CUtensorMap* out);

// out[c] = sum over pixels of x[p*ld + c] (bf16 in, fp32 out), deterministic two-level reduction.
int bsl_channel_sum_bf16(bsl_ctx* ctx, const void* x, long long pixels, int c, int ld, float* out,
                         cudaStream_t stream);

// sums[group][2][c] (fp64) = per-channel sum and sum of squares of a bf16 NHWC tensor (norm.cu).
int bsl_stats_bf16(bsl_ctx* ctx, const void* x, long long pixels_per_group, int groups, int c, int ld, double* sums,
                   cudaStream_t stream);

// (3,3,3) / (1,3,3) stride-1 layers on the halo-tile kernels (conv.cu), used by conv3d.cu when the shape allows.
bool bsl_conv3d_halo_ok(const bsl_conv3d_desc* d);
bool bsl_conv3d_halo_dgrad_strided_ok(const bsl_conv3d_desc* d);
int bsl_conv3d_halo_dgrad_strided(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* dy, const void* w, void* dx,
                                  cudaStream_t s);
// sums (nullable): fp64 [n][2][cout] per (volume, channel) when per_volume, else [2][cout] over the whole batch.
int bsl_conv3d_halo_fprop(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x, const void* w, void* y, cudaStream_t s,
                          double* sums = nullptr, bool per_volume = true);
int bsl_conv3d_halo_dgrad(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* dy, const void* w, void* dx, cudaStream_t s);
bool bsl_conv3d_halo_wgrad_ok(const bsl_conv3d_desc* d);
size_t bsl_conv3d_halo_wgrad_ws(bsl_ctx* ctx, const bsl_conv3d_desc* d);
int bsl_conv3d_halo_wgrad(bsl_ctx* ctx, const bsl_conv3d_desc* d, const void* x, const void* dy, float* dw, void* workspace,
                          size_t workspace_bytes, cudaStream_t s);

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
