// Context, device memory, streams/events/graphs and TMA tensor-map encoding for libbsl_b200.so.
// This is the part of the boundary the TF wrapper would NOT use (TF owns memory and streams,
// SURVEY.md section 8b); the ctypes host in boxsegliver_b200/ uses it instead of PyTorch.
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include "internal.h"

// BSL_PDL=0 in the environment turns the launch attribute off for the whole process (read once), the way to isolate a
// fault from launch overlap; the attribute only changes scheduling, never results.
bool bsl_pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("BSL_PDL");
    return e ? atoi(e) != 0 : true;
  }();
  return on;
}

int bsl_fail(bsl_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) {
    std::lock_guard<std::mutex> g(ctx->mu);
    ctx->err = buf;
  }
  return code;
}

int bsl_check_cuda(bsl_ctx* ctx, cudaError_t e, const char* what) {
  return bsl_fail(ctx, BSL_ECUDA, "CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
}

extern "C" {

const char* bsl_version(void) { return "bsl_b200 0.1 (sm_100a)"; }

// CRC-32C (Castagnoli, reflected polynomial 0x82F63B78), slicing-by-8, host only: the checksum of the TF Saver V2
// bundle format (boxsegliver_b200/checkpoint.py). `crc` is the running value (0 to start); no context needed.
unsigned bsl_crc32c(unsigned crc, const void* data, size_t n) {
  static uint32_t T[8][256];
  static bool ready = [] {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c >> 1) ^ (0x82F63B78u & (0u - (c & 1u)));
      T[0][i] = c;
    }
    for (uint32_t i = 0; i < 256; ++i)
      for (int t = 1; t < 8; ++t) T[t][i] = (T[t - 1][i] >> 8) ^ T[0][T[t - 1][i] & 0xff];
    return true;
  }();
  (void)ready;
  const unsigned char* p = static_cast<const unsigned char*>(data);
  uint32_t c = ~crc;
  while (n >= 8) {
    uint32_t lo, hi;
    memcpy(&lo, p, 4);
    memcpy(&hi, p + 4, 4);
    lo ^= c;
    c = T[7][lo & 0xff] ^ T[6][(lo >> 8) & 0xff] ^ T[5][(lo >> 16) & 0xff] ^ T[4][lo >> 24] ^ T[3][hi & 0xff] ^
        T[2][(hi >> 8) & 0xff] ^ T[1][(hi >> 16) & 0xff] ^ T[0][hi >> 24];
    p += 8;
    n -= 8;
  }
  while (n--) c = (c >> 8) ^ T[0][(c ^ *p++) & 0xff];
  return ~c;
}

int bsl_init(int device, bsl_ctx** out) {
  if (!out) return BSL_EINVAL;
  *out = nullptr;
  bsl_ctx* ctx = new bsl_ctx();
  ctx->device = device;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) {
    fprintf(stderr, "bsl_init: cudaSetDevice(%d) failed: %s\n", device, cudaGetErrorString(e));
    delete ctx;
    return BSL_ECUDA;
  }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess || prop.major != 10) {
    fprintf(stderr, "bsl_init: device %d is not an sm_100 part (cc %d.%d); no fallback path exists\n",
            device, e == cudaSuccess ? prop.major : -1, e == cudaSuccess ? prop.minor : -1);
    delete ctx;
    return BSL_EUNSUPPORTED;
  }
  ctx->sm_count = prop.multiProcessorCount;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || !fn || qres != cudaDriverEntryPointSuccess) {
    fprintf(stderr, "bsl_init: cuTensorMapEncodeTiled not available\n");
    delete ctx;
    return BSL_ECUDA;
  }
  ctx->encode_tiled = reinterpret_cast<bsl_encode_tiled_fn>(fn);
  e = cudaMalloc(&ctx->d_status, sizeof(bsl::DeviceStatus));
  if (e == cudaSuccess) e = cudaMemset(ctx->d_status, 0, sizeof(bsl::DeviceStatus));
  if (e != cudaSuccess) {
    delete ctx;
    return BSL_ECUDA;
  }
  *out = ctx;
  return BSL_OK;
}

void bsl_destroy(bsl_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->d_status) cudaFree(ctx->d_status);
  bsl_scratch_release(ctx, nullptr, true);
  delete ctx;
}

const char* bsl_last_error(bsl_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int bsl_device_status(bsl_ctx* ctx, int* block, int* site) {
  if (!ctx) return BSL_EINVAL;
  bsl::DeviceStatus h;
  BSL_CUDA(ctx, cudaMemcpy(&h, ctx->d_status, sizeof(h), cudaMemcpyDeviceToHost));
  if (block) *block = h.block;
  if (site) *site = h.site;
  if (h.error) {
    BSL_CUDA(ctx, cudaMemset(ctx->d_status, 0, sizeof(h)));
    return bsl_fail(ctx, BSL_EDEVICE, "device pipeline watchdog fired: block %d site %d", h.block, h.site);
  }
  return BSL_OK;
}

int bsl_launch_count(bsl_ctx* ctx, unsigned long long* out) {
  if (!ctx || !out) return BSL_EINVAL;
  *out = ctx->launches;
  return BSL_OK;
}

int bsl_mem_info(bsl_ctx* ctx, size_t* free_bytes, size_t* total_bytes) {
  if (!ctx || !free_bytes || !total_bytes) return BSL_EINVAL;
  BSL_CUDA(ctx, cudaMemGetInfo(free_bytes, total_bytes));
  return BSL_OK;
}

int bsl_malloc(bsl_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return BSL_EINVAL;
  BSL_CUDA(ctx, cudaMalloc(out, bytes ? bytes : 16));
  return BSL_OK;
}
int bsl_free(bsl_ctx* ctx, void* ptr) {
  if (!ctx) return BSL_EINVAL;
  BSL_CUDA(ctx, cudaFree(ptr));
  return BSL_OK;
}
int bsl_memset(bsl_ctx* ctx, void* dst, int value, size_t bytes, void* stream) {
  BSL_CUDA(ctx, cudaMemsetAsync(dst, value, bytes, as_stream(stream)));
  return BSL_OK;
}
int bsl_memcpy_h2d(bsl_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream) {
  BSL_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, as_stream(stream)));
  return BSL_OK;
}
int bsl_memcpy_d2h(bsl_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream) {
  BSL_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, as_stream(stream)));
  return BSL_OK;
}
int bsl_memcpy_d2d(bsl_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream) {
  BSL_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, as_stream(stream)));
  return BSL_OK;
}
int bsl_host_alloc(bsl_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return BSL_EINVAL;
  BSL_CUDA(ctx, cudaMallocHost(out, bytes ? bytes : 16));
  return BSL_OK;
}
int bsl_host_free(bsl_ctx* ctx, void* ptr) {
  BSL_CUDA(ctx, cudaFreeHost(ptr));
  return BSL_OK;
}
int bsl_stream_create(bsl_ctx* ctx, void** out) {
  if (!ctx || !out) return BSL_EINVAL;
  cudaStream_t s;
  BSL_CUDA(ctx, cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  *out = s;
  return BSL_OK;
}
int bsl_stream_destroy(bsl_ctx* ctx, void* stream) {
  if (!ctx) return BSL_EINVAL;
  BSL_CUDA(ctx, cudaStreamSynchronize(as_stream(stream)));
  bsl_scratch_release(ctx, as_stream(stream), false);
  BSL_CUDA(ctx, cudaStreamDestroy(as_stream(stream)));
  return BSL_OK;
}
int bsl_stream_sync(bsl_ctx* ctx, void* stream) {
  BSL_CUDA(ctx, cudaStreamSynchronize(as_stream(stream)));
  return BSL_OK;
}
int bsl_event_create(bsl_ctx* ctx, void** out) {
  if (!ctx || !out) return BSL_EINVAL;
  cudaEvent_t e;
  BSL_CUDA(ctx, cudaEventCreate(&e));
  *out = e;
  return BSL_OK;
}
int bsl_event_destroy(bsl_ctx* ctx, void* ev) {
  BSL_CUDA(ctx, cudaEventDestroy(reinterpret_cast<cudaEvent_t>(ev)));
  return BSL_OK;
}
int bsl_event_record(bsl_ctx* ctx, void* ev, void* stream) {
  BSL_CUDA(ctx, cudaEventRecord(reinterpret_cast<cudaEvent_t>(ev), as_stream(stream)));
  return BSL_OK;
}
int bsl_event_sync(bsl_ctx* ctx, void* ev) {
  BSL_CUDA(ctx, cudaEventSynchronize(reinterpret_cast<cudaEvent_t>(ev)));
  return BSL_OK;
}
int bsl_stream_wait_event(bsl_ctx* ctx, void* stream, void* ev) {
  BSL_CUDA(ctx, cudaStreamWaitEvent(as_stream(stream), reinterpret_cast<cudaEvent_t>(ev), 0));
  return BSL_OK;
}
int bsl_event_elapsed_ms(bsl_ctx* ctx, void* start, void* stop, float* ms) {
  BSL_CUDA(ctx, cudaEventElapsedTime(ms, reinterpret_cast<cudaEvent_t>(start),
                                     reinterpret_cast<cudaEvent_t>(stop)));
  return BSL_OK;
}
int bsl_graph_begin(bsl_ctx* ctx, void* stream) {
  BSL_CUDA(ctx, cudaStreamBeginCapture(as_stream(stream), cudaStreamCaptureModeThreadLocal));
  return BSL_OK;
}
int bsl_graph_end(bsl_ctx* ctx, void* stream, void** graph_exec) {
  cudaGraph_t g;
  BSL_CUDA(ctx, cudaStreamEndCapture(as_stream(stream), &g));
  cudaGraphExec_t ge;
  cudaError_t e = cudaGraphInstantiate(&ge, g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) return bsl_check_cuda(ctx, e, "cudaGraphInstantiate");
  *graph_exec = ge;
  return BSL_OK;
}
int bsl_graph_launch(bsl_ctx* ctx, void* graph_exec, void* stream) {
  BSL_CUDA(ctx, cudaGraphLaunch(reinterpret_cast<cudaGraphExec_t>(graph_exec), as_stream(stream)));
  return BSL_OK;
}
int bsl_graph_destroy(bsl_ctx* ctx, void* graph_exec) {
  BSL_CUDA(ctx, cudaGraphExecDestroy(reinterpret_cast<cudaGraphExec_t>(graph_exec)));
  return BSL_OK;
}

}  // extern "C"

int bsl_get_tmap(bsl_ctx* ctx, const void* base, int rank, const uint64_t* dims,
                 const uint64_t* strides_bytes, const uint32_t* box, CUtensorMap* out) {
  return bsl_get_tmap_es(ctx, base, rank, dims, strides_bytes, box, nullptr, out);
}

int bsl_get_tmap_es(bsl_ctx* ctx, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, const uint32_t* elem_strides, CUtensorMap* out) {
  char key[640];
  int n = snprintf(key, sizeof(key), "%p:%d", base, rank);
  for (int i = 0; i < rank; ++i)
    n += snprintf(key + n, sizeof(key) - n, ":%llu,%llu,%u,%u", (unsigned long long)dims[i],
                  (unsigned long long)(i ? strides_bytes[i] : 2), box[i], elem_strides ? elem_strides[i] : 1u);
  {
    std::lock_guard<std::mutex> g(ctx->mu);
    auto it = ctx->tmaps.find(key);
    if (it != ctx->tmaps.end()) {
      *out = it->second;
      return BSL_OK;
    }
  }
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = elem_strides ? elem_strides[i] : 1;
    if (i) gstr[i - 1] = strides_bytes[i];
  }
  alignas(64) CUtensorMap m;
  CUresult r = ctx->encode_tiled(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base),
                                 gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                 CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return bsl_fail(ctx, BSL_ECUDA, "cuTensorMapEncodeTiled failed (%d) for %s", (int)r, key);
  {
    std::lock_guard<std::mutex> g(ctx->mu);
    ctx->tmaps[key] = m;
  }
  *out = m;
  return BSL_OK;
}
