// tcgen05 implicit-GEMM kernel family for sm_100a. One warp-specialised kernel template covers
// every dense contraction on the U-Net hot path (SURVEY.md §2b K1-K3, K5):
//
//   MODE_PIX_M  rows of the GEMM are 128 output pixels (a TMA box over the NHWC activation
//               tensor, zero-filled out of bounds = TF "SAME" padding for free), columns are
//               output channels, the reduction runs over (filter tap, 64-channel block).
//               conv fprop  (reference call site NetworksV2/UNet.py:79)   : B = HWIO weights, N-major
//               conv dgrad  (tf.gradients of the above, core/solver.py:239): B = HWIO weights, K-major,
//                                                                            taps visited in reverse
//               convT fwd   (NetworksV2/UNet.py:91)  : 1 tap, columns = (tap,cout), scatter epilogue
//               convT dgrad                          : 4 taps through a 5-D view of dOut
//   MODE_PIX_K  the reduction runs over pixels (split-K), rows are (filter tap, input channel),
//               columns are output channels: conv / convT wgrad. Both operands are MN-major views
//               of NHWC tensors; the fp32 partials land in [split][taps*Cin][Cout] = HWIO order.
//
// Operands are bf16, accumulation is fp32 in TMEM. Warp roles: warp 0 = TMA producer,
// warp 1 = UMMA issuer + TMEM owner, warps 2..5 = epilogue (TMEM -> registers -> global).
#pragma once
#include "ptx.cuh"
#include <cuda_bf16.h>

namespace bsl {

enum { MODE_PIX_M = 0, MODE_PIX_K = 1 };

struct IgemmArgs {
  int tdim[4];           // logical pixel-grid extents, dims 1..4 of the activation tensor map
  int tbox[4];           // pixel box per TMA load: product 128 (MODE_PIX_M) or 64 (MODE_PIX_K)
  int ntile[4];          // ceil(tdim / tbox)
  int ntaps;             // filter taps
  int cblocks;           // 64-channel blocks per tap on the A side
  int b_flip;            // MODE_PIX_M: 1 = visit B taps in reverse (stride-1 dgrad), 2 = B tap index from tapb[]
  int b_rows_per_tap;    // MODE_PIX_M, K-major B: B rows per tap
  signed char tapoff[27][4];  // per tap: offsets added to A-map coordinates 1..4
  signed char tapb[27];  // b_flip == 2: filter tap read for loop tap t (phase decomposition of strided dgrad)
  int istride[4];        // A-map coordinate = pixel coordinate * istride + tapoff (strided convs: the A map
                         // carries the same traversal stride, so a box still holds tbox consecutive OUTPUT pixels)
  // ---- epilogue
  void* out;             // bf16 (MODE_PIX_M) or fp32 partials (MODE_PIX_K)
  long long ostride[4];  // MODE_PIX_M: output element stride per pixel-grid dim
  int n_group;           // MODE_PIX_M: columns per output group (== N unless convT scatter)
  long long group_off[8];//             element offset added for column group g
  const float* bias;     // MODE_PIX_M: optional per-column-in-group bias
  int relu;              // MODE_PIX_M: clamp at zero after bias
  int m_total;           // MODE_PIX_K: valid rows (ntaps*cblocks*64)
  int n_total;           // valid columns
  int k_tiles_per_split; // MODE_PIX_K: pixel tiles per split
  int k_tiles_total;     // MODE_PIX_K
  // UMMA shared-memory descriptor strides (bytes) for MN-major operands: LBO = distance between
  // 64-element blocks along M/N, SBO = distance between 8-row groups along K, KADV = start-address
  // step per UMMA_K(16). Constants of the layout TMA produces; kept as arguments so a probe can
  // vary them (bsl_debug_set) without a rebuild.
  int mn_lbo, mn_sbo, mn_kadv;
  DeviceStatus* status;
};

constexpr int IGEMM_THREADS = 192;
constexpr int IGEMM_A_BYTES = 128 * 128;  // 128 rows x 64 bf16 (K-major) or 2 x (64 x 64) MN-major

template <int BN, int STAGES>
constexpr int igemm_smem_bytes() {
  return STAGES * (IGEMM_A_BYTES + BN * 128) + 1024;
}

template <int MODE, bool B_MN, int BN, int STAGES>
__global__ void __launch_bounds__(IGEMM_THREADS)
igemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
             const IgemmArgs p) {
  constexpr int A_BYTES = IGEMM_A_BYTES;
  constexpr int B_BYTES = BN * 128;
  constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr bool A_MN = (MODE == MODE_PIX_K);
  static_assert(MODE == MODE_PIX_M || B_MN, "pixel-reduction GEMM uses MN-major operands");
  static_assert(BN == 64 || BN == 128 || BN == 256, "BN");

  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * STAGES + 1];
  __shared__ uint32_t tmem_slot;
  __shared__ int dead;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t full0 = smem_u32(&bars[0]);
  const uint32_t empty0 = smem_u32(&bars[STAGES]);
  const uint32_t tfull = smem_u32(&bars[2 * STAGES]);
  DeviceStatus* st = p.status;

  if (threadIdx.x == 0) dead = *reinterpret_cast<volatile int*>(&st->error);
  __syncthreads();
  if (dead) return;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmA);
    prefetch_tensormap(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    mbar_init(tfull, 1);
    fence_barrier_init();
  } else if (warp == 1) {
    tmem_alloc<BN>(smem_u32(&tmem_slot));
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();   // the prologue above touches no data of the previous kernel in the stream
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);

  // ---- tile coordinates
  const int n0 = blockIdx.y * BN;
  int x[4] = {0, 0, 0, 0};   // MODE_PIX_M: pixel-box origin of this CTA's 128 rows
  int k_begin = 0, k_end = 0;
  if (MODE == MODE_PIX_M) {
    int t = blockIdx.x;
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      x[d] = (t % p.ntile[d]) * p.tbox[d];
      t /= p.ntile[d];
    }
    k_end = p.ntaps * p.cblocks;
  } else {
    k_begin = blockIdx.z * p.k_tiles_per_split;
    k_end = min(p.k_tiles_total, k_begin + p.k_tiles_per_split);
  }
  const int num_k = k_end - k_begin;

  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kk = 0; kk < num_k; ++kk) {
        if (!mbar_wait(empty0 + 8 * stage, phase ^ 1, st, 1)) break;
        const uint32_t fb = full0 + 8 * stage;
        const uint32_t sa = smem_base + stage * STAGE_BYTES;
        const uint32_t sb = sa + A_BYTES;
        mbar_arrive_expect_tx(fb, STAGE_BYTES);
        if (MODE == MODE_PIX_M) {
          const int tap = kk / p.cblocks;
          const int cb = kk - tap * p.cblocks;
          tma_load_5d(sa, &tmA, fb, cb * 64, x[0] * p.istride[0] + p.tapoff[tap][0],
                      x[1] * p.istride[1] + p.tapoff[tap][1], x[2] * p.istride[2] + p.tapoff[tap][2],
                      x[3] * p.istride[3] + p.tapoff[tap][3]);
          const int tapb = p.b_flip == 2 ? p.tapb[tap] : (p.b_flip ? (p.ntaps - 1 - tap) : tap);
          if (B_MN) {
            const int krow = (tapb * p.cblocks + cb) * 64;
#pragma unroll
            for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * 8192, &tmB, fb, n0 + 64 * j, krow);
          } else {
            tma_load_2d(sb, &tmB, fb, cb * 64, tapb * p.b_rows_per_tap + n0);
          }
        } else {
          int t = k_begin + kk;
          int px[4];
#pragma unroll
          for (int d = 0; d < 4; ++d) {
            px[d] = (t % p.ntile[d]) * p.tbox[d];
            t /= p.ntile[d];
          }
#pragma unroll
          for (int blk = 0; blk < 2; ++blk) {
            int mblk = blockIdx.x * 2 + blk;
            if (mblk >= p.ntaps * p.cblocks) mblk = p.ntaps * p.cblocks - 1;  // rows ignored later
            const int tap = mblk / p.cblocks;
            const int cb = mblk - tap * p.cblocks;
            tma_load_5d(sa + blk * 8192, &tmA, fb, cb * 64, px[0] * p.istride[0] + p.tapoff[tap][0],
                        px[1] * p.istride[1] + p.tapoff[tap][1], px[2] * p.istride[2] + p.tapoff[tap][2],
                        px[3] * p.istride[3] + p.tapoff[tap][3]);
          }
#pragma unroll
          for (int j = 0; j < BN / 64; ++j)
            tma_load_5d(sb + j * 8192, &tmB, fb, n0 + 64 * j, px[0], px[1], px[2], px[3]);
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ============================== UMMA issuer ===============================
    if (elect_one_sync()) {
      constexpr uint32_t idesc = make_idesc_bf16(128, BN, A_MN, B_MN);
      int stage = 0;
      uint32_t phase = 0;
      bool ok = true;
      for (int kk = 0; kk < num_k; ++kk) {
        if (!mbar_wait(full0 + 8 * stage, phase, st, 2)) { ok = false; break; }
        tc_fence_after();
        const uint32_t sa = smem_base + stage * STAGE_BYTES;
        const uint32_t sb = sa + A_BYTES;
#pragma unroll
        for (int k = 0; k < 4; ++k) {  // 4 x UMMA_K(16) = 64 reduction elements per stage
          const uint64_t da = A_MN ? make_smem_desc_sw128(sa + k * p.mn_kadv, p.mn_lbo, p.mn_sbo)
                                   : make_smem_desc_sw128(sa + k * 32, 16, 1024);
          const uint64_t db = B_MN ? make_smem_desc_sw128(sb + k * p.mn_kadv, p.mn_lbo, p.mn_sbo)
                                   : make_smem_desc_sw128(sb + k * 32, 16, 1024);
          umma_bf16(tmem_base, da, db, idesc, (kk | k) != 0);
        }
        umma_commit(empty0 + 8 * stage);  // frees this smem stage once the UMMAs have read it
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (ok) umma_commit(tfull);  // accumulator complete
    }
  } else {
    // ================================ epilogue ================================
    const int q = warp & 3;               // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;          // accumulator row
    const bool alive = mbar_wait(tfull, 0, st, 3);
    tc_fence_after();
    if (alive) {
      const uint32_t trow = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
      if (MODE == MODE_PIX_M) {
        int rr = r;
        bool valid = true;
        long long off = 0;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
          const int i = rr % p.tbox[d];
          rr /= p.tbox[d];
          valid = valid && (x[d] + i < p.tdim[d]);
          off += static_cast<long long>(x[d] + i) * p.ostride[d];
        }
        const int g = n0 / p.n_group;
        const int ng0 = n0 - g * p.n_group;
        __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) + off + p.group_off[g] + ng0;
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(trow + c, v);
          tmem_ld_wait();
          if (valid && n0 + c < p.n_total) {
            uint32_t packed[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float a = __uint_as_float(v[2 * j]);
              float b = __uint_as_float(v[2 * j + 1]);
              if (p.bias) {
                a += __ldg(p.bias + ng0 + c + 2 * j);
                b += __ldg(p.bias + ng0 + c + 2 * j + 1);
              }
              if (p.relu) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); }
              __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
              packed[j] = *reinterpret_cast<uint32_t*>(&h);
            }
            if ((reinterpret_cast<uintptr_t>(o + c) & 31) == 0) {   // whole 32-byte sectors per lane
              st_global_v8(o + c, packed[0], packed[1], packed[2], packed[3], packed[4], packed[5], packed[6], packed[7]);
              st_global_v8(o + c + 16, packed[8], packed[9], packed[10], packed[11], packed[12], packed[13], packed[14],
                           packed[15]);
            } else {
              uint4* dst = reinterpret_cast<uint4*>(o + c);
#pragma unroll
              for (int j = 0; j < 4; ++j)
                dst[j] = make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
            }
          }
        }
      } else {
        const int row = blockIdx.x * 128 + r;
        const bool valid = row < p.m_total;
        float* o = reinterpret_cast<float*>(p.out) +
                   (static_cast<long long>(blockIdx.z) * p.m_total + row) * p.n_total + n0;
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(trow + c, v);
          tmem_ld_wait();
          if (valid && n0 + c < p.n_total) {
            if ((reinterpret_cast<uintptr_t>(o + c) & 31) == 0) {
#pragma unroll
              for (int j = 0; j < 4; ++j)
                st_global_v8(o + c + 8 * j, v[8 * j], v[8 * j + 1], v[8 * j + 2], v[8 * j + 3], v[8 * j + 4], v[8 * j + 5],
                             v[8 * j + 6], v[8 * j + 7]);
            } else {
              float4* dst = reinterpret_cast<float4*>(o + c);
#pragma unroll
              for (int j = 0; j < 8; ++j)
                dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                     __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
            }
          }
        }
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<BN>(tmem_base);
  }
}

}  // namespace bsl
