// Halo-tile implicit GEMM for 3x3 / stride-1 / SAME convolutions on sm_100a (tcgen05 + TMEM + TMA).
//
// Measured on B200 (tools/umma_probe.cu, profiles/r01_umma_shifted_descriptor_probe.log): a SWIZZLE_128B
// UMMA shared-memory descriptor may start at any 128-byte aligned address, with any 128-byte multiple
// as the stride between 8-row groups / 64-element blocks, because the swizzle is a function of the
// absolute shared-memory address on both sides (TMA writes, UMMA reads). So the 9 filter taps need not
// be 9 TMA loads of shifted pixel boxes: ONE box with a 1-pixel halo is loaded per 64-channel block and
// tap (r, s) is the same tile read through a descriptor whose start address is moved by
// (r * pitch + s) pixels. That cuts the L2 -> shared-memory traffic of the activation operand ~6x, which
// is what bounded the first-generation kernel (igemm.cuh) on the 64/128-channel layers.
//
//   conv_halo_kernel   fprop / dgrad (and 1x1 / transposed-conv forward as the 1-tap case): persistent CTAs,
//                      static tile schedule, TMEM double-buffered accumulators so the epilogue of tile i
//                      overlaps the MMAs of tile i+1, optional per-channel sum / sum-of-squares of the
//                      bf16-rounded outputs (batch-norm statistics, NetworksV2/base.py:154-162) fused into
//                      the epilogue.   Reference ops: slim.conv2d, NetworksV2/UNet.py:79,85,94.
//   wgrad_halo_kernel  filter gradient: one CTA owns (64 input channels) x (64 output channels) x ALL 9 taps
//                      for a range of pixel tiles; 5 TMEM accumulators hold tap pairs (M = 2 x 64 channels).
//                      Reference op: Conv2DBackpropFilter created by optimizer.minimize, core/solver.py:239.
#pragma once
#include "ptx.cuh"
#include <cuda_bf16.h>

namespace bsl {

// ------------------------------------------------------------------------------------------------ wgrad
struct WgradHaloArgs {
  int ntile_w, ntile_h, n;       // pixel tiles of 16 (w) x 4 (h)
  int k_tiles_total;
  int k_tiles_per_split;
  int cin, cout;                 // padded-to-64 extents of dW
  float* out;                    // [split][kd * 9][cin][cout] fp32 (or dW itself when splits == 1)
  int kd, depth, splits;         // filter depth (blockIdx.z = kdi * splits + split); slices per volume
  DeviceStatus* status;
};

constexpr int WG_THREADS = 192;
constexpr int WG_TW = 16, WG_TH = 4;
constexpr int WG_PITCH = WG_TW + 2;                     // halo tile row pitch in pixels
constexpr int WG_X_ROWS = WG_PITCH * (WG_TH + 2);       // 108 pixels of 128 B
constexpr int WG_X_BYTES = 14336;                       // 108 * 128 = 13824, padded to 1024
constexpr int WG_DY_BYTES = WG_TW * WG_TH * 128;        // 8192
constexpr int WG_STAGE_BYTES = WG_X_BYTES + WG_DY_BYTES;
constexpr int WG_STAGES = 8;
constexpr int WG_SMEM_BYTES = WG_STAGES * WG_STAGE_BYTES + 1024;

// grid = (cin / 64, cout / 64, splits)
__global__ void __launch_bounds__(WG_THREADS)
wgrad_halo_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDY,
                  const WgradHaloArgs p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * WG_STAGES + 1];
  __shared__ uint32_t tmem_slot;
  __shared__ int dead;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t full0 = smem_u32(&bars[0]);
  const uint32_t empty0 = smem_u32(&bars[WG_STAGES]);
  const uint32_t tfull = smem_u32(&bars[2 * WG_STAGES]);
  DeviceStatus* st = p.status;

  if (threadIdx.x == 0) dead = *reinterpret_cast<volatile int*>(&st->error);
  __syncthreads();
  if (dead) return;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmX);
    prefetch_tensormap(&tmDY);
    for (int s = 0; s < WG_STAGES; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    mbar_init(tfull, 1);
    fence_barrier_init();
  } else if (warp == 1) {
    tmem_alloc<512>(smem_u32(&tmem_slot));
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();   // the prologue above touches no data of the previous kernel in the stream
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);

  const int cb = blockIdx.x, nb = blockIdx.y;
  const int kdi = blockIdx.z / p.splits, split = blockIdx.z - kdi * p.splits;
  const int k_begin = split * p.k_tiles_per_split;
  const int k_end = min(p.k_tiles_total, k_begin + p.k_tiles_per_split);
  const int num_k = k_end - k_begin;

  if (warp == 0) {
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kk = 0; kk < num_k; ++kk) {
        if (!mbar_wait(empty0 + 8 * stage, phase ^ 1, st, 11)) break;
        int t = k_begin + kk;
        const int tx = t % p.ntile_w;
        t /= p.ntile_w;
        const int ty = t % p.ntile_h;
        const int img = t / p.ntile_h;
        const uint32_t fb = full0 + 8 * stage;
        const uint32_t sx = smem_base + stage * WG_STAGE_BYTES;
        mbar_arrive_expect_tx(fb, WG_X_ROWS * 128 + WG_DY_BYTES);
        const int z = img % p.depth, vol = img / p.depth;
        tma_load_5d(sx, &tmX, fb, cb * 64, tx * WG_TW - 1, ty * WG_TH - 1, z + kdi - (p.kd >> 1), vol);
        tma_load_5d(sx + WG_X_BYTES, &tmDY, fb, nb * 64, tx * WG_TW, ty * WG_TH, z, vol);
        if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (elect_one_sync()) {
      constexpr uint32_t idesc = make_idesc_bf16(128, 64, true, true);
      // tap pairs (0,1) (2,3) (4,5) (6,7) (8,-): start row of the first tap and distance to the second
      // inside the halo tile, tap t = (r, s) = (t / 3, t % 3) at pixel offset r * PITCH + s.
      int off0[5], lbo[5];
#pragma unroll
      for (int q = 0; q < 5; ++q) {
        const int t0 = 2 * q, t1 = (2 * q + 1 < 9) ? 2 * q + 1 : 2 * q;
        const int o0 = (t0 / 3) * WG_PITCH + t0 % 3, o1 = (t1 / 3) * WG_PITCH + t1 % 3;
        off0[q] = o0 * 128;
        lbo[q] = (o1 > o0 ? o1 - o0 : 1) * 128;  // lone tap 8: second block = garbage rows, never read back
      }
      int stage = 0;
      uint32_t phase = 0;
      bool ok = true;
      for (int kk = 0; kk < num_k; ++kk) {
        if (!mbar_wait(full0 + 8 * stage, phase, st, 12)) { ok = false; break; }
        tc_fence_after();
        const uint32_t sx = smem_base + stage * WG_STAGE_BYTES;
        const uint32_t sdy = sx + WG_X_BYTES;
        const uint64_t db0 = make_smem_desc_sw128(sdy, 8192, 1024);
        uint64_t da0[5];
#pragma unroll
        for (int q = 0; q < 5; ++q) da0[q] = make_smem_desc_sw128(sx + off0[q], lbo[q], 1024);
        const uint32_t first = kk != 0;
#pragma unroll
        for (int y = 0; y < WG_TH; ++y) {
#pragma unroll
          for (int q = 0; q < 5; ++q)
            umma_bf16(tmem_base + q * 64, da0[q] + (uint64_t)((y * WG_PITCH * 128) >> 4),
                      db0 + (uint64_t)((y * WG_TW * 128) >> 4), idesc, first | (uint32_t)(y != 0));
        }
        umma_commit(empty0 + 8 * stage);
        if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
      }
      if (ok) umma_commit(tfull);
    }
  } else {
    const int q4 = warp & 3;
    const int r = q4 * 32 + lane;  // accumulator row: tap-in-pair = r / 64, input channel = r % 64
    const bool alive = mbar_wait(tfull, 0, st, 13);
    tc_fence_after();
    if (alive) {
      const uint32_t trow = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
#pragma unroll 1
      for (int q = 0; q < 5; ++q) {
        const int tap = 2 * q + (r >> 6);
        const bool valid = tap < 9 && !(q == 4 && r >= 64);
        float* o = p.out + ((((long long)split * p.kd + kdi) * 9 + tap) * p.cin + cb * 64 + (r & 63)) * p.cout + nb * 64;
#pragma unroll
        for (int c = 0; c < 64; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(trow + q * 64 + c, v);
          tmem_ld_wait();
          if (valid) {
            float4* dst = reinterpret_cast<float4*>(o + c);
#pragma unroll
            for (int j = 0; j < 8; ++j)
              dst[j] = make_float4(num_k ? __uint_as_float(v[4 * j]) : 0.f, num_k ? __uint_as_float(v[4 * j + 1]) : 0.f,
                                   num_k ? __uint_as_float(v[4 * j + 2]) : 0.f, num_k ? __uint_as_float(v[4 * j + 3]) : 0.f);
          }
        }
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ wgrad, wide
// Filter gradient of layers with cout % 128 == 0. wgrad_halo_kernel issues 128 x 64 x 16 UMMAs, whose operand fetch
// (6 KB per 32 tensor-pipe cycles) saturates the shared-memory read path at ~55 % tensor utilisation
// (profiles/r01_ncu_full_conv_kernels.txt). Here the roles are swapped: A = dy tile (M = 128 output channels), B = THREE
// taps of one filter row read from the halo tile as a 192-wide MN-major operand (the 64-element blocks of the descriptor
// are 128 B = one pixel apart), so one UMMA is 128 x 192 x 16. An earlier version of this kernel (since removed) gave
// each CTA either filter rows 0, 1 or row 2; per-CTA cycle counters (tools/gpu_conv_bench.py
// --ops wgrad --waits, profiles/r02_wgrad_class_timing.log) showed its two CTA classes apart: the rows-0,1 class issues a
// pixel tile's 8 UMMAs (768 tensor cycles) every ~790 cycles, but the row-2 class needs ~630 cycles for 4 UMMAs (384 tensor
// cycles): a CTA cannot take in more than ~48 B per cycle from L2 (30 KB of operands per tile either way), and the split
// planner, which assumed half the time for half the MMAs, left the row-2 CTAs running long after the others had finished.
// Here every CTA fills two 192-column accumulators per pixel tile and loads only the halo rows it reads:
//   class a   filter rows 0, 1 of ONE 64-channel input block:  x box 18 x 5 pixels (11.25 KB) + dy (16 KB) per tile
//   class b   filter row 2 of TWO input blocks:                 2 x box 18 x 4 pixels (18 KB) + dy (16 KB) per tile
// (a lone last input block, cin / 64 odd, runs with one accumulator). Linear grid: all class-a CTAs, then class b, with
// (input block, output block) fastest so that CTAs resident together share x / dy tiles in L2.
struct WgradHalo3Args {
  int ntile_w, ntile_h, n;       // pixel tiles of 16 (w) x 4 (h)
  int k_tiles_total;
  int ncb, nnb, ncb_b;           // cin / 64, cout / 128, ceil(ncb / 2)
  int splits_a, per_a;           // class a: pixel tiles [zi * per_a, ...)
  int splits_b, per_b;
  int n_cta_a;                   // ncb * nnb * kd * splits_a
  int cin, cout;
  float* out_a;                  // [splits_a][kd][6][cin][cout]
  float* out_b;                  // [splits_b][kd][3][cin][cout]
  int kd, depth;                 // filter depth (slice z + kdi - kd / 2 of the volume); slices per volume
  int stages_a, stages_b;        // pipeline depth per class (<= WG3_MAX_STAGES); the launch sizes shared memory to match
  long long* dbg;                // tuning (bsl_debug_set key 3): per CTA {issuer cycles, cycles waiting for a full stage,
                                 // class << 32 | pixel tiles, start ns}
  DeviceStatus* status;
};

constexpr int WG3_DY_BYTES = 2 * WG_DY_BYTES;                         // 128 output channels = two 64-channel blocks
constexpr int WG3_XA_BYTES = 12288;                                  // 18 x 5 pixels x 128 B = 11520, padded to 1024
constexpr int WG3_XB_BYTES = WG_PITCH * WG_TH * 128;                 // 18 x 4 pixels x 128 B = 9216
constexpr int WG3_STAGE_A = WG3_XA_BYTES + WG3_DY_BYTES;             // 28672
constexpr int WG3_STAGE_B = 2 * WG3_XB_BYTES + WG3_DY_BYTES;         // 34816
// Pipeline depth: 8 / 6 stages fit (225 KB), but a CTA that fills the SM's shared memory keeps the HBM-bound passes of
// the main stream from running beside it (the filter gradient runs on a side stream). Timed alone the kernel is equally
// fast with 5 .. 8 stages (4 / 3 stages: 5 % slower); 6 / 5 stages = 171 KB leave room for the neighbours
// (profiles/r02_ab_experiments.md).
constexpr int WG3_MAX_STAGES = 8;
constexpr int WG3_STAGES_A = 6, WG3_STAGES_B = 5;
constexpr int wg3_smem_bytes(int sa, int sb) {
  return (sa * WG3_STAGE_A > sb * WG3_STAGE_B ? sa * WG3_STAGE_A : sb * WG3_STAGE_B) + 1024;
}

__global__ void __launch_bounds__(WG_THREADS)
wgrad_halo3_kernel(const __grid_constant__ CUtensorMap tmXa, const __grid_constant__ CUtensorMap tmXb,
                   const __grid_constant__ CUtensorMap tmDY, const WgradHalo3Args p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * WG3_MAX_STAGES + 1];
  __shared__ uint32_t tmem_slot;
  __shared__ int dead;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t full0 = smem_u32(&bars[0]);
  const uint32_t empty0 = smem_u32(&bars[WG3_MAX_STAGES]);
  const uint32_t tfull = smem_u32(&bars[2 * WG3_MAX_STAGES]);
  DeviceStatus* st = p.status;

  if (threadIdx.x == 0) dead = *reinterpret_cast<volatile int*>(&st->error);
  __syncthreads();
  if (dead) return;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmXa);
    prefetch_tensormap(&tmXb);
    prefetch_tensormap(&tmDY);
    for (int s = 0; s < WG3_MAX_STAGES; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    mbar_init(tfull, 1);
    fence_barrier_init();
  } else if (warp == 1) {
    tmem_alloc<512>(smem_u32(&tmem_slot));
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();   // the prologue above touches no data of the previous kernel in the stream
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);

  // ---- which part of dW this CTA owns
  const bool type_a = (int)blockIdx.x < p.n_cta_a;
  int id = type_a ? blockIdx.x : blockIdx.x - p.n_cta_a;
  const int ncol = type_a ? p.ncb : p.ncb_b;
  const int col = id % ncol;
  id /= ncol;
  const int nb = id % p.nnb;
  const int zz = id / p.nnb;
  const int nsplit = type_a ? p.splits_a : p.splits_b;
  const int kdi = zz / nsplit, zi = zz - kdi * nsplit;
  const int per = type_a ? p.per_a : p.per_b;
  const int k_begin = zi * per;
  const int k_end = min(p.k_tiles_total, k_begin + per);
  const int num_k = max(k_end - k_begin, 0);
  const int cb0 = type_a ? col : 2 * col;                       // first 64-channel input block
  const int nacc = type_a ? 2 : min(2, p.ncb - cb0);            // accumulators: filter rows 0, 1 / input blocks cb0, cb0 + 1
  const int nstage = type_a ? p.stages_a : p.stages_b;
  const int stage_bytes = type_a ? WG3_STAGE_A : WG3_STAGE_B;
  const int dy_off = type_a ? WG3_XA_BYTES : 2 * WG3_XB_BYTES;

  if (warp == 0) {
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t tx_bytes = (type_a ? WG_PITCH * (WG_TH + 1) * 128 : nacc * WG3_XB_BYTES) + WG3_DY_BYTES;
      for (int kk = 0; kk < num_k; ++kk) {
        if (!mbar_wait(empty0 + 8 * stage, phase ^ 1, st, 17)) break;
        int t = k_begin + kk;
        const int tx = t % p.ntile_w;
        t /= p.ntile_w;
        const int ty = t % p.ntile_h;
        const int img = t / p.ntile_h;
        const uint32_t fb = full0 + 8 * stage;
        const uint32_t sx = smem_base + stage * stage_bytes;
        mbar_arrive_expect_tx(fb, tx_bytes);
        const int z = img % p.depth, vol = img / p.depth;
        const int zx = z + kdi - (p.kd >> 1);
        if (type_a) {
          tma_load_5d(sx, &tmXa, fb, cb0 * 64, tx * WG_TW - 1, ty * WG_TH - 1, zx, vol);
        } else {
          tma_load_5d(sx, &tmXb, fb, cb0 * 64, tx * WG_TW - 1, ty * WG_TH + 1, zx, vol);
          if (nacc == 2) tma_load_5d(sx + WG3_XB_BYTES, &tmXb, fb, cb0 * 64 + 64, tx * WG_TW - 1, ty * WG_TH + 1, zx, vol);
        }
        tma_load_5d(sx + dy_off, &tmDY, fb, nb * 128, tx * WG_TW, ty * WG_TH, z, vol);
        tma_load_5d(sx + dy_off + WG_DY_BYTES, &tmDY, fb, nb * 128 + 64, tx * WG_TW, ty * WG_TH, z, vol);
        if (++stage == nstage) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (elect_one_sync()) {
      constexpr uint32_t idesc = make_idesc_bf16(128, 192, true, true);
      int stage = 0;
      uint32_t phase = 0;
      bool ok = true;
      const bool timed = p.dbg != nullptr;
      long long t_all = 0, w_full = 0, t0 = 0;
      unsigned long long ns0 = 0;
      if (timed) { t_all = clock64(); ns0 = globaltimer_ns(); }
      // accumulator a reads the halo tile at acc_off * a: the next filter row (class a) or the next input block (class b)
      const uint32_t acc_off = type_a ? WG_PITCH * 128 : WG3_XB_BYTES;
      for (int kk = 0; kk < num_k; ++kk) {
        if (timed) t0 = clock64();
        if (!mbar_wait(full0 + 8 * stage, phase, st, 18)) { ok = false; break; }
        if (timed) w_full += clock64() - t0;
        tc_fence_after();
        const uint32_t sx = smem_base + stage * stage_bytes;
        const uint64_t da0 = make_smem_desc_sw128(sx + dy_off, WG_DY_BYTES, 1024);
        const uint32_t first = kk != 0;
#pragma unroll
        for (int y = 0; y < WG_TH; ++y) {
          for (int a = 0; a < nacc; ++a) {
            // three taps of one filter row: 64-channel blocks one pixel (128 B) apart, the 16 pixels of row y as K
            const uint64_t db = make_smem_desc_sw128(sx + a * acc_off + (y * WG_PITCH) * 128, 128, 1024);
            umma_bf16(tmem_base + a * 192, da0 + (uint64_t)((y * WG_TW * 128) >> 4), db, idesc,
                      first | (uint32_t)(y != 0));
          }
        }
        umma_commit(empty0 + 8 * stage);
        if (++stage == nstage) { stage = 0; phase ^= 1; }
      }
      if (ok) umma_commit(tfull);
      if (timed && blockIdx.x < 1024) {
        p.dbg[blockIdx.x * 4 + 0] = clock64() - t_all;
        p.dbg[blockIdx.x * 4 + 1] = w_full;
        p.dbg[blockIdx.x * 4 + 2] = ((long long)(type_a ? 0 : 1) << 32) | num_k;
        p.dbg[blockIdx.x * 4 + 3] = (long long)ns0;
      }
    }
  } else {
    const int q4 = warp & 3;
    const int row = q4 * 32 + lane;  // accumulator row = output channel within the 128-block
    const bool alive = mbar_wait(tfull, 0, st, 19);
    tc_fence_after();
    if (alive) {
      const uint32_t trow = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
      const int ntap = type_a ? 6 : 3;
      float* obase = (type_a ? p.out_a : p.out_b) + ((long long)zi * p.kd + kdi) * ntap * p.cin * p.cout + nb * 128 + row;
#pragma unroll 1
      for (int a = 0; a < nacc; ++a) {
        const int tap0 = type_a ? a * 3 : 0;          // first local tap of this accumulator
        const int cblk = type_a ? cb0 : cb0 + a;      // its 64-channel input block
#pragma unroll 1
        for (int c = 0; c < 192; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(trow + a * 192 + c, v);
          tmem_ld_wait();
          float* o = obase + ((long long)(tap0 + c / 64) * p.cin + cblk * 64 + (c & 63)) * p.cout;
#pragma unroll
          for (int j = 0; j < 32; ++j) o[(long long)j * p.cout] = num_k ? __uint_as_float(v[j]) : 0.f;
        }
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------ fprop / dgrad
struct ConvHaloArgs {
  int ntile_w, ntile_h, n;       // sub-tiles of 8 (w) x 16 (h) pixels: ceil(extent / tile)
  int vw, vh;                    // true extents of the pixel grid: rows of a sub-tile outside are neither stored nor counted
  int n_sub_total;               // ntile_w * ntile_h * n
  int n_units;                   // ceil(n_sub_total / NSUB) * n_ntiles
  int n_ntiles;                  // column tiles (N / BN)
  int ntaps;                     // 9 (halo = 1) or 1 (halo = 0)
  int halo;                      // 1: box (10 x 18), 0: box (8 x 16)
  int cblocks;                   // 64-channel blocks of the reduction
  int b_flip;                    // dgrad: B tap = ntaps - 1 - tap
  int b_rows_per_tap;            // K-major B: rows per tap
  // ---- epilogue
  void* out;                     // bf16
  long long ostride_x, ostride_y, ostride_n;  // element strides of the output pixel grid
  int n_group;                   // columns per output group (== N unless transposed-conv scatter)
  long long group_off[8];
  const float* bias;
  int relu;
  int n_total;
  float* stats_part;             // [slot][2][n_total] per-CTA partial sums (nullptr: no statistics)
  // instance statistics (stats_group_imgs > 0): a statistics group is stats_group_imgs consecutive images (1 for 2-D
  // instance norm, the depth of a volume whose slices run as images); each epilogue warp flushes its running sums
  // whenever the group of the sub-tile it is about to add changes (images come in non-decreasing order), into
  // stats_part[group][slot * 4 + lane quarter][2][n_total] (zero-filled by the host: not every CTA meets every group)
  int stats_group_imgs;
  int stats_blocks;              // slots * 4
  int a_stages;                  // B_RES kernels: activation stages that fit beside the resident filter
  int kd;                        // filter depth (1, or 3 for the (3,3,3) layers of UNet3D): the reduction runs over
  int depth;                     //   (kd, 64-channel block, tap); an "image" is slice z = img % depth of volume img / depth
  // ---- transposed-conv backward-data: the A tensor map is upsampled_map (c, b, w, a, n*h); the reduction runs over
  //      (a = kd index, b, 64-channel block): K block cbx -> a = cbx / cblocks, b = cb / up_cpb, channel (cb % up_cpb) * 64
  int up_cpb;                    // 0 = ordinary (c, x, y, z, vol) coordinates
  long long* dbg;                // tuning (bsl_debug_set key 3): per CTA {total, wait acc_empty, wait a_full, wait b_full}
                                 // cycles of the UMMA issuer thread
  // ---- optional per-tap tables (tap_table != 0): one output phase of a STRIDED layer's dgrad is a stride-1 correlation
  //      over dy with a subset of the filter taps -- tap t reads the halo tile at byte offset tap_off[t] and the filter
  //      tap tap_b[kdi * ntaps + t] (conv3d.cu / bsl_conv3d_halo_dgrad_strided)
  int tap_table;
  int tap_off[9];
  signed char tap_b[27];
  DeviceStatus* status;
};

constexpr int CH_SUB_BYTES = 23552;   // (10 x 18) x 128 B = 23040, padded to a multiple of 1024

constexpr int CH_STAGING_BYTES = 2 * 16384;   // TMA-store epilogue: one 128-pixel x 64-channel tile per warp group

// PAIR: a cluster of two CTAs issues 256 x BN x 16 MMAs (cta_group::2) from the even CTA; each CTA owns the pixels of its
// own unit and holds HALF of every filter slice, so a filter stage is half the size (see conv_halo_kernel).
template <int BN, int NSUB, bool TMA_ST = false, bool PAIR = false>
struct ConvHaloCfg {
  static constexpr int ACC_BUFS = (512 / (BN * NSUB)) >= 2 ? 2 : 1;
  static constexpr int TMEM_COLS = BN * NSUB * ACC_BUFS;
  static constexpr int B_BYTES = (PAIR ? BN / 2 : BN) * 128;
  static constexpr int A_BYTES = NSUB * CH_SUB_BYTES;
  // three activation stages hide the HBM latency of the one-block-deep reductions (Cin = 64: a unit is
  // ~1.5 us of MMAs); the widest column tile only occurs with long reductions and keeps two.
  // 256-wide tiles, and 128-wide tiles over sub-tile pairs: two activation stages (a stage is a whole 64-channel block of
  // the reduction, 9 taps of MMAs) leave room for 7 instead of 4 filter stages, which is what the issuer waits for there
  static constexpr int A_STAGES = (BN == 256 || (BN == 128 && NSUB == 2)) ? 2 : 3;
  static constexpr int B_FIT = (212 * 1024 - (TMA_ST ? CH_STAGING_BYTES : 0) - A_STAGES * A_BYTES) / B_BYTES;
  static constexpr int B_STAGES = B_FIT > 8 ? 8 : (B_FIT < 3 ? 3 : B_FIT);
  static constexpr int SMEM_BYTES = A_STAGES * A_BYTES + B_STAGES * B_BYTES + 1024 + (TMA_ST ? CH_STAGING_BYTES : 0);
};

// warp 0: A producer, 1: UMMA issuer, 2..9: epilogue (two warps per TMEM lane quarter), 10: B producer
constexpr int CH_EPI_WARPS = 8;
constexpr int CH_THREADS = (3 + CH_EPI_WARPS) * 32;

// 32 fp32 accumulator columns of one pixel row -> 32 bf16 (64 B) in global memory.
template <bool SCATTER>
__device__ __forceinline__ void ch_store_chunk(const uint32_t (&v)[32], __nv_bfloat16* o, const float* bias,
                                               int relu, uint32_t (&packed)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    float a = __uint_as_float(v[2 * i]);
    float b = __uint_as_float(v[2 * i + 1]);
    if (SCATTER) {
      if (bias) {   // the warp's slice of the bias vector, staged in shared memory by the epilogue loop
        const float2 bb = reinterpret_cast<const float2*>(bias)[i];
        a += bb.x;
        b += bb.y;
      }
      if (relu) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); }
    }
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    packed[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  if ((reinterpret_cast<uintptr_t>(o) & 31) == 0) {
    // two 256-bit stores: every lane fills whole 32-byte sectors (lanes of a warp are different pixels, so a
    // 128-bit store would touch 32 sectors and fill half of each)
    st_global_v8(o, packed[0], packed[1], packed[2], packed[3], packed[4], packed[5], packed[6], packed[7]);
    st_global_v8(o + 16, packed[8], packed[9], packed[10], packed[11], packed[12], packed[13], packed[14], packed[15]);
  } else {
    uint4* dst = reinterpret_cast<uint4*>(o);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      dst[i] = make_uint4(packed[4 * i], packed[4 * i + 1], packed[4 * i + 2], packed[4 * i + 3]);
  }
}

// Sums s1[i], s2[i] (i = column) over the 32 lanes (= rows) of a warp: 5 halving steps, after which lane l holds
// the totals of column l in s1[0], s2[0].
__device__ __forceinline__ void ch_transpose_reduce(float (&s1)[32], float (&s2)[32], int lane) {
#pragma unroll
  for (int w = 16; w >= 1; w >>= 1) {
    const bool hi = (lane & w) != 0;
#pragma unroll
    for (int i = 0; i < w; ++i) {
      const float keep1 = hi ? s1[i + w] : s1[i];
      const float send1 = hi ? s1[i] : s1[i + w];
      const float keep2 = hi ? s2[i + w] : s2[i];
      const float send2 = hi ? s2[i] : s2[i + w];
      s1[i] = keep1 + __shfl_xor_sync(0xffffffffu, send1, w);
      s2[i] = keep2 + __shfl_xor_sync(0xffffffffu, send2, w);
    }
  }
}

// B_RES: the whole filter slice of this CTA's column tile (ntaps x cblocks x BN x 64 channels) is loaded ONCE and
// stays in shared memory; a CTA always owns column tile blockIdx.x % n_ntiles. Chosen by the host when it fits
// (short reductions: the 64- and 128-channel layers, 1x1 and transposed convs), where re-streaming the filter from
// L2 for every unit was 60 % of the TMA bytes and its latency left the tensor pipe idle two thirds of the time
// (profiles/r01_ncu_full_conv_kernels.txt, enc1_2 dgrad). a_stages = p.a_stages activation stages share the rest.
constexpr int CH_MAX_A_STAGES = 4;

// TMA_ST (plain epilogue only: no statistics, no scatter, streamed filter): the bf16 tile goes registers -> swizzled
// shared-memory staging -> one TMA store per 128-pixel x 64-channel block instead of one 32-byte sector per lane and
// store instruction. A lane-per-pixel global store costs one L1 wavefront per 32 bytes on the data path the UMMA
// operand fetch also uses, and left the issuer waiting 16-30 % of the time for the un-overlapped epilogue of the
// 256-wide tiles (gpu_conv_bench --waits); the staged store needs a quarter of the wavefronts and is asynchronous.
//
// PAIR (3x3 windows, sub-tile pairs, plain epilogue, streamed filter): the kernel runs as clusters of two CTAs. Both load
// their own activation tiles and half of every filter slice (rows [rank * BN / 2, ...) of the column tile); the even CTA's
// issuer thread drives BOTH tensor cores with 256 x BN x 16 MMAs, whose rows 0..127 are its own sub-tile and rows 128..255
// the peer's. Per CTA that halves the filter bytes taken in from L2, written to and read back from shared memory -- the
// 128 x 256 x 16 MMA reads 12 KB of operands per 128 cycles (96 B/clk of the 128 B/clk shared memory moves), and the
// filter stream written beside it (32 KB per 1024 cycles) is what the single-CTA kernel's issuer waits for a third of
// the time (`b_full`, tools/gpu_conv_bench.py --waits). Barriers: every TMA load of both CTAs counts its bytes on the
// EVEN CTA's full barriers (cp.async.bulk.tensor.cta_group::2); the issuer's commits arrive on the empty / accumulator
// barriers of both CTAs (multicast); the peer's epilogue warps arrive on the even CTA's acc_empty barrier through DSMEM.
//
// BIAS_RELU (plain epilogue of any schedule, no statistics, no scatter): y = bf16(relu(acc + bias[column])), slim.conv2d
// without a normaliser. The bias of a warp's columns is staged in shared memory once per column tile, as for SCATTER;
// with TMA_ST, whose 256-wide tiles leave no room for 8 KB of staged bias beside the rings, each warp stages the 64
// columns of the chunk it is converting (loaded while the TMEM loads are in flight).
template <int BN, int NSUB, bool B_MN, bool STATS, bool SCATTER, bool B_RES = false, bool TMA_ST = false, bool PAIR = false,
          bool BIAS_RELU = false>
// One CTA per SM: the shared-memory ring takes the SM anyway; with that bound ptxas keeps the epilogue's accumulator
// values in registers instead of spilling them.
__global__ void __launch_bounds__(CH_THREADS, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmO, const ConvHaloArgs p) {
  static_assert(!TMA_ST || (!STATS && !SCATTER && !B_RES), "TMA-store epilogue: plain streamed-filter variant only");
  static_assert(!PAIR || !SCATTER, "CTA pairs: no scatter epilogue");
  static_assert(!BIAS_RELU || (!STATS && !SCATTER), "bias + ReLU epilogue: plain stores only");
  constexpr bool EPI_BIAS = SCATTER || BIAS_RELU;
  constexpr bool TILE_BIAS = SCATTER || (BIAS_RELU && !TMA_ST);   // bias staged per column tile (else per 64-column chunk)
  static_assert(!PAIR || !B_MN || BN >= 128, "CTA pairs: an MN-major filter splits in 64-column blocks");
  using Cfg = ConvHaloCfg<BN, NSUB, TMA_ST, PAIR>;
  constexpr int ACC_BUFS = Cfg::ACC_BUFS;
  constexpr int B_STAGES = Cfg::B_STAGES;
  constexpr int A_BYTES = Cfg::A_BYTES;
  constexpr int B_BYTES = Cfg::B_BYTES;
  constexpr int A_BARS = B_RES ? CH_MAX_A_STAGES : Cfg::A_STAGES;
  const int A_STAGES = B_RES ? p.a_stages : Cfg::A_STAGES;

  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * A_BARS + 2 * B_STAGES + 2 * ACC_BUFS + 2];
  __shared__ uint32_t tmem_slot;
  __shared__ int dead;
  __shared__ float s_stats[STATS ? CH_EPI_WARPS * 2 * BN : 1];
  __shared__ __align__(16) float s_bias[TILE_BIAS ? CH_EPI_WARPS * 256 : (EPI_BIAS ? CH_EPI_WARPS * 64 : 1)];   // per epilogue warp: bias of its columns

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA0 = smem_base;
  const uint32_t sB0 = smem_base + A_STAGES * A_BYTES;
  const uint32_t a_full = smem_u32(&bars[0]);
  const uint32_t a_empty = smem_u32(&bars[A_BARS]);
  const uint32_t b_full = smem_u32(&bars[2 * A_BARS]);
  const uint32_t b_empty = smem_u32(&bars[2 * A_BARS + B_STAGES]);
  const uint32_t acc_full = smem_u32(&bars[2 * A_BARS + 2 * B_STAGES]);
  const uint32_t acc_empty = smem_u32(&bars[2 * A_BARS + 2 * B_STAGES + ACC_BUFS]);
  const uint32_t grp_bar = smem_u32(&bars[2 * A_BARS + 2 * B_STAGES + 2 * ACC_BUFS]);   // TMA_ST: one per warp group
  const uint32_t sStage = sB0 + B_STAGES * B_BYTES;                                     // TMA_ST: 2 x 16 KB
  DeviceStatus* st = p.status;

  // CTA pairs: rank in the cluster; a pair walks "pair units" (one pixel unit per CTA, the same column tile for both)
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const int u_first = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int u_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int u_count = PAIR ? p.n_units >> 1 : p.n_units;
  auto pixel_unit = [&](int u) { return PAIR ? 2 * (u / p.n_ntiles) + (int)rank : u / p.n_ntiles; };

  if (threadIdx.x == 0) dead = *reinterpret_cast<volatile int*>(&st->error);
  if (STATS) {
    for (int i = threadIdx.x; i < CH_EPI_WARPS * 2 * BN; i += CH_THREADS) s_stats[i] = 0.f;
  }
  __syncthreads();
  if (!PAIR && dead) return;   // (a pair never leaves its peer alone at the cluster barriers; the watchdogs unwind it)

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmA);
    prefetch_tensormap(&tmB);
    for (int s = 0; s < A_STAGES; ++s) {
      mbar_init(a_full + 8 * s, 1);
      mbar_init(a_empty + 8 * s, 1);
    }
    for (int s = 0; s < B_STAGES; ++s) {
      mbar_init(b_full + 8 * s, 1);
      mbar_init(b_empty + 8 * s, 1);
    }
    for (int s = 0; s < ACC_BUFS; ++s) {
      mbar_init(acc_full + 8 * s, 1);
      mbar_init(acc_empty + 8 * s, (PAIR ? 2 : 1) * CH_EPI_WARPS);  // one arrival per epilogue warp (of both CTAs)
    }
    mbar_init(grp_bar, 4);       // the four lane-quarter warps of a staging group
    mbar_init(grp_bar + 8, 4);
    if (TMA_ST) prefetch_tensormap(&tmO);
    fence_barrier_init();
  } else if (warp == 1) {
    if (PAIR) {
      tmem_alloc2<Cfg::TMEM_COLS>(smem_u32(&tmem_slot));
      tmem_relinquish2();
    } else {
      tmem_alloc<Cfg::TMEM_COLS>(smem_u32(&tmem_slot));
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // the peer's barriers exist before anything is counted on them
  tc_fence_after();
  pdl_wait();   // the prologue above touches no data of the previous kernel in the stream
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&tmem_slot);

  const int box_w = p.halo ? 10 : 8;
  const int sub_rows = p.halo ? 180 : 128;
  const int kblocks = p.kd * p.cblocks;

  if (warp == 0) {
    // ============================== A producer: one halo'd tile per (sub-tile, 64-channel block)
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      bool ok = true;
      for (int u = u_first; u < u_count && ok; u += u_step) {
        const int pu = pixel_unit(u);
        int nsub = p.n_sub_total - pu * NSUB;
        nsub = nsub > NSUB ? NSUB : nsub;
        int tx[NSUB], ty[NSUB], img[NSUB];
#pragma unroll
        for (int j = 0; j < NSUB; ++j) {
          int s = pu * NSUB + j;
          tx[j] = s % p.ntile_w;
          s /= p.ntile_w;
          ty[j] = s % p.ntile_h;
          img[j] = s / p.ntile_h;
        }
        for (int cbx = 0; cbx < kblocks && ok; ++cbx) {
          if (!mbar_wait(a_empty + 8 * stage, phase ^ 1, st, 21)) { ok = false; break; }
          const uint32_t fb = a_full + 8 * stage;
          const int kdi = cbx / p.cblocks, cb = cbx - kdi * p.cblocks;
          if (PAIR) {   // both CTAs' tiles are counted on the even CTA's barrier
            if (rank == 0) mbar_arrive_expect_tx(fb, 2 * NSUB * sub_rows * 128);
            const uint32_t fbc = mapa_shared(fb, 0);
#pragma unroll
            for (int j = 0; j < NSUB; ++j)
              tma_load_5d_pair(sA0 + stage * A_BYTES + j * CH_SUB_BYTES, &tmA, fbc, cb * 64, tx[j] * 8 - p.halo,
                               ty[j] * 16 - p.halo, img[j] % p.depth + kdi - (p.kd >> 1), img[j] / p.depth);
            if (++stage == A_STAGES) { stage = 0; phase ^= 1; }
            continue;
          }
          mbar_arrive_expect_tx(fb, nsub * sub_rows * 128);
#pragma unroll
          for (int j = 0; j < NSUB; ++j)
            if (j < nsub) {
              if (p.up_cpb != 0)   // (c, b, x, a, row) of the upsampled gradient; rows of all images form one column
                tma_load_5d(sA0 + stage * A_BYTES + j * CH_SUB_BYTES, &tmA, fb, (cb % p.up_cpb) * 64, cb / p.up_cpb,
                            tx[j] * 8, kdi, ty[j] * 16);
              else                 // slices outside the volume are zero-filled by TMA: SAME padding along depth
                tma_load_5d(sA0 + stage * A_BYTES + j * CH_SUB_BYTES, &tmA, fb, cb * 64, tx[j] * 8 - p.halo,
                            ty[j] * 16 - p.halo, img[j] % p.depth + kdi - (p.kd >> 1), img[j] / p.depth);
            }
          if (++stage == A_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 2 + CH_EPI_WARPS) {
    // ============================== B producer: one (tap, 64-channel block) filter slice per stage
    if (B_RES) {
      if (PAIR) {
        // resident filter of a CTA pair (one column tile, n_ntiles == 1): this CTA keeps rows / columns
        // [rank * BN / 2, ...) of every slice; all bytes are counted on the even CTA's barrier
        if (elect_one_sync() && u_first < u_count) {
          if (rank == 0) mbar_arrive_expect_tx(b_full, 2 * kblocks * p.ntaps * B_BYTES);
          const uint32_t fbc = mapa_shared(b_full, 0);
          const int nh = (int)rank * (BN / 2);
          for (int cbx = 0; cbx < kblocks; ++cbx)
            for (int tap = 0; tap < p.ntaps; ++tap) {
              const uint32_t sb = sB0 + (cbx * p.ntaps + tap) * B_BYTES;
              const int kdi = cbx / p.cblocks, cb = cbx - kdi * p.cblocks;
              const int tapb = p.b_flip ? (p.kd * p.ntaps - 1 - (kdi * p.ntaps + tap)) : kdi * p.ntaps + tap;
              if (B_MN) {
                const int krow = (tapb * p.cblocks + cb) * 64;
#pragma unroll
                for (int j = 0; j < BN / 128; ++j) tma_load_2d_pair(sb + j * 8192, &tmB, fbc, nh + 64 * j, krow);
              } else {
                tma_load_2d_pair(sb, &tmB, fbc, cb * 64, tapb * p.b_rows_per_tap + nh);   // box of BN / 2 rows
              }
            }
        }
      } else
      if (elect_one_sync() && (int)blockIdx.x < p.n_units) {
        const int n0 = (blockIdx.x % p.n_ntiles) * BN;
        mbar_arrive_expect_tx(b_full, kblocks * p.ntaps * B_BYTES);
        for (int cbx = 0; cbx < kblocks; ++cbx)
          for (int tap = 0; tap < p.ntaps; ++tap) {
            const uint32_t sb = sB0 + (cbx * p.ntaps + tap) * B_BYTES;
            const int kdi = cbx / p.cblocks, cb = cbx - kdi * p.cblocks;
            const int tapb = p.tap_table ? p.tap_b[kdi * p.ntaps + tap]
                                         : (p.b_flip ? (p.kd * p.ntaps - 1 - (kdi * p.ntaps + tap)) : kdi * p.ntaps + tap);
            if (B_MN) {
              const int krow = (tapb * p.cblocks + cb) * 64;
#pragma unroll
              for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * 8192, &tmB, b_full, n0 + 64 * j, krow);
            } else {
              tma_load_2d(sb, &tmB, b_full, cb * 64, tapb * p.b_rows_per_tap + n0);
            }
          }
      }
    } else if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      bool ok = true;
      for (int u = u_first; u < u_count && ok; u += u_step) {
        const int n0 = (u % p.n_ntiles) * BN;
        for (int cbx = 0; cbx < kblocks && ok; ++cbx) {
          const int kdi = cbx / p.cblocks, cb = cbx - kdi * p.cblocks;
          for (int tap = 0; tap < p.ntaps; ++tap) {
            if (!mbar_wait(b_empty + 8 * stage, phase ^ 1, st, 22)) { ok = false; break; }
            const uint32_t fb = b_full + 8 * stage;
            const uint32_t sb = sB0 + stage * B_BYTES;
            const int tapb = p.tap_table ? p.tap_b[kdi * p.ntaps + tap]
                                         : (p.b_flip ? (p.kd * p.ntaps - 1 - (kdi * p.ntaps + tap)) : kdi * p.ntaps + tap);
            if (PAIR) {   // this CTA's half of the slice: columns / rows [n0 + rank * BN / 2, ...), counted on the even CTA
              if (rank == 0) mbar_arrive_expect_tx(fb, 2 * B_BYTES);
              const uint32_t fbc = mapa_shared(fb, 0);
              const int nh = n0 + (int)rank * (BN / 2);
              if (B_MN) {
                const int krow = (tapb * p.cblocks + cb) * 64;
#pragma unroll
                for (int j = 0; j < BN / 128; ++j) tma_load_2d_pair(sb + j * 8192, &tmB, fbc, nh + 64 * j, krow);
              } else {
                tma_load_2d_pair(sb, &tmB, fbc, cb * 64, tapb * p.b_rows_per_tap + nh);   // box of BN / 2 rows
              }
              if (++stage == B_STAGES) { stage = 0; phase ^= 1; }
              continue;
            }
            mbar_arrive_expect_tx(fb, B_BYTES);
            if (B_MN) {
              const int krow = (tapb * p.cblocks + cb) * 64;
#pragma unroll
              for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * 8192, &tmB, fb, n0 + 64 * j, krow);
            } else {
              tma_load_2d(sb, &tmB, fb, cb * 64, tapb * p.b_rows_per_tap + n0);
            }
            if (++stage == B_STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ============================== UMMA issuer
    if (elect_one_sync() && rank == 0) {   // (the odd CTA of a pair has no issuer: the even one drives both tensor cores)
      constexpr uint32_t idesc = make_idesc_bf16(PAIR ? 256 : 128, BN, false, B_MN);
      auto mma = [](uint32_t d, uint64_t da_, uint64_t db_, uint32_t id, uint32_t accum) {
        if (PAIR) umma2_bf16(d, da_, db_, id, accum); else umma_bf16(d, da_, db_, id, accum);
      };
      auto commit = [](uint32_t bar) { if (PAIR) umma2_commit(bar); else umma_commit(bar); };
      const uint32_t a_sbo = box_w * 128;
      int sa = 0, sb = 0, buf = 0;
      uint32_t pa = 0, pb = 0, pacc = 0;
      bool ok = true;
      long long t_all = clock64(), w_acc = 0, w_a = 0, w_b = 0, t0;
      const bool timed = p.dbg != nullptr;
      const bool fast9 = p.ntaps == 9 && p.halo != 0 && p.tap_table == 0;
      const uint64_t db_base = B_MN ? make_smem_desc_sw128(sB0, 8192, 1024) : make_smem_desc_sw128(sB0, 16, 1024);
      if (B_RES && u_first < u_count) ok = mbar_wait(b_full, 0, st, 27);
      for (int u = u_first; u < u_count && ok; u += u_step) {
        const int pu = pixel_unit(u);
        int nsub = p.n_sub_total - pu * NSUB;
        nsub = nsub > NSUB ? NSUB : nsub;
        t0 = clock64();
        if (!mbar_wait(acc_empty + 8 * buf, pacc ^ 1, st, 23)) { ok = false; break; }
        w_acc += clock64() - t0;
        tc_fence_after();
        const uint32_t acc = tmem_base + buf * (NSUB * BN);
        for (int cb = 0; cb < kblocks && ok; ++cb) {   // cb runs over (kd, 64-channel block) here
          t0 = clock64();
          if (!mbar_wait(a_full + 8 * sa, pa, st, 24)) { ok = false; break; }
          w_a += clock64() - t0;
          const uint32_t a_stage = sA0 + sa * A_BYTES;
          if (B_RES) tc_fence_after();
          if (fast9 && nsub == NSUB) {
            // 3x3 window over a full unit, straight-line: every descriptor is a base plus an IMMEDIATE (tap offset inside
            // the halo tile, sub-tile, K slice): ~2.5 instructions per UMMA. The generic loop below spends ~10 (offset
            // arithmetic, parameter loads, vector-to-uniform moves) in this single thread, which bounded the 128-wide tiles
            // (8 UMMAs of 64 cycles per tap): -14 % on those layers, -4 % on the 64-wide, -2 % on the 256-wide ones
            // (tools/gpu_conv_bench.py against the generic loop; profiles/r02_ab_experiments.md).
            const uint64_t da = make_smem_desc_sw128(a_stage, 16, 10 * 128);
            const uint64_t db_res = db_base + (uint64_t)((cb * 9 * B_BYTES) >> 4);
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              uint64_t db0;
              if (B_RES) {
                db0 = db_res + (uint64_t)((tap * B_BYTES) >> 4);
              } else {
                if (timed) t0 = clock64();
                if (!mbar_wait(b_full + 8 * sb, pb, st, 25)) { ok = false; break; }
                if (timed) w_b += clock64() - t0;
                tc_fence_after();
                db0 = db_base + (uint64_t)((sb * B_BYTES) >> 4);
              }
              const int toff = ((tap / 3) * 10 + tap % 3) * 128;
#pragma unroll
              for (int j = 0; j < NSUB; ++j) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  mma(acc + j * BN, da + (uint64_t)((toff + j * CH_SUB_BYTES + k * 32) >> 4),
                            db0 + (uint64_t)((B_MN ? k * 2048 : k * 32) >> 4), idesc,
                            (tap == 0 && k == 0) ? (uint32_t)(cb != 0) : 1u);
              }
              if (!B_RES) {
                commit(b_empty + 8 * sb);
                if (++sb == B_STAGES) { sb = 0; pb ^= 1; }
              }
            }
          } else
          for (int tap = 0; tap < p.ntaps; ++tap) {
            if (!B_RES) {
              t0 = clock64();
              if (!mbar_wait(b_full + 8 * sb, pb, st, 25)) { ok = false; break; }
              w_b += clock64() - t0;
              tc_fence_after();
            }
            const uint32_t b_stage = B_RES ? sB0 + (cb * p.ntaps + tap) * B_BYTES : sB0 + sb * B_BYTES;
            const int toff = p.tap_table ? p.tap_off[tap] : (p.halo ? ((tap / 3) * box_w + tap % 3) * 128 : 0);
            // descriptors differ only in the 14-bit start-address field: one add per operand per UMMA
            const uint64_t da0 = make_smem_desc_sw128(a_stage + toff, 16, a_sbo);
            const uint64_t db0 = B_MN ? make_smem_desc_sw128(b_stage, 8192, 1024) : make_smem_desc_sw128(b_stage, 16, 1024);
            const uint32_t first = (cb | tap) != 0;
#pragma unroll
            for (int j = 0; j < NSUB; ++j) {
              if (j < nsub) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  mma(acc + j * BN, da0 + (uint64_t)((j * CH_SUB_BYTES + k * 32) >> 4),
                            db0 + (uint64_t)((B_MN ? k * 2048 : k * 32) >> 4), idesc, first | (uint32_t)(k != 0));
              }
            }
            if (!B_RES) {
              commit(b_empty + 8 * sb);
              if (++sb == B_STAGES) { sb = 0; pb ^= 1; }
            }
          }
          commit(a_empty + 8 * sa);
          if (++sa == A_STAGES) { sa = 0; pa ^= 1; }
        }
        if (ok) commit(acc_full + 8 * buf);
        if (++buf == ACC_BUFS) { buf = 0; pacc ^= 1; }
      }
      if (p.dbg != nullptr) {
        p.dbg[blockIdx.x * 4 + 0] = clock64() - t_all;
        p.dbg[blockIdx.x * 4 + 1] = w_acc;
        p.dbg[blockIdx.x * 4 + 2] = w_a;
        p.dbg[blockIdx.x * 4 + 3] = w_b;
      }
    }
  } else {
    // ============================== epilogue (warps 2..9): TMEM -> registers -> bf16 global (+ statistics)
    // Warp e handles TMEM lane quarter (warp & 3); the two warps of a quarter split the work of a unit:
    // NSUB == 2: one sub-tile each; NSUB == 1: half of the columns each.
    const int e = warp - 2;
    const int q = warp & 3;
    const int half = e >> 2;
    const int r = q * 32 + lane;        // accumulator row = pixel (x = r % 8, y = r / 8) of the sub-tile
    constexpr int COLS = NSUB == 2 ? BN : BN / 2;   // columns this warp handles per unit
    const int c_begin = NSUB == 2 ? 0 : half * COLS;
    constexpr int SC = BN / 2;                      // STATS: columns per warp
    constexpr bool PERSIST = STATS && BN == 64;
    const int sc0 = half * SC;
    float acc1[PERSIST ? SC : 1], acc2[PERSIST ? SC : 1];
    if (PERSIST) {
#pragma unroll
      for (int i = 0; i < SC; ++i) acc1[i] = acc2[i] = 0.f;
    }
    int buf = 0;
    uint32_t pacc = 0;
    int bias_n0 = -1;
    uint32_t gphase = 0;
    float* sb = s_bias + (TILE_BIAS ? e * 256 : (EPI_BIAS ? e * 64 : 0));
    // instance statistics: this warp's sums of statistics group `g` -> stats_part[g][slot * 4 + q][2][n_total]
    int cur_grp = -1, last_n0 = 0;
    auto flush_group = [&](int g, int n0) {
      if (!STATS) return;
      float* dst = p.stats_part + ((long long)g * p.stats_blocks + (blockIdx.x / p.n_ntiles) * 4 + q) * (2LL * p.n_total) +
                   n0 + sc0;
#pragma unroll
      for (int c = 0; c < SC; c += 32) {
        if (PERSIST) {
          float s1[32], s2[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            s1[i] = acc1[c + i];
            s2[i] = acc2[c + i];
            acc1[c + i] = acc2[c + i] = 0.f;
          }
          ch_transpose_reduce(s1, s2, lane);
          dst[c + lane] = s1[0];
          dst[p.n_total + c + lane] = s2[0];
        } else {
          const int i0 = (e * 2 + 0) * BN + sc0 + c + lane;
          dst[c + lane] = s_stats[i0];
          dst[p.n_total + c + lane] = s_stats[i0 + BN];
          s_stats[i0] = 0.f;
          s_stats[i0 + BN] = 0.f;
        }
      }
    };
    for (int u = u_first; u < u_count; u += u_step) {
      const int pu = pixel_unit(u);
      const int n0 = (u % p.n_ntiles) * BN;
      int nsub = p.n_sub_total - pu * NSUB;
      nsub = nsub > NSUB ? NSUB : nsub;
      if (TILE_BIAS && p.bias != nullptr && n0 != bias_n0) {
        // (re)stage the bias of this warp's columns: 32 scalar global loads per chunk in the store loop left the
        // epilogue waiting on the long scoreboard (ncu: 4.7 stalled warps per issue, tensor pipe 11 % active)
        __syncwarp();
        for (int i = lane; i < COLS; i += 32) sb[i] = __ldg(p.bias + (n0 + c_begin + i) % p.n_group);
        __syncwarp();
        bias_n0 = n0;
      }
      if (!mbar_wait(acc_full + 8 * buf, pacc, st, 26)) break;
      tc_fence_after();
      const int j = NSUB == 2 ? half : 0;
      if (TMA_ST && j < nsub) {
        // group = the four warps (lane quarters 0..3) with the same `half`: one staging tile, one barrier
        int s = pu * NSUB + j;
        const int tx = s % p.ntile_w;
        s /= p.ntile_w;
        const int ty = s % p.ntile_h;
        const int img = s / p.ntile_h;
        const uint32_t trow = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * (NSUB * BN) + j * BN;
        const uint32_t stg = sStage + half * 16384;
        const uint32_t gb = grp_bar + 8 * half;
        const bool leader = q == 0 && lane == 0;
        const uint32_t rowaddr = stg + r * 128;
#pragma unroll 1
        for (int c = c_begin; c < c_begin + COLS; c += 64) {
          uint32_t v0[32], v1[32], pk[32];
          float bl0 = 0.f, bl1 = 0.f;
          if (BIAS_RELU) {
            bl0 = __ldg(p.bias + n0 + c + lane);
            bl1 = __ldg(p.bias + n0 + c + 32 + lane);
          }
          tmem_ld_32x32(trow + c, v0);
          tmem_ld_32x32(trow + c + 32, v1);
          tmem_ld_wait();
          if (BIAS_RELU) {
            // (the previous chunk's reads of sb ended before the group barriers below)
            sb[lane] = bl0;
            sb[32 + lane] = bl1;
            __syncwarp();
            const float2* bb = reinterpret_cast<const float2*>(sb);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 b0 = bb[i], b1 = bb[16 + i];
              v0[2 * i] = __float_as_uint(fmaxf(__uint_as_float(v0[2 * i]) + b0.x, 0.f));
              v0[2 * i + 1] = __float_as_uint(fmaxf(__uint_as_float(v0[2 * i + 1]) + b0.y, 0.f));
              v1[2 * i] = __float_as_uint(fmaxf(__uint_as_float(v1[2 * i]) + b1.x, 0.f));
              v1[2 * i + 1] = __float_as_uint(fmaxf(__uint_as_float(v1[2 * i + 1]) + b1.y, 0.f));
            }
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            __nv_bfloat162 h0 = __floats2bfloat162_rn(__uint_as_float(v0[2 * i]), __uint_as_float(v0[2 * i + 1]));
            __nv_bfloat162 h1 = __floats2bfloat162_rn(__uint_as_float(v1[2 * i]), __uint_as_float(v1[2 * i + 1]));
            pk[i] = *reinterpret_cast<uint32_t*>(&h0);
            pk[16 + i] = *reinterpret_cast<uint32_t*>(&h1);
          }
          // (1) the previous store of this group has finished reading the staging tile
          if (leader) bulk_wait_read_all();
          __syncwarp();
          if (lane == 0) mbar_arrive(gb);
          if (!mbar_wait(gb, gphase, st, 29)) break;
          gphase ^= 1;
          // (2) row r -> 8 chunks of 16 B at chunk position (i ^ (r & 7)): the tensor map's 128-byte swizzle
#pragma unroll
          for (int i = 0; i < 8; ++i)
            st_shared_v4(rowaddr + (static_cast<uint32_t>(i ^ (r & 7)) << 4), pk[4 * i], pk[4 * i + 1], pk[4 * i + 2],
                         pk[4 * i + 3]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(gb);
          if (!mbar_wait(gb, gphase, st, 30)) break;
          gphase ^= 1;
          if (leader) {
            tma_store_4d(&tmO, stg, n0 + c, tx * 8, ty * 16, img);
            bulk_commit_group();
          }
        }
      }
      if (!TMA_ST && !STATS && j < nsub) {
        int s = pu * NSUB + j;
        const int tx = s % p.ntile_w;
        s /= p.ntile_w;
        const int ty = s % p.ntile_h;
        const int img = s / p.ntile_h;
        const long long off = (long long)(tx * 8 + (r & 7)) * p.ostride_x + (long long)(ty * 16 + (r >> 3)) * p.ostride_y +
                              (long long)img * p.ostride_n;
        const bool inside = tx * 8 + (r & 7) < p.vw && ty * 16 + (r >> 3) < p.vh;   // ragged edge tiles
        __nv_bfloat16* obase = reinterpret_cast<__nv_bfloat16*>(p.out) + off;
        const uint32_t trow = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * (NSUB * BN) + j * BN;
        {
          // two chunks in flight: both TMEM loads are issued before the first is consumed
#pragma unroll 1
          for (int c = c_begin; c < c_begin + COLS; c += 64) {
            uint32_t v0[32], v1[32], packed[16];
            tmem_ld_32x32(trow + c, v0);
            if (COLS >= 64) tmem_ld_32x32(trow + c + 32, v1);
            tmem_ld_wait();
#pragma unroll
            for (int hc = 0; hc < (COLS >= 64 ? 2 : 1); ++hc) {
              const int col = n0 + c + 32 * hc;
              __nv_bfloat16* o;
              const float* bias = nullptr;
              if (SCATTER) {
                const int g = col / p.n_group;          // transposed-conv scatter: column group = filter tap
                const int ngc = col - g * p.n_group;
                o = obase + p.group_off[g] + ngc;
                bias = p.bias ? sb + (c - c_begin) + 32 * hc : nullptr;
              } else {
                o = obase + col;
                if (BIAS_RELU) bias = sb + (c - c_begin) + 32 * hc;
              }
              if (inside) ch_store_chunk<EPI_BIAS>(hc ? v1 : v0, o, bias, BIAS_RELU ? 1 : p.relu, packed);
            }
          }
        }
      }
      if (STATS) {
        // Statistics variant: the two warps of a lane quarter split the COLUMNS (SC each) and walk every sub-tile,
        // so a thread always sees the same SC channels. BN == 64: per-thread running sums over all units of this
        // CTA (fixed order), transposed across the 32 rows once at the end. BN == 128: the sub-tiles' values are
        // added first, then one transpose-reduce per 32-column strip and unit.
        const uint32_t tq = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * (NSUB * BN) + sc0;
        __nv_bfloat16* ob[NSUB];
        int grp[NSUB];
        bool inside[NSUB];
#pragma unroll
        for (int jj = 0; jj < NSUB; ++jj) {
          int s = pu * NSUB + jj;
          const int tx = s % p.ntile_w;
          s /= p.ntile_w;
          const int ty = s % p.ntile_h;
          const int img = s / p.ntile_h;
          inside[jj] = tx * 8 + (r & 7) < p.vw && ty * 16 + (r >> 3) < p.vh;
          grp[jj] = p.stats_group_imgs > 0 ? img / p.stats_group_imgs : 0;
          ob[jj] = reinterpret_cast<__nv_bfloat16*>(p.out) + (long long)(tx * 8 + (r & 7)) * p.ostride_x +
                   (long long)(ty * 16 + (r >> 3)) * p.ostride_y + (long long)img * p.ostride_n + n0 + sc0;
        }
        // sub-tiles [j0, j1) of this unit, all of one statistics group
        auto body = [&](int j0, int j1) {
#pragma unroll
          for (int c = 0; c < SC; c += 32) {
            float s1[32], s2[32];
            if (!PERSIST) {
#pragma unroll
              for (int i = 0; i < 32; ++i) s1[i] = s2[i] = 0.f;
            }
#pragma unroll
            for (int jj = 0; jj < NSUB; ++jj) {
              if (jj >= j0 && jj < j1) {
                uint32_t v[32], packed[16];
                tmem_ld_32x32(tq + jj * BN + c, v);
                tmem_ld_wait();
                if (inside[jj]) {
                  ch_store_chunk<false>(v, ob[jj] + c, nullptr, 0, packed);
                } else {                         // a row of a ragged edge tile outside the image: no store, no count
#pragma unroll
                  for (int i = 0; i < 16; ++i) packed[i] = 0u;
                }
#pragma unroll
                for (int i = 0; i < 16; ++i) {   // the bf16 values just stored: what the normalisation pass reads back
                  const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&packed[i]));
                  if (PERSIST) {
                    acc1[c + 2 * i] += f.x;
                    acc1[c + 2 * i + 1] += f.y;
                    acc2[c + 2 * i] = fmaf(f.x, f.x, acc2[c + 2 * i]);
                    acc2[c + 2 * i + 1] = fmaf(f.y, f.y, acc2[c + 2 * i + 1]);
                  } else {
                    s1[2 * i] += f.x;
                    s1[2 * i + 1] += f.y;
                    s2[2 * i] = fmaf(f.x, f.x, s2[2 * i]);
                    s2[2 * i + 1] = fmaf(f.y, f.y, s2[2 * i + 1]);
                  }
                }
              }
            }
            if (!PERSIST) {
              ch_transpose_reduce(s1, s2, lane);
              s_stats[(e * 2 + 0) * BN + sc0 + c + lane] += s1[0];
              s_stats[(e * 2 + 1) * BN + sc0 + c + lane] += s2[0];
            }
          }
        };
        if (p.stats_group_imgs > 0) {
          int j0 = 0;
          while (j0 < nsub) {
            int j1 = j0 + 1;
            while (j1 < nsub && grp[j1] == grp[j0]) ++j1;
            if (grp[j0] != cur_grp) {
              if (cur_grp >= 0) flush_group(cur_grp, n0);
              cur_grp = grp[j0];
            }
            body(j0, j1);
            j0 = j1;
          }
          last_n0 = n0;
        } else {
          body(0, nsub);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR && rank != 0) mbar_arrive_cluster(mapa_shared(acc_empty + 8 * buf, 0));   // the issuer lives in the even CTA
        else mbar_arrive(acc_empty + 8 * buf);
      }
      if (++buf == ACC_BUFS) { buf = 0; pacc ^= 1; }
    }
    if (TMA_ST && q == 0 && lane == 0) bulk_wait_all();   // the staging tiles stay valid until the last store is done
    if (STATS && p.stats_group_imgs > 0) {
      if (cur_grp >= 0) flush_group(cur_grp, last_n0);
    } else if (PERSIST) {
#pragma unroll
      for (int c = 0; c < SC; c += 32) {
        float s1[32], s2[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) { s1[i] = acc1[c + i]; s2[i] = acc2[c + i]; }
        ch_transpose_reduce(s1, s2, lane);
        s_stats[(e * 2 + 0) * BN + sc0 + c + lane] = s1[0];
        s_stats[(e * 2 + 1) * BN + sc0 + c + lane] = s2[0];
      }
    }
  }

  __syncthreads();
  if (STATS && p.stats_part != nullptr && p.stats_group_imgs == 0) {
    // this CTA always works on column tile blockIdx.x % n_ntiles (the host makes gridDim.x a multiple of it)
    const int n0 = (blockIdx.x % p.n_ntiles) * BN;
    const int slot = blockIdx.x / p.n_ntiles;
    for (int i = threadIdx.x; i < 2 * BN; i += CH_THREADS) {
      const int k = i / BN, c = i - k * BN;
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < CH_EPI_WARPS; ++w) t += s_stats[(w * 2 + k) * BN + c];  // fixed order
      if (n0 + c < p.n_total) p.stats_part[((long long)slot * 2 + k) * p.n_total + n0 + c] = t;
    }
  }
  if (PAIR) cluster_sync_all();   // neither CTA leaves while the other may still signal its barriers
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) tmem_dealloc2<Cfg::TMEM_COLS>(tmem_base);
    else tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

}  // namespace bsl
