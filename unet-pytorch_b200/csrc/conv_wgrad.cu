// conv_wgrad.cu -- weight gradient of the 3x3 (pad 1) / 1x1 convolutions for sm_100a.
//
//   dW[co][(r,s)][ci] = sum_{n,h,w} dz[n,h,w,co] * x[n,h+r-1,w+s-1,ci]
//
// Replaces the autograd wgrad (cuDNN bwd-filter) behind loss.backward() in the reference
// (utils_fit.py:92) for nn.Conv2d at nets/vgg.py:53, nets/unet.py:11-12.
//
// GEMM view: M = 128 output channels (rows of dz, MN-major), N = 3 vertical taps x 64 input
// channels, K = pixels.  Both operands are NHWC (channels contiguous) so both are "MN-major"
// UMMA operands: a TMA box [pixels][64 ch] with 128B swizzle IS the canonical MN-major SW128
// tile (row = one K index, 8 rows = one swizzle atom).
//   * K block = a 16(w) x 8(h) pixel patch; one tcgen05.mma (K=16) consumes one image row of the
//     patch: A = dz rows [j*16, j*16+16), B = x box rows [(j+r)*16, ...) for r = 0..2.
//   * The three vertical taps are ONE instruction with N = 192: the B descriptor's leading-dim
//     byte offset (distance between 64-channel MN atoms) is set to one image row of the box
//     (16 px * 128 B = 2048 B), so "atom r" is the same box shifted down by r rows.
//   * The horizontal taps s are separate work units (separate TMA boxes shifted by s-1).
//   * Work unit = (cout block, cin block, s, K split); fp32 partial sums go to a workspace
//     [split][Cout][taps][Cin]; wgrad_reduce sums the splits and writes OIHW fp32 (deterministic).
//   * Warp roles: warp0 TMA producer, warp1 MMA issuer, warps 2..5 epilogue (TMEM -> global), warps 6-7 bias sums
//     (db = column sums of dz, read from the dz tiles while they sit in shared memory for the MMA).
#include "b2u_internal.h"
#include "b2u_ptx.cuh"

namespace b2u {

constexpr int kWb = 16, kHb = 8;

struct WgradParams {
  int N, H, W;
  int C0, C1, Cout;
  int tiles_w, tiles_h, kblocks;   // kblocks = N * tiles_h * tiles_w
  int num_mblk, num_cblk, splits, units;
  float* partial;                  // [splits][Cout][taps][C0+C1]
  float* bias_partial;             // [splits][Cout] or null: db = column sums of dz (warp 6 sums the staged dz tiles)
};

template <int TAPS, int STAGES>
struct WgCfg {
  static constexpr int kXRows = (TAPS == 9 ? kHb + 2 : kHb) * kWb;
  static constexpr int kXBytes = kXRows * 128;
  static constexpr int kDzHalf = kHb * kWb * 128;       // 64 couts x 128 px
  static constexpr int kDzBytes = 2 * kDzHalf;
  static constexpr int kStage = kDzBytes + kXBytes;
  static constexpr int kOffBar = STAGES * kStage;
  static constexpr int kNumBar = 2 * STAGES + 4;
  static constexpr int kOffTmem = kOffBar + kNumBar * 8;
  static constexpr int kSmemBytes = kOffTmem + 16 + 1024;
  static constexpr int kAccN = TAPS == 9 ? 192 : 64;    // accumulator columns per unit
  static constexpr int kTmemCols = TAPS == 9 ? 512 : 256;
  static constexpr int kAccStride = kTmemCols / 2;
  static_assert(kStage % 1024 == 0, "stage alignment");
  static_assert(kSmemBytes <= 232448, "shared memory budget exceeded");
};

template <int TAPS, int STAGES>
__global__ void __launch_bounds__(256, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap tmX0, const __grid_constant__ CUtensorMap tmX1,
                  const __grid_constant__ CUtensorMap tmDZ, const WgradParams p) {
  using Cfg = WgCfg<TAPS, STAGES>;
  constexpr int S_TAPS = TAPS == 9 ? 3 : 1;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bars = smem_base + Cfg::kOffBar;
  auto full = [&](int i) { return bars + 8u * i; };
  auto empty = [&](int i) { return bars + 8u * (STAGES + i); };
  auto t_full = [&](int i) { return bars + 8u * (2 * STAGES + i); };
  auto t_empty = [&](int i) { return bars + 8u * (2 * STAGES + 2 + i); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::kOffTmem);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmX0);
    tma_prefetch_desc(&tmX1);
    tma_prefetch_desc(&tmDZ);
    // a stage is free again after the MMAs that read it committed AND (bias wanted) warps 6 and 7 have summed / skipped it
    for (int i = 0; i < STAGES; ++i) { mbar_init(full(i), 1); mbar_init(empty(i), p.bias_partial ? 3 : 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(t_full(i), 1); mbar_init(t_empty(i), 4); }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int ctot = p.C0 + p.C1;
  const bool two_halves = p.Cout >= 128;   // cout block = 128 (two 64-channel boxes) or 64

  // unit -> (split, mblk, cblk, s); units sharing the dz tile (same split, mblk) are adjacent
  auto decode = [&](int unit, int& split, int& mblk, int& cblk, int& s) {
    s = unit % S_TAPS; unit /= S_TAPS;
    cblk = unit % p.num_cblk; unit /= p.num_cblk;
    mblk = unit % p.num_mblk;
    split = unit / p.num_mblk;
  };
  auto krange = [&](int split, int& k0, int& k1) {
    const long long kb = p.kblocks;
    k0 = static_cast<int>(kb * split / p.splits);
    k1 = static_cast<int>(kb * (split + 1) / p.splits);
  };

  if (warp == 0) {
    if (lane == 0) {
      int st = 0; uint32_t ph = 0;
      for (int unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
        int split, mblk, cblk, s, k0, k1;
        decode(unit, split, mblk, cblk, s);
        krange(split, k0, k1);
        const int cin0 = cblk * 64;
        const CUtensorMap* tmx = cin0 < p.C0 ? &tmX0 : &tmX1;
        const int cx = cin0 < p.C0 ? cin0 : cin0 - p.C0;
        const int co0 = mblk * 128;
        for (int kb = k0; kb < k1; ++kb) {
          int t = kb;
          const int tw = t % p.tiles_w; t /= p.tiles_w;
          const int th = t % p.tiles_h;
          const int img = t / p.tiles_h;
          const int w0 = tw * kWb, h0 = th * kHb;
          mbar_wait(empty(st), ph ^ 1u);
          const uint32_t base = smem_base + st * Cfg::kStage;
          mbar_expect_tx(full(st), (two_halves ? Cfg::kDzBytes : Cfg::kDzHalf) + Cfg::kXBytes);
          tma_load_4d(base, &tmDZ, full(st), co0, w0, h0, img);
          if (two_halves) tma_load_4d(base + Cfg::kDzHalf, &tmDZ, full(st), co0 + 64, w0, h0, img);
          if (TAPS == 9) tma_load_4d(base + Cfg::kDzBytes, tmx, full(st), cx, w0 + s - 1, h0 - 1, img);
          else           tma_load_4d(base + Cfg::kDzBytes, tmx, full(st), cx, w0, h0, img);
          if (++st == STAGES) { st = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // A = dz (M x K, MN-major), B = x (N x K, MN-major)
      constexpr uint32_t idesc = umma_idesc_bf16(128, Cfg::kAccN, 1, 1);
      const uint32_t lbo_a = two_halves ? Cfg::kDzHalf : 0u;   // Cout == 64: rows 64..127 alias rows 0..63
      // descriptor templates: per MMA only the 14-bit start-address field moves (+128 = one 16-pixel image row)
      const uint64_t a_desc0 = umma_smem_desc(smem_base, lbo_a, 1024, 2u);
      const uint64_t b_desc0 = umma_smem_desc(smem_base + Cfg::kDzBytes, 2048, 1024, 2u);
      int st = 0, as = 0; uint32_t ph = 0, pacc = 0;
      for (int unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
        int split, mblk, cblk, s, k0, k1;
        decode(unit, split, mblk, cblk, s);
        krange(split, k0, k1);
        mbar_wait(t_empty(as), pacc ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * Cfg::kAccStride);
        uint32_t acc = 0;
        for (int kb = k0; kb < k1; ++kb) {
          mbar_wait(full(st), ph);
          tc_fence_after();
          const uint64_t a_st = a_desc0 + static_cast<uint64_t>((st * Cfg::kStage) >> 4);
          const uint64_t b_st = b_desc0 + static_cast<uint64_t>((st * Cfg::kStage) >> 4);
#pragma unroll
          for (int j = 0; j < kHb; ++j)
            tc_mma_bf16(d_tmem, a_st + j * 128, b_st + j * 128, idesc, j == 0 ? acc : 1u);
          acc = 1;
          tc_commit(empty(st));
          if (++st == STAGES) { st = 0; ph ^= 1u; }
        }
        tc_commit(t_full(as));
        if (++as == 2) { as = 0; pacc ^= 1u; }
      }
    }
  } else if (warp >= 6) {
    // ===================== bias warps (6: couts 0..63 of the block, 7: couts 64..127): db[co] = sum over pixels of dz[., co]
    // Mirrors the MMA warp's walk over the stages.  In the one unit per (split, cout block) that owns the bias
    // (cblk == 0, s == 0) it sums the dz tile of every stage from shared memory: lane = (16-byte chunk c of 8
    // channels, row group g), rows g, g+4, ...; the 128-byte swizzle puts logical chunk c of row r at chunk c ^ (r & 7),
    // and the 8 lanes of a quarter warp read one full 128-byte row, so the loads are conflict-free.
    if (p.bias_partial != nullptr) {
      const int c = lane & 7, g = lane >> 3;
      int st = 0; uint32_t ph = 0;
      for (int unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
        int split, mblk, cblk, s, k0, k1;
        decode(unit, split, mblk, cblk, s);
        krange(split, k0, k1);
        const bool bias_unit = cblk == 0 && s == 0;
        const int h = warp - 6;                         // which 64-channel half of the dz tile this warp sums
        const bool mine = bias_unit && (h == 0 || two_halves);
        float sum[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) sum[k] = 0.f;
        for (int kb = k0; kb < k1; ++kb) {
          mbar_wait(full(st), ph);
          if (mine) {
            const uint8_t* tile = smem_gen + st * Cfg::kStage + h * Cfg::kDzHalf;
#pragma unroll 8
            for (int it = 0; it < (kHb * kWb) / 4; ++it) {
              const int row = it * 4 + g;
              const uint4 v = *reinterpret_cast<const uint4*>(tile + row * 128 + ((c ^ (row & 7)) << 4));
              sum[0] += bf16_lo(v.x); sum[1] += bf16_hi(v.x); sum[2] += bf16_lo(v.y); sum[3] += bf16_hi(v.y);
              sum[4] += bf16_lo(v.z); sum[5] += bf16_hi(v.z); sum[6] += bf16_lo(v.w); sum[7] += bf16_hi(v.w);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(empty(st));
          if (++st == STAGES) { st = 0; ph ^= 1u; }
        }
        if (mine) {
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float t = sum[k];
            t += __shfl_xor_sync(0xffffffffu, t, 8);
            t += __shfl_xor_sync(0xffffffffu, t, 16);
            const int co = mblk * 128 + h * 64 + c * 8 + k;
            if (g == 0 && co < p.Cout) p.bias_partial[static_cast<size_t>(split) * p.Cout + co] = t;   // zero for an empty split
          }
        }
      }
    }
  } else {
    const int ew = warp & 3;
    int as = 0; uint32_t pacc = 0;
    for (int unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
      int split, mblk, cblk, s, k0, k1;
      decode(unit, split, mblk, cblk, s);
      krange(split, k0, k1);
      mbar_wait(t_full(as), pacc);
      tc_fence_after();
      const int co = mblk * 128 + ew * 32 + lane;
      const bool valid = co < p.Cout && (two_halves || ew < 2);
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + static_cast<uint32_t>(as * Cfg::kAccStride);
#pragma unroll 1
      for (int c32 = 0; c32 < Cfg::kAccN / 32; ++c32) {
        uint32_t v[32];
        tmem_ld_32x32(t_row + c32 * 32, v);
        tmem_ld_wait();
        if (valid) {
          const int r = (c32 * 32) / 64;
          const int ci = cblk * 64 + (c32 * 32) % 64;
          const int tap = r * S_TAPS + s;
          float4* dst = reinterpret_cast<float4*>(
              p.partial + ((static_cast<size_t>(split) * p.Cout + co) * TAPS + tap) * ctot + ci);
          const bool nz = k1 > k0;
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float4 o;
            o.x = nz ? __uint_as_float(v[q * 4 + 0]) : 0.f;
            o.y = nz ? __uint_as_float(v[q * 4 + 1]) : 0.f;
            o.z = nz ? __uint_as_float(v[q * 4 + 2]) : 0.f;
            o.w = nz ? __uint_as_float(v[q * 4 + 3]) : 0.f;
            dst[q] = o;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(t_empty(as));
      if (++as == 2) { as = 0; pacc ^= 1u; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ----------------------------------------------------------------------------------------------------------------
// Cout == 64, 3x3: operand roles swapped so that no half of the 128-row datapath carries duplicates.
//   A (M x K) = x: the halo box [10 rows][16 px][64 ci]; the two M atoms of one MMA are vertical taps r and r+1 (atom stride
//               = one image row of the box, 2048 B), so M = 128 = 2 taps x 64 input channels.  A second MMA starting
//               at tap 2 supplies r = 2 (its second atom reads past the halo and is discarded).
//   B (N x K) = dz: three boxes [8 rows][16 px][64 co] shifted horizontally by +1, 0, -1 pixels (TMA zero-fills outside
//               the image); sum_c dz[c - (s-1)] x[c] is the tap with x offset s-1, so ONE x box (offset 0) serves all
//               three horizontal taps and N = 192 = 3 taps x 64 output channels.
//   D1[(r in {0,1}, ci)][(s, co)], D2[(r = 2, ci)][(s, co)]: 2 MMAs of N = 192 per image row deliver all 9 taps, where
//   the generic kernel needs 3 (one per horizontal tap, each with its M rows duplicated).
//   The second M atom of D2 would be waste; it is pointed (per-row descriptor, LBO = distance to the tile) at a tile of
//   ones, so rows 64..127 of D2 hold sum_p dz[p][co] -- the bias gradient -- at no extra MMA.
// Work unit = (K split, cin block); accumulators are single-buffered (a unit spans hundreds of K blocks).
// ----------------------------------------------------------------------------------------------------------------
struct Wg64Params {
  int N, H, W, C0, C1;
  int tiles_w, tiles_h, kblocks;
  int num_cblk, splits, units;
  float* partial;                  // [splits][64][9][C0+C1]
  float* bias_partial;             // [splits][64] or null
};

struct Wg64Cfg {
  static constexpr int kStages = 3;
  static constexpr int kXBytes = (kHb + 2) * kWb * 128;     // 20480
  static constexpr int kDzBox = kHb * kWb * 128;            // 16384
  static constexpr int kStage = kXBytes + 3 * kDzBox;       // 69632
  static constexpr int kOffOnes = kStages * kStage;         // one M atom (16 K rows x 128 B) of bf16 1.0
  static constexpr int kOffBar = kOffOnes + 2048;
  static constexpr int kNumBar = 2 * kStages + 2;
  static constexpr int kOffTmem = kOffBar + kNumBar * 8;
  static constexpr int kSmemBytes = kOffTmem + 16 + 1024;
  static constexpr int kTmemCols = 512;                     // D1 at column 0, D2 at column 256 (192 columns each)
  static_assert(kStage % 1024 == 0 && kXBytes % 1024 == 0, "stage alignment");
  static_assert(kSmemBytes <= 232448, "shared memory budget exceeded");
};

__global__ void __launch_bounds__(192, 1)
conv_wgrad64_kernel(const __grid_constant__ CUtensorMap tmX0, const __grid_constant__ CUtensorMap tmX1,
                    const __grid_constant__ CUtensorMap tmDZ, const Wg64Params p) {
  using Cfg = Wg64Cfg;
  constexpr int STAGES = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bars = smem_base + Cfg::kOffBar;
  auto full = [&](int i) { return bars + 8u * i; };
  auto empty = [&](int i) { return bars + 8u * (STAGES + i); };
  const uint32_t t_full = bars + 8u * (2 * STAGES), t_empty = bars + 8u * (2 * STAGES + 1);
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::kOffTmem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmX0); tma_prefetch_desc(&tmX1); tma_prefetch_desc(&tmDZ);
    for (int i = 0; i < STAGES; ++i) { mbar_init(full(i), 1); mbar_init(empty(i), 1); }
    mbar_init(t_full, 1); mbar_init(t_empty, 4);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), Cfg::kTmemCols);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 2048 / 4; i += blockDim.x)
    reinterpret_cast<uint32_t*>(smem_gen + Cfg::kOffOnes)[i] = 0x3F803F80u;   // two bf16 1.0
  fence_proxy_async_smem();        // generic-proxy writes -> visible to the tensor core's async proxy
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int ctot = p.C0 + p.C1;

  auto decode = [&](int unit, int& split, int& cblk) { cblk = unit % p.num_cblk; split = unit / p.num_cblk; };
  auto krange = [&](int split, int& k0, int& k1) {
    const long long kb = p.kblocks;
    k0 = static_cast<int>(kb * split / p.splits);
    k1 = static_cast<int>(kb * (split + 1) / p.splits);
  };

  if (warp == 0) {
    if (lane == 0) {
      int st = 0; uint32_t ph = 0;
      for (int unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
        int split, cblk, k0, k1;
        decode(unit, split, cblk);
        krange(split, k0, k1);
        const int cin0 = cblk * 64;
        const CUtensorMap* tmx = cin0 < p.C0 ? &tmX0 : &tmX1;
        const int cx = cin0 < p.C0 ? cin0 : cin0 - p.C0;
        for (int kb = k0; kb < k1; ++kb) {
          int t = kb;
          const int tw = t % p.tiles_w; t /= p.tiles_w;
          const int th = t % p.tiles_h;
          const int img = t / p.tiles_h;
          const int w0 = tw * kWb, h0 = th * kHb;
          mbar_wait(empty(st), ph ^ 1u);
          const uint32_t base = smem_base + st * Cfg::kStage;
          mbar_expect_tx(full(st), Cfg::kStage);
          tma_load_4d(base, tmx, full(st), cx, w0, h0 - 1, img);
          // N atom s holds dz shifted so that it meets x with offset s - 1: columns w0 - (s - 1) ...
          tma_load_4d(base + Cfg::kXBytes, &tmDZ, full(st), 0, w0 + 1, h0, img);
          tma_load_4d(base + Cfg::kXBytes + Cfg::kDzBox, &tmDZ, full(st), 0, w0, h0, img);
          tma_load_4d(base + Cfg::kXBytes + 2 * Cfg::kDzBox, &tmDZ, full(st), 0, w0 - 1, h0, img);
          if (++st == STAGES) { st = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, 192, 1, 1);
      const uint64_t a_desc0 = umma_smem_desc(smem_base, 2048, 1024, 2u);                         // M atoms: taps r, r+1
      const uint64_t b_desc0 = umma_smem_desc(smem_base + Cfg::kXBytes, Cfg::kDzBox, 1024, 2u);    // N atoms: 3 shifted dz boxes
      // D2's operand: atom 0 = tap r = 2 of image row j, atom 1 = the ones tile (LBO = its distance from atom 0)
      uint64_t a2_desc[STAGES][kHb];
#pragma unroll
      for (int s_ = 0; s_ < STAGES; ++s_)
#pragma unroll
        for (int j = 0; j < kHb; ++j) {
          const uint32_t a0 = smem_base + s_ * Cfg::kStage + (j + 2) * 2048;
          a2_desc[s_][j] = umma_smem_desc(a0, smem_base + Cfg::kOffOnes - a0, 1024, 2u);
        }
      int st = 0; uint32_t ph = 0, pacc = 0;
      for (int unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
        int split, cblk, k0, k1;
        decode(unit, split, cblk);
        krange(split, k0, k1);
        mbar_wait(t_empty, pacc ^ 1u);
        tc_fence_after();
        uint32_t acc = 0;
        for (int kb = k0; kb < k1; ++kb) {
          mbar_wait(full(st), ph);
          tc_fence_after();
          const uint64_t a_st = a_desc0 + static_cast<uint64_t>((st * Cfg::kStage) >> 4);
          const uint64_t b_st = b_desc0 + static_cast<uint64_t>((st * Cfg::kStage) >> 4);
#pragma unroll
          for (int j = 0; j < kHb; ++j) {
            const uint32_t accj = j == 0 ? acc : 1u;
            tc_mma_bf16(tmem_base, a_st + j * 128, b_st + j * 128, idesc, accj);                  // taps r = 0, 1
            uint64_t a2 = a2_desc[0][j];                                                          // tap r = 2 | ones
#pragma unroll
            for (int s_ = 1; s_ < STAGES; ++s_) if (s_ == st) a2 = a2_desc[s_][j];
            tc_mma_bf16(tmem_base + 256, a2, b_st + j * 128, idesc, accj);
          }
          acc = 1;
          tc_commit(empty(st));
          if (++st == STAGES) { st = 0; ph ^= 1u; }
        }
        tc_commit(t_full);
        pacc ^= 1u;
      }
    }
  } else {
    const int ew = warp & 3;
    uint32_t pacc = 0;
    for (int unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
      int split, cblk, k0, k1;
      decode(unit, split, cblk);
      krange(split, k0, k1);
      mbar_wait(t_full, pacc);
      tc_fence_after();
      const bool nz = k1 > k0;
      const int m = ew * 32 + lane;                  // accumulator row = (tap r index, input channel)
      const int ci = cblk * 64 + (m & 63);
#pragma unroll 1
      for (int part = 0; part < 2; ++part) {         // part 0: D1 (r = m / 64), part 1: D2 (r = 2, rows 0..63 only)
        const int r = part == 0 ? (m >> 6) : 2;
        const bool valid = part == 0 || m < 64;
        const uint32_t t_row = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + static_cast<uint32_t>(part * 256);
#pragma unroll 1
        for (int c32 = 0; c32 < 6; ++c32) {
          uint32_t v[32];
          tmem_ld_32x32(t_row + c32 * 32, v);
          tmem_ld_wait();
          if (valid) {
            const int s = (c32 * 32) / 64, co0 = (c32 * 32) % 64;
            float* dst = p.partial + ((static_cast<size_t>(split) * 64 + co0) * 9 + r * 3 + s) * ctot + ci;
#pragma unroll
            for (int q = 0; q < 32; ++q)             // consecutive lanes = consecutive ci: 128-byte stores
              dst[static_cast<size_t>(q) * 9 * ctot] = nz ? __uint_as_float(v[q]) : 0.f;
          }
        }
      }
      if (p.bias_partial != nullptr && cblk == 0 && ew == 2) {
        // rows 64..127 of D2 all hold the column sums of dz; columns 64..127 belong to the unshifted box: db[co]
        uint32_t v[32];
#pragma unroll 1
        for (int c32 = 2; c32 < 4; ++c32) {
          tmem_ld_32x32(tmem_base + (64u << 16) + 256u + c32 * 32, v);
          tmem_ld_wait();
          if (lane == 0) {
#pragma unroll
            for (int q = 0; q < 32; ++q)
              p.bias_partial[static_cast<size_t>(split) * 64 + (c32 - 2) * 32 + q] = nz ? __uint_as_float(v[q]) : 0.f;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(t_empty);
      pacc ^= 1u;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// out[co][ci][r][s] (OIHW fp32) = sum_split partial[split][co][tap][ci]; one thread per (co, ci).
// cin_real < cin_pitch handles the first layer (im2col columns k = tap*cin_real + c, see layout.cu).
// generic path (1x1 convs and the first layer's im2col columns): 256 threads = 64 outputs x 4 split lanes
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, int splits, int Cout, int taps,
                    int cin_pitch, int cin_real, int first_layer) {
  __shared__ float sred[4][64];
  const int o = blockIdx.x * 64 + (threadIdx.x & 63);      // output index in OIHW order: (co, ci, tap)
  const int sl = threadIdx.x >> 6;
  const int total = Cout * cin_real * taps;
  float acc = 0.f;
  if (o < total) {
    const int t = o % taps, ci = (o / taps) % cin_real, co = o / (taps * cin_real);
    // partial is [split][Cout][taps][cin_pitch], or for the first layer [split][Cout][cin_pitch] with k = tap*cin_real + ci
    const size_t split_stride = static_cast<size_t>(Cout) * (first_layer ? 1 : taps) * cin_pitch;
    const float* src = first_layer ? partial + static_cast<size_t>(co) * cin_pitch + t * cin_real + ci
                                   : partial + (static_cast<size_t>(co) * taps + t) * cin_pitch + ci;
    for (int s = sl; s < splits; s += 4) acc += __ldg(src + s * split_stride);
    // first layer with the two-term image split (im2col_first): columns [9 cin, 18 cin) carry the lo halves of the same
    // pixels, so their partial sums belong to the same weight
    if (first_layer == 2)
      for (int s = sl; s < splits; s += 4) acc += __ldg(src + taps * cin_real + s * split_stride);
  }
  sred[sl][threadIdx.x & 63] = acc;
  __syncthreads();
  if (sl == 0 && o < total) dw[o] = (sred[0][threadIdx.x] + sred[1][threadIdx.x]) + (sred[2][threadIdx.x] + sred[3][threadIdx.x]);
}

// 3x3 fast path: block = (co, 64-channel block of ci); 144 threads = 9 taps x 16 float4 columns sum the splits with
// coalesced 16-byte loads, then the 576 results leave through shared memory as one contiguous OIHW run
// (dw[co][ci0..ci0+63][0..8]).
__global__ void __launch_bounds__(160)
wgrad_reduce9_kernel(const float* __restrict__ partial, float* __restrict__ dw, int splits, int Cout, int ctot) {
  __shared__ float tile[9][65];
  const int co = blockIdx.y, ci0 = blockIdx.x * 64;
  const int tid = threadIdx.x;
  if (tid < 144) {
    const int tap = tid / 16, q = tid % 16;
    const size_t split_stride = static_cast<size_t>(Cout) * 9 * ctot;
    const float4* src = reinterpret_cast<const float4*>(partial + (static_cast<size_t>(co) * 9 + tap) * ctot + ci0 + q * 4);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int s = 0;
    for (; s + 4 <= splits; s += 4) {
      const float4 a = __ldg(src + (s * split_stride) / 4), b = __ldg(src + ((s + 1) * split_stride) / 4);
      const float4 c = __ldg(src + ((s + 2) * split_stride) / 4), d = __ldg(src + ((s + 3) * split_stride) / 4);
      acc.x += (a.x + b.x) + (c.x + d.x); acc.y += (a.y + b.y) + (c.y + d.y);
      acc.z += (a.z + b.z) + (c.z + d.z); acc.w += (a.w + b.w) + (c.w + d.w);
    }
    for (; s < splits; ++s) {
      const float4 a = __ldg(src + (s * split_stride) / 4);
      acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
    }
    tile[tap][q * 4 + 0] = acc.x; tile[tap][q * 4 + 1] = acc.y; tile[tap][q * 4 + 2] = acc.z; tile[tap][q * 4 + 3] = acc.w;
  }
  __syncthreads();
  float* out = dw + (static_cast<size_t>(co) * ctot + ci0) * 9;
  for (int j = tid; j < 576; j += blockDim.x) out[j] = tile[j % 9][j / 9];
}

__global__ void wgrad_bias_reduce_kernel(const float* __restrict__ bias_partial, float* __restrict__ db, int splits, int Cout) {
  const int co = blockIdx.x * blockDim.x + threadIdx.x;
  if (co >= Cout) return;
  float acc = 0.f;
  for (int s = 0; s < splits; ++s) acc += bias_partial[static_cast<size_t>(s) * Cout + co];
  db[co] = acc;
}

// Split-K factor: the grid is persistent (one CTA per SM, static round-robin over work units), so the kernel ends
// when the CTA with the most units ends.  Search the split counts that give 3..8 units per SM for the one wasting
// the fewest unit slots in the last round; keep at least 8 K blocks per unit so prologue/epilogue stay amortised.
static int choose_splits(int base_units, int kblocks) {
  const int sms = num_sms();
  int lo = (3 * sms + base_units - 1) / base_units, hi = (8 * sms + base_units - 1) / base_units;
  int cap = kblocks / 8;
  if (cap < 1) cap = 1;
  if (lo > cap) lo = cap;
  if (hi > cap) hi = cap;
  if (lo < 1) lo = 1;
  int best = lo;
  double best_waste = 1e30;
  for (int sp = lo; sp <= hi; ++sp) {
    const long long units = static_cast<long long>(base_units) * sp;
    const long long rounds = (units + sms - 1) / sms;
    const double waste = static_cast<double>(rounds * sms) / static_cast<double>(units);
    if (waste < best_waste - 1e-9) { best_waste = waste; best = sp; }
  }
  return best;
}

struct WgradPlan {
  int num_mblk, num_cblk, s_taps, splits, units, kblocks;
  size_t ws_bytes;
};

static WgradPlan plan_wgrad(int N, int H, int W, int Cin_tot, int Cout, int taps) {
  WgradPlan pl;
  pl.num_mblk = (Cout + 127) / 128;
  pl.num_cblk = Cin_tot / 64;
  pl.s_taps = taps == 9 ? 3 : 1;
  const int tiles_w = (W + kWb - 1) / kWb, tiles_h = (H + kHb - 1) / kHb;
  pl.kblocks = N * tiles_h * tiles_w;
  const int base = pl.num_mblk * pl.num_cblk * pl.s_taps;
  pl.splits = choose_splits(base, pl.kblocks);
  pl.units = base * pl.splits;
  pl.ws_bytes = static_cast<size_t>(pl.splits) * Cout * taps * Cin_tot * sizeof(float)   // weight partials
              + static_cast<size_t>(pl.splits) * Cout * sizeof(float);                // bias partials
  return pl;
}

template <int TAPS, int STAGES>
static int launch_wgrad_cfg(const void* x0, int C0, const void* x1, int C1, const void* dz, int Cout, float* partial,
                            float* bias_partial, const WgradPlan& pl, int N, int H, int W, cudaStream_t st) {
  using Cfg = WgCfg<TAPS, STAGES>;
  auto kern = conv_wgrad_kernel<TAPS, STAGES>;
  static bool attr_done[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "cudaFuncSetAttribute(wgrad): %s", cudaGetErrorString(e));
    attr_done[dev] = true;
  }
  const CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B;
  const int x_box_h = TAPS == 9 ? kHb + 2 : kHb;
  CUtensorMap tmX0, tmX1, tmDZ;
  int rc;
  if ((rc = make_tmap_nhwc(&tmX0, x0, N, H, W, C0, 64, kWb, x_box_h, swz))) return rc;
  if (C1 > 0) {
    if ((rc = make_tmap_nhwc(&tmX1, x1, N, H, W, C1, 64, kWb, x_box_h, swz))) return rc;
  } else {
    tmX1 = tmX0;
  }
  if ((rc = make_tmap_nhwc(&tmDZ, dz, N, H, W, Cout, 64, kWb, kHb, swz))) return rc;
  WgradParams p;
  p.N = N; p.H = H; p.W = W; p.C0 = C0; p.C1 = C1; p.Cout = Cout;
  p.tiles_w = (W + kWb - 1) / kWb; p.tiles_h = (H + kHb - 1) / kHb; p.kblocks = pl.kblocks;
  p.num_mblk = pl.num_mblk; p.num_cblk = pl.num_cblk; p.splits = pl.splits; p.units = pl.units;
  p.partial = partial;
  p.bias_partial = bias_partial;
  const int grid = pl.units < num_sms() ? pl.units : num_sms();
  kern<<<grid, 256, Cfg::kSmemBytes, st>>>(tmX0, tmX1, tmDZ, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "conv_wgrad launch: %s", cudaGetErrorString(e));
  note_launch();
  return 0;
}

struct Wgrad64Plan { int num_cblk, splits, units, kblocks; size_t ws_bytes; };

static Wgrad64Plan plan_wgrad64(int N, int H, int W, int Cin_tot) {
  Wgrad64Plan pl;
  pl.num_cblk = Cin_tot / 64;
  pl.kblocks = N * ((H + kHb - 1) / kHb) * ((W + kWb - 1) / kWb);
  pl.splits = choose_splits(pl.num_cblk, pl.kblocks);
  pl.units = pl.num_cblk * pl.splits;
  pl.ws_bytes = static_cast<size_t>(pl.splits) * 64 * 9 * Cin_tot * sizeof(float) + static_cast<size_t>(pl.splits) * 64 * sizeof(float);
  return pl;
}

static int launch_wgrad64(const void* x0, int C0, const void* x1, int C1, const void* dz, float* partial, float* bias_partial,
                          const Wgrad64Plan& pl, int N, int H, int W, cudaStream_t st) {
  using Cfg = Wg64Cfg;
  static bool attr_done[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "cudaFuncSetAttribute(wgrad64): %s", cudaGetErrorString(e));
    attr_done[dev] = true;
  }
  const CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B;
  CUtensorMap tmX0, tmX1, tmDZ;
  int rc;
  if ((rc = make_tmap_nhwc(&tmX0, x0, N, H, W, C0, 64, kWb, kHb + 2, swz))) return rc;
  if (C1 > 0) {
    if ((rc = make_tmap_nhwc(&tmX1, x1, N, H, W, C1, 64, kWb, kHb + 2, swz))) return rc;
  } else {
    tmX1 = tmX0;
  }
  if ((rc = make_tmap_nhwc(&tmDZ, dz, N, H, W, 64, 64, kWb, kHb, swz))) return rc;
  Wg64Params p;
  p.N = N; p.H = H; p.W = W; p.C0 = C0; p.C1 = C1;
  p.tiles_w = (W + kWb - 1) / kWb; p.tiles_h = (H + kHb - 1) / kHb; p.kblocks = pl.kblocks;
  p.num_cblk = pl.num_cblk; p.splits = pl.splits; p.units = pl.units;
  p.partial = partial;
  p.bias_partial = bias_partial;
  const int grid = pl.units < num_sms() ? pl.units : num_sms();
  conv_wgrad64_kernel<<<grid, 192, Cfg::kSmemBytes, st>>>(tmX0, tmX1, tmDZ, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "conv_wgrad64 launch: %s", cudaGetErrorString(e));
  note_launch();
  return 0;
}

}  // namespace b2u

extern "C" {

size_t b2u_conv_wgrad_workspace(int N, int H, int W, int Cin_tot, int Cout, int taps) {
  if (N <= 0 || H <= 0 || W <= 0 || Cin_tot <= 0 || Cout <= 0) return 0;
  size_t need = b2u::plan_wgrad(N, H, W, Cin_tot, Cout, taps).ws_bytes;
  if (Cout == 64 && taps == 9) {          // the swapped-role kernel may use a different split count
    const size_t n64 = b2u::plan_wgrad64(N, H, W, Cin_tot).ws_bytes;
    if (n64 > need) need = n64;
  }
  return need;
}

// dw: OIHW fp32 [Cout][cin_real][taps]  (cin_real = C0+C1 unless first_cin > 0); db (nullable): [Cout] bias gradient,
// computed in the same pass as column sums of dz.
// first_cin > 0: x0 is the first layer's im2col tensor [N,H,W,64] (taps must be 1, C0 == 64, C1 == 0);
//                dw then is [Cout][first_cin][3][3].
// flags bit1: never use the swapped-role Cout = 64 kernel; every other bit is rejected.
int b2u_conv_wgrad(const void* x0, int C0, const void* x1, int C1, const void* dz, int Cout, float* dw, float* db, void* ws,
                   size_t ws_bytes, int N, int H, int W, int taps, int first_cin, int flags, void* stream) {
  using namespace b2u;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!x1) C1 = 0;
  const int ctot = C0 + C1;
  if (flags & ~2) return set_error(B2U_ERR_ARG, "wgrad: unknown flags 0x%x (only bit 1 is defined)", flags);
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "wgrad: empty tensor");
  if (taps != 9 && taps != 1) return set_error(B2U_ERR_SHAPE, "wgrad: taps must be 9 or 1");
  if (C0 % 64 != 0 || C1 % 64 != 0 || ctot <= 0)
    return set_error(B2U_ERR_SHAPE, "wgrad: input channels (%d,%d) must be multiples of 64", C0, C1);
  if (Cout % 64 != 0) return set_error(B2U_ERR_SHAPE, "wgrad: Cout %d must be a multiple of 64", Cout);   // a ragged last 128-block reads zero-filled (out-of-bounds) dz channels
  if (first_cin > 0 && (taps != 1 || C0 != 64 || C1 != 0 || 9 * first_cin > 64))
    return set_error(B2U_ERR_SHAPE, "wgrad: first-layer mode needs taps=1, C0=64, C1=0, 9*cin<=64");
  if (Cout == 64 && taps == 9 && !(flags & 2)) {
    // flags bit1 forces the generic kernel (tests); otherwise Cout = 64 runs with swapped operand roles
    const Wgrad64Plan p64 = plan_wgrad64(N, H, W, ctot);
    if (ws == nullptr || ws_bytes < p64.ws_bytes)
      return set_error(B2U_ERR_ARG, "wgrad: workspace %zu bytes < required %zu", ws_bytes, p64.ws_bytes);
    float* wp64 = static_cast<float*>(ws);
    float* bp64 = db ? wp64 + static_cast<size_t>(p64.splits) * 64 * 9 * ctot : nullptr;
    int rc64 = launch_wgrad64(x0, C0, x1, C1, dz, wp64, bp64, p64, N, H, W, st);
    if (rc64) return rc64;
    if (db) {
      wgrad_bias_reduce_kernel<<<1, 128, 0, st>>>(bp64, db, p64.splits, 64);
      cudaError_t eb = cudaGetLastError();
      if (eb != cudaSuccess) return set_error(B2U_ERR_CUDA, "wgrad_bias_reduce launch: %s", cudaGetErrorString(eb));
      note_launch();
    }
    wgrad_reduce9_kernel<<<dim3(ctot / 64, 64), 160, 0, st>>>(static_cast<const float*>(ws), dw, p64.splits, 64, ctot);
    cudaError_t e64 = cudaGetLastError();
    if (e64 != cudaSuccess) return set_error(B2U_ERR_CUDA, "wgrad_reduce launch: %s", cudaGetErrorString(e64));
    note_launch();
    return 0;
  }
  const WgradPlan pl = plan_wgrad(N, H, W, ctot, Cout, taps);
  if (ws == nullptr || ws_bytes < pl.ws_bytes)
    return set_error(B2U_ERR_ARG, "wgrad: workspace %zu bytes < required %zu", ws_bytes, pl.ws_bytes);
  int rc;
  float* wpart = static_cast<float*>(ws);
  float* bpart = db ? wpart + static_cast<size_t>(pl.splits) * Cout * taps * ctot : nullptr;
  if (taps == 9) rc = launch_wgrad_cfg<9, 4>(x0, C0, x1, C1, dz, Cout, wpart, bpart, pl, N, H, W, st);
  else           rc = launch_wgrad_cfg<1, 4>(x0, C0, x1, C1, dz, Cout, wpart, bpart, pl, N, H, W, st);
  if (rc) return rc;
  if (db) {
    wgrad_bias_reduce_kernel<<<(Cout + 127) / 128, 128, 0, st>>>(bpart, db, pl.splits, Cout);
    cudaError_t eb = cudaGetLastError();
    if (eb != cudaSuccess) return set_error(B2U_ERR_CUDA, "wgrad_bias_reduce launch: %s", cudaGetErrorString(eb));
    note_launch();
  }
  const int cin_real = first_cin > 0 ? first_cin : ctot;
  const int rtaps = first_cin > 0 ? 9 : taps;
  const int total = Cout * cin_real;
  if (taps == 9)
    wgrad_reduce9_kernel<<<dim3(ctot / 64, Cout), 160, 0, st>>>(static_cast<const float*>(ws), dw, pl.splits, Cout, ctot);
  else
    wgrad_reduce_kernel<<<(total * rtaps + 63) / 64, 256, 0, st>>>(static_cast<const float*>(ws), dw, pl.splits, Cout, rtaps, ctot,
                                                                   cin_real, first_cin > 0 ? (18 * first_cin <= 64 ? 2 : 1) : 0);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "wgrad_reduce launch: %s", cudaGetErrorString(e));
  note_launch();
  return 0;
}

// wgrad of a conv that ran as a 1x1 GEMM over im2col rows (first VGG layer: Kpad 64, 3x3; ResNet stem: Kpad 192, 7x7):
// dw[co][c][tap] = partial column tap*cin + c
int b2u_conv_wgrad_im2col(const void* x0, int Kpad, const void* dz, int Cout, float* dw, void* ws, size_t ws_bytes, int N,
                          int H, int W, int cin, int taps, void* stream) {
  using namespace b2u;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "wgrad_im2col: empty tensor");
  if (Kpad % 64 != 0 || cin <= 0 || taps <= 0 || cin * taps > Kpad) return set_error(B2U_ERR_SHAPE, "wgrad_im2col: bad K layout");
  if (Cout % 64 != 0) return set_error(B2U_ERR_SHAPE, "wgrad_im2col: Cout %d must be a multiple of 64", Cout);
  const WgradPlan pl = plan_wgrad(N, H, W, Kpad, Cout, 1);
  if (ws == nullptr || ws_bytes < pl.ws_bytes) return set_error(B2U_ERR_ARG, "wgrad_im2col: workspace too small");
  int rc = launch_wgrad_cfg<1, 4>(x0, Kpad, nullptr, 0, dz, Cout, static_cast<float*>(ws), nullptr, pl, N, H, W, st);
  if (rc) return rc;
  const int total = Cout * cin * taps;
  wgrad_reduce_kernel<<<(total + 63) / 64, 256, 0, st>>>(static_cast<const float*>(ws), dw, pl.splits, Cout, taps, Kpad, cin, 1);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "wgrad_reduce launch: %s", cudaGetErrorString(e));
  note_launch();
  return 0;
}

}  // extern "C"
