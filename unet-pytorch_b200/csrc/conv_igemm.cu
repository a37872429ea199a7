// conv_igemm.cu -- implicit-GEMM convolution (3x3 pad 1 / 1x1, stride 1) for sm_100a.
//
//   y[n,h,w,co] = act( sum_{r,s,ci} x[n,h+r-1,w+s-1,ci] * Wp[co,(r*3+s)*C+ci] + bias[co] ) (* mask)
//
// Replaces the library calls behind nn.Conv2d(k=3,p=1)+ReLU in the reference
// (nets/vgg.py:53-57, nets/unet.py:11-12,18-21) and, with flipped/transposed packed
// weights, their autograd dgrad (utils_fit.py:92).  The channel concat of unetUp
// (nets/unet.py:17) is never materialised: the K loop walks source 0 (skip) then
// source 1 (upsampled) through two tensor maps; the dgrad of that conv writes its two
// channel ranges to two tensors.
//
// Mapping to the hardware (B200):
//   * GEMM M = 128 output pixels = an 8(w) x 16(h) spatial patch of one image, N = BN output
//     channels, K = taps x input channels in blocks of 64.
//   * A operand: ONE TMA box per channel block: (16 MT + 2) x (8 + 2) pixels x 64 channels, zero-filled outside the
//     image by TMA (this IS the padding), 128-byte swizzled, and all NINE taps read it in place: accumulator row
//     m = h * 8 + w of tap (r, s) is box pixel (h + r) * 10 + (w + s), so the UMMA descriptor of a tap is the box
//     address + (r * 10 + s) * 128 B with a stride of one box row (1280 B) between the 8-pixel groups.  The tensor core
//     applies the 128B swizzle to absolute shared-memory address bits, so an operand may start at any 128-byte row and
//     use any group stride (scripts/umma_unaligned_probe.cu measures exactly that): the input is fetched 1.3-1.4 x per
//     conv (halo only) instead of once per horizontal tap (3.2-3.75 x).
//   * B operand: packed weights [Cout][taps*C] (K-major), one TMA box per tap.
//   * tcgen05.mma (cta_group::1, M=128, N=BN, K=16), fp32 accumulators in TMEM, double
//     buffered so the epilogue of tile i overlaps the main loop of tile i+1.
//   * Warp roles: warp0 = TMA producer, warp1 = MMA issuer (+TMEM alloc), warps 2..5 =
//     epilogue (tcgen05.ld -> bias/ReLU/mask -> bf16 -> swizzled smem -> TMA store).
//   * Persistent: grid = min(tiles, #SM).  Tiles are handed out DYNAMICALLY: the producer thread takes the next tile id
//     with one atomicAdd on a per-launch counter and passes it to the MMA and epilogue warps through a 4-deep
//     shared-memory queue (mbarrier full/empty pairs), so a CTA that lost its SM for a while to another kernel (the NCCL
//     all-reduce of the data-parallel step) simply takes fewer tiles instead of holding the whole grid back.  The
//     cp.async mask-stream variants (MD > 0), whose prefetch runs across tile boundaries, keep the static round robin
//     (the same queue carries the static sequence).
//   * M tiles stacked vertically per CTA step (MT): 1 (small images), 2, or 3 for the unmasked N = 64 layers.
//   * UP = 1 (the first conv of a decoder stage, nets/unet.py:16-18: conv1(cat([skip, up(low)]))): source 1 is the
//     LOW-RESOLUTION tensor [N, H/2, W/2, C1].  Five extra warps (6..10) interpolate its 64-channel blocks (bilinear 2x,
//     align_corners=True, the arithmetic of b2u_bilinear.cuh) straight into the 128B-swizzled A box the tensor core reads,
//     taking the A slots of the channel blocks >= C0 in the same ring the TMA thread fills for the skip tensor: neither the
//     concat nor the upsampled tensor goes through HBM on the way into the conv, and because one box serves all nine
//     taps every up-sampled pixel is interpolated once per tile (plus halo).  Low-resolution rows are fetched one
//     row segment ahead (12 16-byte loads in flight per thread), so their L2 latency hides behind the interpolation of the
//     previous segment.  In training the weight gradient of this conv needs the upsampled tensor as an operand: the
//     warps of N tile 0 also store the box interior to `up_out` (a by-product of the conv, not a separate pass);
//     inference passes up_out = null and the tensor never exists.
#include <atomic>
#include <cstdlib>
#include <mutex>

#include "b2u_internal.h"
#include "b2u_ptx.cuh"
#include "b2u_bilinear.cuh"

namespace b2u {

// Two tile geometries (ConvCfg::kWb x kHb pixels = one M = 128 accumulator tile):
//   plain convs (UP = 0): 16 (w) x 8 (h); one TMA box of (8 MT + 2) x 16 pixels per (channel block, horizontal tap), the
//     three vertical taps re-use it through the descriptor start address (+ r image rows).  Its 2 KB image-row runs
//     suit the HBM-bound launches (masked data gradients, 1x1 head) and four stacked tiles fit for the N = 64 layers;
//   decoder convs (UP = 1): 8 (w) x 16 (h); ONE box of (16 MT + 2) x 10 pixels per channel block serves all nine taps
//     (descriptor start + (r * 10 + s) * 128 B, group stride = one box row), so an interpolated pixel is built once.
// Same-box A/B of the two geometries on the plain convs of the headline step: 22.2-22.3 ms vs 22.6 ms per step in
// favour of 16 x 8 (the N = 64 and masked launches lose 15-25 % with 1 KB runs), so each keeps its own.
constexpr int kTileM = 128;
constexpr int KB = 64;    // channels per K block = one 128-byte swizzle row

struct ConvParams {
  int N, H, W;
  int C0, C1;        // input channels of source 0 / source 1 (C1 == 0: single source)
  int Cout;          // GEMM N extent (multiple of BN)
  int tiles_w, tiles_h;
  int num_m_tiles, num_n_tiles;
  int split_c;       // output channels >= split_c go to the second output tensor map
  int flags;         // bit0 relu, bit1 mask, bit2 classifier head, bit3 the mask is a bit mask (mask_bits)
  float* stat_partial;  // [m tiles][2][Cout] or null: per-tile sums of z and z^2 over the tile's in-image pixels (BatchNorm statistics)
  float* head_out;   // bit2: fp32 NCHW logits [N][head_cls][H][W]
  int head_cls;
  const float* bias; // [Cout] or null (head: [head_cls])
  const float* scale;   // [Cout] or null: per-channel multiplier of the accumulator (folded eval-mode BatchNorm)
  const __nv_bfloat16* mask;  // NHWC [N,H,W,mask_c] or null; keeps y where mask > 0
  int mask_c;
  int* sched;        // dynamic tile scheduler: [0] next tile id, [1] CTAs done (self-resetting); null = static round robin
  const unsigned long long* mask_bits;   // flags bit3: the ReLU mask as one bit per channel, [N,H,W,Cout/64] 64-bit words (bit c%64 of word c/64)
  unsigned long long* bits_out;          // forward + ReLU, nullable: receives (y > 0) in that layout for the backward pass
  const __nv_bfloat16* up_low;  // UP kernels: source 1 = this [N, H/2, W/2, C1] tensor, upsampled 2x on the fly
  __nv_bfloat16* up_out;        // UP kernels, nullable: receives the upsampled tensor [N, H, W, C1] (operand of the weight gradient)
  float up_sh, up_sw;           // (H/2 - 1) / (H - 1), (W/2 - 1) / (W - 1)
};

constexpr int kUpWarps = 5;         // interpolation warps of the UP kernels: 160 threads = 2 row groups x 10 box columns x 8 16-byte chunks

template <int BN, int TAPS, int MT, int RB, int SA, int SB, int MD = 0, int UP = 0>
struct ConvCfg {
  // MD: depth of the cp.async ReLU-mask pipeline (0: mask rows are prefetched into registers one sub-tile ahead)
  // MT: M tiles (8x16 pixel patches, stacked vertically) per CTA step, sharing every B tile
  // RB: vertical taps per B pipeline stage (3: one barrier round trip per 12*MT MMAs, for the small-N tiles)
  static constexpr int kRowBytes = KB * 2;                      // swizzle span (128 B)
  static constexpr int kWb = UP ? 8 : 16;                       // tile width / height in pixels
  static constexpr int kHb = UP ? 16 : 8;
  static constexpr bool kOneBox = UP != 0;                      // one halo box per channel block serves all nine taps
  static constexpr int kPitch = kOneBox ? kWb + 2 : kWb;        // pixels per box row (one box: a halo column each side)
  static constexpr int kBoxRows = TAPS == 9 ? kHb * MT + 2 : kHb * MT;
  static constexpr int kARows = kBoxRows * kPitch;
  static constexpr int kABoxBytes = kARows * kRowBytes;         // bytes one TMA box delivers
  static constexpr int kABytes = (kABoxBytes + 1023) / 1024 * 1024;   // slot size: the swizzle pattern is anchored at 1024 B
  static constexpr int kBTap = BN * kRowBytes;                  // one tap's weight tile
  static constexpr int kBBytes = RB * kBTap;
  static constexpr int kStageBytes = kTileM * 64 * 2;
  static constexpr int kOffA = 0;
  static constexpr int kOffB = kOffA + SA * kABytes;
  static constexpr int kOffStage = kOffB + SB * kBBytes;
  static constexpr int kOffBias = kOffStage + 2 * kStageBytes;
  static constexpr int kOffStat = kOffBias + 2 * 256 * 4;    // [4 row quarters][64 channels][2] fp32 scratch of the BatchNorm-statistics pass
  static constexpr int kOffMask = kOffStat + 4 * 64 * 2 * 4; // MD thread-private mask tiles [128 rows][128 B]
  static constexpr int kOffBar = kOffMask + MD * kTileM * 128;  // (bias of the current N tile is double buffered by tile parity)
  static constexpr int kQ = 4;                                  // depth of the tile-id queue (producer -> MMA / epilogue warps)
  static constexpr int kNumBar = 2 * SA + 2 * SB + 4 + 2 * kQ + (UP ? SA : 0);   // UP: one "slot is yours" barrier per A slot
  static constexpr int kOffTmem = kOffBar + kNumBar * 8;
  static constexpr int kOffTq = kOffTmem + 16;
  static constexpr int kOffRowW = kOffTq + kQ * 4;             // UP: per box row, the two vertical interpolation weights (float2), two tile parities
  static constexpr int kSmemBytes = kOffRowW + (UP ? 2 * kBoxRows * 8 : 0) + 1024;  // + alignment slack
  static constexpr uint32_t kSBO = 8 * kRowBytes;             // B operand: 8-row groups are contiguous
  static constexpr uint32_t kSBO_A = kOneBox ? kPitch * kRowBytes : 8 * kRowBytes;   // A operand: one box: next 8-pixel group = next box row
  static constexpr int kAccCols = MT * BN;                     // accumulator columns per pipeline stage
  static constexpr int kTmemCols = 2 * kAccCols <= 128 ? 128 : (2 * kAccCols <= 256 ? 256 : 512);
  static_assert(BN % 64 == 0 && BN <= 256, "N tile must be 64/128/192/256");
  static_assert(2 * kAccCols <= 512, "TMEM holds 512 columns");
  static_assert(TAPS == 9 || RB == 1, "1x1 convs have a single tap");
  static_assert(kABytes % 1024 == 0 && kBTap % 1024 == 0, "stage buffers must keep 1024B alignment");
  static_assert(kSmemBytes <= 232448, "shared memory budget exceeded");
  static_assert(UP == 0 || (TAPS == 9 && MD == 0), "the interpolating producer exists for the unmasked 3x3 forward tiles");
  static constexpr int kThreads = 192 + (UP ? kUpWarps * 32 : 0);
};

template <int BN, int TAPS, int MT, int RB, int SA, int SB, int MD = 0, int UP = 0>
__global__ void __launch_bounds__(192 + (UP ? kUpWarps * 32 : 0), 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                  const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC0,
                  const __grid_constant__ CUtensorMap tmC1, const ConvParams p) {
  using Cfg = ConvCfg<BN, TAPS, MT, RB, SA, SB, MD, UP>;
  constexpr int S_TAPS = TAPS == 9 ? 3 : 1;
  constexpr int R_TAPS = TAPS == 9 ? 3 : 1;
  constexpr int kWb = Cfg::kWb, kHb = Cfg::kHb;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  const uint32_t sA = smem_base + Cfg::kOffA;
  const uint32_t sB = smem_base + Cfg::kOffB;
  const uint32_t sStage = smem_base + Cfg::kOffStage;
  float* sBias = reinterpret_cast<float*>(smem_gen + Cfg::kOffBias);
  float* sStat = reinterpret_cast<float*>(smem_gen + Cfg::kOffStat);
  const uint32_t bars = smem_base + Cfg::kOffBar;
  auto a_full = [&](int i) { return bars + 8u * i; };
  auto a_empty = [&](int i) { return bars + 8u * (SA + i); };
  auto b_full = [&](int i) { return bars + 8u * (2 * SA + i); };
  auto b_empty = [&](int i) { return bars + 8u * (2 * SA + SB + i); };
  auto t_full = [&](int i) { return bars + 8u * (2 * SA + 2 * SB + i); };
  auto t_empty = [&](int i) { return bars + 8u * (2 * SA + 2 * SB + 2 + i); };
  auto q_full = [&](int i) { return bars + 8u * (2 * SA + 2 * SB + 4 + i); };
  auto q_empty = [&](int i) { return bars + 8u * (2 * SA + 2 * SB + 4 + Cfg::kQ + i); };
  auto u_go = [&](int i) { return bars + 8u * (2 * SA + 2 * SB + 4 + 2 * Cfg::kQ + i); };   // TMA thread -> interpolation warps
  volatile int* tq = reinterpret_cast<volatile int*>(smem_gen + Cfg::kOffTq);
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::kOffTmem);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA0);
    tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmC0);
    tma_prefetch_desc(&tmC1);
    for (int i = 0; i < SA; ++i) { mbar_init(a_full(i), 1); mbar_init(a_empty(i), 1); }
    for (int i = 0; i < SB; ++i) { mbar_init(b_full(i), 1); mbar_init(b_empty(i), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(t_full(i), 1); mbar_init(t_empty(i), 4); }
    for (int i = 0; i < Cfg::kQ; ++i) { mbar_init(q_full(i), 1); mbar_init(q_empty(i), 5 + (UP ? kUpWarps : 0)); }      // readers: MMA thread + 4 epilogue warps (+ interpolation warps)
    if (UP) for (int i = 0; i < SA; ++i) mbar_init(u_go(i), 1);
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

  const int total_tiles = p.num_m_tiles * p.num_n_tiles;
  const int chunks0 = p.C0 / KB;
  const int chunks = (p.C0 + p.C1) / KB;
  const int ctot = p.C0 + p.C1;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      int qs = 0, static_next = blockIdx.x;
      uint32_t qp = 0;
      for (;;) {
        // next tile: one atomic per tile (dynamic) or the round robin (static); published to the consumers through the queue
        int tile;
        if (p.sched != nullptr) tile = atomicAdd(p.sched, 1);
        else { tile = static_next; static_next += gridDim.x; }
        if (tile >= total_tiles) tile = -1;
        mbar_wait(q_empty(qs), qp ^ 1u);
        tq[qs] = tile;
        mbar_arrive(q_full(qs));
        if (++qs == Cfg::kQ) { qs = 0; qp ^= 1u; }
        if (tile < 0) break;
        const int n_tile = tile % p.num_n_tiles;
        int m_tile = tile / p.num_n_tiles;
        const int tw = m_tile % p.tiles_w; m_tile /= p.tiles_w;
        const int th = m_tile % p.tiles_h;
        const int img = m_tile / p.tiles_h;
        const int w0 = tw * kWb, h0 = th * (kHb * MT), n0 = n_tile * BN;
        for (int c = 0; c < chunks; ++c) {
          const CUtensorMap* tm = c < chunks0 ? &tmA0 : &tmA1;
          const int cc = c < chunks0 ? c * KB : c * KB - p.C0;
          if (Cfg::kOneBox) {
            // This thread is the only one that follows the a_empty phases (a parity wait is exact only within one phase of
            // its barrier, and the interpolation warps skip the skip tensor's slots): a free slot of an up-sampled channel
            // block is handed to them through u_go, which by construction never runs more than one phase ahead of them.
            mbar_wait(a_empty(sa), pa ^ 1u);
            if (UP && c >= chunks0) {
              mbar_arrive(u_go(sa));
            } else {
              mbar_expect_tx(a_full(sa), Cfg::kABoxBytes);
              tma_load_4d(sA + sa * Cfg::kABytes, tm, a_full(sa), cc, w0 - 1, h0 - 1, img);
            }
            if (++sa == SA) { sa = 0; pa ^= 1u; }
          }
          for (int s = 0; s < S_TAPS; ++s) {
            if (!Cfg::kOneBox) {
              mbar_wait(a_empty(sa), pa ^ 1u);
              mbar_expect_tx(a_full(sa), Cfg::kABoxBytes);
              if (TAPS == 9) tma_load_4d(sA + sa * Cfg::kABytes, tm, a_full(sa), cc, w0 + s - 1, h0 - 1, img);
              else           tma_load_4d(sA + sa * Cfg::kABytes, tm, a_full(sa), cc, w0, h0, img);
              if (++sa == SA) { sa = 0; pa ^= 1u; }
            }
            for (int rb = 0; rb < R_TAPS / RB; ++rb) {
              mbar_wait(b_empty(sb), pb ^ 1u);
              mbar_expect_tx(b_full(sb), Cfg::kBBytes);
#pragma unroll
              for (int rr = 0; rr < RB; ++rr) {
                const int r = rb * RB + rr;
                tma_load_2d(sB + sb * Cfg::kBBytes + rr * Cfg::kBTap, &tmB, b_full(sb), (r * S_TAPS + s) * ctot + c * KB, n0);
              }
              if (++sb == SB) { sb = 0; pb ^= 1u; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(kTileM, BN, 0, 0);
      // descriptor templates: only the 14-bit start-address field changes per MMA (smem < 256 KB, no carry)
      const uint64_t a_desc0 = umma_smem_desc(sA, 16, Cfg::kSBO_A, 2u);
      const uint64_t b_desc0 = umma_smem_desc(sB, 16, Cfg::kSBO, 2u);
      int sa = 0, sb = 0, as = 0;
      uint32_t pa = 0, pb = 0, pacc = 0;
      int qs = 0;
      uint32_t qp = 0;
      for (;;) {
        mbar_wait(q_full(qs), qp);
        const int tile = tq[qs];
        mbar_arrive(q_empty(qs));
        if (++qs == Cfg::kQ) { qs = 0; qp ^= 1u; }
        if (tile < 0) break;
        mbar_wait(t_empty(as), pacc ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * Cfg::kAccCols);
        uint32_t acc = 0;
        for (int c = 0; c < chunks; ++c) {
          uint64_t a_desc = 0;
          if (Cfg::kOneBox) {
            mbar_wait(a_full(sa), pa);
            tc_fence_after();
            a_desc = a_desc0 + static_cast<uint64_t>((sa * Cfg::kABytes) >> 4);
          }
          for (int s = 0; s < S_TAPS; ++s) {
            if (!Cfg::kOneBox) {
              mbar_wait(a_full(sa), pa);
              tc_fence_after();
              a_desc = a_desc0 + static_cast<uint64_t>((sa * Cfg::kABytes) >> 4);
            }
            // horizontal tap: its own box (start 0), or s pixels into the one halo box
            const int s_off = Cfg::kOneBox ? s : 0;
            for (int rb = 0; rb < R_TAPS / RB; ++rb) {
              mbar_wait(b_full(sb), pb);
              tc_fence_after();
              const uint64_t b_desc = b_desc0 + static_cast<uint64_t>((sb * Cfg::kBBytes) >> 4);
#pragma unroll
              for (int rr = 0; rr < RB; ++rr) {
                const int r = rb * RB + rr;
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
                  for (int k = 0; k < KB / 16; ++k) {
                    // tap row r of stacked tile mt: box pixel (mt * kHb + r) * pitch (+ s), 16 channels further per k
                    const uint64_t ad = a_desc + static_cast<uint64_t>((((mt * kHb + r) * Cfg::kPitch + s_off) * Cfg::kRowBytes + k * 32) >> 4);
                    const uint64_t bd = b_desc + static_cast<uint64_t>((rr * Cfg::kBTap + k * 32) >> 4);
                    tc_mma_bf16(d_tmem + mt * BN, ad, bd, idesc, (k == 0 ? acc : 1u));
                  }
                }
                acc = 1;
              }
              tc_commit(b_empty(sb));
              if (++sb == SB) { sb = 0; pb ^= 1u; }
            }
            if (!Cfg::kOneBox) {
              tc_commit(a_empty(sa));
              if (++sa == SA) { sa = 0; pa ^= 1u; }
            }
          }
          if (Cfg::kOneBox) {
            tc_commit(a_empty(sa));
            if (++sa == SA) { sa = 0; pa ^= 1u; }
          }
        }
        tc_commit(t_full(as));
        if (++as == 2) { as = 0; pacc ^= 1u; }
      }
    }
  } else if (UP && warp >= 6) {
    // ===================== interpolation producers (UP kernels: warps 6..10, 160 threads) =====================
    // thread = (row group g, box column `col` of 10, 16-byte chunk `ch` of the 64-channel block); box pixel q = row * 10 + col
    // lands at byte q * 128 + ((ch ^ (q & 7)) << 4), exactly where a 128B-swizzled TMA box would put it.  A box of
    // 16 MT + 2 rows is built in 2 MT row segments (10 rows, then 8 at a time), even segments by group 0, odd ones by group 1;
    // output rows 2m+1 .. 2m+10 read the low-resolution rows m .. m+5 (b2u_bilinear.cuh), and all 12 16-byte loads of
    // a segment are issued one segment ahead of their use.
    const int ut = threadIdx.x - 192;
    const int ch = ut & 7, col = (ut >> 3) % Cfg::kPitch, grp = (ut >> 3) / Cfg::kPitch;
    const int HL = p.H >> 1, WL = p.W >> 1;
    const int c8 = p.C1 >> 3;                              // 16-byte vectors per low-resolution pixel
    constexpr int R = Cfg::kBoxRows;
    constexpr int SEG_ROWS = 6;
    const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
    uint32_t boxes = 0;                                    // A slots handed out so far (all channel blocks, ring order)
    uint32_t go_phase = 0;                                 // bit i: parity of the next u_go(i) phase to wait for
    int tpar = 0;
    int qs = 0;
    uint32_t qp = 0;
    for (;;) {
      mbar_wait(q_full(qs), qp);
      const int tile = tq[qs];
      __syncwarp();
      if (lane == 0) mbar_arrive(q_empty(qs));
      if (++qs == Cfg::kQ) { qs = 0; qp ^= 1u; }
      if (tile < 0) break;
      const int n_tile = tile % p.num_n_tiles;
      int m_tile = tile / p.num_n_tiles;
      const int tw = m_tile % p.tiles_w; m_tile /= p.tiles_w;
      const int th = m_tile % p.tiles_h;
      const int img = m_tile / p.tiles_h;
      const int wo = tw * kWb - 1 + col, hb = th * (kHb * MT) - 1;       // this thread's image column; image row of box row 0 (odd)
      const bool colok = wo >= 0 && wo < p.W;
      int c0i, c1i; float lw;
      src_index(colok ? wo : 0, p.up_sw, WL, c0i, c1i, lw);
      const float w0l = 1.f - lw;
      const int total = (chunks - chunks0) * MT;           // segments of this thread in the tile
      const uint4* lowimg = reinterpret_cast<const uint4*>(p.up_low) + static_cast<size_t>(img) * HL * WL * c8 + ch;
      const uint4* lowc0 = lowimg + static_cast<size_t>(c0i) * c8;     // this thread's two low-resolution columns
      const uint4* lowc1 = lowimg + static_cast<size_t>(c1i) * c8;
      const size_t lowrow = static_cast<size_t>(WL) * c8, uprow = static_cast<size_t>(p.W) * c8;
      // interior of the box = this tile: by-product store of the up-sampled tensor (N tile 0 only, so once per pixel)
      uint4* upimg = p.up_out != nullptr && n_tile == 0 && colok && col >= 1 && col <= kWb
                         ? reinterpret_cast<uint4*>(p.up_out) + (static_cast<size_t>(img) * p.H * p.W + wo) * c8 + ch : nullptr;
      // vertical weights of the tile's box rows, once per tile (they are the same for every thread and channel block):
      // row r -> weights of low-resolution rows j, j + 1 with j = floor((hb + r - 1) / 2); both zero outside the image
      float2* roww = reinterpret_cast<float2*>(smem_gen + Cfg::kOffRowW) + tpar * R;
      if (ut < R) {
        float wa, wb;
        pair_weights(hb + ut, (hb + ut - 1) >> 1, p.up_sh, HL, p.H, wa, wb);
        roww[ut] = make_float2(wa, wb);
      }
      named_bar_sync(5, kUpWarps * 32);     // (double buffered by tile parity: a fast warp may be one tile ahead of a slow one)
      tpar ^= 1;

      // segment u of this thread -> (up-sampled channel block cu, row segment 2 * (u % MT) + grp)
      auto seg_load = [&](int u, uint4 (&buf)[2 * SEG_ROWS]) {
        const int cu = u / MT, sidx = 2 * (u % MT) + grp;
        const int m = (hb + (sidx == 0 ? 0 : 2 + 8 * sidx) - 1) >> 1;
#pragma unroll
        for (int k = 0; k < SEG_ROWS; ++k) {
          int j = m + k;
          j = j < 0 ? 0 : (j > HL - 1 ? HL - 1 : j);         // rows outside the image carry zero weight
          buf[2 * k] = __ldg(lowc0 + j * lowrow + cu * 8);
          buf[2 * k + 1] = __ldg(lowc1 + j * lowrow + cu * 8);
        }
      };
      auto seg_compute = [&](int u, const uint4 (&buf)[2 * SEG_ROWS]) {
        const int cu = u / MT, sidx = 2 * (u % MT) + grp;
        const uint32_t bidx = boxes + static_cast<uint32_t>(chunks0 + cu);
        const uint32_t slot = bidx % SA;
        if (u % MT == 0) {                                  // the TMA thread saw the slot's previous contents consumed
          mbar_wait(u_go(slot), (go_phase >> slot) & 1u);
          go_phase ^= 1u << slot;
        }
        const int r0 = sidx == 0 ? 0 : 2 + 8 * sidx;
        const uint32_t q0 = static_cast<uint32_t>(r0 * Cfg::kPitch + col);
        const uint32_t box = sA + slot * Cfg::kABytes + q0 * 128;
        uint4* upp = upimg != nullptr ? upimg + (hb + r0) * static_cast<ptrdiff_t>(uprow) + cu * 8 : nullptr;
        float va[8], vb[8];
        hlerp8(buf[0], buf[1], w0l, lw, va);
#pragma unroll
        for (int t = 0; t < 10; ++t) {
          if (t >= 8 && sidx != 0) break;
          if ((t & 1) == 0) {
            if (t > 0) {
#pragma unroll
              for (int k = 0; k < 8; ++k) va[k] = vb[k];
            }
            hlerp8(buf[2 * (t / 2 + 1)], buf[2 * (t / 2 + 1) + 1], w0l, lw, vb);
          }
          const int r = r0 + t, o = hb + r;
          const bool inside = colok && o >= 0 && o < p.H;       // outside the image: the conv's zero padding
          const float2 w2 = roww[r];
          const uint4 v = inside ? vlerp8(va, vb, w2.x, w2.y) : zero4;
          const uint32_t q = q0 + t * Cfg::kPitch;
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(box + t * Cfg::kPitch * 128 + ((ch ^ (q & 7)) << 4)), "r"(v.x), "r"(v.y),
                       "r"(v.z), "r"(v.w) : "memory");
          if (upp != nullptr && inside && r >= 1 && r <= R - 2) upp[t * uprow] = v;
        }
        if (u % MT == MT - 1) {
          fence_proxy_async_smem();          // generic-proxy writes -> visible to the tensor core's async-proxy reads
          named_bar_sync(4, kUpWarps * 32);
          if (ut == 0) mbar_arrive(a_full(slot));
        }
      };

      uint4 bufA[2 * SEG_ROWS], bufB[2 * SEG_ROWS];
      if (total > 0) seg_load(0, bufA);
      for (int u = 0; u < total; u += 2) {
        if (u + 1 < total) seg_load(u + 1, bufB);
        seg_compute(u, bufA);
        if (u + 2 < total) seg_load(u + 2, bufA);
        if (u + 1 < total) seg_compute(u + 1, bufB);
      }
      boxes += static_cast<uint32_t>(chunks);
    }
  } else {
    // ===================== epilogue (4 warps, 128 threads) =====================
    const int ew = warp & 3;  // TMEM sub-partition this warp may read
    const int row = ew * 32 + lane;
    const int ph = row / kWb, pw = row % kWb;
    const bool issuer = (threadIdx.x == 64);
    int as = 0;
    uint32_t pacc = 0;
    uint32_t sbuf = 0;
    uint32_t bpar = 0;
    // ReLU-mask stream for the memory-bound small-N tiles (MD > 0): every thread copies the 128-byte mask row of its
    // pixel with cp.async into a thread-private slot, MD sub-tiles ahead of its use (across tile boundaries), so 16 KB x MD
    // of mask bytes are in flight per SM instead of one register-held row per thread.
    const uint32_t sMask = smem_base + Cfg::kOffMask;
    int pf_tile = blockIdx.x, pf_jj = 0, pf_slot = 0, use_slot = 0;
    auto mask_issue = [&]() {
      if (MD > 0) {
        if (pf_tile < total_tiles) {
          const int n_tile_ = pf_tile % p.num_n_tiles;
          int m_ = pf_tile / p.num_n_tiles;
          const int tw_ = m_ % p.tiles_w; m_ /= p.tiles_w;
          const int th_ = m_ % p.tiles_h;
          const int img_ = m_ / p.tiles_h;
          const int mt_ = pf_jj / (BN / 64), j_ = pf_jj % (BN / 64);
          const int gh_ = th_ * (kHb * MT) + mt_ * kHb + ph, gw_ = tw_ * kWb + pw;
          const bool inb_ = gh_ < p.H && gw_ < p.W;
          const uint4* mrow = reinterpret_cast<const uint4*>(
              p.mask + ((static_cast<size_t>(img_) * p.H + (inb_ ? gh_ : 0)) * p.W + (inb_ ? gw_ : 0)) * p.mask_c + n_tile_ * BN + j_ * 64);
          const uint32_t dst = sMask + pf_slot * (kTileM * 128) + row * 128;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst + ((q ^ (row & 7)) << 4)), "l"(mrow + q),
                         "r"(inb_ ? 16 : 0) : "memory");
          if (++pf_jj == MT * (BN / 64)) { pf_jj = 0; pf_tile += gridDim.x; }
          if (++pf_slot == MD) pf_slot = 0;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");       // always: keeps the wait count uniform at the tail
      }
    };
    if (MD > 0 && (p.flags & 2)) {
#pragma unroll
      for (int i = 0; i < (MD > 0 ? MD : 1); ++i) mask_issue();
    }
    int qs = 0;
    uint32_t qp = 0;
    for (;;) {
      mbar_wait(q_full(qs), qp);
      const int tile = tq[qs];
      __syncwarp();
      if (lane == 0) mbar_arrive(q_empty(qs));
      if (++qs == Cfg::kQ) { qs = 0; qp ^= 1u; }
      if (tile < 0) break;
      const int n_tile = tile % p.num_n_tiles;
      int m_tile = tile / p.num_n_tiles;
      const int tw = m_tile % p.tiles_w; m_tile /= p.tiles_w;
      const int th = m_tile % p.tiles_h;
      const int img = m_tile / p.tiles_h;
      const int w0 = tw * kWb, h0 = th * (kHb * MT), n0 = n_tile * BN;
      const int gw = w0 + pw;

      // ReLU-mask rows are fetched one sub-tile ahead (first one before the accumulator wait) so their latency
      // hides behind the main loop / the previous sub-tile's staging instead of stalling the epilogue
      uint4 mreg[8];
      auto fetch_mask = [&](int jj_) {
        const int mt_ = jj_ / (BN / 64), j_ = jj_ % (BN / 64);
        const int gh_ = h0 + mt_ * kHb + ph;
        const bool inb_ = gh_ < p.H && gw < p.W;
        const uint4* mrow = reinterpret_cast<const uint4*>(
            p.mask + ((static_cast<size_t>(img) * p.H + (inb_ ? gh_ : 0)) * p.W + (inb_ ? gw : 0)) * p.mask_c + n0 + j_ * 64);
#pragma unroll
        for (int q = 0; q < 8; ++q) mreg[q] = inb_ ? __ldg(mrow + q) : make_uint4(0, 0, 0, 0);
      };
      // bit-mask form of the same: 8 bytes per pixel and 64-channel block instead of 128 (ConvParams::mask_bits)
      const int words = p.Cout >> 6;
      unsigned long long mbits = 0ull;
      auto fetch_bits = [&](int jj_) {
        const int mt_ = jj_ / (BN / 64), j_ = jj_ % (BN / 64);
        const int gh_ = h0 + mt_ * kHb + ph;
        mbits = (gh_ < p.H && gw < p.W)
                    ? __ldg(p.mask_bits + ((static_cast<size_t>(img) * p.H + gh_) * p.W + gw) * words + (n0 >> 6) + j_) : 0ull;
      };
      if (MD == 0 && (p.flags & 2)) { if (p.flags & 8) fetch_bits(0); else fetch_mask(0); }
      // this tile's bias slice; the parity double buffer + the barrier keep a fast warp from overwriting values a
      // slow warp of the previous tile still reads
      float* sB = sBias + bpar * 256;
      float* sS = sStat + bpar * 256;      // the statistics scratch doubles as the scale buffer (training vs eval: never both)
      for (int c = threadIdx.x - 64; c < BN; c += 128) {
        // head: column n0 + c is row (n0 + c) % 64 of group (n0 + c) / 64, and the bias [head_cls] is indexed by class
        const int hcol = n0 + c, hcls = (hcol >> 6) * 32 + (hcol & 31);
        sB[c] = !p.bias ? 0.f
                : !(p.flags & 4) ? __ldg(p.bias + n0 + c)
                : ((hcol & 63) < 32 && hcls < p.head_cls) ? __ldg(p.bias + hcls) : 0.f;
        if (p.scale) sS[c] = __ldg(p.scale + n0 + c);
      }
      named_bar_sync(2, 128);
      bpar ^= 1u;

      mbar_wait(t_full(as), pacc);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + static_cast<uint32_t>(as * Cfg::kAccCols);
      float stat_acc[BN / 64];       // thread (c = row & 63, quantity = row >> 6) owns one column sum per 64-channel block
#pragma unroll
      for (int j = 0; j < BN / 64; ++j) stat_acc[j] = 0.f;

#pragma unroll 1
      for (int jj = 0; jj < MT * (BN / 64); ++jj) {
        const int mt = jj / (BN / 64), j = jj % (BN / 64);
        uint32_t v[64];
        tmem_ld_32x32(t_row + mt * BN + j * 64, v);
        tmem_ld_32x32(t_row + mt * BN + j * 64 + 32, v + 32);
        tmem_ld_wait();
        if (jj == MT * (BN / 64) - 1) {
          // all TMEM reads of this accumulator stage are done: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(t_empty(as));
        }
        if (p.flags & 4) {
          // classifier head (nets/unet.py:58,76): each block of 64 accumulator columns is one group [hi(32) | lo(32)] of
          // the two-term bf16 split of the fp32 weights of classes 32g .. 32g + 31, so logits[c] = acc[c] + acc[32 + c] +
          // bias[c] carries them to ~2^-17; written straight to the fp32 NCHW tensor the losses read (a warp covers two
          // 64-byte runs per class).  Groups past the last class (zero-filled rows of a ragged N tile) are skipped.
          const int gh = h0 + mt * kHb + ph;
          const int cls0 = ((n0 + j * 64) >> 6) * 32;
          if (gh < p.H && gw < p.W && cls0 < p.head_cls) {
            const size_t plane = static_cast<size_t>(p.H) * p.W;
            float* o = p.head_out + (static_cast<size_t>(img) * p.head_cls + cls0) * plane + static_cast<size_t>(gh) * p.W + gw;
            const int ncls = p.head_cls - cls0;
#pragma unroll
            for (int c = 0; c < 32; ++c)
              if (c < ncls) o[c * plane] = __uint_as_float(v[c]) + __uint_as_float(v[32 + c]) + sB[j * 64 + c];
          }
          continue;
        }
        const int cbase = n0 + j * 64;
        uint32_t packed[32];
        if (MD == 0 && (p.flags & 8)) {
          // ReLU backward from the bit mask the forward conv left behind: keep column c where bit c of this pixel's word is set
          const uint32_t bw[2] = {static_cast<uint32_t>(mbits), static_cast<uint32_t>(mbits >> 32)};
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            float lo = __uint_as_float(v[2 * e]) + sB[j * 64 + 2 * e];
            float hi = __uint_as_float(v[2 * e + 1]) + sB[j * 64 + 2 * e + 1];
            const uint32_t two = bw[e >> 4] >> ((2 * e) & 31);
            lo = (two & 1u) ? lo : 0.f;
            hi = (two & 2u) ? hi : 0.f;
            packed[e] = pack_bf16x2(lo, hi);
          }
          if (jj + 1 < MT * (BN / 64)) fetch_bits(jj + 1);
        } else if (p.flags & 2) {
          if (MD > 0) {
            asm volatile("cp.async.wait_group %0;" ::"n"(MD > 0 ? MD - 1 : 0) : "memory");
            const uint32_t src = sMask + use_slot * (kTileM * 128) + row * 128;
#pragma unroll
            for (int q = 0; q < 8; ++q)
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(mreg[q].x), "=r"(mreg[q].y), "=r"(mreg[q].z), "=r"(mreg[q].w) : "r"(src + ((q ^ (row & 7)) << 4)));
            if (++use_slot == MD) use_slot = 0;
          }
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const uint32_t mm[4] = {mreg[q].x, mreg[q].y, mreg[q].z, mreg[q].w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float lo = __uint_as_float(v[q * 8 + 2 * e]) + sB[j * 64 + q * 8 + 2 * e];
              float hi = __uint_as_float(v[q * 8 + 2 * e + 1]) + sB[j * 64 + q * 8 + 2 * e + 1];
              lo = bf16_lo(mm[e]) > 0.f ? lo : 0.f;
              hi = bf16_hi(mm[e]) > 0.f ? hi : 0.f;
              packed[q * 4 + e] = pack_bf16x2(lo, hi);
            }
          }
          if (MD > 0) mask_issue();             // refill the slot just consumed (its values now sit in `packed`)
          else if (jj + 1 < MT * (BN / 64)) fetch_mask(jj + 1);
        } else {
          const bool relu = p.flags & 1;
          if (p.scale) {          // y = [relu](acc * s + b'): conv + eval-mode BatchNorm (+ ReLU) in one epilogue
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              float lo = fmaf(__uint_as_float(v[2 * e]), sS[j * 64 + 2 * e], sB[j * 64 + 2 * e]);
              float hi = fmaf(__uint_as_float(v[2 * e + 1]), sS[j * 64 + 2 * e + 1], sB[j * 64 + 2 * e + 1]);
              if (relu) { lo = fmaxf(lo, 0.f); hi = fmaxf(hi, 0.f); }
              packed[e] = pack_bf16x2(lo, hi);
            }
          } else {
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              float lo = __uint_as_float(v[2 * e]) + sB[j * 64 + 2 * e];
              float hi = __uint_as_float(v[2 * e + 1]) + sB[j * 64 + 2 * e + 1];
              if (relu) { lo = fmaxf(lo, 0.f); hi = fmaxf(hi, 0.f); }
              packed[e] = pack_bf16x2(lo, hi);
            }
          }
        }
        if (p.bits_out != nullptr) {
          // (y > 0) of the 64 values this thread just rounded, one bit per channel: the ReLU mask of the backward pass at
          // 1/16 of the bytes of y (a rounded value is positive iff its 15 magnitude bits are not all zero: y >= 0 here)
          uint32_t bw[2] = {0u, 0u};
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const uint32_t t = packed[e] & 0x7FFF7FFFu;
            const uint32_t two = ((t & 0xFFFFu) ? 1u : 0u) | ((t >> 16) ? 2u : 0u);
            bw[e >> 4] |= two << ((2 * e) & 31);
          }
          const int gh = h0 + mt * kHb + ph;
          if (gh < p.H && gw < p.W)
            p.bits_out[((static_cast<size_t>(img) * p.H + gh) * p.W + gw) * words + (n0 >> 6) + j] =
                (static_cast<unsigned long long>(bw[1]) << 32) | bw[0];
        }
        // staging buffer `sbuf` was last read by the TMA store issued two sub-tiles ago
        if (issuer) tma_store_wait_read<1>();
        named_bar_sync(1, 128);
        const uint32_t stage = sStage + sbuf * Cfg::kStageBytes;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const uint32_t off = row * 128 + ((q ^ (row & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stage + off), "r"(packed[q * 4]),
                       "r"(packed[q * 4 + 1]), "r"(packed[q * 4 + 2]), "r"(packed[q * 4 + 3])
                       : "memory");
        }
        fence_proxy_async_smem();
        named_bar_sync(1, 128);
        if (issuer) {
          if (h0 + mt * kHb < p.H) {       // a stacked tile may hang below the image entirely
            if (cbase < p.split_c) tma_store_4d(&tmC0, stage, cbase, w0, h0 + mt * kHb, img);
            else                   tma_store_4d(&tmC1, stage, cbase - p.split_c, w0, h0 + mt * kHb, img);
          }
          tma_store_commit();              // always: the wait_group<1> bookkeeping counts one group per sub-tile
        }
        if (p.stat_partial != nullptr) {
          // BatchNorm statistics of this conv's output, taken from the bf16 tile exactly as it is stored (so they equal a
          // separate pass over z): thread = (channel pair cp, row quarter q) sums its 32 rows of the staged tile (a warp
          // reads one permuted 128-byte row per step: conflict-free), the four quarters meet in a 2 KB scratch, and
          // thread (c, quantity) keeps the running sum of the tile's stacked sub-tiles in a register.
          const int cp = row & 31, q4 = row >> 5;
          float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll 8
          for (int rr = 0; rr < 32; ++rr) {
            const int r = q4 * 32 + rr;
            const bool inimg = (h0 + mt * kHb + r / kWb) < p.H && (w0 + r % kWb) < p.W;
            uint32_t wv;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(wv) : "r"(stage + r * 128 + (((cp >> 2) ^ (r & 7)) << 4) + ((cp & 3) << 2)));
            const float lo = inimg ? bf16_lo(wv) : 0.f, hi = inimg ? bf16_hi(wv) : 0.f;
            s0 += lo; s1 += hi; q0 = fmaf(lo, lo, q0); q1 = fmaf(hi, hi, q1);
          }
          float* sq = sStat + q4 * 128;            // [channel 0..63][2]
          sq[(2 * cp) * 2] = s0; sq[(2 * cp) * 2 + 1] = q0;
          sq[(2 * cp + 1) * 2] = s1; sq[(2 * cp + 1) * 2 + 1] = q1;
          named_bar_sync(3, 128);
          const int c = row & 63, qty = row >> 6;
          const float tsum = sStat[c * 2 + qty] + sStat[128 + c * 2 + qty] + sStat[256 + c * 2 + qty] + sStat[384 + c * 2 + qty];
#pragma unroll
          for (int j2 = 0; j2 < BN / 64; ++j2) if (j2 == j) stat_acc[j2] += tsum;      // static indices keep it in registers
          // the scratch is rewritten only after the two named barriers at the top of the next sub-tile
        }
        sbuf ^= 1u;
      }
      if (p.stat_partial != nullptr) {
        const int c = row & 63, qty = row >> 6;
        float* dst = p.stat_partial + (static_cast<size_t>(tile / p.num_n_tiles) * 2 + qty) * p.Cout + n0 + c;
#pragma unroll
        for (int j = 0; j < BN / 64; ++j) dst[j * 64] = stat_acc[j];
      }
      if (++as == 2) { as = 0; pacc ^= 1u; }
    }
    if (issuer) tma_store_wait_all<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
  if (threadIdx.x == 0 && p.sched != nullptr) {
    // the last CTA to leave re-arms the scheduler slot for its next use (every CTA took its final tile id before this point)
    __threadfence();
    if (atomicAdd(p.sched + 1, 1) == static_cast<int>(gridDim.x) - 1) {
      p.sched[0] = 0;
      p.sched[1] = 0;
      __threadfence();
    }
  }
}

// ----------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------
// Scheduler slots: a ring of self-resetting {next tile, CTAs done} pairs per device; consecutive launches take consecutive
// slots, so kernels that overlap on two streams never share one.  B2U_STATIC_TILES=1 forces the static round robin.
constexpr int kSchedSlots = 256;
static int* sched_slot() {
  static int* base[64] = {nullptr};
  static std::atomic<unsigned> next{0};
  static std::mutex mu;
  static int off = -1;
  if (off < 0) { const char* e = getenv("B2U_STATIC_TILES"); off = (e && e[0] == '1') ? 1 : 0; }
  if (off == 1) return nullptr;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return nullptr;
  if (base[dev] == nullptr) {
    std::lock_guard<std::mutex> lk(mu);
    if (base[dev] == nullptr) {
      int* ptr = nullptr;
      if (cudaMalloc(&ptr, kSchedSlots * 2 * sizeof(int)) != cudaSuccess) return nullptr;
      cudaMemset(ptr, 0, kSchedSlots * 2 * sizeof(int));
      cudaDeviceSynchronize();
      base[dev] = ptr;
    }
  }
  return base[dev] + 2 * (next.fetch_add(1, std::memory_order_relaxed) % kSchedSlots);
}

template <int BN, int TAPS, int MT, int RB, int SA, int SB, int MD = 0, int UP = 0>
static int launch_cfg(const ConvLaunch& a, cudaStream_t st) {
  using Cfg = ConvCfg<BN, TAPS, MT, RB, SA, SB, MD, UP>;
  constexpr int kWb = Cfg::kWb, kHb = Cfg::kHb;
  auto kern = conv_igemm_kernel<BN, TAPS, MT, RB, SA, SB, MD, UP>;
  static bool attr_done[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "cudaFuncSetAttribute(conv): %s", cudaGetErrorString(e));
    attr_done[dev] = true;
  }
  const CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B;
  CUtensorMap tmA0, tmA1, tmB, tmC0, tmC1;
  int rc;
  if ((rc = make_tmap_nhwc(&tmA0, a.x0, a.N, a.H, a.W, a.C0, KB, Cfg::kPitch, Cfg::kBoxRows, swz))) return rc;
  if (a.C1 > 0 && !UP) {
    if ((rc = make_tmap_nhwc(&tmA1, a.x1, a.N, a.H, a.W, a.C1, KB, Cfg::kPitch, Cfg::kBoxRows, swz))) return rc;
  } else {
    tmA1 = tmA0;       // UP: source 1 is read by the interpolation warps, not by TMA
  }
  const int ctot = a.C0 + a.C1;
  if ((rc = make_tmap_2d(&tmB, a.wpacked, (uint64_t)TAPS * ctot, a.Cout, KB, BN, swz))) return rc;
  const int split = (a.y1 != nullptr) ? a.split_c : a.Cout;
  if ((rc = make_tmap_nhwc(&tmC0, a.y0, a.N, a.H, a.W, split, 64, kWb, kHb, swz))) return rc;
  if (a.y1 != nullptr) {
    if ((rc = make_tmap_nhwc(&tmC1, a.y1, a.N, a.H, a.W, a.Cout - split, 64, kWb, kHb, swz))) return rc;
  } else {
    tmC1 = tmC0;
  }
  ConvParams p;
  p.N = a.N; p.H = a.H; p.W = a.W; p.C0 = a.C0; p.C1 = a.C1; p.Cout = a.Cout;
  p.tiles_w = (a.W + kWb - 1) / kWb;
  p.tiles_h = (a.H + kHb * MT - 1) / (kHb * MT);
  p.num_m_tiles = a.N * p.tiles_h * p.tiles_w;
  p.num_n_tiles = (a.Cout + BN - 1) / BN;     // ragged only in head mode (the weight rows past Cout load as zeros)
  p.split_c = split;
  p.flags = a.flags;
  p.stat_partial = a.stat_partial;
  p.head_out = a.head_out;
  p.head_cls = a.head_cls;
  p.bias = a.bias;
  p.scale = a.scale;
  p.mask = a.mask;
  p.mask_c = a.mask_c;
  p.mask_bits = a.mask_bits;
  p.bits_out = a.bits_out;
  p.sched = MD > 0 ? nullptr : sched_slot();      // the mask-stream variants prefetch across tile boundaries: static order
  p.up_low = UP ? static_cast<const __nv_bfloat16*>(a.up_low) : nullptr;
  p.up_out = UP ? static_cast<__nv_bfloat16*>(a.up_out) : nullptr;
  // the scale factors of b2u_upsample2x_fwd (ATen's align_corners=True ratio for a 2x enlargement)
  p.up_sh = a.H > 1 ? static_cast<float>(a.H / 2 - 1) / static_cast<float>(a.H - 1) : 0.f;
  p.up_sw = a.W > 1 ? static_cast<float>(a.W / 2 - 1) / static_cast<float>(a.W - 1) : 0.f;
  const int total = p.num_m_tiles * p.num_n_tiles;
  const int grid = total < num_sms() ? total : num_sms();
  kern<<<grid, Cfg::kThreads, Cfg::kSmemBytes, st>>>(tmA0, tmA1, tmB, tmC0, tmC1, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "conv_igemm launch: %s", cudaGetErrorString(e));
  note_launch();
  return 0;
}

// number of M tiles launch_conv will use for this problem = rows of ConvLaunch::stat_partial
// M tiles stacked vertically per CTA step: the single rule both the launcher and conv_m_tiles follow.
//   plain 3x3 (16 x 8 tiles): N tile 128 / 64 stack two when the image is taller than one tile (halves the weight traffic
//        per pixel); the unmasked N = 64 layers, bound by shared-memory operand traffic (DESIGN.md), stack four from 32 rows on
//   decoder 3x3 (8 x 16 tiles): the same with three instead of four (two 83 KB boxes do not fit), from 48 rows on
//   1x1: N tile 64 stacks two
// tile_flags bit 0 forces one tile, bit 1 caps the stack at two.
int stacked_tiles(int bn, int taps, int H, int tile_flags, bool masked, bool decoder) {
  if (taps != 9) return bn == 64 ? 2 : 1;
  const int hb = decoder ? 16 : 8;
  const bool tall = H > hb && !(tile_flags & 1);
  if (!tall || (bn != 128 && bn != 64)) return 1;
  if (bn == 64 && !masked && !(tile_flags & 2) && H >= (decoder ? 3 : 4) * hb) return decoder ? 3 : 4;
  return 2;
}

// number of M tiles launch_conv will use for this problem = rows of ConvLaunch::stat_partial (forward launches: unmasked);
// bit 18 of bn_override: the decoder conv's tiles (b2u_decoder_conv_fprop)
int conv_m_tiles(int N, int H, int W, int Cout, int taps, int bn_override) {
  int bn = bn_override & 0xffff;
  if (!bn) bn = Cout % 256 == 0 ? 256 : (Cout % 192 == 0 ? 192 : (Cout % 128 == 0 ? 128 : 64));
  const bool decoder = ((bn_override >> 18) & 1) && taps == 9;
  const int mt = stacked_tiles(bn, taps, H, (bn_override >> 16) & 3, false, decoder);
  const int hb = decoder ? 16 : 8, wb = decoder ? 8 : 16;
  return N * ((H + hb * mt - 1) / (hb * mt)) * ((W + wb - 1) / wb);
}

int launch_conv(const ConvLaunch& a, cudaStream_t st) {
  const int ctot = a.C0 + a.C1;
  if (a.N <= 0 || a.H <= 0 || a.W <= 0) return set_error(B2U_ERR_SHAPE, "conv: empty tensor");
  if (a.taps != 9 && a.taps != 1) return set_error(B2U_ERR_SHAPE, "conv: taps must be 9 or 1");
  if (a.Cout <= 0) return set_error(B2U_ERR_SHAPE, "conv: Cout %d must be positive", a.Cout);
  if (a.Cout % 64 != 0) return set_error(B2U_ERR_SHAPE, "conv: Cout %d must be a multiple of 64", a.Cout);
  if ((a.flags & 8) && (!(a.flags & 2) || a.mask_bits == nullptr || a.y1 != nullptr))
    return set_error(B2U_ERR_ARG, "conv: the bit-mask flag needs mask_bits and a single output");
  if (a.bits_out != nullptr && (!(a.flags & 1) || (a.flags & 6) || a.y1 != nullptr || a.scale != nullptr))
    return set_error(B2U_ERR_ARG, "conv: bits_out is written by a forward conv + ReLU with one output");
  if ((a.flags & 2) && !(a.flags & 8) && (a.mask == nullptr || a.mask_c % 8 != 0 || a.mask_c < a.Cout))
    return set_error(B2U_ERR_SHAPE, "conv: mask flag needs a mask tensor with >= Cout channels, %% 8 == 0");
  if (ctot <= 0 || a.C0 % 64 != 0 || a.C1 % 64 != 0)
    return set_error(B2U_ERR_SHAPE, "conv: input channels (%d,%d) must be multiples of 64", a.C0, a.C1);
  if (a.y1 != nullptr && (a.split_c <= 0 || a.split_c >= a.Cout || a.split_c % 64 != 0))
    return set_error(B2U_ERR_SHAPE, "conv: split_c %d must be a multiple of 64 inside (0,Cout)", a.split_c);
  if (a.scale && (a.stat_partial || (a.flags & 6)))
    return set_error(B2U_ERR_ARG, "conv: a per-channel scale excludes the statistics, mask and head epilogues");
  if ((a.flags & 4) && (a.head_out == nullptr || a.head_cls < 1 || a.head_cls > 255 || a.Cout != 64 * ((a.head_cls + 31) / 32) ||
                        a.y1 != nullptr || a.bn_override))
    return set_error(B2U_ERR_SHAPE, "conv: head mode needs 1..255 classes, Cout == 64 * ceil(classes / 32) and an fp32 output");
  int bn = 0;
  if (a.flags & 4) {
    // head: the widest N tile (one pass over the 64-channel input per 4 groups); a ragged last tile runs on zero rows
    bn = a.Cout >= 256 ? 256 : a.Cout;
  } else if (a.bn_override) {
    if (a.Cout % a.bn_override != 0) return set_error(B2U_ERR_SHAPE, "conv: bn_override does not divide Cout");
    bn = a.bn_override;
  } else if (a.Cout % 256 == 0) bn = 256;
  else if (a.Cout % 192 == 0) bn = 192;
  else if (a.Cout % 128 == 0) bn = 128;
  else bn = 64;

  // a bit mask costs 8 bytes per pixel and block: those launches tile like unmasked ones (no cp.async mask stream)
  const bool bf16_mask = (a.flags & 2) && !(a.flags & 8);
  const int mt = stacked_tiles(bn, a.taps, a.H, a.tile_flags, bf16_mask, a.up_low != nullptr);
  if (a.up_low != nullptr) {
    // decoder conv over [skip, upsample2x(low)]: 8 x 16 tiles, one halo box per channel block, interpolation warps
    if (a.taps != 9 || a.C1 <= 0 || (a.H & 1) || (a.W & 1) || (a.flags & 6) || a.y1 != nullptr)
      return set_error(B2U_ERR_SHAPE, "decoder conv: needs a 3x3 forward conv over even H, W with an up-sampled source");
    switch (bn) {
      case 256: return launch_cfg<256, 9, 1, 1, 2, 4, 0, 1>(a, st);
      case 192: return launch_cfg<192, 9, 1, 1, 2, 5, 0, 1>(a, st);
      case 128: return mt == 2 ? launch_cfg<128, 9, 2, 3, 2, 2, 0, 1>(a, st) : launch_cfg<128, 9, 1, 3, 3, 2, 0, 1>(a, st);
      case 64:
        if (mt == 3) return launch_cfg<64, 9, 3, 3, 2, 2, 0, 1>(a, st);
        return mt == 2 ? launch_cfg<64, 9, 2, 3, 2, 3, 0, 1>(a, st) : launch_cfg<64, 9, 1, 3, 3, 4, 0, 1>(a, st);
    }
    return set_error(B2U_ERR_SHAPE, "conv: unsupported N tile %d", bn);
  }
  if (a.taps == 9) {
    switch (bn) {
      case 256: return launch_cfg<256, 9, 1, 1, 3, 4>(a, st);
      case 192: return launch_cfg<192, 9, 1, 1, 3, 5>(a, st);
      case 128: return mt == 2 ? launch_cfg<128, 9, 2, 3, 2, 2>(a, st) : launch_cfg<128, 9, 1, 3, 3, 2>(a, st);
      case 64:
        // masked (dgrad + ReLU) Cin-side-64 layers are HBM-bound: the mask rows go through the cp.async stream
        // unmasked N = 64 tiles are bound by shared-memory operand traffic (DESIGN.md): four stacked M tiles per CTA step --
        // the weights of a step serve 512 pixels and the A box carries 2 halo rows per 32 instead of per 16, two pipeline
        // stages instead of three, all 512 TMEM columns -- measured 0.344 -> 0.309 ms (64->64) and 0.954 -> 0.879 ms
        // (64+128->64) at 16x512x512, bit-identical results (scripts/tile_variants_bench.py).  The masked variant keeps two
        // tiles: its cp.async mask stream does not fit next to the larger A stages and register prefetch is slower
        // (0.443 vs 0.415 ms).  tile_flags bit 1 forces the two-tile kernel (tests).
        if (mt == 4) return launch_cfg<64, 9, 4, 3, 2, 2>(a, st);
        if (mt == 2 && bf16_mask) return launch_cfg<64, 9, 2, 3, 3, 2, 2>(a, st);
        return mt == 2 ? launch_cfg<64, 9, 2, 3, 3, 3>(a, st) : launch_cfg<64, 9, 1, 3, 4, 4>(a, st);
    }
  } else {
    switch (bn) {
      case 256: return launch_cfg<256, 1, 1, 1, 3, 3>(a, st);
      case 192: return launch_cfg<192, 1, 1, 1, 4, 4>(a, st);
      case 128: return launch_cfg<128, 1, 1, 1, 4, 4>(a, st);
      case 64:  return bf16_mask ? launch_cfg<64, 1, 2, 1, 3, 4, 3>(a, st) : launch_cfg<64, 1, 2, 1, 3, 4>(a, st);
    }
  }
  return set_error(B2U_ERR_SHAPE, "conv: unsupported N tile %d", bn);
}

}  // namespace b2u

// ----------------------------------------------------------------------------
// C ABI (include/b2u.h)
// ----------------------------------------------------------------------------
extern "C" {

int b2u_conv_fprop(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* bias, void* y, int N,
                   int H, int W, int Cout, int taps, int relu, int bn_override, void* stream) {
  b2u::ConvLaunch a;
  a.x0 = x0; a.C0 = C0; a.x1 = x1; a.C1 = x1 ? C1 : 0;
  a.wpacked = wf; a.bias = bias; a.y0 = y;
  a.N = N; a.H = H; a.W = W; a.Cout = Cout; a.taps = taps;
  a.flags = relu ? 1 : 0;
  a.bn_override = bn_override & 0xffff;    // bits 0..15: N tile override; bit 16: one M tile per CTA step
  a.tile_flags = bn_override >> 16;
  return b2u::launch_conv(a, static_cast<cudaStream_t>(stream));
}

// b2u_conv_fprop that also emits the BatchNorm statistics of its output: stat_partial [b2u_conv_stat_rows(...)][2][Cout]
// fp32 receives, per M tile, the sums of z and z^2 over the tile's in-image pixels, taken from the bf16 values as stored.
int b2u_conv_stat_rows(int N, int H, int W, int Cout, int taps, int bn_override) {
  if (N <= 0 || H <= 0 || W <= 0 || Cout <= 0) return 0;
  return b2u::conv_m_tiles(N, H, W, Cout, taps, bn_override);
}

int b2u_conv_fprop_stats(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* bias, void* y, int N,
                         int H, int W, int Cout, int taps, int relu, int bn_override, float* stat_partial, int stat_rows,
                         void* stream) {
  if (stat_partial == nullptr || stat_rows < b2u::conv_m_tiles(N, H, W, Cout, taps, bn_override))
    return b2u::set_error(B2U_ERR_ARG, "conv_fprop_stats: statistics buffer too small");
  b2u::ConvLaunch a;
  a.x0 = x0; a.C0 = C0; a.x1 = x1; a.C1 = x1 ? C1 : 0;
  a.wpacked = wf; a.bias = bias; a.y0 = y;
  a.N = N; a.H = H; a.W = W; a.Cout = Cout; a.taps = taps;
  a.flags = relu ? 1 : 0;
  a.bn_override = bn_override & 0xffff;
  a.tile_flags = bn_override >> 16;
  a.stat_partial = stat_partial;
  return b2u::launch_conv(a, static_cast<cudaStream_t>(stream));
}

// y = [relu](conv(x) * scale[c] + bias[c]): a conv followed by eval-mode nn.BatchNorm2d (+ReLU) in one kernel; scale/bias
// come from b2u_bn_fold (scale = gamma / sqrt(rv + eps), bias = (conv_bias - rm) * scale + beta).
int b2u_conv_fprop_scaled(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* scale, const float* bias,
                          void* y, int N, int H, int W, int Cout, int taps, int relu, int bn_override, void* stream) {
  if (!scale) return b2u::set_error(B2U_ERR_ARG, "conv_fprop_scaled: scale vector missing");
  b2u::ConvLaunch a;
  a.x0 = x0; a.C0 = C0; a.x1 = x1; a.C1 = x1 ? C1 : 0;
  a.wpacked = wf; a.bias = bias; a.scale = scale; a.y0 = y;
  a.N = N; a.H = H; a.W = W; a.Cout = Cout; a.taps = taps;
  a.flags = relu ? 1 : 0;
  a.bn_override = bn_override & 0xffff;
  a.tile_flags = bn_override >> 16;
  return b2u::launch_conv(a, static_cast<cudaStream_t>(stream));
}

// First conv of a decoder stage (nets/unet.py:16-18: conv1(cat([skip, up(low)])) with up = nn.UpsamplingBilinear2d(2)):
// `low` is the LOW-RESOLUTION tensor [N, H/2, W/2, C1]; it is interpolated inside the kernel, on the way into the
// A-operand stage, so neither the concat nor the up-sampled tensor is read from HBM.  up_out (nullable) receives the
// up-sampled tensor [N, H, W, C1] as a by-product (training: operand of this conv's weight gradient).
// scale (nullable): folded eval-mode BatchNorm as in b2u_conv_fprop_scaled; stat_partial (nullable): as in b2u_conv_fprop_stats.
int b2u_decoder_conv_fprop(const void* skip, int C0, const void* low, int C1, const void* wf, const float* scale,
                           const float* bias, void* y, void* up_out, int N, int H, int W, int Cout, int relu, int bn_override,
                           float* stat_partial, int stat_rows, void* stream) {
  if (skip == nullptr || low == nullptr) return b2u::set_error(B2U_ERR_ARG, "decoder_conv_fprop: skip and low tensors are required");
  if (stat_partial != nullptr && stat_rows < b2u::conv_m_tiles(N, H, W, Cout, 9, bn_override | (1 << 18)))
    return b2u::set_error(B2U_ERR_ARG, "decoder_conv_fprop: statistics buffer too small (b2u_conv_stat_rows with bit 18 of bn_override)");
  b2u::ConvLaunch a;
  a.x0 = skip; a.C0 = C0; a.x1 = nullptr; a.C1 = C1;
  a.up_low = low; a.up_out = up_out;
  a.wpacked = wf; a.bias = bias; a.scale = scale; a.y0 = y;
  a.N = N; a.H = H; a.W = W; a.Cout = Cout; a.taps = 9;
  a.flags = relu ? 1 : 0;
  a.bn_override = bn_override & 0xffff;
  a.tile_flags = (bn_override >> 16) & 3;
  a.stat_partial = stat_partial;
  return b2u::launch_conv(a, static_cast<cudaStream_t>(stream));
}

// dx = conv(dz, flipped/transposed weights); channels [0,C0) -> dx0, [C0,C0+C1) -> dx1 (optional).
// `mask` (NHWC bf16, C0 channels, only when dx1 == NULL): dx0 is zeroed where mask <= 0 (ReLU backward).
int b2u_conv_dgrad(const void* dz, int Cz, const void* wd, void* dx0, int C0, void* dx1, int C1, const void* mask,
                   int N, int H, int W, int taps, int bn_override, void* stream) {
  b2u::ConvLaunch a;
  a.x0 = dz; a.C0 = Cz;
  a.wpacked = wd; a.bias = nullptr;
  a.y0 = dx0; a.y1 = dx1; a.split_c = C0;
  a.N = N; a.H = H; a.W = W; a.Cout = C0 + (dx1 ? C1 : 0); a.taps = taps;
  a.flags = 0;
  if (mask) {
    if (dx1) return b2u::set_error(B2U_ERR_ARG, "dgrad: mask is only supported with a single output");
    a.flags = 2; a.mask = static_cast<const __nv_bfloat16*>(mask); a.mask_c = C0;
  }
  a.bn_override = bn_override & 0xffff;
  a.tile_flags = bn_override >> 16;
  return b2u::launch_conv(a, static_cast<cudaStream_t>(stream));
}

// b2u_conv_dgrad that also leaves the per-tile column sums of what it stores (after the ReLU mask) in stat_partial
// [b2u_conv_dgrad_stat_rows(...)][2][C0 + C1]: dx is the pre-activation gradient of the layer below, so its column sums ARE
// that layer's bias gradient (b2u_bias_from_stats) and the separate pass over dz (b2u_bias_grad) disappears.
int b2u_conv_dgrad_stat_rows(int N, int H, int W, int Ctot, int taps, int bn_override, int masked) {
  if (N <= 0 || H <= 0 || W <= 0 || Ctot <= 0) return 0;
  int bn = bn_override & 0xffff;
  if (!bn) bn = Ctot % 256 == 0 ? 256 : (Ctot % 192 == 0 ? 192 : (Ctot % 128 == 0 ? 128 : 64));
  const int mt = b2u::stacked_tiles(bn, taps, H, (bn_override >> 16) & 3, masked != 0, false);
  return N * ((H + 8 * mt - 1) / (8 * mt)) * ((W + 15) / 16);
}

int b2u_conv_dgrad_stats(const void* dz, int Cz, const void* wd, void* dx0, int C0, void* dx1, int C1, const void* mask,
                         int N, int H, int W, int taps, int bn_override, float* stat_partial, int stat_rows, void* stream) {
  const int ctot = C0 + (dx1 ? C1 : 0);
  if (stat_partial == nullptr || stat_rows < b2u_conv_dgrad_stat_rows(N, H, W, ctot, taps, bn_override, mask != nullptr))
    return b2u::set_error(B2U_ERR_ARG, "conv_dgrad_stats: statistics buffer too small");
  b2u::ConvLaunch a;
  a.x0 = dz; a.C0 = Cz;
  a.wpacked = wd; a.bias = nullptr;
  a.y0 = dx0; a.y1 = dx1; a.split_c = C0;
  a.N = N; a.H = H; a.W = W; a.Cout = ctot; a.taps = taps;
  a.flags = 0;
  if (mask) {
    if (dx1) return b2u::set_error(B2U_ERR_ARG, "dgrad: mask is only supported with a single output");
    a.flags = 2; a.mask = static_cast<const __nv_bfloat16*>(mask); a.mask_c = C0;
  }
  a.bn_override = bn_override & 0xffff;
  a.tile_flags = (bn_override >> 16) & 3;
  a.stat_partial = stat_partial;
  return b2u::launch_conv(a, static_cast<cudaStream_t>(stream));
}

// Forward conv + bias + ReLU that also leaves the ReLU decisions behind as a BIT mask: bits_out [N,H,W,Cout/64] 64-bit words,
// bit c % 64 of word c / 64 = (y[n,h,w,c] > 0).  The backward pass then reads 8 bytes per pixel and 64-channel block where
// it would re-read 128 bytes of y (b2u_conv_dgrad_bits).  low != NULL (and x1 == NULL): the decoder conv of
// b2u_decoder_conv_fprop (source 1 = upsample2x(low), up_out = its by-product copy).
int b2u_conv_fprop_relu_bits(const void* x0, int C0, const void* x1, int C1, const void* low, const void* wf, const float* bias,
                             void* y, void* up_out, unsigned long long* bits_out, int N, int H, int W, int Cout, int taps,
                             int bn_override, void* stream) {
  if (bits_out == nullptr) return b2u::set_error(B2U_ERR_ARG, "conv_fprop_relu_bits: bits_out is required");
  if (low != nullptr && x1 != nullptr) return b2u::set_error(B2U_ERR_ARG, "conv_fprop_relu_bits: give x1 or low, not both");
  b2u::ConvLaunch a;
  a.x0 = x0; a.C0 = C0; a.x1 = x1; a.C1 = (x1 || low) ? C1 : 0;
  a.up_low = low; a.up_out = low ? up_out : nullptr;
  a.wpacked = wf; a.bias = bias; a.y0 = y; a.bits_out = bits_out;
  a.N = N; a.H = H; a.W = W; a.Cout = Cout; a.taps = taps;
  a.flags = 1;
  a.bn_override = bn_override & 0xffff;
  a.tile_flags = (bn_override >> 16) & 3;
  return b2u::launch_conv(a, static_cast<cudaStream_t>(stream));
}

// b2u_conv_dgrad (single output) with the ReLU mask given as the bit mask of b2u_conv_fprop_relu_bits: dx0 = 0 where the
// bit is clear.  stat_partial (nullable): per-tile column sums as in b2u_conv_dgrad_stats, rows =
// b2u_conv_dgrad_stat_rows(..., masked = 0) -- a bit-masked launch tiles like an unmasked one.
int b2u_conv_dgrad_bits(const void* dz, int Cz, const void* wd, void* dx0, int C0, const unsigned long long* mask_bits,
                        int N, int H, int W, int taps, int bn_override, float* stat_partial, int stat_rows, void* stream) {
  if (mask_bits == nullptr) return b2u::set_error(B2U_ERR_ARG, "conv_dgrad_bits: mask_bits is required");
  if (stat_partial != nullptr && stat_rows < b2u_conv_dgrad_stat_rows(N, H, W, C0, taps, bn_override, 0))
    return b2u::set_error(B2U_ERR_ARG, "conv_dgrad_bits: statistics buffer too small");
  b2u::ConvLaunch a;
  a.x0 = dz; a.C0 = Cz;
  a.wpacked = wd; a.bias = nullptr;
  a.y0 = dx0; a.split_c = C0;
  a.N = N; a.H = H; a.W = W; a.Cout = C0; a.taps = taps;
  a.flags = 2 | 8; a.mask_bits = mask_bits;
  a.bn_override = bn_override & 0xffff;
  a.tile_flags = (bn_override >> 16) & 3;
  a.stat_partial = stat_partial;
  return b2u::launch_conv(a, static_cast<cudaStream_t>(stream));
}

// Classifier head on the tensor cores: logits[n][c][h][w] = sum_k x[n][h][w][k] W[c][k] + b[c], fp32 NCHW.
// wf: bf16 [64 G][64] from b2u_pack_head_fprop, G = ceil(ncls / 32) groups (in group g, rows [64g, 64g + 32) = bf16(W) and
// rows [64g + 32, 64g + 64) = bf16(W - bf16(W)) of classes 32g..); bias: [ncls].
int b2u_head_fwd_tc(const void* x, const void* wf, const float* bias, float* logits, int N, int H, int W, int ncls,
                    void* stream) {
  if (ncls < 1 || ncls > 255) return b2u::set_error(B2U_ERR_SHAPE, "head_fwd_tc: 1 <= classes <= 255 (got %d)", ncls);
  b2u::ConvLaunch a;
  a.x0 = x; a.C0 = 64;
  a.wpacked = wf; a.bias = bias;
  a.y0 = const_cast<void*>(x);          // never written: the head epilogue bypasses the NHWC store path
  a.N = N; a.H = H; a.W = W; a.Cout = 64 * ((ncls + 31) / 32); a.taps = 1;
  a.flags = 4; a.head_out = logits; a.head_cls = ncls;
  return b2u::launch_conv(a, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
