// hist.cu -- fast_hist: the n x n confusion matrix of get_miou / compute_mIoU (utils/utils_metrics.py:34-43).
//
//   k = (a >= 0) & (a < n);  hist = bincount(n * a[k] + b[k], minlength = n*n).reshape(n, n)
//
// Integer work, bit-exact.  HBM-bound: 2 bytes per pixel (uint8 ground truth + uint8 prediction), read as
// 16-byte vectors.  Each warp owns a private shared-memory histogram (no inter-warp contention); lanes that hit
// the same bin in one step are combined with __match_any_sync so the shared atomic count stays low for the
// few-class case; per-block histograms are flushed with 64-bit global atomics (integer adds: order-free, exact).
// Bins >= n*n (possible when b >= n, where numpy's reshape would raise) are counted in hist[n*n] so the host
// wrapper can raise the same error.
#include <cstdlib>

#include "b2u_internal.h"
#include "b2u_ptx.cuh"

namespace b2u {

constexpr int kHistWarps = 8;

template <typename T, int VEC>
__global__ void __launch_bounds__(kHistWarps * 32)
fast_hist_kernel(const T* __restrict__ a, const T* __restrict__ b, long long len, int n, unsigned long long* __restrict__ hist) {
  extern __shared__ unsigned int sh[];   // [warps][nbins + 1]
  const int nbins = n * n;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned int* mine = sh + warp * (nbins + 1);
  for (int i = threadIdx.x; i < kHistWarps * (nbins + 1); i += blockDim.x) sh[i] = 0;
  __syncthreads();

  auto count = [&](long long av, long long bv, bool live) {
    int bin = -1;
    if (live && av >= 0 && av < n) {
      const long long bb = static_cast<long long>(n) * av + bv;
      bin = (bb >= 0 && bb < nbins) ? static_cast<int>(bb) : nbins;   // nbins = overflow slot
    }
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && lane == (__ffs(peers) - 1)) atomicAdd(&mine[bin], __popc(peers));
  };

  const long long nvec = len / VEC;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < ((nvec + 31) / 32) * 32; i += stride) {
    const bool live = i < nvec;
    T av[VEC], bv[VEC];
    if (live) {
      if (sizeof(T) * VEC == 16) {
        *reinterpret_cast<uint4*>(av) = __ldg(reinterpret_cast<const uint4*>(a) + i);
        *reinterpret_cast<uint4*>(bv) = __ldg(reinterpret_cast<const uint4*>(b) + i);
      } else {
#pragma unroll
        for (int e = 0; e < VEC; ++e) { av[e] = a[i * VEC + e]; bv[e] = b[i * VEC + e]; }
      }
    }
#pragma unroll
    for (int e = 0; e < VEC; ++e) count(live ? static_cast<long long>(av[e]) : 0, live ? static_cast<long long>(bv[e]) : 0, live);
  }
  // tail (len % VEC elements), handled by block 0 warp 0
  if (blockIdx.x == 0 && warp == 0) {
    const long long t0 = nvec * VEC;
    for (long long base = t0; base < len; base += 32) {
      const long long i = base + lane;
      const bool live = i < len;
      count(live ? static_cast<long long>(a[i]) : 0, live ? static_cast<long long>(b[i]) : 0, live);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i <= nbins; i += blockDim.x) {
    unsigned long long s = 0;
    for (int w = 0; w < kHistWarps; ++w) s += sh[w * (nbins + 1) + i];
    if (s) atomicAdd(&hist[i], s);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Fast paths for uint8 masks (the get_miou case).  Shared-memory atomics top out near 0.5 pixel/clock/SM, ~5 % of what
// HBM delivers (11.5 pixel/clock/SM at 2 B/pixel), so the hot variants count without atomics:
//
//  * n*n <= 32 bins ("vote"): per 32 pixels one __ballot_sync per bin; popcounts accumulate in registers.
//  * otherwise ("private"): every lane owns a byte counter per bin, laid out [bin][lane] in shared memory, so an
//    increment is a plain LDS.U8 / STS.U8 on an address no other lane ever touches; byte counters are folded into
//    per-warp 32-bit sums before they can overflow (every 240 pixels per lane).
// Both finish with per-block 64-bit global atomics (integer adds: exact, order-free).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kVoteMaxBins = 32;      // (historical name) largest n*n handled by the register-counter kernel

// n*n <= 32 bins: every lane keeps all its counters in registers, packed as 8-bit fields of NW 64-bit words
// (bin k -> word k/8, byte k%8), so counting a pixel is one shift and one 64-bit add on a word selected by predicate.
// Fields are widened into 32-bit registers every 240 pixels (before a byte can wrap).  Slot nbins counts out-of-range
// bins; ignored pixels add zero.
struct HistItem;
template <int NW>      // 64-bit words: (n*n + 1 + 7) / 8 <= NW
__global__ void __launch_bounds__(256)
fast_hist_packed_batch_kernel(const HistItem* __restrict__ items, int count, long long total_chunks, int n,
                              unsigned long long* __restrict__ hist);

template <int NW>      // 64-bit words: (n*n + 1 + 7) / 8 <= NW
__global__ void __launch_bounds__(256)
fast_hist_packed_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, long long nvec, int n,
                        unsigned long long* __restrict__ hist) {
  const int nbins = n * n;
  unsigned long long pk[NW];
  unsigned int wide[NW * 8];
#pragma unroll
  for (int i = 0; i < NW; ++i) pk[i] = 0ull;
#pragma unroll
  for (int i = 0; i < NW * 8; ++i) wide[i] = 0u;
  auto widen = [&]() {
#pragma unroll
    for (int i = 0; i < NW; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) wide[i * 8 + k] += static_cast<unsigned int>(pk[i] >> (8 * k)) & 0xffu;
      pk[i] = 0ull;
    }
  };
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  int since = 0;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    const uint4 va = __ldg(a + i), vb = __ldg(b + i);
    const unsigned wa[4] = {va.x, va.y, va.z, va.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
    for (int wsel = 0; wsel < 4; ++wsel) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const unsigned av = (wa[wsel] >> (8 * k)) & 0xffu, bv = (wb[wsel] >> (8 * k)) & 0xffu;
        unsigned bin = n * av + bv;
        if (bin > static_cast<unsigned>(nbins)) bin = nbins;                   // overflow slot
        const unsigned long long inc = av < static_cast<unsigned>(n) ? 1ull << (8 * (bin & 7u)) : 0ull;
        const unsigned word = bin >> 3;
#pragma unroll
        for (int q = 0; q < NW; ++q) pk[q] += (word == static_cast<unsigned>(q)) ? inc : 0ull;
      }
    }
    since += 16;
    if (since >= 240) { widen(); since = 0; }
  }
  widen();
  // lanes -> warp -> block -> global
  __shared__ unsigned int sblk[NW * 8];
  if (threadIdx.x < NW * 8) sblk[threadIdx.x] = 0;
  __syncthreads();
#pragma unroll
  for (int v = 0; v < NW * 8; ++v) {
    const unsigned t = __reduce_add_sync(0xffffffffu, wide[v]);
    if ((threadIdx.x & 31) == (v & 31) && t) atomicAdd(&sblk[v], t);
  }
  __syncthreads();
  if (threadIdx.x <= nbins && sblk[threadIdx.x]) atomicAdd(&hist[threadIdx.x], static_cast<unsigned long long>(sblk[threadIdx.x]));
}

__global__ void __launch_bounds__(256)
fast_hist_private_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, long long nvec, int n,
                         unsigned long long* __restrict__ hist, int warps) {
  extern __shared__ __align__(16) unsigned char smem_h[];
  const int nbins = n * n;
  const int slots = nbins + 2;                                  // + overflow slot + trash slot (ignored pixels)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // layout: [warps][slots][32] byte counters, then [warps][slots] u32 sums
  unsigned char* mine = smem_h + static_cast<size_t>(warp) * slots * 32;
  unsigned int* sums = reinterpret_cast<unsigned int*>(smem_h + static_cast<size_t>(warps) * slots * 32) + warp * slots;
  for (int i = lane; i < slots * 8; i += 32) reinterpret_cast<unsigned int*>(mine)[i] = 0;
  for (int i = lane; i < slots; i += 32) sums[i] = 0;
  __syncwarp();

  auto fold = [&]() {       // byte counters -> 32-bit sums; lane l owns slots l, l+32, ...
    __syncwarp();
    for (int s = lane; s < slots; s += 32) {
      uint4* row = reinterpret_cast<uint4*>(mine + s * 32);
      const uint4 r0 = row[0], r1 = row[1];
      unsigned t = 0;
      t = __dp4a(r0.x, 0x01010101u, t); t = __dp4a(r0.y, 0x01010101u, t); t = __dp4a(r0.z, 0x01010101u, t); t = __dp4a(r0.w, 0x01010101u, t);
      t = __dp4a(r1.x, 0x01010101u, t); t = __dp4a(r1.y, 0x01010101u, t); t = __dp4a(r1.z, 0x01010101u, t); t = __dp4a(r1.w, 0x01010101u, t);
      sums[s] += t;
      row[0] = make_uint4(0, 0, 0, 0); row[1] = make_uint4(0, 0, 0, 0);
    }
    __syncwarp();
  };

  unsigned char* col = mine + lane;                              // this lane's counter column
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  int since_fold = 0;
  // i0 is the warp's first index: every lane of a warp runs the same number of iterations (fold() is warp-collective)
  for (long long i0 = static_cast<long long>(blockIdx.x) * blockDim.x + warp * 32; i0 < nvec; i0 += stride) {
    const long long i = i0 + lane;
    uint4 va = make_uint4(~0u, ~0u, ~0u, ~0u), vb = make_uint4(0, 0, 0, 0);      // a = 255: ignored
    if (i < nvec) { va = __ldg(a + i); vb = __ldg(b + i); }
    const unsigned wa[4] = {va.x, va.y, va.z, va.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
    for (int wsel = 0; wsel < 4; ++wsel) {
      // four pixels at a time: the four counter loads are independent (latency overlaps); pixels that share a bin
      // all store old + multiplicity, so aliasing stores agree.  Ignored pixels go to a trash slot: no branches.
      unsigned char* pc[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int av = (wa[wsel] >> (8 * k)) & 0xff, bv = (wb[wsel] >> (8 * k)) & 0xff;
        int bin = n * av + bv;
        if (bin > nbins) bin = nbins;                 // out-of-range prediction -> overflow slot
        if (av >= n) bin = nbins + 1;                 // ignored ground truth -> trash slot
        pc[k] = col + bin * 32;
      }
      unsigned c[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) c[k] = *pc[k];
      const unsigned e01 = pc[0] == pc[1], e02 = pc[0] == pc[2], e03 = pc[0] == pc[3];
      const unsigned e12 = pc[1] == pc[2], e13 = pc[1] == pc[3], e23 = pc[2] == pc[3];
      *pc[0] = static_cast<unsigned char>(c[0] + 1 + e01 + e02 + e03);
      *pc[1] = static_cast<unsigned char>(c[1] + 1 + e01 + e12 + e13);
      *pc[2] = static_cast<unsigned char>(c[2] + 1 + e02 + e12 + e23);
      *pc[3] = static_cast<unsigned char>(c[3] + 1 + e03 + e13 + e23);
    }
    since_fold += 16;
    if (since_fold >= 240) { fold(); since_fold = 0; }       // byte counters hold at most 240 increments
  }
  fold();
  __syncthreads();
  // block total -> global
  for (int s = threadIdx.x; s <= nbins; s += blockDim.x) {      // the trash slot is not published
    unsigned long long t = 0;
    for (int w2 = 0; w2 < warps; ++w2)
      t += reinterpret_cast<unsigned int*>(smem_h + static_cast<size_t>(warps) * slots * 32)[w2 * slots + s];
    if (t) atomicAdd(&hist[s], t);
  }
}


// ---------------------------------------------------------------------------------------------------------------
// "lanes" kernels (round 2): the uint8 hot path for any n with n*n + 1 <= 1024 bins.
//
// Every lane owns a private byte counter per bin, laid out [bin / 4][lane][bin % 4]: lane l only ever touches shared-memory
// bank l, so every LDS.U8 / STS.U8 of the warp is conflict-free whatever the data (the round-1 [bin][lane] layout left
// lanes 4k..4k+3 to fight over four banks: ~2.1-way conflicts on random masks).  The pixel arithmetic is done two pixels
// per 32-bit register (PRMT pairs -> one IMAD for n*a+b -> one VMNMX clamp -> one shift/mask to the byte offset), ignored
// pixels (a >= n) fall into the same clamp slot as out-of-range bins and are told apart by one SIMD compare + POPC per four
// pixels, and instead of folding the byte counters every 240 pixels a wrapped byte (255 -> 0) adds 256 to a per-warp
// 32-bit table through a predicated shared-memory atomic (never taken on ordinary masks).  A lane increments its pixels
// strictly in order (aliasing needs no comparison logic); 12 warps per SM and a 3-deep register prefetch of the 16-byte
// loads cover the latency.
// ---------------------------------------------------------------------------------------------------------------
struct HistSmem {
  unsigned char* bytes;     // [warps][rows][32 lanes][4]
  unsigned int* wraps;      // [warps][slots]: multiples of 256 carried out of the byte counters
};

// Rare path: some byte counter of this lane wrapped (255 -> 0) while the `npix` pixels (4 per 32-bit word of wa / wb) were
// counted.  A bin with m hits in the batch wrapped iff its counter now reads < m (m <= 16); each wrap carries 256 into the
// warp's 32-bit table.
__device__ __noinline__ void hist_carry(const unsigned* wa, const unsigned* wb, int npix, unsigned n, unsigned nbins,
                                        const unsigned char* col, unsigned int* wraps) {
  unsigned bins[16];
  for (int k = 0; k < npix; ++k) {
    const unsigned av = (wa[k >> 2] >> (8 * (k & 3))) & 0xffu, bv = (wb[k >> 2] >> (8 * (k & 3))) & 0xffu;
    const unsigned bin = av * n + bv;
    bins[k] = bin < nbins ? bin : nbins;
  }
  for (int k = 0; k < npix; ++k) {
    unsigned m = 0;
    bool first = true;
    for (int j = 0; j < npix; ++j) {
      if (bins[j] == bins[k]) { ++m; if (j < k) first = false; }
    }
    if (first && col[(bins[k] >> 2) * 128 + (bins[k] & 3)] < m) atomicAdd(wraps + bins[k], 256u);
  }
}

// Four pixels (one 32-bit word of ground truth + one of predictions).  Pixels are counted in pairs: both counter loads are
// issued before either store (two shared-memory round trips in flight per lane); a pair that hits the same counter stores
// c + 1 then c + 2.  `carry` collects bit 8 of every incremented value (set iff a byte wrapped).
__device__ __forceinline__ void hist_count4(unsigned wa, unsigned wb, unsigned n, unsigned clamp2, unsigned char* col,
                                            unsigned& ign, unsigned& carry, unsigned n4) {
  ign += __popc(__vcmpgeu4(wa, n4));                            // 8 set bits per ignored pixel (a >= n)
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const unsigned a2 = __byte_perm(wa, 0u, h ? 0x4342u : 0x4140u);      // two pixels as 16-bit halves
    const unsigned b2 = __byte_perm(wb, 0u, h ? 0x4342u : 0x4140u);
    unsigned bin2 = a2 * n + b2;                                   // 255 * 64 + 255 < 2^16: the halves never carry
    bin2 = __vminu2(bin2, clamp2);                                 // >= n*n (ignored or out of range) -> slot n*n
    const unsigned off2 = (bin2 & 0x00030003u) | ((bin2 & 0xfffcfffcu) << 5);      // (bin >> 2) * 128 + (bin & 3)
    unsigned char* p0 = col + (off2 & 0xffffu);
    unsigned char* p1 = col + (off2 >> 16);
    unsigned c0 = *p0, c1 = *p1;
    c0 += 1u;
    c1 += p0 == p1 ? 2u : 1u;
    *p0 = static_cast<unsigned char>(c0);
    *p1 = static_cast<unsigned char>(c1);
    carry |= c0 | c1;
  }
}

__device__ __forceinline__ void hist_count16(const uint4& va, const uint4& vb, unsigned n, unsigned nbins, unsigned clamp2,
                                             unsigned char* col, unsigned int* wraps, unsigned& ign, unsigned n4) {
  unsigned carry = 0;
  hist_count4(va.x, vb.x, n, clamp2, col, ign, carry, n4);
  hist_count4(va.y, vb.y, n, clamp2, col, ign, carry, n4);
  hist_count4(va.z, vb.z, n, clamp2, col, ign, carry, n4);
  hist_count4(va.w, vb.w, n, clamp2, col, ign, carry, n4);
  if (carry & 0x100u) {
    const unsigned wa[4] = {va.x, va.y, va.z, va.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
    hist_carry(wa, wb, 16, n, nbins, col, wraps);
  }
}

// block totals -> global.  slot n*n holds ignored + out-of-range pixels; only the latter are published.
__device__ __forceinline__ void hist_publish(const HistSmem& sm, int warps, int rows, int slots, unsigned ign_lane,
                                             unsigned long long* __restrict__ hist, unsigned int* s_ign) {
  const unsigned ign_warp = __reduce_add_sync(0xffffffffu, ign_lane);
  if ((threadIdx.x & 31) == 0 && ign_warp) atomicAdd(s_ign, ign_warp);
  __syncthreads();
  for (int s = threadIdx.x; s < slots; s += blockDim.x) {
    unsigned long long t = 0;
    const int row = s >> 2, sh = 8 * (s & 3);
    for (int w = 0; w < warps; ++w) {
      const unsigned int* words = reinterpret_cast<const unsigned int*>(sm.bytes + (static_cast<size_t>(w) * rows + row) * 128);
      unsigned acc = 0;
#pragma unroll 8
      for (int j = 0; j < 32; ++j) acc += (words[(j + row) & 31] >> sh) & 0xffu;      // staggered: conflict-free across rows
      t += acc + sm.wraps[w * slots + s];
    }
    if (s == slots - 1) t -= (*s_ign >> 3);                       // drop the ignored pixels from the overflow slot
    if (t) atomicAdd(&hist[s], t);
  }
}

__device__ __forceinline__ HistSmem hist_smem_init(unsigned char* smem, int warps, int rows, int slots) {
  HistSmem sm;
  sm.bytes = smem;
  sm.wraps = reinterpret_cast<unsigned int*>(smem + static_cast<size_t>(warps) * rows * 128);
  uint4* z = reinterpret_cast<uint4*>(smem);
  const int total16 = (warps * rows * 128 + warps * slots * 4 + 15) / 16;
  for (int i = threadIdx.x; i < total16; i += blockDim.x) z[i] = make_uint4(0, 0, 0, 0);
  return sm;
}

struct HistItem {            // one (ground truth, prediction) pair of a batched call (32 bytes)
  const unsigned char* a;
  const unsigned char* b;
  long long len;
  long long first_chunk;     // sum over the previous items of max(1, ceil((len / 16) / kHistChunkVec))
};
constexpr long long kHistChunkVec = 16384;     // 16-byte vectors per work unit of a batched call (256 KB of each mask = one 512x512 mask)
constexpr int kHistDepth = 4;                  // 16-byte load pairs in flight per lane

// Batched form of fast_hist_packed_kernel (n*n + 1 <= 32 bins, counters in registers): work units as in the lanes kernel.
template <int NW>
__global__ void __launch_bounds__(256)
fast_hist_packed_batch_kernel(const HistItem* __restrict__ items, int count, long long total_chunks, int n,
                              unsigned long long* __restrict__ hist) {
  const int nbins = n * n;
  unsigned long long pk[NW];
  unsigned int wide[NW * 8];
#pragma unroll
  for (int i = 0; i < NW; ++i) pk[i] = 0ull;
#pragma unroll
  for (int i = 0; i < NW * 8; ++i) wide[i] = 0u;
  auto widen = [&]() {
#pragma unroll
    for (int i = 0; i < NW; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) wide[i * 8 + k] += static_cast<unsigned int>(pk[i] >> (8 * k)) & 0xffu;
      pk[i] = 0ull;
    }
  };
  auto count1 = [&](unsigned av, unsigned bv) {
    unsigned bin = n * av + bv;
    if (bin > static_cast<unsigned>(nbins)) bin = nbins;                   // overflow slot
    const unsigned long long inc = av < static_cast<unsigned>(n) ? 1ull << (8 * (bin & 7u)) : 0ull;
    const unsigned word = bin >> 3;
#pragma unroll
    for (int q = 0; q < NW; ++q) pk[q] += (word == static_cast<unsigned>(q)) ? inc : 0ull;
  };
  int since = 0;
  for (long long u = blockIdx.x; u < total_chunks; u += gridDim.x) {
    int lo = 0, hi = count - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (__ldg(&items[mid].first_chunk) <= u) lo = mid; else hi = mid - 1;
    }
    const unsigned char *pa = items[lo].a, *pb = items[lo].b;
    const long long len = items[lo].len, nvec = len / 16;
    const long long v0 = (u - items[lo].first_chunk) * kHistChunkVec;
    const long long v1 = v0 + kHistChunkVec < nvec ? v0 + kHistChunkVec : nvec;
    const uint4 *qa = reinterpret_cast<const uint4*>(pa), *qb = reinterpret_cast<const uint4*>(pb);
    for (long long i = v0 + threadIdx.x; i < v1; i += blockDim.x) {
      const uint4 va = __ldg(qa + i), vb = __ldg(qb + i);
      const unsigned wa[4] = {va.x, va.y, va.z, va.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
      for (int wsel = 0; wsel < 4; ++wsel) {
#pragma unroll
        for (int k = 0; k < 4; ++k) count1((wa[wsel] >> (8 * k)) & 0xffu, (wb[wsel] >> (8 * k)) & 0xffu);
      }
      since += 16;
      if (since >= 240) { widen(); since = 0; }
    }
    if (v1 == nvec && threadIdx.x < 16) {                                     // the pair's len % 16 tail
      const long long t = nvec * 16 + threadIdx.x;
      if (t < len) { count1(pa[t], pb[t]); if (++since >= 240) { widen(); since = 0; } }
    }
  }
  widen();
  __shared__ unsigned int sblk[NW * 8];
  if (threadIdx.x < NW * 8) sblk[threadIdx.x] = 0;
  __syncthreads();
#pragma unroll
  for (int v = 0; v < NW * 8; ++v) {
    const unsigned t = __reduce_add_sync(0xffffffffu, wide[v]);
    if ((threadIdx.x & 31) == (v & 31) && t) atomicAdd(&sblk[v], t);
  }
  __syncthreads();
  if (threadIdx.x <= nbins && sblk[threadIdx.x]) atomicAdd(&hist[threadIdx.x], static_cast<unsigned long long>(sblk[threadIdx.x]));
}

// Work unit = one chunk of one pair; blocks take units round-robin, so a thousand 512x512 masks keep every SM busy on its own
// mask.  items == nullptr: the single pair (a0, b0, len0).  Pointers must be 16-byte aligned; the len % 16 tail of a pair is
// counted by warp 0 of the block that owns the pair's last chunk, one pixel per lane.
__global__ void __launch_bounds__(384, 1)
fast_hist_lanes_kernel(const HistItem* __restrict__ items, int count, long long total_chunks, long long chunk_vec,
                       const unsigned char* a0, const unsigned char* b0, long long len0, int n,
                       unsigned long long* __restrict__ hist, int warps) {
  extern __shared__ __align__(16) unsigned char smem_h[];
  __shared__ unsigned int s_ign;
  const int nbins = n * n, slots = nbins + 1, rows = (slots + 3) / 4;
  const HistSmem sm = hist_smem_init(smem_h, warps, rows, slots);
  if (threadIdx.x == 0) s_ign = 0;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* col = sm.bytes + static_cast<size_t>(warp) * rows * 128 + lane * 4;
  unsigned int* wraps = sm.wraps + warp * slots;
  const unsigned un = static_cast<unsigned>(n), n4 = un * 0x01010101u, clamp2 = static_cast<unsigned>(nbins) * 0x00010001u;
  unsigned ign = 0;
  const uint4 skip_a = make_uint4(~0u, ~0u, ~0u, ~0u), skip_b = make_uint4(0, 0, 0, 0);
  const long long step = blockDim.x;
  for (long long u = blockIdx.x; u < total_chunks; u += gridDim.x) {
    const unsigned char *pa = a0, *pb = b0;
    long long len = len0, first = 0;
    if (items) {                                   // last item whose first_chunk <= u (every thread: broadcast loads)
      int lo = 0, hi = count - 1;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&items[mid].first_chunk) <= u) lo = mid; else hi = mid - 1;
      }
      pa = items[lo].a; pb = items[lo].b; len = items[lo].len; first = items[lo].first_chunk;
    }
    const long long nvec = len / 16;
    const long long v0 = (u - first) * chunk_vec;
    const long long v1 = v0 + chunk_vec < nvec ? v0 + chunk_vec : nvec;
    const uint4* qa = reinterpret_cast<const uint4*>(pa);
    const uint4* qb = reinterpret_cast<const uint4*>(pb);
    // kHistDepth vector pairs in flight per lane (ncu on the 3-deep version: "long scoreboard" was the top stall, the loads of
    // a slot are re-issued as soon as its previous contents have been copied out)
    uint4 ra[kHistDepth], rb[kHistDepth];
#pragma unroll
    for (int k = 0; k < kHistDepth; ++k) {
      const long long j = v0 + threadIdx.x + k * step;
      ra[k] = skip_a; rb[k] = skip_b;
      if (j < v1) { ra[k] = __ldg(qa + j); rb[k] = __ldg(qb + j); }
    }
    for (long long i = v0 + threadIdx.x; i < v1; i += kHistDepth * step) {
#pragma unroll
      for (int k = 0; k < kHistDepth; ++k) {
        const uint4 ca = ra[k], cb = rb[k];
        const long long j = i + (k + kHistDepth) * step;
        ra[k] = skip_a; rb[k] = skip_b;
        if (j < v1) { ra[k] = __ldg(qa + j); rb[k] = __ldg(qb + j); }
        if (i + k * step < v1) hist_count16(ca, cb, un, static_cast<unsigned>(nbins), clamp2, col, wraps, ign, n4);
      }
    }
    if (v1 == nvec && warp == 0) {                 // this unit ends the pair: tail pixels, one per lane, padded with ignored pixels
      for (long long t = nvec * 16 + lane; t < len; t += 32)
        hist_count16(make_uint4(0xffffff00u | pa[t], ~0u, ~0u, ~0u), make_uint4(pb[t], 0u, 0u, 0u), un, static_cast<unsigned>(nbins),
                     clamp2, col, wraps, ign, n4);
    }
  }
  __syncthreads();
  hist_publish(sm, warps, rows, slots, ign, hist, &s_ign);
}

// get_miou without the mask round trip (get_miou.py:45-65 + utils_metrics.py:74-95): pred = argmax_c logits[n][c][h][w]
// (lowest index on ties, like numpy), optionally written as a uint8 mask, and (gt, pred) counted in the same pass.
// HBM-bound on the logits (4C B/pixel); one thread = four consecutive pixels (float4 per class plane).
__global__ void __launch_bounds__(384, 1)
argmax_hist_kernel(const float* __restrict__ logits, const unsigned char* __restrict__ gt, unsigned char* __restrict__ pred,
                   int N, int C, long long HW, int n, unsigned long long* __restrict__ hist, int warps) {
  extern __shared__ __align__(16) unsigned char smem_h[];
  __shared__ unsigned int s_ign;
  const int nbins = n * n, slots = nbins + 1, rows = (slots + 3) / 4;
  const HistSmem sm = hist_smem_init(smem_h, warps, rows, slots);
  if (threadIdx.x == 0) s_ign = 0;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* col = sm.bytes + static_cast<size_t>(warp) * rows * 128 + lane * 4;
  unsigned int* wraps = sm.wraps + warp * slots;
  const unsigned un = static_cast<unsigned>(n), n4 = un * 0x01010101u, clamp2 = static_cast<unsigned>(nbins) * 0x00010001u;
  unsigned ign = 0;
  const long long q_per_img = HW / 4;                     // HW % 4 == 0 (checked by the host)
  const long long total = static_cast<long long>(N) * q_per_img;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < total; q += stride) {
    const long long img = q / q_per_img, p4 = q - img * q_per_img;
    const float4* plane = reinterpret_cast<const float4*>(logits + static_cast<size_t>(img) * C * HW) + p4;
    float4 best = __ldg(plane);
    unsigned idx = 0;                                     // four class indices, one per byte
    for (int c0 = 1; c0 < C; c0 += 16) {                  // sixteen class planes requested before any is compared
      float4 v[16];
#pragma unroll
      for (int k = 0; k < 16; ++k)
        if (c0 + k < C) v[k] = __ldg(plane + static_cast<size_t>(c0 + k) * q_per_img);
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const unsigned c = static_cast<unsigned>(c0 + k);
        if (c0 + k < C) {
          if (v[k].x > best.x) { best.x = v[k].x; idx = (idx & 0xffffff00u) | c; }
          if (v[k].y > best.y) { best.y = v[k].y; idx = (idx & 0xffff00ffu) | (c << 8); }
          if (v[k].z > best.z) { best.z = v[k].z; idx = (idx & 0xff00ffffu) | (c << 16); }
          if (v[k].w > best.w) { best.w = v[k].w; idx = (idx & 0x00ffffffu) | (c << 24); }
        }
      }
    }
    if (pred) reinterpret_cast<unsigned int*>(pred)[q] = idx;
    if (gt) {
      const unsigned wa = __ldg(reinterpret_cast<const unsigned int*>(gt) + q);
      unsigned carry = 0;
      hist_count4(wa, idx, un, clamp2, col, ign, carry, n4);
      if (carry & 0x100u) hist_carry(&wa, &idx, 4, un, static_cast<unsigned>(nbins), col, wraps);
    }
  }
  __syncthreads();
  if (gt) hist_publish(sm, warps, rows, slots, ign, hist, &s_ign);
}

// ---------------------------------------------------------------------------------------------------------------
// 64 < n <= 256 ("wide"): n*n + 1 bins no longer fit lane-private byte counters.  One shared-memory table per block;
// lanes of a warp holding the same bin (real masks are piecewise constant) are combined with __match_any_sync so one
// atomic covers them; the table is flushed to the 64-bit global histogram with integer atomics (exact, order-free).
// Counters are 32-bit while n*n + 1 of them fit a block's 227 KB (n <= 241).  Beyond that (C16) two 16-bit counters
// share a word and the table is flushed after every 63 pixels per thread (at most 64512 < 2^16 increments per counter).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kWideThreads = 1024;
constexpr size_t kWideSmemMax = 227 * 1024;

__host__ __device__ inline bool hist_wide_c16(int n) { return static_cast<size_t>(n * n + 1) * 4 > kWideSmemMax; }
__host__ __device__ inline int hist_wide_words(int n) { return hist_wide_c16(n) ? (n * n + 2) / 2 : n * n + 1; }

template <bool C16>
__device__ __forceinline__ void wide_flush(unsigned int* sh, int n, unsigned long long* __restrict__ hist) {
  const int slots = n * n + 1, words = hist_wide_words(n);
  for (int i = threadIdx.x; i < words; i += blockDim.x) {
    const unsigned v = sh[i];
    if (!v) continue;
    sh[i] = 0u;
    if (C16) {
      if (v & 0xffffu) atomicAdd(&hist[2 * i], static_cast<unsigned long long>(v & 0xffffu));
      if ((v >> 16) && 2 * i + 1 < slots) atomicAdd(&hist[2 * i + 1], static_cast<unsigned long long>(v >> 16));
    } else {
      atomicAdd(&hist[i], static_cast<unsigned long long>(v));
    }
  }
}

// counts pixels [p0, p1) of a block-uniform range; fetch(i, a, b) returns the pair of pixel i (fast_hist's semantics:
// a outside [0, n) is ignored, n * a + b outside [0, n*n) goes to the overflow slot n*n)
template <bool C16, typename Fetch>
__device__ __forceinline__ void wide_count_range(long long p0, long long p1, int n, unsigned int* sh,
                                                 unsigned long long* __restrict__ hist, Fetch fetch) {
  const int lane = threadIdx.x & 31, nbins = n * n;
  const long long step = C16 ? 63LL * blockDim.x : p1 - p0;
  for (long long s0 = p0; s0 < p1; s0 += step) {
    const long long s1 = s0 + step < p1 ? s0 + step : p1;
    for (long long i0 = s0 + (threadIdx.x & ~31); i0 < s1; i0 += blockDim.x) {    // warp-uniform: full-warp match below
      const long long i = i0 + lane;
      int bin = -1;
      if (i < s1) {
        long long av, bv;
        fetch(i, av, bv);
        if (av >= 0 && av < n) {
          const long long bb = static_cast<long long>(n) * av + bv;
          bin = (bb >= 0 && bb < nbins) ? static_cast<int>(bb) : nbins;
        }
      }
      const unsigned peers = __match_any_sync(0xffffffffu, bin);
      if (bin >= 0 && lane == __ffs(peers) - 1) {
        if (C16) atomicAdd(&sh[bin >> 1], static_cast<unsigned>(__popc(peers)) << ((bin & 1) * 16));
        else atomicAdd(&sh[bin], static_cast<unsigned>(__popc(peers)));
      }
    }
    if (C16) { __syncthreads(); wide_flush<true>(sh, n, hist); __syncthreads(); }
  }
}

template <bool C16>
__device__ __forceinline__ unsigned int* wide_table_init(int n) {
  extern __shared__ __align__(16) unsigned int sh_wide[];
  for (int i = threadIdx.x; i < hist_wide_words(n); i += blockDim.x) sh_wide[i] = 0u;
  __syncthreads();
  return sh_wide;
}

template <typename T, bool C16>
__global__ void __launch_bounds__(kWideThreads)
fast_hist_wide_kernel(const T* __restrict__ a, const T* __restrict__ b, long long len, long long unit, int n,
                      unsigned long long* __restrict__ hist) {
  unsigned int* sh = wide_table_init<C16>(n);
  for (long long p0 = blockIdx.x * unit; p0 < len; p0 += gridDim.x * unit) {
    const long long p1 = p0 + unit < len ? p0 + unit : len;
    wide_count_range<C16>(p0, p1, n, sh, hist, [&](long long i, long long& av, long long& bv) {
      av = static_cast<long long>(a[i]); bv = static_cast<long long>(b[i]);
    });
  }
  __syncthreads();
  wide_flush<C16>(sh, n, hist);
}

// batched form: work units are the item table's chunks (as in fast_hist_lanes_kernel); the last chunk of a pair also
// takes its len % 16 tail pixels
template <bool C16>
__global__ void __launch_bounds__(kWideThreads)
fast_hist_wide_batch_kernel(const HistItem* __restrict__ items, int count, long long total_chunks, int n,
                            unsigned long long* __restrict__ hist) {
  unsigned int* sh = wide_table_init<C16>(n);
  for (long long u = blockIdx.x; u < total_chunks; u += gridDim.x) {
    int lo = 0, hi = count - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (__ldg(&items[mid].first_chunk) <= u) lo = mid; else hi = mid - 1;
    }
    const unsigned char *pa = items[lo].a, *pb = items[lo].b;
    const long long len = items[lo].len, nvec = len / 16;
    const long long v0 = (u - items[lo].first_chunk) * kHistChunkVec;
    const long long p0 = 16 * v0, p1 = v0 + kHistChunkVec >= nvec ? len : 16 * (v0 + kHistChunkVec);
    wide_count_range<C16>(p0, p1, n, sh, hist, [&](long long i, long long& av, long long& bv) {
      av = __ldg(pa + i); bv = __ldg(pb + i);
    });
  }
  __syncthreads();
  wide_flush<C16>(sh, n, hist);
}

// argmax_hist_kernel for 64 < n: one thread per pixel, arg-max over the class planes (lowest index on ties)
template <bool C16>
__global__ void __launch_bounds__(kWideThreads)
argmax_hist_wide_kernel(const float* __restrict__ logits, const unsigned char* __restrict__ gt, unsigned char* __restrict__ pred,
                        int N, int C, long long HW, long long unit, int n, unsigned long long* __restrict__ hist) {
  unsigned int* sh = wide_table_init<C16>(n);
  const long long total = static_cast<long long>(N) * HW;
  for (long long p0 = blockIdx.x * unit; p0 < total; p0 += gridDim.x * unit) {
    const long long p1 = p0 + unit < total ? p0 + unit : total;
    wide_count_range<C16>(p0, p1, n, sh, hist, [&](long long i, long long& av, long long& bv) {
      const long long img = i / HW, hw = i - img * HW;
      const float* z = logits + img * C * HW + hw;
      float best = __ldg(z); int arg = 0;
      for (int c = 1; c < C; ++c) { const float v = __ldg(z + c * HW); if (v > best) { best = v; arg = c; } }
      if (pred) pred[i] = static_cast<unsigned char>(arg);
      av = __ldg(gt + i); bv = arg;
    });
  }
  __syncthreads();
  wide_flush<C16>(sh, n, hist);
}

}  // namespace b2u

extern "C" {
using namespace b2u;

static int hist_lanes_warps(int n) {       // warps per block that fit 200 KB of byte counters + wrap tables (0: does not fit)
  const int slots = n * n + 1, rows = (slots + 3) / 4;
  const size_t per_warp = static_cast<size_t>(rows) * 128 + static_cast<size_t>(slots) * 4;
  int w = static_cast<int>((200 * 1024) / per_warp);
  return w > 12 ? 12 : w;
}
static int hist_set_attr(const void* fn) {
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 204 * 1024);
  return e == cudaSuccess ? 0 : set_error(B2U_ERR_CUDA, "fast_hist: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
}
static int launch_hist_lanes(const HistItem* items, int count, long long total_chunks, const unsigned char* a, const unsigned char* b,
                             long long len, int n, unsigned long long* hist, cudaStream_t st) {
  const int warps = hist_lanes_warps(n);
  const int slots = n * n + 1, rows = (slots + 3) / 4;
  const size_t smem = static_cast<size_t>(warps) * (static_cast<size_t>(rows) * 128 + static_cast<size_t>(slots) * 4) + 16;
  static bool attr_done[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !attr_done[dev]) {
    if (int rc = hist_set_attr(reinterpret_cast<const void*>(fast_hist_lanes_kernel))) return rc;
    if (int rc = hist_set_attr(reinterpret_cast<const void*>(argmax_hist_kernel))) return rc;
    attr_done[dev] = true;
  }
  long long chunk_vec = kHistChunkVec;
  if (!items) {
    // a single pair: units sized so that every SM gets one (at least kHistDepth rounds of the block per unit)
    const long long nvec = len / 16, min_chunk = static_cast<long long>(warps) * 32 * kHistDepth;
    chunk_vec = (nvec + num_sms() - 1) / num_sms();
    if (chunk_vec < min_chunk) chunk_vec = min_chunk;
    total_chunks = (nvec + chunk_vec - 1) / chunk_vec;
    if (total_chunks < 1) total_chunks = 1;
  }
  int grid = num_sms();
  if (total_chunks < grid) grid = static_cast<int>(total_chunks);
  fast_hist_lanes_kernel<<<grid, warps * 32, smem, st>>>(items, count, total_chunks, chunk_vec, a, b, len, n, hist, warps);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "fast_hist_lanes launch: %s", cudaGetErrorString(e));
  note_launch();
  return 0;
}

// the wide kernels' dynamic shared memory: set once per device for every instantiation
static int hist_wide_attr() {
  static bool attr_done[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && attr_done[dev]) return 0;
  const void* fns[] = {reinterpret_cast<const void*>(fast_hist_wide_kernel<unsigned char, false>),
                       reinterpret_cast<const void*>(fast_hist_wide_kernel<unsigned char, true>),
                       reinterpret_cast<const void*>(fast_hist_wide_kernel<int, false>),
                       reinterpret_cast<const void*>(fast_hist_wide_kernel<int, true>),
                       reinterpret_cast<const void*>(fast_hist_wide_kernel<long long, false>),
                       reinterpret_cast<const void*>(fast_hist_wide_kernel<long long, true>),
                       reinterpret_cast<const void*>(fast_hist_wide_batch_kernel<false>),
                       reinterpret_cast<const void*>(fast_hist_wide_batch_kernel<true>),
                       reinterpret_cast<const void*>(argmax_hist_wide_kernel<false>),
                       reinterpret_cast<const void*>(argmax_hist_wide_kernel<true>)};
  for (const void* fn : fns) {
    const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kWideSmemMax));
    if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "fast_hist (wide): cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  }
  if (dev >= 0 && dev < 64) attr_done[dev] = true;
  return 0;
}
static size_t hist_wide_smem(int n) { return static_cast<size_t>(hist_wide_words(n)) * sizeof(unsigned int); }
// pixels per work unit: about one unit per SM (at least 64K pixels)
static long long hist_wide_unit(long long len) {
  long long u = (len + num_sms() - 1) / num_sms();
  return u < 65536 ? 65536 : u;
}
static int hist_wide_grid(long long units) { return static_cast<int>(units < num_sms() ? (units < 1 ? 1 : units) : num_sms()); }

static int fast_hist_wide(const void* a, const void* b, long long len, int n, int dtype, unsigned long long* hist, cudaStream_t st) {
  if (int rc = hist_wide_attr()) return rc;
  const long long unit = hist_wide_unit(len);
  const int grid = hist_wide_grid((len + unit - 1) / unit);
  const size_t sm = hist_wide_smem(n);
  const bool c16 = hist_wide_c16(n);
#define B2U_WIDE(T_) do { const T_* pa = static_cast<const T_*>(a); const T_* pb = static_cast<const T_*>(b);                       \
    if (c16) fast_hist_wide_kernel<T_, true><<<grid, kWideThreads, sm, st>>>(pa, pb, len, unit, n, hist);                         \
    else fast_hist_wide_kernel<T_, false><<<grid, kWideThreads, sm, st>>>(pa, pb, len, unit, n, hist); } while (0)
  if (dtype == 0) B2U_WIDE(unsigned char);
  else if (dtype == 1) B2U_WIDE(int);
  else if (dtype == 2) B2U_WIDE(long long);
  else return set_error(B2U_ERR_ARG, "fast_hist: dtype must be 0 (u8), 1 (i32) or 2 (i64)");
#undef B2U_WIDE
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "fast_hist_wide launch: %s", cudaGetErrorString(e));
  note_launch();
  return 0;
}

// hist: n*n + 1 uint64 on device, ACCUMULATED into (caller zeroes it); hist[n*n] counts out-of-range bins.
// dtype: 0 = uint8, 1 = int32, 2 = int64.  Blocks of 2^31 elements at most per call keep uint32 counters exact.
// 1 <= n <= 256 (64 < n: the shared-table kernels above).
int b2u_fast_hist(const void* a, const void* b, long long len, int n, int dtype, unsigned long long* hist, void* stream) {
  if (n <= 0 || n > 256) return set_error(B2U_ERR_SHAPE, "fast_hist: 1 <= n <= 256 (got %d)", n);
  if (len < 0) return set_error(B2U_ERR_SHAPE, "fast_hist: negative length");
  if (len == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n > 64) {
    const long long chunk = 1ll << 31;
    const size_t esz = dtype == 0 ? 1 : (dtype == 1 ? 4 : 8);
    for (long long off = 0; off < len; off += chunk) {
      const long long l = len - off < chunk ? len - off : chunk;
      if (int rc = fast_hist_wide(static_cast<const char*>(a) + off * esz, static_cast<const char*>(b) + off * esz, l, n, dtype, hist, st))
        return rc;
    }
    return 0;
  }
  const size_t sm = static_cast<size_t>(kHistWarps) * (n * n + 1) * sizeof(unsigned int);
  if (sm > 48 * 1024) {
    static bool big_done[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !big_done[dev]) {
      cudaFuncSetAttribute(fast_hist_kernel<unsigned char, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
      cudaFuncSetAttribute(fast_hist_kernel<unsigned char, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
      cudaFuncSetAttribute(fast_hist_kernel<int, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
      cudaFuncSetAttribute(fast_hist_kernel<long long, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
      big_done[dev] = true;
    }
  }
  const long long chunk = 1ll << 31;
  for (long long off = 0; off < len; off += chunk) {
    const long long l = len - off < chunk ? len - off : chunk;
    int grid = 8 * num_sms();
    if (dtype == 0) {
      const bool aligned = ((reinterpret_cast<uintptr_t>(a) + off) % 16 == 0) && ((reinterpret_cast<uintptr_t>(b) + off) % 16 == 0);
      const unsigned char* pa = static_cast<const unsigned char*>(a) + off;
      const unsigned char* pb = static_cast<const unsigned char*>(b) + off;
      long long want = (l / 16 + kHistWarps * 32 - 1) / (kHistWarps * 32);
      if (want < 1) want = 1;
      if (grid > want) grid = static_cast<int>(want);
      const long long nvec = l / 16;
      const int slots = n * n + 2;
      auto tail = [&]() {
        if (l % 16) fast_hist_kernel<unsigned char, 1><<<1, kHistWarps * 32, sm, st>>>(pa + nvec * 16, pb + nvec * 16, l % 16, n, hist);
      };
      // few bins (n*n + 1 <= 32): successive pixels keep hitting the same counter, a shared-memory round trip each; the
      // register-counter kernel below is 3-4x faster there (measured: 2.1 vs 0.56 TB/s at n = 2)
      if (aligned && n * n + 1 > kVoteMaxBins && hist_lanes_warps(n) >= 4) {
        int rc = launch_hist_lanes(nullptr, 1, 0, pa, pb, l, n, hist, st);
        if (rc) return rc;
        continue;
      } else if (aligned && nvec > 0 && n * n + 1 <= kVoteMaxBins) {
        int g2 = 8 * num_sms();
        const long long w2 = (nvec + 255) / 256;
        if (g2 > w2) g2 = static_cast<int>(w2);
        const uint4 *qa = reinterpret_cast<const uint4*>(pa), *qb = reinterpret_cast<const uint4*>(pb);
        if (n * n + 1 <= 8)       fast_hist_packed_kernel<1><<<g2, 256, 0, st>>>(qa, qb, nvec, n, hist);
        else if (n * n + 1 <= 24) fast_hist_packed_kernel<3><<<g2, 256, 0, st>>>(qa, qb, nvec, n, hist);
        else                      fast_hist_packed_kernel<4><<<g2, 256, 0, st>>>(qa, qb, nvec, n, hist);
        note_launch();
        tail();
      } else if (aligned && nvec > 0 && static_cast<size_t>(slots) * 36 * 2 <= 200 * 1024) {
        int warps = static_cast<int>((200 * 1024) / (static_cast<size_t>(slots) * 36));
        if (warps > 8) warps = 8;
        const size_t sm2 = static_cast<size_t>(warps) * slots * 36;
        static bool attr_done[64] = {false};
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev >= 0 && dev < 64 && !attr_done[dev]) {
          cudaFuncSetAttribute(fast_hist_private_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
          attr_done[dev] = true;
        }
        int g2 = num_sms();
        const long long w2 = (nvec + warps * 32 - 1) / (warps * 32);
        if (g2 > w2) g2 = static_cast<int>(w2);
        fast_hist_private_kernel<<<g2, warps * 32, sm2, st>>>(reinterpret_cast<const uint4*>(pa), reinterpret_cast<const uint4*>(pb), nvec, n, hist, warps);
        note_launch();
        tail();
      } else if (aligned) {
        fast_hist_kernel<unsigned char, 16><<<grid, kHistWarps * 32, sm, st>>>(pa, pb, l, n, hist);
      } else {
        fast_hist_kernel<unsigned char, 1><<<grid, kHistWarps * 32, sm, st>>>(pa, pb, l, n, hist);
      }
    } else if (dtype == 1) {
      fast_hist_kernel<int, 1><<<grid, kHistWarps * 32, sm, st>>>(static_cast<const int*>(a) + off, static_cast<const int*>(b) + off, l, n, hist);
    } else if (dtype == 2) {
      fast_hist_kernel<long long, 1><<<grid, kHistWarps * 32, sm, st>>>(static_cast<const long long*>(a) + off,
                                                                        static_cast<const long long*>(b) + off, l, n, hist);
    } else {
      return set_error(B2U_ERR_ARG, "fast_hist: dtype must be 0 (u8), 1 (i32) or 2 (i64)");
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "fast_hist launch: %s", cudaGetErrorString(e));
    note_launch();
  }
  return 0;
}

// Many (ground truth, prediction) uint8 mask pairs in ONE launch: compute_mIoU's loop over an evaluation set
// (utils/utils_metrics.py:74-95) without a launch per image.  items: `count` x {const uint8* a; const uint8* b; int64 len;
// int64 first_chunk} (32 bytes each) in DEVICE memory, first_chunk = running sum of b2u_fast_hist_chunks(len) over the previous
// items, total_chunks = the sum over all items; every pointer 16-byte aligned.  hist as in b2u_fast_hist.
int b2u_fast_hist_batch(const void* items, int count, long long total_chunks, int n, unsigned long long* hist, void* stream) {
  if (n <= 0 || n > 256) return set_error(B2U_ERR_SHAPE, "fast_hist_batch: 1 <= n <= 256 (got %d)", n);
  if (count < 0 || (count > 0 && (!items || total_chunks < count))) return set_error(B2U_ERR_ARG, "fast_hist_batch: bad item table");
  if (count == 0) return 0;
  if (n > 64) {
    if (int rc = hist_wide_attr()) return rc;
    const int grid = hist_wide_grid(total_chunks);
    const HistItem* it = static_cast<const HistItem*>(items);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (hist_wide_c16(n)) fast_hist_wide_batch_kernel<true><<<grid, kWideThreads, hist_wide_smem(n), st>>>(it, count, total_chunks, n, hist);
    else fast_hist_wide_batch_kernel<false><<<grid, kWideThreads, hist_wide_smem(n), st>>>(it, count, total_chunks, n, hist);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "fast_hist_wide_batch launch: %s", cudaGetErrorString(e));
    note_launch();
    return 0;
  }
  if (n * n + 1 <= kVoteMaxBins) {         // few bins: register counters (see b2u_fast_hist)
    int grid = 8 * num_sms();
    if (total_chunks < grid) grid = static_cast<int>(total_chunks);
    const HistItem* it = static_cast<const HistItem*>(items);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n * n + 1 <= 8)       fast_hist_packed_batch_kernel<1><<<grid, 256, 0, st>>>(it, count, total_chunks, n, hist);
    else if (n * n + 1 <= 24) fast_hist_packed_batch_kernel<3><<<grid, 256, 0, st>>>(it, count, total_chunks, n, hist);
    else                      fast_hist_packed_batch_kernel<4><<<grid, 256, 0, st>>>(it, count, total_chunks, n, hist);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "fast_hist_packed_batch launch: %s", cudaGetErrorString(e));
    note_launch();
    return 0;
  }
  if (hist_lanes_warps(n) < 1) return set_error(B2U_ERR_SHAPE, "fast_hist_batch: n = %d does not fit the shared-memory counters", n);
  return launch_hist_lanes(static_cast<const HistItem*>(items), count, total_chunks, nullptr, nullptr, 0, n, hist,
                           static_cast<cudaStream_t>(stream));
}
long long b2u_fast_hist_chunks(long long len) {      // work units of one pair of `len` pixels (for the table's first_chunk column)
  const long long c = (len / 16 + b2u::kHistChunkVec - 1) / b2u::kHistChunkVec;
  return c < 1 ? 1 : c;
}

// logits fp32 NCHW -> per-pixel class (argmax, lowest index on ties; unet.py:246-250) -> optional uint8 mask `pred` [N][H][W]
// and, with a ground-truth mask `gt` (uint8 [N][H][W], values >= n ignored), the n x n confusion matrix accumulated into
// hist (n*n + 1 uint64) in the same pass: Unet.get_miou_png + compute_mIoU (get_miou.py:45-65) as one kernel.
int b2u_argmax_hist(const float* logits, const unsigned char* gt, unsigned char* pred, int N, int C, int H, int W, int n,
                    unsigned long long* hist, void* stream) {
  if (N <= 0 || C <= 0 || C > 255 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "argmax_hist: bad shape");
  const long long HW = static_cast<long long>(H) * W;
  if (HW % 4 != 0) return set_error(B2U_ERR_SHAPE, "argmax_hist: H*W must be a multiple of 4");
  if (gt && (n <= 0 || n > 256 || !hist || (n <= 64 && hist_lanes_warps(n) < 1)))
    return set_error(B2U_ERR_ARG, "argmax_hist: bad n / hist");
  if (!gt && !pred) return set_error(B2U_ERR_ARG, "argmax_hist: nothing to produce");
  if (gt && n > 64) {
    if (int rc = hist_wide_attr()) return rc;
    const long long total = static_cast<long long>(N) * HW, unit = hist_wide_unit(total);
    const int grid = hist_wide_grid((total + unit - 1) / unit);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (hist_wide_c16(n)) argmax_hist_wide_kernel<true><<<grid, kWideThreads, hist_wide_smem(n), st>>>(logits, gt, pred, N, C, HW, unit, n, hist);
    else argmax_hist_wide_kernel<false><<<grid, kWideThreads, hist_wide_smem(n), st>>>(logits, gt, pred, N, C, HW, unit, n, hist);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "argmax_hist_wide launch: %s", cudaGetErrorString(e));
    note_launch();
    return 0;
  }
  const int nn = gt ? n : 1;
  const int warps = hist_lanes_warps(nn);
  const int slots = nn * nn + 1, rows = (slots + 3) / 4;
  const size_t smem = static_cast<size_t>(warps) * (static_cast<size_t>(rows) * 128 + static_cast<size_t>(slots) * 4) + 16;
  static bool attr_done[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !attr_done[dev]) {
    if (int rc = hist_set_attr(reinterpret_cast<const void*>(argmax_hist_kernel))) return rc;
    attr_done[dev] = true;
  }
  const long long total = static_cast<long long>(N) * (HW / 4);
  long long work = (total + warps * 32 - 1) / (warps * 32);
  int grid = 2 * num_sms();
  if (work < grid) grid = static_cast<int>(work < 1 ? 1 : work);
  argmax_hist_kernel<<<grid, warps * 32, smem, static_cast<cudaStream_t>(stream)>>>(logits, gt, pred, N, C, HW, nn, hist, warps);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "argmax_hist launch: %s", cudaGetErrorString(e));
  note_launch();
  return 0;
}

}  // extern "C"
