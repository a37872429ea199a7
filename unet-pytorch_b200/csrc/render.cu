// render.cu -- detect_image's rendering (unet.py:150-203) for a batch of images on the device: the class masks of the
// batched tail and the staged uint8 RGB sources in, the rendered uint8 RGB images (and per-image class counts) out.
//
//   mix_type 0: Image.blend(old, palette[m], 0.7).  Pillow (Blend.c) computes out = (UINT8)(a + alpha * (b - a)) with a
//               float alpha and int operands, i.e. in float32, with no fused multiply-add, truncated; the same operations
//               are written here as __fmul_rn / __fadd_rn, so no contraction can move a byte.
//   mix_type 1: palette[m].
//   mix_type 2: the source pixel where m != 0, else 0 (np.where((pr != 0)[..., None], old, 0)).
//   mix_type -1: no image; counts only.
// Counts are per-block shared-memory histograms added to the [count][C] uint64 output with integer atomics, so the result
// does not depend on the order of the blocks.
#include "b2u_internal.h"

namespace b2u {

constexpr int kRenderThreads = 256;
constexpr int kRenderBlocksPerImage = 256;    // pixel quads are strided over at most this many blocks per image

// one image of a batch (32 bytes, include/b2u.h)
struct RenderItem {
  const uint8_t* src;                    // uint8 [ih][iw][3], device
  const uint8_t* mask;                   // uint8 [ih][iw], device
  long long out_off;                     // byte offset of the rendered [ih][iw][3] image in `out`
  int ih, iw;
};
static_assert(sizeof(RenderItem) == 32, "RenderItem is part of the ABI");

__device__ __forceinline__ uint8_t blend07(uint8_t a, uint8_t b) {
  const float r = __fadd_rn(static_cast<float>(a), __fmul_rn(0.7f, static_cast<float>(static_cast<int>(b) - static_cast<int>(a))));
  return static_cast<uint8_t>(__float2int_rz(r));
}

// one pixel: s = its source bytes, m = its class, pal = the [C][3] palette in shared memory
template <int MODE>
__device__ __forceinline__ void render_px(const uint8_t* s, int m, int C, const uint8_t* pal, uint8_t* d) {
  const bool known = m < C;
  if (MODE == 2) {
    const bool keep = m != 0;
    d[0] = keep ? s[0] : 0; d[1] = keep ? s[1] : 0; d[2] = keep ? s[2] : 0;
    return;
  }
  const uint8_t p0 = known ? pal[3 * m] : 0, p1 = known ? pal[3 * m + 1] : 0, p2 = known ? pal[3 * m + 2] : 0;
  if (MODE == 1) {
    d[0] = p0; d[1] = p1; d[2] = p2;
  } else {
    d[0] = blend07(s[0], p0); d[1] = blend07(s[1], p1); d[2] = blend07(s[2], p2);
  }
}

// blockIdx.y = image; each thread takes four pixels at a time (12 source bytes, 4 mask bytes, 12 output bytes as 32-bit
// words when the three pointers are 4-byte aligned)
template <int MODE>
__global__ void __launch_bounds__(kRenderThreads)
render_batch_kernel(const RenderItem* __restrict__ items, const uint8_t* __restrict__ palette, int C, uint8_t* __restrict__ out,
                    unsigned long long* __restrict__ counts) {
  __shared__ uint8_t pal[3 * 256];
  __shared__ unsigned int hist[256];
  const RenderItem it = items[blockIdx.y];
  if (MODE == 0 || MODE == 1)
    for (int i = threadIdx.x; i < 3 * C; i += blockDim.x) pal[i] = palette[i];
  if (counts)
    for (int i = threadIdx.x; i < C; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  const long long npx = static_cast<long long>(it.ih) * it.iw;
  const long long quads = (npx + 3) / 4;
  uint8_t* dst = MODE >= 0 ? out + it.out_off : nullptr;
  const bool vec = ((reinterpret_cast<uintptr_t>(it.src) | reinterpret_cast<uintptr_t>(it.mask) |
                     reinterpret_cast<uintptr_t>(dst)) & 3) == 0;
  for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < quads;
       q += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long p0 = 4 * q;
    if (vec && npx - p0 >= 4) {                          // four pixels as 32-bit words, every index static
      uint32_t mw = __ldg(reinterpret_cast<const uint32_t*>(it.mask + p0));
      const uint8_t* m = reinterpret_cast<const uint8_t*>(&mw);
      if (counts) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (m[k] < C) atomicAdd(&hist[m[k]], 1u);
      }
      if (MODE < 0) continue;
      uint32_t sw[3] = {0, 0, 0}, dw[3];
      if (MODE != 1) {
        const uint32_t* sp = reinterpret_cast<const uint32_t*>(it.src + 3 * p0);
        sw[0] = __ldg(sp); sw[1] = __ldg(sp + 1); sw[2] = __ldg(sp + 2);
      }
      const uint8_t* sb = reinterpret_cast<const uint8_t*>(sw);
      uint8_t* db = reinterpret_cast<uint8_t*>(dw);
#pragma unroll
      for (int k = 0; k < 4; ++k) render_px<MODE>(sb + 3 * k, m[k], C, pal, db + 3 * k);
      uint32_t* dp = reinterpret_cast<uint32_t*>(dst + 3 * p0);
      dp[0] = dw[0]; dp[1] = dw[1]; dp[2] = dw[2];
    } else {                                             // the last pixels of an image, or unaligned pointers
      for (long long p = p0; p < p0 + 4 && p < npx; ++p) {
        const int m = it.mask[p];
        if (counts && m < C) atomicAdd(&hist[m], 1u);
        if (MODE < 0) continue;
        uint8_t sp[3] = {0, 0, 0}, d[3];
        if (MODE != 1) { sp[0] = it.src[3 * p]; sp[1] = it.src[3 * p + 1]; sp[2] = it.src[3 * p + 2]; }
        render_px<MODE>(sp, m, C, pal, d);
        dst[3 * p] = d[0]; dst[3 * p + 1] = d[1]; dst[3 * p + 2] = d[2];
      }
    }
  }
  if (counts) {
    __syncthreads();
    unsigned long long* row = counts + static_cast<size_t>(blockIdx.y) * C;
    for (int i = threadIdx.x; i < C; i += blockDim.x)
      if (hist[i]) atomicAdd(row + i, static_cast<unsigned long long>(hist[i]));
  }
}

}  // namespace b2u

extern "C" {
using namespace b2u;

int b2u_render_batch(const void* items, int count, const unsigned char* palette, int C, int mix_type, unsigned char* out,
                     unsigned long long* counts, long long max_pixels, void* stream) {
  if (!items || count <= 0 || count > 65535 || C < 1 || C > 255 || max_pixels <= 0 || mix_type < -1 || mix_type > 2)
    return set_error(B2U_ERR_SHAPE, "render_batch: bad arguments (count %d, C %d, mix_type %d, max_pixels %lld)", count, C,
                     mix_type, max_pixels);
  if ((mix_type >= 0 && !out) || (mix_type <= 1 && mix_type >= 0 && !palette) || (mix_type < 0 && !counts))
    return set_error(B2U_ERR_ARG, "render_batch: mix_type %d needs %s", mix_type,
                     mix_type < 0 ? "counts" : mix_type == 2 ? "out" : "out and palette");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (counts) {
    cudaError_t e = cudaMemsetAsync(counts, 0, sizeof(unsigned long long) * static_cast<size_t>(count) * C, st);
    if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "render_batch: clearing the counts: %s", cudaGetErrorString(e));
  }
  long long blocks = (max_pixels + 4LL * kRenderThreads - 1) / (4LL * kRenderThreads);
  if (blocks > kRenderBlocksPerImage) blocks = kRenderBlocksPerImage;
  const dim3 grid(static_cast<unsigned>(blocks), static_cast<unsigned>(count));
  const RenderItem* it = static_cast<const RenderItem*>(items);
  const uint8_t* pal = static_cast<const uint8_t*>(palette);
  switch (mix_type) {
    case 0: render_batch_kernel<0><<<grid, kRenderThreads, 0, st>>>(it, pal, C, out, counts); break;
    case 1: render_batch_kernel<1><<<grid, kRenderThreads, 0, st>>>(it, pal, C, out, counts); break;
    case 2: render_batch_kernel<2><<<grid, kRenderThreads, 0, st>>>(it, pal, C, out, counts); break;
    default: render_batch_kernel<-1><<<grid, kRenderThreads, 0, st>>>(it, pal, C, out, counts); break;
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "render_batch launch: %s", cudaGetErrorString(e));
  note_launch();
  return 0;
}

}  // extern "C"
