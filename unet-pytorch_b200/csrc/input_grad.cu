// input_grad.cu -- the gradient with respect to the input image (x.grad of the drop-in modules): the data gradient of the
// layer that reads the image, written as NCHW fp32 like the image itself.
//
//   first_conv_dgrad_input : 3x3 s1 p1 conv over the im2col rows of b2u_im2col_first (Unet-VGG16 features.0,
//                            TraditionalUnet inc.double_conv.0; nets/vgg.py:53, nets/TraditionalUnet.py:9)
//   stem_dgrad_input       : 7x7 s2 p3 ResNet stem over the rows of b2u_im2col_stem (nets/resnet.py:109)
//   nhwc_bf16_padded_to_nchw_f32 : the first C of Cpad channels of an NHWC bf16 gradient -> NCHW fp32 (the image convs of
//                            the graph families, whose dgrad already yields the gradient wrt the padded NHWC image)
//
// The two conv kernels are gathers: every thread owns a few output pixels and sums over the (tap, output channel) pairs that
// reach them -- no atomics, one fixed summation order, fp32 accumulation of bf16 dz times the fp32 OIHW weights.  Reading
// the fp32 weights (not the packed bf16 operand) also sidesteps the two-term image split of the forward: the lo columns
// of the im2col rows carry the same weights, and the gradient wrt the image is that of the hi columns alone.
// Per block, dz is staged through shared memory in 16-channel chunks with a row pitch of 1 mod 8 uint4 units, so the
// 16-byte loads of a warp (4 rows x 8 pixel groups) fall into 8 distinct bank groups.
#include "b2u_internal.h"
#include "b2u_ptx.cuh"

namespace b2u {

#define B2U_CHECK_LAUNCH(name)                                                                           \
  do {                                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                                \
    if (e__ != cudaSuccess) return b2u::set_error(B2U_ERR_CUDA, name " launch: %s", cudaGetErrorString(e__)); \
    b2u::note_launch();                                                                                  \
  } while (0)

__device__ __forceinline__ float chan8(const uint4& v, int k) {      // k is a compile-time constant after unrolling
  const uint32_t w = k < 2 ? v.x : k < 4 ? v.y : k < 6 ? v.z : v.w;
  return (k & 1) ? bf16_hi(w) : bf16_lo(w);
}

constexpr int kIgCo = 16;       // output channels (of the forward conv) staged per step

// Loads dz rows [r0, r0 + rows) x cols [c0, c0 + cols) of channels [co0, co0 + 16) into s[2][rows][pitch] (zeros outside).
__device__ __forceinline__ void stage_dz(uint4* s, const __nv_bfloat16* dz, int Cz, int n, int Hz, int Wz, int r0, int c0,
                                         int rows, int cols, int pitch, int co0) {
  const int items = 2 * rows * cols;
  for (int i = threadIdx.x; i < items; i += blockDim.x) {
    const int q = i / (rows * cols), rc = i - q * rows * cols;
    const int r = rc / cols, c = rc - r * cols;
    const int hh = r0 + r, ww = c0 + c;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (hh >= 0 && hh < Hz && ww >= 0 && ww < Wz)
      v = __ldg(reinterpret_cast<const uint4*>(dz + ((static_cast<size_t>(n) * Hz + hh) * Wz + ww) * Cz + co0) + q);
    s[(q * rows + r) * pitch + c] = v;
  }
}

// ---------------------------------------------------------------------------------------------- first 3x3 conv
// dx[n,c,h,w] = sum_{co,r,s} dz[n, h+1-r, w+1-s, co] * W[co,c,r,s].  Block = 16 x 64 output pixels; thread = 4 adjacent
// pixels of one row x CI channels.  Warp w covers rows 4 (w / 2) .. +3 and pixel groups 8 (w % 2) .. +7.
constexpr int kFcTh = 16, kFcTw = 64, kFcRows = kFcTh + 2, kFcCols = kFcTw + 2, kFcPitch = 73;
template <int CI>
__global__ void __launch_bounds__(256)
first_conv_dgrad_input_kernel(const __nv_bfloat16* __restrict__ dz, int Cz, const float* __restrict__ w, float* __restrict__ dx,
                              int H, int W, int Cout, int vec) {
  constexpr int CIP = CI <= 4 ? 4 : 8;
  __shared__ uint4 s_dz[2 * kFcRows * kFcPitch];
  __shared__ __align__(16) float s_w[kIgCo * 9 * CIP];
  const int n = blockIdx.z, h0 = blockIdx.y * kFcTh, w0 = blockIdx.x * kFcTw;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ty = (warp >> 1) * 4 + (lane >> 3), gx = (warp & 1) * 8 + (lane & 7);
  float acc[4][CI];
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int c = 0; c < CI; ++c) acc[p][c] = 0.f;

  for (int co0 = 0; co0 < Cz; co0 += kIgCo) {
    __syncthreads();
    stage_dz(s_dz, dz, Cz, n, H, W, h0 - 1, w0 - 1, kFcRows, kFcCols, kFcPitch, co0);
    for (int i = threadIdx.x; i < kIgCo * 9 * CIP; i += blockDim.x) {
      const int c = i % CIP, tap = (i / CIP) % 9, co = co0 + i / (9 * CIP);
      s_w[i] = (c < CI && co < Cout) ? __ldg(w + (static_cast<size_t>(co) * CI + c) * 9 + tap) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 2; ++q) {
#pragma unroll
      for (int j = 0; j < 3; ++j) {                 // halo row ty + j holds dz row h + 1 - r with r = 2 - j
        const uint4* row = s_dz + (q * kFcRows + ty + j) * kFcPitch + 4 * gx;
        uint4 v[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) v[k] = row[k];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          float f[6];
#pragma unroll
          for (int i = 0; i < 6; ++i) f[i] = chan8(v[i], k);
#pragma unroll
          for (int sh = 0; sh < 3; ++sh) {          // halo column 4 gx + p + sh holds dz column w + 1 - s with s = 2 - sh
            const float* wp = s_w + ((q * 8 + k) * 9 + (2 - j) * 3 + (2 - sh)) * CIP;
            float wv[CIP];
#pragma unroll
            for (int c4 = 0; c4 < CIP; c4 += 4) {
              const float4 t = *reinterpret_cast<const float4*>(wp + c4);
              wv[c4] = t.x; wv[c4 + 1] = t.y; wv[c4 + 2] = t.z; wv[c4 + 3] = t.w;
            }
#pragma unroll
            for (int p = 0; p < 4; ++p)
#pragma unroll
              for (int c = 0; c < CI; ++c) acc[p][c] = fmaf(f[p + sh], wv[c], acc[p][c]);
          }
        }
      }
    }
  }
  const int h = h0 + ty, x0 = w0 + 4 * gx;
  if (h >= H) return;
  const size_t HW = static_cast<size_t>(H) * W;
#pragma unroll
  for (int c = 0; c < CI; ++c) {
    float* out = dx + (static_cast<size_t>(n) * CI + c) * HW + static_cast<size_t>(h) * W + x0;
    if (vec && (W & 3) == 0 && x0 + 3 < W) {
      *reinterpret_cast<float4*>(out) = make_float4(acc[0][c], acc[1][c], acc[2][c], acc[3][c]);
    } else {
#pragma unroll
      for (int p = 0; p < 4; ++p)
        if (x0 + p < W) out[p] = acc[p][c];
    }
  }
}

// ---------------------------------------------------------------------------------------------- 7x7 s2 p3 stem
// dx[n,c,h,w] = sum over co and the taps with h + 3 - r, w + 3 - s even of dz[n, (h+3-r)/2, (w+3-s)/2, co] * W[co,c,r,s].
// Thread = the 2 x 2 output pixels (2a + dy, 2m + dx): they read dz rows a-1 .. a+2 and columns m-1 .. m+2, where dz row
// a-1+jj meets output row 2a+dy through tap r = dy + 5 - 2 jj (when 0 <= r < 7) -- per axis 3 taps for even and 4 for odd
// pixels, the same pattern for every thread.  Block = 8 x 32 quads = 16 x 64 output pixels.
constexpr int kStQh = 8, kStQw = 32, kStRows = kStQh + 3, kStCols = kStQw + 3, kStPitch = 41;
__global__ void __launch_bounds__(256)
stem_dgrad_input_kernel(const __nv_bfloat16* __restrict__ dz, int Cz, const float* __restrict__ w, float* __restrict__ dx, int Cin,
                        int H, int W, int Ho, int Wo, int Cout, int vec) {
  __shared__ uint4 s_dz[2 * kStRows * kStPitch];
  __shared__ __align__(16) float s_w[kIgCo * 49 * 4];
  const int n = blockIdx.z, a0 = blockIdx.y * kStQh, m0 = blockIdx.x * kStQw;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int qa = (warp >> 2) * 4 + (lane >> 3), qm = (warp & 3) * 8 + (lane & 7);
  float acc[2][2][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[i][j][c] = 0.f;

  for (int co0 = 0; co0 < Cz; co0 += kIgCo) {
    __syncthreads();
    stage_dz(s_dz, dz, Cz, n, Ho, Wo, a0 - 1, m0 - 1, kStRows, kStCols, kStPitch, co0);
    for (int i = threadIdx.x; i < kIgCo * 49 * 4; i += blockDim.x) {
      const int c = i & 3, tap = (i >> 2) % 49, co = co0 + i / (49 * 4);
      s_w[i] = (c < Cin && co < Cout) ? __ldg(w + (static_cast<size_t>(co) * Cin + c) * 49 + tap) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 2; ++q) {
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const uint4 v = s_dz[(q * kStRows + qa + jj) * kStPitch + qm + kk];
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float f = chan8(v, k);
            const float* wp = s_w + (q * 8 + k) * 49 * 4;
#pragma unroll
            for (int dy = 0; dy < 2; ++dy) {
              const int r = dy + 5 - 2 * jj;
              if (r < 0 || r > 6) continue;
#pragma unroll
              for (int dxx = 0; dxx < 2; ++dxx) {
                const int s = dxx + 5 - 2 * kk;
                if (s < 0 || s > 6) continue;
                const float4 t = *reinterpret_cast<const float4*>(wp + (r * 7 + s) * 4);
                acc[dy][dxx][0] = fmaf(f, t.x, acc[dy][dxx][0]);
                acc[dy][dxx][1] = fmaf(f, t.y, acc[dy][dxx][1]);
                acc[dy][dxx][2] = fmaf(f, t.z, acc[dy][dxx][2]);
                acc[dy][dxx][3] = fmaf(f, t.w, acc[dy][dxx][3]);
              }
            }
          }
        }
      }
    }
  }
  const size_t HW = static_cast<size_t>(H) * W;
#pragma unroll
  for (int dy = 0; dy < 2; ++dy) {
    const int h = 2 * (a0 + qa) + dy;
    if (h >= H) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if (c >= Cin) break;
      const int x0 = 2 * (m0 + qm);
      float* out = dx + (static_cast<size_t>(n) * Cin + c) * HW + static_cast<size_t>(h) * W + x0;
      if (vec && (W & 1) == 0 && x0 + 1 < W) {
        *reinterpret_cast<float2*>(out) = make_float2(acc[dy][0][c], acc[dy][1][c]);
      } else {                                      // odd W (rows start at odd offsets) or the image's last column
        if (x0 < W) out[0] = acc[dy][0][c];
        if (x0 + 1 < W) out[1] = acc[dy][1][c];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- padded NHWC -> NCHW
// thread = one pixel x 8 channels: a 16-byte read of the NHWC row, eight fp32 stores that are coalesced across the pixels
__global__ void nhwc_bf16_padded_to_nchw_f32_kernel(const uint4* __restrict__ x, float* __restrict__ y, int C, long long HW,
                                                    int Cpad8) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int n = blockIdx.z, q = blockIdx.y;
  if (i >= HW) return;
  const uint4 v = __ldg(x + (static_cast<size_t>(n) * HW + i) * Cpad8 + q);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int c = q * 8 + k;
    if (c < C) y[(static_cast<size_t>(n) * C + c) * HW + i] = chan8(v, k);
  }
}

}  // namespace b2u

extern "C" {
using namespace b2u;

int b2u_first_conv_dgrad_input(const void* dz, int Cz, const float* w, float* dx, int N, int Cin, int H, int W, int Cout,
                               void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || Cin <= 0 || 9 * Cin > 64 || Cout <= 0 || Cout > Cz || Cz % kIgCo != 0)
    return set_error(B2U_ERR_SHAPE, "first_conv_dgrad_input: bad shape (Cin=%d Cout=%d Cz=%d)", Cin, Cout, Cz);
  if (N > 65535 || (H + kFcTh - 1) / kFcTh > 65535) return set_error(B2U_ERR_SHAPE, "first_conv_dgrad_input: grid too large");
  if (reinterpret_cast<uintptr_t>(dz) % 16 != 0) return set_error(B2U_ERR_ARG, "first_conv_dgrad_input: dz must be 16-byte aligned");
  const dim3 grid((W + kFcTw - 1) / kFcTw, (H + kFcTh - 1) / kFcTh, N);
  const auto* d = static_cast<const __nv_bfloat16*>(dz);
  const int vec = reinterpret_cast<uintptr_t>(dx) % 16 == 0;      // float4 stores; scalar ones for an offset view
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (Cin) {
    case 1: first_conv_dgrad_input_kernel<1><<<grid, 256, 0, st>>>(d, Cz, w, dx, H, W, Cout, vec); break;
    case 2: first_conv_dgrad_input_kernel<2><<<grid, 256, 0, st>>>(d, Cz, w, dx, H, W, Cout, vec); break;
    case 3: first_conv_dgrad_input_kernel<3><<<grid, 256, 0, st>>>(d, Cz, w, dx, H, W, Cout, vec); break;
    case 4: first_conv_dgrad_input_kernel<4><<<grid, 256, 0, st>>>(d, Cz, w, dx, H, W, Cout, vec); break;
    case 5: first_conv_dgrad_input_kernel<5><<<grid, 256, 0, st>>>(d, Cz, w, dx, H, W, Cout, vec); break;
    case 6: first_conv_dgrad_input_kernel<6><<<grid, 256, 0, st>>>(d, Cz, w, dx, H, W, Cout, vec); break;
    default: first_conv_dgrad_input_kernel<7><<<grid, 256, 0, st>>>(d, Cz, w, dx, H, W, Cout, vec); break;
  }
  B2U_CHECK_LAUNCH("first_conv_dgrad_input");
  return 0;
}

int b2u_stem_dgrad_input(const void* dz, int Cz, const float* w, float* dx, int N, int Cin, int H, int W, int Cout, void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || Cin <= 0 || 49 * Cin > 192 || Cout <= 0 || Cout > Cz || Cz % kIgCo != 0)
    return set_error(B2U_ERR_SHAPE, "stem_dgrad_input: bad shape (Cin=%d Cout=%d Cz=%d)", Cin, Cout, Cz);
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  if (N > 65535 || (Ho + kStQh - 1) / kStQh > 65535) return set_error(B2U_ERR_SHAPE, "stem_dgrad_input: grid too large");
  if (reinterpret_cast<uintptr_t>(dz) % 16 != 0) return set_error(B2U_ERR_ARG, "stem_dgrad_input: dz must be 16-byte aligned");
  const dim3 grid((Wo + kStQw - 1) / kStQw, (Ho + kStQh - 1) / kStQh, N);
  const int vec = reinterpret_cast<uintptr_t>(dx) % 8 == 0;       // float2 stores; scalar ones for an offset view
  stem_dgrad_input_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(dz), Cz, w, dx,
                                                                               Cin, H, W, Ho, Wo, Cout, vec);
  B2U_CHECK_LAUNCH("stem_dgrad_input");
  return 0;
}

int b2u_nhwc_bf16_padded_to_nchw_f32(const void* x, float* y, int N, int C, int H, int W, int Cpad, void* stream) {
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || Cpad < C || Cpad % 8 != 0 || N > 65535)
    return set_error(B2U_ERR_SHAPE, "nhwc_bf16_padded_to_nchw_f32: bad shape (C=%d Cpad=%d)", C, Cpad);
  if (reinterpret_cast<uintptr_t>(x) % 16 != 0) return set_error(B2U_ERR_ARG, "nhwc_bf16_padded_to_nchw_f32: x must be 16-byte aligned");
  const long long HW = static_cast<long long>(H) * W;
  const dim3 grid(static_cast<unsigned>((HW + 255) / 256), (C + 7) / 8, N);
  nhwc_bf16_padded_to_nchw_f32_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const uint4*>(x), y, C, HW,
                                                                                           Cpad / 8);
  B2U_CHECK_LAUNCH("nhwc_bf16_padded_to_nchw_f32");
  return 0;
}

}  // extern "C"
