// head_loss.cu -- classifier head (final 1x1 conv) and the CE / Focal / Dice / f_score kernels.
//
//   head_fwd : logits[n,c,h,w] (NCHW fp32) = sum_k x[n,h,w,k] * W[c][k] + b[c]     nets/unet.py:58,76
//   head_bwd : dx (NHWC bf16, ReLU-masked by x), dW, db from dlogits (NCHW fp32)
//   loss_stats / loss_finalize / loss_bwd : nets/unet_training.py:9-56 and utils/utils_metrics.py:12-31
//     one pass over the logits accumulates everything CE_Loss, Focal_Loss, Dice_loss and f_score need;
//     the backward pass recomputes the softmax and writes dlogits for any linear combination of them.
//
// All of these are HBM-bound (AI <= 16 flop/B): coalesced NCHW plane accesses, fp32 math, block-level
// partial sums reduced by a second tiny kernel so results are deterministic.
#include "b2u_internal.h"
#include "b2u_ptx.cuh"

namespace b2u {

#define B2U_CHECK_LAUNCH(name)                                                                           \
  do {                                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                                \
    if (e__ != cudaSuccess) return b2u::set_error(B2U_ERR_CUDA, name " launch: %s", cudaGetErrorString(e__)); \
    b2u::note_launch();                                                                                  \
  } while (0)

constexpr int kMaxCls = 32;        // the register-array kernels below; wider heads take the *_wide kernels
constexpr int kMaxClsWide = 255;   // uint8 masks: the reference's ignore label (= num_classes) must still fit a byte
#ifndef B2U_FP32_VALIDATION
constexpr int kHeadK = 64;
#endif

#ifndef B2U_FP32_VALIDATION   // the fp32 validation build (validation_fp32.cu) brings its own head / operand kernels
// ------------------------------------------------------------------------------------------
// head forward: one thread per pixel; x row (64 bf16 = 128 B) in registers, weights in smem
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
head_fwd_kernel(const uint4* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                float* __restrict__ logits, long long HW, long long P, int ncls) {
  __shared__ float sw[kMaxCls * kHeadK];
  __shared__ float sb[kMaxCls];
  for (int i = threadIdx.x; i < ncls * kHeadK; i += blockDim.x) sw[i] = w[i];
  for (int i = threadIdx.x; i < ncls; i += blockDim.x) sb[i] = b ? b[i] : 0.f;
  __syncthreads();
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  float xv[kHeadK];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const uint4 v = __ldg(x + p * 8 + q);
    xv[q * 8 + 0] = bf16_lo(v.x); xv[q * 8 + 1] = bf16_hi(v.x); xv[q * 8 + 2] = bf16_lo(v.y); xv[q * 8 + 3] = bf16_hi(v.y);
    xv[q * 8 + 4] = bf16_lo(v.z); xv[q * 8 + 5] = bf16_hi(v.z); xv[q * 8 + 6] = bf16_lo(v.w); xv[q * 8 + 7] = bf16_hi(v.w);
  }
  const long long n = p / HW, hw = p % HW;
  float* out = logits + n * ncls * HW + hw;
  for (int c = 0; c < ncls; ++c) {
    float acc = sb[c];
    const float4* wr = reinterpret_cast<const float4*>(sw + c * kHeadK);
#pragma unroll
    for (int k = 0; k < kHeadK / 4; ++k) {
      const float4 ww = wr[k];
      acc = fmaf(xv[4 * k + 0], ww.x, acc); acc = fmaf(xv[4 * k + 1], ww.y, acc);
      acc = fmaf(xv[4 * k + 2], ww.z, acc); acc = fmaf(xv[4 * k + 3], ww.w, acc);
    }
    out[c * HW] = acc;
  }
}

// head backward, data part: dx[p][k] = (x[p][k] > 0) * sum_c g[p][c] W[c][k]
__global__ void __launch_bounds__(128)
head_dgrad_kernel(const float* __restrict__ dlogits, const uint4* __restrict__ x, const float* __restrict__ w,
                  uint4* __restrict__ dx, long long HW, long long P, int ncls, int relu_mask) {
  __shared__ float sw[kMaxCls * kHeadK];
  for (int i = threadIdx.x; i < ncls * kHeadK; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const long long n = p / HW, hw = p % HW;
  const float* g = dlogits + n * ncls * HW + hw;
  float acc[kHeadK];
#pragma unroll
  for (int k = 0; k < kHeadK; ++k) acc[k] = 0.f;
  for (int c = 0; c < ncls; ++c) {
    const float gc = __ldg(g + c * HW);
    const float4* wr = reinterpret_cast<const float4*>(sw + c * kHeadK);
#pragma unroll
    for (int k = 0; k < kHeadK / 4; ++k) {
      const float4 ww = wr[k];
      acc[4 * k + 0] = fmaf(gc, ww.x, acc[4 * k + 0]); acc[4 * k + 1] = fmaf(gc, ww.y, acc[4 * k + 1]);
      acc[4 * k + 2] = fmaf(gc, ww.z, acc[4 * k + 2]); acc[4 * k + 3] = fmaf(gc, ww.w, acc[4 * k + 3]);
    }
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    float o[8];
    if (relu_mask) {
      const uint4 v = __ldg(x + p * 8 + q);
      const float m[8] = {bf16_lo(v.x), bf16_hi(v.x), bf16_lo(v.y), bf16_hi(v.y),
                          bf16_lo(v.z), bf16_hi(v.z), bf16_lo(v.w), bf16_hi(v.w)};
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = m[e] > 0.f ? acc[q * 8 + e] : 0.f;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = acc[q * 8 + e];
    }
    uint4 r;
    r.x = pack_bf16x2(o[0], o[1]); r.y = pack_bf16x2(o[2], o[3]); r.z = pack_bf16x2(o[4], o[5]); r.w = pack_bf16x2(o[6], o[7]);
    dx[p * 8 + q] = r;
  }
}

// head backward, weight part: partial[block][c][k] = sum over the block's pixels of g[p][c] * x[p][k];
// column 64 of each row holds sum g (bias gradient).  Block = 128 threads, pixel tiles of 64.
constexpr int kHwTile = 64;
__global__ void __launch_bounds__(128)
head_wgrad_kernel(const float* __restrict__ dlogits, const __nv_bfloat16* __restrict__ x, float* __restrict__ partial,
                  long long HW, long long P, int ncls) {
  __shared__ float sg[kMaxCls][kHwTile];          // [class][pixel]
  __shared__ float sx[kHwTile][kHeadK + 4];       // [pixel][k]
  const int tid = threadIdx.x;
  const int kg = tid & 15;        // 16 groups of 4 k
  const int cg = tid >> 4;        // 8 groups of 4 classes (ncls <= 32)
  float acc[4][4];
  float bacc[4] = {0, 0, 0, 0};
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const long long ntiles = (P + kHwTile - 1) / kHwTile;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long p0 = tile * kHwTile;
    for (int i = tid; i < kMaxCls * kHwTile; i += 128) {
      const int c = i / kHwTile, pp = i % kHwTile;
      const long long p = p0 + pp;
      float v = 0.f;
      if (c < ncls && p < P) { const long long n = p / HW, hw = p % HW; v = __ldg(dlogits + (n * ncls + c) * HW + hw); }
      sg[c][pp] = v;
    }
    for (int i = tid; i < kHwTile * kHeadK / 2; i += 128) {
      const int pp = i / (kHeadK / 2), k2 = i % (kHeadK / 2);
      const long long p = p0 + pp;
      uint32_t v = 0;
      if (p < P) v = __ldg(reinterpret_cast<const uint32_t*>(x) + p * (kHeadK / 2) + k2);
      sx[pp][2 * k2] = bf16_lo(v); sx[pp][2 * k2 + 1] = bf16_hi(v);
    }
    __syncthreads();
#pragma unroll 4
    for (int pp = 0; pp < kHwTile; ++pp) {
      const float4 xv = *reinterpret_cast<const float4*>(&sx[pp][kg * 4]);
      float g[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) g[i] = sg[cg * 4 + i][pp];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[i][0] = fmaf(g[i], xv.x, acc[i][0]); acc[i][1] = fmaf(g[i], xv.y, acc[i][1]);
        acc[i][2] = fmaf(g[i], xv.z, acc[i][2]); acc[i][3] = fmaf(g[i], xv.w, acc[i][3]);
        if (kg == 0) bacc[i] += g[i];
      }
    }
    __syncthreads();
  }
  float* out = partial + static_cast<size_t>(blockIdx.x) * kMaxCls * (kHeadK + 1);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = cg * 4 + i;
#pragma unroll
    for (int j = 0; j < 4; ++j) out[c * (kHeadK + 1) + kg * 4 + j] = acc[i][j];
    if (kg == 0) out[c * (kHeadK + 1) + kHeadK] = bacc[i];
  }
}
__global__ void head_wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, float* __restrict__ db,
                                         int blocks, int ncls) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ncls * (kHeadK + 1)) return;
  const int c = i / (kHeadK + 1), k = i % (kHeadK + 1);
  float acc = 0.f;
  for (int b = 0; b < blocks; ++b) acc += partial[static_cast<size_t>(b) * kMaxCls * (kHeadK + 1) + c * (kHeadK + 1) + k];
  if (k < kHeadK) { if (dw) dw[c * kHeadK + k] = acc; }
  else if (db) db[c] = acc;
}

// ---- more than 32 classes: the same three computations, the weights staged through shared memory 32 classes at a time
__global__ void __launch_bounds__(128)
head_fwd_wide_kernel(const uint4* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                     float* __restrict__ logits, long long HW, long long P, int ncls) {
  __shared__ float sw[kMaxCls * kHeadK];
  __shared__ float sb[kMaxCls];
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const bool live = p < P;
  float xv[kHeadK];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const uint4 v = live ? __ldg(x + p * 8 + q) : make_uint4(0u, 0u, 0u, 0u);
    xv[q * 8 + 0] = bf16_lo(v.x); xv[q * 8 + 1] = bf16_hi(v.x); xv[q * 8 + 2] = bf16_lo(v.y); xv[q * 8 + 3] = bf16_hi(v.y);
    xv[q * 8 + 4] = bf16_lo(v.z); xv[q * 8 + 5] = bf16_hi(v.z); xv[q * 8 + 6] = bf16_lo(v.w); xv[q * 8 + 7] = bf16_hi(v.w);
  }
  const long long n = live ? p / HW : 0, hw = live ? p % HW : 0;
  float* out = logits + n * ncls * HW + hw;
  for (int c0 = 0; c0 < ncls; c0 += kMaxCls) {
    const int cn = ncls - c0 < kMaxCls ? ncls - c0 : kMaxCls;
    __syncthreads();
    for (int i = threadIdx.x; i < cn * kHeadK; i += blockDim.x) sw[i] = w[c0 * kHeadK + i];
    for (int i = threadIdx.x; i < cn; i += blockDim.x) sb[i] = b ? b[c0 + i] : 0.f;
    __syncthreads();
    if (!live) continue;
    for (int c = 0; c < cn; ++c) {
      float acc = sb[c];
      const float4* wr = reinterpret_cast<const float4*>(sw + c * kHeadK);
#pragma unroll
      for (int k = 0; k < kHeadK / 4; ++k) {
        const float4 ww = wr[k];
        acc = fmaf(xv[4 * k + 0], ww.x, acc); acc = fmaf(xv[4 * k + 1], ww.y, acc);
        acc = fmaf(xv[4 * k + 2], ww.z, acc); acc = fmaf(xv[4 * k + 3], ww.w, acc);
      }
      out[(c0 + c) * HW] = acc;
    }
  }
}

__global__ void __launch_bounds__(128)
head_dgrad_wide_kernel(const float* __restrict__ dlogits, const uint4* __restrict__ x, const float* __restrict__ w,
                       uint4* __restrict__ dx, long long HW, long long P, int ncls, int relu_mask) {
  __shared__ float sw[kMaxCls * kHeadK];
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const bool live = p < P;
  const long long n = live ? p / HW : 0, hw = live ? p % HW : 0;
  const float* g = dlogits + n * ncls * HW + hw;
  float acc[kHeadK];
#pragma unroll
  for (int k = 0; k < kHeadK; ++k) acc[k] = 0.f;
  for (int c0 = 0; c0 < ncls; c0 += kMaxCls) {
    const int cn = ncls - c0 < kMaxCls ? ncls - c0 : kMaxCls;
    __syncthreads();
    for (int i = threadIdx.x; i < cn * kHeadK; i += blockDim.x) sw[i] = w[c0 * kHeadK + i];
    __syncthreads();
    if (!live) continue;
    for (int c = 0; c < cn; ++c) {
      const float gc = __ldg(g + (c0 + c) * HW);
      const float4* wr = reinterpret_cast<const float4*>(sw + c * kHeadK);
#pragma unroll
      for (int k = 0; k < kHeadK / 4; ++k) {
        const float4 ww = wr[k];
        acc[4 * k + 0] = fmaf(gc, ww.x, acc[4 * k + 0]); acc[4 * k + 1] = fmaf(gc, ww.y, acc[4 * k + 1]);
        acc[4 * k + 2] = fmaf(gc, ww.z, acc[4 * k + 2]); acc[4 * k + 3] = fmaf(gc, ww.w, acc[4 * k + 3]);
      }
    }
  }
  if (!live) return;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    float o[8];
    if (relu_mask) {
      const uint4 v = __ldg(x + p * 8 + q);
      const float m[8] = {bf16_lo(v.x), bf16_hi(v.x), bf16_lo(v.y), bf16_hi(v.y),
                          bf16_lo(v.z), bf16_hi(v.z), bf16_lo(v.w), bf16_hi(v.w)};
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = m[e] > 0.f ? acc[q * 8 + e] : 0.f;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = acc[q * 8 + e];
    }
    uint4 r;
    r.x = pack_bf16x2(o[0], o[1]); r.y = pack_bf16x2(o[2], o[3]); r.z = pack_bf16x2(o[4], o[5]); r.w = pack_bf16x2(o[6], o[7]);
    dx[p * 8 + q] = r;
  }
}

// blockIdx.y selects the group of 32 classes; partial[(group * gridDim.x + block)][32][65] as in head_wgrad_kernel
__global__ void __launch_bounds__(128)
head_wgrad_wide_kernel(const float* __restrict__ dlogits, const __nv_bfloat16* __restrict__ x, float* __restrict__ partial,
                       long long HW, long long P, int ncls) {
  __shared__ float sg[kMaxCls][kHwTile];
  __shared__ float sx[kHwTile][kHeadK + 4];
  const int tid = threadIdx.x;
  const int kg = tid & 15;
  const int cg = tid >> 4;
  const int c0 = blockIdx.y * kMaxCls;
  float acc[4][4];
  float bacc[4] = {0, 0, 0, 0};
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const long long ntiles = (P + kHwTile - 1) / kHwTile;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long p0 = tile * kHwTile;
    for (int i = tid; i < kMaxCls * kHwTile; i += 128) {
      const int c = i / kHwTile, pp = i % kHwTile;
      const long long p = p0 + pp;
      float v = 0.f;
      if (c0 + c < ncls && p < P) { const long long n = p / HW, hw = p % HW; v = __ldg(dlogits + (n * ncls + c0 + c) * HW + hw); }
      sg[c][pp] = v;
    }
    for (int i = tid; i < kHwTile * kHeadK / 2; i += 128) {
      const int pp = i / (kHeadK / 2), k2 = i % (kHeadK / 2);
      const long long p = p0 + pp;
      uint32_t v = 0;
      if (p < P) v = __ldg(reinterpret_cast<const uint32_t*>(x) + p * (kHeadK / 2) + k2);
      sx[pp][2 * k2] = bf16_lo(v); sx[pp][2 * k2 + 1] = bf16_hi(v);
    }
    __syncthreads();
#pragma unroll 4
    for (int pp = 0; pp < kHwTile; ++pp) {
      const float4 xv = *reinterpret_cast<const float4*>(&sx[pp][kg * 4]);
      float g[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) g[i] = sg[cg * 4 + i][pp];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[i][0] = fmaf(g[i], xv.x, acc[i][0]); acc[i][1] = fmaf(g[i], xv.y, acc[i][1]);
        acc[i][2] = fmaf(g[i], xv.z, acc[i][2]); acc[i][3] = fmaf(g[i], xv.w, acc[i][3]);
        if (kg == 0) bacc[i] += g[i];
      }
    }
    __syncthreads();
  }
  float* out = partial + (static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x) * kMaxCls * (kHeadK + 1);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = cg * 4 + i;
#pragma unroll
    for (int j = 0; j < 4; ++j) out[c * (kHeadK + 1) + kg * 4 + j] = acc[i][j];
    if (kg == 0) out[c * (kHeadK + 1) + kHeadK] = bacc[i];
  }
}
__global__ void head_wgrad_wide_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, float* __restrict__ db,
                                              int blocks, int ncls) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ncls * (kHeadK + 1)) return;
  const int c = i / (kHeadK + 1), k = i % (kHeadK + 1);
  const float* src = partial + static_cast<size_t>(c / kMaxCls) * blocks * kMaxCls * (kHeadK + 1) + (c % kMaxCls) * (kHeadK + 1) + k;
  float acc = 0.f;
  for (int b = 0; b < blocks; ++b) acc += src[static_cast<size_t>(b) * kMaxCls * (kHeadK + 1)];
  if (k < kHeadK) { if (dw) dw[c * kHeadK + k] = acc; }
  else if (db) db[c] = acc;
}
#endif  // !B2U_FP32_VALIDATION

// ------------------------------------------------------------------------------------------
// losses
// ------------------------------------------------------------------------------------------
// stats layout (doubles), L = 5*C + 4:
//   [0]            sum_i w[y_i] * nll_i      (valid pixels)            -> CE numerator
//   [1]            sum_i w[y_i]                                          -> CE denominator
//   [2]            sum_i focal_i             (all pixels; ignored contribute 0)
//   [3]            pixel count
//   [4 + c]        tp_c   = sum t_ic p_ic          [4 + C + c]   P_c = sum p_ic      [4 + 2C + c] T_c = sum t_ic
//   [4 + 3C + c]   tpf_c  = sum t_ic [p_ic > thr]  [4 + 4C + c]  Pf_c = sum [p_ic > thr]
constexpr int kLossThreads = 256;

template <bool ONEHOT>
__global__ void __launch_bounds__(kLossThreads)
loss_stats_kernel(const float* __restrict__ logits, const long long* __restrict__ target, const float* __restrict__ onehot,
                  const float* __restrict__ cls_w, double* __restrict__ partial, long long HW, long long P, int C,
                  float focal_alpha, float focal_gamma, float thr) {
  __shared__ float swt[kMaxCls];
  extern __shared__ double sred[];   // [L][warps]
  for (int i = threadIdx.x; i < C; i += blockDim.x) swt[i] = cls_w ? cls_w[i] : 1.f;
  __syncthreads();
  const int L = 5 * C + 4;
  float a_ce = 0.f, a_w = 0.f, a_focal = 0.f, a_cnt = 0.f;
  float tp[kMaxCls], Ps[kMaxCls], Ts[kMaxCls], tpf[kMaxCls], Pf[kMaxCls];
#pragma unroll
  for (int c = 0; c < kMaxCls; ++c) { tp[c] = Ps[c] = Ts[c] = tpf[c] = Pf[c] = 0.f; }

  for (long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; p < P;
       p += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = p / HW, hw = p % HW;
    const float* z = logits + n * C * HW + hw;
    float v[kMaxCls];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < kMaxCls; ++c) if (c < C) { v[c] = __ldg(z + c * HW); m = fmaxf(m, v[c]); }
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxCls; ++c) if (c < C) { v[c] = __expf(v[c] - m); sum += v[c]; }
    const float inv = 1.f / sum;
    const float lse = m + logf(sum);
    long long y = target ? target[p] : -1;
    if (target && y >= 0 && y < C) {
      const float zy = __ldg(z + y * HW);
      const float nll = lse - zy;
      const float wy = swt[y];
      a_ce += wy * nll; a_w += wy;
      const float logpt = -wy * nll;
      const float pt = expf(logpt);
      a_focal += -powf(fmaxf(1.f - pt, 0.f), focal_gamma) * (focal_alpha * logpt);
    }
    a_cnt += 1.f;
#pragma unroll
    for (int c = 0; c < kMaxCls; ++c) if (c < C) {
      const float pc = v[c] * inv;
      float t;
      if (ONEHOT) t = __ldg(onehot + p * (C + 1) + c);
      else t = (y == c) ? 1.f : 0.f;
      const float hard = pc > thr ? 1.f : 0.f;
      tp[c] += t * pc; Ps[c] += pc; Ts[c] += t; tpf[c] += t * hard; Pf[c] += hard;
    }
  }
  // block reduction (fp32 per thread over <= a few hundred pixels, fp64 across threads)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  auto red = [&](float val, int slot) {
    double d = static_cast<double>(val);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
    if (lane == 0) sred[slot * nwarps + warp] = d;
  };
  red(a_ce, 0); red(a_w, 1); red(a_focal, 2); red(a_cnt, 3);
#pragma unroll
  for (int c = 0; c < kMaxCls; ++c) if (c < C) {
    red(tp[c], 4 + c); red(Ps[c], 4 + C + c); red(Ts[c], 4 + 2 * C + c); red(tpf[c], 4 + 3 * C + c); red(Pf[c], 4 + 4 * C + c);
  }
  __syncthreads();
  for (int s = threadIdx.x; s < L; s += blockDim.x) {
    double d = 0.0;
    for (int w2 = 0; w2 < nwarps; ++w2) d += sred[s * nwarps + w2];
    partial[static_cast<size_t>(blockIdx.x) * L + s] = d;
  }
}

// Label-map variant (the training loop's case): only P_c and Pf_c need a per-class register; the three sums that
// involve the pixel's own class (tp, T, tpf) go to per-warp shared-memory tables.  tp is accumulated in 2^-32
// fixed point so the result does not depend on the order in which lanes reach the table.
template <int CM>
__global__ void __launch_bounds__(kLossThreads, 2)
loss_stats_map_kernel(const float* __restrict__ logits, const long long* __restrict__ target,
                      const float* __restrict__ cls_w, double* __restrict__ partial, long long HW, long long P, int C,
                      float focal_alpha, float focal_gamma, float thr) {
  constexpr int kWarps = kLossThreads / 32;
  __shared__ float swt[kMaxCls];
  __shared__ unsigned long long s_tp[kWarps][kMaxCls];
  __shared__ unsigned int s_T[kWarps][kMaxCls], s_tpf[kWarps][kMaxCls];
  extern __shared__ double sred[];   // [2C + 4][warps]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < C; i += blockDim.x) swt[i] = cls_w ? cls_w[i] : 1.f;
  for (int i = threadIdx.x; i < kWarps * kMaxCls; i += blockDim.x) {
    (&s_tp[0][0])[i] = 0ull; (&s_T[0][0])[i] = 0u; (&s_tpf[0][0])[i] = 0u;
  }
  __syncthreads();
  float a_ce = 0.f, a_w = 0.f, a_focal = 0.f, a_cnt = 0.f;
  float Ps[CM], Pf[CM];
#pragma unroll
  for (int c = 0; c < CM; ++c) { Ps[c] = Pf[c] = 0.f; }
  const bool small = P < 0x7fffffffLL && static_cast<long long>(C) * HW < 0x7fffffffLL;

  // warp-uniform loop (every lane stays in it, `inb` guards the tail) so the class-wise aggregation below can use
  // full-warp collectives
  for (long long p0 = static_cast<long long>(blockIdx.x) * blockDim.x + warp * 32; p0 < P;
       p0 += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long p = p0 + lane;
    const bool inb = p < P;
    const long long pc_ = inb ? p : P - 1;
    // (32-bit index arithmetic whenever the plane fits: a 64-bit division and 21 64-bit multiplies per pixel were a third of
    // this kernel's instructions)
    long long n, hw;
    if (small) { const unsigned pu = static_cast<unsigned>(pc_), hwu = static_cast<unsigned>(HW); n = pu / hwu; hw = pu - static_cast<unsigned>(n) * hwu; }
    else { n = pc_ / HW; hw = pc_ % HW; }
    const float* z = logits + n * C * HW + hw;
    float v[CM];
    float m = -INFINITY;
    if (small) {
      const int hwi = static_cast<int>(HW);
#pragma unroll
      for (int c = 0; c < CM; ++c) if (c < C) { v[c] = __ldg(z + c * hwi); m = fmaxf(m, v[c]); }
    } else {
#pragma unroll
      for (int c = 0; c < CM; ++c) if (c < C) { v[c] = __ldg(z + c * HW); m = fmaxf(m, v[c]); }
    }
    const long long y64 = target[pc_];
    const bool valid = inb && y64 >= 0 && y64 < C;
    const int y = valid ? static_cast<int>(y64) : -1;
    const float zy = valid ? __ldg(z + y * HW) : 0.f;
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < CM; ++c) if (c < C) { v[c] = __expf(v[c] - m); sum += v[c]; }   // arguments <= 0: ex2.approx, <= 2 ulp near the max class
    const float inv = 1.f / sum;
    if (inb) {
#pragma unroll
      for (int c = 0; c < CM; ++c) if (c < C) {
        const float pc = v[c] * inv;
        Ps[c] += pc;
        Pf[c] += pc > thr ? 1.f : 0.f;
      }
      a_cnt += 1.f;
    }
    float py = 0.f;
    if (valid) {
      const float nll = m + logf(sum) - zy;
      const float wy = swt[y];
      a_ce += wy * nll; a_w += wy;
      if (focal_alpha != 0.f) {          // (host passes alpha = 0 when the focal term is not requested: powf / expf are ~100 instructions)
        const float logpt = -wy * nll;
        const float pt = expf(logpt);
        a_focal += -powf(fmaxf(1.f - pt, 0.f), focal_gamma) * (focal_alpha * logpt);
      }
      py = __expf(zy - m) * inv;
    }
    // own-class sums: lanes holding the same class are grouped (label maps are blob-structured, so a warp usually holds
    // one or two classes) and one lane per group updates the warp's table -- integer arithmetic, order-independent
    const unsigned gm = __match_any_sync(0xffffffffu, y);
    if (valid) {
      const unsigned fx = __reduce_add_sync(gm, __float2uint_rn(py * 16777216.f));      // 2^-24 fixed point, <= 2^29
      const unsigned hard = __popc(__ballot_sync(gm, py > thr));
      if (lane == __ffs(gm) - 1) {
        atomicAdd(&s_tp[warp][y], static_cast<unsigned long long>(fx) << 8);            // table is 2^-32 fixed point
        atomicAdd(&s_T[warp][y], static_cast<unsigned>(__popc(gm)));
        if (hard) atomicAdd(&s_tpf[warp][y], hard);
      }
    }
  }
  const int nwarps = kWarps;
  auto red = [&](float val, int slot) {
    double d = static_cast<double>(val);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
    if (lane == 0) sred[slot * nwarps + warp] = d;
  };
  red(a_ce, 0); red(a_w, 1); red(a_focal, 2); red(a_cnt, 3);
#pragma unroll
  for (int c = 0; c < CM; ++c) if (c < C) { red(Ps[c], 4 + c); red(Pf[c], 4 + C + c); }
  __syncthreads();
  const int L = 5 * C + 4;
  double* out = partial + static_cast<size_t>(blockIdx.x) * L;
  for (int sI = threadIdx.x; sI < 2 * C + 4; sI += blockDim.x) {
    double d = 0.0;
    for (int w2 = 0; w2 < nwarps; ++w2) d += sred[sI * nwarps + w2];
    if (sI < 4) out[sI] = d;
    else if (sI < 4 + C) out[4 + C + (sI - 4)] = d;              // P_c
    else out[4 + 4 * C + (sI - 4 - C)] = d;                      // Pf_c
  }
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    unsigned long long tp = 0; unsigned int T = 0, tpf = 0;
    for (int w2 = 0; w2 < nwarps; ++w2) { tp += s_tp[w2][c]; T += s_T[w2][c]; tpf += s_tpf[w2][c]; }
    out[4 + c] = static_cast<double>(tp) / 4294967296.0;         // tp_c
    out[4 + 2 * C + c] = static_cast<double>(T);                 // T_c
    out[4 + 3 * C + c] = static_cast<double>(tpf);               // tpf_c
  }
}

// out (floats): [0] CE  [1] Focal  [2] Dice loss  [3] f_score, then per class A_c (4..4+C) and B_c (4+C..4+2C)
// (Dice backward coefficients, see DESIGN.md), then [4+2C] = 1/sum_w, [4+2C+1] = 1/pixel count.
__global__ void __launch_bounds__(1024)
loss_finalize_kernel(const double* __restrict__ partial, int blocks, int C, float beta, float smooth,
                     float* __restrict__ out, double* __restrict__ stats_out) {
  extern __shared__ double tot[];            // [L] totals, then [4][L] staging
  const int L = 5 * C + 4;
  double* part = tot + L;
  // 4 lanes per slot walk the block partials with stride 4 (fixed order -> deterministic), then fold
  const int lanes = 4;
  for (int i = threadIdx.x; i < L * lanes; i += blockDim.x) {
    const int s = i % L, q = i / L;
    double d = 0.0;
    for (int b = q; b < blocks; b += lanes) d += partial[static_cast<size_t>(b) * L + s];
    part[q * L + s] = d;
  }
  __syncthreads();
  for (int s = threadIdx.x; s < L; s += blockDim.x) {
    const double d = (part[s] + part[L + s]) + (part[2 * L + s] + part[3 * L + s]);
    tot[s] = d;
    if (stats_out) stats_out[s] = d;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const double b2 = static_cast<double>(beta) * beta, a = 1.0 + b2, eps = smooth;
    out[0] = tot[1] > 0.0 ? static_cast<float>(tot[0] / tot[1]) : nanf("");
    out[1] = static_cast<float>(tot[2] / tot[3]);
    double dice = 0.0, fs = 0.0;
    for (int c = 0; c < C; ++c) {
      const double tp = tot[4 + c], Pc = tot[4 + C + c], Tc = tot[4 + 2 * C + c];
      const double D = b2 * Tc + Pc + eps;           // (1+b2)tp + b2(T-tp) + (P-tp) + eps
      dice += (a * tp + eps) / D;
      out[4 + c] = static_cast<float>(-a / (C * D));                  // A_c
      out[4 + C + c] = static_cast<float>((a * tp + eps) / (C * D * D));  // B_c
      const double tpf = tot[4 + 3 * C + c], Pf = tot[4 + 4 * C + c];
      fs += (a * tpf + eps) / (b2 * Tc + Pf + eps);
    }
    out[2] = static_cast<float>(1.0 - dice / C);
    out[3] = static_cast<float>(fs / C);
    out[4 + 2 * C] = tot[1] > 0.0 ? static_cast<float>(1.0 / tot[1]) : 0.f;
    out[4 + 2 * C + 1] = static_cast<float>(1.0 / tot[3]);
  }
}

// dlogits = g_ce * dCE/dz + g_focal * dFocal/dz + g_dice * dDice/dz   (coefficients from loss_finalize)
// NHWC64: dlogits leave as bf16 [pixel][64] (channels >= C zero) = the dz operand of the tensor-core 1x1 dgrad/wgrad
template <bool ONEHOT, bool NHWC64, int CM>
__global__ void __launch_bounds__(kLossThreads)
loss_bwd_kernel(const float* __restrict__ logits, const long long* __restrict__ target, const float* __restrict__ onehot,
                const float* __restrict__ cls_w, const float* __restrict__ fin, const float* __restrict__ gscale,
                float* __restrict__ dlogits, long long HW, long long P, int C, float focal_alpha, float focal_gamma) {
  __shared__ float swt[kMaxCls], sA[kMaxCls], sB[kMaxCls];
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    swt[i] = cls_w ? cls_w[i] : 1.f; sA[i] = fin[4 + i]; sB[i] = fin[4 + C + i];
  }
  __syncthreads();
  const float g_ce = gscale[0] * fin[4 + 2 * C];       // upstream grad / sum_w
  const float g_focal = gscale[1] * fin[4 + 2 * C + 1];  // upstream grad / pixel count
  const float g_dice = gscale[2];
  const long long p_raw = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (!NHWC64 && p_raw >= P) return;
  const bool inb = p_raw < P;                  // NHWC64: every lane stays for the warp's cooperative store
  const long long p = inb ? p_raw : P - 1;
  // 32-bit index arithmetic whenever the tensor fits (see loss_stats_map_kernel)
  const bool small = P < 0x7fffffffLL && static_cast<long long>(C) * HW < 0x7fffffffLL;
  long long n, hw;
  if (small) { const unsigned pu = static_cast<unsigned>(p), hwu = static_cast<unsigned>(HW); n = pu / hwu; hw = pu - static_cast<unsigned>(n) * hwu; }
  else { n = p / HW; hw = p % HW; }
  const float* z = logits + n * C * HW + hw;
  float* dzp = dlogits + n * C * HW + hw;
  float v[CM];
  float m = -INFINITY;
  if (small) {
    const int hwi = static_cast<int>(HW);
#pragma unroll
    for (int c = 0; c < CM; ++c) if (c < C) { v[c] = __ldg(z + c * hwi); m = fmaxf(m, v[c]); }
  } else {
#pragma unroll
    for (int c = 0; c < CM; ++c) if (c < C) { v[c] = __ldg(z + c * HW); m = fmaxf(m, v[c]); }
  }
  const long long y64 = target ? target[p] : -1;
  const bool valid = target && y64 >= 0 && y64 < C;
  const int y = valid ? static_cast<int>(y64) : -1;
  float zy = 0.f;
#pragma unroll
  for (int c = 0; c < CM; ++c) if (c < C) { if (valid && c == y) zy = v[c]; }
  float sum = 0.f;
#pragma unroll
  for (int c = 0; c < CM; ++c) if (c < C) { v[c] = __expf(v[c] - m); sum += v[c]; }   // arguments <= 0: ex2.approx, <= 2 ulp near the max class
  const float inv = 1.f / sum;
  // per-pixel scalar multiplying (p - onehot_y): CE and focal share the direction
  float k_py = 0.f;
  if (valid) {
    const float wy = swt[y];
    k_py = g_ce * wy;
    if (g_focal != 0.f) {
      const float nll = m + logf(sum) - zy;
      const float logpt = -wy * nll;
      const float pt = expf(logpt);
      const float om = fmaxf(1.f - pt, 0.f);
      // focal = -(1-pt)^g * alpha * logpt ; d/dlogpt = alpha * ( g (1-pt)^(g-1) pt logpt - (1-pt)^g )
      const float dF = focal_alpha * (focal_gamma * powf(om, focal_gamma - 1.f) * pt * logpt - powf(om, focal_gamma));
      // logpt = -wy * nll, dnll/dz = p - onehot  ->  dfocal/dz = dF * (-wy) * (p - onehot)
      k_py += g_focal * dF * (-wy);
    }
  }
  // dice: g_c = A_c t_c + B_c ; ddice/dz_k = p_k (g_k - sum_c g_c p_c)
  float gdot = 0.f;
  float t[CM];
  if (g_dice != 0.f) {
#pragma unroll
    for (int c = 0; c < CM; ++c) if (c < C) {
      if (ONEHOT) t[c] = __ldg(onehot + p * (C + 1) + c);
      else t[c] = (y == c) ? 1.f : 0.f;
      gdot += (sA[c] * t[c] + sB[c]) * (v[c] * inv);
    }
  }
  float dv[CM];
#pragma unroll
  for (int c = 0; c < CM; ++c) {
    float d = 0.f;
    if (c < C) {
      const float pc = v[c] * inv;
      d = k_py * (pc - ((valid && c == y) ? 1.f : 0.f));
      if (g_dice != 0.f) d += g_dice * pc * (sA[c] * t[c] + sB[c] - gdot);
      if (!NHWC64) dzp[c * HW] = d;
    }
    dv[c] = d;
  }
  if (NHWC64) {
    // channels [0,32): bf16(d); channels [32,64): bf16(d - hi).  The two halves meet the SAME weights in the 1x1
    // dgrad/wgrad (K resp. M is padded to 64 anyway), so the head's backward sees dlogits to ~2^-17 at no cost.
    // Each lane owns one pixel row of 128 B; the warp's 32 rows are contiguous (4 KB), so they go through a
    // warp-private shared-memory tile and leave as fully coalesced 512-byte stores.
    __shared__ uint4 tile[kLossThreads / 32][32][9];          // [warp][pixel][8 + 1 pad]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float lo[CM];
#pragma unroll
    for (int c = 0; c < CM; ++c) lo[c] = dv[c] - __bfloat162float(__float2bfloat16_rn(dv[c]));
#pragma unroll
    for (int q = 0; q < kMaxCls / 8; ++q) {
      uint4 r = make_uint4(0u, 0u, 0u, 0u), l = make_uint4(0u, 0u, 0u, 0u);
      if (q * 8 < CM) {       // classes >= CM (>= C) are zero columns
        r.x = pack_bf16x2(dv[q * 8 + 0], dv[q * 8 + 1]); r.y = pack_bf16x2(dv[q * 8 + 2], dv[q * 8 + 3]);
        r.z = pack_bf16x2(dv[q * 8 + 4], dv[q * 8 + 5]); r.w = pack_bf16x2(dv[q * 8 + 6], dv[q * 8 + 7]);
        l.x = pack_bf16x2(lo[q * 8 + 0], lo[q * 8 + 1]); l.y = pack_bf16x2(lo[q * 8 + 2], lo[q * 8 + 3]);
        l.z = pack_bf16x2(lo[q * 8 + 4], lo[q * 8 + 5]); l.w = pack_bf16x2(lo[q * 8 + 6], lo[q * 8 + 7]);
      }
      tile[warp][lane][q] = r;
      tile[warp][lane][kMaxCls / 8 + q] = l;
    }
    __syncwarp();
    const long long p_warp = p_raw - lane;                     // first pixel of this warp
    uint4* o = reinterpret_cast<uint4*>(dlogits) + p_warp * 8;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int idx = it * 32 + lane, px = idx >> 3, q = idx & 7;
      if (p_warp + px < P) o[idx] = tile[warp][px][q];
    }
  }
}

// ------------------------------------------------------------------------------------------
// losses, more than 32 classes: no per-class register arrays.  A pixel's logits are read twice (a block's 256 pixels
// span C KB, served from L2): an online pass gives the max and the sum of exponentials, a second pass forms p_c.
// ------------------------------------------------------------------------------------------
// online softmax over one pixel's classes: on return m = max_c z_c and s = sum_c exp(z_c - m)
__device__ __forceinline__ void online_max_sum(float v, float& m, float& s) {
  if (v > m) { s = s * __expf(m - v) + 1.f; m = v; }
  else s += __expf(v - m);
}

// v[i] on every lane -> lane l returns the sum over the warp of v[l] (reduce-scatter: 31 shuffles for 32 values, fixed
// order, so the sums are deterministic)
__device__ __forceinline__ float warp_transpose_sum32(float (&v)[32], int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int i = 0; i < s; ++i) {
      const float send = up ? v[i] : v[i + s];
      const float keep = up ? v[i + s] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
  return v[0];
}

// Same statistics layout as loss_stats_kernel.  A warp holds 32 pixels (one per lane); for each group of 32 classes the
// per-class sums over those pixels are transposed so lane l owns class 32g + l, and the lane adds them to its warp's
// shared-memory table (only that lane writes that entry: no atomics, fixed order).  Tables are folded in fp64 per block.
template <bool ONEHOT>
__global__ void __launch_bounds__(kLossThreads)
loss_stats_wide_kernel(const float* __restrict__ logits, const long long* __restrict__ target, const float* __restrict__ onehot,
                       const float* __restrict__ cls_w, double* __restrict__ partial, long long HW, long long P, int C,
                       float focal_alpha, float focal_gamma, float thr) {
  constexpr int kWarps = kLossThreads / 32;
  __shared__ float swt[kMaxClsWide];
  __shared__ float tab[kWarps][5 * kMaxClsWide];     // [warp][q * C + c], q = tp, P, T, tpf, Pf
  __shared__ double sred[4][kWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < C; i += blockDim.x) swt[i] = cls_w ? cls_w[i] : 1.f;
  for (int i = threadIdx.x; i < kWarps * 5 * kMaxClsWide; i += blockDim.x) (&tab[0][0])[i] = 0.f;
  __syncthreads();
  float a_ce = 0.f, a_w = 0.f, a_focal = 0.f, a_cnt = 0.f;
  float* mytab = tab[warp];
  for (long long p0 = static_cast<long long>(blockIdx.x) * blockDim.x + warp * 32; p0 < P;
       p0 += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long p = p0 + lane;
    const bool inb = p < P;
    const long long pc_ = inb ? p : P - 1;
    const long long n = pc_ / HW, hw = pc_ % HW;
    const float* z = logits + n * C * HW + hw;
    float m = -INFINITY, s = 0.f;
    for (int c = 0; c < C; ++c) online_max_sum(__ldg(z + c * HW), m, s);
    const float inv = 1.f / s;
    const long long y64 = (target && inb) ? target[pc_] : -1;
    const bool valid = y64 >= 0 && y64 < C;
    const int y = valid ? static_cast<int>(y64) : -1;
    if (valid) {
      const float nll = m + logf(s) - __ldg(z + y * HW);
      const float wy = swt[y];
      a_ce += wy * nll; a_w += wy;
      const float logpt = -wy * nll;
      const float pt = expf(logpt);
      a_focal += -powf(fmaxf(1.f - pt, 0.f), focal_gamma) * (focal_alpha * logpt);
    }
    if (inb) a_cnt += 1.f;
    for (int c0 = 0; c0 < C; c0 += 32) {
      float pc[32], t[32], v[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int c = c0 + i;
        pc[i] = (inb && c < C) ? __expf(__ldg(z + c * HW) - m) * inv : 0.f;
        if (ONEHOT) t[i] = (inb && c < C) ? __ldg(onehot + pc_ * (C + 1) + c) : 0.f;
        else t[i] = (y == c) ? 1.f : 0.f;
      }
      const int cl = c0 + lane;
      float r;
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = t[i] * pc[i];
      r = warp_transpose_sum32(v, lane);
      if (cl < C) mytab[cl] += r;
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = pc[i];
      r = warp_transpose_sum32(v, lane);
      if (cl < C) mytab[C + cl] += r;
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = t[i];
      r = warp_transpose_sum32(v, lane);
      if (cl < C) mytab[2 * C + cl] += r;
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = pc[i] > thr ? t[i] : 0.f;
      r = warp_transpose_sum32(v, lane);
      if (cl < C) mytab[3 * C + cl] += r;
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = (inb && c0 + i < C && pc[i] > thr) ? 1.f : 0.f;
      r = warp_transpose_sum32(v, lane);
      if (cl < C) mytab[4 * C + cl] += r;
    }
  }
  auto red = [&](float val, int slot) {
    double d = static_cast<double>(val);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
    if (lane == 0) sred[slot][warp] = d;
  };
  red(a_ce, 0); red(a_w, 1); red(a_focal, 2); red(a_cnt, 3);
  __syncthreads();
  const int L = 5 * C + 4;
  double* out = partial + static_cast<size_t>(blockIdx.x) * L;
  for (int sI = threadIdx.x; sI < L; sI += blockDim.x) {
    double d = 0.0;
    for (int w2 = 0; w2 < kWarps; ++w2) d += sI < 4 ? sred[sI][w2] : static_cast<double>(tab[w2][sI - 4]);
    out[sI] = d;
  }
}

// loss_bwd_kernel for more than 32 classes.  The online pass also accumulates sum_c (A_c t_c + B_c) exp(z_c - m), the
// Dice term's dot product, so the second pass can write dz_c directly.
// NHWC64: bf16 [pixel][64 G], group g = [hi(32) | lo(32)] of classes 32g .. 32g + 31 (padded classes exactly zero).
template <bool ONEHOT, bool NHWC64>
__global__ void __launch_bounds__(kLossThreads)
loss_bwd_wide_kernel(const float* __restrict__ logits, const long long* __restrict__ target, const float* __restrict__ onehot,
                     const float* __restrict__ cls_w, const float* __restrict__ fin, const float* __restrict__ gscale,
                     void* __restrict__ dlogits, long long HW, long long P, int C, float focal_alpha, float focal_gamma) {
  __shared__ float swt[kMaxClsWide], sA[kMaxClsWide], sB[kMaxClsWide];
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    swt[i] = cls_w ? cls_w[i] : 1.f; sA[i] = fin[4 + i]; sB[i] = fin[4 + C + i];
  }
  __syncthreads();
  const float g_ce = gscale[0] * fin[4 + 2 * C];
  const float g_focal = gscale[1] * fin[4 + 2 * C + 1];
  const float g_dice = gscale[2];
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const long long n = p / HW, hw = p % HW;
  const float* z = logits + n * C * HW + hw;
  const long long y64 = target ? target[p] : -1;
  const bool valid = target && y64 >= 0 && y64 < C;
  const int y = valid ? static_cast<int>(y64) : -1;
  auto tgt = [&](int c) -> float {
    if (ONEHOT) return __ldg(onehot + p * (C + 1) + c);
    return c == y ? 1.f : 0.f;
  };
  float m = -INFINITY, s = 0.f, gs = 0.f;
  if (g_dice != 0.f) {
    for (int c = 0; c < C; ++c) {
      const float v = __ldg(z + c * HW), gc = sA[c] * tgt(c) + sB[c];
      if (v > m) { const float r = __expf(m - v); s = s * r + 1.f; gs = gs * r + gc; m = v; }
      else { const float e = __expf(v - m); s += e; gs = fmaf(gc, e, gs); }
    }
  } else {
    for (int c = 0; c < C; ++c) online_max_sum(__ldg(z + c * HW), m, s);
  }
  const float inv = 1.f / s;
  const float gdot = gs * inv;
  float k_py = 0.f;
  if (valid) {
    const float wy = swt[y];
    k_py = g_ce * wy;
    if (g_focal != 0.f) {
      const float nll = m + logf(s) - __ldg(z + y * HW);
      const float logpt = -wy * nll;
      const float pt = expf(logpt);
      const float om = fmaxf(1.f - pt, 0.f);
      const float dF = focal_alpha * (focal_gamma * powf(om, focal_gamma - 1.f) * pt * logpt - powf(om, focal_gamma));
      k_py += g_focal * dF * (-wy);
    }
  }
  auto dz = [&](int c) -> float {
    const float pc = __expf(__ldg(z + c * HW) - m) * inv;
    float d = k_py * (pc - (c == y ? 1.f : 0.f));
    if (g_dice != 0.f) d += g_dice * pc * (sA[c] * tgt(c) + sB[c] - gdot);
    return d;
  };
  if (!NHWC64) {
    float* dzp = static_cast<float*>(dlogits) + n * C * HW + hw;
    for (int c = 0; c < C; ++c) dzp[c * HW] = dz(c);
  } else {
    const int G = (C + 31) / 32;
    uint4* row = static_cast<uint4*>(dlogits) + p * 8 * G;
    for (int g = 0; g < G; ++g) {
      float d[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) d[i] = 32 * g + i < C ? dz(32 * g + i) : 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 h, l;
        float lo[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) lo[e] = d[q * 8 + e] - __bfloat162float(__float2bfloat16_rn(d[q * 8 + e]));
        h.x = pack_bf16x2(d[q * 8 + 0], d[q * 8 + 1]); h.y = pack_bf16x2(d[q * 8 + 2], d[q * 8 + 3]);
        h.z = pack_bf16x2(d[q * 8 + 4], d[q * 8 + 5]); h.w = pack_bf16x2(d[q * 8 + 6], d[q * 8 + 7]);
        l.x = pack_bf16x2(lo[0], lo[1]); l.y = pack_bf16x2(lo[2], lo[3]); l.z = pack_bf16x2(lo[4], lo[5]); l.w = pack_bf16x2(lo[6], lo[7]);
        row[8 * g + q] = h;
        row[8 * g + 4 + q] = l;
      }
    }
  }
}

#ifndef B2U_FP32_VALIDATION
// The tensor-core head works on G = ceil(C / 32) groups of 64 columns; group g covers classes 32g .. 32g + 31 as
// [hi(32) | lo(32)].
// final.weight [C][64] fp32 -> dgrad operand wd[ci][co] bf16, 64 x 64G: columns [64g, 64g + 32) and [64g + 32, 64g + 64)
// both hold the weights of classes 32g.. (they multiply the hi and lo halves of the split dlogits), classes >= C are zero
__global__ void pack_head_dgrad_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wd, int C) {
  const int cols = 64 * ((C + kMaxCls - 1) / kMaxCls);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * cols) return;
  const int ci = i / cols, col = i % cols, co = (col / 64) * kMaxCls + (col % 64) % kMaxCls;
  wd[i] = __float2bfloat16_rn(co < C ? w[co * 64 + ci] : 0.f);
}

// final.weight [C][64] fp32 -> fprop operand wf[co'][k] bf16, 64G x 64: in group g, rows [64g, 64g + 32) = bf16(W) and rows
// [64g + 32, 64g + 64) = the bf16 remainder W - bf16(W) of classes 32g..; the head epilogue adds the two halves (classes
// >= C are zero rows)
__global__ void pack_head_fprop_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wf, int C) {
  const int rows = 64 * ((C + kMaxCls - 1) / kMaxCls);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * 64) return;
  const int co = i / 64, k = i % 64, r = co % 64, c = (co / 64) * kMaxCls + r % kMaxCls;
  float v = 0.f;
  if (c < C) {
    const float full = w[c * 64 + k];
    const float hi = __bfloat162float(__float2bfloat16_rn(full));
    v = r < kMaxCls ? hi : full - hi;
  }
  wf[i] = __float2bfloat16_rn(v);
}
#endif  // !B2U_FP32_VALIDATION

// arg-max over classes (lowest index on ties, like numpy/torch): logits NCHW fp32 -> uint8 mask [N,H,W]
__global__ void argmax_u8_kernel(const float* __restrict__ logits, uint8_t* __restrict__ mask, long long HW, long long P, int C) {
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const long long n = p / HW, hw = p % HW;
  const float* z = logits + n * C * HW + hw;
  float best = __ldg(z); int arg = 0;
  for (int c = 1; c < C; ++c) { const float v = __ldg(z + c * HW); if (v > best) { best = v; arg = c; } }
  mask[p] = static_cast<uint8_t>(arg);
}

// Inference tail of the reference's predictor (unet.py:135-148, 324-340): softmax over classes, crop of the letterbox
// bars, cv2.resize(pr, (w, h), INTER_LINEAR) of the probabilities back to the original image size, argmax -- fused:
// one thread per output pixel interpolates the softmax of its 4 source pixels and keeps the best class, so only a
// uint8 mask ever leaves the GPU.  cv2's float INTER_LINEAR: f = (d + 0.5) * in/out - 0.5, s = floor(f), f -= s;
// s < 0 -> (s, f) = (0, 0); s >= in - 1 -> (s, f) = (in - 1, 0) (second tap clamped).
// The per-pixel bodies are shared by the single-crop kernels and the batched kernel (one crop and output size per image),
// so both give the same class for the same pixel.
struct SraTaps {
  size_t o[4];       // offsets of the 4 source pixels inside a class plane
  float wgt[4];      // their bilinear weights
};

__device__ __forceinline__ SraTaps sra_taps(int W, int cy, int cx, int ch, int cw, int x, int y, float sy, float sx) {
  float fy = (y + 0.5f) * sy - 0.5f, fx = (x + 0.5f) * sx - 0.5f;
  int y0 = static_cast<int>(floorf(fy)), x0 = static_cast<int>(floorf(fx));
  fy -= y0; fx -= x0;
  if (y0 < 0) { y0 = 0; fy = 0.f; }
  if (y0 >= ch - 1) { y0 = ch - 1; fy = 0.f; }
  if (x0 < 0) { x0 = 0; fx = 0.f; }
  if (x0 >= cw - 1) { x0 = cw - 1; fx = 0.f; }
  const int y1 = y0 + 1 < ch ? y0 + 1 : ch - 1, x1 = x0 + 1 < cw ? x0 + 1 : cw - 1;
  SraTaps t;
  t.o[0] = static_cast<size_t>(cy + y0) * W + cx + x0; t.o[1] = static_cast<size_t>(cy + y0) * W + cx + x1;
  t.o[2] = static_cast<size_t>(cy + y1) * W + cx + x0; t.o[3] = static_cast<size_t>(cy + y1) * W + cx + x1;
  t.wgt[0] = (1.f - fy) * (1.f - fx); t.wgt[1] = (1.f - fy) * fx; t.wgt[2] = fy * (1.f - fx); t.wgt[3] = fy * fx;
  return t;
}

// class of one output pixel, C <= CM <= 32; base = the image's logits [C][H][W]
template <int CM>
__device__ __forceinline__ int sra_pixel(const float* __restrict__ base, size_t plane, int C, const SraTaps& tp) {
  float acc[CM];
#pragma unroll
  for (int c = 0; c < CM; ++c) acc[c] = 0.f;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    float v[CM];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < CM; ++c) if (c < C) { v[c] = __ldg(base + c * plane + tp.o[t]); m = fmaxf(m, v[c]); }
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < CM; ++c) if (c < C) { v[c] = __expf(v[c] - m); sum += v[c]; }   // arguments <= 0: ex2.approx, <= 2 ulp near the max class
    const float k = tp.wgt[t] / sum;
#pragma unroll
    for (int c = 0; c < CM; ++c) if (c < C) acc[c] = fmaf(k, v[c], acc[c]);
  }
  float best = acc[0]; int arg = 0;
#pragma unroll
  for (int c = 1; c < CM; ++c) if (c < C && acc[c] > best) { best = acc[c]; arg = c; }
  return arg;
}

// the same for more than 32 classes, without per-class arrays: loop 1 gives each tap's max and sum (the same max-then-sum
// order as sra_pixel), loop 2 interpolates each class's probability and keeps a running arg-max (strict >, so the lowest
// index wins ties)
__device__ __forceinline__ int sra_pixel_wide(const float* __restrict__ base, size_t plane, int C, const SraTaps& tp) {
  float m[4], k[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    m[t] = -INFINITY;
    for (int c = 0; c < C; ++c) m[t] = fmaxf(m[t], __ldg(base + c * plane + tp.o[t]));
    float sum = 0.f;
    for (int c = 0; c < C; ++c) sum += __expf(__ldg(base + c * plane + tp.o[t]) - m[t]);
    k[t] = tp.wgt[t] / sum;
  }
  float best = -INFINITY; int arg = 0;
  for (int c = 0; c < C; ++c) {
    float acc = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) acc = fmaf(k[t], __expf(__ldg(base + c * plane + tp.o[t]) - m[t]), acc);
    if (c == 0 || acc > best) { best = acc; arg = c; }
  }
  return arg;
}

// CM = 0: the wide body (the batched kernel's dispatch)
template <int CM>
__device__ __forceinline__ int sra_class(const float* __restrict__ base, size_t plane, int C, const SraTaps& tp) {
  if constexpr (CM == 0) return sra_pixel_wide(base, plane, C, tp);
  else return sra_pixel<CM>(base, plane, C, tp);
}

template <int CM>
__global__ void __launch_bounds__(128)
softmax_resize_argmax_kernel(const float* __restrict__ logits, uint8_t* __restrict__ mask, int C, int H, int W, int cy,
                             int cx, int ch, int cw, int oh, int ow, float sy, float sx) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, n = blockIdx.z;
  if (x >= ow) return;
  const size_t plane = static_cast<size_t>(H) * W;
  const SraTaps tp = sra_taps(W, cy, cx, ch, cw, x, y, sy, sx);
  mask[(static_cast<size_t>(n) * oh + y) * ow + x] =
      static_cast<uint8_t>(sra_pixel<CM>(logits + static_cast<size_t>(n) * C * plane, plane, C, tp));
}

__global__ void __launch_bounds__(128)
softmax_resize_argmax_wide_kernel(const float* __restrict__ logits, uint8_t* __restrict__ mask, int C, int H, int W, int cy,
                                  int cx, int ch, int cw, int oh, int ow, float sy, float sx) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, n = blockIdx.z;
  if (x >= ow) return;
  const size_t plane = static_cast<size_t>(H) * W;
  const SraTaps tp = sra_taps(W, cy, cx, ch, cw, x, y, sy, sx);
  mask[(static_cast<size_t>(n) * oh + y) * ow + x] =
      static_cast<uint8_t>(sra_pixel_wide(logits + static_cast<size_t>(n) * C * plane, plane, C, tp));
}

// one image of a batched tail call (32 bytes, include/b2u.h)
struct SraItem {
  int cy, cx, ch, cw, oh, ow;
  long long mask_off;   // byte offset of the image's [oh][ow] mask in the flat output
};
static_assert(sizeof(SraItem) == 32, "SraItem is part of the ABI");

// blockIdx.z = image; rows and columns are strided over the grid, which is sized for the largest image of the batch
template <int CM>
__global__ void __launch_bounds__(128)
softmax_resize_argmax_batch_kernel(const float* __restrict__ logits, const SraItem* __restrict__ items,
                                   uint8_t* __restrict__ masks, int C, int H, int W) {
  const SraItem it = items[blockIdx.z];
  if (it.cy < 0 || it.cx < 0 || it.ch <= 0 || it.cw <= 0 || it.cy + it.ch > H || it.cx + it.cw > W) return;
  const float sy = static_cast<float>(__ddiv_rn(static_cast<double>(it.ch), static_cast<double>(it.oh)));
  const float sx = static_cast<float>(__ddiv_rn(static_cast<double>(it.cw), static_cast<double>(it.ow)));
  const size_t plane = static_cast<size_t>(H) * W;
  const float* base = logits + static_cast<size_t>(blockIdx.z) * C * plane;
  uint8_t* mask = masks + it.mask_off;
  for (int y = blockIdx.y; y < it.oh; y += gridDim.y)
    for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < it.ow; x += gridDim.x * blockDim.x)
      mask[static_cast<size_t>(y) * it.ow + x] =
          static_cast<uint8_t>(sra_class<CM>(base, plane, C, sra_taps(W, it.cy, it.cx, it.ch, it.cw, x, y, sy, sx)));
}

}  // namespace b2u

extern "C" {
using namespace b2u;

#ifndef B2U_FP32_VALIDATION
int b2u_head_fwd(const void* x, const float* w, const float* b, float* logits, int N, int H, int W, int Cin, int ncls,
                 void* stream) {
  if (Cin != kHeadK || ncls <= 0 || ncls > kMaxClsWide) return set_error(B2U_ERR_SHAPE, "head_fwd: needs Cin == 64 and 1 <= classes <= 255 (got %d, %d)", Cin, ncls);
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "head_fwd: empty tensor");
  const long long HW = static_cast<long long>(H) * W, P = HW * N;
  const unsigned grid = static_cast<unsigned>((P + 127) / 128);
  if (ncls <= kMaxCls)
    head_fwd_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const uint4*>(x), w, b, logits, HW, P, ncls);
  else
    head_fwd_wide_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const uint4*>(x), w, b, logits, HW, P, ncls);
  B2U_CHECK_LAUNCH("head_fwd");
  return 0;
}

// workspace of b2u_head_bwd: one [32][65] fp32 partial per block and group of 32 classes
size_t b2u_head_bwd_workspace_cls(int ncls) {
  const int groups = ncls > kMaxCls ? (ncls + kMaxCls - 1) / kMaxCls : 1;
  return static_cast<size_t>(4 * 148) * groups * kMaxCls * (kHeadK + 1) * sizeof(float);
}
size_t b2u_head_bwd_workspace(void) { return b2u_head_bwd_workspace_cls(kMaxCls); }   // enough for up to 32 classes

// dx may be NULL (frozen everything below); dw/db may be NULL.
int b2u_head_bwd(const float* dlogits, const void* x, const float* w, void* dx, float* dw, float* db, void* ws,
                 size_t ws_bytes, int N, int H, int W, int Cin, int ncls, int relu_mask, void* stream) {
  if (Cin != kHeadK || ncls <= 0 || ncls > kMaxClsWide) return set_error(B2U_ERR_SHAPE, "head_bwd: needs Cin == 64 and 1 <= classes <= 255");
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "head_bwd: empty tensor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long HW = static_cast<long long>(H) * W, P = HW * N;
  const bool wide = ncls > kMaxCls;
  if (dx) {
    const unsigned grid = static_cast<unsigned>((P + 127) / 128);
    if (!wide)
      head_dgrad_kernel<<<grid, 128, 0, st>>>(dlogits, static_cast<const uint4*>(x), w, static_cast<uint4*>(dx), HW, P, ncls, relu_mask);
    else
      head_dgrad_wide_kernel<<<grid, 128, 0, st>>>(dlogits, static_cast<const uint4*>(x), w, static_cast<uint4*>(dx), HW, P, ncls, relu_mask);
    B2U_CHECK_LAUNCH("head_dgrad");
  }
  if (dw || db) {
    const int blocks = 4 * 148;
    if (!ws || ws_bytes < b2u_head_bwd_workspace_cls(ncls)) return set_error(B2U_ERR_ARG, "head_bwd: workspace too small");
    if (!wide) {
      head_wgrad_kernel<<<blocks, 128, 0, st>>>(dlogits, static_cast<const __nv_bfloat16*>(x), static_cast<float*>(ws), HW, P, ncls);
      B2U_CHECK_LAUNCH("head_wgrad");
      head_wgrad_reduce_kernel<<<(ncls * (kHeadK + 1) + 127) / 128, 128, 0, st>>>(static_cast<const float*>(ws), dw, db, blocks, ncls);
    } else {
      const dim3 grid(blocks, (ncls + kMaxCls - 1) / kMaxCls);
      head_wgrad_wide_kernel<<<grid, 128, 0, st>>>(dlogits, static_cast<const __nv_bfloat16*>(x), static_cast<float*>(ws), HW, P, ncls);
      B2U_CHECK_LAUNCH("head_wgrad");
      head_wgrad_wide_reduce_kernel<<<(ncls * (kHeadK + 1) + 127) / 128, 128, 0, st>>>(static_cast<const float*>(ws), dw, db, blocks, ncls);
    }
    B2U_CHECK_LAUNCH("head_wgrad_reduce");
  }
  return 0;
}

#endif  // !B2U_FP32_VALIDATION

static const int kLossBlocks = 4 * 148;
size_t b2u_loss_workspace(int C) { return static_cast<size_t>(kLossBlocks) * (5 * C + 4) * sizeof(double); }
int b2u_loss_out_len(int C) { return 4 + 2 * C + 2; }

// target: int64 [N,H,W] (values outside [0,C) are ignored by CE/Focal and count as "no class" for Dice when
// onehot == NULL); onehot: optional fp32 [N,H,W,C+1] exactly as the reference's Dice_loss/f_score receive it.
// out: b2u_loss_out_len(C) floats (device); stats (optional): 5C+4 doubles (device).
int b2u_loss_fwd(const float* logits, const long long* target, const float* onehot, const float* cls_w, float* out,
                 double* stats, void* ws, size_t ws_bytes, int N, int C, int H, int W, float beta, float smooth,
                 float focal_alpha, float focal_gamma, float thr, void* stream) {
  if (C <= 0 || C > kMaxClsWide) return set_error(B2U_ERR_SHAPE, "loss: 1 <= classes <= 255 (got %d)", C);
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "loss: empty tensor");
  if (!ws || ws_bytes < b2u_loss_workspace(C)) return set_error(B2U_ERR_ARG, "loss: workspace too small");
  if (!target && !onehot) return set_error(B2U_ERR_ARG, "loss: need a target map or a one-hot tensor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long HW = static_cast<long long>(H) * W, P = HW * N;
  const int L = 5 * C + 4;
  long long want = (P + kLossThreads - 1) / kLossThreads;
  const int blocks = static_cast<int>(want < kLossBlocks ? want : kLossBlocks);
  const size_t sm = static_cast<size_t>(L) * (kLossThreads / 32) * sizeof(double);
  const size_t fin_sm = 5 * L * sizeof(double);
  if (fin_sm > 48 * 1024) {        // from C = 245 on the finalize's staging passes the default dynamic shared-memory limit
    static bool attr_done[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !attr_done[dev]) {
      const cudaError_t e = cudaFuncSetAttribute(loss_finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 static_cast<int>(5 * (5 * kMaxClsWide + 4) * sizeof(double)));
      if (e != cudaSuccess) return set_error(B2U_ERR_CUDA, "loss: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      if (dev >= 0 && dev < 64) attr_done[dev] = true;
    }
  }
  if (C > kMaxCls) {
    if (onehot)
      loss_stats_wide_kernel<true><<<blocks, kLossThreads, 0, st>>>(logits, target, onehot, cls_w, static_cast<double*>(ws), HW, P, C,
                                                                    focal_alpha, focal_gamma, thr);
    else
      loss_stats_wide_kernel<false><<<blocks, kLossThreads, 0, st>>>(logits, target, nullptr, cls_w, static_cast<double*>(ws), HW, P, C,
                                                                     focal_alpha, focal_gamma, thr);
  } else if (onehot) {
    loss_stats_kernel<true><<<blocks, kLossThreads, sm, st>>>(logits, target, onehot, cls_w, static_cast<double*>(ws), HW, P, C,
                                                              focal_alpha, focal_gamma, thr);
  } else {
    // class loops are unrolled to the smallest bucket >= C (a runtime bound would run all 32 predicated iterations)
    const size_t smm = static_cast<size_t>(2 * C + 4) * (kLossThreads / 32) * sizeof(double);
#define B2U_STATS(CM_) loss_stats_map_kernel<CM_><<<blocks, kLossThreads, smm, st>>>( \
        logits, target, cls_w, static_cast<double*>(ws), HW, P, C, focal_alpha, focal_gamma, thr)
    if (C <= 8) B2U_STATS(8); else if (C <= 16) B2U_STATS(16); else if (C <= 24) B2U_STATS(24); else B2U_STATS(32);
#undef B2U_STATS
  }
  B2U_CHECK_LAUNCH("loss_stats");
  loss_finalize_kernel<<<1, 1024, fin_sm, st>>>(static_cast<const double*>(ws), blocks, C, beta, smooth, out, stats);
  B2U_CHECK_LAUNCH("loss_finalize");
  return 0;
}

// fin: the `out` vector of b2u_loss_fwd; gscale: 3 floats on device = upstream gradients of (CE, Focal, Dice)
// out_mode 0: dlogits fp32 NCHW [N,C,H,W]; 1: bf16 NHWC [N,H,W,64 G], G = ceil(C / 32), group g = [hi(32) | lo(32)] of
// classes 32g.. with padded classes zero (feeds b2u_conv_dgrad/wgrad, taps=1)
int b2u_loss_bwd(const float* logits, const long long* target, const float* onehot, const float* cls_w, const float* fin,
                 const float* gscale, void* dlogits, int out_mode, int N, int C, int H, int W, float focal_alpha,
                 float focal_gamma, void* stream) {
  if (C <= 0 || C > kMaxClsWide) return set_error(B2U_ERR_SHAPE, "loss_bwd: 1 <= classes <= 255");
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "loss_bwd: empty tensor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long HW = static_cast<long long>(H) * W, P = HW * N;
  const unsigned blocks = static_cast<unsigned>((P + kLossThreads - 1) / kLossThreads);
  if (C > kMaxCls) {
#define B2U_LBWDW(OH_, NH_) loss_bwd_wide_kernel<OH_, NH_><<<blocks, kLossThreads, 0, st>>>( \
      logits, target, onehot, cls_w, fin, gscale, dlogits, HW, P, C, focal_alpha, focal_gamma)
    if (out_mode == 1) {
#ifdef B2U_FP32_VALIDATION
      return set_error(B2U_ERR_ARG, "loss_bwd: the bf16 [hi | lo] output is not part of the fp32 validation build");
#else
      if (onehot) B2U_LBWDW(true, true); else B2U_LBWDW(false, true);
#endif
    } else if (out_mode == 0) {
      if (onehot) B2U_LBWDW(true, false); else B2U_LBWDW(false, false);
    } else {
      return set_error(B2U_ERR_ARG, "loss_bwd: out_mode must be 0 or 1");
    }
#undef B2U_LBWDW
    B2U_CHECK_LAUNCH("loss_bwd");
    return 0;
  }
  float* out = static_cast<float*>(dlogits);
#define B2U_LBWD(OH_, NH_, CM_) loss_bwd_kernel<OH_, NH_, CM_><<<blocks, kLossThreads, 0, st>>>( \
      logits, target, onehot, cls_w, fin, gscale, out, HW, P, C, focal_alpha, focal_gamma)
#define B2U_LBWD_C(OH_, NH_) do { if (C <= 8) B2U_LBWD(OH_, NH_, 8); else if (C <= 16) B2U_LBWD(OH_, NH_, 16); \
                                  else if (C <= 24) B2U_LBWD(OH_, NH_, 24); else B2U_LBWD(OH_, NH_, 32); } while (0)
  if (out_mode == 1) {
#ifdef B2U_FP32_VALIDATION
    return set_error(B2U_ERR_ARG, "loss_bwd: the bf16 [hi | lo] output is not part of the fp32 validation build");
#else
    if (onehot) B2U_LBWD_C(true, true); else B2U_LBWD_C(false, true);
#endif
  } else if (out_mode == 0) {
    if (onehot) B2U_LBWD_C(true, false); else B2U_LBWD_C(false, false);
  } else {
    return set_error(B2U_ERR_ARG, "loss_bwd: out_mode must be 0 or 1");
  }
#undef B2U_LBWD_C
#undef B2U_LBWD
  B2U_CHECK_LAUNCH("loss_bwd");
  return 0;
}

#ifndef B2U_FP32_VALIDATION
int b2u_pack_head_dgrad(const float* w, void* wd, int ncls, void* stream) {
  if (ncls <= 0 || ncls > kMaxClsWide) return set_error(B2U_ERR_SHAPE, "pack_head_dgrad: 1 <= classes <= 255");
  const int groups = (ncls + kMaxCls - 1) / kMaxCls;
  pack_head_dgrad_kernel<<<16 * groups, 256, 0, static_cast<cudaStream_t>(stream)>>>(w, static_cast<__nv_bfloat16*>(wd), ncls);
  B2U_CHECK_LAUNCH("pack_head_dgrad");
  return 0;
}

int b2u_pack_head_fprop(const float* w, void* wf, int ncls, void* stream) {
  if (ncls <= 0 || ncls > kMaxClsWide) return set_error(B2U_ERR_SHAPE, "pack_head_fprop: 1 <= classes <= 255");
  const int groups = (ncls + kMaxCls - 1) / kMaxCls;
  pack_head_fprop_kernel<<<16 * groups, 256, 0, static_cast<cudaStream_t>(stream)>>>(w, static_cast<__nv_bfloat16*>(wf), ncls);
  B2U_CHECK_LAUNCH("pack_head_fprop");
  return 0;
}
#endif  // !B2U_FP32_VALIDATION

int b2u_argmax_u8(const float* logits, unsigned char* mask, int N, int C, int H, int W, void* stream) {
  if (N <= 0 || C <= 0 || C > 256 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "argmax: bad shape");
  const long long HW = static_cast<long long>(H) * W, P = HW * N;
  argmax_u8_kernel<<<static_cast<unsigned>((P + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(logits, mask, HW, P, C);
  B2U_CHECK_LAUNCH("argmax_u8");
  return 0;
}

// logits [N][C][H][W] fp32; crop (cy, cx, ch, cw) inside H x W; mask [N][oh][ow] uint8 (class index, lowest on ties)
int b2u_softmax_resize_argmax_u8(const float* logits, unsigned char* mask, int N, int C, int H, int W, int cy, int cx,
                                 int ch, int cw, int oh, int ow, void* stream) {
  if (N <= 0 || C <= 0 || C > kMaxClsWide || H <= 0 || W <= 0 || oh <= 0 || ow <= 0 || N > 65535 || oh > 65535)
    return set_error(B2U_ERR_SHAPE, "softmax_resize_argmax: bad shape");
  if (cy < 0 || cx < 0 || ch <= 0 || cw <= 0 || cy + ch > H || cx + cw > W)
    return set_error(B2U_ERR_SHAPE, "softmax_resize_argmax: crop outside the logits");
  const float sy = static_cast<float>(static_cast<double>(ch) / oh), sx = static_cast<float>(static_cast<double>(cw) / ow);
  const dim3 grid((ow + 127) / 128, oh, N);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define B2U_SRA(CM_) softmax_resize_argmax_kernel<CM_><<<grid, 128, 0, st>>>(logits, mask, C, H, W, cy, cx, ch, cw, oh, ow, sy, sx)
  if (C <= 8) B2U_SRA(8); else if (C <= 16) B2U_SRA(16); else if (C <= 24) B2U_SRA(24); else if (C <= 32) B2U_SRA(32);
  else softmax_resize_argmax_wide_kernel<<<grid, 128, 0, st>>>(logits, mask, C, H, W, cy, cx, ch, cw, oh, ow, sy, sx);
#undef B2U_SRA
  B2U_CHECK_LAUNCH("softmax_resize_argmax");
  return 0;
}

// logits [count][C][H][W] fp32; items: count x {int cy, cx, ch, cw, oh, ow; int64 mask_off} (32 B each) in DEVICE memory,
// every crop inside H x W (an item whose crop is not is left unwritten); masks: flat uint8, image i's [oh][ow] mask at
// mask_off; max_oh / max_ow: the largest oh / ow of the batch (grid size only)
int b2u_softmax_resize_argmax_u8_batch(const float* logits, const void* items, int count, int C, int H, int W,
                                       unsigned char* masks, int max_oh, int max_ow, void* stream) {
  if (!logits || !items || !masks || count <= 0 || count > 65535 || C <= 0 || C > kMaxClsWide || H <= 0 || W <= 0 ||
      max_oh <= 0 || max_ow <= 0)
    return set_error(B2U_ERR_SHAPE, "softmax_resize_argmax_batch: bad shape");
  const dim3 grid((max_ow + 127) / 128, max_oh < 65535 ? max_oh : 65535, count);
  const SraItem* it = static_cast<const SraItem*>(items);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define B2U_SRAB(CM_) softmax_resize_argmax_batch_kernel<CM_><<<grid, 128, 0, st>>>(logits, it, masks, C, H, W)
  if (C <= 8) B2U_SRAB(8); else if (C <= 16) B2U_SRAB(16); else if (C <= 24) B2U_SRAB(24); else if (C <= 32) B2U_SRAB(32);
  else B2U_SRAB(0);
#undef B2U_SRAB
  B2U_CHECK_LAUNCH("softmax_resize_argmax_batch");
  return 0;
}

}  // extern "C"
