// bn.cu -- nn.BatchNorm2d (+ReLU) forward and backward on NHWC bf16 activations.
//
// Replaces nn.BatchNorm2d + nn.ReLU(inplace=True) after every conv of the reference's BN models
// (nets/TraditionalUnet.py:9-14, nets/resnet.py:65-71,110,140, nets/LightWeightUnet.py:9-11) and their autograd.
//
//   train fwd : mean_c, var_c (biased) over the N*H*W pixels of z; y = [relu](gamma (z - mean) invstd + beta);
//               running_mean = (1-m) rm + m mean, running_var = (1-m) rv + m var P/(P-1)   (torch semantics)
//   eval fwd  : y = [relu](gamma (z - rm) / sqrt(rv + eps) + beta)
//   bwd       : g = dy (y > 0 if relu); dbeta = sum g; dgamma = sum g xhat;
//               dz = gamma invstd (g - dbeta/P - xhat dgamma/P)
//
// All HBM-bound: a column-sum pass (z read once, 2 B/element) + an elementwise pass (4 B/element) forward; a
// column-sum pass (4 B/element; 6 with a residual) + an elementwise pass (6 B/element; 8 / 10 with a residual) backward.  Partial sums are fp32 per block,
// combined in fp64 in block order by a one-block finalize kernel (deterministic).
#include "b2u_internal.h"
#include "b2u_ptx.cuh"

namespace b2u {

#define B2U_CHECK_LAUNCH(name)                                                                           \
  do {                                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                                \
    if (e__ != cudaSuccess) return b2u::set_error(B2U_ERR_CUDA, name " launch: %s", cudaGetErrorString(e__)); \
    b2u::note_launch();                                                                                  \
  } while (0)

constexpr int kBnBlocks = 2 * 148;      // column-sum grid: 2 resident blocks of 256 threads per SM

__device__ __forceinline__ void bn_unpack8(const uint4& v, float* f) {
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x); f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z); f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}
__device__ __forceinline__ uint4 bn_pack8(const float* f) {
  uint4 v;
  v.x = pack_bf16x2(f[0], f[1]); v.y = pack_bf16x2(f[2], f[3]);
  v.z = pack_bf16x2(f[4], f[5]); v.w = pack_bf16x2(f[6], f[7]);
  return v;
}
// 8 consecutive per-channel fp32 coefficients as two 16-byte loads
__device__ __forceinline__ void bn_load8(const float* __restrict__ p, float* f) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
// The forward's affine form, reproducible bit for bit from (gamma, beta, save_mean, save_invstd): the backward
// recomputes the ReLU mask as fmaf(z, scale, shift) > 0 instead of re-reading y.
__device__ __forceinline__ void bn_affine(float g, float bt, float mean, float invstd, float* scale, float* shift) {
  const double sc = static_cast<double>(g) * static_cast<double>(invstd);
  *scale = static_cast<float>(sc);
  *shift = static_cast<float>(static_cast<double>(bt) - static_cast<double>(mean) * sc);
}

// Column sums of two per-element quantities.  MODE 0: (z - K, (z - K)^2) with the per-channel pivot K = row 0 of z when
// `pivot` is set (K = 0 otherwise).  MODE 1: (g, g * xhat) with g = dy * mask, where the mask is y > 0 (y given: residual
// blocks) or recomputed from z (y null).  partial layout: [block][2][C].
// The pivot keeps the one-pass variance accurate at training scale: with raw sums, var = E[z^2] - mean^2 loses the fp32
// rounding of E[z^2] amplified by (mean / std)^2 (1.2e-2 relative at mean = 64 std over 4M pixels).  Shifted by a value of
// the same channel, both sums are of the channel's spread; z - K of two bf16 values is exact in fp32.
// blockDim.x = 256; thread -> (row lane, 8-channel chunk); kBnUnroll rows (independent 16-byte loads per operand) are
// requested before any is consumed: ~64 KB in flight per SM.
template <int MODE>
__global__ void __launch_bounds__(256, 2)
bn_colsum_kernel(const uint4* __restrict__ a, const uint4* __restrict__ y, const uint4* __restrict__ z,
                 const float* __restrict__ gamma, const float* __restrict__ beta,
                 const float* __restrict__ mean, const float* __restrict__ invstd, float* __restrict__ partial,
                 long long P, int C8, int relu, int pivot) {
  constexpr int kBnUnroll = MODE == 0 ? 8 : 4;
  extern __shared__ float sred[];          // [256][16]
  const int tid = threadIdx.x;
  const int cpt = C8 < 256 ? C8 : 256;
  const int rows = 256 / cpt;
  const int cc = tid % cpt, rr = tid / cpt;
  const long long stride = static_cast<long long>(gridDim.x) * rows;
  for (int c0 = 0; c0 < C8; c0 += cpt) {
    const int c = c0 + cc;
    float s0[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s1[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (c < C8 && rr < rows) {
      float mu[8], is[8], sc[8], sh[8];
      if (MODE == 1) {
        bn_load8(mean + c * 8, mu); bn_load8(invstd + c * 8, is);
        if (relu && !y) {
#pragma unroll
          for (int k = 0; k < 8; ++k)
            bn_affine(gamma ? gamma[c * 8 + k] : 1.f, beta ? beta[c * 8 + k] : 0.f, mu[k], is[k], &sc[k], &sh[k]);
        }
      }
      // rows past the end load the pivot itself: they add exactly 0 to both sums
      const uint4 zero = MODE == 0 && pivot ? __ldg(a + c) : make_uint4(0u, 0u, 0u, 0u);
      float kp[8];
      bn_unpack8(zero, kp);
      for (long long p = static_cast<long long>(blockIdx.x) * rows + rr; p < P; p += kBnUnroll * stride) {
        uint4 va[kBnUnroll], vz[kBnUnroll], vy[kBnUnroll];
#pragma unroll
        for (int u = 0; u < kBnUnroll; ++u) {
          const long long q = p + u * stride;
          const bool ok = q < P;
          va[u] = ok ? __ldg(a + q * C8 + c) : zero;
          if (MODE == 1) {
            vz[u] = ok ? __ldg(z + q * C8 + c) : zero;
            if (relu && y) vy[u] = ok ? __ldg(y + q * C8 + c) : zero;
          }
        }
#pragma unroll
        for (int u = 0; u < kBnUnroll; ++u) {
          float f[8];
          bn_unpack8(va[u], f);
          if (MODE == 0) {
#pragma unroll
            for (int k = 0; k < 8; ++k) { const float d = f[k] - kp[k]; s0[k] += d; s1[k] = fmaf(d, d, s1[k]); }
          } else {
            float zz[8], yy[8];
            bn_unpack8(vz[u], zz);
            if (relu && y) bn_unpack8(vy[u], yy);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const bool on = !relu || (y ? yy[k] > 0.f : fmaf(zz[k], sc[k], sh[k]) > 0.f);
              const float g = on ? f[k] : 0.f;      // rows past the end carry dy = 0
              s0[k] += g;
              s1[k] = fmaf(g, (zz[k] - mu[k]) * is[k], s1[k]);
            }
          }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) { sred[tid * 16 + k] = s0[k]; sred[tid * 16 + 8 + k] = s1[k]; }
    __syncthreads();
    if (rr == 0 && c < C8) {
      for (int r = 1; r < rows; ++r)
#pragma unroll
        for (int k = 0; k < 8; ++k) { s0[k] += sred[(r * cpt + cc) * 16 + k]; s1[k] += sred[(r * cpt + cc) * 16 + 8 + k]; }
      float* out = partial + static_cast<size_t>(blockIdx.x) * 2 * C8 * 8;
#pragma unroll
      for (int k = 0; k < 8; ++k) { out[c * 8 + k] = s0[k]; out[C8 * 8 + c * 8 + k] = s1[k]; }
    }
    __syncthreads();
  }
}

// rows [R][L] fp32 -> out[L] (fp64 accumulation, fixed order): folds the per-tile statistics a conv epilogue wrote
__global__ void __launch_bounds__(256)
bn_rows_reduce_kernel(const float* __restrict__ rows, float* __restrict__ out, int R, int L) {
  __shared__ double sred[8][33];
  const int col = threadIdx.x & 31, lane_r = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + col;
  double acc = 0.0;
  if (i < L)
    for (int r = lane_r; r < R; r += 8) acc += static_cast<double>(__ldg(rows + static_cast<size_t>(r) * L + i));
  sred[lane_r][col] = acc;
  __syncthreads();
  if (lane_r == 0 && i < L) {
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sred[k][col];
    out[i] = static_cast<float>(t);
  }
}

// (mean, biased variance) of channel c from the column sums of bn_colsum_kernel<0>, combined in fp64 in block order.
// pivot_z (nullable): z itself when the sums are of z - K with K = row 0 of z (bn_colsum_kernel<0> with pivot set)
__device__ __forceinline__ void bn_sums_to_moments(const float* __restrict__ partial, const __nv_bfloat16* __restrict__ pivot_z,
                                                   int blocks, int C, long long P, int c, double* mean, double* var) {
  double s = 0.0, ss = 0.0;
  for (int b = 0; b < blocks; ++b) {
    s += partial[static_cast<size_t>(b) * 2 * C + c];
    ss += partial[static_cast<size_t>(b) * 2 * C + C + c];
  }
  const double ms = s / static_cast<double>(P);      // mean of the shifted values
  *mean = (pivot_z ? static_cast<double>(__bfloat162float(pivot_z[c])) : 0.0) + ms;
  const double v = ss / static_cast<double>(P) - ms * ms;
  *var = v < 0.0 ? 0.0 : v;
}

// the forward finalize from channel c's statistics over P rows: (scale, shift) for the apply pass, saved mean / invstd,
// running-statistic update
__device__ __forceinline__ void bn_fwd_finish(int c, double mean, double var, long long P, const float* __restrict__ gamma,
                                              const float* __restrict__ beta, float* __restrict__ running_mean,
                                              float* __restrict__ running_var, float* __restrict__ save_mean,
                                              float* __restrict__ save_invstd, float* __restrict__ scale,
                                              float* __restrict__ shift, float eps, float momentum, int centered) {
  const double invstd = 1.0 / sqrt(var + static_cast<double>(eps));
  const float mean_f = static_cast<float>(mean), invstd_f = static_cast<float>(invstd);
  save_mean[c] = mean_f;
  save_invstd[c] = invstd_f;
  bn_affine(gamma ? gamma[c] : 1.f, beta ? beta[c] : 0.f, mean_f, invstd_f, scale + c, shift + c);
  // centered: the producing conv stored z - running_mean (the old value, still in place here), so `mean` is the mean of
  // the shifted tensor; everything downstream (y, saved statistics, the backward) is shift-invariant, only the running
  // mean has to see the true mean
  if (running_mean) {
    const float rm_old = running_mean[c];
    running_mean[c] = (1.f - momentum) * rm_old + momentum * (static_cast<float>(mean) + (centered ? rm_old : 0.f));
  }
  if (running_var) {
    const double unbiased = P > 1 ? var * static_cast<double>(P) / static_cast<double>(P - 1) : var;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
  }
}

// forward finalize from the column sums of bn_colsum_kernel<0> (`blocks` rows of [2][C])
__global__ void bn_fwd_finalize_kernel(const float* __restrict__ partial, const __nv_bfloat16* __restrict__ pivot_z, int blocks, int C, long long P,
                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                       float* __restrict__ running_mean, float* __restrict__ running_var,
                                       float* __restrict__ save_mean, float* __restrict__ save_invstd,
                                       float* __restrict__ scale, float* __restrict__ shift, float eps, float momentum,
                                       int centered) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double mean, var;
  bn_sums_to_moments(partial, pivot_z, blocks, C, P, c, &mean, &var);
  bn_fwd_finish(c, mean, var, P, gamma, beta, running_mean, running_var, save_mean, save_invstd, scale, shift, eps, momentum,
                centered);
}

// SyncBatchNorm, one rank: moments [2][C] = (mean, biased variance) of this rank's rows
__global__ void bn_moments_kernel(const float* __restrict__ partial, const __nv_bfloat16* __restrict__ pivot_z, int blocks, int C,
                                  long long P, float* __restrict__ moments) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double mean, var;
  bn_sums_to_moments(partial, pivot_z, blocks, C, P, c, &mean, &var);
  moments[c] = static_cast<float>(mean);
  moments[C + c] = static_cast<float>(var);
}

// SyncBatchNorm forward finalize from the moments [world][2][C] of `world` ranks of P rows each, combined in fp64 like
// nn.SyncBatchNorm: mean = mean of the means, var = mean of (var_r + (mean_r - mean)^2); the running variance's unbiased
// factor counts the rows of all ranks
__global__ void bn_fwd_finalize_moments_kernel(const float* __restrict__ moments, int world, int C, long long P,
                                               const float* __restrict__ gamma, const float* __restrict__ beta,
                                               float* __restrict__ running_mean, float* __restrict__ running_var,
                                               float* __restrict__ save_mean, float* __restrict__ save_invstd,
                                               float* __restrict__ scale, float* __restrict__ shift, float eps, float momentum,
                                               int centered) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double mean = 0.0, var = 0.0;
  for (int r = 0; r < world; ++r) mean += moments[static_cast<size_t>(r) * 2 * C + c];
  mean /= world;
  for (int r = 0; r < world; ++r) {
    const double d = static_cast<double>(moments[static_cast<size_t>(r) * 2 * C + c]) - mean;
    var += static_cast<double>(moments[static_cast<size_t>(r) * 2 * C + C + c]) + d * d;
  }
  var /= world;
  bn_fwd_finish(c, mean, var, P * world, gamma, beta, running_mean, running_var, save_mean, save_invstd, scale, shift, eps,
                momentum, centered);
}

__global__ void bn_eval_coeff_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                     const float* __restrict__ running_mean, const float* __restrict__ running_var,
                                     float* __restrict__ scale, float* __restrict__ shift, int C, float eps) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float g = gamma ? gamma[c] : 1.f, bt = beta ? beta[c] : 0.f;
  const float is = 1.f / sqrtf(running_var[c] + eps);
  scale[c] = g * is;
  shift[c] = bt - running_mean[c] * g * is;
}

// eval-mode BatchNorm folded into the preceding conv: y = acc * scale + bias with scale = gamma / sqrt(rv + eps),
// bias = (conv_bias - rm) * scale + beta
__global__ void bn_fold_kernel(const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ rm,
                               const float* __restrict__ rv, const float* __restrict__ conv_bias, float* __restrict__ scale,
                               float* __restrict__ bias, int C, float eps) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float s = (gamma ? gamma[c] : 1.f) / sqrtf(rv[c] + eps);
  scale[c] = s;
  bias[c] = ((conv_bias ? conv_bias[c] : 0.f) - rm[c]) * s + (beta ? beta[c] : 0.f);
}

// y = [relu](z * scale + shift).  One thread = one 8-channel chunk of kBnApplyRows rows spaced G rows apart (so a warp's
// loads stay contiguous): the per-channel coefficients are loaded once and all the rows' 16-byte loads are in flight
// together.
constexpr int kBnApplyRows = 4;

__global__ void __launch_bounds__(256)
bn_apply_kernel(const uint4* __restrict__ z, const uint4* __restrict__ res, uint4* __restrict__ y,
                const float* __restrict__ scale, const float* __restrict__ shift, long long P, long long G, int C8, int relu) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= G * C8) return;
  const long long g = i / C8;
  const int c = static_cast<int>(i - g * C8);
  uint4 vz[kBnApplyRows], vr[kBnApplyRows];
#pragma unroll
  for (int u = 0; u < kBnApplyRows; ++u) {
    const long long row = g + u * G;
    if (row < P) {
      vz[u] = __ldg(z + row * C8 + c);
      if (res) vr[u] = __ldg(res + row * C8 + c);      // residual branch of a bottleneck: y = relu(bn(z) + identity)
    }
  }
  float sc[8], sh[8];
  bn_load8(scale + c * 8, sc); bn_load8(shift + c * 8, sh);
#pragma unroll
  for (int u = 0; u < kBnApplyRows; ++u) {
    const long long row = g + u * G;
    if (row >= P) break;
    float f[8], rs[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    bn_unpack8(vz[u], f);
    if (res) bn_unpack8(vr[u], rs);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float v = fmaf(f[k], sc[k], sh[k]) + rs[k];
      f[k] = relu ? fmaxf(v, 0.f) : v;
    }
    y[row * C8 + c] = bn_pack8(f);
  }
}

// backward finalize: dgamma, dbeta and the per-channel coefficients of the apply pass.
// dz = a (g - b - xhat c) with a = gamma invstd, b = dbeta / P, c = dgamma / P, written as dz = a g + kz z + k0.
// coef: [5][C] = a, kz, k0, scale, shift (the last two reproduce the forward's ReLU mask).
__global__ void bn_bwd_finalize_kernel(const float* __restrict__ partial, int blocks, int C, long long P,
                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                       const float* __restrict__ mean, const float* __restrict__ invstd,
                                       float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ coef) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double sg = 0.0, sgx = 0.0;
  for (int b = 0; b < blocks; ++b) {
    sg += partial[static_cast<size_t>(b) * 2 * C + c];
    sgx += partial[static_cast<size_t>(b) * 2 * C + C + c];
  }
  if (dbeta) dbeta[c] = static_cast<float>(sg);
  if (dgamma) dgamma[c] = static_cast<float>(sgx);
  const float g = gamma ? gamma[c] : 1.f;
  const double a = static_cast<double>(g) * invstd[c];
  const double kz = -a * (sgx / static_cast<double>(P)) * invstd[c];
  coef[c] = static_cast<float>(a);
  coef[C + c] = static_cast<float>(kz);
  coef[2 * C + c] = static_cast<float>(-a * (sg / static_cast<double>(P)) - kz * mean[c]);
  bn_affine(g, beta ? beta[c] : 0.f, mean[c], invstd[c], coef + 3 * C + c, coef + 4 * C + c);
}

__global__ void __launch_bounds__(256)
bn_bwd_apply_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ y, const uint4* __restrict__ z,
                    const float* __restrict__ coef, uint4* __restrict__ dz, uint4* __restrict__ gout, long long P,
                    long long G, int C8, int relu) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= G * C8) return;
  const long long gr = i / C8;
  const int c = static_cast<int>(i - gr * C8);
  const int C = C8 * 8;
  const bool from_y = relu && y;
  uint4 vg[kBnApplyRows], vz[kBnApplyRows], vy[kBnApplyRows];
#pragma unroll
  for (int u = 0; u < kBnApplyRows; ++u) {
    const long long row = gr + u * G;
    if (row < P) {
      vg[u] = __ldg(dy + row * C8 + c);
      vz[u] = __ldg(z + row * C8 + c);
      if (from_y) vy[u] = __ldg(y + row * C8 + c);
    }
  }
  float ca[8], kz[8], k0[8], sc[8], sh[8];
  bn_load8(coef + c * 8, ca); bn_load8(coef + C + c * 8, kz); bn_load8(coef + 2 * C + c * 8, k0);
  if (relu && !y) { bn_load8(coef + 3 * C + c * 8, sc); bn_load8(coef + 4 * C + c * 8, sh); }
#pragma unroll
  for (int u = 0; u < kBnApplyRows; ++u) {
    const long long row = gr + u * G;
    if (row >= P) break;
    float g[8], yy[8], zz[8], o[8], gm[8];
    bn_unpack8(vg[u], g);
    bn_unpack8(vz[u], zz);
    if (from_y) bn_unpack8(vy[u], yy);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const bool on = !relu || (from_y ? yy[k] > 0.f : fmaf(zz[k], sc[k], sh[k]) > 0.f);
      const float gg = on ? g[k] : 0.f;
      o[k] = fmaf(ca[k], gg, fmaf(kz[k], zz[k], k0[k]));
      gm[k] = gg;
    }
    if (gout) gout[row * C8 + c] = bn_pack8(gm);      // ReLU-masked dy: the gradient of the residual (identity) branch
    dz[row * C8 + c] = bn_pack8(o);
  }
}

}  // namespace b2u

extern "C" {
using namespace b2u;

// workspace: [blocks][2][C] fp32 partial sums + 5*C coefficients
size_t b2u_bn_workspace(int C) { return (static_cast<size_t>(kBnBlocks) * 2 * C + 5 * static_cast<size_t>(C)) * sizeof(float); }

static int bn_check(long long P, int C, const void* ws, size_t ws_bytes, const char* who) {
  if (P <= 0 || C <= 0 || C % 8 != 0) return set_error(B2U_ERR_SHAPE, "%s: needs P > 0 and C %% 8 == 0 (C=%d)", who, C);
  if (P * (C / 8) >= (1ll << 31)) return set_error(B2U_ERR_SHAPE, "%s: tensor too large (P*C/8 must be < 2^31)", who);
  if (!ws || ws_bytes < b2u_bn_workspace(C)) return set_error(B2U_ERR_ARG, "%s: workspace too small", who);
  return 0;
}

int b2u_bn_fwd_train(const void* z, const void* residual, void* y, const float* gamma, const float* beta, float* running_mean,
                     float* running_var, float* save_mean, float* save_invstd, void* ws, size_t ws_bytes, long long P,
                     int C, float eps, float momentum, int relu, void* stream) {
  int rc = bn_check(P, C, ws, ws_bytes, "bn_fwd_train");
  if (rc) return rc;
  const int centered = (relu >> 1) & 1;      // bit 1 of `relu`: z is stored centred on the running mean (see finalize)
  relu &= 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(ws);
  float* coef = partial + static_cast<size_t>(kBnBlocks) * 2 * C;
  bn_colsum_kernel<0><<<kBnBlocks, 256, 256 * 16 * sizeof(float), st>>>(static_cast<const uint4*>(z), nullptr, nullptr, nullptr,
                                                                        nullptr, nullptr, nullptr, partial, P, C / 8, 0, 1);
  B2U_CHECK_LAUNCH("bn_colsum");
  bn_fwd_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(partial, static_cast<const __nv_bfloat16*>(z), kBnBlocks, C, P, gamma,
                                                          beta, running_mean, running_var,
                                                          save_mean, save_invstd, coef, coef + C, eps, momentum, centered);
  B2U_CHECK_LAUNCH("bn_fwd_finalize");
  const long long G = (P + kBnApplyRows - 1) / kBnApplyRows;
  bn_apply_kernel<<<static_cast<unsigned>((G * (C / 8) + 255) / 256), 256, 0, st>>>(static_cast<const uint4*>(z), static_cast<const uint4*>(residual),
                                                                                   static_cast<uint4*>(y), coef, coef + C, P, G, C / 8, relu);
  B2U_CHECK_LAUNCH("bn_apply");
  return 0;
}

// b2u_bn_fwd_train with the column sums supplied by the producing conv (b2u_conv_fprop_stats): stat_rows rows of
// [2][C] fp32 per-tile sums of z and z^2 replace the statistics pass over z (one tensor read less).
int b2u_bn_fwd_train_stats(const void* z, const void* residual, void* y, const float* gamma, const float* beta,
                           float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                           const float* stat_partial, int stat_rows, void* ws, size_t ws_bytes, long long P, int C, float eps,
                           float momentum, int relu, void* stream) {
  int rc = bn_check(P, C, ws, ws_bytes, "bn_fwd_train_stats");
  if (rc) return rc;
  const int centered = (relu >> 1) & 1;      // bit 1 of `relu`: z is stored centred on the running mean (see finalize)
  relu &= 1;
  if (!stat_partial || stat_rows <= 0) return set_error(B2U_ERR_ARG, "bn_fwd_train_stats: statistics missing");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(ws);
  float* coef = partial + static_cast<size_t>(kBnBlocks) * 2 * C;
  bn_rows_reduce_kernel<<<(2 * C + 31) / 32, 256, 0, st>>>(stat_partial, partial, stat_rows, 2 * C);
  B2U_CHECK_LAUNCH("bn_rows_reduce");
  bn_fwd_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(partial, nullptr, 1, C, P, gamma, beta, running_mean, running_var,
                                                          save_mean, save_invstd, coef, coef + C, eps, momentum, centered);
  B2U_CHECK_LAUNCH("bn_fwd_finalize");
  const long long G = (P + kBnApplyRows - 1) / kBnApplyRows;
  bn_apply_kernel<<<static_cast<unsigned>((G * (C / 8) + 255) / 256), 256, 0, st>>>(static_cast<const uint4*>(z), static_cast<const uint4*>(residual),
                                                                                   static_cast<uint4*>(y), coef, coef + C, P, G, C / 8, relu);
  B2U_CHECK_LAUNCH("bn_apply");
  return 0;
}

// ---- SyncBatchNorm building blocks (nn.SyncBatchNorm.convert_sync_batchnorm, train.py:335-336): the statistics pass and the
// apply pass as separate calls, so the caller can gather the per-rank moments in between.  A per-rank pivot does not survive
// a sum across ranks, so the ranks exchange moments, not sums, and combine them the way nn.SyncBatchNorm does: each rank's
// (mean, var) keeps the one-GPU path's accuracy at any channel mean, and so does their combination.
// moments [2][C] fp32 = (mean, biased variance) of this rank's P rows, from the column sums about the row-0 pivot.
int b2u_bn_moments(const void* z, float* moments, void* ws, size_t ws_bytes, long long P, int C, void* stream) {
  int rc = bn_check(P, C, ws, ws_bytes, "bn_moments");
  if (rc) return rc;
  if (!moments) return set_error(B2U_ERR_ARG, "bn_moments: moments missing");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(ws);
  bn_colsum_kernel<0><<<kBnBlocks, 256, 256 * 16 * sizeof(float), st>>>(static_cast<const uint4*>(z), nullptr, nullptr, nullptr,
                                                                        nullptr, nullptr, nullptr, partial, P, C / 8, 0, 1);
  B2U_CHECK_LAUNCH("bn_colsum");
  bn_moments_kernel<<<(C + 127) / 128, 128, 0, st>>>(partial, static_cast<const __nv_bfloat16*>(z), kBnBlocks, C, P, moments);
  B2U_CHECK_LAUNCH("bn_moments");
  return 0;
}

// forward from the gathered moments [world][2][C] of `world` ranks holding P rows each; running statistics and saved
// mean / invstd are the global ones
int b2u_bn_fwd_train_moments(const void* z, const void* residual, void* y, const float* gamma, const float* beta,
                             float* running_mean, float* running_var, float* save_mean, float* save_invstd, const float* moments,
                             int world, void* ws, size_t ws_bytes, long long P, int C, float eps, float momentum, int relu,
                             void* stream) {
  int rc = bn_check(P, C, ws, ws_bytes, "bn_fwd_train_moments");
  if (rc) return rc;
  const int centered = (relu >> 1) & 1;      // bit 1 of `relu`: z is stored centred on the running mean (see finalize)
  relu &= 1;
  if (!moments || world < 1) return set_error(B2U_ERR_ARG, "bn_fwd_train_moments: moments missing or world < 1");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* coef = static_cast<float*>(ws) + static_cast<size_t>(kBnBlocks) * 2 * C;
  bn_fwd_finalize_moments_kernel<<<(C + 127) / 128, 128, 0, st>>>(moments, world, C, P, gamma, beta, running_mean, running_var,
                                                                  save_mean, save_invstd, coef, coef + C, eps, momentum, centered);
  B2U_CHECK_LAUNCH("bn_fwd_finalize_moments");
  const long long G = (P + kBnApplyRows - 1) / kBnApplyRows;
  bn_apply_kernel<<<static_cast<unsigned>((G * (C / 8) + 255) / 256), 256, 0, st>>>(static_cast<const uint4*>(z), static_cast<const uint4*>(residual),
                                                                                   static_cast<uint4*>(y), coef, coef + C, P, G, C / 8, relu);
  B2U_CHECK_LAUNCH("bn_apply");
  return 0;
}

// backward statistics of this rank: sums [2][C] = (sum g, sum g xhat) with g = dy masked by the ReLU (= dbeta, dgamma of
// this rank: torch's SyncBatchNorm keeps the affine gradients local and lets DDP average them)
int b2u_bn_bwd_sums(const void* dy, const void* y, const void* z, const float* gamma, const float* beta, const float* save_mean,
                    const float* save_invstd, float* sums, void* ws, size_t ws_bytes, long long P, int C, int relu,
                    void* stream) {
  int rc = bn_check(P, C, ws, ws_bytes, "bn_bwd_sums");
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(ws);
  bn_colsum_kernel<1><<<kBnBlocks, 256, 256 * 16 * sizeof(float), st>>>(static_cast<const uint4*>(dy), static_cast<const uint4*>(y),
                                                                        static_cast<const uint4*>(z), gamma, beta, save_mean,
                                                                        save_invstd, partial, P, C / 8, relu, 0);
  B2U_CHECK_LAUNCH("bn_bwd_colsum");
  bn_rows_reduce_kernel<<<(2 * C + 31) / 32, 256, 0, st>>>(partial, sums, kBnBlocks, 2 * C);
  B2U_CHECK_LAUNCH("bn_rows_reduce");
  return 0;
}

// dz from given (all-reduced) sums over P_stat rows
int b2u_bn_bwd_apply_sums(const void* dy, const void* y, const void* z, const float* gamma, const float* beta,
                          const float* save_mean, const float* save_invstd, void* dz, void* gout, const float* sums,
                          long long P_stat, void* ws, size_t ws_bytes, long long P, int C, int relu, void* stream) {
  int rc = bn_check(P, C, ws, ws_bytes, "bn_bwd_apply_sums");
  if (rc) return rc;
  if (!sums || P_stat < P) return set_error(B2U_ERR_ARG, "bn_bwd_apply_sums: sums missing or P_stat < P");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* coef = static_cast<float*>(ws) + static_cast<size_t>(kBnBlocks) * 2 * C;
  bn_bwd_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums, 1, C, P_stat, gamma, beta, save_mean, save_invstd, nullptr,
                                                          nullptr, coef);
  B2U_CHECK_LAUNCH("bn_bwd_finalize");
  const long long G = (P + kBnApplyRows - 1) / kBnApplyRows;
  bn_bwd_apply_kernel<<<static_cast<unsigned>((G * (C / 8) + 255) / 256), 256, 0, st>>>(
      static_cast<const uint4*>(dy), static_cast<const uint4*>(y), static_cast<const uint4*>(z), coef,
      static_cast<uint4*>(dz), static_cast<uint4*>(gout), P, G, C / 8, relu);
  B2U_CHECK_LAUNCH("bn_bwd_apply");
  return 0;
}

int b2u_bn_fold(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                const float* conv_bias, float* scale, float* bias, int C, float eps, void* stream) {
  if (C <= 0 || !running_mean || !running_var || !scale || !bias) return set_error(B2U_ERR_ARG, "bn_fold: bad arguments");
  bn_fold_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(gamma, beta, running_mean, running_var, conv_bias,
                                                                                scale, bias, C, eps);
  B2U_CHECK_LAUNCH("bn_fold");
  return 0;
}

int b2u_bn_fwd_eval(const void* z, const void* residual, void* y, const float* gamma, const float* beta, const float* running_mean,
                    const float* running_var, void* ws, size_t ws_bytes, long long P, int C, float eps, int relu,
                    void* stream) {
  int rc = bn_check(P, C, ws, ws_bytes, "bn_fwd_eval");
  if (rc) return rc;
  if (!running_mean || !running_var) return set_error(B2U_ERR_ARG, "bn_fwd_eval: running statistics required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* coef = static_cast<float*>(ws);
  bn_eval_coeff_kernel<<<(C + 127) / 128, 128, 0, st>>>(gamma, beta, running_mean, running_var, coef, coef + C, C, eps);
  B2U_CHECK_LAUNCH("bn_eval_coeff");
  const long long G = (P + kBnApplyRows - 1) / kBnApplyRows;
  bn_apply_kernel<<<static_cast<unsigned>((G * (C / 8) + 255) / 256), 256, 0, st>>>(static_cast<const uint4*>(z), static_cast<const uint4*>(residual),
                                                                                   static_cast<uint4*>(y), coef, coef + C, P, G, C / 8, relu);
  B2U_CHECK_LAUNCH("bn_apply");
  return 0;
}

// dy: gradient wrt y = [relu](bn(z) [+ residual]); dz (may alias dy) = gradient wrt the BN input z; gout (nullable,
// must not alias dy/dz) = dy masked by the ReLU = gradient wrt the residual input.
// y: the forward output, needed only when a residual was added before the ReLU; y == NULL (no residual) recomputes the
// ReLU mask from z, gamma, beta and the saved statistics exactly as the forward evaluated it, saving one tensor read
// in each of the two passes.
int b2u_bn_bwd(const void* dy, const void* y, const void* z, const float* gamma, const float* beta, const float* save_mean,
               const float* save_invstd, void* dz, void* gout, float* dgamma, float* dbeta, void* ws, size_t ws_bytes,
               long long P, int C, int relu, void* stream) {
  int rc = bn_check(P, C, ws, ws_bytes, "bn_bwd");
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(ws);
  float* coef = partial + static_cast<size_t>(kBnBlocks) * 2 * C;
  bn_colsum_kernel<1><<<kBnBlocks, 256, 256 * 16 * sizeof(float), st>>>(static_cast<const uint4*>(dy), static_cast<const uint4*>(y),
                                                                        static_cast<const uint4*>(z), gamma, beta, save_mean,
                                                                        save_invstd, partial, P, C / 8, relu, 0);
  B2U_CHECK_LAUNCH("bn_bwd_colsum");
  bn_bwd_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(partial, kBnBlocks, C, P, gamma, beta, save_mean, save_invstd, dgamma,
                                                          dbeta, coef);
  B2U_CHECK_LAUNCH("bn_bwd_finalize");
  const long long G = (P + kBnApplyRows - 1) / kBnApplyRows;
  bn_bwd_apply_kernel<<<static_cast<unsigned>((G * (C / 8) + 255) / 256), 256, 0, st>>>(
      static_cast<const uint4*>(dy), static_cast<const uint4*>(y), static_cast<const uint4*>(z), coef,
      static_cast<uint4*>(dz), static_cast<uint4*>(gout), P, G, C / 8, relu);
  B2U_CHECK_LAUNCH("bn_bwd_apply");
  return 0;
}

}  // extern "C"
