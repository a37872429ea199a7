// validation_fp32.cu -- the fp32 VALIDATION BUILD of the UNet hot path (libb200unet_fp32.so).
//
// BASELINE.json asks for two numeric bars: bf16 (rel-L2 <= 1e-2, the product path: tcgen05 kernels on NHWC bf16) and
// "<= 1e-5 for an fp32 validation build".  This translation unit is that build: the SAME C ABI (include/b2u.h), the same
// operand layouts, channel padding, virtual concat, split dgrad outputs, fused ReLU masks and call sequence -- so the
// host engine (engine.py) runs unchanged -- but every activation/gradient tensor ("void*" in the header) is NHWC fp32 and
// every contraction is an fp32 FMA chain on the CUDA cores.  What it validates is everything around the bf16 rounding:
// index arithmetic, weight packing, tap flips, mask placement, gradient routing, reductions, loss gradients.
// It is NOT a product path and is never loaded unless ops.set_validation_fp32(True) / B2U_FP32_VALIDATION=1 asks for it
// (tests/test_fp32_validation_gpu.py); no attention is paid to speed beyond a shared-memory tiled SGEMM.
//
// Covered: the entry points UNetEngine uses (Unet-VGG16 of nets/unet.py + nets/vgg.py, and the conv+BatchNorm+ReLU
// TraditionalUnet of nets/TraditionalUnet.py).  The loss / metric / optimizer kernels already compute in fp32 and are
// compiled into this library from their own sources (head_loss.cu with -DB2U_FP32_VALIDATION, hist.cu, optim.cu).
#include "b2u_internal.h"

#include <math.h>

namespace b2u {

#define B2U_CHECK_LAUNCH(name)                                                                           \
  do {                                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                                \
    if (e__ != cudaSuccess) return b2u::set_error(B2U_ERR_CUDA, name " launch: %s", cudaGetErrorString(e__)); \
    b2u::note_launch();                                                                                  \
  } while (0)

static inline unsigned blocks_for(long long n, int block) {
  long long g = (n + block - 1) / block;
  return static_cast<unsigned>(g < 1 ? 1 : g);
}

// ---------------------------------------------------------------------------------------------
// layout / packing (same operand layouts as elementwise.cu, fp32 elements)
// ---------------------------------------------------------------------------------------------
// col[n,h,w,k] = x[n,c,h+r-1,w+s-1] for k = (r*3+s)*Cin + c < 9*Cin, else 0   (nets/vgg.py:53 with C_in = 3)
__global__ void v32_im2col_first_kernel(const float* __restrict__ x, float* __restrict__ col, int N, int Cin, int H, int W) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(N) * H * W * 64;
  if (idx >= total) return;
  const int k = static_cast<int>(idx & 63);
  long long p = idx >> 6;
  const int w = static_cast<int>(p % W); p /= W;
  const int h = static_cast<int>(p % H);
  const int n = static_cast<int>(p / H);
  float v = 0.f;
  if (k < 9 * Cin) {
    const int tap = k / Cin, c = k - tap * Cin;
    const int hh = h + tap / 3 - 1, ww = w + tap % 3 - 1;
    if (hh >= 0 && hh < H && ww >= 0 && ww < W) v = x[((static_cast<size_t>(n) * Cin + c) * H + hh) * W + ww];
  }
  col[idx] = v;
}

// wf[co][tap*Cin + ci] = w[co][ci][tap];  wd[ci][tap*Cout + co] = w[co][ci][taps-1-tap]
__global__ void v32_pack_weights_kernel(const float* __restrict__ w, float* __restrict__ wf, float* __restrict__ wd, int Cout,
                                        int Cin, int taps) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(Cout) * Cin * taps;
  if (idx >= total) return;
  const int ci = static_cast<int>(idx % Cin);
  const int tap = static_cast<int>((idx / Cin) % taps);
  const int co = static_cast<int>(idx / (static_cast<long long>(Cin) * taps));
  const float v = w[(static_cast<size_t>(co) * Cin + ci) * taps + tap];
  if (wf) wf[idx] = v;
  if (wd) wd[(static_cast<size_t>(ci) * taps + (taps - 1 - tap)) * Cout + co] = v;
}
__global__ void v32_pack_weights_first_kernel(const float* __restrict__ w, float* __restrict__ wf, int Cout, int Cin) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= Cout * 64) return;
  const int co = idx / 64, k = idx % 64;
  float v = 0.f;
  if (k < 9 * Cin) { const int tap = k / Cin, c = k % Cin; v = w[(static_cast<size_t>(co) * Cin + c) * 9 + tap]; }
  wf[idx] = v;
}

// the table of b2u_pack_weights_multi (include/b2u.h): same 64-byte records, operands are fp32 here
struct V32PackEntry {
  const float* w;
  float* wf;
  float* wd;
  long long start;
  int Cout, Cin, taps, first;
  int C0, C0_pad;
  int Ctot_pad, Cout_pad;
};
__global__ void v32_pack_weights_multi_kernel(const V32PackEntry* __restrict__ table, int n) {
  int lo = 0, hi = n - 1;
  const long long b = blockIdx.x;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (table[mid].start <= b) lo = mid; else hi = mid - 1;
  }
  const V32PackEntry e = table[lo];
  const int lb = static_cast<int>(b - e.start);
  if (e.first) {
    for (int i = threadIdx.x; i < 32 * 64; i += blockDim.x) {
      const int co = lb * 32 + i / 64, k = i % 64;
      if (co >= e.Cout) continue;
      float v = 0.f;
      if (k < 9 * e.Cin) { const int tap = k / e.Cin, c = k % e.Cin; v = e.w[(static_cast<size_t>(co) * e.Cin + c) * 9 + tap]; }
      e.wf[static_cast<size_t>(co) * 64 + k] = v;
    }
    return;
  }
  const int tiles_ci = (e.Cin + 31) / 32;
  const int co0 = (lb / tiles_ci) * 32, ci0 = (lb % tiles_ci) * 32;
  const size_t kf = static_cast<size_t>(e.taps) * e.Ctot_pad, kd = static_cast<size_t>(e.taps) * e.Cout_pad;
  for (int i = threadIdx.x; i < 32 * 32 * e.taps; i += blockDim.x) {
    const int t = i % e.taps, ci = (i / e.taps) & 31, r = i / (32 * e.taps);
    const int co = co0 + r, gci = ci0 + ci;
    if (co >= e.Cout || gci >= e.Cin) continue;
    const float v = e.w[(static_cast<size_t>(co) * e.Cin + gci) * e.taps + t];
    const int pc = gci < e.C0 ? gci : gci - e.C0 + e.C0_pad;       // padded position of this input channel
    e.wf[co * kf + static_cast<size_t>(t) * e.Ctot_pad + pc] = v;
    if (e.wd) e.wd[pc * kd + static_cast<size_t>(e.taps - 1 - t) * e.Cout_pad + co] = v;
  }
}

// ---------------------------------------------------------------------------------------------
// convolution as an implicit-GEMM SGEMM: 64 pixels x 64 output channels per block, 4 x 4 per thread, K step 16
//   y[m][co] = epilogue( sum_k A[m][k] * Wp[co][k] ),  k = tap * Ctot + ci,  A[m][k] = x(pixel m shifted by tap)[ci]
// (fprop with the fprop operand; dgrad = the same kernel over dz with the flipped/transposed operand)
// ---------------------------------------------------------------------------------------------
struct V32Conv {
  const float* x0; const float* x1; int C0, C1;
  const float* wp;                 // [Cout][taps * (C0 + C1)]
  const float* bias; const float* scale;
  const float* mask; int mask_c;   // keep y where mask > 0
  float* y0; float* y1; int split_c;   // channels >= split_c go to y1 (channel pitch Cout - split_c)
  int N, H, W, Cout, taps, relu;
};
constexpr int kTM = 64, kTN = 64, kTK = 16;

__global__ void __launch_bounds__(256)
v32_conv_kernel(const V32Conv p) {
  __shared__ float As[kTK][kTM + 4];
  __shared__ float Bs[kTK][kTN + 4];
  const int ctot = p.C0 + p.C1;
  const int K = p.taps * ctot;
  const long long M = static_cast<long long>(p.N) * p.H * p.W;
  const long long m0 = static_cast<long long>(blockIdx.x) * kTM;
  const int n0 = blockIdx.y * kTN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;      // tx: channel group, ty: pixel group
  // loader roles: thread -> (row = tid / 4, 4 consecutive k = (tid % 4) * 4)
  const int lrow = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;
  const long long am = m0 + lrow;
  int an = 0, ah = 0, aw = 0;
  const bool a_ok = am < M;
  if (a_ok) {
    long long t = am;
    aw = static_cast<int>(t % p.W); t /= p.W;
    ah = static_cast<int>(t % p.H);
    an = static_cast<int>(t / p.H);
  }
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += kTK) {
    // a 16-wide k chunk never straddles a tap or a source: C0, C1 are multiples of 64
    const int tap = k0 / ctot, c = k0 - tap * ctot;
    const float* src; int cs, cc;
    if (c < p.C0) { src = p.x0; cs = p.C0; cc = c; } else { src = p.x1; cs = p.C1; cc = c - p.C0; }
    float4 av = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a_ok) {
      const int hh = p.taps == 9 ? ah + tap / 3 - 1 : ah, ww = p.taps == 9 ? aw + tap % 3 - 1 : aw;
      if (hh >= 0 && hh < p.H && ww >= 0 && ww < p.W)
        av = *reinterpret_cast<const float4*>(src + ((static_cast<size_t>(an) * p.H + hh) * p.W + ww) * cs + cc + lk);
    }
    As[lk + 0][lrow] = av.x; As[lk + 1][lrow] = av.y; As[lk + 2][lrow] = av.z; As[lk + 3][lrow] = av.w;
    const float4 bv = *reinterpret_cast<const float4*>(p.wp + static_cast<size_t>(n0 + lrow) * K + k0 + lk);
    Bs[lk + 0][lrow] = bv.x; Bs[lk + 1][lrow] = bv.y; Bs[lk + 2][lrow] = bv.z; Bs[lk + 3][lrow] = bv.w;
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kTK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int co = n0 + tx * 4 + j;
      float v = acc[i][j];
      if (p.scale) v = fmaf(v, p.scale[co], p.bias ? p.bias[co] : 0.f);
      else if (p.bias) v += p.bias[co];
      if (p.relu) v = fmaxf(v, 0.f);
      if (p.mask && !(p.mask[m * p.mask_c + co] > 0.f)) v = 0.f;
      if (co < p.split_c) p.y0[m * p.split_c + co] = v;
      else p.y1[m * (p.Cout - p.split_c) + (co - p.split_c)] = v;
    }
  }
}

static int v32_launch_conv(const V32Conv& p, cudaStream_t st) {
  if (p.N <= 0 || p.H <= 0 || p.W <= 0) return set_error(B2U_ERR_SHAPE, "conv: empty tensor");
  if (p.taps != 9 && p.taps != 1) return set_error(B2U_ERR_SHAPE, "conv: taps must be 9 or 1");
  if (p.Cout <= 0 || p.Cout % 64 != 0) return set_error(B2U_ERR_SHAPE, "conv: Cout %d must be a multiple of 64", p.Cout);
  if (p.C0 + p.C1 <= 0 || p.C0 % 64 != 0 || p.C1 % 64 != 0)
    return set_error(B2U_ERR_SHAPE, "conv: input channels (%d,%d) must be multiples of 64", p.C0, p.C1);
  if (p.y1 != nullptr && (p.split_c <= 0 || p.split_c >= p.Cout || p.split_c % 64 != 0))
    return set_error(B2U_ERR_SHAPE, "conv: split_c %d must be a multiple of 64 inside (0,Cout)", p.split_c);
  const long long M = static_cast<long long>(p.N) * p.H * p.W;
  dim3 grid(blocks_for(M, kTM), p.Cout / kTN, 1);
  v32_conv_kernel<<<grid, 256, 0, st>>>(p);
  B2U_CHECK_LAUNCH("conv_fp32");
  return 0;
}

// ---------------------------------------------------------------------------------------------
// weight gradient: dw[co][ci][tap] = sum_m dz[m][co] * x(pixel m shifted by tap)[ci]
// block = (64 co) x (64 ci) for one tap; the pixel sum runs in chunks of 16, fp32 FMA chains per thread
// ---------------------------------------------------------------------------------------------
struct V32Wgrad {
  const float* x0; const float* x1; int C0, C1;
  const float* dz; int Cout;
  float* dw;                     // OIHW [Cout][C0 + C1][taps], or [Cout][first_cin][9] when first_cin > 0
  int N, H, W, taps, first_cin;
};
__global__ void __launch_bounds__(256)
v32_wgrad_kernel(const V32Wgrad p) {
  __shared__ float As[kTK][kTM + 4];   // dz chunk: [pixel][co]
  __shared__ float Bs[kTK][kTN + 4];   // x chunk:  [pixel][ci]
  const int ctot = p.C0 + p.C1;
  const int co0 = blockIdx.x * 64, ci0 = blockIdx.y * 64, tap = blockIdx.z;
  const long long M = static_cast<long long>(p.N) * p.H * p.W;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;      // tx: ci group, ty: co group
  const int lp = threadIdx.x >> 4, lc = (threadIdx.x & 15) * 4;   // loader: pixel lp of the chunk, 4 channels from lc
  const float* src; int cs, cc;
  if (ci0 < p.C0) { src = p.x0; cs = p.C0; cc = ci0; } else { src = p.x1; cs = p.C1; cc = ci0 - p.C0; }
  const int dh = p.taps == 9 ? tap / 3 - 1 : 0, dwv = p.taps == 9 ? tap % 3 - 1 : 0;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (long long m0 = 0; m0 < M; m0 += kTK) {
    const long long m = m0 + lp;
    float4 av = make_float4(0.f, 0.f, 0.f, 0.f), bv = av;
    if (m < M) {
      av = *reinterpret_cast<const float4*>(p.dz + m * p.Cout + co0 + lc);
      long long t = m;
      const int w = static_cast<int>(t % p.W); t /= p.W;
      const int h = static_cast<int>(t % p.H);
      const int n = static_cast<int>(t / p.H);
      const int hh = h + dh, ww = w + dwv;
      if (hh >= 0 && hh < p.H && ww >= 0 && ww < p.W)
        bv = *reinterpret_cast<const float4*>(src + ((static_cast<size_t>(n) * p.H + hh) * p.W + ww) * cs + cc + lc);
    }
    *reinterpret_cast<float4*>(&As[lp][lc]) = av;
    *reinterpret_cast<float4*>(&Bs[lp][lc]) = bv;
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kTK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int co = co0 + ty * 4 + i;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ci = ci0 + tx * 4 + j;
      if (p.first_cin > 0) {
        // x0 is the im2col tensor: column k = tap' * cin + c of a 3x3 conv over first_cin channels
        if (ci < 9 * p.first_cin) {
          const int t9 = ci / p.first_cin, c = ci - t9 * p.first_cin;
          p.dw[(static_cast<size_t>(co) * p.first_cin + c) * 9 + t9] = acc[i][j];
        }
      } else {
        p.dw[(static_cast<size_t>(co) * ctot + ci) * p.taps + tap] = acc[i][j];
      }
    }
  }
}

// db[c] = sum over pixels of dz[., c]: one block per 32 channels, 8 pixel lanes, double accumulators
__global__ void __launch_bounds__(256)
v32_colsum_kernel(const float* __restrict__ dz, float* __restrict__ db, long long P, int C) {
  __shared__ double red[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), lane = threadIdx.x >> 5;
  double s = 0.0;
  if (c < C)
    for (long long p = lane; p < P; p += 8) s += static_cast<double>(dz[p * C + c]);
  red[lane][threadIdx.x & 31] = s;
  __syncthreads();
  if (lane == 0 && c < C) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    db[c] = static_cast<float>(t);
  }
}

// ---------------------------------------------------------------------------------------------
// pooling / upsampling
// ---------------------------------------------------------------------------------------------
__global__ void v32_maxpool_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int H, int W, int C) {
  const int Ho = H / 2, Wo = W / 2;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * Ho * Wo * C) return;
  const int c = static_cast<int>(idx % C);
  long long t = idx / C;
  const int wo = static_cast<int>(t % Wo); t /= Wo;
  const int ho = static_cast<int>(t % Ho);
  const int n = static_cast<int>(t / Ho);
  const size_t base = ((static_cast<size_t>(n) * H + 2 * ho) * W + 2 * wo) * C + c;
  const size_t rs = static_cast<size_t>(W) * C;
  y[idx] = fmaxf(fmaxf(x[base], x[base + C]), fmaxf(x[base + rs], x[base + rs + C]));
}
// dz[pos] = ((pos == first max of the window ? dpool : 0) + dskip[pos]) * (y[pos] > 0 if use_mask)
__global__ void v32_maxpool_bwd_kernel(const float* __restrict__ dpool, const float* __restrict__ dskip, const float* __restrict__ y,
                                       float* __restrict__ dz, int N, int H, int W, int C, int use_mask) {
  const int Ho = H / 2, Wo = W / 2;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * Ho * Wo * C) return;
  const int c = static_cast<int>(idx % C);
  long long t = idx / C;
  const int wo = static_cast<int>(t % Wo); t /= Wo;
  const int ho = static_cast<int>(t % Ho);
  const int n = static_cast<int>(t / Ho);
  const size_t base = ((static_cast<size_t>(n) * H + 2 * ho) * W + 2 * wo) * C + c;
  const size_t rs = static_cast<size_t>(W) * C;
  const size_t off[4] = {base, base + C, base + rs, base + rs + C};
  float yv[4];
  for (int q = 0; q < 4; ++q) yv[q] = y[off[q]];
  int a = 0; float m = yv[0];
  for (int q = 1; q < 4; ++q) if (yv[q] > m) { m = yv[q]; a = q; }
  const float g = dpool[idx];
  for (int q = 0; q < 4; ++q) {
    float v = (a == q ? g : 0.f) + (dskip ? dskip[off[q]] : 0.f);
    if (use_mask && !(yv[q] > 0.f)) v = 0.f;
    dz[off[q]] = v;
  }
}

// ATen area_pixel_compute_source_index(align_corners=True)
__device__ __forceinline__ void v32_src_index(int o, float scale, int in_size, int& i0, int& i1, float& lam) {
  const float src = scale * static_cast<float>(o);
  i0 = static_cast<int>(src);
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  lam = src - static_cast<float>(i0);
}
__global__ void v32_upsample_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int H, int W, int C, float sh,
                                        float sw) {
  const int Ho = 2 * H, Wo = 2 * W;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * Ho * Wo * C) return;
  const int c = static_cast<int>(idx % C);
  long long t = idx / C;
  const int wo = static_cast<int>(t % Wo); t /= Wo;
  const int ho = static_cast<int>(t % Ho);
  const int n = static_cast<int>(t / Ho);
  int h0, h1, w0, w1; float lh, lw;
  v32_src_index(ho, sh, H, h0, h1, lh);
  v32_src_index(wo, sw, W, w0, w1, lw);
  const float* img = x + static_cast<size_t>(n) * H * W * C + c;
  const float x00 = img[(static_cast<size_t>(h0) * W + w0) * C], x01 = img[(static_cast<size_t>(h0) * W + w1) * C];
  const float x10 = img[(static_cast<size_t>(h1) * W + w0) * C], x11 = img[(static_cast<size_t>(h1) * W + w1) * C];
  y[idx] = (1.f - lh) * ((1.f - lw) * x00 + lw * x01) + lh * ((1.f - lw) * x10 + lw * x11);
}
// adjoint in gather form: low-res (i, j) collects from the output rows/columns whose stencil touches it
__global__ void v32_upsample_bwd_kernel(const float* __restrict__ dup, const float* __restrict__ ylow, float* __restrict__ dlow,
                                        int N, int H, int W, int C, float sh, float sw) {
  const int Ho = 2 * H, Wo = 2 * W;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * H * W * C) return;
  const int c = static_cast<int>(idx % C);
  long long t = idx / C;
  const int j = static_cast<int>(t % W); t /= W;
  const int i = static_cast<int>(t % H);
  const int n = static_cast<int>(t / H);
  const float* img = dup + static_cast<size_t>(n) * Ho * Wo * C + c;
  float acc = 0.f;
  for (int oh = max(0, 2 * i - 3); oh <= min(Ho - 1, 2 * i + 3); ++oh) {
    int h0, h1; float lh;
    v32_src_index(oh, sh, H, h0, h1, lh);
    const float wh = (h0 == i ? 1.f - lh : 0.f) + (h1 == i ? lh : 0.f);
    if (wh == 0.f) continue;
    for (int ow = max(0, 2 * j - 3); ow <= min(Wo - 1, 2 * j + 3); ++ow) {
      int w0, w1; float lw;
      v32_src_index(ow, sw, W, w0, w1, lw);
      const float ww = (w0 == j ? 1.f - lw : 0.f) + (w1 == j ? lw : 0.f);
      if (ww != 0.f) acc = fmaf(wh * ww, img[(static_cast<size_t>(oh) * Wo + ow) * C], acc);
    }
  }
  if (ylow && !(ylow[idx] > 0.f)) acc = 0.f;
  dlow[idx] = acc;
}

// ---------------------------------------------------------------------------------------------
// classifier head: nn.Conv2d(64, num_classes, 1) (nets/unet.py:58,76), x NHWC fp32 [P][64], logits NCHW fp32
// ---------------------------------------------------------------------------------------------
__global__ void v32_head_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                                    float* __restrict__ logits, long long HW, long long P, int C) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= P * C) return;
  const long long p = idx % P;          // pixel fastest: coalesced logits stores
  const int c = static_cast<int>(idx / P);
  const float* xr = x + p * 64;
  float acc = 0.f;
  for (int k = 0; k < 64; ++k) acc = fmaf(xr[k], w[c * 64 + k], acc);
  const long long n = p / HW, hw = p % HW;
  logits[(n * C + c) * HW + hw] = acc + (b ? b[c] : 0.f);
}
__global__ void v32_head_dgrad_kernel(const float* __restrict__ dl, const float* __restrict__ x, const float* __restrict__ w,
                                      float* __restrict__ dx, long long HW, long long P, int C, int relu_mask) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= P * 64) return;
  const int k = static_cast<int>(idx & 63);
  const long long p = idx >> 6;
  const long long n = p / HW, hw = p % HW;
  float acc = 0.f;
  for (int c = 0; c < C; ++c) acc = fmaf(dl[(n * C + c) * HW + hw], w[c * 64 + k], acc);
  if (relu_mask && !(x[idx] > 0.f)) acc = 0.f;
  dx[idx] = acc;
}
// dw[c][k] = sum_p dl[p][c] x[p][k]; db[c] = sum_p dl[p][c]: one block per (class, k or bias), double accumulators
__global__ void __launch_bounds__(256)
v32_head_wgrad_kernel(const float* __restrict__ dl, const float* __restrict__ x, float* __restrict__ dw, float* __restrict__ db,
                      long long HW, long long P, int C) {
  __shared__ double red[256];
  const int c = blockIdx.x / 65, k = blockIdx.x % 65;     // k == 64: the bias column
  double s = 0.0;
  for (long long p = threadIdx.x; p < P; p += 256) {
    const long long n = p / HW, hw = p % HW;
    const float g = dl[(n * C + c) * HW + hw];
    s += k < 64 ? static_cast<double>(g) * static_cast<double>(x[p * 64 + k]) : static_cast<double>(g);
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (k < 64) { if (dw) dw[c * 64 + k] = static_cast<float>(red[0]); }
    else if (db) db[c] = static_cast<float>(red[0]);
  }
}

// ---------------------------------------------------------------------------------------------
// batch normalisation (nn.BatchNorm2d [+ ReLU], nets/TraditionalUnet.py:9-14): statistics in double
// ---------------------------------------------------------------------------------------------
// sums[c] = sum z, sums[C + c] = sum (z - mean)^2 would need two passes; instead one pass in double over (z, z^2)
__global__ void __launch_bounds__(256)
v32_bn_stats_kernel(const float* __restrict__ z, double* __restrict__ sums, long long P, int C) {
  __shared__ double r0[8][33], r1[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), lane = threadIdx.x >> 5;
  double s = 0.0, q = 0.0;
  if (c < C)
    for (long long p = lane; p < P; p += 8) { const double v = z[p * C + c]; s += v; q += v * v; }
  r0[lane][threadIdx.x & 31] = s; r1[lane][threadIdx.x & 31] = q;
  __syncthreads();
  if (lane == 0 && c < C) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < 8; ++i) { a += r0[i][threadIdx.x]; b += r1[i][threadIdx.x]; }
    sums[c] = a; sums[C + c] = b;
  }
}
__global__ void v32_bn_finalize_kernel(const double* __restrict__ sums, float* __restrict__ running_mean, float* __restrict__ running_var,
                                       float* __restrict__ save_mean, float* __restrict__ save_invstd, long long P, int C, float eps,
                                       float momentum) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = sums[c] / static_cast<double>(P);
  double var = sums[C + c] / static_cast<double>(P) - mean * mean;
  if (var < 0.0) var = 0.0;
  save_mean[c] = static_cast<float>(mean);
  save_invstd[c] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * static_cast<float>(mean);
  if (running_var) {
    const double unbiased = P > 1 ? var * static_cast<double>(P) / static_cast<double>(P - 1) : var;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
  }
}
__device__ __forceinline__ float v32_bn_eval(float z, float mean, float invstd, float g, float b) {
  return (z - mean) * invstd * g + b;
}
__global__ void v32_bn_apply_kernel(const float* __restrict__ z, const float* __restrict__ residual, float* __restrict__ y,
                                    const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                                    const float* __restrict__ invstd_or_var, long long total, int C, float eps, int var_mode,
                                    int relu) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = static_cast<int>(idx % C);
  const float is = var_mode ? 1.f / sqrtf(invstd_or_var[c] + eps) : invstd_or_var[c];
  float v = v32_bn_eval(z[idx], mean[c], is, gamma ? gamma[c] : 1.f, beta ? beta[c] : 0.f);
  if (residual) v += residual[idx];
  if (relu) v = fmaxf(v, 0.f);
  y[idx] = v;
}
// pass 1 of the backward: sums[c] = sum g, sums[C + c] = sum g * xhat with g = dy masked by the ReLU
__global__ void __launch_bounds__(256)
v32_bn_bwd_stats_kernel(const float* __restrict__ dy, const float* __restrict__ y, const float* __restrict__ z,
                        const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                        const float* __restrict__ invstd, double* __restrict__ sums, long long P, int C, int relu) {
  __shared__ double r0[8][33], r1[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), lane = threadIdx.x >> 5;
  double s = 0.0, q = 0.0;
  if (c < C) {
    const float mu = mean[c], is = invstd[c], g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
    for (long long p = lane; p < P; p += 8) {
      const float zz = z[p * C + c];
      const bool on = !relu || (y ? y[p * C + c] > 0.f : v32_bn_eval(zz, mu, is, g, b) > 0.f);
      const double gv = on ? static_cast<double>(dy[p * C + c]) : 0.0;
      s += gv; q += gv * static_cast<double>((zz - mu) * is);
    }
  }
  r0[lane][threadIdx.x & 31] = s; r1[lane][threadIdx.x & 31] = q;
  __syncthreads();
  if (lane == 0 && c < C) {
    double a = 0.0, b2 = 0.0;
    for (int i = 0; i < 8; ++i) { a += r0[i][threadIdx.x]; b2 += r1[i][threadIdx.x]; }
    sums[c] = a; sums[C + c] = b2;
  }
}
// pass 2: dz = gamma * invstd * (g - mean(g) - xhat * mean(g xhat)); gout = g
__global__ void v32_bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ y, const float* __restrict__ z,
                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                        const float* __restrict__ mean, const float* __restrict__ invstd,
                                        const double* __restrict__ sums, float* __restrict__ dz, float* __restrict__ gout,
                                        float* __restrict__ dgamma, float* __restrict__ dbeta, long long P, int C, int relu) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx < C) {
    if (dbeta) dbeta[idx] = static_cast<float>(sums[idx]);
    if (dgamma) dgamma[idx] = static_cast<float>(sums[C + idx]);
  }
  if (idx >= P * C) return;
  const int c = static_cast<int>(idx % C);
  const float mu = mean[c], is = invstd[c], g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
  const float zz = z[idx];
  const bool on = !relu || (y ? y[idx] > 0.f : v32_bn_eval(zz, mu, is, g, b) > 0.f);
  const float gv = on ? dy[idx] : 0.f;
  const float xhat = (zz - mu) * is;
  const float m1 = static_cast<float>(sums[c] / static_cast<double>(P)), m2 = static_cast<float>(sums[C + c] / static_cast<double>(P));
  if (gout) gout[idx] = gv;
  dz[idx] = g * is * (gv - m1 - xhat * m2);
}
__global__ void v32_bn_fold_kernel(const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ rm,
                                   const float* __restrict__ rv, const float* __restrict__ conv_bias, float* __restrict__ scale,
                                   float* __restrict__ bias, int C, float eps) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double s = static_cast<double>(gamma ? gamma[c] : 1.f) / sqrt(static_cast<double>(rv[c]) + static_cast<double>(eps));
  scale[c] = static_cast<float>(s);
  bias[c] = static_cast<float>((static_cast<double>(conv_bias ? conv_bias[c] : 0.f) - static_cast<double>(rm[c])) * s +
                               static_cast<double>(beta ? beta[c] : 0.f));
}


// ---------------------------------------------------------------------------------------------
// ResNet50 encoder helpers (resnet_ops.cu in fp32): stem im2col, stride-2 helpers, 3x3 s2 ceil-mode max-pool, joins
// ---------------------------------------------------------------------------------------------
__global__ void v32_im2col_stem_kernel(const float* __restrict__ x, float* __restrict__ col, int N, int Cin, int H, int W, int Ho,
                                       int Wo) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * Ho * Wo * 192) return;
  const int k = static_cast<int>(idx % 192);
  long long t = idx / 192;
  const int wo = static_cast<int>(t % Wo); t /= Wo;
  const int ho = static_cast<int>(t % Ho);
  const int n = static_cast<int>(t / Ho);
  float v = 0.f;
  if (k < 49 * Cin) {
    const int tap = k / Cin, c = k - tap * Cin;
    const int hh = 2 * ho + tap / 7 - 3, ww = 2 * wo + tap % 7 - 3;
    if (hh >= 0 && hh < H && ww >= 0 && ww < W) v = x[((static_cast<size_t>(n) * Cin + c) * H + hh) * W + ww];
  }
  col[idx] = v;
}
__global__ void v32_pack_weights_im2col_kernel(const float* __restrict__ w, float* __restrict__ wf, int Cout, int Cin, int taps,
                                               int Kpad) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= Cout * Kpad) return;
  const int co = idx / Kpad, k = idx - co * Kpad;
  float v = 0.f;
  if (k < taps * Cin) { const int tap = k / Cin, c = k - tap * Cin; v = w[(static_cast<size_t>(co) * Cin + c) * taps + tap]; }
  wf[idx] = v;
}
// dw[co][c][tap] = sum_p dz[p][co] * col[p][tap * cin + c]: one block per output element row, double accumulators
__global__ void __launch_bounds__(256)
v32_wgrad_im2col_kernel(const float* __restrict__ col, const float* __restrict__ dz, float* __restrict__ dw, long long P, int Kpad,
                        int Cout, int cin, int taps) {
  __shared__ double red[256];
  const int co = blockIdx.x / (cin * taps), k = blockIdx.x % (cin * taps);    // k = tap * cin + c
  double s = 0.0;
  for (long long p = threadIdx.x; p < P; p += 256) s += static_cast<double>(dz[p * Cout + co]) * static_cast<double>(col[p * Kpad + k]);
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) { const int tap = k / cin, c = k - tap * cin; dw[(static_cast<size_t>(co) * cin + c) * taps + tap] = static_cast<float>(red[0]); }
}
__global__ void v32_subsample2_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int H, int W, int C) {
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * Ho * Wo * C) return;
  const int c = static_cast<int>(idx % C);
  long long t = idx / C;
  const int wo = static_cast<int>(t % Wo); t /= Wo;
  const int ho = static_cast<int>(t % Ho);
  const int n = static_cast<int>(t / Ho);
  y[idx] = x[((static_cast<size_t>(n) * H + 2 * ho) * W + 2 * wo) * C + c];
}
__global__ void v32_zero_insert2_kernel(const float* __restrict__ y, float* __restrict__ x, int N, int H, int W, int C) {
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * H * W * C) return;
  const int c = static_cast<int>(idx % C);
  long long t = idx / C;
  const int w = static_cast<int>(t % W); t /= W;
  const int h = static_cast<int>(t % H);
  const int n = static_cast<int>(t / H);
  x[idx] = (!(h & 1) && !(w & 1)) ? y[((static_cast<size_t>(n) * Ho + h / 2) * Wo + w / 2) * C + c] : 0.f;
}
__global__ void v32_maxpool3_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int H, int W, int Ho, int Wo,
                                        int C) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * Ho * Wo * C) return;
  const int c = static_cast<int>(idx % C);
  long long t = idx / C;
  const int wo = static_cast<int>(t % Wo); t /= Wo;
  const int ho = static_cast<int>(t % Ho);
  const int n = static_cast<int>(t / Ho);
  float m = -INFINITY;
  for (int r = 0; r < 3; ++r)
    for (int q = 0; q < 3; ++q) {
      const int h = 2 * ho + r, w = 2 * wo + q;
      if (h < H && w < W) m = fmaxf(m, x[((static_cast<size_t>(n) * H + h) * W + w) * C + c]);
    }
  y[idx] = m;
}
// dx[h,w] = sum of dy over the windows containing (h,w) whose FIRST maximum (row-major scan, like ATen) is (h,w)
__global__ void v32_maxpool3_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x, float* __restrict__ dx, int N,
                                        int H, int W, int Ho, int Wo, int C) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * H * W * C) return;
  const int c = static_cast<int>(idx % C);
  long long t = idx / C;
  const int w = static_cast<int>(t % W); t /= W;
  const int h = static_cast<int>(t % H);
  const int n = static_cast<int>(t / H);
  const float* ximg = x + static_cast<size_t>(n) * H * W * C + c;
  const float xv = x[idx];
  const int ho_lo = h >= 2 ? (h - 1) / 2 : 0, ho_hi = min(h / 2, Ho - 1);
  const int wo_lo = w >= 2 ? (w - 1) / 2 : 0, wo_hi = min(w / 2, Wo - 1);
  float acc = 0.f;
  for (int ho = ho_lo; ho <= ho_hi; ++ho)
    for (int wo = wo_lo; wo <= wo_hi; ++wo) {
      bool first = true;
      for (int r = 0; r < 3 && first; ++r)
        for (int q = 0; q < 3; ++q) {
          const int hh = 2 * ho + r, ww = 2 * wo + q;
          if (hh >= H || ww >= W || (hh == h && ww == w)) continue;
          const float f = ximg[(static_cast<size_t>(hh) * W + ww) * C];
          const bool before = hh < h || (hh == h && ww < w);
          if (!(before ? f < xv : f <= xv)) { first = false; break; }
        }
      if (first) acc += dy[((static_cast<size_t>(n) * Ho + ho) * Wo + wo) * C + c];
    }
  dx[idx] = acc;
}
// mode 0: a + b; 1: relu(a + b); 2: a * (b > 0)
__global__ void v32_join_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long long n, int mode) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = a[i], y = b[i];
  out[i] = mode == 0 ? x + y : (mode == 1 ? fmaxf(x + y, 0.f) : (y > 0.f ? x : 0.f));
}
// NCHW fp32 -> NHWC fp32 with the channel dimension zero-padded to Cpad
__global__ void v32_nchw_to_nhwc_padded_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int C, long long HW, int Cpad) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * HW * Cpad) return;
  const int c = static_cast<int>(idx % Cpad);
  const long long p = idx / Cpad;
  const long long n = p / HW, hw = p % HW;
  y[idx] = c < C ? x[(n * C + c) * HW + hw] : 0.f;
}
// the gradient wrt the input image (input_grad.cu in fp32): one thread per NCHW output element, gather over (co, tap)
// dx[n,c,h,w] = sum over co and the taps (r, s) with (h + pad - r) and (w + pad - s) divisible by the stride of
// dz[n, (h+pad-r)/stride, (w+pad-s)/stride, co] * W[co,c,r,s]
__global__ void v32_conv_dgrad_input_kernel(const float* __restrict__ dz, int Cz, const float* __restrict__ w, float* __restrict__ dx,
                                            int N, int Cin, int H, int W, int Hz, int Wz, int Cout, int K, int stride, int pad) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * Cin * H * W) return;
  const int x = static_cast<int>(idx % W);
  long long t = idx / W;
  const int y = static_cast<int>(t % H); t /= H;
  const int c = static_cast<int>(t % Cin);
  const int n = static_cast<int>(t / Cin);
  float acc = 0.f;
  for (int r = 0; r < K; ++r) {
    const int hs = y + pad - r;
    if (hs < 0 || hs % stride) continue;
    const int hz = hs / stride;
    if (hz >= Hz) continue;
    for (int s = 0; s < K; ++s) {
      const int ws = x + pad - s;
      if (ws < 0 || ws % stride) continue;
      const int wz = ws / stride;
      if (wz >= Wz) continue;
      const float* g = dz + ((static_cast<size_t>(n) * Hz + hz) * Wz + wz) * Cz;
      for (int co = 0; co < Cout; ++co) acc = fmaf(g[co], w[((static_cast<size_t>(co) * Cin + c) * K + r) * K + s], acc);
    }
  }
  dx[idx] = acc;
}
__global__ void v32_nhwc_padded_to_nchw_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int C, long long HW, int Cpad) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * C * HW) return;
  const long long hw = idx % HW, nc = idx / HW;
  y[idx] = x[((nc / C) * HW + hw) * Cpad + nc % C];
}
// F.interpolate(x, size, mode="bilinear", align_corners=True) on NCHW fp32 planes, and its adjoint (gather form)
__global__ void v32_resize_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, long long NC, int Hi, int Wi, int Ho, int Wo,
                                      float sh, float sw) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= NC * Ho * Wo) return;
  const int wo = static_cast<int>(idx % Wo);
  const int ho = static_cast<int>((idx / Wo) % Ho);
  const long long nc = idx / (static_cast<long long>(Wo) * Ho);
  int h0, h1, w0, w1; float lh, lw;
  v32_src_index(ho, sh, Hi, h0, h1, lh);
  v32_src_index(wo, sw, Wi, w0, w1, lw);
  const float* img = x + nc * Hi * Wi;
  y[idx] = (1.f - lh) * ((1.f - lw) * img[h0 * Wi + w0] + lw * img[h0 * Wi + w1]) +
           lh * ((1.f - lw) * img[h1 * Wi + w0] + lw * img[h1 * Wi + w1]);
}
__global__ void v32_resize_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, long long NC, int Hi, int Wi, int Ho, int Wo,
                                      float sh, float sw) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= NC * Hi * Wi) return;
  const int j = static_cast<int>(idx % Wi);
  const int i = static_cast<int>((idx / Wi) % Hi);
  const long long nc = idx / (static_cast<long long>(Wi) * Hi);
  const float* img = dy + nc * Ho * Wo;
  // outputs whose source interval touches i: src in (i-1, i+1)  ->  o in ((i-1)/s, (i+1)/s)
  const int oh_lo = sh > 0.f ? max(0, static_cast<int>((i - 1) / sh) - 1) : 0, oh_hi = sh > 0.f ? min(Ho - 1, static_cast<int>((i + 1) / sh) + 1) : Ho - 1;
  const int ow_lo = sw > 0.f ? max(0, static_cast<int>((j - 1) / sw) - 1) : 0, ow_hi = sw > 0.f ? min(Wo - 1, static_cast<int>((j + 1) / sw) + 1) : Wo - 1;
  float acc = 0.f;
  for (int oh = oh_lo; oh <= oh_hi; ++oh) {
    int h0, h1; float lh;
    v32_src_index(oh, sh, Hi, h0, h1, lh);
    const float wh = (h0 == i ? 1.f - lh : 0.f) + (h1 == i ? lh : 0.f);
    if (wh == 0.f) continue;
    for (int ow = ow_lo; ow <= ow_hi; ++ow) {
      int w0, w1; float lw;
      v32_src_index(ow, sw, Wi, w0, w1, lw);
      const float ww = (w0 == j ? 1.f - lw : 0.f) + (w1 == j ? lw : 0.f);
      if (ww != 0.f) acc = fmaf(wh * ww, img[static_cast<size_t>(oh) * Wo + ow], acc);
    }
  }
  dx[idx] = acc;
}

// ---------------------------------------------------------------------------------------------
// depthwise 3x3, per-(image, channel) reductions and scaling (dw_se.cu in fp32)
// ---------------------------------------------------------------------------------------------
__global__ void v32_dwconv_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                                  float* __restrict__ y, int N, int H, int W, int C, int flip) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(N) * H * W * C) return;
  const int c = static_cast<int>(idx % C);
  long long t = idx / C;
  const int ww = static_cast<int>(t % W); t /= W;
  const int hh = static_cast<int>(t % H);
  const int n = static_cast<int>(t / H);
  float acc = bias ? bias[c] : 0.f;
  for (int tap = 0; tap < 9; ++tap) {
    const int h = hh + tap / 3 - 1, v = ww + tap % 3 - 1;
    if (h >= 0 && h < H && v >= 0 && v < W)
      acc = fmaf(x[((static_cast<size_t>(n) * H + h) * W + v) * C + c], w[c * 9 + (flip ? 8 - tap : tap)], acc);
  }
  y[idx] = acc;
}
// dw[c][tap] = sum_p dy[p][c] x[p + tap][c]; column 9 = sum dy (bias): block = (channel, quantity), double accumulators
__global__ void __launch_bounds__(256)
v32_dwconv_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dw, float* __restrict__ db,
                        int N, int H, int W, int C) {
  __shared__ double red[256];
  const int c = blockIdx.x / 10, tap = blockIdx.x % 10;
  const long long P = static_cast<long long>(N) * H * W;
  double s = 0.0;
  for (long long p = threadIdx.x; p < P; p += 256) {
    const double g = dy[p * C + c];
    if (tap == 9) { s += g; continue; }
    const int ww = static_cast<int>(p % W), hh = static_cast<int>((p / W) % H);
    const long long n = p / (static_cast<long long>(W) * H);
    const int h = hh + tap / 3 - 1, v = ww + tap % 3 - 1;
    if (h >= 0 && h < H && v >= 0 && v < W) s += g * static_cast<double>(x[((n * H + h) * W + v) * C + c]);
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (tap < 9) { if (dw) dw[c * 9 + tap] = static_cast<float>(red[0]); }
    else if (db) db[c] = static_cast<float>(red[0]);
  }
}
// out[n][c] = scale * sum over the image's pixels of a (b == NULL) or a * b
__global__ void __launch_bounds__(256)
v32_spatial_reduce_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long long HW, int C,
                          float scale) {
  __shared__ double red[8][33];
  const int n = blockIdx.y, c = blockIdx.x * 32 + (threadIdx.x & 31), lane = threadIdx.x >> 5;
  double s = 0.0;
  if (c < C)
    for (long long p = lane; p < HW; p += 8) {
      const size_t i = (static_cast<size_t>(n) * HW + p) * C + c;
      s += b ? static_cast<double>(a[i]) * static_cast<double>(b[i]) : static_cast<double>(a[i]);
    }
  red[lane][threadIdx.x & 31] = s;
  __syncthreads();
  if (lane == 0 && c < C) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    out[static_cast<size_t>(n) * C + c] = static_cast<float>(t * static_cast<double>(scale));
  }
}
__global__ void v32_scale_nc_kernel(const float* __restrict__ x, const float* __restrict__ s, const float* __restrict__ a,
                                    float* __restrict__ y, long long HW, int C, long long total) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = static_cast<int>(idx % C);
  const long long n = idx / (HW * C);
  y[idx] = fmaf(x[idx], s[n * C + c], a ? a[n * C + c] : 0.f);
}

}  // namespace b2u

// ----------------------------------------------------------------------------
// C ABI (include/b2u.h): same names and argument meaning, activations fp32
// ----------------------------------------------------------------------------
extern "C" {
using namespace b2u;

int b2u_validation_fp32(void) { return 1; }

int b2u_im2col_first(const float* x, void* col, int N, int Cin, int H, int W, void* stream) {
  if (Cin <= 0 || 9 * Cin > 64) return set_error(B2U_ERR_SHAPE, "im2col_first: 9*Cin must fit 64 columns (Cin=%d)", Cin);
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "im2col_first: empty tensor");
  const long long total = static_cast<long long>(N) * H * W * 64;
  v32_im2col_first_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, static_cast<float*>(col), N, Cin, H, W);
  B2U_CHECK_LAUNCH("im2col_first_fp32");
  return 0;
}

int b2u_pack_weights(const float* w, void* wf, void* wd, int Cout, int Cin, int taps, void* stream) {
  if (Cout <= 0 || Cin <= 0 || (taps != 1 && taps != 9)) return set_error(B2U_ERR_SHAPE, "pack_weights: bad shape");
  const long long total = static_cast<long long>(Cout) * Cin * taps;
  v32_pack_weights_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w, static_cast<float*>(wf), static_cast<float*>(wd), Cout, Cin, taps);
  B2U_CHECK_LAUNCH("pack_weights_fp32");
  return 0;
}

int b2u_pack_weights_first(const float* w, void* wf, int Cout, int Cin, void* stream) {
  if (Cout <= 0 || Cin <= 0 || 9 * Cin > 64) return set_error(B2U_ERR_SHAPE, "pack_weights_first: bad shape");
  v32_pack_weights_first_kernel<<<blocks_for(Cout * 64, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(w, static_cast<float*>(wf), Cout, Cin);
  B2U_CHECK_LAUNCH("pack_weights_first_fp32");
  return 0;
}

int b2u_pack_weights_multi(const void* table, int n, long long total_blocks, void* stream) {
  if (!table || n <= 0 || total_blocks <= 0) return set_error(B2U_ERR_ARG, "pack_weights_multi: empty table");
  v32_pack_weights_multi_kernel<<<static_cast<unsigned>(total_blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const V32PackEntry*>(table), n);
  B2U_CHECK_LAUNCH("pack_weights_multi_fp32");
  return 0;
}

static int v32_fprop(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* scale, const float* bias, void* y,
                     int N, int H, int W, int Cout, int taps, int relu, void* stream) {
  V32Conv p{};
  p.x0 = static_cast<const float*>(x0); p.C0 = C0;
  p.x1 = static_cast<const float*>(x1); p.C1 = x1 ? C1 : 0;
  p.wp = static_cast<const float*>(wf); p.bias = bias; p.scale = scale;
  p.y0 = static_cast<float*>(y); p.y1 = nullptr; p.split_c = Cout;
  p.N = N; p.H = H; p.W = W; p.Cout = Cout; p.taps = taps; p.relu = relu ? 1 : 0;
  return v32_launch_conv(p, static_cast<cudaStream_t>(stream));
}

int b2u_conv_fprop(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* bias, void* y, int N, int H,
                   int W, int Cout, int taps, int relu, int /*bn_override*/, void* stream) {
  return v32_fprop(x0, C0, x1, C1, wf, nullptr, bias, y, N, H, W, Cout, taps, relu, stream);
}

// the validation build takes BatchNorm statistics from z itself (b2u_bn_fwd_train_stats ignores the partials)
int b2u_conv_stat_rows(int N, int H, int W, int Cout, int /*taps*/, int /*bn_override*/) {
  return (N <= 0 || H <= 0 || W <= 0 || Cout <= 0) ? 0 : 1;
}
int b2u_conv_fprop_stats(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* bias, void* y, int N, int H,
                         int W, int Cout, int taps, int relu, int /*bn_override*/, float* /*stat_partial*/, int /*stat_rows*/,
                         void* stream) {
  return v32_fprop(x0, C0, x1, C1, wf, nullptr, bias, y, N, H, W, Cout, taps, relu, stream);
}
int b2u_conv_fprop_scaled(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* scale, const float* bias,
                          void* y, int N, int H, int W, int Cout, int taps, int relu, int /*bn_override*/, void* stream) {
  if (!scale) return set_error(B2U_ERR_ARG, "conv_fprop_scaled: scale vector missing");
  return v32_fprop(x0, C0, x1, C1, wf, scale, bias, y, N, H, W, Cout, taps, relu, stream);
}

int b2u_upsample2x_fwd(const void* x, void* y, int N, int H, int W, int C, void* stream);
// the validation build keeps the two steps apart: it up-samples into up_out (required here) and convolves the pair
int b2u_decoder_conv_fprop(const void* skip, int C0, const void* low, int C1, const void* wf, const float* scale, const float* bias,
                           void* y, void* up_out, int N, int H, int W, int Cout, int relu, int /*bn_override*/,
                           float* /*stat_partial*/, int /*stat_rows*/, void* stream) {
  if (!skip || !low) return set_error(B2U_ERR_ARG, "decoder_conv_fprop: skip and low tensors are required");
  if (!up_out) return set_error(B2U_ERR_ARG, "decoder_conv_fprop (fp32 validation build): up_out buffer is required");
  if ((H & 1) || (W & 1)) return set_error(B2U_ERR_SHAPE, "decoder_conv_fprop: H and W must be even");
  const int rc = b2u_upsample2x_fwd(low, up_out, N, H / 2, W / 2, C1, stream);
  if (rc) return rc;
  return v32_fprop(skip, C0, up_out, C1, wf, scale, bias, y, N, H, W, Cout, 9, relu, stream);
}

int b2u_conv_dgrad(const void* dz, int Cz, const void* wd, void* dx0, int C0, void* dx1, int C1, const void* mask, int N, int H,
                   int W, int taps, int /*bn_override*/, void* stream) {
  if (mask && dx1) return set_error(B2U_ERR_ARG, "dgrad: mask is only supported with a single output");
  V32Conv p{};
  p.x0 = static_cast<const float*>(dz); p.C0 = Cz; p.x1 = nullptr; p.C1 = 0;
  p.wp = static_cast<const float*>(wd);
  p.y0 = static_cast<float*>(dx0); p.y1 = static_cast<float*>(dx1);
  p.Cout = C0 + (dx1 ? C1 : 0); p.split_c = dx1 ? C0 : p.Cout;
  p.mask = static_cast<const float*>(mask); p.mask_c = C0;
  p.N = N; p.H = H; p.W = W; p.taps = taps; p.relu = 0;
  return v32_launch_conv(p, static_cast<cudaStream_t>(stream));
}

size_t b2u_conv_wgrad_workspace(int, int, int, int, int, int) { return 16; }

int b2u_conv_wgrad(const void* x0, int C0, const void* x1, int C1, const void* dz, int Cout, float* dw, float* db, void* /*ws*/,
                   size_t /*ws_bytes*/, int N, int H, int W, int taps, int first_cin, int flags, void* stream) {
  if (flags & ~2) return set_error(B2U_ERR_ARG, "wgrad: unknown flags 0x%x (only bit 1 is defined)", flags);
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "wgrad: empty tensor");
  if (taps != 9 && taps != 1) return set_error(B2U_ERR_SHAPE, "wgrad: taps must be 9 or 1");
  const int c1 = x1 ? C1 : 0;
  if (Cout <= 0 || Cout % 64 != 0 || C0 % 64 != 0 || c1 % 64 != 0 || C0 + c1 <= 0)
    return set_error(B2U_ERR_SHAPE, "wgrad: channels (%d,%d)->%d must be multiples of 64", C0, c1, Cout);
  if (first_cin > 0 && (taps != 1 || C0 != 64 || x1 || 9 * first_cin > 64))
    return set_error(B2U_ERR_SHAPE, "wgrad: first-layer mode needs the 64-column im2col tensor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dw) {
    V32Wgrad p{};
    p.x0 = static_cast<const float*>(x0); p.C0 = C0; p.x1 = static_cast<const float*>(x1); p.C1 = c1;
    p.dz = static_cast<const float*>(dz); p.Cout = Cout; p.dw = dw;
    p.N = N; p.H = H; p.W = W; p.taps = taps; p.first_cin = first_cin;
    dim3 grid(Cout / 64, (C0 + c1) / 64, taps);
    v32_wgrad_kernel<<<grid, 256, 0, st>>>(p);
    B2U_CHECK_LAUNCH("wgrad_fp32");
  }
  if (db) {
    v32_colsum_kernel<<<(Cout + 31) / 32, 256, 0, st>>>(static_cast<const float*>(dz), db, static_cast<long long>(N) * H * W, Cout);
    B2U_CHECK_LAUNCH("wgrad_bias_fp32");
  }
  return 0;
}

size_t b2u_bias_grad_workspace(int) { return 16; }
int b2u_bias_grad(const void* dz, float* db, void* /*ws*/, size_t /*ws_bytes*/, long long P, int C, void* stream) {
  if (P <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "bias_grad: empty tensor");
  v32_colsum_kernel<<<(C + 31) / 32, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const float*>(dz), db, P, C);
  B2U_CHECK_LAUNCH("bias_grad_fp32");
  return 0;
}

int b2u_maxpool2x2_fwd(const void* x, void* y, int N, int H, int W, int C, void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0 || (H & 1) || (W & 1)) return set_error(B2U_ERR_SHAPE, "maxpool: needs even H, W");
  const long long total = static_cast<long long>(N) * (H / 2) * (W / 2) * C;
  v32_maxpool_fwd_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(x), static_cast<float*>(y), N, H, W, C);
  B2U_CHECK_LAUNCH("maxpool_fwd_fp32");
  return 0;
}
int b2u_maxpool2x2_bwd(const void* dpool, const void* dskip, const void* y, void* dz, int N, int H, int W, int C, int relu_mask,
                       void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0 || (H & 1) || (W & 1)) return set_error(B2U_ERR_SHAPE, "maxpool_bwd: needs even H, W");
  const long long total = static_cast<long long>(N) * (H / 2) * (W / 2) * C;
  v32_maxpool_bwd_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(dpool), static_cast<const float*>(dskip), static_cast<const float*>(y), static_cast<float*>(dz), N, H,
      W, C, relu_mask);
  B2U_CHECK_LAUNCH("maxpool_bwd_fp32");
  return 0;
}

static inline float v32_ac_scale(int in, int out) { return out > 1 ? static_cast<float>(in - 1) / static_cast<float>(out - 1) : 0.f; }

int b2u_upsample2x_fwd(const void* x, void* y, int N, int H, int W, int C, void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "upsample: empty tensor");
  const long long total = static_cast<long long>(N) * 4 * H * W * C;
  v32_upsample_fwd_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(x), static_cast<float*>(y), N, H, W, C, v32_ac_scale(H, 2 * H), v32_ac_scale(W, 2 * W));
  B2U_CHECK_LAUNCH("upsample_fwd_fp32");
  return 0;
}
int b2u_upsample2x_bwd(const void* dup, const void* ylow, void* dlow, int N, int H, int W, int C, void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "upsample_bwd: empty tensor");
  const long long total = static_cast<long long>(N) * H * W * C;
  v32_upsample_bwd_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(dup), static_cast<const float*>(ylow), static_cast<float*>(dlow), N, H, W, C, v32_ac_scale(H, 2 * H),
      v32_ac_scale(W, 2 * W));
  B2U_CHECK_LAUNCH("upsample_bwd_fp32");
  return 0;
}

int b2u_head_fwd(const void* x, const float* w, const float* b, float* logits, int N, int H, int W, int Cin, int ncls, void* stream) {
  if (Cin != 64 || ncls <= 0 || ncls > 255) return set_error(B2U_ERR_SHAPE, "head_fwd: needs Cin == 64 and 1 <= classes <= 255 (got %d, %d)", Cin, ncls);
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "head_fwd: empty tensor");
  const long long HW = static_cast<long long>(H) * W, P = HW * N;
  v32_head_fwd_kernel<<<blocks_for(P * ncls, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const float*>(x), w, b,
                                                                                                 logits, HW, P, ncls);
  B2U_CHECK_LAUNCH("head_fwd_fp32");
  return 0;
}
size_t b2u_head_bwd_workspace(void) { return 16; }
size_t b2u_head_bwd_workspace_cls(int /*ncls*/) { return 16; }
int b2u_head_bwd(const float* dlogits, const void* x, const float* w, void* dx, float* dw, float* db, void* /*ws*/,
                 size_t /*ws_bytes*/, int N, int H, int W, int Cin, int ncls, int relu_mask, void* stream) {
  if (Cin != 64 || ncls <= 0 || ncls > 255) return set_error(B2U_ERR_SHAPE, "head_bwd: needs Cin == 64 and 1 <= classes <= 255");
  if (N <= 0 || H <= 0 || W <= 0) return set_error(B2U_ERR_SHAPE, "head_bwd: empty tensor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long HW = static_cast<long long>(H) * W, P = HW * N;
  if (dx) {
    v32_head_dgrad_kernel<<<blocks_for(P * 64, 256), 256, 0, st>>>(dlogits, static_cast<const float*>(x), w, static_cast<float*>(dx),
                                                                   HW, P, ncls, relu_mask);
    B2U_CHECK_LAUNCH("head_dgrad_fp32");
  }
  if (dw || db) {
    v32_head_wgrad_kernel<<<ncls * 65, 256, 0, st>>>(dlogits, static_cast<const float*>(x), dw, db, HW, P, ncls);
    B2U_CHECK_LAUNCH("head_wgrad_fp32");
  }
  return 0;
}

// workspace: [2C] doubles for the statistics
size_t b2u_bn_workspace(int C) { return static_cast<size_t>(2 * C) * sizeof(double) + 16; }

static int v32_bn_fwd_train(const void* z, const void* residual, void* y, const float* gamma, const float* beta, float* running_mean,
                            float* running_var, float* save_mean, float* save_invstd, void* ws, size_t ws_bytes, long long P, int C,
                            float eps, float momentum, int relu, void* stream) {
  if (P <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "bn: empty tensor");
  if (!ws || ws_bytes < b2u_bn_workspace(C) || !save_mean || !save_invstd) return set_error(B2U_ERR_ARG, "bn: workspace / save buffers missing");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double* sums = static_cast<double*>(ws);
  v32_bn_stats_kernel<<<(C + 31) / 32, 256, 0, st>>>(static_cast<const float*>(z), sums, P, C);
  B2U_CHECK_LAUNCH("bn_stats_fp32");
  v32_bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums, running_mean, running_var, save_mean, save_invstd, P, C, eps, momentum);
  B2U_CHECK_LAUNCH("bn_finalize_fp32");
  v32_bn_apply_kernel<<<blocks_for(P * C, 256), 256, 0, st>>>(static_cast<const float*>(z), static_cast<const float*>(residual),
                                                             static_cast<float*>(y), gamma, beta, save_mean, save_invstd, P * C, C, eps, 0,
                                                             relu);
  B2U_CHECK_LAUNCH("bn_apply_fp32");
  return 0;
}
int b2u_bn_fwd_train(const void* z, const void* residual, void* y, const float* gamma, const float* beta, float* running_mean,
                     float* running_var, float* save_mean, float* save_invstd, void* ws, size_t ws_bytes, long long P, int C, float eps,
                     float momentum, int relu, void* stream) {
  return v32_bn_fwd_train(z, residual, y, gamma, beta, running_mean, running_var, save_mean, save_invstd, ws, ws_bytes, P, C, eps,
                          momentum, relu, stream);
}
int b2u_bn_fwd_train_stats(const void* z, const void* residual, void* y, const float* gamma, const float* beta, float* running_mean,
                           float* running_var, float* save_mean, float* save_invstd, const float* /*stat_partial*/, int /*stat_rows*/,
                           void* ws, size_t ws_bytes, long long P, int C, float eps, float momentum, int relu, void* stream) {
  return v32_bn_fwd_train(z, residual, y, gamma, beta, running_mean, running_var, save_mean, save_invstd, ws, ws_bytes, P, C, eps,
                          momentum, relu, stream);
}
int b2u_bn_fwd_eval(const void* z, const void* residual, void* y, const float* gamma, const float* beta, const float* running_mean,
                    const float* running_var, void* /*ws*/, size_t /*ws_bytes*/, long long P, int C, float eps, int relu, void* stream) {
  if (P <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "bn: empty tensor");
  v32_bn_apply_kernel<<<blocks_for(P * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(z), static_cast<const float*>(residual), static_cast<float*>(y), gamma, beta, running_mean, running_var,
      P * C, C, eps, 1, relu);
  B2U_CHECK_LAUNCH("bn_eval_fp32");
  return 0;
}
int b2u_bn_bwd(const void* dy, const void* y, const void* z, const float* gamma, const float* beta, const float* save_mean,
               const float* save_invstd, void* dz, void* gout, float* dgamma, float* dbeta, void* ws, size_t ws_bytes, long long P, int C,
               int relu, void* stream) {
  if (P <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "bn_bwd: empty tensor");
  if (!ws || ws_bytes < b2u_bn_workspace(C)) return set_error(B2U_ERR_ARG, "bn_bwd: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double* sums = static_cast<double*>(ws);
  v32_bn_bwd_stats_kernel<<<(C + 31) / 32, 256, 0, st>>>(static_cast<const float*>(dy), static_cast<const float*>(y),
                                                         static_cast<const float*>(z), gamma, beta, save_mean, save_invstd, sums, P, C, relu);
  B2U_CHECK_LAUNCH("bn_bwd_stats_fp32");
  v32_bn_bwd_apply_kernel<<<blocks_for(P * C, 256), 256, 0, st>>>(static_cast<const float*>(dy), static_cast<const float*>(y),
                                                                 static_cast<const float*>(z), gamma, beta, save_mean, save_invstd, sums,
                                                                 static_cast<float*>(dz), static_cast<float*>(gout), dgamma, dbeta, P, C, relu);
  B2U_CHECK_LAUNCH("bn_bwd_apply_fp32");
  return 0;
}
int b2u_bn_fold(const float* gamma, const float* beta, const float* running_mean, const float* running_var, const float* conv_bias,
                float* scale, float* bias, int C, float eps, void* stream) {
  if (C <= 0 || !running_mean || !running_var || !scale || !bias) return set_error(B2U_ERR_ARG, "bn_fold: missing vectors");
  v32_bn_fold_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(gamma, beta, running_mean, running_var, conv_bias,
                                                                                    scale, bias, C, eps);
  B2U_CHECK_LAUNCH("bn_fold_fp32");
  return 0;
}


// ---- ResNet50 helpers, joins, resizes ----
int b2u_im2col_stem(const float* x, void* col, int N, int Cin, int H, int W, void* stream) {
  if (N <= 0 || Cin <= 0 || 49 * Cin > 192 || H < 1 || W < 1) return set_error(B2U_ERR_SHAPE, "im2col_stem: bad shape (Cin=%d)", Cin);
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  v32_im2col_stem_kernel<<<blocks_for(static_cast<long long>(N) * Ho * Wo * 192, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, static_cast<float*>(col), N, Cin, H, W, Ho, Wo);
  B2U_CHECK_LAUNCH("im2col_stem_fp32");
  return 0;
}
int b2u_pack_weights_im2col(const float* w, void* wf, int Cout, int Cin, int taps, int Kpad, void* stream) {
  if (Cout <= 0 || Cin <= 0 || taps <= 0 || taps * Cin > Kpad) return set_error(B2U_ERR_SHAPE, "pack_weights_im2col: bad shape");
  v32_pack_weights_im2col_kernel<<<(Cout * Kpad + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(w, static_cast<float*>(wf), Cout,
                                                                                                         Cin, taps, Kpad);
  B2U_CHECK_LAUNCH("pack_weights_im2col_fp32");
  return 0;
}
int b2u_conv_wgrad_im2col(const void* x0, int Kpad, const void* dz, int Cout, float* dw, void* /*ws*/, size_t /*ws_bytes*/, int N, int H,
                          int W, int cin, int taps, void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || Cout <= 0 || cin <= 0 || taps * cin > Kpad) return set_error(B2U_ERR_SHAPE, "wgrad_im2col: bad shape");
  v32_wgrad_im2col_kernel<<<Cout * cin * taps, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(x0), static_cast<const float*>(dz), dw, static_cast<long long>(N) * H * W, Kpad, Cout, cin, taps);
  B2U_CHECK_LAUNCH("wgrad_im2col_fp32");
  return 0;
}
int b2u_subsample2(const void* x, void* y, int N, int H, int W, int C, void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "subsample2: bad shape");
  const long long total = static_cast<long long>(N) * ((H + 1) / 2) * ((W + 1) / 2) * C;
  v32_subsample2_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const float*>(x),
                                                                                              static_cast<float*>(y), N, H, W, C);
  B2U_CHECK_LAUNCH("subsample2_fp32");
  return 0;
}
int b2u_zero_insert2(const void* y, void* x, int N, int H, int W, int C, void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "zero_insert2: bad shape");
  v32_zero_insert2_kernel<<<blocks_for(static_cast<long long>(N) * H * W * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(y), static_cast<float*>(x), N, H, W, C);
  B2U_CHECK_LAUNCH("zero_insert2_fp32");
  return 0;
}
int b2u_maxpool3x3s2_fwd(const void* x, void* y, int N, int H, int W, int C, void* stream) {
  if (N <= 0 || H < 3 || W < 3 || C <= 0) return set_error(B2U_ERR_SHAPE, "maxpool3x3s2: needs H,W >= 3");
  const int Ho = (H - 3 + 1) / 2 + 1, Wo = (W - 3 + 1) / 2 + 1;
  v32_maxpool3_fwd_kernel<<<blocks_for(static_cast<long long>(N) * Ho * Wo * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(x), static_cast<float*>(y), N, H, W, Ho, Wo, C);
  B2U_CHECK_LAUNCH("maxpool3x3s2_fwd_fp32");
  return 0;
}
int b2u_maxpool3x3s2_bwd(const void* dy, const void* x, void* dx, int N, int H, int W, int C, void* stream) {
  if (N <= 0 || H < 3 || W < 3 || C <= 0) return set_error(B2U_ERR_SHAPE, "maxpool3x3s2_bwd: needs H,W >= 3");
  const int Ho = (H - 3 + 1) / 2 + 1, Wo = (W - 3 + 1) / 2 + 1;
  v32_maxpool3_bwd_kernel<<<blocks_for(static_cast<long long>(N) * H * W * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(dy), static_cast<const float*>(x), static_cast<float*>(dx), N, H, W, Ho, Wo, C);
  B2U_CHECK_LAUNCH("maxpool3x3s2_bwd_fp32");
  return 0;
}
static int v32_join(const void* a, const void* b, void* out, long long n, int mode, void* stream) {
  if (n <= 0) return set_error(B2U_ERR_SHAPE, "join: empty tensor");
  v32_join_kernel<<<blocks_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const float*>(a), static_cast<const float*>(b),
                                                                                   static_cast<float*>(out), n, mode);
  B2U_CHECK_LAUNCH("join_fp32");
  return 0;
}
/* the ABI names say bf16; in this build the element type is fp32 like every other activation */
int b2u_add_bf16(const void* a, const void* b, void* out, long long n, void* stream) { return v32_join(a, b, out, n, 0, stream); }
int b2u_add_relu_bf16(const void* a, const void* b, void* out, long long n, void* stream) { return v32_join(a, b, out, n, 1, stream); }
int b2u_relu_bwd_bf16(const void* dy, const void* y, void* dx, long long n, void* stream) { return v32_join(dy, y, dx, n, 2, stream); }
int b2u_nchw_f32_to_nhwc_bf16_padded(const float* x, void* y, int N, int C, int H, int W, int Cpad, void* stream) {
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || Cpad < C) return set_error(B2U_ERR_SHAPE, "nchw_to_nhwc_padded: bad shape");
  const long long HW = static_cast<long long>(H) * W;
  v32_nchw_to_nhwc_padded_kernel<<<blocks_for(N * HW * Cpad, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, static_cast<float*>(y), N, C,
                                                                                                              HW, Cpad);
  B2U_CHECK_LAUNCH("nchw_to_nhwc_padded_fp32");
  return 0;
}
int b2u_first_conv_dgrad_input(const void* dz, int Cz, const float* w, float* dx, int N, int Cin, int H, int W, int Cout,
                               void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || Cin <= 0 || 9 * Cin > 64 || Cout <= 0 || Cout > Cz || Cz % 16 != 0)
    return set_error(B2U_ERR_SHAPE, "first_conv_dgrad_input: bad shape (Cin=%d Cout=%d Cz=%d)", Cin, Cout, Cz);
  if (reinterpret_cast<uintptr_t>(dz) % 16 != 0) return set_error(B2U_ERR_ARG, "first_conv_dgrad_input: dz must be 16-byte aligned");
  v32_conv_dgrad_input_kernel<<<blocks_for(static_cast<long long>(N) * Cin * H * W, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(dz), Cz, w, dx, N, Cin, H, W, H, W, Cout, 3, 1, 1);
  B2U_CHECK_LAUNCH("first_conv_dgrad_input_fp32");
  return 0;
}
int b2u_stem_dgrad_input(const void* dz, int Cz, const float* w, float* dx, int N, int Cin, int H, int W, int Cout, void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || Cin <= 0 || 49 * Cin > 192 || Cout <= 0 || Cout > Cz || Cz % 16 != 0)
    return set_error(B2U_ERR_SHAPE, "stem_dgrad_input: bad shape (Cin=%d Cout=%d Cz=%d)", Cin, Cout, Cz);
  if (reinterpret_cast<uintptr_t>(dz) % 16 != 0) return set_error(B2U_ERR_ARG, "stem_dgrad_input: dz must be 16-byte aligned");
  v32_conv_dgrad_input_kernel<<<blocks_for(static_cast<long long>(N) * Cin * H * W, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(dz), Cz, w, dx, N, Cin, H, W, (H - 1) / 2 + 1, (W - 1) / 2 + 1, Cout, 7, 2, 3);
  B2U_CHECK_LAUNCH("stem_dgrad_input_fp32");
  return 0;
}
int b2u_nhwc_bf16_padded_to_nchw_f32(const void* x, float* y, int N, int C, int H, int W, int Cpad, void* stream) {
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || Cpad < C || Cpad % 8 != 0)
    return set_error(B2U_ERR_SHAPE, "nhwc_bf16_padded_to_nchw_f32: bad shape (C=%d Cpad=%d)", C, Cpad);
  if (reinterpret_cast<uintptr_t>(x) % 16 != 0) return set_error(B2U_ERR_ARG, "nhwc_bf16_padded_to_nchw_f32: x must be 16-byte aligned");
  const long long HW = static_cast<long long>(H) * W;
  v32_nhwc_padded_to_nchw_kernel<<<blocks_for(N * C * HW, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(x), y, N, C, HW, Cpad);
  B2U_CHECK_LAUNCH("nhwc_padded_to_nchw_fp32");
  return 0;
}
int b2u_resize_bilinear_f32_fwd(const float* x, float* y, long long NC, int Hi, int Wi, int Ho, int Wo, void* stream) {
  if (NC <= 0 || Hi <= 0 || Wi <= 0 || Ho <= 0 || Wo <= 0) return set_error(B2U_ERR_SHAPE, "resize_bilinear: bad shape");
  v32_resize_fwd_kernel<<<blocks_for(NC * Ho * Wo, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, NC, Hi, Wi, Ho, Wo,
                                                                                                     v32_ac_scale(Hi, Ho), v32_ac_scale(Wi, Wo));
  B2U_CHECK_LAUNCH("resize_bilinear_fwd_fp32");
  return 0;
}
int b2u_resize_bilinear_f32_bwd(const float* dy, float* dx, long long NC, int Hi, int Wi, int Ho, int Wo, void* stream) {
  if (NC <= 0 || Hi <= 0 || Wi <= 0 || Ho <= 0 || Wo <= 0) return set_error(B2U_ERR_SHAPE, "resize_bilinear_bwd: bad shape");
  v32_resize_bwd_kernel<<<blocks_for(NC * Hi * Wi, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(dy, dx, NC, Hi, Wi, Ho, Wo,
                                                                                                     v32_ac_scale(Hi, Ho), v32_ac_scale(Wi, Wo));
  B2U_CHECK_LAUNCH("resize_bilinear_bwd_fp32");
  return 0;
}

// ---- depthwise / squeeze-excite support ----
int b2u_dwconv3x3_fwd(const void* x, const float* w, const float* bias, void* y, int N, int H, int W, int C, int flip, void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "dwconv3x3: bad shape");
  v32_dwconv_kernel<<<blocks_for(static_cast<long long>(N) * H * W * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(x), w, bias, static_cast<float*>(y), N, H, W, C, flip);
  B2U_CHECK_LAUNCH("dwconv3x3_fp32");
  return 0;
}
size_t b2u_dwconv3x3_wgrad_workspace(int) { return 16; }
int b2u_dwconv3x3_wgrad(const void* x, const void* dy, float* dw, float* db, void* /*ws*/, size_t /*ws_bytes*/, int N, int H, int W, int C,
                        void* stream) {
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "dwconv3x3_wgrad: bad shape");
  v32_dwconv_wgrad_kernel<<<C * 10, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const float*>(x), static_cast<const float*>(dy),
                                                                               dw, db, N, H, W, C);
  B2U_CHECK_LAUNCH("dwconv3x3_wgrad_fp32");
  return 0;
}
int b2u_spatial_reduce_workspace_floats(int, int) { return 4; }
int b2u_spatial_reduce(const void* a, const void* b, float* out, void* /*ws*/, size_t /*ws_bytes*/, int N, long long HW, int C, float scale,
                       void* stream) {
  if (N <= 0 || HW <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "spatial_reduce: bad shape");
  v32_spatial_reduce_kernel<<<dim3((C + 31) / 32, N), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const float*>(a), static_cast<const float*>(b), out, HW, C, scale);
  B2U_CHECK_LAUNCH("spatial_reduce_fp32");
  return 0;
}
int b2u_scale_nc(const void* x, const float* s, const float* a, void* y, int N, long long HW, int C, void* stream) {
  if (N <= 0 || HW <= 0 || C <= 0) return set_error(B2U_ERR_SHAPE, "scale_nc: bad shape");
  const long long total = static_cast<long long>(N) * HW * C;
  v32_scale_nc_kernel<<<blocks_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const float*>(x), s, a,
                                                                                            static_cast<float*>(y), HW, C, total);
  B2U_CHECK_LAUNCH("scale_nc_fp32");
  return 0;
}

}  // extern "C"
