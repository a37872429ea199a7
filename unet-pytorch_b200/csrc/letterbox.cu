// letterbox.cu -- the predictor's front end on the device (utils/utils.py:22-34 resize_image + preprocess_input + the
// NCHW transpose of unet.py:116-120) for a batch of uint8 RGB images of different sizes, bit for bit what PIL 12's
// Image.resize(..., BICUBIC) pasted on a (128, 128, 128) canvas and numpy's float32 / 255.0 give.
//
// Pillow's 8-bit resampling (Resample.c), restated:
//   per axis: scale = in / out, fs = max(scale, 1), support = 2 fs, ksize = 2 ceil(support) + 1; for output o:
//   center = (o + 0.5) scale, xmin = max(int(center - support + 0.5), 0), n = min(int(center + support + 0.5), in) - xmin,
//   w[k] = bicubic((k + xmin - center + 0.5) * (1 / fs)) (a = -0.5), normalised by their double sum (k ascending),
//   quantised to 22 fractional bits (round half away from zero, then truncation).
//   Each pass: acc = 2^21 + sum src * w in int32, stored as clamp(acc >> 22, 0, 255); horizontal first -- vertical first
//   for an image more than 100 times taller than wide whose height shrinks -- and an axis whose size does not change is
//   not resampled.
// The coefficients are computed here in double with explicit _rn intrinsics, so that no FMA contraction can move a
// weight by one unit.  Three launches per batch: coefficients, first pass into a uint8 intermediate, second pass +
// canvas + IEEE fp32 division by 255 written as NCHW fp32 (x * (1/255.f) differs on 126 byte values).
#include "b2u_internal.h"

namespace b2u {

#define B2U_CHECK_LAUNCH(name)                                                                           \
  do {                                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                                \
    if (e__ != cudaSuccess) return b2u::set_error(B2U_ERR_CUDA, name " launch: %s", cudaGetErrorString(e__)); \
    b2u::note_launch();                                                                                  \
  } while (0)

constexpr int kLbThreads = 128;
constexpr int kLbRowBlocks = 256;        // first pass: rows are strided over this many blocks per image
constexpr int kLbPrecision = 22;

// one image of a batch (64 bytes, include/b2u.h); the last five fields are filled by b2u_letterbox_workspace
struct LetterboxItem {
  const uint8_t* src;                    // uint8 [ih][iw][3], device
  int ih, iw, nh, nw, dy, dx;
  int kx, ky;                            // taps per output column / row (0: the axis is not resampled)
  long long coef_x, coef_y, tmp;         // workspace offsets: int2 bounds [nw] + int weights [nw][kx]; the same for y;
                                         // uint8 first-pass image ([ih][nw][3], or [nh][iw][3] when vertical_first)
};
static_assert(sizeof(LetterboxItem) == 64, "LetterboxItem is part of the ABI");

static inline long long align16(long long v) { return (v + 15) & ~15LL; }

// Image.resize of PIL >= 9 resamples an image more than 100 times taller than wide vertically first when it shrinks its
// height (two single-axis calls); the rounding of the uint8 intermediate makes the order visible
__host__ __device__ __forceinline__ bool vertical_first(int ih, int iw, int nh) {
  return static_cast<long long>(ih) > 100LL * iw && nh < ih;
}

// Pillow's ksize for one axis; the device recomputes the same scale, so the table stride matches what it writes
static int bicubic_ksize(int in, int out) {
  double fs = static_cast<double>(in) / out;
  if (fs < 1.0) fs = 1.0;
  return static_cast<int>(ceil(2.0 * fs)) * 2 + 1;
}

__device__ __forceinline__ double bicubic_rn(double x) {
  if (x < 0.0) x = -x;
  if (x < 1.0) return __dadd_rn(__dmul_rn(__dmul_rn(__dsub_rn(__dmul_rn(1.5, x), 2.5), x), x), 1.0);   // ((a+2)x-(a+3))x*x+1
  if (x < 2.0) return __dmul_rn(__dsub_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dsub_rn(x, 5.0), x), 8.0), x), 4.0), -0.5);
  return 0.0;
}

// blockIdx.z = axis (0: x, 1: y), blockIdx.y = image, one thread per output index
__global__ void __launch_bounds__(kLbThreads)
letterbox_coeffs_kernel(const LetterboxItem* __restrict__ items, uint8_t* __restrict__ ws) {
  const LetterboxItem it = items[blockIdx.y];
  const bool xa = blockIdx.z == 0;
  const int in = xa ? it.iw : it.ih, out = xa ? it.nw : it.nh, K = xa ? it.kx : it.ky;
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (K == 0 || o >= out) return;
  int2* bounds = reinterpret_cast<int2*>(ws + (xa ? it.coef_x : it.coef_y));
  int* kk = reinterpret_cast<int*>(bounds + out) + static_cast<size_t>(o) * K;
  const double scale = __ddiv_rn(static_cast<double>(in), static_cast<double>(out));
  const double fs = scale < 1.0 ? 1.0 : scale;
  const double support = __dmul_rn(2.0, fs), ss = __ddiv_rn(1.0, fs);
  const double center = __dmul_rn(__dadd_rn(static_cast<double>(o), 0.5), scale);
  int xmin = static_cast<int>(__dadd_rn(__dsub_rn(center, support), 0.5));
  if (xmin < 0) xmin = 0;
  int xmax = static_cast<int>(__dadd_rn(__dadd_rn(center, support), 0.5));
  if (xmax > in) xmax = in;
  const int n = xmax - xmin;
  double ww = 0.0;
  for (int k = 0; k < n; ++k) ww = __dadd_rn(ww, bicubic_rn(__dmul_rn(__dadd_rn(__dsub_rn(static_cast<double>(k + xmin), center), 0.5), ss)));
  for (int k = 0; k < n; ++k) {
    double w = bicubic_rn(__dmul_rn(__dadd_rn(__dsub_rn(static_cast<double>(k + xmin), center), 0.5), ss));
    if (ww != 0.0) w = __ddiv_rn(w, ww);
    const double q = __dmul_rn(w, static_cast<double>(1 << kLbPrecision));
    kk[k] = static_cast<int>(w < 0.0 ? __dadd_rn(-0.5, q) : __dadd_rn(0.5, q));
  }
  bounds[o] = make_int2(xmin, n);
}

__device__ __forceinline__ uint8_t clip8(int acc) {
  const int v = acc >> kLbPrecision;
  return static_cast<uint8_t>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// n taps of one output pixel: p = the first tap's pixel, step = bytes between taps
__device__ __forceinline__ void resample3(const uint8_t* __restrict__ p, size_t step, const int* __restrict__ k, int n, int v[3]) {
  int a0 = 1 << (kLbPrecision - 1), a1 = a0, a2 = a0;
  for (int t = 0; t < n; ++t, p += step) {
    const int w = k[t];
    a0 += p[0] * w; a1 += p[1] * w; a2 += p[2] * w;
  }
  v[0] = clip8(a0); v[1] = clip8(a1); v[2] = clip8(a2);
}

__device__ __forceinline__ int2 lb_bounds(const uint8_t* ws, long long off, int o) { return reinterpret_cast<const int2*>(ws + off)[o]; }
__device__ __forceinline__ const int* lb_weights(const uint8_t* ws, long long off, int out, int K, int o) {
  return reinterpret_cast<const int*>(reinterpret_cast<const int2*>(ws + off) + out) + static_cast<size_t>(o) * K;
}

// first pass into the uint8 intermediate: horizontal, [ih][iw] -> [ih][nw]; or, for a tall image (vertical_first),
// vertical, [ih][iw] -> [nh][iw].  blockIdx.x * blockDim.x + threadIdx.x = column, rows strided over blockIdx.y; z = image
__global__ void __launch_bounds__(kLbThreads)
letterbox_first_pass_kernel(const LetterboxItem* __restrict__ items, uint8_t* __restrict__ ws) {
  const LetterboxItem it = items[blockIdx.z];
  const bool vfirst = vertical_first(it.ih, it.iw, it.nh);
  if (vfirst ? it.ky == 0 : it.kx == 0) return;
  const int rows = vfirst ? it.nh : it.ih, cols = vfirst ? it.iw : it.nw;
  uint8_t* tmp = ws + it.tmp;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cols; c += gridDim.x * blockDim.x) {
    for (int r = blockIdx.y; r < rows; r += gridDim.y) {
      int v[3];
      if (vfirst) {
        const int2 b = lb_bounds(ws, it.coef_y, r);
        resample3(it.src + (static_cast<size_t>(b.x) * it.iw + c) * 3, static_cast<size_t>(it.iw) * 3,
                  lb_weights(ws, it.coef_y, it.nh, it.ky, r), b.y, v);
      } else {
        const int2 b = lb_bounds(ws, it.coef_x, c);
        resample3(it.src + (static_cast<size_t>(r) * it.iw + b.x) * 3, 3, lb_weights(ws, it.coef_x, it.nw, it.kx, c), b.y, v);
      }
      uint8_t* d = tmp + (static_cast<size_t>(r) * cols + c) * 3;
      d[0] = static_cast<uint8_t>(v[0]); d[1] = static_cast<uint8_t>(v[1]); d[2] = static_cast<uint8_t>(v[2]);
    }
  }
}

// second pass + paste on the grey canvas + / 255: out [count][3][H][W] fp32; blockIdx.y = canvas row, blockIdx.z = image
__global__ void __launch_bounds__(kLbThreads)
letterbox_second_pass_kernel(const LetterboxItem* __restrict__ items, const uint8_t* __restrict__ ws, float* __restrict__ out,
                             int H, int W) {
  const LetterboxItem it = items[blockIdx.z];
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= W) return;
  const size_t plane = static_cast<size_t>(H) * W;
  float* o = out + static_cast<size_t>(blockIdx.z) * 3 * plane + static_cast<size_t>(y) * W + x;
  const int ox = x - it.dx, oy = y - it.dy;
  if (ox < 0 || ox >= it.nw || oy < 0 || oy >= it.nh) {
    const float grey = __fdiv_rn(128.f, 255.f);
    o[0] = grey; o[plane] = grey; o[2 * plane] = grey;
    return;
  }
  int v[3];
  if (vertical_first(it.ih, it.iw, it.nh)) {          // intermediate [nh][iw]; horizontal pass left
    const uint8_t* img = ws + it.tmp;
    if (it.kx) {
      const int2 b = lb_bounds(ws, it.coef_x, ox);
      resample3(img + (static_cast<size_t>(oy) * it.iw + b.x) * 3, 3, lb_weights(ws, it.coef_x, it.nw, it.kx, ox), b.y, v);
    } else {
      const uint8_t* s = img + (static_cast<size_t>(oy) * it.iw + ox) * 3;
      v[0] = s[0]; v[1] = s[1]; v[2] = s[2];
    }
  } else {                                            // intermediate [ih][nw] (the source itself when nw == iw); vertical left
    const uint8_t* img = it.kx ? ws + it.tmp : it.src;
    if (it.ky) {
      const int2 b = lb_bounds(ws, it.coef_y, oy);
      resample3(img + (static_cast<size_t>(b.x) * it.nw + ox) * 3, static_cast<size_t>(it.nw) * 3,
                lb_weights(ws, it.coef_y, it.nh, it.ky, oy), b.y, v);
    } else {
      const uint8_t* s = img + (static_cast<size_t>(oy) * it.nw + ox) * 3;
      v[0] = s[0]; v[1] = s[1]; v[2] = s[2];
    }
  }
  o[0] = __fdiv_rn(static_cast<float>(v[0]), 255.f);
  o[plane] = __fdiv_rn(static_cast<float>(v[1]), 255.f);
  o[2 * plane] = __fdiv_rn(static_cast<float>(v[2]), 255.f);
}

}  // namespace b2u

extern "C" {
using namespace b2u;

// host_items: count LetterboxItems in HOST memory with src, ih, iw, nh, nw, dy, dx set; fills kx, ky and the workspace
// offsets and returns the workspace size in bytes (0 on a bad item, with the message in b2u_last_error)
size_t b2u_letterbox_workspace(void* host_items, int count, int H, int W) {
  if (!host_items || count <= 0 || H <= 0 || W <= 0 || H > 65535) {
    set_error(B2U_ERR_SHAPE, "letterbox_workspace: bad batch (count %d, H %d, W %d)", count, H, W);
    return 0;
  }
  LetterboxItem* items = static_cast<LetterboxItem*>(host_items);
  long long off = 0;
  for (int i = 0; i < count; ++i) {
    LetterboxItem& it = items[i];
    if (!it.src || it.ih <= 0 || it.iw <= 0 || it.nh <= 0 || it.nw <= 0 || it.dy < 0 || it.dx < 0 ||
        it.dy + it.nh > H || it.dx + it.nw > W) {
      set_error(B2U_ERR_SHAPE, "letterbox_workspace: item %d (%dx%d -> %dx%d at %d,%d) does not fit a %dx%d canvas", i,
                it.iw, it.ih, it.nw, it.nh, it.dx, it.dy, W, H);
      return 0;
    }
    it.kx = it.nw != it.iw ? bicubic_ksize(it.iw, it.nw) : 0;
    it.ky = it.nh != it.ih ? bicubic_ksize(it.ih, it.nh) : 0;
    it.coef_x = off;
    if (it.kx) off = align16(off + static_cast<long long>(it.nw) * (8 + 4LL * it.kx));
    it.coef_y = off;
    if (it.ky) off = align16(off + static_cast<long long>(it.nh) * (8 + 4LL * it.ky));
    it.tmp = off;
    if (vertical_first(it.ih, it.iw, it.nh)) off = align16(off + static_cast<long long>(it.nh) * it.iw * 3);
    else if (it.kx) off = align16(off + static_cast<long long>(it.ih) * it.nw * 3);
  }
  return static_cast<size_t>(off < 16 ? 16 : off);
}

// items: the table b2u_letterbox_workspace filled, copied to DEVICE memory; out: fp32 [count][3][H][W];
// ws: device workspace of the size b2u_letterbox_workspace returned for the same table
int b2u_letterbox_bicubic(const void* items, int count, float* out, int H, int W, void* ws, size_t ws_bytes, void* stream) {
  if (!items || !out || !ws || count <= 0 || count > 65535 || H <= 0 || W <= 0 || H > 65535 || ws_bytes < 16)
    return set_error(B2U_ERR_SHAPE, "letterbox_bicubic: bad arguments (count %d, H %d, W %d)", count, H, W);
  const LetterboxItem* it = static_cast<const LetterboxItem*>(items);
  uint8_t* w = static_cast<uint8_t*>(ws);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned side = static_cast<unsigned>(((H > W ? H : W) + kLbThreads - 1) / kLbThreads);
  letterbox_coeffs_kernel<<<dim3(side, count, 2), kLbThreads, 0, st>>>(it, w);
  B2U_CHECK_LAUNCH("letterbox_coeffs");
  const unsigned cols = static_cast<unsigned>((W + kLbThreads - 1) / kLbThreads);
  letterbox_first_pass_kernel<<<dim3(cols, kLbRowBlocks, count), kLbThreads, 0, st>>>(it, w);
  B2U_CHECK_LAUNCH("letterbox_first_pass");
  letterbox_second_pass_kernel<<<dim3(cols, H, count), kLbThreads, 0, st>>>(it, w, out, H, W);
  B2U_CHECK_LAUNCH("letterbox_second_pass");
  return 0;
}

}  // extern "C"
