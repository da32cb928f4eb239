// imgproc.cuh — §10 f6: CLIP's image preprocessing on the device, from decoded uint8 RGB pixels to the vision
// tower's pixel_values [n, 3, crop, crop], bit for bit what the HuggingFace processor returns.
//
// Per image: resize so the shorter side is shortest_edge (transformers' get_resize_output_image_size), BICUBIC with
// the chosen library's uint8 arithmetic, center crop (top = (H' - crop) / 2), then rescale / normalise as that
// processor does.  The two numerics (restated in tests/helpers/resample_ref.py, which the CPU tests hold to the
// installed libraries):
//   backend 0  CLIPImageProcessor (torchvision backend): aten's uint8 antialiased bicubic — int16 coefficients at the
//              largest precision p that keeps round(max weight of the axis * 2^(p+1)) below 2^15; then
//              (float(x) - m) / s with m = float(mean) * float(1 / rescale), s likewise (the fused rescale+normalise).
//   backend 1  CLIPImageProcessorPil: Pillow's Image.resize(BICUBIC) — 22-bit coefficients; then
//              float(double(x) * rescale), (v - float(mean)) / float(std).
// Both: filterscale = max(n_in / n_out, 1), support = 2 * filterscale, center = (i + 0.5) * n_in / n_out,
// taps [max(int(center - support + 0.5), 0), min(int(center + support + 0.5), n_in)), cubic a = -0.5 at
// (j + xmin - center + 0.5) / filterscale, normalised by the taps' sum, rounded half away from zero; the horizontal
// pass first into uint8 ((2^(p-1) + sum w q) >> p clipped to 0..255), then the vertical pass; a pass whose axis keeps
// its size is skipped.  The two cubics differ only in how the outer lobe is evaluated (kept literally, see
// cubic_w).  The coefficient arithmetic is IEEE double (the library is built with --fmad=false, so nothing is
// contracted), on the device: only (H, W) per image crosses the bus besides the pixels.
//
// Kernels, per chunk of images of any sizes (packed HWC uint8, per-image byte offset):
//   imgproc_bits_kernel   one CTA per (image, axis): the precision p (aten: from the axis' largest weight over ALL its
//                         outputs);
//   imgproc_coeff_kernel  one CTA per (image, axis): the integer taps of the outputs the crop keeps (the double
//                         divisions of the two steps sit in separate kernels, so neither spills around the division's
//                         slow-path call);
//   imgproc_hpass_kernel  horizontal pass of the input rows the kept output rows read, the kept columns only, into a
//                         uint8 intermediate [rows][crop_w][3];
//   imgproc_vpass_kernel  vertical pass fused with the crop, the float rescale / normalise and the CHW layout,
//                         writing straight into pixel_values.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace rse {

constexpr int kIpThreads = 256;
constexpr int kIpMaxScale = 32;                    // largest downscale per axis on the device (n_in / n_out)
constexpr int kIpMaxTaps = 2 * (2 * kIpMaxScale) + 1;

// one image of a chunk, filled by the host
struct IpImage {
  long long off;        // byte offset of the HWC pixels in the chunk's input buffer
  int H, W;             // input
  int nh, nw;           // resized
  int top, left;        // crop origin in the resized image
  int ylo, rows;        // input rows the vertical pass reads: [ylo, ylo + rows)
  long long mid_off;    // byte offset of this image's intermediate [rows][crop_w][3]
  int out;              // output image index of the call
  int pad;
};

// per-axis output of imgproc_coeff_kernel: for output k of the kept range (k = 0 .. crop - 1), the first input
// index and the tap count; weights [K] (zero past the count); bits = p (0: the axis keeps its size, no pass)
struct IpAxis {
  int bits, pad;
};

__device__ __forceinline__ double cubic_w(double x, int backend) {
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return backend == 1 ? ((a + 2.0) * x - (a + 3.0)) * x * x + 1 : ((a + 2) * x - (a + 3)) * x * x + 1;
  if (x < 2.0) return backend == 1 ? (((x - 5) * x + 8) * x - 4) * a : ((a * x - 5 * a) * x + 8 * a) * x - 4 * a;
  return 0.0;
}

// taps of output i of an axis n_in -> n_out: first index, count, their sum (the normaliser) — the sum is taken in tap
// order, as both libraries do
__device__ __forceinline__ void ip_taps(int i, int n_in, int n_out, int K, int backend, double& center, double& inv,
                                        int& lo, int& cnt, double& tot) {
  const double scale = static_cast<double>(n_in) / n_out;
  const double fs = scale > 1.0 ? scale : 1.0;
  const double support = 2.0 * fs;
  inv = 1.0 / fs;
  center = (i + 0.5) * scale;
  lo = static_cast<int>(center - support + 0.5);
  if (lo < 0) lo = 0;
  int hi = static_cast<int>(center + support + 0.5);
  if (hi > n_in) hi = n_in;
  cnt = hi - lo;
  if (cnt < 0) cnt = 0;
  if (cnt > K) cnt = K;
  tot = 0.0;
  for (int j = 0; j < cnt; ++j) tot += cubic_w((j + lo - center + 0.5) * inv, backend);
}

// the axis' precision p into axes[(image, axis)]: 0 when the axis keeps its size (no pass), Pillow's fixed 22, or
// aten's from the largest normalised weight over ALL outputs of the axis.  grid (n_img, 2): axis 0 horizontal
// (W -> nw), axis 1 vertical (H -> nh).
__global__ void __launch_bounds__(kIpThreads)
imgproc_bits_kernel(const IpImage* __restrict__ imgs, int backend, int K, IpAxis* __restrict__ axes) {
  __shared__ double s_max[kIpThreads / 32];
  const IpImage im = imgs[blockIdx.x];
  const int axis = blockIdx.y;
  const int n_in = axis == 0 ? im.W : im.H, n_out = axis == 0 ? im.nw : im.nh;
  const size_t t = static_cast<size_t>(blockIdx.x) * 2 + axis;
  if (n_in == n_out || backend == 1) {
    if (threadIdx.x == 0) axes[t].bits = n_in == n_out ? 0 : 22;     // Pillow: PRECISION_BITS = 32 - 8 - 2
    return;
  }
  double m = 0.0;
  for (int i = threadIdx.x; i < n_out; i += kIpThreads) {
    double center, inv, tot; int lo, cnt;
    ip_taps(i, n_in, n_out, K, backend, center, inv, lo, cnt, tot);
    for (int j = 0; j < cnt; ++j) {
      double w = cubic_w((j + lo - center + 0.5) * inv, backend);
      if (tot != 0.0) w /= tot;
      m = fmax(m, w);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x != 0) return;
  m = s_max[0];
  for (int wi = 1; wi < kIpThreads / 32; ++wi) m = fmax(m, s_max[wi]);
  int bits = 0;
  while (bits < 22 && static_cast<int>(0.5 + m * static_cast<double>(1 << (bits + 1))) < (1 << 15)) ++bits;
  axes[t].bits = bits;
}

// the integer taps of the outputs the crop keeps: axis 0 [left, left + crop_w), axis 1 [top, top + crop_h).
// Tables: span [n_img][2][crop_max] int2 {first, count}, w [n_img][2][crop_max][K] int32.  grid (n_img, 2), after
// imgproc_bits_kernel.
__global__ void __launch_bounds__(kIpThreads)
imgproc_coeff_kernel(const IpImage* __restrict__ imgs, int backend, int crop_h, int crop_w, int crop_max, int K,
                     const IpAxis* __restrict__ axes, int2* __restrict__ span, int* __restrict__ wq) {
  const IpImage im = imgs[blockIdx.x];
  const int axis = blockIdx.y;
  const int n_in = axis == 0 ? im.W : im.H, n_out = axis == 0 ? im.nw : im.nh;
  const int first = axis == 0 ? im.left : im.top, kept = axis == 0 ? crop_w : crop_h;
  const size_t t = static_cast<size_t>(blockIdx.x) * 2 + axis;
  const int bits = axes[t].bits;
  if (bits == 0) return;
  const double q = static_cast<double>(1 << bits);
  // per tile of kept outputs: the taps' first index, count and sum into shared memory, then one thread per
  // (output, tap) — few values live across the division, and the table rows are written contiguously
  __shared__ double s_center[kIpThreads], s_inv[kIpThreads], s_tot[kIpThreads];
  __shared__ int s_lo[kIpThreads], s_cnt[kIpThreads];
  for (int k0 = 0; k0 < kept; k0 += kIpThreads) {
    const int n_k = min(kIpThreads, kept - k0);
    __syncthreads();
    if (threadIdx.x < n_k) {
      double center, inv, tot; int lo, cnt;
      ip_taps(first + k0 + threadIdx.x, n_in, n_out, K, backend, center, inv, lo, cnt, tot);
      s_center[threadIdx.x] = center; s_inv[threadIdx.x] = inv; s_tot[threadIdx.x] = tot;
      s_lo[threadIdx.x] = lo; s_cnt[threadIdx.x] = cnt;
      span[t * crop_max + k0 + threadIdx.x] = make_int2(lo, cnt);
    }
    __syncthreads();
    int* w = wq + (t * crop_max + k0) * K;
    for (int e = threadIdx.x; e < n_k * K; e += kIpThreads) {
      const int k = e / K, j = e - k * K;
      int v = 0;
      if (j < s_cnt[k]) {
        double x = cubic_w((j + s_lo[k] - s_center[k] + 0.5) * s_inv[k], backend);
        if (s_tot[k] != 0.0) x /= s_tot[k];
        x *= q;
        v = x < 0 ? static_cast<int>(-0.5 + x) : static_cast<int>(0.5 + x);
      }
      w[e] = v;
    }
  }
}

__device__ __forceinline__ int ip_clip8(int acc, int bits) {
  const int v = acc >> bits;
  return v < 0 ? 0 : (v > 255 ? 255 : v);
}

// grid (ceil(max rows * crop_w / 256), n_img): one thread per (input row of [ylo, ylo + rows), kept output column),
// all three channels.  An axis without a pass copies the kept columns.
__global__ void __launch_bounds__(kIpThreads)
imgproc_hpass_kernel(const IpImage* __restrict__ imgs, const uint8_t* __restrict__ in, int crop_w, int crop_max,
                     int K, const IpAxis* __restrict__ axes, const int2* __restrict__ span,
                     const int* __restrict__ wq, uint8_t* __restrict__ mid) {
  const IpImage im = imgs[blockIdx.y];
  const int idx = blockIdx.x * kIpThreads + threadIdx.x;
  if (idx >= im.rows * crop_w) return;
  const int r = idx / crop_w, ox = idx - r * crop_w;
  const uint8_t* row = in + im.off + (static_cast<long long>(im.ylo + r) * im.W) * 3;
  uint8_t* o = mid + im.mid_off + static_cast<long long>(idx) * 3;
  const size_t t = static_cast<size_t>(blockIdx.y) * 2;
  const int bits = axes[t].bits;
  if (bits == 0) {
    const uint8_t* p = row + (im.left + ox) * 3;
    o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
    return;
  }
  const int2 sp = span[t * crop_max + ox];
  const int* w = wq + (t * crop_max + ox) * K;
  int a0 = 1 << (bits - 1), a1 = a0, a2 = a0;
  const uint8_t* p = row + sp.x * 3;
  for (int j = 0; j < sp.y; ++j, p += 3) {
    const int c = w[j];
    a0 += c * p[0]; a1 += c * p[1]; a2 += c * p[2];
  }
  o[0] = static_cast<uint8_t>(ip_clip8(a0, bits));
  o[1] = static_cast<uint8_t>(ip_clip8(a1, bits));
  o[2] = static_cast<uint8_t>(ip_clip8(a2, bits));
}

// the float step after the resize, per channel: v = x; rescale_mode 1: v = v * rf (float), 2: v = float(double(x) *
// rd); normalise: v = (v - m[c]) / s[c] (float, correctly rounded)
struct IpNorm {
  int rescale_mode, normalize;
  float rf;
  double rd;
  float m[3], s[3];
};

// grid (ceil(crop_h * crop_w / 256), n_img): one thread per output pixel, three channels, written CHW into
// out [n, 3, crop_h, crop_w]
__global__ void __launch_bounds__(kIpThreads)
imgproc_vpass_kernel(const IpImage* __restrict__ imgs, int crop_h, int crop_w, int crop_max, int K,
                     const IpAxis* __restrict__ axes, const int2* __restrict__ span, const int* __restrict__ wq,
                     const uint8_t* __restrict__ mid, IpNorm nm, float* __restrict__ out) {
  const IpImage im = imgs[blockIdx.y];
  const int idx = blockIdx.x * kIpThreads + threadIdx.x;
  if (idx >= crop_h * crop_w) return;
  const int oy = idx / crop_w, ox = idx - oy * crop_w;
  const uint8_t* col = mid + im.mid_off + static_cast<long long>(ox) * 3;
  const long long pitch = static_cast<long long>(crop_w) * 3;
  const size_t t = static_cast<size_t>(blockIdx.y) * 2 + 1;
  const int bits = axes[t].bits;
  int x[3];
  if (bits == 0) {
    const uint8_t* p = col + (im.top + oy - im.ylo) * pitch;
    x[0] = p[0]; x[1] = p[1]; x[2] = p[2];
  } else {
    const int2 sp = span[t * crop_max + oy];
    const int* w = wq + (t * crop_max + oy) * K;
    int a0 = 1 << (bits - 1), a1 = a0, a2 = a0;
    const uint8_t* p = col + (sp.x - im.ylo) * pitch;
    for (int j = 0; j < sp.y; ++j, p += pitch) {
      const int c = w[j];
      a0 += c * p[0]; a1 += c * p[1]; a2 += c * p[2];
    }
    x[0] = ip_clip8(a0, bits); x[1] = ip_clip8(a1, bits); x[2] = ip_clip8(a2, bits);
  }
  const long long plane = static_cast<long long>(crop_h) * crop_w;
  float* o = out + static_cast<long long>(im.out) * 3 * plane + idx;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float v = static_cast<float>(x[c]);
    if (nm.rescale_mode == 1) v = __fmul_rn(v, nm.rf);
    else if (nm.rescale_mode == 2) v = __double2float_rn(__dmul_rn(static_cast<double>(x[c]), nm.rd));
    if (nm.normalize) v = __fdiv_rn(__fsub_rn(v, nm.m[c]), nm.s[c]);
    o[c * plane] = v;
  }
}

}  // namespace rse
