// Training-time augmentation on the device: the config's train_pipeline transforms RandomResize (mmcv, keep_ratio),
// RandomCrop (mmseg, cat_max_ratio), RandomFlip (mmcv, horizontal) and PhotoMetricDistortion (mmseg), fused with what
// SegDataPreProcessor does after them (BGR -> RGB, (x - mean) / std, right / bottom padding of stack_batch).
//
//  * crop_select_kernel   : one block per (sample, candidate box).  Counts the classes of the nearest-resized label inside
//      the box, reading each pixel straight from the source label (the resized label is never built), and applies
//      RandomCrop's acceptance rule `len(cnt) > 1 and max(cnt) / sum(cnt) < cat_max_ratio` in float64.  The first
//      accepted candidate (or the last one, which RandomCrop uses unchecked) wins through an integer atomicMin, so the
//      parallel check gives the sequential loop's answer; the counts are integers, so any summation order gives them.
//  * train_augment_kernel : one thread per output pixel of [N, 3, Hp, Wp] (+ the int64 label): chosen box, flip within
//      the cropped extent, the resized-frame coordinate, cv2's fixed-point INTER_LINEAR taps on the uint8 CHW source,
//      the photometric chain in cv2 / numpy's own integer and float32 arithmetic, the channel swap and normalisation.
//      The label is cv2's INTER_NEAREST of the source label.  Only the outputs reach memory.
//  * view_resize_kernel   : the test-time views (TestTimeAug's Resize x RandomFlip, or the test pipeline's Resize): one
//      thread per pixel of the padded frame, the same INTER_LINEAR taps (sample_linear), written to the unflipped view
//      and to the mirrored pixel of the flipped one, then stack_pad_kernel's swap and normalisation, bit for bit.
//
// The restatement these kernels are checked against is tests/augment_oracle.py; the cv2 formulations it follows:
//   INTER_LINEAR (imgproc/resize.cpp): scale = 1 / (dst / src) in double, fx = (float)((dx + 0.5) * scale - 0.5),
//     sx = floor(fx), clamped at both edges, short coefficients rint(c * 2048), the horizontal pass into int and the
//     vertical pass in the SIMD rounding (((S0 >> 4) * b0 >> 16) + ((S1 >> 4) * b1 >> 16) + 2) >> 2.
//   INTER_NEAREST: sx = min(floor(dx * scale), src - 1).
//   BGR2HSV (uint8): the integer form with hsv_shift = 12 and the rint-rounded sdiv / hdiv tables.
//   HSV2BGR (uint8): the float SIMD form: s, v scaled by 1/255, h by 6/180, v * (1 - s * h) with the product and the
//     difference fused (the compiler contracts the vector intrinsics into FMA), the result * 255 truncated.
#include <algorithm>
#include <string>

#include "kernels.h"

namespace ledb {
namespace {

constexpr int kAugMaxSamples = 64;
constexpr int kAugMaxCandidates = 11;

struct AugSample {
  const uint8_t* img;            // [3, h, w] CHW
  const void* label;             // [h, w]
  int h, w, rh, rw;
  int eh, ew;                    // cropped extent: min(crop, resized frame)
  int count;                     // candidate boxes
  int oy[kAugMaxCandidates], ox[kAugMaxCandidates];
  int flip, contrast_mode, brightness, contrast, saturation, hue, hue_delta;
  float beta, contrast_alpha, saturation_alpha;
  double sy, sx;                 // cv2's source-per-destination scales, 1 / (rh / h) and 1 / (rw / w)
};

struct AugArgs {
  AugSample s[kAugMaxSamples];
  int N;
  double cat_max_ratio;
  int ignore_index;
  const int32_t* crop_index;     // [N], null when every sample has one candidate
  int32_t* crop_index_out;
  float mean[3], stdv[3], pad_val;
  int swap_rb, normalize, seg_pad_val, Hp, Wp;
  float* out;                    // [N, 3, Hp, Wp]
  int64_t* label_out;            // [N, Hp, Wp]
};

__device__ __forceinline__ int nearest_src(int d, double scale, int src) {
  const int s = (int)floor(__dmul_rn((double)d, scale));
  return s < src - 1 ? s : src - 1;
}

template <typename TL>
__device__ __forceinline__ int label_bin(const TL* lab, int64_t i) {
  const int64_t v = (int64_t)lab[i];
  return (v >= 0 && v < 256) ? (int)v : 256;        // values outside [0, 255] count as one class
}

constexpr int kSelThreads = 512;
constexpr int kSelWarps = kSelThreads / 32;
constexpr int kBins = 257;

template <typename TL>
__global__ void __launch_bounds__(kSelThreads) crop_select_kernel(const __grid_constant__ AugArgs a) {
  const int n = blockIdx.x / kAugMaxCandidates, k = blockIdx.x % kAugMaxCandidates;
  const AugSample& s = a.s[n];
  if (k >= s.count) return;
  if (k == s.count - 1) {                             // the last box is used without a check
    if (threadIdx.x == 0) atomicMin(a.crop_index_out + n, k);
    return;
  }
  __shared__ unsigned hist[kSelWarps][kBins];
  __shared__ long long red_sum[kSelWarps];
  __shared__ unsigned red_max[kSelWarps], red_nnz[kSelWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < kSelWarps * kBins; i += kSelThreads) (&hist[0][0])[i] = 0u;
  __syncthreads();
  const TL* lab = reinterpret_cast<const TL*>(s.label);
  const int oy = s.oy[k], ox = s.ox[k];
  for (int y = warp; y < s.eh; y += kSelWarps) {
    const int64_t row = (int64_t)nearest_src(oy + y, s.sy, s.h) * s.w;
    for (int x0 = 0; x0 < s.ew; x0 += 32) {
      const int x = x0 + lane;
      const int bin = x < s.ew ? label_bin(lab, row + nearest_src(ox + x, s.sx, s.w)) : -1;
      const unsigned same = __match_any_sync(0xffffffffu, bin);
      if (bin >= 0 && lane == __ffs(same) - 1) hist[warp][bin] += __popc(same);
    }
  }
  __syncthreads();
  // per bin: sum over the warps' histograms; then the block's sum / max / number of classes, ignore_index dropped
  long long sum = 0;
  unsigned mx = 0, nnz = 0;
  for (int b = threadIdx.x; b < kBins; b += kSelThreads) {
    if (b == a.ignore_index) continue;
    unsigned c = 0;
    for (int w = 0; w < kSelWarps; ++w) c += hist[w][b];
    sum += c; mx = c > mx ? c : mx; nnz += c > 0;
  }
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    nnz += __shfl_xor_sync(0xffffffffu, nnz, o);
  }
  if (lane == 0) { red_sum[warp] = sum; red_max[warp] = mx; red_nnz[warp] = nnz; }
  __syncthreads();
  if (threadIdx.x == 0) {
    long long tsum = 0;
    unsigned tmax = 0, tnnz = 0;
    for (int w = 0; w < kSelWarps; ++w) { tsum += red_sum[w]; tmax = max(tmax, red_max[w]); tnnz += red_nnz[w]; }
    if (tnnz > 1 && __ddiv_rn((double)tmax, (double)tsum) < a.cat_max_ratio) atomicMin(a.crop_index_out + n, k);
  }
}

// cv2's linear coefficients for destination index d: source index i0, i1 and the short weights c0, c1
__device__ __forceinline__ void linear_taps(int d, double scale, int src, int& i0, int& i1, int& c0, int& c1) {
  float f = (float)__dsub_rn(__dmul_rn((double)d + 0.5, scale), 0.5);
  int i = (int)floorf(f);
  f = __fsub_rn(f, (float)i);
  if (i < 0) { f = 0.f; i = 0; }
  if (i >= src - 1) { f = 0.f; i = src - 1; }
  i0 = i;
  i1 = i < src - 1 ? i + 1 : i;
  c0 = (int)rintf(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
  c1 = (int)rintf(__fmul_rn(f, 2048.f));
}

// cv2 INTER_LINEAR of the uint8 CHW source [3, h, w] at resized-frame pixel (ry, rx): the taps of both axes, the horizontal
// sums into int and the vertical pass in the SIMD rounding.  c[ch] is the resized uint8 value of source channel ch.
__device__ __forceinline__ void sample_linear(const uint8_t* img, int h, int w, double sy, double sx, int ry, int rx,
                                              int* c) {
  int y0, y1, b0, b1, x0, x1, a0, a1;
  linear_taps(ry, sy, h, y0, y1, b0, b1);
  linear_taps(rx, sx, w, x0, x1, a0, a1);
  const int64_t plane = (int64_t)h * w;
  const uint8_t* r0p = img + (int64_t)y0 * w;
  const uint8_t* r1p = img + (int64_t)y1 * w;
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const int S0 = __ldg(r0p + ch * plane + x0) * a0 + __ldg(r0p + ch * plane + x1) * a1;
    const int S1 = __ldg(r1p + ch * plane + x0) * a0 + __ldg(r1p + ch * plane + x1) * a1;
    const int v = ((((S0 >> 4) * b0) >> 16) + (((S1 >> 4) * b1) >> 16) + 2) >> 2;
    c[ch] = min(max(v, 0), 255);
  }
}

// numpy: clip(x.astype(float32) * alpha + beta, 0, 255).astype(uint8), two roundings, truncation
__device__ __forceinline__ int convert_u8(int x, float alpha, float beta) {
  const float v = __fadd_rn(__fmul_rn((float)x, alpha), beta);
  return (int)fminf(fmaxf(v, 0.f), 255.f);
}

__device__ __forceinline__ void bgr2hsv(int b, int g, int r, int& h, int& s, int& v, const int* sdiv, const int* hdiv) {
  v = max(max(b, g), r);
  const int vmin = min(min(b, g), r), diff = v - vmin;
  const int vr = v == r ? -1 : 0, vg = v == g ? -1 : 0;
  s = (diff * sdiv[v] + (1 << 11)) >> 12;
  h = (vr & (g - b)) + (~vr & ((vg & (b - r + 2 * diff)) + ((~vg) & (r - g + 4 * diff))));
  h = (h * hdiv[diff] + (1 << 11)) >> 12;
  h += h < 0 ? 180 : 0;
}

__device__ __forceinline__ void hsv2bgr(int h, int s, int v, int& b, int& g, int& r) {
  const float inv255 = 1.f / 255.f, hscale = 6.f / 180.f;
  const float sf = __fmul_rn((float)s, inv255), vf = __fmul_rn((float)v, inv255);
  float hh = __fmul_rn((float)h, hscale);
  const float sector_f = truncf(hh);
  hh = __fsub_rn(hh, sector_f);
  const int sector = (int)sector_f % 6;
  float tab[4];
  tab[0] = vf;
  tab[1] = __fmul_rn(vf, __fsub_rn(1.f, sf));
  tab[2] = __fmul_rn(vf, __fmaf_rn(-sf, hh, 1.f));
  tab[3] = __fmul_rn(vf, __fmaf_rn(-sf, __fsub_rn(1.f, hh), 1.f));
  int ib, ig, ir;
  switch (sector) {
    case 0: ib = 1; ig = 3; ir = 0; break;
    case 1: ib = 1; ig = 0; ir = 2; break;
    case 2: ib = 3; ig = 0; ir = 1; break;
    case 3: ib = 0; ig = 2; ir = 1; break;
    case 4: ib = 0; ig = 1; ir = 3; break;
    default: ib = 2; ig = 1; ir = 0; break;
  }
  b = (int)__fmul_rn(tab[ib], 255.f);
  g = (int)__fmul_rn(tab[ig], 255.f);
  r = (int)__fmul_rn(tab[ir], 255.f);
}

template <typename TL>
__global__ void __launch_bounds__(256) train_augment_kernel(const __grid_constant__ AugArgs a) {
  __shared__ int sdiv[256], hdiv[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    // saturate_cast<int>((255 << 12) / (1. * i)) and ((180 << 12) / (6. * i)): round half to even of a rational
    int q0 = 0, q1 = 0;
    if (i > 0) {
      const int n0 = 255 << 12, d0 = i, n1 = 180 << 12, d1 = 6 * i;
      q0 = n0 / d0; int r0 = 2 * (n0 % d0);
      q0 += (r0 > d0 || (r0 == d0 && (q0 & 1))) ? 1 : 0;
      q1 = n1 / d1; int r1 = 2 * (n1 % d1);
      q1 += (r1 > d1 || (r1 == d1 && (q1 & 1))) ? 1 : 0;
    }
    sdiv[i] = q0; hdiv[i] = q1;
  }
  __syncthreads();
  const int64_t HWp = (int64_t)a.Hp * a.Wp;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.N * HWp) return;
  const int n = (int)(idx / HWp);
  const int64_t pix = idx % HWp;
  const int y = (int)(pix / a.Wp), x = (int)(pix % a.Wp);
  const AugSample& s = a.s[n];
  float* out = a.out + (int64_t)n * 3 * HWp + pix;
  int64_t* lout = a.label_out + idx;
  if (y >= s.eh || x >= s.ew) {
    out[0] = a.pad_val; out[HWp] = a.pad_val; out[2 * HWp] = a.pad_val;
    *lout = a.seg_pad_val;
    return;
  }
  int k = 0;
  if (s.count > 1) k = min(max(__ldg(a.crop_index + n), 0), s.count - 1);
  const int ry = s.oy[k] + y;
  const int rx = s.ox[k] + (s.flip ? s.ew - 1 - x : x);

  *lout = (int64_t)reinterpret_cast<const TL*>(s.label)[(int64_t)nearest_src(ry, s.sy, s.h) * s.w +
                                                        nearest_src(rx, s.sx, s.w)];

  int c[3];
  sample_linear(s.img, s.h, s.w, s.sy, s.sx, ry, rx, c);
  // PhotoMetricDistortion: brightness; contrast if mode 1; saturation; hue; contrast if mode 0
  if (s.brightness) {
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) c[ch] = convert_u8(c[ch], 1.f, s.beta);
  }
  if (s.contrast && s.contrast_mode == 1) {
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) c[ch] = convert_u8(c[ch], s.contrast_alpha, 0.f);
  }
  if (s.saturation) {
    int h, sat, v;
    bgr2hsv(c[0], c[1], c[2], h, sat, v, sdiv, hdiv);
    hsv2bgr(h, convert_u8(sat, s.saturation_alpha, 0.f), v, c[0], c[1], c[2]);
  }
  if (s.hue) {
    int h, sat, v;
    bgr2hsv(c[0], c[1], c[2], h, sat, v, sdiv, hdiv);
    h = ((h + s.hue_delta) % 180 + 180) % 180;
    hsv2bgr(h, sat, v, c[0], c[1], c[2]);
  }
  if (s.contrast && s.contrast_mode == 0) {
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) c[ch] = convert_u8(c[ch], s.contrast_alpha, 0.f);
  }
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const float v = (float)c[a.swap_rb ? 2 - ch : ch];
    out[ch * HWp] = a.normalize ? __fdiv_rn(v - a.mean[ch], a.stdv[ch]) : v;
  }
}

// ---- test-time views: mmcv Resize (keep_ratio, cv2 INTER_LINEAR) + RandomFlip (horizontal) + SegDataPreProcessor ----
constexpr int kViewMax = 64;

struct View {
  const uint8_t* src;            // [3, h, w] CHW
  float* out;                    // [3, Hp, Wp] or null
  float* out_flip;               // [3, Hp, Wp] or null
  int h, w, rh, rw;
  double sy, sx;                 // cv2's source-per-destination scales, as in fill_samples
};

struct ViewArgs {
  View v[kViewMax];
  int n, Hp, Wp, swap_rb, normalize;
  float mean[3], stdv[3], pad_val;
};

// One thread per pixel of the padded frame of one view.  Inside the resized frame the pixel is sampled once and written
// to out[y][x] and to out_flip[y][rw - 1 - x]; outside it both outputs get pad_val at [y][x].
__global__ void __launch_bounds__(256) view_resize_kernel(const __grid_constant__ ViewArgs a) {
  const int64_t HWp = (int64_t)a.Hp * a.Wp;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.n * HWp) return;
  const int n = (int)(idx / HWp);
  const int64_t pix = idx % HWp;
  const int y = (int)(pix / a.Wp), x = (int)(pix % a.Wp);
  const View& v = a.v[n];
  if (y >= v.rh || x >= v.rw) {
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      if (v.out) v.out[ch * HWp + pix] = a.pad_val;
      if (v.out_flip) v.out_flip[ch * HWp + pix] = a.pad_val;
    }
    return;
  }
  int c[3];
  sample_linear(v.src, v.h, v.w, v.sy, v.sx, y, x, c);
  const int64_t fpix = pix + (v.rw - 1 - 2 * x);
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const float f = (float)c[a.swap_rb ? 2 - ch : ch];
    const float o = a.normalize ? __fdiv_rn(f - a.mean[ch], a.stdv[ch]) : f;   // stack_pad_kernel's expression
    if (v.out) v.out[ch * HWp + pix] = o;
    if (v.out_flip) v.out_flip[ch * HWp + fpix] = o;
  }
}

int fill_samples(const ledb200_aug_sample* smp, int32_t N, int32_t crop_h, int32_t crop_w, int32_t label_dtype,
                 AugArgs& a, const char* what) {
  const std::string w(what);
  if (!smp) return fail(LEDB200_EINVAL, w + ": null sample descriptors");
  if (N < 1 || N > kAugMaxSamples) return fail(LEDB200_EINVAL, w + ": between 1 and 64 samples per call");
  if (crop_h < 1 || crop_w < 1) return fail(LEDB200_EINVAL, w + ": crop size must be at least 1 x 1");
  if (label_dtype != LEDB200_U8 && label_dtype != LEDB200_I64)
    return fail(LEDB200_EINVAL, w + ": label dtype must be U8 or I64");
  a.N = N;
  for (int i = 0; i < N; ++i) {
    const ledb200_aug_sample& d = smp[i];
    AugSample& s = a.s[i];
    if (!d.img || !d.label) return fail(LEDB200_EINVAL, w + ": null image or label");
    if (d.h < 1 || d.w < 1 || d.rh < 1 || d.rw < 1) return fail(LEDB200_EINVAL, w + ": empty image or resized frame");
    if (d.num_candidates < 1 || d.num_candidates > kAugMaxCandidates)
      return fail(LEDB200_EINVAL, w + ": between 1 and 11 candidate boxes per sample");
    if (d.flip < 0 || d.flip > 1) return fail(LEDB200_EINVAL, w + ": flip must be 0 or 1 (horizontal)");
    s.img = d.img; s.label = d.label; s.h = d.h; s.w = d.w; s.rh = d.rh; s.rw = d.rw;
    s.eh = std::min(crop_h, d.rh); s.ew = std::min(crop_w, d.rw);
    s.count = d.num_candidates;
    for (int k = 0; k < kAugMaxCandidates; ++k) {
      s.oy[k] = s.ox[k] = 0;
      if (k >= d.num_candidates) continue;
      const int oy = d.offsets[k][0], ox = d.offsets[k][1];
      if (oy < 0 || ox < 0 || oy > std::max(d.rh - crop_h, 0) || ox > std::max(d.rw - crop_w, 0))
        return fail(LEDB200_EINVAL, w + ": candidate box outside the resized frame");
      s.oy[k] = oy; s.ox[k] = ox;
    }
    s.flip = d.flip; s.contrast_mode = d.contrast_mode ? 1 : 0;
    s.brightness = d.brightness ? 1 : 0; s.contrast = d.contrast ? 1 : 0;
    s.saturation = d.saturation ? 1 : 0; s.hue = d.hue ? 1 : 0; s.hue_delta = d.hue_delta;
    s.beta = d.beta; s.contrast_alpha = d.contrast_alpha; s.saturation_alpha = d.saturation_alpha;
    s.sy = 1.0 / ((double)d.rh / d.h);
    s.sx = 1.0 / ((double)d.rw / d.w);
  }
  return LEDB200_OK;
}

}  // namespace
}  // namespace ledb

using namespace ledb;

extern "C" {

int ledb200_crop_select(const ledb200_aug_sample* samples, int32_t N, int32_t crop_h, int32_t crop_w, int32_t label_dtype,
                        double cat_max_ratio, int32_t ignore_index, int32_t* crop_index, void* stream) {
  AugArgs a;
  if (!crop_index) return fail(LEDB200_EINVAL, "crop_select: null crop_index");
  if (ignore_index < 0 || ignore_index > 255) return fail(LEDB200_EINVAL, "crop_select: ignore_index must lie in [0, 255]");
  int rc = fill_samples(samples, N, crop_h, crop_w, label_dtype, a, "crop_select");
  if (rc != LEDB200_OK) return rc;
  a.cat_max_ratio = cat_max_ratio; a.ignore_index = ignore_index; a.crop_index_out = crop_index;
  cudaStream_t st = (cudaStream_t)stream;
  LEDB_CUDA_OK(cudaMemsetAsync(crop_index, 0x7f, sizeof(int32_t) * N, st));   // above any index: atomicMin starts here
  const unsigned grid = (unsigned)(N * kAugMaxCandidates);
  if (label_dtype == LEDB200_I64) crop_select_kernel<int64_t><<<grid, kSelThreads, 0, st>>>(a);
  else crop_select_kernel<uint8_t><<<grid, kSelThreads, 0, st>>>(a);
  LEDB_LAUNCH_OK("crop_select_kernel");
  return LEDB200_OK;
}

int ledb200_train_augment(const ledb200_aug_sample* samples, int32_t N, int32_t crop_h, int32_t crop_w,
                          int32_t label_dtype, const int32_t* crop_index, int32_t swap_rb, const float* mean3,
                          const float* std3, float pad_val, float* out, int32_t Hp, int32_t Wp, int64_t* label_out,
                          int32_t seg_pad_val, void* stream) {
  AugArgs a;
  if (!out || !label_out) return fail(LEDB200_EINVAL, "train_augment: null buffer");
  if ((mean3 == nullptr) != (std3 == nullptr)) return fail(LEDB200_EINVAL, "train_augment: mean and std come together");
  int rc = fill_samples(samples, N, crop_h, crop_w, label_dtype, a, "train_augment");
  if (rc != LEDB200_OK) return rc;
  for (int i = 0; i < N; ++i) {
    if (a.s[i].count > 1 && !crop_index)
      return fail(LEDB200_EINVAL, "train_augment: crop_index is needed when a sample has several candidate boxes");
    if (a.s[i].eh > Hp || a.s[i].ew > Wp)
      return fail(LEDB200_EINVAL, "train_augment: the padded size is smaller than a cropped sample");
  }
  a.crop_index = crop_index;
  a.normalize = mean3 ? 1 : 0;
  for (int c = 0; c < 3; ++c) { a.mean[c] = mean3 ? mean3[c] : 0.f; a.stdv[c] = std3 ? std3[c] : 1.f; }
  a.pad_val = pad_val; a.swap_rb = swap_rb ? 1 : 0; a.seg_pad_val = seg_pad_val; a.Hp = Hp; a.Wp = Wp;
  a.out = out; a.label_out = label_out;
  const unsigned grid = (unsigned)ceil_div64((int64_t)N * Hp * Wp, 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (label_dtype == LEDB200_I64) train_augment_kernel<int64_t><<<grid, 256, 0, st>>>(a);
  else train_augment_kernel<uint8_t><<<grid, 256, 0, st>>>(a);
  LEDB_LAUNCH_OK("train_augment_kernel");
  return LEDB200_OK;
}

int ledb200_view_resize(const ledb200_view_desc* views, int32_t n, int32_t Hp, int32_t Wp, int32_t swap_rb,
                        const float* mean3, const float* std3, float pad_val, void* stream) {
  if (!views) return fail(LEDB200_EINVAL, "view_resize: null view descriptors");
  if (n < 1 || n > kViewMax) return fail(LEDB200_EINVAL, "view_resize: between 1 and 64 views per call");
  if ((mean3 == nullptr) != (std3 == nullptr)) return fail(LEDB200_EINVAL, "view_resize: mean and std come together");
  ViewArgs a;
  for (int i = 0; i < n; ++i) {
    const ledb200_view_desc& d = views[i];
    if (!d.src) return fail(LEDB200_EINVAL, "view_resize: null source image");
    if (!d.out && !d.out_flip) return fail(LEDB200_EINVAL, "view_resize: a view needs out or out_flip");
    if (d.h < 1 || d.w < 1 || d.rh < 1 || d.rw < 1) return fail(LEDB200_EINVAL, "view_resize: empty image or resized frame");
    if (d.rh > Hp || d.rw > Wp) return fail(LEDB200_EINVAL, "view_resize: the padded size is smaller than a resized view");
    View& v = a.v[i];
    v.src = d.src; v.out = d.out; v.out_flip = d.out_flip;
    v.h = d.h; v.w = d.w; v.rh = d.rh; v.rw = d.rw;
    v.sy = 1.0 / ((double)d.rh / d.h);
    v.sx = 1.0 / ((double)d.rw / d.w);
  }
  a.n = n; a.Hp = Hp; a.Wp = Wp; a.swap_rb = swap_rb ? 1 : 0; a.normalize = mean3 ? 1 : 0; a.pad_val = pad_val;
  for (int c = 0; c < 3; ++c) { a.mean[c] = mean3 ? mean3[c] : 0.f; a.stdv[c] = std3 ? std3[c] : 1.f; }
  const unsigned grid = (unsigned)ceil_div64((int64_t)n * Hp * Wp, 256);
  view_resize_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
  LEDB_LAUNCH_OK("view_resize_kernel");
  return LEDB200_OK;
}

}  // extern "C"
