// Result post-processing on the device (SURVEY section 8a rows H3 and E2).
//
//  * postprocess_kernel : BaseSegmentor.postprocess_result (mmseg/models/segmentors/base.py:153-198) for one
//      image: remove the padding border, undo a horizontal / vertical test-time flip, bilinear-resize the
//      logits to `ori_shape` (mmseg/models/utils/wrappers.py:8-27 -> F.interpolate, align_corners as the
//      decode head's) and take argmax(dim=0) (C > 1) or sigmoid > threshold (C == 1) - in ONE pass: the
//      resized [K, oh, ow] logits are written only when the caller asks for them.  The real Apple-Branch
//      pipeline needs the general ratio (512x910 -> 720x1280, scale 1.40625); all BASELINE configs are the
//      identity case, which the fused tail kernel already covers.
//  * slide_accumulate / slide_finalize : EncoderDecoder.slide_inference (encoder_decoder.py:241-292):
//      `preds += F.pad(crop_logits, ...)`, `count_mat[..., y1:y2, x1:x2] += 1` without materialising the padded
//      full-size tensor per crop, then `preds / count_mat` (+ optional argmax) in one pass.
//  * slide_merge : the same for ALL crops at once (they ran as one batch of the engine): per output pixel the crops that
//      cover it are summed in the reference's grid order (fp32, starting from 0: bit-identical to the sequential
//      `preds +=`), divided by their number, and optionally arg-maxed - no full-size read-modify-write per crop.
//  * tta_merge : SegTTAModel.merge_preds (mmseg/models/segmentors/seg_tta.py) for every view of a batch at once: per output
//      pixel each view is sampled through postprocess_kernel's own geometry (un-pad, un-flip, resize), soft-maxed (or
//      sigmoid-ed) over K and summed in view order in registers; then / V and argmax (or > threshold).  Only the labels
//      (and, on request, the merged probabilities) reach memory.
//  * stack_pad : SegDataPreProcessor.forward + stack_batch for one sample (mmseg/models/data_preprocessor.py:112-149,
//      mmseg/utils/misc.py:30-128): BGR<->RGB swap, float, (x - mean) / std, right / bottom padding with `pad_val`
//      (applied AFTER the normalisation, as the reference does), label map padded with `seg_pad_val`.
// All tensors are the reference's NCHW fp32; one thread per output pixel, consecutive threads on consecutive x.
#include <type_traits>
#include <vector>

#include "kernels.h"

namespace ledb {
namespace {

// The geometry of one post-processed view: stored [K, H, W] logits, the padding to remove, the flip to undo and the
// ATen resize scales from the cropped extent [ch, cw] to the output size.  Shared by postprocess_kernel and
// tta_merge_kernel, so a merged view samples exactly the values ledb200_postprocess writes for it.
struct ViewGeom {
  int H, W;
  int pl, pt;            // left / top padding (right / bottom only shorten the cropped extent)
  int ch, cw;            // cropped extent
  int flip;              // 0 none, 1 horizontal, 2 vertical
  float sy, sx;          // ATen scales
};

// false when the padding is negative or removes the whole image
bool make_geom(int H, int W, const int32_t* pad_lrtb, int flip, int oh, int ow, int align_corners, ViewGeom& g) {
  const int pl = pad_lrtb ? pad_lrtb[0] : 0, pr = pad_lrtb ? pad_lrtb[1] : 0;
  const int pt = pad_lrtb ? pad_lrtb[2] : 0, pb = pad_lrtb ? pad_lrtb[3] : 0;
  g.H = H; g.W = W; g.pl = pl; g.pt = pt; g.ch = H - pt - pb; g.cw = W - pl - pr; g.flip = flip;
  if (pl < 0 || pr < 0 || pt < 0 || pb < 0 || g.ch < 1 || g.cw < 1) return false;
  if (align_corners) {
    g.sy = oh > 1 ? (float)(g.ch - 1) / (float)(oh - 1) : 0.f;
    g.sx = ow > 1 ? (float)(g.cw - 1) / (float)(ow - 1) : 0.f;
  } else {
    g.sy = (float)g.ch / (float)oh; g.sx = (float)g.cw / (float)ow;
  }
  return true;
}

struct PostArgs {
  const float* logits;   // [K, H, W] of one image
  int K;
  ViewGeom g;
  int oh, ow, align_corners;
  float threshold;       // C == 1
  void* pred; int pred_dtype;
  float* out_logits;     // optional [K, oh, ow]
};

__device__ __forceinline__ void src_index(int dst, float scale, int in_size, int align, int& i0, int& i1, float& l1) {
  if (align) {
    const float src = scale * (float)dst;                         // area_pixel_compute_source_index, align_corners
    i0 = min((int)src, in_size - 1);
    i1 = i0 + ((i0 < in_size - 1) ? 1 : 0);
    l1 = src - (float)i0;
  } else {
    float l0;
    bilinear_coord(dst, scale, in_size, i0, i1, l0, l1);
  }
}

// the four source taps of output pixel (oy, ox) in the stored logits, and the lerp weights
struct Taps {
  int64_t o00, o01, o10, o11;
  float ly, lx;
};

__device__ __forceinline__ Taps view_taps(const ViewGeom& g, int oy, int ox, int align_corners) {
  int y0, y1, x0, x1;
  Taps t;
  src_index(oy, g.sy, g.ch, align_corners, y0, y1, t.ly);
  src_index(ox, g.sx, g.cw, align_corners, x0, x1, t.lx);
  // cropped (and flipped) coordinates -> coordinates of the stored logits
  if (g.flip == 1) { x0 = g.cw - 1 - x0; x1 = g.cw - 1 - x1; }
  if (g.flip == 2) { y0 = g.ch - 1 - y0; y1 = g.ch - 1 - y1; }
  t.o00 = (int64_t)(y0 + g.pt) * g.W + x0 + g.pl; t.o01 = (int64_t)(y0 + g.pt) * g.W + x1 + g.pl;
  t.o10 = (int64_t)(y1 + g.pt) * g.W + x0 + g.pl; t.o11 = (int64_t)(y1 + g.pt) * g.W + x1 + g.pl;
  return t;
}

// postprocess_result's value of one class plane `p` at the taps (sigmoid applied when K == 1, base.py:190)
__device__ __forceinline__ float view_value(const float* p, const Taps& t, int K) {
  const float hy = 1.f - t.ly, hx = 1.f - t.lx;
  // ATen upsample_bilinear2d: h0lambda * (w0lambda * v00 + w1lambda * v01) + h1lambda * (w0lambda * v10 + w1lambda * v11)
  float v = hy * (hx * __ldg(p + t.o00) + t.lx * __ldg(p + t.o01)) + t.ly * (hx * __ldg(p + t.o10) + t.lx * __ldg(p + t.o11));
  if (K == 1) v = 1.f / (1.f + __expf(-v));
  return v;
}

template <typename TP>
__global__ void __launch_bounds__(256) postprocess_kernel(PostArgs a) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.oh * a.ow) return;
  const int ox = (int)(idx % a.ow), oy = (int)(idx / a.ow);
  const Taps t = view_taps(a.g, oy, ox, a.align_corners);
  float best = -INFINITY;
  int bi = 0;
  float v = 0.f;
  for (int k = 0; k < a.K; ++k) {
    v = view_value(a.logits + (int64_t)k * a.g.H * a.g.W, t, a.K);
    if (a.out_logits) a.out_logits[(int64_t)k * a.oh * a.ow + idx] = v;
    if (v > best) { best = v; bi = k; }                           // strict >: torch.argmax's first-max rule
  }
  TP* pred = reinterpret_cast<TP*>(a.pred);
  if (pred) pred[idx] = (TP)(a.K == 1 ? (v > a.threshold ? 1 : 0) : bi);
}

// ---- tta_merge: SegTTAModel.merge_preds over every view of a batch -----------------------------------------------
constexpr int kMaxViews = 32;
struct TtaView {
  const float* logits;   // image n at logits + n * image_stride
  int64_t image_stride;
  ViewGeom g;
};
struct TtaArgs {
  TtaView v[kMaxViews];
  int V, N, K, oh, ow, align_corners;
  float threshold;       // sigmoid mode
  void* pred;            // softmax mode: labels [N, oh, ow]; sigmoid mode: float mask [N, K, oh, ow]
  float* probs;          // optional merged [N, K, oh, ow]
};

__device__ __forceinline__ float sigmoid_ref(float v) { return 1.f / (1.f + expf(-v)); }

// Both paths: TP == float selects the sigmoid mode (out_channels == 1), whose prediction is the float mask
// (logits > threshold).to(logits) of [N, K, oh, ow]; otherwise TP is the label type of argmax(dim=0).

// Register path, K <= KT: one thread per output pixel, the per-class accumulator and the view's values in registers.
// EXACT: K == KT (no per-class guards).
template <int KT, bool EXACT, typename TP>
__global__ void __launch_bounds__(256) tta_merge_kernel(const __grid_constant__ TtaArgs a) {
  constexpr bool kSigmoid = std::is_same<TP, float>::value;
  const int K = EXACT ? KT : a.K;
  const int64_t OHW = (int64_t)a.oh * a.ow;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.N * OHW) return;
  const int n = (int)(idx / OHW);
  const int64_t pix = idx % OHW;
  const int oy = (int)(pix / a.ow), ox = (int)(pix % a.ow);
  float acc[KT];
#pragma unroll
  for (int k = 0; k < KT; ++k) acc[k] = 0.f;                     // logits = zeros_like(views[0])
  for (int i = 0; i < a.V; ++i) {
    const TtaView& vw = a.v[i];
    const Taps t = view_taps(vw.g, oy, ox, a.align_corners);
    const float* base = vw.logits + (int64_t)n * vw.image_stride;
    const int64_t plane = (int64_t)vw.g.H * vw.g.W;
    float v[KT];
    float m = -INFINITY;
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (EXACT || k < K) { v[k] = view_value(base + k * plane, t, K); m = fmaxf(m, v[k]); }
    if constexpr (kSigmoid) {
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (EXACT || k < K) acc[k] += sigmoid_ref(v[k]);          // logits += seg_logit.sigmoid()
    } else {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (EXACT || k < K) { v[k] = expf(v[k] - m); s += v[k]; }
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (EXACT || k < K) acc[k] += v[k] / s;                   // logits += seg_logit.softmax(dim=0)
    }
  }
  float best = -INFINITY;
  int bi = 0;
#pragma unroll
  for (int k = 0; k < KT; ++k) {
    if (EXACT || k < K) {
      const float mk = acc[k] / (float)a.V;                       // logits /= len(views)
      const int64_t o = ((int64_t)n * K + k) * OHW + pix;
      if (a.probs) a.probs[o] = mk;
      if constexpr (kSigmoid) {
        if (a.pred) reinterpret_cast<float*>(a.pred)[o] = mk > a.threshold ? 1.f : 0.f;
      }
      if (mk > best) { best = mk; bi = k; }                       // strict >: torch.argmax's first-max rule
    }
  }
  if constexpr (!kSigmoid) {
    if (a.pred) reinterpret_cast<TP*>(a.pred)[idx] = (TP)bi;
  }
}

// General path, 32 < K <= 255: the accumulator of thread t lives in shared memory at acc[k * 32 + t] (one warp per
// block, K * 128 bytes); each view's values are recomputed per pass from the same taps instead of held.
template <typename TP>
__global__ void __launch_bounds__(32) tta_merge_general_kernel(const __grid_constant__ TtaArgs a) {
  extern __shared__ float tta_acc[];
  float* acc = tta_acc + threadIdx.x;
  const int K = a.K;
  const int64_t OHW = (int64_t)a.oh * a.ow;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.N * OHW) return;
  const int n = (int)(idx / OHW);
  const int64_t pix = idx % OHW;
  const int oy = (int)(pix / a.ow), ox = (int)(pix % a.ow);
  for (int k = 0; k < K; ++k) acc[k * 32] = 0.f;
  for (int i = 0; i < a.V; ++i) {
    const TtaView& vw = a.v[i];
    const Taps t = view_taps(vw.g, oy, ox, a.align_corners);
    const float* base = vw.logits + (int64_t)n * vw.image_stride;
    const int64_t plane = (int64_t)vw.g.H * vw.g.W;
    if constexpr (std::is_same<TP, float>::value) {
      for (int k = 0; k < K; ++k) acc[k * 32] += sigmoid_ref(view_value(base + k * plane, t, K));
    } else {
      float m = -INFINITY, s = 0.f;
      for (int k = 0; k < K; ++k) m = fmaxf(m, view_value(base + k * plane, t, K));
      for (int k = 0; k < K; ++k) s += expf(view_value(base + k * plane, t, K) - m);
      for (int k = 0; k < K; ++k) acc[k * 32] += expf(view_value(base + k * plane, t, K) - m) / s;
    }
  }
  const float V = (float)a.V;
  float best = -INFINITY;
  int bi = 0;
  for (int k = 0; k < K; ++k) {
    const float mk = acc[k * 32] / V;
    const int64_t o = ((int64_t)n * K + k) * OHW + pix;
    if (a.probs) a.probs[o] = mk;
    if constexpr (std::is_same<TP, float>::value) {
      if (a.pred) reinterpret_cast<float*>(a.pred)[o] = mk > a.threshold ? 1.f : 0.f;
    }
    if (mk > best) { best = mk; bi = k; }
  }
  if constexpr (!std::is_same<TP, float>::value) {
    if (a.pred) reinterpret_cast<TP*>(a.pred)[idx] = (TP)bi;
  }
}

template <typename TP>
int launch_tta_merge(const TtaArgs& a, cudaStream_t st) {
  const unsigned grid = (unsigned)ceil_div64((int64_t)a.N * a.oh * a.ow, 256);
  switch (a.K) {
    case 2: tta_merge_kernel<2, true, TP><<<grid, 256, 0, st>>>(a); break;       // Apple-Branch
    case 19: tta_merge_kernel<19, true, TP><<<grid, 256, 0, st>>>(a); break;     // Cityscapes
    default:
      if (a.K <= 8) tta_merge_kernel<8, false, TP><<<grid, 256, 0, st>>>(a);
      else if (a.K <= 16) tta_merge_kernel<16, false, TP><<<grid, 256, 0, st>>>(a);
      else if (a.K <= 32) tta_merge_kernel<32, false, TP><<<grid, 256, 0, st>>>(a);
      else
        tta_merge_general_kernel<TP><<<(unsigned)ceil_div64((int64_t)a.N * a.oh * a.ow, 32), 32,
                                       (size_t)a.K * 32 * sizeof(float), st>>>(a);
  }
  LEDB_LAUNCH_OK("tta_merge_kernel");
  return LEDB200_OK;
}

__global__ void __launch_bounds__(256) slide_accumulate_kernel(float* preds, float* count, const float* crop, int N, int K,
                                                               int H, int W, int hc, int wc, int y1, int x1) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)N * (K + 1) * hc * wc;            // plane K of every image = the count matrix
  if (idx >= total) return;
  const int x = (int)(idx % wc);
  int64_t t = idx / wc;
  const int y = (int)(t % hc); t /= hc;
  const int k = (int)(t % (K + 1));
  const int n = (int)(t / (K + 1));
  const int64_t pix = (int64_t)(y1 + y) * W + x1 + x;
  if (k < K) preds[((int64_t)n * K + k) * H * W + pix] += crop[(((int64_t)n * K + k) * hc + y) * wc + x];
  else count[(int64_t)n * H * W + pix] += 1.f;
}

template <typename TP>
__global__ void __launch_bounds__(256) slide_finalize_kernel(float* preds, const float* count, int N, int K, int64_t HW,
                                                             TP* pred) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * HW) return;
  const int n = (int)(idx / HW);
  const int64_t pix = idx % HW;
  const float c = count[idx];
  float best = -INFINITY;
  int bi = 0;
  for (int k = 0; k < K; ++k) {
    float* p = preds + ((int64_t)n * K + k) * HW + pix;
    const float v = *p / c;                                        // preds / count_mat (encoder_decoder.py:290)
    *p = v;
    if (v > best) { best = v; bi = k; }
  }
  if (pred) pred[idx] = (TP)bi;
}

constexpr int kMaxCrops = 64;
struct MergeArgs {
  const float* crops;    // [G * N, K, hc, wc], crop g of image n at index g * N + n
  int G, N, K, H, W, hc, wc;
  int y1[kMaxCrops], x1[kMaxCrops];
  float* out;            // optional [N, K, H, W]
  void* pred;            // optional [N, H, W]
};

template <typename TP>
__global__ void __launch_bounds__(256) slide_merge_kernel(const __grid_constant__ MergeArgs a) {
  const int64_t HW = (int64_t)a.H * a.W;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.N * HW) return;
  const int n = (int)(idx / HW);
  const int64_t pix = idx % HW;
  const int y = (int)(pix / a.W), x = (int)(pix % a.W);
  const int64_t plane = (int64_t)a.hc * a.wc;
  float cnt = 0.f;
  for (int g = 0; g < a.G; ++g)
    cnt += (y >= a.y1[g] && y < a.y1[g] + a.hc && x >= a.x1[g] && x < a.x1[g] + a.wc) ? 1.f : 0.f;
  float best = -INFINITY;
  int bi = 0;
  for (int k = 0; k < a.K; ++k) {
    float s = 0.f;                                               // preds = zeros; preds += pad(crop) in grid order
    for (int g = 0; g < a.G; ++g) {
      const int yy = y - a.y1[g], xx = x - a.x1[g];
      if (yy >= 0 && yy < a.hc && xx >= 0 && xx < a.wc)
        s += __ldg(a.crops + (((int64_t)g * a.N + n) * a.K + k) * plane + (int64_t)yy * a.wc + xx);
    }
    const float v = s / cnt;
    if (a.out) a.out[((int64_t)n * a.K + k) * HW + pix] = v;
    if (v > best) { best = v; bi = k; }
  }
  if (a.pred) reinterpret_cast<TP*>(a.pred)[idx] = (TP)bi;
}

struct StackPadArgs {
  const void* img; int h, w, swap_rb, normalize;
  float mean[3], stdv[3], pad_val;
  float* out; int Hp, Wp;
  const void* label; int64_t* label_out; int seg_pad_val;
};

template <typename TI, typename TL>
__global__ void __launch_bounds__(256) stack_pad_kernel(const __grid_constant__ StackPadArgs a) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t HWp = (int64_t)a.Hp * a.Wp;
  if (idx >= HWp) return;
  const int y = (int)(idx / a.Wp), x = (int)(idx % a.Wp);
  const bool inside = y < a.h && x < a.w;
  const int64_t src = (int64_t)y * a.w + x, hw = (int64_t)a.h * a.w;
  const TI* img = reinterpret_cast<const TI*>(a.img);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float v = a.pad_val;
    if (inside) {
      v = (float)img[(a.swap_rb ? 2 - c : c) * hw + src];
      if (a.normalize) v = __fdiv_rn(v - a.mean[c], a.stdv[c]);   // (_input - self.mean) / self.std, channel c AFTER the swap
    }
    a.out[c * HWp + idx] = v;
  }
  if (a.label_out)
    a.label_out[idx] = inside ? (int64_t)reinterpret_cast<const TL*>(a.label)[src] : (int64_t)a.seg_pad_val;
}

}  // namespace
}  // namespace ledb

using namespace ledb;

extern "C" {

int ledb200_postprocess(const float* logits, int32_t K, int32_t H, int32_t W, const int32_t* padding_lrtb,
                        int32_t flip, int32_t out_h, int32_t out_w, int32_t align_corners, float threshold,
                        void* pred, int32_t pred_dtype, float* out_logits, void* stream) {
  if (!logits || (!pred && !out_logits)) return fail(LEDB200_EINVAL, "postprocess: null buffer");
  if (K < 1 || H < 1 || W < 1 || out_h < 1 || out_w < 1) return fail(LEDB200_EINVAL, "postprocess: empty tensor");
  if (flip < 0 || flip > 2) return fail(LEDB200_EINVAL, "postprocess: flip must be 0 (none), 1 (horizontal) or 2 (vertical)");
  if (pred && pred_dtype != LEDB200_U8 && pred_dtype != LEDB200_I64 && pred_dtype != LEDB200_F32)
    return fail(LEDB200_EINVAL, "postprocess: pred dtype must be U8, I64 or F32");
  PostArgs a;
  a.logits = logits; a.K = K;
  a.oh = out_h; a.ow = out_w; a.align_corners = align_corners ? 1 : 0;
  if (!make_geom(H, W, padding_lrtb, flip, out_h, out_w, a.align_corners, a.g))
    return fail(LEDB200_EINVAL, "postprocess: padding removes the whole image");
  a.threshold = threshold; a.pred = pred; a.pred_dtype = pred_dtype; a.out_logits = out_logits;
  const unsigned grid = (unsigned)ceil_div64((int64_t)out_h * out_w, 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (pred_dtype == LEDB200_I64) postprocess_kernel<int64_t><<<grid, 256, 0, st>>>(a);
  else if (pred_dtype == LEDB200_F32) postprocess_kernel<float><<<grid, 256, 0, st>>>(a);
  else postprocess_kernel<uint8_t><<<grid, 256, 0, st>>>(a);
  LEDB_LAUNCH_OK("postprocess_kernel");
  return LEDB200_OK;
}

int ledb200_slide_accumulate(float* preds, float* count, const float* crop_logits, int32_t N, int32_t K, int32_t H,
                             int32_t W, int32_t hc, int32_t wc, int32_t y1, int32_t x1, void* stream) {
  if (!preds || !count || !crop_logits) return fail(LEDB200_EINVAL, "slide_accumulate: null buffer");
  if (N < 1 || K < 1 || hc < 1 || wc < 1 || y1 < 0 || x1 < 0 || y1 + hc > H || x1 + wc > W)
    return fail(LEDB200_EINVAL, "slide_accumulate: crop window outside the image");
  const int64_t total = (int64_t)N * (K + 1) * hc * wc;
  slide_accumulate_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, (cudaStream_t)stream>>>(preds, count, crop_logits, N, K,
                                                                                          H, W, hc, wc, y1, x1);
  LEDB_LAUNCH_OK("slide_accumulate_kernel");
  return LEDB200_OK;
}

int ledb200_slide_finalize(float* preds, const float* count, int32_t N, int32_t K, int32_t H, int32_t W, void* pred,
                           int32_t pred_dtype, void* stream) {
  if (!preds || !count) return fail(LEDB200_EINVAL, "slide_finalize: null buffer");
  if (pred && pred_dtype != LEDB200_U8 && pred_dtype != LEDB200_I64)
    return fail(LEDB200_EINVAL, "slide_finalize: pred dtype must be U8 or I64");
  const int64_t HW = (int64_t)H * W;
  const unsigned grid = (unsigned)ceil_div64((int64_t)N * HW, 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (pred_dtype == LEDB200_I64) slide_finalize_kernel<int64_t><<<grid, 256, 0, st>>>(preds, count, N, K, HW, (int64_t*)pred);
  else slide_finalize_kernel<uint8_t><<<grid, 256, 0, st>>>(preds, count, N, K, HW, (uint8_t*)pred);
  LEDB_LAUNCH_OK("slide_finalize_kernel");
  return LEDB200_OK;
}

int ledb200_slide_merge(const float* crop_logits, int32_t G, const int32_t* y1, const int32_t* x1, int32_t N, int32_t K,
                        int32_t H, int32_t W, int32_t hc, int32_t wc, float* out_logits, void* pred, int32_t pred_dtype,
                        void* stream) {
  if (!crop_logits || !y1 || !x1 || (!out_logits && !pred)) return fail(LEDB200_EINVAL, "slide_merge: null buffer");
  if (G < 1 || G > kMaxCrops) return fail(LEDB200_EINVAL, "slide_merge: between 1 and 64 crops per call");
  if (N < 1 || K < 1 || hc < 1 || wc < 1 || hc > H || wc > W) return fail(LEDB200_EINVAL, "slide_merge: bad shape");
  if (pred && pred_dtype != LEDB200_U8 && pred_dtype != LEDB200_I64)
    return fail(LEDB200_EINVAL, "slide_merge: pred dtype must be U8 or I64");
  MergeArgs a;
  a.crops = crop_logits; a.G = G; a.N = N; a.K = K; a.H = H; a.W = W; a.hc = hc; a.wc = wc; a.out = out_logits; a.pred = pred;
  // encoder_decoder.py:289 asserts count_mat != 0 everywhere.  The reference's windows are a cartesian product of row
  // and column offsets, so the image is covered iff every row and every column lies in some window: checked here.
  std::vector<char> rows(H, 0), cols(W, 0);
  for (int g = 0; g < G; ++g) {
    if (y1[g] < 0 || x1[g] < 0 || y1[g] + hc > H || x1[g] + wc > W)
      return fail(LEDB200_EINVAL, "slide_merge: crop window outside the image");
    a.y1[g] = y1[g]; a.x1[g] = x1[g];
  }
  for (int g = 0; g < G; ++g) {
    for (int y = y1[g]; y < y1[g] + hc; ++y) rows[y] = 1;
    for (int x = x1[g]; x < x1[g] + wc; ++x) cols[x] = 1;
  }
  for (int y = 0; y < H; ++y) if (!rows[y]) return fail(LEDB200_EINVAL, "slide_merge: the crop windows leave rows uncovered");
  for (int x = 0; x < W; ++x) if (!cols[x]) return fail(LEDB200_EINVAL, "slide_merge: the crop windows leave columns uncovered");
  const unsigned grid = (unsigned)ceil_div64((int64_t)N * H * W, 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (pred_dtype == LEDB200_I64) slide_merge_kernel<int64_t><<<grid, 256, 0, st>>>(a);
  else slide_merge_kernel<uint8_t><<<grid, 256, 0, st>>>(a);
  LEDB_LAUNCH_OK("slide_merge_kernel");
  return LEDB200_OK;
}

int ledb200_stack_pad(const void* img, int32_t img_dtype, int32_t h, int32_t w, int32_t swap_rb, const float* mean3,
                      const float* std3, float pad_val, float* out, int32_t Hp, int32_t Wp, const void* label,
                      int32_t label_dtype, int64_t* label_out, int32_t seg_pad_val, void* stream) {
  if (!img || !out) return fail(LEDB200_EINVAL, "stack_pad: null buffer");
  if (h < 1 || w < 1 || Hp < h || Wp < w) return fail(LEDB200_EINVAL, "stack_pad: the padded size is smaller than the image");
  if (img_dtype != LEDB200_U8 && img_dtype != LEDB200_F32) return fail(LEDB200_EINVAL, "stack_pad: image dtype must be U8 or F32");
  if ((mean3 == nullptr) != (std3 == nullptr)) return fail(LEDB200_EINVAL, "stack_pad: mean and std come together");
  if ((label == nullptr) != (label_out == nullptr)) return fail(LEDB200_EINVAL, "stack_pad: label and label_out come together");
  if (label && label_dtype != LEDB200_U8 && label_dtype != LEDB200_I64)
    return fail(LEDB200_EINVAL, "stack_pad: label dtype must be U8 or I64");
  StackPadArgs a;
  a.img = img; a.h = h; a.w = w; a.swap_rb = swap_rb ? 1 : 0; a.normalize = mean3 ? 1 : 0;
  for (int c = 0; c < 3; ++c) { a.mean[c] = mean3 ? mean3[c] : 0.f; a.stdv[c] = std3 ? std3[c] : 1.f; }
  a.pad_val = pad_val; a.out = out; a.Hp = Hp; a.Wp = Wp; a.label = label; a.label_out = label_out; a.seg_pad_val = seg_pad_val;
  const unsigned grid = (unsigned)ceil_div64((int64_t)Hp * Wp, 256);
  cudaStream_t st = (cudaStream_t)stream;
  const bool l64 = label && label_dtype == LEDB200_I64;
  if (img_dtype == LEDB200_U8) {
    if (l64) stack_pad_kernel<uint8_t, int64_t><<<grid, 256, 0, st>>>(a);
    else stack_pad_kernel<uint8_t, uint8_t><<<grid, 256, 0, st>>>(a);
  } else {
    if (l64) stack_pad_kernel<float, int64_t><<<grid, 256, 0, st>>>(a);
    else stack_pad_kernel<float, uint8_t><<<grid, 256, 0, st>>>(a);
  }
  LEDB_LAUNCH_OK("stack_pad_kernel");
  return LEDB200_OK;
}

int ledb200_tta_merge(const ledb200_tta_view* views, int32_t V, int32_t N, int32_t K, int32_t oh, int32_t ow,
                      int32_t align_corners, int32_t mode, float threshold, void* pred, int32_t pred_dtype,
                      float* probs_opt, void* stream) {
  if (!views || (!pred && !probs_opt)) return fail(LEDB200_EINVAL, "tta_merge: null buffer");
  if (V < 1 || V > kMaxViews) return fail(LEDB200_EINVAL, "tta_merge: between 1 and 32 views per call");
  if (K < 1 || K > 255) return fail(LEDB200_EINVAL, "tta_merge: K must lie in [1, 255]");
  if (N < 1 || oh < 1 || ow < 1) return fail(LEDB200_EINVAL, "tta_merge: empty tensor");
  if (mode != 0 && mode != 1) return fail(LEDB200_EINVAL, "tta_merge: mode must be 0 (softmax) or 1 (sigmoid)");
  if (pred && mode == 0 && pred_dtype != LEDB200_U8 && pred_dtype != LEDB200_I64)
    return fail(LEDB200_EINVAL, "tta_merge: softmax-mode pred dtype must be U8 or I64");
  if (pred && mode == 1 && pred_dtype != LEDB200_F32)
    return fail(LEDB200_EINVAL, "tta_merge: sigmoid-mode pred (the float mask) must be F32");
  TtaArgs a;
  a.V = V; a.N = N; a.K = K; a.oh = oh; a.ow = ow; a.align_corners = align_corners ? 1 : 0;
  a.threshold = threshold; a.pred = pred; a.probs = probs_opt;
  for (int i = 0; i < V; ++i) {
    const ledb200_tta_view& v = views[i];
    if (!v.logits) return fail(LEDB200_EINVAL, "tta_merge: null view logits");
    if (v.H < 1 || v.W < 1) return fail(LEDB200_EINVAL, "tta_merge: empty view");
    if (v.flip < 0 || v.flip > 2) return fail(LEDB200_EINVAL, "tta_merge: flip must be 0 (none), 1 (horizontal) or 2 (vertical)");
    if (N > 1 && v.image_stride < (int64_t)K * v.H * v.W)
      return fail(LEDB200_EINVAL, "tta_merge: image_stride smaller than one image's [K, H, W] logits");
    a.v[i].logits = v.logits; a.v[i].image_stride = v.image_stride;
    if (!make_geom(v.H, v.W, v.pad_lrtb, v.flip, oh, ow, a.align_corners, a.v[i].g))
      return fail(LEDB200_EINVAL, "tta_merge: a view's padding removes the whole image");
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == 1) return launch_tta_merge<float>(a, st);
  if (pred_dtype == LEDB200_I64) return launch_tta_merge<int64_t>(a, st);
  return launch_tta_merge<uint8_t>(a, st);
}

}  // extern "C"
