// Segmentation overlays (SegLocalVisualizer / SegVisualizationHook, mmseg's `tools/test.py --show-dir`) on the device.
//
// mmseg's _draw_sem_seg colours every pixel with palette[label] (labels >= K stay black), draws a label box and the class
// name at each class's _get_center_loc, and blends `image * (1 - alpha) + mask * alpha` in float64, truncated to uint8.
//
//  * seg_row_hist_kernel   : one block per (row, image) counts the row's pixels of every class < K in a shared-memory
//      histogram and writes the K counts to a [N,K,H] table.
//  * seg_locate_kernel     : one warp per (image, class) finds the row with the most pixels of the class (the first on a
//      tie: _get_center_loc's argmax over np.unique's ascending rows), then walks that row 32 pixels at a time with a
//      ballot to the pixel at index count / 2 in x order.
//  * seg_overlay_kernel    : one thread per output pixel: table[image channel][palette channel] per channel, where the
//      table is the caller's 256 x 256 blend (exact float64 truncation, built on the host).  Panels are side by side
//      (gt | pred), each reading its own label map.
//  * seg_stamp_kernel      : one block per (image, panel) writes that panel's label stamps in array order (a barrier
//      between stamps, so the last stamp touching a pixel wins, as the last cv2 call does on the host).  A stamp is the
//      label box and text that cv2 drew on the host: per pixel a colour and a "touched" flag.
#include <algorithm>

#include "kernels.h"

namespace ledb {
namespace {

__device__ __forceinline__ int64_t load_label(const void* p, int32_t dtype, int64_t i) {
  return dtype == LEDB200_U8 ? (int64_t)static_cast<const uint8_t*>(p)[i] : static_cast<const int64_t*>(p)[i];
}

__global__ void __launch_bounds__(256) seg_row_hist_kernel(const void* __restrict__ labels, int32_t dtype, int H, int W,
                                                          int K, int32_t* __restrict__ counts) {
  __shared__ uint32_t hist[256];
  const int row = blockIdx.x, n = blockIdx.y;
  hist[threadIdx.x] = 0;
  __syncthreads();
  const int64_t base = ((int64_t)n * H + row) * W;
  for (int x = threadIdx.x; x < W; x += blockDim.x) {
    const int64_t v = load_label(labels, dtype, base + x);
    if (v >= 0 && v < K) atomicAdd(&hist[v], 1u);
  }
  __syncthreads();
  if (threadIdx.x < K) counts[((int64_t)n * K + threadIdx.x) * H + row] = (int32_t)hist[threadIdx.x];
}

__global__ void __launch_bounds__(256) seg_locate_kernel(const void* __restrict__ labels, int32_t dtype, int N, int H,
                                                        int W, int K, const int32_t* __restrict__ counts,
                                                        int32_t* __restrict__ out) {
  const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= (int64_t)N * K) return;                       // the whole warp leaves together
  const int64_t n = gw / K;
  const int k = (int)(gw % K);
  const int32_t* c = counts + gw * H;
  int best = 0, brow = H;
  for (int r = lane; r < H; r += 32) {
    const int v = c[r];
    if (v > best) { best = v; brow = r; }                   // rows ascend per lane: strict > keeps the first
  }
  for (int o = 16; o; o >>= 1) {
    const int ob = __shfl_xor_sync(0xffffffffu, best, o), orow = __shfl_xor_sync(0xffffffffu, brow, o);
    if (ob > best || (ob == best && orow < brow)) { best = ob; brow = orow; }
  }
  int32_t* o3 = out + gw * 3;
  if (best == 0) {
    if (lane == 0) { o3[0] = 0; o3[1] = 0; o3[2] = 0; }
    return;
  }
  int target = best / 2;
  const int64_t base = (n * H + brow) * W;
  for (int x0 = 0; x0 < W; x0 += 32) {
    const int x = x0 + lane;
    const bool hit = x < W && load_label(labels, dtype, base + x) == k;
    const uint32_t m = __ballot_sync(0xffffffffu, hit);
    const int pc = __popc(m);
    if (target < pc) {                                      // uniform over the warp
      if (hit && __popc(m & ((1u << lane) - 1u)) == target) { o3[0] = 1; o3[1] = x; o3[2] = brow; }
      break;
    }
    target -= pc;
  }
}

__device__ __forceinline__ void blend_pixel(const uint8_t* __restrict__ img, int64_t plane, int64_t at,
                                            const uint8_t* __restrict__ table, uint32_t r, uint32_t g, uint32_t b,
                                            uint8_t* __restrict__ o) {
  const uint32_t ib = img[at], ig = img[at + plane], ir = img[at + 2 * plane];
  o[0] = __ldg(table + ir * 256 + r);
  o[1] = __ldg(table + ig * 256 + g);
  o[2] = __ldg(table + ib * 256 + b);
}

__global__ void __launch_bounds__(256) seg_overlay_kernel(const uint8_t* __restrict__ images, const void* gt,
                                                         int32_t gt_dtype, const void* pred, int32_t pred_dtype, int N,
                                                         int H, int W, int P, int K, const uint8_t* __restrict__ palette,
                                                         const uint8_t* __restrict__ table, uint8_t* __restrict__ out) {
  __shared__ uint8_t pal[256 * 3];
  for (int i = threadIdx.x; i < K * 3; i += blockDim.x) pal[i] = palette[i];
  __syncthreads();
  const int64_t PW = (int64_t)P * W, total = (int64_t)N * H * PW;
  const int64_t plane = (int64_t)H * W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t xo = i % PW, t = i / PW, y = t % H, n = t / H;
    const int p = (int)(xo / W);
    const int64_t x = xo - (int64_t)p * W, pix = (n * H + y) * W + x;
    const bool use_gt = p == 0 && gt != nullptr;
    const int64_t lab = use_gt ? load_label(gt, gt_dtype, pix) : load_label(pred, pred_dtype, pix);
    uint32_t r = 0, g = 0, b = 0;
    if (lab >= 0 && lab < K) { r = pal[3 * lab]; g = pal[3 * lab + 1]; b = pal[3 * lab + 2]; }
    blend_pixel(images + n * 3 * plane, plane, y * W + x, table, r, g, b, out + i * 3);
  }
}

__global__ void __launch_bounds__(256) seg_stamp_kernel(const uint8_t* __restrict__ images, int N, int H, int W, int P,
                                                       const uint8_t* __restrict__ table,
                                                       const ledb200_seg_stamp* __restrict__ stamps, int num_stamps,
                                                       const uint8_t* __restrict__ data, int64_t data_bytes,
                                                       uint8_t* __restrict__ out) {
  const int n = blockIdx.x / P, p = blockIdx.x % P;
  const int64_t plane = (int64_t)H * W, PW = (int64_t)P * W;
  for (int s = 0; s < num_stamps; ++s) {
    const ledb200_seg_stamp d = stamps[s];
    if (d.image != n || d.panel != p) continue;
    if (d.x0 < 0 || d.y0 < 0 || d.w < 1 || d.h < 1 || d.x0 + (int64_t)d.w > W || d.y0 + (int64_t)d.h > H ||
        d.offset < 0 || d.offset + 4 * (int64_t)d.w * d.h > data_bytes)
      continue;
    const uint8_t* src = data + d.offset;
    for (int64_t j = threadIdx.x; j < (int64_t)d.w * d.h; j += blockDim.x) {
      const uint8_t* q = src + 4 * j;
      if (!q[3]) continue;
      const int64_t y = d.y0 + j / d.w, x = d.x0 + j % d.w;
      blend_pixel(images + (int64_t)n * 3 * plane, plane, y * W + x, table, q[0], q[1], q[2],
                  out + (((int64_t)n * H + y) * PW + (int64_t)p * W + x) * 3);
    }
    __syncthreads();
  }
}

}  // namespace
}  // namespace ledb

using namespace ledb;

extern "C" {

int64_t ledb200_seg_locate_workspace_bytes(int32_t N, int32_t H, int32_t K) {
  if (N < 1 || H < 1 || K < 1 || K > 255)
    return fail(LEDB200_EINVAL, "seg_locate_workspace_bytes: N, H >= 1 and 1 <= K <= 255");
  return (int64_t)N * K * H * 4;
}

int ledb200_seg_label_locations(const void* labels, int32_t dtype, int32_t N, int32_t H, int32_t W, int32_t K,
                                int32_t* out, void* workspace, void* stream) {
  if (N < 1 || H < 1 || W < 1) return fail(LEDB200_EINVAL, "seg_label_locations: N, H and W must be at least 1");
  if (K < 1 || K > 255) return fail(LEDB200_EINVAL, "seg_label_locations: K must be in 1 .. 255");
  if (N > 65535) return fail(LEDB200_EINVAL, "seg_label_locations: at most 65535 maps per call");
  if (dtype != LEDB200_U8 && dtype != LEDB200_I64) return fail(LEDB200_EINVAL, "seg_label_locations: labels must be U8 or I64");
  if (!labels || !out || !workspace) return fail(LEDB200_EINVAL, "seg_label_locations: null buffer");
  cudaStream_t st = (cudaStream_t)stream;
  int32_t* counts = (int32_t*)workspace;
  seg_row_hist_kernel<<<dim3((unsigned)H, (unsigned)N), 256, 0, st>>>(labels, dtype, H, W, K, counts);
  LEDB_LAUNCH_OK("seg_row_hist_kernel");
  const int64_t warps = (int64_t)N * K;
  seg_locate_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, st>>>(labels, dtype, N, H, W, K, counts, out);
  LEDB_LAUNCH_OK("seg_locate_kernel");
  return LEDB200_OK;
}

int ledb200_seg_overlay(const uint8_t* images, const void* gt, int32_t gt_dtype, const void* pred, int32_t pred_dtype,
                        int32_t N, int32_t H, int32_t W, int32_t K, const uint8_t* palette, const uint8_t* table,
                        const ledb200_seg_stamp* stamps, int32_t num_stamps, const uint8_t* stamp_data,
                        int64_t stamp_bytes, uint8_t* out, void* stream) {
  if (N < 1 || H < 1 || W < 1) return fail(LEDB200_EINVAL, "seg_overlay: N, H and W must be at least 1");
  if (K < 1 || K > 255) return fail(LEDB200_EINVAL, "seg_overlay: K must be in 1 .. 255");
  if (!gt && !pred) return fail(LEDB200_EINVAL, "seg_overlay: no label map (gt and pred are both null)");
  for (int k = 0; k < 2; ++k) {
    const int32_t dt = k ? pred_dtype : gt_dtype;
    if ((k ? pred : gt) && dt != LEDB200_U8 && dt != LEDB200_I64)
      return fail(LEDB200_EINVAL, "seg_overlay: label maps must be U8 or I64");
  }
  if (!images || !palette || !table || !out) return fail(LEDB200_EINVAL, "seg_overlay: null buffer");
  if (num_stamps < 0 || (num_stamps > 0 && (!stamps || !stamp_data)))
    return fail(LEDB200_EINVAL, "seg_overlay: stamps without their descriptors or data");
  const int P = (gt ? 1 : 0) + (pred ? 1 : 0);
  if ((int64_t)N * P > INT32_MAX) return fail(LEDB200_EINVAL, "seg_overlay: too many panels in one call");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t total = (int64_t)N * H * P * W;
  const int64_t blocks = std::min<int64_t>((total + 255) / 256, (int64_t)1 << 20);
  seg_overlay_kernel<<<(unsigned)blocks, 256, 0, st>>>(images, gt, gt_dtype, pred, pred_dtype, N, H, W, P, K, palette,
                                                       table, out);
  LEDB_LAUNCH_OK("seg_overlay_kernel");
  if (num_stamps > 0) {
    seg_stamp_kernel<<<(unsigned)(N * P), 256, 0, st>>>(images, N, H, W, P, table, stamps, num_stamps, stamp_data,
                                                        stamp_bytes, out);
    LEDB_LAUNCH_OK("seg_stamp_kernel");
  }
  return LEDB200_OK;
}

}  // extern "C"
