// Cityscapes pixel-level statistics (CityscapesMetric: cityscapesscripts' evalPixelLevelSemanticLabeling.evaluatePair
// with evalInstLevelScore) on the device, for a batch of same-shape images, reading each input once.
//
// Per pixel: the prediction (a trainId, uint8 or int64) goes through the trainId -> labelId table, then
//   * the 34 x 34 confusion matrix of (GT labelId, predicted labelId) gains one count;
//   * when the GT instanceId is above 1000 and its class l = instanceId / 1000 is a counted instance class (the host
//     table says which: person .. bicycle without caravan / trailer), the instance's size, tp (predicted labelId == l)
//     and catTp (predicted labelId in l's category) gain one count.  Counted classes are ids 24 .. 33, so every counted
//     instance id lies in the dense range 24000 .. 33999.
// Statuses per image (bits): a GT labelId above 33, a predicted labelId outside 0 .. 33, an instance id whose class is
// neither counted nor skipped (CSEval's KeyError), an int64 prediction outside 0 .. 255.
//
//  * cityscapes_stats_kernel   : a grid of (blocks per image, N); each block of 1024 threads owns a contiguous chunk of
//      one image, each thread 8 consecutive pixels at a time (vector loads when the image allows).  A thread merges
//      runs of equal confusion bins and of equal instance ids in registers and adds a finished run to the block's
//      shared-memory histograms (1156 confusion bins, 3 x 10000 instance counters: 125 KB) with one atomic each.  At the
//      end the block adds its non-zero bins to the int64 matrix and the per-image int32 instance counters in global
//      memory.  Every count is an integer, so the result does not depend on the order of the atomics.
//  * cityscapes_count_kernel / cityscapes_compact_kernel : one block per image counts the instance ids seen, then
//      writes their records (instId, size, tp, catTp) in ascending instId (np.unique's order), the images' records back
//      to back after the statuses and counts, so the host fetches everything with one copy.
#include <algorithm>

#include "kernels.h"

namespace ledb {
namespace {

constexpr int kIds = 34;                      // labelIds 0 .. 33
constexpr int kBins = kIds * kIds;
constexpr int kInstBase = 24000, kInstIds = 10000;
constexpr int kThreads = 1024;
constexpr int kStrip = 8;                     // pixels per thread per step (16 would spill at 64 registers)
constexpr int kRuleError = 0, kRuleSkip = 1, kRuleCount = 2;
constexpr int kStGt = 1, kStPred = 2, kStInst = 4, kStRange = 8;

struct Tables {
  int32_t train_to_id[256];
  int8_t category[kIds];                      // -1: not in an instance category
  int8_t rule[kIds];
};

struct StatsSmem {
  uint32_t cm[kBins];
  uint32_t size[kInstIds], tp[kInstIds], cat[kInstIds];
  int32_t train_to_id[256];
  int8_t category[kIds], rule[kIds];
  int status;
};

// a prediction as an index of the trainId table, 256 when it is outside 0 .. 255
__device__ __forceinline__ int clamp_pred(int64_t v) { return (uint64_t)v > 255 ? 256 : (int)v; }

template <typename TP>
__device__ __forceinline__ void load_strip(const TP* __restrict__ pred, const uint8_t* __restrict__ gt,
                                           const int32_t* __restrict__ inst, int64_t i, int64_t end, bool vec,
                                           int (&p)[kStrip], int (&g)[kStrip], int (&q)[kStrip]) {
  if (vec) {
    const uint2 gv = __ldg(reinterpret_cast<const uint2*>(gt + i));
    const uint32_t gw[2] = {gv.x, gv.y};
#pragma unroll
    for (int k = 0; k < kStrip; ++k) g[k] = (gw[k / 4] >> (8 * (k % 4))) & 0xff;
#pragma unroll
    for (int v = 0; v < kStrip / 4; ++v) {
      const int4 qv = __ldg(reinterpret_cast<const int4*>(inst + i) + v);
      q[4 * v] = qv.x; q[4 * v + 1] = qv.y; q[4 * v + 2] = qv.z; q[4 * v + 3] = qv.w;
    }
    if constexpr (sizeof(TP) == 1) {
      const uint2 pv = __ldg(reinterpret_cast<const uint2*>(pred + i));
      const uint32_t pw[2] = {pv.x, pv.y};
#pragma unroll
      for (int k = 0; k < kStrip; ++k) p[k] = (pw[k / 4] >> (8 * (k % 4))) & 0xff;
    } else {
#pragma unroll
      for (int v = 0; v < kStrip / 2; ++v) {
        const longlong2 pv = __ldg(reinterpret_cast<const longlong2*>(pred + i) + v);
        p[2 * v] = clamp_pred(pv.x); p[2 * v + 1] = clamp_pred(pv.y);
      }
    }
    return;
  }
#pragma unroll
  for (int k = 0; k < kStrip; ++k) {
    const bool in = i + k < end;
    p[k] = in ? clamp_pred((int64_t)__ldg(pred + i + k)) : 0;
    g[k] = in ? __ldg(gt + i + k) : -1;       // -1: past the end, counted nowhere
    q[k] = in ? __ldg(inst + i + k) : 0;
  }
}

template <typename TP>
__global__ void __launch_bounds__(kThreads, 1)
cityscapes_stats_kernel(const TP* __restrict__ pred, const uint8_t* __restrict__ gt, const int32_t* __restrict__ inst,
                        int64_t npix, int64_t chunk, bool vec, const __grid_constant__ Tables tables,
                        unsigned long long* __restrict__ cm, unsigned long long* __restrict__ cm_last, int last_image,
                        uint32_t* __restrict__ counters, int32_t* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  StatsSmem& sm = *reinterpret_cast<StatsSmem*>(smem_raw);
  const int t = threadIdx.x;
  const int img = blockIdx.y;
  for (int i = t; i < kBins; i += kThreads) sm.cm[i] = 0;
  for (int i = t; i < kInstIds; i += kThreads) { sm.size[i] = 0; sm.tp[i] = 0; sm.cat[i] = 0; }
  if (t < 256) sm.train_to_id[t] = tables.train_to_id[t];
  if (t < kIds) { sm.category[t] = tables.category[t]; sm.rule[t] = tables.rule[t]; }
  if (t == 0) sm.status = 0;
  __syncthreads();

  const int64_t base = (int64_t)img * npix;
  const int64_t c0 = (int64_t)blockIdx.x * chunk, c1 = min(npix, c0 + chunk);
  int flags = 0;
  int cur_bin = -1;                            // open confusion run
  uint32_t bin_n = 0;
  int cur_k = -1;                              // open instance run: dense index, size, tp, catTp
  uint32_t k_size = 0, k_tp = 0, k_cat = 0;
  for (int64_t s = c0 + (int64_t)t * kStrip; s < c1; s += (int64_t)kThreads * kStrip) {
    int p[kStrip], g[kStrip], q[kStrip];
    load_strip(pred, gt, inst, base + s, base + c1, vec, p, g, q);
#pragma unroll
    for (int k = 0; k < kStrip; ++k) {
      if (g[k] < 0) continue;
      int pid = -1;
      if (p[k] > 255) flags |= kStRange;
      else pid = sm.train_to_id[p[k]];
      if (pid < 0 || pid >= kIds) { flags |= kStPred; pid = -1; }
      if (g[k] >= kIds) flags |= kStGt;
      const int bin = (pid >= 0 && g[k] < kIds) ? g[k] * kIds + pid : -1;
      if (bin != cur_bin) {
        if (cur_bin >= 0) atomicAdd(&sm.cm[cur_bin], bin_n);
        cur_bin = bin; bin_n = 0;
      }
      ++bin_n;
      const int id = q[k];
      int kk = -1;
      if (id > 1000) {
        const int l = id / 1000;
        const int rule = l < kIds ? sm.rule[l] : kRuleError;
        if (rule == kRuleError) flags |= kStInst;
        else if (rule == kRuleCount) kk = id - kInstBase;
        if (kk >= 0) {
          if (kk != cur_k) {
            if (cur_k >= 0) {
              atomicAdd(&sm.size[cur_k], k_size); atomicAdd(&sm.tp[cur_k], k_tp); atomicAdd(&sm.cat[cur_k], k_cat);
            }
            cur_k = kk; k_size = 0; k_tp = 0; k_cat = 0;
          }
          ++k_size;
          k_tp += pid == l;
          k_cat += pid >= 0 && sm.category[pid] >= 0 && sm.category[pid] == sm.category[l];
        }
      }
    }
  }
  if (cur_bin >= 0) atomicAdd(&sm.cm[cur_bin], bin_n);
  if (cur_k >= 0) { atomicAdd(&sm.size[cur_k], k_size); atomicAdd(&sm.tp[cur_k], k_tp); atomicAdd(&sm.cat[cur_k], k_cat); }
  if (flags) atomicOr(&sm.status, flags);
  __syncthreads();

  for (int i = t; i < kBins; i += kThreads) {
    const uint32_t v = sm.cm[i];
    if (!v) continue;
    atomicAdd(cm + i, (unsigned long long)v);
    if (img == last_image && cm_last) atomicAdd(cm_last + i, (unsigned long long)v);
  }
  uint32_t* cnt = counters + (int64_t)img * 3 * kInstIds;
  for (int i = t; i < kInstIds; i += kThreads) {
    if (!sm.size[i]) continue;
    atomicAdd(cnt + i, sm.size[i]);
    if (sm.tp[i]) atomicAdd(cnt + kInstIds + i, sm.tp[i]);
    if (sm.cat[i]) atomicAdd(cnt + 2 * kInstIds + i, sm.cat[i]);
  }
  if (t == 0 && sm.status) atomicOr(status + img, sm.status);
}

// the number of instance ids of image blockIdx.x into counts[img]
__global__ void __launch_bounds__(kThreads) cityscapes_count_kernel(const uint32_t* __restrict__ counters,
                                                                     int32_t* __restrict__ counts) {
  const uint32_t* sz = counters + (int64_t)blockIdx.x * 3 * kInstIds;
  int n = 0;
  for (int i0 = 0; i0 < kInstIds; i0 += kThreads) {
    const int i = i0 + threadIdx.x;
    n += __syncthreads_count(i < kInstIds && sz[i] > 0);
  }
  if (threadIdx.x == 0) counts[blockIdx.x] = n;
}

// image blockIdx.x's records at its offset (the counts of the images before it), in ascending instance id
__global__ void __launch_bounds__(kThreads) cityscapes_compact_kernel(const uint32_t* __restrict__ counters,
                                                                       const int32_t* __restrict__ counts,
                                                                       int32_t* __restrict__ records) {
  __shared__ int warp_n[kThreads / 32];
  __shared__ int64_t off_s;
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int img = blockIdx.x;
  if (t == 0) {
    int64_t o = 0;
    for (int m = 0; m < img; ++m) o += counts[m];
    off_s = o;
  }
  __syncthreads();
  int64_t off = off_s;
  const uint32_t* cnt = counters + (int64_t)img * 3 * kInstIds;
  for (int i0 = 0; i0 < kInstIds; i0 += kThreads) {
    const int i = i0 + t;
    const bool has = i < kInstIds && cnt[i] > 0;
    const unsigned ball = __ballot_sync(0xffffffffu, has);
    if (lane == 0) warp_n[wid] = __popc(ball);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < kThreads / 32; ++w) {
      const int v = warp_n[w];
      before += w < wid ? v : 0;
      total += v;
    }
    if (has) {
      int32_t* r = records + 4 * (off + before + __popc(ball & ((1u << lane) - 1)));
      r[0] = kInstBase + i; r[1] = (int32_t)cnt[i]; r[2] = (int32_t)cnt[kInstIds + i];
      r[3] = (int32_t)cnt[2 * kInstIds + i];
    }
    off += total;
    __syncthreads();
  }
}

}  // namespace
}  // namespace ledb

using namespace ledb;

extern "C" {

int64_t ledb200_cityscapes_out_ints(int32_t N) {
  if (N < 1) return fail(LEDB200_EINVAL, "cityscapes_out_ints: N must be at least 1");
  return 2 * (int64_t)N + 4 * (int64_t)N * kInstIds;
}

int64_t ledb200_cityscapes_workspace_bytes(int32_t N) {
  if (N < 1) return fail(LEDB200_EINVAL, "cityscapes_workspace_bytes: N must be at least 1");
  return (int64_t)N * 3 * kInstIds * 4;
}

int ledb200_cityscapes_accumulate(const void* pred, int32_t pred_dtype, const uint8_t* gt, const int32_t* inst,
                                  int32_t N, int32_t H, int32_t W, const int32_t* train_to_id, const int8_t* category,
                                  const int8_t* inst_rule, int64_t* cm_inout, int64_t* cm_last_out, int32_t* out,
                                  void* workspace, void* stream) {
  if (N < 1 || H < 1 || W < 1) return fail(LEDB200_EINVAL, "cityscapes_accumulate: N, H and W must be at least 1");
  if (N > 65535) return fail(LEDB200_EINVAL, "cityscapes_accumulate: at most 65535 images per call");
  if ((int64_t)H * W >= (int64_t)1 << 31) return fail(LEDB200_EINVAL, "cityscapes_accumulate: H * W must be below 2^31");
  if (pred_dtype != LEDB200_U8 && pred_dtype != LEDB200_I64)
    return fail(LEDB200_EINVAL, "cityscapes_accumulate: predictions must be U8 or I64");
  if (!pred || !gt || !inst || !train_to_id || !category || !inst_rule || !cm_inout || !out || !workspace)
    return fail(LEDB200_EINVAL, "cityscapes_accumulate: null buffer or table");
  Tables tab;
  for (int i = 0; i < 256; ++i) tab.train_to_id[i] = train_to_id[i];
  for (int i = 0; i < kIds; ++i) {
    if (category[i] < -1) return fail(LEDB200_EINVAL, "cityscapes_accumulate: categories are -1 or non-negative");
    if (inst_rule[i] != kRuleError && inst_rule[i] != kRuleSkip && inst_rule[i] != kRuleCount)
      return fail(LEDB200_EINVAL, "cityscapes_accumulate: instance rules are 0 (error), 1 (skip) or 2 (count)");
    if (inst_rule[i] == kRuleCount && (i < kInstBase / 1000 || category[i] < 0))
      return fail(LEDB200_EINVAL, "cityscapes_accumulate: counted instance classes are ids 24 .. 33 of a category");
    tab.category[i] = category[i];
    tab.rule[i] = inst_rule[i];
  }
  cudaStream_t st = (cudaStream_t)stream;
  uint32_t* counters = (uint32_t*)workspace;
  const int64_t npix = (int64_t)H * W;
  LEDB_CUDA_OK(cudaMemsetAsync(out, 0, 2 * (size_t)N * sizeof(int32_t), st));
  LEDB_CUDA_OK(cudaMemsetAsync(counters, 0, (size_t)ledb200_cityscapes_workspace_bytes(N), st));
  if (cm_last_out) LEDB_CUDA_OK(cudaMemsetAsync(cm_last_out, 0, kBins * sizeof(int64_t), st));

  // about one block per SM in all: each block zeroes and flushes 125 KB of shared histograms once
  int sms = 148;
  { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
  const int64_t per_img = std::max<int64_t>(1, std::min<int64_t>((sms + N - 1) / N, ceil_div64(npix, kThreads * kStrip)));
  const int64_t chunk = ceil_div64(ceil_div64(npix, per_img), kStrip) * kStrip;
  const int64_t blocks = ceil_div64(npix, chunk);
  const bool vec = npix % kStrip == 0 && (uintptr_t)pred % 16 == 0 && (uintptr_t)gt % 16 == 0 &&
                   (uintptr_t)inst % 16 == 0;
  const size_t smem = sizeof(StatsSmem);
  const dim3 grid((unsigned)blocks, (unsigned)N);
  auto* cmu = reinterpret_cast<unsigned long long*>(cm_inout);
  auto* cml = reinterpret_cast<unsigned long long*>(cm_last_out);
  if (pred_dtype == LEDB200_U8) {
    LEDB_CUDA_OK(cudaFuncSetAttribute(cityscapes_stats_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cityscapes_stats_kernel<uint8_t><<<grid, kThreads, smem, st>>>((const uint8_t*)pred, gt, inst, npix, chunk, vec, tab,
                                                                   cmu, cml, N - 1, counters, out);
  } else {
    LEDB_CUDA_OK(cudaFuncSetAttribute(cityscapes_stats_kernel<int64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cityscapes_stats_kernel<int64_t><<<grid, kThreads, smem, st>>>((const int64_t*)pred, gt, inst, npix, chunk, vec, tab,
                                                                   cmu, cml, N - 1, counters, out);
  }
  LEDB_LAUNCH_OK("cityscapes_stats_kernel");
  cityscapes_count_kernel<<<(unsigned)N, kThreads, 0, st>>>(counters, out + N);
  LEDB_LAUNCH_OK("cityscapes_count_kernel");
  cityscapes_compact_kernel<<<(unsigned)N, kThreads, 0, st>>>(counters, out + N, out + 2 * N);
  LEDB_LAUNCH_OK("cityscapes_compact_kernel");
  return LEDB200_OK;
}

}  // extern "C"
