// The logit ladder of LEDHead on the tensor cores (north_star kernels 1 + 3 + 4 fused).
//
// Replaces, per rung,
//   `_make_base_head` 3x3 conv + folded BN + ReLU on a stem tap (mmseg/models/decode_heads/led_head.py:84-99),
//   the rung of the patched `BaseDecodeHead.predict_by_feat` (mmseg/models/decode_heads/decode_head.py:362-379):
//        r2 = head_x2(x2) + up2(x_c)        r1 = head_x1(x1) + up2(r2)        out = up2(r1)
//   and, for the last rung, `postprocess_result`'s argmax(dim=0) (mmseg/models/segmentors/base.py:187-188).
//
//   ladder_kernel<false>  (rung):  out[N,H,W,24] fp16 = relu(conv3x3(in) + b) + up2(up)          head_x2 always;
//                                  head_x1 only when the caller wants the full-resolution logits (tail2 follows)
//   ladder_kernel<true>   (final): label[N,2H,2W] = argmax_k up2(relu(conv3x3(in) + b) + up2(up))   head_x1 hot path:
//                                  r1 (402 MB per 16-image batch as fp16) never reaches HBM.
//
// GEMM side (same machinery as conv_tc.cu, MODE 0 / KC = 32 / resident weights): M = 128 pixels (16 x 8 tile),
// N = 32 (K <= 24 classes, zero padded), K = 9 taps x Cin; ONE TMA halo slab (18 x 10 pixels x 32 ch, 64 B swizzle)
// per Cin block, nine shifted UMMA descriptors into it; fp32 accumulators in TMEM, EIGHT 32-column stages.
//
// Epilogue:
//   * 16 epilogue warps = four groups of four; group g owns every fourth tile of the CTA.  With a per-tile epilogue
//     of ~700 instructions per thread the warp schedulers are the limiter, so each gets 4 epilogue warps;
//   * the `up` corner patch (10 x 6 pixels x 24 ch fp16 = 2.9 KB) arrives by TMA per tile (its own full / empty
//     barrier ring, loaded with the A slab), so the gather is 12 conflict-free LDS.128 (48 B pixel stride) at 29 clk
//     instead of L2 round trips, and nothing has to be prefetched into registers across the accumulator wait;
//   * bilinear border clamps are index clamps at READ time (TMA zero fill outside the image is never consumed),
//     which is ATen's align_corners=False rule: weights (1/4, 3/4) by parity, fma(v, 3/4, v/4) == v exactly;
//   * final rung: tiles OVERLAP by one r1 row / column (stride 15 x 7 over a 16 x 8 MMA tile; the last tile of a row /
//     column is shifted back so that it ends at the image edge, like every other TMA box of this library it then
//     leaves the tensor by at most one pixel).  The group writes its r1 tile (fp16, 48 B per pixel) to a
//     double-buffered shared exchange tile, one named barrier, then thread (i, j) owns the 2 x 2 outputs BETWEEN r1
//     pixels (i, j) .. (i+1, j+1) - rows 2y+1, 2y+2 - from its own pixel (registers) and three neighbours (LDS), with
//     packed f32x2 lerps in tail2_kernel's operation order (horizontal with (1/4, 3/4), then vertical: bit-identical
//     logits) and a strict `>` running argmax in ascending class order = torch.argmax's first-max rule.  Output row 0 /
//     column 0 (source index clamped: a pure copy of the first r1 row / column) are written by the threads of r1 row 0
//     / column 0 in a second, rare pass.  22 % of the MMA work is recomputed (pixels covered by two tiles get
//     bit-identical values, so the duplicate label stores are benign); in exchange r1 never makes the 0.8 GB per step
//     round trip through HBM and no separate tail launch is needed.
//   * one producer thread per operand (warp 0: A slabs, warp 3: `up` patches), tile coordinates advanced as
//     mixed-radix digits: a single thread doing both plus three integer divisions per tile bounded the kernel at
//     ~800 clk per tile (probe: 239 us with every other role switched off).
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <mutex>

#include "tc_common.cuh"

namespace ledb {
namespace {

using namespace tc;

constexpr int LTH = 16, LTW = 8;                 // MMA tile in rung pixels
constexpr int L_GROUPS = 4;                      // epilogue groups of 4 warps
constexpr int L_EPI_WARP0 = 4;                   // first epilogue warp (multiple of 4: TMEM lane quadrant = warp & 3)
constexpr int L_THREADS = 32 * (L_EPI_WARP0 + 4 * L_GROUPS);
constexpr int L_NST = 8;                         // accumulator stages (32 columns each)
constexpr int L_NU = 8;                          // `up` patch ring
constexpr int L_SA = 8;                          // A slab ring
constexpr int L_NP = 32;                         // UMMA N
constexpr int L_CH = 24;                         // stored channels per rung pixel (48 B)
constexpr int UP_H = 10, UP_W = 6;               // `up` patch
constexpr uint32_t UP_BYTES = UP_H * UP_W * L_CH * 2;          // 2880
constexpr uint32_t UP_STAGE = 3072;
constexpr uint32_t A_BOX = (LTH + 2) * (LTW + 2) * 64;          // 11520
constexpr uint32_t A_STAGE = 12288;
constexpr uint32_t B_TILE = L_NP * 64;                          // 2048
constexpr uint32_t X_TILE = 128 * L_CH * 2;                     // 6144: r1 exchange tile of one group

struct LadderParams {
  int N, H, W;                 // rung size (= conv output = conv input size)
  int Cin, nchunks;            // Cin = 32 * nchunks
  int K;                       // classes (<= 24)
  int up_h, up_w;              // H == 2 up_h, W == 2 up_w
  int tiles_h, tiles_w;
  uint32_t total_tiles;
  int th_step, tw_step;        // tile stride (16 x 8; final: 15 x 7)
  int r_max, c_max;            // largest tile origin (final: H - 16, W - 8: the last tile ends at the image edge)
  int step[3][3];              // tile-index step of 1, 2 and 4 grids as digits (tile col, tile row, image)
  const float* bias;
  __half* out;                 // rung: [N,H,W,24] fp16
  void* pred; int pred_i64;    // final: [N,2H,2W] uint8 or int64
  int dbg;                     // LEDB200_LADDER_DBG probe bits (timing / diagnosis only): 1 no output phase, 2 no `up` gather,
                               // 4 no MMAs, 8 final mode also stores r1 to `out`, 16 single MMA issuer, 32 release the accumulator stage and the
                               // `up` patch at the END of the tile, 64 no uniform-corner shortcut in the final rung
};

__device__ __forceinline__ void tc_ld8(uint32_t taddr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds128f(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
// source row of an exact x2 bilinear upsample (align_corners=False): output y reads rows lo(y), lo(y) + 1 with
// weights (1/4, 3/4) for even y and (3/4, 1/4) for odd y
__device__ __forceinline__ int lo2(int y) { return (y - 1) >> 1; }
__device__ __forceinline__ float2 lerp2(float2 a, float2 b, float2 w0, float2 w1) {
  return __ffma2_rn(b, w1, __fmul2_rn(a, w0));   // b*w1 + a*w0 per lane (tail.cu lerp2: same bits)
}

template <bool FINAL>
__global__ void __launch_bounds__(L_THREADS, 1)
ladder_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
              const __grid_constant__ CUtensorMap tmU, const __grid_constant__ LadderParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                                        // [L_SA][A_STAGE]
  uint8_t* sB = sA + (size_t)L_SA * A_STAGE;                 // [nchunks * 9][B_TILE]   (resident weights)
  uint8_t* sU = sB + (size_t)P.nchunks * 9 * B_TILE;         // [L_NU][UP_STAGE]
  uint8_t* sX = sU + (size_t)L_NU * UP_STAGE;                // [L_GROUPS][2][X_TILE]   (final rung only)
  float* s_bias = reinterpret_cast<float*>(sX + (FINAL ? (size_t)L_GROUPS * 2 * X_TILE : 0));   // [32]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_bias + L_NP);
  uint64_t* a_full = bars;                  // [L_SA]
  uint64_t* a_empty = a_full + L_SA;        // [L_SA]
  uint64_t* u_full = a_empty + L_SA;        // [L_NU]
  uint64_t* u_empty = u_full + L_NU;        // [L_NU]
  uint64_t* t_full = u_empty + L_NU;        // [L_NST]
  uint64_t* t_empty = t_full + L_NST;       // [L_NST]
  uint64_t* b_full = t_empty + L_NST;       // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t total = P.total_tiles;

  if (threadIdx.x == 0) {
    prefetch_tensormap(&tmA); prefetch_tensormap(&tmB); prefetch_tensormap(&tmU);
    for (int i = 0; i < L_SA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < L_NU; ++i) { mbar_init(&u_full[i], 1); mbar_init(&u_empty[i], 4); }
    for (int i = 0; i < L_NST; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 4); }
    mbar_init(b_full, 1);
    mbar_fence_init();
    // resident weights: one barrier, one expect_tx (requested before the CTA-wide sync, as in conv_tc.cu)
    mbar_expect_tx(b_full, (uint32_t)(P.nchunks * 9) * B_TILE);
    for (int ch = 0; ch < P.nchunks; ++ch)
      for (int t = 0; t < 9; ++t)
        tma_load_2d(smem_u32(sB + (size_t)(ch * 9 + t) * B_TILE), &tmB, smem_u32(b_full), t * P.Cin + ch * 32, 0);
  }
  if (warp == 1) tmem_alloc(tmem_slot, L_NST * L_NP);
  uint32_t tmem_base = 0;
  if (warp == 0) {
    __syncwarp();
    asm volatile("bar.arrive 1, %0;" ::"n"(L_THREADS) : "memory");
  } else {
    if (threadIdx.x >= 32 && threadIdx.x < 32 + L_NP) {
      const int c = threadIdx.x - 32;
      s_bias[c] = (P.bias && c < P.K) ? P.bias[c] : 0.f;
    }
    tc_fence_before();
    asm volatile("bar.sync 1, %0;" ::"n"(L_THREADS) : "memory");
    tc_fence_after();
    tmem_base = *tmem_slot;
  }

  // tile coordinates: (tile col, tile row, image) digits advanced by `k` grids at a time (no per-tile divisions)
  struct TileIt {
    int tw, th, n;
    __device__ __forceinline__ void init(uint32_t t, const LadderParams& P) {
      tw = (int)(t % (uint32_t)P.tiles_w); t /= (uint32_t)P.tiles_w;
      th = (int)(t % (uint32_t)P.tiles_h);
      n = (int)(t / (uint32_t)P.tiles_h);
    }
    __device__ __forceinline__ void step(const int* d, const LadderParams& P) {
      tw += d[0]; if (tw >= P.tiles_w) { tw -= P.tiles_w; ++th; }
      th += d[1]; if (th >= P.tiles_h) { th -= P.tiles_h; ++n; }
      n += d[2];
    }
    __device__ __forceinline__ int r0(const LadderParams& P) const { return min(th * P.th_step, P.r_max); }
    __device__ __forceinline__ int c0(const LadderParams& P) const { return min(tw * P.tw_step, P.c_max); }
  };

  if (warp == 0) {
    // =========================== TMA producer, A slabs (one elected lane) ==========================
    if (elect_one()) {
      int sa = 0, pa = 0;
      TileIt it; it.init(blockIdx.x, P);
      for (uint32_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int r0 = it.r0(P), c0 = it.c0(P);
        for (int ch = 0; ch < P.nchunks; ++ch) {
          mbar_wait(&a_empty[sa], pa ^ 1);
          mbar_expect_tx(&a_full[sa], A_BOX);
          tma_load_4d(smem_u32(sA + (size_t)sa * A_STAGE), &tmA, smem_u32(&a_full[sa]), ch * 32, c0 - 1, r0 - 1, it.n);
          if (++sa == L_SA) { sa = 0; pa ^= 1; }
        }
        it.step(P.step[0], P);
      }
    }
    __syncwarp();
  } else if (warp == 3) {
    // =========================== TMA producer, `up` patches (one elected lane) =====================
    if (elect_one()) {
      int su = 0, pu = 0;
      TileIt it; it.init(blockIdx.x, P);
      for (uint32_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
        mbar_wait(&u_empty[su], pu ^ 1);
        mbar_expect_tx(&u_full[su], UP_BYTES);
        tma_load_4d(smem_u32(sU + (size_t)su * UP_STAGE), &tmU, smem_u32(&u_full[su]), 0, lo2(it.c0(P)), lo2(it.r0(P)), it.n);
        if (++su == L_NU) { su = 0; pu ^= 1; }
        it.step(P.step[0], P);
      }
    }
    __syncwarp();
  } else if (warp == 1 || warp == 2) {
    // =========================== MMA issuers: two elected threads alternate tiles =================
    // (see conv_tc.cu for why two: the issuing thread stalls on its uniform registers until its MMAs have drained)
    const int mw = warp - 1;
    const int nmw = (P.dbg & 16) ? 1 : 2;
    if (mw < nmw && elect_one()) {
      const uint32_t idesc = make_idesc_bf16_m128(L_NP);
      const uint32_t a_hi = desc_hi((LTW + 2) * 64, 4u);          // SBO = one slab row (10 pixels x 64 B), 64 B swizzle
      const uint32_t b_hi = desc_hi(8 * 64, 4u);
      const uint32_t a_lo0 = ((smem_u32(sA) >> 4) & 0x3FFFu) | (1u << 16), b_lo0 = ((smem_u32(sB) >> 4) & 0x3FFFu) | (1u << 16);
      constexpr uint32_t a_stage16 = A_STAGE >> 4, b_tile16 = B_TILE >> 4;
      int sa = 0, pa = 0, ts = 0, tp = 0;
      mbar_wait(b_full, 0);
      tc_fence_after();
      auto skip_tile = [&]() {
        for (int i = 0; i < P.nchunks; ++i) if (++sa == L_SA) { sa = 0; pa ^= 1; }
        if (++ts == L_NST) { ts = 0; tp ^= 1; }
      };
      if (mw == 1) skip_tile();
      for (uint32_t tile = blockIdx.x + (uint32_t)mw * gridDim.x; tile < total; tile += (uint32_t)nmw * gridDim.x) {
        mbar_wait(&t_empty[ts], tp ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ts * L_NP);
        for (int ch = 0; ch < P.nchunks; ++ch) {
          const uint32_t acc_first = ch ? 1u : 0u;
          const uint32_t b_chunk = b_lo0 + (uint32_t)(ch * 9) * b_tile16;
          mbar_wait(&a_full[sa], pa);
          tc_fence_after();
          const uint32_t a_lo = a_lo0 + (uint32_t)sa * a_stage16;
          if (!(P.dbg & 4))
#pragma unroll
          for (int t = 0; t < 9; ++t) {
            const uint32_t b_lo = b_chunk + (uint32_t)t * b_tile16;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const uint32_t al = a_lo + (((uint32_t)((t / 3) * (LTW + 2) + (t % 3)) * 64 + k * 32) >> 4);
              if (t == 0 && k == 0) tc_mma2(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc, acc_first);
              else tc_mma2_acc(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc);
            }
          }
          tc_commit(&a_empty[sa]);
          if (++sa == L_SA) { sa = 0; pa ^= 1; }
        }
        tc_commit(&t_full[ts]);
        if (++ts == L_NST) { ts = 0; tp ^= 1; }
        if (nmw == 2) skip_tile();                         // the other issuer's tile
      }
    }
    __syncwarp();
  } else if (warp >= L_EPI_WARP0) {
    // =========================== epilogue: four groups of four warps ===============================
    const int ew = warp - L_EPI_WARP0, grp = ew >> 2, q = warp & 3;
    const int m = q * 32 + lane, ph = m >> 3, pw = m & 7;        // this thread's pixel of the 16 x 8 tile
    const uint32_t taddr_q = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t bias_u = smem_u32(s_bias), sU_u = smem_u32(sU);
    const uint32_t sX_u = smem_u32(sX) + (uint32_t)grp * 2 * X_TILE;
    const int H = P.H, W = P.W, K = P.K;
    uint32_t ts = (uint32_t)grp, tp = 0, su = (uint32_t)grp, pu = 0, xb = 0;     // L_NST, L_NU multiples of L_GROUPS
    TileIt it; it.init(blockIdx.x + (uint32_t)grp * gridDim.x, P);
    for (uint32_t tile = blockIdx.x + (uint32_t)grp * gridDim.x; tile < total; tile += (uint32_t)L_GROUPS * gridDim.x) {
      const int n = it.n, r0 = it.r0(P), c0 = it.c0(P);
      const int y = r0 + ph, x = c0 + pw;                         // >= 0; may lie beyond the rung in ragged last tiles
      // ---- `up` corner addresses in the patch (index clamps = ATen's border rule) and parity weights
      const int uy0 = lo2(r0), ux0 = lo2(c0);
      // (pixels beyond the rung may clamp outside the patch: keep every read inside it, their values are never consumed)
      const int ya = clampi(clampi(lo2(y), 0, P.up_h - 1) - uy0, 0, UP_H - 1), yb = clampi(clampi(lo2(y) + 1, 0, P.up_h - 1) - uy0, 0, UP_H - 1);
      const int xa = clampi(clampi(lo2(x), 0, P.up_w - 1) - ux0, 0, UP_W - 1), xb_ = clampi(clampi(lo2(x) + 1, 0, P.up_w - 1) - ux0, 0, UP_W - 1);
      const uint32_t ub = sU_u + su * UP_STAGE;
      const uint32_t u00 = ub + (uint32_t)((ya * UP_W + xa) * (L_CH * 2)), u01 = ub + (uint32_t)((ya * UP_W + xb_) * (L_CH * 2));
      const uint32_t u10 = ub + (uint32_t)((yb * UP_W + xa) * (L_CH * 2)), u11 = ub + (uint32_t)((yb * UP_W + xb_) * (L_CH * 2));
      const __half2 hwx0 = __float2half2_rn((x & 1) ? 0.75f : 0.25f), hwx1 = __float2half2_rn((x & 1) ? 0.25f : 0.75f);
      const __half2 hwy0 = __float2half2_rn((y & 1) ? 0.75f : 0.25f), hwy1 = __float2half2_rn((y & 1) ? 0.25f : 0.75f);

      mbar_wait(&t_full[ts], tp);
      tc_fence_after();
      uint32_t v[24];
      tc_ld16(taddr_q + ts * (uint32_t)L_NP, v);
      tc_ld8(taddr_q + ts * (uint32_t)L_NP + 16, v + 16);
      tc_wait_ld();
      // the accumulator stage is free as soon as it is in registers
      tc_fence_before();
      __syncwarp();
      if (lane == 0 && !(P.dbg & 32)) mbar_arrive(&t_empty[ts]);
      mbar_wait(&u_full[su], pu);

      uint4 o[3];                                              // this pixel's rung value, 24 x fp16
#pragma unroll
      for (int g = 0; g < 3; ++g) {
        float f[8];
        const float4 b0 = lds128f(bias_u + 32 * g), b1 = lds128f(bias_u + 32 * g + 16);
        f[0] = fmaxf(__uint_as_float(v[8 * g + 0]) + b0.x, 0.f); f[1] = fmaxf(__uint_as_float(v[8 * g + 1]) + b0.y, 0.f);
        f[2] = fmaxf(__uint_as_float(v[8 * g + 2]) + b0.z, 0.f); f[3] = fmaxf(__uint_as_float(v[8 * g + 3]) + b0.w, 0.f);
        f[4] = fmaxf(__uint_as_float(v[8 * g + 4]) + b1.x, 0.f); f[5] = fmaxf(__uint_as_float(v[8 * g + 5]) + b1.y, 0.f);
        f[6] = fmaxf(__uint_as_float(v[8 * g + 6]) + b1.z, 0.f); f[7] = fmaxf(__uint_as_float(v[8 * g + 7]) + b1.w, 0.f);
        if (P.dbg & 2) { o[g] = make_uint4(pack_f16x2_sat(f[0], f[1]), pack_f16x2_sat(f[2], f[3]), pack_f16x2_sat(f[4], f[5]), pack_f16x2_sat(f[6], f[7])); continue; }
        const uint4 ca = lds128(u00 + 16 * g), cb = lds128(u01 + 16 * g), cc = lds128(u10 + 16 * g), cd = lds128(u11 + 16 * g);
        const __half2* a = reinterpret_cast<const __half2*>(&ca);
        const __half2* b = reinterpret_cast<const __half2*>(&cb);
        const __half2* c = reinterpret_cast<const __half2*>(&cc);
        const __half2* d = reinterpret_cast<const __half2*>(&cd);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          // packed half2 interpolation (the weights are exact; same order as round 1's conv_tc ladder epilogue)
          const __half2 h0 = __hfma2(b[j], hwx1, __hmul2(a[j], hwx0));
          const __half2 h1 = __hfma2(d[j], hwx1, __hmul2(c[j], hwx0));
          const float2 u2 = __half22float2(__hfma2(h1, hwy1, __hmul2(h0, hwy0)));
          f[2 * j] += u2.x; f[2 * j + 1] += u2.y;
        }
        o[g] = make_uint4(pack_f16x2_sat(f[0], f[1]), pack_f16x2_sat(f[2], f[3]), pack_f16x2_sat(f[4], f[5]),
                          pack_f16x2_sat(f[6], f[7]));
      }
      __syncwarp();
      if (lane == 0 && !(P.dbg & 32)) mbar_arrive(&u_empty[su]);   // patch consumed

      if (!FINAL) {
        if (y < H && x < W) {
          __half* op = P.out + (((int64_t)n * H + y) * W + x) * L_CH;
#pragma unroll
          for (int g = 0; g < 3; ++g)
            if (8 * g < K) *reinterpret_cast<uint4*>(op + 8 * g) = o[g];
        }
      } else {
        // ---- exchange the r1 tile inside the group, then the last x2 upsample + argmax
        if ((P.dbg & 8) && P.out && y < H && x < W) {
          __half* op = P.out + (((int64_t)n * H + y) * W + x) * L_CH;
#pragma unroll
          for (int g = 0; g < 3; ++g) *reinterpret_cast<uint4*>(op + 8 * g) = o[g];
        }
        const uint32_t xt = sX_u + xb * X_TILE;
        const uint32_t mine = xt + (uint32_t)m * (L_CH * 2);
        // ---- uniform-corner shortcut.  Every output of the 2 x 2 block between four r1 pixels is a convex combination
        // of them (weights 1/16 .. 9/16), and each lerp is a monotone fp32 operation: when the four pixels share one
        // first-max class k*, every output has v[k*] >= v[k] for all k, strictly for k < k* (the corner gaps are at least
        // one fp16 ulp of the largest magnitude involved, 2^-11 M, times a weight >= 1/16, against <= 6 roundings of
        // 2^-24 M), i.e. the same first-max class.  So each thread takes the arg-max of ITS r1 pixel (K compares instead
        // of 4 K lerped outputs), publishes it in the exchange tile's spare channel 23, and a warp whose 32 blocks are
        // all uniform skips the per-class lerps.  Bit-identical labels; 92 % of the warps on the benchmark input.
        const bool shortcut = K < L_CH && !(P.dbg & 64);
        int amax = 0;
        if (shortcut) {
          float bv = -INFINITY;
#pragma unroll
          for (int g = 0; g < 3; ++g) {
            const __half2* h = reinterpret_cast<const __half2*>(&o[g]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int k = 8 * g + 2 * j;
              const float2 v2 = __half22float2(h[j]);
              if (k < K && v2.x > bv) { bv = v2.x; amax = k; }
              if (k + 1 < K && v2.y > bv) { bv = v2.y; amax = k + 1; }
            }
          }
        }
#pragma unroll
        for (int g = 0; g < 2; ++g) sts128(mine + 16 * g, o[g]);
        sts128(mine + 32, shortcut ? make_uint4(o[2].x, o[2].y, o[2].z, (o[2].w & 0xFFFFu) | ((uint32_t)amax << 16)) : o[2]);
        asm volatile("bar.sync %0, 128;" ::"r"(2 + grp) : "memory");
        // This thread's r1 pixel (y, x) is the TOP-LEFT corner of the outputs it owns: rows 2y+1 (3/4 top, 1/4 bottom)
        // and 2y+2 (1/4, 3/4), columns 2x+1 and 2x+2.  The bottom / right neighbour is clamped at the rung's edge
        // (ATen's index clamp); tile row 15 / column 7 have their neighbour in the NEXT tile and only own outputs
        // when they are the rung's last row / column (neighbour = themselves).
        const bool has_b = y + 1 <= H - 1, has_r = x + 1 <= W - 1;
        const bool act = y <= H - 1 && x <= W - 1 && (ph < LTH - 1 || !has_b) && (pw < LTW - 1 || !has_r);
        const uint32_t pTR = mine + (has_r ? (uint32_t)(L_CH * 2) : 0u);
        const uint32_t pBL = mine + (has_b ? (uint32_t)(LTW * L_CH * 2) : 0u);
        const uint32_t pBR = pBL + (has_r ? (uint32_t)(L_CH * 2) : 0u);
        bool uni = true;
        if (shortcut && act) {
          uint32_t i1, i2, i3;
          asm volatile("ld.shared.u16 %0, [%1];" : "=r"(i1) : "r"(pTR + 46) : "memory");
          asm volatile("ld.shared.u16 %0, [%1];" : "=r"(i2) : "r"(pBL + 46) : "memory");
          asm volatile("ld.shared.u16 %0, [%1];" : "=r"(i3) : "r"(pBR + 46) : "memory");
          uni = (i1 == (uint32_t)amax) & (i2 == (uint32_t)amax) & (i3 == (uint32_t)amax);
        }
        const bool fast = shortcut && __all_sync(0xffffffffu, uni);
        if (act && !(P.dbg & 1)) {
          const float2 q14 = make_float2(0.25f, 0.25f), q34 = make_float2(0.75f, 0.75f);
          float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};       // (Y1,X1) (Y1,X2) (Y2,X1) (Y2,X2)
          int bidx[4] = {amax, amax, amax, amax};
          if (!fast)
#pragma unroll
          for (int g = 0; g < 3; ++g) {
            if (8 * g >= K) break;
            const uint4 tr = lds128(pTR + 16 * g), bl = lds128(pBL + 16 * g), br = lds128(pBR + 16 * g);
            const __half2* htl = reinterpret_cast<const __half2*>(&o[g]);           // own pixel: registers
            const __half2* htr = reinterpret_cast<const __half2*>(&tr);
            const __half2* hbl = reinterpret_cast<const __half2*>(&bl);
            const __half2* hbr = reinterpret_cast<const __half2*>(&br);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int k = 8 * g + 2 * j;
              if (k >= K) break;
              const bool two = k + 1 < K;
              const float2 TL = __half22float2(htl[j]), TR = __half22float2(htr[j]);
              const float2 BL = __half22float2(hbl[j]), BR = __half22float2(hbr[j]);
              // horizontal first, then vertical (tail2_kernel's order)
              const float2 t1 = lerp2(TL, TR, q34, q14), t2 = lerp2(TL, TR, q14, q34);
              const float2 b1 = lerp2(BL, BR, q34, q14), b2 = lerp2(BL, BR, q14, q34);
              const float2 o11 = lerp2(t1, b1, q34, q14), o12 = lerp2(t2, b2, q34, q14);
              const float2 o21 = lerp2(t1, b1, q14, q34), o22 = lerp2(t2, b2, q14, q34);
              if (o11.x > best[0]) { best[0] = o11.x; bidx[0] = k; }
              if (o12.x > best[1]) { best[1] = o12.x; bidx[1] = k; }
              if (o21.x > best[2]) { best[2] = o21.x; bidx[2] = k; }
              if (o22.x > best[3]) { best[3] = o22.x; bidx[3] = k; }
              if (two) {
                if (o11.y > best[0]) { best[0] = o11.y; bidx[0] = k + 1; }
                if (o12.y > best[1]) { best[1] = o12.y; bidx[1] = k + 1; }
                if (o21.y > best[2]) { best[2] = o21.y; bidx[2] = k + 1; }
                if (o22.y > best[3]) { best[3] = o22.y; bidx[3] = k + 1; }
              }
            }
          }
          const int Wo = 2 * W;
          const int64_t base = ((int64_t)n * (2 * H) + (2 * y + 1)) * Wo + (2 * x + 1);
          if (P.pred_i64) {
            int64_t* pr = reinterpret_cast<int64_t*>(P.pred);
            pr[base] = bidx[0];
            if (has_r) pr[base + 1] = bidx[1];
            if (has_b) pr[base + Wo] = bidx[2];
            if (has_b && has_r) pr[base + Wo + 1] = bidx[3];
          } else {
            uint8_t* pr = reinterpret_cast<uint8_t*>(P.pred);
            pr[base] = (uint8_t)bidx[0];
            if (has_r) pr[base + 1] = (uint8_t)bidx[1];
            if (has_b) pr[base + Wo] = (uint8_t)bidx[2];
            if (has_b && has_r) pr[base + Wo + 1] = (uint8_t)bidx[3];
          }
          if (y == 0 || x == 0) {
            // ---- output row 0 / column 0: the source index is clamped there, so they interpolate along the edge only
            //      (fma(v, 3/4, v/4) == v exactly).  e0 = (0,0), e1 = (0,2x+1), e2 = (0,2x+2), e3 = (2y+1,0), e4 = (2y+2,0)
            float eb[5] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY, -INFINITY};
            int ei[5] = {amax, amax, amax, amax, amax};
            if (!fast)
            for (int g = 0; g < 3; ++g) {
              if (8 * g >= K) break;
              const uint4 tl = lds128(mine + 16 * g), tr = lds128(pTR + 16 * g), bl = lds128(pBL + 16 * g);
              const __half2* htl = reinterpret_cast<const __half2*>(&tl);
              const __half2* htr = reinterpret_cast<const __half2*>(&tr);
              const __half2* hbl = reinterpret_cast<const __half2*>(&bl);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int k = 8 * g + 2 * j;
                if (k >= K) break;
                const bool two = k + 1 < K;
                const float2 TL = __half22float2(htl[j]), TR = __half22float2(htr[j]), BL = __half22float2(hbl[j]);
                const float2 e[5] = {TL, lerp2(TL, TR, q34, q14), lerp2(TL, TR, q14, q34), lerp2(TL, BL, q34, q14),
                                     lerp2(TL, BL, q14, q34)};
#pragma unroll
                for (int c = 0; c < 5; ++c) {
                  if (e[c].x > eb[c]) { eb[c] = e[c].x; ei[c] = k; }
                  if (two && e[c].y > eb[c]) { eb[c] = e[c].y; ei[c] = k + 1; }
                }
              }
            }
            const int64_t row0 = ((int64_t)n * (2 * H)) * Wo, r1o = row0 + (int64_t)(2 * y + 1) * Wo;
            auto put = [&](int64_t off, int v) {
              if (P.pred_i64) reinterpret_cast<int64_t*>(P.pred)[off] = v; else reinterpret_cast<uint8_t*>(P.pred)[off] = (uint8_t)v;
            };
            if (y == 0 && x == 0) put(row0, ei[0]);
            if (y == 0) { put(row0 + 2 * x + 1, ei[1]); if (has_r) put(row0 + 2 * x + 2, ei[2]); }
            if (x == 0) { put(r1o, ei[3]); if (has_b) put(r1o + Wo, ei[4]); }
          }
        }
        xb ^= 1;
      }
      if (P.dbg & 32) { __syncwarp(); if (lane == 0) { mbar_arrive(&t_empty[ts]); mbar_arrive(&u_empty[su]); } }
      ts += L_GROUPS; if (ts >= (uint32_t)L_NST) { ts -= L_NST; tp ^= 1; }
      su += L_GROUPS; if (su >= (uint32_t)L_NU) { su -= L_NU; pu ^= 1; }
      it.step(P.step[2], P);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, L_NST * L_NP);
  }
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn get_encode() {
  static EncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  });
  return fn;
}
int encode(CUtensorMap* m, CUtensorMapDataType dt, const void* base, int rank, const uint64_t* dims,
           const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle sw) {
  EncodeFn fn = get_encode();
  if (!fn) return fail(LEDB200_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t d[5], s[4];
  cuuint32_t b[5], es[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) s[i] = strides_bytes[i];
  CUresult r = fn(m, dt, (cuuint32_t)rank, const_cast<void*>(base), d, s, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LEDB200_ECUDA, "ladder: cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
  return LEDB200_OK;
}

}  // namespace

bool ladder_eligible(const LadderArgs& a) {
  if (!a.in || !a.up || !a.w_tc) return false;
  if (a.Cin != 32 && a.Cin != 64) return false;                 // 32-channel K blocks, weights resident
  if (a.in_ld % 8 || a.in_ld < a.Cin) return false;
  if (a.K < 1 || a.K > L_CH || a.cout_pad_tc != L_NP) return false;
  if (a.up_ld != L_CH || a.H != 2 * a.up_h || a.W != 2 * a.up_w) return false;
  if (((uintptr_t)a.in | (uintptr_t)a.up | (uintptr_t)a.w_tc) & 15) return false;
  if (a.final_argmax) { if (!a.pred) return false; }
  else if (!a.out || a.out_ld != L_CH || ((uintptr_t)a.out & 15)) return false;
  if ((int64_t)a.N * (ceil_div(a.H, 15) + 1) * (ceil_div(a.W, 7) + 1) >= (1ll << 29)) return false;
  return true;
}

int launch_ladder(const LadderArgs& a, cudaStream_t st) {
  if (!ladder_eligible(a)) return fail(LEDB200_EINVAL, "ladder: shape not eligible");
  LadderParams P{};
  P.N = a.N; P.H = a.H; P.W = a.W; P.Cin = a.Cin; P.nchunks = a.Cin / 32; P.K = a.K;
  P.up_h = a.up_h; P.up_w = a.up_w; P.bias = a.bias;
  P.out = (__half*)a.out; P.pred = a.pred; P.pred_i64 = a.pred_i64;
  { const char* e = getenv("LEDB200_LADDER_DBG"); P.dbg = e ? atoi(e) : 0; }
  if (a.final_argmax) {
    // overlapping tiles: tile row i and i+1 produce output rows 2i+1, 2i+2, so a tile of 16 rung rows advances by 15
    // (the rung's last row needs no lower neighbour: it may sit in tile row 15); the last tile is shifted back to end
    // at the edge
    P.th_step = LTH - 1; P.tw_step = LTW - 1;
    P.tiles_h = std::max(1, ceil_div(a.H - 1, LTH - 1)); P.tiles_w = std::max(1, ceil_div(a.W - 1, LTW - 1));
    P.r_max = std::max(0, a.H - LTH); P.c_max = std::max(0, a.W - LTW);
  } else {
    P.th_step = LTH; P.tw_step = LTW;
    P.tiles_h = ceil_div(a.H, LTH); P.tiles_w = ceil_div(a.W, LTW);
    P.r_max = P.c_max = 1 << 30;
  }
  P.total_tiles = (uint32_t)((int64_t)a.N * P.tiles_h * P.tiles_w);
  CUtensorMap tmA, tmB, tmU;
  int rc;
  {
    const uint64_t ld = (uint64_t)a.in_ld;
    const uint64_t dims[4] = {(uint64_t)a.Cin, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.N};
    const uint64_t str[3] = {ld * 2, (uint64_t)a.W * ld * 2, (uint64_t)a.H * a.W * ld * 2};
    const uint32_t box[4] = {32, LTW + 2, LTH + 2, 1};
    if ((rc = encode(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, a.in, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B))) return rc;
  }
  {
    const uint64_t dims[2] = {(uint64_t)9 * a.Cin, (uint64_t)L_NP};
    const uint64_t str[1] = {(uint64_t)9 * a.Cin * 2};
    const uint32_t box[2] = {32, L_NP};
    if ((rc = encode(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, a.w_tc, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B))) return rc;
  }
  {
    const uint64_t dims[4] = {(uint64_t)L_CH, (uint64_t)a.up_w, (uint64_t)a.up_h, (uint64_t)a.N};
    const uint64_t str[3] = {(uint64_t)L_CH * 2, (uint64_t)a.up_w * L_CH * 2, (uint64_t)a.up_h * a.up_w * L_CH * 2};
    const uint32_t box[4] = {L_CH, UP_W, UP_H, 1};
    if ((rc = encode(&tmU, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, a.up, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_NONE))) return rc;
  }
  const size_t smem = 1024 + (size_t)L_SA * A_STAGE + (size_t)P.nchunks * 9 * B_TILE + (size_t)L_NU * UP_STAGE +
                      (a.final_argmax ? (size_t)L_GROUPS * 2 * X_TILE : 0) + L_NP * 4 + (2 * L_SA + 2 * L_NU + 2 * L_NST + 1) * 8 + 16;
  static std::once_flag attr_once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once, [] {
    cudaError_t e = cudaFuncSetAttribute(ladder_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
    if (e != cudaSuccess) attr_err = e;
    e = cudaFuncSetAttribute(ladder_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
    if (e != cudaSuccess) attr_err = e;
  });
  if (attr_err != cudaSuccess) return fail(LEDB200_ECUDA, std::string("ladder: cudaFuncSetAttribute: ") + cudaGetErrorString(attr_err));
  static int sms = 0;
  if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
  const int grid = (int)std::min<uint32_t>(P.total_tiles, (uint32_t)sms);
  for (int k = 0; k < 3; ++k) {
    uint32_t stp = (uint32_t)grid << k;
    P.step[k][0] = (int)(stp % (uint32_t)P.tiles_w); stp /= (uint32_t)P.tiles_w;
    P.step[k][1] = (int)(stp % (uint32_t)P.tiles_h);
    P.step[k][2] = (int)(stp / (uint32_t)P.tiles_h);
  }
  if (a.final_argmax) ladder_kernel<true><<<grid, L_THREADS, smem, st>>>(tmA, tmB, tmU, P);
  else ladder_kernel<false><<<grid, L_THREADS, smem, st>>>(tmA, tmB, tmU, P);
  LEDB_LAUNCH_OK("ladder_kernel");
  return LEDB200_OK;
}

}  // namespace ledb
