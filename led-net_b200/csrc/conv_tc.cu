// Implicit-GEMM convolution on the 5th-gen tensor cores (north_star kernel 1).
//
// Replaces mmcv ConvModule = Conv2d(3x3 pad 1 | 1x1, stride 1 | 2) + folded BatchNorm (+ReLU)
// (+ residual add of BasicBlock/Bottleneck.forward) for every dense layer of the trunk and head:
//   mmseg/models/utils/basic_block.py:43-75, 186-221, mmseg/models/backbones/ddrnet.py:68-105,
//   mmseg/models/utils/ppm.py:57-117, mmseg/models/decode_heads/led_head.py:84-99,
//   mmseg/models/decode_heads/decode_head.py:241-246 (cls_seg).
//
// GEMM view: D[M = 128 output pixels (TH x TW tile)][N = Cout] += A[M][K] * B[N][K]^T with
// K = taps * Cin walked as (Cin chunk of KC channels) x (filter tap).
//   A  NHWC bf16 activations.  TMA (cp.async.bulk.tensor, tiled mode, hardware zero fill for the
//      conv padding) stages, per Cin chunk, one "slab" per filter column: (TH+2) x TW pixels x KC
//      channels, 128B- (KC=64) or 64B-swizzled (KC=32).  The three filter rows of that column are
//      three row-shifted windows of the same slab: the UMMA shared-memory descriptor just starts
//      TW*kh pixels later, so the input is fetched 3x (not 9x) from L2 and never re-laid out.
//      Stride 2 uses a 5-D view [N][H/2][2][W/2][2*C] of the same tensor (row/column parity
//      split), which turns the strided taps back into dense boxes.
//   B  folded weights bf16 [CoutPad][taps*Cin] (K-major), TMA 2-D boxes of NT x KC; kept resident in
//      shared memory for the whole persistent CTA when they fit, else streamed through a ring.
//   D  fp32 accumulators in TMEM (tcgen05.mma cta_group::1, M=128, N=NT<=256), double buffered so
//      the epilogue of tile i overlaps the MMAs of tile i+1.
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + single-thread MMA issuer,
// warps 2-5 = epilogue (tcgen05.ld 32x32b -> +bias (+residual) -> ReLU -> bf16 -> 16 B stores; an
// optional second output relu(s*v+b) feeds the next layer's pre-activation BN+ReLU).
// Persistent grid of min(tiles, #SM) CTAs, static round-robin tile schedule.
#include <cuda.h>

#include <map>
#include <mutex>
#include <tuple>
#include <type_traits>
#include <vector>
#include <cstdlib>

#include "tc_common.cuh"

namespace ledb {
namespace {

constexpr int kThreads = 352;            // TMA warp, MMA warp, 2 x 4 epilogue warps, second MMA issuer (warp 10)
constexpr int TH = 16, TW = 8;            // output tile: 16 rows x 8 cols = 128 pixels = UMMA M
constexpr int MAX_SLABS = 6, MAX_TAPS = 9;
constexpr uint32_t SMEM_BUDGET = 220 * 1024;

struct Slab {
  int c_mul;      // channel offset multiplier (stride 2: column parity -> + c_mul * ld)
  int dw, dh;     // box origin offsets (in units of the tensor-map W / H dims)
  int ph;         // stride 2: row parity coordinate
  int ntaps;
  int tap_pix[MAX_TAPS];   // first pixel of the tap's window inside the slab
  int tap_id[MAX_TAPS];    // filter tap index kh*3+kw (weight column block)
};

struct TcParams {
  Slab slabs[MAX_SLABS];
  int nslabs;
  int Cin, Cout, NT, ntiles_n;       // NT = N tile (<=256, multiple of 16)
  int ntaps_total;                   // ksize * ksize
  int KC, nchunks;                   // channels per k-block, Cin / KC
  int N, Ho, Wo, tiles_h, tiles_w;
  int64_t total_tiles;
  int in_ld;                         // pixel stride of the input (elements)
  int sbo_bytes;                     // stride between 8-row groups of the A window
  uint32_t a_stage_bytes, b_tile_bytes;   // padded to 1024 B (ring strides)
  uint32_t a_box_bytes, b_box_bytes;      // bytes one TMA box actually writes (expect_tx)
  int SA, SB, b_resident;
  int cp;                            // Cout padded to the N tiling (ntiles_n * NT)
  uint32_t stage_bytes;              // epilogue staging: 32 KB (+32 KB with a second output)
  int step1[4], step2[4];            // grid and 2*grid tiles as digits (n-tile, tile col, tile row, image)
  uint32_t tmem_cols;
  int nst;                           // accumulator stages in TMEM: 4 when 4*NT <= 512 columns, else 2
  int nmw;                           // MMA issuer threads: 2 when weights are resident and the A ring allows it
  // epilogue
  __nv_bfloat16* out; int out_ld;
  __nv_bfloat16* out2; int out2_ld;
  const float* o2_scale; const float* o2_shift;
  const __nv_bfloat16* res; int res_ld;
  const float* bias;
  int relu;
  int out_f16;                       // `out` holds IEEE fp16 (conv_seg's x_c, the bottom rung of the head ladder)
  int fast_epi;                      // interior tiles take the epilogue fast path (decided once per launch, launch_conv_tc)
  // TF32 epilogue only: output pixel (oy, ox) of image n lands at ((n * o_H + oy * o_mul + o_a) * o_W + ox * o_mul + o_b):
  // o_mul = 2 writes one parity class of a twice-as-large tensor (data gradient of a stride-2 convolution)
  int o_mul, o_a, o_b, o_H, o_W;
  // three-pass mode: the two correction passes (x_hi*w_lo, x_lo*w_hi) accumulate into their OWN TMEM columns, lo_off columns
  // after the main accumulator of the same stage, and the epilogue adds the two.  The tensor core's accumulator truncates at
  // the magnitude of the running sum; small addends kept apart lose nothing to it (measured: 2e-5 -> 7e-6 at K = 2304).
  int lo_off;
  // three-pass 3x3 stride-1 launches: kacc = 3 main accumulators, one per filter ROW, added by the epilogue.  The tensor
  // core's accumulator truncates at every accumulation step, so the error of a long reduction grows with its length (measured
  // 8.6e-7 at K = 9 x 32, 6.8e-6 at K = 9 x 256 with one accumulator); three chains of a third of the length cut it.
  // Accumulator j of stage ts lives at column j * acc_plane + ts * NT (j = kacc is the correction accumulator: lo_off).
  int kacc, acc_plane;
  int tl_launch;                     // launch ordinal (timeline probe builds only: slot of g_tc_tl)
  int dbg;                           // LEDB200_TC_DBG probe bits: 1 no global stores, 2 no MMAs, 4 no A TMA, 8 no residual loads, 32 atom-aligned A row groups, 64 empty epilogue, 128 single MMA issuer
};

using namespace tc;   // PTX wrappers: tc_common.cuh

// Timeline probe (tools/probes/tc_timeline.sh builds a second library with -DLEDB_TC_TIMELINE; the product build
// compiles none of it): CTA 0 of every launch stamps clock64 at the points of its ramp into slot `tl_launch`.
#ifdef LEDB_TC_TIMELINE
__device__ unsigned long long g_tc_tl[128][16];
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t;
}
#define TL(slot, cond) do { if (blockIdx.x == 0 && (cond)) g_tc_tl[P.tl_launch & 127][slot] = clock64(); } while (0)
#define TLG(slot, cond) do { if (blockIdx.x == 0 && (cond)) g_tc_tl[P.tl_launch & 127][slot] = gtimer(); } while (0)
#else
#define TL(slot, cond) do {} while (0)
#define TLG(slot, cond) do {} while (0)
#endif

__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
// 256-bit global accesses (sm_100): one full 32 B sector per thread and instruction
__device__ __forceinline__ void ldg256(const void* p, uint4& a, uint4& b) {
  asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}
__device__ __forceinline__ void stg256(void* p, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}
__device__ __forceinline__ float4 lds128f(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

// Epilogue of the persistent conv kernel, run by warps 2..9 as two groups of four.
//   N tile >= 64: both groups work on EVERY tile, group g drains column half g of the accumulator (all
//     128 lanes), so a tile's epilogue takes half as long and the epilogue warps never idle waiting for
//     "their" accumulator stage while the MMAs of the next tile run into the other TMEM stage;
//   N tile < 64: group g owns accumulator stage g and every second tile (per-tile fixed costs dominate).
// Per tile and block of up to 32 columns:
//   tcgen05.ld (thread = output pixel) -> +bias (+residual) -> ReLU -> bf16 -> warp-private XOR-swizzled
//   staging (up to 64 channels x 32 pixels) -> 16 B global stores with consecutive lanes on consecutive
//   addresses (full 32 B sectors; 8 lanes cover one 128 B pixel row of a 64-channel slice).
// The second output relu(s*y + b) (pre-activation BN+ReLU of the consumer) goes through its own
// staging tile.  Templated on which tensors exist so the hot loop has no per-element branches; ReLU is
// a max against 0 or -inf.
template <bool HAS_RES, bool HAS_OUT, bool HAS_OUT2>
__device__ __forceinline__ void epilogue_loop(const TcParams& P, int warp, int lane, uint32_t tmem_base,
                                              uint64_t* t_full, uint64_t* t_empty, uint32_t st_u, uint32_t bias_u,
                                              uint32_t o2s_u, uint32_t o2b_u) {
  const int ew = warp - 2;                      // 0..7
  const int grp = ew >> 2;                      // column half of every accumulator
  const int q = warp & 3;                       // TMEM lane quadrant this warp may access
  const int m = q * 32 + lane;                  // tile row = output pixel within the tile
  const int ph = m >> 3, pw = m & 7;            // TW == 8
  const uint32_t st1 = st_u + (uint32_t)ew * 4096, st2 = st_u + 32768 + (uint32_t)ew * 4096;
  const int NT = P.NT, Ho = P.Ho, Wo = P.Wo;
  const int cout8 = (P.Cout + 7) & ~7;          // stores cover whole 8-channel groups (buffers are padded)
  const float relu_lo = P.relu ? 0.f : -INFINITY;
  const uint32_t taddr_q = tmem_base + ((uint32_t)(q * 32) << 16);
  const bool split = NT >= 64;                  // split columns between the groups, else alternate tiles
  const int ncols_g = split ? NT / 2 : NT;
  const int cbeg = split ? grp * ncols_g : 0, cend = cbeg + ncols_g;
  // staging slice geometry (constant per launch: ncols_g is 16, 32, 64 or a multiple of 64)
  const int slice_cols = max(16, min(64, ncols_g));
  const int sh = 31 - __clz(slice_cols * 2);    // log2(bytes per staged pixel): 5, 6 or 7
  const int ppi = 512 >> sh;                    // pixels covered by one warp-wide 16 B store
  const int niter = slice_cols >> 3;            // stores per slice = 32 px * slice bytes / 512
  const int pl = lane >> (sh - 4);              // pixel of this lane inside a store
  const int cl = (lane & ((1 << (sh - 4)) - 1)) * 8;   // channel of this lane inside the slice
  const uint32_t row_off = (uint32_t)lane << sh;
  uint32_t tp = 0, ts = split ? 0u : (uint32_t)grp;
  // tile coordinates, advanced incrementally by the tile step (mixed-radix digits from the host)
  const uint32_t first = blockIdx.x + (split ? 0u : (uint32_t)grp * gridDim.x);
  const int* stepd = split ? P.step1 : P.step2;
  uint32_t t0 = first;
  int nt = (int)(t0 % (uint32_t)P.ntiles_n); t0 /= (uint32_t)P.ntiles_n;
  int tw = (int)(t0 % (uint32_t)P.tiles_w); t0 /= (uint32_t)P.tiles_w;
  int th = (int)(t0 % (uint32_t)P.tiles_h);
  int n = (int)(t0 / (uint32_t)P.tiles_h);
  const uint32_t total = (uint32_t)P.total_tiles, step = split ? gridDim.x : 2 * gridDim.x;
  // ---- fast path: interior tiles, 32-column blocks, registers -> global directly.
  // Measured on B200 (profiles/r1c_notes.md): with N tile <= 64 every tcgen05.mma re-reads its 4 KB A window
  // from shared memory (6 KB per MMA at 128 B/clk = 48 clk against a 32 clk tensor floor), so the 3x3 layers
  // are bound by the shared-memory port; the staged epilogue of the generic path below adds another
  // 32-64 KB of st.shared/ld.shared per tile on the same port plus ~520 instructions per warp.  Here each
  // thread owns one output pixel: 32 channels = 64 contiguous bytes = two 256-bit stores (full 32 B sectors),
  // the residual comes in as two 256-bit loads issued before the accumulator wait, and nothing touches shared
  // memory except the bias broadcast.
  const int lane_px = ph * Wo + pw;                                         // this thread's pixel inside the tile
  for (uint32_t tile = first; tile < total; tile += step) {
    if (P.fast_epi && th * TH + TH <= Ho && tw * TW + TW <= Wo) {
      const int64_t pix = ((int64_t)n * Ho + th * TH) * Wo + tw * TW + lane_px;
      const int cgt = nt * NT;
      const __nv_bfloat16* res_px = HAS_RES ? P.res + pix * P.res_ld + cgt : nullptr;
      __nv_bfloat16* out_px = HAS_OUT ? P.out + pix * P.out_ld + cgt : nullptr;
      __nv_bfloat16* out2_px = HAS_OUT2 ? P.out2 + pix * P.out2_ld + cgt : nullptr;
      uint4 rr[HAS_RES ? 4 : 1];
      if (HAS_RES) { ldg256(res_px + cbeg, rr[0], rr[1]); ldg256(res_px + cbeg + 16, rr[2], rr[3]); }
      if (HAS_RES && tile + step < total) {
        // L1 prefetch of the residual row the NEXT tile of this warp will read: the residual epilogue is bound by
        // that L2 latency (probe r1c: 52 us with the MMAs off against 29 us without a residual), and a register
        // prefetch does not fit under the 168-register cap (tried: slower)
        int nt2 = nt + stepd[0], tw2 = tw, th2 = th, n2 = n;
        if (nt2 >= P.ntiles_n) { nt2 -= P.ntiles_n; ++tw2; }
        tw2 += stepd[1]; if (tw2 >= P.tiles_w) { tw2 -= P.tiles_w; ++th2; }
        th2 += stepd[2]; if (th2 >= P.tiles_h) { th2 -= P.tiles_h; ++n2; }
        n2 += stepd[3];
        if (th2 * TH + TH <= Ho && tw2 * TW + TW <= Wo) {
          const __nv_bfloat16* rn = P.res + (((int64_t)n2 * Ho + th2 * TH) * Wo + tw2 * TW + lane_px) * P.res_ld + nt2 * NT + cbeg;
          prefetch_l1(rn);
          if (ncols_g > 64) prefetch_l1(rn + 64);
        }
      }
      mbar_wait(&t_full[ts], tp);
      tc_fence_after();
      TL(7, tile == blockIdx.x && warp == 2 && lane == 0);
      const uint32_t taddr0 = taddr_q + ts * (uint32_t)NT;
      for (int c0 = (P.dbg & 64) ? cend : cbeg; c0 < cend; c0 += 32) {     // probe bit 64: epilogue only hands the stage back
        uint32_t v[32];
        tc_ld16(taddr0 + c0, v);
        tc_ld16(taddr0 + c0 + 16, v + 16);
        tc_wait_ld();
        const uint32_t bias_b = bias_u + (uint32_t)(cgt + c0) * 4;
        uint4 o[4], o2[HAS_OUT2 ? 4 : 1];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float f[8];
          const float4 b0 = lds128f(bias_b + 32 * g);
          const float4 b1 = lds128f(bias_b + 32 * g + 16);
          f[0] = __uint_as_float(v[8 * g + 0]) + b0.x; f[1] = __uint_as_float(v[8 * g + 1]) + b0.y;
          f[2] = __uint_as_float(v[8 * g + 2]) + b0.z; f[3] = __uint_as_float(v[8 * g + 3]) + b0.w;
          f[4] = __uint_as_float(v[8 * g + 4]) + b1.x; f[5] = __uint_as_float(v[8 * g + 5]) + b1.y;
          f[6] = __uint_as_float(v[8 * g + 6]) + b1.z; f[7] = __uint_as_float(v[8 * g + 7]) + b1.w;
          if (HAS_RES) {
            float t[8];
            unpack8(rr[g], t);
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] += t[j];
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], relu_lo);
          if (P.out_f16) {                             // cvt.rn.satfinite: saturates at +-65504, never inf
            o[g] = make_uint4(pack_f16x2_sat(f[0], f[1]), pack_f16x2_sat(f[2], f[3]), pack_f16x2_sat(f[4], f[5]),
                              pack_f16x2_sat(f[6], f[7]));
          } else if (HAS_OUT) {
            o[g] = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
          }
          if (HAS_OUT2) {
            const uint32_t q2 = (uint32_t)(cgt + c0) * 4 + 32 * g;
            const float4 s0 = lds128f(o2s_u + q2), s1 = lds128f(o2s_u + q2 + 16);
            const float4 h0 = lds128f(o2b_u + q2), h1 = lds128f(o2b_u + q2 + 16);
            o2[g] = make_uint4(
                pack_bf16x2(fmaxf(fmaf(f[0], s0.x, h0.x), 0.f), fmaxf(fmaf(f[1], s0.y, h0.y), 0.f)),
                pack_bf16x2(fmaxf(fmaf(f[2], s0.z, h0.z), 0.f), fmaxf(fmaf(f[3], s0.w, h0.w), 0.f)),
                pack_bf16x2(fmaxf(fmaf(f[4], s1.x, h1.x), 0.f), fmaxf(fmaf(f[5], s1.y, h1.y), 0.f)),
                pack_bf16x2(fmaxf(fmaf(f[6], s1.z, h1.z), 0.f), fmaxf(fmaf(f[7], s1.w, h1.w), 0.f)));
          }
        }
        if (HAS_RES && c0 + 32 < cend) { ldg256(res_px + c0 + 32, rr[0], rr[1]); ldg256(res_px + c0 + 48, rr[2], rr[3]); }
        if (!(P.dbg & 1)) {
          if (HAS_OUT) { stg256(out_px + c0, o[0], o[1]); stg256(out_px + c0 + 16, o[2], o[3]); }
          if (HAS_OUT2) { stg256(out2_px + c0, o2[0], o2[1]); stg256(out2_px + c0 + 16, o2[2], o2[3]); }
        }
      }
    } else {
    if (P.stage_bytes == 0) __trap();            // host promised an all-interior fast-path launch
    const bool pvalid = (th * TH + ph < Ho) && (tw * TW + pw < Wo);
    const int64_t pix0 = ((int64_t)n * Ho + th * TH) * Wo + tw * TW;       // first pixel of the tile
    const int cgt = nt * NT;                                               // first output channel of this N tile
    const __nv_bfloat16* res_px = HAS_RES ? P.res + (pix0 + ph * Wo + pw) * P.res_ld + cgt : nullptr;
    __nv_bfloat16* out_t = HAS_OUT ? P.out + pix0 * P.out_ld + cgt : nullptr;
    __nv_bfloat16* out2_t = HAS_OUT2 ? P.out2 + pix0 * P.out2_ld + cgt : nullptr;
    const int rows_ok = Ho - th * TH - q * 4, cols_ok = Wo - tw * TW;      // valid rows (of this warp's 4) / cols
    // residual prefetch for one 32-column block; issued BEFORE the accumulator wait for the first block and
    // one block ahead afterwards, so the L2 latency hides behind the MMAs
    uint4 rr[4];
    bool rv[4];
    auto prefetch = [&](int c0) {
      const int ncol = min(32, cend - c0);
      if (HAS_RES) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          rv[g] = pvalid && (8 * g < ncol) && (cgt + c0 + 8 * g < cout8) && !(P.dbg & 8);
          if (rv[g]) rr[g] = __ldg(reinterpret_cast<const uint4*>(res_px + c0 + 8 * g));
        }
      }
    };
    prefetch(cbeg);
    mbar_wait(&t_full[ts], tp);
    tc_fence_after();
    TL(7, tile == blockIdx.x && warp == 2 && lane == 0);
    const uint32_t taddr0 = taddr_q + ts * (uint32_t)NT;
    for (int c0 = cbeg; c0 < cend; c0 += 32) {
      const int ncol = min(32, cend - c0);       // 16 or 32
      uint32_t v[32];
      tc_ld16(taddr0 + c0, v);
      if (ncol == 32) tc_ld16(taddr0 + c0 + 16, v + 16);
      tc_wait_ld();
      const int slice_c = (c0 - cbeg) & 63;      // column of this block inside the staging slice
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        if (8 * g < ncol) {
          float f[8];
          const float4 b0 = lds128f(bias_u + (uint32_t)(cgt + c0 + 8 * g) * 4);
          const float4 b1 = lds128f(bias_u + (uint32_t)(cgt + c0 + 8 * g + 4) * 4);
          f[0] = __uint_as_float(v[8 * g + 0]) + b0.x; f[1] = __uint_as_float(v[8 * g + 1]) + b0.y;
          f[2] = __uint_as_float(v[8 * g + 2]) + b0.z; f[3] = __uint_as_float(v[8 * g + 3]) + b0.w;
          f[4] = __uint_as_float(v[8 * g + 4]) + b1.x; f[5] = __uint_as_float(v[8 * g + 5]) + b1.y;
          f[6] = __uint_as_float(v[8 * g + 6]) + b1.z; f[7] = __uint_as_float(v[8 * g + 7]) + b1.w;
          if (HAS_RES) {
            if (rv[g]) {
              float t[8];
              unpack8(rr[g], t);
#pragma unroll
              for (int j = 0; j < 8; ++j) f[j] += t[j];
            }
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], relu_lo);
          if (P.relu == 2) {                          // ReLU6 (GETB Mlp): generic path only
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] = fminf(f[j], 6.f);
          }
          const uint32_t so = swz(row_off + (uint32_t)(slice_c + 8 * g) * 2);
          if (P.out_f16) {
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] = fminf(fmaxf(f[j], -65504.f), 65504.f);   // saturate, never inf
            sts128(st1 + so, pack_f16x2(f[0], f[1]), pack_f16x2(f[2], f[3]), pack_f16x2(f[4], f[5]), pack_f16x2(f[6], f[7]));
          } else if (HAS_OUT)
            sts128(st1 + so, pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
          if (HAS_OUT2) {
            const float4 s0 = lds128f(o2s_u + (uint32_t)(cgt + c0 + 8 * g) * 4);
            const float4 s1 = lds128f(o2s_u + (uint32_t)(cgt + c0 + 8 * g + 4) * 4);
            const float4 h0 = lds128f(o2b_u + (uint32_t)(cgt + c0 + 8 * g) * 4);
            const float4 h1 = lds128f(o2b_u + (uint32_t)(cgt + c0 + 8 * g + 4) * 4);
            sts128(st2 + so,
                   pack_bf16x2(fmaxf(fmaf(f[0], s0.x, h0.x), 0.f), fmaxf(fmaf(f[1], s0.y, h0.y), 0.f)),
                   pack_bf16x2(fmaxf(fmaf(f[2], s0.z, h0.z), 0.f), fmaxf(fmaf(f[3], s0.w, h0.w), 0.f)),
                   pack_bf16x2(fmaxf(fmaf(f[4], s1.x, h1.x), 0.f), fmaxf(fmaf(f[5], s1.y, h1.y), 0.f)),
                   pack_bf16x2(fmaxf(fmaf(f[6], s1.z, h1.z), 0.f), fmaxf(fmaf(f[7], s1.w, h1.w), 0.f)));
          }
        }
      }
      if (HAS_RES && c0 + 32 < cend) prefetch(c0 + 32);
      // ---- flush a completed staging slice with coalesced stores
      if (slice_c + ncol == slice_cols) {
        __syncwarp();
        const int c = c0 - slice_c + cl;                       // this lane's channel inside the N tile
        const bool c_ok = (cgt + c < cout8) && !(P.dbg & 1);
#pragma unroll 4
        for (int i = 0; i < niter; ++i) {
          const int p = i * ppi + pl;                          // staged pixel 0..31
          const int prow = p >> 3, pcol = p & 7;
          if (c_ok && prow < rows_ok && pcol < cols_ok) {
            const uint32_t so = swz((uint32_t)i * 512 + (uint32_t)lane * 16);
            const int po = (q * 4 + prow) * Wo + pcol;
            if (HAS_OUT) *reinterpret_cast<uint4*>(out_t + (int64_t)po * P.out_ld + c) = lds128(st1 + so);
            if (HAS_OUT2) *reinterpret_cast<uint4*>(out2_t + (int64_t)po * P.out2_ld + c) = lds128(st2 + so);
          }
        }
        __syncwarp();
      }
    }
    }   // generic (edge-tile) body
    TL(8, tile == blockIdx.x && warp == 2 && lane == 0);
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&t_empty[ts]);
    ts += split ? 1u : 2u;
    if (ts >= (uint32_t)P.nst) { ts -= (uint32_t)P.nst; tp ^= 1; }
    // advance the tile coordinates by the tile step
    nt += stepd[0]; if (nt >= P.ntiles_n) { nt -= P.ntiles_n; ++tw; }
    tw += stepd[1]; if (tw >= P.tiles_w) { tw -= P.tiles_w; ++th; }
    th += stepd[2]; if (th >= P.tiles_h) { th -= P.tiles_h; ++n; }
    n += stepd[3];
  }
}

// Epilogue of the TF32 instantiations (training: forward and data-gradient convolutions on fp32 NHWC tensors, train.cu):
// the raw convolution (+ bias) goes out as fp32 - BatchNorm's batch statistics need the un-normalised values, so nothing
// else is fused here.  Same work split as epilogue_loop; the host only launches all-interior tilings, thread = output pixel,
// 32 channels = 128 contiguous bytes = four 256-bit stores.
__device__ __forceinline__ void epilogue_f32(const TcParams& P, int warp, int lane, uint32_t tmem_base,
                                             uint64_t* t_full, uint64_t* t_empty, uint32_t bias_u) {
  const int ew = warp - 2, grp = ew >> 2, q = warp & 3;
  const int m = q * 32 + lane, ph = m >> 3, pw = m & 7;
  const int NT = P.NT, Ho = P.Ho, Wo = P.Wo, Cout = P.Cout;
  const float relu_lo = P.relu ? 0.f : -INFINITY;
  const uint32_t taddr_q = tmem_base + ((uint32_t)(q * 32) << 16);
  const bool split = NT >= 64;
  const int ncols_g = split ? NT / 2 : NT;
  const int cbeg = split ? grp * ncols_g : 0, cend = cbeg + ncols_g;
  float* const outp = reinterpret_cast<float*>(P.out);
  const bool vec_ok = (P.out_ld % 8 == 0) && ((uintptr_t)outp % 32 == 0);
  uint32_t tp = 0, ts = split ? 0u : (uint32_t)grp;
  const uint32_t first = blockIdx.x + (split ? 0u : (uint32_t)grp * gridDim.x);
  const int* stepd = split ? P.step1 : P.step2;
  uint32_t t0 = first;
  int nt = (int)(t0 % (uint32_t)P.ntiles_n); t0 /= (uint32_t)P.ntiles_n;
  int tw = (int)(t0 % (uint32_t)P.tiles_w); t0 /= (uint32_t)P.tiles_w;
  int th = (int)(t0 % (uint32_t)P.tiles_h);
  int n = (int)(t0 / (uint32_t)P.tiles_h);
  const uint32_t total = (uint32_t)P.total_tiles, step = split ? gridDim.x : 2 * gridDim.x;
  for (uint32_t tile = first; tile < total; tile += step) {
    const int64_t pix = ((int64_t)n * P.o_H + (th * TH + ph) * P.o_mul + P.o_a) * P.o_W + (tw * TW + pw) * P.o_mul + P.o_b;
    const int cgt = nt * NT;
    float* out_px = outp + pix * P.out_ld + cgt;
    mbar_wait(&t_full[ts], tp);
    tc_fence_after();
    const uint32_t taddr0 = taddr_q + ts * (uint32_t)NT;
    for (int c0 = cbeg; c0 < cend; c0 += 32) {
      uint32_t v[32];
      tc_ld16(taddr0 + c0, v);
      tc_ld16(taddr0 + c0 + 16, v + 16);
      tc_wait_ld();
      if (P.lo_off) {
        uint32_t u[32];
        for (int a = 1; a < P.kacc; ++a) {                      // the other filter rows' accumulators
          tc_ld16(taddr0 + (uint32_t)(a * P.acc_plane) + c0, u);
          tc_ld16(taddr0 + (uint32_t)(a * P.acc_plane) + c0 + 16, u + 16);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
        }
        tc_ld16(taddr0 + (uint32_t)P.lo_off + c0, u);
        tc_ld16(taddr0 + (uint32_t)P.lo_off + c0 + 16, u + 16);
        tc_wait_ld();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
      }
      const uint32_t bias_b = bias_u + (uint32_t)(cgt + c0) * 4;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const float4 b0 = lds128f(bias_b + 32 * g), b1 = lds128f(bias_b + 32 * g + 16);
        float f[8];
        f[0] = __uint_as_float(v[8 * g + 0]) + b0.x; f[1] = __uint_as_float(v[8 * g + 1]) + b0.y;
        f[2] = __uint_as_float(v[8 * g + 2]) + b0.z; f[3] = __uint_as_float(v[8 * g + 3]) + b0.w;
        f[4] = __uint_as_float(v[8 * g + 4]) + b1.x; f[5] = __uint_as_float(v[8 * g + 5]) + b1.y;
        f[6] = __uint_as_float(v[8 * g + 6]) + b1.z; f[7] = __uint_as_float(v[8 * g + 7]) + b1.w;
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], relu_lo);
        const int c = cgt + c0 + 8 * g;
        if (vec_ok && c + 8 <= Cout) {
          stg256(out_px + c0 + 8 * g,
                 make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3])),
                 make_uint4(__float_as_uint(f[4]), __float_as_uint(f[5]), __float_as_uint(f[6]), __float_as_uint(f[7])));
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (c + j < Cout) out_px[c0 + 8 * g + j] = f[j];
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&t_empty[ts]);
    ts += split ? 1u : 2u;
    if (ts >= (uint32_t)P.nst) { ts -= (uint32_t)P.nst; tp ^= 1; }
    nt += stepd[0]; if (nt >= P.ntiles_n) { nt -= P.ntiles_n; ++tw; }
    tw += stepd[1]; if (tw >= P.tiles_w) { tw -= P.tiles_w; ++th; }
    th += stepd[2]; if (th >= P.tiles_h) { th -= P.tiles_h; ++n; }
    n += stepd[3];
  }
}

// Tap tables, compile-time so the MMA issue loop unrolls into immediate-offset descriptor adds
// (a single thread issues every MMA: any dependent address arithmetic there is on the critical path).
//   MODE 0: 3x3 stride 1, one halo slab, 9 taps      MODE 1: 1x1 (stride 1 or 2), one slab, one tap
//   MODE 2: 3x3 stride 2, six parity slabs: slab 2*kw -> taps (kh=0, kh=2), slab 2*kw+1 -> tap kh=1
//   MODE 3: one halo slab, taps from the launch's table (P.slabs[0]) - the four parity sub-convolutions of a stride-2 data gradient
template <int MODE> __device__ __forceinline__ constexpr int mode_slabs() { return MODE == 2 ? 6 : 1; }
template <int MODE> __device__ __forceinline__ constexpr int mode_taps(int s) {
  return MODE == 0 ? 9 : (MODE == 1 ? 1 : ((s & 1) ? 1 : 2));
}
template <int MODE> __device__ __forceinline__ constexpr int mode_tap_pix(int s, int t) {
  return MODE == 0 ? (t / 3) * (TW + 2) + (t % 3) : (MODE == 1 ? 0 : (((s & 1) == 0 && t == 1) ? TW : 0));
}
template <int MODE> __device__ __forceinline__ constexpr int mode_tap_id(int s, int t) {
  return MODE == 0 ? t : (MODE == 1 ? 0 : ((s & 1) ? 3 + (s >> 1) : (t ? 6 + (s >> 1) : (s >> 1))));
}

// TF32: 0 = bf16 operands (inference); 1 = one kind::tf32 pass over the raw fp32 operands (the tensor core keeps 10 mantissa
// bits and TRUNCATES the rest); 3 = error-compensated "3 x TF32": x = x_hi + x_lo, w = w_hi + w_lo and
//   x*w ~= x_hi*w_hi + x_hi*w_lo + x_lo*w_hi        (dropped: x_lo*w_lo ~ 2^-22; products exact, fp32 accumulation)
// - fp32-grade results from the tensor pipe, which the training step needs: train-mode BatchNorm makes LED-Net's gradient
// so ill-conditioned that tf32-level operand rounding alone moves it by tens of percent (tools/diag_tf32_grads.py).
// x_hi is what the hardware truncation of the raw slab yields; x_lo = x - trunc(x) is written next to every TMA-staged
// slab by four converter warps (11..14); w_hi / w_lo come pre-split from the host side (rows [0, cp) and [cp, 2 cp)).
template <int TF32> __device__ __forceinline__ constexpr int conv_tc_threads() { return TF32 == 3 ? kThreads + 128 : kThreads; }

template <int MODE, int KSTEPS, bool S2, bool BRES, int TF32 = 0>
__global__ void __launch_bounds__(conv_tc_threads<TF32>(), 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ TcParams P) {
  constexpr int NTHR = conv_tc_threads<TF32>();
  constexpr bool X3 = TF32 == 3;
#define NTAPS(s) (MODE == 3 ? P.slabs[0].ntaps : mode_taps<MODE == 3 ? 0 : MODE>(s))
#define TAPPIX(s, t) (MODE == 3 ? P.slabs[0].tap_pix[t] : mode_tap_pix<MODE == 3 ? 0 : MODE>(s, t))
#define TAPID(s, t) (MODE == 3 ? P.slabs[0].tap_id[t] : mode_tap_id<MODE == 3 ? 0 : MODE>(s, t))
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve: [A ring][B ring or resident B][epilogue staging][bias / out2 affine][barriers]
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = sA + (size_t)P.SA * P.a_stage_bytes;
  const int nb_tiles = P.b_resident ? P.nchunks * 9 : P.SB;   // resident: indexed [chunk][tap]
  uint8_t* sStage = sB + (size_t)nb_tiles * P.b_tile_bytes;   // 4 warps x (1 or 2) x 4 KB
  float* s_bias = reinterpret_cast<float*>(sStage + P.stage_bytes);   // [cp]
  float* s_o2s = s_bias + P.cp;                                       // [cp]
  float* s_o2b = s_o2s + P.cp;                                        // [cp]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_o2b + P.cp);
  uint64_t* a_full = bars;                 // [8]
  uint64_t* a_empty = a_full + 8;          // [8]
  uint64_t* b_full = a_empty + 8;          // [8] (resident: [0] only)
  uint64_t* b_empty = b_full + 8;          // [8]
  uint64_t* t_full = b_empty + 8;          // [4]
  uint64_t* t_empty = t_full + 4;          // [4]
  uint64_t* a_lo_full = t_empty + 4;       // [8] X3: the low-part slab next to A stage i is written
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_lo_full + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  TL(0, threadIdx.x == 0); TLG(12, threadIdx.x == 0);

  if (threadIdx.x == 0) {
    // descriptor fetch starts now instead of at the first TMA (part of the fixed cost per launch, r1c_notes.md 3b)
    prefetch_tensormap(&tmA);
    prefetch_tensormap(&tmB);
    for (int i = 0; i < 8; ++i) {
      mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1);
      mbar_init(&a_lo_full[i], 4);
    }
    for (int i = 0; i < 4; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], P.NT >= 64 ? 8 : 4); }
    mbar_fence_init();
    if (BRES) {
      // whole folded weight matrix once per persistent CTA: one barrier, one expect_tx for all boxes.  Issued by
      // the thread that initialised the barriers, BEFORE the CTA-wide sync: the weight fetch (up to 150 KB, the
      // longest latency of the ramp) overlaps the TMEM allocation and the bias loads instead of following them
      mbar_expect_tx(&b_full[0], (uint32_t)(P.nchunks * P.ntaps_total) * P.b_box_bytes * (X3 ? 2u : 1u));
      for (int ch = 0; ch < P.nchunks; ++ch)
        for (int t = 0; t < P.ntaps_total; ++t) {
          tma_load_2d(smem_u32(sB + (size_t)(ch * 9 + t) * P.b_tile_bytes), &tmB, smem_u32(&b_full[0]),
                      t * P.Cin + ch * P.KC, 0);
          if (X3) tma_load_2d(smem_u32(sB + (size_t)(ch * 9 + t) * P.b_tile_bytes + P.b_tile_bytes / 2), &tmB,
                              smem_u32(&b_full[0]), t * P.Cin + ch * P.KC, P.cp);
        }
    }
    TL(1, true);
  }
  if (warp == 1) {   // TMEM allocation: one full warp, address lands in shared memory
    tmem_alloc(tmem_slot, P.tmem_cols);
  }
  // Set-up barrier (named barrier 1).  The producer warp needs neither TMEM nor the epilogue constants: it only
  // ARRIVES (its barrier initialisation is ordered before the other warps' bar.sync) and requests the first A slabs
  // while the other warps are still allocating TMEM and waiting for their bias loads - measured with the timeline
  // probe (tools/probes/tc_timeline.py): first A request 2.0 us after kernel entry when it waited for the sync.
  uint32_t tmem_base = 0;
  if (warp == 0) {
    __syncwarp();
    asm volatile("bar.arrive 1, %0;" ::"n"(NTHR) : "memory");
  } else {
    // per-channel epilogue constants, zero padded to cp so no channel guard is needed later
    for (int c = threadIdx.x - 32; c < P.cp; c += NTHR - 32) {
      const bool in = c < P.Cout;
      s_bias[c] = (P.bias && in) ? P.bias[c] : 0.f;
      s_o2s[c] = in ? (P.o2_scale ? P.o2_scale[c] : 1.f) : 0.f;
      s_o2b[c] = (P.o2_shift && in) ? P.o2_shift[c] : 0.f;
    }
    tc_fence_before();
    asm volatile("bar.sync 1, %0;" ::"n"(NTHR) : "memory");
    tc_fence_after();
    TL(2, threadIdx.x == 32);
    tmem_base = *tmem_slot;
  }

  const uint32_t row_bytes = P.KC * 2;
  const uint32_t layout_type = (P.KC == 64) ? 2u : (P.KC == 32 ? 4u : 6u);   // SW128 / SW64 / SW32

  if (warp == 0) {
    // =========================== TMA producer: ONE elected lane runs the whole role ================
    if (elect_one()) {
      int sa = 0, pa = 0, sb = 0, pb = 0;
      // (resident weights were requested by thread 0 before the CTA-wide sync)
      // tile coordinates as mixed-radix digits advanced by the grid step (no per-tile divisions)
      uint32_t t0 = blockIdx.x;
      int nt = (int)(t0 % (uint32_t)P.ntiles_n); t0 /= (uint32_t)P.ntiles_n;
      int tw = (int)(t0 % (uint32_t)P.tiles_w); t0 /= (uint32_t)P.tiles_w;
      int th = (int)(t0 % (uint32_t)P.tiles_h);
      int n = (int)(t0 / (uint32_t)P.tiles_h);
      const uint32_t total = (uint32_t)P.total_tiles;
      for (uint32_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int h0 = th * TH, w0 = tw * TW;
        for (int ch = 0; ch < P.nchunks; ++ch) {
          for (int s = 0; s < P.nslabs; ++s) {
            const Slab& sl = P.slabs[s];
            mbar_wait(&a_empty[sa], pa ^ 1);
            if (P.dbg & 4) {
              mbar_arrive(&a_full[sa]);
            } else {
              mbar_expect_tx(&a_full[sa], P.a_box_bytes);
              const uint32_t dst = smem_u32(sA + (size_t)sa * P.a_stage_bytes);
              if (S2) tma_load_5d(dst, &tmA, smem_u32(&a_full[sa]), sl.c_mul * P.in_ld + ch * P.KC, w0 + sl.dw, sl.ph, h0 + sl.dh, n);
              else    tma_load_4d(dst, &tmA, smem_u32(&a_full[sa]), ch * P.KC, w0 + sl.dw, h0 + sl.dh, n);
            }
            TL(3, tile == blockIdx.x && ch == 0 && s == 0);
            if (++sa == P.SA) { sa = 0; pa ^= 1; }
            if (!BRES) {
              for (int t = 0; t < sl.ntaps; ++t) {
                mbar_wait(&b_empty[sb], pb ^ 1);
                mbar_expect_tx(&b_full[sb], P.b_box_bytes * (X3 ? 2u : 1u));
                tma_load_2d(smem_u32(sB + (size_t)sb * P.b_tile_bytes), &tmB, smem_u32(&b_full[sb]),
                            sl.tap_id[t] * P.Cin + ch * P.KC, nt * P.NT);
                if (X3) tma_load_2d(smem_u32(sB + (size_t)sb * P.b_tile_bytes + P.b_tile_bytes / 2), &tmB,
                                    smem_u32(&b_full[sb]), sl.tap_id[t] * P.Cin + ch * P.KC, P.cp + nt * P.NT);
                if (++sb == P.SB) { sb = 0; pb ^= 1; }
              }
            }
          }
        }
        nt += P.step1[0]; if (nt >= P.ntiles_n) { nt -= P.ntiles_n; ++tw; }
        tw += P.step1[1]; if (tw >= P.tiles_w) { tw -= P.tiles_w; ++th; }
        th += P.step1[2]; if (th >= P.tiles_h) { th -= P.tiles_h; ++n; }
        n += P.step1[3];
      }
    }
    __syncwarp();
  } else if (warp == 1 || warp == 10) {
    // =========================== MMA issuers: ONE elected lane of warp 1 (and of warp 10) ==========
    // Two issuers alternate tiles when the weights are resident.  Measured (ncu r1c, profiles/r1c_notes.md): after
    // the last tcgen05.mma of a tile the issuing thread rewrites a uniform register the queued MMAs still read
    // (write-after-read scoreboard), so it sits until the MMA queue has drained and only then runs its ~250
    // instructions of barrier waits and descriptor set-up for the next tile - the tensor pipe idles ~1250 clk per
    // tile (83 clk per MMA against 48 in isolation).  With a second issuer that bubble is covered by the other
    // thread's tile: the two tiles use different accumulator stages and A slabs, so their MMAs may interleave.
    // (a branch on elect.sync, not a per-lane predicate on each MMA: ptxas then knows a single thread is
    // active and issues each tcgen05.mma straight from uniform registers; the predicated form cost an
    // ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall of 17 instructions per MMA, and this thread's issue
    // rate is the per-tile critical path of every 3x3 layer - ncu r1b: producer and epilogue both wait on it)
    const int nmw = (P.dbg & 128) ? 1 : P.nmw;              // host: 2 only with resident weights and SA % (2 * slabs per tile) == 0
    const int mw = (warp == 1) ? 0 : 1;
    if (mw < nmw && elect_one()) {
      const bool mma_on = !(P.dbg & 2);
      const uint32_t idesc = TF32 != 0 ? make_idesc_tf32_m128(P.NT) : make_idesc_bf16_m128(P.NT);
      // probe bit 32 (timing only, results wrong): 8-row groups 1024 B apart (atom aligned) instead of one slab row
      const uint32_t a_hi = desc_hi((P.dbg & 32) ? 8 * row_bytes : (uint32_t)P.sbo_bytes, layout_type);
      const uint32_t b_hi = desc_hi(8 * row_bytes, layout_type);
      const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB);
      constexpr uint32_t ROWB = KSTEPS * 32;        // bytes per A/B row = KC * 2
      // descriptor low words advance by (bytes >> 4); the 14-bit address field cannot overflow (smem < 256 KB)
      const uint32_t a_lo0 = ((sA_u >> 4) & 0x3FFFu) | (1u << 16), b_lo0 = ((sB_u >> 4) & 0x3FFFu) | (1u << 16);
      const uint32_t a_stage16 = P.a_stage_bytes >> 4, b_tile16 = P.b_tile_bytes >> 4;
      int sa = 0, pa = 0, sb = 0, pb = 0;
      int ts = 0, tp = 0;
      if (BRES) { mbar_wait(&b_full[0], 0); tc_fence_after(); }
      TL(4, mw == 0);
      const uint32_t total = (uint32_t)P.total_tiles;
      // the j-th tile of this CTA owns accumulator stage j % nst and the next nchunks * slabs A stages of the ring
      const int slabs_per_tile = P.nchunks * mode_slabs<MODE>();
      auto skip_tile = [&]() {
        for (int i = 0; i < slabs_per_tile; ++i) if (++sa == P.SA) { sa = 0; pa ^= 1; }
        if (++ts == P.nst) { ts = 0; tp ^= 1; }
      };
      if (mw == 1) skip_tile();
      for (uint32_t tile = blockIdx.x + (uint32_t)mw * gridDim.x; tile < total; tile += (uint32_t)nmw * gridDim.x) {
        mbar_wait(&t_empty[ts], tp ^ 1);            // epilogue has drained this accumulator stage
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ts * P.NT);
        for (int ch = 0; ch < P.nchunks; ++ch) {
          // accumulate flag: 0 only for the very first MMA of a tile.  It must NOT be a loop-carried register:
          // ptxas then re-materialises it into the uniform register the in-flight UTCHMMAs still read (R2UR per
          // tap), and that write-after-read wait drains the MMA queue at every tap (measured: 158 clk stall per
          // tap, 83 clk per MMA instead of 48 - profiles/r1c_notes.md).  Every MMA but the chunk's first takes a
          // literal 1.
          const uint32_t acc_first = ch ? 1u : 0u;
          const uint32_t b_chunk = b_lo0 + (uint32_t)(ch * 9) * b_tile16;   // resident weights of this chunk
#pragma unroll
          for (int s = 0; s < mode_slabs<MODE>(); ++s) {
            mbar_wait(&a_full[sa], pa);
            tc_fence_after();
            TL(5, tile == blockIdx.x && ch == 0 && s == 0);
            const uint32_t a_lo = a_lo0 + (uint32_t)sa * a_stage16;
            if constexpr (X3) {
              // three passes per (tap, k-step); the low-part slab is only needed for the third, so its barrier is waited
              // for after the raw-slab MMAs of the slab (resident weights) or of the first tap (streamed weights) are queued
              const uint32_t a_half16 = a_stage16 >> 1, b_half16 = b_tile16 >> 1;
              const uint32_t d_lo = d_tmem + (uint32_t)P.lo_off;        // correction passes: their own accumulator
              if (BRES) {
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                  if (t < NTAPS(s)) {
                    const uint32_t b_lo = b_chunk + (uint32_t)TAPID(s, t) * b_tile16;
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k) {
                      const uint32_t al = a_lo + (((uint32_t)TAPPIX(s, t) * ROWB + k * 32) >> 4);
                      // main product into the accumulator of this tap's filter row (kacc = 3) or the single one
                      const uint32_t d_main = d_tmem + ((MODE == 0 && P.kacc == 3) ? (uint32_t)((t / 3) * P.acc_plane) : 0u);
                      if (s == 0 && k == 0 && (t == 0 || (MODE == 0 && P.kacc == 3 && t % 3 == 0)))
                        tc_mma2_tf32(d_main, al, a_hi, b_lo + 2 * k, b_hi, idesc, acc_first);
                      else
                        tc_mma2_acc_tf32(d_main, al, a_hi, b_lo + 2 * k, b_hi, idesc);
                      if (s == 0 && t == 0 && k == 0) tc_mma2_tf32(d_lo, al, a_hi, b_lo + b_half16 + 2 * k, b_hi, idesc, acc_first);
                      else tc_mma2_acc_tf32(d_lo, al, a_hi, b_lo + b_half16 + 2 * k, b_hi, idesc);
                    }
                  }
                }
                mbar_wait(&a_lo_full[sa], pa);
                tc_fence_after();
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                  if (t < NTAPS(s)) {
                    const uint32_t b_lo = b_chunk + (uint32_t)TAPID(s, t) * b_tile16;
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k) {
                      const uint32_t al = a_lo + a_half16 + (((uint32_t)TAPPIX(s, t) * ROWB + k * 32) >> 4);
                      tc_mma2_acc_tf32(d_lo, al, a_hi, b_lo + 2 * k, b_hi, idesc);
                    }
                  }
                }
              } else {
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                  if (t < NTAPS(s)) {
                    mbar_wait(&b_full[sb], pb);
                    tc_fence_after();
                    const uint32_t b_lo = b_lo0 + (uint32_t)sb * b_tile16;
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k) {
                      const uint32_t al = a_lo + (((uint32_t)TAPPIX(s, t) * ROWB + k * 32) >> 4);
                      // main product into the accumulator of this tap's filter row (kacc = 3) or the single one
                      const uint32_t d_main = d_tmem + ((MODE == 0 && P.kacc == 3) ? (uint32_t)((t / 3) * P.acc_plane) : 0u);
                      if (s == 0 && k == 0 && (t == 0 || (MODE == 0 && P.kacc == 3 && t % 3 == 0)))
                        tc_mma2_tf32(d_main, al, a_hi, b_lo + 2 * k, b_hi, idesc, acc_first);
                      else
                        tc_mma2_acc_tf32(d_main, al, a_hi, b_lo + 2 * k, b_hi, idesc);
                      if (s == 0 && t == 0 && k == 0) tc_mma2_tf32(d_lo, al, a_hi, b_lo + b_half16 + 2 * k, b_hi, idesc, acc_first);
                      else tc_mma2_acc_tf32(d_lo, al, a_hi, b_lo + b_half16 + 2 * k, b_hi, idesc);
                    }
                    if (t == 0) { mbar_wait(&a_lo_full[sa], pa); tc_fence_after(); }
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k) {
                      const uint32_t al = a_lo + a_half16 + (((uint32_t)TAPPIX(s, t) * ROWB + k * 32) >> 4);
                      tc_mma2_acc_tf32(d_lo, al, a_hi, b_lo + 2 * k, b_hi, idesc);
                    }
                    tc_commit(&b_empty[sb]);
                    if (++sb == P.SB) { sb = 0; pb ^= 1; }
                  }
                }
              }
            } else
            if (BRES) {
              // resident weights: no per-tap waits, so the slab's MMAs are ONE straight-line block - every
              // descriptor word is the per-slab base plus an immediate and the uniform registers the in-flight
              // UTCHMMAs read are not rewritten between taps
              if (mma_on) {
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                  if (t < NTAPS(s)) {
                    const uint32_t b_lo = b_chunk + (uint32_t)TAPID(s, t) * b_tile16;
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k) {
                      const uint32_t al = a_lo + (((uint32_t)TAPPIX(s, t) * ROWB + k * 32) >> 4);
                      if constexpr (TF32 != 0) {
                        if (s == 0 && t == 0 && k == 0) tc_mma2_tf32(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc, acc_first);
                        else tc_mma2_acc_tf32(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc);
                      } else {
                        if (s == 0 && t == 0 && k == 0) tc_mma2(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc, acc_first);
                        else tc_mma2_acc(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc);
                      }
                    }
                  }
                }
              }
            } else {
#pragma unroll
              for (int t = 0; t < 9; ++t) {
                if (t < NTAPS(s)) {
                  mbar_wait(&b_full[sb], pb);
                  tc_fence_after();
                  const uint32_t b_lo = b_lo0 + (uint32_t)sb * b_tile16;
                  if (mma_on) {
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k) {
                      const uint32_t al = a_lo + (((uint32_t)TAPPIX(s, t) * ROWB + k * 32) >> 4);
                      if constexpr (TF32 != 0) {
                        if (s == 0 && t == 0 && k == 0) tc_mma2_tf32(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc, acc_first);
                        else tc_mma2_acc_tf32(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc);
                      } else {
                        if (s == 0 && t == 0 && k == 0) tc_mma2(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc, acc_first);
                        else tc_mma2_acc(d_tmem, al, a_hi, b_lo + 2 * k, b_hi, idesc);
                      }
                    }
                  }
                  tc_commit(&b_empty[sb]);                  // frees the B stage when these MMAs retire
                  if (++sb == P.SB) { sb = 0; pb ^= 1; }
                }
              }
            }
            tc_commit(&a_empty[sa]);                        // frees the A slab
            if (++sa == P.SA) { sa = 0; pa ^= 1; }
          }
        }
        tc_commit(&t_full[ts]);                             // accumulator complete -> epilogue
        TL(6, tile == blockIdx.x);
        if (++ts == P.nst) { ts = 0; tp ^= 1; }
        if (nmw == 2) skip_tile();                          // the other issuer's tile
      }
    }
    __syncwarp();
  } else if (warp >= 11) {
    // =========================== X3 only: low-part converter, warps 11..14 ========================
    // walks the A ring exactly like the producer; for every landed slab writes x - trunc_tf32(x) (exact in fp32) into the
    // second half of the stage.  The swizzle is a permutation of 16-byte chunks, so an element-wise pass over the raw
    // bytes keeps the layout.  generic-proxy writes -> fence.proxy.async -> the MMAs (async proxy) may read them.
    if constexpr (X3) {
      const uint32_t ctid = threadIdx.x - 11 * 32;
      int sa = 0, pa = 0;
      const uint32_t total = (uint32_t)P.total_tiles;
      const int slabs_per_tile = P.nchunks * P.nslabs;
      for (uint32_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
        for (int i = 0; i < slabs_per_tile; ++i) {
          mbar_wait(&a_full[sa], pa);
          const uint32_t src = smem_u32(sA + (size_t)sa * P.a_stage_bytes), dst = src + P.a_stage_bytes / 2;
          for (uint32_t o = ctid * 16; o < P.a_box_bytes; o += 128 * 16) {
            const uint4 v = lds128(src + o);
            sts128(dst + o, __float_as_uint(__uint_as_float(v.x) - __uint_as_float(v.x & 0xFFFFE000u)),
                   __float_as_uint(__uint_as_float(v.y) - __uint_as_float(v.y & 0xFFFFE000u)),
                   __float_as_uint(__uint_as_float(v.z) - __uint_as_float(v.z & 0xFFFFE000u)),
                   __float_as_uint(__uint_as_float(v.w) - __uint_as_float(v.w & 0xFFFFE000u)));
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(&a_lo_full[sa]);
          if (++sa == P.SA) { sa = 0; pa ^= 1; }
        }
      }
    }
  } else if (warp < 10) {
    // =========================== epilogue: two groups of 4 warps (see epilogue_loop) ==============
    const uint32_t st_u = smem_u32(sStage), bias_u = smem_u32(s_bias), o2s_u = smem_u32(s_o2s), o2b_u = smem_u32(s_o2b);
    const int variant = (P.res ? 1 : 0) | (P.out ? 2 : 0) | (P.out2 ? 4 : 0);
    if constexpr (TF32 != 0) {
      epilogue_f32(P, warp, lane, tmem_base, t_full, t_empty, bias_u);
    } else
    switch (variant) {
      case 2: epilogue_loop<false, true, false>(P, warp, lane, tmem_base, t_full, t_empty, st_u, bias_u, o2s_u, o2b_u); break;
      case 3: epilogue_loop<true, true, false>(P, warp, lane, tmem_base, t_full, t_empty, st_u, bias_u, o2s_u, o2b_u); break;
      case 4: epilogue_loop<false, false, true>(P, warp, lane, tmem_base, t_full, t_empty, st_u, bias_u, o2s_u, o2b_u); break;
      case 5: epilogue_loop<true, false, true>(P, warp, lane, tmem_base, t_full, t_empty, st_u, bias_u, o2s_u, o2b_u); break;
      case 6: epilogue_loop<false, true, true>(P, warp, lane, tmem_base, t_full, t_empty, st_u, bias_u, o2s_u, o2b_u); break;
      default: epilogue_loop<true, true, true>(P, warp, lane, tmem_base, t_full, t_empty, st_u, bias_u, o2s_u, o2b_u); break;
    }
  }

  TL(9, threadIdx.x == 0);              // producer role finished (its warp reaches the final sync)
  TL(14, warp == 2 && lane == 0);       // first epilogue warp finished
  tc_fence_before();
  __syncthreads();
  TL(10, threadIdx.x == 32);
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, P.tmem_cols);
  }
  TL(11, threadIdx.x == 32); TLG(13, threadIdx.x == 32);
}

#undef NTAPS
#undef TAPPIX
#undef TAPID

// ------------------------------------------------------------------ host side
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

int encode(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
           const uint32_t* box, int kc) {
  EncodeFn fn = get_encode();
  if (!fn) return fail(LEDB200_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t d[5], s[4];
  cuuint32_t b[5], es[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) s[i] = strides_bytes[i];
  // kc = 1064: 128 B rows swizzled in 32-byte chunks (the only layout tcgen05 reads MN-major tf32 operands from, wgrad_tc.cu)
  const CUtensorMapSwizzle sw = kc == 1064 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B
                                : kc == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (kc == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), d, s, b, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LEDB200_ECUDA, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
  return LEDB200_OK;
}

int pick_kc(int cin) { return cin % 64 == 0 ? 64 : 32; }
int num_sms() {
  static int n = 0;
  if (!n) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); if (n <= 0) n = 148; }
  return n;
}
}  // namespace

// tensor-map encoder for the other tcgen05 kernels of the library (wgrad_tc.cu): tiled, 2-byte units, swizzle by box width
int tc_encode_tiled(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, int kc) {
  return encode(m, base, rank, dims, strides_bytes, box, kc);
}

// 32 is the smallest N tile: the epilogue fast path works on 32-column blocks, and an N = 16 MMA costs the same A fetch
int conv_tc_pad(int cout) { return cout <= 32 ? 32 : (cout + 63) / 64 * 64; }

bool conv_tc_eligible(const ConvArgs& a) {
  if (a.tf32) {
    // training convolutions: fp32 NHWC in, raw fp32 (+ bias) out, TF32 tensor-core arithmetic (see epilogue_f32)
    if (a.in_dtype != LEDB200_F32 || a.out_dtype != LEDB200_F32 || !a.out) return false;
    if (a.pre_scale || a.res || a.out2 || a.relu == 2) return false;
    if (a.ksize != 1 && a.ksize != 3) return false;
    if (a.stride != 1 && a.stride != 2) return false;
    if (a.dil != 1 && a.ksize == 3) return false;
    if (a.Cin < 32 || a.Cin % 32) return false;                      // K blocks of 32 fp32 channels (128 B rows)
    if (a.in_sc != 1 || a.in_sw % 4) return false;
    if (a.stride == 2 && ((a.H & 1) || (a.W & 1))) return false;
    if (a.Ho % TH || a.Wo % TW) return false;                        // all-interior tilings only (else: CUDA-core kernels)
    if (a.sub && a.stride != 1) return false;
    if (a.out_ld < a.Cout) return false;
    const int cp = a.cout_pad_tc > 0 ? a.cout_pad_tc : conv_tc_pad(a.Cout);
    if (cp > 256 && cp % 128) return false;                          // wide outputs: 128-column N tiles (e.g. 640 = 5 x 128)
    if (cp != 32 && cp % 64) return false;
    if ((int64_t)a.N * (a.Ho / TH) * (a.Wo / TW) * (cp > 256 ? cp / 128 : 1) >= (1ll << 31)) return false;
    return true;
  }
  if (a.in_dtype != LEDB200_BF16 || a.out_dtype != LEDB200_BF16) return false;
  if (a.pre_scale) return false;
  if (a.ksize != 1 && a.ksize != 3) return false;
  if (a.stride != 1 && a.stride != 2) return false;
  if (a.dil != 1 && a.ksize == 3) return false;
  if (a.Cin < 32 || a.Cin % 32) return false;                        // K blocks of 32 or 64 channels
  if (a.in_sc != 1 || a.in_sw % 8) return false;                     // NHWC, 16 B aligned pixels
  if (a.stride == 2 && ((a.H & 1) || (a.W & 1))) return false;       // parity-split view needs even H, W
  const int c8 = (a.Cout + 7) / 8 * 8;                               // stores cover whole 8-channel groups
  if (a.out && (a.out_ld % 8 || a.out_ld < c8)) return false;
  if (a.out2 && (a.out2_ld % 8 || a.out2_ld < c8)) return false;
  if (a.res && (a.res_ld % 8 || a.res_ld < c8)) return false;
  const int cp = a.cout_pad_tc > 0 ? a.cout_pad_tc : conv_tc_pad(a.Cout);
  if (cp > 256 && cp % 256) return false;
  if (cp != 16 && cp != 32 && cp % 64) return false;                 // epilogue staging slices are 16/32/64 channels
  if ((int64_t)a.N * ceil_div(a.Ho, TH) * ceil_div(a.Wo, TW) * (cp > 256 ? cp / 256 : 1) >= (1ll << 31)) return false;
  return true;
}

int launch_conv_tc(const ConvArgs& a, cudaStream_t st) {
  if (!conv_tc_eligible(a)) return fail(LEDB200_EINVAL, "conv_tc: shape not eligible");
  TcParams P{};
  const bool s2 = a.stride == 2;
  // TF32 launches move fp32 words: every shared-memory / TMA quantity below is in 2-byte units, so an fp32 tensor of C
  // channels is described as 2C units (128 B rows = 32 fp32 channels = "KC 64"); only the MMA kind and the epilogue differ
  const bool tf32 = a.tf32 != 0;
  const bool x3 = a.tf32 == 3;          // error-compensated three-pass mode: low-part slab / weight rows next to every tile
  const int es = tf32 ? 2 : 1;
  const int cinE = a.Cin * es;
  P.Cin = cinE; P.Cout = a.Cout;
  const int cp = a.cout_pad_tc > 0 ? a.cout_pad_tc : conv_tc_pad(a.Cout);
  // N tile: the whole (padded) Cout when it is 16 / 32 / 64 / 128 / 256, 256 for multiples of 256, else 64-column
  // tiles (e.g. 192 = GETB qkv of a 64-channel block): the epilogue's column split needs a power-of-two tile
  P.NT = cp > 256 ? 256 : ((cp & (cp - 1)) == 0 ? cp : 64);
  if (x3 && P.NT > 128) P.NT = 128;     // two weight halves per tile: keep the B ring inside shared memory
  if (tf32 && cp > 256) P.NT = 128;     // wide training outputs (DAPPM's 640-channel data gradient): any multiple of 128
  const bool kacc3 = x3 && a.ksize == 3 && !s2 && !a.sub;     // one main accumulator per filter row (see TcParams::kacc)
  if (kacc3 && P.NT > 64) P.NT = 64;    // (3 main + 1 correction) x 64 columns x 2 stages = the whole TMEM
  P.ntiles_n = cp / P.NT;
  P.KC = tf32 ? 64 : pick_kc(a.Cin);
  P.nchunks = cinE / P.KC;
  P.N = a.N; P.Ho = a.Ho; P.Wo = a.Wo;
  P.tiles_h = ceil_div(a.Ho, TH); P.tiles_w = ceil_div(a.Wo, TW);
  P.total_tiles = (int64_t)a.N * P.tiles_h * P.tiles_w * P.ntiles_n;
  P.in_ld = (int)a.in_sw * es;
  const int row_bytes = P.KC * 2;
  int box_w = TW, box_rows = TH;
  P.sbo_bytes = 8 * row_bytes;
  // ---- slab tables
  int sub_taps = 0;
  if (a.sub && a.ksize == 3) {
    // parity class of a stride-2 data gradient: the halo slab of a 3x3 convolution, taps at offsets {0, +1} (odd parity)
    // or {0} (even parity) per axis, in the order the class's weight matrix is packed (train.cu pack mode 2)
    P.nslabs = 1; box_rows = TH + 2; box_w = TW + 2;
    P.sbo_bytes = box_w * row_bytes;
    Slab& s = P.slabs[0];
    s.c_mul = 0; s.dw = -1; s.dh = -1; s.ph = 0;
    for (int ir = 0; ir < (a.sub_a ? 2 : 1); ++ir)
      for (int ic = 0; ic < (a.sub_b ? 2 : 1); ++ic) {
        const int dr = a.sub_a ? 1 - ir : 0, dc = a.sub_b ? 1 - ic : 0;   // filter row 0 reads dY row i + 1, row 2 reads row i
        s.tap_pix[sub_taps] = (1 + dr) * box_w + (1 + dc);
        s.tap_id[sub_taps] = sub_taps;
        ++sub_taps;
      }
    s.ntaps = sub_taps;
  } else
  if (a.ksize == 3 && !s2) {
    // ONE halo slab (TH+2) x (TW+2) per Cin chunk; every tap is a row- AND column-shifted window of it:
    // the descriptor start address is not swizzle-atom aligned and SBO = (TW+2) rows.  The hardware
    // applies the swizzle XOR on absolute shared-memory address bits (probed on B200, see
    // profiles/r1_notes.md), so this reads exactly what TMA wrote.  Input fetch 1.4x instead of the
    // 3.4x of three column-shifted slabs, one TMA per chunk instead of three.
    P.nslabs = 1; box_rows = TH + 2; box_w = TW + 2;
    P.sbo_bytes = box_w * row_bytes;
    Slab& s = P.slabs[0];
    s.c_mul = 0; s.dw = -1; s.dh = -1; s.ph = 0; s.ntaps = 9;
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) { s.tap_pix[kh * 3 + kw] = kh * box_w + kw; s.tap_id[kh * 3 + kw] = kh * 3 + kw; }
  } else if (a.ksize == 1 && !s2) {
    P.nslabs = 1;
    Slab& s = P.slabs[0];
    s.c_mul = 0; s.dw = 0; s.dh = 0; s.ph = 0; s.ntaps = 1; s.tap_pix[0] = 0; s.tap_id[0] = 0;
  } else if (a.ksize == 3 && s2) {
    // input row 2*oh-1+kh -> (parity, half-row): kh=0 -> (1, oh-1), kh=1 -> (0, oh), kh=2 -> (1, oh); same for columns
    P.nslabs = 6; box_rows = TH + 1;
    int i = 0;
    for (int kw = 0; kw < 3; ++kw) {
      const int pw = (kw == 1) ? 0 : 1, dw = (kw == 0) ? -1 : 0;
      Slab& s1 = P.slabs[i++];
      s1.c_mul = pw; s1.dw = dw; s1.ph = 1; s1.dh = -1; s1.ntaps = 2;
      s1.tap_pix[0] = 0; s1.tap_id[0] = 0 * 3 + kw;          // kh = 0: half-row oh-1
      s1.tap_pix[1] = TW; s1.tap_id[1] = 2 * 3 + kw;         // kh = 2: half-row oh
      Slab& s0 = P.slabs[i++];
      s0.c_mul = pw; s0.dw = dw; s0.ph = 0; s0.dh = 0; s0.ntaps = 1;
      s0.tap_pix[0] = 0; s0.tap_id[0] = 1 * 3 + kw;          // kh = 1
    }
  } else {   // 1x1 stride 2: parity (0,0) only
    P.nslabs = 1;
    Slab& s = P.slabs[0];
    s.c_mul = 0; s.dw = 0; s.dh = 0; s.ph = 0; s.ntaps = 1; s.tap_pix[0] = 0; s.tap_id[0] = 0;
  }
  P.a_stage_bytes = (uint32_t)((box_rows * box_w * row_bytes + 1023) / 1024 * 1024) * (x3 ? 2u : 1u);
  P.b_tile_bytes = (uint32_t)((P.NT * row_bytes + 1023) / 1024 * 1024) * (x3 ? 2u : 1u);
  P.a_box_bytes = (uint32_t)(box_rows * box_w * row_bytes);
  P.b_box_bytes = (uint32_t)(P.NT * row_bytes);
  const int taps = sub_taps ? sub_taps : a.ksize * a.ksize;
  P.ntaps_total = taps;
  // ---- shared-memory plan
  P.cp = cp;
  {
    // Epilogue fast path for interior tiles (epilogue_loop): whole 32-column blocks per epilogue group, no ReLU6, no
    // channel padding beyond the 8-channel groups, 32 B aligned pixels for the 256-bit accesses.
    const int cout8 = (a.Cout + 7) & ~7;
    const int ncols_g = P.NT >= 64 ? P.NT / 2 : P.NT;
    const bool al32 = ((a.out_ld | a.out2_ld | a.res_ld) % 16 == 0) &&
                      (((uintptr_t)a.out | (uintptr_t)a.out2 | (uintptr_t)a.res) % 32 == 0);
    P.fast_epi = (ncols_g % 32 == 0) && a.relu != 2 && cout8 == cp && al32;
  }
  // When every tile is interior and takes the fast path (or the TF32 epilogue), the staging tiles are never touched:
  // their 32-64 KB go to the A ring / resident weights.
  P.stage_bytes = (tf32 || (P.fast_epi && a.Ho % TH == 0 && a.Wo % TW == 0)) ? 0u : (a.out2 ? 65536u : 32768u);
  const uint32_t bar_bytes = (uint32_t)((3 * cp * 4 + 48 * 8 + 16 + 1023) / 1024 * 1024) + P.stage_bytes;
  const uint32_t b_res_bytes = (uint32_t)(P.nchunks * 9) * P.b_tile_bytes;
  P.b_resident = (P.ntiles_n == 1 && b_res_bytes <= (P.stage_bytes ? 100u : 150u) * 1024) ? 1 : 0;
  static const bool no_resident = getenv("LEDB200_TC_NO_RESIDENT") != nullptr;
  if (no_resident) P.b_resident = 0;
  uint32_t left = SMEM_BUDGET - bar_bytes - 1024;
  if (x3) {
    // three-pass mode: an A stage is two slabs (raw + low part, ~47 KB for a 3x3 halo slab), so the A ring is sized first
    if (P.b_resident && b_res_bytes + 2 * P.a_stage_bytes > left) P.b_resident = 0;
    if (P.b_resident) {
      left -= b_res_bytes;
      P.SB = 1;
      P.SA = (int)std::min<uint32_t>(8, left / P.a_stage_bytes);
    } else {
      if (left < 2 * P.a_stage_bytes + 2 * P.b_tile_bytes) return fail(LEDB200_EINVAL, "conv_tc: shared memory plan does not fit");
      P.SB = (int)std::min<uint32_t>(8, (left - 2 * P.a_stage_bytes) / P.b_tile_bytes);
      left -= P.SB * P.b_tile_bytes;
      P.SA = (int)std::min<uint32_t>(8, left / P.a_stage_bytes);
    }
  } else {
  if (P.b_resident) {
    left -= b_res_bytes;
    P.SB = 1;
  } else {
    P.SB = (int)std::min<uint32_t>(8, std::max<uint32_t>(2, (left * 6 / 10) / P.b_tile_bytes));
    left -= P.SB * P.b_tile_bytes;
  }
  P.SA = (int)std::min<uint32_t>(8, left / P.a_stage_bytes);
  }
  if (P.SA < 2) return fail(LEDB200_EINVAL, "conv_tc: shared memory plan does not fit");
  {
    // Two MMA issuers alternate tiles (see the kernel).  An mbarrier parity wait is only sound when the waiter is at
    // most one phase behind, so every A stage must always be consumed by the SAME issuer: the ring length has to be
    // a multiple of 2 x (slabs per tile).  Trim the ring to that, or fall back to one issuer (stride-2 layers: 6 slabs).
    const int slabs_per_tile = P.nchunks * P.nslabs;
    const int sa2 = P.SA / (2 * slabs_per_tile) * (2 * slabs_per_tile);
    P.nmw = 1;
    if (P.b_resident && sa2 >= 2 * slabs_per_tile && sa2 >= 2) { P.nmw = 2; P.SA = sa2; }
  }
  const size_t smem = 1024 + (size_t)P.SA * P.a_stage_bytes +
                      (size_t)(P.b_resident ? P.nchunks * 9 : P.SB) * P.b_tile_bytes + bar_bytes;
  P.kacc = kacc3 ? 3 : 1;
  const int nacc = x3 ? P.kacc + 1 : 1;          // accumulators per stage
  P.nst = (4 * P.NT * nacc <= 512) ? 4 : 2;
  P.acc_plane = P.nst * P.NT;
  P.lo_off = x3 ? P.kacc * P.acc_plane : 0;
  uint32_t cols = 32;
  while (cols < (uint32_t)(P.acc_plane * nacc)) cols <<= 1;
  P.tmem_cols = cols;
  P.out = (__nv_bfloat16*)a.out; P.out_ld = a.out_ld;
  P.out2 = (__nv_bfloat16*)a.out2; P.out2_ld = a.out2_ld; P.o2_scale = a.o2_scale; P.o2_shift = a.o2_shift;
  P.res = (const __nv_bfloat16*)a.res; P.res_ld = a.res_ld; P.bias = a.bias; P.relu = a.relu;
  { const char* e = getenv("LEDB200_TC_DBG"); P.dbg = e ? atoi(e) : 0; }
  { static int tl_counter = 0; P.tl_launch = tl_counter++; }
  P.out_f16 = a.out_f16;
  P.o_mul = a.sub ? 2 : 1; P.o_a = a.sub ? a.sub_a : 0; P.o_b = a.sub ? a.sub_b : 0;
  P.o_H = a.Ho * P.o_mul; P.o_W = a.Wo * P.o_mul;

  // ---- tensor maps
  CUtensorMap tmA, tmB;
  const uint64_t ld = (uint64_t)a.in_sw * es;
  int rc;
  if (!s2) {
    const uint64_t dims[4] = {(uint64_t)cinE, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.N};
    const uint64_t str[3] = {ld * 2, (uint64_t)a.W * ld * 2, (uint64_t)a.H * a.W * ld * 2};
    const uint32_t box[4] = {(uint32_t)P.KC, (uint32_t)box_w, (uint32_t)box_rows, 1};
    rc = encode(&tmA, a.in, 4, dims, str, box, P.KC);
  } else {
    const uint64_t dims[5] = {ld + (uint64_t)cinE, (uint64_t)a.W / 2, 2, (uint64_t)a.H / 2, (uint64_t)a.N};
    const uint64_t str[4] = {2 * ld * 2, (uint64_t)a.W * ld * 2, 2 * (uint64_t)a.W * ld * 2, (uint64_t)a.H * a.W * ld * 2};
    const uint32_t box[5] = {(uint32_t)P.KC, (uint32_t)box_w, 1, (uint32_t)box_rows, 1};
    rc = encode(&tmA, a.in, 5, dims, str, box, P.KC);
  }
  if (rc) return rc;
  {
    const uint64_t dims[2] = {(uint64_t)taps * cinE, (uint64_t)cp * (tf32 ? 2 : 1)};   // tf32: rows [cp, 2 cp) = low parts
    const uint64_t str[1] = {(uint64_t)taps * cinE * 2};
    const uint32_t box[2] = {(uint32_t)P.KC, (uint32_t)P.NT};
    rc = encode(&tmB, tf32 ? (const void*)a.w_tc32 : (const void*)a.w_tc, 2, dims, str, box, P.KC);
  }
  if (rc) return rc;

  const int grid = (int)std::min<int64_t>(P.total_tiles, num_sms());
  {
    for (int k = 1; k <= 2; ++k) {
      int* d = k == 1 ? P.step1 : P.step2;
      uint32_t stp = (uint32_t)(k * grid);
      d[0] = (int)(stp % (uint32_t)P.ntiles_n); stp /= (uint32_t)P.ntiles_n;
      d[1] = (int)(stp % (uint32_t)P.tiles_w); stp /= (uint32_t)P.tiles_w;
      d[2] = (int)(stp % (uint32_t)P.tiles_h);
      d[3] = (int)(stp / (uint32_t)P.tiles_h);
    }
  }
  const int mode = (a.ksize == 1) ? 1 : (sub_taps ? 3 : (s2 ? 2 : 0));
  const int ksteps = P.KC / 16;
  using KernelFn = void (*)(const CUtensorMap, const CUtensorMap, const TcParams);
  // [mode][stride 2][KC == 64][weights resident]
  static const KernelFn kernels[3][2][2][2] = {
      {{{conv_tc_kernel<0, 2, false, false>, conv_tc_kernel<0, 2, false, true>},
        {conv_tc_kernel<0, 4, false, false>, conv_tc_kernel<0, 4, false, true>}},
       {{nullptr, nullptr}, {nullptr, nullptr}}},
      {{{conv_tc_kernel<1, 2, false, false>, conv_tc_kernel<1, 2, false, true>},
        {conv_tc_kernel<1, 4, false, false>, conv_tc_kernel<1, 4, false, true>}},
       {{conv_tc_kernel<1, 2, true, false>, conv_tc_kernel<1, 2, true, true>},
        {conv_tc_kernel<1, 4, true, false>, conv_tc_kernel<1, 4, true, true>}}},
      {{{nullptr, nullptr}, {nullptr, nullptr}},
       {{conv_tc_kernel<2, 2, true, false>, conv_tc_kernel<2, 2, true, true>},
        {conv_tc_kernel<2, 4, true, false>, conv_tc_kernel<2, 4, true, true>}}}};
  // TF32 instantiations (KSTEPS = 4: four 32-byte k-steps per 128 B row): [three-pass][mode][stride 2][weights resident]
  static const KernelFn kernels_tf32[2][4][2][2] = {
      {{{conv_tc_kernel<0, 4, false, false, 1>, conv_tc_kernel<0, 4, false, true, 1>}, {nullptr, nullptr}},
       {{conv_tc_kernel<1, 4, false, false, 1>, conv_tc_kernel<1, 4, false, true, 1>},
        {conv_tc_kernel<1, 4, true, false, 1>, conv_tc_kernel<1, 4, true, true, 1>}},
       {{nullptr, nullptr}, {conv_tc_kernel<2, 4, true, false, 1>, conv_tc_kernel<2, 4, true, true, 1>}},
       {{conv_tc_kernel<3, 4, false, false, 1>, conv_tc_kernel<3, 4, false, true, 1>}, {nullptr, nullptr}}},
      {{{conv_tc_kernel<0, 4, false, false, 3>, conv_tc_kernel<0, 4, false, true, 3>}, {nullptr, nullptr}},
       {{conv_tc_kernel<1, 4, false, false, 3>, conv_tc_kernel<1, 4, false, true, 3>},
        {conv_tc_kernel<1, 4, true, false, 3>, conv_tc_kernel<1, 4, true, true, 3>}},
       {{nullptr, nullptr}, {conv_tc_kernel<2, 4, true, false, 3>, conv_tc_kernel<2, 4, true, true, 3>}},
       {{conv_tc_kernel<3, 4, false, false, 3>, conv_tc_kernel<3, 4, false, true, 3>}, {nullptr, nullptr}}}};
  static std::once_flag attr_once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once, [] {
    for (int x = 0; x < 2; ++x)
      for (int m = 0; m < 4; ++m)
        for (int s = 0; s < 2; ++s)
          for (int r = 0; r < 2; ++r)
            if (kernels_tf32[x][m][s][r]) {
              cudaError_t e = cudaFuncSetAttribute(kernels_tf32[x][m][s][r], cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   (int)SMEM_BUDGET + 2048);
              if (e != cudaSuccess) attr_err = e;
            }
    for (int m = 0; m < 3; ++m)
      for (int s = 0; s < 2; ++s)
        for (int k = 0; k < 2; ++k)
          for (int r = 0; r < 2; ++r)
            if (kernels[m][s][k][r]) {
              cudaError_t e = cudaFuncSetAttribute(kernels[m][s][k][r], cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   (int)SMEM_BUDGET + 2048);
              if (e != cudaSuccess) attr_err = e;
            }
  });
  if (attr_err != cudaSuccess) return fail(LEDB200_ECUDA, std::string("conv_tc: cudaFuncSetAttribute: ") + cudaGetErrorString(attr_err));
  const KernelFn fn = tf32 ? kernels_tf32[x3 ? 1 : 0][mode][s2 ? 1 : 0][P.b_resident ? 1 : 0]
                           : kernels[mode][s2 ? 1 : 0][ksteps == 4][P.b_resident ? 1 : 0];
  fn<<<grid, x3 ? kThreads + 128 : kThreads, smem, st>>>(tmA, tmB, P);
  LEDB_LAUNCH_OK("conv_tc_kernel");
  return LEDB200_OK;
}

}  // namespace ledb

#ifdef LEDB_TC_TIMELINE
// probe builds only: copy the 128 x 16 stamp table of the last launches to the host (after a device sync)
extern "C" int ledb200_probe_tc_timeline(unsigned long long* out) {
  if (cudaDeviceSynchronize() != cudaSuccess) return 1;
  return cudaMemcpyFromSymbol(out, ledb::g_tc_tl, sizeof(unsigned long long) * 128 * 16) == cudaSuccess ? 0 : 1;
}
#endif
