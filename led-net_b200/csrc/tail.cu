// Fused head tail (north_star kernel 4b): 3-level bilinear ladder + argmax in ONE kernel, so the
// full-resolution logits [N,K,H,W] (159 MB / image at K=19, 1024x2048) never reach HBM.
//
// Replaces BaseDecodeHead.predict_by_feat as patched by the reference's author
//   (mmseg/models/decode_heads/decode_head.py:362-379):
//       size = ceil(2 * head_x1.HW)
//       r = head_x2 + resize(x_c, ceil(size/4));  r = head_x1 + resize(r, ceil(size/2));
//       out = resize(r, size)                      (bilinear, align_corners=False)
//   and BaseSegmentor.postprocess_result's `argmax(dim=0, keepdim=True)`
//   (mmseg/models/segmentors/base.py:187-188; torch.argmax returns the FIRST maximal index).
//
// One CTA (128 threads) produces a 32 x 64 output tile; three CTAs are resident per SM.  Classes are
// processed in passes of up to 24 (one pass for K <= 24).  Per pass the CTA stages, in shared memory
// and fp32,
//   xc patch -> r2 patch (= hx2 + up(xc)) -> r1 patch (= hx1 + up(r2)), r1 laid out [k][row][col],
// with the bilinear source indices / weights of every patch row and column computed ONCE per tile into
// small tables (ATen's align_corners=False formula, any size ratio), 8 classes (16 B bf16 / 32 B fp32)
// per load.  Then every thread interpolates its own 4 x 4 output block from a 4 x 4 window of r1 (the
// last stage is always an exact x2 upsample because size = 2*head_x1.HW) with 8 LDS.64 per class,
// keeping a running (max, index) pair per pixel in registers.  Strict `>` in ascending class order is
// torch.argmax's first-max rule.  Every input element is read once per CTA (plus the 1-pixel clamped
// halo); output is 1 byte per pixel (or int64 when asked).  The kernel is instruction-issue bound
// (about 7.5 instructions per output logit in the last stage), not HBM bound: DESIGN.md section 3.
#include "kernels.h"

namespace ledb {
namespace {

constexpr int KP = 24;                      // classes per pass (three 8-class groups)
constexpr int TROWS = 8, TCOLS = 16;        // thread grid: each thread owns a 4x4 output block
constexpr int TAIL_THREADS = TROWS * TCOLS; // 128
constexpr int OT_H = 4 * TROWS, OT_W = 4 * TCOLS;           // 32 x 64 output tile
constexpr int R1_H = 2 * TROWS + 2, R1_W = 2 * TCOLS + 2;   // 18 x 34 r1 patch (with clamped halo)
constexpr int R2_H = 12, R2_W = 20;         // capacity of the r2 patch
constexpr int XC_H = 9, XC_W = 13;          // capacity of the xc patch
constexpr int R1_PLANE = R1_H * R1_W;       // 612 floats per class

struct TailTables {                         // per-tile bilinear tables
  int r1_gy[R1_H], r1_gx[R1_W];             // clamped global hx1 row / col of each patch row / col
  int r1_y0[R1_H], r1_y1[R1_H], r1_x0[R1_W], r1_x1[R1_W];   // r2-patch-relative source rows / cols
  float r1_wy[R1_H], r1_wx[R1_W];           // weight of the second source
  int r2_y0[R2_H], r2_y1[R2_H], r2_x0[R2_W], r2_x1[R2_W];   // xc-patch-relative source rows / cols
  float r2_wy[R2_H], r2_wx[R2_W];
};

template <typename T>
__device__ __forceinline__ void load_group(const T* p, int c0, int K, bool vec, float v[8]) {
  if (vec) {
    load8(p + c0, v);
  } else {
#pragma unroll
    for (int c = 0; c < 8; ++c) v[c] = (c0 + c < K) ? to_f32(p[c0 + c]) : 0.f;
  }
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// v[c] += bilinear(4 corners) for 8 classes; corner pointers are fp32 [8] in shared memory
__device__ __forceinline__ void add_bilerp8(float v[8], const float* p00, const float* p01, const float* p10,
                                            const float* p11, float wx, float wy) {
  const float4 a0 = *reinterpret_cast<const float4*>(p00), a1 = *reinterpret_cast<const float4*>(p00 + 4);
  const float4 b0 = *reinterpret_cast<const float4*>(p01), b1 = *reinterpret_cast<const float4*>(p01 + 4);
  const float4 c0 = *reinterpret_cast<const float4*>(p10), c1 = *reinterpret_cast<const float4*>(p10 + 4);
  const float4 d0 = *reinterpret_cast<const float4*>(p11), d1 = *reinterpret_cast<const float4*>(p11 + 4);
  const float ux = 1.f - wx, uy = 1.f - wy;
  const float A[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
  const float B[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
  const float C[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
  const float D[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const float r0 = fmaf(B[c], wx, A[c] * ux);
    const float r1 = fmaf(D[c], wx, C[c] * ux);
    v[c] += fmaf(r1, wy, r0 * uy);
  }
}

template <typename T, typename TP>
__global__ void __launch_bounds__(TAIL_THREADS, 3)
tail_kernel(TailArgs a, float s2h, float s2w, float sch, float scw, int vec, int planes) {
  extern __shared__ __align__(16) float sm[];
  float* s1 = sm;                                 // [planes][R1_H][R1_W]; the xc patch aliases its start
  float* sc = sm;                                 // [XC_H*XC_W][KP]   (dead once r2 is built)
  float* s2 = s1 + planes * R1_PLANE;             // [R2_H*R2_W][KP]
  TailTables* tb = reinterpret_cast<TailTables*>(s2 + R2_H * R2_W * KP);

  const int Ho = 2 * a.h2, Wo = 2 * a.w2;
  const int tiles_x = (Wo + OT_W - 1) / OT_W;
  const int n = blockIdx.y;
  const int a0 = (blockIdx.x / tiles_x) * TROWS;    // first thread-row (units of 4 output rows)
  const int b0 = (blockIdx.x % tiles_x) * TCOLS;
  const int t = threadIdx.x;
  const int tr = t / TCOLS, tc = t % TCOLS;

  // ---- patch extents (uniform): r1 patch (i,j) <-> global (clamp(2*a0-1+i), clamp(2*b0-1+j))
  const int g1y_min = clampi(2 * a0 - 1, 0, a.h2 - 1), g1y_max = clampi(2 * a0 - 1 + R1_H - 1, 0, a.h2 - 1);
  const int g1x_min = clampi(2 * b0 - 1, 0, a.w2 - 1), g1x_max = clampi(2 * b0 - 1 + R1_W - 1, 0, a.w2 - 1);
  int y2a, y2b, x2a, x2b, tmp;
  float f0, f1;
  bilinear_coord(g1y_min, s2h, a.h4, y2a, tmp, f0, f1);
  bilinear_coord(g1y_max, s2h, a.h4, tmp, y2b, f0, f1);
  bilinear_coord(g1x_min, s2w, a.w4, x2a, tmp, f0, f1);
  bilinear_coord(g1x_max, s2w, a.w4, tmp, x2b, f0, f1);
  const int r2h = y2b - y2a + 1, r2w = x2b - x2a + 1;
  int yca, ycb, xca, xcb;
  bilinear_coord(y2a, sch, a.hc, yca, tmp, f0, f1);
  bilinear_coord(y2b, sch, a.hc, tmp, ycb, f0, f1);
  bilinear_coord(x2a, scw, a.wc, xca, tmp, f0, f1);
  bilinear_coord(x2b, scw, a.wc, tmp, xcb, f0, f1);
  const int rch = ycb - yca + 1, rcw = xcb - xca + 1;

  // ---- per-tile tables (one thread per row / column)
  if (t < R1_H) {
    const int y = clampi(2 * a0 - 1 + t, 0, a.h2 - 1);
    int i0, i1; float l0, l1;
    bilinear_coord(y, s2h, a.h4, i0, i1, l0, l1);
    tb->r1_gy[t] = y; tb->r1_y0[t] = i0 - y2a; tb->r1_y1[t] = i1 - y2a; tb->r1_wy[t] = l1;
  } else if (t >= 32 && t < 32 + R1_W) {
    const int j = t - 32;
    const int x = clampi(2 * b0 - 1 + j, 0, a.w2 - 1);
    int i0, i1; float l0, l1;
    bilinear_coord(x, s2w, a.w4, i0, i1, l0, l1);
    tb->r1_gx[j] = x; tb->r1_x0[j] = i0 - x2a; tb->r1_x1[j] = i1 - x2a; tb->r1_wx[j] = l1;
  } else if (t >= 72 && t < 72 + R2_H) {
    const int i = t - 72;
    if (i < r2h) {
      int i0, i1; float l0, l1;
      bilinear_coord(y2a + i, sch, a.hc, i0, i1, l0, l1);
      tb->r2_y0[i] = i0 - yca; tb->r2_y1[i] = i1 - yca; tb->r2_wy[i] = l1;
    }
  } else if (t >= 96 && t < 96 + R2_W) {
    const int j = t - 96;
    if (j < r2w) {
      int i0, i1; float l0, l1;
      bilinear_coord(x2a + j, scw, a.wc, i0, i1, l0, l1);
      tb->r2_x0[j] = i0 - xca; tb->r2_x1[j] = i1 - xca; tb->r2_wx[j] = l1;
    }
  }

  const T* xc = reinterpret_cast<const T*>(a.xc) + (int64_t)n * a.hc * a.wc * a.xc_ld;
  const T* hx2 = reinterpret_cast<const T*>(a.hx2) + (int64_t)n * a.h4 * a.w4 * a.hx2_ld;
  const T* hx1 = reinterpret_cast<const T*>(a.hx1) + (int64_t)n * a.h2 * a.w2 * a.hx1_ld;

  // per-thread output coordinates and vertical/horizontal weights (exact x2 stage)
  const int oy0 = 4 * (a0 + tr), ox0 = 4 * (b0 + tc);
  float wy1[4], wx1[4], wy0[4], wx0[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    int i0, i1; float l0, l1;
    bilinear_coord(min(oy0 + r, Ho - 1), 0.5f, a.h2, i0, i1, l0, l1); wy1[r] = l1; wy0[r] = 1.f - l1;
    bilinear_coord(min(ox0 + r, Wo - 1), 0.5f, a.w2, i0, i1, l0, l1); wx1[r] = l1; wx0[r] = 1.f - l1;
  }
  float best[4][4];
  int bidx[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) { best[r][c] = -INFINITY; bidx[r][c] = 0; }

  for (int k0 = 0; k0 < a.K; k0 += KP) {
    const int kc = min(KP, a.K - k0);
    const int ng = (kc + 7) >> 3;                 // 8-class groups in this pass
    // ---- A: xc patch -> sc[pixel][KP]
    {
      const int npix = rch * rcw;
      for (int i = t; i < npix * ng; i += TAIL_THREADS) {
        const int g = i / npix, p = i - g * npix;
        const int y = yca + p / rcw, x = xca + p % rcw;
        float v[8];
        load_group(xc + ((int64_t)y * a.wc + x) * a.xc_ld, k0 + 8 * g, a.K, vec, v);
        float4* d = reinterpret_cast<float4*>(sc + p * KP + 8 * g);
        d[0] = make_float4(v[0], v[1], v[2], v[3]);
        d[1] = make_float4(v[4], v[5], v[6], v[7]);
      }
    }
    __syncthreads();
    // ---- B: r2 = hx2 + up(xc) -> s2[pixel][KP]
    {
      const int npix = r2h * r2w;
      for (int i = t; i < npix * ng; i += TAIL_THREADS) {
        const int g = i / npix, p = i - g * npix;
        const int py = p / r2w, px = p - py * r2w;
        float v[8];
        load_group(hx2 + ((int64_t)(y2a + py) * a.w4 + (x2a + px)) * a.hx2_ld, k0 + 8 * g, a.K, vec, v);
        const int yy0 = tb->r2_y0[py], yy1 = tb->r2_y1[py], xx0 = tb->r2_x0[px], xx1 = tb->r2_x1[px];
        add_bilerp8(v, sc + (yy0 * rcw + xx0) * KP + 8 * g, sc + (yy0 * rcw + xx1) * KP + 8 * g,
                    sc + (yy1 * rcw + xx0) * KP + 8 * g, sc + (yy1 * rcw + xx1) * KP + 8 * g, tb->r2_wx[px], tb->r2_wy[py]);
        float4* d = reinterpret_cast<float4*>(s2 + p * KP + 8 * g);
        d[0] = make_float4(v[0], v[1], v[2], v[3]);
        d[1] = make_float4(v[4], v[5], v[6], v[7]);
      }
    }
    __syncthreads();
    // ---- C: r1 = hx1 + up(r2) on the (clamped) 18 x 34 patch -> s1[k][i][j]  (overwrites sc)
    for (int i = t; i < R1_PLANE * ng; i += TAIL_THREADS) {
      const int g = i / R1_PLANE, p = i - g * R1_PLANE;
      const int pi = p / R1_W, pj = p - pi * R1_W;
      float v[8];
      load_group(hx1 + ((int64_t)tb->r1_gy[pi] * a.w2 + tb->r1_gx[pj]) * a.hx1_ld, k0 + 8 * g, a.K, vec, v);
      const int yy0 = tb->r1_y0[pi], yy1 = tb->r1_y1[pi], xx0 = tb->r1_x0[pj], xx1 = tb->r1_x1[pj];
      add_bilerp8(v, s2 + (yy0 * r2w + xx0) * KP + 8 * g, s2 + (yy0 * r2w + xx1) * KP + 8 * g,
                  s2 + (yy1 * r2w + xx0) * KP + 8 * g, s2 + (yy1 * r2w + xx1) * KP + 8 * g, tb->r1_wx[pj], tb->r1_wy[pi]);
#pragma unroll
      for (int c = 0; c < 8; ++c)
        if (8 * g + c < planes) s1[(8 * g + c) * R1_PLANE + p] = v[c];
    }
    __syncthreads();
    // ---- D: 4x4 outputs per thread from a 4x4 r1 window; window (wi,wj) = patch (2*tr+wi, 2*tc+wj)
    for (int k = 0; k < kc; ++k) {
      const float* base = s1 + k * R1_PLANE + (2 * tr) * R1_W + 2 * tc;
      float hrow[4][4];   // horizontally interpolated: [window row][output col]
#pragma unroll
      for (int wi = 0; wi < 4; ++wi) {
        const float2 p = *reinterpret_cast<const float2*>(base + wi * R1_W);
        const float2 q = *reinterpret_cast<const float2*>(base + wi * R1_W + 2);
        // output col c uses window cols (0,1),(1,2),(1,2),(2,3)
        hrow[wi][0] = fmaf(p.y, wx1[0], p.x * wx0[0]);
        hrow[wi][1] = fmaf(q.x, wx1[1], p.y * wx0[1]);
        hrow[wi][2] = fmaf(q.x, wx1[2], p.y * wx0[2]);
        hrow[wi][3] = fmaf(q.y, wx1[3], q.x * wx0[3]);
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float o[4];
        o[0] = fmaf(hrow[1][c], wy1[0], hrow[0][c] * wy0[0]);
        o[1] = fmaf(hrow[2][c], wy1[1], hrow[1][c] * wy0[1]);
        o[2] = fmaf(hrow[2][c], wy1[2], hrow[1][c] * wy0[2]);
        o[3] = fmaf(hrow[3][c], wy1[3], hrow[2][c] * wy0[3]);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          if (o[r] > best[r][c]) { best[r][c] = o[r]; bidx[r][c] = k0 + k; }   // strict > : first max wins
          hrow[r][c] = o[r];          // reuse as the logits staging for the optional store below
        }
      }
      if (a.logits) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int oy = oy0 + r;
          if (oy < Ho) {
            float* lp = a.logits + (((int64_t)n * a.K + k0 + k) * Ho + oy) * Wo + ox0;
            if (ox0 + 3 < Wo && (Wo & 3) == 0) {
              *reinterpret_cast<float4*>(lp) = make_float4(hrow[r][0], hrow[r][1], hrow[r][2], hrow[r][3]);
            } else {
#pragma unroll
              for (int c = 0; c < 4; ++c) if (ox0 + c < Wo) lp[c] = hrow[r][c];
            }
          }
        }
      }
    }
    __syncthreads();
  }

  // ---- labels
  TP* pred = reinterpret_cast<TP*>(a.pred) + (int64_t)n * Ho * Wo;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int oy = oy0 + r;
    if (oy >= Ho) continue;
    if (sizeof(TP) == 1 && ox0 + 3 < Wo && (Wo & 3) == 0) {
      uchar4 u = make_uchar4((unsigned char)bidx[r][0], (unsigned char)bidx[r][1], (unsigned char)bidx[r][2],
                             (unsigned char)bidx[r][3]);
      *reinterpret_cast<uchar4*>(reinterpret_cast<uint8_t*>(pred) + (int64_t)oy * Wo + ox0) = u;
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (ox0 + c < Wo) pred[(int64_t)oy * Wo + ox0 + c] = (TP)bidx[r][c];
    }
  }
}


// ---------------------------------------------------------------------------------------------
// tail2: the LAST stage only, for callers that want the full-resolution logits.  The ladder kernel (ladder_tc.cu) has
// already formed r1 = head_x1 + up(head_x2 + up(x_c)) at half resolution (fp16, NHWC, pixel stride `ld`); the outputs
// are its exact x2 bilinear upsample as fp32 NCHW logits and their argmax_k (decode_head.py:373-378 + base.py:187-188).
//
// CTA = 128 threads = 8 x 16 thread grid, 32 x 64 output tile, 18 x 34 r1 patch (clamped halo) staged in
// shared memory as fp32 CLASS PAIRS: plane[kp][row][col] = float2(class 2kp, class 2kp+1), so one LDS.128
// brings two columns of two classes and the interpolation runs on packed f32x2 FMAs (FMUL2/FFMA2: two
// classes per instruction, each lane an IEEE fp32 op - same rounding as the scalar formula of tail_kernel).
// Per thread and class pair: 8 LDS.128, 16 + 16 packed ops for a 4 x 4 output block, then the running
// (max, index) update per class in ascending order with strict `>` (torch.argmax's first-max rule).
constexpr int T2_PAIRS = 12;                // class pairs per pass (24 classes)
constexpr int T2_PLANE = R1_H * R1_W;       // float2 elements per pair plane

__device__ __forceinline__ float2 lerp2(float2 a, float2 b, float2 w0, float2 w1) {
  return __ffma2_rn(b, w1, __fmul2_rn(a, w0));   // b*w1 + a*w0 per lane: fmaf(b, w1, a*w0)
}

template <typename TP>
__global__ void __launch_bounds__(TAIL_THREADS, 4)
tail2_kernel(const __half* __restrict__ r1, int ld, int K, int h2, int w2, TP* __restrict__ pred_base,
             float* __restrict__ logits, int planes) {
  extern __shared__ __align__(16) float2 sp[];          // [pairs][R1_H][R1_W]
  const int Ho = 2 * h2, Wo = 2 * w2;
  const int tiles_x = (Wo + OT_W - 1) / OT_W;
  const int n = blockIdx.y;
  const int a0 = (blockIdx.x / tiles_x) * TROWS, b0 = (blockIdx.x % tiles_x) * TCOLS;
  const int t = threadIdx.x;
  const int tr = t / TCOLS, tc = t % TCOLS;
  const __half* src = r1 + (int64_t)n * h2 * w2 * ld;

  const int oy0 = 4 * (a0 + tr), ox0 = 4 * (b0 + tc);
  // exact x2, align_corners=False: even outputs take (1/4, 3/4) of window (i-1, i), odd ones (3/4, 1/4) of
  // (i, i+1).  At the image border ATen clamps the source index (weights 1/0); the patch below replicates the
  // border pixel instead, and fma(a, 3/4, a/4) == a exactly, so constant weights give the same bits.
  const float2 q14 = make_float2(0.25f, 0.25f), q34 = make_float2(0.75f, 0.75f);
  float best[4][4];
  int bidx[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) { best[r][c] = -INFINITY; bidx[r][c] = 0; }

  for (int k0 = 0; k0 < K; k0 += 2 * T2_PAIRS) {
    const int kc = min(2 * T2_PAIRS, K - k0);
    const int ng = (kc + 7) >> 3;                 // 8-class groups in this pass (source is padded to 8)
    if (k0) __syncthreads();
    // ---- stage the patch: item = (pixel, 8-class group); consecutive lanes read consecutive 16 B
    for (int i = t; i < T2_PLANE * ng; i += TAIL_THREADS) {
      const int p = i / ng, g = i - p * ng;
      const int pi = p / R1_W, pj = p - pi * R1_W;
      const int gy = clampi(2 * a0 - 1 + pi, 0, h2 - 1), gx = clampi(2 * b0 - 1 + pj, 0, w2 - 1);
      float v[8];
      load8(src + ((int64_t)gy * w2 + gx) * ld + k0 + 8 * g, v);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (4 * g + j < planes) sp[(4 * g + j) * T2_PLANE + p] = make_float2(v[2 * j], v[2 * j + 1]);
    }
    __syncthreads();
    const int npair = (kc + 1) >> 1;
    for (int kp = 0; kp < npair; ++kp) {
      const float2* base = sp + kp * T2_PLANE + (2 * tr) * R1_W + 2 * tc;
      float2 hrow[4][4];   // [window row][output col], lanes = (class k, class k+1)
#pragma unroll
      for (int wi = 0; wi < 4; ++wi) {
        const float4 pq = *reinterpret_cast<const float4*>(base + wi * R1_W);       // window cols 0, 1
        const float4 rs = *reinterpret_cast<const float4*>(base + wi * R1_W + 2);   // window cols 2, 3
        const float2 c0 = make_float2(pq.x, pq.y), c1 = make_float2(pq.z, pq.w);
        const float2 c2 = make_float2(rs.x, rs.y), c3 = make_float2(rs.z, rs.w);
        // output col c uses window cols (0,1),(1,2),(1,2),(2,3)
        hrow[wi][0] = lerp2(c0, c1, q14, q34);
        hrow[wi][1] = lerp2(c1, c2, q34, q14);
        hrow[wi][2] = lerp2(c1, c2, q14, q34);
        hrow[wi][3] = lerp2(c2, c3, q34, q14);
      }
      const int k = k0 + 2 * kp;
      const bool two = (2 * kp + 1) < kc;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float2 o[4];
        o[0] = lerp2(hrow[0][c], hrow[1][c], q14, q34);
        o[1] = lerp2(hrow[1][c], hrow[2][c], q34, q14);
        o[2] = lerp2(hrow[1][c], hrow[2][c], q14, q34);
        o[3] = lerp2(hrow[2][c], hrow[3][c], q34, q14);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          if (o[r].x > best[r][c]) { best[r][c] = o[r].x; bidx[r][c] = k; }        // strict > : first max wins
          if (two && o[r].y > best[r][c]) { best[r][c] = o[r].y; bidx[r][c] = k + 1; }
          hrow[r][c] = o[r];          // staging for the logits store
        }
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        if (half && !two) break;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int oy = oy0 + r;
          if (oy < Ho) {
            float* lp = logits + (((int64_t)n * K + k + half) * Ho + oy) * Wo + ox0;
            float vv[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) vv[c] = half ? hrow[r][c].y : hrow[r][c].x;
            if (ox0 + 3 < Wo && (Wo & 3) == 0) {
              *reinterpret_cast<float4*>(lp) = make_float4(vv[0], vv[1], vv[2], vv[3]);
            } else {
#pragma unroll
              for (int c = 0; c < 4; ++c) if (ox0 + c < Wo) lp[c] = vv[c];
            }
          }
        }
      }
    }
  }

  TP* pred = pred_base + (int64_t)n * Ho * Wo;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int oy = oy0 + r;
    if (oy >= Ho) continue;
    if (sizeof(TP) == 1 && ox0 + 3 < Wo && (Wo & 3) == 0) {
      uchar4 u = make_uchar4((unsigned char)bidx[r][0], (unsigned char)bidx[r][1], (unsigned char)bidx[r][2],
                             (unsigned char)bidx[r][3]);
      *reinterpret_cast<uchar4*>(reinterpret_cast<uint8_t*>(pred) + (int64_t)oy * Wo + ox0) = u;
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (ox0 + c < Wo) pred[(int64_t)oy * Wo + ox0 + c] = (TP)bidx[r][c];
    }
  }
}

}  // namespace

int launch_tail(const TailArgs& a, cudaStream_t st) {
  if (a.K < 1 || a.K > 255) return fail(LEDB200_EINVAL, "tail: K must be in [1,255]");
  if (a.N < 1 || a.h2 < 1 || a.w2 < 1 || a.h4 < 1 || a.w4 < 1 || a.hc < 1 || a.wc < 1)
    return fail(LEDB200_EINVAL, "tail: empty input");
  const float s2h = (float)a.h4 / (float)a.h2, s2w = (float)a.w4 / (float)a.w2;
  const float sch = (float)a.hc / (float)a.h4, scw = (float)a.wc / (float)a.w4;
  // patch capacities (worst case over tiles): span*scale + 2 rows/cols
  auto fits = [](int span, float scale, int cap, int level) {
    const int need = (int)(span * scale) + 3;
    return (need < level ? need : level) <= cap;
  };
  if (!fits(R1_H, s2h, R2_H, a.h4) || !fits(R1_W, s2w, R2_W, a.w4) || !fits(R2_H, sch, XC_H, a.hc) ||
      !fits(R2_W, scw, XC_W, a.wc))
    return fail(LEDB200_EINVAL,
                "tail: level sizes must follow the reference ladder (each level ~2x the one below); got "
                "hc/h4/h2 = " + std::to_string(a.hc) + "/" + std::to_string(a.h4) + "/" + std::to_string(a.h2));
  const int Ho = 2 * a.h2, Wo = 2 * a.w2;
  const int esz = (int)dtype_size(a.dtype);
  const bool vec = (a.xc_ld % 8 == 0) && (a.hx2_ld % 8 == 0) && (a.hx1_ld % 8 == 0) &&
                   ((uintptr_t)a.xc % (8 * esz) == 0) && ((uintptr_t)a.hx2 % (8 * esz) == 0) &&
                   ((uintptr_t)a.hx1 % (8 * esz) == 0) && (a.xc_ld >= (a.K + 7) / 8 * 8) &&
                   (a.hx2_ld >= (a.K + 7) / 8 * 8) && (a.hx1_ld >= (a.K + 7) / 8 * 8);
  dim3 grid(ceil_div(Wo, OT_W) * ceil_div(Ho, OT_H), a.N);
  const int planes = a.K < KP ? a.K : KP;
  // the xc patch aliases the r1 planes; make sure it fits even for tiny K
  const size_t s1_floats = std::max<size_t>((size_t)planes * R1_PLANE, (size_t)XC_H * XC_W * KP);
  const int planes_alloc = (int)((s1_floats + R1_PLANE - 1) / R1_PLANE);
  const size_t smem = ((size_t)planes_alloc * R1_PLANE + (size_t)R2_H * R2_W * KP) * sizeof(float) + sizeof(TailTables);
#define LEDB_TAIL(T, TP)                                                                              \
  do {                                                                                                \
    LEDB_CUDA_OK(cudaFuncSetAttribute(tail_kernel<T, TP>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                      (int)smem));                                                    \
    tail_kernel<T, TP><<<grid, TAIL_THREADS, smem, st>>>(a, s2h, s2w, sch, scw, vec ? 1 : 0, planes_alloc); \
  } while (0)
  if (a.dtype == LEDB200_BF16 && a.pred_dtype == LEDB200_U8) LEDB_TAIL(__nv_bfloat16, uint8_t);
  else if (a.dtype == LEDB200_BF16 && a.pred_dtype == LEDB200_I64) LEDB_TAIL(__nv_bfloat16, int64_t);
  else if (a.dtype == LEDB200_F32 && a.pred_dtype == LEDB200_U8) LEDB_TAIL(float, uint8_t);
  else if (a.dtype == LEDB200_F32 && a.pred_dtype == LEDB200_I64) LEDB_TAIL(float, int64_t);
  else return fail(LEDB200_EINVAL, "tail: dtype must be F32/BF16 and pred dtype U8/I64");
#undef LEDB_TAIL
  LEDB_LAUNCH_OK("tail_kernel");
  return LEDB200_OK;
}

int launch_tail2(const Tail2Args& a, cudaStream_t st) {
  if (a.K < 1 || a.K > 255) return fail(LEDB200_EINVAL, "tail2: K must be in [1,255]");
  if (a.N < 1 || a.h2 < 1 || a.w2 < 1) return fail(LEDB200_EINVAL, "tail2: empty input");
  if (!a.logits) return fail(LEDB200_EINVAL, "tail2: logits output required (labels alone come from the ladder kernel)");
  if (a.ld % 8 || a.ld < (a.K + 7) / 8 * 8 || ((uintptr_t)a.r1 & 15))
    return fail(LEDB200_EINVAL, "tail2: r1 must be fp16 NHWC with a 16-byte aligned pixel stride covering K rounded up to 8");
  if (a.pred_dtype != LEDB200_U8 && a.pred_dtype != LEDB200_I64)
    return fail(LEDB200_EINVAL, "tail2: pred dtype must be U8 or I64");
  const int Ho = 2 * a.h2, Wo = 2 * a.w2;
  dim3 grid(ceil_div(Wo, OT_W) * ceil_div(Ho, OT_H), a.N);
  const int pairs = std::min(T2_PAIRS, (a.K + 1) / 2);
  const size_t smem = (size_t)pairs * T2_PLANE * sizeof(float2);
#define LEDB_TAIL2(TP)                                                                                   \
  do {                                                                                                   \
    LEDB_CUDA_OK(cudaFuncSetAttribute(tail2_kernel<TP>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                      (int)smem));                                                       \
    tail2_kernel<TP><<<grid, TAIL_THREADS, smem, st>>>(a.r1, a.ld, a.K, a.h2, a.w2, (TP*)a.pred, a.logits, pairs); \
  } while (0)
  if (a.pred_dtype == LEDB200_U8) LEDB_TAIL2(uint8_t); else LEDB_TAIL2(int64_t);
#undef LEDB_TAIL2
  LEDB_LAUNCH_OK("tail2_kernel");
  return LEDB200_OK;
}

}  // namespace ledb
