// GETB block (global-local window attention + MLP) behind a small handle API (SURVEY section 8a row B6).
//
// Replaces GETBBlock.forward (mmseg/models/backbones/UNetFormer_GETB.py:221-226) with GlobalLocalAttention
// (:97-206) and Mlp (:79-94), eval mode (drop / drop_path are identities):
//   z   = BN1(x)
//   qkv = conv1x1(reflect_pad(z)) ; per (8x8 window, head): softmax(q k^T * scale + rel_pos_bias) v   (:171-190)
//   a   = crop(attn) ; o = avgpool_8x1(reflect-pad-bottom(a)) + avgpool_1x8(reflect-pad-right(a)) + z   (:196-199)
//   y   = x + conv1x1(BN(depthwise8x8(reflect_pad_(0,1,0,1)(o))))                                       (:200-204)
//   out = y + fc2(ReLU6(fc1(BN2(y))))                                                                   (:225)
// Lowering:
//   * all four 1x1 convolutions (qkv, proj, fc1, fc2 = 97 % of the FLOPs) go through the SAME launchers the
//     trunk uses: tcgen05 implicit GEMM in bf16 mode, CUDA-core fp32 in the parity mode.  BN1 is folded into
//     the qkv weights and BN2 into fc1 by the caller; a 1x1 conv commutes with reflect padding (a gather),
//     so qkv is computed on the UNPADDED map and the attention kernel gathers padded tokens by reflection;
//     the two residual adds and ReLU6 ride in the conv epilogues.
//   * getb_attn_kernel  : one thread per query token, K/V of the (window, head) in shared memory, scores in
//                         registers (64 keys), fp32 softmax.
//   * getb_pool_kernel  : the two 8-tap box filters with the reference's reflect (index H -> H-2) / zero
//                         (AvgPool2d padding 3, count_include_pad) borders, + BN1(x).
//   * getb_dw_kernel    : depthwise 8x8 over the virtually reflect-padded map, zero padding 3, + folded BN.
#include <vector>

#include "kernels.h"

namespace ledb {
namespace {

constexpr int WS = 8, NTOK = WS * WS;

struct GetbDev {
  PackedConv conv[4];   // qkv, proj, fc1, fc2
  float *n1s = nullptr, *n1b = nullptr, *relb = nullptr, *wdw = nullptr, *dws = nullptr, *dwb = nullptr;
};

}  // namespace
}  // namespace ledb

struct ledb200_getb {
  int dim = 0, heads = 0, hidden = 0, dtype = 0;
  ledb::GetbDev d;
  void* ws = nullptr;
  size_t ws_bytes = 0;
};

namespace ledb {
namespace {

__device__ __forceinline__ int reflect(int t, int size) { return t < size ? t : 2 * (size - 1) - t; }

struct AttnArgs {
  const void* qkv;     // [N,H,W,3C]
  void* attn;          // [N,H,W,C]
  const float* relb;   // [heads][64][64]
  int N, H, W, C, heads, hh, ww;
  float scale;
};

template <typename T, int D, int HPB>
__global__ void __launch_bounds__(NTOK * HPB) getb_attn_kernel(AttnArgs a) {
  __shared__ float sk[HPB][NTOK][D];
  __shared__ float sv[HPB][NTOK][D];
  const int tok = threadIdx.x, hl = threadIdx.y;
  const int head = blockIdx.y * HPB + hl;
  int win = blockIdx.x;
  const int wx = win % a.ww; win /= a.ww;
  const int wy = win % a.hh;
  const int n = win / a.hh;
  const int yp = wy * WS + tok / WS, xp = wx * WS + tok % WS;        // padded coordinates of this token
  const int ys = reflect(yp, a.H), xs = reflect(xp, a.W);            // source pixel (1x1 conv commutes with the pad)
  const T* px = reinterpret_cast<const T*>(a.qkv) + (((int64_t)n * a.H + ys) * a.W + xs) * (3 * a.C) + head * D;
  float q[D];
  if (D >= 8) {
#pragma unroll
    for (int j = 0; j < D; j += 8) {
      float t[8];
      load8(px + j, q + j);
      load8(px + a.C + j, t);
#pragma unroll
      for (int e = 0; e < 8; ++e) sk[hl][tok][j + e] = t[e];
      load8(px + 2 * a.C + j, t);
#pragma unroll
      for (int e = 0; e < 8; ++e) sv[hl][tok][j + e] = t[e];
    }
  } else {
#pragma unroll
    for (int j = 0; j < D; ++j) {
      q[j] = to_f32(px[j]);
      sk[hl][tok][j] = to_f32(px[a.C + j]);
      sv[hl][tok][j] = to_f32(px[2 * a.C + j]);
    }
  }
  __syncthreads();
  const float* rb = a.relb + ((int64_t)head * NTOK + tok) * NTOK;
  float s[NTOK];
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < NTOK; ++j) {
    float acc = 0.f;
#pragma unroll
    for (int e = 0; e < D; ++e) acc = fmaf(q[e], sk[hl][j][e], acc);
    s[j] = fmaf(acc, a.scale, __ldg(rb + j));
    mx = fmaxf(mx, s[j]);
  }
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < NTOK; ++j) { s[j] = __expf(s[j] - mx); sum += s[j]; }
  float o[D];
#pragma unroll
  for (int e = 0; e < D; ++e) o[e] = 0.f;
#pragma unroll
  for (int j = 0; j < NTOK; ++j) {
#pragma unroll
    for (int e = 0; e < D; ++e) o[e] = fmaf(s[j], sv[hl][j][e], o[e]);
  }
  if (yp >= a.H || xp >= a.W) return;                                 // crop (:194)
  const float inv = 1.f / sum;
  T* dst = reinterpret_cast<T*>(a.attn) + (((int64_t)n * a.H + yp) * a.W + xp) * a.C + head * D;
  if (D >= 8) {
#pragma unroll
    for (int j = 0; j < D; j += 8) {
      float t[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) t[e] = o[j + e] * inv;
      store8(dst + j, t);
    }
  } else {
#pragma unroll
    for (int j = 0; j < D; ++j) dst[j] = from_f32<T>(o[j] * inv);
  }
}

struct PoolLocalArgs {
  const void* attn;    // [N,H,W,C]
  const void* x;       // [N,H,W,C]
  void* out;           // [N,H,W,C]
  const float *n1s, *n1b;
  int N, H, W, C;
};

template <typename T>
__global__ void __launch_bounds__(256) getb_pool_kernel(PoolLocalArgs a) {
  const int cgs = a.C / 8;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.N * a.H * a.W * cgs) return;
  const int cg = (int)(idx % cgs);
  int64_t p = idx / cgs;
  const int x = (int)(p % a.W); p /= a.W;
  const int y = (int)(p % a.H);
  const int n = (int)(p / a.H);
  const T* A = reinterpret_cast<const T*>(a.attn) + (int64_t)n * a.H * a.W * a.C + cg * 8;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < WS; ++k) {
    // rows: F.pad(attn, (0,0,0,1), reflect) then AvgPool2d((8,1), padding (3,0)): padded row t in [0, H] else zero
    const int t = y - (WS / 2 - 1) + k;
    if (t >= 0 && t <= a.H) {
      float v[8];
      load8(A + ((int64_t)reflect(t, a.H) * a.W + x) * a.C, v);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += v[e];
    }
    const int u = x - (WS / 2 - 1) + k;
    if (u >= 0 && u <= a.W) {
      float v[8];
      load8(A + ((int64_t)y * a.W + reflect(u, a.W)) * a.C, v);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += v[e];
    }
  }
  const int64_t off = (((int64_t)n * a.H + y) * a.W + x) * a.C + cg * 8;
  float xv[8];
  load8(reinterpret_cast<const T*>(a.x) + off, xv);
#pragma unroll
  for (int e = 0; e < 8; ++e)
    acc[e] = acc[e] * (1.f / WS) + fmaf(xv[e], a.n1s[cg * 8 + e], a.n1b[cg * 8 + e]);
  store8(reinterpret_cast<T*>(a.out) + off, acc);
}

struct DwArgs {
  const void* in;      // [N,H,W,C]
  void* out;           // [N,H,W,C]
  const float *w;      // [ws*ws][C]  (tap major)
  const float *s, *b;  // folded BN
  int N, H, W, C;
};

template <typename T>
__global__ void __launch_bounds__(256) getb_dw_kernel(DwArgs a) {
  const int cgs = a.C / 8;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.N * a.H * a.W * cgs) return;
  const int cg = (int)(idx % cgs);
  int64_t p = idx / cgs;
  const int x = (int)(p % a.W); p /= a.W;
  const int y = (int)(p % a.H);
  const int n = (int)(p / a.H);
  const T* I = reinterpret_cast<const T*>(a.in) + (int64_t)n * a.H * a.W * a.C + cg * 8;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int i = 0; i < WS; ++i) {
    const int u = y - (WS - 1) / 2 + i;            // row of the (H+1) x (W+1) reflect-padded map; outside: zero
    if (u < 0 || u > a.H) continue;
    const int ur = reflect(u, a.H);
#pragma unroll
    for (int j = 0; j < WS; ++j) {
      const int v = x - (WS - 1) / 2 + j;
      if (v < 0 || v > a.W) continue;
      float t[8], w[8];
      load8(I + ((int64_t)ur * a.W + reflect(v, a.W)) * a.C, t);
      load8(a.w + (i * WS + j) * a.C + cg * 8, w);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] = fmaf(t[e], w[e], acc[e]);
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = fmaf(acc[e], a.s[cg * 8 + e], a.b[cg * 8 + e]);
  store8(reinterpret_cast<T*>(a.out) + (((int64_t)n * a.H + y) * a.W + x) * a.C + cg * 8, acc);
}

// 1x1 conv weights [Cout][Cin] fp32 (host) -> both device layouts + padded bias
int pack_conv1x1(PackedConv& c, const float* w, const float* bias, int cin, int cout) {
  c.cin = cin; c.cout = cout;
  return pack_conv(w, bias, nullptr, nullptr, c);
}

int conv1x1(const ledb200_getb& g, int i, const void* in, void* out, const void* res, int relu, int N, int H, int W,
            cudaStream_t st) {
  const PackedConv& c = g.d.conv[i];
  ConvArgs a = conv_args(c, N, H, W);
  a.in = in; a.in_dtype = g.dtype; a.in_sc = 1; a.in_sw = c.cin; a.in_sh = (int64_t)W * c.cin; a.in_sn = (int64_t)H * W * c.cin;
  a.out = out; a.out_dtype = g.dtype; a.out_ld = c.cout; a.res = res; a.res_ld = c.cout; a.relu = relu;
  return launch_conv(a, 0, "getb_forward", st);
}

template <typename T, int D>
int launch_attn_d(const AttnArgs& a, cudaStream_t st) {
  const dim3 grid((unsigned)(a.N * a.hh * a.ww), 1);
  if constexpr (D <= 16) {
    if (a.heads % 4 == 0) {
      getb_attn_kernel<T, D, 4><<<dim3(grid.x, a.heads / 4), dim3(NTOK, 4), 0, st>>>(a);
      LEDB_LAUNCH_OK("getb_attn_kernel");
      return LEDB200_OK;
    }
  }
  if (a.heads % 2 == 0) {
    getb_attn_kernel<T, D, 2><<<dim3(grid.x, a.heads / 2), dim3(NTOK, 2), 0, st>>>(a);
  } else {
    getb_attn_kernel<T, D, 1><<<dim3(grid.x, a.heads), dim3(NTOK, 1), 0, st>>>(a);
  }
  LEDB_LAUNCH_OK("getb_attn_kernel");
  return LEDB200_OK;
}

template <typename T>
int launch_attn(const AttnArgs& a, int d, cudaStream_t st) {
  switch (d) {
    case 4: return launch_attn_d<T, 4>(a, st);
    case 8: return launch_attn_d<T, 8>(a, st);
    case 16: return launch_attn_d<T, 16>(a, st);
    case 32: return launch_attn_d<T, 32>(a, st);
    default: return fail(LEDB200_EINVAL, "getb: head dimension must be 4, 8, 16 or 32");
  }
}

}  // namespace
}  // namespace ledb

using namespace ledb;

extern "C" {

// floats of the host parameter block of ledb200_getb_create (window 8):
//   w_qkv[3C][C], b_qkv[3C], n1_scale[C], n1_shift[C], rel_bias[heads][64][64], w_dw[C][64], dw_scale[C],
//   dw_shift[C], w_proj[C][C], w_fc1[hidden][C], b_fc1[hidden], w_fc2[C][hidden], b_fc2[C]
int64_t ledb200_getb_param_floats(int32_t dim, int32_t heads, int32_t hidden) {
  const int64_t C = dim;
  return 3 * C * C + 3 * C + 2 * C + (int64_t)heads * NTOK * NTOK + C * NTOK + 2 * C + C * C + (int64_t)hidden * C + hidden +
         C * hidden + C;
}

int ledb200_getb_create(int32_t dim, int32_t heads, int32_t hidden, int32_t window, int32_t dtype,
                        const float* params, ledb200_getb** out) {
  if (!params || !out) return fail(LEDB200_EINVAL, "getb_create: null pointer");
  if (window != WS) return fail(LEDB200_EINVAL, "getb_create: window_size must be 8");
  if (dtype != LEDB200_F32 && dtype != LEDB200_BF16) return fail(LEDB200_EINVAL, "getb_create: dtype must be F32 or BF16");
  if (dim < 8 || dim % 8 || heads < 1 || dim % heads) return fail(LEDB200_EINVAL, "getb_create: dim must be a multiple of 8 and of num_heads");
  const int d = dim / heads;
  if (d != 4 && d != 8 && d != 16 && d != 32) return fail(LEDB200_EINVAL, "getb_create: dim / num_heads must be 4, 8, 16 or 32");
  if (hidden < 8 || hidden % 8) return fail(LEDB200_EINVAL, "getb_create: hidden must be a multiple of 8");
  ledb200_getb* g = new ledb200_getb();
  g->dim = dim; g->heads = heads; g->hidden = hidden; g->dtype = dtype;
  const int C = dim;
  const float* p = params;
  const float* w_qkv = p; p += 3 * C * C;
  const float* b_qkv = p; p += 3 * C;
  const float* n1s = p; p += C;
  const float* n1b = p; p += C;
  const float* relb = p; p += heads * NTOK * NTOK;
  const float* w_dw = p; p += C * NTOK;
  const float* dws = p; p += C;
  const float* dwb = p; p += C;
  const float* w_proj = p; p += C * C;
  const float* w_fc1 = p; p += hidden * C;
  const float* b_fc1 = p; p += hidden;
  const float* w_fc2 = p; p += C * hidden;
  const float* b_fc2 = p;
  std::vector<float> dwt((size_t)NTOK * C);                 // tap-major depthwise weights
  for (int c = 0; c < C; ++c)
    for (int t = 0; t < NTOK; ++t) dwt[(size_t)t * C + c] = w_dw[(size_t)c * NTOK + t];
  int rc = pack_conv1x1(g->d.conv[0], w_qkv, b_qkv, C, 3 * C);
  if (!rc) rc = pack_conv1x1(g->d.conv[1], w_proj, nullptr, C, C);
  if (!rc) rc = pack_conv1x1(g->d.conv[2], w_fc1, b_fc1, C, hidden);
  if (!rc) rc = pack_conv1x1(g->d.conv[3], w_fc2, b_fc2, hidden, C);
  if (!rc) rc = upload(n1s, C * 4, (void**)&g->d.n1s);
  if (!rc) rc = upload(n1b, C * 4, (void**)&g->d.n1b);
  if (!rc) rc = upload(relb, (size_t)heads * NTOK * NTOK * 4, (void**)&g->d.relb);
  if (!rc) rc = upload(dwt, &g->d.wdw);
  if (!rc) rc = upload(dws, C * 4, (void**)&g->d.dws);
  if (!rc) rc = upload(dwb, C * 4, (void**)&g->d.dwb);
  if (rc) { ledb200_getb_destroy(g); return rc; }
  *out = g;
  return LEDB200_OK;
}

int ledb200_getb_destroy(ledb200_getb* g) {
  if (!g) return LEDB200_OK;
  for (PackedConv& c : g->d.conv) free_conv(c);
  cudaFree(g->d.n1s); cudaFree(g->d.n1b); cudaFree(g->d.relb); cudaFree(g->d.wdw); cudaFree(g->d.dws); cudaFree(g->d.dwb);
  cudaFree(g->ws);
  delete g;
  return LEDB200_OK;
}

int ledb200_getb_forward(ledb200_getb* g, const void* x, void* out, int32_t N, int32_t H, int32_t W, void* stream) {
  if (!g || !x || !out) return fail(LEDB200_EINVAL, "getb_forward: null pointer");
  if (N < 1 || H < 2 || W < 2) return fail(LEDB200_EINVAL, "getb_forward: needs N >= 1 and H, W >= 2 (reflect padding)");
  const int padh = (WS - H % WS) % WS, padw = (WS - W % WS) % WS;
  if (padh >= H || padw >= W)
    return fail(LEDB200_EINVAL, "getb_forward: reflect padding to a multiple of 8 must be smaller than the input (as in F.pad)");
  cudaStream_t st = (cudaStream_t)stream;
  const int C = g->dim;
  const size_t es = dtype_size(g->dtype);
  const size_t npix = (size_t)N * H * W;
  // workspace: qkv (3C) | attn (C) | o (C) | t (C) | y (C) | hidden  -- qkv is dead once attn exists, so the
  // MLP's hidden map reuses qkv's space when it fits
  const size_t hid_units = (size_t)g->hidden > 3 * (size_t)C ? g->hidden : 3 * (size_t)C;
  const size_t need = npix * es * (hid_units + 4 * (size_t)C);
  if (need > g->ws_bytes) {          // grows on a new (larger) shape only; steady state allocates nothing
    LEDB_CUDA_OK(cudaStreamSynchronize(st));
    cudaFree(g->ws); g->ws = nullptr; g->ws_bytes = 0;
    LEDB_CUDA_OK(cudaMalloc(&g->ws, need));
    g->ws_bytes = need;
  }
  char* base = reinterpret_cast<char*>(g->ws);
  void* qkv = base;                                   // also the MLP hidden map later
  void* attn = base + npix * es * hid_units;
  void* o = reinterpret_cast<char*>(attn) + npix * es * C;
  void* t = reinterpret_cast<char*>(o) + npix * es * C;
  void* y = reinterpret_cast<char*>(t) + npix * es * C;
  int rc = conv1x1(*g, 0, x, qkv, nullptr, 0, N, H, W, st);
  if (rc) return rc;
  AttnArgs aa;
  aa.qkv = qkv; aa.attn = attn; aa.relb = g->d.relb; aa.N = N; aa.H = H; aa.W = W; aa.C = C; aa.heads = g->heads;
  aa.hh = (H + padh) / WS; aa.ww = (W + padw) / WS;
  aa.scale = 1.f / sqrtf((float)(C / g->heads));
  rc = g->dtype == LEDB200_BF16 ? launch_attn<__nv_bfloat16>(aa, C / g->heads, st) : launch_attn<float>(aa, C / g->heads, st);
  if (rc) return rc;
  const unsigned eb = (unsigned)ceil_div64((int64_t)npix * (C / 8), 256);
  PoolLocalArgs pa{attn, x, o, g->d.n1s, g->d.n1b, N, H, W, C};
  DwArgs da{o, t, g->d.wdw, g->d.dws, g->d.dwb, N, H, W, C};
  if (g->dtype == LEDB200_BF16) {
    getb_pool_kernel<__nv_bfloat16><<<eb, 256, 0, st>>>(pa);
    LEDB_LAUNCH_OK("getb_pool_kernel");
    getb_dw_kernel<__nv_bfloat16><<<eb, 256, 0, st>>>(da);
  } else {
    getb_pool_kernel<float><<<eb, 256, 0, st>>>(pa);
    LEDB_LAUNCH_OK("getb_pool_kernel");
    getb_dw_kernel<float><<<eb, 256, 0, st>>>(da);
  }
  LEDB_LAUNCH_OK("getb_dw_kernel");
  rc = conv1x1(*g, 1, t, y, x, 0, N, H, W, st);                 // y = x + proj(...)
  if (rc) return rc;
  rc = conv1x1(*g, 2, y, qkv, nullptr, 2, N, H, W, st);         // hidden = ReLU6(fc1(BN2(y)))   (BN2 folded)
  if (rc) return rc;
  return conv1x1(*g, 3, qkv, out, y, 0, N, H, W, st);           // out = y + fc2(hidden)
}

}  // extern "C"
