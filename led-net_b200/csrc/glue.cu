// Layer-level C-ABI operators for module compositions outside the R0 engine plan (the LED wiring, led_variant.py):
//   * conv layer handles: one ConvModule with its BatchNorm folded on the host, weights resident on the device in both
//     layouts, forward = ONE launch of conv_tc (bf16, eligible shapes) or conv_direct - the same launchers as the engine;
//   * depthwise 3x3 (STDCModule's stride-2 downsample, mmseg/models/backbones/stdc.py:52-61);
//   * AvgPool2d (count_include_pad=True) / global average, bilinear resize (align_corners=False), add(+ReLU).
// All tensors NHWC fp32 or bf16 with explicit pixel strides, so a producer can write straight into a channel slice of a
// concat buffer (STDCModule.forward_cat, DAPPM) and no concat copy exists.
#include <vector>

#include "kernels.h"

using namespace ledb;

struct ledb200_conv_layer {
  PackedConv c;                               // depthwise: only cin .. stride, bias
  int depthwise = 0;
  float* w_dw = nullptr;                      // depthwise: [9][C]
};

namespace ledb {
namespace {

constexpr int kT = 256;
inline unsigned grid_for(int64_t work) {
  int64_t b = ceil_div64(work, kT);
  const int64_t cap = 148 * 16;
  return (unsigned)(b < cap ? (b < 1 ? 1 : b) : cap);
}

template <typename T>
__global__ void __launch_bounds__(kT)
dwconv3x3_kernel(const T* __restrict__ in, T* __restrict__ out, const float* __restrict__ w, const float* __restrict__ bias,
                 int N, int H, int W, int C, int Ho, int Wo, int stride, int relu, int in_ld, int out_ld) {
  const int cg = C / 8;
  const int64_t total = (int64_t)N * Ho * Wo * cg;
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int g = (int)(i % cg);
    int64_t p = i / cg;
    const int ox = (int)(p % Wo), oy = (int)((p / Wo) % Ho), n = (int)(p / ((int64_t)Wo * Ho));
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = bias ? bias[g * 8 + c] : 0.f;
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int y = oy * stride - 1 + kh;
      if (y < 0 || y >= H) continue;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int x = ox * stride - 1 + kw;
        if (x < 0 || x >= W) continue;
        float v[8], wv[8];
        load8(in + (((int64_t)n * H + y) * W + x) * in_ld + g * 8, v);
        load8(w + (kh * 3 + kw) * C + g * 8, wv);
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[c] = fmaf(v[c], wv[c], acc[c]);
      }
    }
    if (relu) {
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[c] = fmaxf(acc[c], 0.f);
    }
    store8(out + p * out_ld + g * 8, acc);
  }
}

template <typename T>
__global__ void __launch_bounds__(kT)
avgpool2d_kernel(const T* __restrict__ in, T* __restrict__ out, int N, int H, int W, int C, int Ho, int Wo, int k, int s,
                 int pd, int in_ld, int out_ld) {
  const int cg = C / 8;
  const int64_t total = (int64_t)N * Ho * Wo * cg;
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int g = (int)(i % cg);
    int64_t p = i / cg;
    const int ox = (int)(p % Wo), oy = (int)((p / Wo) % Ho), n = (int)(p / ((int64_t)Wo * Ho));
    int y0, y1, x0, x1;
    float inv;
    if (k == 0) { y0 = 0; y1 = H; x0 = 0; x1 = W; inv = 1.f / (float)(H * W); }
    else {
      y0 = oy * s - pd; y1 = y0 + k; x0 = ox * s - pd; x1 = x0 + k;
      const int hend = min(y1, H + pd), wend = min(x1, W + pd);       // ATen pool_size: window clipped to the PADDED extent
      inv = 1.f / (float)((hend - y0) * (wend - x0));
      y0 = max(y0, 0); x0 = max(x0, 0); y1 = min(y1, H); x1 = min(x1, W);
    }
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int y = y0; y < y1; ++y)
      for (int x = x0; x < x1; ++x) {
        float v[8];
        load8(in + (((int64_t)n * H + y) * W + x) * in_ld + g * 8, v);
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[c] += v[c];
      }
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] *= inv;
    store8(out + p * out_ld + g * 8, acc);
  }
}

template <typename T>
__global__ void __launch_bounds__(kT)
resize_kernel(const T* __restrict__ in, T* __restrict__ out, int N, int h, int w, int H, int W, int C, int in_ld, int out_ld,
              float sh, float sw) {
  const int cg = C / 8;
  const int64_t total = (int64_t)N * H * W * cg;
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int g = (int)(i % cg);
    int64_t p = i / cg;
    const int x = (int)(p % W), y = (int)((p / W) % H), n = (int)(p / ((int64_t)W * H));
    int y0, y1, x0, x1;
    float ly0, ly1, lx0, lx1;
    bilinear_coord(y, sh, h, y0, y1, ly0, ly1);
    bilinear_coord(x, sw, w, x0, x1, lx0, lx1);
    const T* s = in + (int64_t)n * h * w * in_ld + g * 8;
    float a[8], b[8], c[8], d[8], o[8];
    load8(s + ((int64_t)y0 * w + x0) * in_ld, a); load8(s + ((int64_t)y0 * w + x1) * in_ld, b);
    load8(s + ((int64_t)y1 * w + x0) * in_ld, c); load8(s + ((int64_t)y1 * w + x1) * in_ld, d);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float r0 = fmaf(b[j], lx1, a[j] * lx0);
      const float r1 = fmaf(d[j], lx1, c[j] * lx0);
      o[j] = fmaf(r1, ly1, r0 * ly0);
    }
    store8(out + p * out_ld + g * 8, o);
  }
}

template <typename T>
__global__ void __launch_bounds__(kT)
add_relu_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ out, int64_t npix, int C, int a_ld, int b_ld,
                int out_ld, int relu) {
  const int cg = C / 8;
  const int64_t total = npix * cg;
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int g = (int)(i % cg);
    const int64_t p = i / cg;
    float v[8];
    load8(a + p * a_ld + g * 8, v);
    if (b) {
      float u[8];
      load8(b + p * b_ld + g * 8, u);
#pragma unroll
      for (int c = 0; c < 8; ++c) v[c] += u[c];
    }
    if (relu) {
#pragma unroll
      for (int c = 0; c < 8; ++c) v[c] = fmaxf(v[c], 0.f);
    }
    store8(out + p * out_ld + g * 8, v);
  }
}

bool dt_ok(int dt) { return dt == LEDB200_F32 || dt == LEDB200_BF16; }

}  // namespace
}  // namespace ledb

extern "C" {

int ledb200_conv_layer_create(const float* weight, const float* bias, const float* pre_scale, const float* pre_shift,
                              int32_t Cin, int32_t Cout, int32_t ksize, int32_t stride, int32_t groups,
                              ledb200_conv_layer** out) {
  if (!weight || !out) return fail(LEDB200_EINVAL, "conv_layer_create: null pointer");
  if (ksize != 1 && ksize != 3) return fail(LEDB200_EINVAL, "conv_layer_create: ksize must be 1 or 3");
  if (stride != 1 && stride != 2) return fail(LEDB200_EINVAL, "conv_layer_create: stride must be 1 or 2");
  if (Cin < 1 || Cout < 1) return fail(LEDB200_EINVAL, "conv_layer_create: empty layer");
  if ((pre_scale == nullptr) != (pre_shift == nullptr)) return fail(LEDB200_EINVAL, "conv_layer_create: pre_scale and pre_shift come together");
  const bool dw = groups != 1;
  if (dw && (groups != Cin || Cin != Cout || ksize != 3 || Cin % 8 || pre_scale))
    return fail(LEDB200_EINVAL, "conv_layer_create: grouped convolutions are depthwise 3x3 (groups == Cin == Cout, Cin % 8 == 0)");
  ledb200_conv_layer* L = new ledb200_conv_layer();
  L->c.cin = Cin; L->c.cout = Cout; L->c.k = ksize; L->c.stride = stride; L->depthwise = dw ? 1 : 0;
  int rc = LEDB200_OK;
  if (dw) {
    std::vector<float> w((size_t)9 * Cin);                      // weight [C][1][3][3] -> [tap][C]
    for (int c = 0; c < Cin; ++c)
      for (int t = 0; t < 9; ++t) w[(size_t)t * Cin + c] = weight[(size_t)c * 9 + t];
    rc = upload(w, &L->w_dw);
    if (!rc && bias) rc = upload(bias, Cout * 4, (void**)&L->c.bias);
  } else {
    rc = pack_conv(weight, bias, nullptr, nullptr, L->c);
  }
  if (!rc && pre_scale) {
    rc = upload(pre_scale, Cin * 4, (void**)&L->c.pre_scale);
    if (!rc) rc = upload(pre_shift, Cin * 4, (void**)&L->c.pre_shift);
  }
  if (rc) { ledb200_conv_layer_destroy(L); return rc; }
  *out = L;
  return LEDB200_OK;
}

int ledb200_conv_layer_destroy(ledb200_conv_layer* L) {
  if (!L) return LEDB200_OK;
  free_conv(L->c);
  cudaFree(L->w_dw);
  delete L;
  return LEDB200_OK;
}

int ledb200_conv_layer_forward(ledb200_conv_layer* L, const void* in, void* out, const void* residual, int32_t dtype, int32_t N,
                               int32_t H, int32_t W, int32_t in_ld, int32_t out_ld, int32_t res_ld, int32_t relu,
                               int32_t backend, void* stream) {
  if (!L || !in || !out) return fail(LEDB200_EINVAL, "conv_layer_forward: null pointer");
  if (!dt_ok(dtype)) return fail(LEDB200_EINVAL, "conv_layer_forward: dtype must be F32 or BF16");
  if (N < 1 || H < 1 || W < 1) return fail(LEDB200_EINVAL, "conv_layer_forward: empty input");
  const PackedConv& c = L->c;
  if (in_ld == 0) in_ld = c.cin;
  if (out_ld == 0) out_ld = c.cout;
  if (res_ld == 0) res_ld = c.cout;
  if (in_ld < c.cin || out_ld < c.cout || (residual && res_ld < c.cout))
    return fail(LEDB200_EINVAL, "conv_layer_forward: pixel stride smaller than the channel count");
  cudaStream_t st = (cudaStream_t)stream;
  ConvArgs a = conv_args(c, N, H, W);
  if (L->depthwise) {
    if (residual) return fail(LEDB200_EINVAL, "conv_layer_forward: the depthwise layer takes no residual");
    if (in_ld % 8 || out_ld % 8) return fail(LEDB200_EINVAL, "conv_layer_forward: depthwise pixel strides must be multiples of 8");
    const int64_t total = (int64_t)N * a.Ho * a.Wo * (c.cin / 8);
    if (dtype == LEDB200_BF16)
      dwconv3x3_kernel<__nv_bfloat16><<<grid_for(total), kT, 0, st>>>((const __nv_bfloat16*)in, (__nv_bfloat16*)out, L->w_dw, c.bias, N,
                                                                      H, W, c.cin, a.Ho, a.Wo, c.stride, relu, in_ld, out_ld);
    else
      dwconv3x3_kernel<float><<<grid_for(total), kT, 0, st>>>((const float*)in, (float*)out, L->w_dw, c.bias, N, H, W, c.cin, a.Ho,
                                                              a.Wo, c.stride, relu, in_ld, out_ld);
    LEDB_LAUNCH_OK("dwconv3x3_kernel");
    return LEDB200_OK;
  }
  a.in = in; a.in_dtype = dtype; a.in_sc = 1; a.in_sw = in_ld; a.in_sh = (int64_t)W * in_ld; a.in_sn = (int64_t)H * W * in_ld;
  a.out = out; a.out_dtype = dtype; a.out_ld = out_ld; a.res = residual; a.res_ld = res_ld; a.relu = relu;
  return launch_conv(a, backend, "conv_layer_forward", st);
}

int ledb200_conv_layer_forward_image(ledb200_conv_layer* L, const void* img, int32_t img_layout, void* out, int32_t dtype, int32_t N,
                                     int32_t H, int32_t W, int32_t out_ld, int32_t relu, void* stream) {
  if (!L || !img || !out) return fail(LEDB200_EINVAL, "conv_layer_forward_image: null pointer");
  if (L->depthwise || L->c.cin != 3 || L->c.k != 3) return fail(LEDB200_EINVAL, "conv_layer_forward_image: a dense 3x3 layer on 3 input channels");
  if (!dt_ok(dtype)) return fail(LEDB200_EINVAL, "conv_layer_forward_image: output dtype must be F32 or BF16");
  if (img_layout != LEDB200_IMG_NCHW_F32) return fail(LEDB200_EINVAL, "conv_layer_forward_image: image layout must be NCHW fp32");
  if (out_ld == 0) out_ld = L->c.cout;
  ConvArgs a = conv_args(L->c, N, H, W);
  const int64_t HW = (int64_t)H * W;
  a.in = img; a.in_dtype = LEDB200_F32; a.in_sn = 3 * HW; a.in_sc = HW; a.in_sh = W; a.in_sw = 1;
  a.out = out; a.out_dtype = dtype; a.out_ld = out_ld; a.relu = relu;
  cudaStream_t st = (cudaStream_t)stream;
  if (stem_tc_eligible(a)) return launch_stem_tc(a, st);       // bf16 output, stride 2, Cout 16 / 32: tensor cores
  return launch_conv_direct(a, st);
}

int ledb200_avgpool2d(const void* in, void* out, int32_t dtype, int32_t N, int32_t H, int32_t W, int32_t C, int32_t k, int32_t s,
                      int32_t p, int32_t in_ld, int32_t out_ld, void* stream) {
  if (!in || !out) return fail(LEDB200_EINVAL, "avgpool2d: null buffer");
  if (!dt_ok(dtype) || C < 8 || C % 8) return fail(LEDB200_EINVAL, "avgpool2d: F32 / BF16, C a multiple of 8");
  if (in_ld == 0) in_ld = C;
  if (out_ld == 0) out_ld = C;
  if (in_ld % 8 || out_ld % 8 || in_ld < C || out_ld < C) return fail(LEDB200_EINVAL, "avgpool2d: bad pixel stride");
  if (k < 0 || (k > 0 && (s < 1 || p < 0 || 2 * p > k))) return fail(LEDB200_EINVAL, "avgpool2d: bad window (pad must be at most half the kernel)");
  const int Ho = k ? (H + 2 * p - k) / s + 1 : 1, Wo = k ? (W + 2 * p - k) / s + 1 : 1;
  if (Ho < 1 || Wo < 1) return fail(LEDB200_EINVAL, "avgpool2d: window larger than the padded input");
  const int64_t total = (int64_t)N * Ho * Wo * (C / 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == LEDB200_BF16)
    avgpool2d_kernel<__nv_bfloat16><<<grid_for(total), kT, 0, st>>>((const __nv_bfloat16*)in, (__nv_bfloat16*)out, N, H, W, C, Ho, Wo, k,
                                                                    s, p, in_ld, out_ld);
  else
    avgpool2d_kernel<float><<<grid_for(total), kT, 0, st>>>((const float*)in, (float*)out, N, H, W, C, Ho, Wo, k, s, p, in_ld, out_ld);
  LEDB_LAUNCH_OK("avgpool2d_kernel");
  return LEDB200_OK;
}

int ledb200_resize_bilinear(const void* in, void* out, int32_t dtype, int32_t N, int32_t h, int32_t w, int32_t H, int32_t W, int32_t C,
                            int32_t in_ld, int32_t out_ld, void* stream) {
  if (!in || !out) return fail(LEDB200_EINVAL, "resize_bilinear: null buffer");
  if (!dt_ok(dtype) || C < 8 || C % 8) return fail(LEDB200_EINVAL, "resize_bilinear: F32 / BF16, C a multiple of 8");
  if (h < 1 || w < 1 || H < 1 || W < 1 || N < 1) return fail(LEDB200_EINVAL, "resize_bilinear: empty tensor");
  if (in_ld == 0) in_ld = C;
  if (out_ld == 0) out_ld = C;
  if (in_ld % 8 || out_ld % 8 || in_ld < C || out_ld < C) return fail(LEDB200_EINVAL, "resize_bilinear: bad pixel stride");
  const int64_t total = (int64_t)N * H * W * (C / 8);
  cudaStream_t st = (cudaStream_t)stream;
  const float sh = (float)h / (float)H, sw = (float)w / (float)W;
  if (dtype == LEDB200_BF16)
    resize_kernel<__nv_bfloat16><<<grid_for(total), kT, 0, st>>>((const __nv_bfloat16*)in, (__nv_bfloat16*)out, N, h, w, H, W, C, in_ld,
                                                                 out_ld, sh, sw);
  else
    resize_kernel<float><<<grid_for(total), kT, 0, st>>>((const float*)in, (float*)out, N, h, w, H, W, C, in_ld, out_ld, sh, sw);
  LEDB_LAUNCH_OK("resize_kernel");
  return LEDB200_OK;
}

int ledb200_add_relu(const void* a, const void* b, void* out, int32_t dtype, int64_t npix, int32_t C, int32_t a_ld, int32_t b_ld,
                     int32_t out_ld, int32_t relu, void* stream) {
  if (!a || !out) return fail(LEDB200_EINVAL, "add_relu: null buffer");
  if (!dt_ok(dtype) || C < 8 || C % 8) return fail(LEDB200_EINVAL, "add_relu: F32 / BF16, C a multiple of 8");
  if (a_ld == 0) a_ld = C;
  if (b_ld == 0) b_ld = C;
  if (out_ld == 0) out_ld = C;
  if (a_ld % 8 || b_ld % 8 || out_ld % 8) return fail(LEDB200_EINVAL, "add_relu: bad pixel stride");
  const int64_t total = npix * (C / 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == LEDB200_BF16)
    add_relu_kernel<__nv_bfloat16><<<grid_for(total), kT, 0, st>>>((const __nv_bfloat16*)a, (const __nv_bfloat16*)b, (__nv_bfloat16*)out,
                                                                   npix, C, a_ld, b_ld, out_ld, relu);
  else
    add_relu_kernel<float><<<grid_for(total), kT, 0, st>>>((const float*)a, (const float*)b, (float*)out, npix, C, a_ld, b_ld, out_ld, relu);
  LEDB_LAUNCH_OK("add_relu_kernel");
  return LEDB200_OK;
}

// ---- the whole DAPPM as a handle: parameters folded and resident, scratch grown on demand; forward = the two launches
//      of dappm.cu (bf16, <= 8 tiles of 16 x 8 pixels per image)
struct ledb200_dappm {
  int C = 0, P = 0, Cout = 0;
  std::vector<void*> allocs;
  const float *a_scale[5] = {}, *b_scale[5] = {}, *a_proc[4] = {}, *b_proc[4] = {}, *a_comp = nullptr, *b_comp = nullptr,
              *a_sc = nullptr, *b_sc = nullptr;
  const __nv_bfloat16 *w_scale[5] = {}, *w_proc[4] = {}, *w_comp = nullptr, *w_sc = nullptr;
  const float *bias_scale[5] = {}, *bias_proc[4] = {}, *bias_comp = nullptr, *bias_sc = nullptr;
  void* scratch = nullptr; size_t scratch_bytes = 0;
};

namespace {
int dappm_upload_conv(ledb200_dappm* D, const ledb200_preact_conv& pc, int cin, int cout, int k, const float** a, const float** b,
                      const __nv_bfloat16** w, const float** bias) {
  if (!pc.weight || !pc.bn_scale || !pc.bn_shift) return fail(LEDB200_EINVAL, "dappm_create: null parameter");
  float *da = nullptr, *db = nullptr, *dbias = nullptr;
  __nv_bfloat16* dw = nullptr;
  int rc = upload(pc.bn_scale, cin * 4, (void**)&da);
  if (!rc) { D->allocs.push_back(da); rc = upload(pc.bn_shift, cin * 4, (void**)&db); }
  if (!rc) { D->allocs.push_back(db); rc = upload_kmajor_bf16(pc.weight, nullptr, cin, cout, k, &dw); }
  if (!rc) D->allocs.push_back(dw);
  if (!rc && pc.bias) {
    rc = upload(pc.bias, cout * 4, (void**)&dbias);
    if (!rc) D->allocs.push_back(dbias);
  }
  *a = da; *b = db; *w = dw; *bias = dbias;
  return rc;
}
}  // namespace

int ledb200_dappm_destroy(ledb200_dappm* D) {
  if (!D) return LEDB200_OK;
  for (void* p : D->allocs) cudaFree(p);
  cudaFree(D->scratch);
  delete D;
  return LEDB200_OK;
}

int ledb200_dappm_create(int32_t C, int32_t P, int32_t Cout, const ledb200_preact_conv* scales5, const ledb200_preact_conv* processes4,
                         const ledb200_preact_conv* compression, const ledb200_preact_conv* shortcut, ledb200_dappm** out) {
  if (!scales5 || !processes4 || !compression || !shortcut || !out) return fail(LEDB200_EINVAL, "dappm_create: null pointer");
  DappmArgs probe;
  probe.N = 1; probe.H = 8; probe.W = 8; probe.C = C; probe.P = P; probe.Cout = Cout; probe.out_ld = Cout;
  if (!dappm_eligible(probe)) return fail(LEDB200_EINVAL, "dappm_create: the fused DAPPM needs C % 64 == 0, ppm channels = out channels = 128");
  ledb200_dappm* D = new ledb200_dappm();
  D->C = C; D->P = P; D->Cout = Cout;
  int rc = LEDB200_OK;
  for (int i = 0; i < 5 && !rc; ++i) rc = dappm_upload_conv(D, scales5[i], C, P, 1, &D->a_scale[i], &D->b_scale[i], &D->w_scale[i], &D->bias_scale[i]);
  for (int i = 0; i < 4 && !rc; ++i) rc = dappm_upload_conv(D, processes4[i], P, P, 3, &D->a_proc[i], &D->b_proc[i], &D->w_proc[i], &D->bias_proc[i]);
  if (!rc) rc = dappm_upload_conv(D, *compression, 5 * P, Cout, 1, &D->a_comp, &D->b_comp, &D->w_comp, &D->bias_comp);
  if (!rc) rc = dappm_upload_conv(D, *shortcut, C, Cout, 1, &D->a_sc, &D->b_sc, &D->w_sc, &D->bias_sc);
  if (rc) { ledb200_dappm_destroy(D); return rc; }
  *out = D;
  return LEDB200_OK;
}

int ledb200_dappm_eligible(int32_t dtype, int32_t N, int32_t H, int32_t W, int32_t C, int32_t P, int32_t Cout) {
  DappmArgs a;
  a.N = N; a.H = H; a.W = W; a.C = C; a.P = P; a.Cout = Cout; a.out_ld = Cout;
  return (dtype == LEDB200_BF16 && dappm_eligible(a)) ? 1 : 0;
}

int ledb200_dappm_forward(ledb200_dappm* D, const void* x, void* out, int32_t dtype, int32_t N, int32_t H, int32_t W, void* stream) {
  if (!D || !x || !out) return fail(LEDB200_EINVAL, "dappm_forward: null pointer");
  if (dtype != LEDB200_BF16) return fail(LEDB200_EINVAL, "dappm_forward: the fused DAPPM runs bf16 tensors");
  DappmArgs a;
  a.x = x; a.N = N; a.H = H; a.W = W; a.C = D->C; a.P = D->P; a.Cout = D->Cout; a.out = out; a.out_ld = D->Cout;
  if (!dappm_eligible(a)) return fail(LEDB200_EINVAL, "dappm_forward: shape not eligible (more than 8 tiles of 16 x 8 pixels per image)");
  static const int ks[3] = {5, 9, 17}, ss[3] = {2, 4, 8}, ps[3] = {2, 4, 8};
  size_t need = 0, off[6];
  for (int i = 0; i < 4; ++i) {
    a.pool_k[i] = i < 3 ? ks[i] : 0; a.pool_s[i] = i < 3 ? ss[i] : 1; a.pool_p[i] = i < 3 ? ps[i] : 0;
    a.sh[i] = i < 3 ? (H + 2 * ps[i] - ks[i]) / ss[i] + 1 : 1;
    a.sw[i] = i < 3 ? (W + 2 * ps[i] - ks[i]) / ss[i] + 1 : 1;
    if (a.sh[i] < 1 || a.sw[i] < 1) return fail(LEDB200_EINVAL, "dappm_forward: feature map smaller than a pooling window allows");
    off[i] = need; need += ((size_t)N * a.sh[i] * a.sw[i] * D->P * 2 + 255) / 256 * 256;
  }
  for (int i = 4; i < 6; ++i) { off[i] = need; need += ((size_t)N * H * W * D->P * 2 + 255) / 256 * 256; }
  if (need > D->scratch_bytes) {
    LEDB_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    cudaFree(D->scratch); D->scratch = nullptr; D->scratch_bytes = 0;
    LEDB_CUDA_OK(cudaMalloc(&D->scratch, need));
    D->scratch_bytes = need;
  }
  char* base = (char*)D->scratch;
  for (int i = 0; i < 4; ++i) {
    a.s[i] = base + off[i];
    a.a_scale[i] = D->a_scale[i + 1]; a.b_scale[i] = D->b_scale[i + 1]; a.w_scale[i] = D->w_scale[i + 1]; a.bias_scale[i] = D->bias_scale[i + 1];
    a.a_proc[i] = D->a_proc[i]; a.b_proc[i] = D->b_proc[i]; a.w_proc[i] = D->w_proc[i]; a.bias_proc[i] = D->bias_proc[i];
  }
  a.t0 = base + off[4]; a.t1 = base + off[5];
  a.a_s0 = D->a_scale[0]; a.b_s0 = D->b_scale[0]; a.w_s0 = D->w_scale[0]; a.bias_s0 = D->bias_scale[0];
  a.a_sc = D->a_sc; a.b_sc = D->b_sc; a.w_sc = D->w_sc; a.bias_sc = D->bias_sc;
  a.a_comp = D->a_comp; a.b_comp = D->b_comp; a.w_comp = D->w_comp; a.bias_comp = D->bias_comp;
  return launch_dappm(a, (cudaStream_t)stream);
}

}  // extern "C"
