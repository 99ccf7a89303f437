// The packed inference convolution (PackedConv, kernels.h): the one owner of the device weight layouts conv_direct and
// conv_tc read, of the weight upload, of the ConvArgs fields that follow from the layer, and of the choice between the
// tensor-core and the CUDA-core kernel.  Host code only.
#include <algorithm>

#include "kernels.h"

namespace ledb {

int upload(const void* host, size_t bytes, void** dev) {
  void* p = nullptr;
  LEDB_CUDA_OK(cudaMalloc(&p, std::max<size_t>(bytes, 16)));
  const cudaError_t e = cudaMemcpy(p, host, bytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(p); return fail(LEDB200_ECUDA, std::string("weight upload: ") + cudaGetErrorString(e)); }
  *dev = p;
  return LEDB200_OK;
}

int upload_kmajor_bf16(const float* w_oihw, const float* scale, int cin, int cout, int k, __nv_bfloat16** dev) {
  const int taps = k * k;
  std::vector<__nv_bfloat16> wt((size_t)conv_tc_pad(cout) * taps * cin, __float2bfloat16(0.f));
  for (int o = 0; o < cout; ++o) {
    const float s = scale ? scale[o] : 1.f;
    for (int c = 0; c < cin; ++c)
      for (int t = 0; t < taps; ++t) wt[((size_t)o * taps + t) * cin + c] = __float2bfloat16(w_oihw[((size_t)o * cin + c) * taps + t] * s);
  }
  return upload(wt, dev);
}

int pack_conv(const float* w_oihw, const float* bias, const float* scale, const float* shift, PackedConv& c) {
  const int taps = c.k * c.k;
  c.cout_pad16 = (c.cout + 15) / 16 * 16;
  c.cout_pad_tc = conv_tc_pad(c.cout);
  std::vector<float> wd((size_t)taps * c.cin * c.cout_pad16, 0.f);
  std::vector<float> bv(std::max(c.cout_pad16, c.cout_pad_tc), 0.f);
  for (int o = 0; o < c.cout; ++o) {
    const float s = scale ? scale[o] : 1.f;
    if (bias) bv[o] = bias[o] * s;
    if (shift) bv[o] += shift[o];
    for (int ci = 0; ci < c.cin; ++ci)
      for (int t = 0; t < taps; ++t) wd[((size_t)t * c.cin + ci) * c.cout_pad16 + o] = w_oihw[((size_t)o * c.cin + ci) * taps + t] * s;
  }
  int rc = upload(wd, &c.w_direct);
  if (!rc) rc = upload_kmajor_bf16(w_oihw, scale, c.cin, c.cout, c.k, &c.w_tc);
  if (!rc && (bias || shift)) rc = upload(bv, &c.bias);
  return rc;
}

void free_conv(PackedConv& c) {
  cudaFree(c.w_direct); cudaFree(c.w_tc); cudaFree(c.bias); cudaFree(c.pre_scale); cudaFree(c.pre_shift);
  c.w_direct = nullptr; c.w_tc = nullptr; c.bias = c.pre_scale = c.pre_shift = nullptr;
}

ConvArgs conv_args(const PackedConv& c, int N, int H, int W) {
  ConvArgs a;
  a.bias = c.bias; a.w_direct = c.w_direct; a.w_tc = c.w_tc; a.cout_pad16 = c.cout_pad16; a.cout_pad_tc = c.cout_pad_tc;
  a.pre_scale = c.pre_scale; a.pre_shift = c.pre_shift;
  a.N = N; a.H = H; a.W = W; a.Cin = c.cin; a.Cout = c.cout;
  a.ksize = c.k; a.stride = c.stride; a.pad = c.k / 2; a.dil = 1;
  a.Ho = (H + 2 * a.pad - c.k) / c.stride + 1; a.Wo = (W + 2 * a.pad - c.k) / c.stride + 1;
  return a;
}

bool conv_use_tc(const ConvArgs& a, int backend) { return backend != 1 && conv_tc_eligible(a); }

int launch_conv(const ConvArgs& a, int backend, const char* who, cudaStream_t st) {
  const bool tc = conv_use_tc(a, backend);
  if (backend == 2 && !tc) return fail(LEDB200_EINVAL, std::string(who) + ": shape not eligible for the tcgen05 path");
  return tc ? launch_conv_tc(a, st) : launch_conv_direct(a, st);
}

}  // namespace ledb
