// Launcher declarations shared by the engine (engine.cu), the layer handles (glue.cu, getb.cu, ...) and the raw C-ABI
// ops (api.cu), and the one packed-weight format of their inference convolutions (PackedConv: fp32 Cout padded to 16 for
// the CUDA cores, bf16 K-major with conv_tc_pad(Cout) = 32 or a multiple of 64 rows for the tensor cores).
#pragma once
#include <vector>

#include "common.cuh"

namespace ledb {

// cudaMalloc + host-to-device copy of `bytes` (at least 16 are allocated).  On failure nothing stays allocated.
int upload(const void* host, size_t bytes, void** dev);
template <typename T>
int upload(const std::vector<T>& host, T** dev) { return upload(host.data(), host.size() * sizeof(T), (void**)dev); }

// One convolution layer (BN folded by the host side).  NHWC unless strides say otherwise.
struct ConvArgs {
  const void* in = nullptr;
  int in_dtype = LEDB200_F32;
  int64_t in_sn = 0, in_sh = 0, in_sw = 0, in_sc = 1;   // element strides of the input
  void* out = nullptr;          // may be null when only out2 is wanted
  int out_dtype = LEDB200_F32;
  int out_ld = 0;               // pixel stride (elements) of out
  void* out2 = nullptr;         // optional: relu(o2_scale*y + o2_shift), y = the primary output value (after `relu`)
  int out2_ld = 0;
  const float* o2_scale = nullptr;  // null => identity affine
  const float* o2_shift = nullptr;
  const void* res = nullptr;    // optional residual, same dtype as out
  int res_ld = 0;
  const float* bias = nullptr;  // [Cout] (device)
  int out_f16 = 0;              // tensor-core path only: `out` holds IEEE fp16 instead of bf16 (x_c, the ladder's bottom rung)
  const float* pre_scale = nullptr;  // [Cin] prologue affine (device), CUDA-core path only
  const float* pre_shift = nullptr;
  int pre_relu = 1;
  const float* w_direct = nullptr;         // [k*k][Cin][cout_pad16] fp32 (device)
  const __nv_bfloat16* w_tc = nullptr;     // [cout_pad_tc][k*k*Cin] bf16 (device), K-major
  const float* w_tc32 = nullptr;           // tf32 launches: the same matrix as fp32 words (tf32-rounded)
  int tf32 = 0;                            // 1 / 3: fp32 tensors through the kind::tf32 instantiations, passes per product (training, train.cu)
  // tf32 only - one parity class (sub_a, sub_b) of the data gradient of a stride-2 convolution: a stride-1 convolution over
  // dY whose taps are the filter rows / columns of that parity (offsets 0 / +1) and whose output pixel (i, j) is written to
  // (2 i + sub_a, 2 j + sub_b) of the [N, 2 Ho, 2 Wo] gradient.  w_tc32 then holds that class's own K-major matrix.
  int sub = 0, sub_a = 0, sub_b = 0;
  int cout_pad16 = 0;
  int cout_pad_tc = 0;
  int N = 0, H = 0, W = 0, Cin = 0, Ho = 0, Wo = 0, Cout = 0;
  int ksize = 3, stride = 1, pad = 1, dil = 1;
  int relu = 0;                  // 0 none, 1 ReLU, 2 ReLU6 (GETB Mlp, UNetFormer_GETB.py:80)
  // CUDA-core path only: the input is a zero-inserted view (factor in_up) of a real [Hr x Wr] tensor;
  // H/W are then the VIRTUAL extents.  Used for the data gradient of stride-2 convolutions (train.cu).
  int in_up = 1, Hr = 0, Wr = 0;
};

int launch_conv_direct(const ConvArgs& a, cudaStream_t st);
// tcgen05/TMEM implicit GEMM (conv_tc.cu).  conv_tc_eligible() says whether the shape fits.
bool conv_tc_eligible(const ConvArgs& a);
int conv_tc_pad(int cout);   // rows of the K-major bf16 weight matrix: 32 or a multiple of 64
int launch_conv_tc(const ConvArgs& a, cudaStream_t st);

// One inference convolution resident on the device (packed_conv.cu), BatchNorm already folded, in the layouts both
// kernels read.  k x k, padding k / 2, dilation 1.
struct PackedConv {
  int cin = 0, cout = 0, k = 1, stride = 1;
  float* w_direct = nullptr;        // [k*k][cin][cout_pad16] fp32 (conv_direct)
  __nv_bfloat16* w_tc = nullptr;    // [cout_pad_tc][k*k*cin] bf16, K-major (conv_tc)
  float* bias = nullptr;            // [max(cout_pad16, cout_pad_tc)]; null when the conv has neither a bias nor a shift
  float* pre_scale = nullptr;       // optional [cin] prologue BN + ReLU (CUDA-core path only)
  float* pre_shift = nullptr;
  int cout_pad16 = 0, cout_pad_tc = 0;
};
// Packs OIHW fp32 weights of c.cin -> c.cout, c.k for both kernels and uploads them.  Per output channel o the weights
// are scaled by scale[o] and the bias is bias[o] * scale[o] + shift[o]; any of bias / scale / shift may be null.
int pack_conv(const float* w_oihw, const float* bias, const float* scale, const float* shift, PackedConv& c);
// The bf16 K-major matrix alone: conv_tc_pad(cout) rows (zero beyond cout), uploaded to *dev.
int upload_kmajor_bf16(const float* w_oihw, const float* scale, int cin, int cout, int k, __nv_bfloat16** dev);
void free_conv(PackedConv& c);
// Weight / padding fields, Cin, Cout, ksize, stride, pad, dil, N, H, W, Ho and Wo of c on an N x H x W input.  The
// caller sets the tensors, their strides and dtypes, relu, residual and out2.
ConvArgs conv_args(const PackedConv& c, int N, int H, int W);
// backend 0 = tensor cores when conv_tc_eligible, else CUDA cores; 1 = CUDA cores; 2 = tensor cores.
bool conv_use_tc(const ConvArgs& a, int backend);
// Launches on the kernel conv_use_tc picks; backend 2 on a shape the tensor cores do not take fails with
// LEDB200_EINVAL ("<who>: shape not eligible for the tcgen05 path").
int launch_conv(const ConvArgs& a, int backend, const char* who, cudaStream_t st);

// One rung of the LEDHead logit ladder on the tensor cores (ladder_tc.cu):
//   rung : out[N,H,W,24] fp16 = relu(conv3x3(in) + bias) + up2(up)
//   final: pred[N,2H,2W] = argmax_k up2(relu(conv3x3(in) + bias) + up2(up))      (no rung tensor in HBM)
struct LadderArgs {
  const void* in = nullptr;                // [N,H,W,in_ld] bf16, already BN+ReLU pre-activated (Cin = 32 or 64)
  int in_ld = 0;
  const __nv_bfloat16* w_tc = nullptr;     // [32][9*Cin] bf16, K-major, BN folded
  int cout_pad_tc = 0;
  const float* bias = nullptr;
  const void* up = nullptr;                // [N,up_h,up_w,24] fp16: the rung below
  int up_ld = 0, up_h = 0, up_w = 0;
  void* out = nullptr;                     // rung mode: [N,H,W,24] fp16
  int out_ld = 0;
  int final_argmax = 0;
  void* pred = nullptr;                    // final mode: [N,2H,2W]
  int pred_i64 = 0;
  int N = 0, H = 0, W = 0, Cin = 0, K = 0;
};
bool ladder_eligible(const LadderArgs& a);
int launch_ladder(const LadderArgs& a, cudaStream_t st);

// stem conv 0 (3 -> C, 3x3 s2) on the tensor cores with a thread-built im2col tile (stem_tc.cu)
bool stem_tc_eligible(const ConvArgs& a);
int launch_stem_tc(const ConvArgs& a, cudaStream_t st);

// out = [relu](base + bilinear(src -> base HW)), out2 = relu(s2*v + b2) ; NHWC, same dtype.
struct UpAddArgs {
  const void* base = nullptr;   // [N,H,W,C]; may be null (pure upsample)
  const void* src = nullptr;    // [N,h,w,C]
  void* out = nullptr;          // optional
  void* out2 = nullptr;         // optional
  int out_ld = 0, out2_ld = 0;
  const float* o2_scale = nullptr;
  const float* o2_shift = nullptr;
  int dtype = LEDB200_F32;
  int N = 0, H = 0, W = 0, C = 0, h = 0, w = 0;
  int relu = 0;
};
int launch_upsample_add(const UpAddArgs& a, cudaStream_t st);

// AvgPool2d(k,s,p, count_include_pad=True) or global average (k == 0), followed by the
// consumer's pre-activation BN+ReLU: out = relu(scale*avg + shift).  (ppm.py:68-90)
struct PoolArgs {
  const void* in = nullptr;
  void* out = nullptr;
  const float* scale = nullptr;
  const float* shift = nullptr;
  int dtype = LEDB200_F32;
  int N = 0, H = 0, W = 0, C = 0, Ho = 0, Wo = 0, k = 0, s = 1, p = 0;
};
int launch_avgpool_bnrelu(const PoolArgs& a, cudaStream_t st);

// The whole DAPPM (ppm.py:57-130) as two launches (dappm.cu): pooled branches, then one clustered tcgen05 kernel for the
// 1x1 / 3x3 chain, the concat-free compression and the shortcut.  All tensors NHWC bf16, dense; BN as y = relu(a x + b).
struct DappmArgs {
  const void* x = nullptr;                         // [N,H,W,C] raw context features
  int N = 0, H = 0, W = 0, C = 0, P = 0, Cout = 0; // P = ppm channels (128), Cout = 4 * channels (128)
  // pooled branches i = 1..4: window / stride / pad (k == 0: global), pooled size, BN, 1x1 conv [P][C], output [N,sh,sw,P]
  int pool_k[4] = {0, 0, 0, 0}, pool_s[4] = {1, 1, 1, 1}, pool_p[4] = {0, 0, 0, 0}, sh[4] = {0, 0, 0, 0}, sw[4] = {0, 0, 0, 0};
  const float* a_scale[4] = {nullptr, nullptr, nullptr, nullptr};
  const float* b_scale[4] = {nullptr, nullptr, nullptr, nullptr};
  const __nv_bfloat16* w_scale[4] = {nullptr, nullptr, nullptr, nullptr};
  const float* bias_scale[4] = {nullptr, nullptr, nullptr, nullptr};
  void* s[4] = {nullptr, nullptr, nullptr, nullptr};
  // scales[0] and shortcut (1x1, [P][C] / [Cout][C]), processes[0..3] (3x3, [P][9*P]), compression (1x1, [Cout][5*P])
  const float *a_s0 = nullptr, *b_s0 = nullptr, *a_sc = nullptr, *b_sc = nullptr, *a_comp = nullptr, *b_comp = nullptr;
  const float* a_proc[4] = {nullptr, nullptr, nullptr, nullptr};
  const float* b_proc[4] = {nullptr, nullptr, nullptr, nullptr};
  const __nv_bfloat16 *w_s0 = nullptr, *w_sc = nullptr, *w_comp = nullptr;
  const __nv_bfloat16* w_proc[4] = {nullptr, nullptr, nullptr, nullptr};
  const float *bias_s0 = nullptr, *bias_sc = nullptr, *bias_comp = nullptr;
  const float* bias_proc[4] = {nullptr, nullptr, nullptr, nullptr};
  void *t0 = nullptr, *t1 = nullptr;               // ping-pong scratch [N,H,W,P]
  void* out = nullptr; int out_ld = 0;             // [N,H,W,Cout]
};
bool dappm_eligible(const DappmArgs& a);
int launch_dappm(const DappmArgs& a, cudaStream_t st);

// out = relu(scale*x + shift) per channel; up to two outputs from one read.
struct AffineArgs {
  const void* in = nullptr;
  void* out_a = nullptr;
  void* out_b = nullptr;
  const float *sa = nullptr, *ba = nullptr, *sb = nullptr, *bb = nullptr;
  int dtype = LEDB200_F32;
  int64_t npix = 0;
  int C = 0;
};
int launch_affine_relu(const AffineArgs& a, cudaStream_t st);

// layout conversion helpers (engine boundary): NCHW fp32 <-> NHWC T
int launch_nchw_to_nhwc(const float* in, void* out, int out_dtype, int N, int C, int H, int W, cudaStream_t st);
int launch_nhwc_to_nchw(const void* in, int in_dtype, float* out, int N, int C, int H, int W, int in_ld, cudaStream_t st);

// fused head tail: 3-level bilinear ladder + argmax (tail.cu)
struct TailArgs {
  const void* xc = nullptr;   // [N,hc,wc,K]
  const void* hx2 = nullptr;  // [N,h4,w4,K]
  const void* hx1 = nullptr;  // [N,h2,w2,K]
  int xc_ld = 0, hx2_ld = 0, hx1_ld = 0;   // pixel strides (elements)
  int dtype = LEDB200_F32;
  int N = 0, K = 0, hc = 0, wc = 0, h4 = 0, w4 = 0, h2 = 0, w2 = 0;
  void* pred = nullptr;       // [N,2*h2,2*w2]
  int pred_dtype = LEDB200_U8;
  float* logits = nullptr;    // optional fp32 NCHW
};
int launch_tail(const TailArgs& a, cudaStream_t st);

// last ladder stage only: r1 [N,h2,w2,ld] fp16 (the top rung written by ladder_kernel)
// -> logits and argmax of its exact x2 upsample (tail.cu, tail2_kernel)
struct Tail2Args {
  const __half* r1 = nullptr;
  int ld = 0;
  int N = 0, K = 0, h2 = 0, w2 = 0;
  void* pred = nullptr;       // [N,2*h2,2*w2]
  int pred_dtype = LEDB200_U8;
  float* logits = nullptr;    // fp32 NCHW, required
};
int launch_tail2(const Tail2Args& a, cudaStream_t st);

int launch_confusion(const void* pred, const void* gt, int pred_dtype, int gt_dtype, int64_t n, int K,
                     int ignore_index, int64_t* cm, cudaStream_t st);

int64_t ohem_workspace_bytes(int64_t npix);
int launch_ohem(const float* logits, const int64_t* target, int N, int K, int H, int W, int ignore_label,
                float thres, int64_t min_kept, float loss_weight, const float* class_weight, float* out3,
                float* dlogits, void* workspace, cudaStream_t st);

// fused ladder top + OHEM CE: the loss (and its gradient) of the bilinear upsample of the NHWC rung r1 [N,h,w,K] to [N,H,W]
// without the full-resolution logits (ohem.cu); same workspace as launch_ohem
int launch_ohem_up(const float* r1, const int64_t* target, int N, int K, int h, int w, int H, int W, int ignore_label,
                   float thres, int64_t min_kept, float loss_weight, const float* class_weight, float* out3,
                   void* workspace, cudaStream_t st);
int launch_ohem_up_bwd(const float* r1, const int64_t* target, int N, int K, int h, int w, int H, int W, int ignore_label,
                       float loss_weight, const float* class_weight, const float* gscale, const void* workspace, float* dr1,
                       cudaStream_t st);

}  // namespace ledb
