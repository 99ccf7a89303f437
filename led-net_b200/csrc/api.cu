// Stand-alone C-ABI operators (no handle): the fused head tail, the confusion matrix, OHEM CE and a
// single convolution through the same launchers the engine uses.  See include/ledb200.h.
#include "kernels.h"

using namespace ledb;

extern "C" {

int ledb200_head_fuse_argmax(const void* xc, const void* hx2, const void* hx1, int32_t dtype, int32_t N, int32_t K,
                             int32_t hc, int32_t wc, int32_t h4, int32_t w4, int32_t h2, int32_t w2, void* pred,
                             int32_t pred_dtype, float* logits_opt, void* stream) {
  if (!xc || !hx2 || !hx1 || !pred) return fail(LEDB200_EINVAL, "head_fuse_argmax: null buffer");
  TailArgs a;
  a.xc = xc; a.hx2 = hx2; a.hx1 = hx1; a.xc_ld = a.hx2_ld = a.hx1_ld = K; a.dtype = dtype;
  a.N = N; a.K = K; a.hc = hc; a.wc = wc; a.h4 = h4; a.w4 = w4; a.h2 = h2; a.w2 = w2;
  a.pred = pred; a.pred_dtype = pred_dtype; a.logits = logits_opt;
  return launch_tail(a, (cudaStream_t)stream);
}

int ledb200_confusion_accumulate(const void* pred, const void* gt, int32_t pred_dtype, int32_t gt_dtype, int64_t n,
                                 int32_t K, int32_t ignore_index, int64_t* cm_inout, void* stream) {
  if ((!pred || !gt) && n > 0) return fail(LEDB200_EINVAL, "confusion: null buffer");
  if (!cm_inout) return fail(LEDB200_EINVAL, "confusion: null matrix");
  return launch_confusion(pred, gt, pred_dtype, gt_dtype, n, K, ignore_index, cm_inout, (cudaStream_t)stream);
}

int64_t ledb200_ohem_workspace_bytes(int64_t npix) { return ohem_workspace_bytes(npix); }

int ledb200_ohem_up_fwd(const float* r1_nhwc, const int64_t* target, int32_t N, int32_t K, int32_t h, int32_t w, int32_t H,
                        int32_t W, int32_t ignore_label, float thres, int64_t min_kept, float loss_weight,
                        const float* class_weight_opt, float* out3, void* workspace, void* stream) {
  if (!out3) return fail(LEDB200_EINVAL, "ohem_up: null output");
  if ((!r1_nhwc || !target) && (int64_t)N * H * W > 0) return fail(LEDB200_EINVAL, "ohem_up: null input");
  return launch_ohem_up(r1_nhwc, target, N, K, h, w, H, W, ignore_label, thres, min_kept, loss_weight, class_weight_opt, out3,
                        workspace, (cudaStream_t)stream);
}

int ledb200_ohem_up_bwd(const float* r1_nhwc, const int64_t* target, int32_t N, int32_t K, int32_t h, int32_t w, int32_t H,
                        int32_t W, int32_t ignore_label, float loss_weight, const float* class_weight_opt,
                        const float* grad_scale_opt, const void* workspace, float* d_r1, void* stream) {
  if (!r1_nhwc || !target) return fail(LEDB200_EINVAL, "ohem_up_bwd: null input");
  return launch_ohem_up_bwd(r1_nhwc, target, N, K, h, w, H, W, ignore_label, loss_weight, class_weight_opt, grad_scale_opt,
                            workspace, d_r1, (cudaStream_t)stream);
}

int ledb200_ohem_ce(const float* logits, const int64_t* target, int32_t N, int32_t K, int32_t H, int32_t W,
                    int32_t ignore_label, float thres, int64_t min_kept, float loss_weight,
                    const float* class_weight_opt, float* out3, float* dlogits_opt, void* workspace, void* stream) {
  if (!out3) return fail(LEDB200_EINVAL, "ohem: null output");
  if ((!logits || !target) && (int64_t)N * H * W > 0) return fail(LEDB200_EINVAL, "ohem: null input");
  return launch_ohem(logits, target, N, K, H, W, ignore_label, thres, min_kept, loss_weight, class_weight_opt, out3,
                     dlogits_opt, workspace, (cudaStream_t)stream);
}

int ledb200_conv2d(const void* in, void* out, const void* residual, int32_t dtype, int32_t N, int32_t H, int32_t W,
                   int32_t Cin, int32_t Cout, int32_t ksize, int32_t stride, int32_t relu, const float* weight_oihw,
                   const float* bias, const float* pre_scale, const float* pre_shift, int32_t backend, int32_t in_ld,
                   int32_t out_ld, int32_t res_ld, void* stream) {
  if (!in || !out || !weight_oihw) return fail(LEDB200_EINVAL, "conv2d: null buffer");
  if (ksize != 1 && ksize != 3) return fail(LEDB200_EINVAL, "conv2d: ksize must be 1 or 3");
  if (stride != 1 && stride != 2) return fail(LEDB200_EINVAL, "conv2d: stride must be 1 or 2");
  if (dtype != LEDB200_F32 && dtype != LEDB200_BF16) return fail(LEDB200_EINVAL, "conv2d: dtype must be F32 or BF16");
  if (in_ld == 0) in_ld = Cin;
  if (out_ld == 0) out_ld = Cout;
  if (res_ld == 0) res_ld = Cout;
  if (in_ld < Cin || out_ld < Cout || res_ld < Cout) return fail(LEDB200_EINVAL, "conv2d: pixel stride smaller than the channel count");
  cudaStream_t st = (cudaStream_t)stream;
  PackedConv c;
  c.cin = Cin; c.cout = Cout; c.k = ksize; c.stride = stride;
  int rc = pack_conv(weight_oihw, bias, nullptr, nullptr, c);
  if (!rc && pre_scale) rc = upload(pre_scale, Cin * 4, (void**)&c.pre_scale);
  if (!rc && pre_shift) rc = upload(pre_shift, Cin * 4, (void**)&c.pre_shift);
  if (!rc) {
    ConvArgs a = conv_args(c, N, H, W);
    a.in = in; a.in_dtype = dtype; a.in_sc = 1; a.in_sw = in_ld; a.in_sh = (int64_t)W * in_ld; a.in_sn = (int64_t)H * W * in_ld;
    a.out = out; a.out_dtype = dtype; a.out_ld = out_ld; a.res = residual; a.res_ld = res_ld; a.relu = relu;
    rc = launch_conv(a, backend, "conv2d", st);
  }
  cudaError_t ce = cudaStreamSynchronize(st);
  if (!rc && ce != cudaSuccess) rc = fail(LEDB200_ECUDA, std::string("conv2d: ") + cudaGetErrorString(ce));
  free_conv(c);
  return rc;
}

}  // extern "C"
