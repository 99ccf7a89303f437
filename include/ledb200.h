/*
 * ledb200.h - C ABI of libledb200.so: hand-written sm_100a CUDA kernels for the
 * LED-Net data-parallel hot path (backbone forward -> bilateral fusion -> seg head
 * -> 3-level logit fusion -> argmax -> IoU confusion matrix; OHEM cross-entropy).
 *
 * The reference (ly27253/LED-Net, an mmsegmentation-1.2.2 fork) is pure Python on
 * stock PyTorch; it has no FFI of its own.  The boundary the reference exposes for
 * this path is the mmseg registry (mmseg/registry/registry.py:56 MODELS, :90 METRICS)
 * and the module methods built from it.  Each entry point below names the reference
 * method(s) whose device work it replaces; the Python modules registered under the
 * reference names (led-net_b200/{backbone,head,losses,metrics,segmentor}.py) bind
 * these through ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - return 0 on success, a negative LEDB200_E* code otherwise; nothing throws or
 *     aborts across the ABI; ledb200_last_error() returns a thread-local message.
 *   - the caller owns every input/output buffer (device pointers unless the name
 *     says host); the library owns only a handle's folded weights and its
 *     activation workspace (allocated at first use of a shape, grown on demand -
 *     no cudaMalloc in steady state).
 *   - all work is enqueued on the cudaStream_t passed in (as void*); no implicit
 *     synchronisation.  One handle per (process, GPU); a handle is not re-entrant.
 *   - activations inside the library are NHWC; dtype mode 0 = fp32 storage with
 *     fp32 CUDA-core math (parity mode, 1e-4), 1 = bf16 storage, fp32 accumulate,
 *     tcgen05/TMEM implicit-GEMM convolutions.
 */
#ifndef LEDB200_H_
#define LEDB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LEDB200_VERSION 100 /* 0.1.0 */

enum {
  LEDB200_OK = 0,
  LEDB200_EINVAL = -1,   /* bad argument / unsupported shape            */
  LEDB200_ECUDA = -2,    /* CUDA runtime / driver error                 */
  LEDB200_ESTATE = -3,   /* call order (e.g. forward before finalize)   */
  LEDB200_ENOMEM = -4,
  LEDB200_ENOTFOUND = -5 /* unknown parameter / buffer name             */
};

enum { LEDB200_F32 = 0, LEDB200_BF16 = 1, LEDB200_U8 = 2, LEDB200_I64 = 3, LEDB200_I32 = 4 };

/* image layouts accepted by the forward entry points */
enum {
  LEDB200_IMG_NCHW_F32 = 0, /* normalised float, what LEDNet.forward(x) receives        */
  LEDB200_IMG_NCHW_U8 = 1,  /* raw BGR uint8 CHW: SegDataPreProcessor fused into stem   */
  LEDB200_IMG_NHWC_U8 = 2   /* raw BGR uint8 HWC (decoder output order)                 */
};

typedef struct ledb200_handle ledb200_handle;

/* Constructor arguments of the two registered modules
 * (configs/LED_Net/LEDNet_80k_cityscapes-1024x1024.py:24-52). */
typedef struct ledb200_cfg {
  int32_t in_channels;   /* LEDNet(in_channels=3)                         */
  int32_t channels;      /* LEDNet(channels=32)                           */
  int32_t ppm_channels;  /* LEDNet(ppm_channels=128)                      */
  int32_t head_channels; /* LEDHead(channels=64)                          */
  int32_t num_classes;   /* LEDHead(num_classes=K)                        */
  int32_t align_corners; /* must be 0 (config); 1 is rejected             */
  int32_t dtype;         /* LEDB200_F32 or LEDB200_BF16 (activation mode) */
  int32_t device;        /* CUDA device ordinal                           */
  int32_t variant;       /* 0 = R0 trunk (DDRNet-23-slim body + stem taps) */
  int32_t conv_backend;  /* 0 = auto (tcgen05 where eligible in bf16 mode), 1 = force CUDA-core */
  float mean[3];         /* SegDataPreProcessor mean (RGB order)          */
  float std[3];          /* SegDataPreProcessor std                       */
  int32_t bgr_to_rgb;    /* SegDataPreProcessor bgr_to_rgb                */
  int32_t reserved[7];
} ledb200_cfg;

int ledb200_version(void);
const char* ledb200_last_error(void);

/* ---- handle life cycle --------------------------------------------------------------
 * Replaces MODELS.build(dict(type='LEDNet', ...)) / MODELS.build(dict(type='LEDHead', ...))
 * (mmseg/models/segmentors/encoder_decoder.py:89,102) for the device side. */
int ledb200_create(const ledb200_cfg* cfg, ledb200_handle** out);
int ledb200_destroy(ledb200_handle* h);

/* Feed one state-dict entry under its reference name, e.g.
 * "backbone.stem.0.conv.weight", "decode_head.head.0.bn.running_var",
 * "decode_head.conv_seg.bias" (module paths of ddrnet.py / led_head.py / decode_head.py:158).
 * `data` is HOST memory, fp32 (dtype LEDB200_F32) or int64 (ignored: num_batches_tracked).
 * Replaces load_state_dict / load_checkpoint (mmseg/apis/inference.py:60). */
int ledb200_set_param(ledb200_handle* h, const char* name, const void* data,
                      const int64_t* shape, int32_t ndim, int32_t dtype);
/* Number of parameters the engine expects, and the i-th expected name (for diagnostics). */
int ledb200_num_params(ledb200_handle* h);
const char* ledb200_param_name(ledb200_handle* h, int32_t i);

/* Fold eval-mode BatchNorm into the convolutions (W*g/sqrt(v+eps), b-m*g/sqrt(v+eps)),
 * repack OIHW fp32 -> [Cout][kh][kw][Cin] bf16 (tensor-core path) and
 * [kh][kw][Cin][Cout] fp32 (CUDA-core path), upload.  Fails with LEDB200_ESTATE and a
 * message listing what is missing if any expected parameter was not set. */
int ledb200_finalize(ledb200_handle* h);

/* ---- inference ----------------------------------------------------------------------
 * Whole path in one call: EncoderDecoder.predict (encoder_decoder.py:187-222) =
 * extract_feat (:117-122) -> LEDHead.forward eval (led_head.py:76-81) ->
 * predict_by_feat fusion (decode_head.py:362-379) -> postprocess_result argmax
 * (segmentors/base.py:187-188).
 *   img        device, layout per img_layout, N x 3 x H x W
 *   pred       device, [N, Ho, Wo] with Ho = 2*ceil(H/2), Wo = 2*ceil(W/2)
 *              (the reference's output size is 2*head_x1.shape, decode_head.py:363);
 *              pred_dtype LEDB200_U8 or LEDB200_I64 (argmax(dim=0) returns int64)
 *   logits_opt device or NULL: full-resolution fused logits [N, K, Ho, Wo] fp32 NCHW
 *              (what predict_by_feat returns); NULL keeps them out of HBM entirely. */
int ledb200_forward_infer(ledb200_handle* h, const void* img, int32_t img_layout, int32_t N,
                          int32_t H, int32_t W, void* pred, int32_t pred_dtype,
                          float* logits_opt, void* stream);

/* LEDNet.forward in eval mode (contract: led_head.py:76-81 consumes (c5, x1, x2)).
 * Outputs are fp32 NCHW device tensors owned by the caller:
 *   c5 [N,4C,ceil(H/8),ceil(W/8)], x1 [N,C,H/2,W/2], x2 [N,C,H/4,W/4]. */
int ledb200_backbone_forward(ledb200_handle* h, const void* img, int32_t img_layout, int32_t N,
                             int32_t H, int32_t W, float* c5, float* x1, float* x2, void* stream);

/* LEDHead.forward in eval mode (led_head.py:76-81) on caller-supplied fp32 NCHW features:
 * returns x_c [N,K,h8,w8], head_x1 [N,K,h2,w2], head_x2 [N,K,h4,w4] (fp32 NCHW). */
int ledb200_head_forward(ledb200_handle* h, const float* c5, const float* x1, const float* x2,
                         int32_t N, int32_t h8, int32_t w8, int32_t h2, int32_t w2, int32_t h4,
                         int32_t w4, float* xc, float* hx1, float* hx2, void* stream);
/* Head + fused tail on caller-owned features: c5 [N,h8,w8,4*channels], x1 [N,h2,w2,channels], x2 [N,h4,w4,channels], NHWC,
 * dense, in the handle's dtype (F32 or BF16) - for a trunk that is not the R0 plan (LEDNet(variant='led')).  The
 * pre-activation BN + ReLU of the three base heads (led_head.py:84-99), the head convs, predict_by_feat's ladder
 * (decode_head.py:362-379) and the argmax (base.py:187-188) run as in ledb200_forward_infer: pred [N,2*h2,2*w2] (U8 or
 * I64); logits_opt (nullable) fp32 [N,K,2*h2,2*w2]. */
int ledb200_head_infer(ledb200_handle* h, const void* c5, const void* x1, const void* x2, int32_t N, int32_t h8, int32_t w8,
                       int32_t h2, int32_t w2, int32_t h4, int32_t w4, void* pred, int32_t pred_dtype, float* logits_opt,
                       void* stream);

/* Copy a named internal activation of the last forward to HOST as fp32 NCHW (tests /
 * layer-wise parity).  `capacity` in floats; writes the shape to shape4 = {N,C,H,W}.
 * Synchronises the stream. */
int ledb200_debug_fetch(ledb200_handle* h, const char* buffer_name, float* host_out,
                        int64_t capacity, int32_t* shape4, void* stream);
/* Per-op timing of the last plan (runs each op `iters` times between CUDA events);
 * writes up to `cap` entries; names via ledb200_op_name.  Returns the op count. */
int ledb200_profile_ops(ledb200_handle* h, int32_t iters, float* ms_out, int32_t cap, void* stream);
const char* ledb200_op_name(ledb200_handle* h, int32_t i);
/* Algorithmic work of op i of the last plan: out3 = {FLOPs, bytes, kind} with kind
 * 0 conv (CUDA cores), 1 conv (tcgen05), 2 upsample+add, 3 avg-pool, 4 affine+ReLU, 5 fused tail,
 * 6 layout conversion.  bench.py builds the per-layer roofline from these (DESIGN.md section 4). */
int ledb200_op_info(ledb200_handle* h, int32_t i, double* out3);
/* Number of kernel launches one forward of the current plan issues. */
int ledb200_plan_launches(ledb200_handle* h);

/* ---- stand-alone fused kernels --------------------------------------------------------
 * BaseDecodeHead.predict_by_feat (decode_head.py:362-379) + postprocess argmax
 * (base.py:187-188) in one kernel: r = hx2 + up(xc); r = hx1 + up(r); out = up(r -> 2*hx1.HW);
 * pred = first-max argmax over K.  Inputs NHWC, dtype F32 or BF16:
 * xc [N,hc,wc,K], hx2 [N,h4,w4,K], hx1 [N,h2,w2,K]; output [N,2*h2,2*w2].
 * logits_opt: optional fp32 NCHW [N,K,2*h2,2*w2]. */
int ledb200_head_fuse_argmax(const void* xc, const void* hx2, const void* hx1, int32_t dtype,
                             int32_t N, int32_t K, int32_t hc, int32_t wc, int32_t h4, int32_t w4,
                             int32_t h2, int32_t w2, void* pred, int32_t pred_dtype,
                             float* logits_opt, void* stream);

/* IoUMetric.intersect_and_union (evaluation/metrics/iou_metric.py:163-200) and
 * calculate_confusion_matrix (tools/analysis_tools/confusion_matrix.py:66-74):
 * cm[(K+1) x K] int64 += bincount(K*gt + pred) over pixels with gt != ignore_index;
 * rows = GT, cols = prediction; row K collects GT values outside [0,K) that are not
 * ignore_index (histc drops those from area_label but keeps them in area_pred_label).
 * pred_dtype / gt_dtype: LEDB200_U8 or LEDB200_I64.  Accumulates (does not zero). */
int ledb200_confusion_accumulate(const void* pred, const void* gt, int32_t pred_dtype,
                                 int32_t gt_dtype, int64_t n, int32_t K, int32_t ignore_index,
                                 int64_t* cm_inout, void* stream);

/* OhemCrossEntropy.forward (+ autograd backward) (losses/ohem_cross_entropy_loss.py:52-90)
 * and accuracy (losses/accuracy.py:41-60) in one pass family:
 *   logits  fp32 NCHW [N,K,H,W]; target int64 [N,H,W]
 *   class_weight_opt device fp32 [K] or NULL
 *   out3    device fp32[3]: {loss (already * loss_weight), kept count, top-1 accuracy in %}
 *   dlogits_opt device fp32 NCHW or NULL: d(loss)/d(logits)
 *   workspace device, >= ledb200_ohem_workspace_bytes(N*H*W) bytes */
int64_t ledb200_ohem_workspace_bytes(int64_t npix);
int ledb200_ohem_ce(const float* logits, const int64_t* target, int32_t N, int32_t K, int32_t H,
                    int32_t W, int32_t ignore_label, float thres, int64_t min_kept,
                    float loss_weight, const float* class_weight_opt, float* out3,
                    float* dlogits_opt, void* workspace, void* stream);

/* The same loss taken over logits = resize(r1, (H, W), mode='bilinear', align_corners=False) WITHOUT materialising them:
 * r1 is the last rung of LEDHead's training ladder (led_head.py:101-146 / decode_head.py:362-379), device fp32 NHWC
 * [N,h,w,K], K <= 32.  Every full-resolution pixel interpolates its K logits in registers (bit-identical to the resize
 * kernel's values); the backward gathers, per r1 pixel, the outputs that read it and re-derives their softmax, in the
 * resize backward's summation order.  fwd fills out3 and leaves the per-pixel probabilities and the selection threshold in
 * `workspace` (>= ledb200_ohem_workspace_bytes(N*H*W)); bwd reads them and writes d(loss)/d(r1) [N,h,w,K], scaled by the
 * device scalar grad_scale_opt (the upstream gradient of the loss; NULL = 1). */
int ledb200_ohem_up_fwd(const float* r1_nhwc, const int64_t* target, int32_t N, int32_t K, int32_t h, int32_t w,
                        int32_t H, int32_t W, int32_t ignore_label, float thres, int64_t min_kept, float loss_weight,
                        const float* class_weight_opt, float* out3, void* workspace, void* stream);
int ledb200_ohem_up_bwd(const float* r1_nhwc, const int64_t* target, int32_t N, int32_t K, int32_t h, int32_t w,
                        int32_t H, int32_t W, int32_t ignore_label, float loss_weight, const float* class_weight_opt,
                        const float* grad_scale_opt, const void* workspace, float* d_r1, void* stream);

/* One convolution through the same launchers the engine uses (unit tests, SESP etc.).
 * NHWC in/out of `dtype`; weight host fp32 OIHW [Cout,Cin,kh,kw] folded by the caller;
 * bias host fp32 [Cout] or NULL; pre_scale/pre_shift host fp32 [Cin] or NULL
 * (pre-activation BN+ReLU applied before zero padding, mmcv ConvModule order
 * ('norm','act','conv'): led_head.py:94, ppm.py:42-43); residual NHWC or NULL.
 * backend 0 auto, 1 CUDA-core, 2 tcgen05 (fails if the shape is not eligible).
 * in_ld / out_ld / res_ld: pixel strides in elements (0 = dense, i.e. Cin / Cout / Cout); the
 * tcgen05 path needs them to be multiples of 8 (16-byte pixels), so a 19-class output is
 * stored with out_ld = 24 exactly as the engine does. */
int ledb200_conv2d(const void* in, void* out, const void* residual, int32_t dtype, int32_t N,
                   int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t ksize, int32_t stride,
                   int32_t relu, const float* weight_oihw, const float* bias,
                   const float* pre_scale, const float* pre_shift, int32_t backend,
                   int32_t in_ld, int32_t out_ld, int32_t res_ld, void* stream);

/* ---- training step (SURVEY section 8a rows T1/T4; north_star kernel 6) -----------------------------
 * The reference trains through autograd over ATen/cuDNN (encoder_decoder.py:161-185 -> led_head.py:101-146,
 * SGD per configs/LED_Net/LEDNet_80k_cityscapes-1024x1024.py:64-65).  These entry points are the forward
 * and backward kernels of every op on that path; led-net_b200/train_ops.py wraps them as
 * torch.autograd.Function so PyTorch supplies only the tape.  All tensors are DEVICE fp32 NHWC, dense. */

/* Weights stay in the reference's OIHW fp32 state-dict layout; each step repacks them on the device.
 * mode 0 -> forward layout [tap][Cin][Cout16]; mode 1 -> data-gradient layout [tap flipped][Cout][Cin16]. */
int64_t ledb200_train_packed_weight_floats(int32_t Cout, int32_t Cin, int32_t k, int32_t mode);
int ledb200_train_pack_weight(const float* w_oihw, float* out, int32_t Cout, int32_t Cin, int32_t k,
                              int32_t mode, void* stream);
/* nn.Conv2d(k in {1,3}, padding k/2, stride in {1,2}) forward: y[N,Ho,Wo,Cout] (bias_opt [Cout] or NULL). */
int ledb200_train_conv_fwd(const float* x, const float* w_packed, const float* bias_opt, float* y,
                           int32_t N, int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t k,
                           int32_t stride, void* stream);
/* d(loss)/dx [N,H,W,Cin] from dy [N,Ho,Wo,Cout] (H, W are the conv INPUT extents). */
int ledb200_train_conv_dgrad(const float* dy, const float* w_packed_dgrad, float* dx, int32_t N,
                             int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t k, int32_t stride,
                             void* stream);
/* Tensor-core forms of the forward / data-gradient convolution (north_star kernel 6: dgrad / wgrad implicit GEMM; the
 * reference gets cuDNN's through encoder_decoder.py:161-185 -> led_head.py:101-146): conv_tc.cu's tcgen05 implicit GEMM with
 * kind::tf32 operands read straight from the fp32 NHWC tensors (TMA halo slabs), fp32 accumulation in TMEM, raw fp32 output.
 * ledb200_train_conv_tc_ok(op, ...) says whether they take a shape (op 0 forward, 1 data gradient, 2 weight gradient;
 * H, W = conv INPUT extents): Cin % 32 == 0 (of the GEMM's reduction side), output extents multiples of the 16 x 8 tile.
 * The data gradient of a stride-2 convolution runs as its four parity classes (3x3; weights from pack mode 2) or as the
 * even-even class over a zeroed gradient (1x1; pack mode 1).  Everything else stays on the CUDA-core entry points above.  Weights: K-major fp32
 * [pad(Cout)][k*k*Cin] (mode 0) / [pad(Cin)][k*k*Cout] rotated (mode 1) rounded to tf32 on the device, followed by a second
 * matrix of the same shape holding the remainders w - tf32(w) (the three-pass mode's w_lo). */
/* tf32 storage mode of the training element-wise kernels (BatchNorm apply / backward, resize, add, pool, concat): on = every
 * tensor they write is rounded to tf32 (nearest), because the tensor core truncates raw fp32 operands.  Process-wide;
 * returns the previous setting.  train_ops.set_tensor_cores() keeps it in step with the convolution path. */
int ledb200_train_set_tf32_rounding(int32_t on);
/* Tensor-core passes per product of the *_tc entry points below.  3 (default): error-compensated "3 x TF32" -
 * x = x_hi + x_lo, w = w_hi + w_lo, x*w ~= x_hi*w_hi + x_hi*w_lo + x_lo*w_hi with exact products and fp32 accumulation:
 * fp32-grade results from the tensor pipe (the low parts are formed in shared memory next to every TMA-staged slab).
 * 1: a single tf32 pass (10-bit mantissa operands, cuDNN's allow_tf32 numerics).  Process-wide; returns the previous value. */
int ledb200_train_set_tf32_passes(int32_t passes);
/* Passes of ledb200_train_conv_wgrad_tc alone (default 1).  The weight gradient is a leaf of the backward pass - its rounding
 * is not fed back into the chain - and a sum over 1e5..1e6 pixels: one tf32 pass leaves a uniform ~7e-4 shrink (the tensor
 * core truncates raw fp32 operands) against the 1e-2 gate; 3 = fp32-grade like the forward / data-gradient kernels. */
int ledb200_train_set_wgrad_passes(int32_t passes);
int32_t ledb200_train_conv_tc_ok(int32_t op, int32_t N, int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t k,
                                 int32_t stride);
int64_t ledb200_train_packed_weight_tc_floats(int32_t Cout, int32_t Cin, int32_t k, int32_t mode);
int ledb200_train_pack_weight_tc(const float* w_oihw, float* out, int32_t Cout, int32_t Cin, int32_t k,
                                 int32_t mode, void* stream);
int ledb200_train_conv_fwd_tc(const float* x, const float* w_tc, const float* bias_opt, float* y, int32_t N,
                              int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t k, int32_t stride,
                              void* stream);
int ledb200_train_conv_dgrad_tc(const float* dy, const float* w_tc_dgrad, float* dx, int32_t N, int32_t H,
                                int32_t W, int32_t Cin, int32_t Cout, int32_t k, int32_t stride, void* stream);
/* Weight gradient on the tensor cores (wgrad_tc.cu): 3x3, stride 1 or 2, Cin and Cout multiples of 32, no bias gradient.
 * The pixel is the GEMM's reduction dimension: both operands are read MN-major straight from the TMA-staged NHWC slabs, the
 * accumulators stay in TMEM for the CTA's whole life, per-CTA partials are added in a fixed order (bit-reproducible).
 * workspace: device, >= ledb200_train_wgrad_tc_workspace_bytes(...) bytes. */
int64_t ledb200_train_wgrad_tc_workspace_bytes(int32_t N, int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t k,
                                               int32_t stride);
int ledb200_train_conv_wgrad_tc(const float* x, const float* dy, float* dw_oihw, int32_t N, int32_t H, int32_t W,
                                int32_t Cin, int32_t Cout, int32_t k, int32_t stride, void* workspace, void* stream);
/* The stem's first layer (mmcv ConvModule 3 -> C, 3x3, stride 2; ddrnet.py:121-139) on the NCHW image as the caller holds
 * it: forward into an NHWC tensor and the weight gradient, without the NHWC copy of the image the generic entry points need.
 * Cin <= 4; forward: Cout a multiple of 16, <= 128.  workspace: ledb200_train_wgrad_workspace_bytes(Cin, Cout, 3). */
int ledb200_train_stem_fwd(const float* x_nchw, const float* w_oihw, const float* bias_opt, float* y, int32_t N,
                           int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t stride, void* stream);
int ledb200_train_stem_wgrad(const float* x_nchw, const float* dy, float* dw_oihw, int32_t N, int32_t H, int32_t W,
                             int32_t Cin, int32_t Cout, int32_t stride, void* workspace, void* stream);
/* d(loss)/dW in OIHW (overwritten) and optionally d(loss)/dbias.  Every reduction of the training kernels is order-fixed
 * (per-CTA / per-block partial sums in `workspace`, added in index order: no floating-point atomics), so a training step
 * is bit-reproducible run to run.  workspace: device, >= ledb200_train_wgrad_workspace_bytes(Cin, Cout, k) bytes. */
int64_t ledb200_train_wgrad_workspace_bytes(int32_t Cin, int32_t Cout, int32_t k);
int64_t ledb200_train_bn_workspace_bytes(int32_t C);
int ledb200_train_conv_wgrad(const float* x, const float* dy, float* dw_oihw, float* dbias_opt, int32_t N,
                             int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t k, int32_t stride,
                             void* workspace, void* stream);
/* nn.BatchNorm2d in training mode fused with the block's residual add and ReLU
 * (basic_block.py:62-75): out = [relu](bn(y) [+ res]); saves batch mean / inverse std for backward and
 * updates the running statistics (momentum, unbiased variance) in place.  workspace: device, >= ledb200_train_bn_workspace_bytes(C) bytes
 * (doubles [0,2C) hold the statistics after a reduce step, [2C,4C+8) are free for the caller - SyncBN keeps the all-reduced copy
 * and the sample count there -, the rest are block partials). */
int ledb200_train_bn_fwd(const float* y, const float* gamma, const float* beta, const float* res_opt,
                         float* out, float* save_mean, float* save_invstd, float* running_mean_opt,
                         float* running_var_opt, float momentum, float eps, int32_t relu, int64_t npix,
                         int32_t C, void* workspace, void* stream);
/* All-reduce (sum) of n <= nmax doubles over the `world` GPUs of one NVSwitch box through peer memory, for the SyncBN
 * statistics (2C + 1 doubles per layer and direction; NCCL's small-message latency was 6.7 ms of a 41 ms step at N = 8).
 * peer_buffers[r] = rank r's symmetric buffer as mapped into THIS process (>= ledb200_peer_allreduce_buffer_bytes(nmax)
 * bytes, zeroed before the first call, e.g. torch.distributed._symmetric_memory); seq = 1, 2, 3, ... advanced identically on
 * every rank.  One launch: P2P stores of the local vector into every peer's slot, release / acquire flags, slots added in
 * rank order (identical bits on all ranks).  local may alias out. */
int64_t ledb200_peer_allreduce_buffer_bytes(int32_t nmax);
int ledb200_peer_allreduce_f64(const double* local, int32_t n, int32_t rank, int32_t world, const uint64_t* peer_buffers,
                               uint32_t seq, int32_t nmax, double* out, void* stream);
/* backward of the above: dy, dres_opt (= masked dout), dgamma, dbeta. */
int ledb200_train_bn_bwd(const float* dout, const float* y, const float* out, const float* gamma,
                         const float* save_mean, const float* save_invstd, float* dy, float* dres_opt,
                         float* dgamma, float* dbeta, int32_t relu, int64_t npix, int32_t C, void* workspace,
                         void* stream);
/* The same in separate steps, so that the per-channel statistics can be all-reduced between ranks - SyncBN
 * (configs/LED_Net/LEDNet_80k_cityscapes-1024x1024.py:20; torch.nn.SyncBatchNorm semantics):
 *   reduce(mode 0): workspace[0:2C] (double) = (sum y, sum y^2)
 *   reduce(mode 1): workspace[0:2C]          = (sum dz, sum dz * xhat), dz = dout masked by the ReLU
 *   reduce(mode 0) also leaves this rank's sample count at workspace[2C]; reduce(mode 3) = mode 1 on the FORWARD pass's
 *                   workspace: the global count it still holds at [2C] moves to [4C], the sums land at [0:2C] and [2C:4C]
 *                   (mode 4: the same without the move, for a repeated backward pass)
 *   fwd_apply     : mean / invstd / running stats from workspace[0:2C] over `total_count` samples, then apply
 *                   (total_count < 0: the count is read on the device, from workspace[2C] here and workspace[4C] in bwd_apply -
 *                   the all-reduced count of a SyncBN layer never visits the host)
 *   bwd_apply     : dgamma / dbeta from workspace[0:2C] (this rank), dy from workspace[2C:4C] (all ranks). */
int ledb200_train_bn_reduce(const float* a, const float* y_opt, const float* out_opt, const float* mean_opt,
                            const float* invstd_opt, int32_t mode, int32_t relu, int64_t npix, int32_t C,
                            void* workspace, void* stream);
int ledb200_train_bn_fwd_apply(const float* y, const float* gamma, const float* beta, const float* res_opt,
                               float* out, float* save_mean, float* save_invstd, float* running_mean_opt,
                               float* running_var_opt, float momentum, float eps, int32_t relu, int64_t npix,
                               double total_count, int32_t C, const void* workspace, void* stream);
int ledb200_train_bn_bwd_apply(const float* dout, const float* y, const float* out, const float* gamma,
                               const float* save_mean, const float* save_invstd, float* dy, float* dres_opt,
                               float* dgamma, float* dbeta, int32_t relu, int64_t npix, double total_count,
                               int32_t C, const void* workspace, void* stream);
/* resize(mode='bilinear', align_corners=False) (utils/wrappers.py:8-27) and its backward (dsrc overwritten). */
int ledb200_train_resize_fwd(const float* src, float* out, int32_t N, int32_t h, int32_t w, int32_t H,
                             int32_t W, int32_t C, void* stream);
int ledb200_train_resize_bwd(const float* dout, float* dsrc, int32_t N, int32_t h, int32_t w, int32_t H,
                             int32_t W, int32_t C, void* stream);
/* out = [relu](a [+ b_opt]); relu backward dx = dout * (out > 0). */
int ledb200_train_add_relu(const float* a, const float* b_opt, float* out, int32_t relu, int64_t n,
                           void* stream);
int ledb200_train_relu_bwd(const float* dout, const float* out, float* dx, int64_t n, void* stream);
/* nn.AvgPool2d(k,s,p) (count_include_pad=True) or AdaptiveAvgPool2d(1) when k == 0 (ppm.py:66-90). */
int ledb200_train_avgpool_fwd(const float* in, float* out, int32_t N, int32_t H, int32_t W, int32_t C,
                              int32_t Ho, int32_t Wo, int32_t k, int32_t s, int32_t p, void* stream);
int ledb200_train_avgpool_bwd(const float* dout, float* din, int32_t N, int32_t H, int32_t W, int32_t C,
                              int32_t Ho, int32_t Wo, int32_t k, int32_t s, int32_t p, void* stream);
/* channel slice copy (torch.cat(dim=1) of ppm.py:128 and its backward). */
int ledb200_train_copy_channels(const float* src, int32_t src_ld, int32_t src_off, float* dst,
                                int32_t dst_ld, int32_t dst_off, int64_t npix, int32_t C, void* stream);
/* NCHW <-> NHWC fp32 (the boundary to the reference's tensors). */
int ledb200_train_layout(const float* in, float* out, int32_t N, int32_t C, int32_t H, int32_t W,
                         int32_t to_nhwc, void* stream);
/* torch.optim.SGD(momentum, weight_decay) over one flat parameter arena; grad is multiplied by
 * grad_scale first (1/world_size after a sum all-reduce). */
int ledb200_train_sgd_step(float* param, const float* grad, float* momentum_buf, int64_t n, float lr,
                           float momentum, float weight_decay, int32_t first_step, float grad_scale,
                           void* stream);

/* ---- SESP block (SURVEY section 8a row B5; north_star kernel 2) ---------------------------------
 * SESP.forward (mmseg/models/nn_layers/eesp.py:76-118; CBR/BR/CB/CDilated of espnet_utils.py:8-145),
 * eval mode, stride 1, k = 4 branches, as ONE kernel: grouped 1x1 + BN + PReLU -> 4 depthwise dilated
 * 3x3 with hierarchical fusion -> (SESPV2) second depthwise 3x3 with dilation d+1 -> concat, BN + PReLU,
 * grouped 1x1 + BN -> + input (when nIn == nOut) -> PReLU.  NHWC in/out of `dtype` (F32 or BF16).
 * `params`: device fp32 block of ledb200_sesp_param_floats(nIn, nOut) floats, BatchNorm already
 * folded to per-channel scale/shift by the caller, in this order:
 *   w_proj[n][nIn/4], proj_scale[n], proj_shift[n], proj_slope[n], w_dw[4][n][9], w_dw2[4][n][9],
 *   br_scale[nOut], br_shift[nOut], br_slope[nOut], w_exp[nOut][n], exp_scale[nOut], exp_shift[nOut],
 *   act_slope[nOut]            (n = nOut/4).
 * dilations4: host int32[4], the first depthwise dilation of each branch (eesp.py:40-57). */
int64_t ledb200_sesp_param_floats(int32_t nIn, int32_t nOut);
int ledb200_sesp_forward(const void* in, void* out, int32_t dtype, int32_t N, int32_t H, int32_t W,
                         int32_t nIn, int32_t nOut, const int32_t* dilations4, int32_t v2,
                         const float* params, void* stream);

/* ---- MFAF gate (SURVEY section 8a row B7) ---------------------------------------------------------
 * Replaces Muti_AFF.forward (mmseg/models/classification/model_utils.py:410-429), eval mode:
 *   xa = x + residual;  att = local(xa) + global(avgpool(xa)) + sum_{L=4,8,16} nearest_up(ctx_L(adaptive_avgpool_L(xa)));
 *   out = 2 x sigmoid(att) + 2 residual (1 - sigmoid(att)).
 * NHWC x / residual / out of `dtype` (F32 or BF16), C channels (multiple of 8, <= 256), CI = C // r in
 * {8, 16, 32, 64}.  `params`: device fp32 block of ledb200_mfaf_param_floats(C, CI) floats, five paths in the
 * order local_att, context1 (4x4), context2 (8x8), context3 (16x16), global_att, each as
 *   w1[CI][C], a1[CI], b1[CI], w2[C][CI], a2[C], b2[C]
 * with the conv bias and BatchNorm folded by the caller to y = a * (W x) + b.
 * `workspace`: device scratch of ledb200_mfaf_workspace_bytes(N, C) bytes (pooled sums + context table). */
int64_t ledb200_mfaf_param_floats(int32_t C, int32_t CI);
int64_t ledb200_mfaf_workspace_bytes(int32_t N, int32_t C);
int ledb200_mfaf_forward(const void* x, const void* residual, void* out, int32_t dtype, int32_t N, int32_t H,
                         int32_t W, int32_t C, int32_t CI, const float* params, void* workspace, void* stream);

/* ---- GETB block (SURVEY section 8a row B6) ---------------------------------------------------------
 * Replaces GETBBlock.forward (mmseg/models/backbones/UNetFormer_GETB.py:221-226; GlobalLocalAttention :97-206,
 * Mlp :79-94), eval mode, window_size 8: out = y + fc2(ReLU6(fc1(BN2(y)))), y = x + attn(BN1(x)).
 * A handle owns the device copies of the weights (both conv layouts) and a workspace that grows only when a
 * larger shape arrives.  `params`: HOST fp32 block of ledb200_getb_param_floats(dim, heads, hidden) floats:
 *   w_qkv[3C][C] (BN1 folded in), b_qkv[3C], n1_scale[C], n1_shift[C] (BN1 as y = s x + t),
 *   rel_bias[heads][64][64] (relative_position_bias_table gathered by relative_position_index),
 *   w_dw[C][64] (depthwise 8x8), dw_scale[C], dw_shift[C] (proj BN), w_proj[C][C],
 *   w_fc1[hidden][C] (BN2 folded in), b_fc1[hidden], w_fc2[C][hidden], b_fc2[C].
 * x / out: NHWC [N,H,W,dim] of the handle's dtype (F32 or BF16); H, W >= 2 and the reflect padding to a multiple
 * of 8 must be smaller than the input (PyTorch's own F.pad rule). */
typedef struct ledb200_getb ledb200_getb;
int64_t ledb200_getb_param_floats(int32_t dim, int32_t heads, int32_t hidden);
int ledb200_getb_create(int32_t dim, int32_t heads, int32_t hidden, int32_t window, int32_t dtype,
                        const float* params, ledb200_getb** out);
int ledb200_getb_destroy(ledb200_getb* g);
int ledb200_getb_forward(ledb200_getb* g, const void* x, void* out, int32_t N, int32_t H, int32_t W, void* stream);

/* ---- result post-processing (SURVEY section 8a rows H3, E2) -------------------------------------------
 * ledb200_postprocess: BaseSegmentor.postprocess_result (mmseg/models/segmentors/base.py:153-198) for ONE image:
 *   logits fp32 [K,H,W] (NCHW plane layout) -> remove `padding_lrtb` (left, right, top, bottom; NULL = none) -> undo
 *   `flip` (0 none, 1 horizontal, 2 vertical) -> bilinear resize to [out_h, out_w] (align_corners as the head's) ->
 *   pred [out_h,out_w] = argmax over K (first max), or sigmoid(v) > threshold when K == 1 (pred dtype U8, I64 or F32);
 *   `out_logits` (nullable) receives the resized fp32 [K,out_h,out_w] logits (sigmoid applied when K == 1).
 * ledb200_slide_accumulate / ledb200_slide_finalize: EncoderDecoder.slide_inference (encoder_decoder.py:241-292):
 *   preds[:, :, y1:y1+hc, x1:x1+wc] += crop_logits; count[:, 0, same window] += 1; then preds /= count in place and,
 *   when `pred` is given, argmax over K into [N,H,W] (U8 or I64).  preds [N,K,H,W], count [N,1,H,W], fp32. */
int ledb200_postprocess(const float* logits, int32_t K, int32_t H, int32_t W, const int32_t* padding_lrtb,
                        int32_t flip, int32_t out_h, int32_t out_w, int32_t align_corners, float threshold,
                        void* pred, int32_t pred_dtype, float* out_logits, void* stream);
int ledb200_slide_accumulate(float* preds, float* count, const float* crop_logits, int32_t N, int32_t K, int32_t H,
                             int32_t W, int32_t hc, int32_t wc, int32_t y1, int32_t x1, void* stream);
int ledb200_slide_finalize(float* preds, const float* count, int32_t N, int32_t K, int32_t H, int32_t W, void* pred,
                           int32_t pred_dtype, void* stream);

/* ledb200_slide_merge: slide_inference's accumulation for ALL crop windows in one pass (the crops ran as ONE engine batch):
 *   crop_logits fp32 [G*N,K,hc,wc] (window g of image n at index g*N+n), window origins y1[g], x1[g] (HOST arrays, G <= 64, in
 *   the reference's grid order).  Per output pixel the covering windows are summed in that order starting from 0 (bit-identical
 *   to the sequential `preds += F.pad(crop)`, encoder_decoder.py:283-287), divided by their number (:290) and, when `pred` is
 *   given, arg-maxed (U8 or I64).  out_logits (nullable) [N,K,H,W].  Windows that leave a row or a column uncovered are an error
 *   (the reference asserts count_mat != 0, :289).
 * ledb200_stack_pad: SegDataPreProcessor.forward + stack_batch for ONE sample (mmseg/models/data_preprocessor.py:112-149,
 *   mmseg/utils/misc.py:30-128): img [3,h,w] (U8 or F32, CHW) -> out [3,Hp,Wp] fp32: channel c reads input channel 2-c when
 *   swap_rb, (v - mean3[c]) / std3[c] when mean3/std3 (HOST, both or neither) are given, `pad_val` right of / below the image;
 *   label (nullable, [h,w] U8 or I64) -> label_out [Hp,Wp] int64 padded with seg_pad_val. */
int ledb200_slide_merge(const float* crop_logits, int32_t G, const int32_t* y1, const int32_t* x1, int32_t N, int32_t K,
                        int32_t H, int32_t W, int32_t hc, int32_t wc, float* out_logits, void* pred, int32_t pred_dtype,
                        void* stream);
int ledb200_stack_pad(const void* img, int32_t img_dtype, int32_t h, int32_t w, int32_t swap_rb, const float* mean3,
                      const float* std3, float pad_val, float* out, int32_t Hp, int32_t Wp, const void* label,
                      int32_t label_dtype, int64_t* label_out, int32_t seg_pad_val, void* stream);

/* ledb200_tta_merge: SegTTAModel.merge_preds (mmseg/models/segmentors/seg_tta.py) over V views of N images in ONE launch.
 *   views (HOST array, 1 <= V <= 32, in the augmentation list order): image n of view v is the fp32 [K,H,W] plane stack at
 *   logits + n * image_stride (elements); pad_lrtb / flip (0 none, 1 horizontal, 2 vertical) are that view's padding to
 *   remove and flip to undo.  Per output pixel of [oh, ow] and per view, the value of class k is exactly what
 *   ledb200_postprocess writes to out_logits for that view (same source taps and lerp); then mode 0 (out_channels > 1):
 *   softmax over K, mode 1 (out_channels == 1): sigmoid per class, summed over the views in order in fp32 registers
 *   (shared memory for K > 32) and divided by V.  pred: mode 0 argmax over K (first max) [N,oh,ow] U8 or I64; mode 1
 *   (merged > threshold) as F32 [N,K,oh,ow].  probs_opt (nullable): the merged fp32 [N,K,oh,ow].  1 <= K <= 255. */
typedef struct {
  const float* logits;
  int64_t image_stride;
  int32_t H, W;
  int32_t pad_lrtb[4];
  int32_t flip;
} ledb200_tta_view;
int ledb200_tta_merge(const ledb200_tta_view* views, int32_t V, int32_t N, int32_t K, int32_t oh, int32_t ow,
                      int32_t align_corners, int32_t mode, float threshold, void* pred, int32_t pred_dtype,
                      float* probs_opt, void* stream);

/* ---- training augmentation (csrc/augment.cu) ---------------------------------------------------------------------------
 * The config's train_pipeline RandomResize (keep_ratio) -> RandomCrop (cat_max_ratio) -> RandomFlip (horizontal) ->
 * PhotoMetricDistortion, then SegDataPreProcessor's swap / normalisation / padding, for up to 64 samples per call; the
 * random draws are the caller's (one descriptor per sample, HOST array).  img: [3,h,w] uint8 CHW as decoded (BGR);
 * label: [h,w] of `label_dtype` (U8 or I64).  (rh, rw): the RandomResize size of the sample (cv2 INTER_LINEAR for the
 * image, INTER_NEAREST for the label).  offsets[k] = (offset_h, offset_w) of candidate box k in the resized frame, each
 * in [0, max(rh - crop_h, 0)] x [0, max(rw - crop_w, 0)]; the box is clipped to the frame.  flip: 1 mirrors the cropped
 * extent horizontally.  Photometric steps fire when their flag is 1, in the order brightness (+beta), contrast if
 * contrast_mode == 1 (*contrast_alpha), saturation (*saturation_alpha on S of HSV), hue (H + hue_delta mod 180), contrast
 * if contrast_mode == 0, each step in uint8 arithmetic as mmseg's PhotoMetricDistortion computes it. */
typedef struct {
  const uint8_t* img;
  const void* label;
  int32_t h, w;
  int32_t rh, rw;
  int32_t num_candidates;        /* 1 .. 11 */
  int32_t offsets[11][2];
  int32_t flip;
  int32_t contrast_mode;
  int32_t brightness, contrast, saturation, hue;
  float beta, contrast_alpha, saturation_alpha;
  int32_t hue_delta;
} ledb200_aug_sample;
/* ledb200_crop_select: RandomCrop's cat_max_ratio loop for every sample at once.  Candidate k < num_candidates - 1 is
 *   accepted when the nearest-resized label inside its box, ignore_index (in [0, 255]) dropped, holds more than one class
 *   and max(count) / sum(count) < cat_max_ratio (float64); label values outside [0, 255] count as one class.
 *   crop_index [N] int32 (device) receives the first accepted candidate, else num_candidates - 1. */
int ledb200_crop_select(const ledb200_aug_sample* samples, int32_t N, int32_t crop_h, int32_t crop_w, int32_t label_dtype,
                        double cat_max_ratio, int32_t ignore_index, int32_t* crop_index, void* stream);
/* ledb200_train_augment: out [N,3,Hp,Wp] fp32 and label_out [N,Hp,Wp] int64 of the augmented batch, the box of sample n
 *   being candidate crop_index[n] (device; nullable when every sample has one candidate).  Channel c of out reads
 *   augmented channel 2 - c when swap_rb, then (v - mean3[c]) / std3[c] when mean3 / std3 (HOST, both or neither) are
 *   given; pixels right of / below the cropped extent get pad_val and seg_pad_val. */
int ledb200_train_augment(const ledb200_aug_sample* samples, int32_t N, int32_t crop_h, int32_t crop_w,
                          int32_t label_dtype, const int32_t* crop_index, int32_t swap_rb, const float* mean3,
                          const float* std3, float pad_val, float* out, int32_t Hp, int32_t Wp, int64_t* label_out,
                          int32_t seg_pad_val, void* stream);

/* ---- test-time views (csrc/augment.cu) ---------------------------------------------------------------------------------
 * mmcv Resize (keep_ratio; cv2 INTER_LINEAR, the same taps as ledb200_train_augment) of a decoded image, optionally
 * followed by RandomFlip (horizontal), then SegDataPreProcessor's swap / normalisation / padding: the views of
 * TestTimeAug and the test pipeline's own Resize.  One descriptor per (image, resized size), HOST array.
 * src: [3,h,w] uint8 CHW as decoded (BGR).  (rh, rw): the resized size, computed by the caller with mmcv's arithmetic.
 * out / out_flip: [3,Hp,Wp] fp32 of the unflipped / horizontally flipped view, either may be NULL but not both; a flip
 * pair costs one sampling pass. */
typedef struct {
  const uint8_t* src;
  float* out;
  float* out_flip;
  int32_t h, w;
  int32_t rh, rw;
} ledb200_view_desc;
/* ledb200_view_resize: 1 <= n <= 64 views of one padded size Hp x Wp (rh <= Hp, rw <= Wp).  Channel c of an output reads
 *   resized channel 2 - c when swap_rb, then (v - mean3[c]) / std3[c] when mean3 / std3 (HOST, both or neither) are
 *   given; pixels right of / below the resized frame get pad_val. */
int ledb200_view_resize(const ledb200_view_desc* views, int32_t n, int32_t Hp, int32_t Wp, int32_t swap_rb,
                        const float* mean3, const float* std3, float pad_val, void* stream);

/* ---- label maps -> PNG files (csrc/png.cu) ------------------------------------------------------------------------------
 * What IoUMetric(output_dir=...) writes for each prediction (mmseg: Image.fromarray((pred + reduce_zero_label)
 * .astype(np.uint8)).save(path)): an 8-bit grayscale PNG (colour type 0, no interlace) of (label + add) mod 256, one
 * IDAT holding one zlib stream.  Files decode to exactly those pixels; they are not byte-identical to PIL's.
 * ledb200_png_bound: the largest file an H x W map can give (headers plus the whole image in stored blocks), or
 *   LEDB200_EINVAL when H or W < 1 or the map does not fit one IDAT chunk.
 * ledb200_png_workspace_bytes: device workspace of ledb200_png_encode for N maps of H x W.
 * ledb200_png_encode: labels [N,H,W] contiguous, dtype LEDB200_U8 | LEDB200_I64, add 0 | 1.  out (capacity N * bound)
 *   receives the files back to back, file i at out[offsets[i] : offsets[i + 1]]; offsets: device int64 [N + 1].  The
 *   host reads offsets, then offsets[N] bytes of out.
 * ledb200_png_encode_lut: the same with pixels lut[label & 255] (lut: HOST 256 bytes; ledb200_png_encode is the table
 *   (i + add) & 255).  palette 1 writes colour type 3 and, before the IDAT, the 256-entry grey PLTE (entry i = (i, i, i))
 *   that PIL's Image.convert('P') gives a grayscale image (CityscapesMetric's labelId files); out then holds
 *   N * ledb200_png_lut_bound(H, W, 1) bytes.
 * ledb200_png_lut_bound: ledb200_png_bound plus the PLTE chunk when palette is 1.
 * ledb200_png_encode_rgb: rgb [N,H,W,3] uint8 contiguous (device) -> 8-bit RGB files (colour type 2), the drawn
 *   pictures of SegLocalVisualizer.  Each scanline takes the filter (None, Sub, Up, Average, Paeth) with the least sum
 *   of |signed residual| (libpng's heuristic).  ledb200_png_rgb_bound / ledb200_png_rgb_workspace_bytes size it; out
 *   and offsets as for ledb200_png_encode. */
int64_t ledb200_png_bound(int32_t H, int32_t W);
int64_t ledb200_png_lut_bound(int32_t H, int32_t W, int32_t palette);
int64_t ledb200_png_workspace_bytes(int32_t N, int32_t H, int32_t W);
int ledb200_png_encode(const void* labels, int32_t dtype, int32_t N, int32_t H, int32_t W, int32_t add, uint8_t* out,
                       int64_t* offsets, void* workspace, void* stream);
int ledb200_png_encode_lut(const void* labels, int32_t dtype, int32_t N, int32_t H, int32_t W, const uint8_t* lut,
                           int32_t palette, uint8_t* out, int64_t* offsets, void* workspace, void* stream);
int64_t ledb200_png_rgb_bound(int32_t H, int32_t W);
int64_t ledb200_png_rgb_workspace_bytes(int32_t N, int32_t H, int32_t W);
int ledb200_png_encode_rgb(const uint8_t* rgb, int32_t N, int32_t H, int32_t W, uint8_t* out, int64_t* offsets,
                           void* workspace, void* stream);

/* ---- segmentation overlays (csrc/visualize.cu) ---------------------------------------------------------------------------
 * mmseg's SegLocalVisualizer._draw_sem_seg on the device.
 * ledb200_seg_label_locations: labels [N,H,W] (LEDB200_U8 | LEDB200_I64, device, contiguous), 1 <= K <= 255.  out: device
 *   int32 [N,K,3] = (present, x, y) per class k < K: the row holding the most pixels of k (the first on a tie) and the
 *   pixel at index count / 2 of that row in x order (mmseg's _get_center_loc); (0, 0, 0) for an absent class.  Labels
 *   outside 0 .. K - 1 are not counted.  workspace: device, ledb200_seg_locate_workspace_bytes(N, H, K).
 * ledb200_seg_overlay: images [N,3,H,W] uint8 BGR (the decoders' layout), gt / pred [N,H,W] label maps of their own
 *   dtype (LEDB200_U8 | LEDB200_I64) or NULL (not both).  out [N,H,P*W,3] uint8 RGB, P = the number of non-NULL maps,
 *   gt panel first.  Pixel (y, x) of a panel is table[i * 256 + c] per channel, i the image's channel and c: the colour
 *   of the last stamp of that panel touching the pixel, else palette[label] for 0 <= label < K, else 0.  palette: device
 *   K x 3 RGB; table: device 256 x 256 (the caller's blend, e.g. uint8(i * (1 - alpha) + c * alpha) in float64).
 *   stamps: device array of num_stamps descriptors, drawn in array order; stamp_data: device bytes, 4 per stamp pixel
 *   (R, G, B, touched), row-major over the stamp's w x h box, stamp_bytes in all.  A descriptor whose box leaves its
 *   panel, the batch or stamp_data is skipped. */
typedef struct {
  int32_t image, panel;       /* batch index, panel 0 .. P - 1 */
  int32_t x0, y0, w, h;       /* the box in panel coordinates */
  int64_t offset;             /* byte offset of the box's pixels in stamp_data */
} ledb200_seg_stamp;
int64_t ledb200_seg_locate_workspace_bytes(int32_t N, int32_t H, int32_t K);
int ledb200_seg_label_locations(const void* labels, int32_t dtype, int32_t N, int32_t H, int32_t W, int32_t K,
                                int32_t* out, void* workspace, void* stream);
int ledb200_seg_overlay(const uint8_t* images, const void* gt, int32_t gt_dtype, const void* pred, int32_t pred_dtype,
                        int32_t N, int32_t H, int32_t W, int32_t K, const uint8_t* palette, const uint8_t* table,
                        const ledb200_seg_stamp* stamps, int32_t num_stamps, const uint8_t* stamp_data,
                        int64_t stamp_bytes, uint8_t* out, void* stream);

/* ---- PNG files -> decoded images and label maps (csrc/png_decode.cu) -----------------------------------------------------
 * The dataset feed of LoadImageFromFile (mmcv imfrombytes, cv2 backend, flag 'color') and LoadAnnotations (pillow backend,
 * 'unchanged') on the device.  Bit depth 8, colour types 0 / 2 / 3 / 4 / 6, no interlace; the caller reads the IHDR (at
 * its fixed offset) and rejects everything else before the call.
 *   LEDB200_PNG_COLOR: out [3,h,w] uint8 BGR, bit-identical to cv2.imdecode(buf, IMREAD_COLOR) transposed to CHW (grey
 *     replicated, palette expanded through PLTE, alpha dropped, tRNS / gAMA / other ancillary chunks ignored).
 *   LEDB200_PNG_LABEL: colour types 0 and 3 only; out [1,h,w] uint8 = lut[grey value or palette index] (lut: HOST 256
 *     bytes, NULL = identity), i.e. np.array(Image.open(f)) through the table.
 *   LEDB200_PNG_GREY16: bit depth 16, colour type 0 only (Cityscapes' *_gtFine_instanceIds.png); out [1,h,w] int32 =
 *     np.array(Image.open(f)), the big-endian 16-bit samples; lut is ignored.  The other modes read bit depth 8.
 * One descriptor per file (HOST array): data / size = the whole file (device), out = its output (device), h / w /
 * color_type as the IHDR states them (the device checks that they do).  status: device int32 [n], one LEDB200_PNG_*
 * code per file; a file with a non-zero status leaves its output undefined.  Every file is decoded at once (one warp
 * inflates each file; a block per file undoes the filters).  No file makes the kernels read outside it or write
 * outside its output and its workspace slot, whatever its content.
 * ledb200_png_decode_workspace_bytes: device workspace of one ledb200_png_decode call over these descriptors in the
 *   colour or label mode; ledb200_png_decode_mode_workspace_bytes: the same for any mode.
 * ledb200_png_decode_host: the same decoder on the CPU (diagnostics, like ledb200_debug_fetch): every pointer of the
 *   descriptors, status and lut are HOST memory; the statuses equal the device's. */
enum { LEDB200_PNG_COLOR = 0, LEDB200_PNG_LABEL = 1, LEDB200_PNG_GREY16 = 16 };
enum {
  LEDB200_PNG_OK = 0,
  LEDB200_PNG_EHEADER = 1,      /* signature or IHDR differs from the descriptor                                 */
  LEDB200_PNG_ECHUNK = 2,       /* chunk past the end of the file, bad chunk name, chunk order (PLTE after IDAT,
                                   split IDAT run, second PLTE / IHDR), unknown critical chunk, no IDAT / IEND     */
  LEDB200_PNG_ECRC = 3,         /* CRC-32 of a critical chunk (IDAT, PLTE, IEND)                                 */
  LEDB200_PNG_EPLTE = 4,        /* palette image without a valid PLTE                                            */
  LEDB200_PNG_EUNSUPPORTED = 5, /* an eXIf chunk (cv2 would apply its orientation)                               */
  LEDB200_PNG_EZLIB = 6,        /* zlib header (method, window, preset dictionary, check bits), data after the
                                   end of the zlib stream                                                        */
  LEDB200_PNG_EDEFLATE = 7,     /* invalid deflate data: block type, stored length, Huffman code (over-subscribed,
                                   incomplete, no end-of-block), symbol, distance before the start of the stream */
  LEDB200_PNG_ETRUNC = 8,       /* the zlib stream ends early                                                    */
  LEDB200_PNG_ESIZE = 9,        /* the inflated scanlines are not exactly h * (1 + w * bytes per pixel) bytes     */
  LEDB200_PNG_EADLER = 10,      /* Adler-32 of the inflated scanlines                                            */
  LEDB200_PNG_EFILTER = 11      /* a scanline filter type above 4                                                */
};
typedef struct {
  const uint8_t* data;
  int64_t size;
  uint8_t* out;
  int32_t h, w, color_type;
} ledb200_png_file;
int64_t ledb200_png_decode_workspace_bytes(const ledb200_png_file* files, int32_t n);
int64_t ledb200_png_decode_mode_workspace_bytes(const ledb200_png_file* files, int32_t n, int32_t mode);
int ledb200_png_decode(const ledb200_png_file* files, int32_t n, int32_t mode, const uint8_t* lut, void* workspace,
                       int32_t* status, void* stream);
int ledb200_png_decode_host(const ledb200_png_file* files, int32_t n, int32_t mode, const uint8_t* lut, int32_t* status);

/* ---- Cityscapes pixel-level statistics (csrc/cityscapes.cu) --------------------------------------------------------------
 * CityscapesMetric's evaluation (cityscapesscripts evalPixelLevelSemanticLabeling.evaluatePair, evalInstLevelScore) for N
 * same-shape images: pred [N,H,W] trainIds (LEDB200_U8 | LEDB200_I64), gt [N,H,W] uint8 labelIds, inst [N,H,W] int32
 * instanceIds, all device and contiguous.  Tables (HOST): train_to_id[256] maps a trainId to its labelId; category[34]
 * is each labelId's instance category (-1: none); inst_rule[34] says what an instance id id > 1000 of class id / 1000
 * does: 0 error, 1 skipped (ignoreInEval), 2 counted (only ids 24 .. 33 of a category).
 * cm_inout: device int64 [34,34] (rows GT, columns prediction), accumulated; cm_last_out (device int64 [34,34] or NULL)
 * receives the matrix of image N - 1 alone.  out: device int32 of ledb200_cityscapes_out_ints(N): statuses [N] (bits:
 * 1 a GT labelId above 33, 2 a predicted labelId outside 0 .. 33, 4 an instance id of a class neither counted nor
 * skipped or above 33, 8 an int64 prediction outside 0 .. 255), record counts [N], then the records (instId, size, tp,
 * catTp) of every counted instance, image after image, in ascending instId.  workspace: device,
 * ledb200_cityscapes_workspace_bytes(N).  Every count is an exact integer. */
int64_t ledb200_cityscapes_out_ints(int32_t N);
int64_t ledb200_cityscapes_workspace_bytes(int32_t N);
int ledb200_cityscapes_accumulate(const void* pred, int32_t pred_dtype, const uint8_t* gt, const int32_t* inst,
                                  int32_t N, int32_t H, int32_t W, const int32_t* train_to_id, const int8_t* category,
                                  const int8_t* inst_rule, int64_t* cm_inout, int64_t* cm_last_out, int32_t* out,
                                  void* workspace, void* stream);

/* ---- baseline JPEG files -> decoded images (csrc/jpeg_decode.cu) ---------------------------------------------------------
 * LoadImageFromFile (mmcv imfrombytes, cv2 backend, flag 'color') on the device for JPEG files: out [3,h,w] uint8 BGR,
 * bit-identical to cv2.imdecode(buf, IMREAD_COLOR) transposed to CHW (libjpeg-turbo, JDCT_ISLOW, fancy upsampling).
 * Supported: SOF0 / SOF1, 8-bit precision, Huffman coding, one interleaved scan carrying every component; 1 component
 * (grey, replicated) or 3 that libjpeg treats as YCbCr, with luma sampling factors in {1, 2} x {1, 2} and chroma 1 x 1
 * (4:4:4, 4:2:2, 4:2:0, 4:4:0); any restart interval.  The caller walks the markers to the first SOS and refuses the
 * rest before the call (lednet_b200.ops.jpeg_info); the device refuses them too, with LEDB200_JPEG_EUNSUPPORTED.
 * Unlike libjpeg, which warns and fills the rest of the image with grey, corrupt entropy-coded data is an error.
 * One descriptor per file (HOST array): data / size = the whole file (device, size < 2^28), out = its output (device),
 * h / w / components as the frame header states them (the device checks that they do).  status: device int32 [n], one
 * LEDB200_JPEG_* code per file; a file with a non-zero status leaves its output undefined.  Every file of a call is
 * decoded by one sequence of launches, and every stage but the header walk splits each file over many threads.  No
 * file makes the kernels read outside it or write outside its output and its workspace slot, whatever its content.
 * ledb200_jpeg_decode_workspace_bytes: device workspace of one ledb200_jpeg_decode call over these descriptors (a
 *   bound that holds for every accepted sampling).
 * ledb200_jpeg_decode_host: the same decoder on the CPU (diagnostics): every pointer of the descriptors and status is
 *   HOST memory; the statuses equal the device's. */
enum {
  LEDB200_JPEG_OK = 0,
  LEDB200_JPEG_EHEADER = 1,     /* no SOI, or the frame header's height, width or components differ from the
                                   descriptor                                                                    */
  LEDB200_JPEG_ESEGMENT = 2,    /* marker structure: a segment length past the end of the file or wrong for its
                                   marker, a marker out of place (a second SOF, SOS before SOF, RSTn / EOI / DNL
                                   before the scan, an unknown marker), the scan not followed by EOI, zero width   */
  LEDB200_JPEG_EUNSUPPORTED = 3,/* progressive, lossless, hierarchical or arithmetic-coded, not 8-bit, 2 or 4
                                   components, RGB colour space, other sampling factors, a non-interleaved scan,
                                   height 0 (DNL), an Exif orientation other than 1 (cv2 would rotate)             */
  LEDB200_JPEG_ETABLE = 4,      /* bad DQT / DHT (table class or id, length, over-subscribed or all-ones Huffman
                                   code, DC symbol above 15), or a table the frame or scan refers to is missing  */
  LEDB200_JPEG_EHUFF = 5,       /* a bit pattern that is no code of the Huffman table in use                     */
  LEDB200_JPEG_ETRUNC = 6,      /* the entropy-coded data ends before the last MCU (of the scan or an interval) */
  LEDB200_JPEG_ERESTART = 7,    /* an RSTn out of sequence, or more or fewer RSTn than the restart interval needs */
  LEDB200_JPEG_EZZ = 8          /* an AC run that takes the coefficient index past 63                            */
};
typedef struct {
  const uint8_t* data;
  int64_t size;
  uint8_t* out;
  int32_t h, w, components;
} ledb200_jpeg_file;
int64_t ledb200_jpeg_decode_workspace_bytes(const ledb200_jpeg_file* files, int32_t n);
int ledb200_jpeg_decode(const ledb200_jpeg_file* files, int32_t n, void* workspace, int32_t* status, void* stream);
int ledb200_jpeg_decode_host(const ledb200_jpeg_file* files, int32_t n, int32_t* status);

/* ---- layer-level operators for module compositions outside the R0 plan (the LED wiring, led_variant.py) ---------------
 * A conv layer handle is ONE mmcv ConvModule (mmcv/cnn/bricks/conv_module.py; conv k = 1 | 3, stride 1 | 2, padding k/2)
 * whose BatchNorm the caller folded into `weight` (OIHW, HOST fp32) / `bias` (nullable); `pre_scale` / `pre_shift`
 * (nullable, HOST [Cin]) are the folded BN of a pre-activation module (order norm, act, conv: ppm.py:57-117), applied
 * as relu(a x + b) in the conv prologue.  groups == Cin == Cout selects the depthwise 3x3 (stdc.py:52-61).  The weights
 * stay on the device in both conv layouts; forward is one launch: the tcgen05 kernel for bf16 tensors of eligible
 * shape (backend 0 / 2), else the CUDA-core kernel (backend 1 forces it).  out = [relu](conv(in) + bias [+ residual]).
 * in / out / residual: NHWC of `dtype` (F32 | BF16) with pixel strides in elements (0 = dense), so a layer can read /
 * write a channel slice of a wider buffer (concat without a copy). */
typedef struct ledb200_conv_layer ledb200_conv_layer;
int ledb200_conv_layer_create(const float* weight, const float* bias, const float* pre_scale, const float* pre_shift,
                              int32_t Cin, int32_t Cout, int32_t ksize, int32_t stride, int32_t groups,
                              ledb200_conv_layer** out);
int ledb200_conv_layer_forward(ledb200_conv_layer* layer, const void* in, void* out, const void* residual, int32_t dtype,
                               int32_t N, int32_t H, int32_t W, int32_t in_ld, int32_t out_ld, int32_t res_ld, int32_t relu,
                               int32_t backend, void* stream);
int ledb200_conv_layer_destroy(ledb200_conv_layer* layer);
/* The same layer fed by the caller's image (NCHW fp32, 3 channels): the stem convolution of a composed trunk.  bf16 output
 * with stride 2 and Cout 16 / 32 runs the tensor-core stem kernel (csrc/stem_tc.cu), anything else the CUDA-core one. */
int ledb200_conv_layer_forward_image(ledb200_conv_layer* layer, const void* img, int32_t img_layout, void* out, int32_t dtype,
                                     int32_t N, int32_t H, int32_t W, int32_t out_ld, int32_t relu, void* stream);
/* The whole DAPPM (mmseg/models/utils/ppm.py:57-130) as a handle: two launches per forward (csrc/dappm.cu: pooled branches,
 * then ONE clustered tcgen05 kernel for scales[0], the four 3x3 processes, the concat-free compression and the shortcut).
 * Every ConvModule of the module is pre-activation (norm, act, conv): `weight` OIHW HOST fp32, `bias` nullable, bn_scale /
 * bn_shift = the folded BatchNorm on the INPUT channels (y = relu(a x + b)).  scales5[0] is scales[0], scales5[i] the conv of
 * the pooled branch i.  x [N,H,W,C], out [N,H,W,Cout], NHWC dense BF16; ledb200_dappm_eligible() says whether a shape fits
 * (C % 64 == 0, ppm = out channels = 128, at most 8 tiles of 16 x 8 pixels per image). */
typedef struct { const float* weight; const float* bias; const float* bn_scale; const float* bn_shift; } ledb200_preact_conv;
typedef struct ledb200_dappm ledb200_dappm;
int ledb200_dappm_create(int32_t C, int32_t P, int32_t Cout, const ledb200_preact_conv* scales5,
                         const ledb200_preact_conv* processes4, const ledb200_preact_conv* compression,
                         const ledb200_preact_conv* shortcut, ledb200_dappm** out);
int ledb200_dappm_eligible(int32_t dtype, int32_t N, int32_t H, int32_t W, int32_t C, int32_t P, int32_t Cout);
int ledb200_dappm_forward(ledb200_dappm* d, const void* x, void* out, int32_t dtype, int32_t N, int32_t H, int32_t W, void* stream);
int ledb200_dappm_destroy(ledb200_dappm* d);
/* nn.AvgPool2d(k, s, p) with count_include_pad=True (stdc.py:80, ppm.py:68-90), or the global average when k == 0;
 * F.interpolate(mode='bilinear', align_corners=False) (mmseg/models/utils/wrappers.py:8-27); out = [relu](a [+ b]).
 * NHWC F32 | BF16, C a multiple of 8, pixel strides in elements (0 = dense). */
int ledb200_avgpool2d(const void* in, void* out, int32_t dtype, int32_t N, int32_t H, int32_t W, int32_t C, int32_t k, int32_t s,
                      int32_t p, int32_t in_ld, int32_t out_ld, void* stream);
int ledb200_resize_bilinear(const void* in, void* out, int32_t dtype, int32_t N, int32_t h, int32_t w, int32_t H, int32_t W,
                            int32_t C, int32_t in_ld, int32_t out_ld, void* stream);
int ledb200_add_relu(const void* a, const void* b, void* out, int32_t dtype, int64_t npix, int32_t C, int32_t a_ld, int32_t b_ld,
                     int32_t out_ld, int32_t relu, void* stream);

/* ---- SEAM edge gate (SURVEY section 8(f) rank 1) -----------------------------------------------------
 * The inline edge path of the authors' speed prototype (tools/speed/ddrnet_speed.py:282-338, 388-389), eval mode:
 *   e = minmax_normalise(BN(conv3x3 C->1 (x))) over the whole tensor; b_s = [clamp(laplacian_stride_s(e), 0) > t] for
 *   s = 1, 2, 4 (strided maps nearest-upsampled); m = [0.6 b_1 + 0.3 b_2 + 0.1 b_4 > t]; out = BN(conv3x3 1->C (m)) * x_s + x_s.
 * x / x_s / out: NHWC of `dtype` (F32 or BF16), C a multiple of 8.  `params`: device fp32 block of
 * ledb200_seam_param_floats(C) floats: w1[9][C] (tap major), a1, b1, six pad floats, w2[9][C], a2[C], b2[C] (BatchNorm folded to
 * y = a * conv + b).  `workspace`: ledb200_seam_workspace_bytes(N, H, W) bytes. */
int64_t ledb200_seam_param_floats(int32_t C);
int64_t ledb200_seam_workspace_bytes(int32_t N, int32_t H, int32_t W);
int ledb200_seam_forward(const void* x, const void* x_s, void* out, int32_t dtype, int32_t N, int32_t H, int32_t W,
                         int32_t C, float threshold, const float* params, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LEDB200_H_ */
