"""Functional wrappers over the stand-alone C-ABI kernels (include/ledb200.h).

Layout changes between the reference's NCHW tensors and the library's NHWC are views/copies made
with torch (plumbing); the arithmetic is in the CUDA kernels.
"""
import ctypes as C
import struct
import zlib

import numpy as np
import torch

from . import lib as L


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def fold_bn(bn):
    """Eval BatchNorm as a per-channel affine in float64: (scale, shift) = (gamma / sqrt(var + eps), beta - mean * scale)."""
    scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps)
    return scale, bn.bias.detach().double() - bn.running_mean.detach().double() * scale


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise L.LedB200Error('LED-Net B200 ops need CUDA tensors (no CPU fallback)')


def head_fuse_argmax(xc, hx2, hx1, pred_dtype=torch.uint8, want_logits=False, channels_last=False):
    """predict_by_feat + argmax (decode_head.py:362-379, base.py:187-188).

    xc/hx2/hx1: [N,K,h,w] (NCHW, default) or [N,h,w,K] (channels_last=True), fp32 or bf16.
    Returns (pred [N,2*h2,2*w2], logits or None)."""
    _need_cuda(xc, hx2, hx1)
    if not channels_last:
        xc, hx2, hx1 = (t.permute(0, 2, 3, 1).contiguous() for t in (xc, hx2, hx1))
    else:
        xc, hx2, hx1 = (t.contiguous() for t in (xc, hx2, hx1))
    assert xc.dtype == hx2.dtype == hx1.dtype and xc.dtype in (torch.float32, torch.bfloat16)
    N, hc, wc, K = xc.shape
    _, h4, w4, _ = hx2.shape
    _, h2, w2, _ = hx1.shape
    pred = torch.empty((N, 2 * h2, 2 * w2), dtype=pred_dtype, device=xc.device)
    logits = torch.empty((N, K, 2 * h2, 2 * w2), dtype=torch.float32, device=xc.device) if want_logits else None
    L.check(L.get().ledb200_head_fuse_argmax(
        _p(xc), _p(hx2), _p(hx1), L.torch_dtype_code(xc), N, K, hc, wc, h4, w4, h2, w2, _p(pred),
        L.torch_dtype_code(pred), _p(logits), L.stream_ptr(xc.device)), 'ledb200_head_fuse_argmax')
    return pred, logits


def confusion_accumulate(pred, gt, num_classes, ignore_index=255, cm=None):
    """cm[(K+1),K] int64 += bincount(K*gt+pred) over gt != ignore (rows GT; row K = out-of-range GT)."""
    _need_cuda(pred, gt)
    pred, gt = pred.contiguous(), gt.contiguous()
    assert pred.numel() == gt.numel(), 'prediction and label must have the same number of pixels'
    if cm is None:
        cm = torch.zeros((num_classes + 1, num_classes), dtype=torch.int64, device=pred.device)
    L.check(L.get().ledb200_confusion_accumulate(
        _p(pred), _p(gt), L.torch_dtype_code(pred), L.torch_dtype_code(gt), pred.numel(), num_classes,
        ignore_index, _p(cm), L.stream_ptr(pred.device)), 'ledb200_confusion_accumulate')
    return cm


def ohem_ce(score, target, ignore_label=255, thres=0.7, min_kept=100000, loss_weight=1.0,
            class_weight=None, want_grad=False):
    """Returns (out3 = [loss, kept, accuracy%] device tensor, dlogits or None)."""
    _need_cuda(score, target)
    score = score.contiguous().float()
    target = target.contiguous().to(torch.int64)
    N, K, H, W = score.shape
    lib = L.get()
    ws = torch.empty(lib.ledb200_ohem_workspace_bytes(N * H * W), dtype=torch.uint8, device=score.device)
    out3 = torch.empty(3, dtype=torch.float32, device=score.device)
    grad = torch.empty_like(score) if want_grad else None
    cw = None
    if class_weight is not None:
        cw = torch.as_tensor(class_weight, dtype=torch.float32, device=score.device).contiguous()
        assert cw.numel() == K
    L.check(lib.ledb200_ohem_ce(_p(score), _p(target), N, K, H, W, ignore_label, float(thres),
                                int(min_kept), float(loss_weight), _p(cw), _p(out3), _p(grad), _p(ws),
                                L.stream_ptr(score.device)), 'ledb200_ohem_ce')
    return out3, grad


def conv2d(x_nhwc, weight_oihw, bias=None, stride=1, relu=False, residual=None, pre_scale=None,
           pre_shift=None, backend=0):
    """One convolution (3x3 pad 1 or 1x1) on an NHWC fp32/bf16 CUDA tensor; weights host fp32."""
    _need_cuda(x_nhwc, residual)
    x = x_nhwc.contiguous()
    N, H, W, Cin = x.shape
    w = weight_oihw.detach().to('cpu', torch.float32).contiguous()
    Cout, _, k, _ = w.shape
    pad = k // 2
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    # 16-byte pixels for the tensor-core path: Cout 19 -> pixel stride 24, like the engine's buffers
    ld = (Cout + 7) // 8 * 8
    out_full = torch.empty((N, Ho, Wo, ld), dtype=x.dtype, device=x.device)
    host = [None if t is None else t.detach().to('cpu', torch.float32).contiguous()
            for t in (bias, pre_scale, pre_shift)]
    res = None
    if residual is not None:
        res = residual.new_zeros((N, Ho, Wo, ld))
        res[..., :Cout] = residual
    L.check(L.get().ledb200_conv2d(_p(x), _p(out_full), _p(res), L.torch_dtype_code(x), N, H, W, Cin, Cout, k,
                                   stride, int(relu), _p(w), _p(host[0]), _p(host[1]), _p(host[2]),
                                   backend, Cin, ld, ld, L.stream_ptr(x.device)), 'ledb200_conv2d')
    return out_full[..., :Cout]


_FLIP = {None: 0, False: 0, 'horizontal': 1, 'vertical': 2}


def postprocess(seg_logit, padding=None, flip=None, ori_shape=None, align_corners=False, threshold=0.3,
                pred_dtype=torch.int64, want_logits=True):
    """BaseSegmentor.postprocess_result for ONE image (base.py:153-198): seg_logit fp32 [K,H,W] -> crop `padding`
    (left, right, top, bottom), undo `flip` ('horizontal' | 'vertical' | None), bilinear resize to `ori_shape`,
    argmax (K > 1) or sigmoid > threshold (K == 1).  Returns (pred [1,h,w], logits [K,h,w] or None)."""
    _need_cuda(seg_logit)
    x = seg_logit.contiguous().float()
    K, H, W = x.shape
    pad = tuple(int(v) for v in (padding if padding is not None else (0, 0, 0, 0)))
    assert flip in (None, False, 'horizontal', 'vertical'), flip
    oh, ow = (int(v) for v in ori_shape) if ori_shape is not None else (H - pad[2] - pad[3], W - pad[0] - pad[1])
    if K == 1:
        pred_dtype = torch.float32                    # (sigmoid > threshold).to(seg_logits) in the reference
    pred = torch.empty((1, oh, ow), dtype=pred_dtype, device=x.device)
    out = torch.empty((K, oh, ow), dtype=torch.float32, device=x.device) if want_logits else None
    pad_c = (C.c_int32 * 4)(*pad)
    L.check(L.get().ledb200_postprocess(_p(x), K, H, W, pad_c, _FLIP[flip],
                                        oh, ow, int(bool(align_corners)), float(threshold), _p(pred),
                                        L.torch_dtype_code(pred), _p(out), L.stream_ptr(x.device)), 'ledb200_postprocess')
    return pred, out


def tta_merge(views, ori_shape, align_corners=False, mode=0, threshold=0.3, pred_dtype=torch.int64, want_pred=True,
              want_probs=False, pred=None):
    """SegTTAModel.merge_preds (seg_tta.py) over every view of N images in ONE launch.

    views: list (1..32, augmentation order) of (logits, padding, flip): logits fp32 [N,K,H,W] on the device whose images
    are each [K,H,W]-contiguous (a slice of a larger engine batch is used in place), padding (left, right, top, bottom)
    or None, flip 'horizontal' | 'vertical' | None.  Each view is post-processed exactly as `postprocess` does (un-pad,
    un-flip, bilinear resize to `ori_shape`), soft-maxed over K (mode 0: out_channels > 1) or sigmoid-ed (mode 1:
    out_channels == 1), summed in order and divided by the number of views.
    Returns (pred, probs): pred = argmax [N,oh,ow] of `pred_dtype` (mode 0) or the float mask merged > threshold
    [N,K,oh,ow] (mode 1), None unless want_pred (written into `pred` when given); probs = the merged fp32 [N,K,oh,ow]
    when want_probs, else None."""
    V = len(views)
    flat = []
    for lg, _, _ in views:
        _need_cuda(lg)
        lg = lg.float()
        assert lg.dim() == 4, 'view logits are [N,K,H,W]'
        if not lg[0].is_contiguous():
            lg = lg.contiguous()
        flat.append(lg)
    N, K = (flat[0].shape[0], flat[0].shape[1]) if flat else (1, 1)
    assert all(t.shape[0] == N for t in flat), 'every view must hold the same images'
    assert all(t.shape[1] == K for t in flat), 'every view must have the same number of classes'
    oh, ow = (int(v) for v in ori_shape)
    arr = (L.TtaView * max(V, 1))()
    for d, t, (_, padding, flip) in zip(arr, flat, views):
        d.logits, d.image_stride, d.H, d.W = t.data_ptr(), t.stride(0), t.shape[2], t.shape[3]
        d.pad_lrtb[:] = [int(v) for v in (padding if padding is not None else (0, 0, 0, 0))]
        d.flip = _FLIP[flip]
    dev = flat[0].device if flat else torch.device('cuda', torch.cuda.current_device())
    if pred is not None:
        _need_cuda(pred)
        assert pred.is_contiguous() and pred.numel() == N * oh * ow * (K if mode == 1 else 1), 'pred has the wrong shape'
    elif want_pred:
        pred = (torch.empty((N, K, oh, ow), dtype=torch.float32, device=dev) if mode == 1 else
                torch.empty((N, oh, ow), dtype=pred_dtype, device=dev))
    probs = torch.empty((N, K, oh, ow), dtype=torch.float32, device=dev) if want_probs else None
    L.check(L.get().ledb200_tta_merge(arr, V, N, K, oh, ow, int(bool(align_corners)), int(mode), float(threshold),
                                      _p(pred), L.torch_dtype_code(pred) if pred is not None else L.I64, _p(probs),
                                      L.stream_ptr(dev)), 'ledb200_tta_merge')
    return pred, probs


def slide_accumulate(preds, count, crop_logits, y1, x1):
    """preds[:, :, y1:y1+hc, x1:x1+wc] += crop_logits; count[:, :, same] += 1 (encoder_decoder.py:283-287)."""
    _need_cuda(preds, count, crop_logits)
    assert preds.is_contiguous() and count.is_contiguous() and preds.dtype == count.dtype == torch.float32
    crop = crop_logits.contiguous().float()
    N, K, H, W = preds.shape
    _, _, hc, wc = crop.shape
    L.check(L.get().ledb200_slide_accumulate(_p(preds), _p(count), _p(crop), N, K, H, W, hc, wc, int(y1), int(x1),
                                             L.stream_ptr(preds.device)), 'ledb200_slide_accumulate')


def slide_finalize(preds, count, want_pred=False, pred_dtype=torch.int64):
    """preds /= count in place (encoder_decoder.py:290); optionally also argmax over K -> [N,H,W]."""
    _need_cuda(preds, count)
    N, K, H, W = preds.shape
    pred = torch.empty((N, H, W), dtype=pred_dtype, device=preds.device) if want_pred else None
    L.check(L.get().ledb200_slide_finalize(_p(preds), _p(count), N, K, H, W, _p(pred),
                                           L.torch_dtype_code(pred) if want_pred else L.I64,
                                           L.stream_ptr(preds.device)), 'ledb200_slide_finalize')
    return preds, pred


def slide_merge(crop_logits, origins, n_images, image_hw, want_logits=True, want_pred=False, pred_dtype=torch.int64):
    """All crop windows of slide_inference at once: crop_logits fp32 [G*N,K,hc,wc] (window g of image n at g*N+n),
    origins = [(y1, x1)] * G in the reference's grid order -> (logits [N,K,H,W] or None, pred [N,H,W] or None)."""
    _need_cuda(crop_logits)
    crop = crop_logits.contiguous().float()
    G, N = len(origins), int(n_images)
    GN, K, hc, wc = crop.shape
    assert GN == G * N, 'crop batch must hold every window of every image'
    H, W = (int(v) for v in image_hw)
    out = torch.empty((N, K, H, W), dtype=torch.float32, device=crop.device) if want_logits else None
    pred = torch.empty((N, H, W), dtype=pred_dtype, device=crop.device) if want_pred else None
    y1 = (C.c_int32 * G)(*[int(o[0]) for o in origins])
    x1 = (C.c_int32 * G)(*[int(o[1]) for o in origins])
    L.check(L.get().ledb200_slide_merge(_p(crop), G, y1, x1, N, K, H, W, hc, wc, _p(out), _p(pred),
                                        L.torch_dtype_code(pred) if want_pred else L.I64,
                                        L.stream_ptr(crop.device)), 'ledb200_slide_merge')
    return out, pred


def stack_pad(img, out, swap_rb=False, mean=None, std=None, pad_val=0.0, label=None, label_out=None, seg_pad_val=255):
    """SegDataPreProcessor + stack_batch for one sample: img [3,h,w] uint8 / fp32 -> out [3,Hp,Wp] fp32 (a slice of the
    batch tensor), label [h,w] or [1,h,w] uint8 / int64 -> label_out [Hp,Wp] int64."""
    _need_cuda(img, out, label, label_out)
    img = img.contiguous()
    assert img.dim() == 3 and img.shape[0] == 3 and out.is_contiguous() and out.dtype == torch.float32
    if img.dtype not in (torch.uint8, torch.float32):
        img = img.float()
    if label is not None:
        label = label.reshape(label.shape[-2:]).contiguous()
        if label.dtype not in (torch.uint8, torch.int64):
            label = label.to(torch.int64)
        assert label_out.is_contiguous() and label_out.dtype == torch.int64
    m3 = (C.c_float * 3)(*[float(v) for v in mean]) if mean is not None else None
    s3 = (C.c_float * 3)(*[float(v) for v in std]) if std is not None else None
    L.check(L.get().ledb200_stack_pad(_p(img), L.torch_dtype_code(img), img.shape[1], img.shape[2], int(bool(swap_rb)),
                                      m3, s3, float(pad_val), _p(out), out.shape[-2], out.shape[-1], _p(label),
                                      L.torch_dtype_code(label) if label is not None else L.U8, _p(label_out),
                                      int(seg_pad_val), L.stream_ptr(img.device)), 'ledb200_stack_pad')
    return out


MAX_AUG_SAMPLES = 64          # ledb200_train_augment's descriptors per call


def _aug_desc(p, img, lab):
    d = L.AugSample()
    d.img, d.label = img.data_ptr(), lab.data_ptr()
    d.h, d.w = img.shape[1], img.shape[2]
    d.rh, d.rw = (int(v) for v in p['resized_hw'])
    cands = p['candidates']
    if not 1 <= len(cands) <= 11:
        raise L.LedB200Error(f'train_augment: {len(cands)} candidate boxes (1 .. 11 per sample)')
    d.num_candidates = len(cands)
    for k, (oy, ox) in enumerate(cands):
        d.offsets[k][0], d.offsets[k][1] = int(oy), int(ox)
    d.flip = int(bool(p['flip']))
    d.contrast_mode = int(p['contrast_mode'])
    d.brightness, d.beta = p['brightness'] is not None, p['brightness'] or 0.0
    d.contrast, d.contrast_alpha = p['contrast'] is not None, p['contrast'] or 1.0
    d.saturation, d.saturation_alpha = p['saturation'] is not None, p['saturation'] or 1.0
    d.hue, d.hue_delta = p['hue'] is not None, int(p['hue'] or 0)
    return d


def train_augment(imgs, labels, params, crop_size, out, label_out, cat_max_ratio=1.0, ignore_index=255,
                  swap_rb=False, mean=None, std=None, pad_val=0.0, seg_pad_val=255, crop_index=None):
    """RandomResize -> RandomCrop -> RandomFlip -> PhotoMetricDistortion -> SegDataPreProcessor on the device, with the
    random draws given: imgs [3,h,w] uint8 (BGR as decoded), labels [h,w] or [1,h,w] uint8 / int64, params one dict per
    sample (lednet_b200.augment.draw_sample's format: resized_hw, candidates [(offset_h, offset_w)] (1 .. 11),
    flip, brightness / contrast / saturation / hue (None when the step does not fire), contrast_mode).
    crop_size (h, w); out [N,3,Hp,Wp] fp32 and label_out [N,Hp,Wp] int64, contiguous.  When a sample has several
    candidates, crop_select picks the first that passes cat_max_ratio (the last one otherwise) into crop_index
    (int32 [N], allocated when None) and that box is used.  Returns crop_index (None when every sample has one)."""
    N = len(imgs)
    assert len(labels) == N == len(params) and N >= 1
    _need_cuda(out, label_out, *imgs, *labels)
    assert out.is_contiguous() and out.dtype == torch.float32 and out.shape[:2] == (N, 3)
    assert label_out.is_contiguous() and label_out.dtype == torch.int64 and label_out.numel() == N * out[0, 0].numel()
    for t in imgs:
        if t.dtype != torch.uint8 or t.dim() != 3 or t.shape[0] != 3:
            raise L.LedB200Error('train_augment: images are [3, h, w] uint8')
    imgs = [t.contiguous() for t in imgs]
    ldt = torch.uint8 if all(t.dtype == torch.uint8 for t in labels) else torch.int64
    labels = [t.reshape(t.shape[-2:]).to(ldt).contiguous() for t in labels]
    for t, lab in zip(imgs, labels):
        if tuple(lab.shape) != tuple(t.shape[1:]):
            raise L.LedB200Error('train_augment: a label differs in size from its image')
    ch, cw = (int(v) for v in crop_size)
    Hp, Wp = out.shape[-2:]
    select = any(len(p['candidates']) > 1 for p in params)
    if select and crop_index is None:
        crop_index = torch.empty(N, dtype=torch.int32, device=out.device)
    lab_code = L.torch_dtype_code(labels[0])
    m3 = (C.c_float * 3)(*[float(v) for v in mean]) if mean is not None else None
    s3 = (C.c_float * 3)(*[float(v) for v in std]) if std is not None else None
    lib, st = L.get(), L.stream_ptr(out.device)
    lout = label_out.view(N, Hp, Wp)
    for i0 in range(0, N, MAX_AUG_SAMPLES):
        i1 = min(N, i0 + MAX_AUG_SAMPLES)
        arr = (L.AugSample * (i1 - i0))(*[_aug_desc(params[i], imgs[i], labels[i]) for i in range(i0, i1)])
        ci = crop_index[i0:i1] if crop_index is not None else None
        if select:
            L.check(lib.ledb200_crop_select(arr, i1 - i0, ch, cw, lab_code, float(cat_max_ratio), int(ignore_index),
                                            _p(ci), st), 'ledb200_crop_select')
        L.check(lib.ledb200_train_augment(arr, i1 - i0, ch, cw, lab_code, _p(ci), int(bool(swap_rb)), m3, s3,
                                          float(pad_val), _p(out[i0:i1]), Hp, Wp, _p(lout[i0:i1]), int(seg_pad_val),
                                          st), 'ledb200_train_augment')
    return crop_index


MAX_VIEWS = 64                # ledb200_view_resize's descriptors per call


def view_resize(imgs, resized_hw, out=None, out_flip=None, swap_rb=False, mean=None, std=None, pad_val=0.0):
    """mmcv Resize (keep_ratio, cv2 INTER_LINEAR) + optional horizontal RandomFlip + SegDataPreProcessor on the device:
    imgs N [3,h,w] uint8 (BGR as decoded), resized_hw one (rh, rw) for all or one per image (mmcv's arithmetic,
    lednet_b200.augment.view_size).  out / out_flip: [N,3,Hp,Wp] fp32 contiguous (one may be None) receive the unflipped
    / flipped view of image n at index n, swapped, normalised and padded with pad_val to Hp x Wp, as SegDataPreProcessor
    writes a view the CPU pipeline resized.  Returns (out, out_flip)."""
    N = len(imgs)
    assert N >= 1 and (out is not None or out_flip is not None)
    _need_cuda(out, out_flip, *imgs)
    for t in imgs:
        if t.dtype != torch.uint8 or t.dim() != 3 or t.shape[0] != 3:
            raise L.LedB200Error('view_resize: images are [3, h, w] uint8')
    imgs = [t.contiguous() for t in imgs]
    if len(resized_hw) == 2 and not isinstance(resized_hw[0], (tuple, list)):
        resized_hw = [resized_hw] * N
    assert len(resized_hw) == N
    ref = out if out is not None else out_flip
    Hp, Wp = ref.shape[-2:]
    for t in (out, out_flip):
        if t is not None:
            assert t.is_contiguous() and t.dtype == torch.float32 and tuple(t.shape) == (N, 3, Hp, Wp)
    m3 = (C.c_float * 3)(*[float(v) for v in mean]) if mean is not None else None
    s3 = (C.c_float * 3)(*[float(v) for v in std]) if std is not None else None
    lib, st = L.get(), L.stream_ptr(ref.device)
    for i0 in range(0, N, MAX_VIEWS):
        i1 = min(N, i0 + MAX_VIEWS)
        arr = (L.ViewDesc * (i1 - i0))()
        for d, i in zip(arr, range(i0, i1)):
            d.src = imgs[i].data_ptr()
            d.out = out[i].data_ptr() if out is not None else None
            d.out_flip = out_flip[i].data_ptr() if out_flip is not None else None
            d.h, d.w = imgs[i].shape[1], imgs[i].shape[2]
            d.rh, d.rw = (int(v) for v in resized_hw[i])
        L.check(lib.ledb200_view_resize(arr, i1 - i0, Hp, Wp, int(bool(swap_rb)), m3, s3, float(pad_val), st),
                'ledb200_view_resize')
    return out, out_flip


def png_encode(labels, add=0, lut=None, palette=False):
    """Label maps or RGB images -> PNG files on the device.

    A [N,H,W,3] uint8 tensor is N RGB images: each file is an 8-bit RGB PNG (colour type 2) that decodes to exactly
    those pixels (cv2.imdecode gives them in BGR order); add / lut / palette do not apply.
    Otherwise labels [H,W], [1,H,W] or [N,H,W], CUDA uint8 or int64.  Returns N `bytes`,
    each an 8-bit grayscale PNG of (label + add) mod 256 (add 0 or 1: mmseg's reduce_zero_label), which decodes to the
    pixels of `Image.fromarray((label + add).astype(np.uint8))`.  With `lut` (256 values in 0 .. 255) the pixels are
    lut[label mod 256] instead; `add` and `lut` do not go together.  palette=True writes a palette file (colour type 3)
    with PIL's 256-entry grey palette, what `Image.fromarray(x).convert('P').save(f)` writes: the same pixel values, read
    back in mode 'P'.  One launch sequence, then two copies back: the offsets and the files."""
    _need_cuda(labels)
    if lut is not None and add:
        raise L.LedB200Error('png_encode: give either add or lut, not both')
    if labels.dim() == 4:
        return _png_encode_rgb(labels, add, lut, palette)
    if labels.dtype not in (torch.uint8, torch.int64):
        raise L.LedB200Error('png_encode: labels must be uint8 or int64')
    if labels.dim() == 2:
        labels = labels[None]
    if labels.dim() != 3:
        raise L.LedB200Error('png_encode: labels must be [H, W] or [N, H, W]')
    labels = labels.contiguous()
    N, H, W = labels.shape
    lib, dev = L.get(), labels.device
    table = None
    if lut is not None:
        lut = np.asarray(lut)
        if lut.shape != (256,) or lut.min() < 0 or lut.max() > 255:
            raise L.LedB200Error('png_encode: lut must hold 256 values in 0 .. 255')
        table = (C.c_uint8 * 256)(*lut.astype(np.uint8).tolist())
    bound = L.check(lib.ledb200_png_lut_bound(H, W, int(bool(palette))), 'ledb200_png_lut_bound')
    ws = torch.empty(L.check(lib.ledb200_png_workspace_bytes(N, H, W), 'ledb200_png_workspace_bytes'),
                     dtype=torch.uint8, device=dev)
    out = torch.empty(N * bound, dtype=torch.uint8, device=dev)
    offsets = torch.empty(N + 1, dtype=torch.int64, device=dev)
    if table is None and not palette:
        L.check(lib.ledb200_png_encode(_p(labels), L.torch_dtype_code(labels), N, H, W, int(add), _p(out), _p(offsets),
                                       _p(ws), L.stream_ptr(dev)), 'ledb200_png_encode')
    else:
        if table is None:
            if add not in (0, 1):
                raise L.LedB200Error('png_encode: add must be 0 or 1')
            table = (C.c_uint8 * 256)(*[(i + int(add)) & 255 for i in range(256)])
        L.check(lib.ledb200_png_encode_lut(_p(labels), L.torch_dtype_code(labels), N, H, W, table, int(bool(palette)),
                                           _p(out), _p(offsets), _p(ws), L.stream_ptr(dev)), 'ledb200_png_encode_lut')
    return _fetch_files(out, offsets)


def _fetch_files(out, offsets):
    offs = offsets.cpu().tolist()
    data = out[:offs[-1]].cpu().numpy().tobytes()
    return [data[offs[i]:offs[i + 1]] for i in range(len(offs) - 1)]


def _png_encode_rgb(rgb, add, lut, palette):
    if add or lut is not None or palette:
        raise L.LedB200Error('png_encode: add, lut and palette apply to label maps, not to RGB images')
    if rgb.dtype != torch.uint8 or rgb.shape[-1] != 3:
        raise L.LedB200Error('png_encode: RGB images are [N, H, W, 3] uint8')
    rgb = rgb.contiguous()
    N, H, W, _ = rgb.shape
    lib, dev = L.get(), rgb.device
    bound = L.check(lib.ledb200_png_rgb_bound(H, W), 'ledb200_png_rgb_bound')
    ws = torch.empty(L.check(lib.ledb200_png_rgb_workspace_bytes(N, H, W), 'ledb200_png_rgb_workspace_bytes'),
                     dtype=torch.uint8, device=dev)
    out = torch.empty(N * bound, dtype=torch.uint8, device=dev)
    offsets = torch.empty(N + 1, dtype=torch.int64, device=dev)
    L.check(lib.ledb200_png_encode_rgb(_p(rgb), N, H, W, _p(out), _p(offsets), _p(ws), L.stream_ptr(dev)),
            'ledb200_png_encode_rgb')
    return _fetch_files(out, offsets)


def blend_table(alpha):
    """The 256 x 256 uint8 table of mmseg's blend `(image * (1 - alpha) + mask * alpha).astype(np.uint8)`: entry
    [i, c] for image value i and mask value c, computed with numpy's own float64 expression (a float32 or fused
    multiply-add restatement truncates differently for some pairs)."""
    v = np.arange(256, dtype=np.uint8)
    return (v[:, None] * (1 - alpha) + v[None, :] * alpha).astype(np.uint8)


def _label_map(t, who):
    _need_cuda(t)
    if t.dim() == 2:
        t = t[None]
    if t.dim() != 3 or t.dtype not in (torch.uint8, torch.int64):
        raise L.LedB200Error(f'{who}: label maps are [N, H, W] (or [H, W]) uint8 or int64')
    return t.contiguous()


def seg_label_locations(labels, num_classes):
    """mmseg's SegLocalVisualizer._get_center_loc for every class of N label maps in one launch sequence.

    labels [N,H,W] (or [H,W]) CUDA uint8 / int64, 1 <= num_classes <= 255.  Returns int32 [N, K, 3] on the device:
    (present, x, y) per class k < K, where y is the first row holding the most pixels of k and x the pixel at index
    count // 2 of that row in x order; (0, 0, 0) when k is absent.  Labels outside 0 .. K - 1 are not counted."""
    labels = _label_map(labels, 'seg_label_locations')
    N, H, W = labels.shape
    K = int(num_classes)
    lib, dev = L.get(), labels.device
    ws = torch.empty(L.check(lib.ledb200_seg_locate_workspace_bytes(N, H, K), 'ledb200_seg_locate_workspace_bytes'),
                     dtype=torch.uint8, device=dev)
    out = torch.empty((N, K, 3), dtype=torch.int32, device=dev)
    L.check(lib.ledb200_seg_label_locations(_p(labels), L.torch_dtype_code(labels), N, H, W, K, _p(out), _p(ws),
                                            L.stream_ptr(dev)), 'ledb200_seg_label_locations')
    return out


STAMP_DTYPE = np.dtype([('image', '<i4'), ('panel', '<i4'), ('x0', '<i4'), ('y0', '<i4'), ('w', '<i4'), ('h', '<i4'),
                        ('offset', '<i8')])        # ledb200_seg_stamp


def seg_overlay(images, gt, pred, palette, table, stamps=None, stamp_data=None):
    """mmseg's _draw_sem_seg blend for N same-shape images, with the gt | pred panels side by side, in one call.

    images [N,3,H,W] CUDA uint8 BGR (what the decoders give); gt / pred [N,H,W] label maps (uint8 / int64), either may
    be None.  palette: CUDA uint8 [K, 3] RGB (K <= 255); table: CUDA uint8 [256, 256] (blend_table(alpha)).  stamps:
    an optional CUDA tensor holding a STAMP_DTYPE array as bytes (drawn in order: the last one touching a pixel wins),
    stamp_data its CUDA uint8 pixels, 4 bytes (R, G, B, touched) each.  Returns CUDA uint8 [N, H, P*W, 3] RGB."""
    _need_cuda(images, palette, table, stamps, stamp_data)
    if gt is None and pred is None:
        raise L.LedB200Error('seg_overlay: neither a gt nor a pred label map')
    if images.dim() != 4 or images.shape[1] != 3 or images.dtype != torch.uint8:
        raise L.LedB200Error('seg_overlay: images are [N, 3, H, W] uint8')
    images = images.contiguous()
    N, _, H, W = images.shape
    maps = [None if m is None else _label_map(m, 'seg_overlay') for m in (gt, pred)]
    for m in maps:
        if m is not None and tuple(m.shape) != (N, H, W):
            raise L.LedB200Error(f'seg_overlay: a label map of {tuple(m.shape)} for images of {(N, H, W)}')
    palette = palette.contiguous()
    if palette.dtype != torch.uint8 or palette.dim() != 2 or palette.shape[1] != 3:
        raise L.LedB200Error('seg_overlay: palette is [K, 3] uint8')
    if table.dtype != torch.uint8 or table.numel() != 65536:
        raise L.LedB200Error('seg_overlay: table is [256, 256] uint8')
    P = sum(m is not None for m in maps)
    out = torch.empty((N, H, P * W, 3), dtype=torch.uint8, device=images.device)
    ns = 0 if stamps is None else stamps.numel() // STAMP_DTYPE.itemsize
    codes = [L.torch_dtype_code(m) if m is not None else L.U8 for m in maps]
    L.check(L.get().ledb200_seg_overlay(_p(images), _p(maps[0]), codes[0], _p(maps[1]), codes[1], N, H, W,
                                        palette.shape[0], _p(palette), _p(table.contiguous()), _p(stamps), ns,
                                        _p(stamp_data), 0 if stamp_data is None else stamp_data.numel(), _p(out),
                                        L.stream_ptr(images.device)), 'ledb200_seg_overlay')
    return out


CITYSCAPES_RECORDS_PER_COPY = 256   # records per image fetched with the statuses; a batch with more costs a second copy


def cityscapes_accumulate(pred, gt, inst, train_to_id, category, inst_rule, cm=None, cm_last=None):
    """cityscapesscripts' evaluatePair statistics for N same-shape images in one call (csrc/cityscapes.cu).

    pred [N,H,W] (or [H,W]) uint8 / int64 trainIds, gt uint8 labelIds, inst int32 instanceIds, all CUDA.  Tables:
    train_to_id (256 labelIds), category (34 instance categories, -1 none), inst_rule (34: 0 error, 1 skip, 2 count).
    cm: int64 [34, 34] CUDA matrix accumulated (allocated when None); cm_last: when given, receives the matrix of the
    batch's last image alone.  Returns (cm, statuses, records): statuses an int32 numpy [N] of LEDB200 bit flags
    (lib.CITYSCAPES_STATUS), records one int64 numpy [k, 4] per image of (instId, size, tp, catTp) in ascending instId.
    One small copy brings statuses, counts and records back (a second one when a batch holds more than
    CITYSCAPES_RECORDS_PER_COPY instances per image)."""
    _need_cuda(pred, gt, inst, cm, cm_last)
    if pred.dim() == 2:
        pred, gt, inst = pred[None], gt[None], inst[None]
    if pred.dtype not in (torch.uint8, torch.int64) or gt.dtype != torch.uint8 or inst.dtype != torch.int32:
        raise L.LedB200Error('cityscapes_accumulate: predictions uint8 / int64, labelIds uint8, instanceIds int32')
    if pred.dim() != 3 or pred.shape != gt.shape or pred.shape != inst.shape:
        raise L.LedB200Error(f'cityscapes_accumulate: shapes differ ({tuple(pred.shape)}, {tuple(gt.shape)}, '
                             f'{tuple(inst.shape)})')
    pred, gt, inst = pred.contiguous(), gt.contiguous(), inst.contiguous()
    N, H, W = pred.shape
    dev, lib = pred.device, L.get()
    if cm is None:
        cm = torch.zeros((34, 34), dtype=torch.int64, device=dev)
    assert cm.dtype == torch.int64 and cm.is_contiguous() and cm.numel() == 34 * 34
    if cm_last is not None:
        assert cm_last.dtype == torch.int64 and cm_last.is_contiguous() and cm_last.numel() == 34 * 34
    out = torch.empty(L.check(lib.ledb200_cityscapes_out_ints(N), 'ledb200_cityscapes_out_ints'), dtype=torch.int32,
                      device=dev)
    ws = torch.empty(L.check(lib.ledb200_cityscapes_workspace_bytes(N), 'ledb200_cityscapes_workspace_bytes'),
                     dtype=torch.uint8, device=dev)
    t2i = (C.c_int32 * 256)(*[int(v) for v in train_to_id])
    cat = (C.c_int8 * 34)(*[int(v) for v in category])
    rule = (C.c_int8 * 34)(*[int(v) for v in inst_rule])
    L.check(lib.ledb200_cityscapes_accumulate(_p(pred), L.torch_dtype_code(pred), _p(gt), _p(inst), N, H, W, t2i, cat,
                                              rule, _p(cm), _p(cm_last), _p(out), _p(ws), L.stream_ptr(dev)),
            'ledb200_cityscapes_accumulate')
    cap = N * CITYSCAPES_RECORDS_PER_COPY
    head = out[:2 * N + 4 * cap].cpu().numpy()
    statuses, counts = head[:N].copy(), head[N:2 * N].astype(np.int64)
    total = int(counts.sum())
    rec = head[2 * N:2 * N + 4 * min(total, cap)]
    if total > cap:
        rec = np.concatenate([rec, out[2 * N + 4 * cap:2 * N + 4 * total].cpu().numpy()])
    rec = rec.astype(np.int64).reshape(-1, 4)
    ends = np.cumsum(counts)
    return cm, statuses, [rec[e - c:e] for c, e in zip(counts, ends)]


PNG_SIGNATURE = b'\x89PNG\r\n\x1a\n'
MAX_PNG_PIXELS = 1 << 30      # OpenCV's default CV_IO_MAX_IMAGE_PIXELS


def _head(f, n):
    """the first n bytes of a file given as bytes-like or a 1-D uint8 tensor (a device tensor costs one small copy)"""
    if isinstance(f, torch.Tensor):
        if f.dtype != torch.uint8 or f.dim() != 1:
            raise L.LedB200Error('files are bytes or 1-D uint8 tensors')
        return f[:n].cpu().numpy().tobytes()
    return bytes(memoryview(f)[:n])


def png_info(f, kind='color'):
    """(h, w, colour type) from the IHDR of a PNG file (bytes-like or 1-D uint8 tensor), which sits at a fixed offset
    after the signature.  Checks the signature, the IHDR's length, name and CRC, and the sizes; a malformed header raises
    LedB200Error, a valid PNG outside what png_decode supports raises NotImplementedError: bit depths other than 8
    (kind 'color' and 'label') or 16 (kind 'grey16'), interlaced (Adam7) files, for kind='label' colour types 2 / 4 / 6
    and for kind='grey16' every colour type but 0."""
    b = _head(f, 33)
    if len(b) < 33 or b[:8] != PNG_SIGNATURE:
        raise L.LedB200Error('not a PNG file (no PNG signature)')
    if b[8:16] != b'\x00\x00\x00\x0dIHDR':
        raise L.LedB200Error('the first chunk is not a 13-byte IHDR')
    if zlib.crc32(b[12:29]) != struct.unpack('>I', b[29:33])[0]:
        raise L.LedB200Error('IHDR CRC-32 mismatch')
    w, h, depth, ct, comp, filt, interlace = struct.unpack('>IIBBBBB', b[16:29])
    if not (1 <= w < 1 << 31 and 1 <= h < 1 << 31):
        raise L.LedB200Error(f'IHDR: invalid size {w} x {h}')
    if ct not in (0, 2, 3, 4, 6) or depth not in (1, 2, 4, 8, 16) or comp or filt or interlace > 1:
        raise L.LedB200Error(f'IHDR: invalid header (bit depth {depth}, colour type {ct}, compression {comp}, '
                             f'filter {filt}, interlace {interlace})')
    if kind == 'grey16':
        if depth != 16 or ct != 0:
            raise NotImplementedError(f'{depth}-bit PNG files of colour type {ct} as grey16 (16-bit grey only)')
    elif depth != 8:
        raise NotImplementedError(f'{depth}-bit PNG files (png_decode reads bit depth 8, 16 for kind grey16)')
    if interlace:
        raise NotImplementedError('interlaced (Adam7) PNG files')
    if kind == 'label' and ct not in (0, 3):
        raise NotImplementedError(f'label maps of colour type {ct} (grey or palette only)')
    if h * w > MAX_PNG_PIXELS:
        raise L.LedB200Error(f'{w} x {h} is more than {MAX_PNG_PIXELS} pixels')
    return h, w, ct


def label_lut(reduce_zero_label=False, label_map=None):
    """The 256-entry uint8 table that maps a stored label value to what LoadAnnotations._load_seg_map gives.

    mmseg 1.2.2, mmseg/datasets/transforms/loading.py, LoadAnnotations._load_seg_map, restated here from the released
    source (the reference checkout is not part of this repository), applies, to the uint8 map:
      1. reduce_zero_label: 0 -> 255, then v - 1 (uint8), then 254 -> 255;
      2. label_map: for each (old, new), map[copy == old] = new, where `copy` is the map after step 1 (every
         replacement reads the values before any of them)."""
    v = np.arange(256, dtype=np.uint8)
    if reduce_zero_label:
        v[v == 0] = 255
        v = v - np.uint8(1)
        v[v == 254] = 255
    if label_map is not None:
        src = v.copy()
        for old, new in label_map.items():
            if not 0 <= int(new) <= 255:
                raise ValueError(f'label_map value {new} does not fit a uint8 label map')
            v[src == old] = new
    return v


def _decode_files(files, names, infos, ch, device, who, launch, status_names, dtype=torch.uint8):
    """The host side shared by png_decode and jpeg_decode: files (bytes-like or 1-D uint8 tensors, host or device) are
    staged, the host ones packed into one pinned buffer and uploaded with one copy; one [ch, h, w] output of `dtype` per
    file (infos[i] starts with h, w) is carved from one allocation; launch(arr_args) runs the decode call, given the
    device copies of the files, their sizes and the outputs, and returns the int32 status tensor, read back with one
    copy.  A file with a non-zero status raises LedB200Error naming it and status_names' reason."""
    n = len(files)
    if device is None:
        device = next((f.device for f in files if isinstance(f, torch.Tensor) and f.is_cuda), None)
    if device is None:
        if not torch.cuda.is_available():
            raise L.LedB200Error(f'{who} decodes on a CUDA device (no CPU fallback)')
        device = torch.device('cuda', torch.cuda.current_device())
    dev = torch.device(device)
    if dev.type != 'cuda':
        raise L.LedB200Error(f'{who} decodes on a CUDA device (no CPU fallback)')
    # host files: one pinned staging buffer, one host-to-device copy
    host = [i for i, f in enumerate(files) if not (isinstance(f, torch.Tensor) and f.is_cuda)]
    sizes = [f.numel() if isinstance(f, torch.Tensor) else memoryview(f).nbytes for f in files]
    data = [None] * n
    if host:
        offs = np.cumsum([0] + [sizes[i] for i in host])
        pinned = torch.empty(int(offs[-1]), dtype=torch.uint8, pin_memory=True)
        view = pinned.numpy()
        for k, i in enumerate(host):
            f = files[i]
            src = f.contiguous().numpy() if isinstance(f, torch.Tensor) else np.frombuffer(f, np.uint8)
            view[offs[k]:offs[k + 1]] = src
        up = pinned.to(dev, non_blocking=True)
        for k, i in enumerate(host):
            data[i] = up[offs[k]:offs[k + 1]]
    for i, f in enumerate(files):
        if data[i] is None:
            data[i] = f.to(dev).contiguous()
    numel = [ch * info[0] * info[1] for info in infos]
    flat = torch.empty(sum(numel), dtype=dtype, device=dev)
    outs, at = [], 0
    for info, m in zip(infos, numel):
        outs.append(flat[at:at + m].view(ch, info[0], info[1]))
        at += m
    st = launch(data, sizes, outs, dev).cpu().tolist()
    bad = [(names[i], status_names.get(c, f'status {c}')) for i, c in enumerate(st) if c]
    if bad:
        raise L.LedB200Error(f'{who}: ' + '; '.join(f'{nm}: {why}' for nm, why in bad))
    return outs


def _infos(files, names, parse):
    """parse(f) for every file, its errors prefixed with the file's name"""
    infos = []
    for f, name in zip(files, names):
        try:
            infos.append(parse(f))
        except NotImplementedError as e:
            raise NotImplementedError(f'{name}: {e}') from None
        except L.LedB200Error as e:
            raise L.LedB200Error(f'{name}: {e}') from None
    return infos


def png_decode(files, kind='color', reduce_zero_label=False, label_map=None, names=None, device=None):
    """PNG files -> CUDA uint8 tensors, decoded on the device (csrc/png_decode.cu).

    files: bytes-like objects or 1-D uint8 tensors (host or device), bit depth 8, not interlaced.
    kind='color': each result is [3, h, w] BGR, bit-identical to cv2.imdecode(buf, cv2.IMREAD_COLOR).transpose(2, 0, 1)
      (what LoadImageFromFile gives): grey replicated, palettes expanded, alpha dropped, ancillary chunks ignored.
    kind='label': grey or palette files; each result is [1, h, w], the stored values (palette indices, not colours: what
      np.array(Image.open(f)) gives) through label_lut(reduce_zero_label, label_map), as LoadAnnotations gives them.
    kind='grey16': 16-bit grey files only (Cityscapes' *_instanceIds.png); each result is [1, h, w] int32, the values
      np.array(Image.open(f)) gives.
    The host reads each IHDR (png_info), packs the host files into one pinned buffer and uploads it with one copy; one
    decode call covers every file and one small copy brings the statuses back.  A file that fails raises LedB200Error
    naming it (names[i], default 'file i') and the reason."""
    if kind not in ('color', 'label', 'grey16'):
        raise ValueError(f"kind must be 'color', 'label' or 'grey16', not {kind!r}")
    files = list(files)
    n = len(files)
    if n == 0:
        return []
    names = list(names) if names is not None else [f'file {i}' for i in range(n)]
    infos = _infos(files, names, lambda f: png_info(f, kind))

    def launch(data, sizes, outs, dev):
        arr = (L.PngFile * n)()
        for d, t, o, (h, w, ct), sz in zip(arr, data, outs, infos, sizes):
            d.data, d.size, d.out, d.h, d.w, d.color_type = t.data_ptr(), sz, o.data_ptr(), h, w, ct
        lib = L.get()
        mode = {'color': L.PNG_COLOR, 'label': L.PNG_LABEL, 'grey16': L.PNG_GREY16}[kind]
        ws = torch.empty(max(1, L.check(lib.ledb200_png_decode_mode_workspace_bytes(arr, n, mode),
                                        'ledb200_png_decode_mode_workspace_bytes')), dtype=torch.uint8, device=dev)
        status = torch.empty(n, dtype=torch.int32, device=dev)
        lut = None
        if kind == 'label':
            lut = (C.c_uint8 * 256)(*label_lut(reduce_zero_label, label_map).tolist())
        L.check(lib.ledb200_png_decode(arr, n, mode, lut, _p(ws), _p(status), L.stream_ptr(dev)), 'ledb200_png_decode')
        return status

    return _decode_files(files, names, infos, 3 if kind == 'color' else 1, device, 'png_decode', launch, L.PNG_STATUS,
                         torch.int32 if kind == 'grey16' else torch.uint8)


JPEG_SOI = b'\xff\xd8'
_JPEG_SOF_REFUSED = {0xC2: 'progressive', 0xC3: 'lossless', 0xC5: 'hierarchical', 0xC6: 'hierarchical progressive',
                     0xC7: 'hierarchical lossless', 0xC9: 'arithmetic-coded', 0xCA: 'arithmetic-coded progressive',
                     0xCB: 'arithmetic-coded lossless', 0xCD: 'hierarchical arithmetic-coded',
                     0xCE: 'hierarchical arithmetic-coded progressive', 0xCF: 'hierarchical arithmetic-coded lossless'}


def _exif_orientation(d):
    """the orientation tag of an APP1 Exif payload (IFD0), 0 when there is none"""
    if len(d) < 14 or d[:6] != b'Exif\x00\x00':
        return 0
    t = d[6:]
    if t[:2] not in (b'II', b'MM'):
        return 0
    e = '<' if t[:2] == b'II' else '>'
    if struct.unpack(e + 'H', t[2:4])[0] != 42:
        return 0
    ifd = struct.unpack(e + 'I', t[4:8])[0]
    if ifd > len(t) - 2:
        return 0
    for i in range(struct.unpack(e + 'H', t[ifd:ifd + 2])[0]):
        at = ifd + 2 + 12 * i
        if at + 12 > len(t):
            break
        if struct.unpack(e + 'H', t[at:at + 2])[0] == 0x0112:
            return struct.unpack(e + 'H', t[at + 8:at + 10])[0]
    return 0


def _jpeg_markers(b):
    """(h, w, components) from a JPEG header prefix b; None when b ends before the first SOS"""
    if len(b) < 2 or b[:2] != JPEG_SOI:
        raise L.LedB200Error('not a JPEG file (no SOI marker)')
    p, frame, jfif, adobe, transform, orient = 2, None, False, False, 0, 0
    while True:
        if p >= len(b):
            return None
        if b[p] != 0xFF:
            raise L.LedB200Error(f'no marker at byte {p}')
        while p < len(b) and b[p] == 0xFF:
            p += 1
        if p + 3 > len(b):
            return None
        m, n = b[p], (b[p + 1] << 8 | b[p + 2]) - 2
        p += 3
        if n < 0:
            raise L.LedB200Error(f'marker 0x{m:02X}: segment length {n + 2}')
        if p + n > len(b):
            return None
        s = b[p:p + n]
        p += n
        if m in _JPEG_SOF_REFUSED or m == 0xCC:
            raise NotImplementedError(f'{_JPEG_SOF_REFUSED.get(m, "arithmetic-coded")} JPEG files (baseline only)')
        if m in (0xC0, 0xC1):
            if frame is not None:
                raise L.LedB200Error('a second frame header')
            if n < 6 or n != 6 + 3 * s[5]:
                raise L.LedB200Error('frame header length')
            prec, h, w, nf = s[0], s[1] << 8 | s[2], s[3] << 8 | s[4], s[5]
            if prec != 8:
                raise NotImplementedError(f'{prec}-bit JPEG files (8-bit only)')
            if h == 0:
                raise NotImplementedError('JPEG files whose height is given by a DNL marker')
            if w == 0:
                raise L.LedB200Error('frame width 0')
            if nf not in (1, 3):
                raise NotImplementedError(f'JPEG files of {nf} components (grey or YCbCr only)')
            comps = [(s[6 + 3 * c], s[7 + 3 * c] >> 4, s[7 + 3 * c] & 15) for c in range(nf)]
            if any(not (1 <= hs <= 4 and 1 <= vs <= 4) for _, hs, vs in comps):
                raise L.LedB200Error('invalid sampling factors')
            if nf == 3 and not (comps[0][1] <= 2 and comps[0][2] <= 2 and all(c[1:] == (1, 1) for c in comps[1:])):
                raise NotImplementedError('sampling factors ' + ', '.join(f'{hs}x{vs}' for _, hs, vs in comps) +
                                          ' (4:4:4, 4:2:2, 4:2:0 and 4:4:0 only)')
            frame = (h, w, nf, [c[0] for c in comps])
        elif m == 0xDA:
            if frame is None:
                raise L.LedB200Error('SOS before the frame header')
            h, w, nf, ids = frame
            if n < 1 or s[0] != nf:
                raise NotImplementedError('non-interleaved (multi-scan) JPEG files')
            if [s[1 + 2 * c] for c in range(nf)] != ids:
                raise NotImplementedError('a scan whose components are not in frame order')
            if nf == 3 and (False if jfif else transform == 0 if adobe else ids == [82, 71, 66]):
                raise NotImplementedError('RGB JPEG files (YCbCr or grey only)')
            if 2 <= orient <= 8:
                raise NotImplementedError(f'Exif orientation {orient} (cv2.imdecode would rotate the image)')
            if h * w > MAX_PNG_PIXELS:
                raise L.LedB200Error(f'{w} x {h} is more than {MAX_PNG_PIXELS} pixels')
            return h, w, nf
        elif m == 0xE0:
            jfif |= n >= 14 and s[:5] == b'JFIF\x00'
        elif m == 0xE1:
            orient = orient or _exif_orientation(s)
        elif m == 0xEE and n >= 12 and s[:5] == b'Adobe':
            adobe, transform = True, s[11]
        elif m == 0xDC:
            raise NotImplementedError('JPEG files whose height is given by a DNL marker')
        elif not (m in (0xC4, 0xDB, 0xDD, 0xFE) or 0xE0 <= m <= 0xEF):
            raise L.LedB200Error(f'unexpected marker 0x{m:02X} before the scan')


def jpeg_info(f):
    """(h, w, components) of a JPEG file (bytes-like or 1-D uint8 tensor), from its markers up to the first SOS (a device
    tensor costs small copies of the header prefix).  A malformed header raises LedB200Error; a valid JPEG outside what
    jpeg_decode supports raises NotImplementedError: progressive, lossless, hierarchical or arithmetic-coded files,
    precision other than 8 bits, 2 or 4 components, RGB colour space, sampling other than 4:4:4 / 4:2:2 / 4:2:0 /
    4:4:0, non-interleaved scans, a DNL height and an Exif orientation other than 1."""
    size = f.numel() if isinstance(f, torch.Tensor) else memoryview(f).nbytes
    n = 1 << 16
    while True:
        info = _jpeg_markers(_head(f, n))
        if info is not None:
            return info
        if n >= size:
            raise L.LedB200Error('the file ends before the first SOS')
        n *= 4


def jpeg_decode(files, names=None, device=None):
    """Baseline JPEG files -> CUDA [3, h, w] uint8 BGR tensors decoded on the device (csrc/jpeg_decode.cu),
    bit-identical to cv2.imdecode(buf, cv2.IMREAD_COLOR).transpose(2, 0, 1) (what LoadImageFromFile gives).

    files: bytes-like objects or 1-D uint8 tensors (host or device).  The host walks each file's markers (jpeg_info),
    packs the host files into one pinned buffer and uploads it with one copy; one decode call covers every file and
    one small copy brings the statuses back.  A file that fails raises LedB200Error naming it (names[i], default
    'file i') and the reason: corrupt entropy-coded data is an error, where libjpeg would warn and fill with grey."""
    files = list(files)
    n = len(files)
    if n == 0:
        return []
    names = list(names) if names is not None else [f'file {i}' for i in range(n)]
    infos = _infos(files, names, jpeg_info)

    def launch(data, sizes, outs, dev):
        arr = (L.JpegFile * n)()
        for d, t, o, (h, w, nc), sz in zip(arr, data, outs, infos, sizes):
            d.data, d.size, d.out, d.h, d.w, d.components = t.data_ptr(), sz, o.data_ptr(), h, w, nc
        lib = L.get()
        ws = torch.empty(L.check(lib.ledb200_jpeg_decode_workspace_bytes(arr, n), 'ledb200_jpeg_decode_workspace_bytes'),
                         dtype=torch.uint8, device=dev)
        status = torch.empty(n, dtype=torch.int32, device=dev)
        L.check(lib.ledb200_jpeg_decode(arr, n, _p(ws), _p(status), L.stream_ptr(dev)), 'ledb200_jpeg_decode')
        return status

    return _decode_files(files, names, infos, 3, device, 'jpeg_decode', launch, L.JPEG_STATUS)
