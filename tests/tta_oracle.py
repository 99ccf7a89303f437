"""CPU restatement of the reference's test-time-augmentation tail (TEST INFRASTRUCTURE): BaseSegmentor.postprocess_result
(mmseg/models/segmentors/base.py:153-198) per view, then SegTTAModel.merge_preds (mmseg/models/segmentors/seg_tta.py),
in plain PyTorch built on the oracle's `resize`.  The tests of SegTTAModel / ops.tta_merge compare against it."""
import torch

from oracle import resize


def postprocess_view(lg, padding=None, flip=None, ori_shape=None, align_corners=False):
    """base.py:153-198 for ONE image's [K,H,W] logits: crop padding (l, r, t, b), undo the flip, resize to ori_shape,
    sigmoid when K == 1; returns the seg_logits postprocess_result stores."""
    K, H, W = lg.shape
    l, r, t, b = padding if padding is not None else (0, 0, 0, 0)
    x = lg[None, :, t:H - b, l:W - r]
    if flip == 'horizontal':
        x = x.flip(dims=(3,))
    elif flip == 'vertical':
        x = x.flip(dims=(2,))
    if ori_shape is not None:
        x = resize(x, ori_shape, align_corners)
    x = x.squeeze(0)
    return x.sigmoid() if K == 1 else x


def merge_preds(view_logits, out_channels, threshold=0.3):
    """seg_tta.py SegTTAModel.merge_preds for ONE image: view_logits = the views' post-processed [K,H,W] seg_logits.
    Returns (merged logits [K,H,W], seg_pred)."""
    logits = torch.zeros(view_logits[0].shape).to(view_logits[0])
    for seg_logit in view_logits:
        if out_channels > 1:
            logits += seg_logit.softmax(dim=0)
        else:
            logits += seg_logit.sigmoid()
    logits /= len(view_logits)
    if out_channels == 1:
        seg_pred = (logits > threshold).to(logits).squeeze(1)
    else:
        seg_pred = logits.argmax(dim=0)
    return logits, seg_pred


def tta_merge(view_logits, metas, out_channels, threshold=0.3, align_corners=False):
    """The reference's TTA tail on CPU: view_logits = per view [N,K,H,W] (module.inference output), metas = per view
    the N images' metainfo (img_padding_size / padding_size, flip, flip_direction, ori_shape).  Each view goes through
    postprocess_result, then merge_preds per image.  Returns (merged [N,K,oh,ow], seg_pred stacked over images)."""
    merged, preds = [], []
    for i in range(view_logits[0].shape[0]):
        views = []
        for lg, mv in zip(view_logits, metas):
            m = mv[i].get('metainfo', mv[i])
            padding = m.get('img_padding_size', m.get('padding_size', None))
            flip = m.get('flip_direction') if m.get('flip', None) else None
            views.append(postprocess_view(lg[i], padding, flip, m.get('ori_shape'), align_corners))
        lg, pred = merge_preds(views, out_channels, threshold)
        merged.append(lg)
        preds.append(pred)
    return torch.stack(merged, 0), torch.stack(preds, 0)

