"""SegTTAModel and ops.tta_merge (csrc/postprocess.cu tta_merge_kernel) against the reference's TTA tail restated on
the CPU (tests/tta_oracle.py: postprocess_result per view, then SegTTAModel.merge_preds)."""
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle
import lednet_b200 as L
from lednet_b200 import ops, synth
from lednet_b200.tta import SegTTAModel
from util import build_pair
import trained
import tta_oracle

pytestmark = pytest.mark.gpu
DEV = 'cuda'


def _check_labels(pred, ref_pred, merged, tol):
    """labels identical except pixels whose top-2 merged probabilities lie within `tol`"""
    top2 = merged.topk(2, dim=1).values
    tie = (top2[:, 0] - top2[:, 1]) <= tol
    mism = pred.cpu().long() != ref_pred.long()
    assert not (mism & ~tie).any(), int((mism & ~tie).sum())


# ------------------------------------------------------------------ 1. kernel against the CPU restatement
# (K, [(view hw, padding, flip)], ori_shape, align_corners)
CASES = [
    (19, [((24, 40), None, None)] * 3, (24, 40), False),                                    # identity
    (19, [((40, 56), (0, 3, 0, 5), 'horizontal'), ((40, 56), (0, 3, 0, 5), None)], (64, 96), False),  # pad + flip + up
    (5, [((37, 29), (2, 1, 3, 0), 'vertical'), ((37, 29), None, None)], (20, 17), True),   # v-flip + down, align_corners
    (2, [((64, 114), None, None), ((64, 114), None, 'horizontal')], (90, 160), False),     # Apple ratio 1.40625
    (19, [((16, 24), None, None), ((24, 36), None, 'horizontal'), ((32, 48), None, None),
          ((40, 64), (0, 4, 0, 0), 'vertical')], (32, 48), False),                          # several view sizes
    (2, [((12, 20), None, None), ((18, 30), None, 'horizontal'), ((24, 40), (0, 0, 0, 0), 'horizontal')], (24, 40), True),
    (40, [((20, 30), None, None), ((30, 45), (1, 0, 0, 2), 'horizontal'), ((40, 60), None, 'vertical')], (40, 60), False),
    (12, [((20, 30), None, None)] * 2 + [((26, 38), (0, 2, 1, 1), 'horizontal')], (21, 31), False),
]


def _case_logits(K, views, n, seed):
    """per view [n,K,H,W]; views of one shape are slices of one batch (the engine's layout for a flip pair)"""
    g = torch.Generator().manual_seed(seed)
    out, batches = [None] * len(views), {}
    for v, (hw, _, _) in enumerate(views):
        batches.setdefault(hw, []).append(v)
    for hw, idx in batches.items():
        big = torch.randn(len(idx) * n, K, *hw, generator=g) * 3
        for j, v in enumerate(idx):
            out[v] = big[j * n:(j + 1) * n]
    return out


@pytest.mark.parametrize('mode', [0, 1])
@pytest.mark.parametrize('case', range(len(CASES)))
def test_tta_merge_kernel_matches_restatement(case, mode):
    K, views, ori, ac = CASES[case]
    n = 2
    logits = _case_logits(K, views, n, seed=case * 10 + mode)
    metas = [[dict(img_padding_size=p or (0, 0, 0, 0), flip=f is not None, flip_direction=f, ori_shape=ori)] * n
             for (_, p, f) in views]
    ref_merged, ref_pred = tta_oracle.tta_merge(logits, metas, K if mode == 0 else 1, 0.3, ac)
    dev_logits = [lg.to(DEV) for lg in logits]
    if len({v[0] for v in views}) == 1:                 # same-shape views: slices of one device batch, no copy
        big = torch.cat(logits, 0).to(DEV)
        dev_logits = [big[v * n:(v + 1) * n] for v in range(len(views))]
    vd = [(lg, p, f) for lg, (_, p, f) in zip(dev_logits, views)]
    pred, probs = ops.tta_merge(vd, ori, ac, mode, 0.3, torch.int64, want_probs=True)
    assert probs.shape == ref_merged.shape
    assert (probs.cpu() - ref_merged).abs().max().item() <= 1e-5
    if mode == 0:
        assert pred.dtype == torch.int64 and tuple(pred.shape) == (n,) + ori
        _check_labels(pred, ref_pred, ref_merged, 1e-5)
        assert torch.equal(probs.argmax(dim=1), pred)                     # self-consistent
        pred_u8, _ = ops.tta_merge(vd, ori, ac, mode, 0.3, torch.uint8)
        assert torch.equal(pred_u8.long(), pred)
    else:
        assert pred.dtype == torch.float32 and pred.shape == ref_pred.shape
        near = (ref_merged - 0.3).abs() < 1e-6
        assert torch.equal(pred.cpu()[~near], ref_pred[~near])
        assert torch.equal(pred, (probs > 0.3).float())


# ------------------------------------------------------------------ 2. agreement with ops.postprocess
@pytest.mark.parametrize('K', [2, 19, 40])
def test_tta_merge_equals_postprocess_softmax_mean(K):
    _, views, ori, ac = CASES[4]
    logits = _case_logits(K, views, 1, seed=K)
    acc = None
    for lg, (_, p, f) in zip(logits, views):
        _, out = ops.postprocess(lg[0].to(DEV), padding=p, flip=f, ori_shape=ori, align_corners=ac)
        sm = torch.softmax(out, dim=0)
        acc = sm if acc is None else acc + sm
    acc = acc / len(views)
    pred, probs = ops.tta_merge([(lg.to(DEV), p, f) for lg, (_, p, f) in zip(logits, views)], ori, ac,
                                want_probs=True)
    assert (probs[0] - acc).abs().max().item() <= 1e-6
    _check_labels(pred[0:1].cpu(), acc.argmax(dim=0)[None].cpu(), acc[None].cpu(), 1e-6)


# ------------------------------------------------------------------ SegTTAModel end to end
def _resize_u8(img, hw):
    """view images of the TTA pipeline (test plumbing: torch bilinear on the device, not cv2's Resize)"""
    if tuple(img.shape[-2:]) == tuple(hw):
        return img.clone()
    return F.interpolate(img.float(), size=hw, mode='bilinear', align_corners=False).round().clamp(0, 255).to(torch.uint8)


def _tta_data(img, ratios, flip=True, img_path='img'):
    """mmseg TestTimeAug output after pseudo_collate: per view a list of images and of data samples"""
    n, _, h, w = img.shape
    inputs, samples = [], []
    for r in ratios:
        base = _resize_u8(img, (int(h * r + 0.5), int(w * r + 0.5)))
        for fl in ([False, True] if flip else [False]):
            x = base.flip(dims=(3,)) if fl else base
            inputs.append([x[i] for i in range(n)])
            samples.append([dict(metainfo=dict(ori_shape=(h, w), img_shape=tuple(x.shape[-2:]), flip=fl,
                                               flip_direction='horizontal' if fl else None, scale_factor=r,
                                               img_path=f'{img_path}{i}_{r}_{fl}.png'))
                            for i in range(n)])
    return dict(inputs=inputs, data_samples=samples)


def _oracle_views(o, data, pp_test_cfg=None):
    """the reference's per-view path on CPU: preprocess (+ stack_batch padding) -> inference; returns the logits and the
    metainfo postprocess_result reads"""
    logits, metas = [], []
    for inputs, samples in zip(data['inputs'], data['data_samples']):
        x = oracle.preprocess(torch.stack(inputs).cpu())
        ms = [dict(s['metainfo']) for s in samples]
        if pp_test_cfg:
            d = pp_test_cfg['size_divisor']
            hp, wp = -(-x.shape[-2] // d) * d, -(-x.shape[-1] // d) * d
            pad = (0, wp - x.shape[-1], 0, hp - x.shape[-2])
            x = F.pad(x, pad, value=0)
            for m in ms:
                m['img_padding_size'] = pad
        with torch.no_grad():
            logits.append(o.inference(x))
        metas.append(ms)
    return logits, metas


def _tta_pair(K, dtype='fp32'):
    o, m = build_pair(K, dtype=dtype)
    return o, m.to(DEV), SegTTAModel(m)


def test_tta_end_to_end_fp32():
    K = 19
    o, m, tta = _tta_pair(K)
    m.data_preprocessor.test_cfg = dict(size_divisor=32)        # pads the 0.5 and 1.5 views (32x48, 96x144)
    img = synth.make_images_u8(2, 64, 96, seed=21)
    data = _tta_data(img, (0.5, 1.0, 1.5))
    for s in data['data_samples'][0]:
        s['gt_sem_seg'] = dict(data=torch.zeros(1, 64, 96, dtype=torch.int64))
    ref_logits, ref_metas = _oracle_views(o, data, dict(size_divisor=32))
    assert any(any(mm['img_padding_size']) for mm in ref_metas[0])
    ref_merged, ref_pred = tta_oracle.tta_merge(ref_logits, ref_metas, K, 0.3, False)
    res = tta.test_step(data)
    assert len(res) == 2
    pred = torch.stack([r['pred_sem_seg']['data'] for r in res])
    assert pred.dtype == torch.int64 and tuple(pred.shape) == (2, 64, 96)
    # merged probabilities through the same views the model ran
    views = [m.data_preprocessor(dict(inputs=i, data_samples=[dict(s) for s in ss]), False)
             for i, ss in zip(data['inputs'], data['data_samples'])]
    lg = tta._view_logits([v['inputs'] for v in views])
    _, probs = ops.tta_merge([(lg[v], ref_metas[v][0]['img_padding_size'], 'horizontal' if ref_metas[v][0]['flip'] else None)
                              for v in range(len(lg))], (64, 96), want_pred=False, want_probs=True)
    assert (probs.cpu() - ref_merged).abs().max().item() <= 1e-4
    _check_labels(pred, ref_pred, ref_merged, 1e-4)
    for i, r in enumerate(res):                                 # reference-shaped: the last view's sample
        last = data['data_samples'][-1][i]
        assert set(r) >= {'seg_logits', 'pred_sem_seg', 'metainfo', 'gt_sem_seg'}
        assert r['metainfo']['scale_factor'] == 1.5 and r['metainfo']['flip'] is True
        assert r['metainfo']['img_path'] == data['data_samples'][0][i]['metainfo']['img_path']
        assert last['metainfo']['img_path'] != r['metainfo']['img_path']         # the input samples are not mutated
        assert r['gt_sem_seg'] is data['data_samples'][0][i]['gt_sem_seg']
        assert tuple(r['seg_logits']['data'].shape) == (K, 64, 96)
    list_res = tta.test_step([data['inputs'], data['data_samples']])              # list-shaped data
    assert torch.equal(torch.stack([r['pred_sem_seg']['data'] for r in list_res]), pred)


def test_merge_preds_equals_test_step():
    K = 19
    _, m, tta = _tta_pair(K)
    img = synth.make_images_u8(2, 64, 96, seed=22)
    data = _tta_data(img, (0.75, 1.0))
    res = tta.test_step(data)
    per_view = []
    for inputs, samples in zip(data['inputs'], data['data_samples']):
        per_view.append(m.test_step(dict(inputs=inputs, data_samples=[dict(s) for s in samples])))
    merged = tta.merge_preds([[pv[i] for pv in per_view] for i in range(2)])
    for i, (a, b) in enumerate(zip(res, merged)):
        _, probs = ops.tta_merge([(pv[i]['seg_logits']['data'][None], None, None) for pv in per_view], (64, 96),
                                 want_pred=False, want_probs=True)
        _check_labels(a['pred_sem_seg']['data'][None], b['pred_sem_seg']['data'][None].cpu(), probs.cpu(), 1e-6)
    # one unflipped ratio-1 view == module.predict, except near-ties
    one = _tta_data(img, (1.0,), flip=False)
    r1 = tta.test_step(one)
    x = m.data_preprocessor(dict(inputs=one['inputs'][0]), False)['inputs']
    logits = m.inference(x)
    pr = m.predict(x)
    sm = torch.softmax(logits, dim=1).cpu()
    for i in range(2):
        _check_labels(r1[i]['pred_sem_seg']['data'][None], pr[i]['pred_sem_seg']['data'].cpu(), sm[i:i + 1], 1e-5)


def test_tta_bf16_trained_fullsize():
    K = 19
    o, m = build_pair(K, dtype='bf16')
    sd = trained.train_product(K, [(2, (512, 1024), (4, 8)), (1, (1024, 2048), (8, 16)), (2, (512, 1024), (8, 16))],
                               steps=300)
    o.load_state_dict(sd)
    m.load_state_dict(sd, strict=True)
    tta = SegTTAModel(m.to(DEV))
    imgs, labs = [], []
    for i in range(2):
        im, lb = synth.make_scene(1, 512, 1024, K, seed=700 + i, coarse=(4, 8), ignore_frac=0.03)
        imgs.append(im), labs.append(lb)
    img, lab = torch.cat(imgs), torch.cat(labs)
    data = _tta_data(img, (0.75, 1.0, 1.25))
    ref_logits, ref_metas = _oracle_views(o, data)
    _, ref_pred = tta_oracle.tta_merge(ref_logits, ref_metas, K, 0.3, False)
    res = tta.test_step(data)
    pred = torch.stack([r['pred_sem_seg']['data'] for r in res])
    agree = (pred.cpu() == ref_pred).float().mean().item()
    assert agree >= 0.999, agree
    labels = tta.predict_labels([m.data_preprocessor(dict(inputs=v), False)['inputs'] for v in data['inputs']],
                                data['data_samples'])
    assert labels.dtype == torch.uint8 and torch.equal(labels.long(), pred)
    cm = ops.confusion_accumulate(labels, lab.to(DEV), K)
    ref_cm = oracle.confusion_matrix(labels.cpu().numpy().astype(np.int64), lab.numpy(), K, 255)
    np.testing.assert_array_equal(cm.cpu().numpy(), ref_cm)


def _self_consistent(tta, data):
    """labels of test_step == the CPU restatement over the module's own per-view inference logits"""
    views = [tta.module.data_preprocessor(dict(inputs=i, data_samples=[dict(s) for s in ss]), False)
             for i, ss in zip(data['inputs'], data['data_samples'])]
    lg = [t.cpu() for t in tta._view_logits([v['inputs'] for v in views])]
    metas = [[s['metainfo'] for s in ss] for ss in data['data_samples']]
    merged, ref_pred = tta_oracle.tta_merge(lg, metas, tta.module.out_channels, 0.3, tta.module.align_corners)
    res = tta.test_step(data)
    pred = torch.stack([r['pred_sem_seg']['data'] for r in res])
    _check_labels(pred, ref_pred, merged, 1e-5)
    return pred


def test_tta_led_variant_and_slide_and_chunking():
    K = 19
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        m = L.EncoderDecoder(dict(type='LEDNet', variant='led'),
                             dict(type='LEDHead', in_channels=128, channels=64, num_classes=K, dropout_ratio=0.),
                             data_preprocessor=dict(type='SegDataPreProcessor', mean=list(L.engine.MEAN),
                                                    std=list(L.engine.STD), bgr_to_rgb=True), compute_dtype='fp32').eval()
    sd = synth.make_state_dict(m.state_dict(), seed=4)
    sd['backbone.fusion_kernel'] = m.state_dict()['backbone.fusion_kernel'].clone()
    m.load_state_dict(sd)
    tta = SegTTAModel(m.to(DEV))
    _self_consistent(tta, _tta_data(synth.make_images_u8(1, 512, 512, seed=23), (1.0, 1.125)))

    _, ms, tta_s = _tta_pair(K)
    ms.test_cfg = dict(mode='slide', crop_size=(64, 64), stride=(48, 48))
    data = _tta_data(synth.make_images_u8(2, 96, 128, seed=24), (0.75, 1.0))
    pred = _self_consistent(tta_s, data)
    tta_s.MAX_TTA_BATCH = 1                                      # every module.inference call gets one image
    pred1 = torch.stack([r['pred_sem_seg']['data'] for r in tta_s.test_step(data)])
    assert torch.equal(pred1, pred)

    _, mw, tta_w = _tta_pair(K)
    data = _tta_data(synth.make_images_u8(2, 64, 96, seed=25), (0.5, 1.0))
    pred = torch.stack([r['pred_sem_seg']['data'] for r in tta_w.test_step(data)])
    tta_w.MAX_TTA_BATCH = 1
    assert torch.equal(torch.stack([r['pred_sem_seg']['data'] for r in tta_w.test_step(data)]), pred)


def test_tta_sigmoid_mode_through_the_model():
    """LEDHead(out_channels=1) broadcasts to num_classes channels: the sigmoid branch yields a float [K, H, W] mask"""
    K = 2
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        m1 = L.EncoderDecoder(dict(type='LEDNet'), dict(type='LEDHead', in_channels=128, channels=64, num_classes=K,
                                                         out_channels=1, dropout_ratio=0., tap_channels=32),
                              data_preprocessor=dict(type='SegDataPreProcessor', mean=list(L.engine.MEAN),
                                                     std=list(L.engine.STD), bgr_to_rgb=True), compute_dtype='fp32').eval()
    m1.load_state_dict(synth.make_state_dict(m1.state_dict(), seed=6))
    tta = SegTTAModel(m1.to(DEV))
    assert tta._mode() == (1, 0.3)
    data = _tta_data(synth.make_images_u8(2, 64, 96, seed=26), (0.75, 1.0))
    res = tta.test_step(data)
    mask = torch.stack([r['pred_sem_seg']['data'] for r in res])
    assert mask.dtype == torch.float32 and tuple(mask.shape) == (2, K, 64, 96)
    views = [m1.data_preprocessor(dict(inputs=i), False)['inputs'] for i in data['inputs']]
    lg = [t.cpu() for t in tta._view_logits(views)]
    metas = [[s['metainfo'] for s in ss] for ss in data['data_samples']]
    merged, ref = tta_oracle.tta_merge(lg, metas, 1, 0.3, False)
    near = (merged - 0.3).abs() < 1e-6
    assert torch.equal(mask.cpu()[~near], ref[~near])


# ------------------------------------------------------------------ 7. error conventions
def test_tta_merge_errors():
    lg = torch.randn(1, 3, 8, 8, device=DEV)
    with pytest.raises(L.LedB200Error):
        ops.tta_merge([], (8, 8))
    with pytest.raises(L.LedB200Error):
        ops.tta_merge([(lg, None, None)] * 33, (8, 8))
    with pytest.raises(L.LedB200Error):
        ops.tta_merge([(torch.randn(1, 256, 4, 4, device=DEV), None, None)], (4, 4))
    with pytest.raises(L.LedB200Error):
        ops.tta_merge([(lg, (0, 0, 4, 4), None)], (8, 8))             # the crop removes the whole view
    with pytest.raises(L.LedB200Error):
        ops.tta_merge([(lg, (0, 9, 0, 0), None)], (8, 8))
    with pytest.raises(AssertionError):
        ops.tta_merge([(lg, None, None), (torch.randn(2, 3, 8, 8, device=DEV), None, None)], (8, 8))
    with pytest.raises(L.LedB200Error):
        ops.tta_merge([(lg, None, None)], (8, 8), mode=0, pred_dtype=torch.float32)
    torch.cuda.synchronize()                                          # nothing was launched, nothing faulted
    pred, _ = ops.tta_merge([(lg, None, None)], (8, 8))
    assert torch.equal(pred, lg.argmax(dim=1))
