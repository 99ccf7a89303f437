"""The training augmentation kernels (csrc/augment.cu) bit for bit against the numpy restatement
(tests/augment_oracle.py), DeviceAugSegDataPreProcessor end to end, one training step fed by it, and the C ABI's error
conventions."""
import warnings

import numpy as np
import pytest
import torch

import lednet_b200 as L
from lednet_b200 import lib as LIB, ops, synth
from lednet_b200.augment import DeviceAugSegDataPreProcessor
import augment_oracle as A

pytestmark = pytest.mark.gpu
DEV = 'cuda'
MEAN, STD = [123.675, 116.28, 103.53], [58.395, 57.12, 57.375]
ALL_PM = dict(brightness=-17.3, contrast_mode=0, contrast=1.31, saturation=0.62, hue=-7)
NO_PM = dict(brightness=None, contrast_mode=0, contrast=None, saturation=None, hue=None)


def _images(n, h, w, K, seed, label_dtype=np.uint8, ignore=True):
    rng = np.random.default_rng(seed)
    # smooth-ish images: random blocks upsampled, plus noise, so resizes and HSV see real gradients
    base = rng.integers(0, 256, (n, 3, h // 8 + 1, w // 8 + 1)).repeat(8, 2).repeat(8, 3)[:, :, :h, :w]
    img = np.clip(base + rng.integers(-40, 40, (n, 3, h, w)), 0, 255).astype(np.uint8)
    lab = rng.integers(0, K, (n, h // 4 + 1, w // 4 + 1)).repeat(4, 1).repeat(4, 2)[:, :h, :w]
    if ignore:
        lab[:, : h // 6] = 255
    return img, lab.astype(label_dtype)


def _params(h, w, ratio, crop, rng, n_cand=1, flip=False, pm=NO_PM):
    rh, rw = int(h * ratio + 0.5), int(w * ratio + 0.5)
    mh, mw = max(rh - crop[0], 0), max(rw - crop[1], 0)
    cands = [(int(rng.integers(0, mh + 1)), int(rng.integers(0, mw + 1))) for _ in range(n_cand)]
    return dict(resized_hw=(rh, rw), candidates=cands, flip=flip, **pm)


def _oracle(img, lab, params, crop, Hp, Wp, cat=1.0, ignore_index=255, mean=MEAN, std=STD):
    outs, labs, ks = [], [], []
    for i, p in enumerate(params):
        im, seg, k = A.augment(img[i], lab[i], p, crop, cat, ignore_index)
        o, lb = A.preprocess(im, seg, Hp, Wp, mean, std, bgr_to_rgb=True)
        outs.append(o); labs.append(lb); ks.append(k)
    return np.stack(outs), np.stack(labs), ks


def _device(img, lab, params, crop, Hp, Wp, cat=1.0, ignore_index=255, mean=MEAN, std=STD):
    n = len(params)
    imgs = [torch.from_numpy(x).to(DEV) for x in img]
    labs = [torch.from_numpy(x).to(DEV) for x in lab]
    out = torch.empty((n, 3, Hp, Wp), dtype=torch.float32, device=DEV)
    lout = torch.empty((n, Hp, Wp), dtype=torch.int64, device=DEV)
    ci = ops.train_augment(imgs, labs, params, crop, out, lout, cat_max_ratio=cat, ignore_index=ignore_index,
                           swap_rb=True, mean=mean, std=std, pad_val=0.0, seg_pad_val=255)
    torch.cuda.synchronize()
    return out.cpu().numpy(), lout.cpu().numpy(), (ci.cpu().tolist() if ci is not None else [0] * n)


def _check(img, lab, params, crop, Hp, Wp, **kw):
    o_ref, l_ref, k_ref = _oracle(img, lab, params, crop, Hp, Wp, **kw)
    o, lb, k = _device(img, lab, params, crop, Hp, Wp, **kw)
    assert k == k_ref
    assert np.array_equal(lb, l_ref)
    bad = o.view(np.int32) != o_ref.view(np.int32)
    assert not bad.any(), f'{int(bad.sum())} of {bad.size} image values differ, first at {np.argwhere(bad)[0]}'
    return k


@pytest.mark.parametrize('ratio', [0.5, 1.0, 2.0, 'random'])
@pytest.mark.parametrize('flip', [False, True])
def test_ratios_bit_exact(ratio, flip):
    rng = np.random.default_rng(1)
    h, w, crop = 120, 200, (96, 160)
    img, lab = _images(3, h, w, 19, seed=2)
    params = []
    for i in range(3):
        r = float(rng.uniform(0.5, 2.0)) if ratio == 'random' else ratio
        params.append(_params(h, w, r, crop, rng, flip=flip, pm=ALL_PM))
    _check(img, lab, params, crop, 96, 160)


def test_crop_larger_than_resized_frame_pads_and_flips_inside_extent():
    rng = np.random.default_rng(3)
    h, w, crop = 100, 150, (128, 256)
    img, lab = _images(2, h, w, 5, seed=4)
    params = [_params(h, w, 0.5, crop, rng, flip=True, pm=ALL_PM), _params(h, w, 1.3, crop, rng, flip=False, pm=NO_PM)]
    _check(img, lab, params, crop, 128, 256)


@pytest.mark.parametrize('step', ['none', 'brightness', 'contrast0', 'contrast1', 'saturation', 'hue', 'all', 'all_mode1'])
def test_photometric_branches_bit_exact(step):
    pm = dict(NO_PM)
    if step == 'brightness':
        pm['brightness'] = 23.7
    elif step.startswith('contrast'):
        pm.update(contrast=0.71, contrast_mode=int(step[-1]))
    elif step == 'saturation':
        pm['saturation'] = 1.43
    elif step == 'hue':
        pm['hue'] = 17
    elif step.startswith('all'):
        pm = dict(ALL_PM, contrast_mode=1 if step == 'all_mode1' else 0)
    rng = np.random.default_rng(5)
    img, lab = _images(2, 90, 130, 19, seed=6)
    params = [_params(90, 130, r, (64, 96), rng, flip=bool(i), pm=pm) for i, r in enumerate((0.77, 1.61))]
    _check(img, lab, params, (64, 96), 64, 96)


def test_photometric_exhaustive_colours():
    """every colour of a 256^3 cube through saturation + hue (two lossy HSV round trips) and both contrast orders at
    ratio 1 (the taps reduce to the source pixel)"""
    b, g, r = np.meshgrid(np.arange(256), np.arange(256), np.arange(256), indexing='ij')
    img = np.stack([b, g, r]).astype(np.uint8).reshape(1, 3, 4096, 4096)
    lab = np.zeros((1, 4096, 4096), np.uint8)
    for pm in (ALL_PM, dict(ALL_PM, contrast_mode=1, hue=11, saturation=1.37, brightness=9.6)):
        params = [dict(resized_hw=(4096, 4096), candidates=[(0, 0)], flip=False, **pm)]
        _check(img, lab, params, (4096, 4096), 4096, 4096)


@pytest.mark.parametrize('K', [2, 19])
@pytest.mark.parametrize('ldt', [np.uint8, np.int64], ids=['u8', 'i64'])
def test_crop_select_bit_exact(K, ldt):
    rng = np.random.default_rng(7 + K)
    h, w, crop = 160, 240, (64, 96)
    img, lab = _images(4, h, w, K, seed=K, label_dtype=ldt)
    params = [_params(h, w, float(rng.uniform(0.5, 2.0)), crop, rng, n_cand=11, flip=bool(i % 2), pm=ALL_PM)
              for i in range(4)]
    _check(img, lab, params, crop, 64, 96, cat=0.75)
    _check(img, lab, params, crop, 64, 96, cat=0.3)                 # nearly every box fails: the eleventh is used


@pytest.mark.parametrize('ldt', [np.uint8, np.int64], ids=['u8', 'i64'])
def test_first_k_candidates_fail(ldt):
    """left half one class (every box there fails), right half two classes (every box there passes): with the first
    k boxes on the left the kernel picks box k; with all ten on the left, the eleventh"""
    h, w, crop = 64, 128, (16, 16)
    lab = np.zeros((1, h, w), ldt)
    lab[0, :, 64:] = np.tile(np.arange(2).repeat(4), 8)[None, :64]
    lab[0, :8, :] = 255                                            # ignore_index rows
    img = _images(1, h, w, 2, seed=9)[0]
    left, right = (20, 10), (20, 90)
    params, want = [], []
    for k in range(11):
        params.append(dict(resized_hw=(h, w), candidates=[left] * k + [right] * (11 - k), flip=False, **ALL_PM))
        want.append(min(k, 10))
    imgs, labs = np.repeat(img, 11, 0), np.repeat(lab, 11, 0)
    assert _check(imgs, labs, params, crop, 16, 16, cat=0.75) == want


def test_chunks_of_64_and_seed_reproducible():
    pipe = [dict(type='RandomResize', scale=(160, 80), ratio_range=(0.5, 2.0), keep_ratio=True),
            dict(type='RandomCrop', crop_size=(64, 64), cat_max_ratio=0.75),
            dict(type='RandomFlip', prob=0.5), dict(type='PhotoMetricDistortion')]
    img, lab = _images(70, 60, 110, 7, seed=11)

    def run(seed):
        pp = DeviceAugSegDataPreProcessor(train_pipeline=pipe, seed=seed, mean=MEAN, std=STD, bgr_to_rgb=True,
                                          size=(64, 64), seg_pad_val=255)
        samples = [dict(gt_sem_seg=dict(data=torch.from_numpy(lab[i:i + 1]).to(DEV))) for i in range(70)]
        out = pp(dict(inputs=[torch.from_numpy(x).to(DEV) for x in img], data_samples=samples), training=True)
        return out, samples

    (o1, s1), (o2, s2), (o3, _) = run(5), run(5), run(6)
    assert torch.equal(o1['inputs'], o2['inputs']) and not torch.equal(o1['inputs'], o3['inputs'])
    # replay every sample through the restatement from its recorded parameters
    params = [s['metainfo']['aug_params'] for s in s1]
    o_ref, l_ref, k_ref = _oracle(img, lab, params, (64, 64), 64, 64, cat=0.75)
    assert [int(p['crop_index']) for p in params] == k_ref
    assert np.array_equal(o1['inputs'].cpu().numpy().view(np.int32), o_ref.view(np.int32))
    assert np.array_equal(torch.stack([s['gt_sem_seg']['data'] for s in s1]).cpu().numpy()[:, 0], l_ref)
    m = s1[0]['metainfo']
    p = params[0]
    eh, ew = min(64, p['resized_hw'][0]), min(64, p['resized_hw'][1])
    assert m['img_shape'] == (eh, ew) and m['pad_shape'] == (64, 64) and m['padding_size'] == (0, 64 - ew, 0, 64 - eh)
    assert m['scale_factor'] == (p['resized_hw'][1] / 110, p['resized_hw'][0] / 60)
    assert m['flip'] == p['flip'] and m['flip_direction'] == ('horizontal' if p['flip'] else None)


def test_eval_mode_is_the_plain_preprocessor():
    pipe = [dict(type='RandomResize', scale=(160, 80), ratio_range=(0.5, 2.0), keep_ratio=True),
            dict(type='RandomCrop', crop_size=(64, 64), cat_max_ratio=0.75),
            dict(type='RandomFlip', prob=0.5), dict(type='PhotoMetricDistortion')]
    img, _ = _images(2, 60, 110, 7, seed=12)
    x = torch.from_numpy(img).to(DEV)
    a = DeviceAugSegDataPreProcessor(train_pipeline=pipe, mean=MEAN, std=STD, bgr_to_rgb=True)(dict(inputs=x), False)
    b = L.SegDataPreProcessor(mean=MEAN, std=STD, bgr_to_rgb=True)(dict(inputs=x), False)
    assert torch.equal(a['inputs'], b['inputs'])


def test_train_step_same_loss_bits_as_restated_batch():
    """one EncoderDecoder.train_step fed through the device augmentation gives the loss bits of the same weights fed the
    restatement's batch through the plain path"""
    K, N = 5, 2
    pipe = [dict(type='RandomResize', scale=(256, 128), ratio_range=(0.5, 2.0), keep_ratio=True),
            dict(type='RandomCrop', crop_size=(64, 128), cat_max_ratio=0.75),
            dict(type='RandomFlip', prob=0.5), dict(type='PhotoMetricDistortion')]
    img, lab = _images(N, 96, 192, K, seed=13)

    def model(pp):
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            m = L.EncoderDecoder(dict(type='LEDNet'),
                                 dict(type='LEDHead', in_channels=128, channels=64, num_classes=K, dropout_ratio=0.),
                                 data_preprocessor=pp, compute_dtype='fp32')
        m.load_state_dict(synth.make_state_dict(m.state_dict(), seed=2))
        return m.to(DEV).train()

    pp = dict(type='DeviceAugSegDataPreProcessor', train_pipeline=pipe, seed=1, mean=MEAN, std=STD, bgr_to_rgb=True,
              size=(64, 128), seg_pad_val=255)
    m1 = model(pp)
    samples = [dict(gt_sem_seg=dict(data=torch.from_numpy(lab[i:i + 1]).to(DEV))) for i in range(N)]
    log1 = m1.train_step(dict(inputs=[torch.from_numpy(x).to(DEV) for x in img], data_samples=samples),
                         L.FlatSGD(m1.parameters(), lr=0.01))
    params = [s['metainfo']['aug_params'] for s in samples]
    o_ref, l_ref, _ = _oracle(img, lab, params, (64, 128), 64, 128, cat=0.75)
    m2 = model(None)
    ref_samples = [dict(gt_sem_seg=dict(data=torch.from_numpy(l_ref[i:i + 1]).to(DEV))) for i in range(N)]
    log2 = m2.train_step(dict(inputs=torch.from_numpy(o_ref).to(DEV), data_samples=ref_samples),
                         L.FlatSGD(m2.parameters(), lr=0.01))
    l1, l2 = float(log1['loss'].detach()), float(log2['loss'].detach())
    assert np.float32(l1).tobytes() == np.float32(l2).tobytes(), (l1, l2)


def test_error_conventions():
    lib = LIB.get()
    img = torch.zeros((3, 16, 16), dtype=torch.uint8, device=DEV)
    lab = torch.zeros((16, 16), dtype=torch.uint8, device=DEV)
    out = torch.empty((1, 3, 16, 16), device=DEV)
    lout = torch.empty((1, 16, 16), dtype=torch.int64, device=DEV)
    ci = torch.empty(1, dtype=torch.int32, device=DEV)
    p = dict(resized_hw=(16, 16), candidates=[(0, 0)] * 3, flip=False, **NO_PM)

    def desc(**kw):
        d = ops._aug_desc(p, img, lab)
        for k, v in kw.items():
            setattr(d, k, v)
        return (LIB.AugSample * 1)(d)

    st = LIB.stream_ptr()

    def aug(arr, n=1, ch=16, cw=16, dt=LIB.U8, o=out):
        return lib.ledb200_train_augment(arr, n, ch, cw, dt, ops._p(ci), 1, None, None, 0.0, ops._p(o), 16, 16,
                                         ops._p(lout), 255, st)

    def sel(arr, n=1, ign=255, idx=ci):
        return lib.ledb200_crop_select(arr, n, 16, 16, LIB.U8, 0.75, ign, ops._p(idx), st)

    assert sel(desc()) == 0 and aug(desc()) == 0
    assert aug(None) == LIB_EINVAL and sel(None) == LIB_EINVAL
    assert aug(desc(), n=0) == LIB_EINVAL and aug(desc(), n=65) == LIB_EINVAL
    assert aug(desc(img=None)) == LIB_EINVAL and aug(desc(label=None)) == LIB_EINVAL
    assert aug(desc(), o=None) == LIB_EINVAL and sel(desc(), idx=None) == LIB_EINVAL
    assert aug(desc(h=0)) == LIB_EINVAL and aug(desc(rw=0)) == LIB_EINVAL
    assert aug(desc(num_candidates=12)) == LIB_EINVAL and aug(desc(num_candidates=0)) == LIB_EINVAL
    assert aug(desc(), dt=LIB.F32) == LIB_EINVAL and aug(desc(), dt=LIB.I32) == LIB_EINVAL
    assert aug(desc(), ch=0) == LIB_EINVAL and aug(desc(), cw=0) == LIB_EINVAL
    assert aug(desc(flip=2)) == LIB_EINVAL and sel(desc(), ign=-1) == LIB_EINVAL
    bad = desc()
    bad[0].offsets[1][0] = 1                                       # outside [0, max(rh - crop_h, 0)]
    assert aug(bad) == LIB_EINVAL
    assert b'candidate' in lib.ledb200_last_error()
    with pytest.raises(L.LedB200Error):
        ops.train_augment([img], [lab], [dict(p, candidates=[(0, 0)] * 12)], (16, 16), out, lout)
    with pytest.raises(L.LedB200Error):
        ops.train_augment([img.float()], [lab], [p], (16, 16), out, lout)
    torch.cuda.synchronize()


LIB_EINVAL = -1
