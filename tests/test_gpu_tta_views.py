"""The test-time views built on the device (csrc/augment.cu view_resize_kernel) bit for bit against the INTER_LINEAR
restatement (tests/augment_oracle.py) plus SegDataPreProcessor's arithmetic; SegTTAModel(tta_transforms=...) against
the existing SegTTAModel fed the restated views; the test pipeline's Resize in DeviceAugSegDataPreProcessor; and the
C ABI's error conventions."""
import ctypes
import functools
import warnings

import numpy as np
import pytest
import torch

import lednet_b200 as L
from lednet_b200 import lib as LIB, ops, synth
from lednet_b200.augment import DeviceAugSegDataPreProcessor, parse_resize, view_size
from lednet_b200.tta import SegTTAModel
from util import build_pair
import augment_oracle as A
import trained

pytestmark = pytest.mark.gpu
DEV = 'cuda'
MEAN, STD = [123.675, 116.28, 103.53], [58.395, 57.12, 57.375]
RATIOS = [0.5, 0.75, 1.0, 1.25, 1.5, 1.75]
FLIPS = [dict(type='RandomFlip', prob=0., direction='horizontal'),
         dict(type='RandomFlip', prob=1., direction='horizontal')]
VOC_RESIZE = dict(type='Resize', scale=(2048, 512), keep_ratio=True)
TRAIN = [dict(type='RandomResize', scale=(2048, 512), ratio_range=(0.5, 2.0), keep_ratio=True),
         dict(type='RandomCrop', crop_size=(512, 512), cat_max_ratio=0.75),
         dict(type='RandomFlip', prob=0.5), dict(type='PhotoMetricDistortion')]


def _tta(ratios, flips=True):
    t = [[dict(type='Resize', scale_factor=float(r), keep_ratio=True) for r in ratios]]
    return t + [FLIPS] if flips else t


def _images(n, h, w, seed):
    """smooth-ish uint8 [n, 3, h, w]: random blocks plus noise, so the resize sees real gradients"""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (n, 3, h // 8 + 1, w // 8 + 1)).repeat(8, 2).repeat(8, 3)[:, :, :h, :w]
    return np.clip(base + rng.integers(-40, 40, (n, 3, h, w)), 0, 255).astype(np.uint8)


def _restated_u8(img_chw, rh, rw, flip=False):
    """cv2 INTER_LINEAR (restated) of one [3, h, w] uint8 image, then RandomFlip: [3, rh, rw] uint8"""
    v = A.resize_linear(np.ascontiguousarray(img_chw.transpose(1, 2, 0)), rh, rw)
    if flip:
        v = v[:, ::-1]
    return np.ascontiguousarray(v.transpose(2, 0, 1))


def _bits(t):
    return t.detach().cpu().numpy().view(np.int32)


# ------------------------------------------------------------------ 1. kernel against the restatement
def _check_views(img, sizes, Hp, Wp, swap, norm, pad_val=0., outs=(True, True)):
    """view_resize of every image (sizes: one (rh, rw) per image) against the restatement + A.preprocess (numpy) and
    + SegDataPreProcessor's stack_pad kernel on the restated uint8 view"""
    n = len(img)
    mean, std = (MEAN, STD) if norm else (None, None)
    out = torch.full((n, 3, Hp, Wp), float('nan'), device=DEV) if outs[0] else None
    out_f = torch.full((n, 3, Hp, Wp), float('nan'), device=DEV) if outs[1] else None
    ops.view_resize([torch.from_numpy(x).to(DEV) for x in img], sizes, out=out, out_flip=out_f, swap_rb=swap,
                    mean=mean, std=std, pad_val=pad_val)
    for t, flip in ((out, False), (out_f, True)):
        if t is None:
            continue
        for i in range(n):
            rh, rw = sizes[i]
            u8 = _restated_u8(img[i], rh, rw, flip)
            ref, _ = A.preprocess(u8.transpose(1, 2, 0), np.zeros((rh, rw), np.uint8), Hp, Wp, mean, std,
                                  bgr_to_rgb=swap, pad_val=pad_val)
            got = _bits(t[i])
            bad = got != ref.view(np.int32)
            assert not bad.any(), f'image {i} flip {flip}: {int(bad.sum())} values differ, first {np.argwhere(bad)[0]}'
            sp = torch.empty((3, Hp, Wp), device=DEV)
            ops.stack_pad(torch.from_numpy(u8).to(DEV), sp, swap_rb=swap, mean=mean, std=std, pad_val=pad_val)
            assert np.array_equal(_bits(sp), got)


@pytest.mark.parametrize('ratio', RATIOS)
def test_base_ratios_fullsize_bit_exact(ratio):
    img = _images(2, 1024, 2048, seed=1)
    rh, rw = view_size(1024, 2048, ('scale_factor', ratio))
    _check_views(img, [(rh, rw)] * 2, rh, rw, swap=True, norm=True)


@pytest.mark.parametrize('swap,norm', [(False, False), (True, False), (False, True)])
@pytest.mark.parametrize('ratio', RATIOS)
def test_odd_size_swap_and_normalisation(ratio, swap, norm):
    img = _images(1, 511, 1023, seed=2)
    rh, rw = view_size(511, 1023, ('scale_factor', ratio))
    _check_views(img, [(rh, rw)], rh, rw, swap=swap, norm=norm)


@pytest.mark.parametrize('hw,resize', [((720, 1280), VOC_RESIZE), ((512, 910), VOC_RESIZE),
                                       ((37, 53), dict(type='Resize', scale_factor=2.7, keep_ratio=True)),
                                       ((300, 200), dict(type='Resize', scale_factor=0.33, keep_ratio=True))])
def test_size_divisor_padding_up_and_down(hw, resize):
    h, w = hw
    rh, rw = view_size(h, w, parse_resize(resize))
    Hp, Wp = -(-rh // 32) * 32, -(-rw // 32) * 32
    img = _images(2, h, w, seed=h)
    _check_views(img, [(rh, rw)] * 2, Hp, Wp, swap=True, norm=True, pad_val=0.)
    _check_views(img, [(rh, rw)] * 2, Hp, Wp, swap=False, norm=False, pad_val=7.5, outs=(False, True))
    _check_views(img, [(rh, rw)] * 2, Hp, Wp, swap=True, norm=True, pad_val=-1., outs=(True, False))


def test_mixed_sources_and_chunks_of_64():
    rng = np.random.default_rng(3)
    img, sizes = [], []
    for i in range(70):
        h, w = int(rng.integers(9, 60)), int(rng.integers(9, 60))
        img.append(_images(1, h, w, seed=100 + i)[0])
        sizes.append((int(rng.integers(1, 65)), int(rng.integers(1, 97))))
    _check_views(img, sizes, 64, 96, swap=True, norm=True, pad_val=3.)


def test_ratio_one_equals_stack_pad():
    img = torch.from_numpy(_images(2, 1024, 2048, seed=4)).to(DEV)
    for swap, norm in ((True, True), (False, False)):
        mean, std = (MEAN, STD) if norm else (None, None)
        out = torch.empty((2, 3, 1024, 2048), device=DEV)
        out_f = torch.empty_like(out)
        ops.view_resize(list(img), (1024, 2048), out=out, out_flip=out_f, swap_rb=swap, mean=mean, std=std)
        for i in range(2):
            sp = torch.empty((3, 1024, 2048), device=DEV)
            ops.stack_pad(img[i], sp, swap_rb=swap, mean=mean, std=std)
            assert torch.equal(out[i].view(torch.int32), sp.view(torch.int32))
            ops.stack_pad(img[i].flip(-1), sp, swap_rb=swap, mean=mean, std=std)
            assert torch.equal(out_f[i].view(torch.int32), sp.view(torch.int32))


# ------------------------------------------------------------------ 2. SegTTAModel(tta_transforms) end to end
@functools.lru_cache(maxsize=None)
def _trained_sd(K):
    return trained.train_product(K, [(2, (512, 1024), (4, 8)), (1, (1024, 2048), (8, 16)), (2, (512, 1024), (8, 16))],
                                 steps=300)


@functools.lru_cache(maxsize=None)
def _scene(n, h, w, K, seed):
    imgs, labs = [], []
    for i in range(n):
        im, lb = synth.make_scene(1, h, w, K, seed=seed + i, coarse=(4, 8), ignore_frac=0.03)
        imgs.append(im), labs.append(lb)
    return torch.cat(imgs).numpy(), torch.cat(labs)


def _restated_tta_data(img, lab, ratios, flips=(False, True)):
    """what TestTimeAug + LoadAnnotations + PackSegInputs hand over, with the restated cv2 resize: one list per view"""
    n, _, h, w = img.shape
    inputs, samples = [], []
    for r in ratios:
        rh, rw = view_size(h, w, ('scale_factor', float(r)))
        for f in flips:
            inputs.append([torch.from_numpy(_restated_u8(img[i], rh, rw, f)) for i in range(n)])
            samples.append([dict(metainfo=dict(ori_shape=(h, w), img_shape=(rh, rw), scale_factor=(rw / w, rh / h),
                                               keep_ratio=True, flip=f, flip_direction='horizontal' if f else None,
                                               img_path=f'img{i}.png'),
                                 gt_sem_seg=dict(data=lab[i:i + 1].clone())) for i in range(n)])
    return dict(inputs=inputs, data_samples=samples)


def _decoded_data(img, lab):
    n, _, h, w = img.shape
    return dict(inputs=[torch.from_numpy(img[i]) for i in range(n)],
                data_samples=[dict(metainfo=dict(ori_shape=(h, w), img_path=f'img{i}.png'),
                                   gt_sem_seg=dict(data=lab[i:i + 1].clone())) for i in range(n)])


def _compare(m, ratios, img, lab, flips=True):
    ref = SegTTAModel(m).test_step(_restated_tta_data(img, lab, ratios, (False, True) if flips else (False,)))
    tta = SegTTAModel(m, tta_transforms=_tta(ratios, flips))
    res = tta.test_step(_decoded_data(img, lab))
    assert len(res) == len(ref)
    for a, b in zip(res, ref):
        assert a['pred_sem_seg']['data'].dtype == b['pred_sem_seg']['data'].dtype
        assert torch.equal(a['pred_sem_seg']['data'], b['pred_sem_seg']['data'])
        assert torch.equal(a['seg_logits']['data'].view(torch.int32), b['seg_logits']['data'].view(torch.int32))
        for k in ('ori_shape', 'img_shape', 'scale_factor', 'keep_ratio', 'flip', 'flip_direction', 'img_path',
                  'img_padding_size', 'pad_shape'):
            assert a['metainfo'].get(k) == b['metainfo'].get(k), k
        assert torch.equal(a['gt_sem_seg']['data'], b['gt_sem_seg']['data'])
    return tta, res


def _trained_model(K, dtype):
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        m = L.EncoderDecoder(dict(type='LEDNet'), dict(type='LEDHead', in_channels=128, channels=64, num_classes=K,
                                                       dropout_ratio=0.),
                             data_preprocessor=dict(type='SegDataPreProcessor', mean=MEAN, std=STD, bgr_to_rgb=True),
                             compute_dtype=dtype).eval()
    m.load_state_dict(_trained_sd(K), strict=True)
    return m.to(DEV)


@pytest.mark.parametrize('dtype', ['bf16', 'fp32'])
def test_tta_device_views_trained_whole(dtype):
    K = 19
    m = _trained_model(K, dtype)
    img, lab = _scene(2, 512, 1024, K, 700)
    tta, res = _compare(m, RATIOS, img, lab)
    labels = tta.predict_image_labels(torch.from_numpy(img).to(DEV), [{'ori_shape': (512, 1024)}] * 2)
    assert labels.dtype == torch.uint8
    assert torch.equal(labels.long(), torch.stack([r['pred_sem_seg']['data'] for r in res]))


def test_tta_device_views_trained_slide():
    K = 19
    m = _trained_model(K, 'bf16')
    m.test_cfg = dict(mode='slide', crop_size=(512, 512), stride=(384, 384))
    img, lab = _scene(2, 512, 1024, K, 710)
    _compare(m, (0.75, 1.0, 1.25), img, lab)


def test_tta_device_views_padding_and_chunking():
    K = 19
    _, m = build_pair(K)
    m = m.to(DEV)
    m.data_preprocessor.test_cfg = dict(size_divisor=32)              # pads the 0.75 and 1.25 views of 100x150
    img, lab = _scene(2, 100, 150, K, 720)
    tta, res = _compare(m, (0.75, 1.0, 1.25), img, lab)
    assert any(res[0]['metainfo']['img_padding_size'])
    tta.MAX_TTA_BATCH = 1
    again = tta.test_step(_decoded_data(img, lab))
    assert all(torch.equal(a['pred_sem_seg']['data'], b['pred_sem_seg']['data']) for a, b in zip(again, res))
    _compare(m, (0.5, 1.5), img, lab, flips=False)                   # no flip list


def test_tta_device_views_sigmoid_mode():
    K = 2
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        m1 = L.EncoderDecoder(dict(type='LEDNet'), dict(type='LEDHead', in_channels=128, channels=64, num_classes=K,
                                                         out_channels=1, dropout_ratio=0., tap_channels=32),
                              data_preprocessor=dict(type='SegDataPreProcessor', mean=MEAN, std=STD, bgr_to_rgb=True),
                              compute_dtype='fp32').eval()
    m1.load_state_dict(synth.make_state_dict(m1.state_dict(), seed=6))
    img, lab = _scene(2, 512, 1024, K, 730)
    tta, res = _compare(m1.to(DEV), (0.75, 1.0, 1.25), img, lab)
    assert res[0]['pred_sem_seg']['data'].dtype == torch.float32
    with pytest.raises(ValueError):
        tta.predict_image_labels(torch.from_numpy(img).to(DEV))


def test_tta_device_views_input_errors():
    _, m = build_pair(19)
    tta = SegTTAModel(m.to(DEV), tta_transforms=_tta((1.0,)))
    x = torch.zeros((3, 32, 48), dtype=torch.uint8)
    with pytest.raises(NotImplementedError):
        tta.test_step(dict(inputs=[x.float()]))
    with pytest.raises(NotImplementedError):
        tta.test_step(dict(inputs=[x, torch.zeros((3, 32, 40), dtype=torch.uint8)]))
    with pytest.raises(NotImplementedError):
        tta.test_step(dict(inputs=[torch.zeros((1, 32, 48), dtype=torch.uint8)]))
    with pytest.raises(ValueError):
        SegTTAModel(m).predict_image_labels(x[None])


# ------------------------------------------------------------------ 3. the test pipeline's Resize
@pytest.mark.parametrize('test_cfg', [None, dict(size_divisor=32)])
def test_device_test_resize_equals_plain_preprocessor(test_cfg):
    K = 19
    img, _ = _scene(2, 720, 1280, K, 740)
    kw = dict(mean=MEAN, std=STD, bgr_to_rgb=True, test_cfg=test_cfg)
    dev_pp = DeviceAugSegDataPreProcessor(train_pipeline=TRAIN, test_pipeline=[VOC_RESIZE], **kw)
    ref_pp = L.SegDataPreProcessor(**kw)
    rh, rw = 512, 910
    samples = [dict(metainfo=dict(ori_shape=(720, 1280), img_path=f'{i}.png')) for i in range(2)]
    out = dev_pp(dict(inputs=[torch.from_numpy(x) for x in img], data_samples=[dict(s, metainfo=dict(s['metainfo']))
                                                                               for s in samples]), False)
    ref_samples = [dict(metainfo=dict(s['metainfo'], img_shape=(rh, rw), scale_factor=(rw / 1280, rh / 720),
                                      keep_ratio=True)) for s in samples]
    ref = ref_pp(dict(inputs=[torch.from_numpy(_restated_u8(x, rh, rw)) for x in img], data_samples=ref_samples), False)
    assert torch.equal(out['inputs'].view(torch.int32), ref['inputs'].view(torch.int32))
    for a, b in zip(out['data_samples'], ref['data_samples']):
        assert a['metainfo'] == b['metainfo']
    if test_cfg:
        assert out['inputs'].shape[-2:] == (512, 928) and out['data_samples'][0]['metainfo']['pad_shape'] == (512, 928)
    _, m = build_pair(K)
    m = m.to(DEV)
    p1 = m.predict(out['inputs'], out['data_samples'])
    p2 = m.predict(ref['inputs'], ref['data_samples'])
    for a, b in zip(p1, p2):
        assert tuple(a['pred_sem_seg']['data'].shape[-2:]) == (720, 1280)
        assert torch.equal(a['pred_sem_seg']['data'], b['pred_sem_seg']['data'])
    # without a test pipeline, eval stays the plain preprocessor
    plain = DeviceAugSegDataPreProcessor(train_pipeline=TRAIN, **kw)(dict(inputs=torch.from_numpy(img)), False)
    assert torch.equal(plain['inputs'], ref_pp(dict(inputs=torch.from_numpy(img)), False)['inputs'])


# ------------------------------------------------------------------ 4. error conventions
def test_error_conventions_write_nothing():
    lib = LIB.get()
    img = torch.zeros((3, 16, 16), dtype=torch.uint8, device=DEV)
    out = torch.full((3, 16, 16), 7.0, device=DEV)
    out_f = torch.full((3, 16, 16), 7.0, device=DEV)
    m3, s3 = (ctypes.c_float * 3)(1., 2., 3.), (ctypes.c_float * 3)(1., 1., 1.)
    st = LIB.stream_ptr()

    def desc(**kw):
        d = LIB.ViewDesc()
        d.src, d.out, d.out_flip, d.h, d.w, d.rh, d.rw = img.data_ptr(), out.data_ptr(), out_f.data_ptr(), 16, 16, 8, 8
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    def call(descs, n=None, Hp=16, Wp=16, mean=m3, std=s3):
        arr = (LIB.ViewDesc * max(len(descs), 1))(*descs)
        return lib.ledb200_view_resize(arr if descs else None, len(descs) if n is None else n, Hp, Wp, 1, mean, std,
                                       0.0, st)

    EINVAL = -1
    bad = [call([]), call([desc()], n=0), call([desc()] * 65), call([desc(src=None)]),
           call([desc(out=None, out_flip=None)]), call([desc(h=0)]), call([desc(w=0)]), call([desc(rh=0)]),
           call([desc(rw=0)]), call([desc(rh=17)]), call([desc(rw=17)]), call([desc()], Hp=7), call([desc()], Wp=7),
           call([desc()], mean=None), call([desc()], std=None)]
    assert bad == [EINVAL] * len(bad)
    assert b'view_resize' in lib.ledb200_last_error()
    torch.cuda.synchronize()
    assert (out == 7.0).all() and (out_f == 7.0).all()                  # nothing was launched
    assert call([desc()]) == 0 and call([desc(out=None)], mean=None, std=None) == 0
    torch.cuda.synchronize()
    assert not (out == 7.0).all()
    with pytest.raises(L.LedB200Error):
        ops.view_resize([img.float()], (8, 8), out=out[None])
