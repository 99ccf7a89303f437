"""CPU checks of the training augmentation: the numpy restatement (tests/augment_oracle.py) against cv2, the rescale
arithmetic, the host sampler of DeviceAugSegDataPreProcessor and its config validation."""
import copy

import numpy as np
import pytest

import lednet_b200 as L
from lednet_b200.augment import DeviceAugSegDataPreProcessor, draw_sample, parse_pipeline, rescale_size
import augment_oracle as A

cv2 = pytest.importorskip('cv2')

VOC = [dict(type='RandomResize', scale=(2048, 512), ratio_range=(0.5, 2.0), keep_ratio=True),
       dict(type='RandomCrop', crop_size=(512, 512), cat_max_ratio=0.75),
       dict(type='RandomFlip', prob=0.5),
       dict(type='PhotoMetricDistortion')]


def _all_colours():
    b, g, r = np.meshgrid(np.arange(256), np.arange(256), np.arange(256), indexing='ij')
    return np.stack([b, g, r], -1).astype(np.uint8).reshape(4096, 4096, 3)


def test_bgr2hsv_exhaustive_bit_exact():
    img = _all_colours()
    for rows in (slice(0, 2048), slice(2048, 4096)):
        part = np.ascontiguousarray(img[rows])
        assert np.array_equal(A.bgr2hsv(part), cv2.cvtColor(part, cv2.COLOR_BGR2HSV))


def test_hsv2bgr_exhaustive_bit_exact():
    h, s, v = np.meshgrid(np.arange(180), np.arange(256), np.arange(256), indexing='ij')
    hsv = np.stack([h, s, v], -1).astype(np.uint8).reshape(180 * 256, 256, 3)
    for rows in (slice(0, 90 * 256), slice(90 * 256, 180 * 256)):
        part = np.ascontiguousarray(hsv[rows])
        assert np.array_equal(A.hsv2bgr(part), cv2.cvtColor(part, cv2.COLOR_HSV2BGR))


@pytest.mark.parametrize('seed', range(6))
def test_inter_linear_within_one_lsb(seed):
    """cv2 runs a scalar tail on the last columns of a row, which rounds the vertical pass differently"""
    rng = np.random.default_rng(seed)
    h, w = int(rng.integers(20, 600)), int(rng.integers(20, 800))
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    for ratio in (0.5, 1.0, 2.0, float(rng.uniform(0.5, 2.0))):
        dh, dw = int(h * ratio + 0.5), int(w * ratio + 0.5)
        d = np.abs(A.resize_linear(img, dh, dw).astype(int) -
                   cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR).astype(int))
        assert d.max() <= 1 and (d > 0).mean() < 0.01, (ratio, d.max(), (d > 0).mean())


@pytest.mark.parametrize('seed', range(6))
def test_inter_nearest_exact(seed):
    rng = np.random.default_rng(100 + seed)
    h, w = int(rng.integers(20, 600)), int(rng.integers(20, 800))
    lab = rng.integers(0, 20, (h, w), dtype=np.uint8)
    for ratio in (0.5, 1.0, 2.0, float(rng.uniform(0.5, 2.0))):
        dh, dw = int(h * ratio + 0.5), int(w * ratio + 0.5)
        assert np.array_equal(A.resize_nearest(lab, dh, dw), cv2.resize(lab, (dw, dh), interpolation=cv2.INTER_NEAREST))


def test_convert_two_roundings_and_truncation():
    x = np.arange(256, dtype=np.uint8)
    ref = np.clip(x.astype(np.float32) * 1.3 + 0, 0, 255).astype(np.uint8)
    assert np.array_equal(A.convert(x, alpha=1.3), ref)
    assert np.array_equal(A.convert(x, beta=-20.7), np.clip(x.astype(np.float32) - np.float32(20.7), 0, 255).astype(np.uint8))


def test_rescale_size():
    """mmcv.rescale_size(keep_ratio): the scale factor fits the long side into max(scale), the short into min(scale)"""
    assert rescale_size(1024, 2048, (2048, 1024)) == (1024, 2048)
    assert rescale_size(1024, 2048, (1024, 512)) == (512, 1024)
    assert rescale_size(1024, 2048, (4096, 2048)) == (2048, 4096)
    assert rescale_size(375, 500, (2048, 512)) == (512, 683)          # short side bound: 375 * 512 / 375, 500 * 1.3653
    assert rescale_size(500, 333, (3000, 768)) == (1153, 768)
    h, w, s = 481, 771, (1357, 377)
    f = min(max(s) / max(h, w), min(s) / min(h, w))
    assert rescale_size(h, w, s) == (int(h * f + 0.5), int(w * f + 0.5))


def _replay(rng, cfg, h, w):
    """draw_sample's draw order written out"""
    lo, hi = cfg['ratio_range']
    ratio = rng.random() * (hi - lo) + lo
    rh, rw = rescale_size(h, w, (int(cfg['scale'][0] * ratio), int(cfg['scale'][1] * ratio)))
    cands = [(int(rng.integers(0, max(rh - cfg['crop_size'][0], 0) + 1)),
              int(rng.integers(0, max(rw - cfg['crop_size'][1], 0) + 1))) for _ in range(11 if cfg['cat_max_ratio'] < 1 else 1)]
    flip = rng.random() < cfg['prob']
    seq = [ratio, (rh, rw), cands, flip]
    b = float(rng.uniform(-32, 32)) if rng.integers(2) else None
    mode = int(rng.integers(2))
    c = float(rng.uniform(0.5, 1.5)) if mode == 1 and rng.integers(2) else None
    s = float(rng.uniform(0.5, 1.5)) if rng.integers(2) else None
    hu = int(rng.integers(-18, 18)) if rng.integers(2) else None
    if mode == 0:
        c = float(rng.uniform(0.5, 1.5)) if rng.integers(2) else None
    return seq + [b, mode, c, s, hu]


def test_sampler_draw_order_and_ranges():
    cfg = parse_pipeline(VOC)
    g1, g2 = np.random.default_rng(7), np.random.default_rng(7)
    seen = dict(flip=set(), mode=set(), b=0, c=0, s=0, h=0)
    for i in range(400):
        h, w = (1024, 2048) if i % 2 else (375, 500)
        p = draw_sample(g1, cfg, h, w)
        r = _replay(g2, cfg, h, w)
        assert [p['ratio'], p['resized_hw'], p['candidates'], p['flip'], p['brightness'], p['contrast_mode'],
                p['contrast'], p['saturation'], p['hue']] == r
        assert 0.5 <= p['ratio'] < 2.0 and len(p['candidates']) == 11
        rh, rw = p['resized_hw']
        for oy, ox in p['candidates']:
            assert 0 <= oy <= max(rh - 512, 0) and 0 <= ox <= max(rw - 512, 0)
        assert p['brightness'] is None or -32 <= p['brightness'] < 32
        assert p['contrast'] is None or 0.5 <= p['contrast'] < 1.5
        assert p['saturation'] is None or 0.5 <= p['saturation'] < 1.5
        assert p['hue'] is None or -18 <= p['hue'] < 18
        seen['flip'].add(p['flip']); seen['mode'].add(p['contrast_mode'])
        for k, key in (('b', 'brightness'), ('c', 'contrast'), ('s', 'saturation'), ('h', 'hue')):
            seen[k] += p[key] is not None
    assert seen['flip'] == {True, False} and seen['mode'] == {0, 1}
    assert all(100 < seen[k] < 300 for k in 'bcsh')


def test_sampler_seed_reproducible_and_one_box_without_cat_max_ratio():
    a = DeviceAugSegDataPreProcessor(train_pipeline=VOC, seed=3)
    b = DeviceAugSegDataPreProcessor(train_pipeline=VOC, seed=3)
    c = DeviceAugSegDataPreProcessor(train_pipeline=VOC, seed=4)
    shapes = [(1024, 2048), (500, 375)]
    pa, pb, pc = a.draw(shapes), b.draw(shapes), c.draw(shapes)
    assert pa == pb and pa != pc
    assert a.draw(shapes) != pa                                   # the stream advances from batch to batch
    voc = copy.deepcopy(VOC)
    del voc[1]['cat_max_ratio']
    p = DeviceAugSegDataPreProcessor(train_pipeline=voc).draw(shapes)
    assert all(len(q['candidates']) == 1 for q in p)


def test_crop_rule_eleventh_box_unchecked():
    """the first passing box of the first ten wins; when all ten fail the eleventh is used without a check"""
    seg = np.zeros((40, 40), np.uint8)
    seg[:, 20:] = 1                                               # two classes only in boxes that straddle x = 20
    seg[30:, :] = 255
    bad, good = (0, 0), (0, 15)                                   # 10 x 10 boxes: x 0..9 one class; x 15..24 two
    for k in range(11):
        cands = [bad] * k + [good] * (11 - k)
        assert A.choose_crop(seg, cands, (10, 10), 0.75) == min(k, 10)
    assert A.choose_crop(seg, [bad] * 11, (10, 10), 0.75) == 10
    assert A.choose_crop(seg, [(30, 15)] * 10 + [bad], (10, 10), 0.75) == 10   # ignore_index only: no class left
    assert A.choose_crop(seg, [good, bad], (10, 10), 1.0) == 1                 # cat_max_ratio >= 1: the last box
    assert A.crop_accepted(seg[0:10, 15:25], 0.75) and not A.crop_accepted(seg[0:10, 15:25], 0.5)


def test_config_validation():
    P = DeviceAugSegDataPreProcessor
    P(train_pipeline=VOC, mean=[1., 2., 3.], std=[1., 1., 1.], size=(512, 512), bgr_to_rgb=True)
    with pytest.raises(NotImplementedError):
        P(train_pipeline=VOC[:3])
    with pytest.raises(NotImplementedError):
        P(train_pipeline=[VOC[1], VOC[0], VOC[2], VOC[3]])
    with pytest.raises(NotImplementedError):
        P(train_pipeline=VOC[:3] + [dict(type='RandomRotate', prob=0.5, degree=10)])
    with pytest.raises(NotImplementedError):
        P(train_pipeline=None)
    bad = [(0, dict(keep_ratio=False)), (0, dict(clip_object_border=False)), (1, dict(crop_size=(512, 512, 3))),
           (1, dict(ignore_index=-1)), (2, dict(direction='vertical')), (2, dict(prob=[0.5])), (3, dict(foo=1))]
    for i, kw in bad:
        pipe = copy.deepcopy(VOC)
        pipe[i].update(kw)
        with pytest.raises(NotImplementedError):
            P(train_pipeline=pipe)
    for i, kw, exc in [(1, dict(crop_size=(0, 512)), AssertionError), (2, dict(prob=1.5), AssertionError),
                       (2, dict(prob=1), ValueError), (0, dict(ratio_range=(2.0, 0.5)), AssertionError)]:
        pipe = copy.deepcopy(VOC)
        pipe[i].update(kw)
        with pytest.raises(exc):
            P(train_pipeline=pipe)
    assert L.MODELS.get('DeviceAugSegDataPreProcessor') is P


def test_restatement_end_to_end_shapes():
    """one sample through the restatement: the cropped extent, padding and label padding"""
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (3, 60, 90), dtype=np.uint8)
    lab = rng.integers(0, 5, (60, 90), dtype=np.uint8)
    cfg = parse_pipeline([dict(VOC[0], scale=(90, 60)), dict(VOC[1], crop_size=(48, 64)), VOC[2], VOC[3]])
    p = draw_sample(rng, cfg, 60, 90)
    im, seg, k = A.augment(img, lab, p, (48, 64), 0.75)
    rh, rw = p['resized_hw']
    assert im.shape == (min(48, rh), min(64, rw), 3) and seg.shape == im.shape[:2] and 0 <= k <= 10
    x, y = A.preprocess(im, seg, 64, 80, mean=[1., 2., 3.], std=[2., 2., 2.])
    assert x.shape == (3, 64, 80) and y.shape == (64, 80)
    assert (y[im.shape[0]:] == 255).all() and (x[:, :, im.shape[1]:] == 0).all()
