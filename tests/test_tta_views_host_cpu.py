"""CPU checks of the test-time views built on the device: the view sizes and metainfo against mmcv's Resize / imrescale /
RandomFlip arithmetic restated literally, TestTimeAug's view order, the INTER_LINEAR restatement (tests/augment_oracle.py)
against cv2 at the test-time sizes, and the strict parsing of the transform dicts."""
import copy
import itertools

import numpy as np
import pytest
import torch.nn as nn

from lednet_b200.augment import DeviceAugSegDataPreProcessor, parse_resize, view_size
from lednet_b200.tta import SegTTAModel
import augment_oracle as A

RATIOS = [0.5, 0.75, 1.0, 1.25, 1.5, 1.75]
FLIPS = [dict(type='RandomFlip', prob=0., direction='horizontal'),
         dict(type='RandomFlip', prob=1., direction='horizontal')]
TTA = [[dict(type='Resize', scale_factor=r, keep_ratio=True) for r in RATIOS], FLIPS]
VOC_RESIZE = dict(type='Resize', scale=(2048, 512), keep_ratio=True)
SIZES = [(1024, 2048), (720, 1280), (512, 910), (511, 1023), (375, 500)]
TRAIN = [dict(type='RandomResize', scale=(2048, 512), ratio_range=(0.5, 2.0), keep_ratio=True),
         dict(type='RandomCrop', crop_size=(512, 512), cat_max_ratio=0.75),
         dict(type='RandomFlip', prob=0.5),
         dict(type='PhotoMetricDistortion')]


# ---- mmcv 2.x, restated line by line (mmcv/image/geometric.py, mmcv/transforms/processing.py) ----
def _scale_size(size, scale):
    if isinstance(scale, (float, int)):
        scale = (scale, scale)
    w, h = size
    return int(w * float(scale[0]) + 0.5), int(h * float(scale[1]) + 0.5)


def _rescale_size(old_size, scale, return_scale=False):
    w, h = old_size
    if isinstance(scale, (float, int)):
        scale_factor = scale
    elif isinstance(scale, tuple):
        max_long_edge = max(scale)
        max_short_edge = min(scale)
        scale_factor = min(max_long_edge / max(h, w), max_short_edge / min(h, w))
    new_size = _scale_size((w, h), scale_factor)
    return (new_size, scale_factor) if return_scale else new_size


def _mmcv_resize(results, t):
    """Resize(keep_ratio=True).transform on the image: results['scale'], then imrescale and the metainfo."""
    if t.get('scale') is not None:
        results['scale'] = tuple(t['scale'])
    else:
        factor = (t['scale_factor'], t['scale_factor'])                 # Resize.__init__ stores a float as a pair
        results['scale'] = _scale_size(results['img_shape'][::-1], factor)
    h, w = results['img_shape']
    new_w, new_h = _rescale_size((w, h), results['scale'])               # imrescale -> imresize(img, new_size)
    results['img_shape'] = (new_h, new_w)
    results['scale_factor'] = (new_w / w, new_h / h)
    results['keep_ratio'] = True
    return results


def _mmcv_flip(results, t):
    cur_dir = 'horizontal' if t['prob'] == 1. else None                 # RandomFlip._choose_direction
    results['flip'] = cur_dir is not None
    results['flip_direction'] = cur_dir
    return results


def _test_time_aug(h, w, transforms):
    """TestTimeAug.transform: one results dict per itertools.product of the transform lists"""
    out = []
    for combo in itertools.product(*transforms):
        r = dict(img_shape=(h, w), ori_shape=(h, w))
        for t in combo:
            r = (_mmcv_resize if t['type'] == 'Resize' else _mmcv_flip)(r, t)
        out.append({k: r[k] for k in ('img_shape', 'scale_factor', 'keep_ratio', 'flip', 'flip_direction') if k in r})
    return out


@pytest.mark.parametrize('hw', SIZES, ids=[f'{h}x{w}' for h, w in SIZES])
def test_view_plan_matches_mmcv(hw):
    h, w = hw
    tta = SegTTAModel(nn.Identity(), tta_transforms=TTA)
    assert tta.view_plan(h, w) == _test_time_aug(h, w, TTA)
    # ratio-major: the flip pair of every ratio is adjacent, unflipped first as listed
    plan = tta.view_plan(h, w)
    assert [p['flip'] for p in plan] == [False, True] * len(RATIOS)
    assert [p['img_shape'] for p in plan[::2]] == [p['img_shape'] for p in plan[1::2]]
    # the flip list in the other order, and no flip list
    rev = SegTTAModel(nn.Identity(), tta_transforms=[TTA[0], FLIPS[::-1]]).view_plan(h, w)
    assert rev == _test_time_aug(h, w, [TTA[0], FLIPS[::-1]]) and rev[0]['flip'] is True
    one = SegTTAModel(nn.Identity(), tta_transforms=[TTA[0]]).view_plan(h, w)
    assert [dict(p, flip=False, flip_direction=None) for p in plan[::2]] == one
    # the dataset's own Resize
    vs = _test_time_aug(h, w, [[VOC_RESIZE]])[0]
    assert view_size(h, w, parse_resize(VOC_RESIZE)) == vs['img_shape']


def test_known_sizes():
    assert view_size(720, 1280, parse_resize(VOC_RESIZE)) == (512, 910)
    assert view_size(1024, 2048, parse_resize(VOC_RESIZE)) == (512, 1024)
    assert [view_size(1024, 2048, ('scale_factor', r)) for r in RATIOS] == \
        [(512, 1024), (768, 1536), (1024, 2048), (1280, 2560), (1536, 3072), (1792, 3584)]
    assert view_size(511, 1023, ('scale_factor', 0.75)) == (383, 767)


def _smooth_image(h, w, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (h // 8 + 1, w // 8 + 1, 3)).repeat(8, 0).repeat(8, 1)[:h, :w]
    return np.clip(base + rng.integers(-40, 40, (h, w, 3)), 0, 255).astype(np.uint8)


@pytest.mark.parametrize('hw', SIZES[:4], ids=[f'{h}x{w}' for h, w in SIZES[:4]])
def test_inter_linear_restatement_at_view_sizes(hw):
    """within 1 LSB on under 1 % of values; exact at ratio 1.0 (cv2 copies) and at ratio 0.5 on even sizes (cv2's area
    fast path (a + b + c + d + 2) >> 2, which the linear formula gives at weights 1024 / 1024)"""
    cv2 = pytest.importorskip('cv2')
    h, w = hw
    img = _smooth_image(h, w, seed=h + w)
    sizes = {r: view_size(h, w, ('scale_factor', r)) for r in RATIOS}
    sizes['voc'] = view_size(h, w, parse_resize(VOC_RESIZE))
    for key, (dh, dw) in sizes.items():
        ref = cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR)
        d = np.abs(A.resize_linear(img, dh, dw).astype(int) - ref.astype(int))
        assert d.max() <= 1 and (d > 0).mean() < 0.01, (key, d.max(), (d > 0).mean())
        if key == 1.0 or (key == 0.5 and h % 2 == 0 and w % 2 == 0):
            assert d.max() == 0, key


BAD_RESIZE = [dict(keep_ratio=False), dict(keep_ratio=None), dict(scale=(2048, 512)), dict(scale_factor=None),
              dict(scale_factor=(0.5, 0.5)), dict(scale_factor=1), dict(scale_factor=-0.5),
              dict(interpolation='nearest'), dict(backend='pillow'), dict(foo=1)]
BAD_FLIP = [dict(prob=0.5), dict(prob=1), dict(prob=[1.]), dict(direction='vertical'), dict(swap_seg_labels=[(1, 2)])]


def test_tta_transforms_validation():
    SegTTAModel(nn.Identity(), tta_transforms=TTA)
    SegTTAModel(nn.Identity(), tta_transforms=[[dict(VOC_RESIZE, clip_object_border=False)], FLIPS])
    assert SegTTAModel(nn.Identity()).tta is None
    for kw in BAD_RESIZE:
        t = copy.deepcopy(TTA)
        t[0][2].update(kw)
        with pytest.raises(NotImplementedError):
            SegTTAModel(nn.Identity(), tta_transforms=t)
    for kw in BAD_FLIP:
        t = copy.deepcopy(TTA)
        t[1][1].update(kw)
        with pytest.raises(NotImplementedError):
            SegTTAModel(nn.Identity(), tta_transforms=t)
    for t in ([], [[]], [TTA[0], []], TTA + [[dict(type='LoadAnnotations')]], [FLIPS, TTA[0]],
              [TTA[0], [FLIPS[0], FLIPS[0]]], [TTA[0] + [dict(type='RandomFlip', prob=1.)]],
              [[dict(type='RandomResize', scale=(2048, 512), ratio_range=(0.5, 2.0), keep_ratio=True)]], 'Resize'):
        with pytest.raises(NotImplementedError):
            SegTTAModel(nn.Identity(), tta_transforms=t)


def test_test_pipeline_validation():
    P = DeviceAugSegDataPreProcessor
    assert P(train_pipeline=TRAIN).test_resize is None
    assert P(train_pipeline=TRAIN, test_pipeline=[VOC_RESIZE]).test_resize == ('scale', (2048, 512))
    assert P(train_pipeline=TRAIN, test_pipeline=[dict(type='Resize', scale_factor=0.5, keep_ratio=True)]).test_resize \
        == ('scale_factor', 0.5)
    for kw in BAD_RESIZE:
        with pytest.raises(NotImplementedError):
            P(train_pipeline=TRAIN, test_pipeline=[dict(TTA[0][2], **kw)])
    for scale in ((2048,), (2048, 512.), 2048, (0, 512)):
        with pytest.raises(NotImplementedError):
            P(train_pipeline=TRAIN, test_pipeline=[dict(VOC_RESIZE, scale=scale)])
    for pipe in ([], [VOC_RESIZE, VOC_RESIZE], [dict(type='LoadImageFromFile'), VOC_RESIZE], [FLIPS[1]], VOC_RESIZE):
        with pytest.raises(NotImplementedError):
            P(train_pipeline=TRAIN, test_pipeline=pipe)
