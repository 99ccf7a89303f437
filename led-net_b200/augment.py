"""`DeviceAugSegDataPreProcessor` (MODELS): the config's training augmentations on the device.

Reference surface: ``mmcv/transforms/processing.py`` (RandomResize -> Resize(keep_ratio=True) -> mmcv.imrescale,
RandomFlip), ``mmseg/datasets/transforms/transforms.py`` (RandomCrop with cat_max_ratio, PhotoMetricDistortion) and
``mmseg/models/data_preprocessor.py`` (SegDataPreProcessor).  The dataloader keeps decoding (LoadImageFromFile,
LoadAnnotations, PackSegInputs); the four transform dicts move from `train_pipeline` into this preprocessor, which draws
their random parameters on the host and runs them, with the swap / normalisation / padding, as two kernel launches per
batch (csrc/augment.cu).
"""
import numpy as np
import torch

from .registry import MODELS
from .png_feed import decode_batch
from .segmentor import SegDataPreProcessor, _meta
from . import ops

PIPELINE = ('RandomResize', 'RandomCrop', 'RandomFlip', 'PhotoMetricDistortion')
NUM_CANDIDATES = 11           # RandomCrop: the first box plus up to 10 redraws


def rescale_size(h, w, scale):
    """mmcv.rescale_size for keep_ratio: (new_h, new_w) of an (h, w) image fitted into `scale` (w, h)."""
    f = min(max(scale) / max(h, w), min(scale) / min(h, w))
    return int(h * f + 0.5), int(w * f + 0.5)


def _pair(v, what):
    if isinstance(v, (list, tuple)) and len(v) == 2:
        return tuple(v)
    raise NotImplementedError(f'{what}: a pair is supported, got {v!r}')


def _check_keys(t, allowed):
    extra = set(t) - {'type'} - set(allowed)
    if extra:
        raise NotImplementedError(f"{t['type']}: unsupported arguments {sorted(extra)}")


def parse_pipeline(pipeline):
    """The four transform dicts of the config, verbatim and in order -> one flat dict of their parameters.
    Any other transform, order or argument raises NotImplementedError; a bad value raises what the reference raises."""
    types = tuple(t.get('type') if isinstance(t, dict) else None for t in pipeline or ())
    if types != PIPELINE:
        raise NotImplementedError(f'train_pipeline must be exactly {list(PIPELINE)} in that order, got {list(types)}')
    rr, rc, rf, pmd = (dict(t) for t in pipeline)
    _check_keys(rr, ('scale', 'ratio_range', 'keep_ratio', 'resize_type'))
    if rr.get('resize_type', 'Resize') != 'Resize' or not rr.get('keep_ratio', False):
        raise NotImplementedError('RandomResize: only resize_type=Resize with keep_ratio=True')
    if rr.get('ratio_range') is None:
        raise NotImplementedError('RandomResize: only the ratio_range form')
    scale = _pair(rr.get('scale'), 'RandomResize scale')
    lo, hi = _pair(rr['ratio_range'], 'RandomResize ratio_range')
    assert lo <= hi                                              # mmcv RandomResize._random_sample_ratio
    _check_keys(rc, ('crop_size', 'cat_max_ratio', 'ignore_index'))
    crop = rc['crop_size']
    crop = (crop, crop) if isinstance(crop, int) else _pair(crop, 'RandomCrop crop_size')
    assert crop[0] > 0 and crop[1] > 0                           # mmseg RandomCrop.__init__
    ignore_index = rc.get('ignore_index', 255)
    if not 0 <= ignore_index <= 255:
        raise NotImplementedError('RandomCrop: ignore_index must lie in [0, 255] (uint8 label maps)')
    _check_keys(rf, ('prob', 'direction'))
    prob = rf.get('prob')
    if isinstance(prob, list):
        raise NotImplementedError('RandomFlip: a single probability')
    if not isinstance(prob, float):
        raise ValueError(f'probs must be float or list of float, but got `{type(prob)}`.')   # mmcv RandomFlip
    assert 0 <= prob <= 1
    direction = rf.get('direction', 'horizontal')
    if direction != 'horizontal':
        raise NotImplementedError("RandomFlip: direction='horizontal' only")
    _check_keys(pmd, ('brightness_delta', 'contrast_range', 'saturation_range', 'hue_delta'))
    return dict(scale=scale, ratio_range=(lo, hi), crop_size=crop, cat_max_ratio=float(rc.get('cat_max_ratio', 1.)),
                ignore_index=int(ignore_index), prob=prob,
                brightness_delta=pmd.get('brightness_delta', 32),
                contrast_range=_pair(pmd.get('contrast_range', (0.5, 1.5)), 'contrast_range'),
                saturation_range=_pair(pmd.get('saturation_range', (0.5, 1.5)), 'saturation_range'),
                hue_delta=int(pmd.get('hue_delta', 18)))


def parse_resize(t):
    """One test-time mmcv Resize dict -> ('scale', (a, b)) or ('scale_factor', r).  keep_ratio=True with cv2's bilinear
    only; exactly one of a `scale` pair or a float `scale_factor`; anything else raises NotImplementedError."""
    if not isinstance(t, dict) or t.get('type') != 'Resize':
        raise NotImplementedError(f'a Resize dict is supported here, got {t!r}')
    _check_keys(t, ('scale', 'scale_factor', 'keep_ratio', 'clip_object_border', 'backend', 'interpolation'))
    if t.get('keep_ratio') is not True:
        raise NotImplementedError('Resize: only keep_ratio=True')
    if t.get('interpolation', 'bilinear') != 'bilinear' or t.get('backend', 'cv2') != 'cv2':
        raise NotImplementedError("Resize: only interpolation='bilinear' with backend='cv2'")
    scale, factor = t.get('scale'), t.get('scale_factor')
    if (scale is None) == (factor is None):
        raise NotImplementedError('Resize: exactly one of scale and scale_factor')
    if scale is not None:
        scale = _pair(scale, 'Resize scale')
        if not all(isinstance(v, int) and v > 0 for v in scale):
            raise NotImplementedError(f'Resize: scale must be two positive ints, got {scale!r}')
        return 'scale', scale
    if not isinstance(factor, float) or not factor > 0:
        raise NotImplementedError(f'Resize: scale_factor must be one positive float, got {factor!r}')
    return 'scale_factor', factor


def view_size(h, w, resize):
    """mmcv Resize.transform (keep_ratio) of an (h, w) image: `_scale_size((w, h), scale_factor)` when the dict gives a
    factor, then mmcv.imrescale's rescale_size.  Returns (rh, rw)."""
    kind, v = resize
    scale = (int(w * v + 0.5), int(h * v + 0.5)) if kind == 'scale_factor' else v
    return rescale_size(h, w, scale)


def parse_flip(t):
    """One test-time RandomFlip dict -> flip (bool): prob exactly 0. or 1., direction='horizontal'."""
    if not isinstance(t, dict) or t.get('type') != 'RandomFlip':
        raise NotImplementedError(f'a RandomFlip dict is supported here, got {t!r}')
    _check_keys(t, ('prob', 'direction'))
    prob = t.get('prob')
    if not isinstance(prob, float) or prob not in (0., 1.):
        raise NotImplementedError(f'RandomFlip: prob must be exactly 0. or 1. at test time, got {prob!r}')
    if t.get('direction', 'horizontal') != 'horizontal':
        raise NotImplementedError("RandomFlip: direction='horizontal' only")
    return prob == 1.


def parse_tta_transforms(transforms):
    """The first two lists of TestTimeAug.transforms, verbatim: [[Resize ...], [RandomFlip ...]] (the flip list is
    optional) -> (resizes, flips).  Each flip state may appear once."""
    if not isinstance(transforms, (list, tuple)) or len(transforms) not in (1, 2):
        raise NotImplementedError('tta_transforms: [[Resize, ...]] or [[Resize, ...], [RandomFlip, ...]]')
    if not all(isinstance(ts, (list, tuple)) and len(ts) > 0 for ts in transforms):
        raise NotImplementedError('tta_transforms: each entry is a non-empty list of transform dicts')
    resizes = [parse_resize(t) for t in transforms[0]]
    flips = [parse_flip(t) for t in transforms[1]] if len(transforms) == 2 else [False]
    if len(set(flips)) != len(flips):
        raise NotImplementedError('tta_transforms: each flip state at most once')
    return resizes, flips


def view_meta(h, w, rh, rw):
    """The metainfo mmcv Resize (keep_ratio) leaves on an (h, w) image resized to (rh, rw)."""
    return dict(img_shape=(rh, rw), scale_factor=(rw / w, rh / h), keep_ratio=True)


def draw_sample(rng, cfg, h, w):
    """One sample's random parameters, drawn from `rng` (numpy Generator) in the reference's order: the resize ratio,
    the crop boxes (offset_h then offset_w each), the flip, then PhotoMetricDistortion's draws.  All 11 crop boxes are
    drawn up front when cat_max_ratio < 1 (the reference draws a box only when the previous one fails), so the random
    stream differs from the reference's while every parameter has the reference's distribution."""
    lo, hi = cfg['ratio_range']
    ratio = rng.random() * (hi - lo) + lo
    scale = (int(cfg['scale'][0] * ratio), int(cfg['scale'][1] * ratio))
    rh, rw = rescale_size(h, w, scale)
    ch, cw = cfg['crop_size']
    mh, mw = max(rh - ch, 0), max(rw - cw, 0)
    n = NUM_CANDIDATES if cfg['cat_max_ratio'] < 1. else 1
    cands = []
    for _ in range(n):
        oy = int(rng.integers(0, mh + 1))
        ox = int(rng.integers(0, mw + 1))
        cands.append((oy, ox))
    flip = bool(rng.random() < cfg['prob'])
    p = dict(ratio=ratio, scale=scale, resized_hw=(rh, rw), candidates=cands, flip=flip,
             brightness=None, contrast=None, saturation=None, hue=None)
    d = cfg['brightness_delta']
    if rng.integers(2):
        p['brightness'] = float(rng.uniform(-d, d))
    p['contrast_mode'] = int(rng.integers(2))

    def contrast():
        if rng.integers(2):
            p['contrast'] = float(rng.uniform(*cfg['contrast_range']))
    if p['contrast_mode'] == 1:
        contrast()
    if rng.integers(2):
        p['saturation'] = float(rng.uniform(*cfg['saturation_range']))
    if rng.integers(2):
        p['hue'] = int(rng.integers(-cfg['hue_delta'], cfg['hue_delta']))
    if p['contrast_mode'] == 0:
        contrast()
    return p


def device_images(inputs):
    """The decoded uint8 [3, h, w] images of a batch (list or [N, 3, h, w] tensor) on the device; anything else raises
    NotImplementedError."""
    inputs = list(inputs) if isinstance(inputs, (list, tuple)) else list(inputs.unbind(0))
    if not inputs or any(not isinstance(t, torch.Tensor) or t.dtype != torch.uint8 or t.dim() != 3 or t.shape[0] != 3
                         for t in inputs):
        raise NotImplementedError('the device augmentation takes decoded uint8 [3, h, w] images')
    dev = next((t.device for t in inputs if t.is_cuda), None) or torch.device('cuda', torch.cuda.current_device())
    return [t.to(dev, non_blocking=True) for t in inputs]


@MODELS.register_module()
class DeviceAugSegDataPreProcessor(SegDataPreProcessor):
    """SegDataPreProcessor that also runs the config's training augmentations.

    `train_pipeline` holds the four dicts RandomResize, RandomCrop, RandomFlip, PhotoMetricDistortion verbatim from the
    config (in that order); `seed` seeds a numpy Generator (seed + rank under torch.distributed) that draws every random
    parameter on the host.  forward(data, training=True) takes the decoded uint8 [3, h, w] BGR images and their label
    maps, and returns the normalised, padded batch with the padded int64 labels, as SegDataPreProcessor does after the
    CPU pipeline, plus the metainfo those transforms leave (img_shape, scale_factor, flip, flip_direction, pad_shape,
    padding_size) and the drawn parameters under `aug_params` (with `crop_index`, the chosen box as a device tensor).
    The crop boxes are all drawn up front (see `draw_sample`): the random stream differs from the reference's lazy
    redraws, the distribution does not.

    `test_pipeline` (optional) holds the test pipeline's one Resize dict (keep_ratio=True, `scale` pair or float
    `scale_factor`), moved verbatim from the dataset: forward(data, training=False) then resizes the decoded uint8 images
    with cv2's INTER_LINEAR on the device, fused with the swap / normalisation / test_cfg padding (ops.view_resize), and
    sets img_shape, scale_factor and keep_ratio (ori_shape stays the decoded size, so predict resizes back to it).
    Without it, forward(data, training=False) is SegDataPreProcessor.forward."""

    def __init__(self, train_pipeline=None, seed=0, test_pipeline=None, **kwargs):
        super().__init__(**kwargs)
        self.aug = parse_pipeline(train_pipeline)
        self.test_resize = None
        if test_pipeline is not None:
            if not isinstance(test_pipeline, (list, tuple)) or len(test_pipeline) != 1:
                raise NotImplementedError('test_pipeline must be exactly [Resize(...)]')
            self.test_resize = parse_resize(test_pipeline[0])
        rank = 0
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            rank = torch.distributed.get_rank()
        self.rng = np.random.default_rng(int(seed) + rank)

    def draw(self, shapes):
        """Random parameters of a batch of (h, w) source images."""
        return [draw_sample(self.rng, self.aug, h, w) for h, w in shapes]

    def forward(self, data, training=False):
        decode_batch(data)
        if not training:
            if self.test_resize is None:
                return super().forward(data, False)
            return self._forward_test(data)
        samples = data.get('data_samples', None)
        assert samples is not None, 'During training, `data_samples` must be define.'
        inputs = device_images(data['inputs'])
        dev = inputs[0].device
        labels = [s['gt_sem_seg']['data'].to(dev, non_blocking=True) for s in samples]
        params = self.draw([tuple(t.shape[-2:]) for t in inputs])
        ch, cw = self.aug['crop_size']
        shapes = [(min(ch, p['resized_hw'][0]), min(cw, p['resized_hw'][1])) for p in params]
        Hp, Wp = self._padded_hw(shapes, self.size, self.size_divisor)
        N = len(inputs)
        out = torch.empty((N, 3, Hp, Wp), dtype=torch.float32, device=dev)
        lab_out = torch.empty((N, 1, Hp, Wp), dtype=torch.int64, device=dev)
        mean, std = self.mean_std() if self._enable_normalize else (None, None)
        crop_index = ops.train_augment(inputs, labels, params, (ch, cw), out, lab_out,
                                       cat_max_ratio=self.aug['cat_max_ratio'], ignore_index=self.aug['ignore_index'],
                                       swap_rb=self.channel_conversion, mean=mean, std=std, pad_val=self.pad_val,
                                       seg_pad_val=self.seg_pad_val)
        for i, (s, p) in enumerate(zip(samples, params)):
            (h, w), (rh, rw), (eh, ew) = inputs[i].shape[-2:], p['resized_hw'], shapes[i]
            s['gt_sem_seg']['data'] = lab_out[i]
            _meta(s).update(img_shape=(eh, ew), scale_factor=(rw / w, rh / h), flip=p['flip'],
                            flip_direction='horizontal' if p['flip'] else None, pad_shape=(Hp, Wp),
                            padding_size=(0, Wp - ew, 0, Hp - eh),
                            aug_params=dict(p, crop_index=crop_index[i] if crop_index is not None else 0))
        return dict(inputs=out, data_samples=samples)

    def _forward_test(self, data):
        """The test pipeline's Resize + SegDataPreProcessor.forward(training=False) in one launch per 64 images."""
        samples = data.get('data_samples', None)
        inputs = device_images(data['inputs'])
        src = [tuple(t.shape[-2:]) for t in inputs]
        sizes = [view_size(h, w, self.test_resize) for h, w in src]
        if self.test_cfg:
            Hp, Wp = self._padded_hw(sizes, self.test_cfg.get('size', None), self.test_cfg.get('size_divisor', None))
        else:
            assert all(sh == sizes[0] for sh in sizes), 'The image size in a batch should be the same.'
            Hp, Wp = sizes[0]
        out = torch.empty((len(inputs), 3, Hp, Wp), dtype=torch.float32, device=inputs[0].device)
        mean, std = self.mean_std() if self._enable_normalize else (None, None)
        ops.view_resize(inputs, sizes, out=out, swap_rb=self.channel_conversion, mean=mean, std=std,
                        pad_val=self.pad_val)
        if samples is not None:
            for s, (h, w), (rh, rw) in zip(samples, src, sizes):
                if not isinstance(s, dict):
                    continue
                m = _meta(s)
                m.update(view_meta(h, w, rh, rw))
                m.setdefault('ori_shape', (h, w))
                if self.test_cfg:
                    m.update(img_padding_size=(0, Wp - rw, 0, Hp - rh), pad_shape=(Hp, Wp))
        return dict(inputs=out, data_samples=samples)
