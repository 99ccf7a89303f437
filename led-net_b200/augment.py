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
    redraws, the distribution does not.  forward(data, training=False) is SegDataPreProcessor.forward."""

    def __init__(self, train_pipeline=None, seed=0, **kwargs):
        super().__init__(**kwargs)
        self.aug = parse_pipeline(train_pipeline)
        rank = 0
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            rank = torch.distributed.get_rank()
        self.rng = np.random.default_rng(int(seed) + rank)

    def draw(self, shapes):
        """Random parameters of a batch of (h, w) source images."""
        return [draw_sample(self.rng, self.aug, h, w) for h, w in shapes]

    def forward(self, data, training=False):
        if not training:
            return super().forward(data, False)
        inputs = data['inputs']
        samples = data.get('data_samples', None)
        assert samples is not None, 'During training, `data_samples` must be define.'
        inputs = list(inputs) if isinstance(inputs, (list, tuple)) else list(inputs.unbind(0))
        dev = next((t.device for t in inputs if t.is_cuda), None) or torch.device('cuda', torch.cuda.current_device())
        inputs = [t.to(dev, non_blocking=True) for t in inputs]
        if any(t.dtype != torch.uint8 or t.dim() != 3 or t.shape[0] != 3 for t in inputs):
            raise NotImplementedError('the device augmentation takes decoded uint8 [3, h, w] images')
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
