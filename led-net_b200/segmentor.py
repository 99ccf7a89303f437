"""`EncoderDecoder` and `SegDataPreProcessor` (MODELS) - the callers either side of the hot path.

Reference surface: ``mmseg/models/segmentors/encoder_decoder.py:117-132, 187-345``,
``mmseg/models/segmentors/base.py:127-200`` and ``mmseg/models/data_preprocessor.py:98-151``.
`predict_labels` is the fused fast path (one C-ABI call: image batch -> label map, full-resolution
logits never materialised); `predict` keeps the reference's return shape (seg_logits + pred_sem_seg
per image) and therefore does materialise the logits.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .engine import Engine, MEAN, STD
from .registry import MODELS
from . import ops
from .png_feed import decode_batch


def _meta(sample):
    """Where a dict-style data sample keeps its metainfo (SegDataSample.metainfo)."""
    return sample.setdefault('metainfo', {}) if 'metainfo' in sample or 'gt_sem_seg' in sample else sample


def _view_geometry(meta):
    """(padding (left, right, top, bottom), flip direction or None) that postprocess_result undoes (base.py:163-176)."""
    padding = meta.get('img_padding_size', meta.get('padding_size', [0] * 4))
    flip = None
    if meta.get('flip', None):
        flip = meta.get('flip_direction', None)
        assert flip in ['horizontal', 'vertical']
    return padding, flip


@MODELS.register_module()
class SegDataPreProcessor(nn.Module):
    """mmseg/models/data_preprocessor.py:98-151 on the device: per sample ONE kernel (ops.stack_pad) does the BGR<->RGB
    swap, the float conversion, (x - mean) / std, the right / bottom padding of `stack_batch` (mmseg/utils/misc.py:30-128:
    to `size`, or to the batch maximum rounded up to `size_divisor`; `pad_val` after the normalisation) and pads the label
    map with `seg_pad_val`.  mean / std default to None = no normalisation, as in the reference.  On the fused inference
    path (raw uint8 into `predict_labels`) the same mean / std / swap are the stem convolution's prologue instead."""

    def __init__(self, mean=None, std=None, size=None, size_divisor=None, pad_val=0, seg_pad_val=255,
                 bgr_to_rgb=False, rgb_to_bgr=False, batch_augments=None, test_cfg=None):
        super().__init__()
        assert not (bgr_to_rgb and rgb_to_bgr), '`bgr2rgb` and `rgb2bgr` cannot be set to True at the same time'
        assert (mean is None) == (std is None), 'mean and std should be both None or tuple'
        if batch_augments is not None:
            raise NotImplementedError('batch_augments are outside the LED-Net path (the config has none)')
        self.channel_conversion = bgr_to_rgb or rgb_to_bgr
        self.size, self.size_divisor, self.pad_val, self.seg_pad_val = size, size_divisor, pad_val, seg_pad_val
        self.test_cfg = test_cfg
        self._enable_normalize = mean is not None
        if self._enable_normalize:
            self.register_buffer('mean', torch.tensor(mean, dtype=torch.float32).view(-1, 1, 1), False)
            self.register_buffer('std', torch.tensor(std, dtype=torch.float32).view(-1, 1, 1), False)
        else:
            self.mean = self.std = None

    def mean_std(self):
        """(mean, std) tuples for the engine's fused prologue (identity when normalisation is off)."""
        if not self._enable_normalize:
            return (0., 0., 0.), (1., 1., 1.)
        return tuple(self.mean.flatten().tolist()), tuple(self.std.flatten().tolist())

    @staticmethod
    def _padded_hw(shapes, size, size_divisor):
        """stack_batch's target shape; exactly one of size / size_divisor (misc.py:64-66)."""
        assert (size is not None) ^ (size_divisor is not None), 'only one of size and size_divisor should be valid'
        if size is not None:
            hw = {(h + max(size[-2] - h, 0), w + max(size[-1] - w, 0)) for h, w in shapes}
            assert len(hw) == 1, f'samples padded to `size` still differ in shape: {sorted(hw)}'   # torch.stack would fail
            return hw.pop()
        mh, mw = max(h for h, _ in shapes), max(w for _, w in shapes)
        if size_divisor > 1:
            mh, mw = -(-mh // size_divisor) * size_divisor, -(-mw // size_divisor) * size_divisor
        return mh, mw

    def forward(self, data, training=False):
        decode_batch(data)
        inputs = data['inputs']
        samples = data.get('data_samples', None)
        inputs = list(inputs) if isinstance(inputs, (list, tuple)) else list(inputs.unbind(0))
        dev = next((t.device for t in inputs if t.is_cuda), None) or torch.device('cuda', torch.cuda.current_device())
        inputs = [t.to(dev, non_blocking=True) for t in inputs]                     # BaseDataPreprocessor.cast_data
        assert all(t.dim() == 3 and t.shape[0] == inputs[0].shape[0] for t in inputs)
        if inputs[0].shape[0] != 3:
            raise NotImplementedError('the device preprocessor handles 3-channel images (the LED-Net pipeline)')
        shapes = [tuple(t.shape[-2:]) for t in inputs]
        pad_labels = False
        if training:
            assert samples is not None, 'During training, `data_samples` must be define.'
            Hp, Wp = self._padded_hw(shapes, self.size, self.size_divisor)
            pad_labels = True
        else:
            assert all(sh == shapes[0] for sh in shapes), 'The image size in a batch should be the same.'
            if self.test_cfg:
                Hp, Wp = self._padded_hw(shapes, self.test_cfg.get('size', None), self.test_cfg.get('size_divisor', None))
            else:
                Hp, Wp = shapes[0]
        out = torch.empty((len(inputs), 3, Hp, Wp), dtype=torch.float32, device=dev)
        mean, std = self.mean_std() if self._enable_normalize else (None, None)
        for i, t in enumerate(inputs):
            h, w = shapes[i]
            padding = (0, Wp - w, 0, Hp - h)                                        # (left, right, top, bottom)
            s = samples[i] if samples is not None else None
            lab = lab_out = None
            if pad_labels and isinstance(s, dict) and 'gt_sem_seg' in s:
                lab = s['gt_sem_seg']['data'].to(dev)
                lab_out = torch.empty((1, Hp, Wp), dtype=torch.int64, device=dev)
            ops.stack_pad(t, out[i], swap_rb=self.channel_conversion, mean=mean, std=std, pad_val=self.pad_val,
                          label=lab, label_out=lab_out[0] if lab_out is not None else None, seg_pad_val=self.seg_pad_val)
            if isinstance(s, dict):
                if lab_out is not None:
                    s['gt_sem_seg']['data'] = lab_out
                if training:
                    _meta(s).update(img_shape=(h, w), pad_shape=(Hp, Wp) if lab_out is not None else None,
                                    padding_size=padding)
                elif self.test_cfg:
                    _meta(s).update(img_padding_size=padding, pad_shape=(Hp, Wp))
        return dict(inputs=out, data_samples=samples)


@MODELS.register_module()
class EncoderDecoder(nn.Module):

    def __init__(self, backbone, decode_head, neck=None, auxiliary_head=None, train_cfg=None,
                 test_cfg=None, data_preprocessor=None, pretrained=None, init_cfg=None,
                 compute_dtype='bf16'):
        super().__init__()
        assert neck is None and auxiliary_head is None, 'the LED-Net config has neither'
        self.backbone = MODELS.build(backbone) if isinstance(backbone, dict) else backbone
        self.decode_head = MODELS.build(decode_head) if isinstance(decode_head, dict) else decode_head
        self.data_preprocessor = (MODELS.build(data_preprocessor) if isinstance(data_preprocessor, dict)
                                  else data_preprocessor)
        self.align_corners = self.decode_head.align_corners       # encoder_decoder.py:103-105
        self.num_classes = self.decode_head.num_classes
        self.out_channels = self.decode_head.out_channels
        self.train_cfg, self.test_cfg = train_cfg, dict(test_cfg or dict(mode='whole'))
        self.compute_dtype = compute_dtype
        self._engine = None
        for part in (self.backbone, self.decode_head):          # stand-alone module engines (mode='tensor') follow
            if hasattr(part, 'set_compute_dtype'):
                part.set_compute_dtype(compute_dtype)
        self.register_load_state_dict_post_hook(lambda m, keys: m.reset_engine())

    # -- engine ---------------------------------------------------------------------------
    def reset_engine(self):
        self._engine = None

    def set_compute_dtype(self, dtype):
        if dtype != self.compute_dtype:
            self.compute_dtype, self._engine = dtype, None
        for part in (self.backbone, self.decode_head):
            if hasattr(part, 'set_compute_dtype'):
                part.set_compute_dtype(dtype)
        return self

    @property
    def _composed(self):
        """layer-by-layer backbone (LEDNet(variant='led')) instead of the fused R0 engine plan"""
        return getattr(self.backbone, 'composed', False)

    def _float_inputs(self, inputs):
        """raw uint8 batches go through the device preprocessor when the backbone is not the fused engine"""
        if inputs.dtype != torch.uint8:
            return inputs
        pp = self.data_preprocessor or SegDataPreProcessor()
        return pp(dict(inputs=inputs if inputs.shape[1] == 3 else inputs.permute(0, 3, 1, 2)))['inputs']

    def engine(self):
        if self._composed:
            raise RuntimeError("LEDNet(variant='led') runs layer by layer; there is no fused engine plan for it")
        if self._engine is None:
            state = {'backbone.' + k: v for k, v in self.backbone.state_dict().items()}
            state.update(self.decode_head.engine_state() if hasattr(self.decode_head, 'engine_state') else
                         {'decode_head.' + k: v for k, v in self.decode_head.state_dict().items()})
            pp = self.data_preprocessor
            kw = {}
            if pp is not None:
                mean, std = pp.mean_std()
                kw = dict(mean=mean, std=std, bgr_to_rgb=pp.channel_conversion)
            self._engine = Engine(state, self.num_classes, self.backbone.channels,
                                  self.backbone.ppm_channels, self.decode_head.channels,
                                  dtype=self.compute_dtype, **kw)
        return self._engine

    # -- reference API --------------------------------------------------------------------
    def extract_feat(self, inputs):
        if self.training:
            return self.backbone(inputs)            # train-mode tape over csrc/train.cu
        if self._composed:
            return self.backbone(self._float_inputs(inputs))
        return self.engine().backbone_forward(inputs)

    def train(self, mode=True):
        if mode:
            self.reset_engine()                     # folded eval weights go stale once training resumes
        return super().train(mode)

    def loss(self, inputs, data_samples):
        """encoder_decoder.py:161-185: decode-head losses under the 'decode.' prefix."""
        x = self.extract_feat(inputs)
        out = self.decode_head.loss(x, data_samples, self.train_cfg)
        return {'decode.' + k: v for k, v in out.items()}

    @staticmethod
    def parse_losses(losses):
        """mmengine BaseModel.parse_losses: total = sum of every entry whose key contains 'loss'."""
        log = {k: (v.mean() if isinstance(v, torch.Tensor) else sum(x.mean() for x in v))
               for k, v in losses.items()}
        total = sum(v for k, v in log.items() if 'loss' in k)
        log['loss'] = total
        return total, log

    def train_step(self, data, optimizer):
        """mmengine BaseModel.train_step: preprocess -> loss -> backward -> optimiser step.
        `optimizer` is a lednet_b200.optim.FlatSGD (or any object with zero_grad()/step())."""
        if self.data_preprocessor is not None and isinstance(data, dict) and 'inputs' in data:
            data = self.data_preprocessor(data, training=True)
        total, log = self.parse_losses(self.loss(data['inputs'], data['data_samples']))
        optimizer.zero_grad()
        total.backward()
        optimizer.step()
        return log

    def test_step(self, data):
        """mmengine BaseModel.test_step: data_preprocessor(data, False), then forward(mode='predict').  `data` is a dict
        (inputs, data_samples) or an (inputs, data_samples) sequence."""
        if isinstance(data, (list, tuple)):
            data = dict(zip(('inputs', 'data_samples'), data))
        data = (self.data_preprocessor or SegDataPreProcessor())(data, False)
        return self.predict(data['inputs'], data.get('data_samples'))

    val_step = test_step                            # mmengine's val_step is the same call

    def encode_decode(self, inputs, batch_img_metas=None):
        """encoder_decoder.py:124-132: full-resolution logits [N,K,H,W] (fused, one call)."""
        if self._composed:
            return self.decode_head.engine().head_infer(*self.extract_feat(inputs), want_logits=True)[1]
        return self.engine().forward_infer(inputs, want_logits=True)[1]

    def whole_inference(self, inputs, batch_img_metas=None):
        return self.encode_decode(inputs, batch_img_metas)

    def _slide_windows(self, h_img, w_img):
        """Window origins in the reference's grid order (encoder_decoder.py:262-278)."""
        h_stride, w_stride = self.test_cfg['stride']
        h_crop, w_crop = self.test_cfg['crop_size']
        h_grids = max(h_img - h_crop + h_stride - 1, 0) // h_stride + 1
        w_grids = max(w_img - w_crop + w_stride - 1, 0) // w_stride + 1
        wins = []
        for hi in range(h_grids):
            for wi in range(w_grids):
                y1, x1 = hi * h_stride, wi * w_stride
                y2, x2 = min(y1 + h_crop, h_img), min(x1 + w_crop, w_img)
                wins.append((max(y2 - h_crop, 0), max(x2 - w_crop, 0), y2, x2))
        return wins

    MAX_SLIDE_BATCH = 64          # crop images per engine call on the batched path

    def slide_inference(self, inputs, batch_img_metas=None, want_pred=False):
        """encoder_decoder.py:241-292.  The crop windows are independent, so they run as ONE batch of the fused engine
        (window g of image n at batch index g*n_img + n) and ops.slide_merge sums, divides (and optionally arg-maxes)
        per output pixel in the reference's accumulation order - no full-size `preds` read-modify-write per crop.
        More than MAX_SLIDE_BATCH crop images, or crops whose logits are not crop-sized (odd crop sizes round up),
        take the sequential slide_accumulate / slide_finalize kernels instead."""
        n, _, h_img, w_img = inputs.shape
        wins = self._slide_windows(h_img, w_img)
        hc, wc = wins[0][2] - wins[0][0], wins[0][3] - wins[0][1]
        even = hc % 2 == 0 and wc % 2 == 0
        if even and len(wins) * n <= self.MAX_SLIDE_BATCH:
            crops = torch.cat([inputs[:, :, y1:y2, x1:x2] for (y1, x1, y2, x2) in wins], 0).contiguous()
            logit = self.encode_decode(crops)
            out, pred = ops.slide_merge(logit, [(y1, x1) for (y1, x1, _, _) in wins], n, (h_img, w_img),
                                        want_logits=True, want_pred=want_pred)
            return (out, pred) if want_pred else out
        k = self.num_classes                       # channels of the fused logits (decode_head.py:362-379 broadcasts to K)
        preds = torch.zeros((n, k, h_img, w_img), dtype=torch.float32, device=inputs.device)
        count = torch.zeros((n, 1, h_img, w_img), dtype=torch.float32, device=inputs.device)
        for (y1, x1, y2, x2) in wins:
            logit = self.encode_decode(inputs[:, :, y1:y2, x1:x2].contiguous())
            ops.slide_accumulate(preds, count, logit, y1, x1)
        assert (count == 0).sum() == 0
        out, pred = ops.slide_finalize(preds, count, want_pred=want_pred)
        return (out, pred) if want_pred else out

    def inference(self, inputs, batch_img_metas=None):
        mode = self.test_cfg.get('mode', 'whole')
        assert mode in ['slide', 'whole'], \
            f'Only "slide" or "whole" test mode are supported, but got {mode}.'
        return self.slide_inference(inputs, batch_img_metas) if mode == 'slide' \
            else self.whole_inference(inputs, batch_img_metas)

    def postprocess_result(self, seg_logits, data_samples=None):
        """base.py:153-198: per image remove the padding, undo the test-time flip, resize to `ori_shape`, argmax
        (or sigmoid > threshold for one class) - one kernel per image (ops.postprocess).  `data_samples` are dicts
        whose 'metainfo' (or the dict itself) carries img_padding_size / padding_size, flip, flip_direction, ori_shape."""
        out = []
        for i in range(seg_logits.shape[0]):
            meta = {}
            if data_samples is not None and isinstance(data_samples[i], dict):
                meta = data_samples[i].get('metainfo', data_samples[i])
            padding, flip = _view_geometry(meta)
            pred, lg = ops.postprocess(seg_logits[i], padding=padding, flip=flip, ori_shape=meta.get('ori_shape'),
                                       align_corners=self.align_corners,
                                       threshold=getattr(self.decode_head, 'threshold', None) or 0.3)
            out.append({'seg_logits': {'data': lg}, 'pred_sem_seg': {'data': pred}})
        return out

    def predict(self, inputs, data_samples=None):
        """encoder_decoder.py:187-222: list of {'seg_logits','pred_sem_seg'} per image."""
        def _plain(s):                       # no crop / flip / resize requested for this sample
            m = s.get('metainfo', s) if isinstance(s, dict) else {}
            return not (m.get('flip') or m.get('ori_shape') is not None and tuple(m['ori_shape']) != tuple(inputs.shape[-2:])
                        or any(m.get('img_padding_size', m.get('padding_size', [0] * 4))))
        if (not self._composed and self.test_cfg.get('mode', 'whole') == 'whole'
                and (data_samples is None or all(_plain(s) for s in data_samples))):
            pred, logits = self.engine().forward_infer(inputs, pred_dtype=torch.int64, want_logits=True)
            res = [{'seg_logits': {'data': logits[i]}, 'pred_sem_seg': {'data': pred[i:i + 1]}}
                   for i in range(pred.shape[0])]
        else:
            res = self.postprocess_result(self.inference(inputs), data_samples)
        if data_samples is not None:
            for r, s in zip(res, data_samples):
                if isinstance(s, dict):
                    r.update({k: v for k, v in s.items() if k not in r})
        return res

    @torch.no_grad()
    def predict_labels(self, inputs, pred=None, pred_dtype=torch.uint8):
        """Fused fast path: [N,3,H,W] float (normalised) or uint8 (raw BGR) -> labels [N,H,W]."""
        if self._composed:       # composed trunk -> head engine on its NHWC features (fused ladder + argmax)
            return self.decode_head.engine().head_infer(*self.extract_feat(inputs), pred=pred, pred_dtype=pred_dtype)
        return self.engine().forward_infer(inputs, pred=pred, pred_dtype=pred_dtype)

    def forward(self, inputs, data_samples=None, mode='tensor'):
        if mode == 'predict':
            return self.predict(inputs, data_samples)
        if mode == 'tensor':
            return self.decode_head.forward(self.extract_feat(inputs))
        if mode == 'loss':
            return self.loss(inputs, data_samples)
        raise RuntimeError(f'Invalid mode "{mode}". Only supports loss, predict and tensor mode')
