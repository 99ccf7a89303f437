"""`SegTTAModel` (MODELS): multi-scale + flip test-time augmentation (`tools/test.py --tta`).

Reference surface: ``mmseg/models/segmentors/seg_tta.py`` (merge_preds) over mmengine's ``BaseTTAModel.test_step``
(split the per-augmentation lists into one batch per view, run each through the module, merge per image).  Here every
view runs through the module's own `inference`; views whose preprocessed batches share a shape (the flip pair of every
scale ratio) run as ONE batch, and ONE ops.tta_merge post-processes (un-pad, un-flip, resize), soft-maxes, sums,
divides and arg-maxes all views per output pixel: the per-view probabilities never reach memory.

With `tta_transforms` (the Resize and RandomFlip lists of the config's TestTimeAug) the views are built on the device
from one decoded image per sample (ops.view_resize: cv2's INTER_LINEAR, the flip and SegDataPreProcessor in one pass),
so the dataloader decodes and packs each image once instead of resizing, flipping and uploading 12 views.
"""
import torch
import torch.nn as nn

from .augment import device_images, parse_tta_transforms, view_meta, view_size
from .png_feed import decode_batch
from .registry import MODELS
from .segmentor import SegDataPreProcessor, _meta, _view_geometry
from . import ops


def split_views(data):
    """BaseTTAModel.test_step's split: a dict of per-augmentation lists -> one dict per view; a list / tuple of such
    lists -> one list per view; augmentation order."""
    if isinstance(data, dict):
        num_augs = len(data[next(iter(data))])
        return [{key: value[idx] for key, value in data.items()} for idx in range(num_augs)]
    if isinstance(data, (tuple, list)):
        num_augs = len(data[0])
        return [[_data[idx] for _data in data] for idx in range(num_augs)]
    raise TypeError(f'data given by dataLoader should be a dict, list or tuple, but got {type(data)}')


def _sample_meta(s):
    return s.get('metainfo', s) if isinstance(s, dict) else {}


def view_descriptor(meta, view_hw):
    """((padding l, r, t, b), flip or None, ori_shape) of one image of one view: what postprocess_result undoes and the
    size it resizes to (the cropped extent when the metainfo carries no ori_shape)."""
    padding, flip = _view_geometry(meta)
    padding = tuple(int(v) for v in padding)
    ori = meta.get('ori_shape')
    if ori is None:
        ori = (view_hw[0] - padding[2] - padding[3], view_hw[1] - padding[0] - padding[1])
    return padding, flip, tuple(int(v) for v in ori[:2])


def _with_meta(sample, meta):
    """a shallow copy of a data sample with `meta` merged into its metainfo"""
    r = dict(sample) if isinstance(sample, dict) else {}
    if 'metainfo' in r or 'gt_sem_seg' in r:
        r['metainfo'] = dict(r.get('metainfo', {}), **meta)
    else:
        r.update(meta)
    return r


@MODELS.register_module()
class SegTTAModel(nn.Module):
    """SegTTAModel(module, data_preprocessor=None, tta_transforms=None).  `module` is an EncoderDecoder or its config
    dict.  `data_preprocessor` is accepted for config compatibility; as in mmengine, each view goes through the module's.

    `tta_transforms` takes the first two lists of the config's TestTimeAug.transforms verbatim:
    [[Resize(scale_factor=r, keep_ratio=True) ...], [RandomFlip(prob=0., ...), RandomFlip(prob=1., ...)]] (the flip
    list is optional; any other transform or argument raises NotImplementedError).  test_step then takes an ordinary
    single-view batch of decoded uint8 [3, h, w] images of one size and builds the views itself, in TestTimeAug's order
    (ratio-major), with the metainfo mmcv's Resize / RandomFlip and the module's SegDataPreProcessor would give them."""

    MAX_TTA_BATCH = 64            # images per module.inference call; larger same-shape view groups are chunked

    def __init__(self, module, data_preprocessor=None, tta_transforms=None):
        super().__init__()
        self.module = MODELS.build(module) if isinstance(module, dict) else module
        self.tta = parse_tta_transforms(tta_transforms) if tta_transforms is not None else None

    # -- merge -------------------------------------------------------------------------------
    def _mode(self):
        """(mode, threshold) of ops.tta_merge: softmax when out_channels > 1, else sigmoid > threshold."""
        m = self.module
        if m.out_channels > 1:
            return 0, 0.3
        return 1, float(getattr(m.decode_head, 'threshold', None) or 0.3)

    def _view_logits(self, inputs):
        """module.inference of every view: views of one shape run as one concatenated batch (at most MAX_TTA_BATCH
        images per call).  Returns one [N,K,H,W] logits tensor per view (slices of the group's output)."""
        groups = {}
        for v, x in enumerate(inputs):
            groups.setdefault(tuple(x.shape), []).append(v)
        out = [None] * len(inputs)
        for idx in groups.values():
            n = inputs[idx[0]].shape[0]
            x = torch.cat([inputs[v] for v in idx], 0) if len(idx) > 1 else inputs[idx[0]]
            lg = self._inference(x)
            for j, v in enumerate(idx):
                out[v] = lg[j * n:(j + 1) * n]
        return out

    def _inference(self, x):
        """module.inference of one batch, at most MAX_TTA_BATCH images per call"""
        cap = max(1, int(self.MAX_TTA_BATCH))
        parts = [self.module.inference(x[i:i + cap]) for i in range(0, x.shape[0], cap)]
        return torch.cat(parts, 0) if len(parts) > 1 else parts[0]

    def view_plan(self, h, w):
        """The metainfo of every view of an (h, w) image in TestTimeAug's order (itertools.product of the Resize and
        RandomFlip lists: ratio-major): img_shape, scale_factor, keep_ratio, flip, flip_direction."""
        resizes, flips = self.tta
        plan = []
        for rs in resizes:
            rh, rw = view_size(h, w, rs)
            plan += [dict(view_meta(h, w, rh, rw), flip=f, flip_direction='horizontal' if f else None) for f in flips]
        return plan

    def _device_views(self, images, metas):
        """The TestTimeAug views of decoded uint8 images of one size, built on the device ratio by ratio: per ratio ONE
        ops.view_resize writes the flip pair into the [F*N, 3, Hp, Wp] batch module.inference takes, and only the
        logits outlive the ratio.  Returns (per view logits [N,K,H,W], per view the N images' metainfo)."""
        pp = self.module.data_preprocessor or SegDataPreProcessor()
        flips = self.tta[1]
        n, (h, w) = len(images), images[0].shape[-2:]
        mean, std = pp.mean_std() if pp._enable_normalize else (None, None)
        ori = [tuple(m['ori_shape'][:2]) if m.get('ori_shape') is not None else (h, w) for m in metas]
        plan = self.view_plan(h, w)
        logits, view_metas = [], []
        for r in range(0, len(plan), len(flips)):
            rh, rw = plan[r]['img_shape']
            pad = {}
            if pp.test_cfg:
                Hp, Wp = pp._padded_hw([(rh, rw)], pp.test_cfg.get('size', None), pp.test_cfg.get('size_divisor', None))
                pad = dict(img_padding_size=(0, Wp - rw, 0, Hp - rh), pad_shape=(Hp, Wp))
            else:
                Hp, Wp = rh, rw
            x = torch.empty((len(flips) * n, 3, Hp, Wp), dtype=torch.float32, device=images[0].device)
            part = {f: x[j * n:(j + 1) * n] for j, f in enumerate(flips)}
            ops.view_resize(images, (rh, rw), out=part.get(False), out_flip=part.get(True),
                            swap_rb=pp.channel_conversion, mean=mean, std=std, pad_val=pp.pad_val)
            lg = self._inference(x)
            del x, part
            for j in range(len(flips)):
                logits.append(lg[j * n:(j + 1) * n])
                view_metas.append([dict(plan[r + j], ori_shape=o, **pad) for o in ori])
        return logits, view_metas

    @staticmethod
    def _images(inputs):
        images = device_images(inputs)
        if len({tuple(t.shape) for t in images}) != 1:
            raise NotImplementedError('the device augmentation takes decoded uint8 [3, h, w] images of one size')
        return images

    def _merge(self, logits, metas, pred=None, pred_dtype=torch.int64):
        """ops.tta_merge of per-view logits [N,K,H,W] with per-view, per-image metainfo: one launch for the batch
        when every image shares its views' geometry (the fixed-size case), else one per image."""
        n = logits[0].shape[0]
        assert all(lg.shape[0] == n for lg in logits), 'every view must hold the same images'
        desc = [[view_descriptor(metas[v][i], lg.shape[-2:]) for i in range(n)] for v, lg in enumerate(logits)]
        for i in range(n):
            assert len({desc[v][i][2] for v in range(len(logits))}) == 1, 'the views of an image differ in ori_shape'
        uniform = all(len(set(d)) == 1 for d in desc)
        mode, thr = self._mode()
        chunks = [range(n)] if uniform else [range(i, i + 1) for i in range(n)]
        preds = []
        for ch in chunks:
            i0, i1 = ch[0], ch[-1] + 1
            views = [(lg[i0:i1], desc[v][i0][0], desc[v][i0][1]) for v, lg in enumerate(logits)]
            p, _ = ops.tta_merge(views, desc[0][i0][2], self.module.align_corners, mode, thr, pred_dtype,
                                 pred=pred[i0:i1] if pred is not None else None)
            preds.append(p)
        return preds[0] if len(preds) == 1 else torch.cat(preds, 0)

    @staticmethod
    def _result(first, last, pred, seg_logits):
        """seg_tta.py merge_preds: the LAST view's sample with pred_sem_seg replaced, gt_sem_seg and img_path from the
        first view's."""
        r = dict(last) if isinstance(last, dict) else {}
        if 'metainfo' in r:
            r['metainfo'] = dict(r['metainfo'])
        r['seg_logits'] = {'data': seg_logits}
        r['pred_sem_seg'] = {'data': pred}
        if isinstance(first, dict) and 'gt_sem_seg' in first:
            r['gt_sem_seg'] = first['gt_sem_seg']
        fm = _sample_meta(first)
        if 'img_path' in fm:
            _meta(r)['img_path'] = fm['img_path']
        return r

    @staticmethod
    def _squeeze(pred, mode):
        """argmax(dim=0) gives [H, W]; the sigmoid branch's (logits > threshold).to(logits).squeeze(1) keeps [K, H, W]"""
        return pred if mode == 0 else pred.squeeze(1)

    # -- reference API ---------------------------------------------------------------------------
    @torch.no_grad()
    def test_step(self, data):
        """BaseTTAModel.test_step + SegTTAModel.merge_preds: one list per augmentation in `data` (dict or list form);
        returns one reference-shaped result dict per image.  With `tta_transforms`, `data` is one ordinary batch
        (inputs, data_samples) of decoded images and the views are built on the device."""
        if self.tta is not None:
            return self._test_step_device_views(data)
        m = self.module
        pp = m.data_preprocessor or SegDataPreProcessor()
        inputs, samples = [], []
        for view in split_views(data):
            if isinstance(view, (list, tuple)):
                view = dict(zip(('inputs', 'data_samples'), view))
            out = pp(view, False)
            inputs.append(out['inputs'])
            samples.append(out.get('data_samples'))
        n = inputs[0].shape[0]
        samples = [s if s is not None else [{} for _ in range(n)] for s in samples]
        metas = [[_sample_meta(s) for s in ss] for ss in samples]
        logits = self._view_logits(inputs)
        pred = self._merge(logits, metas)
        mode, thr = self._mode()
        res = []
        for i in range(n):
            pad, flip, ori = view_descriptor(metas[-1][i], logits[-1].shape[-2:])
            _, lg = ops.postprocess(logits[-1][i], padding=pad, flip=flip, ori_shape=ori,
                                    align_corners=m.align_corners, threshold=thr)
            res.append(self._result(samples[0][i], samples[-1][i], self._squeeze(pred[i], mode), lg))
        return res

    def _test_step_device_views(self, data):
        if isinstance(data, (list, tuple)):
            data = dict(zip(('inputs', 'data_samples'), data))
        decode_batch(data)
        images = self._images(data['inputs'])
        n = len(images)
        samples = data.get('data_samples') or [{} for _ in range(n)]
        metas = [_sample_meta(s) for s in samples]
        logits, view_metas = self._device_views(images, metas)
        pred = self._merge(logits, view_metas)
        mode, thr = self._mode()
        res = []
        for i in range(n):
            pad, flip, ori = view_descriptor(view_metas[-1][i], logits[-1].shape[-2:])
            _, lg = ops.postprocess(logits[-1][i], padding=pad, flip=flip, ori_shape=ori,
                                    align_corners=self.module.align_corners, threshold=thr)
            last = _with_meta(samples[i], view_metas[-1][i])
            res.append(self._result(samples[i], last, self._squeeze(pred[i], mode), lg))
        return res

    val_step = test_step

    @torch.no_grad()
    def merge_preds(self, data_samples_list):
        """seg_tta.py merge_preds on already post-processed samples: per image a list of view dicts carrying
        seg_logits.data [K,H,W].  The same kernel with identity geometry (one launch per image)."""
        mode, _ = self._mode()
        res = []
        for views in data_samples_list:
            lgs = [s['seg_logits']['data'] for s in views]
            if lgs[0].shape[0] == 1:
                # postprocess_result already applied the one-class sigmoid, which the kernel's view sampling repeats
                raise NotImplementedError('merge_preds of one-class seg_logits: use test_step')
            pred = self._merge([lg[None] for lg in lgs], [[{}] for _ in lgs])
            res.append(self._result(views[0], views[-1], self._squeeze(pred[0], mode), lgs[-1]))
        return res

    @torch.no_grad()
    def predict_labels(self, views, metas, pred=None, pred_dtype=torch.uint8):
        """Labels-only fast path (for IoUMetric.process_batch): views = one input batch [N,3,H,W] per augmentation
        (whatever module.inference takes: normalised float, or raw uint8 on the fused engine), metas = per view the
        N images' metainfo dicts (padding / flip / ori_shape).  Returns labels [N, oh, ow] (written into `pred`)."""
        if self._mode()[0] != 0:
            raise ValueError('predict_labels is the argmax path (out_channels > 1)')
        metas = [[_sample_meta(s) for s in ss] for ss in metas]
        return self._merge(self._view_logits(list(views)), metas, pred=pred, pred_dtype=pred_dtype)

    @torch.no_grad()
    def predict_image_labels(self, images, metas=None, pred=None, pred_dtype=torch.uint8):
        """Labels-only counterpart of the `tta_transforms` test_step (for IoUMetric.process_batch): decoded uint8
        images [N,3,h,w] (or a list) of one size, optional per-image metainfo (ori_shape).  The views are built on the
        device.  Returns labels [N, oh, ow] (written into `pred`)."""
        if self.tta is None:
            raise ValueError('predict_image_labels builds the views from tta_transforms; none were given')
        if self._mode()[0] != 0:
            raise ValueError('predict_image_labels is the argmax path (out_channels > 1)')
        images = self._images(images)
        metas = [_sample_meta(s) for s in metas] if metas is not None else [{} for _ in images]
        logits, view_metas = self._device_views(images, metas)
        return self._merge(logits, view_metas, pred=pred, pred_dtype=pred_dtype)
