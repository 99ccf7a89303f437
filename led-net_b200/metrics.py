"""`IoUMetric` (METRICS) - reference surface of ``mmseg/evaluation/metrics/iou_metric.py:18-295``.

Device work is one confusion-matrix kernel launch per image (csrc/metrics.cu) instead of two
boolean gathers, three float32 `histc` calls and three device->host syncs; nothing leaves the GPU
until `compute_metrics`.  With `output_dir`, the predictions are written as PNG files encoded on the device
(csrc/png.cu, one launch sequence per shape of a `process` call); only the files come back to the host.  Across ranks the (K+1) x K int64 matrix is summed with ONE NCCL
all-reduce (2.9 KB at K=19) instead of mmengine's pickled `collect_results` object gather.
"""
import logging
import os
from collections import OrderedDict

import numpy as np
import torch

from . import ops
from .registry import METRICS


def _is_main_process():
    d = torch.distributed
    return not (d.is_available() and d.is_initialized()) or d.get_rank() == 0


def _sample_meta(sample, key, default=None):
    """`key` of a data sample or of its `metainfo` (a SegDataSample or its dict form)."""
    v = sample.get(key, None)
    if v is None:
        meta = sample.get('metainfo', None)
        v = meta.get(key, None) if meta is not None else None
    return default if v is None else v


def _areas_from_cm(cm):
    """[K+1,K] int64 -> (intersect, union, pred_label, label) int64 [K] (rows GT, cols pred)."""
    k = cm.shape[1]
    inter = torch.diagonal(cm[:k])
    area_l = cm[:k].sum(1)
    area_p = cm.sum(0)
    return inter, area_p + area_l - inter, area_p, area_l


@METRICS.register_module()
class IoUMetric:

    def __init__(self, ignore_index=255, iou_metrics=('mIoU',), nan_to_num=None, beta=1,
                 collect_device='cpu', output_dir=None, format_only=False, prefix=None, **kwargs):
        self.ignore_index = ignore_index
        self.metrics = list(iou_metrics) if not isinstance(iou_metrics, str) else [iou_metrics]
        self.nan_to_num, self.beta = nan_to_num, beta
        self.collect_device, self.output_dir, self.format_only, self.prefix = \
            collect_device, output_dir, format_only, prefix
        if output_dir and _is_main_process():
            os.makedirs(output_dir, exist_ok=True)
        self.results = []
        self.dataset_meta = None
        self._cm = None
        self._n_samples = 0          # images this rank has processed since the last evaluate()
        self._last = None            # (pred, label, K) of the most recent image: see evaluate(size)

    # -- reference API --------------------------------------------------------------------
    def process(self, data_batch, data_samples):
        """iou_metric.py:67-100: one entry per image in self.results (here: its int64 matrix).  With `format_only`
        no matrix is computed and `gt_sem_seg` may be missing.  With `output_dir`, each prediction is written to
        `{splitext(basename(img_path))[0]}.png`, plus one when the sample's `reduce_zero_label` is set."""
        preds = []
        for s in data_samples:
            pred = s['pred_sem_seg']['data'].squeeze()
            preds.append(pred)
            if not self.format_only:
                num_classes = len(self.dataset_meta['classes'])
                label = s['gt_sem_seg']['data'].squeeze().to(pred.device)
                self.results.append(ops.confusion_accumulate(pred, label, num_classes, self.ignore_index))
                self._last = (pred, label, num_classes)
            self._n_samples += 1
        if self.output_dir is not None:
            self._write_pngs(preds, [_sample_meta(s, 'img_path') for s in data_samples],
                             [bool(_sample_meta(s, 'reduce_zero_label', False)) for s in data_samples])

    def process_batch(self, pred, label=None, num_classes=None, img_paths=None, reduce_zero_label=False):
        """Batched fast path: accumulate a whole [N,H,W] prediction/label pair into the running matrix (not with
        `format_only` or without a label), and with `output_dir` write image n to the PNG named from img_paths[n]."""
        preds = list(pred) if pred.dim() == 3 else [pred]
        if label is not None and not self.format_only:
            k = num_classes or len(self.dataset_meta['classes'])
            self._cm = ops.confusion_accumulate(pred, label, k, self.ignore_index, self._cm)
            self._last = (preds[-1], label[-1] if label.dim() == 3 else label, k)
        self._n_samples += len(preds)
        if self.output_dir is not None and img_paths is not None:
            if isinstance(img_paths, str):
                img_paths = [img_paths]
            assert len(img_paths) == len(preds), 'one img_path per image'
            self._write_pngs(preds, img_paths, [bool(reduce_zero_label)] * len(preds))
        return self._cm

    def _write_pngs(self, preds, img_paths, reduce_zero_label):
        """One ops.png_encode call per (shape, dtype, reduce_zero_label) group, then the files."""
        groups = OrderedDict()
        for i, (p, z) in enumerate(zip(preds, reduce_zero_label)):
            groups.setdefault((tuple(p.shape), p.dtype, z), []).append(i)
        for (_, _, z), idx in groups.items():
            batch = preds[idx[0]][None] if len(idx) == 1 else torch.stack([preds[i] for i in idx])
            for i, data in zip(idx, ops.png_encode(batch, add=int(z))):
                base = os.path.splitext(os.path.basename(img_paths[i]))[0]
                with open(os.path.abspath(os.path.join(self.output_dir, f'{base}.png')), 'wb') as f:
                    f.write(data)

    @staticmethod
    def intersect_and_union(pred_label, label, num_classes, ignore_index):
        """iou_metric.py:163-200: four float32 [K] CPU tensors (exact while counts <= 2**24)."""
        cm = ops.confusion_accumulate(pred_label, label.to(pred_label.device), num_classes, ignore_index)
        return tuple(a.to(torch.float32).cpu() for a in _areas_from_cm(cm))

    def total_confusion(self, results=None, reduce_ranks=True):
        """Sum of every per-image matrix + the running matrix; all-reduced over ranks (int64)."""
        results = self.results if results is None else results
        mats = [r for r in results if torch.is_tensor(r)]
        if self._cm is not None:
            mats.append(self._cm)
        if not mats:
            return None
        total = torch.stack(mats).sum(0) if len(mats) > 1 else mats[0].clone()
        if reduce_ranks and torch.distributed.is_available() and torch.distributed.is_initialized() \
                and torch.distributed.get_world_size() > 1:
            torch.distributed.all_reduce(total, op=torch.distributed.ReduceOp.SUM)
        return total

    def compute_metrics(self, results=None):
        """iou_metric.py:102-161.  Accepts this class's matrices or reference-style 4-tuples.  With `format_only`
        nothing is computed: an empty OrderedDict, and a log line saying where the files went."""
        if self.format_only:
            logging.getLogger(__name__).info(f'results are saved to {self.output_dir}')
            return OrderedDict()
        results = self.results if results is None else results
        if len(results) and not torch.is_tensor(results[0]):
            cols = tuple(zip(*results))
            assert len(cols) == 4
            tot = [sum(c) for c in cols]
        else:
            cm = self.total_confusion(results)
            if cm is None:
                raise ValueError('IoUMetric.compute_metrics: no sample has been processed')
            # the reference sums float32 histograms; int64 counts converted once are exact <= 2**24
            tot = [a.to(torch.float32).cpu() for a in _areas_from_cm(cm)]
        ret = self.total_area_to_metrics(*tot, self.metrics, self.nan_to_num, self.beta)
        out = {}
        for k, v in ret.items():
            val = np.round(np.nanmean(v) * 100, 2)
            out[k if k == 'aAcc' else 'm' + k] = val
        self.per_class = OrderedDict((k, np.round(v * 100, 2)) for k, v in ret.items() if k != 'aAcc')
        return out

    def evaluate(self, size=None):
        """mmengine BaseMetric.evaluate(size): `size` is the dataset length.  A DistributedSampler pads the index list
        to a multiple of the world size by repeating samples, and `collect_results(results, size)` interleaves the ranks'
        lists and drops that padded tail - i.e. the LAST sample of every rank >= size % world_size.  The all-reduce here
        has no per-sample list to truncate, so those ranks subtract their last image's matrix before the sum."""
        import torch.distributed as dist
        if (size is not None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
                and self._last is not None):
            world, rank = dist.get_world_size(), dist.get_rank()
            per_rank = -(-int(size) // world)
            if int(size) % world and self._n_samples == per_rank and rank >= int(size) % world:
                pred, label, k = self._last
                dup = ops.confusion_accumulate(pred, label.to(pred.device), k, self.ignore_index)
                self.results.append(-dup)
        m = self.compute_metrics(self.results)
        self.results.clear()
        self._cm, self._n_samples, self._last = None, 0, None
        return m

    @staticmethod
    def total_area_to_metrics(total_area_intersect, total_area_union, total_area_pred_label,
                              total_area_label, metrics=('mIoU',), nan_to_num=None, beta=1):
        """iou_metric.py:202-295 (host-side float math on [K] vectors; negligible cost)."""
        def f_score(p, r):
            return (1 + beta ** 2) * (p * r) / ((beta ** 2 * p) + r)
        if isinstance(metrics, str):
            metrics = [metrics]
        if not set(metrics).issubset({'mIoU', 'mDice', 'mFscore'}):
            raise KeyError(f'metrics {metrics} is not supported')
        ti, tu, tp, tl = (torch.as_tensor(np.asarray(a)) if not torch.is_tensor(a) else a
                          for a in (total_area_intersect, total_area_union, total_area_pred_label,
                                    total_area_label))
        ret = OrderedDict(aAcc=ti.sum() / tl.sum())
        for m in metrics:
            if m == 'mIoU':
                ret['IoU'], ret['Acc'] = ti / tu, ti / tl
            if m in ('mIoU', 'mFscore'):
                p, r = ti / tp, ti / tl
                ret['Fscore'] = torch.tensor([f_score(a, b) for a, b in zip(p, r)])
                ret['Precision'], ret['Recall'] = p, r
            if m == 'mDice':
                ret['Dice'], ret['Acc'] = 2 * ti / (tp + tl), ti / tl
        ret = OrderedDict((k, v.numpy()) for k, v in ret.items())
        if nan_to_num is not None:
            ret = OrderedDict((k, np.nan_to_num(v, nan=nan_to_num)) for k, v in ret.items())
        return ret
