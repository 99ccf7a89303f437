"""`CityscapesMetric` (METRICS) - mmseg 1.2.2 ``mmseg/evaluation/metrics/citys_metric.py`` with cityscapesscripts'
pixel-level evaluation (``evaluation/evalPixelLevelSemanticLabeling.py``) computed on the device.

mmseg converts every prediction from trainIds to labelIds, saves it as a palette PNG, and hands the files to
``CSEval.evaluateImgLists``, which reads each one back with the GT ``*_gtFine_labelIds.png`` and
``*_gtFine_instanceIds.png`` and, per image, runs ``np.unique`` and one boolean mask per instance.  Here, per group of
same-shape samples of a `process` call:
  * the labelId files are encoded on the device (``ops.png_encode(lut=trainId -> labelId, palette=True)``, one call)
    and written when `keep_results` is set;
  * the GT files are decoded on the device (``ops.png_decode``: one 'label' call, one 'grey16' call);
  * ``ops.cityscapes_accumulate`` (csrc/cityscapes.cu, one call) adds the 34 x 34 confusion matrix and returns integer
    records (instId, size, tp, catTp) per image in np.unique's order.
The weighted float sums of the instance scores run on the host over those records, in CSEval's order, so the scores are
the ones CSEval computes from the same files.  The label table below is cityscapesscripts' ``helpers/labels.py``
(2.2.x) restated; the kernel gets its tables from here.
"""
import logging
import math
import os
from collections import OrderedDict

import numpy as np
import torch

from . import ops
from .lib import LedB200Error, CITYSCAPES_STATUS
from .metrics import _is_main_process, _sample_meta
from .registry import METRICS

# (name, id, trainId, category, hasInstances, ignoreInEval), cityscapesscripts helpers/labels.py
LABELS = [
    ('unlabeled', 0, 255, 'void', False, True),
    ('ego vehicle', 1, 255, 'void', False, True),
    ('rectification border', 2, 255, 'void', False, True),
    ('out of roi', 3, 255, 'void', False, True),
    ('static', 4, 255, 'void', False, True),
    ('dynamic', 5, 255, 'void', False, True),
    ('ground', 6, 255, 'void', False, True),
    ('road', 7, 0, 'flat', False, False),
    ('sidewalk', 8, 1, 'flat', False, False),
    ('parking', 9, 255, 'flat', False, True),
    ('rail track', 10, 255, 'flat', False, True),
    ('building', 11, 2, 'construction', False, False),
    ('wall', 12, 3, 'construction', False, False),
    ('fence', 13, 4, 'construction', False, False),
    ('guard rail', 14, 255, 'construction', False, True),
    ('bridge', 15, 255, 'construction', False, True),
    ('tunnel', 16, 255, 'construction', False, True),
    ('pole', 17, 5, 'object', False, False),
    ('polegroup', 18, 255, 'object', False, True),
    ('traffic light', 19, 6, 'object', False, False),
    ('traffic sign', 20, 7, 'object', False, False),
    ('vegetation', 21, 8, 'nature', False, False),
    ('terrain', 22, 9, 'nature', False, False),
    ('sky', 23, 10, 'sky', False, False),
    ('person', 24, 11, 'human', True, False),
    ('rider', 25, 12, 'human', True, False),
    ('car', 26, 13, 'vehicle', True, False),
    ('truck', 27, 14, 'vehicle', True, False),
    ('bus', 28, 15, 'vehicle', True, False),
    ('caravan', 29, 255, 'vehicle', True, True),
    ('trailer', 30, 255, 'vehicle', True, True),
    ('train', 31, 16, 'vehicle', True, False),
    ('motorcycle', 32, 17, 'vehicle', True, False),
    ('bicycle', 33, 18, 'vehicle', True, False),
    ('license plate', -1, -1, 'vehicle', False, True),
]
CATEGORIES = ['void', 'flat', 'construction', 'object', 'nature', 'sky', 'human', 'vehicle']
# evalPixelLevelSemanticLabeling.py: args.avgClassSize
AVG_CLASS_SIZE = {
    'bicycle': 4672.3249222261, 'caravan': 36771.8241758242, 'motorcycle': 6298.7200839748,
    'rider': 3930.4788056518, 'bus': 35732.1511111111, 'train': 67583.7075812274, 'car': 12794.0202738185,
    'person': 3462.4756337644, 'truck': 27855.1264367816, 'trailer': 16926.9763313609,
}
NUM_IDS = 34                                  # evalLabels: ids 0 .. 33

_BY_ID = {lab[1]: lab for lab in LABELS}
NAMES = [_BY_ID[i][0] for i in range(NUM_IDS)]
IGNORED = np.array([_BY_ID[i][5] for i in range(NUM_IDS)])
_CAT_OF = [_BY_ID[i][3] for i in range(NUM_IDS)]
# trainId2label is built over reversed(labels): for trainId 255 the first label in id order (unlabeled) wins
_TRAIN2ID = {}
for _lab in reversed(LABELS):
    _TRAIN2ID[_lab[2]] = _lab[1]
# mmseg's _convert_to_label_id on a uint8 map: trainIds 0 .. 18 and 255 are replaced, every other value stays
TRAIN_TO_ID = np.array([_TRAIN2ID.get(t, t) for t in range(256)], np.int64)
# categories with instance statistics: those whose labels (id >= 0) all have instances, with all their ids
INST_CATEGORIES = OrderedDict()
for _c in CATEGORIES:
    _labs = [lab for lab in LABELS if lab[3] == _c and lab[1] >= 0]
    if all(lab[4] for lab in _labs):
        INST_CATEGORIES[_c] = [lab[1] for lab in _labs]
# classes with instance statistics
INST_CLASSES = [lab[0] for lab in LABELS if lab[4] and not lab[5]]
# the kernel's tables: the instance category of each id (-1 none) and what an instance id of class id does
KERNEL_CATEGORY = [list(INST_CATEGORIES).index(_CAT_OF[i]) if any(i in v for v in INST_CATEGORIES.values()) else -1
                   for i in range(NUM_IDS)]
RULE_ERROR, RULE_SKIP, RULE_COUNT = 0, 1, 2
KERNEL_RULE = [RULE_SKIP if IGNORED[i] else RULE_COUNT if NAMES[i] in AVG_CLASS_SIZE else RULE_ERROR
               for i in range(NUM_IDS)]


# ---- scores (CSEval's functions over the matrix and the instance records) ------------------------------------------------
def _not_ignored_except(label):
    return [l for l in range(NUM_IDS) if not IGNORED[l] and l != label]


def _not_ignored_outside(category):
    return [l for l in range(NUM_IDS) if not IGNORED[l] and _CAT_OF[l] != category]


def _class_iou(label, cm):
    if IGNORED[label]:
        return float('nan')
    tp = np.longlong(cm[label, label])
    fn = np.longlong(cm[label, :].sum()) - tp
    fp = np.longlong(cm[_not_ignored_except(label), label].sum())
    denom = tp + fp + fn
    if denom == 0:
        return float('nan')
    return float(tp) / denom


def _class_iiou(label, cm, inst):
    if IGNORED[label] or NAMES[label] not in inst['classes']:
        return float('nan')
    tp, fn = inst['classes'][NAMES[label]]['tpWeighted'], inst['classes'][NAMES[label]]['fnWeighted']
    fp = np.longlong(cm[_not_ignored_except(label), label].sum())
    denom = tp + fp + fn
    if denom == 0:
        return float('nan')
    return float(tp) / denom


def _category_iou(category, cm):
    ids = [l for l in range(NUM_IDS) if _CAT_OF[l] == category and not IGNORED[l]]
    if not ids:
        return float('nan')
    tp = np.longlong(cm[ids, :][:, ids].sum())
    fn = np.longlong(cm[ids, :].sum()) - tp
    fp = np.longlong(cm[_not_ignored_outside(category), :][:, ids].sum())
    denom = tp + fp + fn
    if denom == 0:
        return float('nan')
    return float(tp) / denom


def _category_iiou(category, cm, inst):
    if category not in inst['categories']:
        return float('nan')
    ids = INST_CATEGORIES[category]
    tp, fn = inst['categories'][category]['tpWeighted'], inst['categories'][category]['fnWeighted']
    fp = np.longlong(cm[_not_ignored_outside(category), :][:, ids].sum())
    denom = tp + fp + fn
    if denom == 0:
        return float('nan')
    return float(tp) / denom


def _average(scores):
    valid, total = 0, 0.0
    for v in scores.values():
        if not math.isnan(v):
            valid += 1
            total += v
    return float('nan') if valid == 0 else total / valid


def instance_stats(records):
    """CSEval's instanceStats from the per-image records (instId, size, tp, catTp), images and instances in order."""
    zero = dict(tp=0, tpWeighted=0.0, fn=0, fnWeighted=0.0)
    inst = dict(classes={c: dict(zero) for c in INST_CLASSES},
                categories={c: dict(zero, labelIds=ids) for c, ids in INST_CATEGORIES.items()})
    for rec in records:
        for inst_id, size, tp, cat_tp in np.asarray(rec, np.int64).reshape(-1, 4).tolist():
            name = NAMES[inst_id // 1000]
            fn = size - tp
            weight = AVG_CLASS_SIZE[name] / float(size)
            c = inst['classes'][name]
            c['tp'] += tp
            c['fn'] += fn
            c['tpWeighted'] += float(tp) * weight
            c['fnWeighted'] += float(fn) * weight
            category = _CAT_OF[inst_id // 1000]
            if category in inst['categories']:
                cat_fn = size - cat_tp
                cat_weight = AVG_CLASS_SIZE[name] / float(size)
                k = inst['categories'][category]
                k['tp'] += cat_tp
                k['fn'] += cat_fn
                k['tpWeighted'] += float(cat_tp) * cat_weight
                k['fnWeighted'] += float(cat_fn) * cat_weight
    return inst


def result_dict(cm, records):
    """CSEval.evaluateImgLists' result (createResultDict, without perImageScores) from the int64 [34, 34] matrix and the
    per-image records in dataset order.  confMatrix is the int64 matrix."""
    cm = np.asarray(cm, np.int64)
    inst = instance_stats(records)
    class_scores = OrderedDict((NAMES[l], _class_iou(l, cm)) for l in range(NUM_IDS))
    class_inst = OrderedDict((NAMES[l], _class_iiou(l, cm, inst)) for l in range(NUM_IDS))
    cat_scores = OrderedDict((c, _category_iou(c, cm)) for c in CATEGORIES)
    cat_inst = OrderedDict((c, _category_iiou(c, cm, inst)) for c in CATEGORIES)
    total = cm.sum()
    return dict(
        confMatrix=cm,
        priors={NAMES[l]: float(cm[l, :].sum()) / total for l in range(NUM_IDS)},
        labels={NAMES[l]: l for l in range(NUM_IDS)},
        classScores=class_scores, classInstScores=class_inst, categoryScores=cat_scores, categoryInstScores=cat_inst,
        averageScoreClasses=_average(class_scores), averageScoreInstClasses=_average(class_inst),
        averageScoreCategories=_average(cat_scores), averageScoreInstCategories=_average(cat_inst))


def combine(states, size=None):
    """The dataset's result dict from every rank's state (rank order).  A state is dict(cm, last_cm, records): the
    rank's int64 [34, 34] matrix, the matrix of its last image alone, and its images' records in processing order.
    Rank-local image i of rank r is dataset image i * world + r (a DistributedSampler's interleaving); with `size`,
    images at or past it (the sampler's padded tail, the last image of a rank) are dropped, as collect_results does."""
    world = len(states)
    cm = np.zeros((NUM_IDS, NUM_IDS), np.int64)
    order = []
    for r, s in enumerate(states):
        recs = list(s['records'])
        cm += np.asarray(s['cm'], np.int64)
        for i, rec in enumerate(recs):
            g = i * world + r
            if size is not None and g >= size:
                if i != len(recs) - 1:
                    raise ValueError(f'combine: rank {r} holds {len(recs)} images, more than the padded tail allows')
                cm -= np.asarray(s['last_cm'], np.int64)
                continue
            order.append((g, rec))
    order.sort(key=lambda x: x[0])
    return result_dict(cm, [rec for _, rec in order])


# ---- the metric ----------------------------------------------------------------------------------------------------------
@METRICS.register_module()
class CityscapesMetric:
    """mmseg's CityscapesMetric(output_dir, ignore_index=255, format_only=False, keep_results=False,
    collect_device='cpu', prefix=None).  `evaluate` returns {'averageScoreCategories', 'averageScoreInstCategories'} as
    CSEval's fractions; the whole result dict stays in `cityscapes_results`.  Unlike mmseg, files are written only with
    keep_results (which format_only requires), predictions are never read back from disk, and output_dir is not removed.
    cityscapesscripts is not needed."""

    def __init__(self, output_dir, ignore_index=255, format_only=False, keep_results=False, collect_device='cpu',
                 prefix=None, **kwargs):
        if format_only:
            assert keep_results, ('When format_only is True, the results must be kept, please set keep_results as '
                                  f'True, but got {keep_results}')
        self.output_dir, self.ignore_index = output_dir, ignore_index
        self.format_only, self.keep_results = format_only, keep_results
        self.collect_device, self.prefix = collect_device, prefix
        if _is_main_process():
            os.makedirs(output_dir, exist_ok=True)
        self.dataset_meta = None
        self.cityscapes_results = None
        self._reset()

    def _reset(self):
        self._cm = None                         # running int64 [34, 34] on the device
        self._last_cm = None                    # the matrix of the last image processed
        self._records = []                      # per image, in processing order
        self.results = []                       # (png_filename, gt_filename) per image, as mmseg records them

    def process(self, data_batch, data_samples):
        preds = [s['pred_sem_seg']['data'][0] for s in data_samples]
        img_paths = [_sample_meta(s, 'img_path') for s in data_samples]
        seg_paths = None if self.format_only else [_sample_meta(s, 'seg_map_path') for s in data_samples]
        self._process(preds, img_paths, seg_paths)

    def process_batch(self, pred, seg_map_paths=None, img_paths=None):
        """The labels-only path: pred [N, H, W] (or [H, W]) trainIds on the device; the GT files from seg_map_paths
        (unless format_only); the labelId files named from img_paths (with keep_results)."""
        preds = list(pred) if pred.dim() == 3 else [pred]
        if isinstance(img_paths, str):
            img_paths = [img_paths]
        if isinstance(seg_map_paths, str):
            seg_map_paths = [seg_map_paths]
        if img_paths is None:
            if self.keep_results:
                raise ValueError('CityscapesMetric.process_batch: keep_results needs img_paths to name the files')
            img_paths = [None] * len(preds)
        if not self.format_only and (seg_map_paths is None or len(seg_map_paths) != len(preds)):
            raise ValueError('CityscapesMetric.process_batch: one seg_map_path per image')
        self._process(preds, img_paths, None if self.format_only else seg_map_paths)

    def _process(self, preds, img_paths, seg_paths):
        groups = OrderedDict()
        for i, p in enumerate(preds):
            groups.setdefault((tuple(p.shape), p.dtype), []).append(i)
        records = [None] * len(preds)
        pngs = [None if p is None else os.path.abspath(os.path.join(
            self.output_dir, os.path.splitext(os.path.basename(p))[0] + '.png')) for p in img_paths]
        gts = None
        if seg_paths is not None:
            gts = [p.replace('labelTrainIds.png', 'labelIds.png') for p in seg_paths]
        for idx in groups.values():
            batch = torch.stack([preds[i] for i in idx]) if len(idx) > 1 else preds[idx[0]][None]
            if gts is None and batch.dtype == torch.int64:
                lo, hi = torch.aminmax(batch)
                if lo.item() < 0 or hi.item() > 255:
                    raise LedB200Error(f'CityscapesMetric: {img_paths[idx[0]]} ..: int64 predictions outside 0 .. 255')
            if gts is not None:
                recs, last = self._evaluate_group(batch, [gts[i] for i in idx], [img_paths[i] for i in idx])
                for i, r in zip(idx, recs):
                    records[i] = r
                if idx[-1] == len(preds) - 1:
                    self._last_cm = last
            if self.keep_results:
                for i, data in zip(idx, ops.png_encode(batch, lut=TRAIN_TO_ID, palette=True)):
                    with open(pngs[i], 'wb') as f:
                        f.write(data)
        for i in range(len(preds)):
            self.results.append((pngs[i], '' if gts is None else gts[i]))
        if gts is not None:
            self._records.extend(records)

    def _evaluate_group(self, batch, gts, names):
        insts = [g.replace('labelIds', 'instanceIds') for g in gts]
        gt_bytes, inst_bytes = [], []
        for path, store in ((gts, gt_bytes), (insts, inst_bytes)):
            for p in path:
                try:
                    with open(p, 'rb') as f:
                        store.append(f.read())
                except OSError as e:
                    raise LedB200Error(f'CityscapesMetric: {p}: {e.strerror or e}') from None
        dev = batch.device
        labels = ops.png_decode(gt_bytes, 'label', names=gts, device=dev)
        inst = ops.png_decode(inst_bytes, 'grey16', names=insts, device=dev)
        H, W = batch.shape[1:]
        for g, gi, l, i, name in zip(gts, insts, labels, inst, names):
            if tuple(l.shape[1:]) != (H, W) or tuple(i.shape[1:]) != (H, W):
                raise LedB200Error(f'CityscapesMetric: {g} is {l.shape[2]} x {l.shape[1]}, {gi} {i.shape[2]} x '
                                   f'{i.shape[1]} and the prediction of {name} {W} x {H}: the sizes must be equal')
        if self._cm is None:
            self._cm = torch.zeros((NUM_IDS, NUM_IDS), dtype=torch.int64, device=dev)
        last = torch.empty((NUM_IDS, NUM_IDS), dtype=torch.int64, device=dev)
        _, st, recs = ops.cityscapes_accumulate(batch, torch.cat(labels), torch.cat(inst), TRAIN_TO_ID,
                                                KERNEL_CATEGORY, KERNEL_RULE, self._cm, last)
        bad = [f'{g}: ' + ', '.join(why for bit, why in CITYSCAPES_STATUS.items() if s & bit)
               for g, s in zip(gts, st.tolist()) if s]
        if bad:
            raise LedB200Error('CityscapesMetric: ' + '; '.join(bad))
        return recs, last

    def state(self):
        """This rank's state for combine(): host copies of the matrices and the records."""
        z = np.zeros((NUM_IDS, NUM_IDS), np.int64)
        return dict(cm=self._cm.cpu().numpy() if self._cm is not None else z,
                    last_cm=self._last_cm.cpu().numpy() if self._last_cm is not None else z,
                    records=list(self._records))

    def compute_metrics(self, results=None, size=None):
        """citys_metric.py compute_metrics: {} with format_only, else the two category averages of CSEval."""
        if self.format_only:
            logging.getLogger(__name__).info(f'results are saved to {os.path.dirname(self.output_dir)}')
            return OrderedDict()
        states = [self.state()]
        d = torch.distributed
        if d.is_available() and d.is_initialized() and d.get_world_size() > 1:
            states = [None] * d.get_world_size()
            d.all_gather_object(states, self.state())
        if not any(len(s['records']) for s in states):
            raise ValueError('CityscapesMetric.compute_metrics: no sample has been processed')
        self.cityscapes_results = combine(states, size)
        return dict(averageScoreCategories=self.cityscapes_results['averageScoreCategories'],
                    averageScoreInstCategories=self.cityscapes_results['averageScoreInstCategories'])

    def evaluate(self, size=None):
        """mmengine BaseMetric.evaluate(size): `size` is the dataset length (the padded tail past it is dropped)."""
        m = self.compute_metrics(size=size)
        self._reset()
        return m
