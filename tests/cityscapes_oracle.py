"""A numpy restatement of the Cityscapes pixel-level evaluation, the reference CityscapesMetric is checked against.

Sources, restated from the released packages (neither is a dependency of this repository):
  * cityscapesscripts 2.2.x, cityscapesscripts/helpers/labels.py: the label table, trainId2label (built over
    reversed(labels)), category2labels;
  * cityscapesscripts 2.2.x, cityscapesscripts/evaluation/evalPixelLevelSemanticLabeling.py: args.avgClassSize,
    generateMatrix (np.ulonglong), generateInstanceStats, evaluatePair (the confusion matrix, np.unique over the instance
    ids above 1000, one mask per instance, the weighted tp / fn in Python floats), getIouScoreForLabel,
    getInstanceIouScoreForLabel, getIouScoreForCategory, getInstanceIouScoreForCategory, getScoreAverage, getPrior and
    createResultDict, evaluateImgLists (images in list order);
  * mmseg 1.2.2, mmseg/evaluation/metrics/citys_metric.py: CityscapesMetric._convert_to_label_id.
Per-image pixel accuracy (perImageScores) is left out.  Where cityscapesscripts can be imported,
tests/test_cityscapes_host_cpu.py runs the real evaluateImgLists on files and compares its result with this one."""
import math
from collections import namedtuple

import numpy as np

Label = namedtuple('Label', 'name id trainId category catId hasInstances ignoreInEval')
labels = [
    Label('unlabeled', 0, 255, 'void', 0, False, True),
    Label('ego vehicle', 1, 255, 'void', 0, False, True),
    Label('rectification border', 2, 255, 'void', 0, False, True),
    Label('out of roi', 3, 255, 'void', 0, False, True),
    Label('static', 4, 255, 'void', 0, False, True),
    Label('dynamic', 5, 255, 'void', 0, False, True),
    Label('ground', 6, 255, 'void', 0, False, True),
    Label('road', 7, 0, 'flat', 1, False, False),
    Label('sidewalk', 8, 1, 'flat', 1, False, False),
    Label('parking', 9, 255, 'flat', 1, False, True),
    Label('rail track', 10, 255, 'flat', 1, False, True),
    Label('building', 11, 2, 'construction', 2, False, False),
    Label('wall', 12, 3, 'construction', 2, False, False),
    Label('fence', 13, 4, 'construction', 2, False, False),
    Label('guard rail', 14, 255, 'construction', 2, False, True),
    Label('bridge', 15, 255, 'construction', 2, False, True),
    Label('tunnel', 16, 255, 'construction', 2, False, True),
    Label('pole', 17, 5, 'object', 3, False, False),
    Label('polegroup', 18, 255, 'object', 3, False, True),
    Label('traffic light', 19, 6, 'object', 3, False, False),
    Label('traffic sign', 20, 7, 'object', 3, False, False),
    Label('vegetation', 21, 8, 'nature', 4, False, False),
    Label('terrain', 22, 9, 'nature', 4, False, False),
    Label('sky', 23, 10, 'sky', 5, False, False),
    Label('person', 24, 11, 'human', 6, True, False),
    Label('rider', 25, 12, 'human', 6, True, False),
    Label('car', 26, 13, 'vehicle', 7, True, False),
    Label('truck', 27, 14, 'vehicle', 7, True, False),
    Label('bus', 28, 15, 'vehicle', 7, True, False),
    Label('caravan', 29, 255, 'vehicle', 7, True, True),
    Label('trailer', 30, 255, 'vehicle', 7, True, True),
    Label('train', 31, 16, 'vehicle', 7, True, False),
    Label('motorcycle', 32, 17, 'vehicle', 7, True, False),
    Label('bicycle', 33, 18, 'vehicle', 7, True, False),
    Label('license plate', -1, -1, 'vehicle', 7, False, True),
]
id2label = {label.id: label for label in labels}
trainId2label = {label.trainId: label for label in reversed(labels)}
category2labels = {}
for label in labels:
    category2labels.setdefault(label.category, []).append(label)

avgClassSize = {
    'bicycle': 4672.3249222261, 'caravan': 36771.8241758242, 'motorcycle': 6298.7200839748,
    'rider': 3930.4788056518, 'bus': 35732.1511111111, 'train': 67583.7075812274, 'car': 12794.0202738185,
    'person': 3462.4756337644, 'truck': 27855.1264367816, 'trailer': 16926.9763313609,
}
evalLabels = [label.id for label in labels if label.id >= 0]


class CSEvalError(Exception):
    pass


def convert_to_label_id(pred):
    """mmseg CityscapesMetric._convert_to_label_id, then .astype(np.uint8) as the saved file holds it"""
    out = pred.copy()
    for train_id, label in trainId2label.items():
        out[pred == train_id] = label.id
    return out.astype(np.uint8)


def generate_matrix():
    return np.zeros((max(evalLabels) + 1, max(evalLabels) + 1), dtype=np.ulonglong)


def generate_instance_stats():
    stats = {'classes': {}, 'categories': {}}
    for label in labels:
        if label.hasInstances and not label.ignoreInEval:
            stats['classes'][label.name] = dict(tp=0, tpWeighted=0.0, fn=0, fnWeighted=0.0)
    for category in category2labels:
        ids, all_inst = [], True
        for label in category2labels[category]:
            if label.id < 0:
                continue
            if not label.hasInstances:
                all_inst = False
                break
            ids.append(label.id)
        if all_inst:
            stats['categories'][category] = dict(tp=0, tpWeighted=0.0, fn=0, fnWeighted=0.0, labelIds=ids)
    return stats


def instance_records(pred, inst):
    """(instId, size, tp, catTp) of every instance evaluatePair counts, in its order"""
    masks = {c: np.isin(pred, v['labelIds']) for c, v in generate_instance_stats()['categories'].items()}
    out = []
    for inst_id in np.unique(inst[inst > 1000]):
        label_id = int(inst_id / 1000)
        if label_id not in id2label:
            raise CSEvalError(f'KeyError: {label_id}')
        label = id2label[label_id]
        if label.ignoreInEval:
            continue
        if label.name not in avgClassSize:
            raise CSEvalError(f'KeyError: {label.name}')
        mask = inst == inst_id
        size = np.count_nonzero(mask)
        tp = np.count_nonzero(pred[mask] == label_id)
        cat_tp = np.count_nonzero(np.logical_and(mask, masks[label.category])) if label.category in masks else tp
        out.append((int(inst_id), int(size), int(tp), int(cat_tp)))
    return out


def evaluate_pair(pred, gt, inst, cm, stats):
    """evaluatePair on decoded arrays: pred labelIds (uint8), gt labelIds, inst instanceIds"""
    if pred.shape != gt.shape or inst.shape != gt.shape:
        raise CSEvalError('image sizes differ')
    for v in np.unique(gt):
        if v not in evalLabels:
            raise CSEvalError(f'Unknown label with id {v}')
    for v in np.unique(pred):
        if v not in evalLabels:
            raise CSEvalError(f'Unknown label with id {v}')
    enc = gt.astype(np.int32) * 34 + pred.astype(np.int32)
    values, counts = np.unique(enc, return_counts=True)
    for value, c in zip(values, counts):
        cm[value // 34][value % 34] += c
    cat_masks = {c: np.isin(pred, v['labelIds']).reshape(pred.shape) for c, v in stats['categories'].items()}
    for inst_id in np.unique(inst[inst > 1000]):
        label_id = int(inst_id / 1000)
        if label_id not in id2label:
            raise CSEvalError(f'KeyError: {label_id}')
        label = id2label[label_id]
        if label.ignoreInEval:
            continue
        mask = inst == inst_id
        size = np.count_nonzero(mask)
        tp = np.count_nonzero(pred[mask] == label_id)
        fn = size - tp
        if label.name not in avgClassSize:
            raise CSEvalError(f'KeyError: {label.name}')
        weight = avgClassSize[label.name] / float(size)
        s = stats['classes'][label.name]
        s['tp'] += tp
        s['fn'] += fn
        s['tpWeighted'] += float(tp) * weight
        s['fnWeighted'] += float(fn) * weight
        if label.category in stats['categories']:
            cat_tp = np.count_nonzero(np.logical_and(mask, cat_masks[label.category]))
            cat_fn = size - cat_tp
            cat_weight = avgClassSize[label.name] / float(size)
            k = stats['categories'][label.category]
            k['tp'] += cat_tp
            k['fn'] += cat_fn
            k['tpWeighted'] += float(cat_tp) * cat_weight
            k['fnWeighted'] += float(cat_fn) * cat_weight


def iou_label(label, cm):
    if id2label[label].ignoreInEval:
        return float('nan')
    tp = np.longlong(cm[label, label])
    fn = np.longlong(cm[label, :].sum()) - tp
    not_ignored = [l for l in evalLabels if not id2label[l].ignoreInEval and not l == label]
    fp = np.longlong(cm[not_ignored, label].sum())
    denom = tp + fp + fn
    if denom == 0:
        return float('nan')
    return float(tp) / denom


def iiou_label(label, cm, stats):
    if id2label[label].ignoreInEval:
        return float('nan')
    name = id2label[label].name
    if name not in stats['classes']:
        return float('nan')
    tp, fn = stats['classes'][name]['tpWeighted'], stats['classes'][name]['fnWeighted']
    not_ignored = [l for l in evalLabels if not id2label[l].ignoreInEval and not l == label]
    fp = np.longlong(cm[not_ignored, label].sum())
    denom = tp + fp + fn
    if denom == 0:
        return float('nan')
    return float(tp) / denom


def iou_category(category, cm):
    ids = [label.id for label in category2labels[category] if not label.ignoreInEval and label.id in evalLabels]
    if not ids:
        return float('nan')
    tp = np.longlong(cm[ids, :][:, ids].sum())
    fn = np.longlong(cm[ids, :].sum()) - tp
    outside = [l for l in evalLabels if not id2label[l].ignoreInEval and id2label[l].category != category]
    fp = np.longlong(cm[outside, :][:, ids].sum())
    denom = tp + fp + fn
    if denom == 0:
        return float('nan')
    return float(tp) / denom


def iiou_category(category, cm, stats):
    if category not in stats['categories']:
        return float('nan')
    ids = stats['categories'][category]['labelIds']
    tp, fn = stats['categories'][category]['tpWeighted'], stats['categories'][category]['fnWeighted']
    outside = [l for l in evalLabels if not id2label[l].ignoreInEval and id2label[l].category != category]
    fp = np.longlong(cm[outside, :][:, ids].sum())
    denom = tp + fp + fn
    if denom == 0:
        return float('nan')
    return float(tp) / denom


def score_average(scores):
    valid, total = 0, 0.0
    for k in scores:
        if not math.isnan(scores[k]):
            valid += 1
            total += scores[k]
    if valid == 0:
        return float('nan')
    return total / valid


def evaluate_arrays(triples):
    """evaluateImgLists over (pred labelIds, gt labelIds, instanceIds) triples in list order: createResultDict's keys
    except perImageScores (confMatrix as the ulonglong matrix)"""
    cm, stats = generate_matrix(), generate_instance_stats()
    for pred, gt, inst in triples:
        evaluate_pair(pred, gt, inst, cm, stats)
    class_scores = {id2label[l].name: iou_label(l, cm) for l in evalLabels}
    class_inst = {id2label[l].name: iiou_label(l, cm, stats) for l in evalLabels}
    cat_scores = {c: iou_category(c, cm) for c in category2labels}
    cat_inst = {c: iiou_category(c, cm, stats) for c in category2labels}
    return dict(
        confMatrix=cm,
        priors={id2label[l].name: float(cm[l, :].sum()) / cm.sum() for l in evalLabels},
        labels={id2label[l].name: l for l in evalLabels},
        classScores=class_scores, classInstScores=class_inst, categoryScores=cat_scores, categoryInstScores=cat_inst,
        averageScoreClasses=score_average(class_scores), averageScoreInstClasses=score_average(class_inst),
        averageScoreCategories=score_average(cat_scores), averageScoreInstCategories=score_average(cat_inst))


def same(a, b):
    """bit-for-bit equality of two result dicts (nan equals nan; confMatrix by value)"""
    if isinstance(a, dict):
        return isinstance(b, dict) and list(a) == list(b) and all(same(a[k], b[k]) for k in a)
    if isinstance(a, np.ndarray) or isinstance(b, np.ndarray) or isinstance(a, list):
        return np.array_equal(np.asarray(a, np.int64), np.asarray(b, np.int64))
    if isinstance(a, str):
        return a == b
    fa, fb = float(a), float(b)
    return (math.isnan(fa) and math.isnan(fb)) or fa.hex() == fb.hex()
