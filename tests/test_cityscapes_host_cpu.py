"""CityscapesMetric's host side (no GPU): the oracle on hand-computed scenes, the scores and `combine` against the oracle,
the 16-bit PNG decoder on the CPU (ledb200_png_decode_host, the kernels' __host__ __device__ code) and what the decoder
still refuses; and, where cityscapesscripts is installed, the oracle against the real evaluateImgLists."""
import io
import math
import os

import numpy as np
import pytest
import torch
from PIL import Image

import lednet_b200 as L
from lednet_b200 import cityscapes as CS, lib, ops
import cityscapes_corpus as CC
import cityscapes_oracle as O
import png_corpus as P


# ---- the oracle by hand --------------------------------------------------------------------------------------------------
def test_oracle_matches_a_hand_computed_scene():
    gt = np.array([[7, 7, 8, 8], [24, 24, 0, 0]], np.uint8)
    inst = np.array([[7, 7, 8, 8], [24001, 24001, 0, 0]], np.int32)
    pred = np.array([[7, 8, 8, 8], [24, 7, 0, 24]], np.uint8)
    r = O.evaluate_arrays([(pred, gt, inst)])
    cs = r['classScores']
    assert cs['road'] == 1 / 3 and cs['sidewalk'] == 2 / 3 and cs['person'] == 0.5
    assert all(math.isnan(v) for k, v in cs.items() if k not in ('road', 'sidewalk', 'person'))
    assert r['averageScoreClasses'] == 0.5
    assert r['classInstScores']['person'] == 0.5
    assert all(math.isnan(v) for k, v in r['classInstScores'].items() if k != 'person')
    assert r['averageScoreInstClasses'] == 0.5
    cat = r['categoryScores']
    assert cat['flat'] == 0.8 and cat['human'] == 0.5
    assert all(math.isnan(cat[c]) for c in ('void', 'construction', 'object', 'nature', 'sky', 'vehicle'))
    assert r['averageScoreCategories'] == 0.65
    assert r['categoryInstScores']['human'] == 0.5 and math.isnan(r['categoryInstScores']['vehicle'])
    assert r['averageScoreInstCategories'] == 0.5
    assert r['confMatrix'][24, 7] == 1 and r['confMatrix'].sum() == 8


def test_oracle_nan_cases():
    gt = np.full((3, 3), 7, np.uint8)
    r = O.evaluate_arrays([(gt.copy(), gt, gt.astype(np.int32))])     # no instances
    assert r['classScores']['road'] == 1.0
    assert all(math.isnan(v) for v in r['classInstScores'].values())
    assert math.isnan(r['averageScoreInstClasses']) and math.isnan(r['averageScoreInstCategories'])
    void = np.zeros((3, 3), np.uint8)                                  # every pixel ignored: zero denominators
    r = O.evaluate_arrays([(void, void, void.astype(np.int32))])
    assert all(math.isnan(v) for v in r['classScores'].values()) and math.isnan(r['averageScoreCategories'])


def test_oracle_errors():
    gt = np.full((2, 2), 7, np.uint8)
    for pred, g, inst in ((gt, gt + 33, gt.astype(np.int32)), (gt + 30, gt, gt.astype(np.int32)),
                          (gt, gt, np.full((2, 2), 7001, np.int32)), (gt, gt, np.full((2, 2), 34001, np.int32))):
        with pytest.raises(O.CSEvalError):
            O.evaluate_arrays([(pred, g, inst)])
    O.evaluate_arrays([(gt, gt, np.full((2, 2), 29001, np.int32))])   # caravan: skipped


# ---- tables, scores and combine ---------------------------------------------------------------------------------------------
def test_tables():
    want = {t: i for t, i in enumerate([7, 8, 11, 12, 13, 17, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 31, 32, 33])}
    want[255] = 0
    assert CS.TRAIN_TO_ID.tolist() == [want.get(t, t) for t in range(256)]
    v = np.arange(256)
    assert np.array_equal(CS.TRAIN_TO_ID, O.convert_to_label_id(v.astype(np.int64)).astype(np.int64))
    assert [i for i in range(34) if CS.KERNEL_RULE[i] == CS.RULE_COUNT] == [24, 25, 26, 27, 28, 31, 32, 33]
    assert [i for i in range(34) if CS.KERNEL_RULE[i] == CS.RULE_SKIP] == [0, 1, 2, 3, 4, 5, 6, 9, 10, 14, 15, 16, 18,
                                                                           29, 30]
    assert CS.INST_CATEGORIES == {'human': [24, 25], 'vehicle': list(range(26, 34))}
    assert L.METRICS.get('CityscapesMetric') is L.CityscapesMetric


def _scenes(n=7, h=96, w=160):
    out = []
    for i in range(n):
        gt, inst, pred = CC.scene(h, w, seed=100 + i, cell=16)
        out.append((O.convert_to_label_id(pred), gt, inst))
    return out


def _per_image(triples):
    """each image's own matrix and records, from the oracle"""
    out = []
    for pred, gt, inst in triples:
        cm = O.generate_matrix()
        O.evaluate_pair(pred, gt, inst, cm, O.generate_instance_stats())
        out.append((cm.astype(np.int64), np.array(O.instance_records(pred, inst), np.int64).reshape(-1, 4)))
    return out


def test_result_dict_equals_the_oracle():
    triples = _scenes()
    per = _per_image(triples)
    got = CS.result_dict(sum(cm for cm, _ in per), [r for _, r in per])
    assert O.same(got, O.evaluate_arrays(triples))
    assert sum(len(r) for _, r in per) > 20


@pytest.mark.parametrize('world,size', [(1, 7), (2, 6), (3, 7), (4, 7), (2, 7)])
def test_combine_restores_dataset_order_and_drops_the_padded_tail(world, size):
    per = _per_image(_scenes(size))
    single = CS.combine([dict(cm=sum(cm for cm, _ in per), last_cm=per[-1][0], records=[r for _, r in per])], size)
    per_rank = -(-size // world)
    states = []
    for r in range(world):
        idx = [i * world + r for i in range(per_rank)]
        idx = [g if g < size else g - size for g in idx]             # DistributedSampler pads from the start
        states.append(dict(cm=sum(per[g][0] for g in idx), last_cm=per[idx[-1]][0], records=[per[g][1] for g in idx]))
    got = CS.combine(states, size)
    assert O.same(got, single)
    if size % world:
        assert not O.same(CS.combine(states), single)               # without size the duplicates count


# ---- the 16-bit decoder on the CPU ----------------------------------------------------------------------------------------
def test_host_grey16_corpus_matches_pil():
    corpus = CC.grey16_corpus()
    rc, st, outs = CC.host16([b for _, b in corpus])
    assert rc == 0
    for (name, b), s, o in zip(corpus, st, outs):
        assert s == 0, (name, lib.PNG_STATUS.get(s))
        assert Image.open(io.BytesIO(b)).mode.startswith('I'), name
        assert np.array_equal(o, CC.pil16_ref(b)), name


@pytest.mark.parametrize('name,data,status', CC.corrupt16(), ids=[c[0] for c in CC.corrupt16()])
def test_host_grey16_rejects_corrupt_files(name, data, status):
    rc, st, _ = CC.host16([data])
    assert rc == 0 and st == [status], lib.PNG_STATUS.get(st[0])


def test_host_grey16_fuzz():
    valid = 0
    for f, want in CC.fuzz16(300, seed=2):
        _, st, outs = CC.host16([f])
        if want is None:
            assert st[0] != 0
            continue
        valid += 1
        assert st[0] == 0 and np.array_equal(outs[0], want)
        assert np.array_equal(outs[0], CC.pil16_ref(f))
    assert valid >= 40


def test_sixteen_bit_files_stay_refused_by_the_other_kinds():
    f = CC.pil16(np.arange(12).reshape(3, 4) * 1000)
    assert ops.png_info(f, 'grey16') == (3, 4, 0)
    for kind in ('color', 'label'):
        with pytest.raises(NotImplementedError):
            ops.png_info(f, kind)
    with pytest.raises(NotImplementedError):
        ops.png_info(P.png(np.zeros((2, 2), np.uint8), 0), 'grey16')          # 8-bit grey
    with pytest.raises(NotImplementedError):
        ops.png_info(P.SIG + P.ihdr(4, 4, 2, 16), 'grey16')                   # 16-bit colour
    with pytest.raises(ValueError):
        ops.png_decode([f], 'grey8')
    rc, st, _ = CC.host16([f], mode=lib.PNG_LABEL)                                 # the label mode reads bit depth 8
    assert rc == 0 and st == [1]
    for mode in (2, 3, 15, 17):
        assert CC.host16([f], mode=mode)[0] == -1
    assert CC.host16([f], ct=3)[0] == -1                                          # grey16 takes colour type 0 only


def test_grey16_decode_needs_cuda():
    if torch.cuda.is_available():
        pytest.skip('checks the no-device error')
    with pytest.raises(lib.LedB200Error):
        ops.png_decode([CC.pil16(np.ones((2, 2)))], 'grey16')


# ---- against the real package ---------------------------------------------------------------------------------------------
def test_oracle_against_cityscapesscripts(tmp_path):
    CSEval = pytest.importorskip('cityscapesscripts.evaluation.evalPixelLevelSemanticLabeling')
    scenes = [CC.scene(64, 96, seed=200 + i, cell=16) for i in range(4)]
    samples = CC.write_dataset(str(tmp_path), scenes)
    preds, gts = [], []
    for i, ((gt, inst, pred), (_, seg)) in enumerate(zip(scenes, samples)):
        p = str(tmp_path / f'pred_{i}.png')
        Image.fromarray(O.convert_to_label_id(pred)).convert('P').save(p)
        preds.append(p)
        gts.append(seg.replace('labelTrainIds.png', 'labelIds.png'))
    args = CSEval.args
    args.evalInstLevelScore, args.evalPixelAccuracy, args.JSONOutput, args.quiet = True, False, False, True
    args.predictionPath = str(tmp_path)
    real = CSEval.evaluateImgLists(preds, gts, args)
    mine = O.evaluate_arrays([(O.convert_to_label_id(p), g, i) for g, i, p in scenes])
    for k in mine:
        assert O.same(mine[k], real[k]), k
