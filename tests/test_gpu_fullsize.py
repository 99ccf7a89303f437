"""Parity AT THE BENCHMARKED SIZES (BASELINE configs 2 and 5), through the C ABI, against the CPU oracle.

The batch-16 1024x2048 plan is not the small-test plan: it replays a CUDA graph, walks ~110 tiles per persistent
CTA with both MMA issuers active, has no epilogue staging tiles (every tile interior) and runs the label-only ladder.
These tests run exactly that plan (and the batch-128 512x512 K=2 plan of config 5) and compare whole images with the
oracle: labels, logits and the confusion matrix.

Weights are TRAINED (tests/trained.py: a few hundred steps of the repo's own training step on learnable blocky
scenes, seeded), because north_star's bf16 gate - >= 99.9 % argmax agreement - presumes trained logit margins; the
same state dict is loaded into the oracle and the engine.  The near-tie analysis stays as a diagnostic only.
"""
import numpy as np
import pytest
import torch

import oracle
from lednet_b200 import ops, synth
import trained
from util import build_pair, rel_err, near_tie_mask

pytestmark = pytest.mark.gpu
DEV = 'cuda'

SCHED19 = [(2, (512, 1024), (4, 8)), (1, (1024, 2048), (8, 16)), (2, (512, 1024), (8, 16))]
SCHED2 = [(8, (512, 512), (4, 4)), (8, (512, 512), (8, 8)), (4, (512, 1024), (4, 8))]


def _pair(k, dtype, sched):
    o, m = build_pair(k, dtype=dtype)
    sd = trained.train_product(k, sched, steps=300)
    o.load_state_dict(sd)
    m.load_state_dict(sd, strict=True)
    return o, m


def _scenes(n, h, w, k, coarse, seed):
    imgs, labs = [], []
    for i in range(n):                      # one scene per image: every image of the batch is different
        im, lb = synth.make_scene(1, h, w, k, seed=seed + i, coarse=coarse, ignore_frac=0.03)
        imgs.append(im), labs.append(lb)
    return torch.cat(imgs), torch.cat(labs)


def _check_cm(pred_dev, lab, k):
    cm = ops.confusion_accumulate(pred_dev, lab.to(DEV), k)
    ref = oracle.confusion_matrix(pred_dev.cpu().numpy().astype(np.int64), lab.numpy(), k, 255)
    np.testing.assert_array_equal(cm.cpu().numpy(), ref)                        # bit-exact given identical predictions
    return cm


def _run_bf16(k, n, h, w, coarse, sched, check):
    o, m = _pair(k, 'bf16', sched)
    img, lab = _scenes(n, h, w, k, coarse, seed=500)
    x = oracle.preprocess(img)
    xd = x.to(DEV)
    eng = m.engine()
    pred = eng.forward_infer(xd)                                   # the benchmarked call: labels only, graph replay
    pred_again = eng.forward_infer(xd)                             # second call = graph REPLAY of the captured plan
    assert torch.equal(pred, pred_again)
    pred_u8 = m.predict_labels(img.to(DEV))                        # raw uint8 BGR -> fused preprocessing in the stem
    assert (pred_u8 != pred).float().mean() < 1e-4
    pred_lg, logits = eng.forward_infer(xd, want_logits=True)      # logits export variant of the tail
    assert torch.equal(pred_lg, pred)                              # label-only ladder == tail2 labels, bit for bit
    stats = []
    for i in check:
        ref_logits, ref_pred = o.predict(x[i:i + 1])
        agree = (pred[i].cpu().long() == ref_pred[0, 0]).float().mean().item()
        acc = (ref_pred[0, 0] == lab[i])[lab[i] != 255].float().mean().item()
        err = rel_err(logits[i:i + 1].cpu(), ref_logits)
        mism = pred[i].cpu().long() != ref_pred[0, 0]
        unexplained = (mism & ~near_tie_mask(ref_logits, 4e-2)[0]).sum().item()
        stats.append((i, agree, err, acc, unexplained))
    print('bf16 full-size', (k, n, h, w), stats)
    for i, agree, err, acc, unexplained in stats:
        assert err < 2e-2, (i, err)                                # north_star bf16 logit gate
        assert agree >= 0.999, (i, agree)                          # north_star bf16 argmax gate, as stated
        assert acc > 0.9, (i, acc)                                 # the weights ARE trained (margins are realistic)
        assert unexplained == 0, (i, unexplained)                  # diagnostic: every flip is a near-tie
    cm = _check_cm(pred, lab, k)
    assert int(cm.sum()) == int((lab != 255).sum())


def test_config2_bf16_batch16_1024x2048_vs_oracle():
    _run_bf16(19, 16, 1024, 2048, (8, 16), SCHED19, check=(0, 15))


def test_config5_bf16_batch128_512x512_vs_oracle():
    _run_bf16(2, 128, 512, 512, (4, 4), SCHED2, check=(0, 77, 127))


def test_config2_fp32_batch16_1024x2048_vs_oracle():
    o, m = _pair(19, 'fp32', SCHED19)
    img, lab = _scenes(16, 1024, 2048, 19, (8, 16), seed=500)
    x = oracle.preprocess(img)
    pred, logits = m.engine().forward_infer(x.to(DEV), want_logits=True)
    for i in (0, 15):
        ref_logits, ref_pred = o.predict(x[i:i + 1])
        err = rel_err(logits[i:i + 1].cpu(), ref_logits)
        assert err < 1e-4, (i, err)                                # north_star fp32 gate
        mism = pred[i].cpu().long() != ref_pred[0, 0]
        assert not (mism & ~near_tie_mask(ref_logits, 1e-4)[0]).any()
        assert mism.float().mean() < 1e-4
    _check_cm(pred, lab, 19)


def test_bf16_random_init_diagnostic():
    """Random-init weights (no trained margins): the bf16 engine must still be within the bf16 logit gate and every
    flip must be a near-tie; the agreement figure itself is only reported (DESIGN.md section 5)."""
    o, m = build_pair(19, dtype='bf16')
    img = synth.make_images_u8(16, 1024, 2048, seed=3)
    x = oracle.preprocess(img)
    pred, logits = m.engine().forward_infer(x.to(DEV), want_logits=True)
    ref_logits, ref_pred = o.predict(x[5:6])
    assert rel_err(logits[5:6].cpu(), ref_logits) < 2e-2
    mism = pred[5].cpu().long() != ref_pred[0, 0]
    print('random-init bf16 agreement at 1024x2048:', 1 - mism.float().mean().item())
    assert not (mism & ~near_tie_mask(ref_logits, 4e-2)[0]).any()
    assert mism.float().mean() < 0.01
