#!/usr/bin/env python
"""CityscapesMetric's device path against cityscapesscripts' evaluation restated on the host.

    python tools/bench_cityscapes_metric.py [--min-seconds 1.0]

Workload: seeded 2048x1024 Cityscapes-like scenes (tests/cityscapes_corpus.py: blocky labelIds with 32-pixel cells, 12
instance blobs and 2 crowd regions, trainId predictions with perturbed blocks), GT written by PIL (labelIds 8-bit,
instanceIds 16-bit), batches of 8 and 16 (8 distinct scenes, repeated for 16).  Reported per batch:
  * gt_label_decode_ms / gt_inst_decode_ms: one ops.png_decode call each ('label', 'grey16'), host parse, staging,
    upload and status read-back included, CUDA events over repetitions of at least --min-seconds;
  * accumulate_ms: ops.cityscapes_accumulate (uint8 and int64 predictions), the three kernels and the copy back, with
    the bytes the kernel reads (prediction + labelIds + instanceIds) and their rate;
  * encode_ms: ops.png_encode(lut=trainId -> labelId, palette=True) with the files copied back;
  * combine_ms: the host's scores over the batch's records (lednet_b200.cityscapes.combine);
  * oracle_ms_per_image: the restated evaluatePair on the host, the three files decoded by PIL;
  * the GPU name and power limit, read in the same run.
Prints ONE JSON line.  Writes nothing to the tree.
"""
import argparse
import io
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from bench_png_decode import gpu_info, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--min-seconds', type=float, default=1.0)
    ap.add_argument('--oracle-images', type=int, default=3)
    args = ap.parse_args()
    import numpy as np
    import torch
    from PIL import Image
    from lednet_b200 import cityscapes as CS, ops
    import cityscapes_corpus as CC
    import cityscapes_oracle as O

    res = dict(bench='cityscapes_metric', shape=[1024, 2048], **gpu_info())
    if not torch.cuda.is_available():
        raise SystemExit('bench_cityscapes_metric measures on a CUDA device')
    h, w = 1024, 2048
    scenes = [CC.scene(h, w, seed=i) for i in range(8)]
    gt_files = [CC.pil_png(g) for g, _, _ in scenes]
    inst_files = [CC.pil16(i) for _, i, _ in scenes]
    res['gt_label_kb'] = round(float(np.mean([len(b) for b in gt_files])) / 1e3, 1)
    res['gt_inst_kb'] = round(float(np.mean([len(b) for b in inst_files])) / 1e3, 1)
    for n in (8, 16):
        gf, inf = (gt_files * 2)[:n], (inst_files * 2)[:n]
        r = {}
        r['gt_label_decode_ms'] = round(timed(lambda: ops.png_decode(gf, 'label'), args.min_seconds), 2)
        r['gt_inst_decode_ms'] = round(timed(lambda: ops.png_decode(inf, 'grey16'), args.min_seconds), 2)
        gt = torch.cat(ops.png_decode(gf, 'label'))
        inst = torch.cat(ops.png_decode(inf, 'grey16'))
        pred64 = torch.from_numpy(np.stack([(s[2]) for s in (scenes * 2)[:n]])).cuda()
        for name, pred in (('u8', pred64.to(torch.uint8)), ('i64', pred64)):
            ms = timed(lambda: ops.cityscapes_accumulate(pred, gt, inst, CS.TRAIN_TO_ID, CS.KERNEL_CATEGORY,
                                                         CS.KERNEL_RULE), args.min_seconds)
            nbytes = n * h * w * (pred.element_size() + 1 + 4)
            r[f'accumulate_{name}_ms'] = round(ms, 3)
            r[f'accumulate_{name}_bytes'] = nbytes
            r[f'accumulate_{name}_GBps'] = round(nbytes / ms / 1e6, 1)
        r['encode_ms'] = round(timed(lambda: ops.png_encode(pred64, lut=CS.TRAIN_TO_ID, palette=True),
                                     args.min_seconds), 2)
        cm, st, recs = ops.cityscapes_accumulate(pred64, gt, inst, CS.TRAIN_TO_ID, CS.KERNEL_CATEGORY, CS.KERNEL_RULE)
        assert not st.any()
        state = dict(cm=cm.cpu().numpy(), last_cm=np.zeros((34, 34), np.int64), records=recs)
        t0, reps = time.perf_counter(), 0
        while time.perf_counter() - t0 < args.min_seconds or reps < 3:
            CS.combine([state], n)
            reps += 1
        r['combine_ms'] = round((time.perf_counter() - t0) / reps * 1e3, 2)
        r['instances_per_image'] = round(sum(len(x) for x in recs) / n, 1)
        res[f'batch{n}'] = r
    preds = []
    for _, _, p in scenes[:args.oracle_images]:
        bio = io.BytesIO()
        Image.fromarray(O.convert_to_label_id(p)).convert('P').save(bio, format='PNG')
        preds.append(bio.getvalue())
    t0 = time.perf_counter()
    cm, stats = O.generate_matrix(), O.generate_instance_stats()
    for pb, gb, ib in zip(preds, gt_files, inst_files):
        arrs = [np.array(Image.open(io.BytesIO(b))) for b in (pb, gb, ib)]
        O.evaluate_pair(arrs[0], arrs[1], arrs[2], cm, stats)
    res['oracle_ms_per_image'] = round((time.perf_counter() - t0) / len(preds) * 1e3, 1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
