#!/usr/bin/env python
"""SegLocalVisualizer's device path (what `tools/test.py --show-dir` draws) against mmseg's drawing restated on the host.

    python tools/bench_visualize.py [--min-seconds 2.0] [--oracle-images 2]

Workload: 16 seeded 1024x2048 images (tests/vis_oracle.py photo) with 19-class blocky gt and pred maps (16-pixel cells,
5 % ignore pixels in the gt), both panels drawn (a 1024x4096 picture per image), Cityscapes classes and palette.
Reported:
  * batch_ms_labels / batch_ms_no_labels: one SegLocalVisualizer.add_datasamples call over the 16 images with a
    LocalVisBackend writing into a temporary directory: locations (with labels: one locate call and its copy back, the
    cv2 stamps, their upload), the overlay, the RGB PNG encode, the copy back and the 16 file writes; host wall clock
    from the call to its return (every step ends in a device synchronise), mean over repetitions of at least
    --min-seconds;
  * locate_ms, overlay_ms, encode_ms: the three device calls alone on the same batch (CUDA events; locate_ms and
    encode_ms include their copies back);
  * stamp_batch_ms: the labels' whole share: the locate call, its copy back, the cv2 stamps and their upload (wall);
  * files_equal_oracle: the first --oracle-images files written with labels decode to the oracle's pictures;
  * oracle_ms_per_image: the numpy + cv2 restatement (both panels with labels) plus cv2.imwrite of the picture, per
    image, on one host thread;
  * device_kb_per_image / cv2_kb_per_image: the PNG sizes of the same pictures, ours and cv2.imwrite's (level 1
    default);
  * the GPU name and power limit, read in the same run.
Prints ONE JSON line.  Writes nothing to the tree.
"""
import argparse
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from bench_png_decode import gpu_info, timed  # noqa: E402


def wall(fn, min_seconds):
    import torch
    fn()
    torch.cuda.synchronize()
    t0, reps = time.perf_counter(), 0
    while time.perf_counter() - t0 < min_seconds or reps < 3:
        fn()
        torch.cuda.synchronize()
        reps += 1
    return (time.perf_counter() - t0) / reps * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--min-seconds', type=float, default=2.0)
    ap.add_argument('--oracle-images', type=int, default=2)
    args = ap.parse_args()
    import cv2
    import numpy as np
    import torch
    from lednet_b200 import ops, visualization as V
    import vis_oracle as O

    if not torch.cuda.is_available():
        raise SystemExit('bench_visualize measures on a CUDA device')
    res = dict(bench='visualize', batch=16, shape=[1024, 2048], panels=2, classes=19, **gpu_info(),
               torch_device=torch.cuda.get_device_name(0))
    n, h, w = 16, 1024, 2048
    imgs = [O.photo(h, w, seed=i) for i in range(n)]
    gts = [O.blocky_map(h, w, 19, seed=100 + i) for i in range(n)]
    preds = [O.blocky_map(h, w, 19, seed=200 + i, ignore=0) for i in range(n)]
    dev = torch.device('cuda', 0)
    timgs = [torch.from_numpy(np.ascontiguousarray(im[..., ::-1].transpose(2, 0, 1))).to(dev) for im in imgs]
    samples = [dict(gt_sem_seg=dict(data=torch.from_numpy(g)[None].to(dev)),
                    pred_sem_seg=dict(data=torch.from_numpy(p.astype(np.int64))[None].to(dev)))
               for g, p in zip(gts, preds)]
    names = [f'img{i}.png' for i in range(n)]
    with tempfile.TemporaryDirectory() as tmp:
        vis = V.SegLocalVisualizer(save_dir=tmp, vis_backends=[dict(type='LocalVisBackend')])
        for key, labels in (('batch_ms_no_labels', False), ('batch_ms_labels', True)):
            res[key] = round(wall(lambda: vis.add_datasamples(names, timgs, samples, list(range(n)),
                                                              with_labels=labels), args.min_seconds), 2)
        img_dir = vis.get_backend('LocalVisBackend').img_dir
        files = [open(os.path.join(img_dir, f'{nm}_{i}.png'), 'rb').read() for i, nm in enumerate(names)]
        sizes = [len(f) for f in files]
    res['images_per_s_labels'] = round(n / res['batch_ms_labels'] * 1e3, 1)
    res['device_kb_per_image'] = round(float(np.mean(sizes)) / 1e3, 1)

    x = torch.stack(timgs)
    g = torch.stack([s['gt_sem_seg']['data'][0] for s in samples])
    p = torch.stack([s['pred_sem_seg']['data'][0] for s in samples])
    both = torch.cat([g.to(torch.int64), p])
    res['locate_ms'] = round(timed(lambda: ops.seg_label_locations(both, 19).cpu(), args.min_seconds), 3)
    res['stamp_batch_ms'] = round(wall(lambda: vis._stamp_batch(g, p, V.CITYSCAPES_CLASSES, (h, w)),
                                       args.min_seconds), 2)
    palette, table = vis._tables(dev)
    res['overlay_ms'] = round(timed(lambda: ops.seg_overlay(x, g, p, palette, table), args.min_seconds), 3)
    drawn = ops.seg_overlay(x, g, p, palette, table)
    res['encode_ms'] = round(timed(lambda: ops.png_encode(drawn), args.min_seconds), 2)

    k = args.oracle_images
    t0 = time.perf_counter()
    with tempfile.TemporaryDirectory() as tmp:
        for i in range(k):
            pic = O.add_datasample(imgs[i], gts[i], preds[i])
            cv2.imwrite(os.path.join(tmp, f'{i}.png'), cv2.cvtColor(pic, cv2.COLOR_RGB2BGR))
    res['oracle_ms_per_image'] = round((time.perf_counter() - t0) / k * 1e3, 1)
    ref = [O.add_datasample(imgs[i], gts[i], preds[i]) for i in range(k)]
    res['cv2_kb_per_image'] = round(float(np.mean([len(O.local_file(r)) for r in ref])) / 1e3, 1)
    dec = [cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_COLOR)[..., ::-1] for f in files[:k]]
    res['files_equal_oracle'] = all(np.array_equal(a, b) for a, b in zip(dec, ref))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
