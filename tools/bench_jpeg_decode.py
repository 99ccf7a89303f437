#!/usr/bin/env python
"""JPEG decoding of the dataset feed (ops.jpeg_decode, PackSegFiles) on the device against cv2 on the host.

    python tools/bench_jpeg_decode.py [--min-seconds 1.0] [--stages]

Workload: seeded photo-like images (smooth colour gradients, edges, mild noise) at 500x375 (Pascal VOC-sized) and
2048x1024, encoded three ways: cv2 defaults (quality 95, 4:2:0), PIL defaults (quality 75, 4:2:0) and cv2 quality 95 at
4:4:4.  Reported:
  * file sizes per encoder;
  * decode_ms per call of ops.jpeg_decode for N = 16, 64 (500x375) and N = 12, 16, 64 (2048x1024) files of each
    encoder (host marker walk, pinned staging, one upload, the five kernels, the status read-back), CUDA events over
    repetitions of at least --min-seconds; img/s; MB uploaded against MB decoded;
  * cv2_ms_per_image: cv2.imdecode(IMREAD_COLOR) on one host thread, and img/s with a thread pool of every host CPU;
  * feed: DeviceAugSegDataPreProcessor (the config's train pipeline, batch 12 of 2048x1024) from PackSegFiles batches of
    cv2-default JPEG files against the same batch from decoded images already pinned on the host, ms per batch (host
    clock around a device synchronise), and whether the two batches are identical;
  * the GPU name and power limit, read in the same run.
--stages instead profiles one workload (16 cv2-default 2048x1024 files) with torch.profiler and reports the device
time of each decoder kernel per call: which stage bounds the decode.
Prints ONE JSON line.  Writes nothing to the tree.
"""
import argparse
import json
import os
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from bench_png_decode import gpu_info, timed  # noqa: E402


def encoders(imgs):
    import jpeg_corpus as J
    return {
        'cv2_default': [J.cv2_jpeg(a, 95) for a in imgs],
        'pil_default': [J.pil_jpeg(a) for a in imgs],
        'cv2_q95_444': [J.cv2_jpeg(a, 95, '444') for a in imgs],
    }


def stages(args):
    import torch
    from torch.profiler import ProfilerActivity, profile
    import jpeg_corpus as J
    from lednet_b200 import ops
    files = encoders([J.photo(1024, 2048, seed=s) for s in range(16)])['cv2_default']
    for _ in range(2):
        ops.jpeg_decode(files)
    torch.cuda.synchronize()
    reps = 10
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ops.jpeg_decode(files)
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        if 'jpeg_' in e.key:
            name = e.key.split('jpeg_')[1].split('(')[0].split('<')[0]
            per['jpeg_' + name] = round(e.device_time_total / 1e3 / reps, 3)
    ms = timed(lambda: ops.jpeg_decode(files), args.min_seconds)
    return dict(workload='16 x 2048x1024 cv2-default JPEG files (quality 95, 4:2:0)', **gpu_info(),
                kernel_ms_per_call=per, decode_ms_per_call=round(ms, 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--min-seconds', type=float, default=1.0)
    ap.add_argument('--stages', action='store_true')
    args = ap.parse_args()
    import cv2
    import numpy as np
    import torch
    import lednet_b200 as L
    from lednet_b200 import ops
    import jpeg_corpus as J
    import png_corpus as P
    assert torch.cuda.is_available(), 'bench_jpeg_decode measures on a CUDA device'
    torch.cuda.set_device(0)
    if args.stages:
        print(json.dumps(stages(args)))
        return
    cv2.setNumThreads(1)
    res = dict(workload='photo-like images at 500x375 and 2048x1024; cv2 q95 4:2:0, PIL q75 4:2:0, cv2 q95 4:4:4',
               **gpu_info())
    sizes = {'500x375': (375, 500), '2048x1024': (1024, 2048)}
    counts = {'500x375': (16, 64), '2048x1024': (12, 16, 64)}
    imgs = {k: [J.photo(h, w, seed=s) for s in range(16)] for k, (h, w) in sizes.items()}
    enc = {k: encoders(v) for k, v in imgs.items()}
    for k, by_enc in enc.items():                          # every encoder's files decode to cv2's pixels
        for e, fs in by_enc.items():
            for f, o in zip(fs[:2], ops.jpeg_decode(fs[:2])):
                assert np.array_equal(o.cpu().numpy(), J.cv2_ref(f)), (k, e)
    res['file_mb'] = {f'{k}_{e}': round(sum(map(len, fs)) / len(fs) / 1e6, 4) for k, v in enc.items()
                      for e, fs in v.items()}
    dev, host = {}, {}
    nthreads = os.cpu_count() or 1
    for k, by_enc in enc.items():
        h, w = sizes[k]
        decoded_mb = h * w * 3 / 1e6
        for e, fs in by_enc.items():
            for n in counts[k]:
                batch = [fs[i % len(fs)] for i in range(n)]
                ms = timed(lambda: ops.jpeg_decode(batch), args.min_seconds)
                dev[f'{k}_{e}_n{n}'] = dict(decode_ms=round(ms, 3), img_per_s=round(n / ms * 1e3, 1),
                                            uploaded_mb=round(sum(map(len, batch)) / 1e6, 2),
                                            decoded_mb=round(n * decoded_mb, 2))
            bufs = [np.frombuffer(f, np.uint8) for f in fs]
            t = time.perf_counter()
            for b in bufs[:8]:
                cv2.imdecode(b, cv2.IMREAD_COLOR)
            one = (time.perf_counter() - t) / 8
            work = bufs * max(1, (4 * nthreads) // len(bufs))
            with ThreadPoolExecutor(nthreads) as ex:
                list(ex.map(lambda b: cv2.imdecode(b, cv2.IMREAD_COLOR), work[:nthreads]))
                t = time.perf_counter()
                list(ex.map(lambda b: cv2.imdecode(b, cv2.IMREAD_COLOR), work))
                pool = len(work) / (time.perf_counter() - t)
            host[f'{k}_{e}'] = dict(cv2_ms_per_image=round(one * 1e3, 3), threads=nthreads,
                                    pool_img_per_s=round(pool, 1), pool_ms_per_16=round(16 / pool * 1e3, 2))
    res['device'] = dev
    res['host'] = host
    # the preprocessor fed JPEG files against the same batch decoded on the host
    train = [dict(type='RandomResize', scale=(2048, 1024), ratio_range=(0.5, 2.0), keep_ratio=True),
             dict(type='RandomCrop', crop_size=(1024, 1024), cat_max_ratio=0.75),
             dict(type='RandomFlip', prob=0.5), dict(type='PhotoMetricDistortion')]
    N = 12
    files = enc['2048x1024']['cv2_default']
    labs = [P.blocky_labels(1024, 2048, seed=40 + i) for i in range(16)]
    with tempfile.TemporaryDirectory() as d:
        items = []
        for i in range(N):
            ip, lp = os.path.join(d, f'{i}.jpg'), os.path.join(d, f'{i}_gt.png')
            open(ip, 'wb').write(files[i % 16])
            open(lp, 'wb').write(P.png(labs[i % 16][..., None], 0, level=1))
            items.append(L.PackSegFiles()(dict(img_path=ip, seg_map_path=lp, reduce_zero_label=False)))
        dec_imgs = [torch.from_numpy(np.ascontiguousarray(J.cv2_ref(files[i % 16]))).pin_memory() for i in range(N)]
        dec_labs = [torch.from_numpy(labs[i % 16][None]).pin_memory() for i in range(N)]

        def batch(from_files):
            if from_files:
                return dict(inputs=[it['inputs'] for it in items], data_samples=[dict(it['data_samples']) for it in items])
            return dict(inputs=list(dec_imgs), data_samples=[dict(gt_sem_seg=dict(data=l)) for l in dec_labs])

        def pp():
            return L.DeviceAugSegDataPreProcessor(train_pipeline=train, seed=0, size=(1024, 1024), bgr_to_rgb=True,
                                                  mean=[123.675, 116.28, 103.53], std=[58.395, 57.12, 57.375])

        def feed(from_files):
            p = pp()
            p(batch(from_files), training=True)
            torch.cuda.synchronize()
            t = time.perf_counter()
            k = 0
            while time.perf_counter() - t < args.min_seconds or k < 3:
                p(batch(from_files), training=True)
                torch.cuda.synchronize()
                k += 1
            return (time.perf_counter() - t) / k * 1e3

        ms_files, ms_dec = feed(True), feed(False)
        a, b = pp()(batch(True), True), pp()(batch(False), True)
        same = torch.equal(a['inputs'], b['inputs']) and all(
            torch.equal(x['gt_sem_seg']['data'], y['gt_sem_seg']['data'])
            for x, y in zip(a['data_samples'], b['data_samples']))
    res['feed_batch12_2048x1024'] = dict(from_files_ms=round(ms_files, 2), from_decoded_pinned_ms=round(ms_dec, 2),
                                         identical_batches=bool(same))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
