#!/usr/bin/env python
"""PNG decoding of the dataset feed (ops.png_decode, PackSegPNGFiles) on the device against cv2 on the host.

    python tools/bench_png_decode.py [--min-seconds 1.0]

Workload: seeded 2048x1024 RGB images (a gradient with blocks and noise, compressing like a street scene rather than
like noise) and blocky 19-class label maps (16x16 cells, 2 % ignore pixels), encoded by cv2 (default level and level 9)
and PIL (default).  Reported:
  * file sizes per encoder;
  * decode_ms per call of ops.png_decode for N = 12, 16, 64 files of each encoder (host IHDR parse, pinned staging, one
    upload, the two kernels, the status read-back), CUDA events over repetitions of at least --min-seconds; img/s; MB
    uploaded against MB decoded;
  * cv2_ms_per_image: cv2.imdecode(IMREAD_COLOR) on one host thread, and img/s with a thread pool of every host CPU;
  * feed: DeviceAugSegDataPreProcessor (the config's train pipeline, batch 12) from PackSegPNGFiles batches against the
    same batch from decoded images already on the host, ms per batch (host clock around a device synchronise);
  * the GPU name and power limit, read in the same run.
Prints ONE JSON line.  Writes nothing to the tree.
"""
import argparse
import io
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = (v.strip() for v in out.split(','))
        return dict(gpu=name, power_limit=plim, sm_clock_max=clk)
    except Exception as e:  # noqa: BLE001
        return dict(power_limit=f'unavailable ({type(e).__name__})')


def images(n, h=1024, w=2048, seed=0):
    import numpy as np
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    out = []
    for i in range(n):
        base = np.stack([(x * 3 + y + 17 * i) % 256, (y * 5 + x // 3) % 256, ((x // 7 + y // 5) * 37) % 256], -1)
        noise = rng.integers(0, 6, (h, w, 3)) * (rng.random((h, w, 1)) < 0.4)
        out.append(((base + noise) % 256).astype(np.uint8))
    return out


def labels(n, h=1024, w=2048, seed=1):
    import numpy as np
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        lab = np.kron(rng.integers(0, 19, (h // 16, w // 16)), np.ones((16, 16), np.int64))
        lab[rng.random((h, w)) < 0.02] = 255
        out.append(lab.astype(np.uint8))
    return out


def timed(fn, min_seconds):
    import torch
    fn()
    torch.cuda.synchronize()
    reps, total = 0, 0.0
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while total < min_seconds * 1e3 or reps < 3:
        s.record()
        fn()
        e.record()
        e.synchronize()
        total += s.elapsed_time(e)
        reps += 1
    return total / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--min-seconds', type=float, default=1.0)
    args = ap.parse_args()
    import cv2
    import numpy as np
    import torch
    from PIL import Image
    import lednet_b200 as L
    from lednet_b200 import ops
    assert torch.cuda.is_available(), 'bench_png_decode measures on a CUDA device'
    torch.cuda.set_device(0)
    cv2.setNumThreads(1)
    res = dict(workload='2048x1024 RGB images, 19-class label maps', **gpu_info())
    imgs, labs = images(16), labels(16)

    def pil(a):
        bio = io.BytesIO()
        Image.fromarray(a).save(bio, format='PNG')
        return bio.getvalue()

    enc = {
        'cv2_default': [cv2.imencode('.png', a)[1].tobytes() for a in imgs],
        'cv2_level9': [cv2.imencode('.png', a, [cv2.IMWRITE_PNG_COMPRESSION, 9])[1].tobytes() for a in imgs],
        'pil_default': [pil(a[..., ::-1]) for a in imgs],
    }
    lab_files = [pil(a) for a in labs]
    for k, fs in enc.items():                              # every encoder decodes to the same pixels
        for f, a in zip(fs[:2], imgs):
            assert np.array_equal(ops.png_decode([f])[0].cpu().numpy(), a.transpose(2, 0, 1)), k
    res['file_mb'] = {k: round(sum(map(len, fs)) / len(fs) / 1e6, 3) for k, fs in enc.items()}
    res['file_mb']['label_pil'] = round(sum(map(len, lab_files)) / len(lab_files) / 1e6, 4)
    decoded_mb = 1024 * 2048 * 3 / 1e6
    res['decoded_mb_per_image'] = decoded_mb
    dev = {}
    for k, fs in enc.items():
        for n in (12, 16, 64):
            batch = [fs[i % len(fs)] for i in range(n)]
            ms = timed(lambda: ops.png_decode(batch), args.min_seconds)
            up = sum(map(len, batch)) / 1e6
            dev[f'{k}_n{n}'] = dict(decode_ms=round(ms, 3), img_per_s=round(n / ms * 1e3, 1),
                                    uploaded_mb=round(up, 2), decoded_mb=round(n * decoded_mb, 2))
    for n in (12, 64):
        batch = [lab_files[i % len(lab_files)] for i in range(n)]
        ms = timed(lambda: ops.png_decode(batch, 'label'), args.min_seconds)
        dev[f'label_pil_n{n}'] = dict(decode_ms=round(ms, 3), img_per_s=round(n / ms * 1e3, 1))
    res['device'] = dev
    host = {}
    for k, fs in enc.items():
        bufs = [np.frombuffer(f, np.uint8) for f in fs]
        t = time.perf_counter()
        for b in bufs[:6]:
            cv2.imdecode(b, cv2.IMREAD_COLOR)
        one = (time.perf_counter() - t) / 6
        nthreads = os.cpu_count() or 1
        work = bufs * max(1, (2 * nthreads) // len(bufs))
        with ThreadPoolExecutor(nthreads) as ex:
            list(ex.map(lambda b: cv2.imdecode(b, cv2.IMREAD_COLOR), work[:nthreads]))
            t = time.perf_counter()
            list(ex.map(lambda b: cv2.imdecode(b, cv2.IMREAD_COLOR), work))
            pool = len(work) / (time.perf_counter() - t)
        host[k] = dict(cv2_ms_per_image=round(one * 1e3, 2), threads=nthreads, pool_img_per_s=round(pool, 1))
    res['host'] = host
    # the preprocessor fed files against the same batch decoded on the host
    import tempfile
    train = [dict(type='RandomResize', scale=(2048, 1024), ratio_range=(0.5, 2.0), keep_ratio=True),
             dict(type='RandomCrop', crop_size=(1024, 1024), cat_max_ratio=0.75),
             dict(type='RandomFlip', prob=0.5), dict(type='PhotoMetricDistortion')]
    N = 12
    with tempfile.TemporaryDirectory() as d:
        items = []
        for i in range(N):
            ip, lp = os.path.join(d, f'{i}.png'), os.path.join(d, f'{i}_gt.png')
            open(ip, 'wb').write(enc['cv2_default'][i % 16])
            open(lp, 'wb').write(lab_files[i % 16])
            items.append(L.PackSegPNGFiles()(dict(img_path=ip, seg_map_path=lp, reduce_zero_label=False)))
        dec_imgs = [torch.from_numpy(np.ascontiguousarray(imgs[i % 16].transpose(2, 0, 1))).pin_memory() for i in range(N)]
        dec_labs = [torch.from_numpy(labs[i % 16][None]).pin_memory() for i in range(N)]

        def feed(files):
            pp = L.DeviceAugSegDataPreProcessor(train_pipeline=train, seed=0, size=(1024, 1024), bgr_to_rgb=True,
                                                mean=[123.675, 116.28, 103.53], std=[58.395, 57.12, 57.375])

            def run():
                if files:
                    batch = dict(inputs=[it['inputs'] for it in items],
                                 data_samples=[dict(it['data_samples']) for it in items])
                else:
                    batch = dict(inputs=list(dec_imgs), data_samples=[dict(gt_sem_seg=dict(data=l)) for l in dec_labs])
                out = pp(batch, training=True)
                torch.cuda.synchronize()
                return out
            run()
            t = time.perf_counter()
            k = 0
            while time.perf_counter() - t < args.min_seconds or k < 3:
                run()
                k += 1
            return (time.perf_counter() - t) / k * 1e3, pp

        ms_files, _ = feed(True)
        ms_dec, _ = feed(False)
        a = L.DeviceAugSegDataPreProcessor(train_pipeline=train, seed=0, size=(1024, 1024))(
            dict(inputs=[it['inputs'] for it in items], data_samples=[dict(it['data_samples']) for it in items]), True)
        b = L.DeviceAugSegDataPreProcessor(train_pipeline=train, seed=0, size=(1024, 1024))(
            dict(inputs=list(dec_imgs), data_samples=[dict(gt_sem_seg=dict(data=l)) for l in dec_labs]), True)
        same = torch.equal(a['inputs'], b['inputs']) and all(
            torch.equal(x['gt_sem_seg']['data'], y['gt_sem_seg']['data']) for x, y in zip(a['data_samples'], b['data_samples']))
    res['feed_batch12'] = dict(from_files_ms=round(ms_files, 2), from_decoded_pinned_ms=round(ms_dec, 2),
                               identical_batches=bool(same))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
