#!/usr/bin/env python
"""PNG output of label maps (IoUMetric(output_dir=...), `tools/test.py --out`): the device encoder against PIL.

    python tools/bench_png.py [--batch 16] [--height 1024] [--width 2048] [--min-seconds 1.0]

Workload: batches of seeded uint8 label maps of 1024x2048, one batch per kind:
  * blocky: 32x32 cells of 19 classes; smooth: a Gaussian field (sigma 30) cut into 19 levels; noise: uniform bytes,
    which takes the stored path (the worst case for the encoder's output size).
For each kind:
  * encode_ms: the launch sequence of ledb200_png_encode for the whole batch (filter, band, size, scan and assemble
    kernels), timed with CUDA events over repetitions of at least --min-seconds; the input GB/s counts the label bytes
    read once;
  * bytes: the files of the batch in total and per image;
  * copy_write_ms: ops.png_encode's two copies back (offsets, then the files) plus writing every file to a temporary
    directory, host clock after the encode, per batch;
  * pil_ms_per_image / pil_bytes at compress_level 1 and 6: `Image.fromarray(a).save(path)` on one host thread, as
    mmseg's IoUMetric writes a prediction, measured in the same run on a few maps of the batch.
Prints ONE JSON line; the GPU name and power limit are read in the same run.  Writes nothing to the tree.
"""
import argparse
import io
import json
import os
import subprocess
import sys
import tempfile
import time

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


def make_maps(kind, n, h, w):
    import numpy as np
    import scipy.ndimage as nd
    out = []
    for i in range(n):
        rng = np.random.default_rng(i)
        if kind == 'blocky':
            small = rng.integers(0, 19, (-(-h // 32), -(-w // 32)))
            a = np.kron(small, np.ones((32, 32), np.int64))[:h, :w]
        elif kind == 'smooth':
            f = nd.gaussian_filter(rng.standard_normal((h, w)), 30)
            a = np.digitize(f, np.linspace(f.min(), f.max(), 20)[1:-1])
        else:
            a = rng.integers(0, 256, (h, w))
        out.append(a.astype(np.uint8))
    return np.stack(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=16)
    ap.add_argument('--height', type=int, default=1024)
    ap.add_argument('--width', type=int, default=2048)
    ap.add_argument('--min-seconds', type=float, default=1.0)
    ap.add_argument('--pil-images', type=int, default=4)
    args = ap.parse_args()
    import torch
    from PIL import Image
    from lednet_b200 import lib, ops
    if not torch.cuda.is_available():
        raise SystemExit('bench_png needs a CUDA device')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    N, H, W = args.batch, args.height, args.width
    l = lib.get()
    bound = l.ledb200_png_bound(H, W)
    ws = torch.empty(l.ledb200_png_workspace_bytes(N, H, W), dtype=torch.uint8, device=dev)
    out = torch.empty(N * bound, dtype=torch.uint8, device=dev)
    offs = torch.empty(N + 1, dtype=torch.int64, device=dev)
    res = dict(bench='png_encode', batch=N, height=H, width=W, torch_device=torch.cuda.get_device_name(dev),
               **gpu_info())
    for kind in ('blocky', 'smooth', 'noise'):
        maps = make_maps(kind, N, H, W)
        t = torch.from_numpy(maps).to(dev)

        def enc():
            lib.check(l.ledb200_png_encode(t.data_ptr(), lib.U8, N, H, W, 0, out.data_ptr(), offs.data_ptr(),
                                           ws.data_ptr(), lib.stream_ptr(dev)), 'ledb200_png_encode')
        for _ in range(3):
            enc()
        torch.cuda.synchronize()
        reps, el = 4, 0.0
        while True:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                enc()
            e1.record()
            e1.synchronize()
            el = e0.elapsed_time(e1)
            if el >= args.min_seconds * 1e3:
                break
            reps *= 2
        enc_ms = el / reps
        # copies back + files
        files = ops.png_encode(t)
        torch.cuda.synchronize()
        cw = []
        with tempfile.TemporaryDirectory() as d:
            for r in range(5):
                enc()
                torch.cuda.synchronize()
                c0 = time.perf_counter()
                o = offs.cpu().tolist()
                data = out[:o[-1]].cpu().numpy().tobytes()
                for i in range(N):
                    with open(os.path.join(d, f'{r}_{i}.png'), 'wb') as f:
                        f.write(data[o[i]:o[i + 1]])
                cw.append((time.perf_counter() - c0) * 1e3)
        total = sum(len(b) for b in files)
        k = dict(encode_ms=round(enc_ms, 4), encode_reps=reps, input_gbps=round(maps.nbytes / enc_ms / 1e6, 2),
                 images_per_s=round(N / enc_ms * 1e3, 1), bytes_total=total, bytes_per_image=round(total / N, 1),
                 copy_write_ms=round(sorted(cw)[len(cw) // 2], 3))
        for level in (1, 6):
            ms, sizes = [], []
            for a in maps[:args.pil_images]:
                buf = io.BytesIO()
                c0 = time.perf_counter()
                Image.fromarray(a).save(buf, format='PNG', compress_level=level)
                ms.append((time.perf_counter() - c0) * 1e3)
                sizes.append(len(buf.getvalue()))
            k[f'pil{level}_ms_per_image'] = round(sum(ms) / len(ms), 2)
            k[f'pil{level}_bytes_per_image'] = round(sum(sizes) / len(sizes), 1)
        res[kind] = k
    print(json.dumps(res))


if __name__ == '__main__':
    main()
