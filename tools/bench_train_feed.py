#!/usr/bin/env python
"""Training feed benchmark: the Cityscapes train_pipeline augmentations (RandomResize (2048, 1024) x [0.5, 2.0],
RandomCrop 1024x1024 with cat_max_ratio 0.75, RandomFlip 0.5, PhotoMetricDistortion) plus SegDataPreProcessor on the
device (DeviceAugSegDataPreProcessor), for a batch of 12 decoded 1024x2048 uint8 images and label maps, K = 19.
Prints one JSON line: the augmentation time per batch (CUDA events, host parameter draws included), its algorithmic
bytes and GB/s, the training step fed by it next to the step on synthetic, already normalised input, the numpy
restatement's host ms per image (tests/augment_oracle.py, one thread), and the GPU name / power limit.

    python tools/bench_train_feed.py [--batch 12] [--steps 20] [--warmup 3] [--out profiles/train_feed_1gpu.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

PIPELINE = [dict(type='RandomResize', scale=(2048, 1024), ratio_range=(0.5, 2.0), keep_ratio=True),
            dict(type='RandomCrop', crop_size=(1024, 1024), cat_max_ratio=0.75),
            dict(type='RandomFlip', prob=0.5),
            dict(type='PhotoMetricDistortion')]


def gpu_info():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:                                        # noqa: BLE001
        return f'unavailable ({e})'


def algorithmic_bytes(params, shapes, crop, Hp, Wp, label_bytes):
    """outputs written (fp32 image + int64 label) + the source pixels under each chosen box (3 image bytes + the label)
    + the source label pixels under every checked candidate box"""
    total = 12 * Hp * Wp * len(params)
    for p, (h, w) in zip(params, shapes):
        rh, rw = p['resized_hw']
        eh, ew = min(crop[0], rh), min(crop[1], rw)
        foot = min(h, -(-eh * h // rh) + 1) * min(w, -(-ew * w // rw) + 1)
        total += foot * (3 + label_bytes) + foot * label_bytes * (len(p['candidates']) - 1)
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=12)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--host-images', type=int, default=2, help='images timed through the numpy restatement')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import lednet_b200 as L
    from lednet_b200 import synth
    assert torch.cuda.is_available(), 'this benchmark measures the B200: no CUDA device found'
    dev = torch.device('cuda', 0)
    N, H, W, K = args.batch, 1024, 2048, 19
    img = synth.make_images_u8(N, H, W, seed=100).to(dev)
    lab = synth.make_labels(N, H, W, K, seed=200).to(torch.uint8).to(dev)
    lab[:, :64] = 255
    mean, std = list(L.engine.MEAN), list(L.engine.STD)
    pp = L.DeviceAugSegDataPreProcessor(train_pipeline=PIPELINE, seed=0, mean=mean, std=std, bgr_to_rgb=True,
                                        size=(1024, 1024), pad_val=0, seg_pad_val=255)

    def feed():
        samples = [dict(gt_sem_seg=dict(data=lab[i:i + 1])) for i in range(N)]
        return pp(dict(inputs=list(img.unbind(0)), data_samples=samples), training=True)

    # -- augmentation alone
    for _ in range(args.warmup):
        feed()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nbytes = 0
    e0.record()
    for _ in range(args.steps):
        d = feed()
        p = [s['metainfo']['aug_params'] for s in d['data_samples']]
        nbytes += algorithmic_bytes(p, [(H, W)] * N, (1024, 1024), 1024, 1024, 1)
    e1.record()
    torch.cuda.synchronize()
    aug_ms = e0.elapsed_time(e1) / args.steps
    gbps = nbytes / args.steps / (aug_ms * 1e-3) / 1e9

    # -- training step: synthetic normalised input vs fed by the augmentation
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        m = L.EncoderDecoder(dict(type='LEDNet'),
                             dict(type='LEDHead', in_channels=128, channels=64, num_classes=K, dropout_ratio=0.),
                             data_preprocessor=None, compute_dtype='fp32')
    m.load_state_dict(synth.make_state_dict(m.state_dict(), seed=2))
    m.to(dev).train()
    opt = L.FlatSGD(m.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4)
    s_img = synth.make_images_u8(N, 1024, 1024, seed=300).to(dev)
    mt, st = torch.tensor(mean, device=dev).view(1, 3, 1, 1), torch.tensor(std, device=dev).view(1, 3, 1, 1)
    x_syn = ((s_img[:, [2, 1, 0]].float() - mt) / st).contiguous()
    l_syn = synth.make_labels(N, 1024, 1024, K, seed=301).to(dev)
    syn_samples = [dict(gt_sem_seg=dict(data=l_syn[i:i + 1])) for i in range(N)]

    def step(data):
        total, log = m.parse_losses(m.loss(data['inputs'], data['data_samples']))
        opt.zero_grad()
        total.backward()
        opt.step()
        return log

    def timed(make):
        for _ in range(args.warmup):
            step(make())
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            step(make())
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    syn_ms = timed(lambda: dict(inputs=x_syn, data_samples=syn_samples))
    fed_ms = timed(feed)

    # -- the numpy restatement on the host, one thread
    import augment_oracle as A
    from lednet_b200.augment import draw_sample
    A._fma_tables()
    rng = np.random.default_rng(0)
    img_np, lab_np = img[:args.host_images].cpu().numpy(), lab[:args.host_images].cpu().numpy()
    t0 = time.perf_counter()
    for i in range(args.host_images):
        p = draw_sample(rng, pp.aug, H, W)
        A.augment(img_np[i], lab_np[i], p, (1024, 1024), 0.75)
    host_ms = (time.perf_counter() - t0) * 1e3 / args.host_images

    res = dict(metric='LED-Net train feed: device augmentation ms / batch', value=aug_ms, unit='ms', batch=N,
               source=f'{H}x{W} uint8 + uint8 labels', crop='1024x1024', steps=args.steps, warmup=args.warmup,
               aug_ms_per_batch=aug_ms, aug_algorithmic_bytes_per_batch=nbytes / args.steps, aug_gbps=gbps,
               train_step_ms_synthetic=syn_ms, train_step_ms_fed=fed_ms,
               train_img_s_synthetic=N / (syn_ms * 1e-3), train_img_s_fed=N / (fed_ms * 1e-3),
               restatement_host_ms_per_image=host_ms, restatement_images=args.host_images,
               dtype=L.train_ops.compute_mode(), gpu=gpu_info(), device=torch.cuda.get_device_name(0))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
