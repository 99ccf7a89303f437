#!/usr/bin/env python
"""Multi-scale + flip test-time augmentation throughput (SegTTAModel over the fused engine + tta_merge_kernel).

    python tools/bench_tta.py [--batch 2] [--height 1024] [--width 2048] [--min-seconds 1.0]

Workload: the mmseg base dataset configs' `tta_pipeline` - scale ratios 0.5 .. 1.75 x {no flip, horizontal flip} =
12 views per image - on seeded uint8 images of 1024x2048, K = 19, bf16 activations, batch 2 (random-init weights:
the throughput does not depend on them).  The views are resized and flipped on the device BEFORE the timed region
(F.interpolate, test plumbing standing in for the CPU pipeline's cv2 Resize, which is not what is measured) and
normalised like SegDataPreProcessor.  Timed with CUDA events:
  * tta: SegTTAModel.predict_labels over all 12 views (6 engine calls, one per flip pair, + ONE tta_merge launch);
  * per ratio group: module.inference of the flip pair (2 x batch images, fp32 logits exported);
  * merge: ops.tta_merge alone (labels only) with its algorithmic bytes (every view's fp32 logits read once + the
    uint8 labels written) and the achieved GB/s, against MEASURED_PEAKS.json when present;
  * single: the plain single-view fused path (forward_infer, labels only) at the same batch, for contrast.
The fields above keep those definitions.  The views built on the device (SegTTAModel(tta_transforms=...)) add:
  * view_build: all 12 views of the batch through ops.view_resize (one launch per ratio writes the flip pair), with
    its algorithmic bytes (the uint8 sources read once per ratio + the fp32 views written) and the achieved GB/s;
  * tta_device_views: SegTTAModel.predict_image_labels from device-resident uint8 images, view building included;
  * tta_device_views_from_host: the same from pinned host uint8 images, one upload of the N images per step;
  * host_views_ms_per_image: what a dataloader worker does per image for TestTimeAug on one host thread (6 cv2.resize
    INTER_LINEAR + 6 flips + 12 HWC -> CHW packs), and upload_bytes_per_image: the 12 uint8 views against the image.
Prints ONE JSON line; the GPU name and power limit are read in the same run.  Writes nothing to the tree.
"""
import argparse
import json
import os
import subprocess
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RATIOS = (0.5, 0.75, 1.0, 1.25, 1.5, 1.75)


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = (s.strip() for s in out.split(','))
        return dict(gpu=name, power_limit=plim, sm_clock_max=clk)
    except Exception as e:                  # the name from torch still identifies the card
        return dict(power_limit=f'unavailable ({type(e).__name__})')


def timed(fn, min_seconds, min_steps=5):
    """mean ms per call of fn over at least min_seconds (CUDA events), after one warm call."""
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    steps = max(min_steps, int(min_seconds * 1000.0 / max(e0.elapsed_time(e1), 1e-3)) + 1)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, steps


def host_views_ms(img_hwc, sizes, repeats=3):
    """ms per image of TestTimeAug's per-image host work on one thread: per ratio cv2.resize (INTER_LINEAR), np.flip
    (mmcv.imflip) and PackSegInputs' np.ascontiguousarray(img.transpose(2, 0, 1)) of both views"""
    import time
    import cv2
    import numpy as np
    cv2.setNumThreads(0)                                  # OpenCV runs sequentially on the calling thread
    best = float('inf')
    for _ in range(repeats):
        t0 = time.perf_counter()
        for rh, rw in sizes:
            v = cv2.resize(img_hwc, (rw, rh), interpolation=cv2.INTER_LINEAR)
            for x in (v, np.flip(v, axis=1)):
                np.ascontiguousarray(x.transpose(2, 0, 1))
        best = min(best, (time.perf_counter() - t0) * 1e3)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=2)
    ap.add_argument('--height', type=int, default=1024)
    ap.add_argument('--width', type=int, default=2048)
    ap.add_argument('--min-seconds', type=float, default=1.0)
    args = ap.parse_args()

    import torch
    import torch.nn.functional as F
    import lednet_b200 as L
    from lednet_b200 import ops, synth
    from lednet_b200.augment import view_size

    if not torch.cuda.is_available():
        raise SystemExit('bench_tta.py measures on the GPU; no CUDA device found')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    N, H, W, K = args.batch, args.height, args.width, 19
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        m = L.EncoderDecoder(dict(type='LEDNet'), dict(type='LEDHead', in_channels=128, channels=64, num_classes=K,
                                                       dropout_ratio=0.),
                             data_preprocessor=dict(type='SegDataPreProcessor', mean=list(L.engine.MEAN),
                                                    std=list(L.engine.STD), bgr_to_rgb=True),
                             compute_dtype='bf16').eval()
    m.load_state_dict(synth.make_state_dict(m.state_dict(), seed=2))
    m.to(dev)
    tta = L.SegTTAModel(m)

    img_host = synth.make_images_u8(N, H, W, seed=100)
    img = img_host.to(dev)
    mean = torch.tensor(L.engine.MEAN, device=dev).view(1, 3, 1, 1)
    std = torch.tensor(L.engine.STD, device=dev).view(1, 3, 1, 1)

    def norm(u8):
        return ((u8[:, [2, 1, 0]].float() - mean) / std).contiguous()

    views, metas = [], []
    for r in RATIOS:
        hw = (int(H * r + 0.5), int(W * r + 0.5))
        base = img if r == 1.0 else \
            F.interpolate(img.float(), size=hw, mode='bilinear', align_corners=False).round().clamp(0, 255).to(torch.uint8)
        for flip in (False, True):
            views.append(norm(base.flip(dims=(3,)) if flip else base))
            metas.append([dict(ori_shape=(H, W), flip=flip, flip_direction='horizontal') for _ in range(N)])
    pred = torch.empty((N, H, W), dtype=torch.uint8, device=dev)
    tta_cfg = [[dict(type='Resize', scale_factor=r, keep_ratio=True) for r in RATIOS],
               [dict(type='RandomFlip', prob=0., direction='horizontal'),
                dict(type='RandomFlip', prob=1., direction='horizontal')]]
    tta_dev = L.SegTTAModel(m, tta_transforms=tta_cfg)
    sizes = [view_size(H, W, ('scale_factor', r)) for r in RATIOS]

    with torch.no_grad():
        # warm every view shape (engine plans are built per input shape)
        tta.predict_labels(views, metas, pred=pred)
        torch.cuda.synchronize()
        tta_ms, tta_steps = timed(lambda: tta.predict_labels(views, metas, pred=pred), args.min_seconds)

        group_ms = {}
        for j, r in enumerate(RATIOS):
            pair = torch.cat([views[2 * j], views[2 * j + 1]], 0)
            group_ms[str(r)] = round(timed(lambda: m.inference(pair), args.min_seconds / 4)[0], 3)
            del pair

        logits = tta._view_logits(views)
        desc = [(lg, None, 'horizontal' if v % 2 else None) for v, lg in enumerate(logits)]
        merge_ms, merge_steps = timed(lambda: ops.tta_merge(desc, (H, W), False, 0, 0.3, pred=pred),
                                      args.min_seconds)
        bytes_read = sum(lg.numel() * 4 for lg in logits)
        merge_bytes = bytes_read + N * H * W
        del logits, desc

        x1 = views[4]                                        # ratio 1.0, unflipped
        eng = m.engine()
        single_ms, _ = timed(lambda: eng.forward_infer(x1, pred=pred), args.min_seconds)
        n_views = len(views)
        del views, x1

        # the 12 views built on the device: one view_resize per ratio, the flip pair in one [2N, 3, rh, rw] batch
        pp = m.data_preprocessor
        mean_l, std_l = pp.mean_std()
        vbufs = [torch.empty((2 * N, 3, rh, rw), dtype=torch.float32, device=dev) for rh, rw in sizes]
        imgs = list(img)

        def build_views():
            for (rh, rw), x in zip(sizes, vbufs):
                ops.view_resize(imgs, (rh, rw), out=x[:N], out_flip=x[N:], swap_rb=True, mean=mean_l, std=std_l)
        view_ms, view_steps = timed(build_views, args.min_seconds)
        view_bytes = len(sizes) * N * 3 * H * W + sum(x.numel() * 4 for x in vbufs)
        del vbufs

        dmetas = [dict(ori_shape=(H, W)) for _ in range(N)]
        tta_dev.predict_image_labels(img, dmetas, pred=pred)
        torch.cuda.synchronize()
        dev_ms, dev_steps = timed(lambda: tta_dev.predict_image_labels(img, dmetas, pred=pred), args.min_seconds)
        pinned = img_host.pin_memory()
        host_ms, host_steps = timed(lambda: tta_dev.predict_image_labels(pinned.to(dev, non_blocking=True), dmetas,
                                                                         pred=pred), args.min_seconds)
    try:
        host_views = round(host_views_ms(img_host[0].permute(1, 2, 0).contiguous().numpy(), sizes), 2)
    except ImportError as e:
        host_views = f'not measured ({e})'

    gbs = merge_bytes / (merge_ms * 1e-3) / 1e9
    peak, src = 6650.0, 'fallback'
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        peak, src = float(json.load(open(p))['hbm_gbs']), 'MEASURED_PEAKS.json'
    out = dict(metric='LED-Net TTA img/s @1024x2048 bf16 (6 ratios x flip)', batch=N, height=H, width=W,
               num_classes=K, views=n_views,
               tta_img_s=round(N / (tta_ms * 1e-3), 2), tta_ms_per_batch=round(tta_ms, 3), tta_steps=tta_steps,
               inference_ms_per_ratio_pair=group_ms,
               merge_ms=round(merge_ms, 4), merge_steps=merge_steps, merge_bytes=merge_bytes,
               merge_gbs=round(gbs, 1), merge_hbm_peak_gbs=peak, merge_peak_source=src,
               merge_share_of_hbm_peak=round(gbs / peak, 3),
               single_view_img_s=round(N / (single_ms * 1e-3), 2), single_view_ms_per_batch=round(single_ms, 3),
               view_build_ms=round(view_ms, 4), view_build_steps=view_steps, view_build_bytes=view_bytes,
               view_build_gbs=round(view_bytes / (view_ms * 1e-3) / 1e9, 1),
               tta_device_views_img_s=round(N / (dev_ms * 1e-3), 2), tta_device_views_ms_per_batch=round(dev_ms, 3),
               tta_device_views_steps=dev_steps,
               tta_device_views_from_host_img_s=round(N / (host_ms * 1e-3), 2),
               tta_device_views_from_host_ms_per_batch=round(host_ms, 3), tta_device_views_from_host_steps=host_steps,
               host_views_ms_per_image=host_views,
               upload_bytes_per_image=dict(views=2 * sum(3 * rh * rw for rh, rw in sizes), image=3 * H * W),
               torch_device=torch.cuda.get_device_name(dev), **gpu_info())
    print(json.dumps(out))


if __name__ == '__main__':
    main()
