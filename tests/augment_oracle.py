"""numpy restatement of the training augmentations (RandomResize -> RandomCrop -> RandomFlip -> PhotoMetricDistortion ->
SegDataPreProcessor) for explicit random parameters (lednet_b200.augment.draw_sample's dict), in cv2 4.x's own
integer and float arithmetic (see csrc/augment.cu).  tests/test_augment_host_cpu.py checks each operation against cv2;
tests/test_gpu_augment.py checks the kernels against this file bit for bit."""
from fractions import Fraction

import numpy as np

F32 = np.float32
HSV_SHIFT = 12
SDIV = np.array([0] + [int(np.rint((255 << HSV_SHIFT) / (1. * i))) for i in range(1, 256)], np.int64)
HDIV = np.array([0] + [int(np.rint((180 << HSV_SHIFT) / (6. * i))) for i in range(1, 256)], np.int64)


def cv_scale(src, dst):
    """cv2.resize's source-per-destination scale: 1 / (dst / src) in double"""
    return 1. / (dst / src)


def linear_coefs(src, dst):
    """INTER_LINEAR taps along one axis: (i0, i1, c0, c1), short coefficients out of 2048"""
    d = np.arange(dst, dtype=np.float64)
    f = ((d + 0.5) * cv_scale(src, dst) - 0.5).astype(F32)
    i = np.floor(f).astype(np.int64)
    f = (f - i.astype(F32)).astype(F32)
    lo, hi = i < 0, i >= src - 1
    f[lo], i[lo] = 0, 0
    f[hi], i[hi] = 0, src - 1
    c0 = np.rint((F32(1) - f) * F32(2048)).astype(np.int64)
    c1 = np.rint(f * F32(2048)).astype(np.int64)
    return i, np.minimum(i + 1, src - 1), c0, c1


def resize_linear(img, dh, dw):
    """cv2.resize(img, (dw, dh), INTER_LINEAR) of an [h, w, C] uint8 image, the SIMD rounding of the vertical pass"""
    h, w = img.shape[:2]
    x0, x1, a0, a1 = linear_coefs(w, dw)
    y0, y1, b0, b1 = linear_coefs(h, dh)
    im = img.astype(np.int64)
    hz = im[:, x0] * a0[None, :, None] + im[:, x1] * a1[None, :, None]
    s0, s1 = hz[y0], hz[y1]
    o = ((((s0 >> 4) * b0[:, None, None]) >> 16) + (((s1 >> 4) * b1[:, None, None]) >> 16) + 2) >> 2
    return np.clip(o, 0, 255).astype(np.uint8)


def nearest_index(src, dst):
    return np.minimum(np.floor(np.arange(dst) * cv_scale(src, dst)).astype(np.int64), src - 1)


def resize_nearest(lab, dh, dw):
    """cv2.resize(lab, (dw, dh), INTER_NEAREST)"""
    h, w = lab.shape[:2]
    return lab[nearest_index(h, dh)][:, nearest_index(w, dw)]


def bgr2hsv(img):
    """cv2.cvtColor(img, COLOR_BGR2HSV) of uint8 [..., 3]: the integer form"""
    b, g, r = (img[..., c].astype(np.int64) for c in range(3))
    v = np.maximum(np.maximum(b, g), r)
    diff = v - np.minimum(np.minimum(b, g), r)
    vr = np.where(v == r, -1, 0)
    vg = np.where(v == g, -1, 0)
    s = (diff * SDIV[v] + (1 << (HSV_SHIFT - 1))) >> HSV_SHIFT
    h = (vr & (g - b)) + (~vr & ((vg & (b - r + 2 * diff)) + (~vg & (r - g + 4 * diff))))
    h = (h * HDIV[diff] + (1 << (HSV_SHIFT - 1))) >> HSV_SHIFT
    h = h + np.where(h < 0, 180, 0)
    return np.stack([h, s, v], -1).astype(np.uint8)


_SECTOR = np.array([[1, 3, 0], [1, 0, 2], [3, 0, 1], [0, 2, 1], [0, 1, 3], [2, 1, 0]])
_FMA = None


def _fma_tables():
    """1 - s * hh and 1 - s * (1 - hh) with ONE rounding (cv2's vector code is contracted into FMA) for every
    (H < 180, S) pair, computed exactly in rationals and rounded once to float32"""
    global _FMA
    if _FMA is None:
        H, S = np.meshgrid(np.arange(180), np.arange(256), indexing='ij')
        sf = S.astype(F32) * F32(1 / 255.)
        hh = H.astype(F32) * F32(6 / 180.)
        hh = (hh - np.trunc(hh)).astype(F32)
        one_m = (F32(1) - hh).astype(F32)
        t2, t3 = np.empty((180, 256), F32), np.empty((180, 256), F32)
        for idx in np.ndindex(180, 256):
            s = Fraction(float(sf[idx]))
            t2[idx] = np.float32(_round_f32(1 - s * Fraction(float(hh[idx]))))
            t3[idx] = np.float32(_round_f32(1 - s * Fraction(float(one_m[idx]))))
        _FMA = t2, t3
    return _FMA


def _round_f32(q):
    """round a non-negative rational to the nearest float32 (ties to even)"""
    x = F32(float(q))                       # nearest double, then float32: may double-round, fixed below
    cands = [x, np.nextafter(x, F32(np.inf)), np.nextafter(x, F32(-np.inf))]
    best = min(cands, key=lambda c: (abs(Fraction(float(c)) - q), int(np.frombuffer(c.tobytes(), np.uint32)[0]) & 1))
    return best


def hsv2bgr(hsv):
    """cv2.cvtColor(hsv, COLOR_HSV2BGR) of uint8 [..., 3] with H < 180: the float SIMD form, truncated"""
    H, S, V = (hsv[..., c].astype(np.int64) for c in range(3))
    t2tab, t3tab = _fma_tables()
    sf = S.astype(F32) * F32(1 / 255.)
    vf = V.astype(F32) * F32(1 / 255.)
    hh = H.astype(F32) * F32(6 / 180.)
    sector = np.trunc(hh).astype(np.int64) % 6
    tab = np.stack([vf, vf * (F32(1) - sf), vf * t2tab[H, S], vf * t3tab[H, S]], -1).astype(F32)
    out = np.take_along_axis(tab, _SECTOR[sector], -1) * F32(255)
    return np.trunc(out.astype(F32)).astype(np.uint8)


def convert(img, alpha=1, beta=0):
    """PhotoMetricDistortion.convert: float32 x * alpha + beta (two roundings), clip, truncate to uint8"""
    x = img.astype(F32) * F32(alpha)
    x = (x + F32(beta)).astype(F32)
    return np.clip(x, 0, 255).astype(np.uint8)


def photometric(img, p):
    """PhotoMetricDistortion.transform of an [h, w, 3] BGR uint8 image with the drawn parameters"""
    if p['brightness'] is not None:
        img = convert(img, beta=p['brightness'])
    if p['contrast_mode'] == 1 and p['contrast'] is not None:
        img = convert(img, alpha=p['contrast'])
    if p['saturation'] is not None:
        hsv = bgr2hsv(img)
        hsv[..., 1] = convert(hsv[..., 1], alpha=p['saturation'])
        img = hsv2bgr(hsv)
    if p['hue'] is not None:
        hsv = bgr2hsv(img)
        hsv[..., 0] = (hsv[..., 0].astype(int) + p['hue']) % 180
        img = hsv2bgr(hsv)
    if p['contrast_mode'] == 0 and p['contrast'] is not None:
        img = convert(img, alpha=p['contrast'])
    return img


def crop_accepted(seg, cat_max_ratio, ignore_index=255):
    """RandomCrop's test of one box"""
    labels, cnt = np.unique(seg, return_counts=True)
    cnt = cnt[labels != ignore_index]
    return len(cnt) > 1 and np.max(cnt) / np.sum(cnt) < cat_max_ratio


def choose_crop(seg, candidates, crop_size, cat_max_ratio, ignore_index=255):
    """RandomCrop.crop_bbox's loop over pre-drawn boxes: the first of the first len - 1 that passes, else the last"""
    ch, cw = crop_size
    if cat_max_ratio < 1.:
        for k, (oy, ox) in enumerate(candidates[:-1]):
            if crop_accepted(seg[oy:oy + ch, ox:ox + cw], cat_max_ratio, ignore_index):
                return k
    return len(candidates) - 1


def augment(img_chw, label, p, crop_size, cat_max_ratio=1., ignore_index=255):
    """One sample through the four transforms: (image [h', w', 3] uint8 BGR, label [h', w'], chosen box index)"""
    img = np.ascontiguousarray(img_chw.transpose(1, 2, 0))
    rh, rw = p['resized_hw']
    img = resize_linear(img, rh, rw)
    seg = resize_nearest(label, rh, rw)
    k = choose_crop(seg, p['candidates'], crop_size, cat_max_ratio, ignore_index)
    oy, ox = p['candidates'][k]
    ch, cw = crop_size
    img, seg = img[oy:oy + ch, ox:ox + cw], seg[oy:oy + ch, ox:ox + cw]
    if p['flip']:
        img, seg = img[:, ::-1], seg[:, ::-1]
    return photometric(np.ascontiguousarray(img), p), np.ascontiguousarray(seg), k


def preprocess(img_hwc, seg, Hp, Wp, mean=None, std=None, bgr_to_rgb=True, pad_val=0., seg_pad_val=255):
    """SegDataPreProcessor + stack_batch of one sample: fp32 [3, Hp, Wp], int64 [Hp, Wp]"""
    x = img_hwc.transpose(2, 0, 1).astype(F32)
    if bgr_to_rgb:
        x = x[::-1]
    if mean is not None:
        x = (x - np.asarray(mean, F32)[:, None, None]) / np.asarray(std, F32)[:, None, None]
    h, w = seg.shape
    out = np.full((3, Hp, Wp), F32(pad_val), F32)
    out[:, :h, :w] = x
    lab = np.full((Hp, Wp), seg_pad_val, np.int64)
    lab[:h, :w] = seg
    return out, lab
