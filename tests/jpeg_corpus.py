"""Seeded JPEG files for the decoder tests (tests/test_jpeg_decode_host_cpu.py, tests/test_gpu_jpeg_decode.py): files
written by cv2 and PIL at several qualities, samplings, restart intervals and sizes, refused files, corrupt files with
the status the decoder must give, a fuzz of valid files, cv2's decode as the reference and a ctypes call of
ledb200_jpeg_decode_host."""
import ctypes as C
import io
import struct

import cv2
import numpy as np
from PIL import Image

from lednet_b200 import lib as LIB, ops

SAMPLING = {'444': cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, '422': cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            '420': cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, '440': cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440}
SIZES = [(1, 1), (2, 3), (7, 9), (17, 33), (375, 500)]


# ---- pixels ----------------------------------------------------------------------------------------------------------
def photo(h, w, seed=0):
    """smooth colour gradients with edges and mild noise: what a photograph compresses like"""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    b = 128 + 100 * np.sin(x / (7 + seed) + y / 13)
    g = 128 + 90 * np.cos(y / (5 + seed) - x / 17)
    r = (x * 3 + y * 2) % 256
    img = np.stack([b, g, r], -1) + rng.normal(0, 6, (h, w, 3))
    img[(x.astype(int) // 16 + y.astype(int) // 16) % 5 == 0] *= 0.5
    return np.clip(img, 0, 255).astype(np.uint8)


def noise(h, w, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3)).astype(np.uint8)


def flat(h, w, v=(40, 120, 200)):
    return np.broadcast_to(np.array(v, np.uint8), (h, w, 3)).copy()


# ---- encoders ----------------------------------------------------------------------------------------------------------
def cv2_jpeg(img, quality=95, sampling=None, rst=None, optimize=False, progressive=False):
    params = [cv2.IMWRITE_JPEG_QUALITY, quality]
    if sampling is not None:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sampling]]
    if rst is not None:
        params += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    if optimize:
        params += [cv2.IMWRITE_JPEG_OPTIMIZE, 1]
    if progressive:
        params += [cv2.IMWRITE_JPEG_PROGRESSIVE, 1]
    ok, enc = cv2.imencode('.jpg', img, params)
    assert ok
    return enc.tobytes()


def pil_jpeg(img_bgr, mode='RGB', **kw):
    bio = io.BytesIO()
    a = img_bgr[..., ::-1] if img_bgr.ndim == 3 else img_bgr
    Image.fromarray(np.ascontiguousarray(a)).convert(mode).save(bio, format='JPEG', **kw)
    return bio.getvalue()


def exif(orientation):
    e = Image.Exif()
    e[0x0112] = orientation
    return e.tobytes()


# ---- reference decoder and the host entry point ------------------------------------------------------------------------
def cv2_ref(b):
    return cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR).transpose(2, 0, 1)


def host_decode(files, infos=None):
    """ledb200_jpeg_decode_host over the files: (statuses, outputs)"""
    n = len(files)
    srcs = [np.frombuffer(b, np.uint8).copy() for b in files]
    infos = infos or [ops.jpeg_info(b) for b in files]
    outs = [np.zeros((3, h, w), np.uint8) for h, w, _ in infos]
    arr = (LIB.JpegFile * n)()
    for d, s, o, (h, w, nc) in zip(arr, srcs, outs, infos):
        d.data, d.size, d.out, d.h, d.w, d.components = s.ctypes.data, s.size, o.ctypes.data, h, w, nc
    st = (C.c_int32 * n)()
    LIB.check(LIB.get().ledb200_jpeg_decode_host(arr, n, st))
    return list(st), outs


# ---- corpora ------------------------------------------------------------------------------------------------------------
def corpus():
    """(name, file) pairs of supported files, all decoded by cv2"""
    out = []
    img = photo(45, 67, seed=1)
    for q in (50, 75, 95, 100):
        out.append((f'cv2-q{q}', cv2_jpeg(img, q)))
    for s in SAMPLING:
        for h, w in SIZES:
            out.append((f'cv2-{s}-{h}x{w}', cv2_jpeg(photo(h, w, seed=h + w), 90, s)))
    for rst in (1, 3, 64):
        for s in ('420', '444'):
            out.append((f'cv2-rst{rst}-{s}', cv2_jpeg(photo(37, 53, seed=rst), 85, s, rst=rst)))
    out.append(('cv2-optimize', cv2_jpeg(img, 90, optimize=True)))
    out.append(('cv2-optimize-rst2', cv2_jpeg(img, 80, '422', rst=2, optimize=True)))
    grey = cv2.cvtColor(photo(29, 41, seed=5), cv2.COLOR_BGR2GRAY)
    for q in (60, 100):
        out.append((f'cv2-grey-q{q}', cv2_jpeg(grey, q)))
    out.append(('cv2-grey-rst5', cv2_jpeg(grey, 90, rst=5)))
    out.append(('pil-L', pil_jpeg(grey, 'L', quality=80)))
    for sub in (0, 1, 2):
        out.append((f'pil-sub{sub}', pil_jpeg(img, subsampling=sub, quality=75)))
        out.append((f'pil-sub{sub}-odd', pil_jpeg(photo(19, 23, seed=sub), subsampling=sub, quality=88)))
    out.append(('pil-default', pil_jpeg(img)))
    out.append(('pil-rst-blocks', pil_jpeg(img, quality=90, restart_marker_blocks=5)))
    out.append(('pil-optimize', pil_jpeg(img, quality=70, optimize=True)))
    out.append(('pil-exif-orientation-1', pil_jpeg(img, quality=90, exif=exif(1))))
    out.append(('flat-420', cv2_jpeg(flat(64, 256), 95, '420')))          # subsequences of EOB-only blocks
    out.append(('flat-grey', cv2_jpeg(flat(40, 300)[..., 0], 75)))
    out.append(('noise-q100-444', cv2_jpeg(noise(48, 64, seed=3), 100, '444')))   # blocks longer than a subsequence
    out.append(('noise-q100-420-rst7', cv2_jpeg(noise(33, 47, seed=4), 100, '420', rst=7)))
    return out


def large_corpus():
    """larger files: VOC-sized and 2048x1024 photos"""
    out = []
    for s in ('420', '444'):
        out.append((f'cv2-500x375-{s}', cv2_jpeg(photo(375, 500, seed=7), 95, s)))
    out.append(('cv2-2048x1024-420', cv2_jpeg(photo(1024, 2048, seed=8), 95, '420')))
    out.append(('pil-2048x1024', pil_jpeg(photo(1024, 2048, seed=9))))
    return out


def _replace_byte(b, off, v):
    return b[:off] + bytes([v]) + b[off + 1:]


def _sof_offset(b):
    for m in (b'\xff\xc0', b'\xff\xc1'):
        i = b.find(m)
        if i >= 0:
            return i
    raise ValueError('no SOF')


def refused():
    """(name, file) pairs that jpeg_info refuses with NotImplementedError"""
    img = photo(24, 40, seed=2)
    good = cv2_jpeg(img, 90)
    sof = _sof_offset(good)
    out = [('progressive', cv2_jpeg(img, 90, progressive=True)),
           ('pil-cmyk', pil_jpeg(img, 'CMYK', quality=90)),
           ('pil-keep-rgb', pil_jpeg(img, quality=90, keep_rgb=True)),
           ('exif-orientation-6', pil_jpeg(photo(30, 40, seed=3), quality=90, exif=exif(6))),
           ('sof9-arithmetic', _replace_byte(good, sof + 1, 0xC9)),
           ('sof3-lossless', _replace_byte(good, sof + 1, 0xC3)),
           ('12-bit', _replace_byte(good, sof + 4, 12)),
           ('dnl-height-0', good[:sof + 5] + b'\x00\x00' + good[sof + 7:]),
           ('sampling-411', cv2_sampling(good, 0x41)),
           ('pil-sub-411-like', cv2_sampling(good, 0x42))]
    return out


def cv2_sampling(b, hv):
    """b with the luma sampling byte replaced"""
    sof = _sof_offset(b)
    return _replace_byte(b, sof + 11, hv)


def _scan_start(b):
    i = b.index(b'\xff\xda')
    return i + 2 + (b[i + 2] << 8 | b[i + 3])


def _segment(b, marker):
    i = b.index(marker)
    return i, i + 2 + (b[i + 2] << 8 | b[i + 3])


CORRUPT_INFO = (32, 48, 3)


def corrupt():
    """(name, file, expected status) of files the decoder must reject, statuses as lib.JPEG_STATUS lists them; every
    file is decoded with the descriptor CORRUPT_INFO of the valid file it was made from"""
    img = photo(32, 48, seed=6)
    good = cv2_jpeg(img, 90, '420')
    s0 = _scan_start(good)
    out = []
    out.append(('truncated-scan', good[:s0 + (len(good) - s0) // 2], 6))
    out.append(('scan-cut-before-eoi', good[:s0 + (len(good) - s0) // 2] + b'\xff\xd9', 6))
    # flipped code bits: all-ones bytes are no code of the tables cv2 writes
    out.append(('flipped-code-bits', good[:s0 + 8] + b'\xff\x00' * 6 + good[s0 + 20:], 5))
    rst = cv2_jpeg(img, 90, '420', rst=1)
    k = rst.index(b'\xff\xd1', _scan_start(rst))
    out.append(('wrong-rst-number', _replace_byte(rst, k + 1, 0xD3), 7))
    k0 = rst.index(b'\xff\xd0', _scan_start(rst))
    out.append(('missing-rst', rst[:k0] + rst[k0 + 2:], 7))
    a, e = _segment(good, b'\xff\xc4')
    out.append(('missing-dht', good[:a] + good[e:], 4))
    # DHT segments placed just before SOS, so they replace the luma DC table cv2 wrote (class 0, id 0)
    sos = good.index(b'\xff\xda')

    def dht(counts, vals):
        body = b'\x00' + bytes(counts) + bytes(vals)
        return b'\xff\xc4' + struct.pack('>H', 2 + len(body)) + body

    out.append(('oversubscribed-dht', good[:sos] + dht([2, 1] + [0] * 14, [0, 1, 2]) + good[sos:], 4))
    out.append(('all-ones-dht', good[:sos] + dht([2] + [0] * 15, [0, 1]) + good[sos:], 4))
    out.append(('dc-symbol-16', good[:sos] + dht([1, 1] + [0] * 14, [0, 16]) + good[sos:], 4))
    out.append(('segment-past-end', good[:2] + b'\xff\xe0\xff\xf0' + good[4:40], 2))
    q, _ = _segment(good, b'\xff\xdb')
    out.append(('dqt-table-id-4', _replace_byte(good, q + 4, 0x04), 4))
    out.append(('no-eoi-marker-after-scan', good[:-2] + b'\xff\xd8', 2))
    return out


def fuzz(n=300, seed=0):
    """seeded mutations of small valid files: flipped bits and bytes in the entropy-coded data, truncations, flips
    anywhere"""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        h, w = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        s = list(SAMPLING)[i % 4]
        b = bytearray(cv2_jpeg(photo(h, w, seed=i), int(rng.integers(30, 101)), s,
                               rst=[None, 1, 2, 5][int(rng.integers(4))]))
        s0 = _scan_start(bytes(b))
        kind = int(rng.integers(5))
        if kind == 0:                                                     # flip bits in the scan
            for _ in range(int(rng.integers(1, 4))):
                j = int(rng.integers(s0, len(b) - 2))
                b[j] ^= 1 << int(rng.integers(8))
        elif kind == 1:                                                   # a random byte in the scan
            b[int(rng.integers(s0, len(b) - 2))] = int(rng.integers(256))
        elif kind == 2:                                                   # cut
            b = b[:int(rng.integers(s0, len(b)))]
        elif kind == 3:                                                   # flip a bit anywhere after SOI
            j = int(rng.integers(2, len(b)))
            b[j] ^= 1 << int(rng.integers(8))
        out.append(bytes(b))
    return out
