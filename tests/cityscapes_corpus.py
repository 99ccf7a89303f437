"""Seeded Cityscapes-like scenes and their files (tests/test_cityscapes_host_cpu.py, tests/test_gpu_cityscapes.py,
tools/bench_cityscapes_metric.py): blocky labelIds using every id 0 .. 33, instanceIds id * 1000 + k in instance blobs of
classes 24 .. 33 (caravan and trailer included), crowd regions of instance classes stored as the bare labelId, and trainId
predictions made from the GT with perturbed blocks.  16-bit instance files are written by PIL, by cv2 and by hand (every
filter type), plus corrupt and fuzzed 16-bit files."""
import ctypes as C
import io
import os
import struct
import zlib

import cv2
import numpy as np
from PIL import Image

from lednet_b200 import lib as LIB
import png_corpus as P

# labelId -> trainId (ignored ids -> 255), cityscapesscripts helpers/labels.py
ID_TO_TRAIN = np.full(34, 255, np.int64)
for _i, _t in zip([7, 8, 11, 12, 13, 17, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 31, 32, 33], range(19)):
    ID_TO_TRAIN[_i] = _t


def scene(h, w, seed=0, cell=32, blobs=12, crowd=2):
    """(gt labelIds uint8 [h, w], instanceIds int32 [h, w], trainId prediction int64 [h, w])"""
    rng = np.random.default_rng(seed)
    ch, cw = -(-h // cell), -(-w // cell)
    ids = np.resize(rng.permutation(34), ch * cw)           # every id 0 .. 33 when the map has >= 34 cells
    rng.shuffle(ids)
    gt = np.kron(ids.reshape(ch, cw), np.ones((cell, cell), np.int64))[:h, :w].astype(np.uint8)
    inst = gt.astype(np.int32).copy()
    y, x = np.mgrid[0:h, 0:w]
    counters = {}
    for b in range(blobs + crowd):
        c = int(rng.integers(24, 34))
        cy, cx = rng.integers(0, h), rng.integers(0, w)
        ry, rx = rng.integers(2, max(3, h // 5)), rng.integers(2, max(3, w // 5))
        m = ((y - cy) / ry) ** 2 + ((x - cx) / rx) ** 2 <= 1
        gt[m] = c
        if b < blobs:
            k = counters.get(c, 0)
            counters[c] = k + 1
            inst[m] = c * 1000 + k
        else:
            inst[m] = c                                       # a crowd region: the bare labelId
    pred = ID_TO_TRAIN[gt].copy()
    for _ in range(max(1, (ch * cw) // 3)):
        py, px = rng.integers(0, h), rng.integers(0, w)
        sy, sx = rng.integers(1, max(2, cell)), rng.integers(1, max(2, cell))
        pred[py:py + sy, px:px + sx] = rng.choice(np.r_[np.arange(19), 255])
    return gt, inst, pred


def many_instances(h, w, n, seed=0):
    """a scene whose instance map holds n small person / car instances (more than one copy's worth of records)"""
    rng = np.random.default_rng(seed)
    gt = np.full((h, w), 7, np.uint8)
    inst = gt.astype(np.int32)
    side = int(np.ceil(np.sqrt(n)))
    bh, bw = h // side, w // side
    assert bh >= 2 and bw >= 2
    for k in range(n):
        c = 24 if k % 2 else 26
        y0, x0 = (k // side) * bh, (k % side) * bw
        gt[y0:y0 + bh - 1, x0:x0 + bw - 1] = c
        inst[y0:y0 + bh - 1, x0:x0 + bw - 1] = c * 1000 + k
    pred = ID_TO_TRAIN[gt].copy()
    pred[rng.random((h, w)) < 0.2] = 13
    return gt, inst, pred


# ---- files ---------------------------------------------------------------------------------------------------------------
def pil_png(a):
    bio = io.BytesIO()
    Image.fromarray(a).save(bio, format='PNG')
    return bio.getvalue()


def pil16(inst, **kw):
    bio = io.BytesIO()
    Image.fromarray(inst.astype(np.uint16)).save(bio, format='PNG', **kw)
    return bio.getvalue()


def cv2_16(inst, level=3):
    ok, enc = cv2.imencode('.png', inst.astype(np.uint16), [cv2.IMWRITE_PNG_COMPRESSION, level])
    assert ok
    return enc.tobytes()


def be_bytes(inst):
    """[h, 2 w] uint8: each 16-bit sample as its big-endian byte pair"""
    return inst.astype('>u2').view(np.uint8).reshape(inst.shape[0], -1)


def hand16(inst, filters=(0,), zdata=None, level=6):
    """a 16-bit grey PNG by hand; the scanlines filtered with 2 bytes per pixel (png_corpus's colour type 4 has that)"""
    h, w = inst.shape
    if zdata is None:
        zdata = zlib.compress(P.filter_rows(be_bytes(inst), 4, filters), level)
    return P.SIG + P.ihdr(w, h, 0, 16) + P.chunk(b'IDAT', zdata) + P.chunk(b'IEND', b'')


def pil16_ref(b):
    return np.array(Image.open(io.BytesIO(b))).astype(np.int32)


def grey16_corpus():
    """(name, file) pairs of valid 16-bit grey files"""
    _, inst, _ = scene(45, 67, seed=3, cell=8, blobs=6)
    out = [(f'pil-l{lv}', pil16(inst, compress_level=lv)) for lv in (0, 1, 6, 9)]
    out += [('pil-opt', pil16(inst, optimize=True))]
    out += [(f'cv2-l{lv}', cv2_16(inst, lv)) for lv in (0, 1, 3, 9)]
    rng = np.random.default_rng(4)
    noise = rng.integers(0, 65536, (9, 13)).astype(np.int64)
    for ft in range(5):
        out.append((f'hand-filter{ft}', hand16(noise, (ft,))))
    out.append(('hand-filters-mixed', hand16(inst, (4, 0, 1, 2, 3))))
    out.append(('hand-stored', hand16(inst, (1,), level=0)))
    for h, w in ((1, 1), (1, 9), (7, 1), (5, 33)):
        out.append((f'size-{h}x{w}', hand16(rng.integers(0, 65536, (h, w)), (4, 3))))
    return out


def corrupt16():
    """(name, file, expected LEDB200_PNG_* status) of 16-bit files the decoder must reject"""
    inst = np.random.default_rng(5).integers(0, 34000, (6, 10))
    raw = P.filter_rows(be_bytes(inst), 4, (0,))
    z = zlib.compress(raw)
    good = hand16(inst)
    idat = good.index(b'IDAT') - 4
    n = struct.unpack('>I', good[idat:idat + 4])[0]
    bad = bytearray(good)
    bad[idat + 8 + n] ^= 0xff
    return [
        ('idat-crc', bytes(bad), 3),
        ('no-iend', good[:-12], 2),
        ('truncated-zlib', hand16(inst, zdata=z[:len(z) // 2]), 8),
        ('bad-adler', hand16(inst, zdata=z[:-4] + bytes([z[-4] ^ 1]) + z[-3:]), 10),
        ('8-bit-sized-data', hand16(inst, zdata=zlib.compress(P.filter_rows(be_bytes(inst)[:, ::2], 0, (0,)))), 9),
        ('too-many-bytes', hand16(inst, zdata=zlib.compress(raw + b'\x00')), 9),
        ('filter-type-5', hand16(inst, zdata=zlib.compress(bytes([5]) + raw[1:])), 11),
    ]


def fuzz16(n=200, seed=0):
    """(file, expected int32 [h, w] or None) of seeded mutations of small 16-bit files' zlib streams"""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        h, w = int(rng.integers(1, 10)), int(rng.integers(1, 10))
        inst = rng.integers(0, 3, (h, w)) * 12000 + rng.integers(0, 2, (h, w))
        co = zlib.compressobj(int(rng.integers(0, 10)), zlib.DEFLATED, 15, 9,
                              [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE][i % 4])
        z = bytearray(co.compress(P.filter_rows(be_bytes(inst), 4, (int(rng.integers(0, 5)),))) + co.flush())
        kind = rng.integers(4)
        if kind == 0:
            for _ in range(int(rng.integers(1, 4))):
                j = int(rng.integers(len(z)))
                z[j] ^= 1 << int(rng.integers(8))
        elif kind == 1:
            z = z[:int(rng.integers(len(z)))]
        elif kind == 2:
            z[min(2, len(z) - 1)] ^= 1 << int(rng.integers(3))
        z = bytes(z)
        px = P.fuzz_expect(z, h, w, 4)
        want = None if px is None else (px[:, 0::2].astype(np.int32) << 8 | px[:, 1::2])
        out.append((hand16(inst, zdata=z), want))
    return out


def host16(files, mode=LIB.PNG_GREY16, ct=None):
    """ledb200_png_decode_host over 16-bit files: (return code, statuses, int32 [h, w] outputs)"""
    n = len(files)
    srcs = [np.frombuffer(b, np.uint8).copy() for b in files]
    infos = [P.ops.png_info(b, 'grey16') for b in files]
    outs = [np.zeros((1, h, w), np.int32) for h, w, _ in infos]
    arr = (LIB.PngFile * n)()
    for d, s, o, (h, w, c) in zip(arr, srcs, outs, infos):
        d.data, d.size, d.out, d.h, d.w, d.color_type = s.ctypes.data, s.size, o.ctypes.data, h, w, c if ct is None else ct
    st = (C.c_int32 * n)()
    rc = LIB.get().ledb200_png_decode_host(arr, n, mode, None, st)
    return rc, list(st), [o[0] for o in outs]


def write_dataset(root, scenes, inst_writer=pil16):
    """Cityscapes' layout under root: gtFine/<city>/<name>_gtFine_labelTrainIds.png (what the dataset's seg_map_path
    names), _labelIds.png and _instanceIds.png; returns the samples' (img_path, seg_map_path)."""
    out = []
    d = os.path.join(root, 'gtFine', 'val', 'city')
    os.makedirs(d, exist_ok=True)
    for i, (gt, inst, _) in enumerate(scenes):
        stem = os.path.join(d, f'city_{i:06d}_000019_gtFine_')
        with open(stem + 'labelIds.png', 'wb') as f:
            f.write(pil_png(gt))
        with open(stem + 'instanceIds.png', 'wb') as f:
            f.write(inst_writer(inst))
        out.append((f'leftImg8bit/val/city/city_{i:06d}_000019_leftImg8bit.png', stem + 'labelTrainIds.png'))
    return out
