"""PNG files of label maps encoded on the device (csrc/png.cu, ops.png_encode) and IoUMetric's output_dir / format_only.

Every file is decoded twice: by PIL, and by a strict reader here that checks the signature, the chunk order, every chunk's
CRC-32 and the zlib stream (zlib.decompress checks the Adler-32), then undoes the filter bytes."""
import io
import os
import struct
import zlib

import numpy as np
import pytest
import scipy.ndimage as nd
import torch
from PIL import Image

import lednet_b200 as L
from lednet_b200 import lib, ops

pytestmark = pytest.mark.gpu


# ---- seeded maps ---------------------------------------------------------------------------------------------------
def constant(h, w, seed=0):
    return np.full((h, w), 7, np.uint8)


def blocky(h, w, seed=0, cell=32, k=19):
    rng = np.random.default_rng(seed)
    small = rng.integers(0, k, (-(-h // cell), -(-w // cell)))
    return np.kron(small, np.ones((cell, cell), np.int64))[:h, :w].astype(np.uint8)


def smooth(h, w, seed=0, k=19):
    rng = np.random.default_rng(seed)
    f = nd.gaussian_filter(rng.standard_normal((h, w)), 30 if min(h, w) > 64 else 2)
    return np.digitize(f, np.linspace(f.min(), f.max(), k + 1)[1:-1]).astype(np.uint8)


def noise(h, w, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (h, w)).astype(np.uint8)


MAPS = dict(constant=constant, blocky=blocky, smooth=smooth, noise=noise)


# ---- decoders --------------------------------------------------------------------------------------------------------
def strict_decode(b):
    assert b[:8] == b'\x89PNG\r\n\x1a\n'
    pos, chunks = 8, []
    while pos < len(b):
        n, = struct.unpack('>I', b[pos:pos + 4])
        typ, data = b[pos + 4:pos + 8], b[pos + 8:pos + 8 + n]
        crc, = struct.unpack('>I', b[pos + 8 + n:pos + 12 + n])
        assert zlib.crc32(typ + data) == crc, f'bad CRC in {typ}'
        chunks.append((typ, data))
        pos += 12 + n
    assert pos == len(b)
    types = [t for t, _ in chunks]
    assert types[0] == b'IHDR' and types[-1] == b'IEND' and set(types[1:-1]) == {b'IDAT'}
    w, h, depth, ctype, comp, filt, inter = struct.unpack('>IIBBBBB', chunks[0][1])
    assert (depth, ctype, comp, filt, inter) == (8, 0, 0, 0, 0)
    raw = zlib.decompress(b''.join(d for t, d in chunks if t == b'IDAT'))
    rows = np.frombuffer(raw, np.uint8).reshape(h, w + 1)
    assert (rows[:, 0] == 0).all()
    return rows[:, 1:]


def pil_decode(b):
    im = Image.open(io.BytesIO(b))
    assert im.mode == 'L'
    return np.asarray(im)


def check_files(files, labels, add):
    want = ((labels.astype(np.int64) + add) % 256).astype(np.uint8)
    if want.ndim == 2:
        want = want[None]
    assert len(files) == want.shape[0]
    bound = lib.get().ledb200_png_bound(want.shape[1], want.shape[2])
    for b, w in zip(files, want):
        assert len(b) <= bound
        assert np.array_equal(strict_decode(b), w)
        assert np.array_equal(pil_decode(b), w)


def pil_size(a, level):
    buf = io.BytesIO()
    Image.fromarray(a).save(buf, format='PNG', compress_level=level)
    return len(buf.getvalue())


# ---- round trips ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('shape', [(1, 1), (1, 2048), (2048, 1), (7, 13), (512, 910), (4, 40000)])
@pytest.mark.parametrize('kind', sorted(MAPS))
@pytest.mark.parametrize('dtype', [torch.uint8, torch.int64])
@pytest.mark.parametrize('add', [0, 1])
def test_round_trip(shape, kind, dtype, add):
    a = MAPS[kind](*shape, seed=3)
    t = torch.from_numpy(a).to(dtype).cuda()
    check_files(ops.png_encode(t, add=add), a, add)


@pytest.mark.parametrize('add', [0, 1])
def test_int64_wraps_and_255(add):
    rng = np.random.default_rng(5)
    a = rng.integers(0, 1000, (3, 61, 77))
    a[0, :10] = 255
    a[1, 5:40, 3:50] = 511
    a[2] = rng.integers(-300, 300, (61, 77))
    check_files(ops.png_encode(torch.from_numpy(a).cuda(), add=add), a, add)


def test_shapes_of_pred_sem_seg():
    a = blocky(64, 96, seed=1)
    t = torch.from_numpy(a).cuda()
    one = ops.png_encode(t)
    assert len(one) == 1 and ops.png_encode(t[None]) == one
    check_files(one, a, 0)


def test_batch_16_full_size_mixed_and_sizes():
    h, w = 1024, 2048
    kinds = ['blocky', 'smooth', 'noise', 'constant'] * 4
    maps = np.stack([MAPS[k](h, w, seed=i) for i, k in enumerate(kinds)])
    t = torch.from_numpy(maps).cuda()
    files = ops.png_encode(t)
    check_files(files, maps, 0)
    stored = h * (w + 1)
    for k, a, b in zip(kinds, maps, files):
        if k == 'noise':
            assert len(b) >= stored                   # incompressible: the stored path
        if k in ('blocky', 'smooth'):
            assert len(b) <= pil_size(a, 1), k
    assert ops.png_encode(t) == files              # deterministic
    files64 = ops.png_encode(t.long())
    assert files64 == files


def test_errors():
    l = lib.get()
    t = torch.zeros(4, 4, dtype=torch.uint8, device='cuda')
    with pytest.raises(lib.LedB200Error):
        ops.png_encode(t, add=2)
    with pytest.raises(lib.LedB200Error):
        ops.png_encode(t.float())
    ws = torch.empty(l.ledb200_png_workspace_bytes(1, 4, 4), dtype=torch.uint8, device='cuda')
    out = torch.empty(l.ledb200_png_bound(4, 4), dtype=torch.uint8, device='cuda')
    offs = torch.empty(2, dtype=torch.int64, device='cuda')
    st = lib.stream_ptr()
    args = [t.data_ptr(), lib.U8, 1, 4, 4, 0, out.data_ptr(), offs.data_ptr(), ws.data_ptr(), st]
    assert l.ledb200_png_encode(*args) == 0
    for i, bad in [(1, lib.F32), (2, 0), (3, 0), (4, 0), (5, -1), (0, None), (6, None), (7, None), (8, None)]:
        a = list(args)
        a[i] = bad
        assert l.ledb200_png_encode(*a) == -1, (i, bad)


# ---- IoUMetric -------------------------------------------------------------------------------------------------------
def _samples(n=4, h=48, w=80, with_gt=True, rzl=None, meta=False):
    out = []
    for i in range(n):
        pred = torch.from_numpy(blocky(h, w, seed=10 + i, cell=8)).long().cuda()
        s = dict(pred_sem_seg=dict(data=pred[None]))
        if with_gt:
            s['gt_sem_seg'] = dict(data=torch.from_numpy(blocky(h, w, seed=20 + i, cell=8)).long().cuda()[None])
        info = dict(img_path=f'/data/city/img_{i}.leftImg8bit.jpg', reduce_zero_label=bool(rzl and rzl[i]))
        if meta:
            s['metainfo'] = info
        else:
            s.update(info)
        out.append(s)
    return out


def _metric(**kw):
    m = L.IoUMetric(**kw)
    m.dataset_meta = dict(classes=[str(i) for i in range(19)])
    return m


def _expected_name(i):
    return f'img_{i}.leftImg8bit.png'


@pytest.mark.parametrize('meta', [False, True])
def test_metric_output_dir(tmp_path, meta):
    d = str(tmp_path / 'out')
    samples = _samples(rzl=[0, 1, 0, 1], meta=meta)
    m, ref = _metric(output_dir=d), _metric()
    m.process(None, samples)
    ref.process(None, samples)
    assert sorted(os.listdir(d)) == sorted(_expected_name(i) for i in range(4))
    for i, s in enumerate(samples):
        pred = s['pred_sem_seg']['data'][0].cpu().numpy()
        got = np.asarray(Image.open(os.path.join(d, _expected_name(i))))
        assert np.array_equal(got, (pred + (i % 2)).astype(np.uint8))
    assert m.evaluate(4) == ref.evaluate(4)


def test_metric_mixed_shapes(tmp_path):
    d = str(tmp_path)
    samples = _samples(2, 48, 80) + _samples(2, 33, 17)
    for i, s in enumerate(samples):
        s['img_path'] = f'x{i}.png'
    m = _metric(output_dir=d, format_only=True)
    m.process(None, samples)
    for i, s in enumerate(samples):
        got = np.asarray(Image.open(os.path.join(d, f'x{i}.png')))
        assert np.array_equal(got, s['pred_sem_seg']['data'][0].cpu().numpy().astype(np.uint8))


def test_metric_format_only(tmp_path):
    d = str(tmp_path / 'fmt')
    m = _metric(output_dir=d, format_only=True, keep_results=True)
    m.process(None, _samples(with_gt=False))
    assert len(os.listdir(d)) == 4
    assert m.evaluate(4) == {}


def test_process_batch_writes_the_same_files(tmp_path):
    d1, d2 = str(tmp_path / 'a'), str(tmp_path / 'b')
    samples = _samples(rzl=[1, 1, 1, 1])
    m1, m2 = _metric(output_dir=d1), _metric(output_dir=d2)
    m1.process(None, samples)
    pred = torch.cat([s['pred_sem_seg']['data'] for s in samples])
    lab = torch.cat([s['gt_sem_seg']['data'] for s in samples])
    m2.process_batch(pred, lab, img_paths=[s['img_path'] for s in samples], reduce_zero_label=True)
    for i in range(4):
        with open(os.path.join(d1, _expected_name(i)), 'rb') as f1, open(os.path.join(d2, _expected_name(i)), 'rb') as f2:
            assert f1.read() == f2.read()
    assert m1.evaluate(4) == m2.evaluate(4)
    m3 = _metric(output_dir=str(tmp_path / 'c'), format_only=True)
    m3.process_batch(pred.to(torch.uint8), img_paths=[s['img_path'] for s in samples])
    assert len(os.listdir(str(tmp_path / 'c'))) == 4 and m3.evaluate(4) == {}
