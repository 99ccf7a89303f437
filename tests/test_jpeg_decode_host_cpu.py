"""Host side of the JPEG decoder (no GPU): the marker walk and what jpeg_decode refuses before a launch, PackSegFiles /
PackSegPNGFiles and decode_batch's grouping, and the decoder itself run on the CPU through ledb200_jpeg_decode_host
(the same __host__ __device__ code as the kernels) over the seeded corpus, the corrupt files and a fuzz of valid
files, against cv2.imdecode."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

import lednet_b200 as L
from lednet_b200 import lib, ops
import jpeg_corpus as J
import png_corpus as P


# ---- the marker walk ---------------------------------------------------------------------------------------------------
def test_jpeg_info_reads_the_frame():
    assert ops.jpeg_info(J.cv2_jpeg(J.photo(13, 70), 90, '420')) == (13, 70, 3)
    grey = J.cv2_jpeg(J.photo(9, 5)[..., 0], 90)
    assert ops.jpeg_info(grey) == (9, 5, 1)
    assert ops.jpeg_info(torch.frombuffer(bytearray(grey), dtype=torch.uint8)) == (9, 5, 1)


def test_jpeg_info_walks_past_a_large_exif_segment():
    from PIL import Image
    e = Image.Exif()
    e[0x0112] = 1
    e[0x010E] = 'x' * 60000                                              # ImageDescription: a long APP1
    b = J.pil_jpeg(J.photo(20, 30), quality=80, exif=e.tobytes())
    assert ops.jpeg_info(b) == (20, 30, 3)


@pytest.mark.parametrize('name,data', J.refused(), ids=[r[0] for r in J.refused()])
def test_refused_files_are_not_implemented(name, data):
    with pytest.raises(NotImplementedError):
        ops.jpeg_info(data)


@pytest.mark.parametrize('name,data', J.refused(), ids=[r[0] for r in J.refused()])
def test_refused_files_are_unsupported_on_the_device_path_too(name, data):
    """the decoder itself refuses them, whatever descriptor it is given"""
    st, _ = J.host_decode([data], [(30, 40, 3) if 'exif' in name else (24, 40, 3)])
    assert st == [3], lib.JPEG_STATUS.get(st[0])


def test_malformed_headers_raise():
    good = J.cv2_jpeg(J.photo(8, 8), 90)
    for bad in (b'', b'\xff', good[:1] + b'\xd9' + good[2:], good[:2] + b'\x00' + good[3:], good[:2] + b'\xff\xe0\x00',
                good[:2] + b'\xff\xd9\x00\x02' + good[2:], good[:50]):
        with pytest.raises(lib.LedB200Error):
            ops.jpeg_info(bad)


def test_jpeg_decode_needs_cuda():
    if torch.cuda.is_available():
        pytest.skip('checks the no-device error')
    with pytest.raises(lib.LedB200Error):
        ops.jpeg_decode([J.cv2_jpeg(J.photo(8, 8))])


# ---- PackSegFiles / PackSegPNGFiles / decode_batch --------------------------------------------------------------------------
def test_pack_seg_files_reads_png_and_jpeg_images(tmp_path):
    jpg, png = J.cv2_jpeg(J.photo(12, 20), 90), P.png(P.smooth_rgb(12, 20), 2)
    lab = P.png(P.blocky_labels(12, 20)[..., None], 0)
    (tmp_path / 'a.jpg').write_bytes(jpg)
    (tmp_path / 'b.png').write_bytes(png)
    (tmp_path / 'a_gt.png').write_bytes(lab)
    t = L.TRANSFORMS.build(dict(type='PackSegFiles'))
    for name, data in (('a.jpg', jpg), ('b.png', png)):
        out = t(dict(img_path=str(tmp_path / name), seg_map_path=str(tmp_path / 'a_gt.png'), reduce_zero_label=False))
        assert out['inputs'].numpy().tobytes() == data
        s = out['data_samples']
        assert s['gt_seg_map_file'].numpy().tobytes() == lab
        assert s['metainfo'] == dict(img_path=str(tmp_path / name), seg_map_path=str(tmp_path / 'a_gt.png'),
                                     ori_shape=(12, 20), img_shape=(12, 20), reduce_zero_label=False, label_map=None)
    (tmp_path / 'p.jpg').write_bytes(J.refused()[0][1])
    with pytest.raises(NotImplementedError):
        t(dict(img_path=str(tmp_path / 'p.jpg')))
    (tmp_path / 'jpg_gt.jpg').write_bytes(jpg)
    with pytest.raises(lib.LedB200Error):                                 # label maps stay PNG
        t(dict(img_path=str(tmp_path / 'b.png'), seg_map_path=str(tmp_path / 'jpg_gt.jpg')))


def test_pack_seg_png_files_still_refuses_jpeg(tmp_path):
    (tmp_path / 'a.jpg').write_bytes(J.cv2_jpeg(J.photo(12, 20), 90))
    with pytest.raises(lib.LedB200Error, match='not a PNG file'):
        L.TRANSFORMS.build(dict(type='PackSegPNGFiles'))(dict(img_path=str(tmp_path / 'a.jpg')))
    assert issubclass(L.PackSegPNGFiles, L.PackSegFiles)


def test_decode_batch_groups_images_by_format(monkeypatch):
    jpg = [torch.frombuffer(bytearray(J.cv2_jpeg(J.photo(4 + i, 6), 90)), dtype=torch.uint8) for i in range(3)]
    png = [torch.frombuffer(bytearray(P.png(P.smooth_rgb(9, 5 + i), 2)), dtype=torch.uint8) for i in range(2)]
    calls = []

    def fake(kind):
        def dec(files, names=None, **kw):
            calls.append((kind, list(names)))
            return [f'{kind}:{n}' for n in names]
        return dec

    monkeypatch.setattr(ops, 'png_decode', fake('png'))
    monkeypatch.setattr(ops, 'jpeg_decode', fake('jpeg'))
    inputs = [jpg[0], png[0], jpg[1], jpg[2], png[1]]
    d = dict(inputs=inputs, data_samples=[dict(metainfo=dict(img_path=f'f{i}')) for i in range(5)])
    L.decode_batch(d)
    assert calls == [('png', ['f1', 'f4']), ('jpeg', ['f0', 'f2', 'f3'])]
    assert d['inputs'] == ['jpeg:f0', 'png:f1', 'jpeg:f2', 'jpeg:f3', 'png:f4']


# ---- the decoder on the CPU ----------------------------------------------------------------------------------------------
def test_host_decode_corpus_matches_cv2():
    corpus = J.corpus() + J.large_corpus()
    st, outs = J.host_decode([b for _, b in corpus])
    for (name, b), s, o in zip(corpus, st, outs):
        assert s == 0, (name, lib.JPEG_STATUS.get(s))
        assert np.array_equal(o, J.cv2_ref(b)), name


@pytest.mark.parametrize('name,data,status', J.corrupt(), ids=[c[0] for c in J.corrupt()])
def test_host_decode_rejects_corrupt_files(name, data, status):
    st, _ = J.host_decode([data], [J.CORRUPT_INFO])
    assert st == [status], lib.JPEG_STATUS.get(st[0])


def test_host_decode_checks_the_descriptor_against_the_frame():
    b = J.cv2_jpeg(J.photo(6, 10), 90)
    for info in ((6, 11, 3), (7, 10, 3), (6, 10, 1)):
        st, _ = J.host_decode([b], [info])
        assert st == [1]


def test_descriptors_are_validated():
    b = J.cv2_jpeg(J.photo(6, 10), 90)
    src = np.frombuffer(b, np.uint8).copy()
    out = np.zeros((3, 6, 10), np.uint8)
    st = (C.c_int32 * 1)()
    l = lib.get()
    for kw in (dict(h=0), dict(components=2), dict(size=3), dict(w=70000), dict(data=None)):
        arr = (lib.JpegFile * 1)()
        d = dict(data=src.ctypes.data, size=src.size, out=out.ctypes.data, h=6, w=10, components=3)
        d.update(kw)
        for k, v in d.items():
            setattr(arr[0], k, v)
        assert l.ledb200_jpeg_decode_host(arr, 1, st) == -1
        assert l.ledb200_jpeg_decode_workspace_bytes(arr, 1) == -1
    assert l.ledb200_jpeg_decode_host(arr, 0, st) == -1


def fuzz_outcomes(files):
    """(statuses, outputs) of the host build over fuzzed files; None where jpeg_info refuses the header"""
    out = []
    for b in files:
        try:
            info = ops.jpeg_info(b)
        except (NotImplementedError, lib.LedB200Error):
            out.append(None)
            continue
        st, o = J.host_decode([b], [info])
        out.append((st[0], o[0]))
    return out


def test_host_decode_fuzz_gives_a_status_or_cv2_pixels():
    import cv2
    decoded = 0
    files = J.fuzz(400, seed=1)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for b, r in zip(files, fuzz_outcomes(files)):
            if r is None or r[0] != 0:
                continue
            decoded += 1
            ref = cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR)
            assert ref is not None and np.array_equal(r[1], ref.transpose(2, 0, 1))
    assert decoded >= 100
