"""Host side of the PNG decoder (no GPU): IHDR parsing and what png_decode rejects before a launch, PackSegPNGFiles, the
label lookup table, and the decoder itself run on the CPU through ledb200_png_decode_host (the same __host__ __device__
code as the kernels) over the seeded corpus, the corrupt files and a fuzz of zlib payloads."""
import ctypes as C

import numpy as np
import pytest
import torch

import lednet_b200 as L
from lednet_b200 import lib, ops
import png_corpus as P


# ---- IHDR ------------------------------------------------------------------------------------------------------------
def _hdr(w, h, ct, depth=8, interlace=0):
    return P.SIG + P.ihdr(w, h, ct, depth, interlace)


@pytest.mark.parametrize('ct', [0, 2, 3, 4, 6])
def test_png_info_reads_the_ihdr(ct):
    assert ops.png_info(_hdr(70000, 3, ct)) == (3, 70000, ct)
    assert ops.png_info(torch.frombuffer(bytearray(_hdr(5, 9, ct)), dtype=torch.uint8)) == (9, 5, ct)


@pytest.mark.parametrize('depth,ct', [(1, 0), (2, 3), (4, 0), (16, 0), (16, 2), (16, 6)])
def test_other_bit_depths_are_not_implemented(depth, ct):
    with pytest.raises(NotImplementedError):
        ops.png_info(_hdr(4, 4, ct, depth))


def test_interlace_and_colour_labels_are_not_implemented():
    with pytest.raises(NotImplementedError):
        ops.png_info(_hdr(4, 4, 2, interlace=1))
    for ct in (2, 4, 6):
        ops.png_info(_hdr(4, 4, ct))
        with pytest.raises(NotImplementedError):
            ops.png_info(_hdr(4, 4, ct), 'label')


def test_malformed_headers_raise():
    good = _hdr(4, 4, 2)
    for bad in (b'', good[:32], b'\x88' + good[1:], good[:8] + b'\x00\x00\x00\x0eIHDR' + good[16:],
                good[:-1] + bytes([good[-1] ^ 1]), _hdr(0, 4, 2), _hdr(4, 0, 2), _hdr(4, 4, 5), _hdr(4, 4, 2, 3),
                _hdr(4, 4, 2, interlace=2), _hdr(1 << 16, 1 << 15, 0)):
        with pytest.raises(lib.LedB200Error):
            ops.png_info(bad)


def test_png_decode_needs_cuda():
    if torch.cuda.is_available():
        pytest.skip('checks the no-device error')
    with pytest.raises(lib.LedB200Error):
        ops.png_decode([P.png(np.zeros((2, 2, 3), np.uint8), 2)])


# ---- PackSegPNGFiles / decode_batch --------------------------------------------------------------------------------------
def test_pack_seg_png_files(tmp_path):
    img = P.png(P.smooth_rgb(12, 20), 2)
    lab = P.png(P.blocky_labels(12, 20)[..., None], 0)
    (tmp_path / 'a.png').write_bytes(img)
    (tmp_path / 'a_gt.png').write_bytes(lab)
    t = L.TRANSFORMS.build(dict(type='PackSegPNGFiles'))
    out = t(dict(img_path=str(tmp_path / 'a.png'), seg_map_path=str(tmp_path / 'a_gt.png'), reduce_zero_label=True,
                 label_map={1: 2}))
    assert out['inputs'].dtype == torch.uint8 and out['inputs'].dim() == 1
    assert out['inputs'].numpy().tobytes() == img
    s = out['data_samples']
    assert s['gt_seg_map_file'].numpy().tobytes() == lab and 'gt_sem_seg' not in s
    assert s['metainfo'] == dict(img_path=str(tmp_path / 'a.png'), seg_map_path=str(tmp_path / 'a_gt.png'),
                                 ori_shape=(12, 20), img_shape=(12, 20), reduce_zero_label=True, label_map={1: 2})
    only = t(dict(img_path=str(tmp_path / 'a.png'), reduce_zero_label=False))
    assert 'gt_seg_map_file' not in only['data_samples']
    assert only['data_samples']['metainfo']['reduce_zero_label'] is False
    with pytest.raises(AssertionError):
        L.PackSegPNGFiles(reduce_zero_label=False)(dict(img_path=str(tmp_path / 'a.png'),
                                                        seg_map_path=str(tmp_path / 'a_gt.png'), reduce_zero_label=True))
    (tmp_path / 'rgb_gt.png').write_bytes(img)
    with pytest.raises(NotImplementedError):
        t(dict(img_path=str(tmp_path / 'a.png'), seg_map_path=str(tmp_path / 'rgb_gt.png')))


def test_decode_batch_leaves_decoded_batches_alone():
    x = torch.zeros(2, 3, 4, 4, dtype=torch.uint8)
    d = dict(inputs=x, data_samples=[{}, {}])
    assert L.decode_batch(d) is d and d['inputs'] is x
    imgs = [torch.zeros(3, 4, 4, dtype=torch.uint8)]
    d = dict(inputs=imgs)
    assert L.decode_batch(d)['inputs'] is imgs


# ---- the label table -------------------------------------------------------------------------------------------------------
def _load_annotations(seg, reduce_zero_label, label_map):
    """mmseg 1.2.2 LoadAnnotations._load_seg_map on a decoded uint8 map, restated"""
    seg = seg.copy()
    if reduce_zero_label:
        seg[seg == 0] = 255
        seg = seg - 1
        seg[seg == 254] = 255
    if label_map is not None:
        copy = seg.copy()
        for old, new in label_map.items():
            seg[copy == old] = new
    return seg


@pytest.mark.parametrize('rzl', [False, True])
@pytest.mark.parametrize('label_map', [None, {0: 3, 3: 0, 255: 7}, {i: (i * 7) % 19 for i in range(19)}])
def test_label_lut_matches_load_annotations(rzl, label_map):
    seg = np.arange(256, dtype=np.uint8).reshape(16, 16)
    assert np.array_equal(ops.label_lut(rzl, label_map)[seg], _load_annotations(seg, rzl, label_map))


def test_label_lut_rejects_values_outside_uint8():
    with pytest.raises(ValueError):
        ops.label_lut(False, {1: 256})


# ---- the decoder on the CPU ---------------------------------------------------------------------------------------------------
def test_host_decode_colour_corpus_matches_cv2():
    corpus = P.color_corpus()
    st, outs = P.host_decode([b for _, b in corpus])
    for (name, b), s, o in zip(corpus, st, outs):
        assert s == 0, (name, s)
        assert np.array_equal(o, P.cv2_ref(b)), name


@pytest.mark.parametrize('rzl,label_map', [(False, None), (True, None), (True, {3: 7, 7: 3})])
def test_host_decode_label_corpus_matches_pil(rzl, label_map):
    corpus = P.label_corpus()
    st, outs = P.host_decode([b for _, b in corpus], 'label', rzl, label_map)
    for (name, b), s, o in zip(corpus, st, outs):
        assert s == 0, (name, s)
        assert np.array_equal(o, P.pil_label_ref(b, rzl, label_map)), name


@pytest.mark.parametrize('name,data,status', P.corrupt_corpus(), ids=[c[0] for c in P.corrupt_corpus()])
def test_host_decode_rejects_corrupt_files(name, data, status):
    st, _ = P.host_decode([data])
    assert st == [status], lib.PNG_STATUS.get(st[0])


def test_host_decode_checks_the_descriptor_against_the_ihdr():
    b = P.png(P.smooth_rgb(6, 10), 2)
    src = np.frombuffer(b, np.uint8).copy()
    out = np.zeros((3, 6, 11), np.uint8)
    arr = (lib.PngFile * 1)()
    arr[0].data, arr[0].size, arr[0].out, arr[0].h, arr[0].w, arr[0].color_type = src.ctypes.data, src.size, \
        out.ctypes.data, 6, 11, 2
    st = (C.c_int32 * 1)()
    assert lib.get().ledb200_png_decode_host(arr, 1, lib.PNG_COLOR, None, st) == 0 and st[0] == 1


def test_descriptors_are_validated():
    b = P.png(P.smooth_rgb(6, 10), 2)
    src = np.frombuffer(b, np.uint8).copy()
    out = np.zeros((3, 6, 10), np.uint8)
    st = (C.c_int32 * 1)()
    l = lib.get()
    for kw in (dict(h=0), dict(color_type=5), dict(size=20), dict(h=1 << 16, w=1 << 15)):
        arr = (lib.PngFile * 1)()
        d = dict(data=src.ctypes.data, size=src.size, out=out.ctypes.data, h=6, w=10, color_type=2)
        d.update(kw)
        for k, v in d.items():
            setattr(arr[0], k, v)
        assert l.ledb200_png_decode_host(arr, 1, lib.PNG_COLOR, None, st) == -1
    arr = (lib.PngFile * 1)()
    arr[0].data, arr[0].size, arr[0].out, arr[0].h, arr[0].w, arr[0].color_type = src.ctypes.data, src.size, \
        out.ctypes.data, 6, 10, 2
    assert l.ledb200_png_decode_host(arr, 1, lib.PNG_LABEL, None, st) == -1     # a colour file as a label map
    assert l.ledb200_png_decode_host(arr, 0, lib.PNG_COLOR, None, st) == -1
    assert l.ledb200_png_decode_host(arr, 1, 2, None, st) == -1


def test_host_decode_fuzzed_zlib_payloads():
    valid = 0
    for f, z, (h, w, ct) in P.fuzz_corpus(400, seed=1):
        want = P.fuzz_expect(z, h, w, ct)
        st, outs = P.host_decode([f])
        if want is None:
            assert st[0] != 0
            continue
        valid += 1
        assert st[0] == 0
        got = outs[0]
        ref = P.cv2_ref(f)
        assert np.array_equal(got, ref)
        px = want.reshape(h, w, P.BPP[ct])
        rgb = px[..., :1].repeat(3, -1) if ct in (0, 4) else px[..., :3]
        assert np.array_equal(got, rgb[..., ::-1].transpose(2, 0, 1))
    assert valid >= 40
