"""JPEG files decoded on the device (csrc/jpeg_decode.cu, ops.jpeg_decode) against cv2.imdecode(IMREAD_COLOR), the
device statuses against the CPU build of the same code, and the preprocessors fed PackSegFiles batches of JPEG images
against the same batches decoded by cv2."""
import ctypes as C

import cv2
import numpy as np
import pytest
import torch

import lednet_b200 as L
from lednet_b200 import lib, ops
from lednet_b200.tta import SegTTAModel
import jpeg_corpus as J
import png_corpus as P
from test_gpu_png_decode import MEAN, STD, TRAIN, _confusion, _model, _same_samples

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda', 0)


def _device_status(files, infos):
    """ledb200_jpeg_decode over device copies of the files: (statuses, outputs as numpy)"""
    n = len(files)
    data = [torch.frombuffer(bytearray(b), dtype=torch.uint8).to(DEV) for b in files]
    outs = [torch.zeros((3, h, w), dtype=torch.uint8, device=DEV) for h, w, _ in infos]
    arr = (lib.JpegFile * n)()
    for d, t, o, (h, w, nc) in zip(arr, data, outs, infos):
        d.data, d.size, d.out, d.h, d.w, d.components = t.data_ptr(), t.numel(), o.data_ptr(), h, w, nc
    l = lib.get()
    ws = torch.empty(lib.check(l.ledb200_jpeg_decode_workspace_bytes(arr, n)), dtype=torch.uint8, device=DEV)
    st = torch.full((n,), -7, dtype=torch.int32, device=DEV)
    lib.check(l.ledb200_jpeg_decode(arr, n, C.c_void_p(ws.data_ptr()), C.c_void_p(st.data_ptr()), lib.stream_ptr(DEV)))
    return st.cpu().tolist(), [o.cpu().numpy() for o in outs]


# ---- bit-exact decoding ------------------------------------------------------------------------------------------------------
def test_corpus_bit_exact_in_one_call():
    corpus = J.corpus() + J.large_corpus()                  # sizes, samplings and restart intervals mixed in one call
    outs = ops.jpeg_decode([b for _, b in corpus], names=[n for n, _ in corpus])
    for (name, b), o in zip(corpus, outs):
        assert o.is_cuda and o.dtype == torch.uint8
        assert np.array_equal(o.cpu().numpy(), J.cv2_ref(b)), name


def test_device_tensor_inputs():
    files = [J.cv2_jpeg(J.photo(375, 500, seed=s), 95, '420') for s in range(3)]
    outs = ops.jpeg_decode([torch.frombuffer(bytearray(files[0]), dtype=torch.uint8).to(DEV), files[1],
                            torch.frombuffer(bytearray(files[2]), dtype=torch.uint8)])
    for f, o in zip(files, outs):
        assert np.array_equal(o.cpu().numpy(), J.cv2_ref(f))


def test_batch_of_16_full_size_files():
    files = [J.cv2_jpeg(J.photo(1024, 2048, seed=s), 95, '420') for s in range(4)]
    files += [J.pil_jpeg(J.photo(1024, 2048, seed=10 + s)) for s in range(4)]
    files += [J.cv2_jpeg(J.photo(1024, 2048, seed=20 + s), 95, '444') for s in range(4)]
    files += [J.cv2_jpeg(J.photo(1024, 2048, seed=30 + s), 90, '422', rst=8) for s in range(4)]
    outs = ops.jpeg_decode(files)
    for f, o in zip(files, outs):
        assert np.array_equal(o.cpu().numpy(), J.cv2_ref(f))


def test_repeated_calls_give_the_same_output():
    files = [b for _, b in J.corpus()]
    a = ops.jpeg_decode(files)
    for _ in range(3):
        for x, y in zip(a, ops.jpeg_decode(files)):
            assert torch.equal(x, y)


# ---- corrupt files -----------------------------------------------------------------------------------------------------------
def test_corrupt_files_have_the_cpu_status():
    corrupt = J.corrupt()
    st, _ = _device_status([b for _, b, _ in corrupt], [J.CORRUPT_INFO] * len(corrupt))
    assert st == [s for _, _, s in corrupt]


def test_refused_files_are_unsupported_on_the_device():
    ref = J.refused()
    st, _ = _device_status([b for _, b in ref], [(30, 40, 3) if 'exif' in n else (24, 40, 3) for n, _ in ref])
    assert st == [3] * len(ref)


@pytest.mark.parametrize('name,data,status', J.corrupt(), ids=[c[0] for c in J.corrupt()])
def test_corrupt_file_raises_naming_it(name, data, status):
    try:
        ops.jpeg_info(data)
    except lib.LedB200Error:
        pytest.skip('refused by the host marker walk before any launch')
    good = J.cv2_jpeg(J.photo(8, 8), 90)
    with pytest.raises(lib.LedB200Error) as e:
        ops.jpeg_decode([good, data, good], names=['good0.jpg', f'{name}.jpg', 'good2.jpg'])
    msg = str(e.value)
    assert f'{name}.jpg' in msg and 'good0.jpg' not in msg


def test_fuzzed_files_match_the_cpu_build():
    files, infos = [], []
    for b in J.fuzz(400, seed=1) + J.fuzz(200, seed=2):
        try:
            infos.append(ops.jpeg_info(b))
            files.append(b)
        except (NotImplementedError, lib.LedB200Error):
            pass
    st_d, out_d = _device_status(files, infos)
    st_h, out_h = J.host_decode(files, infos)
    assert st_d == st_h
    assert sum(s == 0 for s in st_d) >= 100
    for s, a, b in zip(st_d, out_d, out_h):
        if s == 0:
            assert np.array_equal(a, b)


# ---- the preprocessors fed files ------------------------------------------------------------------------------------------------
def _dataset(tmp_path, n, h, w, K=19, png_every=0):
    """n image / label-map pairs on disk (JPEG images, every png_every-th a PNG), and PackSegFiles' outputs for them"""
    pack = L.PackSegFiles()
    items = []
    for i in range(n):
        img = J.photo(h, w, seed=20 + i)
        lab = P.blocky_labels(h, w, seed=40 + i, k=K)
        is_png = png_every and i % png_every == 0
        ip, lp = tmp_path / (f'img{i}.png' if is_png else f'img{i}.jpg'), tmp_path / f'img{i}_gt.png'
        ip.write_bytes(cv2.imencode('.png', img)[1].tobytes() if is_png else J.cv2_jpeg(img, 95, '420'))
        lp.write_bytes(P.png(lab[..., None], 0))
        items.append(pack(dict(img_path=str(ip), seg_map_path=str(lp), reduce_zero_label=False, label_map=None)))
    return items


def _file_batch(items):
    return dict(inputs=[it['inputs'] for it in items],
                data_samples=[dict(it['data_samples'], metainfo=dict(it['data_samples']['metainfo'])) for it in items])


def _decoded_batch(items):
    """the batch LoadImageFromFile + LoadAnnotations + PackSegInputs give: cv2 images, PIL label maps"""
    inputs, samples = [], []
    for it in items:
        m = it['data_samples']['metainfo']
        img = cv2.imread(m['img_path'], cv2.IMREAD_COLOR)
        inputs.append(torch.from_numpy(np.ascontiguousarray(img.transpose(2, 0, 1))))
        lab = P.pil_label_ref(open(m['seg_map_path'], 'rb').read())
        samples.append(dict(metainfo=dict(m), gt_sem_seg=dict(data=torch.from_numpy(lab))))
    return dict(inputs=inputs, data_samples=samples)


def test_mixed_png_and_jpeg_batch(tmp_path):
    items = _dataset(tmp_path, 5, 40, 56, png_every=2)
    a, b = L.decode_batch(_file_batch(items)), _decoded_batch(items)
    for x, y in zip(a['inputs'], b['inputs']):
        assert torch.equal(x.cpu(), y)
    _same_samples(a['data_samples'], b['data_samples'])


def test_device_augmentation_batch_from_jpeg_files(tmp_path):
    items = _dataset(tmp_path, 4, 96, 160)

    def run(batch):
        pp = L.DeviceAugSegDataPreProcessor(train_pipeline=TRAIN, seed=3, mean=MEAN, std=STD, bgr_to_rgb=True,
                                            size=(64, 96))
        return pp(batch, training=True)

    a, b = run(_file_batch(items)), run(_decoded_batch(items))
    assert torch.equal(a['inputs'], b['inputs'])
    _same_samples(a['data_samples'], b['data_samples'])


@pytest.mark.parametrize('path', ['plain', 'test_resize', 'tta'])
def test_eval_batches_from_jpeg_files(tmp_path, path):
    K = 19
    items = _dataset(tmp_path, 3, 128, 256, K)
    m = _model(K)
    if path == 'test_resize':
        m.data_preprocessor = L.DeviceAugSegDataPreProcessor(
            train_pipeline=TRAIN, test_pipeline=[dict(type='Resize', scale=(384, 192), keep_ratio=True)], mean=MEAN,
            std=STD, bgr_to_rgb=True)
    if path == 'tta':
        flips = [dict(type='RandomFlip', prob=0., direction='horizontal'),
                 dict(type='RandomFlip', prob=1., direction='horizontal')]
        runner = SegTTAModel(m, tta_transforms=[[dict(type='Resize', scale_factor=r, keep_ratio=True)
                                                  for r in (0.75, 1.0, 1.5)], flips])
    else:
        runner = m
    with torch.no_grad():
        a, b = runner.test_step(_file_batch(items)), runner.test_step(_decoded_batch(items))
    for x, y in zip(a, b):
        assert torch.equal(x['pred_sem_seg']['data'], y['pred_sem_seg']['data'])
        assert torch.equal(x['seg_logits']['data'], y['seg_logits']['data'])
    _same_samples(a, b)
    assert torch.equal(_confusion(a, K), _confusion(b, K))
