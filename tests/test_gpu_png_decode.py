"""PNG files decoded on the device (csrc/png_decode.cu, ops.png_decode) against cv2.imdecode(IMREAD_COLOR) and
np.array(Image.open) + the label table, the device statuses against the CPU build of the same code, and the
preprocessors fed PackSegPNGFiles batches against the same batches decoded by cv2 / PIL."""
import ctypes as C
import warnings

import cv2
import numpy as np
import pytest
import torch

import lednet_b200 as L
from lednet_b200 import lib, ops, synth
from lednet_b200.tta import SegTTAModel
import png_corpus as P

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda', 0)
MEAN, STD = [123.675, 116.28, 103.53], [58.395, 57.12, 57.375]
TRAIN = [dict(type='RandomResize', scale=(320, 160), ratio_range=(0.5, 2.0), keep_ratio=True),
         dict(type='RandomCrop', crop_size=(64, 96), cat_max_ratio=0.75),
         dict(type='RandomFlip', prob=0.5), dict(type='PhotoMetricDistortion')]


def _device_status(files, kind='color'):
    """ledb200_png_decode over device copies of the files: (statuses, outputs as numpy)"""
    n = len(files)
    data = [torch.frombuffer(bytearray(b), dtype=torch.uint8).to(DEV) for b in files]
    infos = [ops.png_info(b, kind) for b in files]
    ch = 3 if kind == 'color' else 1
    outs = [torch.zeros((ch, h, w), dtype=torch.uint8, device=DEV) for h, w, _ in infos]
    arr = (lib.PngFile * n)()
    for d, t, o, (h, w, ct) in zip(arr, data, outs, infos):
        d.data, d.size, d.out, d.h, d.w, d.color_type = t.data_ptr(), t.numel(), o.data_ptr(), h, w, ct
    l = lib.get()
    ws = torch.empty(l.ledb200_png_decode_workspace_bytes(arr, n), dtype=torch.uint8, device=DEV)
    st = torch.full((n,), -7, dtype=torch.int32, device=DEV)
    lib.check(l.ledb200_png_decode(arr, n, lib.PNG_LABEL if kind == 'label' else lib.PNG_COLOR, None,
                                   C.c_void_p(ws.data_ptr()), C.c_void_p(st.data_ptr()), lib.stream_ptr(DEV)))
    return st.cpu().tolist(), [o.cpu().numpy() for o in outs]


# ---- bit-exact decoding ------------------------------------------------------------------------------------------------------
def test_colour_corpus_bit_exact_in_one_call():
    corpus = P.color_corpus()                              # sizes and colour types mixed in one call
    outs = ops.png_decode([b for _, b in corpus], names=[n for n, _ in corpus])
    for (name, b), o in zip(corpus, outs):
        assert o.is_cuda and o.dtype == torch.uint8
        assert np.array_equal(o.cpu().numpy(), P.cv2_ref(b)), name


@pytest.mark.parametrize('rzl,label_map', [(False, None), (True, None), (True, {3: 7, 7: 3})])
def test_label_corpus_bit_exact(rzl, label_map):
    corpus = P.label_corpus()
    outs = ops.png_decode([b for _, b in corpus], 'label', rzl, label_map)
    for (name, b), o in zip(corpus, outs):
        assert np.array_equal(o.cpu().numpy(), P.pil_label_ref(b, rzl, label_map)), name


def test_device_tensor_inputs_and_full_size():
    img = P.smooth_rgb(1024, 2048, seed=9)
    files = [cv2.imencode('.png', img, [cv2.IMWRITE_PNG_COMPRESSION, lvl])[1].tobytes() for lvl in (1, 9)]
    outs = ops.png_decode([torch.frombuffer(bytearray(files[0]), dtype=torch.uint8).to(DEV), files[1]])
    for o in outs:
        assert np.array_equal(o.cpu().numpy(), img.transpose(2, 0, 1))


def test_round_trip_through_png_encode():
    lab = torch.from_numpy(np.stack([P.blocky_labels(97, 131, seed=s) for s in range(3)])).to(DEV)
    files = ops.png_encode(lab)
    outs = ops.png_decode(files, 'label')
    for f, o, l in zip(files, outs, lab):
        assert torch.equal(o[0], l)
    assert torch.equal(ops.png_decode(ops.png_encode(lab, add=1), 'label', reduce_zero_label=True)[0][0], lab[0])


# ---- corrupt files -----------------------------------------------------------------------------------------------------------
def test_corrupt_files_have_the_cpu_status():
    corrupt = P.corrupt_corpus()
    st, _ = _device_status([b for _, b, _ in corrupt])
    assert st == [s for _, _, s in corrupt]


@pytest.mark.parametrize('name,data,status', P.corrupt_corpus(), ids=[c[0] for c in P.corrupt_corpus()])
def test_corrupt_file_raises_naming_it(name, data, status):
    good = P.png(P.smooth_rgb(8, 8), 2)
    with pytest.raises(lib.LedB200Error) as e:
        ops.png_decode([good, data, good], names=['good0.png', f'{name}.png', 'good2.png'])
    msg = str(e.value)
    assert f'{name}.png' in msg and lib.PNG_STATUS[status] in msg and 'good0.png' not in msg


def test_fuzzed_payloads_match_the_cpu_build():
    fz = P.fuzz_corpus(400, seed=1)
    files = [f for f, _, _ in fz]
    st_d, out_d = _device_status(files)
    st_h, out_h = P.host_decode(files)
    assert st_d == st_h
    for s, a, b in zip(st_d, out_d, out_h):
        if s == 0:
            assert np.array_equal(a, b)


# ---- the preprocessors fed files ------------------------------------------------------------------------------------------------
def _dataset(tmp_path, n, h, w, K=19):
    """n image / label-map PNG pairs on disk, and PackSegPNGFiles' outputs for them"""
    pack = L.PackSegPNGFiles()
    items = []
    for i in range(n):
        img = P.smooth_rgb(h, w, seed=20 + i)
        lab = P.blocky_labels(h, w, seed=40 + i, k=K)
        ip, lp = tmp_path / f'img{i}.png', tmp_path / f'img{i}_gt.png'
        ip.write_bytes(cv2.imencode('.png', img)[1].tobytes())
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


def _same_samples(a, b):
    for x, y in zip(a, b):
        assert x['metainfo'].keys() == y['metainfo'].keys()
        for k in x['metainfo']:
            if k != 'aug_params':
                assert x['metainfo'][k] == y['metainfo'][k], k
        assert torch.equal(x['gt_sem_seg']['data'].to(DEV), y['gt_sem_seg']['data'].to(DEV))


def test_device_augmentation_batch_from_files(tmp_path):
    items = _dataset(tmp_path, 4, 96, 160)
    def run(batch):
        pp = L.DeviceAugSegDataPreProcessor(train_pipeline=TRAIN, seed=3, mean=MEAN, std=STD, bgr_to_rgb=True,
                                            size=(64, 96))
        return pp(batch, training=True)

    a, b = run(_file_batch(items)), run(_decoded_batch(items))
    assert torch.equal(a['inputs'], b['inputs'])
    _same_samples(a['data_samples'], b['data_samples'])
    for x, y in zip(a['data_samples'], b['data_samples']):
        assert {k: v for k, v in x['metainfo']['aug_params'].items() if k != 'crop_index'} == \
            {k: v for k, v in y['metainfo']['aug_params'].items() if k != 'crop_index'}


def _model(K):
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        m = L.EncoderDecoder(dict(type='LEDNet'), dict(type='LEDHead', in_channels=128, channels=64, num_classes=K,
                                                       dropout_ratio=0.),
                             data_preprocessor=dict(type='SegDataPreProcessor', mean=MEAN, std=STD, bgr_to_rgb=True),
                             compute_dtype='bf16').eval()
    m.load_state_dict(synth.make_state_dict(m.state_dict(), seed=2))
    return m.to(DEV)


def _confusion(results, K):
    metric = L.IoUMetric()
    metric.dataset_meta = dict(classes=[str(k) for k in range(K)])
    metric.process(None, results)
    return metric.total_confusion(reduce_ranks=False)


@pytest.mark.parametrize('path', ['plain', 'test_resize', 'tta'])
def test_eval_batches_from_files(tmp_path, path):
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
