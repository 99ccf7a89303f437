"""CPU checks of the test-time-augmentation host logic: mmengine's split of the per-augmentation data, the view
descriptors read from metainfo, the registry entry, and the CPU restatement of merge_preds (tests/tta_oracle.py)
against a literal transcription of the reference - and against the reference file itself when it is mounted."""
import importlib.util
import os
import sys
import types
import warnings

import pytest
import torch

import lednet_b200 as L
from lednet_b200.tta import split_views, view_descriptor
from oracle import ref_loader
import tta_oracle


def test_split_dict_and_list_data():
    a, b = torch.zeros(3, 4, 4), torch.ones(3, 4, 4)
    data = dict(inputs=[[a, a], [b, b]], data_samples=[[{'i': 0}, {'i': 1}], [{'i': 2}, {'i': 3}]])
    views = split_views(data)
    assert len(views) == 2
    assert views[1]['inputs'][0] is b and views[0]['data_samples'][1] == {'i': 1}
    lst = split_views([[a, b, a], [{'i': 0}, {'i': 1}, {'i': 2}]])
    assert len(lst) == 3 and lst[1][0] is b and lst[2][1] == {'i': 2}
    with pytest.raises(TypeError):
        split_views(a)


def test_view_descriptor_from_metainfo():
    meta = dict(img_padding_size=(0, 4, 0, 8), padding_size=(1, 1, 1, 1), flip=True, flip_direction='vertical',
                ori_shape=(80, 100, 3))
    assert view_descriptor(meta, (72, 104)) == ((0, 4, 0, 8), 'vertical', (80, 100))
    assert view_descriptor(dict(padding_size=[1, 2, 3, 4], flip=False, flip_direction='horizontal'), (20, 30)) == \
        ((1, 2, 3, 4), None, (13, 27))                     # no ori_shape: the cropped extent
    assert view_descriptor({}, (16, 24)) == ((0, 0, 0, 0), None, (16, 24))
    with pytest.raises(AssertionError):
        view_descriptor(dict(flip=True, flip_direction='diagonal'), (8, 8))


def test_registry_builds_tta_model():
    assert 'SegTTAModel' in L.MODELS
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        tta = L.MODELS.build(dict(type='SegTTAModel', module=dict(
            type='EncoderDecoder', backbone=dict(type='LEDNet'),
            decode_head=dict(type='LEDHead', in_channels=128, channels=64, num_classes=19, dropout_ratio=0.))))
    assert isinstance(tta, L.SegTTAModel) and isinstance(tta.module, L.EncoderDecoder)
    assert tta._mode() == (0, 0.3)
    assert L.SegTTAModel(tta.module).module is tta.module


def _literal_merge_preds(data_samples_list, out_channels, threshold):
    """seg_tta.py SegTTAModel.merge_preds transcribed line by line over attribute-style samples."""
    predictions = []
    for data_samples in data_samples_list:
        seg_logits = data_samples[0].seg_logits.data
        logits = torch.zeros(seg_logits.shape).to(seg_logits)
        for data_sample in data_samples:
            seg_logit = data_sample.seg_logits.data
            if out_channels > 1:
                logits += seg_logit.softmax(dim=0)
            else:
                logits += seg_logit.sigmoid()
        logits /= len(data_samples)
        if out_channels == 1:
            seg_pred = (logits > threshold).to(logits).squeeze(1)
        else:
            seg_pred = logits.argmax(dim=0)
        predictions.append(seg_pred)
    return predictions


def _views(K, V, n, hw, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(n, K, *hw, generator=g) * 3 for _ in range(V)]


@pytest.mark.parametrize('out_channels', [19, 1])
def test_oracle_merge_equals_literal_merge_preds(out_channels):
    K, V, n, hw = 19, 4, 2, (12, 20)
    logits = _views(K, V, n, hw, seed=out_channels)
    metas = [[{}] * n for _ in range(V)]
    merged, pred = tta_oracle.tta_merge(logits, metas, out_channels, 0.3)
    samples = [[types.SimpleNamespace(seg_logits=types.SimpleNamespace(data=lg[i])) for lg in logits] for i in range(n)]
    ref = _literal_merge_preds(samples, out_channels, 0.3)
    for i in range(n):
        assert torch.equal(pred[i], ref[i])
    assert merged.shape == (n, K) + hw and pred.dtype == (torch.int64 if out_channels > 1 else torch.float32)


def test_oracle_postprocess_view_geometry():
    lg = torch.arange(2 * 6 * 8, dtype=torch.float32).view(2, 6, 8)
    out = tta_oracle.postprocess_view(lg, (1, 2, 0, 1), 'horizontal', None, False)
    assert torch.equal(out, lg[:, 0:5, 1:6].flip(dims=(2,)))
    out = tta_oracle.postprocess_view(lg, None, 'vertical', (6, 8), False)
    assert torch.equal(out, lg.flip(dims=(1,)))


def _load_reference_seg_tta():
    """seg_tta.py loaded verbatim behind stubs of the mmengine / mmseg names it imports."""
    path = os.path.join(ref_loader.REF_ROOT, 'mmseg/models/segmentors/seg_tta.py')

    class BaseTTAModel:
        def __init__(self, module=None, data_preprocessor=None):
            self.module = module

    class PixelData:
        def __init__(self, **kw):
            self.__dict__.update(kw)

    class _Registry:
        def register_module(self, *a, **k):
            return lambda cls: cls

    stubs = {'mmengine': types.ModuleType('mmengine'),
             'mmengine.model': types.ModuleType('mmengine.model'),
             'mmengine.structures': types.ModuleType('mmengine.structures'),
             'mmseg': types.ModuleType('mmseg'),
             'mmseg.registry': types.ModuleType('mmseg.registry'),
             'mmseg.utils': types.ModuleType('mmseg.utils')}
    stubs['mmengine.model'].BaseTTAModel = BaseTTAModel
    stubs['mmengine.structures'].PixelData = PixelData
    stubs['mmseg.registry'].MODELS = _Registry()
    stubs['mmseg.utils'].SampleList = list
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    try:
        spec = importlib.util.spec_from_file_location('_ledref_seg_tta', path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod


class _Sample:
    """the SegDataSample surface merge_preds touches"""

    def __init__(self, seg_logits, img_path):
        self.seg_logits = types.SimpleNamespace(data=seg_logits)
        self.img_path = img_path

    def set_data(self, d):
        for k, v in d.items():
            setattr(self, k, v)

    def set_metainfo(self, d):
        for k, v in d.items():
            setattr(self, k, v)


@pytest.mark.skipif(not os.path.isfile(os.path.join(ref_loader.REF_ROOT, 'mmseg/models/segmentors/seg_tta.py')),
                    reason='reference tree not mounted')
@pytest.mark.parametrize('out_channels', [19, 1])
def test_oracle_merge_against_reference_seg_tta(out_channels):
    ref = _load_reference_seg_tta()
    module = types.SimpleNamespace(out_channels=out_channels, decode_head=types.SimpleNamespace(threshold=0.3))
    tta = ref.SegTTAModel(module=module)
    tta.module = module
    K, V, n, hw = 19, 3, 2, (10, 14)
    logits = _views(K, V, n, hw, seed=7 + out_channels)
    _, pred = tta_oracle.tta_merge(logits, [[{}] * n for _ in range(V)], out_channels, 0.3)
    samples = [[_Sample(lg[i], f'img{i}_{v}.png') for v, lg in enumerate(logits)] for i in range(n)]
    out = tta.merge_preds(samples)
    for i in range(n):
        assert torch.equal(out[i].pred_sem_seg.data, pred[i])
        assert out[i] is samples[i][-1] and out[i].img_path == f'img{i}_0.png'
