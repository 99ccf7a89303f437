"""CityscapesMetric on the device: 16-bit decoding, palette labelId files, cityscapes_accumulate and the metric against the
numpy restatement of cityscapesscripts' evaluation (tests/cityscapes_oracle.py), and its errors."""
import io
import os
import struct

import numpy as np
import pytest
import torch
from PIL import Image

import lednet_b200 as L
from lednet_b200 import cityscapes as CS, lib, ops
import cityscapes_corpus as CC
import cityscapes_oracle as O

pytestmark = pytest.mark.gpu


def _chunks(b):
    pos, out = 8, []
    while pos < len(b):
        n, = struct.unpack('>I', b[pos:pos + 4])
        out.append((b[pos + 4:pos + 8], b[pos:pos + 12 + n]))
        pos += 12 + n
    return out


# ---- decoding and encoding ------------------------------------------------------------------------------------------------
def test_grey16_decode_equals_host_and_pil():
    corpus = CC.grey16_corpus() + [('scene-2048x1024', CC.pil16(CC.scene(1024, 2048, seed=1)[1]))]
    files = [b for _, b in corpus]
    outs = ops.png_decode(files, 'grey16', names=[n for n, _ in corpus])
    _, st, host = CC.host16(files)
    for (name, b), o, h in zip(corpus, outs, host):
        assert o.dtype == torch.int32 and o.shape[0] == 1
        got = o[0].cpu().numpy()
        assert np.array_equal(got, CC.pil16_ref(b)), name
        assert np.array_equal(got, h), name
    assert st == [0] * len(files)
    bad = CC.corrupt16()
    for name, data, status in bad:
        with pytest.raises(lib.LedB200Error, match=name):
            ops.png_decode([data], 'grey16', names=[name])


def test_palette_files_match_pil():
    rng = np.random.default_rng(1)
    pred = rng.integers(0, 256, (37, 53))
    pred[:10] = rng.integers(0, 19, (10, 53))
    for dt in (torch.uint8, torch.int64):
        files = ops.png_encode(torch.from_numpy(pred).to(dt).cuda(), lut=CS.TRAIN_TO_ID, palette=True)
        want = O.convert_to_label_id(pred)
        bio = io.BytesIO()
        Image.fromarray(want).convert('P').save(bio, format='PNG')
        ref = dict(_chunks(bio.getvalue()))
        im = Image.open(io.BytesIO(files[0]))
        assert im.mode == 'P' and np.array_equal(np.asarray(im), want)
        got = dict(_chunks(files[0]))
        assert got[b'IHDR'] == ref[b'IHDR'] and got[b'PLTE'] == ref[b'PLTE']
        assert [t for t, _ in _chunks(files[0])] == [b'IHDR', b'PLTE', b'IDAT', b'IEND']
        assert len(files[0]) <= lib.get().ledb200_png_lut_bound(37, 53, 1)
    dec = ops.png_decode(files, 'label')[0][0].cpu().numpy()
    assert np.array_equal(dec, O.convert_to_label_id(pred))


@pytest.mark.parametrize('add', [0, 1])
def test_lut_without_palette_gives_todays_bytes(add):
    t = torch.from_numpy(CC.scene(96, 130, seed=4)[2]).cuda()
    assert ops.png_encode(t, lut=(np.arange(256) + add) % 256) == ops.png_encode(t, add=add)
    assert ops.png_encode(t, add=add, palette=False) == ops.png_encode(t, add=add)
    with pytest.raises(lib.LedB200Error):
        ops.png_encode(t, add=1, lut=np.arange(256))
    with pytest.raises(lib.LedB200Error):
        ops.png_encode(t, lut=np.arange(255))


# ---- cityscapes_accumulate --------------------------------------------------------------------------------------------------
def _accumulate(scenes, dtype):
    pred = torch.from_numpy(np.stack([p for _, _, p in scenes])).to(dtype).cuda()
    gt = torch.from_numpy(np.stack([g for g, _, _ in scenes])).cuda()
    inst = torch.from_numpy(np.stack([i for _, i, _ in scenes])).cuda()
    last = torch.empty((34, 34), dtype=torch.int64, device='cuda')
    cm, st, recs = ops.cityscapes_accumulate(pred, gt, inst, CS.TRAIN_TO_ID, CS.KERNEL_CATEGORY, CS.KERNEL_RULE,
                                             cm_last=last)
    return cm.cpu().numpy(), st, recs, last.cpu().numpy()


def _oracle_stats(g, i, p):
    pl = O.convert_to_label_id(p)
    cm = O.generate_matrix()
    O.evaluate_pair(pl, g, i, cm, O.generate_instance_stats())
    return cm.astype(np.int64), np.array(O.instance_records(pl, i), np.int64).reshape(-1, 4)


@pytest.mark.parametrize('dtype', [torch.uint8, torch.int64])
@pytest.mark.parametrize('shape,n', [((1024, 2048), 2), ((37, 53), 3), ((1, 1), 2), ((61, 7), 1)])
def test_accumulate_equals_the_oracle(dtype, shape, n):
    scenes = [CC.scene(*shape, seed=10 + k, cell=max(1, min(shape) // 4), blobs=20) for k in range(n)]
    cm, st, recs, last = _accumulate(scenes, dtype)
    assert st.tolist() == [0] * n
    want = [_oracle_stats(*s) for s in scenes]
    assert np.array_equal(cm, sum(c for c, _ in want))
    assert np.array_equal(last, want[-1][0])
    for (_, r), g in zip(want, recs):
        assert np.array_equal(g, r)
    if shape == (1024, 2048):
        assert all(len(r) > 5 for r in recs)
        assert _accumulate(scenes, dtype)[2][0].tolist() == recs[0].tolist()       # repeats run to run


def test_accumulate_many_instances_take_a_second_copy():
    scenes = [CC.many_instances(120, 160, 400, seed=k) for k in range(2)]
    _, st, recs, _ = _accumulate(scenes, torch.uint8)
    assert st.tolist() == [0, 0] and sum(len(r) for r in recs) > 2 * ops.CITYSCAPES_RECORDS_PER_COPY
    for s, r in zip(scenes, recs):
        assert np.array_equal(r, _oracle_stats(*s)[1])


def test_accumulate_statuses():
    g, i, p = CC.scene(40, 60, seed=3)
    cases = []
    gg = g.copy(); gg[5, 5] = 40; cases.append((gg, i, p, 1))
    pp = p.copy(); pp[0, 0] = 200; cases.append((g, i, pp, 2))                      # trainId 200 stays labelId 200
    for bad in (7001, 34001):
        ii = i.copy(); ii[3, 3] = bad; cases.append((g, ii, p, 4))
    pp = p.copy(); pp[1, 1] = 300; cases.append((g, i, pp, 8))
    pp = p.copy(); pp[1, 1] = -1; cases.append((g, i, pp, 8))
    for gg, ii, pp, bit in cases:
        _, st, _, _ = _accumulate([(g, i, p), (gg, ii, pp)], torch.int64)
        assert st[0] == 0 and st[1] & bit, (bit, st)


# ---- the metric ---------------------------------------------------------------------------------------------------------------
def _samples(scenes, paths, dtype=torch.int64):
    return [dict(pred_sem_seg=dict(data=torch.from_numpy(p).to(dtype).cuda()[None]), img_path=img, seg_map_path=seg)
            for (_, _, p), (img, seg) in zip(scenes, paths)]


def _oracle(scenes):
    return O.evaluate_arrays([(O.convert_to_label_id(p), g, i) for g, i, p in scenes])


@pytest.mark.parametrize('inst_writer', [CC.pil16, CC.cv2_16])
def test_metric_equals_the_oracle(tmp_path, inst_writer):
    scenes = [CC.scene(128, 256, seed=30 + k, cell=16, blobs=15) for k in range(5)] + \
             [CC.scene(64, 96, seed=40 + k, cell=8) for k in range(2)]
    paths = CC.write_dataset(str(tmp_path / 'data'), scenes, inst_writer)
    samples = _samples(scenes, paths)
    out = str(tmp_path / 'out')
    m = L.METRICS.build(dict(type='CityscapesMetric', output_dir=out, keep_results=True))
    m.process(None, samples[:3])
    m.process(None, samples[3:])
    got = m.evaluate(len(samples))
    want = _oracle(scenes)
    assert got == dict(averageScoreCategories=want['averageScoreCategories'],
                       averageScoreInstCategories=want['averageScoreInstCategories'])
    assert O.same(m.cityscapes_results, want)
    assert m.cityscapes_results['confMatrix'].dtype == np.int64
    assert sorted(os.listdir(out)) == sorted(os.path.basename(p) for p, _ in paths)
    for (_, _, p), (img, _) in zip(scenes, paths):
        im = Image.open(os.path.join(out, os.path.basename(img)))
        assert im.mode == 'P' and np.array_equal(np.asarray(im), O.convert_to_label_id(p))
    # the labels-only path, uint8 predictions, no files
    m2 = L.CityscapesMetric(output_dir=str(tmp_path / 'out2'))
    for k in (0, 5):
        n = 5 if k == 0 else 2
        pred = torch.stack([s['pred_sem_seg']['data'][0] for s in samples[k:k + n]]).to(torch.uint8)
        m2.process_batch(pred, seg_map_paths=[s for _, s in paths[k:k + n]])
    assert m2.evaluate() == got and O.same(m2.cityscapes_results, want)
    assert os.listdir(str(tmp_path / 'out2')) == []


def test_format_only_and_keep_results(tmp_path):
    scenes = [CC.scene(48, 80, seed=50 + k, cell=8) for k in range(3)]
    paths = [(f'a/x{k}_leftImg8bit.png', None) for k in range(3)]
    with pytest.raises(AssertionError):
        L.CityscapesMetric(output_dir=str(tmp_path / 'f'), format_only=True)
    m = L.CityscapesMetric(output_dir=str(tmp_path / 'f'), format_only=True, keep_results=True)
    m.process(None, _samples(scenes, paths))
    assert sorted(os.listdir(str(tmp_path / 'f'))) == [f'x{k}_leftImg8bit.png' for k in range(3)]
    assert m.evaluate(3) == {}
    bad = scenes[0][2].copy()
    bad[0, 0] = 300
    with pytest.raises(lib.LedB200Error, match='x0_leftImg8bit'):
        m.process(None, [dict(pred_sem_seg=dict(data=torch.from_numpy(bad).cuda()[None]), img_path=paths[0][0])])
    data = CC.write_dataset(str(tmp_path / 'data'), scenes)
    d = str(tmp_path / 'kept')
    m = L.CityscapesMetric(output_dir=d)
    assert os.path.isdir(d)
    m.process(None, _samples(scenes, data))
    m.evaluate(3)
    assert os.path.isdir(d) and os.listdir(d) == []


def test_metric_errors_name_the_file(tmp_path):
    g, i, p = CC.scene(40, 60, seed=7)
    base = str(tmp_path / 'data')

    def run(gt, inst, pred, mutate=None):
        paths = CC.write_dataset(base, [(gt, inst, pred)])
        if mutate:
            mutate(paths[0][1].replace('labelTrainIds', 'instanceIds'))
        m = L.CityscapesMetric(output_dir=str(tmp_path / 'o'))
        with pytest.raises(lib.LedB200Error, match='city_000000_000019_gtFine') as e:
            m.process(None, _samples([(gt, inst, pred)], paths))
        return str(e.value)

    gg = g.copy(); gg[2, 2] = 40
    assert 'labelId above 33' in run(gg, i, p)
    for bad in (7001, 34001):
        ii = i.copy(); ii[2, 2] = bad
        assert 'instance id' in run(g, ii, p)
    pp = p.copy(); pp[1, 1] = 300
    assert 'outside 0 .. 255' in run(g, i, pp)
    assert 'instanceIds' in run(g, i, p, os.remove)
    assert 'instanceIds' in run(g, i, p, lambda f: open(f, 'wb').write(CC.pil16(np.zeros((40, 61)))))
