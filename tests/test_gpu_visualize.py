"""SegLocalVisualizer / SegVisualizationHook on the device against the numpy + cv2 restatement of mmseg's drawing
(tests/vis_oracle.py): label locations, drawn files decoded by cv2 and PIL, RGB PNG files, the grey / palette PNG bytes
pinned from before the RGB encoder, and the hook end to end after EncoderDecoder.test_step."""
import hashlib
import io
import os
import types
import zlib

import cv2
import numpy as np
import pytest
import torch
from PIL import Image

import lednet_b200 as L
from lednet_b200 import lib, ops, visualization as V
import jpeg_corpus as J
import png_corpus as P
import vis_oracle as O
from test_gpu_png_decode import _model

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda', 0)


def center_locs(m, K):
    """_get_center_loc of every class k < K of one map, with numpy row counts (the oracle's sort is too slow at full
    size; test_center_locs_fast_equals_the_oracle ties the two together)"""
    H, W = m.shape
    out = np.zeros((K, 3), np.int32)
    for k in np.unique(m):
        if k >= K:
            continue
        hit = m == k
        rows = hit.sum(1)
        y = int(rows.argmax())
        xs = np.flatnonzero(hit[y])
        out[k] = (1, xs[len(xs) // 2], y)
    return out


def _maps(kind, h, w, K, seed):
    rng = np.random.default_rng(seed)
    if kind == 'random':
        return rng.integers(0, min(K + 3, 256), (h, w)).astype(np.uint8)
    m = O.blocky_map(h, w, K, seed, cell=max(1, min(h, w) // 8))
    m[rng.random((h, w)) < 0.02] = rng.integers(0, K)
    return m


def test_center_locs_fast_equals_the_oracle():
    for seed in range(6):
        m = _maps('structured' if seed % 2 else 'random', 23, 31, 5, seed)
        want = center_locs(m, 5)
        for k in range(5):
            if want[k, 0]:
                assert O.get_center_loc((m == k).astype(np.uint8)).tolist() == want[k, 1:].tolist()


# ---- seg_label_locations -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', [torch.uint8, torch.int64])
@pytest.mark.parametrize('K', [2, 19, 150])
@pytest.mark.parametrize('kind,shape,n', [('structured', (1024, 2048), 2), ('random', (37, 53), 3),
                                          ('structured', (300, 41), 2), ('random', (1, 1), 2), ('random', (5, 1000), 1)])
def test_label_locations_equal_the_oracle(dtype, K, kind, shape, n):
    maps = [_maps(kind, *shape, K, seed=K + k) for k in range(n)]
    got = ops.seg_label_locations(torch.from_numpy(np.stack(maps)).to(dtype).to(DEV), K).cpu().numpy()
    assert got.shape == (n, K, 3) and got.dtype == np.int32
    for g, m in zip(got, maps):
        assert np.array_equal(g, center_locs(m, K))


def test_label_locations_ties_and_out_of_range():
    m = np.full((6, 9), 255, np.int64)
    m[1, [2, 3, 4]] = 1
    m[4, [0, 5, 8]] = 1
    m[0, 0] = 0
    m[2, 2] = -3
    m[3, 3] = 7
    got = ops.seg_label_locations(torch.from_numpy(m).to(DEV), 4).cpu().numpy()[0]
    assert got.tolist() == [[1, 0, 0], [1, 3, 1], [0, 0, 0], [0, 0, 0]]


# ---- drawn pictures --------------------------------------------------------------------------------------------------------
def _decoded(data):
    a = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_UNCHANGED)
    im = Image.open(io.BytesIO(data))
    im.load()                                 # PIL checks the CRCs of the chunks it reads
    b = np.asarray(im.convert('RGB'))
    assert im.mode == 'RGB' and np.array_equal(a[..., ::-1], b)
    return b


def _draw_files(tmp_path, imgs, gts, preds, with_labels=True, alpha=0.8, classes=None, palette=None, tensor_images=False):
    vis = V.SegLocalVisualizer(save_dir=str(tmp_path), vis_backends=[dict(type='LocalVisBackend')], alpha=alpha,
                               classes=classes, palette=palette)
    names = [f'img{i}.png' for i in range(len(imgs))]
    samples = []
    for g, p in zip(gts, preds):
        s = {}
        if g is not None:
            s['gt_sem_seg'] = dict(data=torch.from_numpy(g)[None].to(DEV))
        if p is not None:
            s['pred_sem_seg'] = dict(data=torch.from_numpy(p.astype(np.int64))[None].to(DEV))
        samples.append(s)
    images = [torch.from_numpy(np.ascontiguousarray(im[..., ::-1].transpose(2, 0, 1))).to(DEV) for im in imgs] \
        if tensor_images else imgs
    vis.add_datasamples(names, images, samples, list(range(1, len(imgs) + 1)), with_labels=with_labels)
    d = os.path.join(str(tmp_path), 'vis_data', 'vis_image')
    return [_decoded(open(os.path.join(d, f'{n}_{i + 1}.png'), 'rb').read()) for i, n in enumerate(names)]


def _case(h, w, n, K=19, seed=0):
    imgs = [O.photo(h, w, seed + i) for i in range(n)]
    gts = [O.blocky_map(h, w, K, seed + 10 + i, cell=max(4, min(h, w) // 6)) for i in range(n)]
    preds = [O.blocky_map(h, w, K, seed + 20 + i, cell=max(4, min(h, w) // 5), ignore=0) for i in range(n)]
    return imgs, gts, preds


@pytest.mark.parametrize('panels', ['both', 'pred', 'gt'])
@pytest.mark.parametrize('with_labels', [True, False])
def test_drawn_files_equal_the_oracle(tmp_path, panels, with_labels):
    imgs, gts, preds = _case(256, 384, 3)
    gts = gts if panels != 'pred' else [None] * 3
    preds = preds if panels != 'gt' else [None] * 3
    got = _draw_files(tmp_path, imgs, gts, preds, with_labels, tensor_images=panels == 'both')
    for g, im, gt, pr in zip(got, imgs, gts, preds):
        assert np.array_equal(g, O.add_datasample(im, gt, pr, with_labels=with_labels))


@pytest.mark.parametrize('alpha', [0.8, 0.6, 0.5, 1.0])
@pytest.mark.parametrize('hw', [(120, 170), (299, 433), (301, 317), (57, 1)])
def test_alphas_and_sizes(tmp_path, alpha, hw):
    imgs, gts, preds = _case(*hw, 2, seed=hw[0])
    got = _draw_files(tmp_path, imgs, gts, preds, alpha=alpha)
    for g, im, gt, pr in zip(got, imgs, gts, preds):
        assert np.array_equal(g, O.add_datasample(im, gt, pr, alpha=alpha))


def test_given_palette_and_full_size(tmp_path):
    rng = np.random.default_rng(5)
    classes = [f'class {k}' for k in range(150)]
    palette = rng.integers(0, 256, (150, 3)).tolist()
    imgs, gts, preds = _case(512, 640, 2, K=150, seed=7)
    got = _draw_files(tmp_path / 'a', imgs, gts, preds, classes=classes, palette=palette)
    for g, im, gt, pr in zip(got, imgs, gts, preds):
        assert np.array_equal(g, O.add_datasample(im, gt, pr, classes, palette))
    imgs, gts, preds = _case(1024, 2048, 2, seed=9)
    got = _draw_files(tmp_path / 'b', imgs, gts, preds, tensor_images=True)
    for g, im, gt, pr in zip(got, imgs, gts, preds):
        assert np.array_equal(g, O.add_datasample(im, gt, pr))


def test_row_wider_than_the_far_match_limit(tmp_path):
    """gt | pred rows of 2 * 5500 pixels: a scanline of 33001 bytes, past deflate's 32768 window (no match one row up)
    and alone in its band"""
    imgs, gts, preds = _case(24, 5500, 1, seed=3)
    got = _draw_files(tmp_path, imgs, gts, preds)
    assert np.array_equal(got[0], O.add_datasample(imgs[0], gts[0], preds[0]))


def test_out_file_and_other_backends(tmp_path):
    imgs, gts, preds = _case(90, 130, 1, seed=11)
    seen = []
    fake = types.SimpleNamespace(name='fake', add_image=lambda name, img, step=0: seen.append((name, img.copy(), step)))
    vis = V.SegLocalVisualizer(vis_backends=[fake])
    sample = dict(gt_sem_seg=dict(data=torch.from_numpy(gts[0])[None]),
                  pred_sem_seg=dict(data=torch.from_numpy(preds[0].astype(np.int64))[None].to(DEV)))
    want = O.add_datasample(imgs[0], gts[0], preds[0])
    vis.add_datasample('pic', imgs[0], sample, step=4)
    assert len(seen) == 1 and seen[0][0] == 'pic' and seen[0][2] == 4 and np.array_equal(seen[0][1], want)
    f = str(tmp_path / 'sub' / 'pic.png')
    vis.add_datasample('pic', imgs[0], sample, out_file=f, draw_gt=False)
    assert np.array_equal(_decoded(open(f, 'rb').read()), O.add_datasample(imgs[0], None, preds[0]))
    assert len(seen) == 1


# ---- RGB files and the pinned grey / palette bytes -------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['noise', 'smooth', 'flat'])
@pytest.mark.parametrize('hw', [(1, 1), (7, 13), (200, 333), (1024, 2048)])
def test_rgb_png_round_trips(kind, hw):
    h, w = hw
    rng = np.random.default_rng(h * w)
    if kind == 'noise':
        img = rng.integers(0, 256, (2, h, w, 3)).astype(np.uint8)
    elif kind == 'smooth':
        img = np.stack([O.photo(h, w, s) for s in range(2)])
    else:
        img = np.broadcast_to(rng.integers(0, 256, (2, 1, 1, 3)), (2, h, w, 3)).astype(np.uint8)
    files = ops.png_encode(torch.from_numpy(np.ascontiguousarray(img)).to(DEV))
    for f, want in zip(files, img):
        assert len(f) <= lib.get().ledb200_png_rgb_bound(h, w)
        assert np.array_equal(_decoded(f), want)
        assert f[25] == 2                                   # IHDR colour type
        raw = zlib.decompress(f[41:41 + int.from_bytes(f[33:37], 'big')])
        assert len(raw) == h * (3 * w + 1) and set(raw[::3 * w + 1]) <= set(range(5))
    if kind == 'smooth' and h > 100:
        assert len(set(zlib.decompress(files[0][41:41 + int.from_bytes(files[0][33:37], 'big')])[::3 * w + 1])) > 1
    with pytest.raises(lib.LedB200Error):
        ops.png_encode(torch.from_numpy(np.ascontiguousarray(img)).to(DEV), add=1)


def hash_cases():
    """seeded label maps whose grey / palette PNG bytes are pinned below (computed by the encoder before RGB support)"""
    rng = np.random.default_rng(2024)
    u8 = torch.from_numpy(rng.integers(0, 256, (3, 61, 97)).astype(np.uint8))
    i64 = torch.from_numpy(rng.integers(0, 40, (2, 45, 300)))
    full = torch.from_numpy(np.stack([P.blocky_labels(1024, 2048, seed=s) for s in range(2)]).astype(np.uint8))
    lut = rng.permutation(256)
    return [('u8_add0', u8, {}), ('u8_add1', u8, dict(add=1)), ('i64_add1', i64, dict(add=1)),
            ('i64_lut', i64, dict(lut=lut)), ('u8_palette', u8, dict(lut=lut, palette=True)),
            ('i64_palette', i64, dict(palette=True)), ('full_u8', full, {}), ('full_palette', full, dict(palette=True))]


def hashes():
    return {name: hashlib.sha256(b''.join(ops.png_encode(t.to(DEV), **kw))).hexdigest() for name, t, kw in hash_cases()}


# SHA-256 of each case's files, concatenated, as the encoder wrote them before it learned RGB files
PINNED = {
    'u8_add0': '1fdb21b4475eca983ba67156b6e3d03ba06c0c88b37b9aa451618115940f7420',
    'u8_add1': '9b35d6a0b9c64ab3d3c7fd0a2a1876d4e71f8c863437b53151bdc8f8c6dc4d9a',
    'i64_add1': '67a74e9e622deadc1ccd71c6024c77cf245c9db00ae32d3569843013fd3ae31d',
    'i64_lut': '432e4d3a41acdc5eb66e80bb8ed47cb0567f8f31e00e2ffa4210da1472118a4c',
    'u8_palette': '5644909d0ca75490a6fc375f7811f4dd8d5c50e3b2b9e25586a6f9847e942049',
    'i64_palette': 'b16de08723f1db06e9d02683962303f8c08235160ebcba348466b15d2377fbe9',
    'full_u8': 'db292dab4bdbfe39d28e346719689c1d295cf98f227c59ec19fcfad86e5823ec',
    'full_palette': 'ee3b22d65ed625b8cf869396e03439d08cb9df240a092ddda9130056f3e45086',
}


def test_grey_and_palette_bytes_are_unchanged():
    assert hashes() == PINNED


# ---- the hook -------------------------------------------------------------------------------------------------------------
def _dataset(tmp_path, n, h, w, K=19, jpeg=True):
    pack = L.PackSegFiles()
    items = []
    for i in range(n):
        img = J.photo(h, w, seed=60 + i)
        lab = P.blocky_labels(h, w, seed=70 + i, k=K)
        use_jpeg = jpeg and i % 2 == 0
        ip, lp = tmp_path / (f'img{i}.jpg' if use_jpeg else f'img{i}.png'), tmp_path / f'img{i}_gt.png'
        ip.write_bytes(J.cv2_jpeg(img, 95, '420') if use_jpeg else cv2.imencode('.png', img)[1].tobytes())
        lp.write_bytes(P.png(lab[..., None], 0))
        items.append(pack(dict(img_path=str(ip), seg_map_path=str(lp), reduce_zero_label=False, label_map=None)))
    return items


def _batch(items):
    return dict(inputs=[it['inputs'] for it in items],
                data_samples=[dict(it['data_samples'], metainfo=dict(it['data_samples']['metainfo'])) for it in items])


def _want(path, seg_path, pred):
    img = cv2.imread(path, cv2.IMREAD_COLOR)[..., ::-1]             # mmcv.imfrombytes(channel_order='rgb')
    gt = np.array(Image.open(seg_path))
    return O.add_datasample(np.ascontiguousarray(img), gt, pred)


@pytest.mark.parametrize('decoded', [True, False])
def test_hook_after_test_iter_writes_the_oracle_pictures(tmp_path, decoded):
    K = 19
    (tmp_path / 'data').mkdir()
    items = _dataset(tmp_path / 'data', 3, 128, 256, K)
    m = _model(K)
    save = str(tmp_path / 'show')
    V.SegLocalVisualizer(save_dir=save, vis_backends=[dict(type='LocalVisBackend')])
    hook = V.SegVisualizationHook(draw=True)
    runner = types.SimpleNamespace(iter=0)
    steps = []
    for b0 in (0, 2):
        batch = _batch(items[b0:b0 + 2])
        with torch.no_grad():
            outs = m.test_step(batch)
        if decoded:
            assert isinstance(batch['inputs'], L.png_feed.DecodedFiles)
        else:
            batch['inputs'] = list(batch['inputs'])                   # as if decoded elsewhere: read the files again
        hook.after_test_iter(runner, b0 // 2, batch, outs)
        for k, (o, s) in enumerate(zip(outs, batch['data_samples'])):
            meta = s['metainfo']
            steps.append(b0 + k + 1)
            f = os.path.join(save, 'vis_data', 'vis_image', f'{os.path.basename(meta["img_path"])}_{b0 + k + 1}.png')
            got = _decoded(open(f, 'rb').read())
            pred = o['pred_sem_seg']['data'][0].cpu().numpy()
            assert np.array_equal(got, _want(meta['img_path'], meta['seg_map_path'], pred))
    assert hook._test_index == 3 and steps == [1, 2, 3]


def test_hook_after_val_iter_interval_and_names(tmp_path):
    items = _dataset(tmp_path, 2, 64, 96, jpeg=False)
    m = _model(19)
    seen = []
    fake = types.SimpleNamespace(name='fake', add_image=lambda name, img, step=0: seen.append((name, img, step)))
    V.SegLocalVisualizer(vis_backends=[fake])
    hook = V.SegVisualizationHook(draw=True, interval=4)
    for it, bi in ((3, 1), (5, 0), (2, 2)):
        batch = _batch(items)
        with torch.no_grad():
            outs = m.test_step(batch)
        hook.after_val_iter(types.SimpleNamespace(iter=it), bi, batch, outs)
    assert [(n, s) for n, _, s in seen] == [('val_img0.png', 4), ('val_img0.png', 4)]
    meta = items[0]['data_samples']['metainfo']
    pred = outs[0]['pred_sem_seg']['data'][0].cpu().numpy()
    assert np.array_equal(seen[-1][1], _want(meta['img_path'], meta['seg_map_path'], pred))
    with pytest.warns(UserWarning):
        off = V.SegVisualizationHook(draw=False)
    off.after_val_iter(types.SimpleNamespace(iter=0), 0, _batch(items), outs)
    assert len(seen) == 2
