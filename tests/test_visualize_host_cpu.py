"""SegLocalVisualizer's host side without a GPU: the oracle (tests/vis_oracle.py) on hand-made cases, the cv2 label stamps
against drawing on the full mask, the blend table against numpy, the refused cases and the registry entries."""
import subprocess
import sys
import os

import numpy as np
import pytest

import lednet_b200 as L
from lednet_b200 import ops, visualization as V
import vis_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the oracle ----------------------------------------------------------------------------------------------------------------
def test_center_loc_ties_and_single_pixels():
    m = np.zeros((6, 9), np.uint8)
    m[1, [2, 3, 4]] = 1
    m[4, [0, 5, 8]] = 1                       # a tie of three: the first row wins
    assert O.get_center_loc(m).tolist() == [3, 1]
    m[4, 7] = 1                               # row 4 now has four: index 2 in x order is x = 7
    assert O.get_center_loc(m).tolist() == [7, 4]
    s = np.zeros((5, 5), np.uint8)
    s[3, 2] = 1
    assert O.get_center_loc(s).tolist() == [2, 3]


def test_labels_at_or_above_k_are_not_drawn():
    img = O.photo(20, 30, 0)
    sem = np.full((20, 30), 255, np.uint8)
    sem[:5] = 19
    out = O.draw_sem_seg(img, sem, O.CITYSCAPES_CLASSES, O.CITYSCAPES_PALETTE, True)
    assert np.array_equal(out, (img * 0.19999999999999996).astype(np.uint8))     # no legal label: a black mask
    sem[10:, :4] = 3
    out = O.draw_sem_seg(img, sem, O.CITYSCAPES_CLASSES, O.CITYSCAPES_PALETTE, False)
    want = (img * (1 - 0.8)).astype(np.uint8)
    want[10:, :4] = (img[10:, :4] * (1 - 0.8) + np.array(O.CITYSCAPES_PALETTE[3]) * 0.8).astype(np.uint8)
    assert np.array_equal(out, want)


@pytest.mark.parametrize('hw,style', [((299, 1000), (299 / 500, 1)), ((300, 300), (300 / 500, 2)),
                                      ((1024, 2048), (1024 / 500, 2)), ((512, 200), (200 / 500, 1))])
def test_text_style_thickness_switch(hw, style):
    fs, th = O.text_style(*hw)
    assert th == style[1] and abs(fs - style[0]) < 1e-12
    assert V.text_style(*hw) == O.text_style(*hw)


def test_blend_table_equals_numpy():
    rng = np.random.default_rng(0)
    i = rng.integers(0, 256, 5000).astype(np.uint8)
    c = rng.integers(0, 256, 5000).astype(np.uint8)
    for alpha in (0.8, 0.6, 0.5, 0.3, 1.0, 0.0, 0.75):
        t = ops.blend_table(alpha)
        assert t.shape == (256, 256) and t.dtype == np.uint8
        assert np.array_equal(t[i, c], (i * (1 - alpha) + c * alpha).astype(np.uint8))
    # float32 arithmetic would not do: the table differs from it at 0.8
    v = np.arange(256, dtype=np.float32)
    f32 = (v[:, None] * np.float32(1 - 0.8) + v[None, :] * np.float32(0.8)).astype(np.uint8)
    assert (f32 != ops.blend_table(0.8)).sum() > 0


# ---- stamps --------------------------------------------------------------------------------------------------------------------
def _stamped(mask_hw, labels):
    """the labels drawn through V._Stamps onto a mask whose untouched pixels are the palette colours"""
    H, W = mask_hw
    fs, th = O.text_style(H, W)
    st = V._Stamps()
    rng = np.random.default_rng(1)
    base = rng.integers(0, 256, (H, W, 3)).astype(np.uint8)
    full, via = base.copy(), base.copy()
    for text, color, x, y in labels:
        O.draw_label(full, (x, y), text, color, fs, th)
        x0, y0, pix = st.make(text, color, fs, th, x, y, H, W)
        h, w = pix.shape[:2]
        assert 0 <= x0 and 0 <= y0 and x0 + w <= W and y0 + h <= H
        region = via[y0:y0 + h, x0:x0 + w]
        region[pix[..., 3] == 1] = pix[..., :3][pix[..., 3] == 1]
    return full, via, st


@pytest.mark.parametrize('hw', [(1024, 2048), (200, 260), (512, 512), (40, 30)])
def test_stamps_equal_drawing_on_the_full_mask(hw):
    H, W = hw
    rng = np.random.default_rng(H + W)
    names = ['road', 'traffic light', 'sky', 'motorcycle', 'vegetation']
    labels = []
    for k in range(120):
        edge = k % 4
        x = int(rng.integers(0, W)) if edge != 1 else int(W - 1 - rng.integers(0, 8))
        y = int(rng.integers(0, H)) if edge != 2 else int(H - 1 - rng.integers(0, 8))
        if edge == 3:
            x, y = int(rng.integers(0, 4)), int(rng.integers(0, 4))
        labels.append((names[k % 5], O.CITYSCAPES_PALETTE[k % 19], x, y))
    full, via, st = _stamped(hw, labels)          # overlapping labels, later ones over earlier ones
    assert np.array_equal(full, via)


def test_stamp_cache_reuses_inner_stamps():
    full, via, st = _stamped((600, 800), [('car', (0, 0, 142), 100, 100), ('car', (0, 0, 142), 400, 300),
                                         ('car', (0, 0, 142), 795, 590)])
    assert np.array_equal(full, via)
    assert len(st._cache) == 1


def test_device_composition_equals_the_oracle_on_the_host():
    """the device path's arithmetic restated on the host: table[image][stamp or palette colour] with the oracle's
    locations must give the oracle's picture"""
    H, W = 180, 240
    img = O.photo(H, W, 3)
    sem = O.blocky_map(H, W, 19, seed=4, cell=30)
    classes, palette = O.CITYSCAPES_CLASSES, O.CITYSCAPES_PALETTE
    for alpha in (0.8, 0.6):
        want = O.draw_sem_seg(img, sem, classes, palette, True, alpha)
        pal = np.array(palette + [[0, 0, 0]] * (256 - 19), np.uint8)
        colour = pal[sem]
        fs, th = O.text_style(H, W)
        st = V._Stamps()
        for k in sorted(set(np.unique(sem)) - {255}, reverse=True):
            x, y = O.get_center_loc((sem == k).astype(np.uint8))
            x0, y0, pix = st.make(classes[k], palette[k], fs, th, int(x), int(y), H, W)
            h, w = pix.shape[:2]
            t = pix[..., 3] == 1
            colour[y0:y0 + h, x0:x0 + w][t] = pix[..., :3][t]
        got = ops.blend_table(alpha)[img, colour]
        assert np.array_equal(got, want)


# ---- refused cases, registry, imports ------------------------------------------------------------------------------------------
def test_refused_cases(tmp_path):
    vis = V.SegLocalVisualizer()
    sample = dict(pred_sem_seg=dict(data=np.zeros((1, 4, 4), np.int64)))
    with pytest.raises(NotImplementedError, match='show'):
        vis.add_datasample('x', np.zeros((4, 4, 3), np.uint8), sample, show=True)
    with pytest.raises(NotImplementedError, match='PNG'):
        vis.add_datasample('x', np.zeros((4, 4, 3), np.uint8), sample, out_file=str(tmp_path / 'x.jpg'))
    with pytest.raises(NotImplementedError, match='show'):
        V.SegVisualizationHook(draw=True, show=True)
    with pytest.raises(NotImplementedError):
        V.SegLocalVisualizer(dataset_name='ade20k')


def test_defaults_and_registry(tmp_path):
    vis = L.VISUALIZERS.build(dict(type='SegLocalVisualizer', save_dir=str(tmp_path),
                                   vis_backends=[dict(type='LocalVisBackend')]))
    assert isinstance(vis, V.SegLocalVisualizer) and vis.alpha == 0.8
    assert list(vis.dataset_meta['classes']) == list(O.CITYSCAPES_CLASSES)
    assert [list(p) for p in vis.dataset_meta['palette']] == O.CITYSCAPES_PALETTE
    b = vis.get_backend('LocalVisBackend')
    assert isinstance(b, V.LocalImageBackend) and b.img_dir == os.path.join(str(tmp_path), 'vis_data', 'vis_image')
    hook = L.HOOKS.build(dict(type='SegVisualizationHook', draw=True, interval=5))
    assert hook._visualizer is vis and hook.interval == 5
    assert V.SegLocalVisualizer.get_current_instance() is vis
    with pytest.warns(UserWarning):
        V.SegVisualizationHook()
    vis.set_dataset_meta(classes=['a', 'b'], palette=[[1, 2, 3], [4, 5, 6]])
    assert vis.dataset_meta == {'classes': ['a', 'b'], 'palette': [[1, 2, 3], [4, 5, 6]]}


def test_importing_the_package_does_not_import_cv2():
    code = 'import sys, lednet_b200; print("cv2" in sys.modules)'
    out = subprocess.run([sys.executable, '-c', code], cwd=ROOT, capture_output=True, text=True, check=True)
    assert out.stdout.strip() == 'False'
