"""Segmentation overlays on the device: `SegLocalVisualizer` (VISUALIZERS) and `SegVisualizationHook` (HOOKS), what
mmseg's `tools/test.py --show-dir` draws.

mmseg 1.2.2's SegLocalVisualizer._draw_sem_seg colours each pixel with palette[label] (labels >= len(classes) stay
black), draws every present class's name in a box at its _get_center_loc (classes in descending order, later boxes over
earlier ones) and blends `(image * (1 - alpha) + mask * alpha).astype(np.uint8)`; add_datasample puts the gt and pred
panels side by side and LocalVisBackend writes the picture as a PNG.  Here:
  * ops.seg_label_locations finds every class's location of a whole batch in one launch sequence; one copy brings the
    locations back (only with `with_labels`);
  * cv2 draws each label box and its text on the host, but only into a small stamp (see `_Stamps`), since only cv2
    draws its Hershey text bit for bit;
  * ops.seg_overlay blends every pixel through a 256 x 256 table built with numpy's float64 expression
    (ops.blend_table), which is exact where float32 or fused multiply-add arithmetic is not, and writes the stamps;
  * ops.png_encode writes the RGB files on the device; only their bytes come back for LocalVisBackend.  Any other
    backend (TensorboardVisBackend, or an instance passed in) receives the drawn HWC RGB array through add_image.
Every step runs per shape group of a batch.  cv2 is imported only when labels are drawn.
"""
import os
import warnings
from collections import OrderedDict

import numpy as np
import torch

from . import ops
from .lib import LedB200Error
from .metrics import _sample_meta
from .png_feed import DecodedFiles, _is_jpeg, _read
from .registry import HOOKS, VISUALIZERS

CITYSCAPES_CLASSES = ('road', 'sidewalk', 'building', 'wall', 'fence', 'pole', 'traffic light', 'traffic sign',
                      'vegetation', 'terrain', 'sky', 'person', 'rider', 'car', 'truck', 'bus', 'train', 'motorcycle',
                      'bicycle')
CITYSCAPES_PALETTE = [[128, 64, 128], [244, 35, 232], [70, 70, 70], [102, 102, 156], [190, 153, 153], [153, 153, 153],
                      [250, 170, 30], [220, 220, 0], [107, 142, 35], [152, 251, 152], [70, 130, 180], [220, 20, 60],
                      [255, 0, 0], [0, 0, 142], [0, 0, 70], [0, 60, 100], [0, 80, 100], [0, 0, 230], [119, 11, 32]]


def _get(obj, key):
    """a field of a dict or of an attribute-style data sample (SegDataSample, PixelData)"""
    if obj is None:
        return None
    if isinstance(obj, dict):
        return obj.get(key, None)
    return getattr(obj, key, None)


def text_style(h, w):
    """(fontScale, thickness) of _draw_sem_seg's labels on an h x w image"""
    scale = 0.05
    return min(h, w) / (25 / scale), 1 if h < 300 or w < 300 else 2


class _Stamps:
    """Label boxes drawn by cv2 into small stamps.

    A stamp covers a label's box plus a margin wide enough for the outline and the text.  cv2 draws the box, outline and
    text (exactly _draw_sem_seg's three calls) onto two canvases of that size, one black and one white; a pixel is
    "touched" where the two agree, and then holds the drawn colour.  Where the margin box crosses an image edge the
    canvas is cut at that edge, so cv2 clips there exactly as it does on the full mask.  A stamp that reaches no edge
    depends only on (text, colour, fontScale, thickness) and is cached."""

    def __init__(self):
        self._cache = {}

    @staticmethod
    def _draw(cv2, canvas, x, y, text, color, font_scale, thickness):
        (lw, lh), base = cv2.getTextSize(text, cv2.FONT_HERSHEY_SIMPLEX, font_scale, thickness)
        cv2.rectangle(canvas, (x, y), (x + lw + base, y + lh + base), color, -1)
        cv2.rectangle(canvas, (x, y), (x + lw + base, y + lh + base), (0, 0, 0), thickness)
        cv2.putText(canvas, text, (x, y + lh), cv2.FONT_HERSHEY_SIMPLEX, font_scale, (255, 255, 255), thickness, 2)

    def make(self, text, color, font_scale, thickness, x, y, H, W):
        """(x0, y0, pixels [h, w, 4] uint8 (R, G, B, touched)) of the label at (x, y) on an H x W panel"""
        import cv2
        color = tuple(int(c) for c in color)
        (lw, lh), base = cv2.getTextSize(text, cv2.FONT_HERSHEY_SIMPLEX, font_scale, thickness)
        m = lh + base + 2 * thickness + 2
        x0, y0, x1, y1 = x - m, y - m, x + lw + base + m + 1, y + lh + base + m + 1
        cx0, cy0, cx1, cy1 = max(0, x0), max(0, y0), min(W, x1), min(H, y1)
        inner = (cx0, cy0, cx1, cy1) == (x0, y0, x1, y1)
        key = (text, color, font_scale, thickness)
        if inner and key in self._cache:
            return x0, y0, self._cache[key]
        a = np.zeros((cy1 - cy0, cx1 - cx0, 3), np.uint8)
        b = np.full_like(a, 255)
        for canvas in (a, b):
            self._draw(cv2, canvas, x - cx0, y - cy0, text, color, font_scale, thickness)
        pix = np.concatenate([a, np.all(a == b, axis=-1, keepdims=True).astype(np.uint8)], axis=-1)
        if inner:
            self._cache[key] = pix
        return cx0, cy0, pix


class LocalImageBackend:
    """mmengine's LocalVisBackend for images, fed device-encoded PNG bytes: `{save_dir}/{img_save_dir}/{name}_{step}.png`.
    Other calls (scalars, config) go to `inner`, mmengine's own LocalVisBackend when mmengine is importable."""

    def __init__(self, save_dir, img_save_dir='vis_image', inner=None, **kwargs):
        self.save_dir = save_dir
        self.img_dir = os.path.join(save_dir, img_save_dir)
        self._inner = inner

    def write(self, name, step, data):
        os.makedirs(self.img_dir, exist_ok=True)
        with open(os.path.join(self.img_dir, f'{name}_{step}.png'), 'wb') as f:
            f.write(data)

    def add_image(self, name, image, step=0, **kwargs):
        """a host HWC RGB uint8 image, encoded on the current device"""
        t = torch.from_numpy(np.ascontiguousarray(image)).cuda()
        self.write(name, step, ops.png_encode(t[None])[0])

    def __getattr__(self, key):
        inner = self.__dict__.get('_inner')
        if inner is None:
            raise AttributeError(key)
        return getattr(inner, key)


def _build_backend(cfg, save_dir):
    cfg = dict(cfg)
    typ = cfg.pop('type')
    cfg.pop('name', None)
    cfg.setdefault('save_dir', save_dir)
    try:
        from mmengine.registry import VISBACKENDS
    except Exception:
        VISBACKENDS = None
    if typ in ('LocalVisBackend', 'mmengine.LocalVisBackend'):
        inner = VISBACKENDS.build(dict(cfg, type=typ)) if VISBACKENDS is not None else None
        return LocalImageBackend(inner=inner, **cfg)
    if VISBACKENDS is None:
        raise ImportError(f'{typ} needs mmengine (only LocalVisBackend is built without it)')
    return VISBACKENDS.build(dict(cfg, type=typ))


@VISUALIZERS.register_module()
class SegLocalVisualizer:
    """mmseg's SegLocalVisualizer (mmseg/visualization/local_visualizer.py) drawing on the device.

    vis_backends: dicts (LocalVisBackend is written natively; other types are built through mmengine's VISBACKENDS) or
    backend instances.  As in mmengine, dict backends are built only with a save_dir, under `{save_dir}/vis_data`.
    classes / palette default to Cityscapes'; the runner replaces them with the dataset's metainfo through
    `dataset_meta`.  At most 255 classes."""

    _current = None

    def __init__(self, name='visualizer', image=None, vis_backends=None, save_dir=None, classes=None, palette=None,
                 dataset_name=None, alpha=0.8, **kwargs):
        self.name = name
        self.alpha = alpha
        self._backends = OrderedDict()
        for k, b in enumerate(vis_backends or []):
            if isinstance(b, dict):
                if save_dir is None:
                    warnings.warn('SegLocalVisualizer: backend dicts are ignored without a save_dir')
                    continue
                key = b.get('name', b['type'])
                self._backends[key] = _build_backend(b, os.path.join(save_dir, 'vis_data'))
            else:
                self._backends[getattr(b, 'name', f'backend{k}')] = b
        self.set_dataset_meta(classes, palette, dataset_name)
        self._stamps = _Stamps()
        self._dev_tables = {}
        SegLocalVisualizer._current = self

    @classmethod
    def get_current_instance(cls):
        """the SegLocalVisualizer built last (mmengine's ManagerMixin.get_current_instance)"""
        if SegLocalVisualizer._current is None:
            raise RuntimeError('no SegLocalVisualizer has been built yet')
        return SegLocalVisualizer._current

    def set_dataset_meta(self, classes=None, palette=None, dataset_name='cityscapes'):
        if dataset_name not in (None, 'cityscapes') and not (classes and palette):
            raise NotImplementedError(f"the default classes and palette of {dataset_name!r} (only 'cityscapes' is built "
                                      'in: give classes and palette)')
        classes = classes if classes else CITYSCAPES_CLASSES
        palette = palette if palette else CITYSCAPES_PALETTE
        assert len(classes) == len(palette), 'The length of classes should be equal to palette'
        self.dataset_meta = {'classes': classes, 'palette': palette}

    def get_backend(self, name):
        return self._backends.get(name)

    def _forward(self, method, *args, **kwargs):
        for b in self._backends.values():
            fn = getattr(b, method, None)
            if fn is not None:
                fn(*args, **kwargs)

    def add_config(self, config, **kwargs):
        self._forward('add_config', config, **kwargs)

    def add_graph(self, model, data_batch, **kwargs):
        self._forward('add_graph', model, data_batch, **kwargs)

    def add_scalar(self, name, value, step=0, **kwargs):
        self._forward('add_scalar', name, value, step, **kwargs)

    def add_scalars(self, scalar_dict, step=0, file_path=None, **kwargs):
        self._forward('add_scalars', scalar_dict, step, file_path, **kwargs)

    def close(self):
        self._forward('close')

    # -- drawing ---------------------------------------------------------------------------------------------------------
    def _tables(self, device):
        """(palette [K,3], blend table [256,256]) on `device`, built once per (device, palette, alpha)"""
        pal = np.asarray(self.dataset_meta['palette'], dtype=np.int64).reshape(-1, 3)
        if len(pal) > 255 or pal.min() < 0 or pal.max() > 255:
            raise LedB200Error('SegLocalVisualizer: at most 255 classes, palette values in 0 .. 255')
        key = (str(device), pal.tobytes(), float(self.alpha))
        if key not in self._dev_tables:
            self._dev_tables[key] = (torch.from_numpy(pal.astype(np.uint8)).to(device),
                                     torch.from_numpy(ops.blend_table(self.alpha)).to(device))
        return self._dev_tables[key]

    @staticmethod
    def _as_image(image):
        """[3, h, w] uint8 BGR CUDA tensor from the decoders' tensor or mmseg's HWC RGB array"""
        if isinstance(image, torch.Tensor):
            if image.dtype != torch.uint8 or image.dim() != 3 or image.shape[0] != 3:
                raise LedB200Error('SegLocalVisualizer: image tensors are [3, h, w] uint8 BGR')
            return image if image.is_cuda else image.cuda()
        image = np.asarray(image)
        if image.dtype != np.uint8 or image.ndim != 3 or image.shape[2] != 3:
            raise LedB200Error('SegLocalVisualizer: image arrays are HWC RGB uint8')
        return torch.from_numpy(np.ascontiguousarray(image[..., ::-1].transpose(2, 0, 1))).cuda()

    @staticmethod
    def _as_map(m, device, hw):
        if m is None:
            return None
        m = torch.as_tensor(m).to(device)
        if m.dtype not in (torch.uint8, torch.int64):
            m = m.to(torch.int64)
        if m.numel() != hw[0] * hw[1]:
            raise LedB200Error(f'SegLocalVisualizer: a label map of {tuple(m.shape)} for an image of {tuple(hw)}')
        return m.reshape(hw)

    def add_datasample(self, name, image, data_sample=None, draw_gt=True, draw_pred=True, show=False, wait_time=0,
                       out_file=None, step=0, with_labels=True):
        """mmseg's add_datasample for one image: image HWC RGB uint8 (numpy) or the decoders' [3, h, w] uint8 BGR
        tensor.  With out_file the picture is written there (PNG only); otherwise it goes to every backend."""
        self.add_datasamples([name], [image], [data_sample], [step], draw_gt, draw_pred, show, wait_time,
                             None if out_file is None else [out_file], with_labels)

    def add_datasamples(self, names, images, data_samples, steps, draw_gt=True, draw_pred=True, show=False,
                        wait_time=0, out_files=None, with_labels=True):
        """add_datasample for a batch: per group of same-shape images one seg_label_locations call (with labels), one
        seg_overlay call and one png_encode call, then the files."""
        if show:
            raise NotImplementedError('SegLocalVisualizer: show=True (windows) is not supported; write files with '
                                      'out_file or a save_dir')
        if out_files is not None:
            for f in out_files:
                if os.path.splitext(f)[1].lower() != '.png':
                    raise NotImplementedError(f'{f}: SegLocalVisualizer writes PNG files only')
        classes = self.dataset_meta['classes']
        K = len(classes)
        groups = OrderedDict()
        items = []
        for i, (image, s) in enumerate(zip(images, data_samples)):
            img = self._as_image(image)
            hw = tuple(img.shape[1:])
            gt = self._as_map(_get(_get(s, 'gt_sem_seg'), 'data'), img.device, hw) if draw_gt else None
            pred = self._as_map(_get(_get(s, 'pred_sem_seg'), 'data'), img.device, hw) if draw_pred else None
            if gt is None and pred is None:
                raise LedB200Error(f'{names[i]}: the data sample has neither gt_sem_seg nor pred_sem_seg to draw')
            items.append((img, gt, pred))
            key = (hw, str(img.device), None if gt is None else gt.dtype, None if pred is None else pred.dtype)
            groups.setdefault(key, []).append(i)
        for (hw, _, _, _), idx in groups.items():
            imgs = torch.stack([items[i][0] for i in idx])
            gts = None if items[idx[0]][1] is None else torch.stack([items[i][1] for i in idx])
            preds = None if items[idx[0]][2] is None else torch.stack([items[i][2] for i in idx])
            palette, table = self._tables(imgs.device)
            stamps = data = None
            if with_labels:
                stamps, data = self._stamp_batch(gts, preds, classes, hw)
            drawn = ops.seg_overlay(imgs, gts, preds, palette, table, stamps, data)
            self._emit(drawn, [names[i] for i in idx], [steps[i] for i in idx],
                       None if out_files is None else [out_files[i] for i in idx])

    def _stamp_batch(self, gts, preds, classes, hw):
        """every label stamp of a group: one locate call over all panels, one copy back, cv2 stamps, one upload"""
        maps = [m for m in (gts, preds) if m is not None]
        if len(maps) == 2 and maps[0].dtype != maps[1].dtype:
            maps = [m.to(torch.int64) for m in maps]
        K, (H, W) = len(classes), hw
        loc = ops.seg_label_locations(torch.cat(maps) if len(maps) == 2 else maps[0], K).cpu().numpy()
        n = len(maps[0])
        palette = self.dataset_meta['palette']
        font_scale, thickness = text_style(H, W)
        desc, chunks, at, placed = [], [], 0, {}           # a cached stamp's pixels are uploaded once per call
        for p in range(len(maps)):
            for j in range(n):
                lj = loc[p * n + j]
                for k in range(K - 1, -1, -1):
                    if not lj[k, 0]:
                        continue
                    x0, y0, pix = self._stamps.make(classes[k], palette[k], font_scale, thickness, int(lj[k, 1]),
                                                    int(lj[k, 2]), H, W)
                    if id(pix) not in placed:
                        placed[id(pix)] = at
                        chunks.append(pix.reshape(-1))
                        at += pix.size
                    desc.append((j, p, x0, y0, pix.shape[1], pix.shape[0], placed[id(pix)]))
        if not desc:
            return None, None
        head = np.array(desc, dtype=ops.STAMP_DTYPE).view(np.uint8)
        host = torch.empty(len(head) + at, dtype=torch.uint8, pin_memory=True)
        view = host.numpy()
        view[:len(head)] = head
        view[len(head):] = np.concatenate(chunks)
        dev = host.to(maps[0].device, non_blocking=True)
        return dev[:len(head)], dev[len(head):]

    def _emit(self, drawn, names, steps, out_files):
        """the drawn [n, H, P*W, 3] RGB pictures to out_files or to every backend"""
        local = [b for b in self._backends.values() if isinstance(b, LocalImageBackend)]
        files = ops.png_encode(drawn) if out_files is not None or local else None
        if out_files is not None:
            for f, data in zip(out_files, files):
                d = os.path.dirname(os.path.abspath(f))
                os.makedirs(d, exist_ok=True)
                with open(f, 'wb') as fh:
                    fh.write(data)
            return
        for b in local:
            for name, step, data in zip(names, steps, files):
                b.write(name, step, data)
        others = [b for b in self._backends.values() if not isinstance(b, LocalImageBackend)]
        if others:
            host = drawn.cpu().numpy()
            for b in others:
                for name, step, img in zip(names, steps, host):
                    b.add_image(name, img, step)


@HOOKS.register_module()
class SegVisualizationHook:
    """mmseg's SegVisualizationHook (mmseg/engine/hooks/visualization_hook.py) over the batched device visualizer.

    The image drawn under each prediction is the file's pixels (mmcv.imfrombytes(channel_order='rgb') in mmseg).  When
    the batch came through PackSegFiles, decode_batch has already decoded it on the device (data_batch['inputs']);
    otherwise each img_path is read and decoded with ops.png_decode / ops.jpeg_decode, bit-identical to cv2.  A sample's
    img_path and gt_sem_seg are taken from the output, else from the batch's data sample."""

    priority = 'NORMAL'

    def __init__(self, draw=False, interval=50, show=False, wait_time=0., backend_args=None):
        if show:
            raise NotImplementedError('SegVisualizationHook: show=True (windows) is not supported; use --show-dir')
        self._visualizer = SegLocalVisualizer.get_current_instance()
        self.interval = interval
        self.show = show
        self.wait_time = wait_time
        self.backend_args = backend_args.copy() if backend_args else None
        if self.backend_args:
            raise NotImplementedError('SegVisualizationHook: backend_args (files are read from the local disk)')
        self.draw = draw
        if not self.draw:
            warnings.warn('The draw is False, it means that the hook for visualization will not take effect. The '
                          'results will NOT be visualized or stored.')
        self._test_index = 0

    @staticmethod
    def _merged(out, batch_sample):
        """(img_path, the sample to draw: pred from the output, gt from the output or else the batch)"""
        path = _sample_meta(out, 'img_path') if isinstance(out, dict) else getattr(out, 'img_path', None)
        if path is None and batch_sample is not None:
            path = _sample_meta(batch_sample, 'img_path') if isinstance(batch_sample, dict) else \
                getattr(batch_sample, 'img_path', None)
        gt = _get(out, 'gt_sem_seg')
        if gt is None:
            gt = _get(batch_sample, 'gt_sem_seg')
        return path, dict(gt_sem_seg=gt, pred_sem_seg=_get(out, 'pred_sem_seg'))

    @staticmethod
    def _images(data_batch, indices, paths):
        inputs = data_batch.get('inputs', None) if isinstance(data_batch, dict) else None
        if isinstance(inputs, DecodedFiles):
            return [inputs[i] for i in indices]
        files = [_read(p) for p in paths]
        images = [None] * len(files)
        for is_jpeg, decode in ((False, ops.png_decode), (True, ops.jpeg_decode)):
            idx = [k for k, f in enumerate(files) if _is_jpeg(f) == is_jpeg]
            if idx:
                for k, img in zip(idx, decode([files[k] for k in idx], names=[paths[k] for k in idx])):
                    images[k] = img
        return images

    def _batch_samples(self, data_batch, n):
        samples = data_batch.get('data_samples', None) if isinstance(data_batch, dict) else None
        return list(samples) if samples is not None else [None] * n

    def after_val_iter(self, runner, batch_idx, data_batch, outputs):
        if self.draw is False:
            return
        step = runner.iter + batch_idx
        if step % self.interval != 0:
            return
        path, sample = self._merged(outputs[0], self._batch_samples(data_batch, len(outputs))[0])
        img = self._images(data_batch, [0], [path])[0]
        self._visualizer.add_datasamples([f'val_{os.path.basename(path)}'], [img], [sample], [step],
                                         wait_time=self.wait_time)

    def after_test_iter(self, runner, batch_idx, data_batch, outputs):
        if self.draw is False:
            return
        batch = self._batch_samples(data_batch, len(outputs))
        merged = [self._merged(o, b) for o, b in zip(outputs, batch)]
        paths = [p for p, _ in merged]
        steps = []
        for _ in outputs:
            self._test_index += 1
            steps.append(self._test_index)
        images = self._images(data_batch, list(range(len(outputs))), paths)
        self._visualizer.add_datasamples([os.path.basename(p) for p in paths], images, [s for _, s in merged], steps,
                                         wait_time=self.wait_time)
