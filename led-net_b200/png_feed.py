"""Image and label files straight into the device preprocessors: `PackSegFiles` / `PackSegPNGFiles` (TRANSFORMS) and
`decode_batch`.

A dataset pipeline of LoadImageFromFile, LoadAnnotations and PackSegInputs decodes every file on a dataloader worker
(cv2 / PIL) and moves the decoded uint8 arrays.  `PackSegFiles` replaces the three: it reads the files' bytes and their
headers (PNG IHDR, JPEG markers up to the scan), and packs the file bytes with the metainfo PackSegInputs would set.
Images are PNG or baseline JPEG, label maps PNG.  `decode_batch`, called at the top of SegDataPreProcessor.forward,
DeviceAugSegDataPreProcessor.forward and SegTTAModel's device-view test_step, decodes such a batch on the device
(ops.png_decode for the PNG images, ops.jpeg_decode for the JPEG ones, ops.png_decode for the label maps: one call
each) into exactly the batch the decoded path delivers, so everything after it runs unchanged.
"""
import torch

from .registry import TRANSFORMS
from . import ops


def _read(path):
    with open(path, 'rb') as f:
        return f.read()


def _as_tensor(b):
    return torch.frombuffer(bytearray(b), dtype=torch.uint8)


def _is_jpeg(f):
    return ops._head(f, 2) == ops.JPEG_SOI


@TRANSFORMS.register_module()
class PackSegFiles:
    """LoadImageFromFile + LoadAnnotations + PackSegInputs for PNG and JPEG datasets, without decoding.

    Returns dict(inputs=<the image file as a 1-D uint8 tensor>, data_samples=<sample dict>), the sample holding
    `metainfo` (img_path, ori_shape and img_shape from the file's header, and with a label map seg_map_path,
    reduce_zero_label and label_map) and, when `seg_map_path` is set, the label file as `gt_seg_map_file`.  Images are
    PNG or baseline JPEG, told apart by their signature; label maps are PNG.  reduce_zero_label: None takes the dataset's
    results['reduce_zero_label'], as LoadAnnotations does.  A file the decoders cannot read (16-bit or interlaced PNG, a
    colour label map, progressive / CMYK / RGB JPEG, an Exif orientation other than 1) raises NotImplementedError here,
    on the worker."""

    jpeg_images = True

    def __init__(self, reduce_zero_label=None):
        self.reduce_zero_label = reduce_zero_label

    def __call__(self, results):
        img_path = results['img_path']
        img = _read(img_path)
        h, w, _ = ops.jpeg_info(img) if self.jpeg_images and _is_jpeg(img) else ops.png_info(img)
        meta = dict(img_path=img_path, ori_shape=(h, w), img_shape=(h, w))
        sample = dict(metainfo=meta)
        seg_path = results.get('seg_map_path', None)
        if seg_path is not None:
            rzl = self.reduce_zero_label
            if rzl is None:
                rzl = results.get('reduce_zero_label', False)
            assert rzl == results.get('reduce_zero_label', rzl), \
                f'Initialize dataset with `reduce_zero_label` consistently with {type(self).__name__}'
            seg = _read(seg_path)
            ops.png_info(seg, 'label')
            meta.update(seg_map_path=seg_path, reduce_zero_label=bool(rzl), label_map=results.get('label_map', None))
            sample['gt_seg_map_file'] = _as_tensor(seg)
        elif 'reduce_zero_label' in results:
            meta['reduce_zero_label'] = results['reduce_zero_label']
        return dict(inputs=_as_tensor(img), data_samples=sample)

    def __repr__(self):
        return f'{self.__class__.__name__}(reduce_zero_label={self.reduce_zero_label})'


@TRANSFORMS.register_module()
class PackSegPNGFiles(PackSegFiles):
    """PackSegFiles for PNG datasets: images and label maps are PNG files (a JPEG image raises LedB200Error)."""

    jpeg_images = False


def _is_file(x):
    if isinstance(x, torch.Tensor):
        return x.dtype == torch.uint8 and x.dim() == 1
    return isinstance(x, (bytes, bytearray, memoryview))


def _meta(s):
    return s.get('metainfo', s) if isinstance(s, dict) else {}


class DecodedFiles(list):
    """The images decode_batch decoded from a batch's files: the files' pixels by construction, so
    SegVisualizationHook draws on them without reading the files again."""


def decode_batch(data):
    """Decodes a batch of PackSegFiles outputs in place: data['inputs'] becomes the [3, h, w] uint8 BGR images (one
    png_decode call for the PNG images and one jpeg_decode call for the JPEG ones, back in batch order) and each
    sample's `gt_seg_map_file` becomes gt_sem_seg['data'], the [1, h, w] uint8 label map.  A batch of decoded images is
    returned untouched.  Returns `data`."""
    inputs = data.get('inputs', None) if isinstance(data, dict) else None
    if not isinstance(inputs, (list, tuple)) or not inputs or not all(_is_file(x) for x in inputs):
        return data
    samples = data.get('data_samples', None)
    metas = [_meta(s) for s in samples] if samples is not None else [{} for _ in inputs]
    names = [m.get('img_path', f'image {i}') for i, m in enumerate(metas)]
    jpeg = [_is_jpeg(x) for x in inputs]
    images = [None] * len(inputs)
    for is_jpeg, decode in ((False, ops.png_decode), (True, ops.jpeg_decode)):
        idx = [i for i, j in enumerate(jpeg) if j == is_jpeg]
        if idx:
            for i, img in zip(idx, decode([inputs[i] for i in idx], names=[names[i] for i in idx])):
                images[i] = img
    data['inputs'] = DecodedFiles(images)
    withlab = [i for i, s in enumerate(samples or []) if isinstance(s, dict) and 'gt_seg_map_file' in s]
    if withlab:
        rzl = {bool(metas[i].get('reduce_zero_label', False)) for i in withlab}
        lmaps = {repr(metas[i].get('label_map', None)) for i in withlab}
        if len(rzl) != 1 or len(lmaps) != 1:
            raise NotImplementedError('the label maps of one batch must share reduce_zero_label and label_map')
        labels = ops.png_decode([samples[i].pop('gt_seg_map_file') for i in withlab], 'label',
                                reduce_zero_label=rzl.pop(), label_map=metas[withlab[0]].get('label_map', None),
                                names=[metas[i].get('seg_map_path', f'label map {i}') for i in withlab])
        for i, lab in zip(withlab, labels):
            samples[i]['gt_sem_seg'] = dict(data=lab)
    return data
