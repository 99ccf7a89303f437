"""numpy + cv2 restatement of mmseg 1.2.2's SegLocalVisualizer drawing and mmengine's LocalVisBackend file, the reference
the device path (ops.seg_label_locations, ops.seg_overlay, lednet_b200.visualization) is tested against.

Restated from the released mmseg 1.2.2 source (mmseg/visualization/local_visualizer.py: _get_center_loc, _draw_sem_seg,
add_datasample) and mmengine 0.x (LocalVisBackend.add_image); neither is installed here.  If a real install is ever
available, check this file against it.
"""
import cv2
import numpy as np

CITYSCAPES_CLASSES = ('road', 'sidewalk', 'building', 'wall', 'fence', 'pole', 'traffic light', 'traffic sign',
                      'vegetation', 'terrain', 'sky', 'person', 'rider', 'car', 'truck', 'bus', 'train', 'motorcycle',
                      'bicycle')
CITYSCAPES_PALETTE = [[128, 64, 128], [244, 35, 232], [70, 70, 70], [102, 102, 156], [190, 153, 153], [153, 153, 153],
                      [250, 170, 30], [220, 220, 0], [107, 142, 35], [152, 251, 152], [70, 130, 180], [220, 20, 60],
                      [255, 0, 0], [0, 0, 142], [0, 0, 70], [0, 60, 100], [0, 80, 100], [0, 0, 230], [119, 11, 32]]


def get_center_loc(mask):
    """_get_center_loc: (x, y) of the pixel at index count // 2 (x order) of the first row with the most mask pixels"""
    loc = np.argwhere(mask == 1)
    loc_sort = np.array(sorted(loc.tolist(), key=lambda row: (row[0], row[1])))
    y_list = loc_sort[:, 0]
    unique, indices, counts = np.unique(y_list, return_index=True, return_counts=True)
    y_loc = unique[counts.argmax()]
    y_most_freq_loc = loc[loc_sort[:, 0] == y_loc]
    center_num = len(y_most_freq_loc) // 2
    x = y_most_freq_loc[center_num][1]
    y = y_most_freq_loc[center_num][0]
    return np.array([x, y])


def text_style(h, w):
    """(fontScale, thickness) of _draw_sem_seg's labels for an h x w image"""
    scale = 0.05
    font_scale = min(h, w) / (25 / scale)
    thickness = 1 if h < 300 or w < 300 else 2
    return font_scale, thickness


def draw_label(mask, loc, text, color, font_scale, thickness):
    """one label of _draw_sem_seg: a filled box in the class colour, its black outline, the white class name"""
    font = cv2.FONT_HERSHEY_SIMPLEX
    (lw, lh), baseline = cv2.getTextSize(text, font, font_scale, thickness)
    x, y = int(loc[0]), int(loc[1])
    color = tuple(int(c) for c in color)
    mask = cv2.rectangle(mask, (x, y), (x + lw + baseline, y + lh + baseline), color, -1)
    mask = cv2.rectangle(mask, (x, y), (x + lw + baseline, y + lh + baseline), (0, 0, 0), thickness)
    mask = cv2.putText(mask, text, (x, y + lh), font, font_scale, (255, 255, 255), thickness, 2)
    return mask


def draw_sem_seg(image, sem_seg, classes, palette, with_labels=True, alpha=0.8):
    """_draw_sem_seg: image HWC RGB uint8, sem_seg [1,H,W] (or [H,W]) -> the blended HWC RGB uint8 picture"""
    sem_seg = np.asarray(sem_seg).reshape((1,) + image.shape[:2])
    num_classes = len(classes)
    ids = np.unique(sem_seg)[::-1]
    ids = ids[ids < num_classes]
    labels = np.array(ids, dtype=np.int64)
    colors = [palette[label] for label in labels]
    mask = np.zeros_like(image, dtype=np.uint8)
    for label, color in zip(labels, colors):
        mask[sem_seg[0] == label, :] = color
    if with_labels:
        font_scale, thickness = text_style(image.shape[0], image.shape[1])
        masks = (sem_seg[0] == labels[:, None, None]).astype(np.uint8)
        for k in range(len(labels)):
            loc = get_center_loc(masks[k])
            mask = draw_label(mask, loc, classes[labels[k]], colors[k], font_scale, thickness)
    return (image * (1 - alpha) + mask * alpha).astype(np.uint8)


def add_datasample(image, gt=None, pred=None, classes=CITYSCAPES_CLASSES, palette=CITYSCAPES_PALETTE,
                   with_labels=True, alpha=0.8):
    """add_datasample's drawn picture (HWC RGB): the gt panel, the pred panel, or both side by side"""
    panels = [draw_sem_seg(image, m, classes, palette, with_labels, alpha) for m in (gt, pred) if m is not None]
    return np.concatenate(panels, axis=1) if len(panels) == 2 else panels[0]


def local_file(drawn):
    """the PNG LocalVisBackend.add_image writes (cv2.imwrite of the RGB picture turned BGR)"""
    return cv2.imencode('.png', cv2.cvtColor(drawn, cv2.COLOR_RGB2BGR))[1].tobytes()


def blocky_map(h, w, k, seed, cell=16, ignore=0.05):
    """a seeded label map of k classes in cell x cell blocks, with some 255 (ignore) pixels"""
    rng = np.random.default_rng(seed)
    small = rng.integers(0, k, (-(-h // cell), -(-w // cell)))
    m = np.kron(small, np.ones((cell, cell), np.int64))[:h, :w]
    m[rng.random((h, w)) < ignore] = 255
    return m.astype(np.uint8)


def photo(h, w, seed):
    """a seeded smooth-plus-noise HWC RGB uint8 image"""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    base = np.stack([(x * 255 // max(w - 1, 1)), (y * 255 // max(h - 1, 1)), ((x + y) * 127 // max(h + w - 2, 1))], -1)
    return np.clip(base + rng.integers(-20, 21, (h, w, 3)), 0, 255).astype(np.uint8)
