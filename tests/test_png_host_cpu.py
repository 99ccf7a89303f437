"""Host side of the PNG output (no GPU): IoUMetric's format_only construction, ledb200_png_bound against the stored
encoding, and no CPU fallback in ops.png_encode."""
import os

import pytest
import torch

import lednet_b200 as L
from lednet_b200 import lib, ops


def test_format_only_metric_constructs(tmp_path):
    d = str(tmp_path / 'preds' / 'test')
    m = L.IoUMetric(output_dir=d, format_only=True, keep_results=True)
    assert os.path.isdir(d)
    assert m.compute_metrics([]) == {}
    assert m.evaluate(0) == {}


def _stored_png_size(h, w):
    """Signature + IHDR + IEND + one IDAT of a zlib stream whose deflate data is stored blocks of <= 65535 bytes, each
    band of rows ending its own blocks (one band per <= 65535 bytes of rows where a row allows it)."""
    s = w + 1
    rows = max(1, min(h, 65535 // s))
    data = 0
    for r0 in range(0, h, rows):
        n = min(rows, h - r0) * s
        data += n + 5 * -(-n // 65535)
    return 8 + 25 + 12 + (12 + 2 + data + 4)


@pytest.mark.parametrize('h,w', [(1, 1), (1, 2048), (2048, 1), (7, 13), (512, 910), (1024, 2048), (4, 40000),
                                 (3, 70000), (33, 65534)])
def test_bound_covers_the_stored_encoding(h, w):
    b = lib.get().ledb200_png_bound(h, w)
    assert b >= _stored_png_size(h, w)


def test_bound_and_workspace_reject_bad_sizes():
    l = lib.get()
    assert l.ledb200_png_bound(0, 4) == -1 and l.ledb200_png_bound(4, 0) == -1
    assert l.ledb200_png_bound(46341, 46341) == -1          # larger than one IDAT chunk can hold
    assert l.ledb200_png_workspace_bytes(0, 4, 4) == -1
    assert l.ledb200_png_workspace_bytes(2, 4, 4) > 2 * 4 * 5


def test_png_encode_needs_cuda():
    with pytest.raises(lib.LedB200Error):
        ops.png_encode(torch.zeros(4, 4, dtype=torch.uint8))
