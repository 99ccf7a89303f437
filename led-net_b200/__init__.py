"""led-net_b200: the LED-Net data-parallel hot path as hand-written sm_100a CUDA kernels behind
the reference's mmseg registry surface (MODELS: LEDNet, LEDHead, OhemCrossEntropy, EncoderDecoder,
SegDataPreProcessor, DeviceAugSegDataPreProcessor, SegTTAModel; METRICS: IoUMetric, CityscapesMetric; TRANSFORMS: PackSegFiles, PackSegPNGFiles; VISUALIZERS: SegLocalVisualizer; HOOKS: SegVisualizationHook).  Host code is Python/PyTorch plumbing over the C ABI in
include/ledb200.h; there is no CPU fallback."""
__version__ = '0.1.0'

from .registry import MODELS, METRICS, TRANSFORMS, VISUALIZERS, HOOKS, Registry, register_into_mmseg  # noqa: F401
from .lib import LedB200Error  # noqa: F401
from .losses import OhemCrossEntropy, accuracy  # noqa: F401
from .modules import LEDNet, LEDHead  # noqa: F401
from .metrics import IoUMetric  # noqa: F401
from .cityscapes import CityscapesMetric  # noqa: F401
from .segmentor import EncoderDecoder, SegDataPreProcessor  # noqa: F401
from .tta import SegTTAModel  # noqa: F401
from .augment import DeviceAugSegDataPreProcessor  # noqa: F401
from .png_feed import PackSegFiles, PackSegPNGFiles, decode_batch  # noqa: F401
from .visualization import SegLocalVisualizer, SegVisualizationHook  # noqa: F401
from .engine import Engine  # noqa: F401
from .sesp import SESP  # noqa: F401
from .mfaf import Muti_AFF  # noqa: F401
from .getb import GETBBlock  # noqa: F401
from .seam import SEAM  # noqa: F401
from .optim import FlatSGD, PolyLR  # noqa: F401
from . import ops, synth, train_ops  # noqa: F401
