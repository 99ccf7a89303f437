"""The registry surface the drop-in sits behind.

The reference selects modules by ``type=`` strings resolved in ``mmseg.registry.MODELS``
(``mmseg/registry/registry.py:56``) and ``METRICS`` (``:90``); the LED-Net config
(``configs/LED_Net/LEDNet_80k_cityscapes-1024x1024.py:21-56``) names ``EncoderDecoder``,
``SegDataPreProcessor``, ``LEDNet``, ``LEDHead`` and ``OhemCrossEntropy``, and the dataset base
config names ``IoUMetric``.  This file offers the same two registries with the same
``register_module()`` / ``build(cfg)`` calls.  When a real mmseg/mmengine install is importable,
``register_into_mmseg()`` additionally registers the B200 classes under the reference names in
mmseg's own registries (``force=True``), which is all a reference checkout needs to pick them up.
"""
import inspect


class Registry:

    def __init__(self, name):
        self.name = name
        self._table = {}

    def register_module(self, name=None, force=False, module=None):
        def deco(cls):
            key = name or cls.__name__
            if key in self._table and not force:
                raise KeyError(f'{key} is already registered in {self.name}')
            self._table[key] = cls
            return cls
        return deco(module) if module is not None else deco

    def get(self, key):
        return self._table.get(key)

    def build(self, cfg, **default_args):
        if not isinstance(cfg, dict) or 'type' not in cfg:
            raise TypeError(f'cfg must be a dict with a "type" key, got {cfg!r}')
        args = dict(cfg)
        typ = args.pop('type')
        cls = typ if inspect.isclass(typ) else self._table.get(typ)
        if cls is None:
            raise KeyError(f'{typ} is not in the {self.name} registry')
        for k, v in default_args.items():
            args.setdefault(k, v)
        return cls(**args)

    def __contains__(self, key):
        return key in self._table


MODELS = Registry('model')
METRICS = Registry('metric')
TRANSFORMS = Registry('transform')      # dataset pipeline steps (mmseg/registry/registry.py TRANSFORMS)
VISUALIZERS = Registry('visualizer')    # SegLocalVisualizer (mmseg/registry/registry.py VISUALIZERS)
HOOKS = Registry('hook')                # SegVisualizationHook (mmseg/registry/registry.py HOOKS)


def register_into_mmseg():
    """Register the B200 modules in a real mmseg install (returns False if mmseg is absent)."""
    try:
        from mmseg.registry import MODELS as MM, METRICS as MT, TRANSFORMS as TR, VISUALIZERS as VI, HOOKS as HK
    except Exception:
        return False
    for k, v in MODELS._table.items():
        MM.register_module(name=k, force=True, module=v)
    for k, v in METRICS._table.items():
        MT.register_module(name=k, force=True, module=v)
    for k, v in TRANSFORMS._table.items():
        TR.register_module(name=k, force=True, module=v)
    for k, v in VISUALIZERS._table.items():
        VI.register_module(name=k, force=True, module=v)
    try:                                # mmengine's runner calls every Hook method: give the hooks its base class
        from mmengine.hooks import Hook
    except Exception:
        Hook = None
    for k, v in HOOKS._table.items():
        HK.register_module(name=k, force=True, module=type(k, (v, Hook), {}) if Hook is not None else v)
    return True
