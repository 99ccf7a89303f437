"""MFAF gate behind the reference's module surface (SURVEY section 8a row B7).

``Muti_AFF`` mirrors ``mmseg/models/classification/model_utils.py:356-429``: same constructor
``(channels=64, r=4)``, same sub-module / parameter names (``local_att.0.weight`` ... ``global_att.4.running_var``)
so reference checkpoints load, same ``forward(x, residual)``.  Eval-mode forward runs the three kernels of
``csrc/mfaf.cu`` through ``ledb200_mfaf_forward``; there is no CPU fallback.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import lib as L
from .ops import fold_bn
from .registry import MODELS


def _att(channels, inter, pool):
    layers = [] if pool is None else [nn.AdaptiveAvgPool2d(pool)]
    layers += [nn.Conv2d(channels, inter, kernel_size=1, stride=1, padding=0), nn.BatchNorm2d(inter),
               nn.ReLU(inplace=True), nn.Conv2d(inter, channels, kernel_size=1, stride=1, padding=0),
               nn.BatchNorm2d(channels)]
    return nn.Sequential(*layers)


def _fold_conv_bn(conv, bn):
    """y = BN(W x + bias)  ->  y = a * (W x) + b  (float64 fold, fp32 result)."""
    a = fold_bn(bn)[0]
    b = bn.bias.detach().double() + (conv.bias.detach().double() - bn.running_mean.detach().double()) * a
    return conv.weight.detach().reshape(conv.out_channels, conv.in_channels).float(), a.float(), b.float()


@MODELS.register_module()
class Muti_AFF(nn.Module):

    def __init__(self, channels=64, r=4):
        super().__init__()
        inter_channels = int(channels // r)
        if channels % 8 or not 8 <= channels <= 256 or inter_channels not in (8, 16, 32, 64):
            raise NotImplementedError('the B200 MFAF kernel needs channels % 8 == 0, channels <= 256 and '
                                      'channels // r in {8, 16, 32, 64}')
        self.channels, self.inter_channels = channels, inter_channels
        self.local_att = _att(channels, inter_channels, None)
        self.context1 = _att(channels, inter_channels, (4, 4))
        self.context2 = _att(channels, inter_channels, (8, 8))
        self.context3 = _att(channels, inter_channels, (16, 16))
        self.global_att = _att(channels, inter_channels, 1)
        self.sigmoid = nn.Sigmoid()
        self._packed = None
        self._ws = None
        self.register_load_state_dict_post_hook(lambda m, keys: m.reset_engine())

    def reset_engine(self):
        self._packed = None

    def packed_params(self, device):
        if self._packed is None or self._packed.device != device:
            parts = []
            for seq in (self.local_att, self.context1, self.context2, self.context3, self.global_att):
                mods = [m for m in seq if isinstance(m, (nn.Conv2d, nn.BatchNorm2d))]
                w1, a1, b1 = _fold_conv_bn(mods[0], mods[1])
                w2, a2, b2 = _fold_conv_bn(mods[2], mods[3])
                parts += [w1.reshape(-1), a1, b1, w2.reshape(-1), a2, b2]
            flat = torch.cat([p.cpu().reshape(-1) for p in parts])
            assert flat.numel() == L.get().ledb200_mfaf_param_floats(self.channels, self.inter_channels)
            self._packed = flat.to(device)
        return self._packed

    def _workspace(self, n, device):
        need = L.get().ledb200_mfaf_workspace_bytes(n, self.channels)
        if self._ws is None or self._ws.device != device or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=device)
        return self._ws

    def forward(self, x, residual):
        if self.training:
            raise NotImplementedError('Muti_AFF: only the eval-mode block is built (SURVEY section 8a row B7)')
        if not (x.is_cuda and residual.is_cuda):
            raise L.LedB200Error('Muti_AFF needs CUDA tensors (no CPU fallback)')
        if x.dtype not in (torch.float32, torch.bfloat16) or residual.dtype != x.dtype:
            raise L.LedB200Error(f'Muti_AFF: x and residual must both be float32 or bfloat16, got {x.dtype} / '
                                 f'{residual.dtype}')
        assert x.shape == residual.shape and x.shape[1] == self.channels, \
            f'Muti_AFF expects two [N, {self.channels}, H, W] tensors, got {tuple(x.shape)} / {tuple(residual.shape)}'
        N, Cc, H, W = x.shape
        xs = [t.permute(0, 2, 3, 1) for t in (x, residual)]
        xs = [t if t.is_contiguous() else t.contiguous() for t in xs]   # NCHW caller: one layout pass (plumbing)
        out = torch.empty((N, H, W, Cc), dtype=x.dtype, device=x.device)
        L.check(L.get().ledb200_mfaf_forward(
            C.c_void_p(xs[0].data_ptr()), C.c_void_p(xs[1].data_ptr()), C.c_void_p(out.data_ptr()),
            L.torch_dtype_code(x), N, H, W, Cc, self.inter_channels,
            C.c_void_p(self.packed_params(x.device).data_ptr()),
            C.c_void_p(self._workspace(N, x.device).data_ptr()), L.stream_ptr(x.device)), 'ledb200_mfaf_forward')
        return out.permute(0, 3, 1, 2)               # NCHW-shaped view over NHWC memory
