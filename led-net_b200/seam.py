"""SEAM edge gate as a registered module (SURVEY section 8(f) rank 1).

Upstream has no class for it: the gate is inline code in the authors' speed prototype
(``tools/speed/ddrnet_speed.py``: parameters ``:88-113``, edge map ``:282-338``, gate ``:388-389``).  ``SEAM`` keeps that
code's parameter names (``conv_1.conv.weight``, ``conv_1.bn.*``, ``conv_2.conv.weight``, ``conv_2.bn.*``,
``fusion_kernel``) so the prototype's checkpoints load, and exposes it as ``forward(x, x_s) -> conv_2(mask(x)) * x_s + x_s``.
Eval-mode forward runs the three kernels of ``csrc/seam.cu``; there is no CPU fallback.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import lib as L
from .ops import fold_bn
from .registry import MODELS


class _ConvBN(nn.Module):
    """mmcv ConvModule(k=3, padding=1, norm_cfg=BN, act_cfg=None): conv (no bias) + BatchNorm."""

    def __init__(self, cin, cout):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, 3, padding=1, bias=False)
        self.bn = nn.BatchNorm2d(cout)


@MODELS.register_module()
class SEAM(nn.Module):

    def __init__(self, channels=64, boundary_threshold=0.1):
        super().__init__()
        if channels % 8:
            raise NotImplementedError('the B200 SEAM kernel needs channels % 8 == 0')
        self.channels, self.boundary_threshold = channels, boundary_threshold
        self.conv_1 = _ConvBN(channels, 1)
        self.conv_2 = _ConvBN(1, channels)
        self.fusion_kernel = nn.Parameter(torch.tensor([[6. / 10], [3. / 10], [1. / 10]],
                                                       dtype=torch.float32).reshape(1, 3, 1, 1), requires_grad=False)
        self._packed = None
        self._ws = None
        self.register_load_state_dict_post_hook(lambda m, keys: m.reset_engine())

    def reset_engine(self):
        self._packed = None

    def packed_params(self, device):
        if self._packed is None or self._packed.device != device:
            if not torch.allclose(self.fusion_kernel.detach().reshape(-1).cpu(), torch.tensor([0.6, 0.3, 0.1])):
                raise NotImplementedError('the B200 SEAM kernel hard-codes fusion_kernel = (0.6, 0.3, 0.1)')
            a1, b1 = fold_bn(self.conv_1.bn)
            a2, b2 = fold_bn(self.conv_2.bn)
            w1 = self.conv_1.conv.weight.detach().reshape(self.channels, 9).t().contiguous()      # [tap][C]
            w2 = self.conv_2.conv.weight.detach().reshape(self.channels, 9).t().contiguous()      # [tap][C]
            flat = torch.cat([t.float().cpu().reshape(-1) for t in (w1, a1, b1, torch.zeros(6), w2, a2, b2)])
            assert flat.numel() == L.get().ledb200_seam_param_floats(self.channels)
            self._packed = flat.to(device)
        return self._packed

    def forward(self, x, x_s):
        if self.training:
            raise NotImplementedError('SEAM: only the eval-mode block is built (SURVEY section 8f)')
        if not (x.is_cuda and x_s.is_cuda):
            raise L.LedB200Error('SEAM needs CUDA tensors (no CPU fallback)')
        if x.dtype not in (torch.float32, torch.bfloat16) or x_s.dtype != x.dtype:
            raise L.LedB200Error(f'SEAM: x and x_s must both be float32 or bfloat16, got {x.dtype} / {x_s.dtype}')
        assert x.shape == x_s.shape and x.shape[1] == self.channels, \
            f'SEAM expects two [N, {self.channels}, H, W] tensors, got {tuple(x.shape)} / {tuple(x_s.shape)}'
        N, Cc, H, W = x.shape
        ts = [t.permute(0, 2, 3, 1) for t in (x, x_s)]
        ts = [t if t.is_contiguous() else t.contiguous() for t in ts]
        out = torch.empty((N, H, W, Cc), dtype=x.dtype, device=x.device)
        need = L.get().ledb200_seam_workspace_bytes(N, H, W)
        if self._ws is None or self._ws.device != x.device or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=x.device)
        L.check(L.get().ledb200_seam_forward(
            C.c_void_p(ts[0].data_ptr()), C.c_void_p(ts[1].data_ptr()), C.c_void_p(out.data_ptr()), L.torch_dtype_code(x),
            N, H, W, Cc, float(self.boundary_threshold), C.c_void_p(self.packed_params(x.device).data_ptr()),
            C.c_void_p(self._ws.data_ptr()), L.stream_ptr(x.device)), 'ledb200_seam_forward')
        return out.permute(0, 3, 1, 2)
