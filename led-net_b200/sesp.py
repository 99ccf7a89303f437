"""`SESP` (MODELS) - the reference's SESP block behind its own constructor signature and state-dict
names (``mmseg/models/nn_layers/eesp.py:15-118``), computed by ONE fused CUDA kernel (csrc/sesp.cu).

Input / output follow the reference: NCHW-shaped tensors.  channels_last (NHWC memory) tensors are
consumed and produced without any copy; contiguous NCHW ones go through one layout kernel each way.
fp32 or bf16.  Eval mode only (the block's training backward is outside SURVEY section 8a row B5).
"""
import ctypes as C

import torch
import torch.nn as nn

from . import lib as L
from .ops import fold_bn
from .registry import MODELS


def sesp_dilations(k=4, r_lim=7, spatial=True):
    """eesp.py:40-57."""
    if spatial:
        return [1] * k
    table = {3: 1, 5: 2, 7: 3, 9: 4, 11: 5, 13: 6, 15: 7, 17: 6, 19: 12, 21: 18, 23: 24}
    ks = sorted((3 + 2 * i) if (3 + 2 * i) <= r_lim else 3 for i in range(k))
    return [table[s] for s in ks]


class _CBR(nn.Module):
    def __init__(self, nin, nout, groups):
        super().__init__()
        self.conv = nn.Conv2d(nin, nout, 1, bias=False, groups=groups)
        self.bn = nn.BatchNorm2d(nout)
        self.act = nn.PReLU(nout)


class _BR(nn.Module):
    def __init__(self, nout):
        super().__init__()
        self.bn = nn.BatchNorm2d(nout)
        self.act = nn.PReLU(nout)


class _CB(nn.Module):
    def __init__(self, nin, nout, groups):
        super().__init__()
        self.conv = nn.Conv2d(nin, nout, 1, bias=False, groups=groups)
        self.bn = nn.BatchNorm2d(nout)


class _CDilated(nn.Module):
    def __init__(self, n, d):
        super().__init__()
        self.conv = nn.Conv2d(n, n, 3, 1, d, d, groups=n, bias=False)


@MODELS.register_module()
class SESP(nn.Module):

    def __init__(self, nIn, nOut, stride=1, k=4, r_lim=7, down_method='esp', Spatial=True,
                 SPASPP_Flag=False, SESPV2=True):
        super().__init__()
        assert down_method in ['avg', 'esp'], 'One of these is suppported (avg or esp)'
        n = int(nOut / k)
        n1 = nOut - (k - 1) * n
        assert n == n1, 'n(={}) and n1(={}) should be equal for Depth-wise Convolution '.format(n, n1)
        if stride != 1 or k != 4 or SPASPP_Flag:
            raise NotImplementedError('the B200 SESP kernel covers stride=1, k=4, SPASPP_Flag=False '
                                      '(the configurations on the LED-Net path)')
        if nIn % 32 or nOut % 32:
            raise NotImplementedError('the B200 SESP kernel needs nIn and nOut to be multiples of 32')
        self.nIn, self.nOut, self.stride, self.Spatial, self.SESPV2 = nIn, nOut, stride, Spatial, SESPV2
        self.dilations = sesp_dilations(k, r_lim, Spatial)
        self.proj_1x1 = _CBR(nIn, n, k)
        self.spp_dw = nn.ModuleList([_CDilated(n, d) for d in self.dilations])
        if SESPV2:
            self.spp_dw_v2 = nn.ModuleList([_CDilated(n, d + 1) for d in self.dilations])
        self.conv_1x1_exp = _CB(nOut, nOut, k)
        self.br_after_cat = _BR(nOut)
        self.module_act = nn.PReLU(nOut)
        self._packed = None
        self.register_load_state_dict_post_hook(lambda m, keys: m.reset_engine())

    def reset_engine(self):
        self._packed = None

    def packed_params(self, device):
        """BN folded to scale/shift, everything in the one fp32 block csrc/sesp.cu expects."""
        if self._packed is None or self._packed.device != device:
            n = self.nOut // 4
            ps, pb = fold_bn(self.proj_1x1.bn)
            bs, bb = fold_bn(self.br_after_cat.bn)
            es, eb = fold_bn(self.conv_1x1_exp.bn)
            dw2 = ([m.conv.weight.detach().reshape(-1) for m in self.spp_dw_v2] if self.SESPV2
                   else [torch.zeros(n * 9)] * 4)
            parts = [self.proj_1x1.conv.weight.detach().reshape(-1), ps, pb,
                     self.proj_1x1.act.weight.detach()]
            parts += [m.conv.weight.detach().reshape(-1) for m in self.spp_dw] + list(dw2)
            parts += [bs, bb, self.br_after_cat.act.weight.detach(),
                      self.conv_1x1_exp.conv.weight.detach().reshape(-1), es, eb,
                      self.module_act.weight.detach()]
            flat = torch.cat([p.float().cpu().reshape(-1) for p in parts])
            assert flat.numel() == L.get().ledb200_sesp_param_floats(self.nIn, self.nOut)
            self._packed = flat.to(device)
        return self._packed

    def forward(self, input):
        if self.training:
            raise NotImplementedError('SESP: only the eval-mode block is built (SURVEY section 8a row B5)')
        if not input.is_cuda:
            raise L.LedB200Error('SESP needs a CUDA tensor (no CPU fallback)')
        if input.dtype not in (torch.float32, torch.bfloat16):
            raise L.LedB200Error(f'SESP: dtype must be float32 or bfloat16, got {input.dtype}')
        N, Cc, H, W = input.shape
        assert Cc == self.nIn, f'SESP expects {self.nIn} input channels, got {Cc}'
        x = input.permute(0, 2, 3, 1)
        if not x.is_contiguous():
            x = x.contiguous()                       # NCHW-contiguous caller: one layout pass (plumbing)
        out = torch.empty((N, H, W, self.nOut), dtype=input.dtype, device=input.device)
        dil = (C.c_int32 * 4)(*self.dilations)
        L.check(L.get().ledb200_sesp_forward(
            C.c_void_p(x.data_ptr()), C.c_void_p(out.data_ptr()), L.torch_dtype_code(x), N, H, W, self.nIn,
            self.nOut, dil, int(self.SESPV2), C.c_void_p(self.packed_params(input.device).data_ptr()),
            L.stream_ptr(input.device)), 'ledb200_sesp_forward')
        return out.permute(0, 3, 1, 2)               # NCHW-shaped view over NHWC memory
