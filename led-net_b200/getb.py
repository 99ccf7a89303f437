"""GETB block behind the reference's module surface (SURVEY section 8a row B6).

``GETBBlock`` mirrors ``mmseg/models/backbones/UNetFormer_GETB.py:209-226`` (with ``GlobalLocalAttention``
:97-206 and ``Mlp`` :79-94): same constructor, same sub-module / parameter / buffer names
(``norm1``, ``attn.qkv.0.weight``, ``attn.relative_position_bias_table``, ``attn.relative_position_index``,
``attn.proj.{0,1,2}``, ``mlp.fc1``, ``mlp.fc2``, ``norm2``) so reference checkpoints load.  Eval-mode forward runs
``csrc/getb.cu`` through a ``ledb200_getb`` handle (the four 1x1 convolutions on the tcgen05 conv kernel in bf16
mode); there is no CPU fallback.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import lib as L
from .ops import fold_bn
from .registry import MODELS


def _relative_position_index(ws):
    """UNetFormer_GETB.py:131-141."""
    coords = torch.stack(torch.meshgrid([torch.arange(ws), torch.arange(ws)], indexing='ij'))
    flat = torch.flatten(coords, 1)
    rel = (flat[:, :, None] - flat[:, None, :]).permute(1, 2, 0).contiguous()
    rel[:, :, 0] += ws - 1
    rel[:, :, 1] += ws - 1
    rel[:, :, 0] *= 2 * ws - 1
    return rel.sum(-1)


class GlobalLocalAttention(nn.Module):
    """Parameter container with the reference's names; the arithmetic lives in csrc/getb.cu."""

    def __init__(self, dim=256, num_heads=16, qkv_bias=False, window_size=8, relative_pos_embedding=True):
        super().__init__()
        if not relative_pos_embedding:
            raise NotImplementedError('the B200 GETB kernel always adds the relative position bias')
        self.num_heads, self.ws = num_heads, window_size
        self.scale = (dim // num_heads) ** -0.5
        ws = window_size
        self.qkv = nn.Sequential(nn.Conv2d(dim, 3 * dim, kernel_size=1, bias=qkv_bias))
        self.proj = nn.Sequential(
            nn.Conv2d(dim, dim, ws, stride=1, dilation=1, padding=(ws - 1) // 2, groups=dim, bias=False),
            nn.BatchNorm2d(dim), nn.Conv2d(dim, dim, kernel_size=1, bias=False))
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * ws - 1) * (2 * ws - 1), num_heads))
        self.register_buffer('relative_position_index', _relative_position_index(ws))
        nn.init.trunc_normal_(self.relative_position_bias_table, std=.02)


class Mlp(nn.Module):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.ReLU6, drop=0.):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Conv2d(in_features, hidden_features, 1, 1, 0, bias=True)
        self.act = act_layer()
        self.fc2 = nn.Conv2d(hidden_features, out_features, 1, 1, 0, bias=True)
        self.drop = nn.Dropout(drop, inplace=True)


@MODELS.register_module()
class GETBBlock(nn.Module):

    def __init__(self, dim=256, num_heads=16, mlp_ratio=4., qkv_bias=False, drop=0., attn_drop=0.,
                 drop_path=0., act_layer=nn.ReLU6, norm_layer=nn.BatchNorm2d, window_size=8):
        super().__init__()
        if window_size != 8:
            raise NotImplementedError('the B200 GETB kernel is built for window_size = 8 (64 tokens per window)')
        if act_layer is not nn.ReLU6 or norm_layer is not nn.BatchNorm2d:
            raise NotImplementedError('the B200 GETB kernel covers act_layer=ReLU6, norm_layer=BatchNorm2d')
        if dim % 8 or dim % num_heads or dim // num_heads not in (4, 8, 16, 32):
            raise NotImplementedError('the B200 GETB kernel needs dim % 8 == 0 and dim / num_heads in {4, 8, 16, 32}')
        self.dim, self.num_heads, self.window_size = dim, num_heads, window_size
        self.hidden = int(dim * mlp_ratio)
        if self.hidden % 8:
            raise NotImplementedError('the B200 GETB kernel needs int(dim * mlp_ratio) % 8 == 0')
        self.norm1 = norm_layer(dim)
        self.attn = GlobalLocalAttention(dim, num_heads=num_heads, qkv_bias=qkv_bias, window_size=window_size)
        self.drop_path = nn.Identity()          # eval: DropPath is the identity
        self.mlp = Mlp(in_features=dim, hidden_features=self.hidden, out_features=dim, act_layer=act_layer, drop=drop)
        self.norm2 = norm_layer(dim)
        self._handles = {}
        self.register_load_state_dict_post_hook(lambda m, keys: m.reset_engine())

    def reset_engine(self):
        for h in self._handles.values():
            L.get().ledb200_getb_destroy(h)
        self._handles = {}

    def __del__(self):
        try:
            self.reset_engine()
        except Exception:
            pass

    def packed_params(self):
        """host fp32 block in the order include/ledb200.h documents; BN1 folded into qkv, BN2 into fc1."""
        Cc, a = self.dim, self.attn
        s1, t1 = fold_bn(self.norm1)
        s2, t2 = fold_bn(self.norm2)
        sp, tp = fold_bn(a.proj[1])
        wq = a.qkv[0].weight.detach().double().reshape(3 * Cc, Cc)
        bq = wq @ t1 + (a.qkv[0].bias.detach().double() if a.qkv[0].bias is not None else 0.)
        relb = a.relative_position_bias_table.detach()[a.relative_position_index.view(-1)]
        relb = relb.view(64, 64, self.num_heads).permute(2, 0, 1).contiguous()
        w1 = self.mlp.fc1.weight.detach().double().reshape(self.hidden, Cc)
        b1 = w1 @ t2 + self.mlp.fc1.bias.detach().double()
        parts = [wq * s1[None, :], bq, s1, t1, relb, a.proj[0].weight.detach().reshape(Cc, 64), sp, tp,
                 a.proj[2].weight.detach().reshape(Cc, Cc), w1 * s2[None, :], b1,
                 self.mlp.fc2.weight.detach().reshape(Cc, self.hidden), self.mlp.fc2.bias.detach()]
        flat = torch.cat([p.float().cpu().reshape(-1) for p in parts]).contiguous()
        assert flat.numel() == L.get().ledb200_getb_param_floats(Cc, self.num_heads, self.hidden)
        return flat

    def _handle(self, x):
        key = (x.dtype, x.device.index)
        if key not in self._handles:
            flat = self.packed_params()
            h = C.c_void_p()
            with torch.cuda.device(x.device):
                L.check(L.get().ledb200_getb_create(self.dim, self.num_heads, self.hidden, self.window_size,
                                                    L.torch_dtype_code(x), C.c_void_p(flat.data_ptr()),
                                                    C.byref(h)), 'ledb200_getb_create')
            self._handles[key] = h
        return self._handles[key]

    def forward(self, x):
        if self.training:
            raise NotImplementedError('GETBBlock: only the eval-mode block is built (SURVEY section 8a row B6)')
        if not x.is_cuda:
            raise L.LedB200Error('GETBBlock needs a CUDA tensor (no CPU fallback)')
        if x.dtype not in (torch.float32, torch.bfloat16):
            raise L.LedB200Error(f'GETBBlock: dtype must be float32 or bfloat16, got {x.dtype}')
        N, Cc, H, W = x.shape
        assert Cc == self.dim, f'GETBBlock expects {self.dim} channels, got {Cc}'
        xn = x.permute(0, 2, 3, 1)
        if not xn.is_contiguous():
            xn = xn.contiguous()                     # NCHW-contiguous caller: one layout pass (plumbing)
        out = torch.empty((N, H, W, Cc), dtype=x.dtype, device=x.device)
        with torch.cuda.device(x.device):
            L.check(L.get().ledb200_getb_forward(self._handle(x), C.c_void_p(xn.data_ptr()), C.c_void_p(out.data_ptr()),
                                                 N, H, W, L.stream_ptr(x.device)), 'ledb200_getb_forward')
        return out.permute(0, 3, 1, 2)               # NCHW-shaped view over NHWC memory
