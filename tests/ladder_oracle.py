"""Plain float64 references for the head's logit ladder (TEST INFRASTRUCTURE).

The bf16 engine runs LEDHead's last stages as

    c5h, x1h, x2h = bf16(relu(scale * feature + shift))          pre-activation BatchNorm of each base head
    head.feat     = bf16(relu(conv3x3(c5h) + shift))             head (BatchNorm .1 folded into the conv)
    xc            = fp16_satfinite(conv1x1(head.feat) + bias)    conv_seg (conv_tc.cu, out_f16)
    r2            = rung(x2h, head_x2, up = xc)                  ladder_tc.cu, ladder_kernel<false>
    r1            = rung(x1h, head_x1, up = r2)
    logits        = up2(r1), labels = argmax_k                   tail.cu tail2_kernel, or ladder_kernel<true>

    rung(in, conv, up) = fp16_satfinite(f32(f32(relu(conv3x3(in) + b)) + up_fp16(up)))

Everything here works on float64 tensors on any device and models the engine's storage roundings exactly; the one
thing it cannot model is the fp32 accumulation order of the tensor-core sums.  `exact_fold_state` builds head
parameters for which BatchNorm folding introduces no rounding at all, so the folded weights are known exactly.
"""
import numpy as np
import torch
import torch.nn.functional as F

import oracle

F16_MAX = 65504.0


# ---------------------------------------------------------------------------------------------- roundings
def pow2(e):
    """2**e as float64, exactly, for integer tensors e in the normal range (built from the exponent bits)."""
    return ((e.long() + 1023) << 52).view(torch.float64)


def round_to(x, mant, emin):
    """Round float64 `x` to the nearest number with `mant` significant bits and smallest normal exponent `emin`
    (ties to even; no overflow handling).  One rounding, unlike float64 -> float32 -> half casts."""
    _, e = torch.frexp(x)                                    # |x| in [2^(e-1), 2^e)
    ulp_exp = torch.clamp(e - 1, min=emin) - (mant - 1)
    return torch.round(x * pow2(-ulp_exp)) * pow2(ulp_exp)


def rnd16(x):
    """IEEE fp16 round-to-nearest with overflow to +-inf (__hmul2 / __hfma2)."""
    r = round_to(x, 11, -14)
    return torch.where(r.abs() > F16_MAX, torch.copysign(torch.full_like(r, float('inf')), r), r)


def sat16(x):
    """cvt.rn.satfinite.f16: round to nearest, then clamp to +-65504 (never inf)."""
    return round_to(x, 11, -14).clamp(-F16_MAX, F16_MAX)


def rnd_bf16(x):
    return round_to(x, 8, -126)


def fl32(x):
    return x.float().double()


def ulp(x, mant, emin):
    """Spacing of the storage format at |x|."""
    _, e = torch.frexp(x.abs())
    return pow2(torch.clamp(e - 1, min=emin) - (mant - 1))


FMT = {'bf16': (8, -126), 'f16': (11, -14)}


# ---------------------------------------------------------------------------------------------- x2 upsamples
def _taps(n_out, n_in, device):
    """Exact x2 bilinear upsample, align_corners=False, as ladder_tc.cu / tail.cu index it: output i reads source
    rows lo = clamp((i-1)>>1), hi = clamp(((i-1)>>1) + 1) with weights (3/4, 1/4) for odd i and (1/4, 3/4) for even i."""
    i = torch.arange(n_out, device=device)
    lo = (i - 1) >> 1
    a, b = lo.clamp(0, n_in - 1), (lo + 1).clamp(0, n_in - 1)
    w0 = torch.where(i % 2 == 1, 0.75, 0.25).double()
    return a, b, w0, 1.0 - w0


def up_fp16(u, rounding=True):
    """The `up` gather of ladder_tc.cu:280-321 on fp16 values (float64 tensor [N,K,h,w] -> [N,K,2h,2w]):
    h0 = rnd16(b*wx1 + rnd16(a*wx0)), h1 likewise on the bottom pair, out = rnd16(h1*wy1 + rnd16(h0*wy0)).
    Products by 1/4 and 3/4 of fp16 values are exact in float64, so each rnd16 is the single rounding of __hmul2 or
    __hfma2.  rounding=False gives the exact bilinear upsample."""
    R = rnd16 if rounding else (lambda t: t)
    h, w = u.shape[-2:]
    ya, yb, wy0, wy1 = _taps(2 * h, h, u.device)
    xa, xb, wx0, wx1 = _taps(2 * w, w, u.device)
    top, bot = u[..., ya, :], u[..., yb, :]
    h0 = R(top[..., xb] * wx1 + R(top[..., xa] * wx0))
    h1 = R(bot[..., xb] * wx1 + R(bot[..., xa] * wx0))
    return R(h1 * wy1[:, None] + R(h0 * wy0[:, None]))


def up_f32(r):
    """tail2_kernel's last x2 upsample (tail.cu:287-356, and the ladder's final rung): every lerp is
    fmaf(hi, w_hi, lo * w_lo) in fp32, horizontal first, then vertical.  Bit-exact on fp16 / fp32 inputs."""
    def lerp(lo, hi, wlo, whi):
        return fl32(hi * whi + fl32(lo * wlo))
    h, w = r.shape[-2:]
    ya, yb, wy0, wy1 = _taps(2 * h, h, r.device)
    xa, xb, wx0, wx1 = _taps(2 * w, w, r.device)
    rows = lerp(r[..., xa], r[..., xb], wx0, wx1)
    return lerp(rows[..., ya, :], rows[..., yb, :], wy0[:, None], wy1[:, None])


def corner_max(r):
    """max |corner| of every output of an x2 upsample of r: the scale of its fp32 lerp roundings."""
    h, w = r.shape[-2:]
    ya, yb, _, _ = _taps(2 * h, h, r.device)
    xa, xb, _, _ = _taps(2 * w, w, r.device)
    a = r.abs()
    rows = torch.maximum(a[..., xa], a[..., xb])
    return torch.maximum(rows[..., ya, :], rows[..., yb, :])


# ---------------------------------------------------------------------------------------------- parameters
BN_PREFIXES = ('head.0.bn', 'head.1', 'aux_head.0.bn', 'aux_head.1', 'head_x1.0.bn', 'head_x1.1',
               'head_x2.0.bn', 'head_x2.1')


def exact_fold_state(C, HC, K, seed=0):
    """decode_head.* state dict of oracle.OracleLEDHead(4C, HC, K, tap_channels=C) whose BatchNorm folding is exact:
    running_var = 4**j - 1e-5 (sqrt(var + 1e-5f) == 2**j in float32 for j = 0, 1, 2), gamma a power of two,
    running_mean = 0, and every weight and bias bf16-representable."""
    head = oracle.OracleLEDHead(4 * C, HC, K, tap_channels=C)
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, t in head.state_dict().items():
        leaf = name.rsplit('.', 1)[-1]
        if leaf == 'num_batches_tracked':
            v = t.clone()
        elif leaf == 'running_var':
            j = torch.randint(0, 3, t.shape, generator=g).double()
            v = (4.0 ** j - 1e-5).float()
        elif leaf == 'running_mean':
            v = torch.zeros_like(t)
        elif leaf == 'weight' and t.dim() == 1:
            v = 2.0 ** torch.randint(-1, 2, t.shape, generator=g).float()
        elif leaf == 'weight':
            fan_in = t[0].numel()
            v = (torch.randn(t.shape, generator=g) * (2.0 / fan_in) ** 0.5).bfloat16().float()
        else:                                                     # BatchNorm beta, conv_seg / aux_cls_seg bias
            v = (torch.randn(t.shape, generator=g) * 0.1).bfloat16().float()
        out['decode_head.' + name] = v
    return out


def folded_bn(state, prefix):
    """(scale, shift) of a BatchNorm as the engine folds it (engine.cu bn_affine: float32 arithmetic)."""
    p = 'decode_head.' + prefix
    w, b = state[p + '.weight'].numpy(), state[p + '.bias'].numpy()
    m, v = state[p + '.running_mean'].numpy(), state[p + '.running_var'].numpy()
    s = (w / np.sqrt(v + np.float32(1e-5))).astype(np.float32)
    shift = (b - m * s).astype(np.float32)
    return torch.from_numpy(s).double(), torch.from_numpy(shift).double()


def assert_exact_fold(state):
    """Every BatchNorm scale is an exact power of two, every shift is the beta itself, and every weight folded by it
    is still bf16-representable: the engine's folded parameters equal the reference's with no rounding."""
    for pre in BN_PREFIXES:
        s, shift = folded_bn(state, pre)
        mant, _ = np.frexp(s.numpy())
        assert np.all(mant == 0.5), (pre, s)
        beta = state['decode_head.' + pre + '.bias'].double()
        assert torch.equal(shift, beta), pre
        assert torch.equal(rnd_bf16(beta), beta), pre
        if pre.endswith('.1'):
            w = state['decode_head.' + pre[:-2] + '.0.conv.weight'].double() * s[:, None, None, None]
            assert torch.equal(rnd_bf16(w), w), pre


class HeadParams:
    """The head's parameters as the engine uses them (folded, float64) on `device`.  acc=torch.float32 sums the
    convolutions in fp32 instead of exactly: a stand-in for the tensor cores' accumulation-order differences."""

    def __init__(self, state, device, acc=torch.float64):
        self.acc = acc
        def d(t):
            return t.double().to(device)
        self.pre = {n: tuple(d(t) for t in folded_bn(state, n + '.0.bn')) for n in ('head', 'head_x1', 'head_x2')}
        self.conv = {}
        for n in ('head', 'head_x1', 'head_x2'):
            s, shift = folded_bn(state, n + '.1')
            self.conv[n] = (d(state['decode_head.' + n + '.0.conv.weight'].double() * s[:, None, None, None]), d(shift))
        self.conv['conv_seg'] = (d(state['decode_head.conv_seg.weight']), d(state['decode_head.conv_seg.bias']))


# ---------------------------------------------------------------------------------------------- stage references
def pre_act(p, name, feat):
    """c5h / x1h / x2h: bf16(relu(fp32(scale * x + shift)))."""
    s, b = p.pre[name]
    return rnd_bf16(fl32(feat * s[:, None, None] + b[:, None, None]).clamp_min(0))


def conv(p, name, x, absolute=False):
    """Exact conv sum + bias in float64; absolute=True gives sum |w x| + |b| (the accumulation-error scale)."""
    w, b = p.conv[name]
    if absolute:
        w, b, x = w.abs(), b.abs(), x.abs()
    elif p.acc != torch.float64:
        w, b, x = w.to(p.acc), b.to(p.acc), x.to(p.acc)
    return F.conv2d(x, w, b, padding=w.shape[-1] // 2).double()


def head_feat(p, c5h):
    return rnd_bf16(fl32(conv(p, 'head', c5h)).clamp_min(0))


def x_c(p, feat):
    return sat16(fl32(conv(p, 'conv_seg', feat)))


def rung(p, name, inp, up):
    """r = fp16_satfinite(f32(f32(relu(conv3x3(in) + b)) + up_fp16(up)))."""
    t = fl32(conv(p, name, inp)).clamp_min(0)
    return sat16(fl32(t + up_fp16(up)))


def chain(p, c5, x1, x2):
    """Every stored stage of the ladder from the raw features, in storage precision."""
    out = {'c5h': pre_act(p, 'head', c5), 'x1h': pre_act(p, 'head_x1', x1), 'x2h': pre_act(p, 'head_x2', x2)}
    out['head.feat'] = head_feat(p, out['c5h'])
    out['xc'] = x_c(p, out['head.feat'])
    out['hx2'] = rung(p, 'head_x2', out['x2h'], out['xc'])
    out['hx1'] = rung(p, 'head_x1', out['x1h'], out['hx2'])
    return out


def ladder_logits(p, c5, x1, x2):
    """The ladder path's logits from the raw features: tail2's fp32 upsample of the stored r1."""
    return up_f32(chain(p, c5, x1, x2)['hx1'])


def fallback_logits(p, c5, x1, x2):
    """Heads with K <= 16 (tail_kernel): x_c, head_x1 and head_x2 stored in bf16, the three-level upsample in fp32
    (modelled in float64: its fp32 roundings are far below the bf16 ones)."""
    c5h, x1h, x2h = pre_act(p, 'head', c5), pre_act(p, 'head_x1', x1), pre_act(p, 'head_x2', x2)
    xc = rnd_bf16(fl32(conv(p, 'conv_seg', head_feat(p, c5h))))
    h1 = rnd_bf16(fl32(conv(p, 'head_x1', x1h)).clamp_min(0))
    h2 = rnd_bf16(fl32(conv(p, 'head_x2', x2h)).clamp_min(0))
    return oracle.fuse_logits(xc, h1, h2)


def end_to_end(got, labels, model, L64, dev):
    """Engine logits `got` and labels against `model` (the storage-rounded logits from the raw features) and the
    float64 reference L64.  The engine may differ from `model` only by the accumulation order of its fp32 sums,
    which moves a stored value across a rounding boundary now and then: at most dev * (the pixel's largest |logit|).
    The budget of each logit is then its modelled rounding error |model - L64| plus that allowance, and a label may
    differ from L64's argmax only where the top-2 gap of L64 is within the two classes' budgets.
    Returns (logits beyond the allowance, unexplained labels, the measured deviation relative to the scale)."""
    scale = model.abs().amax(1, keepdim=True)
    allow = dev * scale
    off = ~((got - model).abs() <= allow)
    budget = (model - L64).abs() + allow
    ref, lab = L64.argmax(1, keepdim=True), labels.long()[:, None]
    gap = L64.gather(1, ref) - L64.gather(1, lab)
    unexplained = ((lab != ref) & (gap > budget.gather(1, ref) + budget.gather(1, lab)))[:, 0]
    return off, unexplained, ((got - model).abs() / scale.clamp_min(1e-30)).max().item()


def unrounded_chain(p, c5, x1, x2):
    """The same chain with every rounding switched off: LEDHead's math in float64 with folded BatchNorm."""
    c5h = (c5 * p.pre['head'][0][:, None, None] + p.pre['head'][1][:, None, None]).clamp_min(0)
    x1h = (x1 * p.pre['head_x1'][0][:, None, None] + p.pre['head_x1'][1][:, None, None]).clamp_min(0)
    x2h = (x2 * p.pre['head_x2'][0][:, None, None] + p.pre['head_x2'][1][:, None, None]).clamp_min(0)
    xc = conv(p, 'conv_seg', conv(p, 'head', c5h).clamp_min(0))
    r2 = conv(p, 'head_x2', x2h).clamp_min(0) + up_fp16(xc, rounding=False)
    r1 = conv(p, 'head_x1', x1h).clamp_min(0) + up_fp16(r2, rounding=False)
    return up_fp16(r1, rounding=False)


# ---------------------------------------------------------------------------------------------- float64 end to end
def head64(state, C, HC, K, device):
    h = oracle.OracleLEDHead(4 * C, HC, K, tap_channels=C)
    h.load_state_dict({k[len('decode_head.'):]: v for k, v in state.items()})
    return h.double().eval().to(device)


@torch.no_grad()
def logits64(state, C, HC, K, c5, x1, x2):
    """oracle.fuse_logits on float64 head outputs of the original features: no rounding anywhere."""
    xc, h1, h2 = head64(state, C, HC, K, c5.device)((c5, x1, x2))
    return oracle.fuse_logits(xc, h1, h2)
