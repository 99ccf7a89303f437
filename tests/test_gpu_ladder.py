"""The tensor-core logit ladder (ladder_tc.cu), tail2_kernel (tail.cu) and conv_seg's fp16 output, rung by rung.

Harness: `Engine.head_infer` on caller features (the PLAN_HEAD_NHWC plan), so every rung size is chosen directly:
x_c is h8 x w8, r2 2h8 x 2w8, r1 4h8 x 4w8, labels 8h8 x 8w8.  Head parameters fold exactly
(tests/ladder_oracle.py), so each stored stage can be compared with a storage-aware float64 reference computed from
the fetched input of that stage: the one unmodelled difference is the fp32 accumulation order of the tensor-core sums.
Failures name the stage, the pixel and the class.
"""
import pytest
import torch

from lednet_b200.engine import Engine
import ladder_oracle as LO

pytestmark = pytest.mark.gpu
DEV = 'cuda'
ACC = 2.0 ** -16            # fp32 accumulation-order slack, relative to sum |w x| + |b| of the conv
# Engine logits vs the storage-rounded model from the raw features, relative to the pixel's largest |logit|: an fp32
# sum that lands on the other side of a rounding boundary than the exact one moves a stored value by one ulp.  In the
# ladder that is mostly a bf16 ulp of head.feat (2^-7 relative) carried through conv_seg; the B200 reaches 2^-8.1 at
# the 512 x 1024 rung, an fp32-accumulating stand-in for the tensor cores 2^-9.7.  The K <= 16 path stores its rungs
# in bf16: one ulp, 2^-7, as well.
DEV_LADDER = 2.0 ** -7
DEV_FALLBACK = 2.0 ** -7

# (N, h8, w8): r1 = 4h8 x 4w8
SHAPES = [
    (1, 1, 1),          # smaller than one tile in both axes; x_c 1 x 1
    (2, 1, 2),          # one tile wide exactly, short
    (1, 4, 2),          # exactly one final-rung tile
    (1, 5, 3),          # shifted last tile in both axes; ragged r2 tiles
    (3, 9, 15),         # several shifted tiles, odd tile origins, N > 1
    (4, 64, 1),         # tiles_w == 1
    (4, 1, 128),        # tiles_h == 1
    (8, 32, 64),        # more tiles than 4 x 148: persistent loop, both MMA issuers, ring wrap
    (2, 128, 256),      # the rung size of a 1024 x 2048 image
]
CASES = ([(s, K, 32, 64) for s in SHAPES for K in (17, 19, 23, 24)] +
         [(s, K, 64, 64) for s in (SHAPES[0], SHAPES[3], SHAPES[4], SHAPES[7]) for K in (19, 24)] +
         [(SHAPES[4], 19, 32, 128)])


def _id(case):
    (n, h, w), K, C, HC = case
    return f'N{n}_h{h}_w{w}_K{K}_C{C}_HC{HC}'


def features(shape, C, seed, scale=1.0):
    """Seeded bf16 features (c5, x1, x2) in channels_last memory, so that head_infer reads them in place."""
    N, h8, w8 = shape
    g = torch.Generator().manual_seed(seed)

    def f(c, h, w):
        t = (torch.randn((N, c, h, w), generator=g) * scale).bfloat16()
        return t.to(DEV).contiguous(memory_format=torch.channels_last)
    return f(4 * C, h8, w8), f(C, 4 * h8, 4 * w8), f(C, 2 * h8, 2 * w8)


def engine(state, K, C, HC):
    return Engine(state, K, channels=C, head_channels=HC, dtype='bf16', allow_partial=True)


def fill_value(dtype):
    return 255 if dtype == torch.uint8 else -1


def run(eng, feats, pred, want_logits=False):
    """One head_infer call into `pred`, pre-filled so that a pixel the kernels never write cannot look right."""
    pred.fill_(fill_value(pred.dtype))
    out = eng.head_infer(*feats, pred=pred, want_logits=want_logits)
    torch.cuda.synchronize()
    return out


def new_pred(feats, dtype):
    N, _, h8, w8 = feats[0].shape
    return torch.empty((N, 8 * h8, 8 * w8), dtype=dtype, device=DEV)


def ops(eng):
    return {name: kind for name, kind, _, _ in eng.op_info()}


def assert_ladder_path(eng):
    o = ops(eng)
    assert o.get('decode_head.head_x1') == 'conv_tc' and o.get('decode_head.head_x2') == 'conv_tc', o
    assert 'tail.up2_argmax' in o and 'tail.fuse_argmax' not in o, o


def fetch(eng, name):
    return eng.debug_fetch(name).double().to(DEV)


def where(mask):
    """(n, k, y, x) of the first True element."""
    return tuple(int(i) for i in mask.nonzero()[0])


def check_stage(name, got, ref, fmt, acc=None):
    """got within one ulp of its storage format of ref, plus the accumulation-order slack; exact where ref saturates."""
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    mant, emin = LO.FMT[fmt]
    tol = LO.ulp(torch.maximum(got.abs(), ref.abs()), mant, emin)
    if acc is not None:
        tol = tol + ACC * acc
    bad = ~((got - ref).abs() <= tol)
    if fmt == 'f16':
        bad |= (ref.abs() == LO.F16_MAX) & (got != ref)
    same = (got == ref).double().mean().item()
    print(f'{name}: {100 * same:.3f} % bit-identical')
    if bad.any():
        i = where(bad)
        raise AssertionError(f'{name}: {int(bad.sum())} of {bad.numel()} elements beyond 1 ulp; first at (n, k, y, x) = {i}: '
                             f'got {got[i].item()!r}, reference {ref[i].item()!r}, tolerance {tol[i].item()!r}')
    return same


def check_logits(logits, r1):
    """tail2's logits against its exact emulation on the fetched r1, and against the float64 upsample elementwise."""
    got = logits.double()
    ref64 = LO.up_fp16(r1, rounding=False)
    bound = 4 * 2.0 ** -24 * LO.corner_max(r1)
    bad = ~((got - ref64).abs() <= bound)
    if bad.any():
        i = where(bad)
        raise AssertionError(f'logits: {int(bad.sum())} elements off the x2 upsample of r1; first at {i}: '
                             f'got {got[i].item()!r}, reference {ref64[i].item()!r}')
    emu = LO.up_f32(r1)
    diff = got != emu
    print(f'logits: {100 * (1 - diff.double().mean().item()):.3f} % bit-identical to the fp32 lerp emulation')
    if diff.any():
        i = where(diff)
        raise AssertionError(f'logits: {int(diff.sum())} elements differ from the fp32 lerp order; first at {i}: '
                             f'got {got[i].item()!r}, emulation {emu[i].item()!r}')


def check_stages(eng, state, feats, logits):
    """Every stored stage of the last want_logits call against its storage-aware reference from the fetched input."""
    p = LO.HeadParams(state, DEV)
    c5, x1, x2 = (t.double() for t in feats)
    st = {n: fetch(eng, n) for n in ('c5h', 'x1h', 'x2h', 'head.feat', 'xc', 'hx2', 'hx1')}
    check_stage('c5h', st['c5h'], LO.pre_act(p, 'head', c5), 'bf16')
    check_stage('x1h', st['x1h'], LO.pre_act(p, 'head_x1', x1), 'bf16')
    check_stage('x2h', st['x2h'], LO.pre_act(p, 'head_x2', x2), 'bf16')
    check_stage('head.feat', st['head.feat'], LO.head_feat(p, st['c5h']), 'bf16', LO.conv(p, 'head', st['c5h'], True))
    check_stage('xc', st['xc'], LO.x_c(p, st['head.feat']), 'f16', LO.conv(p, 'conv_seg', st['head.feat'], True))
    check_stage('r2 (hx2)', st['hx2'], LO.rung(p, 'head_x2', st['x2h'], st['xc']), 'f16',
                LO.conv(p, 'head_x2', st['x2h'], True))
    check_stage('r1 (hx1)', st['hx1'], LO.rung(p, 'head_x1', st['x1h'], st['hx2']), 'f16',
                LO.conv(p, 'head_x1', st['x1h'], True))
    check_logits(logits, st['hx1'])
    return st


def check_vs_float64(state, C, HC, K, feats, logits, labels):
    """Logits within the accumulation-order allowance of the storage-rounded model computed from the raw features, and
    every label that differs from the float64 reference's argmax where that pixel's top-2 gap is within the modelled
    rounding error of the two classes plus the allowance (ladder_oracle.end_to_end)."""
    p = LO.HeadParams(state, DEV)
    c5, x1, x2 = (t.double() for t in feats)
    ladder = K > 16
    model = (LO.ladder_logits if ladder else LO.fallback_logits)(p, c5, x1, x2)
    L64 = LO.logits64(state, C, HC, K, c5, x1, x2)
    dev = DEV_LADDER if ladder else DEV_FALLBACK
    off, unexplained, measured = LO.end_to_end(logits.double(), labels, model, L64, dev)
    mism = labels.long() != L64.argmax(1)
    print(f'logits vs storage model: largest deviation 2^{torch.tensor(measured).log2().item():.1f} of the pixel scale '
          f'(allowed 2^{torch.tensor(dev).log2().item():.0f}); labels vs float64 argmax: {int(mism.sum())} of '
          f'{mism.numel()} differ, {int(unexplained.sum())} beyond the budget')
    if off.any():
        i = where(off)
        raise AssertionError(f'logits: {int(off.sum())} elements off the storage model beyond the allowance; first at '
                             f'(n, k, y, x) = {i}: got {logits[i].item()!r}, model {model[i].item()!r}, '
                             f'float64 {L64[i].item()!r}')
    if unexplained.any():
        i = tuple(int(v) for v in unexplained.nonzero()[0])
        raise AssertionError(f'label at (n, y, x) = {i} is {int(labels[i])}, float64 reference {int(L64.argmax(1)[i])}: '
                             f'top-2 gap beyond the rounding budget')


def assert_labels(name, got, want):
    if not torch.equal(got, want):
        d = got != want
        i = tuple(int(v) for v in d.nonzero()[0])
        raise AssertionError(f'{name}: {int(d.sum())} labels differ; first at (n, y, x) = {i}: {int(got[i])} vs {int(want[i])}')


# ---------------------------------------------------------------------------------------------- a. stages
@pytest.mark.parametrize('case', CASES, ids=_id)
def test_ladder_stages(case):
    shape, K, C, HC = case
    state = LO.exact_fold_state(C, HC, K, seed=K + C)
    LO.assert_exact_fold(state)
    feats = features(shape, C, seed=sum(shape) + K)
    eng = engine(state, K, C, HC)
    pred, logits = run(eng, feats, new_pred(feats, torch.uint8), want_logits=True)
    assert_ladder_path(eng)
    check_stages(eng, state, feats, logits)


# ---------------------------------------------------------------------------------------------- b. labels
@pytest.mark.parametrize('case', CASES, ids=_id)
def test_ladder_labels(case, monkeypatch):
    shape, K, C, HC = case
    state = LO.exact_fold_state(C, HC, K, seed=K + C)
    feats = features(shape, C, seed=sum(shape) + K)
    eng = engine(state, K, C, HC)
    for dtype in (torch.uint8, torch.int64):
        fill = fill_value(dtype)
        pred_lg, pred = new_pred(feats, dtype), new_pred(feats, dtype)
        _, logits = run(eng, feats, pred_lg, want_logits=True)         # r1 stored, tail2_kernel: logits + labels
        run(eng, feats, pred)                                          # ladder_kernel<true>: labels only
        assert_ladder_path(eng)
        assert not (pred_lg == fill).any() and not (pred == fill).any(), 'a label was never written'
        assert_labels('label-only vs logits path', pred, pred_lg)
        assert_labels('logits path vs logits.argmax', pred_lg, logits.argmax(1).to(dtype))
        first = pred.clone()
        run(eng, feats, pred)                                          # same buffers: graph replay
        assert_labels('graph replay', pred, first)
    check_vs_float64(state, C, HC, K, feats, logits, pred)
    # the uniform-corner shortcut off (read at launch, frozen into the captured graph: a fresh engine)
    monkeypatch.setenv('LEDB200_LADDER_DBG', '64')
    eng64 = engine(state, K, C, HC)
    p64 = run(eng64, feats, new_pred(feats, torch.int64))
    monkeypatch.delenv('LEDB200_LADDER_DBG')
    assert_labels('shortcut off vs on', p64, pred)


# ---------------------------------------------------------------------------------------------- d. content edges
def _tie(state, a, b):
    """Make class b a bitwise copy of class a in conv_seg, head_x1 and head_x2 (weights and folded BatchNorm), and
    give both a larger bias."""
    s = {k: v.clone() for k, v in state.items()}
    s['decode_head.conv_seg.bias'][a] = 2.0                  # a wins often enough for a wrong tie-break to show
    for name in ('conv_seg.weight', 'conv_seg.bias', 'head_x1.0.conv.weight', 'head_x2.0.conv.weight'):
        s['decode_head.' + name][b] = s['decode_head.' + name][a]
    for bn in ('head_x1.1', 'head_x2.1'):
        for leaf in ('weight', 'bias', 'running_mean', 'running_var'):
            s[f'decode_head.{bn}.{leaf}'][b] = s[f'decode_head.{bn}.{leaf}'][a]
    return s


@pytest.mark.parametrize('K,a,b', [(24, 1, 22), (24, 6, 23), (19, 2, 17)])
def test_ladder_ties(K, a, b):
    """Two classes with identical parameters: identical logit planes, and the first-max rule never picks b
    (K = 24 runs without the shortcut, K = 19 with it)."""
    C, HC, shape = 32, 64, (3, 9, 15)
    state = _tie(LO.exact_fold_state(C, HC, K, seed=7), a, b)
    feats = features(shape, C, seed=8)
    eng = engine(state, K, C, HC)
    pred_lg, logits = run(eng, feats, new_pred(feats, torch.int64), want_logits=True)
    for n in ('xc', 'hx2', 'hx1'):
        t = eng.debug_fetch(n)
        assert torch.equal(t[:, a], t[:, b]), n
    assert torch.equal(logits[:, a], logits[:, b])
    pred = run(eng, feats, new_pred(feats, torch.int64))
    assert_ladder_path(eng)
    assert (pred_lg == a).any(), 'the tied class never wins: the test would not see a wrong tie-break'
    assert not (pred_lg == b).any() and not (pred == b).any()
    assert_labels('label-only vs logits path', pred, pred_lg)


@pytest.mark.parametrize('K', [19, 24])
def test_ladder_constant_features(K):
    """All-zero features and per-class biases that are all equal: every logit ties, so every label is 0."""
    C, HC, shape = 32, 64, (3, 9, 15)
    s = LO.exact_fold_state(C, HC, K, seed=11)
    for bn in ('head.0.bn', 'head_x1.0.bn', 'head_x2.0.bn'):
        s[f'decode_head.{bn}.bias'].zero_()
    s['decode_head.head.1.bias'].fill_(-0.5)              # head.feat = relu(-0.5) = 0: x_c = conv_seg.bias
    s['decode_head.conv_seg.bias'].fill_(0.25)
    s['decode_head.head_x1.1.bias'].fill_(0.5)
    s['decode_head.head_x2.1.bias'].fill_(-0.125)
    feats = tuple(torch.zeros_like(t) for t in features(shape, C, seed=0))
    eng = engine(s, K, C, HC)
    for dtype in (torch.uint8, torch.int64):
        pred_lg, logits = run(eng, feats, new_pred(feats, dtype), want_logits=True)
        pred = run(eng, feats, new_pred(feats, dtype))
        assert_ladder_path(eng)
        assert torch.equal(logits, logits[:, :1].expand_as(logits))
        assert (logits[:, 0] == 0.75).all()
        assert (pred_lg == 0).all() and (pred == 0).all()


@pytest.mark.parametrize('K', [17, 24])
def test_ladder_saturation(K):
    """Features scaled so that x_c, r2 and r1 leave fp16's range: the rungs saturate at exactly +-65504 where the
    reference does, the logits stay finite and the labels follow the saturated reference."""
    C, HC, shape = 32, 64, (3, 9, 15)
    state = LO.exact_fold_state(C, HC, K, seed=13)
    feats = features(shape, C, seed=14, scale=2.0 ** 17)
    eng = engine(state, K, C, HC)
    pred_lg, logits = run(eng, feats, new_pred(feats, torch.int64), want_logits=True)
    pred = run(eng, feats, new_pred(feats, torch.int64))
    assert_ladder_path(eng)
    assert torch.isfinite(logits).all()
    st = check_stages(eng, state, feats, logits)
    for n in ('xc', 'hx2', 'hx1'):
        assert (st[n] == LO.F16_MAX).any(), f'{n} never saturates: scale the features up'
    assert (st['hx2'] == -LO.F16_MAX).any() and (st['hx1'] == -LO.F16_MAX).any()
    assert_labels('label-only vs logits path', pred, pred_lg)
    assert_labels('logits path vs logits.argmax', pred_lg, logits.argmax(1))
    p = LO.HeadParams(state, DEV)
    ref = LO.up_f32(LO.rung(p, 'head_x1', st['x1h'], st['hx2']))
    top2 = ref.topk(2, dim=1).values
    mism = pred != ref.argmax(1)
    near = (top2[:, 0] - top2[:, 1]) <= 2 * LO.ulp(top2[:, 0], 11, -14)
    print(f'saturated labels vs reference: {int(mism.sum())} of {mism.numel()} differ')
    assert not (mism & ~near).any()


@pytest.mark.parametrize('K,shape', [(17, (1, 5, 3)), (17, (3, 9, 15)), (24, (3, 9, 15))])
def test_ladder_poisoned_workspace(K, shape, monkeypatch):
    """A workspace filled with the byte 0x7F before first use changes no bit: no kernel reads the never-written pad
    channels K..23 of x_c, r2 and r1, or a halo it did not write.  0x7F7F is NaN in the fp16 buffers (x_c, r2, r1)
    but the finite 3.39e38 in the bf16 ones (c5h, x1h, x2h, head.feat): the test rests on bit equality, not on NaN
    propagation."""
    C, HC = 32, 64
    state = LO.exact_fold_state(C, HC, K, seed=17)
    feats = features(shape, C, seed=18)

    def both(eng):
        pred_lg, logits = run(eng, feats, new_pred(feats, torch.uint8), want_logits=True)
        return pred_lg, logits, run(eng, feats, new_pred(feats, torch.uint8))
    clean = both(engine(state, K, C, HC))
    monkeypatch.setenv('LEDB200_POISON', '127')
    eng = engine(state, K, C, HC)
    poisoned = both(eng)
    monkeypatch.delenv('LEDB200_POISON')
    assert_ladder_path(eng)
    assert_labels('poisoned logits path', poisoned[0], clean[0])
    assert torch.equal(poisoned[1], clean[1])
    assert_labels('poisoned label-only', poisoned[2], clean[2])


# ---------------------------------------------------------------------------------------------- e. fallback pinned
@pytest.mark.parametrize('K', [2, 16])
def test_small_k_heads_take_the_tail_kernel(K):
    """K <= 16 stores x_c and r2 with a pixel stride of kpad(K), not the ladder's 24: those heads run tail_kernel.
    Widening the ladder to them is a deliberate change of this test."""
    C, HC, shape = 32, 64, (3, 9, 15)
    state = LO.exact_fold_state(C, HC, K, seed=19)
    feats = features(shape, C, seed=20)
    eng = engine(state, K, C, HC)
    for dtype in (torch.uint8, torch.int64):
        pred_lg, logits = run(eng, feats, new_pred(feats, dtype), want_logits=True)
        pred = run(eng, feats, new_pred(feats, dtype))
        o = ops(eng)
        assert 'tail.fuse_argmax' in o and 'tail.up2_argmax' not in o, o
        assert not (pred == fill_value(dtype)).any() and not (pred_lg == fill_value(dtype)).any()
        assert_labels('labels vs logits.argmax', pred_lg, logits.argmax(1).to(dtype))
        assert_labels('label-only vs logits path', pred, pred_lg)
    check_vs_float64(state, C, HC, K, feats, logits, pred)
