"""The float64 references of tests/test_gpu_ladder.py, checked on the host: the fp16 `up` gather emulation, the fp32
lerp emulation of tail2, the exact-fold parameters, and the unrounded rung chain against oracle.fuse_logits."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import ladder_oracle as LO
import test_gpu_ladder as G


@pytest.mark.parametrize('h,w', [(1, 1), (1, 2), (2, 1), (2, 2), (3, 5), (4, 7), (9, 6)])
def test_up_unrounded_is_bilinear_x2(h, w):
    u = torch.randn(2, 3, h, w, dtype=torch.float64, generator=torch.Generator().manual_seed(h * 10 + w))
    ref = F.interpolate(u, size=(2 * h, 2 * w), mode='bilinear', align_corners=False)
    got = LO.up_fp16(u, rounding=False)
    assert (got - ref).abs().max().item() <= 1e-12
    # rows / columns 0 and last are copies along the edge
    assert torch.equal(got[..., 0, 0], u[..., 0, 0]) and torch.equal(got[..., -1, -1], u[..., -1, -1])


def test_up_f32_is_bilinear_x2_to_fp32_rounding():
    u = torch.randn(1, 4, 5, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(0)).half().double()
    ref = F.interpolate(u, scale_factor=2, mode='bilinear', align_corners=False)
    got = LO.up_f32(u)
    assert torch.equal(got, got.float().double())
    assert ((got - ref).abs() <= 4 * 2.0 ** -24 * LO.corner_max(u)).all()


def test_up_fp16_hand_computed():
    # one row [a, b]: output columns 0..3 read (a, a), (a, b) 3/4 : 1/4, (a, b) 1/4 : 3/4, (b, b)
    a = 1 + 2.0 ** -10
    u = torch.tensor([[[[a, 0.0]]]], dtype=torch.float64)
    got = LO.up_fp16(u)[0, 0]
    # a * 3/4 = 0.750732421875 is a tie between fp16 neighbours 0.75048828125 and 0.7509765625: to even
    assert got[0].tolist() == [a, 0.7509765625, 0.250244140625, 0.0]
    assert torch.equal(got[0], got[1])                       # one source row: both output rows are copies
    # fp16's top binade: 65504 * 3/4 = 49128 -> 49120, then -16376 + 49120 = 32744, a tie -> 32736 (bilinear: 32752)
    u = torch.tensor([[[[65504.0, -65504.0]]]], dtype=torch.float64)
    assert LO.up_fp16(u)[0, 0, 0].tolist() == [65504.0, 32736.0, -32752.0, -65504.0]


def test_fp16_roundings_hand_computed():
    x = torch.tensor([65519.0, 65520.0, 1e6, -1e6, 2049.0, 2051.0, 2.0 ** -25, 3 * 2.0 ** -26, float('nan')],
                     dtype=torch.float64)
    r = LO.rnd16(x).tolist()
    assert r[:8] == [65504.0, float('inf'), float('inf'), float('-inf'), 2048.0, 2052.0, 0.0, 2.0 ** -24]
    s = LO.sat16(x)
    assert s[:8].tolist() == [65504.0, 65504.0, 65504.0, -65504.0, 2048.0, 2052.0, 0.0, 2.0 ** -24]
    assert torch.isnan(s[8])
    assert LO.rnd_bf16(torch.tensor([1 + 2.0 ** -8, 1 + 3 * 2.0 ** -8], dtype=torch.float64)).tolist() == \
        [1.0, 1 + 2.0 ** -6]


def test_roundings_match_torch_casts():
    x = torch.randn(100000, dtype=torch.float64, generator=torch.Generator().manual_seed(1)) * 100
    x32 = x.float().double()                                 # on fp32 inputs torch's casts round once
    assert torch.equal(LO.rnd16(x32), x32.float().half().double())
    assert torch.equal(LO.rnd_bf16(x32), x32.float().bfloat16().double())


@pytest.mark.parametrize('C,HC,K', [(32, 64, 19), (64, 64, 24), (32, 128, 17)])
def test_exact_fold_state(C, HC, K):
    for j in range(3):                                       # sqrt(fl32(4**j - 1e-5) + 1e-5f) == 2**j in float32
        v = np.float32(4.0 ** j - 1e-5)
        assert np.sqrt(v + np.float32(1e-5)) == np.float32(2.0 ** j)
    state = LO.exact_fold_state(C, HC, K, seed=3)
    LO.assert_exact_fold(state)
    scales = torch.cat([LO.folded_bn(state, p)[0] for p in LO.BN_PREFIXES])
    assert len(set(scales.tolist())) > 1                     # not all ones: the folding is exercised
    # a plain state dict does not fold exactly: the check has teeth
    bad = dict(state)
    bad['decode_head.head_x1.1.running_var'] = torch.full_like(state['decode_head.head_x1.1.running_var'], 2.0)
    with pytest.raises(AssertionError):
        LO.assert_exact_fold(bad)


def test_unrounded_chain_is_fuse_logits():
    C, HC, K = 32, 64, 19
    state = LO.exact_fold_state(C, HC, K, seed=4)
    g = torch.Generator().manual_seed(5)
    c5, x1, x2 = (torch.randn(s, dtype=torch.float64, generator=g) for s in
                  ((2, 4 * C, 3, 5), (2, C, 12, 20), (2, C, 6, 10)))
    p = LO.HeadParams(state, 'cpu')
    got = LO.unrounded_chain(p, c5, x1, x2)
    ref = LO.logits64(state, C, HC, K, c5, x1, x2)
    assert got.shape == ref.shape == (2, K, 24, 40)
    # the oracle folds sqrt(fl32(4**j - 1e-5) + 1e-5) in float64: not exactly 2**j, off by ~1e-8 relative
    scale = ref.abs().amax(1, keepdim=True)
    assert ((got - ref).abs() <= 1e-6 * scale).all()


def _swapped_up(u, rounding=True):
    """up_fp16 with the horizontal weights of the top pair swapped: a wrong `up` gather."""
    R = LO.rnd16
    h, w = u.shape[-2:]
    ya, yb, wy0, wy1 = LO._taps(2 * h, h, u.device)
    xa, xb, wx0, wx1 = LO._taps(2 * w, w, u.device)
    top, bot = u[..., ya, :], u[..., yb, :]
    h0 = R(top[..., xb] * wx0 + R(top[..., xa] * wx1))
    h1 = R(bot[..., xb] * wx1 + R(bot[..., xa] * wx0))
    return R(h1 * wy1[:, None] + R(h0 * wy0[:, None]))


def _case(shape, K, C=32, HC=64):
    """The GPU file's parameters and features for one case, on the host (float64)."""
    state = LO.exact_fold_state(C, HC, K, seed=K + C)
    N, h8, w8 = shape
    g = torch.Generator().manual_seed(sum(shape) + K)
    c5, x1, x2 = (torch.randn(s, generator=g).bfloat16().double() for s in
                  ((N, 4 * C, h8, w8), (N, C, 4 * h8, 4 * w8), (N, C, 2 * h8, 2 * w8)))
    return state, (c5, x1, x2), LO.logits64(state, C, HC, K, c5, x1, x2)


@pytest.mark.parametrize('shape', G.SHAPES[:2])
def test_gpu_references_run_on_cpu(shape):
    """The references of the GPU file at its two smallest shapes: the stored chain rounds where the engine does, and
    an fp32-accumulating stand-in for the engine passes the end-to-end check."""
    K = 24
    state, (c5, x1, x2), L64 = _case(shape, K)
    N, h8, w8 = shape
    p = LO.HeadParams(state, 'cpu')
    st = LO.chain(p, c5, x1, x2)
    for n in ('c5h', 'x1h', 'x2h', 'head.feat'):
        assert torch.equal(st[n], LO.rnd_bf16(st[n])), n
    for n in ('xc', 'hx2', 'hx1'):
        assert torch.equal(st[n], LO.sat16(st[n])), n
    assert st['hx1'].shape == (N, K, 4 * h8, 4 * w8)
    model = LO.up_f32(st['hx1'])
    got = LO.ladder_logits(LO.HeadParams(state, 'cpu', acc=torch.float32), c5, x1, x2)
    off, unexplained, _ = LO.end_to_end(got, got.argmax(1), model, L64, G.DEV_LADDER)
    assert not off.any() and not unexplained.any()


@pytest.mark.parametrize('shape,K', [((3, 9, 15), 24), ((3, 9, 15), 19), ((1, 5, 3), 16), ((3, 9, 15), 2)])
def test_end_to_end_check_rejects_wrong_results(shape, K, monkeypatch):
    """The end-to-end check of the GPU file has teeth: it passes an fp32-accumulating stand-in for the engine, and
    rejects the argmin label, random labels and a wrong `up` gather."""
    state, feats, L64 = _case(shape, K)
    ladder = K > 16
    fn = LO.ladder_logits if ladder else LO.fallback_logits
    dev = G.DEV_LADDER if ladder else G.DEV_FALLBACK
    model = fn(LO.HeadParams(state, 'cpu'), *feats)
    got = fn(LO.HeadParams(state, 'cpu', acc=torch.float32), *feats)
    off, unexplained, _ = LO.end_to_end(got, got.argmax(1), model, L64, dev)
    assert not off.any() and not unexplained.any()
    ref = L64.argmax(1)
    _, unexplained, _ = LO.end_to_end(got, got.argmin(1), model, L64, dev)
    assert unexplained.double().mean() > 0.95
    rnd = torch.randint(0, K, ref.shape, generator=torch.Generator().manual_seed(0))
    _, unexplained, _ = LO.end_to_end(got, rnd, model, L64, dev)
    assert unexplained.sum() >= 0.95 * (rnd != ref).sum()
    if ladder:
        monkeypatch.setattr(LO, 'up_fp16', _swapped_up)
        wrong = fn(LO.HeadParams(state, 'cpu'), *feats)
        monkeypatch.undo()
        off, unexplained, _ = LO.end_to_end(wrong, wrong.argmax(1), model, L64, dev)
        assert off.any() and unexplained.any()
