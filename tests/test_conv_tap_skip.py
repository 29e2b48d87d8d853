"""Tap skipping in conv_tc_kernel: a tile leaves out the taps of the outermost filter dimension with more than one
tap (kt, else kh) whose input box lies wholly in the zero padding.

CPU: the k-blocks each layer of the benchmarked step issues, from dt_conv_plan's tiles and a restatement of the
kernel's range rule (tap_range in csrc/conv_tc.cu).
GPU: outputs with skipping on and off (DT_CONV_TAP_SKIP, read on every dt_conv3d call) are bit-identical; the
skipped products are exact zeros and the remaining k-blocks keep their order."""
import os
from fractions import Fraction

import pytest

from test_conv_plan import R50_FPN_3D, plan


def _cdiv(a, b):
    return -(-a // b)


def _valid_taps(ext, base, n, s, lim):
    """Taps k in [0, ext) whose positions base + k + j*s, j in [0, n), touch [0, lim); all of them when none do."""
    k0 = max(0, -(base + (n - 1) * s))
    k1 = min(ext, lim - base)
    return k1 - k0 if k0 < k1 else ext


def issued_kblocks(o, N, T, H, W, Cout, k, s, p):
    """k-blocks issued over the whole conv with tap skipping: sum over tiles of the tile's [kb, ke) length."""
    To = (T + 2 * p[0] - k[0]) // s[0] + 1
    Ho = (H + 2 * p[1] - k[1]) // s[1] + 1
    Wo = (W + 2 * p[2] - k[2]) // s[2] + 1
    tiles_t, tiles_h = _cdiv(To, o.TT), _cdiv(Ho, o.TH)
    others = _cdiv(Wo, o.TW) * _cdiv(N, o.TB) * _cdiv(Cout, o.BN)
    if k[0] > 1:
        per = o.kiters // k[0]
        walked = sum(_valid_taps(k[0], ti * o.TT * s[0] - p[0], o.TT, s[0], T) for ti in range(tiles_t)) * tiles_h
    elif k[1] > 1:
        per = o.kiters // k[1]
        walked = sum(_valid_taps(k[1], hi * o.TH * s[1] - p[1], o.TH, s[1], H) for hi in range(tiles_h)) * tiles_t
    else:
        return o.tiles * o.kiters
    return walked * per * others


# the post-hoc FPN convs at P3 / P4 (the step also has P2 and P5, listed in R50_FPN_3D)
POST_HOC_P3_P4 = [
    ('fpn post-hoc P3', 8, 3, 100, 168, 256, 256, (3, 3, 3), (1, 1, 1), (1, 1, 1), 0),
    ('fpn post-hoc P4', 8, 3, 50, 84, 256, 256, (3, 3, 3), (1, 1, 1), (1, 1, 1), 0),
]
# issued / full k-blocks of the layers that skip taps; every other layer of the step issues all of them
SKIP_RATIO = {
    'res3 3x3x3': Fraction(7, 9), 'res4 3x3x3': Fraction(7, 9),           # single-frame tiles: frames 0 and 2 drop
    'fpn post-hoc P2': Fraction(7, 9), 'fpn post-hoc P3': Fraction(7, 9),  # one of three kt rows
    'fpn post-hoc P4': Fraction(7, 9),
    'keypoint head conv': Fraction(40, 42),                                 # one-row tiles: rows 0 and 13 drop one kh row
    'keypoint lowres (sub-pixel deconv)': Fraction(40, 42),
    'rpn conv P6': Fraction(14, 15),                                        # the ragged last 3-row tile drops kh = 2
}
LAYERS = R50_FPN_3D + POST_HOC_P3_P4


@pytest.mark.parametrize('layer', LAYERS, ids=[l[0] for l in LAYERS])
def test_issued_kblocks_of_every_bench_layer(layer):
    name, N, T, H, W, Cin, Cout, k, s, p, rm = layer
    o = plan(N, T, H, W, Cin, Cout, k, s, p, res_mode=rm)
    full = o.tiles * o.kiters
    ratio = Fraction(issued_kblocks(o, N, T, H, W, Cout, k, s, p), full)
    assert ratio == SKIP_RATIO.get(name, 1), (ratio, (o.TH, o.TW, o.TT, o.TB))
    if name in SKIP_RATIO and k[0] > 1:
        assert o.TT == 1
    if k[0] == 1 and k[1] == 1:
        assert ratio == 1


def test_range_rule_edge_cases():
    assert _valid_taps(3, -1, 1, 1, 1) == 1                          # T = 1: only the centre tap
    assert _valid_taps(3, 3, 2, 1, 5) == 2                            # ragged stacked tile past the last frame
    assert _valid_taps(3, -1, 2, 1, 5) == 3                           # a stacked box touching frame 0 keeps kt = 0
    assert _valid_taps(3, 1, 1, 2, 3) == 2                            # stride 2: second output frame of T = 3
    assert _valid_taps(3, -5, 1, 1, 3) == 3                           # wholly in the padding: everything is issued


# ---------------------------------------------------------------------------------------------------- GPU
# (N, T, H, W, k, stride, pad, options): kT = 3 with T in {1, 2, 3, 5}, sT in {1, 2}, single-frame tiles, stacked frames
# (t5-stacked: a ragged last stack), stacked images,
# output frame ranges, time-major output, both residual modes, and keypoint-head 3x3s on 14x14 RoI maps (20 RoIs:
# two-row tiles, no row skipped; 18 RoIs: the one-row tiles of the step, rows 0 and 13 skip a kh row)
GPU_CASES = {
    't1': (2, 1, 32, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), {}),
    't2': (2, 2, 32, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), {}),
    't3-plain': (2, 3, 32, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'tt': 1}),
    't3-stacked': (2, 3, 25, 42, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'tt': 3}),
    't3-images': (3, 3, 13, 21, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'tt': 1}),
    't5-plain': (1, 5, 32, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'tt': 1}),
    't5-stacked': (1, 5, 7, 9, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'tt': 2}),
    't1-s2': (2, 1, 24, 40, (3, 3, 3), (2, 1, 1), (1, 1, 1), {}),
    't2-s2': (2, 2, 24, 40, (3, 3, 3), (2, 1, 1), (1, 1, 1), {}),
    't3-s2': (2, 3, 24, 40, (3, 3, 3), (2, 1, 1), (1, 1, 1), {}),
    't5-s2': (1, 5, 24, 40, (3, 3, 3), (2, 2, 2), (1, 1, 1), {}),
    'frames-0-1': (2, 3, 32, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'frames': (0, 1)}),
    'frames-1-2': (2, 3, 13, 21, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'frames': (1, 2)}),
    'time-major': (2, 3, 32, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'time_major': True}),
    'residual': (2, 3, 32, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'res_mode': 1}),
    'upsample-add': (2, 3, 32, 64, (3, 3, 3), (1, 1, 1), (1, 1, 1), {'res_mode': 2}),
    'keypoint-14x14': (20, 1, 14, 14, (1, 3, 3), (1, 1, 1), (0, 1, 1), {'th': 2}),
    'keypoint-14x14-rows': (18, 1, 14, 14, (1, 3, 3), (1, 1, 1), (0, 1, 1), {'th': 1}),
}
MODES = ['bf16', 'bf16x3', 'tf32', 'tf32x3']


def _run_both(fn):
    old = os.environ.get('DT_CONV_TAP_SKIP')
    try:
        os.environ['DT_CONV_TAP_SKIP'] = '0'
        off = fn()
        os.environ['DT_CONV_TAP_SKIP'] = '1'
        on = fn()
    finally:
        if old is None:
            os.environ.pop('DT_CONV_TAP_SKIP', None)
        else:
            os.environ['DT_CONV_TAP_SKIP'] = old
    return off, on


@pytest.mark.gpu
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('case', list(GPU_CASES))
def test_tap_skip_is_bit_identical(case, mode):
    import torch
    from detectandtrack_b200.ops import conv as cv
    N, T, H, W, k, s, p, opt = GPU_CASES[case]
    Cin, Cout = 64, 128
    dtype = cv.MODE_NAMES[mode]
    o = plan(N, T, H, W, Cin, Cout, k, s, p, res_mode=opt.get('res_mode', 0), dtype=cv.kernel_dtype(dtype),
             out_t=opt.get('frames', (0, 0)))
    if 'tt' in opt:
        assert o.TT == opt['tt'], o.TT
    if 'th' in opt:
        assert o.TH == opt['th'], o.TH
    g = torch.Generator().manual_seed(list(GPU_CASES).index(case) * 10 + MODES.index(mode))
    x = torch.randn((N, T, H, W, Cin), generator=g)
    w = torch.randn((Cout, Cin) + k, generator=g) * (2.0 / (Cin * k[0] * k[1] * k[2])) ** 0.5
    scale = (torch.rand(Cout, generator=g) + 0.5).cuda()
    bias = (torch.randn(Cout, generator=g) * 0.1).cuda()
    if dtype in cv.SPLIT_MODES:
        xd = cv.split_for(dtype, x.cuda())
    else:
        xd = x.cuda().to(torch.bfloat16 if dtype == cv.BF16 else torch.float32)
    wp = cv.pack_weight(w, dtype)
    To = (T + 2 * p[0] - k[0]) // s[0] + 1
    Ho = (H + 2 * p[1] - k[1]) // s[1] + 1
    Wo = (W + 2 * p[2] - k[2]) // s[2] + 1
    rm = opt.get('res_mode', 0)
    res = None
    if rm:
        r = torch.randn((N, To, Ho, Wo, Cout) if rm == 1 else (N, To, Ho // 2, Wo // 2, Cout), generator=g).cuda()
        if dtype in cv.SPLIT_MODES:
            res = cv.split_for(dtype, r)
        else:
            res = r.to(torch.bfloat16 if dtype == cv.BF16 else torch.float32)

    def conv():
        y = cv.conv3d(xd, wp, k, s, p, scale, bias, res, rm, True, dtype=dtype, cin=Cin,
                      time_major=opt.get('time_major', False), out_frames=opt.get('frames'))
        torch.cuda.synchronize()
        return y.clone()

    off, on = _run_both(conv)
    assert off.shape == on.shape and off.abs().sum().item() > 0
    assert torch.equal(off, on), (off.float() - on.float()).abs().max().item()
