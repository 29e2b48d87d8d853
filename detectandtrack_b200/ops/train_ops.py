"""Device-tensor API over csrc/train_ops.cu (training step kernels: filter gradient on the tensor cores over
channel-major planes, elementwise backward joins, SGD update).  See include/dt_b200.h."""
import ctypes as C

from .. import _lib as L
from . import conv as cv


def planes_ld(Ho, Wo, pH, pW):
    return int(L.lib().dt_planes_ld(int(Ho), int(Wo), int(pH), int(pW)))


def to_planes(x, pad=(0, 0), stride=(1, 1), channels=None, copies=False):
    """x [N, T, H, W, ld] bf16 -> planes [N, T, C, Pld] (zero border pad, spatial subsampling stride).
    copies=True: the wgrad INPUT operand [2*pad_w + 1, N, T, C, Pld], copy kw pre-shifted by kw - pad_w columns."""
    torch = L.require_cuda()
    N, T, H, W, ld = x.shape
    Cc = channels or ld
    assert x.dtype == torch.bfloat16 and x.is_contiguous()
    Ho, Wo = (H + stride[0] - 1) // stride[0], (W + stride[1] - 1) // stride[1]
    Pld = planes_ld(Ho, Wo, pad[0], pad[1])
    shifts = list(range(-pad[1], pad[1] + 1)) if copies else [0]
    out = torch.empty((len(shifts), N, T, Cc, Pld), dtype=torch.bfloat16, device='cuda')
    L.call('dt_to_planes', L.ptr(x), N * T, H, W, Cc, ld, stride[0], stride[1], pad[0], pad[1], shifts[0], len(shifts), L.ptr(out),
           L.stream_ptr())
    return out if copies else out[0]


def wgrad(gz_planes, x_planes, out_hw, ksize, dW=None):
    """gz_planes [N,T,Cout,Pld], x_planes [kW,N,T,Cin,Pld] (to_planes(copies=True), pad = k // 2) -> dW [taps, Cout, Cin] fp32
    (accumulated into `dW` if given, else a zeroed buffer)."""
    torch = L.require_cuda()
    N, T, Cout, Pld = gz_planes.shape
    kT, kH, kW = ksize
    assert x_planes.dim() == 5 and x_planes.shape[0] == kW, 'x_planes: to_planes(..., copies=True) -> [kW, N, T, Cin, Pld]'
    Cin = x_planes.shape[3]
    assert x_planes.shape[1] == N and x_planes.shape[2] == T and x_planes.shape[4] == Pld and x_planes.is_contiguous()
    assert Pld == planes_ld(out_hw[0], out_hw[1], kH // 2, kW // 2)
    if dW is None:
        dW = L.zeros((kT * kH * kW, Cout, Cin), torch.float32)
    assert dW.dtype == torch.float32 and tuple(dW.shape) == (kT * kH * kW, Cout, Cin) and dW.is_contiguous()
    L.call('dt_wgrad', L.ptr(gz_planes), L.ptr(x_planes), N, T, out_hw[0], out_hw[1], Cout, Cin, kT, kH, kW, L.ptr(dW), L.stream_ptr())
    return dW


def wgrad_nhwc(gz, x, ksize, stride=(1, 1), dW=None, cout=None, cin=None):
    """Filter gradient straight from the NDHWC tensors: gz [N,T,Ho,Wo,ld_g], x [N,T,Hi,Wi,ld_x] bf16 -> dW [taps, Cout, Cin] fp32
    (accumulated into `dW` if given).  stride (sH, sW) > 1 only for pointwise convs."""
    torch = L.require_cuda()
    N, T, Ho, Wo, ld_g = gz.shape
    _, _, Hi, Wi, ld_x = x.shape
    Cout, Cin = cout or ld_g, cin or ld_x
    kT, kH, kW = ksize
    assert gz.dtype == torch.bfloat16 and x.dtype == torch.bfloat16 and gz.is_contiguous() and x.is_contiguous() and x.shape[0] == N and x.shape[1] == T
    if dW is None:
        dW = L.zeros((kT * kH * kW, Cout, Cin), torch.float32)
    assert dW.dtype == torch.float32 and tuple(dW.shape) == (kT * kH * kW, Cout, Cin) and dW.is_contiguous()
    L.call('dt_wgrad_nhwc', L.ptr(gz), ld_g, L.ptr(x), ld_x, N, T, Ho, Wo, Hi, Wi, Cout, Cin, kT, kH, kW, int(stride[0]), int(stride[1]),
           L.ptr(dW), L.stream_ptr())
    return dW


def bwd_pointwise(g1, g2=None, y=None, scale=None, second=False, scale2=None):
    """(g1 + g2) * [y > 0] * scale[c] over NDHWC bf16 tensors of one shape.  second=True: also returns the same masked sum
    times scale2[c] (or unscaled) from the same read of the inputs -> (out, out2)."""
    torch = L.require_cuda()
    Cc = g1.shape[-1]
    out = torch.empty_like(g1)
    for t in (g1, g2, y):
        assert t is None or (t.dtype == torch.bfloat16 and t.is_contiguous() and t.shape == g1.shape)
    if not second:
        L.call('dt_bwd_pointwise', L.ptr(g1), L.ptr(g2), L.ptr(y), L.ptr(scale), g1.numel() // Cc, Cc, L.ptr(out), L.stream_ptr())
        return out
    out2 = torch.empty_like(g1)
    L.call('dt_bwd_pointwise2', L.ptr(g1), L.ptr(g2), L.ptr(y), L.ptr(scale), g1.numel() // Cc, Cc, L.ptr(out), L.ptr(scale2), L.ptr(out2),
           L.stream_ptr())
    return out, out2


def upsample_add_bwd(fine, coarse_in=None):
    """fine [N,T,2Hc,2Wc,C] -> [N,T,Hc,Wc,C] = coarse_in + 2x2 sums (backward of the FPN nearest-2x top-down add)."""
    torch = L.require_cuda()
    N, T, H2, W2, Cc = fine.shape
    out = torch.empty((N, T, H2 // 2, W2 // 2, Cc), dtype=torch.bfloat16, device='cuda')
    L.call('dt_upsample_add_bwd', L.ptr(fine), L.ptr(coarse_in), N * T, H2 // 2, W2 // 2, Cc, L.ptr(out), L.stream_ptr())
    return out


def scatter_stride2(src, hw):
    """src [N,T,ceil(H/2),ceil(W/2),C] -> [N,T,H,W,C] with src on the even positions (dgrad of a stride-2 1x1 conv)."""
    torch = L.require_cuda()
    N, T, Hs, Ws, Cc = src.shape
    out = torch.empty((N, T, hw[0], hw[1], Cc), dtype=torch.bfloat16, device='cuda')
    L.call('dt_scatter_stride2', L.ptr(src), N * T, Hs, Ws, hw[0], hw[1], Cc, L.ptr(out), L.stream_ptr())
    return out


def sgd_update(w, g, m, lr, momentum=0.9, wd=1e-4, grad_scale=1.0, w_fwd=None, w_dgrad=None):
    """MomentumSGDUpdate on packed fp32 master weights [taps, Cout, Cin]; refreshes the bf16 forward / dgrad filters."""
    taps, Cout, Cin = w.shape
    L.call('dt_sgd_update', L.ptr(w), L.ptr(g), L.ptr(m), taps, Cout, Cin, float(lr), float(momentum), float(wd), float(grad_scale),
           L.ptr(w_fwd), L.ptr(w_dgrad), L.stream_ptr())


def pack_dgrad_weight(w):
    """Filter (Cout, Cin, kT, kH, kW) -> the dgrad filter in dt_conv3d's packed order [taps (flipped), Cin, Cout] bf16:
    dX = conv(dY, flip(W)^T) for a stride-1 'same' conv."""
    torch = L.require_cuda()
    if w.dim() == 2:
        w = w[:, :, None, None, None]
    elif w.dim() == 4:
        w = w[:, :, None]
    wt = w.to('cuda').float().flip(2, 3, 4).permute(1, 0, 2, 3, 4).contiguous()      # (Cin, Cout, kT, kH, kW), flipped
    return cv.pack_weight(wt, cv.BF16)


# ---------------------------------------------------------------------- RoI heads (backward) and their losses
def grad_join_f32(acc, g=None):
    """bf16(g + acc): joins the fp32 RoIAlign-backward accumulator with an (optional) bf16 gradient of the same shape."""
    torch = L.require_cuda()
    assert acc.dtype == torch.float32 and acc.is_contiguous() and (g is None or (g.shape == acc.shape and g.dtype == torch.bfloat16))
    out = torch.empty(acc.shape, dtype=torch.bfloat16, device='cuda')
    L.call('dt_grad_join_f32', L.ptr(g), L.ptr(acc), acc.numel(), L.ptr(out), L.stream_ptr())
    return out


def roi_align_bwd(grad, dfeats, scales, rois, levels, P, sampling_ratio, T=1, k_min=2, n_dev=None):
    """grad [R, T, P, P, C] bf16 -> accumulated into dfeats (list of fp32 [Nimg*T, H_l, W_l, C], finest first, zeroed by the
    caller); the arguments mirror dense_ops.roi_align."""
    torch = L.require_cuda()
    nl = len(dfeats)
    Cc = grad.shape[-1]
    R = rois.shape[0]
    assert grad.dtype == torch.bfloat16 and grad.is_contiguous() and grad.numel() == R * T * P * P * Cc
    fp = (C.c_void_p * nl)(*[f.data_ptr() for f in dfeats])
    Hs = (C.c_int * nl)(*[f.shape[1] for f in dfeats])
    Ws = (C.c_int * nl)(*[f.shape[2] for f in dfeats])
    sc = (C.c_float * nl)(*[float(s) for s in scales])
    for f in dfeats:
        assert f.dtype == torch.float32 and f.is_contiguous() and f.shape[-1] == Cc
    rois = rois.contiguous()
    L.call('dt_roi_align_bwd', L.ptr(grad), fp, Hs, Ws, sc, nl, k_min, Cc, L.ptr(rois), rois.shape[1], L.ptr(n_dev), R, T,
           L.ptr(levels), P, sampling_ratio, L.stream_ptr())


def frcnn_loss_grad(out, labels, targets, inside, outside, C_, totals, scale_cls, scale_box, ld_g, loss=None, accuracy=None):
    """out [rows, ld_o] fp32 (C_ logits | 4C_ deltas) -> grad [rows, ld_g] bf16; loss [2] += (cls, bbox)."""
    torch = L.require_cuda()
    rows, ld_o = out.shape
    grad = torch.empty((rows, ld_g), dtype=torch.bfloat16, device='cuda')
    L.call('dt_frcnn_loss_grad', L.ptr(out), ld_o, L.ptr(labels), L.ptr(targets), L.ptr(inside), L.ptr(outside), rows, C_, L.ptr(totals),
           float(scale_cls), float(scale_box), L.ptr(grad), ld_g, L.ptr(loss), L.ptr(accuracy), L.stream_ptr())
    return grad


def frcnn_tube_loss_grad(out, labels, targets, inside, outside, T, C_, totals, scale_cls, scale_box, ld_g, loss=None, accuracy=None):
    """out [R*T, ld_o] fp32 per RoI-frame (C_ logits | 4C_ deltas) -> grad [R*T, ld_g] bf16 through the tube fold;
    labels [R], targets / weights [R, 4*C_*T]; loss [2] += (cls, bbox)."""
    torch = L.require_cuda()
    rows, ld_o = out.shape
    assert rows % T == 0
    grad = torch.empty((rows, ld_g), dtype=torch.bfloat16, device='cuda')
    L.call('dt_frcnn_tube_loss_grad', L.ptr(out), ld_o, L.ptr(labels), L.ptr(targets), L.ptr(inside), L.ptr(outside), rows // T, T, C_,
           L.ptr(totals), float(scale_cls), float(scale_box), L.ptr(grad), ld_g, L.ptr(loss), L.ptr(accuracy), L.stream_ptr())
    return grad


def rpn_tube_loss_grad(out, A, t, scale_cls, scale_box, ld_g, loss=None, normalizer=None, beta=1.0 / 9.0):
    """out [B, T, H, W, ld_o] fp32 per-frame RPN output; t: dt_rpn_targets dict (labels [B,H,W,A], bbox_targets / inside /
    outside [B,H,W,4TA]) -> grad [B, T, H, W, ld_g] bf16; loss [2] += (cls, bbox).  normalizer: [1] fp32 scratch that
    receives the SigmoidCrossEntropyLoss normaliser max(#labels >= 0, 1e-5)."""
    torch = L.require_cuda()
    B, T, H, W, ld_o = out.shape
    assert out.dtype == torch.float32 and out.is_contiguous()
    if normalizer is None:
        normalizer = torch.empty((1,), dtype=torch.float32, device='cuda')
    grad = torch.empty((B, T, H, W, ld_g), dtype=torch.bfloat16, device='cuda')
    L.call('dt_rpn_tube_loss_grad', L.ptr(out), ld_o, L.ptr(t['labels']), L.ptr(t['bbox_targets']), L.ptr(t['inside']), L.ptr(t['outside']),
           B, T, H, W, A, float(scale_cls), float(scale_box), float(beta), L.ptr(normalizer), L.ptr(grad), ld_g, L.ptr(loss), L.stream_ptr())
    return grad


def spatial_mean_bwd(g, hw, y=None, scale=None, second=False, scale2=None):
    """g [N, C] bf16 (gradient wrt the spatial mean) -> [N, H, W, C] = g / (H*W) * [y > 0] * scale[c]; second=True also returns
    the same masked value times scale2[c] (or unscaled), like bwd_pointwise(second=True)."""
    torch = L.require_cuda()
    N, Cc = g.shape
    H, W = hw
    assert g.dtype == torch.bfloat16 and g.is_contiguous()
    assert y is None or (y.dtype == torch.bfloat16 and y.is_contiguous() and tuple(y.shape) == (N, H, W, Cc))
    out = torch.empty((N, H, W, Cc), dtype=torch.bfloat16, device='cuda')
    out2 = torch.empty_like(out) if second else None
    L.call('dt_spatial_mean_bwd', L.ptr(g), N, H, W, Cc, L.ptr(y), L.ptr(scale), L.ptr(out), L.ptr(scale2), L.ptr(out2), L.stream_ptr())
    return (out, out2) if second else out


def kps_loss_grad(low, K, locations, weights, totals, scale, ld_g, loss=None):
    """low [D, S, S, ld] fp32 (sub-pixel packed kps_score_lowres) -> grad [D, S, S, ld_g] bf16 of the spatial-softmax loss."""
    torch = L.require_cuda()
    D, S, _, ld = low.shape
    grad = L.zeros((D, S, S, ld_g), torch.bfloat16)
    L.call('dt_kps_loss_grad', L.ptr(low), ld, S, K, D, L.ptr(locations), L.ptr(weights), L.ptr(totals), float(scale), L.ptr(grad), ld_g,
           L.ptr(loss), L.stream_ptr())
    return grad


def subpixel_grad_fix(gW, gb, K):
    taps, ldc, Cin = gW.shape
    assert taps == 9
    L.call('dt_subpixel_grad_fix', L.ptr(gW), L.ptr(gb), K, Cin, ldc, L.stream_ptr())
