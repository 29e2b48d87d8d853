"""GPU: the tube keypoint R-CNN training step (modeling/tube_trainer.py; configs/video/3d/03_R-18-3D_PTFromCOCO.yaml
semantics) — its new kernels against torch autograd in fp32 on the same bf16 inputs, one whole step against torch-fp32
autograd of the oracle's tube graph (oracle/net.py) fed with the device's own targets, and the reference CLI.

Loss semantics pinned by the oracle losses below: the tube RPN's SigmoidCrossEntropyLoss runs with Detectron's default
normalize=1 (sum over labels >= 0 divided by max(#labels >= 0, 1e-5), scale 1 / NUM_GPUS), SmoothL1Loss beta 1/9 scaled by
1 / NUM_GPUS / T / batch; the box head's SmoothL1Loss by 1 / NUM_GPUS / T; the keypoint loss is not divided by T."""
import os
import pickle
import re
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import net as onet
from oracle.graph import OracleSpec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _smooth_l1(d, beta):
    ad = d.abs()
    return __import__('torch').where(ad < beta, 0.5 * d * d / beta, ad - 0.5 * beta)


# ---------------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize('all_ignored', [False, True])
def test_rpn_tube_loss_grad_vs_autograd(all_ignored):
    import torch
    import torch.nn.functional as F
    from detectandtrack_b200.ops import train_ops as to
    B, T, H, W, A, ld = 2, 3, 5, 6, 15, 80
    g = torch.Generator().manual_seed(0)
    o = torch.randn((B, T, H, W, ld), generator=g) * 2
    labels = torch.randint(-1, 2, (B, H, W, A), generator=g, dtype=torch.int32)
    labels[1] = -1                                                             # an image with every label ignored
    if all_ignored:
        labels[:] = -1
    tg = torch.randn((B, H, W, 4 * T * A), generator=g) * 0.3
    iw = (torch.rand((B, H, W, 4 * T * A), generator=g) > 0.5).float()
    ow = torch.rand((B, H, W, 4 * T * A), generator=g) / 64
    s_cls, s_box = 0.5, 0.5 / T / B
    t = dict(labels=labels.cuda(), bbox_targets=tg.cuda(), inside=iw.cuda(), outside=ow.cuda())
    loss = torch.zeros(2, device='cuda')
    norm = torch.zeros(1, device='cuda')
    grad = to.rpn_tube_loss_grad(o.cuda(), A, t, s_cls, s_box, ld, loss=loss, normalizer=norm)
    torch.cuda.synchronize()
    x = o.clone().requires_grad_(True)
    lg = x[..., :A].mean(dim=1)                                                # TimePool avg -> [B, H, W, A]
    m = labels >= 0
    cnt = max(float(m.sum()), 1e-5)
    lc = s_cls * F.binary_cross_entropy_with_logits(lg[m], labels[m].float(), reduction='sum') / cnt
    dl = x[..., A:5 * A].reshape(B, T, H, W, A, 4).permute(0, 2, 3, 4, 1, 5).reshape(B, H, W, 4 * T * A)   # a*4T + t*4 + k
    lb = s_box * (ow * _smooth_l1(iw * (dl - tg), 1.0 / 9.0)).sum()
    (lc + lb).backward()
    assert float(norm) == pytest.approx(max(float(m.sum()), 1e-5))
    got = loss.cpu()
    assert abs(float(got[0]) - lc.item()) <= 1e-4 * abs(lc.item()) + 1e-7, (got, lc.item())
    assert abs(float(got[1]) - lb.item()) <= 1e-4 * abs(lb.item()) + 1e-7, (got, lb.item())
    gd = grad.float().cpu()
    assert torch.all(gd[..., 5 * A:] == 0) and torch.isfinite(gd).all()
    assert _rel(gd[..., :A], x.grad[..., :A]) <= 8e-3 if not all_ignored else torch.all(gd[..., :A] == 0)
    assert _rel(gd[..., A:5 * A], x.grad[..., A:5 * A]) <= 8e-3


def test_frcnn_tube_loss_grad_vs_autograd_and_t1_equals_2d():
    import torch
    import torch.nn.functional as F
    from detectandtrack_b200.ops import train_ops as to
    R, T, C, ld = 40, 3, 2, 16
    g = torch.Generator().manual_seed(1)
    o = torch.randn((R * T, ld), generator=g)
    labels = torch.randint(0, C, (R,), generator=g, dtype=torch.int32)
    labels[-8:] = -1                                                           # padding rows
    tg = torch.randn((R, 4 * C * T), generator=g) * 0.5
    iw = (torch.rand((R, 4 * C * T), generator=g) > 0.3).float()
    ow = iw.clone()
    live = labels >= 0
    N = float(live.sum())
    totals = torch.tensor([N, 1.0], device='cuda')
    loss, acc = torch.zeros(2, device='cuda'), torch.zeros(1, device='cuda')
    grad = to.frcnn_tube_loss_grad(o.cuda(), labels.cuda(), tg.cuda(), iw.cuda(), ow.cuda(), T, C, totals, 0.5, 0.5 / T, ld,
                                   loss=loss, accuracy=acc)
    torch.cuda.synchronize()
    x = o.clone().requires_grad_(True)
    xv = x.view(R, T, ld)
    cls = xv[..., :C].mean(dim=1)
    bb = xv[..., C:5 * C].reshape(R, T, C, 4).permute(0, 2, 1, 3).reshape(R, 4 * C * T)        # c*4T + t*4 + k
    l_cls = 0.5 * F.cross_entropy(cls[live], labels[live].long(), reduction='sum') / N
    l_box = (0.5 / T) * (ow[live] * _smooth_l1(iw[live] * (bb[live] - tg[live]), 1.0)).sum() / N
    (l_cls + l_box).backward()
    got = loss.cpu()
    assert abs(float(got[0]) - float(l_cls)) <= 1e-5 * float(l_cls) and abs(float(got[1]) - float(l_box)) <= 1e-5 * float(l_box)
    assert int(acc) == int((cls[live].argmax(1) == labels[live].long()).sum())
    gd = grad.float().cpu()
    assert torch.all(gd.view(R, T, ld)[~live] == 0) and torch.all(gd[:, 5 * C:] == 0)
    assert _rel(gd, x.grad) <= 5e-3
    # T = 1 is the 2-D head: bit-identical to dt_frcnn_loss_grad
    tg1, iw1 = tg[:, :4 * C].contiguous().cuda(), iw[:, :4 * C].contiguous().cuda()
    o1 = o[:R].contiguous().cuda()
    l1, l2 = torch.zeros(2, device='cuda'), torch.zeros(2, device='cuda')
    a1, a2 = torch.zeros(1, device='cuda'), torch.zeros(1, device='cuda')
    g1 = to.frcnn_loss_grad(o1, labels.cuda(), tg1, iw1, iw1, C, totals, 0.5, 0.5, ld, loss=l1, accuracy=a1)
    g2 = to.frcnn_tube_loss_grad(o1, labels.cuda(), tg1, iw1, iw1, 1, C, totals, 0.5, 0.5, ld, loss=l2, accuracy=a2)
    assert torch.equal(g1, g2) and torch.equal(l1, l2) and torch.equal(a1, a2)


def test_spatial_mean_bwd_fused():
    import torch
    from detectandtrack_b200.ops import train_ops as to
    N, H, W, C = 21, 7, 7, 64
    g = torch.Generator(device='cuda').manual_seed(2)
    gm = torch.randn((N, C), generator=g, device='cuda').bfloat16()
    y = torch.randn((N, H, W, C), generator=g, device='cuda').bfloat16()
    s1 = torch.rand(C, generator=g, device='cuda') + 0.5
    s2 = torch.rand(C, generator=g, device='cuda') + 0.5
    out, out2 = to.spatial_mean_bwd(gm, (H, W), y, s1, second=True, scale2=s2)
    base = (gm.float() / (H * W))[:, None, None, :].expand(N, H, W, C) * (y.float() > 0)
    assert _rel(out.float(), base * s1) <= 4e-3 and _rel(out2.float(), base * s2) <= 4e-3
    plain = to.spatial_mean_bwd(gm, (H, W))
    assert _rel(plain.float(), (gm.float() / (H * W))[:, None, None, :].expand(N, H, W, C)) <= 4e-3


@pytest.mark.parametrize('hw', [(8, 10), (9, 11)])
def test_strided_3x3x3_conv_gradients_vs_conv3d(hw):
    """TrainConv's stride-(1,2,2) 3x3x3 backward (zero-inserted gradient + stride-1 dgrad / wgrad) against F.conv3d autograd."""
    import torch
    import torch.nn.functional as F
    from detectandtrack_b200.modeling.trainer import TrainConv
    H, W = hw
    Cin, Cout, N, T = 32, 64, 2, 3
    rng = np.random.RandomState(3)
    w = (rng.randn(Cout, Cin, 3, 3, 3) * 0.05).astype(np.float32)
    c = TrainConv(torch, w, bias=np.zeros(Cout, np.float32), stride=(1, 2, 2))
    c.g = torch.zeros_like(c.w); c.bias_g = torch.zeros_like(c.bias)
    x = torch.randn((N, T, H, W, Cin), device='cuda').bfloat16()
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    gz = torch.randn((N, T, Ho, Wo, Cout), device='cuda').bfloat16()
    dx, _ = c.backward(gz, x)
    torch.cuda.synchronize()
    xr = x.float().cpu().permute(0, 4, 1, 2, 3).contiguous().requires_grad_(True)
    wr = torch.from_numpy(w).bfloat16().float().requires_grad_(True)
    y = F.conv3d(xr, wr, None, (1, 2, 2), (1, 1, 1))
    assert tuple(y.shape[2:]) == (T, Ho, Wo)
    y.backward(gz.float().cpu().permute(0, 4, 1, 2, 3))
    assert _rel(dx.float().cpu().permute(0, 4, 1, 2, 3), xr.grad) <= 1e-2
    dW = c.g.view(3, 3, 3, Cout, Cin).permute(3, 4, 0, 1, 2).cpu()
    assert _rel(dW, wr.grad) <= 2e-3
    assert _rel(c.bias_g.cpu(), gz.float().sum(dim=(0, 1, 2, 3)).cpu()) <= 1e-4


def test_roi_align_bwd_tube_vs_torchvision():
    import torch
    from detectandtrack_b200.ops import train_ops as to
    B, C, T, H, W, R, P = 2, 32, 3, 12, 14, 10, 7
    rng = np.random.RandomState(4)
    feat = torch.from_numpy(rng.randn(B, C, T, H, W).astype(np.float32)).requires_grad_(True)
    x1 = rng.uniform(0, 150, R); y1 = rng.uniform(0, 120, R)
    b0 = np.stack([x1, y1, x1 + rng.uniform(8, 80, R), y1 + rng.uniform(8, 60, R)], 1)
    rois = np.hstack([rng.randint(0, B, (R, 1))] + [b0 + rng.normal(0, 3, (R, 4)) * (t > 0) for t in range(T)]).astype(np.float32)
    out = onet.roi_features_tube(feat, 1 / 16., rois, P, 2)                     # (R, C, T, P, P)
    gout = torch.from_numpy(rng.randn(*out.shape).astype(np.float32)).bfloat16().float()
    out.backward(gout)
    dfe = torch.zeros((B * T, H, W, C), device='cuda')
    to.roi_align_bwd(gout.permute(0, 2, 3, 4, 1).contiguous().cuda().bfloat16(), [dfe], [1 / 16.], torch.from_numpy(rois).cuda(), None, P, 2,
                     T=T)
    ref = feat.grad.permute(0, 2, 3, 4, 1).reshape(B * T, H, W, C)
    assert _rel(dfe.cpu(), ref) <= 1e-5


# ---------------------------------------------------------------------------------------------------- whole step
def _cfg():
    from test_gpu_engine_tube import _cfg as tube_cfg
    cfg = tube_cfg()
    cfg.TEST.SCALES = (96,); cfg.TEST.MAX_SIZE = 128
    cfg.TRAIN.BATCH_SIZE_PER_IM = 32; cfg.TRAIN.RPN_PRE_NMS_TOP_N = 300; cfg.TRAIN.RPN_POST_NMS_TOP_N = 200
    cfg.TRAIN.RPN_BATCH_SIZE_PER_IM = 64
    cfg.KRCNN.CONV_HEAD_DIM = 64
    return cfg


def _tube_gt(rng, T=3, K=17):
    entries = []
    for b in range(2):
        g = 2 + b
        x1 = rng.uniform(0, 60, g); y1 = rng.uniform(0, 40, g)
        base = np.stack([x1, y1, x1 + rng.uniform(30, 60, g), y1 + rng.uniform(30, 50, g)], 1)
        tubes = np.concatenate([np.clip(base + rng.normal(0, 2, (g, 4)) * (t > 0), 0, [127, 95, 127, 95]) for t in range(T)], 1)
        kps = np.zeros((g, 3, K * T), np.int32)
        for i in range(g):
            for t in range(T):
                bx = tubes[i, 4 * t:4 * t + 4]
                kps[i, 0, t * K:(t + 1) * K] = rng.randint(int(bx[0]), int(bx[2]) + 1, K)
                kps[i, 1, t * K:(t + 1) * K] = rng.randint(int(bx[1]), int(bx[3]) + 1, K)
                kps[i, 2, t * K:(t + 1) * K] = rng.randint(0, 3, K)
        entries.append(dict(boxes=tubes.astype(np.float32), gt_keypoints=kps))
    return entries


def _oracle_tube_step(cfg, blobs, frames, rt, smp, T, world=1):
    """The tube keypoint R-CNN loss in torch fp32 on the CPU, teacher-forced with the device's targets."""
    import torch
    import torch.nn.functional as F
    spec = OracleSpec(cfg)
    tb = {k: torch.from_numpy(np.ascontiguousarray(v)).clone() for k, v in blobs.items()}
    pref = ('res3', 'res4', 'res5', 'conv_rpn', 'rpn_', 'cls_score', 'bbox_pred', 'conv_fcn', 'kps_score_lowres')
    train = [k for k in tb if (k.startswith(pref) and not k.endswith(('_bn_s', '_bn_b')))]
    for k in train:
        tb[k].requires_grad_(True)
    means = np.asarray(cfg.PIXEL_MEANS, np.float32).reshape(1, 1, 1, 1, 3)
    data = torch.from_numpy(frames.astype(np.float32) - means).permute(0, 4, 1, 2, 3).contiguous()
    feat = onet.conv_body(tb, spec, data)[spec.stage_blobs[-1]]                 # (B, C, T, h, w)
    B = frames.shape[0]
    lg, dl = onet.rpn_heads_3d(tb, spec, feat)
    lab = torch.from_numpy(rt['labels']).permute(0, 3, 1, 2)
    m = lab >= 0
    lc = F.binary_cross_entropy_with_logits(lg[m], lab[m].float(), reduction='sum') / max(float(m.sum()), 1e-5) / world
    tg, iw, ow = (torch.from_numpy(rt[k]).permute(0, 3, 1, 2) for k in ('bbox_targets', 'inside', 'outside'))
    lb = (ow * _smooth_l1(iw * (dl - tg), 1.0 / 9.0)).sum() / world / T / B
    live = smp['labels'].reshape(-1) >= 0
    N = float(live.sum())
    rois = smp['rois'].reshape(-1, 4 * T + 1)[live]
    labels = torch.from_numpy(smp['labels'].reshape(-1)[live].astype(np.int64))
    rf = onet.roi_features_tube(feat, 1 / 16., rois, cfg.FAST_RCNN.ROI_XFORM_RESOLUTION, cfg.FAST_RCNN.ROI_XFORM_SAMPLING_RATIO)
    cls, bb = onet.box_head_conv5_3d(tb, rf)
    l_cls = F.cross_entropy(cls, labels, reduction='sum') / N / world
    C4 = smp['bbox_targets'].shape[-1]
    tg, iw, ow = (torch.from_numpy(smp[k].reshape(-1, C4)[live]) for k in ('bbox_targets', 'inside', 'outside'))
    l_box = (ow * _smooth_l1(iw * (bb - tg), 1.0)).sum() / N / world / T
    K = cfg.KRCNN.NUM_KEYPOINTS
    kl = np.zeros(smp['kp_rois'].shape[:2], bool)
    for b in range(kl.shape[0]):
        kl[b, :smp['kp_counts'][b]] = True
    kl = kl.reshape(-1)
    krois = smp['kp_rois'].reshape(-1, 4 * T + 1)[kl]
    kf = onet.roi_features_tube(feat, 1 / 16., krois, cfg.KRCNN.ROI_XFORM_RESOLUTION, cfg.KRCNN.ROI_XFORM_SAMPLING_RATIO)
    up = onet.keypoint_head_3d(tb, kf, cfg.KRCNN.NUM_STACKED_CONVS)             # (D, T*K, 56, 56), channel t*K + k
    lp = F.log_softmax(up.reshape(up.shape[0] * T * K, -1), dim=1)
    loc = torch.from_numpy(smp['kp_locations'].reshape(-1, K * T)[kl].reshape(-1).astype(np.int64))
    w = torch.from_numpy(smp['kp_weights'].reshape(-1, K * T)[kl].reshape(-1))
    l_kps = (-(lp[torch.arange(lp.shape[0]), loc]) * w).sum() / w.sum() * cfg.KRCNN.LOSS_WEIGHT / world
    (lc + lb + l_cls + l_box + l_kps).backward()
    return [float(v) for v in (lc, lb, l_cls, l_box, l_kps)], {k: tb[k].grad for k in train}


def test_tube_keypoint_rcnn_training_step_vs_autograd():
    import torch
    import detectandtrack_b200._lib as L
    from test_gpu_engine_tube import _cfg as reset
    from detectandtrack_b200.modeling import params as P, model_builder
    from detectandtrack_b200.modeling.trainer import pack_gt
    from detectandtrack_b200.modeling.tube_trainer import TubeKeypointRcnnTrainer
    cfg = _cfg()
    try:
        blobs, spec = P.random_blobs(cfg, seed=3)
        rng = np.random.RandomState(0)
        T = spec.T_head
        frames = rng.randint(0, 256, (2, T, 96, 128, 3)).astype(np.uint8)
        gt = pack_gt(_tube_gt(rng, T))
        tr = model_builder.create('keypoint_rcnn', train=True, blobs=blobs)
        assert isinstance(tr, TubeKeypointRcnnTrainer)
        tr.lr, tr.wd = 0.01, 1e-4
        exp = tr.export_blobs(blobs)                                             # an exact round trip under the reference's names
        assert set(exp) == set(blobs)
        for k in blobs:
            assert exp[k].shape == blobs[k].shape and np.array_equal(exp[k], blobs[k]), k
        fr = torch.from_numpy(frames).cuda()
        outs = tr.forward_all(fr)
        rt, smp = tr.make_targets(outs, gt, 2, 96, 128, seed=5)
        tr.forward_heads(smp)
        L.call('dt_memset', L.ptr(tr.flat_g), 0, tr.flat_g.numel() * 4, L.stream_ptr())
        tr.reducer.reset()
        hg = tr.backward_heads(smp)
        loss = tr.backward(outs, rt, head_grads=hg, fresh=False).cpu().numpy()
        lh = tr.loss_heads.cpu().numpy()
        assert smp['counts'].cpu().numpy().min() > 8 and int(smp['kp_counts'].sum()) > 0 and float(tr.totals[1]) > 0
        rt_np = {k: v.cpu().numpy() for k, v in rt[0].items()}
        smp_np = {k: v.cpu().numpy() for k, v in smp.items()}
        ref_l, grads = _oracle_tube_step(cfg, blobs, frames, rt_np, smp_np, T)
        got_l = [loss[0], loss[1], lh[0], lh[1], lh[2]]
        print('losses (device, oracle)', list(zip(got_l, ref_l)))
        for name, a, b in zip(('rpn_cls', 'rpn_bbox', 'cls', 'bbox', 'kps'), got_l, ref_l):
            assert abs(a - b) <= 3e-2 * abs(b) + 1e-6, (name, a, b)

        def dev_grad(c):
            kT, kH, kW = c.k
            return c.g.view(kT, kH, kW, c.cout, c.cin).permute(3, 4, 0, 1, 2).cpu()

        bad, errs = [], {}

        def check(name, got, ref, tol=0.25):
            ref = ref.reshape(got.shape)
            err = (got - ref).abs().max().item() / max(ref.abs().max().item(), 1e-30)
            cos = float((got.flatten() * ref.flatten()).sum() / (got.norm() * ref.norm() + 1e-30))
            errs[name] = (round(err, 4), round(cos, 5))
            if err > tol or cos < 0.985:
                bad.append((name, round(err, 4), round(cos, 5)))

        named = {c.name: c for c in tr.convs if hasattr(c, 'name')}
        for n in ('conv_fcn1', 'conv_fcn8', 'res5_0_branch2a', 'res5_0_branch1', 'res5_1_branch2b', 'conv_rpn', 'res4_1_branch2b',
                  'res4_0_branch2a', 'res3_0_branch2a', 'res3_0_branch1'):
            check(n, dev_grad(named[n]), grads[n + '_w'])
        K, C_, A = tr.K, tr.C_, tr.A
        g3 = dev_grad(tr.kps_lowres)[:, :, 0]                                   # sub-pixel filters -> ConvTranspose taps
        gwt = torch.zeros_like(grads['kps_score_lowres_w'])
        for py in range(2):
            for px in range(2):
                for dy in (-1, 0, 1):
                    for dx in (-1, 0, 1):
                        ky, kx = py + 1 - 2 * dy, px + 1 - 2 * dx
                        if 0 <= ky <= 3 and 0 <= kx <= 3:
                            gwt[:, :, ky, kx] = g3[(py * 2 + px) * K:(py * 2 + px + 1) * K, :, dy + 1, dx + 1].t()
        check('kps_score_lowres', gwt, grads['kps_score_lowres_w'])
        gcb = dev_grad(tr.cls_bbox)[:5 * C_, :, 0, 0, 0]
        check('cls_score_1', gcb[:C_], grads['cls_score_1_w']); check('bbox_pred_1', gcb[C_:], grads['bbox_pred_1_w'])
        gro = dev_grad(tr.rpn_out)[:5 * A, :, 0, 0, 0]
        check('rpn_cls_logits_1', gro[:A], grads['rpn_cls_logits_1_w']); check('rpn_bbox_pred_1', gro[A:], grads['rpn_bbox_pred_1_w'])
        print('grad (max-norm rel err, cosine) per layer', errs)
        assert not bad, bad
        # one whole step() runs end to end and moves the weights
        w0 = tr.cls_bbox.w.clone(), tr.stages[0][0]['a'].w.clone()
        l1, l2 = tr.step(fr, gt)
        torch.cuda.synchronize()
        assert torch.isfinite(l1).all() and torch.isfinite(l2).all()
        assert not torch.equal(w0[0], tr.cls_bbox.w) and not torch.equal(w0[1], tr.stages[0][0]['a'].w)
        assert tr.step_flops() > 0
    finally:
        reset()


# ---------------------------------------------------------------------------------------------------- CLI
TUBE_YAML = '''
MODEL:
  TYPE: keypoint_rcnn
  CONV_BODY: ResNet3D.add_ResNet18_conv4_body
  ROI_HEAD: ResNet3D.add_ResNet18_roi_conv5_head
  NUM_CLASSES: 2
  FASTER_RCNN: True
  KEYPOINTS_ON: True
  VIDEO_ON: True
FAST_RCNN:
  ROI_XFORM_METHOD: RoIAlign
  ROI_XFORM_RESOLUTION: 7
  ROI_XFORM_SAMPLING_RATIO: 2
KRCNN:
  ROI_KEYPOINTS_HEAD: keypoint_rcnn_heads.add_roi_pose_head_v1convX_3d
  NUM_STACKED_CONVS: 8
  NUM_KEYPOINTS: 17
  USE_DECONV_OUTPUT: True
  CONV_HEAD_DIM: 128
  UP_SCALE: 2
  HEATMAP_SIZE: 56
  ROI_XFORM_RESOLUTION: 14
  ROI_XFORM_SAMPLING_RATIO: 2
  NO_3D_DECONV_TIME_TO_CH: True
VIDEO:
  NUM_FRAMES: 3
  TIME_INTERVAL: 1
  TIME_KERNEL_DIM: 3
  BODY_HEAD_LINK: ''
TEST:
  DATASET: synthetic_2x3_96x128
  WEIGHTS: random
  SCALES: (96,)
  MAX_SIZE: 128
  NMS: 0.5
  RPN_PRE_NMS_TOP_N: 1000
  RPN_POST_NMS_TOP_N: 300
  COMPETITION_MODE: False
TRAIN:
  DATASET: synthetic_1x2_96x128
  SCALES: (96,)
  MAX_SIZE: 128
  IMS_PER_BATCH: 2
  BATCH_SIZE_PER_IM: 64
  RPN_BATCH_SIZE_PER_IM: 64
  RPN_PRE_NMS_TOP_N: 300
  RPN_POST_NMS_TOP_N: 200
SOLVER:
  BASE_LR: 0.0003
  LR_POLICY: steps_with_decay
  STEPS: [0, 30]
  MAX_ITER: 61
  WARM_UP_ITERS: 5
  WEIGHT_DECAY: 0.0001
NUM_GPUS: 1
'''


def test_train_net_tube_loss_falls_and_test_net_loads_it(tmp_path):
    cfg = tmp_path / 'cfg.yaml'
    cfg.write_text(TUBE_YAML)
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'train_net.py'), '--cfg', str(cfg), 'OUTPUT_DIR', str(tmp_path / 'out'),
                        'TRAIN.DATASET', 'synthetic_1x2_96x128', 'SOLVER.MAX_ITER', '61'], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    losses = [float(m.group(1)) for m in re.finditer(r'iter \d+ lr [\d.]+ loss ([\d.]+)', r.stdout)]
    print('tube train_net losses', losses)
    assert len(losses) == 4 and all(np.isfinite(losses)), r.stdout[-2000:]
    assert losses[-1] < losses[0], losses
    snap = os.path.join(str(tmp_path / 'out'), 'train', 'synthetic_1x2_96x128', 'keypoint_rcnn', 'model_final.pkl')
    w = pickle.load(open(snap, 'rb'))
    assert w['blobs']['rpn_bbox_pred_1_w'].shape == (48, 256, 1, 1, 1) and w['blobs']['res4_0_branch2a_w'].shape == (256, 128, 3, 3, 3)
    r2 = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'test_net.py'), '--cfg', str(cfg), 'OUTPUT_DIR', str(tmp_path / 'out2'),
                         'TEST.WEIGHTS', snap], env=env, capture_output=True, text=True, timeout=600)
    assert r2.returncode == 0, r2.stdout[-2000:] + r2.stderr[-2000:]
    assert os.path.exists(os.path.join(str(tmp_path / 'out2'), 'test', 'synthetic_2x3_96x128', 'keypoint_rcnn', 'detections.pkl'))
