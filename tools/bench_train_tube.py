#!/usr/bin/env python
"""Time the tube keypoint R-CNN training step (modeling/tube_trainer.py) at the geometry of
configs/video/3d/03_R-18-3D_PTFromCOCO.yaml: the largest training scale (TRAIN.SCALES[-1] 256, MAX_SIZE 333) on 256 x 333
frames, T = 3, BATCH_SIZE_PER_IM 512, RPN_PRE_NMS_TOP_N 2000, 2 clips per GPU, seeded synthetic frames, gt tubes and weights.

    python tools/bench_train_tube.py [--steps 30] [--warmup 5] [--out FILE]

Prints one JSON line: ms/step and clips/s (CUDA events over the timed steps, bracketed by a synchronise), the algorithmic FLOPs
of one step (trainer.step_flops()) and the achieved rate, the losses of the last step, the GPU name and power limit, and a
per-phase split from a separate event-timed pass (trunk forward, targets + proposals, heads forward, heads backward, RPN +
trunk backward, update), plus the backward of the two stride-2 3x3x3 convs (res3_0 / res4_0 branch2a) timed on their own."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def tube_cfg():
    from detectandtrack_b200.core.config import cfg, reset_cfg, assert_and_infer_cfg
    reset_cfg()
    cfg.MODEL.TYPE = 'keypoint_rcnn'
    cfg.MODEL.CONV_BODY = 'ResNet3D.add_ResNet18_conv4_body'
    cfg.MODEL.ROI_HEAD = 'ResNet3D.add_ResNet18_roi_conv5_head'
    cfg.MODEL.NUM_CLASSES = 2
    cfg.MODEL.FASTER_RCNN = True; cfg.MODEL.KEYPOINTS_ON = True; cfg.MODEL.VIDEO_ON = True
    cfg.FAST_RCNN.ROI_XFORM_METHOD = 'RoIAlign'; cfg.FAST_RCNN.ROI_XFORM_RESOLUTION = 7; cfg.FAST_RCNN.ROI_XFORM_SAMPLING_RATIO = 2
    cfg.KRCNN.ROI_KEYPOINTS_HEAD = 'keypoint_rcnn_heads.add_roi_pose_head_v1convX_3d'
    cfg.KRCNN.NUM_STACKED_CONVS = 8; cfg.KRCNN.NUM_KEYPOINTS = 17; cfg.KRCNN.USE_DECONV_OUTPUT = True
    cfg.KRCNN.CONV_HEAD_DIM = 512; cfg.KRCNN.UP_SCALE = 2; cfg.KRCNN.HEATMAP_SIZE = 56
    cfg.KRCNN.ROI_XFORM_RESOLUTION = 14; cfg.KRCNN.ROI_XFORM_SAMPLING_RATIO = 2; cfg.KRCNN.NO_3D_DECONV_TIME_TO_CH = True
    cfg.VIDEO.NUM_FRAMES = 3; cfg.VIDEO.TIME_INTERVAL = 1
    for k in ('BODY', 'HEAD_RPN', 'HEAD_KPS', 'HEAD_DET'):
        cfg.VIDEO.TIME_KERNEL_DIM[k] = 3
    cfg.VIDEO.BODY_HEAD_LINK = ''
    cfg.TRAIN.SCALES = (128, 196, 256); cfg.TRAIN.MAX_SIZE = 333
    cfg.TRAIN.BATCH_SIZE_PER_IM = 512; cfg.TRAIN.RPN_PRE_NMS_TOP_N = 2000; cfg.TRAIN.IMS_PER_BATCH = 2
    cfg.TEST.SCALES = (cfg.TRAIN.SCALES[-1],); cfg.TEST.MAX_SIZE = cfg.TRAIN.MAX_SIZE        # the trainer's blob geometry
    cfg.SOLVER.BASE_LR = 0.001; cfg.SOLVER.WEIGHT_DECAY = 1e-4
    assert_and_infer_cfg()
    return cfg


def gpu_info():
    try:
        r = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().split(',')]
        return dict(gpu=name, power_limit=power, sm_max_clock=clk)
    except Exception as e:
        import torch
        return dict(gpu=torch.cuda.get_device_name(0), power_limit='unavailable (%s)' % type(e).__name__)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--out', default=None, help='also write the JSON line to this file')
    a = ap.parse_args()
    import torch
    import detectandtrack_b200._lib as L
    from detectandtrack_b200.modeling import params as P
    from detectandtrack_b200.modeling.trainer import pack_gt
    from detectandtrack_b200.modeling.tube_trainer import TubeKeypointRcnnTrainer
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from train_net import _synthetic_gt
    assert torch.cuda.is_available(), 'bench_train_tube.py measures on the GPU; there is no CPU fallback'
    cfg = tube_cfg()
    B, T, H, W = cfg.TRAIN.IMS_PER_BATCH, cfg.VIDEO.NUM_FRAMES, 256, 333
    blobs, spec = P.random_blobs(cfg, seed=3)
    tr = TubeKeypointRcnnTrainer(cfg, blobs, spec)
    frames = torch.from_numpy(np.random.RandomState(0).randint(0, 256, (B, T, H, W, 3)).astype(np.uint8)).cuda()
    gt = pack_gt([_synthetic_gt(dict(seed=1000003 * b + 1, height=H, width=W), cfg.KRCNN.NUM_KEYPOINTS, T) for b in range(B)],
                 K=cfg.KRCNN.NUM_KEYPOINTS)
    for _ in range(a.warmup):
        tr.step(frames, gt)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(a.steps):
        l_rpn, l_heads = tr.step(frames, gt)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / a.steps
    flops = tr.step_flops()
    # per-phase split: KeypointRcnnTrainer.step's sequence with an event between the phases
    names = ('trunk_fwd', 'targets_proposals', 'heads_fwd', 'heads_bwd', 'rpn_trunk_bwd', 'update')
    acc = dict((n, 0.0) for n in names)
    for _ in range(a.steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        ev[0].record()
        outs = tr.forward_all(frames); ev[1].record()
        rt, smp = tr.make_targets(outs, gt, B, H, W, cfg.RNG_SEED + tr.iter); ev[2].record()
        tr.forward_heads(smp); ev[3].record()
        L.call('dt_memset', L.ptr(tr.flat_g), 0, tr.flat_g.numel() * 4, L.stream_ptr())
        tr.reducer.reset()
        hg = tr.backward_heads(smp); ev[4].record()
        tr.backward(outs, rt, head_grads=hg, fresh=False); ev[5].record()
        tr.update(); ev[6].record()
        tr.iter += 1
        torch.cuda.synchronize()
        for i, n in enumerate(names):
            acc[n] += ev[i].elapsed_time(ev[i + 1]) / a.steps
    # the two strided 3x3x3 convs' backward (zero-insertion + 4x the minimal MMAs) on the saved activations of the last step
    strided = {}
    for sb in tr.saved['blocks']:
        c = sb['blk']['a']
        if c.stride[1] != 2:
            continue
        gz = torch.randn(tuple(sb['a'].shape), device='cuda').bfloat16()
        c.backward(gz, sb['x'])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            c.backward(gz, sb['x'])
        e1.record()
        torch.cuda.synchronize()
        strided[c.name] = round(e0.elapsed_time(e1) / a.steps, 4)
    l = l_rpn.tolist() + l_heads.tolist()
    res = dict(workload='tube_keypoint_rcnn_train R18-3D T=%d %dx%d clips/gpu=%d BATCH_SIZE_PER_IM=%d RPN_PRE_NMS_TOP_N=%d' % (
                   T, H, W, B, cfg.TRAIN.BATCH_SIZE_PER_IM, cfg.TRAIN.RPN_PRE_NMS_TOP_N),
               steps=a.steps, warmup=a.warmup, ms_per_step=round(ms, 3), clips_per_s=round(B * 1000.0 / ms, 2),
               step_gflop=round(flops / 1e9, 2), achieved_tflops=round(flops / (ms / 1e3) / 1e12, 2),
               phases_ms=dict((k, round(v, 3)) for k, v in acc.items()), strided_conv_bwd_ms=strided,
               losses=dict(zip(('rpn_cls', 'rpn_bbox', 'cls', 'bbox', 'kps'), [round(x, 5) for x in l[:5]])),
               live_rois=float(tr.totals[0]), **gpu_info())
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
