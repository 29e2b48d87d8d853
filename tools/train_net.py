#!/usr/bin/env python
"""Training entry point with the reference's command line (tools/train_net.py:40-66,129-229):

    python tools/train_net.py --cfg X.yaml [KEY VALUE ...]                       (one GPU)
    python -m torch.distributed.run --nproc-per-node N tools/train_net.py ...     (one process per GPU, NCCL all-reduce)

The loop: minibatch (TRAIN.IMS_PER_BATCH clips + their ground truth) -> trainer.step (forward, device-side targets, losses,
backward, bucketed gradient all-reduce, SGD with the lr of lib/utils/lr_policy) -> smoothed loss log every 20 iterations.
TRAIN.DATASET 'synthetic_VxF[_HxW]' draws seeded frames and persons (person tubes for the 3-D tube models); any other name is a
JSON list of roidb entries with 'image', 'height', 'width', 'boxes', 'gt_keypoints' (the fields lib/datasets/json_dataset.py
builds; [G,4T] boxes and [G,3,K*T] keypoints for tube models).
"""
import argparse
import logging
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from detectandtrack_b200.core.config import cfg, cfg_from_file, cfg_from_list, assert_and_infer_cfg  # noqa: E402


def parse_args():
    p = argparse.ArgumentParser(description='Train a network with Detectron')
    p.add_argument('--cfg', dest='cfg_file', help='Config file for training (and optionally testing)', default=None, type=str)
    p.add_argument('--multi-gpu-testing', dest='multi_gpu_testing', action='store_true')
    p.add_argument('--skip-test', dest='skip_test', action='store_true')
    p.add_argument('opts', help='See core/config.py for all options', default=None, nargs=argparse.REMAINDER)
    return p.parse_args()


def find_resume_point(output_dir):
    """tools/train_net.py:79-105 (CLUSTER.AUTO_RESUME): ('final', path) if model_final.pkl exists, else (start_iter, path) of
    the newest model_iter<N>.pkl (training resumes at N + 1), else (0, None)."""
    import re
    final = os.path.join(output_dir, 'model_final.pkl')
    if os.path.exists(final):
        return 'final', final
    start, path = 0, None
    for f in os.listdir(output_dir) if os.path.isdir(output_dir) else []:
        m = re.findall(r'(?<=model_iter)\d+(?=\.pkl)', f)
        if m and int(m[0]) + 1 > start:
            start, path = int(m[0]) + 1, os.path.join(output_dir, f)
    return start, path


def _synthetic_gt(entry, K, T=1):
    """Seeded persons of a synthetic clip.  T > 1: tubes, boxes [G,4T] with every frame's box the T == 1 draw shifted by up to
    3 % of the frame size (clipped to the frame), keypoints [G,3,K*T] drawn per frame inside that frame's box."""
    rng = np.random.RandomState(entry['seed'] % (2 ** 31))
    H, W, G = entry['height'], entry['width'], 3
    w = rng.uniform(0.08, 0.2, G) * W; h = rng.uniform(0.2, 0.4, G) * H
    x1 = rng.uniform(0, W - 1 - w); y1 = rng.uniform(0, H - 1 - h)
    boxes = np.stack([x1, y1, x1 + w, y1 + h], 1).astype(np.float32)
    if T == 1:
        kps = np.zeros((G, 3, K), np.int32)
        for i in range(G):
            kps[i, 0] = rng.randint(int(boxes[i, 0]), int(boxes[i, 2]) + 1, K)
            kps[i, 1] = rng.randint(int(boxes[i, 1]), int(boxes[i, 3]) + 1, K)
            kps[i, 2] = rng.randint(0, 3, K)
        return dict(boxes=boxes, gt_keypoints=kps)
    shift = rng.uniform(-0.03, 0.03, (G, T, 2)) * np.array([W, H])
    tubes = np.zeros((G, T, 4), np.float32)
    for t in range(T):
        b = boxes + np.tile(shift[:, t], 2)
        tubes[:, t] = np.clip(b, 0, [W - 1, H - 1, W - 1, H - 1])
    kps = np.zeros((G, 3, K * T), np.int32)
    for i in range(G):
        for t in range(T):
            bx = tubes[i, t]
            kps[i, 0, t * K:(t + 1) * K] = rng.randint(int(bx[0]), int(bx[2]) + 1, K)
            kps[i, 1, t * K:(t + 1) * K] = rng.randint(int(bx[1]), int(bx[3]) + 1, K)
            kps[i, 2, t * K:(t + 1) * K] = rng.randint(0, 3, K)
    return dict(boxes=tubes.reshape(G, 4 * T), gt_keypoints=kps)


def train_model():
    import torch
    import torch.distributed as dist
    from detectandtrack_b200.core import test_engine as te
    from detectandtrack_b200.modeling import model_builder
    from detectandtrack_b200.modeling.trainer import pack_gt
    from detectandtrack_b200.utils.lr_policy import get_lr_at_iter
    log = logging.getLogger('train_net')
    rank, world = int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1'))
    torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', '0')))
    if world > 1:
        dist.init_process_group('nccl')
    cfg.TEST.SCALES, cfg.TEST.MAX_SIZE = (cfg.TRAIN.SCALES[-1],), cfg.TRAIN.MAX_SIZE       # one training scale per run (the blob geometry)
    from detectandtrack_b200.core.config import get_output_dir
    from detectandtrack_b200.modeling import params as P
    import yaml
    output_dir = get_output_dir(training=True)
    start_iter, resume = find_resume_point(output_dir) if (cfg.CLUSTER.ON_CLUSTER and cfg.CLUSTER.AUTO_RESUME) else (0, None)
    if start_iter == 'final':
        log.info('model_final.pkl exists; no need to train!')
        return []
    if resume:
        cfg.TRAIN.WEIGHTS = resume
        log.info('========> Resuming from checkpoint %s with start iter %d', resume, start_iter)
    model = model_builder.create(cfg.MODEL.TYPE, train=True)
    snap_every = max(1, int(cfg.TRAIN.SNAPSHOT_ITERS / max(1, cfg.NUM_GPUS)))

    def snapshot(name):
        path = os.path.join(output_dir, name)
        P.save_weights_file(model.export_blobs(model.blobs0), yaml.dump({'MODEL': {'TYPE': cfg.MODEL.TYPE, 'CONV_BODY': cfg.MODEL.CONV_BODY}}), path)
        log.info('Wrote %s', path)
    roidb = te.get_dataset(cfg.TRAIN.DATASET).get_roidb(gt=True)
    K = cfg.KRCNN.NUM_KEYPOINTS
    T = P.GraphSpec(cfg).T_head                    # frames per gt tube (1: boxes)
    B = cfg.TRAIN.IMS_PER_BATCH
    order = np.random.RandomState(cfg.RNG_SEED).permutation(len(roidb))
    smooth = []
    for it in range(start_iter, cfg.SOLVER.MAX_ITER):
        idx = [order[(it * world * B + rank * B + j) % len(order)] for j in range(B)]
        entries = [roidb[i] for i in idx]
        frames = torch.from_numpy(np.stack([np.stack(te.read_image_video(e)) for e in entries])).cuda()
        gts = [(_synthetic_gt(e, K, T) if e.get('synthetic') else dict(boxes=np.asarray(e['boxes'], np.float32),
                                                                    gt_keypoints=np.asarray(e['gt_keypoints'], np.int32))) for e in entries]
        model.lr = float(get_lr_at_iter(it))
        l_rpn, l_heads = model.step(frames, pack_gt(gts, K=K))
        if rank == 0 and (it + 1) % snap_every == 0 and it > start_iter:      # :208-212
            snapshot('model_iter{}.pkl'.format(it))
        if it % 20 == 0 or it == cfg.SOLVER.MAX_ITER - 1:
            l = l_rpn.tolist() + l_heads.tolist()
            smooth.append(sum(l[:5]))
            if rank == 0:
                log.info('iter %d lr %.6f loss %.4f (rpn_cls %.4f rpn_bbox %.4f cls %.4f bbox %.4f kps %.4f) accuracy_cls %.3f', it, model.lr,
                         sum(l[:5]), l[0], l[1], l[2], l[3], l[4], l[5] / max(1.0, float(model.totals[0])))
    if rank == 0:             # tools/train_net.py:214-218: the final weights under the reference's blob names (TEST.WEIGHTS of test_net.py)
        snapshot('model_final.pkl')
    if world > 1:
        dist.destroy_process_group()
    return smooth


if __name__ == '__main__':
    logging.basicConfig(level=logging.INFO, format='%(levelname)s %(filename)s:%(lineno)4d: %(message)s', stream=sys.stdout)
    args = parse_args()
    if args.cfg_file is not None:
        cfg_from_file(args.cfg_file)
    if args.opts:
        cfg_from_list(args.opts)
    assert_and_infer_cfg()
    train_model()
