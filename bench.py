#!/usr/bin/env python
"""bench.py — clips/sec of the per-clip detect path (BASELINE.json metric) on N B200s.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --config r50fpn2d | r18tube               (BASELINE.json configs[1] / configs[2])
    python bench.py ... --dump-outputs DIR                    (the last timed step's detections as DIR/*.npy)

Workload (config.workload), default = BASELINE.json configs[3]: 3-D ResNet-50-FPN (T=3, time kernel 3) keypoint
R-CNN inference, 800x1333 frames (blob 800x1344), per-clip data parallel: FPN3D body, BODY_HEAD_LINK slice-center,
2mlp box head, 8-conv keypoint head (the reference's runnable FPN semantics, lib/modeling/FPN3D.py:228), R = 1000
proposals, D <= 100 detections, synthetic uint8 frames, seeded random weights (SURVEY.md §8d).  A step = `--clips`
clips per GPU through ONE captured device step; weak scaling (clips are independent: no data-path collective).

  dtype      the HEADLINE arithmetic is `bf16x3` ([hi | lo] bf16 pair storage, 3 bf16 MMAs per k-block): the fastest
             mode whose end-to-end error against the fp32 reference is <= 1e-3 BY TEST (tests/test_gpu_engine.py,
             tests/test_gpu_parity_e2e.py).  bf16 (fast, ~1e-2) / tf32 are timed beside it as labelled extras.
  value      clips/s with the uint8 frames already resident in HBM (CUDA events, max over ranks)
  e2e        the same metric THROUGH THE REFERENCE-FACING API: core.test.ClipPipeline (what test_engine.test_net
             drives and im_detect_all is the 1-clip form of) fed host numpy clips — loader threads copy them into
             pinned memory, H2D of the frames and D2H of boxes + keypoints + conversion to the reference's per-clip
             containers all inside the timed region
  roofline   tensor-core roofline of the dominant kernel (conv_tc_kernel): algorithmic conv/FC FLOPs of a step (2*MACs
             of the fp32 graph) / summed CUDA-event time of those launches, vs the bf16 peak of MEASURED_PEAKS.json
             (bf16x3 issues bf16 MMAs); `tensor_pipe_frac` counts the 3 MMAs actually issued per product
  cpu_baseline / --impl reference : the torch-fp32 CPU restatement of the reference graph (oracle/, test
             infrastructure) on the host cores, one bounded clip per step
  gpu_standin: the same oracle graph on the B200 through cuDNN 9 (fp32 / TF32 / bf16 autocast, batch 1, host NMS as the
             reference does it) — BASELINE.md §3's stand-in for the reference's Caffe2 + cuDNN 7 build
  tracking   config 1 (tools/compute_tracks.py path): frame pairs / s on the device next to cython_bbox + scipy per pair
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

HEADLINE = 'bf16x3'
WORKLOADS = {
    'r50fpn3d': 'R50-FPN-3D (T=3, tk=3) keypoint R-CNN inference, slice-center + 2-D heads, %dx%d, R=1000, D<=100 (BASELINE.json configs[3])',
    'r50fpn2d': '2-D R50-FPN keypoint R-CNN inference, single %dx%d frames batched, R=1000, D<=100 (BASELINE.json configs[1])',
    'r18tube': '3-D R18-conv4 (T=3, tk=3) tube keypoint R-CNN, res5 RoI head + 3-D keypoint head '
               '(configs/video/3d/03_R-18-3D_PTFromCOCO.yaml), %dx%d, R=1000 tubes, D<=100 (BASELINE.json configs[2])',
}


def bench_cfg(h=800, w=1333, name='r50fpn3d'):
    from detectandtrack_b200.core.config import cfg, reset_cfg, assert_and_infer_cfg
    reset_cfg()
    cfg.MODEL.TYPE = 'keypoint_rcnn'
    cfg.MODEL.NUM_CLASSES = 2
    cfg.MODEL.FASTER_RCNN = True
    cfg.MODEL.KEYPOINTS_ON = True
    cfg.FAST_RCNN.ROI_XFORM_METHOD = 'RoIAlign'; cfg.FAST_RCNN.ROI_XFORM_RESOLUTION = 7
    cfg.FAST_RCNN.ROI_XFORM_SAMPLING_RATIO = 2
    cfg.KRCNN.NUM_STACKED_CONVS = 8; cfg.KRCNN.NUM_KEYPOINTS = 17; cfg.KRCNN.USE_DECONV_OUTPUT = True
    cfg.KRCNN.CONV_HEAD_DIM = 512; cfg.KRCNN.UP_SCALE = 2; cfg.KRCNN.HEATMAP_SIZE = 56
    cfg.KRCNN.ROI_XFORM_RESOLUTION = 14; cfg.KRCNN.ROI_XFORM_SAMPLING_RATIO = 2
    if name == 'r18tube':                   # configs/video/3d/03_R-18-3D_PTFromCOCO.yaml at TEST.SCALES (800,) MAX_SIZE 1333
        cfg.MODEL.CONV_BODY = 'ResNet3D.add_ResNet18_conv4_body'
        cfg.MODEL.ROI_HEAD = 'ResNet3D.add_ResNet18_roi_conv5_head'
        cfg.MODEL.VIDEO_ON = True
        cfg.KRCNN.ROI_KEYPOINTS_HEAD = 'keypoint_rcnn_heads.add_roi_pose_head_v1convX_3d'
        cfg.KRCNN.NO_3D_DECONV_TIME_TO_CH = True
        cfg.VIDEO.NUM_FRAMES = 3; cfg.VIDEO.TIME_INTERVAL = 1; cfg.VIDEO.BODY_HEAD_LINK = ''
        for k in ('BODY', 'HEAD_RPN', 'HEAD_KPS', 'HEAD_DET'):
            cfg.VIDEO.TIME_KERNEL_DIM[k] = 3
    else:
        cfg.MODEL.ROI_HEAD = 'head_builder.add_roi_2mlp_head'
        cfg.KRCNN.ROI_KEYPOINTS_HEAD = 'keypoint_rcnn_heads.add_roi_pose_head_v1convX'
        cfg.FPN.FPN_ON = True; cfg.FPN.MULTILEVEL_ROIS = True; cfg.FPN.MULTILEVEL_RPN = True
        if name == 'r50fpn2d':
            cfg.MODEL.CONV_BODY = 'FPN.add_fpn_ResNet50_conv5_body'
            cfg.MODEL.VIDEO_ON = False
        else:
            cfg.MODEL.CONV_BODY = 'FPN3D.add_fpn_ResNet50_conv5_body'
            cfg.MODEL.VIDEO_ON = True
            cfg.VIDEO.NUM_FRAMES = 3; cfg.VIDEO.TIME_INTERVAL = 1
            for k in ('BODY', 'HEAD_RPN', 'HEAD_KPS', 'HEAD_DET'):
                cfg.VIDEO.TIME_KERNEL_DIM[k] = 3
            cfg.VIDEO.BODY_HEAD_LINK = 'slice-center'; cfg.VIDEO.NUM_FRAMES_MID = 1
    cfg.TEST.SCALES = (min(h, w),); cfg.TEST.MAX_SIZE = max(h, w)
    cfg.TEST.NMS = 0.5; cfg.TEST.RPN_PRE_NMS_TOP_N = 1000; cfg.TEST.RPN_POST_NMS_TOP_N = 1000
    cfg.TEST.COMPETITION_MODE = False
    assert_and_infer_cfg()
    return cfg


def frames_per_clip(cfg):
    return cfg.VIDEO.NUM_FRAMES if cfg.MODEL.VIDEO_ON else 1


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=float(d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1413.7))), src='measured (MEASURED_PEAKS.json, bf16 sustained)')
    return dict(tflops=1400.0, src='fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)')


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.25)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) > 8 and r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 8 and r[2].replace('.', '').isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) > 8:
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def synth_frames(B, T, H, W, seed):
    rng = np.random.RandomState(seed)
    return rng.randint(0, 256, (B, T, H, W, 3)).astype(np.uint8)


# ------------------------------------------------------------------------------ reference / CPU arm
def pick_cpu_threads(torch):
    """Thread count for the CPU arm: the fastest of {32, 64, all} on one mid-sized conv (the port's time moved 5x
    between driver runs with all 128+ hardware threads; a calibrated, stated count keeps the baseline stable)."""
    import torch.nn.functional as F
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (32, 64, cores) if c <= cores} or {cores})
    x = torch.randn(1, 128, 3, 100, 168); w = torch.randn(128, 128, 3, 3, 3)
    best, best_t = cands[-1], None
    for c in cands:
        torch.set_num_threads(c)
        F.conv3d(x, w, None, 1, 1)
        t0 = time.perf_counter()
        F.conv3d(x, w, None, 1, 1)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def reference_clip(cfg, blobs, frames, device='cpu', conv_flags=None):
    """One clip through the torch-fp32 restatement of the reference graph with the reference's host ops (oracle/; TEST
    INFRASTRUCTURE used here only as the measured baseline).  Returns (#detections, #keypoint RoIs)."""
    from oracle import pipeline as opipe
    out = opipe.detect_clip(cfg, blobs, frames[0], device=device, conv_flags=conv_flags)
    nd = out['cls_boxes'].shape[0]
    return nd, (nd if out['keyps'] is not None else 0)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    from detectandtrack_b200.modeling import params as P
    cfg = bench_cfg(args.height, args.width, args.config)
    blobs, _ = P.random_blobs(cfg)
    cores = pick_cpu_threads(torch)
    T = frames_per_clip(cfg)
    frames = synth_frames(1, T, args.height, args.width, 7)
    done = args.steps                       # ONE clip per step
    for _ in range(args.warmup):
        reference_clip(cfg, blobs, frames)
    t0 = time.time()
    for _ in range(done):
        reference_clip(cfg, blobs, frames)
    t_total = time.time() - t0
    v = done / t_total
    line = dict(impl='reference', metric='clips/sec (T=3, 800x1333)', value=v, unit='clips/s', n_gpus=args.gpus,
                steps=done, warmup=args.warmup, ms_per_step=1000.0 * t_total / done, higher_is_better=True, scaling='weak',
                vs_baseline=None, dtype='f32', data='synthetic',
                config=dict(workload=WORKLOADS[args.config] % (args.height, args.width),
                            clips_per_step=1, note='torch-fp32 CPU restatement of the reference graph + reference host ops (oracle/); '
                                                   'the reference Caffe2/cuDNN build cannot be produced here (BASELINE.md §2)'),
                cpu_baseline=dict(value=v, unit='clips/s', cores=cores, kind='port',
                                  sample='%d clip(s), full graph, batch 1, %d torch threads (calibrated)' % (done, cores)),
                e2e=dict(value=v, unit='clips/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# ------------------------------------------------------------------------------ our arm
class ConvMeter(object):
    """CUDA-event timing of every conv_tc launch + its algorithmic FLOPs (2*MACs of the fp32 graph)."""

    def __init__(self, torch):
        self.torch, self.ev, self.flops, self.on, self.meta = torch, [], 0.0, False, []
        self.installed = False

    def reset(self):
        self.ev, self.flops, self.meta = [], 0.0, []

    def install(self):
        if self.installed:
            return
        self.installed = True
        from detectandtrack_b200.ops import conv as cv
        meter, orig = self, cv.conv3d

        def timed(x, w_packed, ksize, *a, **kw):
            if not meter.on:
                return orig(x, w_packed, ksize, *a, **kw)
            e0 = meter.torch.cuda.Event(enable_timing=True); e1 = meter.torch.cuda.Event(enable_timing=True)
            e0.record()
            y = orig(x, w_packed, ksize, *a, **kw)
            e1.record()
            split = kw.get('dtype') in cv.SPLIT_MODES           # [hi | lo] rows: half of the row is the channel count
            cin = kw.get('cin') or (min(x.shape[-1], w_packed.shape[-1]) // (2 if split else 1))
            cout = w_packed.shape[1]
            meter.flops += 2.0 * y.shape[0] * y.shape[1] * y.shape[2] * y.shape[3] * cout * cin * ksize[0] * ksize[1] * ksize[2]
            meter.ev.append((e0, e1))
            meter.meta.append((tuple(x.shape), cin, cout, tuple(ksize), tuple(y.shape)))
            return y
        cv.conv3d = timed
        orig1 = cv.conv1_7x7s2

        def timed1(x_padded, w_packed, hw, *a, **kw):
            if not meter.on:
                return orig1(x_padded, w_packed, hw, *a, **kw)
            e0 = meter.torch.cuda.Event(enable_timing=True); e1 = meter.torch.cuda.Event(enable_timing=True)
            e0.record()
            y = orig1(x_padded, w_packed, hw, *a, **kw)
            e1.record()
            cout = w_packed.shape[1]
            meter.flops += 2.0 * y.shape[0] * y.shape[1] * y.shape[2] * cout * 3 * 49      # algorithmic: Cin = 3, 7x7
            meter.ev.append((e0, e1))
            meter.meta.append((tuple(x_padded.shape), 3, cout, (1, 7, 7), (1,) + tuple(y.shape[:3]) + (cout,)))
            return y
        cv.conv1_7x7s2 = timed1

    def result(self):
        ms = sum(a.elapsed_time(b) for a, b in self.ev)
        return ms, self.flops, len(self.ev)

    def layers(self, nsteps):
        """Per-layer median time over the timed steps (layer = position in the launch sequence)."""
        n = len(self.ev) // nsteps
        rows = []
        for i in range(n):
            ts = sorted(self.ev[s * n + i][0].elapsed_time(self.ev[s * n + i][1]) for s in range(nsteps))
            xs, cin, cout, k, ys = self.meta[i]
            fl = 2.0 * ys[0] * ys[1] * ys[2] * ys[3] * cout * cin * k[0] * k[1] * k[2]
            ms = ts[len(ts) // 2]
            rows.append(dict(i=i, x=list(xs), cin=cin, cout=cout, k=list(k), ms=round(ms, 4), gflop=round(fl / 1e9, 2),
                             tflops=round(fl / ms / 1e9, 1)))
        return rows


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, out, num_classes):
    """What a caller of the captured step receives (engine.gather / ClipPipeline read the same rows), as .npy files:
    det_counts [B, C-1], boxes [sum of counts, 5] and keypoints [sum of class-1 counts, 4, K], clip by clip, then class.
    Beyond DUMP_BYTES, a fixed seeded subset of the clips is written; clip_index lists the clips kept."""
    dets = out['dets'].float().cpu().numpy()                              # [B, C-1, cap, 5]
    B, cap = dets.shape[0], dets.shape[2]
    cnt = np.minimum(out['det_counts'].view(B, num_classes - 1).cpu().numpy(), cap)
    xy = None if out['xy'] is None else out['xy'].float().cpu().numpy().reshape((B, cap) + tuple(out['xy'].shape[1:]))
    per_clip = 8 * (num_classes - 1) + dets[0].nbytes + (0 if xy is None else xy[0].nbytes)
    keep = np.arange(B)
    if B * per_clip > DUMP_BYTES:
        keep = np.sort(np.random.RandomState(0).choice(B, DUMP_BYTES // per_clip, replace=False))
    arrays = dict(clip_index=keep.astype(np.float64), det_counts=cnt[keep].astype(np.float64),
                  boxes=np.concatenate([dets[b, j, :cnt[b, j]] for b in keep for j in range(num_classes - 1)]))
    if xy is not None:
        arrays['keypoints'] = np.concatenate([xy[b, :cnt[b, 0]] for b in keep])
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + '.npy'), a)


def measure_mode(mode, cfg, blobs, args, ctx, full):
    """One arithmetic mode: captured step (ClipPipeline), resident + API end-to-end timing; full: also the launch count,
    the eager roofline pass and (rank 0) clock sampling."""
    import torch
    from detectandtrack_b200.modeling import model_builder
    from detectandtrack_b200.core.test import ClipPipeline
    rank, world, local, barrier, meter = ctx['rank'], ctx['world'], ctx['local'], ctx['barrier'], ctx['meter']
    B, T, H, W = args.clips, frames_per_clip(cfg), args.height, args.width
    model = model_builder.create(cfg.MODEL.TYPE, train=False, blobs=blobs, dtype=mode)
    eng = model.engine
    eng.skip_dead_frames = bool(args.dce)
    host_np = ctx['host_np']
    dev = torch.from_numpy(host_np).cuda()
    flush = ctx['flush']
    res = dict(mode=mode)
    # count our kernel launches of one step (eager)
    if full:
        for _ in range(2):
            eng.detect_static(dev)
        torch.cuda.synchronize()
        ctx['ncalls']['n'] = 0
        eng.detect_static(dev)
        torch.cuda.synchronize()
        res['launches_per_step'] = ctx['ncalls']['n']
    pipe = ClipPipeline(model, B, T, H, W)
    pipe.static_in.copy_(dev)

    def step_resident():
        flush.zero_()                       # L2 flush between iterations (256 MiB > 126 MB L2)
        return pipe.replay()

    for _ in range(max(args.warmup, 3)):
        out = step_resident()
    barrier()
    res['ndet'] = out['det_counts'].view(B, -1)[:, 0].tolist()
    sampler = None
    if full and rank == 0:
        sampler = ClockSampler(local)
        sampler.start()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step_resident()
    e1.record()
    barrier()
    res['ms'] = e0.elapsed_time(e1)
    if full and args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, eng.spec.num_classes)
    # ---- end to end through the API: host numpy clips -> ClipPipeline.run -> the reference's per-clip containers ----
    got = []

    def fill(i, dst):
        np.copyto(dst, host_np[i % B])          # pageable host clip -> pinned staging (loader thread)

    def on_result(i, cls_boxes, cls_segms, cls_keyps):
        got.append((i, cls_boxes[1].shape[0], 0 if cls_keyps is None else len(cls_keyps[1])))
    pipe.pre_step = flush.zero_
    pipe.run(2 * B, fill, on_result)                                         # warm-up of the pipelined loop
    barrier()
    del got[:]
    f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
    f0.record()
    pipe.run(args.steps * B, fill, on_result)          # returns when the last clip's containers have been delivered
    f1.record()
    barrier()
    res['ms_e2e'] = f0.elapsed_time(f1)
    assert len(got) == args.steps * B and [g[0] for g in got] == list(range(args.steps * B))
    res['h2d'], res['d2h'] = pipe.h2d_bytes, pipe.d2h_bytes
    pipe.pre_step = None
    if full:
        # ---- roofline pass: the same step, eager, with CUDA events around every conv_tc launch -------
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.detect_static(dev)
        enqueue_s = time.perf_counter() - t0
        torch.cuda.synchronize()
        delay_cycles = int(max(40e6, 1.6 * enqueue_s * 2.0e9))
        meter.reset()
        meter.on = True
        barrier()
        for _ in range(args.steps):
            flush.zero_()
            # keep the GPU busy while the CPU enqueues the step, so the per-conv events bracket kernel
            # execution back to back instead of CPU launch latency (eager mode is launch-bound)
            torch.cuda._sleep(delay_cycles)
            eng.detect_static(dev)
        barrier()
        meter.on = False
        res['conv_ms'], res['conv_flops'], res['conv_n'] = meter.result()
        if args.layers and rank == 0:
            os.makedirs(os.path.join(ROOT, 'gpurun_out'), exist_ok=True)
            json.dump(meter.layers(args.steps), open(os.path.join(ROOT, 'gpurun_out', 'conv_layers.json'), 'w'), indent=0)
        res['clocks'] = sampler.stop() if sampler is not None else None
        # ---- extra (not the headline): the same step with dead-frame elimination ----------------------
        if not args.dce and not args.no_extras and world == 1 and eng.spec.fpn and eng.spec.link == 'slice-center' and T > 1:
            eng.skip_dead_frames = True
            for _ in range(2):
                eng.detect_static(dev)
            s2, run2 = eng.capture(B, T, H, W)
            s2.copy_(dev)
            for _ in range(3):
                flush.zero_(); run2()
            barrier()
            h0 = torch.cuda.Event(enable_timing=True); h1 = torch.cuda.Event(enable_timing=True)
            h0.record()
            for _ in range(args.steps):
                flush.zero_(); run2()
            h1.record()
            barrier()
            res['dce'] = dict(value=B * args.steps / (h0.elapsed_time(h1) / 1000.0), unit='clips/s',
                              note='dead-frame elimination of the post-hoc FPN convs; identical outputs; NOT the headline')
            eng.skip_dead_frames = False
            del s2, run2
    del pipe, model, eng, dev, out
    gc.collect()
    torch.cuda.empty_cache()
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist
    from detectandtrack_b200 import _lib as L
    from detectandtrack_b200.modeling import params as P
    rank = int(os.environ.get('RANK', '0')); world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    cfg = bench_cfg(args.height, args.width, args.config)
    blobs, _ = P.random_blobs(cfg)
    B, T, H, W = args.clips, frames_per_clip(cfg), args.height, args.width
    meter = ConvMeter(torch)
    meter.install()
    ncalls = {'n': 0}
    orig_call = L.call

    def counting_call(name, *a):
        if name not in ('dt_memset', 'dt_nms_workspace_bytes', 'dt_rpn_workspace_bytes', 'dt_conv_plan'):     # kernels only
            ncalls['n'] += 3 if name == 'dt_nms_batched' else 1
        return orig_call(name, *a)
    L.call = counting_call
    for m in ('box_ops', 'rpn_ops', 'dense_ops', 'conv'):
        mod = __import__('detectandtrack_b200.ops.' + m, fromlist=['x'])
        mod.L.call = counting_call

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = dict(rank=rank, world=world, local=local, barrier=barrier, meter=meter, ncalls=ncalls,
               host_np=synth_frames(B, T, H, W, 100 + rank), flush=torch.empty(256 << 20, dtype=torch.uint8, device='cuda'))
    head_mode = HEADLINE if args.dtype == 'auto' else args.dtype
    head = measure_mode(head_mode, cfg, blobs, args, ctx, full=True)
    extras = []
    if args.dtype == 'auto' and world == 1 and not args.no_extras:
        for m in ('bf16x3h', 'bf16', 'tf32'):
            try:
                extras.append(measure_mode(m, cfg, blobs, args, ctx, full=False))
            except Exception as e:                               # an extra must never cost the headline
                extras.append(dict(mode=m, error=str(e)[:200]))
    t = torch.tensor([head['ms'], head['ms_e2e'], head['conv_ms']], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e, conv_ms_max = t.tolist()
    # BASELINE.json configs[4] next to the inference headline, on the same box and process group: the keypoint R-CNN training
    # step with its NCCL gradient all-reduce (every rank takes part; a labelled extra of this line, `bench.py --train` alone
    # prints it as its own line)
    training = None
    if args.dtype == 'auto' and args.config == 'r50fpn3d' and not args.no_extras and not args.dce:
        try:
            import gc
            gc.collect(); torch.cuda.empty_cache()
            tl = _train_measure(args, rank, world, local)
            if tl is not None:
                training = dict(metric=tl['metric'], value=tl['value'], unit=tl['unit'], ms_per_step=tl['ms_per_step'], n_gpus=world,
                                dtype='bf16', e2e=tl['e2e'], roofline=dict(achieved=tl['roofline']['achieved'], frac=tl['roofline']['frac'],
                                                                          unit='TFLOP/s', note=tl['roofline']['note']),
                                allreduce_bytes_per_step=tl['config']['allreduce_bytes_per_step'], allreduce=tl['config']['allreduce'],
                                losses=dict(rpn=tl['config']['loss_rpn'], cls=tl['config'].get('loss_cls'), bbox=tl['config'].get('loss_bbox'),
                                            kps=tl['config'].get('loss_kps')), workload=tl['config']['workload'])
        except Exception as e:                                   # an extra must never cost the headline
            training = dict(error=str(e)[:300])
    if rank == 0:
        pk = peaks()
        value = world * B * args.steps / (ms / 1000.0)
        e2e = world * B * args.steps / (ms_e2e / 1000.0)
        conv_ms, conv_flops, conv_n = head['conv_ms'], head['conv_flops'], head['conv_n']
        achieved = conv_flops / (conv_ms / 1000.0) / 1e12
        mma_factor = 3.0 if head_mode in ('bf16x3', 'tf32x3', 'bf16x3h') else 1.0
        parity = {'bf16x3': '<= 1e-3 end to end vs the fp32 oracle BY TEST (tests/test_gpu_parity_e2e.py, test_gpu_engine.py: <= 5e-4)',
                  'bf16x3h': 'bf16x3 with the four post-hoc FPN convs as one fp16 MMA per product: heat maps ~1e-3 (no margin), 1 of 100 detections differs at 800x1333 (tests/test_gpu_parity_e2e.py) - NOT a parity mode, labelled extra only',
                  'tf32x3': '<= 1e-3 end to end by test (<= 5e-4)', 'tf32': '~1.5e-3 end to end (outside 1e-3)',
                  'bf16': '~1e-2 end to end (outside 1e-3): labelled extra only'}
        tr = conv_traffic(B, head_mode)
        line = dict(metric='clips/sec (T=3, 800x1333)', value=value, unit='clips/s', n_gpus=world, steps=args.steps,
                    warmup=max(args.warmup, 3), ms_per_step=ms / args.steps, higher_is_better=True, scaling='weak',
                    vs_baseline=None, dtype=head_mode, data='synthetic',
                    config=dict(workload=WORKLOADS[args.config] % (H, W),
                                arithmetic='%s: %s' % (head_mode, parity[head_mode]),
                                clips_per_step_per_gpu=B, parallelism='clips sharded over %d GPU(s), no collective' % world,
                                detections_per_clip=head['ndet'], l2='flushed between iterations (256 MiB fill)',
                                dead_frame_elimination=bool(args.dce),
                                conv_gflop_per_clip=conv_flops / 1e9 / (B * args.steps), conv_launches_per_step=conv_n // args.steps,
                                conv_share_of_step=conv_ms / ms, cuda_graph=True,
                                e2e_path='core.test.ClipPipeline.run (the loop of test_engine.test_net; im_detect_all is its 1-clip form): '
                                         'host numpy clips -> loader threads -> pinned -> H2D -> captured step -> D2H -> per-clip cls_boxes / cls_keyps',
                                roofline_pass='same step run eagerly behind a GPU-side delay, CUDA events around every conv_tc launch'),
                    e2e=dict(value=e2e, unit='clips/s', h2d_bytes_per_step=head['h2d'], d2h_bytes_per_step=head['d2h']),
                    gpu_launches=head['launches_per_step'] * args.steps, clocks=head['clocks'],
                    roofline=dict(bound='tensor', kernel='conv_tc_kernel (all conv/FC launches of the step)', achieved=achieved,
                                  peak=pk['tflops'], unit='TFLOP/s', frac=achieved / pk['tflops'],
                                  tensor_pipe_frac=mma_factor * achieved / pk['tflops'],
                                  note='achieved = algorithmic FLOPs (2*MACs of the fp32 graph) / conv_tc time; %s issues %d bf16 MMA(s) per '
                                       'product, so the tensor pipe runs at tensor_pipe_frac of the measured bf16 peak' % (head_mode, int(mma_factor)),
                                  traffic=tr[0], traffic_source=tr[1], peak_source=pk['src']))
        if head.get('dce') is not None:
            line['config']['with_dead_frame_elimination'] = head['dce']
        if extras:
            line['config']['other_modes'] = [
                dict(dtype=x['mode'], parity=parity.get(x['mode']), error=x.get('error')) if 'error' in x else
                dict(dtype=x['mode'], parity=parity.get(x['mode']), value=B * args.steps / (x['ms'] / 1000.0),
                     e2e=B * args.steps / (x['ms_e2e'] / 1000.0), unit='clips/s') for x in extras]
        if training is not None:
            line['training'] = training
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline(cfg, blobs, args)
        if world == 1 and not args.no_extras:
            try:
                line['gpu_standin'] = gpu_standin(cfg, blobs, args)
            except Exception as e:
                line['gpu_standin'] = dict(error=str(e)[:300])
            try:
                line['tracking'] = tracking_leg()
            except Exception as e:
                line['tracking'] = dict(error=str(e)[:300])
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def synth_gt(B, H, W, seed, G=4, K=17):
    """Synthetic ground truth of a training clip batch: G persons per clip (boxes 80..320 px, 17 joints inside, ~2/3 visible)."""
    rng = np.random.RandomState(seed)
    entries = []
    for _ in range(B):
        w = rng.uniform(80, 240, G); h = rng.uniform(160, 320, G)
        x1 = rng.uniform(0, W - 1 - w); y1 = rng.uniform(0, H - 1 - h)
        boxes = np.stack([x1, y1, x1 + w, y1 + h], 1).astype(np.float32)
        kps = np.zeros((G, 3, K), np.int32)
        for i in range(G):
            kps[i, 0] = rng.randint(int(boxes[i, 0]), int(boxes[i, 2]) + 1, K)
            kps[i, 1] = rng.randint(int(boxes[i, 1]), int(boxes[i, 3]) + 1, K)
            kps[i, 2] = rng.randint(0, 3, K)
        entries.append(dict(boxes=boxes, gt_keypoints=kps))
    return entries


def _train_measure(args, rank, world, local):
    """One measured training leg on an initialised process group (all ranks call it); returns the JSON line as a dict on rank 0,
    None elsewhere.  `--train`: BASELINE.json configs[4], the keypoint R-CNN training step (modeling/trainer.KeypointRcnnTrainer): frozen
    stem, bf16 forward of res3..res5 + FPN3D + RPN + both RoI heads, ALL targets generated on the device (RPN anchor targets,
    training proposals, RoI sampling, keypoint labels), losses, backward (dgrad / tcgen05 wgrad / RoIAlign backward), the
    bucketed NCCL gradient all-reduce overlapped with the backward pass, fused SGD.  TRAIN.IMS_PER_BATCH = 2 clips per GPU.
    `--train-trunk` times the RPN-model trunk alone (MODEL.TYPE rpn) under its own metric name."""
    import torch
    import torch.distributed as dist
    from detectandtrack_b200.modeling import params as P
    from detectandtrack_b200.modeling.trainer import RpnTrainer, KeypointRcnnTrainer, pack_gt
    nsteps = args.steps
    cfg = bench_cfg(args.height, args.width, 'r50fpn3d')
    cfg.TRAIN.BATCH_SIZE_PER_IM = 512; cfg.TRAIN.RPN_PRE_NMS_TOP_N = 2000      # the shipped keypoint yamls (configs/video/2d_best)
    blobs, spec = P.random_blobs(cfg)
    B, T, H, W = cfg.TRAIN.IMS_PER_BATCH, 3, args.height, args.width
    full = not getattr(args, 'train_trunk', False)
    frames_h = torch.from_numpy(synth_frames(B, T, H, W, 100 + rank)).pin_memory()
    frames = frames_h.cuda()
    if full:
        tr = KeypointRcnnTrainer(cfg, blobs, spec, world=world, buckets=args.buckets)
        gt = pack_gt(synth_gt(B, H, W, 7 + rank))
        step = lambda fr: tr.step(fr, gt)
    else:
        tr = RpnTrainer(cfg, blobs, spec, world=world, buckets=args.buckets)
        targets = tr.synthetic_targets(B, H, W, seed=rank)
        step = lambda fr: (tr.step(fr, targets), None)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            out = fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), out, sampler.stop() if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step(frames)
    ms, (loss, lh), clocks = timed(lambda: step(frames), nsteps)
    # e2e: the step a training loop makes — pinned host frames -> device every step, losses read back every step
    loss_h = torch.empty(6, dtype=torch.float32).pin_memory()

    def e2e_step():
        fr = frames_h.cuda(non_blocking=True)
        l, h = step(fr)
        loss_h[:2].copy_(l, non_blocking=True)
        if h is not None:
            loss_h[2:6].copy_(h, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return l, h
    e2e_step()
    ms2, _, _ = timed(e2e_step, nsteps)
    if rank == 0:
        nparam = int(tr.flat_g.numel())
        what = ('keypoint R-CNN training step (RPN + Fast R-CNN + keypoint heads, device-side targets)' if full else
                'RPN-model trunk (res3..res5 + FPN3D + RPN heads/losses)')
        cfgd = dict(workload='BASELINE.json configs[4]: R50-FPN-3D (T=3) %s, %d clips/GPU, bf16 forward/backward, fp32 master weights%s'
                             % ('keypoint R-CNN, BATCH_SIZE_PER_IM 512, RPN 2000/level -> 2000, 4 gt persons/clip' if full else 'trunk only', B,
                                '' if full else '; RoI heads / target generators NOT included (partial training step)'),
                    trainable_params=nparam, allreduce_bytes_per_step=4 * nparam if world > 1 else 0,
                    allreduce='NCCL SUM, %d buckets issued as their wgrads are enqueued (overlaps the backward pass)' % len(tr.bucket_ends),
                    loss_rpn=[float(x) for x in loss.cpu().tolist()], eager_launches=True)
        if full:
            l4 = [float(x) for x in lh.cpu().tolist()]
            cfgd.update(loss_cls=l4[0], loss_bbox=l4[1], loss_kps=l4[2], sampled_rois=float(tr.totals[0]), keypoint_targets=float(tr.totals[1]))
        pk = peaks()
        fl = tr.step_flops()
        tf = fl / (ms / nsteps / 1000.0) / 1e12
        peak = pk['tflops']
        roof = dict(bound='tensor', kernel='conv_tc_kernel (forward + dgrad) + wgrad_nhwc_kernel, whole step', achieved=tf, peak=peak, unit='TFLOP/s',
                    frac=tf / peak, traffic=None,
                    note='achieved = algorithmic FLOPs of the trainable convs / FCs (forward + filter gradient + input gradient, %.1f GFLOP per '
                         'step of %d clips; frozen stem excluded) / WHOLE step time incl. targets, losses, joins, all-reduce and SGD' % (fl / 1e9, B),
                    peak_source=pk['src'])
        line = dict(metric='training clips/sec, %s, T=3, %dx%d' % (what, H, W),
                    value=world * B * nsteps / (ms / 1000.0), unit='clips/s', n_gpus=world, steps=nsteps,
                    warmup=max(args.warmup, 3), ms_per_step=ms / nsteps, higher_is_better=True, scaling='weak', vs_baseline=None,
                    dtype='bf16', data='synthetic',
                    e2e=dict(value=world * B * nsteps / (ms2 / 1000.0), unit='clips/s', h2d_bytes_per_step=int(frames_h.numel()),
                             d2h_bytes_per_step=24), roofline=roof, config=cfgd, clocks=clocks)
        return line
    return None


def run_train(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0')); world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    line = _train_measure(args, rank, world, local)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def conv_traffic(clips_per_step, mode):
    """DRAM bytes moved by the conv_tc launches of ONE step (the unit `roofline.achieved` is computed over), from the
    committed ncu capture of this same bench command (profiles/conv_dram_<round>_<mode>.json, tools/ncu_conv_traffic.py);
    scaled if the step size differs.  Returns (bytes or None, provenance string)."""
    for name in ('conv_dram_r02_%s.json' % mode, 'conv_dram_r01.json' if mode == 'bf16' else ''):
        path = os.path.join(ROOT, 'profiles', name)
        if name and os.path.exists(path):
            d = json.load(open(path))
            return (d['dram_bytes'] * clips_per_step / float(d['clips_per_step']),
                    'dram__bytes_read.sum + dram__bytes_write.sum over the %d conv_tc launches of one step, ncu, %d clips/step '
                    '(profiles/%s)' % (d['launches'], d['clips_per_step'], name))
    return None, 'no ncu capture committed for this mode'


def cpu_baseline(cfg, blobs, args):
    import torch
    cores = pick_cpu_threads(torch)
    frames = synth_frames(1, frames_per_clip(cfg), args.height, args.width, 7)
    t0 = time.time()
    nd, nk = reference_clip(cfg, blobs, frames)
    dt = time.time() - t0
    return dict(value=1.0 / dt, unit='clips/s', cores=cores, kind='port',
                sample='1 clip, full graph incl. host NMS/decoding, torch fp32 CPU (oracle/), %d torch threads (calibrated), %d detections' % (cores, nd))


def gpu_standin(cfg, blobs, args):
    """The oracle graph on the SAME B200 through cuDNN 9 with the reference's execution shape: batch 1, the proposal /
    NMS / decode steps on the host with a D2H sync each (lib/core/test.py:158-252, lib/ops/generate_proposals.py).
    It is the stand-in BASELINE.md §3 names for the reference's Caffe2 + cuDNN 7 build, never the reference itself."""
    import torch
    frames = synth_frames(1, frames_per_clip(cfg), args.height, args.width, 7)
    out = {}
    for tag, flags in (('fp32', dict(tf32=False, autocast=None)), ('tf32', dict(tf32=True, autocast=None)),
                       ('bf16_autocast', dict(tf32=True, autocast='bf16'))):
        reference_clip(cfg, blobs, frames, device='cuda', conv_flags=flags)          # warm-up (cuDNN autotune, allocator)
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            nd, _ = reference_clip(cfg, blobs, frames, device='cuda', conv_flags=flags)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        out[tag] = dict(value=1.0 / sorted(ts)[1], unit='clips/s', detections=nd)
    out['note'] = ('torch 2.11 + cuDNN 9 on this B200, batch 1, host proposals/NMS/keypoint decode like the reference '
                   '(oracle/pipeline.py on cuda); stand-in for the reference Caffe2 + cuDNN 7 path, which cannot be built here')
    torch.backends.cudnn.allow_tf32 = True
    gc.collect(); torch.cuda.empty_cache()
    return out


def tracking_leg(videos=64, frames=30, dets=100, cpu_videos=4):
    """BASELINE.json configs[0] / SURVEY §8(d) config 1: V videos x 30 frames x 100 detections linked by
    core.tracking_engine (cost + assignment for every frame pair + id scan on the device, host lists in and out), next
    to what the reference pays per pair on the CPU: compiled cython_bbox.bbox_overlaps + scipy.linear_sum_assignment."""
    import torch
    import scipy.optimize
    from detectandtrack_b200.core import tracking_engine as te
    from detectandtrack_b200.core.config import cfg
    from oracle import tracking as ot
    try:
        from oracle._ref import cython_bbox as ref_bbox
        overlaps, kind = ref_bbox.bbox_overlaps, 'reference cython_bbox (oracle/_ref) + scipy %s' % scipy.__version__
    except Exception:
        from oracle import boxes as obox
        overlaps, kind = obox.bbox_overlaps, 'oracle numpy bbox_overlaps + scipy %s' % scipy.__version__
    saved = (cfg.TRACKING.DISTANCE_METRICS, cfg.TRACKING.DISTANCE_METRIC_WTS, cfg.TRACKING.BIPARTITE_MATCHING_ALGO)
    cfg.TRACKING.DISTANCE_METRICS = ('bbox-overlap',); cfg.TRACKING.DISTANCE_METRIC_WTS = (1.0,)
    cfg.TRACKING.BIPARTITE_MATCHING_ALGO = 'hungarian'
    try:
        out = {}
        for tag, tie_free in (('tie_heavy', False), ('tie_free', True)):
            rng = np.random.default_rng(3)
            vids = [ot.synth_video(rng, n_frames=frames, n_dets=dets) for _ in range(videos)]
            if tie_free:                          # sub-pixel jitter: no exactly-tied costs (SURVEY §8d second variant)
                vids = [[(f + np.concatenate([rng.uniform(0, 1e-2, (f.shape[0], 4)), np.zeros((f.shape[0], 1))], 1)).astype(np.float32)
                         for f in v] for v in vids]
            te._tracks_for_videos(vids[:2])
            torch.cuda.synchronize()
            ts = []
            for _ in range(5):
                t0 = time.perf_counter()
                got = te._tracks_for_videos(vids)
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            t_gpu = sorted(ts)[len(ts) // 2]
            t0 = time.perf_counter()
            npairs = 0
            for v in vids[:cpu_videos]:
                for a, b in zip(v[:-1], v[1:]):
                    C = (np.float32(1) - overlaps(np.ascontiguousarray(a[:, :4]), np.ascontiguousarray(b[:, :4]))).astype(np.float32)
                    scipy.optimize.linear_sum_assignment(C)
                    npairs += 1
            t_cpu = time.perf_counter() - t0
            ref = [ot.compute_tracks_video(v, solver='scipy') for v in vids[:2]]
            out[tag] = dict(value=videos * (frames - 1) / t_gpu, unit='frame-pairs/s',
                            cpu=dict(value=npairs / t_cpu, unit='frame-pairs/s', cores=1, kind=kind),
                            ids_identical_to_cpu=bool(all(ref[i] == got[i] for i in range(2))))
        out['config'] = '%d videos x %d frames x %d detections, host lists in / id lists out (H2D + 3 launches + D2H per call)' % (videos, frames, dets)
        return out
    finally:
        cfg.TRACKING.DISTANCE_METRICS, cfg.TRACKING.DISTANCE_METRIC_WTS, cfg.TRACKING.BIPARTITE_MATCHING_ALGO = saved


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='timed steps (default 10; --impl reference: 2)')
    ap.add_argument('--warmup', type=int, default=None, help='warm-up steps (default 3; --impl reference: 1)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--dtype', default='auto', choices=['auto', 'bf16', 'tf32', 'tf32x3', 'bf16x3', 'bf16x3h'],
                    help='auto: headline bf16x3 (the parity mode) + bf16 / tf32 as labelled extras')
    ap.add_argument('--config', default='r50fpn3d', choices=sorted(WORKLOADS))
    ap.add_argument('--clips', type=int, default=8, help='clips per GPU per step')
    ap.add_argument('--height', type=int, default=800)
    ap.add_argument('--width', type=int, default=1333)
    ap.add_argument('--dce', type=int, default=0, help='1: compute only the consumed centre frame of the post-hoc FPN convs')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the extra modes, the cuDNN stand-in and the tracking leg')
    ap.add_argument('--layers', action='store_true', help='dump per-conv timings to gpurun_out/conv_layers.json')
    ap.add_argument('--graph', type=int, default=1, help='(kept for old command lines; the step is always a captured graph)')
    ap.add_argument('--train', action='store_true', help='BASELINE.json configs[4]: keypoint R-CNN training step with NCCL gradient all-reduce (see run_train)')
    ap.add_argument('--train-trunk', action='store_true', help='with --train: the RPN-model trunk alone')
    ap.add_argument('--buckets', type=int, default=4, help='--train: gradient all-reduce buckets')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write the detections of the last step '
                    '(det_counts, boxes, keypoints, clip_index) as DIR/<name>.npy')
    a = ap.parse_args()
    reference = a.impl == 'reference' and not a.train
    if a.steps is None:
        a.steps = 2 if reference else 10
    if a.warmup is None:
        a.warmup = 1 if reference else 3
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if a.dump_outputs and (a.train or reference):
        ap.error('--dump-outputs applies to the inference benchmark (--impl ours, no --train)')
    if a.train:
        run_train(a)
    elif reference:
        run_reference(a)
    else:
        run_ours(a)
