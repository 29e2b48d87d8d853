"""Data-parallel training step on the device (BASELINE.json configs[4]; reference: tools/train_net.py:129-229,
lib/modeling/model_builder.py:908-985 build_data_parallel_model / add_parameter_update_ops).

Implemented graph: the reference's RPN training model (``MODEL.TYPE rpn``, model_builder.py ``rpn`` + FPN.add_fpn_rpn_outputs
+ FPN.add_fpn_rpn_losses, lib/modeling/FPN.py:205-321) on the FPN / FPN3D ResNet-50/101/152 bodies: conv1 / pool1 / res2
frozen (freeze_at=2, ResNet3D.py:273-274; AffineChannel parameters frozen everywhere), res3..res5 + FPN + RPN heads
trained: forward in bf16 (fp32 accumulate), backward =
    dgrad   dt_conv3d with the flipped / transposed filter (+ dt_scatter_stride2 for the stride-2 1x1 convs)
    wgrad   dt_wgrad on channel-major planes (tcgen05, split-K)
    joins   dt_bwd_pointwise (Relu / Sum / AffineChannelNd gradients), dt_upsample_add_bwd (FPN top-down), dt_bias_grad
    losses  dt_rpn_loss_grad per level (SigmoidCrossEntropyLoss + SmoothL1Loss)
then a bucketed gradient SUM all-reduce over NCCL issued per bucket as soon as its filter gradients are enqueued
(overlapping the rest of the backward pass; losses carry 1/NUM_GPUS like the reference, model_builder.py:484) and the fused
MomentumSGDUpdate on fp32 master weights that re-emits the bf16 forward and dgrad filters.

KeypointRcnnTrainer is config 5 proper (``MODEL.TYPE keypoint_rcnn``, FASTER_RCNN end to end): the trunk above plus, per step
and all on the device,
    targets    dt_rpn_targets (lib/roi_data/rpn.py), proposals with the TRAIN settings (GenerateProposals + collect),
               dt_sample_rois (json_dataset.add_proposals + lib/roi_data/fast_rcnn.py + keypoint_rcnn.py)
    box head   RoIAlign 7x7 -> fc6 -> fc7 -> (cls_score | bbox_pred), SoftmaxWithLoss + SmoothL1Loss (dt_frcnn_loss_grad)
    kps head   RoIAlign 14x14 -> 8 x conv3x3 -> sub-pixel deconv, spatial SoftmaxWithLoss through the fixed bilinear 2x
               upsampling (dt_kps_loss_grad)
    backward   the FC / conv layers through the same dgrad / wgrad kernels (an FC is a 1x1 conv over the RoI axis),
               dt_roi_align_bwd into fp32 per-level accumulators that join the RPN's feature gradients.

The single-level 3-D bodies with tube heads (the R18-3D yaml) train through tube_trainer.TubeKeypointRcnnTrainer."""
import os

import numpy as np

from .. import _lib as L
from ..ops import conv as cv, dense_ops, train_ops as to, rpn_ops, box_ops, target_ops
from . import params as P
from .engine import DetectionEngine
from .generate_anchors import generate_anchors


WGRAD_PLANES = os.environ.get('DT_WGRAD_PLANES', '0') == '1'


def plan_buckets(counts, nbuckets):
    """counts: parameter counts in BACKWARD order -> (cumulative ends per parameter, bucket end offsets).  Buckets hold
    ~equal parameter counts and are cut at parameter boundaries, so a bucket is complete as soon as the gradient of its
    last parameter has been enqueued."""
    bounds, off = [], 0
    for n in counts:
        off += int(n)
        bounds.append(off)
    total = off
    ends, target = [], total / float(max(1, nbuckets))
    for b in bounds:
        if b >= target * (len(ends) + 1) or b == total:
            if not ends or b > ends[-1]:
                ends.append(b)
    return bounds, ends


class BucketReducer(object):
    """Gradient SUM all-reduce of a flat buffer in buckets, each launched (async, on the process group's own stream) as soon
    as the producer says the buffer is complete up to an offset — the data-parallel exchange of
    lib/modeling/model_builder.py:922-942 (one NCCLAllreduce per parameter there), overlapped with the backward pass."""

    def __init__(self, flat, bucket_ends, world):
        self.flat, self.ends, self.world = flat, list(bucket_ends), world
        self.reset()

    def reset(self):
        self.next, self.pending = 0, []

    def ready(self, upto):
        if self.world <= 1:
            return
        import torch.distributed as dist
        while self.next < len(self.ends) and self.ends[self.next] <= upto:
            lo = self.ends[self.next - 1] if self.next else 0
            self.pending.append(dist.all_reduce(self.flat[lo:self.ends[self.next]], op=dist.ReduceOp.SUM, async_op=True))
            self.next += 1

    def wait(self):
        for w in self.pending:
            w.wait()
        assert self.world <= 1 or self.next == len(self.ends), 'a gradient bucket was never marked ready'
        self.pending = []


class TrainConv(object):
    """One trainable conv: packed fp32 master filter [taps, Cout, Cin], momentum, gradient (a view into the trainer's
    flat gradient buffer), the bf16 forward / dgrad filters, and either a frozen AffineChannel (scale, bias) or a
    trainable bias."""

    def __init__(self, torch, w, scale=None, shift=None, bias=None, stride=(1, 1, 1), relu=False):
        w = torch.from_numpy(np.ascontiguousarray(w)).float()
        if w.dim() == 2:                                  # FC layer: a 1x1x1 conv over the RoI axis
            w = w[:, :, None, None, None]
        if w.dim() == 4:
            w = w[:, :, None]
        self.k = tuple(w.shape[2:])
        self.pad = tuple(x // 2 for x in self.k)
        self.stride, self.relu = stride, relu
        self.cout, self.cin = w.shape[0], w.shape[1]
        self.cout_live = self.cout                        # output channels that are not zero padding (set by the builder)
        self._accumulate = 0                              # 1: the conv runs several times per step (RPN heads: once per level)
        self.taps = self.k[0] * self.k[1] * self.k[2]
        self.w = w.permute(2, 3, 4, 0, 1).reshape(self.taps, self.cout, self.cin).contiguous().cuda()
        self.m = torch.zeros_like(self.w)
        self.g = None                                     # assigned by the trainer (view into the flat buffer)
        self.w_fwd = self.w.to(torch.bfloat16)
        self.w_dg = torch.empty((self.taps, self.cin, self.cout), dtype=torch.bfloat16, device='cuda')
        self.w_dg.copy_(to.pack_dgrad_weight(w))
        f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda() if a is not None else None
        self.scale, self.shift = f32(scale), f32(shift)
        self.bias = f32(bias)                             # trainable (FPN / RPN convs); None for AffineChannel convs
        self.bias_m = torch.zeros_like(self.bias) if self.bias is not None else None
        self.bias_g = None

    def nparams(self):
        return self.w.numel() + (self.bias.numel() if self.bias is not None else 0)

    def forward(self, x, residual=None, res_mode=0, out_f32=False, out=None, time_major=False):
        N, T, H, W, _ = x.shape                                  # algorithmic MACs of this launch (the roofline's numerator)
        self.macs = (N * T * ((H + self.stride[1] - 1) // self.stride[1]) * ((W + self.stride[2] - 1) // self.stride[2]) *
                     self.cout_live * self.cin * self.taps) + getattr(self, 'macs', 0) * self._accumulate
        return cv.conv3d(x, self.w_fwd, self.k, self.stride, self.pad, self.scale, self.shift if self.bias is None else self.bias,
                         residual, res_mode, self.relu, out_f32=out_f32, dtype=cv.BF16, out=out, time_major=time_major)

    def backward(self, gz, x, x_planes=None, need_dx=True):
        """gz: gradient wrt the conv's raw output (after the pointwise joins), x: the saved input.  Accumulates dW (and db),
        returns (dx or None, x_planes)."""
        assert self.cout % 8 == 0 and gz.shape[-1] == self.cout
        stride = self.stride[1:]
        spatial = self.stride[1] == 2 and self.k[1] > 1
        if spatial:           # strided 3x3(x3) conv: with gz on the even positions of the input grid (zeros elsewhere) both
            # gradients are stride-1 'same' ones: dx = conv(gz', flip(W)^T), dW[k] = sum_i gz'[i] x[i + k - pad]
            gz = to.scatter_stride2(gz, (x.shape[2], x.shape[3]))
            stride = (1, 1)
        N, T, Ho, Wo, _ = gz.shape
        if WGRAD_PLANES:      # the first implementation: channel-major plane copies of both operands (kept for A/B runs)
            sp = (self.pad[1], self.pad[2])
            if x_planes is None:
                x_planes = to.to_planes(x, pad=sp, stride=stride, channels=self.cin, copies=True)
            to.wgrad(to.to_planes(gz, pad=sp), x_planes, (Ho, Wo), self.k, self.g)
        else:                 # operands read straight from NDHWC (MN-major tcgen05 operands, tap = TMA coordinate shift)
            to.wgrad_nhwc(gz, x, self.k, stride, self.g, cout=self.cout, cin=self.cin)
        if self.bias is not None:
            L.call('dt_bias_grad', L.ptr(gz), gz.numel() // gz.shape[-1], self.cout, gz.shape[-1], L.ptr(self.bias_g), L.stream_ptr())
        dx = None
        if need_dx:
            dx = cv.conv3d(gz, self.w_dg, self.k, (1, 1, 1), self.pad, out_f32=False, dtype=cv.BF16, cin=self.cout)
            if self.stride[1] == 2 and not spatial:
                dx = to.scatter_stride2(dx, (x.shape[2], x.shape[3]))
        return dx, x_planes

    def update(self, lr, momentum, wd, grad_scale):
        to.sgd_update(self.w, self.g, self.m, lr, momentum, wd, grad_scale, self.w_fwd, self.w_dg)
        if self.bias is not None:     # biases: no weight decay, 2x learning rate (model_builder.py:971-976)
            to.sgd_update(self.bias.view(1, 1, -1), self.bias_g.view(1, 1, -1), self.bias_m.view(1, 1, -1), 2.0 * lr, momentum, 0.0,
                          grad_scale)


def _subpixel_taps():
    """(sub-pixel filter (py, px), footprint tap (dy, dx), ConvTranspose tap (ky, kx)) of the k4-s2-p1 ConvTranspose written as
    four 2x2 sub-pixel filters on one 3x3 footprint (engine.py)."""
    for py in range(2):
        for px in range(2):
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    ky, kx = py + 1 - 2 * dy, px + 1 - 2 * dx
                    if 0 <= ky <= 3 and 0 <= kx <= 3:
                        yield py * 2 + px, dy + 1, dx + 1, ky, kx


def subpixel_deconv_conv(torch, blobs):
    """kps_score_lowres (ConvTranspose (Cin, K, 4, 4), stride 2, pad 1) as a trainable 3x3 conv with 4K (padded) outputs
    -> (TrainConv, K, padded output count)."""
    wt = blobs['kps_score_lowres_w']
    cin, K = wt.shape[0], wt.shape[1]
    ldk = (4 * K + 7) // 8 * 8
    w3 = np.zeros((ldk, cin, 3, 3), np.float32)
    for sub, ty, tx, ky, kx in _subpixel_taps():
        w3[sub * K:(sub + 1) * K, :, ty, tx] = wt[:, :, ky, kx].T
    b3 = np.zeros((ldk,), np.float32); b3[:4 * K] = np.tile(blobs['kps_score_lowres_b'], 4)
    c = TrainConv(torch, w3, bias=b3)
    c.cout_live = 4 * K
    return c, K, ldk


def export_subpixel_deconv(tr, blobs, out):
    """The inverse of subpixel_deconv_conv on the trained master filter: kps_score_lowres_{w,b} into `out`."""
    K = tr.K
    w3 = tr._blob_w(tr.kps_lowres, (tr.kp_ld, tr.kps_lowres.cin, 3, 3))                 # [ldk, cin, 3, 3]
    wt = np.zeros_like(blobs['kps_score_lowres_w'])                                      # (cin, K, 4, 4)
    for sub, ty, tx, ky, kx in _subpixel_taps():
        wt[:, :, ky, kx] = w3[sub * K:(sub + 1) * K, :, ty, tx].T
    out['kps_score_lowres_w'] = wt
    out['kps_score_lowres_b'] = tr.kps_lowres.bias.cpu().numpy()[:K].copy()


class RpnTrainer(object):
    def __init__(self, cfg, blobs, spec=None, world=1, buckets=4, lr=None, momentum=None, weight_decay=None):
        torch = L.require_cuda()
        self.torch, self.cfg, self.world = torch, cfg, world
        self.spec = s = spec or P.GraphSpec(cfg)
        assert s.fpn and s.block == 'bottleneck' and not s.head3d, 'RpnTrainer: FPN bottleneck bodies with 2-D RPN heads'
        self.lr = cfg.SOLVER.BASE_LR if lr is None else lr
        self.momentum = cfg.SOLVER.MOMENTUM if momentum is None else momentum
        self.wd = cfg.SOLVER.WEIGHT_DECAY if weight_decay is None else weight_decay
        # frozen stem (conv1, pool1, res2): the inference engine's bf16 kernels
        self.eng = DetectionEngine(cfg, blobs, s, dtype='bf16')
        self.convs = []                                   # forward order
        mk = self._mk
        self.stages = []
        dim_in = s.dims[1]
        for si in range(1, len(s.counts)):
            dim_out, inner = s.dims[si + 1], s.dim_inner * (2 ** si)
            blocks = []
            for i in range(s.counts[si]):
                pre = 'res%d_%d' % (si + 2, i)
                st = (1, 2, 2) if i == 0 else (1, 1, 1)
                s1, s3 = (st, (1, 1, 1)) if s.stride_1x1 else ((1, 1, 1), st)
                assert s3 == (1, 1, 1), 'RpnTrainer: stride on the 1x1 conv (RESNETS.STRIDE_1X1 True, the default)'
                blk = dict(a=mk(blobs, pre + '_branch2a', affine=True, stride=s1, relu=True),
                           b=mk(blobs, pre + '_branch2b', affine=True, relu=True),
                           c=mk(blobs, pre + '_branch2c', affine=True, relu=True),
                           sc=mk(blobs, pre + '_branch1', affine=True, stride=st) if dim_in != dim_out else None)
                blocks.append(blk)
                dim_in = dim_out
            self.stages.append(blocks)
        names = s.stage_blobs[::-1]                       # coarsest first
        self.lat = [mk(blobs, 'fpn_inner_' + names[0])] + [mk(blobs, 'fpn_inner_%s_lateral' % n) for n in names[1:]]
        self.post = [mk(blobs, 'fpn_' + n) for n in names]
        k = str(s.rpn_levels[0])
        A = self.A = s.num_anchors
        self.rpn_conv = mk(blobs, 'conv_rpn_fpn' + k, relu=True)
        self.blobs0 = blobs                                   # the initial weights dict (export_blobs fills the trained ones in)
        w = np.concatenate([blobs['rpn_cls_logits_fpn%s_w' % k], blobs['rpn_bbox_pred_fpn%s_w' % k]], 0)
        b = np.concatenate([blobs['rpn_cls_logits_fpn%s_b' % k], blobs['rpn_bbox_pred_fpn%s_b' % k]], 0)
        ld = self.rpn_ld = (5 * A + 7) // 8 * 8           # padded with zero filters so the planes are 16-byte rows
        wp = np.zeros((ld,) + w.shape[1:], np.float32); wp[:5 * A] = w
        bp = np.zeros((ld,), np.float32); bp[:5 * A] = b
        self.rpn_out = TrainConv(torch, wp, bias=bp)
        self.rpn_out.cout_live = 5 * A
        self.rpn_out._accumulate = self.rpn_conv._accumulate = 1
        self.convs.append(self.rpn_out)
        self._build_heads(blobs)                          # RoI heads of the full model (KeypointRcnnTrainer); none here
        self._alloc_grads(buckets)

    def _alloc_grads(self, buckets):
        """The flat gradient buffer in BACKWARD order (so a bucket finished early in the backward pass is contiguous), its
        all-reduce buckets and the loss accumulator."""
        torch, world = self.torch, self.world
        order = self.convs[::-1]
        total = sum(c.nparams() for c in order)
        self.flat_g = torch.zeros(total, dtype=torch.float32, device='cuda')
        off = 0
        for c in order:
            n = c.w.numel()
            c.g = self.flat_g[off:off + n].view_as(c.w); off += n
            if c.bias is not None:
                c.bias_g = self.flat_g[off:off + c.bias.numel()]; off += c.bias.numel()
        bounds, self.bucket_ends = plan_buckets([c.nparams() for c in order], buckets)
        self._order_end = {id(c): e for c, e in zip(order, bounds)}
        self.reducer = BucketReducer(self.flat_g, self.bucket_ends, world)
        self.loss = torch.zeros(2, dtype=torch.float32, device='cuda')

    def _build_heads(self, blobs):
        pass

    def _mk(self, blobs, name, affine=False, stride=(1, 1, 1), relu=False):
        c = TrainConv(self.torch, blobs[name + '_w'], scale=blobs[name + '_bn_s'] if affine else None,
                      shift=blobs[name + '_bn_b'] if affine else None, bias=None if affine else blobs[name + '_b'],
                      stride=stride, relu=relu)
        c.name = name
        self.convs.append(c)
        return c

    # ------------------------------------------------------------------ forward (activations saved for the backward)
    def forward_all(self, frames_u8):
        """stem -> res2 (frozen) -> res3..5 -> FPN -> RPN heads; returns per level the fp32 RPN outputs [B,1,H,W,ld]."""
        torch, eng, s, cfg = self.torch, self.eng, self.spec, self.cfg
        B, T, H, W, _ = frames_u8.shape
        self.rpn_conv.macs = self.rpn_out.macs = 0
        g = eng._geom_tensors(B, H, W)
        x = eng._blob(frames_u8, g['scale'], g['hr'], g['wr'], g['hp'], g['wp'])
        xs = x.view((B * T,) + tuple(x.shape[2:]))
        y = cv.conv1_7x7s2(xs, eng.conv1_w, (g['hp'], g['wp']), eng.conv1_s, eng.conv1_b, relu=True, dtype=cv.BF16)
        y = dense_ops.maxpool2d(y, 3, 2, 1)
        y = y.view((B, T) + tuple(y.shape[1:]))
        for blk in eng.stages[0]:
            y = eng._run_block(blk, y)
        sv = self.saved = dict(blocks=[], C=[y])                                  # C2 (frozen producer)
        for blocks in self.stages:
            for blk in blocks:
                a = blk['a'].forward(y)
                b = blk['b'].forward(a)
                sc = blk['sc'].forward(y) if blk['sc'] is not None else y
                out = blk['c'].forward(b, residual=sc, res_mode=1)
                sv['blocks'].append(dict(blk=blk, x=y, a=a, b=b, y=out))
                y = out
            sv['C'].append(y)
        Cs = sv['C'][::-1]                                                        # coarsest first
        inner = [self.lat[0].forward(Cs[0])]
        for i in range(1, len(Cs)):
            inner.append(self.lat[i].forward(Cs[i], residual=inner[i - 1], res_mode=2))
        tm = s.link == 'slice-center' and T > 1        # frames-outermost storage: the centre-frame link below is a view
        Ps = [self.post[i].forward(inner[i], time_major=tm) for i in range(len(inner))]   # [B, T, h, w, 256], coarsest first
        sv['inner'], sv['P'] = inner, Ps
        c = int(cfg.VIDEO.NUM_FRAMES_MID / 2) if (s.link == 'slice-center' and T > 1) else 0
        sv['center'] = c
        feats = [p[:, c:c + 1] if T > 1 else p for p in Ps]                       # slice-center link (contiguous [B, 1, h, w, C] views)
        assert all(f.is_contiguous() for f in feats)
        p6 = dense_ops.maxpool2d(feats[0].view((B,) + tuple(feats[0].shape[2:])), 1, 2, 0)
        feats = [p6.view((B, 1) + tuple(p6.shape[1:]))] + feats                   # P6 first (coarsest)
        sv['feats'] = feats
        outs, hs = [], []
        for f in feats:
            h = self.rpn_conv.forward(f)
            o = torch.empty(tuple(h.shape[:4]) + (self.rpn_ld,), dtype=torch.float32, device='cuda')
            self.rpn_out.forward(h, out_f32=True, out=o)
            hs.append(h); outs.append(o)
        sv['rpn_h'] = hs
        return outs[::-1]                                                          # finest (P2) first, like spec.rpn_levels

    # ------------------------------------------------------------------ backward
    def _bucket_ready(self, conv, pending=None):
        """Launch the all-reduce of every bucket whose last filter gradient has just been enqueued."""
        self.reducer.ready(self._order_end[id(conv)])

    def backward(self, rpn_outs, targets, head_grads=None, fresh=True):
        """targets: per level (finest first) dict(labels [B,H,W,A] i32, bbox_targets / inside / outside [B,H,W,4A] f32).
        head_grads: fp32 accumulators of the RoI heads' gradient wrt the per-level features (aligned with saved['feats'],
        coarsest first; None entries for levels the heads do not read).  fresh=False: the gradient buffer already holds the
        heads' filter gradients (KeypointRcnnTrainer zeroes it and resets the reducer itself)."""
        torch, cfg, s, sv = self.torch, self.cfg, self.spec, self.saved
        A = self.A
        if fresh:
            L.call('dt_memset', L.ptr(self.flat_g), 0, self.flat_g.numel() * 4, L.stream_ptr())
            self.reducer.reset()
        L.call('dt_memset', L.ptr(self.loss), 0, 8, L.stream_ptr())
        pending = None
        B = rpn_outs[0].shape[0]
        s_cls = 1.0 / self.world / cfg.TRAIN.RPN_BATCH_SIZE_PER_IM / cfg.TRAIN.IMS_PER_BATCH
        s_box = 1.0 / self.world / B
        feats, hs = sv['feats'], sv['rpn_h']                                    # coarsest first
        nl = len(feats)
        gP6 = None
        gfeat = [None] * nl
        # RPN heads, level by level (shared filters: their gradients accumulate across levels)
        for li in range(nl):
            o = rpn_outs[nl - 1 - li]                                           # level of feats[li]
            t = targets[nl - 1 - li]
            go = torch.empty(tuple(o.shape[:4]) + (self.rpn_ld,), dtype=torch.bfloat16, device='cuda')
            rows = o.numel() // o.shape[-1]
            L.call('dt_rpn_loss_grad', L.ptr(o), o.shape[-1], L.ptr(t['labels']), L.ptr(t['bbox_targets']), L.ptr(t['inside']),
                   L.ptr(t['outside']), rows, A, s_cls, s_box, 1.0 / 9.0, L.ptr(go), self.rpn_ld, L.ptr(self.loss), L.stream_ptr())
            gh, _ = self.rpn_out.backward(go, hs[li])
            gz = to.bwd_pointwise(gh, None, hs[li], None)                      # Relu of conv_rpn (bias conv: no scale)
            gfeat[li], _ = self.rpn_conv.backward(gz, feats[li])
            if head_grads is not None and head_grads[li] is not None:      # + the RoI heads' gradient (RoIAlign backward)
                gfeat[li] = to.grad_join_f32(head_grads[li].view(gfeat[li].shape), gfeat[li])
        self._bucket_ready(self.rpn_conv, pending)
        # P6 = stride-2 subsample of P5's centre frame: its gradient lands on P5's even positions
        Ps, inner = sv['P'], sv['inner']                                         # coarsest first (P5 ... P2)
        T = Ps[0].shape[1]
        c = sv['center']
        gP = []
        for i in range(len(Ps)):
            g = gfeat[i + 1]                                                     # [B,1,h,w,256]
            if i == 0:
                g = to.bwd_pointwise(g, to.scatter_stride2(gfeat[0], (g.shape[2], g.shape[3])))
            if T > 1:                                                            # slice-center: the other frames get zero
                full = torch.empty(tuple(Ps[i].shape), dtype=torch.bfloat16, device='cuda')
                L.call('dt_embed_frame', L.ptr(g), g.shape[0], T, g.numel() // g.shape[0], c, L.ptr(full), L.stream_ptr())
                g = full
            gP.append(g)
        # FPN: finest level first (its inner gradient flows into the next coarser one through the top-down add)
        g_inner = [None] * len(Ps)
        for i in range(len(Ps) - 1, -1, -1):
            gi, _ = self.post[i].backward(gP[i], inner[i])
            if i < len(Ps) - 1:                                                  # add the 2x2 sums of the finer level's inner gradient
                B_, T_, h, w, C_ = gi.shape
                gi = to.upsample_add_bwd(g_inner[i + 1], gi)
            g_inner[i] = gi
        Cs = sv['C'][::-1]
        gC = []
        for i in range(len(Ps)):
            need_dx = i < len(Ps) - 1                                            # C2's producer is frozen
            dx, _ = self.lat[i].backward(g_inner[i], Cs[i], need_dx=need_dx)
            gC.append(dx)
        self._bucket_ready(self.lat[0], pending)
        # body: res5 -> res3
        blocks = sv['blocks']
        bi = len(blocks)
        g_parts = (gC[0], None)                                                  # gradient wrt C5 from its lateral
        stage_of = []
        for si, st_blocks in enumerate(self.stages):
            stage_of += [si] * len(st_blocks)
        for bidx in range(len(blocks) - 1, -1, -1):
            sb = blocks[bidx]
            blk = sb['blk']
            g1, g2 = g_parts
            last_of_trunk = bidx == 0
            # gradient wrt the block output, masked by its ReLU, for BOTH consumers (branch2c and the shortcut) from one read
            gz3, gsc = to.bwd_pointwise(g1, g2, sb['y'], blk['c'].scale, second=True,
                                        scale2=blk['sc'].scale if blk['sc'] is not None else None)
            gb, _ = blk['c'].backward(gz3, sb['b'])
            gz2 = to.bwd_pointwise(gb, None, sb['b'], blk['b'].scale)
            ga, _ = blk['b'].backward(gz2, sb['a'])
            gz1 = to.bwd_pointwise(ga, None, sb['a'], blk['a'].scale)
            need_dx = not last_of_trunk                                          # res2 is frozen: stop at the input of res3_0
            gx1, xpl = blk['a'].backward(gz1, sb['x'], need_dx=need_dx)
            if blk['sc'] is not None:
                gx2, _ = blk['sc'].backward(gsc, sb['x'], x_planes=xpl, need_dx=need_dx)
            else:
                gx2 = gsc
            for cnv in (blk['c'], blk['b'], blk['a'], blk['sc']):
                if cnv is not None:
                    self._bucket_ready(cnv, pending)
            g_parts = (gx1, gx2)
            # a stage boundary: the lateral's gradient wrt this stage output joins the two parts
            if bidx > 0 and stage_of[bidx - 1] != stage_of[bidx]:
                lvl = len(self.stages) - stage_of[bidx - 1] - 1                 # index into gC (coarsest first)
                g_parts = (to.bwd_pointwise(gx1, gx2), gC[lvl])
        self.reducer.wait()
        return self.loss

    def step_flops(self):
        """Algorithmic FLOPs of the last step's tensor-core work: 2 * MACs of every trainable conv / FC, once forward, once for
        the filter gradient and once for the input gradient where one is needed (everything except the first trainable convs
        after the frozen stem).  The frozen stem's forward (conv1, res2) is not counted."""
        first = {id(self.stages[0][0]['a']), id(self.stages[0][0]['sc'])}
        tot = 0
        for c in self.convs:
            m = getattr(c, 'macs', 0)
            tot += 2 * m * (2 if id(c) in first else 3)
        return tot

    # ------------------------------------------------------------------ weights back to the reference's blob names
    @staticmethod
    def _blob_w(c, shape):
        """packed master filter [taps, Cout, Cin] -> the blob layout (Cout, Cin[, kT], kH, kW) of `shape`."""
        kT, kH, kW = c.k
        w = c.w.view(kT, kH, kW, c.cout, c.cin).permute(3, 4, 0, 1, 2).contiguous().cpu().numpy()
        return w.reshape((c.cout, c.cin) + tuple(shape[2:])) if len(shape) >= 2 else w

    def _export_named(self, blobs):
        """A copy of the weights dict with every conv that carries its blob name (filter and bias) replaced by its trained value."""
        out = dict(blobs)
        for c in self.convs:
            n = getattr(c, 'name', None)
            if n is None:
                continue
            out[n + '_w'] = self._blob_w(c, blobs[n + '_w'].shape).astype(np.float32)
            if c.bias is not None:
                out[n + '_b'] = c.bias.cpu().numpy()
        return out

    def export_blobs(self, blobs):
        """The trained parameters written back into a copy of the weights dict under the reference's blob names
        (lib/utils/net.py:252-294 save_model_to_weights_file): what tools/test_net.py loads through TEST.WEIGHTS."""
        out = self._export_named(blobs)
        k = str(self.spec.rpn_levels[0])
        A = self.A
        w = self.rpn_out.w[0].cpu().numpy()                                   # [ld, Cin]
        b = self.rpn_out.bias.cpu().numpy()
        out['rpn_cls_logits_fpn%s_w' % k] = w[:A].reshape(blobs['rpn_cls_logits_fpn%s_w' % k].shape)
        out['rpn_bbox_pred_fpn%s_w' % k] = w[A:5 * A].reshape(blobs['rpn_bbox_pred_fpn%s_w' % k].shape)
        out['rpn_cls_logits_fpn%s_b' % k], out['rpn_bbox_pred_fpn%s_b' % k] = b[:A].copy(), b[A:5 * A].copy()
        return out

    def _sgd_table(self):
        """One dt_sgd_item per parameter tensor (filters, then the biases: 2x learning rate, no weight decay,
        model_builder.py:971-976) + the block prefix of the single-launch update; the pointers are stable for the trainer's life."""
        import ctypes as C
        torch = self.torch
        items, first, nb = [], [], 0

        def add(w, g, m, wf, wdg, taps, co, ci, lr_mult, wd_mult):
            nonlocal nb
            tci, tco = (ci + 31) // 32, (co + 31) // 32
            items.append(L.SgdItem(w.data_ptr(), g.data_ptr(), m.data_ptr(), wf.data_ptr() if wf is not None else None,
                                   wdg.data_ptr() if wdg is not None else None, taps, co, ci, tci, tco, lr_mult, wd_mult))
            first.append(nb)
            nb += taps * tci * tco
        for c in self.convs:
            add(c.w, c.g, c.m, c.w_fwd, c.w_dg, c.taps, c.cout, c.cin, 1.0, 1.0)
            if c.bias is not None:
                add(c.bias, c.bias_g, c.bias_m, None, None, 1, 1, c.bias.numel(), 2.0, 0.0)
        arr = (L.SgdItem * len(items))(*items)
        buf = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).cuda()
        return buf, torch.tensor(first, dtype=torch.int32).cuda(), len(items), nb

    def update(self):
        gs = 1.0            # losses already carry 1/NUM_GPUS; the all-reduce is a SUM (model_builder.py:484,938-942)
        if not hasattr(self, '_sgd'):
            self._sgd = self._sgd_table()
        buf, first, n, nb = self._sgd
        L.call('dt_sgd_update_multi', L.ptr(buf), L.ptr(first), n, nb, float(self.lr), float(self.momentum), float(self.wd), gs, L.stream_ptr())

    def step(self, frames_u8, targets):
        outs = self.forward_all(frames_u8)
        loss = self.backward(outs, targets)
        self.update()
        return loss

    # ------------------------------------------------------------------ synthetic targets (the f1 loaders are out of scope)
    def synthetic_targets(self, B, H, W, seed=0):
        """Per level random RPN targets of the reference's shapes (lib/roi_data/rpn.py): 256 sampled anchors per image
        (half foreground) spread over the levels, unit inside weights on foreground, outside weights 1 / 256."""
        torch = self.torch
        eng = self.eng
        g = eng._geom_tensors(B, H, W)
        rng = np.random.RandomState(seed)
        A = self.A
        out = []
        for lvl in self.spec.rpn_levels:
            h, w = int(np.ceil(g['hp'] / 2. ** lvl)), int(np.ceil(g['wp'] / 2. ** lvl))
            labels = -np.ones((B, h, w, A), np.int32)
            n = max(2, int(256 * (h * w) / float(sum(int(np.ceil(g['hp'] / 2. ** l)) * int(np.ceil(g['wp'] / 2. ** l)) for l in self.spec.rpn_levels))))
            bt = np.zeros((B, h, w, 4 * A), np.float32); iw = np.zeros_like(bt); ow = np.zeros_like(bt)
            for b in range(B):
                idx = rng.choice(h * w * A, size=min(n, h * w * A), replace=False)
                fg = idx[:len(idx) // 2]
                lab = labels[b].reshape(-1)
                lab[idx] = 0; lab[fg] = 1
                pos, a = fg // A, fg % A
                for k in range(4):
                    bt[b].reshape(-1, 4 * A)[pos, a * 4 + k] = rng.normal(0, 0.5, len(fg))
                    iw[b].reshape(-1, 4 * A)[pos, a * 4 + k] = 1.0
                pos_all, a_all = idx // A, idx % A
                for k in range(4):
                    ow[b].reshape(-1, 4 * A)[pos_all, a_all * 4 + k] = 1.0 / 256.0
            out.append(dict(labels=torch.from_numpy(labels).cuda(), bbox_targets=torch.from_numpy(bt).cuda(),
                            inside=torch.from_numpy(iw).cuda(), outside=torch.from_numpy(ow).cuda()))
        return out


def pack_gt(entries, Gmax=None, K=17, device='cuda'):
    """roidb-style entries (dicts with 'boxes' [G,4] in ORIGINAL image coordinates, optional 'gt_classes', 'is_crowd',
    'gt_keypoints' [G,3,K] int32) -> the fixed-capacity device tensors of dt_rpn_targets / dt_sample_rois.  The RPN sees the
    non-crowd boxes only (rpn.py:84-86), the RoI sampler all of them (json_dataset.py:437).
    Tube entries (T > 1 frames): 'boxes' [G,4T] (frame t in columns 4t..4t+3), 'gt_keypoints' [G,3,K*T] (column t*K + k)
    and an optional per-frame visibility 'gt_visible' [G,T]; the latter is returned as 'gt_visible' [B,Gmax,T] uint8,
    aligned with 'rpn_boxes' (the boxes dt_rpn_targets reads)."""
    import torch
    B = len(entries)
    Gmax = Gmax or max(8, max(len(e['boxes']) for e in entries))
    D = max(np.asarray(e['boxes']).reshape(len(e['boxes']), -1).shape[1] if len(e['boxes']) else 4 for e in entries)
    T = D // 4
    boxes = np.zeros((B, Gmax, D), np.float32); rboxes = np.zeros((B, Gmax, D), np.float32)
    classes = np.zeros((B, Gmax), np.int32); crowd = np.zeros((B, Gmax), np.int32)
    kps = np.zeros((B, Gmax, 3, K * T), np.int32)
    vis = np.ones((B, Gmax, T), np.uint8)
    counts = np.zeros((B,), np.int32); rcounts = np.zeros((B,), np.int32)
    for b, e in enumerate(entries):
        g = len(e['boxes'])
        assert g <= Gmax, 'more gt boxes than Gmax'
        boxes[b, :g] = np.asarray(e['boxes'], np.float32).reshape(g, D)
        classes[b, :g] = e.get('gt_classes', np.ones(g, np.int32))
        cr = np.asarray(e.get('is_crowd', np.zeros(g, bool))).astype(bool)
        crowd[b, :g] = cr
        if 'gt_keypoints' in e:
            kps[b, :g] = e['gt_keypoints']
        counts[b] = g
        keep = np.where((classes[b, :g] > 0) & ~cr)[0]
        rboxes[b, :len(keep)] = boxes[b, keep]
        rcounts[b] = len(keep)
        if 'gt_visible' in e:
            vis[b, :len(keep)] = np.asarray(e['gt_visible']).reshape(g, T)[keep]
    t = lambda a: torch.from_numpy(a).to(device)
    out = dict(boxes=t(boxes), classes=t(classes), crowd=t(crowd), keypoints=t(kps), counts=t(counts), rpn_boxes=t(rboxes),
               rpn_counts=t(rcounts))
    if any('gt_visible' in e for e in entries):
        out['gt_visible'] = t(vis)
    return out


class KeypointRcnnTrainer(RpnTrainer):
    """The end-to-end keypoint R-CNN training step (model_builder.py keypoint_rcnn: RPN + Fast R-CNN + keypoint heads)."""

    def _build_heads(self, blobs):
        torch, cfg, s = self.torch, self.cfg, self.spec
        res, fd = cfg.FAST_RCNN.ROI_XFORM_RESOLUTION, s.fpn_dim
        n6 = blobs['fc6_w'].shape[0]
        w6 = blobs['fc6_w'].reshape(n6, fd, res, res).transpose(0, 2, 3, 1).reshape(n6, -1)      # columns in RoIAlign (h, w, c) order
        add = self.convs.append
        self.fc6 = TrainConv(torch, w6, bias=blobs['fc6_b'], relu=True); add(self.fc6)
        self.fc7 = TrainConv(torch, blobs['fc7_w'], bias=blobs['fc7_b'], relu=True); add(self.fc7)
        C_ = self.C_ = s.num_classes
        w = np.concatenate([blobs['cls_score_w'], blobs['bbox_pred_w']], 0)
        b = np.concatenate([blobs['cls_score_b'], blobs['bbox_pred_b']], 0)
        ld = self.cb_ld = (5 * C_ + 7) // 8 * 8
        wp = np.zeros((ld, w.shape[1]), np.float32); wp[:5 * C_] = w
        bp = np.zeros((ld,), np.float32); bp[:5 * C_] = b
        self.cls_bbox = TrainConv(torch, wp, bias=bp); add(self.cls_bbox)
        self.cls_bbox.cout_live = 5 * C_
        self.kps = []
        for i in range(cfg.KRCNN.NUM_STACKED_CONVS):
            c = TrainConv(torch, blobs['conv_fcn%d_w' % (i + 1)], bias=blobs['conv_fcn%d_b' % (i + 1)], relu=True)
            self.kps.append(c); add(c)
        self.kps_lowres, self.K, self.kp_ld = subpixel_deconv_conv(torch, blobs); add(self.kps_lowres)
        self.loss_heads = torch.zeros(4, dtype=torch.float32, device='cuda')      # cls, bbox, kps, #correct
        self.totals = torch.zeros(2, dtype=torch.float32, device='cuda')          # live RoIs, keypoint weight sum (loss normalisers)
        self.iter = 0

    def export_blobs(self, blobs):
        out = RpnTrainer.export_blobs(self, blobs)
        cfg, s = self.cfg, self.spec
        res, fd = cfg.FAST_RCNN.ROI_XFORM_RESOLUTION, s.fpn_dim
        w6 = self.fc6.w[0].cpu().numpy()                                      # columns in (h, w, c) order -> (c, h, w)
        out['fc6_w'] = w6.reshape(-1, res, res, fd).transpose(0, 3, 1, 2).reshape(w6.shape[0], -1).copy()
        out['fc6_b'] = self.fc6.bias.cpu().numpy()
        out['fc7_w'], out['fc7_b'] = self.fc7.w[0].cpu().numpy().copy(), self.fc7.bias.cpu().numpy()
        C_ = self.C_
        w, b = self.cls_bbox.w[0].cpu().numpy(), self.cls_bbox.bias.cpu().numpy()
        out['cls_score_w'], out['bbox_pred_w'] = w[:C_].copy(), w[C_:5 * C_].copy()
        out['cls_score_b'], out['bbox_pred_b'] = b[:C_].copy(), b[C_:5 * C_].copy()
        for i, c in enumerate(self.kps):
            out['conv_fcn%d_w' % (i + 1)] = self._blob_w(c, blobs['conv_fcn%d_w' % (i + 1)].shape).astype(np.float32)
            out['conv_fcn%d_b' % (i + 1)] = c.bias.cpu().numpy()
        export_subpixel_deconv(self, blobs, out)
        return out

    # ------------------------------------------------------------------ geometry / proposals
    def _train_geom(self, B, H, W):
        g = self.eng._geom_tensors(B, H, W)
        if 'im_info_train' not in g:                          # rpn.py:90: im_info = (round(h * scale), round(w * scale), scale)
            g['im_info_train'] = self.torch.tensor([[g['hr'], g['wr'], g['scale']]] * B, dtype=self.torch.float32, device='cuda')
        return g

    def proposals(self, rpn_outs, im_info):
        """GenerateProposals + collect with the TRAIN settings, from the fp32 RPN outputs (finest level first)."""
        torch, cfg, s = self.torch, self.cfg, self.spec
        B, Lv, A = rpn_outs[0].shape[0], len(rpn_outs), self.A
        Kp = int(cfg.TRAIN.RPN_PRE_NMS_TOP_N)
        props = L.zeros((B, Lv, Kp, 5), torch.float32)
        counts = L.zeros((B, Lv), torch.int32)
        levels = []
        for l, o in enumerate(rpn_outs):
            o4 = o.view(o.shape[0], o.shape[2], o.shape[3], o.shape[4])
            levels.append(dict(logits=o4[..., :A], deltas=o4[..., A:5 * A], anchors=self.eng.anchors[l],
                               feat_stride=2. ** s.rpn_levels[l], out=props[:, l], counts=counts[:, l]))
        rpn_ops.rpn_proposals_levels(levels, im_info, Kp, A, float(cfg.TRAIN.RPN_MIN_SIZE), 1)
        post = int(cfg.TRAIN.RPN_POST_NMS_TOP_N)
        keep, nkeep = box_ops.nms_batched(props.view(B * Lv, Kp, 5), counts.view(-1), cfg.TRAIN.RPN_NMS_THRESH, box_ops.NMS_2D_GE,
                                          box_ops.ORDER_INDEX, max_keep=post)
        return rpn_ops.collect(props, keep, nkeep, post)

    def make_targets(self, rpn_outs, gt, B, H, W, seed):
        """All targets of one step on the device: RPN anchor targets, sampled RoIs + box targets, keypoint RoIs + labels."""
        cfg, s = self.cfg, self.spec
        g = self._train_geom(B, H, W)
        shapes = [(o.shape[2], o.shape[3]) for o in rpn_outs]
        rt = target_ops.rpn_targets(shapes, self.eng.anchors, [2. ** l for l in s.rpn_levels], self.A, gt['rpn_boxes'], gt['rpn_counts'],
                                    g['im_info_train'], cfg.TRAIN, seed)
        rois, scores, counts = self.proposals(rpn_outs, g['im_info_train'])
        L.call('dt_memset', L.ptr(self.totals), 0, 8, L.stream_ptr())
        smp = target_ops.sample_rois(rois, scores, counts, gt, g['im_info_train'], cfg, seed, keypoints=True, totals=self.totals)
        return rt, smp

    # ------------------------------------------------------------------ heads
    def _roi_levels(self, rois_flat):
        s, cfg = self.spec, self.cfg
        lv, _, _ = rpn_ops.distribute(rois_flat, None, col0=1, T=1, k_min=s.roi_levels[0], k_max=s.roi_levels[-1],
                                      s0=float(cfg.FPN.ROI_CANONICAL_SCALE), lvl0=float(cfg.FPN.ROI_CANONICAL_LEVEL), want_restore=False)
        return lv

    def forward_heads(self, smp):
        torch, cfg, s, sv = self.torch, self.cfg, self.spec, self.saved
        nl = len(s.roi_levels)
        feats = sv['feats'][::-1][:nl]                        # finest first: P2 .. P5, each [B, 1, h, w, C]
        fl = [f.view((f.shape[0] * f.shape[1],) + tuple(f.shape[2:])) for f in feats]
        scales = [1. / 2 ** l for l in s.roi_levels]
        h = sv['heads'] = dict(fl=fl, scales=scales)
        # box head
        rois = smp['rois'].view(-1, 5)
        R = rois.shape[0]
        lv = self._roi_levels(rois)
        res = cfg.FAST_RCNN.ROI_XFORM_RESOLUTION
        x = dense_ops.roi_align(fl, scales, rois, lv, res, cfg.FAST_RCNN.ROI_XFORM_SAMPLING_RATIO, T=1, k_min=s.roi_levels[0])
        x6 = x.view(1, 1, 1, R, -1)
        h6 = self.fc6.forward(x6)
        h7 = self.fc7.forward(h6)
        o = torch.empty((1, 1, 1, R, self.cb_ld), dtype=torch.float32, device='cuda')
        self.cls_bbox.forward(h7, out_f32=True, out=o)
        h.update(rois=rois, lv=lv, x6=x6, h6=h6, h7=h7, o=o)
        # keypoint head
        krois = smp['kp_rois'].view(-1, 5)
        D = krois.shape[0]
        klv = self._roi_levels(krois)
        kres = cfg.KRCNN.ROI_XFORM_RESOLUTION
        xk = dense_ops.roi_align(fl, scales, krois, klv, kres, cfg.KRCNN.ROI_XFORM_SAMPLING_RATIO, T=1, k_min=s.roi_levels[0])
        acts = [xk.view(D, 1, kres, kres, -1)]
        for c in self.kps:
            acts.append(c.forward(acts[-1]))
        low = torch.empty((D, 1, kres, kres, self.kp_ld), dtype=torch.float32, device='cuda')
        self.kps_lowres.forward(acts[-1], out_f32=True, out=low)
        h.update(krois=krois, klv=klv, kacts=acts, low=low)
        return o.view(R, self.cb_ld), low.view(D, kres, kres, self.kp_ld)

    def backward_heads(self, smp):
        """Losses + backward of both RoI heads; returns the fp32 feature-gradient accumulators (coarsest first, aligned with
        saved['feats']: None for P6)."""
        torch, cfg, s, sv = self.torch, self.cfg, self.spec, self.saved
        h = sv['heads']
        fl, scales = h['fl'], h['scales']
        dfe = [L.zeros(tuple(f.shape), torch.float32) for f in fl]                 # finest first
        w = 1.0 / self.world
        L.call('dt_memset', L.ptr(self.loss_heads), 0, 16, L.stream_ptr())
        # keypoint head (model_builder.py:873-888: scale = KRCNN.LOSS_WEIGHT / NUM_GPUS)
        low = h['low']
        D, _, S, _, ldk = low.shape
        g = to.kps_loss_grad(low.view(D, S, S, ldk), self.K, smp['kp_locations'].view(D, self.K), smp['kp_weights'].view(D, self.K),
                             self.totals, cfg.KRCNN.LOSS_WEIGHT * w, ldk, loss=self.loss_heads[2:3])
        acts = h['kacts']
        gh, _ = self.kps_lowres.backward(g.view(D, 1, S, S, ldk), acts[-1])
        to.subpixel_grad_fix(self.kps_lowres.g, self.kps_lowres.bias_g, self.K)
        self._bucket_ready(self.kps_lowres)
        for i in range(len(self.kps) - 1, -1, -1):
            gz = to.bwd_pointwise(gh, None, acts[i + 1], None)
            gh, _ = self.kps[i].backward(gz, acts[i])
            self._bucket_ready(self.kps[i])
        to.roi_align_bwd(gh, dfe, scales, h['krois'], h['klv'], S, cfg.KRCNN.ROI_XFORM_SAMPLING_RATIO, T=1, k_min=s.roi_levels[0])
        # box head (model_builder.py:481-493: both losses scaled by 1 / NUM_GPUS)
        o = h['o']
        R = o.shape[3]
        C_ = self.C_
        go = to.frcnn_loss_grad(o.view(R, self.cb_ld), smp['labels'].view(-1), smp['bbox_targets'].view(R, 4 * C_),
                                smp['inside'].view(R, 4 * C_), smp['outside'].view(R, 4 * C_), C_, self.totals, w, w, self.cb_ld,
                                loss=self.loss_heads[0:2], accuracy=self.loss_heads[3:4])
        g7, _ = self.cls_bbox.backward(go.view(1, 1, 1, R, self.cb_ld), h['h7'])
        self._bucket_ready(self.cls_bbox)
        g6, _ = self.fc7.backward(to.bwd_pointwise(g7, None, h['h7'], None), h['h6'])
        self._bucket_ready(self.fc7)
        gx, _ = self.fc6.backward(to.bwd_pointwise(g6, None, h['h6'], None), h['x6'])
        self._bucket_ready(self.fc6)
        res = cfg.FAST_RCNN.ROI_XFORM_RESOLUTION
        to.roi_align_bwd(gx.view(R, 1, res, res, -1), dfe, scales, h['rois'], h['lv'], res, cfg.FAST_RCNN.ROI_XFORM_SAMPLING_RATIO, T=1,
                         k_min=s.roi_levels[0])
        nf = len(sv['feats'])
        out = [None] * nf
        for i, d in enumerate(dfe):                                                # dfe[i] = level roi_levels[i]; feats coarsest first
            out[nf - 1 - i] = d
        return out

    def step(self, frames_u8, gt, seed=None):
        """One SGD iteration from uint8 frames and packed ground truth (pack_gt): returns (rpn loss [2], head losses [4])."""
        B, T, H, W, _ = frames_u8.shape
        seed = self.cfg.RNG_SEED + self.iter if seed is None else seed
        outs = self.forward_all(frames_u8)
        rt, smp = self.make_targets(outs, gt, B, H, W, seed)
        self.forward_heads(smp)
        L.call('dt_memset', L.ptr(self.flat_g), 0, self.flat_g.numel() * 4, L.stream_ptr())
        self.reducer.reset()
        hg = self.backward_heads(smp)
        loss = self.backward(outs, rt, head_grads=hg, fresh=False)
        self.update()
        self.iter += 1
        self.last = dict(rpn_targets=rt, sampled=smp)
        return loss, self.loss_heads
