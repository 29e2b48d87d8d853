"""Training step of the 3-D tube keypoint R-CNN (configs/video/3d/03_R-18-3D_PTFromCOCO.yaml: MODEL.TYPE keypoint_rcnn with
VIDEO.BODY_HEAD_LINK '', reference lib/modeling/model_builder.py:179-306,426-493,500-635,755-888, ResNet3D.py:59-146,
251-344).  Everything runs on the device, T = VIDEO.NUM_FRAMES_MID frames per clip:

    trunk      conv1 / pool1 / res2 frozen (the inference engine's bf16 kernels), res3 + res4 basic blocks trained; the
               stride-2 [TIME_KERNEL_DIM.BODY, 3, 3] branch2a convs take their gradients through TrainConv's zero-insertion
               path (dt_scatter_stride2 + stride-1 dgrad / wgrad)
    RPN        conv_rpn [HEAD_RPN, 3, 3] + ReLU, fused rpn_cls_logits_1 | rpn_bbox_pred_1 per frame; dt_rpn_tube_loss_grad
               (TimePool avg of the logits, normalised SigmoidCrossEntropyLoss, SmoothL1Loss on the a*4T + t*4 + k deltas)
    targets    dt_rpn_targets on tube anchors, proposals with the TRAIN settings + tube NMS (mean-over-T IoU), dt_sample_rois(T)
    box head   tube RoIAlign 7x7 -> res5 (two basic blocks, time kernel 1) -> spatial mean -> cls_score_1 | bbox_pred_1 per
               RoI-frame; dt_frcnn_tube_loss_grad folds the frames (and unfolds the gradient); dt_spatial_mean_bwd
    kps head   tube RoIAlign 14x14 -> 8 x [HEAD_KPS, 3, 3] convs -> per-frame sub-pixel deconv; dt_kps_loss_grad on the
               [D*T] frame rows (label index frame*K + joint)
    backward   heads, RPN, res4, res3 through the same dgrad / wgrad kernels as the FPN trainer; both heads' RoIAlign
               backward accumulates into one fp32 [B*T, H, W, C] map that joins conv_rpn's input gradient."""
import numpy as np

from .. import _lib as L
from ..ops import conv as cv, dense_ops, train_ops as to, rpn_ops, box_ops, target_ops
from . import params as P
from .engine import DetectionEngine
from .trainer import KeypointRcnnTrainer, TrainConv, subpixel_deconv_conv, export_subpixel_deconv


class TubeKeypointRcnnTrainer(KeypointRcnnTrainer):
    """The keypoint R-CNN training step for single-level 3-D bodies with tube heads.  step(), update(), the SGD table, the
    gradient buckets and step_flops() are KeypointRcnnTrainer's; the graph-specific parts are overridden here."""

    def __init__(self, cfg, blobs, spec=None, world=1, buckets=4, lr=None, momentum=None, weight_decay=None):
        torch = L.require_cuda()
        self.torch, self.cfg, self.world = torch, cfg, world
        self.spec = s = spec or P.GraphSpec(cfg)
        assert not s.fpn and s.head3d and s.block == 'basic' and 'roi_conv5_head' in s.roi_head and cfg.MODEL.KEYPOINTS_ON, \
            'TubeKeypointRcnnTrainer: single-level basic-block 3-D bodies with the res5 tube box head and 3-D keypoint head'
        assert s.T_head == s.T, 'TubeKeypointRcnnTrainer: the heads see every frame of the clip (VIDEO.NUM_FRAMES_MID == NUM_FRAMES)'
        self.lr = cfg.SOLVER.BASE_LR if lr is None else lr
        self.momentum = cfg.SOLVER.MOMENTUM if momentum is None else momentum
        self.wd = cfg.SOLVER.WEIGHT_DECAY if weight_decay is None else weight_decay
        self.eng = DetectionEngine(cfg, blobs, s, dtype='bf16')          # frozen stem, tube anchors, feature stride
        self.blobs0 = blobs
        self.T = s.T_head
        self.convs = []                                                   # forward order
        mk = self._mk
        # res3, res4 (ResNet3D.py:59-146 basic_transformation: the stride sits on branch2a's 3x3(x3) conv and on branch1)
        self.stages = []
        dim_in = s.dims[1]
        for si in range(1, len(s.counts)):
            dim_out = s.dims[si + 1]
            self.stages.append([self._basic_block(blobs, 'res%d_%d' % (si + 2, i), dim_in if i == 0 else dim_out, dim_out,
                                                  2 if (i == 0 and dim_in != dim_out) else 1) for i in range(s.counts[si])])
            dim_in = dim_out
        # RPN (model_builder.py:500-563): conv_rpn + the fused per-frame [cls | bbox] 1x1x1 output, padded to 16-byte rows
        A = self.A = s.num_anchors
        self.rpn_conv = mk(blobs, 'conv_rpn', relu=True)
        w = np.concatenate([blobs['rpn_cls_logits_1_w'], blobs['rpn_bbox_pred_1_w']], 0).reshape(5 * A, -1)
        b = np.concatenate([blobs['rpn_cls_logits_1_b'], blobs['rpn_bbox_pred_1_b']], 0)
        self.rpn_ld = (5 * A + 7) // 8 * 8
        self.rpn_out = self._padded_fc(w, b, self.rpn_ld)
        # res5 RoI head (ResNet3D.py:301-327, 340-344): time kernel 1, stride_init = ROI_XFORM_RESOLUTION / 7
        arch = s.roi_head.split('add_')[1].split('_')[0]
        n5, dout = P._BLOCKS[arch][0][3], P._BLOCKS[arch][2][4]
        st5 = int(cfg.FAST_RCNN.ROI_XFORM_RESOLUTION / 7)
        self.res5 = [self._basic_block(blobs, 'res5_%d' % i, dim_in if i == 0 else dout, dout, st5 if (i == 0 and dim_in != dout) else 1)
                     for i in range(n5)]
        C_ = self.C_ = s.num_classes
        w = np.concatenate([blobs['cls_score_1_w'], blobs['bbox_pred_1_w']], 0).reshape(5 * C_, -1)
        b = np.concatenate([blobs['cls_score_1_b'], blobs['bbox_pred_1_b']], 0)
        self.cb_ld = (5 * C_ + 7) // 8 * 8
        self.cls_bbox = self._padded_fc(w, b, self.cb_ld)
        # keypoint head (keypoint_rcnn_heads.add_roi_pose_head_v1convX_3d; deconv per frame, NO_3D_DECONV_TIME_TO_CH)
        self.kps = [mk(blobs, 'conv_fcn%d' % (i + 1), relu=True) for i in range(cfg.KRCNN.NUM_STACKED_CONVS)]
        self.kps_lowres, self.K, self.kp_ld = subpixel_deconv_conv(torch, blobs)
        self.convs.append(self.kps_lowres)
        self.loss_heads = torch.zeros(4, dtype=torch.float32, device='cuda')      # cls, bbox, kps, #correct
        self.totals = torch.zeros(2, dtype=torch.float32, device='cuda')          # live RoIs, keypoint weight sum
        self.rpn_norm = torch.zeros(1, dtype=torch.float32, device='cuda')        # SigmoidCrossEntropyLoss normaliser
        self.iter = 0
        self._alloc_grads(buckets)

    def _basic_block(self, blobs, pre, dim_in, dim_out, stride):
        st = (1, stride, stride)
        return dict(a=self._mk(blobs, pre + '_branch2a', affine=True, stride=st, relu=True),
                    b=self._mk(blobs, pre + '_branch2b', affine=True, relu=True),
                    sc=self._mk(blobs, pre + '_branch1', affine=True, stride=st) if dim_in != dim_out else None)

    def _padded_fc(self, w, b, ld):
        wp = np.zeros((ld, w.shape[1]), np.float32); wp[:w.shape[0]] = w
        bp = np.zeros((ld,), np.float32); bp[:w.shape[0]] = b
        c = TrainConv(self.torch, wp, bias=bp)
        c.cout_live = w.shape[0]
        self.convs.append(c)
        return c

    # ------------------------------------------------------------------ blocks
    @staticmethod
    def _block_forward(blk, x):
        a = blk['a'].forward(x)
        sc = blk['sc'].forward(x) if blk['sc'] is not None else x
        return dict(blk=blk, x=x, a=a, y=blk['b'].forward(a, residual=sc, res_mode=1))

    def _block_backward(self, sb, gzb, gsc, need_dx=True):
        """gzb / gsc: the gradient wrt branch2b's and the shortcut's raw outputs -> the two parts of the input gradient."""
        blk = sb['blk']
        ga, _ = blk['b'].backward(gzb, sb['a'])
        gx1, _ = blk['a'].backward(to.bwd_pointwise(ga, None, sb['a'], blk['a'].scale), sb['x'], need_dx=need_dx)
        gx2 = blk['sc'].backward(gsc, sb['x'], need_dx=need_dx)[0] if blk['sc'] is not None else gsc
        for c in (blk['b'], blk['a'], blk['sc']):
            if c is not None:
                self._bucket_ready(c)
        return gx1, gx2

    def _blocks_backward(self, saved, g1, g2, stop_at_input=False):
        """Backward through a chain of basic blocks from the two parts (g1 + g2) of the gradient wrt its output."""
        for i in range(len(saved) - 1, -1, -1):
            sb = saved[i]
            blk = sb['blk']
            gzb, gsc = to.bwd_pointwise(g1, g2, sb['y'], blk['b'].scale, second=True,
                                        scale2=blk['sc'].scale if blk['sc'] is not None else None)
            g1, g2 = self._block_backward(sb, gzb, gsc, need_dx=not (stop_at_input and i == 0))
        return g1, g2

    # ------------------------------------------------------------------ forward
    def forward_all(self, frames_u8):
        """stem (frozen) -> res3, res4 -> RPN head; returns [the fp32 per-frame RPN output [B, T, H, W, rpn_ld]]."""
        torch, eng = self.torch, self.eng
        B, T, H, W, _ = frames_u8.shape
        assert T == self.T, 'clips of %d frames, the graph is built for %d' % (T, self.T)
        g = eng._geom_tensors(B, H, W)
        x = eng._blob(frames_u8, g['scale'], g['hr'], g['wr'], g['hp'], g['wp'])
        hp, wp = 2 * x.shape[3] - 6, x.shape[4] - 8                           # the even physical blob (engine.body)
        y = cv.conv1_7x7s2(x.view((B * T,) + tuple(x.shape[2:])), eng.conv1_w, (hp, wp), eng.conv1_s, eng.conv1_b, relu=True,
                           dtype=cv.BF16)
        y = dense_ops.maxpool2d(y, 3, 2, 1)
        y = y.view((B, T) + tuple(y.shape[1:]))
        for blk in eng.stages[0]:
            y = eng._run_block(blk, y)
        sv = self.saved = dict(blocks=[])
        for blocks in self.stages:
            for blk in blocks:
                sv['blocks'].append(self._block_forward(blk, y))
                y = sv['blocks'][-1]['y']
        sv['feat'] = y
        h = self.rpn_conv.forward(y)
        o = torch.empty(tuple(h.shape[:4]) + (self.rpn_ld,), dtype=torch.float32, device='cuda')
        self.rpn_out.forward(h, out_f32=True, out=o)
        sv['rpn_h'] = h
        return [o]

    def proposals(self, rpn_outs, im_info):
        """GenerateProposals on tube anchors + tube NMS + collect with the TRAIN settings (engine.rpn_tube's path)."""
        torch, cfg = self.torch, self.cfg
        o = rpn_outs[0]
        B, T, H, W, _ = o.shape
        A, Kp = self.A, int(cfg.TRAIN.RPN_PRE_NMS_TOP_N)
        n = H * W * A
        Kc = n if (Kp <= 0 or Kp > n) else Kp
        props = L.zeros((B, 1, Kc, 4 * T + 1), torch.float32)
        counts = L.zeros((B, 1), torch.int32)
        rpn_ops.rpn_proposals(o[..., :A], o[..., A:5 * A], self.eng.anchors[0], self.eng.feat_stride, im_info, Kp,
                              float(cfg.TRAIN.RPN_MIN_SIZE), T, out=props[:, 0], counts=counts[:, 0], time_major=True)
        post = int(cfg.TRAIN.RPN_POST_NMS_TOP_N)
        keep, nkeep = box_ops.nms_batched(props.view(B, Kc, 4 * T + 1), counts.view(-1), cfg.TRAIN.RPN_NMS_THRESH,
                                          box_ops.NMS_TUBE_GT if T > 1 else box_ops.NMS_2D_GE,
                                          box_ops.ORDER_SCORE if T > 1 else box_ops.ORDER_INDEX, max_keep=post)
        return rpn_ops.collect(props, keep, nkeep, post)

    def make_targets(self, rpn_outs, gt, B, H, W, seed):
        cfg = self.cfg
        g = self._train_geom(B, H, W)
        o = rpn_outs[0]
        rt = target_ops.rpn_targets([(o.shape[2], o.shape[3])], self.eng.anchors, [self.eng.feat_stride], self.A, gt['rpn_boxes'],
                                    gt['rpn_counts'], g['im_info_train'], cfg.TRAIN, seed, gt_visible=gt.get('gt_visible'))
        rois, scores, counts = self.proposals(rpn_outs, g['im_info_train'])
        L.call('dt_memset', L.ptr(self.totals), 0, 8, L.stream_ptr())
        smp = target_ops.sample_rois(rois, scores, counts, gt, g['im_info_train'], cfg, seed, keypoints=True, totals=self.totals)
        return rt, smp

    def forward_heads(self, smp):
        torch, cfg, sv, T = self.torch, self.cfg, self.saved, self.T
        feat = sv['feat']
        f = feat.view((feat.shape[0] * T,) + tuple(feat.shape[2:]))          # frames as images b*T + t
        scale = 1.0 / self.eng.feat_stride
        h = sv['heads'] = dict(f=f, scale=scale)
        # box head
        rois = smp['rois'].view(-1, 4 * T + 1)
        R = rois.shape[0]
        x = dense_ops.roi_align([f], [scale], rois, None, cfg.FAST_RCNN.ROI_XFORM_RESOLUTION, cfg.FAST_RCNN.ROI_XFORM_SAMPLING_RATIO, T=T)
        res5 = []
        for blk in self.res5:
            res5.append(self._block_forward(blk, x))
            x = res5[-1]['y']
        _, _, hh, ww, ch = x.shape
        m = dense_ops.spatial_mean(x.view(R * T, hh, ww, ch))                # [R*T, ch]
        o = torch.empty((1, 1, 1, R * T, self.cb_ld), dtype=torch.float32, device='cuda')
        self.cls_bbox.forward(m.view(1, 1, 1, R * T, ch), out_f32=True, out=o)
        h.update(rois=rois, res5=res5, m=m, o=o)
        # keypoint head
        krois = smp['kp_rois'].view(-1, 4 * T + 1)
        D = krois.shape[0]
        kres = cfg.KRCNN.ROI_XFORM_RESOLUTION
        acts = [dense_ops.roi_align([f], [scale], krois, None, kres, cfg.KRCNN.ROI_XFORM_SAMPLING_RATIO, T=T)]
        for c in self.kps:
            acts.append(c.forward(acts[-1]))
        low = torch.empty((D, T, kres, kres, self.kp_ld), dtype=torch.float32, device='cuda')
        self.kps_lowres.forward(acts[-1], out_f32=True, out=low)                # per frame (kT = 1)
        h.update(krois=krois, kacts=acts, low=low)
        return o.view(R * T, self.cb_ld), low

    # ------------------------------------------------------------------ backward
    def backward_heads(self, smp):
        """Losses + backward of both tube heads; returns the fp32 gradient wrt the res4 feature [B*T, H, W, C]."""
        torch, cfg, sv, T = self.torch, self.cfg, self.saved, self.T
        h = sv['heads']
        dfe = L.zeros(tuple(h['f'].shape), torch.float32)
        w = 1.0 / self.world
        L.call('dt_memset', L.ptr(self.loss_heads), 0, 16, L.stream_ptr())
        # keypoint head (model_builder.py:873-888: LOSS_WEIGHT / NUM_GPUS, NOT divided by T).  Frame t of RoI d is row d*T + t
        # of the per-frame output, and its labels are columns t*K .. t*K+K-1 of the RoI's K*T: both views are [D*T, K].
        low = h['low']
        D, _, S, _, ldk = low.shape
        K = self.K
        g = to.kps_loss_grad(low.view(D * T, S, S, ldk), K, smp['kp_locations'].view(D * T, K), smp['kp_weights'].view(D * T, K),
                             self.totals, cfg.KRCNN.LOSS_WEIGHT * w, ldk, loss=self.loss_heads[2:3])
        acts = h['kacts']
        gh, _ = self.kps_lowres.backward(g.view(D, T, S, S, ldk), acts[-1])
        to.subpixel_grad_fix(self.kps_lowres.g, self.kps_lowres.bias_g, K)
        self._bucket_ready(self.kps_lowres)
        for i in range(len(self.kps) - 1, -1, -1):
            gh, _ = self.kps[i].backward(to.bwd_pointwise(gh, None, acts[i + 1], None), acts[i])
            self._bucket_ready(self.kps[i])
        to.roi_align_bwd(gh, [dfe], [h['scale']], h['krois'], None, S, cfg.KRCNN.ROI_XFORM_SAMPLING_RATIO, T=T)
        # box head (model_builder.py:481-493: SoftmaxWithLoss 1 / NUM_GPUS, SmoothL1Loss 1 / NUM_GPUS / T)
        o = h['o']
        RT = o.shape[3]
        R, C_ = RT // T, self.C_
        go = to.frcnn_tube_loss_grad(o.view(RT, self.cb_ld), smp['labels'].view(-1), smp['bbox_targets'].view(R, 4 * C_ * T),
                                     smp['inside'].view(R, 4 * C_ * T), smp['outside'].view(R, 4 * C_ * T), T, C_, self.totals, w, w / T,
                                     self.cb_ld, loss=self.loss_heads[0:2], accuracy=self.loss_heads[3:4])
        gm, _ = self.cls_bbox.backward(go.view(1, 1, 1, RT, self.cb_ld), h['m'].view(1, 1, 1, RT, -1))
        self._bucket_ready(self.cls_bbox)
        # ReduceBackMean backward fused with res5's last ReLU and AffineChannel gradients
        last = h['res5'][-1]
        y, blk = last['y'], last['blk']
        _, _, hh, ww, ch = y.shape
        gzb, gsc = to.spatial_mean_bwd(gm.view(RT, ch), (hh, ww), y.view(RT, hh, ww, ch), blk['b'].scale, second=True,
                                       scale2=blk['sc'].scale if blk['sc'] is not None else None)
        g1, g2 = self._block_backward(last, gzb.view(y.shape), gsc.view(y.shape))
        g1, g2 = self._blocks_backward(h['res5'][:-1], g1, g2)
        gx = to.bwd_pointwise(g1, g2) if g2 is not None else g1
        res = cfg.FAST_RCNN.ROI_XFORM_RESOLUTION
        to.roi_align_bwd(gx, [dfe], [h['scale']], h['rois'], None, res, cfg.FAST_RCNN.ROI_XFORM_SAMPLING_RATIO, T=T)
        return dfe

    def backward(self, rpn_outs, targets, head_grads=None, fresh=True):
        """targets: [dt_rpn_targets dict]; head_grads: backward_heads' fp32 feature gradient (or None: RPN + trunk only)."""
        sv = self.saved
        if fresh:
            L.call('dt_memset', L.ptr(self.flat_g), 0, self.flat_g.numel() * 4, L.stream_ptr())
            self.reducer.reset()
        L.call('dt_memset', L.ptr(self.loss), 0, 8, L.stream_ptr())
        o = rpn_outs[0]
        B, T = o.shape[:2]
        # add_rpn_losses(time_dim=T): cls 1 / NUM_GPUS (normalised by the valid-label count), bbox 1 / NUM_GPUS / T / batch
        go = to.rpn_tube_loss_grad(o, self.A, targets[0], 1.0 / self.world, 1.0 / self.world / T / B, self.rpn_ld, loss=self.loss,
                                   normalizer=self.rpn_norm)
        gh, _ = self.rpn_out.backward(go, sv['rpn_h'])
        self._bucket_ready(self.rpn_out)
        gfeat, _ = self.rpn_conv.backward(to.bwd_pointwise(gh, None, sv['rpn_h'], None), sv['feat'])
        self._bucket_ready(self.rpn_conv)
        if head_grads is not None:
            gfeat = to.grad_join_f32(head_grads.view(gfeat.shape), gfeat)
        self._blocks_backward(sv['blocks'], gfeat, None, stop_at_input=True)      # res4 -> res3 (res2 is frozen)
        self.reducer.wait()
        return self.loss

    # ------------------------------------------------------------------ weights back to the reference's blob names
    def export_blobs(self, blobs):
        out = self._export_named(blobs)
        for c, names in ((self.rpn_out, ('rpn_cls_logits_1', 'rpn_bbox_pred_1')), (self.cls_bbox, ('cls_score_1', 'bbox_pred_1'))):
            n0 = blobs[names[0] + '_w'].shape[0]
            w, b = c.w[0].cpu().numpy(), c.bias.cpu().numpy()
            out[names[0] + '_w'] = w[:n0].reshape(blobs[names[0] + '_w'].shape)
            out[names[1] + '_w'] = w[n0:c.cout_live].reshape(blobs[names[1] + '_w'].shape)
            out[names[0] + '_b'], out[names[1] + '_b'] = b[:n0].copy(), b[n0:c.cout_live].copy()
        export_subpixel_deconv(self, blobs, out)
        return out
