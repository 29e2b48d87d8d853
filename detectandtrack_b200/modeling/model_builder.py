"""``model_builder.create`` with the reference's signature (lib/modeling/model_builder.py:52-61).

The reference resolves MODEL.TYPE to a graph-building function and returns a
DetectionModelHelper holding Caffe2 nets (``net``, ``conv_body_net``, ``keypoint_net``).
Here the returned object is a ``DetectionModel`` wrapping the B200 ``DetectionEngine``; the
three "nets" are methods on it with the same split the reference makes for inference
(:179-306): bbox net (body + RPN + box head), conv-body net, keypoint net.
"""
import logging

from ..core.config import cfg
from . import params as P

logger = logging.getLogger(__name__)

_GENERIC_TYPES = ('keypoint_rcnn', 'mask_rcnn', 'faster_rcnn', 'fast_rcnn', 'generalized_rcnn')


class DetectionModel(object):
    """Stand-in for DetectionModelHelper at inference time."""

    def __init__(self, name, train, blobs, spec, dtype):
        from .engine import DetectionEngine
        self.name = name
        self.train = train
        self.num_classes = cfg.MODEL.NUM_CLASSES
        self.blobs = blobs
        self.spec = spec
        self.engine = DetectionEngine(cfg, blobs, spec, dtype=dtype)
        self.params = list(blobs.keys())

    # the reference's net split, as callables
    def conv_body_net(self, frames_u8):
        return self.engine.forward_features(frames_u8)

    def net(self, frames_u8):
        return self.engine.detect(frames_u8)

    def keypoint_net(self, feats2d, boxes, batch_idx, im_scale):
        return self.engine.keypoint_head(feats2d, boxes, batch_idx, im_scale)


def create(model_name, train=False, init_params=None, blobs=None, dtype=None):
    """model_name is cfg.MODEL.TYPE.  ``init_params`` keeps the reference's meaning (random
    initialisation even at test time); weights are then overwritten from cfg.TEST.WEIGHTS by
    test_engine.initialize_model_from_cfg, exactly like the reference's two-step init."""
    if train:
        # the training graph of the reference (:52-61 with train=True, build_data_parallel_model :908-951) is the trainer
        # object: forward / device-side targets / losses / backward / all-reduce / SGD in its .step()
        from . import trainer as T
        import os
        if blobs is None:
            blobs, spec = (P.load_weights_file(cfg, cfg.TRAIN.WEIGHTS) if cfg.TRAIN.WEIGHTS else P.random_blobs(cfg))
        else:
            spec = P.GraphSpec(cfg)
        world = int(os.environ.get('WORLD_SIZE', '1'))
        if model_name == 'rpn':
            return T.RpnTrainer(cfg, blobs, spec, world=world)
        if model_name == 'keypoint_rcnn' and cfg.MODEL.FASTER_RCNN and cfg.MODEL.KEYPOINTS_ON:
            if spec.head3d:                                   # single-level 3-D body with tube heads
                from .tube_trainer import TubeKeypointRcnnTrainer
                return TubeKeypointRcnnTrainer(cfg, blobs, spec, world=world)
            return T.KeypointRcnnTrainer(cfg, blobs, spec, world=world)
        raise NotImplementedError('training graph for MODEL.TYPE {!r}'.format(model_name))
    if model_name not in _GENERIC_TYPES:
        raise NotImplementedError('MODEL.TYPE {!r}'.format(model_name))
    if cfg.MODEL.MASK_ON:
        raise NotImplementedError('Handle tubes..')          # as lib/core/test.py:917
    if not cfg.MODEL.FASTER_RCNN:
        raise NotImplementedError('precomputed-proposal models are not on the hot path')
    if blobs is None:
        blobs, spec = P.random_blobs(cfg)
    else:
        spec = P.GraphSpec(cfg)
    return DetectionModel(model_name, train, blobs, spec, dtype or cfg.TEST.PRECISION)
