"""CPU: the host side of the tube keypoint R-CNN training step — argument validation of its C-ABI entry points (before any
CUDA call, reported through dt_last_error()), pack_gt on tube entries, and the seeded synthetic tube ground truth of
tools/train_net.py."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest

from detectandtrack_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


_TUBE_CASES = [
    ('dt_rpn_tube_loss_grad', (None, 48, None, None, None, None, 2, 3, 8, 10, 15, 1.0, 1.0, 1.0 / 9, None, None, 48, None, None), b'ld_o=48'),
    ('dt_rpn_tube_loss_grad', (None, 80, None, None, None, None, 2, 9, 8, 10, 15, 1.0, 1.0, 1.0 / 9, None, None, 80, None, None), b'T=9'),
    ('dt_rpn_tube_loss_grad', (None, 80, None, None, None, None, 2, 3, 8, 10, 15, 1.0, 1.0, 1.0 / 9, None, None, 80, None, None), b'null pointer'),
    ('dt_frcnn_tube_loss_grad', (None, 16, None, None, None, None, 4, 0, 2, None, 1.0, 1.0, None, 16, None, None, None), b'T=0'),
    ('dt_frcnn_tube_loss_grad', (None, 8, None, None, None, None, 4, 3, 2, None, 1.0, 1.0, None, 16, None, None, None), b'ld_o=8'),
    ('dt_frcnn_tube_loss_grad', (None, 16, None, None, None, None, 4, 3, 2, None, 1.0, 1.0, None, 16, None, None, None), b'null pointer'),
    ('dt_spatial_mean_bwd', (None, 4, 7, 7, 12, None, None, None, None, None, None), b'C=12'),
    ('dt_spatial_mean_bwd', (None, 4, 7, 7, 512, None, None, None, None, None, None), b'null pointer'),
]


@pytest.mark.parametrize('name,args,msg', _TUBE_CASES)
def test_tube_loss_entry_points_reject_bad_arguments(name, args, msg):
    rc = getattr(L.lib(), name)(*args)
    assert rc != 0
    assert msg in L.lib().dt_last_error()
    with pytest.raises(RuntimeError):
        L.call(name, *args)


def _train3d_header_functions():
    src = open(os.path.join(ROOT, 'include', 'dt_b200_train3d.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return set(re.findall(r'\b(dt_[a-z0-9_]+)\s*\(', src))


def test_train3d_table_matches_its_header_and_the_library_exports_it():
    names = _train3d_header_functions()
    assert names == set(L.TRAIN3D_SIGNATURES), (names, set(L.TRAIN3D_SIGNATURES))
    assert not names & (set(L.SIGNATURES) | set(L.HOST_FUNCS))
    lib = ctypes.CDLL(L.LIB_PATH)
    assert all(hasattr(lib, n) for n in names)


def test_every_train3d_entry_point_has_an_error_case():
    assert set(L.TRAIN3D_SIGNATURES) == {c[0] for c in _TUBE_CASES}


def _tube_entries(T=3, K=17):
    rng = np.random.RandomState(0)
    out = []
    for g in (2, 3):
        boxes = np.tile(rng.uniform(0, 50, (g, 4)).astype(np.float32), (1, T))
        kps = rng.randint(0, 50, (g, 3, K * T)).astype(np.int32)
        out.append(dict(boxes=boxes, gt_keypoints=kps, is_crowd=np.array([False] + [True] + [False] * (g - 2)),
                        gt_visible=np.ones((g, T), np.uint8) * np.arange(g)[:, None] % 2))
    return out


def test_pack_gt_tubes_shapes_and_rpn_alignment():
    from detectandtrack_b200.modeling.trainer import pack_gt
    e = _tube_entries()
    gt = pack_gt(e, device='cpu')
    assert tuple(gt['boxes'].shape) == (2, 8, 12) and tuple(gt['rpn_boxes'].shape) == (2, 8, 12)
    assert tuple(gt['keypoints'].shape) == (2, 8, 3, 51) and tuple(gt['gt_visible'].shape) == (2, 8, 3)
    assert gt['gt_visible'].dtype.is_floating_point is False and gt['gt_visible'].element_size() == 1
    assert gt['counts'].tolist() == [2, 3] and gt['rpn_counts'].tolist() == [1, 2]       # crowd tubes are not RPN gt
    np.testing.assert_array_equal(gt['boxes'][1, :3].numpy(), e[1]['boxes'])
    np.testing.assert_array_equal(gt['keypoints'][1, :3].numpy(), e[1]['gt_keypoints'])
    keep = [0, 2]                                                                          # non-crowd rows of clip 1
    np.testing.assert_array_equal(gt['rpn_boxes'][1, :2].numpy(), e[1]['boxes'][keep])
    np.testing.assert_array_equal(gt['gt_visible'][1, :2].numpy(), e[1]['gt_visible'][keep])


def test_pack_gt_2d_output_unchanged():
    """2-D entries: the same keys, shapes and values as before tubes were accepted (no visibility tensor)."""
    from detectandtrack_b200.modeling.trainer import pack_gt
    rng = np.random.RandomState(1)
    boxes = rng.uniform(0, 50, (3, 4)).astype(np.float32)
    kps = rng.randint(0, 50, (3, 3, 17)).astype(np.int32)
    gt = pack_gt([dict(boxes=boxes, gt_keypoints=kps, is_crowd=np.array([False, True, False]))], device='cpu')
    assert set(gt) == {'boxes', 'classes', 'crowd', 'keypoints', 'counts', 'rpn_boxes', 'rpn_counts'}
    exp_b = np.zeros((1, 8, 4), np.float32); exp_b[0, :3] = boxes
    exp_r = np.zeros((1, 8, 4), np.float32); exp_r[0, :2] = boxes[[0, 2]]
    exp_k = np.zeros((1, 8, 3, 17), np.int32); exp_k[0, :3] = kps
    np.testing.assert_array_equal(gt['boxes'].numpy(), exp_b)
    np.testing.assert_array_equal(gt['rpn_boxes'].numpy(), exp_r)
    np.testing.assert_array_equal(gt['keypoints'].numpy(), exp_k)
    assert gt['classes'].numpy().tolist() == [[1, 1, 1, 0, 0, 0, 0, 0]] and gt['crowd'].numpy().tolist() == [[0, 1, 0, 0, 0, 0, 0, 0]]
    assert gt['counts'].tolist() == [3] and gt['rpn_counts'].tolist() == [2]
    assert gt['boxes'].dtype == gt['rpn_boxes'].dtype and str(gt['keypoints'].dtype) == 'torch.int32'


def _train_net():
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    try:
        import train_net
    finally:
        sys.path.pop(0)
    return train_net


def test_synthetic_tube_gt_is_deterministic_and_inside_the_frame():
    tn = _train_net()
    entry = dict(seed=1000003 * 2 + 5, height=96, width=128)
    a, b = tn._synthetic_gt(entry, 17, T=3), tn._synthetic_gt(entry, 17, T=3)
    assert a['boxes'].shape == (3, 12) and a['gt_keypoints'].shape == (3, 3, 51)
    np.testing.assert_array_equal(a['boxes'], b['boxes'])
    np.testing.assert_array_equal(a['gt_keypoints'], b['gt_keypoints'])
    tub = a['boxes'].reshape(3, 3, 4)
    assert tub[..., 0::2].min() >= 0 and tub[..., 0::2].max() <= 127 and tub[..., 1::2].max() <= 95
    assert np.all(tub[..., 2] > tub[..., 0]) and np.all(tub[..., 3] > tub[..., 1])
    assert not np.array_equal(tub[:, 0], tub[:, 1])                                       # per-frame jitter
    for t in range(3):                                                                     # keypoints inside their frame's box
        k = a['gt_keypoints'][:, :, t * 17:(t + 1) * 17]
        assert np.all(k[:, 0] >= np.floor(tub[:, t, 0:1])) and np.all(k[:, 0] <= tub[:, t, 2:3] + 1)
    # T == 1 draws are exactly the 2-D ones (same stream, same shapes)
    one = tn._synthetic_gt(entry, 17)
    assert one['boxes'].shape == (3, 4) and one['gt_keypoints'].shape == (3, 3, 17)
    np.testing.assert_array_equal(one['boxes'], tn._synthetic_gt(entry, 17, T=1)['boxes'])
