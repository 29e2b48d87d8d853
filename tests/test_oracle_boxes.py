"""CPU: the oracle restatements vs goldens produced by the reference's own code
(tests/golden/gen_golden.py) and by the compiled reference Cython
(tests/golden/gen_golden_compiled.py).  Integer outputs must be identical; fp32
outputs bit-equal unless a tolerance is stated."""
import numpy as np
import pytest

from oracle import boxes as ob
from oracle import proposals as op


def test_iou_golden(golden):
    g = golden('iou2d')
    assert np.array_equal(ob.bbox_overlaps(g['iou2d_a'], g['iou2d_b']), g['iou2d_out'])
    g = golden('iou3')
    assert np.array_equal(ob.bbox_overlaps(g['iou3_a'], g['iou3_b']), g['iou3_out'])
    g = golden('iou5')
    assert np.array_equal(ob.bbox_overlaps(g['iou5_a'], g['iou5_b']), g['iou5_out'])


def test_iou_vs_compiled_reference(golden):
    g = golden('compiled_ref')
    for i in range(3):                                  # box size scales 0.02, 1, 7
        a = g['iou%d_boxes' % i]
        assert np.array_equal(g['iou%d_out' % i], ob.bbox_overlaps_2d(a[:250], a[250:]))


def test_iou_edge_cases():
    a = np.array([[0, 0, 10, 10], [5, 5, 5, 5], [20, 20, 10, 10]], np.float32)   # last one inverted
    o = ob.bbox_overlaps_2d(a, a)
    assert o[0, 0] == 1.0 and o[1, 1] == 1.0
    assert o[0, 2] == 0.0
    assert ob.bbox_overlaps_2d(a[:0], a).shape == (0, 3)


@pytest.mark.parametrize('name', ['nms2d', 'nms2d_small', 'nmst3', 'nmst2'])
def test_nms_golden(golden, name):
    g = golden(name.split('_')[0])
    d = g[name + '_dets']
    for th in (0.3, 0.5, 0.7):
        keep = np.asarray(ob.nms(d, th), dtype=np.int64)
        assert np.array_equal(keep, g['%s_keep_%d' % (name, int(th * 10))])


def test_nms_vs_compiled_reference(golden):
    g = golden('compiled_ref')
    d = g['nms_dets']
    for th in (0.3, 0.7):
        assert np.array_equal(g['nms_keep_%d' % int(th * 10)], ob.nms_2d(d, th))


def test_nms_empty_and_single():
    assert ob.nms(np.zeros((0, 5), np.float32), 0.5) == []
    assert list(ob.nms(np.array([[0, 0, 5, 5, 0.3]], np.float32), 0.5)) == [0]
    assert ob.nms(np.array([[0, 0, 5, 5, 1, 1, 6, 6, 0.3]], np.float32), 0.5) == [0]


def test_anchors_golden(golden):
    g = golden('anchors')
    # the comment block at lib/modeling/generate_anchors.py:21-39 is a known-answer test; it is
    # MATLAB output (1-based pixels): the python function returns the same windows 0-based (-1).
    kat = np.array([[-83, -39, 100, 56], [-175, -87, 192, 104], [-359, -183, 376, 200],
                    [-55, -55, 72, 72], [-119, -119, 136, 136], [-247, -247, 264, 264],
                    [-35, -79, 52, 96], [-79, -167, 96, 184], [-167, -343, 184, 360]], np.float64) - 1
    assert np.array_equal(op.generate_anchors(16, (128, 256, 512), (0.5, 1, 2)), kat)
    assert np.array_equal(g['anchors_s16'], kat)
    assert np.array_equal(op.generate_anchors(), g['anchors_default'])
    assert np.array_equal(op.generate_anchors(16, (64, 128, 256, 512), (0.5, 1, 2), 3), g['anchors_rpn12_T3'])
    for lvl in range(2, 7):
        a = op.generate_anchors(2. ** lvl, (32 * 2. ** (lvl - 2),), (0.5, 1, 2), 1)
        assert np.array_equal(a, g['anchors_fpn%d' % lvl])


def test_bbox_transform_golden(golden):
    g = golden('xform')
    assert np.array_equal(ob.bbox_transform(g['xform_boxes'], g['xform_deltas'], (10., 10., 5., 5.)), g['xform_out_w10'])
    p = ob.bbox_transform(g['xform_boxes'], g['xform_deltas'], (1., 1., 1., 1.))
    assert np.array_equal(p, g['xform_out_w1'])
    assert np.array_equal(ob.clip_tiled_boxes(p.copy(), np.array([800, 1333], np.float32)), g['xform_clip'])
    g = golden('xformT')
    assert np.array_equal(ob.bbox_transform(g['xformT_boxes'], g['xformT_deltas'], (10., 10., 5., 5.)), g['xformT_out'])


def test_bbox_transform_roundtrip():
    """tests/test_bbox_transform.py:42-54 of the reference: inv o fwd == id (5 decimals)."""
    rng = np.random.default_rng(0)
    x1 = rng.uniform(0, 500, 50); y1 = rng.uniform(0, 400, 50)
    src = np.stack([x1, y1, x1 + rng.uniform(5, 200, 50), y1 + rng.uniform(5, 200, 50)], 1).astype(np.float32)
    dst = (src + rng.normal(0, 5, src.shape)).astype(np.float32)
    w = (10., 10., 5., 5.)
    ew, eh = src[:, 2] - src[:, 0] + 1, src[:, 3] - src[:, 1] + 1
    gw, gh = dst[:, 2] - dst[:, 0] + 1, dst[:, 3] - dst[:, 1] + 1
    d = np.stack([w[0] * ((dst[:, 0] + 0.5 * gw) - (src[:, 0] + 0.5 * ew)) / ew,
                  w[1] * ((dst[:, 1] + 0.5 * gh) - (src[:, 1] + 0.5 * eh)) / eh,
                  w[2] * np.log(gw / ew), w[3] * np.log(gh / eh)], 1).astype(np.float32)
    back = ob.bbox_transform(src, d, w)
    # the forward transform returns x2 = ctr + 0.5*w (no -1), as in the reference test
    np.testing.assert_array_almost_equal(back[:, :2], dst[:, :2], decimal=3)
    np.testing.assert_array_almost_equal(back[:, 2:] - 1, dst[:, 2:], decimal=3)


@pytest.mark.parametrize('name', ['gp2d', 'gp3d'])
def test_generate_proposals_golden(golden, name):
    g = golden(name)
    A = 3 if name == 'gp2d' else 12
    ga = golden('anchors')
    anchors = ga['anchors_fpn5'] if name == 'gp2d' else ga['anchors_rpn12_T3']
    props, sc = op.generate_proposals(g[name + '_scores'][0], g[name + '_deltas'][0], g[name + '_im_info'][0],
                                      anchors, float(g[name + '_stride']), 1000, 300, 0.7, 0)
    rois = g[name + '_rois']
    assert rois.shape[0] == props.shape[0]
    assert np.all(rois[:, 0] == 0)
    assert np.array_equal(rois[:, 1:], props)
    assert np.array_equal(g[name + '_probs'], sc)


@pytest.mark.parametrize('name', ['cd2d', 'cd3d'])
def test_collect_distribute_golden(golden, name):
    g = golden(name)
    rois_l = [g['%s_in_rois%d' % (name, i)] for i in range(5)]
    sc_l = [g['%s_in_scores%d' % (name, i)] for i in range(5)]
    rois = op.collect(rois_l, sc_l, 1000)
    assert np.array_equal(rois, g[name + '_rois'])
    assert np.array_equal(op.map_rois_to_fpn_levels(rois[:, 1:], 2, 5), g[name + '_lvls'])
    _, per_level, restore = op.distribute(rois, 2, 5)
    for i in range(4):
        assert np.array_equal(per_level[i], g['%s_rois_fpn%d' % (name, i + 2)])
    assert np.array_equal(restore, g[name + '_idx_restore'])
    # reference tests/test_batch_permutation_op.py:59-60 identity: concat(levels)[restore] == rois
    assert np.array_equal(np.concatenate(per_level)[restore], rois)


def test_roi_to_batch_format_golden(golden):
    g = golden('r2b')
    assert np.array_equal(op.roi_to_batch_format(g['r2b_in']), g['r2b_out'])


def test_pose_pck_distance_vs_reference_golden():
    """oracle.keypoints.pck_distance / pairwise_kpt_distance against the reference's own functions
    (tests/golden/gen_golden_pose_pck.py): the 'pose-pck' tracking cost, SURVEY §8(f) rank 4."""
    import os
    from oracle import keypoints as okp
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'pose_pck.npz'))
    names = [str(x) for x in g['names']]
    for tag in ('small', 'frame', 'far'):
        a = [x for x in g[tag + '_a']]
        b = [x for x in g[tag + '_b']]
        d = okp.pairwise_kpt_distance(a, b, names)
        assert d.dtype == np.float64 and np.array_equal(d, g[tag + '_dist'])
        heads = np.array([okp.compute_head_size(x, names) for x in a], dtype=np.float64)
        assert np.array_equal(heads, g[tag + '_head'])
    assert g['small_dist'].min() == 0.0 and g['far_dist'].max() > 0.8          # the fixtures span both regimes
