"""Golden vectors of the reference's compiled Cython IoU / NMS (oracle/_ref, built by oracle/build_ref.py) on the
seeded inputs of tests/test_oracle_boxes.py::test_{iou,nms}_vs_compiled_reference.  Needs the reference sources that
oracle/build_ref.py compiles; the .npz is committed so the tests run without them.

    python tests/golden/gen_golden_compiled.py      -> tests/golden/compiled_ref.npz
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


def main():
    from oracle import build_ref
    assert build_ref.build(), 'reference not present'
    from oracle._ref import cython_bbox, cython_nms
    out = {}
    rng = np.random.default_rng(5)
    for i, scale in enumerate((0.02, 1.0, 7.0)):
        x1 = rng.uniform(0, 500, 400); y1 = rng.uniform(0, 300, 400)
        a = np.stack([x1, y1, x1 + rng.uniform(0, 200, 400) * scale, y1 + rng.uniform(0, 200, 400) * scale], 1).astype(np.float32)
        out['iou%d_boxes' % i] = a
        out['iou%d_out' % i] = cython_bbox.bbox_overlaps(a[:250], a[250:])
    rng = np.random.default_rng(7)
    c = rng.uniform(0, 600, (60, 2))
    xy = c[rng.integers(0, 60, 1500)] + rng.normal(0, 12, (1500, 2))
    wh = rng.uniform(20, 120, (1500, 2))
    d = np.hstack([xy, xy + wh, rng.permutation(1500)[:, None] / 1500.]).astype(np.float32)
    out['nms_dets'] = d
    for th in (0.3, 0.7):
        out['nms_keep_%d' % int(th * 10)] = np.asarray(cython_nms.nms(d, np.float32(th)), dtype=np.int64)
    np.savez_compressed(os.path.join(HERE, 'compiled_ref.npz'), **out)
    print('wrote compiled_ref.npz', {k: (v.shape, str(v.dtype)) for k, v in out.items()})


if __name__ == '__main__':
    main()
