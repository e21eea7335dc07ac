"""Frame-sequence inputs (``DAVO.inference_sequence``, include/davo_b200.h: davo_forward_sequence).

A sequence of N >= 3 frames holds N-2 samples: sample s is frames (s, s+1, s+2) in the roles (src0, tgt, src1).
``sequence_to_triplets`` is the executable definition of how a sequence maps onto the reference's sample layout.
"""
from __future__ import annotations

import numpy as np


def sequence_to_triplets(img, flow_fwd, flow_bwd, seg, depth=None):
    """The triplet batch (reference test_kitti_pose.py:104-114 layout) that a frame sequence stands for.

    ``img`` uint8 [N,H,W,3], ``flow_fwd`` / ``flow_bwd`` float32 [N-1,H,W,2] (entry i: frame i -> i+1 / frame
    i+1 -> i), ``seg`` float32 [N,H,W,1] or None, ``depth`` float32 [N,H,W,1] or None.  Returns ``(img [B,H,3W,3],
    flow [B,4,H,W,2], seg [B,3,H,W,1] or None, depth [B,3,H,W,1] or None)`` with B = N-2 and, for sample s:

    ====================  =========  ================
    triplet plane         role       sequence source
    ====================  =========  ================
    ``flow[s, 0]``        src0->tgt  ``flow_fwd[s]``
    ``flow[s, 1]``        src1->tgt  ``flow_bwd[s+1]``
    ``flow[s, 2]``        tgt->src0  ``flow_bwd[s]``
    ``flow[s, 3]``        tgt->src1  ``flow_fwd[s+1]``
    ====================  =========  ================

    Image columns and seg / depth planes are frames s, s+1, s+2.  Planes 2 and 3 of the flow are never read by the
    pose graph; they are filled so that the conversion is complete.  ``flow_fwd`` or ``flow_bwd`` may be None (a
    selection that reads no plane of it); its planes are then zeros.
    """
    img = np.asarray(img)
    n = img.shape[0]
    if n < 3:
        raise ValueError("sequence_to_triplets: a sequence has at least 3 frames, got %d" % n)
    b, h, w = n - 2, img.shape[1], img.shape[2]
    trip_img = np.concatenate([img[0:b], img[1:b + 1], img[2:b + 2]], axis=2)
    zeros = np.zeros((n - 1, h, w, 2), np.float32)
    fwd = zeros if flow_fwd is None else np.asarray(flow_fwd, np.float32)
    bwd = zeros if flow_bwd is None else np.asarray(flow_bwd, np.float32)
    for name, f in (("flow_fwd", fwd), ("flow_bwd", bwd)):
        if f.shape != (n - 1, h, w, 2):
            raise ValueError("sequence_to_triplets: %s has shape %s, expected %s" % (name, f.shape, (n - 1, h, w, 2)))
    flow = np.stack([fwd[0:b], bwd[1:b + 1], bwd[0:b], fwd[1:b + 1]], axis=1)

    def planes(x):
        if x is None:
            return None
        x = np.asarray(x, np.float32)
        return np.stack([x[0:b], x[1:b + 1], x[2:b + 2]], axis=1)
    return np.ascontiguousarray(trip_img), np.ascontiguousarray(flow), planes(seg), planes(depth)
