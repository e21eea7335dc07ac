"""sequence_to_triplets (davo_b200.sequence): the executable definition of how a frame sequence maps onto the
reference's sample layout (include/davo_b200.h: davo_forward_sequence).  CPU only."""
import numpy as np
import pytest

from davo_b200 import synthetic as S
from davo_b200.sequence import sequence_to_triplets

H, W = 16, 24


def test_planes_follow_the_table():
    n = 7
    img, fwd, bwd, seg, depth = S.make_sequence(n, H, W, seed=2)
    t_img, flow, t_seg, t_depth = sequence_to_triplets(img, fwd, bwd, seg, depth)
    b = n - 2
    assert t_img.shape == (b, H, 3 * W, 3) and t_img.dtype == np.uint8
    assert flow.shape == (b, 4, H, W, 2) and t_seg.shape == (b, 3, H, W, 1) and t_depth.shape == (b, 3, H, W, 1)
    for s in range(b):
        for f in range(3):                                 # src0, tgt, src1 = frames s, s+1, s+2
            assert np.array_equal(t_img[s, :, f * W:(f + 1) * W], img[s + f])
            assert np.array_equal(t_seg[s, f], seg[s + f]) and np.array_equal(t_depth[s, f], depth[s + f])
        assert np.array_equal(flow[s, 0], fwd[s])          # src0 -> tgt
        assert np.array_equal(flow[s, 1], bwd[s + 1])      # src1 -> tgt
        assert np.array_equal(flow[s, 2], bwd[s])          # tgt -> src0
        assert np.array_equal(flow[s, 3], fwd[s + 1])      # tgt -> src1


def test_two_frame_overlapping_pieces_give_the_whole_conversion():
    n = 12
    seq = S.make_sequence(n, H, W, seed=3)
    whole = sequence_to_triplets(*seq)
    for cut in (3, 5, 10):                                 # piece 1: frames [0, cut); piece 2: [cut - 2, n)
        a = sequence_to_triplets(*(x[:cut] for x in seq[:1]), seq[1][:cut - 1], seq[2][:cut - 1],
                                 seq[3][:cut], seq[4][:cut])
        b = sequence_to_triplets(seq[0][cut - 2:], seq[1][cut - 2:], seq[2][cut - 2:], seq[3][cut - 2:], seq[4][cut - 2:])
        for x, y, z in zip(whole, a, b):
            assert np.array_equal(np.concatenate([y, z]), x)


def test_absent_flow_and_bad_shapes():
    img, fwd, bwd, seg, _ = S.make_sequence(4, H, W, seed=4)
    _, flow, _, depth = sequence_to_triplets(img, None, bwd, seg)
    assert depth is None and not flow[:, 0].any() and not flow[:, 3].any() and np.array_equal(flow[:, 1], bwd[1:])
    with pytest.raises(ValueError):
        sequence_to_triplets(img[:2], fwd[:1], bwd[:1], seg[:2])
    with pytest.raises(ValueError):
        sequence_to_triplets(img, fwd[:2], bwd, seg)


def test_make_sequence_is_seeded():
    a, b = S.make_sequence(5, H, W, seed=9), S.make_sequence(5, H, W, seed=9)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    img, fwd, bwd, seg, depth = a
    assert img.shape == (5, H, W, 3) and fwd.shape == bwd.shape == (4, H, W, 2) and seg.shape == depth.shape == (5, H, W, 1)
    assert seg.min() >= 0 and seg.max() <= 18 and np.all(seg == np.trunc(seg))
