"""Unit tests of tests/tf_shim (the test-only TensorFlow 1.13 stand-in the reference's graph code runs on).

Every TF op semantic the shim restates is checked here against an independent brute-force statement (python
loops / numpy), so that what the fixtures rest on besides the reference's own source is this list.  The last
tests run the reference's source over the shim where the checkout exists (the build container) and check that
the committed fixture is what it produces.
"""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from tests.golden import make_golden as G

SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tf_shim")
HAVE_REF = os.path.isdir(G.REF)


@pytest.fixture()
def tf():
    saved_path, saved = list(sys.path), {k: v for k, v in sys.modules.items() if k.split(".")[0] == "tensorflow"}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, SHIM)
    mod = importlib.import_module("tensorflow")
    mod.shim_configure("float64")
    mod.shim_reset()
    try:
        yield mod
    finally:
        for k in [k for k in sys.modules if k.split(".")[0] == "tensorflow"]:
            del sys.modules[k]
        sys.modules.update(saved)
        sys.path[:] = saved_path


def test_same_padding_table(tf):
    # SURVEY 8a: the strided layers at 128x416 (asymmetric) and the dilated ones (symmetric)
    assert tf.same_padding(128, 7, 2, 1) == (64, 2, 3)
    assert tf.same_padding(416, 7, 2, 1) == (208, 2, 3)
    assert tf.same_padding(64, 5, 2, 1) == (32, 1, 2)
    assert tf.same_padding(104, 3, 2, 1) == (52, 0, 1)
    assert tf.same_padding(32, 3, 1, 8) == (32, 8, 8)
    assert tf.same_padding(13, 3, 2, 1) == (7, 1, 1)
    assert tf.same_padding(4, 3, 2, 1) == (2, 0, 1)


@pytest.mark.parametrize("stride,rate", [(1, 1), (2, 1), (1, 2), (1, 3)])
def test_slim_conv2d_matches_a_python_loop(tf, stride, rate):
    slim = tf.contrib.slim
    rng = np.random.default_rng(0)
    x, w, b = rng.normal(size=(2, 7, 10, 3)), rng.normal(size=(3, 3, 3, 4)), rng.normal(size=(4,))
    tf.shim_reset(feed={"net/c/weights": w, "net/c/biases": b})
    with tf.variable_scope("net"):
        y = slim.conv2d(tf.constant(x), 4, [3, 3], stride=stride, rate=rate, scope="c", activation_fn=None).numpy()
    Ho, pt, _ = tf.same_padding(7, 3, stride, rate)
    Wo, pl, _ = tf.same_padding(10, 3, stride, rate)
    ref = np.zeros((2, Ho, Wo, 4))
    for n in range(2):
        for oh in range(Ho):
            for ow in range(Wo):
                acc = b.copy()
                for ty in range(3):
                    for tx in range(3):
                        ih, iw = oh * stride + ty * rate - pt, ow * stride + tx * rate - pl
                        if 0 <= ih < 7 and 0 <= iw < 10:
                            acc += x[n, ih, iw] @ w[ty, tx]              # HWIO: [kh, kw, in, out]
                ref[n, oh, ow] = acc
    np.testing.assert_allclose(y, ref, rtol=1e-12, atol=1e-12)
    assert tf.shim_initialised() == [] and tf.shim_unused_feed() == []


def test_dilated_conv_equals_space_to_batch_lowering(tf):
    """TF 1.x lowers rate > 1 to space_to_batch -> VALID conv -> batch_to_space (nn_ops.with_space_to_batch):
    the direct dilated conv of the shim gives the same numbers on the layer shapes of the path."""
    rng = np.random.default_rng(1)
    x, w = torch.tensor(rng.normal(size=(1, 8, 12, 2))), torch.tensor(rng.normal(size=(3, 3, 2, 3)))
    r = 2
    direct = tf._conv2d(x, w, (1, 1), (r, r), "SAME")
    xp = torch.nn.functional.pad(x, (0, 0, r, r, r, r))                    # base paddings ((k-1)*r)//2 = r on both sides
    H, W = xp.shape[1], xp.shape[2]
    out = torch.zeros(1, 8, 12, 3, dtype=torch.float64)
    for py in range(r):
        for px in range(r):
            sub = xp[:, py::r, px::r]                                      # one phase of the space_to_batch split
            y = tf._conv2d(sub, w, (1, 1), (1, 1), "VALID")
            out[:, py::r, px::r] = y[:, : (8 - py + r - 1) // r, : (12 - px + r - 1) // r]
    assert H == 12 and W == 16
    np.testing.assert_allclose(direct.numpy(), out.numpy(), rtol=1e-12, atol=1e-12)


def test_batch_norm_uses_batch_statistics_and_creates_no_biases(tf):
    slim = tf.contrib.slim
    rng = np.random.default_rng(2)
    x, w = rng.normal(size=(3, 5, 6, 2)), rng.normal(size=(1, 1, 2, 4))
    with slim.arg_scope([slim.conv2d], normalizer_fn=slim.batch_norm, activation_fn=None):
        y = slim.conv2d(tf.constant(x), 4, [1, 1], scope="c").numpy()
    names = list(tf.shim_variables())
    assert names == ["c/weights", "c/BatchNorm/beta", "c/BatchNorm/moving_mean", "c/BatchNorm/moving_variance"]
    assert [v.name for v in tf.trainable_variables()] == ["c/weights:0", "c/BatchNorm/beta:0"]
    np.testing.assert_allclose(y.mean((0, 1, 2)), 0, atol=1e-12)
    raw = x @ tf.shim_variables()["c/weights"].numpy()[0, 0]
    want = (raw - raw.mean((0, 1, 2))) / np.sqrt(raw.var((0, 1, 2)) + 1e-3)      # biased variance, epsilon 0.001
    np.testing.assert_allclose(y, want, rtol=1e-10, atol=1e-12)


def test_dense_one_hot_cast_and_leaky_relu(tf):
    k, b = np.arange(6.0).reshape(2, 3), np.array([1.0, 2.0, 3.0])
    tf.shim_reset(feed={"s/fc/kernel": k, "s/fc/bias": b})
    with tf.variable_scope("s"):
        y = tf.layers.dense(tf.constant(np.ones((4, 1, 1, 2))), 3, activation=tf.nn.leaky_relu, name="fc").numpy()
    np.testing.assert_allclose(y[0, 0, 0], [4, 7, 10])
    seg = tf.constant(np.array([0.0, 18.0, 19.0, 255.0, -1.0, 3.9, -0.5]).reshape(1, 7, 1, 1))
    oh = tf.squeeze(tf.one_hot(tf.cast(seg, dtype=tf.int32), depth=19, dtype=tf.float32), -2).numpy()[0, :, 0]
    assert oh.shape == (7, 19)
    assert oh.argmax(-1).tolist() == [0, 18, 0, 0, 0, 3, 0] and oh.sum(-1).tolist() == [1, 1, 0, 0, 0, 1, 1]
    np.testing.assert_allclose(tf.nn.leaky_relu(tf.constant([-2.0, 3.0])).numpy(), [-0.4, 3.0])


def test_tensor_equality_is_identity_and_lists_are_packed(tf):
    a = tf.constant([1.0, 2.0])
    assert (a == 2.0) is False and (a == a) is True                       # TF 1.x Tensor.__eq__
    np.testing.assert_allclose(tf.where(a == 2.0, tf.ones_like(a), a).numpy(), [1, 2])      # flow_utils.py:483
    d = [tf.constant(np.full((1, 2, 2, 1), v)) for v in (1.0, 2.0, 3.0)]
    packed = [t for t in d] + d[0]                                        # davo.py:1109: list + Tensor
    assert isinstance(packed, tf.Tensor) and packed.shape.as_list() == [3, 1, 2, 2, 1]
    np.testing.assert_allclose([float(t.numpy().mean()) for t in packed], [2, 3, 4])
    np.testing.assert_allclose(float(tf.reduce_max([-1, tf.reduce_max(a)]).numpy()), 2.0)   # flow_utils.py:260


def test_variable_scope_reuse_rules_and_collection_prefix(tf):
    with tf.variable_scope("pose_exp_net", reuse=tf.AUTO_REUSE):
        v1 = tf.get_variable("se_flow_near/w", shape=[2])
        with tf.variable_scope("inner"):
            tf.get_variable("w", shape=[1])
            assert tf.get_variable("w", shape=[1]) is tf.get_variable("w", shape=[1])      # AUTO_REUSE is inherited
        with tf.variable_scope("pose_exp_net/seg_channel_weight", reuse=tf.AUTO_REUSE):
            tf.get_variable("weight", shape=(19,))
    assert "pose_exp_net/pose_exp_net/seg_channel_weight/weight" in tf.shim_variables()     # posenn.py:386, davo.py:1392
    with tf.variable_scope("pose_exp_net", reuse=tf.AUTO_REUSE):
        assert tf.get_variable("se_flow_near/w", shape=[2]) is v1
    with tf.variable_scope("pose_exp_net"):
        with pytest.raises(ValueError):
            tf.get_variable("se_flow_near/w", shape=[2])                  # exists, reuse not set
    with tf.variable_scope("pose_exp_net", reuse=True):
        with pytest.raises(ValueError):
            tf.get_variable("never_made", shape=[2])
    got = tf.get_collection(tf.GraphKeys.TRAINABLE_VARIABLES, scope="pose_exp_net/se_flow")
    assert [v.name for v in got] == ["pose_exp_net/se_flow_near/w:0"]     # prefix regex: se_flow_near counts (davo.py:1404)
    assert tf.get_collection(tf.GraphKeys.TRAINABLE_VARIABLES, scope="pose_exp_net/se_seg") == []


def test_avg_pool_same_with_a_window_narrower_than_the_stride(tf):
    x = np.arange(1 * 6 * 20 * 1, dtype=np.float64).reshape(1, 6, 20, 1)
    y = tf.nn.avg_pool(tf.constant(x), ksize=[1, 3, 3, 1], strides=[1, 3, 10, 1], padding="SAME").numpy()
    assert y.shape == (1, 2, 2, 1)
    for i in range(2):
        for j in range(2):
            assert y[0, i, j, 0] == x[0, 3 * i:3 * i + 3, 10 * j:10 * j + 3, 0].mean()
    # a window that overhangs: padded cells are not counted
    y = tf.nn.avg_pool(tf.constant(np.ones((1, 5, 5, 1))), ksize=[1, 3, 3, 1], strides=[1, 2, 2, 1], padding="SAME").numpy()
    np.testing.assert_allclose(y, 1.0)


def test_resize_bilinear_legacy_coordinates(tf):
    x = np.arange(6, dtype=np.float64).reshape(1, 2, 3, 1)
    up = tf.image.resize_bilinear(tf.constant(x), [4, 6]).numpy()[0, :, :, 0]
    np.testing.assert_allclose(up[0], [0, 0.5, 1, 1.5, 2, 2])
    np.testing.assert_allclose(up[:, 0], [0, 1.5, 3, 3])


def test_convert_image_dtype_both_ways(tf):
    u8 = tf.constant(np.array([[0, 1, 128, 255]], np.uint8), dtype=tf.uint8)
    f = tf.image.convert_image_dtype(u8, dtype=tf.float32).numpy()
    np.testing.assert_allclose(f, np.array([[0, 1, 128, 255]]) / 255.0, rtol=1e-15)
    back = tf.image.convert_image_dtype(tf.constant([0.0, 0.5, 0.99, 1.0]), dtype=tf.uint8).numpy()
    assert back.tolist() == [0, 127, 252, 255]                            # cast(x * 255.5)


def test_oracle_agrees_with_reference_fixture_variable_counts():
    gold = np.load(os.path.join(os.path.dirname(G.__file__), "poses.npz"))
    from davo_b200 import synthetic as S
    for key, ver in G.CASES.items():
        assert int(gold[key + "/nvars"]) == len(S.init_weights(ver)), key


@pytest.mark.skipif(not HAVE_REF, reason="reference checkout not on this box")
@pytest.mark.parametrize("key", ["headline", "plain_couple_net", "pix_mix_dispflow", "spp21_flow_net"])
def test_committed_fixture_is_what_the_reference_code_produces(key):
    """Re-runs the reference's graph code for a few cases and compares with the committed fixture, entry by entry."""
    gold = np.load(os.path.join(os.path.dirname(G.__file__), "poses.npz"))
    with G.reference_on_path():
        fresh = G.reference_case(key)
    assert sorted(key + "/" + n for n in fresh) == sorted(n for n in gold.files if n.startswith(key + "/"))
    for name, a in fresh.items():
        np.testing.assert_array_equal(gold[key + "/" + name], a, err_msg=name)


def test_reference_rejects_the_version_strings_the_parser_rejects():
    """davo_b200.version raises the same exception type as the reference's graph code for unbuildable strings: the
    types stored in make_golden.REFERENCE_RAISES (which the generator checks against the reference), and, where the
    checkout exists, a fresh run of the reference."""
    from davo_b200 import version as V
    for ver, exc in G.REFERENCE_RAISES.items():
        with pytest.raises(Exception) as ours:
            V.parse_version(ver)
        assert type(ours.value).__name__ == exc, (ver, ours.value)
    if not HAVE_REF:
        return
    img, flow, seg, depth = G.golden_inputs()
    with G.reference_on_path():
        for ver, exc in G.REFERENCE_RAISES.items():
            with pytest.raises(Exception) as theirs:
                G.run_reference(ver, img[:1, :32, :96 * 3], flow[:1, :, :32, :96], seg[:1, :, :32, :96], depth[:1, :, :32, :96], {})
            assert type(theirs.value).__name__ == exc, (ver, theirs.value)


@pytest.mark.skipif(not HAVE_REF, reason="reference checkout not on this box")
@pytest.mark.parametrize("key", ["headline", "se_seg", "pix_mix_segflow"])
def test_unusual_label_values_through_the_reference_graph(key):
    """Fractions, negative fractions, range edges, huge values, infinities and NaN as labels: the oracle equals the
    reference's graph code (tf.cast truncates; one_hot drops what is outside 0..18, NaN -> INT_MIN included)."""
    from davo_b200 import synthetic as S
    from oracle import davo_oracle as O
    from tests.test_gpu_parity import odd_labels
    ver = G.CASES[key]
    w = S.init_weights(ver, random_bias=True)
    img, flow, seg = S.make_inputs(2, 64, 208, seed=3)
    seg = odd_labels(seg)
    depth = S.make_depth(2, 64, 208)
    with G.reference_on_path():
        ref, _ = G.run_reference(ver, img, flow, seg, depth, w, "float64", "pose")
    mine = O.davo_forward(ver, img, flow, seg, w, torch.float64, depth=depth)
    np.testing.assert_allclose(mine, np.asarray(ref["pose"], np.float64), rtol=1e-9, atol=1e-13)


@pytest.mark.skipif(not HAVE_REF, reason="reference checkout not on this box")
def test_random_version_strings_agree_with_the_reference():
    """tests/golden/fuzz_versions.py, a short run: random strings of the version grammar give the same poses (or the
    same exception type) from the reference's graph code and from version.parse_version + the oracle.  Longer runs
    (thousands of strings) are recorded in DESIGN section 2."""
    sys.path.insert(0, os.path.dirname(G.__file__))
    try:
        import fuzz_versions
    finally:
        sys.path.pop(0)
    bad, summary = fuzz_versions.run(40, seed=3, verbose=False)
    assert not bad, (summary, bad)


@pytest.mark.skipif(not HAVE_REF, reason="reference checkout not on this box")
def test_reference_pose_vec2mat_and_composition_loop_over_the_shim():
    """utils/geo_utils.py:93-119 (TF) executed over the shim == the host geo_utils used for the trajectory."""
    from davo_b200 import geo_utils
    rng = np.random.default_rng(3)
    vec = np.concatenate([rng.normal(0, 0.02, size=(5, 6)), rng.uniform(-4, 4, size=(3, 6))]).astype(np.float32)
    with G.reference_on_path():
        import tensorflow as tf
        from utils import geo_utils as ref_geo
        tf.shim_configure("float32")
        tf.shim_reset()
        want = ref_geo.pose_vec2mat(tf.constant(vec)).numpy()
    got = geo_utils.pose_vec2mat(vec)
    assert np.abs(got - want).max() < 1e-6


@pytest.mark.skipif(not HAVE_REF, reason="reference checkout not on this box")
def test_composition_matches_the_reference_cli_loop_at_random_lengths_and_batches():
    """The same comparison on 16 random (number of samples 1..29, batch size 1..8) draws: the reference's loop executed
    from its source against geo_utils / the oracle on the padded sample list (160 draws were run once, worst 3.5e-6)."""
    from davo_b200 import geo_utils, parallel
    from oracle import davo_oracle as O
    rng = np.random.default_rng(0)
    with G.reference_on_path():
        for _ in range(16):
            N, B = int(rng.integers(1, 30)), int(rng.integers(1, 9))
            p = np.zeros((N, 2, 6), np.float32)
            p[..., :3] = rng.normal(0, 0.02, size=(N, 2, 3))
            p[:, 0, 3:] = rng.normal(0, 0.05, size=(N, 3)) + [0, 0, 0.8]
            p[:, 1, 3:] = rng.normal(0, 0.05, size=(N, 3)) - [0, 0, 0.8]
            want = G.reference_cli_loop(p, B)
            order = parallel.complete_batch_size(list(range(N)), B)
            for fn in (geo_utils.compose_trajectory, O.compose_trajectory):
                got = fn(p[order], B, True)
                assert got.shape == want.shape and np.abs(got - want).max() < 5e-6, (N, B)


@pytest.mark.parametrize("B", [1, 4, 5])
def test_composition_matches_the_reference_cli_loop(B):
    """a14 at batch_size > 1: ``reference_batch_semantics`` reproduces what the reference's loop -- executed from
    its own source by make_golden.reference_cli_loop -- produces for 10 samples (4 pads the list to 12): every sample
    of batch 0 contributes tgt->src0, padding duplicates are composed.  At B = 1 the default is the same thing."""
    from davo_b200 import geo_utils, parallel
    from oracle import davo_oracle as O
    gold = np.load(os.path.join(os.path.dirname(G.__file__), "poses.npz"))
    want = gold["cli_loop/B%d" % B]
    p = G.cli_loop_inputs()
    order = parallel.complete_batch_size(list(range(len(p))), B)
    assert len(want) == 1 + min(B, len(order)) + len(order)
    for fn in (geo_utils.compose_trajectory, O.compose_trajectory):
        got = fn(p[order], B, True)
        assert got.shape == want.shape and np.abs(got - want).max() < 5e-6      # fp32 sin / cos of two libms
    if B == 1:
        assert np.abs(geo_utils.compose_trajectory(p) - want).max() < 5e-6
    else:
        assert len(geo_utils.compose_trajectory(p)) == len(p) + 2               # default: the intended trajectory
    if HAVE_REF:
        with G.reference_on_path():
            np.testing.assert_array_equal(G.reference_cli_loop(p, B), want)
