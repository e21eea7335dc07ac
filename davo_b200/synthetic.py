"""Synthetic inputs and TF-default random-init weights for the pose path.

There is no dataset or checkpoint offline, so tests, the CLI's ``--synthetic``
mode and ``bench.py`` use seeded stand-ins with the tensor contract of the
reference's input pipeline (reference ``test_kitti_pose.py:104-114``):

    img  uint8   [B, H, 3W, 3]   src0 | tgt | src1 stacked along width
    flow float32 [B, 4, H, W, 2] [src0->tgt, src1->tgt, tgt->src0, tgt->src1]
    seg  float32 [B, 3, H, W, 1] Cityscapes trainIds 0..18 for [src0, tgt, src1]

Weights follow the initialisers the reference graph would use before a
checkpoint is restored, keyed by TF variable name (checkpoint surface):
``slim.conv2d`` -> xavier uniform, zero bias (reference ``nets/posenn.py:205-215``);
``tf.layers.dense`` with ``variance_scaling_initializer()`` -> truncated normal,
stddev sqrt(1.3 * 2 / fan_in), zero bias (``nets/attention_module.py:60-61``);
``seg_channel_weight/weight`` -> N(0, 0.05) (``nets/posenn.py:388-389``).
"""
from __future__ import annotations

import math
from typing import Dict

import numpy as np

from . import version as V

FLOW_MEAN, FLOW_STD = 0.32140523, 15.384229   # dataset statistics, reference davo.py:1090
NUM_CLASSES = 19


def make_inputs(batch: int, height: int = 128, width: int = 416, seed: int = 1234,
                seg_block: int = 16, bad_label_frac: float = 0.0):
    """Seeded (img, flow, seg) with the reference's shapes and dtypes.

    seg is integer-valued, constant over ``seg_block`` x ``seg_block`` pixel blocks;
    ``bad_label_frac`` > 0 overwrites that fraction of pixels with label 255
    (out of range -> attention 0, reference ``davo.py:1115``).
    """
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, size=(batch, height, 3 * width, 3), dtype=np.uint8)
    flow = rng.normal(FLOW_MEAN, FLOW_STD, size=(batch, 4, height, width, 2)).astype(np.float32)
    hb, wb = -(-height // seg_block), -(-width // seg_block)
    blocks = rng.integers(0, NUM_CLASSES, size=(batch, 3, hb, wb), dtype=np.int64)
    seg = np.repeat(np.repeat(blocks, seg_block, axis=2), seg_block, axis=3)[:, :, :height, :width]
    seg = seg.astype(np.float32)
    if bad_label_frac > 0:
        bad = rng.random(size=seg.shape) < bad_label_frac
        seg[bad] = 255.0
    return img, flow, seg[..., None].copy()


def compact_inputs(flow: np.ndarray, seg: np.ndarray):
    """(flow16 [B,2,H,W,2] float16, seg8 [B,3,H,W] uint8): the compact forms ``DAVO.inference`` accepts as an
    extension -- the two flow planes the graph reads (reference davo.py:978-982) in half precision and the labels as
    ``tf.cast(seg, int32)`` (davo.py:1115) clamped to a byte, 255 standing for every label outside 0..18."""
    lab = np.trunc(np.asarray(seg, np.float32)[..., 0])
    seg8 = np.where((lab >= 0) & (lab <= 18), lab, 255).astype(np.uint8)
    return np.ascontiguousarray(np.asarray(flow)[:, 0:2].astype(np.float16)), seg8


def make_depth(batch: int, height: int = 128, width: int = 416, seed: int = 4321) -> np.ndarray:
    """Seeded input_depth [B,3,H,W,1] (metres, 1..80, smooth over 8x8 blocks): [src0, tgt, src1]
    (reference davo.py:991-996); read only by the se_depth attention sources."""
    rng = np.random.default_rng(seed)
    hb, wb = -(-height // 8), -(-width // 8)
    blocks = rng.uniform(1.0, 80.0, size=(batch, 3, hb, wb))
    d = np.repeat(np.repeat(blocks, 8, axis=2), 8, axis=3)[:, :, :height, :width]
    return d.astype(np.float32)[..., None].copy()


def make_sequence(n_frames: int, height: int = 128, width: int = 416, seed: int = 1234, seg_block: int = 16):
    """A seeded frame sequence in the layout of ``DAVO.inference_sequence``: ``(img [N,H,W,3] uint8,
    flow_fwd [N-1,H,W,2] float32, flow_bwd [N-1,H,W,2] float32, seg [N,H,W,1] float32, depth [N,H,W,1] float32)``.
    ``flow_fwd[i]`` stands for the flow from frame i to i+1 and ``flow_bwd[i]`` for the flow from i+1 to i; labels
    are integer-valued over ``seg_block`` x ``seg_block`` blocks, depth (1..80 m) over 8 x 8 blocks, as in
    ``make_inputs`` / ``make_depth``."""
    if n_frames < 3:
        raise ValueError("make_sequence: a sequence has at least 3 frames")
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, size=(n_frames, height, width, 3), dtype=np.uint8)
    flow_fwd = rng.normal(FLOW_MEAN, FLOW_STD, size=(n_frames - 1, height, width, 2)).astype(np.float32)
    flow_bwd = rng.normal(FLOW_MEAN, FLOW_STD, size=(n_frames - 1, height, width, 2)).astype(np.float32)
    hb, wb = -(-height // seg_block), -(-width // seg_block)
    blocks = rng.integers(0, NUM_CLASSES, size=(n_frames, hb, wb), dtype=np.int64)
    seg = np.repeat(np.repeat(blocks, seg_block, axis=1), seg_block, axis=2)[:, :height, :width].astype(np.float32)
    dblocks = rng.uniform(1.0, 80.0, size=(n_frames, -(-height // 8), -(-width // 8)))
    depth = np.repeat(np.repeat(dblocks, 8, axis=1), 8, axis=2)[:, :height, :width].astype(np.float32)
    return img, flow_fwd, flow_bwd, seg[..., None].copy(), depth[..., None].copy()


def _xavier_uniform(rng, shape):
    kh, kw, cin, cout = shape
    lim = math.sqrt(6.0 / (kh * kw * cin + kh * kw * cout))
    return rng.uniform(-lim, lim, size=shape).astype(np.float32)


def _trunc_normal(rng, shape, std):
    out = rng.normal(0.0, std, size=shape)
    bad = np.abs(out) > 2 * std
    while bad.any():
        out[bad] = rng.normal(0.0, std, size=int(bad.sum()))
        bad = np.abs(out) > 2 * std
    return out.astype(np.float32)


def conv_specs(cfg: V.DavoConfig):
    """[(tf scope under pose_exp_net/, HWIO shape)] of decouple_sharednet_v0_dilation
    (posenn.py:189-254) or couple_sharednet_v0_dilation (:133-187)."""
    shared = cfg.posenn in (V.POSENN_DECOUPLE_SHARED_DIL, V.POSENN_COUPLE_SHARED_DIL)
    nsrc = 1 if shared else 2                            # num_source of one evaluation
    cin = (5 if cfg.in_mode == 1 else 3) * (1 + nsrc)    # (rgb [+ flow]) x (tgt + sources)
    c6 = cfg.cnv6_out
    rep = cfg.posenn_se == V.PSE_REPLACE                 # cnv6 := se_block(cnv5): no cnv6 variables, cnv7 reads 256 channels
    specs = [("cnv1", (7, 7, cin, 16)), ("cnv2", (5, 5, 16, 32)), ("cnv3", (3, 3, 32, 64)),
             ("cnv4", (3, 3, 64, 128)), ("cnv5", (3, 3, 128, 256))]
    if cfg.posenn in (V.POSENN_COUPLE_SHARED_DIL, V.POSENN_COUPLE_DIL, V.POSENN_COUPLE):
        return specs + ([] if rep else [("pose/cnv6", (3, 3, 256, c6))]) + [
            ("pose/cnv7", (3, 3, 256 if rep else c6, 256)), ("pose/pred", (1, 1, 256, 6 * nsrc))]
    for br in ("rotation", "translation"):
        specs += ([] if rep else [("pose/%s/cnv6" % br, (3, 3, 256, c6))]) + [
            ("pose/%s/cnv7" % br, (3, 3, 256 if rep else c6, 256)),
            ("pose/%s/pred" % br, (1, 1, 256, 3 * nsrc))]
    return specs


def init_weights(version: str, seed: int = 8964, random_bias: bool = False
                 ) -> Dict[str, np.ndarray]:
    """{tf variable name: ndarray} for ``version`` (seed 8964 = reference train.py:34).

    ``random_bias`` draws biases from N(0, 0.05) instead of TF's zeros, so that
    tests exercise the bias path the way a trained checkpoint would.
    """
    cfg = V.parse_version(version)
    if cfg.posenn not in (V.POSENN_DECOUPLE_SHARED_DIL, V.POSENN_COUPLE_SHARED_DIL, V.POSENN_DECOUPLE_DIL,
                          V.POSENN_COUPLE_DIL, V.POSENN_COUPLE, V.POSENN_DECOUPLE):
        raise NotImplementedError("init_weights: unknown PoseNN kind")
    rng = np.random.default_rng(seed)
    w: Dict[str, np.ndarray] = {}

    def bias(n):
        if random_bias:
            return rng.normal(0.0, 0.05, size=(n,)).astype(np.float32)
        return np.zeros((n,), np.float32)

    for scope, shape in conv_specs(cfg):
        w["pose_exp_net/%s/weights" % scope] = _xavier_uniform(rng, shape)
        if cfg.batch_norm and not scope.endswith("pred"):
            # normalizer_fn=slim.batch_norm (posenn.py:206): no biases; BatchNorm/beta is the only other trainable
            # variable (scale=False), zeros at initialisation
            w["pose_exp_net/%s/BatchNorm/beta" % scope] = bias(shape[3])
        else:
            w["pose_exp_net/%s/biases" % scope] = bias(shape[3])
    se_scopes = {V.ATT_SE_FLOW: ("se_flow", 2, 8), V.ATT_SE_SEG: ("se_seg", 19, 19),
                 V.ATT_SE_RGB_SEG: ("se_rgb", 3, 8), V.ATT_SE_DEPTH_SEG: ("se_depth", 1, 8),
                 V.ATT_SE_SEGFLOW_SEG: ("se_segflow", 21, 19)}
    if cfg.att_src in se_scopes:
        scope, din, dh = se_scopes[cfg.att_src]
        if cfg.att_src == V.ATT_SE_DEPTH_SEG and cfg.depth_norm == 2:
            scope = "se_disp"                            # se(1. / depth, "se_disp", ...) (davo.py:1257)
        if cfg.att_src == V.ATT_SE_DEPTH_SEG and cfg.pixel_map == 2:
            scope, din = ("se_dispflow" if cfg.depth_norm == 2 else "se_depthflow"), 3     # davo.py:1161, 1171
        if cfg.att_src == V.ATT_SE_SEG and cfg.se_pool in V.SPP_SIZES:
            scope = "se_spp_seg"                         # se_spp_block(seg_19, "se_spp_seg", ...) (davo.py:1326)
        if cfg.se_pool == 1:
            din *= 4                                     # gp2x2: four quadrant means concatenated
        elif cfg.se_pool in V.SPP_SIZES:
            din *= sum(n * n for n in V.SPP_SIZES[cfg.se_pool])   # one mean per pyramid cell
        if cfg.se_hidden:
            dh = cfg.se_hidden
        dout = 19
        if cfg.pixel_map:                                # se_block(..., ratio=1): channel -> channel -> channel
            dh = dout = din
            if cfg.att_src == V.ATT_SE_SEGFLOW_SEG and cfg.se_pool in V.SPP_SIZES:   # se_spp_block(concat(seg_19, flow), "se_spp_segflow")
                scope, dh, dout = "se_spp_segflow", 21, 21
                din = 21 * sum(n * n for n in V.SPP_SIZES[cfg.se_pool])
        for name, (fi, fo) in (("bottleneck_fc", (din, dh)), ("recover_fc", (dh, dout))):
            std = math.sqrt(1.3 * 2.0 / fi)
            w["pose_exp_net/%s/%s/kernel" % (scope, name)] = _trunc_normal(rng, (fi, fo), std)
            w["pose_exp_net/%s/%s/bias" % (scope, name)] = bias(fo)
    if cfg.depth_split:
        # davo.py:1137-1140, 1150: two SEs instead of se_flow, and the threshold variable N(15 | the token's number, 0.1)
        for name in ("bottleneck_fc", "recover_fc"):
            for leaf in ("kernel", "bias"):
                t = w.pop("pose_exp_net/se_flow/%s/%s" % (name, leaf))
                w["pose_exp_net/se_flow_near/%s/%s" % (name, leaf)] = t
                w["pose_exp_net/se_flow_far/%s/%s" % (name, leaf)] = (
                    _trunc_normal(rng, t.shape, math.sqrt(1.3 * 2.0 / t.shape[0])) if leaf == "kernel" else bias(t.shape[0]))
        m = __import__("re").search("-se_flow_on_depthseg_.*layers_([0-9.]+)", version)
        w["pose_exp_net/se_flow/depth_threshold"] = np.float32(rng.normal(15.0 if m is None else float(m.group(1)), 0.1))
    if cfg.att_src == V.ATT_STATIC:
        # double scope is the reference's: prefix "pose_exp_net/" inside scope pose_exp_net
        w["pose_exp_net/pose_exp_net/seg_channel_weight/weight"] = \
            rng.normal(0.0, 0.05, size=(19,)).astype(np.float32)
    if cfg.posenn_se in (V.PSE_INSERT, V.PSE_SKIPADD, V.PSE_REPLACE):
        for br in (("rotation/", "translation/") if cfg.posenn in (V.POSENN_DECOUPLE_SHARED_DIL, V.POSENN_DECOUPLE_DIL,
                                                               V.POSENN_DECOUPLE)
                   else ("",)):
            sc = "pose_exp_net/pose/%s%s_se_attention" % (br, "cnv5" if cfg.posenn_se == V.PSE_INSERT else "cnv6")
            for name, (fi, fo) in (("bottleneck_fc", (256, 32)), ("recover_fc", (32, 256))):
                std = math.sqrt(1.3 * 2.0 / fi)
                w["%s/%s/kernel" % (sc, name)] = _trunc_normal(rng, (fi, fo), std)
                w["%s/%s/bias" % (sc, name)] = bias(fo)
    return w
