"""The front end and the pose head, per element, against the operands they read.

tests/test_conv_stages.py holds every conv layer to an fp64 convolution of what it read.  This file does the same for
the kernels on either side of the conv stack (frontend.cuh), so that every kernel on the pose path is held to its own
operands: front end -> (conv gate) -> head.  Three stages, on the first, a middle and the last unit of the last
micro-batch of every configuration:

(a) ``packed`` (the cnv1 input written by pack8_kernel, pack_kernel, pack_sample_kernel or front_pipeline_kernel)
against a packed tensor rebuilt here from the reference's definitions (davo.py:1115-1450, posenn.py:198) and the class
weights the kernel read (``att_weights:<slot>``, or the static table).  Restated here, not taken from the library:
which frame is target / src0 / src1 and which flow plane belongs to a source (davo.py:978-982); the label rule of
tf.cast (truncation toward zero; NaN, +-inf and everything outside 0..18 has no class); the target map forced to ones
(-se_flow and its pooled variants, ``_wo_tgt``, ``-static``); the masking (-segmask_all: rgb and flow; -segmask_rgb
and ``.555``: rgb only); the depth split with its strict ``<`` (davo.py:1143); and the channel layout of each kernel
(8: tgt rgb, src rgb, src flow; 16: tgt rgb, two zero channels, src rgb, src flow, then residual channels 10-15 that
no cnv1 weight reads; sample units: tgt rgb, src0 rgb, src0 flow, src1 rgb, src1 flow, zeros 13-15).  Two tiers:

  * bit-exact where the arithmetic is a fixed chain of single IEEE operations: class-weight, static and -no_segmask
    maps.  A packed value is rna_tf32(fl32(img_norm(v) * A)) or rna_tf32(fl32(flow * A)), with
    img_norm(v) = fl32(fl32(v * fl32(1/255)) * 2 - 1) (a contraction to fma(t, 2, -1) gives the same bits: 2t is
    exact) and the flow rounded to binary16 first when ``flow_f16`` is on.  numpy float32 reproduces every bit; each
    element (image and flow channels, the channels the layout leaves zero, masked pixels) must be equal.
  * bounded where FMA contraction leaves the order to the compiler: the per-pixel maps sum_i x_i * e_i (-se_rgb,
    -se_depth, -se_disp, -se_mix*).  v = the packed value in fp64 from the device's own excitation e; with S = the sum
    of the magnitudes of the map's n terms and k = 2n the operation count of the chain (n products, n - 1 adds, one
    slack),
        E_A = sum_i |e_i| d_i + k 2^-24 S                    (d_i: error of the SE input x_i, below)
        E   = |c| E_A + 2^-24 |c| (|A| + E_A)                (c: the image or flow value the map multiplies)
        |got - v| <= 2^-11 (|v| + E) + E                     (the conv gate's form: the rna store on top)
    plus the conv gate's summed-offset check (sum sign(v)(got - v) / sum ulp_tf32(v) within +-0.125): a store that
    truncates passes the bound but not the offset.  d_i: -norm_flow takes two fp32 operations with fp32 constants,
    d <= 2^-22 (|flow| + 0.3214) / 15.38; a depth sum, 1 / depth or (d + d_t) / 80 is one or two correctly rounded
    operations, d <= 2^-23 |x|; the image and the one-hot are exact.

(b) ``att_weights:<slot>`` of every slot the variant computes, against fp64 of the slot's frame: the pooling of the
oracle (``se_weights`` / ``spatial_pyramid_pool`` / the one-hot pooling of davo_oracle, pinned to the reference's
code, DESIGN section 2), then both dense layers.  The bound follows the kernels' arithmetic:
  * pooling, per component with mean p and mean magnitude |x|-bar:
        e_p = mean(d) + (L + 1) 2^-24 |x|-bar + 2 * 2^-24 |p|
    mean(d): the per-pixel SE-input error as in (a); L the depth of the kernel's summation tree: se_pool_kernel = the
    per-thread chain (2 adds per flow load, 4 per depth load) + 5 shuffle levels + 8 warp partials + 16 split
    partials; se_spp_kernel / se_segcells_kernel = the lane-strided chain ceil(h*w / 32) + 5 shuffles per cell; the
    last term is fl32(1/n) and the product.  Label counts are exact integers (the L term then only loosens).  rgb sums
    bytes exactly and maps the mean with fl32(1/255), *2, -1: (2/255)(e_bytes + 2 * 2^-24 m) + 2^-24 |p| on top;
    -norm_depth divides by 80: one more 2^-24 |p|; the target's zero flow is the constant se_in(0), error d(0).
  * dense layers:  e_1 = |W1|^T e_p + (D + 1) 2^-24 (|p| |W1| + |b1|);  e_h = e_1 (derivative <= 1 for relu, tanh,
    lrelu) + the activation's own error (tanhf: 2 ulp, 2^-22 |h|; lrelu: the fl32(0.2) constant and the product,
    2^-23 |h|);  e_2 = |W2|^T e_h + (Hd + 1) 2^-24 (|h| |W2| + |b2|);  e_s = e_2 / 4 (sigmoid' <= 1/4) + 2^-21 s
    (expf: 2 ulp, the add and the division: 2^-22 + 2^-24 + 2^-24 <= 2^-21 relative).   |got - s| <= e_s.

(c) the poses written by head_kernel against the channel sums it read: ``cnv7_sum`` (the partials added in the head's
order, so the same fp32 values), m = S / (H7 * W7) with the map proper's size (not the pitched map's), and
v = 0.01 (m . W_pred + b_pred) in fp64.  The fp32 chain: fl32(1/n) and the product (2), 8 lane terms with a product
and an add each (9), 5 shuffle levels (5), then the bias add and the *0.01f (0.01f and the product):
        |got - v| <= 0.01 (16 * 2^-24 sum_c |m_c W_c| + 2^-24 (|m . W| + |b|)) + 2 * 2^-24 |v|.
Each output is looked up where the head must have put it in pose[B, 2, 6] (decouple: rotation | translation per
source; couple: 6 per source; shared nets: one source per unit, by the pair selection; rows a selection does not
compute stay exactly zero).

The CPU self-tests build small inputs that hold every odd label value in source and target planes (at row ends and at
the edges of pack8's 4-pixel groups), distinct class weights and depths exactly at the threshold, and show that a
correct float32 emulation of each kernel passes its tier while each planted bug fails it (the bounded tiers by at
least 10x).  The GPU part prints the worst ratio per (configuration, stage) and holds the set of kernels and
``frame_attention`` branches the configurations reached to every one there is.
"""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

from davo_b200 import synthetic as S
from davo_b200 import version as V
from oracle import davo_oracle as O
from tests.test_conv_stages import OFFSET_BAR, _maps, rna, tf32_clean, ulp_tf32

U = 2.0 ** -24
ODD = np.float32([np.nan, np.inf, -np.inf, -0.5, 18.999, 19.0, 255.0, 1e9, -1e9])
FLOW_C, FLOW_D = 0.32140523, 15.384229        # davo.py:1090, as the oracle writes them
NC = 19
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------ definitions restated --
def pair_of_slot(mode, s):
    """Selection slot -> (sample, source): 0 all, 1 trajectory (tgt->src1), 2 trajectory plus the first tgt->src0,
    3 whole samples (the non-shared nets)."""
    if mode == 0:
        return s >> 1, s & 1
    if mode in (1, 3):
        return s, 1 if mode == 1 else 0
    return (0, 0) if s == 0 else (s - 1, 1)


def tf_labels(seg):
    """tf.cast(seg, int32) followed by one_hot(., 19): truncation toward zero; -1 = no class (NaN, +-inf, < 0 after
    truncation, > 18).  Bytes (the host entry points' narrowed labels) are labels already, 255 = none."""
    s = np.asarray(seg)
    if s.dtype == np.uint8:
        s = s.astype(np.int64)
        return np.where(s <= 18, s, -1)
    s = s.astype(np.float64)
    ok = np.isfinite(s) & (s > -1.0) & (s < 19.0)
    return np.where(ok, np.trunc(np.where(ok, s, 0.0)), -1).astype(np.int64)


def img_norm32(v):
    """davo.py:1519-1522 as the kernels evaluate it in float32."""
    t = np.asarray(v).astype(np.float32) * (np.float32(1.0) / np.float32(255.0))
    return t * np.float32(2.0) - np.float32(1.0)


def flow_q(x):
    """flow_f16: binary16 rounding; values that do not fit a finite half pass through."""
    x = np.asarray(x, np.float32)
    with np.errstate(over="ignore"):
        h = x.astype(np.float16).astype(np.float32)
    return np.where(np.abs(x) < 65520.0, h, x)


def se_in64(v, cfg, axis):
    """SE flow input (davo.py:1087-1102) in fp64 and the error bound of its fp32 evaluation."""
    v = np.asarray(v, np.float64)
    x, d = v, np.zeros_like(v)
    if cfg.flow_norm:
        x = (v - FLOW_C) / FLOW_D
        d = 2.0 ** -22 * (np.abs(v) + FLOW_C) / FLOW_D
    if cfg.flow_abs == V.ABS_BOTH or (cfg.flow_abs == V.ABS_H and axis == 0) or (cfg.flow_abs == V.ABS_V and axis == 1):
        x = np.abs(x)
    return x, d


def se_in32(v, cfg, axis):
    v = np.asarray(v, np.float32)
    if cfg.flow_norm:
        v = (v - np.float32(FLOW_C)) / np.float32(FLOW_D)
    if cfg.flow_abs == V.ABS_BOTH or (cfg.flow_abs == V.ABS_H and axis == 0) or (cfg.flow_abs == V.ABS_V and axis == 1):
        v = np.abs(v)
    return v


def slot_map(cfg, unit_sample, k):
    """Attention-weight slots a unit computes -> (frame plane, weight set): planes 0 src0, 1 tgt, 2 src1; the weight
    set is 0 / 1 = near / far under the depth split, else 0."""
    if cfg.att_src == V.ATT_NONE:
        return {}
    if unit_sample:
        if cfg.depth_split:
            return {0: (0, 0), 1: (0, 1), 2: (2, 0), 3: (2, 1)}
        out = {0: (0, 0), 1: (2, 0)}
        if not cfg.att_tgt_ones:
            out[2] = (1, 0)
        return out
    src = 0 if k == 0 else 2
    if cfg.depth_split:
        return {0: (src, 0), 1: (src, 1)}
    return {0: (src, 0)} if cfg.att_tgt_ones else {0: (src, 0), 1: (1, 0)}


def unit_inputs(img, flow, seg, depth, b, W):
    """Per frame plane f (0 src0, 1 tgt, 2 src1): image [H,W,3] u8, labels, depth, and the flow the frame's SE reads
    (src0: flow[:, 0], src1: flow[:, 1], the target: zeros)."""
    z = np.zeros_like(flow[b, 0])
    return {"img": [img[b][:, f * W:(f + 1) * W] for f in range(3)],
            "lab": [tf_labels(seg[b, f, ..., 0]) for f in range(3)],
            "depth": [None if depth is None else depth[b, f, ..., 0] for f in range(3)],
            "flow": [flow[b, 0], z, flow[b, 1]]}


# --------------------------------------------------------------------------------- (a) the packed input --
def _attention(cfg, u, f, w, w_far, thr, f32, mutate):
    """The attention map of frame f.  Returns (A, E_A): A float32 with E_A None where the map is a table lookup (exact),
    else A in fp64 and its error bound (f32=True: the float32 evaluation, E_A None)."""
    lab = u["lab"][f]
    if mutate == "nan_class0":
        lab = lab.copy()
        lab[u["nan"][f]] = 0
    has = lab >= 0
    li = np.clip(lab, 0, NC - 1)
    w = np.asarray(w, np.float32)
    if not cfg.pixel_map:
        if cfg.depth_split:
            d = u["depth"][f]
            near = d <= thr if mutate == "near_le" else d < thr
            tab = np.where(near, w[li], np.asarray(w_far, np.float32)[li])
        else:
            tab = w[li]
        return np.where(has, tab, np.float32(0)), None
    terms, errs, ws = [], [], []
    if cfg.att_src == V.ATT_SE_RGB_SEG:
        for c in range(3):
            terms.append(img_norm32(u["img"][f][..., c]))
            errs.append(0.0)
            ws.append(w[c])
    elif cfg.att_src == V.ATT_SE_DEPTH_SEG:
        ds, dt = u["depth"][f], u["depth"][1]
        if f32:
            x = (np.float32(1) / ds if cfg.depth_norm == 2 else
                 (ds + dt) / np.float32(80) if cfg.depth_norm == 1 else ds + dt)
            e = 0.0
        else:
            ds64, dt64 = ds.astype(np.float64), dt.astype(np.float64)
            x = 1.0 / ds64 if cfg.depth_norm == 2 else (ds64 + dt64) / 80.0 if cfg.depth_norm == 1 else ds64 + dt64
            e = 2.0 ** -23 * np.abs(x)
        terms.append(x)
        errs.append(e)
        ws.append(w[0])
        if cfg.pixel_map == 2:
            for a in range(2):
                if f32:
                    terms.append(se_in32(u["flow"][f][..., a], cfg, a))
                    errs.append(0.0)
                else:
                    x, e = se_in64(u["flow"][f][..., a], cfg, a)
                    terms.append(x)
                    errs.append(e)
                ws.append(w[1 + a])
    else:                                                   # -se_mixSegFlow: one_hot . e[:19] + SE flow . e[19:]
        cls = np.where(has, w[li], np.float32(0))
        terms.append(cls if f32 else cls.astype(np.float64))
        errs.append(0.0)
        ws.append(np.float32(1))
        for a in range(2):
            if f32:
                terms.append(se_in32(u["flow"][f][..., a], cfg, a))
                errs.append(0.0)
            else:
                x, e = se_in64(u["flow"][f][..., a], cfg, a)
                terms.append(x)
                errs.append(e)
            ws.append(w[NC + a])
    if f32:
        acc = terms[0] * ws[0] if cfg.att_src != V.ATT_SE_SEGFLOW_SEG else terms[0]
        for t, wi in zip(terms[1:], ws[1:]):
            acc = (acc + t * wi).astype(np.float32)
        return acc.astype(np.float32), None
    prods = [np.asarray(t, np.float64) * float(wi) for t, wi in zip(terms, ws)]
    A = sum(prods)
    Sabs = sum(np.abs(p) for p in prods)
    EA = sum(abs(float(wi)) * e for wi, e in zip(ws, errs)) + 2 * len(prods) * U * Sabs
    return A, EA


def _shift_row_ends(u, W):
    """Mutation: the last pixel of every row reads the first pixel of the next row."""
    v = {k: list(x) for k, x in u.items()}
    for key in ("img", "lab", "depth", "flow", "nan"):
        for f in range(3):
            a = v[key][f]
            if a is None:
                continue
            a = a.copy()
            a[:-1, W - 1] = a[1:, 0]
            v[key][f] = a
    return v


def pack_unit(cfg, layout, u, k, slots, static, thr, f32=False, mutate=None):
    """Expected packed tensor of one unit.  layout: 8, 16 (frame-pair units) or "sample".  slots: {slot: weights}
    as read back.  Returns (want [H,W,C] fp64, E [H,W,C]: -1 where the element must be bit-equal, else its bound,
    compared channels).  f32=True: a float32 emulation of the kernel instead (want = its output, E all -1)."""
    H, W = u["lab"][0].shape
    if mutate == "row_end_shift":
        u = _shift_row_ends(u, W)
    if mutate == "swap_rb":
        u = dict(u, img=[x[..., ::-1] for x in u["img"]])
    unit_sample = layout == "sample"

    def table(slot):
        if cfg.att_src == V.ATT_STATIC:
            return static
        return slots[slot]

    ones = (np.ones((H, W), np.float32), None)
    # maps: role -> (A, E_A); roles: "s" (the pair's source) or "s0", "s1"; and "t"
    maps = {}
    src_planes = {"s0": 0, "s1": 2} if unit_sample else {"s": (2 if (k == 1 and mutate != "swap_sources") else 0)}
    if cfg.att_src == V.ATT_NONE:
        for r in list(src_planes) + ["t"]:
            maps[r] = ones
    else:
        for r, f in src_planes.items():
            if unit_sample:
                s = {"s0": 0, "s1": 1}[r] * (2 if cfg.depth_split else 1)
            else:
                s = 0
            far = table(s + 1) if cfg.depth_split else None
            maps[r] = _attention(cfg, u, f, table(s), far, thr, f32, mutate)
        if not cfg.att_tgt_ones:
            ts = 2 if unit_sample else 1
            maps["t"] = _attention(cfg, u, 1, table(ts), None, thr, f32, mutate)
        elif mutate == "tgt_map_not_ones":
            maps["t"] = _attention(cfg, u, 1, table(0), table(1) if cfg.depth_split else None, thr, f32, None)
        else:
            maps["t"] = ones
    mask_rgb = cfg.mask_mode != V.MASK_OFF
    mask_flow = cfg.mask_mode == V.MASK_ALL
    if mutate == "flow_masked":
        mask_flow = mask_rgb
    if mutate == "flow_unmasked":
        mask_flow = False

    def chan(c, role, masked):
        """One packed channel: value c (float32 array) times the role's map (or 1)."""
        A, EA = maps[role] if masked else ones
        if EA is None:
            prod = (c * A.astype(np.float32)).astype(np.float32)
            if mutate == "trunc_store":
                st = (prod.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32).astype(np.float64)
            else:
                st = rna(prod)
            return st, np.full(c.shape, -1.0)
        if f32:
            raise AssertionError("unreachable")
        c64 = c.astype(np.float64)
        v = c64 * A
        E = np.abs(c64) * EA + U * np.abs(c64) * (np.abs(A) + EA)
        return v, E

    rgb = lambda f: [img_norm32(u["img"][f][..., ch]) for ch in range(3)]

    def flows(role):
        f = {"s": src_planes.get("s"), "s0": 0, "s1": 2}[role]
        fl = u["flow"][f]
        if cfg.in_mode != 1:
            fl = np.zeros_like(fl)
        return [fl[..., 0].astype(np.float32), fl[..., 1].astype(np.float32)]

    zero = (np.zeros((H, W)), np.full((H, W), -1.0))
    chans = [chan(c, "t", mask_rgb) for c in rgb(1)]
    if unit_sample:
        for role, f in (("s0", 0), ("s1", 2)):
            chans += [chan(c, role, mask_rgb) for c in rgb(f)]
            chans += [chan(c, role, mask_flow) for c in flows(role)]
        chans += [zero] * 3
        compared = list(range(16))
    else:
        f = src_planes["s"]
        srgb = [chan(c, "s", mask_rgb) for c in rgb(f)]
        sfl = [chan(c, "s", mask_flow) for c in flows("s")]
        if layout == 8:
            chans += srgb + sfl
            compared = list(range(8))
        else:
            chans += [zero, zero] + srgb + sfl + [zero] * 6          # 10-15: residuals no cnv1 weight reads
            compared = list(range(10))
    want = np.stack([c[0] for c in chans], -1)
    E = np.stack([c[1] for c in chans], -1)
    return want, E, compared


class Gate:
    """Per (configuration, stage): mismatches of the exact elements, worst error / bound of the bounded ones, and
    the summed offset in TF32 ulps (sign-aware: a store that truncates pulls every value toward zero)."""

    def __init__(self):
        self.n, self.exact, self.mismatch, self.ratio, self.off_sum, self.off_n, self.where = 0, 0, 0, 0.0, 0.0, 0.0, None

    def add(self, got, want, E, offset=True):
        got = np.asarray(got, np.float64)
        ex = E < 0
        self.n += got.size
        self.exact += int(ex.sum())
        bad = ex & ~((got == want) | (np.isnan(got) & np.isnan(want)))
        self.mismatch += int(bad.sum())
        if bad.any() and self.where is None:
            self.where = ("mismatch", np.argwhere(bad)[0].tolist(), float(got[bad][0]), float(want[bad][0]))
        bd = ~ex
        if bd.any():
            g, v, e = got[bd], want[bd], E[bd]
            if offset:
                r = np.abs(g - v) / np.maximum(2.0 ** -11 * (np.abs(v) + e) + e, 1e-300)
                nz = v != 0
                self.off_sum += float((np.sign(v[nz]) * (g[nz] - v[nz])).sum())
                self.off_n += float(ulp_tf32(v[nz]).sum())
            else:
                r = np.abs(g - v) / np.maximum(e, 1e-300)
            i = int(np.argmax(r))
            if r[i] > self.ratio:
                self.ratio = float(r[i])
                self.where = ("bound", np.argwhere(bd)[i].tolist(), float(g[i]), float(v[i]), float(e[i]))

    @property
    def offset(self):
        return self.off_sum / self.off_n if self.off_n else 0.0

    def ok(self):
        return self.mismatch == 0 and self.ratio <= 1.0 and abs(self.offset) <= OFFSET_BAR

    def as_dict(self):
        return {"n": self.n, "exact": self.exact, "mismatch": self.mismatch, "ratio": self.ratio, "offset": self.offset,
                "where": self.where}


# ------------------------------------------------------------------------------- (b) the SE class weights --
def se_scope(cfg):
    """The SE variables' scope (davo_capi.cu davo_finalize_weights, synthetic.init_weights)."""
    a = cfg.att_src
    if a == V.ATT_SE_FLOW:
        return "se_flow"
    if a == V.ATT_SE_SEG:
        return "se_spp_seg" if cfg.se_pool in V.SPP_SIZES else "se_seg"
    if a == V.ATT_SE_RGB_SEG:
        return "se_rgb"
    if a == V.ATT_SE_DEPTH_SEG:
        if cfg.pixel_map == 2:
            return "se_dispflow" if cfg.depth_norm == 2 else "se_depthflow"
        return "se_disp" if cfg.depth_norm == 2 else "se_depth"
    return "se_spp_segflow" if cfg.se_pool in V.SPP_SIZES else "se_segflow"


def se_kernel(cfg):
    if cfg.att_src in (V.ATT_SE_SEG, V.ATT_SE_SEGFLOW_SEG) and cfg.se_pool != 0:
        return "se_segcells_kernel"
    if cfg.att_src == V.ATT_SE_FLOW and cfg.se_pool >= 2:
        return "se_spp_kernel"
    return "se_pool_kernel"


def se_input(cfg, u, f):
    """The slot's SE input map [H,W,C] in fp64 and its per-pixel error (davo.py:1087-1400)."""
    H, W = u["lab"][0].shape
    onehot = lambda lab: (lab[..., None] == np.arange(NC)).astype(np.float64)
    sflow = lambda: [se_in64(u["flow"][f][..., a], cfg, a) for a in range(2)]
    a = cfg.att_src
    if a == V.ATT_SE_FLOW:
        (x0, d0), (x1, d1) = sflow()
        return np.stack([x0, x1], -1), np.stack([d0, d1], -1)
    if a == V.ATT_SE_SEG:
        return onehot(u["lab"][f]), np.zeros((H, W, NC))
    if a == V.ATT_SE_RGB_SEG:
        return img_norm32(u["img"][f]).astype(np.float64), np.zeros((H, W, 3))
    if a == V.ATT_SE_DEPTH_SEG:
        ds, dt = u["depth"][f].astype(np.float64), u["depth"][1].astype(np.float64)
        x = 1.0 / ds if cfg.depth_norm == 2 else ds + dt         # /80 of -norm_depth: applied to the mean (kernel order)
        chans, errs = [x], [U * np.abs(x)]
        if cfg.pixel_map == 2:
            for x_, d_ in sflow():
                chans.append(x_)
                errs.append(d_)
        return np.stack(chans, -1), np.stack(errs, -1)
    (x0, d0), (x1, d1) = sflow()
    return (np.concatenate([onehot(u["lab"][f]), np.stack([x0, x1], -1)], -1),
            np.concatenate([np.zeros((H, W, NC)), np.stack([d0, d1], -1)], -1))


def pool(cfg, x):
    """The oracle's pooling (davo_oracle.se_weights / spatial_pyramid_pool, attention_module.py:22-86, 137-167)."""
    t = torch.from_numpy(np.ascontiguousarray(x))[None]
    if cfg.se_pool == V.SE_POOL_GP2X2:
        h, w = x.shape[0] // 2, x.shape[1] // 2
        p = torch.cat([t[:, :h, :w].mean(dim=(1, 2)), t[:, :h, w:].mean(dim=(1, 2)),
                       t[:, h:, :w].mean(dim=(1, 2)), t[:, h:, w:].mean(dim=(1, 2))], dim=-1)
    elif cfg.se_pool in V.SPP_SIZES:
        p = O.spatial_pyramid_pool(t, V.SPP_SIZES[cfg.se_pool])
    else:
        p = t.mean(dim=(1, 2))
    return p[0].numpy()


def tree_depth(cfg, H, W):
    """L: the depth of the kernel's summation tree (see the module docstring)."""
    kern = se_kernel(cfg)
    if kern == "se_pool_kernel":
        if cfg.att_src == V.ATT_SE_RGB_SEG:
            return 1 + 5 + 8 + 16
        per_load = 4 if cfg.att_src == V.ATT_SE_DEPTH_SEG else 2
        n4 = H * W // per_load
        iters = -(-(-(-n4 // 16)) // 256)
        return per_load * iters + 5 + 8 + 16
    if cfg.se_pool == V.SE_POOL_GP2X2:
        cell = (H - H // 2) * (W - W // 2)
    else:
        hs = -(-H // min(V.SPP_SIZES[cfg.se_pool]))
        cell = hs * hs
    return -(-cell // 32) + 5


def se_reference(cfg, weights, u, f, wset, H, W):
    """(s, e_s): fp64 excitation of the slot's frame and its bound."""
    x, d = se_input(cfg, u, f)
    p, pa, pd = pool(cfg, x), pool(cfg, np.abs(x)), pool(cfg, d)
    L = tree_depth(cfg, H, W)
    e = pd + (L + 1) * U * pa + 2 * U * np.abs(p)
    if cfg.att_src == V.ATT_SE_RGB_SEG:                     # bytes summed, then fl32(1/255), *2, -1 on the mean
        m = (p + 1.0) * 127.5
        e = (2.0 / 255.0) * ((L + 1) * U * m + 4 * U * m) + U * np.abs(p) + U
    if cfg.att_src == V.ATT_SE_DEPTH_SEG and cfg.depth_norm == 1:
        p = p.copy()
        p[0] /= 80.0
        e = e.copy()
        e[0] = e[0] / 80.0 + U * abs(p[0])
    return dense_reference(cfg, weights, wset, p, e)


def dense_reference(cfg, weights, wset, p, e):
    sc = ("se_flow_near", "se_flow_far")[wset] if cfg.depth_split else se_scope(cfg)
    g = lambda n: np.asarray(weights["pose_exp_net/%s/%s" % (sc, n)], np.float64)
    W1, b1, W2, b2 = g("bottleneck_fc/kernel"), g("bottleneck_fc/bias"), g("recover_fc/kernel"), g("recover_fc/bias")
    z1 = p @ W1 + b1
    e1 = e @ np.abs(W1) + (len(p) + 1) * U * (np.abs(p) @ np.abs(W1) + np.abs(b1))
    if cfg.se_act == V.ACT_TANH:
        h, eh = np.tanh(z1), e1 + 2.0 ** -22 * np.abs(np.tanh(z1))
    elif cfg.se_act == V.ACT_LRELU:
        h = np.where(z1 > 0, z1, 0.2 * z1)
        eh = e1 + 2.0 ** -23 * np.abs(h)
    else:
        h, eh = np.maximum(z1, 0), e1
    z2 = h @ W2 + b2
    e2 = eh @ np.abs(W2) + (len(h) + 1) * U * (np.abs(h) @ np.abs(W2) + np.abs(b2))
    s = 1.0 / (1.0 + np.exp(-z2))
    return s, e2 / 4 + 2.0 ** -21 * s


# ------------------------------------------------------------------------------------------- (c) the head --
def head_reference(S7, n_hw, Wp, bp):
    """S7 [256] channel sums, n_hw the map's pixel count, Wp [256, per], bp [per] -> (v, E) [per]."""
    m = np.asarray(S7, np.float64) / n_hw
    Wp, bp = np.asarray(Wp, np.float64), np.asarray(bp, np.float64)
    dot = m @ Wp
    v = 0.01 * (dot + bp)
    E = 0.01 * (16 * U * (np.abs(m) @ np.abs(Wp)) + U * (np.abs(dot) + np.abs(bp))) + 2 * U * np.abs(v)
    return v, E


def head_emulate(parts, n_hw, Wp, bp, mutate=None):
    """head_kernel in float32: partials added in order, * fl32(1/n), 32 lanes x 8 terms, a 5-level xor shuffle tree,
    + bias, * 0.01f."""
    parts = np.asarray(parts, np.float32)
    if mutate == "drop_partial":
        parts = np.delete(parts, 1, axis=0)
    a = np.zeros(parts.shape[1], np.float32)
    for row in parts:
        a = (a + row).astype(np.float32)
    m = a * (np.float32(1) / np.float32(n_hw))
    Wp = np.asarray(Wp, np.float32)
    out = []
    for j in range(Wp.shape[1]):
        lane = np.zeros(32, np.float32)
        for i in range(256):
            lane[i % 32] = np.float32(lane[i % 32] + np.float32(m[i] * Wp[i, j]))
        for off in (16, 8, 4, 2, 1):
            lane = (lane + lane[np.arange(32) ^ off]).astype(np.float32)
        out.append(np.float32(0.01) * np.float32(lane[0] + np.float32(bp[j])))
    return np.array(out, np.float32)


# ------------------------------------------------------------------------------- CPU self-test: inputs --
def self_inputs(H=12, W=24, seed=3, thr=np.float32(40.03125)):
    """One sample whose label planes hold every odd value at row ends, at both edges of 4-pixel groups and inside,
    in source and target planes; distinct class weights; depths exactly at the threshold."""
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (1, H, 3 * W, 3), dtype=np.uint8)
    flow = rng.normal(0.3, 15.0, (1, 4, H, W, 2)).astype(np.float32)
    seg = rng.integers(0, NC, (1, 3, H, W, 1)).astype(np.float32)
    cols = [W - 1, 0, 3, 4, 7, 8, 11]
    for f in range(3):
        for i, v in enumerate(ODD):
            for j, c in enumerate(cols):
                seg[0, f, (i + f) % H, c, 0] = v
    depth = rng.uniform(1.0, 80.0, (1, 3, H, W, 1)).astype(np.float32)
    depth[rng.random(depth.shape) < 0.2] = thr
    return img, flow, seg, depth, thr


def _assert_odd_coverage(seg, W):
    for f in range(3):
        plane = seg[0, f, ..., 0]
        for v in ODD:
            hit = np.isnan(plane) if np.isnan(v) else plane == v
            assert hit[:, W - 1].any() and hit[:, 0::4].any() and hit[:, 3::4].any(), (f, v)


def _self_unit(img, flow, seg, depth, W):
    u = unit_inputs(img, flow, seg, depth, 0, W)
    u["nan"] = [np.isnan(seg[0, f, ..., 0]) for f in range(3)]
    return u


def _self_weights(cfg, width):
    rng = np.random.default_rng(11)
    base = 0.05 + 0.9 * rng.permutation(np.arange(width)) / width + rng.uniform(0, 1e-3, width)
    return {s: np.float32(base[::-1] if s % 2 else base) for s in range(4)}


SELF_VERSIONS = {
    "headline": "v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh",
    "se_seg_tgt": "v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_seg-fc_tanh",
    "segmask_rgb": "v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_rgb-se_flow-abs_flow-fc_tanh",
    "v1.555": "v1.555-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh",
    "static_tgt": "v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all",
    "depthseg": "v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow_on_depthseg_seplayers_40-abs_flow-fc_tanh",
    "pix_mix_depthflow": "v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_mixDepthFlow-norm_depth-abs_flow-fc_tanh",
    "pix_mix_segflow": "v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_mixSegFlow-abs_flow-norm_flow-fc_tanh",
    "pix_rgb_net": "v1-dilatedPoseNN-cnv6_128-segmask_all-se_rgb-fc_tanh",
    "depthseg_net": "v1-dilatedPoseNN-cnv6_128-segmask_all-se_flow_on_depthseg_seplayers_40-abs_flow-fc_tanh",
}
# (mutation, self configuration, layout, unit k)
PACK_MUTATIONS = [
    ("round_labels", "se_seg_tgt", 8, 1), ("nan_class0", "se_seg_tgt", 8, 1), ("neg_half_no_class", "headline", 8, 0),
    ("255_unmasked", "se_seg_tgt", 16, 1), ("swap_sources", "headline", 8, 1), ("tgt_map_not_ones", "headline", 8, 1),
    ("flow_masked", "segmask_rgb", 8, 1), ("flow_masked", "v1.555", 16, 1), ("flow_unmasked", "headline", 8, 0),
    ("row_end_shift", "headline", 8, 1), ("row_end_shift", "pix_rgb_net", "sample", 0), ("swap_rb", "se_seg_tgt", 16, 0),
    ("swap_rb", "static_tgt", "sample", 0), ("trunc_store", "headline", 8, 1), ("trunc_store", "pix_mix_depthflow", 16, 1),
    ("near_le", "depthseg", 16, 1), ("near_le", "depthseg_net", "sample", 0),
]


def _pack_self(name, layout, k, mutate):
    cfg = V.parse_version(SELF_VERSIONS[name])
    img, flow, seg, depth, thr = self_inputs()
    W = img.shape[2] // 3
    _assert_odd_coverage(seg, W)
    width = NC if not cfg.pixel_map else (3 if cfg.pixel_map == 2 or cfg.att_src == V.ATT_SE_RGB_SEG else
                                          1 if cfg.att_src == V.ATT_SE_DEPTH_SEG else NC + 2)
    slots = _self_weights(cfg, width)
    static = slots[0][:NC]
    u = _self_unit(img, flow, seg, depth, W)
    want, E, ch = pack_unit(cfg, layout, u, k, slots, static, thr)
    if mutate in ("round_labels", "neg_half_no_class", "255_unmasked"):
        rule = {"round_labels": np.round, "neg_half_no_class": np.floor, "255_unmasked": np.trunc}[mutate]
        s = seg[0, :, ..., 0].astype(np.float64)
        with np.errstate(invalid="ignore"):
            t = rule(np.where(np.isfinite(s), s, -5.0))
        if mutate == "255_unmasked":
            t = np.where(t > 18, 18, t)
        lab = np.where((t >= 0) & (t <= 18), t, -1).astype(np.int64)
        u = dict(u, lab=[lab[f] for f in range(3)])
        mutate_k = None
    else:
        mutate_k = mutate
    got, _, _ = pack_unit(cfg, layout, u, k, slots, static, thr, f32=True, mutate=mutate_k)
    g = Gate()
    g.add(got[..., ch], want[..., ch], E[..., ch])
    return g, want, E


@pytest.mark.parametrize("name,layout,k", [(n, l_, k) for n in SELF_VERSIONS for l_, k in ((8, 0), (16, 1), ("sample", 0))
                                           if not (V.parse_version(SELF_VERSIONS[n]).pixel_map and l_ == 8)])
def test_packed_gate_passes_a_correct_kernel(name, layout, k):
    g, want, E = _pack_self(name, layout, k, None)
    assert g.ok(), (name, layout, g.as_dict())
    cfg = V.parse_version(SELF_VERSIONS[name])
    assert (g.exact == g.n) == (not cfg.pixel_map or cfg.mask_mode == V.MASK_OFF), g.as_dict()


@pytest.mark.parametrize("mutation,name,layout,k", PACK_MUTATIONS)
def test_packed_gate_catches_a_subtly_wrong_kernel(mutation, name, layout, k):
    g, _, _ = _pack_self(name, layout, k, mutation)
    if g.exact == g.n or mutation != "trunc_store":
        assert g.mismatch > 0 or g.ratio > 10.0, (mutation, g.as_dict())
    else:                                                   # within the bound, but biased toward zero
        assert g.offset < -OFFSET_BAR, (mutation, g.as_dict())


def test_label_rule_is_tf_cast():
    v = np.float32([np.nan, np.inf, -np.inf, -0.5, -0.999, -1.0, 0.0, 18.999, 19.0, 7.3, 255.0, 1e9, -1e9, 3e38])
    assert tf_labels(v).tolist() == [-1, -1, -1, 0, 0, -1, 0, 18, -1, 7, -1, -1, -1, -1]
    assert tf_labels(np.uint8([0, 18, 19, 255])).tolist() == [0, 18, -1, -1]


# ------------------------------------------------------------------------------ CPU self-test: SE weights --
SE_SELF = {                                       # name -> (version, H, W)
    "flow_gp": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh", 16, 40),
    "flow_gp_norm": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-norm_flow-fc_lrelu", 16, 40),
    "flow_gp2x2": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_gp2x2_flow-abs_flow-fc_tanh", 13, 30),
    "flow_spp864": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_spp_flow-abs_flow-fc_tanh", 14, 30),
    "seg_spp21": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_spp21_seg-fc_tanh", 13, 30),
    "segflow_tgt": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_SegFlow_to_seg-norm_flow-abs_flow-fc_tanh", 16, 40),
    "depth_tgt": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_rgb-se_depth_to_seg-norm_depth-fc_lrelu", 16, 40),
    "rgb": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_rgb_to_seg-fc_tanh", 16, 40),
}
# (mutation, self configuration, frame plane of the slot)
SE_MUTATIONS = [("window_wide", "flow_spp864", 0), ("spp_w_size", "flow_spp864", 0), ("spp_w_size", "seg_spp21", 0),
                ("pad_not_counted", "flow_spp864", 0), ("pad_not_counted", "seg_spp21", 2),
                ("quadrant_up", "flow_gp2x2", 0), ("tgt_flow_nonzero", "segflow_tgt", 1), ("depth_no_tgt", "depth_tgt", 0),
                ("drop_split", "flow_gp", 0), ("drop_split", "rgb", 2)]


def _cells(cfg, H, W, mutate):
    """Pooling windows [(rows, cols, divisor)] as the kernels walk them (with one planted geometry bug)."""
    if cfg.se_pool == V.SE_POOL_GP2X2:
        hh = (H + 1) // 2 if mutate == "quadrant_up" else H // 2
        hw2 = W // 2
        return [(slice(r0, r1), slice(c0, c1), (r1 - r0) * (c1 - c0))
                for r0, r1 in ((0, hh), (hh, H)) for c0, c1 in ((0, hw2), (hw2, W))]
    if cfg.se_pool in V.SPP_SIZES:
        out = []
        for n in V.SPP_SIZES[cfg.se_pool]:
            hs, ws = -(-H // n), -(-W // n)
            cw = ws if mutate == "spp_w_size" else hs + (1 if mutate == "window_wide" else 0)
            for i in range(n):
                for j in range(n):
                    r, c = slice(i * hs, min((i + 1) * hs, H)), slice(j * ws, min(j * ws + cw, W))
                    inside = (r.stop - r.start) * max(c.stop - c.start, 0)
                    out.append((r, c, inside if mutate == "pad_not_counted" else hs * cw))
        return out
    return [(slice(0, H), slice(0, W), H * W)]


def _se_f32(cfg, weights, u, f, mutate):
    """A float32 emulation of the SE kernels: per-cell float32 sums (16 split partials for the global pool), *
    fl32(1/n), the post-ops, then both dense layers and the sigmoid in float32."""
    H, W = u["lab"][0].shape
    if mutate == "tgt_flow_nonzero":
        u = dict(u, flow=[u["flow"][0]] * 3)
    if mutate == "depth_no_tgt":
        u = dict(u, depth=[u["depth"][f], np.zeros_like(u["depth"][1]), u["depth"][2]])
    x = se_input(cfg, u, f)[0].astype(np.float32)
    if cfg.att_src == V.ATT_SE_RGB_SEG:
        x = np.asarray(u["img"][f], np.float32)              # bytes; mapped after the mean
    p = []
    for r, c, n in _cells(cfg, H, W, mutate):
        blk = x[r, c].reshape(-1, x.shape[-1])
        parts = np.array_split(blk, 16) if se_kernel(cfg) == "se_pool_kernel" else [blk]
        if mutate == "drop_split":
            parts = parts[:5] + parts[6:]
        acc = np.zeros(x.shape[-1], np.float32)
        for q in parts:
            acc = (acc + q.sum(0, dtype=np.float32)).astype(np.float32)
        p.append(acc * (np.float32(1) / np.float32(n)))
    p = np.concatenate(p).astype(np.float32)
    if cfg.att_src == V.ATT_SE_RGB_SEG:
        p = p * (np.float32(1) / np.float32(255)) * np.float32(2) - np.float32(1)
    if cfg.att_src == V.ATT_SE_DEPTH_SEG and cfg.depth_norm == 1:
        p[0] = p[0] / np.float32(80)
    sc = se_scope(cfg)
    g = lambda n: np.asarray(weights["pose_exp_net/%s/%s" % (sc, n)], np.float32)
    z1 = p @ g("bottleneck_fc/kernel") + g("bottleneck_fc/bias")
    h = np.tanh(z1) if cfg.se_act == V.ACT_TANH else np.where(z1 > 0, z1, np.float32(0.2) * z1) if cfg.se_act == V.ACT_LRELU \
        else np.maximum(z1, 0)
    z2 = h.astype(np.float32) @ g("recover_fc/kernel") + g("recover_fc/bias")
    return (np.float32(1) / (np.float32(1) + np.exp(-z2.astype(np.float32)))).astype(np.float32)


def _se_self(name, f, mutate):
    ver, H, W = SE_SELF[name]
    cfg = V.parse_version(ver)
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (1, H, 3 * W, 3), dtype=np.uint8)
    flow = rng.normal(0.3, 1.5, (1, 4, H, W, 2)).astype(np.float32)      # SE pools of order 1: no saturated tanh
    seg = rng.integers(0, NC, (1, 3, H, W, 1)).astype(np.float32)
    seg[0, :, :, -1, 0] = 255.0
    depth = rng.uniform(1.0, 80.0, (1, 3, H, W, 1)).astype(np.float32)
    weights = S.init_weights(ver, seed=4, random_bias=True)
    u = _self_unit(img, flow, seg, depth, W)
    s, e = se_reference(cfg, weights, u, f, 0, H, W)
    got = _se_f32(cfg, weights, u, f, mutate)
    r = np.abs(got - s) / e
    return (np.inf if np.isnan(r).any() else float(np.max(r))), cfg


@pytest.mark.parametrize("name", list(SE_SELF))
def test_se_bound_passes_a_correct_kernel(name):
    for f in (0, 1, 2):
        cfg = V.parse_version(SE_SELF[name][0])
        if f == 1 and cfg.att_tgt_ones and cfg.att_src == V.ATT_SE_FLOW:
            continue                                        # no target slot: the target map is ones
        ratio, _ = _se_self(name, f, None)
        assert ratio <= 1.0, (name, f, ratio)


@pytest.mark.parametrize("mutation,name,f", SE_MUTATIONS)
def test_se_bound_catches_a_subtly_wrong_kernel(mutation, name, f):
    ratio, _ = _se_self(name, f, mutation)
    assert ratio > 10.0, (mutation, name, ratio)


def test_se_reference_is_the_oracles():
    """The pooling and dense layers above give what davo_oracle.se_weights gives (fp64, the same inputs)."""
    for name in ("flow_gp", "flow_gp2x2", "flow_spp864", "seg_spp21"):
        ver, H, W = SE_SELF[name]
        cfg = V.parse_version(ver)
        rng = np.random.default_rng(1)
        x = rng.normal(size=(H, W, 2 if cfg.att_src == V.ATT_SE_FLOW else NC))
        w = S.init_weights(ver, seed=4, random_bias=True)
        mode = {V.SE_POOL_GP2X2: "gp2x2"}.get(cfg.se_pool, "spp" if cfg.se_pool in V.SPP_SIZES else "gp")
        act = {V.ACT_TANH: "tanh", V.ACT_LRELU: "lrelu"}.get(cfg.se_act, "relu")
        wt = {k: torch.as_tensor(np.asarray(v), dtype=torch.float64) for k, v in w.items()}
        want = O.se_weights(torch.from_numpy(x)[None], wt, "pose_exp_net/" + se_scope(cfg), act, mode=mode,
                            spp_size=V.SPP_SIZES.get(cfg.se_pool))[0].numpy()
        p = pool(cfg, x)
        got, _ = dense_reference(cfg, w, 0, p, np.zeros_like(p))
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-15)


# ------------------------------------------------------------------------------------ CPU self-test: head --
def _head_self(mutate, hw=(4, 13), pitched=(4, 14)):
    rng = np.random.default_rng(2)
    parts = np.maximum(rng.normal(0.5, 1.0, (28, 256)), 0).astype(np.float32)
    Wp = rng.normal(0, 0.06, (256, 3)).astype(np.float32)
    bp = rng.normal(0, 0.05, 3).astype(np.float32)
    S7 = np.zeros(256, np.float32)
    for row in parts:
        S7 = (S7 + row).astype(np.float32)
    v, E = head_reference(S7, hw[0] * hw[1], Wp, bp)
    n = pitched[0] * pitched[1] if mutate == "pitched_divisor" else hw[0] * hw[1]
    got = head_emulate(parts, n, Wp, bp, mutate if mutate == "drop_partial" else None)
    return float(np.max(np.abs(got - v) / E))


def test_head_bound_passes_a_correct_kernel():
    assert _head_self(None) <= 1.0


@pytest.mark.parametrize("mutation", ["drop_partial", "pitched_divisor"])
def test_head_bound_catches_a_subtly_wrong_kernel(mutation):
    assert _head_self(mutation) > 10.0


# ------------------------------------------------------------------------------------------ the GPU check --
HEADLINE = "v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh"
from tests.golden.make_golden import CASES as G  # noqa: E402

# name -> (version, H, W, batch, environment, options); options: pairs ('all', 'trajectory', 'trajectory_first'),
# entry ('device' triplets, 'host' float labels, 'compact' float16 flow / byte labels, 'sequence' device frames),
# f16 (flow_f16 with values near the binary16 overflow)
CONFIGS = {
    "headline_128x416": (HEADLINE, 128, 416, 2, {}, {}),
    "headline_136x424_traj": (HEADLINE, 136, 424, 2, {}, {"pairs": "trajectory"}),
    "headline_136x200_first": (HEADLINE, 136, 200, 3, {}, {"pairs": "trajectory_first"}),
    "headline_32x64": (HEADLINE, 32, 64, 2, {}, {}),
    "headline_256x832": (HEADLINE, 256, 832, 1, {}, {}),
    "headline_wide0_f16": (HEADLINE, 64, 208, 2, {"DAVO_B200_WIDE": "0"}, {"f16": True}),
    "headline_f16_pack8": (HEADLINE, 64, 208, 2, {}, {"f16": True, "pairs": "trajectory_first"}),
    "headline_front_pipe": (HEADLINE, 128, 416, 2, {"DAVO_B200_FRONT_PIPE": "1"}, {}),
    "headline_fused_front": (HEADLINE, 64, 208, 2, {"DAVO_B200_FUSED_FRONT": "1"}, {}),
    "headline_host": (HEADLINE, 64, 208, 2, {}, {"entry": "host"}),
    "headline_compact": (HEADLINE, 64, 208, 2, {}, {"entry": "compact"}),
    "headline_sequence": (HEADLINE, 64, 208, 3, {}, {"entry": "sequence", "pairs": "trajectory_first"}),
    "segmask_rgb": (G["segmask_rgb"], 64, 208, 2, {}, {}),
    "v1.555": ("v1.555-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh", 64, 200, 2, {}, {}),
    "no_segmask": (G["no_segmask"], 64, 208, 2, {}, {}),
    "static": (G["static"], 64, 208, 2, {}, {}),
    "static_tgt": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all", 136, 200, 2, {}, {"entry": "host"}),
    "v0_lrelu": (G["v0_lrelu"], 64, 208, 2, {}, {"pairs": "trajectory"}),
    "gp2x2_flow": (G["gp2x2_flow"], 136, 200, 2, {}, {}),
    "gp2x2_flow_nobottle": (G["gp2x2_flow_nobottle"], 64, 208, 2, {}, {}),
    "spp864_flow_128": (G["spp864_flow"], 128, 416, 1, {}, {}),
    "spp864_flow_72": (G["spp864_flow"], 72, 232, 2, {}, {}),
    "spp2_flow": ("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_spp2_flow-abs_flow-fc_tanh", 64, 208, 2, {}, {}),
    "spp21_flow_net": (G["spp21_flow_net"], 136, 424, 2, {}, {}),
    "se_seg": (G["se_seg"], 136, 424, 2, {}, {}),
    "se_seg_wo_tgt": (G["se_seg_wo_tgt"], 64, 208, 2, {}, {"entry": "host"}),
    "gp2x2_seg": (G["gp2x2_seg"], 64, 208, 2, {}, {}),
    "spp864_seg_136": (G["spp864_seg"], 136, 200, 2, {}, {}),
    "spp864_seg_72": (G["spp864_seg"], 72, 232, 2, {}, {}),
    "spp21_seg_couple": (G["spp21_seg_couple"], 64, 208, 2, {}, {}),
    "se_rgb_to_seg": (G["se_rgb_to_seg"], 64, 208, 2, {}, {}),
    "se_depth": (G["se_depth"], 64, 208, 2, {}, {}),
    "se_depth_norm_tgt": (G["se_depth_norm_tgt"], 64, 208, 2, {}, {}),
    "se_disp": (G["se_disp"], 64, 208, 2, {}, {}),
    "segflow_to_seg": (G["segflow_to_seg"], 64, 208, 2, {}, {}),
    "segflow_8_wo_tgt": (G["segflow_8_wo_tgt"], 64, 208, 2, {}, {}),
    "pix_rgb": (G["pix_rgb"], 64, 208, 2, {}, {}),
    "pix_depth_wo_tgt": (G["pix_depth_wo_tgt"], 64, 208, 2, {}, {}),
    "pix_disp": (G["pix_disp"], 64, 208, 2, {}, {}),
    "pix_mix_segflow": (G["pix_mix_segflow"], 64, 208, 2, {}, {}),
    "pix_mix_depthflow": (G["pix_mix_depthflow"], 64, 208, 2, {}, {}),
    "pix_mix_dispflow": (G["pix_mix_dispflow"], 64, 208, 2, {}, {}),
    "spp21_mix_segflow": (G["spp21_mix_segflow"], 128, 416, 1, {}, {}),
    "depthseg_seplayers": (G["depthseg_seplayers"], 64, 208, 2, {}, {}),
    "couple_shared": (G["couple_shared"], 64, 208, 2, {}, {"pairs": "trajectory"}),
    "decouple_net": (G["decouple_net"], 64, 208, 2, {}, {}),
    "couple_net_v0": (G["couple_net_v0"], 64, 208, 2, {}, {}),
    "plain_decouple_net": (G["plain_decouple_net"], 128, 416, 2, {}, {}),
    "plain_couple_net": (G["plain_couple_net"], 64, 208, 2, {}, {}),
    "pix_rgb_net": (G["pix_rgb_net"], 64, 208, 2, {}, {}),
    "pix_mix_segflow_net": (G["pix_mix_segflow_net"], 64, 208, 2, {}, {}),
    "pix_mix_depthflow_net": (G["pix_mix_depthflow_net"], 64, 208, 2, {}, {}),
    "pix_disp_wo_tgt_net": (G["pix_disp_wo_tgt_net"], 64, 208, 2, {}, {}),
    "spp21_mix_segflow_net": (G["spp21_mix_segflow_net"], 72, 232, 2, {}, {}),
    "depthseg_seplayers_net": (G["depthseg_seplayers_net"], 64, 208, 2, {}, {}),
    "fuzz_0": ("v1-decay100k-dilatedPoseNN-cnv6_64-segmask_rgb-se_SegFlow_to_seg_wo_tgt-norm_flow-abs_flow_v", 64, 208, 2, {}, {}),
    "fuzz_1": ("v1.555-sharedNN-dilatedCouplePoseNN-cnv6_32-segmask_all-se_seg_wo_tgt-fc_lrelu-abs_flow_h", 64, 208, 2, {}, {}),
    "fuzz_2": ("v0-couplePoseNN-cnv6_256-segmask-se_disp_wo_tgt_to_seg-norm_depth-se_insert", 64, 208, 2, {}, {}),
}
# everything the configurations must reach together
MUST_REACH = (
    {"se_pool_kernel:" + s for s in ("flow", "flow_gp2x2", "seg", "rgb", "depth", "depth_norm", "disp", "segflow",
                                     "mixdepth", "mixdisp")}
    | {"se_spp_kernel:%s" % s for s in ("21", "2", "864")}
    | {"se_segcells_kernel:" + s for s in ("gp2x2_seg", "spp_seg", "spp21_mixsegflow")}
    | {"static", "none", "pack8_kernel", "pack_kernel", "pack_sample_kernel", "front_pipeline_kernel"}
    | {"attention:" + s for s in ("class", "depth_split", "pixel_rgb", "pixel_depth", "pixel_depth_flow", "pixel_segflow")})
STAGES = ("packed", "se", "head")
_RUNS = {}


def _reached(cfg, packed_c, unit_sample, pipe):
    out = set()
    a = cfg.att_src
    if a == V.ATT_NONE:
        out.add("none")
    elif a == V.ATT_STATIC:
        out.add("static")
    else:
        k = se_kernel(cfg)
        if k == "se_spp_kernel":
            out.add("se_spp_kernel:" + "".join(str(n) for n in V.SPP_SIZES[cfg.se_pool]))
        elif k == "se_segcells_kernel":
            out.add("se_segcells_kernel:" + ("gp2x2_seg" if cfg.se_pool == V.SE_POOL_GP2X2 else
                                             "spp21_mixsegflow" if a == V.ATT_SE_SEGFLOW_SEG else "spp_seg"))
        else:
            tag = {V.ATT_SE_FLOW: "flow_gp2x2" if cfg.se_pool else "flow", V.ATT_SE_SEG: "seg", V.ATT_SE_RGB_SEG: "rgb",
                   V.ATT_SE_SEGFLOW_SEG: "segflow"}.get(a)
            if a == V.ATT_SE_DEPTH_SEG:
                tag = ("mixdisp" if cfg.depth_norm == 2 else "mixdepth") if cfg.pixel_map == 2 else \
                    {0: "depth", 1: "depth_norm", 2: "disp"}[cfg.depth_norm]
            out.add("se_pool_kernel:" + tag)
    if a != V.ATT_NONE:
        out.add("attention:" + ("depth_split" if cfg.depth_split else "class" if not cfg.pixel_map else
                                "pixel_rgb" if a == V.ATT_SE_RGB_SEG else "pixel_segflow" if a == V.ATT_SE_SEGFLOW_SEG else
                                "pixel_depth_flow" if cfg.pixel_map == 2 else "pixel_depth"))
    out.add("pack_sample_kernel" if unit_sample else "front_pipeline_kernel" if pipe else
            "pack8_kernel" if packed_c == 8 else "pack_kernel")
    return out


def _inputs(name, cfg, H, W, B, opt, weights):
    rng = np.random.default_rng(zlib.crc32(name.encode()) % 1000)
    seed = int(rng.integers(1000))
    img, flow, seg = S.make_inputs(B, H, W, seed=seed)
    depth = S.make_depth(B, H, W, seed=seed + 1)
    if opt.get("entry") == "sequence":
        img_s, ff, fb, seg_s, depth_s = S.make_sequence(B + 2, H, W, seed=seed)
        seg_s = _odd(seg_s[:, None], rng, W)[:, 0]
        seq = [img_s, ff, fb, seg_s, depth_s]
        from davo_b200.sequence import sequence_to_triplets
        img, flow, seg, depth = sequence_to_triplets(img_s, ff, fb, seg_s, depth_s)
        return img, flow, seg, depth, seq
    seg = _odd(seg, rng, W)
    if cfg.depth_split:
        thr = np.float32(weights["pose_exp_net/se_flow/depth_threshold"])
        d = rng.random(depth.shape)
        depth[d < 0.03] = thr
        depth[(d >= 0.03) & (d < 0.06)] = np.nextafter(thr, np.float32(0))
        depth[(d >= 0.06) & (d < 0.09)] = np.nextafter(thr, np.float32(100))
    if opt.get("f16"):
        near = np.float32([65504.0, 65519.0, -65519.99, 65520.0, -70000.0, 65487.9, 0.000061, -1e-8])
        m = rng.random(flow.shape[:-1]) < 0.002
        flow[m] = near[rng.integers(0, len(near), (int(m.sum()), 2))]
    return img, flow, seg, depth, None


def _odd(seg, rng, W):
    """The odd label values at random places and at row ends and 4-pixel group edges of every plane."""
    seg = seg.copy()
    m = rng.random(seg.shape) < 0.02
    seg[m] = ODD[rng.integers(0, len(ODD), int(m.sum()))]
    B, F, H = seg.shape[:3]
    for b in range(B):
        for f in range(F):
            for i, v in enumerate(ODD):
                for j, c in enumerate((W - 1, 0, 3, 4, W - 4)):
                    seg[b, f, (3 * i + j + f + b) % H, c, 0] = v
    return seg


def _run_subprocess(name):
    code = ("import json, sys; sys.path.insert(0, %r); from tests import test_front_stages as T; "
            "print('RESULT ' + json.dumps(T._run_config(%r, in_process=True)))" % (ROOT, name))
    env = dict(os.environ, **CONFIGS[name][4])
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    line = [x for x in r.stdout.splitlines() if x.startswith("RESULT ")]
    assert r.returncode == 0 and line, r.stderr[-3000:]
    res = json.loads(line[-1][7:])
    res["reached"] = set(res["reached"])
    return res


def _run_config(name, in_process=False):
    """Runs one configuration and checks all three stages; returns {"stats": {stage: Gate dict}, "reached": set,
    "error": str or None, "failures": [str]}."""
    if name in _RUNS:
        return _RUNS[name]
    ver, H, W, B, env, opt = CONFIGS[name]
    if "DAVO_B200_FRONT_PIPE" in env and not in_process:
        res = _RUNS[name] = _run_subprocess(name)         # the knob is read once per process
        return res
    from davo_b200.davo import DAVO
    cfg = V.parse_version(ver)
    weights = S.init_weights(ver, seed=8964, random_bias=True)
    img, flow, seg, depth, seq = _inputs(name, cfg, H, W, B, opt, weights)
    pairs = opt.get("pairs", "all")
    entry = opt.get("entry", "device")
    f16 = bool(opt.get("f16"))
    res = {"stats": {s: Gate() for s in STAGES}, "reached": set(), "error": None, "failures": []}
    with pytest.MonkeyPatch.context() as mp:
        for k, v in env.items():
            mp.setenv(k, v)
        sysm = DAVO(version=ver)
        sysm.setup_inference(H, W, "davo", 3, B, device=0, flow_f16=f16)
        sysm.load_weights(weights)
        cu = lambda x: None if x is None else torch.as_tensor(x).cuda()
        if entry == "sequence":
            out = sysm.inference_sequence(*(cu(x) for x in seq[:4]), depth=cu(seq[4]), pairs=pairs)["pose"]
        elif entry == "host":
            out = sysm.inference(None, "pose", inputs=(img, flow, seg, depth), pairs=pairs)["pose"]
        elif entry == "compact":
            flow16, seg8 = S.compact_inputs(flow, seg)
            out = sysm.inference(None, "pose", inputs=(img, flow16, seg8, depth), pairs=pairs)["pose"]
            flow = np.concatenate([flow16.astype(np.float32), flow[:, 2:]], 1)
        else:
            out = sysm.inference(None, "pose", inputs=tuple(cu(x) for x in (img, flow, seg, depth)), pairs=pairs)["pose"]
    flow_seen = flow_q(flow) if f16 else flow
    unit_sample = cfg.posenn >= V.POSENN_DECOUPLE_DIL
    mode = 3 if unit_sample else {"all": 0, "trajectory": 1, "trajectory_first": 2}[pairs]
    units = B if (unit_sample or mode == 1) else 2 * B if mode == 0 else B + 1
    layout_c = sysm.get_intermediate("packed", 0).size // (H * W)
    layout = "sample" if unit_sample else layout_c
    pipe = "DAVO_B200_FRONT_PIPE" in env and cfg.att_src == V.ATT_SE_FLOW and cfg.se_pool == 0 and layout == 8
    if pipe:
        assert sysm.last_launch_count() == 9, "front_pipeline_kernel did not run"
    res["reached"] = _reached(cfg, layout_c, unit_sample, pipe)
    thr = np.float32(weights["pose_exp_net/se_flow/depth_threshold"]) if cfg.depth_split else None
    static = None
    if cfg.att_src == V.ATT_STATIC:
        static = sysm.get_intermediate("att_weights", 0)
        sw = np.asarray(weights["pose_exp_net/pose_exp_net/seg_channel_weight/weight"], np.float64)
        np.testing.assert_allclose(static, 1 / (1 + np.exp(-sw)), rtol=2.0 ** -21)     # expf, the add, the division
    maps = _maps(cfg, H, W)
    h7, w7 = maps[6][2]
    nbr = 2 if cfg.posenn in (V.POSENN_DECOUPLE_SHARED_DIL, V.POSENN_DECOUPLE_DIL, V.POSENN_DECOUPLE) else 1
    nsrc = 2 if unit_sample else 1
    per = 6 * nsrc // nbr
    pred = lambda br, leaf: np.asarray(weights["pose_exp_net/pose/%spred/%s" % (("rotation/", "translation/")[br] if nbr == 2
                                                                                 else "", leaf)], np.float64)
    written = np.zeros(out.shape, bool)
    check = sorted({0, units - 1} | ({units // 2} if units > 2 else set()))
    for pl in range(units):
        b, k = pair_of_slot(mode, pl)
        # (c) the head
        S7 = sysm.get_intermediate("cnv7_sum", pl).astype(np.float64).reshape(nbr, 256)
        for br in range(nbr):
            v, E = head_reference(S7[br], h7 * w7, pred(br, "weights").reshape(256, per), pred(br, "biases"))
            comps = 6 // nbr
            for j in range(per):
                src = k if nsrc == 1 else j // comps
                comp = br * comps + j % comps
                written[b, src, comp] = True
                res["stats"]["head"].add(np.float64(out[b, src, comp]), np.float64(v[j]), np.float64(E[j]), offset=False)
        if pl not in check:
            continue
        u = unit_inputs(img, flow_seen, seg, depth, b, W)
        smap = slot_map(cfg, unit_sample, k)
        slots = {}
        for s in smap:
            slots[s] = sysm.get_intermediate("att_weights:%d" % s, pl)
        if smap:                                          # plain att_weights: slot 0 (or the static table), 19 wide
            n0 = min(NC, slots[0].size)
            if not np.array_equal(slots[0][:n0], sysm.get_intermediate("att_weights", pl)[:n0]):
                res["failures"].append("att_weights and att_weights:0 differ (unit %d)" % pl)
        try:
            sysm.get_intermediate("att_weights:%d" % len(smap), pl)
            res["failures"].append("att_weights:%d of unit %d was not refused" % (len(smap), pl))
        except RuntimeError as e:
            if "att_weights:%d" % len(smap) not in str(e):
                res["failures"].append("refusal does not name the slot: %s" % e)
        # (b) the SE weights of every live slot
        if cfg.att_src not in (V.ATT_NONE, V.ATT_STATIC):
            for s, (f, wset) in smap.items():
                ref, e = se_reference(cfg, weights, u, f, wset, H, W)
                res["stats"]["se"].add(slots[s].astype(np.float64), ref, e, offset=False)
        # (a) the packed input
        got = sysm.get_intermediate("packed", pl).reshape(H, W, -1)
        want, E, ch = pack_unit(cfg, layout, u, k, slots, static, thr)
        if not tf32_clean(got).all():
            res["failures"].append("unit %d: packed values are not TF32" % pl)
        res["stats"]["packed"].add(got[..., ch].astype(np.float64), want[..., ch], E[..., ch])
    if not unit_sample and mode != 0 and np.any(out[~written] != 0):
        res["failures"].append("rows the selection does not compute are not zero")
    del sysm
    torch.cuda.empty_cache()
    res["stats"] = {s: g.as_dict() for s, g in res["stats"].items()}
    if in_process:
        res["reached"] = sorted(res["reached"])
    _RUNS[name] = res
    return res


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _bad(res):
    out = list(res["failures"])
    for s, st in res["stats"].items():
        if st["mismatch"] or st["ratio"] > 1.0 or abs(st["offset"]) > OFFSET_BAR:
            out.append("%s: %s" % (s, st))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
def test_front_stage_per_element(config):
    _need_gpu()
    res = _run_config(config)
    assert res["error"] is None, res["error"]
    assert not _bad(res), (config, _bad(res))
    assert res["stats"]["head"]["n"] > 0 and res["stats"]["packed"]["n"] > 0


@pytest.mark.gpu
def test_every_front_kernel_and_attention_branch_is_reached(capsys):
    _need_gpu()
    seen, lines = set(), []
    for config in CONFIGS:
        res = _run_config(config)
        seen |= set(res["reached"])
        for s in STAGES:
            st = res["stats"][s]
            if st["n"]:
                lines.append("%-26s %-6s ratio %.4f  offset %+.4f ulp  exact %d / %d, %d mismatch(es)"
                             % (config, s, st["ratio"], st["offset"], st["exact"], st["n"], st["mismatch"]))
    with capsys.disabled():
        print("\nfront stages: largest |error| / bound, summed offset in TF32 ulps, bit-exact elements, per (configuration, stage)")
        print("\n".join(lines))
        print("reached:", sorted(seen))
    missing = MUST_REACH - seen
    assert not missing, sorted(missing)
