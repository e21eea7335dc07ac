"""Every conv kernel plan, per element, against an fp64 convolution of the operands the kernel actually read.

The pose tests see the conv stack through spatial means: an error confined to one border column, one partial tile
or the second CTA of an odd cluster is divided by the map size before it reaches a pose.  Here each stored layer of
each plan is read back with the input it read (``<layer>:in``), the TF32 weights its pack was built from
(``<layer>:w<g>``) and its bias (``<layer>:b``), and compared element by element with

    y = b + sum a*w        s = |b| + sum |a|*|w|            (float64, explicit TF-SAME asymmetric padding)

The operands are TF32 values (10-bit mantissas), so every product is exact in float64 and y is exact to fp64.
Geometry (kernel, stride, dilation, padding) comes from the net type and ``oracle.davo_oracle.tf_same_pad``, never
from the library's planner.

Bound of a stored layer, n = the layer's full K (taps x input channels of a group):

    E = (n + 2) * 2^-22 * s                |got - relu(y)| <= 2^-11 * (|y| + E) + E

E allows two fp32 ulps (2^-23 relative) per accumulated term, measured against s: enough for a tensor-core adder
that truncates instead of rounding (its exact behaviour on sm_100 is not documented).  2^-11 * (|y| + E) is the
round-to-nearest (``cvt.rna.tf32``) store.  One missing tap at one pixel, a padding column read as data, a skipped
32-channel slab, a shifted output pixel or a missing bias move an element by far more (the CPU self-test below
builds each of these mutations and shows it fails).

Two properties the bound cannot see, checked on their own:
  * TF32 storage: every stored activation has its low 13 bits zero (``kind::tf32`` truncates whatever it is
    given, DESIGN section 3);
  * no offset: over the elements with relu(y) > 0, sum (got - y) / sum ulp_tf32(y) lies within +-0.125.
    Round-to-nearest gives about 0, a truncating store about -0.5: the one error that survives the poses' spatial
    mean and builds up along a trajectory (DESIGN section 5).  The errors are summed before dividing: a mean of
    per-element ratios is dominated by the few elements whose sum nearly cancels (|y| << s), where the accumulation
    error is many ulps of y: on a B200 that mean measured +0.14 to +0.24 in configurations whose summed offset is
    within 0.005.

The cnv7 sum epilogue (no TF32 rounding, conv_pm.cuh) is held per branch and channel to
    |sum7 - sum_p relu(y_p)| <= sum_p E_p + (P + 2) * 2^-22 * sum_p (relu(|y_p|) + E_p),   P = pixels of the map.

-batch_norm (bn.cuh): layer = rna(relu((x - mu) * r + beta)) with x = the fp32 conv sums, mu and the biased variance
over the layer's call group in fp64 (the shared nets' two PoseNN calls: pairs with the same source index), r =
1 / sqrt(var + 1e-3).  With Ex = E of an element, Em = the largest E of the group's channel, sigma = sqrt(var):
    the stored mean carries |mu_f - mu| <= Em + 2^-24 |mu|  (the group mean of the x errors, then one float rounding);
    the variance of the fp32 sums moves by at most 2 sigma Em + Em^2, so r moves by at most
    dr = r * ((sigma Em + Em^2 / 2) / (var + eps) + 2^-23)  (plus one float rounding of rstd);
    the three fp32 ops of bn_apply_kernel add 2^-22 (|x - mu| r + |beta|).
    D = r (Ex + Em + 2^-24 |mu|) + |x - mu| dr + 2^-22 (|x - mu| r + |beta|)
    |got - relu(z)| <= 2^-11 (|z| + D) + D,   z = (x - mu) r + beta in fp64.
cnv7 is stored there as the plain conv sums (the raw epilogue): |got - y| <= E.

The largest error / bound ratio per (configuration, layer) and the offset are printed at the end of the GPU run,
together with the set of kernel plans the configurations reached; that set must contain every branch of
``launch_conv`` (davo_capi.cu).
"""
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from davo_b200 import synthetic as S
from oracle.davo_oracle import tf_same_pad

U11, U22, U23, U24 = 2.0 ** -11, 2.0 ** -22, 2.0 ** -23, 2.0 ** -24
OFFSET_BAR = 0.125
NAMES = ("cnv1", "cnv2", "cnv3", "cnv4", "cnv5", "cnv6", "cnv7")
# (k, stride, dilation) per layer, reference nets/posenn.py: the dilated nets (:12-254) and the original stride-2 nets
# (:257-378), where -se_skipadd runs cnv6 at stride 1 (:292, :355)
GEO_DILATED = ((7, 2, 1), (5, 2, 1), (3, 1, 2), (3, 1, 4), (3, 1, 8), (3, 1, 2), (3, 2, 1))
GEO_V0 = ((7, 2, 1), (5, 2, 1), (3, 2, 1), (3, 2, 1), (3, 2, 1), (3, 2, 1), (3, 2, 1))
GEO_V0_SKIPADD = GEO_V0[:5] + ((3, 1, 1), (3, 2, 1))


# ---------------------------------------------------------------------------------------------- the checker --
def rna(x):
    """cvt.rna.tf32.f32 of the float32 value of x, as float64."""
    u = np.asarray(x, np.float32).view(np.uint32)
    return ((u + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32).astype(np.float64)


def tf32_clean(x32):
    """True where a float32 value is a TF32 value (low 13 mantissa bits zero)."""
    return (np.asarray(x32, np.float32).view(np.uint32) & np.uint32(0x1FFF)) == 0


def ulp_tf32(y):
    a = np.maximum(np.abs(y), np.finfo(np.float32).tiny)
    return np.exp2(np.floor(np.log2(a)) - 10)


def ref_conv(a, w, b, k, stride, dil):
    """a [H,W,C], w [k,k,C,Co], b [Co] -> (y, s) [Ho,Wo,Co], float64, TF-SAME padding."""
    H, W_, _ = a.shape
    _, pt, pb = tf_same_pad(H, k, stride, dil)
    _, pl, pr = tf_same_pad(W_, k, stride, dil)
    x = F.pad(torch.from_numpy(np.asarray(a, np.float64)).permute(2, 0, 1)[None], (pl, pr, pt, pb))
    wt = torch.from_numpy(np.asarray(w, np.float64)).permute(3, 2, 0, 1).contiguous()
    bt = torch.from_numpy(np.asarray(b, np.float64))
    y = F.conv2d(x, wt, bt, stride=stride, dilation=dil)
    s = F.conv2d(x.abs(), wt.abs(), bt.abs(), stride=stride, dilation=dil)
    return y[0].permute(1, 2, 0).numpy(), s[0].permute(1, 2, 0).numpy()


def accum_allowance(s, n):
    """E: two fp32 ulps per accumulated term of a K = n reduction, against s = |b| + sum |a||w|."""
    return (n + 2) * U22 * s


class Stat:
    """Worst error / bound ratio and the offset statistic of one (configuration, layer)."""

    def __init__(self):
        self.ratio, self.off_sum, self.off_n, self.n = 0.0, 0.0, 0, 0

    def add(self, got, z, D, rounded=True, relu=True):
        """got: stored values; z: exact pre-activation (fp64); D: allowance on z before the store (rounded: the
        rna store on top; relu=False: the raw epilogue, plain sums)."""
        got = np.asarray(got, np.float64)
        want = np.maximum(z, 0.0) if relu else z
        bound = (U11 * (np.abs(z) + D) + D) if rounded else D
        r = np.abs(got - want) / np.maximum(bound, 1e-300)
        worst = int(np.argmax(r))
        if r.flat[worst] > self.ratio:
            self.ratio, self.where = float(r.flat[worst]), np.unravel_index(worst, r.shape)
        self.n += got.size
        if rounded:
            pos = want > 0
            self.off_sum += float((got[pos] - z[pos]).sum())
            self.off_n += float(ulp_tf32(z[pos]).sum())

    @property
    def offset(self):
        """sum (got - y) / sum ulp_tf32(y) over relu(y) > 0: the mean error in units of the mean TF32 ulp."""
        return self.off_sum / self.off_n if self.off_n else 0.0


# ------------------------------------------------------------------------------------ CPU self-test: the gate --
def _trunc_add(acc32, v64):
    """fp32 add that truncates toward zero."""
    exact = acc32.astype(np.float64) + v64
    r = exact.astype(np.float32)
    over = np.abs(r.astype(np.float64)) > np.abs(exact)
    r[over] = np.nextafter(r[over], np.float32(0))
    return r


def simulated_kernel(a, w, b, k, stride, dil, seed=0, mutate=None, store="rna", tile=(16, 8)):
    """A conv layer the way a tensor-core kernel evaluates it, on the CPU: output tiles of 16 x 8 pixels (partial
    ones at the right and bottom border); per tile the K axis (tap-major, then channel) goes in 8-wide k-steps in a
    shuffled order, each k-step's products summed exactly and added to an fp32 accumulator that TRUNCATES; then the
    bias (truncating add), relu and the store (``rna``, ``trunc`` or ``none``).  ``mutate`` plants one kernel bug."""
    rng = np.random.default_rng(seed)
    H, W_, C = a.shape
    Co = w.shape[3]
    Ho, pt, pb = tf_same_pad(H, k, stride, dil)
    Wo, pl, pr = tf_same_pad(W_, k, stride, dil)
    x = np.pad(np.asarray(a, np.float64), ((pt, pb), (pl, pr), (0, 0)))
    if mutate == "pad_neighbour":              # a SAME padding column read as the neighbouring data column
        if pl > 0:
            x[:, pl - 1] = x[:, pl]
        else:
            x[:, pl + W_] = x[:, pl + W_ - 1]
    cols = np.stack([x[ty * dil: ty * dil + stride * (Ho - 1) + 1: stride, tx * dil: tx * dil + stride * (Wo - 1) + 1: stride]
                     for ty in range(k) for tx in range(k)], axis=2).reshape(Ho, Wo, k * k * C)
    K = cols.shape[2]
    wk = np.asarray(w, np.float64).reshape(K, Co)
    tiles = [(r0, c0) for r0 in range(0, Ho, tile[0]) for c0 in range(0, Wo, tile[1])]
    last = tiles[-1]                           # bottom-right tile: partial whenever the map is not a tile multiple
    if mutate == "drop_tap":                   # last tap of border pixel (0, 0) (in bounds there: it reads data)
        cols[0, 0, (k * k - 1) * C:] = 0.0
    if mutate == "skip_slab":                  # the 32-wide slab around the centre tap, in one (partial) tile
        s0 = ((k * k // 2) * C // 32) * 32
        cols[last[0]:last[0] + tile[0], last[1]:last[1] + tile[1], s0:s0 + 32] = 0.0
    out = np.zeros((Ho, Wo, Co), np.float32)
    bias = np.asarray(b, np.float64).copy()
    if mutate == "no_bias":
        bias[int(np.argmax(np.abs(bias)))] = 0.0
    for r0, c0 in tiles:
        blk = cols[r0:r0 + tile[0], c0:c0 + tile[1]]
        th, tw = blk.shape[:2]
        blk = blk.reshape(th * tw, K)
        acc = np.zeros((th * tw, Co), np.float32)
        for ks in rng.permutation(K // 8):
            acc = _trunc_add(acc, blk[:, 8 * ks:8 * ks + 8] @ wk[8 * ks:8 * ks + 8])
        acc = _trunc_add(acc, bias[None, :])
        out[r0:r0 + th, c0:c0 + tw] = np.maximum(acc, 0).reshape(th, tw, Co)
    if mutate == "shift_pixel":                # one pixel of the partial tile written one column to the right
        r, c = last[0], last[1]
        out[r, c + 1] = out[r, c]
    if store == "rna":
        return rna(out).astype(np.float32)
    if store == "trunc":
        return (out.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
    return out


# (name, input H, W, C, output channels, k, stride, dilation): every layer geometry of the two net families on small
# maps with borders and partial tiles, the odd stride-2 maps of the original nets (7 x 13 -> 4 x 7) included
SELF_GEOMETRIES = [
    ("cnv1_7x7s2", 30, 44, 8, 16, 7, 2, 1),
    ("cnv2_5x5s2", 15, 22, 16, 32, 5, 2, 1),
    ("cnv3_dil2", 12, 20, 32, 64, 3, 1, 2),
    ("cnv4_dil4", 12, 20, 64, 128, 3, 1, 4),
    ("cnv5_dil8", 12, 20, 128, 256, 3, 1, 8),
    ("cnv6_dil2", 10, 20, 256, 256, 3, 1, 2),
    ("v0_s2_odd", 7, 13, 256, 256, 3, 2, 1),
]
MUTATIONS = ["drop_tap", "pad_neighbour", "skip_slab", "shift_pixel", "no_bias"]


def _self_operands(geom, seed=1):
    _, H, W_, C, Co, k, stride, dil = geom
    rng = np.random.default_rng(seed)
    a = rna(np.maximum(rng.normal(0.1, 1.0, (H, W_, C)), 0))         # post-relu activations, TF32
    w = rna(rng.normal(0.0, np.sqrt(2.0 / (k * k * C)), (k, k, C, Co)))
    b = rng.normal(0.0, 0.05, Co).astype(np.float32).astype(np.float64)
    return a, w, b, k, stride, dil


def _gate(geom, **kw):
    a, w, b, k, stride, dil = _self_operands(geom)
    y, s = ref_conv(a, w, b, k, stride, dil)
    got = simulated_kernel(a, w, b, k, stride, dil, **kw)
    st = Stat()
    st.add(got, y, accum_allowance(s, k * k * a.shape[2]))
    return st, got


@pytest.mark.parametrize("geom", SELF_GEOMETRIES, ids=[g[0] for g in SELF_GEOMETRIES])
def test_gate_passes_a_truncating_accumulator(geom):
    """A correct kernel whose fp32 adds all truncate, in a shuffled order, passes the bound, the offset check and
    the TF32-storage check at every layer geometry."""
    st, got = _gate(geom)
    assert st.ratio <= 1.0, (geom[0], st.ratio)
    assert abs(st.offset) <= OFFSET_BAR, (geom[0], st.offset)
    assert tf32_clean(got).all()


@pytest.mark.parametrize("mutation", MUTATIONS)
@pytest.mark.parametrize("geom", SELF_GEOMETRIES, ids=[g[0] for g in SELF_GEOMETRIES])
def test_gate_catches_a_subtly_wrong_kernel(geom, mutation):
    st, _ = _gate(geom, mutate=mutation)
    assert st.ratio > 1.0, (geom[0], mutation, st.ratio)


@pytest.mark.parametrize("geom", SELF_GEOMETRIES[::3], ids=[g[0] for g in SELF_GEOMETRIES[::3]])
def test_gate_catches_a_store_that_truncates_or_skips_the_rounding(geom):
    st, got = _gate(geom, store="trunc")
    assert tf32_clean(got).all() and st.offset < -OFFSET_BAR, st.offset       # within the bound, but biased
    st, got = _gate(geom, store="none")
    assert not tf32_clean(got).all()


def test_reference_convolution_is_tf_same():
    """ref_conv against a loop over taps with explicit TF-SAME indices (asymmetric padding: the extra one after)."""
    rng = np.random.default_rng(3)
    for (H, W_, k, stride, dil) in [(7, 13, 3, 2, 1), (9, 10, 7, 2, 1), (8, 12, 3, 1, 4), (5, 6, 5, 2, 1)]:
        a = rng.normal(size=(H, W_, 3))
        w = rng.normal(size=(k, k, 3, 2))
        b = rng.normal(size=2)
        y, s = ref_conv(a, w, b, k, stride, dil)
        Ho, pt, _ = tf_same_pad(H, k, stride, dil)
        Wo, pl, _ = tf_same_pad(W_, k, stride, dil)
        want = np.tile(b, (Ho, Wo, 1))
        for i in range(Ho):
            for j in range(Wo):
                for ty in range(k):
                    for tx in range(k):
                        r, c = i * stride + ty * dil - pt, j * stride + tx * dil - pl
                        if 0 <= r < H and 0 <= c < W_:
                            want[i, j] += a[r, c] @ w[ty, tx]
        np.testing.assert_allclose(y, want, rtol=1e-12, atol=1e-12)
        assert np.all(s >= np.abs(y) - 1e-12)


# ------------------------------------------------------------------------------------------- the GPU check --
HEADLINE = "v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh"
BN_CASES = {"batch_norm": "v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh-batch_norm",
            "batch_norm_couple_net": "v1-dilatedCouplePoseNN-cnv6_64-no_segmask-batch_norm",
            "batch_norm_plain_net": "v0-cnv6_128-segmask_rgb-static-batch_norm"}
SHARED = "v1-sharedNN-dilatedPoseNN-cnv6_%d-segmask_all-se_flow-abs_flow-fc_tanh"
ST, CL, SM, OR, WI, FF, C7, WR = ("DAVO_B200_CM_STAGED", "DAVO_B200_CLUSTER", "DAVO_B200_SMALL_TILES", "DAVO_B200_ORIENT",
                                  "DAVO_B200_WIDE", "DAVO_B200_FUSED_FRONT", "DAVO_B200_CNV7_CM", "DAVO_B200_WEIGHT_ROUNDING")
# name -> (version, H, W, batch, environment).  Rows of the plan table (see the issue this file was written for):
# a latency plans; b 256-pixel channels-on-M plans and strips; c staged / direct x cluster / not (136 rows: the
# smallest dilated map tall enough for channels-on-M; 3 samples of a non-shared net: an odd tile count, so the last
# cluster's second CTA has no tile);
# d forced orientations; e pair slabs, fused cnv1, channels-on-M sums; f sizes with partial tiles; g cnv6 widths and
# the SE variants; h non-shared nets; i stride-2 nets with odd pitched maps; j -batch_norm; k nearest weight rounding
CONFIGS = {
    "a_headline_b1": (HEADLINE, 128, 416, 1, {}),
    "b_headline_b6": (HEADLINE, 128, 416, 6, {}),
    "b_headline_b1_no_small_tiles": (HEADLINE, 128, 416, 1, {SM: "0"}),
    "c_direct": (HEADLINE, 136, 200, 3, {ST: "0"}),
    "c_staged": (HEADLINE, 136, 200, 3, {ST: "1"}),
    "c_no_cluster": (HEADLINE, 136, 200, 3, {CL: "0", ST: "0"}),
    "c_no_cluster_staged": (HEADLINE, 136, 200, 3, {CL: "0", ST: "1"}),
    "c_no_cluster_256": (HEADLINE, 136, 200, 3, {CL: "0", SM: "0"}),
    "c_odd_tile_count": ("v1-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh", 136, 200, 3, {}),
    "d_orient_pm": (HEADLINE, 64, 208, 2, {OR: "pm"}),
    "d_orient_cm": (HEADLINE, 64, 208, 2, {OR: "cm", WI: "0"}),
    "e_pair_slabs": (HEADLINE, 128, 416, 1, {WI: "0"}),
    "e_fused_front": (HEADLINE, 128, 416, 1, {FF: "1"}),
    "e_cnv7_cm": (HEADLINE, 128, 416, 1, {C7: "1"}),
    "e_cnv7_cm_256": (HEADLINE, 136, 424, 1, {C7: "1"}),
    "e_cnv7_cm_no_cluster": (HEADLINE, 64, 208, 2, {C7: "1", CL: "0"}),
    "e_cnv7_cm_256_no_cluster": (HEADLINE, 136, 424, 1, {C7: "1", CL: "0"}),
    "f_136x424": (HEADLINE, 136, 424, 1, {}),
    "f_128x400": (HEADLINE, 128, 400, 1, {}),
    "f_32x64": (HEADLINE, 32, 64, 1, {}),
    "f_256x832": (HEADLINE, 256, 832, 1, {}),
    "g_cnv6_32": (SHARED % 32, 64, 208, 2, {}),
    "g_cnv6_64": (SHARED % 64, 64, 208, 2, {}),
    "g_cnv6_256": (SHARED % 256, 64, 208, 2, {}),
    "g_cnv6_256_128rows": (SHARED % 256, 128, 416, 1, {}),
    "g_se_insert": ("v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-no_segmask-se_insert", 64, 208, 2, {}),
    "g_se_skipadd": ("v1-sharedNN-dilatedPoseNN-cnv6_256-segmask_all-se_flow-abs_flow-fc_tanh-se_skipadd", 64, 208, 2, {}),
    "g_se_replace": ("v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh-se_replace", 64, 208, 2, {}),
    "g_couple_shared": ("v1-sharedNN-dilatedCouplePoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh", 64, 208, 2, {}),
    "h_decouple_net": ("v1-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh", 64, 208, 2, {}),
    "h_couple_net": ("v0-dilatedCouplePoseNN-cnv6_128-segmask_rgb-se_seg-fc_tanh", 64, 208, 2, {}),
    "i_decouple_v0": ("v1-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh", 128, 416, 1, {}),
    "i_decouple_v0_64x208": ("v1-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh", 64, 208, 2, {}),
    "i_couple_v0": ("v1-couplePoseNN-cnv6_64-segmask_all-static", 64, 208, 2, {}),
    "i_decouple_v0_skipadd": ("v1-cnv6_256-segmask_all-se_flow-abs_flow-fc_tanh-se_skipadd", 128, 416, 1, {}),
    "j_batch_norm": (BN_CASES["batch_norm"], 128, 416, 2, {}),
    "j_batch_norm_couple_net": (BN_CASES["batch_norm_couple_net"], 128, 416, 2, {}),
    "j_batch_norm_plain_net": (BN_CASES["batch_norm_plain_net"], 128, 416, 2, {}),
    "k_nearest_rounding": (HEADLINE, 64, 208, 1, {WR: "nearest"}),
}
# configurations the planner refuses, with the error davo_create / davo_finalize_weights gives
REFUSED = {}
# the plans each row exists for: (layer, field of the ':plan' readback, value)
MUST_REACH = {
    "a_headline_b1": [("cnv1", "wide_G", 8), ("cnv2", "wide_G", 4), ("cnv3", "resident", 1), ("cnv5", "npix", 128),
                      ("cnv7", "epi", 1), ("cnv7", "orient", 0)],
    "b_headline_b6": [("cnv5", "npix", 256), ("cnv5", "strips", 1), ("cnv6", "npix", 256)],
    "b_headline_b1_no_small_tiles": [("cnv5", "npix", 256)],
    "c_direct": [("cnv4", "staged", 0), ("cnv4", "cluster", 1)],
    "c_staged": [("cnv5", "staged", 1), ("cnv5", "cluster", 1)],
    "c_no_cluster": [("cnv4", "cluster", 0), ("cnv4", "npix", 128), ("cnv4", "staged", 0)],
    "c_no_cluster_staged": [("cnv4", "cluster", 0), ("cnv4", "npix", 128), ("cnv4", "staged", 1)],
    "c_no_cluster_256": [("cnv5", "cluster", 0), ("cnv5", "npix", 256)],
    "d_orient_pm": [("cnv5", "orient", 0), ("cnv6", "orient", 0), ("cnv6", "resident", 0)],
    "e_pair_slabs": [("cnv1", "wide_G", 0), ("cnv2", "wide_G", 0)],
    "e_fused_front": [("cnv1", "fused", 1)],
    "e_cnv7_cm": [("cnv7", "orient", 1), ("cnv7", "npix", 128), ("cnv7", "cluster", 1)],
    "e_cnv7_cm_256": [("cnv7", "orient", 1), ("cnv7", "npix", 256)],
    "e_cnv7_cm_256_no_cluster": [("cnv7", "npix", 256), ("cnv7", "cluster", 0)],
    "f_136x424": [("cnv1", "wide_G", 0), ("cnv1", "BN", 16)],
    "f_32x64": [("cnv5", "orient", 0)],
    "g_cnv6_256_128rows": [("cnv6", "m_blocks", 4)],
    "g_se_insert": [("cnv6", "groups", 2)],
    "h_decouple_net": [("cnv1", "wide_G", 8)],
    "i_decouple_v0": [("cnv7", "orient", 0)],
    "j_batch_norm": [("cnv5", "raw", 1)],
}
PLAN_FIELDS = ("orient", "npix", "wide_G", "wide_tw", "staged", "cluster", "strips", "m_blocks", "groups", "raw", "epi",
               "BN", "resident", "fused")
# every branch of launch_conv: (orient, pixels per tile, widened G, staged, cluster, epilogue, pm: channels)
LAUNCH_BRANCHES = (
    {("cm", npix, 0, staged, cl, epi, None) for npix in (128, 256) for cl in (0, 1)
     for staged, epi in ((1, "store"), (0, "store"), (0, "sum"))}
    | {("pm", 128, 8, 0, 0, "store", 16), ("pm", 128, 4, 0, 0, "store", 32), ("pm", 128, 0, 0, 0, "sum", 256)}
    | {("pm", 128, 0, 0, 0, "store", bn) for bn in (16, 32, 64, 128, 256)})

_RUNS = {}            # configuration -> {"stats": {layer: Stat}, "plans": {layer: dict}, "error": str or None}


def _plan(sysm, name):
    v = sysm.get_intermediate(name + ":plan", 0)
    return {f: int(x) for f, x in zip(PLAN_FIELDS, v)}


def _branch(p):
    epi = "sum" if p["epi"] == 1 else "store"
    return ("cm" if p["orient"] else "pm", p["npix"], p["wide_G"], p["staged"], p["cluster"], epi,
            None if p["orient"] else p["BN"])


def _maps(cfg, H, W):
    """Per layer (geometry, input size, output size) from the net type; -se_replace has no cnv6 (cnv7 reads cnv5)."""
    geo = GEO_DILATED if cfg.posenn <= 3 else (GEO_V0_SKIPADD if cfg.posenn_se == 2 else GEO_V0)
    out, h, w = [], H, W
    for li, (k, st, dil) in enumerate(geo):
        ho, wo = tf_same_pad(h, k, st, dil)[0], tf_same_pad(w, k, st, dil)[0]
        out.append(((k, st, dil), (h, w), (ho, wo)))
        if not (li == 5 and cfg.posenn_se == 3):
            h, w = ho, wo
    return out


def _pitched(sysm, name, pair, hw, what):
    """A stored map read back with its pitch: the pad row / column of an odd map must be exactly zero."""
    h, w = hw
    hp, wp = h + (h & 1), w + (w & 1)
    flat = sysm.get_intermediate(name, pair)
    assert flat.size % (hp * wp) == 0, (what, name, flat.size, hp, wp)
    m = flat.reshape(hp, wp, -1)
    assert not m[h:].any() and not m[:, w:].any(), "%s: %s: the pad row / column is not zero" % (what, name)
    return m[:h, :w]


def _layer_operands(sysm, li, pair, geo_in, groups):
    """:in cut into the group's channels, :w<g>, :b, as float64."""
    name = NAMES[li]
    a32 = _pitched(sysm, name + ":in", pair, geo_in, "input")
    a = a32.astype(np.float64)
    b = sysm.get_intermediate(name + ":b", pair).astype(np.float64)
    return a32, a, b


def _conv_layer(a, ws, b, groups, k, stride, dil):
    """y, s of one layer over its groups; ws[g] [k,k,Cin_g,BN]."""
    ys, ss = [], []
    C = a.shape[2]
    for g in range(groups):
        cin_g, bn = ws[g].shape[2], ws[g].shape[3]
        off = 0 if groups * cin_g > C else g * cin_g          # cnv6 groups that all read the same cnv5
        y, s = ref_conv(a[..., off:off + cin_g], ws[g], b[g * bn:(g + 1) * bn], k, stride, dil)
        ys.append(y)
        ss.append(s)
    return np.concatenate(ys, -1), np.concatenate(ss, -1), k * k * ws[0].shape[2]


def _units(sysm, B):
    return B if sysm.config.posenn >= 2 else 2 * B


def _run_config(name, monkeypatch_factory=pytest.MonkeyPatch):
    if name in _RUNS:
        return _RUNS[name]
    from davo_b200.davo import DAVO
    ver, H, W, B, env = CONFIGS[name]
    res = _RUNS[name] = {"stats": {}, "plans": {}, "error": None}
    inputs = [torch.as_tensor(x).cuda() for x in S.make_inputs(B, H, W, seed=zlib.crc32(name.encode()) % 1000, bad_label_frac=0.01)]
    depth = torch.as_tensor(S.make_depth(B, H, W)).cuda()            # read by the depth attention sources only
    weights = S.init_weights(ver, seed=8964, random_bias=True)
    with monkeypatch_factory.context() as mp:               # knobs are read when the weights are finalised
        for k, v in env.items():
            mp.setenv(k, v)
        try:
            sysm = DAVO(version=ver)
            sysm.setup_inference(H, W, "davo", 3, B, inputs[0], input_flow=inputs[1], input_seglabel=inputs[2],
                                 input_depth=depth, device=0)
            sysm.load_weights(weights)
        except RuntimeError as e:
            res["error"] = str(e)
            return res
    sysm.inference(None, "pose")
    cfg = sysm.config
    units = _units(sysm, B)
    pairs = sorted({0, units - 1} | ({units // 2} if units > 4 else set()))
    maps = _maps(cfg, H, W)
    for p in pairs:
        assert tf32_clean(sysm.get_intermediate("packed", p)).all(), (name, "packed")
    bn = bool(cfg.batch_norm)
    for li, (geom, hw_in, hw_out) in enumerate(maps):
        lname = NAMES[li]
        if li == 5 and cfg.posenn_se == 3:
            continue
        plan = res["plans"][lname] = _plan(sysm, lname)
        k, stride, dil = geom
        groups = plan["groups"]
        ws = [sysm.get_intermediate("%s:w%d" % (lname, g), 0) for g in range(groups)]
        stored = li < 6 or bn
        st = res["stats"][lname] = Stat()
        todo = range(units) if bn else pairs
        ys = {}
        for p in todo:
            a32, a, b = _layer_operands(sysm, li, p, hw_in, groups)
            assert tf32_clean(a32).all(), (name, lname, "input", p)
            cin_g = ws[0].size // (k * k * (b.size // groups))
            wg = [x.reshape(k, k, cin_g, -1).astype(np.float64) for x in ws]
            assert all(tf32_clean(x).all() for x in ws), (name, lname, "weights")
            if bn:
                b_conv, beta = np.zeros_like(b), b
            else:
                b_conv, beta = b, None
            ys[p] = _conv_layer(a, wg, b_conv, groups, k, stride, dil)
        if bn:
            _check_bn(sysm, name, li, ys, pairs, hw_out, st, beta, units, cfg)
        elif stored:
            for p in pairs:
                y, s, n = ys[p]
                got32 = _pitched(sysm, lname + ":pitched", p, hw_out, name)
                assert np.array_equal(got32, sysm.get_intermediate(lname, p).reshape(got32.shape)), (name, lname)
                assert tf32_clean(got32).all(), (name, lname, "stored values are not TF32")
                st.add(got32, y, accum_allowance(s, n))
        else:                                               # cnv7 sum epilogue
            P = hw_out[0] * hw_out[1]
            for p in pairs:
                y, s, n = ys[p]
                E = accum_allowance(s, n)
                want = np.maximum(y, 0).sum((0, 1))
                allow = E.sum((0, 1)) + (P + 2) * U22 * (np.abs(np.maximum(y, 0)) + E).sum((0, 1))
                got = sysm.get_intermediate("cnv7_sum", p).astype(np.float64)
                st.add(got, want, allow, rounded=False)
    if cfg.posenn_se in (1, 2, 3):
        _check_se5(sysm, name, weights, pairs, maps, cfg)
    if B > 1 and any((hw[2][0] | hw[2][1]) & 1 for hw in maps):
        # the zero pad row / column of an odd map stays zero after a smaller batch ran through the same buffers
        sysm.inference(None, "pose", inputs=tuple(t[:B - 1] for t in inputs) + (depth[:B - 1],))
        for li, (_, _, hw_out) in enumerate(maps):
            if (li < 6 or bn) and not (li == 5 and cfg.posenn_se == 3):
                for p in range(_units(sysm, B - 1)):
                    _pitched(sysm, NAMES[li] + ":pitched", p, hw_out, name + " after a smaller batch")
    del sysm
    torch.cuda.empty_cache()
    return res


def _check_bn(sysm, name, li, ys, pairs, hw_out, st, beta, units, cfg):
    """-batch_norm: see the module docstring for the bound."""
    lname = NAMES[li]
    shared = cfg.posenn <= 1
    for p in pairs:
        grp = [q for q in ys if (q % 2 == p % 2 or not shared)]
        x = np.stack([ys[q][0] for q in grp])                 # [units of the group, h, w, C]
        Eg = np.stack([accum_allowance(ys[q][1], ys[q][2]) for q in grp])
        mu = x.mean((0, 1, 2))
        var = ((x - mu) ** 2).mean((0, 1, 2))
        r = 1.0 / np.sqrt(var + 1e-3)
        Em = Eg.max((0, 1, 2))
        y, s, n = ys[p]
        Ex = accum_allowance(s, n)
        if li == 6:                                           # the raw epilogue: plain conv sums
            got = _pitched(sysm, lname + ":pitched", p, hw_out, name)
            st.add(got, y, Ex, rounded=False, relu=False)
            continue
        dr = r * ((np.sqrt(var) * Em + Em ** 2 / 2) / (var + 1e-3) + 2 * U23)
        z = (y - mu) * r + beta
        D = r * (Ex + Em + U24 * np.abs(mu)) + np.abs(y - mu) * dr + U22 * (np.abs(y - mu) * r + np.abs(beta))
        got = _pitched(sysm, lname + ":pitched", p, hw_out, name)
        assert tf32_clean(got).all(), (name, lname, "stored values are not TF32")
        st.add(got, z, D)


def _check_se5(sysm, name, weights, pairs, maps, cfg):
    """The SE block on cnv5 / cnv6: the excitation against fp64 (the att_weights tolerance of test_gpu_parity), and
    d_se5out per element against rna(relu(cnv5 * e)) / rna(relu(cnv5 + cnv6 * e)) with the GPU's own e."""
    nbr = 1 if cfg.posenn in (1, 3, 4) else 2
    scope = lambda g: "pose_exp_net/" + ("pose/%s/" % ("rotation", "translation")[g] if nbr == 2 else "pose/")
    blk = "cnv6_se_attention/" if cfg.posenn_se in (2, 3) else "cnv5_se_attention/"
    h5 = maps[4][2]
    for p in pairs:
        c5 = _pitched(sysm, "cnv5:pitched", p, h5, name).astype(np.float64)
        e_gpu = sysm.get_intermediate("se5_scale", p).astype(np.float64).reshape(nbr, 256)
        if cfg.posenn_se == 2:
            c6 = _pitched(sysm, "cnv6:pitched", p, maps[5][2], name).astype(np.float64).reshape(*h5, nbr, 256)
        e_ref, run = [], 1.0
        for g in range(nbr):
            W1, b1, W2, b2 = (np.asarray(weights[scope(g) + blk + v], np.float64) for v in
                              ("bottleneck_fc/kernel", "bottleneck_fc/bias", "recover_fc/kernel", "recover_fc/bias"))
            m = c6[..., g, :].mean((0, 1)) if cfg.posenn_se == 2 else c5.mean((0, 1)) * (run if cfg.posenn_se == 1 else 1.0)
            e = 1.0 / (1.0 + np.exp(-(np.maximum(m @ W1 + b1, 0) @ W2 + b2)))
            run = run * e
            e_ref.append(run if cfg.posenn_se == 1 else e)
        np.testing.assert_allclose(e_gpu, np.stack(e_ref), rtol=2e-6, atol=1e-7, err_msg="%s: se5_scale" % name)
        src = "cnv7:in" if cfg.posenn_se in (2, 3) else "cnv6:in"
        out = _pitched(sysm, src, p, h5, name).astype(np.float64).reshape(*h5, nbr, 256)
        for g in range(nbr):
            if cfg.posenn_se == 2:
                t = c5 + c6[..., g, :] * e_gpu[g]
                allow = U23 * (np.abs(c5) + np.abs(c6[..., g, :] * e_gpu[g]))
            else:
                t = c5 * e_gpu[g]
                allow = U24 * np.abs(t)
            want = np.maximum(t, 0)
            assert np.all(np.abs(out[..., g, :] - want) <= U11 * (want + allow) + allow), (name, "se5 out", g)


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
def test_conv_stage_per_element(config):
    _need_gpu()
    res = _run_config(config)
    if config in REFUSED:
        assert res["error"] is not None and REFUSED[config] in res["error"], res["error"]
        return
    assert res["error"] is None, res["error"]
    for lname, field, value in MUST_REACH.get(config, []):
        assert res["plans"][lname][field] == value, (config, lname, field, res["plans"][lname])
    for lname, st in res["stats"].items():
        assert st.ratio <= 1.0, "%s %s: error / bound %.3g at %s" % (config, lname, st.ratio, getattr(st, "where", None))
        assert abs(st.offset) <= OFFSET_BAR, "%s %s: mean offset %.3f TF32 ulp" % (config, lname, st.offset)


@pytest.mark.gpu
def test_every_launch_conv_branch_is_reached(capsys):
    """Runs whatever configuration has not run yet, prints the ratio table, and holds the plans reached to every
    branch of launch_conv (and the raw epilogue in both orientations, channels-on-M with 1, 2 and 4 m-blocks)."""
    _need_gpu()
    seen, m_blocks, raw = set(), set(), set()
    lines = []
    for config in CONFIGS:
        res = _run_config(config)
        if res["error"] is not None:
            lines.append("%-30s refused: %s" % (config, res["error"]))
            continue
        for lname, p in res["plans"].items():
            if p["raw"]:
                raw.add("cm" if p["orient"] else "pm")
            else:
                seen.add(_branch(p))
            if p["orient"]:
                m_blocks.add(p["m_blocks"])
        for lname, st in res["stats"].items():
            lines.append("%-30s %-5s ratio %.4f  offset %+.4f ulp  (%d elements)" % (config, lname, st.ratio, st.offset, st.n))
    with capsys.disabled():
        print("\nconv stages: largest |error| / bound, mean offset in TF32 ulps, per (configuration, layer)")
        print("\n".join(lines))
        print("plans reached:", sorted(seen, key=str))
    missing = LAUNCH_BRANCHES - seen
    assert not missing, sorted(missing, key=str)
    assert m_blocks >= {1, 2, 4}, m_blocks
    assert raw == {"cm", "pm"}, raw
