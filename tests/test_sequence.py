"""Frame-sequence inputs (include/davo_b200.h: davo_forward_sequence, davo_forward_sequence_host) on the GPU.

The defining property: a sequence call returns the bits davo_forward_pairs returns on the triplet batch that
davo_b200.sequence.sequence_to_triplets builds from the same frames."""
import ctypes as C

import numpy as np
import pytest
import torch

from davo_b200 import _capi, geo_utils, evaluation, synthetic as S, version as V
from davo_b200.davo import DAVO
from davo_b200.sequence import sequence_to_triplets
from tests.golden import make_golden as G

pytestmark = pytest.mark.gpu

H, W = 128, 416
HEADLINE = G.CASES["headline"]
PAIRS = ("all", "trajectory", "trajectory_first")


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _system(ver, max_batch, h=H, w=W, micro_batch=0, flow_f16=False, seed=8964):
    sysm = DAVO(version=ver)
    sysm.setup_inference(h, w, "davo", 3, max_batch, device=0, micro_batch=micro_batch, flow_f16=flow_f16)
    sysm.load_weights(S.init_weights(ver, seed=seed, random_bias=True))
    return sysm


def _cuda(*xs):
    return tuple(None if x is None else torch.as_tensor(x).cuda() for x in xs)


def _triplet_poses(sysm, seq, pairs):
    img, fwd, bwd, seg, depth = seq
    t = sequence_to_triplets(img, fwd, bwd, seg, depth)
    return sysm.inference(None, "pose", inputs=_cuda(*t), pairs=pairs)["pose"].copy()


def _device_poses(sysm, seq, pairs):
    return sysm.inference_sequence(*_cuda(*seq), pairs=pairs)["pose"]


def _seq(n, h=H, w=W, seed=5):
    img, fwd, bwd, seg, depth = S.make_sequence(n, h, w, seed=seed)
    seg[0, :2, :3] = 255.0                      # a few labels without a class
    return img, fwd, bwd, seg, depth


@pytest.mark.parametrize("key", list(G.CASES))
def test_device_sequence_equals_triplets_for_every_variant(key):
    """N = 6 frames (4 samples), every pair selection the variant takes: the bits of davo_forward_pairs."""
    _need_gpu()
    ver = G.CASES[key]
    cfg = V.parse_version(ver)
    sysm = _system(ver, 4)
    seq = _seq(6)
    for pairs in (("all",) if cfg.batch_norm else PAIRS):
        a = _triplet_poses(sysm, seq, pairs)
        b = _device_poses(sysm, seq, pairs)
        assert np.array_equal(a, b), (key, pairs, np.abs(a - b).max())


@pytest.mark.parametrize("case", ["flow_f16", "w_not_16", "stride2_short", "fused_front"])
def test_device_sequence_equals_triplets_at_other_settings(case, monkeypatch):
    """binary16 flow mode; a width that is not a multiple of 16 (16-channel packed fallback); a stride-2 net on a
    frame of fewer than 64 rows; cnv1 building its operand from the raw inputs (DAVO_B200_FUSED_FRONT=1), host
    sequence path included."""
    _need_gpu()
    ver, h, w, f16 = {"flow_f16": (HEADLINE, H, W, True), "w_not_16": (HEADLINE, 64, 136, False),
                      "stride2_short": (G.CASES["plain_decouple_net"], 48, 160, False),
                      "fused_front": (HEADLINE, H, W, False)}[case]
    if case == "fused_front":
        monkeypatch.setenv("DAVO_B200_FUSED_FRONT", "1")
    sysm = _system(ver, 4, h, w, flow_f16=f16)
    seq = _seq(6, h, w, seed=7)
    for pairs in PAIRS:
        d = _device_poses(sysm, seq, pairs)
        assert np.array_equal(_triplet_poses(sysm, seq, pairs), d), (case, pairs)
        if case == "fused_front":
            assert np.array_equal(sysm.inference_sequence(*seq, pairs=pairs)["pose"], d), pairs


@pytest.mark.parametrize("key", ["headline", "se_seg", "decouple_net", "se_depth", "pix_mix_segflow", "static", "no_segmask"])
def test_host_sequence_equals_device_sequence(key, monkeypatch):
    """Blocking and asynchronous host calls against the device call: N = 3, chunk + 2, chunk + 3, max_batch + 2, with
    the labels narrowed to bytes on the CPU and, with flow_f16 = 1, the flow to binary16."""
    _need_gpu()
    monkeypatch.setenv("DAVO_B200_HOST_FLOW16_FRAC", "0.5")
    ver = G.CASES[key]
    for f16 in (False, True):
        sysm = _system(ver, 7, micro_batch=4, flow_f16=f16)
        chunk = 4 if sysm.config.posenn not in (V.POSENN_DECOUPLE_SHARED_DIL, V.POSENN_COUPLE_SHARED_DIL) else 2
        for n in sorted({3, chunk + 2, chunk + 3, 7 + 2}):
            seq = _seq(n, seed=n)
            for pairs in PAIRS:
                d = _device_poses(sysm, seq, pairs)
                h = sysm.inference_sequence(*seq, pairs=pairs)["pose"]
                assert np.array_equal(d, h), (key, f16, n, pairs)
                pend = [sysm.inference_sequence_async(*seq, pairs=pairs) for _ in range(3)]     # calls in flight
                for p in pend:
                    assert np.array_equal(d, p.result()["pose"]), (key, f16, n, pairs)


def test_overlapping_calls_equal_one_call_and_compose_the_same_trajectory():
    """Two calls that share 2 frames give the poses of one call over the whole sequence; the trajectories composed
    from sequence and triplet poses (host loop and davo_compose_trajectory) are identical."""
    _need_gpu()
    sysm = _system(HEADLINE, 12)
    seq = _seq(14, seed=3)
    for pairs in PAIRS:
        whole = sysm.inference_sequence(*seq, pairs=pairs)["pose"]
        img, fwd, bwd, seg, depth = seq                    # frames [0, 8) and [6, 14): flows [0, 7) and [6, 13)
        first = sysm.inference_sequence(img[:8], fwd[:7], bwd[:7], seg[:8], depth[:8], pairs=pairs)["pose"]
        later = "trajectory" if pairs == "trajectory_first" else pairs
        tail = tuple(x[6:] for x in seq)
        second = sysm.inference_sequence(*tail, pairs=later)["pose"]
        assert np.array_equal(np.concatenate([first, second]), whole), pairs
        assert np.array_equal(_device_poses(sysm, tail, later), second)
    poses = sysm.inference_sequence(*seq, pairs="trajectory_first")["pose"]
    trip = _triplet_poses(sysm, seq, "trajectory_first")
    assert np.array_equal(geo_utils.compose_trajectory(poses), geo_utils.compose_trajectory(trip))
    a = evaluation.compose_trajectory_gpu(sysm, torch.as_tensor(poses).cuda()).cpu().numpy()
    b = evaluation.compose_trajectory_gpu(sysm, torch.as_tensor(trip).cuda()).cpu().numpy()
    assert np.array_equal(a, b)


def _expected_h2d(sysm, n, pairs):
    """Bytes the host sequence call must move: the frames and flow entries some computed pair reads, once each."""
    c, hw = sysm.config, H * W
    unit = c.posenn not in (V.POSENN_DECOUPLE_SHARED_DIL, V.POSENN_COUPLE_SHARED_DIL)
    k0 = lambda s: unit or pairs == "all" or (pairs == "trajectory_first" and s == 0)
    b = n - 2
    img = [f for f in range(n) if (1 <= f <= b) or f >= 2 or (f < b and k0(f))]
    flow = c.in_mode == 1 or c.att_src in (1, 6) or c.pixel_map == 2
    labels = c.att_src != 0 and (not c.pixel_map or c.att_src == 6)
    lab = [f for f in range(n) if labels and (f >= 2 or (f < b and k0(f)) or (not c.att_tgt_ones and 1 <= f <= b))]
    depth = c.att_src == V.ATT_SE_DEPTH_SEG or c.depth_split
    fl = (sum(k0(s) for s in range(b)) + b) * hw * 8 if flow else 0
    return len(img) * hw * 3 + len(lab) * hw + (len(img) * hw * 4 if depth else 0) + fl


@pytest.mark.parametrize("key", ["headline", "se_seg", "decouple_net", "se_depth", "pix_rgb", "no_segmask"])
def test_host_sequence_copies_each_read_plane_once(key):
    _need_gpu()
    ver = G.CASES[key]
    sysm = _system(ver, 7, micro_batch=4)
    for n in (3, 6, 9):
        seq = _seq(n, seed=11)
        for pairs in PAIRS:
            sysm.inference_sequence(*seq, pairs=pairs)
            h2d, d2h = sysm.last_host_copy_bytes()
            assert h2d == _expected_h2d(sysm, n, pairs) and d2h == (n - 2) * 48, (key, n, pairs)


def test_trajectory_mode_moves_at_most_045_of_the_triplet_bytes():
    """Headline version, 128 samples (N = 130), trajectory mode: (N-1) images, (N-2) label planes as bytes, (N-2)
    float32 flow entries -- against the triplet host call on the same frames."""
    _need_gpu()
    n, hw = 130, H * W
    sysm = _system(HEADLINE, 128)
    seq = _seq(n, seed=13)
    s = sysm.inference_sequence(*seq, pairs="trajectory")["pose"]
    h2d_seq = sysm.last_host_copy_bytes()[0]
    assert h2d_seq == (n - 1) * 3 * hw + (n - 2) * hw + (n - 2) * 8 * hw
    img, flow, seg, _ = sequence_to_triplets(*seq)
    t = sysm.inference(None, "pose", inputs=(img, flow, seg), pairs="trajectory")["pose"]
    assert np.array_equal(s, t)
    assert h2d_seq <= 0.45 * sysm.last_host_copy_bytes()[0]
    # a flow_fwd nobody reads may be absent
    assert np.array_equal(s, sysm.inference_sequence(seq[0], None, seq[2], seq[3], pairs="trajectory")["pose"])


def test_argument_errors_name_the_input():
    _need_gpu()
    sysm = _system(HEADLINE, 4)
    lib, h = sysm._lib, sysm._h
    n = 6
    img, fwd, bwd, seg, _ = _cuda(*_seq(n))
    out = torch.empty((n - 2, 2, 6), device="cuda")
    p = lambda t, off=0: C.c_void_p(t.data_ptr() + off) if t is not None else None
    ALL, TRAJ = _capi.PAIRS["all"], _capi.PAIRS["trajectory"]

    def call(fn, nf, pairs, args):
        if fn == "dev":
            rc = lib.davo_forward_sequence(h, nf, pairs, *args, p(out), None)
        else:
            rc = lib.davo_forward_sequence_host(h, nf, pairs, *args, p(out), None, None)
        return rc, _capi.last_error(lib, h)

    imgh, fwdh, bwdh, segh, _ = _seq(n)
    hp = lambda a, off=0: C.c_void_p(a.ctypes.data + off) if a is not None else None
    for fn, ptrs in (("dev", p), ("host", hp)):
        im, fw, bw, sg = (img, fwd, bwd, seg) if fn == "dev" else (imgh, fwdh, bwdh, segh)
        good = [ptrs(im), ptrs(fw), ptrs(bw), ptrs(sg), None]
        rc, msg = call(fn, 2, ALL, good)
        assert rc == -1 and "n_frames=2" in msg
        rc, msg = call(fn, 7, ALL, good)
        assert rc == -1 and "max_batch" in msg
        for i, name in ((0, "img"), (2, "flow_bwd"), (3, "seg"), (1, "flow_fwd")):
            args = list(good)
            args[i] = None
            rc, msg = call(fn, n, ALL, args)
            assert rc == -1 and name in msg, (fn, name, msg)
        args = list(good)
        args[1] = None
        assert call(fn, n, TRAJ, args)[0] == 0                # trajectory mode of a shared net reads no flow_fwd
        for i, name in ((0, "img"), (1, "flow_fwd"), (2, "flow_bwd"), (3, "seg")):
            args = list(good)
            args[i] = ptrs((im, fw, bw, sg)[i], 4)
            rc, msg = call(fn, n, ALL, args)
            assert rc == -1 and name in msg and "aligned" in msg, (fn, name, msg)
