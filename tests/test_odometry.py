"""Online odometry sessions (include/davo_b200.h: davo_odometry_*, davo_b200.davo.Odometry).

The defining properties: however a stream is cut into pushes, the poses are the bits of one davo_forward_sequence call
over the whole sequence, and the absolute poses are the same bits for every cut."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from davo_b200 import _capi, evaluation, geo_utils, synthetic as S, version as V
from davo_b200.davo import DAVO
from tests.golden import make_golden as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W = 128, 416
HEADLINE = G.CASES["headline"]
FIRST = {"trajectory": "trajectory_first", "all": "all"}      # the whole-sequence call a session's poses equal


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _system(ver, max_batch, micro_batch=0, flow_f16=False):
    sysm = DAVO(version=ver)
    sysm.setup_inference(H, W, "davo", 3, max_batch, device=0, micro_batch=micro_batch, flow_f16=flow_f16)
    sysm.load_weights(S.init_weights(ver, seed=31, random_bias=True))
    return sysm


def _seq(n, seed=5):
    img, fwd, bwd, seg, depth = S.make_sequence(n, H, W, seed=seed)
    seg[0, :2, :3] = 255.0                      # a few labels without a class
    return img, fwd, bwd, seg, depth


def _pieces(seq, cut):
    """The pushes of a cut: frames [a, b) with flow entries [a-1, b-1) ([0, b-1) for the first)."""
    img, fwd, bwd, seg, depth = seq
    a = 0
    for k in cut:
        b = a + k
        fl = slice(max(a - 1, 0), b - 1)
        yield img[a:b], fwd[fl], bwd[fl], seg[a:b], depth[a:b]
        a = b


def _np(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else x


def _run(od, seq, cut, device=False):
    """Pushes `seq` as `cut`; returns the concatenated poses and trajectory, checking the frame ranges."""
    poses, traj, posed = [], [], 0
    for p in _pieces(seq, cut):
        out = od.push(*(tuple(torch.as_tensor(x).cuda() for x in p) if device else p))
        assert out["frames"] == range(posed, posed + out["trajectory"].shape[0])
        posed += out["trajectory"].shape[0]
        poses.append(_np(out["pose"]))
        traj.append(_np(out["trajectory"]))
    assert od.frames() == (sum(cut), posed)
    return np.concatenate(poses), np.concatenate(traj)


def _random_cut(n, rng, first):
    cut = [first]
    while sum(cut) < n:
        cut.append(int(min(rng.integers(1, 9), n - sum(cut))))
    return cut


@pytest.mark.gpu
@pytest.mark.parametrize("pairs", ["trajectory", "all"])
def test_every_cut_gives_the_whole_sequence_poses_and_one_trajectory(pairs):
    _need_gpu()
    n = 40
    sysm = _system(HEADLINE, n)
    seq = _seq(n, seed=3)
    whole = sysm.inference_sequence(*seq, pairs=FIRST[pairs])["pose"]
    rng = np.random.default_rng(7)
    cuts = [[n], [1] * n, [1, 1, 5, 2, 9, 3, 1, 18], _random_cut(n, rng, 1), _random_cut(n, rng, 2), _random_cut(n, rng, 2)]
    trajs = []
    with sysm.odometry(pairs=pairs) as od:
        for cut in cuts:
            od.reset()
            poses, traj = _run(od, seq, cut)
            assert np.array_equal(poses, whole), cut
            assert traj.shape == (n, 4, 4)
            trajs.append(traj)
    for t in trajs[1:]:
        assert np.array_equal(t, trajs[0])                  # a sequential chain: the bits do not depend on the cut
    host = geo_utils.compose_trajectory(whole)
    got = trajs[0]
    path = float(np.linalg.norm(np.diff(host[:, :3, 3], axis=0), axis=1).sum())
    assert np.array_equal(got[0], np.eye(4)) and np.all(got[:, 3] == [0, 0, 0, 1])
    assert np.abs(got - host)[:, :3, 3].max() <= 2e-6 * path + 1e-6
    assert np.abs(got - host)[:, :3, :3].max() <= 2e-5
    scan = evaluation.compose_trajectory_gpu(sysm, torch.as_tensor(whole).cuda()).cpu().numpy()
    assert np.abs(got - scan).max() <= 1e-9 * path + 1e-12   # the same products, associated differently


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(G.CASES))
def test_every_variant_equals_the_sequence_call(key):
    """One fixed cut, host session in trajectory mode and device session in all mode; -batch_norm is refused."""
    _need_gpu()
    ver = G.CASES[key]
    sysm = _system(ver, 9)
    if V.parse_version(ver).batch_norm:
        with pytest.raises(RuntimeError, match="-batch_norm"):
            sysm.odometry()
        return
    seq = _seq(11, seed=4)
    cut = [2, 3, 1, 5]
    for pairs, device in (("trajectory", False), ("all", True)):
        with sysm.odometry(pairs=pairs, host=not device) as od:
            poses, _ = _run(od, seq, cut, device)
        assert np.array_equal(poses, sysm.inference_sequence(*seq, pairs=FIRST[pairs])["pose"]), (key, pairs)


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["headline", "decouple_net", "se_depth", "se_seg"])
def test_host_sessions_equal_device_sessions(key, monkeypatch):
    """Both flow_f16 modes, half of a chunk's flow narrowed on the CPU, pushes larger than the host chunk (2 samples
    for the shared nets, 4 for the others at micro_batch 4) and equal to max_push."""
    _need_gpu()
    monkeypatch.setenv("DAVO_B200_HOST_FLOW16_FRAC", "0.5")
    ver = G.CASES[key]
    seq = _seq(24, seed=9)
    cut = [1, 7, 3, 7, 1, 5]
    for f16 in (False, True):
        sysm = _system(ver, 22, micro_batch=4, flow_f16=f16)
        for pairs in ("trajectory", "all"):
            with sysm.odometry(pairs, 7, host=True) as h, sysm.odometry(pairs, 7, host=False) as d:
                ph, th = _run(h, seq, cut)
                pd, td = _run(d, seq, cut, device=True)
            assert np.array_equal(ph, pd) and np.array_equal(th, td), (key, f16, pairs)
            assert np.array_equal(ph, sysm.inference_sequence(*seq, pairs=FIRST[pairs])["pose"]), (key, f16, pairs)


@pytest.mark.gpu
def test_pushes_in_flight_equal_blocking_pushes():
    _need_gpu()
    sysm = _system(HEADLINE, 8, micro_batch=4)
    seq = _seq(30, seed=12)
    cut = [2, 1, 8, 4, 1, 6, 8]
    for pairs in ("trajectory", "all"):
        with sysm.odometry(pairs=pairs) as od:
            want = _run(od, seq, cut)
        with sysm.odometry(pairs=pairs) as od:
            pend, outs = [], []
            for p in _pieces(seq, cut):
                pend.append(od.push_async(*p))
                if len(pend) == 3:                          # three pushes in flight
                    outs.append(pend.pop(0).result())
            outs += [p.result() for p in pend]
        assert np.array_equal(np.concatenate([o["pose"] for o in outs]), want[0])
        assert np.array_equal(np.concatenate([o["trajectory"] for o in outs]), want[1])
        assert [o["frames"] for o in outs][-1].stop == 30


@pytest.mark.gpu
@pytest.mark.parametrize("host", [True, False])
def test_sessions_on_one_handle_are_independent(host):
    """Two sessions pushed in turns, with sequence and triplet calls on the handle between pushes: each equals a run of
    it alone; reset() then a new sequence equals a fresh session."""
    _need_gpu()
    sysm = _system(HEADLINE, 8, micro_batch=4)
    sa, sb, other = _seq(17, seed=1), _seq(15, seed=2), _seq(9, seed=6)
    ca, cb = [2, 5, 1, 8, 1], [1, 3, 3, 8]
    with sysm.odometry(host=host) as od:
        alone_a = _run(od, sa, ca, not host)
        od.reset()
        alone_b = _run(od, sb, cb, not host)
    trip = S.make_inputs(3, H, W, seed=2)
    oa, ob = sysm.odometry(host=host), sysm.odometry(pairs="trajectory", host=host)
    res = {"a": ([], []), "b": ([], [])}
    pa, pb = list(_pieces(sa, ca)), list(_pieces(sb, cb))
    for i in range(max(len(pa), len(pb))):
        for name, od, pieces in (("a", oa, pa), ("b", ob, pb)):
            if i < len(pieces):
                p = pieces[i] if host else tuple(torch.as_tensor(x).cuda() for x in pieces[i])
                out = od.push(*p)
                res[name][0].append(_np(out["pose"]))
                res[name][1].append(_np(out["trajectory"]))
            sysm.inference_sequence(*other, pairs="all")
            sysm.inference(None, "pose", inputs=trip)
    for name, alone in (("a", alone_a), ("b", alone_b)):
        assert np.array_equal(np.concatenate(res[name][0]), alone[0]), name
        assert np.array_equal(np.concatenate(res[name][1]), alone[1]), name
    oa.reset()                                              # a new sequence on a used session
    again = _run(oa, sb, cb, not host)
    assert np.array_equal(again[0], alone_b[0]) and np.array_equal(again[1], alone_b[1])
    oa.close()
    ob.close()


def _expected_stream_h2d(sysm, n, pairs, flow_entry_bytes=H * W * 8):
    """Bytes a host session moves over a whole n-frame stream: every frame, label plane, depth plane and flow entry some
    pair of the stream reads, once -- and the last flow_fwd entry of the stream when the sample after the last one
    would read it (a push copies that entry for the next push, which the session cannot know will not come).  A flow
    entry is `flow_entry_bytes`: H*W*8 as float32, H*W*4 as binary16."""
    c, hw = sysm.config, H * W
    unit = c.posenn not in (V.POSENN_DECOUPLE_SHARED_DIL, V.POSENN_COUPLE_SHARED_DIL)
    k0 = lambda s: unit or pairs == "all" or s == 0
    b = n - 2
    flow = c.in_mode == 1 or c.att_src in (1, 6) or c.pixel_map == 2
    labels = c.att_src != 0 and (not c.pixel_map or c.att_src == 6)
    lab = [f for f in range(n) if labels and (f >= 2 or k0(f) or (not c.att_tgt_ones and f >= 1))]
    depth = c.att_src == V.ATT_SE_DEPTH_SEG or c.depth_split
    fwd = sum(k0(s) for s in range(n - 1))                 # flow_fwd entry s is read by sample s (plane 0)
    fl = (fwd + b) * flow_entry_bytes if flow else 0
    return n * hw * 3 + len(lab) * hw + (n * hw * 4 if depth else 0) + fl


@pytest.mark.gpu
@pytest.mark.parametrize("key,f16", [pytest.param(k, False, id=k) for k in
                                     ["headline", "se_seg", "decouple_net", "se_depth", "no_segmask"]] +
                                    [pytest.param("headline", True, id="headline-flow16")])
def test_host_session_sends_each_read_plane_once(key, f16, monkeypatch):
    """f16: flow_f16 with every flow entry a push sends narrowed on the CPU, so every one crosses as binary16."""
    _need_gpu()
    flow_bytes = H * W * (4 if f16 else 8)
    if f16:
        monkeypatch.setenv("DAVO_B200_HOST_FLOW16_FRAC", "1")
    sysm = _system(G.CASES[key], 7, micro_batch=4, flow_f16=f16)
    n = 20
    seq = _seq(n, seed=11)
    for pairs in ("trajectory", "all"):
        for cut in ([1, 1, 1, 7, 2, 1, 7], [2, 7, 7, 4], [3] + [1] * 17):
            total = 0
            with sysm.odometry(pairs=pairs) as od:
                for p in _pieces(seq, cut):
                    out = od.push(*p)
                    h2d, d2h = sysm.last_host_copy_bytes()
                    assert d2h == out["pose"].nbytes + out["trajectory"].nbytes
                    total += h2d
            assert total == _expected_stream_h2d(sysm, n, pairs, flow_bytes), (key, pairs, cut)
    # against the same stream as 3-frame sequence calls, one per new frame
    img, fwd, bwd, seg, depth = seq
    triples = 0
    for s in range(n - 2):
        sysm.inference_sequence(img[s:s + 3], fwd[s:s + 2], bwd[s:s + 2], seg[s:s + 3], depth[s:s + 3],
                                pairs="trajectory_first" if s == 0 else "trajectory")
        triples += sysm.last_host_copy_bytes()[0]
    assert _expected_stream_h2d(sysm, n, "trajectory", flow_bytes) < triples


@pytest.mark.gpu
def test_argument_errors_name_the_input():
    _need_gpu()
    sysm = _system(HEADLINE, 4)
    lib, h = sysm._lib, sysm._h
    img, fwd, bwd, seg, _ = _seq(6)
    ALL = _capi.PAIRS["all"]
    o = C.c_void_p()
    assert lib.davo_odometry_create(h, 5, ALL, 1, C.byref(o)) == -1 and "max_push" in _capi.last_error(lib, h)
    assert lib.davo_odometry_create(h, 4, _capi.PAIRS["trajectory_first"], 1, C.byref(o)) == -1
    assert lib.davo_odometry_create(h, 4, ALL, 1, C.byref(o)) == 0
    pose, traj = np.zeros((4, 2, 6), np.float32), np.zeros((6, 4, 4))
    hp = lambda a, off=0: C.c_void_p(a.ctypes.data + off) if a is not None else None
    ns, nt = C.c_int(-1), C.c_int(-1)

    def push(k, i, f, b, s, off=None):
        args = [i, f, b, s]
        if off is not None:
            args[off] = C.c_void_p(args[off].value + 4)
        rc = lib.davo_odometry_push(o, k, *args, None, hp(pose), hp(traj), C.byref(ns), C.byref(nt), None, None)
        return rc, _capi.last_error(lib, h)

    good = (hp(img), hp(fwd), hp(bwd), hp(seg))
    assert push(0, *good)[0] == -1 and "k=0" in push(0, *good)[1]
    rc, msg = push(5, *good)
    assert rc == -1 and "max_push" in msg
    for i, name in ((0, "img"), (1, "flow_fwd"), (2, "flow_bwd"), (3, "seg")):
        args = list(good)
        args[i] = None
        rc, msg = push(3, *args)
        assert rc == -1 and name in msg, (name, msg)
        rc, msg = push(3, *good, off=i)
        assert rc == -1 and name in msg and "aligned" in msg, (name, msg)
    frames = lambda: (lambda a, b: (lib.davo_odometry_frames(o, C.byref(a), C.byref(b)), a.value, b.value))(C.c_longlong(), C.c_longlong())
    assert frames() == (0, 0, 0)                              # refused pushes change nothing
    assert push(1, hp(img), None, None, hp(seg))[0] == 0      # one frame: no flow, no sample
    assert (ns.value, nt.value) == (0, 0) and frames() == (0, 1, 0)
    rc, msg = lib.davo_odometry_push(o, 1, hp(img[1:]), hp(fwd), hp(bwd), hp(seg[1:]), None, hp(pose), hp(traj), None,
                                     None, None, C.byref(C.c_longlong())), _capi.last_error(lib, h)
    assert rc == 0                                            # a host session takes a ticket
    lib.davo_odometry_destroy(o)
    rc = push(1, *good)[0]
    assert rc == -1 and "destroyed" in _capi.last_error(lib, None)
    od = sysm.odometry(host=False)
    with pytest.raises(ValueError, match="flow_fwd"):        # a first push of k frames has k-1 flow entries
        od.push(*(torch.as_tensor(x).cuda() for x in (img[:3], fwd[:3], bwd[:2], seg[:3])))
    with pytest.raises(ValueError, match="img"):
        od.push(img[:3], fwd[:2], bwd[:2], seg[:3])            # a device session takes CUDA tensors
    rc = lib.davo_odometry_push(od._o, 1, C.c_void_p(torch.as_tensor(img[:1]).cuda().data_ptr()), None, None,
                                C.c_void_p(torch.as_tensor(seg[:1]).cuda().data_ptr()), None, None, None, None, None,
                                None, C.byref(C.c_longlong()))
    assert rc == -1 and "ticket" in _capi.last_error(lib, h)
    od.close()


def _ptxas(text):
    """{kernel: (registers, stack, spill stores, spill loads)} from ptxas -v output."""
    out, cur = {}, None
    for line in text.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            out[cur] = (None,) + tuple(int(x) for x in m.groups())
        m = re.search(r"Used (\d+) registers", line)
        if m and cur in out:
            out[cur] = (int(m.group(1)),) + out[cur][1:]
    return out


def test_forward_kernels_keep_their_registers_and_push_kernels_do_not_spill():
    """The build's ptxas report (davo_b200/csrc/build.log) against profiles/odometry_ptxas.txt: pack8_kernel and every
    conv kernel as recorded; odo_compose_many_kernel (its stack frame holds a matrix) and odo_widen_kernel without
    spills, odo_widen_kernel without a stack frame."""
    log = os.path.join(ROOT, "davo_b200", "csrc", "build.log")
    if not os.path.exists(log):
        pytest.skip("the library was not built by davo_b200/build.py here")
    got = _ptxas(open(log).read())
    rec = {}
    for line in open(os.path.join(ROOT, "profiles", "odometry_ptxas.txt")):
        m = re.match(r"(\S+) regs=(\d+) stack=(\d+) spill=\((\d+), (\d+)\)$", line.strip())
        if m:
            rec[m.group(1)] = tuple(int(x) for x in m.groups()[1:])
    names = [k for k in rec if "pack8_kernel" in k or "conv" in k]
    assert len(names) >= 10
    for k in names:
        assert got[k] == rec[k], (k, got[k], rec[k])
    for name, tail in (("odo_compose_many_kernel", 2), ("odo_widen_kernel", 1)):
        ext = [k for k in got if name in k]
        assert len(ext) == 1 and got[ext[0]][tail:] == (0,) * (4 - tail), (name, got[ext[0]])
