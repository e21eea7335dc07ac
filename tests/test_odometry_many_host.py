"""Batched pushes of host sessions (include/davo_b200.h: davo_odometry_push_many_host,
davo_b200.davo.DAVO.odometry_push_many_host).

The defining property: a batched host push gives every session the bits that pushing it alone with
davo_odometry_push gives, in array order -- its poses, its trajectory, its counts and every later push on it -- and
moves the bytes those single pushes move."""
import ctypes as C
import os
import re
import types

import numpy as np
import pytest
import torch

from davo_b200 import _capi, synthetic as S, version as V
from davo_b200.davo import DAVO, Odometry
from tests.golden import make_golden as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W = 128, 416
HEADLINE = G.CASES["headline"]
FIRST = {"trajectory": "trajectory_first", "all": "all"}      # the whole-sequence call a session's poses equal


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _system(ver, max_batch, micro_batch=0):
    sysm = DAVO(version=ver)
    sysm.setup_inference(H, W, "davo", 3, max_batch, device=0, micro_batch=micro_batch)
    sysm.load_weights(S.init_weights(ver, seed=31, random_bias=True))
    return sysm


def _stream(n, seed, pinned=False):
    """A seeded n-frame stream of host arrays (page-locked with `pinned`)."""
    img, fwd, bwd, seg, depth = S.make_sequence(n, H, W, seed=seed)
    seg[0, :2, :3] = 255.0                                   # a few labels without a class
    seg[-1, 5, :4] = np.nan
    host = (img, fwd, bwd, seg, depth)
    if pinned:
        host = tuple(torch.as_tensor(x).pin_memory().numpy() for x in host)
    return host


def _piece(s, a, k):
    """The push of frames [a, a+k): flow entries [a-1, a+k-1) ([0, k-1) for a first push)."""
    img, fwd, bwd, seg, depth = s
    fl = slice(max(a - 1, 0), a + k - 1)
    return img[a:a + k], fwd[fl], bwd[fl], seg[a:a + k], depth[a:a + k]


def _np(out):
    f = lambda x: x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
    return f(out["pose"]), f(out["trajectory"]), out["frames"]


def _same(a, b, what):
    pa, ta, fa = _np(a)
    pb, tb, fb = _np(b)
    assert np.array_equal(pa, pb) and np.array_equal(ta, tb) and fa == fb, what


class _Twin(object):
    """The same host sessions on two handles with the same weights: `many` pushes batched, `one` pushes each alone."""

    def __init__(self, ver, max_batch, modes, max_push=4, micro_batch=0):
        self.many, self.one = _system(ver, max_batch, micro_batch), _system(ver, max_batch, micro_batch)
        self.sm = [self.many.odometry(m, max_push, host=True) for m in modes]
        self.so = [self.one.odometry(m, max_push, host=True) for m in modes]

    def step(self, entries, what):
        """entries: [(session index, piece)]; checks batched against single, returns the single results."""
        got = self.many.odometry_push_many_host([self.sm[i] for i, _ in entries], *zip(*[p for _, p in entries]))
        want = [self.so[i].push(*p) for i, p in entries]
        for (i, _), g, w in zip(entries, got, want):
            _same(g, w, (what, i))
        for i, _ in entries:
            assert self.sm[i].frames() == self.so[i].frames()
        return want

    def close(self):
        for od in self.sm + self.so:
            od.close()


@pytest.mark.gpu
def test_random_batched_host_pushes_give_the_bits_of_single_pushes():
    """7 host sessions, trajectory and all mode, streams of different lengths, 40 steps of random subsets with k in
    1..4: first pushes of 1, 2 and 4 frames next to mid-stream ones, a reset in the middle.  Every result equals the
    single push, and each session's poses over its stream equal one sequence call."""
    _need_gpu()
    modes = ["trajectory", "all", "trajectory", "trajectory", "all", "trajectory", "all"]
    lens = [43, 30, 52, 25, 38, 61, 47]
    streams = [_stream(n, seed=100 + i) for i, n in enumerate(lens)]
    tw = _Twin(HEADLINE, 28, modes)
    rng = np.random.default_rng(23)
    start = [0, 0, 0, 2, 3, 5, 8]                            # sessions join late: first pushes among mid-stream ones
    first_k = [1, 2, 4, 1, 3, 2, 4]
    pos = [0] * 7
    runs = [[[]] for _ in range(7)]                          # per session: the poses of each segment between resets
    for step in range(40):
        if step == 20:                                       # a reset: a new sequence on a used session
            tw.sm[2].reset()
            tw.so[2].reset()
            pos[2] = 0
            runs[2].append([])
        entries = []
        for i in range(7):
            if step < start[i] or pos[i] >= lens[i] or (step > start[i] and rng.random() < 0.35):
                continue
            k = first_k[i] if pos[i] == 0 and step == start[i] else int(rng.integers(1, 5))
            k = min(k, lens[i] - pos[i])
            entries.append((i, _piece(streams[i], pos[i], k)))
            pos[i] += k
        if not entries:
            continue
        for (i, _), out in zip(entries, tw.step(entries, step)):
            runs[i][-1].append((pos[i], out["pose"]))
    ref = _system(HEADLINE, max(lens))                       # the same weights, a batch the whole streams fit
    for i in range(7):
        for seg_ in runs[i]:
            if not seg_ or seg_[-1][0] < 3:
                continue
            n = seg_[-1][0]
            whole = ref.inference_sequence(*[x[:n] if j in (0, 3, 4) else x[:n - 1] for j, x in enumerate(streams[i])],
                                           pairs=FIRST[modes[i]])["pose"]
            assert np.array_equal(np.concatenate([p for _, p in seg_]), whole), i
    tw.close()


@pytest.mark.gpu
@pytest.mark.parametrize("key", [k for k in G.CASES if not V.parse_version(G.CASES[k]).batch_norm])
def test_every_variant_batched_host_equals_single(key):
    """One fixed schedule of 3 sessions: the non-shared nets, depth and per-pixel sources, static, -no_segmask, v0."""
    _need_gpu()
    tw = _Twin(G.CASES[key], 12, ["trajectory", "all", "trajectory"])
    streams = [_stream(14, seed=40 + i) for i in range(3)]
    pos = [0, 0, 0]
    for step, ks in enumerate([(1, 3, 2), (2, 1, 4), (4, 2, 1), (1, 4, 3), (3, 1, 0)]):
        entries = []
        for i, k in enumerate(ks):
            if k:
                entries.append((i, _piece(streams[i], pos[i], k)))
                pos[i] += k
        tw.step(entries, (key, step))
    tw.close()


@pytest.mark.gpu
def test_single_and_batched_host_pushes_mix_on_the_same_sessions():
    """Batched and single host pushes alternate on the same sessions.  Some steps follow each other with nothing in
    between (the carried state passes from the caller's stream to the copy stream and back); others have host sequence
    calls, host triplet calls, another host session's pushes and a device batched push on the handle between them.
    The results equal an all-single run."""
    _need_gpu()
    modes = ["trajectory", "all", "trajectory"]
    tw = _Twin(HEADLINE, 12, modes)
    streams = [_stream(24, seed=60 + i) for i in range(3)]
    other_seq = S.make_sequence(7, H, W, seed=6)
    trip = S.make_inputs(3, H, W, seed=2)
    other = tw.many.odometry("trajectory", 4, host=True)
    other_stream = _stream(14, seed=70)
    dev_sess = [tw.many.odometry("trajectory", 4, host=False) for _ in range(2)]
    dev_stream = tuple(torch.as_tensor(x).cuda() for x in _stream(14, seed=71))
    pos, opos, dpos = [0, 0, 0], 0, 0
    plan = [(2, 3, 1), (1, 1, 1), (3, 2, 4), (1, 2, 1), (2, 1, 3), (1, 1, 1), (4, 3, 2), (1, 1, 1), (2, 2, 2)]
    for step, ks in enumerate(plan):
        entries = [(i, _piece(streams[i], pos[i], k)) for i, k in enumerate(ks)]
        for i, k in enumerate(ks):
            pos[i] += k
        if step % 2:                                         # single pushes on the batched handle too
            for i, p in entries:
                _same(tw.sm[i].push(*p), tw.so[i].push(*p), (step, i))
        else:
            tw.step(entries, step)
        if step % 4 in (0, 1):                               # back to back with the next step on some steps
            continue
        tw.many.inference_sequence(*other_seq, pairs="all")
        tw.many.inference(None, "pose", inputs=trip)
        if opos < 12:
            other.push(*_piece(other_stream, opos, 2))
            opos += 2
        if dpos < 12:
            tw.many.odometry_push_many(dev_sess, *zip(*[_piece(dev_stream, dpos, 2)] * 2))
            dpos += 2
    other.close()
    for od in dev_sess:
        od.close()
    tw.close()


@pytest.mark.gpu
def test_batched_host_pushes_in_flight_equal_the_blocking_form():
    """Up to 8 asynchronous batched pushes queued from page-locked inputs, then waited for in order and out of order:
    the results equal blocking single pushes."""
    _need_gpu()
    modes = ["trajectory", "all", "trajectory"]
    tw = _Twin(HEADLINE, 12, modes)
    streams = [_stream(40, seed=120 + i, pinned=True) for i in range(3)]
    pos = [0, 0, 0]
    rng = np.random.default_rng(5)
    for rnd, order in enumerate(("in order", "out of order")):
        pend, want = [], []
        for step in range(8):
            ks = [int(rng.integers(1, 4)) for _ in range(3)]
            entries = [(i, _piece(streams[i], pos[i], k)) for i, k in enumerate(ks)]
            for i, k in enumerate(ks):
                pos[i] += k
            pend.append(tw.many.odometry_push_many_host_async(tw.sm, *zip(*[p for _, p in entries])))
            want.append([tw.so[i].push(*p) for i, p in entries])
        idx = list(range(8)) if order == "in order" else [5, 7, 0, 3, 1, 6, 2, 4]
        got = {j: pend[j].result() for j in idx}
        for j in range(8):
            for i in range(3):
                _same(got[j][i], want[j][i], (order, j, i))
    tw.close()


@pytest.mark.gpu
def test_batched_host_pushes_equal_batched_device_pushes():
    """The same schedule as batched host pushes and as batched device pushes gives identical bits."""
    _need_gpu()
    modes = ["trajectory", "all", "trajectory", "all"]
    hs, ds = _system(HEADLINE, 16), _system(HEADLINE, 16)
    sh = [hs.odometry(m, 4, host=True) for m in modes]
    sd = [ds.odometry(m, 4, host=False) for m in modes]
    streams = [_stream(16, seed=140 + i) for i in range(4)]
    dev = [tuple(torch.as_tensor(x).cuda() for x in s) for s in streams]
    pos = [0] * 4
    for step, ks in enumerate([(1, 2, 4, 3), (2, 1, 1, 4), (4, 3, 2, 1), (1, 1, 1, 1), (3, 4, 2, 2)]):
        a = hs.odometry_push_many_host(sh, *zip(*[_piece(streams[i], pos[i], k) for i, k in enumerate(ks)]))
        b = ds.odometry_push_many(sd, *zip(*[_piece(dev[i], pos[i], k) for i, k in enumerate(ks)]))
        for i in range(4):
            _same(a[i], b[i], (step, i))
        pos = [p + k for p, k in zip(pos, ks)]
    for od in sh + sd:
        od.close()


@pytest.mark.gpu
def test_float_labels_give_the_bits_of_single_pushes(monkeypatch):
    """With DAVO_B200_HOST_SEG8=0 labels cross as float32 and the stage kernel narrows them; the results equal single
    pushes on a handle with the same setting."""
    _need_gpu()
    monkeypatch.setenv("DAVO_B200_HOST_SEG8", "0")
    tw = _Twin(HEADLINE, 12, ["trajectory", "all", "trajectory"])
    streams = [_stream(14, seed=150 + i) for i in range(3)]
    pos = [0, 0, 0]
    for step, ks in enumerate([(1, 3, 2), (2, 1, 4), (4, 2, 1), (1, 4, 3)]):
        tw.step([(i, _piece(streams[i], pos[i], k)) for i, k in enumerate(ks)], step)
        pos = [p + k for p, k in zip(pos, ks)]
    tw.close()


@pytest.mark.gpu
def test_max_batch_samples_pass_and_one_more_is_refused():
    """Exactly max_batch samples over several micro-batch passes; max_batch + 1 is refused and changes nothing."""
    _need_gpu()
    tw = _Twin(HEADLINE, 12, ["trajectory", "all", "trajectory"], max_push=6, micro_batch=4)
    streams = [_stream(16, seed=80 + i) for i in range(3)]
    pos = [0, 0, 0]

    def entries(ks):
        return [(i, _piece(streams[i], pos[i], k)) for i, k in enumerate(ks)]

    tw.step(entries((2, 2, 2)), "open")                      # no samples yet
    pos = [2, 2, 2]
    tw.step(entries((4, 4, 4)), "max_batch")                 # 12 samples; 12 pairs of both kinds: 3 passes of 4
    pos = [6, 6, 6]
    with pytest.raises(RuntimeError, match="max_batch"):
        tw.many.odometry_push_many_host(tw.sm, *zip(*[p for _, p in entries((5, 4, 4))]))
    assert [od.frames() for od in tw.sm] == [od.frames() for od in tw.so]
    tw.step(entries((4, 4, 4)), "after")
    tw.close()


@pytest.mark.gpu
def test_copy_bytes_equal_the_sum_of_the_single_pushes():
    """davo_last_host_copy_bytes of a batched push equals the sum over its sessions of the single pushes' counts, both
    ways: first pushes (where trajectory mode skips the second frame's labels) and mid-stream ones, both modes."""
    _need_gpu()
    modes = ["trajectory", "all", "trajectory", "all"]
    tw = _Twin(HEADLINE, 16, modes)
    streams = [_stream(16, seed=160 + i) for i in range(4)]
    pos = [0] * 4
    for step, ks in enumerate([(3, 2, 1, 4), (1, 2, 2, 1), (2, 1, 4, 3), (1, 1, 1, 1), (4, 3, 1, 2)]):
        entries = [(i, _piece(streams[i], pos[i], k)) for i, k in enumerate(ks)]
        got = tw.many.odometry_push_many_host(tw.sm, *zip(*[p for _, p in entries]))
        many = tw.many.last_host_copy_bytes()
        h2d = d2h = 0
        for (i, p), g in zip(entries, got):
            _same(g, tw.so[i].push(*p), (step, i))
            a, b = tw.one.last_host_copy_bytes()
            h2d, d2h = h2d + a, d2h + b
        assert many == (h2d, d2h), (step, many, (h2d, d2h))
        pos = [p + k for p, k in zip(pos, ks)]
    tw.close()


def _profile(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kernels = [n for n in names if not n.startswith(("Memcpy", "Memset"))]
    d2d = [n for n in names if "DtoD" in n or "Device -> Device" in n]
    h2d = [n for n in names if "HtoD" in n or "Host -> Device" in n]
    return kernels, d2d, h2d


@pytest.mark.gpu
def test_launches_do_not_depend_on_the_number_of_sessions():
    """One batched host push of 16 sessions launches as many kernels as one of 2, copies nothing device to device, and
    with one frame per session makes at most one host-to-device copy per input kind per session, plus a constant."""
    _need_gpu()
    sysm = _system(HEADLINE, 32)
    s = _stream(6, seed=90)
    kinds = 4                                                # img, seg, flow_fwd, flow_bwd (no depth in this variant)
    counts = []
    for n in (2, 16):
        sessions = [sysm.odometry("trajectory", 4, host=True) for _ in range(n)]
        sysm.odometry_push_many_host(sessions, *zip(*[_piece(s, 0, 3)] * n))   # mid-stream from here on
        sysm.odometry_push_many_host(sessions, *zip(*[_piece(s, 3, 1)] * n))   # warm
        kernels, d2d, h2d = _profile(lambda: sysm.odometry_push_many_host(sessions, *zip(*[_piece(s, 4, 1)] * n)))
        assert d2d == [], d2d
        assert len(h2d) <= kinds * n + 2, (n, len(h2d))
        counts.append(len(kernels))
        assert any("odo_stage_kernel" in k for k in kernels) and any("odo_compose_many_kernel" in k for k in kernels)
        for od in sessions:
            od.close()
    assert counts[0] == counts[1], counts


class _Raw(object):
    """davo_odometry_push_many_host on numpy buffers, with the argument arrays built once."""

    def __init__(self, sysm, sessions, pieces):
        n = len(sessions)
        self.sysm, self.n = sysm, n
        vp = C.c_void_p
        arr = lambda vals: (vp * n)(*vals)
        ptr = lambda a: a.ctypes.data if a is not None and a.size else None
        self.pieces = [tuple(np.ascontiguousarray(x) for x in p) for p in pieces]
        counts = [od._counts(int(p[0].shape[0])) for od, p in zip(sessions, pieces)]
        self.outs = [(np.zeros((ns, 2, 6), np.float32), np.zeros((nt, 4, 4), np.float64)) for ns, nt in counts]
        self.args = [n, arr([od._o.value for od in sessions]), (C.c_int * n)(*[int(p[0].shape[0]) for p in pieces])]
        self.args += [arr([ptr(p[j]) for p in self.pieces]) for j in range(5)]
        self.args += [arr([ptr(o[0]) for o in self.outs]), arr([ptr(o[1]) for o in self.outs]), None, None]


@pytest.mark.gpu
def test_argument_errors_name_the_input_and_index_and_change_nothing():
    _need_gpu()
    modes = ["trajectory", "all"]
    tw = _Twin(HEADLINE, 6, modes, max_push=4)
    lib, h = tw.many._lib, tw.many._h
    streams = [_stream(14, seed=110 + i) for i in range(2)]
    tw.step([(i, _piece(streams[i], 0, 3)) for i in range(2)], "open")
    pos = [3, 3]
    pieces = [_piece(streams[i], pos[i], 2) for i in range(2)]
    dev_od = tw.many.odometry("trajectory", 4, host=False)
    foreign = tw.one.odometry("trajectory", 4, host=True)
    dead = tw.many.odometry("trajectory", 4, host=True)
    dead_ptr = dead._o.value
    dead.close()
    keep = []

    def call(n=2, sess=None, ks=(2, 2), edit=None, err_handle=h):
        raw = _Raw(tw.many, tw.sm, pieces)
        keep.append(raw)
        args = list(raw.args)
        args[0] = n
        if sess is not None:
            args[1] = (C.c_void_p * 2)(*sess)
        args[2] = (C.c_int * 2)(*ks)
        if edit:
            edit(args)
        rc = lib.davo_odometry_push_many_host(*args, None, None)
        return rc, _capi.last_error(lib, err_handle)

    me = [od._o.value for od in tw.sm]
    assert call(n=0)[0] == -1 and "n=0" in _capi.last_error(lib, None)
    rc, _ = call(sess=[me[0], None])
    assert rc == -1 and "sessions[1]" in _capi.last_error(lib, None)
    rc, _ = call(sess=[dead_ptr, me[1]])
    assert rc == -1 and "sessions[0]" in _capi.last_error(lib, None) and "destroyed" in _capi.last_error(lib, None)
    for sess, words in (([me[0], me[0]], ("sessions[1]", "twice")),
                        ([me[0], dev_od._o.value], ("sessions[1]", "device session", "davo_odometry_push_many takes it")),
                        ([me[0], foreign._o.value], ("sessions[1]", "handle"))):
        rc, msg = call(sess=sess)
        assert rc == -1 and all(w in msg for w in words), msg
    for ks, words in (((2, 0), ("k[1]", "max_push")), ((5, 2), ("k[0]", "max_push"))):
        rc, msg = call(ks=ks)
        assert rc == -1 and all(w in msg for w in words), msg
    # 7 samples from 4 + 3 new frames on mid-stream sessions, max_batch 6
    raw = _Raw(tw.many, tw.sm, [_piece(streams[0], pos[0], 4), _piece(streams[1], pos[1], 3)])
    assert lib.davo_odometry_push_many_host(*raw.args, None, None) == -1 and "max_batch" in _capi.last_error(lib, h)
    for col, name in ((3, "img"), (4, "flow_fwd"), (5, "flow_bwd"), (6, "seg"), (8, "pose_out"), (9, "traj_out")):
        for off, word in ((None, "NULL"), (4, "aligned")):
            def edit(args, col=col, off=off):
                vals = [args[col][0], args[col][1]]
                vals[1] = None if off is None else vals[1] + off
                args[col] = (C.c_void_p * 2)(*vals)
            rc, msg = call(edit=edit)                        # entry 1: an all-mode session, which reads every input
            assert rc == -1 and "%s[1]" % name in msg and word in msg, (name, word, msg)
    with pytest.raises(ValueError, match="session 1 is a device session"):
        tw.many.odometry_push_many_host([tw.sm[0], dev_od], *zip(*pieces))
    with pytest.raises(ValueError, match="session 1 is a host session"):
        tw.many.odometry_push_many([dev_od, tw.sm[0]], *zip(*pieces))
    short = list(pieces[0])
    short[1] = short[1][:1]                                  # one flow_fwd entry for two new frames
    with pytest.raises(ValueError, match="session 0: flow_fwd has shape"):
        tw.many.odometry_push_many_host(tw.sm, *zip(short, pieces[1]))
    # nothing of the above changed a session: they continue as the all-single twins
    for step in range(3):
        tw.step([(i, _piece(streams[i], pos[i], 2)) for i in range(2)], ("after", step))
        pos = [p + 2 for p in pos]
    dev_od.close()
    foreign.close()
    tw.close()


# ---- CPU ---------------------------------------------------------------------------------------------------------

def _stub(host=True, pushed=0, system=None):
    if system is None:
        system = DAVO.__new__(DAVO)
        system.img_height, system.img_width, system.version, system.device = 4, 8, "stub", 0
        system.config = types.SimpleNamespace(att_src=1, depth_split=0)
    od = Odometry.__new__(Odometry)
    od._system, od._host, od._pushed, od._posed, od._o = system, host, pushed, 0, C.c_void_p(1)
    return od


def test_python_checks_refuse_before_any_device_work():
    a = _stub()
    sysm = a._system
    b, d = _stub(system=sysm, pushed=5), _stub(host=False, system=sysm)
    img = lambda k: np.zeros((k, 4, 8, 3), np.uint8)
    fl = lambda k: np.zeros((k, 4, 8, 2), np.float32)
    seg = lambda k: np.zeros((k, 4, 8, 1), np.float32)
    with pytest.raises(ValueError, match="session 1 is a device session"):
        sysm.odometry_push_many_host([a, d], [img(1)] * 2, [fl(0), fl(1)], [fl(0), fl(1)], [seg(1)] * 2)
    with pytest.raises(ValueError, match="session 1 is a host session"):
        sysm.odometry_push_many([d, a], [img(1)] * 2, [fl(0), fl(1)], [fl(0), fl(1)], [seg(1)] * 2)
    with pytest.raises(ValueError, match="session 1 is given twice"):
        sysm.odometry_push_many_host([a, a], [img(1)] * 2, [fl(0)] * 2, [fl(0)] * 2, [seg(1)] * 2)
    with pytest.raises(ValueError, match="flow_bwd has 1 entries for 2 sessions"):
        sysm.odometry_push_many_host([a, b], [img(1)] * 2, [fl(0), fl(1)], [fl(0)], [seg(1)] * 2)
    with pytest.raises(ValueError, match="session 1: flow_fwd has shape"):      # mid-stream: k entries
        sysm.odometry_push_many_host([a, b], [img(2)] * 2, [fl(1), fl(1)], [fl(1), fl(2)], [seg(2)] * 2)
    with pytest.raises(ValueError, match="session 0 is not a session of this handle"):
        sysm.odometry_push_many_host([_stub()], [img(1)], [fl(0)], [fl(0)], [seg(1)])
    with pytest.raises(ValueError, match="no session"):
        sysm.odometry_push_many_host([], [], [], [])
    with pytest.raises(ValueError, match="no session"):
        sysm.odometry_push_many_host_async([], [], [], [])


def test_the_library_declares_and_binds_the_batched_host_push():
    assert "davo_odometry_push_many_host" in _capi.SYMBOLS
    hdr = open(os.path.join(ROOT, "include", "davo_b200.h")).read()
    assert re.search(r"int davo_odometry_push_many_host\(int n, davo_odometry\* const\* sessions", hdr)
    assert re.search(r"int\* n_samples, int\* n_traj, void\* cuda_stream, long long\* ticket\);", hdr)


def test_ptxas_record_shows_no_spills_in_the_touched_kernels():
    rec = {}
    for line in open(os.path.join(ROOT, "profiles", "odometry_many_host_ptxas.txt")):
        m = re.match(r"(\S+) regs=(\d+) stack=(\d+) spill=\((\d+), (\d+)\)$", line.strip())
        if m:
            rec[m.group(1)] = tuple(int(x) for x in m.groups()[1:])
    for name in ("odo_stage_kernel", "odo_carry_kernel"):
        got = [v for k, v in rec.items() if name in k]
        assert len(got) == 1 and got[0][2:] == (0, 0), (name, got)
    pack8 = [v for k, v in rec.items() if "pack8_kernel" in k]
    assert pack8 == [(56, 0, 0, 0)]
