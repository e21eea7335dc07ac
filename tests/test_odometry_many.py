"""Batched odometry pushes (include/davo_b200.h: davo_odometry_push_many, davo_b200.davo.DAVO.odometry_push_many).

The defining property: a batched push gives every session the bits that pushing it alone gives, in array order -- its
poses, its trajectory, its counts, and every later push on it."""
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


def _stream(n, seed):
    """A seeded n-frame stream, host arrays and the same on the device."""
    img, fwd, bwd, seg, depth = S.make_sequence(n, H, W, seed=seed)
    seg[0, :2, :3] = 255.0                                   # a few labels without a class
    seg[-1, 5, :4] = np.nan
    host = (img, fwd, bwd, seg, depth)
    return host, tuple(torch.as_tensor(x).cuda() for x in host)


def _piece(dev, a, k):
    """The push of frames [a, a+k): flow entries [a-1, a+k-1) ([0, k-1) for a first push)."""
    img, fwd, bwd, seg, depth = dev
    fl = slice(max(a - 1, 0), a + k - 1)
    return img[a:a + k], fwd[fl], bwd[fl], seg[a:a + k], depth[a:a + k]


def _cpu(out):
    return out["pose"].cpu().numpy(), out["trajectory"].cpu().numpy(), out["frames"]


def _same(a, b, what):
    pa, ta, fa = _cpu(a)
    pb, tb, fb = _cpu(b)
    assert np.array_equal(pa, pb) and np.array_equal(ta, tb) and fa == fb, what


class _Twin(object):
    """The same sessions on two handles with the same weights: `many` pushes batched, `one` pushes each session alone."""

    def __init__(self, ver, max_batch, modes, max_push=4, micro_batch=0):
        self.many, self.one = _system(ver, max_batch, micro_batch), _system(ver, max_batch, micro_batch)
        self.sm = [self.many.odometry(m, max_push, host=False) for m in modes]
        self.so = [self.one.odometry(m, max_push, host=False) for m in modes]

    def step(self, entries, what):
        """entries: [(session index, piece)]; checks batched against single, returns the single results."""
        got = self.many.odometry_push_many([self.sm[i] for i, _ in entries], *zip(*[p for _, p in entries]))
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
def test_random_batched_pushes_give_the_bits_of_single_pushes():
    """7 sessions, trajectory and all mode, streams of different lengths, 40 steps of random subsets with k in 1..4:
    first pushes of 1, 2 and 4 frames next to mid-stream ones, a reset in the middle.  Every result equals the single
    push, and each session's poses over its stream equal one sequence call."""
    _need_gpu()
    modes = ["trajectory", "all", "trajectory", "trajectory", "all", "trajectory", "all"]
    lens = [43, 30, 52, 25, 38, 61, 47]
    streams = [_stream(n, seed=100 + i) for i, n in enumerate(lens)]
    tw = _Twin(HEADLINE, 28, modes)
    rng = np.random.default_rng(17)
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
            entries.append((i, _piece(streams[i][1], pos[i], k)))
            pos[i] += k
        if not entries:
            continue
        for (i, _), out in zip(entries, tw.step(entries, step)):
            runs[i][-1].append((pos[i], out["pose"].cpu().numpy()))
    ref = _system(HEADLINE, max(lens))                       # the same weights, a batch the whole streams fit
    for i in range(7):
        for seg_ in runs[i]:
            if not seg_ or seg_[-1][0] < 3:
                continue
            n = seg_[-1][0]
            whole = ref.inference_sequence(*[x[:n] if j in (0, 3, 4) else x[:n - 1] for j, x in enumerate(streams[i][0])],
                                              pairs=FIRST[modes[i]])["pose"]
            assert np.array_equal(np.concatenate([p for _, p in seg_]), whole), i
    tw.close()


@pytest.mark.gpu
@pytest.mark.parametrize("key", [k for k in G.CASES if not V.parse_version(G.CASES[k]).batch_norm])
def test_every_variant_batched_equals_single(key):
    """One fixed schedule of 3 sessions: the non-shared nets, depth and per-pixel sources, static, -no_segmask, v0."""
    _need_gpu()
    tw = _Twin(G.CASES[key], 12, ["trajectory", "all", "trajectory"])
    streams = [_stream(14, seed=40 + i)[1] for i in range(3)]
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
def test_single_and_batched_pushes_mix_on_the_same_sessions():
    """Batched and single pushes alternate on the same sessions, with sequence calls, triplet calls and another
    session's pushes on the handle between them: the results equal an all-single run."""
    _need_gpu()
    modes = ["trajectory", "all", "trajectory"]
    tw = _Twin(HEADLINE, 12, modes)
    streams = [_stream(20, seed=60 + i)[1] for i in range(3)]
    other_seq = S.make_sequence(7, H, W, seed=6)
    trip = S.make_inputs(3, H, W, seed=2)
    other = tw.many.odometry("trajectory", 4, host=False)
    other_stream = _stream(12, seed=70)[1]
    pos, opos = [0, 0, 0], 0
    for step, ks in enumerate([(2, 3, 1), (1, 1, 1), (3, 2, 4), (1, 2, 1), (2, 1, 3), (1, 1, 1), (4, 3, 2)]):
        entries = [(i, _piece(streams[i], pos[i], k)) for i, k in enumerate(ks)]
        for i, k in enumerate(ks):
            pos[i] += k
        if step % 2:                                         # single pushes on the batched handle too
            for i, p in entries:
                _same(tw.sm[i].push(*p), tw.so[i].push(*p), (step, i))
        else:
            tw.step(entries, step)
        tw.many.inference_sequence(*other_seq, pairs="all")
        tw.many.inference(None, "pose", inputs=trip)
        if opos < 10:
            other.push(*_piece(other_stream, opos, 2))
            opos += 2
    other.close()
    tw.close()


@pytest.mark.gpu
def test_max_batch_samples_pass_and_one_more_is_refused():
    """Exactly max_batch samples over several micro-batch passes; max_batch + 1 is refused and changes nothing."""
    _need_gpu()
    tw = _Twin(HEADLINE, 12, ["trajectory", "all", "trajectory"], max_push=6, micro_batch=4)
    streams = [_stream(16, seed=80 + i)[1] for i in range(3)]
    pos = [0, 0, 0]

    def entries(ks):
        return [(i, _piece(streams[i], pos[i], k)) for i, k in enumerate(ks)]

    tw.step(entries((2, 2, 2)), "open")                      # no samples yet
    pos = [2, 2, 2]
    tw.step(entries((4, 4, 4)), "max_batch")                 # 12 samples; 12 pairs of both kinds: 3 passes of 4
    pos = [6, 6, 6]
    ks = (5, 4, 4)
    with pytest.raises(RuntimeError, match="max_batch"):
        tw.many.odometry_push_many(tw.sm, *zip(*[p for _, p in entries(ks)]))
    assert [od.frames() for od in tw.sm] == [od.frames() for od in tw.so]
    tw.step(entries((4, 4, 4)), "after")
    tw.close()


def _kernels_and_d2d(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kernels = [n for n in names if not n.startswith(("Memcpy", "Memset"))]
    d2d = [n for n in names if "DtoD" in n or "Device -> Device" in n]
    return kernels, d2d


class _Raw(object):
    """davo_odometry_push_many with every buffer allocated beforehand (so the profile holds the library's work only)."""

    def __init__(self, sysm, sessions, pieces):
        n = len(sessions)
        self.sysm, self.n = sysm, n
        vp = C.c_void_p
        arr = lambda vals: (vp * n)(*vals)
        ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None
        counts = [od._counts(int(p[0].shape[0])) for od, p in zip(sessions, pieces)]
        self.outs = [(torch.zeros((ns, 2, 6), device="cuda"), torch.zeros((nt, 4, 4), dtype=torch.float64, device="cuda"))
                     for ns, nt in counts]
        self.args = [n, arr([od._o.value for od in sessions]), (C.c_int * n)(*[int(p[0].shape[0]) for p in pieces])]
        self.args += [arr([ptr(p[j]) for p in pieces]) for j in range(5)]
        self.args += [arr([ptr(o[0]) for o in self.outs]), arr([ptr(o[1]) for o in self.outs]), None, None]

    def __call__(self):
        stream = torch.cuda.current_stream().cuda_stream
        rc = self.sysm._lib.davo_odometry_push_many(*self.args, C.c_void_p(stream))
        assert rc == 0, _capi.last_error(self.sysm._lib, self.sysm._h)


@pytest.mark.gpu
def test_launches_do_not_depend_on_the_number_of_sessions():
    """One batched push of 16 sessions launches as many kernels as one of 2 and copies nothing device to device."""
    _need_gpu()
    sysm = _system(HEADLINE, 32)
    dev = _stream(6, seed=90)[1]
    counts = []
    for n in (2, 16):
        sessions = [sysm.odometry("trajectory", 4, host=False) for _ in range(n)]
        sysm.odometry_push_many(sessions, *zip(*[_piece(dev, 0, 3)] * n))      # mid-stream from here on
        raw = _Raw(sysm, sessions, [_piece(dev, 3, 1)] * n)
        raw()                                                                   # warm
        raw = _Raw(sysm, sessions, [_piece(dev, 4, 1)] * n)
        kernels, d2d = _kernels_and_d2d(raw)
        assert d2d == [], d2d
        counts.append(len(kernels))
        assert any("odo_stage_kernel" in k for k in kernels) and any("odo_compose_many_kernel" in k for k in kernels)
        for od in sessions:
            od.close()
    assert counts[0] == counts[1], counts


@pytest.mark.gpu
def test_argument_errors_name_the_input_and_index_and_change_nothing():
    _need_gpu()
    modes = ["trajectory", "all"]
    tw = _Twin(HEADLINE, 6, modes, max_push=4)
    lib, h = tw.many._lib, tw.many._h
    streams = [_stream(12, seed=110 + i)[1] for i in range(2)]
    tw.step([(i, _piece(streams[i], 0, 3)) for i in range(2)], "open")
    pos = [3, 3]
    pieces = [_piece(streams[i], pos[i], 2) for i in range(2)]
    host_od = tw.many.odometry("trajectory", 4, host=True)
    foreign = tw.one.odometry("trajectory", 4, host=False)
    dead = tw.many.odometry("trajectory", 4, host=False)
    dead_ptr = dead._o.value
    dead.close()

    def call(n=2, sess=None, ks=(2, 2), edit=None, err_handle=h):
        raw = _Raw(tw.many, tw.sm, pieces)
        args = list(raw.args)
        args[0] = n
        if sess is not None:
            args[1] = (C.c_void_p * 2)(*sess)
        args[2] = (C.c_int * 2)(*ks)
        if edit:
            edit(args)
        rc = lib.davo_odometry_push_many(*args, None)
        return rc, _capi.last_error(lib, err_handle)

    me = [od._o.value for od in tw.sm]
    assert call(n=0)[0] == -1 and "n=0" in _capi.last_error(lib, None)
    rc, _ = call(sess=[me[0], None])
    assert rc == -1 and "sessions[1]" in _capi.last_error(lib, None)
    rc, _ = call(sess=[dead_ptr, me[1]])
    assert rc == -1 and "sessions[0]" in _capi.last_error(lib, None) and "destroyed" in _capi.last_error(lib, None)
    for sess, words in (([me[0], me[0]], ("sessions[1]", "twice")), ([me[0], host_od._o.value], ("sessions[1]", "host")),
                        ([me[0], foreign._o.value], ("sessions[1]", "handle"))):
        rc, msg = call(sess=sess)
        assert rc == -1 and all(w in msg for w in words), msg
    for ks, words in (((2, 0), ("k[1]", "max_push")), ((5, 2), ("k[0]", "max_push"))):
        rc, msg = call(ks=ks)
        assert rc == -1 and all(w in msg for w in words), msg
    # 7 samples from 4 + 3 new frames on mid-stream sessions, max_batch 6
    big = [_piece(streams[0], pos[0], 4), _piece(streams[1], pos[1], 3)]
    raw = _Raw(tw.many, tw.sm, big)
    assert lib.davo_odometry_push_many(*raw.args, None) == -1 and "max_batch" in _capi.last_error(lib, h)
    for col, name in ((3, "img"), (4, "flow_fwd"), (5, "flow_bwd"), (6, "seg"), (8, "pose_out"), (9, "traj_out")):
        for off, word in ((None, "NULL"), (4, "aligned")):
            def edit(args, col=col, off=off):
                vals = [args[col][0], args[col][1]]
                vals[1] = None if off is None else vals[1] + off
                args[col] = (C.c_void_p * 2)(*vals)
            rc, msg = call(edit=edit)                        # entry 1: an all-mode session, which reads every input
            assert rc == -1 and "%s[1]" % name in msg and word in msg, (name, word, msg)
    with pytest.raises(ValueError, match="session 1.*host"):
        tw.many.odometry_push_many([tw.sm[0], host_od], *zip(*pieces))
    short = list(pieces[0])
    short[1] = short[1][:1]                                  # one flow_fwd entry for two new frames
    with pytest.raises(ValueError, match="session 0: flow_fwd has shape"):
        tw.many.odometry_push_many(tw.sm, *zip(short, pieces[1]))
    # nothing of the above changed a session: they continue as the all-single twins
    for step in range(3):
        tw.step([(i, _piece(streams[i], pos[i], 2)) for i in range(2)], ("after", step))
        pos = [p + 2 for p in pos]
    host_od.close()
    foreign.close()
    tw.close()


# ---- CPU ---------------------------------------------------------------------------------------------------------

def _stub(host=False, pushed=0, system=None):
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
    b, h = _stub(system=sysm, pushed=5), _stub(host=True, system=sysm)
    img = lambda k: torch.zeros((k, 4, 8, 3), dtype=torch.uint8)
    fl = lambda k: torch.zeros((k, 4, 8, 2))
    seg = lambda k: torch.zeros((k, 4, 8, 1))
    with pytest.raises(ValueError, match="session 1 is a host session"):
        sysm.odometry_push_many([a, h], [img(1)] * 2, [fl(0), fl(1)], [fl(0), fl(1)], [seg(1)] * 2)
    with pytest.raises(ValueError, match="session 1 is given twice"):
        sysm.odometry_push_many([a, a], [img(1)] * 2, [fl(0)] * 2, [fl(0)] * 2, [seg(1)] * 2)
    with pytest.raises(ValueError, match="flow_bwd has 1 entries for 2 sessions"):
        sysm.odometry_push_many([a, b], [img(1)] * 2, [fl(0), fl(1)], [fl(0)], [seg(1)] * 2)
    with pytest.raises(ValueError, match="session 1: flow_fwd has shape"):      # mid-stream: k entries
        sysm.odometry_push_many([a, b], [img(2)] * 2, [fl(1), fl(1)], [fl(1), fl(2)], [seg(2)] * 2)
    with pytest.raises(ValueError, match="session 0: img must be a contiguous torch.uint8 tensor on cuda:0"):
        sysm.odometry_push_many([a, b], [img(2)] * 2, [fl(1), fl(2)], [fl(1), fl(2)], [seg(2)] * 2)
    with pytest.raises(ValueError, match="session 0 is not a session of this handle"):
        sysm.odometry_push_many([_stub()], [img(1)], [fl(0)], [fl(0)], [seg(1)])
    with pytest.raises(ValueError, match="no session"):
        sysm.odometry_push_many([], [], [], [])


def test_the_library_declares_and_binds_the_batched_push():
    assert "davo_odometry_push_many" in _capi.SYMBOLS
    hdr = open(os.path.join(ROOT, "include", "davo_b200.h")).read()
    assert re.search(r"int davo_odometry_push_many\(int n, davo_odometry\* const\* sessions", hdr)


def test_ptxas_record_shows_no_spills_in_the_new_kernels():
    rec = {}
    for line in open(os.path.join(ROOT, "profiles", "odometry_many_ptxas.txt")):
        m = re.match(r"(\S+) regs=(\d+) stack=(\d+) spill=\((\d+), (\d+)\)$", line.strip())
        if m:
            rec[m.group(1)] = tuple(int(x) for x in m.groups()[1:])
    for name in ("odo_stage_kernel", "odo_carry_kernel", "odo_compose_many_kernel", "traj_extend_kernel"):
        got = [v for k, v in rec.items() if name in k]
        assert len(got) == 1 and got[0][2:] == (0, 0), (name, got)
    pack8 = [v for k, v in rec.items() if "pack8_kernel" in k]
    assert pack8 == [(56, 0, 0, 0)]
