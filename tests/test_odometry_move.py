"""Moving odometry sessions between handles (include/davo_b200.h: davo_odometry_move, davo_b200.davo.Odometry.move_to)
and the camera pool over several handles (davo_b200.odometry_pool.OdometryPool).

The defining property: every push after a move gives the bits it would have given without the move -- poses,
trajectory, counts and host-to-device bytes -- whatever the session's state at the move, and whichever handle (of the
same configuration and weights, on this device or another) it moves to."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from davo_b200 import _capi, synthetic as S
from davo_b200.davo import DAVO, Odometry
from davo_b200.odometry_pool import OdometryPool
from tests.golden import make_golden as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W = 128, 416
HEADLINE = G.CASES["headline"]


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _need_two():
    _need_gpu()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")


def _system(ver, max_batch, device=0, seed=31, micro_batch=0):
    sysm = DAVO(version=ver)
    sysm.setup_inference(H, W, "davo", 3, max_batch, device=device, micro_batch=micro_batch)
    sysm.load_weights(S.init_weights(ver, seed=seed, random_bias=True))
    return sysm


def _stream(n, seed):
    img, fwd, bwd, seg, depth = S.make_sequence(n, H, W, seed=seed)
    seg[0, :2, :3] = 255.0                                   # a few labels without a class
    return img, fwd, bwd, seg, depth


def _piece(s, a, k):
    """The push of frames [a, a+k): flow entries [a-1, a+k-1) ([0, k-1) for a first push)."""
    img, fwd, bwd, seg, depth = s
    fl = slice(max(a - 1, 0), a + k - 1)
    return img[a:a + k], fwd[fl], bwd[fl], seg[a:a + k], depth[a:a + k]


def _on(piece, od):
    """A piece as a device session on its current handle takes it."""
    if od._host:
        return piece
    dev = "cuda:%d" % od._system.device
    return tuple(torch.as_tensor(np.ascontiguousarray(x)).to(dev) for x in piece)


def _np(out):
    f = lambda x: x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
    return f(out["pose"]), f(out["trajectory"]), out["frames"]


def _same(a, b, what):
    pa, ta, fa = _np(a)
    pb, tb, fb = _np(b)
    assert np.array_equal(pa, pb) and np.array_equal(ta, tb) and fa == fb, what


def _push_kind(systems, sessions, entries, kind):
    """entries [(index, piece)]: pushed singly, or batched per current handle; results in entry order."""
    if kind == "single":
        return [sessions[i].push(*_on(p, sessions[i])) for i, p in entries]
    out = {}
    for s in systems:
        mine = [(i, p) for i, p in entries if sessions[i]._system is s]
        if not mine:
            continue
        sess = [sessions[i] for i, _ in mine]
        ins = list(zip(*[_on(p, sessions[i]) for i, p in mine]))
        res = s.odometry_push_many_host(sess, *ins) if sess[0]._host else s.odometry_push_many(sess, *ins)
        out.update({i: r for (i, _), r in zip(mine, res)})
    return [out[i] for i, _ in entries]


def _random_schedule(a, b):
    """7 sessions (4 host, 3 device, both pair modes) on handles a and b, moved between them at random points and at
    the corner cases; a twin of each on a third handle is pushed singly with no move."""
    ref = _system(HEADLINE, 12)
    systems = [a, b]
    modes = ["trajectory", "all", "trajectory", "all", "trajectory", "all", "trajectory"]
    host = [True, True, True, True, False, False, False]
    sm = [systems[i % 2].odometry(m, 4, host=h) for i, (m, h) in enumerate(zip(modes, host))]
    so = [ref.odometry(m, 4, host=h) for m, h in zip(modes, host)]
    lens = [30, 26, 34, 28, 30, 24, 32]
    streams = [_stream(n, seed=200 + i) for i, n in enumerate(lens)]
    other = lambda od: b if od._system is a else a
    rng = np.random.default_rng(17)
    pos = [0] * 7
    sm[0].move_to(other(sm[0]))                              # before the first push
    for step in range(14):
        if step == 6:                                        # a reset, and a move right after it
            sm[2].reset()
            so[2].reset()
            pos[2] = 0
            sm[2].move_to(other(sm[2]))
        if step == 3 and pos[3] + 2 <= lens[3]:              # a host push still in flight when the session moves
            p = _piece(streams[3], pos[3], 2)
            pos[3] += 2
            pend = sm[3].push_async(*p)
            sm[3].move_to(other(sm[3]))
            _same(pend.result(), so[3].push(*p), ("in flight", step))
        entries = []
        for i in range(7):
            if pos[i] >= lens[i] or (step > 0 and rng.random() < 0.3):
                continue
            # first pushes of 1 and 2 frames, moved right after (a carried head shorter than 2)
            k = {1: 1, 4: 2, 5: 1}.get(i, 3) if pos[i] == 0 else int(rng.integers(1, 5))
            k = min(k, lens[i] - pos[i])
            entries.append((i, _piece(streams[i], pos[i], k)))
            pos[i] += k
        hosts = [(i, p) for i, p in entries if host[i]]
        devs = [(i, p) for i, p in entries if not host[i]]
        for group in (hosts, devs):
            kind = "single" if rng.random() < 0.4 else "batched"
            got = _push_kind(systems, sm, group, kind)
            want = [so[i].push(*_on(p, so[i])) for i, p in group]
            for (i, _), g, w in zip(group, got, want):
                _same(g, w, (step, i, kind))
                assert sm[i].frames() == so[i].frames()
        for i in range(7):
            if pos[i] in (1, 2) or rng.random() < 0.25:
                sm[i].move_to(other(sm[i]))
    for od in sm + so:
        od.close()
    ref.close()


@pytest.mark.gpu
def test_random_moves_on_one_device_give_the_bits_of_no_move():
    _need_gpu()
    a, b = _system(HEADLINE, 12), _system(HEADLINE, 20)      # two handles of different max_batch on device 0
    _random_schedule(a, b)
    a.close()
    b.close()


@pytest.mark.gpu
def test_random_moves_across_two_devices_give_the_bits_of_no_move():
    _need_two()
    a, b = _system(HEADLINE, 12, device=0), _system(HEADLINE, 20, device=1)
    _random_schedule(a, b)
    a.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("key,float_labels", [("headline", False), ("se_depth", False), ("decouple_net", False),
                                              ("headline", True)])
def test_moves_keep_the_bits_of_every_kind_of_carried_state(key, float_labels, monkeypatch):
    """Carried state that differs by variant: the headline version in both modes (an all-mode session carries a
    flow_fwd entry), a depth source (carries depth planes), a non-shared net, host sessions with float labels."""
    _need_gpu()
    if float_labels:
        monkeypatch.setenv("DAVO_B200_HOST_SEG8", "0")
    ver = G.CASES[key]
    a, b, ref = _system(ver, 8), _system(ver, 14), _system(ver, 8)
    specs = [("trajectory", True), ("all", True), ("trajectory", False), ("all", False)]
    sm = [a.odometry(m, 4, host=h) for m, h in specs]
    so = [ref.odometry(m, 4, host=h) for m, h in specs]
    streams = [_stream(16, seed=300 + i) for i in range(4)]
    pos = [0] * 4
    for step, k in enumerate([2, 1, 3, 1, 4, 2]):
        for i in range(4):
            p = _piece(streams[i], pos[i], k)
            _same(sm[i].push(*_on(p, sm[i])), so[i].push(*_on(p, so[i])), (key, step, i))
            if sm[i]._host:                                  # the bytes of the push too
                assert sm[i]._system.last_host_copy_bytes() == ref.last_host_copy_bytes(), (key, step, i)
            pos[i] += k
            sm[i].move_to(b if sm[i]._system is a else a)
    for od in sm + so:
        od.close()
    for s in (a, b, ref):
        s.close()


@pytest.mark.gpu
def test_ownership_follows_the_session():
    """After a move the old handle can go and the session still pushes with the same bits; it joins a batched push with
    the new handle's own sessions; when the new handle goes, the session goes with it."""
    _need_gpu()
    a, b, ref = _system(HEADLINE, 8), _system(HEADLINE, 12), _system(HEADLINE, 8)
    for host in (True, False):
        a = a if a._h is not None else _system(HEADLINE, 8)
        b = b if b._h is not None else _system(HEADLINE, 12)
        od, own = a.odometry("trajectory", 4, host=host), b.odometry("all", 4, host=host)
        tw, tw_own = ref.odometry("trajectory", 4, host=host), ref.odometry("all", 4, host=host)
        s, s2 = _stream(12, seed=90), _stream(12, seed=91)
        p = _piece(s, 0, 3)
        _same(od.push(*_on(p, od)), tw.push(*_on(p, tw)), "before")
        od.move_to(b)
        a.close()                                            # the old handle no longer owns it
        p, q = _piece(s, 3, 2), _piece(s2, 0, 3)
        ins = list(zip(_on(p, od), _on(q, own)))
        got = (b.odometry_push_many_host if host else b.odometry_push_many)([od, own], *ins)
        _same(got[0], tw.push(*_on(p, tw)), "batched with dst's own")
        _same(got[1], tw_own.push(*_on(q, tw_own)), "dst's own")
        b.close()                                            # the new one does
        with pytest.raises(RuntimeError, match="destroyed"):
            od.push(*_on(_piece(s, 5, 1), tw))
        for x in (tw, tw_own):
            x.close()
    ref.close()


@pytest.mark.gpu
def test_refused_moves_name_the_reason_and_change_nothing():
    _need_gpu()
    a, ref = _system(HEADLINE, 8), _system(HEADLINE, 8)
    lib = a._lib
    od, tw = a.odometry("all", 4), ref.odometry("all", 4)
    s = _stream(14, seed=95)
    _same(od.push(*_piece(s, 0, 3)), tw.push(*_piece(s, 0, 3)), "open")
    pos = 3

    def refused(dst, words):
        rc = lib.davo_odometry_move(od._o, dst)
        msg = _capi.last_error(lib, a._h)
        assert rc == -1 and all(w in msg for w in words), (words, msg)

    bare = DAVO(version=HEADLINE)
    bare.setup_inference(H, W, "davo", 3, 8, device=0)
    targets = [(None, ("dst is NULL",)),                     # the handles stay referenced until the end
               (_system(HEADLINE, 8, micro_batch=4), ("micro_batch", "max_batch may differ")),
               (_system(G.CASES["no_segmask"], 8), ("att_src",)),
               (_system(HEADLINE, 3), ("max_push 4", "max_batch 3")),
               (bare, ("not finalized",)),
               (_system(HEADLINE, 8, seed=32), ("different weights",))]
    for dst, words in targets:
        refused(None if dst is None else dst._h, words)
    dead = a.odometry("all", 4)
    dead_ptr = dead._o.value
    dead.close()
    rc = lib.davo_odometry_move(C.c_void_p(dead_ptr), ref._h)
    assert rc == -1 and "destroyed" in _capi.last_error(lib, None)
    rc = lib.davo_odometry_move(None, ref._h)
    assert rc == -1 and "NULL" in _capi.last_error(lib, None)
    assert lib.davo_odometry_move(od._o, a._h) == 0               # its own handle: nothing to do
    assert od._system is a and od.move_to(a) is od
    with pytest.raises(ValueError, match="not set up"):
        od.move_to(DAVO(version=HEADLINE))
    with pytest.raises(ValueError, match="no weights"):
        od.move_to(bare)
    other = _system(HEADLINE, 8, seed=33)
    with pytest.raises(RuntimeError, match="different weights"):
        od.move_to(other)
    assert od._system is a
    for step in range(3):                                    # still on its handle, with the bits of no move
        p = _piece(s, pos, 2)
        pos += 2
        _same(od.push(*p), tw.push(*p), ("after", step))
    od.close()
    tw.close()
    for s_ in [other, ref, a] + [d for d, _ in targets if d is not None]:
        s_.close()


@pytest.mark.gpu
def test_pool_pushes_equal_single_pushes_and_rebalance_keeps_the_bits():
    """A host and a device pool over two handles of device 0 (and device 1 where there is one): every push equals
    single pushes on one handle; open and close keep placement at the fewest sessions; rebalance keeps the bits."""
    _need_gpu()
    devices = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    for host in (True, False):
        systems = [_system(HEADLINE, 16, device=d) for d in devices]
        ref = _system(HEADLINE, 16)
        pool = OdometryPool(systems, pairs="trajectory", max_push=2, host=host)
        ids = [pool.open() for _ in range(5)]
        assert pool.counts() == [3, 2]
        twins = {c: ref.odometry("trajectory", 2, host=host) for c in ids}
        streams = {c: _stream(16, seed=400 + c) for c in ids}
        pos = {c: 0 for c in ids}

        def step(cams, k, what):
            pieces = {c: _piece(streams[c], pos[c], k) for c in cams}
            feed = lambda c: pieces[c] if host else tuple(
                torch.as_tensor(np.ascontiguousarray(x)).to("cuda:%d" % pool.device_of(c)) for x in pieces[c])
            got = pool.push(cams, *zip(*[feed(c) for c in cams]))
            for c, g in zip(cams, got):
                _same(g, twins[c].push(*_on(pieces[c], twins[c])), (what, c))
                pos[c] += k

        step(ids, 2, "open")
        step([ids[3], ids[0], ids[4]], 1, "subset, out of order")
        gone = (ids[0], ids[3])                              # one on each handle: [2, 1], the next goes to handle 1
        for c in gone:
            pool.close(c)
        assert pool.counts() == [2, 1]
        ids = [c for c in ids if c not in gone]
        c = pool.open()
        assert pool.counts() == [2, 2]
        twins[c], streams[c], pos[c] = ref.odometry("trajectory", 2, host=host), _stream(16, seed=400 + c), 0
        ids.append(c)
        for c in [x for x in ids if pool.session(x)._system is systems[1]]:
            pool.session(c).move_to(systems[0])              # drain handle 1
        assert pool.counts() == [4, 0]
        step(ids, 2, "drained")
        assert pool.rebalance() == 2 and pool.counts() == [2, 2]
        step(ids, 1, "rebalanced")
        step(ids, 2, "rebalanced again")
        pool.close_all()
        for od in twins.values():
            od.close()
        for s in systems + [ref]:
            s.close()


# ---- CPU ---------------------------------------------------------------------------------------------------------

def _stub_system(version="stub", hw=(4, 8), loaded=True):
    system = DAVO.__new__(DAVO)
    system.img_height, system.img_width = hw
    system.version, system.device, system._h, system._weights_loaded = version, 0, C.c_void_p(1), loaded
    system._lib = None                                       # any library call would fail: none may happen
    return system


def test_move_to_refuses_an_unset_or_mismatched_target_before_any_device_work():
    src = _stub_system()
    od = Odometry.__new__(Odometry)
    od._system, od._host, od._pushed, od._posed, od._o = src, True, 0, 0, C.c_void_p(1)
    with pytest.raises(ValueError, match="not set up"):
        od.move_to(DAVO(version="stub"))
    with pytest.raises(ValueError, match="not set up"):
        od.move_to(object())
    with pytest.raises(ValueError, match="no weights"):
        od.move_to(_stub_system(loaded=False))
    with pytest.raises(ValueError, match="version"):
        od.move_to(_stub_system(version="other"))
    with pytest.raises(ValueError, match="4x16"):
        od.move_to(_stub_system(hw=(4, 16)))
    assert od.move_to(src) is od and od._system is src
    od._o = None
    with pytest.raises(RuntimeError, match="closed"):
        od.move_to(_stub_system())


def test_pool_refuses_handles_that_cannot_share_cameras():
    with pytest.raises(ValueError, match="no handle"):
        OdometryPool([])
    with pytest.raises(ValueError, match="handle 1 is not set up"):
        OdometryPool([_stub_system(), _stub_system(loaded=False)])
    with pytest.raises(ValueError, match="handle 1 runs another version"):
        OdometryPool([_stub_system(), _stub_system(version="other")])
    s = _stub_system()
    with pytest.raises(ValueError, match="handle 1 is given twice"):
        OdometryPool([s, s])
    pool = OdometryPool([s, _stub_system()])
    assert pool.counts() == [0, 0]
    with pytest.raises(ValueError, match="camera 3 is not open"):
        pool.push([3], [None], None, None)


def test_the_library_declares_and_binds_the_move():
    assert "davo_odometry_move" in _capi.SYMBOLS
    hdr = open(os.path.join(ROOT, "include", "davo_b200.h")).read()
    assert re.search(r"int davo_odometry_move\(davo_odometry\*, davo_ctx\* dst\);", hdr)
    src = open(os.path.join(ROOT, "davo_b200", "_capi.py")).read()
    assert "lib.davo_odometry_move.argtypes = [vp, vp]" in src
