"""Saved odometry sessions (include/davo_b200.h: davo_odometry_save / _load and their _many forms; davo_b200.davo:
Odometry.save, DAVO.odometry_load, DAVO.odometry_save_many / odometry_load_many; OdometryPool.save / load).

The defining property: a session loaded from a blob continues the stream with the bits the saved session would have
given -- poses, trajectory, counts and host-to-device bytes -- whatever its state at the save, on whichever handle (of
the same configuration and weights, on this device, another one, or in another process) it is loaded."""
import ctypes as C
import os
import re
import struct
import subprocess
import sys

import numpy as np
import pytest
import torch

from davo_b200 import _capi, synthetic as S
from davo_b200.davo import DAVO, Odometry, odometry_blob_header
from davo_b200.odometry_pool import OdometryPool
from tests.golden import make_golden as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W = 128, 416
HEADLINE = G.CASES["headline"]
HEADER = 272
GOLDEN = 0x9E3779B97F4A7C15


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


def _checksum(blob):
    """numpy reference of the blob checksum (include/davo_b200.h)."""
    w = np.frombuffer(bytes(blob), "<u8").copy()
    w[HEADER // 8 - 1] = 0
    i = np.arange(1, w.size + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = w + i * np.uint64(GOLDEN)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return int(z.sum(dtype=np.uint64))


def _check_blob(blob, od):
    """The blob's header describes od, and its stored checksum is the numpy reference's."""
    h = odometry_blob_header(blob)
    assert h["total_bytes"] == len(bytes(blob)) and len(bytes(blob)) % 16 == 0
    assert (h["host"], h["pairs"], h["max_push"]) == (od._host, od.pairs, od.max_push)
    assert (h["pushed"], h["posed"]) == od.frames() and h["carried_frames"] == min(od.frames()[0], 2)
    assert h["checksum"] == _checksum(blob)
    return h


def _reload(od, dst):
    """od replaced by load(save()) on dst."""
    blob = od.save()
    _check_blob(blob, od)
    new = dst.odometry_load(blob)
    assert new.frames() == od.frames() and (new._host, new.pairs, new.max_push) == (od._host, od.pairs, od.max_push)
    assert new._system is dst
    od.close()
    return new


def _random_schedule(a, b):
    """7 sessions (4 host, 3 device, both pair modes) on handles a and b, replaced by load(save()) on the other handle
    at random points and at the corner cases; a twin of each on a third handle is pushed singly and never saved."""
    ref = _system(HEADLINE, 12)
    systems = [a] if a is b else [a, b]
    modes = ["trajectory", "all", "trajectory", "all", "trajectory", "all", "trajectory"]
    host = [True, True, True, True, False, False, False]
    sm = [systems[i % len(systems)].odometry(m, 4, host=h) for i, (m, h) in enumerate(zip(modes, host))]
    so = [ref.odometry(m, 4, host=h) for m, h in zip(modes, host)]
    lens = [30, 26, 34, 28, 30, 24, 32]
    streams = [_stream(n, seed=200 + i) for i, n in enumerate(lens)]
    other = lambda od: b if od._system is a else a
    rng = np.random.default_rng(17)
    pos = [0] * 7
    sm[0] = _reload(sm[0], other(sm[0]))                     # before the first push
    for step in range(14):
        if step == 6:                                        # a reset, and a reload right after it
            sm[2].reset()
            so[2].reset()
            pos[2] = 0
            sm[2] = _reload(sm[2], other(sm[2]))
        if step == 3 and pos[3] + 2 <= lens[3]:              # a host push still in flight at the save
            p = _piece(streams[3], pos[3], 2)
            pos[3] += 2
            pend = sm[3].push_async(*p)
            blob = sm[3].save()
            _same(pend.result(), so[3].push(*p), ("in flight", step))
            _check_blob(blob, sm[3])
            old, sm[3] = sm[3], other(sm[3]).odometry_load(blob)
            old.close()
        entries = []
        for i in range(7):
            if pos[i] >= lens[i] or (step > 0 and rng.random() < 0.3):
                continue
            # first pushes of 1 and 2 frames, reloaded right after (a carried head shorter than 2)
            k = {1: 1, 4: 2, 5: 1}.get(i, 3) if pos[i] == 0 else int(rng.integers(1, 5))
            k = min(k, lens[i] - pos[i])
            entries.append((i, _piece(streams[i], pos[i], k)))
            pos[i] += k
        for group in ([(i, p) for i, p in entries if host[i]], [(i, p) for i, p in entries if not host[i]]):
            if rng.random() < 0.4:                           # single pushes, host bytes compared push by push
                for i, p in group:
                    _same(sm[i].push(*_on(p, sm[i])), so[i].push(*_on(p, so[i])), (step, i, "single"))
                    if host[i]:
                        assert sm[i]._system.last_host_copy_bytes() == ref.last_host_copy_bytes(), (step, i)
                    assert sm[i].frames() == so[i].frames()
                continue
            for s in systems:                                # batched per current handle
                mine = [(i, p) for i, p in group if sm[i]._system is s]
                if not mine:
                    continue
                sess = [sm[i] for i, _ in mine]
                ins = list(zip(*[_on(p, sm[i]) for i, p in mine]))
                got = s.odometry_push_many_host(sess, *ins) if sess[0]._host else s.odometry_push_many(sess, *ins)
                for (i, p), g in zip(mine, got):
                    _same(g, so[i].push(*_on(p, so[i])), (step, i, "batched"))
                    assert sm[i].frames() == so[i].frames()
        for i in range(7):
            if pos[i] in (1, 2) or rng.random() < 0.25:
                sm[i] = _reload(sm[i], other(sm[i]))
    for od in sm + so:
        od.close()
    ref.close()


@pytest.mark.gpu
def test_random_reloads_on_one_handle_give_the_bits_of_no_save():
    _need_gpu()
    a = _system(HEADLINE, 12)
    _random_schedule(a, a)
    a.close()


@pytest.mark.gpu
def test_random_reloads_across_two_handles_give_the_bits_of_no_save():
    _need_gpu()
    a, b = _system(HEADLINE, 12), _system(HEADLINE, 20)      # two handles of different max_batch on device 0
    _random_schedule(a, b)
    a.close()
    b.close()


@pytest.mark.gpu
def test_random_reloads_across_two_devices_give_the_bits_of_no_save():
    _need_two()
    a, b = _system(HEADLINE, 12, device=0), _system(HEADLINE, 20, device=1)
    _random_schedule(a, b)
    a.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("key,float_labels", [("headline", False), ("se_depth", False), ("decouple_net", False),
                                              ("headline", True)])
def test_reloads_keep_the_bits_of_every_kind_of_carried_state(key, float_labels, monkeypatch):
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
    kinds = set()
    for step, k in enumerate([2, 1, 3, 1, 4, 2]):
        for i in range(4):
            p = _piece(streams[i], pos[i], k)
            _same(sm[i].push(*_on(p, sm[i])), so[i].push(*_on(p, so[i])), (key, step, i))
            if sm[i]._host:                                  # the bytes of the push too
                assert sm[i]._system.last_host_copy_bytes() == ref.last_host_copy_bytes(), (key, step, i)
            pos[i] += k
            h = odometry_blob_header(sm[i].save())
            kinds |= {j for j in range(6) if h["section_bytes"][j]}
            sm[i] = _reload(sm[i], b if sm[i]._system is a else a)
    want = {0, 4, 5} | ({3} if key == "se_depth" else set()) | ({1, 2} if not float_labels else {2})
    assert want <= kinds, (key, sorted(kinds))
    for od in sm + so:
        od.close()
    for s in (a, b, ref):
        s.close()


@pytest.mark.gpu
def test_a_loaded_copy_forks_the_stream_and_save_changes_nothing():
    _need_gpu()
    a, b = _system(HEADLINE, 8), _system(HEADLINE, 8)
    for host in (True, False):
        od = a.odometry("all", 4, host=host)
        s = _stream(14, seed=60)
        od.push(*_on(_piece(s, 0, 3), od))
        blob = od.save()
        assert od.save() == blob and od.frames() == (3, 3)  # a save changes nothing
        forks = [a.odometry_load(blob), b.odometry_load(blob)]
        pos = 3
        for k in (2, 1, 3):
            p = _piece(s, pos, k)
            want = od.push(*_on(p, od))
            for f in forks:
                _same(f.push(*_on(p, f)), want, ("fork", host, pos))
                assert f.frames() == od.frames()
            pos += k
        for x in forks + [od]:
            x.close()
    a.close()
    b.close()


_CHILD = r"""
import sys
sys.path.insert(0, {root!r})
import numpy as np
from davo_b200 import synthetic as S
from davo_b200.davo import DAVO
from tests.test_odometry_save import _system, _stream, _piece, _on, _np
sysm = _system({ver!r}, 8, seed=31)
blobs = np.load({inp!r})
out = {{}}
for name in blobs.files:
    od = sysm.odometry_load(blobs[name].tobytes())
    s = _stream(16, seed=500 + int(name[-1]))
    pos = od.frames()[0]
    for j, k in enumerate((2, 3, 1)):
        pose, traj, frames = _np(od.push(*_on(_piece(s, pos, k), od)))
        out["%s_%d_pose" % (name, j)], out["%s_%d_traj" % (name, j)] = pose, traj
        pos += k
    od.close()
np.savez({outp!r}, **out)
sysm.close()
"""


@pytest.mark.gpu
def test_another_process_continues_the_stream(tmp_path):
    """Blobs written to a file; a child process builds a handle from the same version and weight seed, loads them,
    pushes the rest of each stream and writes its results; they are the bits of the parent's twins."""
    _need_gpu()
    a, ref = _system(HEADLINE, 8), _system(HEADLINE, 8)
    specs = [("trajectory", True), ("all", True), ("trajectory", False), ("all", False)]
    sm = [a.odometry(m, 4, host=h) for m, h in specs]
    tw = [ref.odometry(m, 4, host=h) for m, h in specs]
    blobs = {}
    for i, (od, t) in enumerate(zip(sm, tw)):
        s = _stream(16, seed=500 + i)
        for x in (od, t):
            x.push(*_on(_piece(s, 0, 3), x))
            x.push(*_on(_piece(s, 3, 2), x))
        blobs["s%d" % i] = np.frombuffer(od.save(), np.uint8)
    np.savez(tmp_path / "blobs.npz", **blobs)
    code = _CHILD.format(root=ROOT, ver=HEADLINE, inp=str(tmp_path / "blobs.npz"), outp=str(tmp_path / "out.npz"))
    res = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code], cwd=ROOT,
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    got = np.load(tmp_path / "out.npz")
    for i, t in enumerate(tw):
        s = _stream(16, seed=500 + i)
        pos = 5
        for j, k in enumerate((2, 3, 1)):
            pose, traj, _ = _np(t.push(*_on(_piece(s, pos, k), t)))
            assert np.array_equal(got["s%d_%d_pose" % (i, j)], pose) and np.array_equal(got["s%d_%d_traj" % (i, j)], traj), (i, j)
            pos += k
    for x in sm + tw:
        x.close()
    a.close()
    ref.close()


@pytest.mark.gpu
def test_batched_forms_equal_the_single_forms():
    """save_many writes the bytes of n single saves; load_many sessions equal single-loaded ones; the launches are the
    same for 2 and 16 sessions; a save's device-to-host bytes are the blobs'."""
    _need_gpu()
    a, b = _system(HEADLINE, 8), _system(HEADLINE, 8)
    launches = {}
    for host in (True, False):
        for n in (2, 16):
            sessions = [a.odometry("trajectory" if i % 3 else "all", 4, host=host) for i in range(n)]
            streams = [_stream(8, seed=600 + i) for i in range(n)]
            for i, od in enumerate(sessions):                # every state: fresh, 1, 2, 3+ frames
                if i % 4:
                    od.push(*_on(_piece(streams[i], 0, i % 4), od))
            many = a.odometry_save_many(sessions)
            launches[(host, n, "save")] = a.last_launch_count()
            total = sum(len(bytes(x)) for x in many)
            assert a.last_host_copy_bytes()[1] == total
            singles = [od.save() for od in sessions]
            assert [bytes(x) for x in many] == singles
            loaded = b.odometry_load_many(many)
            launches[(host, n, "load")] = b.last_launch_count()
            alone = [b.odometry_load(x) for x in singles]
            for i, (x, y) in enumerate(zip(loaded, alone)):
                assert x.frames() == y.frames() == sessions[i].frames()
                p = _piece(streams[i], x.frames()[0], 2)
                want = sessions[i].push(*_on(p, sessions[i]))
                _same(x.push(*_on(p, x)), want, (host, n, i, "load_many"))
                _same(y.push(*_on(p, y)), want, (host, n, i, "load"))
            for x in sessions + loaded + alone:
                x.close()
    for host in (True, False):
        for kind in ("save", "load"):
            assert launches[(host, 2, kind)] == launches[(host, 16, kind)] == 1, launches
    a.close()
    b.close()


def _load_rc(dst, blob, lib):
    """davo_odometry_load of raw bytes: (rc, message, whether *out was left untouched)."""
    a = np.frombuffer(bytes(blob), np.uint8)
    out = C.c_void_p(12345)
    rc = lib.davo_odometry_load(dst, C.c_void_p(a.ctypes.data) if a.size else None, a.size, C.byref(out))
    return rc, _capi.last_error(lib, dst), out.value == 12345


@pytest.mark.gpu
def test_refused_loads_and_saves_name_the_reason_and_change_nothing(monkeypatch):
    _need_gpu()
    a, ref = _system(HEADLINE, 8), _system(HEADLINE, 8)
    lib = a._lib
    od, tw = a.odometry("all", 4), ref.odometry("all", 4)
    s = _stream(16, seed=95)
    for x in (od, tw):
        x.push(*_piece(s, 0, 3))
    pos = 3
    blob = od.save()
    h = _check_blob(blob, od)
    assert all(h["section_bytes"][j] for j in (0, 1, 4, 5)), h["section_bytes"]   # img, byte labels, flow_fwd, pose

    def refused(dst, data, words):
        rc, msg, untouched = _load_rc(dst._h if dst is not None else None, data, lib)
        if dst is None:
            msg = _capi.last_error(lib, None)
        assert rc == -1 and untouched and all(w in msg for w in words), (words, msg)

    def patched(at, value, fmt="<I"):
        b = bytearray(blob)
        struct.pack_into(fmt, b, at, value)
        return bytes(b)

    def flipped(at):
        b = bytearray(blob)
        b[at] ^= 0x5A
        return bytes(b)

    refused(a, blob[:-16], ("header says",))                 # truncated
    refused(a, blob[:100], ("shorter than the 272-byte header",))
    refused(a, flipped(0), ("bad magic",))
    refused(a, patched(8, 2), ("format version 2",))
    refused(a, flipped(145), ("checksum",))                  # frames posed: only the checksum sees it
    refused(a, flipped(264), ("checksum",))                  # the checksum itself
    for j in range(6):                                       # one byte of every carried section
        if h["section_bytes"][j]:
            refused(a, flipped(h["section_off"][j] + h["section_bytes"][j] // 2), ("checksum",))
    refused(a, patched(152, 1, "<i"), ("disagree",))         # carried frames that disagree with the counts
    refused(None, blob, ("dst is NULL",))
    bare = DAVO(version=HEADLINE)
    bare.setup_inference(H, W, "davo", 3, 8, device=0)
    monkeypatch.setenv("DAVO_B200_HOST_SEG8", "0")
    floats = _system(HEADLINE, 8)                            # host sessions hold float labels
    monkeypatch.delenv("DAVO_B200_HOST_SEG8")
    monkeypatch.setenv("DAVO_B200_WEIGHT_ROUNDING", "nearest")
    nearest = _system(HEADLINE, 8)
    monkeypatch.delenv("DAVO_B200_WEIGHT_ROUNDING")
    targets = [(_system(HEADLINE, 8, micro_batch=4), ("micro_batch", "max_batch may differ")),
               (_system(G.CASES["no_segmask"], 8), ("att_src",)),
               (_system(HEADLINE, 3), ("max_push 4", "max_batch 3")),
               (bare, ("not finalized",)),
               (_system(HEADLINE, 8, seed=32), ("different weights",)),
               (nearest, ("DAVO_B200_WEIGHT_ROUNDING",)),
               (floats, ("labels", "DAVO_B200_HOST_SEG8"))]
    for dst, words in targets:
        refused(dst, blob, words)
    # NULL pointers
    out = C.c_void_p(12345)
    assert lib.davo_odometry_load(a._h, None, len(blob), C.byref(out)) == -1 and out.value == 12345
    assert "buf is NULL" in _capi.last_error(lib, a._h)
    raw = np.frombuffer(blob, np.uint8)
    assert lib.davo_odometry_load(a._h, C.c_void_p(raw.ctypes.data), len(blob), None) == -1
    assert "out is NULL" in _capi.last_error(lib, a._h)
    # the _many form names the blob
    two = np.frombuffer(blob + flipped(h["section_off"][0] + 7), np.uint8)
    offs = (C.c_int64 * 3)(0, len(blob), 2 * len(blob))
    outs = (C.c_void_p * 2)(1, 2)
    assert lib.davo_odometry_load_many(a._h, 2, C.c_void_p(two.ctypes.data), offs, outs) == -1
    assert "blob[1]: checksum" in _capi.last_error(lib, a._h) and list(outs) == [1, 2]
    # saves: capacity too small reports the size, a destroyed session, sessions of two handles
    size = C.c_int64(0)
    small = np.zeros(16, np.uint8)
    assert lib.davo_odometry_save(od._o, C.c_void_p(small.ctypes.data), 16, C.byref(size)) == -1
    assert size.value == len(blob) and "capacity 16" in _capi.last_error(lib, a._h) and not small.any()
    big = np.zeros(2 * len(blob), np.uint8)
    offs = (C.c_int64 * 3)()
    pair = (C.c_void_p * 2)(od._o.value, tw._o.value)
    assert lib.davo_odometry_save_many(2, pair, C.c_void_p(big.ctypes.data), big.size, offs) == -1
    assert "sessions[1] belongs to another handle" in _capi.last_error(lib, a._h)
    dead = a.odometry("all", 4)
    dead_ptr = dead._o.value
    dead.close()
    assert lib.davo_odometry_save(C.c_void_p(dead_ptr), C.c_void_p(big.ctypes.data), big.size, C.byref(size)) == -1
    assert "destroyed" in _capi.last_error(lib, None)
    with pytest.raises(RuntimeError, match="closed"):
        dead.save()
    # Python checks before any device work
    with pytest.raises(ValueError, match="not set up"):
        DAVO(version=HEADLINE).odometry_load(blob)
    with pytest.raises(ValueError, match="no weights"):
        bare.odometry_load(blob)
    with pytest.raises(ValueError, match="no_segmask|att_src|another version"):
        targets[1][0].odometry_load(blob)
    with pytest.raises(RuntimeError, match="different weights"):
        targets[4][0].odometry_load(blob)
    assert od.save() == blob                                 # nothing changed
    for step in range(3):
        p = _piece(s, pos, 2)
        pos += 2
        _same(od.push(*p), tw.push(*p), ("after", step))
    od.close()
    tw.close()
    for s_ in [a, ref, floats, nearest] + [d for d, _ in targets]:
        s_.close()


@pytest.mark.gpu
def test_pool_save_and_load_restore_every_camera_with_its_bits():
    """OdometryPool.save on one pool, load on a fresh pool over fresh handles: the same ids, placement by the fewest
    sessions, every later pool push the twins' bits, and new ids above the restored ones."""
    _need_gpu()
    devices = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    for host in (True, False):
        systems = [_system(HEADLINE, 16, device=d) for d in devices]
        ref = _system(HEADLINE, 16)
        pool = OdometryPool(systems, pairs="trajectory", max_push=2, host=host)
        ids = [pool.open() for _ in range(5)]
        pool.close(ids.pop(1))                               # ids 0, 2, 3, 4
        twins = {c: ref.odometry("trajectory", 2, host=host) for c in ids}
        streams = {c: _stream(16, seed=700 + c) for c in ids}
        pos = {c: 0 for c in ids}

        def step(p, cams, k, what):
            pieces = {c: _piece(streams[c], pos[c], k) for c in cams}
            feed = lambda c: pieces[c] if host else tuple(
                torch.as_tensor(np.ascontiguousarray(x)).to("cuda:%d" % p.device_of(c)) for x in pieces[c])
            got = p.push(cams, *zip(*[feed(c) for c in cams]))
            for c, g in zip(cams, got):
                _same(g, twins[c].push(*_on(pieces[c], twins[c])), (what, c))
                pos[c] += k

        step(pool, ids, 2, "open")
        step(pool, ids[:3], 1, "subset")
        blobs = pool.save()
        assert sorted(blobs) == ids
        for c in ids:
            assert bytes(blobs[c]) == pool.session(c).save()
        pool.close_all()
        for s in systems:
            s.close()
        systems = [_system(HEADLINE, 12, device=d) for d in devices]          # a restarted process's handles
        fresh = OdometryPool(systems, pairs="trajectory", max_push=2, host=host)
        assert fresh.load(blobs) == ids and fresh.counts() == [2, 2]
        with pytest.raises(ValueError, match="camera 0 is open"):
            fresh.load({0: blobs[0]})
        for c in ids:
            assert fresh.session(c).frames() == twins[c].frames()
        step(fresh, ids, 2, "restored")
        step(fresh, ids[::-1], 1, "restored, out of order")
        assert fresh.open() == 5
        fresh.close_all()
        for od in twins.values():
            od.close()
        for s in systems + [ref]:
            s.close()


# ---- CPU ---------------------------------------------------------------------------------------------------------

def _blob(fields=None, sections=(96, 0, 0, 0, 32, 128), seed=0):
    """A blob laid out by the documented format, with random section bytes and the numpy reference's checksum."""
    f = dict(magic=b"DAVOSESS", version=1, header=HEADER, config=list(range(1, 21)), digest=0x1234567890ABCDEF,
             rounding=1, conv=0, host=1, label=1, pairs=1, max_push=4, pushed=7, posed=7, frames=2, fwd=1, pose=1)
    f.update(fields or {})
    off, at = [], HEADER
    for b in sections:
        off.append(at)
        at += (b + 15) // 16 * 16
    rng = np.random.default_rng(seed)
    body = bytearray(at)
    for o, b in zip(off, sections):
        body[o:o + b] = rng.integers(0, 256, b, dtype=np.uint8).tobytes()
    struct.pack_into("<8sIIQ20iQ6i2q4i6Q6QQ", body, 0, f["magic"], f["version"], f["header"], at, *f["config"],
                     f["digest"], f["rounding"], f["conv"], f["host"], f["label"], f["pairs"], f["max_push"],
                     f["pushed"], f["posed"], f["frames"], f["fwd"], f["pose"], 0, *off, *sections, 0)
    struct.pack_into("<Q", body, HEADER - 8, _checksum(body))
    return bytes(body)


def test_the_checksum_reference_is_splitmix64_and_order_free():
    # a blob of zero words: term 0 is splitmix64's first output from state 0, 0xE220A8397B1DCDAF
    b = bytes(HEADER + 16)
    ref = 0
    for i in range(len(b) // 8):
        z = (i + 1) * GOLDEN % 2 ** 64
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9 % 2 ** 64
        z = (z ^ (z >> 27)) * 0x94D049BB133111EB % 2 ** 64
        z ^= z >> 31
        if i == 0:
            assert z == 0xE220A8397B1DCDAF
        ref = (ref + z) % 2 ** 64
    assert _checksum(b) == ref
    # the stored checksum word does not count, and every other word does, wherever it is
    blob = _blob()
    assert _checksum(blob) == struct.unpack_from("<Q", blob, HEADER - 8)[0]
    c = bytearray(blob)
    c[HEADER - 3] ^= 1
    assert _checksum(c) == _checksum(blob)
    for at in (0, 145, HEADER, len(blob) - 1):
        c = bytearray(blob)
        c[at] ^= 1
        assert _checksum(c) != _checksum(blob), at


def test_the_header_parses_as_documented():
    blob = _blob()
    h = odometry_blob_header(blob)
    assert h["total_bytes"] == len(blob) == HEADER + 96 + 32 + 128
    assert h["config"]["H"] == 1 and h["config"]["W"] == 2 and h["config"]["posenn"] == 3 and h["config"]["batch_norm"] == 20
    assert "max_batch" not in h["config"]
    assert (h["host"], h["pairs"], h["max_push"], h["pushed"], h["posed"]) == (True, "trajectory", 4, 7, 7)
    assert (h["carried_frames"], h["carried_fwd"], h["carried_pose"], h["label_form"]) == (2, True, True, 1)
    assert h["section_off"] == [HEADER, HEADER + 96, HEADER + 96, HEADER + 96, HEADER + 96, HEADER + 128]
    assert h["section_bytes"] == [96, 0, 0, 0, 32, 128] and h["weights_digest"] == 0x1234567890ABCDEF
    assert h["checksum"] == _checksum(blob)
    assert odometry_blob_header(memoryview(bytearray(blob)))["checksum"] == h["checksum"]
    with pytest.raises(ValueError, match="truncated"):
        odometry_blob_header(blob[:200])
    with pytest.raises(ValueError, match="bad magic"):
        odometry_blob_header(_blob({"magic": b"DAVOSES?"}))
    with pytest.raises(ValueError, match="version 3"):
        odometry_blob_header(_blob({"version": 3}))


def _stub_system(version="stub", hw=(4, 8), loaded=True, **cfg):
    system = DAVO.__new__(DAVO)
    system.img_height, system.img_width = hw
    system.version, system.device, system._h, system._weights_loaded = version, 0, C.c_void_p(1), loaded
    system._lib = None                                       # any library call would fail: none may happen
    c = dict(zip([n for n, _ in _capi.DavoConfigC._fields_], range(1, 22)))
    c.update(H=hw[0], W=hw[1], **cfg)
    system._cfg = _capi.DavoConfigC(**c)
    return system


def _stub_blob(**fields):
    cfg = [v for n, v in zip([n for n, _ in _capi.DavoConfigC._fields_], range(1, 22)) if n != "max_batch"]
    cfg[0], cfg[1] = 4, 8
    return _blob({"config": cfg, **fields})


def test_loads_refuse_an_unset_handle_or_a_foreign_blob_before_any_device_work():
    blob = _stub_blob()
    with pytest.raises(ValueError, match="not set up"):
        DAVO(version="stub").odometry_load(blob)
    with pytest.raises(ValueError, match="no weights"):
        _stub_system(loaded=False).odometry_load(blob)
    with pytest.raises(ValueError, match="4x8, this handle's 4x16"):
        _stub_system(hw=(4, 16)).odometry_load(blob)
    with pytest.raises(ValueError, match="davo_config.att_src"):
        _stub_system(att_src=99).odometry_load(blob)
    with pytest.raises(ValueError, match="bad magic"):
        _stub_system().odometry_load(_stub_blob(magic=b"XXXXXXXX"))
    with pytest.raises(ValueError, match="version 2"):
        _stub_system().odometry_load_many([blob, _stub_blob(version=2)])
    with pytest.raises(ValueError, match="blob 1: .*truncated"):
        _stub_system().odometry_load_many([blob, blob[:100]])
    with pytest.raises(ValueError, match="no blob"):
        _stub_system().odometry_load_many([])
    s = _stub_system()
    with pytest.raises(ValueError, match="session 0 is not a session of this handle"):
        s.odometry_save_many([object()])
    pool = OdometryPool([_stub_system(), _stub_system()], pairs="trajectory", max_push=4, host=True)
    with pytest.raises(ValueError, match="camera 3 was saved as a device session"):
        pool.load({2: blob, 3: _stub_blob(host=0)})
    with pytest.raises(ValueError, match="max_push=4"):
        OdometryPool([_stub_system()], pairs="trajectory", max_push=2, host=True).load({0: blob})
    with pytest.raises(ValueError, match="another version"):
        pool.load({0: blob, 1: _stub_blob(config=[4, 8] + [0] * 18)})
    assert pool.counts() == [0, 0]


def test_the_library_declares_and_binds_save_and_load():
    names = ("davo_odometry_state_bytes", "davo_odometry_save", "davo_odometry_load", "davo_odometry_save_many",
             "davo_odometry_load_many")
    assert all(n in _capi.SYMBOLS for n in names)
    hdr = open(os.path.join(ROOT, "include", "davo_b200.h")).read()
    assert re.search(r"int davo_odometry_state_bytes\(const davo_odometry\*, int64_t\* bytes\);", hdr)
    assert re.search(r"int davo_odometry_save\(davo_odometry\*, void\* buf, int64_t capacity, int64_t\* bytes\);", hdr)
    assert re.search(r"int davo_odometry_load\(davo_ctx\* dst, const void\* buf, int64_t bytes, davo_odometry\*\* out\);", hdr)
    assert re.search(r"int davo_odometry_save_many\(int n, davo_odometry\* const\* sessions, void\* buf, int64_t capacity, "
                     r"int64_t\* offsets\);", hdr)
    assert re.search(r"int davo_odometry_load_many\(davo_ctx\* dst, int n, const void\* buf, const int64_t\* offsets, "
                     r"davo_odometry\*\* out\);", hdr)
    src = open(os.path.join(ROOT, "davo_b200", "_capi.py")).read()
    for n in names:
        assert "lib.%s.argtypes" % n in src


def test_ptxas_record_shows_no_spills_in_the_new_kernels():
    rec = {}
    for line in open(os.path.join(ROOT, "profiles", "odometry_save_ptxas.txt")):
        m = re.match(r"(\S+) regs=(\d+) stack=(\d+) spill=\((\d+), (\d+)\)$", line.strip())
        if m:
            rec[m.group(1)] = tuple(int(x) for x in m.groups()[1:])
    for name in ("odo_save_kernel", "odo_load_kernel"):
        got = [v for k, v in rec.items() if name in k]
        assert len(got) == 1 and got[0][1:] == (0, 0, 0), (name, got)
    assert [v for k, v in rec.items() if "pack8_kernel" in k] == [(56, 0, 0, 0)]
