"""Attention out of the streaming paths (include/davo_b200.h: davo_forward_sequence_features, davo_odometry_attention).

The defining properties:
- mode='feature' on a frame sequence gives every output of mode='feature' on the triplets of the same frames, bit for bit;
- each posed frame's map from an odometry push is a plane of davo_forward_features on the triplets of the whole stream
  (frame 0: attention[1][0], frame 1: attention[0][0], frame s+2: attention[2][s]), and its weight rows are the tables
  davo_get_intermediate("att_weights:<k>") returns;
- asking for attention changes no pose, trajectory, count or later push, and adds one launch per micro-batch."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from davo_b200 import _capi, synthetic as S, version as V
from davo_b200.davo import DAVO
from davo_b200.odometry_pool import OdometryPool
from davo_b200.sequence import sequence_to_triplets
from tests.golden import make_golden as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W = 128, 416
HEADLINE = G.CASES["headline"]
SESSION_CASES = [k for k in G.CASES if not V.parse_version(G.CASES[k]).batch_norm]
NEW_SYMBOLS = ("davo_forward_sequence_features", "davo_odometry_push_attention", "davo_odometry_push_many_attention",
               "davo_odometry_push_many_host_attention")


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _system(ver, max_batch, micro_batch=0):
    sysm = DAVO(version=ver)
    sysm.setup_inference(H, W, "davo", 3, max_batch, device=0, micro_batch=micro_batch)
    sysm.load_weights(S.init_weights(ver, seed=31, random_bias=True))
    return sysm


def _stream(n, seed):
    img, fwd, bwd, seg, depth = S.make_sequence(n, H, W, seed=seed)
    seg[0, :2, :3] = 255.0                                   # a few labels without a class
    seg[-1, 5, :4] = np.nan
    seg[1, 7, 8:12] = -3.0
    return img, fwd, bwd, seg, depth


def _piece(x, a, k):
    """The push of frames [a, a+k): flow entries [a-1, a+k-1) ([0, k-1) for a first push)."""
    img, fwd, bwd, seg, depth = x
    fl = slice(max(a - 1, 0), a + k - 1)
    return img[a:a + k], fwd[fl], bwd[fl], seg[a:a + k], depth[a:a + k]


def _cuts(rng, n, first, kmax):
    ks = [first]
    while sum(ks) < n:
        ks.append(int(min(rng.integers(1, kmax + 1), n - sum(ks))))
    return ks


def _np(x):
    return x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x)


def _reference(sysm, stream):
    """Per frame of the stream: the map (features of the whole stream's triplets) and the weight rows [2,24]
    (davo_get_intermediate after one davo_forward_sequence over every pair)."""
    img, fwd, bwd, seg, depth = stream
    n = img.shape[0]
    c = sysm.config
    uses_depth = c.att_src == V.ATT_SE_DEPTH_SEG or c.depth_split
    t_img, t_flow, t_seg, t_depth = sequence_to_triplets(img, fwd, bwd, seg, depth if uses_depth else None)
    feat = sysm.inference(None, 'feature', inputs=(t_img, t_flow, t_seg, t_depth))
    att = [_np(a)[..., 0] for a in feat['masks']['attention']]          # [tgt, src0, src1] x [B,H,W]
    maps = [att[1][0], att[0][0]] + [att[2][s] for s in range(n - 2)]
    dev = [torch.as_tensor(x).cuda() for x in stream]
    sysm.inference_sequence(*dev[:4], depth=dev[4] if uses_depth else None, pairs='all', as_torch=True)
    torch.cuda.synchronize()
    slots, width = sysm._att_shape()
    unit_sample = c.posenn >= 2                              # the non-shared nets: one unit per sample

    def table(b, f):
        out = np.zeros((2, 24), np.float32)
        if c.att_src == 0 or (f == 0 and c.att_tgt_ones):
            return out                                       # a map of ones
        if unit_sample:
            unit = b
            slot = 2 * (f - 1) if c.depth_split else (2 if f == 0 else f - 1)
        else:
            unit = 2 * b + (1 if f == 2 else 0)
            slot = 1 if f == 0 else 0
        for r in range(2 if c.depth_split else 1):
            out[r, :width] = sysm.get_intermediate("att_weights:%d" % (0 if c.att_src == 2 else slot + r), unit)[:width]
        return out
    weights = [table(0, 1), table(0, 0)] + [table(s, 2) for s in range(n - 2)]
    return np.stack(maps), np.stack(weights)[:, :slots, :width]


def _push_stream(od, stream, ks, attention, host):
    """Pushes the stream cut into ks; returns the concatenated (pose, trajectory, maps, weights, frames)."""
    res, a = [], 0
    for i, k in enumerate(ks):
        p = _piece(stream, a, k)
        if not host:
            p = tuple(torch.as_tensor(x).cuda() for x in p)
        att = attention(i) if callable(attention) else attention
        res.append(od.push(*p, attention=att))
        a += k
    cat = lambda key: np.concatenate([_np(r[key]) for r in res if key in r]) if any(key in r for r in res) else None
    return cat('pose'), cat('trajectory'), cat('attention'), cat('att_weights'), [f for r in res for f in r['frames']]


# ------------------------------------------------------------------------------------------------ CPU
def test_header_declares_the_attention_entry_points(tmp_path):
    """The header compiles as C99 with the new struct and functions, and a C program links them."""
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "att.c"
    src.write_text('#include <stdio.h>\n#include "davo_b200.h"\n'
                   'int main(void) { davo_odometry_attention a = {0, 0}; (void)a;\n'
                   '  void* f[4] = {(void*)davo_forward_sequence_features, (void*)davo_odometry_push_attention,\n'
                   '                (void*)davo_odometry_push_many_attention, (void*)davo_odometry_push_many_host_attention};\n'
                   '  printf("%d\\n", (int)(sizeof a + (f[0] != 0) + (f[3] != 0))); return 0; }\n')
    lib = _capi.lib_path()
    _capi.load()
    exe = tmp_path / "att"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                    lib, "-Wl,-rpath," + os.path.dirname(lib), "-o", str(exe)], check=True, capture_output=True)
    assert subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split() == [str(2 * C.sizeof(C.c_void_p) + 2)]


def test_capi_binds_the_attention_entry_points():
    lib = _capi.load()
    for s in NEW_SYMBOLS:
        assert s in _capi.SYMBOLS and getattr(lib, s).argtypes, s
    assert C.sizeof(_capi.DavoOdometryAttentionC) == 2 * C.sizeof(C.c_void_p)


def test_python_checks_raise_before_device_work():
    d = DAVO(version=HEADLINE)
    with pytest.raises(ValueError, match="pairs='all'"):
        d.inference_sequence(None, None, None, None, pairs='trajectory', mode='feature')
    with pytest.raises(NotImplementedError, match="'pose', 'feature'"):
        d.inference_sequence(None, None, None, None, mode='features')


def test_ptxas_profile_shows_the_attention_kernel_without_spills():
    text = open(os.path.join(ROOT, "profiles", "odometry_attention_ptxas.txt")).read()
    m = re.search(r"^(\S*attention_out_kernel\S*) regs=(\d+) stack=(\d+) spill=\((\d+), (\d+)\)", text, re.M)
    assert m, text
    assert int(m.group(2)) <= 255 and m.group(4) == "0" and m.group(5) == "0"
    assert re.search(r"^\S*pack8_kernel\S* regs=56 stack=0 spill=\(0, 0\)", text, re.M)


# ------------------------------------------------------------------------------------------------ GPU
FEATURE_CASES = ["headline", "se_seg", "se_seg_wo_tgt", "static", "no_segmask", "pix_rgb", "pix_mix_depthflow",
                 "depthseg_seplayers", "decouple_net", "pix_mix_segflow_net", "se_skipadd", "batch_norm"]


@pytest.mark.gpu
@pytest.mark.parametrize("key", FEATURE_CASES)
def test_sequence_features_equal_triplet_features(key):
    """Every output of mode='feature' on a 7-frame sequence equals the triplet call on sequence_to_triplets."""
    _need_gpu()
    ver = G.CASES[key]
    sysm = _system(ver, 5)
    img, fwd, bwd, seg, depth = _stream(7, seed=5)
    uses_depth = sysm.config.att_src == V.ATT_SE_DEPTH_SEG or sysm.config.depth_split
    depth = depth if uses_depth else None
    got = sysm.inference_sequence(img, fwd, bwd, seg, depth, mode='feature')
    want = sysm.inference(None, 'feature', inputs=sequence_to_triplets(img, fwd, bwd, seg, depth))

    def walk(a, b, path):
        if isinstance(a, dict):
            assert sorted(a) == sorted(b), path
            for k in a:
                walk(a[k], b[k], path + (k,))
        elif isinstance(a, list):
            assert len(a) == len(b), path
            for i, (x, y) in enumerate(zip(a, b)):
                walk(x, y, path + (i,))
        else:
            x, y = _np(a), _np(b)
            assert x.shape == y.shape and x.dtype == y.dtype, path
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), path
    walk(got, want, ())
    dev = [torch.as_tensor(x).cuda() for x in (img, fwd, bwd, seg)]
    got_dev = sysm.inference_sequence(*dev, depth=None if depth is None else torch.as_tensor(depth).cuda(), mode='feature',
                                      as_torch=True)
    assert np.array_equal(_np(got_dev['masks']['attention'][2]), _np(want['masks']['attention'][2]))
    if key == "headline":                                     # one pass only: 2B units <= micro_batch
        small = _system(ver, 8, micro_batch=10)
        small.inference_sequence(*_stream(7, seed=6)[:4], mode='feature')        # B = 5: 10 units
        with pytest.raises(RuntimeError, match=r"n_frames=8 \(B=6 samples\) needs 12 units, one pass holds 10"):
            small.inference_sequence(*_stream(8, seed=6)[:4], mode='feature')


@pytest.mark.gpu
@pytest.mark.parametrize("key", SESSION_CASES)
def test_session_attention_equals_triplet_features(key):
    """A 40-frame stream pushed under random cuts (first pushes of 1 and 2 frames) in both pair modes, device sessions:
    the maps are the feature planes of the whole stream, the weights davo_get_intermediate's tables, and the poses,
    trajectory and frames those of the same pushes without attention."""
    _need_gpu()
    sysm = _system(G.CASES[key], 40)
    stream = _stream(40, seed=70)
    maps, weights = _reference(sysm, stream)
    rng = np.random.default_rng(3)
    for mode in ("trajectory", "all"):
        for first in (1, 2):
            ks = _cuts(rng, 40, first, 6)
            with sysm.odometry(mode, 6, host=False) as od, sysm.odometry(mode, 6, host=False) as plain:
                pose, traj, m, w, fr = _push_stream(od, stream, ks, True, False)
                pose0, traj0, _, _, fr0 = _push_stream(plain, stream, ks, False, False)
                assert np.array_equal(pose, pose0) and np.array_equal(traj, traj0) and fr == fr0, (mode, first)
                assert od.frames() == plain.frames() == (40, 40)
                assert np.array_equal(m, maps), (mode, first)
                assert np.array_equal(w, weights), (mode, first)


@pytest.mark.gpu
def test_mixed_pushes_and_launch_counts():
    """Attention on some pushes of a session gives the plain stream's bits; a push with attention launches one kernel
    more per micro-batch than the same push without (micro_batch 6: pushes of 1 to 2 passes)."""
    _need_gpu()
    sysm = _system(HEADLINE, 12, micro_batch=6)
    stream = _stream(30, seed=9)
    maps, weights = _reference(_system(HEADLINE, 28), stream)
    for mode in ("trajectory", "all"):
        ks = [2, 1, 5, 3, 6, 4, 1, 6, 2]
        od, plain = sysm.odometry(mode, 6, host=False), sysm.odometry(mode, 6, host=False)
        a = 0
        got_m, got_p, want_p = [], [], []
        for i, k in enumerate(ks):
            p = tuple(torch.as_tensor(x).cuda() for x in _piece(stream, a, k))
            want = plain.push(*p)
            n_plain = sysm.last_launch_count()
            got = od.push(*p, attention=i % 2 == 0)
            n_att = sysm.last_launch_count()
            ns = _np(want['pose']).shape[0]
            if i % 2 == 0 and ns > 0:
                units = 2 * ns if mode == "all" else ns + (1 if a == 0 else 0)
                assert n_att == n_plain + -(-units // 6), (mode, i)
                got_m.append((list(got['frames']), _np(got['attention'])))
            elif ns > 0:
                assert n_att == n_plain
            got_p.append(_np(got['trajectory']))
            want_p.append(_np(want['trajectory']))
            assert np.array_equal(_np(got['pose']), _np(want['pose'])), (mode, i)
            a += k
        assert np.array_equal(np.concatenate(got_p), np.concatenate(want_p))
        for frames, m in got_m:
            assert np.array_equal(m, maps[frames]), (mode, frames)
        od.close()
        plain.close()


def _entries(streams, pos, ks, host):
    out = []
    for i, k in enumerate(ks):
        p = _piece(streams[i], pos[i], k)
        out.append(p if host else tuple(torch.as_tensor(x).cuda() for x in p))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["headline", "depthseg_seplayers", "se_seg_wo_tgt", "decouple_net", "no_segmask"])
@pytest.mark.parametrize("host", [False, True])
def test_batched_attention_equals_single(key, host):
    """Batched pushes (device and host) with random k, sessions in mixed states and both pair modes, give each session
    the maps and weights of single pushes; micro_batch 8 makes some calls several passes (host: several chunks)."""
    _need_gpu()
    ver = G.CASES[key]
    many, one = _system(ver, 24, micro_batch=8), _system(ver, 24, micro_batch=8)
    modes = ["trajectory", "all", "trajectory", "all", "trajectory"]
    sm = [many.odometry(m, 5, host=host) for m in modes]
    so = [one.odometry(m, 5, host=host) for m in modes]
    streams = [_stream(16, seed=200 + i) for i in range(5)]
    pos = [0] * 5
    rng = np.random.default_rng(11)
    for step in range(6):
        ids = [i for i in range(5) if pos[i] < 16 and (step == 0 or rng.random() < 0.8)]
        ks = [int(min(rng.integers(1, 6), 16 - pos[i])) for i in ids]
        ins = _entries([streams[i] for i in ids], [pos[i] for i in ids], ks, host)
        args = [list(x) for x in zip(*ins)]
        if host:
            got = many.odometry_push_many_host([sm[i] for i in ids], *args, attention=True)
        else:
            got = many.odometry_push_many([sm[i] for i in ids], *args, attention=True)
        for j, i in enumerate(ids):
            want = so[i].push(*ins[j], attention=True)
            for name in ('pose', 'trajectory', 'attention', 'att_weights'):
                assert np.array_equal(_np(got[j][name]), _np(want[name])), (step, i, name)
            assert got[j]['frames'] == want['frames']
            pos[i] += ks[j]
    for od in sm + so:
        od.close()


@pytest.mark.gpu
def test_batched_launch_count_does_not_depend_on_sessions():
    _need_gpu()
    sysm = _system(HEADLINE, 40)
    counts = {}
    for n in (2, 16):
        sess = [sysm.odometry("trajectory", 3, host=False) for _ in range(n)]
        streams = [_stream(6, seed=300 + i) for i in range(n)]
        dev = lambda i, a, k: tuple(torch.as_tensor(x).cuda() for x in _piece(streams[i], a, k))
        sysm.odometry_push_many(sess, *[list(x) for x in zip(*[dev(i, 0, 3) for i in range(n)])])
        sysm.odometry_push_many(sess, *[list(x) for x in zip(*[dev(i, 3, 1) for i in range(n)])])
        plain = sysm.last_launch_count()
        sysm.odometry_push_many(sess, *[list(x) for x in zip(*[dev(i, 4, 1) for i in range(n)])], attention=True)
        counts[n] = (plain, sysm.last_launch_count())
        for od in sess:
            od.close()
    assert counts[2] == counts[16] and counts[2][1] == counts[2][0] + 1, counts


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["headline", "depthseg_seplayers", "pix_mix_segflow_net"])
def test_host_sessions_equal_device_sessions(key):
    """Host pushes, blocking and with tickets, return the device sessions' maps and weights; the device-to-host byte
    count grows by exactly the maps and weights."""
    _need_gpu()
    sysm = _system(G.CASES[key], 12, micro_batch=8)
    stream = _stream(20, seed=41)
    ks = [2, 3, 1, 6, 4, 4]
    for mode in ("trajectory", "all"):
        dev = _push_stream(sysm.odometry(mode, 6, host=False), stream, ks, True, False)
        blk = _push_stream(sysm.odometry(mode, 6, host=True), stream, ks, True, True)
        for x, y in zip(dev[:4], blk[:4]):
            assert np.array_equal(x, y), mode
        od, plain = sysm.odometry(mode, 6, host=True), sysm.odometry(mode, 6, host=True)
        pend, a = [], 0
        for k in ks:
            p = _piece(stream, a, k)
            plain.push(*p)
            d2h_plain = sysm.last_host_copy_bytes()[1]
            pend.append(od.push_async(*p, attention=True))
            n_t = len(pend[-1]._out['frames'])
            assert sysm.last_host_copy_bytes()[1] == d2h_plain + n_t * (H * W * 4 + 2 * 24 * 4)
            a += k
        res = [q.result() for q in pend]
        assert np.array_equal(np.concatenate([r['attention'] for r in res]), dev[2])
        assert np.array_equal(np.concatenate([r['att_weights'] for r in res]), dev[3])


@pytest.mark.gpu
def test_pool_push_returns_the_single_push_maps():
    _need_gpu()
    for host in (False, True):
        pool = OdometryPool([_system(HEADLINE, 16)], pairs="trajectory", max_push=4, host=host)
        ref = _system(HEADLINE, 16)
        cams = [pool.open() for _ in range(3)]
        singles = [ref.odometry("trajectory", 4, host=host) for _ in range(3)]
        streams = [_stream(9, seed=500 + i) for i in range(3)]
        for a, k in ((0, 3), (3, 4), (7, 2)):
            ins = _entries(streams, [a] * 3, [k] * 3, host)
            got = pool.push(cams, *[list(x) for x in zip(*ins)], attention=True)
            for j in range(3):
                want = singles[j].push(*ins[j], attention=True)
                assert np.array_equal(_np(got[j]['attention']), _np(want['attention']))
                assert np.array_equal(_np(got[j]['att_weights']), _np(want['att_weights']))
        pool.close_all()


@pytest.mark.gpu
def test_refusals_name_the_entry_and_change_nothing():
    _need_gpu()
    sysm = _system(HEADLINE, 8)
    lib = sysm._lib
    s = [sysm.odometry("trajectory", 4, host=False) for _ in range(2)]
    streams = [_stream(6, seed=600 + i) for i in range(2)]
    ins = [tuple(torch.as_tensor(x).cuda() for x in _piece(st, 0, 4)) for st in streams]
    n = 2
    vp = C.c_void_p
    arr = lambda vals: (vp * n)(*vals)
    ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None
    pose = [torch.zeros((2, 2, 6), device="cuda") for _ in range(n)]
    traj = [torch.zeros((4, 4, 4), dtype=torch.float64, device="cuda") for _ in range(n)]
    maps = [torch.zeros((4, H, W), device="cuda") for _ in range(n)]
    wts = [torch.zeros((4, 2, 24), device="cuda") for _ in range(n)]
    cols = [arr([ptr(x[j]) for x in ins]) for j in range(5)]

    def call(att):
        return lib.davo_odometry_push_many_attention(
            n, arr([od._o.value for od in s]), (C.c_int * n)(4, 4), *cols, arr([ptr(p) for p in pose]),
            arr([ptr(t) for t in traj]), att, None, None, None)
    A = _capi.DavoOdometryAttentionC
    bad = [((A * 2)(A(ptr(maps[0]), ptr(wts[0])), A(None, None)), r"att\[1\] has neither map nor weights"),
           ((A * 2)(A(ptr(maps[0]) + 4, ptr(wts[0])), A(ptr(maps[1]), ptr(wts[1]))), r"att\[0\]\.map is not 16-byte"),
           ((A * 2)(A(ptr(maps[0]), ptr(wts[0])), A(ptr(maps[1]), ptr(wts[1]) + 8)), r"att\[1\]\.weights is not 16-byte")]
    for att, msg in bad:
        assert call(att) != 0
        assert re.search(msg, _capi.last_error(lib, sysm._h)), _capi.last_error(lib, sysm._h)
        assert [od.frames() for od in s] == [(0, 0), (0, 0)]
        pushed = C.c_longlong(-1)
        lib.davo_odometry_frames(s[0]._o, C.byref(pushed), None)
        assert pushed.value == 0
    rc = lib.davo_odometry_push_attention(s[0]._o, 4, *[vp(ptr(x)) for x in ins[0]], vp(ptr(pose[0])), vp(ptr(traj[0])),
                                          C.byref(A(None, None)), None, None, None, None)
    assert rc != 0 and "att has neither map nor weights; 4 row(s) are due" in _capi.last_error(lib, sysm._h)
    assert call((A * 2)(A(ptr(maps[0]), None), A(None, ptr(wts[1])))) == 0        # either output alone
    torch.cuda.synchronize()
    for od in s:
        od.close()
