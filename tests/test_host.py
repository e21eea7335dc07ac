"""CPU tests of the host side: geometry, sharding, C-ABI exports, DAVO wrapper errors."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from davo_b200 import _capi, geo_utils, parallel
from davo_b200.davo import DAVO
from oracle import davo_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADLINE = "v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh"


# ------------------------------------------------------------------ geometry --
def test_pose_vec2mat_matches_oracle_and_is_rotation():
    rng = np.random.default_rng(0)
    v = rng.normal(0, 0.3, size=(50, 6)).astype(np.float32)
    v[0, :3] = [4.0, -5.0, 3.5]                      # beyond +-pi: clipped (geo_utils.py:29-31)
    m = geo_utils.pose_vec2mat(v)
    np.testing.assert_allclose(m, O.pose_vec2mat(v), atol=1e-6)
    r = m[:, :3, :3].astype(np.float64)
    np.testing.assert_allclose(r @ r.transpose(0, 2, 1), np.broadcast_to(np.eye(3), r.shape), atol=1e-5)
    np.testing.assert_allclose(m[:, :3, 3], v[:, 3:])
    c = np.cos(np.float32(np.pi))
    assert abs(m[0, 0, 0] - c * c) < 1e-6           # rz, ry clipped to pi: cos(pi)^2


def test_euler_order_is_rx_ry_rz():
    z, y, x = 0.3, -0.2, 0.5
    m = geo_utils.euler2mat([z], [y], [x])[0].astype(np.float64)
    rz = np.array([[np.cos(z), -np.sin(z), 0], [np.sin(z), np.cos(z), 0], [0, 0, 1]])
    ry = np.array([[np.cos(y), 0, np.sin(y)], [0, 1, 0], [-np.sin(y), 0, np.cos(y)]])
    rx = np.array([[1, 0, 0], [0, np.cos(x), -np.sin(x)], [0, np.sin(x), np.cos(x)]])
    np.testing.assert_allclose(m, rx @ ry @ rz, atol=1e-6)


def test_compose_trajectory_matches_reference_loop():
    rng = np.random.default_rng(1)
    poses = rng.normal(0, 0.05, size=(40, 2, 6)).astype(np.float32)
    traj = geo_utils.compose_trajectory(poses)
    ref = O.compose_trajectory(poses)
    assert traj.shape == (42, 4, 4)
    np.testing.assert_allclose(traj, ref, atol=1e-9)
    np.testing.assert_array_equal(traj[0], np.eye(4))
    # the second pose is T(tgt->src0) of the first sample; then inverses of tgt->src1
    np.testing.assert_allclose(traj[1], geo_utils.pose_vec2mat(poses[:1, 0])[0], atol=1e-7)
    np.testing.assert_allclose(traj[2], traj[1] @ np.linalg.inv(geo_utils.pose_vec2mat(poses[:1, 1])[0]), atol=1e-7)


def test_kitti_text_format(tmp_path):
    poses = np.zeros((3, 2, 6), np.float32)
    poses[:, :, 5] = 1.0
    traj = geo_utils.compose_trajectory(poses)
    p = tmp_path / "09-pred_kitti_pose.txt"
    geo_utils.write_kitti_trajectory(str(p), traj)
    lines = p.read_text().strip().split("\n")
    assert len(lines) == 5 and all(len(l.split()) == 12 for l in lines)
    assert lines == O.kitti_lines(traj)
    assert lines[0].split()[0] == "1.0"              # str(float) formatting


def _mat2euler(r):
    """Inverse of euler2mat for R = Rx Ry Rz (reference utils/geo_utils.py:66-91, branch f1)."""
    cy = np.sqrt(r[2, 2] ** 2 + r[1, 2] ** 2)
    return np.arctan2(-r[0, 1], r[0, 0]), np.arctan2(r[0, 2], cy), np.arctan2(-r[1, 2], r[2, 2])


def _gt_trajectory(turn=0.0):
    """300 frames of seeded random motion, translation steps up to about a metre.  turn = 0: small rotation steps;
    turn > 0: a steady yaw of `turn` rad per frame and larger rotation noise, so that the heading sweeps several full
    turns (every yaw in -pi..pi) and the steps' Euler angles reach a few tenths of a radian."""
    rng = np.random.default_rng(2)
    std = [0.005, 0.02, 0.005, 0.03, 0.02, 0.8] if turn == 0.0 else [0.03, 0.1, 0.03, 0.03, 0.02, 0.8]
    gt = [np.eye(4)]
    for _ in range(299):
        step = geo_utils.pose_vec2mat(rng.normal([0.0, turn, 0.0, 0.0, 0.0, 0.0], std, size=(1, 6)))[0]
        gt.append(gt[-1] @ step.astype(np.float64))
    return np.stack(gt)


def test_ground_truth_round_trip_through_pose_vectors():
    """encode GT steps as the network's [rz,ry,rx,t] vectors -> compose -> the GT trajectory again, for gentle motion
    and for a trajectory that turns through every heading."""
    for turn in (0.0, 0.05):
        gt = _gt_trajectory(turn)
        n = gt.shape[0] - 2                           # samples for a stream of n+2 frames
        poses = np.zeros((n, 2, 6), np.float32)
        for s in range(n):
            # pose[s,1] is tgt->src1 with tgt = frame s+1: inv(step s+1 -> s+2) (test_kitti_pose.py:145)
            t_fwd = np.linalg.inv(gt[s + 1]) @ gt[s + 2]
            m = np.linalg.inv(t_fwd)
            poses[s, 1, :3] = _mat2euler(m[:3, :3])
            poses[s, 1, 3:] = m[:3, 3]
        first = np.linalg.inv(gt[0]) @ gt[1]          # pose[0,0] = tgt->src0 of the first sample
        poses[0, 0, :3] = _mat2euler(first[:3, :3])
        poses[0, 0, 3:] = first[:3, 3]
        traj = geo_utils.compose_trajectory(poses)
        assert traj.shape == gt.shape
        assert O.ate(traj, gt) < 2e-3 * max(1.0, np.abs(gt[:, :3, 3]).max() / 100), turn


# ------------------------------------------------------------------ sharding --
def test_complete_batch_size_and_valid_sample():
    assert parallel.complete_batch_size([1, 2, 3], 2) == [1, 2, 3, 3]
    assert parallel.complete_batch_size([1, 2, 3, 4], 2) == [1, 2, 3, 4]
    frames = ["09 %06d" % i for i in range(5)] + ["10 000000"]
    assert [parallel.is_valid_sample(frames, i, 3) for i in range(6)] == [False, True, True, True, False, False]


@pytest.mark.parametrize("n,world", [(4539, 8), (4539, 2), (7, 4), (3, 4), (16, 4)])
def test_shard_ranges_cover_stream_in_order(n, world):
    seen = []
    for r in range(world):
        idx = parallel.padded_indices(n, r, world)
        assert len(idx) == -(-n // world)
        seen.extend(idx)
    assert seen[:n] == list(range(n))
    assert all(i == n - 1 for i in seen[n:])


def test_gloo_world2_gather_matches_single_process():
    """world_size 2, gloo: the N>1 host path (shard -> local 'forward' -> all-gather -> trim)."""
    script = r'''
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %r)
from davo_b200 import parallel
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
n = 11
full = torch.arange(n * 12, dtype=torch.float32).reshape(n, 2, 6)     # stand-in for per-sample poses
idx = parallel.padded_indices(n, rank, world)
local = full[idx] * 2 + 1                                               # the per-rank 'forward'
out = parallel.gather_poses(local, n)
assert out.shape == (n, 2, 6) and torch.equal(out, full * 2 + 1), (rank, out)
dist.destroy_process_group()
print("OK", rank)
''' % ROOT
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29571", "--no-python",
                          sys.executable, "-c", script],
                         capture_output=True, text=True, env=env, timeout=240)
    assert res.returncode == 0, res.stdout + res.stderr
    assert res.stdout.count("OK") == 2


# ------------------------------------------------------------------- C ABI ----
def _declared_functions():
    hdr = open(os.path.join(ROOT, "include", "davo_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(davo_[a-z_0-9]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    lib = _capi.load()                                # builds with nvcc if stale (no GPU needed)
    names = _declared_functions()
    assert "davo_forward" in names and "davo_create" in names and len(names) >= 12
    for n in names:
        assert hasattr(lib, n), n
    assert set(names) == set(_capi.SYMBOLS)
    assert b"sm_100a" in lib.davo_build_info()


def test_library_contains_tcgen05_and_tma_sass():
    sass = subprocess.run(["cuobjdump", "-sass", _capi.lib_path()], capture_output=True, text=True).stdout
    if not sass:
        pytest.skip("cuobjdump not available")
    assert "UTCHMMA" in sass or "UTCMMA" in sass      # tcgen05.mma
    assert "UTMALDG" in sass                          # TMA tensor loads
    assert "LDTM" in sass                             # tcgen05.ld


def test_create_without_gpu_fails_loudly_not_silently():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _capi.load()
    cfg = _capi.DavoConfigC(H=128, W=416, max_batch=1, posenn=0, cnv6_out=128, in_mode=1, att_src=1,
                            att_tgt_ones=1, mask_mode=2, se_act=1, flow_abs=1)
    h = ctypes.c_void_p()
    rc = lib.davo_create(ctypes.byref(cfg), 0, ctypes.byref(h))
    assert rc != 0 and not h.value
    assert b"no CPU fallback" in lib.davo_last_error(None)
    sysm = DAVO(version=HEADLINE)
    with pytest.raises(RuntimeError, match="davo_create failed"):
        sysm.setup_inference(128, 416, "davo", 3, 1)


def test_create_rejects_bad_config_before_touching_cuda():
    lib = _capi.load()
    h = ctypes.c_void_p()
    cfg = _capi.DavoConfigC(H=100, W=416, max_batch=1, cnv6_out=128, in_mode=1)
    assert lib.davo_create(ctypes.byref(cfg), 0, ctypes.byref(h)) == -1
    assert b"multiples of 8" in lib.davo_last_error(None)
    cfg = _capi.DavoConfigC(H=128, W=416, max_batch=1, cnv6_out=128, in_mode=1, posenn=6)     # no such PoseNN
    assert lib.davo_create(ctypes.byref(cfg), 0, ctypes.byref(h)) == -1


def test_wrapper_raises_like_the_reference():
    with pytest.raises(NameError, match="unknown PoseNN type."):
        DAVO(version="v1-sharedNN").setup_inference(128, 416, "davo", 3, 1)
    with pytest.raises(AssertionError):
        DAVO().setup_inference(128, 416, "davo", 3, 1)
    # any other mode builds nothing, as in the reference (davo.py:1548)
    DAVO(version=HEADLINE).setup_inference(128, 416, "other", 3, 1)


def test_product_package_does_not_import_oracle():
    pkg = os.path.join(ROOT, "davo_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def _write_dump(root, seq, n_frames, h, w, seed=3):
    """A dump in the reference's layout (doc/preprocessing.md:50-113, test_kitti_pose.py:45-49):
    <root>/<seq>/<id>.jpg (src0|tgt|src1 side by side), <id>-flownet2.npy (4,H,W,2),
    <id>-seglabel.npy (3,H,W,1), one triple per valid target frame."""
    from PIL import Image
    d = os.path.join(root, "%.2d" % seq)
    os.makedirs(d)
    rng = np.random.default_rng(seed)
    out = []
    for t in range(1, n_frames - 1):
        fid = "%.6d" % t
        img = rng.integers(0, 256, size=(h, 3 * w, 3), dtype=np.uint8)
        Image.fromarray(img).save(os.path.join(d, fid + ".jpg"), quality=95)
        flow = rng.normal(0.3, 15.0, size=(4, h, w, 2)).astype(np.float32)
        seg = rng.integers(0, 19, size=(3, h, w, 1)).astype(np.uint8)
        np.save(os.path.join(d, fid + "-flownet2.npy"), flow)
        np.save(os.path.join(d, fid + "-seglabel.npy"), seg)
        np.save(os.path.join(d, fid + "-monodepth2_depth.npy"), rng.uniform(1.0, 80.0, size=(3, h, w, 1)).astype(np.float32))
        out.append((flow, seg))
    return out


def test_dump_stream_reads_the_reference_layout(tmp_path):
    from PIL import Image
    from davo_b200.test_kitti_pose import DumpStream
    h, w, n = 16, 32, 6
    ref = _write_dump(str(tmp_path), 9, n, h, w)
    stream = DumpStream(str(tmp_path), 9, h, w, 3)
    assert stream.n == n - 2 and stream.ids[0] == "000001" and stream.ids[-1] == "%.6d" % (n - 2)
    for i in range(stream.n):
        img, flow, seg = stream.sample(i)
        assert img.shape == (h, 3 * w, 3) and img.dtype == np.uint8
        assert flow.shape == (4, h, w, 2) and flow.dtype == np.float32
        assert seg.shape == (3, h, w, 1) and seg.dtype == np.float32
        assert np.array_equal(flow, ref[i][0]) and np.array_equal(seg, ref[i][1].astype(np.float32))
        assert np.array_equal(img, np.asarray(Image.open(str(tmp_path / "09" / (stream.ids[i] + ".jpg"))).convert("RGB")))


# ---- TensorFlow checkpoint (tensor bundle) reader ----
def _pb_varint(v):
    out = bytearray()
    v &= (1 << 64) - 1
    while True:
        b = v & 0x7F
        v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _pb(field, wt, payload):
    return _pb_varint((field << 3) | wt) + payload


def _write_bundle(prefix, tensors, extra_entries=(), block_bytes=300):
    """A writer of the tensor-bundle format independent of the reader: LevelDB-style table with
    prefix-compressed keys, restart points every 4 entries, several data blocks, masked crc32c."""
    import struct
    from davo_b200 import tf_checkpoint as T
    data = bytearray()
    entries = {b"": _pb(1, 0, _pb_varint(1)) + _pb(3, 2, _pb_varint(2) + _pb(1, 0, _pb_varint(1)))}   # header
    for name in sorted(tensors):
        a = np.require(np.asarray(tensors[name]), requirements="C")      # (ascontiguousarray would make a scalar 1-d)
        raw = a.astype("<f4").tobytes() if a.dtype != np.int64 else a.astype("<i8").tobytes()
        shape = b"".join(_pb(2, 2, _pb_varint(len(_pb(1, 0, _pb_varint(d)))) + _pb(1, 0, _pb_varint(d))) for d in a.shape)
        e = _pb(1, 0, _pb_varint(1 if a.dtype != np.int64 else 9)) + _pb(2, 2, _pb_varint(len(shape)) + shape)
        e += _pb(4, 0, _pb_varint(len(data))) + _pb(5, 0, _pb_varint(len(raw))) + _pb(6, 5, struct.pack("<I", T.masked_crc32c(raw)))
        entries[name.encode()] = e
        data += raw
    for k, v in extra_entries:
        entries[k] = v
    with open(prefix + ".data-00000-of-00001", "wb") as f:
        f.write(bytes(data))

    def build_block(kvs, interval=4):
        out, restarts, prev = bytearray(), [], b""
        for i, (k, v) in enumerate(kvs):
            shared = 0
            if i % interval == 0:
                restarts.append(len(out))
            else:
                while shared < min(len(prev), len(k)) and prev[shared] == k[shared]:
                    shared += 1
            out += _pb_varint(shared) + _pb_varint(len(k) - shared) + _pb_varint(len(v)) + k[shared:] + v
            prev = k
        for r in restarts or [0]:
            out += struct.pack("<I", r)
        out += struct.pack("<I", len(restarts) or 1)
        return bytes(out)

    table, handles = bytearray(), []

    def emit(block):
        off = len(table)
        table.extend(block + b"\x00" + struct.pack("<I", T.masked_crc32c(block + b"\x00")))
        return _pb_varint(off) + _pb_varint(len(block))

    cur, size = [], 0
    for k in sorted(entries):
        cur.append((k, entries[k]))
        size += len(k) + len(entries[k])
        if size >= block_bytes:
            handles.append((cur[-1][0], emit(build_block(cur))))
            cur, size = [], 0
    if cur:
        handles.append((cur[-1][0], emit(build_block(cur))))
    meta = emit(build_block([]))
    index = emit(build_block(handles, interval=1))
    footer = meta + index
    footer += b"\x00" * (40 - len(footer)) + struct.pack("<Q", T.TABLE_MAGIC)
    with open(prefix + ".index", "wb") as f:
        f.write(bytes(table) + footer)


def test_tf_checkpoint_reader_round_trip(tmp_path):
    """tf_checkpoint.read_checkpoint on a bundle written by an independent writer of the same format:
    all pose variables come back bit for bit, optimizer slots / non-float variables are skipped,
    crc32c is checked, damage is reported."""
    from davo_b200 import tf_checkpoint as T
    from davo_b200 import synthetic as S
    assert T.crc32c(b"123456789") == 0xE3069283                      # the Castagnoli check value
    # a variant with a SCALAR variable (se_flow/depth_threshold, rank 0) next to the conv and dense ones
    w = S.init_weights("v1-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow_on_depthseg_seplayers_15-abs_flow-fc_tanh",
                       random_bias=True)
    assert np.asarray(w["pose_exp_net/se_flow/depth_threshold"]).shape == ()
    extra = {"global_step": np.array([1600000], np.int64),
             "pose_exp_net/cnv1/weights/Adam": np.zeros((7, 7, 10, 16), np.float32),
             "depth_net/cnv1/weights": np.ones((3, 3, 3, 8), np.float32)}
    prefix = str(tmp_path / "model-1600000")
    _write_bundle(prefix, {**w, **extra})
    assert T.is_checkpoint_prefix(prefix) and not T.is_checkpoint_prefix(str(tmp_path / "nothing"))
    header, entries = T.read_index(prefix + ".index")
    assert header["num_shards"] == 1 and set(entries) == set(w) | set(extra)
    got = T.read_checkpoint(prefix, T.pose_variables, verify_data_crc=True)
    assert set(got) == set(w)
    for k in w:
        assert got[k].dtype == np.float32 and got[k].shape == np.shape(w[k]) and np.array_equal(got[k], w[k])
    assert "depth_net/cnv1/weights" in T.read_checkpoint(prefix) and "global_step" not in T.read_checkpoint(prefix)
    # damage: a flipped byte in the index fails the block crc; a flipped tensor byte fails the data crc
    raw = bytearray(open(prefix + ".index", "rb").read())
    raw[10] ^= 0xFF
    open(str(tmp_path / "bad.index"), "wb").write(bytes(raw))
    with pytest.raises(ValueError, match="crc32c"):
        T.read_index(str(tmp_path / "bad.index"))
    d = bytearray(open(prefix + ".data-00000-of-00001", "rb").read())
    d[entries["pose_exp_net/cnv1/biases"]["offset"] + 5] ^= 0x01
    open(prefix + ".data-00000-of-00001", "wb").write(bytes(d))
    with pytest.raises(ValueError, match="crc32c"):
        T.read_checkpoint(prefix, T.pose_variables, verify_data_crc=True)
    with pytest.raises(ValueError, match="magic"):
        open(str(tmp_path / "junk.index"), "wb").write(b"x" * 100)
        T.read_index(str(tmp_path / "junk.index"))


def test_comm_unique_id_binds_nccl_at_run_time():
    """davo_comm_unique_id (include/davo_b200.h): NCCL is dlopen'ed, ids are 128 bytes and differ per call."""
    import ctypes as C
    from davo_b200 import _capi
    lib = _capi.load()
    a, b = (C.c_ubyte * 128)(), (C.c_ubyte * 128)()
    assert lib.davo_comm_unique_id(a) == 0, lib.davo_last_error(None)
    assert lib.davo_comm_unique_id(b) == 0
    assert bytes(a) != bytes(b) and any(bytes(a))
    assert lib.davo_comm_unique_id(None) != 0 and b"null argument" in lib.davo_last_error(None)


def test_host_flow_conversion_is_ieee_binary16_round_to_nearest_even():
    """davo_debug_flows_to_half (the CPU side of the host entry point, csrc/host_convert.cpp): both the
    F16C and the scalar path equal numpy's float16 cast bit for bit, subnormals and ties included, and
    report values that have no finite half."""
    import ctypes as C
    from davo_b200 import _capi
    lib = _capi.load()
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.normal(0.32, 15.38, 100003), rng.normal(0, 1e-5, 5000), rng.normal(0, 1e-7, 5000),
                        [0.0, -0.0, 65504, 65519.9, -65519.9, 6.1e-5, 5.96e-8, 2.98e-8, 2.9802322e-08, 8.9e-8, 1e-30,
                         2048.5, 2049.5, 1.00048828125, 1.00146484375]]).astype(np.float32)
    want = x.astype(np.float16).view(np.uint16)
    for portable in (0, 1):
        out = np.zeros(x.size, np.uint16)
        assert lib.davo_debug_flows_to_half(x.ctypes.data, out.ctypes.data, x.size, portable) == 0
        assert np.array_equal(out, want)
        for poison in (65520.0, -1e9, np.nan, np.inf):
            bad = x.copy()
            bad[777] = poison
            assert lib.davo_debug_flows_to_half(bad.ctypes.data, out.ctypes.data, bad.size, portable) == 1


def test_host_label_conversion_truncates_and_marks_invalid_labels():
    """davo_debug_labels_to_bytes (csrc/host_convert.cpp): the vector and the scalar path agree with
    tf.cast(label, int32) followed by one_hot(depth=19)'s treatment of out-of-range indices, at every tail length."""
    from davo_b200 import _capi
    lib = _capi.load()
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.integers(0, 19, 4099).astype(np.float32), rng.uniform(-3, 22, 4000).astype(np.float32),
                        np.float32([-0.0, -0.5, -0.999, -1.0, 18.0, 18.999, 19.0, 255.0, 256.0, 1e9, -1e9, 3e38, -3e38,
                                    np.inf, -np.inf, np.nan])])
    with np.errstate(invalid="ignore"):
        t = np.trunc(x)
    want = np.where(np.isnan(x), 255, np.where((t >= 0) & (t <= 18), t, 255)).astype(np.uint8)      # NaN: no class (tf.cast -> INT_MIN on the CPU)
    for portable in (0, 1):
        for n in (x.size, 31, 32, 33, 47, 48, 15, 1, 0):
            src = np.ascontiguousarray(x[x.size - n:])
            out = np.full(n + 8, 0xAB, np.uint8)
            assert lib.davo_debug_labels_to_bytes(src.ctypes.data, out.ctypes.data, n, portable) == 0
            assert np.array_equal(out[:n], want[x.size - n:]) and np.all(out[n:] == 0xAB)


def test_binding_struct_matches_the_header():
    """The ctypes davo_config has the header's fields in the header's order, and the library's size."""
    import ctypes as C, re
    from davo_b200 import _capi
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "davo_b200.h")).read()
    body = hdr[hdr.index("typedef struct davo_config {"):hdr.index("} davo_config;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"int32_t\s+([a-z_0-9, A-Z]+);", body)
    names = [n.strip() for f in fields for n in f.split(",")]
    assert names == [n for n, _ in _capi.DavoConfigC._fields_]
    assert _capi.load().davo_config_bytes() == C.sizeof(_capi.DavoConfigC) == 4 * len(names)


def test_header_is_plain_c_and_links_against_the_library(tmp_path):
    """include/davo_b200.h compiles as C99 (the boundary is a C ABI, not a C++ one) and a C program that
    links the shared library sees the config size the Python binding sees."""
    import shutil, subprocess, ctypes as C
    from davo_b200 import _capi
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "host.c"
    src.write_text('#include <stdio.h>\n#include "davo_b200.h"\n'
                   'int main(void) { davo_config c; davo_features f; (void)c; (void)f;\n'
                   '  printf("%d %d %s\\n", davo_config_bytes(), (int)sizeof(davo_config), davo_build_info()); return 0; }\n')
    exe = tmp_path / "host"
    lib = _capi.lib_path()
    _capi.load()
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(root, "include"),
                    str(src), lib, "-Wl,-rpath," + os.path.dirname(lib), "-o", str(exe)], check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert int(out[0]) == int(out[1]) == C.sizeof(_capi.DavoConfigC)


def test_cli_depth_source_mirrors_the_reference_cli(tmp_path):
    """Which file feeds input_depth: reference test_kitti_pose.py:91 reads the depth file only when "depth" is in the
    version, while the graph reads input_depth for "depth" OR "disp" (davo.py:960): a disp-only version gets the
    SEGLABEL file as its depth (:59-62).  DumpStream / SyntheticStream return the 4-tuple DAVO.inference needs."""
    from davo_b200 import test_kitti_pose as cli
    assert cli.depth_source("v1-sharedNN-dilatedPoseNN-segmask_all-se_depth_wo_tgt_to_seg") == "depth"
    assert cli.depth_source("v1-sharedNN-dilatedPoseNN-segmask_all-se_disp_to_seg-norm_depth") == "depth"
    assert cli.depth_source("v1-sharedNN-dilatedPoseNN-segmask_all-se_disp_to_seg") == "seglabel"
    assert cli.depth_source("v1-sharedNN-dilatedPoseNN-segmask_all-se_flow") == "none"
    _write_dump(str(tmp_path / "dump"), 9, 5, 16, 24)
    d = os.path.join(str(tmp_path / "dump"), "09")
    s3 = cli.DumpStream(str(tmp_path / "dump"), 9, 16, 24, 3).sample(0)
    s4 = cli.DumpStream(str(tmp_path / "dump"), 9, 16, 24, 3, "depth").sample(1)
    sl = cli.DumpStream(str(tmp_path / "dump"), 9, 16, 24, 3, "seglabel").sample(1)
    assert len(s3) == 3 and len(s4) == 4 and s4[3].shape == (3, 16, 24, 1) and s4[3].dtype == np.float32
    assert np.array_equal(s4[3], np.load(os.path.join(d, "000002-monodepth2_depth.npy")))
    assert np.array_equal(sl[3], sl[2])
    syn = cli.SyntheticStream(10, 16, 24, 5, "depth").sample(3)
    assert len(syn) == 4 and syn[3].shape == (3, 16, 24, 1) and syn[3].min() >= 1.0
    assert len(cli.SyntheticStream(10, 16, 24, 5).sample(3)) == 3


def test_data_loader_mirrors_load_test_batch_flow(tmp_path):
    """davo_b200/data_loader.py: the reference's file lists (test_kitti_pose.py:32-72) and its batch iterator
    (data_loader.py:241-325): tuple order image, pose, flow, depth, seglabel; batches in list order, the last one
    partial; contents equal the files; worker threads and prefetch do not reorder anything."""
    from PIL import Image
    from davo_b200.data_loader import DataLoader, load_kitti_image_sequence_names
    h, w = 16, 24
    _write_dump(str(tmp_path / "dump"), 9, 9, h, w)                       # 9 frames -> 7 samples
    frames = ["%.2d %.6d" % (9, n) for n in range(9)]
    names, tgt, poses, flows, depths, segs = load_kitti_image_sequence_names(str(tmp_path / "dump"), frames, 3, load_pose=True,
                                                                          load_flow=True, load_depth=False, load_seglabel=True)
    assert tgt == list(range(1, 8)) and names[0].endswith("09/000001.jpg") and flows[6].endswith("000007-flownet2.npy")
    assert depths == segs                                                  # load_depth False: the seglabel files (:59-62)
    assert load_kitti_image_sequence_names(str(tmp_path / "dump"), frames, 3, load_depth=True)[4][0].endswith("-monodepth2_depth.npy")
    loader = DataLoader(str(tmp_path / "dump"), 3, h, w, 2, read_flow=True, read_depth=True, read_seglabel=True)
    it = loader.load_test_batch_flow(names, poses, flows, depths, segs, workers=3, prefetch=2)
    assert len(it) == 3
    seen = 0
    for img, pose, flow, depth, seg in it:
        n = img.shape[0]
        assert pose is None and img.dtype == np.uint8 and flow.shape == (n, 4, h, w, 2) and seg.shape == (n, 3, h, w, 1)
        for k in range(n):
            assert np.array_equal(img[k], np.asarray(Image.open(names[seen + k]).convert("RGB")))
            assert np.array_equal(flow[k], np.load(flows[seen + k]))
            assert np.array_equal(seg[k][..., 0], np.load(segs[seen + k])[..., 0].astype(np.float32))
            assert np.array_equal(depth[k], seg[k])                        # the depth list IS the seglabel list here
        seen += n
    assert seen == 7
    # hold=3: a batch's arrays stay untouched while two later batches are fetched (a consumer with two asynchronous
    # inferences in flight); with hold=1 they may be refilled as soon as the next batch is asked for
    one = DataLoader(str(tmp_path / "dump"), 1, h, w, 2, read_flow=True, read_seglabel=True)
    it = one.load_test_batch_flow(names, poses, flows, depths, segs, workers=2, prefetch=1, hold=3)
    first = it.get_next()
    snap = first[2].copy()
    for _ in range(2):
        it.get_next()
    assert np.array_equal(first[2], snap) and np.array_equal(snap[0], np.load(flows[0]))
    it.close()
    bad = loader.load_test_batch_flow(names[:2] + [str(tmp_path / "missing.jpg")], poses[:3], flows[:3], depths[:3], segs[:3])
    with pytest.raises(FileNotFoundError):
        list(bad)
    with pytest.raises(ValueError):
        loader.load_test_batch_flow(names, poses, flows, depths, segs, decode="nvjpeg")      # needs a DAVO handle


def test_bench_reference_arm_prints_one_contract_line_also_when_started_plainly_with_gpus_2(tmp_path):
    """`python bench.py --impl reference --gpus 2` (no torchrun around it): bench.py becomes the 2-rank launch itself
    (127.0.0.1 rendezvous), rank 0 alone times the CPU port and prints ONE JSON line with the contract's keys; the other
    rank exits 0 without work.  --dump-outputs writes the poses of the last timed step, the same ones on every run."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if k not in ("WORLD_SIZE", "RANK", "LOCAL_RANK")}
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
                        "--dump-outputs", str(tmp_path / "a")], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["steps"] == 1 and d["warmup"] == 1
    for key in ("metric", "value", "unit", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["value"] > 0
    assert sorted(os.listdir(tmp_path / "a")) == ["pose.npy"]
    pose = np.load(tmp_path / "a" / "pose.npy")
    assert pose.shape == (16, 2, 6) and pose.dtype == np.float64 and np.all(np.isfinite(pose))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--dump-outputs", str(tmp_path / "b")], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert np.array_equal(np.load(tmp_path / "b" / "pose.npy"), pose)
