"""Online odometry on one GPU: per-frame latency and bulk rate of davo_odometry sessions against sequence calls.

Headline version, 128x416, a seeded frame stream (synthetic.make_sequence) in pinned host memory.

* Per-frame latency: the wall time from pushing one frame to holding its absolute pose in host memory, p50 and p99 over
  `--latency-frames` frames after a warm-up: a host session (numpy in, numpy out), a device session (the frames
  already on the GPU, the trajectory row copied to the host), and the same frames as 3-frame inference_sequence calls
  with the composition step on the host (T = pose_vec2mat, its inverse, one fp64 product).
* Bulk rate: a host session fed pushes of 1, 16 and 128 frames with two pushes in flight, alternated in the same run
  with inference_sequence_async calls of 130 frames starting every 128 frames (two in flight) on the same frames.
* Host-to-device bytes per frame for both (davo_last_host_copy_bytes).

    python tools/odometry_stream.py [--frames 1026] [--reps 3] [--latency-frames 2000] [--log profiles/odometry_stream.log]

Prints one JSON line with the card's name and power limit and appends it to the log.
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from davo_b200 import geo_utils, synthetic as S              # noqa: E402
from davo_b200.davo import DAVO                              # noqa: E402
from tests.golden.make_golden import CASES                   # noqa: E402

H, W, PER_CALL = 128, 416, 128


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:
        return "unknown (%s)" % e


def pinned(a):
    import torch
    t = torch.empty(a.shape, dtype=getattr(torch, str(a.dtype))).pin_memory()
    t.numpy()[...] = a
    return t.numpy()


def pieces(seq, cut, start=0):
    img, fwd, bwd, seg = seq
    a = start
    for k in cut:
        b = a + k
        fl = slice(max(a - 1, 0), b - 1)
        yield img[a:b], fwd[fl], bwd[fl], seg[a:b]
        a = b


def pct(ms):
    return {"p50_ms": float(np.percentile(ms, 50)), "p99_ms": float(np.percentile(ms, 99)), "frames": len(ms)}


def latency(system, seq, n_lat, warm):
    """Frame-by-frame pushes over laps of the stream; times only frames that return a pose."""
    import torch
    n = seq[0].shape[0]
    out = {}
    dev_seq = tuple(torch.as_tensor(x).cuda() for x in seq)
    for name, host in (("host_session", True), ("device_session", False)):
        ms = []
        with system.odometry(max_push=1, host=host) as od:
            src = seq if host else dev_seq
            done = 0
            while len(ms) < n_lat:
                od.reset()
                for f, p in enumerate(pieces(src, [1] * n)):
                    t0 = time.perf_counter()
                    r = od.push(*p)
                    last = r["trajectory"][-1:] if f >= 2 else None
                    if last is not None and not host:
                        last = last.cpu()
                    t1 = time.perf_counter()
                    done += 1
                    if last is not None and done > warm and len(ms) < n_lat:
                        ms.append((t1 - t0) * 1e3)
        out[name] = pct(ms)
    # the same frames as overlapping 3-frame sequence calls, composed on the host
    img, fwd, bwd, seg = seq
    ms, done = [], 0
    while len(ms) < n_lat:
        P = np.eye(4)
        for s in range(n - 2):
            t0 = time.perf_counter()
            pose = system.inference_sequence(img[s:s + 3], fwd[s:s + 2], bwd[s:s + 2], seg[s:s + 3],
                                             pairs="trajectory_first" if s == 0 else "trajectory")["pose"]
            if s == 0:
                P = P @ geo_utils.pose_vec2mat(pose[:1, 0])[0].astype(np.float64)
            P = P @ np.linalg.inv(geo_utils.pose_vec2mat(pose[:, 1]))[0].astype(np.float64)
            t1 = time.perf_counter()
            done += 1
            if done > warm and len(ms) < n_lat:
                ms.append((t1 - t0) * 1e3)
    out["sequence_calls_3_frames"] = pct(ms)
    return out


def bulk_session(system, seq, k, in_flight=2):
    """Frames per second and H2D bytes per frame of a host session fed pushes of k frames."""
    n = seq[0].shape[0]
    cut = [k] * (n // k) + ([n % k] if n % k else [])
    with system.odometry(max_push=max(k, 1)) as od:
        for p in pieces(seq, [k, k] if k > 1 else [1, 1, 1]):  # warm: staging, pinned ring, pass shapes
            od.push(*p)
        od.reset()
        pend, h2d, poses = collections.deque(), 0, []
        t0 = time.perf_counter()
        for p in pieces(seq, cut):
            pend.append(od.push_async(*p))
            h2d += system.last_host_copy_bytes()[0]
            if len(pend) == in_flight:
                poses.append(pend.popleft().result()["pose"])
        poses += [q.result()["pose"] for q in pend]
        dt = time.perf_counter() - t0
    return n / dt, h2d / n, np.concatenate(poses)


def bulk_sequence(system, seq, in_flight=2):
    img, fwd, bwd, seg = seq
    n = img.shape[0]
    starts = list(range(0, n - 2, PER_CALL))
    pend, h2d, poses = collections.deque(), 0, []
    t0 = time.perf_counter()
    for i, a in enumerate(starts):
        b = min(a + PER_CALL + 2, n)
        pend.append(system.inference_sequence_async(img[a:b], fwd[a:b - 1], bwd[a:b - 1], seg[a:b],
                                                    pairs="trajectory_first" if i == 0 else "trajectory"))
        h2d += system.last_host_copy_bytes()[0]
        if len(pend) == in_flight:
            poses.append(pend.popleft().result()["pose"])
    poses += [q.result()["pose"] for q in pend]
    dt = time.perf_counter() - t0
    return n / dt, h2d / n, np.concatenate(poses)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1026)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--latency-frames", type=int, default=2000)
    ap.add_argument("--warm", type=int, default=50)
    ap.add_argument("--log", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles",
                                                  "odometry_stream.log"))
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("odometry_stream.py measures on a GPU; there is none")
    ver = CASES["headline"]
    system = DAVO(version=ver)
    system.setup_inference(H, W, "davo", 3, PER_CALL, device=0)
    system.load_weights(S.init_weights(ver, seed=1, random_bias=True))
    img, fwd, bwd, seg, _ = S.make_sequence(a.frames, H, W, seed=21)
    seq = tuple(pinned(x) for x in (img, fwd, bwd, seg))
    res = {"workload": "host-fed online odometry, headline version, %dx%d, %d-frame seeded stream, trajectory mode"
                       % (H, W, a.frames), "gpus": 1, "card": card()}
    # bulk first (it warms every pass shape), alternating session and sequence calls rep by rep
    rates = {k: [] for k in ("push_1", "push_16", "push_128", "sequence_calls_130")}
    ref = None
    identical = True
    for _ in range(a.reps):
        for k in (1, 16, 128):
            r, b, p = bulk_session(system, seq, k)
            rates["push_%d" % k].append(r)
            res["push_%d_h2d_bytes_per_frame" % k] = b
            identical &= ref is None or np.array_equal(p, ref)
            ref = p if ref is None else ref
        r, b, p = bulk_sequence(system, seq)
        rates["sequence_calls_130"].append(r)
        res["sequence_calls_h2d_bytes_per_frame"] = b
        identical &= np.array_equal(p, ref)
    res["bulk_frames_per_s"] = {k: {"median": float(np.median(v)), "all": [float(x) for x in v]} for k, v in rates.items()}
    res["push_128_over_sequence_calls"] = (res["bulk_frames_per_s"]["push_128"]["median"]
                                           / res["bulk_frames_per_s"]["sequence_calls_130"]["median"])
    res["poses_identical"] = bool(identical)
    n_lat = a.latency_frames
    res["latency"] = latency(system, tuple(x[:min(a.frames, 514)] for x in seq), n_lat, a.warm)
    res["latency"]["note"] = "wall time from push of one frame to its absolute pose in host memory"
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.log)), exist_ok=True)
    with open(a.log, "a") as f:
        f.write(line + "\n")
    system.close()


if __name__ == "__main__":
    main()
