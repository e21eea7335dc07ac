"""What each posed frame's attention costs an odometry push (include/davo_b200.h: davo_odometry_attention).

Three cases of the headline variant at 128x416, each run as two twin session sets on one handle -- one pushing plainly,
one asking for attention -- stepped in alternation so that both see the same machine:
  single   one device session with max_push 1, one frame per push;
  device   C device cameras, one batched push (davo_odometry_push_many) of one frame each per step;
  host     a host OdometryPool of C cameras, one push of one frame each per step.
Per case and mode: frames/s over the timed steps and the p50 / p90 of a step's wall time (each step ends in a device
synchronise, or in the host push's own wait).  The GPU's name and power limit are read in the same run.

    python tools/odometry_attention.py --steps 200 --warmup 20 --out profiles/odometry_attention.log
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

VERSION = "v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh"
H, W = 128, 416


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:                                   # the record says so rather than guessing
        return "unknown (%s)" % e


def system(max_batch):
    from davo_b200 import synthetic as S
    from davo_b200.davo import DAVO
    s = DAVO(version=VERSION)
    s.setup_inference(H, W, "davo", 3, max_batch, device=0)
    s.load_weights(S.init_weights(VERSION, seed=31, random_bias=True))
    return s


def frames(n, device):
    """n frames of one synthetic stream: (img, fwd, bwd, seg) per frame index, numpy or CUDA."""
    import torch
    from davo_b200 import synthetic as S
    img, fwd, bwd, seg, _ = S.make_sequence(n + 1, H, W, seed=5)
    x = (img, fwd, bwd, seg)
    return tuple(torch.as_tensor(a).cuda() for a in x) if device else x


def piece(x, a, k):
    img, fwd, bwd, seg = x
    fl = slice(max(a - 1, 0), a + k - 1)
    return img[a:a + k], fwd[fl], bwd[fl], seg[a:a + k]


def run_case(name, cams, steps, warmup):
    """Steps both modes in alternation; returns {mode: record}."""
    import torch
    from davo_b200.odometry_pool import OdometryPool
    n = steps + warmup + 2
    host = name == "host"
    sysm = system(max(cams, 1) * (2 if name == "single" else 1))
    x = frames(n, not host)
    if name == "host":
        pools = {m: OdometryPool([sysm], "trajectory", max_push=1, host=True) for m in ("plain", "attention")}
        ids = {m: [p.open() for _ in range(cams)] for m, p in pools.items()}

        def push(m, a):
            p = piece(x, a, 1)
            return pools[m].push(ids[m], *[[t] * cams for t in p], attention=m == "attention")
    else:
        sess = {m: [sysm.odometry("trajectory", 1, host=False) for _ in range(cams)] for m in ("plain", "attention")}

        def push(m, a):
            p = piece(x, a, 1)
            if name == "single":
                r = sess[m][0].push(*p, attention=m == "attention")
            else:
                r = sysm.odometry_push_many(sess[m], *[[t] * cams for t in p], attention=m == "attention")
            torch.cuda.synchronize()
            return r
    times = {"plain": [], "attention": []}
    for a in range(n - 1):
        for m in (("plain", "attention") if a % 2 == 0 else ("attention", "plain")):
            t0 = time.perf_counter()
            push(m, a)
            if a >= warmup + 1:                             # frames 0 and 1 pose no sample; then warm-up
                times[m].append(time.perf_counter() - t0)
    out = {}
    for m, t in times.items():
        t = np.asarray(t)
        out[m] = {"case": name, "cameras": cams, "mode": m, "steps": int(t.size),
                  "frames_per_s": round(cams * t.size / t.sum(), 1),
                  "step_ms_p50": round(float(np.median(t)) * 1e3, 3), "step_ms_p90": round(float(np.quantile(t, 0.9)) * 1e3, 3)}
    out["attention"]["cost_vs_plain"] = round(out["plain"]["frames_per_s"] / out["attention"]["frames_per_s"] - 1, 4)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--device-cams", type=int, default=128)
    ap.add_argument("--host-cams", type=int, default=256)
    ap.add_argument("--out", default=None, help="append the JSON lines here as well")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("odometry_attention.py measures on a GPU; there is none here")
    gpu = gpu_info()
    lines = []
    for name, cams in (("single", 1), ("device", a.device_cams), ("host", a.host_cams)):
        for rec in run_case(name, cams, a.steps, a.warmup).values():
            rec["gpu"] = gpu
            rec["frame"] = "%dx%d" % (H, W)
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
