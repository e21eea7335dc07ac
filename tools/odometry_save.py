"""Saving and loading odometry sessions: davo_odometry_save_many / load_many against S single saves and loads.

S sessions (headline version, 128x416, trajectory mode, max_push 2), each three frames into its stream so that it
carries two frames with their labels and a pose, as host sessions and as device sessions, S in {1, 16, 128, 1024}.
The C ABI is called directly on page-locked buffers, so that the numbers are the library's and not the wrapper's.
For each (kind, S) it records:
  - the time of one save_many and of one load_many of all S sessions, and of S davo_odometry_save / davo_odometry_load
    calls one after the other (host clock around the synchronous calls; median of --rounds);
  - bytes per session;
  - the blobs' bytes per second against the pinned copy rate measured in the same run at the same size
    (device to host for a save, host to device for a load);
  - that save_many wrote the bytes of the single saves, and that one more push on every loaded session gives the bits
    of the same push on the original.
It prints the name and power limit of the card, read in the same run.  Writes profiles/odometry_save.log unless --out
says otherwise.

    python tools/odometry_save.py [--sizes 1,16,128,1024] [--rounds 5] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np      # noqa: E402
import torch            # noqa: E402

from davo_b200 import _capi, synthetic as S     # noqa: E402
from davo_b200.davo import DAVO, Odometry       # noqa: E402
from tests.golden import make_golden as G       # noqa: E402

H, W = 128, 416


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if q.returncode == 0 and q.stdout.strip():
        return q.stdout.strip().splitlines()
    return [torch.cuda.get_device_name(d) for d in range(torch.cuda.device_count())]


def copy_rate(nbytes, d2h, rounds):
    """Bytes per second of one pinned copy of nbytes (median of rounds)."""
    dev = torch.empty((nbytes,), dtype=torch.uint8, device="cuda:0")
    host = torch.empty((nbytes,), dtype=torch.uint8).pin_memory()
    ts = []
    for _ in range(rounds + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        (host.copy_(dev, non_blocking=True) if d2h else dev.copy_(host, non_blocking=True))
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return nbytes / float(np.median(ts[1:]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,16,128,1024")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "odometry_save.log"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("odometry_save.py measures on the GPU; there is none here")
    sizes = [int(s) for s in a.sizes.split(",")]
    ver = G.CASES["headline"]
    sysm = DAVO(version=ver)
    sysm.setup_inference(H, W, "davo", 3, max(sizes), device=0)
    sysm.load_weights(S.init_weights(ver, seed=31, random_bias=True))
    lib, h = sysm._lib, sysm._h
    img, fwd, bwd, seg, _ = S.make_sequence(8, H, W, seed=21)
    vp = C.c_void_p
    result = {"workload": "S odometry sessions of the headline version, %dx%d, trajectory mode, max_push 2, three frames "
                          "into their streams; one handle on cuda:0" % (H, W),
              "cards": cards(), "rounds": a.rounds, "runs": {}}

    def check(rc):
        assert rc == 0, _capi.last_error(lib, h)

    for host in (True, False):
        name = "host" if host else "device"
        for n in sizes:
            sess = [sysm.odometry("trajectory", 2, host=host) for _ in range(n)]
            feed = (lambda x: x) if host else (lambda x: torch.as_tensor(np.ascontiguousarray(x)).cuda())
            first = tuple(feed(x) for x in (img[0:2], fwd[0:1], bwd[0:1], seg[0:2]))
            nxt = tuple(feed(x) for x in (img[2:3], fwd[1:2], bwd[1:2], seg[2:3]))
            push = sysm.odometry_push_many_host if host else sysm.odometry_push_many
            push(sess, *[[x] * n for x in first])
            push(sess, *[[x] * n for x in nxt])
            torch.cuda.synchronize()
            ptrs = (vp * n)(*[od._o.value for od in sess])
            size = C.c_int64(0)
            sizes_b = []
            for od in sess:
                check(lib.davo_odometry_state_bytes(od._o, C.byref(size)))
                sizes_b.append(size.value)
            total = sum(sizes_b)
            buf = torch.empty((total,), dtype=torch.uint8).pin_memory().numpy()
            one = torch.empty((max(sizes_b),), dtype=torch.uint8).pin_memory().numpy()
            offs = (C.c_int64 * (n + 1))()
            out = (vp * n)()
            t_save, t_load, t_save1, t_load1 = [], [], [], []
            for r in range(a.rounds + 1):                    # round 0 warms (staging, descriptor areas)
                t0 = time.perf_counter()
                check(lib.davo_odometry_save_many(n, ptrs, vp(buf.ctypes.data), total, offs))
                t1 = time.perf_counter()
                check(lib.davo_odometry_load_many(h, n, vp(buf.ctypes.data), offs, out))
                t2 = time.perf_counter()
                loaded = [out[i] for i in range(n)]
                for p in loaded[:-1] if r == a.rounds else loaded:
                    lib.davo_odometry_destroy(vp(p))
                t3 = time.perf_counter()
                for od in sess:
                    check(lib.davo_odometry_save(od._o, vp(one.ctypes.data), one.size, C.byref(size)))
                t4 = time.perf_counter()
                singles = []
                for i in range(n):
                    o = vp()
                    check(lib.davo_odometry_load(h, vp(buf.ctypes.data + offs[i]), offs[i + 1] - offs[i], C.byref(o)))
                    singles.append(o.value)
                t5 = time.perf_counter()
                for p in singles:
                    lib.davo_odometry_destroy(vp(p))
                if r:
                    t_save.append(t1 - t0)
                    t_load.append(t2 - t1)
                    t_save1.append(t4 - t3)
                    t_load1.append(t5 - t4)
            singles_same = all(bytes(od.save()) == bytes(buf[offs[i]:offs[i + 1]]) for i, od in enumerate(sess[:64]))
            # one more push on the last loaded session and on its original: the same bits
            hdr = {"host": host, "max_push": 2, "pairs": "trajectory"}
            copy = Odometry._adopt(sysm, vp(loaded[-1]), hdr)
            third = tuple(feed(x) for x in (img[3:4], fwd[2:3], bwd[2:3], seg[3:4]))
            pa, pb = sess[-1].push(*third), copy.push(*third)
            f = lambda x: x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
            identical = bool(np.array_equal(f(pa["pose"]), f(pb["pose"])) and
                             np.array_equal(f(pa["trajectory"]), f(pb["trajectory"])))
            d2h, h2d = copy_rate(total, True, a.rounds), copy_rate(total, False, a.rounds)
            med = lambda v: float(np.median(v))
            row = {"kind": name, "S": n, "bytes_per_session": total / n, "total_bytes": total,
                   "save_many_ms": 1e3 * med(t_save), "saves_ms": 1e3 * med(t_save1),
                   "load_many_ms": 1e3 * med(t_load), "loads_ms": 1e3 * med(t_load1),
                   "save_many_GBps": total / med(t_save) / 1e9, "load_many_GBps": total / med(t_load) / 1e9,
                   "copy_d2h_GBps": d2h / 1e9, "copy_h2d_GBps": h2d / 1e9,
                   "save_many_over_copy": total / med(t_save) / d2h, "load_many_over_copy": total / med(t_load) / h2d,
                   "save_many_bytes_equal_single_saves": bool(singles_same), "identical_after_load": identical}
            result["runs"]["%s_S%d" % (name, n)] = row
            print(json.dumps(row), flush=True)
            copy.close()
            for od in sess:
                od.close()
    result["cards_after"] = cards()
    sysm.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(result) + "\n")
    print(json.dumps({"cards": result["cards"], "runs": len(result["runs"])}))


if __name__ == "__main__":
    main()
