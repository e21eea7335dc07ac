"""Many cameras, one frame each, at the same time: batched odometry pushes against pushing each session alone.

S device sessions (headline version, 128x416, trajectory mode) follow seeded streams resident in HBM and push one frame
per step, S in {1, 4, 16, 64, 128, 256}.  For each S, in the same run and alternating:
  - frames/s of davo_odometry_push_many against the same pushes as S davo_odometry_push calls;
  - p50 / p99 step latency, from the call to traj_out ready (CUDA events around an idle-started step);
  - odo_stage_kernel time (torch.profiler, a run of its own) and its bytes over that time against the copy peak of
    DESIGN.md section 8.
It checks that both ways give identical poses and trajectories, and prints the card name and power limit read in the
same run.  Writes profiles/odometry_many.log unless --out says otherwise.  The C ABI is called directly, with every
buffer allocated beforehand, so that the numbers are the library's and not the wrapper's.

    python tools/odometry_many.py [--sizes 1,4,16,64,128,256] [--steps 64] [--out FILE]
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
from davo_b200.davo import DAVO                 # noqa: E402
from tests.golden import make_golden as G       # noqa: E402

H, W = 128, 416
POOL = 96                     # frames of the resident pool; session i starts 7 i frames into it
COPY_PEAK_GBS = 6458.0        # DESIGN.md section 4.2 / 8: measured device copy peak on one B200


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def stage_bytes(sysm, n):
    """Bytes odo_stage_kernel reads and writes for n mid-stream trajectory samples (tgt and src1 only)."""
    c, hw = sysm.config, H * W
    flow = c.in_mode == 1 or c.att_src in (1, 6) or c.pixel_map == 2
    labels = c.att_src != 0 and (not c.pixel_map or c.att_src == 6)
    nlab = (2 if not c.att_tgt_ones else 1) if labels else 0
    per = 2 * 2 * hw * 3 + nlab * hw * (4 + 1) + (2 * hw * 8 if flow else 0)
    return n * per


class Fleet(object):
    """S sessions on one handle, their pushes as prebuilt C argument arrays."""

    def __init__(self, sysm, pool, n, steps):
        self.sysm, self.lib, self.n = sysm, sysm._lib, n
        self.sessions = [sysm.odometry("trajectory", 2, host=False) for _ in range(n)]
        img, fwd, bwd, seg = pool
        self.pose = torch.zeros((steps + 1, n, 1, 2, 6), device="cuda")
        self.traj = torch.zeros((steps + 1, n, 3, 4, 4), dtype=torch.float64, device="cuda")
        vp, ip = C.c_void_p, C.c_int
        arr = lambda vals: (vp * n)(*vals)
        self.sess = arr([od._o.value for od in self.sessions])
        self.args = []
        for t in range(steps + 1):
            # session i follows the pool from frame 7 i on (cyclically: only the timing reads past the end); step 0
            # pushes two frames, so that every later step is a mid-stream push of one frame and its flow entry
            k = 2 if t == 0 else 1
            fr = [(7 * i + (t + 1 if t else 0)) % (POOL - 1) for i in range(n)]
            fl = [x if t == 0 else (x - 1) % (POOL - 1) for x in fr]
            im = [img[x:x + k].data_ptr() for x in fr]
            sg = [seg[x:x + k].data_ptr() for x in fr]
            fw = [fwd[e].data_ptr() for e in fl]
            bw = [bwd[e].data_ptr() for e in fl]
            po = [self.pose[t, i].data_ptr() for i in range(n)]
            tr = [self.traj[t, i].data_ptr() for i in range(n)]
            self.args.append(((ip * n)(*[k] * n), arr(im), arr(fw), arr(bw), arr(sg), arr(po), arr(tr), k, im, fw, bw,
                              sg, po, tr))

    def many(self, t, stream):
        a = self.args[t]
        rc = self.lib.davo_odometry_push_many(self.n, self.sess, a[0], a[1], a[2], a[3], a[4], None, a[5], a[6], None, None,
                                              C.c_void_p(stream))
        assert rc == 0, _capi.last_error(self.lib, self.sysm._h)

    def single(self, t, stream):
        a = self.args[t]
        k, im, fw, bw, sg, po, tr = a[7:]
        for i, od in enumerate(self.sessions):
            rc = self.lib.davo_odometry_push(od._o, k, C.c_void_p(im[i]), C.c_void_p(fw[i]), C.c_void_p(bw[i]),
                                             C.c_void_p(sg[i]), None, C.c_void_p(po[i]), C.c_void_p(tr[i]), None, None,
                                             C.c_void_p(stream), None)
            assert rc == 0, _capi.last_error(self.lib, self.sysm._h)

    def reset(self):
        for od in self.sessions:
            od.reset()

    def close(self):
        for od in self.sessions:
            od.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,4,16,64,128,256")
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--lat", type=int, default=200, help="latency steps per way")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "odometry_many.log"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("odometry_many.py measures on the GPU; there is none here")
    sizes = [int(s) for s in a.sizes.split(",")]
    steps = a.steps
    ver = G.CASES["headline"]
    sysm = DAVO(version=ver)
    sysm.setup_inference(H, W, "davo", 3, max(sizes) + 2, device=0)
    sysm.load_weights(S.init_weights(ver, seed=31, random_bias=True))
    img, fwd, bwd, seg, _ = S.make_sequence(POOL, H, W, seed=21)
    pool = tuple(torch.as_tensor(x).cuda() for x in (img, fwd, bwd, seg))
    stream = torch.cuda.current_stream().cuda_stream
    result = {"workload": "S device odometry sessions, one frame per step each, headline version, %dx%d, trajectory "
                          "mode, frames resident in HBM" % (H, W), "card": card(), "steps": steps, "sizes": {}}
    for n in sizes:
        fa, fb = Fleet(sysm, pool, n, max(steps, a.lat)), Fleet(sysm, pool, n, max(steps, a.lat))
        row = {}
        # identical results, and warm-up of every shape: the whole schedule once each way
        for f, go in ((fa, fa.many), (fb, fb.single)):
            for t in range(steps + 1):
                go(t, stream)
        torch.cuda.synchronize()
        same = bool(torch.equal(fa.pose[:steps + 1], fb.pose[:steps + 1]) and torch.equal(fa.traj[:steps + 1], fb.traj[:steps + 1]))
        row["identical"] = same
        # throughput: rounds of `steps` steps, batched and single alternating, the sessions reset between rounds
        rates = {"many": [], "single": []}
        for r in range(3):
            for name, f, go in (("many", fa, fa.many), ("single", fb, fb.single)):
                f.reset()
                go(0, stream)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for t in range(1, steps + 1):
                    go(t, stream)
                torch.cuda.synchronize()
                rates[name].append(n * steps / (time.perf_counter() - t0))
        row["frames_per_s"] = {k: {"median": float(np.median(v)), "all": v} for k, v in rates.items()}
        row["many_over_single"] = row["frames_per_s"]["many"]["median"] / row["frames_per_s"]["single"]["median"]
        # latency: each step starts on an idle device; the events bracket the call and its last kernel
        lat = {"many": [], "single": []}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for name, f, go in (("many", fa, fa.many), ("single", fb, fb.single)):
            f.reset()
            go(0, stream)
            for t in range(1, a.lat + 1):
                torch.cuda.synchronize()
                ev0.record()
                go(t, stream)
                ev1.record()
                ev1.synchronize()
                lat[name].append(ev0.elapsed_time(ev1))
        row["step_latency_ms"] = {k: {"p50": float(np.percentile(v, 50)), "p99": float(np.percentile(v, 99)),
                                      "steps": len(v)} for k, v in lat.items()}
        # the stage kernel, in a profiled run of its own
        from torch.profiler import ProfilerActivity, profile
        fa.reset()
        fa.many(0, stream)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for t in range(1, 17):
                fa.many(t, stream)
            torch.cuda.synchronize()
        us = [e for e in prof.key_averages() if "odo_stage_kernel" in e.key]
        if us:
            tot = getattr(us[0], "device_time_total", None) or getattr(us[0], "cuda_time_total", 0.0)
            per = tot / max(us[0].count, 1)
            b = stage_bytes(sysm, n)
            row["stage_kernel"] = {"us": per, "bytes": b, "GB_per_s": b / per / 1e3,
                                   "of_copy_peak": b / per / 1e3 / COPY_PEAK_GBS}
        result["sizes"][str(n)] = row
        print(json.dumps({str(n): row}), flush=True)
        fa.close()
        fb.close()
    result["copy_peak_GB_per_s"] = COPY_PEAK_GBS
    result["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(result) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
