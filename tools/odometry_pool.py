"""Many cameras over several GPUs: an OdometryPool of G handles, one per GPU, in one process.

S cameras (headline version, 128x416, trajectory mode) follow seeded streams and push one frame per step, S in
{64, 256, 1024}, G in {1, 2, 4, 8} as far as the box has GPUs, as a host pool (frames in pinned host memory) and as a
device pool (frames resident in each camera's GPU).  Each step is one batched push per handle, all queued before any is
waited for -- what OdometryPool.push does -- with the C ABI called directly and every argument array built beforehand,
so that the numbers are the library's and not the wrapper's.  For each (G, S, pool) it records:
  - frames/s with two steps in flight, and its ratio to G = 1;
  - p50 / p99 step latency (steps queued on idle devices, to every camera's results ready);
  - host-to-device bytes per frame of a mid-stream step (davo_last_host_copy_bytes summed over the handles);
  - midway through the latency run, the time of draining handle G-1 into handle 0 and of the rebalance() that moves
    those S/G sessions back;
  - that every camera's poses and trajectory over the whole run, moves included, equal the G = 1 run's bits.
It prints the name and power limit of every card, read in the same run.  Writes profiles/odometry_pool.log unless --out
says otherwise.

    python tools/odometry_pool.py [--gpus 1,2,4,8] [--sizes 64,256,1024] [--steps 32] [--out FILE]
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
from davo_b200.odometry_pool import OdometryPool     # noqa: E402
from tests.golden import make_golden as G       # noqa: E402

H, W = 128, 416
POOL = 130                    # frames of the stream pool; camera i starts 7 i frames into it (cyclically)


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if q.returncode == 0 and q.stdout.strip():
        return q.stdout.strip().splitlines()
    return [torch.cuda.get_device_name(d) for d in range(torch.cuda.device_count())]


def pinned(a):
    t = torch.empty(a.shape, dtype=getattr(torch, str(a.dtype))).pin_memory()
    t.numpy()[...] = a
    return t.numpy()


class Run(object):
    """The pushes of S cameras of a pool for steps 0..steps as prebuilt per-handle C argument arrays (rebuilt after
    moves), writing each camera's results at [step, camera]."""

    def __init__(self, pool, systems, cams, frames, steps, host):
        self.pool, self.systems, self.cams, self.frames, self.steps, self.host = pool, systems, cams, frames, steps, host
        self.lib = systems[0]._lib
        n = len(cams)
        if host:
            self.pose = pinned(np.zeros((steps + 1, n, 1, 2, 6), np.float32))
            self.traj = pinned(np.zeros((steps + 1, n, 3, 4, 4), np.float64))
        else:      # each camera's results on the device it is on at that step: one buffer per device
            devs = sorted({s.device for s in systems})
            self.pose = {d: torch.zeros((steps + 1, n, 1, 2, 6), device="cuda:%d" % d) for d in devs}
            self.traj = {d: torch.zeros((steps + 1, n, 3, 4, 4), dtype=torch.float64, device="cuda:%d" % d) for d in devs}
        self.tickets = [[C.c_longlong(0) for _ in systems] for _ in range(2)]     # two steps in flight
        self.events = {s.device: [torch.cuda.Event() for _ in range(2)] for s in systems}
        self.placed = [[] for _ in range(steps + 1)]        # per step: (device, camera positions) that wrote it
        self.build()

    def build(self):
        """Per handle and step: (n, sessions, k, img, fwd, bwd, seg, pose, traj, positions)."""
        vp = C.c_void_p
        self.args = []
        for t in range(self.steps + 1):
            k = 2 if t == 0 else 1
            per = []
            for s in self.systems:
                pos = [j for j, c in enumerate(self.cams) if self.pool.session(c)._system is s]
                if not pos:
                    per.append(None)
                    continue
                n = len(pos)
                arr = lambda vals: (vp * n)(*vals)
                img, fwd, bwd, seg = self.frames if self.host else self.frames[s.device]
                fr = [(7 * j + (t + 1 if t else 0)) % (POOL - 2) for j in pos]
                fl = [x if t == 0 else (x - 1) % (POOL - 2) for x in fr]
                addr = (lambda a: a.ctypes.data) if self.host else (lambda a: a.data_ptr())
                pose = self.pose if self.host else self.pose[s.device]
                traj = self.traj if self.host else self.traj[s.device]
                per.append((n, arr([self.pool.session(self.cams[j])._o.value for j in pos]), (C.c_int * n)(*[k] * n),
                            arr([addr(img[x:x + k]) for x in fr]), arr([addr(fwd[e]) for e in fl]),
                            arr([addr(bwd[e]) for e in fl]), arr([addr(seg[x:x + k]) for x in fr]),
                            arr([addr(pose[t, j]) for j in pos]), arr([addr(traj[t, j]) for j in pos]), pos))
            self.args.append(per)

    def queue(self, t):
        self.placed[t] = [(s.device, a[9]) for s, a in zip(self.systems, self.args[t]) if a is not None]
        for g, (s, a) in enumerate(zip(self.systems, self.args[t])):
            if a is None:
                continue
            if self.host:
                rc = self.lib.davo_odometry_push_many_host(a[0], a[1], a[2], a[3], a[4], a[5], a[6], None, a[7], a[8],
                                                           None, None, None, C.byref(self.tickets[t % 2][g]))
            else:
                rc = self.lib.davo_odometry_push_many(a[0], a[1], a[2], a[3], a[4], a[5], a[6], None, a[7], a[8], None,
                                                      None, C.c_void_p(torch.cuda.default_stream(s.device).cuda_stream))
            assert rc == 0, _capi.last_error(self.lib, s._h)
            if not self.host:
                self.events[s.device][t % 2].record(torch.cuda.default_stream(s.device))

    def wait(self, t):
        for g, (s, a) in enumerate(zip(self.systems, self.args[t])):
            if a is None:
                continue
            if self.host:
                assert self.lib.davo_host_wait(s._h, self.tickets[t % 2][g]) == 0
            else:
                self.events[s.device][t % 2].synchronize()

    def results(self):
        """Every camera's poses and trajectory rows of every step, gathered from wherever it was."""
        if self.host:
            return np.array(self.pose), np.array(self.traj)
        pose = np.zeros((self.steps + 1, len(self.cams), 1, 2, 6), np.float32)
        traj = np.zeros((self.steps + 1, len(self.cams), 3, 4, 4), np.float64)
        for t, placed in enumerate(self.placed):
            for d, pos in placed:
                pose[t, pos] = self.pose[d][t, pos].cpu().numpy()
                traj[t, pos] = self.traj[d][t, pos].cpu().numpy()
        return pose, traj


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--sizes", default="64,256,1024")
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=3, help="throughput rounds per (G, S, pool)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "odometry_pool.log"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("odometry_pool.py measures on the GPU; there is none here")
    ndev = torch.cuda.device_count()
    gpus = sorted({1} | {g for g in (int(x) for x in a.gpus.split(",")) if g <= ndev})   # G = 1: the reference bits
    sizes = [int(s) for s in a.sizes.split(",")]
    steps = a.steps
    ver = G.CASES["headline"]
    weights = S.init_weights(ver, seed=31, random_bias=True)
    img, fwd, bwd, seg, _ = S.make_sequence(POOL, H, W, seed=21)
    host_frames = tuple(pinned(x) for x in (img, fwd, bwd, seg))
    dev_frames = {}
    result = {"workload": "S cameras over G handles (one per GPU) in one process, one frame per camera per step, headline "
                          "version, %dx%d, trajectory mode; host pool: frames in pinned host memory; device pool: frames "
                          "resident in each camera's GPU" % (H, W),
              "cards": cards(), "gpus_on_box": ndev, "steps": steps, "runs": {}}
    ref = {}                                                  # (S, pool) -> the G = 1 bits
    rate1 = {}
    for g in gpus:
        systems = []
        for d in range(g):
            s = DAVO(version=ver)
            s.setup_inference(H, W, "davo", 3, max(sizes), device=d)
            s.load_weights(weights)
            systems.append(s)
            if d not in dev_frames:
                dev_frames[d] = tuple(torch.as_tensor(x).to("cuda:%d" % d) for x in (img, fwd, bwd, seg))
        for n in sizes:
            for host in (True, False):
                name = "host" if host else "device"
                pool = OdometryPool(systems, pairs="trajectory", max_push=2, host=host)
                cams = [pool.open() for _ in range(n)]
                run = Run(pool, systems, cams, host_frames if host else dev_frames, steps, host)
                row = {"G": g, "S": n, "pool": name, "placement": pool.counts()}
                # latency run over the whole schedule, idle devices at each step; warms every shape; a drain and a
                # rebalance halfway
                lat = []
                for t in range(steps + 1):
                    if t == steps // 2 and g > 1:
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        drained = 0
                        for c in cams:
                            if pool.session(c)._system is systems[-1]:
                                pool.session(c).move_to(systems[0])
                                drained += 1
                        t1 = time.perf_counter()
                        moved = pool.rebalance()
                        t2 = time.perf_counter()
                        row["drain"] = {"sessions": drained, "s": t1 - t0}
                        row["rebalance"] = {"sessions": moved, "s": t2 - t1, "ms_per_session": 1e3 * (t2 - t1) / max(moved, 1)}
                        row["placement_after"] = pool.counts()
                        run.build()
                    for d in range(g):
                        torch.cuda.synchronize(d)
                    t0 = time.perf_counter()
                    run.queue(t)
                    run.wait(t)
                    if t > 0:
                        lat.append(1e3 * (time.perf_counter() - t0))
                    if t == 2 and host:                   # a mid-stream step
                        row["h2d_bytes_per_frame"] = sum(s.last_host_copy_bytes()[0] for s in systems) / n
                row["step_latency_ms"] = {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)),
                                          "steps": len(lat)}
                bits = run.results()
                if g == 1:
                    ref[(n, name)] = bits
                row["identical_to_one_handle"] = bool(np.array_equal(bits[0], ref[(n, name)][0]) and
                                                      np.array_equal(bits[1], ref[(n, name)][1]))
                # throughput: the sessions reset, steps 1..steps two in flight after a blocking step 0
                rates = []
                for r in range(a.rounds):
                    for c in cams:
                        pool.session(c).reset()
                    run.queue(0)
                    run.wait(0)
                    for d in range(g):
                        torch.cuda.synchronize(d)
                    t0 = time.perf_counter()
                    for t in range(1, steps + 1):
                        run.queue(t)
                        if t > 1:
                            run.wait(t - 1)
                    run.wait(steps)
                    rates.append(n * steps / (time.perf_counter() - t0))
                bits = run.results()
                row["identical_after_throughput_rounds"] = bool(np.array_equal(bits[0], ref[(n, name)][0]) and
                                                                np.array_equal(bits[1], ref[(n, name)][1]))
                med = float(np.median(rates))
                if g == 1:
                    rate1[(n, name)] = med
                row["frames_per_s"] = {"median": med, "all": rates, "per_gpu": med / g,
                                       "over_G1": med / rate1[(n, name)]}
                result["runs"]["G%d_S%d_%s" % (g, n, name)] = row
                print(json.dumps(row), flush=True)
                pool.close_all()
                del run
        for s in systems:
            s.close()
    result["cards_after"] = cards()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(result) + "\n")
    print(json.dumps({"cards": result["cards"], "runs": len(result["runs"])}))


if __name__ == "__main__":
    main()
