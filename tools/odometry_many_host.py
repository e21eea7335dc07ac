"""Many cameras fed from host memory: batched pushes of host sessions against pushing each session alone.

S host sessions (headline version, 128x416, trajectory mode) follow seeded streams in pinned host memory and push one
frame per step, S in {1, 4, 16, 64, 128}, two steps in flight.  For each S, in the same run and alternating:
  - frames/s of davo_odometry_push_many_host against the same pushes as S davo_odometry_push calls;
  - frames/s of inference_sequence_async with 130-frame calls every 128 frames on the same pinned frames, the host-fed
    ceiling of DESIGN.md section 8.2;
  - p50 / p99 step latency, from the call to every session's poses and trajectory in host memory (blocking calls on an
    idle device);
  - host-to-device bytes per frame (davo_last_host_copy_bytes) of both ways;
  - the host time spent inside the asynchronous batched call per step, against the step time, and the rate the
    measured pinned host-to-device bandwidth alone would allow at those bytes: which of the host thread and the copies
    bounds the step.
It checks that both ways give identical poses and trajectories, and prints the card name and power limit read in the
same run.  Writes profiles/odometry_many_host.log unless --out says otherwise.  The C ABI is called directly, with every
argument array built beforehand, so that the numbers are the library's and not the wrapper's.

    python tools/odometry_many_host.py [--sizes 1,4,16,64,128] [--steps 64] [--out FILE]
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
POOL = 130                    # frames of the pinned pool: one 130-frame sequence call, and the sessions' streams
PER_CALL = 128


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def pinned(a):
    t = torch.empty(a.shape, dtype=getattr(torch, str(a.dtype))).pin_memory()
    t.numpy()[...] = a
    return t.numpy()


class Fleet(object):
    """S host sessions on one handle, their pushes as prebuilt C argument arrays, outputs page-locked."""

    def __init__(self, sysm, pool, n, steps):
        self.sysm, self.lib, self.n = sysm, sysm._lib, n
        self.sessions = [sysm.odometry("trajectory", 2, host=True) for _ in range(n)]
        img, fwd, bwd, seg = pool
        self.pose = pinned(np.zeros((steps + 1, n, 1, 2, 6), np.float32))
        self.traj = pinned(np.zeros((steps + 1, n, 3, 4, 4), np.float64))
        vp, ip = C.c_void_p, C.c_int
        arr = lambda vals: (vp * n)(*vals)
        self.sess = arr([od._o.value for od in self.sessions])
        self.args = []
        for t in range(steps + 1):
            # session i follows the pool from frame 7 i on (cyclically); step 0 pushes two frames, so that every later
            # step is a mid-stream push of one frame and its flow entry
            k = 2 if t == 0 else 1
            fr = [(7 * i + (t + 1 if t else 0)) % (POOL - 2) for i in range(n)]
            fl = [x if t == 0 else (x - 1) % (POOL - 2) for x in fr]
            im = [img[x:x + k].ctypes.data for x in fr]
            sg = [seg[x:x + k].ctypes.data for x in fr]
            fw = [fwd[e].ctypes.data for e in fl]
            bw = [bwd[e].ctypes.data for e in fl]
            po = [self.pose[t, i].ctypes.data for i in range(n)]
            tr = [self.traj[t, i].ctypes.data for i in range(n)]
            self.args.append(((ip * n)(*[k] * n), arr(im), arr(fw), arr(bw), arr(sg), arr(po), arr(tr), k, im, fw, bw,
                              sg, po, tr))
        self.ticket = C.c_longlong(0)

    def many(self, t, block=False):
        a = self.args[t]
        rc = self.lib.davo_odometry_push_many_host(self.n, self.sess, a[0], a[1], a[2], a[3], a[4], None, a[5], a[6],
                                                   None, None, None, None if block else C.byref(self.ticket))
        assert rc == 0, _capi.last_error(self.lib, self.sysm._h)

    def single(self, t, block=False):
        a = self.args[t]
        k, im, fw, bw, sg, po, tr = a[7:]
        for i, od in enumerate(self.sessions):
            rc = self.lib.davo_odometry_push(od._o, k, C.c_void_p(im[i]), C.c_void_p(fw[i]), C.c_void_p(bw[i]),
                                             C.c_void_p(sg[i]), None, C.c_void_p(po[i]), C.c_void_p(tr[i]), None, None,
                                             None, None if block else C.byref(self.ticket))
            assert rc == 0, _capi.last_error(self.lib, self.sysm._h)

    def reset(self):
        for od in self.sessions:
            od.reset()

    def close(self):
        for od in self.sessions:
            od.close()


def two_in_flight(go, steps, in_call=None):
    """Steps 1..steps of `go`, each queued while the one before runs: after queueing step t, wait for step t-1 (an event
    on the default stream, which both ways enqueue on).  Returns the wall time; `in_call` collects the host time inside
    each call."""
    evs = [torch.cuda.Event() for _ in range(2)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t in range(1, steps + 1):
        c0 = time.perf_counter()
        go(t)
        if in_call is not None:
            in_call.append(time.perf_counter() - c0)
        evs[t % 2].record(torch.cuda.default_stream())
        if t > 1:
            evs[(t - 1) % 2].synchronize()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def h2d_bandwidth(nbytes=1 << 30, reps=5):
    """Pinned host -> device copy rate of one large buffer (GB/s), median of `reps`."""
    src = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    dst = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dst.copy_(src, non_blocking=True)
    rates = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        rates.append(nbytes / (time.perf_counter() - t0) / 1e9)
    return float(np.median(rates))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,4,16,64,128")
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--lat", type=int, default=200, help="latency steps per way")
    ap.add_argument("--seq-calls", type=int, default=16, help="sequence calls per round of the ceiling")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "odometry_many_host.log"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("odometry_many_host.py measures on the GPU; there is none here")
    sizes = [int(s) for s in a.sizes.split(",")]
    steps = a.steps
    ver = G.CASES["headline"]
    sysm = DAVO(version=ver)
    sysm.setup_inference(H, W, "davo", 3, max(max(sizes), PER_CALL) + 2, device=0)
    sysm.load_weights(S.init_weights(ver, seed=31, random_bias=True))
    img, fwd, bwd, seg, _ = S.make_sequence(POOL, H, W, seed=21)
    pool = tuple(pinned(x) for x in (img, fwd, bwd, seg))
    result = {"workload": "S host odometry sessions, one frame per step each, headline version, %dx%d, trajectory mode, "
                          "frames in pinned host memory, two steps in flight" % (H, W), "card": card(), "steps": steps,
              "sizes": {}}
    bw = h2d_bandwidth()
    result["pinned_h2d_GB_per_s"] = bw

    def seq_round():
        """inference_sequence_async calls of 130 frames on the pinned pool, two in flight; frames/s."""
        pend = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.seq_calls):
            pend.append(sysm.inference_sequence_async(pool[0], pool[1], pool[2], pool[3], pairs="trajectory"))
            if len(pend) > 1:
                pend.pop(0).result()
        for p in pend:
            p.result()
        return PER_CALL * a.seq_calls / (time.perf_counter() - t0)

    seq_round()                                                           # warm
    seq_bytes = sysm.last_host_copy_bytes()[0] / PER_CALL
    for n in sizes:
        fa, fb = Fleet(sysm, pool, n, max(steps, a.lat)), Fleet(sysm, pool, n, max(steps, a.lat))
        row = {}
        # identical results, and warm-up of every shape: the whole schedule once each way, blocking
        for go in (fa.many, fb.single):
            for t in range(steps + 1):
                go(t, block=True)
        row["identical"] = bool(np.array_equal(fa.pose[:steps + 1], fb.pose[:steps + 1]) and
                                np.array_equal(fa.traj[:steps + 1], fb.traj[:steps + 1]))
        # bytes of one mid-stream step each way
        fa.many(1, block=True)
        many_b = sysm.last_host_copy_bytes()[0]
        single_b = 0
        for i in range(n):                                                # the single pushes' counts, summed
            a_ = fb.args[1]
            rc = sysm._lib.davo_odometry_push(fb.sessions[i]._o, 1, C.c_void_p(a_[8][i]), C.c_void_p(a_[9][i]),
                                              C.c_void_p(a_[10][i]), C.c_void_p(a_[11][i]), None, C.c_void_p(a_[12][i]),
                                              C.c_void_p(a_[13][i]), None, None, None, None)
            assert rc == 0, _capi.last_error(sysm._lib, sysm._h)
            single_b += sysm.last_host_copy_bytes()[0]
        row["h2d_bytes_per_frame"] = {"many": many_b / n, "single": single_b / n, "sequence_calls": seq_bytes}
        # throughput: rounds of `steps` steps, batched, single and sequence calls alternating, sessions reset between
        rates = {"many": [], "single": [], "sequence_calls_130": []}
        in_call = []
        for r in range(3):
            for name, f, go in (("many", fa, fa.many), ("single", fb, fb.single)):
                f.reset()
                go(0, block=True)
                dt = two_in_flight(go, steps, in_call if name == "many" else None)
                rates[name].append(n * steps / dt)
            rates["sequence_calls_130"].append(seq_round())
        row["frames_per_s"] = {k: {"median": float(np.median(v)), "all": v} for k, v in rates.items()}
        med = row["frames_per_s"]
        row["many_over_single"] = med["many"]["median"] / med["single"]["median"]
        row["many_over_sequence_calls"] = med["many"]["median"] / med["sequence_calls_130"]["median"]
        step_ms = 1e3 * n / med["many"]["median"]
        row["many_host"] = {"in_call_ms_per_step_p50": 1e3 * float(np.percentile(in_call, 50)),
                            "step_ms": step_ms,
                            "in_call_share_of_step": 1e3 * float(np.percentile(in_call, 50)) / step_ms,
                            "copy_bound_frames_per_s": bw * 1e9 / (many_b / n),
                            "of_copy_bound": med["many"]["median"] / (bw * 1e9 / (many_b / n))}
        # latency: each step starts on an idle device, blocking call to results in host memory
        lat = {"many": [], "single": []}
        for name, f, go in (("many", fa, fa.many), ("single", fb, fb.single)):
            f.reset()
            go(0, block=True)
            for t in range(1, a.lat + 1):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                go(t, block=True)
                lat[name].append(1e3 * (time.perf_counter() - t0))
        row["step_latency_ms"] = {k: {"p50": float(np.percentile(v, 50)), "p99": float(np.percentile(v, 99)),
                                      "steps": len(v)} for k, v in lat.items()}
        result["sizes"][str(n)] = row
        print(json.dumps({str(n): row}), flush=True)
        fa.close()
        fb.close()
    result["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(result) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
