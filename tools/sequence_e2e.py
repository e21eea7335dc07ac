"""End-to-end rate of host-fed trajectory inference: a seeded frame stream fed as triplets vs as a frame sequence.

The same N-frame stream (seeded frames, flows, labels; headline version, 128x416) sits in pinned host memory twice:
as the reference's triplet batches (davo_forward_host_pairs_async, 128 samples per call) and as frames
(davo_forward_sequence_host, calls of 130 frames that start every 128 frames).  Both keep two calls in flight.  For
each it reports target frames per second, host->device bytes per frame (davo_last_host_copy_bytes) and the same loop
with DAVO_B200_HOST_COPY_ONLY=1 (copies only, no kernels).  The poses of the two ways are compared bit for bit.

    python tools/sequence_e2e.py [--frames 1026] [--reps 5]
    torchrun --nproc_per_node 8 tools/sequence_e2e.py        # each rank streams its own contiguous frame range

Every rank streams frames [r*F, (r+1)*F + 2) of its own seeded stream.  Rank 0 prints one JSON line (rates summed
over ranks, with the card name and power limit) and appends it to profiles/sequence_e2e.log.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from davo_b200 import synthetic as S                      # noqa: E402
from davo_b200.davo import DAVO                            # noqa: E402
from davo_b200.sequence import sequence_to_triplets        # noqa: E402
from tests.golden.make_golden import CASES                 # noqa: E402

H, W, PER_CALL = 128, 416, 128


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:          # the numbers still stand; say that the card could not be read
        return "unknown (%s)" % e


def pinned(a):
    import torch
    t = torch.empty(a.shape, dtype=getattr(torch, str(a.dtype))).pin_memory()
    t.numpy()[...] = a
    return t.numpy()


def run(calls, reps, copy_only):
    """Issues every call `reps` times with two in flight; returns (seconds, poses of the last rep)."""
    if copy_only:
        os.environ["DAVO_B200_HOST_COPY_ONLY"] = "1"
    else:
        os.environ.pop("DAVO_B200_HOST_COPY_ONLY", None)
    for c in calls[:2]:
        c().result()                                       # warm: staging, pinned rings, every pass shape
    out = []
    t0 = time.perf_counter()
    for r in range(reps):
        pend, out = [], []
        for c in calls:
            pend.append(c())
            if len(pend) == 2:
                out.append(pend.pop(0).result()["pose"])
        out += [p.result()["pose"] for p in pend]
    dt = time.perf_counter() - t0
    os.environ.pop("DAVO_B200_HOST_COPY_ONLY", None)
    return dt, np.concatenate(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8 * PER_CALL + 2, help="frames per rank (a multiple of 128, + 2)")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    import torch
    dev = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(dev)
    n = args.frames
    samples = n - 2
    if samples % PER_CALL:
        raise SystemExit("--frames must be a multiple of %d plus 2" % PER_CALL)
    # this rank's contiguous frame range of one long seeded stream: a seed per range stands for it
    img, fwd, bwd, seg, _ = (pinned(x) for x in S.make_sequence(n, H, W, seed=1000 + rank))
    sysm = DAVO(version=CASES["headline"])
    sysm.setup_inference(H, W, "davo", 3, PER_CALL, device=dev)
    sysm.load_weights(S.init_weights(CASES["headline"]))
    starts = range(0, samples, PER_CALL)
    trip = []
    for s0 in starts:                                      # the same frames as triplet batches, pinned
        t_img, t_flow, t_seg, _ = sequence_to_triplets(img[s0:s0 + PER_CALL + 2], fwd[s0:s0 + PER_CALL + 1],
                                                       bwd[s0:s0 + PER_CALL + 1], seg[s0:s0 + PER_CALL + 2])
        trip.append(tuple(pinned(x) for x in (t_img, t_flow, t_seg)))
    ways = {
        "triplet": [lambda t=t: sysm.inference_async(t, pairs="trajectory") for t in trip],
        "sequence": [lambda s0=s0: sysm.inference_sequence_async(img[s0:s0 + PER_CALL + 2], None, bwd[s0:s0 + PER_CALL + 1],
                                                                  seg[s0:s0 + PER_CALL + 2], pairs="trajectory")
                     for s0 in starts],
    }
    res, poses = {}, {}
    for name, calls in ways.items():
        if world > 1:
            torch.distributed.barrier()
        dt, poses[name] = run(calls, args.reps, False)
        calls[0]().result()
        h2d = sysm.last_host_copy_bytes()[0]
        if world > 1:
            torch.distributed.barrier()
        dt_copy, _ = run(calls, args.reps, True)
        res[name] = {"frames_per_s": samples * args.reps / dt, "h2d_bytes_per_frame": h2d / PER_CALL,
                     "copy_only_frames_per_s": samples * args.reps / dt_copy}
    same = bool(np.array_equal(poses["triplet"], poses["sequence"]))
    if world > 1:
        vals = torch.tensor([[res[w][k] for k in ("frames_per_s", "copy_only_frames_per_s")] for w in ("triplet", "sequence")]
                            + [[float(same), 0.0]], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(vals)
        for i, w in enumerate(("triplet", "sequence")):
            res[w]["frames_per_s"], res[w]["copy_only_frames_per_s"] = vals[i].tolist()
        same = vals[2, 0].item() == world
    if rank == 0:
        line = {"workload": "host-fed trajectory mode, headline version, %dx%d, %d frames per rank, %d samples per call, "
                            "2 calls in flight" % (H, W, n, PER_CALL),
                "gpus": world, "card": card(), "poses_identical": same, **res,
                "speedup": res["sequence"]["frames_per_s"] / res["triplet"]["frames_per_s"]}
        print(json.dumps(line))
        root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
        out = os.environ.get("SEQUENCE_E2E_LOG", os.path.join(root, "profiles", "sequence_e2e.log"))
        with open(out, "a") as f:
            f.write(json.dumps(line) + "\n")
    sysm.close()


if __name__ == "__main__":
    if int(os.environ.get("WORLD_SIZE", 1)) > 1:
        import torch.distributed
        torch.distributed.init_process_group("nccl")
    main()
    if int(os.environ.get("WORLD_SIZE", 1)) > 1:
        torch.distributed.destroy_process_group()
