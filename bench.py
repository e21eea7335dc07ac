#!/usr/bin/env python
"""Benchmark of the DAVO pose forward path (BASELINE.json metric: frame pairs / second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A step is one pass of the hot path (attention front end -> dilated PoseNN -> 6-DoF
head) over one batch of synthetic 128x416 samples: 128 samples = 256 frame pairs
per GPU (BASELINE.json configs[1]).  Under torchrun every rank runs its own batch
(weak scaling) and the poses are all-gathered once per step over NCCL; started
plainly with ``--gpus N`` > 1, bench.py re-launches itself under
``torch.distributed.run`` with N ranks on 127.0.0.1.

Prints ONE JSON line (rank 0).  ``value`` is device-resident throughput, ``e2e``
the same metric through ``DAVO.inference`` with host numpy inputs (host<->device
copies inside the timed region), ``roofline`` the dominant kernel (cnv6) against
the measured tensor peak, ``cpu_baseline`` the oracle's fp32 CPU restatement of
the reference graph timed on this box's host cores.  Correctness travels with the
numbers: ``parity`` compares the poses of the timed batch (device-resident and
host-fed) with the fp32 oracle on the same inputs (tolerance 1e-4 + 1e-3 |ref|,
BASELINE.json north_star); under N > 1 the per-step gather is the library's own
``davo_allgather_poses`` and ``gather_check`` says whether the gathered
[N*B,2,6] equals, bit for bit, what rank 0 computes alone from every rank's
seeded inputs.  ``stream_4541`` is BASELINE configs[2]: the 4541-frame stream
sharded over the N ranks (strong scaling), gathered and composed.

``--dump-outputs DIR`` writes (rank 0) what the last timed step returned to its
caller as ``DIR/pose.npy``: the CUDA path's [N*B,2,6] float32 poses (gathered
over the N ranks), or under ``--impl reference`` the oracle's [16,2,6] float64
poses of its CPU sample.  Inputs and weights are seeded, so two builds run with
the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

VERSION = "v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh"
H, W = 128, 416
FLOP_PER_PAIR = 7780171776            # SURVEY.md 8(d): 2 x 3 890 085 888 MACs, all conv layers
FLOP_PER_PAIR_LAYER = {               # 2 x MACs per frame pair (SURVEY.md 8a table)
    "cnv1": 2 * 104366080, "cnv2": 2 * 42598400, "cnv3": 2 * 61341696, "cnv4": 2 * 245366784,
    "cnv5": 2 * 981467136, "cnv6": 2 * 1962934272, "cnv7": 2 * 490733568,
}
FRONT_BYTES_PER_PAIR = 3008512        # SURVEY.md 8(d) minimum front-end traffic
METRIC = "PoseNN+attention frame-pairs/sec @128x416"
UNIT = "frame-pairs/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "of measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "of fallback"


def ncu_traffic(layer):
    """DRAM bytes (read + write) per launch of `layer`'s kernel from the newest committed
    `ncu --set full` capture (profiles/r*_ncu_traffic.json), or None.  Not measured by this run."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_traffic.json")))
    if not files:
        return None, None
    with open(files[-1]) as f:
        d = json.load(f)
    e = d.get("layers", {}).get(layer)
    if not e:
        return None, None
    return e["dram_bytes_read"] + e["dram_bytes_write"], {
        "file": os.path.relpath(files[-1], ROOT), "pairs_per_launch": e.get("pairs_per_launch"),
        "tensor_pipe_pct": e.get("tensor_pipe_pct")}


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def live_tf32_gemm_tflops(dev, n=8192, reps=10):
    """cuBLAS TF32 GEMM (torch.matmul, allow_tf32) n^3, best of `reps`: a live tensor-pipe peak for
    the arithmetic type this path computes in (MEASURED_PEAKS.json only holds bf16)."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(3):
            a @ b
        best = None
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def cpu_oracle_rate(batch, iters, threads=None, min_seconds=0.0, inputs=None):
    """Frame pairs / s of the oracle's fp32 torch-CPU restatement on the host cores; also returns the
    poses it computed (for the given `inputs`' first `batch` samples when given)."""
    import torch
    from davo_b200 import synthetic as S
    from oracle import davo_oracle as O
    if threads:
        torch.set_num_threads(threads)
    w = S.init_weights(VERSION)
    if inputs is None:
        img, flow, seg = S.make_inputs(batch, H, W, seed=4321)
    else:
        img, flow, seg = (a[:batch] for a in inputs)
    O.davo_forward(VERSION, img[:1], flow[:1], seg[:1], w, torch.float32)     # warm
    t0 = time.perf_counter()
    done = 0
    poses = None
    while done < iters or time.perf_counter() - t0 < min_seconds:
        poses = O.davo_forward(VERSION, img, flow, seg, w, torch.float32)
        done += 1
    dt = time.perf_counter() - t0
    return 2 * batch * done / dt, dt, torch.get_num_threads(), done, poses


def parity_block(ref, **got):
    """max |gpu - oracle32| of each given pose array against the north_star tolerance 1e-4 + 1e-3 |ref|."""
    import numpy as np
    out = {"n_samples": int(ref.shape[0]), "against": "fp32 oracle (CPU restatement held to the reference's own graph "
           "code by tests/golden/poses.npz)", "tolerance": "abs(gpu - ref) <= 1e-4 + 1e-3 * abs(ref)", "ok": True}
    for name, g in got.items():
        g = np.asarray(g, np.float64)[: ref.shape[0]]
        err = np.abs(g - ref)
        ok = bool(np.all(np.isfinite(g)) and np.all(err <= 1e-4 + 1e-3 * np.abs(ref)))
        out[name] = {"max_abs": float(err.max()), "max_abs_ref": float(np.abs(ref).max()), "ok": ok}
        out["ok"] = out["ok"] and ok
    return out


def dump_outputs(out_dir, **arrays):
    """Writes each array as ``out_dir/<name>.npy``, float64 kept, anything else as float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def run_reference(args):
    """--impl reference: the reference graph's CPU restatement (oracle port) on host cores.

    TensorFlow 1.13 cannot be installed here, so this arm times the oracle, with
    every host thread torch will use, on a bounded sample of the same workload.
    """
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = 16
    cores = os.cpu_count() or 1
    for _ in range(max(args.warmup, 1) - 1):
        cpu_oracle_rate(batch, 1, cores)
    steps = max(1, args.steps)                   # a step = 16 samples: ~0.2 s of CPU work
    rate, dt, thr, steps, poses = cpu_oracle_rate(batch, steps, cores)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, pose=poses)
    sample = "%d steps x %d samples (%d frame pairs each) of the 128-sample batch, fp32 torch-CPU" % (
        steps, batch, 2 * batch)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "configs[1]: 256 frame pairs (128 samples) @128x416, headline variant; "
                               "bounded CPU sample", "version": VERSION},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": thr, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle port of the TF 1.13 graph (TF not installable); not TensorFlow itself",
    }
    print(json.dumps(line), flush=True)


def stream_4541(system, dev, rank, world, dist, n_samples=4539, batch=128):
    """BASELINE.json configs[2]: the 4541-frame stream (4539 samples) sharded by sample over the ranks (contiguous
    blocks, the last padded by the reference's complete_batch_size rule), each rank's shard resident in HBM, run in
    128-sample batches in trajectory mode (only the poses reference test_kitti_pose.py:143-145 composes), gathered
    once by davo_allgather_poses, composed on rank 0.  STRONG scaling: the stream is fixed, the ranks divide it.
    Returns (on rank 0) ms per stream = max over ranks of the device time, frames/s and the host composition time."""
    import numpy as np
    import torch
    from davo_b200 import geo_utils, parallel
    from davo_b200 import synthetic as S
    idx = parallel.padded_indices(n_samples, rank, world)
    n_local = len(idx)
    # the shard's inputs: a seeded 64-sample block tiled over the shard, resident (2.8 MB per sample)
    base = [torch.as_tensor(x).to(dev) for x in S.make_inputs(64, H, W, seed=1000 + rank)]
    reps = -(-n_local // 64)
    shard = [t.repeat((reps,) + (1,) * (t.dim() - 1))[:n_local].contiguous() for t in base]
    del base
    poses = torch.empty((n_local, 2, 6), dtype=torch.float32, device=dev)

    def run_stream():
        for b0 in range(0, n_local, batch):
            b1 = min(b0 + batch, n_local)
            mode = "trajectory_first" if (rank == 0 and b0 == 0) else "trajectory"
            out = system.inference(None, "pose", inputs=tuple(t[b0:b1] for t in shard), as_torch=True, pairs=mode)["pose"]
            poses[b0:b1] = out
        return parallel.gather_poses(poses, n_samples, system)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(2):
        allp = run_stream()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps_t = 5
    e0.record()
    for _ in range(reps_t):
        allp = run_stream()
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1) / reps_t], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    del shard
    if rank != 0:
        return None
    allp = allp.cpu().numpy()
    t0 = time.perf_counter()
    traj = geo_utils.compose_trajectory(allp)
    t_host = time.perf_counter() - t0
    ms = float(ms.item())
    return {"workload": "configs[2]: 4541-frame stream = 4539 samples, sample-sharded x%d (%d per rank), trajectory mode, "
                        "inputs resident in HBM, one davo_allgather_poses, host composition on rank 0" % (world, n_local),
            "scaling": "strong", "n_gpus": world, "frames": int(traj.shape[0]), "ms_per_stream": ms,
            "frames_per_s": 4541 / (ms * 1e-3), "frame_pairs_computed": n_samples + 1,
            "host_composition_ms": 1e3 * t_host, "finite": bool(np.all(np.isfinite(traj))),
            "passes_per_rank": -(-n_local // batch), "last_pass_samples": n_local - (n_local - 1) // batch * batch}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from davo_b200 import synthetic as S
    from davo_b200.davo import DAVO
    from davo_b200 import parallel

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the davo_b200 path has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    B = args.batch
    peaks, peak_kind = measured_peaks()

    weights = S.init_weights(VERSION)
    img, flow, seg = S.make_inputs(B, H, W, seed=1234 + rank)
    d_img, d_flow, d_seg = (torch.as_tensor(x).to(dev) for x in (img, flow, seg))
    system = DAVO(version=VERSION)
    system.setup_inference(H, W, "davo", 3, B, d_img, input_flow=d_flow, input_seglabel=d_seg,
                           device=local, micro_batch=args.micro_batch)
    system.load_weights(weights)
    # ranks that share a host: keep each rank's threads and pinned staging on the NUMA node of its GPU
    numa_node = system.bind_host_numa() if (world > 1 and os.environ.get("DAVO_B200_NUMA_BIND", "1") != "0") else -1

    if world > 1:
        system.init_comm(rank, world)            # the handle's own NCCL communicator (davo_comm_create)

    def step():
        out = system.inference(None, "pose", as_torch=True)["pose"]
        if world > 1:
            out = parallel.gather_poses(out, world * B, system)      # davo_allgather_poses (ncclAllGather, compute stream)
        return out

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(args.steps):
        timed_out = step()
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    launches = system.last_launch_count() * args.steps
    timed_out = timed_out.cpu().numpy()          # [world*B,2,6] under N > 1 (gathered), [B,2,6] at N = 1
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pose=timed_out)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * 2 * B * args.steps / (ms * 1e-3)

    # end to end: host numpy in, host numpy out, through the public API
    h_img, h_flow, h_seg = (torch.as_tensor(x).pin_memory().numpy() for x in (img, flow, seg))
    e2e_steps = max(2, min(args.steps, 50))
    for _ in range(2):
        system.inference(None, "pose", inputs=(h_img, h_flow, h_seg))
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        pose_host = system.inference(None, "pose", inputs=(h_img, h_flow, h_seg))["pose"]
    torch.cuda.synchronize()
    dt_sync = torch.tensor([time.perf_counter() - t0], device=dev)
    # the same loop through the asynchronous form of the same call (DAVO.inference_async): step k+1's copies are queued
    # while step k computes, as tf.data's prefetch does for the reference's sess.run loop; every step's inputs still
    # cross PCIe inside the region and every step's poses are read back on the host
    sync_all()
    t0 = time.perf_counter()
    pending = None
    for _ in range(e2e_steps):
        nxt = system.inference_async((h_img, h_flow, h_seg))
        if pending is not None:
            pose_host = pending.result()["pose"]
        pending = nxt
    pose_host = pending.result()["pose"].copy()
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dt_sync, op=dist.ReduceOp.MAX)
    e2e_sync_value = world * 2 * B * e2e_steps / float(dt_sync.item())
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = world * 2 * B * e2e_steps / float(dt.item())
    h2d, d2h = system.last_host_copy_bytes()      # counted by the library from the copies it issues
    # the same, for a caller whose loader already holds byte labels and half-precision flow (extension, labelled)
    c_flow, c_seg = S.compact_inputs(flow, seg)
    c_flow, c_seg = (torch.as_tensor(x).pin_memory().numpy() for x in (c_flow, c_seg))
    for _ in range(2):
        pose_compact = system.inference(None, "pose", inputs=(h_img, c_flow, c_seg))["pose"]
    sync_all()
    t0 = time.perf_counter()
    pending = None
    for _ in range(e2e_steps):
        nxt = system.inference_async((h_img, c_flow, c_seg))
        if pending is not None:
            pose_compact = pending.result()["pose"]
        pending = nxt
    pose_compact = pending.result()["pose"].copy()
    torch.cuda.synchronize()
    dtk = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dtk, op=dist.ReduceOp.MAX)
    compact_value = world * 2 * B * e2e_steps / float(dtk.item())
    compact_h2d = system.last_host_copy_bytes()[0]
    system.inference(None, "pose", inputs=(h_img, h_flow, h_seg))     # leave the float-input state behind for what follows
    # What the host's links give when EVERY rank copies at once: a plain pinned host->device copy of the same number
    # of bytes, all ranks released together by a barrier, timed on each rank's device; the bound uses the slowest.
    pin = torch.empty(h2d, dtype=torch.uint8).pin_memory()
    dst = torch.empty(h2d, dtype=torch.uint8, device=dev)
    dst.copy_(pin, non_blocking=True)
    sync_all()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(5):
        dst.copy_(pin, non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    gb = torch.tensor([5 * h2d / (c0.elapsed_time(c1) * 1e-3) / 1e9], device=dev)
    gb_min = gb.clone()
    if world > 1:
        dist.all_reduce(gb_min, op=dist.ReduceOp.MIN)
        dist.all_reduce(gb, op=dist.ReduceOp.SUM)
    pcie_gbs, pcie_gbs_sum = float(gb_min.item()), float(gb.item())
    del pin, dst
    # the library's own copies without compute (DAVO_B200_HOST_COPY_ONLY): staging + H2D of exactly what it moves
    os.environ["DAVO_B200_HOST_COPY_ONLY"] = "1"
    sync_all()
    t0 = time.perf_counter()
    pending = None
    for _ in range(5):
        nxt = system.inference_async((h_img, h_flow, h_seg))
        if pending is not None:
            pending.result()
        pending = nxt
    pending.result()
    torch.cuda.synchronize()
    dtc = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dtc, op=dist.ReduceOp.MAX)
    os.environ.pop("DAVO_B200_HOST_COPY_ONLY")
    copy_only_value = world * 2 * B * 5 / float(dtc.item())
    stream = None if os.environ.get("DAVO_BENCH_SKIP_STREAM") else stream_4541(system, dev, rank, world, dist)   # skipped under ncu

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # dominant kernel (cnv6) timed alone, live, with CUDA events on the launch stream
    system.inference(None, "pose", as_torch=True)   # rank-local (no collective): rebinds the device-resident inputs
    torch.cuda.synchronize()
    # SURVEY 8(f)1: what the trajectory CLI runs -- only the poses test_kitti_pose.py:143-145 composes
    for _ in range(3):
        system.inference(None, "pose", as_torch=True, pairs="trajectory_first")
    t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0e.record()
    for _ in range(20):
        system.inference(None, "pose", as_torch=True, pairs="trajectory_first")
    t1e.record()
    torch.cuda.synchronize()
    traj_ms = t0e.elapsed_time(t1e) / 20
    system.inference(None, "pose", as_torch=True)
    torch.cuda.synchronize()
    layer_ms, npairs = system.profile_layers(iters=20)
    dom = max((k for k in layer_ms if k.startswith("cnv")), key=lambda k: layer_ms[k])
    # Tensor peak for TF32: MEASURED_PEAKS.json holds bf16 only, so the denominator is the larger of
    # bf16/2 and a cuBLAS TF32 GEMM timed live here (burst, best of 10) -- never the smaller.
    live_tf32 = live_tf32_gemm_tflops(dev)
    peak_tf32 = max(peaks["bf16_tflops"] / 2.0, live_tf32)
    achieved = FLOP_PER_PAIR_LAYER[dom] * npairs / (layer_ms[dom] * 1e-3) / 1e12
    conv_ms = sum(v for k, v in layer_ms.items() if k.startswith("cnv"))
    stack_tflops = FLOP_PER_PAIR * npairs / (conv_ms * 1e-3) / 1e12
    traffic, traffic_src = ncu_traffic(dom)
    if traffic is not None and traffic_src["pairs_per_launch"] not in (None, npairs):
        traffic = traffic * npairs / traffic_src["pairs_per_launch"]      # same kernel, other pass size
    roofline = {
        "bound": "tensor", "kernel": "conv_tc_kernel<%s>" % dom, "achieved": achieved,
        "peak": peak_tf32, "unit": "TFLOP/s", "frac": achieved / peak_tf32, "traffic": traffic,
        "traffic_note": None if traffic is None else
        "dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full capture %s "
        "(tensor pipe active %.1f %%); algorithmic in+out bytes of this launch: %d" % (
            traffic_src["file"], traffic_src["tensor_pipe_pct"] or 0.0,
            npairs * {"cnv4": 851968 + 1703936, "cnv5": 1703936 + 3407872, "cnv6": 2 * 3407872,
                      "cnv7": 3407872}.get(dom, 0)),
        "flop_per_launch": FLOP_PER_PAIR_LAYER[dom] * npairs, "launch_ms": layer_ms[dom],
        "nominal_peak": 1100.0, "frac_nominal": achieved / 1100.0,     # B200 TF32 dense, for context only
        "peak_note": "TF32 dense = max(MEASURED_PEAKS bf16_tflops (burst) / 2 = %.1f %s, live cuBLAS TF32 8192^3 GEMM = %.1f)"
                     % (peaks["bf16_tflops"] / 2.0, peak_kind, live_tf32),
        "pairs_per_launch": npairs, "layer_ms": layer_ms,
        "conv_stack_tflops": stack_tflops, "conv_stack_frac": stack_tflops / peak_tf32,
        "front_end_gbs": FRONT_BYTES_PER_PAIR * npairs / (layer_ms["front"] * 1e-3) / 1e9,
        "front_end_frac_hbm": FRONT_BYTES_PER_PAIR * npairs / (layer_ms["front"] * 1e-3) / 1e9 / peaks["hbm_gbs"],
        "whole_step_tflops": value / world * FLOP_PER_PAIR / 1e12,
        "whole_step_frac": value / world * FLOP_PER_PAIR / 1e12 / peak_tf32,
        # the timed region is a long step under the power cap: beside the burst denominator above, the same number
        # against MEASURED_PEAKS' sustained bf16 figure / 2 (what a long tensor-bound run on this pool's B200s keeps up)
        "whole_step_frac_of_sustained": value / world * FLOP_PER_PAIR / 1e12 / (peaks["bf16_tflops_sustained"] / 2.0)
        if peaks.get("bf16_tflops_sustained") else None,
    }
    # CPU baseline leg = the fp32 oracle on the FIRST 16 SAMPLES OF THE TIMED BATCH; its poses are the parity reference
    rate, cdt, thr, n, ref16 = cpu_oracle_rate(16, 1, min_seconds=12.0, inputs=(img, flow, seg))
    cpu = {"value": rate, "unit": UNIT, "cores": thr, "kind": "port",
           "sample": "%d x the first 16 samples (32 frame pairs) of the timed batch, fp32 torch-CPU oracle "
                     "(restatement of the TF graph, not TF), %.1f s" % (n, cdt)}
    parity = parity_block(ref16, device_resident=timed_out[:16], host_fed=pose_host[:16], host_fed_compact=pose_compact[:16])
    gather_check = None
    if world > 1:
        # what every rank contributed, recomputed by rank 0 alone from that rank's seeded inputs: same kernels, same
        # per-sample reduction order, so the gathered block must be the same BITS
        equal, worst = True, 0.0
        for r in range(world):
            ri = S.make_inputs(B, H, W, seed=1234 + r)
            alone = system.inference(None, "pose", inputs=tuple(torch.as_tensor(x).to(dev) for x in ri))["pose"]
            blk = timed_out[r * B:(r + 1) * B]
            equal = equal and bool(np.array_equal(alone, blk))
            worst = max(worst, float(np.abs(alone.astype(np.float64) - blk).max()))
        gather_check = {"via": "davo_allgather_poses (ncclAllGather on the compute stream, the handle's communicator)",
                        "ranks": world, "shape": list(timed_out.shape), "bit_equal_to_single_gpu": equal,
                        "max_abs_diff": worst, "ok": equal and timed_out.shape[0] == world * B}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "tf32 operands (activations and weights), fp32 accumulate; inputs read as given (uint8 frames, float32 "
                 "flow and labels; flow_f16 off)", "data": "synthetic",
        "config": {"workload": "configs[1]: 256 frame pairs (128 samples) per GPU @128x416, headline variant",
                   "version": VERSION, "samples_per_gpu": B, "frame_pairs_per_step": world * 2 * B,
                   "micro_batch_pairs": npairs,
                   "l2": "inputs (361 MB per step) exceed the 126 MB L2; no flush needed",
                   "parallelism": "sample-sharded x%d, NCCL all-gather of poses" % world},
        "clocks": clocks, "gpu_launches": launches, "parity": parity, "gather_check": gather_check,
        "stream_4541": stream,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "pcie_h2d_gbs": pcie_gbs, "pcie_h2d_gbs_all_ranks": pcie_gbs_sum,
                "copy_only": copy_only_value, "frac_of_copy_only": e2e_value / copy_only_value,
                "one_call_at_a_time": e2e_sync_value,
                "api": "DAVO.inference_async(host arrays).result(): one step in flight behind the one being read "
                       "(davo_forward_host_pairs_async / davo_host_wait); one_call_at_a_time = the blocking "
                       "DAVO.inference(inputs=host arrays) loop, where each step's pipeline fill and drain are exposed",
                "compact_inputs": {"value": compact_value, "unit": UNIT, "h2d_bytes_per_step": compact_h2d,
                                   "note": "NOT the reference's input contract: the caller supplies uint8 labels and "
                                           "binary16 flow planes (davo_forward_host_compact); no CPU pass, fewer bytes"},
                "numa_node": numa_node,
                "host_input_bytes_per_step": world * B * (128 * 416 * (9 + 4 * 2 * 4 + 3 * 4)),
                "note": "host inputs (uint8 frames, float32 flow and labels, as the reference feeds them) enter the "
                        "timed region as numpy arrays; the library copies only the planes the graph reads and, on "
                        "the CPU inside the timed region, narrows the labels to bytes (lossless: the graph casts them "
                        "to int32); the flow crosses as float32 (flow_f16 off), so h2d_bytes_per_step is what crossed "
                        "PCIe.  pcie_h2d_gbs = plain pinned copies of that many bytes issued by ALL ranks at once "
                        "(barrier-released), slowest rank (context: its value depends on which NUMA node the "
                        "probe's buffer landed on); copy_only = the library's own staging + copies with the kernels skipped "
                        "(DAVO_B200_HOST_COPY_ONLY), same ranks, same buffers: the ceiling e2e can reach"},
        "roofline": roofline, "cpu_baseline": cpu,
        "trajectory_mode": {"samples_per_s": B / (traj_ms * 1e-3), "ms_per_step": traj_ms, "frame_pairs_computed": B + 1,
                            "note": "pairs='trajectory_first' (rank 0, device-resident): the same output file as the "
                                    "reference CLI from half the evaluations; not part of `value`"},
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=128, help="samples per GPU per step (2 frame pairs each)")
    ap.add_argument("--micro-batch", type=int, default=0, help="frame pairs per pass of the conv stack")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the poses of the last timed step to DIR/pose.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # started as plain `python bench.py --gpus N`: become the N-rank launch the contract describes
        # (torch.distributed.run, one rank per GPU, rendezvous on 127.0.0.1)
        import socket
        import subprocess
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
