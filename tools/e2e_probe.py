import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from davo_b200 import synthetic as S
from davo_b200.davo import DAVO
ver = "v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh"
B = 128
inputs = S.make_inputs(B, 128, 416, seed=3)
pinned = tuple(torch.as_tensor(x).pin_memory().numpy() for x in inputs)
w = S.init_weights(ver)
for chunk in (4, 8, 16, 32, 64):
    os.environ["DAVO_B200_HOST_CHUNK"] = str(chunk)
    sysm = DAVO(version=ver)
    sysm.setup_inference(128, 416, "davo", 3, B, device=0)
    sysm.load_weights(w)
    for _ in range(3):
        sysm.inference(None, "pose", inputs=pinned)
    t0 = time.perf_counter()
    for _ in range(30):
        sysm.inference(None, "pose", inputs=pinned)
    dt = (time.perf_counter() - t0) / 30
    print("chunk %3d samples: %.3f ms per 256 pairs -> %.0f pairs/s" % (chunk, dt * 1e3, 256 / dt), flush=True)
    sysm.close()
os.environ["DAVO_B200_HOST_CHUNK"] = "16"
sysm = DAVO(version=ver)
sysm.setup_inference(128, 416, "davo", 3, B, device=0)
sysm.load_weights(w)
for sel in ("all", "trajectory"):
    for _ in range(3):
        sysm.inference(None, "pose", inputs=pinned, pairs=sel)
    t0 = time.perf_counter()
    for _ in range(30):
        sysm.inference(None, "pose", inputs=pinned, pairs=sel)
    dt = (time.perf_counter() - t0) / 30
    print("pairs=%s: %.3f ms per 128 samples" % (sel, dt * 1e3), flush=True)
# the same bytes as plain copies, no compute: contiguous, and in the library's pattern (per chunk: img, 2 of 4 flow planes, 2 of 3 seg planes)
timg, tflow, tseg = (torch.as_tensor(x) for x in pinned)
dimg = torch.empty_like(timg, device="cuda"); dflow = torch.empty((B, 2) + tuple(tflow.shape[2:]), device="cuda"); dseg = torch.empty((B, 2) + tuple(tseg.shape[2:]), device="cuda")
def pattern():
    for s0 in range(0, B, 16):
        dimg[s0:s0 + 16].copy_(timg[s0:s0 + 16], non_blocking=True)
        dflow[s0:s0 + 16].copy_(tflow[s0:s0 + 16, 0:2], non_blocking=True)
        dseg[s0:s0 + 16, 0].copy_(tseg[s0:s0 + 16, 0], non_blocking=True)
        dseg[s0:s0 + 16, 1].copy_(tseg[s0:s0 + 16, 2], non_blocking=True)
for _ in range(2):
    pattern()
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(20):
    pattern()
torch.cuda.synchronize()
dt = (time.perf_counter() - t0) / 20
nbytes = dimg.numel() + 4 * dflow.numel() + 4 * dseg.numel()
print("copy pattern alone: %.3f ms, %.1f GB/s (%d bytes)" % (dt * 1e3, nbytes / dt / 1e9, nbytes), flush=True)
