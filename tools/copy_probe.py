import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from davo_b200 import synthetic as S
from davo_b200.davo import DAVO
ver = "v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh"
B = 128
inputs = S.make_inputs(B, 128, 416, seed=3)
pinned = tuple(torch.as_tensor(x).pin_memory().numpy() for x in inputs)
sysm = DAVO(version=ver)
sysm.setup_inference(128, 416, "davo", 3, B, device=0)
sysm.load_weights(S.init_weights(ver))
for _ in range(3):
    sysm.inference(None, "pose", inputs=pinned)
t0 = time.perf_counter()
for _ in range(30):
    sysm.inference(None, "pose", inputs=pinned)
dt = (time.perf_counter() - t0) / 30
h2d, _ = sysm.last_host_copy_bytes()
print("copy_only=%s: %.3f ms per 128 samples, %d bytes host->device (%.1f GB/s)" % (os.environ.get("DAVO_B200_HOST_COPY_ONLY"), dt * 1e3, h2d, h2d / dt / 1e9))
