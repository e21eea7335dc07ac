import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from davo_b200 import synthetic as S
from davo_b200.davo import DAVO
from oracle import davo_oracle as O
ver = "v1-decay100k-sharedNN-dilatedPoseNN-cnv6_128-segmask_all-se_flow-abs_flow-fc_tanh"
for (H, W, B) in [(256, 832, 2), (64, 208, 3), (128, 400, 2), (136, 424, 1)]:
    w = S.init_weights(ver, random_bias=True)
    inputs = S.make_inputs(B, H, W, seed=11, bad_label_frac=0.01)
    ref = O.davo_forward(ver, *inputs, w, torch.float64)
    try:
        sysm = DAVO(version=ver)
        d = [torch.as_tensor(x).cuda() for x in inputs]
        sysm.setup_inference(H, W, "davo", 3, B, d[0], input_flow=d[1], input_seglabel=d[2], device=0)
        sysm.load_weights(w)
        out = sysm.inference(None, "pose")["pose"]
        print(H, W, B, "max err %.3e" % np.abs(out - ref).max(), "max |ref| %.3e" % np.abs(ref).max(), flush=True)
    except Exception as e:
        print(H, W, B, "FAILED", repr(e)[:300], flush=True)
