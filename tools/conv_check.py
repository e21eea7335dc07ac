"""The per-element conv-stage check of tests/test_conv_stages.py over more frame sizes, batches and fuzzed version
strings (tests/golden/fuzz_versions.py).  One line per (configuration, layer): the largest |error| / bound (must stay
<= 1) and the summed offset in TF32 ulps (must stay within +-0.125).  A change to a conv kernel plan should leave
the ratios where profiles/conv_check.log has them.

    python tools/conv_check.py [--fuzz 12] [--seed 5]
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from davo_b200 import version as V  # noqa: E402
from tests import test_conv_stages as T  # noqa: E402
from tests.golden import fuzz_versions  # noqa: E402

SIZES = [(64, 208, 1), (96, 320, 3), (128, 416, 4), (136, 424, 2), (256, 832, 1)]


def fuzz_strings(n, seed):
    rng, out = np.random.default_rng(seed), []
    while len(out) < n:
        ver = fuzz_versions.draw(rng)
        try:
            V.parse_version(ver)
        except Exception:  # noqa: BLE001  (strings the reference cannot build either)
            continue
        if ver not in out:
            out.append(ver)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fuzz", type=int, default=12, help="fuzzed version strings (64x208, batch 2)")
    ap.add_argument("--seed", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "conv_check needs a CUDA device"
    configs = {"size_%dx%d_b%d" % s: (T.HEADLINE,) + s + ({},) for s in SIZES}
    configs.update(("fuzz_%02d %s" % (i, v), (v, 64, 208, 2, {})) for i, v in enumerate(fuzz_strings(args.fuzz, args.seed)))
    configs.update(T.CONFIGS)
    worst, failures = 0.0, 0
    for name, cfg in configs.items():
        T.CONFIGS[name] = cfg
        try:
            res = T._run_config(name)
        except AssertionError as e:
            print("%-40s FAILS %s" % (name, str(e).splitlines()[0][:200]), flush=True)
            failures += 1
            continue
        if res["error"] is not None:
            print("%-40s refused: %s" % (name, res["error"]), flush=True)
            continue
        for lname, st in res["stats"].items():
            bad = st.ratio > 1.0 or abs(st.offset) > T.OFFSET_BAR
            failures += bad
            worst = max(worst, st.ratio)
            print("%-40s %-5s ratio %.4f  offset %+.4f ulp  %s%s" % (name, lname, st.ratio, st.offset, T._branch(res["plans"][lname]),
                                                                     "   <-- FAILS" if bad else ""), flush=True)
    print("worst ratio %.4f, %d failure(s)" % (worst, failures))
    return 1 if failures else 0


if __name__ == "__main__":
    sys.exit(main())
