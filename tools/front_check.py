"""The per-element front-end and head check of tests/test_front_stages.py over more frame sizes, batches and fuzzed
version strings (tests/golden/fuzz_versions.py).  One line per (configuration, stage): the largest |error| / bound
(must stay <= 1), the summed offset in TF32 ulps (within +-0.125) and the bit-exact elements with their mismatches
(must be 0).  A change to a front-end kernel or the head should leave the ratios where profiles/front_check.log has
them.

    python tools/front_check.py [--fuzz 12] [--seed 7]
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from davo_b200 import version as V  # noqa: E402
from tests import test_front_stages as T  # noqa: E402
from tests.golden import fuzz_versions  # noqa: E402

SIZES = [(64, 208, 1), (96, 320, 3), (128, 416, 4), (136, 424, 2), (136, 200, 5), (256, 832, 1), (32, 64, 6)]
SIZED = {"spp864": T.CONFIGS["spp864_flow_72"][0], "pix_mix_depthflow": T.CONFIGS["pix_mix_depthflow"][0],
         "decouple_net": T.CONFIGS["decouple_net"][0], "gp2x2_seg": T.CONFIGS["gp2x2_seg"][0]}


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
    ap.add_argument("--seed", type=int, default=7)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "front_check needs a CUDA device"
    configs = {"size_%dx%d_b%d" % s: (T.HEADLINE,) + s + ({}, {}) for s in SIZES}
    configs.update(("%s_%dx%d_b%d" % ((k,) + s), (v,) + s + ({}, {})) for k, v in SIZED.items() for s in SIZES[1:4]
                   if s[0] <= s[1])
    configs.update(("fuzz_%02d %s" % (i, v), (v, 64, 208, 2, {}, {})) for i, v in enumerate(fuzz_strings(args.fuzz, args.seed)))
    configs.update(T.CONFIGS)
    worst, failures = 0.0, 0
    for name, cfg in configs.items():
        T.CONFIGS[name] = cfg
        try:
            res = T._run_config(name)
        except (AssertionError, RuntimeError) as e:
            print("%-44s FAILS %s" % (name, str(e).splitlines()[0][:200]), flush=True)
            failures += 1
            continue
        bad = T._bad(res)
        failures += bool(bad)
        for s in T.STAGES:
            st = res["stats"][s]
            if not st["n"]:
                continue
            worst = max(worst, st["ratio"])
            print("%-44s %-6s ratio %.4f  offset %+.4f ulp  exact %d / %d, %d mismatch(es)%s"
                  % (name, s, st["ratio"], st["offset"], st["exact"], st["n"], st["mismatch"], "   <-- FAILS" if bad else ""),
                  flush=True)
        for b in bad:
            print("    " + b[:300], flush=True)
    print("worst ratio %.4f, %d failing configuration(s)" % (worst, failures))
    return 1 if failures else 0


if __name__ == "__main__":
    sys.exit(main())
