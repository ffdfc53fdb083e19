"""Bring-up check of the CTA-pair (cta_group::2) path of conv_tc_kernel: every eligible case of tests/test_conv_gpu.py and
the res4 / FPN shapes of the detector, computed with B2_PAIR on and off in one process -- the two paths do the same
arithmetic in the same order, so the outputs must be bit-identical.  On a mismatch prints which 128-row x 64-column blocks
differ (a swapped B half or m-block shows as a pattern).
Usage: python tools/pair_check.py [min_kb]      exit code 0 = all identical"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from object_detection_tracking_b200 import engine   # noqa: E402
from test_conv_gpu import CASES, reference   # noqa: E402

EXTRA = {
    "res4_3x3_b2":   (2, 46, 80, 256, 256, 3, 1, 1, (1, 1, 1, 1), 1, 1, 0, 0),     # 58 m-blocks (even), 2 n-blocks, 36 K-blocks
    "res4_1x1_k1024": (1, 46, 80, 1024, 256, 1, 1, 1, (0, 0, 0, 0), 1, 1, 0, 0),   # 29 m-blocks (odd), 16 K-blocks
    "odd_3x3":       (1, 25, 37, 128, 256, 3, 1, 1, (1, 1, 1, 1), 1, 1, 1, 0),     # 8 m-blocks, ragged, residual
}


def run(spec, x, w, bias, res, pair):
    os.environ.pop("B2_PAIR", None)
    if pair:
        os.environ["B2_PAIR"] = str(pair)
    try:
        return engine.op_conv2d(x, w, bias, res, stride=spec[6], dil=spec[7], pad=spec[8], relu=bool(spec[10]),
                                res_shift=spec[12], impl="tcgen05", split=True)
    finally:
        os.environ.pop("B2_PAIR", None)


def block_map(a, b):
    m = a.reshape(-1, a.shape[-1]) != b.reshape(-1, b.shape[-1])
    rows, cols = m.shape
    lines = []
    for r0 in range(0, rows, 128):
        lines.append("".join("x" if m[r0:r0 + 128, c0:c0 + 64].any() else "." for c0 in range(0, cols, 64)))
    return lines


def main():
    min_kb = int(sys.argv[1]) if len(sys.argv) > 1 else 1
    bad = 0
    cases = dict(CASES)
    cases.update(EXTRA)
    for name in sorted(cases):
        spec = cases[name]
        x, w, bias, res, ref = reference(spec, seed=len(name))
        base = run(spec, x, w, bias, res, 0)
        try:
            got = run(spec, x, w, bias, res, min_kb)
        except Exception as e:   # the diag build reports a timed-out wait through the error string
            print("%-20s PAIR FAILED: %s" % (name, e), flush=True)
            bad += 1
            break
        same = np.array_equal(base, got)
        err = np.abs(got - ref).max() / np.abs(ref).max()
        print("%-20s %s  rel err vs torch %.2e  (base %.2e)" % (name, "identical" if same else "DIFFERENT", err,
                                                                  np.abs(base - ref).max() / np.abs(ref).max()), flush=True)
        if not same:
            bad += 1
            bm = block_map(base, got)
            print("   blocks (rows of 128 down, columns of 64 across; first 12 rows): ")
            for ln in bm[:12]:
                print("   " + ln)
            d = np.abs(got.astype(np.float64) - base)
            print("   max |diff| %.3e at %s, finite %s" % (d.max(), np.unravel_index(d.argmax(), d.shape), np.isfinite(got).all()),
                  flush=True)
    print("pair_check: %s" % ("ALL IDENTICAL" if bad == 0 else "%d case(s) differ / failed" % bad))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
