#!/usr/bin/env python3
"""Cost of the seam step width in the batch seam loop: N distinct 1920x1080 RGB frames (ol.synth_image, seeds
0x1920108 + i) reduced to 1440 wide (480 vertical seams) with delta_x = 1, 2 and 4, rigidity 0.  Every shape and step
width runs once untimed before it is timed.  For every N it runs, in the same process, REPS alternations of: for each
delta_x, load (untimed), then CarverBatch.resize_width(480), device events around the call.  Every delta_x launches
per seam the seam DP, jump and trace kernels (at this size every step width takes the parallel back-track), with the
step rule of delta_x = 1 or the step table of delta_x > 1.
Reports the time per batch seam and the ratio to delta_x = 1.
python tools/time_delta_x_batch.py [N ...]   (DCTC_LIB=<path> loads an alternative build)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import dct_carver_b200 as dc  # noqa: E402
if os.environ.get("DCTC_LIB"):
    dc.LIB_PATH = os.environ["DCTC_LIB"]
import oracle_lib as ol  # noqa: E402  (synthetic image generator only)

W, H, NEW_W, REPS = 1920, 1080, 1440, 3
SEAMS = W - NEW_W
DXS = (1, 2, 4)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception:
        return "unknown"


def run(ctx, b, frames, dx):
    b.set_delta_x(dx)
    b.load(frames)
    ctx.timer_begin()
    b.resize_width(SEAMS)
    return ctx.timer_end()


def main():
    ns = [int(a) for a in sys.argv[1:]] or [1, 8, 64]
    gpu = card()
    n_max = max(ns)
    frames = np.stack([ol.synth_image(W, H, 3, 0x1920108 + i, 0).reshape(H, W, 3) for i in range(n_max)])
    ctx = dc.Context(0, blocksize=8, edges=0.5, textures=0.5)
    print("card, power limit: %s" % gpu)
    print("%dx%d RGB -> %d wide, rigidity 0, min-max of %d runs each" % (W, H, NEW_W, REPS))
    print("%4s | %s" % ("N", " | ".join("dx %d ms (us/seam)" % d for d in DXS)) + " | ratios to dx 1 (median)")
    rows = []
    for n in ns:
        b = dc.CarverBatch(ctx, frames[:n])
        try:
            for dx in DXS:                                 # warm-up of every kernel
                run(ctx, b, frames[:n], dx)
            ms = {dx: [] for dx in DXS}
            for _ in range(REPS):
                for dx in DXS:
                    ms[dx].append(run(ctx, b, frames[:n], dx))
        finally:
            b.close()
        med = {dx: float(np.median(ms[dx])) for dx in DXS}
        row = {"n": n, "ms": {str(dx): ms[dx] for dx in DXS},
               "us_per_seam": {str(dx): 1e3 * med[dx] / SEAMS for dx in DXS},
               "ratio_to_dx1": {str(dx): med[dx] / med[1] for dx in DXS}}
        rows.append(row)
        print("%4d | %s | %s" % (n, " | ".join("%7.1f-%7.1f (%6.1f)" % (min(ms[dx]), max(ms[dx]), 1e3 * med[dx] / SEAMS)
                                               for dx in DXS),
                                 ", ".join("%.2f" % (med[dx] / med[1]) for dx in DXS)))
        sys.stdout.flush()
    ctx.close()
    print(json.dumps({"card": gpu, "w": W, "h": H, "new_w": NEW_W, "rows": rows}))


if __name__ == "__main__":
    main()
