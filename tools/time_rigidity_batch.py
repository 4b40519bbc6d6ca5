#!/usr/bin/env python3
"""Cost of the rigidity in the batch seam loop: N distinct 1920x1080 RGB frames (ol.synth_image, seeds 0x1920108 + i)
reduced to 1440 wide (480 vertical seams), rigid against rigidity 0.  The rigidity gives pen = rigidity / 1080 = the
mean operator energy of frame 0, so that the seams really change.  Every shape runs once untimed before it is timed.
For every N it runs, in the same process, REPS alternations of:
  plain  load (untimed), then CarverBatch.resize_width(480) with rigidity 0, device events around the call;
  rigid  load (untimed), then resize_width(480) with the rigidity, device events around the call.  It launches per seam
         what the plain loop launches: the RIG instantiations of the seam DP, jump and trace kernels.
Reports the time per batch seam and the frame-seams per second.
python tools/time_rigidity_batch.py [N ...]   (DCTC_LIB=<path> loads an alternative build)"""
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception:
        return "unknown"


def run(ctx, b, frames, rigidity):
    b.set_rigidity(rigidity)
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
    ctx.carver_load(frames[0])
    rigidity = float(np.float32(float(np.mean(ctx.carver_energy())) * H))
    print("card, power limit: %s" % gpu)
    print("%dx%d RGB -> %d wide, rigidity %.4g (pen %.4g), min-max of %d runs each" % (W, H, NEW_W, rigidity, rigidity / H, REPS))
    print("%4s | %17s | %17s | %13s | %13s | %s" % ("N", "plain ms", "rigid ms", "plain us/seam", "rigid us/seam",
                                                     "rigid / plain (median); frame-seams/s plain, rigid"))
    rows = []
    for n in ns:
        b = dc.CarverBatch(ctx, frames[:n])
        try:
            run(ctx, b, frames[:n], 0.0)                 # warm-up of both instantiations
            run(ctx, b, frames[:n], rigidity)
            mp, mr = [], []
            for _ in range(REPS):
                mp.append(run(ctx, b, frames[:n], 0.0))
                mr.append(run(ctx, b, frames[:n], rigidity))
        finally:
            b.close()
        p, r = float(np.median(mp)), float(np.median(mr))
        row = {"n": n, "plain_ms": mp, "rigid_ms": mr, "ratio_median": r / p,
               "plain_us_per_seam": 1e3 * p / SEAMS, "rigid_us_per_seam": 1e3 * r / SEAMS,
               "plain_frame_seams_per_s": n * SEAMS / (p * 1e-3), "rigid_frame_seams_per_s": n * SEAMS / (r * 1e-3)}
        rows.append(row)
        print("%4d | %8.1f-%8.1f | %8.1f-%8.1f | %13.1f | %13.1f | %.3f; %.0f, %.0f" % (
            n, min(mp), max(mp), min(mr), max(mr), row["plain_us_per_seam"], row["rigid_us_per_seam"], r / p,
            row["plain_frame_seams_per_s"], row["rigid_frame_seams_per_s"]))
        sys.stdout.flush()
    ctx.close()
    print(json.dumps({"card": gpu, "w": W, "h": H, "new_w": NEW_W, "rigidity": rigidity, "rows": rows}))


if __name__ == "__main__":
    main()
