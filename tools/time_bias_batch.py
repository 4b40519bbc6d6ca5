#!/usr/bin/env python3
"""Cost of the bias in the batch seam loop: N distinct 1920x1080 RGB frames (ol.synth_image, seeds 0x1920108 + i)
reduced to 1440 wide (480 vertical seams), with and without a bias plane per frame (signed noise and a preserved
rectangle).  Every shape runs once untimed before it is timed.  For every N it runs, in the same process, REPS
alternations of:
  unbiased  load, then CarverBatch.resize_width(480), device events around the call;
  biased    load and set_bias (untimed: one K1 and one bias-add launch), then resize_width(480), device events around
            the call.  Per seam it launches what the unbiased loop launches; the carve also compacts the bias plane
            (one more float plane per frame and seam) and the band K1 reads it.
python tools/time_bias_batch.py [N ...]   (DCTC_LIB=<path> loads an alternative build)"""
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception:
        return "unknown"


def run(ctx, b, frames, bias):
    b.load(frames)
    if bias is not None:
        b.set_bias(bias)
    ctx.timer_begin()
    b.resize_width(W - NEW_W)
    return ctx.timer_end()


def main():
    ns = [int(a) for a in sys.argv[1:]] or [1, 8, 64]
    gpu = card()
    n_max = max(ns)
    frames = np.stack([ol.synth_image(W, H, 3, 0x1920108 + i, 0).reshape(H, W, 3) for i in range(n_max)])
    rng = np.random.default_rng(0x1920108)
    bias = (rng.standard_normal((n_max, H, W)) * 50.0).astype(np.float32)
    bias[:, 300:700, 800:1100] = 1e6
    ctx = dc.Context(0, blocksize=8, edges=0.5, textures=0.5)
    print("card, power limit: %s" % gpu)
    print("%dx%d RGB -> %d wide, min-max of %d runs each" % (W, H, NEW_W, REPS))
    print("%4s | %17s | %17s | %s" % ("N", "unbiased ms", "biased ms", "biased / unbiased (median)"))
    rows = []
    for n in ns:
        b = dc.CarverBatch(ctx, frames[:n])
        try:
            run(ctx, b, frames[:n], None)                # warm-up of both instantiations
            run(ctx, b, frames[:n], bias[:n])
            mu, mb = [], []
            for _ in range(REPS):
                mu.append(run(ctx, b, frames[:n], None))
                mb.append(run(ctx, b, frames[:n], bias[:n]))
        finally:
            b.close()
        ratio = float(np.median(mb) / np.median(mu))
        rows.append({"n": n, "unbiased_ms": mu, "biased_ms": mb, "ratio_median": ratio})
        print("%4d | %8.1f-%8.1f | %8.1f-%8.1f | %.3f" % (n, min(mu), max(mu), min(mb), max(mb), ratio))
        sys.stdout.flush()
    ctx.close()
    print(json.dumps({"card": gpu, "w": W, "h": H, "new_w": NEW_W, "rows": rows}))


if __name__ == "__main__":
    main()
