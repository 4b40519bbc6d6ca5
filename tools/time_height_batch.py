#!/usr/bin/env python3
"""Batch height retargeting throughput: N distinct 1920x1080 RGB frames (ol.synth_image, seeds 0x2391080 + i) -> 1920x800
(280 horizontal seams each, 16:9 -> 2.39:1).  Every shape runs once untimed before it is timed.  For every N it runs,
in the same process, REPS alternations of:
  height   one CarverBatch.resize_height(280) over the N frames, device events around the call (includes the device
           transpose of the frames and the K1 of the transposed frames);
  twidth   the same frames transposed on the host, loaded into a CarverBatch of 1080x1920 frames, resize_width(280),
           device events around the call: the same seam work without the transpose and without that K1;
and once:
  host     the host carver's vertically path for one frame (host.render(frame, -280, vertically=True, ctx=ctx): host
           transpose, device seam loop, host transpose back), host clock around the call.
The seams of height and twidth must be equal.
python tools/time_height_batch.py [N ...]   (DCTC_LIB=<path> loads an alternative build)"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import dct_carver_b200 as dc  # noqa: E402
if os.environ.get("DCTC_LIB"):
    dc.LIB_PATH = os.environ["DCTC_LIB"]
import oracle_lib as ol  # noqa: E402  (synthetic image generator only)

W, H, K, REPS = 1920, 1080, 280, 3


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception:
        return "unknown"


def timed(ctx, batch, frames, call):
    batch.load(frames)
    ctx.timer_begin()
    seams = call(K)
    return ctx.timer_end(), seams


def main():
    ns = [int(a) for a in sys.argv[1:]] or [1, 8, 64]
    gpu = card()
    frames = np.stack([ol.synth_image(W, H, 3, 0x2391080 + i, 0) for i in range(max(ns))])
    tframes = np.ascontiguousarray(np.swapaxes(frames, 1, 2))
    ctx = dc.Context(0, blocksize=8, edges=0.5, textures=0.5)
    print("card, power limit: %s" % gpu)
    print("%dx%d RGB -> %dx%d, %d seams per frame, all timed; frame-seams/s = N * %d / time; min-max of %d runs"
          % (W, H, W, H - K, K, K, REPS))
    print("%4s | %17s %19s | %17s %19s | %s" % ("N", "height ms", "height fs/s", "twidth ms", "twidth fs/s", "height / twidth"))
    rows = []
    for n in ns:
        bh = dc.CarverBatch(ctx, frames[:n])
        bw = dc.CarverBatch(ctx, tframes[:n])
        try:
            bh.resize_height(K)             # warm-up of both batch shapes
            bw.resize_width(K)
            mh, mw = [], []
            same = True
            for _ in range(REPS):
                ms, sh = timed(ctx, bh, frames[:n], bh.resize_height)
                mh.append(ms)
                ms, sw = timed(ctx, bw, tframes[:n], bw.resize_width)
                mw.append(ms)
                same = same and bool(np.array_equal(sh, sw))
        finally:
            bh.close()
            bw.close()
        rate = lambda m: n * K / (m * 1e-3)  # noqa: E731
        r = {"n": n, "height_ms": mh, "twidth_ms": mw, "height_frame_seams_per_s": [rate(m) for m in mh],
             "twidth_frame_seams_per_s": [rate(m) for m in mw], "same_seams": same}
        rows.append(r)
        print("%4d | %8.1f-%8.1f %9.0f-%9.0f | %8.1f-%8.1f %9.0f-%9.0f | %.3f-%.3fx%s" % (
            n, min(mh), max(mh), rate(max(mh)), rate(min(mh)), min(mw), max(mw), rate(max(mw)), rate(min(mw)),
            min(mw) / max(mh), max(mw) / min(mh), "" if same else "  SEAMS DIFFER"))
        sys.stdout.flush()
    from dct_carver_b200 import host
    host.render(frames[0], -K, 8, 0.5, 0.5, vertically=True, ctx=ctx)   # warm-up
    t0 = time.perf_counter()
    got = host.render(frames[0], -K, 8, 0.5, 0.5, vertically=True, ctx=ctx)
    host_ms = 1e3 * (time.perf_counter() - t0)
    b1 = dc.CarverBatch(ctx, frames[:1])
    try:
        host_same = bool(np.array_equal(got["seams"], b1.resize_height(K)[0]))
    finally:
        b1.close()
    print("host carver, vertically, one frame: %.1f ms (%.0f frame-seams/s), seams %s the batch's" % (
        host_ms, K / (host_ms * 1e-3), "equal to" if host_same else "DIFFERENT FROM"))
    ctx.close()
    print(json.dumps({"card": gpu, "w": W, "h": H, "seams": K, "rows": rows, "host_ms": host_ms, "host_same_seams": host_same}))


if __name__ == "__main__":
    main()
