#!/usr/bin/env python3
"""Batch enlarge throughput: N distinct 1440x1080 RGB frames (ol.synth_image, seeds 0xE41A26E0 + i) enlarged to 1920
(480 seams each, 4:3 -> 16:9).  Every shape is enlarged once untimed before it is timed.  For every N it runs, in the
same process:
  batch    one CarverBatch.enlarge_width(480) over the N frames, device events around the call;
  shrink   one CarverBatch.resize_width(480) of the same frames, device events around the call (enlarge - shrink is the
           cost of the start-frame copy, the visibility maps, the inflate kernel and the enlarged frames' energy maps);
  single   one single-frame session on one context, carver_enlarge_width(480) of the N frames one after another (device
           events per frame, summed);
  threads  N contexts driven from N host threads at once (ctypes releases the GIL), host clock from a barrier to the
           last thread's return (each enlarge ends in a stream synchronise).
python tools/time_enlarge_batch.py [N ...]   (DCTC_LIB=<path> loads an alternative build)"""
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import dct_carver_b200 as dc  # noqa: E402
if os.environ.get("DCTC_LIB"):
    dc.LIB_PATH = os.environ["DCTC_LIB"]
import oracle_lib as ol  # noqa: E402  (synthetic image generator only)

W, H, K = 1440, 1080, 480


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception:
        return "unknown"


def time_batch(ctx, frames):
    """(enlarge ms, shrink ms, enlarge seams, shrink seams) of one batch over the frames."""
    b = dc.CarverBatch(ctx, frames)
    try:
        b.enlarge_width(K)                  # warm-up of this batch shape (the shrink runs the same seam loop)
        b.load(frames)
        ctx.timer_begin()
        grow = b.enlarge_width(K)
        ms_grow = ctx.timer_end()
        b.load(frames)
        ctx.timer_begin()
        shrink = b.resize_width(K)
        ms_shrink = ctx.timer_end()
    finally:
        b.close()
    return ms_grow, ms_shrink, grow, shrink


def time_single(ctx, frames):
    ms, seams = 0.0, []
    for f in frames:
        ctx.carver_load(f)
        ctx.timer_begin()
        seams.append(ctx.carver_enlarge_width(K))
        ms += ctx.timer_end()
    return ms, np.stack(seams)


def time_threads(frames):
    n = len(frames)
    ctxs = [dc.Context(0, blocksize=8, edges=0.5, textures=0.5) for _ in range(n)]
    try:
        for c, f in zip(ctxs, frames):
            c.carver_load(f)
            c.carver_enlarge_width(K)       # warm-up of every context at the timed shape
            c.carver_load(f)
        go = threading.Barrier(n + 1)
        out = [None] * n

        def work(i):
            go.wait()
            out[i] = ctxs[i].carver_enlarge_width(K)

        ts = [threading.Thread(target=work, args=(i,)) for i in range(n)]
        for t in ts:
            t.start()
        go.wait()
        t0 = time.perf_counter()
        for t in ts:
            t.join()
        ms = 1e3 * (time.perf_counter() - t0)
    finally:
        for c in ctxs:
            c.close()
    return ms, np.stack(out)


def main():
    ns = [int(a) for a in sys.argv[1:]] or [1, 2, 4, 8, 16, 32, 64]
    gpu = card()
    frames = np.stack([ol.synth_image(W, H, 3, 0xE41A26E0 + i, 0) for i in range(max(ns))])
    ctx = dc.Context(0, blocksize=8, edges=0.5, textures=0.5)
    ctx.carver_load(frames[0])              # warm-up of the single session at the timed shape
    ctx.carver_enlarge_width(K)
    print("card, power limit: %s" % gpu)
    print("%dx%d RGB -> %dx%d, %d seams per frame, all timed; frame-seams/s = N * %d / time" % (W, H, W + K, H, K, K))
    print("%4s | %12s %12s | %12s %12s | %12s | %12s | %s" % ("N", "batch ms", "batch fs/s", "shrink ms", "shrink fs/s",
                                                             "single fs/s", "threads fs/s", "batch / single, batch / threads"))
    rows = []
    for n in ns:
        fr = frames[:n]
        mg, mk, sg, sk = time_batch(ctx, fr)
        ms, ss = time_single(ctx, fr)
        mt, st = time_threads(fr)
        same = bool(np.array_equal(sg, ss) and np.array_equal(sg, st) and np.array_equal(sg, sk))
        rate = lambda m: n * K / (m * 1e-3)  # noqa: E731
        r = {"n": n, "batch_ms": mg, "batch_frame_seams_per_s": rate(mg), "shrink_ms": mk,
             "shrink_frame_seams_per_s": rate(mk), "single_ms": ms, "single_frame_seams_per_s": rate(ms),
             "threads_ms": mt, "threads_frame_seams_per_s": rate(mt), "same_seams": same}
        rows.append(r)
        print("%4d | %12.1f %12.0f | %12.1f %12.0f | %12.0f | %12.0f | %.2fx, %.2fx%s" % (
            n, mg, r["batch_frame_seams_per_s"], mk, r["shrink_frame_seams_per_s"], r["single_frame_seams_per_s"],
            r["threads_frame_seams_per_s"], r["batch_frame_seams_per_s"] / r["single_frame_seams_per_s"],
            r["batch_frame_seams_per_s"] / r["threads_frame_seams_per_s"], "" if same else "  SEAMS DIFFER"))
        sys.stdout.flush()
    ctx.close()
    print(json.dumps({"card": gpu, "w": W, "h": H, "seams": K, "rows": rows}))


if __name__ == "__main__":
    main()
