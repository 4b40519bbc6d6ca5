#!/usr/bin/env python3
"""Batch retarget throughput: N distinct 1920x1080 RGB frames (ol.synth_image, seeds 0xD0C7CA14 + i), 480 seams each;
the first 240 warm up, the next 240 are timed.  For every N it runs, in the same process:
  batch    one CarverBatch over the N frames (one launch per phase for all frames), device events around its resize;
  single   one single-frame session on one context, the N frames one after another (device events per frame, summed);
  threads  N contexts driven from N host threads at once (ctypes releases the GIL), host clock from a barrier to the
           last thread's return (each resize ends in a stream synchronise).
python tools/time_seamloop_batch.py [N ...]   (DCTC_LIB=<path> loads an alternative build)"""
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

W, H, WARM, TIMED = 1920, 1080, 240, 240


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception:
        return "unknown"


def warm_up(ctx):
    # as tools/time_seamloop.py: one small session loads every kernel of the loop
    img = ol.synth_image(256, 256, 3, 0xD0C7CA14, 0)
    ctx.carver_load(img)
    ctx.carver_resize_width(8)


def time_batch(ctx, frames):
    b = dc.CarverBatch(ctx, frames)
    try:
        first = b.resize_width(WARM)
        ctx.timer_begin()
        second = b.resize_width(TIMED)
        ms = ctx.timer_end()
    finally:
        b.close()
    return ms, np.concatenate([first, second], axis=1)


def time_single(ctx, frames):
    ms, seams = 0.0, []
    for f in frames:
        ctx.carver_load(f)
        first = ctx.carver_resize_width(WARM)
        ctx.timer_begin()
        second = ctx.carver_resize_width(TIMED)
        ms += ctx.timer_end()
        seams.append(np.concatenate([first, second]))
    return ms, np.stack(seams)


def time_threads(frames):
    n = len(frames)
    ctxs = [dc.Context(0, blocksize=8, edges=0.5, textures=0.5) for _ in range(n)]
    try:
        for c, f in zip(ctxs, frames):
            warm_up(c)
            c.carver_load(f)
        go = threading.Barrier(n + 1)
        out = [None] * n

        def work(i):
            first = ctxs[i].carver_resize_width(WARM)
            go.wait()
            second = ctxs[i].carver_resize_width(TIMED)
            out[i] = np.concatenate([first, second])

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
    frames = np.stack([ol.synth_image(W, H, 3, 0xD0C7CA14 + i, 0) for i in range(max(ns))])
    ctx = dc.Context(0, blocksize=8, edges=0.5, textures=0.5)
    warm_up(ctx)
    print("card, power limit: %s" % gpu)
    print("%dx%d RGB, seams %d..%d of %d timed; frame-seams/s = N * %d / time" % (W, H, WARM + 1, WARM + TIMED, WARM + TIMED, TIMED))
    print("%4s | %14s %14s | %14s %14s | %14s %14s | %s" % ("N", "batch us/seam", "batch fs/s", "single us/seam", "single fs/s",
                                                            "threads us/seam", "threads fs/s", "batch / single, batch / threads"))
    rows = []
    for n in ns:
        fr = frames[:n]
        mb, sb = time_batch(ctx, fr)
        ms, ss = time_single(ctx, fr)
        mt, st = time_threads(fr)
        same = bool(np.array_equal(sb, ss) and np.array_equal(sb, st))
        rate = lambda m: n * TIMED / (m * 1e-3)  # noqa: E731
        r = {"n": n, "batch_us_per_seam": 1e3 * mb / TIMED, "batch_frame_seams_per_s": rate(mb),
             "single_us_per_seam": 1e3 * ms / TIMED, "single_frame_seams_per_s": rate(ms),
             "threads_us_per_seam": 1e3 * mt / TIMED, "threads_frame_seams_per_s": rate(mt), "same_seams": same}
        rows.append(r)
        print("%4d | %14.1f %14.0f | %14.1f %14.0f | %14.1f %14.0f | %.2fx, %.2fx%s" % (
            n, r["batch_us_per_seam"], r["batch_frame_seams_per_s"], r["single_us_per_seam"], r["single_frame_seams_per_s"],
            r["threads_us_per_seam"], r["threads_frame_seams_per_s"], r["batch_frame_seams_per_s"] / r["single_frame_seams_per_s"],
            r["batch_frame_seams_per_s"] / r["threads_frame_seams_per_s"], "" if same else "  SEAMS DIFFER"))
        sys.stdout.flush()
    ctx.close()
    print(json.dumps({"card": gpu, "w": W, "h": H, "timed_seams": TIMED, "rows": rows}))


if __name__ == "__main__":
    main()
