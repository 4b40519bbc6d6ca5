#!/usr/bin/env python3
"""Both axes in one batch call: N distinct 1920x1080 RGB frames (ol.synth_image, seeds 0x1920108 + i) resized to
1440x810 (480 vertical seams removed, then 270 horizontal ones) and to 2400x900 (480 vertical seams inserted, then 180
horizontal ones removed).  Every shape runs once untimed before it is timed.  For every N and target it runs, in the same
process, REPS alternations of:
  resize      one CarverBatch.resize(new_w, new_h) over the loaded frames, device events around the call (the width
              pass, the device transpose of the frames it left and their K1, the height pass);
  workaround  what a caller did before: the batch's width call (resize_width or enlarge_width), the images downloaded,
              loaded into a second batch created at the intermediate size (created once, outside the timed region),
              its resize_height; device events around the whole sequence.
The seams and the final images of the two must be equal.
python tools/time_resize_batch.py [N ...]   (DCTC_LIB=<path> loads an alternative build)"""
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

W, H, REPS = 1920, 1080, 3
TARGETS = [(1440, 810), (2400, 900)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception:
        return "unknown"


def run_resize(ctx, b, frames, new_w, new_h):
    b.load(frames)
    ctx.timer_begin()
    passes = b.resize(new_w, new_h)
    ms = ctx.timer_end()
    return ms, [p["seams"] for p in passes], b.images()


def run_workaround(ctx, b, mid, frames, new_w, new_h):
    b.load(frames)
    ctx.timer_begin()
    first = b.enlarge_width(new_w - W) if new_w > W else b.resize_width(W - new_w)
    mid.load(b.images())
    second = mid.resize_height(H - new_h)
    ms = ctx.timer_end()
    return ms, [first, second], mid.images()


def main():
    ns = [int(a) for a in sys.argv[1:]] or [1, 8, 64]
    gpu = card()
    frames = np.stack([ol.synth_image(W, H, 3, 0x1920108 + i, 0).reshape(H, W, 3) for i in range(max(ns))])
    ctx = dc.Context(0, blocksize=8, edges=0.5, textures=0.5)
    print("card, power limit: %s" % gpu)
    print("%dx%d RGB, min-max of %d runs each; workaround / resize > 1 means the combined call is faster" % (W, H, REPS))
    print("%4s %10s | %17s | %17s | %s" % ("N", "target", "resize ms", "workaround ms", "workaround / resize"))
    rows = []
    for n in ns:
        for new_w, new_h in TARGETS:
            for p in dc.resize_plan(W, H, new_w, new_h):
                assert p["n_seams"] == abs((new_w if p["axis"] == "width" else new_h) - (W if p["axis"] == "width" else H))
            b = dc.CarverBatch(ctx, frames[:n])
            mid = dc.CarverBatch(ctx, np.zeros((n, H, new_w, 3), np.uint8))
            try:
                run_resize(ctx, b, frames[:n], new_w, new_h)             # warm-up of every shape
                run_workaround(ctx, b, mid, frames[:n], new_w, new_h)
                mr, mw, same = [], [], True
                for _ in range(REPS):
                    ms, sr, ir = run_resize(ctx, b, frames[:n], new_w, new_h)
                    mr.append(ms)
                    ms, sw, iw = run_workaround(ctx, b, mid, frames[:n], new_w, new_h)
                    mw.append(ms)
                    same = same and all(np.array_equal(x, y) for x, y in zip(sr, sw)) and bool(np.array_equal(ir, iw))
            finally:
                b.close()
                mid.close()
            r = {"n": n, "target": [new_w, new_h], "resize_ms": mr, "workaround_ms": mw, "same": same}
            rows.append(r)
            print("%4d %10s | %8.1f-%8.1f | %8.1f-%8.1f | %.3f-%.3fx%s" % (
                n, "%dx%d" % (new_w, new_h), min(mr), max(mr), min(mw), max(mw), min(mw) / max(mr), max(mw) / min(mr),
                "" if same else "  RESULTS DIFFER"))
            sys.stdout.flush()
    ctx.close()
    print(json.dumps({"card": gpu, "w": W, "h": H, "rows": rows}))


if __name__ == "__main__":
    main()
