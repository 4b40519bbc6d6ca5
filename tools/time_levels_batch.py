#!/usr/bin/env python3
"""Interactive resizing of a batch: N distinct 1920x1080 RGB frames (ol.synth_image, seeds 0x1920108 + i), one levels
build to depth 480, then renders of 16 widths, against what a caller needs without levels for the same 16 widths.
  build     CarverBatch.levels_width(480) after a load, device events around the call;
  shrink    render_levels_dev of 1440, 1472, ..., 1920 (16 widths <= the start width: one gather launch), REPS runs;
  enlarge   render_levels_dev of 1950, 1980, ..., 2400 (16 widths > the start width: one inflate launch each), REPS runs;
  today     per width, a batch load plus resize_width(1920 - e) or enlarge_width(e - 1920), device events around each
            pair, summed over the 16 widths (one run).
Every width of "today" is compared with its rendered level.  The render's GB/s count the algorithmic bytes of one call:
the gather reads every frame's map (4 bytes a pixel) and image (3 bytes a pixel) once and writes every level's rows; each
inflate launch reads map and image once more for its level.  The working set of N >= 8 is larger than the L2.
python tools/time_levels_batch.py [N ...]   (DCTC_LIB=<path> loads an alternative build)"""
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

W, H, CH, DEPTH, REPS = 1920, 1080, 3, 480, 5
SHRINK = [1440 + 32 * i for i in range(16)]
ENLARGE = [1920 + 30 * (i + 1) for i in range(16)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception:
        return "unknown"


def render_bytes(n, extents):
    """Algorithmic bytes of one render call: one gather over every shrink level, one inflate per enlarge level."""
    src = n * H * W * (4 + CH)
    reads = (src if any(e <= W for e in extents) else 0) + src * sum(e > W for e in extents)
    return reads + n * H * CH * sum(extents)


def timed_render(ctx, b, extents, d_out):
    b.render_levels_dev(extents, d_out)   # warm-up of the shape
    ms = []
    for _ in range(REPS):
        ctx.timer_begin()
        b.render_levels_dev(extents, d_out)
        ms.append(ctx.timer_end())
    return ms


def today(ctx, b, frames, extents, d_out):
    """Load + resize / enlarge per width; each result compared with the rendered level at the same index."""
    n = frames.shape[0]
    total, same, off = 0.0, True, 0
    for e in extents:
        b.load(frames)
        ctx.timer_begin()
        if e <= W:
            b.resize_width(W - e)
        else:
            b.enlarge_width(e - W)
        total += ctx.timer_end()
        got = np.empty((n, H, e, CH), np.uint8)
        ctx.d2h(got, d_out + off)
        same = same and bool(np.array_equal(got, b.images()))
        off += got.nbytes
    return total, same


def main():
    ns = [int(a) for a in sys.argv[1:]] or [1, 8, 64]
    gpu = card()
    frames_all = np.stack([ol.synth_image(W, H, CH, 0x1920108 + i, 0).reshape(H, W, CH) for i in range(max(ns))])
    ctx = dc.Context(0, blocksize=8, edges=0.5, textures=0.5)
    print("card, power limit: %s" % gpu)
    print("%dx%d RGB, build to depth %d, 16 widths per render; min-max of %d render runs" % (W, H, DEPTH, REPS))
    rows = []
    for n in ns:
        frames = frames_all[:n]
        b = dc.CarverBatch(ctx, frames)
        d_out = ctx.dev_alloc(n * H * CH * max(sum(SHRINK), sum(ENLARGE)))
        try:
            b.levels_width(DEPTH)               # warm-up of the build
            b.load(frames)
            ctx.timer_begin()
            b.levels_width(DEPTH)
            build_ms = ctx.timer_end()
            r = {"n": n, "build_ms": build_ms}
            for name, ext in (("shrink", SHRINK), ("enlarge", ENLARGE)):
                ms = timed_render(ctx, b, ext, d_out)
                nbytes = render_bytes(n, ext)
                r[name] = {"render_ms": ms, "bytes": nbytes, "gbs": nbytes / (min(ms) * 1e-3) / 1e9}
            # today's way; the rendered levels are compared level by level (the batch is reloaded, so render first)
            for name, ext in (("shrink", SHRINK), ("enlarge", ENLARGE)):
                b.load(frames)
                b.levels_width(DEPTH)
                b.render_levels_dev(ext, d_out)
                ms, same = today(ctx, b, frames, ext, d_out)
                r[name]["today_ms"] = ms
                r[name]["same"] = same
        finally:
            ctx.dev_free(d_out)
            b.close()
        rows.append(r)
        print("N %3d  build %8.1f ms" % (n, build_ms))
        for name in ("shrink", "enlarge"):
            x = r[name]
            print("       %-7s render %7.3f-%7.3f ms (%6.0f GB/s)  today %9.1f ms  today / (build + render) %6.2fx%s" % (
                name, min(x["render_ms"]), max(x["render_ms"]), x["gbs"], x["today_ms"],
                x["today_ms"] / (build_ms + min(x["render_ms"])), "" if x["same"] else "  RESULTS DIFFER"))
        sys.stdout.flush()
    ctx.close()
    print(json.dumps({"card": gpu, "w": W, "h": H, "depth": DEPTH, "rows": rows}))


if __name__ == "__main__":
    main()
