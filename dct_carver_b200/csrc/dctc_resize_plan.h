// Pass plan of lqr_carver_resize(new_w, new_h): the one definition of the passes dctc_carver_resize and
// dctc_carver_batch_resize run (dctc_resize_plan exports it).  It restates the host carver's dctc_lqr_carver_resize /
// resize_axis (host/dctc_lqr.c): the width first, then the height; along each axis either one shrink pass of
// extent - new_extent seams, or enlarge passes of min(new_extent - extent, extent - 1) seams until the target is reached.
// Plain C++ without CUDA, so a host compiler can check it (tests/test_resize_plan_cpu.py).
#pragma once
#include <cstddef>
#include "../../include/dctc.h"

// An enlarge pass that does not reach the target doubles extent - 1, so an int extent takes at most 31 passes per axis
constexpr int DCTC_RESIZE_MAX_PASSES = 64;

// Writes the first max_passes passes (passes may be null when max_passes is 0) and returns the number of passes:
// DCTC_ERR_INVALID for a non-positive size, DCTC_ERR_STATE when a pass cannot make progress (an extent of 1 cannot grow).
inline int dctc_resize_passes(int w, int h, int new_w, int new_h, DctcResizePass* passes, int max_passes)
{
    if (w <= 0 || h <= 0 || new_w <= 0 || new_h <= 0 || max_passes < 0 || (max_passes > 0 && !passes)) return DCTC_ERR_INVALID;
    int count = 0;
    size_t seams_offset = 0, vmap_offset = 0;
    for (int axis = DCTC_RESIZE_WIDTH; axis <= DCTC_RESIZE_HEIGHT; axis++) {
        int& e = axis == DCTC_RESIZE_WIDTH ? w : h;
        const int e1 = axis == DCTC_RESIZE_WIDTH ? new_w : new_h;
        const int len = axis == DCTC_RESIZE_WIDTH ? h : w;   // seam length: one entry per row (column) of the image
        while (e != e1) {
            const int enlarge = e1 > e;
            const int n = enlarge ? (e1 - e < e - 1 ? e1 - e : e - 1) : e - e1;
            if (n <= 0) return DCTC_ERR_STATE;
            if (count < max_passes) passes[count] = DctcResizePass{axis, enlarge, n, w, h, seams_offset, vmap_offset};
            count++;
            seams_offset += (size_t) n * len;
            vmap_offset += (size_t) w * h;
            e += enlarge ? n : -n;
        }
    }
    return count;
}
