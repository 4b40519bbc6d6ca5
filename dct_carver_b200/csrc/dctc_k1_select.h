// K1 kernel selection: the one place that decides which kernel computes a launch (dctc_run_k1 launches exactly what
// dctc_k1_select returns).  Plain C++ without CUDA, so a host compiler can check the policy (tests/test_k1_select_cpu.py).
#pragma once
#include "../../include/dctc.h"

enum class DctcK1Variant { Tile, Small, March8, Tc8, Tc16 };

// kernel: the requested DCTC_KERNEL_*; band: per-seam update (DctcK1Args::seam set); preview: preview operator;
// fast_layout: dctc_k1_fast_layout, which the Small, Tc8 and Tc16 kernels need.  The tile kernel serves every block size
// and mode, so it takes whatever the faster kernels do not.
inline DctcK1Variant dctc_k1_select(int kernel, int blocksize, bool band, bool preview, bool fast_layout)
{
    if (band || preview) return DctcK1Variant::Tile;
    switch (blocksize) {
    case 8:   // block size 8 has no streaming kernel: FP32_STREAM runs its register-march kernel
        if (kernel == DCTC_KERNEL_FP32_TILE) return DctcK1Variant::Tile;
        if (kernel == DCTC_KERNEL_FP32_MARCH || kernel == DCTC_KERNEL_FP32_STREAM || !fast_layout) return DctcK1Variant::March8;
        return DctcK1Variant::Tc8;
    case 16:
        if (kernel == DCTC_KERNEL_FP32_TILE || kernel == DCTC_KERNEL_FP32_MARCH || !fast_layout) return DctcK1Variant::Tile;
        return DctcK1Variant::Tc16;
    default:  // 2, 4
        if ((kernel == DCTC_KERNEL_AUTO || kernel == DCTC_KERNEL_FP32_STREAM) && fast_layout) return DctcK1Variant::Small;
        return DctcK1Variant::Tile;
    }
}
