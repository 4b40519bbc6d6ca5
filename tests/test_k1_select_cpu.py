"""CPU test of the K1 kernel selection (csrc/dctc_k1_select.h): the tile, march and streaming kernels give bit-identical
maps, so no GPU test sees which of them ran.  This pins the choice for every input of dctc_k1_select against the
table below (DESIGN.md, "K1 kernel selection")."""
import itertools
import os
import subprocess

import dct_carver_b200 as dc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dct_carver_b200", "csrc")
KERNELS = (dc.KERNEL_AUTO, dc.KERNEL_FP32_TILE, dc.KERNEL_FP32_MARCH, dc.KERNEL_TC_SPLIT, dc.KERNEL_FP32_STREAM)

DRIVER = r"""
#include <cstdio>
#include <initializer_list>
#include "dctc_k1_select.h"
int main()
{
    const char* names[] = {"Tile", "Small", "March8", "Tc8", "Tc16"};
    for (int kernel : {%s})
        for (int b : {2, 4, 8, 16})
            for (int band = 0; band < 2; band++)
                for (int preview = 0; preview < 2; preview++)
                    for (int fast = 0; fast < 2; fast++)
                        std::printf("%%d %%d %%d %%d %%d %%s\n", kernel, b, band, preview, fast,
                                    names[(int) dctc_k1_select(kernel, b, band, preview, fast)]);
}
""" % ", ".join(str(k) for k in KERNELS)


def expected(kernel, b, band, preview, fast):
    """First matching row wins."""
    if band or preview:
        return "Tile"
    if b == 8:
        if kernel == dc.KERNEL_FP32_TILE:
            return "Tile"
        if kernel in (dc.KERNEL_FP32_MARCH, dc.KERNEL_FP32_STREAM):
            return "March8"
        return "Tc8" if fast else "March8"   # AUTO, TC_SPLIT
    if b in (2, 4):
        return "Small" if kernel in (dc.KERNEL_AUTO, dc.KERNEL_FP32_STREAM) and fast else "Tile"
    return "Tc16" if kernel in (dc.KERNEL_AUTO, dc.KERNEL_TC_SPLIT, dc.KERNEL_FP32_STREAM) and fast else "Tile"


def test_k1_select_matches_the_table(tmp_path):
    src, exe = tmp_path / "select.cpp", tmp_path / "select"
    src.write_text(DRIVER)
    subprocess.check_call(["c++", "-std=c++17", "-Wall", "-Werror", "-I", CSRC, str(src), "-o", str(exe)])
    got = {}
    for line in subprocess.check_output([str(exe)], text=True).splitlines():
        *key, variant = line.split()
        got[tuple(int(v) for v in key)] = variant
    inputs = list(itertools.product(KERNELS, (2, 4, 8, 16), (0, 1), (0, 1), (0, 1)))
    assert len(inputs) == 160 and sorted(got) == sorted(inputs)
    for key in inputs:
        assert got[key] == expected(*key), key
