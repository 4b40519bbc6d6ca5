"""CPU test of the resize plan (csrc/dctc_resize_plan.h): the passes dctc_carver_resize and dctc_carver_batch_resize run
must be those of the host carver's dctc_lqr_carver_resize / resize_axis (host/dctc_lqr.c), restated below."""
import os
import subprocess

import pytest

import dct_carver_b200 as dc

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "dct_carver_b200", "csrc")

DRIVER = r"""
#include <cstdio>
#include <cstdlib>
#include "dctc_resize_plan.h"
int main(int argc, char** argv)
{
    for (int i = 1; i + 3 < argc; i += 4) {
        const int w = atoi(argv[i]), h = atoi(argv[i + 1]), nw = atoi(argv[i + 2]), nh = atoi(argv[i + 3]);
        DctcResizePass p[DCTC_RESIZE_MAX_PASSES];
        const int n = dctc_resize_passes(w, h, nw, nh, p, DCTC_RESIZE_MAX_PASSES);
        std::printf("%d", n);
        for (int k = 0; k < n; k++)
            std::printf(" %d,%d,%d,%d,%d,%zu,%zu", p[k].axis, p[k].enlarge, p[k].n_seams, p[k].w, p[k].h, p[k].seams_offset,
                        p[k].vmap_offset);
        std::printf("\n");
    }
}
"""


def expected(w, h, new_w, new_h):
    """dctc_lqr_carver_resize: the width, then the height through a transpose; resize_axis shrinks once or enlarges by
    min(target - extent, extent - 1) until it gets there, and fails when that is not positive.  Returns the passes as
    (axis, enlarge, n_seams, w, h, seams_offset, vmap_offset) or the refusal status."""
    if min(w, h, new_w, new_h) <= 0:
        return dc.ERR_INVALID
    passes, size = [], [w, h]

    def add(axis, enlarge, k):
        so = passes[-1][5] + passes[-1][2] * passes[-1][4 - passes[-1][0]] if passes else 0
        vo = passes[-1][6] + passes[-1][3] * passes[-1][4] if passes else 0
        passes.append((axis, enlarge, k, size[0], size[1], so, vo))
        size[axis] += k if enlarge else -k

    for axis, target in ((dc.RESIZE_WIDTH, new_w), (dc.RESIZE_HEIGHT, new_h)):
        if target < size[axis]:
            add(axis, 0, size[axis] - target)
        while target > size[axis]:
            k = min(target - size[axis], size[axis] - 1)
            if k <= 0:
                return dc.ERR_STATE
            add(axis, 1, k)
    return passes


GRID = [
    (64, 48, 64, 48), (1, 1, 1, 1),                                   # no change
    (64, 48, 40, 48), (64, 48, 64, 30), (64, 48, 90, 48), (64, 48, 64, 70),   # one axis only
    (1920, 1080, 1440, 810), (1920, 1080, 2400, 900), (1920, 1080, 1600, 1300), (100, 80, 150, 60),   # both axes
    (64, 48, 127, 48), (64, 48, 128, 48), (64, 48, 192, 48), (64, 48, 64, 95), (64, 48, 64, 96), (64, 48, 64, 144),
    (40, 30, 130, 30), (640, 360, 1920, 360), (2, 2, 1000, 3), (3, 2, 7, 1), (2, 7, 2, 1 << 30),
    (64, 48, 1, 1), (1, 48, 1, 10), (48, 1, 10, 1), (1, 5, 1, 9), (5, 2, 1, 2),
    (1, 5, 3, 5), (5, 1, 5, 3), (1, 1, 2, 1), (1, 1, 1, 2), (30, 1, 10, 2),        # an extent of 1 cannot grow
    (0, 5, 3, 5), (5, 5, 0, 5), (5, 5, 5, -1), (-3, 4, 4, 4),                      # non-positive sizes
]


@pytest.fixture(scope="module")
def plans(tmp_path_factory):
    d = tmp_path_factory.mktemp("plan")
    src, exe = d / "plan.cpp", d / "plan"
    src.write_text(DRIVER)
    subprocess.check_call(["c++", "-std=c++17", "-Wall", "-Werror", "-I", CSRC, str(src), "-o", str(exe)])
    out = subprocess.check_output([str(exe)] + [str(v) for case in GRID for v in case], text=True).splitlines()
    assert len(out) == len(GRID)
    got = {}
    for case, line in zip(GRID, out):
        n, *passes = line.split()
        got[case] = int(n) if int(n) < 0 else [tuple(int(v) for v in p.split(",")) for p in passes]
        if int(n) >= 0:
            assert len(got[case]) == int(n)
    return got


@pytest.mark.parametrize("case", GRID)
def test_plan_matches_the_host_carver(plans, case):
    assert plans[case] == expected(*case)


def test_plan_examples(plans):
    W, H = dc.RESIZE_WIDTH, dc.RESIZE_HEIGHT
    assert plans[(64, 48, 64, 48)] == []
    assert plans[(1920, 1080, 1440, 810)] == [(W, 0, 480, 1920, 1080, 0, 0),
                                              (H, 0, 270, 1440, 1080, 480 * 1080, 1920 * 1080)]
    assert plans[(64, 48, 127, 48)] == [(W, 1, 63, 64, 48, 0, 0)]
    assert plans[(64, 48, 128, 48)] == [(W, 1, 63, 64, 48, 0, 0), (W, 1, 1, 127, 48, 63 * 48, 64 * 48)]
    assert [p[2] for p in plans[(64, 48, 192, 48)]] == [63, 65]
    assert [p[2] for p in plans[(40, 30, 130, 30)]] == [39, 51]
    assert plans[(1, 5, 3, 5)] == plans[(1, 1, 1, 2)] == dc.ERR_STATE
    assert plans[(5, 5, 0, 5)] == dc.ERR_INVALID


def test_exported_plan_is_the_header_plan(plans):
    """dctc_resize_plan in the library (and resize_plan in Python) return the header's plan."""
    for case in GRID:
        want = plans[case]
        if isinstance(want, int):
            with pytest.raises(dc.DctcError) as e:
                dc.resize_plan(*case)
            assert e.value.status == want
            continue
        got = [(dc.RESIZE_WIDTH if p["axis"] == "width" else dc.RESIZE_HEIGHT, int(p["enlarge"]), p["n_seams"], p["w"],
                p["h"], p["seams_offset"], p["vmap_offset"]) for p in dc.resize_plan(*case)]
        assert got == want, case
    assert dc.lib().dctc_resize_plan(64, 48, 192, 48, None, 0) == 2
    assert dc.lib().dctc_resize_plan(64, 48, 192, 48, None, 1) == dc.ERR_INVALID
    assert dc.lib().dctc_resize_plan(64, 48, 192, 48, None, -1) == dc.ERR_INVALID
