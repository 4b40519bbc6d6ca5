"""CPU tests of the host carver's seam step width (dctc_lqr_carver_init(carver, delta_x, rigidity), driven through
dctc_render_ext): a seam may move up to delta_x columns per row, a step of |d| columns costing
fl(fl(rigidity * |d|^1.5) / h) more.  The host carver, fed the per-pixel callback, is compared against the NumPy float32
restatement of test_carver_rigidity_cpu.py for delta_x 3 and 4 (that file covers 1 and 2)."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
from dct_carver_b200 import host
from test_carver_cpu import energy_source
from test_carver_rigidity_cpu import mean_energy, ref_shrink


@pytest.mark.parametrize("dx", [3, 4])
@pytest.mark.parametrize("factor", [0.0, 0.01])
def test_wide_steps_host_carver_matches_numpy_restatement(dx, factor):
    img = ol.synth_image(44, 30, 3, 1400 + dx, 0)
    cbp, ep, energy = energy_source(8, 0.5, 0.5)
    rigidity = float(np.float32(factor * mean_energy(energy, img) * 30))
    got = host.render(img, -7, 8, callback=cbp, callback_extra=C.byref(ep), rigidity=rigidity, delta_x=dx)
    seams, out = ref_shrink(img, 7, rigidity, dx, energy)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], out)
    steps = np.abs(np.diff(got["seams"], axis=1))
    assert steps.max() == dx                               # some seam really takes a step of dx columns
    for k, s in enumerate(got["seams"]):
        assert s.min() >= 0 and s.max() < 44 - k
