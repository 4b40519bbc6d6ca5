"""CPU tests of the host carver's rigidity (dctc_lqr_carver_init(carver, delta_x, rigidity), driven through
dctc_render_ext): a seam step of |d| columns costs rigidity_map[d] = fl(fl(rigidity * |d|^1.5) / h) more in the
cumulative map and in the back-track.  The host carver, fed the per-pixel callback, is compared against a NumPy
float32 restatement of the whole loop for delta_x 1 and 2."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
from dct_carver_b200 import host
from test_carver_cpu import energy_source


def rigidity_map(rigidity, h, dx):
    """fl(fl(rigidity * fl(d * fl(sqrt(d)))) / h) for d = 0 .. dx: the host carver's |d|^1.5, correctly rounded steps"""
    d = np.arange(dx + 1, dtype=np.float32)
    return (np.float32(rigidity) * (d * np.sqrt(d))) / np.float32(h)


def ref_shrink(img, n, rigidity, dx, energy):
    """NumPy restatement of the rigid seam loop with delta_x = dx: seams [n, h] and the carved image"""
    cur = img.copy()
    h = cur.shape[0]
    rmap = rigidity_map(rigidity, h, dx)
    inf = np.float32(np.inf)
    seams = np.zeros((n, h), np.int32)
    for s in range(n):
        w = cur.shape[1]
        E = energy(cur)
        assert E.dtype == np.float32
        m = np.empty_like(E)
        m[0] = E[0]
        for y in range(1, h):
            p = np.concatenate((np.full(dx, inf), m[y - 1], np.full(dx, inf)))
            best = np.full(w, inf, np.float32)
            for d in range(-dx, dx + 1):
                best = np.minimum(best, p[dx + d:dx + d + w] + rmap[abs(d)])
            m[y] = E[y] + best
        x = int(np.argmin(m[h - 1]))                              # leftmost minimum of the last row
        seam = np.empty(h, np.int32)
        seam[h - 1] = x
        for y in range(h - 1, 0, -1):
            cand = [c for c in range(x - dx, x + dx + 1) if 0 <= c < w]
            vals = np.array([m[y - 1][c] + rmap[abs(c - x)] for c in cand], np.float32)
            x = cand[int(np.argmin(vals))]                        # first strict minimum scanning left to right
            seam[y - 1] = x
        seams[s] = seam
        keep = np.ones((h, w), bool)
        keep[np.arange(h), seam] = False
        cur = cur[keep].reshape(h, w - 1, -1)
    return seams, cur


def mean_energy(energy, img):
    return float(np.mean(energy(img)))


@pytest.mark.parametrize("dx", [1, 2])
@pytest.mark.parametrize("factor", [0.1, 1.0, 10.0])
def test_rigid_host_carver_matches_numpy_restatement(dx, factor):
    img = ol.synth_image(44, 30, 3, 1300 + dx, 0)
    cbp, ep, energy = energy_source(8, 0.5, 0.5)
    rigidity = float(np.float32(factor * mean_energy(energy, img) * 30))   # pen = rigidity / h ~ factor x mean energy
    got = host.render(img, -7, 8, callback=cbp, callback_extra=C.byref(ep), rigidity=rigidity, delta_x=dx)
    seams, out = ref_shrink(img, 7, rigidity, dx, energy)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], out)
    assert got["vmap_depth"] == 7 and (got["vmap"] > 0).sum() == 7 * 30
    for k, s in enumerate(got["seams"]):
        assert np.abs(np.diff(s)).max() <= dx and s.min() >= 0 and s.max() < 44 - k


def test_rigidity_changes_the_seams_and_zero_keeps_them():
    img = ol.synth_image(40, 28, 3, 1310, 0)
    cbp, ep, energy = energy_source(4, 0.5, 0.5)
    plain = host.render(img, -6, 4, callback=cbp, callback_extra=C.byref(ep))
    zero = host.render(img, -6, 4, callback=cbp, callback_extra=C.byref(ep), rigidity=0.0, delta_x=1)
    assert np.array_equal(plain["seams"], zero["seams"]) and np.array_equal(plain["image"], zero["image"])
    rigid = host.render(img, -6, 4, callback=cbp, callback_extra=C.byref(ep),
                        rigidity=float(np.float32(mean_energy(energy, img) * 28)))
    assert not np.array_equal(plain["seams"], rigid["seams"])
    jumps = lambda r: np.abs(np.diff(r["seams"], axis=1)).mean()
    assert jumps(rigid) < jumps(plain)


def test_rigid_height_is_the_width_call_on_the_transpose():
    """Horizontal seams are w long: the transposed frame's h is the image width."""
    img = ol.synth_image(34, 46, 3, 1320, 0)
    cbp, ep, energy = energy_source(8, 0.5, 0.5)
    rigidity = float(np.float32(mean_energy(energy, img) * 34))
    a = host.render(img, -5, 8, vertically=True, callback=cbp, callback_extra=C.byref(ep), rigidity=rigidity)
    t = np.ascontiguousarray(img.transpose(1, 0, 2))
    seams, out = ref_shrink(t, 5, rigidity, 1, energy)
    assert np.array_equal(a["seams"], seams)
    assert np.array_equal(a["image"], out.transpose(1, 0, 2))
