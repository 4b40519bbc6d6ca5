"""GPU tests of the rigidity (dctc_carver_set_rigidity, dctc_carver_batch_set_rigidity): a seam step to a neighbouring
column costs pen = fl(rigidity / h) more, h the seam length,
    m[y][x] = fl(E[y][x] + min(fl(m[y-1][x-1] + pen), m[y-1][x], fl(m[y-1][x+1] + pen)))
with the parent the first strict minimum of those candidates.  The reference is a NumPy float32 seam loop whose operator
energies come from a second context; height, enlarge, combined resizes, levels, incremental mode and batches are checked
against the definitions they have without rigidity, bit for bit."""
import numpy as np
import pytest

import dct_carver_b200 as dc
import oracle_lib as ol
from test_carver_batch_gpu import DP_VARIANT_SIZES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)
    yield c
    c.carver_set_rigidity(0)
    c.close()


@pytest.fixture(scope="module")
def ectx():
    """Operator energies of the NumPy restatement (carver_load + carver_energy of each intermediate image)."""
    c = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)
    yield c
    c.close()


@pytest.fixture(autouse=True)
def _reset(ctx):
    ctx.set_params(8, 0.5, 0.5)
    yield
    ctx.carver_set_rigidity(0)
    ctx.carver_set_incremental(False)
    ctx.carver_set_dump_vmaps(False)


def image(w, h, ch, seed, pattern=0):
    return ol.synth_image(w, h, ch, seed, pattern).reshape(h, w, ch)


def op_energy(ectx, img):
    ectx.carver_load(img)
    return ectx.carver_energy()


def rigidity_for(ectx, img, factor):
    """The rigidity whose pen is factor x the mean operator energy of img (seams as long as img is tall)."""
    return float(np.float32(factor * (float(np.mean(op_energy(ectx, img))) + 1e-3) * img.shape[0]))


def ref_shrink(ectx, img, rigidity, n, bias=None):
    """NumPy restatement of a rigid (and optionally biased) width seam loop.  rigidity: a value or one per seam.
    Returns (seams [n, h], image, visibility map [h, w0])."""
    h, w0 = img.shape[:2]
    rig = np.broadcast_to(np.asarray(rigidity, np.float32), (n,))
    cur = img.copy()
    B = None if bias is None else bias.astype(np.float32).copy()
    raw = np.tile(np.arange(w0), (h, 1))
    vmap = np.zeros((h, w0), np.int32)
    seams = np.zeros((n, h), np.int32)
    inf = np.float32(np.inf)
    for s in range(n):
        w = cur.shape[1]
        pen = np.float32(rig[s]) / np.float32(h)                 # float32 IEEE division
        E = op_energy(ectx, cur)
        if B is not None:
            E = E + B / np.float32(w0)
        assert E.dtype == np.float32 and pen.dtype == np.float32
        m = np.empty_like(E)
        m[0] = E[0]
        for y in range(1, h):
            p = np.concatenate(([inf], m[y - 1], [inf]))
            m[y] = E[y] + np.minimum(np.minimum(p[:-2] + pen, p[1:-1]), p[2:] + pen)
        x = int(np.argmin(m[h - 1]))                            # leftmost minimum
        seam = np.empty(h, np.int64)
        seam[h - 1] = x
        for y in range(h - 1, 0, -1):
            cand = [c for c in (x - 1, x, x + 1) if 0 <= c < w]
            vals = np.array([m[y - 1][c] + pen if c != x else m[y - 1][c] for c in cand], np.float32)
            x = cand[int(np.argmin(vals))]                      # first strict minimum scanning x-1, x, x+1
            seam[y - 1] = x
        seams[s] = seam
        keep = np.ones((h, w), bool)
        keep[np.arange(h), seam] = False
        vmap[np.arange(h), raw[np.arange(h), seam]] = s + 1
        cur = cur[keep].reshape(h, w - 1, -1)
        raw = raw[keep].reshape(h, w - 1)
        if B is not None:
            B = B[keep].reshape(h, w - 1)
    return seams, cur, vmap


def inflate(img, vmap, n):
    """The enlarge of img by the first n seams of vmap: integer mean with the left neighbour (a copy in column 0)."""
    h, w0 = vmap.shape
    rows = []
    for y in range(h):
        px = []
        for x in range(w0):
            if 0 < vmap[y, x] <= n:
                a = img[y, x].astype(np.int32)
                left = img[y, x - 1].astype(np.int32) if x > 0 else a
                px.append(((left + a) // 2).astype(np.uint8))
            px.append(img[y, x])
        rows.append(np.stack(px))
    return np.stack(rows)


def single(ctx, img, rigidity, call, n, vmaps=True):
    """Loads img, sets the rigidity (None: never set) and runs one seam call: everything it shows afterwards."""
    ctx.carver_load(img)
    if rigidity is not None:
        ctx.carver_set_rigidity(rigidity)
    ctx.carver_set_dump_vmaps(vmaps)
    before = ctx.launches
    seams = getattr(ctx, call)(n)
    out = dict(seams=seams, image=ctx.carver_image(), energy=ctx.carver_energy(), launches=ctx.launches - before)
    if vmaps:
        h, w = img.shape[:2]
        out["vmap"] = ctx.carver_vmap(w, h)[0]
    ctx.carver_set_dump_vmaps(False)
    return out


def check_width(ctx, ectx, img, rigidity, n):
    got = single(ctx, img, rigidity, "carver_resize_width", n)
    seams, want_img, want_vmap = ref_shrink(ectx, img, rigidity, n)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], want_img)
    assert np.array_equal(got["vmap"], want_vmap)
    assert np.array_equal(got["energy"], op_energy(ectx, want_img))
    return got


def mean_jump(seams):
    return float(np.abs(np.diff(seams.astype(np.int64), axis=-1)).mean())


# ---- against the NumPy restatement -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("factor", [0.1, 1.0, 10.0])
def test_width_matches_numpy_restatement(ctx, ectx, ch, factor):
    img = image(96, 64, ch, 8100 + ch)
    rigidity = rigidity_for(ectx, img, factor)
    got = check_width(ctx, ectx, img, rigidity, 30)
    plain = single(ctx, img, 0.0, "carver_resize_width", 30)
    assert not np.array_equal(got["seams"], plain["seams"])     # the rigidity really changes the seams


def test_1080p_prefix(ctx, ectx):
    img = image(1920, 1080, 3, 8200)
    check_width(ctx, ectx, img, rigidity_for(ectx, img, 1.0), 3)


# strip width P of the seam DP and its energy staging (the width map of test_carver_batch_gpu.py)
@pytest.mark.parametrize("w,h", DP_VARIANT_SIZES)
def test_dp_variants(ctx, ectx, w, h):
    img = image(w, h, 1, w + 8300, pattern=2)
    check_width(ctx, ectx, img, rigidity_for(ectx, img, 1.0), 3)


def test_tall_frame_serial_backtrack(ctx, ectx):
    """2800 rows: the DP kernel walks the seam back itself (no jump / trace kernels)."""
    img = image(64, 2800, 3, 8400)
    check_width(ctx, ectx, img, rigidity_for(ectx, img, 1.0), 3)


def test_pitch_equals_width(ctx, ectx):
    """w = 160: energy and cumulative rows have no padding, the back-track's right sentinel lands in the window's pad."""
    img = image(160, 50, 3, 8500)
    check_width(ctx, ectx, img, rigidity_for(ectx, img, 1.0), 12)


# ---- rigidity 0, launches, straightness ----------------------------------------------------------------------------------

@pytest.mark.parametrize("call", ["carver_resize_width", "carver_resize_height", "carver_enlarge_width"])
def test_zero_equals_never_set(ctx, ectx, call):
    img = image(80, 60, 3, 8600)
    want = single(ctx, img, None, call, 17)
    ctx.carver_set_rigidity(rigidity_for(ectx, img, 1.0))
    ctx.carver_set_rigidity(0)
    got = single(ctx, img, None, call, 17)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
    frames = np.stack([image(48, 36, 3, 8601 + i) for i in range(3)])
    outs = []
    for r in (None, 0.0):
        b = dc.CarverBatch(ctx, frames, dump_vmaps=True)
        try:
            if r is not None:
                b.set_rigidity(r)
            before = ctx.launches
            outs.append((b.resize_width(9), b.images(), b.energy(), b.vmap()[0], ctx.launches - before))
        finally:
            b.close()
    for g, w in zip(*outs):
        assert np.array_equal(g, w)


def test_rigid_loop_launches_what_a_plain_loop_launches(ctx, ectx):
    img = image(200, 120, 3, 8700)
    r = rigidity_for(ectx, img, 1.0)
    for call in ("carver_resize_width", "carver_resize_height", "carver_enlarge_width"):
        for n in (5, 12):
            assert single(ctx, img, r, call, n)["launches"] == single(ctx, img, 0.0, call, n)["launches"], (call, n)
    tall = image(40, 2800, 1, 8701)        # serial back-track
    assert (single(ctx, tall, rigidity_for(ectx, tall, 1.0), "carver_resize_width", 3)["launches"] ==
            single(ctx, tall, 0.0, "carver_resize_width", 3)["launches"])


def test_seams_straighten_as_rigidity_grows(ctx, ectx):
    img = np.random.default_rng(8800).integers(0, 256, (90, 120, 3), dtype=np.uint8)
    jumps = []
    for factor in (0.0, 0.1, 1.0, 10.0):
        jumps.append(mean_jump(single(ctx, img, rigidity_for(ectx, img, factor), "carver_resize_width", 20)["seams"]))
    assert all(b <= a for a, b in zip(jumps, jumps[1:])), jumps
    assert jumps[-1] < jumps[0], jumps
    straight = single(ctx, img, rigidity_for(ectx, img, 1e6), "carver_resize_width", 20)["seams"]
    assert mean_jump(straight) == 0.0


# ---- the other operations keep their definitions -------------------------------------------------------------------------

def test_height_is_width_on_the_transpose(ctx, ectx):
    img = image(70, 90, 3, 8900)
    t = np.ascontiguousarray(img.transpose(1, 0, 2))
    r = rigidity_for(ectx, t, 1.0)                    # horizontal seams are 70 long
    got = single(ctx, img, r, "carver_resize_height", 15)
    seams, want_t, want_vmap_t = ref_shrink(ectx, t, r, 15)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], want_t.transpose(1, 0, 2))
    assert np.array_equal(got["vmap"], want_vmap_t.T)


@pytest.mark.parametrize("axis", ["width", "height"])
def test_enlarge_is_the_inflate_of_the_rigid_shrink(ctx, ectx, axis):
    img = image(64, 56, 3, 9000)
    src = img if axis == "width" else np.ascontiguousarray(img.transpose(1, 0, 2))
    r = rigidity_for(ectx, src, 1.0)
    got = single(ctx, img, r, "carver_enlarge_" + axis, 11)
    seams, _, vmap = ref_shrink(ectx, src, r, 11)
    want = inflate(src, vmap, 11)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], want if axis == "width" else want.transpose(1, 0, 2))


@pytest.mark.parametrize("target", [(50, 40), (90, 44), (62, 70)])
def test_combined_resize_is_the_per_axis_chain(ctx, ectx, target):
    img = image(70, 52, 3, 9100)
    r = rigidity_for(ectx, img, 1.0)
    ctx.carver_set_rigidity(r)
    ctx.carver_load(img)
    got = ctx.carver_resize(*target)
    final = ctx.carver_image()
    cur = img
    plan = dc.resize_plan(70, 52, *target)
    assert len(got) == len(plan)
    for g, p in zip(got, plan):
        ctx.carver_load(cur)
        fn = "carver_%s_%s" % ("enlarge" if p["enlarge"] else "resize", p["axis"])
        want = getattr(ctx, fn)(p["n_seams"])
        assert np.array_equal(g["seams"], want), p
        cur = ctx.carver_image()
    assert np.array_equal(final, cur)


@pytest.mark.parametrize("axis", ["width", "height"])
def test_levels_render_the_rigid_resizes(ctx, ectx, axis):
    img = image(72, 60, 3, 9200)
    r = rigidity_for(ectx, img, 1.0)
    ctx.carver_set_rigidity(r)
    ctx.carver_load(img)
    getattr(ctx, "carver_levels_" + axis)(20)
    e0 = 72 if axis == "width" else 60
    ext = [e0 - 20, e0 - 7, e0, e0 + 5, e0 + 20]
    got = ctx.carver_render_levels(ext)
    for e, g in zip(ext, got):
        ctx.carver_load(img)
        if e < e0:
            getattr(ctx, "carver_resize_" + axis)(e0 - e)
        elif e > e0:
            getattr(ctx, "carver_enlarge_" + axis)(e - e0)
        assert np.array_equal(g, ctx.carver_image()), e


def test_bias_and_rigidity(ctx, ectx):
    img = image(96, 64, 3, 9300)
    ectx.carver_load(img)
    en = ectx.carver_energy()
    bias = (np.random.default_rng(9300).standard_normal((64, 96)) * 2.0 * float(np.mean(en)) * 96).astype(np.float32)
    r = rigidity_for(ectx, img, 1.0)
    ctx.carver_load(img)
    ctx.carver_set_bias(bias)
    ctx.carver_set_rigidity(r)
    ctx.carver_set_dump_vmaps(True)
    seams = ctx.carver_resize_width(25)
    want_seams, want_img, want_vmap = ref_shrink(ectx, img, r, 25, bias=bias)
    assert np.array_equal(seams, want_seams)
    assert np.array_equal(ctx.carver_image(), want_img)
    assert np.array_equal(ctx.carver_vmap(96, 64)[0], want_vmap)


def test_incremental_equals_rebuild(ctx, ectx):
    img = image(300, 200, 3, 9400)
    r = rigidity_for(ectx, img, 1.0)
    want = single(ctx, img, r, "carver_resize_width", 40)
    ctx.carver_set_incremental(True)
    got = single(ctx, img, r, "carver_resize_width", 40)
    assert ctx.carver_rebuild_count() < 40          # the walk served seams
    for k in ("seams", "image", "energy", "vmap"):
        assert np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("method,n", [("resize_width", 9), ("resize_height", 7), ("enlarge_width", 11),
                                      ("enlarge_height", 6)])
def test_batch_frames_equal_single_sessions(ctx, ectx, method, n):
    frames = np.stack([image(80, 48, 3, 9500 + i, pattern=i % 4) for i in range(4)])
    r = rigidity_for(ectx, frames[0], 1.0)
    b = dc.CarverBatch(ctx, frames)
    try:
        b.set_rigidity(r)
        seams, imgs, en = getattr(b, method)(n), b.images(), b.energy()
    finally:
        b.close()
    for i, f in enumerate(frames):
        s = single(ctx, f, r, "carver_" + method, n, vmaps=False)
        assert np.array_equal(seams[i], s["seams"]), i
        assert np.array_equal(imgs[i], s["image"]), i
        assert np.array_equal(en[i], s["energy"]), i


def test_batch_resize_and_levels_equal_single_sessions(ctx, ectx):
    frames = np.stack([image(64, 40, 3, 9600 + i) for i in range(3)])
    r = rigidity_for(ectx, frames[0], 1.0)
    b = dc.CarverBatch(ctx, frames)
    try:
        b.set_rigidity(r)
        got = b.resize(50, 33)
        got_img = b.images()
        b.load(frames)                               # the rigidity survives the load
        b.levels_width(10)
        lv = b.render_levels([54, 60, 70])
    finally:
        b.close()
    for i, f in enumerate(frames):
        ctx.carver_set_rigidity(r)
        ctx.carver_load(f)
        want = ctx.carver_resize(50, 33)
        for g, w in zip(got, want):
            assert np.array_equal(g["seams"][i], w["seams"])
        assert np.array_equal(got_img[i], ctx.carver_image())
        ctx.carver_load(f)
        ctx.carver_levels_width(10)
        for g, w in zip(lv, ctx.carver_render_levels([54, 60, 70])):
            assert np.array_equal(g[i], w)


# ---- rules ---------------------------------------------------------------------------------------------------------------

def test_invalid_values_are_refused(ctx):
    frames = np.stack([image(32, 20, 1, 9700)])
    b = dc.CarverBatch(ctx, frames)
    try:
        for bad in (-1.0, -1e-30, float("nan"), float("inf"), -float("inf")):
            with pytest.raises(dc.DctcError) as e:
                ctx.carver_set_rigidity(bad)
            assert e.value.status == dc.ERR_INVALID
            with pytest.raises(dc.DctcError) as e:
                b.set_rigidity(bad)
            assert e.value.status == dc.ERR_INVALID
    finally:
        b.close()
    L = dc.lib()
    assert L.dctc_carver_set_rigidity(None, 1.0) == dc.ERR_INVALID
    assert L.dctc_carver_batch_set_rigidity(None, 1.0) == dc.ERR_INVALID


def test_option_persists_across_loads(ctx, ectx):
    img = image(90, 60, 3, 9800)
    r = rigidity_for(ectx, img, 1.0)
    ctx.carver_set_rigidity(r)
    ctx.carver_load(image(40, 30, 3, 9801))
    ctx.carver_resize_width(3)
    got = single(ctx, img, None, "carver_resize_width", 20)   # loaded again without setting it: still rigid
    seams, want_img, want_vmap = ref_shrink(ectx, img, r, 20)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], want_img) and np.array_equal(got["vmap"], want_vmap)


@pytest.mark.parametrize("incremental", [False, True])
def test_change_between_split_resizes_applies_to_the_second(ctx, ectx, incremental):
    """Incremental mode: the change drops the map built with the old pen, so the result equals the NumPy loop."""
    img = image(120, 80, 3, 9900)
    r1, r2 = rigidity_for(ectx, img, 0.1), rigidity_for(ectx, img, 10.0)
    ctx.carver_set_incremental(incremental)
    ctx.carver_set_rigidity(r1)
    ctx.carver_load(img)
    a = ctx.carver_resize_width(10)
    ctx.carver_set_rigidity(r2)
    bseams = ctx.carver_resize_width(10)
    seams, want_img, _ = ref_shrink(ectx, img, [r1] * 10 + [r2] * 10, 20)
    assert np.array_equal(np.concatenate([a, bseams]), seams)
    assert np.array_equal(ctx.carver_image(), want_img)


def test_levels_build_is_not_affected_by_a_later_change(ctx, ectx):
    img = image(72, 48, 3, 9950)
    r = rigidity_for(ectx, img, 1.0)
    ctx.carver_set_rigidity(r)
    ctx.carver_load(img)
    ctx.carver_levels_width(12)
    before = ctx.carver_render_levels([60, 66, 84])
    ctx.carver_set_rigidity(0)
    after = ctx.carver_render_levels([60, 66, 84])
    for x, y in zip(before, after):
        assert np.array_equal(x, y)


# ---- the host carver -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("seams_number,vertically", [(-12, False), (-9, True), (10, False)])
def test_host_carver_device_loop_equals_host_loop(ctx, ectx, seams_number, vertically):
    from dct_carver_b200 import host
    img = image(88, 64, 3, 9990)
    src = img if not vertically else np.ascontiguousarray(img.transpose(1, 0, 2))
    r = rigidity_for(ectx, src, 1.0)
    dev = host.render(img, seams_number, 8, 0.5, 0.5, vertically=vertically, ctx=ctx, device_loop=True, rigidity=r)
    hst = host.render(img, seams_number, 8, 0.5, 0.5, vertically=vertically, ctx=ctx, device_loop=False, rigidity=r)
    plain = host.render(img, seams_number, 8, 0.5, 0.5, vertically=vertically, ctx=ctx, device_loop=True)
    for k in ("seams", "image", "vmap"):
        assert np.array_equal(dev[k], hst[k]), k
    assert not np.array_equal(dev["seams"], plain["seams"])
    if seams_number < 0 and not vertically:
        seams, want_img, _ = ref_shrink(ectx, img, r, -seams_number)
        assert np.array_equal(dev["seams"], seams) and np.array_equal(dev["image"], want_img)
