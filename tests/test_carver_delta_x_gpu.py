"""GPU tests of the seam step width (dctc_carver_set_delta_x, dctc_carver_batch_set_delta_x): a seam may move up to dx
columns from one row to the next, a step of |d| columns costing pen[|d|] = fl(fl(rigidity * fl(d * fl(sqrt(d)))) / h)
more,
    m[y][x] = fl(E[y][x] + min over |d| <= dx of fl(m[y-1][x+d] + pen[|d|]))
with the parent the first strict minimum scanning x-dx .. x+dx.  The reference is a NumPy float32 seam loop whose
operator energies come from a second context; height, enlarge, combined resizes, levels, bias, incremental mode, batches
and the host carver are checked against the definitions they have with dx = 1, bit for bit.  Every comparison with the
NumPy loop also checks that some seam takes a step of dx columns."""
import numpy as np
import pytest

import dct_carver_b200 as dc
from test_carver_batch_gpu import DP_VARIANT_SIZES
from test_carver_rigidity_gpu import image, inflate, op_energy, rigidity_for

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)
    yield c
    c.carver_set_delta_x(1)
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
    ctx.carver_set_delta_x(1)
    ctx.carver_set_rigidity(0)
    ctx.carver_set_incremental(False)
    ctx.carver_set_dump_vmaps(False)


def pen_table(rigidity, h, dx):
    d = np.arange(dx + 1, dtype=np.float32)
    return (np.float32(rigidity) * (d * np.sqrt(d))) / np.float32(h)


def ref_shrink(ectx, img, dx, rigidity, n, bias=None):
    """NumPy restatement of the width seam loop with step width dx (and optionally a bias).  Returns (seams [n, h],
    image, visibility map [h, w0])."""
    h, w0 = img.shape[:2]
    pen = pen_table(rigidity, h, dx)
    cur = img.copy()
    B = None if bias is None else bias.astype(np.float32).copy()
    raw = np.tile(np.arange(w0), (h, 1))
    vmap = np.zeros((h, w0), np.int32)
    seams = np.zeros((n, h), np.int32)
    inf = np.float32(np.inf)
    for s in range(n):
        w = cur.shape[1]
        E = op_energy(ectx, cur)
        if B is not None:
            E = E + B / np.float32(w0)
        assert E.dtype == np.float32
        m = np.empty_like(E)
        m[0] = E[0]
        for y in range(1, h):
            p = np.concatenate((np.full(dx, inf), m[y - 1], np.full(dx, inf)))
            best = p[dx:dx + w].copy()
            for d in range(1, dx + 1):
                best = np.minimum(best, np.minimum(p[dx - d:dx - d + w] + pen[d], p[dx + d:dx + d + w] + pen[d]))
            m[y] = E[y] + best
        x = int(np.argmin(m[h - 1]))                              # leftmost minimum
        seam = np.empty(h, np.int64)
        seam[h - 1] = x
        for y in range(h - 1, 0, -1):
            cand = [c for c in range(x - dx, x + dx + 1) if 0 <= c < w]
            vals = np.array([m[y - 1][c] + pen[abs(c - x)] if c != x else m[y - 1][c] for c in cand], np.float32)
            x = cand[int(np.argmin(vals))]                        # first strict minimum scanning x-dx .. x+dx
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


def max_step(seams):
    return int(np.abs(np.diff(np.asarray(seams, np.int64), axis=-1)).max())


def single(ctx, img, dx, rigidity, call, n, vmaps=True):
    """Loads img, sets dx and the rigidity (None: never set) and runs one seam call: everything it shows afterwards."""
    ctx.carver_load(img)
    if dx is not None:
        ctx.carver_set_delta_x(dx)
    ctx.carver_set_rigidity(rigidity or 0.0)
    ctx.carver_set_dump_vmaps(vmaps)
    before = ctx.launches
    seams = getattr(ctx, call)(n)
    out = dict(seams=seams, image=ctx.carver_image(), energy=ctx.carver_energy(), launches=ctx.launches - before)
    if vmaps:
        h, w = img.shape[:2]
        out["vmap"] = ctx.carver_vmap(w, h)[0]
    ctx.carver_set_dump_vmaps(False)
    return out


def check_width(ctx, ectx, img, dx, rigidity, n):
    got = single(ctx, img, dx, rigidity, "carver_resize_width", n)
    seams, want_img, want_vmap = ref_shrink(ectx, img, dx, rigidity, n)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], want_img)
    assert np.array_equal(got["vmap"], want_vmap)
    assert np.array_equal(got["energy"], op_energy(ectx, want_img))
    assert max_step(seams) == dx                      # some seam really takes a step of dx columns
    return got


# ---- against the NumPy restatement -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("factor", [0.0, 0.01])
@pytest.mark.parametrize("dx", [2, 3, 4])
def test_width_matches_numpy_restatement(ctx, ectx, dx, factor, ch):
    img = image(96, 48, ch, 7100 + 10 * dx + ch)
    check_width(ctx, ectx, img, dx, rigidity_for(ectx, img, factor) if factor else 0.0, 12)


def test_1080p(ctx, ectx):
    img = image(1920, 1080, 3, 7200)
    check_width(ctx, ectx, img, 4, rigidity_for(ectx, img, 0.01), 32)


# every strip width P of the seam DP and its energy staging (the width map of test_carver_batch_gpu.py)
@pytest.mark.parametrize("w,h", DP_VARIANT_SIZES)
@pytest.mark.parametrize("dx", [2, 4])
def test_dp_variants(ctx, ectx, dx, w, h):
    img = image(w, h, 1, w + 7300 + dx)
    check_width(ctx, ectx, img, dx, 0.0, 3)


def parallel_backtrack(w, h, dx):
    """Whether the loop traces the seams back with the jump and trace kernels (bt_plan in dctc_k2_carver.cu): the cone
    of jump entries fits into shared memory and, for dx > 1, the cumulative rows hold the trace window (264 floats)."""
    jb = 32 if dx == 1 else 31
    nb = (h - 1 + jb - 1) // jb
    j = max(nb - 1, 0)
    if dx == 1:
        return nb > 0 and 32 * j * j + 16 * j + 16 <= 200 * 1024
    r8 = (31 * dx + 7) & ~7
    m_pitch = max((w + 3) & ~3, 144)
    return nb > 0 and r8 * j * max(j - 1, 0) + 48 * j + 16 <= 180 * 1024 and m_pitch >= 264


# (300, 90): the parallel back-track for every dx; (96, 90): the serial walk (narrower than the trace window);
# (264, 70): parallel, rows exactly one trace window wide; (300, 1600): parallel for dx 2, serial for dx 3 and 4 (cone too
# large), parallel for dx 1; (64, 2800): serial for all
@pytest.mark.parametrize("w,h,n", [(300, 90, 8), (96, 90, 8), (264, 70, 8), (300, 1600, 3), (64, 2800, 3)])
@pytest.mark.parametrize("dx", [2, 3, 4])
def test_parallel_and_serial_backtrack(ctx, ectx, dx, w, h, n):
    img = image(w, h, 3, 7400 + w + h + dx)
    got = check_width(ctx, ectx, img, dx, rigidity_for(ectx, img, 0.01), n)
    plain = single(ctx, img, 1, None, "carver_resize_width", n)
    # per seam: DP, vmap update, carve (2), band K1, and jump + trace on the parallel path
    assert got["launches"] - plain["launches"] == 2 * n * (parallel_backtrack(w, h, dx) - parallel_backtrack(w, h, 1))


def test_pitch_equals_width(ctx, ectx):
    """w = 160: no row padding; the walk's right sentinels land in the window's pad."""
    img = image(160, 50, 3, 7500)
    check_width(ctx, ectx, img, 4, 0.0, 12)


# ---- dx = 1, launches ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("call", ["carver_resize_width", "carver_resize_height", "carver_enlarge_width"])
def test_one_equals_never_set(ctx, call):
    img = image(80, 60, 3, 7600)
    want = single(ctx, img, None, None, call, 17)
    ctx.carver_set_delta_x(3)
    got = single(ctx, img, 1, None, call, 17)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
    frames = np.stack([image(48, 36, 3, 7601 + i) for i in range(3)])
    outs = []
    for dx in (None, 1):
        b = dc.CarverBatch(ctx, frames, dump_vmaps=True)
        try:
            if dx is not None:
                b.set_delta_x(4)
                b.set_delta_x(dx)
            before = ctx.launches
            outs.append((b.resize_width(9), b.images(), b.energy(), b.vmap()[0], ctx.launches - before))
        finally:
            b.close()
    for g, w in zip(*outs):
        assert np.array_equal(g, w)


def test_wide_loop_launches(ctx):
    """dx > 1 launches per seam what dx = 1 launches where both trace the seams back in parallel or both walk; a frame
    narrower than the wide trace window walks back in the DP kernel (no jump and trace launches)."""
    for w, h, seed in ((300, 120, 7700), (40, 2800, 7701)):
        img = image(w, h, 1, seed)
        for n in (5, 12):
            assert single(ctx, img, 3, None, "carver_resize_width", n)["launches"] == \
                single(ctx, img, 1, None, "carver_resize_width", n)["launches"], (w, h, n)
    img = image(200, 120, 3, 7702)
    assert single(ctx, img, 3, None, "carver_resize_width", 5)["launches"] == \
        single(ctx, img, 1, None, "carver_resize_width", 5)["launches"] - 2 * 5


# ---- the other operations keep their definitions -------------------------------------------------------------------------

def test_height_is_width_on_the_transpose(ctx, ectx):
    img = image(70, 90, 3, 7800)
    t = np.ascontiguousarray(img.transpose(1, 0, 2))
    r = rigidity_for(ectx, t, 0.01)                   # horizontal seams are 70 long
    got = single(ctx, img, 3, r, "carver_resize_height", 15)
    seams, want_t, want_vmap_t = ref_shrink(ectx, t, 3, r, 15)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], want_t.transpose(1, 0, 2))
    assert np.array_equal(got["vmap"], want_vmap_t.T)
    assert max_step(seams) == 3


@pytest.mark.parametrize("axis", ["width", "height"])
def test_enlarge_is_the_inflate_of_the_shrink(ctx, ectx, axis):
    img = image(64, 56, 3, 7900)
    src = img if axis == "width" else np.ascontiguousarray(img.transpose(1, 0, 2))
    got = single(ctx, img, 4, None, "carver_enlarge_" + axis, 11)
    seams, _, vmap = ref_shrink(ectx, src, 4, 0.0, 11)
    want = inflate(src, vmap, 11)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], want if axis == "width" else want.transpose(1, 0, 2))
    assert max_step(seams) == 4


@pytest.mark.parametrize("target", [(50, 40), (90, 44), (62, 70)])
def test_combined_resize_is_the_per_axis_chain(ctx, target):
    img = image(70, 52, 3, 8000)
    ctx.carver_set_delta_x(2)
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
    assert max(max_step(g["seams"]) for g in got) == 2


@pytest.mark.parametrize("axis", ["width", "height"])
def test_levels_render_the_resizes(ctx, axis):
    img = image(72, 60, 3, 8100)
    ctx.carver_set_delta_x(3)
    ctx.carver_load(img)
    seams = getattr(ctx, "carver_levels_" + axis)(20)
    assert max_step(seams) == 3
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


def test_bias(ctx, ectx):
    img = image(96, 64, 3, 8200)
    en = op_energy(ectx, img)
    bias = (np.random.default_rng(8200).standard_normal((64, 96)) * 2.0 * float(np.mean(en)) * 96).astype(np.float32)
    r = rigidity_for(ectx, img, 0.01)
    ctx.carver_load(img)
    ctx.carver_set_bias(bias)
    ctx.carver_set_delta_x(4)
    ctx.carver_set_rigidity(r)
    ctx.carver_set_dump_vmaps(True)
    seams = ctx.carver_resize_width(25)
    want_seams, want_img, want_vmap = ref_shrink(ectx, img, 4, r, 25, bias=bias)
    assert np.array_equal(seams, want_seams)
    assert np.array_equal(ctx.carver_image(), want_img)
    assert np.array_equal(ctx.carver_vmap(96, 64)[0], want_vmap)
    assert max_step(seams) == 4


def test_incremental_mode_rebuilds(ctx):
    img = image(300, 200, 3, 8300)
    want = single(ctx, img, 2, None, "carver_resize_width", 20)
    ctx.carver_set_incremental(True)
    got = single(ctx, img, 2, None, "carver_resize_width", 20)
    for k in ("seams", "image", "energy", "vmap", "launches"):
        assert np.array_equal(got[k], want[k]), k
    assert max_step(got["seams"]) == 2


@pytest.mark.parametrize("method,n", [("resize_width", 9), ("resize_height", 7), ("enlarge_width", 11)])
def test_batch_frames_equal_single_sessions(ctx, ectx, method, n):
    frames = np.stack([image(80, 48, 3, 8400 + i, pattern=i % 4) for i in range(4)])
    r = rigidity_for(ectx, frames[0], 0.01)
    b = dc.CarverBatch(ctx, frames)
    try:
        b.set_delta_x(3)
        b.set_rigidity(r)
        seams, imgs, en = getattr(b, method)(n), b.images(), b.energy()
    finally:
        b.close()
    for i, f in enumerate(frames):
        s = single(ctx, f, 3, r, "carver_" + method, n, vmaps=False)
        assert np.array_equal(seams[i], s["seams"]), i
        assert np.array_equal(imgs[i], s["image"]), i
        assert np.array_equal(en[i], s["energy"]), i
    assert max_step(seams) == 3


# ---- dctc_carve_and_update -------------------------------------------------------------------------------------------------

def test_carve_and_update_takes_steps_up_to_delta_x(ctx, ectx):
    h, w = 48, 80
    img = image(w, h, 3, 8500)
    seam = np.array([30 + (3 * (y % 4) if (y // 4) % 2 == 0 else 12 - 3 * (y % 4)) for y in range(h)], np.int32)
    assert max_step(seam) == 3
    ctx.carver_load(img)
    with pytest.raises(dc.DctcError) as e:            # dx = 1: a step of 3 is refused
        ctx.carve_and_update(seam)
    assert e.value.status == dc.ERR_INVALID
    ctx.carver_set_delta_x(2)
    with pytest.raises(dc.DctcError) as e:
        ctx.carve_and_update(seam)
    assert e.value.status == dc.ERR_INVALID
    for bs in (8, 16):
        ctx.set_params(bs, 0.5, 0.5)
        ectx.set_params(bs, 0.5, 0.5)
        ctx.carver_load(img)
        ctx.carver_set_delta_x(3)
        band, xmin, xmax = ctx.carve_and_update(seam)
        keep = np.ones((h, w), bool)
        keep[np.arange(h), seam] = False
        full = op_energy(ectx, img[keep].reshape(h, w - 1, 3))
        assert np.array_equal(ctx.carver_energy(), full)
        r = bs // 2
        assert int((xmax - xmin + 1).max()) <= 2 * r * 4
        k = 0
        for y in range(h):
            n = xmax[y] - xmin[y] + 1
            assert np.array_equal(band[k:k + n], full[y, xmin[y]:xmax[y] + 1]), (bs, y)
            k += n
    ectx.set_params(8, 0.5, 0.5)


# ---- rules ---------------------------------------------------------------------------------------------------------------

def test_setter_errors(ctx):
    frames = np.stack([image(32, 20, 1, 8600)])
    b = dc.CarverBatch(ctx, frames)
    try:
        for bad, status in ((0, dc.ERR_INVALID), (-1, dc.ERR_INVALID), (dc.MAX_DELTA_X + 1, dc.ERR_UNSUPPORTED),
                            (100, dc.ERR_UNSUPPORTED)):
            with pytest.raises(dc.DctcError) as e:
                ctx.carver_set_delta_x(bad)
            assert e.value.status == status
            with pytest.raises(dc.DctcError) as e:
                b.set_delta_x(bad)
            assert e.value.status == status
        for ok in range(1, dc.MAX_DELTA_X + 1):
            ctx.carver_set_delta_x(ok)
            b.set_delta_x(ok)
    finally:
        b.close()
    L = dc.lib()
    assert L.dctc_carver_set_delta_x(None, 2) == dc.ERR_INVALID
    assert L.dctc_carver_batch_set_delta_x(None, 2) == dc.ERR_INVALID


def test_option_persists_across_loads(ctx, ectx):
    img = image(90, 60, 3, 8700)
    ctx.carver_set_delta_x(3)
    ctx.carver_load(image(40, 30, 3, 8701))
    ctx.carver_resize_width(3)
    got = single(ctx, img, None, None, "carver_resize_width", 10)
    seams, want_img, _ = ref_shrink(ectx, img, 3, 0.0, 10)
    assert np.array_equal(got["seams"], seams) and np.array_equal(got["image"], want_img)
    assert max_step(got["seams"]) == 3


# ---- the host carver -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dx", [2, 3, 4])
@pytest.mark.parametrize("seams_number,vertically", [(-12, False), (-9, True), (10, False)])
def test_host_carver_device_loop_equals_host_loop(ctx, ectx, dx, seams_number, vertically):
    from dct_carver_b200 import host
    img = image(88, 64, 3, 8800 + dx)
    src = img if not vertically else np.ascontiguousarray(img.transpose(1, 0, 2))
    r = rigidity_for(ectx, src, 0.01)
    dev = host.render(img, seams_number, 8, 0.5, 0.5, vertically=vertically, ctx=ctx, device_loop=True, delta_x=dx, rigidity=r)
    hst = host.render(img, seams_number, 8, 0.5, 0.5, vertically=vertically, ctx=ctx, device_loop=False, delta_x=dx, rigidity=r)
    for k in ("seams", "image", "vmap"):
        assert np.array_equal(dev[k], hst[k]), k
    assert max_step(dev["seams"]) == dx
    if seams_number < 0 and not vertically:
        seams, want_img, _ = ref_shrink(ectx, img, dx, r, -seams_number)
        assert np.array_equal(dev["seams"], seams) and np.array_equal(dev["image"], want_img)
