"""GPU tests of height retargeting on the device (dctc_carver_resize_height / _enlarge_height and the batch's _height
calls).  One reference defines every result: transpose the image with numpy, load it into a single session, run the
width call and transpose the results back.  Seams, image, energy plane, visibility map, energy image and painted seams
must match it bit for bit; every frame of a batch must match its single session's height call."""
import ctypes as C

import numpy as np
import pytest

import dct_carver_b200 as dc
import oracle_lib as ol

pytestmark = pytest.mark.gpu

DP_MAX_W = 8 * 8 * (512 - 2 * 32)   # widest frame the device seam DP covers (dctc_k2_carver.cu)


@pytest.fixture(scope="module")
def ctx():
    # the single session's arithmetic: FP32 march (full maps) + FP32 tile (band updates)
    c = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)
    yield c
    c.close()


def T(a):
    """The transpose of an image [h, w(, ch)] or plane [h, w]."""
    return np.ascontiguousarray(np.swapaxes(a, 0, 1))


def image(w, h, ch, seed, pattern=0):
    img = ol.synth_image(w, h, ch, seed, pattern)
    return img.reshape(h, w, ch)


def results(ctx, start, seams, vmaps, orient):
    """Everything the session shows after a seam call, turned into image orientation by orient."""
    out = dict(seams=seams, image=orient(ctx.carver_image()), energy=orient(ctx.carver_energy()),
               energy_image=orient(ctx.carver_energy_image()))
    if vmaps:
        h, w = start.shape[:2]
        vm, depth = ctx.carver_vmap(w, h)
        out["vmap"], out["depth"] = orient(vm), depth
        out["paint"] = orient(ctx.carver_paint_seams(start))
    return out


def reference(ctx, img, n, vmaps=False, enlarge=False):
    t = T(img)
    ctx.carver_load(t)
    ctx.carver_set_dump_vmaps(vmaps)
    try:
        seams = ctx.carver_enlarge_width(n) if enlarge else ctx.carver_resize_width(n)
        return results(ctx, t, seams, vmaps, T)
    finally:
        ctx.carver_set_dump_vmaps(False)


def device(ctx, img, n, vmaps=False, enlarge=False):
    ctx.carver_load(img)
    ctx.carver_set_dump_vmaps(vmaps)
    try:
        seams = ctx.carver_enlarge_height(n) if enlarge else ctx.carver_resize_height(n)
        return results(ctx, img, seams, vmaps, lambda a: a)
    finally:
        ctx.carver_set_dump_vmaps(False)


def assert_same(got, want):
    assert got.keys() == want.keys()
    for k in want:
        if k == "depth":
            assert got[k] == want[k]
        else:
            assert got[k].shape == want[k].shape, k
            assert np.array_equal(got[k], want[k]), k


# ---- single session -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("b", [2, 4, 8, 16])
@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("w,h", [(203, 144), (144, 203)])
def test_resize_height_equals_transposed_width_call(ctx, b, ch, w, h):
    img = image(w, h, ch, 1000 + 10 * b + ch, pattern=(b + ch) % 4)
    ctx.set_params(b, 0.5, 0.5)
    got = device(ctx, img, 9, vmaps=True)
    assert got["image"].shape == (h - 9, w, ch) and got["seams"].shape == (9, w)
    assert_same(got, reference(ctx, img, 9, vmaps=True))


@pytest.mark.parametrize("w,h", [(203, 144), (144, 203)])
@pytest.mark.parametrize("which", ["one", "all_but_one"])
def test_one_and_all_but_one_seam(ctx, w, h, which):
    img = image(w, h, 3, 77 + w)
    n = 1 if which == "one" else h - 1
    ctx.set_params(8, 0.5, 0.5)
    got = device(ctx, img, n, vmaps=True)
    assert got["image"].shape == (h - n, w, 3)
    assert_same(got, reference(ctx, img, n, vmaps=True))


def test_non_uniform_weights(ctx):
    img = image(150, 120, 3, 31)
    ctx.set_params(8, 0.8, 0.2)
    try:
        assert_same(device(ctx, img, 17, vmaps=True), reference(ctx, img, 17, vmaps=True))
    finally:
        ctx.set_params(8, 0.5, 0.5)


@pytest.mark.parametrize("incremental", [False, True])
def test_split_resizes(ctx, incremental):
    img = image(130, 110, 3, 41, pattern=1)
    ctx.set_params(8, 0.5, 0.5)
    want = reference(ctx, img, 23, vmaps=True)
    ctx.carver_load(img)
    ctx.carver_set_dump_vmaps(True)
    ctx.carver_set_incremental(incremental)
    try:
        seams = np.concatenate([ctx.carver_resize_height(10), ctx.carver_resize_height(13)])
        got = results(ctx, img, seams, True, lambda a: a)
    finally:
        ctx.carver_set_incremental(False)
        ctx.carver_set_dump_vmaps(False)
    assert_same(got, want)


def test_set_params_mid_session_rebuilds_the_transposed_map(ctx):
    img = image(120, 100, 3, 51)
    ctx.set_params(8, 0.5, 0.5)
    t = T(img)
    ctx.carver_load(t)
    first = ctx.carver_resize_width(6)
    ctx.set_params(4, 0.6, 0.4)
    want = results(ctx, t, np.concatenate([first, ctx.carver_resize_width(8)]), False, T)
    ctx.set_params(8, 0.5, 0.5)
    ctx.carver_load(img)
    first = ctx.carver_resize_height(6)
    ctx.set_params(4, 0.6, 0.4)
    got = results(ctx, img, np.concatenate([first, ctx.carver_resize_height(8)]), False, lambda a: a)
    ctx.set_params(8, 0.5, 0.5)
    assert_same(got, want)


def test_pixel_energy_speaks_image_orientation(ctx):
    img = image(40, 30, 3, 61)
    ctx.set_params(8, 0.5, 0.5)
    ctx.carver_load(img)
    ctx.carver_resize_height(3)
    en = ctx.carver_energy()
    assert en.shape == (27, 40)
    p = dc.CarverEnergyParams()
    p.base.edges, p.base.textures, p.base.blocksize = 0.5, 0.5, 8
    p.gpu = ctx.handle.value
    L = dc.lib()
    for x, y in [(7, 9), (39, 0), (0, 26), (20, 13)]:
        assert L.dctc_pixel_energy(x, y, 40, 27, None, C.byref(p)) == en[y, x]
    assert np.isnan(L.dctc_pixel_energy(7, 9, 27, 40, None, C.byref(p)))   # the transposed size is not the image's


@pytest.mark.parametrize("ch", [1, 3, 4])
def test_enlarge_height_then_resize_height(ctx, ch):
    img = image(97, 80, ch, 71 + ch)
    ctx.set_params(8, 0.5, 0.5)
    want = reference(ctx, img, 25, vmaps=True, enlarge=True)
    more_want = ctx.carver_resize_width(11)
    want_after = results(ctx, None, more_want, False, T)
    got = device(ctx, img, 25, vmaps=True, enlarge=True)
    assert got["image"].shape == (105, 97, ch)
    assert_same(got, want)
    more = ctx.carver_resize_height(11)
    assert_same(results(ctx, None, more, False, lambda a: a), want_after)


def test_plugin_path_matches_the_device_call(ctx):
    """host.render(vertically=True) transposes on the host and runs the width loop; the device call must agree, and
    the host carver's map is the transpose of the device map."""
    from dct_carver_b200 import host
    img = image(120, 90, 3, 81)
    ctx.set_params(8, 0.5, 0.5)
    want = host.render(img, -14, 8, 0.5, 0.5, vertically=True, ctx=ctx)
    got = device(ctx, img, 14, vmaps=True)
    assert np.array_equal(got["image"], want["image"])
    assert np.array_equal(got["seams"], want["seams"])
    assert want["vmap"].shape == (120, 90) and want["vmap_depth"] == got["depth"] == 14
    assert np.array_equal(got["vmap"], want["vmap"].T)


def test_wide_image_takes_the_serial_backtrack(ctx):
    """3840 x 64: the transposed frame is 3840 rows tall, beyond the parallel back-track's shared-memory cone."""
    img = image(3840, 64, 3, 91)
    ctx.set_params(8, 0.5, 0.5)
    assert_same(device(ctx, img, 5, vmaps=True), reference(ctx, img, 5, vmaps=True))


def test_tall_narrow_image_takes_the_register_ring(ctx):
    """16 x 9000: the transposed frame is 9000 wide, where the seam DP keeps its energies in a register ring (P = 2)."""
    img = image(16, 9000, 3, 101)
    ctx.set_params(8, 0.5, 0.5)
    assert_same(device(ctx, img, 7), reference(ctx, img, 7))


def test_launch_counts(ctx):
    img = image(160, 120, 3, 111)
    ctx.set_params(8, 0.5, 0.5)
    ctx.carver_load(T(img))
    ctx.carver_set_dump_vmaps(True)
    try:
        n0 = ctx.launches
        ctx.carver_resize_width(6)
        n1 = ctx.launches
        ctx.carver_resize_width(6)
        width_first, width_next = n1 - n0, ctx.launches - n1
        n0 = ctx.launches
        ctx.carver_image()
        assert ctx.launches == n0                                  # an untransposed download launches nothing
        ctx.carver_load(img)
        n0 = ctx.launches
        ctx.carver_resize_height(6)
        n1 = ctx.launches
        ctx.carver_resize_height(6)
        assert n1 - n0 == width_first + 2                          # transpose + K1 of the transposed image
        assert ctx.launches - n1 == width_next
        for read in (ctx.carver_image, ctx.carver_energy):
            n0 = ctx.launches
            read()
            assert ctx.launches == n0 + 1                          # one transpose on the way out
    finally:
        ctx.carver_set_dump_vmaps(False)


def test_states_and_errors(ctx):
    L = dc.lib()
    h = ctx.handle
    ctx.set_params(8, 0.5, 0.5)
    fresh = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)   # nothing loaded
    try:
        assert L.dctc_carver_resize_height(fresh.handle, 1, None) == dc.ERR_STATE
        assert L.dctc_carver_enlarge_height(fresh.handle, 1, None) == dc.ERR_STATE
    finally:
        fresh.close()
    assert L.dctc_carver_resize_height(None, 1, None) == dc.ERR_INVALID
    img = image(48, 32, 3, 121)
    ctx.carver_load(img)
    assert L.dctc_carver_resize_height(h, -1, None) == dc.ERR_INVALID
    assert L.dctc_carver_enlarge_height(h, -1, None) == dc.ERR_INVALID
    assert L.dctc_carver_resize_height(h, 32, None) == dc.ERR_STATE       # n >= height
    assert L.dctc_carver_enlarge_height(h, 32, None) == dc.ERR_STATE
    assert L.dctc_carver_resize_height(h, 0, None) == dc.OK
    assert ctx.carver_size() == (48, 32)
    # height after width
    ctx.carver_resize_width(2)
    assert L.dctc_carver_resize_height(h, 1, None) == dc.ERR_STATE
    assert L.dctc_carver_enlarge_height(h, 1, None) == dc.ERR_STATE
    # a reload clears the axis; width after height
    ctx.carver_load(img)
    ctx.carver_resize_height(2)
    assert ctx.carver_size() == (48, 30)
    assert L.dctc_carver_resize_width(h, 1, None) == dc.ERR_STATE
    assert L.dctc_carver_enlarge_width(h, 1, None) == dc.ERR_STATE
    seam = np.full(30, 3, np.int32)
    assert L.dctc_carve_and_update(h, seam.ctypes.data, None, None, None) == dc.ERR_STATE   # the vertical-seam hook
    assert L.dctc_carver_resize_height(h, 30, None) == dc.ERR_STATE       # n >= current height
    assert L.dctc_carver_resize_height(h, 29, None) == dc.OK
    assert ctx.carver_size() == (48, 1)
    ctx.carver_load(img)
    ctx.carver_resize_width(1)
    ctx.carver_load(img)
    ctx.carver_enlarge_height(3)
    assert ctx.carver_size() == (48, 35)
    # taller than the seam DP covers: refused before any work, the session stays loaded and keeps no axis
    tall = np.zeros((DP_MAX_W + 1, 4), np.uint8)
    ctx.carver_load(tall)
    for fn in (L.dctc_carver_resize_height, L.dctc_carver_enlarge_height):
        assert fn(h, 1, None) == dc.ERR_UNSUPPORTED
    assert ctx.carver_size() == (4, DP_MAX_W + 1)
    assert ctx.carver_resize_width(1).shape == (1, DP_MAX_W + 1)
    assert ctx.carver_size() == (3, DP_MAX_W + 1)


# ---- batch session --------------------------------------------------------------------------------------------------

def frames_of(w, h, ch, seeds, patterns=(0,)):
    return np.stack([image(w, h, ch, s, patterns[i % len(patterns)]) for i, s in enumerate(seeds)])


def run_batch(ctx, frames, n, vmaps=False, enlarge=False):
    b = dc.CarverBatch(ctx, frames, dump_vmaps=vmaps)
    try:
        seams = b.enlarge_height(n) if enlarge else b.resize_height(n)
        assert (b.width, b.height) == (frames.shape[2], frames.shape[1] + (n if enlarge else -n))
        return seams, b.images(), b.energy(), (b.vmap() if vmaps else None)
    finally:
        b.close()


def assert_frames_match_single(ctx, frames, n, got, vmaps=False, enlarge=False):
    seams, imgs, en, vm = got
    assert seams.shape == (len(frames), n, frames.shape[2])
    for i, f in enumerate(frames):
        want = device(ctx, f, n, vmaps, enlarge)
        assert np.array_equal(seams[i], want["seams"]), "frame %d: seams" % i
        assert np.array_equal(imgs[i], want["image"]), "frame %d: image" % i
        assert np.array_equal(en[i], want["energy"]), "frame %d: energy" % i
        if vmaps:
            assert vm[1] == want["depth"] == n
            assert np.array_equal(vm[0][i], want["vmap"]), "frame %d: visibility map" % i


@pytest.mark.parametrize("b", [2, 4, 8, 16])
@pytest.mark.parametrize("ch", [1, 2, 3, 4])
def test_batch_frames_equal_single_sessions(ctx, b, ch):
    frames = frames_of(97, 75, ch, [500 + 7 * b + ch, 600 + b, 700 + ch], patterns=(0, 3, 1))
    ctx.set_params(b, 0.5, 0.5)
    vmaps = ch % 2 == 1
    assert_frames_match_single(ctx, frames, 20, run_batch(ctx, frames, 20, vmaps), vmaps)


@pytest.mark.parametrize("which", ["one", "all_but_one"])
def test_batch_one_and_all_but_one_seam(ctx, which):
    frames = frames_of(144, 203, 3, [801, 802])
    n = 1 if which == "one" else 202
    ctx.set_params(8, 0.5, 0.5)
    assert_frames_match_single(ctx, frames, n, run_batch(ctx, frames, n, vmaps=True), vmaps=True)


@pytest.mark.parametrize("vmaps", [False, True])
@pytest.mark.parametrize("ch", [1, 3, 4])
def test_batch_enlarge_height(ctx, vmaps, ch):
    frames = frames_of(203, 144, ch, [811 + ch, 812, 813])
    ctx.set_params(8, 0.5, 0.5)
    got = run_batch(ctx, frames, 30, vmaps, enlarge=True)
    assert got[1].shape == (3, 174, 203, ch)
    assert_frames_match_single(ctx, frames, 30, got, vmaps, enlarge=True)


def test_batch_reloads_and_axes(ctx):
    """Both axes and an enlarge through one batch: each load clears the axis, the buffers are reused."""
    a = frames_of(120, 90, 3, [821, 822, 823])
    c = frames_of(120, 90, 3, [831, 832, 833], patterns=(1, 0, 3))
    ctx.set_params(8, 0.5, 0.5)
    L = dc.lib()
    b = dc.CarverBatch(ctx, a, dump_vmaps=True)
    try:
        s = b.resize_height(12)
        assert L.dctc_carver_batch_resize_width(b.handle, 1, None) == dc.ERR_STATE
        assert L.dctc_carver_batch_enlarge_width(b.handle, 1, None) == dc.ERR_STATE
        assert_frames_match_single(ctx, a, 12, (s, b.images(), b.energy(), b.vmap()), vmaps=True)
        b.load(c)
        s = b.resize_width(5)
        assert L.dctc_carver_batch_resize_height(b.handle, 1, None) == dc.ERR_STATE
        assert L.dctc_carver_batch_enlarge_height(b.handle, 1, None) == dc.ERR_STATE
        assert (b.width, b.height) == (115, 90)
        b.load(c)
        s = np.concatenate([b.resize_height(7), b.resize_height(8)], axis=1)
        assert_frames_match_single(ctx, c, 15, (s, b.images(), b.energy(), b.vmap()), vmaps=True)
        for frames, n in ((a, 20), (c, 20), (a, 9)):
            b.load(frames)
            s = b.enlarge_height(n)
            assert L.dctc_carver_batch_resize_height(b.handle, 1, None) == dc.ERR_STATE
            assert_frames_match_single(ctx, frames, n, (s, b.images(), b.energy(), b.vmap()), vmaps=True, enlarge=True)
        b.load(a)
        s = b.enlarge_width(6)
        assert b.images().shape == (3, 90, 126, 3)
    finally:
        b.close()


def test_batch_errors(ctx):
    L = dc.lib()
    ctx.set_params(8, 0.5, 0.5)
    out = C.c_void_p()
    assert L.dctc_carver_batch_create(ctx.handle, 2, 16, 8, 3, 0, C.byref(out)) == dc.OK
    b = out
    try:
        assert L.dctc_carver_batch_resize_height(b, 2, None) == dc.ERR_STATE             # before a load
        assert L.dctc_carver_batch_enlarge_height(b, 2, None) == dc.ERR_STATE
        imgs = frames_of(16, 8, 3, [1, 2])
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 48) == dc.OK
        assert L.dctc_carver_batch_resize_height(None, 2, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_resize_height(b, -1, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_enlarge_height(b, -1, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_resize_height(b, 8, None) == dc.ERR_STATE             # n_seams >= height
        assert L.dctc_carver_batch_resize_height(b, 0, None) == dc.OK
        assert L.dctc_carver_batch_height(b) == 8 and L.dctc_carver_batch_height(None) == 0
        assert L.dctc_carver_batch_resize_height(b, 7, None) == dc.OK
        assert (L.dctc_carver_batch_width(b), L.dctc_carver_batch_height(b)) == (16, 1)
        assert L.dctc_carver_batch_enlarge_height(b, 1, None) == dc.ERR_STATE            # not at the loaded height
    finally:
        L.dctc_carver_batch_destroy(b)
    tall = np.zeros((2, DP_MAX_W + 1, 2), np.uint8)
    bt = dc.CarverBatch(ctx, tall)
    try:
        with pytest.raises(dc.DctcError) as e:
            bt.resize_height(1)
        assert e.value.status == dc.ERR_UNSUPPORTED
        assert bt.resize_width(1).shape == (2, 1, DP_MAX_W + 1)                         # still loaded, no axis fixed
    finally:
        bt.close()


def test_batch_1080p_to_2_39_to_1(ctx):
    """Eight distinct 1920x1080 RGB frames -> 1920x800 (280 horizontal seams each)."""
    frames = np.stack([image(1920, 1080, 3, 0x2391080 + i) for i in range(8)])
    ctx.set_params(8, 0.5, 0.5)
    got = run_batch(ctx, frames, 280)
    assert got[1].shape == (8, 800, 1920, 3)
    assert_frames_match_single(ctx, frames, 280, got)
