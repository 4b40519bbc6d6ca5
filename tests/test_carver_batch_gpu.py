"""GPU tests of the batch carver session (dctc_carver_batch_*): n equally sized frames through one device seam loop.
The reference for every frame is a single carver session on the same context (carver_load + carver_resize_width);
every frame must match it bit for bit in seams, image, energy plane and visibility map."""
import ctypes as C

import numpy as np
import pytest

import dct_carver_b200 as dc
import oracle_lib as ol

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    # same arithmetic as the single session's references in test_k2_gpu.py (FP32 march + FP32 tile kernels)
    c = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)
    yield c
    c.close()


def single(ctx, frame, n, vmaps=False):
    """(seams [n, h], image [h, w - n, ch], energy [h, w - n], (vmap, depth) or None) of one single-frame session."""
    h, w = frame.shape[:2]
    ctx.carver_load(frame)
    ctx.carver_set_dump_vmaps(vmaps)
    try:
        seams = ctx.carver_resize_width(n)
        vm = ctx.carver_vmap(w, h) if vmaps else None
    finally:
        ctx.carver_set_dump_vmaps(False)
    return seams, ctx.carver_image(), ctx.carver_energy(), vm


def run_batch(ctx, frames, n, vmaps=False):
    b = dc.CarverBatch(ctx, frames, dump_vmaps=vmaps)
    try:
        seams = b.resize_width(n)
        assert b.width == frames.shape[2] - n
        return seams, b.images(), b.energy(), (b.vmap() if vmaps else None)
    finally:
        b.close()


def assert_matches_single(ctx, frames, n, got, vmaps=False):
    seams, imgs, en, vm = got
    assert seams.shape == (len(frames), n, frames.shape[1])
    for i, f in enumerate(frames):
        s, im, e, v = single(ctx, f, n, vmaps)
        assert np.array_equal(seams[i], s), "frame %d: seams" % i
        assert np.array_equal(imgs[i].reshape(im.shape), im), "frame %d: image" % i
        assert np.array_equal(en[i], e), "frame %d: energy" % i
        if vmaps:
            assert vm[1] == v[1] == n
            assert np.array_equal(vm[0][i], v[0]), "frame %d: visibility map" % i


def frames_of(w, h, ch, seeds, patterns=(0,)):
    fs = [ol.synth_image(w, h, ch, s, patterns[i % len(patterns)]) for i, s in enumerate(seeds)]
    return np.stack(fs)


@pytest.mark.parametrize("b", [2, 4, 8, 16])
@pytest.mark.parametrize("ch", [1, 3, 4])
def test_small_frames_equal_single_sessions(ctx, b, ch):
    frames = frames_of(97, 75, ch, [100 + 7 * b + ch, 200 + b, 300 + ch], patterns=(0, 3, 1))
    ctx.set_params(b, 0.5, 0.5)
    vmaps = b == 8
    assert_matches_single(ctx, frames, 20, run_batch(ctx, frames, 20, vmaps), vmaps)


def test_non_uniform_weights_equal_single_sessions(ctx):
    frames = frames_of(120, 64, 3, [11, 12, 13, 14])
    ctx.set_params(8, 0.8, 0.2)
    try:
        assert_matches_single(ctx, frames, 15, run_batch(ctx, frames, 15))
    finally:
        ctx.set_params(8, 0.5, 0.5)


# The seam DP's variant per frame width (dp_plan in csrc/dctc_k2_carver.cu): P float4 groups per lane (strips of
# 128 * P columns), energies staged in nst stages of SR rows by tensor copies, or SR = 0: a register ring.
#   width             P  SR  nst    test width
#   1 - 2560          1  32   2     300
#   2561 - 3584       1  16   3     3000
#   3585 - 4096       1  16   2     4000
#   4097 - 4608       2  16   3     4500
#   4609 - 7680       2  16   2     5000
#   7681 - 12288      2   0   -     9000
#   12289 - 28672     4   0   -     13000
# The 16-row cases are tall enough to have more chunks than stages, so each of them refills a stage.
DP_VARIANT_SIZES = [(300, 40), (3000, 56), (4000, 40), (4500, 56), (5000, 40), (9000, 16), (13000, 12)]


@pytest.mark.parametrize("w,h", DP_VARIANT_SIZES)
def test_strip_widths_and_staging_variants(ctx, w, h):
    frames = frames_of(w, h, 1, [w + 1, w + 2, w + 3], patterns=(0, 2, 0))
    ctx.set_params(8, 0.5, 0.5)
    assert_matches_single(ctx, frames, 3, run_batch(ctx, frames, 3))


def test_tall_frames_take_the_serial_backtrack(ctx):
    """2800 rows: the trace kernel's cone would exceed 200 KB of shared memory, so the DP kernel walks the seam back
    itself, per frame."""
    frames = frames_of(64, 2800, 3, [41, 42])
    ctx.set_params(8, 0.5, 0.5)
    assert_matches_single(ctx, frames, 4, run_batch(ctx, frames, 4, vmaps=True), vmaps=True)


def test_permuted_frames_give_permuted_results(ctx):
    frames = frames_of(150, 90, 3, [51, 52, 53, 54], patterns=(0, 1, 3, 0))
    ctx.set_params(8, 0.5, 0.5)
    a = run_batch(ctx, frames, 12, vmaps=True)
    perm = np.array([2, 0, 3, 1])
    b = run_batch(ctx, frames[perm], 12, vmaps=True)
    for x, y in zip(a[:3], b[:3]):
        assert np.array_equal(x[perm], y)
    assert np.array_equal(a[3][0][perm], b[3][0])


def test_identical_frames_give_identical_results(ctx):
    f = ol.synth_image(130, 70, 3, 61, 0)
    frames = np.stack([f] * 5)
    ctx.set_params(8, 0.5, 0.5)
    got = run_batch(ctx, frames, 10)
    for x in got[:3]:
        assert all(np.array_equal(x[0], x[i]) for i in range(1, 5))
    assert_matches_single(ctx, frames[:1], 10, tuple(x[:1] for x in got[:3]) + (None,))


def test_frame_between_flat_neighbours_keeps_its_seams(ctx):
    """Flat frames remove column 0 in every row; a textured frame between them must still get its own seams."""
    f = ol.synth_image(110, 60, 3, 71, 0)
    flat = np.full_like(f, 77)
    frames = np.stack([flat, f, flat])
    ctx.set_params(8, 0.5, 0.5)
    got = run_batch(ctx, frames, 9)
    assert (got[0][0] == 0).all() and (got[0][2] == 0).all()
    assert_matches_single(ctx, frames, 9, got)


def test_two_resize_calls_equal_one(ctx):
    frames = frames_of(140, 80, 3, [81, 82, 83])
    ctx.set_params(8, 0.5, 0.5)
    n = 17
    b = dc.CarverBatch(ctx, frames, dump_vmaps=True)
    try:
        parts = np.concatenate([b.resize_width(n // 2), b.resize_width(n - n // 2)], axis=1)
        got = (parts, b.images(), b.energy(), b.vmap())
    finally:
        b.close()
    want = run_batch(ctx, frames, n, vmaps=True)
    for x, y in zip(got[:3], want[:3]):
        assert np.array_equal(x, y)
    assert got[3][1] == want[3][1] == n and np.array_equal(got[3][0], want[3][0])


@pytest.mark.parametrize("vmaps", [False, True])
def test_launch_count_does_not_grow_with_the_frame_count(ctx, vmaps):
    ctx.set_params(8, 0.5, 0.5)
    growth = []
    for n in (1, 8):
        b = dc.CarverBatch(ctx, frames_of(200, 100, 3, range(90, 90 + n)), dump_vmaps=vmaps)
        try:
            before = ctx.launches
            b.resize_width(6)
            growth.append(ctx.launches - before)
        finally:
            b.close()
    assert growth[0] == growth[1] > 0


def test_single_session_survives_batch_calls(ctx):
    img = ol.synth_image(150, 90, 3, 95, 0)
    ctx.set_params(8, 0.5, 0.5)
    ctx.carver_load(img)
    ctx.carver_resize_width(5)
    size, im, en = ctx.carver_size(), ctx.carver_image(), ctx.carver_energy()
    b = dc.CarverBatch(ctx, frames_of(150, 90, 3, [96, 97]))
    b.resize_width(7)
    b.close()
    assert ctx.carver_size() == size
    assert np.array_equal(ctx.carver_image(), im)
    assert np.array_equal(ctx.carver_energy(), en)
    # the single session carries on as if no batch had run
    more = ctx.carver_resize_width(4)
    want = single(ctx, img, 9)
    assert np.array_equal(more, want[0][5:])


def test_errors(ctx):
    L = dc.lib()
    ctx.set_params(8, 0.5, 0.5)
    out = C.c_void_p()
    h = ctx.handle
    assert L.dctc_carver_batch_create(None, 2, 16, 8, 3, 0, C.byref(out)) == dc.ERR_INVALID
    assert L.dctc_carver_batch_create(h, 2, 16, 8, 3, 0, None) == dc.ERR_INVALID
    for n, w, hh, ch in [(0, 16, 8, 3), (-1, 16, 8, 3), (2, 16, 8, 0), (2, 16, 8, 5), (2, 0, 8, 3), (2, 16, 0, 3)]:
        assert L.dctc_carver_batch_create(h, n, w, hh, ch, 0, C.byref(out)) == dc.ERR_INVALID, (n, w, hh, ch)
    assert L.dctc_carver_batch_create(h, 2, 16, 8, 3, 0, C.byref(out)) == dc.OK
    b = out
    try:
        imgs = frames_of(16, 8, 3, [1, 2])
        buf = np.empty(2 * 8 * 16 * 3, np.uint8)
        en = np.empty(2 * 8 * 16, np.float32)
        # before a load: nothing to resize or read
        assert L.dctc_carver_batch_resize_width(b, 2, None) == dc.ERR_STATE
        assert L.dctc_carver_batch_images(b, buf.ctypes.data) == dc.ERR_STATE
        assert L.dctc_carver_batch_energy(b, en.ctypes.data) == dc.ERR_STATE
        assert L.dctc_carver_batch_load(None, imgs.ctypes.data, 8 * 48, 48) == dc.ERR_INVALID
        assert L.dctc_carver_batch_load(b, None, 8 * 48, 48) == dc.ERR_INVALID
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 47) == dc.ERR_INVALID        # pitch < w * ch
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48 - 1, 48) == dc.ERR_INVALID    # frames overlap
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 48) == dc.OK
        assert L.dctc_carver_batch_resize_width(None, 2, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_resize_width(b, -1, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_resize_width(b, 16, None) == dc.ERR_STATE                      # n_seams >= width
        assert L.dctc_carver_batch_images(b, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_energy(b, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_vmap(b, None, None) == dc.ERR_STATE                            # no dump_vmaps
        assert L.dctc_carver_batch_vmap(None, None, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_resize_width(b, 0, None) == dc.OK
        assert L.dctc_carver_batch_width(b) == 16 and L.dctc_carver_batch_width(None) == 0
        assert L.dctc_carver_batch_resize_width(b, 15, None) == dc.OK
        assert L.dctc_carver_batch_width(b) == 1
    finally:
        L.dctc_carver_batch_destroy(b)
    L.dctc_carver_batch_destroy(None)
    # wider than the seam DP's cluster covers: refused like the single session refuses it
    wide = 8 * 8 * (512 - 2 * 32) + 1
    frames = np.zeros((2, 2, wide), np.uint8)
    bt = dc.CarverBatch(ctx, frames)
    try:
        with pytest.raises(dc.DctcError) as e:
            bt.resize_width(1)
        assert e.value.status == dc.ERR_UNSUPPORTED
    finally:
        bt.close()
    ctx.carver_load(frames[0])
    with pytest.raises(dc.DctcError) as e:
        ctx.carver_resize_width(1)
    assert e.value.status == dc.ERR_UNSUPPORTED


def test_full_size_1080p_to_75_percent(ctx):
    """8 distinct 1920x1080 RGB frames, 480 seams each (the retarget of BASELINE config 3, frame by frame)."""
    frames = np.stack([ol.synth_image(1920, 1080, 3, 0xD0C7CA14 + i, 0) for i in range(8)])
    ctx.set_params(8, 0.5, 0.5)
    got = run_batch(ctx, frames, 480)
    assert got[1].shape == (8, 1080, 1440, 3)
    assert_matches_single(ctx, frames, 480, got)
