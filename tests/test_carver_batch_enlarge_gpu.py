"""GPU tests of enlarging a batch (dctc_carver_batch_enlarge_width, CarverBatch.enlarge_width): n equally sized frames
made wider by one device seam loop plus one inflate launch.  The reference for every frame is a single carver session
on the same context (carver_load + carver_enlarge_width); every frame must match it bit for bit in seams, enlarged
image, energy plane of the enlarged frame and the start frame's visibility map."""
import ctypes as C

import numpy as np
import pytest

import dct_carver_b200 as dc
import oracle_lib as ol
from test_carver_batch_gpu import DP_VARIANT_SIZES
from test_carver_cpu import inflate_from_vmap

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    # same arithmetic as the single session's references in test_k2_gpu.py (FP32 march + FP32 tile kernels)
    c = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)
    yield c
    c.close()


def single(ctx, frame, k):
    """(seams [k, h], image [h, w + k, ch], energy [h, w + k], (vmap [h, w], depth)) of one single-frame session."""
    h, w = frame.shape[:2]
    ctx.carver_load(frame)
    seams = ctx.carver_enlarge_width(k)
    return seams, ctx.carver_image(), ctx.carver_energy(), ctx.carver_vmap(w, h)


def run_batch(ctx, frames, k, vmaps=True):
    b = dc.CarverBatch(ctx, frames, dump_vmaps=vmaps)
    try:
        seams = b.enlarge_width(k)
        assert b.width == frames.shape[2] + k
        return seams, b.images(), b.energy(), (b.vmap() if vmaps else None)
    finally:
        b.close()


def assert_matches_single(ctx, frames, k, got, inflate=False):
    seams, imgs, en, vm = got
    n, h, w = frames.shape[:3]
    assert seams.shape == (n, k, h)
    assert imgs.shape[:3] == (n, h, w + k) and en.shape == (n, h, w + k)
    for i, f in enumerate(frames):
        s, im, e, (v, depth) = single(ctx, f, k)
        assert depth == k
        assert np.array_equal(seams[i], s), "frame %d: seams" % i
        assert np.array_equal(imgs[i].reshape(im.shape), im), "frame %d: image" % i
        assert np.array_equal(en[i], e), "frame %d: energy" % i
        if vm is not None:
            assert vm[1] == k
            assert np.array_equal(vm[0][i], v), "frame %d: visibility map" % i
        if inflate:
            assert np.array_equal(im, inflate_from_vmap(f.reshape(h, w, -1), v, k)), "frame %d: pixel synthesis" % i


def frames_of(w, h, ch, seeds, patterns=(0,)):
    fs = [ol.synth_image(w, h, ch, s, patterns[i % len(patterns)]) for i, s in enumerate(seeds)]
    return np.stack(fs)


@pytest.mark.parametrize("b", [2, 4, 8, 16])
@pytest.mark.parametrize("ch", [1, 3, 4])
def test_small_frames_equal_single_sessions(ctx, b, ch):
    frames = frames_of(97, 75, ch, [110 + 7 * b + ch, 210 + b, 310 + ch], patterns=(0, 3, 1))
    ctx.set_params(b, 0.5, 0.5)
    assert_matches_single(ctx, frames, 20, run_batch(ctx, frames, 20), inflate=True)


@pytest.mark.parametrize("k", [1, 96])
def test_one_seam_and_all_but_one_column(ctx, k):
    frames = frames_of(97, 75, 3, [401, 402, 403], patterns=(0, 3, 1))
    ctx.set_params(8, 0.5, 0.5)
    assert_matches_single(ctx, frames, k, run_batch(ctx, frames, k), inflate=True)


def test_non_uniform_weights_equal_single_sessions(ctx):
    frames = frames_of(120, 64, 3, [21, 22, 23, 24])
    ctx.set_params(8, 0.8, 0.2)
    try:
        assert_matches_single(ctx, frames, 15, run_batch(ctx, frames, 15))
    finally:
        ctx.set_params(8, 0.5, 0.5)


# the seam DP's strip widths and energy staging variants (the width map of test_carver_batch_gpu.py)
@pytest.mark.parametrize("w,h", DP_VARIANT_SIZES)
def test_strip_widths_and_staging_variants(ctx, w, h):
    frames = frames_of(w, h, 1, [w + 11, w + 12, w + 13], patterns=(0, 2, 0))
    ctx.set_params(8, 0.5, 0.5)
    assert_matches_single(ctx, frames, 3, run_batch(ctx, frames, 3))


def test_tall_frames_take_the_serial_backtrack(ctx):
    """2800 rows: the trace kernel's cone would exceed 200 KB of shared memory, so the DP kernel walks the seam back
    itself, per frame."""
    frames = frames_of(64, 2800, 3, [43, 44])
    ctx.set_params(8, 0.5, 0.5)
    assert_matches_single(ctx, frames, 4, run_batch(ctx, frames, 4))


def test_permuted_frames_give_permuted_results(ctx):
    frames = frames_of(150, 90, 3, [55, 56, 57, 58], patterns=(0, 1, 3, 0))
    ctx.set_params(8, 0.5, 0.5)
    a = run_batch(ctx, frames, 12)
    perm = np.array([2, 0, 3, 1])
    b = run_batch(ctx, frames[perm], 12)
    for x, y in zip(a[:3], b[:3]):
        assert np.array_equal(x[perm], y)
    assert a[3][1] == b[3][1] == 12 and np.array_equal(a[3][0][perm], b[3][0])


def test_identical_frames_give_identical_results(ctx):
    f = ol.synth_image(130, 70, 3, 63, 0)
    frames = np.stack([f] * 5)
    ctx.set_params(8, 0.5, 0.5)
    got = run_batch(ctx, frames, 10)
    for x in got[:3] + (got[3][0],):
        assert all(np.array_equal(x[0], x[i]) for i in range(1, 5))
    assert_matches_single(ctx, frames[:1], 10, tuple(x[:1] for x in got[:3]) + (None,))


def test_batch_without_visibility_maps_enlarges_the_same(ctx):
    frames = frames_of(140, 80, 3, [85, 86, 87])
    ctx.set_params(8, 0.5, 0.5)
    with_maps = run_batch(ctx, frames, 17, vmaps=True)
    fresh = dc.CarverBatch(ctx, frames, dump_vmaps=False)
    try:
        before = ctx.launches
        want = (fresh.resize_width(5), fresh.images(), fresh.energy())
        shrink_launches = ctx.launches - before
    finally:
        fresh.close()
    b = dc.CarverBatch(ctx, frames, dump_vmaps=False)
    try:
        got = (b.enlarge_width(17), b.images(), b.energy())
        with pytest.raises(dc.DctcError) as e:
            b.vmap()
        assert e.value.status == dc.ERR_STATE
        # after a reload the batch shrinks as one that never enlarged (no visibility-map updates either)
        b.load(frames)
        before = ctx.launches
        again = (b.resize_width(5), b.images(), b.energy())
        assert ctx.launches - before == shrink_launches
        with pytest.raises(dc.DctcError) as e:
            b.vmap()
        assert e.value.status == dc.ERR_STATE
    finally:
        b.close()
    for x, y in zip(got, with_maps[:3]):
        assert np.array_equal(x, y)
    for x, y in zip(again, want):
        assert np.array_equal(x, y)


def test_load_after_enlarge_restarts_the_batch(ctx):
    frames = frames_of(140, 80, 3, [91, 92, 93])
    other = frames_of(140, 80, 3, [94, 95, 96], patterns=(1, 0, 3))
    ctx.set_params(8, 0.5, 0.5)
    b = dc.CarverBatch(ctx, frames, dump_vmaps=True)
    try:
        first = (b.enlarge_width(9), b.images(), b.energy(), b.vmap())
        # the same frames again: the buffers of the first enlarge are reused
        for _ in range(2):
            b.load(frames)
            assert b.width == 140
            again = (b.enlarge_width(9), b.images(), b.energy(), b.vmap())
            for x, y in zip(first[:3], again[:3]):
                assert np.array_equal(x, y)
            assert again[3][1] == 9 and np.array_equal(first[3][0], again[3][0])
        # another seam count: the enlarged frames' buffers are reallocated
        b.load(frames)
        other_k = (b.enlarge_width(4), b.images(), b.energy(), b.vmap())
        # then a shrink of other frames: what a fresh batch gives
        b.load(other)
        assert b.width == 140
        got = (b.resize_width(13), b.images(), b.energy(), b.vmap())
    finally:
        b.close()
    fresh = dc.CarverBatch(ctx, other, dump_vmaps=True)
    try:
        want = (fresh.resize_width(13), fresh.images(), fresh.energy(), fresh.vmap())
    finally:
        fresh.close()
    for x, y in zip(got[:3], want[:3]):
        assert np.array_equal(x, y)
    assert got[3][1] == want[3][1] == 13 and np.array_equal(got[3][0], want[3][0])
    want_k = run_batch(ctx, frames, 4)
    for x, y in zip(other_k[:3], want_k[:3]):
        assert np.array_equal(x, y)
    assert other_k[3][1] == 4 and np.array_equal(other_k[3][0], want_k[3][0])


@pytest.mark.parametrize("vmaps", [False, True])
def test_launch_count_does_not_grow_with_the_frame_count(ctx, vmaps):
    ctx.set_params(8, 0.5, 0.5)
    growth = []
    for n in (1, 8):
        b = dc.CarverBatch(ctx, frames_of(200, 100, 3, range(190, 190 + n)), dump_vmaps=vmaps)
        try:
            before = ctx.launches
            b.enlarge_width(6)
            growth.append(ctx.launches - before)
        finally:
            b.close()
    assert growth[0] == growth[1] > 0


def test_single_session_survives_batch_enlarge(ctx):
    img = ol.synth_image(150, 90, 3, 99, 0)
    ctx.set_params(8, 0.5, 0.5)
    ctx.carver_load(img)
    ctx.carver_resize_width(5)
    size, im, en = ctx.carver_size(), ctx.carver_image(), ctx.carver_energy()
    b = dc.CarverBatch(ctx, frames_of(150, 90, 3, [100, 101]))
    b.enlarge_width(7)
    b.close()
    assert ctx.carver_size() == size
    assert np.array_equal(ctx.carver_image(), im)
    assert np.array_equal(ctx.carver_energy(), en)
    # the single session carries on as if no batch had run
    more = ctx.carver_resize_width(4)
    ctx.carver_load(img)
    want = ctx.carver_resize_width(9)
    assert np.array_equal(more, want[5:])


def test_errors(ctx):
    L = dc.lib()
    ctx.set_params(8, 0.5, 0.5)
    out = C.c_void_p()
    assert L.dctc_carver_batch_enlarge_width(None, 1, None) == dc.ERR_INVALID
    assert L.dctc_carver_batch_create(ctx.handle, 2, 16, 8, 3, 1, C.byref(out)) == dc.OK
    b = out
    try:
        imgs = frames_of(16, 8, 3, [1, 2])
        assert L.dctc_carver_batch_enlarge_width(b, 2, None) == dc.ERR_STATE                      # before a load
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 48) == dc.OK
        assert L.dctc_carver_batch_enlarge_width(b, -1, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_enlarge_width(b, 0, None) == dc.OK
        assert L.dctc_carver_batch_width(b) == 16
        assert L.dctc_carver_batch_enlarge_width(b, 16, None) == dc.ERR_STATE                     # n_seams >= width
        assert L.dctc_carver_batch_resize_width(b, 2, None) == dc.OK
        assert L.dctc_carver_batch_enlarge_width(b, 2, None) == dc.ERR_STATE                      # not at the loaded width
        assert L.dctc_carver_batch_width(b) == 14
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 48) == dc.OK
        seams = np.empty(2 * 15 * 8, np.int32)
        assert L.dctc_carver_batch_enlarge_width(b, 15, seams.ctypes.data) == dc.OK              # w - 1 seams
        assert L.dctc_carver_batch_width(b) == 31
        # the enlarged frames stay readable; neither a resize nor another enlarge continues from them
        for fn in (L.dctc_carver_batch_enlarge_width, L.dctc_carver_batch_resize_width):
            for k in (0, 1):
                assert fn(b, k, None) == dc.ERR_STATE, (fn, k)
        assert L.dctc_carver_batch_width(b) == 31
        buf = np.empty(2 * 8 * 31 * 3, np.uint8)
        en = np.empty(2 * 8 * 31, np.float32)
        depth = C.c_int(0)
        assert L.dctc_carver_batch_images(b, buf.ctypes.data) == dc.OK
        assert L.dctc_carver_batch_energy(b, en.ctypes.data) == dc.OK
        assert L.dctc_carver_batch_vmap(b, None, C.byref(depth)) == dc.OK and depth.value == 15
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 48) == dc.OK
        assert L.dctc_carver_batch_width(b) == 16
        assert L.dctc_carver_batch_resize_width(b, 3, None) == dc.OK
    finally:
        L.dctc_carver_batch_destroy(b)
    # wider than the seam DP's cluster covers: refused before any work, the batch stays loaded with its frames
    wide = 8 * 8 * (512 - 2 * 32) + 1
    frames = np.random.default_rng(5).integers(0, 256, (2, 2, wide), dtype=np.uint8)
    bt = dc.CarverBatch(ctx, frames)
    try:
        en = bt.energy()
        with pytest.raises(dc.DctcError) as e:
            bt.enlarge_width(1)
        assert e.value.status == dc.ERR_UNSUPPORTED
        assert bt.width == wide
        assert np.array_equal(bt.images()[..., 0], frames)
        assert np.array_equal(bt.energy(), en)
    finally:
        bt.close()


def test_full_size_4_3_to_16_9(ctx):
    """8 distinct 1440x1080 RGB frames enlarged to 1920x1080 (480 seams each)."""
    frames = np.stack([ol.synth_image(1440, 1080, 3, 0xE41A26E0 + i, 0) for i in range(8)])
    ctx.set_params(8, 0.5, 0.5)
    got = run_batch(ctx, frames, 480)
    assert got[1].shape == (8, 1080, 1920, 3)
    assert_matches_single(ctx, frames, 480, got)
