"""GPU tests of levels (dctc_carver_levels_width / _height, dctc_carver_render_levels and the batch's): liblqr's
interactive resize.  One seam loop to depth n keeps the start image and the visibility map; a render of any extent within
n of the start is then, bit for bit, what a fresh load and the resize or enlarge to that extent gives, and what a NumPy
gather over the start image and the map gives."""
import numpy as np
import pytest

import dct_carver_b200 as dc
import oracle_lib as ol
from test_carver_cpu import inflate_from_vmap

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)
    yield c
    c.close()


# ---- NumPy restatement -----------------------------------------------------------------------------------------------
def shrink_np(img, vmap, k):
    """The start image without the pixels of the first k seams: vs == 0 || vs > k, in their original order."""
    h, w, ch = img.shape
    keep = (vmap == 0) | (vmap > k)
    return img[keep].reshape(h, w - k, ch)


def inflate_np(img, vmap, m):
    """inflate_from_vmap (tests/test_carver_cpu.py) without the Python loop."""
    h, w, ch = img.shape
    flag = (vmap > 0) & (vmap <= m)
    pos = np.arange(w)[None, :] + np.cumsum(flag, axis=1)
    rows = np.broadcast_to(np.arange(h)[:, None], (h, w))
    out = np.zeros((h, w + m, ch), np.uint8)
    out[rows, pos] = img
    left = np.concatenate([img[:, :1], img[:, :-1]], axis=1).astype(np.int32)
    mean = ((left + img.astype(np.int32)) // 2).astype(np.uint8)
    mean[:, 0] = img[:, 0]
    out[rows[flag], pos[flag] - 1] = mean[flag]
    return out


def level_np(img, vmap, e):
    w = img.shape[1]
    return shrink_np(img, vmap, w - e) if e <= w else inflate_np(img, vmap, e - w)


def turn(a):
    return np.ascontiguousarray(np.swapaxes(a, -3, -2))


# ---- references ------------------------------------------------------------------------------------------------------
def fresh(ctx, img, axis, e, bias=None):
    """The image a fresh load (with bias) and the resize / enlarge to extent e along axis give."""
    ctx.carver_load(img)
    if bias is not None:
        ctx.carver_set_bias(bias)
    e0 = img.shape[1] if axis == "width" else img.shape[0]
    if e < e0:
        getattr(ctx, "carver_resize_" + axis)(e0 - e)
    elif e > e0:
        getattr(ctx, "carver_enlarge_" + axis)(e - e0)
    return ctx.carver_image()


def single_levels(ctx, img, axis, depth, extents, bias=None):
    """(seams, renders, vmap) of a single session's build and render."""
    ctx.carver_load(img)
    if bias is not None:
        ctx.carver_set_bias(bias)
    seams = getattr(ctx, "carver_levels_" + axis)(depth)
    h, w = img.shape[:2]
    vm, d = ctx.carver_vmap(w, h)
    assert d == depth
    return seams, ctx.carver_render_levels(extents), vm


def image(w, h, ch, seed, pattern=0):
    return ol.synth_image(w, h, ch, seed, pattern).reshape(h, w, ch)


def extents_for(e0, depth):
    ks = sorted({0, 1, depth // 2, depth - 1, depth})
    ms = sorted({1, depth // 2, depth})
    return [e0 - k for k in ks] + [e0 + m for m in ms]


def check_single(ctx, img, axis, depth):
    h, w, ch = img.shape
    e0 = w if axis == "width" else h
    ext = extents_for(e0, depth)
    seams, got, vm = single_levels(ctx, img, axis, depth, ext)
    ctx.carver_load(img)
    assert np.array_equal(seams, getattr(ctx, "carver_resize_" + axis)(depth))
    for e, g in zip(ext, got):
        assert g.shape == ((h, e, ch) if axis == "width" else (e, w, ch))
        if axis == "width":
            assert np.array_equal(g, level_np(img, vm, e)), ("numpy", e)
        else:
            assert np.array_equal(g, turn(level_np(turn(img), vm.T, e))), ("numpy", e)
        assert np.array_equal(g, fresh(ctx, img, axis, e)), ("session", e)
    return ext, got


def test_numpy_inflate_matches_the_loop_restatement():
    img = image(37, 11, 3, 5)
    rng = np.random.default_rng(3)
    vm = np.zeros((11, 37), np.int32)
    for y in range(11):
        vm[y, rng.permutation(37)[:9]] = np.arange(1, 10)
    for m in (1, 4, 9):
        assert np.array_equal(inflate_np(img, vm, m), inflate_from_vmap(img, vm, m))


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("w,h,depth", [(203, 61, 60), (204, 60, 71), (144, 50, 143)])
def test_width_levels_equal_fresh_sessions(ctx, ch, w, h, depth):
    ctx.set_params(8, 0.5, 0.5)
    check_single(ctx, image(w, h, ch, 1000 + w + ch), "width", depth)


@pytest.mark.parametrize("ch", [1, 2, 3, 4])
@pytest.mark.parametrize("w,h,depth", [(61, 203, 60), (60, 204, 71), (50, 144, 143)])
def test_height_levels_equal_fresh_sessions(ctx, ch, w, h, depth):
    ctx.set_params(8, 0.5, 0.5)
    img = image(w, h, ch, 2000 + h + ch)
    ext, got = check_single(ctx, img, "height", depth)
    # and the width levels of the transposed image, turned back
    _, want, _ = single_levels(ctx, turn(img), "width", depth, ext)
    for g, t in zip(got, want):
        assert np.array_equal(g, turn(t))


def test_full_hd_width_and_height_levels(ctx):
    ctx.set_params(8, 0.5, 0.5)
    img = image(1920, 1080, 3, 0x1920108)
    check_single(ctx, img, "width", 480)
    check_single(ctx, img, "height", 270)


def test_incremental_mode_levels(ctx):
    ctx.set_params(8, 0.5, 0.5)
    img = image(203, 96, 3, 77)
    ctx.carver_set_incremental(True)
    try:
        check_single(ctx, img, "width", 90)
    finally:
        ctx.carver_set_incremental(False)


def bias_plane(w, h, seed):
    rng = np.random.default_rng(seed)
    b = np.zeros((h, w), np.float32)
    b[:, w // 3: w // 3 + 12] = 5e4                      # preserve a band
    b[h // 4: h // 2, 2 * w // 3: 2 * w // 3 + 9] = -1e6    # discard a block
    return b + rng.random((h, w), dtype=np.float32)


@pytest.mark.parametrize("axis", ["width", "height"])
def test_biased_levels_equal_biased_fresh_sessions(ctx, axis):
    ctx.set_params(8, 0.5, 0.5)
    w, h = 150, 120
    img = image(w, h, 3, 88)
    bias = bias_plane(w, h, 8)
    e0, depth = (w, 60) if axis == "width" else (h, 50)
    ext = extents_for(e0, depth)
    _, got, _ = single_levels(ctx, img, axis, depth, ext, bias=bias)
    for e, g in zip(ext, got):
        assert np.array_equal(g, fresh(ctx, img, axis, e, bias=bias)), e
    # a biased batch gives every frame its biased single session's render
    frames = np.stack([img, image(w, h, 3, 89)])
    biases = np.stack([bias, bias_plane(w, h, 9)])
    b = dc.CarverBatch(ctx, frames)
    try:
        b.set_bias(biases)
        getattr(b, "levels_" + axis)(depth)
        got_b = b.render_levels(ext)
    finally:
        b.close()
    for i in range(2):
        _, want, _ = single_levels(ctx, frames[i], axis, depth, ext, bias=biases[i])
        for g, t in zip(got_b, want):
            assert np.array_equal(g[i], t)


# ---- batch -------------------------------------------------------------------------------------------------------------
def check_batch(ctx, frames, axis, depth, ext):
    n, h, w, ch = frames.shape
    b = dc.CarverBatch(ctx, frames)
    try:
        seams = getattr(b, "levels_" + axis)(depth)
        got = b.render_levels(ext)
        d = ctx.dev_alloc(sum(g.nbytes for g in got))
        try:
            nbytes = b.render_levels_dev(ext, d)
            flat = np.empty(nbytes, np.uint8)
            ctx.d2h(flat, d)
        finally:
            ctx.dev_free(d)
    finally:
        b.close()
    assert np.array_equal(flat, np.concatenate([g.ravel() for g in got]))
    for i in range(n):
        s, want, _ = single_levels(ctx, frames[i], axis, depth, ext)
        assert np.array_equal(seams[i], s), i
        for e, g, t in zip(ext, got, want):
            assert g.shape == (n,) + t.shape
            assert np.array_equal(g[i], t), (i, e)


@pytest.mark.parametrize("axis", ["width", "height"])
def test_batch_mixed_extents_equal_single_sessions(ctx, axis):
    ctx.set_params(8, 0.5, 0.5)
    frames = np.stack([image(203, 144, 3, 500 + i, i % 4) for i in range(3)])
    e0 = 203 if axis == "width" else 144
    ext = [e0 - 5, e0 + 7, e0, e0 - 60, e0 + 60, e0 - 5, e0 + 1, e0 - 1, e0 + 7]
    check_batch(ctx, frames, axis, 60, ext)


def test_batch_full_hd(ctx):
    ctx.set_params(8, 0.5, 0.5)
    frames = np.stack([image(1920, 1080, 3, 0x1920108 + i) for i in range(8)])
    ext = [1700, 2400, 1440, 1920, 2100, 1500, 1700]
    check_batch(ctx, frames, "width", 480, ext)


def test_more_shrink_levels_than_one_launch_takes(ctx):
    """40 shrink extents: two gather launches, every level still right."""
    ctx.set_params(8, 0.5, 0.5)
    img = image(180, 70, 3, 321)
    ext = list(range(180, 140, -1))
    ctx.carver_load(img)
    ctx.carver_levels_width(40)
    vm, _ = ctx.carver_vmap(180, 70)
    before = ctx.launches
    got = ctx.carver_render_levels(ext)
    assert ctx.launches - before == 2
    for e, g in zip(ext, got):
        assert np.array_equal(g, shrink_np(img, vm, 180 - e)), e


# ---- rules ----------------------------------------------------------------------------------------------------------
def status(fn, *args):
    with pytest.raises(dc.DctcError) as e:
        fn(*args)
    return e.value.status


@pytest.mark.parametrize("axis", ["width", "height"])
def test_launch_counts(ctx, axis):
    ctx.set_params(8, 0.5, 0.5)
    img = image(160, 120, 3, 42)
    e0, depth = (160, 30) if axis == "width" else (120, 30)
    ctx.carver_set_dump_vmaps(True)
    try:
        ctx.carver_load(img)
        before = ctx.launches
        getattr(ctx, "carver_resize_" + axis)(depth)
        want = ctx.launches - before
    finally:
        ctx.carver_set_dump_vmaps(False)
    ctx.carver_load(img)
    before = ctx.launches
    getattr(ctx, "carver_levels_" + axis)(depth)
    assert ctx.launches - before == want
    per_level = 1 if axis == "height" else 0
    for ext, gathers, inflates in (([e0 - 3, e0 - 30, e0], 1, 0), ([e0 + 4, e0 + 30], 0, 2),
                                   ([e0 + 4, e0 - 3, e0 + 4, e0, e0 - 3], 1, 2)):
        before = ctx.launches
        ctx.carver_render_levels(ext)
        assert ctx.launches - before == gathers + inflates + per_level * len(ext), ext


def test_rules_single_session(ctx):
    ctx.set_params(8, 0.5, 0.5)
    L = dc.lib()
    w, h, depth = 160, 90, 40
    img = image(w, h, 3, 7)
    # no session, or a session without a build: STATE
    other = dc.Context(0)
    try:
        assert status(other.carver_render_levels, [w]) == dc.ERR_STATE
        assert status(other.carver_levels_width, 3) == dc.ERR_STATE
    finally:
        other.close()
    ctx.carver_load(img)
    assert status(ctx.carver_render_levels, [w]) == dc.ERR_STATE
    assert L.dctc_carver_levels_width(ctx.handle, -1, None) == dc.ERR_INVALID
    assert L.dctc_carver_levels_width(None, 1, None) == dc.ERR_INVALID
    assert status(ctx.carver_levels_width, w) == dc.ERR_STATE
    assert status(ctx.carver_levels_height, h) == dc.ERR_STATE
    # after a seam operation: STATE
    ctx.carver_resize_width(1)
    assert status(ctx.carver_levels_width, 3) == dc.ERR_STATE
    # the build
    ctx.carver_load(img)
    ctx.carver_levels_width(depth)
    got = ctx.carver_render_levels([w - depth, w, w + depth])
    size, im, en, eimg = ctx.carver_size(), ctx.carver_image(), ctx.carver_energy(), ctx.carver_energy_image()
    vm = ctx.carver_vmap(w, h)
    painted = ctx.carver_paint_seams(img)
    ctx.carver_set_dump_vmaps(True)
    try:
        ctx.carver_load(img)
        ctx.carver_resize_width(depth)
        assert size == ctx.carver_size() == (w - depth, h)
        assert np.array_equal(im, ctx.carver_image())
        assert np.array_equal(en, ctx.carver_energy())
        assert np.array_equal(eimg, ctx.carver_energy_image())
        want_vm = ctx.carver_vmap(w, h)
        assert vm[1] == want_vm[1] == depth and np.array_equal(vm[0], want_vm[0])
        assert np.array_equal(painted, ctx.carver_paint_seams(img))
    finally:
        ctx.carver_set_dump_vmaps(False)
    ctx.carver_load(img)
    ctx.carver_levels_width(depth)
    # argument checks
    ext = np.array([w], np.int32)
    out = np.empty(w * h * 3, np.uint8)
    assert L.dctc_carver_render_levels(ctx.handle, 0, ext.ctypes.data, out.ctypes.data) == dc.ERR_INVALID
    assert L.dctc_carver_render_levels(ctx.handle, 1, None, out.ctypes.data) == dc.ERR_INVALID
    assert L.dctc_carver_render_levels(ctx.handle, 1, ext.ctypes.data, None) == dc.ERR_INVALID
    for bad in (0, -4):
        assert status(ctx.carver_render_levels, [w, bad]) == dc.ERR_INVALID
    for far in (w - depth - 1, w + depth + 1):
        assert status(ctx.carver_render_levels, [w, far]) == dc.ERR_STATE
    # every seam operation, the combined resize, the bias and another build: STATE; the session stays as it was
    for fn, args in ((ctx.carver_resize_width, (0,)), (ctx.carver_resize_width, (1,)), (ctx.carver_enlarge_width, (1,)),
                     (ctx.carver_resize_height, (1,)), (ctx.carver_enlarge_height, (1,)), (ctx.carver_resize, (w - 1, h)),
                     (ctx.carver_set_bias, (np.zeros((h, w - depth), np.float32),)), (ctx.carver_levels_width, (1,)),
                     (ctx.carver_levels_height, (1,)), (ctx.carver_levels_width, (0,)),
                     (ctx.carve_and_update, (np.zeros(h, np.int32),))):
        assert status(fn, *args) == dc.ERR_STATE, fn.__name__
    assert ctx.carver_size() == size and np.array_equal(ctx.carver_image(), im)
    # renders are repeatable, change nothing, and survive dctc_set_params (which rebuilds the energy map)
    for _ in range(2):
        again = ctx.carver_render_levels([w - depth, w, w + depth])
        assert all(np.array_equal(a, b) for a, b in zip(got, again))
        assert ctx.carver_size() == size and np.array_equal(ctx.carver_image(), im)
        assert np.array_equal(ctx.carver_energy(), en)
    ctx.set_params(4, 0.5, 0.5)
    try:
        assert np.array_equal(ctx.carver_energy(), ctx.energy_full(im))
        again = ctx.carver_render_levels([w - depth, w, w + depth])
        assert all(np.array_equal(a, b) for a, b in zip(got, again))
    finally:
        ctx.set_params(8, 0.5, 0.5)
    # a load drops the levels
    ctx.carver_load(img)
    assert status(ctx.carver_render_levels, [w]) == dc.ERR_STATE
    # depth 0: only the start extent renders, as the loaded image
    ctx.carver_levels_height(0)
    assert ctx.carver_size() == (w, h)
    (same,) = ctx.carver_render_levels([h])
    assert np.array_equal(same, img)
    for far in (h - 1, h + 1):
        assert status(ctx.carver_render_levels, [far]) == dc.ERR_STATE


def test_unsupported_width_leaves_the_session_loaded(ctx):
    ctx.set_params(8, 0.5, 0.5)
    wide = 8 * 8 * (512 - 2 * 32) + 1
    img = np.random.default_rng(5).integers(0, 256, (2, wide, 1), dtype=np.uint8)
    ctx.carver_load(img)
    assert status(ctx.carver_levels_width, 1) == dc.ERR_UNSUPPORTED
    assert ctx.carver_size() == (wide, 2)
    assert np.array_equal(ctx.carver_image(), img)
    b = dc.CarverBatch(ctx, np.stack([img[..., 0]] * 2))
    try:
        assert status(b.levels_width, 1) == dc.ERR_UNSUPPORTED
        assert b.width == wide
        assert np.array_equal(b.images()[..., 0], np.stack([img[..., 0]] * 2))
    finally:
        b.close()


@pytest.mark.parametrize("dump_vmaps", [False, True])
def test_rules_batch(ctx, dump_vmaps):
    ctx.set_params(8, 0.5, 0.5)
    L = dc.lib()
    w, h, depth = 120, 80, 30
    frames = np.stack([image(w, h, 3, 60 + i) for i in range(2)])
    b = dc.CarverBatch(ctx, frames, dump_vmaps=dump_vmaps)
    try:
        assert status(b.render_levels, [w]) == dc.ERR_STATE
        assert L.dctc_carver_batch_levels_width(None, 1, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_levels_height(b.handle, -1, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_render_levels_dev(b.handle, 1, None, None) == dc.ERR_INVALID
        assert status(b.levels_height, h) == dc.ERR_STATE
        b.resize_width(2)
        assert status(b.levels_width, 2) == dc.ERR_STATE
        b.load(frames)
        b.levels_height(depth)
        assert (b.width, b.height) == (w, h - depth)
        if dump_vmaps:
            vm, d = b.vmap()
            assert d == depth
            for i in range(2):
                ctx.carver_load(frames[i])
                ctx.carver_levels_height(depth)
                assert np.array_equal(vm[i], ctx.carver_vmap(w, h)[0])
        else:
            assert status(b.vmap) == dc.ERR_STATE
        for fn, args in ((b.resize_width, (0,)), (b.resize_height, (1,)), (b.enlarge_height, (1,)), (b.resize, (w, h - 1)),
                         (b.set_bias, (None,)), (b.levels_height, (1,)), (b.levels_width, (1,))):
            assert status(fn, *args) == dc.ERR_STATE, fn.__name__
        for far in (h - depth - 1, h + depth + 1):
            assert status(b.render_levels, [h, far]) == dc.ERR_STATE
        got = b.render_levels([h - depth, h + depth, h])
        assert np.array_equal(got[2], frames)
        before = ctx.launches
        again = b.render_levels([h - depth, h + depth, h])
        assert ctx.launches - before == 1 + 1 + 3
        assert all(np.array_equal(x, y) for x, y in zip(got, again))
        im = b.images()
        b.load(frames)
        assert status(b.render_levels, [h]) == dc.ERR_STATE
        b.resize_height(depth)
        assert np.array_equal(b.images(), im)
    finally:
        b.close()
