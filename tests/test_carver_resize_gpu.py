"""GPU tests of both axes in one call (dctc_carver_resize, dctc_carver_batch_resize).  The reference is the chain of
per-axis calls the plan stands for, with a host reload at the start of each axis: load, the width passes, carver_image,
load, the height passes.  Every pass's seams and visibility map and the final image, energy plane and energy image must
match it bit for bit; every frame of a batch must match its single session's dctc_carver_resize."""
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


def image(w, h, ch, seed, pattern=0):
    return ol.synth_image(w, h, ch, seed, pattern).reshape(h, w, ch)


def final(ctx):
    return dict(image=ctx.carver_image(), energy=ctx.carver_energy(), energy_image=ctx.carver_energy_image())


def chain(ctx, img, new_w, new_h, vmaps=False):
    """The per-axis calls of the plan with a host reload at each axis: (passes, final frame, launches of the seam calls
    and map reads)."""
    h, w = img.shape[:2]
    calls = {("width", False): ctx.carver_resize_width, ("width", True): ctx.carver_enlarge_width,
             ("height", False): ctx.carver_resize_height, ("height", True): ctx.carver_enlarge_height}
    passes, axis, launches = [], None, 0
    cur = img
    try:
        for p in dc.resize_plan(w, h, new_w, new_h):
            if p["axis"] != axis:
                ctx.carver_load(cur)
                ctx.carver_set_dump_vmaps(vmaps)
                axis = p["axis"]
            n0 = ctx.launches
            e = dict(axis=p["axis"], enlarge=p["enlarge"], seams=calls[(p["axis"], p["enlarge"])](p["n_seams"]))
            if vmaps:
                vm, depth = ctx.carver_vmap(p["w"], p["h"])
                assert depth == p["n_seams"]
                e["vmap"] = vm
            launches += ctx.launches - n0
            passes.append(e)
            cur = ctx.carver_image()
    finally:
        ctx.carver_set_dump_vmaps(False)
    if not passes:
        ctx.carver_load(img)
    return passes, final(ctx), launches


def combined(ctx, img, new_w, new_h, vmaps=False):
    ctx.carver_load(img)
    n0 = ctx.launches
    passes = ctx.carver_resize(new_w, new_h, vmaps=vmaps)
    launches = ctx.launches - n0
    return passes, final(ctx), launches


def assert_passes_equal(got, want):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.keys() == w.keys(), i
        assert (g["axis"], g["enlarge"]) == (w["axis"], w["enlarge"]), i
        for k in ("seams", "vmap"):
            if k in w:
                assert g[k].shape == w[k].shape, (i, k)
                assert np.array_equal(g[k], w[k]), (i, k)


def assert_final_equal(got, want):
    for k in want:
        assert got[k].shape == want[k].shape, k
        assert np.array_equal(got[k], want[k]), k


def check(ctx, img, new_w, new_h, vmaps=True):
    got_p, got_f, got_n = combined(ctx, img, new_w, new_h, vmaps)
    want_p, want_f, want_n = chain(ctx, img, new_w, new_h, vmaps)
    assert got_f["image"].shape[:2] == (new_h, new_w)
    assert_passes_equal(got_p, want_p)
    assert_final_equal(got_f, want_f)
    assert got_n == want_n          # the same launches: per-seam work, axis switch, maps on the way out
    return got_p


# ---- single session against the per-axis chain ------------------------------------------------------------------------

TARGETS = [(70, 55), (85, 40), (65, 75)]   # from 90 x 70: shrink/shrink, enlarge/shrink, shrink/enlarge


@pytest.mark.parametrize("b", [2, 4, 8, 16])
@pytest.mark.parametrize("ch", [1, 2, 3, 4])
def test_resize_equals_the_per_axis_chain(ctx, b, ch):
    img = image(90, 70, ch, 2000 + 10 * b + ch, pattern=(b + ch) % 4)
    ctx.set_params(b, 0.5, 0.5)
    new_w, new_h = TARGETS[(b + ch) % 3]
    passes = check(ctx, img, new_w, new_h)
    assert [p["axis"] for p in passes] == ["width", "height"]


@pytest.mark.parametrize("target", [(130, 30), (40, 70), (130, 70), (25, 95), (79, 59), (80, 60)])
def test_multi_pass_enlarges(ctx, target):
    """40 x 30 -> 130 wide takes passes of 39 and 51 seams; 30 -> 70 tall 29 and 11; 2w - 1 and 2w exactly."""
    img = image(40, 30, 3, 2101)
    ctx.set_params(8, 0.5, 0.5)
    passes = check(ctx, img, *target)
    assert len(passes) == len(dc.resize_plan(40, 30, *target))


def test_non_uniform_weights(ctx):
    img = image(100, 80, 3, 2201, pattern=1)
    ctx.set_params(8, 0.8, 0.2)
    try:
        check(ctx, img, 120, 64)
    finally:
        ctx.set_params(8, 0.5, 0.5)


@pytest.mark.parametrize("target", [(70, 80), (110, 50)])
def test_incremental_mode(ctx, target):
    img = image(90, 70, 3, 2301)
    ctx.set_params(8, 0.5, 0.5)
    ctx.carver_set_incremental(True)
    try:
        check(ctx, img, *target)
    finally:
        ctx.carver_set_incremental(False)


def test_without_maps_and_one_axis(ctx):
    img = image(90, 70, 3, 2401)
    ctx.set_params(8, 0.5, 0.5)
    for target in ((60, 50), (90, 40), (60, 70), (150, 70)):
        passes = check(ctx, img, *target, vmaps=False)
        assert all("vmap" not in p for p in passes)


def test_dump_vmaps_setting_does_not_matter(ctx):
    img = image(64, 48, 3, 2501)
    ctx.set_params(8, 0.5, 0.5)
    want = combined(ctx, img, 50, 40, vmaps=True)
    ctx.carver_load(img)
    ctx.carver_set_dump_vmaps(True)
    try:
        got = ctx.carver_resize(50, 40)
    finally:
        ctx.carver_set_dump_vmaps(False)
    assert_passes_equal(got, [{k: v for k, v in p.items() if k != "vmap"} for p in want[0]])
    assert_final_equal(final(ctx), want[1])


def test_each_axis_switch_adds_one_transpose_and_one_k1(ctx):
    img = image(120, 90, 3, 2601)
    ctx.set_params(8, 0.5, 0.5)
    ctx.carver_load(img)
    n0 = ctx.launches
    ctx.carver_resize_width(20)
    width = ctx.launches - n0
    mid = ctx.carver_image()
    ctx.carver_load(np.ascontiguousarray(np.swapaxes(mid, 0, 1)))   # the height passes as width calls on the transpose
    n0 = ctx.launches
    ctx.carver_resize_width(15)
    height = ctx.launches - n0
    ctx.carver_load(img)
    n0 = ctx.launches
    ctx.carver_resize(100, 75)
    assert ctx.launches - n0 == width + height + 2


def test_one_axis_plans_match_the_host_carver(ctx):
    """host.render (the host carver with its device loop, reloading between passes) along one axis, including its
    multi-pass enlarge: the seams of all passes and the image."""
    from dct_carver_b200 import host
    img = image(40, 30, 3, 2701)
    ctx.set_params(8, 0.5, 0.5)
    for seams_number, vertically in ((90, False), (-12, False), (45, True), (-9, True)):
        want = host.render(img, seams_number, 8, 0.5, 0.5, vertically=vertically, ctx=ctx)
        ctx.carver_load(img)
        new_w, new_h = (40, 30 + seams_number) if vertically else (40 + seams_number, 30)
        passes = ctx.carver_resize(new_w, new_h)
        assert np.array_equal(np.concatenate([p["seams"] for p in passes]), want["seams"]), (seams_number, vertically)
        assert np.array_equal(ctx.carver_image(), want["image"]), (seams_number, vertically)


def test_after_the_call(ctx):
    """Getters, dctc_pixel_energy and dctc_set_params work on the final frame; seam operations, maps and painting
    wait for the next load."""
    L = dc.lib()
    h = ctx.handle
    img = image(80, 60, 3, 2801)
    ctx.set_params(8, 0.5, 0.5)
    want = chain(ctx, img, 70, 66)[1]
    ctx.carver_load(img)
    ctx.carver_resize(70, 66, vmaps=True)
    assert ctx.carver_size() == (70, 66)
    assert_final_equal(final(ctx), want)
    p = dc.CarverEnergyParams()
    p.base.edges, p.base.textures, p.base.blocksize = 0.5, 0.5, 8
    p.gpu = h.value
    for x, y in [(0, 0), (69, 65), (31, 17)]:
        assert L.dctc_pixel_energy(x, y, 70, 66, None, C.byref(p)) == want["energy"][y, x]
    ctx.set_params(4, 0.6, 0.4)
    try:   # the final frame is a height pass's: its map is the transposed image's, turned back
        t = np.ascontiguousarray(np.swapaxes(want["image"], 0, 1))
        assert np.array_equal(ctx.carver_energy(), np.ascontiguousarray(ctx.energy_full(t).T))
    finally:
        ctx.set_params(8, 0.5, 0.5)
    for fn in (L.dctc_carver_resize_width, L.dctc_carver_resize_height, L.dctc_carver_enlarge_width,
               L.dctc_carver_enlarge_height):
        assert fn(h, 1, None) == dc.ERR_STATE
    assert L.dctc_carver_resize(h, 60, 60, None, None) == dc.ERR_STATE
    assert L.dctc_carver_resize(h, 70, 66, None, None) == dc.ERR_STATE
    vm = np.empty(80 * 60, np.int32)
    assert L.dctc_carver_vmap(h, vm.ctypes.data, None) == dc.ERR_STATE
    assert L.dctc_carver_paint_seams(h, img.ctypes.data, 3, 240) == dc.ERR_STATE
    seam = np.zeros(66, np.int32)
    assert L.dctc_carve_and_update(h, seam.ctypes.data, None, None, None) == dc.ERR_STATE
    ctx.carver_load(img)                                                      # a load starts over
    assert ctx.carver_resize_width(3).shape == (3, 60)


def test_states_and_errors(ctx):
    L = dc.lib()
    h = ctx.handle
    ctx.set_params(8, 0.5, 0.5)
    fresh = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)   # nothing loaded
    try:
        assert L.dctc_carver_resize(fresh.handle, 10, 10, None, None) == dc.ERR_STATE
    finally:
        fresh.close()
    assert L.dctc_carver_resize(None, 10, 10, None, None) == dc.ERR_INVALID
    img = image(48, 32, 3, 2901)
    ctx.carver_load(img)
    for nw, nh in ((0, 32), (48, 0), (-1, 5)):
        assert L.dctc_carver_resize(h, nw, nh, None, None) == dc.ERR_INVALID
    n0 = ctx.launches
    assert L.dctc_carver_resize(h, 48, 32, None, None) == dc.OK                # nothing changes
    assert ctx.launches == n0 and ctx.carver_size() == (48, 32)
    assert ctx.carver_resize(40, 30)[0]["seams"].shape == (8, 32)            # the no-op left the session fresh
    # a seam operation since the load
    for op in (lambda: ctx.carver_resize_width(1), lambda: ctx.carver_enlarge_height(2),
               lambda: ctx.carve_and_update(np.full(32, 5, np.int32), want_band=False)):
        ctx.carver_load(img)
        op()
        assert L.dctc_carver_resize(h, 40, 30, None, None) == dc.ERR_STATE
    # an extent of 1 cannot grow
    ctx.carver_load(image(1, 32, 3, 2902))
    assert L.dctc_carver_resize(h, 3, 32, None, None) == dc.ERR_STATE
    assert ctx.carver_size() == (1, 32)
    # a pass wider than the seam DP covers: refused on the plan before any work, the session stays loaded and fresh
    ctx.carver_load(np.zeros((4, 20000), np.uint8))          # enlarge passes from 20000 (fine) and 39999 (too wide)
    assert L.dctc_carver_resize(h, 50000, 4, None, None) == dc.ERR_UNSUPPORTED
    assert ctx.carver_size() == (20000, 4)
    assert ctx.carver_resize_width(1).shape == (1, 4)
    ctx.carver_load(np.zeros((DP_MAX_W + 1, 4), np.uint8))   # width pass fine, height pass too tall
    assert L.dctc_carver_resize(h, 3, DP_MAX_W, None, None) == dc.ERR_UNSUPPORTED
    assert ctx.carver_size() == (4, DP_MAX_W + 1)
    assert ctx.carver_resize_width(1).shape == (1, DP_MAX_W + 1)


# ---- batch session --------------------------------------------------------------------------------------------------

def frames_of(w, h, ch, seeds, patterns=(0,)):
    return np.stack([image(w, h, ch, s, patterns[i % len(patterns)]) for i, s in enumerate(seeds)])


def batch_final(b):
    return dict(image=b.images(), energy=b.energy())


def assert_frames_match_single(ctx, frames, new_w, new_h, passes, fin, vmaps):
    for i, f in enumerate(frames):
        want_p, want_f, _ = combined(ctx, f, new_w, new_h, vmaps)
        got_p = [{k: (v[i] if isinstance(v, np.ndarray) else v) for k, v in p.items()} for p in passes]
        assert_passes_equal(got_p, want_p)
        for k in fin:
            assert np.array_equal(fin[k][i], want_f[k]), (i, k)


@pytest.mark.parametrize("b", [2, 4, 8, 16])
@pytest.mark.parametrize("ch", [1, 3, 4])
def test_batch_frames_equal_single_sessions(ctx, b, ch):
    frames = frames_of(90, 70, ch, [3000 + 7 * b + ch, 3100 + b, 3200 + ch], patterns=(0, 3, 1))
    ctx.set_params(b, 0.5, 0.5)
    vmaps = ch != 4
    new_w, new_h = TARGETS[(b + ch) % 3]
    bt = dc.CarverBatch(ctx, frames, dump_vmaps=(b == 8))
    try:
        passes = bt.resize(new_w, new_h, vmaps=vmaps)
        assert (bt.width, bt.height) == (new_w, new_h)
        assert_frames_match_single(ctx, frames, new_w, new_h, passes, batch_final(bt), vmaps)
    finally:
        bt.close()


@pytest.mark.parametrize("target", [(130, 70), (25, 95), (79, 20)])
def test_batch_multi_pass(ctx, target):
    frames = frames_of(40, 30, 3, [3301, 3302, 3303])
    ctx.set_params(8, 0.5, 0.5)
    bt = dc.CarverBatch(ctx, frames)
    try:
        passes = bt.resize(*target, vmaps=True)
        assert_frames_match_single(ctx, frames, *target, passes, batch_final(bt), True)
    finally:
        bt.close()


def test_batch_reuses_and_reallocates_its_frame_sets(ctx):
    a = frames_of(96, 72, 3, [3401, 3402, 3403])
    c = frames_of(96, 72, 3, [3411, 3412, 3413], patterns=(1, 0, 3))
    ctx.set_params(8, 0.5, 0.5)
    L = dc.lib()
    bt = dc.CarverBatch(ctx, a, dump_vmaps=True)
    try:
        for frames, target in ((a, (80, 60)), (c, (200, 50)), (a, (80, 60)), (c, (60, 150)), (a, (96, 40))):
            bt.load(frames)
            passes = bt.resize(*target, vmaps=True)
            assert_frames_match_single(ctx, frames, *target, passes, batch_final(bt), True)
            assert L.dctc_carver_batch_resize(bt.handle, 50, 50, None, None) == dc.ERR_STATE
        # per-axis calls after a load match a fresh batch
        for call, n in (("resize_height", 11), ("enlarge_height", 20), ("resize_width", 9), ("enlarge_width", 30)):
            bt.load(c)
            s = getattr(bt, call)(n)
            got = (s, bt.images(), bt.energy(), bt.vmap())
            fresh = dc.CarverBatch(ctx, c, dump_vmaps=True)
            try:
                want = (getattr(fresh, call)(n), fresh.images(), fresh.energy(), fresh.vmap())
            finally:
                fresh.close()
            for g, w in zip(got[:3], want[:3]):
                assert np.array_equal(g, w), call
            assert np.array_equal(got[3][0], want[3][0]) and got[3][1] == want[3][1], call
    finally:
        bt.close()


def test_batch_states_and_errors(ctx):
    L = dc.lib()
    ctx.set_params(8, 0.5, 0.5)
    out = C.c_void_p()
    assert L.dctc_carver_batch_create(ctx.handle, 2, 16, 8, 3, 1, C.byref(out)) == dc.OK
    b = out
    try:
        assert L.dctc_carver_batch_resize(b, 10, 6, None, None) == dc.ERR_STATE              # before a load
        imgs = frames_of(16, 8, 3, [1, 2])
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 48) == dc.OK
        assert L.dctc_carver_batch_resize(None, 10, 6, None, None) == dc.ERR_INVALID
        for nw, nh in ((0, 6), (10, 0)):
            assert L.dctc_carver_batch_resize(b, nw, nh, None, None) == dc.ERR_INVALID
        assert L.dctc_carver_batch_resize(b, 16, 8, None, None) == dc.OK                    # nothing changes
        assert L.dctc_carver_batch_resize_width(b, 2, None) == dc.OK                         # a seam operation
        assert L.dctc_carver_batch_resize(b, 10, 6, None, None) == dc.ERR_STATE
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 48) == dc.OK
        assert L.dctc_carver_batch_enlarge_height(b, 2, None) == dc.OK
        assert L.dctc_carver_batch_resize(b, 10, 6, None, None) == dc.ERR_STATE
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 48) == dc.OK
        assert L.dctc_carver_batch_resize(b, 10, 12, None, None) == dc.OK
        assert (L.dctc_carver_batch_width(b), L.dctc_carver_batch_height(b)) == (10, 12)
        for fn in (L.dctc_carver_batch_resize_width, L.dctc_carver_batch_resize_height,
                   L.dctc_carver_batch_enlarge_width, L.dctc_carver_batch_enlarge_height):
            assert fn(b, 1, None) == dc.ERR_STATE
        assert L.dctc_carver_batch_resize(b, 9, 9, None, None) == dc.ERR_STATE
        vm = np.empty(2 * 16 * 8, np.int32)
        assert L.dctc_carver_batch_vmap(b, vm.ctypes.data, None) == dc.ERR_STATE
        assert L.dctc_carver_batch_load(b, imgs.ctypes.data, 8 * 48, 48) == dc.OK           # the load starts over
        assert (L.dctc_carver_batch_width(b), L.dctc_carver_batch_height(b)) == (16, 8)
        assert L.dctc_carver_batch_vmap(b, vm.ctypes.data, None) == dc.OK
    finally:
        L.dctc_carver_batch_destroy(b)
    thin = dc.CarverBatch(ctx, np.zeros((2, 5, 1, 3), np.uint8))
    try:
        assert L.dctc_carver_batch_resize(thin.handle, 3, 5, None, None) == dc.ERR_STATE    # an extent of 1 cannot grow
    finally:
        thin.close()
    wide = dc.CarverBatch(ctx, np.zeros((2, 3, 20000), np.uint8))
    try:
        with pytest.raises(dc.DctcError) as e:
            wide.resize(50000, 3)
        assert e.value.status == dc.ERR_UNSUPPORTED
        assert wide.resize_width(1).shape == (2, 1, 3)                                     # still loaded and fresh
    finally:
        wide.close()


def test_batch_1080p_to_1440x810(ctx):
    """Eight distinct 1920x1080 RGB frames -> 1440x810 (480 vertical, then 270 horizontal seams each)."""
    frames = np.stack([image(1920, 1080, 3, 0x1440810 + i) for i in range(8)])
    ctx.set_params(8, 0.5, 0.5)
    bt = dc.CarverBatch(ctx, frames)
    try:
        passes = bt.resize(1440, 810)
        assert [p["seams"].shape for p in passes] == [(8, 480, 1080), (8, 270, 1440)]
        fin = batch_final(bt)
    finally:
        bt.close()
    assert fin["image"].shape == (8, 810, 1440, 3)
    assert_frames_match_single(ctx, frames, 1440, 810, passes, fin, False)
