"""GPU tests of the bias (dctc_carver_set_bias, dctc_carver_batch_set_bias): a per-pixel plane B that the seam search
adds to the operator energy as E_seam = fl(en_op + fl(B / ext)), ext = the start width of the frame the seam loop runs
on.  The reference is a NumPy seam loop in float32 whose operator energies come from a second context; height, enlarge,
combined resizes and batches are checked against the single-session width call they are defined by, bit for bit."""
import ctypes as C

import numpy as np
import pytest

import dct_carver_b200 as dc
import oracle_lib as ol

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    # the single session's arithmetic: FP32 march (full maps) + FP32 tile (band updates)
    c = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ectx():
    """Operator energies of the NumPy restatement (carver_load + carver_energy of each intermediate image)."""
    c = dc.Context(0, kernel=dc.KERNEL_FP32_MARCH)
    yield c
    c.close()


def image(w, h, ch, seed, pattern=0):
    return ol.synth_image(w, h, ch, seed, pattern).reshape(h, w, ch)


def noise_bias(ectx, img, seed, scale=2.0):
    """Signed noise of the order of ext times the image's energies, so that it changes the seams."""
    ectx.carver_load(img)
    en = ectx.carver_energy()
    rng = np.random.default_rng(seed)
    s = scale * (float(np.mean(en)) + 1e-3) * img.shape[1]
    return (rng.standard_normal(img.shape[:2]) * s).astype(np.float32)


def op_energy(ectx, img):
    ectx.carver_load(img)
    return ectx.carver_energy()


def ref_shrink(ectx, img, bias, n):
    """NumPy restatement of a biased width seam loop: (seams [n, h], image, bias, visibility map [h, w0])."""
    h, w0 = img.shape[:2]
    ext = np.float32(w0)
    cur, B = img.copy(), bias.astype(np.float32).copy()
    raw = np.tile(np.arange(w0), (h, 1))
    vmap = np.zeros((h, w0), np.int32)
    seams = np.zeros((n, h), np.int32)
    inf = np.float32(np.inf)
    for s in range(n):
        w = cur.shape[1]
        E = op_energy(ectx, cur) + B / ext                       # float32 division and add
        assert E.dtype == np.float32
        m = np.empty_like(E)
        m[0] = E[0]
        for y in range(1, h):
            p = np.concatenate(([inf], m[y - 1], [inf]))
            m[y] = E[y] + np.minimum(np.minimum(p[:-2], p[1:-1]), p[2:])
        x = int(np.argmin(m[h - 1]))                            # leftmost minimum
        seam = np.empty(h, np.int64)
        seam[h - 1] = x
        for y in range(h - 1, 0, -1):
            cand = [c for c in (x - 1, x, x + 1) if 0 <= c < w]
            x = cand[int(np.argmin(m[y - 1][cand]))]            # first strict minimum scanning x-1, x, x+1
            seam[y - 1] = x
        seams[s] = seam
        keep = np.ones((h, w), bool)
        keep[np.arange(h), seam] = False
        vmap[np.arange(h), raw[np.arange(h), seam]] = s + 1
        cur = cur[keep].reshape(h, w - 1, -1)
        B = B[keep].reshape(h, w - 1)
        raw = raw[keep].reshape(h, w - 1)
    return seams, cur, B, vmap


def inflate(img, bias, vmap, n):
    """The enlarge of the frames the first n seams of vmap went through: the image by the integer mean rule (a copy in
    column 0), the bias by the copy rule."""
    h, w0 = vmap.shape
    rows_i, rows_b = [], []
    for y in range(h):
        pi, pb = [], []
        for x in range(w0):
            if 0 < vmap[y, x] <= n:
                a = img[y, x].astype(np.int32)
                left = img[y, x - 1].astype(np.int32) if x > 0 else a
                pi.append(((left + a) // 2).astype(np.uint8))
                pb.append(bias[y, x])
            pi.append(img[y, x])
            pb.append(bias[y, x])
        rows_i.append(np.stack(pi))
        rows_b.append(np.array(pb, np.float32))
    return np.stack(rows_i), np.stack(rows_b)


def single(ctx, img, bias, call, n, vmaps=True):
    """Loads img with bias (None: no bias) and runs one seam call: everything it shows afterwards."""
    ctx.carver_load(img)
    if bias is not None:
        ctx.carver_set_bias(bias)
    ctx.carver_set_dump_vmaps(vmaps)
    try:
        seams = getattr(ctx, call)(n)
        out = dict(seams=seams, image=ctx.carver_image(), energy=ctx.carver_energy(), energy_image=ctx.carver_energy_image())
        if vmaps:
            h, w = img.shape[:2]
            out["vmap"] = ctx.carver_vmap(w, h)[0]
        if bias is not None:
            out["bias"] = ctx.carver_bias()
    finally:
        ctx.carver_set_dump_vmaps(False)
    return out


def assert_same(got, want, keys=None):
    for k in keys or want:
        assert got[k].shape == want[k].shape, k
        assert np.array_equal(got[k], want[k]), k


# ---- zero bias == no bias ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("call", ["carver_resize_width", "carver_resize_height", "carver_enlarge_width", "carver_enlarge_height"])
def test_zero_bias_equals_no_bias(ctx, call):
    img = image(80, 60, 3, 7001)
    ctx.set_params(8, 0.5, 0.5)
    zero = np.zeros((60, 80), np.float32)
    got = single(ctx, img, zero, call, 17)
    want = single(ctx, img, None, call, 17)
    assert_same(got, want)
    assert np.array_equal(got["bias"], np.zeros_like(got["energy"]))


def test_zero_bias_equals_no_bias_combined_and_batch(ctx):
    ctx.set_params(4, 0.5, 0.5)
    img = image(40, 30, 3, 7002)
    for target in ((30, 22), (130, 20)):
        ctx.carver_load(img)
        want = ctx.carver_resize(*target, vmaps=True)
        want_f = (ctx.carver_image(), ctx.carver_energy(), ctx.carver_energy_image())
        ctx.carver_load(img)
        ctx.carver_set_bias(np.zeros((30, 40), np.float32))
        got = ctx.carver_resize(*target, vmaps=True)
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert np.array_equal(g["seams"], w["seams"]) and np.array_equal(g["vmap"], w["vmap"])
        for g, w in zip((ctx.carver_image(), ctx.carver_energy(), ctx.carver_energy_image()), want_f):
            assert np.array_equal(g, w)
    imgs = np.stack([image(48, 36, 3, 7003 + i) for i in range(3)])
    for method, n in (("resize_width", 9), ("resize_height", 7), ("enlarge_width", 11)):
        outs = []
        for bias in (None, np.zeros((3, 36, 48), np.float32)):
            b = dc.CarverBatch(ctx, imgs, dump_vmaps=True)
            try:
                if bias is not None:
                    b.set_bias(bias)
                outs.append((getattr(b, method)(n), b.images(), b.energy(), b.vmap()[0]))
            finally:
                b.close()
        for g, w in zip(*outs):
            assert np.array_equal(g, w), method


# ---- against the NumPy restatement -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("b", [2, 4, 8, 16])
@pytest.mark.parametrize("ch", [1, 2, 3, 4])
def test_width_matches_numpy_restatement(ctx, ectx, b, ch):
    wts = (0.5, 0.5) if (b + ch) % 2 else (0.8, 0.2)
    incremental = (ch + b.bit_length()) % 2 == 0     # every weight pair with and without incremental mode
    w, h, n = (96, 64, 40) if b == 8 else (72, 48, 25)
    img = image(w, h, ch, 7100 + 10 * b + ch, pattern=(b + ch) % 4)
    for c in (ctx, ectx):
        c.set_params(b, *wts)
    bias = noise_bias(ectx, img, 7100 + b * ch)
    ctx.carver_set_incremental(incremental)
    try:
        got = single(ctx, img, bias, "carver_resize_width", n)
    finally:
        ctx.carver_set_incremental(False)
    seams, want_img, want_bias, want_vmap = ref_shrink(ectx, img, bias, n)
    assert np.array_equal(got["seams"], seams)
    assert np.array_equal(got["image"], want_img)
    assert np.array_equal(got["bias"], want_bias)
    assert np.array_equal(got["vmap"], want_vmap)
    assert np.array_equal(got["energy"], op_energy(ectx, want_img))   # the getters show the operator map


@pytest.mark.parametrize("incremental", [False, True])
def test_split_resizes_continue_the_biased_loop(ctx, ectx, incremental):
    img = image(90, 60, 3, 7201)
    for c in (ctx, ectx):
        c.set_params(8, 0.8, 0.2)
    bias = noise_bias(ectx, img, 7201)
    ctx.carver_load(img)
    ctx.carver_set_bias(bias)
    ctx.carver_set_incremental(incremental)
    try:
        s = np.concatenate([ctx.carver_resize_width(k) for k in (5, 1, 14)])
    finally:
        ctx.carver_set_incremental(False)
    seams, want_img, want_bias, _ = ref_shrink(ectx, img, bias, 20)
    assert np.array_equal(s, seams)
    assert np.array_equal(ctx.carver_image(), want_img) and np.array_equal(ctx.carver_bias(), want_bias)


def test_set_params_keeps_the_bias(ctx, ectx):
    img = image(64, 48, 3, 7202)
    ctx.set_params(4, 0.5, 0.5)
    ectx.set_params(8, 0.8, 0.2)
    bias = noise_bias(ectx, img, 7202)
    ctx.carver_load(img)
    ctx.carver_set_bias(bias)
    ctx.set_params(8, 0.8, 0.2)        # rebuilds the seam energy with the new operator
    seams = ctx.carver_resize_width(12)
    want = ref_shrink(ectx, img, bias, 12)
    assert np.array_equal(seams, want[0]) and np.array_equal(ctx.carver_image(), want[1])


# ---- height --------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("b,ch", [(2, 1), (4, 3), (8, 3), (16, 4)])
@pytest.mark.parametrize("call", ["resize", "enlarge"])
def test_height_is_the_width_call_on_the_transpose(ctx, ectx, b, ch, call):
    img = image(70, 52, ch, 7300 + b + ch, pattern=b % 4)
    ctx.set_params(b, 0.5, 0.5)
    ectx.set_params(b, 0.5, 0.5)
    bias = noise_bias(ectx, img, 7300 + b)
    got = single(ctx, img, bias, "carver_%s_height" % call, 19)
    t = single(ctx, np.ascontiguousarray(img.transpose(1, 0, 2)), np.ascontiguousarray(bias.T), "carver_%s_width" % call, 19)
    assert np.array_equal(got["seams"], t["seams"])
    for k in ("energy", "energy_image", "vmap", "bias"):
        assert np.array_equal(got[k], t[k].T), k
    assert np.array_equal(got["image"], t["image"].transpose(1, 0, 2))
    if call == "resize":   # ext = the image height: the restatement on the transpose
        seams, want_img, want_bias, _ = ref_shrink(ectx, np.ascontiguousarray(img.transpose(1, 0, 2)), bias.T, 19)
        assert np.array_equal(got["seams"], seams)
        assert np.array_equal(got["bias"], want_bias.T)


# ---- enlarge --------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("b,ch", [(2, 3), (8, 1), (8, 3), (16, 2)])
def test_enlarge_follows_the_biased_shrink(ctx, ectx, b, ch):
    img = image(60, 40, ch, 7400 + b + ch)
    ctx.set_params(b, 0.5, 0.5)
    ectx.set_params(b, 0.5, 0.5)
    bias = noise_bias(ectx, img, 7400 + b)
    n = 23
    shrink = single(ctx, img, bias, "carver_resize_width", n)
    got = single(ctx, img, bias, "carver_enlarge_width", n)
    assert np.array_equal(got["seams"], shrink["seams"])
    assert np.array_equal(got["vmap"], shrink["vmap"])
    want_img, want_bias = inflate(img, bias, shrink["vmap"], n)
    assert np.array_equal(got["image"], want_img)
    assert np.array_equal(got["bias"], want_bias)
    assert np.array_equal(got["energy"], op_energy(ectx, want_img))
    # the enlarged frame's seam loop divides by the enlarged width: a reload with the inflated bias
    more = ctx.carver_resize_width(9)
    want = ref_shrink(ectx, want_img, want_bias, 9)
    assert np.array_equal(more, want[0]) and np.array_equal(ctx.carver_image(), want[1])


# ---- combined resize -------------------------------------------------------------------------------------------------------

def chain(ctx, img, bias, new_w, new_h):
    """The per-axis calls of the plan with a host reload before every pass that re-sets the bias read back."""
    calls = {("width", False): ctx.carver_resize_width, ("width", True): ctx.carver_enlarge_width,
             ("height", False): ctx.carver_resize_height, ("height", True): ctx.carver_enlarge_height}
    h, w = img.shape[:2]
    passes, cur, B = [], img, bias
    ctx.carver_set_dump_vmaps(True)
    try:
        for p in dc.resize_plan(w, h, new_w, new_h):
            ctx.carver_load(cur)
            ctx.carver_set_bias(B)
            seams = calls[(p["axis"], p["enlarge"])](p["n_seams"])
            passes.append(dict(seams=seams, vmap=ctx.carver_vmap(p["w"], p["h"])[0]))
            cur, B = ctx.carver_image(), ctx.carver_bias()
    finally:
        ctx.carver_set_dump_vmaps(False)
    return passes, dict(image=cur, bias=B, energy=ctx.carver_energy(), energy_image=ctx.carver_energy_image())


def combined(ctx, img, bias, new_w, new_h):
    ctx.carver_load(img)
    ctx.carver_set_bias(bias)
    passes = ctx.carver_resize(new_w, new_h, vmaps=True)
    return passes, dict(image=ctx.carver_image(), bias=ctx.carver_bias(), energy=ctx.carver_energy(),
                        energy_image=ctx.carver_energy_image())


@pytest.mark.parametrize("size,target", [((90, 70), (70, 55)), ((40, 30), (130, 20)), ((50, 30), (38, 70))])
@pytest.mark.parametrize("b", [4, 8])
def test_combined_resize_equals_the_chain(ctx, ectx, size, target, b):
    """Both shrinks; two enlarge passes (39 + 51 seams) then a height shrink; a shrink then two height enlarges."""
    img = image(*size, 3, 7500 + b + size[0])
    ctx.set_params(b, 0.5, 0.5)
    ectx.set_params(b, 0.5, 0.5)
    bias = noise_bias(ectx, img, 7500 + b)
    got_p, got_f = combined(ctx, img, bias, *target)
    want_p, want_f = chain(ctx, img, bias, *target)
    assert got_f["image"].shape[:2] == target[::-1]
    assert len(got_p) == len(want_p)
    for i, (g, w) in enumerate(zip(got_p, want_p)):
        assert np.array_equal(g["seams"], w["seams"]), i
        assert np.array_equal(g["vmap"], w["vmap"]), i
    assert_same(got_f, want_f)


# ---- batch ----------------------------------------------------------------------------------------------------------------

def batch_run(ctx, imgs, biases, method, *args):
    b = dc.CarverBatch(ctx, imgs, dump_vmaps=method != "resize")
    try:
        b.set_bias(biases)
        r = getattr(b, method)(*args)
        out = dict(image=b.images(), bias=b.bias(), energy=b.energy())
        if method == "resize":
            out["passes"] = r
        else:
            out["seams"] = r
            out["vmap"] = b.vmap()[0]
        return out
    finally:
        b.close()


@pytest.mark.parametrize("method,n", [("resize_width", 21), ("resize_height", 13), ("enlarge_width", 17), ("enlarge_height", 11)])
def test_batch_frames_equal_their_single_sessions(ctx, ectx, method, n):
    ctx.set_params(8, 0.8, 0.2)
    ectx.set_params(8, 0.8, 0.2)
    imgs = np.stack([image(64, 40, 3, 7600 + i, pattern=i % 4) for i in range(4)])
    biases = np.stack([noise_bias(ectx, imgs[i], 7600 + i) for i in range(4)])
    got = batch_run(ctx, imgs, biases, method, n)
    for i in range(4):
        want = single(ctx, imgs[i], biases[i], "carver_" + method, n)
        for k in ("seams", "image", "bias", "energy", "vmap"):
            assert np.array_equal(got[k][i], want[k]), (i, k)


def test_batch_combined_resize_equals_single_sessions(ctx, ectx):
    ctx.set_params(4, 0.5, 0.5)
    ectx.set_params(4, 0.5, 0.5)
    imgs = np.stack([image(40, 30, 3, 7700 + i) for i in range(3)])
    biases = np.stack([noise_bias(ectx, imgs[i], 7700 + i) for i in range(3)])
    got = batch_run(ctx, imgs, biases, "resize", 130, 20)
    for i in range(3):
        want_p, want_f = combined(ctx, imgs[i], biases[i], 130, 20)
        for g, w in zip(got["passes"], want_p):
            assert np.array_equal(g["seams"][i], w["seams"])
        for k in ("image", "bias", "energy"):
            assert np.array_equal(got[k][i], want_f[k]), (i, k)


def test_batch_eight_1080p_frames_to_1440(ctx):
    ctx.set_params(8, 0.5, 0.5)
    imgs = np.stack([image(1920, 1080, 3, 7800 + i, pattern=i % 4) for i in range(8)])
    rng = np.random.default_rng(7800)
    biases = (rng.standard_normal((8, 1080, 1920)) * 50.0).astype(np.float32)
    biases[:, 300:700, 800:1100] = 1e6          # a preserved region in every frame
    got = batch_run(ctx, imgs, biases, "resize_width", 480)
    assert got["image"].shape == (8, 1080, 1440, 3)
    for i in range(8):
        want = single(ctx, imgs[i], biases[i], "carver_resize_width", 480)
        for k in ("seams", "image", "bias", "energy", "vmap"):
            assert np.array_equal(got[k][i], want[k]), (i, k)
        assert not want["vmap"][300:700, 800:1100].any()


# ---- behaviour -----------------------------------------------------------------------------------------------------------

def test_preserve_mask_is_never_removed(ctx):
    ctx.set_params(8, 0.5, 0.5)
    img = image(96, 64, 3, 7901)
    bias = np.zeros((64, 96), np.float32)
    bias[10:50, 30:60] = 1e6                  # 30 columns wide, narrower than w - n = 56
    out = single(ctx, img, bias, "carver_resize_width", 40)
    assert not out["vmap"][10:50, 30:60].any()
    assert (out["bias"] == 1e6).sum() == 40 * 30


@pytest.mark.parametrize("k", [1, 5, 12])
def test_discard_mask_is_removed_by_k_seams(ctx, k):
    ctx.set_params(8, 0.5, 0.5)
    img = image(96, 64, 3, 7902 + k)
    bias = np.zeros((64, 96), np.float32)
    bias[:, 41:41 + k] = -1e6
    out = single(ctx, img, bias, "carver_resize_width", k)
    strip = out["vmap"][:, 41:41 + k]
    assert np.all((strip >= 1) & (strip <= k))
    assert not (out["bias"] < 0).any()        # object removal: nothing of the strip is left


# ---- launches --------------------------------------------------------------------------------------------------------------

def launches(c, fn):
    n0 = c.launches
    r = fn()
    return c.launches - n0, r


def test_launch_counts(ctx):
    ctx.set_params(8, 0.5, 0.5)
    img = image(80, 56, 3, 8001)
    bias = np.ones((56, 80), np.float32)
    ctx.carver_load(img)
    assert launches(ctx, lambda: ctx.carver_set_bias(None))[0] == 0   # clearing no bias does nothing
    assert launches(ctx, lambda: ctx.carver_set_bias(bias))[0] == 2   # K1 + bias add
    per_call = {}
    for call, n in (("carver_resize_width", 5), ("carver_resize_width", 12), ("carver_resize_height", 9),
                    ("carver_enlarge_width", 7), ("carver_enlarge_height", 7)):
        counts = []
        for biased in (False, True):
            ctx.carver_load(img)
            if biased:
                ctx.carver_set_bias(bias)
            counts.append(launches(ctx, lambda: getattr(ctx, call)(n))[0])
        per_call[(call, n)] = counts
        extra = {"carver_resize_width": 0, "carver_resize_height": 2, "carver_enlarge_width": 1, "carver_enlarge_height": 3}[call]
        assert counts[1] == counts[0] + extra, (call, counts)
    # per seam: the same launches with and without a bias
    un = per_call[("carver_resize_width", 12)][0] - per_call[("carver_resize_width", 5)][0]
    bi = per_call[("carver_resize_width", 12)][1] - per_call[("carver_resize_width", 5)][1]
    assert un == bi
    # getters: one K1 more for the operator map, nothing more for the image
    ctx.carver_load(img)
    un_e, un_i = launches(ctx, ctx.carver_energy)[0], launches(ctx, ctx.carver_image)[0]
    ctx.carver_set_bias(bias)
    ctx.carver_resize_width(3)
    assert launches(ctx, ctx.carver_energy)[0] == un_e + 1
    assert launches(ctx, ctx.carver_image)[0] == un_i
    # batch
    imgs = np.stack([img, img[:, ::-1]])
    counts = []
    for biased in (False, True):
        b = dc.CarverBatch(ctx, imgs)
        try:
            if biased:
                assert launches(ctx, lambda: b.set_bias(np.stack([bias, bias])))[0] == 2
            counts.append(launches(ctx, lambda: b.resize_height(6))[0])
        finally:
            b.close()
    assert counts[1] == counts[0] + 2


# ---- state and error rules ---------------------------------------------------------------------------------------------------

def test_state_and_error_rules(ctx):
    ctx.set_params(8, 0.5, 0.5)
    L = dc.lib()
    img = image(64, 40, 3, 8101)
    bias = np.ones((40, 64), np.float32)
    c2 = dc.Context(0)
    try:   # before a load
        assert L.dctc_carver_set_bias(c2.handle, bias.ctypes.data, 64 * 4) == dc.ERR_STATE
    finally:
        c2.close()
    ctx.carver_load(img)
    out = np.empty((40, 64), np.float32)
    assert L.dctc_carver_bias(ctx.handle, out.ctypes.data) == dc.ERR_STATE          # no bias set
    assert L.dctc_carver_set_bias(ctx.handle, bias.ctypes.data, 63 * 4) == dc.ERR_INVALID
    ctx.carver_set_bias(bias)
    assert np.array_equal(ctx.carver_bias(), bias)
    seam = np.full(40, 10, np.int32)
    assert L.dctc_carve_and_update(ctx.handle, seam.ctypes.data, None, None, None) == dc.ERR_STATE
    ctx.carver_resize_width(2)
    assert L.dctc_carver_set_bias(ctx.handle, bias[:, :62].copy().ctypes.data, 62 * 4) == dc.ERR_STATE   # after a seam operation
    assert L.dctc_carver_set_bias(ctx.handle, None, 0) == dc.ERR_STATE
    ctx.carver_load(img)                                                             # a load clears the bias
    assert L.dctc_carver_bias(ctx.handle, out.ctypes.data) == dc.ERR_STATE
    ctx.carver_set_bias(bias)
    ctx.carver_set_bias(None)
    assert L.dctc_carver_bias(ctx.handle, out.ctypes.data) == dc.ERR_STATE
    # wrappers
    for bad in (np.ones((40, 63), np.float32), np.ones((64, 40), np.float32), np.full((40, 64), np.nan, np.float32),
                np.where(np.eye(40, 64) > 0, np.inf, 0).astype(np.float32)):
        with pytest.raises(ValueError):
            ctx.carver_set_bias(bad)
    b = dc.CarverBatch(ctx, np.stack([img, img]))
    try:
        with pytest.raises(ValueError):
            b.set_bias(np.ones((1, 40, 64), np.float32))
        with pytest.raises(ValueError):
            b.set_bias(np.full((2, 40, 64), -np.inf, np.float32))
        with pytest.raises(dc.DctcError):
            b.bias()
        b.set_bias(np.stack([bias, 2 * bias]))
        assert np.array_equal(b.bias()[1], 2 * bias)
        b.resize_width(3)
        assert L.dctc_carver_batch_set_bias(b.handle, None, 0, 0) == dc.ERR_STATE
        b.load(np.stack([img, img]))                                                 # a load clears the bias
        with pytest.raises(dc.DctcError):
            b.bias()
    finally:
        b.close()


@pytest.mark.parametrize("axis", ["width", "height"])
def test_operator_getters_after_carving_equal_an_unbiased_reload(ctx, axis):
    """The getters show the operator map of the carved image: what an unbiased load of it shows (for a height session:
    of its transpose, turned back, as every height result is defined)."""
    ctx.set_params(8, 0.5, 0.5)
    img = image(80, 48, 3, 8201)
    rng = np.random.default_rng(8201)
    ctx.carver_load(img)
    ctx.carver_set_bias((rng.standard_normal((48, 80)) * 1e3).astype(np.float32))
    getattr(ctx, "carver_resize_" + axis)(9)
    got = dict(energy=ctx.carver_energy(), energy_image=ctx.carver_energy_image())
    w, h = ctx.carver_size()
    p = dc.CarverEnergyParams()
    p.gpu = ctx.handle.value
    pts = ((0, 0), (17, 30), (w - 1, h - 1))
    pix = [dc.lib().dctc_pixel_energy(x, y, w, h, None, C.byref(p)) for (x, y) in pts]
    carved = ctx.carver_image()
    if axis == "width":
        ctx.carver_load(carved)
        want = dict(energy=ctx.carver_energy(), energy_image=ctx.carver_energy_image())
    else:
        ctx.carver_load(np.ascontiguousarray(carved.transpose(1, 0, 2)))
        want = dict(energy=ctx.carver_energy().T, energy_image=ctx.carver_energy_image().T)
    assert_same(got, want)
    assert pix == [want["energy"][y, x] for (x, y) in pts]
