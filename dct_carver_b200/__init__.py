"""dct_carver_b200 — B200-native DCT-Carver energy hot path.

Thin ctypes mirror of the C ABI in include/dctc.h (the product is the CUDA library, not this file).
Names follow the reference: EnergyParameters (src/render.h:9-18), blocksize / edges / textures
(src/main.h:12-22).  There is no CPU fallback: if libdctc.so is missing or no CUDA device is present,
loading / context creation raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DCTC_LIB") or os.path.join(_HERE, "libdctc.so")   # DCTC_LIB: experimental builds (tools/build_exp.sh)

OK = 0
ERR_INVALID, ERR_BLOCKSIZE, ERR_NOMEM, ERR_CUDA, ERR_NO_DEVICE, ERR_STATE, ERR_UNSUPPORTED = -1, -2, -3, -4, -5, -6, -7
KERNEL_AUTO, KERNEL_FP32_TILE, KERNEL_FP32_MARCH, KERNEL_TC_SPLIT, KERNEL_FP32_STREAM = 0, 1, 2, 3, 4
MAX_DELTA_X = 4   # DCTC_MAX_DELTA_X: the widest seam step the device seam loop takes

# every symbol include/dctc.h declares (tests check that the library exports exactly these)
ABI_SYMBOLS = [
    "dctc_create", "dctc_destroy", "dctc_set_params", "dctc_set_kernel", "dctc_last_cuda_error", "dctc_strerror",
    "dctc_version", "dctc_device_count", "dctc_stream", "dctc_launch_count",
    "dctc_energy_full", "dctc_energy_full_dev", "dctc_energy_batch_dev", "dctc_energy_band_dev", "dctc_energy_band_dev_at", "dctc_energy_batch",
    "dctc_carver_load", "dctc_carver_width", "dctc_carver_height", "dctc_carver_energy", "dctc_carve_and_update",
    "dctc_carver_image", "dctc_carver_resize_width", "dctc_carver_enlarge_width", "dctc_carver_resize_height",
    "dctc_carver_enlarge_height", "dctc_carver_set_incremental", "dctc_carver_rebuild_count", "dctc_pixel_energy",
    "dctc_energy_minmax_dev", "dctc_energy_image_dev", "dctc_carver_energy_image", "dctc_preview_energy",
    "dctc_carver_set_dump_vmaps", "dctc_carver_vmap", "dctc_carver_paint_seams",
    "dctc_carver_batch_create", "dctc_carver_batch_destroy", "dctc_carver_batch_load", "dctc_carver_batch_resize_width",
    "dctc_carver_batch_enlarge_width", "dctc_carver_batch_width", "dctc_carver_batch_images", "dctc_carver_batch_energy",
    "dctc_carver_batch_vmap", "dctc_carver_batch_resize_height", "dctc_carver_batch_enlarge_height", "dctc_carver_batch_height",
    "dctc_resize_plan", "dctc_carver_resize", "dctc_carver_batch_resize",
    "dctc_carver_set_bias", "dctc_carver_bias", "dctc_carver_batch_set_bias", "dctc_carver_batch_bias",
    "dctc_carver_set_rigidity", "dctc_carver_batch_set_rigidity", "dctc_carver_set_delta_x", "dctc_carver_batch_set_delta_x",
    "dctc_carver_levels_width", "dctc_carver_levels_height", "dctc_carver_render_levels", "dctc_carver_batch_levels_width",
    "dctc_carver_batch_levels_height", "dctc_carver_batch_render_levels", "dctc_carver_batch_render_levels_dev",
    "dctc_synth_fill_dev", "dctc_synth_byte", "dctc_ipc_export", "dctc_ipc_open", "dctc_ipc_close",
    "dctc_dev_alloc", "dctc_dev_free", "dctc_host_alloc_pinned", "dctc_host_alloc_pinned_wc", "dctc_host_free_pinned", "dctc_memcpy_h2d",
    "dctc_memcpy_d2h", "dctc_memset_dev", "dctc_sync", "dctc_timer_begin", "dctc_timer_end",
    # multi-GPU host layer (csrc/dctc_multi.cu)
    "dctc_band_plan", "dctc_multi_create", "dctc_multi_destroy", "dctc_multi_device_count", "dctc_multi_context",
    "dctc_multi_set_params", "dctc_multi_set_kernel", "dctc_multi_launch_count", "dctc_multi_energy_batch",
    "dctc_multi_energy_bands", "dctc_multi_bands_create", "dctc_multi_bands_destroy", "dctc_multi_bands_geometry",
    "dctc_multi_bands_upload", "dctc_multi_bands_synth", "dctc_multi_bands_energy", "dctc_multi_bands_download",
    "dctc_multi_bands_energy_image", "dctc_rendezvous_allgather", "dctc_band_runner_create", "dctc_band_runner_geometry",
    "dctc_band_runner_image_dev", "dctc_band_runner_energy_dev", "dctc_band_runner_synth", "dctc_band_runner_upload",
    "dctc_band_runner_connect", "dctc_band_runner_barrier", "dctc_band_runner_energy", "dctc_band_runner_download",
    "dctc_band_runner_energy_image", "dctc_band_runner_destroy", "dctc_pcie_probe",
]


class EnergyParameters(C.Structure):
    """Bit-for-bit the reference's EnergyParameters (src/render.h:9-18)."""
    _fields_ = [("edges", C.c_float), ("textures", C.c_float), ("blocksize", C.c_int),
                ("ip", C.POINTER(C.c_int)), ("w", C.POINTER(C.c_double)), ("data", C.POINTER(C.POINTER(C.c_double)))]


class CarverEnergyParams(C.Structure):
    _fields_ = [("base", EnergyParameters), ("gpu", C.c_void_p)]


RESIZE_WIDTH, RESIZE_HEIGHT = 0, 1


class ResizePass(C.Structure):
    """DctcResizePass (include/dctc.h): one pass of a resize plan."""
    _fields_ = [("axis", C.c_int), ("enlarge", C.c_int), ("n_seams", C.c_int), ("w", C.c_int), ("h", C.c_int),
                ("seams_offset", C.c_size_t), ("vmap_offset", C.c_size_t)]


class DctcError(RuntimeError):
    def __init__(self, status, what=""):
        self.status = status
        msg = "%s failed: %d" % (what, status)
        try:
            msg += " (%s)" % lib().dctc_strerror(status).decode()
        except Exception:
            pass
        super().__init__(msg)


_lib = None


def lib():
    """Loads libdctc.so; fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("dct_carver_b200: %s is missing — run `python -m dct_carver_b200.build` "
                          "(needs nvcc). There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, sz, i32, u32, f32 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint32, C.c_float
    sig = {
        "dctc_create": (i32, [C.POINTER(vp), i32]),
        "dctc_destroy": (None, [vp]),
        "dctc_set_params": (i32, [vp, C.POINTER(EnergyParameters)]),
        "dctc_set_kernel": (i32, [vp, i32]),
        "dctc_last_cuda_error": (i32, [vp]),
        "dctc_strerror": (C.c_char_p, [i32]),
        "dctc_version": (i32, []),
        "dctc_device_count": (i32, []),
        "dctc_stream": (vp, [vp]),
        "dctc_launch_count": (C.c_ulonglong, [vp]),
        "dctc_energy_full": (i32, [vp, vp, i32, i32, i32, sz, vp]),
        "dctc_energy_full_dev": (i32, [vp, vp, i32, i32, i32, sz, vp, sz, i32]),
        "dctc_energy_batch_dev": (i32, [vp, vp, i32, sz, i32, i32, i32, sz, vp, sz, sz, i32]),
        "dctc_energy_band_dev": (i32, [vp, vp, i32, i32, i32, sz, vp, i32, sz, vp, i32, sz, vp, sz, i32]),
        "dctc_energy_band_dev_at": (i32, [vp, vp, i32, i32, i32, i32, sz, vp, i32, sz, vp, i32, sz, vp, sz, i32]),
        "dctc_energy_batch": (i32, [vp, vp, i32, sz, i32, i32, i32, sz, vp, sz]),
        "dctc_carver_load": (i32, [vp, vp, i32, i32, i32, sz]),
        "dctc_carver_width": (i32, [vp]),
        "dctc_carver_height": (i32, [vp]),
        "dctc_carver_energy": (i32, [vp, vp]),
        "dctc_carve_and_update": (i32, [vp, vp, vp, vp, vp]),
        "dctc_carver_image": (i32, [vp, vp]),
        "dctc_carver_resize_width": (i32, [vp, i32, vp]),
        "dctc_carver_enlarge_width": (i32, [vp, i32, vp]),
        "dctc_carver_resize_height": (i32, [vp, i32, vp]),
        "dctc_carver_enlarge_height": (i32, [vp, i32, vp]),
        "dctc_carver_rebuild_count": (i32, [vp]),
        "dctc_carver_set_incremental": (i32, [vp, i32]),
        "dctc_energy_minmax_dev": (i32, [vp, vp, C.c_size_t, i32, i32, vp]),
        "dctc_energy_image_dev": (i32, [vp, vp, C.c_size_t, i32, i32, vp, vp, C.c_size_t, i32]),
        "dctc_carver_energy_image": (i32, [vp, vp]),
        "dctc_preview_energy": (i32, [vp, vp, i32, i32, i32, C.c_size_t, vp, vp]),
        "dctc_carver_set_dump_vmaps": (i32, [vp, i32]),
        "dctc_carver_vmap": (i32, [vp, vp, vp]),
        "dctc_carver_paint_seams": (i32, [vp, vp, i32, C.c_size_t]),
        "dctc_carver_batch_create": (i32, [vp, i32, i32, i32, i32, i32, C.POINTER(vp)]),
        "dctc_carver_batch_destroy": (None, [vp]),
        "dctc_carver_batch_load": (i32, [vp, vp, sz, sz]),
        "dctc_carver_batch_resize_width": (i32, [vp, i32, vp]),
        "dctc_carver_batch_enlarge_width": (i32, [vp, i32, vp]),
        "dctc_carver_batch_width": (i32, [vp]),
        "dctc_carver_batch_resize_height": (i32, [vp, i32, vp]),
        "dctc_carver_batch_enlarge_height": (i32, [vp, i32, vp]),
        "dctc_carver_batch_height": (i32, [vp]),
        "dctc_carver_batch_images": (i32, [vp, vp]),
        "dctc_carver_batch_energy": (i32, [vp, vp]),
        "dctc_carver_batch_vmap": (i32, [vp, vp, vp]),
        "dctc_resize_plan": (i32, [i32, i32, i32, i32, vp, i32]),
        "dctc_carver_resize": (i32, [vp, i32, i32, vp, vp]),
        "dctc_carver_batch_resize": (i32, [vp, i32, i32, vp, vp]),
        "dctc_carver_set_bias": (i32, [vp, vp, sz]),
        "dctc_carver_bias": (i32, [vp, vp]),
        "dctc_carver_batch_set_bias": (i32, [vp, vp, sz, sz]),
        "dctc_carver_batch_bias": (i32, [vp, vp]),
        "dctc_carver_set_rigidity": (i32, [vp, f32]),
        "dctc_carver_batch_set_rigidity": (i32, [vp, f32]),
        "dctc_carver_set_delta_x": (i32, [vp, i32]),
        "dctc_carver_batch_set_delta_x": (i32, [vp, i32]),
        "dctc_carver_levels_width": (i32, [vp, i32, vp]),
        "dctc_carver_levels_height": (i32, [vp, i32, vp]),
        "dctc_carver_render_levels": (i32, [vp, i32, vp, vp]),
        "dctc_carver_batch_levels_width": (i32, [vp, i32, vp]),
        "dctc_carver_batch_levels_height": (i32, [vp, i32, vp]),
        "dctc_carver_batch_render_levels": (i32, [vp, i32, vp, vp]),
        "dctc_carver_batch_render_levels_dev": (i32, [vp, i32, vp, vp]),
        "dctc_pixel_energy": (f32, [i32, i32, i32, i32, vp, vp]),
        "dctc_synth_fill_dev": (i32, [vp, vp, i32, sz, i32, i32, i32, sz, u32, i32, i32, i32]),
        "dctc_synth_byte": (C.c_uint8, [u32, u32, u32, u32, u32, i32]),
        "dctc_ipc_export": (i32, [vp, vp, vp]),
        "dctc_ipc_open": (i32, [vp, vp, C.POINTER(vp)]),
        "dctc_ipc_close": (i32, [vp, vp]),
        "dctc_dev_alloc": (i32, [vp, C.POINTER(vp), sz]),
        "dctc_dev_free": (i32, [vp, vp]),
        "dctc_host_alloc_pinned": (i32, [C.POINTER(vp), sz]),
        "dctc_host_alloc_pinned_wc": (i32, [C.POINTER(vp), sz]),
        "dctc_host_free_pinned": (i32, [vp]),
        "dctc_memcpy_h2d": (i32, [vp, vp, vp, sz]),
        "dctc_memcpy_d2h": (i32, [vp, vp, vp, sz]),
        "dctc_memset_dev": (i32, [vp, vp, i32, sz]),
        "dctc_sync": (i32, [vp]),
        "dctc_timer_begin": (i32, [vp]),
        "dctc_timer_end": (i32, [vp, C.POINTER(f32)]),
        "dctc_band_plan": (i32, [i32, i32, i32, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
        "dctc_multi_create": (i32, [C.POINTER(vp), C.POINTER(i32), i32]),
        "dctc_multi_destroy": (None, [vp]),
        "dctc_multi_device_count": (i32, [vp]),
        "dctc_multi_context": (vp, [vp, i32]),
        "dctc_multi_set_params": (i32, [vp, C.POINTER(EnergyParameters)]),
        "dctc_multi_set_kernel": (i32, [vp, i32]),
        "dctc_multi_launch_count": (C.c_ulonglong, [vp]),
        "dctc_multi_energy_batch": (i32, [vp, vp, i32, sz, i32, i32, i32, sz, vp, sz]),
        "dctc_multi_energy_bands": (i32, [vp, vp, i32, i32, i32, sz, vp, vp]),
        "dctc_multi_bands_create": (i32, [vp, i32, i32, i32, C.POINTER(vp)]),
        "dctc_multi_bands_destroy": (None, [vp]),
        "dctc_multi_bands_geometry": (i32, [vp, i32, C.POINTER(i32), C.POINTER(i32)]),
        "dctc_multi_bands_upload": (i32, [vp, vp, sz]),
        "dctc_multi_bands_synth": (i32, [vp, u32, i32]),
        "dctc_multi_bands_energy": (i32, [vp, i32]),
        "dctc_multi_bands_download": (i32, [vp, vp]),
        "dctc_multi_bands_energy_image": (i32, [vp, vp]),
        "dctc_rendezvous_allgather": (i32, [C.c_char_p, i32, i32, vp, sz, vp, i32]),
        "dctc_band_runner_create": (i32, [vp, C.c_char_p, i32, i32, i32, i32, i32, C.POINTER(vp)]),
        "dctc_band_runner_geometry": (i32, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(sz)]),
        "dctc_band_runner_image_dev": (vp, [vp]),
        "dctc_band_runner_energy_dev": (vp, [vp]),
        "dctc_band_runner_synth": (i32, [vp, u32, i32]),
        "dctc_band_runner_upload": (i32, [vp, vp, sz]),
        "dctc_band_runner_connect": (i32, [vp]),
        "dctc_band_runner_barrier": (i32, [vp]),
        "dctc_band_runner_energy": (i32, [vp, i32]),
        "dctc_band_runner_download": (i32, [vp, vp]),
        "dctc_band_runner_energy_image": (i32, [vp, vp]),
        "dctc_band_runner_destroy": (None, [vp]),
        "dctc_pcie_probe": (i32, [vp, sz, i32, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _check(status, what):
    if status != OK:
        raise DctcError(status, what)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def resize_plan(w, h, new_w, new_h):
    """The passes lqr_carver_resize(new_w, new_h) runs from w x h (dctc_resize_plan), in order: dicts with axis ("width"
    or "height"), enlarge, n_seams, the image size w, h at the start of the pass, and the pass's per-frame offsets (in
    ints) in the seams and maps buffers of Context.carver_resize / CarverBatch.resize."""
    n = lib().dctc_resize_plan(w, h, new_w, new_h, None, 0)
    if n < 0:
        raise DctcError(n, "dctc_resize_plan")
    passes = (ResizePass * max(n, 1))()
    lib().dctc_resize_plan(w, h, new_w, new_h, passes, n)
    return [dict(axis="width" if p.axis == RESIZE_WIDTH else "height", enlarge=bool(p.enlarge), n_seams=p.n_seams, w=p.w,
                 h=p.h, seams_offset=p.seams_offset, vmap_offset=p.vmap_offset) for p in passes[:n]]


def _resize(fn, handle, w, h, new_w, new_h, vmaps, n_frames):
    """Runs dctc_carver_resize / dctc_carver_batch_resize (fn) and splits its buffers into one entry per pass: axis,
    enlarge, seams ([n_frames,] n_seams, len) and, with vmaps, the map ([n_frames,] h, w) of the pass's start frame."""
    try:
        plan = resize_plan(w, h, new_w, new_h) if min(w, h, new_w, new_h) > 0 else []
    except DctcError:
        plan = []   # the entry point refuses the same sizes and reports its own status
    lens = [p["h"] if p["axis"] == "width" else p["w"] for p in plan]
    n_seams = sum(p["n_seams"] * n for p, n in zip(plan, lens))
    n_maps = sum(p["w"] * p["h"] for p in plan)
    nf = n_frames or 1
    seams = np.empty(nf * n_seams, np.int32)
    maps = np.empty(nf * n_maps, np.int32) if vmaps else None
    _check(fn(handle, int(new_w), int(new_h), _ptr(seams) if n_seams else None, _ptr(maps) if vmaps and n_maps else None),
           fn.__name__)
    lead = (n_frames,) if n_frames else ()
    out = []
    for p, n in zip(plan, lens):
        so, vo = nf * p["seams_offset"], nf * p["vmap_offset"]
        e = dict(axis=p["axis"], enlarge=p["enlarge"],
                 seams=seams[so:so + nf * p["n_seams"] * n].reshape(lead + (p["n_seams"], n)))
        if vmaps:
            e["vmap"] = maps[vo:vo + nf * p["w"] * p["h"]].reshape(lead + (p["h"], p["w"]))
        out.append(e)
    return out


def _render_levels(fn, handle, levels, extents, n_frames, ch, out=None):
    """Runs dctc_carver_render_levels / dctc_carver_batch_render_levels (fn) after a build along levels = (axis, w, h),
    the image size at the build (None: no build, fn reports the state), and splits its buffer into one uint8 array
    ([n_frames,] H_i, W_i, ch) per extent."""
    ext = np.ascontiguousarray([int(e) for e in extents], np.int32)
    if levels is None:
        shapes = [(0, 0)] * len(ext)
    else:
        axis, w, h = levels
        shapes = [(h, max(int(e), 0)) if axis == "width" else (max(int(e), 0), w) for e in ext]
    nf = n_frames or 1
    sizes = [nf * H * W * ch for H, W in shapes]
    buf = np.empty(max(sum(sizes), 1), np.uint8)
    _check(fn(handle, len(ext), _ptr(ext) if len(ext) else None, _ptr(buf)), fn.__name__)
    lead = (n_frames,) if n_frames else ()
    res, o = [], 0
    for (H, W), s in zip(shapes, sizes):
        res.append(buf[o:o + s].reshape(lead + (H, W, ch)))
        o += s
    return res


def _bias_plane(bias, shape):
    """bias as a C-contiguous float32 array of `shape`; ValueError for another shape or a non-finite value."""
    b = np.asarray(bias, dtype=np.float32)
    if b.shape != tuple(shape):
        raise ValueError("bias must have shape %s, got %s" % (tuple(shape), b.shape))
    if not np.isfinite(b).all():
        raise ValueError("bias values must be finite")
    return np.ascontiguousarray(b)


def pinned_array(shape, dtype, write_combined=False):
    """numpy array over cudaMallocHost memory (kept alive by the returned array's base); write_combined: for input frames
    the host only writes."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    if write_combined:
        _check(lib().dctc_host_alloc_pinned_wc(C.byref(p), n), "dctc_host_alloc_pinned_wc")
    else:
        _check(lib().dctc_host_alloc_pinned(C.byref(p), n), "dctc_host_alloc_pinned")
    buf = (C.c_uint8 * max(n, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED[id(buf)] = (buf, p.value)
    return arr


_PINNED = {}


class Context:
    """One GPU context (one caller at a time, like the reference's single-threaded callback)."""

    def __init__(self, device=0, blocksize=8, edges=0.5, textures=0.5, kernel=KERNEL_AUTO):
        self._h = C.c_void_p()
        _check(lib().dctc_create(C.byref(self._h), device), "dctc_create")
        self.device = device
        self.set_params(blocksize, edges, textures)
        if kernel != KERNEL_AUTO:
            self.set_kernel(kernel)

    # -- parameters ------------------------------------------------------------------------------------
    def set_params(self, blocksize, edges, textures):
        p = EnergyParameters(edges=edges, textures=textures, blocksize=blocksize)
        _check(lib().dctc_set_params(self._h, C.byref(p)), "dctc_set_params")
        self.blocksize, self.edges, self.textures = blocksize, edges, textures

    def set_kernel(self, kernel):
        _check(lib().dctc_set_kernel(self._h, kernel), "dctc_set_kernel")

    @property
    def handle(self):
        return self._h

    @property
    def launches(self):
        return int(lib().dctc_launch_count(self._h))

    def close(self):
        if self._h:
            lib().dctc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- K1 ---------------------------------------------------------------------------------------------
    def energy_full(self, img):
        """img: uint8 array [h, w] or [h, w, channels] (C-contiguous rows) -> float32 [h, w]."""
        img = np.asarray(img)
        if img.dtype != np.uint8:
            raise TypeError("image must be uint8")
        if img.ndim == 2:
            img = img[:, :, None]
        img = np.ascontiguousarray(img)
        h, w, ch = img.shape
        out = np.empty((h, w), np.float32)
        _check(lib().dctc_energy_full(self._h, _ptr(img), w, h, ch, w * ch, _ptr(out)), "dctc_energy_full")
        return out

    def energy_batch(self, imgs, out=None):
        """imgs: uint8 [n, h, w, ch] host array (pinned for full speed) -> float32 [n, h, w]."""
        n, h, w, ch = imgs.shape
        if out is None:
            out = np.empty((n, h, w), np.float32)
        _check(lib().dctc_energy_batch(self._h, _ptr(imgs), n, h * w * ch, w, h, ch, w * ch, _ptr(out), h * w),
               "dctc_energy_batch")
        return out

    # -- device memory helpers ----------------------------------------------------------------------------
    def dev_alloc(self, nbytes):
        p = C.c_void_p()
        _check(lib().dctc_dev_alloc(self._h, C.byref(p), nbytes), "dctc_dev_alloc")
        return p.value

    def dev_free(self, p):
        _check(lib().dctc_dev_free(self._h, C.c_void_p(p)), "dctc_dev_free")

    def h2d(self, d_ptr, arr):
        arr = np.ascontiguousarray(arr)
        _check(lib().dctc_memcpy_h2d(self._h, C.c_void_p(d_ptr), _ptr(arr), arr.nbytes), "dctc_memcpy_h2d")

    def d2h(self, arr, d_ptr):
        _check(lib().dctc_memcpy_d2h(self._h, _ptr(arr), C.c_void_p(d_ptr), arr.nbytes), "dctc_memcpy_d2h")

    def sync(self):
        _check(lib().dctc_sync(self._h), "dctc_sync")

    def ipc_export(self, d_ptr):
        buf = (C.c_ubyte * 64)()
        _check(lib().dctc_ipc_export(self._h, C.c_void_p(d_ptr), buf), "dctc_ipc_export")
        return bytes(buf)

    def ipc_open(self, handle):
        buf = (C.c_ubyte * 64).from_buffer_copy(handle)
        p = C.c_void_p()
        _check(lib().dctc_ipc_open(self._h, buf, C.byref(p)), "dctc_ipc_open")
        return p.value

    def ipc_close(self, d_ptr):
        _check(lib().dctc_ipc_close(self._h, C.c_void_p(d_ptr)), "dctc_ipc_close")

    def timer_begin(self):
        _check(lib().dctc_timer_begin(self._h), "dctc_timer_begin")

    def timer_end(self):
        ms = C.c_float()
        _check(lib().dctc_timer_end(self._h, C.byref(ms)), "dctc_timer_end")
        return ms.value

    def synth_fill_dev(self, d_img, n_frames, frame_stride, w, h, ch, pitch, seed, pattern=0, first_frame=0, y_offset=0):
        _check(lib().dctc_synth_fill_dev(self._h, C.c_void_p(d_img), n_frames, frame_stride, w, h, ch, pitch, seed,
                                         pattern, first_frame, y_offset), "dctc_synth_fill_dev")

    def energy_batch_dev(self, d_imgs, n, frame_stride, w, h, ch, pitch, d_out, out_frame_stride, out_pitch, sync=False):
        _check(lib().dctc_energy_batch_dev(self._h, C.c_void_p(d_imgs), n, frame_stride, w, h, ch, pitch,
                                           C.c_void_p(d_out), out_frame_stride, out_pitch, int(sync)),
               "dctc_energy_batch_dev")

    def energy_band_dev(self, d_band, w, rows, ch, pitch, d_top, top_rows, top_pitch, d_bot, bot_rows, bot_pitch, d_out,
                        out_pitch, sync=False, band_y0=0):
        """band_y0: image row of the band's first row (dctc_energy_band_dev_at); 0 = dctc_energy_band_dev."""
        _check(lib().dctc_energy_band_dev_at(self._h, C.c_void_p(d_band), w, rows, band_y0, ch, pitch,
                                             C.c_void_p(d_top) if d_top else None, top_rows, top_pitch,
                                             C.c_void_p(d_bot) if d_bot else None, bot_rows, bot_pitch,
                                             C.c_void_p(d_out), out_pitch, int(sync)), "dctc_energy_band_dev_at")

    # -- K2 carver session ----------------------------------------------------------------------------------
    def carver_load(self, img):
        img = np.asarray(img)
        if img.ndim == 2:
            img = img[:, :, None]
        img = np.ascontiguousarray(img, dtype=np.uint8)
        h, w, ch = img.shape
        self._carver_levels = None
        _check(lib().dctc_carver_load(self._h, _ptr(img), w, h, ch, w * ch), "dctc_carver_load")
        self._carver_ch = ch

    def carver_size(self):
        return lib().dctc_carver_width(self._h), lib().dctc_carver_height(self._h)

    def carver_energy(self):
        w, h = self.carver_size()
        out = np.empty((h, w), np.float32)
        _check(lib().dctc_carver_energy(self._h, _ptr(out)), "dctc_carver_energy")
        return out

    def carver_image(self):
        w, h = self.carver_size()
        out = np.empty((h, w, self._carver_ch), np.uint8)
        _check(lib().dctc_carver_image(self._h, _ptr(out)), "dctc_carver_image")
        return out

    def carver_resize_width(self, n_seams):
        """Whole retarget loop on the device (seam DP, back-track, carve, band energy update per seam); returns the
        removed columns, shape (n_seams, h), in the coordinates of the image at the time of removal."""
        w, h = self.carver_size()
        seams = np.empty((n_seams, h), np.int32)
        _check(lib().dctc_carver_resize_width(self._h, int(n_seams), _ptr(seams) if n_seams else None),
               "dctc_carver_resize_width")
        return seams

    def carver_enlarge_width(self, n_seams):
        """lqr_carver_resize to a larger width on the device: returns the n_seams seams (as carver_resize_width does);
        the session continues on the enlarged image."""
        w, h = self.carver_size()
        seams = np.empty((n_seams, h), np.int32)
        _check(lib().dctc_carver_enlarge_width(self._h, int(n_seams), _ptr(seams) if n_seams else None),
               "dctc_carver_enlarge_width")
        return seams

    def carver_resize_height(self, n_seams):
        """Removes n_seams horizontal seams on the device (lqr_carver_resize(carver, w, h - n_seams)); returns the removed
        rows, shape (n_seams, w), in the coordinates of the image at the time of removal.  The first seam operation after
        carver_load fixes the axis: width calls fail until the next load."""
        w, h = self.carver_size()
        seams = np.empty((n_seams, w), np.int32)
        _check(lib().dctc_carver_resize_height(self._h, int(n_seams), _ptr(seams) if n_seams else None),
               "dctc_carver_resize_height")
        return seams

    def carver_enlarge_height(self, n_seams):
        """lqr_carver_resize to a larger height on the device: returns the n_seams seams (as carver_resize_height does);
        the session continues on the enlarged image."""
        w, h = self.carver_size()
        seams = np.empty((n_seams, w), np.int32)
        _check(lib().dctc_carver_enlarge_height(self._h, int(n_seams), _ptr(seams) if n_seams else None),
               "dctc_carver_enlarge_height")
        return seams

    def carver_resize(self, new_w, new_h, vmaps=False):
        """lqr_carver_resize(carver, new_w, new_h) on the device (dctc_carver_resize): the width passes, then the height
        passes of resize_plan.  Returns one dict per pass: axis, enlarge, seams shaped as the per-axis method returns
        them and, with vmaps, "vmap", the pass's start-frame visibility map [h, w].  Needs a freshly loaded session;
        afterwards no seam operation until the next carver_load."""
        w, h = self.carver_size()
        return _resize(lib().dctc_carver_resize, self._h, w, h, new_w, new_h, vmaps, None)

    def carver_levels_width(self, depth):
        """The interactive dialog's build (dctc_carver_levels_width): one seam loop to depth with visibility maps and a
        copy of the start image, after which carver_render_levels shows any width within depth of the start.  Returns the
        seams as carver_resize_width does.  Needs a freshly loaded session; afterwards no seam operation until the next
        carver_load, and the getters show the image carved by depth."""
        return self._carver_levels_build(lib().dctc_carver_levels_width, "width", depth)

    def carver_levels_height(self, depth):
        """carver_levels_width along the other axis (dctc_carver_levels_height); seams as carver_resize_height."""
        return self._carver_levels_build(lib().dctc_carver_levels_height, "height", depth)

    def _carver_levels_build(self, fn, axis, depth):
        w, h = self.carver_size()
        seams = np.empty((depth, h if axis == "width" else w), np.int32)
        _check(fn(self._h, int(depth), _ptr(seams) if depth else None), fn.__name__)
        self._carver_levels = (axis, w, h)
        return seams

    def carver_render_levels(self, extents):
        """dctc_carver_render_levels: one uint8 (H_i, W_i, ch) image per extent along the built axis, each bit for bit
        what a fresh load and the resize (extent below the start) or enlarge (above) to that extent gives."""
        return _render_levels(lib().dctc_carver_render_levels, self._h, getattr(self, "_carver_levels", None), extents,
                              None, getattr(self, "_carver_ch", 1))

    def carver_set_bias(self, bias):
        """Per-pixel bias of the seam search (liblqr's lqr_carver_bias_add): float (h, w) at the current size, or None to
        clear it.  Every seam operation then runs on energy + bias / ext, ext = the start width of the frame the seam
        loop runs on (include/dctc.h); positive values preserve pixels, large negative values remove them first.  Needs
        a freshly loaded session; carver_load clears the bias."""
        if bias is None:
            _check(lib().dctc_carver_set_bias(self._h, None, 0), "dctc_carver_set_bias")
            return
        w, h = self.carver_size()
        b = _bias_plane(bias, (h, w))
        _check(lib().dctc_carver_set_bias(self._h, _ptr(b), w * 4), "dctc_carver_set_bias")

    def carver_bias(self):
        """The current bias plane (h, w): carved, transposed back and inflated with the pixels."""
        w, h = self.carver_size()
        out = np.empty((h, w), np.float32)
        _check(lib().dctc_carver_bias(self._h, _ptr(out)), "dctc_carver_bias")
        return out

    def carver_set_rigidity(self, rigidity):
        """liblqr's rigidity (lqr_carver_init): a seam step to a neighbouring column costs rigidity / h more, h the seam
        length, so larger values give straighter seams (include/dctc.h).  Applies from the next seam operation and
        survives carver_load; 0 (the default) is the plain seam search.  Raises for a negative or non-finite value."""
        _check(lib().dctc_carver_set_rigidity(self._h, float(rigidity)), "dctc_carver_set_rigidity")

    def carver_set_delta_x(self, delta_x):
        """liblqr's delta_x (lqr_carver_init): the largest number of columns a seam may move from one row to the next,
        1 .. MAX_DELTA_X (include/dctc.h).  Applies from the next seam operation and survives carver_load; 1 (the
        default) is the plug-in's value.  Raises for delta_x < 1 or above MAX_DELTA_X."""
        _check(lib().dctc_carver_set_delta_x(self._h, int(delta_x)), "dctc_carver_set_delta_x")

    def carver_set_incremental(self, on):
        """Device seam loop: update the cumulative map incrementally (liblqr's update_mmap) instead of rebuilding it."""
        _check(lib().dctc_carver_set_incremental(self._h, int(bool(on))), "dctc_carver_set_incremental")

    def carver_rebuild_count(self):
        """Full cumulative-map rebuilds the device seam loop needed since carver_load (the other seams were served by
        the incremental update)."""
        return int(lib().dctc_carver_rebuild_count(self._h))

    def preview_energy(self, img, want_image=True):
        """Preview-path operator (dct_energy_preview, src/render.c:421-501): returns (energy float map, normalised
        8-bit image with the input's channel count)."""
        img = np.asarray(img)
        if img.ndim == 2:
            img = img[:, :, None]
        img = np.ascontiguousarray(img, dtype=np.uint8)
        h, w, ch = img.shape
        en = np.empty((h, w), np.float32)
        out = np.empty((h, w, ch), np.uint8) if want_image else None
        _check(lib().dctc_preview_energy(self._h, _ptr(img), w, h, ch, w * ch, _ptr(en), _ptr(out) if want_image else None),
               "dctc_preview_energy")
        return en, out

    def carver_set_dump_vmaps(self, on=True):
        _check(lib().dctc_carver_set_dump_vmaps(self._h, int(on)), "dctc_carver_set_dump_vmaps")

    def carver_vmap(self, w0, h):
        """(visibility map of the original w0 x h pixels, depth): removal order per pixel, 0 = never removed (by vertical
        seams, or by horizontal ones after carver_resize_height / carver_enlarge_height)."""
        out = np.empty((h, w0), np.int32)
        depth = C.c_int(0)
        _check(lib().dctc_carver_vmap(self._h, _ptr(out), C.byref(depth)), "dctc_carver_vmap")
        return out, depth.value

    def carver_paint_seams(self, img):
        """display_carver_seams (src/render.c:204-240) on a copy of the original image."""
        img = np.array(img, dtype=np.uint8, order="C")
        if img.ndim == 2:
            img = img[:, :, None]
        h, w, ch = img.shape
        _check(lib().dctc_carver_paint_seams(self._h, _ptr(img), ch, w * ch), "dctc_carver_paint_seams")
        return img

    def carver_energy_image(self):
        """8-bit grey energy image of the session's current map (liblqr get_energy_image semantics)."""
        w, h = self.carver_size()
        out = np.empty((h, w), np.uint8)
        _check(lib().dctc_carver_energy_image(self._h, _ptr(out)), "dctc_carver_energy_image")
        return out

    def energy_minmax_dev(self, d_en, en_pitch, w, h):
        lo_hi = np.empty(2, np.float32)
        _check(lib().dctc_energy_minmax_dev(self._h, C.c_void_p(d_en), en_pitch, w, h, _ptr(lo_hi)), "dctc_energy_minmax_dev")
        return lo_hi

    def energy_image_dev(self, d_en, en_pitch, w, h, d_out, out_pitch, lo_hi=None, sync=True):
        p = None
        if lo_hi is not None:
            lo_hi = np.ascontiguousarray(lo_hi, dtype=np.float32)
            p = _ptr(lo_hi)
        _check(lib().dctc_energy_image_dev(self._h, C.c_void_p(d_en), en_pitch, w, h, p, C.c_void_p(d_out), out_pitch,
                                           int(sync)), "dctc_energy_image_dev")

    def carve_and_update(self, seam_x, want_band=True):
        """Removes one vertical seam; returns (band_values, xmin, xmax) like liblqr's update_emap would visit."""
        w, h = self.carver_size()
        seam = np.ascontiguousarray(seam_x, dtype=np.int32)
        if seam.shape != (h,):
            raise ValueError("seam must have one column per row")
        xmin = np.empty(h, np.int32)
        xmax = np.empty(h, np.int32)
        # at most 2 r (delta_x + 1) values per row (include/dctc.h), r = blocksize / 2
        band = np.empty(h * 2 * (self.blocksize // 2) * (MAX_DELTA_X + 1), np.float32) if want_band else None
        _check(lib().dctc_carve_and_update(self._h, _ptr(seam), _ptr(band) if want_band else None, _ptr(xmin),
                                           _ptr(xmax)), "dctc_carve_and_update")
        if want_band:
            n = int(np.maximum(xmax - xmin + 1, 0).sum())
            band = band[:n]
        return band, xmin, xmax


    def pcie_probe(self, nbytes=256 << 20, iters=8):
        """Pinned host <-> device copy bandwidth (GB/s): H2D alone, D2H alone, per direction with both running."""
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        _check(lib().dctc_pcie_probe(self._h, nbytes, iters, C.byref(a), C.byref(b), C.byref(c)), "dctc_pcie_probe")
        return {"h2d_gbs": a.value, "d2h_gbs": b.value, "bidir_gbs_per_dir": c.value}


class CarverBatch:
    """n equally sized frames retargeted together by one device seam loop (dctc_carver_batch_*): every phase of the loop
    is one launch for all frames, and each frame gets exactly what a single carver session on the same context gives
    it.  imgs: uint8 [n, h, w] or [n, h, w, ch].  Uses the context's operator and kernel selection at load time."""

    def __init__(self, ctx, imgs, dump_vmaps=False):
        imgs = self._frames(imgs)
        self.ctx = ctx
        self.n, self.h, self.w0, self.ch = imgs.shape
        self._b = C.c_void_p()
        _check(lib().dctc_carver_batch_create(ctx.handle, self.n, self.w0, self.h, self.ch, int(bool(dump_vmaps)),
                                              C.byref(self._b)), "dctc_carver_batch_create")
        try:
            self.load(imgs)
        except Exception:
            self.close()
            raise

    @staticmethod
    def _frames(imgs):
        imgs = np.asarray(imgs)
        if imgs.dtype != np.uint8:
            raise TypeError("frames must be uint8")
        if imgs.ndim == 3:
            imgs = imgs[..., None]
        if imgs.ndim != 4:
            raise ValueError("frames must be [n, h, w] or [n, h, w, ch]")
        return np.ascontiguousarray(imgs)

    def load(self, imgs):
        """Loads new frames of the batch's shape and restarts it at the original width (also after enlarge_width)."""
        imgs = self._frames(imgs)
        if imgs.shape != (self.n, self.h, self.w0, self.ch):
            raise ValueError("frames must have the batch's shape %s" % ((self.n, self.h, self.w0, self.ch),))
        self._levels = None
        _check(lib().dctc_carver_batch_load(self._b, _ptr(imgs), self.h * self.w0 * self.ch, self.w0 * self.ch),
               "dctc_carver_batch_load")

    @property
    def handle(self):
        return self._b

    @property
    def width(self):
        return int(lib().dctc_carver_batch_width(self._b))

    @property
    def height(self):
        return int(lib().dctc_carver_batch_height(self._b))

    def resize_width(self, n_seams):
        """Removes n_seams vertical seams from every frame; returns int32 [n, n_seams, h], the removed columns in the
        coordinates of each frame at the time of removal."""
        seams = np.empty((self.n, n_seams, self.h), np.int32)
        _check(lib().dctc_carver_batch_resize_width(self._b, int(n_seams), _ptr(seams) if n_seams else None),
               "dctc_carver_batch_resize_width")
        return seams

    def enlarge_width(self, n_seams):
        """lqr_carver_resize to a larger width for every frame: returns int32 [n, n_seams, h], the seams a shrink by
        n_seams would remove (as resize_width), every pixel of which is then doubled.  The frames become w0 + n_seams
        wide; vmap() keeps the start frames' maps.  No further resize until the next load()."""
        seams = np.empty((self.n, n_seams, self.h), np.int32)
        _check(lib().dctc_carver_batch_enlarge_width(self._b, int(n_seams), _ptr(seams) if n_seams else None),
               "dctc_carver_batch_enlarge_width")
        return seams

    def resize_height(self, n_seams):
        """Removes n_seams horizontal seams from every frame; returns int32 [n, n_seams, w], the removed rows in the
        coordinates of each frame at the time of removal.  The first seam operation after a load fixes the axis: width
        calls fail until the next load(), and the other way round."""
        seams = np.empty((self.n, n_seams, self.width), np.int32)
        _check(lib().dctc_carver_batch_resize_height(self._b, int(n_seams), _ptr(seams) if n_seams else None),
               "dctc_carver_batch_resize_height")
        return seams

    def enlarge_height(self, n_seams):
        """lqr_carver_resize to a larger height for every frame (enlarge_width along the other axis): returns int32
        [n, n_seams, w]; the frames become h + n_seams tall.  No further resize until the next load()."""
        seams = np.empty((self.n, n_seams, self.width), np.int32)
        _check(lib().dctc_carver_batch_enlarge_height(self._b, int(n_seams), _ptr(seams) if n_seams else None),
               "dctc_carver_batch_enlarge_height")
        return seams

    def resize(self, new_w, new_h, vmaps=False):
        """Context.carver_resize for every frame (dctc_carver_batch_resize): one dict per pass with seams
        [n, n_seams, len] and, with vmaps, "vmap" [n, h, w].  Needs a freshly loaded batch; afterwards no seam operation
        until the next load()."""
        return _resize(lib().dctc_carver_batch_resize, self._b, self.width, self.height, new_w, new_h, vmaps, self.n)

    def levels_width(self, depth):
        """Context.carver_levels_width for every frame: returns int32 [n, depth, h]."""
        return self._levels_build(lib().dctc_carver_batch_levels_width, "width", depth)

    def levels_height(self, depth):
        """Context.carver_levels_height for every frame: returns int32 [n, depth, w]."""
        return self._levels_build(lib().dctc_carver_batch_levels_height, "height", depth)

    def _levels_build(self, fn, axis, depth):
        w, h = self.width, self.height
        seams = np.empty((self.n, depth, h if axis == "width" else w), np.int32)
        _check(fn(self._b, int(depth), _ptr(seams) if depth else None), fn.__name__)
        self._levels = (axis, w, h)
        return seams

    def render_levels(self, extents):
        """Context.carver_render_levels for every frame: one uint8 (n, H_i, W_i, ch) array per extent."""
        return _render_levels(lib().dctc_carver_batch_render_levels, self._b, self._levels, extents, self.n, self.ch)

    def render_levels_dev(self, extents, d_out):
        """dctc_carver_batch_render_levels_dev into device memory at d_out (the layout of render_levels back to back);
        returns the bytes written."""
        ext = np.ascontiguousarray([int(e) for e in extents], np.int32)
        _check(lib().dctc_carver_batch_render_levels_dev(self._b, len(ext), _ptr(ext) if len(ext) else None,
                                                         C.c_void_p(d_out)), "dctc_carver_batch_render_levels_dev")
        other = self.h if self._levels is None or self._levels[0] == "width" else self._levels[1]
        return int(ext.sum()) * other * self.n * self.ch

    def set_bias(self, bias):
        """Context.carver_set_bias for every frame: float (n, h, w0), or None to clear.  Needs a freshly loaded batch;
        load() clears the bias."""
        if bias is None:
            _check(lib().dctc_carver_batch_set_bias(self._b, None, 0, 0), "dctc_carver_batch_set_bias")
            return
        b = _bias_plane(bias, (self.n, self.h, self.w0))
        _check(lib().dctc_carver_batch_set_bias(self._b, _ptr(b), self.h * self.w0 * 4, self.w0 * 4),
               "dctc_carver_batch_set_bias")

    def set_rigidity(self, rigidity):
        """Context.carver_set_rigidity for every frame of the batch: applies from the next seam operation and survives
        load()."""
        _check(lib().dctc_carver_batch_set_rigidity(self._b, float(rigidity)), "dctc_carver_batch_set_rigidity")

    def set_delta_x(self, delta_x):
        """Context.carver_set_delta_x for every frame of the batch: applies from the next seam operation and survives
        load()."""
        _check(lib().dctc_carver_batch_set_delta_x(self._b, int(delta_x)), "dctc_carver_batch_set_delta_x")

    def bias(self):
        """The current bias planes (n, height, width)."""
        out = np.empty((self.n, self.height, self.width), np.float32)
        _check(lib().dctc_carver_batch_bias(self._b, _ptr(out)), "dctc_carver_batch_bias")
        return out

    def images(self):
        out = np.empty((self.n, self.height, self.width, self.ch), np.uint8)
        _check(lib().dctc_carver_batch_images(self._b, _ptr(out)), "dctc_carver_batch_images")
        return out

    def energy(self):
        out = np.empty((self.n, self.height, self.width), np.float32)
        _check(lib().dctc_carver_batch_energy(self._b, _ptr(out)), "dctc_carver_batch_energy")
        return out

    def vmap(self):
        """(visibility maps int32 [n, h, w0], depth): removal order per original pixel, 0 = never removed (by the
        horizontal seams after resize_height / enlarge_height)."""
        out = np.empty((self.n, self.h, self.w0), np.int32)
        depth = C.c_int(0)
        _check(lib().dctc_carver_batch_vmap(self._b, _ptr(out), C.byref(depth)), "dctc_carver_batch_vmap")
        return out, depth.value

    def close(self):
        if self._b:
            lib().dctc_carver_batch_destroy(self._b)
            self._b = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def band_plan(h, world, rank, blocksize):
    """(first row, rows, halo rows needed above, below) of `rank`'s band: dctc_band_plan."""
    y0, rows, tn, bn = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    _check(lib().dctc_band_plan(h, world, rank, blocksize, C.byref(y0), C.byref(rows), C.byref(tn), C.byref(bn)), "dctc_band_plan")
    return y0.value, rows.value, tn.value, bn.value


def rendezvous_allgather(name, rank, world, blob, timeout_ms=60000):
    """All-gather of equal-sized byte strings over the ranks of one box through POSIX shared memory (no framework)."""
    blob = bytes(blob)
    mine = (C.c_ubyte * max(len(blob), 1)).from_buffer_copy(blob or b"\0")
    out = (C.c_ubyte * max(len(blob) * world, 1))()
    _check(lib().dctc_rendezvous_allgather(name.encode(), rank, world, mine, len(blob), out, timeout_ms), "dctc_rendezvous_allgather")
    raw = bytes(out)
    return [raw[i * len(blob):(i + 1) * len(blob)] for i in range(world)]


class BandRunner:
    """One rank's row band of a w x h image (one process per GPU): dctc_band_runner_*.  The halo rows are read from the
    neighbour ranks' HBM by the energy kernel (CUDA IPC peer mappings exchanged through the C rendezvous)."""

    def __init__(self, ctx, rendezvous, rank, world, w, h, ch):
        self.ctx, self.rank, self.world, self.w, self.h, self.ch = ctx, rank, world, w, h, ch
        self._r = C.c_void_p()
        _check(lib().dctc_band_runner_create(ctx.handle, rendezvous.encode(), rank, world, w, h, ch, C.byref(self._r)),
               "dctc_band_runner_create")
        y0, rows, pitch = C.c_int(), C.c_int(), C.c_size_t()
        _check(lib().dctc_band_runner_geometry(self._r, C.byref(y0), C.byref(rows), C.byref(pitch)), "dctc_band_runner_geometry")
        self.y0, self.band_rows, self.pitch = y0.value, rows.value, pitch.value

    def synth(self, seed, pattern=0):
        _check(lib().dctc_band_runner_synth(self._r, seed, pattern), "dctc_band_runner_synth")

    def upload(self, band_rows):
        a = np.ascontiguousarray(band_rows, dtype=np.uint8)
        _check(lib().dctc_band_runner_upload(self._r, _ptr(a), self.w * self.ch), "dctc_band_runner_upload")

    def connect(self):
        _check(lib().dctc_band_runner_connect(self._r), "dctc_band_runner_connect")

    def barrier(self):
        _check(lib().dctc_band_runner_barrier(self._r), "dctc_band_runner_barrier")

    def step(self, sync=False):
        _check(lib().dctc_band_runner_energy(self._r, int(sync)), "dctc_band_runner_energy")

    def fetch(self):
        out = np.empty((self.band_rows, self.w), np.float32)
        _check(lib().dctc_band_runner_download(self._r, _ptr(out)), "dctc_band_runner_download")
        return out

    def energy_image(self):
        out = np.empty((self.band_rows, self.w), np.uint8)
        _check(lib().dctc_band_runner_energy_image(self._r, _ptr(out)), "dctc_band_runner_energy_image")
        return out

    def energy_dev(self):
        """Device address of this band's float32 energy rows (row pitch w)."""
        return lib().dctc_band_runner_energy_dev(self._r)

    def close(self):
        if self._r:
            lib().dctc_band_runner_destroy(self._r)
            self._r = C.c_void_p()


class Multi:
    """All GPUs of the box from one process: dctc_multi_* (frames round-robin, row bands with peer halo reads)."""

    def __init__(self, devices=None, blocksize=8, edges=0.5, textures=0.5, kernel=KERNEL_AUTO):
        self._m = C.c_void_p()
        if devices is None:
            _check(lib().dctc_multi_create(C.byref(self._m), None, 0), "dctc_multi_create")
        else:
            arr = (C.c_int * len(devices))(*devices)
            _check(lib().dctc_multi_create(C.byref(self._m), arr, len(devices)), "dctc_multi_create")
        self.n = lib().dctc_multi_device_count(self._m)
        self.set_params(blocksize, edges, textures)
        if kernel != KERNEL_AUTO:
            _check(lib().dctc_multi_set_kernel(self._m, kernel), "dctc_multi_set_kernel")
        self._bands = C.c_void_p()

    def set_params(self, blocksize, edges, textures):
        p = EnergyParameters(edges=edges, textures=textures, blocksize=blocksize)
        _check(lib().dctc_multi_set_params(self._m, C.byref(p)), "dctc_multi_set_params")

    @property
    def launches(self):
        return int(lib().dctc_multi_launch_count(self._m))

    def energy_batch(self, imgs, out=None):
        n, h, w, ch = imgs.shape
        if out is None:
            out = np.empty((n, h, w), np.float32)
        _check(lib().dctc_multi_energy_batch(self._m, _ptr(imgs), n, h * w * ch, w, h, ch, w * ch, _ptr(out), h * w),
               "dctc_multi_energy_batch")
        return out

    def energy_bands(self, img, want_image=False):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        if img.ndim == 2:
            img = img[:, :, None]
        h, w, ch = img.shape
        out = np.empty((h, w), np.float32)
        im8 = np.empty((h, w), np.uint8) if want_image else None
        _check(lib().dctc_multi_energy_bands(self._m, _ptr(img), w, h, ch, w * ch, _ptr(out), _ptr(im8) if want_image else None),
               "dctc_multi_energy_bands")
        return (out, im8) if want_image else out

    # device-resident bands (bench)
    def bands_create(self, w, h, ch):
        self.bands_destroy()
        _check(lib().dctc_multi_bands_create(self._m, w, h, ch, C.byref(self._bands)), "dctc_multi_bands_create")
        self._bw, self._bh = w, h

    def bands_synth(self, seed, pattern=0):
        _check(lib().dctc_multi_bands_synth(self._bands, seed, pattern), "dctc_multi_bands_synth")

    def bands_energy(self, sync=False):
        _check(lib().dctc_multi_bands_energy(self._bands, int(sync)), "dctc_multi_bands_energy")

    def bands_download(self):
        out = np.empty((self._bh, self._bw), np.float32)
        _check(lib().dctc_multi_bands_download(self._bands, _ptr(out)), "dctc_multi_bands_download")
        return out

    def bands_destroy(self):
        if self._bands:
            lib().dctc_multi_bands_destroy(self._bands)
            self._bands = C.c_void_p()

    def close(self):
        self.bands_destroy()
        if self._m:
            lib().dctc_multi_destroy(self._m)
            self._m = C.c_void_p()
