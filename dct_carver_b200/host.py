"""ctypes mirror of the host-side C (dct_carver_b200/host/dctc_lqr.h): the carver that stands where liblqr stands
for the reference, and the render()-like driver (src/render.c:327-419)."""
import ctypes as C
import os

import numpy as np

from . import DctcError, lib as _corelib

_HERE = os.path.dirname(os.path.abspath(__file__))
HOST_LIB_PATH = os.path.join(_HERE, "libdctc_host.so")
_host = None

ENERGY_FUNC = C.CFUNCTYPE(C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p)


class PlugInVals(C.Structure):
    """src/main.h:12-22"""
    _fields_ = [("edges", C.c_float), ("textures", C.c_float), ("blocksize", C.c_int), ("seams_number", C.c_int),
                ("new_layer", C.c_int), ("resize_canvas", C.c_int), ("output_energy", C.c_int),
                ("output_seams", C.c_int), ("vertically", C.c_int)]


class RenderResult(C.Structure):
    _fields_ = [("image", C.POINTER(C.c_uint8)), ("new_w", C.c_int), ("new_h", C.c_int), ("channels", C.c_int),
                ("energy_image", C.POINTER(C.c_uint8)), ("vmap", C.POINTER(C.c_int)), ("vmap_depth", C.c_int),
                ("seams", C.POINTER(C.c_int)), ("n_seams", C.c_int), ("seam_len", C.c_int),
                ("t_energy", C.c_double), ("t_mmap", C.c_double), ("t_seam", C.c_double), ("t_total", C.c_double)]


def hostlib():
    global _host
    if _host is None:
        if not os.path.exists(HOST_LIB_PATH):
            raise ImportError("%s missing — run `make -C dct_carver_b200/host`" % HOST_LIB_PATH)
        _corelib()
        L = C.CDLL(HOST_LIB_PATH)
        L.dctc_render.restype = C.c_int
        L.dctc_render.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(PlugInVals), C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.POINTER(RenderResult)]
        L.dctc_render_ext.restype = C.c_int
        L.dctc_render_ext.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(PlugInVals), C.c_int, C.c_float,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RenderResult)]
        L.dctc_host_set_device_seam_loop.restype = None
        L.dctc_host_set_device_seam_loop.argtypes = [C.c_int]
        L.dctc_render_result_free.restype = None
        L.dctc_render_result_free.argtypes = [C.POINTER(RenderResult)]
        _host = L
    return _host


def render(img, seams_number, blocksize=8, edges=0.5, textures=0.5, vertically=False, ctx=None, callback=None,
           callback_extra=None, output_energy=False, output_seams=True, device_loop=True, delta_x=1, rigidity=0.0):
    """Retargets `img` by `seams_number` (negative = shrink, as PlugInVals.seams_number) along the width
    (vertically=False) or height.  Energy comes from the GPU context `ctx`, or from a per-pixel `callback`
    (address of an LqrEnergyFunc; checker use only).  device_loop=False keeps the cumulative map, seam search and
    carve on the host (energy batches still on the GPU): the cross-check of the device-resident seam loop.
    delta_x, rigidity: lqr_carver_init's (dctc_render_ext); the defaults are the plug-in's."""
    img = np.ascontiguousarray(img, dtype=np.uint8)
    if img.ndim == 2:
        img = img[:, :, None]
    h, w, ch = img.shape
    hostlib().dctc_host_set_device_seam_loop(int(device_loop))
    vals = PlugInVals(edges, textures, blocksize, seams_number, 0, 1, int(output_energy), int(output_seams), int(vertically))
    res = RenderResult()
    rc = hostlib().dctc_render_ext(img.ctypes.data, w, h, ch, C.byref(vals), int(delta_x), float(rigidity),
                                   ctx.handle if ctx is not None else None, callback, callback_extra, C.byref(res))
    if rc != 0:
        raise DctcError(rc, "dctc_render")
    out = dict(
        image=np.ctypeslib.as_array(res.image, (res.new_h, res.new_w, res.channels)).copy(),
        seams=(np.ctypeslib.as_array(res.seams, (res.n_seams, res.seam_len)).copy() if res.n_seams else
               np.zeros((0, 0), np.int32)),
        energy_image=(np.ctypeslib.as_array(res.energy_image, (h, w)).copy() if output_energy else None),
        vmap=(np.ctypeslib.as_array(res.vmap, (h, w) if not vertically else (w, h)).copy() if bool(res.vmap) else None),
        vmap_depth=res.vmap_depth,
        t_energy=res.t_energy, t_mmap=res.t_mmap, t_seam=res.t_seam, t_total=res.t_total,
    )
    hostlib().dctc_render_result_free(C.byref(res))
    return out
