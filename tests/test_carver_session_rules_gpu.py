"""The state rules of the two carver sessions side by side: the context's single session (dctc_carver_*) and a batch
session of two frames (dctc_carver_batch_*) run the same scripted sequences, and after every call the status, the
launches it made (dctc_launch_count), the width and height, and the CRC-32 of every returned array (per frame) must
match the table below.  Frame 0 of the batch is the single session's image, so where the rules agree the two columns
agree too; where they differ the table says how:
  - operator: the single session uses the context's operator at each call, a batch the one it had at its load;
  - after an enlarge: the single session continues on the enlarged frames, a batch refuses seam operations
    (n_seams = 0 included) until the next load;
  - n_seams = 0 after a combined resize: DCTC_OK for the single session, DCTC_ERR_STATE for a batch;
  - visibility maps: requested per call on the single session (made by the first recording loop, refused once that
    frame is carved), fixed at create for a batch (reset at load and at the axis switch); an enlarge always records.
Steps: load, bias / nobias (set or clear the bias), rw / rh / ew / eh k (resize or enlarge width / height by k), rs /
rsv w h (combined resize without / with maps), img / en / bi / vm / ps (image, energy, bias, visibility map, painted
seams), par4 / par8 (dctc_set_params block size), tile / auto (dctc_set_kernel), dv1 / dv0 (single session only:
dctc_carver_set_dump_vmaps).  "ps" and "dv" do not apply to a batch ("-")."""
import ctypes as C
import zlib

import numpy as np
import pytest

import dct_carver_b200 as dc
import oracle_lib as ol

pytestmark = pytest.mark.gpu

W, H, CH, N = 24, 16, 3, 2
WIDE = 8 * 8 * (512 - 2 * 32) + 1   # one column wider than the device seam DP covers
STATUS = {dc.OK: "OK", dc.ERR_INVALID: "INVALID", dc.ERR_STATE: "STATE", dc.ERR_UNSUPPORTED: "UNSUPPORTED"}

# name: (frame width, height, channels, batch created with dump_vmaps, steps)
SCENARIOS = {
    "load_getters": (W, H, CH, True, "img en bi vm ps load img en bi vm ps rw 0 rh 0 vm ps"),
    "bias": (W, H, CH, False, "load bias bi en img rw 2 bias nobias bi en load bi bias rh 1 bi en img load bias ew 2 bi en "
                              "rw 1 load bias rsv 20 18 bi en load bias nobias bi en"),
    "zero_one": (W, H, CH, True, "dv1 load rw 0 rh 0 ew 0 eh 0 rw 1 rh 0 rh 1 eh 0 eh 1 ew 0 ew 1 vm ps img en rw 1 vm ps "
                                 "load rh 1 rw 0 rw 1 ew 0 ew 1 vm ps img en"),
    "enlarge_width": (W, H, CH, True, "dv1 load ew 3 img en vm ps rw 0 rh 0 rh 1 eh 0 eh 1 ew 0 ew 2 img en vm ps rw 1 vm "
                                      "ps ew 1 rs 20 20 rsv 20 20 img en"),
    "enlarge_width_maps_off": (W, H, CH, False, "load ew 3 vm ps rw 1 vm ps dv1 rw 1 ew 1 vm dv0 rw 1 img en vm"),
    "enlarge_height": (W, H, CH, True, "dv1 load eh 3 img en vm ps rh 0 rw 0 rw 1 ew 0 ew 1 eh 0 eh 2 img en vm rh 1 vm "
                                       "ps rs 20 20 img en"),
    "enlarge_height_maps_off": (W, H, CH, False, "load eh 2 vm ps dv1 rh 1 vm ps eh 1 dv0 rh 1 vm img en"),
    "resize_then": (W, H, CH, True, "dv1 load rsv 20 19 img en vm ps bi rw 0 rw 1 rh 0 rh 1 ew 0 ew 1 eh 0 eh 1 rs 20 19 "
                                    "rs 24 16 img en load rs 24 16 rw 1 img load rsv 50 40 img en vm load rs 30 12 img "
                                    "en rw 0 vm"),
    "params": (W, H, CH, False, "load par4 rw 2 img en par8 tile rw 1 img en auto load ew 2 par4 rw 1 en img par8 load "
                                "rh 1 tile rh 1 en auto rs 20 12 img"),
    "dump_toggle": (W, H, CH, True, "load dv1 rw 2 vm ps dv0 rw 1 vm dv1 rw 1 vm ps dv0 load rh 2 vm dv1 rh 1 vm dv0 "
                                    "load dv1 rh 1 vm ps rsv 20 12 vm"),
    "dp_wide": (WIDE, 2, 1, False, "load rw 1 ew 1 rs 100 2 img rh 1 img"),
    "dp_tall": (2, WIDE, 1, False, "load rh 1 eh 1 rs 2 100 img rw 1 img"),
}


def frames(w, h, ch):
    return np.stack([ol.synth_image(w, h, ch, seed, 0).reshape(h, w, ch) for seed in (1, 2)])


def bias_planes(w, h):
    return np.random.default_rng(7).uniform(-300, 300, (N, h, w)).astype(np.float32)


def crc(a, n):
    """CRC-32 of each of the n frames of a flat array"""
    return ",".join("%08x" % zlib.crc32(p.tobytes()) for p in np.split(a, n))


class Session:
    """One session driven through the raw C ABI: the single session (batch=None) or a batch of N frames"""

    def __init__(self, ctx, w, h, ch, batch):
        self.L, self.ctx, self.w0, self.h0, self.ch = dc.lib(), ctx, w, h, ch
        self.imgs = frames(w, h, ch)
        self.bias = bias_planes(w, h)
        self.b = batch
        self.n = N if batch else 1
        self.s = batch if batch else ctx.handle

    def size(self):
        if self.b:
            return self.L.dctc_carver_batch_width(self.b), self.L.dctc_carver_batch_height(self.b)
        return self.L.dctc_carver_width(self.s), self.L.dctc_carver_height(self.s)

    def call(self, single, batch, *args):
        return getattr(self.L, batch if self.b else single)(self.s, *args)

    def step(self, op, arg):
        """(status, checksums) of one step; None for a step that does not apply to the session"""
        L, n = self.L, self.n
        w, h = self.size()
        if op in ("dv1", "dv0"):
            return None if self.b else (L.dctc_carver_set_dump_vmaps(self.s, int(op == "dv1")), "")
        if op == "ps":
            if self.b:
                return None
            img = np.full((256, 256, self.ch), 77, np.uint8)
            st = L.dctc_carver_paint_seams(self.s, img.ctypes.data, self.ch, 256 * self.ch)
            return st, crc(img.ravel(), 1) if st == dc.OK else ""
        if op in ("par4", "par8"):
            p = dc.EnergyParameters(edges=0.5, textures=0.5, blocksize=int(op[3:]))
            return L.dctc_set_params(self.ctx.handle, C.byref(p)), ""
        if op in ("tile", "auto"):
            return L.dctc_set_kernel(self.ctx.handle, dc.KERNEL_FP32_TILE if op == "tile" else dc.KERNEL_AUTO), ""
        if op == "load":
            if self.b:
                st = L.dctc_carver_batch_load(self.b, self.imgs.ctypes.data, self.imgs[0].nbytes, self.w0 * self.ch)
            else:
                st = L.dctc_carver_load(self.s, self.imgs[0].ctypes.data, self.w0, self.h0, self.ch, self.w0 * self.ch)
            return st, ""
        if op in ("bias", "nobias"):
            p = self.bias.ctypes.data if op == "bias" else None
            if self.b:
                return L.dctc_carver_batch_set_bias(self.b, p, self.bias[0].nbytes, self.w0 * 4), ""
            return L.dctc_carver_set_bias(self.s, p, self.w0 * 4), ""
        if op in ("img", "en", "bi"):
            out = np.full(max(n * w * h * (self.ch if op == "img" else 1), 1), 0xAB,
                          np.uint8 if op == "img" else np.float32)
            fn = {"img": ("dctc_carver_image", "dctc_carver_batch_images"),
                  "en": ("dctc_carver_energy", "dctc_carver_batch_energy"),
                  "bi": ("dctc_carver_bias", "dctc_carver_batch_bias")}[op]
            st = self.call(*fn, out.ctypes.data)
            return st, crc(out, n) if st == dc.OK else ""
        if op == "vm":
            out = np.full(n * 4096, -1, np.int32)
            depth = C.c_int(-1)
            st = self.call("dctc_carver_vmap", "dctc_carver_batch_vmap", out.ctypes.data, C.byref(depth))
            return st, "d%d:%s" % (depth.value, crc(out, n)) if st == dc.OK else ""
        raise ValueError(op)

    def seams(self, op, k):
        w, h = self.size()
        out = np.full(max(self.n * k * (h if op[1] == "w" else w), 1), -1, np.int32)
        fn = {"rw": "resize_width", "rh": "resize_height", "ew": "enlarge_width", "eh": "enlarge_height"}[op]
        st = self.call("dctc_carver_" + fn, "dctc_carver_batch_" + fn, k, out.ctypes.data if k else None)
        return st, crc(out, self.n) if st == dc.OK and k else ""

    def resize(self, op, new_w, new_h):
        seams = np.full(self.n * 8192, -1, np.int32)
        maps = np.full(self.n * 16384, -1, np.int32) if op == "rsv" else None
        st = self.call("dctc_carver_resize", "dctc_carver_batch_resize", new_w, new_h, seams.ctypes.data,
                       maps.ctypes.data if maps is not None else None)
        sums = "%08x" % zlib.crc32(seams.tobytes() + (maps.tobytes() if maps is not None else b""))
        return st, sums if st == dc.OK else ""


def record(name, batched):
    """The rows of one scenario on one session: 'step: status +launches wxh checksums'"""
    w, h, ch, dump, script = SCENARIOS[name]
    ctx = dc.Context(0)
    b = C.c_void_p()
    try:
        if batched:
            assert dc.lib().dctc_carver_batch_create(ctx.handle, N, w, h, ch, int(dump), C.byref(b)) == dc.OK
        s = Session(ctx, w, h, ch, b if batched else None)
        tok, rows = script.split(), []
        while tok:
            op = tok.pop(0)
            args = []
            if op in ("rw", "rh", "ew", "eh"):
                args = [int(tok.pop(0))]
            elif op in ("rs", "rsv"):
                args = [int(tok.pop(0)), int(tok.pop(0))]
            label = " ".join([op] + [str(a) for a in args])
            l0 = ctx.launches
            r = s.seams(op, *args) if len(args) == 1 else s.resize(op, *args) if args else s.step(op, None)
            if r is None:
                rows.append(label + ": -")
                continue
            st, sums = r
            sw, sh = s.size()
            rows.append(("%s: %s +%d %dx%d %s" % (label, STATUS.get(st, st), ctx.launches - l0, sw, sh, sums)).rstrip())
        return rows
    finally:
        if batched:
            dc.lib().dctc_carver_batch_destroy(b)
        ctx.close()


EXPECTED = {('bias', 'batch'): ['load: OK +1 24x16',
                     'bias: OK +2 24x16',
                     'bi: OK +0 24x16 df7e7071,cc89ffac',
                     'en: OK +1 24x16 c6aa44c0,3add3ad6',
                     'img: OK +0 24x16 7d9bfc4e,574f3dca',
                     'rw 2: OK +10 22x16 926c46fa,773a0b78',
                     'bias: STATE +0 22x16',
                     'nobias: STATE +0 22x16',
                     'bi: OK +0 22x16 f49740c9,4e9d40c9',
                     'en: OK +1 22x16 1a14eda6,526cab12',
                     'load: OK +1 24x16',
                     'bi: STATE +0 24x16',
                     'bias: OK +2 24x16',
                     'rh 1: OK +9 24x15 db980363,59277d10',
                     'bi: OK +1 24x15 30789f22,1a198a0a',
                     'en: OK +2 24x15 6c3faf98,1e61ce82',
                     'img: OK +1 24x15 e24934dc,a729fe15',
                     'load: OK +1 24x16',
                     'bias: OK +2 24x16',
                     'ew 2: OK +16 26x16 926c46fa,773a0b78',
                     'bi: OK +0 26x16 e74aa292,189aa3df',
                     'en: OK +1 26x16 15f049ca,ed3e1103',
                     'rw 1: STATE +0 26x16',
                     'load: OK +1 24x16',
                     'bias: OK +2 24x16',
                     'rsv 20 18: OK +46 20x18 c6370943',
                     'bi: OK +1 20x18 34e763ac,53ae3aed',
                     'en: OK +2 20x18 ce0aa951,8193716a',
                     'load: OK +1 24x16',
                     'bias: OK +2 24x16',
                     'nobias: OK +1 24x16',
                     'bi: STATE +0 24x16',
                     'en: OK +0 24x16 c6aa44c0,3add3ad6'],
 ('bias', 'single'): ['load: OK +1 24x16',
                      'bias: OK +2 24x16',
                      'bi: OK +0 24x16 df7e7071',
                      'en: OK +1 24x16 c6aa44c0',
                      'img: OK +0 24x16 7d9bfc4e',
                      'rw 2: OK +10 22x16 926c46fa',
                      'bias: STATE +0 22x16',
                      'nobias: STATE +0 22x16',
                      'bi: OK +0 22x16 f49740c9',
                      'en: OK +1 22x16 1a14eda6',
                      'load: OK +1 24x16',
                      'bi: STATE +0 24x16',
                      'bias: OK +2 24x16',
                      'rh 1: OK +9 24x15 db980363',
                      'bi: OK +1 24x15 30789f22',
                      'en: OK +2 24x15 6c3faf98',
                      'img: OK +1 24x15 e24934dc',
                      'load: OK +1 24x16',
                      'bias: OK +2 24x16',
                      'ew 2: OK +16 26x16 926c46fa',
                      'bi: OK +0 26x16 e74aa292',
                      'en: OK +1 26x16 15f049ca',
                      'rw 1: OK +5 25x16 6090078a',
                      'load: OK +1 24x16',
                      'bias: OK +2 24x16',
                      'rsv 20 18: OK +46 20x18 8846cdb5',
                      'bi: OK +1 20x18 34e763ac',
                      'en: OK +2 20x18 ce0aa951',
                      'load: OK +1 24x16',
                      'bias: OK +2 24x16',
                      'nobias: OK +1 24x16',
                      'bi: STATE +0 24x16',
                      'en: OK +0 24x16 c6aa44c0'],
 ('dp_tall', 'batch'): ['load: OK +1 2x28673',
                        'rh 1: UNSUPPORTED +0 2x28673',
                        'eh 1: UNSUPPORTED +0 2x28673',
                        'rs 2 100: UNSUPPORTED +0 2x28673',
                        'img: OK +0 2x28673 3792a7cf,e9038969',
                        'rw 1: OK +3 1x28673 92e6bed7,3274f7b5',
                        'img: OK +0 1x28673 c1c75de8,70fd8a7c'],
 ('dp_tall', 'single'): ['load: OK +1 2x28673',
                         'rh 1: UNSUPPORTED +0 2x28673',
                         'eh 1: UNSUPPORTED +0 2x28673',
                         'rs 2 100: UNSUPPORTED +0 2x28673',
                         'img: OK +0 2x28673 3792a7cf',
                         'rw 1: OK +3 1x28673 92e6bed7',
                         'img: OK +0 1x28673 c1c75de8'],
 ('dp_wide', 'batch'): ['load: OK +1 28673x2',
                        'rw 1: UNSUPPORTED +0 28673x2',
                        'ew 1: UNSUPPORTED +0 28673x2',
                        'rs 100 2: UNSUPPORTED +0 28673x2',
                        'img: OK +0 28673x2 b0e6431b,f8d9a23f',
                        'rh 1: OK +5 28673x1 36c56f12,08984038',
                        'img: OK +1 28673x1 5fe8a98d,b2964d40'],
 ('dp_wide', 'single'): ['load: OK +1 28673x2',
                         'rw 1: UNSUPPORTED +0 28673x2',
                         'ew 1: UNSUPPORTED +0 28673x2',
                         'rs 100 2: UNSUPPORTED +0 28673x2',
                         'img: OK +0 28673x2 b0e6431b',
                         'rh 1: OK +5 28673x1 36c56f12',
                         'img: OK +1 28673x1 5fe8a98d'],
 ('dump_toggle', 'batch'): ['load: OK +2 24x16',
                            'dv1: -',
                            'rw 2: OK +12 22x16 1a1c5295,bcc63558',
                            'vm: OK +0 22x16 d2:79093999,690b37d3',
                            'ps: -',
                            'dv0: -',
                            'rw 1: OK +6 21x16 9d693235,109c6499',
                            'vm: OK +0 21x16 d3:4f379022,690b37d3',
                            'dv1: -',
                            'rw 1: OK +6 20x16 4609a845,71534ba0',
                            'vm: OK +0 20x16 d4:3a6c8b6a,690b37d3',
                            'ps: -',
                            'dv0: -',
                            'load: OK +2 24x16',
                            'rh 2: OK +15 24x14 dcc20a17,890f262d',
                            'vm: OK +1 24x14 d2:3af388cd,690b37d3',
                            'dv1: -',
                            'rh 1: OK +6 24x13 1c85c46e,088d75a6',
                            'vm: OK +1 24x13 d3:41dc8d9f,690b37d3',
                            'dv0: -',
                            'load: OK +2 24x16',
                            'dv1: -',
                            'rh 1: OK +9 24x15 45cd0f61,f24c7d9c',
                            'vm: OK +1 24x15 d1:8aa5638e,690b37d3',
                            'ps: -',
                            'rsv 20 12: STATE +0 24x15',
                            'vm: OK +1 24x15 d1:8aa5638e,690b37d3'],
 ('dump_toggle', 'single'): ['load: OK +1 24x16',
                             'dv1: OK +0 24x16',
                             'rw 2: OK +13 22x16 1a1c5295',
                             'vm: OK +0 22x16 d2:d04bb1c5',
                             'ps: OK +1 22x16 4a584464',
                             'dv0: OK +0 22x16',
                             'rw 1: OK +5 21x16 9d693235',
                             'vm: OK +0 21x16 d2:d04bb1c5',
                             'dv1: OK +0 21x16',
                             'rw 1: OK +6 20x16 4609a845',
                             'vm: OK +0 20x16 d3:2c9e7702',
                             'ps: OK +1 20x16 465da414',
                             'dv0: OK +0 20x16',
                             'load: OK +1 24x16',
                             'rh 2: OK +12 24x14 dcc20a17',
                             'vm: STATE +0 24x14',
                             'dv1: OK +0 24x14',
                             'rh 1: STATE +0 24x14',
                             'vm: STATE +0 24x14',
                             'dv0: OK +0 24x14',
                             'load: OK +1 24x16',
                             'dv1: OK +0 24x16',
                             'rh 1: OK +9 24x15 45cd0f61',
                             'vm: OK +1 24x15 d1:974e1280',
                             'ps: OK +2 24x15 290afbbe',
                             'rsv 20 12: STATE +0 24x15',
                             'vm: OK +1 24x15 d1:974e1280'],
 ('enlarge_height', 'batch'): ['dv1: -',
                               'load: OK +2 24x16',
                               'eh 3: OK +23 24x19 23c456e0,619f21f3',
                               'img: OK +1 24x19 afee2efe,efdc105b',
                               'en: OK +1 24x19 6d49d72d,2f1242de',
                               'vm: OK +1 24x19 d3:41dc8d9f,690b37d3',
                               'ps: -',
                               'rh 0: STATE +0 24x19',
                               'rw 0: STATE +0 24x19',
                               'rw 1: STATE +0 24x19',
                               'ew 0: STATE +0 24x19',
                               'ew 1: STATE +0 24x19',
                               'eh 0: STATE +0 24x19',
                               'eh 2: STATE +0 24x19',
                               'img: OK +1 24x19 afee2efe,efdc105b',
                               'en: OK +1 24x19 6d49d72d,2f1242de',
                               'vm: OK +1 24x19 d3:41dc8d9f,690b37d3',
                               'rh 1: STATE +0 24x19',
                               'vm: OK +1 24x19 d3:41dc8d9f,690b37d3',
                               'ps: -',
                               'rs 20 20: STATE +0 24x19',
                               'img: OK +1 24x19 afee2efe,efdc105b',
                               'en: OK +1 24x19 6d49d72d,2f1242de'],
 ('enlarge_height', 'single'): ['dv1: OK +0 0x0',
                                'load: OK +1 24x16',
                                'eh 3: OK +23 24x19 23c456e0',
                                'img: OK +1 24x19 afee2efe',
                                'en: OK +1 24x19 6d49d72d',
                                'vm: OK +1 24x19 d3:bdb504b0',
                                'ps: OK +2 24x19 53446bbf',
                                'rh 0: OK +0 24x19',
                                'rw 0: OK +0 24x19',
                                'rw 1: STATE +0 24x19',
                                'ew 0: OK +0 24x19',
                                'ew 1: STATE +0 24x19',
                                'eh 0: OK +0 24x19',
                                'eh 2: OK +15 24x21 da4def95',
                                'img: OK +1 24x21 5d10cbc6',
                                'en: OK +1 24x21 ca5beef2',
                                'vm: OK +1 24x21 d2:3e5855bd',
                                'rh 1: OK +7 24x20 1faa4840',
                                'vm: OK +1 24x20 d1:8fbbade6',
                                'ps: OK +2 24x20 c324ebe3',
                                'rs 20 20: STATE +0 24x20',
                                'img: OK +1 24x20 c2c21c77',
                                'en: OK +1 24x20 f24f8771'],
 ('enlarge_height_maps_off', 'batch'): ['load: OK +1 24x16',
                                        'eh 2: OK +17 24x18 dcc20a17,890f262d',
                                        'vm: STATE +0 24x18',
                                        'ps: -',
                                        'dv1: -',
                                        'rh 1: STATE +0 24x18',
                                        'vm: STATE +0 24x18',
                                        'ps: -',
                                        'eh 1: STATE +0 24x18',
                                        'dv0: -',
                                        'rh 1: STATE +0 24x18',
                                        'vm: STATE +0 24x18',
                                        'img: OK +1 24x18 bcd413b6,5e42b707',
                                        'en: OK +1 24x18 9de56c00,ca59aba4'],
 ('enlarge_height_maps_off', 'single'): ['load: OK +1 24x16',
                                         'eh 2: OK +17 24x18 dcc20a17',
                                         'vm: OK +1 24x18 d2:8478e522',
                                         'ps: OK +2 24x18 cd01e21a',
                                         'dv1: OK +0 24x18',
                                         'rh 1: OK +7 24x17 e8e1fdfd',
                                         'vm: OK +1 24x17 d1:92e45b09',
                                         'ps: OK +2 24x17 8e561a40',
                                         'eh 1: STATE +0 24x17',
                                         'dv0: OK +0 24x17',
                                         'rh 1: OK +5 24x16 94209077',
                                         'vm: OK +1 24x16 d1:92e45b09',
                                         'img: OK +1 24x16 2a180fc5',
                                         'en: OK +1 24x16 acc5c1e1'],
 ('enlarge_width', 'batch'): ['dv1: -',
                              'load: OK +2 24x16',
                              'ew 3: OK +20 27x16 dfbbf99c,4d5385e6',
                              'img: OK +0 27x16 8568cbc6,97dfa1ec',
                              'en: OK +0 27x16 0878a69b,80c73214',
                              'vm: OK +0 27x16 d3:4f379022,690b37d3',
                              'ps: -',
                              'rw 0: STATE +0 27x16',
                              'rh 0: STATE +0 27x16',
                              'rh 1: STATE +0 27x16',
                              'eh 0: STATE +0 27x16',
                              'eh 1: STATE +0 27x16',
                              'ew 0: STATE +0 27x16',
                              'ew 2: STATE +0 27x16',
                              'img: OK +0 27x16 8568cbc6,97dfa1ec',
                              'en: OK +0 27x16 0878a69b,80c73214',
                              'vm: OK +0 27x16 d3:4f379022,690b37d3',
                              'ps: -',
                              'rw 1: STATE +0 27x16',
                              'vm: OK +0 27x16 d3:4f379022,690b37d3',
                              'ps: -',
                              'ew 1: STATE +0 27x16',
                              'rs 20 20: STATE +0 27x16',
                              'rsv 20 20: STATE +0 27x16',
                              'img: OK +0 27x16 8568cbc6,97dfa1ec',
                              'en: OK +0 27x16 0878a69b,80c73214'],
 ('enlarge_width', 'single'): ['dv1: OK +0 0x0',
                               'load: OK +1 24x16',
                               'ew 3: OK +21 27x16 dfbbf99c',
                               'img: OK +0 27x16 8568cbc6',
                               'en: OK +0 27x16 0878a69b',
                               'vm: OK +0 27x16 d3:e91fe95d',
                               'ps: OK +1 27x16 13b6c0f7',
                               'rw 0: OK +0 27x16',
                               'rh 0: OK +0 27x16',
                               'rh 1: STATE +0 27x16',
                               'eh 0: OK +0 27x16',
                               'eh 1: STATE +0 27x16',
                               'ew 0: OK +0 27x16',
                               'ew 2: OK +15 29x16 c07bdcbb',
                               'img: OK +0 29x16 31de8707',
                               'en: OK +0 29x16 19477c1d',
                               'vm: OK +0 29x16 d2:83ec6131',
                               'ps: OK +1 29x16 0fb8b626',
                               'rw 1: OK +7 28x16 d3bbf101',
                               'vm: OK +0 28x16 d1:f2024187',
                               'ps: OK +1 28x16 dab16035',
                               'ew 1: STATE +0 28x16',
                               'rs 20 20: STATE +0 28x16',
                               'rsv 20 20: STATE +0 28x16',
                               'img: OK +0 28x16 080704e2',
                               'en: OK +0 28x16 b8090a42'],
 ('enlarge_width_maps_off', 'batch'): ['load: OK +1 24x16',
                                       'ew 3: OK +21 27x16 dfbbf99c,4d5385e6',
                                       'vm: STATE +0 27x16',
                                       'ps: -',
                                       'rw 1: STATE +0 27x16',
                                       'vm: STATE +0 27x16',
                                       'ps: -',
                                       'dv1: -',
                                       'rw 1: STATE +0 27x16',
                                       'ew 1: STATE +0 27x16',
                                       'vm: STATE +0 27x16',
                                       'dv0: -',
                                       'rw 1: STATE +0 27x16',
                                       'img: OK +0 27x16 8568cbc6,97dfa1ec',
                                       'en: OK +0 27x16 0878a69b,80c73214',
                                       'vm: STATE +0 27x16'],
 ('enlarge_width_maps_off', 'single'): ['load: OK +1 24x16',
                                        'ew 3: OK +21 27x16 dfbbf99c',
                                        'vm: OK +0 27x16 d3:e91fe95d',
                                        'ps: OK +1 27x16 13b6c0f7',
                                        'rw 1: OK +5 26x16 ba9972d4',
                                        'vm: OK +0 26x16 d3:e91fe95d',
                                        'ps: OK +1 26x16 13b6c0f7',
                                        'dv1: OK +0 26x16',
                                        'rw 1: STATE +0 26x16',
                                        'ew 1: STATE +0 26x16',
                                        'vm: OK +0 26x16 d3:e91fe95d',
                                        'dv0: OK +0 26x16',
                                        'rw 1: OK +5 25x16 ee4b053c',
                                        'img: OK +0 25x16 ded11155',
                                        'en: OK +0 25x16 2c8a349a',
                                        'vm: OK +0 25x16 d3:e91fe95d'],
 ('load_getters', 'batch'): ['img: STATE +0 24x16',
                             'en: STATE +0 24x16',
                             'bi: STATE +0 24x16',
                             'vm: STATE +0 24x16',
                             'ps: -',
                             'load: OK +2 24x16',
                             'img: OK +0 24x16 7d9bfc4e,574f3dca',
                             'en: OK +0 24x16 c6aa44c0,3add3ad6',
                             'bi: STATE +0 24x16',
                             'vm: OK +0 24x16 d0:3f7fc867,690b37d3',
                             'ps: -',
                             'rw 0: OK +0 24x16',
                             'rh 0: OK +0 24x16',
                             'vm: OK +0 24x16 d0:3f7fc867,690b37d3',
                             'ps: -'],
 ('load_getters', 'single'): ['img: STATE +0 0x0',
                              'en: STATE +0 0x0',
                              'bi: STATE +0 0x0',
                              'vm: STATE +0 0x0',
                              'ps: STATE +0 0x0',
                              'load: OK +1 24x16',
                              'img: OK +0 24x16 7d9bfc4e',
                              'en: OK +0 24x16 c6aa44c0',
                              'bi: STATE +0 24x16',
                              'vm: STATE +0 24x16',
                              'ps: STATE +0 24x16',
                              'rw 0: OK +0 24x16',
                              'rh 0: OK +0 24x16',
                              'vm: STATE +0 24x16',
                              'ps: STATE +0 24x16'],
 ('params', 'batch'): ['load: OK +1 24x16',
                       'par4: OK +0 24x16',
                       'rw 2: OK +10 22x16 1a1c5295,bcc63558',
                       'img: OK +0 22x16 5821884c,958f5619',
                       'en: OK +0 22x16 3ba29277,5430a62f',
                       'par8: OK +0 22x16',
                       'tile: OK +0 22x16',
                       'rw 1: OK +5 21x16 9d693235,109c6499',
                       'img: OK +0 21x16 edde5e13,7bde899e',
                       'en: OK +0 21x16 8bd3b002,ea008b81',
                       'auto: OK +0 21x16',
                       'load: OK +1 24x16',
                       'ew 2: OK +15 26x16 1a1c5295,bcc63558',
                       'par4: OK +0 26x16',
                       'rw 1: STATE +0 26x16',
                       'en: OK +0 26x16 e3c8a6ab,7944525d',
                       'img: OK +0 26x16 5343ba8c,3fa56df3',
                       'par8: OK +0 26x16',
                       'load: OK +1 24x16',
                       'rh 1: OK +7 24x15 45cd0f61,f24c7d9c',
                       'tile: OK +0 24x15',
                       'rh 1: OK +5 24x14 36bbf2b7,f37a452b',
                       'en: OK +1 24x14 4179677b,8994e54b',
                       'auto: OK +0 24x14',
                       'rs 20 12: STATE +0 24x14',
                       'img: OK +1 24x14 62bbb264,9a9fdcb2'],
 ('params', 'single'): ['load: OK +1 24x16',
                        'par4: OK +1 24x16',
                        'rw 2: OK +10 22x16 fb5377ba',
                        'img: OK +0 22x16 e9849c73',
                        'en: OK +0 22x16 c2ad3ef0',
                        'par8: OK +1 22x16',
                        'tile: OK +0 22x16',
                        'rw 1: OK +5 21x16 9150c18e',
                        'img: OK +0 21x16 51dafcc7',
                        'en: OK +0 21x16 44da9ce4',
                        'auto: OK +0 21x16',
                        'load: OK +1 24x16',
                        'ew 2: OK +15 26x16 1a1c5295',
                        'par4: OK +1 26x16',
                        'rw 1: OK +5 25x16 6d614d46',
                        'en: OK +0 25x16 48172728',
                        'img: OK +0 25x16 46091c1a',
                        'par8: OK +1 25x16',
                        'load: OK +1 24x16',
                        'rh 1: OK +7 24x15 45cd0f61',
                        'tile: OK +0 24x15',
                        'rh 1: OK +5 24x14 36bbf2b7',
                        'en: OK +1 24x14 4179677b',
                        'auto: OK +0 24x14',
                        'rs 20 12: STATE +0 24x14',
                        'img: OK +1 24x14 62bbb264'],
 ('resize_then', 'batch'): ['dv1: -',
                            'load: OK +2 24x16',
                            'rsv 20 19: OK +48 20x19 feacde88',
                            'img: OK +1 20x19 6e6c26f2,471aa5d2',
                            'en: OK +1 20x19 b813b667,0f58ef94',
                            'vm: STATE +0 20x19',
                            'ps: -',
                            'bi: STATE +0 20x19',
                            'rw 0: STATE +0 20x19',
                            'rw 1: STATE +0 20x19',
                            'rh 0: STATE +0 20x19',
                            'rh 1: STATE +0 20x19',
                            'ew 0: STATE +0 20x19',
                            'ew 1: STATE +0 20x19',
                            'eh 0: STATE +0 20x19',
                            'eh 1: STATE +0 20x19',
                            'rs 20 19: STATE +0 20x19',
                            'rs 24 16: STATE +0 20x19',
                            'img: OK +1 20x19 6e6c26f2,471aa5d2',
                            'en: OK +1 20x19 b813b667,0f58ef94',
                            'load: OK +2 24x16',
                            'rs 24 16: OK +0 24x16 deab7e4e',
                            'rw 1: OK +6 23x16 8c9fcb8c,a500dcf4',
                            'img: OK +0 23x16 e495f868,3bd3d96c',
                            'load: OK +2 24x16',
                            'rsv 50 40: OK +315 50x40 1aa231ce',
                            'img: OK +1 50x40 4ce39652,9855ffde',
                            'en: OK +1 50x40 5cd1094e,6084b9b3',
                            'vm: STATE +0 50x40',
                            'load: OK +2 24x16',
                            'rs 30 12: OK +60 30x12 26b7e410',
                            'img: OK +1 30x12 3a58a581,e5bc8873',
                            'en: OK +1 30x12 04e98f84,b09d4c91',
                            'rw 0: STATE +0 30x12',
                            'vm: STATE +0 30x12'],
 ('resize_then', 'single'): ['dv1: OK +0 0x0',
                             'load: OK +1 24x16',
                             'rsv 20 19: OK +49 20x19 c54072df',
                             'img: OK +1 20x19 6e6c26f2',
                             'en: OK +1 20x19 b813b667',
                             'vm: STATE +0 20x19',
                             'ps: STATE +0 20x19',
                             'bi: STATE +0 20x19',
                             'rw 0: OK +0 20x19',
                             'rw 1: STATE +0 20x19',
                             'rh 0: OK +0 20x19',
                             'rh 1: STATE +0 20x19',
                             'ew 0: OK +0 20x19',
                             'ew 1: STATE +0 20x19',
                             'eh 0: OK +0 20x19',
                             'eh 1: STATE +0 20x19',
                             'rs 20 19: STATE +0 20x19',
                             'rs 24 16: STATE +0 20x19',
                             'img: OK +1 20x19 6e6c26f2',
                             'en: OK +1 20x19 b813b667',
                             'load: OK +1 24x16',
                             'rs 24 16: OK +0 24x16 1b43eabd',
                             'rw 1: OK +7 23x16 8c9fcb8c',
                             'img: OK +0 23x16 e495f868',
                             'load: OK +1 24x16',
                             'rsv 50 40: OK +316 50x40 af177859',
                             'img: OK +1 50x40 4ce39652',
                             'en: OK +1 50x40 5cd1094e',
                             'vm: STATE +0 50x40',
                             'load: OK +1 24x16',
                             'rs 30 12: OK +61 30x12 ebd2cfca',
                             'img: OK +1 30x12 3a58a581',
                             'en: OK +1 30x12 04e98f84',
                             'rw 0: OK +0 30x12',
                             'vm: STATE +0 30x12'],
 ('zero_one', 'batch'): ['dv1: -',
                         'load: OK +2 24x16',
                         'rw 0: OK +0 24x16',
                         'rh 0: OK +0 24x16',
                         'ew 0: OK +0 24x16',
                         'eh 0: OK +0 24x16',
                         'rw 1: OK +6 23x16 8c9fcb8c,a500dcf4',
                         'rh 0: OK +0 23x16',
                         'rh 1: STATE +0 23x16',
                         'eh 0: OK +0 23x16',
                         'eh 1: STATE +0 23x16',
                         'ew 0: OK +0 23x16',
                         'ew 1: STATE +0 23x16',
                         'vm: OK +0 23x16 d1:bcbcbab6,690b37d3',
                         'ps: -',
                         'img: OK +0 23x16 e495f868,3bd3d96c',
                         'en: OK +0 23x16 a5a654b9,870eef12',
                         'rw 1: OK +6 22x16 3fd06464,c463130d',
                         'vm: OK +0 22x16 d2:79093999,690b37d3',
                         'ps: -',
                         'load: OK +2 24x16',
                         'rh 1: OK +9 24x15 45cd0f61,f24c7d9c',
                         'rw 0: OK +0 24x15',
                         'rw 1: STATE +0 24x15',
                         'ew 0: OK +0 24x15',
                         'ew 1: STATE +0 24x15',
                         'vm: OK +1 24x15 d1:8aa5638e,690b37d3',
                         'ps: -',
                         'img: OK +1 24x15 b09f7a97,c0f2e186',
                         'en: OK +1 24x15 a77f8af7,4d043457'],
 ('zero_one', 'single'): ['dv1: OK +0 0x0',
                          'load: OK +1 24x16',
                          'rw 0: OK +0 24x16',
                          'rh 0: OK +0 24x16',
                          'ew 0: OK +0 24x16',
                          'eh 0: OK +0 24x16',
                          'rw 1: OK +7 23x16 8c9fcb8c',
                          'rh 0: OK +0 23x16',
                          'rh 1: STATE +0 23x16',
                          'eh 0: OK +0 23x16',
                          'eh 1: STATE +0 23x16',
                          'ew 0: OK +0 23x16',
                          'ew 1: STATE +0 23x16',
                          'vm: OK +0 23x16 d1:6c2ff098',
                          'ps: OK +1 23x16 42de5e05',
                          'img: OK +0 23x16 e495f868',
                          'en: OK +0 23x16 a5a654b9',
                          'rw 1: OK +6 22x16 3fd06464',
                          'vm: OK +0 22x16 d2:d04bb1c5',
                          'ps: OK +1 22x16 4a584464',
                          'load: OK +1 24x16',
                          'rh 1: OK +9 24x15 45cd0f61',
                          'rw 0: OK +0 24x15',
                          'rw 1: STATE +0 24x15',
                          'ew 0: OK +0 24x15',
                          'ew 1: STATE +0 24x15',
                          'vm: OK +1 24x15 d1:974e1280',
                          'ps: OK +2 24x15 290afbbe',
                          'img: OK +1 24x15 b09f7a97',
                          'en: OK +1 24x15 a77f8af7']}


@pytest.mark.parametrize("batched", [False, True], ids=["single", "batch"])
@pytest.mark.parametrize("name", list(SCENARIOS))
def test_session_rules(name, batched):
    got = record(name, batched)
    want = EXPECTED[(name, "batch" if batched else "single")]
    assert got == want, "\n".join("%s %-70s | %s" % ("  " if e == g else "!!", e, g) for e, g in zip(want, got))
