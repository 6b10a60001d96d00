"""TEST INFRASTRUCTURE — ctypes bindings of the parity oracles.  Not part of the product.

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline / --impl reference
legs import this module; nothing under blinky_b200/ does.

* :class:`RefOracle`   — oracle/_ref/libblinky_ref.so: the UNMODIFIED reference
  engine/NQ/fisheye.c compiled headless (needs a prebuilt .so; building it needs
  /root/reference).  One per process (the reference keeps its state in statics).
* :class:`Restatement` — oracle/liboracle.so: the plain-C restatement
  (blinky_oracle.c) + C transcriptions of shipped lenses/globes (oracle_lenses.c).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_void_p

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(HERE, "_ref", "libblinky_ref.so")
REF_FAST_SO = os.path.join(HERE, "_ref", "libblinky_ref_fastmath.so")
RESTATE_SO = os.path.join(HERE, "liboracle.so")
REFERENCE_GAME_DIR = "/root/reference/game"

ZOOM = {"f_fov": 1, "f_vfov": 2, "f_cover": 3, "f_contain": 4}


def _p(a):
    return a.ctypes.data_as(c_void_p)


_short_dirs = {}


def _short_basedir(basedir: str) -> str:
    """The reference formats "<basedir>/lua-scripts/lenses/<name>.lua" into a char[100] with sprintf
    (engine/NQ/fisheye.c:1665-1666, 1758-1759): from a checkout a few directories deep the longer lens
    names overflow it and the process aborts.  It gets the directory through a short symlink instead."""
    if basedir not in _short_dirs:
        import atexit
        import shutil
        import tempfile

        d = tempfile.mkdtemp(prefix="bref")
        atexit.register(shutil.rmtree, d, True)
        os.symlink(os.path.abspath(basedir), os.path.join(d, "s"))
        _short_dirs[basedir] = os.path.join(d, "s")
    return _short_dirs[basedir]


# ---------------------------------------------------------------------------
# the compiled reference
# ---------------------------------------------------------------------------
class RefOracle:
    _instance = None

    @staticmethod
    def available(fastmath: bool = False) -> bool:
        return os.path.exists(REF_FAST_SO if fastmath else REF_SO)

    @classmethod
    def get(cls, basedir: str, palette: np.ndarray) -> "RefOracle":
        """process-wide singleton (F_Init can only run once per loaded library)"""
        if cls._instance is None:
            cls._instance = cls(basedir, palette)
        else:
            cls._instance.set_basedir(basedir)
        return cls._instance

    def __init__(self, basedir: str, palette: np.ndarray, fastmath: bool = False):
        self.lib = L = ctypes.CDLL(REF_FAST_SO if fastmath else REF_SO)
        L.ref_log.restype = c_char_p
        L.ref_unhandled_commands.restype = c_char_p
        for f in ("ref_scale", "ref_lens_width", "ref_lens_height", "ref_plate_fov"):
            getattr(L, f).restype = c_double
        L.ref_time_render.restype = c_double
        L.ref_time_render.argtypes = [c_int, POINTER(c_double)]
        L.ref_lens_inverse.argtypes = [c_double, c_double, c_void_p]
        L.ref_lens_forward.argtypes = [c_void_p, POINTER(c_double), POINTER(c_double)]
        self.palette = np.ascontiguousarray(palette, np.uint8).reshape(768)
        rc = L.ref_init(_short_basedir(basedir).encode(), _p(self.palette))
        if rc != 0:
            raise RuntimeError("ref_init failed (already initialised in this process?)")
        self.W = self.H = 0

    def set_basedir(self, basedir: str):
        self.lib.ref_set_basedir(_short_basedir(basedir).encode())

    def command(self, text: str):
        self.lib.ref_command(text.encode())

    @property
    def log(self) -> str:
        return self.lib.ref_log().decode(errors="replace")

    def clear_log(self):
        self.lib.ref_log_clear()

    def set_screen(self, w, h, rowbytes=None, vx=0, vy=0, vw=None, vh=None):
        rowbytes = rowbytes or w
        vw = vw if vw is not None else w
        vh = vh if vh is not None else h
        self.lib.ref_set_screen(w, h, rowbytes, vx, vy, vw, vh)
        self.scr = (w, h, rowbytes, vx, vy, vw, vh)

    def build(self, w, h, ps) -> int:
        self.W, self.H, self.ps = w, h, ps
        return self.lib.ref_build(w, h, ps)

    def lensmap(self):
        idx = np.zeros((self.H, self.W), np.int32)
        tint = np.zeros((self.H, self.W), np.uint8)
        self.lib.ref_get_lensmap(_p(idx), _p(tint))
        return idx, tint

    def palmaps(self):
        out = np.zeros((6, 256), np.uint8)
        self.lib.ref_get_palmaps(_p(out))
        return out

    def display(self):
        d = (c_int * 6)()
        self.lib.ref_get_display(d)
        return list(d)

    def plates(self):
        n = self.lib.ref_numplates()
        out = np.zeros((6, 11), np.float32)
        self.lib.ref_get_plates(_p(out))
        return out[:n]

    scale = property(lambda s: s.lib.ref_scale())
    numplates = property(lambda s: s.lib.ref_numplates())
    map_type = property(lambda s: s.lib.ref_map_type())
    rubix_enabled = property(lambda s: bool(s.lib.ref_rubix_enabled()))

    def render(self, faces: np.ndarray, background: np.ndarray | None = None) -> np.ndarray:
        """render_lensmap() over `faces` ([P][ps][ps]) on top of `background` ([h][rowbytes])"""
        w, h, rowbytes = self.scr[0], self.scr[1], self.scr[2]
        out = np.zeros((h, rowbytes), np.uint8)
        faces = np.ascontiguousarray(faces, np.uint8)
        bg = None if background is None else np.ascontiguousarray(background, np.uint8)
        if bg is None:
            bg = np.zeros((h, rowbytes), np.uint8)
        self.lib.ref_render(_p(faces), int(faces.shape[0]), _p(bg), _p(out))
        return out

    def frame(self, faces: np.ndarray, background: np.ndarray) -> tuple[np.ndarray, int]:
        """one full engine frame through the real F_RenderView (platesize = min(w,h))"""
        w, h, rowbytes = self.scr[0], self.scr[1], self.scr[2]
        out = np.zeros((h, rowbytes), np.uint8)
        faces = np.ascontiguousarray(faces, np.uint8)
        bg = np.ascontiguousarray(background, np.uint8)
        n = self.lib.ref_frame(_p(faces), _p(bg), _p(out))
        return out, n

    def time_render(self, reps: int) -> tuple[float, float]:
        total = c_double()
        best = self.lib.ref_time_render(reps, ctypes.byref(total))
        return best, total.value

    def write_config(self, path: str) -> str:
        self.lib.ref_write_config(path.encode())
        return open(path).read()

    def lens_inverse(self, x, y):
        ray = np.zeros(3, np.float32)
        st = self.lib.ref_lens_inverse(x, y, _p(ray))
        return st, ray


# ---------------------------------------------------------------------------
# the plain-C restatement
# ---------------------------------------------------------------------------
class _Plate(ctypes.Structure):
    _fields_ = [("forward", c_float * 3), ("right", c_float * 3), ("up", c_float * 3), ("fov", c_float),
                ("dist", c_float), ("display", c_int)]


class _Globe(ctypes.Structure):
    _fields_ = [("numplates", c_int), ("platesize", c_int), ("plates", _Plate * 6), ("plate_fn", c_void_p),
                ("plate_ud", c_void_p)]


class _Rubix(ctypes.Structure):
    _fields_ = [("numcells", c_int), ("cell_size", c_double), ("pad_size", c_double)]


class _LensMap(ctypes.Structure):
    _fields_ = [("w", c_int), ("h", c_int), ("scale", c_double), ("idx", c_void_p), ("tint", c_void_p)]


class _LensDef(ctypes.Structure):
    _fields_ = [("name", c_char_p), ("inverse", c_void_p), ("forward", c_void_p), ("max_fov", c_int),
                ("max_vfov", c_int), ("lens_width", c_double), ("lens_height", c_double), ("onload", c_char_p)]


INVERSE_CB = ctypes.CFUNCTYPE(c_int, c_double, c_double, POINTER(c_double), c_void_p)
FORWARD_CB = ctypes.CFUNCTYPE(c_int, c_double, c_double, c_double, POINTER(c_double), POINTER(c_double), c_void_p)

TRANSCRIBED_LENSES = ["panini", "stereographic", "rectilinear", "equirect", "cylinder", "mercator", "hammer",
                      "fisheye1", "fisheye2", "quincuncial", "sinusoidal", "winkel1", "mollweide", "vandergrinten", "cube",
                      "winkeltripel", "eckert4", "miller", "gallstereo", "fahey", "eckert1", "eckert5", "kavrayskiy7", "winkel2",
                      "wagner6", "larrivee", "gins8", "polyconic", "gumby", "cubestereo", "debug"]
TRANSCRIBED_GLOBES = ["cube", "trism", "tetra", "cube_edge", "cube_corner", "fast"]


class Restatement:
    @staticmethod
    def available() -> bool:
        return os.path.exists(RESTATE_SO)

    def __init__(self):
        self.lib = L = ctypes.CDLL(RESTATE_SO)
        L.orc_calc_zoom.argtypes = [c_int, c_int, c_int, c_int, c_double, c_double, c_int, c_int, c_void_p, c_void_p,
                                    POINTER(c_double)]
        L.orc_render_lensmap.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int]
        L.orc_render_lensmap_omp.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int]

    def time_render(self, idx, tint, faces, palmaps, rubix: bool, threads: int, reps: int):
        """(best seconds, total seconds) of `reps` calls of the restated render_lensmap"""
        h, w = idx.shape
        idx = np.ascontiguousarray(idx, np.int32)
        tint = np.ascontiguousarray(tint, np.uint8)
        faces = np.ascontiguousarray(faces, np.uint8)
        palmaps = np.ascontiguousarray(palmaps, np.uint8)
        out = np.zeros((h, w), np.uint8)
        LM = _LensMap(w, h, 0.0, idx.ctypes.data, tint.ctypes.data)
        total = c_double()
        self.lib.orc_time_render.restype = c_double
        self.lib.orc_time_render.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, POINTER(c_double)]
        best = self.lib.orc_time_render(ctypes.byref(LM), _p(faces), _p(palmaps), int(rubix), _p(out), w, threads, reps,
                                        ctypes.byref(total))
        return best, total.value

    def max_threads(self) -> int:
        return self.lib.orc_max_threads()

    def lens_inverse(self, lens: str, x: float, y: float):
        """raw result of the C transcription of <lens>.lua's lens_inverse: (status, (rx, ry, rz))"""
        D = _LensDef()
        if lens == "debug" or not self.lib.orc_find_lens(lens.encode(), ctypes.byref(D)) or not D.inverse:
            raise KeyError(lens)   # (debug needs a globe: only through build())
        fn = INVERSE_CB(D.inverse)
        out = (c_double * 3)()
        st = fn(x, y, out, None)
        return st, (out[0], out[1], out[2])

    def lens_forward(self, lens: str, rx: float, ry: float, rz: float):
        D = _LensDef()
        if not self.lib.orc_find_lens(lens.encode(), ctypes.byref(D)) or not D.forward:
            raise KeyError(lens)
        fn = FORWARD_CB(D.forward)
        x, y = c_double(), c_double()
        st = fn(rx, ry, rz, ctypes.byref(x), ctypes.byref(y), None)
        return st, (x.value, y.value)

    def palmaps(self, palette: np.ndarray) -> np.ndarray:
        pal = np.ascontiguousarray(palette, np.uint8).reshape(768)
        out = np.zeros((6, 256), np.uint8)
        self.lib.orc_create_palmap(_p(pal), _p(out))
        return out

    def build(self, globe: str, lens: str, w: int, h: int, ps: int, zoom: tuple[str, int] | None = None,
              rubixgrid=(10, 4.0, 1.0), inverse_cb=None):
        """lensmap from the C transcriptions; returns dict(idx, tint, scale, display, plates)"""
        L = self.lib
        G = _Globe()
        G.platesize = ps
        if not L.orc_load_globe(globe.encode(), ctypes.byref(G)):
            raise KeyError(globe)
        D = _LensDef()
        if not L.orc_find_lens(lens.encode(), ctypes.byref(D)):
            raise KeyError(lens)
        ud = None
        if lens == "debug":   # sizes itself from numplates, calls plate_to_ray
            L.orc_debug_lens(G.numplates, ctypes.byref(D))
            ud = ctypes.byref(G)
        if zoom is None:
            parts = D.onload.decode().split()
            zoom = (parts[0], int(parts[1]) if len(parts) > 1 else 0)
        scale = c_double()
        ok = L.orc_calc_zoom(ZOOM[zoom[0]], zoom[1], D.max_fov, D.max_vfov, D.lens_width, D.lens_height, w, h,
                             D.forward, None, ctypes.byref(scale))
        if not ok:
            raise ValueError("calc_zoom failed")
        idx = np.zeros((h, w), np.int32)
        tint = np.zeros((h, w), np.uint8)
        LM = _LensMap(w, h, scale.value, idx.ctypes.data, tint.ctypes.data)
        rb = _Rubix(int(rubixgrid[0]), float(rubixgrid[1]), float(rubixgrid[2]))
        if inverse_cb is not None:
            rc = L.orc_build_inverse(ctypes.byref(G), ctypes.byref(rb), ctypes.byref(LM), inverse_cb, None)
        elif D.inverse:
            rc = L.orc_build_inverse(ctypes.byref(G), ctypes.byref(rb), ctypes.byref(LM), c_void_p(D.inverse), ud)
        else:
            rc = L.orc_build_forward(ctypes.byref(G), ctypes.byref(rb), ctypes.byref(LM), c_void_p(D.forward), None)
        plates = np.array([list(G.plates[i].forward) + list(G.plates[i].right) + list(G.plates[i].up) +
                           [G.plates[i].fov, G.plates[i].dist] for i in range(G.numplates)], np.float32)
        return dict(rc=rc, idx=idx, tint=tint, scale=scale.value, numplates=G.numplates,
                    display=[G.plates[i].display for i in range(6)], plates=plates)

    def render(self, idx: np.ndarray, tint: np.ndarray, faces: np.ndarray, palmaps: np.ndarray, rubix: bool,
               background: np.ndarray | None = None, rowbytes: int | None = None, vx: int = 0, vy: int = 0,
               threads: int = 0) -> np.ndarray:
        """render_lensmap restated: writes only mapped pixels over `background`"""
        h, w = idx.shape
        idx = np.ascontiguousarray(idx, np.int32)
        tint = np.ascontiguousarray(tint, np.uint8)
        faces = np.ascontiguousarray(faces, np.uint8)
        palmaps = np.ascontiguousarray(palmaps, np.uint8)
        if background is None:
            rowbytes = rowbytes or w
            out = np.zeros((h + vy, rowbytes), np.uint8)
        else:
            out = np.array(background, np.uint8, copy=True, order="C")
            rowbytes = out.shape[1]
        LM = _LensMap(w, h, 0.0, idx.ctypes.data, tint.ctypes.data)
        if threads and threads > 1:
            self.lib.orc_render_lensmap_omp(ctypes.byref(LM), _p(faces), _p(palmaps), int(rubix), _p(out), rowbytes, vx,
                                            vy, threads)
        else:
            self.lib.orc_render_lensmap(ctypes.byref(LM), _p(faces), _p(palmaps), int(rubix), _p(out), rowbytes, vx, vy)
        return out
