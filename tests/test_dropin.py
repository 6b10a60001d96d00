"""The C drop-in (blinky_b200/host/fisheye_b200.c): same engine seam as the reference's
fisheye.c.  It is compiled against the reference engine's own headers with the same
headless engine stubs as the compiled reference (oracle/Makefile -> oracle/_ref/
libdropin_b200.so), then driven with the command sequence the compiled reference was driven
with (tests/golden/make_golden.py): console text, config text and whole F_RenderView frames
must be identical."""
import ctypes
import json
import os

import numpy as np
import pytest

from conftest import sha

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "oracle", "_ref", "libdropin_b200.so")

needs_so = pytest.mark.skipif(not os.path.exists(SO), reason="oracle/_ref/libdropin_b200.so not built (needs the reference engine's headers)")


@pytest.fixture(scope="module")
def want():
    """the compiled reference's console text, frames and config for the sequences below"""
    return json.load(open(os.path.join(ROOT, "tests", "golden", "reference_live.json")))["dropin"]


@pytest.fixture()
def dropin(bb, palette, cuda_device):
    """the drop-in after F_Init, shut down again even when the test fails"""
    D = ctypes.CDLL(SO)
    D.dropin_log.restype = ctypes.c_char_p
    D.dropin_plate_fov.restype = ctypes.c_double
    assert D.dropin_init(bb.SCRIPT_DIR.encode(), palette.ctypes.data_as(ctypes.c_void_p)) == 0
    yield D
    D.dropin_shutdown()


@needs_so
def test_dropin_exports_the_engine_seam(bb):
    lib = ctypes.CDLL(SO)
    for sym in ("F_Init", "F_Shutdown", "F_RenderView", "F_WriteConfig", "fisheye_enabled", "fisheye_plate_fov"):
        assert hasattr(lib, sym), sym


@needs_so
def test_dropin_fails_loudly_without_a_gpu(bb, palette):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = ctypes.CDLL(SO)
    lib.dropin_log.restype = ctypes.c_char_p
    rc = lib.dropin_init(bb.SCRIPT_DIR.encode(), palette.ctypes.data_as(ctypes.c_void_p))
    assert rc == -2
    assert b"fisheye_b200:" in lib.dropin_log() and not lib.dropin_fisheye_enabled()


@needs_so
@pytest.mark.gpu
def test_dropin_matches_compiled_reference(bb, want, dropin, tmp_path):
    D = dropin
    assert D.dropin_fisheye_enabled() == 1

    for c in ("fisheye 1", "f_globe cube", "f_lens panini", "f_fov 180", "f_rubixgrid 10 4 1"):
        D.dropin_command(c.encode())
    D.dropin_log_clear()
    D.dropin_recalc_refdef()  # clear what F_Init's own "fisheye 1" set
    for c in ("f_help", "f_fov", "f_lens hammer", "f_lens", "f_globe trism", "f_globe", "f_rubix", "f_rubix", "f_vfov 70", "f_cover",
              "f_rubixgrid", "fisheye", "f_lens panini", "f_globe cube"):
        D.dropin_command(c.encode())
    assert want["log"] == D.dropin_log().decode()
    assert D.dropin_recalc_refdef() == 0  # only `fisheye <n>` touches it
    D.dropin_command(b"fisheye 1")
    assert D.dropin_recalc_refdef() == 1

    # whole frames through F_RenderView, view rectangle inside a wider screen (the reference started with rubix off)
    rubix_on = False
    for (g, l, rubix, scr) in [("cube", "panini", False, (96, 64, 96, 0, 0, 96, 64)), ("cube", "fisheye1", True, (128, 80, 136, 16, 8, 96, 64)),
                               ("trism", "equirect", True, (96, 64, 96, 0, 0, 96, 64)), ("tetra", "winkel1", False, (104, 72, 104, 8, 8, 88, 56))]:
        D.dropin_command(f"f_globe {g}".encode())
        D.dropin_command(f"f_lens {l}".encode())
        if rubix_on != rubix:
            D.dropin_command(b"f_rubix")
            rubix_on = rubix
        w, h, rowbytes, vx, vy, vw, vh = scr
        D.dropin_set_screen(w, h, rowbytes, vx, vy, vw, vh)
        ps = min(vw, vh)
        faces = bb.synthetic_faces({"cube": 6, "trism": 5, "tetra": 4}[g], ps, 4)
        bg = np.random.default_rng(3).integers(0, 256, (h, w), dtype=np.uint8)
        got = np.zeros((h, rowbytes), np.uint8)
        n2 = D.dropin_frame(faces.ctypes.data_as(ctypes.c_void_p), bg.ctypes.data_as(ctypes.c_void_p), got.ctypes.data_as(ctypes.c_void_p))
        assert n2 == want["frames"][f"{g}__{l}"]["calls"], (g, l)  # same plates rendered (display flags)
        assert sha(got) == want["frames"][f"{g}__{l}"]["sha"], (g, l)
        # a second frame without changes: no rebuild, same bytes
        got2 = np.zeros((h, rowbytes), np.uint8)
        D.dropin_frame(faces.ctypes.data_as(ctypes.c_void_p), bg.ctypes.data_as(ctypes.c_void_p), got2.ctypes.data_as(ctypes.c_void_p))
        assert np.array_equal(got2, got)
    if rubix_on:
        D.dropin_command(b"f_rubix")
    cfg = tmp_path / "dropin_cfg.txt"
    D.dropin_write_config(str(cfg).encode())
    assert open(cfg).read() == want["config"]


@needs_so
@pytest.mark.gpu
def test_dropin_rebuild_never_holds_a_frame_up(bb, want, dropin):
    """The reference's lens builder is time-sliced so that no frame waits for it (engine/NQ/fisheye.c:744-746,
    819-826).  The drop-in builds on a worker thread in a second context: across an f_lens change every
    F_RenderView call must return within a frame time, frames shown meanwhile are the PREVIOUS lens's,
    and the frame after the swap is the reference's frame for the new lens."""
    import time

    D = dropin
    w, h = 640, 480
    ps = min(w, h)

    for c in ("fisheye 1", "f_globe cube", "f_lens panini", "f_fov 180"):
        D.dropin_command(c.encode())
    D.dropin_set_screen(w, h, w, 0, 0, w, h)
    faces = bb.synthetic_faces(6, ps, 9)
    bg = np.random.default_rng(5).integers(0, 256, (h, w), dtype=np.uint8)
    fp, bp = faces.ctypes.data_as(ctypes.c_void_p), bg.ctypes.data_as(ctypes.c_void_p)
    old = np.zeros((h, w), np.uint8)
    D.dropin_frame(fp, bp, old.ctypes.data_as(ctypes.c_void_p))          # panini, built and shown
    assert sha(old) == want["rebuild_old_sha"]

    D.dropin_command(b"f_lens winkeltripel")   # an expensive lens: NVRTC + thousands of interpreter re-evaluations
    D.dropin_command(b"f_contain")
    times, during = [], []
    got = np.zeros((h, w), np.uint8)
    for it in range(100000):
        t0 = time.perf_counter()
        D.dropin_frame_nowait(fp, bp, got.ctypes.data_as(ctypes.c_void_p))
        times.append(time.perf_counter() - t0)
        if not D.dropin_building():
            break
        during.append(got.copy())
    assert len(times) >= 2, "the rebuild finished inside the first F_RenderView call: it was not asynchronous"
    assert max(times) < 1 / 60 + 0.010, f"a frame waited {max(times) * 1e3:.1f} ms for the lens build"
    assert all(np.array_equal(f, old) for f in during[:50]), "frames during the build must show the previous lensmap"
    D.dropin_frame_nowait(fp, bp, got.ctypes.data_as(ctypes.c_void_p))     # first frame after the swap
    assert sha(got) == want["rebuild_new_sha"]
