"""The oracle is pinned before it is trusted (CPU suite).

1. the plain-C restatement (oracle/blinky_oracle.c + oracle_lenses.c) against the
   committed golden vectors, which were produced by the compiled, unmodified
   reference (tests/golden/make_golden.py), for every transcribed globe x lens;
2. where oracle/_ref exists, the compiled reference against the committed vectors
   (they reproduce)."""
import json
import os

import numpy as np
import pytest

from conftest import sha
from oracle.pyoracle import TRANSCRIBED_GLOBES, TRANSCRIBED_LENSES

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = (128, 96, 48)


@pytest.fixture(scope="module")
def golden():
    lm = np.load(os.path.join(G, "lensmaps_small.npz"))
    meta = json.load(open(os.path.join(G, "meta_small.json")))
    return lm, meta


def transcribed_keys(meta):
    for key in sorted(meta):
        g, l = key.split("__")
        if g in TRANSCRIBED_GLOBES and l in TRANSCRIBED_LENSES:
            yield key, g, l


def test_restatement_reproduces_golden_lensmaps(restate, golden):
    lm, meta = golden
    W, H, PS = SMALL
    n = 0
    for key, g, l in transcribed_keys(meta):
        got = restate.build(g, l, W, H, PS)
        assert got["rc"] == 0
        assert got["scale"] == meta[key]["scale"], key
        assert got["display"] == meta[key]["display"], key
        assert np.array_equal(got["idx"], lm[key + "__idx"]), key
        assert np.array_equal(got["tint"], lm[key + "__tint"]), key
        assert sha(got["plates"]) == meta[key]["plates_sha"], key
        n += 1
    assert n >= 20


def test_restatement_palmaps_match_golden(restate):
    g = np.load(os.path.join(G, "palmaps.npz"))
    assert np.array_equal(restate.palmaps(g["palette"]), g["palmaps"])


def test_palmap_known_answers(restate):
    # a grey ramp palette: every tint LUT must map into the ramp, plate 0 (white tint)
    # brightens by (42*(255-c))>>8 and picks the first nearest grey
    pal = np.repeat(np.arange(256, dtype=np.uint8)[:, None], 3, axis=1).reshape(768)
    pm = restate.palmaps(pal)
    for c in (0, 1, 100, 200, 255):
        assert pm[0][c] == c + ((42 * (255 - c)) >> 8)
    # all-black palette: everything maps to index 0 (first minimum wins)
    assert not restate.palmaps(np.zeros(768, np.uint8)).any()


def test_restatement_render_matches_golden_frames(restate, bb, palette):
    frames = np.load(os.path.join(G, "frames_small.npz"))
    W, H, PS = SMALL
    pm = restate.palmaps(palette)
    checked = 0
    for key in frames.files:
        g, l, r = key.split("__")
        if g not in TRANSCRIBED_GLOBES or l not in TRANSCRIBED_LENSES:
            continue
        rubix = r == "rubix1"
        m = restate.build(g, l, W, H, PS)
        faces = bb.synthetic_faces(m["numplates"], PS, 0)
        bg = np.random.default_rng(3).integers(0, 256, (120, 160), dtype=np.uint8)
        out = restate.render(m["idx"], m["tint"], faces, pm, rubix, background=bg, vx=8, vy=6)
        assert np.array_equal(out, frames[key]), key
        # threaded baseline variant is the same function
        out_t = restate.render(m["idx"], m["tint"], faces, pm, rubix, background=bg, vx=8, vy=6, threads=3)
        assert np.array_equal(out_t, frames[key]), key
        checked += 1
    assert checked >= 5


def test_c1_golden(restate, bb, palette):
    """BASELINE config C1: 640x480, cube 6x256^2, panini f_fov 180, rubix off and on"""
    c1 = json.load(open(os.path.join(G, "c1.json")))
    arr = np.load(os.path.join(G, "c1.npz"))
    m = restate.build("cube", "panini", 640, 480, 256, zoom=("f_fov", 180))
    assert m["scale"] == c1["scale"] == 2 / 320  # closed form: x(90 deg) = 2 for d = 1
    assert np.array_equal(m["idx"], arr["idx"]) and np.array_equal(m["tint"], arr["tint"])
    assert sha(m["idx"]) == c1["idx_sha"] and sha(m["tint"]) == c1["tint_sha"]
    assert int((m["idx"] >= 0).sum()) == c1["mapped"] == 640 * 480  # panini maps every pixel
    faces = bb.synthetic_faces(6, 256, 0)
    bg = bb.synthetic_background(640, 480)
    assert sha(faces) == c1["faces_sha"] and sha(bg) == c1["bg_sha"]
    pm = restate.palmaps(palette)
    assert sha(restate.render(m["idx"], m["tint"], faces, pm, False, background=bg)) == c1["render_rubix_off_sha"]
    assert sha(restate.render(m["idx"], m["tint"], faces, pm, True, background=bg)) == c1["render_rubix_on_sha"]


def test_quirks_pinned(restate):
    W, H, PS = 128, 96, 64
    # 1. centre-pixel hole: r = 0 -> x/r = NaN -> unmapped (stereographic, rectilinear, fisheye1/2)
    for lens in ("stereographic", "rectilinear", "fisheye1", "fisheye2"):
        m = restate.build("cube", lens, W, H, PS)
        assert m["idx"][H // 2, W // 2] == -1, lens
        assert m["idx"][H // 2, W // 2 + 1] >= 0
    # panini has no hole
    assert restate.build("cube", "panini", W, H, PS)["idx"][H // 2, W // 2] >= 0
    # 3./5. plates never looked at keep display = 0 (panini at 180 deg never sees the back plate)
    assert restate.build("cube", "panini", W, H, PS)["display"] == [1, 1, 1, 0, 1, 1]
    # mapped fractions from geometry
    f1 = (restate.build("cube", "fisheye1", 192, 108, 64)["idx"] >= 0).mean()
    assert abs(f1 - np.pi / 4 * 108 / 192) < 0.01  # inscribed disc
    eq = (restate.build("cube", "equirect", 192, 108, 64)["idx"] >= 0).mean()
    assert abs(eq - (192 / 2) / 108) < 0.02  # 2:1 strip inside 16:9


def test_tint_is_plate_inside_cells_only(restate):
    m = restate.build("cube", "panini", 128, 96, 48)
    idx, tint = m["idx"], m["tint"]
    plate = idx // (48 * 48)
    inside = tint != 255
    assert inside.any() and (~inside).any()
    assert np.array_equal(tint[inside], plate[inside].astype(np.uint8))


# ---- against the compiled reference ------------------------------------------

def test_restatement_vs_compiled_reference(restate):
    W, H, PS = 200, 150, 100
    want = json.load(open(os.path.join(G, "reference_live.json")))["combos_200x150x100"]
    for g in TRANSCRIBED_GLOBES:
        for l in TRANSCRIBED_LENSES:
            r = want[f"{g}__{l}"]
            assert r["rc"] == 0
            m = restate.build(g, l, W, H, PS)
            assert m["scale"] == r["scale"], (g, l)
            assert sha(m["idx"]) == r["idx_sha"], (g, l)
            assert sha(m["tint"]) == r["tint_sha"], (g, l)
            assert m["display"] == r["display"], (g, l)
            assert sha(m["plates"]) == r["plates_sha"], (g, l)


def test_compiled_reference_reproduces_golden(ref, golden):
    lm, meta = golden
    W, H, PS = SMALL
    ref.set_screen(W, H)
    for key in list(sorted(meta))[::4]:
        g, l = key.split("__")
        ref.clear_log()
        ref.command(f"f_globe {g}")
        ref.command(f"f_lens {l}")
        ref.build(W, H, PS)
        idx, tint = ref.lensmap()
        assert np.array_equal(idx, lm[key + "__idx"]) and np.array_equal(tint, lm[key + "__tint"]), key
        assert ref.scale == meta[key]["scale"] and ref.log == meta[key]["log"]


def test_transcribed_lenses_equal_the_scripts_per_call(restate, host):
    """per-call pin of the Lua evaluator: raw lens_inverse/lens_forward results of the script
    (product evaluator) == the C transcription, bit for bit"""
    rng = np.random.default_rng(11)
    host.command("f_globe cube")
    for l in TRANSCRIBED_LENSES:
        host.command(f"f_lens {l}")
        for _ in range(300):
            x, y = rng.uniform(-3.2, 3.2), rng.uniform(-1.7, 1.7)
            try:
                st_c, ray_c = restate.lens_inverse(l, x, y)
            except KeyError:
                break
            st_p, ray_p = host.lens_inverse(x, y)
            assert st_c == st_p, (l, x, y)
            if st_c == 1:
                assert np.array_equal(np.array(ray_c).view(np.uint64), np.array(ray_p).view(np.uint64)), (l, x, y)
        for _ in range(300):
            v = rng.normal(size=3)
            v = (v / np.linalg.norm(v)).astype(np.float32).astype(np.float64)
            try:
                st_c, xy_c = restate.lens_forward(l, *v)
            except KeyError:
                break
            st_p, xy_p = host.lens_forward(*v)
            assert st_c == st_p
            if st_c == 1:
                assert np.array_equal(np.array(xy_c).view(np.uint64), np.array(xy_p).view(np.uint64)), (l, v)


def test_fastmath_drift(ref):
    """The reference ships with -ffast-math (engine/Makefile:270-277); the oracle is the same source without it.
    scripts/fastmath_drift.py builds every lens with both compiled references and counts differing lensmap entries
    (committed numbers: profiles/r2_fastmath_drift.txt).  Here: the machinery works and the drift stays what the
    report says — a handful of pixels landing on the neighbouring texel, never a mapped<->unmapped flip."""
    import io
    import sys

    from oracle.pyoracle import RefOracle

    if not RefOracle.available(fastmath=True):
        pytest.skip("oracle/_ref/libblinky_ref_fastmath.so not built")
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import fastmath_drift

    rows = fastmath_drift.drift(lenses=["panini", "stereographic", "equirect", "quincuncial"], size=(320, 200, 128), out=io.StringIO(), exact=ref)
    for lens, ndiff, flips, dx, dy in rows:
        assert ndiff <= 0.01 * 320 * 200 and flips == 0 and dx <= 1 and dy <= 1, (lens, ndiff, flips, dx, dy)
    assert os.path.exists(os.path.join(ROOT, "profiles", "r2_fastmath_drift.txt"))
