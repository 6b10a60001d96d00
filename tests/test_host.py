"""Host logic of the product (CPU suite): scripts, console surface, zoom, palette and the
lensmap build of libblinky_b200.so, through the C ABI, against the golden vectors the compiled
reference produced (tests/golden/make_golden.py)."""
import json
import os

import numpy as np
import pytest

from conftest import ALL_GLOBES, ALL_LENSES, sha

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SMALL = (128, 96, 48)


@pytest.fixture(scope="module")
def live():
    """the compiled reference's side of the comparisons below"""
    return json.load(open(os.path.join(G, "reference_live.json")))


def build(fe, globe, lens, w, h, ps, threads=1, extra=()):
    fe.clear_log()
    fe.command(f"f_globe {globe}")
    fe.command(f"f_lens {lens}")
    for c in extra:
        fe.command(c)
    try:
        fe.build_lensmap(w, h, ps, threads)
        rc = 0
    except Exception as e:  # noqa: BLE001
        rc = e.code
    return rc


def test_lensmaps_match_golden(host):
    lm = np.load(os.path.join(G, "lensmaps_small.npz"))
    meta = json.load(open(os.path.join(G, "meta_small.json")))
    W, H, PS = SMALL
    assert len(meta) >= 50
    for key in sorted(meta):
        g, l = key.split("__")
        rc = build(host, g, l, W, H, PS)
        assert rc == 0 if meta[key]["rc"] == 0 else rc != 0, key
        idx, tint = host.lensmap()
        assert np.array_equal(idx, lm[key + "__idx"]), key
        assert np.array_equal(tint, lm[key + "__tint"]), key
        assert host.scale == meta[key]["scale"], key
        assert host.display() == meta[key]["display"], key
        assert host.numplates == meta[key]["numplates"] and host.map_type == meta[key]["map_type"]
        assert sha(host.plates()) == meta[key]["plates_sha"], key
        assert host.log == meta[key]["log"], key


def test_palmaps_match_golden(host):
    g = np.load(os.path.join(G, "palmaps.npz"))
    host.set_palette(g["palette"])
    assert np.array_equal(host.palmaps(), g["palmaps"])


def test_c1_lensmap_matches_golden(host):
    c1 = json.load(open(os.path.join(G, "c1.json")))
    arr = np.load(os.path.join(G, "c1.npz"))
    assert build(host, "cube", "panini", 640, 480, 256, threads=4, extra=["f_fov 180"]) == 0
    idx, tint = host.lensmap()
    assert np.array_equal(idx, arr["idx"]) and np.array_equal(tint, arr["tint"])
    assert host.scale == c1["scale"] and host.display() == c1["display"]
    assert host.mapped_pixels == c1["mapped"]


def test_packed_lensmap_encodes_idx_and_tint(bb, host):
    for g, l in [("cube", "panini"), ("cube", "hammer"), ("trism", "winkel1")]:
        assert build(host, g, l, 96, 72, 40) == 0
        idx, tint = host.lensmap()
        p = host.lensmap_packed()
        valid = (p & bb.LM_VALID) != 0
        assert np.array_equal(valid, idx >= 0)
        assert np.array_equal((p & bb.LM_INDEX_MASK)[valid].astype(np.int32), idx[valid])
        t = ((p >> bb.LM_TINT_SHIFT) & 7).astype(np.uint8)
        assert np.array_equal(t[valid] == bb.LM_TINT_NONE, tint[valid] == 255)
        assert np.array_equal(t[valid][tint[valid] != 255], tint[valid][tint[valid] != 255])
        assert host.mapped_pixels == int(valid.sum())


def test_threaded_build_equals_sequential(bb, palette):
    with bb.Fisheye(device=None, palette=palette) as a, bb.Fisheye(device=None, palette=palette) as b:
        for g, l in [("cube", "quincuncial"), ("fast", "panini"), ("cube", "eckert4"), ("tetra", "debug"),
                     ("cube", "winkeltripel"), ("cube", "sinusoidal"), ("cube", "mollweide")]:
            assert build(a, g, l, 120, 90, 50, threads=1) == 0
            assert build(b, g, l, 120, 90, 50, threads=5) == 0
            ia, ta = a.lensmap()
            ib, tb = b.lensmap()
            assert np.array_equal(ia, ib) and np.array_equal(ta, tb), (g, l)
            assert a.display() == b.display() and a.scale == b.scale


def test_all_combinations_against_compiled_reference(host, live):
    W, H, PS = 96, 64, 40
    want = live["combos_96x64x40"]
    for g in ALL_GLOBES:
        for l in ALL_LENSES:
            r = want[f"{g}__{l}"]
            build(host, g, l, W, H, PS)
            idx, tint = host.lensmap()
            assert sha(idx) == r["idx_sha"] and sha(tint) == r["tint_sha"], (g, l)
            assert r["display"] == host.display() and r["scale"] == host.scale, (g, l)
            assert r["log"] == host.log, (g, l)
            assert sha(host.plates()) == r["plates_sha"], (g, l)


def test_own_scripts_equal_reference_scripts(bb, live, palette):
    """the repo's script set must drive the lensmap exactly like the reference's scripts do"""
    want = live["reference_scripts_112x80x56"]
    with bb.Fisheye(device=None, palette=palette) as b:
        for g in ALL_GLOBES:
            for l in ALL_LENSES:
                r = want[f"{g}__{l}"]
                rb = build(b, g, l, 112, 80, 56, threads=4)
                ib, tb = b.lensmap()
                assert r["rc"] == rb and r["idx_sha"] == sha(ib) and r["tint_sha"] == sha(tb), (g, l)
                assert r["scale"] == b.scale and r["display"] == b.display() and r["log"] == b.log, (g, l)
                assert (r["onload"], r["max_fov"], r["max_vfov"], r["lens_width"], r["lens_height"], r["map_type"]) == \
                       (b.onload, b.max_fov, b.max_vfov, b.lens_width, b.lens_height, b.map_type), (g, l)


def test_console_surface_against_compiled_reference(host, live):
    script = ["fisheye 1", "f_rubixgrid 10 4 1", "fisheye", "fisheye 0", "fisheye 1", "f_help", "f_rubix", "f_rubix", "f_rubixgrid", "f_rubixgrid 7 3.5 0.25",
              "f_rubixgrid", "f_fov", "f_fov 100", "f_fov", "f_vfov 60", "f_vfov", "f_cover", "f_fov", "f_contain",
              "f_fov", "f_lens", "f_globe", "f_lens hammer", "f_lens", "f_globe trism", "f_globe", "f_lens nosuchlens",
              "f_globe nosuchglobe", "f_lens panini", "f_globe cube", "f_rubixgrid 10 4 1", "F_FOV 90"]
    for c in ("fisheye 1", "f_globe cube", "f_lens panini", "f_fov 180", "f_rubixgrid 10 4 1"):  # same starting state
        host.command(c)
    if host.rubix_enabled:  # the reference's run started with rubix off
        host.command("f_rubix")
    host.clear_log()
    for c in script:
        host.command(c)
    # the only difference allowed: the file-open error text of luaL_loadfile vs ours (the stored log has none)
    assert live["console"]["log"] == "\n".join(x for x in host.log.split("\n") if not x.startswith("ERROR:"))
    assert live["console"]["config"] == host.write_config()
    assert host.zoom_type == 1 and host.zoom_fov == 90


def test_write_config_matches_golden(host):
    for c in ["fisheye 1", "f_globe cube", "f_lens panini", "f_lens hammer", "f_globe trism", "f_fov 123", "f_rubixgrid 7 3.5 0.25"]:
        host.command(c)
    assert host.write_config() == open(os.path.join(G, "config.txt")).read()


def test_zoom_modes_and_failures(bb, host):
    host.command("f_globe cube")
    host.command("f_lens panini")
    # closed forms: panini x(lon) = 2 sin(lon)/(1+cos(lon)) = 2 tan(lon/2)
    for fov in (60, 90, 170, 180):
        host.command(f"f_fov {fov}")
        host.build_lensmap(640, 480, 64)
        assert abs(host.scale - 2 * np.tan(np.radians(fov) / 4) / 320) < 1e-7
    host.command("f_vfov 90")
    host.build_lensmap(640, 480, 64)
    assert abs(host.scale - 2 * np.tan(np.radians(45)) / (1 + 1) / 240) < 1e-7  # S*tan(lat), S = 1 at lon 0
    # fov above the lens maximum
    host.clear_log()
    host.command("f_vfov 181")
    with pytest.raises(bb.BlinkyError) as e:
        host.build_lensmap(64, 48, 32)
    assert e.value.code == bb.E_ZOOM and "vfov must be less than 180" in host.log
    # cover/contain need lens_width/lens_height; panini has neither
    host.clear_log()
    host.command("f_cover")
    with pytest.raises(bb.BlinkyError) as e:
        host.build_lensmap(64, 48, 32)
    assert e.value.code == bb.E_ZOOM and "neither lens_height nor lens_width" in host.log
    # the failed map is empty but published (the reference renders nothing)
    idx, _ = host.lensmap()
    assert (idx == -1).all()
    # f_fov on a lens without max_fov
    host.command("f_lens quincuncial")
    host.command("f_fov 90")
    host.clear_log()
    with pytest.raises(bb.BlinkyError):
        host.build_lensmap(64, 48, 32)
    assert "max_fov & max_vfov not specified" in host.log
    # cover vs contain on a 1:1 lens in a 4:3 view
    host.command("f_contain")
    host.build_lensmap(64, 48, 32)
    s_contain = host.scale
    host.command("f_cover")
    host.build_lensmap(64, 48, 32)
    assert s_contain == 2 * np.sqrt(2) / 48 and host.scale == 2 * np.sqrt(2) / 64


def test_scripts_from_source_and_error_paths(bb, host):
    host.load_globe("mini", "plates = { { {0,0,1}, {0,1,0}, 120 } }")
    assert host.globe_valid and host.numplates == 1
    # a lens that returns a plain direction; onload picks the zoom
    host.load_lens("flat", """
lens_width = 2
lens_height = 2
onload = "f_contain"
function lens_inverse(x, y) return x, y, 1 end
""")
    assert host.onload == "f_contain" and host.zoom_type == bb.ZOOM_CONTAIN
    host.build_lensmap(40, 40, 16)
    idx, _ = host.lensmap()
    assert (idx >= 0).mean() > 0.9 and host.display() == [1, 0, 0, 0, 0, 0]
    # wrong number of return values aborts the build (status -1, :1581-1583)
    host.load_lens("bad2", "lens_width=2 lens_height=2 onload='f_contain' function lens_inverse(x,y) return x, y end")
    host.clear_log()
    with pytest.raises(bb.BlinkyError) as e:
        host.build_lensmap(40, 40, 16)
    assert e.value.code == bb.E_SCRIPT and "returned 2 values instead of 3" in host.log
    # a single non-nil value too
    host.load_lens("bad1", "lens_width=2 lens_height=2 onload='f_contain' function lens_inverse(x,y) return 5 end")
    host.clear_log()
    with pytest.raises(bb.BlinkyError):
        host.build_lensmap(40, 40, 16)
    assert "single non-nil value" in host.log
    # non-number values
    host.load_lens("bad3", "lens_width=2 lens_height=2 onload='f_contain' function lens_inverse(x,y) return x, {}, 1 end")
    host.clear_log()
    with pytest.raises(bb.BlinkyError):
        host.build_lensmap(40, 40, 16)
    assert "non-number value" in host.log
    # a runtime error inside the script is reported, not fatal (the reference would panic)
    host.load_lens("boom", "lens_width=2 lens_height=2 onload='f_contain' function lens_inverse(x,y) return x + nil, 0, 1 end")
    host.clear_log()
    with pytest.raises(bb.BlinkyError):
        host.build_lensmap(40, 40, 16, threads=3)
    assert "attempt to perform arithmetic" in host.log
    # syntax error at load
    with pytest.raises(bb.BlinkyError):
        host.load_lens("syn", "function lens_inverse(x,y) return x,, end")
    assert not host.lens_valid and host.lens_name == ""
    # unsupported `map`
    with pytest.raises(bb.BlinkyError):
        host.load_lens("m", "map = 'sideways' function lens_inverse(x,y) return x,y,1 end")
    assert "Unsupported map function: sideways" in host.log
    # `map` forces the forward builder even when both functions exist
    host.load_lens("both", """
map = "lens_forward"
lens_width = 4 lens_height = 4 onload = "f_contain"
function lens_inverse(x, y) return x, y, 1 end
function lens_forward(x, y, z) return x/z, y/z end
""")
    assert host.map_type == bb.MAP_FORWARD
    # globe errors
    for src, msg in [("plates = 3", "plates must be an array"), ("plates = { { {0,0,1}, {0,1}, 90 } }", "up vector is not a 3d vector"),
                     ("plates = { { {0,0,'x'}, {0,1,0}, 90 } }", "element 3 not a number"),
                     ("plates = { { {0,0,1}, {0,1,0}, 0 } }", "fov must > 0"),
                     ("plates = {} for i=1,7 do plates[i] = { {0,0,1}, {0,1,0}, 90 } end", "more than 6 plates")]:
        host.clear_log()
        with pytest.raises(bb.BlinkyError):
            host.load_globe("g", src)
        assert msg in host.log and not host.globe_valid


def test_lua_state_is_shared_between_scripts(host):
    # quirk 6: one Lua state for everything; only the 8+2 reserved names are cleared
    host.load_globe("g", "leak = 41 plates = { { {0,0,1}, {0,1,0}, 90 } }")
    host.load_lens("l", "lens_width = leak + 1 lens_height = 1 onload = 'f_contain' function lens_inverse(x,y) return x,y,1 end")
    assert host.lens_width == 42
    # numplates is visible to the lens (debug.lua relies on it) and refreshed on rebuild
    host.load_lens("n", "lens_width = numplates lens_height = 1 onload='f_cover' function lens_inverse(x,y) return x,y,1 end")
    assert host.lens_width == 1
    host.load_globe("g2", "plates = { { {0,0,1}, {0,1,0}, 90 }, { {0,0,-1}, {0,1,0}, 90 } }")
    host.build_lensmap(32, 32, 16)  # re-runs the lens script (:737)
    assert host.lens_width == 2
    # reserved lens names are cleared between lenses
    host.load_lens("p", "max_fov = 100 max_vfov = 50 function lens_inverse(x,y) return x,y,1 end")
    assert (host.max_fov, host.max_vfov) == (100, 50)
    host.load_lens("q", "function lens_inverse(x,y) return x,y,1 end")
    assert (host.max_fov, host.max_vfov, host.lens_width, host.onload) == (0, 0, 0.0, "")


def test_needs_rebuild_tracks_the_change_flags(host):
    host.command("f_globe cube")
    host.command("f_lens panini")
    assert host.needs_rebuild(64, 48, 32)
    host.build_lensmap(64, 48, 32)
    assert not host.needs_rebuild(64, 48, 32)
    assert host.needs_rebuild(64, 50, 32) and host.needs_rebuild(64, 48, 16)
    for c in ("f_fov 120", "f_rubixgrid 5 2 1", "f_lens panini", "f_globe cube"):
        host.command(c)
        assert host.needs_rebuild(64, 48, 32), c
        host.build_lensmap(64, 48, 32)
        assert not host.needs_rebuild(64, 48, 32)
    host.command("f_rubix")  # toggling the overlay does not touch the map (checked at render time, :2416)
    assert not host.needs_rebuild(64, 48, 32)
    # default plate size is min(w,h) like the reference (:707)
    host.build_lensmap(64, 48, 0)
    assert host.platesize == 48


def test_rubixgrid_changes_tints_only(host):
    assert build(host, "cube", "panini", 96, 72, 60) == 0
    i0, t0 = host.lensmap()
    host.command("f_rubixgrid 3 2 1")
    host.build_lensmap(96, 72, 60)
    i1, t1 = host.lensmap()
    assert np.array_equal(i0, i1) and not np.array_equal(t0, t1)
    # numcells=3, cell=2, pad=1 -> 10 units of 6 px; texel (px,py) is in a cell iff both
    # fmod(px/6, 3) >= 1 and fmod(py/6, 3) >= 1
    px, py = (i1 % 3600) % 60, (i1 % 3600) // 60
    incell = (np.fmod(px / 6.0, 3) >= 1) & (np.fmod(py / 6.0, 3) >= 1)
    assert np.array_equal(t1 != 255, incell)
    host.command("f_rubixgrid 10 4 1")


def test_saveglobe_pcx_matches_compiled_reference(bb, host, live, tmp_path):
    """f_saveglobe: the PCX files (header, escaped pixel stream, 0xFE blanking of texels another
    plate owns, palette trailer) must be byte-identical to the reference's WritePCXplate output"""
    want = np.load(os.path.join(G, "reference_pcx.npz"))
    w, h = 48, 40
    ps = min(w, h)
    for globe in ("cube", "trism", "fast"):
        for margins in (0, 1):
            mine = tmp_path / f"{globe}{margins}"
            os.makedirs(mine)
            host.command(f"f_globe {globe}")
            host.command("f_lens equirect")  # shows every plate
            faces = bb.synthetic_faces(host.numplates, ps, 6)
            host.command(f"f_saveglobe g{margins}_ {margins}")
            host.clear_log()
            host.build_lensmap(w, h, ps)
            assert host.saveglobe_pending
            host.save_globe(faces, str(mine))
            assert not host.saveglobe_pending
            assert live["saveglobe_logs"][f"{globe}__{margins}"] == host.log  # "Wrote <name>" lines
            for i in range(host.numplates):
                a = want[f"{globe}__g{margins}_{i}"].tobytes()
                b = open(mine / f"g{margins}_{i}.pcx", "rb").read()
                assert a == b, (globe, margins, i, len(a), len(b))
    host.clear_log()
    host.command("f_saveglobe")
    assert "f_saveglobe <name> [full flag=0]" in host.log


def test_tile_plan_and_lensmap_do_not_depend_on_the_thread_count(host):
    """the per-pixel host passes (lensmap finish, tile planning) are split over threads"""
    for globe, lens, size in [("cube", "panini", (333, 201, 96)), ("tetra", "quincuncial", (160, 97, 64)), ("cube", "hammer", (256, 128, 80))]:
        host.command(f"f_globe {globe}")
        host.command(f"f_lens {lens}")
        host.build_lensmap(*size, threads=1)
        packed = host.lensmap_packed().copy()
        d1 = host.plan_digest(1)
        assert d1 != 0 and d1 == host.plan_digest(3) == host.plan_digest(16)
        host.build_lensmap(*size, threads=5)
        assert np.array_equal(packed, host.lensmap_packed())
        assert d1 == host.plan_digest(7)
