"""Generates the committed golden vectors from the COMPILED REFERENCE (oracle/_ref,
i.e. the unmodified /root/reference/engine/NQ/fisheye.c) driving the repo's own
script set.  Run here (needs oracle/_ref built):

    python tests/golden/make_golden.py <reference checkout>

Outputs (all under tests/golden/):
  lensmaps_small.npz   idx/tint per (globe, lens) at 128x96, plates 48
  meta_small.json      scale, display flags, plate count, console log per combo
  c1.npz / c1.json     BASELINE config C1 (640x480, cube 6x256^2, panini f_fov 180):
                       lensmap + sha256 of rendered frames (rubix off / on)
  frames_small.npz     render_lensmap outputs for seeded faces/background, incl. a view
                       rectangle inside a wider screen (rowbytes > width)
  engine_frame.npz     whole F_RenderView frames (platesize = min(w,h))
  palmaps.npz          the six rubix LUTs for the seeded palette
  config.txt           F_WriteConfig output
  reference_live.json  the reference's side of every test that used to drive the compiled
                       reference live (lensmap digests of every globe x lens, console
                       and config text, rendered frame digests, the reference's own
                       scripts run by the product)
  reference_pcx.npz    f_saveglobe PCX files written by the reference

The tests compare against these files only, so they need neither the reference
checkout nor oracle/_ref.
"""
import hashlib
import json
import os
import shutil
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import blinky_b200 as bb  # noqa: E402  (inputs only: seeded palette/faces/background, script dir)
from oracle.pyoracle import RefOracle  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))

LENSES = ["cube", "cubestereo", "cylinder", "debug", "eckert1", "eckert4", "eckert5", "equirect", "fahey", "fisheye1",
          "fisheye2", "gallstereo", "gins8", "gumby", "hammer", "kavrayskiy7", "larrivee", "mercator", "miller",
          "mollweide", "panini", "polyconic", "quincuncial", "rectilinear", "sinusoidal", "stereographic",
          "vandergrinten", "wagner6", "winkel1", "winkel2", "winkeltripel"]
GLOBES = ["cube", "cube_corner", "cube_edge", "fast", "tetra", "trism"]
SMALL = (128, 96, 48)


def small_combos():
    combos = [("cube", l) for l in LENSES]
    for g in GLOBES[1:]:
        for l in ("panini", "quincuncial", "debug", "stereographic", "sinusoidal"):
            combos.append((g, l))
    return combos


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    pal = bb.synthetic_palette()
    R = RefOracle.get(bb.SCRIPT_DIR, pal)
    np.savez_compressed(os.path.join(OUT, "palmaps.npz"), palette=pal, palmaps=R.palmaps())

    # ---- small lensmaps ---------------------------------------------------
    W, H, PS = SMALL
    R.set_screen(W, H)
    arrays, meta = {}, {}
    for g, l in small_combos():
        R.clear_log()
        R.command(f"f_globe {g}")
        R.command(f"f_lens {l}")
        rc = R.build(W, H, PS)
        idx, tint = R.lensmap()
        key = f"{g}__{l}"
        arrays[key + "__idx"] = idx
        arrays[key + "__tint"] = tint
        meta[key] = dict(rc=rc, scale=R.scale, display=R.display(), numplates=R.numplates, map_type=R.map_type,
                         log=R.log, plates_sha=sha(R.plates()))
    np.savez_compressed(os.path.join(OUT, "lensmaps_small.npz"), **arrays)
    json.dump(meta, open(os.path.join(OUT, "meta_small.json"), "w"), indent=1, sort_keys=True)

    # ---- rendered frames (small) -------------------------------------------
    frames = {}
    for g, l, rubix in [("cube", "panini", False), ("cube", "panini", True), ("cube", "hammer", True),
                        ("trism", "stereographic", True), ("cube", "winkel1", True), ("fast", "quincuncial", False)]:
        R.command(f"f_globe {g}")
        R.command(f"f_lens {l}")
        if R.rubix_enabled != rubix:
            R.command("f_rubix")
        # view rectangle inside a wider screen: rowbytes 160, vrect at (8, 6)
        R.set_screen(160, 120, 160, 8, 6, W, H)
        R.build(W, H, PS)
        faces = bb.synthetic_faces(R.numplates, PS, 0)
        bg = np.random.default_rng(3).integers(0, 256, (120, 160), dtype=np.uint8)
        out = R.render(faces, bg)
        frames[f"{g}__{l}__rubix{int(rubix)}"] = out
    if R.rubix_enabled:
        R.command("f_rubix")
    np.savez_compressed(os.path.join(OUT, "frames_small.npz"), **frames)

    # ---- whole engine frames through F_RenderView ---------------------------
    eng = {}
    for g, l in [("cube", "panini"), ("cube", "fisheye1"), ("trism", "equirect")]:
        w, h = 96, 64
        R.set_screen(w, h)
        R.command(f"f_globe {g}")
        R.command(f"f_lens {l}")
        ps = min(w, h)
        faces = bb.synthetic_faces(R.numplates, ps, 1)
        bg = bb.synthetic_background(w, h)
        out, ncalls = R.frame(faces, bg)
        eng[f"{g}__{l}"] = out
        eng[f"{g}__{l}__calls"] = np.array([ncalls])
    np.savez_compressed(os.path.join(OUT, "engine_frame.npz"), **eng)

    # ---- C1 -----------------------------------------------------------------
    W1, H1, PS1 = 640, 480, 256
    R.set_screen(W1, H1)
    R.command("f_globe cube")
    R.command("f_lens panini")
    R.command("f_fov 180")
    R.command("f_rubixgrid 10 4 1")
    R.build(W1, H1, PS1)
    idx, tint = R.lensmap()
    faces = bb.synthetic_faces(6, PS1, 0)
    bg = bb.synthetic_background(W1, H1)
    off = R.render(faces, bg)
    R.command("f_rubix")
    on = R.render(faces, bg)
    R.command("f_rubix")
    np.savez_compressed(os.path.join(OUT, "c1.npz"), idx=idx, tint=tint)
    json.dump(dict(scale=R.scale, display=R.display(), idx_sha=sha(idx), tint_sha=sha(tint), faces_sha=sha(faces),
                   bg_sha=sha(bg), render_rubix_off_sha=sha(off), render_rubix_on_sha=sha(on),
                   mapped=int((idx >= 0).sum())),
              open(os.path.join(OUT, "c1.json"), "w"), indent=1, sort_keys=True)

    # ---- config ---------------------------------------------------------------
    R.command("f_lens hammer")
    R.command("f_globe trism")
    R.command("f_fov 123")
    R.command("f_rubixgrid 7 3.5 0.25")
    txt = R.write_config("/tmp/_blinky_cfg.txt")
    open(os.path.join(OUT, "config.txt"), "w").write(txt)
    R.command("f_rubixgrid 10 4 1")
    reference_live(R, pal, sys.argv[1])
    print("golden vectors written to", OUT)


def lensmap_digest(R, w, h, ps):
    rc = R.build(w, h, ps)
    idx, tint = R.lensmap()
    return dict(rc=rc, idx_sha=sha(idx), tint_sha=sha(tint), scale=R.scale, display=R.display(), plates_sha=sha(R.plates()),
                log=R.log)


def reference_live(R, pal, reference_dir):
    """The reference's results for the command sequences of the tests that compare with it
    (tests/test_host.py, test_oracle.py, test_gpu_parity.py, test_dropin.py)."""
    import tempfile

    tmp = tempfile.mkdtemp()
    cfg = os.path.join(tmp, "config.cfg")
    live = {}

    # every globe x lens at two sizes (test_host: all combinations; test_oracle: the restatement)
    for key, (w, h, ps) in (("combos_96x64x40", (96, 64, 40)), ("combos_200x150x100", (200, 150, 100))):
        R.set_screen(w, h)
        live[key] = {}
        for g in GLOBES:
            for l in LENSES:
                R.clear_log()
                R.command(f"f_globe {g}")
                R.command(f"f_lens {l}")
                live[key][f"{g}__{l}"] = lensmap_digest(R, w, h, ps)

    # the reference's own lua-scripts, run by the product (test_host: own scripts equal the reference's)
    scripts = {}
    with bb.Fisheye(device=None, basedir=os.path.join(reference_dir, "game"), palette=pal) as fe:
        for g in GLOBES:
            for l in LENSES:
                fe.clear_log()
                fe.command(f"f_globe {g}")
                fe.command(f"f_lens {l}")
                try:
                    fe.build_lensmap(112, 80, 56, 4)
                    rc = 0
                except bb.BlinkyError as e:
                    rc = e.code
                idx, tint = fe.lensmap()
                scripts[f"{g}__{l}"] = dict(rc=rc, idx_sha=sha(idx), tint_sha=sha(tint), scale=fe.scale, display=fe.display(),
                                            log=fe.log, onload=fe.onload, max_fov=fe.max_fov, max_vfov=fe.max_vfov,
                                            lens_width=fe.lens_width, lens_height=fe.lens_height, map_type=fe.map_type)
    live["reference_scripts_112x80x56"] = scripts

    # console surface (test_host)
    for c in ("fisheye 1", "f_globe cube", "f_lens panini", "f_fov 180", "f_rubixgrid 10 4 1"):
        R.command(c)
    if R.rubix_enabled:
        R.command("f_rubix")
    R.clear_log()
    for c in CONSOLE_SCRIPT:
        R.command(c)
    # the ERROR: lines are luaL_loadfile's message, which names the reference's script directory; the test
    # ignores them (the product words its file-open errors differently)
    log = "\n".join(x for x in R.log.split("\n") if not x.startswith("ERROR:"))
    live["console"] = dict(log=log, config=R.write_config(cfg))

    # f_saveglobe PCX files (test_host)
    pcx, saveglobe_logs = {}, {}
    w, h = 48, 40
    ps = min(w, h)
    R.set_screen(w, h)
    with tempfile.TemporaryDirectory() as d:
        R.lib.ref_set_write_dir(d.encode())
        for globe in ("cube", "trism", "fast"):
            for margins in (0, 1):
                R.command(f"f_globe {globe}")
                R.command("f_lens equirect")
                faces = bb.synthetic_faces(R.numplates, ps, 6)
                R.command(f"f_saveglobe g{margins}_ {margins}")
                R.clear_log()
                R.frame(faces, bb.synthetic_background(w, h))
                saveglobe_logs[f"{globe}__{margins}"] = R.log
                for i in range(R.numplates):
                    pcx[f"{globe}__g{margins}_{i}"] = np.frombuffer(open(os.path.join(d, f"g{margins}_{i}.pcx"), "rb").read(), np.uint8)
    live["saveglobe_logs"] = saveglobe_logs
    np.savez_compressed(os.path.join(OUT, "reference_pcx.npz"), **pcx)

    # rendered frames at 320x200 (test_gpu_parity)
    frames = {}
    W, H, PS = 320, 200, 128
    R.set_screen(W, H)
    for g, l, rubix in LIVE_FRAMES:
        R.command(f"f_globe {g}")
        R.command(f"f_lens {l}")
        if R.rubix_enabled != rubix:
            R.command("f_rubix")
        R.build(W, H, PS)
        frames[f"{g}__{l}__rubix{int(rubix)}"] = sha(R.render(bb.synthetic_faces(R.numplates, PS, 9), bb.synthetic_background(W, H)))
    if R.rubix_enabled:
        R.command("f_rubix")
    live["frames_320x200x128"] = frames

    # the drop-in's engine seam: console, whole F_RenderView frames, config (test_dropin)
    for c in ("fisheye 1", "f_globe cube", "f_lens panini", "f_fov 180", "f_rubixgrid 10 4 1"):
        R.command(c)
    if R.rubix_enabled:
        R.command("f_rubix")
    R.clear_log()
    for c in DROPIN_CONSOLE:
        R.command(c)
    dropin = {"log": R.log, "frames": {}}
    for g, l, rubix, scr in DROPIN_FRAMES:
        R.command(f"f_globe {g}")
        R.command(f"f_lens {l}")
        if R.rubix_enabled != rubix:
            R.command("f_rubix")
        w, h, rowbytes, vx, vy, vw, vh = scr
        R.set_screen(w, h, rowbytes, vx, vy, vw, vh)
        faces = bb.synthetic_faces(R.numplates, min(vw, vh), 4)
        out, ncalls = R.frame(faces, np.random.default_rng(3).integers(0, 256, (h, w), dtype=np.uint8))
        dropin["frames"][f"{g}__{l}"] = dict(sha=sha(out), calls=ncalls)
    if R.rubix_enabled:
        R.command("f_rubix")
    dropin["config"] = R.write_config(cfg)
    # 640x480 frames before and after an f_lens change (test_dropin: the rebuild never holds a frame up)
    for c in ("fisheye 1", "f_globe cube", "f_lens panini", "f_fov 180"):
        R.command(c)
    if R.rubix_enabled:
        R.command("f_rubix")
    R.set_screen(640, 480, 640, 0, 0, 640, 480)
    faces = bb.synthetic_faces(6, 480, 9)
    bg = np.random.default_rng(5).integers(0, 256, (480, 640), dtype=np.uint8)
    dropin["rebuild_old_sha"] = sha(R.frame(faces, bg)[0])
    R.command("f_lens winkeltripel")
    R.command("f_contain")
    dropin["rebuild_new_sha"] = sha(R.frame(faces, bg)[0])
    live["dropin"] = dropin

    json.dump(live, open(os.path.join(OUT, "reference_live.json"), "w"), indent=0, sort_keys=True)
    shutil.rmtree(tmp)


CONSOLE_SCRIPT = ["fisheye 1", "f_rubixgrid 10 4 1", "fisheye", "fisheye 0", "fisheye 1", "f_help", "f_rubix", "f_rubix", "f_rubixgrid",
                  "f_rubixgrid 7 3.5 0.25", "f_rubixgrid", "f_fov", "f_fov 100", "f_fov", "f_vfov 60", "f_vfov", "f_cover", "f_fov",
                  "f_contain", "f_fov", "f_lens", "f_globe", "f_lens hammer", "f_lens", "f_globe trism", "f_globe", "f_lens nosuchlens",
                  "f_globe nosuchglobe", "f_lens panini", "f_globe cube", "f_rubixgrid 10 4 1", "F_FOV 90"]
LIVE_FRAMES = [("cube", "panini", True), ("trism", "stereographic", False), ("tetra", "hammer", True), ("cube", "winkeltripel", True),
               ("fast", "panini", False), ("cube", "polyconic", True)]
DROPIN_CONSOLE = ["f_help", "f_fov", "f_lens hammer", "f_lens", "f_globe trism", "f_globe", "f_rubix", "f_rubix", "f_vfov 70", "f_cover",
                  "f_rubixgrid", "fisheye", "f_lens panini", "f_globe cube"]
DROPIN_FRAMES = [("cube", "panini", False, (96, 64, 96, 0, 0, 96, 64)), ("cube", "fisheye1", True, (128, 80, 136, 16, 8, 96, 64)),
                 ("trism", "equirect", True, (96, 64, 96, 0, 0, 96, 64)), ("tetra", "winkel1", False, (104, 72, 104, 8, 8, 88, 56))]


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_golden.py <reference checkout (its game/ holds the reference's lua-scripts)>")
    main()
