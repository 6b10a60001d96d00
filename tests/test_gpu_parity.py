"""Parity of the CUDA path (GPU suite, everything through the C ABI).

The checker is the CPU oracle: the plain-C restatement of render_lensmap
(oracle/blinky_oracle.c) over the lensmap the oracle builds itself from its C
transcription of the lens, and the committed golden frames and frame digests produced
by the compiled reference.  Integer byte work: every comparison is exact."""
import json
import os

import numpy as np
import pytest

from conftest import sha
from oracle.pyoracle import TRANSCRIBED_GLOBES, TRANSCRIBED_LENSES

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def torch_mod(cuda_device):
    import torch

    return torch


@pytest.fixture()
def fe(bb, palette, cuda_device):
    f = bb.Fisheye(device=cuda_device, palette=palette)
    yield f
    f.close()


def setup(fe, globe, lens, w, h, ps, zoom=None, rubix=False, threads=8):
    fe.command(f"f_globe {globe}")
    fe.command(f"f_lens {lens}")
    if zoom:
        fe.command(zoom)
    fe.set_rubix(rubix)
    fe.build_lensmap(w, h, ps, threads)


def gpu_warp(torch, fe, faces, nframes=1, rgba=False):
    d_faces = torch.from_numpy(np.ascontiguousarray(faces)).cuda()
    shape = (nframes, fe.height, fe.width)
    d_out = torch.zeros(shape, dtype=torch.int32 if rgba else torch.uint8, device="cuda")
    fe.warp(d_faces, d_out, nframes=nframes, stream=torch.cuda.current_stream().cuda_stream, rgba=rgba)
    torch.cuda.synchronize()
    return d_out.cpu().numpy()


def test_native_library_is_what_runs(bb, fe):
    """the hot path is this repo's in-tree .so; report it for the driver's loaded-library check"""
    maps = open("/proc/self/maps").read()
    assert bb.LIB_PATH in maps


RING_KNOBS = [
    {},                                                      # shipped defaults
    {"BLINKY_SERIAL_GATHER": "1"},                           # GATHER tiles in K3 instead of as CTAs of the ring kernel's launch
    {"BLINKY_MERGED_ITEMS": "1000000"},                      # ... and the other way round: always in the ring kernel's launch
    {"BLINKY_RING_CTAS": "2", "BLINKY_STATIC_PCT": "0"},     # few warps, every unit from the ticket counter: long unit sequences per warp
    {"BLINKY_RING_CTAS": "16", "BLINKY_STATIC_PCT": "100"},  # as many warps as the registers allow, no tickets
    {"BLINKY_RING_BYTES": "128", "BLINKY_RING_BOXES": "6"},  # the smallest ring the plan allows (its largest box): wraps all the time
    {"BLINKY_RING_BYTES": "32768", "BLINKY_RING_BOXES": "6", "BLINKY_RING_CTAS": "4"},  # a deep ring: six boxes of a warp in flight
    {"BLINKY_FCHUNK": "1"}, {"BLINKY_FCHUNK": "3"}, {"BLINKY_FCHUNK": "16"},             # unit = 1 / 3 / all frames
]


@pytest.mark.parametrize("knobs", RING_KNOBS, ids=lambda k: ",".join(f"{a[7:]}={b}" for a, b in k.items()) or "default")
def test_ring_kernel_schedules_and_ring_geometries(bb, restate, palette, torch_mod, cuda_device, knobs, monkeypatch):
    """The ring kernel's tuning knobs change how units are handed out, how many boxes a warp keeps in flight and
    where they sit in its byte ring — never the pixels.  Two plans: one with BOX, GATHER and EMPTY tiles and the
    rubix overlay (hammer on a tetrahedron), one with large boxes (quincuncial), five frames each, against the oracle."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    pm = restate.palmaps(palette)
    for globe, lens, zoom, (W, H, PS), rubix in (("tetra", "hammer", "f_contain", (1000, 562, 512), True),
                                                 ("cube", "quincuncial", "f_cover", (1280, 720, 1024), False)):
        with bb.Fisheye(device=cuda_device, palette=palette) as f:   # the knobs are read when the context is created
            setup(f, globe, lens, W, H, PS, zoom, rubix)
            bg = bb.synthetic_background(W, H)
            f.set_background(bg)
            idx, tint = f.lensmap()
            nf = 5
            faces = np.stack([bb.synthetic_faces(f.numplates, PS, 40 + i) for i in range(nf)])
            got = gpu_warp(torch_mod, f, faces, nframes=nf)
            assert "warp_ring_kernel" in f.last_kernel
            for i in range(nf):
                want = restate.render(idx, tint, faces[i], pm, rubix, background=bg)
                assert np.array_equal(got[i], want), (knobs, lens, i, f.last_kernel)
            one = gpu_warp(torch_mod, f, faces[3:4], nframes=1)[0]
            assert np.array_equal(one, got[3]), (knobs, lens, "single frame", f.last_kernel)


@pytest.mark.parametrize("rubix", [False, True])
@pytest.mark.parametrize("kernel", [0, 1])
def test_c1_against_oracle_and_golden(bb, fe, restate, palette, torch_mod, rubix, kernel):
    """BASELINE C1: 640x480, cube 6x256^2, panini f_fov 180 — bit-exact, rubix off and on,
    both kernel variants (0 = tiled TMA, 1 = flat gather)"""
    W, H, PS = 640, 480, 256
    setup(fe, "cube", "panini", W, H, PS, "f_fov 180", rubix)
    fe.set_kernel(kernel)
    bg = bb.synthetic_background(W, H)
    fe.set_background(bg)
    faces = bb.synthetic_faces(6, PS, 0)
    got = gpu_warp(torch_mod, fe, faces)[0]
    assert ("warp_ring_kernel" if kernel == 0 else "warp_gather_kernel") in fe.last_kernel
    om = restate.build("cube", "panini", W, H, PS, zoom=("f_fov", 180))
    idx, tint = fe.lensmap()
    assert np.array_equal(idx, om["idx"]) and np.array_equal(tint, om["tint"])
    want = restate.render(om["idx"], om["tint"], faces, restate.palmaps(palette), rubix, background=bg)
    assert np.array_equal(got, want)
    c1 = json.load(open(os.path.join(G, "c1.json")))
    assert sha(got) == c1["render_rubix_on_sha" if rubix else "render_rubix_off_sha"]
    # the end-to-end host path gives the same bytes
    host = fe.warp_host(faces.reshape(1, -1))[0]
    assert np.array_equal(host, want)


def test_lens_globe_matrix_against_oracle(bb, fe, restate, palette, torch_mod):
    W, H, PS = 256, 160, 96
    pm = restate.palmaps(palette)
    bg = bb.synthetic_background(W, H)
    for g in TRANSCRIBED_GLOBES:
        for l in TRANSCRIBED_LENSES:
            for rubix in (False, True):
                setup(fe, g, l, W, H, PS, None, rubix)
                fe.set_background(bg)
                om = restate.build(g, l, W, H, PS)
                idx, tint = fe.lensmap()
                assert np.array_equal(idx, om["idx"]) and np.array_equal(tint, om["tint"]), (g, l)
                faces = bb.synthetic_faces(fe.numplates, PS, 3)
                want = restate.render(om["idx"], om["tint"], faces, pm, rubix, background=bg)
                for kernel in (0, 1):
                    fe.set_kernel(kernel)
                    got = gpu_warp(torch_mod, fe, faces)[0]
                    assert np.array_equal(got, want), (g, l, rubix, kernel)


def test_all_shipped_lenses_against_oracle_render(bb, fe, restate, palette, torch_mod):
    """lenses without a C transcription: the oracle renders the product's lensmap (the
    lensmap itself is pinned by the CPU suite against the compiled reference / golden)"""
    from conftest import ALL_LENSES

    W, H, PS = 192, 128, 80
    pm = restate.palmaps(palette)
    bg = bb.synthetic_background(W, H)
    for l in ALL_LENSES:
        setup(fe, "cube", l, W, H, PS, None, True)
        fe.set_background(bg)
        idx, tint = fe.lensmap()
        faces = bb.synthetic_faces(6, PS, 5)
        want = restate.render(idx, tint, faces, pm, True, background=bg)
        assert np.array_equal(gpu_warp(torch_mod, fe, faces)[0], want), l


def test_golden_frames_with_view_rectangle(bb, fe, torch_mod):
    """frames_small.npz were rendered by the compiled reference into a 160x120 screen with
    scr_vrect = (8, 6, 128, 96): the host path with keep_unmapped reproduces them exactly"""
    frames = np.load(os.path.join(G, "frames_small.npz"))
    W, H, PS = 128, 96, 48
    for key in frames.files:
        g, l, r = key.split("__")
        setup(fe, g, l, W, H, PS, None, r == "rubix1")
        faces = bb.synthetic_faces(fe.numplates, PS, 0)
        screen = np.random.default_rng(3).integers(0, 256, (120, 160), dtype=np.uint8)  # what Draw_TileClear left
        fe.warp_host(faces.reshape(1, -1), screen.reshape(1, 120, 160), keep_unmapped=True, x0=8, y0=6)
        assert np.array_equal(screen, frames[key]), key


def test_against_compiled_reference_live(bb, fe, torch_mod):
    """frames the compiled reference rendered (tests/golden/make_golden.py), as digests"""
    want = json.load(open(os.path.join(G, "reference_live.json")))["frames_320x200x128"]
    W, H, PS = 320, 200, 128
    for g, l, rubix in [("cube", "panini", True), ("trism", "stereographic", False), ("tetra", "hammer", True),
                        ("cube", "winkeltripel", True), ("fast", "panini", False), ("cube", "polyconic", True)]:
        setup(fe, g, l, W, H, PS, None, rubix)
        faces = bb.synthetic_faces(fe.numplates, PS, 9)
        bg = bb.synthetic_background(W, H)
        fe.set_background(bg)
        assert sha(gpu_warp(torch_mod, fe, faces)[0]) == want[f"{g}__{l}__rubix{int(rubix)}"], (g, l)


def test_ragged_and_tiny_sizes(bb, fe, restate, palette, torch_mod):
    pm = restate.palmaps(palette)
    for (w, h, ps) in [(101, 37, 33), (4, 4, 16), (1, 1, 8), (36, 3, 48), (130, 66, 50), (64, 64, 16), (260, 100, 112)]:
        setup(fe, "cube", "fisheye1", w, h, ps, None, True)
        bg = bb.synthetic_background(w, h)
        fe.set_background(bg)
        idx, tint = fe.lensmap()
        faces = bb.synthetic_faces(6, ps, 2)
        want = restate.render(idx, tint, faces, pm, True, background=bg)
        got = gpu_warp(torch_mod, fe, faces)[0]
        assert np.array_equal(got, want), (w, h, ps, fe.last_kernel)
        assert np.array_equal(fe.warp_host(faces.reshape(1, -1))[0], want), (w, h, ps)


def test_empty_map_and_unmapped_pixels(bb, fe, restate, palette, torch_mod):
    W, H, PS = 96, 64, 32
    # a lens that maps nothing: the frame is the background
    fe.load_globe("cube")
    fe.load_lens("none", "lens_width=1 lens_height=1 onload='f_contain' function lens_inverse(x,y) return nil end")
    fe.build_lensmap(W, H, PS)
    bg = bb.synthetic_background(W, H)
    fe.set_background(bg)
    faces = bb.synthetic_faces(6, PS, 0)
    assert np.array_equal(gpu_warp(torch_mod, fe, faces)[0], bg)
    assert fe.display() == [0] * 6 and fe.mapped_pixels == 0
    # keep_unmapped leaves the caller's pixels alone
    screen = np.full((1, H, W), 77, np.uint8)
    fe.warp_host(faces.reshape(1, -1), screen, keep_unmapped=True)
    assert (screen == 77).all()
    # default background is zeros
    fe.set_background(None)
    assert not gpu_warp(torch_mod, fe, faces).any()


def test_batches_and_strides(bb, fe, restate, palette, torch_mod):
    torch = torch_mod
    W, H, PS, N = 224, 96, 64, 7
    setup(fe, "trism", "stereographic", W, H, PS, None, True)
    bg = bb.synthetic_background(W, H)
    fe.set_background(bg)
    idx, tint = fe.lensmap()
    pm = restate.palmaps(palette)
    faces = np.stack([bb.synthetic_faces(5, PS, f) for f in range(N)])
    want = np.stack([restate.render(idx, tint, faces[f], pm, True, background=bg) for f in range(N)])
    for kernel in (0, 1):
        fe.set_kernel(kernel)
        assert np.array_equal(gpu_warp(torch, fe, faces, nframes=N), want)
    # padded strides: frames and outputs embedded in larger buffers
    fstride, ostride = 5 * PS * PS + 4096, W * H + 512
    big_f = torch.zeros(N * fstride, dtype=torch.uint8, device="cuda")
    for f in range(N):
        big_f[f * fstride:f * fstride + 5 * PS * PS] = torch.from_numpy(faces[f].reshape(-1)).cuda()
    big_o = torch.zeros(N * ostride, dtype=torch.uint8, device="cuda")
    fe.set_kernel(0)
    fe.warp(big_f, big_o, nframes=N, face_stride=fstride, out_stride=ostride)
    torch.cuda.synchronize()
    got = big_o.cpu().numpy()
    for f in range(N):
        assert np.array_equal(got[f * ostride:f * ostride + W * H].reshape(H, W), want[f])
    # end-to-end over a batch, plates the lens never looks at are not uploaded
    out = fe.warp_host(faces.reshape(N, -1))
    assert np.array_equal(out, want)
    # on a non-default stream
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_f = torch.from_numpy(faces).cuda()
        d_o = torch.zeros((N, H, W), dtype=torch.uint8, device="cuda")
        fe.warp(d_f, d_o, nframes=N, stream=s.cuda_stream)
    s.synchronize()
    assert np.array_equal(d_o.cpu().numpy(), want)


def test_pinned_host_buffers(bb, fe, restate, palette):
    W, H, PS, N = 128, 64, 32, 4
    setup(fe, "cube", "hammer", W, H, PS, None, False)
    idx, tint = fe.lensmap()
    pm = restate.palmaps(palette)
    src = fe.alloc_pinned(N * 6 * PS * PS)
    dst = fe.alloc_pinned(N * W * H)
    faces = np.stack([bb.synthetic_faces(6, PS, 20 + f) for f in range(N)])
    src[:] = faces.reshape(-1)
    dst[:] = 0
    fe.warp_host(src, dst.reshape(N, H, W))
    want = np.stack([restate.render(idx, tint, faces[f], pm, False) for f in range(N)])
    assert np.array_equal(dst.reshape(N, H, W), want)
    fe.free_pinned(src)
    fe.free_pinned(dst)


def test_rgba_expansion(bb, fe, restate, palette, torch_mod):
    """fused 8-bit -> 32-bit palette expansion (engine/common/vid_sdl.c:539-546)"""
    W, H, PS = 160, 96, 64
    setup(fe, "cube", "panini", W, H, PS, None, True)
    table = np.random.default_rng(5).integers(0, 2**32, 256, dtype=np.uint64).astype(np.uint32)
    fe.set_rgba_table(table)
    idx, tint = fe.lensmap()
    faces = bb.synthetic_faces(6, PS, 1)
    want8 = restate.render(idx, tint, faces, restate.palmaps(palette), True)
    for kernel in (0, 1):
        fe.set_kernel(kernel)
        got = gpu_warp(torch_mod, fe, faces, rgba=True)[0].view(np.uint32)
        assert np.array_equal(got, table[want8]), kernel


def test_rubix_toggle_and_palette_change_need_no_rebuild(bb, fe, restate, palette, torch_mod):
    W, H, PS = 128, 96, 48
    setup(fe, "cube", "panini", W, H, PS, None, False)
    idx, tint = fe.lensmap()
    faces = bb.synthetic_faces(6, PS, 0)
    off = gpu_warp(torch_mod, fe, faces)[0]
    fe.command("f_rubix")
    assert not fe.needs_rebuild(W, H, PS)
    on = gpu_warp(torch_mod, fe, faces)[0]
    assert np.array_equal(off, restate.render(idx, tint, faces, restate.palmaps(palette), False))
    assert np.array_equal(on, restate.render(idx, tint, faces, restate.palmaps(palette), True))
    pal2 = bb.synthetic_palette(99)
    fe.set_palette(pal2)
    assert np.array_equal(gpu_warp(torch_mod, fe, faces)[0], restate.render(idx, tint, faces, restate.palmaps(pal2), True))


def test_plate_sizes_tma_cannot_address(bb, fe, restate, palette, torch_mod):
    """plate rows that are not a multiple of 16 bytes: every tile uses the direct gather path"""
    W, H, PS = 200, 120, 100
    setup(fe, "cube", "stereographic", W, H, PS, None, True)
    assert " 0 box" in fe.plan_summary
    idx, tint = fe.lensmap()
    faces = bb.synthetic_faces(6, PS, 0)
    want = restate.render(idx, tint, faces, restate.palmaps(palette), True)
    assert np.array_equal(gpu_warp(torch_mod, fe, faces)[0], want)


def test_device_memory_and_ipc_export(bb, fe):
    """peer-memory plumbing on one GPU: allocate, warp straight into the raw buffer, export a handle
    (opening it needs a second process: bench.py --gpus 2 does that and checks the bytes)"""
    import torch

    W, H, PS = 128, 64, 32
    setup(fe, "cube", "panini", W, H, PS)
    ptr = fe.alloc_device(2 * W * H)
    handle = fe.ipc_export(ptr)
    assert len(handle) == 64 and any(handle)
    faces = np.stack([bb.synthetic_faces(6, PS, f) for f in range(2)])
    d_faces = torch.from_numpy(faces).cuda()
    fe.warp(d_faces, ptr, nframes=2)
    ref_out = torch.zeros((2, H, W), dtype=torch.uint8, device="cuda")
    fe.warp(d_faces, ref_out, nframes=2)
    torch.cuda.synchronize()

    class Raw:
        __cuda_array_interface__ = {"shape": (2, H, W), "typestr": "|u1", "data": (ptr, False), "version": 2}

    assert torch.equal(torch.as_tensor(Raw(), device="cuda"), ref_out)
    fe.free_device(ptr)
