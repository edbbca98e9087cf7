"""Adaptive anti-aliased frames (tcrt_render_columns_adaptive & co.): the supersampled pixel of tcrt_render_columns_ss where
the plain frame shows contrast, the plain pixel elsewhere.  A frame is checked bit for bit against
where(refine_mask(render()), render_ss(), render()), with the mask restated in numpy below."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import assert_bit_identical, make_scene, pixel_md5, quant8

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

ENTRY_POINTS = ("tcrt_render_columns_adaptive", "tcrt_render_columns_adaptive_rgb8")
SS = (1, 2, 3, 4, 8)
CONTRASTS = (-1, 0, 8, 32, 255)
PIECE_SAMPLES = 1 << 22          # samples per list piece (tcrt_api.cu kPieceSamples)


def refine_mask(frame, contrast):
    """The contract's mask: P -> quant8 -> for each pixel, the largest channel difference to any neighbour (x', z') != (x, z)
    with |x'-x| <= 1, |z'-z| <= 1 inside the frame; refined where that exceeds contrast, everywhere when contrast < 0.
    frame: (W, H, 3) x-major."""
    q = quant8(np.nan_to_num(np.asarray(frame, np.float32), nan=0.0))     # quant8 maps NaN to 0
    W, H, _ = q.shape
    if contrast < 0:
        return np.ones((W, H), bool)
    m = np.zeros((W, H), bool)
    for dx in (-1, 0, 1):
        for dz in (-1, 0, 1):
            if dx == 0 and dz == 0:
                continue
            # pixel (x, z) against (x + dx, z + dz), for the x, z where that neighbour is inside the frame
            xs, xd = slice(max(0, -dx), W - max(0, dx)), slice(max(0, dx), W - max(0, -dx))
            zs, zd = slice(max(0, -dz), H - max(0, dz)), slice(max(0, dz), H - max(0, -dz))
            m[xs, zs] |= np.abs(q[xs, zs] - q[xd, zd]).max(-1) > contrast
    return m


def q8(img):
    return quant8(img).astype(np.uint8)


def expected(plain, ss_frame, contrast):
    mask = refine_mask(plain, contrast)
    return np.where(mask[..., None], ss_frame, plain), mask


def halo_columns(w, x0, x1):
    return min(w, x1 + 1) - max(0, x0 - 1)


def plain_chunks(cols, h):
    """Column chunks of a plain band of `cols` columns going to host memory (tcrt_api.cu plan_chunks)."""
    return min(16, cols, max(1, cols * h // (256 * 1024)))


def assert_bytes_equal(got, want, what=""):
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    bad = int((got != want).any(-1).sum()) if got.ndim == 3 else int((got != want).sum())
    assert bad == 0, f"{what}: {bad} pixels differ"


# ---- no device needed ------------------------------------------------------------------------------------------------

def test_adaptive_symbols_are_exported():
    lib = C.CDLL(_ffi.LIB_PATH)
    for name in ENTRY_POINTS:
        assert hasattr(lib, name), name


def test_adaptive_entry_points_refuse_a_null_context():
    lib = _ffi.load()
    p = api.default_params(8, 8, 2)
    f = np.zeros(8 * 8 * 3, np.float32)
    b = np.zeros(8 * 8 * 3, np.uint8)
    m = np.zeros(8 * 8, np.uint8)
    n = C.c_ulonglong(7)
    st = _ffi.TcrtStats()
    for ss, contrast in ((1, 0), (2, 8), (0, 8), (9, 8), (2, -2), (2, 256)):
        assert lib.tcrt_render_columns_adaptive(None, C.byref(p), ss, contrast, 0, 8, f.ctypes.data_as(C.c_void_p),
                                                m.ctypes.data_as(C.c_void_p), C.byref(n), C.byref(st)) == _ffi.TCRT_ERR_INVALID
        assert lib.tcrt_render_columns_adaptive_rgb8(None, C.byref(p), ss, contrast, 0, 8, b.ctypes.data_as(C.c_void_p),
                                                     m.ctypes.data_as(C.c_void_p), C.byref(n), C.byref(st)) == \
            _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_columns_adaptive(None, None, 2, 8, 0, 8, None, None, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_columns_adaptive_rgb8(None, C.byref(p), 2, 8, 0, 8, None, None, None, None) == _ffi.TCRT_ERR_INVALID
    assert (f == 0).all() and (b == 0).all() and (m == 0).all() and n.value == 7


def test_mask_restatement_on_crafted_frames():
    # a vertical step edge between columns 2 and 3 of a 6 x 4 frame: columns 2 and 3 are refined up to contrast 254
    f = np.zeros((6, 4, 3), np.float32)
    f[3:] = 1.0
    for c in (0, 8, 254):
        m = refine_mask(f, c)
        assert m[2].all() and m[3].all() and not m[[0, 1, 4, 5]].any(), c
    assert not refine_mask(f, 255).any()
    assert refine_mask(f, -1).all()
    # a step of 9 levels in one channel: refined at contrast 8, not at 9
    f = np.zeros((4, 4, 3), np.float32)
    f[2:, :, 1] = 9.0 / 255.0
    assert refine_mask(f, 8)[1:3].all() and not refine_mask(f, 9).any()
    # a corner pixel sees only its 3 in-frame neighbours: the far corner of the frame is not one of them
    f = np.zeros((5, 5, 3), np.float32)
    f[4, 4] = 1.0
    m = refine_mask(f, 0)
    assert m[4, 4] and m[3, 3] and m[3, 4] and m[4, 3] and m.sum() == 4
    f = np.zeros((5, 5, 3), np.float32)
    f[2, 2] = 1.0                                    # an interior pixel: itself and its 8 neighbours
    assert refine_mask(f, 0).sum() == 9
    # NaN quantises to 0 and values above 1 to 255: NaN next to 0 is flat, 7.5 next to 1.0 is flat, 7.5 next to 0 is an edge
    f = np.zeros((3, 1, 3), np.float32)
    f[0, 0] = np.nan
    assert not refine_mask(f, 0).any()
    f[:] = 1.0
    f[1, 0] = 7.5
    assert not refine_mask(f, 0).any()
    f[0, 0] = 0.0
    assert refine_mask(f, 254)[:2].all() and not refine_mask(f, 254)[2].any()
    # a 1 x 1 frame has no neighbours: only contrast -1 refines it
    assert refine_mask(np.zeros((1, 1, 3), np.float32), -1).all() and not refine_mask(np.zeros((1, 1, 3), np.float32), 0).any()


def test_mask_on_golden_frames(golden_frames):
    for key in golden_frames.files:
        fr = golden_frames[key]
        assert refine_mask(fr, -1).all(), key
        assert not refine_mask(fr, 255).any(), key


def test_mask_on_an_oracle_frame():
    """The default scene at 500 x 504 depth 50 (the oracle renders it bit-identically to the GPU): its refined pixels at six
    contrasts, counted once from the oracle frame and pinned here."""
    scene, cam = make_scene("default")
    fr, _ = O.render(scene.flatten(), cam.export(), api.default_params(500, 504, 50))
    counts = {c: int(refine_mask(fr, c).sum()) for c in (-1, 0, 8, 32, 254, 255)}
    assert counts == {-1: 252000, 0: 123207, 8: 34386, 32: 26107, 254: 30, 255: 0}


# ---- on the GPU ------------------------------------------------------------------------------------------------------

def _inside_sphere_scene():
    from test_gpu_parity import _lattice, _lights_and_ground

    cam = api.Camera()
    c = cam.export()
    s = api.Scene()
    _lights_and_ground(s)
    _lattice(s, 5, 5, 3, 1.8, .75)
    eye = (-3 + 1.8 * 2 + .1, -1 + 1.8 * 2 - .2, .8 + 1.8)       # inside the sphere (2, 2, 1)
    for k in range(3):
        delta = eye[k] - c.eye[k]
        c.eye[k] += delta
        c.screen_origin[k] += delta
    return s, c


def _upload(ctx, spec):
    if spec == "inside_sphere":
        s, c = _inside_sphere_scene()
        ctx.upload_flat(s.flatten(), c)              # the flattened scene points into s: keep s alive across the upload
        assert ctx.scene_structures()["grid_cells"] > 0
        return
    scene, cam = make_scene(spec)
    ctx.upload(scene, cam)
    if spec == "synth256":
        assert ctx.scene_structures()["grid_cells"] > 0            # the grid kernel's list mode


SCENES = [("default", 96, 72, 50), ("two_mirrors", 64, 48, 50), ("synth256", 96, 80, 10), ("boxes:3:14", 96, 80, 12),
          ("random:15:90", 88, 64, 8), ("inside_sphere", 64, 48, 8)]


@gpu
@pytest.mark.parametrize("spec,w,h,d", SCENES)
@pytest.mark.parametrize("ss", SS)
def test_adaptive_equals_mask_of_plain_and_ss(gpu_ctx, spec, w, h, d, ss):
    _upload(gpu_ctx, spec)
    p = api.default_params(w, h, d)
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    full, _ = gpu_ctx.render_ss(p, ss)
    full = full.copy()
    m = ss * ss - 1
    for contrast in CONTRASTS:
        want, want_mask = expected(plain, full, contrast)
        mask = np.full((w, h), 0xAB, np.uint8)
        got, gmask, n, st = gpu_ctx.render_adaptive(p, ss, contrast, mask=mask)
        what = f"{spec} ss={ss} contrast={contrast}"
        assert_bit_identical(got, want, what)
        assert np.array_equal(gmask, want_mask.astype(np.uint8)), what
        assert n == int(want_mask.sum()), what
        assert st.rays_primary == w * h + m * n, what
        assert st.bands == [(0, w)]
        if contrast == -1:
            assert_bit_identical(got, full, what)
        if contrast == 255 or ss == 1:
            assert_bit_identical(got, plain, what)
            assert st.gpu_launches == plain_chunks(w, h) + 3, what      # plain pass and classification: no sample launch
        elif n:
            assert st.gpu_launches == plain_chunks(w, h) + 3 + 2, what  # one piece: list render + resolve
        got8, mask8, n8, _ = gpu_ctx.render_adaptive_rgb8(p, ss, contrast)
        assert_bytes_equal(got8, q8(want), what + " RGB8")
        assert mask8 is None and n8 == n


@gpu
@pytest.mark.parametrize("w,h,d,count", [(1920, 1080, 5, 135373), (3840, 2160, 50, 294377)])
def test_reference_size_refine_counts(gpu_ctx, w, h, d, count):
    """The default scene at contrast 8: the refined counts of the 1080p d5 and 4K d50 frames (counted on oracle frames), and
    the 1080p frame against render_ss."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    p = api.default_params(w, h, d)
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    want_mask = refine_mask(plain, 8)
    assert int(want_mask.sum()) == count
    got, mask, n, st = gpu_ctx.render_adaptive(p, 4, 8, mask=np.empty((w, h), np.uint8))
    assert n == count and np.array_equal(mask, want_mask.astype(np.uint8))
    assert st.rays_primary == w * h + 15 * count
    assert_bit_identical(got[~want_mask], plain[~want_mask], "unrefined pixels")
    if w == 1920:
        full, _ = gpu_ctx.render_ss(p, 4)
        assert_bit_identical(got, np.where(want_mask[..., None], full, plain), "1080p ss=4 contrast 8")


@gpu
def test_adaptive_bands_equal_slices_of_the_frame(gpu_ctx):
    """Bands anywhere, one column wide, at both frame edges and of untileable widths: the halo columns make every band a
    slice of the whole frame."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    w, h, ss = 161, 121, 3
    p = api.default_params(w, h, 20)
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    full, _ = gpu_ctx.render_ss(p, ss)
    full = full.copy()
    for contrast in (0, 8):
        want, want_mask = expected(plain, full, contrast)
        for x0, x1 in ((0, 1), (w - 1, w), (80, 81), (0, 7), (3, 50), (50, 53), (w - 13, w), (1, w - 1), (0, w)):
            mask = np.full(((x1 - x0) * h + 64,), 0xAB, np.uint8)
            got, gmask, n, st = gpu_ctx.render_adaptive(p, ss, contrast, x0, x1, mask=mask[:(x1 - x0) * h])
            what = f"[{x0},{x1}) contrast={contrast}"
            assert_bit_identical(got, want[x0:x1], what)
            assert np.array_equal(gmask, want_mask[x0:x1].astype(np.uint8)), what
            assert (mask[(x1 - x0) * h:] == 0xAB).all(), what + ": a guard byte was overwritten"
            assert n == int(want_mask[x0:x1].sum()) and st.bands == [(x0, x1)], what
            assert st.rays_primary == halo_columns(w, x0, x1) * h + (ss * ss - 1) * n, what
            got8, _, _, _ = gpu_ctx.render_adaptive_rgb8(p, ss, contrast, x0, x1)
            assert_bytes_equal(got8, q8(want[x0:x1]), what + " RGB8")


@gpu
@pytest.mark.parametrize("spec,w,h,d,ss,contrast", [("synth256", 3840, 2160, 10, 2, 0), ("synth256", 640, 360, 10, 8, -1),
                                                    ("default", 1920, 1080, 5, 8, 0)])
def test_adaptive_list_pieces(gpu_ctx, spec, w, h, d, ss, contrast):
    """Lists long enough to be traced in three or more pieces, round robin over the render streams."""
    scene, cam = make_scene(spec)
    gpu_ctx.upload(scene, cam)
    p = api.default_params(w, h, d)
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    want_mask = refine_mask(plain, contrast)
    n_want = int(want_mask.sum())
    per_piece = PIECE_SAMPLES // (ss * ss - 1)
    pieces = -(-n_want // per_piece)
    assert pieces >= 3, pieces
    hb = api.HostBuffer(w * h * 12)
    got, mask, n, st = gpu_ctx.render_adaptive(p, ss, contrast, out=hb.array(np.float32, (w, h, 3)),
                                               mask=np.empty((w, h), np.uint8))
    assert n == n_want and np.array_equal(mask, want_mask.astype(np.uint8))
    assert st.gpu_launches == plain_chunks(w, h) + 3 + 2 * pieces
    full, _ = gpu_ctx.render_ss(p, ss)
    assert_bit_identical(got, np.where(want_mask[..., None], full, plain), f"{spec} {w}x{h} ss={ss} contrast={contrast}")
    del got, hb


GUARD = 4096


@gpu
def test_adaptive_destinations(gpu_ctx):
    """Pinned and pageable destinations (1920 x 1080 is staged when pageable), masks with guard bytes, the device-only
    form; RGB8 is quant8 of the float frame."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    w, h, ss, contrast = 1920, 1080, 2, 8
    p = api.default_params(w, h, 5)
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    full, _ = gpu_ctx.render_ss(p, ss)
    want, want_mask = expected(plain, full.copy(), contrast)
    want8, wmask8 = q8(want), want_mask.astype(np.uint8)
    for x0, x1 in ((0, w), (13, 1002)):
        n = (x1 - x0) * h
        hf, h8, hm = api.HostBuffer(12 * n + GUARD), api.HostBuffer(3 * n + GUARD), api.HostBuffer(n + GUARD)
        for kind, fbuf, bbuf, mbuf in (("pinned", hf.array(np.float32, (3 * n + GUARD // 4,)), h8.array(np.uint8, (3 * n + GUARD,)),
                                        hm.array(np.uint8, (n + GUARD,))),
                                       ("pageable", np.empty(3 * n + GUARD // 4, np.float32), np.empty(3 * n + GUARD, np.uint8),
                                        np.empty(n + GUARD, np.uint8))):
            what = f"[{x0},{x1}) {kind}"
            fbuf.view(np.uint8)[:] = 0xAB
            mbuf[:] = 0xAB
            gpu_ctx.render_adaptive(p, ss, contrast, x0, x1, out=fbuf[:3 * n].reshape(x1 - x0, h, 3), mask=mbuf[:n])
            assert_bit_identical(fbuf[:3 * n].reshape(x1 - x0, h, 3), want[x0:x1], what)
            assert np.array_equal(mbuf[:n].reshape(x1 - x0, h), wmask8[x0:x1]), what
            assert (fbuf[3 * n:].view(np.uint8) == 0xAB).all() and (mbuf[n:] == 0xAB).all(), what + ": guard bytes"
            bbuf[:] = 0xAB
            mbuf[:] = 0xAB
            gpu_ctx.render_adaptive_rgb8(p, ss, contrast, x0, x1, out=bbuf[:3 * n].reshape(x1 - x0, h, 3), mask=mbuf[:n])
            assert_bytes_equal(bbuf[:3 * n].reshape(x1 - x0, h, 3), want8[x0:x1], what + " RGB8")
            assert np.array_equal(mbuf[:n].reshape(x1 - x0, h), wmask8[x0:x1]), what + " RGB8 mask"
            assert (bbuf[3 * n:] == 0xAB).all() and (mbuf[n:] == 0xAB).all(), what + " RGB8: guard bytes"
        del hf, h8, hm
    n_dev, st = gpu_ctx.render_adaptive_device(p, ss, contrast)
    assert n_dev == int(want_mask.sum()) and st.d2h_ms == [0.0]
    assert_bit_identical(gpu_ctx.download(np.empty((w, h, 3), np.float32)), want, "device-only + download (pageable)")
    hb = api.HostBuffer(w * h * 12)
    assert_bit_identical(gpu_ctx.download(hb.array(np.float32, (w, h, 3))), want, "device-only + download (pinned)")
    del hb


@gpu
def test_adaptive_frame_is_the_last_render(gpu_ctx, tmp_path):
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    w, h = 160, 120
    p = api.default_params(w, h, 20)
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    full, _ = gpu_ctx.render_ss(p, 4)
    want, _ = expected(plain, full.copy(), 8)
    got8, _, _, _ = gpu_ctx.render_adaptive_rgb8(p, 4, 8)
    assert_bytes_equal(got8, q8(want), "RGB8")
    assert_bit_identical(gpu_ctx.download(np.empty((w, h, 3), np.float32)), want, "download")
    lib = _ffi.load()
    ptr, n = C.c_void_p(), C.c_size_t()
    assert lib.tcrt_device_frame(gpu_ctx._h, 0, C.byref(ptr), C.byref(n)) == 0
    assert n.value == w * h * 3
    torch = pytest.importorskip("torch")

    class _DeviceFrame:
        __cuda_array_interface__ = {"shape": (n.value,), "typestr": "<f4", "data": (ptr.value, False), "version": 3}

    dev = torch.as_tensor(_DeviceFrame(), device="cuda:0").cpu().numpy().reshape(w, h, 3)
    assert_bit_identical(dev, want, "tcrt_device_frame")
    gpu_ctx.write_ppm(p, str(tmp_path / "a.ppm"))
    ppm = (tmp_path / "a.ppm").read_bytes()
    head = b"P6\n160 120\n255\n"
    assert ppm[:len(head)] == head
    assert np.array_equal(np.frombuffer(ppm[len(head):], np.uint8).reshape(h, w, 3), q8(want).transpose(1, 0, 2)[::-1])
    gpu_ctx.write_txt(p, str(tmp_path / "a.txt"))
    assert pixel_md5((tmp_path / "a.txt").read_bytes()) == pixel_md5(O.format_txt(want))
    gpu_ctx.write_bin(p, str(tmp_path / "a.bin"))
    raw = (tmp_path / "a.bin").read_bytes()
    assert_bit_identical(np.frombuffer(raw[32:], np.float32).reshape(w, h, 3), want, "write_bin")


@gpu
def test_adaptive_with_two_frames_in_flight(gpu_ctx):
    """As for the synchronous supersampled call: refused while the current frame set has an asynchronous frame pending,
    and the frames in flight are not disturbed by one in between."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    w, h = 240, 150
    p = api.default_params(w, h, 12)
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    full, _ = gpu_ctx.render_ss(p, 2)
    want, _ = expected(plain, full.copy(), 8)
    hbs = [api.HostBuffer(w * h * 12) for _ in range(2)]
    outs = [hb.array(np.float32, (w, h, 3)) for hb in hbs]
    t0 = gpu_ctx.render_async_ss(p, 2, 0, w, outs[0])
    got, _, _, _ = gpu_ctx.render_adaptive(p, 2, 8)            # one frame in flight, in the other set
    assert_bit_identical(got, want, "adaptive with one frame in flight")
    t1 = gpu_ctx.render_async(p, out=outs[1])
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.render_adaptive(p, 2, 8)
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    gpu_ctx.wait(t0)
    gpu_ctx.wait(t1)
    assert_bit_identical(outs[0], full, "ss frame in flight")
    assert_bit_identical(outs[1], plain, "plain frame in flight")
    del outs, hbs


@gpu
def test_adaptive_error_codes(gpu_ctx):
    lib = _ffi.load()
    fresh = api.Context([0])
    p = api.default_params(8, 8, 2)
    with pytest.raises(api.TcrtError) as e:
        fresh.render_adaptive(p, 2, 8)
    assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    scene, cam = make_scene("default")
    fresh.upload(scene, cam)
    plain, _ = fresh.render(p)
    plain = plain.copy()
    full, _ = fresh.render_ss(p, 2)
    want, _ = expected(plain, full.copy(), 0)
    st = _ffi.TcrtStats()
    n = C.c_ulonglong(7)
    buf = np.zeros(8 * 8 * 3, np.float32)
    buf8 = np.zeros(8 * 8 * 3, np.uint8)
    mask = np.zeros(8 * 8, np.uint8)
    fdst, bdst, mdst = buf.ctypes.data_as(C.c_void_p), buf8.ctypes.data_as(C.c_void_p), mask.ctypes.data_as(C.c_void_p)
    wide = api.default_params((1 << 24) // 2 + 1, 1, 0)             # ss * width = 2^24 + 2
    tall = api.default_params(1, (1 << 22) + 1, 0)                   # ss * height = 2^24 + 4 at ss = 4
    cases = [(p, 0, 8, _ffi.TCRT_ERR_INVALID), (p, -1, 8, _ffi.TCRT_ERR_INVALID), (p, 2, -2, _ffi.TCRT_ERR_INVALID),
             (p, 2, 256, _ffi.TCRT_ERR_INVALID), (p, 9, 8, _ffi.TCRT_ERR_UNSUPPORTED), (wide, 2, 8, _ffi.TCRT_ERR_UNSUPPORTED),
             (tall, 4, 8, _ffi.TCRT_ERR_UNSUPPORTED)]
    for q, ss, contrast, code in cases:
        for dst, mdst_ in ((fdst, mdst), (None, None)):
            assert lib.tcrt_render_columns_adaptive(fresh._h, C.byref(q), ss, contrast, 0, 1, dst, mdst_, C.byref(n),
                                                    C.byref(st)) == code, (ss, contrast, code)
        assert lib.tcrt_render_columns_adaptive_rgb8(fresh._h, C.byref(q), ss, contrast, 0, 1, bdst, mdst, C.byref(n),
                                                     C.byref(st)) == code, (ss, contrast, code)
    assert lib.tcrt_render_columns_adaptive_rgb8(fresh._h, C.byref(p), 2, 8, 0, 8, None, mdst, C.byref(n), C.byref(st)) == \
        _ffi.TCRT_ERR_INVALID
    for x0, x1 in ((3, 3), (5, 2), (-1, 4), (0, 9)):
        assert lib.tcrt_render_columns_adaptive(fresh._h, C.byref(p), 2, 8, x0, x1, fdst, mdst, C.byref(n), C.byref(st)) == \
            _ffi.TCRT_ERR_INVALID
    deep = api.default_params(8, 8, _ffi.TCRT_MAX_DEPTH + 1)
    assert lib.tcrt_render_columns_adaptive(fresh._h, C.byref(deep), 2, 8, 0, 8, fdst, mdst, C.byref(n), C.byref(st)) == \
        _ffi.TCRT_ERR_UNSUPPORTED
    assert (buf == 0).all() and (buf8 == 0).all() and (mask == 0).all() and n.value == 7
    got, _, _, _ = fresh.render_adaptive(p, 2, 0)
    assert_bit_identical(got, want, "after the refusals")
    fresh.close()


def _expected_cut(st_plain, width):
    """The cut a multi-device ctx derives from a whole plain frame's measured band times (tcrt_rebalance_columns)."""
    lib = _ffi.load()
    nb = st_plain.n_devices
    bounds = (C.c_int * (nb + 1))(*([b0 for b0, _ in st_plain.bands] + [width]))
    ms = (C.c_double * nb)(*st_plain.render_ms)
    out = (C.c_int * (nb + 1))()
    assert lib.tcrt_rebalance_columns(bounds, ms, nb, width, out) == 0
    return [(out[i], out[i + 1]) for i in range(nb)]


@gpu
@pytest.mark.parametrize("n_bands", [2, 3, 8])
def test_adaptive_multi_device(gpu_ctx, n_bands):
    """Band states on every visible GPU, device ids repeating when fewer are visible: equal-width bands, the single-device
    frame, and the balancer's cut untouched (the plain frame after an adaptive one is cut from the plain frame before it)."""
    n = api.device_count()
    devs = [i % n for i in range(n_bands)]
    scene, cam = make_scene("default")
    w, h, ss, contrast = 1920, 1080, 2, 8
    p = api.default_params(w, h, 5)
    gpu_ctx.upload(scene, cam)
    one, mask1, n1, st1 = gpu_ctx.render_adaptive(p, ss, contrast, mask=np.empty((w, h), np.uint8))
    one, mask1 = one.copy(), mask1.copy()
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    multi = api.Context(devs)
    multi.upload(scene, cam)
    _, st_p = multi.render(p)
    for kind in ("float pageable", "rgb8", "device"):
        if kind == "float pageable":
            got, mask, nn, st = multi.render_adaptive(p, ss, contrast, mask=np.empty((w, h), np.uint8))
            assert_bit_identical(got, one, f"{n_bands} bands")
            assert np.array_equal(mask, mask1)
        elif kind == "rgb8":
            got8, _, nn, st = multi.render_adaptive_rgb8(p, ss, contrast)
            assert_bytes_equal(got8, q8(one), f"{n_bands} bands RGB8")
        else:
            nn, st = multi.render_adaptive_device(p, ss, contrast)
            assert_bit_identical(multi.download(np.empty((w, h, 3), np.float32)), one, f"{n_bands} bands device-only")
        assert nn == n1 and st.n_devices == n_bands and st.rays_primary == sum(
            halo_columns(w, b0, b1) * h for b0, b1 in st.bands) + (ss * ss - 1) * n1
        assert st.bands == [(w * i // n_bands, w * (i + 1) // n_bands) for i in range(n_bands)]
    want_cut = _expected_cut(st_p, w)
    got, st_after = multi.render(p)
    assert st_after.bands == want_cut
    assert_bit_identical(got, plain, f"plain frame on {n_bands} bands after adaptive frames")
    multi.close()


CPP_PROGRAM = r"""
#include <stdio.h>
#include <vector>
#include "Camera.h"
#include "RayTracer.h"
#include "Scene.h"

int main() {
    using namespace CelioRayTracer;
    Scene scene;
    Camera camera;
    if (scene.initialize()) return 1;
    RenderSettings rs;
    rs.width = 100; rs.height = 76; rs.max_depth = 50; rs.samples = 4; rs.contrast = 8;
    if (raytrace_main(scene, camera, rs, "raytracer_screen.txt")) return 1;
    GpuRayTracer rt;
    std::vector<unsigned char> px((size_t)rs.width * rs.height * 3);
    tcrt_stats st;
    if (!rt.ok() || rt.setScene(scene, camera) || rt.renderRGB8(rs, px.data(), &st)) {
        fprintf(stderr, "%s\n", rt.lastError());
        return 1;
    }
    printf("%llu\n", st.rays_primary[0]);
    FILE* f = fopen("frame.rgb8", "wb");
    if (!f || fwrite(px.data(), 1, px.size(), f) != px.size()) return 1;
    return fclose(f) ? 1 : 0;
}
"""


@gpu
def test_cpp_render_settings_contrast(gpu_ctx, tmp_path):
    src = tmp_path / "render_adaptive.cpp"
    src.write_text(CPP_PROGRAM)
    libdir = os.path.join(ROOT, "tilecoderaytracer_b200")
    exe = tmp_path / "render_adaptive"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-ltcrt", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    p = api.default_params(100, 76, 50)
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    full, _ = gpu_ctx.render_ss(p, 4)
    want, want_mask = expected(plain, full.copy(), 8)
    assert int(r.stdout.split()[-1]) == 100 * 76 + 15 * int(want_mask.sum())   # the adaptive path, not render_ss
    txt = (tmp_path / "raytracer_screen.txt").read_bytes()
    lines = [ln for ln in txt.split(b"\n") if ln.startswith(b"(")]
    assert b"\n".join(lines) + b"\n" == O.format_txt(want)
    got8 = np.fromfile(tmp_path / "frame.rgb8", dtype=np.uint8).reshape(100, 76, 3)
    assert_bytes_equal(got8, q8(want), "GpuRayTracer::renderRGB8 with samples = 4, contrast = 8")
