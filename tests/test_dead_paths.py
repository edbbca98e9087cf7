"""Dead paths: the grid kernel stops shading a path's levels once every channel has met a zero object colour above them
(DESIGN.md §4.1c).  The frames and every ray counter stay the reference's: scenes whose paths die at the first level, the
second and deep down, -0.0 colours, a scene whose colours overflow (the zero then makes NaN, and pruning must be off),
depths 0, 1 and the cap, shadows and reflections off, adaptive and supersampled frames; the same scenes in a plane/BVH
form for the other render kernel."""
from __future__ import annotations

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import api

from _util import bits, make_scene

gpu = pytest.mark.gpu

# scenes where a colour the reference forms overflows: pruning must be off there
OVERFLOWING = ("overflow", "tiny_colours")

# exact 0/1 colours, so that neighbouring mirrors multiply every channel by zero within a bounce or two
PALETTE = [(1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 1, 1), (0, 0, 1), (1, 1, 1), (1, 0, 1)]


def _lights(s, case):
    if case == "tiny_colours":   # colours of 1e-12, intensities of 1e20: cosine * diffuse * intensity alone overflows
        for pos in ((-2, -6, 12), (8, 2, 10)):
            s.addSphere(pos, .15).setAsLightSource(1e20).setColor(1e-12, 1e-12, 1e-12)
        return
    s.addSphere((-2, -6, 12), .15).setAsLightSource(.75)
    s.addSphere((8, 2, 10), .15).setAsLightSource(1.0)


def _floor(s, case):
    light, dark, diffuse = (1, 1, 1), (0, 0, 0), .5
    if case == "neg_zero":
        dark = (-0.0, -0.0, -0.0)
    if case == "tiny_colours":
        light, diffuse = (1e-12, 1e-12, 1e-12), 1e20
    floor = s.addInfinitePlane((0, 0, 0), (0, 0, 1), (1, 0, 0))
    if case == "tiny_colours":
        floor.setColor(*light)
    floor.setCheckerBoard(light, dark, 3, 3).setReflectiveFactor(.5).setDiffuseFactor(diffuse)


def _color(case, i):
    c = PALETTE[i % len(PALETTE)]
    if case == "neg_zero":
        return tuple(-0.0 if v == 0 else float(v) for v in c)
    if case == "overflow":
        return tuple(2.0 * v for v in c)      # a mirror that doubles its child: 3e38 light -> inf, then a zero -> NaN
    if case == "tiny_colours":
        return tuple(1e-12 * v for v in c)
    return tuple(float(v) for v in c)


def dying_scene(case, kind):
    """kind "grid": a lattice of 108 mirror spheres (the sphere grid, render_grid_kernel); "planes": a mirror box of six
    finite planes around 12 mirror spheres (box clusters and a linear sweep, render_kernel)."""
    s = api.Scene()
    _lights(s, case)
    if case == "overflow":   # a large light that many mirrored rays meet: its colour times 3e38 overflows behind a mirror
        s.addSphere((2, 3, 40) if kind == "grid" else (2, 5, 11), 20 if kind == "grid" else 2.5).setAsLightSource(3e38)
    _floor(s, case)
    diffuse = 1e20 if case == "tiny_colours" else None
    n = 0
    if kind == "grid":
        for k in range(3):
            for j in range(6):
                for i in range(6):
                    s.addSphere((-3 + 1.8 * i, -1 + 1.8 * j, .8 + 1.8 * k), .75).setColor(*_color(case, n)) \
                        .setReflectiveFactor(1.0 if n % 5 else .6).setDiffuseFactor(diffuse or .3).setSpecularFactor(.4)
                    n += 1
    else:
        for face in s.makeSceneBox((-8, -6, 0), (20, 22, 14)):
            face.setColor(*_color(case, n)).setReflectiveFactor(.8).setDiffuseFactor(diffuse or .4)
            n += 1
        for i in range(12):
            s.addSphere((-2 + 1.7 * (i % 4), 1 + 2.0 * (i // 4), 1.5 + .4 * (i % 3)), .7).setColor(*_color(case, n)) \
                .setReflectiveFactor(1.0).setDiffuseFactor(diffuse or .3).setSpecularFactor(.4)
            n += 1
    return s


def _params(w, h, d, null=None, **kw):
    p = api.default_params(w, h, d, **kw)
    if null is not None:
        for k in range(3):
            p.null_color[k] = null
    return p


def assert_same_bits_or_both_nan(got, want, what):
    g, e = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert g.shape == e.shape, what
    nan_g, nan_e = np.isnan(g), np.isnan(e)
    assert np.array_equal(nan_g, nan_e), f"{what}: NaN at {int((nan_g != nan_e).sum())} channels of one side only"
    bad = int(((bits(g) != bits(e)) & ~nan_e).any(-1).sum())
    assert bad == 0, f"{what}: {bad} of {g.shape[0] * g.shape[1]} pixels differ bitwise"


def _check_counters(stats, cnt, what):
    assert (stats.rays_primary, stats.rays_shadow, stats.rays_reflect) == \
        (cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"]), what


# ---- the guard's decision, no device needed ------------------------------------------------------------------------------

def test_guard_prunes_the_flagship_scene():
    scene, _ = make_scene("synth256")
    flat = scene.flatten()
    assert api.plan_dead_paths(flat, _params(7680, 4320, 10))
    assert api.plan_dead_paths(flat, _params(64, 48, 254))            # the depth cap: tails grow linearly at k = 1
    assert api.plan_dead_paths(flat, _params(64, 48, 10, null=-0.0))


def test_guard_refuses_overflowing_and_non_finite_colours():
    for kind in ("grid", "planes"):
        for case in OVERFLOWING:
            s = dying_scene(case, kind)
            assert not api.plan_dead_paths(s.flatten(), _params(64, 48, 10)), (kind, case)
        s = dying_scene("primary", kind)
        assert api.plan_dead_paths(s.flatten(), _params(64, 48, 10)), kind
        assert not api.plan_dead_paths(s.flatten(), _params(64, 48, 10, null=float("inf"))), kind
        assert not api.plan_dead_paths(s.flatten(), _params(64, 48, 10, null=1e35)), kind
    s = dying_scene("primary", "grid")
    s.addSphere((30, 30, 30), .5).setColor(float("nan"), 0, 0)
    assert not api.plan_dead_paths(s.flatten(), _params(64, 48, 10))


@pytest.mark.parametrize("case", OVERFLOWING)
def test_overflow_scenes_make_nan_in_the_reference(case):
    """The overflowing cases are what they claim to be: the oracle's frame has NaN channels."""
    s = dying_scene(case, "grid")
    want, _ = O.render(s.flatten(), api.Camera().export(), _params(96, 64, 8))
    assert np.isnan(want).any()


def test_guard_refuses_bad_params():
    flat = dying_scene("primary", "grid").flatten()
    with pytest.raises(api.TcrtError):
        api.plan_dead_paths(flat, _params(64, 48, 10000))
    p = _params(64, 48, 10)
    p.max_depth = -1
    with pytest.raises(api.TcrtError):
        api.plan_dead_paths(flat, p)


# ---- frames and counters against the oracle ---------------------------------------------------------------------------------

CASES = [("primary", 112, 80, 10, {}), ("primary", 64, 48, 0, {}), ("primary", 64, 48, 1, {}), ("primary", 32, 24, 254, {}),
         ("primary", 96, 64, 8, {"shadows": False}), ("primary", 96, 64, 8, {"reflections": False}),
         ("neg_zero", 112, 80, 10, {}), ("neg_zero", 96, 64, 10, {"null": -0.0}), ("overflow", 96, 64, 8, {}),
         ("tiny_colours", 96, 64, 8, {})]


@gpu
@pytest.mark.parametrize("kind", ["grid", "planes"])
@pytest.mark.parametrize("case,w,h,d,kw", CASES)
def test_dying_paths_match_the_oracle(gpu_ctx, kind, case, w, h, d, kw):
    s, cam = dying_scene(case, kind), api.Camera()
    flat, c = s.flatten(), cam.export()
    p = _params(w, h, d, **kw)
    gpu_ctx.upload_flat(flat, c)
    structures = gpu_ctx.scene_structures()
    assert (structures["grid_cells"] > 0) == (kind == "grid"), structures
    assert api.plan_dead_paths(flat, p) == (case not in OVERFLOWING)
    img, stats = gpu_ctx.render(p)
    want, cnt = O.render(flat, c, p)
    what = f"{kind} {case} {w}x{h} d{d} {kw}"
    assert_same_bits_or_both_nan(img, want, what)
    _check_counters(stats, cnt, what)
    if case in OVERFLOWING:
        assert np.isnan(want).any(), what


@gpu
@pytest.mark.parametrize("kind", ["grid", "planes"])
def test_dying_paths_in_supersampled_and_adaptive_frames(gpu_ctx, kind):
    """ss = 2 frames (the band kernel at the sample size) and adaptive frames (the list kernel) of a dying scene."""
    s, cam = dying_scene("primary", kind), api.Camera()
    flat, c = s.flatten(), cam.export()
    ss, p = 2, _params(48, 32, 10)
    sp = _params(ss * p.width, ss * p.height, p.max_depth)
    gpu_ctx.upload_flat(flat, c)
    samples, cnt = O.render(flat, c, sp)
    acc = samples[0::ss, 0::ss].copy()
    for i in range(ss):
        for j in range(ss):
            if i or j:
                acc = acc + samples[i::ss, j::ss]
    want = acc / np.float32(ss * ss)
    got, st = gpu_ctx.render_ss(p, ss)
    assert_same_bits_or_both_nan(got, want, f"{kind} ss={ss}")
    _check_counters(st, cnt, f"{kind} ss={ss}")
    got, _, n, _ = gpu_ctx.render_adaptive(p, ss, -1)             # contrast -1 refines every pixel through the list kernel
    assert n == p.width * p.height
    assert_same_bits_or_both_nan(got, want, f"{kind} adaptive ss={ss}")
