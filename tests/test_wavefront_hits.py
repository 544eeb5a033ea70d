"""The hits of the render kernels, pixel by pixel.

Every rendered pixel takes its hits from two kernels of ptb_engine.cu: k_trace, the persistent-warp traversal (refill cursor,
postponed triangle groups, warp-quorum triangle phase), and k_exact, which finishes the rays k_trace could not decide (near-edge
hits, alpha-tested triangles, discs): it walks up to PTB_DEFER_K stored candidates and re-traces with traverse<> a ray that left more.
`check_ids` (parity_cases.py) measures `primary_ids`, which runs k_primary, a one-thread-per-ray kernel over the plain traverse<>:
none of the code above.  The image checks are too loose to see a bug that touches only the deferred rays (one in two hundred).

The probe: the denoiser-input render runs k_shade<..., AOV=true> on each sample's first hit, straight out of k_trace / k_exact, and
with the box filter `first_hit_normal` is the normalised sum of those first-hit shading normals.  Give every vertex its own random
normal and render at 1 spp: a pixel's first-hit normal then encodes both the triangle that was hit and the barycentrics of the hit,
and the oracle (oracle/port) computes the same output from the same seeded camera rays.

The scenes send most rays down the rare routes: a random soup (irregular leaves, many postponed groups, many near-edge rays), stacks
of N alpha-mapped sheets (one deferred candidate per sheet crossed: N = 4 fills PTB_DEFER_K, N = 5 and 8 force the re-trace), shadow
rays through such a stack (k_trace<ANY_HIT> deferral and k_exact<true, false>), the scheduling knobs of k_trace, and the device refit
(k_refit_tris / k_refit_level) against a fresh commit at the same pose.

The *_devsim tests run the same scenes and bounds through tests/devsim, which steps the device headers on the host with traverse<>
for every ray: it has no k_trace and no k_exact, so those tests check the scenes, their coverage claims and the tolerances, not the
kernels.  The knob sweep and the refit have no devsim variant (devsim ignores the options and does not refit).
"""
import numpy as np
import pytest
from parity_cases import check_ids, quad_mesh, triangle_soup

from pathtracer_b200 import _abi, scenes
from pathtracer_b200.api import Texture, TriMesh

PTB_DEFER_K = 4      # ptb_scene.h: candidates a ray can leave for k_exact before it is re-traced there

# check_first_hits, per pixel of first_hit_normal (largest component difference):
# (measured on a B200 at 1000 W, of 196,608 pixels: the soup 0 and 1 (5e-6), the refit 2 and 4 (2e-5); every stack 0)
FAR_PX = 1e-4        # > 1e-3: another triangle or other barycentrics
# (measured likewise: the soup 17 and 32 pixels (1.6e-4), the refit at 8x 145 (7.4e-4) and at 1/16 222 (1.1e-3); every stack 0)
NEAR_PX = 2e-3       # > 1e-4: rounding of the hit arithmetic


# ---- the probe ------------------------------------------------------------------------------------------------------
def cone_normals(n, rng, axis=(0, 1, 0), half_angle=0.8):
    """n random unit normals, uniform over the cap within `half_angle` of `axis`.  Every convex combination of them keeps a component
    of at least cos(half_angle) along the axis, so an interpolated normal never comes near zero and normalising it is well conditioned."""
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    t = np.cross(a, (1, 0, 0) if abs(a[0]) < 0.9 else (0, 1, 0))
    t /= np.linalg.norm(t)
    b = np.cross(a, t)
    z = 1 - rng.random(n) * (1 - np.cos(half_angle))
    phi = 2 * np.pi * rng.random(n)
    s = np.sqrt(1 - z * z)
    return ((s * np.cos(phi))[:, None] * t + (s * np.sin(phi))[:, None] * b + z[:, None] * a).astype(np.float32)


def first_hits(rt):
    """The denoiser inputs at the scene's spp: (first_hit_normal, imagedouble, stats)."""
    rt.render_denoiser_inputs()
    return rt.first_hit_normal.copy(), rt.imagedouble.copy(), dict(rt.stats)


def first_hit_errors(test, oracle):
    """(NaN patterns equal, share of pixels off by > 1e-3, share off by > 1e-4) between two first_hit_normal images."""
    fa, fb = np.isnan(test).any(-1), np.isnan(oracle).any(-1)
    e = np.abs(test - oracle).max(-1)
    e[fa | fb] = 0
    return bool(np.array_equal(fa, fb)), float(np.mean(e > 1e-3)), float(np.mean(e > 1e-4))


def check_first_hits(test, oracle, far=FAR_PX, near=NEAR_PX):
    same_nan, f3, f4 = first_hit_errors(test, oracle)
    assert same_nan, "the pixels without a first-hit normal differ"
    assert f3 <= far, f"{f3:.2e} of the pixels have another first hit (normal off by > 1e-3; bound {far})"
    assert f4 <= near, f"{f4:.2e} of the pixels have a first-hit normal off by > 1e-4 (bound {near})"


def compare_render(test_lib, oracle_lib, mk, need_mesh=True):
    """Commit `mk(lib)` on both sides, compare the first hits of the render, the sample counts and the k_primary ids."""
    a, b = mk(oracle_lib).commit(), mk(test_lib).commit()
    na, ia, sa = first_hits(a)
    nb, ib, sb = first_hits(b)
    check_first_hits(nb, na)
    assert sb["samples"] == sa["samples"] == a.W * a.H * a.nrays
    check_ids(b, a, need_mesh=need_mesh)
    return a, b, (na, ia, sa), (nb, ib, sb)


# ---- scenes ---------------------------------------------------------------------------------------------------------
def soup_mesh(n, seed=11, half_angle=0.8):
    """triangle_soup (n unconnected triangles of very different sizes) with a random normal per vertex"""
    v, _, uv, tri = triangle_soup(n, seed)
    return TriMesh(v, cone_normals(len(v), np.random.default_rng(seed + 1), half_angle=half_angle), uv, tri)


def soup_scene(L, W=512, H=384, spp=1, n=100000, view=0):
    rt = scenes.base(L, W, H, spp)
    m = scenes._place_like_gui(soup_mesh(n), scale=22.0)
    m.set_material(0, **scenes.phong((.6, .5, .4), 0.1, 20.0))
    rt.s.addObject(m)
    if view == 1:            # the second view point of case_triangle_soup: from above and the side, through the whole soup
        rt.cam.position = np.array([25, 10, -30], np.float32)
        d = np.array([-0.55, -0.45, 0.7], np.float32)
        rt.cam.direction = d / np.float32(np.linalg.norm(d))
        rt.cam.up = np.array([0, 1, 0], np.float32)
    return rt


SHEET_QUADS, SHEET_TEX = 16, 128      # 512 triangles per sheet; a triangle covers about 32 texels of its alpha map


def sheet(seed, clear=0.6, opaque=False):
    """A wavy sheet (quad_mesh, flattened) with random per-vertex normals and an alpha map of random texels, `clear` of them holes.
    Every sheet draws its own map, so the holes of two sheets do not line up."""
    rng = np.random.default_rng(1000 + seed)
    v, _, uv, tri = quad_mesh(SHEET_QUADS)
    v[:, 1] *= 0.15
    m = TriMesh(v, cone_normals(len(v), rng), uv, tri)
    alpha = np.repeat((rng.random((SHEET_TEX, SHEET_TEX)) >= clear).astype(np.float32)[..., None], 3, -1)
    mat = scenes.phong((.3 + .07 * (seed % 8), .5, .8 - .07 * (seed % 8)), 0.0, 1.0)
    if not opaque:
        mat["alpha"] = Texture(1.0, alpha)
    m.set_material(0, **mat)
    m.alpha_map = alpha
    return m


def straddles(m):
    """Whether every triangle of sheet `m` reads both opaque and clear texels (nearest texel (int)(u * (W - 1)), as alpha_rejects
    reads it; the rows in either order).  Otherwise the commit-time classification (scene_host.cpp) makes it plainly opaque or leaves
    it out, and it is never deferred."""
    a = m.alpha_map[..., 0] >= 0.5
    g = np.linspace(0.02, 0.98, 12)
    b1, b2 = np.meshgrid(g, g)
    keep = b1 + b2 <= 0.98
    b1, b2 = b1[keep], b2[keep]
    uv = m.uvs[m.tri[:, 3:6]]                                                     # (n, 3, 2)
    p = uv[:, :1] * (1 - b1 - b2)[None, :, None] + uv[:, 1:2] * b1[None, :, None] + uv[:, 2:3] * b2[None, :, None]
    i = (p * (SHEET_TEX - 1)).astype(np.int64)
    ok = True
    for rows in (i[..., 1], SHEET_TEX - 1 - i[..., 1]):
        s = a[rows, i[..., 0]]
        ok &= bool((s.any(1) & ~s.all(1)).all())
    return ok


def stack_scene(L, n_sheets, W=256, H=192, spp=1, only=None, opaque=False, soup=0):
    """n_sheets alpha-mapped sheets facing the camera one behind the other, 8 units apart, each with its own small tilt; the dome
    (or, with `soup`, a random soup) behind them.  `only=k` keeps sheet k alone (and `opaque` drops the alpha maps): the coverage
    probes of sheet_crossings."""
    rt = scenes.base(L, W, H, spp)
    rt.cam.position = np.array([0, 60, 70], np.float32)
    rt.cam.direction = np.array([0, 0, -1], np.float32)
    rt.cam.up = np.array([0, 1, 0], np.float32)
    rt.cam.aperture = np.float32(0.0)
    for k in range(n_sheets):
        m = sheet(k, opaque=opaque)
        m.scale = 110.0
        m.mat_rotation = scenes._rot(np.pi / 2 + 0.05 * np.sin(2.1 * k + 1), 0.05 * np.cos(1.7 * k))
        m.max_translation = np.array([0, 60, -8 * k], np.float32)
        if only is None or only == k:
            rt.s.addObject(m)
    if soup:
        s = soup_mesh(soup, seed=5)
        s.set_material(0, **scenes.phong((.6, .5, .4), 0.1, 20.0))
        s.scale, s.max_translation = 70.0, np.array([0, 60, -80], np.float32)
        rt.s.addObject(s)
    return rt


def sheet_crossings(oracle_lib, n_sheets, **kw):
    """Per pixel, how many sheets the camera ray crosses: each sheet alone and opaque, through the oracle's primary_ids.  (Nothing
    opaque stands in front of the stack, so every crossing is a candidate that k_trace leaves for k_exact.)"""
    n = 0
    for k in range(n_sheets):
        rt = stack_scene(oracle_lib, n_sheets, only=k, opaque=True, **kw).commit()
        n = n + (rt.primary_ids()[0] == 3)
        rt.close()
    return n


def check_stack_coverage(a, oracle_lib, n_sheets, **kw):
    """The stack scene does what it is for: every triangle of every sheet straddles opaque and clear texels (so the commit keeps it
    and alpha-tests it), and most camera rays leave exactly N candidates (N <= PTB_DEFER_K) or more than PTB_DEFER_K (N >= 5);
    their first hits spread over the sheets."""
    assert a.scene_info()["n_triangles"] == n_sheets * 2 * SHEET_QUADS ** 2
    assert all(straddles(sheet(k)) for k in range(n_sheets))
    cross = sheet_crossings(oracle_lib, n_sheets, **kw)
    if n_sheets <= PTB_DEFER_K:
        assert (cross == n_sheets).mean() > 0.95, (cross == n_sheets).mean()
    else:
        assert (cross > PTB_DEFER_K).mean() > 0.95, (cross > PTB_DEFER_K).mean()
    obj = a.primary_ids()[0]
    for k in range(n_sheets):   # (holes are 60 % of each map: sheet k takes about 0.4 * 0.6^k of the pixels)
        assert (obj == 3 + k).mean() > 0.4 * 0.6 ** k / 3, (k, (obj == 3 + k).mean())


def shadow_stack_scene(L, n_sheets, W=256, H=192, only=None, opaque=False):
    """The stack laid flat between the floor and the light (the sphere at y = 13..33), nb_bounces = 1: at 1 spp a pixel's radiance
    is its direct term alone, so it shows whether its one shadow ray got through every sheet.  The camera sits under the stack and
    looks down at the floor."""
    rt = scenes.base(L, W, H, 1, depth=1)
    rt.cam.position = np.array([0, -12, 50], np.float32)
    d = np.array([0, -0.45, -1], np.float32)
    rt.cam.direction = d / np.float32(np.linalg.norm(d))
    rt.cam.up = np.array([0, 1, 0], np.float32)
    rt.cam.aperture = np.float32(0.0)
    for k in range(n_sheets):
        m = sheet(k, clear=0.7, opaque=opaque)
        m.scale = 130.0
        m.mat_rotation = scenes._rot(0.01 * np.sin(2.1 * k + 1), 0.3 * k)
        m.max_translation = np.array([0, -8 + 2.5 * k, -5], np.float32)
        if only is None or only == k:
            rt.s.addObject(m)
    return rt


# ---- 1/2: the soup and the stacks against the oracle ------------------------------------------------------------------
def case_soup(test_lib, oracle_lib, W=512, H=384):
    for view in (0, 1):
        a, b, _, _ = compare_render(test_lib, oracle_lib, lambda L: soup_scene(L, W, H, view=view))
        assert b.scene_info()["n_triangles"] == 100000
        assert (a.primary_ids()[0] == 3).mean() > 0.3, "the soup must fill much of the view"
        a.close(); b.close()


def case_alpha_stack(test_lib, oracle_lib, n_sheets):
    a, b, _, _ = compare_render(test_lib, oracle_lib, lambda L: stack_scene(L, n_sheets))
    check_stack_coverage(a, oracle_lib, n_sheets)
    a.close(); b.close()


# pixels whose first hits agree but whose direct term differs by > 1e-4 relative (measured on a B200 at 1000 W: 2 of 49,152 at
# N = 5, 0 at N = 8; no pixel is lit on one side and shadowed on the other)
ANYHIT_PX = 2e-4


def case_anyhit_stack(test_lib, oracle_lib, n_sheets):
    a, b, (na, ia, _), (nb, ib, _) = compare_render(test_lib, oracle_lib, lambda L: shadow_stack_scene(L, n_sheets), need_mesh=False)
    floor = a.primary_ids()[0] == 2
    assert floor.mean() > 0.5, "the camera must see the floor under the stack"
    # every shadow ray from the floor crosses every sheet: each sheet alone and opaque shadows the whole floor in view
    for k in range(n_sheets):
        one = shadow_stack_scene(oracle_lib, n_sheets, only=k, opaque=True).commit()
        img = one.render_image_nopreviz()
        assert (img.max(-1)[::-1][floor] == 0).all(), f"sheet {k} leaves floor pixels lit"
        one.close()
    # the first hits agree: so must the direct terms (whether the shadow ray got through)
    same = np.abs(na - nb).max(-1) <= 1e-4
    rel = np.abs(ia - ib).max(-1) / np.maximum(np.abs(ia).max(-1), 1e-30)
    rel[(ia.max(-1) == 0) & (ib.max(-1) == 0)] = 0
    bad = float(np.mean(same & (rel > 1e-4)))
    assert bad <= ANYHIT_PX, f"{bad:.2e} of the pixels with the same first hit differ in their direct term (bound {ANYHIT_PX})"
    lit = (ia.max(-1) > 0)[::-1][floor]
    assert 0.02 < lit.mean() < 0.5, f"{lit.mean():.3f} of the floor pixels see the light: the stack must block most shadow rays, not all"
    a.close(); b.close()


def test_soup_devsim(devsim, port):
    case_soup(devsim, port)


@pytest.mark.gpu
def test_soup_gpu(gpu, port):
    case_soup(gpu, port)


@pytest.mark.parametrize("n_sheets", [3, 4, 5, 8])
def test_alpha_stack_devsim(devsim, port, n_sheets):
    case_alpha_stack(devsim, port, n_sheets)


@pytest.mark.gpu
@pytest.mark.parametrize("n_sheets", [3, 4, 5, 8])
def test_alpha_stack_gpu(gpu, port, n_sheets):
    case_alpha_stack(gpu, port, n_sheets)


@pytest.mark.parametrize("n_sheets", [5, 8])
def test_anyhit_through_the_stack_devsim(devsim, port, n_sheets):
    case_anyhit_stack(devsim, port, n_sheets)


@pytest.mark.gpu
@pytest.mark.parametrize("n_sheets", [5, 8])
def test_anyhit_through_the_stack_gpu(gpu, port, n_sheets):
    case_anyhit_stack(gpu, port, n_sheets)


# ---- 3: the scheduling knobs of k_trace cannot change a hit -------------------------------------------------------------
# Every setting runs on a fresh context, so no setting outlives its render.  PTB_OPT_PIPES = 1 throughout: with more than one
# pipeline, passes on different streams add into the frame in varying order.  With one pipeline and the box filter the order of the
# adds does not depend on the scheduling, so a changed pixel is a changed hit.  The only hit that may depend on the scheduling is an
# exact tie in t, which k_exact resolves in the order the candidates were deferred.  The extremes TRI_MIN_PCT = 100 and
# REFILL_BELOW = 1 cannot stall a warp: once none of its live lanes has node work left, they all hold triangles and meet the
# quorum (k_trace, ptb_engine.cu).
KNOBS = ([(_abi.OPT_REFILL_BELOW, v) for v in (1, 2, 32, 33)] + [(_abi.OPT_TRI_FRACTION, v) for v in (1, 2, 64)]
         + [(_abi.OPT_TRI_MIN_PCT, v) for v in (0, 50, 100)] + [(_abi.OPT_TRACE_BLOCKS, v) for v in (1, 3)]
         + [(_abi.OPT_COUNT_TRAVERSAL, 1), (_abi.OPT_POOL_PATHS, 4096)])
KNOB_PX = 1e-4       # pixels not bit-equal to the default render (measured on a B200 at 1000 W: 0 for every setting)
KNOB_SHEETS, KNOB_SOUP = 5, 30000


def knob_scene(L):
    """the 5-sheet stack in front of a 30,000-triangle soup with random per-vertex normals, 256x192 at 4 spp"""
    return stack_scene(L, KNOB_SHEETS, spp=4, soup=KNOB_SOUP)


def knob_render(gpu, option=None, value=None):
    rt = knob_scene(gpu).commit()
    rt.set_option(_abi.OPT_PIPES, 1)
    if option is not None:
        rt.set_option(option, value)
    out = first_hits(rt)
    rt.close()
    return out


def knob_differences(ref, got):
    """pixels of (first_hit_normal, imagedouble) that are not bit-equal"""
    both_nan = (np.isnan(ref[0]) & np.isnan(got[0])).all(-1)
    return ((ref[0] != got[0]).any(-1) & ~both_nan) | (ref[1] != got[1]).any(-1)


@pytest.mark.gpu
def test_scheduling_knobs_do_not_change_a_hit_gpu(gpu):
    rt = knob_scene(gpu).commit()
    assert rt.scene_info()["n_triangles"] == KNOB_SHEETS * 2 * SHEET_QUADS ** 2 + KNOB_SOUP
    obj = rt.primary_ids()[0]
    assert (obj == 3 + KNOB_SHEETS).mean() > 0.02 and all((obj == 3 + k).mean() > 0.01 for k in range(KNOB_SHEETS)), "sheets and soup in view"
    rt.close()
    ref = knob_render(gpu)
    assert ref[2]["samples"] == 256 * 192 * 4
    for option, value in KNOBS:
        got = knob_render(gpu, option, value)
        for k in ("samples", "rays_closest", "rays_shadow"):
            assert got[2][k] == ref[2][k], (option, value, k)
        diff = knob_differences(ref, got)
        assert diff.mean() <= KNOB_PX, f"option {option} = {value}: {int(diff.sum())} pixels differ from the default render"


# ---- 4: the device refit against a fresh commit at the same pose -----------------------------------------------------
REFIT_TRIS = 50000


def refit_scene(L, frame, small=False, W=512, H=384):
    """A soup with random per-vertex normals keyed from a pose at frame 0 to a pose at frame 10 that is rotated far and 8x the size
    a few hundred units away, or 1/16 the size a few of its own sizes away (there the quantisation slack of the node boxes,
    node_coord_slack + 4e-3 cell, is largest against the triangles); the camera looks at the frame-10 pose.  The normals keep to a
    narrower cone than elsewhere: far from the origin the barycentrics of the two implementations differ by more, and a narrow
    cone keeps that below the bounds of check_first_hits while another triangle still moves the normal by far more than 1e-3."""
    rt = scenes.base(L, W, H, 1)
    m = soup_mesh(REFIT_TRIS, seed=23, half_angle=0.3)
    m.set_material(0, **scenes.phong((.6, .5, .4), 0.1, 20.0))
    s0 = 4.0
    m.scale, m.max_translation = s0, np.array([0, -20, 0], np.float32)
    m.add_keyframe(0)
    s1 = s0 / 16 if small else 8 * s0
    T = np.array([2.0, 1.5, -2.5] if small else [260, 140, -310], np.float32)
    m.scale, m.mat_rotation, m.max_translation = s1, scenes._rot(1.1, 2.3), T
    m.add_keyframe(10)
    rt.s.addObject(m)
    rt.s.current_frame = frame
    pos = T + np.float32(s1) * np.array([0.3, 0.4, 1.6], np.float32)
    d = T - pos
    rt.cam.position, rt.cam.direction = pos, d / np.float32(np.linalg.norm(d))
    rt.cam.up = np.array([0, 1, 0], np.float32)
    return rt


REFIT_AGREE = 0.99999     # (measured on a B200 at 1000 W: first hits and ids identical on every pixel at both poses)


def refit_against_fresh(gpu, port, small):
    """(refit first hits, fresh first hits, oracle first hits, refit ids, fresh ids)"""
    rt = refit_scene(gpu, 0, small).commit()
    rt.render_image_nopreviz()
    rt.set_frame(10)
    got = first_hits(rt)
    assert rt.scene_info()["ms_refit"] > 0, "the re-pose ran on the device"
    fresh = refit_scene(gpu, 10, small).commit()
    want = first_hits(fresh)
    ora = refit_scene(port, 10, small).commit()
    return rt, fresh, ora, got, want, first_hits(ora)


@pytest.mark.gpu
@pytest.mark.parametrize("small", [False, True], ids=["x8", "x1_16"])
def test_refit_equals_a_fresh_commit_gpu(gpu, port, small):
    rt, fresh, ora, got, want, oracle = refit_against_fresh(gpu, port, small)
    assert (ora.primary_ids()[0] == 3).mean() > 0.3, "the re-posed soup must fill much of the view"
    same = ((got[0] == want[0]) | (np.isnan(got[0]) & np.isnan(want[0]))).all(-1)
    assert same.mean() >= REFIT_AGREE, f"first hits identical on {same.mean():.6f} of the pixels"
    oa, ta, _ = fresh.primary_ids()
    ob, tb, _ = rt.primary_ids()
    ids = (oa == ob) & (ta == tb)
    assert ids.mean() >= REFIT_AGREE, f"primary ids identical on {ids.mean():.6f} of the pixels"
    check_first_hits(got[0], oracle[0])
    assert got[2]["samples"] == oracle[2]["samples"]
