"""Parity cases shared by the CPU suite (tests/devsim: the device headers host-compiled) and the GPU suite
(the real kernels through the C-ABI).  Each case renders the same seeded scene with the implementation under
test and with the oracle and states its tolerance next to the assertion.

Tolerances (float32 paths; the oracle and the CUDA path draw the same pcg32 numbers per (pixel,sample)):
  ID_AGREE      primary-hit (object, triangle) ids agree on >= 99.99 % of pixels (BASELINE.json north_star)
  FRAC_1SPP     at equal seed and spp at most 0.5 % of pixels differ by more than 1e-3 relative
                (a path changes when a rounding difference flips a branch: lobe choice, Fresnel choice, edge hit)
  MEAN_REL      image means agree within 0.2 %
  RRMSE_FACTOR  relRMSE(test_N, oracle_hi) <= 1.1 * relRMSE(oracle_N, oracle_hi) + 0.005  (converged-image bound)
"""
import numpy as np

from pathtracer_b200 import _abi, scenes
from pathtracer_b200.api import Plane, Sphere, Texture, TriMesh, Yarns

ID_AGREE = 0.9999
FRAC_1SPP = 0.005
MEAN_REL = 2e-3
RRMSE_FACTOR = 1.1


def rel_err(a, b):
    return np.abs(a - b).max(-1) / np.maximum(np.abs(a).max(-1), 1e-3 * float(np.abs(a).mean()) + 1e-30)


def rrmse(a, ref):
    return float(np.sqrt(np.mean((a - ref) ** 2)) / np.mean(ref))


def check_images(img, ref, frac=FRAC_1SPP, mean_rel=MEAN_REL):
    assert np.isfinite(img).all()
    e = rel_err(ref, img)
    bad = float(np.mean(e > 1e-3))
    assert bad <= frac, f"{bad:.5f} of pixels differ by > 1e-3 relative (bound {frac})"
    assert abs(float(img.mean()) / float(ref.mean()) - 1) <= mean_rel


def check_ids(rt_test, rt_oracle, W=None, H=None, agree=ID_AGREE, need_mesh=True):
    oa, ta, da = rt_oracle.primary_ids(W, H)
    ob, tb, db = rt_test.primary_ids(W, H)
    same = (oa == ob) & (ta == tb)
    assert same.mean() >= agree, f"primary-hit ids agree on {same.mean():.6f} of pixels (need {agree})"
    if need_mesh:
        assert (ta >= 0).mean() > 0.05, "the test scene must actually show the mesh"
    hit = same & (oa >= 0)
    assert np.allclose(da[hit], db[hit], rtol=2e-4), "hit distances"


def case_scene(test_lib, oracle_lib, mk, nrays=None, frac=FRAC_1SPP, agree=ID_AGREE):
    a, b = mk(oracle_lib).commit(), mk(test_lib).commit()
    if nrays:
        a.nrays = b.nrays = nrays
    check_ids(b, a, agree=agree, need_mesh=len(a.s.objects) > 5 or any(hasattr(o, "tri") for o in a.s.objects))
    ia, ib = a.render_image_nopreviz().copy(), b.render_image_nopreviz().copy()
    check_images(ib, ia, frac)
    assert np.allclose(a.sample_count, b.sample_count, rtol=1e-5)
    # ray counters: identical paths except where a branch flipped
    for k in ("rays_closest", "rays_shadow"):
        assert abs(a.stats[k] - b.stats[k]) <= 0.002 * a.stats[k] + 8, k
    assert b.stats["samples"] == a.stats["samples"]
    d = np.abs(a.image.astype(int) - b.image.astype(int))
    assert np.mean(d > 1) <= 2 * frac
    a.close(); b.close()


def yarn_inside_scene(lib, W=64, H=64, spp=2):
    """A fat yarn segment seen by a camera that sits between the tube and the prism that covers it in the BVH8, inside a small sphere:
    every primary ray meets the tube (t = 0.1 .. 0.5) before the sphere's inner side (t = 1) and leaves the covering prism only
    beyond it (t > 4).  The covering faces must therefore not be cut at the nearest hit so far (their e2.w = 0, ptb_scene.h)."""
    rt = scenes.base(lib, W, H, spp)
    rt.s.addObject(Sphere((0, 0, 2.1), 1.0).set_material(0, **scenes.phong((.3, .8, .3), 0.3, 50.0)))
    # (the third segment has no length: its axis is 0 / 0 and Cylinder::intersection answers t = NaN, which never wins `localt < t`;
    #  the fourth has no radius: the reference can only graze its axis; both must stay harmless on every side)
    rt.s.addObject(Yarns([[-10, 0, 0], [-4, 0.5, -6], [1, 1, -3], [-2, -1, -4]], [[10, 0, 0], [-3, 2, -9], [1, 1, -3], [2, -1, -4]], [2.0, 0.7, 0.5, 0.0]))
    rt.cam.position = np.array([0, 0, 2.1], np.float32)
    rt.cam.direction = np.array([0, 0, -1], np.float32)
    rt.cam.up = np.array([0, 1, 0], np.float32)
    rt.cam.aperture = np.float32(0.0)
    return rt


def case_yarn_from_inside(test_lib, oracle_lib):
    a, b = yarn_inside_scene(oracle_lib).commit(), yarn_inside_scene(test_lib).commit()
    oa, ta, da = a.primary_ids()
    assert (oa == 4).mean() > 0.9 and (ta[oa == 4] == 0).all() and da[oa == 4].max() < 0.9, "the scene must show the tube in front of the sphere"
    check_ids(b, a, need_mesh=False)
    check_images(b.render_image_nopreviz().copy(), a.render_image_nopreviz().copy())
    a.close(); b.close()


def yarn_cloth_scene(lib, W=512, H=512, spp=1, n=120, seg=300, radius=0.003):
    """A cloth of 2 n yarns x `seg` segments (72,000 by default) of the reference's own proportions (its reader gives radius 0.1 to
    curves of extent 50: 2e-3; here 0.12 at distance 50).  Thinner yarns are not a parity case: `delta = b*b - 4*a*c` of
    Cylinder::intersection cancels log10((distance / radius)^2) digits, so within a few per cent of a thin tube's silhouette the
    REFERENCE's answer is rounding noise that its own tight boxes then cull or keep (measured: 99.998 % of the primary ids agree
    at radius 0.18, 99.994 % at 0.12, 99.97 % at 0.064)."""
    rt = scenes.base(lib, W, H, spp)
    y = Yarns(*scenes.weave_segments(n, n, seg, radius=radius))
    y.scale, y.mat_rotation, y.max_translation = 40.0, scenes._rot(1.0, 0.4), np.array([0, -14, 0], np.float32)
    rt.s.addObject(y)
    return rt


def case_yarn_cloth(test_lib, oracle_lib, W=512, H=512):
    a, b = yarn_cloth_scene(oracle_lib, W, H).commit(), yarn_cloth_scene(test_lib, W, H).commit()
    assert (a.primary_ids()[0] == 3).mean() > 0.5, "the cloth must fill the view"
    check_ids(b, a, need_mesh=False)
    # direct light only: camera rays are bit-identical on both sides, so the usual equal-seed bound holds (measured 0.15 % on the GPU)
    a.nb_bounces = b.nb_bounces = 1
    check_images(b.render_image_nopreviz().copy(), a.render_image_nopreviz().copy())
    # full depth: a bounced ray differs in its last bits between the two implementations, and for such a ray the REFERENCE's
    # hit-or-miss near the silhouette of a far, thin tube is a coin toss (the docstring above); the flips are unbiased, so the image
    # means and the ray counters still agree closely while single pixels do not (measured on the GPU, profiles/r02ae_yarn_cloth.txt:
    # 1.7 % of the pixels off by more than 1e-3 at radius 0.12, 1.0 % at 0.18, 0.4 % at 0.36, 0.13 % at 0.8; means within 5e-5)
    a.nb_bounces = b.nb_bounces = 5
    check_images(b.render_image_nopreviz().copy(), a.render_image_nopreviz().copy(), frac=0.05, mean_rel=5e-4)
    for k in ("rays_closest", "rays_shadow"):
        assert abs(a.stats[k] - b.stats[k]) <= 0.001 * a.stats[k], k
    a.close(); b.close()


def case_branch_scene(test_lib, oracle_lib, mk, frac=FRAC_1SPP, gold=None):
    """getColor's branching modes (fog, ghost objects, background photograph).  Same per-contribution pcg32 streams on both
    sides (oracle/build_ref.py patch 7), so the images are compared at equal seed like the linear scenes.  Ray counters are
    NOT equal by construction: the reference traces the in-scattering ray of fogContribution twice (once for its visibility,
    once when the contribution is popped) where the wavefront traces it once, and a ghost's straight-through ray is traced
    before its shadow ray can cancel it; they are only bracketed."""
    a, b = mk(oracle_lib).commit(), mk(test_lib).commit()
    check_ids(b, a, agree=0.998, need_mesh=any(hasattr(o, "tri") for o in a.s.objects))     # 2304 pixels of a coarse mesh: a few silhouette pixels may flip (99.99 % is checked at 512x512)
    ia, ib = a.render_image_nopreviz().copy(), b.render_image_nopreviz().copy()
    check_images(ib, ia, frac)
    if gold is not None:
        check_images(ib, gold["imagedouble"], max(frac, 0.01))
    assert np.allclose(a.sample_count, b.sample_count, rtol=1e-5)
    assert b.stats["samples"] == a.stats["samples"]
    assert abs(a.stats["rays_shadow"] - b.stats["rays_shadow"]) <= 0.01 * a.stats["rays_shadow"] + 8
    assert 0.5 * a.stats["rays_closest"] <= b.stats["rays_closest"] <= 1.2 * a.stats["rays_closest"]
    assert np.mean(np.abs(a.image.astype(int) - b.image.astype(int)) > 1) <= 2 * frac
    a.close(); b.close()


def case_branch_converged(test_lib, oracle_lib):
    """Fog at equal spp against a high-spp oracle image (the converged-image bound of the north star).  The medium is a
    high-variance estimator (relRMSE of a 16-spp image is > 1), so the bound is stated at equal seed like case_converged."""
    mk = lambda L: scenes.config_fog(L, 32, 32, 16, fog_type=1, phase=1)
    hi = mk(oracle_lib).commit()
    hi.nrays, hi.seed = 768, 99
    ref_hi = hi.render_image_nopreviz().copy()
    a, b = mk(oracle_lib).commit(), mk(test_lib).commit()
    ia, ib = a.render_image_nopreviz().copy(), b.render_image_nopreviz().copy()
    ea, eb = rrmse(ia, ref_hi), rrmse(ib, ref_hi)
    assert eb <= RRMSE_FACTOR * ea + 0.005, (ea, eb)
    # equal seed: nearly the same image.  A pixel sums 16 samples x up to 31 contributions, and one flipped firefly moves an
    # RMSE a lot, so this is stated per pixel: at most 3 % of the pixels differ by more than 1e-3 relative
    assert float(np.mean(rel_err(ia, ib) > 1e-3)) <= 0.03


def case_sss_converged(test_lib, oracle_lib, spp=64, mk=None):
    """Subsurface scattering.  The reference picks the re-emergence point by reservoir sampling over the hits of a probe ray,
    one draw per hit in the traversal order of ITS binary BVH; a different BVH meets the hits in another order, so the two
    sides cannot draw the same numbers and the comparison is the north star's converged-image bound: at equal spp the test
    image is as close to a high-spp oracle image as the oracle's own image of that spp, and the means agree within 2 %.
    `mk(lib)`: another subsurface scene (default: config_sss at 40 x 40, `spp`)."""
    mk = mk or (lambda L: scenes.config_sss(L, 40, 40, spp))
    hi = mk(oracle_lib).commit()
    hi.nrays, hi.seed = 1024, 99
    ref_hi = hi.render_image_nopreviz().copy()
    a, b = mk(oracle_lib).commit(), mk(test_lib).commit()
    check_ids(b, a, agree=0.998)
    ia, ib = a.render_image_nopreviz().copy(), b.render_image_nopreviz().copy()
    assert np.isfinite(ib).all() and (ib >= 0).all()
    ea, eb = rrmse(ia, ref_hi), rrmse(ib, ref_hi)
    assert eb <= 1.15 * ea + 0.01, (ea, eb)
    assert abs(float(ib.mean()) / float(ref_hi.mean()) - 1) < 0.02
    # the branch must actually be exercised: without Ksub the image is a different one
    plain = mk(test_lib)
    for o in plain.s.objects:
        for slots in o.materials.values():
            slots.pop("Ksub", None)
    ip = plain.commit().render_image_nopreviz()
    assert rrmse(ip, ref_hi) > 2 * eb
    assert abs(b.stats["rays_closest"] / a.stats["rays_closest"] - 1) < 0.02


def case_branch_passes(test_lib):
    """Splitting a branching render into passes (small contribution pool) must not change the image; an exhausted pool is an error."""
    mk = lambda: scenes.config_fog(test_lib, 40, 24, 3, fog_type=0, phase=2).commit()
    whole, small = mk(), mk()
    ref = whole.render_image_nopreviz().copy()
    small.set_option(_abi.OPT_POOL_PATHS, 40 * 24 * 32)   # 32 slots per sample at depth 5: one sample per pass
    img = small.render_image_nopreviz()
    assert np.allclose(img, ref, rtol=2e-5, atol=1e-3)
    assert small.stats["rays_closest"] == whole.stats["rays_closest"]
    g = scenes.config_ghost(test_lib, 40, 24, 3).commit()
    gi = g.render_image_nopreviz().copy()
    g.set_option(_abi.OPT_POOL_PATHS, 1024)
    assert np.allclose(g.render_image_nopreviz(), gi, rtol=2e-5, atol=1e-3)
    s1, s2 = scenes.config_sss(test_lib, 40, 24, 3).commit(), scenes.config_sss(test_lib, 40, 24, 3).commit()
    si = s1.render_image_nopreviz().copy()
    s2.set_option(_abi.OPT_POOL_PATHS, 1024)
    assert np.allclose(s2.render_image_nopreviz(), si, rtol=2e-5, atol=1e-3), "subsurface probes draw from per-contribution streams: pass splitting cannot matter"


def case_branch_errors(test_lib):
    rt = scenes.config_C1(test_lib, 8, 8, 1)
    rt.s.objects[3].set_material(0, Ksub=Texture((.5, .4, .3)))
    try:
        rt.commit(); raised = False
    except _abi.PtbError:
        raised = True
    assert raised, "subsurface scattering is refused, not approximated"
    rt = scenes.config_C1(test_lib, 8, 8, 1)
    rt.s.objects[3].set_material(0, Ksub=Texture((0, 0, 0)))     # the reference default: accepted
    rt.commit(); rt.close()
    rt = scenes.base(test_lib, 8, 8, 1)
    rt.s.objects.pop()                                            # no object 2: the medium has no ground level
    rt.s.fog_density = 0.2
    try:
        rt.commit(); raised = False
    except _abi.PtbError:
        raised = True
    assert raised
    rt = scenes.config_fog(test_lib, 16, 16, 1).commit()
    try:
        rt.render_denoiser_inputs(); raised = False
    except _abi.PtbError:
        raised = True
    assert raised, "the denoiser-input mode is not combined with the branching modes"


def case_converged(test_lib, oracle_lib):
    mk = lambda L: scenes.config_C2(L, 40, 40, 8, nv=24, env=(128, 64))
    hi = mk(oracle_lib).commit()
    hi.nrays, hi.seed = 512, 99
    ref_hi = hi.render_image_nopreviz().copy()
    a, b = mk(oracle_lib).commit(), mk(test_lib).commit()
    ia, ib = a.render_image_nopreviz().copy(), b.render_image_nopreviz().copy()
    ea, eb = rrmse(ia, ref_hi), rrmse(ib, ref_hi)
    assert eb <= RRMSE_FACTOR * ea + 0.005, (ea, eb)
    assert rrmse(ib, ia) <= 0.02, "equal-seed images should be nearly the same image"


def kat_tolerances():
    # (rtol, atol, fraction of rows allowed outside) per building block
    return {
        _abi.KAT_PCG32: (0, 0, 0), _abi.KAT_LATTICE: (0, 0, 0), _abi.KAT_FAST_EXP: (0, 0, 0), _abi.KAT_RANDOM_PER_PIXEL: (0, 0, 0),
        _abi.KAT_FILTER_RATIO: (0, 0, 0), _abi.KAT_FAST_NORMALIZE: (4e-7, 0, 0), _abi.KAT_CAMERA: (2e-6, 2e-6, 0),
        _abi.KAT_RANDOM_COS: (2e-5, 2e-6, 0), _abi.KAT_RANDOM_PHONG: (2e-5, 2e-6, 0), _abi.KAT_PHONG_EVAL: (1e-4, 1e-7, 0),
        _abi.KAT_MERL_EVAL: (0, 0, 0.02),   # a lookup without interpolation: bin flips at bin borders only
    }


def case_kats(test_lib, gold):
    from golden_scenes import KAT_INPUTS
    rt = scenes.config_C4(test_lib, 32, 32, 1, nv=10).commit()
    for which, (inp, kw) in KAT_INPUTS().items():
        rtol, atol, frac = kat_tolerances()[which]
        got, want = rt.kat(which, inp, **kw), gold[f"out_{which}"]
        ok = np.isclose(got, want, rtol=rtol, atol=atol).all(-1)
        assert 1 - ok.mean() <= frac, f"KAT {which}: {(~ok).sum()} of {len(ok)} rows outside rtol={rtol} atol={atol}"
    rt.close()


def case_merl_index_fast(test_lib, n=400000):
    """The float evaluation of the MERL bin index (merl_index_fast) either declines or returns the bin of the double path
    (MERLBRDFRead.cpp:76-207): random pairs as the integrator makes them, plus the ill-conditioned corners (direction next to the
    normal, half vector next to the normal, coincident directions, grazing directions)."""
    rng = np.random.default_rng(20261017)
    def hemi(m):
        r2, ph = rng.random(m), 2 * np.pi * rng.random(m)
        s = np.sqrt(1 - r2)
        return np.stack([np.cos(ph) * s, np.sin(ph) * s, np.sqrt(r2)], -1)
    a, b = hemi(n), hemi(n)
    k = n // 8
    b[:k] = a[:k] + 1e-3 * (rng.random((k, 3)) - .5)                                       # theta_diff -> 0
    b[k:2 * k] = a[k:2 * k] * np.array([-1, -1, 1]) + 1e-3 * (rng.random((k, 3)) - .5)        # half vector -> normal
    b[2 * k:3 * k] = np.array([0, 0, 1]) + 3e-3 * (rng.random((k, 3)) - .5)                  # wo -> normal
    a[3 * k:4 * k, 2] = 1e-3 * rng.random(k)                                                 # grazing wi
    a /= np.linalg.norm(a, axis=1, keepdims=True); b /= np.linalg.norm(b, axis=1, keepdims=True)
    inp = np.concatenate([a, b], -1).astype(np.float32).astype(np.float64)
    rt = scenes.config_C4(test_lib, 16, 16, 1, nv=8).commit()
    out = rt.kat(_abi.KAT_MERL_INDEX, inp)
    rt.close()
    fast, exact = out[:, 0].astype(np.int64), out[:, 1].astype(np.int64)
    took = fast >= 0
    assert (fast[took] == exact[took]).all(), f"{(fast[took] != exact[took]).sum()} bins differ"
    assert took[4 * k:].mean() > 0.97, "the float path should answer almost every ordinary pair"
    assert (exact >= 0).all() and (exact < 90 * 90 * 180).all()


def triangle_soup(n, seed=7):
    """n unconnected random triangles of very different sizes in a unit cube (file axes): irregular trees, leaves of 1-3 triangles in
    arbitrary slots, overlapping boxes - what a displaced torus never produces."""
    rng = np.random.default_rng(seed)
    c = rng.random((n, 1, 3)) * 2 - 1
    size = (0.02 + 0.5 * rng.random((n, 1, 1)) ** 4)
    v = (c + size * (rng.random((n, 3, 3)) - 0.5)).reshape(-1, 3).astype(np.float32)
    nrm = np.cross(v[1::3] - v[0::3], v[2::3] - v[0::3])
    nrm = np.repeat(nrm / np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-20), 3, 0).astype(np.float32)
    idx = np.arange(3 * n, dtype=np.int32).reshape(n, 3)
    tri = np.concatenate([idx, np.full((n, 3), -1, np.int32), idx, np.zeros((n, 1), np.int32)], 1)
    return v, nrm, np.zeros((0, 2), np.float32), tri


def case_triangle_soup(test_lib, oracle_lib, n=3000, agree=ID_AGREE):
    """closest hits (primary ids from two view points) and a path-traced image (closest + shadow rays) over a random soup"""
    def mk(L):
        rt = scenes.base(L, 96, 72, 2)
        m = scenes._place_like_gui(TriMesh(*triangle_soup(n)), scale=22.0)
        m.set_material(0, **scenes.phong((.6, .5, .4), 0.1, 20.0))
        rt.s.addObject(m)
        return rt.commit()
    a, b = mk(oracle_lib), mk(test_lib)
    check_ids(b, a, agree=agree)
    ia, ib = a.render_image_nopreviz().copy(), b.render_image_nopreviz().copy()
    check_images(ib, ia, frac=0.01)
    for rt in (a, b):
        rt.cam.position = np.array([25, 10, -30], np.float32)
        d = np.array([-0.55, -0.45, 0.7], np.float32)
        rt.cam.direction = d / np.float32(np.linalg.norm(d))
        rt.cam.up = np.array([0, 1, 0], np.float32)
    check_ids(b, a, agree=agree)


# ---- edge cases -------------------------------------------------------------------------------------------------
def quad_mesh(n=6, with_uv=True, with_normals=True, groups=False):
    """A wavy (n x n)-quad sheet in file axes."""
    g = np.linspace(-1, 1, n + 1)
    x, z = np.meshgrid(g, g, indexing="xy")
    y = 0.15 * np.sin(3 * x) * np.cos(2 * z)
    v = np.stack([x, y, z], -1).reshape(-1, 3).astype(np.float32)
    nrm = np.stack([-0.45 * np.cos(3 * x) * np.cos(2 * z), np.ones_like(x), 0.3 * np.sin(3 * x) * np.sin(2 * z)], -1).reshape(-1, 3)
    nrm = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype(np.float32)
    uv = np.stack([(x + 1) / 2, (z + 1) / 2], -1).reshape(-1, 2).astype(np.float32)
    tri = []
    for r in range(n):
        for c in range(n):
            a = r * (n + 1) + c
            b, cc, d = a + 1, a + n + 1, a + n + 2
            for t in ((a, cc, b), (b, cc, d)):
                grp = ((r + c) % 2) if groups else 0
                tri.append([*t, *(t if with_uv else (-1, -1, -1)), *(t if with_normals else (-1, -1, -1)), grp])
    return v, (nrm if with_normals else np.zeros((0, 3), np.float32)), (uv if with_uv else np.zeros((0, 2), np.float32)), np.array(tri, np.int32)


def edge_scene(L, variant, W=37, H=23, spp=3):
    rt = scenes.base(L, W, H, spp)
    if variant == "mirror_and_flip":
        s = Sphere((0, -17.3, 0), 10, mirror=True).set_material(0, **scenes.phong((.8, .8, .8), 0.0, 1.0))
        s2 = Sphere((-14, -20, 8), 6, normal_swapped=False).set_material(0, **scenes.phong((.2, .5, .9), 0.4, 20.0, transp=Texture(0.0), refr=Texture(1.4)))
        rt.s.addObject(s); rt.s.addObject(s2)
    elif variant == "mesh_no_uv_groups":
        m = scenes._place_like_gui(TriMesh(*quad_mesh(with_uv=False, groups=True)))
        m.set_material(0, **scenes.phong((.7, .2, .2), 0.1, 30.0)); m.set_material(1, **scenes.phong((.2, .7, .2), 0.0, 1.0))
        rt.s.addObject(m)
    elif variant == "mesh_flat":
        m = scenes._place_like_gui(TriMesh(*quad_mesh(groups=True)))
        m.interp_normals = False
        m.set_material(0, **scenes.phong((.6, .6, .2), 0.2, 40.0))   # group 1 has no material: defaults Kd=1
        rt.s.addObject(m)
    elif variant == "textured_rotated":
        v, n, uv, tri = quad_mesh(groups=False)
        m = scenes._place_like_gui(TriMesh(v, n, uv, tri))
        th = 0.6
        m.mat_rotation = np.array([[np.cos(th), 0, np.sin(th)], [0, 1, 0], [-np.sin(th), 0, np.cos(th)]], np.float32)
        yy, xx = np.mgrid[0:16, 0:16]
        kd = np.stack([(xx % 4 < 2) * .8 + .1, (yy % 4 < 2) * .8 + .1, np.full((16, 16), .3)], -1).astype(np.float32)
        mat = scenes.phong((1, 1, 1), 0.1, 25.0, normal=Texture((0, 0, 1), scenes.wave_normal_map(32)), alpha=Texture(1.0, scenes.checker_alpha_map(32)))
        mat["Kd"] = Texture((1, 1, 1), kd)
        m.set_material(0, **mat)
        rt.s.addObject(m)
        pl = rt.s.objects[2]
        pl.set_material(0, Kd=Texture((1, 1, 1), kd))
    elif variant == "alpha_classes":
        # the commit-time alpha classification (scene_host.cpp): a fine mesh under a coarse alpha map has triangles that are
        # entirely opaque, entirely transparent (left out of the BVH) and straddling (still tested); uvs run over [-1.5, 2.5]
        # so that the wrap is exercised; a second group has a constant alpha below 0.5 (never hit)
        v, n, uv, tri = quad_mesh(n=24, groups=True)
        uv = (uv * 4.0 - 1.5).astype(np.float32)
        m = scenes._place_like_gui(TriMesh(v, n, uv, tri))
        a = np.ones((8, 8, 3), np.float32); a[::2, 1::3] = 0.0; a[5, :] = 0.0
        m.set_material(0, **scenes.phong((.7, .7, .3), 0.1, 25.0, alpha=Texture(1.0, a)))
        m.set_material(1, **scenes.phong((.2, .3, .8), 0.1, 25.0, alpha=Texture(0.25)))
        rt.s.addObject(m)
        m2 = scenes._place_like_gui(TriMesh(*quad_mesh(n=8)), scale=14.0)
        m2.max_translation = m2.max_translation + np.array([0, 6, -4], np.float32)
        m2.set_material(0, **scenes.phong((.8, .3, .3), 0.0, 1.0, alpha=Texture(1.0, scenes.checker_alpha_map(64))))
        rt.s.addObject(m2)
    elif variant in ("mesh_one_triangle", "mesh_four_triangles"):
        # the smallest trees: a root that holds a single leaf, and a root with four one-triangle leaves (valid24 / compact indices)
        v = np.array([[-1, 0, -1], [1, 0, -1], [1, 0.3, 1], [-1, 0.2, 1], [0, 1, 0]], np.float32)
        n = np.tile(np.array([[0, 1, 0]], np.float32), (5, 1))
        uv = np.array([[0, 0], [1, 0], [1, 1], [0, 1], [.5, .5]], np.float32)
        faces = [(0, 2, 1), (0, 3, 2), (0, 1, 4), (1, 2, 4)][:1 if variant == "mesh_one_triangle" else 4]
        tri = np.array([[*f, *f, *f, 0] for f in faces], np.int32)
        m = scenes._place_like_gui(TriMesh(v, n, uv, tri))
        m.set_material(0, **scenes.phong((.7, .4, .3), 0.1, 20.0))
        rt.s.addObject(m)
    elif variant == "many_spheres":      # more analytic objects than the kernel-parameter table holds (8)
        for k in range(9):
            c = (-16 + 4 * k, -22.3 + (k % 3), -6 + 3 * (k % 4))
            rt.s.addObject(Sphere(c, 2.5 + 0.3 * (k % 3)).set_material(0, **scenes.phong((.2 + .08 * k, .5, .9 - .08 * k), 0.1 * (k % 2), 20.0)))
    elif variant == "wide_filter":
        rt.sigma_filter = 1.0
        rt.s.addObject(Sphere((0, -17.3, 0), 10).set_material(0, **scenes.phong((.8, .3, .3), 0.0, 1.0)))
    elif variant == "depth_one":
        rt.nb_bounces = 1
        rt.s.addObject(Sphere((0, -17.3, 0), 10).set_material(0, **scenes.phong((.8, .3, .3), 0.3, 10.0)))
    else:
        raise KeyError(variant)
    return rt


EDGE_VARIANTS = ["many_spheres", "mirror_and_flip", "mesh_no_uv_groups", "mesh_flat", "textured_rotated", "alpha_classes", "mesh_one_triangle", "mesh_four_triangles", "wide_filter", "depth_one"]


def case_edge(test_lib, oracle_lib, variant):
    a, b = edge_scene(oracle_lib, variant).commit(), edge_scene(test_lib, variant).commit()
    ia, ib = a.render_image_nopreviz().copy(), b.render_image_nopreviz().copy()
    check_images(ib, ia, frac=0.01)
    assert np.allclose(a.sample_count, b.sample_count, rtol=1e-5)
    oa, ta, _ = a.primary_ids(); ob, tb, _ = b.primary_ids()
    assert ((oa == ob) & (ta == tb)).mean() >= 0.998   # 851 pixels: at most one edge pixel may flip
    if variant == "alpha_classes":
        info = b.scene_info()
        assert info["n_triangles"] == 2 * 24 * 24 + 2 * 8 * 8
        if "bytes_triangles" in info and info["bytes_triangles"]:
            assert info["bytes_triangles"] < 48 * info["n_triangles"] * 0.8, "the constant-transparent group and the all-transparent footprints are not resident"


def case_passes_and_shards(test_lib):
    """Size-independent properties: splitting the work into passes or shards must not change the image."""
    mk = lambda: scenes.config_C2(test_lib, 150, 70, 5, nv=16, env=(64, 32)).commit()
    whole = mk()
    ref = whole.render_image_nopreviz().copy()
    cnt = whole.sample_count.copy()
    small = mk()
    small.set_option(_abi.OPT_POOL_PATHS, 4096)      # forces several slot passes and one sample per pass
    img = small.render_image_nopreviz()
    assert np.allclose(img, ref, rtol=2e-5, atol=1e-3) and np.allclose(small.sample_count, cnt, rtol=2e-5)
    assert small.stats["rays_closest"] == whole.stats["rays_closest"] and small.stats["samples"] == whole.stats["samples"]
    return whole, ref, cnt


def case_errors(test_lib):
    import ctypes as C
    from pathtracer_b200.api import Raytracer
    rt = Raytracer(test_lib)
    rt.s.addObject(Sphere((0, 0, 0), 1))
    try:
        rt.commit()
        raised = False
    except _abi.PtbError:
        raised = True
    assert raised, "commit without the dome must fail (object ids 0/1 are hard-wired)"
    rt = scenes.base(test_lib, 8, 8, 1)
    rt.s.addObject(TriMesh(np.zeros((0, 3)), np.zeros((0, 3)), np.zeros((0, 2)), np.zeros((0, 10), np.int32)))
    try:
        rt.commit()
        raised = False
    except _abi.PtbError:
        raised = True
    assert raised, "an empty mesh is rejected"
    # yarns: missing arrays, no segment, a negative or NaN radius are refused at the boundary
    ctx = C.c_void_p()
    test_lib.check(test_lib.create(0, C.byref(ctx)))
    a = np.zeros((2, 3), np.float32); b = np.ones((2, 3), np.float32)
    for desc in (_abi.YarnsDesc(None, None, None, 2), _abi.YarnsDesc(_abi.fptr(a), _abi.fptr(b), _abi.fptr(np.array([.1, .1], np.float32)), 0),
                 _abi.YarnsDesc(_abi.fptr(a), _abi.fptr(b), _abi.fptr(np.array([.1, -1], np.float32)), 2),
                 _abi.YarnsDesc(_abi.fptr(a), _abi.fptr(b), _abi.fptr(np.array([np.nan, .1], np.float32)), 2)):
        assert test_lib.add_yarns(ctx, C.byref(desc), None, 0, None) == _abi.ERR_INVALID
    oid = C.c_int(-1)
    ok = _abi.YarnsDesc(_abi.fptr(a), _abi.fptr(b), _abi.fptr(np.array([.1, .2], np.float32)), 2)
    assert test_lib.add_yarns(ctx, C.byref(ok), None, 0, C.byref(oid)) == _abi.OK and oid.value == 0
    test_lib.destroy(ctx)


# ---- the other two renderers of the reference over the same integrator -------------------------------------------------
def mode_scene(L, W=56, H=40, spp=6):
    """A ragged frame (not a multiple of 16 or of the tile) with every path type: mesh + textured plane + mirror sphere + dome."""
    rt = scenes.config_C2(L, W, H, spp, nv=20, env=(64, 32))
    # (a sphere WITHOUT any slot keeps whatever material the previous object of Scene::intersection's loop left in `localmat`,
    #  Geometry.h:979 — its albedo AOV is undefined in the reference, so the mirror gets a slot)
    rt.s.addObject(Sphere((-14, -20, 8), 6, mirror=True).set_material(0, Kd=Texture((.9, .9, .9))))
    rt.s.objects[2].set_material(0, Kd=Texture((.7, .6, .5)), Ks=Texture(.1), Ne=Texture(30.0))
    return rt


def mode_scene_exotic(L, W=56, H=40, spp=6):
    """The same ragged frame over the primitives of row f4 (yarns, a point set, a cylinder) on the linear path."""
    return scenes.config_exotic_modes(L, W, H, spp, mode="plain")


def case_progressive(test_lib, oracle_lib, frac=FRAC_1SPP, mode_scene=mode_scene):
    """Raytracer::render_image: un-normalised sums, weight sums, the /max(count,1) display image, the 16x16 low-resolution preview;
    stopping after k passes; and sums == nopreviz sums (same per-(pixel,sample) streams)."""
    a, b = mode_scene(oracle_lib).commit(), mode_scene(test_lib).commit()
    ia, ib = a.render_image().copy(), b.render_image(passes_per_call=4).copy()      # 6 passes as 4 + 2
    assert a.current_nb_rays == b.current_nb_rays == 6
    check_images(ib, ia, frac)
    assert np.allclose(a.sample_count, b.sample_count, rtol=1e-5)
    assert np.mean(np.abs(a.image.astype(int) - b.image.astype(int)) > 1) <= 2 * frac
    assert b.imagedouble_lowres.shape == (3, 4, 3) and np.allclose(b.imagedouble_lowres, a.imagedouble_lowres, rtol=2e-3)
    # un-normalised: dividing by the weights gives the nopreviz image
    nb = b.render_image_nopreviz().copy()
    assert np.allclose(ib / b.sample_count[..., None], nb, rtol=1e-4, atol=1e-2)
    # a stop request after 2 passes (the GUI's `stopped`, Raytracer.cpp:1452)
    def stop_after_two(rt):
        rt.stopped = rt.current_nb_rays >= 2
    a.render_image(on_pass=stop_after_two); b.render_image(on_pass=stop_after_two)
    assert a.current_nb_rays == b.current_nb_rays == 2
    check_images(b.imagedouble, a.imagedouble, frac)
    assert np.allclose(a.sample_count, b.sample_count, rtol=1e-5)
    a.close(); b.close()


def case_denoiser_inputs(test_lib, oracle_lib, frac=FRAC_1SPP, mode_scene=mode_scene):
    """render_image_nopreviz with has_denoiser: unsplatted means, first-hit albedo, the reference's `normalImage`, and the first-hit normals."""
    a, b = mode_scene(oracle_lib).commit(), mode_scene(test_lib).commit()
    a.render_denoiser_inputs(); b.render_denoiser_inputs()
    check_images(b.imagedouble, a.imagedouble, frac)
    assert np.array_equal(a.sample_count, b.sample_count) and (b.sample_count == 6).all()
    assert np.mean(np.abs(a.albedoImage - b.albedoImage).max(-1) > 1e-4) <= frac
    ok = np.isfinite(a.normalImage).all(-1) & np.isfinite(b.normalImage).all(-1)
    assert np.array_equal(np.isfinite(a.normalImage).all(-1), np.isfinite(b.normalImage).all(-1)) or ok.mean() > 0.99
    assert np.mean(np.abs(a.normalImage - b.normalImage)[ok].reshape(-1, 3).max(-1) > 1e-3) <= 2 * frac
    if np.isfinite(a.first_hit_normal).any():          # the compiled reference cannot produce this one (it sums colours instead)
        fin = np.isfinite(a.first_hit_normal).all(-1) & np.isfinite(b.first_hit_normal).all(-1)
        assert fin.mean() > 0.95 and np.mean(np.abs(a.first_hit_normal - b.first_hit_normal)[fin].reshape(-1, 3).max(-1) > 1e-3) <= 2 * frac
        assert np.allclose(np.linalg.norm(b.first_hit_normal[fin], axis=-1), 1, atol=1e-5)
    a.close(); b.close()
