"""Pins the oracle: oracle/port (plain-C restatement) must reproduce the REFERENCE's own outputs —
(1) the known answers recorded in SURVEY.md App. E, (2) the golden vectors under tests/golden/ that
tests/golden/make_golden.py generated from oracle/_ref, bit for bit, and (3) oracle/_ref itself when it is
present in this checkout (it is whenever PTB_REFERENCE_DIR names a checkout of the reference at build time)."""
import os

import numpy as np
import pytest
from golden_scenes import ANIM_SCENES, BRANCH_SCENES, KAT_INPUTS, SCENES, STAT_SCENES

ALL_SCENES = {**SCENES, **BRANCH_SCENES, **STAT_SCENES, **ANIM_SCENES}

from pathtracer_b200 import _abi, scenes

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def port_rt(port):
    return scenes.config_C4(port, 32, 32, 1, nv=10).commit()


def test_known_answers_from_the_survey(port_rt):
    rt = port_rt
    assert rt.kat(_abi.KAT_PCG32, [[12345, 7]])[0].tolist() == [1852478230, 3367905088, 934649197, 1102233149]
    lat = rt.kat(_abi.KAT_LATTICE, [[0], [1], [2], [3], [4]]).astype(np.float32)
    want = np.array([(0.456789136, 0.123456791), (0.956789136, 0.625), (0.706789136, 0.875), (0.206789136, 0.375), (0.581789136, 0.498046875)], np.float32)
    assert np.array_equal(lat, want)
    fe = rt.kat(_abi.KAT_FAST_EXP, [[0], [-0.5], [-1], [-2], [-4]]).ravel()
    assert np.allclose(fe, [0.971007824, 0.61033392, 0.374830246, 0.13207829, 0.018300578], rtol=2e-9)
    assert np.allclose(rt.cam.direction, [0, -0.37460658, -0.927183867], atol=1e-8) and np.allclose(rt.cam.up, [0, 0.927183867, -0.37460658], atol=1e-8)
    assert rt.s.intensite_lumiere == 3183098.75
    cam = rt.kat(_abi.KAT_CAMERA, [[0, 0, 0, 0, 0, 0], [300, 200, .25, -.125, .03, -.02]], W=512, H=512).astype(np.float32)
    assert np.allclose(cam[0], [0, 0, 50, -0.287498534, -0.608809531, -0.739388645], rtol=0, atol=1e-9)
    assert np.allclose(cam[1], [0.0299999993, -0.0185436774, 50.0074921, -0.0683836266, -0.322315991, -0.944158912], rtol=1e-7, atol=0)
    N = np.array([0.3, 0.8, -0.52]) / np.linalg.norm([0.3, 0.8, -0.52])
    assert np.allclose(rt.kat(_abi.KAT_RANDOM_COS, [[*N, .37, .61]])[0], [-0.200019926, 0.506198049, -0.838901401], atol=1e-8)
    assert np.allclose(rt.kat(_abi.KAT_RANDOM_PHONG, [[*N, 50, .37, .61]])[0], [0.200695038, 0.765834928, -0.610915959], atol=1e-8)
    wo, wi = np.array([.1, .9, .2]), np.array([-.2, .85, -.3])
    ev = rt.kat(_abi.KAT_PHONG_EVAL, [[.5, .4, .3, .2, .2, .2, 50, 50, 50, *(wi / np.linalg.norm(wi)), *(wo / np.linalg.norm(wo)), *N]])[0]
    assert np.allclose(ev, [0.159154937, 0.127323955, 0.0954929665], atol=1e-8)


def test_kat_golden_bit_exact(port_rt):
    gold = np.load(os.path.join(GOLD, "kat.npz"))
    for which, (inp, kw) in KAT_INPUTS().items():
        assert np.array_equal(inp, gold[f"in_{which}"]), which
        got = port_rt.kat(which, inp, **kw)
        assert np.array_equal(got, gold[f"out_{which}"]), f"KAT {which} differs from the reference's output"


@pytest.mark.parametrize("name", sorted(ALL_SCENES))
def test_scene_golden_bit_exact(port, name):
    gold = np.load(os.path.join(GOLD, f"scene_{name}.npz"))
    rt = ALL_SCENES[name](port).commit()
    rt.set_option(_abi.ORC_OPT_THREADS, 1)
    obj, tri, t = rt.primary_ids()
    assert np.array_equal(obj, gold["obj"]) and np.array_equal(tri, gold["tri"]) and np.array_equal(t, gold["t"])
    img = rt.render_image_nopreviz()
    assert np.array_equal(img, gold["imagedouble"]), "linear image differs from the reference's"
    assert np.array_equal(rt.sample_count, gold["sample_count"]) and np.array_equal(rt.image, gold["image"])
    assert [rt.stats["rays_closest"], rt.stats["rays_shadow"]] == gold["rays"].tolist()


@pytest.mark.parametrize("name", sorted(ALL_SCENES))
def test_port_equals_compiled_reference(port, ref, name):
    a, b = ALL_SCENES[name](ref).commit(), ALL_SCENES[name](port).commit()
    for rt in (a, b):
        rt.set_option(_abi.ORC_OPT_THREADS, 1)
        rt.nrays, rt.seed = 3, 7          # a seed and spp the golden files do not cover
    ia, ib = a.render_image_nopreviz(), b.render_image_nopreviz()
    assert np.array_equal(ia, ib) and np.array_equal(a.image, b.image)
    assert a.stats["rays_closest"] == b.stats["rays_closest"] and a.stats["rays_shadow"] == b.stats["rays_shadow"]
    assert a.scene_info()["n_bvh_nodes"] == b.scene_info()["n_bvh_nodes"]


def test_port_is_thread_count_invariant_up_to_summation_order(port):
    a, b = SCENES["C2"](port).commit(), SCENES["C2"](port).commit()
    a.set_option(_abi.ORC_OPT_THREADS, 1)
    b.set_option(_abi.ORC_OPT_THREADS, 4)
    ia, ib = a.render_image_nopreviz(), b.render_image_nopreviz()
    assert np.allclose(ia, ib, rtol=1e-5)
    assert a.stats["rays_closest"] == b.stats["rays_closest"]


def test_modes_golden_bit_exact(port):
    """Raytracer::render_image (progressive) and the has_denoiser accumulation of render_image_nopreviz, against the reference's own outputs."""
    from parity_cases import mode_scene
    gold = np.load(os.path.join(GOLD, "modes.npz"))
    rt = mode_scene(port).commit()
    rt.set_option(_abi.ORC_OPT_THREADS, 1)
    rt.render_image()
    for k in ("imagedouble", "sample_count", "image", "imagedouble_lowres"):
        assert np.array_equal(getattr(rt, k), gold[f"progressive/{k}"]), k

    def stop_after_two(r):
        r.stopped = r.current_nb_rays >= 2
    rt.render_image(on_pass=stop_after_two)
    for k in ("imagedouble", "sample_count", "image", "imagedouble_lowres"):
        assert np.array_equal(getattr(rt, k), gold[f"progressive2/{k}"]), k
    rt.render_denoiser_inputs()
    for k in ("imagedouble", "sample_count", "albedoImage"):
        assert np.array_equal(getattr(rt, k), gold[f"denoiser/{k}"]), k
    assert np.array_equal(np.nan_to_num(rt.normalImage, nan=-9), np.nan_to_num(gold["denoiser/normalImage"], nan=-9))
    fin = np.isfinite(rt.first_hit_normal).all(-1)
    assert fin.mean() > 0.95 and np.allclose(np.linalg.norm(rt.first_hit_normal[fin], axis=-1), 1, atol=1e-5)
