"""CPU coverage of everything that is host code or host-checkable: scene ingestion (TriMesh::init semantics,
tangents, matrices), the BVH8 builder, the shard/tile arithmetic — and, through tests/devsim (the device headers
compiled for the host, test-only), the device logic itself against the oracle.  No GPU needed."""
import os
import sys

import numpy as np
import pytest
from golden_scenes import ANIM_SCENES, BRANCH_SCENES, SCENES
from parity_cases import (EDGE_VARIANTS, case_branch_converged, case_branch_errors, case_branch_scene, case_converged, case_sss_converged, case_denoiser_inputs, case_edge, case_errors, case_kats, case_merl_index_fast, case_triangle_soup, case_passes_and_shards,
                          case_progressive, case_scene, mode_scene_exotic, case_yarn_cloth, case_yarn_from_inside, check_ids)

from pathtracer_b200 import _abi, scenes

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_kats_devsim(devsim):
    case_kats(devsim, np.load(os.path.join(GOLD, "kat.npz")))


def test_merl_index_fast_devsim(devsim):
    case_merl_index_fast(devsim)


@pytest.mark.parametrize("name", sorted(SCENES))
def test_scenes_devsim_vs_oracle(devsim, port, name):
    case_scene(devsim, port, SCENES[name])


@pytest.mark.parametrize("variant", EDGE_VARIANTS)
def test_edge_cases_devsim(devsim, port, variant):
    case_edge(devsim, port, variant)


def test_yarn_seen_from_inside_its_covering_prism_devsim(devsim, port):
    case_yarn_from_inside(devsim, port)


def test_yarn_cloth_of_72000_segments_devsim(devsim, port):
    case_yarn_cloth(devsim, port, 256, 256)


def test_progressive_devsim(devsim, port):
    case_progressive(devsim, port)


def test_denoiser_inputs_devsim(devsim, port):
    case_denoiser_inputs(devsim, port)


def test_progressive_and_denoiser_inputs_over_yarns_discs_cylinders_devsim(devsim, port):
    case_progressive(devsim, port, mode_scene=mode_scene_exotic)
    case_denoiser_inputs(devsim, port, mode_scene=mode_scene_exotic)


def test_converged_devsim(devsim, port):
    case_converged(devsim, port)


@pytest.mark.parametrize("name", sorted(ANIM_SCENES))
def test_keyframed_scenes_devsim_vs_oracle(devsim, port, name):
    case_scene(devsim, port, ANIM_SCENES[name], agree=0.998)   # 2304 pixels of a coarse, rotated mesh: a silhouette pixel may flip


@pytest.mark.parametrize("name", sorted(BRANCH_SCENES))
def test_branch_scenes_devsim_vs_oracle(devsim, port, name):
    case_branch_scene(devsim, port, BRANCH_SCENES[name])


def test_branch_converged_devsim(devsim, port):
    case_branch_converged(devsim, port)


def test_sss_converged_devsim(devsim, port):
    case_sss_converged(devsim, port, spp=48)


def test_bvh8_against_oracle_on_a_larger_mesh(devsim, port):
    """160k triangles, 200x200 picking rays from two view points: exercises deep trees, quantisation slack and leaf packing."""
    mk = lambda L: scenes.config_C2(L, 200, 200, 1, nv=200, env=(64, 32))
    a, b = mk(port).commit(), mk(devsim).commit()
    check_ids(b, a)
    info = b.scene_info()
    assert info["n_triangles"] == 160000 and 0 < info["n_bvh_nodes"] < 160000 / 2 and info["bvh_depth"] <= 12
    for rt in (a, b):
        rt.cam.position = np.array([30, 5, 30], np.float32)
        rt.cam.direction = np.array([-0.6, -0.35, -0.72], np.float32) / np.float32(np.linalg.norm([-0.6, -0.35, -0.72]))
        rt.cam.up = np.array([0, 1, 0], np.float32)
    check_ids(b, a)


def test_triangle_soup_devsim(devsim, port):
    case_triangle_soup(devsim, port)


def test_passes_and_shards_devsim(devsim):
    whole, ref, cnt = case_passes_and_shards(devsim)
    # shards: three ranks accumulate into one buffer == the whole frame (ragged 150x70 frame, 32-pixel tiles)
    acc = np.zeros((whole.H * whole.W, 4), np.float32)
    total = 0
    for r in range(3):
        st = whole.render_accum(acc.ctypes.data, r, 3, 32)
        total += st["samples"]
    assert total == whole.W * whole.H * whole.nrays
    img = whole.resolve(acc.ctypes.data)
    assert np.allclose(img, ref, rtol=2e-5, atol=1e-3) and np.allclose(whole.sample_count, cnt, rtol=2e-5)


def test_shard_pack_roundtrip_devsim(devsim):
    import ctypes as C
    rt = scenes.config_C1(devsim, 150, 70, 2).commit()
    full = np.zeros((rt.H * rt.W, 4), np.float32)
    rt.render_accum(full.ctypes.data, 0, 1, 32)
    merged = np.zeros_like(full)
    for world in (2, 3, 4):
        merged[:] = 0
        for r in range(world):
            part = np.zeros_like(full)
            rt.render_accum(part.ctypes.data, r, world, 32)
            n = C.c_int64()
            p = rt.params(r, world, 32)
            devsim.check(devsim.shard_pack_size(C.byref(p), r, C.byref(n)))
            packed = np.zeros(n.value, np.float32)
            devsim.check(devsim.shard_pack(rt._ctx, C.byref(p), r, C.c_void_p(part.ctypes.data), C.c_void_p(packed.ctypes.data)))
            devsim.check(devsim.shard_unpack_add(rt._ctx, C.byref(p), r, C.c_void_p(packed.ctypes.data), C.c_void_p(merged.ctypes.data)))
        assert np.allclose(merged, full, rtol=2e-5, atol=1e-2), world


def test_tile_ownership_is_a_spread_bijection(devsim):
    """ptb_scene.h shard_tile_shift / tile_physical / tile_logical: every tile belongs to exactly one shard, shard sizes differ by at
    most one tile, and when the tile columns are a multiple of the shard count (the case that used to give vertical stripes) every row
    AND every column of tiles holds every shard equally often."""
    import ctypes
    raw = ctypes.CDLL(os.path.join(os.path.dirname(os.path.abspath(__file__)), "devsim", "libptb_devsim.so"))
    for tiles_x, tiles_y, count in [(16, 16, 8), (16, 16, 4), (16, 16, 2), (60, 34, 8), (30, 17, 8), (5, 3, 3), (13, 7, 8), (1, 9, 4), (7, 1, 3), (32, 32, 8), (3, 3, 1)]:
        owner = np.full(tiles_x * tiles_y, -7, np.int32); order = owner.copy()
        ip = ctypes.POINTER(ctypes.c_int32)
        shift = raw.devsim_tile_owners(tiles_x, tiles_y, count, owner.ctypes.data_as(ip), order.ctypes.data_as(ip))
        assert shift >= 0, (tiles_x, tiles_y, count, shift)
        assert (owner >= 0).all() and (owner < count).all()
        sizes = np.bincount(owner, minlength=count)
        assert sizes.max() - sizes.min() <= 1
        for r in range(count):                                   # a shard's render order enumerates its tiles 0..n-1
            assert sorted(order[owner == r]) == list(range(sizes[r]))
        if count == 1:
            assert shift == 0 and (order == np.arange(tiles_x * tiles_y)).all()     # one GPU keeps the plain row-major order
        if count > 1 and tiles_x % count == 0 and tiles_y % count == 0:
            grid = owner.reshape(tiles_y, tiles_x)
            for r in range(count):
                assert ((grid == r).sum(0) == tiles_y // count).all() and ((grid == r).sum(1) == tiles_x // count).all()


def test_errors_devsim(devsim):
    case_errors(devsim)


def test_generators_are_deterministic_and_sized():
    v, n, uv, tri = scenes.displaced_torus(10)
    assert len(tri) == 400 and tri[:, :3].max() < len(v) and np.allclose(np.linalg.norm(n, axis=1), 1, atol=1e-6)
    assert 4 * 500 ** 2 == 1000000 and 4 * 791 ** 2 == 2502724 and 4 * 255 ** 2 == 260100 and 8 * 4 * 866 ** 2 == 23998592
    env = scenes.sky_envmap(64, 32)
    assert env.dtype == np.uint8 and env.shape == (32, 64, 3) and env.max() == 255
    t = scenes.merl_table()
    assert t.shape == (3, 90, 90, 180) and np.allclose(t[0] * (1.0 / 1500), t[1] * (1.15 / 1500)) and np.allclose(t[0] * (1.0 / 1500), t[2] * (1.66 / 1500))


def test_material_presets_equal_the_reference_menu():
    """Phong / Ngan material presets (north_star: "Phong/Ngan/MERL materials"): the table of the Python mirror, the table inside the
    library (ptb_preset_get) and the constants of the reference's object menu (mainApp.cpp:1499-1597, committed as
    tests/golden/presets.json by tests/golden/make_presets.py; re-parsed live when PTB_REFERENCE_DIR names the reference) are the same numbers."""
    import ctypes as C
    import json
    import pathtracer_b200
    from pathtracer_b200 import api
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "presets.json")))
    from oracles import reference_dir
    menu = os.path.join(reference_dir(), "mainApp.cpp") if reference_dir() else None
    if menu and os.path.exists(menu):
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
        import make_presets
        assert make_presets.parse(menu) == gold
    assert sorted(gold) == sorted(api.PRESETS) and len(gold) == 14 and sum(k.endswith("_ngan") for k in gold) == 7
    lib = pathtracer_b200.load()
    assert lib.preset_count() == 14 and lib.preset_find(b"nope") == -1
    for name, g in gold.items():
        kd, ks, ne = api.PRESETS[name]
        f32 = lambda v: [float(np.float32(x)) for x in v]
        assert f32(kd) == f32(g["Kd"]) and f32(ks) == f32(g["Ks"]) and f32([ne] * 3) == f32(g["Ne"]), name
        i = lib.preset_find(name.encode())
        assert i >= 0
        nm, a, b, c = C.c_char_p(), (C.c_float * 3)(), (C.c_float * 3)(), C.c_float()
        assert lib.preset_get(i, C.byref(nm), a, b, C.byref(c)) == 0 and nm.value.decode() == name
        assert list(a) == f32(g["Kd"]) and list(b) == f32(g["Ks"]) and float(c.value) == f32(g["Ne"])[0], name
    # Object::set_col_*: only the multiplier of an EXISTING slot changes, the texels stay; a missing slot index is ignored
    o = api.Sphere((0, 0, 0), 1).set_material(0, Kd=api.Texture((1, 1, 1), np.ones((2, 2, 3), np.float32)), Ks=api.Texture(0.5), Ne=api.Texture(9.0))
    o.set_preset("gold_ngan", 0).set_preset("chrome", 3)
    assert o.materials[0]["Kd"].values is not None and o.materials[0]["Kd"].multiplier == tuple(f32(gold["gold_ngan"]["Kd"]))
    assert o.materials[0]["Ne"].multiplier == tuple(f32(gold["gold_ngan"]["Ne"])) and 3 not in o.materials


def test_cpp_host_mirror_builds_and_fails_loudly_without_a_gpu(tmp_path):
    """host/ptb_raytracer.hpp + ptb_cli.cpp (the C++ side of the boundary) build against include/ptb200.h; without a device the
    driver reports the library's error and exits 1 (no CPU path), with or without --gpus."""
    import subprocess
    import torch
    cli = os.path.join(ROOT, "pathtracer_b200", "csrc", "ptb_cli")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "pathtracer_b200", "csrc"), "-s", "ptb_cli"])
    r = subprocess.run([cli], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr
    r = subprocess.run([cli, "--gpus", "0", "C1", str(tmp_path / "x.ppm")], capture_output=True, text=True)
    assert r.returncode == 2
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: tests/test_parity_gpu.py::test_cpp_cli_* cover the render")
    for extra in ([], ["--gpus", "2"]):
        r = subprocess.run([cli] + extra + ["C1", str(tmp_path / "x.ppm"), "32", "32", "1"], capture_output=True, text=True)
        assert r.returncode == 1 and "no CPU path" in r.stderr, r.stderr
    r = subprocess.run([cli, "--preset", "nope", "C1", str(tmp_path / "x.ppm")], capture_output=True, text=True)
    assert r.returncode == 1 and "unknown material preset" in r.stderr
