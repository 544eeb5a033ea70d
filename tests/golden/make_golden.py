#!/usr/bin/env python3
"""Generate the golden vectors under tests/golden/ from oracle/_ref — the REFERENCE's own sources
compiled headless by oracle/build_ref.py (only possible where PTB_REFERENCE_DIR names a checkout of the reference).

The fixtures pin oracle/port (and through it the CUDA path) to outputs of the reference itself:
  kat.npz        function-level known answers: inputs + reference outputs for every PTB_KAT_* block
  sceneio.npz    what the reference's own FILE READERS (load_image, Texture::loadColors/loadNormals, TriMesh::readOBJ/readOFF,
                 Raytracer::load_scene) leave in memory for the fixtures under tests/golden/assets/, and the reference's render of
                 the .scn fixtures loaded by its own load_scene (ids, image, ray counters)
  modes.npz      the reference's progressive renderer (Raytracer::render_image: sums, weights, display image, low-resolution preview,
                 after all passes and after a stop at 2) and its has_denoiser accumulation (means, albedo, normalImage)
  scene_<n>.npz  for five miniature versions of the BASELINE.json configurations and for the branching modes of getColor
                 (background photograph, ghost objects, fog: golden_scenes.BRANCH_SCENES): primary-hit object /
                 triangle ids and t (the picking query), the linear image (imagedouble), sample_count,
                 the 8-bit image and the ray counters of a single-thread render
Run:  python tests/golden/make_golden.py        (rewrites the .npz files; they are committed)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import ctypes as C  # noqa: E402
import json  # noqa: E402

import sceneio_cases as sio  # noqa: E402
from golden_scenes import ANIM_SCENES, BRANCH_SCENES, KAT_INPUTS, SCENES, STAT_SCENES  # noqa: E402
from oracles import ref_lib  # noqa: E402

from pathtracer_b200 import _abi, scenes  # noqa: E402


def render_scn_with_reference(R, RIO, name):
    """The reference's own load_scene + render_image_nopreviz + picking query on a .scn fixture (cwd = assets)."""
    ctx = C.c_void_p()
    R.check(R.create(0, C.byref(ctx)))
    cam, p = _abi.Camera(), _abi.Params()
    RIO.check(RIO.load_scene(ctx, name.encode(), None, C.byref(cam), C.byref(p)))
    R.check(R.commit(ctx), ctx)
    R.check(R.set_option(ctx, _abi.ORC_OPT_THREADS, 1), ctx)
    img, cnt, st = np.empty((p.H, p.W, 3), np.float32), np.empty((p.H, p.W), np.float32), _abi.Stats()
    u8 = np.empty((p.H, p.W, 3), np.uint8)
    R.check(R.render(ctx, C.byref(cam), C.byref(p), _abi.fptr(img), _abi.fptr(cnt), u8.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(st)), ctx)
    obj, tri, t = np.empty((p.H, p.W), np.int32), np.empty((p.H, p.W), np.int32), np.empty((p.H, p.W), np.float32)
    i32 = C.POINTER(C.c_int32)
    R.check(R.primary_ids(ctx, C.byref(cam), p.W, p.H, obj.ctypes.data_as(i32), tri.ctypes.data_as(i32), _abi.fptr(t)), ctx)
    R.destroy(ctx)
    return dict(obj=obj.astype(np.int16), tri=tri, t=t, imagedouble=img, sample_count=cnt, image=u8, rays=np.array([st.rays_closest, st.rays_shadow], np.int64))


def sceneio_golden(R):
    RIO = sio.sceneio_of(R.cdll, "ref_")
    out, meta = {}, {}
    with sio.in_assets():
        for n in sio.IMAGES:
            out[f"image/{n}"] = sio.dump_image(RIO, n)
        for n, k in sio.TEXTURES:
            out[f"texture/{n}/{k}"] = sio.dump_texture(RIO, n, k)
        for n, lt in sio.MESHES:
            d = sio.dump_mesh(RIO, n, lt)
            for key in ("vertices", "normals", "uvs", "vertex_colors", "tri"):
                out[f"mesh/{n}/{lt}/{key}"] = d[key]
            meta[f"mesh/{n}/{lt}"] = {"n_groups": d["n_groups"], "groups": d["groups"], "slots": {str(g): {str(k): v for k, v in per.items()} for g, per in d["slots"].items()}}
        for n in sio.YARNS:
            out[f"yarn/{n}"] = sio.dump_yarn(RIO, n)
        for n in sio.SCENES:
            meta[f"scn/{n}"] = sio.dump_scn(RIO, n)
        for n in sio.RENDER_SCENES:
            for k, v in render_scn_with_reference(R, RIO, n).items():
                out[f"render/{n}/{k}"] = v
    out["meta_json"] = np.frombuffer(json.dumps(meta, sort_keys=True).encode(), np.uint8)
    np.savez_compressed(os.path.join(HERE, "sceneio.npz"), **out)
    print("sceneio.npz:", len(out), "arrays")


def modes_golden(R):
    """The reference's progressive renderer (render_image) and its has_denoiser accumulation on tests/parity_cases.mode_scene."""
    from parity_cases import mode_scene
    rt = mode_scene(R).commit()
    rt.set_option(_abi.ORC_OPT_THREADS, 1)
    out = {}
    rt.render_image()
    for k in ("imagedouble", "sample_count", "image", "imagedouble_lowres"):
        out[f"progressive/{k}"] = getattr(rt, k).copy()

    def stop_after_two(r):
        r.stopped = r.current_nb_rays >= 2
    rt.render_image(on_pass=stop_after_two)
    for k in ("imagedouble", "sample_count", "image", "imagedouble_lowres"):
        out[f"progressive2/{k}"] = getattr(rt, k).copy()
    rt.render_denoiser_inputs()
    for k in ("imagedouble", "sample_count", "albedoImage", "normalImage"):
        out[f"denoiser/{k}"] = getattr(rt, k).copy()
    np.savez_compressed(os.path.join(HERE, "modes.npz"), **out)
    print("modes.npz:", {k: v.shape for k, v in out.items()})


def main():
    R = ref_lib()
    assert R is not None, "oracle/_ref is not built (set PTB_REFERENCE_DIR to a checkout of the reference)"
    only = [a.split("=", 1)[1].split(",") for a in sys.argv if a.startswith("--only=")]      # --only=NGAN,C1: just these scene fixtures
    if "--sceneio-only" in sys.argv:
        sceneio_golden(R)
        return
    if not only:
        sceneio_golden(R)
        modes_golden(R)
    todo = {**BRANCH_SCENES, **STAT_SCENES, **ANIM_SCENES}
    if "--new-only" not in sys.argv:
        todo.update(SCENES)
    if only:
        todo = {k: v for k, v in {**todo, **SCENES}.items() if k in only[0]}
    if "--new-only" not in sys.argv and not only:
        rt = scenes.config_C4(R, 32, 32, 1, nv=10).commit()   # any committed scene with a MERL table
        out = {}
        for which, (inp, kw) in KAT_INPUTS().items():
            out[f"in_{which}"] = inp
            out[f"out_{which}"] = rt.kat(which, inp, **kw)
        np.savez_compressed(os.path.join(HERE, "kat.npz"), **out)
    for name, mk in todo.items():
        rt = mk(R).commit()
        rt.set_option(_abi.ORC_OPT_THREADS, 1)
        obj, tri, t = rt.primary_ids()
        img = rt.render_image_nopreviz().copy()
        np.savez_compressed(os.path.join(HERE, f"scene_{name}.npz"), obj=obj.astype(np.int16), tri=tri, t=t, imagedouble=img,
                            sample_count=rt.sample_count, image=rt.image, rays=np.array([rt.stats["rays_closest"], rt.stats["rays_shadow"]], np.int64))
        print(name, img.shape, float(img.mean()), rt.stats["rays_closest"], rt.stats["rays_shadow"])


if __name__ == "__main__":
    main()
