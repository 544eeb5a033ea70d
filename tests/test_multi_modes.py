"""The denoiser-input and progressive renderers sharded by image tiles, like render_image_nopreviz: a shard renders the tiles it owns
(ptb_params shard_rank / shard_count / tile_size), a group renders one frame on all the GPUs of the process (ptb_group_*), and one
process per GPU renders it over NCCL after multi.init_comm (ptb_*_sharded).  Per-(pixel, sample) random streams make every form
draw the same samples as one GPU, so the results must match it up to the order of float additions.

The devsim cases pin the shard semantics on the CPU; the GPU cases run the kernels, the gather and both host mirrors."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
from parity_cases import mode_scene

from pathtracer_b200 import _abi, scenes
from pathtracer_b200._abi import fptr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RAD = dict(rtol=2e-5, atol=1e-3)          # radiance, as tests/test_parity_gpu.py::test_group_render_equals_single


# ---- the tile rule of ptb_scene.h (shard_tile_shift, tile_logical), restated ----------------------------------------------
def tile_shift(tiles_x, count):
    if count <= 1 or tiles_x <= 1:
        return 0
    for s in range(1, count + 1):
        if math.gcd((tiles_x + s) % count, count) == 1:
            return s % tiles_x
    return 1 % tiles_x


def owner_map(W, H, tile, count):
    """(H, W) shard that owns each pixel, in the output row order (camera row i lands in row H-1-i)."""
    tiles_x = -(-W // tile)
    shift = tile_shift(tiles_x, count)
    ty, tx = np.meshgrid(np.arange(H) // tile, np.arange(W) // tile, indexing="ij")
    logical = ty * tiles_x + (tx + ty * shift) % tiles_x
    return np.flipud(logical % count)


# ---- direct calls of the C-ABI ------------------------------------------------------------------------------------------
def denoiser(L, ctx, rt, p, call="render_denoiser_inputs", handle=None):
    o = {k: np.full((rt.H, rt.W, 3), -7, np.float32) for k in ("img", "albedo", "normal", "fhn")}
    o["cnt"] = np.full((rt.H, rt.W), -7, np.float32)
    st, cam = _abi.Stats(), rt.cam.c_struct()
    h = handle if handle is not None else ctx
    rc = getattr(L, call)(h, C.byref(cam), C.byref(p), fptr(o["img"]), fptr(o["cnt"]), fptr(o["albedo"]), fptr(o["normal"]), fptr(o["fhn"]), C.byref(st))
    assert rc == _abi.OK, (L.group_last_error(h) if call.startswith("group") else L.last_error(ctx))
    o["stats"] = st.as_dict()
    return o


def prog_read(L, handle, rt, call="progressive_read"):
    o = {"img": np.empty((rt.H, rt.W, 3), np.float32), "cnt": np.empty((rt.H, rt.W), np.float32),
         "u8": np.empty((rt.H, rt.W, 3), np.uint8), "lowres": np.empty((-(-rt.H // 16), -(-rt.W // 16), 3), np.float32)}
    n = C.c_int32(0)
    rc = getattr(L, call)(handle, fptr(o["img"]), fptr(o["cnt"]), o["u8"].ctypes.data_as(C.POINTER(C.c_uint8)), fptr(o["lowres"]), C.byref(n))
    assert rc == _abi.OK, rc
    o["n"] = n.value
    return o


def prog_pass(L, handle, n_spp, call="progressive_pass"):
    st = _abi.Stats()
    assert getattr(L, call)(handle, n_spp, C.byref(st)) == _abi.OK
    return st.as_dict()


STAT_KEYS = ("samples", "rays_closest", "rays_shadow")


def check_denoiser_shards(L, mk, k, tile, exact):
    """Shards 0..k-1 merged by owner == the whole frame."""
    whole_rt = mk(L).commit()
    whole = denoiser(L, whole_rt._ctx, whole_rt, whole_rt.params())
    own = owner_map(whole_rt.W, whole_rt.H, tile, k)
    merged = {key: np.zeros_like(whole[key]) for key in ("img", "cnt", "albedo", "normal", "fhn")}
    tot = dict.fromkeys(STAT_KEYS, 0)
    for r in range(k):
        s = denoiser(L, whole_rt._ctx, whole_rt, whole_rt.params(r, k, tile))
        mask = s["cnt"] > 0
        assert np.array_equal(mask, own == r), f"shard {r} of {k}: the pixels with samples are not its tiles"
        for key in merged:
            merged[key][mask] = s[key][mask]
        for key in STAT_KEYS:
            tot[key] += s["stats"][key]
    assert np.array_equal(merged["cnt"], whole["cnt"]) and (whole["cnt"] == whole_rt.nrays).all()
    for key in STAT_KEYS:
        assert tot[key] == whole["stats"][key], key
    cmp = (lambda a, b, **kw: np.array_equal(a, b, equal_nan=True)) if exact else (lambda a, b, **kw: np.allclose(a, b, equal_nan=True, **kw))
    assert cmp(merged["img"], whole["img"], **RAD) and cmp(merged["albedo"], whole["albedo"], rtol=2e-5, atol=1e-5)
    assert cmp(merged["fhn"], whole["fhn"], rtol=0, atol=1e-5)
    assert np.array_equal(np.isnan(merged["normal"]), np.isnan(whole["normal"]))
    assert cmp(merged["normal"], whole["normal"], rtol=0, atol=1e-5)
    whole_rt.close()


def check_progressive_shards(L, mk, k, tile, steps=(2, 4)):
    """Progressive sessions of shards 0..k-1, each on a context of its own, summed == the whole-frame session."""
    rts = [mk(L).commit() for _ in range(k + 1)]
    cam = rts[0].cam.c_struct()
    for r, rt in enumerate(rts):
        p = rt.params() if r == k else rt.params(r, k, tile)
        assert L.progressive_begin(rt._ctx, C.byref(cam), C.byref(p)) == _abi.OK
    tot = [dict.fromkeys(STAT_KEYS, 0) for _ in rts]
    for n_spp in steps:            # the passes of the sessions interleave
        for r, rt in enumerate(rts):
            st = prog_pass(L, rt._ctx, n_spp)
            for key in STAT_KEYS:
                tot[r][key] += st[key]
    outs = [prog_read(L, rt._ctx, rt) for rt in rts]
    whole, shards = outs[k], outs[:k]
    for r, s in enumerate(shards):
        assert s["n"] == sum(steps) == rts[0].nrays
        assert (s["cnt"][owner_map(rts[0].W, rts[0].H, tile, k) == r] > 0).all(), f"shard {r}: a pixel of its tiles has no sample"
    for key, tol in (("img", RAD), ("cnt", dict(rtol=2e-5, atol=1e-6)), ("lowres", dict(rtol=2e-5, atol=1e-3))):
        assert np.allclose(sum(s[key] for s in shards), whole[key], **tol), key
    for key in STAT_KEYS:
        assert sum(t[key] for t in tot[:k]) == tot[k][key], key
    for rt in rts:
        rt.close()


# ---- CPU: the shard semantics on tests/devsim -----------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 3])
def test_denoiser_input_shards_merge_to_the_whole_frame_devsim(devsim, k):
    check_denoiser_shards(devsim, mode_scene, k, 16, exact=True)


@pytest.mark.parametrize("k", [2, 3])
def test_progressive_shards_sum_to_the_whole_frame_devsim(devsim, k):
    check_progressive_shards(devsim, mode_scene, k, 16)


# ---- GPU: one device ----------------------------------------------------------------------------------------------------
W, H, SPP = 256, 192, 4


def mk_gpu(L):
    return mode_scene(L, W, H, SPP)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3])
def test_denoiser_input_shards_merge_to_the_whole_frame(gpu, k):
    check_denoiser_shards(gpu, mk_gpu, k, 32, exact=False)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3])
def test_progressive_shards_sum_to_the_whole_frame(gpu, k):
    check_progressive_shards(gpu, mk_gpu, k, 32, steps=(1, 2, 1))


def n_gpus():
    import torch
    return min(torch.cuda.device_count(), 8)


class GroupLib:
    """The product library with `create` / `commit` / `destroy` going to a ptb_group of `devices` (a group of one on a one-GPU box):
    a Raytracer built on it hands its scene to the group's leader."""

    def __init__(self, lib, devices):
        self._lib, self.devices, self.group = lib, list(devices), None

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def create(self, device, out):
        g = C.c_void_p()
        rc = self._lib.group_create((C.c_int * len(self.devices))(*self.devices), len(self.devices), C.byref(g))
        if rc == _abi.OK:
            self.group = g
            out._obj.value = self._lib.group_ctx(g, 0)
        return rc

    def commit(self, ctx):
        return self._lib.group_commit(self.group)

    def destroy(self, ctx):
        self._lib.group_destroy(self.group)
        self.group = None


def assert_denoiser_equal(a, b):
    assert np.allclose(a["img"], b["img"], **RAD) and np.array_equal(a["cnt"], b["cnt"])
    assert np.allclose(a["albedo"], b["albedo"], rtol=2e-5, atol=1e-5)
    assert np.allclose(a["fhn"], b["fhn"], rtol=0, atol=1e-5, equal_nan=True)
    assert np.array_equal(np.isnan(a["normal"]), np.isnan(b["normal"]))


def assert_progressive_equal(a, b):
    assert a["n"] == b["n"]
    assert np.allclose(a["img"], b["img"], **RAD) and np.allclose(a["cnt"], b["cnt"], rtol=2e-5, atol=1e-6)
    assert np.allclose(a["lowres"], b["lowres"], rtol=2e-5, atol=1e-3)
    assert (np.abs(a["u8"].astype(int) - b["u8"].astype(int)) <= 1).all()


@pytest.mark.gpu
def test_group_modes_equal_a_single_context(gpu):
    """ptb_group_render_denoiser_inputs and a group progressive session (read after 3 passes, then after 8) == one context."""
    gl = GroupLib(gpu, range(n_gpus()))
    one, grp = mk_gpu(gpu).commit(), mk_gpu(gl).commit()
    ref = denoiser(gpu, one._ctx, one, one.params())
    got = denoiser(gl, grp._ctx, grp, grp.params(), call="group_render_denoiser_inputs", handle=gl.group)
    assert_denoiser_equal(got, ref)
    for key in STAT_KEYS:
        assert got["stats"][key] == ref["stats"][key], key
    assert got["stats"]["samples"] == W * H * SPP
    one.nrays = grp.nrays = 10
    cam, p = one.cam.c_struct(), one.params()
    assert gpu.progressive_begin(one._ctx, C.byref(cam), C.byref(p)) == _abi.OK
    assert gpu.group_progressive_begin(gl.group, C.byref(cam), C.byref(p)) == _abi.OK
    for n_spp, times in ((1, 3), (5, 1)):       # a read after 3 passes, then after 8: a gather that adds into a rank's sums counts twice
        for _ in range(times):
            a = prog_pass(gpu, one._ctx, n_spp)
            b = prog_pass(gpu, gl.group, n_spp, call="group_progressive_pass")
            for key in STAT_KEYS:
                assert a[key] == b[key], key
        assert_progressive_equal(prog_read(gpu, gl.group, grp, call="group_progressive_read"), prog_read(gpu, one._ctx, one))
    one.close(); grp.close()


@pytest.mark.gpu
def test_group_modes_repose_a_keyframed_scene(gpu):
    """set_frame between two group renders re-poses every device (as ptb_group_render does) == one context at that frame."""
    gl = GroupLib(gpu, range(n_gpus()))
    mk = lambda L: scenes.config_anim(L, W, H, SPP, frame=0)
    one, grp = mk(gpu).commit(), mk(gl).commit()
    denoiser(gl, grp._ctx, grp, grp.params(), call="group_render_denoiser_inputs", handle=gl.group)
    one.set_frame(5); grp.set_frame(5)
    ref = denoiser(gpu, one._ctx, one, one.params())
    assert_denoiser_equal(denoiser(gl, grp._ctx, grp, grp.params(), call="group_render_denoiser_inputs", handle=gl.group), ref)
    one.set_frame(8); grp.set_frame(8)
    cam, p = one.cam.c_struct(), one.params()
    assert gpu.progressive_begin(one._ctx, C.byref(cam), C.byref(p)) == _abi.OK
    assert gpu.group_progressive_begin(gl.group, C.byref(cam), C.byref(p)) == _abi.OK
    prog_pass(gpu, one._ctx, 2); prog_pass(gpu, gl.group, 2, call="group_progressive_pass")
    assert_progressive_equal(prog_read(gpu, gl.group, grp, call="group_progressive_read"), prog_read(gpu, one._ctx, one))
    one.close(); grp.close()


@pytest.mark.gpu
def test_raytracer_with_devices_renders_both_modes_on_all_of_them(gpu):
    """Raytracer(devices=[...]).render_denoiser_inputs() / .render_image() go through the group: stats of every device, one GPU's result."""
    n = n_gpus()
    one, grp = mk_gpu(gpu), mk_gpu(gpu)
    grp.devices = list(range(n)) if n > 1 else [0]
    one.commit(); grp.commit()
    assert (grp._group is not None) == (n > 1)
    one.render_denoiser_inputs(); grp.render_denoiser_inputs()
    assert grp.stats["samples"] == W * H * SPP and grp.stats["rays_closest"] == one.stats["rays_closest"]
    assert np.allclose(grp.imagedouble, one.imagedouble, **RAD) and np.array_equal(grp.sample_count, one.sample_count)
    assert np.allclose(grp.albedoImage, one.albedoImage, rtol=2e-5, atol=1e-5)
    stop = lambda rt: setattr(rt, "stopped", rt.current_nb_rays >= 3)      # on_pass keeps its meaning: the process decides between passes
    a, b = one.render_image(on_pass=stop).copy(), grp.render_image(on_pass=stop).copy()
    assert one.current_nb_rays == grp.current_nb_rays == 3 and grp.stats["samples"] == W * H * 3
    assert np.allclose(b, a, **RAD) and np.allclose(grp.imagedouble_lowres, one.imagedouble_lowres, rtol=2e-5, atol=1e-3)
    a, b = one.render_image(passes_per_call=3).copy(), grp.render_image(passes_per_call=3).copy()
    assert grp.current_nb_rays == SPP and np.allclose(b, a, **RAD) and np.allclose(grp.sample_count, one.sample_count, rtol=2e-5, atol=1e-6)
    one.close(); grp.close()


DRIVER = r'''
#include <cstdio>
#include <cstdlib>
#include "pathtracer_b200/host/ptb_raytracer.hpp"
static void put(const char* dir, const char* name, const std::vector<float>& v) {
    std::string path = std::string(dir) + "/" + name;
    FILE* f = fopen(path.c_str(), "wb");
    fwrite(v.data(), sizeof(float), v.size(), f);
    fclose(f);
}
int main(int argc, char** argv) {            // driver <n devices> <out dir>
    std::vector<int> devices;
    for (int i = 0; i < atoi(argv[1]); i++) devices.push_back(i);
    ptbhost::Raytracer rt(devices);
    rt.loadScene();
    rt.W = 160; rt.H = 96; rt.nrays = 4;
    try {
        rt.render_denoiser_inputs();
        put(argv[2], "d_img", rt.imagedouble); put(argv[2], "d_cnt", rt.sample_count); put(argv[2], "d_albedo", rt.albedoImage);
        printf("denoiser samples %llu\n", (unsigned long long)rt.stats.samples);
        rt.render_image([](ptbhost::Raytracer&) {}, 3);
        put(argv[2], "p_img", rt.imagedouble); put(argv[2], "p_cnt", rt.sample_count); put(argv[2], "p_lowres", rt.imagedouble_lowres);
        printf("progressive passes %d\n", rt.current_nb_rays);
    } catch (const ptbhost::Error& e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    return 0;
}
'''


@pytest.mark.gpu
def test_cpp_mirror_renders_both_modes_on_every_device(gpu, tmp_path):
    """ptb_raytracer.hpp with several devices routes render_denoiser_inputs() / render_image() through the group."""
    from pathtracer_b200.api import Raytracer
    n = n_gpus()
    src, exe = tmp_path / "driver.cpp", tmp_path / "driver"
    src.write_text(DRIVER)
    csrc = os.path.join(ROOT, "pathtracer_b200", "csrc")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", ROOT, "-o", str(exe), str(src), "-L", csrc, "-lptb200", f"-Wl,-rpath,{csrc}"])
    r = subprocess.run([str(exe), str(n), str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert f"denoiser samples {160 * 96 * 4}" in r.stdout and "progressive passes 4" in r.stdout
    rt = Raytracer(gpu).loadScene()
    rt.W, rt.H, rt.nrays = 160, 96, 4
    rt.render_denoiser_inputs()
    got = lambda name: np.fromfile(str(tmp_path / name), np.float32)
    near = lambda a, b: np.mean(~np.isclose(a, b.reshape(-1), rtol=1e-4, atol=1e-2)) < 1e-3     # the two camera set-ups may differ in the last bit
    assert np.array_equal(got("d_cnt"), rt.sample_count.reshape(-1))
    assert near(got("d_img"), rt.imagedouble) and near(got("d_albedo"), rt.albedoImage)
    rt.render_image(passes_per_call=3)
    assert near(got("p_img"), rt.imagedouble) and near(got("p_cnt"), rt.sample_count) and near(got("p_lowres"), rt.imagedouble_lowres)
    rt.close()


@pytest.mark.gpu
def test_mode_errors_are_refused_on_the_host(gpu):
    """Pass or read before begin, the wrong read for the session kind, a group call on a closed group: error codes, no launch."""
    rt = mk_gpu(gpu).commit()
    ctx, cam, p = rt._ctx, rt.cam.c_struct(), rt.params()
    n = C.c_int32(0)
    assert gpu.progressive_pass(ctx, 1, None) == _abi.ERR_STATE
    assert gpu.progressive_read(ctx, None, None, None, None, C.byref(n)) == _abi.ERR_STATE
    assert gpu.progressive_read_sharded(ctx, None, None, None, None, C.byref(n)) == _abi.ERR_STATE
    assert gpu.progressive_begin(ctx, C.byref(cam), C.byref(p)) == _abi.OK
    assert gpu.progressive_read_sharded(ctx, None, None, None, None, C.byref(n)) == _abi.ERR_STATE
    assert b"ptb_progressive_read" in gpu.last_error(ctx)
    assert gpu.progressive_begin_sharded(ctx, C.byref(cam), C.byref(p)) == _abi.OK
    assert gpu.progressive_read(ctx, None, None, None, None, C.byref(n)) == _abi.ERR_STATE
    assert b"ptb_progressive_read_sharded" in gpu.last_error(ctx)
    assert gpu.progressive_read_sharded(ctx, None, None, None, None, C.byref(n)) == _abi.OK and n.value == 0
    rt.close()
    gl = GroupLib(gpu, range(n_gpus()))
    grp = mk_gpu(gl).commit()
    g = gl.group
    assert gpu.group_progressive_pass(g, 1, None) == _abi.ERR_STATE
    assert gpu.group_progressive_read(g, None, None, None, None, C.byref(n)) == _abi.ERR_STATE
    assert b"before progressive_begin" in gpu.group_last_error(g)
    grp.close()
    assert gl.group is None
    assert gpu.group_progressive_pass(gl.group, 1, None) == _abi.ERR_INVALID
    assert gpu.group_progressive_read(gl.group, None, None, None, None, C.byref(n)) == _abi.ERR_INVALID
    assert gpu.group_progressive_begin(gl.group, C.byref(cam), C.byref(p)) == _abi.ERR_INVALID
    assert gpu.group_render_denoiser_inputs(gl.group, C.byref(cam), C.byref(p), None, None, None, None, None, None) == _abi.ERR_INVALID


# ---- GPU: one process per GPU over NCCL ---------------------------------------------------------------------------------
def _nccl_worker(rank, world, port_no, out_path):
    import sys
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port_no)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import pathtracer_b200
    from pathtracer_b200 import multi
    L = pathtracer_b200.load()
    rt = mode_scene(L, W, H, SPP)
    rt.device = rank
    rt.nrays = 10
    multi.init_comm(rt, rank, world)
    rt.commit()
    out = {}
    img = rt.render_denoiser_inputs()
    assert (img is None) == (rank != 0)
    if rank == 0:
        out.update(d_img=rt.imagedouble, d_cnt=rt.sample_count, d_albedo=rt.albedoImage, d_fhn=rt.first_hit_normal, d_normal=rt.normalImage)
    cam, p = rt.cam.c_struct(), rt.params()
    L.check(L.progressive_begin_sharded(rt._ctx, C.byref(cam), C.byref(p)), rt._ctx)
    for n_spp, times, tag in ((1, 3, "a"), (5, 1, "b")):     # read after 3 passes, then after 8
        for _ in range(times):
            L.check(L.progressive_pass(rt._ctx, n_spp, None), rt._ctx)
        got = rt.read_progressive()
        assert (got is None) == (rank != 0) and rt.current_nb_rays == (3 if tag == "a" else 8)
        if rank == 0:
            out.update({f"{tag}_img": rt.imagedouble, f"{tag}_cnt": rt.sample_count, f"{tag}_lowres": rt.imagedouble_lowres})
    try:
        rt.render_image(on_pass=lambda r: None)
        refused = False
    except _abi.PtbError:
        refused = True
    assert refused, "a stop decision cannot be taken by one process of several"
    got = rt.render_image(passes_per_call=4)
    assert rt.current_nb_rays == 10 and (got is None) == (rank != 0)
    if rank == 0:
        out.update(f_img=rt.imagedouble, f_cnt=rt.sample_count)
        np.savez(out_path, **out)
    dist.barrier()
    rt.close()
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_nccl_sharded_modes_equal_a_single_gpu(gpu, tmp_path, world):
    """2 and 4 ranks (as many as the box shows): denoiser inputs on rank 0 and a progressive session read twice mid-way == one GPU."""
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    out = str(tmp_path / "out.npz")
    mp.spawn(_nccl_worker, args=(world, 29700 + world + os.getpid() % 1000, out), nprocs=world, join=True)
    got = np.load(out)
    rt = mode_scene(gpu, W, H, SPP).commit()
    rt.render_denoiser_inputs()
    assert np.allclose(got["d_img"], rt.imagedouble, **RAD) and np.array_equal(got["d_cnt"], rt.sample_count)
    assert np.allclose(got["d_albedo"], rt.albedoImage, rtol=2e-5, atol=1e-5)
    assert np.allclose(got["d_fhn"], rt.first_hit_normal, rtol=0, atol=1e-5, equal_nan=True)
    assert np.array_equal(np.isnan(got["d_normal"]), np.isnan(rt.normalImage))
    rt.nrays = 10
    cam, p = rt.cam.c_struct(), rt.params()
    gpu.check(gpu.progressive_begin(rt._ctx, C.byref(cam), C.byref(p)), rt._ctx)
    for n_spp, times, tag in ((1, 3, "a"), (5, 1, "b")):
        for _ in range(times):
            gpu.check(gpu.progressive_pass(rt._ctx, n_spp, None), rt._ctx)
        rt.read_progressive()
        assert np.allclose(got[f"{tag}_img"], rt.imagedouble, **RAD) and np.allclose(got[f"{tag}_cnt"], rt.sample_count, rtol=2e-5, atol=1e-6), tag
        assert np.allclose(got[f"{tag}_lowres"], rt.imagedouble_lowres, rtol=2e-5, atol=1e-3), tag
    rt.render_image(passes_per_call=4)
    assert np.allclose(got["f_img"], rt.imagedouble, **RAD) and np.allclose(got["f_cnt"], rt.sample_count, rtol=2e-5, atol=1e-6)
    rt.close()
