"""ctypes mirror of include/ptb200.h.

`Lib(cdll, prefix)` binds the C-ABI entry points of one shared library.  The product binds
libptb200.so with prefix "ptb_" (see pathtracer_b200/__init__.py); the tests bind the CPU checkers
under oracle/ with their own prefixes through the same class, so one scene description can be fed
to each implementation unchanged.
"""
import ctypes as C

import numpy as np

OK = 0
ERR_INVALID, ERR_STATE, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED = -1, -2, -3, -4, -5
SLOT_KD, SLOT_KS, SLOT_NE, SLOT_TRANSP, SLOT_REFR, SLOT_NORMAL, SLOT_ALPHA, SLOT_KSUB = (1 << i for i in range(8))
OBJ_MIRROR, OBJ_FLIP_NORMALS, OBJ_FLAT_NORMALS, OBJ_GHOST, OBJ_DISPLAY_EDGES = 1, 2, 4, 8, 16
BRDF_PHONG, BRDF_MERL = 0, 1
KEY_SCALE, KEY_TRANSLATION, KEY_ROTATION = 0, 1, 2
OPT_COUNT_TRAVERSAL, OPT_POOL_PATHS, OPT_TIME_KERNELS, OPT_REFILL_BELOW, OPT_TRACE_BLOCKS, OPT_TRI_FRACTION, OPT_TRI_MIN_PCT = 1, 2, 3, 4, 5, 6, 7
OPT_PIPES = 9   # 8 is retired (terminal-hit compaction, removed): do not reuse
OPT_BUILD_THREADS, OPT_STACK_LIMIT = 10, 11
COMM_ID_BYTES = 128
KERNEL_NAMES = ["raygen", "extend", "shade", "shadow", "splat"]
ORC_OPT_THREADS = 100
(KAT_PCG32, KAT_LATTICE, KAT_CAMERA, KAT_RANDOM_COS, KAT_RANDOM_PHONG, KAT_PHONG_EVAL, KAT_MERL_EVAL,
 KAT_FAST_EXP, KAT_FAST_NORMALIZE, KAT_RANDOM_PER_PIXEL, KAT_FILTER_RATIO, KAT_MERL_INDEX) = range(1, 13)
# KAT 13 is retired (the half-factor node test, removed): do not reuse
KAT_SHAPES = {  # which -> (n_in, n_out)
    KAT_PCG32: (2, 4), KAT_LATTICE: (1, 2), KAT_CAMERA: (6, 6), KAT_RANDOM_COS: (5, 3),
    KAT_RANDOM_PHONG: (6, 3), KAT_PHONG_EVAL: (18, 3), KAT_MERL_EVAL: (9, 3), KAT_FAST_EXP: (1, 1),
    KAT_FAST_NORMALIZE: (3, 3), KAT_RANDOM_PER_PIXEL: (1, 2), KAT_FILTER_RATIO: (3, 1), KAT_MERL_INDEX: (6, 2),
}

_fp = C.POINTER(C.c_float)


class Tex(C.Structure):
    _fields_ = [("texels", _fp), ("W", C.c_int32), ("H", C.c_int32), ("mult", C.c_float * 3)]


class Material(C.Structure):
    _fields_ = [("present", C.c_uint32), ("Kd", Tex), ("Ks", Tex), ("Ne", Tex), ("transp", Tex),
                ("refr", Tex), ("normal", Tex), ("alpha", Tex), ("Ksub", Tex)]


class Fog(C.Structure):
    _fields_ = [("density", C.c_float), ("absorption", C.c_float), ("density_decay", C.c_float), ("absorption_decay", C.c_float),
                ("type", C.c_int32), ("phase_type", C.c_int32), ("phase_aniso", C.c_float)]


class Xform(C.Structure):
    _fields_ = [("scale", C.c_float), ("rotation", C.c_float * 9), ("rotation_center", C.c_float * 3),
                ("translation", C.c_float * 3)]


class Mesh(C.Structure):
    _fields_ = [("vertices", _fp), ("n_vertices", C.c_int32), ("normals", _fp), ("n_normals", C.c_int32),
                ("uvs", _fp), ("n_uvs", C.c_int32), ("tri", C.POINTER(C.c_int32)), ("n_tri", C.c_int32),
                ("scaling", C.c_float), ("offset", C.c_float * 3), ("center", C.c_int32)]


class PointSetDesc(C.Structure):
    _fields_ = [("points", _fp), ("normals", _fp), ("radii", _fp), ("colors", _fp), ("n", C.c_int32)]


class YarnsDesc(C.Structure):
    _fields_ = [("A", _fp), ("B", _fp), ("R", _fp), ("n", C.c_int32)]


class Camera(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("direction", C.c_float * 3), ("up", C.c_float * 3),
                ("fov", C.c_float), ("focus_distance", C.c_float), ("aperture", C.c_float)]


class Params(C.Structure):
    _fields_ = [("W", C.c_int32), ("H", C.c_int32), ("nrays", C.c_int32), ("nb_bounces", C.c_int32),
                ("sigma_filter", C.c_float), ("gamma", C.c_float), ("seed", C.c_uint32),
                ("shard_rank", C.c_int32), ("shard_count", C.c_int32), ("tile_size", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("rays_closest", C.c_uint64), ("rays_shadow", C.c_uint64),
                ("node_visits", C.c_uint64), ("tri_tests", C.c_uint64), ("ms_device", C.c_double),
                ("ms_wall", C.c_double), ("kernel_launches", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class SceneInfo(C.Structure):
    _fields_ = [("n_triangles", C.c_int64), ("n_bvh_nodes", C.c_int64), ("bytes_nodes", C.c_int64),
                ("bytes_triangles", C.c_int64), ("bytes_attributes", C.c_int64), ("bytes_textures", C.c_int64),
                ("n_objects", C.c_int32), ("bvh_depth", C.c_int32), ("ms_bvh_build", C.c_double),
                ("ms_upload", C.c_double), ("ms_refit", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class KernelTimes(C.Structure):
    _fields_ = [("ms", C.c_double * 5), ("launches", C.c_uint64 * 5), ("items", C.c_uint64 * 5), ("node_visits", C.c_uint64 * 5),
                ("tri_tests", C.c_uint64 * 5)]

    def as_dict(self):
        return {n: {k: getattr(self, k)[i] for k, _ in self._fields_} for i, n in enumerate(KERNEL_NAMES)}


# every symbol include/ptb200.h declares (tests check the product library exports all of them)
SYMBOLS = ["create", "destroy", "last_error", "version", "add_sphere", "add_plane", "add_cylinder", "add_pointset", "add_yarns", "add_mesh",
           "set_group_material", "set_brdf", "add_merl", "set_envmap", "set_light", "set_fog", "set_background", "set_keyframes", "set_frame", "commit", "render",
           "render_accum", "resolve", "shard_pack_size", "shard_pack", "shard_unpack_add", "primary_ids",
           "set_option", "get_scene_info", "kat", "get_kernel_times", "render_denoiser_inputs", "progressive_begin", "progressive_pass",
           "progressive_read"]
# material presets, multi-GPU and host-buffer entry points: the CUDA library only (the CPU checkers under oracle/ and tests/devsim do not have them)
MULTI_SYMBOLS = ["preset_count", "preset_get", "preset_find", "comm_unique_id", "comm_init", "comm_destroy", "render_sharded", "resolve_last", "group_create", "group_destroy", "group_last_error",
                 "group_size", "group_ctx", "group_commit", "group_set_option", "group_render", "pin_host_buffer", "unpin_host_buffer",
                 "render_denoiser_inputs_sharded", "progressive_begin_sharded", "progressive_read_sharded", "group_render_denoiser_inputs",
                 "group_progressive_begin", "group_progressive_pass", "group_progressive_read"]


# ---- include/ptb_sceneio.h -------------------------------------------------------------------------
PATH_MAX = 512
KIND_KD, KIND_NORMAL, KIND_SUBSURF, KIND_KS, KIND_ALPHA, KIND_NE, KIND_TRANSP, KIND_REFR = range(8)
N_KINDS = 8
SCN_MESH, SCN_SPHERE, SCN_PLANE, SCN_POINTSET = range(4)


class Slot(C.Structure):
    _fields_ = [("file", C.c_char * PATH_MAX), ("mult", C.c_float * 3)]


class MeshfileInfo(C.Structure):
    _fields_ = [("vertices", _fp), ("n_vertices", C.c_int32), ("normals", _fp), ("n_normals", C.c_int32), ("uvs", _fp), ("n_uvs", C.c_int32),
                ("vertex_colors", _fp), ("n_vertex_colors", C.c_int32), ("tri", C.POINTER(C.c_int32)), ("n_tri", C.c_int32),
                ("n_groups", C.c_int32), ("has_materials", C.c_int32)]


class ScnHeader(C.Structure):
    _fields_ = [("W", C.c_int32), ("H", C.c_int32), ("nrays", C.c_int32), ("nbframes", C.c_int32), ("nb_bounces", C.c_int32),
                ("has_denoiser", C.c_int32), ("is_lenticular", C.c_int32), ("n_objects", C.c_int32), ("cam", Camera),
                ("sigma_filter", C.c_float), ("gamma", C.c_float), ("intensite_lumiere", C.c_float), ("envmap_intensity", C.c_float),
                ("fog_density", C.c_float), ("fog_absorption", C.c_float), ("fog_density_decay", C.c_float), ("fog_absorption_decay", C.c_float),
                ("fog_type", C.c_int32), ("fog_phase_type", C.c_int32), ("double_frustum_start_t", C.c_float), ("background", C.c_char * PATH_MAX)]


class ScnObject(C.Structure):
    _fields_ = [("type", C.c_int32), ("name", C.c_char * PATH_MAX), ("miroir", C.c_int32), ("ghost", C.c_int32), ("display_edges", C.c_int32),
                ("interp_normals", C.c_int32), ("flip_normals", C.c_int32), ("n_keyframes", C.c_int32), ("xform", Xform),
                ("n_slots", C.c_int32 * N_KINDS), ("is_envmap", C.c_int32), ("envmap", C.c_char * PATH_MAX), ("O", C.c_float * 3), ("R", C.c_float),
                ("A", C.c_float * 3), ("N", C.c_float * 3), ("is_centered", C.c_int32), ("has_csv", C.c_int32), ("csv_file", C.c_char * PATH_MAX)]


# every symbol include/ptb_sceneio.h declares
SCENEIO_SYMBOLS = ["sceneio_last_error", "image_load", "image_free", "texture_load", "meshfile_read", "meshfile_free", "meshfile_get",
                   "meshfile_group_name", "meshfile_group_slot", "yarnfile_read", "yarnfile_free", "scn_load", "scn_free", "scn_get_header", "scn_get_object", "scn_get_slot", "scn_get_keyframes",
                   "scn_save", "load_scene"]


class PtbError(RuntimeError):
    pass


class SceneIO:
    """Bound entry points of include/ptb_sceneio.h (host-side readers; they need no GPU)."""

    def __init__(self, cdll, prefix="ptb_"):
        vp, ip32 = C.c_void_p, C.POINTER(C.c_int32)
        sig = {
            "sceneio_last_error": (C.c_char_p, []),
            "image_load": (C.c_int, [C.c_char_p, C.POINTER(C.POINTER(C.c_uint8)), ip32, ip32]),
            "image_free": (None, [vp]),
            "texture_load": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(_fp), ip32, ip32]),
            "meshfile_read": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(vp)]),
            "meshfile_free": (None, [vp]),
            "meshfile_get": (C.c_int, [vp, C.POINTER(MeshfileInfo)]),
            "meshfile_group_name": (C.c_int, [vp, C.c_int, C.c_char_p]),
            "meshfile_group_slot": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(Slot)]),
            "yarnfile_read": (C.c_int, [C.c_char_p, C.POINTER(_fp), C.POINTER(_fp), C.POINTER(_fp), ip32]),
            "yarnfile_free": (None, [vp]),
            "scn_load": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(vp)]),
            "scn_free": (None, [vp]),
            "scn_get_header": (C.c_int, [vp, C.POINTER(ScnHeader)]),
            "scn_get_object": (C.c_int, [vp, C.c_int, C.POINTER(ScnObject)]),
            "scn_get_slot": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.POINTER(Slot)]),
            "scn_get_keyframes": (C.c_int, [vp, C.c_int, C.c_int, _fp, _fp, C.c_int]),
            "scn_save": (C.c_int, [vp, C.c_char_p]),
            "load_scene": (C.c_int, [vp, C.c_char_p, C.c_char_p, C.POINTER(Camera), C.POINTER(Params)]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(cdll, prefix + name)
            fn.restype, fn.argtypes = res, args
            setattr(self, name, fn)

    def check(self, rc):
        if rc != OK:
            msg = self.sceneio_last_error()
            raise PtbError(f"scene reader failed rc={rc}: {msg.decode() if msg else ''}")


class Lib:
    """Bound entry points of one implementation of the ptb200 C-ABI."""

    def __init__(self, cdll, prefix="ptb_"):
        self.cdll, self.prefix = cdll, prefix
        vp, ip = C.c_void_p, C.POINTER(C.c_int)
        sig = {
            "create": (C.c_int, [C.c_int, C.POINTER(vp)]),
            "destroy": (None, [vp]),
            "last_error": (C.c_char_p, [vp]),
            "version": (C.c_char_p, []),
            "add_sphere": (C.c_int, [vp, _fp, C.c_float, C.POINTER(Xform), C.c_int, ip]),
            "add_plane": (C.c_int, [vp, _fp, _fp, C.POINTER(Xform), C.c_int, ip]),
            "add_cylinder": (C.c_int, [vp, _fp, _fp, C.c_float, C.POINTER(Xform), C.c_int, ip]),
            "add_pointset": (C.c_int, [vp, C.POINTER(PointSetDesc), C.POINTER(Xform), C.c_int, ip]),
            "add_yarns": (C.c_int, [vp, C.POINTER(YarnsDesc), C.POINTER(Xform), C.c_int, ip]),
            "add_mesh": (C.c_int, [vp, C.POINTER(Mesh), C.POINTER(Xform), C.c_int, ip]),
            "set_group_material": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(Material)]),
            "set_brdf": (C.c_int, [vp, C.c_int, C.c_int, C.c_int]),
            "add_merl": (C.c_int, [vp, C.POINTER(C.c_double), ip]),
            "set_envmap": (C.c_int, [vp, C.POINTER(C.c_uint8), C.c_int, C.c_int]),
            "set_light": (C.c_int, [vp, C.c_float, C.c_float]),
            "set_fog": (C.c_int, [vp, C.POINTER(Fog)]),
            "set_background": (C.c_int, [vp, _fp, C.c_int, C.c_int]),
            "set_keyframes": (C.c_int, [vp, C.c_int, C.c_int, _fp, _fp, C.c_int]),
            "set_frame": (C.c_int, [vp, C.c_float]),
            "commit": (C.c_int, [vp]),
            "render": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params), _fp, _fp, C.POINTER(C.c_uint8), C.POINTER(Stats)]),
            "render_accum": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params), vp, C.POINTER(Stats)]),
            "resolve": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_float, _fp, _fp, C.POINTER(C.c_uint8)]),
            "shard_pack_size": (C.c_int, [C.POINTER(Params), C.c_int, C.POINTER(C.c_int64)]),
            "shard_pack": (C.c_int, [vp, C.POINTER(Params), C.c_int, vp, vp]),
            "shard_unpack_add": (C.c_int, [vp, C.POINTER(Params), C.c_int, vp, vp]),
            "primary_ids": (C.c_int, [vp, C.POINTER(Camera), C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32), _fp]),
            "set_option": (C.c_int, [vp, C.c_int, C.c_int64]),
            "get_scene_info": (C.c_int, [vp, C.POINTER(SceneInfo)]),
            "get_kernel_times": (C.c_int, [vp, C.POINTER(KernelTimes)]),
            "render_denoiser_inputs": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params), _fp, _fp, _fp, _fp, _fp, C.POINTER(Stats)]),
            "progressive_begin": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params)]),
            "progressive_pass": (C.c_int, [vp, C.c_int, C.POINTER(Stats)]),
            "progressive_read": (C.c_int, [vp, _fp, _fp, C.POINTER(C.c_uint8), _fp, C.POINTER(C.c_int32)]),
            "kat": (C.c_int, [vp, C.c_int, C.POINTER(Camera), C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int,
                              C.POINTER(C.c_double), C.c_int]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(cdll, prefix + name)  # AttributeError if the symbol is missing: loud by design
            fn.restype, fn.argtypes = res, args
            setattr(self, name, fn)
        u8p = C.POINTER(C.c_uint8)
        multi = {
            "preset_count": (C.c_int, []),
            "preset_get": (C.c_int, [C.c_int, C.POINTER(C.c_char_p), _fp, _fp, _fp]),
            "preset_find": (C.c_int, [C.c_char_p]),
            "comm_unique_id": (C.c_int, [vp]),
            "comm_init": (C.c_int, [vp, C.c_int, C.c_int, vp]),
            "comm_destroy": (C.c_int, [vp]),
            "render_sharded": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params), _fp, _fp, u8p, C.POINTER(Stats)]),
            "resolve_last": (C.c_int, [vp, C.c_int, C.c_int, C.c_float, _fp, _fp, u8p]),
            "group_create": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]),
            "group_destroy": (None, [vp]),
            "group_last_error": (C.c_char_p, [vp]),
            "group_size": (C.c_int, [vp]),
            "group_ctx": (vp, [vp, C.c_int]),
            "group_commit": (C.c_int, [vp]),
            "group_set_option": (C.c_int, [vp, C.c_int, C.c_int64]),
            "group_render": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params), _fp, _fp, u8p, C.POINTER(Stats)]),
            "pin_host_buffer": (C.c_int, [vp, vp, C.c_int64]),
            "unpin_host_buffer": (C.c_int, [vp, vp]),
            "render_denoiser_inputs_sharded": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params), _fp, _fp, _fp, _fp, _fp, C.POINTER(Stats)]),
            "progressive_begin_sharded": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params)]),
            "progressive_read_sharded": (C.c_int, [vp, _fp, _fp, u8p, _fp, C.POINTER(C.c_int32)]),
            "group_render_denoiser_inputs": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params), _fp, _fp, _fp, _fp, _fp, C.POINTER(Stats)]),
            "group_progressive_begin": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(Params)]),
            "group_progressive_pass": (C.c_int, [vp, C.c_int, C.POINTER(Stats)]),
            "group_progressive_read": (C.c_int, [vp, _fp, _fp, u8p, _fp, C.POINTER(C.c_int32)]),
        }
        assert sorted(multi) == sorted(MULTI_SYMBOLS)
        self.has_multi = hasattr(cdll, prefix + "render_sharded")
        if self.has_multi or prefix == "ptb_":       # the product must export all of them (AttributeError otherwise)
            for name, (res, args) in multi.items():
                fn = getattr(cdll, prefix + name)
                fn.restype, fn.argtypes = res, args
                setattr(self, name, fn)
            self.has_multi = True

    def check_group(self, rc, group=None):
        if rc != OK:
            msg = self.group_last_error(group)
            raise PtbError(f"{self.prefix}group call failed rc={rc}: {msg.decode() if msg else ''}")

    def check(self, rc, ctx=None):
        if rc != OK:
            msg = self.last_error(ctx)
            raise PtbError(f"{self.prefix}* call failed rc={rc}: {msg.decode() if msg else ''}")


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def fptr(a):
    return a.ctypes.data_as(_fp) if a is not None else None
