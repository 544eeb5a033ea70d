"""Host-side mirror of the reference's operator surface for the radiance loop.

Names and argument meaning follow the reference (`Raytracer`, `Scene`, `Sphere`, `Plane`, `TriMesh`,
`Camera`; Raytracer.h:25-121, Geometry.h:849-1217, TriangleMesh.h:113-255, Vector.h:720-840) so the
parity tests read like reference code.  Everything here is description + plumbing: the objects only
record what the reference's objects hold and hand it to a C-ABI implementation (`_abi.Lib`) — the
CUDA library for the product, a CPU checker in the tests.  No rendering arithmetic lives in Python.
"""
import ctypes as C
import math

import numpy as np

from . import _abi
from ._abi import f32, fptr


class Camera:
    """Vector.h:720-840 (non-lenticular).  rotate() follows Camera::rotate (738-765)."""

    def __init__(self, position=(0, 0, 50), direction=(0, 0, -1), up=(0, 1, 0)):
        self.position = np.array(position, np.float32)
        self.direction = np.array(direction, np.float32)
        self.up = np.array(up, np.float32)
        self.fov = np.float32(35 * math.pi / 180)
        self.focus_distance = np.float32(50)
        self.aperture = np.float32(0.1)

    def rotate(self, angle_x, angle_y, time):
        ax, ay = np.float32(time * angle_x), np.float32(time * angle_y)
        cx, sx, cy, sy = (np.float32(f(a)) for f, a in ((math.cos, ax), (math.sin, ax), (math.cos, ay), (math.sin, ay)))

        def rot(v):
            t = np.array([v[0], cy * v[1] - sy * v[2], sy * v[1] + cy * v[2]], np.float32)
            return np.array([cx * t[0] - sx * t[2], t[1], sx * t[0] + cx * t[2]], np.float32)

        self.direction, self.up = rot(self.direction), rot(self.up)

    def c_struct(self):
        c = _abi.Camera()
        c.position[:] = [float(x) for x in self.position]
        c.direction[:] = [float(x) for x in self.direction]
        c.up[:] = [float(x) for x in self.up]
        c.fov, c.focus_distance, c.aperture = float(self.fov), float(self.focus_distance), float(self.aperture)
        return c


class Texture:
    """BRDF.h:252-426: `values` (H,W,3) float32 post-load, or a constant `multiplier`."""

    def __init__(self, multiplier=(1, 1, 1), values=None):
        self.multiplier = tuple(float(x) for x in (multiplier if np.ndim(multiplier) else (multiplier,) * 3))
        self.values = None if values is None else f32(values)

    def c_struct(self):
        t = _abi.Tex()
        t.mult[:] = self.multiplier
        if self.values is not None:
            h, w, _ = self.values.shape
            t.texels, t.W, t.H = fptr(self.values), w, h
        return t


# Material presets of the reference's object menu (mainApp.cpp:1499-1597): name -> (Kd, Ks, Ne).  "<name>": OpenGL-style table entry
# (Ne = shininess * 128); "<name>_ngan": Phong fit to the measured BRDF (Ngan et al. 2005).  The same table lives in the library
# (ptb_preset_get, csrc/scene_host.cpp); tests/test_host_logic.py checks the two against each other and against the reference's source.
PRESETS = {
    "gold": ((0.75164, 0.60648, 0.22648), (0.628281, 0.555802, 0.366065), 0.4 * 128),
    "gold_ngan": ((0.069, 0.0323, 0.00638), (0.0738, 0.0434, 0.0104), 41.9),
    "silver": ((0.50754, 0.50754, 0.50754), (0.508273, 0.508273, 0.508273), 0.4 * 128),
    "silver_ngan": ((0.0695, 0.0628, 0.0446), (0.0742, 0.0615, 0.0412), 75.0),
    "pearl": ((1.0, 0.829, 0.829), (0.296648, 0.296648, 0.296648), 0.088 * 128),
    "pearl_ngan": ((0.189, 0.146, 0.0861), (0.0485, 0.0346, 0.0161), 27.7),
    "white_plastic": ((0.55, 0.55, 0.55), (0.70, 0.70, 0.70), 0.25 * 128),
    "white_plastic_ngan": ((0.102, 0.0887, 0.0573), (0.00699, 0.00566, 0.0036), 1040.0),
    "chrome": ((0.4, 0.4, 0.4), (0.774597, 0.774597, 0.774597), 0.6 * 128),
    "chrome_ngan": ((0.00817, 0.0063, 0.00474), (0.0213, 0.0151, 0.00766), 17900.0),
    "bronze": ((0.714, 0.4284, 0.18144), (0.393548, 0.271906, 0.166721), 0.2 * 128),
    "bronze_ngan": ((0.0864, 0.0597, 0.0302), (0.015, 0.00818, 0.00381), 1290.0),
    "copper": ((0.7038, 0.27048, 0.0828), (0.256777, 0.137622, 0.086014), 0.1 * 128),
    "copper_ngan": ((0.0749, 0.0414, 0.027), (0.0756, 0.0437, 0.0202), 33200.0),
}


def _io():
    from . import sceneio
    return sceneio()


def load_image(path):
    """load_image<unsigned char> (utils.cpp:98-170): (H,W,3) uint8, rows flipped like the reference keeps them."""
    io = _io()
    p, w, h = C.POINTER(C.c_uint8)(), C.c_int32(), C.c_int32()
    io.check(io.image_load(str(path).encode(), C.byref(p), C.byref(w), C.byref(h)))
    a = np.ctypeslib.as_array(p, shape=(h.value, w.value, 3)).copy()
    io.image_free(p)
    return a


def load_texture_values(path, normals=False):
    """Texture::loadColors / loadNormals (BRDF.h:393-419): (H,W,3) float32 `Texture::values`, or None if the file cannot be read
    (the reference then keeps a constant slot)."""
    io = _io()
    p, w, h = C.POINTER(C.c_float)(), C.c_int32(), C.c_int32()
    if io.texture_load(str(path).encode(), 1 if normals else 0, C.byref(p), C.byref(w), C.byref(h)) != _abi.OK:
        return None
    a = np.ctypeslib.as_array(p, shape=(h.value, w.value, 3)).copy()
    io.image_free(p)
    return a


_KIND_NAMES = {_abi.KIND_KD: "Kd", _abi.KIND_NORMAL: "normal", _abi.KIND_SUBSURF: "Ksub", _abi.KIND_KS: "Ks", _abi.KIND_ALPHA: "alpha",
               _abi.KIND_NE: "Ne", _abi.KIND_TRANSP: "transp", _abi.KIND_REFR: "refr"}


def _texture_from_slot(slot, kind):
    f = slot.file.decode()
    vals = load_texture_values(f, kind == _abi.KIND_NORMAL) if f else None
    t = Texture(tuple(slot.mult), vals)
    t.filename = f or "Null"
    return t


_SLOTS = [("Kd", _abi.SLOT_KD), ("Ks", _abi.SLOT_KS), ("Ne", _abi.SLOT_NE), ("transp", _abi.SLOT_TRANSP),
          ("refr", _abi.SLOT_REFR), ("normal", _abi.SLOT_NORMAL), ("alpha", _abi.SLOT_ALPHA), ("Ksub", _abi.SLOT_KSUB)]


class Object:
    """Geometry.h:240-672: placement, flags, BRDF pointer and per-group texture slots."""

    def __init__(self):
        self.scale = 1.0
        self.mat_rotation = np.eye(3, dtype=np.float32)
        self.rotation_center = None            # None -> the object's own default
        self.max_translation = np.zeros(3, np.float32)
        self.miroir = False
        self.flip_normals = False
        self.interp_normals = True
        self.brdf = ("phong", None)            # or ("merl", table ndarray float64 of 3*90*90*180)
        self.materials = {}                    # group -> {slot name: Texture}
        self.ghost = False
        self.name = ""
        # Object::{scale,translation,rotation}_keyframes (Geometry.h:318-320): frame -> value, like the reference's std::maps
        self.scale_keyframes, self.translation_keyframes, self.rotation_keyframes = {}, {}, {}

    def add_keyframe(self, frame):
        """Object::add_keyframe (Geometry.h:313-317): the current placement becomes the key of `frame`."""
        self.rotation_keyframes[float(frame)] = np.array(self.mat_rotation, np.float32).reshape(3, 3).copy()
        self.translation_keyframes[float(frame)] = np.array(self.max_translation, np.float32).copy()
        self.scale_keyframes[float(frame)] = float(self.scale)
        return self

    def set_material(self, group=0, **slots):
        """e.g. set_material(0, Kd=Texture((.5,.5,.5)), Ks=Texture(.2), Ne=Texture(50))"""
        self.materials.setdefault(group, {}).update(slots)
        return self

    # ---- Object::set_col_texture / set_col_specular / set_col_roughness (Geometry.cpp:165-177, 229-234): the slot KEEPS its texels,
    #      only its multiplier changes; a slot index that does not exist is left alone, like the reference does ----
    def _set_col(self, name, col, idx):
        t = self.materials.get(idx, {}).get(name)
        if t is not None:
            t.multiplier = tuple(float(np.float32(x)) for x in col)
        return self

    def set_col_texture(self, col, idx=0):
        return self._set_col("Kd", col, idx)

    def set_col_specular(self, col, idx=0):
        return self._set_col("Ks", col, idx)

    def set_col_roughness(self, col, idx=0):
        return self._set_col("Ne", col, idx)

    def set_preset(self, name, idx=0):
        """A material preset of the reference's object menu (mainApp.cpp:1499-1597), e.g. "gold", "gold_ngan" (the Phong fit of
        Ngan et al. to the measured BRDF), "copper_ngan": set_col_texture + set_col_specular + set_col_roughness on slot `idx`."""
        kd, ks, ne = PRESETS[name]
        return self.set_col_texture(kd, idx).set_col_specular(ks, idx).set_col_roughness((ne, ne, ne), idx)

    def _flags(self):
        return ((_abi.OBJ_MIRROR if self.miroir else 0) | (_abi.OBJ_FLIP_NORMALS if self.flip_normals else 0)
                | (0 if self.interp_normals else _abi.OBJ_FLAT_NORMALS) | (_abi.OBJ_GHOST if self.ghost else 0)
                | (_abi.OBJ_DISPLAY_EDGES if getattr(self, "display_edges", False) else 0))

    def _xform(self):
        x = _abi.Xform()
        x.scale = float(self.scale)
        x.rotation[:] = [float(v) for v in np.asarray(self.mat_rotation, np.float32).reshape(9)]
        rc = self.rotation_center if self.rotation_center is not None else (float("nan"),) * 3
        x.rotation_center[:] = [float(v) for v in rc]
        x.translation[:] = [float(v) for v in self.max_translation]
        return x


class Sphere(Object):
    def __init__(self, O, R, mirror=False, normal_swapped=False):
        super().__init__()
        self.O, self.R = np.array(O, np.float32), float(R)
        self.miroir, self.flip_normals = mirror, normal_swapped
        self.envmap = None                     # (H,W,3) uint8 on the dome (object 1)


class Plane(Object):
    def __init__(self, A, N, mirror=False):
        super().__init__()
        self.A, self.vecN = np.array(A, np.float32), np.array(N, np.float32)
        self.miroir = mirror


class Cylinder(Object):
    """Geometry.h:731-846: the open tube of radius R around the segment A-B (the reference's yarn segments, TriangleMesh.h:281)."""

    def __init__(self, A, B, R, mirror=False):
        super().__init__()
        self.A, self.B, self.R = np.array(A, np.float32), np.array(B, np.float32), float(R)
        self.miroir = mirror


class PointSet(Object):
    """PointSet.h / PointSet.cpp as the object stands after init: every point a disc (centre, normal, radius, colour).  The
    reference fills normals and radii with estimate_normals (k-NN + PCA, PointSet.h:124-176); here they are given."""

    def __init__(self, points, normals, radii, colors=None, mirror=False, normal_swapped=False, display_edges=False):
        super().__init__()
        self.points, self.normals = f32(points).reshape(-1, 3), f32(normals).reshape(-1, 3)
        self.radii = f32(radii).reshape(-1)
        self.colors = None if colors is None else f32(colors).reshape(-1, 3)
        assert len(self.points) == len(self.normals) == len(self.radii) and (self.colors is None or len(self.colors) == len(self.points))
        self.miroir, self.flip_normals, self.display_edges = mirror, normal_swapped, display_edges
        self.rotation_center = np.full(3, np.nan, np.float32)      # init: the mean of the points


class Yarns(Object):
    """TriangleMesh.h:265-312: a bundle of yarn curves, every segment an open Cylinder under one BVH.  The reference shades a yarn
    with its segments' default material (white diffuse) whatever the object's slots hold; transform, BRDF, mirror and ghost flags
    are the object's."""

    def __init__(self, A, B, R, mirror=False):
        super().__init__()
        self.A, self.B = f32(A).reshape(-1, 3), f32(B).reshape(-1, 3)
        self.R = f32(np.broadcast_to(np.asarray(R, np.float32), (len(self.A),))).reshape(-1)
        assert len(self.A) == len(self.B) == len(self.R) and len(self.A) > 0
        self.miroir = mirror
        self.rotation_center = np.zeros(3, np.float32)

    @classmethod
    def from_file(cls, path):
        """`new Yarns(file)` (TriangleMesh.h:268-290): `nbyarns`, then per yarn `nbsegments` and that many points; consecutive points
        times 50 are joined by cylinders of radius 0.1."""
        io = _io()
        fp = C.POINTER(C.c_float)
        a, b, r, n = fp(), fp(), fp(), C.c_int32()
        io.check(io.yarnfile_read(str(path).encode(), C.byref(a), C.byref(b), C.byref(r), C.byref(n)))
        A, B = np.ctypeslib.as_array(a, shape=(n.value, 3)).copy(), np.ctypeslib.as_array(b, shape=(n.value, 3)).copy()
        R = np.ctypeslib.as_array(r, shape=(n.value,)).copy()
        for p in (a, b, r):
            io.yarnfile_free(p)
        return cls(A, B, R)


class TriMesh(Object):
    """In-memory equivalent of `new TriMesh(scene, file, scaling, offset, mirror, NULL, false, center)`
    (TriangleMesh.cpp:714-841): arrays as a file reader would have produced them."""

    def __init__(self, vertices, normals, uvs, tri, scaling=1.0, offset=(0, 0, 0), mirror=False, center=True):
        super().__init__()
        self.vertices, self.normals = f32(vertices).reshape(-1, 3), f32(normals).reshape(-1, 3)
        self.uvs = f32(uvs).reshape(-1, 2)
        self.tri = np.ascontiguousarray(tri, np.int32).reshape(-1, 10)
        self.scaling, self.offset, self.center = float(scaling), tuple(float(x) for x in offset), bool(center)
        self.miroir = mirror

    @classmethod
    def from_file(cls, path, scaling=1.0, offset=(0, 0, 0), mirror=False, center=True, load_textures=True):
        """`new TriMesh(scene, file, scaling, offset, mirror, NULL, false, center)` for an .obj (+ .mtl) or .off file
        (TriangleMesh.cpp:714-841 with readOBJ 240-569 / readOFF 107-130)."""
        io = _io()
        h = C.c_void_p()
        io.check(io.meshfile_read(str(path).encode(), int(load_textures), C.byref(h)))
        try:
            info = _abi.MeshfileInfo()
            io.check(io.meshfile_get(h, C.byref(info)))
            arr = lambda p, n, k, dt: (np.ctypeslib.as_array(p, shape=(n, k)).astype(dt, copy=True) if n else np.zeros((0, k), dt))
            m = cls(arr(info.vertices, info.n_vertices, 3, np.float32), arr(info.normals, info.n_normals, 3, np.float32),
                    arr(info.uvs, info.n_uvs, 2, np.float32), arr(info.tri, info.n_tri, 10, np.int32), scaling, offset, mirror, center)
            m.vertex_colors = arr(info.vertex_colors, info.n_vertex_colors, 3, np.float32)
            m.name = str(path)
            m.group_names = {}
            for g in range(info.n_groups):
                buf = C.create_string_buffer(_abi.PATH_MAX)
                if io.meshfile_group_name(h, g, buf) == _abi.OK:
                    m.group_names[buf.value.decode()] = g
            if info.has_materials:
                n_mat = max(1, max(m.group_names.values(), default=0) + 1)
                for g in range(n_mat):
                    slots = {}
                    for kind, name in _KIND_NAMES.items():
                        sl = _abi.Slot()
                        if io.meshfile_group_slot(h, g, kind, C.byref(sl)) == _abi.OK:
                            slots[name] = _texture_from_slot(sl, kind)
                    m.materials[g] = slots
        finally:
            io.meshfile_free(h)
        return m


class Scene:
    """Geometry.h:1238-1400: object list; ids 0/1 are the light and the dome."""

    def __init__(self):
        self.objects = []
        self.intensite_lumiere = 0.0
        self.envmap_intensity = 1.0
        self.fog_density = self.fog_absorption = self.fog_density_decay = self.fog_absorption_decay = 0.0
        self.fog_type = self.fog_phase_type = 0
        self.phase_aniso = 0.0
        self.current_frame = 0                 # Scene::current_frame (an int, Geometry.h:1372)
        self.background = None                 # (H,W,3) uint8 as load_image returns it, or None
        self.background_gamma = 2.2            # the `gamma` argument of Scene::load_background (Geometry.h:1355-1363)
        self.background_values = None          # (H,W,3) float32 in Scene::background scale; overrides `background` when set

    def _background_floats(self):
        """Scene::load_background (Geometry.h:1355-1363): pow(v/255, gamma) * 196964.699, kept as float."""
        if self.background_values is not None:
            return np.ascontiguousarray(self.background_values, np.float32)
        if self.background is None:
            return None
        return np.ascontiguousarray(np.power(np.asarray(self.background, np.float64) / 255., float(self.background_gamma)) * 196964.699, np.float32)

    def addObject(self, o):
        self.objects.append(o)
        return len(self.objects) - 1


class Raytracer:
    """Raytracer.h:25-121.  Fill the public fields, then `render_image_nopreviz()`; outputs land in
    `imagedouble`, `sample_count`, `image` like the reference's public buffers."""

    def __init__(self, lib, device=0, devices=None):
        """`devices=[0, 1, ...]`: render every frame on several GPUs of this process (tile-sharded, gathered over NCCL inside the
        library: ptb_group_*, include/ptb200.h); the interface stays the reference's single render_image_nopreviz() call."""
        self.lib = lib
        self.devices = list(devices) if devices is not None else None
        self.device = self.devices[0] if self.devices else device
        self._group = None
        self._comm = (1, 0)          # (ranks, rank) of the one-process-per-GPU communicator, see comm_init
        self.W, self.H, self.nrays, self.nb_bounces = 1000, 800, 100, 3
        self.sigma_filter, self.gamma = 0.5, 2.2
        self.seed = 0
        self.cam = Camera()
        self.s = Scene()
        self.imagedouble = self.sample_count = self.image = None
        # the reference's Raytracer OWNS imagedouble / sample_count / image (std::vector members resized when the frame size
        # changes, Raytracer.h:90-105).  True: the output arrays are kept across renders like that (no fresh, untouched pages for
        # the device-to-host copies of every call); False (default): every render returns new arrays.
        self.reuse_buffers = False
        self.stats = None
        self._ctx = None
        self._keep = []
        self._pinned = {}

    # ---- Raytracer::loadScene (Raytracer.cpp:1238-1274) ----
    def loadScene(self):
        self.W, self.H, self.nrays, self.nb_bounces = 1000, 800, 100, 3
        self.cam = Camera((0, 0, 50), (0, 0, -1), (0, 1, 0))
        self.cam.fov, self.cam.focus_distance, self.cam.aperture = np.float32(35 * math.pi / 180), np.float32(50), np.float32(0.1)
        self.sigma_filter = 0.5
        self.s = Scene()
        slum = Sphere((10, 23, 15), 10)
        s2 = Sphere((0, 0, 0), 1000000, normal_swapped=True)
        plane = Plane((0, 0, 0), (0, 1, 0))
        plane.max_translation = np.array((0, -27.3, 0), np.float32)
        for o in (slum, s2, plane):
            self.s.addObject(o)
        self.s.intensite_lumiere = float(np.float32(1000000000 * 4. * math.pi / (4. * math.pi * slum.R * slum.R * math.pi)))
        self.s.envmap_intensity = 1.0
        self.cam.rotate(0, -22 * math.pi / 180, 1)
        return self

    # ---- Raytracer::load_scene (Raytracer.cpp:1149-1236) ----
    def load_scene(self, filename, replacedNames=None):
        """Parse a .scn file written by Raytracer::save_scene, read the meshes / textures / environment map it names and
        fill this Raytracer's fields like the reference does.  Parsing happens in the native reader (include/ptb_sceneio.h)."""
        io = _io()
        h = C.c_void_p()
        io.check(io.scn_load(str(filename).encode(), replacedNames.encode() if replacedNames else None, C.byref(h)))
        try:
            hd = _abi.ScnHeader()
            io.check(io.scn_get_header(h, C.byref(hd)))
            self.W, self.H, self.nrays, self.nb_bounces = hd.W, hd.H, hd.nrays, hd.nb_bounces
            self.sigma_filter, self.gamma, self.has_denoiser = float(hd.sigma_filter), float(hd.gamma), bool(hd.has_denoiser)
            self.cam = Camera(tuple(hd.cam.position), tuple(hd.cam.direction), tuple(hd.cam.up))
            self.cam.fov, self.cam.focus_distance, self.cam.aperture = np.float32(hd.cam.fov), np.float32(hd.cam.focus_distance), np.float32(hd.cam.aperture)
            self.cam.is_lenticular = bool(hd.is_lenticular)
            self.s = Scene()
            s = self.s
            s.intensite_lumiere, s.envmap_intensity = float(hd.intensite_lumiere), float(hd.envmap_intensity)
            s.fog_density, s.fog_absorption = float(hd.fog_density), float(hd.fog_absorption)
            s.fog_density_decay, s.fog_absorption_decay = float(hd.fog_density_decay), float(hd.fog_absorption_decay)
            s.fog_type, s.fog_phase_type = hd.fog_type, hd.fog_phase_type
            if hd.background:
                s.background = load_image(hd.background.decode())
                s.background_gamma = float(hd.gamma)
            for i in range(hd.n_objects):
                o = _abi.ScnObject()
                io.check(io.scn_get_object(h, i, C.byref(o)))
                name = o.name.decode()
                if o.type == _abi.SCN_SPHERE:
                    obj = Sphere(tuple(o.O), float(o.R))
                    if o.is_envmap:
                        obj.envmap = load_image(o.envmap.decode())
                elif o.type == _abi.SCN_PLANE:
                    obj = Plane(tuple(o.A), tuple(o.N))
                elif o.type == _abi.SCN_MESH:
                    obj = TriMesh.from_file(name, 1.0, (0, 0, 0), bool(o.miroir), bool(o.is_centered), load_textures=False)
                else:
                    raise _abi.PtbError(f"load_scene: object {i} ({name}): PointSet objects are not rendered")
                obj.name = name
                obj.miroir, obj.ghost = bool(o.miroir), bool(o.ghost)
                obj.flip_normals, obj.interp_normals = bool(o.flip_normals), bool(o.interp_normals)
                obj.scale = float(o.xform.scale)
                obj.mat_rotation = np.array(o.xform.rotation, np.float32).reshape(3, 3)
                obj.rotation_center = tuple(o.xform.rotation_center)
                obj.max_translation = np.array(o.xform.translation, np.float32)
                if o.n_keyframes > 0:      # the three keyframe maps (Geometry.h:544-567)
                    for kind, width, store in ((_abi.KEY_SCALE, 1, obj.scale_keyframes), (_abi.KEY_TRANSLATION, 3, obj.translation_keyframes),
                                               (_abi.KEY_ROTATION, 9, obj.rotation_keyframes)):
                        n = io.scn_get_keyframes(h, i, kind, None, None, 0)
                        fr, val = np.zeros(max(n, 1), np.float32), np.zeros(max(n, 1) * width, np.float32)
                        io.scn_get_keyframes(h, i, kind, fptr(fr), fptr(val), n)
                        for k in range(n):
                            v = val[k * width:(k + 1) * width]
                            store[float(fr[k])] = float(v[0]) if width == 1 else (v.copy() if width == 3 else v.reshape(3, 3).copy())
                for kind, slot_name in _KIND_NAMES.items():
                    for g in range(o.n_slots[kind]):
                        sl = _abi.Slot()
                        io.check(io.scn_get_slot(h, i, kind, g, C.byref(sl)))
                        obj.materials.setdefault(g, {})[slot_name] = _texture_from_slot(sl, kind)
                s.addObject(obj)
        finally:
            io.scn_free(h)
        return self

    def load_scene_native(self, filename, replacedNames=None, io=None):
        """The C-level route a C/C++ caller takes: `ptb_load_scene` parses the file, reads meshes / textures / envmap and feeds the
        context itself (include/ptb_sceneio.h); this object only receives the camera and frame parameters.  Commits the scene."""
        io = io or _io()
        L = self.lib
        self.close()
        ctx = C.c_void_p()
        L.check(L.create(self.device, C.byref(ctx)))
        self._ctx = ctx
        cam, p = _abi.Camera(), _abi.Params()
        io.check(io.load_scene(ctx, str(filename).encode(), replacedNames.encode() if replacedNames else None, C.byref(cam), C.byref(p)))
        L.check(L.set_frame(ctx, float(int(self.s.current_frame))), ctx)
        self.W, self.H, self.nrays, self.nb_bounces = p.W, p.H, p.nrays, p.nb_bounces
        self.sigma_filter, self.gamma = float(p.sigma_filter), float(p.gamma)
        self.cam = Camera(tuple(cam.position), tuple(cam.direction), tuple(cam.up))
        self.cam.fov, self.cam.focus_distance, self.cam.aperture = np.float32(cam.fov), np.float32(cam.focus_distance), np.float32(cam.aperture)
        L.check(L.commit(ctx), ctx)
        return self

    def _unsupported(self):
        """Scene features of the reference that the CUDA path does not render: refused, never approximated."""
        s = self.s
        if getattr(self.cam, "is_lenticular", False):
            return "lenticular camera"
        for i, o in enumerate(s.objects):
            if getattr(o, "vertex_colors", None) is not None and len(o.vertex_colors):
                return f"per-vertex colours on object {i}"
            if i != 1 and getattr(o, "envmap", None) is not None:
                return f"environment map on object {i} (only the dome, object 1)"
            if not isinstance(o, TriMesh):
                for slots in o.materials.values():
                    t = slots.get("Ksub")
                    if t is not None and (t.values is not None or sum(x * x for x in t.multiplier) > 1e-8):
                        return f"subsurface scattering on object {i}: the reference defines it for triangle meshes only"
        return None

    # ---- scene hand-over -------------------------------------------------------------------------
    def commit(self):
        bad = self._unsupported()
        if bad:
            raise _abi.PtbError(f"unsupported by this renderer: {bad}")
        L = self.lib
        comm = getattr(self, "_comm_args", None)
        self.close()
        ctx = C.c_void_p()
        if self.devices and len(self.devices) > 1:
            g = C.c_void_p()
            L.check_group(L.group_create((C.c_int * len(self.devices))(*self.devices), len(self.devices), C.byref(g)))
            self._group = g
            ctx = C.c_void_p(L.group_ctx(g, 0))
            for opt, val in getattr(self, "_group_options", {}).items():
                L.check_group(L.group_set_option(g, opt, val), g)
        else:
            L.check(L.create(self.device, C.byref(ctx)))
        self._ctx = ctx
        if comm is not None:
            self.comm_init(*comm)
        if getattr(self, "build_threads", 0):
            L.check(L.set_option(ctx, _abi.OPT_BUILD_THREADS, int(self.build_threads)), ctx)
        merl_ids = {}
        for o in self.s.objects:
            oid = C.c_int(-1)
            xf = o._xform()
            if isinstance(o, Sphere):
                L.check(L.add_sphere(ctx, fptr(f32(o.O)), o.R, C.byref(xf), o._flags(), C.byref(oid)), ctx)
            elif isinstance(o, Plane):
                L.check(L.add_plane(ctx, fptr(f32(o.A)), fptr(f32(o.vecN)), C.byref(xf), o._flags(), C.byref(oid)), ctx)
            elif isinstance(o, PointSet):
                d = _abi.PointSetDesc(fptr(o.points), fptr(o.normals), fptr(o.radii), fptr(o.colors), len(o.points))
                L.check(L.add_pointset(ctx, C.byref(d), C.byref(xf), o._flags(), C.byref(oid)), ctx)
            elif isinstance(o, Yarns):
                d = _abi.YarnsDesc(fptr(o.A), fptr(o.B), fptr(o.R), len(o.A))
                L.check(L.add_yarns(ctx, C.byref(d), C.byref(xf), o._flags(), C.byref(oid)), ctx)
            elif isinstance(o, Cylinder):
                L.check(L.add_cylinder(ctx, fptr(f32(o.A)), fptr(f32(o.B)), o.R, C.byref(xf), o._flags(), C.byref(oid)), ctx)
            elif isinstance(o, TriMesh):
                m = _abi.Mesh()
                m.vertices, m.n_vertices = fptr(o.vertices), len(o.vertices)
                m.normals, m.n_normals = fptr(o.normals), len(o.normals)
                m.uvs, m.n_uvs = fptr(o.uvs), len(o.uvs)
                m.tri, m.n_tri = o.tri.ctypes.data_as(C.POINTER(C.c_int32)), len(o.tri)
                m.scaling, m.center = o.scaling, int(o.center)
                m.offset[:] = o.offset
                L.check(L.add_mesh(ctx, C.byref(m), C.byref(xf), o._flags(), C.byref(oid)), ctx)
            else:
                raise TypeError(type(o))
            for kind, keys, width in ((_abi.KEY_SCALE, o.scale_keyframes, 1), (_abi.KEY_TRANSLATION, o.translation_keyframes, 3),
                                      (_abi.KEY_ROTATION, o.rotation_keyframes, 9)):
                if keys:
                    fr = f32(sorted(keys))
                    val = f32(np.stack([np.asarray(keys[k], np.float32).reshape(width) for k in sorted(keys)]))
                    L.check(L.set_keyframes(ctx, oid.value, kind, fptr(fr), fptr(val), len(fr)), ctx)
            for group, slots in sorted(o.materials.items()):
                mat = _abi.Material()
                for name, bit in _SLOTS:
                    if name in slots:
                        mat.present |= bit
                        setattr(mat, name, slots[name].c_struct())
                L.check(L.set_group_material(ctx, oid.value, group, C.byref(mat)), ctx)
            if o.brdf[0] == "merl":
                key = id(o.brdf[1])
                if key not in merl_ids:
                    tab = np.ascontiguousarray(o.brdf[1], np.float64).reshape(-1)
                    assert tab.size == 3 * 90 * 90 * 180
                    mid = C.c_int(-1)
                    L.check(L.add_merl(ctx, tab.ctypes.data_as(C.POINTER(C.c_double)), C.byref(mid)), ctx)
                    merl_ids[key] = mid.value
                L.check(L.set_brdf(ctx, oid.value, _abi.BRDF_MERL, merl_ids[key]), ctx)
        dome = self.s.objects[1] if len(self.s.objects) > 1 else None
        if getattr(dome, "envmap", None) is not None:
            env = np.ascontiguousarray(dome.envmap, np.uint8)
            L.check(L.set_envmap(ctx, env.ctypes.data_as(C.POINTER(C.c_uint8)), env.shape[1], env.shape[0]), ctx)
        L.check(L.set_light(ctx, float(self.s.intensite_lumiere), float(self.s.envmap_intensity)), ctx)
        s = self.s
        L.check(L.set_frame(ctx, float(int(s.current_frame))), ctx)
        if s.fog_density > 0:
            fog = _abi.Fog(float(s.fog_density), float(s.fog_absorption), float(s.fog_density_decay), float(s.fog_absorption_decay),
                           int(s.fog_type), int(s.fog_phase_type), float(s.phase_aniso))
            L.check(L.set_fog(ctx, C.byref(fog)), ctx)
        bg = s._background_floats()
        if bg is not None:
            L.check(L.set_background(ctx, fptr(bg), bg.shape[1], bg.shape[0]), ctx)
        if self._group is not None:
            L.check_group(L.group_commit(self._group), self._group)
        else:
            L.check(L.commit(ctx), ctx)
        return self

    # ---- multi-GPU, one process per GPU: every rank builds the same scene, then calls render_image_nopreviz() ----
    def comm_init(self, n_ranks, rank, id_bytes):
        """Join the NCCL communicator of a tile-sharded render (ptb_comm_init).  `id_bytes`: the 128 bytes rank 0 got from
        `comm_unique_id()` and distributed (e.g. torch.distributed.broadcast_object_list).  Survives commit()."""
        self._comm_args = (int(n_ranks), int(rank), bytes(id_bytes) if id_bytes is not None else None)
        if self._ctx is not None:
            buf = C.create_string_buffer(self._comm_args[2], _abi.COMM_ID_BYTES) if self._comm_args[2] is not None else None
            if int(n_ranks) > 1 or self.lib.has_multi:
                self.lib.check(self.lib.comm_init(self._ctx, int(n_ranks), int(rank), buf), self._ctx)
        self._comm = (int(n_ranks), int(rank))
        return self

    def comm_unique_id(self):
        buf = C.create_string_buffer(_abi.COMM_ID_BYTES)
        self.lib.check(self.lib.comm_unique_id(buf), None)
        return buf.raw

    def set_frame(self, frame):
        """Scene::current_frame for the next render (mainApp.cpp:790, 874-877).  On a committed scene nothing is rebuilt: the library
        re-poses the key-framed objects on the device before the next render (ptb_set_frame: matrices, triangles, BVH8 refit)."""
        self.s.current_frame = frame
        if self._ctx is not None:
            self.lib.check(self.lib.set_frame(self._ctx, float(int(frame))), self._ctx)
        return self

    def params(self, shard_rank=0, shard_count=1, tile_size=0):
        p = _abi.Params()
        p.W, p.H, p.nrays, p.nb_bounces = self.W, self.H, self.nrays, self.nb_bounces
        p.sigma_filter, p.gamma, p.seed = self.sigma_filter, self.gamma, self.seed
        p.shard_rank, p.shard_count, p.tile_size = shard_rank, shard_count, tile_size
        return p

    # ---- Raytracer::render_image_nopreviz (Raytracer.cpp:1565-1798) ----
    def _out(self, name, shape, dtype):
        a = getattr(self, name, None)
        if not (self.reuse_buffers and a is not None and a.shape == shape and a.dtype == dtype):
            if a is not None and id(a) in self._pinned and self._ctx is not None:
                self.lib.unpin_host_buffer(self._ctx, C.c_void_p(a.ctypes.data)); self._pinned.pop(id(a))
            a = np.empty(shape, dtype)
            setattr(self, name, a)
        if self.reuse_buffers and self.lib.has_multi and id(a) not in self._pinned and self._ctx is not None:
            # the Raytracer owns these arrays across frames (Raytracer.h:90-105): page-lock them once
            if self.lib.pin_host_buffer(self._ctx, C.c_void_p(a.ctypes.data), a.nbytes) == 0:
                self._pinned[id(a)] = a
        return a

    def render_image_nopreviz(self, want_image=True):
        L, ctx = self.lib, self._ctx
        if ctx is None:
            self.commit()
            ctx = self._ctx
        st, cam, p = _abi.Stats(), self.cam.c_struct(), self.params()
        if self._group is None and self._comm[0] > 1 and self._comm[1] != 0:
            # one process per GPU, not rank 0: this rank renders its tiles and sends them; the frame lands on rank 0
            L.check(L.render_sharded(ctx, C.byref(cam), C.byref(p), None, None, None, C.byref(st)), ctx)
            self.stats = st.as_dict()
            return None
        self._out("imagedouble", (self.H, self.W, 3), np.float32)
        self._out("sample_count", (self.H, self.W), np.float32)
        if want_image:
            self._out("image", (self.H, self.W, 3), np.uint8)
        else:
            self.image = None
        u8 = self.image.ctypes.data_as(C.POINTER(C.c_uint8)) if want_image else None
        if self._group is not None:        # several GPUs of this process under the one call
            L.check_group(L.group_render(self._group, C.byref(cam), C.byref(p), fptr(self.imagedouble), fptr(self.sample_count), u8, C.byref(st)), self._group)
        elif self._comm[0] > 1:            # one process per GPU, rank 0: its own tiles + the gather
            L.check(L.render_sharded(ctx, C.byref(cam), C.byref(p), fptr(self.imagedouble), fptr(self.sample_count), u8, C.byref(st)), ctx)
        else:
            L.check(L.render(ctx, C.byref(cam), C.byref(p), fptr(self.imagedouble), fptr(self.sample_count), u8, C.byref(st)), ctx)
        self.stats = st.as_dict()
        return self.imagedouble

    def render_resident(self):
        """The same render with the frame left on the device (rank 0 / device 0 holds the gathered sums; `resolve_last()` reads them)."""
        L, ctx = self.lib, self._ctx
        st, cam, p = _abi.Stats(), self.cam.c_struct(), self.params()
        if self._group is not None:
            L.check_group(L.group_render(self._group, C.byref(cam), C.byref(p), None, None, None, C.byref(st)), self._group)
        else:
            L.check(L.render_sharded(ctx, C.byref(cam), C.byref(p), None, None, None, C.byref(st)), ctx)
        self.stats = st.as_dict()
        return self.stats

    def resolve_last(self, want_image=True):
        L, ctx = self.lib, self._ctx
        self._out("imagedouble", (self.H, self.W, 3), np.float32)
        self._out("sample_count", (self.H, self.W), np.float32)
        if want_image:
            self._out("image", (self.H, self.W, 3), np.uint8)
        else:
            self.image = None
        L.check(L.resolve_last(ctx, self.W, self.H, self.gamma, fptr(self.imagedouble), fptr(self.sample_count),
                               self.image.ctypes.data_as(C.POINTER(C.c_uint8)) if want_image else None), ctx)
        return self.imagedouble

    # ---- Raytracer::render_image (Raytracer.cpp:1424-1563): the progressive renderer ----
    def _route(self):
        """Where a render goes: "group" (devices=[...]), "sharded" (one process per GPU after comm_init) or "single"."""
        return "group" if self._group is not None else ("sharded" if self._comm[0] > 1 else "single")

    def render_image(self, passes_per_call=1, on_pass=None):
        """One sample per pixel per pass until `nrays` passes are done or `self.stopped` is set by `on_pass` (the reference's GUI
        sets `stopped` from another thread, 1452).  Fills `imagedouble` (UN-normalised sums, as the reference leaves them),
        `sample_count`, `image`, `imagedouble_lowres` and `current_nb_rays`.  With devices=[...] every pass runs on all of them; with
        one process per GPU every rank runs to `nrays` (a stop would have to be agreed by all ranks: `on_pass` is refused) and
        ranks other than 0 return None."""
        L, ctx = self.lib, self._ctx
        if ctx is None:
            self.commit()
            ctx = self._ctx
        route = self._route()
        if route == "sharded" and on_pass is not None:
            raise _abi.PtbError("render_image: on_pass needs one process (devices=[...]); with one process per GPU every rank renders to nrays")
        cam, p = self.cam.c_struct(), self.params()
        if route == "group":
            L.check_group(L.group_progressive_begin(self._group, C.byref(cam), C.byref(p)), self._group)
        elif route == "sharded":
            L.check(L.progressive_begin_sharded(ctx, C.byref(cam), C.byref(p)), ctx)
        else:
            L.check(L.progressive_begin(ctx, C.byref(cam), C.byref(p)), ctx)
        self.stopped = False
        self.current_nb_rays = 0
        tot = {"samples": 0, "rays_closest": 0, "rays_shadow": 0, "ms_device": 0.0, "kernel_launches": 0}
        while self.current_nb_rays < self.nrays and not self.stopped:
            st = _abi.Stats()
            if route == "group":
                L.check_group(L.group_progressive_pass(self._group, int(passes_per_call), C.byref(st)), self._group)
            else:
                L.check(L.progressive_pass(ctx, int(passes_per_call), C.byref(st)), ctx)
            for k in tot:
                tot[k] += getattr(st, k)
            self.current_nb_rays = min(self.nrays, self.current_nb_rays + int(passes_per_call))
            if on_pass is not None:
                on_pass(self)
        self.stats = tot
        return self.read_progressive()

    def read_progressive(self):
        """The outputs of the session so far (collective with one process per GPU: every rank calls it; rank 0 gets them)."""
        L, ctx = self.lib, self._ctx
        route = self._route()
        n = C.c_int32(0)
        self.stopped = True                      # Raytracer.cpp:1559
        if route == "sharded" and self._comm[1] != 0:
            L.check(L.progressive_read_sharded(ctx, None, None, None, None, C.byref(n)), ctx)
            self.current_nb_rays = n.value
            return None
        wlr, hlr = -(-self.W // 16), -(-self.H // 16)
        self.imagedouble = np.empty((self.H, self.W, 3), np.float32)
        self.sample_count = np.empty((self.H, self.W), np.float32)
        self.image = np.empty((self.H, self.W, 3), np.uint8)
        self.imagedouble_lowres = np.empty((hlr, wlr, 3), np.float32)
        outs = (fptr(self.imagedouble), fptr(self.sample_count), self.image.ctypes.data_as(C.POINTER(C.c_uint8)), fptr(self.imagedouble_lowres), C.byref(n))
        if route == "group":
            L.check_group(L.group_progressive_read(self._group, *outs), self._group)
        elif route == "sharded":
            L.check(L.progressive_read_sharded(ctx, *outs), ctx)
        else:
            L.check(L.progressive_read(ctx, *outs), ctx)
        self.current_nb_rays = n.value
        return self.imagedouble

    # ---- render_image_nopreviz with has_denoiser (Raytracer.cpp:1631-1645, 1676-1693), up to the OIDN hand-over ----
    def render_denoiser_inputs(self):
        """Fills `imagedouble` (mean radiance, unsplatted), `sample_count`, `albedoImage`, `normalImage` (as the reference computes it:
        the normalised COLOUR sum) and `first_hit_normal` (the normalised sum of first-hit shading normals).  Routed like
        render_image_nopreviz: all the devices of devices=[...], or every rank after comm_init (ranks other than 0 return None)."""
        L, ctx = self.lib, self._ctx
        if ctx is None:
            self.commit()
            ctx = self._ctx
        route = self._route()
        st, cam, p = _abi.Stats(), self.cam.c_struct(), self.params()
        if route == "sharded" and self._comm[1] != 0:
            L.check(L.render_denoiser_inputs_sharded(ctx, C.byref(cam), C.byref(p), None, None, None, None, None, C.byref(st)), ctx)
            self.stats = st.as_dict()
            return None
        mk = lambda: np.empty((self.H, self.W, 3), np.float32)
        self.imagedouble, self.albedoImage, self.normalImage, self.first_hit_normal = mk(), mk(), mk(), mk()
        self.sample_count = np.empty((self.H, self.W), np.float32)
        outs = (fptr(self.imagedouble), fptr(self.sample_count), fptr(self.albedoImage), fptr(self.normalImage), fptr(self.first_hit_normal), C.byref(st))
        if route == "group":
            L.check_group(L.group_render_denoiser_inputs(self._group, C.byref(cam), C.byref(p), *outs), self._group)
        elif route == "sharded":
            L.check(L.render_denoiser_inputs_sharded(ctx, C.byref(cam), C.byref(p), *outs), ctx)
        else:
            L.check(L.render_denoiser_inputs(ctx, C.byref(cam), C.byref(p), *outs), ctx)
        self.stats = st.as_dict()
        return self.imagedouble

    def render_accum(self, d_rgbw_ptr, shard_rank=0, shard_count=1, tile_size=0):
        """Sharded form: add this shard's sums into a caller-owned DEVICE float4 buffer."""
        L, ctx = self.lib, self._ctx
        st, cam, p = _abi.Stats(), self.cam.c_struct(), self.params(shard_rank, shard_count, tile_size)
        L.check(L.render_accum(ctx, C.byref(cam), C.byref(p), C.c_void_p(d_rgbw_ptr), C.byref(st)), ctx)
        self.stats = st.as_dict()
        return self.stats

    def resolve(self, d_rgbw_ptr, want_image=True):
        L, ctx = self.lib, self._ctx
        self._out("imagedouble", (self.H, self.W, 3), np.float32)
        self._out("sample_count", (self.H, self.W), np.float32)
        if want_image:
            self._out("image", (self.H, self.W, 3), np.uint8)
        else:
            self.image = None
        L.check(L.resolve(ctx, C.c_void_p(d_rgbw_ptr), self.W, self.H, self.gamma, fptr(self.imagedouble), fptr(self.sample_count),
                          self.image.ctypes.data_as(C.POINTER(C.c_uint8)) if want_image else None), ctx)
        return self.imagedouble

    def primary_ids(self, W=None, H=None):
        """The picking query (mainApp.h:686-692) over the whole frame."""
        L, ctx = self.lib, self._ctx
        W, H = W or self.W, H or self.H
        obj = np.empty((H, W), np.int32)
        tri = np.empty((H, W), np.int32)
        t = np.empty((H, W), np.float32)
        cam = self.cam.c_struct()
        i32 = C.POINTER(C.c_int32)
        L.check(L.primary_ids(ctx, C.byref(cam), W, H, obj.ctypes.data_as(i32), tri.ctypes.data_as(i32), fptr(t)), ctx)
        return obj, tri, t

    def kat(self, which, inputs, W=None, H=None):
        L, ctx = self.lib, self._ctx
        n_in, n_out = _abi.KAT_SHAPES[which]
        a = np.ascontiguousarray(inputs, np.float64).reshape(-1, n_in)
        out = np.zeros((len(a), n_out), np.float64)
        cam = self.cam.c_struct()
        dp = C.POINTER(C.c_double)
        L.check(L.kat(ctx, which, C.byref(cam), W or self.W, H or self.H, a.ctypes.data_as(dp), len(a), n_in,
                      out.ctypes.data_as(dp), n_out), ctx)
        return out

    def set_option(self, option, value):
        if self._group is not None:
            self.lib.check_group(self.lib.group_set_option(self._group, option, int(value)), self._group)
        else:
            self.lib.check(self.lib.set_option(self._ctx, option, int(value)), self._ctx)

    def kernel_times(self):
        kt = _abi.KernelTimes()
        self.lib.check(self.lib.get_kernel_times(self._ctx, C.byref(kt)), self._ctx)
        return kt.as_dict()

    def scene_info(self):
        info = _abi.SceneInfo()
        self.lib.check(self.lib.get_scene_info(self._ctx, C.byref(info)), self._ctx)
        return info.as_dict()

    def close(self):
        self._pinned = {}                      # ptb_destroy unregisters what was page-locked
        if self._group is not None:
            self.lib.group_destroy(self._group)
            self._group = None
            self._ctx = None
        if self._ctx is not None:
            self.lib.destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
