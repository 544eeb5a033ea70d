"""The BVH8 traversal ray by ray, on rays chosen to break it.

Every render's hits come from ray_prep / node_hitmask / tri_test* / walk<> (ptb_bvh8.h), run either by the plain walk (traverse<>, as
k_primary runs it) or by the persistent k_trace + k_exact of the wavefront loop.  The other hit tests reach them only through camera
rays and whole images; here the known-answer test PTB_KAT_RAY (input row o[3], d[3], tmax, any_hit; output row object id, original
triangle id, t, b1, b2, or occluded 0/1) feeds them single rays, and PTB_KAT_RAY_WAVEFRONT puts the same rows through k_trace and k_exact
(the path pool for closest hits, the shadow queue for any hits).  Each answer is held against
  (a) the oracle port (oracle/port), row by row: the reference's decisions near edges, and
  (b) a float64 brute force over all world-space triangles: two-sided, barycentrics >= 0, 0 <= t < tmax (any hit: t < 0.999 * tmax,
      ghosts passing), the nearest wins, a texel of alpha < 0.5 rejects.
The meshes are built so that their world-space vertices are exact in float32 (a power-of-two scale, an identity or 90-degree rotation,
integer translations, vertices on a dyadic grid): (b) sees the very triangles the device tests.

Where (b) calls a row clearly (barycentric margin >= MARGIN, no other candidate within T_REL of the winner's t, t not within T_REL of
the bound, no alpha lookup within TEXEL_EPS of a texel border) the answer must be (b)'s: the same ids, t within T_REL (t_tol: never
below one rounding of the coordinates), a miss a miss.  Inside that band the answer must be the port's (its hit or miss, its t, its
triangle or one (b) finds tied with it) or (b)'s (a candidate (b) cannot rule out, at (b)'s t; a miss or no occlusion where (b) finds
no candidate).  The reference's own node tests decide some rows of the band against all triangles: a ray lying in a plane through
vertices with a zero direction component makes its slab test compute 0 * inf = NaN and drop the node (a ray sliding along a face of an
axis-aligned mesh), and its box rounding can drop a ray that only touches a corner; the BVH8 walk keeps both, as (b) does.

Families: signed zeros (axis-parallel rays with +-0 in the other components: these missed every node whose slab held the origin
until ray_prep took the sign of its substitute from `d < 0`), flat nodes (a planar grid: every box flat on one axis), shared edges and
vertices of closed meshes, the same probes far from the origin and at extreme scales, tmax edges with ghosts and alpha-mapped sheets,
the device refit at a pose turned by exactly 90 degrees, random rays through a 100k-triangle soup, and the subsurface render of an
axis-aligned cube (whose probes run along -N0, Tg, Tg2: all carry a -0.0).

devsim (tests/devsim) steps the same headers on the host with the plain walk for both ids; the GPU runs both routes.
"""
import numpy as np
import pytest
from parity_cases import case_sss_converged, triangle_soup

from pathtracer_b200 import _abi, scenes
from pathtracer_b200.api import Raytracer, Sphere, Texture, TriMesh

MARGIN = 1e-4        # barycentric margin of a clear row
T_REL = 1e-5         # t: agreement, runner-up distance and distance to the bound, relative (measured worst on devsim against (b): 1e-7
                     # on the axis-aligned meshes; 6e-5 on a soup ray 5e-4 from a triangle, 0.24 of t_tol)
TEXEL_EPS = 1e-3     # alpha: a texel coordinate this close to a texel border is not clear
INF = float("inf")
F32 = np.float32


def routes(lib):
    return [_abi.KAT_RAY, _abi.KAT_RAY_WAVEFRONT] if lib.prefix == "ptb_" else [_abi.KAT_RAY]


# ---- meshes with exact float32 world-space vertices ---------------------------------------------------------------------------------
def cube(lo, hi):
    """12 triangles of the box [lo, hi] (vertices (8, 3), triangles (12, 3))"""
    lo, hi = np.asarray(lo, np.float64), np.asarray(hi, np.float64)
    v = np.array([[(hi if (k >> a) & 1 else lo)[a] for a in range(3)] for k in range(8)])
    f = [(0, 2, 3, 1), (4, 5, 7, 6), (0, 1, 5, 4), (2, 6, 7, 3), (0, 4, 6, 2), (1, 3, 7, 5)]
    t = [(a, b, c) for a, b, c, d in f] + [(a, c, d) for a, b, c, d in f]
    return v, np.array(t)


def merge(parts):
    vs, ts, n = [], [], 0
    for v, t in parts:
        vs.append(v); ts.append(t + n); n += len(v)
    return np.concatenate(vs), np.concatenate(ts)


def stacked_cubes():
    """four unit-shaped boxes stacked along y with gaps, extent [-0.875, 1] in y"""
    return merge([cube((-0.25, -0.875 + 0.5 * k, -0.25), (0.25, -0.5 + 0.5 * k, 0.25)) for k in range(4)])


def staircase():
    """a voxel staircase of 0.25 cells over x in [-1, 1] (coincident faces between neighbours included)"""
    return merge([cube((-1 + 0.25 * i, -1 + 0.25 * j, -0.25), (-0.75 + 0.25 * i, -0.75 + 0.25 * j, 0.25)) for i in range(8) for j in range(i // 2 + 1)])


def flat_grid(nx=128, nz=40):
    """2 * nx * nz triangles in the plane y = 0, cells of 1/64"""
    x, z = np.arange(nx + 1) / 64 - 1, (np.arange(nz + 1) - nz / 2) / 64
    X, Z = np.meshgrid(x, z, indexing="ij")
    v = np.stack([X, np.zeros_like(X), Z], -1).reshape(-1, 3)
    i = np.arange(nx)[:, None] * (nz + 1) + np.arange(nz)[None, :]
    a, b, c, d = i, i + 1, i + nz + 1, i + nz + 2
    return v, np.concatenate([np.stack([a, c, b], -1).reshape(-1, 3), np.stack([b, c, d], -1).reshape(-1, 3)])


def icosphere(grid=2.0 ** -8):
    """an icosahedron subdivided once (80 triangles, closed), vertices rounded to a dyadic grid"""
    p = (1 + 5 ** 0.5) / 2
    v = [(-1, p, 0), (1, p, 0), (-1, -p, 0), (1, -p, 0), (0, -1, p), (0, 1, p), (0, -1, -p), (0, 1, -p), (p, 0, -1), (p, 0, 1), (-p, 0, -1), (-p, 0, 1)]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6), (7, 1, 8),
         (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7), (9, 8, 1)]
    v = [np.array(x, np.float64) / np.linalg.norm(x) for x in v]
    mid, tris = {}, []

    def m(a, b):
        if (min(a, b), max(a, b)) not in mid:
            c = v[a] + v[b]
            v.append(c / np.linalg.norm(c))
            mid[(min(a, b), max(a, b))] = len(v) - 1
        return mid[(min(a, b), max(a, b))]
    for a, b, c in f:
        ab, bc, ca = m(a, b), m(b, c), m(c, a)
        tris += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
    return np.round(np.array(v) / grid) * grid, np.array(tris)


class Placed:
    """a mesh in unit space (vertices (n, 3), triangles (m, 3)) at scale s (a power of two), rotation R (entries 0, +-1) and integer
    translation T: world = s * R u + T, exact in float32"""

    def __init__(self, v, t, s=1.0, T=(0, 0, 0), R=None, ghost=False, alpha=None, uv=None):
        self.v, self.t, self.s, self.T = np.asarray(v, np.float64), np.asarray(t), float(s), np.asarray(T, np.float64)
        self.R = np.eye(3) if R is None else np.asarray(R, np.float64)
        self.ghost, self.alpha, self.uv = ghost, alpha, uv

    def world(self):
        w = self.s * (self.v @ self.R.T) + self.T
        assert np.array_equal(w.astype(F32).astype(np.float64), w), "world-space vertices must be exact in float32"
        return w[self.t]

    def trimesh(self, R=None, T=None):
        """TriMesh::init swaps (x, y, z) -> (-z, y, x) and is told not to centre: the input is the inverse swap of the unit-space mesh"""
        u = self.v
        vin = np.stack([u[:, 2], u[:, 1], -u[:, 0]], 1).astype(F32)
        n = len(self.t)
        uvi = self.t if self.uv is not None else np.full((n, 3), -1)
        tri = np.concatenate([self.t, uvi, np.full((n, 3), -1), np.zeros((n, 1))], 1).astype(np.int32)
        m = TriMesh(vin, np.zeros((0, 3), F32), self.uv if self.uv is not None else np.zeros((0, 2), F32), tri, center=False)
        m.scale, m.rotation_center = self.s, np.zeros(3, F32)
        m.mat_rotation = (self.R if R is None else np.asarray(R)).astype(F32)
        m.max_translation = (self.T if T is None else np.asarray(T)).astype(F32)
        mat = scenes.phong((.6, .5, .4), 0.1, 20.0)
        if self.alpha is not None:
            mat["alpha"] = Texture(1.0, self.alpha)
        m.set_material(0, **mat)
        m.ghost = self.ghost
        return m


def ray_scene(L, meshes, setup=None):
    """the light and the dome far away (object ids 0 and 1), then the meshes (ids 2...); no ground plane"""
    rt = Raytracer(L).loadScene()
    rt.s.objects = [Sphere((70000, 90000, -50000), 1.0), Sphere((0, 0, 0), 1000000, normal_swapped=True)]
    for p in meshes:
        rt.s.addObject(p.trimesh())
    if setup:
        setup(rt)
    return rt.commit()


# ---- (b): the float64 brute force -----------------------------------------------------------------------------------------------------
def alpha_clear(p, k, u, v):
    """(rejects, certain) of an alpha lookup on triangle k of mesh p at barycentrics (u, v): the map depends on the column only"""
    uv = p.uv[p.t[k]]
    uu = uv[..., 0, 0] * (1 - u - v) + uv[..., 1, 0] * u + uv[..., 2, 0] * v
    x = uu * (p.alpha.shape[1] - 1)
    col = np.clip(np.floor(x), 0, p.alpha.shape[1] - 1).astype(np.int64)
    frac = x - np.floor(x)
    return p.alpha[0, col, 0] < 0.5, (np.minimum(frac, 1 - frac) >= TEXEL_EPS) & (uu > 0) & (uu < 1)


def brute(meshes, rows):
    """per row: (object id, original triangle id, t, b1, b2) of (b) (misses -1; any-hit rows: occluded 0/1, 0, ...), whether (b) calls
    the row clearly, and the candidates it cannot rule out ({object id * 10^7 + triangle id: t}: near an edge, a texel border or t = 0)"""
    W = np.concatenate([p.world() for p in meshes])
    owner = np.concatenate([np.full(len(p.t), 2 + i) for i, p in enumerate(meshes)])
    local = np.concatenate([np.arange(len(p.t)) for p in meshes])
    ghost = np.concatenate([np.full(len(p.t), p.ghost) for p in meshes])
    v0, e1, e2 = W[:, 0], W[:, 1] - W[:, 0], W[:, 2] - W[:, 0]
    n = len(rows)
    out = np.zeros((n, 5)); out[:, :3] = -1
    clear = np.zeros(n, bool)
    near_sets = []
    chunk = max(1, 2000000 // len(W))
    for s in range(0, n, chunk):
        r = rows[s:s + chunk]
        o, d, lim, anyh = r[:, None, :3], r[:, None, 3:6], r[:, 6].copy(), r[:, 7] != 0
        lim[anyh] *= 0.999
        with np.errstate(all="ignore"):
            pv = np.cross(d, e2[None])
            det = (e1[None] * pv).sum(-1)
            inv = 1 / det
            tv = o - v0[None]
            u = (tv * pv).sum(-1) * inv
            q = np.cross(tv, e1[None])
            v = (d * q).sum(-1) * inv
            t = (e2[None] * q).sum(-1) * inv
            m = np.minimum(np.minimum(u, v), 1 - u - v)
        L = lim[:, None]
        tol = 1e-6 * max(p.s for p in meshes)
        rej = np.zeros(m.shape, bool)
        unsure = np.zeros(m.shape, bool)
        for i, p in enumerate(meshes):
            if p.alpha is None:
                continue
            sel = owner == 2 + i
            with np.errstate(all="ignore"):
                rr, cc = alpha_clear(p, local[sel][None, :], u[:, sel], v[:, sel])
            rej[:, sel], unsure[:, sel] = rr, ~cc
        skip = ghost[None] & anyh[:, None]
        ok = np.isfinite(t) & (det != 0) & ~skip
        valid = ok & (m >= 0) & (t >= 0) & (t < L) & ~rej
        near = ok & (m > -MARGIN) & (t > -tol) & (t < L * (1 + T_REL)) & ~(rej & ~unsure)
        sure = valid & (m >= MARGIN) & ((t == 0) | (t >= tol)) & (t < L * (1 - T_REL)) & ~unsure
        tv_ = np.where(valid, t, INF)
        w = np.argmin(tv_, 1)
        hit = np.isfinite(tv_[np.arange(len(r)), w])
        for k in range(len(r)):
            row = s + k
            if anyh[k]:
                out[row, :] = 0
                out[row, 0] = float(hit[k])
                clear[row] = sure[k].any() or not near[k].any()
                continue
            if not hit[k]:
                clear[row] = not near[k].any()
                continue
            j = w[k]
            tw = t[k, j]
            others = near[k].copy(); others[j] = False
            clear[row] = sure[k, j] and not (others & (t[k] <= tw + T_REL * abs(tw) + tol)).any()
            out[row] = (owner[j], local[j], tw, u[k, j], v[k, j])
        near_sets += [dict(zip(owner[near[k]] * 10 ** 7 + local[near[k]], t[k][near[k]])) for k in range(len(r))]
    return out, clear, near_sets


# ---- the comparison ---------------------------------------------------------------------------------------------------------------------
def hits_a_triangle(rows):
    return rows[:, 1] >= 0


def t_tol(rows, t):
    """T_REL of t, and no less than what one rounding of the coordinates (origin, hit point) moves t by: a ray that starts next to a
    triangle has a tiny t whose relative error is large"""
    o, d = rows[:, :3], rows[:, 3:6]
    p = np.abs(o + np.where(np.isfinite(t), t, 0)[:, None] * d).max(1)
    return T_REL * np.abs(t) + 2.0 ** -22 * np.maximum(np.abs(o).max(1), p) / np.linalg.norm(d, axis=1)


def check_rows(got, port, bf, clear, near_sets, rows, label):
    """the rules of the module docstring; returns (clear rows, rows of the band, worst |t - t_(b)| / t_tol on clear hits)"""
    anyh = rows[:, 7] != 0
    cl = clear & ~anyh
    # any hit: (b) where it is clear, the port's or (b)'s answer in the band
    bad = anyh & clear & (got[:, 0] != bf[:, 0])
    assert not bad.any(), f"{label}: {int(bad.sum())} clear any-hit rows differ from the brute force, e.g. {rows[bad][:3].tolist()}"
    bad = anyh & ~clear & (got[:, 0] != port[:, 0]) & (got[:, 0] != bf[:, 0])
    assert not bad.any(), f"{label}: {int(bad.sum())} any-hit rows of the band differ from the port and the brute force"
    # closest hit, clear rows: (b)'s answer (a non-triangle answer is a miss for (b))
    gt, bt, pt = hits_a_triangle(got), hits_a_triangle(bf), hits_a_triangle(port)
    bad = cl & ((gt != bt) | (gt & ((got[:, 0] != bf[:, 0]) | (got[:, 1] != bf[:, 1]))))
    assert not bad.any(), (f"{label}: {int(bad.sum())} of {int(cl.sum())} clear rows differ from the brute force, e.g. rows "
                           f"{rows[bad][:3].tolist()} -> {got[bad][:3].tolist()}, want {bf[bad][:3].tolist()}")
    both = cl & gt
    r = np.abs(got[both, 2] - bf[both, 2]) / t_tol(rows[both], bf[both, 2])
    worst = float(r.max()) if len(r) else 0.0
    assert worst <= 1, f"{label}: t off by {worst:.2f} x its tolerance on a clear row"
    # closest hit, the band: the port's answer (its triangle, or one (b) finds tied with it), or (b)'s (a candidate it cannot rule
    # out, at its t; a miss where it finds none)
    tol_p = t_tol(rows, port[:, 2])
    for k in np.nonzero(~clear & ~anyh)[0]:
        if not gt[k]:
            if (not pt[k] and got[k, 0] == port[k, 0]) or not bt[k]:
                continue
        else:
            key = int(got[k, 0]) * 10 ** 7 + int(got[k, 1])
            tn = near_sets[k].get(key)
            if pt[k] and abs(got[k, 2] - port[k, 2]) <= tol_p[k] and (
                    (got[k, 0] == port[k, 0] and got[k, 1] == port[k, 1]) or (tn is not None and abs(tn - port[k, 2]) <= tol_p[k])):
                continue
            if tn is not None and abs(tn - got[k, 2]) <= t_tol(rows[k:k + 1], np.array([tn]))[0]:
                continue
        raise AssertionError(f"{label}: row {rows[k].tolist()} of the band answers {got[k].tolist()}, the port {port[k].tolist()}, "
                             f"and (b) has no candidate that matches")
    return int(clear.sum()), int((~clear).sum()), worst


def run_family(lib, port, meshes, rows, label, setup=None, min_clear=0.5):
    """commit on both sides, ask every route of `lib` and the port, hold them against (b)"""
    rows = np.asarray(rows, np.float64)
    assert np.array_equal(rows[:, :7].astype(F32).astype(np.float64), rows[:, :7], equal_nan=True), "rows must be float32 values"
    bf, clear, near = brute(meshes, rows)
    assert clear.mean() >= min_clear, f"{label}: only {clear.mean():.3f} of the rows are clear: the probes miss their purpose"
    a = ray_scene(port, meshes, setup)
    want = a.kat(_abi.KAT_RAY, rows)
    a.close()
    b = ray_scene(lib, meshes, setup)
    stats = []
    for which in routes(lib):
        got = b.kat(which, rows)
        stats.append(check_rows(got, want, bf, clear, near, rows, f"{label} / KAT {which}"))
    b.close()
    return bf, clear, stats


# ---- rays ------------------------------------------------------------------------------------------------------------------------------
def signed_zero_dirs():
    """the 24 axis-parallel directions: +-1 on one axis, each of +0 and -0 on the two others"""
    out = []
    for ax in range(3):
        for sg in (1.0, -1.0):
            for z1 in (0.0, -0.0):
                for z2 in (0.0, -0.0):
                    d = [z1, z2]
                    d.insert(ax, sg)
                    out.append(d)
    return np.array(out)


LATERAL = (-1, -0.875, -0.625, -0.5, -0.25, -0.125, 0, 0.0625, 0.25, 0.375, 0.5, 0.625, 0.875, 1)   # box planes and cell centres of both meshes
AXIAL = (-3, -0.875, -0.4375, 0, 0.25, 0.625, 3)


def rows_from(o, d, tmax, any_hit):
    o, d = np.atleast_2d(o), np.atleast_2d(d)
    n = max(len(o), len(d))
    return np.concatenate([np.broadcast_to(o, (n, 3)), np.broadcast_to(d, (n, 3)), np.broadcast_to(np.reshape(tmax, (-1, 1)), (n, 1)),
                           np.full((n, 1), float(any_hit))], 1)


def both_kinds(o, d, dist):
    """every ray as a closest-hit query (tmax = inf) and as a shadow query of length `dist`"""
    return np.concatenate([rows_from(o, d, INF, 0), rows_from(o, d, dist, 1)])


def signed_zero_rows(s=1.0, T=(0, 0, 0), stride=1):
    o, d = [], []
    for dv in signed_zero_dirs():
        ax = int(np.argmax(np.abs(dv)))
        for a in AXIAL:
            for l1 in LATERAL:
                for l2 in LATERAL:
                    p = [l1, l2]
                    p.insert(ax, a)
                    o.append(p); d.append(dv)
    o, d = np.array(o)[::stride], np.array(d)[::stride]
    return both_kinds(s * o + np.asarray(T, np.float64), d, 2.5 * s)


def edge_vertex_rows(p, rng, n_origins=3):
    """rays at the midpoints of the edges and at the vertices of mesh p, from outside (distance 3) and from the centre"""
    v = p.v
    edges = {tuple(sorted((a, b))) for tri in p.t for a, b in ((tri[0], tri[1]), (tri[1], tri[2]), (tri[2], tri[0]))}
    targets = np.concatenate([np.array([(v[a] + v[b]) / 2 for a, b in sorted(edges)]), v])
    o, d = [], []
    for tg in targets:
        for k in range(n_origins):
            q = rng.normal(size=3)
            src = np.round((tg + 3 * q / np.linalg.norm(q)) * 16) / 16
            o.append(src); d.append(tg - src)
        o.append(np.zeros(3)); d.append(tg)
    o, d = p.s * np.array(o) + p.T, (p.s * np.array(d)).astype(F32).astype(np.float64)
    return both_kinds(o, d, 2.0)       # t is in units of d: the target lies at t = 1


# ---- 1: signed zeros ------------------------------------------------------------------------------------------------------------------
def case_signed_zeros(lib, port):
    out = []
    for name, mesh in (("stacked cubes", stacked_cubes()), ("staircase", staircase())):
        bf, clear, st = run_family(lib, port, [Placed(*mesh)], signed_zero_rows(), f"signed zeros, {name}")
        # the family does what it is for: many clear hits on rays with a -0 component
        rows = signed_zero_rows()
        negz = (np.signbit(rows[:, 3:6]) & (rows[:, 3:6] == 0)).any(1)
        assert (clear & negz & (bf[:, 1] >= 0) & (rows[:, 7] == 0)).sum() > 300
        out.append(st)
    return out


def test_signed_zeros_devsim(devsim, port):
    case_signed_zeros(devsim, port)


@pytest.mark.gpu
def test_signed_zeros_gpu(gpu, port):
    case_signed_zeros(gpu, port)


# ---- 2: flat nodes -----------------------------------------------------------------------------------------------------------------------
def flat_rows(rng, n=600):
    """a planar grid at y = 0: steep and grazing rays from above, rays in the plane (det = 0: a miss on either side), and origins on a
    face (t = 0: a hit)"""
    px = (rng.integers(-60, 60, n) + rng.integers(1, 16, n) / 16) / 64
    pz = (rng.integers(-18, 18, n) + rng.integers(1, 16, n) / 16) / 64
    one = np.ones(n)
    steep = np.stack([rng.integers(-8, 9, n) / 64, -one, rng.integers(-8, 9, n) / 64], 1)
    graze = np.stack([one, -np.full(n, 2.0 ** -7), rng.integers(-8, 9, n) / 32], 1)
    inplane = np.stack([one, np.where(rng.random(n) < 0.5, 0.0, -0.0), rng.integers(-8, 9, n) / 16], 1)
    up = np.stack([rng.integers(-4, 5, n) / 16, np.where(rng.random(n) < 0.5, 1.0, -1.0), rng.integers(-4, 5, n) / 16], 1)
    o_above = np.stack([px, np.full(n, 0.5), pz], 1)
    o_graze = np.stack([px - 1, np.full(n, 2.0 ** -8), pz], 1)
    o_on = np.stack([px, np.where(rng.random(n) < 0.5, 0.0, -0.0), pz], 1)
    o_par = np.stack([px - 1, np.full(n, 0.25), pz], 1)
    return np.concatenate([both_kinds(o_above, steep, 2.0), both_kinds(o_graze, graze, 4.0), both_kinds(o_on, inplane, 4.0),
                           both_kinds(o_par, inplane, 4.0), both_kinds(o_on, up, 4.0)])


def case_flat_nodes(lib, port):
    g = Placed(*flat_grid())
    assert len(g.t) >= 10000
    rows = flat_rows(np.random.default_rng(3))
    bf, clear, st = run_family(lib, port, [g], rows, "flat grid")
    n = len(rows) // 10
    inplane = slice(4 * n, 8 * n)
    assert (bf[inplane, 0][rows[inplane, 7] == 0] == -1).all() and (bf[inplane, 0][rows[inplane, 7] != 0] == 0).all(), "in-plane rays miss"
    t0 = slice(8 * n, 9 * n)
    assert (bf[t0, 2] == 0).all() and clear[t0].mean() > 0.8, "rays from a face hit it at t = 0"
    return st


def test_flat_nodes_devsim(devsim, port):
    case_flat_nodes(devsim, port)


@pytest.mark.gpu
def test_flat_nodes_gpu(gpu, port):
    case_flat_nodes(gpu, port)


# ---- 3 / 4: shared edges and vertices; scale and distance --------------------------------------------------------------------------------
PLACEMENTS = [(1.0, (1000, 0, 0)), (1.0, (10000, -10000, 10000)), (1.0, (30000, 0, -30000)), (2.0 ** -10, (0, 0, 0)), (2.0 ** 10, (0, 0, 0))]


def case_edges(lib, port, s=1.0, T=(0, 0, 0), stride=1):
    rng = np.random.default_rng(5)
    out = []
    for name, mesh in (("cube", cube((-1, -1, -1), (1, 1, 1))), ("icosphere", icosphere())):
        p = Placed(*mesh, s=s, T=T)
        rows = edge_vertex_rows(p, rng)
        if name == "cube":
            rows = np.concatenate([rows, signed_zero_rows(s, T, stride)])
        out.append(run_family(lib, port, [p], rows, f"edges, {name}, scale {s}, at {T}", min_clear=0.2)[2])
    return out


def test_edges_devsim(devsim, port):
    case_edges(devsim, port)


@pytest.mark.gpu
def test_edges_gpu(gpu, port):
    case_edges(gpu, port)


@pytest.mark.parametrize("s,T", PLACEMENTS)
def test_scale_and_distance_devsim(devsim, port, s, T):
    case_edges(devsim, port, s, T, stride=3)


@pytest.mark.gpu
@pytest.mark.parametrize("s,T", PLACEMENTS)
def test_scale_and_distance_gpu(gpu, port, s, T):
    case_edges(gpu, port, s, T, stride=3)


# ---- 5: tmax edges, ghosts, alpha-mapped sheets ----------------------------------------------------------------------------------------------
def alpha_sheet(z):
    """an 8 x 8-quad sheet in the plane z with an alpha map of columns 2 texels wide (each triangle straddles opaque and clear)"""
    g = np.arange(9) / 4 - 1
    X, Y = np.meshgrid(g, g, indexing="ij")
    v = np.stack([X, Y, np.full_like(X, z)], -1).reshape(-1, 3)
    uv = np.stack([(X + 1) / 2, (Y + 1) / 2], -1).reshape(-1, 2).astype(F32)
    i = np.arange(8)[:, None] * 9 + np.arange(8)[None, :]
    t = np.concatenate([np.stack([i, i + 9, i + 1], -1).reshape(-1, 3), np.stack([i + 1, i + 9, i + 10], -1).reshape(-1, 3)])
    cols = ((np.arange(64) // 2) % 2).astype(np.float32)
    alpha = np.repeat(np.broadcast_to(cols[None, :, None], (4, 64, 1)), 3, -1).copy()
    return v, t, uv, alpha


def case_tmax_edges(lib, port):
    rng = np.random.default_rng(9)
    # tmax just beyond / short of a clear hit, shadow rays of length t_hit / 0.999 (1 +- 2^-20), t_hit and 2 t_hit
    p = Placed(*stacked_cubes())
    base = signed_zero_rows()[::5]
    base = base[base[:, 7] == 0]
    bf, clear, _ = brute([p], base)
    keep = clear & (bf[:, 1] >= 0) & (bf[:, 2] > 0)
    o, d, th = base[keep, :3], base[keep, 3:6], bf[keep, 2]
    e = 2.0 ** -20
    rows = [rows_from(o, d, th * (1 + e), 0), rows_from(o, d, th * (1 - e), 0)]
    for dist in (th / 0.999 * (1 + e), th / 0.999 * (1 - e), th, 2 * th):
        rows.append(rows_from(o, d, dist, 1))
    rows = np.concatenate(rows)
    rows[:, 6] = rows[:, 6].astype(F32)
    run_family(lib, port, [p], rows, "tmax edges", min_clear=0.0)
    # a ghost box in front of an opaque one: closest hits see it, shadow rays pass through it
    ghost, solid = Placed(*cube((-1, -1, 0.5), (1, 1, 1)), ghost=True), Placed(*cube((-0.5, -0.5, -1), (0.5, 0.5, 0)))
    xy = (rng.integers(-15, 16, (400, 2)) + 0.5) / 16
    o = np.concatenate([xy, np.full((400, 1), 3.0)], 1)
    rows = both_kinds(o, np.array([0.0, -0.0, -1.0]), 5.0)
    bf, _, _ = run_family(lib, port, [ghost, solid], rows, "ghost")
    assert (bf[:400, 0] == 2).mean() > 0.9 and 0.1 < bf[400:, 0].mean() < 0.6, "closest hits on the ghost, shadow rays through it"
    # two alpha-mapped sheets in front of a box
    v1, t1, uv, alpha = alpha_sheet(0.5)
    v2 = v1.copy(); v2[:, 2] = 0.25
    sheets = [Placed(v1, t1, alpha=alpha, uv=uv), Placed(v2, t1, alpha=alpha[:, ::-1].copy(), uv=uv), Placed(*cube((-1, -1, -1), (1, 1, -0.5)))]
    xy = (rng.integers(-255, 256, (800, 2)) + rng.random((800, 2)).round(3)) / 256
    o = np.concatenate([xy, np.full((800, 1), 2.0)], 1)
    d = np.concatenate([rng.integers(-8, 9, (800, 2)) / 128, -np.ones((800, 1))], 1)
    rows = both_kinds(o.astype(F32).astype(np.float64), d, 3.0)
    bf, _, _ = run_family(lib, port, sheets, rows, "alpha sheets")
    cl = rows[:, 7] == 0
    assert all(0.02 < (bf[cl, 0] == k).mean() < 0.8 for k in (2, 3, 4)), "both sheets and the box take hits"
    # three alpha-tested triangles 1/8 apart, small enough to share a node: their tests run in the node's slot order whichever side
    # the ray comes from, so from one side k_trace leaves the farther candidates for k_exact first, which must keep the nearest
    v, _, uv, alpha = alpha_sheet(0)
    tri = np.array([[0, 72, 8]])
    stack = merge([(np.concatenate([v[:, :2], np.full((81, 1), z)], 1), tri) for z in (0.0, 0.125, 0.25)])
    uv3 = np.concatenate([uv] * 3)
    p = Placed(*stack, alpha=alpha, uv=uv3)
    xy = (rng.integers(-240, 200, (600, 2)) + 0.5) / 256
    keep = xy[:, 0] + xy[:, 1] < -0.1                    # inside the triangle (-1, -1), (1, -1), (-1, 1)
    xy = xy[keep]
    o = np.concatenate([np.concatenate([xy, np.full((len(xy), 1), 1.0)], 1), np.concatenate([xy, np.full((len(xy), 1), -1.0)], 1)])
    d = np.concatenate([np.tile([[2.0 ** -9, 0.0, -1.0]], (len(xy), 1)), np.tile([[2.0 ** -9, -0.0, 1.0]], (len(xy), 1))])
    rows = both_kinds(o, d, 3.0)
    bf, _, _ = run_family(lib, port, [p], rows, "alpha stack")
    n = len(xy)
    assert ((bf[:2 * n, 1] >= 0).mean() > 0.3 and np.isin(bf[:n, 1], [2]).mean() > 0.2 and np.isin(bf[n:2 * n, 1], [0]).mean() > 0.2), \
        "the nearest triangle of the stack takes the opaque rays from either side"


def test_tmax_edges_devsim(devsim, port):
    case_tmax_edges(devsim, port)


@pytest.mark.gpu
def test_tmax_edges_gpu(gpu, port):
    case_tmax_edges(gpu, port)


# ---- 6: the refit at a pose turned by exactly 90 degrees ----------------------------------------------------------------------------------------
R90 = np.array([[0, 0, 1], [0, 1, 0], [-1, 0, 0]], np.float64)     # about y: +x -> -z


@pytest.mark.gpu
def test_refit_at_a_right_angle_gpu(gpu, port):
    T1 = np.array([1000, 7, -1000], np.float64)
    meshes0 = [Placed(*stacked_cubes()), Placed(*icosphere(), T=(3, 0, 0))]
    meshes1 = [Placed(p.v, p.t, R=R90, T=p.T + T1) for p in meshes0]

    def keyed(rt):
        for m, p in zip(rt.s.objects[2:], meshes0):
            m.add_keyframe(0)
            m.mat_rotation, m.max_translation = R90.astype(F32), (p.T + T1).astype(F32)
            m.add_keyframe(10)
            m.mat_rotation, m.max_translation = np.eye(3, dtype=F32), p.T.astype(F32)
    rows = np.concatenate([signed_zero_rows(1.0, T1, stride=2), edge_vertex_rows(meshes1[1], np.random.default_rng(2))])
    bf, clear, near = brute(meshes1, rows)
    rt = ray_scene(gpu, meshes0, keyed)
    first = rt.kat(_abi.KAT_RAY, rows[:64])     # a query at frame 0, so that the re-pose is a refit of a committed scene
    rt.set_frame(10)
    fresh = ray_scene(gpu, meshes1)
    ora = ray_scene(port, meshes1)
    want = ora.kat(_abi.KAT_RAY, rows)
    assert rt.scene_info()["ms_refit"] >= 0 and first.shape == (64, 5)
    for which in routes(gpu):
        got, ref = rt.kat(which, rows), fresh.kat(which, rows)
        assert rt.scene_info()["ms_refit"] > 0, "the re-pose ran on the device"
        # the refit keeps the committed tree, so ties at shared edges may be met in another order than in a fresh tree; every clear
        # row must be answered bit for bit alike
        same = (got == ref).all(1)
        assert same[clear].all(), f"KAT {which}: the refit answers {int((~same[clear]).sum())} clear rows unlike a fresh commit"
        check_rows(got, want, bf, clear, near, rows, f"refit / KAT {which}")
    for x in (rt, fresh, ora):
        x.close()


# ---- 7: random rays over the 100k soup -----------------------------------------------------------------------------------------------------------
def case_soup_rays(lib, port, n=400):
    v, _, _, tri = triangle_soup(100000, 11)
    p = Placed(np.stack([-v[:, 2], v[:, 1], v[:, 0]], 1).astype(np.float64), tri[:, :3], s=16.0)   # TriMesh::init's axes of the file's
    rng = np.random.default_rng(17)
    o_out = rng.normal(size=(n, 3)); o_out = 40 * o_out / np.linalg.norm(o_out, axis=1, keepdims=True)
    o_in = rng.uniform(-12, 12, (n, 3))
    tgt = rng.uniform(-14, 14, (n, 3))
    o = np.concatenate([o_out, o_in]).astype(F32).astype(np.float64)
    d = np.concatenate([tgt - o_out, rng.normal(size=(n, 3))]).astype(F32).astype(np.float64)
    rows = both_kinds(o, d, rng.uniform(0.05, 1.0, 2 * n).astype(F32) * np.linalg.norm(d, axis=1))
    rows[:, 6] = rows[:, 6].astype(F32)
    bf, clear, st = run_family(lib, port, [p], rows, "soup", min_clear=0.9)
    assert (bf[: 2 * n, 1] >= 0).mean() > 0.5 and 0.2 < bf[2 * n:, 0].mean() < 0.9
    return st


def test_soup_rays_devsim(devsim, port):
    case_soup_rays(devsim, port)


@pytest.mark.gpu
def test_soup_rays_gpu(gpu, port):
    case_soup_rays(gpu, port)


# ---- 8: the subsurface render of an axis-aligned cube ---------------------------------------------------------------------------------------------
def ksub_cube_scene(L, W=48, H=48, spp=64):
    """config_sss's material on a cube with axis-aligned faces (12 triangles, one normal per face): every subsurface probe of this
    mesh runs along an axis with -0.0 in its other components"""
    rt = scenes.base(L, W, H, spp)
    v, t = cube((-1, -1, -1), (1, 1, 1))
    nrm = np.array([(0, 0, -1), (0, 0, 1), (0, -1, 0), (0, 1, 0), (-1, 0, 0), (1, 0, 0)] * 2, np.float32)
    tri = np.concatenate([t, np.full((12, 3), -1), np.repeat(np.arange(12)[:, None], 3, 1), np.zeros((12, 1))], 1).astype(np.int32)
    m = scenes._place_like_gui(TriMesh(v.astype(F32), nrm, np.zeros((0, 2), F32), tri), scale=24.0)
    m.set_material(0, **scenes.phong((.5, .45, .4), (.1, .1, .1), 30.0, Ksub=Texture((.8, .5, .4))))
    rt.s.addObject(m)
    rt.cam.position = np.array([22, 12, 45], F32)
    d = np.array([0, -15, 0], F32) - rt.cam.position
    rt.cam.direction = d / F32(np.linalg.norm(d))
    return rt


def test_ksub_cube_devsim(devsim, port):
    case_sss_converged(devsim, port, mk=ksub_cube_scene)


@pytest.mark.gpu
def test_ksub_cube_gpu(gpu, port):
    case_sss_converged(gpu, port, mk=ksub_cube_scene)
