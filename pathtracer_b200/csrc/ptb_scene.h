// ptb_scene.h — device-side scene description and the per-path stages of the wavefront integrator.
//
// The stages restate Raytracer::getColor (Raytracer.cpp:196-664) as per-path functions that the kernels in
// ptb_engine.cu call once per queue entry.  The linear path (no fog, ghost object, background photograph or
// subsurface material in the scene: every loop iteration pushes at most one contribution) is:
//     raygen_one  — precomputeRayBatch + Camera::generateDirection (Raytracer.cpp:1404-1420)
//     extend_one  — Scene::intersection (Geometry.cpp:589-688)
//     shade_one   — getColor's per-bounce body: emission, mirror, dielectric, NEE sample, BSDF sample
//     shadow_one  — Scene::intersection_shadow (Geometry.cpp:691-744) + the deferred direct term
//     splat_pixel — the Gaussian splat (Raytracer.cpp:1604-1659)
// Scenes with a medium, ghosts, a background photograph or subsurface scattering take shade_branch_one instead
// of shade_one: the same loop body with those branches, walking the contribution tree level by level
// (DESIGN.md section 10).
#pragma once
#include "../../include/ptb200.h"
#include "ptb_bvh8.h"

namespace ptb {

enum { OBJ_MESH = 0, OBJ_SPHERE = 1, OBJ_PLANE = 2, OBJ_CYLINDER = 3, OBJ_POINTSET = 4, OBJ_YARNS = 5 };
enum { FLAG_MIRROR = 1, FLAG_FLIP = 2, FLAG_FLAT = 4, FLAG_GHOST = 8, FLAG_DISPLAY_EDGES = 16, FLAG_NOT_INLINE = 1 << 16 };
// A point-set disc sits in the BVH8 as the triangle circumscribed about it (in its plane, inscribed radius 1.1 r): every ray that can
// hit the disc hits that triangle's interior, the threshold in its e1.w is +inf, so k_trace classifies it "left for k_exact" like a
// near-edge candidate, with no disc code and no extra test in the traversal loop; k_exact runs the reference's disc test.
PTB_HD void disc_cover_triangle(V3 c, V3 n, float r, V3& v0, V3& v1, V3& v2) {
    const float nn = sqrtf(norm2(n));
    const V3 z = nn > 0.f ? n / nn : v3(0, 0, 1);
    const V3 a = fabsf(z.x) < 0.57f ? v3(1, 0, 0) : (fabsf(z.y) < 0.57f ? v3(0, 1, 0) : v3(0, 0, 1));
    const V3 u = normalize(cross(z, a)), w = cross(z, u);
    const float R = 2.2f * r;
    v0 = c + R * w;
    v1 = c + R * (-0.8660254f * u - 0.5f * w);
    v2 = c + R * (0.8660254f * u - 0.5f * w);
}
#define PTB_GROUP_DISC (-2)   /* TriUV::group of a point-set disc (its TriShade holds normal, colour, centre, radius) */
// A yarn segment (an open Cylinder of a Yarns object) sits in the BVH8 as the EIGHT triangles of a prism around it (equilateral cross-
// section of inscribed radius 1.1 r, the ends 0.1 r beyond A and B): a ray that meets the tube between its end planes is inside the prism
// there, so it crosses the prism's boundary before (entering) or after (leaving: a ray that starts inside).  Like the disc's triangle
// these are always "left for k_exact" (e1.w = +inf).  The face a ray leaves through may lie beyond a nearer hit although the tube
// itself does not, so (a) their e2.w = 0 switches the `t < t_best` cut of the fast test off and (b) all eight enter the BVH8 with the
// TUBE's box (yarn_box), not their own: a ray reaches them whenever it can reach the tube.  idx 0..5: the three side faces, 6 / 7: the ends.
#define PTB_YARN_COVER 8
PTB_HD void yarn_cover_triangle(V3 a, V3 b, float r, int idx, V3& v0, V3& v1, V3& v2) {
    const V3 ab = b - a;
    const float l = sqrtf(norm2(ab));
    const V3 z = l > 0.f ? ab / l : v3(0, 0, 1);
    const V3 h = fabsf(z.x) < 0.57f ? v3(1, 0, 0) : (fabsf(z.y) < 0.57f ? v3(0, 1, 0) : v3(0, 0, 1));
    const V3 u = normalize(cross(z, h)), w = cross(z, u);
    const float slack = 2e-6f * fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(b.x))), fmaxf(fabsf(b.y), fabsf(b.z))) + 1e-3f * r;
    const float R = 2.2f * r + 2.f * slack, pad = 0.1f * r + slack;
    const V3 a2 = a - pad * z, b2 = b + pad * z;
    const V3 c0 = R * w, c1 = R * (-0.8660254f * u - 0.5f * w), c2 = R * (0.8660254f * u - 0.5f * w);
    if (idx >= 6) {
        const V3 e = idx == 6 ? a2 : b2;
        v0 = e + c0; v1 = e + c1; v2 = e + c2;
        return;
    }
    const int j = idx >> 1;
    const V3 cj = j == 0 ? c0 : (j == 1 ? c1 : c2), ck = j == 0 ? c1 : (j == 1 ? c2 : c0);
    if (idx & 1) { v0 = b2 + cj; v1 = a2 + ck; v2 = b2 + ck; }
    else { v0 = a2 + cj; v1 = a2 + ck; v2 = b2 + cj; }
}
// The box all covering triangles of a yarn segment enter the BVH8 with: the tube's own (A +- r, B +- r like Yarns::build_bbox,
// TriangleMesh.cpp:1519-1533), with a few ulps of the coordinates of slack.
PTB_HD void yarn_box(V3 a, V3 b, float r, float lo[3], float hi[3]) {
    const float s = r * (1.f + 1e-3f) + 2e-6f * fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(b.x))), fmaxf(fabsf(b.y), fabsf(b.z)));
    lo[0] = fminf(a.x, b.x) - s; lo[1] = fminf(a.y, b.y) - s; lo[2] = fminf(a.z, b.z) - s;
    hi[0] = fmaxf(a.x, b.x) + s; hi[1] = fmaxf(a.y, b.y) + s; hi[2] = fmaxf(a.z, b.z) + s;
}
#define PTB_GROUP_YARN (-3)   /* TriUV::group of a yarn segment's covering triangle (its TriShade holds the axis d and the end point A) */
enum { SLOT_KD = 1, SLOT_KS = 2, SLOT_NE = 4, SLOT_TRANSP = 8, SLOT_REFR = 16, SLOT_NORMAL = 32, SLOT_ALPHA = 64, SLOT_KSUB = 128 };

struct ObjectDev {          // Object / Sphere / Plane fields the path reads (Geometry.h:240-672, 849-1217)
    int32_t type, flags, brdf, merl;
    int32_t mat_base, n_groups;   // materials[mat_base + group], group < n_groups else defaults
    int32_t slot_mask;            // union of the slots present on the object (Geometry.h:979 test for spheres)
    int32_t pad;
    float trans[12], inv_trans[12], rot[9];
    float a[3];                   // Sphere::O / Plane::A / Cylinder::A
    float n[3];                   // Plane::vecN / Cylinder::d (unit axis)
    float R, R2;
    float len, pad2;              // Cylinder::len
};
struct MaterialDev {
    uint32_t present;
    TexDev Kd, Ks, Ne, transp, refr, normal, alpha, Ksub;
};
struct alignas(16) TriUV {     // what the in-traversal alpha test and the uv interpolation need (32 B)
    float u0, v0, u1, v1, u2, v2;
    int32_t group;             // TriangleIndices::group (-1: no uv / default material)
    int32_t object_has_uv;     // object id | (has_uv << 31)
};
struct alignas(16) TriShade {  // object-space vertex normals and tangents + original triangle id (80 B)
    float n0[3], n1[3], n2[3], t0[3], t1[3], t2[3];
    int32_t orig;
    int32_t pad;
};

// The handful of analytic objects every ray is tested against travel INSIDE the kernel parameter block (constant
// bank, uniform loads) instead of being gathered from global memory by every thread.
#define PTB_INLINE_ANALYTIC 8
struct AnalyticDev {
    int32_t type, id;           // OBJ_SPHERE / OBJ_PLANE, scene object id (bit 30 of `type`: Object::ghost, skipped by shadow rays)
    float inv_trans[12];
    float a[3], n[3], R2;
    float len;                  // Cylinder::len
};

#define PTB_ANALYTIC_GHOST (1 << 30)
#define PTB_ANALYTIC_LINEAR_ID (1 << 29)   /* inv_trans = [I | t] exactly */
struct FogDev {                 // Scene::fog_* (Geometry.h:1371-1377) + the ground level fogContribution reads (Raytracer.cpp:54)
    float density, absorption, density_decay, absorption_decay, phase_aniso, ground;
    int32_t type, phase_type;
};

struct SceneDev {
    const F4* nodes;            // 5 x F4 per Node8
    const F4* tris;             // 3 x F4 per triangle, leaf order
    const F4* tris_obj;         // the same triangles as the reference holds them: OBJECT-space corners A, B, C (A.w = object id); read by
                                // tri_exact for rays near an edge and by the key-frame refit (null: the fast test decides everything)
    const TriUV* tri_uv;
    const TriShade* tri_shade;
    const ObjectDev* objects;
    const MaterialDev* materials;
    const float* texels;
    const uint8_t* envmap;
    const float* merl;          // per table 3*PTB_MERL_N floats, pre-scaled (see merl_eval)
    int32_t n_objects, has_mesh, envW, envH, has_envmap;
    int32_t has_exotic;         // some Cylinder / PointSet / Yarns object: the kernels that carry their code
    float envmap_intensity, lightPower, radiusLight;
    V3 centerLight;
    int32_t n_inline, n_extra;  // analytic objects held inline below / left in `objects` (flag FLAG_NOT_INLINE)
    int32_t has_fog, has_ghost; // fog_density > 1e-8 (Raytracer.cpp:206) / any Object::ghost
    int32_t has_sss;            // some mesh group carries a non-zero subsurface albedo Ksub (Raytracer.cpp:270)
    const float* background;    // Scene::background (Geometry.h:1365), bgW*bgH*3 floats, or null
    int32_t bgW, bgH;
    FogDev fog;
    AnalyticDev analytic[PTB_INLINE_ANALYTIC];
};

struct AlphaCtx {
    const TriUV* tri_uv;
    const ObjectDev* objects;
    const MaterialDev* materials;
    const float* texels;
    const F4* tris_obj;         // object-space corners, see SceneDev
};

PTB_HD V3 xf_point(const float* m, V3 v) {   // Object::apply_transformation (Geometry.h:362-368)
    return v3(m[0] * v.x + m[1] * v.y + m[2] * v.z + m[3], m[4] * v.x + m[5] * v.y + m[6] * v.z + m[7],
              m[8] * v.x + m[9] * v.y + m[10] * v.z + m[11]);
}
PTB_HD V3 xf_dir(const float* m, V3 v) {     // apply_rotation_scaling (369-375)
    return v3(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[4] * v.x + m[5] * v.y + m[6] * v.z, m[8] * v.x + m[9] * v.y + m[10] * v.z);
}
PTB_HD V3 xf_rot(const float* m, V3 v) {     // apply_rotation (376-382), 3x3
    return v3(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[3] * v.x + m[4] * v.y + m[5] * v.z, m[6] * v.x + m[7] * v.y + m[8] * v.z);
}

PTB_HD bool tri_exact_available(const AlphaCtx* c) { return c != nullptr && c->tris_obj != nullptr; }
// apply_inverse_rotation_scaling / apply_(inverse_)transformation (Geometry.h:362-397) with one rounding per operation, in the reference's order
PTB_HD V3 xf_dir_rn(const float* m, V3 d) {
    return v3(add_rn(add_rn(mul_rn(m[0], d.x), mul_rn(m[1], d.y)), mul_rn(m[2], d.z)), add_rn(add_rn(mul_rn(m[4], d.x), mul_rn(m[5], d.y)), mul_rn(m[6], d.z)),
              add_rn(add_rn(mul_rn(m[8], d.x), mul_rn(m[9], d.y)), mul_rn(m[10], d.z)));
}
PTB_HD V3 xf_point_rn(const float* m, V3 v) {
    return v3(add_rn(add_rn(add_rn(mul_rn(m[0], v.x), mul_rn(m[1], v.y)), mul_rn(m[2], v.z)), m[3]),
              add_rn(add_rn(add_rn(mul_rn(m[4], v.x), mul_rn(m[5], v.y)), mul_rn(m[6], v.z)), m[7]),
              add_rn(add_rn(add_rn(mul_rn(m[8], v.x), mul_rn(m[9], v.y)), mul_rn(m[10], v.z)), m[11]));
}
// Cylinder::intersection (Geometry.h:740-754) in the reference's own arithmetic, one rounding per operation.  For a thin yarn far from the
// ray origin `delta = b*b - 4*a*c` cancels five digits: an FMA anywhere in it moves t by 1e-6 relative, which is 1e-4 of the tube's
// radius and hence of the radial shading normal.  (The analytic Cylinder objects, radius of the order of their distance, keep cylinder_t.)
PTB_HD bool cylinder_t_rn(V3 a0, V3 ax, float R, float len, V3 o, V3 d, float& t) {
    const V3 X = sub3_rn(d, scale_rn(dot_rn(d, ax), ax));
    const V3 oa = sub3_rn(o, a0);
    const V3 Y = sub3_rn(oa, scale_rn(dot_rn(oa, ax), ax));
    const float a = dot_rn(X, X);
    const float b = mul_rn(2.f, dot_rn(X, Y));
    const float c = sub_rn(dot_rn(Y, Y), mul_rn(R, R));
    const float delta = sub_rn(mul_rn(b, b), mul_rn(mul_rn(4.f, a), c));
    if (delta < 0) return false;
    const float sdelta = sqrt_rn(delta);
    const float t2 = div_rn(add_rn(-b, sdelta), mul_rn(2.f, a));
    if (t2 < 0) return false;
    const float t1 = div_rn(sub_rn(-b, sdelta), mul_rn(2.f, a));
    t = (t1 > 0) ? t1 : t2;
    const V3 P = add3_rn(o, scale_rn(t, d));
    const float dP = dot_rn(sub3_rn(P, a0), ax);
    if (dP < 0 || dP > len) return false;
    return true;
}

// Scene::intersection's ray transform (Geometry.cpp:603-605, Geometry.h:383-397) + the Triangle constructor and
// Triangle::intersection (TriangleMesh.h:70-104) + the `localt < t` of the traversal (TriangleMesh.cpp:1197), one rounding per operation.
PTB_HD_NOINLINE bool tri_exact(const AlphaCtx* c, int prim, V3 o, V3 d, float tbest, float& t, float& b1, float& b2) {
#if defined(__CUDA_ARCH__)
    const float4 qa = __ldg(reinterpret_cast<const float4*>(c->tris_obj) + 3 * (size_t)prim), qb = __ldg(reinterpret_cast<const float4*>(c->tris_obj) + 3 * (size_t)prim + 1),
                 qc = __ldg(reinterpret_cast<const float4*>(c->tris_obj) + 3 * (size_t)prim + 2);
    const int obj = __float_as_int(qa.w) & 0x0fffffff;     // (bits 28..30: which covering triangle of a yarn segment, see scene_host.cpp)
#else
    const F4 qa = c->tris_obj[3 * (size_t)prim], qb = c->tris_obj[3 * (size_t)prim + 1], qc = c->tris_obj[3 * (size_t)prim + 2];
    const int obj = (int)(f2u(qa.w) & 0x0fffffffu);
#endif
    const float* m = c->objects[obj].inv_trans;
    if (c->objects[obj].type == OBJ_YARNS) {
        // cyls[i]->intersection (Geometry.h:740-766) on the object-space ray + the `localt < t` of Yarns::intersection (TriangleMesh.cpp:1711):
        // A = end point, B.w = radius, C = unit axis d and length
        float tt;
        if (!cylinder_t_rn(v3(qa.x, qa.y, qa.z), v3(qc.x, qc.y, qc.z), qb.w, qc.w, xf_point_rn(m, o), xf_dir_rn(m, d), tt)) return false;
        if (!(tt < tbest)) return false;
        t = tt; b1 = 0; b2 = 0;
        return true;
    }
    if (c->objects[obj].type == OBJ_POINTSET) {
        // Disk::intersection (Geometry.h:1110-1118) on the object-space ray (xf_dir / xf_point are the reference's own expressions;
        // this path is not compared bit for bit): A = centre, B.xyz = normal, B.w = radius
        const V3 dl = xf_dir(m, d), ol = xf_point(m, o);
        const V3 ctr = v3(qa.x, qa.y, qa.z), N = v3(qb.x, qb.y, qb.z);
        const float tt = dot(ctr - ol, N) / dot(dl, N);
        if (tt < 0 || tt != tt) return false;
        const V3 P = ol + tt * dl;
        if (!(norm2(P - ctr) <= qb.w * qb.w)) return false;
        if (!(tt < tbest)) return false;
        t = tt; b1 = 0; b2 = 0;
        return true;
    }
    const V3 dl = xf_dir_rn(m, d), ol = xf_point_rn(m, o);
    const V3 A = v3(qa.x, qa.y, qa.z);
    const V3 u = sub3_rn(v3(qb.x, qb.y, qb.z), A), v = sub3_rn(v3(qc.x, qc.y, qc.z), A);
    const V3 N = cross_rn(u, v);
    const float m11 = dot_rn(u, u), m22 = dot_rn(v, v), m12 = dot_rn(u, v);
    // `1. / (m11*m22 - m12*m12)` narrowed to float (TriangleMesh.h:77): the correctly rounded float quotient equals the narrowed double
    // quotient except when the latter falls within 2^-29 of a rounding midpoint
    const float invdetm = div_rn(1.f, sub_rn(mul_rn(m11, m22), mul_rn(m12, m12)));
    const float tt = div_rn(dot_rn(sub3_rn(A, ol), N), dot_rn(dl, N));
    if (tt < 0 || tt != tt) return false;
    const V3 w = sub3_rn(add3_rn(ol, scale_rn(tt, dl)), A);
    const float b11 = dot_rn(w, u), b21 = dot_rn(w, v);
    const float beta = mul_rn(sub_rn(mul_rn(b11, m22), mul_rn(b21, m12)), invdetm);
    if (beta < 0) return false;
    const float gamma = mul_rn(sub_rn(mul_rn(b21, m11), mul_rn(b11, m12)), invdetm);
    if (gamma < 0) return false;
    const float alpha = sub_rn(sub_rn(1.f, beta), gamma);
    if (alpha < 0) return false;
    if (!(tt < tbest)) return false;
    if (beta != beta || gamma != gamma) return false;   // (sliver: the reference accepts NaN barycentrics and patches them up later, App. D#17)
    t = tt; b1 = beta; b2 = gamma;
    return true;
}

// TriangleMesh.cpp:1198-1205: reject the hit when the group's alpha map reads < 0.5 at the hit's uv
PTB_HD bool alpha_rejects(const AlphaCtx* c, int prim, float b1, float b2) {
#if defined(__CUDA_ARCH__)
    const float4 q0 = __ldg(reinterpret_cast<const float4*>(c->tri_uv + prim));
    const float4 q1 = __ldg(reinterpret_cast<const float4*>(c->tri_uv + prim) + 1);
    TriUV tu; tu.u0 = q0.x; tu.v0 = q0.y; tu.u1 = q0.z; tu.v1 = q0.w; tu.u2 = q1.x; tu.v2 = q1.y;
    tu.group = __float_as_int(q1.z); tu.object_has_uv = __float_as_int(q1.w);
#else
    const TriUV tu = c->tri_uv[prim];
#endif
    if (tu.group < 0 || tu.object_has_uv >= 0) return false;  // needs a group and uvs
    const ObjectDev& ob = c->objects[tu.object_has_uv & 0x7fffffff];
    if (tu.group >= ob.n_groups) return false;
    const MaterialDev& m = c->materials[ob.mat_base + tu.group];
    if (!(m.present & SLOT_ALPHA)) return false;
    // rounded operation by operation (TriangleMesh.cpp:1200-1201): which texel (int)(u * (W - 1)) names must not depend on an FMA
    const float alpha = sub_rn(sub_rn(1.f, b1), b2);
    float u = add_rn(add_rn(mul_rn(tu.u0, alpha), mul_rn(tu.u1, b1)), mul_rn(tu.u2, b2));
    float v = add_rn(add_rn(mul_rn(tu.v0, alpha), mul_rn(tu.v1, b1)), mul_rn(tu.v2, b2));
    u = tex_wrap(u); v = tex_wrap(v);
    return tex_red(m.alpha, c->texels, u, v) < 0.5f;
}

// Sphere::intersection roots (Geometry.h:943-962): object-space ray, non-unit direction
PTB_HD bool sphere_t(const float* A, float R2, V3 o, V3 d, float& t) {
    const V3 O = v3(A[0], A[1], A[2]);
    const V3 oc = o - O;
    const float b = dot(d, oc);
    const float a = norm2(d);
    const float c = norm2(oc) - R2;
    const float delta = b * b - a * c;
    if (delta < 0) return false;
    const float sq = sqrtf(delta);
    const float inva = 1.f / a;
    const float t2 = (-b + sq) * inva;
    if (t2 < 0) return false;
    const float t1 = (-b - sq) * inva;
    t = (t1 > 0) ? t1 : t2;
    return true;
}
// Plane::intersection (Geometry.h:1142-1148)
PTB_HD bool plane_t(const float* A, const float* Nn, V3 o, V3 d, float& t) {
    const V3 N = v3(Nn[0], Nn[1], Nn[2]);
    const float ddot = dot(d, N);
    if (fabsf(ddot) < 1E-9f) return false;
    t = dot(v3(A[0], A[1], A[2]) - o, N) / ddot;
    if (t <= 0.f) return false;
    return true;
}

// Cylinder::intersection (Geometry.h:740-766): roots of |X t + Y|^2 = R^2 with X, Y the parts of direction / origin - A orthogonal to
// the axis; the nearer positive root must lie between the end planes (the farther one is never tried).  No test against the best t
// so far; a ray parallel to the axis yields NaN, which the caller's `t < min_t` discards.
PTB_HD bool cylinder_t(const float* A, const float* D, float R2, float len, V3 o, V3 d, float& t) {
    const V3 a0 = v3(A[0], A[1], A[2]), ax = v3(D[0], D[1], D[2]);
    const V3 X = d - dot(d, ax) * ax;
    const V3 oa = o - a0;
    const V3 Y = oa - dot(oa, ax) * ax;
    const float a = norm2(X);
    const float b = 2 * dot(X, Y);
    const float c = norm2(Y) - R2;
    const float delta = b * b - 4 * a * c;
    if (delta < 0) return false;
    const float sdelta = sqrtf(delta);
    const float t2 = (-b + sdelta) / (2 * a);
    if (t2 < 0) return false;
    const float t1 = (-b - sdelta) / (2 * a);
    t = (t1 > 0) ? t1 : t2;
    const V3 P = o + t * d;
    const float dP = dot(P - a0, ax);
    if (dP < 0 || dP > len) return false;
    return true;
}

#define PTB_HIT_MISS (-1)
PTB_HD int32_t hit_id_analytic(int obj) { return -2 - obj; }

// Nearest hit over the analytic objects (Sphere / Plane) of Scene::intersection's loop (Geometry.cpp:601-626):
// object-space rays, world t.  Meshes are handled by the wide BVH afterwards.
// EXOTIC = the scene holds Cylinder or PointSet objects.  The kernels of the linear path are also compiled without their code
// (EXOTIC = false; the benchmark configurations have none): it costs the 64-register k_shade spills otherwise (+3 %, profiles/r02j).
template <bool EXOTIC = true>
PTB_HD bool analytic_t(int type, const float* inv_trans, const float* A, const float* N, float R2, float len, V3 o, V3 d, float& t) {
    V3 dl, ol;
    if (type & PTB_ANALYTIC_LINEAR_ID) {   // uniform per object; same bits as the general form for m = [I | t]
        dl = d;
        ol = v3(o.x + inv_trans[3], o.y + inv_trans[7], o.z + inv_trans[11]);
    } else {
        dl = xf_dir(inv_trans, d);
        ol = xf_point(inv_trans, o);
    }
    if (EXOTIC && (type & 0xff) == OBJ_CYLINDER) return cylinder_t(A, N, R2, len, ol, dl, t);
    return ((type & 0xff) == OBJ_SPHERE) ? sphere_t(A, R2, ol, dl, t) : plane_t(A, N, ol, dl, t);
}
template <bool EXOTIC = true>
PTB_HD void analytic_closest(const SceneDev& sc, V3 o, V3 d, float& tmin, int32_t& id) {
    tmin = INFINITY;
    id = PTB_HIT_MISS;
    int best = -1;
    // object order matters only for exact ties (strict `t < min_t`, Geometry.cpp:615): inline objects keep scene order
    for (int i = 0; i < sc.n_inline; i++) {
        const AnalyticDev& ob = sc.analytic[i];
        float t;
        if (analytic_t<EXOTIC>(ob.type, ob.inv_trans, ob.a, ob.n, ob.R2, ob.len, o, d, t) && t < tmin) { tmin = t; best = ob.id; }
    }
    if (sc.n_extra > 0)
        for (int i = 0; i < sc.n_objects; i++) {
            const ObjectDev& ob = sc.objects[i];
            if (ob.type == OBJ_MESH || !(ob.flags & FLAG_NOT_INLINE)) continue;
            float t;
            if (analytic_t<EXOTIC>(ob.type, ob.inv_trans, ob.a, ob.n, ob.R2, ob.len, o, d, t) && (t < tmin || (t == tmin && i < best))) { tmin = t; best = i; }
        }
    if (best >= 0) id = hit_id_analytic(best);
}
// Analytic part of Scene::intersection_shadow (Geometry.cpp:721-741): any object closer than 0.999*dist_light
template <bool EXOTIC = true>
PTB_HD bool analytic_occluded(const SceneDev& sc, V3 o, V3 d, float dist_light) {
    const double lim = (double)dist_light * 0.999;
    for (int i = 0; i < sc.n_inline; i++) {
        const AnalyticDev& ob = sc.analytic[i];
        if (ob.type & PTB_ANALYTIC_GHOST) continue;   // avoid_ghosts (Geometry.cpp:722)
        float t;
        if (analytic_t<EXOTIC>(ob.type, ob.inv_trans, ob.a, ob.n, ob.R2, ob.len, o, d, t) && (double)t < lim) return true;
    }
    if (sc.n_extra > 0)
        for (int i = 0; i < sc.n_objects; i++) {
            const ObjectDev& ob = sc.objects[i];
            if (ob.type == OBJ_MESH || !(ob.flags & FLAG_NOT_INLINE) || (ob.flags & FLAG_GHOST)) continue;
            float t;
            if (analytic_t<EXOTIC>(ob.type, ob.inv_trans, ob.a, ob.n, ob.R2, ob.len, o, d, t) && (double)t < lim) return true;
        }
    return false;
}
PTB_HD AlphaCtx alpha_ctx(const SceneDev& sc) {
    AlphaCtx ac; ac.tri_uv = sc.tri_uv; ac.objects = sc.objects; ac.materials = sc.materials; ac.texels = sc.texels; ac.tris_obj = sc.tris_obj;
    return ac;
}

// Scene::intersection: analytic objects, then the wide BVH with the analytic t as the upper bound.
template <bool COUNT>
PTB_HD void extend_ray(const SceneDev& sc, V3 o, V3 d, Hit& hit, int32_t& id, TraverseCounters* cnt) {
    float tmin;
    analytic_closest(sc, o, d, tmin, id);
    hit.b1 = 0; hit.b2 = 0; hit.prim = -1;
    if (sc.has_mesh) {
        const AlphaCtx ac = alpha_ctx(sc);
        Hit h;
        if (traverse<false, COUNT>(sc.nodes, sc.tris, &ac, o, d, tmin, h, cnt)) { hit = h; id = h.prim; tmin = h.t; }
    }
    hit.t = tmin;
}

struct Surface {   // MaterialValues (BRDF.h:7-20) + what getColor needs about the object
    V3 P, N, Kd, Ks, Ne, Ke, Ksub;
    float refr_index;
    bool transp;
    int32_t object;
};

// Object::queryMaterial (Geometry.h:399-445)
PTB_HD void query_material(const SceneDev& sc, const ObjectDev& ob, int group, float u, float v, Surface& s) {
    u = tex_wrap(u); v = tex_wrap(v);
    const bool in_range = group >= 0 && group < ob.n_groups;
    const MaterialDev* m = in_range ? &sc.materials[ob.mat_base + group] : nullptr;
    const uint32_t present = m ? m->present : 0u;
    s.Kd = (present & SLOT_KD) ? tex_vec(m->Kd, sc.texels, u, v) : v3(1, 1, 1);
    s.Ks = (present & SLOT_KS) ? tex_vec(m->Ks, sc.texels, u, v) : v3(0, 0, 0);
    s.Ne = (present & SLOT_NE) ? tex_vec(m->Ne, sc.texels, u, v) : v3(1, 1, 1);
    s.transp = (present & SLOT_TRANSP) ? (tex_red(m->transp, sc.texels, u, v) < 0.5f) : false;
    s.refr_index = (present & SLOT_REFR) ? tex_red(m->refr, sc.texels, u, v) : 1.3f;
    s.Ke = v3(0, 0, 0);
    s.Ksub = (present & SLOT_KSUB) ? tex_vec(m->Ksub, sc.texels, u, v) : v3(0, 0, 0);   // read by the branching shader only
}

// Rebuild the shading point of a hit: Object::intersection's material part + the tail of Scene::intersection.
template <bool EXOTIC = true>
PTB_HD void surface_from_hit(const SceneDev& sc, V3 o, V3 d, const Hit& hit, int32_t id, Surface& s) {
    V3 Nl;  // object-space shading normal before rotation
    const ObjectDev* obp;
    if (id >= 0) {
        // ---- TriMesh::getMaterial (TriangleMesh.cpp:919-1026) ----
        const TriUV tu = sc.tri_uv[id];
        const TriShade ts = sc.tri_shade[id];
        s.object = tu.object_has_uv & 0x7fffffff;
        obp = &sc.objects[s.object];
        if (EXOTIC && tu.group == PTB_GROUP_YARN) {
            // ---- the tail of cyls[i]->intersection (Geometry.h:756-763) on the segment's OWN default material: n0 = axis d, n1 = A ----
            // (one rounding per operation: the radial normal is the small difference of two points far from the origin)
            const V3 dl = xf_dir_rn(obp->inv_trans, d), ol = xf_point_rn(obp->inv_trans, o);
            const V3 Pl = add3_rn(ol, scale_rn(hit.t, dl));
            const V3 a0 = v3(ts.n1[0], ts.n1[1], ts.n1[2]), ax = v3(ts.n0[0], ts.n0[1], ts.n0[2]);
            const V3 proj = add3_rn(a0, scale_rn(dot_rn(sub3_rn(Pl, a0), ax), ax));
            s.Kd = v3(1, 1, 1); s.Ks = v3(0, 0, 0); s.Ne = v3(1, 1, 1); s.transp = false; s.refr_index = 1.3f; s.Ke = v3(0, 0, 0); s.Ksub = v3(0, 0, 0);
            s.P = xf_point(obp->trans, Pl);
            s.N = fast_normalize(xf_rot(obp->rot, sub3_rn(Pl, proj)));      // never flipped: the segment's flip_normals, not the Yarns object's
            return;
        }
        if (EXOTIC && tu.group == PTB_GROUP_DISC) {
            // ---- PointSet::intersection's tail (PointSet.cpp:192-217): n0 = normal, t0 = colour, n1 = centre, n2[0] = radius ----
            const V3 dl = xf_dir(obp->inv_trans, d), ol = xf_point(obp->inv_trans, o);
            const V3 Pl = ol + hit.t * dl;
            Nl = normalize(v3(ts.n0[0], ts.n0[1], ts.n0[2]));
            query_material(sc, *obp, 0, 0.f, 0.f, s);
            if (dot(Nl, dl) > 0 && !s.transp) Nl = -Nl;
            if (obp->flags & FLAG_FLIP) Nl = -Nl;
            s.Kd = v3(ts.t0[0], ts.t0[1], ts.t0[2]);
            if (obp->flags & FLAG_DISPLAY_EDGES) {
                const float r2 = norm2(Pl - v3(ts.n1[0], ts.n1[1], ts.n1[2]));
                if ((double)r2 > (double)ts.n2[0] * (double)ts.n2[0] * 0.95 * 0.95) s.Kd = v3(0, 0, 0);
            }
            s.P = xf_point(obp->trans, Pl);
            s.N = fast_normalize(xf_rot(obp->rot, Nl));
            return;
        }
        float beta = hit.b1, gamma = hit.b2;
        float alpha = 1.f - beta - gamma;
        const bool has_uv = tu.object_has_uv < 0;
        float u = 0, v = 0;
        if (has_uv) {
            u = tu.u0 * alpha + tu.u1 * beta + tu.u2 * gamma;
            v = tu.v0 * alpha + tu.v1 * beta + tu.v2 * gamma;
        }
        query_material(sc, *obp, tu.group, u, v, s);
        Nl = v3(ts.n0[0], ts.n0[1], ts.n0[2]) * alpha + v3(ts.n1[0], ts.n1[1], ts.n1[2]) * beta + v3(ts.n2[0], ts.n2[1], ts.n2[2]) * gamma;
        Nl = normalize(Nl);
        const bool in_range = tu.group >= 0 && tu.group < obp->n_groups;
        if (has_uv && in_range && (sc.materials[obp->mat_base + tu.group].present & SLOT_NORMAL)) {
            const MaterialDev& m = sc.materials[obp->mat_base + tu.group];
            V3 tangent = v3(ts.t0[0], ts.t0[1], ts.t0[2]) * alpha + v3(ts.t1[0], ts.t1[1], ts.t1[2]) * beta + v3(ts.t2[0], ts.t2[1], ts.t2[2]) * gamma;
            tangent = normalize(tangent);
            const V3 bitangent = cross(Nl, tangent);
            const V3 nl = tex_normal(m.normal, sc.texels, u, v);  // un-wrapped uv, as getMaterial passes them (TriangleMesh.cpp:961)
            V3 Ns = nl.x * tangent + nl.y * bitangent + nl.z * Nl;
            if (Ns.x == 0.f && Ns.y == 0.f && Ns.z == 0.f) Ns = Nl;
            Nl = normalize(Ns);
        }
        if (obp->flags & FLAG_FLIP) Nl = -Nl;
        s.P = o + hit.t * d;  // world-space triangles: same point as apply_transformation(o' + t d')
    } else {
        s.object = -2 - id;
        obp = &sc.objects[s.object];
        const ObjectDev& ob = *obp;
        const V3 dl = xf_dir(ob.inv_trans, d);
        const V3 ol = xf_point(ob.inv_trans, o);
        const V3 Pl = ol + hit.t * dl;
        if (ob.type == OBJ_SPHERE) {
            V3 N = Pl - v3(ob.a[0], ob.a[1], ob.a[2]);
            if (s.object == 1 && sc.has_envmap) {
                // Geometry.h:963-977: the dome with an environment map
                N = fast_normalize(N);
                const float theta = 1.f - acosf(N.y) / PTB_PI_F;
                const float phi = (float)(((double)atan2f(-N.z, N.x) + PTB_PI_D) / (double)(2.f * PTB_PI_F));
                query_material(sc, ob, 0, theta, phi, s);
                Nl = -N;
                const int idx = 3 * ((int)(theta * ((float)sc.envH - 1.f)) * sc.envW + (int)(phi * ((float)sc.envW - 1.f)));
                if (idx < 0 || idx >= 3 * sc.envW * sc.envH) s.Ke = v3(0, 0, 0);
                else s.Ke = v3((float)sc.envmap[idx], (float)sc.envmap[idx + 1], (float)sc.envmap[idx + 2]) * (100000.f / 255.f);
            } else {
                // MaterialValues() defaults when the sphere has no slot at all (BRDF.h:9-16)
                s.Kd = v3(.5f, .5f, .5f); s.Ks = v3(0, 0, 0); s.Ne = v3(100, 100, 100); s.transp = false; s.refr_index = 1.3f; s.Ksub = v3(0, 0, 0);
                if (ob.slot_mask & (SLOT_KD | SLOT_KS | SLOT_NE | SLOT_TRANSP | SLOT_REFR)) {
                    N = fast_normalize(N);
                    const float theta = 1.f - acosf(N.y) / PTB_PI_F;
                    const float phi = (atan2f(-N.z, N.x) + PTB_PI_F) / (2.f * PTB_PI_F);
                    query_material(sc, ob, 0, theta, phi, s);
                }
                s.Ke = v3(0, 0, 0);
                Nl = (ob.flags & FLAG_FLIP) ? -N : N;
            }
        } else if (EXOTIC && ob.type == OBJ_CYLINDER) {   // Geometry.h:758-763
            const V3 a0 = v3(ob.a[0], ob.a[1], ob.a[2]), ax = v3(ob.n[0], ob.n[1], ob.n[2]);
            const float dP = dot(Pl - a0, ax);
            const V3 proj = a0 + dP * ax;
            query_material(sc, ob, 0, dP / ob.len, 0.5f, s);
            Nl = Pl - proj;                      // not normalised here: Scene::intersection's fast_normalize does it
            if (ob.flags & FLAG_FLIP) Nl = -Nl;
        } else {
            Nl = v3(ob.n[0], ob.n[1], ob.n[2]);
            query_material(sc, ob, 0, Pl.x * 0.1f, Pl.z * 0.1f, s);
        }
        s.P = xf_point(ob.trans, Pl);
    }
    s.N = fast_normalize(xf_rot(obp->rot, Nl));  // Geometry.cpp:677-684
}

// ---- path pool (structure of arrays in HBM) ---------------------------------------------------------
#define PTB_DEFER_K 4    /* candidates a ray can leave for k_exact; a ray with more is re-traced there with the immediate exact test */
struct PoolDev {
    F4* ray_o;        // xyz origin
    F4* ray_d;        // xyz direction
    F4* weight;       // xyz path weight; w = bits: depth (low 16) | show_lights << 16
    F4* radiance;     // xyz accumulated radiance of the sample
    F4* hit;          // t, b1, b2, id bits
    uint64_t* rng;    // pcg32 state (inc follows from pixel/sample/seed)
    uint32_t* pixel;  // i*W + j, or 0xffffffff for an empty slot
    F4* sh_o;         // shadow queue: xyz origin, w = dist_light
    F4* sh_d;         // xyz direction, w = path slot bits
    F4* sh_c;         // xyz = path weight * direct contribution
    F4* aov_n;        // first-hit shading normal (normalValue, Raytracer.cpp:254-257); null unless the denoiser-input mode renders
    F4* aov_kd;       // first-hit albedo mat.Kd (albedoValue)
    uint32_t* root;   // branching renders (fog / ghost objects): the sample slot a contribution belongs to; null otherwise
    F4* probe_o;      // subsurface probes (entry-indexed): xyz origin, w = tmax
    F4* probe_d;      // xyz axis, w = path slot bits
    F4* probe_x;      // x,y = pcg32 state of the probe's own stream (lo, hi), z = object id bits
    F4* hit2;         // slot-indexed: the probe's answer t, b1, b2, prim bits (prim -1: nothing found)
    uint32_t* defer_prims;  // PTB_DEFER_K per ray (closest: path slot, any hit: shadow entry): triangle | flags << 28 left for k_exact
    U2* defer_rays;         // queue of the rays that left some: {path slot or shadow entry, how many}
};
// a hit as the pool stores it (hit, hit2)
PTB_HD F4 hit_record(const Hit& h) {
    F4 q; q.x = h.t; q.y = h.b1; q.z = h.b2; q.w = u2f((uint32_t)h.prim);
    return q;
}

struct FrameDev {     // per-render constants (Raytracer fields + prepare_render results)
    CameraDev cam;
    FilterDev filter;
    int32_t W, H, nb_bounces, spp_pass, k0;   // this pass traces samples k0 .. k0+spp_pass-1 of each pixel
    uint32_t seed;
    int32_t tile, tiles_x, tiles_y, shard_rank, shard_count, n_my_tiles;
    int32_t tile_shift;                       // row rotation of the tile numbering (shard_tile_shift)
    int32_t slot0;                            // first pixel slot (in the shard's tile-major pixel order) of this pass
    int32_t n_pixel_slots;                    // pixel slots in this pass
    const float* rpp;                         // randomPerPixel, 2 floats per pixel (Raytracer.cpp:1341-1344)
    int32_t box_filter;                       // has_denoiser accumulation: each sample adds (L, 1) to its own pixel, no splat (Raytracer.cpp:1631-1645)
    int32_t lowresW, lowresH;                 // progressive preview grid ceil(W/16) x ceil(H/16) (Raytracer.cpp:1329-1330)
    float* lowres;                            // imagedouble_lowres sums (Raytracer.cpp:1508-1510), or null
    F4* accum_albedo;                         // box_filter mode: per-pixel sums of the first-hit albedo / normal, or null
    F4* accum_normal;
};

// ---- tile ownership ----------------------------------------------------------------------------------------------
// Tiles are numbered row by row, every row rotated by `shift` more columns than the one above: logical id
// l = ty * tiles_x + (tx + ty * shift) % tiles_x; shard r of n owns the tiles with l % n == r and renders them in the order of l.
// Without the rotation a frame whose tile columns are a multiple of n (1024 / 64 = 16 tiles for 2, 4, 8 GPUs) is cut into vertical
// stripes, and the GPUs that get the columns with the mesh finish last (measured at 8 GPUs on C2: slowest rank 7 % over the mean).
// The shift is chosen so that owners advance by a step coprime to n from one row to the next; one shard keeps the plain order.
// default tile edge: 64 for a whole frame, 32 when the frame is shared, 16 among 8 or more (finer granularity balances the shards
// better: slowest of 8 shards of C2 at 1.034 of the mean with 64-pixel tiles, 1.020 with 32, 1.004 with 16, where the mean itself
// is 0.6 % up for the shorter tile rows; profiles/r01m_shard_balance.txt, r02s_shard_balance.txt)
inline int ptb_default_tile(int shard_count) { return shard_count >= 8 ? 16 : shard_count > 1 ? 32 : 64; }
PTB_HD int shard_tile_shift(int tiles_x, int count) {
    if (count <= 1 || tiles_x <= 1) return 0;
    for (int s = 1; s <= count; s++) {
        int a = (tiles_x + s) % count, b = count;
        while (a) { const int t = b % a; b = a; a = t; }
        if (b == 1) return s % tiles_x;
    }
    return 1 % tiles_x;
}
PTB_HD int tile_logical(int ty, int tx, int tiles_x, int shift) { return ty * tiles_x + (tx + ty * shift) % tiles_x; }
PTB_HD void tile_physical(int l, int tiles_x, int shift, int& ty, int& tx) {
    ty = l / tiles_x;
    const int lx = l - ty * tiles_x;
    tx = (lx + tiles_x - (ty * shift) % tiles_x) % tiles_x;
}

// pixel slot (tile-major order over the shard's tiles) -> (i, j); false if outside the image
PTB_HD bool slot_to_pixel(const FrameDev& f, int slot, int& i, int& j) {
    const int tp = f.tile * f.tile;
    const int lt = slot / tp, r = slot - lt * tp;
    const int tile_id = f.shard_rank + lt * f.shard_count;
    if (tile_id >= f.tiles_x * f.tiles_y) return false;
    int ty, tx;
    tile_physical(tile_id, f.tiles_x, f.tile_shift, ty, tx);
    i = ty * f.tile + r / f.tile;
    j = tx * f.tile + (r % f.tile);
    return i < f.H && j < f.W;
}

// Tile gather: does own tile `tile_id` (logical) carry frame pixel (i,j) in its (tile + apron) block?  Every pixel a shard
// touched must travel exactly once: inside an own tile it goes with that tile; in a foreign tile it goes with the first own
// tile, in row-major scan order of the 3x3 neighbourhood, whose apron covers it (two own tiles can flank the same foreign pixel).
PTB_HD bool shard_block_sends(int tile_id, int i, int j, int W, int H, int tile, int apron, int tiles_x, int tiles_y, int rank, int count, int shift) {
    if (i < 0 || i >= H || j < 0 || j >= W) return false;
    const int pty = i / tile, ptx = j / tile;
    const int pid = tile_logical(pty, ptx, tiles_x, shift);
    if (pid % count == rank) return pid == tile_id;
    for (int ty = pty - 1; ty <= pty + 1; ty++)
        for (int tx = ptx - 1; tx <= ptx + 1; tx++) {
            if (ty < 0 || ty >= tiles_y || tx < 0 || tx >= tiles_x) continue;
            const int id = tile_logical(ty, tx, tiles_x, shift);
            if (id % count != rank) continue;
            if (i < ty * tile - apron || i >= ty * tile + tile + apron || j < tx * tile - apron || j >= tx * tile + tile + apron) continue;
            return id == tile_id;
        }
    return false;
}

// sample index of a path within its pass: path % spp_pass.  spp_pass is a power of two for every frame whose pixel count is one (pool / pixels);
// the general remainder is 30 instructions and was taken twice per shaded path (ncu r02x: 5 % of k_shade's instructions).
PTB_HD int path_sample(const FrameDev& f, int path) {
    const int m = f.spp_pass - 1;
    return (f.spp_pass & m) == 0 ? (path & m) : path % f.spp_pass;
}
PTB_HD uint64_t path_inc(const FrameDev& f, int path) {  // pcg32 stream increment of the path's (pixel,sample) stream
    return (((uint64_t)(uint32_t)(f.k0 + path_sample(f, path)) ^ ((uint64_t)f.seed << 32)) << 1) | 1ULL;
}
// path state word (weight.w): depth (low 16) | show_lights | showenvmap | has_had_subsurface_interaction | pcg32 stream kind
// (0: the sample's own stream, 1: fog fork, 2: ghost fork; oracle/build_ref.py patch 7) | fog contribution awaiting its hit
enum { ST_SHOW_LIGHTS = 0x10000u, ST_SHOW_ENV = 0x20000u, ST_HAD_SS = 0x40000u, ST_KIND_SHIFT = 19, ST_KIND_MASK = 3u << 19,
       ST_FOG_PENDING = 1u << 21, ST_FOG_UNIFORM = 1u << 22, ST_SSS_WAIT = 1u << 23 /* the subsurface probe of this hit is in flight / answered */ };
PTB_HD uint32_t pack_state(int depth, bool show_lights) { return (uint32_t)depth | (show_lights ? ST_SHOW_LIGHTS : 0u) | ST_SHOW_ENV; }

// the hit record of a new ray before the BVH has seen it: the analytic half of Scene::intersection rides with the ray producer
template <bool EXOTIC = true>
PTB_HD F4 analytic_hit(const SceneDev& sc, V3 o, V3 d) {
    Hit h; h.b1 = 0; h.b2 = 0;
    analytic_closest<EXOTIC>(sc, o, d, h.t, h.prim);
    return hit_record(h);
}

// ---- stage 1: camera samples --------------------------------------------------------------------------
template <bool EXOTIC = true>
PTB_HD void raygen_one(const SceneDev& sc, const FrameDev& f, PoolDev& p, int path) {
    const int ps = path / f.spp_pass, s = path - ps * f.spp_pass;
    int i, j;
    if (!slot_to_pixel(f, f.slot0 + ps, i, j)) {   // slot of an edge tile that lies outside the frame: an empty path
        p.pixel[path] = 0xffffffffu;
        p.hit[path] = hit_record(Hit{INFINITY, 0, 0, PTB_HIT_MISS});
        return;
    }
    const uint32_t pix = (uint32_t)(i * f.W + j);
    const uint32_t k = (uint32_t)(f.k0 + s);
    Pcg32 e = pcg32_for_sample(pix, k, f.seed);
    const float dx = pcg32_uniform(e) - 0.5f;
    const float dy = pcg32_uniform(e) - 0.5f;
    const float ax = (pcg32_uniform(e) - 0.5f) * f.cam.aperture;
    const float ay = (pcg32_uniform(e) - 0.5f) * f.cam.aperture;
    V3 o, d;
    camera_ray(f.cam, i, j, dx, dy, ax, ay, o, d);
    F4 q;
    q.x = o.x; q.y = o.y; q.z = o.z; q.w = 0; p.ray_o[path] = q;
    q.x = d.x; q.y = d.y; q.z = d.z; q.w = 0; p.ray_d[path] = q;
    q.x = 1; q.y = 1; q.z = 1; q.w = u2f(pack_state(f.nb_bounces, true)); p.weight[path] = q;
    q.x = 0; q.y = 0; q.z = 0; q.w = 0; p.radiance[path] = q;
    if (f.accum_albedo) { p.aov_n[path] = q; p.aov_kd[path] = q; }   // `Vector normal, albedo;` start at zero (Vector.h:45) and stay there on a miss
    p.hit[path] = analytic_hit<EXOTIC>(sc, o, d);
    p.rng[path] = e.state;
    p.pixel[path] = pix;
    if (p.root) p.root[path] = (uint32_t)path;
}

// ---- stage 2: closest hit in the wide BVH (the analytic objects were tested by the ray's producer) ----------------
template <bool COUNT>
PTB_HD void extend_one(const SceneDev& sc, PoolDev& p, int path, TraverseCounters* cnt) {
    const F4 o = p.ray_o[path], d = p.ray_d[path];
    const F4 h0 = p.hit[path];
    const AlphaCtx ac = alpha_ctx(sc);
    Hit h;
    if (traverse<false, COUNT>(sc.nodes, sc.tris, &ac, v3(o.x, o.y, o.z), v3(d.x, d.y, d.z), h0.x, h, cnt)) p.hit[path] = hit_record(h);
}

// ---- stage 3: shade ---------------------------------------------------------------------------------------
struct ShadeOut {
    bool cont;          // the path continues: ray_o/ray_d/weight/hit were rewritten
    bool shadow;        // a shadow ray must still be traced through the BVH
    bool shadow_query;  // an intersection_shadow-equivalent query was made (ray statistics)
    F4 sh_o, sh_d, sh_c;
};

// ---- pieces of one getColor iteration shared by shade_one and shade_branch_one ------------------------------------------------
// next-event estimation: a point of the spherical light seen from P (Raytracer.cpp:494-510) and the density of its direction
struct LightSample { V3 axeOP, dirl, xl, wi; float d2; };
PTB_HD LightSample light_sample(const SceneDev& sc, V3 P, Pcg32& e) {
    LightSample l;
    l.axeOP = fast_normalize(P - sc.centerLight);
    const float l1 = pcg32_uniform(e);
    const float l2 = pcg32_uniform(e);
    l.dirl = random_cos(l.axeOP, l1, l2);
    l.xl = l.dirl * sc.radiusLight + sc.centerLight;
    const V3 toL = l.xl - P;
    l.wi = fast_normalize(toL);
    l.d2 = norm2(toL);
    return l;
}
PTB_HD float light_proba(const SceneDev& sc, const LightSample& l) {
#if defined(__CUDA_ARCH__)
    return dot(l.axeOP, l.dirl) / (PTB_PI_F * (sc.radiusLight * sc.radiusLight));
#else
    return (float)((double)dot(l.axeOP, l.dirl) / (PTB_PI_D * (double)(sc.radiusLight * sc.radiusLight)));
#endif
}
// the MERL-or-Phong choice of shade_branch_one.  shade_one spells it out: through a helper nvcc fuses different products of the MERL
// lookup into FMAs, and the linear render would no longer compute what it did.
template <bool MERL>
PTB_HD V3 brdf_eval(const SceneDev& sc, const ObjectDev& ob, const Surface& s, V3 wi, V3 wo, V3 N) {
    if (MERL && ob.brdf == 1) return merl_eval(sc.merl + (size_t)ob.merl * 3 * PTB_MERL_N, wi, wo, N);
    return phong_eval(s.Kd, s.Ks, s.Ne, wi, wo, N);
}
// the shadow ray of a direct term, for the BVH: `owner` = path or sample slot, `tag` = sh_c.w
PTB_HD void queue_shadow(ShadeOut& out, V3 so, V3 wi, float dist, uint32_t owner, V3 c, uint32_t tag) {
    out.shadow = true;
    out.sh_o.x = so.x; out.sh_o.y = so.y; out.sh_o.z = so.z; out.sh_o.w = (float)((double)dist * 0.999);
    out.sh_d.x = wi.x; out.sh_d.y = wi.y; out.sh_d.z = wi.z; out.sh_d.w = u2f(owner);
    out.sh_c.x = c.x; out.sh_c.y = c.y; out.sh_c.z = c.z; out.sh_c.w = u2f(tag);
}
// the path's next ray, with the analytic half of its closest hit
template <bool EXOTIC = true>
PTB_HD void set_next_ray(const SceneDev& sc, PoolDev& p, int path, V3 no, V3 nd, V3 nw, uint32_t state) {
    F4 q;
    q.x = no.x; q.y = no.y; q.z = no.z; q.w = 0; p.ray_o[path] = q;
    q.x = nd.x; q.y = nd.y; q.z = nd.z; q.w = 0; p.ray_d[path] = q;
    q.x = nw.x; q.y = nw.y; q.z = nw.z; q.w = u2f(state); p.weight[path] = q;
    p.hit[path] = analytic_hit<EXOTIC>(sc, no, nd);
}

// MERL = the scene holds at least one IsoMERLBRDF object; scenes without one get a kernel free of the double-precision
// lookup code (fewer registers, higher occupancy).
// AOV = this launch shades the camera rays of a denoiser-input render: the first hit's shading normal and albedo are recorded
// (`if (has_inter && nbrebonds == nb_bounces) { normalValue = N; albedoValue = mat.Kd; }`, Raytracer.cpp:254-257).
template <bool MERL, bool AOV = false, bool EXOTIC = true>
PTB_HD void shade_one(const SceneDev& sc, const FrameDev& f, PoolDev& p, int path, ShadeOut& out) {
    out.cont = false; out.shadow = false; out.shadow_query = false;
    const F4 hq = p.hit[path];
    const int32_t id = (int32_t)f2u(hq.w);
    if (id == PTB_HIT_MISS) return;                                  // Raytracer.cpp:654-657
    const F4 oq = p.ray_o[path], dq = p.ray_d[path], wq = p.weight[path];
    const V3 ro = v3(oq.x, oq.y, oq.z), rd = v3(dq.x, dq.y, dq.z);
    const V3 w = v3(wq.x, wq.y, wq.z);
    const uint32_t st = f2u(wq.w);
    const int depth = (int)(st & 0xffffu);
    const bool show_lights = (st & 0x10000u) != 0;
    Hit hit; hit.t = hq.x; hit.b1 = hq.y; hit.b2 = hq.z; hit.prim = id;
    F4 Lq = p.radiance[path];
    if (AOV && depth == f.nb_bounces) {
        Surface s0;
        surface_from_hit<EXOTIC>(sc, ro, rd, hit, id, s0);
        F4 q; q.w = 0;
        q.x = s0.N.x; q.y = s0.N.y; q.z = s0.N.z; p.aov_n[path] = q;
        q.x = s0.Kd.x; q.y = s0.Kd.y; q.z = s0.Kd.z; p.aov_kd[path] = q;
    }
    if (id == hit_id_analytic(0)) {                                  // the light, Raytracer.cpp:303-316
        const float lp = show_lights ? sc.lightPower : 0.f;
        Lq.x += w.x * lp; Lq.y += w.y * lp; Lq.z += w.z * lp;
        p.radiance[path] = Lq;
        return;
    }
    if (id == hit_id_analytic(1) && !sc.has_envmap) return;          // dome without a map: Ke = 0
    Surface s;
    surface_from_hit<EXOTIC>(sc, ro, rd, hit, id, s);
    if (s.object == 1) {                                             // env dome, Raytracer.cpp:275-301
        const V3 c = (w * sc.envmap_intensity) * s.Ke;
        Lq.x += c.x; Lq.y += c.y; Lq.z += c.z;
        p.radiance[path] = Lq;
        return;
    }
    const ObjectDev& ob = sc.objects[s.object];
    const V3 N = s.N, P = s.P;
    V3 no, nd, nw = w;
    bool nshow = show_lights;
    if (ob.flags & FLAG_MIRROR) {                                    // 413-436
        nd = reflect(rd, N);
        no = P + 0.001f * N;
    } else if (s.transp) {                                           // 438-489
        // (shade_branch_one has the same lines: as a shared helper nvcc fuses dot(Nt, rd) into FMAs the other way round)
        float n1 = 1.f, n2 = s.refr_index;
        V3 Nt = N;
        bool entering = true;
        if (dot(rd, N) > 0) { n1 = s.refr_index; n2 = 1; Nt = -N; entering = false; }
        const float c0 = dot(Nt, rd);
        const float radical = 1.f - (n1 / n2) * (n1 / n2) * (1.f - c0 * c0);
        if (radical > 0) {
            const V3 refr = (n1 / n2) * (rd - dot(rd, Nt) * Nt) - Nt * sqrtf(radical);
            const float r0 = (n1 - n2) / (n1 + n2);
            const float R0 = r0 * r0;
            float R;
            if (entering) R = R0 + (1 - R0) * pow5(1.f + dot(rd, N));
            else R = R0 + (1 - R0) * pow5(1.f - dot(refr, N));
            Pcg32 e; e.state = p.rng[path]; e.inc = path_inc(f, path);
            const float u = pcg32_uniform(e);
            p.rng[path] = e.state;
            if (u < R) { no = P + 0.001f * Nt; nd = reflect(rd, N); }
            else { no = P - 0.001f * Nt; nd = refr; }
        } else {
            no = P + 0.001f * Nt; nd = reflect(rd, N);
        }
    } else {                                                         // opaque, 490-649
        Pcg32 e; e.state = p.rng[path]; e.inc = path_inc(f, path);
        // -- next-event estimation on the spherical light (494-566)
        const LightSample l = light_sample(sc, P, e);
        const V3 wi = l.wi;
        const float d2 = l.d2;
        if (!(dot(N, wi) < 0)) {
            V3 fr;
            if (MERL && ob.brdf == 1) fr = merl_eval(sc.merl + (size_t)ob.merl * 3 * PTB_MERL_N, wi, -rd, N);
            else fr = phong_eval(s.Kd, s.Ks, s.Ne, wi, -rd, N);
            const float J = dot(l.dirl, -wi) / d2;
            const float proba = light_proba(sc, l);
            if (proba > 0.f) {
                const float g = sc.lightPower * fmaxf(0.f, dot(N, wi)) * J / proba;
                const V3 c = w * (g * fr);
                const V3 so = P + 0.01f * wi;
                const float dist = sqrtf(d2) - 0.01f;
                out.shadow_query = true;
                // analytic occluders (incl. the light itself and the dome, App. D#8) are tested here, coherently;
                // only rays they do not block go on to the BVH
                if (!analytic_occluded<EXOTIC>(sc, so, wi, dist)) {
                    if (sc.has_mesh) queue_shadow(out, so, wi, dist, (uint32_t)path, c, 0u);
                    else {
                        Lq.x += c.x; Lq.y += c.y; Lq.z += c.z;
                        p.radiance[path] = Lq;
                    }
                }
            } else {
                out.shadow_query = true;   // the reference traces this ray too; its result is unused
            }
        }
        // -- continuation (570-632)
        const uint32_t pix = p.pixel[path];
        float sx, sy;
        extensible_lattice_2d((uint32_t)(f.k0 + path_sample(f, path)), sx, sy);
        const float r1 = frac_pos(f.rpp[2 * pix] + sx);
        const float r2 = frac_pos(f.rpp[2 * pix + 1] + sy);
        float pdf;
        V3 dir;
        if (MERL && ob.brdf == 1) {
            dir = random_cos(N, r1, r2);
            pdf = (float)((double)dot(N, dir) / PTB_PI_D);
        } else {
            bool diffuse;
            const float u = pcg32_uniform(e);
            dir = phong_sample(s.Ks, s.Ne, -rd, N, r1, r2, u, pdf, diffuse);
        }
        p.rng[path] = e.state;
        if (dot(dir, N) < 0 || dot(dir, reflect(rd, N)) < 0 || pdf <= 0) return;
        V3 fi;
        if (MERL && ob.brdf == 1) fi = merl_eval(sc.merl + (size_t)ob.merl * 3 * PTB_MERL_N, dir, -rd, N);
        else fi = phong_eval(s.Kd, s.Ks, s.Ne, dir, -rd, N);
        nw = (w * fi) * (dot(N, dir) / pdf);
        no = P + 0.01f * dir;
        nd = dir;
        nshow = false;
    }
    const int ndepth = depth - 1;
    // loop-top tests of the next iteration (240-241): depth exhausted or weight below 0.01
    if (ndepth == 0 || norm2(nw) < 0.01f * 0.01f) return;
    // NaN weights fall through `<` like the reference; keep tracing them as it does
    set_next_ray<EXOTIC>(sc, p, path, no, nd, nw, pack_state(ndepth, nshow));
    out.cont = true;
}

// ---- stage 4: shadow rays through the wide BVH; unoccluded ones deliver the deferred direct term -----------------------
// an unoccluded shadow ray of a linear render adds its deferred direct term to its path's radiance (Raytracer.cpp:545-566)
PTB_HD void deliver_direct(PoolDev& p, uint32_t entry, uint32_t path) {
    const F4 c = p.sh_c[entry];
    F4 L = p.radiance[path];
    L.x += c.x; L.y += c.y; L.z += c.z;
    p.radiance[path] = L;
}
template <bool COUNT>
PTB_HD void shadow_one(const SceneDev& sc, PoolDev& p, int entry, TraverseCounters* cnt) {
    const F4 o = p.sh_o[entry], d = p.sh_d[entry];
    const AlphaCtx ac = alpha_ctx(sc);
    Hit h;
    if (!traverse<true, COUNT>(sc.nodes, sc.tris, &ac, v3(o.x, o.y, o.z), v3(d.x, d.y, d.z), o.w, h, cnt)) deliver_direct(p, (uint32_t)entry, f2u(d.w));
}

// ---- branching contributions: participating medium, ghost objects, background photograph ----------------------------
// getColor's ring of `Contrib` (Raytracer.cpp:213-247) becomes a level-synchronous tree walk: every contribution lives in a
// pool slot; a slot's continuation stays in the slot, a side branch (the in-scattered contribution of fogContribution, the
// straight-through ray of a ghost object) takes a fresh slot and its own pcg32 (oracle/build_ref.py patch 7: seed = two
// draws of a copy of the parent engine, stream = 1 fog / 2 ghost).  Radiance of every contribution is added to the sample
// slot `root` it descends from.
struct ChildOut {
    bool want;
    F4 o, d, w;        // ray origin (.w: fog: squared distance to the sampled light point, < 0 for a uniform direction), direction
                       // (.w: fog: weight factor still to be divided by proba_dir), weight + state word
    uint64_t rng;
};
struct BranchOut {
    ShadeOut base;
    ChildOut fog, ghost;
    bool ghost_pending;   // the ghost child lives only if the shadow ray in base.sh_* turns out unoccluded (Raytracer.cpp:519-537)
    bool probe;           // a subsurface probe must be answered before this hit can be shaded (get_random_intersection, Raytracer.cpp:377)
    F4 probe_o, probe_d, probe_x;
};

PTB_HD uint64_t stream_inc(const FrameDev& f, uint32_t root, uint32_t state) {
    const uint32_t kind = (state & ST_KIND_MASK) >> ST_KIND_SHIFT;
    return kind == 0 ? path_inc(f, (int)root) : (((uint64_t)kind << 1) | 1ULL);
}
PTB_HD uint64_t pcg32_fork(const Pcg32& e, uint64_t tag) {   // returns the STATE of pcg32(seed, stream = tag); its inc is (tag << 1) | 1
    Pcg32 t = e;
    const uint64_t a = pcg32_next(t), b = pcg32_next(t);
    return pcg32_seed((a << 32) | b, tag).state;
}
PTB_HD void radiance_add(PoolDev& p, uint32_t root, V3 c) {
#if defined(__CUDA_ARCH__)
    float* q = reinterpret_cast<float*>(p.radiance + root);
    atomicAdd(q, c.x); atomicAdd(q + 1, c.y); atomicAdd(q + 2, c.z);
#else
    F4& L = p.radiance[root];
    L.x += c.x; L.y += c.y; L.z += c.z;
#endif
}
PTB_HD V3 background_at(const SceneDev& sc, const FrameDev& f, uint32_t pix) {   // Raytracer.cpp:261-265, 615-619
    const int screenI = (int)(pix / (uint32_t)f.W), screenJ = (int)(pix % (uint32_t)f.W);
    int i = (int)((float)screenI / (float)f.H * (float)sc.bgH), j = (int)((float)screenJ / (float)f.W * (float)sc.bgW);
    i = i < 0 ? 0 : (i > sc.bgH - 1 ? sc.bgH - 1 : i);
    j = j < 0 ? 0 : (j > sc.bgW - 1 ? sc.bgW - 1 : j);
    const float* b = sc.background + ((size_t)i * sc.bgW + j) * 3;
    return v3(b[0], b[1], b[2]);
}
PTB_HD float int_exponential(float y0, float ysol, float beta, float s, float uy) {   // Raytracer.cpp:20-38
    if (fabsf(uy * beta) < 0.0001f) return expf(-beta * (y0 - ysol)) * s;
    return (expf(-beta * (y0 - ysol)) - expf(-beta * (y0 + s * uy - ysol))) / (uy * beta);
}
// Raytracer::fogContribution (Raytracer.cpp:40-192) up to the visibility ray: draws the scattering distance and direction from
// `e`, describes the in-scattered contribution in `ch` (its weight is completed by shade_branch_one once the ray's hit is known,
// lines 146-187) and returns the transmittance T (`attenuationFactor`).  When fogContribution returns before setting
// attenuationFactor (scatter point below the ground, line 110) the reference goes on with the previous call's value; here T.
PTB_HD float fog_sample(const SceneDev& sc, V3 ro, V3 rd, V3 lightPos, float t, V3 w, uint32_t child_state, Pcg32& e, ChildOut& ch) {
    const FogDev& fg = sc.fog;
    const bool uniform_fog = fg.type == 0;
    const float alpha = fg.absorption, sigmaT = fg.absorption_decay, ground = fg.ground;
    const float int_ext = uniform_fog ? (float)((double)(alpha * t) * 0.05) : alpha * int_exponential(ro.y, ground, sigmaT, t, rd.y);
    const float T = expf(-int_ext);
    float proba_t, random_t;
    const float clamped_t = fminf(1000.f, t);
    const float a = dot(lightPos - ro, rd);
    if (a > 0) {                                                          // equi-angular sampling, 71-84
        const V3 projP = ro + a * rd;
        const float D = sqrtf(norm2(lightPos - projP));
        const float thetaA = -atan2f(a, D);
        const float b = t - a;
        const float thetaB = atan2f(b, D);
        const float x = pcg32_uniform(e);
        random_t = D * tanf((1 - x) * thetaA + x * thetaB);
        proba_t = D / ((thetaB - thetaA) * (D * D + random_t * random_t));
        random_t += a;
    } else {                                                              // truncated exponential, 90-99
        const float alpha2 = 5.f / clamped_t;
        int guard = 0;
        do { random_t = -logf(pcg32_uniform(e)) / alpha2; } while (random_t > clamped_t && ++guard < 64);
        const float normalization = 1.f / alpha2 * (1.f - expf(-alpha2 * clamped_t));
        proba_t = expf(-alpha2 * random_t) / normalization;
    }
    const float int_ext_p = uniform_fog ? (float)((double)(alpha * random_t) * 0.05) : alpha * int_exponential(ro.y, ground, sigmaT, random_t, rd.y);
    const V3 P = ro + random_t * rd;
    if (P.y < ground) return T;
    const V3 axeOP = normalize(P - sc.centerLight);
    V3 dir;
    float d_light2 = -1.f;
    if (pcg32_uniform(e) < 0.5f) {                                        // random_uniform_sphere<float>, Vector.h:604-615
        const float r1 = pcg32_uniform(e), r2 = pcg32_uniform(e);
        const float twopi = 2.f * PTB_PI_F, sq = sqrtf(r2 * (1 - r2));
        float sn, cs;
#if defined(__CUDA_ARCH__)
        sincosf(twopi * r1, &sn, &cs);
#else
        sn = sinf(twopi * r1); cs = cosf(twopi * r1);
#endif
        dir = v3(2.f * cs * sq, 2.f * sn * sq, 1.f - 2.f * r2);
    } else {
        const float r1 = pcg32_uniform(e), r2 = pcg32_uniform(e);
        const V3 xl = random_cos(axeOP, r1, r2) * sc.radiusLight + sc.centerLight;
        dir = normalize(xl - P);
        d_light2 = norm2(xl - P);
    }
    float phase;
    const float k = fg.phase_aniso;
    if (fg.phase_type == 1) phase = (float)((double)(1 - k * k) / (4. * PTB_PI_D * (double)(1 + k * dot(dir, -rd))));
    else if (fg.phase_type == 2) { const float dd = dot(dir, rd); phase = (float)(3 / (16 * PTB_PI_D) * (double)(1 + dd * dd)); }
    else phase = (float)(1. / (4. * PTB_PI_D));
    const float ext = uniform_fog ? (float)((double)fg.density * 0.05) : fg.density * expf(-fg.density_decay * (P.y - ground));
    if ((child_state & 0xffffu) == 0) return T;   // a depth-0 contribution is dropped at the top of the loop (Raytracer.cpp:240)
    ch.want = true;
    ch.o.x = P.x; ch.o.y = P.y; ch.o.z = P.z; ch.o.w = d_light2;
    ch.d.x = dir.x; ch.d.y = dir.y; ch.d.z = dir.z; ch.d.w = phase * ext * expf(-int_ext_p) / proba_t;
    ch.w.x = w.x; ch.w.y = w.y; ch.w.z = w.z;
    ch.w.w = u2f((child_state & ~(uint32_t)ST_KIND_MASK) | (1u << ST_KIND_SHIFT) | ST_FOG_PENDING | ST_SHOW_ENV | (d_light2 < 0 ? ST_FOG_UNIFORM : 0u));
    ch.rng = pcg32_fork(e, 1);
    return T;
}

// One iteration of getColor's loop (Raytracer.cpp:227-660) for the contribution in slot `path`, with the fog, ghost and
// background and subsurface (318-406) branches.
template <bool MERL>
PTB_HD void shade_branch_one(const SceneDev& sc, const FrameDev& f, PoolDev& p, int path, BranchOut& out) {
    out.base.cont = false; out.base.shadow = false; out.base.shadow_query = false;
    out.fog.want = false; out.ghost.want = false; out.ghost_pending = false; out.probe = false;
    const F4 wq = p.weight[path];
    uint32_t st = f2u(wq.w);
    const int depth = (int)(st & 0xffffu);
    if (depth == 0) return;                                          // 240; also a ghost child whose shadow ray was blocked
    const F4 hq = p.hit[path];
    const int32_t id = (int32_t)f2u(hq.w);
    const F4 oq = p.ray_o[path], dq = p.ray_d[path];
    const V3 ro = v3(oq.x, oq.y, oq.z), rd = v3(dq.x, dq.y, dq.z);
    V3 w = v3(wq.x, wq.y, wq.z);
    const uint32_t root = p.root[path], pix = p.pixel[path];
    Hit hit; hit.t = hq.x; hit.b1 = hq.y; hit.b2 = hq.z; hit.prim = id;
    Surface s;
    bool have_surface = false;
    if (st & ST_FOG_PENDING) {                                       // tail of fogContribution with the hit of L_ray, 146-187
        const bool inter = id != PTB_HIT_MISS;
        V3 interP = v3(0, 0, 0), interN = fast_normalize(v3(0, 1, 0));
        int interobj = -1;
        if (inter) { surface_from_hit(sc, ro, rd, hit, id, s); have_surface = true; interP = s.P; interN = s.N; interobj = s.object; }
        if (!(st & ST_FOG_UNIFORM) && inter && (double)(hit.t * hit.t) < (double)oq.w * 0.99) return;   // V == 0
        const float pdf_uniform = (float)(1. / (4. * PTB_PI_D));
        const float J = dot(interN, -rd) / norm2(interP - ro);
        float pdf_light = 0.f;
        if (inter && interobj == 0) {
            const V3 axeOP = normalize(ro - sc.centerLight);
            pdf_light = (float)((double)dot(normalize(interP - sc.centerLight), axeOP) / (PTB_PI_D * (double)(sc.radiusLight * sc.radiusLight)) / (double)J);
        }
        const float proba_dir = 0.5f * pdf_uniform + (1 - 0.5f) * pdf_light;
        w = w * (dq.w / proba_dir);
        st &= ~(uint32_t)(ST_FOG_PENDING | ST_FOG_UNIFORM);
        if (norm2(w) < 0.01f * 0.01f) return;                        // 241
    }
    if (depth == f.nb_bounces && sc.bgW > 0 && (id == PTB_HIT_MISS || id == hit_id_analytic(1))) {   // 260-268
        radiance_add(p, root, w * background_at(sc, f, pix));
        return;
    }
    if (id == PTB_HIT_MISS) return;                                  // 654-657 (with fog the reference abandons the whole sample here)
    if (!have_surface) surface_from_hit(sc, ro, rd, hit, id, s);
    const bool show_lights = (st & ST_SHOW_LIGHTS) != 0, show_envmap = (st & ST_SHOW_ENV) != 0;
    const uint32_t hadSS = st & ST_HAD_SS, kind_bits = st & ST_KIND_MASK;
    const bool has_fog = sc.has_fog != 0;
    const float t = hit.t;
    Pcg32 e; e.state = p.rng[path]; e.inc = stream_inc(f, root, st);
    // state of a contribution pushed from here: same stream, same subsurface flag
    const uint32_t st_next = (uint32_t)(depth - 1) | hadSS | kind_bits;
    const uint32_t st_fogchild = (uint32_t)(depth - 1) | hadSS | (show_lights ? ST_SHOW_LIGHTS : 0u);
    if (s.object == 1) {                                             // 275-301
        float att = 1.f;
        if (has_fog) att = fog_sample(sc, ro, rd, sc.centerLight, t, w, st_fogchild, e, out.fog);
        if (show_envmap) radiance_add(p, root, ((w * att) * sc.envmap_intensity) * s.Ke);
        return;
    }
    if (s.object == 0) {                                             // 303-316
        float att = 1.f;
        if (has_fog) att = fog_sample(sc, ro, rd, sc.centerLight, t, w, st_fogchild, e, out.fog);
        const float lp = show_lights ? sc.lightPower : 0.f;
        radiance_add(p, root, (w * att) * lp);
        return;
    }
    const ObjectDev& ob = sc.objects[s.object];
    // -- subsurface scattering (318-406): with probability 0.6 the path re-emerges at a random nearby point of the same mesh.
    //    The probe (Scene::get_random_intersection, reservoir sampling over all hits of a short ray) needs a traversal of its
    //    own: the first visit of the hit only emits the probe (ST_SSS_WAIT), the second one redraws the same numbers and goes on.
    //    The reservoir draws come from a fork of the engine (tag 3): their number depends on the traversal order of the
    //    reference's binary BVH, so no stream alignment with the reference survives this branch anyway.
    const V3 cur_d = rd;                                             // currentRay.direction: what fogContribution keeps seeing
    V3 sd = rd;                                                      // rayDirection
    V3 subsW = v3(1, 1, 1);
    bool sub_interaction = false;
    if (sc.has_sss) {
        const bool is_subsurface = (double)norm2(s.Ksub) > 1E-8;
        const float subsProba = (hadSS || !is_subsurface) ? 0.f : 0.6f;
        const float inv1M = 1.f / (1.f - subsProba);
        subsW = v3(inv1M, inv1M, inv1M);
        if (is_subsurface && pcg32_uniform(e) < subsProba) {
            sub_interaction = true;
            const float invp = 1.f / subsProba;
            subsW = v3(invp, invp, invp);
            const float sigmasub = 1.5f;
            const float diskR = sqrtf(12.46f) * sigmasub;
            const float integ = 1.f - expf(-diskR * diskR / (2.f * sigmasub * sigmasub));
            const float randR = sigmasub * sqrtf(-2.f * logf(1.f - pcg32_uniform(e) * integ));
            const float randangle = pcg32_uniform(e) * 2.f * PTB_PI_F;
            const float g0 = randR * sinf(randangle), g1 = randR * cosf(randangle), g2 = randR;
            const float gaussval = (float)((1. / (double)(sigmasub * sigmasub * 2.f * PTB_PI_F)) * (double)expf(-(g2 * g2) / (2.f * sigmasub * sigmasub)));
            const float pdfgauss = gaussval / integ;
            const V3 N0 = s.N, P0 = s.P;
            const V3 Tg = get_tangent(N0), Tg2 = cross(N0, Tg);
            const V3 above = P0 + g0 * Tg + g1 * Tg2 + N0 * diskR;
            const float r1 = pcg32_uniform(e);
            V3 axis = -N0;
            float tmax, wAxis;
            const float h = sqrtf(diskR * diskR - g2 * g2);
            V3 so = above + (diskR - h) * (-N0);
            if (r1 < 0.5f) { wAxis = 0.5f; tmax = 2.f * h; }
            else {
                wAxis = 0.25f; tmax = 2.f * g2;
                axis = r1 < 0.75f ? Tg : Tg2;
                const float r2 = pcg32_uniform(e);
                if (r2 < 0.5f) so = so - h * N0;
            }
            if (!(st & ST_SSS_WAIT)) {
                out.probe = true;
                out.probe_o.x = so.x; out.probe_o.y = so.y; out.probe_o.z = so.z; out.probe_o.w = tmax;
                out.probe_d.x = axis.x; out.probe_d.y = axis.y; out.probe_d.z = axis.z; out.probe_d.w = u2f((uint32_t)path);
                const uint64_t fs = pcg32_fork(e, 3);
                out.probe_x.x = u2f((uint32_t)fs); out.probe_x.y = u2f((uint32_t)(fs >> 32)); out.probe_x.z = u2f((uint32_t)s.object); out.probe_x.w = 0;
                reinterpret_cast<uint32_t*>(p.weight + path)[3] |= ST_SSS_WAIT;
                return;                                              // nothing of this visit is kept: the second visit redraws from p.rng
            }
            const F4 h2 = p.hit2[path];
            const int32_t prim2 = (int32_t)f2u(h2.w);
            if (prim2 >= 0) {
                Hit hh; hh.t = h2.x; hh.b1 = h2.y; hh.b2 = h2.z; hh.prim = prim2;
                Surface s2;
                surface_from_hit(sc, so, axis, hh, prim2, s2);
                const float chris = (float)exp(-(double)norm2(P0 - s2.P) / (2. * (double)sigmasub * (double)sigmasub));
                const float a0 = dot(s2.N, N0), a1 = dot(s2.N, Tg), a2 = dot(s2.N, Tg2);
                const float sumpdfs = (float)((0.5 * a0) * (0.5 * a0) + (0.25 * a1) * (0.25 * a1) + (0.25 * a2) * (0.25 * a2));
                const float pdfdisk = wAxis * fabsf(dot(axis, s2.N)) / sumpdfs;
                subsW = subsW * (pdfdisk / fmaxf(pdfgauss, 0.05f) * chris);
                sd = normalize(s2.P - P0);
                subsW = subsW * (r1 < 0.5f ? 2.f : 4.f);
                subsW = subsW * (s.Ksub / PTB_PI_F);
                const V3 newP = s2.P + 0.005f * s2.N;
                s = s2;
                s.P = newP;
            }
        }
    }
    const V3 N = s.N, P = s.P;
    V3 no, nd, nw = w;
    uint32_t nstate;
    if (ob.flags & FLAG_MIRROR) {                                    // 413-436
        nd = reflect(sd, N);
        no = P + 0.001f * N;
        if (has_fog) nw = w * fog_sample(sc, ro, cur_d, sc.centerLight, t, w, st_fogchild, e, out.fog);
        nstate = st_next | (show_lights ? ST_SHOW_LIGHTS : 0u) | ST_SHOW_ENV;
    } else if (s.transp) {                                           // 438-489
        float n1 = 1.f, n2 = s.refr_index;
        V3 Nt = N;
        bool entering = true;
        if (dot(sd, N) > 0) { n1 = s.refr_index; n2 = 1; Nt = -N; entering = false; }
        const float c0 = dot(Nt, sd);
        const float radical = 1.f - (n1 / n2) * (n1 / n2) * (1.f - c0 * c0);
        if (radical > 0) {
            const V3 refr = (n1 / n2) * (sd - dot(sd, Nt) * Nt) - Nt * sqrtf(radical);
            const float r0 = (n1 - n2) / (n1 + n2);
            const float R0 = r0 * r0;
            float R;
            if (entering) R = R0 + (1 - R0) * pow5(1.f + dot(sd, N));
            else R = R0 + (1 - R0) * pow5(1.f - dot(refr, N));
            const float u = pcg32_uniform(e);
            if (u < R) { no = P + 0.001f * Nt; nd = reflect(sd, N); }
            else { no = P - 0.001f * Nt; nd = refr; }
        } else {
            no = P + 0.001f * Nt; nd = reflect(sd, N);
        }
        if (has_fog) nw = w * fog_sample(sc, ro, cur_d, sc.centerLight, t, w, st_fogchild, e, out.fog);
        nstate = st_next | (show_lights ? ST_SHOW_LIGHTS : 0u) | ST_SHOW_ENV;
    } else {                                                         // opaque, 490-649
        const bool ghost = (ob.flags & FLAG_GHOST) != 0;
        const LightSample l = light_sample(sc, P, e);
        const V3 wi = l.wi, xl = l.xl;
        const float d2 = l.d2;
        bool shadowed = true, pending = false;                       // pending: only the BVH can tell
        const V3 so = P + 0.01f * wi;
        const float dist = sqrtf(d2) - 0.01f;
        if (!(dot(N, wi) < 0)) {
            out.base.shadow_query = true;
            if (!analytic_occluded(sc, so, wi, dist)) { shadowed = false; pending = sc.has_mesh != 0; }
        }
        V3 direct = v3(0, 0, 0);
        if (!shadowed) {
            if (ghost) {                                             // 522-537: straight through the ghost, same depth, same flags
                const V3 offset = dot(N, sd) > 0 ? N : -N;
                const V3 go = P + sd * 0.001f + offset * 0.001f;
                out.ghost.want = true;
                out.ghost.o.x = go.x; out.ghost.o.y = go.y; out.ghost.o.z = go.z; out.ghost.o.w = 0;
                out.ghost.d.x = sd.x; out.ghost.d.y = sd.y; out.ghost.d.z = sd.z; out.ghost.d.w = 0;
                out.ghost.w.x = w.x; out.ghost.w.y = w.y; out.ghost.w.z = w.z;
                out.ghost.w.w = u2f((uint32_t)depth | hadSS | (show_lights ? ST_SHOW_LIGHTS : 0u) | (show_envmap ? ST_SHOW_ENV : 0u) | (2u << ST_KIND_SHIFT));
                out.ghost.rng = pcg32_fork(e, 2);
                out.ghost_pending = pending;
            } else {
                V3 fr;
                if (sub_interaction) fr = s.Ksub / PTB_PI_F;
                else fr = brdf_eval<MERL>(sc, ob, s, wi, -sd, N);
                const float J = dot(l.dirl, -wi) / d2;
                const float proba = light_proba(sc, l);
                if (proba > 0.f) direct = (subsW * (sc.lightPower * fmaxf(0.f, dot(N, wi)) * J / proba)) * fr;
            }
        }
        float att = 1.f;
        // (with a ghost hit the reference hands fogContribution the straight-through ray, i.e. samples the medium BEHIND the
        //  surface over the distance in front of it, Raytracer.cpp:529, 556; the incoming ray is used here)
        if (has_fog) att = fog_sample(sc, ro, cur_d, xl, t, w, st_fogchild, e, out.fog);
        const V3 c = (w * att) * direct;
        if (!shadowed && !ghost) {
            if (pending) queue_shadow(out.base, so, wi, dist, root, c, 0u);
            else radiance_add(p, root, c);
        } else if (ghost && out.ghost_pending) {                     // the shadow ray decides the ghost child's fate and showenvmap below
            queue_shadow(out.base, so, wi, dist, (uint32_t)path, v3(0, 0, 0), 0x80000000u);   // | child slot, set by the kernel
        }
        // -- continuation (570-632)
        float sx, sy;
        extensible_lattice_2d((uint32_t)(f.k0 + path_sample(f, (int)root)), sx, sy);
        const float r1 = frac_pos(f.rpp[2 * pix] + sx);
        const float r2 = frac_pos(f.rpp[2 * pix + 1] + sy);
        float pdf;
        V3 dir;
        bool diffuse = false;
        if (sub_interaction) {                                       // 598-601
            dir = random_cos(N, r1, r2);
            pdf = dot(N, dir) / PTB_PI_F;
            diffuse = true;
        } else if (MERL && ob.brdf == 1) {
            dir = random_cos(N, r1, r2);
            pdf = (float)((double)dot(N, dir) / PTB_PI_D);
        } else {
            const float u = pcg32_uniform(e);
            dir = phong_sample(s.Ks, s.Ne, -sd, N, r1, r2, u, pdf, diffuse);
        }
        if (dot(dir, N) < 0 || dot(dir, reflect(sd, N)) < 0 || pdf <= 0) return;
        const V3 fi = sub_interaction ? s.Ksub / PTB_PI_F : brdf_eval<MERL>(sc, ob, s, dir, -sd, N);
        nw = ((w * subsW) * fi) * (dot(N, dir) / pdf);
        if (ghost && sc.bgW > 0) nw = nw * (background_at(sc, f, pix) / 196964.699f);   // 614-621
        if (has_fog) nw = att * nw;
        no = P + 0.01f * dir;
        nd = dir;
        // showenvmap of the continuation (626, 629): a ghost passes the dome on only below a blocked shadow ray; when the BVH
        // still has to answer, "blocked" is assumed here and the any-hit kernel clears the bit for an unoccluded ray
        const bool nenv = !ghost || (show_envmap && diffuse && (shadowed || pending));
        nstate = st_next | (nenv ? ST_SHOW_ENV : 0u) | (sub_interaction ? (uint32_t)ST_HAD_SS : 0u);
    }
    p.rng[path] = e.state;
    if (depth - 1 == 0 || norm2(nw) < 0.01f * 0.01f) return;         // 240-241 of the next iteration
    set_next_ray(sc, p, path, no, nd, nw, nstate);
    out.base.cont = true;
}
// Scene::get_random_intersection restricted to one TriMesh (Geometry.cpp:339-472, TriangleMesh.cpp:1321-1424): a uniformly random
// one of the object's intersections with 0 <= t < tmax, by reservoir sampling in (this BVH's) traversal order.
struct ReservoirPick {
    const SceneDev* sc;
    int32_t obj;
    Pcg32 e;
    int count;
    Hit best;
    PTB_HD void operator()(int32_t prim, float t, float b1, float b2) {
        if ((sc->tri_uv[prim].object_has_uv & 0x7fffffff) != obj) return;
        count++;
        const float r1 = pcg32_uniform(e);
        if ((double)r1 < 1. / (double)count) { best.t = t; best.b1 = b1; best.b2 = b2; best.prim = prim; }
    }
};
PTB_HD void probe_one(const SceneDev& sc, PoolDev& p, int entry) {
    const F4 o = p.probe_o[entry], d = p.probe_d[entry], x = p.probe_x[entry];
    ReservoirPick pick;
    pick.sc = &sc; pick.obj = (int32_t)f2u(x.z); pick.count = 0;
    pick.e.state = (uint64_t)f2u(x.x) | ((uint64_t)f2u(x.y) << 32); pick.e.inc = (3ULL << 1) | 1ULL;
    pick.best.t = 0; pick.best.b1 = 0; pick.best.b2 = 0; pick.best.prim = -1;
    if (sc.has_mesh && o.w > 0.f) {
        const AlphaCtx ac = alpha_ctx(sc);
        traverse_all(sc.nodes, sc.tris, &ac, v3(o.x, o.y, o.z), v3(d.x, d.y, d.z), o.w, pick);
    }
    p.hit2[f2u(d.w)] = hit_record(pick.best);
}

// Store a side branch in pool slot `slot` (the kernel / host loop allocated it) and give its ray the analytic hit record.
PTB_HD void store_child(const SceneDev& sc, PoolDev& p, uint32_t slot, const ChildOut& ch, uint32_t root, uint32_t pix) {
    p.ray_o[slot] = ch.o; p.ray_d[slot] = ch.d; p.weight[slot] = ch.w;
    p.rng[slot] = ch.rng; p.pixel[slot] = pix; p.root[slot] = root;
    p.hit[slot] = analytic_hit(sc, v3(ch.o.x, ch.o.y, ch.o.z), v3(ch.d.x, ch.d.y, ch.d.z));
}
// What the any-hit pass does with a finished shadow ray of a branching render: deliver the deferred direct term to the sample
// slot, or settle a ghost hit (Raytracer.cpp:519-537, 626-629): blocked -> the straight-through child dies; clear -> the
// continuation must not show the dome.
PTB_HD void shadow_settle_branch(PoolDev& p, int entry, uint32_t item, bool occluded) {
    const F4 c = p.sh_c[entry];
    const uint32_t tag = f2u(c.w);
    if (tag & 0x80000000u) {
        if (occluded) {
            const uint32_t child = tag & 0x7fffffffu;
            if (child != 0x7fffffffu) reinterpret_cast<uint32_t*>(p.weight + child)[3] &= ~0xffffu;
        } else reinterpret_cast<uint32_t*>(p.weight + item)[3] &= ~(uint32_t)ST_SHOW_ENV;
    } else if (!occluded) radiance_add(p, item, v3(c.x, c.y, c.z));
}

// ---- stage 5: Gaussian splat of a pixel's samples of this pass (Raytracer.cpp:1604-1659) --------------------------
// ADD(addr, value) adds a float4 {r*w, g*w, b*w, w} into the frame accumulator: red.global.add.v4.f32 on the device.
template <class ADD>
PTB_HD void splat_pixel(const FrameDev& f, const PoolDev& p, int ps, F4* accum, ADD add) {
    int i, j;
    if (!slot_to_pixel(f, f.slot0 + ps, i, j)) return;
    int bmin_i, bmax_i, bmin_j, bmax_j;
    const float ratio = filter_ratio(f.filter, i, j, f.W, f.H, bmin_i, bmax_i, bmin_j, bmax_j);
    const float denom1 = (float)((double)ratio / ((double)(f.filter.sigma * f.filter.sigma) * 2. * PTB_PI_D));
    const uint32_t pix = (uint32_t)(i * f.W + j);
    if (f.box_filter) {                                  // Raytracer.cpp:1631-1645: unsplatted sums + first-hit AOVs
        F4 c, a, n;
        c.x = c.y = c.z = c.w = 0; a = c; n = c;
        for (int s = 0; s < f.spp_pass; s++) {
            const F4 L = p.radiance[ps * f.spp_pass + s];
            c.x += L.x; c.y += L.y; c.z += L.z; c.w += 1.f;
            if (f.accum_albedo) {
                const F4 ka = p.aov_kd[ps * f.spp_pass + s], kn = p.aov_n[ps * f.spp_pass + s];
                a.x += ka.x; a.y += ka.y; a.z += ka.z; n.x += kn.x; n.y += kn.y; n.z += kn.z;
            }
        }
        const size_t o = (size_t)(f.H - i - 1) * f.W + j;
        add(accum + o, c);
        if (f.accum_albedo) { add(f.accum_albedo + o, a); add(f.accum_normal + o, n); }
        return;
    }
    if (f.lowres) {                                      // Raytracer.cpp:1508-1510: every sample adds colour/256 to its 16x16 block
        float r = 0, g = 0, b = 0;
        for (int s = 0; s < f.spp_pass; s++) { const F4 L = p.radiance[ps * f.spp_pass + s]; r += L.x * (1.f / 256.f); g += L.y * (1.f / 256.f); b += L.z * (1.f / 256.f); }
        float* q = f.lowres + ((size_t)(f.lowresH - i / 16 - 1) * f.lowresW + j / 16) * 3;
#if defined(__CUDA_ARCH__)
        atomicAdd(q, r); atomicAdd(q + 1, g); atomicAdd(q + 2, b);
#else
        q[0] += r; q[1] += g; q[2] += b;
#endif
    }
    if (f.filter.size == 1) {
        F4 acc[9];
#pragma unroll
        for (int q = 0; q < 9; q++) { acc[q].x = 0; acc[q].y = 0; acc[q].z = 0; acc[q].w = 0; }
        for (int s = 0; s < f.spp_pass; s++) {
            Pcg32 e = pcg32_for_sample(pix, (uint32_t)(f.k0 + s), f.seed);
            const float dx = pcg32_uniform(e) - 0.5f;
            const float dy = pcg32_uniform(e) - 0.5f;
            const F4 L = p.radiance[ps * f.spp_pass + s];
#pragma unroll
            for (int a = 0; a < 3; a++)
#pragma unroll
                for (int b = 0; b < 3; b++) {
                    const float w = filter_weight(f.filter, denom1, i + a - 1, j + b - 1, i, j, dx, dy);
                    F4& c = acc[a * 3 + b];
                    c.x += L.x * w; c.y += L.y * w; c.z += L.z * w; c.w += w;
                }
        }
#pragma unroll
        for (int a = 0; a < 3; a++)
#pragma unroll
            for (int b = 0; b < 3; b++) {
                const int i2 = i + a - 1, j2 = j + b - 1;
                if (i2 < bmin_i || i2 > bmax_i || j2 < bmin_j || j2 > bmax_j) continue;
                add(accum + ((size_t)(f.H - i2 - 1) * f.W + j2), acc[a * 3 + b]);
            }
    } else {
        for (int s = 0; s < f.spp_pass; s++) {
            Pcg32 e = pcg32_for_sample(pix, (uint32_t)(f.k0 + s), f.seed);
            const float dx = pcg32_uniform(e) - 0.5f;
            const float dy = pcg32_uniform(e) - 0.5f;
            const F4 L = p.radiance[ps * f.spp_pass + s];
            for (int i2 = bmin_i; i2 <= bmax_i; i2++)
                for (int j2 = bmin_j; j2 <= bmax_j; j2++) {
                    const float w = filter_weight(f.filter, denom1, i2, j2, i, j, dx, dy);
                    F4 c; c.x = L.x * w; c.y = L.y * w; c.z = L.z * w; c.w = w;
                    add(accum + ((size_t)(f.H - i2 - 1) * f.W + j2), c);
                }
        }
    }
}

// ---- resolve: normalise by the weight and tonemap (Raytracer.cpp:1687-1708) ----------------------------------------
PTB_HD void resolve_pixel(const F4* accum, size_t idx, float gamma, float* imagedouble, float* sample_count, uint8_t* image) {
    const F4 a = accum[idx];
    const float r = div_rn(a.x, a.w), g = div_rn(a.y, a.w), b = div_rn(a.z, a.w);     // (the library is compiled with -prec-div=false)
    if (imagedouble) { imagedouble[idx * 3] = r; imagedouble[idx * 3 + 1] = g; imagedouble[idx * 3 + 2] = b; }
    if (sample_count) sample_count[idx] = a.w;
    if (image) {
        const double ig = (double)div_rn(1.f, gamma);
        const float c[3] = {r, g, b};
        for (int q = 0; q < 3; q++) {
            double v = 255. * pow((double)c[q] / 196964.7, ig);
            v = v > 0. ? v : 0.;     // std::max(0., v): NaN -> 0
            v = v < 255. ? v : 255.;
            image[idx * 3 + q] = (uint8_t)v;
        }
    }
}

// has_denoiser tail of render_image_nopreviz (Raytracer.cpp:1676-1693): colour and albedo means, and the two normal images:
// `normalImage` as the reference computes it (it sums the COLOUR buffers there, 1680-1682, then normalises) and the normalised sum of
// the first-hit shading normals that line was meant to produce.
PTB_HD void resolve_denoiser_pixel(const F4* accum, const F4* albedo, const F4* normal, size_t idx, float* imagedouble, float* sample_count,
                                   float* albedoImage, float* normalImage, float* first_hit_normal) {
    const F4 a = accum[idx], k = albedo[idx], m = normal[idx];
    const float nn = sqrtf(a.x * a.x + a.y * a.y + a.z * a.z), nm = sqrtf(m.x * m.x + m.y * m.y + m.z * m.z);
    if (imagedouble) { imagedouble[idx * 3] = a.x / a.w; imagedouble[idx * 3 + 1] = a.y / a.w; imagedouble[idx * 3 + 2] = a.z / a.w; }
    if (sample_count) sample_count[idx] = a.w;
    if (albedoImage) { albedoImage[idx * 3] = k.x / a.w; albedoImage[idx * 3 + 1] = k.y / a.w; albedoImage[idx * 3 + 2] = k.z / a.w; }
    if (normalImage) { normalImage[idx * 3] = a.x / nn; normalImage[idx * 3 + 1] = a.y / nn; normalImage[idx * 3 + 2] = a.z / nn; }
    if (first_hit_normal) { first_hit_normal[idx * 3] = m.x / nm; first_hit_normal[idx * 3 + 1] = m.y / nm; first_hit_normal[idx * 3 + 2] = m.z / nm; }
}

// tail of the progressive Raytracer::render_image (Raytracer.cpp:1540-1547): imagedouble stays the un-normalised sums, the display
// image divides by max(sample_count, 1)
PTB_HD void resolve_progressive_pixel(const F4* accum, size_t idx, float gamma, float* imagedouble, float* sample_count, uint8_t* image) {
    const F4 a = accum[idx];
    if (imagedouble) { imagedouble[idx * 3] = a.x; imagedouble[idx * 3 + 1] = a.y; imagedouble[idx * 3 + 2] = a.z; }
    if (sample_count) sample_count[idx] = a.w;
    if (image) {
        const double ig = (double)(1 / gamma);
        const float d = fmaxf(a.w, 1.f);
        const float c[3] = {a.x, a.y, a.z};
        for (int q = 0; q < 3; q++) {
            double v = 255. * pow((double)c[q] / 196964.7 / (double)d, ig);
            v = v > 0. ? v : 0.;
            v = v < 255. ? v : 255.;
            image[idx * 3 + q] = (uint8_t)v;
        }
    }
}

// ---- multi-GPU gather: texel `idx` of shard `rank`'s packed tiles, each tile with its apron ((tile + 2 apron)^2 texels, tile-major) ----
// pack: the frame texel if this tile's block sends it (shard_block_sends), else zero; unpack: ADD(addr, value) a non-zero texel into the frame.
template <class ADD>
PTB_HD void shard_texel(F4* rgbw, F4* packed, long long idx, int W, int H, int tile, int apron, int tiles_x, int n_tiles_total, int shift,
                        int rank, int count, int unpack, ADD add) {
    const int side = tile + 2 * apron;
    const long long per = (long long)side * side;
    const int lt = (int)(idx / per);
    const int r = (int)(idx - (long long)lt * per);
    const int tile_id = rank + lt * count;
    if (tile_id >= n_tiles_total) return;
    int ty, tx;
    tile_physical(tile_id, tiles_x, shift, ty, tx);
    const int i = ty * tile - apron + r / side, j = tx * tile - apron + r % side;
    const bool inside = i >= 0 && i < H && j >= 0 && j < W;
    if (!unpack) {
        const int tiles_y = (H + tile - 1) / tile;
        const bool send = shard_block_sends(tile_id, i, j, W, H, tile, apron, tiles_x, tiles_y, rank, count, shift);
        F4 z; z.x = z.y = z.z = z.w = 0;
        packed[idx] = send ? rgbw[(size_t)(H - 1 - i) * W + j] : z;
    } else if (inside) {
        const F4 v = packed[idx];
        if (v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f) add(rgbw + (size_t)(H - 1 - i) * W + j, v);
    }
}

// ---- ray queries of the known-answer tests (PTB_KAT_RAY, PTB_KAT_RAY_WAVEFRONT) ------------------------------------------------------
// input row: o[3], d[3], tmax, any_hit, narrowed to float (the sign of a zero survives the narrowing)
PTB_HD void kat_ray_in(const double* a, V3& o, V3& d, float& tmax) {
    o = v3((float)a[0], (float)a[1], (float)a[2]);
    d = v3((float)a[3], (float)a[4], (float)a[5]);
    tmax = (float)a[6];
}
// output row of a closest hit in extend_ray's convention (id >= 0: stored triangle, PTB_HIT_MISS, or an analytic object): object id,
// original triangle id, t, b1, b2; a miss is -1, -1, -1, 0, 0
PTB_HD void kat_ray_out(const SceneDev& sc, const Hit& h, int32_t id, double* o) {
    o[0] = -1; o[1] = -1; o[2] = -1; o[3] = 0; o[4] = 0;
    if (id >= 0) { o[0] = sc.tri_uv[id].object_has_uv & 0x7fffffff; o[1] = sc.tri_shade[id].orig; o[2] = h.t; o[3] = h.b1; o[4] = h.b2; }
    else if (id != PTB_HIT_MISS) { o[0] = -2 - id; o[2] = h.t; }
}
// the analytic half of a closest-hit query, cut at tmax: the hit record a ray producer writes (analytic_hit) before the BVH sees the ray
PTB_HD Hit kat_ray_analytic(const SceneDev& sc, V3 o, V3 d, float tmax) {
    Hit h; h.b1 = 0; h.b2 = 0;
    analytic_closest(sc, o, d, h.t, h.prim);
    if (!(h.t < tmax)) { h.t = tmax; h.prim = PTB_HIT_MISS; }
    return h;
}
// Closest hit: extend_ray (as k_primary runs it) with the analytic objects' t cut at tmax.  Any hit: the shadow query of shade_one,
// analytic_occluded then the BVH8 up to 0.999 * dist_light (queue_shadow's bound), ghosts passing.
PTB_HD void kat_ray(const SceneDev& sc, const double* a, double* out) {
    V3 o, d;
    float tmax;
    kat_ray_in(a, o, d, tmax);
    const AlphaCtx ac = alpha_ctx(sc);
    Hit h;
    if (a[7] != 0) {
        const bool occ = analytic_occluded(sc, o, d, tmax) ||
                         (sc.has_mesh && traverse<true, false>(sc.nodes, sc.tris, &ac, o, d, (float)((double)tmax * 0.999), h, nullptr));
        out[0] = occ ? 1 : 0; out[1] = out[2] = out[3] = out[4] = 0;
        return;
    }
    h = kat_ray_analytic(sc, o, d, tmax);
    int32_t id = h.prim;
    Hit m;
    if (sc.has_mesh && traverse<false, false>(sc.nodes, sc.tris, &ac, o, d, h.t, m, nullptr)) { h = m; id = m.prim; }
    kat_ray_out(sc, h, id, out);
}

// ---- known-answer tests (ptb_kat): one input row `a` of test `which` -> its output row `o`; false for an unknown test --------------
PTB_HD bool kat_one(int which, const SceneDev& sc, const CameraDev& cam, const FilterDev& filt, int W, int H, const double* a, double* o) {
    switch (which) {
    case PTB_KAT_PCG32: { Pcg32 e = pcg32_seed((uint64_t)a[0], (uint64_t)a[1]); for (int q = 0; q < 4; q++) o[q] = (double)pcg32_next(e); } break;
    case PTB_KAT_LATTICE: { float x, y; extensible_lattice_2d((uint32_t)a[0], x, y); o[0] = x; o[1] = y; } break;
    case PTB_KAT_CAMERA: { V3 ro, rd; camera_ray(cam, (int)a[0], (int)a[1], (float)a[2], (float)a[3], (float)a[4], (float)a[5], ro, rd);
        o[0] = ro.x; o[1] = ro.y; o[2] = ro.z; o[3] = rd.x; o[4] = rd.y; o[5] = rd.z; } break;
    case PTB_KAT_RANDOM_COS: { V3 v = random_cos(v3((float)a[0], (float)a[1], (float)a[2]), (float)a[3], (float)a[4]); o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
    case PTB_KAT_RANDOM_PHONG: { V3 v = random_phong(v3((float)a[0], (float)a[1], (float)a[2]), (float)a[3], (float)a[4], (float)a[5]); o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
    case PTB_KAT_PHONG_EVAL: { V3 v = phong_eval(v3((float)a[0], (float)a[1], (float)a[2]), v3((float)a[3], (float)a[4], (float)a[5]), v3((float)a[6], (float)a[7], (float)a[8]),
                                               v3((float)a[9], (float)a[10], (float)a[11]), v3((float)a[12], (float)a[13], (float)a[14]), v3((float)a[15], (float)a[16], (float)a[17]));
        o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
    case PTB_KAT_MERL_EVAL: { V3 v = merl_eval(sc.merl, v3((float)a[0], (float)a[1], (float)a[2]), v3((float)a[3], (float)a[4], (float)a[5]), v3((float)a[6], (float)a[7], (float)a[8]));
        o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
    case PTB_KAT_FAST_EXP: o[0] = fast_exp(a[0]); break;
    case PTB_KAT_FAST_NORMALIZE: { V3 v = fast_normalize(v3((float)a[0], (float)a[1], (float)a[2])); o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
    case PTB_KAT_RANDOM_PER_PIXEL: { float x, y; random_per_pixel((uint32_t)a[0], x, y); o[0] = x; o[1] = y; } break;
    case PTB_KAT_FILTER_RATIO: { int b0, b1, b2, b3; o[0] = filter_ratio(filt, (int)a[0], (int)a[1], W, H, b0, b1, b2, b3); } break;
    case PTB_KAT_MERL_INDEX: { int f, e; merl_index_both(v3((float)a[0], (float)a[1], (float)a[2]), v3((float)a[3], (float)a[4], (float)a[5]), f, e); o[0] = f; o[1] = e; } break;
    case PTB_KAT_RAY: kat_ray(sc, a, o); break;
    default: return false;
    }
    return true;
}

}  // namespace ptb
