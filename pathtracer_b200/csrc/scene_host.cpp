// scene_host.cpp — scene ingestion behind the C-ABI: what the reference does between "a reader filled the
// arrays" and "the render loop starts", restated for a flat, upload-once device scene.
//   TriMesh::init        (TriangleMesh.cpp:718-841): axis swap, centre/normalise, rotation centre
//   TriMesh::setup_tangents (601-711): per-vertex tangents (Lengyel), missing normals -> face normals
//   Object::build_matrix (Geometry.h:322-360)
//   Raytracer::prepare_render light constants (Raytracer.cpp:1377-1380)
#include <chrono>
#include <cmath>
#include <cstring>

#include "ptb_host.h"

namespace ptb {

static ptb_xform identity_xform() {
    ptb_xform x;
    memset(&x, 0, sizeof(x));
    x.scale = 1.f;
    x.rotation[0] = x.rotation[4] = x.rotation[8] = 1.f;
    x.rotation_center[0] = x.rotation_center[1] = x.rotation_center[2] = NAN;
    return x;
}

static void take_xform(HostObject& o, const ptb_xform* xf, const float default_center[3]) {
    o.xf = xf ? *xf : identity_xform();
    if (o.xf.rotation_center[0] != o.xf.rotation_center[0])
        for (int k = 0; k < 3; k++) o.xf.rotation_center[k] = default_center[k];
}

int HostScene::add_sphere(const float O[3], float R, const ptb_xform* xf, int flags) {
    HostObject o;
    o.type = OBJ_SPHERE; o.flags = flags;
    for (int k = 0; k < 3; k++) o.a[k] = O[k];
    o.R = R;
    take_xform(o, xf, O);  // Sphere::init: rotation_center = origin (Geometry.h:869)
    objects.push_back(std::move(o));
    return (int)objects.size() - 1;
}

int HostScene::add_plane(const float A[3], const float N[3], const ptb_xform* xf, int flags) {
    HostObject o;
    o.type = OBJ_PLANE; o.flags = flags;
    for (int k = 0; k < 3; k++) { o.a[k] = A[k]; o.n[k] = N[k]; }
    const float zero[3] = {0, 0, 0};
    take_xform(o, xf, zero);
    objects.push_back(std::move(o));
    return (int)objects.size() - 1;
}

// Cylinder(A, B, R) (Geometry.h:734-738): d = (B - A).getNormalized(), len = sqrt((B - A).getNorm2())
int HostScene::add_cylinder(const float A[3], const float B[3], float R, const ptb_xform* xf, int flags) {
    HostObject o;
    o.type = OBJ_CYLINDER; o.flags = flags;
    const V3 ab = v3(B[0], B[1], B[2]) - v3(A[0], A[1], A[2]);
    const V3 d = normalize(ab);
    o.a[0] = A[0]; o.a[1] = A[1]; o.a[2] = A[2];
    o.n[0] = d.x; o.n[1] = d.y; o.n[2] = d.z;
    o.R = R; o.len = sqrtf(norm2(ab));
    const float zero[3] = {0, 0, 0};
    take_xform(o, xf, zero);   // Object(): rotation_center = Vector() = 0
    objects.push_back(std::move(o));
    return (int)objects.size() - 1;
}

int HostScene::add_pointset(const ptb_pointset* p, const ptb_xform* xf, int flags, std::string& err) {
    if (!p || !p->points || !p->normals || !p->radii || p->n <= 0) { err = "add_pointset: points, normals and radii are needed"; return PTB_ERR_INVALID; }
    HostObject o;
    o.type = OBJ_POINTSET; o.flags = flags;
    const size_t n = (size_t)p->n;
    o.pt_pos.assign(p->points, p->points + 3 * n); o.pt_nrm.assign(p->normals, p->normals + 3 * n); o.pt_rad.assign(p->radii, p->radii + n);
    if (p->colors) o.pt_col.assign(p->colors, p->colors + 3 * n);
    for (size_t i = 0; i < n; i++) if (!(o.pt_rad[i] >= 0.f)) { err = "add_pointset: negative or NaN radius"; return PTB_ERR_INVALID; }
    float rc[3] = {0, 0, 0};      // PointSet::init: rotation_center = mean of the points, accumulated in float (PointSet.h:113-121)
    for (size_t i = 0; i < n; i++) for (int k = 0; k < 3; k++) rc[k] += o.pt_pos[3 * i + k];
    for (int k = 0; k < 3; k++) rc[k] = rc[k] / (float)n;
    take_xform(o, xf, rc);
    objects.push_back(std::move(o));
    return (int)objects.size() - 1;
}

// `new Yarns(file)` after its constructor (TriangleMesh.h:268-290): cyls[i] = Cylinder(A, B, R); Object(): rotation_center = 0
int HostScene::add_yarns(const ptb_yarns* y, const ptb_xform* xf, int flags, std::string& err) {
    if (!y || !y->A || !y->B || !y->R || y->n <= 0) { err = "add_yarns: segment end points and radii are needed"; return PTB_ERR_INVALID; }
    if ((int64_t)y->n * PTB_YARN_COVER >= (int64_t)1 << 28) { err = "add_yarns: too many segments"; return PTB_ERR_UNSUPPORTED; }
    HostObject o;
    o.type = OBJ_YARNS; o.flags = flags;
    const size_t n = (size_t)y->n;
    o.yarn_a.assign(y->A, y->A + 3 * n); o.yarn_b.assign(y->B, y->B + 3 * n); o.yarn_r.assign(y->R, y->R + n);
    for (size_t i = 0; i < n; i++) if (!(o.yarn_r[i] >= 0.f)) { err = "add_yarns: negative or NaN radius"; return PTB_ERR_INVALID; }
    const float zero[3] = {0, 0, 0};
    take_xform(o, xf, zero);
    objects.push_back(std::move(o));
    return (int)objects.size() - 1;
}

static inline V3 V(const std::vector<float>& a, int i) { return v3(a[3 * (size_t)i], a[3 * (size_t)i + 1], a[3 * (size_t)i + 2]); }

int HostScene::add_mesh(const ptb_mesh* m, const ptb_xform* xf, int flags, std::string& err) {
    if (!m || !m->vertices || !m->tri || m->n_tri <= 0 || m->n_vertices <= 0) { err = "add_mesh: empty mesh"; return PTB_ERR_INVALID; }
    HostObject o;
    o.type = OBJ_MESH; o.flags = flags;
    const int nv = m->n_vertices, nn = m->normals ? m->n_normals : 0, nuv = m->uvs ? m->n_uvs : 0, nt = m->n_tri;
    o.vertices.assign(m->vertices, m->vertices + 3 * (size_t)nv);
    if (nn) o.normals.assign(m->normals, m->normals + 3 * (size_t)nn);
    if (nuv) o.uvs.assign(m->uvs, m->uvs + 2 * (size_t)nuv);
    o.tri.assign(m->tri, m->tri + 10 * (size_t)nt);
    for (int i = 0; i < nt; i++) {
        const int32_t* t = &o.tri[10 * (size_t)i];
        for (int k = 0; k < 3; k++) {
            if (t[k] < 0 || t[k] >= nv) { err = "add_mesh: vertex index out of range"; return PTB_ERR_INVALID; }
            // -1 is the only "absent" value (TriangleIndices defaults, TriangleMesh.h:55); anything below it would index before the arrays
            if (t[3 + k] >= nuv || t[6 + k] >= nn || t[3 + k] < -1 || t[6 + k] < -1) { err = "add_mesh: uv/normal index out of range"; return PTB_ERR_INVALID; }
        }
    }
    // (x,y,z) -> (-z,y,x) on vertices and normals (TriangleMesh.cpp:742-751)
    for (int i = 0; i < nv; i++) { float* v = &o.vertices[3 * (size_t)i]; std::swap(v[0], v[2]); v[0] = -v[0]; }
    for (int i = 0; i < nn; i++) { float* v = &o.normals[3 * (size_t)i]; std::swap(v[0], v[2]); v[0] = -v[0]; }
    float lo[3] = {1E9f, 1E9f, 1E9f}, hi[3] = {-1E9f, -1E9f, -1E9f};
    for (int i = 0; i < nv; i++)
        for (int k = 0; k < 3; k++) { lo[k] = std::min(lo[k], o.vertices[3 * (size_t)i + k]); hi[k] = std::max(hi[k], o.vertices[3 * (size_t)i + k]); }
    if (m->center) {  // 760-770
        const float s = std::max(hi[0] - lo[0], std::max(hi[1] - lo[1], hi[2] - lo[2]));
        float c[3];
        for (int k = 0; k < 3; k++) c[k] = (lo[k] + hi[k]) * 0.5f;
        for (int i = 0; i < nv; i++)
            for (int k = 0; k < 3; k++) {
                float& v = o.vertices[3 * (size_t)i + k];
                v = (v - c[k]) / s * m->scaling + m->offset[k];
            }
    }
    // bbox over referenced vertices -> default rotation centre (build_bbox 844-860, 831-835)
    float blo[3], bhi[3];
    for (int k = 0; k < 3; k++) blo[k] = bhi[k] = o.vertices[3 * (size_t)o.tri[0] + k];
    for (int i = 0; i < nt; i++)
        for (int c = 0; c < 3; c++)
            for (int k = 0; k < 3; k++) {
                const float v = o.vertices[3 * (size_t)o.tri[10 * (size_t)i + c] + k];
                blo[k] = std::min(blo[k], v); bhi[k] = std::max(bhi[k], v);
            }
    float rc[3];
    for (int k = 0; k < 3; k++) rc[k] = (blo[k] + bhi[k]) * 0.5f;
    take_xform(o, xf, rc);

    // ---- setup_tangents (601-711) ----
    std::vector<V3> tan1(nv, v3(0, 0, 0)), tan2(nv, v3(0, 0, 0));
    for (int i = 0; i < nt; i++) {
        const int32_t* t = &o.tri[10 * (size_t)i];
        if (t[3] == -1 || t[4] == -1 || t[5] == -1) continue;
        const int a = t[0], b = t[1], c = t[2];
        const V3 vA = V(o.vertices, b) - V(o.vertices, a), vB = V(o.vertices, c) - V(o.vertices, a);
        const float sA0 = o.uvs[2 * (size_t)t[4]] - o.uvs[2 * (size_t)t[3]], sA1 = o.uvs[2 * (size_t)t[4] + 1] - o.uvs[2 * (size_t)t[3] + 1];
        const float sB0 = o.uvs[2 * (size_t)t[5]] - o.uvs[2 * (size_t)t[3]], sB1 = o.uvs[2 * (size_t)t[5] + 1] - o.uvs[2 * (size_t)t[3] + 1];
        const float det = (sA0 * sB1 - sB0 * sA1);
        V3 sdir, tdir;
        if (det != 0) { sdir = (sB1 * vA - sA1 * vB) / det; tdir = (sA0 * vB - sB0 * vA) / det; }
        else { sdir = vA * 0.00001f; tdir = vB * 0.00001f; }
        tan1[a] = tan1[a] + sdir; tan1[b] = tan1[b] + sdir; tan1[c] = tan1[c] + sdir;
        tan2[a] = tan2[a] + tdir; tan2[b] = tan2[b] + tdir; tan2[c] = tan2[c] + tdir;
    }
    // missing normal indices -> a fresh face normal (649-668)
    for (int i = 0; i < nt; i++) {
        int32_t* t = &o.tri[10 * (size_t)i];
        if (t[6] != -1 && t[7] != -1 && t[8] != -1) continue;
        const V3 fn = normalize(cross(V(o.vertices, t[1]) - V(o.vertices, t[0]), V(o.vertices, t[2]) - V(o.vertices, t[0])));
        o.normals.push_back(fn.x); o.normals.push_back(fn.y); o.normals.push_back(fn.z);
        const int id = (int)(o.normals.size() / 3) - 1;
        for (int k = 6; k < 9; k++) if (t[k] == -1) t[k] = id;
    }
    std::vector<int> vtn(nv, 0);
    for (int i = 0; i < nt; i++) { const int32_t* t = &o.tri[10 * (size_t)i]; vtn[t[0]] = t[6]; vtn[t[1]] = t[7]; vtn[t[2]] = t[8]; }
    o.tangents.resize(3 * (size_t)nv);
    for (int i = 0; i < nv; i++) {
        const V3 N = normalize(V(o.normals, vtn[i]));
        const V3 tg = normalize(tan1[i] - N * dot(tan1[i], N));
        o.tangents[3 * (size_t)i] = tg.x; o.tangents[3 * (size_t)i + 1] = tg.y; o.tangents[3 * (size_t)i + 2] = tg.z;
    }
    if (nn == 0) o.flags |= FLAG_FLAT;  // no vertex normals in the input: face normals (the reference yields NaN here, App. D#12)
    objects.push_back(std::move(o));
    return (int)objects.size() - 1;
}

static void take_tex(HostTex& d, const ptb_tex& s) {
    for (int k = 0; k < 3; k++) d.mult[k] = s.mult[k];
    if (s.texels && s.W > 0 && s.H > 0) { d.W = s.W; d.H = s.H; d.texels.assign(s.texels, s.texels + (size_t)s.W * s.H * 3); }
    else { d.W = d.H = 0; d.texels.clear(); }
}

int HostScene::set_group_material(int obj, int group, const ptb_material* m, std::string& err) {
    if (obj < 0 || obj >= (int)objects.size() || group < 0 || !m) { err = "set_group_material: bad object/group"; return PTB_ERR_INVALID; }
    HostObject& o = objects[obj];
    if ((int)o.groups.size() <= group) o.groups.resize(group + 1);
    HostMaterial& g = o.groups[group];
    const bool ksub = (m->present & PTB_SLOT_KSUB) && ((m->Ksub.texels && m->Ksub.W > 0) || m->Ksub.mult[0] * m->Ksub.mult[0] + m->Ksub.mult[1] * m->Ksub.mult[1] + m->Ksub.mult[2] * m->Ksub.mult[2] > 1E-8f);
    if (ksub && o.type != OBJ_MESH) {
        // Sphere::reservoir_sampling_intersection returns true without a point or a material (Geometry.h:994-1012): the subsurface
        // branch is only defined on triangle meshes
        err = "set_group_material: subsurface scattering (Ksub != 0) is only defined for triangle meshes";
        return PTB_ERR_UNSUPPORTED;
    }
    g.present |= m->present & ~(uint32_t)PTB_SLOT_KSUB;
    if (ksub) { g.present |= PTB_SLOT_KSUB; take_tex(g.Ksub, m->Ksub); }   // a zero Ksub is the reference default: slot left absent
    if (m->present & PTB_SLOT_KD) take_tex(g.Kd, m->Kd);
    if (m->present & PTB_SLOT_KS) take_tex(g.Ks, m->Ks);
    if (m->present & PTB_SLOT_NE) take_tex(g.Ne, m->Ne);
    if (m->present & PTB_SLOT_TRANSP) take_tex(g.transp, m->transp);
    if (m->present & PTB_SLOT_REFR) take_tex(g.refr, m->refr);
    if (m->present & PTB_SLOT_NORMAL) take_tex(g.normal, m->normal);
    if (m->present & PTB_SLOT_ALPHA) take_tex(g.alpha, m->alpha);
    return PTB_OK;
}

void build_matrix(HostObject& o) {
    const float* m = o.xf.rotation;
    float mt[9];
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) mt[j * 3 + i] = m[i * 3 + j];
    const float s = o.xf.scale;
    const float* tr = o.xf.translation;
    const float* rc = o.xf.rotation_center;
    for (int i = 0; i < 3; i++) {
        float v2[3] = {m[0 * 3 + i], m[1 * 3 + i], m[2 * 3 + i]};
        o.trans[0 * 4 + i] = v2[0] * s; o.trans[1 * 4 + i] = v2[1] * s; o.trans[2 * 4 + i] = v2[2] * s;
        o.rot[0 * 3 + i] = v2[0]; o.rot[1 * 3 + i] = v2[1]; o.rot[2 * 3 + i] = v2[2];
        float w2[3] = {mt[0 * 3 + i], mt[1 * 3 + i], mt[2 * 3 + i]};
        o.inv_trans[0 * 4 + i] = w2[0] / s; o.inv_trans[1 * 4 + i] = w2[1] / s; o.inv_trans[2 * 4 + i] = w2[2] / s;
    }
    auto mul = [](const float* M, const float* b, float* r) {
        for (int i = 0; i < 3; i++) { float v = 0; for (int j = 0; j < 3; j++) v += M[i * 3 + j] * b[j]; r[i] = v; }
    };
    float nrc[3] = {-rc[0], -rc[1], -rc[2]}, v2[3];
    mul(m, nrc, v2);
    for (int k = 0; k < 3; k++) o.trans[k * 4 + 3] = v2[k] * s + rc[k] + tr[k];
    float b[3] = {-rc[0] - tr[0], -rc[1] - tr[1], -rc[2] - tr[2]};
    mul(mt, b, v2);
    for (int k = 0; k < 3; k++) o.inv_trans[k * 4 + 3] = v2[k] / s + rc[k];
}

static TexDev put_tex(const HostTex& t, std::vector<float>& pool) {
    TexDev d;
    for (int k = 0; k < 3; k++) d.mult[k] = t.mult[k];
    d.W = t.W; d.H = t.H; d.offset = 0;
    if (t.W > 0) { d.offset = (uint32_t)pool.size(); pool.insert(pool.end(), t.texels.begin(), t.texels.end()); }
    return d;
}

// ---- alpha-map pre-classification ------------------------------------------------------------------------------
// The reference rejects a hit whose alpha texel reads < 0.5 inside the traversal (TriangleMesh.cpp:1198-1205).  Which texels a
// triangle can ever read is known at commit time: the uv of a hit is a convex combination of the corner uvs, the lookup is
// nearest-texel after wrapping (BRDF.h:270-300).  With a summed-area table of "this texel rejects" per alpha map, a triangle whose
// (conservatively padded) texel rectangle holds no rejecting texel needs no test in the traversal, and one whose rectangle holds
// only rejecting texels can never be hit by anything (closest hit, shadow ray, subsurface probe all apply the same rejection) and
// is left out of the BVH.  Hits and images are exactly those of testing every triangle; only triangles that straddle a border of
// the map's opaque / transparent regions keep PTB_TRI_FLAG_ALPHA.
struct AlphaSat {
    int W = 0, H = 0;
    std::vector<uint32_t> sat;   // (W+1) x (H+1) inclusive prefix counts of rejecting texels
    void build(const HostTex& a) {
        W = a.W; H = a.H;
        sat.assign((size_t)(W + 1) * (H + 1), 0u);
        for (int y = 0; y < H; y++) {
            uint32_t row = 0;
            for (int x = 0; x < W; x++) {
                row += (a.texels[((size_t)y * W + x) * 3] * a.mult[0] < 0.5f) ? 1u : 0u;   // tex_red(...) < 0.5f
                sat[(size_t)(y + 1) * (W + 1) + (x + 1)] = sat[(size_t)y * (W + 1) + (x + 1)] + row;
            }
        }
    }
    uint32_t count(int x0, int y0, int x1, int y1) const {   // inclusive rectangle
        return sat[(size_t)(y1 + 1) * (W + 1) + (x1 + 1)] - sat[(size_t)y0 * (W + 1) + (x1 + 1)] - sat[(size_t)(y1 + 1) * (W + 1) + x0] + sat[(size_t)y0 * (W + 1) + x0];
    }
};
enum { ALPHA_TEST = 0, ALPHA_OPAQUE = 1, ALPHA_INVISIBLE = 2 };
// texel range [lo, hi] that tex_wrap + tex_index can produce for coordinates in [cmin, cmax]; false when the range crosses an
// integer (the wrap is not monotonic there) or is not finite
static bool texel_range(float cmin, float cmax, int n, int& lo, int& hi) {
    if (!(cmin <= cmax) || !std::isfinite(cmin) || !std::isfinite(cmax) || std::fabs(cmin) > 1e6f || std::fabs(cmax) > 1e6f) return false;
    const float pad = 1e-5f * std::max(1.f, std::max(std::fabs(cmin), std::fabs(cmax)));   // barycentric rounding of the interpolated uv
    const float a = cmin - pad, b = cmax + pad;
    if (std::floor(a) != std::floor(b)) return false;
    const float wa = tex_wrap(a), wb = tex_wrap(b);
    if (!(wa <= wb)) return false;
    lo = (int)(wa * (float)(n - 1)) - 1; hi = (int)(wb * (float)(n - 1)) + 1;
    lo = std::max(lo, 0); hi = std::min(hi, n - 1);
    return lo <= hi;
}
static int alpha_class(const AlphaSat& s, const float* uv0, const float* uv1, const float* uv2) {
    int x0, x1, y0, y1;
    if (!texel_range(std::min(uv0[0], std::min(uv1[0], uv2[0])), std::max(uv0[0], std::max(uv1[0], uv2[0])), s.W, x0, x1)) return ALPHA_TEST;
    if (!texel_range(std::min(uv0[1], std::min(uv1[1], uv2[1])), std::max(uv0[1], std::max(uv1[1], uv2[1])), s.H, y0, y1)) return ALPHA_TEST;
    const uint32_t n = s.count(x0, y0, x1, y1), area = (uint32_t)(x1 - x0 + 1) * (uint32_t)(y1 - y0 + 1);
    return n == 0 ? ALPHA_OPAQUE : (n == area ? ALPHA_INVISIBLE : ALPHA_TEST);
}

void HostScene::replace_placements(FlatScene& f) {
    for (size_t i = 0; i < objects.size() && i < f.objects.size(); i++) {
        HostObject& o = objects[i];
        const ptb_xform static_xf = o.xf;
        o.xf = placement_at(o, current_frame);          // Object::build_matrix(current_frame), Geometry.cpp:283
        build_matrix(o);
        o.xf = static_xf;
        ObjectDev& d = f.objects[i];
        memcpy(d.trans, o.trans, sizeof(d.trans)); memcpy(d.inv_trans, o.inv_trans, sizeof(d.inv_trans)); memcpy(d.rot, o.rot, sizeof(d.rot));
    }
    const HostObject& L = objects[0];                   // light constants (Raytracer.cpp:1377-1380)
    const V3 c = xf_point(L.trans, v3(L.a[0], L.a[1], L.a[2]));
    f.centerLight[0] = c.x; f.centerLight[1] = c.y; f.centerLight[2] = c.z;
    const float lum_scale = placement_at(L, current_frame).scale;
    f.radiusLight = lum_scale * L.R;
    f.lightPower = intensite_lumiere / (lum_scale * lum_scale);
    f.envmap_intensity = envmap_intensity;
}

int HostScene::flatten(FlatScene& out, std::string& err) {
    if (objects.size() < 2 || objects[0].type != OBJ_SPHERE || objects[1].type != OBJ_SPHERE) {
        err = "commit: object 0 must be the spherical light and object 1 the environment dome (Raytracer.cpp:1257-1266)";
        return PTB_ERR_STATE;
    }
    out = FlatScene();
    int64_t n_tri = 0;
    for (auto& o : objects) {
        const ptb_xform static_xf = o.xf;
        o.xf = placement_at(o, current_frame);          // Scene::prepare_render -> build_matrix(current_frame) (Geometry.cpp:283)
        build_matrix(o);
        o.xf = static_xf;
        ObjectDev d;
        memset(&d, 0, sizeof(d));
        d.type = o.type; d.flags = o.flags; d.brdf = o.brdf; d.merl = o.merl;
        d.mat_base = (int32_t)out.materials.size(); d.n_groups = (int32_t)o.groups.size();
        for (auto& g : o.groups) {
            MaterialDev m;
            memset(&m, 0, sizeof(m));
            m.present = g.present;
            m.Kd = put_tex(g.Kd, out.texels); m.Ks = put_tex(g.Ks, out.texels); m.Ne = put_tex(g.Ne, out.texels);
            m.transp = put_tex(g.transp, out.texels); m.refr = put_tex(g.refr, out.texels);
            m.normal = put_tex(g.normal, out.texels); m.alpha = put_tex(g.alpha, out.texels);
            if (g.present & SLOT_KSUB) { m.Ksub = put_tex(g.Ksub, out.texels); out.has_sss = true; }
            out.materials.push_back(m);
            d.slot_mask |= (int32_t)g.present;
        }
        memcpy(d.trans, o.trans, sizeof(d.trans)); memcpy(d.inv_trans, o.inv_trans, sizeof(d.inv_trans)); memcpy(d.rot, o.rot, sizeof(d.rot));
        for (int k = 0; k < 3; k++) { d.a[k] = o.a[k]; d.n[k] = o.n[k]; }
        d.R = o.R; d.R2 = o.R * o.R; d.len = o.len;
        out.objects.push_back(d);
        if (o.type == OBJ_MESH) n_tri += (int64_t)o.tri.size() / 10;
        if (o.type == OBJ_POINTSET) n_tri += (int64_t)o.pt_rad.size();
        if (o.type == OBJ_YARNS) n_tri += (int64_t)o.yarn_r.size() * PTB_YARN_COVER;
    }
    if (out.texels.size() >= (size_t)4294967295u) { err = "commit: texture pool exceeds 2^32 floats"; return PTB_ERR_UNSUPPORTED; }
    if (out.materials.empty()) out.materials.emplace_back();  // keep pointers valid
    if (out.texels.empty()) out.texels.push_back(0.f);
    // light constants (Raytracer.cpp:1377-1380)
    {
        const HostObject& L = objects[0];
        const V3 c = xf_point(L.trans, v3(L.a[0], L.a[1], L.a[2]));
        out.centerLight[0] = c.x; out.centerLight[1] = c.y; out.centerLight[2] = c.z;
        const float lum_scale = placement_at(L, current_frame).scale;     // s.lumiere->get_scale(time) (Raytracer.cpp:1378)
        out.radiusLight = lum_scale * L.R;
        out.lightPower = intensite_lumiere / (lum_scale * lum_scale);
        out.envmap_intensity = envmap_intensity;
    }
    out.envmap = envmap; out.envW = envW; out.envH = envH;
    // MERL tables: channel scales folded in, narrowed exactly like `result[c] = r` (BRDF.h:240-243)
    for (auto& t : merl_tables) {
        const double scale[3] = {1.0 / 1500.0, 1.15 / 1500.0, 1.66 / 1500.0};
        const size_t base = out.merl.size();
        out.merl.resize(base + 3 * (size_t)PTB_MERL_N);
        for (int c = 0; c < 3; c++)
            for (size_t i = 0; i < (size_t)PTB_MERL_N; i++) out.merl[base + c * (size_t)PTB_MERL_N + i] = (float)(t[c * (size_t)PTB_MERL_N + i] * scale[c]);
    }
    if (out.merl.empty()) out.merl.push_back(0.f);

    // ---- world-space triangle soup over all meshes ----
    // (k_trace hands a candidate to k_exact as triangle index | flags << 28, ptb_engine.cu)
    if (n_tri >= (int64_t)1 << 28) { err = "commit: more than 2^28 triangles (discs and yarn faces included)"; return PTB_ERR_UNSUPPORTED; }
    out.n_tri_scene = n_tri;
    struct Src { int obj; int tri; uint8_t alpha; };
    std::vector<float> verts9(9 * (size_t)n_tri);
    std::vector<Src> src(n_tri);
    std::vector<float> boxes6;      // only with yarns in the scene: the box a covering triangle enters the BVH with (NaN: its own)
    if (n_tri > 0) {
        int64_t w = 0;
        for (int oi = 0; oi < (int)objects.size(); oi++) {
            const HostObject& o = objects[oi];
            if (o.type == OBJ_POINTSET) {
                // a disc enters the BVH as the triangle circumscribed about it (disc_cover_triangle, ptb_scene.h)
                const float sc_ = placement_at(o, current_frame).scale;
                for (size_t i = 0; i < o.pt_rad.size(); i++) {
                    const V3 cw = xf_point(o.trans, v3(o.pt_pos[3 * i], o.pt_pos[3 * i + 1], o.pt_pos[3 * i + 2]));
                    const V3 nw = xf_rot(o.rot, v3(o.pt_nrm[3 * i], o.pt_nrm[3 * i + 1], o.pt_nrm[3 * i + 2]));
                    V3 p0, p1, p2;
                    disc_cover_triangle(cw, nw, o.pt_rad[i] * fabsf(sc_), p0, p1, p2);
                    float* v = &verts9[9 * (size_t)w];
                    v[0] = p0.x; v[1] = p0.y; v[2] = p0.z; v[3] = p1.x; v[4] = p1.y; v[5] = p1.z; v[6] = p2.x; v[7] = p2.y; v[8] = p2.z;
                    src[w].obj = oi; src[w].tri = (int)i; src[w].alpha = ALPHA_OPAQUE;
                    w++;
                }
                continue;
            }
            if (o.type == OBJ_YARNS) {
                // a yarn segment enters the BVH as the eight triangles of a prism around it (yarn_cover_triangle, ptb_scene.h)
                const float sc_ = placement_at(o, current_frame).scale;
                for (size_t i = 0; i < o.yarn_r.size(); i++) {
                    const V3 aw = xf_point(o.trans, v3(o.yarn_a[3 * i], o.yarn_a[3 * i + 1], o.yarn_a[3 * i + 2]));
                    const V3 bw = xf_point(o.trans, v3(o.yarn_b[3 * i], o.yarn_b[3 * i + 1], o.yarn_b[3 * i + 2]));
                    if (boxes6.empty()) boxes6.assign(6 * (size_t)n_tri, NAN);
                    for (int f = 0; f < PTB_YARN_COVER; f++) {
                        yarn_box(aw, bw, o.yarn_r[i] * fabsf(sc_), &boxes6[6 * (size_t)w], &boxes6[6 * (size_t)w + 3]);
                        V3 p0, p1, p2;
                        yarn_cover_triangle(aw, bw, o.yarn_r[i] * fabsf(sc_), f, p0, p1, p2);
                        float* v = &verts9[9 * (size_t)w];
                        v[0] = p0.x; v[1] = p0.y; v[2] = p0.z; v[3] = p1.x; v[4] = p1.y; v[5] = p1.z; v[6] = p2.x; v[7] = p2.y; v[8] = p2.z;
                        src[w].obj = oi; src[w].tri = (int)(i * PTB_YARN_COVER + f); src[w].alpha = ALPHA_OPAQUE;
                        w++;
                    }
                }
                continue;
            }
            if (o.type != OBJ_MESH) continue;
            const int nt = (int)(o.tri.size() / 10);
            std::vector<AlphaSat> sats(o.groups.size());
            for (int i = 0; i < nt; i++) {
                const int32_t* t = &o.tri[10 * (size_t)i];
                // same condition as the PTB_TRI_FLAG_ALPHA decision below
                uint8_t cls = ALPHA_OPAQUE;
                const int group = t[9];
                const bool uv_all = !o.uvs.empty() && t[3] >= 0 && t[4] >= 0 && t[5] >= 0;
                if (uv_all && group >= 0 && group < (int)o.groups.size() && (o.groups[group].present & SLOT_ALPHA)) {
                    const HostTex& a = o.groups[group].alpha;
                    if (a.W > 0 && a.H > 0) {
                        if (sats[group].W == 0) sats[group].build(a);
                        cls = (uint8_t)alpha_class(sats[group], &o.uvs[2 * (size_t)t[3]], &o.uvs[2 * (size_t)t[4]], &o.uvs[2 * (size_t)t[5]]);
                    } else if (a.mult[0] < 0.5f) cls = ALPHA_INVISIBLE;   // a constant below 0.5 rejects every hit
                    if (cls == ALPHA_OPAQUE && a.W > 0) out.n_tri_alpha_opaque++;
                    else if (cls == ALPHA_INVISIBLE) out.n_tri_alpha_invisible++;
                    else if (cls == ALPHA_TEST) out.n_tri_alpha_tested++;
                }
                if (cls == ALPHA_INVISIBLE) continue;
                for (int c = 0; c < 3; c++) {
                    const V3 p = xf_point(o.trans, V(o.vertices, t[c]));
                    verts9[9 * (size_t)w + 3 * c] = p.x; verts9[9 * (size_t)w + 3 * c + 1] = p.y; verts9[9 * (size_t)w + 3 * c + 2] = p.z;
                }
                src[w].obj = oi; src[w].tri = i; src[w].alpha = cls;
                w++;
            }
        }
        n_tri = w;
    }
    if (n_tri > 0) {
        auto t0 = std::chrono::steady_clock::now();
        std::vector<uint32_t> order;
        build_bvh8(verts9.data(), n_tri, out.nodes, order, out.bvh, boxes6.empty() ? nullptr : boxes6.data());
        out.ms_bvh = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        out.tris.resize(3 * (size_t)n_tri); out.tris_obj.resize(3 * (size_t)n_tri); out.tri_uv.resize(n_tri); out.tri_shade.resize(n_tri);
#pragma omp parallel for schedule(static)
        for (int64_t k = 0; k < n_tri; k++) {
            const uint32_t in = order[k];
            const HostObject& o = objects[src[in].obj];
            if (o.type == OBJ_POINTSET) {
                const size_t i = (size_t)src[in].tri;
                uint32_t fl = PTB_TRI_FLAG_DISC | ((o.flags & FLAG_GHOST) ? PTB_TRI_FLAG_GHOST : 0u);
                F4 q;
                const float* v = &verts9[9 * (size_t)in];                                   // the covering triangle; e1.w = +inf: always left for k_exact
                q.x = v[0]; q.y = v[1]; q.z = v[2]; q.w = u2f(fl); out.tris[3 * (size_t)k] = q;
                q.x = v[3] - v[0]; q.y = v[4] - v[1]; q.z = v[5] - v[2]; q.w = INFINITY; out.tris[3 * (size_t)k + 1] = q;
                q.x = v[6] - v[0]; q.y = v[7] - v[1]; q.z = v[8] - v[2]; q.w = PTB_TRI_T_CUT; out.tris[3 * (size_t)k + 2] = q;
                q.x = o.pt_pos[3 * i]; q.y = o.pt_pos[3 * i + 1]; q.z = o.pt_pos[3 * i + 2]; q.w = u2f((uint32_t)src[in].obj); out.tris_obj[3 * (size_t)k] = q;
                q.x = o.pt_nrm[3 * i]; q.y = o.pt_nrm[3 * i + 1]; q.z = o.pt_nrm[3 * i + 2]; q.w = o.pt_rad[i]; out.tris_obj[3 * (size_t)k + 1] = q;
                q.x = q.y = q.z = q.w = 0; out.tris_obj[3 * (size_t)k + 2] = q;
                TriUV tu; memset(&tu, 0, sizeof(tu));
                tu.group = PTB_GROUP_DISC; tu.object_has_uv = src[in].obj;
                out.tri_uv[k] = tu;
                TriShade ts; memset(&ts, 0, sizeof(ts));
                for (int c = 0; c < 3; c++) {
                    ts.n0[c] = o.pt_nrm[3 * i + c]; ts.n1[c] = o.pt_pos[3 * i + c];
                    ts.t0[c] = o.pt_col.empty() ? 0.5f : o.pt_col[3 * i + c];
                }
                ts.n2[0] = o.pt_rad[i];
                ts.orig = (int32_t)i;
                out.tri_shade[k] = ts;
                continue;
            }
            if (o.type == OBJ_YARNS) {
                const size_t i = (size_t)src[in].tri / PTB_YARN_COVER, face = (size_t)src[in].tri % PTB_YARN_COVER;
                const uint32_t fl = PTB_TRI_FLAG_DISC | ((o.flags & FLAG_GHOST) ? PTB_TRI_FLAG_GHOST : 0u);    // "decided by k_exact", like a disc
                F4 q;
                const float* v = &verts9[9 * (size_t)in];                                   // e1.w = +inf: always left for k_exact; e2.w = 0: no t cut
                q.x = v[0]; q.y = v[1]; q.z = v[2]; q.w = u2f(fl); out.tris[3 * (size_t)k] = q;
                q.x = v[3] - v[0]; q.y = v[4] - v[1]; q.z = v[5] - v[2]; q.w = INFINITY; out.tris[3 * (size_t)k + 1] = q;
                q.x = v[6] - v[0]; q.y = v[7] - v[1]; q.z = v[8] - v[2]; q.w = 0; out.tris[3 * (size_t)k + 2] = q;
                // Cylinder(A, B, R) (Geometry.h:734-738): d = (B - A).getNormalized(), len = sqrt((B - A).getNorm2())
                const V3 A = v3(o.yarn_a[3 * i], o.yarn_a[3 * i + 1], o.yarn_a[3 * i + 2]), B = v3(o.yarn_b[3 * i], o.yarn_b[3 * i + 1], o.yarn_b[3 * i + 2]);
                const V3 d = normalize(B - A);
                q.x = A.x; q.y = A.y; q.z = A.z; q.w = u2f((uint32_t)src[in].obj | ((uint32_t)face << 28)); out.tris_obj[3 * (size_t)k] = q;
                q.x = B.x; q.y = B.y; q.z = B.z; q.w = o.yarn_r[i]; out.tris_obj[3 * (size_t)k + 1] = q;
                q.x = d.x; q.y = d.y; q.z = d.z; q.w = sqrtf(norm2(B - A)); out.tris_obj[3 * (size_t)k + 2] = q;
                TriUV tu; memset(&tu, 0, sizeof(tu));
                tu.group = PTB_GROUP_YARN; tu.object_has_uv = src[in].obj;
                out.tri_uv[k] = tu;
                TriShade ts; memset(&ts, 0, sizeof(ts));
                ts.n0[0] = d.x; ts.n0[1] = d.y; ts.n0[2] = d.z; ts.n1[0] = A.x; ts.n1[1] = A.y; ts.n1[2] = A.z;
                ts.orig = (int32_t)i;
                out.tri_shade[k] = ts;
                continue;
            }
            const int32_t* t = &o.tri[10 * (size_t)src[in].tri];
            const float* v = &verts9[9 * (size_t)in];
            const int group = t[9];
            const bool uv_all = !o.uvs.empty() && t[3] >= 0 && t[4] >= 0 && t[5] >= 0;
            const bool has_uv = !o.uvs.empty() && group >= 0 && t[3] >= 0;      // TriangleMesh.cpp:928
            uint32_t flags = 0;
            if (src[in].alpha == ALPHA_TEST) flags |= PTB_TRI_FLAG_ALPHA;   // a constant >= 0.5 or an all-opaque footprint can never reject
            (void)uv_all;
            if (o.flags & FLAG_GHOST) flags |= PTB_TRI_FLAG_GHOST;
            F4 q;
            q.x = v[0]; q.y = v[1]; q.z = v[2]; q.w = u2f(flags); out.tris[3 * (size_t)k] = q;
            q.x = v[3] - v[0]; q.y = v[4] - v[1]; q.z = v[5] - v[2];
            q.w = (flags & PTB_TRI_FLAG_ALPHA) ? INFINITY : PTB_EDGE_EPS;     // see tri_test_classify (ptb_bvh8.h)
            out.tris[3 * (size_t)k + 1] = q;
            q.x = v[6] - v[0]; q.y = v[7] - v[1]; q.z = v[8] - v[2]; q.w = PTB_TRI_T_CUT; out.tris[3 * (size_t)k + 2] = q;   // see tri_test_classify: the fast test's t cut
            for (int c = 0; c < 3; c++) {      // what Triangle(vertices[vtxi], vertices[vtxj], vertices[vtxk]) is built from (TriangleMesh.cpp:812-815)
                const V3 pv = V(o.vertices, t[c]);
                q.x = pv.x; q.y = pv.y; q.z = pv.z; q.w = c == 0 ? u2f((uint32_t)src[in].obj) : 0.f;
                out.tris_obj[3 * (size_t)k + c] = q;
            }
            TriUV tu;
            memset(&tu, 0, sizeof(tu));
            auto uvc = [&](int idx, float& u, float& vv) {
                if (idx >= 0 && !o.uvs.empty()) { u = o.uvs[2 * (size_t)idx]; vv = o.uvs[2 * (size_t)idx + 1]; } else { u = 0; vv = 0; }
            };
            uvc(t[3], tu.u0, tu.v0); uvc(t[4], tu.u1, tu.v1); uvc(t[5], tu.u2, tu.v2);
            tu.group = group;
            tu.object_has_uv = src[in].obj | (has_uv ? (int32_t)0x80000000 : 0);
            out.tri_uv[k] = tu;
            TriShade ts;
            memset(&ts, 0, sizeof(ts));
            if (o.flags & FLAG_FLAT) {
                const V3 fn = normalize(cross(V(o.vertices, t[1]) - V(o.vertices, t[0]), V(o.vertices, t[2]) - V(o.vertices, t[0])));
                for (int c = 0; c < 3; c++) { float* d = c == 0 ? ts.n0 : (c == 1 ? ts.n1 : ts.n2); d[0] = fn.x; d[1] = fn.y; d[2] = fn.z; }
            } else {
                for (int c = 0; c < 3; c++) {
                    float* d = c == 0 ? ts.n0 : (c == 1 ? ts.n1 : ts.n2);
                    const V3 nn = V(o.normals, t[6 + c]);
                    d[0] = nn.x; d[1] = nn.y; d[2] = nn.z;
                }
            }
            for (int c = 0; c < 3; c++) {
                float* d = c == 0 ? ts.t0 : (c == 1 ? ts.t1 : ts.t2);
                const V3 tg = V(o.tangents, t[c]);
                d[0] = tg.x; d[1] = tg.y; d[2] = tg.z;
            }
            ts.orig = src[in].tri;
            out.tri_shade[k] = ts;
        }
    }
    return PTB_OK;
}

}  // namespace ptb

// ---- material presets: the Phong constants behind the reference's object menu (mainApp.cpp:1499-1597) --------------------------------
// "<name>": the classic OpenGL material table the reference cites (Ne = shininess * 128); "<name>_ngan": the Phong lobes fitted to
// measured BRDFs (Ngan, Durand, Matusik 2005) as the reference lists them.  Each preset does what the menu entry does:
// set_col_texture(Kd), set_col_specular(Ks), set_col_roughness(Ne, Ne, Ne) on one slot index.
namespace {
struct Preset { const char* name; float Kd[3], Ks[3], Ne; };
const Preset kPresets[] = {
    {"gold", {0.75164f, 0.60648f, 0.22648f}, {0.628281f, 0.555802f, 0.366065f}, (float)(0.4 * 128)},
    {"gold_ngan", {0.069f, 0.0323f, 0.00638f}, {0.0738f, 0.0434f, 0.0104f}, 41.9f},
    {"silver", {0.50754f, 0.50754f, 0.50754f}, {0.508273f, 0.508273f, 0.508273f}, (float)(0.4 * 128)},
    {"silver_ngan", {0.0695f, 0.0628f, 0.0446f}, {0.0742f, 0.0615f, 0.0412f}, 75.f},
    {"pearl", {1.f, 0.829f, 0.829f}, {0.296648f, 0.296648f, 0.296648f}, (float)(0.088 * 128)},
    {"pearl_ngan", {0.189f, 0.146f, 0.0861f}, {0.0485f, 0.0346f, 0.0161f}, 27.7f},
    {"white_plastic", {0.55f, 0.55f, 0.55f}, {0.70f, 0.70f, 0.70f}, (float)(0.25 * 128)},
    {"white_plastic_ngan", {0.102f, 0.0887f, 0.0573f}, {0.00699f, 0.00566f, 0.0036f}, 1040.f},
    {"chrome", {0.4f, 0.4f, 0.4f}, {0.774597f, 0.774597f, 0.774597f}, (float)(0.6 * 128)},
    {"chrome_ngan", {0.00817f, 0.0063f, 0.00474f}, {0.0213f, 0.0151f, 0.00766f}, 17900.f},
    {"bronze", {0.714f, 0.4284f, 0.18144f}, {0.393548f, 0.271906f, 0.166721f}, (float)(0.2 * 128)},
    {"bronze_ngan", {0.0864f, 0.0597f, 0.0302f}, {0.015f, 0.00818f, 0.00381f}, 1290.f},
    {"copper", {0.7038f, 0.27048f, 0.0828f}, {0.256777f, 0.137622f, 0.086014f}, (float)(0.1 * 128)},
    {"copper_ngan", {0.0749f, 0.0414f, 0.027f}, {0.0756f, 0.0437f, 0.0202f}, 33200.f},
};
const int kNumPresets = (int)(sizeof(kPresets) / sizeof(kPresets[0]));
}  // namespace

extern "C" {
int ptb_preset_count(void) { return kNumPresets; }
int ptb_preset_get(int index, const char** name, float Kd[3], float Ks[3], float* Ne) {
    if (index < 0 || index >= kNumPresets) return PTB_ERR_INVALID;
    const Preset& p = kPresets[index];
    if (name) *name = p.name;
    for (int k = 0; k < 3; k++) { if (Kd) Kd[k] = p.Kd[k]; if (Ks) Ks[k] = p.Ks[k]; }
    if (Ne) *Ne = p.Ne;
    return PTB_OK;
}
int ptb_preset_find(const char* name) {
    if (!name) return -1;
    for (int i = 0; i < kNumPresets; i++) if (!strcmp(kPresets[i].name, name)) return i;
    return -1;
}
}
