// ptb_host.h — host-side scene model behind the C-ABI (no CUDA types here).
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/ptb200.h"
#include "ptb_keyframes.h"
#include "ptb_scene.h"

namespace ptb {

struct Bvh8Stats {
    int64_t n_nodes = 0, n_binary_nodes = 0, leaves = 0;
    int depth = 0;
    int e_floor = 0;                       // no node cell finer than 2^e_floor = 2^-25 of the root's cells (the builder's and the refit's floor)
    std::vector<uint32_t> level_start;     // nodes are emitted breadth first: level l is [level_start[l], level_start[l + 1]) (refit walks them bottom-up)
};
// verts9: 9 floats per triangle (world space).  leaf_order[k] = input index of the k-th stored triangle.  boxes6 (or null): lo[3], hi[3]
// per triangle, used instead of the triangle's own bounds where lo[0] <= hi[0] (NaN = no override).
void build_bvh8(const float* verts9, int64_t n_tri, std::vector<Node8>& nodes, std::vector<uint32_t>& leaf_order, Bvh8Stats& stats, const float* boxes6 = nullptr);

struct HostTex {
    float mult[3] = {1, 1, 1};
    int W = 0, H = 0;
    std::vector<float> texels;
};
struct HostMaterial {
    uint32_t present = 0;
    HostTex Kd, Ks, Ne, transp, refr, normal, alpha, Ksub;
};
struct HostObject {
    int type = OBJ_SPHERE, flags = 0, brdf = 0, merl = 0;
    ptb_xform xf;
    float a[3] = {0, 0, 0}, n[3] = {0, 1, 0}, R = 0, len = 0;
    std::vector<HostMaterial> groups;      // index = group
    // mesh data AFTER TriMesh::init processing (object space)
    std::vector<float> vertices, normals, uvs, tangents;   // tangents: per vertex
    std::vector<int32_t> tri;              // n x 10
    std::vector<float> pt_pos, pt_nrm, pt_rad, pt_col;     // point set (PointSet::vertices / normals / radius / colors)
    std::vector<float> yarn_a, yarn_b, yarn_r;             // yarns (Yarns::cyls[i]->A / B / R)
    float trans[12], inv_trans[12], rot[9];
    KeyTrack keys[3];                      // PTB_KEY_SCALE / _TRANSLATION / _ROTATION (Geometry.h:318-320)
};

// The object's placement at `frame`: keyed tracks replace the static fields (Object::build_matrix(frame), Geometry.h:322-328)
inline ptb_xform placement_at(const HostObject& o, float frame) {
    ptb_xform x = o.xf;
    key_eval(o.keys[PTB_KEY_SCALE], frame, &x.scale);
    key_eval(o.keys[PTB_KEY_TRANSLATION], frame, x.translation);
    key_eval(o.keys[PTB_KEY_ROTATION], frame, x.rotation);
    return x;
}

// Everything ptb_commit produces, ready to upload.
struct FlatScene {
    std::vector<Node8> nodes;
    std::vector<F4> tris;                  // 3 per triangle, leaf order
    std::vector<F4> tris_obj;              // 3 per triangle, leaf order: object-space corners, .w of the first = object id
    std::vector<TriUV> tri_uv;
    std::vector<TriShade> tri_shade;
    std::vector<ObjectDev> objects;
    std::vector<MaterialDev> materials;
    std::vector<float> texels;
    std::vector<uint8_t> envmap;
    std::vector<float> merl;
    int envW = 0, envH = 0;
    float envmap_intensity = 1, lightPower = 0, radiusLight = 0, centerLight[3] = {0, 0, 0};
    Bvh8Stats bvh;
    double ms_bvh = 0;
    bool has_sss = false;                  // some mesh group carries a subsurface albedo
    int64_t n_tri_scene = 0;               // triangles handed over (tris holds those that can ever be hit, see alpha classification)
    int64_t n_tri_alpha_opaque = 0, n_tri_alpha_invisible = 0, n_tri_alpha_tested = 0;
};

struct HostScene {
    std::vector<HostObject> objects;
    std::vector<std::vector<double>> merl_tables;
    std::vector<uint8_t> envmap;
    int envW = 0, envH = 0;
    float intensite_lumiere = 0, envmap_intensity = 1;
    ptb_fog fog = {0, 0, 0, 0, 0, 0, 0};            // Scene::fog_* (Geometry.h:1371-1377)
    std::vector<float> background;                  // Scene::background (Geometry.h:1365), bgW*bgH*3
    int bgW = 0, bgH = 0;
    float current_frame = 0;                        // Scene::current_frame

    int add_sphere(const float O[3], float R, const ptb_xform* xf, int flags);
    int add_plane(const float A[3], const float N[3], const ptb_xform* xf, int flags);
    int add_cylinder(const float A[3], const float B[3], float R, const ptb_xform* xf, int flags);
    int add_mesh(const ptb_mesh* m, const ptb_xform* xf, int flags, std::string& err);
    int add_pointset(const ptb_pointset* p, const ptb_xform* xf, int flags, std::string& err);
    int add_yarns(const ptb_yarns* y, const ptb_xform* xf, int flags, std::string& err);
    int set_group_material(int obj, int group, const ptb_material* m, std::string& err);
    int flatten(FlatScene& out, std::string& err);
    // Scene::prepare_render at another frame for an already flattened scene: every object's matrices (build_matrix(current_frame)) and
    // the light constants are recomputed into `f.objects` / `f`; geometry, materials and the BVH topology are untouched (refit).
    void replace_placements(FlatScene& f);
    bool has_keyframes() const { for (const HostObject& o : objects) for (int k = 0; k < 3; k++) if (!o.keys[k].frames.empty()) return true; return false; }
};

void build_matrix(HostObject& o);          // Object::build_matrix (Geometry.h:322-360)

// Fill the by-value part of SceneDev from a flattened scene (pointers are the caller's business).
inline void scene_header(SceneDev& sc, FlatScene& f) {
    sc.n_objects = (int32_t)f.objects.size();
    sc.has_mesh = f.nodes.empty() ? 0 : 1;
    sc.envW = f.envW; sc.envH = f.envH; sc.has_envmap = (f.envW > 0 && f.envH > 0) ? 1 : 0;
    sc.envmap_intensity = f.envmap_intensity; sc.lightPower = f.lightPower; sc.radiusLight = f.radiusLight;
    sc.centerLight = v3(f.centerLight[0], f.centerLight[1], f.centerLight[2]);
    sc.n_inline = 0; sc.n_extra = 0;
    sc.has_ghost = 0; sc.has_exotic = 0;
    sc.has_sss = f.has_sss ? 1 : 0;
    for (size_t i = 0; i < f.objects.size(); i++) {
        ObjectDev& o = f.objects[i];
        if (o.flags & FLAG_GHOST) sc.has_ghost = 1;
        if (o.type == OBJ_POINTSET || o.type == OBJ_CYLINDER || o.type == OBJ_YARNS) sc.has_exotic = 1;   // kernels with the Cylinder / PointSet / Yarns code
        if (o.type == OBJ_MESH || o.type == OBJ_POINTSET || o.type == OBJ_YARNS) continue;
        if (sc.n_inline < PTB_INLINE_ANALYTIC) {
            AnalyticDev& a = sc.analytic[sc.n_inline++];
            a.type = o.type | ((o.flags & FLAG_GHOST) ? PTB_ANALYTIC_GHOST : 0); a.id = (int32_t)i; a.R2 = o.R2;
            for (int k = 0; k < 12; k++) a.inv_trans[k] = o.inv_trans[k];
            // the light, the dome and the ground plane are normally placed without rotation or scaling: mark an exact identity linear
            // part so that the ray producers skip the 3x3 products (m = I gives bit-identical results: 1*x + 0*y + 0*z == x)
            const float* m = a.inv_trans;
            if (m[0] == 1.f && m[1] == 0.f && m[2] == 0.f && m[4] == 0.f && m[5] == 1.f && m[6] == 0.f && m[8] == 0.f && m[9] == 0.f && m[10] == 1.f)
                a.type |= PTB_ANALYTIC_LINEAR_ID;
            for (int k = 0; k < 3; k++) { a.a[k] = o.a[k]; a.n[k] = o.n[k]; }
            a.len = o.len;
        } else { o.flags |= FLAG_NOT_INLINE; sc.n_extra++; }
    }
}

// Medium / compositing modes of the scene (by-value part; the background pointer is the caller's business).
inline int scene_modes(SceneDev& sc, const HostScene& h, std::string& err) {
    sc.has_fog = h.fog.density > 1E-8f ? 1 : 0;                          // Raytracer.cpp:206
    sc.fog.density = h.fog.density; sc.fog.absorption = h.fog.absorption; sc.fog.density_decay = h.fog.density_decay;
    sc.fog.absorption_decay = h.fog.absorption_decay; sc.fog.phase_aniso = h.fog.phase_aniso;
    sc.fog.type = h.fog.type; sc.fog.phase_type = h.fog.phase_type; sc.fog.ground = 0;
    if (sc.has_fog) {
        if (h.objects.size() < 3) { err = "fog needs object 2 (its translation is the ground level, Raytracer.cpp:54)"; return PTB_ERR_STATE; }
        sc.fog.ground = placement_at(h.objects[2], h.current_frame).translation[1];   // get_translation(r.time)[1], r.time = current_frame
    }
    sc.bgW = h.bgW; sc.bgH = h.bgH; sc.background = nullptr;
    return PTB_OK;
}

}  // namespace ptb
