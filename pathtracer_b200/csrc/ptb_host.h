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

// ---- frame and pass geometry (host only: the engine and the test-only devsim share it) -------------------------------------------
#define PTB_MAX_BOUNCES 64
#define PTB_MAX_PIPES 4
#define PTB_BRANCH_MAX_LEVELS 512   // a branching render's contribution tree is cut off below this many levels

// Camera, filter and the shard's tiles of a render; the per-pass fields and the buffers (rpp, AOV sums, preview) are the caller's.
inline int frame_geometry(const ptb_camera* cam, const ptb_params* p, FrameDev& f, std::string& err) {
    if (!cam || !p || p->W <= 0 || p->H <= 0 || p->nrays <= 0 || p->nb_bounces < 0 || p->nb_bounces > PTB_MAX_BOUNCES || !(p->sigma_filter > 0)) {
        err = "render: invalid parameters"; return PTB_ERR_INVALID;
    }
    if ((int)ceilf(p->sigma_filter * 2) > PTB_MAX_FILTER) { err = "render: sigma_filter too large (filter_size > 4)"; return PTB_ERR_UNSUPPORTED; }
    if ((int64_t)p->W * p->H >= ((int64_t)1 << 31)) { err = "render: frame too large"; return PTB_ERR_UNSUPPORTED; }
    memset(&f, 0, sizeof(f));
    camera_setup(f.cam, cam->position, cam->direction, cam->up, cam->fov, cam->focus_distance, cam->aperture, p->W, p->H);
    filter_setup(f.filter, p->sigma_filter);
    f.W = p->W; f.H = p->H; f.nb_bounces = p->nb_bounces; f.seed = p->seed;
    f.tile = p->tile_size > 0 ? p->tile_size : ptb_default_tile(p->shard_count);
    // a splat reaches ceil(2 sigma) pixels into the neighbouring tiles and the gather looks at the 3x3 tile neighbourhood only
    if (f.tile < (int)ceilf(p->sigma_filter * 2) || f.tile > 4096) { err = "render: tile_size must lie in [ceil(2*sigma_filter), 4096]"; return PTB_ERR_INVALID; }
    f.tiles_x = (p->W + f.tile - 1) / f.tile; f.tiles_y = (p->H + f.tile - 1) / f.tile;
    f.shard_count = p->shard_count > 0 ? p->shard_count : 1;
    f.shard_rank = p->shard_rank;
    if (f.shard_rank < 0 || f.shard_rank >= f.shard_count) { err = "render: shard_rank out of range"; return PTB_ERR_INVALID; }
    f.tile_shift = shard_tile_shift(f.tiles_x, f.shard_count);
    const int total_tiles = f.tiles_x * f.tiles_y;
    f.n_my_tiles = total_tiles > f.shard_rank ? (total_tiles - f.shard_rank + f.shard_count - 1) / f.shard_count : 0;
    return PTB_OK;
}

// in-image pixels of the shard's pixel slots [s0, s0 + ns) (edge tiles are partial)
inline unsigned long long tile_range_pixels(const FrameDev& f, int64_t s0, int64_t ns) {
    const int tp = f.tile * f.tile;
    unsigned long long n = 0;
    for (int64_t lt = s0 / tp; lt * tp < s0 + ns; lt++) {
        int ty, tx;
        tile_physical(f.shard_rank + (int)lt * f.shard_count, f.tiles_x, f.tile_shift, ty, tx);
        n += (unsigned long long)std::min(f.tile, f.H - ty * f.tile) * std::min(f.tile, f.W - tx * f.tile);
    }
    return n;
}

// The tiles of shard `rank` in the multi-GPU gather: each travels with an apron of ceil(2 sigma) pixels, (tile + 2 apron)^2 texels
struct ShardGeometry {
    int tile, apron, tiles_x, total, count, shift, mine;   // total: tiles of the frame; mine: tiles of this shard
    int64_t texels() const { return (int64_t)mine * (tile + 2 * apron) * (tile + 2 * apron); }
};
inline ShardGeometry shard_geometry(const ptb_params* p, int rank) {
    ShardGeometry g;
    g.tile = p->tile_size > 0 ? p->tile_size : ptb_default_tile(p->shard_count);
    g.apron = (int)ceilf(p->sigma_filter * 2);
    g.tiles_x = (p->W + g.tile - 1) / g.tile;
    g.total = g.tiles_x * ((p->H + g.tile - 1) / g.tile);
    g.count = p->shard_count > 0 ? p->shard_count : 1;
    g.shift = shard_tile_shift(g.tiles_x, g.count);
    g.mine = g.total > rank ? (g.total - rank + g.count - 1) / g.count : 0;
    return g;
}

// Branching renders (fog, ghost objects, a background photograph, subsurface scattering) walk each sample's contribution tree.
inline bool is_branching(const SceneDev& sc) { return sc.has_fog || sc.has_ghost || sc.bgW > 0 || sc.has_sss; }
// Pool slots one sample may hold at once.  A branching render keeps every live contribution of a sample in the pool: the
// continuation reuses its slot, each side branch takes a new one.  A fogged path forks once per iteration (at most 2^depth - 1
// forks per sample), a ghost hit once; a background photograph or a subsurface material forks nothing.
inline int slots_per_sample(const SceneDev& sc, int nb_bounces) {
    if (!is_branching(sc)) return 1;
    return sc.has_fog ? (1 << std::min(nb_bounces, 6)) : (sc.has_ghost ? 8 : 1);
}

// How a render of `pixel_slots` pixel slots x `nrays` samples is cut into passes.
struct PassPlan {
    bool branch;
    int n_pipes;           // pipelines the passes go round-robin to (branching renders: one)
    int spp_pass;          // samples per pixel of a pass
    int64_t slots_pass;    // pixel slots of a pass
    int64_t stride;        // paths of a pass = the pool slice of one pipeline
    int64_t pool_paths;    // paths the pool must hold
};
inline PassPlan plan_passes(const SceneDev& sc, int nb_bounces, int tile, int64_t pixel_slots, int nrays, int64_t pool_paths, int n_pipes) {
    PassPlan pl;
    pl.branch = is_branching(sc);
    const int fan = slots_per_sample(sc, nb_bounces);
    const int64_t pool_cap_slots = std::max<int64_t>(pool_paths, 1024);
    int64_t pool = std::max<int64_t>(pool_cap_slots / fan, 1024);
    pl.n_pipes = pl.branch ? 1 : std::max(1, std::min(n_pipes, PTB_MAX_PIPES));
    if (pl.n_pipes > 1 && pixel_slots * nrays < pool * pl.n_pipes)   // a frame smaller than the pools is still split so that every pipeline gets a pass
        pool = std::max<int64_t>((pixel_slots * nrays + pl.n_pipes - 1) / pl.n_pipes, (int64_t)1 << 18);
    if (pixel_slots * nrays <= pool) { pl.spp_pass = nrays; pl.slots_pass = pixel_slots; }
    else if (pixel_slots <= pool) { pl.spp_pass = (int)std::max<int64_t>(1, pool / pixel_slots); pl.slots_pass = pixel_slots; }
    else { pl.spp_pass = 1; pl.slots_pass = (pool / (tile * tile)) * (tile * tile); if (pl.slots_pass <= 0) pl.slots_pass = tile * tile; }
    pl.stride = pl.slots_pass * pl.spp_pass;
    pl.pool_paths = pl.branch ? std::max<int64_t>(pl.stride * fan, pool_cap_slots) : pl.stride * pl.n_pipes;
    return pl;
}

// ---- the path pool's arrays ------------------------------------------------------------------------------------------------------
// Every array of PoolDev with its bytes per path and the renders that need it; allocation, release and slicing all walk this list.
// `queue` (or null) adds the two bounce queues, which live outside PoolDev, in their place of the allocation order.
enum { POOL_ALWAYS, POOL_AOV, POOL_BRANCH, POOL_SSS };
struct PoolArray { void** ptr; size_t bytes; int need; };
inline std::vector<PoolArray> pool_arrays(PoolDev& p, uint32_t** queue = nullptr) {
    std::vector<PoolArray> a = {{(void**)&p.ray_o, sizeof(F4), POOL_ALWAYS}, {(void**)&p.ray_d, sizeof(F4), POOL_ALWAYS},
                                {(void**)&p.weight, sizeof(F4), POOL_ALWAYS}, {(void**)&p.radiance, sizeof(F4), POOL_ALWAYS},
                                {(void**)&p.hit, sizeof(F4), POOL_ALWAYS}, {(void**)&p.rng, sizeof(uint64_t), POOL_ALWAYS},
                                {(void**)&p.pixel, sizeof(uint32_t), POOL_ALWAYS}, {(void**)&p.sh_o, sizeof(F4), POOL_ALWAYS},
                                {(void**)&p.sh_d, sizeof(F4), POOL_ALWAYS}, {(void**)&p.sh_c, sizeof(F4), POOL_ALWAYS}};
    if (queue) { a.push_back({(void**)&queue[0], sizeof(uint32_t), POOL_ALWAYS}); a.push_back({(void**)&queue[1], sizeof(uint32_t), POOL_ALWAYS}); }
    a.insert(a.end(), {{(void**)&p.defer_prims, PTB_DEFER_K * sizeof(uint32_t), POOL_ALWAYS}, {(void**)&p.defer_rays, sizeof(U2), POOL_ALWAYS},
                       {(void**)&p.aov_n, sizeof(F4), POOL_AOV}, {(void**)&p.aov_kd, sizeof(F4), POOL_AOV},
                       {(void**)&p.root, sizeof(uint32_t), POOL_BRANCH},
                       {(void**)&p.probe_o, sizeof(F4), POOL_SSS}, {(void**)&p.probe_d, sizeof(F4), POOL_SSS},
                       {(void**)&p.probe_x, sizeof(F4), POOL_SSS}, {(void**)&p.hit2, sizeof(F4), POOL_SSS}});
    return a;
}

}  // namespace ptb
