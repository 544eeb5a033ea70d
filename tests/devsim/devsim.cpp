// tests/devsim/devsim.cpp — TEST-ONLY host-compiled stepping of the DEVICE code.
//
// The CUDA kernels in pathtracer_b200/csrc/ptb_engine.cu are thin wrappers over the PTB_HD per-path
// functions of ptb_core.h / ptb_bvh8.h / ptb_scene.h.  This file compiles those same headers with g++ and
// runs the same stage order in plain loops, so the device logic (BVH8 traversal, shading, splat) can be
// debugged against the oracles in a container without a GPU.  It is NOT part of libptb200.so, is never
// loaded by the product, and no parity claim rests on it: the `-m gpu` tests run the real kernels.
#define ORACLE_PREFIX sim_
#include "../../oracle/prefix.h"
#include "../../pathtracer_b200/csrc/ptb_host.h"

#include <chrono>
#include <cstring>

using namespace ptb;

struct ptb_ctx {
    std::string err;
    HostScene host;
    FlatScene flat;
    SceneDev sc;
    bool committed = false;
    bool count = false;
    // progressive session
    bool prog = false; ptb_camera prog_cam; ptb_params prog_p; int prog_iter = 0;
    std::vector<F4> prog_accum; std::vector<float> prog_lowres;
};
struct Extras {          // what the denoiser-input and progressive modes add to a render
    int k_first = 0; bool box = false; F4* albedo = nullptr; F4* normal = nullptr; float* lowres = nullptr;
};
static std::string g_err;

struct PlainAdd {
    void operator()(F4* a, const F4& v) const { a->x += v.x; a->y += v.y; a->z += v.z; a->w += v.w; }
};

extern "C" {
const char* ptb_version(void) { return "ptb200 devsim (host-stepped device code, test only)"; }
const char* ptb_last_error(const ptb_ctx* c) { return c ? c->err.c_str() : g_err.c_str(); }
int ptb_create(int, ptb_ctx** out) { *out = new ptb_ctx(); memset(&(*out)->sc, 0, sizeof(SceneDev)); return PTB_OK; }
void ptb_destroy(ptb_ctx* c) { delete c; }
int ptb_add_sphere(ptb_ctx* c, const float O[3], float R, const ptb_xform* xf, int flags, int* id) { int i = c->host.add_sphere(O, R, xf, flags); if (id) *id = i; return PTB_OK; }
int ptb_add_plane(ptb_ctx* c, const float A[3], const float N[3], const ptb_xform* xf, int flags, int* id) { int i = c->host.add_plane(A, N, xf, flags); if (id) *id = i; return PTB_OK; }
int ptb_add_cylinder(ptb_ctx* c, const float A[3], const float B[3], float R, const ptb_xform* xf, int flags, int* id) { int i = c->host.add_cylinder(A, B, R, xf, flags); if (id) *id = i; return PTB_OK; }
int ptb_add_pointset(ptb_ctx* c, const ptb_pointset* p, const ptb_xform* xf, int flags, int* id) { int i = c->host.add_pointset(p, xf, flags, c->err); if (i < 0) return i; if (id) *id = i; return PTB_OK; }
int ptb_add_yarns(ptb_ctx* c, const ptb_yarns* y, const ptb_xform* xf, int flags, int* id) { int i = c->host.add_yarns(y, xf, flags, c->err); if (i < 0) return i; if (id) *id = i; return PTB_OK; }
int ptb_add_mesh(ptb_ctx* c, const ptb_mesh* m, const ptb_xform* xf, int flags, int* id) { int i = c->host.add_mesh(m, xf, flags, c->err); if (i < 0) return i; if (id) *id = i; return PTB_OK; }
int ptb_set_group_material(ptb_ctx* c, int obj, int group, const ptb_material* m) { return c->host.set_group_material(obj, group, m, c->err); }
int ptb_set_brdf(ptb_ctx* c, int obj, int kind, int merl) { c->host.objects[obj].brdf = kind; c->host.objects[obj].merl = merl; return PTB_OK; }
int ptb_add_merl(ptb_ctx* c, const double* t, int* id) { c->host.merl_tables.emplace_back(t, t + 3 * (size_t)PTB_MERL_N); if (id) *id = (int)c->host.merl_tables.size() - 1; return PTB_OK; }
int ptb_set_envmap(ptb_ctx* c, const uint8_t* rgb, int W, int H) { c->host.envmap.assign(rgb, rgb + (size_t)W * H * 3); c->host.envW = W; c->host.envH = H; return PTB_OK; }
int ptb_set_light(ptb_ctx* c, float a, float b) { c->host.intensite_lumiere = a; c->host.envmap_intensity = b; return PTB_OK; }
int ptb_set_fog(ptb_ctx* c, const ptb_fog* f) { c->host.fog = *f; return PTB_OK; }
int ptb_set_keyframes(ptb_ctx* c, int obj, int kind, const float* frames, const float* values, int n) {
    static const int width[3] = {1, 3, 9};
    key_track_set(c->host.objects[obj].keys[kind], frames, values, n, width[kind]);
    return PTB_OK;
}
int ptb_set_frame(ptb_ctx* c, float frame) { c->host.current_frame = frame; return PTB_OK; }
int ptb_set_background(ptb_ctx* c, const float* rgb, int W, int H) {
    c->host.background.clear(); c->host.bgW = c->host.bgH = 0;
    if (!rgb || W <= 0 || H <= 0) return PTB_OK;
    c->host.background.assign(rgb, rgb + (size_t)W * H * 3); c->host.bgW = W; c->host.bgH = H;
    return PTB_OK;
}
int ptb_commit(ptb_ctx* c) {
    int rc = c->host.flatten(c->flat, c->err);
    if (rc) return rc;
    FlatScene& f = c->flat; SceneDev& sc = c->sc;
    sc.nodes = reinterpret_cast<const F4*>(f.nodes.data()); sc.tris = f.tris.data(); sc.tris_obj = f.tris_obj.empty() ? nullptr : f.tris_obj.data(); sc.tri_uv = f.tri_uv.data(); sc.tri_shade = f.tri_shade.data();
    sc.objects = f.objects.data(); sc.materials = f.materials.data(); sc.texels = f.texels.data(); sc.envmap = f.envmap.data(); sc.merl = f.merl.data();
    scene_header(sc, f);
    if ((rc = scene_modes(sc, c->host, c->err))) return rc;
    sc.background = c->host.background.data();
    c->committed = true;
    return PTB_OK;
}

static int render_into(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, F4* accum_out, ptb_stats* stats, const Extras& x = Extras()) {
    if (!c->committed) return PTB_ERR_STATE;
    auto t0 = std::chrono::steady_clock::now();
    FrameDev f;
    int rc = frame_geometry(cam, p, f, c->err);
    if (rc) return rc;
    const size_t npix = (size_t)p->W * p->H;
    std::vector<float> rpp(2 * npix);
    for (size_t i = 0; i < npix; i++) random_per_pixel((uint32_t)i, rpp[2 * i], rpp[2 * i + 1]);
    f.rpp = rpp.data();
    f.spp_pass = p->nrays; f.k0 = x.k_first; f.slot0 = 0; f.n_pixel_slots = f.n_my_tiles * f.tile * f.tile;
    f.box_filter = x.box ? 1 : 0; f.accum_albedo = x.albedo; f.accum_normal = x.normal;
    f.lowres = x.lowres; f.lowresW = (int)ceilf(p->W / 16.f); f.lowresH = (int)ceilf(p->H / 16.f);
    // one pass holds every sample: the pool the engine would need for it
    const bool branch = is_branching(c->sc);
    const size_t n_roots = (size_t)f.n_pixel_slots * f.spp_pass;
    const size_t P = n_roots * slots_per_sample(c->sc, f.nb_bounces);
    PoolDev pool = {};
    const bool need[] = {true, x.albedo != nullptr, branch, c->sc.has_sss != 0};   // by PoolArray::need
    std::vector<std::vector<F4>> arrays;                                             // zeroed, F4-aligned storage of the pool arrays
    for (const PoolArray& a : pool_arrays(pool))
        if (need[a.need]) { arrays.emplace_back((P * a.bytes + sizeof(F4) - 1) / sizeof(F4)); *a.ptr = arrays.back().data(); }
    std::vector<uint32_t> q0, q1;
    unsigned long long closest = 0, shadow = 0, nodes = 0, tris = 0, samples = 0;
#pragma omp parallel for schedule(static)
    for (long long i = 0; i < (long long)n_roots; i++) raygen_one(c->sc, f, pool, (int)i);
    for (size_t i = 0; i < n_roots; i++) if (pool.pixel[i] != 0xffffffffu) { q0.push_back((uint32_t)i); }
    samples = q0.size();
    if (branch) {   // the engine's branching level loop (run_branch_levels), single-threaded
        size_t next_slot = n_roots;
        for (int b = 0; b < PTB_BRANCH_MAX_LEVELS && !q0.empty() && f.nb_bounces > 0; b++) {
            closest += q0.size();
            q1.clear();
            size_t ns = 0;
            for (size_t i = 0; i < q0.size(); i++) {
                const int path = (int)q0[i];
                TraverseCounters tc{0, 0};
                if (c->sc.has_mesh) extend_one<true>(c->sc, pool, path, &tc);
                nodes += tc.nodes; tris += tc.tris;
            }
            std::vector<uint32_t> visit(q0.begin(), q0.end());
            for (size_t i = 0; i < visit.size(); i++) {     // hits that emit a subsurface probe are answered and revisited at the end of the list
                const int path = (int)visit[i];
                BranchOut out;
                if (getenv("PTB_DBG") && (f2u(pool.weight[path].w) & 0xffffu)) {
                    const int32_t hid = (int32_t)f2u(pool.hit[path].w);
                    fprintf(stderr, "P %u %u %d %.4f\n", pool.pixel[path], f2u(pool.weight[path].w) & 0xffffu, hid >= 0 ? (c->sc.tri_uv[hid].object_has_uv & 0x7fffffff) : (hid == -1 ? -1 : -2 - hid), hid == -1 ? 0.f : pool.hit[path].x);
                }
                shade_branch_one<true>(c->sc, f, pool, path, out);
                uint32_t ghost_slot = 0x7fffffffu;
                for (int k = 0; k < 2; k++) {
                    const ChildOut& ch = k == 0 ? out.fog : out.ghost;
                    if (!ch.want) continue;
                    if (next_slot >= P) { c->err = "devsim: branching pool exhausted"; return PTB_ERR_NOMEM; }
                    store_child(c->sc, pool, (uint32_t)next_slot, ch, pool.root[path], pool.pixel[path]);
                    if (k == 1) ghost_slot = (uint32_t)next_slot;
                    q1.push_back((uint32_t)next_slot++);
                }
                if (out.base.cont) q1.push_back((uint32_t)path);
                if (out.base.shadow) {
                    F4 cc = out.base.sh_c;
                    if (out.ghost_pending) cc.w = u2f(0x80000000u | ghost_slot);
                    pool.sh_o[ns] = out.base.sh_o; pool.sh_d[ns] = out.base.sh_d; pool.sh_c[ns] = cc; ns++;
                }
                if (out.base.shadow_query) shadow++;
                if (out.probe) { pool.probe_o[0] = out.probe_o; pool.probe_d[0] = out.probe_d; pool.probe_x[0] = out.probe_x; probe_one(c->sc, pool, 0); visit.push_back((uint32_t)path); }
            }
            for (size_t i = 0; i < ns; i++) {
                TraverseCounters tc{0, 0};
                const AlphaCtx ac = alpha_ctx(c->sc);
                Hit h;
                const bool occ = traverse<true, true>(c->sc.nodes, c->sc.tris, &ac, v3(pool.sh_o[i].x, pool.sh_o[i].y, pool.sh_o[i].z), v3(pool.sh_d[i].x, pool.sh_d[i].y, pool.sh_d[i].z), pool.sh_o[i].w, h, &tc);
                shadow_settle_branch(pool, (int)i, f2u(pool.sh_d[i].w), occ);
                nodes += tc.nodes; tris += tc.tris;
            }
            q0.swap(q1);
        }
    }
    for (int b = 0; b < f.nb_bounces && !branch; b++) {
        closest += q0.size();
        const long long n = (long long)q0.size();
#pragma omp parallel for schedule(dynamic, 256) reduction(+ : nodes, tris)
        for (long long i = 0; i < n; i++) { TraverseCounters tc{0, 0}; if (c->sc.has_mesh) extend_one<true>(c->sc, pool, (int)q0[i], &tc); nodes += tc.nodes; tris += tc.tris; }
        std::vector<ShadeOut> outs(n);
#pragma omp parallel for schedule(dynamic, 256)
        for (long long i = 0; i < n; i++) { if (x.albedo && b == 0) shade_one<true, true>(c->sc, f, pool, (int)q0[i], outs[i]); else shade_one<true>(c->sc, f, pool, (int)q0[i], outs[i]); }
        q1.clear();
        size_t ns = 0;
        for (long long i = 0; i < n; i++) {
            if (outs[i].cont) q1.push_back(q0[i]);
            if (outs[i].shadow) { pool.sh_o[ns] = outs[i].sh_o; pool.sh_d[ns] = outs[i].sh_d; pool.sh_c[ns] = outs[i].sh_c; ns++; }
            if (outs[i].shadow_query) shadow++;
        }
#pragma omp parallel for schedule(dynamic, 256) reduction(+ : nodes, tris)
        for (long long i = 0; i < (long long)ns; i++) { TraverseCounters tc{0, 0}; shadow_one<true>(c->sc, pool, (int)i, &tc); nodes += tc.nodes; tris += tc.tris; }
        q0.swap(q1);
    }
    for (int ps = 0; ps < f.n_pixel_slots; ps++) splat_pixel(f, pool, ps, accum_out, PlainAdd());
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->samples = samples; stats->rays_closest = closest; stats->rays_shadow = shadow; stats->node_visits = nodes; stats->tri_tests = tris;
        stats->ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    return PTB_OK;
}
int ptb_render(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, float* imagedouble, float* sample_count, uint8_t* image, ptb_stats* stats) {
    const size_t npix = (size_t)p->W * p->H;
    std::vector<F4> accum(npix);
    memset(accum.data(), 0, npix * sizeof(F4));
    int rc = render_into(c, cam, p, accum.data(), stats);
    if (rc) return rc;
    for (size_t i = 0; i < npix; i++) resolve_pixel(accum.data(), i, p->gamma, imagedouble, sample_count, image);
    return PTB_OK;
}
int ptb_render_denoiser_inputs(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, float* imagedouble, float* sample_count, float* albedoImage,
                               float* normalImage, float* first_hit_normal, ptb_stats* stats) {
    const size_t n = (size_t)p->W * p->H;
    std::vector<F4> acc(n), alb(n), nrm(n);
    memset(acc.data(), 0, n * sizeof(F4)); memset(alb.data(), 0, n * sizeof(F4)); memset(nrm.data(), 0, n * sizeof(F4));
    Extras x; x.box = true; x.albedo = alb.data(); x.normal = nrm.data();
    int rc = render_into(c, cam, p, acc.data(), stats, x);
    if (rc) return rc;
    for (size_t i = 0; i < n; i++) resolve_denoiser_pixel(acc.data(), alb.data(), nrm.data(), i, imagedouble, sample_count, albedoImage, normalImage, first_hit_normal);
    return PTB_OK;
}
int ptb_progressive_begin(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p) {
    if (!c->committed) return PTB_ERR_STATE;
    c->prog = true; c->prog_cam = *cam; c->prog_p = *p; c->prog_iter = 0;
    c->prog_accum.assign((size_t)p->W * p->H, F4{0, 0, 0, 0});
    c->prog_lowres.assign((size_t)ceilf(p->W / 16.f) * (size_t)ceilf(p->H / 16.f) * 3, 0.f);
    return PTB_OK;
}
int ptb_progressive_pass(ptb_ctx* c, int n_spp, ptb_stats* stats) {
    if (!c->prog) return PTB_ERR_STATE;
    const int n = std::min(n_spp, c->prog_p.nrays - c->prog_iter);
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n <= 0) return PTB_OK;
    ptb_params p = c->prog_p; p.nrays = n;
    Extras x; x.k_first = c->prog_iter; x.lowres = c->prog_lowres.data();
    int rc = render_into(c, &c->prog_cam, &p, c->prog_accum.data(), stats, x);
    if (rc) return rc;
    c->prog_iter += n;
    return PTB_OK;
}
int ptb_progressive_read(ptb_ctx* c, float* imagedouble, float* sample_count, uint8_t* image, float* imagedouble_lowres, int32_t* current_nb_rays) {
    if (!c->prog) return PTB_ERR_STATE;
    const ptb_params& p = c->prog_p;
    for (size_t i = 0; i < (size_t)p.W * p.H; i++) resolve_progressive_pixel(c->prog_accum.data(), i, p.gamma, imagedouble, sample_count, image);
    if (imagedouble_lowres) memcpy(imagedouble_lowres, c->prog_lowres.data(), c->prog_lowres.size() * sizeof(float));
    if (current_nb_rays) *current_nb_rays = c->prog_iter;
    return PTB_OK;
}
// in the sim the "device" buffers are plain host memory
int ptb_render_accum(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, float* d_rgbw, ptb_stats* stats) { return render_into(c, cam, p, reinterpret_cast<F4*>(d_rgbw), stats); }
int ptb_resolve(ptb_ctx*, const float* d_rgbw, int W, int H, float gamma, float* imagedouble, float* sample_count, uint8_t* image) {
    for (size_t i = 0; i < (size_t)W * H; i++) resolve_pixel(reinterpret_cast<const F4*>(d_rgbw), i, gamma, imagedouble, sample_count, image);
    return PTB_OK;
}
int ptb_shard_pack_size(const ptb_params* p, int rank, int64_t* out) {
    *out = shard_geometry(p, rank).texels() * 4;
    return PTB_OK;
}
static int shard_move(const ptb_params* p, int rank, F4* rgbw, F4* packed, int unpack) {
    const ShardGeometry g = shard_geometry(p, rank);
    for (long long idx = 0; idx < g.texels(); idx++) shard_texel(rgbw, packed, idx, p->W, p->H, g.tile, g.apron, g.tiles_x, g.total, g.shift, rank, g.count, unpack, PlainAdd());
    return PTB_OK;
}
int ptb_shard_pack(ptb_ctx*, const ptb_params* p, int rank, const float* d_rgbw, float* d_packed) { return shard_move(p, rank, (F4*)d_rgbw, (F4*)d_packed, 0); }
int ptb_shard_unpack_add(ptb_ctx*, const ptb_params* p, int rank, const float* d_packed, float* d_rgbw) { return shard_move(p, rank, (F4*)d_rgbw, (F4*)d_packed, 1); }

int ptb_primary_ids(ptb_ctx* c, const ptb_camera* cam, int W, int H, int32_t* obj_id, int32_t* tri_id, float* tout) {
    if (!c->committed) return PTB_ERR_STATE;
    CameraDev cd; camera_setup(cd, cam->position, cam->direction, cam->up, cam->fov, cam->focus_distance, cam->aperture, W, H);
#pragma omp parallel for schedule(dynamic, 64)
    for (int idx = 0; idx < W * H; idx++) {
        const int i = idx / W, j = idx - i * W;
        V3 o, d; camera_ray(cd, i, j, 0, 0, 0, 0, o, d);
        Hit h; int32_t id;
        extend_ray<false>(c->sc, o, d, h, id, nullptr);
        int32_t oid = -1, tid = -1;
        if (id >= 0) { oid = c->sc.tri_uv[id].object_has_uv & 0x7fffffff; tid = c->sc.tri_shade[id].orig; }
        else if (id != PTB_HIT_MISS) oid = -2 - id;
        if (obj_id) obj_id[idx] = oid;
        if (tri_id) tri_id[idx] = tid;
        if (tout) tout[idx] = id == PTB_HIT_MISS ? -1.f : h.t;
    }
    return PTB_OK;
}
int ptb_set_option(ptb_ctx*, int, int64_t) { return PTB_OK; }
int ptb_get_scene_info(const ptb_ctx* c, ptb_scene_info* info) {
    memset(info, 0, sizeof(*info));
    info->n_triangles = c->flat.n_tri_scene; info->n_bvh_nodes = c->flat.bvh.n_nodes; info->bvh_depth = c->flat.bvh.depth;
    info->bytes_nodes = info->n_bvh_nodes * 80; info->bytes_triangles = (int64_t)c->flat.tris.size() / 3 * 48; info->ms_bvh_build = c->flat.ms_bvh;
    info->n_objects = (int)c->host.objects.size();
    return PTB_OK;
}
int ptb_get_kernel_times(const ptb_ctx*, ptb_kernel_times*) { return PTB_ERR_UNSUPPORTED; }
int ptb_kat(ptb_ctx* c, int which, const ptb_camera* cam, int W, int H, const double* in, int n, int is, double* out, int os) {
    CameraDev cd; memset(&cd, 0, sizeof(cd));
    if (cam) camera_setup(cd, cam->position, cam->direction, cam->up, cam->fov, cam->focus_distance, cam->aperture, W, H);
    FilterDev fd; memset(&fd, 0, sizeof(fd));
    if (which == PTB_KAT_FILTER_RATIO) filter_setup(fd, (float)in[2]);
    if (which == PTB_KAT_MERL_EVAL && (!c->committed || c->host.merl_tables.empty())) return PTB_ERR_STATE;
    if (which == PTB_KAT_RAY_WAVEFRONT) which = PTB_KAT_RAY;   // no k_trace / k_exact here: the rows take the plain walk
    if (which == PTB_KAT_RAY && !c->committed) return PTB_ERR_STATE;
    for (int k = 0; k < n; k++)
        if (!kat_one(which, c->sc, cd, fd, W, H, in + (size_t)k * is, out + (size_t)k * os)) return PTB_ERR_UNSUPPORTED;
    return PTB_OK;
}

// test hook: the tile ownership arithmetic of ptb_scene.h (shard_tile_shift, tile_physical, tile_logical) for one frame layout:
// owner[ty * tiles_x + tx] = shard that renders the tile, order[...] = its position in that shard's render order
int devsim_tile_owners(int tiles_x, int tiles_y, int count, int32_t* owner, int32_t* order) {
    const int shift = shard_tile_shift(tiles_x, count), total = tiles_x * tiles_y;
    for (int i = 0; i < total; i++) owner[i] = order[i] = -1;
    for (int r = 0; r < count; r++)
        for (int lt = 0, l = r; l < total; lt++, l += count) {
            int ty, tx;
            tile_physical(l, tiles_x, shift, ty, tx);
            if (ty < 0 || ty >= tiles_y || tx < 0 || tx >= tiles_x) return -1;
            if (owner[ty * tiles_x + tx] != -1) return -2;                       // a tile handed out twice
            if (tile_logical(ty, tx, tiles_x, shift) != l) return -3;            // the two directions disagree
            owner[ty * tiles_x + tx] = r; order[ty * tiles_x + tx] = lt;
        }
    return shift;
}
}
