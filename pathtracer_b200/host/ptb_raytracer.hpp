// ptb_raytracer.hpp — C++ host side above the C-ABI, shaped like the reference's own classes so that code written
// against `Raytracer` / `Scene` / `Sphere` / `Plane` / `TriMesh` / `Camera` (Raytracer.h:25-121, Geometry.h:849-1400,
// TriangleMesh.h:113-255, Vector.h:720-840) ports by changing an include.  The objects only hold description; all
// rendering happens in libptb200.so (CUDA).  Errors surface as ptb::Error (the reference reports nothing).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <array>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/ptb200.h"
#include "../../include/ptb_sceneio.h"

namespace ptbhost {

struct Error : std::runtime_error { using std::runtime_error::runtime_error; };

struct Vector {
    float v[3];
    Vector(float x = 0, float y = 0, float z = 0) { v[0] = x; v[1] = y; v[2] = z; }
    float& operator[](int i) { return v[i]; }
    float operator[](int i) const { return v[i]; }
};

// Vector.h:720-840 (non-lenticular)
struct Camera {
    Vector position{0, 0, 50}, direction{0, 0, -1}, up{0, 1, 0};
    float fov = 35.f * (float)M_PI / 180.f, focus_distance = 50.f, aperture = 0.1f;
    Camera() = default;
    Camera(const Vector& p, const Vector& d, const Vector& u) : position(p), direction(d), up(u) {}
    void rotate(float angle_x, float angle_y, float time) {   // Camera::rotate, Vector.h:738-765
        const float ax = time * angle_x, ay = time * angle_y;
        auto rot = [&](Vector& d) {
            Vector t(d[0], std::cos(ay) * d[1] - std::sin(ay) * d[2], std::sin(ay) * d[1] + std::cos(ay) * d[2]);
            d = Vector(std::cos(ax) * t[0] - std::sin(ax) * t[2], t[1], std::sin(ax) * t[0] + std::cos(ax) * t[2]);
        };
        rot(direction); rot(up);
    }
};

// BRDF.h:252-426
struct Texture {
    Vector multiplier{1, 1, 1};
    int W = 0, H = 0;
    std::vector<float> values;   // W*H*3 post-load
    Texture() = default;
    explicit Texture(const Vector& m) : multiplier(m) {}
    explicit Texture(float m) : multiplier(m, m, m) {}
};

struct Material {                // one slot index of Object::textures / specularmap / ... (Geometry.h:672)
    uint32_t present = 0;
    Texture Kd, Ks, Ne, transp, refr, normal, alpha;
    Material& set(uint32_t slot, const Texture& t) {
        present |= slot;
        switch (slot) {
        case PTB_SLOT_KD: Kd = t; break; case PTB_SLOT_KS: Ks = t; break; case PTB_SLOT_NE: Ne = t; break;
        case PTB_SLOT_TRANSP: transp = t; break; case PTB_SLOT_REFR: refr = t; break;
        case PTB_SLOT_NORMAL: normal = t; break; case PTB_SLOT_ALPHA: alpha = t; break;
        default: throw Error("unknown slot");
        }
        return *this;
    }
};

enum ObjectType { OT_TRIMESH, OT_SPHERE, OT_PLANE, OT_POINTSET, OT_CYLINDER, OT_YARNS };   // Geometry.h:29

struct Object {                  // Geometry.h:240-672
    ObjectType type;
    bool miroir = false, flip_normals = false, interp_normals = true, ghost = false;
    float scale = 1.f;
    float mat_rotation[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    Vector rotation_center{NAN, NAN, NAN};   // NaN: the object's own default
    Vector max_translation;
    int brdf_kind = PTB_BRDF_PHONG;
    std::shared_ptr<std::vector<double>> merl;   // IsoMERLBRDF::data
    std::vector<Material> materials;             // index = group
    std::map<float, float> scale_keyframes;                  // Geometry.h:318-320
    std::map<float, Vector> translation_keyframes;
    std::map<float, std::array<float, 9>> rotation_keyframes;
    void add_keyframe(int frame) {                           // Geometry.h:313-317
        std::array<float, 9> m; std::memcpy(m.data(), mat_rotation, sizeof(mat_rotation));
        rotation_keyframes[(float)frame] = m; translation_keyframes[(float)frame] = max_translation; scale_keyframes[(float)frame] = scale;
    }
    // Object::set_col_texture / set_col_specular / set_col_roughness (Geometry.cpp:165-177, 229-234): only the multiplier of an
    // EXISTING slot changes (its texels stay); an index past the end is ignored like the reference does
    void set_col_texture(const Vector& col, int idx) { if (idx >= 0 && idx < (int)materials.size() && (materials[idx].present & PTB_SLOT_KD)) materials[idx].Kd.multiplier = col; }
    void set_col_specular(const Vector& col, int idx) { if (idx >= 0 && idx < (int)materials.size() && (materials[idx].present & PTB_SLOT_KS)) materials[idx].Ks.multiplier = col; }
    void set_col_roughness(const Vector& col, int idx) { if (idx >= 0 && idx < (int)materials.size() && (materials[idx].present & PTB_SLOT_NE)) materials[idx].Ne.multiplier = col; }
    // a material preset of the reference's object menu (mainApp.cpp:1499-1597): "gold", "gold_ngan", ..., "copper_ngan" (ptb_preset_get)
    void set_preset(const char* name, int idx = 0) {
        const int k = ptb_preset_find(name);
        float kd[3], ks[3], ne;
        if (k < 0 || ptb_preset_get(k, nullptr, kd, ks, &ne) != PTB_OK) throw Error(std::string("unknown material preset: ") + name);
        set_col_texture(Vector(kd[0], kd[1], kd[2]), idx); set_col_specular(Vector(ks[0], ks[1], ks[2]), idx); set_col_roughness(Vector(ne, ne, ne), idx);
    }
    explicit Object(ObjectType t) : type(t) {}
    virtual ~Object() = default;
};
struct Sphere : Object {
    Vector O; float R;
    std::vector<uint8_t> envtex; int envW = 0, envH = 0;   // Sphere::load_envmap (object 1 only)
    Sphere(const Vector& origin, float rayon, bool mirror = false, bool normal_swapped = false) : Object(OT_SPHERE), O(origin), R(rayon) {
        miroir = mirror; flip_normals = normal_swapped;
    }
};
struct Plane : Object {
    Vector A, vecN;
    Plane(const Vector& a, const Vector& n, bool mirror = false) : Object(OT_PLANE), A(a), vecN(n) { miroir = mirror; }
};
struct PointSet : Object {       // PointSet.h as it stands after init: one disc per point
    std::vector<float> vertices, normals, colors;   // x3 (colors may stay empty: 0.5 grey)
    std::vector<float> radius;
    bool display_edges = false;
    PointSet() : Object(OT_POINTSET) {}
};
struct Cylinder : Object {       // Geometry.h:731-846
    Vector A, B; float R;
    Cylinder(const Vector& a, const Vector& b, float r) : Object(OT_CYLINDER), A(a), B(b), R(r) {}
};
struct Yarns : Object {          // TriangleMesh.h:265-312: `cyls` as three flat arrays (segment i = Cylinder(A[i], B[i], R[i]))
    std::vector<float> A, B, R;  // x3, x3, x1
    Yarns() : Object(OT_YARNS) { rotation_center = Vector(0, 0, 0); }
    explicit Yarns(const char* filename) : Object(OT_YARNS) {      // Yarns::Yarns(filename): points times 50, radius 0.1
        rotation_center = Vector(0, 0, 0);
        float *a = nullptr, *b = nullptr, *r = nullptr; int32_t n = 0;
        if (ptb_yarnfile_read(filename, &a, &b, &r, &n) != PTB_OK) throw Error(std::string("Yarns: ") + ptb_sceneio_last_error());
        A.assign(a, a + 3 * (size_t)n); B.assign(b, b + 3 * (size_t)n); R.assign(r, r + n);
        ptb_yarnfile_free(a); ptb_yarnfile_free(b); ptb_yarnfile_free(r);
    }
};
struct TriMesh : Object {        // arrays as a reader fills them (TriangleMesh.cpp:240-569), before init's processing
    std::vector<float> vertices, normals, uvs;   // x3, x3, x2
    std::vector<int32_t> indices;                // x10: vtx ijk, uv ijk, normal ijk, group
    float scaling = 1.f; Vector offset; bool center = true;
    TriMesh() : Object(OT_TRIMESH) {}
};

struct Scene {                   // Geometry.h:1238-1400
    std::vector<std::shared_ptr<Object>> objects;
    float intensite_lumiere = 0.f, envmap_intensity = 1.f;
    float fog_density = 0.f, fog_absorption = 0.f, fog_density_decay = 0.f, fog_absorption_decay = 0.f, phase_aniso = 0.f;   // Geometry.h:1371-1377
    int fog_type = 0, fog_phase_type = 0;
    int current_frame = 0;                                                                                                 // Geometry.h:1372
    std::vector<float> background; int backgroundW = 0, backgroundH = 0;                                                   // Geometry.h:1365-1366
    int addObject(std::shared_ptr<Object> o) { objects.push_back(std::move(o)); return (int)objects.size() - 1; }
};

class Raytracer {                // Raytracer.h:25-121
public:
    int W = 1000, H = 800, nrays = 100, nb_bounces = 3;
    Camera cam;
    float sigma_filter = 0.5f, gamma = 2.2f;
    uint32_t seed = 0;
    Scene s;
    std::vector<unsigned char> image;     // W*H*3
    std::vector<float> imagedouble;       // W*H*3 linear
    std::vector<float> sample_count;      // W*H
    ptb_stats stats{};

    explicit Raytracer(int device = 0) : device_(device) {}
    // several GPUs of this process under the same single call: the frame is tile-sharded and gathered over NCCL inside the library
    // (ptb_group_*, include/ptb200.h); `devices` = CUDA device ids
    explicit Raytracer(const std::vector<int>& devices) : device_(devices.empty() ? 0 : devices[0]), devices_(devices) {}
    ~Raytracer() { release(); }
    Raytracer(const Raytracer&) = delete;

    void loadScene() {               // Raytracer.cpp:1238-1274
        W = 1000; H = 800; nrays = 100; nb_bounces = 3;
        cam = Camera(Vector(0, 0, 50), Vector(0, 0, -1), Vector(0, 1, 0));
        cam.fov = (float)(35 * M_PI / 180); cam.focus_distance = 50; cam.aperture = 0.1f; sigma_filter = 0.5f;
        s = Scene();
        auto slum = std::make_shared<Sphere>(Vector(10, 23, 15), 10.f);
        auto s2 = std::make_shared<Sphere>(Vector(0, 0, 0), 1000000.f, false, true);
        auto plane = std::make_shared<Plane>(Vector(0, 0, 0), Vector(0, 1, 0));
        plane->max_translation = Vector(0, -27.3f, 0);
        s.addObject(slum); s.addObject(s2); s.addObject(plane);
        s.intensite_lumiere = (float)(1000000000 * 4. * M_PI / (4. * M_PI * slum->R * slum->R * M_PI));
        s.envmap_intensity = 1;
        cam.rotate(0, (float)(-22 * M_PI / 180), 1);
    }

    // Raytracer::load_scene (Raytracer.cpp:1149-1236): the native reader parses the .scn, reads the meshes / textures /
    // environment map it names and feeds the device context; this object receives the camera and frame parameters.
    // The scene is committed on return (`s.objects` stays empty: the description lives in the context).
    void load_scene(const char* filename, const char* replacedNames = nullptr) {
        acquire();
        ptb_camera c; ptb_params p;
        if (ptb_load_scene(ctx_, filename, replacedNames, &c, &p) != PTB_OK) throw Error(std::string("load_scene: ") + ptb_sceneio_last_error());
        W = p.W; H = p.H; nrays = p.nrays; nb_bounces = p.nb_bounces; sigma_filter = p.sigma_filter; gamma = p.gamma;
        cam = Camera(Vector(c.position[0], c.position[1], c.position[2]), Vector(c.direction[0], c.direction[1], c.direction[2]), Vector(c.up[0], c.up[1], c.up[2]));
        cam.fov = c.fov; cam.focus_distance = c.focus_distance; cam.aperture = c.aperture;
        ck(ptb_set_frame(ctx_, (float)s.current_frame));
        commit_device();
    }
    // One frame of an animation (mainApp.cpp:874-877): key-framed objects are placed at `frame`.  Nothing is rebuilt: the library
    // re-poses the scene on the device before the next render (matrices, world-space triangles, BVH8 refit).
    void set_frame(int frame) {
        s.current_frame = frame;
        if (!ctx_) { commit(); return; }
        ck(ptb_set_frame(ctx_, (float)frame));
    }

    // hands the scene to the device: TriMesh::init + build_bvh + Scene::prepare_render equivalents
    void commit() {
        acquire();
        std::vector<std::pair<const std::vector<double>*, int>> merl_ids;
        for (auto& op : s.objects) {
            Object& o = *op;
            ptb_xform xf;
            xf.scale = o.scale; std::memcpy(xf.rotation, o.mat_rotation, sizeof(xf.rotation));
            for (int k = 0; k < 3; k++) { xf.rotation_center[k] = o.rotation_center[k]; xf.translation[k] = o.max_translation[k]; }
            const int flags = (o.miroir ? PTB_OBJ_MIRROR : 0) | (o.flip_normals ? PTB_OBJ_FLIP_NORMALS : 0) | (o.interp_normals ? 0 : PTB_OBJ_FLAT_NORMALS) | (o.ghost ? PTB_OBJ_GHOST : 0);
            int id = -1;
            if (o.type == OT_SPHERE) { auto& sp = static_cast<Sphere&>(o); ck(ptb_add_sphere(ctx_, sp.O.v, sp.R, &xf, flags, &id)); }
            else if (o.type == OT_PLANE) { auto& pl = static_cast<Plane&>(o); ck(ptb_add_plane(ctx_, pl.A.v, pl.vecN.v, &xf, flags, &id)); }
            else if (o.type == OT_POINTSET) {
                auto& ps = static_cast<PointSet&>(o);
                ptb_pointset d;
                d.points = ps.vertices.data(); d.normals = ps.normals.data(); d.radii = ps.radius.data(); d.colors = ps.colors.empty() ? nullptr : ps.colors.data();
                d.n = (int32_t)ps.radius.size();
                ck(ptb_add_pointset(ctx_, &d, &xf, flags | (ps.display_edges ? PTB_OBJ_DISPLAY_EDGES : 0), &id));
            }
            else if (o.type == OT_CYLINDER) { auto& cy = static_cast<Cylinder&>(o); ck(ptb_add_cylinder(ctx_, cy.A.v, cy.B.v, cy.R, &xf, flags, &id)); }
            else if (o.type == OT_YARNS) {
                auto& ys = static_cast<Yarns&>(o);
                ptb_yarns d;
                d.A = ys.A.data(); d.B = ys.B.data(); d.R = ys.R.data(); d.n = (int32_t)ys.R.size();
                ck(ptb_add_yarns(ctx_, &d, &xf, flags, &id));
            }
            else {
                auto& g = static_cast<TriMesh&>(o);
                ptb_mesh m;
                m.vertices = g.vertices.data(); m.n_vertices = (int)g.vertices.size() / 3;
                m.normals = g.normals.data(); m.n_normals = (int)g.normals.size() / 3;
                m.uvs = g.uvs.data(); m.n_uvs = (int)g.uvs.size() / 2;
                m.tri = g.indices.data(); m.n_tri = (int)g.indices.size() / 10;
                m.scaling = g.scaling; m.center = g.center ? 1 : 0;
                for (int k = 0; k < 3; k++) m.offset[k] = g.offset[k];
                ck(ptb_add_mesh(ctx_, &m, &xf, flags, &id));
            }
            {
                std::vector<float> fr, val;
                for (auto& k : o.scale_keyframes) { fr.push_back(k.first); val.push_back(k.second); }
                if (!fr.empty()) ck(ptb_set_keyframes(ctx_, id, PTB_KEY_SCALE, fr.data(), val.data(), (int)fr.size()));
                fr.clear(); val.clear();
                for (auto& k : o.translation_keyframes) { fr.push_back(k.first); for (int q = 0; q < 3; q++) val.push_back(k.second[q]); }
                if (!fr.empty()) ck(ptb_set_keyframes(ctx_, id, PTB_KEY_TRANSLATION, fr.data(), val.data(), (int)fr.size()));
                fr.clear(); val.clear();
                for (auto& k : o.rotation_keyframes) { fr.push_back(k.first); for (int q = 0; q < 9; q++) val.push_back(k.second[q]); }
                if (!fr.empty()) ck(ptb_set_keyframes(ctx_, id, PTB_KEY_ROTATION, fr.data(), val.data(), (int)fr.size()));
            }
            for (size_t gi = 0; gi < o.materials.size(); gi++) {
                const Material& mm = o.materials[gi];
                ptb_material pm;
                std::memset(&pm, 0, sizeof(pm));
                pm.present = mm.present;
                auto tex = [](const Texture& t) { ptb_tex r; r.texels = t.W > 0 ? t.values.data() : nullptr; r.W = t.W; r.H = t.H; for (int k = 0; k < 3; k++) r.mult[k] = t.multiplier[k]; return r; };
                pm.Kd = tex(mm.Kd); pm.Ks = tex(mm.Ks); pm.Ne = tex(mm.Ne); pm.transp = tex(mm.transp); pm.refr = tex(mm.refr); pm.normal = tex(mm.normal); pm.alpha = tex(mm.alpha);
                ck(ptb_set_group_material(ctx_, id, (int)gi, &pm));
            }
            if (o.brdf_kind == PTB_BRDF_MERL && o.merl) {
                int mid = -1;
                for (auto& pr : merl_ids) if (pr.first == o.merl.get()) mid = pr.second;
                if (mid < 0) { ck(ptb_add_merl(ctx_, o.merl->data(), &mid)); merl_ids.push_back({o.merl.get(), mid}); }
                ck(ptb_set_brdf(ctx_, id, PTB_BRDF_MERL, mid));
            }
        }
        if (s.objects.size() > 1 && s.objects[1]->type == OT_SPHERE) {
            auto& dome = static_cast<Sphere&>(*s.objects[1]);
            if (dome.envW > 0) ck(ptb_set_envmap(ctx_, dome.envtex.data(), dome.envW, dome.envH));
        }
        ck(ptb_set_light(ctx_, s.intensite_lumiere, s.envmap_intensity));
        const ptb_fog fog = {s.fog_density, s.fog_absorption, s.fog_density_decay, s.fog_absorption_decay, s.fog_type, s.fog_phase_type, s.phase_aniso};
        ck(ptb_set_fog(ctx_, &fog));
        ck(ptb_set_background(ctx_, s.backgroundW > 0 ? s.background.data() : nullptr, s.backgroundW, s.backgroundH));
        ck(ptb_set_frame(ctx_, (float)s.current_frame));
        commit_device();
    }

    // Raytracer::render_image_nopreviz (Raytracer.cpp:1565-1798): fills imagedouble / sample_count / image
    void render_image_nopreviz() {
        if (!ctx_) commit();
        ptb_camera c; ptb_params p;
        fill(c, p);
        const bool grown = image.size() != (size_t)W * H * 3;
        if (grown) {     // the output vectors are members that live across frames (Raytracer.h:90-105): page-lock them once per size
            unpin();
            image.resize((size_t)W * H * 3); imagedouble.resize((size_t)W * H * 3); sample_count.resize((size_t)W * H);
            ptb_pin_host_buffer(ctx_, imagedouble.data(), (int64_t)(imagedouble.size() * sizeof(float)));
            ptb_pin_host_buffer(ctx_, sample_count.data(), (int64_t)(sample_count.size() * sizeof(float)));
            ptb_pin_host_buffer(ctx_, image.data(), (int64_t)image.size());
            pinned_ = true;
        }
        if (group_) gck(ptb_group_render(group_, &c, &p, imagedouble.data(), sample_count.data(), image.data(), &stats));
        else ck(ptb_render(ctx_, &c, &p, imagedouble.data(), sample_count.data(), image.data(), &stats));
    }

    // Raytracer::render_image (Raytracer.cpp:1424-1563): progressive; `stopped` may be set from `on_pass` (the GUI sets it from
    // another thread).  imagedouble holds UN-normalised sums afterwards, like the reference's.  With several devices every pass
    // runs on all of them (ptb_group_progressive_*).
    bool stopped = true;
    int current_nb_rays = 0;
    std::vector<float> imagedouble_lowres;   // ceil(W/16) x ceil(H/16) x 3
    template <class F>
    void render_image(F on_pass, int passes_per_call = 1) {
        if (!ctx_) commit();
        ptb_camera c; ptb_params p;
        fill(c, p);
        if (group_) gck(ptb_group_progressive_begin(group_, &c, &p));
        else ck(ptb_progressive_begin(ctx_, &c, &p));
        stopped = false; current_nb_rays = 0;
        while (current_nb_rays < nrays && !stopped) {
            if (group_) gck(ptb_group_progressive_pass(group_, passes_per_call, &stats));
            else ck(ptb_progressive_pass(ctx_, passes_per_call, &stats));
            current_nb_rays = std::min(nrays, current_nb_rays + passes_per_call);
            on_pass(*this);
        }
        const int Wlr = (W + 15) / 16, Hlr = (H + 15) / 16;
        image.resize((size_t)W * H * 3); imagedouble.resize((size_t)W * H * 3); sample_count.resize((size_t)W * H); imagedouble_lowres.resize((size_t)Wlr * Hlr * 3);
        int32_t n = 0;
        if (group_) gck(ptb_group_progressive_read(group_, imagedouble.data(), sample_count.data(), image.data(), imagedouble_lowres.data(), &n));
        else ck(ptb_progressive_read(ctx_, imagedouble.data(), sample_count.data(), image.data(), imagedouble_lowres.data(), &n));
        current_nb_rays = n; stopped = true;
    }
    void render_image() { render_image([](Raytracer&) {}); }

    // render_image_nopreviz with has_denoiser (Raytracer.cpp:1631-1645, 1676-1693) up to the hand-over to the denoiser (on every
    // device of a group, like render_image_nopreviz)
    std::vector<float> albedoImage, normalImage, first_hit_normal;
    void render_denoiser_inputs() {
        if (!ctx_) commit();
        ptb_camera c; ptb_params p;
        fill(c, p);
        const size_t n = (size_t)W * H;
        imagedouble.resize(n * 3); sample_count.resize(n); albedoImage.resize(n * 3); normalImage.resize(n * 3); first_hit_normal.resize(n * 3);
        if (group_) gck(ptb_group_render_denoiser_inputs(group_, &c, &p, imagedouble.data(), sample_count.data(), albedoImage.data(), normalImage.data(), first_hit_normal.data(), &stats));
        else ck(ptb_render_denoiser_inputs(ctx_, &c, &p, imagedouble.data(), sample_count.data(), albedoImage.data(), normalImage.data(), first_hit_normal.data(), &stats));
    }

    ptb_ctx* ctx() { return ctx_; }

private:
    void fill(ptb_camera& c, ptb_params& p) const {
        for (int k = 0; k < 3; k++) { c.position[k] = cam.position[k]; c.direction[k] = cam.direction[k]; c.up[k] = cam.up[k]; }
        c.fov = cam.fov; c.focus_distance = cam.focus_distance; c.aperture = cam.aperture;
        p.W = W; p.H = H; p.nrays = nrays; p.nb_bounces = nb_bounces; p.sigma_filter = sigma_filter; p.gamma = gamma; p.seed = seed;
        p.shard_rank = 0; p.shard_count = 1; p.tile_size = 0;
    }
    void ck(int rc) { if (rc != PTB_OK) throw Error(std::string("ptb error ") + std::to_string(rc) + ": " + ptb_last_error(ctx_)); }
    void gck(int rc) { if (rc != PTB_OK) throw Error(std::string("group render: ") + ptb_group_last_error(group_)); }
    void unpin() {
        if (pinned_ && ctx_) { ptb_unpin_host_buffer(ctx_, imagedouble.data()); ptb_unpin_host_buffer(ctx_, sample_count.data()); ptb_unpin_host_buffer(ctx_, image.data()); }
        pinned_ = false;
    }
    void release() {
        unpin();
        image.clear();      // the next render pins afresh
        if (group_) { ptb_group_destroy(group_); group_ = nullptr; ctx_ = nullptr; }
        if (ctx_) { ptb_destroy(ctx_); ctx_ = nullptr; }
    }
    void acquire() {        // a fresh context (one GPU) or group (several): the scene is handed to ctx_ either way
        release();
        if (devices_.size() > 1) {
            if (ptb_group_create(devices_.data(), (int)devices_.size(), &group_) != PTB_OK) throw Error(std::string("ptb_group_create: ") + ptb_group_last_error(nullptr));
            ctx_ = ptb_group_ctx(group_, 0);
        } else if (ptb_create(device_, &ctx_) != PTB_OK) throw Error(std::string("ptb_create: ") + ptb_last_error(nullptr));
    }
    void commit_device() {
        if (group_) { if (ptb_group_commit(group_) != PTB_OK) throw Error(std::string("group commit: ") + ptb_group_last_error(group_)); }
        else ck(ptb_commit(ctx_));
    }
    int device_;
    std::vector<int> devices_;
    ptb_group* group_ = nullptr;
    bool pinned_ = false;
    ptb_ctx* ctx_ = nullptr;
};

}  // namespace ptbhost
