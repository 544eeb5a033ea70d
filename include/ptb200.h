/*
 * ptb200.h — C-ABI of the B200-native radiance loop for nbonneel/pathtracer.
 *
 * The reference has no plugin/FFI interface: its callers reach the hot path through C++ member
 * calls on a by-value `Raytracer` (reference mainApp.h:768, mainApp.cpp:39-47).  This header is the
 * boundary a maintainer binds instead.  Each entry point names the reference interface it replaces
 * (file:line into the reference tree).  Plain pointers and sizes only; no C++ or torch types.
 *
 * Conventions
 *   - every function returns PTB_OK (0) or a negative error code; ptb_last_error() gives the text.
 *     (the reference reports nothing: failures there are crashes or silent garbage.)
 *   - the caller owns all input arrays; the library copies what it needs before returning.
 *   - one ptb_ctx is bound to one CUDA device and is used from one host thread at a time.
 *   - streams: every context works on its own non-blocking CUDA stream and each call returns only after its device work has
 *     finished.  DEVICE buffers handed in by the caller (ptb_render_accum, ptb_resolve, ptb_shard_*) must therefore be ready
 *     before the call (synchronise the stream that produced them), and what the call wrote is complete when it returns.
 *   - object ids are assigned in call order exactly like Scene::addObject (Geometry.cpp:249-252):
 *     id 0 is the spherical light, id 1 the environment dome (Raytracer.cpp:1257-1266, hard-wired
 *     in getColor at Raytracer.cpp:275, 303).
 *   - images use the reference's row convention: pixel (i,j) of the camera lands in row (H-1-i)
 *     (Raytracer.cpp:1651).
 *
 * The same declarations, with the prefix `ref_` / `orc_` instead of `ptb_`, are exported by the two
 * CPU checkers under oracle/ (test infrastructure only): oracle/_ref (the reference's own sources
 * compiled headless) and oracle/port (plain-C restatement).
 */
#ifndef PTB200_H
#define PTB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PTB_OK                0
#define PTB_ERR_INVALID      -1   /* bad argument */
#define PTB_ERR_STATE        -2   /* call order (e.g. render before commit) */
#define PTB_ERR_CUDA         -3   /* CUDA runtime / launch failure */
#define PTB_ERR_NOMEM        -4
#define PTB_ERR_UNSUPPORTED  -5

typedef struct ptb_ctx ptb_ctx;

/* Texture slot == reference `Texture` {values, W, H, multiplier} (BRDF.h:252-426).
 * texels are the POST-LOAD float values, W*H*3, in Texture::values order: colour maps already
 * /255 and ^2.2 (BRDF.h:393-404), normal maps already (v-128) normalised (BRDF.h:406-419), rows
 * already flipped by load_image (utils.cpp:98-170).  W==0 (or texels==NULL) is a constant slot
 * whose value is `mult` (Texture::getVec else-branch, BRDF.h:306-308). */
typedef struct ptb_tex {
    const float* texels;
    int32_t      W, H;
    float        mult[3];
} ptb_tex;

/* Which per-group slots exist.  Object::queryMaterial (Geometry.h:399-445) falls back to
 * Kd=1, Ks=0, Ne=1, opaque, refr 1.3 when `idx >= slot.size()`; an absent bit selects that. */
#define PTB_SLOT_KD      (1u << 0)   /* Object::textures         */
#define PTB_SLOT_KS      (1u << 1)   /* Object::specularmap      */
#define PTB_SLOT_NE      (1u << 2)   /* Object::roughnessmap     */
#define PTB_SLOT_TRANSP  (1u << 3)   /* Object::transparent_map  (transparent iff value < 0.5) */
#define PTB_SLOT_REFR    (1u << 4)   /* Object::refr_index_map   */
#define PTB_SLOT_NORMAL  (1u << 5)   /* Object::normal_map       */
#define PTB_SLOT_ALPHA   (1u << 6)   /* Object::alphamap (hit rejected in traversal iff value < 0.5,
                                        TriangleMesh.cpp:1198-1205, 1298-1305) */
#define PTB_SLOT_KSUB    (1u << 7)   /* Object::subsurface (subsurface albedo Ksub; a surface scatters below itself iff
                                        |Ksub|^2 > 1e-8, Raytracer.cpp:270, 318-406) */

typedef struct ptb_material {
    uint32_t present;               /* PTB_SLOT_* mask */
    ptb_tex  Kd, Ks, Ne, transp, refr, normal, alpha, Ksub;
} ptb_material;

/* Object placement == the fields Object::build_matrix reads (Geometry.h:322-360). */
typedef struct ptb_xform {
    float scale;                    /* Object::scale            */
    float rotation[9];              /* Object::mat_rotation, row-major */
    float rotation_center[3];       /* Object::rotation_center  */
    float translation[3];           /* Object::max_translation  */
} ptb_xform;

#define PTB_OBJ_MIRROR        (1 << 0)   /* Object::miroir        */
#define PTB_OBJ_FLIP_NORMALS  (1 << 1)   /* Object::flip_normals  */
#define PTB_OBJ_FLAT_NORMALS  (1 << 2)   /* !TriMesh::interp_normals (default interpolates) */
#define PTB_OBJ_GHOST         (1 << 3)   /* Object::ghost (Geometry.h:721): invisible to camera paths and shadow rays, but it
                                            receives shadows and shows the background photo (Raytracer.cpp:522-537, 547-549,
                                            614-621; skipped by intersection_shadow, Geometry.cpp:722) */

#define PTB_BRDF_PHONG 0                 /* PhongBRDF   (BRDF.h:37-97), the Object default */
#define PTB_BRDF_MERL  1                 /* IsoMERLBRDF (BRDF.h:192-248) */

/* Triangle mesh as TriMesh::init receives it from a reader (TriangleMesh.cpp:718-841): arrays in
 * FILE order and FILE axes.  The library applies what init applies: axis swap (x,y,z)->(-z,y,x) on
 * vertices and normals (742-751), optional centre + normalise to `scaling` (760-770), per-vertex
 * tangents (601-711).  tri is nTri x 10 int32: {vtx i,j,k, uv i,j,k, normal i,j,k, group}
 * (TriangleIndices, TriangleMesh.h:53-65; -1 = absent).  Triangle ids reported back are indices
 * into this array (the reference's own-BVH path reports BVH-permuted ids, mapped back through
 * permuted_triangle_index, TriangleMesh.cpp:1113). */
typedef struct ptb_mesh {
    const float*   vertices;  int32_t n_vertices;   /* n x 3 */
    const float*   normals;   int32_t n_normals;    /* n x 3 (mandatory for defined shading, see DESIGN.md) */
    const float*   uvs;       int32_t n_uvs;        /* n x 2 */
    const int32_t* tri;       int32_t n_tri;        /* n x 10 */
    float          scaling;                         /* TriMesh ctor `scaling` */
    float          offset[3];                       /* TriMesh ctor `offset`  */
    int32_t        center;                          /* TriMesh ctor `center`  */
} ptb_mesh;

/* Camera == the fields Camera::generateDirection reads (Vector.h:792-825), non-lenticular branch. */
typedef struct ptb_camera {
    float position[3], direction[3], up[3];
    float fov;              /* radians */
    float focus_distance;
    float aperture;
} ptb_camera;

/* Frame parameters == the Raytracer fields render_image_nopreviz reads (Raytracer.h:73-111). */
typedef struct ptb_params {
    int32_t  W, H;
    int32_t  nrays;          /* samples per pixel            */
    int32_t  nb_bounces;     /* path depth                   */
    float    sigma_filter;   /* Gaussian splat sigma         */
    float    gamma;          /* display gamma                */
    uint32_t seed;           /* global seed of the per-(pixel,sample) pcg32 streams (DESIGN.md "RNG") */
    int32_t  shard_rank;     /* image tiles with (tile_id % shard_count) == shard_rank are rendered; tile ids count row by row with
                                every row rotated against the previous one (ptb_scene.h shard_tile_shift), so that shards are
                                spread over the frame instead of forming vertical stripes */
    int32_t  shard_count;    /* 1 = whole frame */
    int32_t  tile_size;      /* tile edge in pixels for sharding; 0 = default (64 for a whole frame, 32 for a shared one) */
} ptb_params;

typedef struct ptb_stats {
    uint64_t samples;        /* camera samples traced                                */
    uint64_t rays_closest;   /* Scene::intersection-equivalent queries               */
    uint64_t rays_shadow;    /* Scene::intersection_shadow-equivalent queries        */
    uint64_t node_visits;    /* wide-node visits   (only when the ctx counts, see ptb_set_option) */
    uint64_t tri_tests;      /* triangle tests     (idem) */
    double   ms_device;      /* CUDA-event time of the render on the device          */
    double   ms_wall;        /* host steady_clock around the call                    */
    uint64_t kernel_launches;
} ptb_stats;

/* ---- lifetime ------------------------------------------------------------------------------- */
/* replaces: `Raytracer` construction (Raytracer.h:28-41) + Scene() (Geometry.h:1240-1281). */
int  ptb_create(int device_id, ptb_ctx** out);
void ptb_destroy(ptb_ctx*);
const char* ptb_last_error(const ptb_ctx*);          /* ctx may be NULL: last error of a failed create */
const char* ptb_version(void);

/* ---- scene ingestion (all before ptb_commit) -------------------------------------------------- */
/* replaces: `new Sphere(O,R)` + Scene::addObject (Geometry.h:852-873, Geometry.cpp:249-252). */
int ptb_add_sphere(ptb_ctx*, const float O[3], float R, const ptb_xform*, int flags, int* out_id);
/* replaces: `new Plane(A,N)` + addObject (Geometry.h:1130-1140). */
int ptb_add_plane(ptb_ctx*, const float A[3], const float N[3], const ptb_xform*, int flags, int* out_id);
/* replaces: `new Cylinder(A, B, R)` + addObject (Geometry.h:731-846): the open tube of radius R around the segment A-B (no caps; a
 * ray that meets the infinite cylinder outside the segment first is a miss even if its second root lies inside, like the
 * reference's test).  Material slot 0 is looked up at (u, v) = (position along the axis / length, 0.5).  The reference builds
 * these for its yarn curves (TriangleMesh.h:281); its default rotation centre is the origin. */
int ptb_add_cylinder(ptb_ctx*, const float A[3], const float B[3], float R, const ptb_xform*, int flags, int* out_id);
/* replaces: `new PointSet(file, nbcols, cols, mirror, normal_swapped, centered)` + addObject (PointSet.h:38-122, PointSet.cpp) with the
 * results of its reader and of estimate_normals (PointSet.h:124-176: nanoflann 10-NN + CImg eigen-solver, not part of this library)
 * passed in memory, as PointSet holds them after init: every point is a DISC (Disk, Geometry.h:1106-1122) with a centre, a normal
 * (used as stored: not normalised for the plane test, normalised for shading), a radius and a colour (PointSet::colors, already
 * /255; NULL = 0.5 grey, the reference's `colors.size() > i` fallback).  Material slot 0 is looked up at uv (0,0) and Kd replaced
 * by the point's colour; the shading normal is turned towards the ray unless the slot is transparent (PointSet.cpp:192-206).
 * PTB_OBJ_DISPLAY_EDGES blackens the outer 5 % ring of every disc (Object::display_edges, PointSet.cpp:212-216).  Triangle ids
 * reported for a point set are point indices into these arrays.  xform->rotation_center NaN: the mean of the points (PointSet.h:113-121). */
typedef struct ptb_pointset {
    const float* points;    /* n x 3  PointSet::vertices */
    const float* normals;   /* n x 3  PointSet::normals  */
    const float* radii;     /* n      PointSet::radius   */
    const float* colors;    /* n x 3  PointSet::colors, or NULL */
    int32_t      n;
} ptb_pointset;
#define PTB_OBJ_DISPLAY_EDGES (1 << 4)
int ptb_add_pointset(ptb_ctx*, const ptb_pointset*, const ptb_xform*, int flags, int* out_id);
/* replaces: `new Yarns(file)` + addObject (TriangleMesh.h:265-312, TriangleMesh.cpp:1519-1737; the GUI adds one for a dropped `.yarn`
 * file, mainApp.cpp:2413-2416) with the segments passed in memory, as Yarns holds them in `cyls` after its constructor: segment i is
 * the open tube `Cylinder(A[i], B[i], R[i])` (Geometry.h:731-846: no caps, only the nearer positive root is tried).  The reference's
 * constructor scales the file's points by 50 and uses R = 0.1 (ptb_yarnfile_read does the same).  Every segment is its own
 * default-constructed Object there, so a yarn is always shaded with queryMaterial's no-texture defaults (Kd = 1, Ks = 0, Ne = 1,
 * opaque: Geometry.h:404-441) and the unnormalised radial normal, never flipped; the Yarns object contributes its transform, its
 * BRDF and its mirror / ghost flags.  Materials set on a yarns object are therefore ignored, like there.  Segments are a third leaf
 * type of the BVH8 (each enters as the triangles of a prism around it and is decided by Cylinder::intersection's arithmetic on the
 * object-space ray).  Triangle ids reported for a yarns object are segment indices into these arrays. */
typedef struct ptb_yarns {
    const float* A;         /* n x 3  cyls[i]->A */
    const float* B;         /* n x 3  cyls[i]->B */
    const float* R;         /* n      cyls[i]->R */
    int32_t      n;
} ptb_yarns;
int ptb_add_yarns(ptb_ctx*, const ptb_yarns*, const ptb_xform*, int flags, int* out_id);
/* replaces: `new TriMesh(scene, file, scaling, offset, mirror, NULL, false, center)` + addObject
 * (TriangleMesh.cpp:714-841), with the reader's arrays passed in memory. */
int ptb_add_mesh(ptb_ctx*, const ptb_mesh*, const ptb_xform*, int flags, int* out_id);
/* replaces: Object::{add,set}_{col_,}{texture,specular,roughness,transp,refr,alpha,normalmap}
 * (Geometry.cpp:56-245) for slot index `group` of object `obj`. */
int ptb_set_group_material(ptb_ctx*, int obj, int group, const ptb_material*);
/* replaces: the material presets of the reference's object menu (mainApp.cpp:1499-1597, ID_GOLD ... ID_COPPER_NGAN): Phong constants
 * {Kd, Ks, Ne}.  "<name>" is the OpenGL-style table entry (Ne = shininess * 128), "<name>_ngan" the Phong fit to the measured BRDF of
 * that material (Ngan et al. 2005) as the reference lists it: gold, silver, pearl, white_plastic, chrome, bronze, copper.  A menu
 * entry does set_col_texture(Kd) + set_col_specular(Ks) + set_col_roughness(Ne,Ne,Ne) on one slot index; the host mirrors do the same
 * (pathtracer_b200/api.py Object.set_preset, ptb_raytracer.hpp Object::set_preset).  ptb_preset_find: index or -1. */
int ptb_preset_count(void);
int ptb_preset_get(int index, const char** name, float Kd[3], float Ks[3], float* Ne);
int ptb_preset_find(const char* name);

/* replaces: `obj->brdf = new IsoMERLBRDF(path)` (mainApp.cpp:2436) / the PhongBRDF default. */
int ptb_set_brdf(ptb_ctx*, int obj, int brdf_kind, int merl_id);
/* replaces: read_brdf (MERLBRDFRead.cpp:212-235): table = 3 x (90*90*180) doubles as stored in the file. */
int ptb_add_merl(ptb_ctx*, const double* table, int* out_merl_id);
/* replaces: Sphere::load_envmap on object 1 (Geometry.h:912-916): 8-bit RGB, rows as load_image returns them. */
int ptb_set_envmap(ptb_ctx*, const uint8_t* rgb, int W, int H);
/* replaces: Scene::intensite_lumiere / Scene::envmap_intensity (Raytracer.cpp:1270-1271). */
int ptb_set_light(ptb_ctx*, float intensite_lumiere, float envmap_intensity);

/* replaces: the Scene::fog_* fields the GUI sliders write (Geometry.h:1371-1377, mainApp.cpp:767-773) and
 * Raytracer::fogContribution reads (Raytracer.cpp:40-192).  density <= 1e-8 switches the medium off (Raytracer.cpp:206).
 * The ground level of the medium is the y translation of object 2 (Raytracer.cpp:54), so a fogged scene needs >= 3 objects. */
typedef struct ptb_fog {
    float   density;            /* Scene::fog_density           */
    float   absorption;         /* Scene::fog_absorption        */
    float   density_decay;      /* Scene::fog_density_decay     */
    float   absorption_decay;   /* Scene::fog_absorption_decay  */
    int32_t type;               /* Scene::fog_type        0 uniform, 1 exponential in height */
    int32_t phase_type;         /* Scene::fog_phase_type  0 isotropic, 1 Schlick, 2 Rayleigh */
    float   phase_aniso;        /* Scene::phase_aniso     Schlick k */
} ptb_fog;
int ptb_set_fog(ptb_ctx*, const ptb_fog*);
/* replaces: Scene::load_background / clear_background (Geometry.h:1348-1366): the photo behind the scene, W*H*3 floats in
 * Scene::background order and scale (already pow(v/255, gamma) * 196964.699).  rgb == NULL or W == 0 clears it.  Camera rays
 * that leave the scene or reach the dome show it (Raytracer.cpp:260-268) and ghost objects tint their indirect light with
 * it (614-621). */
int ptb_set_background(ptb_ctx*, const float* rgb, int W, int H);

/* replaces: Object::{scale,translation,rotation}_keyframes (Geometry.h:313-320; one key of each kind per Object::add_keyframe,
 * nb_transforms rows each in a .scn) and Scene::current_frame (mainApp.cpp:790).  At ptb_commit every object with keys is placed
 * by Object::get_scale / get_translation / get_rotation at the current frame (Geometry.h:258-312: clamped outside the keyed
 * range, linear inside, quaternion Slerp between rotation keys, Vector.h:222-269) exactly like Scene::prepare_render ->
 * Object::build_matrix(current_frame) (Geometry.cpp:283).
 * An animation is: commit once, then per frame ptb_set_frame + ptb_render.  ptb_set_frame on a committed scene does NOT rebuild: the
 * next render (or picking query) first re-poses the scene on the device: object matrices and light constants are recomputed, the
 * world-space triangles are re-derived from the object-space corners resident on the device and the BVH8 boxes are refitted
 * bottom-up with the builder's conservative quantisation (well under a millisecond per million triangles; ptb_scene_info.ms_refit).
 * The tree keeps the topology of the commit frame, which rigid motion preserves; ptb_commit again rebuilds it for the current frame.
 * values: n x 1 (scale), n x 3 (translation), n x 9 (rotation, row-major Matrix33); n == 0 clears the track. */
#define PTB_KEY_SCALE        0
#define PTB_KEY_TRANSLATION  1
#define PTB_KEY_ROTATION     2
int ptb_set_keyframes(ptb_ctx*, int obj, int kind, const float* frames, const float* values, int n);
int ptb_set_frame(ptb_ctx*, float frame);

/* replaces: TriMesh::build_bvh (TriangleMesh.cpp:878-885, 1029-1130) + Scene::prepare_render
 * (Geometry.cpp:280-308): builds the wide BVH over all meshes and uploads the scene to the device. */
int ptb_commit(ptb_ctx*);

/* ---- the hot path ------------------------------------------------------------------------------ */
/* replaces: Raytracer::render_image_nopreviz (Raytracer.cpp:1565-1798) up to and including the
 * tonemap.  HOST outputs, any may be NULL:
 *   imagedouble  W*H*3 float  linear radiance / weight     (Raytracer::imagedouble, 1687-1694)
 *   sample_count W*H   float  filter weight sum            (Raytracer::sample_count)
 *   image        W*H*3 uint8  tonemapped                   (Raytracer::image, 1701-1708)  */
int ptb_render(ptb_ctx*, const ptb_camera*, const ptb_params*,
               float* imagedouble, float* sample_count, uint8_t* image, ptb_stats* stats);

/* replaces: Raytracer::render_image_nopreviz with `has_denoiser == true` (Raytracer.cpp:1631-1645, 1676-1693), up to the hand-over
 * to Open Image Denoise (the denoiser itself is not part of this library).  In this mode the reference does NOT splat: every
 * sample adds its radiance and a count of 1 to its own pixel, and the first hit's albedo (mat.Kd) and shading normal are
 * accumulated next to it (getColor, Raytracer.cpp:254-257).  HOST outputs, W*H*3 floats each (sample_count: W*H), any may be NULL:
 *   imagedouble       mean radiance                           albedoImage   mean first-hit albedo
 *   normalImage       what the reference stores there: it sums the COLOUR buffers instead of the normals (1680-1682) and
 *                     normalises, i.e. the normalised radiance sum (NaN where it is zero)
 *   first_hit_normal  the normalised sum of the first-hit shading normals, the quantity 1680-1682 was written to produce
 * With p->shard_count > 1 only the shard's tiles are rendered: the outputs stay full-frame, sample_count 0 outside them. */
int ptb_render_denoiser_inputs(ptb_ctx*, const ptb_camera*, const ptb_params*, float* imagedouble, float* sample_count,
                               float* albedoImage, float* normalImage, float* first_hit_normal, ptb_stats* stats);

/* replaces: Raytracer::render_image (Raytracer.cpp:1424-1563), the progressive renderer of the GUI thread: one sample per pixel
 * per pass into buffers that persist between passes.  The reference interleaves each pass over 8x8 pixel phases so that a
 * preview fills in evenly on the CPU; the order does not change what is accumulated and a pass takes about a millisecond here,
 * so a pass is simply all pixels.  begin = prepare_render (buffers zeroed, 1382-1389); pass(n) = the next n iterations of the
 * `realtime_ray_iter` loop (1444), fewer if `nrays` is reached; the caller checks its own `stopped` flag between calls (1452).
 * read, HOST outputs, any may be NULL:
 *   imagedouble         W*H*3 UN-normalised weighted sums (the progressive path never divides them, 1491-1493)
 *   sample_count        W*H   filter weight sums (1495)
 *   image               W*H*3 255*(imagedouble/196964.7/max(sample_count,1))^(1/gamma) (1543-1545)
 *   imagedouble_lowres  ceil(W/16)*ceil(H/16)*3: every sample adds colour/256 to its 16x16 block (1508-1510)
 *   current_nb_rays     passes accumulated so far (Raytracer::current_nb_rays, 1445)
 * With p->shard_count > 1 the session renders the shard's tiles only (sample_count 0 outside them, and their splat apron). */
int ptb_progressive_begin(ptb_ctx*, const ptb_camera*, const ptb_params*);
int ptb_progressive_pass(ptb_ctx*, int n_spp, ptb_stats* stats);
int ptb_progressive_read(ptb_ctx*, float* imagedouble, float* sample_count, uint8_t* image, float* imagedouble_lowres,
                         int32_t* current_nb_rays);

/* Sharded form for one-process-per-GPU runs: adds this shard's un-normalised sums into a DEVICE
 * buffer d_rgbw (W*H float4 = {sum r, sum g, sum b, sum weight}, reference row convention) owned
 * by the caller (e.g. a torch tensor, so NCCL can move it).  The buffer is NOT cleared. */
int ptb_render_accum(ptb_ctx*, const ptb_camera*, const ptb_params*, float* d_rgbw, ptb_stats* stats);
/* Normalise + tonemap a DEVICE rgbw buffer into HOST outputs (the tail of render_image_nopreviz,
 * Raytracer.cpp:1687-1708).  Outputs may be NULL. */
int ptb_resolve(ptb_ctx*, const float* d_rgbw, int W, int H, float gamma,
                float* imagedouble, float* sample_count, uint8_t* image);
/* Tile gather support (multi-GPU): pack / unpack-add the tiles owned by a shard, each with a
 * ceil(2*sigma) apron, between a full-frame DEVICE rgbw buffer and a dense DEVICE staging buffer.
 * ptb_shard_pack_size gives the staging size in floats for a shard. */
int ptb_shard_pack_size(const ptb_params*, int shard_rank, int64_t* out_floats);
int ptb_shard_pack(ptb_ctx*, const ptb_params*, int shard_rank, const float* d_rgbw, float* d_packed);
int ptb_shard_unpack_add(ptb_ctx*, const ptb_params*, int shard_rank, const float* d_packed, float* d_rgbw);

/* ---- multi-GPU: the tile-sharded render under ONE call ---------------------------------------------- */
/* The reference's callers make one call per frame, Raytracer::render_image_nopreviz() (mainApp.cpp:38-49).  With several GPUs the
 * frame is sharded by image tiles (owner = tile id % n_ranks, rows rotated), every GPU holds the whole scene, and the only exchange
 * is the gather of the owned tiles (+ a ceil(2 sigma) splat apron) on rank 0: pack -> ncclSend/ncclRecv over NVLink -> unpack-add
 * -> resolve, all inside the call and all on the context's own stream.  NCCL is bound at run time (dlopen of libnccl.so.2: the
 * copy already in the process if there is one; PTB_NCCL_PATH overrides).
 *
 * (1) One process per GPU (e.g. torchrun).  Rank 0 calls ptb_comm_unique_id and hands the 128 bytes to every rank by any means
 * (torch.distributed broadcast, MPI, a file); every rank calls ptb_comm_init on its context (collective), commits the same scene,
 * and then calls ptb_render_sharded with the same camera and parameters (p->shard_rank / shard_count are taken from the
 * communicator).  Rank 0 receives the outputs of ptb_render; on the other ranks the output pointers are ignored.  With all
 * three outputs NULL on rank 0 the gathered sums stay on its device (ptb_resolve_last reads them later).  stats are per rank. */
#define PTB_COMM_ID_BYTES 128
int ptb_comm_unique_id(void* out_id128);
int ptb_comm_init(ptb_ctx*, int n_ranks, int rank, const void* id128);
int ptb_comm_destroy(ptb_ctx*);
int ptb_render_sharded(ptb_ctx*, const ptb_camera*, const ptb_params*,
                       float* imagedouble, float* sample_count, uint8_t* image, ptb_stats* stats);
int ptb_resolve_last(ptb_ctx*, int W, int H, float gamma, float* imagedouble, float* sample_count, uint8_t* image);
/* The other two renderers on every rank of the communicator, called like ptb_render_sharded (same camera and parameters on every
 * rank; the shard comes from the communicator, one rank renders the whole frame).
 * replaces: Raytracer::render_image_nopreviz with has_denoiser (ptb_render_denoiser_inputs).  Rank 0 receives the outputs of
 * ptb_render_denoiser_inputs; the other ranks ignore their output pointers.  The samples are box-filtered, so the tiles travel
 * without an apron (colour, albedo and normal sums: 48 bytes per owned pixel).
 * replaces: Raytracer::render_image (ptb_progressive_begin / _read).  begin_sharded starts a session over this rank's tiles and
 * ptb_progressive_pass renders them.  read_sharded is COLLECTIVE: every rank calls it after the same passes; rank 0 receives the
 * outputs of ptb_progressive_read (the 16x16 preview is summed over the ranks) and the session goes on.  ptb_progressive_read on
 * a session begun here, and ptb_progressive_read_sharded on one begun with ptb_progressive_begin, return PTB_ERR_STATE. */
int ptb_render_denoiser_inputs_sharded(ptb_ctx*, const ptb_camera*, const ptb_params*, float* imagedouble, float* sample_count,
                                       float* albedoImage, float* normalImage, float* first_hit_normal, ptb_stats* stats);
int ptb_progressive_begin_sharded(ptb_ctx*, const ptb_camera*, const ptb_params*);
int ptb_progressive_read_sharded(ptb_ctx*, float* imagedouble, float* sample_count, uint8_t* image, float* imagedouble_lowres,
                                 int32_t* current_nb_rays);

/* (2) One process, several GPUs: a group owns one context (and, during a render, one host thread) per device.  The scene is handed
 * to the LEADER context, ptb_group_ctx(g, 0), with the ptb_add_* / ptb_set_* calls above; ptb_group_commit flattens it and builds
 * the BVH ONCE and uploads it to every device; ptb_group_render is render_image_nopreviz() on all of them (stats: sums over the
 * devices, ms_device of the slowest).  Do not call ptb_commit / ptb_render on the member contexts directly. */
typedef struct ptb_group ptb_group;
int  ptb_group_create(const int* device_ids, int n_devices, ptb_group** out);
void ptb_group_destroy(ptb_group*);
const char* ptb_group_last_error(const ptb_group*);      /* group may be NULL: last error of a failed create */
int  ptb_group_size(const ptb_group*);
ptb_ctx* ptb_group_ctx(ptb_group*, int i);
int  ptb_group_commit(ptb_group*);
int  ptb_group_set_option(ptb_group*, int option, int64_t value);
int  ptb_group_render(ptb_group*, const ptb_camera*, const ptb_params*,
                      float* imagedouble, float* sample_count, uint8_t* image, ptb_stats* stats);
/* replaces: ptb_render_denoiser_inputs on all the group's devices (stats as ptb_group_render) */
int  ptb_group_render_denoiser_inputs(ptb_group*, const ptb_camera*, const ptb_params*, float* imagedouble, float* sample_count,
                                      float* albedoImage, float* normalImage, float* first_hit_normal, ptb_stats* stats);
/* replaces: ptb_progressive_begin / _pass / _read on all the group's devices (pass stats as ptb_group_render).  Pass or read
 * before begin returns PTB_ERR_STATE.  Like ptb_group_render, begin re-poses a key-framed scene after ptb_set_frame on the leader. */
int  ptb_group_progressive_begin(ptb_group*, const ptb_camera*, const ptb_params*);
int  ptb_group_progressive_pass(ptb_group*, int n_spp, ptb_stats* stats);
int  ptb_group_progressive_read(ptb_group*, float* imagedouble, float* sample_count, uint8_t* image, float* imagedouble_lowres,
                                int32_t* current_nb_rays);

/* Host output buffers that live across frames (Raytracer::imagedouble / sample_count / image are members, Raytracer.h:90-105) can
 * be page-locked once, so that the device->host copies that end a render run at PCIe speed without a staging copy.  The buffer
 * must stay allocated until ptb_unpin_host_buffer or ptb_destroy. */
int ptb_pin_host_buffer(ptb_ctx*, void* ptr, int64_t bytes);
int ptb_unpin_host_buffer(ptb_ctx*, void* ptr);

/* replaces: the picking query (mainApp.h:686-692): pixel-centre rays
 * cam.generateDirection(0,i,j,0,0,0,0,0,W,H) + Scene::intersection.  HOST outputs W*H each, row i,
 * column j at [i*W+j] (camera order, not flipped); obj_id -1 = miss; tri_id -1 = not a mesh. */
int ptb_primary_ids(ptb_ctx*, const ptb_camera*, int W, int H,
                    int32_t* obj_id, int32_t* tri_id, float* t);

/* ---- options and introspection ----------------------------------------------------------------- */
#define PTB_OPT_COUNT_TRAVERSAL  1   /* 1: count node visits / triangle tests (instrumented kernels) */
#define PTB_OPT_POOL_PATHS       2   /* paths in flight per pass (default 1<<25, about 5.7 GB of HBM) */
#define PTB_OPT_TIME_KERNELS     3   /* 1: bracket every kernel launch with CUDA events (see ptb_get_kernel_times) */
#define PTB_OPT_REFILL_BELOW     4   /* tuning: a traversal warp refills idle lanes when fewer than this many are live (1..33) */
#define PTB_OPT_TRI_FRACTION     6   /* tuning: triangle steps repeat while >= 1/value of a warp's live lanes have triangle work */
#define PTB_OPT_TRI_MIN_PCT      7   /* tuning: the triangle phase of a warp starts once this % of its live lanes hold triangle work */
/* option 8 is retired (a terminal-hit compaction pass, measured slower and removed); ptb_set_option ignores it.  Do not reuse the number. */
#define PTB_OPT_TRACE_BLOCKS     5   /* tuning: persistent grid size of the traversal kernels (default: SMs x resident blocks) */
#define PTB_OPT_PIPES            9   /* pass pipelines (1..4): consecutive passes of a render run on this many streams, each with its own slice of
                                        the path pool, so that the shade kernels of one pass overlap the traversal kernels of another */
#define PTB_OPT_BUILD_THREADS    10   /* OpenMP threads of the host BVH build at ptb_commit (0 = the OpenMP runtime's default; launchers such as
                                        torchrun export OMP_NUM_THREADS=1, which would serialise the build) */
#define PTB_OPT_STACK_LIMIT      11   /* ptb_commit fails with PTB_ERR_UNSUPPORTED when the BVH8 needs more traversal-stack entries (two per level)
                                        than this; default and maximum: the kernels' 64 entries (32 levels).  The reference's own 50-entry stack
                                        overflows silently (TriangleMesh.cpp:1158). */
int ptb_set_option(ptb_ctx*, int option, int64_t value);

/* Per-kernel device time of the LAST render, measured with CUDA events on the launching stream
 * (PTB_OPT_TIME_KERNELS).  Index: 0 raygen, 1 extend (closest hit), 2 shade, 3 shadow (any hit), 4 splat.
 * ms[k] = summed duration of kernel k's launches, launches[k] = how many, rays[k] = queue entries processed
 * (paths or shadow rays), node_visits/tri_tests per kernel need PTB_OPT_COUNT_TRAVERSAL. */
#define PTB_N_KERNELS 5
typedef struct ptb_kernel_times {
    double   ms[PTB_N_KERNELS];
    uint64_t launches[PTB_N_KERNELS];
    uint64_t items[PTB_N_KERNELS];
    uint64_t node_visits[PTB_N_KERNELS];
    uint64_t tri_tests[PTB_N_KERNELS];
} ptb_kernel_times;
int ptb_get_kernel_times(const ptb_ctx*, ptb_kernel_times*);

typedef struct ptb_scene_info {
    int64_t n_triangles, n_bvh_nodes, bytes_nodes, bytes_triangles, bytes_attributes, bytes_textures;
    int32_t n_objects, bvh_depth;
    double  ms_bvh_build, ms_upload;
    double  ms_refit;        /* device time of the last key-frame re-pose (ptb_set_frame after ptb_commit), 0 if none */
} ptb_scene_info;
int ptb_get_scene_info(const ptb_ctx*, ptb_scene_info*);

/* Function-level probes used by the parity tests: run the DEVICE implementation of one building
 * block on n inputs.  `which` selects the block, in/out layouts are documented in DESIGN.md §KAT. */
#define PTB_KAT_PCG32          1   /* in: u64 {state_seed, stream} x n  -> out: 4 x u32 draws as double */
#define PTB_KAT_LATTICE        2   /* in: k                    -> out: x, y                  (Raytracer.cpp:1311-1319) */
#define PTB_KAT_CAMERA         3   /* in: i,j,dx,dy,ax,ay      -> out: o[3], d[3]            (Vector.h:792-825) */
#define PTB_KAT_RANDOM_COS     4   /* in: N[3], r1, r2         -> out: v[3]                  (Vector.h:581-589) */
#define PTB_KAT_RANDOM_PHONG   5   /* in: R[3], n, r1, r2      -> out: v[3]                  (BRDF.h:41-61) */
#define PTB_KAT_PHONG_EVAL     6   /* in: Kd3,Ks3,Ne3,wi3,wo3,N3 -> out: f[3]                (BRDF.h:88-96) */
#define PTB_KAT_MERL_EVAL      7   /* in: wi3,wo3,N3 (merl id 0) -> out: f[3]                (BRDF.h:204-246) */
#define PTB_KAT_FAST_EXP       8   /* in: y                    -> out: fast_exp(y)           (Raytracer.cpp:1294-1299) */
#define PTB_KAT_FAST_NORMALIZE 9   /* in: v[3]                 -> out: v[3]                  (Vector.h:294-309, 376-382) */
#define PTB_KAT_RANDOM_PER_PIXEL 10 /* in: pixel index p       -> out: randomPerPixel[p].x,.y (Raytracer.cpp:1341-1344) */
#define PTB_KAT_FILTER_RATIO   11  /* in: i,j,W,H,sigma        -> out: ratio                 (Raytracer.cpp:1604-1608) */
#define PTB_KAT_MERL_INDEX     12  /* in: wi3,wo3 (local frame, z = normal) -> out: bin index of the float path (-1: it declined), bin index of
                                      the double path (MERLBRDFRead.cpp:76-207); the two must agree wherever the first is >= 0 */
/* KAT 13 is retired (the half-factor node test, measured slower and removed).  Do not reuse the number. */
int ptb_kat(ptb_ctx*, int which, const ptb_camera* cam, int W, int H,
            const double* in, int n, int in_stride, double* out, int out_stride);

#ifdef __cplusplus
}
#endif
#endif /* PTB200_H */
