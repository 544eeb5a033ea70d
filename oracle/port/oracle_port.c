/*
 * oracle/port/oracle_port.c — TEST INFRASTRUCTURE ONLY.  Plain-C CPU restatement of the reference's
 * radiance loop (nbonneel/pathtracer), used as the parity checker for the CUDA path and as the
 * "port" CPU baseline of bench.py.  Nothing in pathtracer_b200/ may link, import or execute it.
 *
 * PINNED: this restatement is checked against oracle/_ref (the reference's own sources compiled
 * headless, oracle/build_ref.py) by tests/test_oracle_pinning.py — function-level known answers are
 * bit-identical and single-thread images agree bit for bit on the committed scenes — and against the
 * golden vectors under tests/golden/ generated from oracle/_ref (tests/golden/make_golden.py).
 *
 * Every function cites the reference file:line it restates.  Same algorithm, same float/double
 * evaluation order (C++ overload resolution written out: cosf vs cos, powf vs pow ...), same binary
 * BVH (TriangleMesh.cpp:1029-1130), same traversal order, same per-(pixel,sample) pcg32 streams that
 * oracle/build_ref.py patches into the reference copy (DESIGN.md "RNG").  Fog, subsurface, ghost and
 * background-photo branches are outside the contract (SURVEY.md §8a last row) and are not restated.
 */
#define ORACLE_PREFIX orc_
#include "../prefix.h"
#include "../../include/ptb200.h"

#include <float.h>
#include <math.h>
#include <omp.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif
#define M_TWO_PI_REF 6.28318530718 /* Vector.h:16-18 */

typedef struct { float x, y, z; } vec;
static inline vec V(float x, float y, float z) { vec r = {x, y, z}; return r; }
static inline vec vadd(vec a, vec b) { return V(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline vec vsub(vec a, vec b) { return V(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline vec vneg(vec a) { return V(-a.x, -a.y, -a.z); }
static inline vec vmul(vec a, vec b) { return V(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline vec vscale(float s, vec a) { return V(s * a.x, s * a.y, s * a.z); }
static inline vec vdiv(vec a, float s) { return V(a.x / s, a.y / s, a.z / s); }
static inline float vdot(vec a, vec b) { return a.x * b.x + a.y * b.y + a.z * b.z; }      /* Vector.h:553-556 */
static inline float vnorm2(vec a) { return a.x * a.x + a.y * a.y + a.z * a.z; }          /* Vector.h:367-369 */
static inline vec vcross(vec a, vec b) { return V(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
static inline vec vnormalize(vec a) { float n = sqrtf(vnorm2(a)); return V(a.x / n, a.y / n, a.z / n); } /* Vector.h:371-376 */
static inline vec vreflect(vec d, vec N) { return vsub(d, vscale(2.f * vdot(d, N), N)); } /* Vector.h:388-391 */
static inline float vget(vec a, int k) { return k == 0 ? a.x : (k == 1 ? a.y : a.z); }

/* Vector.h:294-309 with the 4-byte pun of the author's platform (build_ref.py patch 4) */
static inline float inv_sq_root(float n) {
    float y = n;
    int32_t i;
    memcpy(&i, &y, 4);
    i = 0x5f3759df - (i >> 1);
    memcpy(&y, &i, 4);
    y = y * (1.5F - ((n * 0.5F) * y * y));
    y = y * (1.5F - ((n * 0.5F) * y * y));
    return y;
}
static inline vec vfast_normalize(vec a) { float inv = inv_sq_root(vnorm2(a)); return V(a.x * inv, a.y * inv, a.z * inv); } /* Vector.h:376-382 */

/* ---- pcg32 (pcg_random.hpp:1866, 845-873, 484-501, 158-159) ------------------------------------- */
typedef struct { uint64_t state, inc; } pcg;
#define PCG_MULT 6364136223846793005ULL
#define PCG_DEFAULT_INC 1442695040888963407ULL
static inline pcg pcg_seed2(uint64_t seed, uint64_t stream) { pcg r; r.inc = (stream << 1) | 1ULL; r.state = (seed + r.inc) * PCG_MULT + r.inc; return r; }
static inline pcg pcg_seed1(uint64_t seed) { pcg r; r.inc = PCG_DEFAULT_INC; r.state = (seed + r.inc) * PCG_MULT + r.inc; return r; }
static inline uint32_t pcg_next(pcg* r) {
    uint64_t old = r->state;
    r->state = old * PCG_MULT + r->inc;
    uint32_t xs = (uint32_t)(((old >> 18u) ^ old) >> 27u), rot = (uint32_t)(old >> 59u);
    return (xs >> rot) | (xs << ((32u - rot) & 31u));
}
static const float INVMAX = 1.f / 4294967296.f; /* 1.f/engine.max(): max() = 2^32-1 rounds to 2^32 as float (Raytracer.h:28) */
static inline float pcg_unif(pcg* r) { return (float)pcg_next(r) * INVMAX; }

/* ---- Raytracer.cpp:1294-1319 -------------------------------------------------------------------- */
static double fast_exp(double y) {
    int32_t hi = (int32_t)(1512775 * y + 1072632447);
    uint64_t bits = ((uint64_t)(uint32_t)hi) << 32;
    double d; memcpy(&d, &bits, 8); return d;
}
static uint32_t reverse_bits(uint32_t n) {
    n = (n << 16) | (n >> 16);
    n = ((n & 0x00ff00ff) << 8) | ((n & 0xff00ff00) >> 8);
    n = ((n & 0x0f0f0f0f) << 4) | ((n & 0xf0f0f0f0) >> 4);
    n = ((n & 0x33333333) << 2) | ((n & 0xcccccccc) >> 2);
    n = ((n & 0x55555555) << 1) | ((n & 0xaaaaaaaa) >> 1);
    return n;
}
static void lattice2d(uint32_t id, float* x, float* y) {
    uint32_t rid = reverse_bits(id);
    float phi = (float)(rid * pow(2.0, -32));
    float tmp;
    *x = modff((float)(phi * 1 + 0.456789123), &tmp);      /* modf(float,float*) overload: narrowed first */
    *y = modff((float)(phi * 182667 + 0.123456789), &tmp);
}

/* ---- Vector.h:566-589, BRDF.h:41-97 ---------------------------------------------------------------- */
static vec get_tangent(vec N) {
    float ax = fabsf(N.x), ay = fabsf(N.y), az = fabsf(N.z);
    vec t;
    if (ax <= ay && ax <= az) t = V(0, -N.z, N.y);
    else if (ay <= ax && ay <= az) t = V(-N.z, 0, N.x);
    else t = V(-N.y, N.x, 0);
    return vnormalize(t);
}
static vec random_cos(vec N, float r1, float r2) {
    float sr2 = sqrtf(1.f - r2);
    float twopi = (float)(2. * M_PI);
    vec l = V(cosf(twopi * r1) * sr2, sinf(twopi * r1) * sr2, sqrtf(r2));
    vec t1 = get_tangent(N), t2 = vcross(t1, N);
    return vadd(vadd(vscale(l.z, N), vscale(l.x, t1)), vscale(l.y, t2));
}
static vec random_phong(vec R, float n, float r1, float r2) {
    float facteur = sqrtf(1 - powf(r2, 2.f / (n + 1.f)));
    vec l = V((float)(cos(2 * M_PI * r1) * facteur), (float)(sin(2 * M_PI * r1) * facteur), (float)pow(r2, 1. / (n + 1)));
    vec t1 = get_tangent(R), t2 = vcross(t1, R);
    return vadd(vadd(vscale(l.z, R), vscale(l.x, t1)), vscale(l.y, t2));
}
typedef struct { vec shadingN, Kd, Ks, Ne, Ke, Ksub; int transp; float refr_index; } matvals; /* BRDF.h:7-20 */
static matvals matvals_default(void) {
    matvals m; m.shadingN = V(0, 1, 0); m.Kd = V(.5f, .5f, .5f); m.Ne = V(100, 100, 100); m.Ks = V(0, 0, 0); m.Ke = V(0, 0, 0); m.Ksub = V(0, 0, 0);
    m.transp = 0; m.refr_index = 1.3f; /* uninitialised in the reference; only read after queryMaterial set them */
    return m;
}
static vec phong_eval(const matvals* m, vec wi, vec wo, vec N) {
    vec refl = vreflect(vneg(wo), N);
    float d = vdot(refl, wi);
    if (d < 0) return vdiv(m->Kd, (float)M_PI);
    vec lobe = V((float)(powf(d, m->Ne.x) * (m->Ne.x + 2.f) / M_TWO_PI_REF), (float)(powf(d, m->Ne.y) * (m->Ne.y + 2.f) / M_TWO_PI_REF),
                 (float)(powf(d, m->Ne.z) * (m->Ne.z + 2.f) / M_TWO_PI_REF));
    return vadd(vdiv(m->Kd, (float)M_PI), vmul(lobe, m->Ks));
}
static vec phong_sample(const matvals* m, vec wo, vec N, float* pdf, float r1, float r2, pcg* e, int* has_sampled_diffuse) {
    float avgNe = (m->Ne.x + m->Ne.y + m->Ne.z) / 3.f;
    float p = 1 - (m->Ks.x + m->Ks.y + m->Ks.z) / 3.f;
    vec R = vreflect(vneg(wo), N), dir;
    if (pcg_next(e) / 4294967296.f < p) { *has_sampled_diffuse = 1; dir = random_cos(N, r1, r2); }
    else { *has_sampled_diffuse = 0; dir = random_phong(R, avgNe, r1, r2); }
    float proba_phong = (float)((avgNe + 1) / (2.f * M_PI) * powf(vdot(R, dir), avgNe));
    *pdf = (float)(p * vdot(N, dir) / (M_PI) + (1.f - p) * proba_phong);
    return dir;
}

/* ---- MERLBRDFRead.cpp:50-207, BRDF.h:204-246 ---------------------------------------------------- */
static void merl_rotate(const double* v, const double* axis, double angle, double* out) {
    double c = cos(angle), s = sin(angle), temp;
    out[0] = v[0] * c; out[1] = v[1] * c; out[2] = v[2] * c;
    temp = axis[0] * v[0] + axis[1] * v[1] + axis[2] * v[2];
    temp = temp * (1.0 - c);
    out[0] += axis[0] * temp; out[1] += axis[1] * temp; out[2] += axis[2] * temp;
    double cr[3] = {axis[1] * v[2] - axis[2] * v[1], axis[2] * v[0] - axis[0] * v[2], axis[0] * v[1] - axis[1] * v[0]};
    out[0] += cr[0] * s; out[1] += cr[1] * s; out[2] += cr[2] * s;
}
static void dnormalize(double* v) { double len = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); v[0] /= len; v[1] /= len; v[2] /= len; }
static vec merl_eval(const double* brdf, vec wi, vec wo, vec N) {
    const double PI = 3.1415926535897932384626433832795;
    vec t1 = get_tangent(N), t2 = vcross(t1, N);
    vec wil = V(vdot(wi, t1), vdot(wi, t2), vdot(wi, N)), wol = V(vdot(wo, t1), vdot(wo, t2), vdot(wo, N));
    float thetai = acosf(wil.z);
    if (thetai >= M_PI / 2) return V(0, 0, 0);
    float thetao = acosf(wol.z);
    if (thetao >= M_PI / 2) return V(0, 0, 0);
    float phio = atan2f(wol.y, wol.x);
    if (phio < 0) phio = (float)(phio + 2 * M_PI);
    float phii = atan2f(wil.y, wil.x);
    if (phii < 0) phii = (float)(phii + 2 * M_PI);
    double theta_in = thetai, fi_in = phii, theta_out = thetao, fi_out = phio;
    double in_z = cos(theta_in), pin = sin(theta_in), in_x = pin * cos(fi_in), in_y = pin * sin(fi_in);
    double in[3] = {in_x, in_y, in_z};
    dnormalize(in);
    double out_z = cos(theta_out), pout = sin(theta_out), out_x = pout * cos(fi_out), out_y = pout * sin(fi_out);
    double half[3] = {(in_x + out_x) / 2.0f, (in_y + out_y) / 2.0f, (in_z + out_z) / 2.0f};
    dnormalize(half);
    double theta_half = acos(half[2]), fi_half = atan2(half[1], half[0]);
    const double bi_normal[3] = {0.0, 1.0, 0.0}, normal[3] = {0.0, 0.0, 1.0};
    double temp[3], diff[3];
    merl_rotate(in, normal, -fi_half, temp);
    merl_rotate(temp, bi_normal, -theta_half, diff);
    double theta_diff = acos(diff[2]), fi_diff = atan2(diff[1], diff[0]);
    int ih, id, ip;
    if (theta_half <= 0.0) ih = 0;
    else { double deg = ((theta_half / (PI / 2.0)) * 90); double t = sqrt(deg * 90); ih = (int)t; if (ih < 0) ih = 0; if (ih >= 90) ih = 89; }
    id = (int)(theta_diff / (PI * 0.5) * 90);
    if (id < 0) id = 0; else if (id >= 89) id = 89;
    if (fi_diff < 0.0) fi_diff += PI;
    ip = (int)(fi_diff / PI * 360 / 2);
    if (ip < 0) ip = 0; else if (ip >= 179) ip = 179;
    int ind = ip + id * 360 / 2 + ih * 360 / 2 * 90;
    double r = brdf[ind] * (1.0 / 1500.0), g = brdf[ind + 90 * 90 * 360 / 2] * (1.15 / 1500.0), b = brdf[ind + 90 * 90 * 360] * (1.66 / 1500.0);
    return V((float)r, (float)g, (float)b);
}

/* ---- Texture (BRDF.h:252-426) --------------------------------------------------------------------- */
typedef struct { float mult[3]; size_t W, H; float* values; } tex;
typedef struct { tex* t; int n; } slotv; /* std::vector<Texture> */
enum { S_KD, S_KS, S_NE, S_TRANSP, S_REFR, S_NORMAL, S_ALPHA, S_KSUB, S_COUNT };
static float tex_wrap(float u) { u -= (int)u; if (u < 0) u += 1; return u; }
static size_t tex_idx(const tex* t, float u, float v) { int x = (int)(u * (t->W - 1)); int y = (int)(v * (t->H - 1)); return (y * t->W + x) * 3; }
static vec tex_vec(const tex* t, float u, float v) {
    if (t->W > 0) { size_t i = tex_idx(t, u, v); return V(t->values[i] * t->mult[0], t->values[i + 1] * t->mult[1], t->values[i + 2] * t->mult[2]); }
    return V(t->mult[0], t->mult[1], t->mult[2]);
}
static float tex_red(const tex* t, float u, float v) { if (t->W > 0) return t->values[tex_idx(t, u, v)] * t->mult[0]; return t->mult[0]; }
static vec tex_normal(const tex* t, float u, float v) {
    if (t->W > 0) { size_t i = tex_idx(t, u, v); return V(t->values[i], t->values[i + 1], t->values[i + 2]); }
    return V(0.f, 0.f, 1.f);
}

/* ---- objects --------------------------------------------------------------------------------------- */
typedef struct { vec lo, hi; } box;
typedef struct { int isleaf, fg, fd; box bb; } bnode;                       /* BVHNodesT, TriangleMesh.h:6-13 */
typedef struct { int vtx[3], uv[3], n[3], group; } tindex;                  /* TriangleIndices, TriangleMesh.h:53-65 */
typedef struct { vec A, u, v, N; float m11, m12, m22, invdetm; float uvs[3][2]; vec normals[3]; } tsoup; /* Triangle, 67-111 */
enum { T_MESH, T_SPHERE, T_PLANE, T_CYLINDER, T_POINTSET, T_YARNS };
typedef struct {
    int type, miroir, flip_normals, interp_normals, brdf, ghost;
    const double* merl;
    float scale, rot[9]; vec rc, tr;
    int nkey[3]; float* kframe[3]; float* kval[3];      /* scale / translation / rotation keyframes (Geometry.h:318-320), frames ascending */
    float scale_at, rot_at[9]; vec tr_at;               /* the placement at Scene::current_frame (get_scale / get_rotation / get_translation) */
    float trans[12], inv[12], rotm[9];
    slotv slots[S_COUNT];
    vec O; float R, R2; int has_envmap; const uint8_t* envtex; int envW, envH;   /* Sphere */
    vec A, vecN;                                                              /* Plane (Cylinder: A) */
    int np, display_edges; vec *pt_pos, *pt_nrm, *pt_col; double* pt_rad; int* pt_perm;   /* PointSet: vertices, normals, colors (NULL: none), radius; perm: original index */
    int ny; vec *yA, *yB, *yd; float *yR, *ylen; int* y_perm;                 /* Yarns: cyls[i]->A, B, d, R, len (TriangleMesh.h:265-312); perm: index handed in */
    vec cylB, cyld; float cyllen;                                             /* Cylinder: B, d, len (Geometry.h:734-738, 843-844) */
    int nv, nn, nuv, nt;                                                      /* TriMesh */
    vec *vertices, *normals; float* uvs; tindex* indices; tsoup* soup; vec* tangent_soup; int* permuted;
    bnode* nodes; int n_nodes, cap_nodes; box bvh_bbox; int bvh_depth;
} object;

struct ptb_ctx {
    object** objs; int n_objs;
    double** merl; int n_merl;
    uint8_t* env; int envW, envH;
    float intensite_lumiere, envmap_intensity;
    ptb_fog fog; float* bg; int bgW, bgH;      /* Scene::fog_*, Scene::background (Geometry.h:1365-1377) */
    int current_frame;                          /* Scene::current_frame (an int, Geometry.h:1372) */
    int committed, threads;
    char err[256];
    double ms_build; long long n_tri;
    /* frame state (Raytracer fields) */
    int W, H, nrays, nb_bounces; float sigma_filter, gamma; uint32_t seed;
    vec cam_pos, cam_dir, cam_up; float fov, focus_distance, aperture;
    vec centerLight; float radiusLight, lightPower;
    int filter_size, filter_total_width; float filter_integral[81];
    vec* randomPerPixel; int rpp_n;
    /* progressive session (Raytracer::render_image): the buffers that persist between passes */
    int prog_active, prog_iter; float* prog_img; float* prog_cnt; float* prog_lowres; vec* prog_samples2d;
    unsigned long long prog_counters[64][8];
};
static char g_err[256];

/* Matrix<3,3,float>::toQuaternion / fromQuaternion (Vector.h:104-160), Slerp (Vector.h:222-269) */
static void mat_to_quat(const float* v, float q[4]) {
    float m00 = v[0], m01 = v[3], m02 = v[6], m10 = v[1], m11 = v[4], m12 = v[7], m20 = v[2], m21 = v[5], m22 = v[8];
    float tr = m00 + m11 + m22, qw, qx, qy, qz;
    if (tr > 0) { float S = (float)(sqrt(tr + 1.0) * 2); qw = (float)(0.25 * S); qx = (m21 - m12) / S; qy = (m02 - m20) / S; qz = (m10 - m01) / S; }
    else if ((m00 > m11) & (m00 > m22)) { float S = (float)(sqrt(1.0 + m00 - m11 - m22) * 2); qw = (m21 - m12) / S; qx = (float)(0.25 * S); qy = (m01 + m10) / S; qz = (m02 + m20) / S; }
    else if (m11 > m22) { float S = (float)(sqrt(1.0 + m11 - m00 - m22) * 2); qw = (m02 - m20) / S; qx = (m01 + m10) / S; qy = (float)(0.25 * S); qz = (m12 + m21) / S; }
    else { float S = (float)(sqrt(1.0 + m22 - m00 - m11) * 2); qw = (m10 - m01) / S; qx = (m02 + m20) / S; qy = (m12 + m21) / S; qz = (float)(0.25 * S); }
    q[0] = qw; q[1] = qx; q[2] = qy; q[3] = qz;
}
static void slerp33(const float* a, const float* b, float t, float* v) {
    float q1[4], q2[4];
    mat_to_quat(a, q1); mat_to_quat(b, q2);
    float w1 = q1[0], x1 = q1[1], y1 = q1[2], z1 = q1[3], w2 = q2[0], x2 = q2[1], y2 = q2[2], z2 = q2[3];
    if (w1 * w2 + x1 * x2 + y1 * y2 + z1 * z2 < 0) { w2 = -w2; x2 = -x2; y2 = -y2; z2 = -z2; }
    float theta = acosf(w1 * w2 + x1 * x2 + y1 * y2 + z1 * z2), mult1, mult2;
    if (theta > 0.000001) { mult1 = sinf((1 - t) * theta) / sinf(theta); mult2 = sinf(t * theta) / sinf(theta); }
    else { mult1 = 1 - t; mult2 = t; }
    float w = mult1 * w1 + mult2 * w2, x = mult1 * x1 + mult2 * x2, y = mult1 * y1 + mult2 * y2, z = mult1 * z1 + mult2 * z2;
    v[0] = w * w + x * x - y * y - z * z; v[1] = (float)(2.0 * x * y + 2.0 * w * z); v[2] = (float)(2.0 * x * z - 2.0 * y * w);
    v[3] = (float)(2.0 * x * y - 2.0 * w * z); v[4] = w * w - x * x + y * y - z * z; v[5] = (float)(2.0 * y * z + 2.0 * w * x);
    v[6] = (float)(2.0 * x * z + 2.0 * w * y); v[7] = (float)(2.0 * y * z - 2.0 * w * x); v[8] = w * w - x * x - y * y + z * z;
}
/* Object::get_scale / get_translation / get_rotation (Geometry.h:258-312) for track `kind` (width 1 / 3 / 9) */
static int key_eval(const object* o, int kind, float frame, float* out) {
    static const int width[3] = {1, 3, 9};
    int n = o->nkey[kind], w = width[kind];
    if (n == 0) return 0;
    const float* fr = o->kframe[kind]; const float* val = o->kval[kind];
    int up = 0;
    while (up < n && !(fr[up] > frame)) up++;                          /* upper_bound */
    if (up == n) { memcpy(out, val + (size_t)(n - 1) * w, w * sizeof(float)); return 1; }
    if (up == 0) { memcpy(out, val, w * sizeof(float)); return 1; }
    float t = (frame - fr[up - 1]) / (fr[up] - fr[up - 1]);
    const float* a = val + (size_t)(up - 1) * w; const float* b = val + (size_t)up * w;
    if (w == 9) slerp33(a, b, t, out);
    else if (w == 3) for (int i = 0; i < 3; i++) out[i] = (1 - t) * a[i] + t * b[i];
    else out[0] = (1.f - t) * a[0] + t * b[0];
    return 1;
}
/* Object::build_matrix(frame) (Geometry.h:322-360) */
static void build_matrix(object* o, float frame) {
    o->scale_at = o->scale; memcpy(o->rot_at, o->rot, sizeof(o->rot)); o->tr_at = o->tr;
    float tv[3];
    key_eval(o, PTB_KEY_SCALE, frame, &o->scale_at);
    if (key_eval(o, PTB_KEY_TRANSLATION, frame, tv)) o->tr_at = V(tv[0], tv[1], tv[2]);
    key_eval(o, PTB_KEY_ROTATION, frame, o->rot_at);
    const float* m = o->rot_at; float mt[9];
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) mt[j * 3 + i] = m[i * 3 + j];
    float s = o->scale_at;
    for (int i = 0; i < 3; i++) {
        vec v2 = V(m[0 * 3 + i], m[1 * 3 + i], m[2 * 3 + i]);
        o->trans[0 * 4 + i] = v2.x * s; o->trans[1 * 4 + i] = v2.y * s; o->trans[2 * 4 + i] = v2.z * s;
        o->rotm[0 * 3 + i] = v2.x; o->rotm[1 * 3 + i] = v2.y; o->rotm[2 * 3 + i] = v2.z;
        v2 = V(mt[0 * 3 + i], mt[1 * 3 + i], mt[2 * 3 + i]);
        o->inv[0 * 4 + i] = v2.x / s; o->inv[1 * 4 + i] = v2.y / s; o->inv[2 * 4 + i] = v2.z / s;
    }
    float b[3] = {-o->rc.x, -o->rc.y, -o->rc.z}, r[3];
    for (int i = 0; i < 3; i++) { float v = 0; for (int j = 0; j < 3; j++) v += m[i * 3 + j] * b[j]; r[i] = v; }
    o->trans[3] = r[0] * s + o->rc.x + o->tr_at.x; o->trans[7] = r[1] * s + o->rc.y + o->tr_at.y; o->trans[11] = r[2] * s + o->rc.z + o->tr_at.z;
    vec q = vsub(vneg(o->rc), o->tr_at);
    float b2[3] = {q.x, q.y, q.z};
    for (int i = 0; i < 3; i++) { float v = 0; for (int j = 0; j < 3; j++) v += mt[i * 3 + j] * b2[j]; r[i] = v; }
    o->inv[3] = r[0] / s + o->rc.x; o->inv[7] = r[1] / s + o->rc.y; o->inv[11] = r[2] / s + o->rc.z;
}
static vec xf_point(const float* m, vec v) { return V(m[0] * v.x + m[1] * v.y + m[2] * v.z + m[3], m[4] * v.x + m[5] * v.y + m[6] * v.z + m[7], m[8] * v.x + m[9] * v.y + m[10] * v.z + m[11]); }
static vec xf_dir(const float* m, vec v) { return V(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[4] * v.x + m[5] * v.y + m[6] * v.z, m[8] * v.x + m[9] * v.y + m[10] * v.z); }
static vec xf_rot(const float* m, vec v) { return V(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[3] * v.x + m[4] * v.y + m[5] * v.z, m[6] * v.x + m[7] * v.y + m[8] * v.z); }

/* Object::queryMaterial (Geometry.h:399-445); idx is compared as size_t in the reference, so -1 selects the defaults */
static void query_material(const object* o, int idx, float u, float v, matvals* m) {
    u = tex_wrap(u); v = tex_wrap(v);
    size_t i = (size_t)idx;
    if (i >= (size_t)o->slots[S_KD].n) m->Kd = V(1, 1, 1); else m->Kd = tex_vec(&o->slots[S_KD].t[i], u, v);
    if (i >= (size_t)o->slots[S_KS].n) m->Ks = V(0, 0, 0); else m->Ks = tex_vec(&o->slots[S_KS].t[i], u, v);
    if (i >= (size_t)o->slots[S_KSUB].n) m->Ksub = V(0, 0, 0); else m->Ksub = tex_vec(&o->slots[S_KSUB].t[i], u, v);
    if (i >= (size_t)o->slots[S_NE].n) m->Ne = V(1, 1, 1); else m->Ne = tex_vec(&o->slots[S_NE].t[i], u, v);
    if (i >= (size_t)o->slots[S_TRANSP].n) m->transp = 0; else m->transp = tex_red(&o->slots[S_TRANSP].t[i], u, v) < 0.5f;
    if (i >= (size_t)o->slots[S_REFR].n) m->refr_index = 1.3f; else m->refr_index = tex_red(&o->slots[S_REFR].t[i], u, v);
    m->Ke = V(0, 0, 0);
}

/* ---- BBox slab tests (Geometry.h:114-204) ----------------------------------------------------------- */
typedef struct { vec o, id; } invray;
static inline float bnd(const box* b, int hi, int k) { return vget(hi ? b->hi : b->lo, k); }
static int box_invd(const box* b, const invray* r, const char s[3], float* t) { /* 114-141 */
    float tmax = (bnd(b, s[0], 0) - r->o.x) * r->id.x;
    if (tmax < 0) return 0;
    *t = (bnd(b, 1 - s[0], 0) - r->o.x) * r->id.x;
    float tmaxy = (bnd(b, s[1], 1) - r->o.y) * r->id.y;
    if (tmaxy < 0) return 0;
    float tminy = (bnd(b, 1 - s[1], 1) - r->o.y) * r->id.y;
    if (tminy > tmax || tmaxy < *t) return 0;
    if (tminy > *t) *t = tminy;
    if (tmaxy < tmax) tmax = tmaxy;
    float tmaxz = (bnd(b, s[2], 2) - r->o.z) * r->id.z;
    if (tmaxz < 0) return 0;
    float tminz = (bnd(b, 1 - s[2], 2) - r->o.z) * r->id.z;
    if (*t > tmaxz || tminz > tmax) return 0;
    if (tminz > *t) *t = tminz;
    if (*t < 0) *t = 0;
    return 1;
}
static int box_invd_x(const box* b, const invray* r, const char s[3], float* t, int positive) { /* 143-204 */
    float tmax;
    if (positive) { tmax = (b->hi.x - r->o.x); if (tmax < 0) return 0; tmax *= r->id.x; *t = (b->lo.x - r->o.x) * r->id.x; }
    else { tmax = (b->lo.x - r->o.x); if (tmax > 0) return 0; tmax *= r->id.x; *t = (b->hi.x - r->o.x) * r->id.x; }
    float tmaxy = (bnd(b, s[1], 1) - r->o.y) * r->id.y;
    if (tmaxy < 0) return 0;
    float tminy = (bnd(b, 1 - s[1], 1) - r->o.y) * r->id.y;
    if (tminy > tmax || tmaxy < *t) return 0;
    if (tminy > *t) *t = tminy;
    if (tmaxy < tmax) tmax = tmaxy;
    float tmaxz = (bnd(b, s[2], 2) - r->o.z) * r->id.z;
    if (tmaxz < 0) return 0;
    float tminz = (bnd(b, 1 - s[2], 2) - r->o.z) * r->id.z;
    if (*t > tmaxz || tminz > tmax) return 0;
    if (tminz > *t) *t = tminz;
    if (*t < 0) *t = 0;
    return 1;
}

/* Triangle ctor + Triangle::intersection (TriangleMesh.h:70-104) */
static tsoup soup_make(vec A, vec B, vec C) {
    tsoup s; memset(&s, 0, sizeof(s));
    s.A = A; s.u = vsub(B, A); s.v = vsub(C, A); s.N = vcross(s.u, s.v);
    s.m11 = vnorm2(s.u); s.m22 = vnorm2(s.v); s.m12 = vdot(s.u, s.v);
    s.invdetm = (float)(1. / (s.m11 * s.m22 - s.m12 * s.m12));
    return s;
}
static int soup_hit(const tsoup* s, vec o, vec d, vec* P, float* t, float* alpha, float* beta, float* gamma) {
    *t = vdot(vsub(s->A, o), s->N) / vdot(d, s->N);
    if (*t < 0 || *t != *t) return 0;
    *P = vadd(o, vscale(*t, d));
    vec w = vsub(*P, s->A);
    float b11 = vdot(w, s->u), b21 = vdot(w, s->v);
    float detb = b11 * s->m22 - b21 * s->m12;
    *beta = detb * s->invdetm;
    if (*beta < 0) return 0;
    float detg = b21 * s->m11 - b11 * s->m12;
    *gamma = detg * s->invdetm;
    if (*gamma < 0) return 0;
    *alpha = 1 - *beta - *gamma;
    if (*alpha < 0) return 0;
    return 1;
}

/* ---- binary BVH build (TriangleMesh.cpp:844-885, 1029-1130) ----------------------------------------- */
static vec vmin3(vec a, vec b) { return V(a.x < b.x ? a.x : b.x, a.y < b.y ? a.y : b.y, a.z < b.z ? a.z : b.z); } /* std::min(a,b): b<a?b:a */
static vec vmax3(vec a, vec b) { return V(a.x < b.x ? b.x : a.x, a.y < b.y ? b.y : a.y, a.z < b.z ? b.z : a.z); }
static float fminr(float a, float b) { return b < a ? b : a; } /* std::min */
static float fmaxr(float a, float b) { return a < b ? b : a; } /* std::max */
static box mesh_bbox(const object* g, int i0, int i1) {
    box r; r.hi = g->vertices[g->indices[i0].vtx[0]]; r.lo = r.hi;
    for (int i = i0; i < i1; i++)
        for (int c = 0; c < 3; c++) { vec p = g->vertices[g->indices[i].vtx[c]]; r.lo = vmin3(r.lo, p); r.hi = vmax3(r.hi, p); }
    return r;
}
static vec tri_center(const object* g, int i) {
    const tindex* t = &g->indices[i];
    return vdiv(vadd(vadd(g->vertices[t->vtx[0]], g->vertices[t->vtx[1]]), g->vertices[t->vtx[2]]), 3.f);
}
static box centers_bbox(const object* g, int i0, int i1) {
    box r; r.hi = tri_center(g, i0); r.lo = r.hi;
    for (int i = i0; i < i1; i++) { vec c = tri_center(g, i); r.lo = vmin3(r.lo, c); r.hi = vmax3(r.hi, c); }
    return r;
}
static float box_area(const box* b) { vec s = vsub(b->hi, b->lo); return 2 * (s.x * s.y + s.x * s.z + s.y * s.z); }
static float center_dim(const object* g, int i, int d) { /* (a+b+c)/3. : double division, narrowed */
    const tindex* t = &g->indices[i];
    return (float)((vget(g->vertices[t->vtx[0]], d) + vget(g->vertices[t->vtx[1]], d) + vget(g->vertices[t->vtx[2]], d)) / 3.);
}
static void bvh_recur(object* g, int node, int i0, int i1, int depth) {
    if (g->n_nodes == g->cap_nodes) { g->cap_nodes *= 2; g->nodes = (bnode*)realloc(g->nodes, sizeof(bnode) * (size_t)g->cap_nodes); }
    bnode n; n.bb = mesh_bbox(g, i0, i1); n.fg = i0; n.fd = i1; n.isleaf = 1;
    g->nodes[g->n_nodes++] = n;
    if (depth > g->bvh_depth) g->bvh_depth = depth;
    box cb = centers_bbox(g, i0, i1);
    vec diag = vsub(cb.hi, cb.lo);
    int dim;
    if (diag.x >= diag.y && diag.x >= diag.z) dim = 0; else if (diag.y >= diag.x && diag.y >= diag.z) dim = 1; else dim = 2;
    float best_factor = 0.5f, best_area = INFINITY; /* 1E50 as float */
    for (int k = 0; k < 16; k++) {
        float f = (k + 1) / (float)(16 + 1);
        float split = vget(cb.lo, dim) + vget(diag, dim) * f;
        box L = {V(1E10f, 1E10f, 1E10f), V(-1E10f, -1E10f, -1E10f)}, Rb = L;
        int nl = 0, nr = 0;
        for (int i = i0; i < i1; i++) {
            float c = center_dim(g, i, dim);
            const tindex* t = &g->indices[i];
            box* bb = (c <= split) ? &L : &Rb;
            for (int q = 0; q < 3; q++) bb->lo = vmin3(bb->lo, g->vertices[t->vtx[q]]);
            for (int q = 0; q < 3; q++) bb->hi = vmax3(bb->hi, g->vertices[t->vtx[q]]);
            if (c <= split) nl++; else nr++;
        }
        float sum = box_area(&L) * nl + box_area(&Rb) * nr;
        if (sum < best_area) { best_factor = f; best_area = sum; }
    }
    float split = vget(cb.lo, dim) + vget(diag, dim) * best_factor;
    int pivot = i0 - 1;
    for (int i = i0; i < i1; i++) {
        if (center_dim(g, i, dim) <= split) {
            pivot++;
            tindex t = g->indices[i]; g->indices[i] = g->indices[pivot]; g->indices[pivot] = t;
            int p = g->permuted[i]; g->permuted[i] = g->permuted[pivot]; g->permuted[pivot] = p;
        }
    }
    if (pivot < i0 || pivot >= i1 - 1 || i1 <= i0 + 4) return;
    g->nodes[node].isleaf = 0;
    g->nodes[node].fg = g->n_nodes;
    bvh_recur(g, g->nodes[node].fg, i0, pivot + 1, depth + 1);
    g->nodes[node].fd = g->n_nodes;
    bvh_recur(g, g->nodes[node].fd, pivot + 1, i1, depth + 1);
}

/* TriMesh::setup_tangents (TriangleMesh.cpp:601-711) */
static void setup_tangents(object* g) {
    vec* tan1 = (vec*)calloc((size_t)g->nv, sizeof(vec));
    vec* tan2 = (vec*)calloc((size_t)g->nv, sizeof(vec));
    for (int i = 0; i < g->nt; i++) {
        const tindex* t = &g->indices[i];
        if (t->uv[0] == -1 || t->uv[1] == -1 || t->uv[2] == -1) continue;
        int a = t->vtx[0], b = t->vtx[1], c = t->vtx[2];
        vec vA = vsub(g->vertices[b], g->vertices[a]), vB = vsub(g->vertices[c], g->vertices[a]);
        float sA0 = g->uvs[2 * t->uv[1]] - g->uvs[2 * t->uv[0]], sA1 = g->uvs[2 * t->uv[1] + 1] - g->uvs[2 * t->uv[0] + 1];
        float sB0 = g->uvs[2 * t->uv[2]] - g->uvs[2 * t->uv[0]], sB1 = g->uvs[2 * t->uv[2] + 1] - g->uvs[2 * t->uv[0] + 1];
        float det = (sA0 * sB1 - sB0 * sA1);
        vec sdir, tdir;
        if (det != 0) { sdir = vdiv(vsub(vscale(sB1, vA), vscale(sA1, vB)), det); tdir = vdiv(vsub(vscale(sA0, vB), vscale(sB0, vA)), det); }
        else { sdir = vscale(0.00001f, vA); tdir = vscale(0.00001f, vB); }
        tan1[a] = vadd(tan1[a], sdir); tan1[b] = vadd(tan1[b], sdir); tan1[c] = vadd(tan1[c], sdir);
        tan2[a] = vadd(tan2[a], tdir); tan2[b] = vadd(tan2[b], tdir); tan2[c] = vadd(tan2[c], tdir);
    }
    for (int i = 0; i < g->nt; i++) { /* missing normals -> face normal (649-668) */
        tindex* t = &g->indices[i];
        if (t->n[0] != -1 && t->n[1] != -1 && t->n[2] != -1) continue;
        vec fn = vnormalize(vcross(vsub(g->vertices[t->vtx[1]], g->vertices[t->vtx[0]]), vsub(g->vertices[t->vtx[2]], g->vertices[t->vtx[0]])));
        g->normals = (vec*)realloc(g->normals, sizeof(vec) * (size_t)(g->nn + 1));
        g->normals[g->nn] = fn;
        for (int k = 0; k < 3; k++) if (t->n[k] == -1) t->n[k] = g->nn;
        g->nn++;
    }
    int* vtn = (int*)calloc((size_t)g->nv, sizeof(int));
    for (int i = 0; i < g->nt; i++) for (int k = 0; k < 3; k++) vtn[g->indices[i].vtx[k]] = g->indices[i].n[k];
    vec* tangents = (vec*)malloc(sizeof(vec) * (size_t)g->nv);
    for (int i = 0; i < g->nv; i++) {
        vec N = vnormalize(g->normals[vtn[i]]);
        tangents[i] = vnormalize(vsub(tan1[i], vscale(vdot(tan1[i], N), N)));
    }
    g->tangent_soup = (vec*)malloc(sizeof(vec) * 3 * (size_t)g->nt);
    for (int i = 0; i < g->nt; i++) for (int k = 0; k < 3; k++) g->tangent_soup[i * 3 + k] = tangents[g->indices[i].vtx[k]];
    free(tan1); free(tan2); free(vtn); free(tangents);
}

/* TriMesh::getMaterial (TriangleMesh.cpp:919-1026) */
static void mesh_material(const object* g, int tri, float alpha, float beta, float gamma, matvals* m) {
    float u = 0, v = 0;
    const tindex* t = &g->indices[tri];
    const tsoup* s = &g->soup[tri];
    int has_uv = 0;
    if (g->nuv != 0 && t->group >= 0 && t->uv[0] >= 0 && !(t->uv[0] >= g->nuv)) {
        u = (s->uvs[0][0] * alpha + s->uvs[1][0] * beta + s->uvs[2][0] * gamma);
        v = (s->uvs[0][1] * alpha + s->uvs[1][1] * beta + s->uvs[2][1] * gamma);
        has_uv = 1;
    }
    query_material(g, t->group, u, v, m);
    if (!g->interp_normals || t->n[0] == -1) m->shadingN = s->N;
    else m->shadingN = vadd(vadd(vscale(alpha, s->normals[0]), vscale(beta, s->normals[1])), vscale(gamma, s->normals[2]));
    m->shadingN = vnormalize(m->shadingN);
    if (g->slots[S_NORMAL].n != 0 && has_uv && (size_t)t->group < (size_t)g->slots[S_NORMAL].n) {
        vec tangent = vadd(vadd(vscale(alpha, g->tangent_soup[tri * 3]), vscale(beta, g->tangent_soup[tri * 3 + 1])), vscale(gamma, g->tangent_soup[tri * 3 + 2]));
        tangent = vnormalize(tangent);
        vec bitangent = vcross(m->shadingN, tangent);
        vec nl = tex_normal(&g->slots[S_NORMAL].t[t->group], u, v);
        vec Ns = vadd(vadd(vscale(nl.x, tangent), vscale(nl.y, bitangent)), vscale(nl.z, m->shadingN));
        if (Ns.x == 0. && Ns.y == 0 && Ns.z == 0) Ns = m->shadingN;
        m->shadingN = vnormalize(Ns);
    }
    if (g->flip_normals) m->shadingN = vneg(m->shadingN);
}

/* alpha test inside traversal (TriangleMesh.cpp:1198-1205) */
static int alpha_skip(const object* g, int i, float alpha, float beta, float gamma) {
    const tindex* t = &g->indices[i];
    int tid = t->group;
    if (g->nuv > 0 && (size_t)g->slots[S_ALPHA].n > (size_t)tid && t->uv[0] >= 0 && t->uv[1] >= 0 && t->uv[2] >= 0) {
        float u = g->uvs[2 * t->uv[0]] * alpha + g->uvs[2 * t->uv[1]] * beta + g->uvs[2 * t->uv[2]] * gamma;
        float v = g->uvs[2 * t->uv[0] + 1] * alpha + g->uvs[2 * t->uv[1] + 1] * beta + g->uvs[2 * t->uv[2] + 1] * gamma;
        u = tex_wrap(u); v = tex_wrap(v);
        if (tex_red(&g->slots[S_ALPHA].t[tid], u, v) < 0.5) return 1;
    }
    return 0;
}

/* TriMesh::intersection (TriangleMesh.cpp:1133-1235) / intersection_shadow (1239-1319) */
static int mesh_hit(const object* g, vec o, vec d, vec* P, float* t, matvals* mat, float cur_best_t, int* tri_id, int shadow, float dist_light) {
    *t = cur_best_t;
    int has = 0, best = -1;
    float tl, tr_, lt, alpha, beta, gamma;
    vec lp;
    invray r; r.o = o; r.id = V((float)(1. / d.x), (float)(1. / d.y), (float)(1. / d.z));
    char s[3] = {(char)(r.id.x >= 0 ? 1 : 0), (char)(r.id.y >= 0 ? 1 : 0), (char)(r.id.z >= 0 ? 1 : 0)};
    if (!box_invd(&g->bvh_bbox, &r, s, &tl)) return 0;
    if (tl > cur_best_t || (shadow && tl > dist_light)) return 0;
    int l[50]; float tn[50]; int top = -1;
    l[++top] = 0; tn[top] = tl;
    while (top >= 0) {
        if (tn[top] > *t) { top--; continue; }
        int cur = l[top--];
        int fg = g->nodes[cur].fg, fd = g->nodes[cur].fd;
        if (!g->nodes[cur].isleaf) {
            int gl, gr;
            if (shadow) {
                gl = box_invd(&g->nodes[fg].bb, &r, s, &tl) && tl < *t && tl < dist_light;
                gr = box_invd(&g->nodes[fd].bb, &r, s, &tr_) && tr_ < *t && tr_ < dist_light;
            } else {
                gl = box_invd_x(&g->nodes[fg].bb, &r, s, &tl, s[0] == 1) && tl < *t;
                gr = box_invd_x(&g->nodes[fd].bb, &r, s, &tr_, s[0] == 1) && tr_ < *t;
            }
            if (gl && gr) {
                if (tl < tr_) { l[++top] = fd; tn[top] = tr_; l[++top] = fg; tn[top] = tl; }
                else { l[++top] = fg; tn[top] = tl; l[++top] = fd; tn[top] = tr_; }
            } else {
                if (gl) { l[++top] = fg; tn[top] = tl; }
                if (gr) { l[++top] = fd; tn[top] = tr_; }
            }
        } else {
            for (int i = fg; i < fd; i++) {
                if (soup_hit(&g->soup[i], o, d, &lp, &lt, &alpha, &beta, &gamma) && lt < *t) {
                    if (alpha_skip(g, i, alpha, beta, gamma)) continue;
                    has = 1; best = i; *t = lt;
                    if (shadow && *t < dist_light * 0.999) return 1;
                }
            }
        }
    }
    if (has && !shadow) {
        *tri_id = best;
        soup_hit(&g->soup[best], o, d, &lp, &lt, &alpha, &beta, &gamma);
        if (isnan(alpha) && isnan(beta) && isnan(gamma)) { alpha = 1; beta = 0; gamma = 0; }
        if (isnan(alpha)) alpha = 0;
        if (isnan(beta)) beta = 0;
        if (isnan(gamma)) gamma = 0;
        if (isinf(alpha)) alpha = 1;
        if (isinf(beta)) beta = 1;
        if (isinf(gamma)) gamma = 1;
        *P = lp;
        mesh_material(g, best, alpha, beta, gamma, mat);
    }
    return has;
}

/* TriMesh::reservoir_sampling_intersection (TriangleMesh.cpp:1321-1424): a uniformly random one of the mesh's intersections with
 * min_t <= t < max_t, by reservoir sampling in BVH traversal order (one draw per accepted hit) */
static int mesh_reservoir(const object* g, vec o, vec d, vec* P, float* t, matvals* mat, int* tri_id, int* nb_intersections, float min_t, float max_t, pcg* e) {
    int has = 0, best = -1;
    float tl, tr_, lt, alpha, beta, gamma;
    vec lp;
    invray r; r.o = o; r.id = V((float)(1. / d.x), (float)(1. / d.y), (float)(1. / d.z));
    char s[3] = {(char)(r.id.x >= 0 ? 1 : 0), (char)(r.id.y >= 0 ? 1 : 0), (char)(r.id.z >= 0 ? 1 : 0)};
    if (!box_invd(&g->bvh_bbox, &r, s, &tl)) return 0;
    if (tl > max_t) return 0;
    int l[50]; float tn[50]; int top = -1;
    l[++top] = 0; tn[top] = tl;
    while (top >= 0) {
        if (tn[top] > max_t) { top--; continue; }
        int cur = l[top--];
        int fg = g->nodes[cur].fg, fd = g->nodes[cur].fd;
        if (!g->nodes[cur].isleaf) {
            int gl = box_invd_x(&g->nodes[fg].bb, &r, s, &tl, s[0] == 1) && tl < max_t;
            int gr = box_invd_x(&g->nodes[fd].bb, &r, s, &tr_, s[0] == 1) && tr_ < max_t;
            if (gl && gr) {
                if (tl < tr_) { l[++top] = fd; tn[top] = tr_; l[++top] = fg; tn[top] = tl; }
                else { l[++top] = fg; tn[top] = tl; l[++top] = fd; tn[top] = tr_; }
            } else {
                if (gl) { l[++top] = fg; tn[top] = tl; }
                if (gr) { l[++top] = fd; tn[top] = tr_; }
            }
        } else {
            for (int i = fg; i < fd; i++) {
                if (soup_hit(&g->soup[i], o, d, &lp, &lt, &alpha, &beta, &gamma)) {
                    if (lt < max_t && lt >= min_t) {
                        if (alpha_skip(g, i, alpha, beta, gamma)) continue;
                        (*nb_intersections)++;
                        float r1 = pcg_unif(e);
                        if (r1 < 1. / *nb_intersections) { has = 1; best = i; *t = lt; }
                    }
                }
            }
        }
    }
    if (has) {
        *tri_id = best;
        soup_hit(&g->soup[best], o, d, &lp, &lt, &alpha, &beta, &gamma);
        if (isnan(alpha) && isnan(beta) && isnan(gamma)) { alpha = 1; beta = 0; gamma = 0; }
        if (isnan(alpha)) alpha = 0;
        if (isnan(beta)) beta = 0;
        if (isnan(gamma)) gamma = 0;
        if (isinf(alpha)) alpha = 1;
        if (isinf(beta)) beta = 1;
        if (isinf(gamma)) gamma = 1;
        *P = lp;
        mesh_material(g, best, alpha, beta, gamma, mat);
    }
    return has;
}

/* Sphere::intersection (Geometry.h:918-992) / intersection_shadow (1071-1094) */
static int sphere_hit(const object* sp, vec o, vec d, vec* P, float* t, matvals* mat, int shadow) {
    float b = vdot(d, vsub(o, sp->O));
    float a = vnorm2(d);
    float c = vnorm2(vsub(o, sp->O)) - sp->R2;
    float delta = b * b - a * c;
    if (delta < 0) return 0;
    float sq = sqrtf(delta);
    float inva = shadow ? (float)(1. / a) : 1.f / a;
    float t2 = (-b + sq) * inva;
    if (t2 < 0) return 0;
    float t1 = (-b - sq) * inva;
    *t = t1 > 0 ? t1 : t2;
    if (shadow) return 1;
    *P = vadd(o, vscale(*t, d));
    vec N = vsub(*P, sp->O);
    if (sp->has_envmap) {
        N = vfast_normalize(N);
        float theta = 1.f - acosf(N.y) / (float)M_PI;
        float phi = (float)((atan2f(-N.z, N.x) + M_PI) / (2.f * (float)M_PI));
        query_material(sp, 0, theta, phi, mat);
        mat->shadingN = vneg(N);
        int idx = 3 * ((int)(theta * (sp->envH - 1.f)) * sp->envW + (int)(phi * (sp->envW - 1.f)));
        if (idx < 0 || idx >= 3 * sp->envW * sp->envH) mat->Ke = V(0, 0, 0);
        else mat->Ke = vscale(100000.f / 255.f, V(sp->envtex[idx], sp->envtex[idx + 1], sp->envtex[idx + 2]));
        return 1;
    }
    if (sp->slots[S_KD].n || sp->slots[S_KS].n || sp->slots[S_NE].n || sp->slots[S_TRANSP].n || sp->slots[S_REFR].n) {
        N = vfast_normalize(N);
        float theta = 1.f - acosf(N.y) / (float)M_PI;
        float phi = (atan2f(-N.z, N.x) + (float)M_PI) / (2.f * (float)M_PI);
        query_material(sp, 0, theta, phi, mat);
    }
    mat->shadingN = N;
    mat->Ke = V(0, 0, 0);
    if (sp->flip_normals) mat->shadingN = vneg(mat->shadingN);
    return 1;
}
/* Plane::intersection (Geometry.h:1142-1157) / intersection_shadow (1185-1191) */
static int plane_hit(const object* pl, vec o, vec d, vec* P, float* t, matvals* mat, int shadow) {
    if (!shadow) mat->shadingN = pl->vecN;
    float ddot = vdot(d, pl->vecN);
    if (fabsf(ddot) < 1E-9) return 0;
    *t = vdot(vsub(pl->A, o), pl->vecN) / ddot;
    if (*t <= 0.) return 0;
    if (shadow) return 1;
    *P = vadd(o, vscale(*t, d));
    query_material(pl, 0, P->x * 0.1f, P->z * 0.1f, mat);
    return 1;
}

/* ---- PointSet (PointSet.cpp): its own binary BVH over discs ---------------------------------------------- */
static vec rad3(const object* g, int i) { float r = (float)g->pt_rad[i]; return V(r, r, r); }   /* Vector(radius[i], radius[i], radius[i]) */
static box pts_bbox(const object* g, int i0, int i1) {                                            /* build_bbox, 4-14 */
    box r; r.hi = vadd(g->pt_pos[i0], rad3(g, i0)); r.lo = vsub(g->pt_pos[i0], rad3(g, i0));
    for (int i = i0; i < i1; i++) { r.lo = vmin3(r.lo, vsub(g->pt_pos[i], rad3(g, i))); r.hi = vmax3(r.hi, vadd(g->pt_pos[i], rad3(g, i))); }
    return r;
}
static box pts_centers_bbox(const object* g, int i0, int i1) {                                    /* build_centers_bbox, 16-26 */
    box r; r.hi = g->pt_pos[i0]; r.lo = g->pt_pos[i0];
    for (int i = i0; i < i1; i++) { r.lo = vmin3(r.lo, g->pt_pos[i]); r.hi = vmax3(r.hi, g->pt_pos[i]); }
    return r;
}
static void pts_bvh_recur(object* g, int node, int i0, int i1, int depth) {                       /* build_bvh_recur, 34-122 */
    if (g->n_nodes == g->cap_nodes) { g->cap_nodes *= 2; g->nodes = (bnode*)realloc(g->nodes, sizeof(bnode) * (size_t)g->cap_nodes); }
    bnode n; n.bb = pts_bbox(g, i0, i1); n.fg = i0; n.fd = i1; n.isleaf = 1;
    g->nodes[g->n_nodes++] = n;
    if (depth > g->bvh_depth) g->bvh_depth = depth;
    box cb = pts_centers_bbox(g, i0, i1);
    vec diag = vsub(cb.hi, cb.lo);
    int dim;
    if (diag.x >= diag.y && diag.x >= diag.z) dim = 0; else if (diag.y >= diag.x && diag.y >= diag.z) dim = 1; else dim = 2;
    double best_factor = 0.5, best_area = 1E50;
    for (int k = 0; k < 16; k++) {
        double f = (k + 1) / (double)(16 + 1);
        double split = vget(cb.lo, dim) + vget(diag, dim) * f;
        box L = {V(1E10f, 1E10f, 1E10f), V(-1E10f, -1E10f, -1E10f)}, Rb = L;
        int nl = 0, nr = 0;
        for (int i = i0; i < i1; i++) {
            double c = vget(g->pt_pos[i], dim);
            if (c <= split) { L.lo = vmin3(L.lo, vsub(g->pt_pos[i], rad3(g, i))); L.hi = vmax3(L.hi, vadd(g->pt_pos[i], rad3(g, i))); nl++; }
            else { Rb.lo = vmin3(Rb.lo, vsub(g->pt_pos[i], rad3(g, i))); Rb.hi = vmax3(Rb.hi, vadd(g->pt_pos[i], rad3(g, i))); nr++; }
        }
        double sum = box_area(&L) * nl + box_area(&Rb) * nr;       /* float area() * int, summed in float, widened */
        if (sum < best_area) { best_factor = f; best_area = sum; }
    }
    double split = vget(cb.lo, dim) + vget(diag, dim) * best_factor;
    int pivot = i0 - 1;
    for (int i = i0; i < i1; i++) {
        double c = vget(g->pt_pos[i], dim);
        if (c <= split) {
            pivot++;
            vec tv = g->pt_pos[i]; g->pt_pos[i] = g->pt_pos[pivot]; g->pt_pos[pivot] = tv;
            if (g->pt_col) { tv = g->pt_col[i]; g->pt_col[i] = g->pt_col[pivot]; g->pt_col[pivot] = tv; }
            tv = g->pt_nrm[i]; g->pt_nrm[i] = g->pt_nrm[pivot]; g->pt_nrm[pivot] = tv;
            double tr = g->pt_rad[i]; g->pt_rad[i] = g->pt_rad[pivot]; g->pt_rad[pivot] = tr;
            int tp = g->pt_perm[i]; g->pt_perm[i] = g->pt_perm[pivot]; g->pt_perm[pivot] = tp;
        }
    }
    if (pivot < i0 || pivot >= i1 - 1 || i1 <= i0 + 4) return;
    g->nodes[node].isleaf = 0;
    g->nodes[node].fg = g->n_nodes;
    pts_bvh_recur(g, g->nodes[node].fg, i0, pivot + 1, depth + 1);
    g->nodes[node].fd = g->n_nodes;
    pts_bvh_recur(g, g->nodes[node].fd, pivot + 1, i1, depth + 1);
}
/* Disk::intersection (Geometry.h:1110-1118) */
static int disk_hit(vec c, vec n, float r, vec o, vec d, vec* P, float* t) {
    *t = vdot(vsub(c, o), n) / vdot(d, n);
    if (*t < 0 || *t != *t) return 0;
    *P = vadd(o, vscale(*t, d));
    float r2 = vnorm2(vsub(*P, c));
    return r2 <= r * r;
}
/* PointSet::intersection (PointSet.cpp:124-220) / intersection_shadow (247-315) */
static int pts_hit(const object* g, vec o, vec d, vec* P, float* t, matvals* mat, float cur_best_t, int* tri_id, int shadow, float dist_light) {
    *t = cur_best_t;
    int has = 0, best = -1;
    float tl, tr_, lt;
    vec lp;
    invray r; r.o = o; r.id = V(1.f / d.x, 1.f / d.y, 1.f / d.z);
    char s[3] = {(char)(r.id.x >= 0 ? 1 : 0), (char)(r.id.y >= 0 ? 1 : 0), (char)(r.id.z >= 0 ? 1 : 0)};
    if (!box_invd(&g->bvh_bbox, &r, s, &tl)) return 0;
    if (tl > cur_best_t || (shadow && tl > dist_light)) return 0;
    int l[50]; float tn[50]; int top = -1;
    l[++top] = 0; tn[top] = tl;
    while (top >= 0) {
        if (tn[top] > *t) { top--; continue; }
        int cur = l[top--];
        int fg = g->nodes[cur].fg, fd = g->nodes[cur].fd;
        if (!g->nodes[cur].isleaf) {
            int gl = box_invd(&g->nodes[fg].bb, &r, s, &tl) && tl < *t && (!shadow || tl < dist_light);
            int gr = box_invd(&g->nodes[fd].bb, &r, s, &tr_) && tr_ < *t && (!shadow || tr_ < dist_light);
            if (gl && gr) {
                if (tl < tr_) { l[++top] = fd; tn[top] = tr_; l[++top] = fg; tn[top] = tl; }
                else { l[++top] = fg; tn[top] = tl; l[++top] = fd; tn[top] = tr_; }
            } else {
                if (gl) { l[++top] = fg; tn[top] = tl; }
                if (gr) { l[++top] = fd; tn[top] = tr_; }
            }
        } else {
            for (int i = fg; i < fd; i++)
                if (disk_hit(g->pt_pos[i], g->pt_nrm[i], (float)g->pt_rad[i], o, d, &lp, &lt) && lt < *t) { has = 1; best = i; *t = lt; }
        }
    }
    if (has && !shadow) {
        int i = best;
        *tri_id = best;
        disk_hit(g->pt_pos[i], g->pt_nrm[i], (float)g->pt_rad[i], o, d, &lp, &lt);
        vec N = vnormalize(g->pt_nrm[i]);
        *P = lp;
        query_material(g, 0, 0, 0, mat);
        mat->shadingN = N;
        if (vdot(mat->shadingN, d) > 0 && !mat->transp) mat->shadingN = vneg(mat->shadingN);
        if (g->flip_normals) mat->shadingN = vneg(mat->shadingN);
        if (g->pt_col) mat->Kd = g->pt_col[i]; else mat->Kd = V(0.5f, 0.5f, 0.5f);
        if (g->display_edges) {
            float r2 = vnorm2(vsub(lp, g->pt_pos[i]));
            if (r2 > (g->pt_rad[i] * g->pt_rad[i] * 0.95 * 0.95)) mat->Kd = V(0, 0, 0);
        }
    }
    return has;
}

/* Cylinder::intersection (Geometry.h:740-766); intersection_shadow is the same call (836-841) */
static int cylinder_hit(const object* cy, vec o, vec d, vec* P, float* t, matvals* mat) {
    vec X = vsub(d, vscale(vdot(d, cy->cyld), cy->cyld));
    vec oa = vsub(o, cy->A);
    vec Y = vsub(oa, vscale(vdot(oa, cy->cyld), cy->cyld));
    float a = vnorm2(X);
    float b = 2 * vdot(X, Y);
    float c = vnorm2(Y) - cy->R * cy->R;
    float delta = b * b - 4 * a * c;
    if (delta < 0) return 0;
    float sdelta = sqrtf(delta);
    float t2 = (-b + sdelta) / (2 * a);
    if (t2 < 0) return 0;
    float t1 = (-b - sdelta) / (2 * a);
    if (t1 > 0) *t = t1; else *t = t2;
    *P = vadd(o, vscale(*t, d));
    float dP = vdot(vsub(*P, cy->A), cy->cyld);
    if (dP < 0 || dP > cy->cyllen) return 0;
    vec proj = vadd(cy->A, vscale(dP, cy->cyld));
    query_material(cy, 0, dP / cy->cyllen, 0.5f, mat);
    mat->shadingN = vsub(*P, proj);
    if (cy->flip_normals) mat->shadingN = vneg(mat->shadingN);
    return 1;
}

/* ---- Yarns (TriangleMesh.h:265-312, TriangleMesh.cpp:1519-1737): a binary BVH over Cylinder segments --------------------- */
static vec yr3(const object* g, int i) { return V(g->yR[i], g->yR[i], g->yR[i]); }
static box yarn_bbox(const object* g, int i0, int i1) {                                           /* build_bbox, 1519-1533 */
    box r; r.hi = V(-FLT_MAX, -FLT_MAX, -FLT_MAX); r.lo = V(FLT_MAX, FLT_MAX, FLT_MAX);
    for (int i = i0; i < i1; i++) {
        r.lo = vmin3(r.lo, vsub(g->yA[i], yr3(g, i))); r.hi = vmax3(r.hi, vadd(g->yA[i], yr3(g, i)));
        r.lo = vmin3(r.lo, vsub(g->yB[i], yr3(g, i))); r.hi = vmax3(r.hi, vadd(g->yB[i], yr3(g, i)));
    }
    return r;
}
static vec yarn_center(const object* g, int i) { return vdiv(vadd(g->yA[i], g->yB[i]), 2.f); }
static box yarn_centers_bbox(const object* g, int i0, int i1) {                                   /* build_centers_bbox, 1535-1548 */
    box r; r.hi = yarn_center(g, i0); r.lo = r.hi;
    for (int i = i0; i < i1; i++) { vec c = yarn_center(g, i); r.lo = vmin3(r.lo, c); r.hi = vmax3(r.hi, c); }
    return r;
}
static float yarn_center_dim(const object* g, int i, int dim) { return (float)((vget(g->yA[i], dim) + vget(g->yB[i], dim)) / 2.); }
static void yarn_bvh_recur(object* g, int node, int i0, int i1, int depth) {                      /* build_bvh_recur, 1556-1647 */
    if (g->n_nodes == g->cap_nodes) { g->cap_nodes *= 2; g->nodes = (bnode*)realloc(g->nodes, sizeof(bnode) * (size_t)g->cap_nodes); }
    bnode n; n.bb = yarn_bbox(g, i0, i1); n.fg = i0; n.fd = i1; n.isleaf = 1;
    g->nodes[g->n_nodes++] = n;
    if (depth > g->bvh_depth) g->bvh_depth = depth;
    box cb = yarn_centers_bbox(g, i0, i1);
    vec diag = vsub(cb.hi, cb.lo);
    int dim;
    if (diag.x >= diag.y && diag.x >= diag.z) dim = 0; else if (diag.y >= diag.x && diag.y >= diag.z) dim = 1; else dim = 2;
    float best_factor = 0.5f, best_area = INFINITY; /* 1E50 as float */
    for (int k = 0; k < 16; k++) {
        float f = (k + 1) / (float)(16 + 1);
        float split = vget(cb.lo, dim) + vget(diag, dim) * f;
        box L = {V(1E10f, 1E10f, 1E10f), V(-1E10f, -1E10f, -1E10f)}, Rb = L;
        int nl = 0, nr = 0;
        for (int i = i0; i < i1; i++) {
            box* bb = (yarn_center_dim(g, i, dim) <= split) ? &L : &Rb;
            bb->lo = vmin3(bb->lo, vsub(g->yA[i], yr3(g, i))); bb->lo = vmin3(bb->lo, vsub(g->yB[i], yr3(g, i)));
            bb->hi = vmax3(bb->hi, vadd(g->yA[i], yr3(g, i))); bb->hi = vmax3(bb->hi, vadd(g->yB[i], yr3(g, i)));
            if (bb == &L) nl++; else nr++;
        }
        float sum = box_area(&L) * nl + box_area(&Rb) * nr;
        if (sum < best_area) { best_factor = f; best_area = sum; }
    }
    float split = vget(cb.lo, dim) + vget(diag, dim) * best_factor;
    int pivot = i0 - 1;
    for (int i = i0; i < i1; i++) {
        if (yarn_center_dim(g, i, dim) <= split) {
            pivot++;                                                  /* std::swap(cyls[i], cyls[pivot]) */
            vec tv = g->yA[i]; g->yA[i] = g->yA[pivot]; g->yA[pivot] = tv;
            tv = g->yB[i]; g->yB[i] = g->yB[pivot]; g->yB[pivot] = tv;
            tv = g->yd[i]; g->yd[i] = g->yd[pivot]; g->yd[pivot] = tv;
            float tf = g->yR[i]; g->yR[i] = g->yR[pivot]; g->yR[pivot] = tf;
            tf = g->ylen[i]; g->ylen[i] = g->ylen[pivot]; g->ylen[pivot] = tf;
            int tp = g->y_perm[i]; g->y_perm[i] = g->y_perm[pivot]; g->y_perm[pivot] = tp;
        }
    }
    if (pivot < i0 || pivot >= i1 - 1 || i1 <= i0 + 4) return;
    g->nodes[node].isleaf = 0;
    g->nodes[node].fg = g->n_nodes;
    yarn_bvh_recur(g, g->nodes[node].fg, i0, pivot + 1, depth + 1);
    g->nodes[node].fd = g->n_nodes;
    yarn_bvh_recur(g, g->nodes[node].fd, pivot + 1, i1, depth + 1);
}
/* cyls[i]->intersection (Geometry.h:740-766): the segment's own Object is default-constructed, so queryMaterial answers with its
 * no-texture defaults (white diffuse, Geometry.h:404-441) and flip_normals is false whatever the Yarns object's flags say */
static int yarn_cyl_hit(const object* g, int i, vec o, vec d, vec* P, float* t, matvals* mat) {
    vec ax = g->yd[i];
    vec X = vsub(d, vscale(vdot(d, ax), ax));
    vec oa = vsub(o, g->yA[i]);
    vec Y = vsub(oa, vscale(vdot(oa, ax), ax));
    float a = vnorm2(X);
    float b = 2 * vdot(X, Y);
    float c = vnorm2(Y) - g->yR[i] * g->yR[i];
    float delta = b * b - 4 * a * c;
    if (delta < 0) return 0;
    float sdelta = sqrtf(delta);
    float t2 = (-b + sdelta) / (2 * a);
    if (t2 < 0) return 0;
    float t1 = (-b - sdelta) / (2 * a);
    if (t1 > 0) *t = t1; else *t = t2;
    *P = vadd(o, vscale(*t, d));
    float dP = vdot(vsub(*P, g->yA[i]), ax);
    if (dP < 0 || dP > g->ylen[i]) return 0;
    vec proj = vadd(g->yA[i], vscale(dP, ax));
    mat->Kd = V(1, 1, 1); mat->Ks = V(0, 0, 0); mat->Ksub = V(0, 0, 0); mat->Ne = V(1, 1, 1); mat->transp = 0; mat->refr_index = 1.3f; mat->Ke = V(0, 0, 0);
    mat->shadingN = vsub(*P, proj);
    return 1;
}
/* Yarns::intersection (TriangleMesh.cpp:1652-1737); intersection_shadow is the same call (TriangleMesh.h:293-298) */
static int yarn_hit(const object* g, vec o, vec d, vec* P, float* t, matvals* mat, float cur_best_t, int* tri_id) {
    *t = cur_best_t;
    int has = 0, best = -1;
    float tl, tr_, lt;
    vec lp;
    invray r; r.o = o; r.id = V(1.f / d.x, 1.f / d.y, 1.f / d.z);
    char s[3] = {(char)(r.id.x >= 0 ? 1 : 0), (char)(r.id.y >= 0 ? 1 : 0), (char)(r.id.z >= 0 ? 1 : 0)};
    if (!box_invd(&g->bvh_bbox, &r, s, &tl)) return 0;
    if (tl > cur_best_t) return 0;
    int l[50]; float tn[50]; int top = -1;
    l[++top] = 0; tn[top] = tl;
    while (top >= 0) {
        if (tn[top] > *t) { top--; continue; }
        int cur = l[top--];
        int fg = g->nodes[cur].fg, fd = g->nodes[cur].fd;
        if (!g->nodes[cur].isleaf) {
            int gl = box_invd_x(&g->nodes[fg].bb, &r, s, &tl, s[0] == 1) && tl < *t;
            int gr = box_invd_x(&g->nodes[fd].bb, &r, s, &tr_, s[0] == 1) && tr_ < *t;
            if (gl && gr) {
                if (tl < tr_) { l[++top] = fd; tn[top] = tr_; l[++top] = fg; tn[top] = tl; }
                else { l[++top] = fg; tn[top] = tl; l[++top] = fd; tn[top] = tr_; }
            } else {
                if (gl) { l[++top] = fg; tn[top] = tl; }
                if (gr) { l[++top] = fd; tn[top] = tr_; }
            }
        } else {
            for (int i = fg; i < fd; i++)
                if (yarn_cyl_hit(g, i, o, d, &lp, &lt, mat) && lt < *t) { has = 1; best = i; *t = lt; }
        }
    }
    if (has) {
        *tri_id = best;
        yarn_cyl_hit(g, best, o, d, &lp, &lt, mat);
        *P = lp;
    }
    return has;
}

/* Scene::intersection (Geometry.cpp:589-688) */
static int scene_hit(const struct ptb_ctx* c, vec o, vec d, vec* P, int* id, float* min_t, matvals* mat, int* tri_id, unsigned long long* counter) {
    int has = 0;
    *min_t = INFINITY; /* 1E99 as float */
    if (counter) counter[0]++;
    vec lp; matvals lm = matvals_default(); float t;
    for (int i = 0; i < c->n_objs; i++) {
        const object* ob = c->objs[i];
        vec dl = xf_dir(ob->inv, d), ol = xf_point(ob->inv, o);
        int h;
        if (ob->type == T_MESH) h = mesh_hit(ob, ol, dl, &lp, &t, &lm, *min_t, tri_id, 0, 0);
        else if (ob->type == T_SPHERE) { h = sphere_hit(ob, ol, dl, &lp, &t, &lm, 0); if (h) *tri_id = -1; }
        else if (ob->type == T_CYLINDER) { h = cylinder_hit(ob, ol, dl, &lp, &t, &lm); if (h) *tri_id = -1; }
        else if (ob->type == T_POINTSET) h = pts_hit(ob, ol, dl, &lp, &t, &lm, *min_t, tri_id, 0, 0);
        else if (ob->type == T_YARNS) h = yarn_hit(ob, ol, dl, &lp, &t, &lm, *min_t, tri_id);
        else { h = plane_hit(ob, ol, dl, &lp, &t, &lm, 0); if (h) *tri_id = -1; }
        if (h && t < *min_t) { has = 1; *min_t = t; *P = lp; *id = i; *mat = lm; }
    }
    if (has) { *P = xf_point(c->objs[*id]->trans, *P); mat->shadingN = xf_rot(c->objs[*id]->rotm, mat->shadingN); }
    mat->shadingN = vfast_normalize(mat->shadingN);
    return has;
}
/* Scene::intersection_shadow (Geometry.cpp:691-744) */
static int scene_shadow(const struct ptb_ctx* c, vec o, vec d, float dist_light, unsigned long long* counter) {
    float min_t = INFINITY;
    if (counter) counter[1]++;
    for (int i = 0; i < c->n_objs; i++) {
        const object* ob = c->objs[i];
        if (ob->ghost) continue;                                         /* avoid_ghosts == true from getColor (Raytracer.cpp:513, Geometry.cpp:722) */
        vec dl = xf_dir(ob->inv, d), ol = xf_point(ob->inv, o);
        float t; int h, tid; vec P; matvals m;
        if (ob->type == T_MESH) h = mesh_hit(ob, ol, dl, &P, &t, &m, min_t, &tid, 1, dist_light);
        else if (ob->type == T_SPHERE) h = sphere_hit(ob, ol, dl, &P, &t, &m, 1);
        else if (ob->type == T_CYLINDER) { m = matvals_default(); h = cylinder_hit(ob, ol, dl, &P, &t, &m); }
        else if (ob->type == T_POINTSET) h = pts_hit(ob, ol, dl, &P, &t, &m, min_t, &tid, 1, dist_light);
        else if (ob->type == T_YARNS) { m = matvals_default(); h = yarn_hit(ob, ol, dl, &P, &t, &m, min_t, &tid); }
        else h = plane_hit(ob, ol, dl, &P, &t, &m, 1);
        if (h && t < dist_light * 0.999) return 1;
    }
    return 0;
}

/* Scene::get_random_intersection (Geometry.cpp:339-472) restricted to object `id`, a TriMesh (the only kind whose
 * reservoir_sampling_intersection the subsurface branch can use: Sphere's returns true without a point, Geometry.h:994-1012) */
static int scene_random_hit(const struct ptb_ctx* c, vec o, vec d, vec* P, int id, float* min_t, matvals* mat, int* tri_id, float tmin, float tmax, pcg* e) {
    const object* ob = c->objs[id];
    *min_t = INFINITY;
    int nb = 0;
    vec dl = xf_dir(ob->inv, d), ol = xf_point(ob->inv, o);
    int has = mesh_reservoir(ob, ol, dl, P, min_t, mat, tri_id, &nb, tmin, tmax, e);
    if (has) { *P = xf_point(ob->trans, *P); mat->shadingN = xf_rot(ob->rotm, mat->shadingN); }
    mat->shadingN = vfast_normalize(mat->shadingN);
    return has;
}

/* Camera::generateDirection (Vector.h:792-825), non-lenticular */
static void camera_ray(const struct ptb_ctx* c, float init_t, int i, int j, float dxs, float dys, float dxa, float dya, int W, int H, vec* ro, vec* rd) {
    float k = W / (2 * tanf(c->fov / 2));
    vec right = vcross(c->cam_dir, c->cam_up);
    vec dv = V((float)(j - W / 2 + 0.5 + dxs), (float)(i - H / 2 + 0.5 + dys), k);
    dv = vnormalize(dv);
    dv = vadd(vadd(vscale(dv.x, right), vscale(dv.y, c->cam_up)), vscale(dv.z, c->cam_dir));
    vec dest = vadd(c->cam_pos, vscale(c->focus_distance / fabsf(vdot(dv, c->cam_dir)), dv));
    vec no = vadd(vadd(c->cam_pos, vscale(dxa, right)), vscale(dya, c->cam_up));
    vec nd = vnormalize(vsub(dest, no));
    *ro = vadd(no, vdiv(vscale(init_t, nd), vdot(nd, c->cam_dir)));
    *rd = nd;
}

/* ---- per-contribution engines (oracle/build_ref.py patch 7) ---------------------------------------- */
typedef struct { vec w, o, d; int depth, show_lights, hadSS, showenv; pcg rng; } contrib; /* Contrib, Raytracer.h:15-23 (+ rng) */
#define RING 200                                                                        /* sizeCircArray, Raytracer.h:114 */
static pcg pcg_fork(const pcg* e, uint64_t tag) { pcg t = *e; uint64_t a = pcg_next(&t); uint64_t b = pcg_next(&t); return pcg_seed2((a << 32) | b, tag); }
static contrib mk_contrib(vec w, vec o, vec d, int depth, int show_lights, int hadSS, int showenv) {
    contrib k; k.w = w; k.o = o; k.d = d; k.depth = depth; k.show_lights = show_lights; k.hadSS = hadSS; k.showenv = showenv; k.rng.state = 0; k.rng.inc = 1; return k;
}

/* int_exponential (Raytracer.cpp:20-38) */
static float int_exponential(float y0, float ysol, float beta, float s, float uy) {
    float result;
    if (fabsf(uy * beta) < 0.0001) result = expf(-beta * (y0 - ysol)) * (s);
    else result = (expf(-beta * (y0 - ysol)) - expf(-beta * (y0 + s * uy - ysol))) / (uy * beta);
    return result;
}
/* random_uniform_sphere<float> (Vector.h:604-615) */
static vec random_uniform_sphere(pcg* e) {
    float r1 = pcg_unif(e), r2 = pcg_unif(e);
    float twopi = (float)(2. * M_PI);
    return V(2.f * cosf(twopi * r1) * sqrtf(r2 * (1 - r2)), 2.f * sinf(twopi * r1) * sqrtf(r2 * (1 - r2)), 1.f - 2.f * r2);
}
/* Raytracer::fogContribution (Raytracer.cpp:40-192).  Returns 1 and fills *out when the in-scattered contribution exists. */
static int fog_contribution(const struct ptb_ctx* c, vec ro, vec rd, vec sampleLightPos, float t, vec curWeight, int nbrebonds, int showLight, int hadSS,
                            contrib* out, float* attenuationFactor, pcg* e, unsigned long long* counter) {
    if (vnorm2(curWeight) < 1E-12) return 0;
    const float p_uniform = 0.5f;
    const int is_uniform_fog = (c->fog.type == 0);
    const float alpha = c->fog.absorption, sigmaT = c->fog.absorption_decay;
    const float groundLevel = c->objs[2]->tr_at.y;                         /* objects[2]->get_translation(r.time)[1], 54 */
    float int_ext;
    if (is_uniform_fog) int_ext = (float)(alpha * t * 0.05);
    else int_ext = alpha * int_exponential(ro.y, groundLevel, sigmaT, t, rd.y);
    float T = expf(-int_ext);
    float proba_t, random_t;
    float clamped_t = fminr(1000.f, t);
    float a = vdot(vsub(sampleLightPos, ro), rd);
    if (a > 0) {                                                           /* equi-angular sampling, 71-84 */
        vec projP = vadd(ro, vscale(a, rd));
        float D = sqrtf(vnorm2(vsub(sampleLightPos, projP)));
        float thetaA = -atan2f(a, D);
        float b = t - a;
        float thetaB = atan2f(b, D);
        float x = pcg_unif(e);
        random_t = D * tanf((1 - x) * thetaA + x * thetaB);
        proba_t = D / ((thetaB - thetaA) * (D * D + random_t * random_t));
        random_t += a;
    } else {                                                               /* truncated exponential, 90-99 */
        float alpha2 = 5.f / clamped_t;
        do { random_t = -logf(pcg_unif(e)) / alpha2; } while (random_t > clamped_t);
        float normalization = 1.f / alpha2 * (1.f - expf(-alpha2 * clamped_t));
        proba_t = expf(-alpha2 * random_t) / normalization;
    }
    float int_ext_partielle;
    if (is_uniform_fog) int_ext_partielle = (float)(alpha * random_t * 0.05);
    else int_ext_partielle = alpha * int_exponential(ro.y, groundLevel, sigmaT, random_t, rd.y);
    vec random_P = vadd(ro, vscale(random_t, rd));
    if (random_P.y < groundLevel) return 0;
    vec random_dir, point_aleatoire = V(0, 0, 0);
    vec axeOP = vnormalize(vsub(random_P, c->centerLight));
    int is_uniform;
    if (pcg_unif(e) < p_uniform) { random_dir = random_uniform_sphere(e); is_uniform = 1; }
    else {
        float r1 = pcg_unif(e), r2 = pcg_unif(e);
        vec dir_aleatoire = random_cos(axeOP, r1, r2);
        point_aleatoire = vadd(vscale(c->radiusLight, dir_aleatoire), c->centerLight);
        random_dir = vnormalize(vsub(point_aleatoire, random_P));
        is_uniform = 0;
    }
    float phase_func = 0, k = c->fog.phase_aniso;
    switch (c->fog.phase_type) {                                           /* 134-144 */
    case 0: phase_func = (float)(1. / (4. * M_PI)); break;
    case 1: phase_func = (float)((1 - k * k) / (4. * M_PI * (1 + k * vdot(random_dir, vneg(rd))))); break;
    case 2: { float dd = vdot(random_dir, rd); phase_func = (float)(3 / (16 * M_PI) * (1 + dd * dd)); break; }
    }
    vec interP = V(0, 0, 0); matvals interMat = matvals_default(); int interid = -1, intertri = -1; float intert;
    int interinter = scene_hit(c, random_P, random_dir, &interP, &interid, &intert, &interMat, &intertri, counter);
    vec interN = interMat.shadingN;
    float Vis;
    if (is_uniform) Vis = 1;
    else {
        float d_light2 = vnorm2(vsub(point_aleatoire, random_P));
        if (interinter && intert * intert < d_light2 * 0.99) Vis = 0; else Vis = 1;
    }
    *attenuationFactor = T;
    if (Vis == 0) return 0;
    float pdf_uniform = (float)(1. / (4. * M_PI));
    float J = vdot(interN, vneg(random_dir)) / vnorm2(vsub(interP, random_P));
    float pdf_light = (interinter && interid == 0) ? (float)(vdot(vnormalize(vsub(interP, c->centerLight)), axeOP) / (M_PI * (c->radiusLight * c->radiusLight)) / J) : 0.f;
    float proba_dir = p_uniform * pdf_uniform + (1 - p_uniform) * pdf_light;
    float ext;
    if (is_uniform_fog) ext = (float)(c->fog.density * 0.05);
    else ext = c->fog.density * expf(-c->fog.density_decay * (random_P.y - groundLevel));
    vec newweight = vscale(phase_func * ext * expf(-int_ext_partielle) / (proba_t * proba_dir), curWeight);
    *out = mk_contrib(newweight, random_P, random_dir, nbrebonds - 1, showLight, hadSS, 1);
    return 1;
}

/* Scene::background lookup of getColor (Raytracer.cpp:261-265, 615-619) */
static vec background_at(const struct ptb_ctx* c, int screenI, int screenJ) {
    int i = (int)(screenI / (float)c->H * c->bgH); if (i < 0) i = 0; if (i > c->bgH - 1) i = c->bgH - 1;
    int j = (int)(screenJ / (float)c->W * c->bgW); if (j < 0) j = 0; if (j > c->bgW - 1) j = c->bgW - 1;
    const float* b = c->bg + ((size_t)i * c->bgW + j) * 3;
    return V(b[0], b[1], b[2]);
}

/* Raytracer::getColor (Raytracer.cpp:196-664): the ring of contributions with fog, ghost objects and the background photograph;
 * the subsurface branch (318-406) is restated for TriMesh objects (the only kind it is defined for). */
#define PUSH(k_) do { ring[end] = (k_); end++; if (end >= RING) end = 0; } while (0)
static vec get_color(const struct ptb_ctx* c, vec ro0, vec rd0, int sampleID, int pix, pcg* e, unsigned long long* counter, const vec* samples2d,
                     vec* normalValue, vec* albedoValue) {
    contrib ring[RING];
    int start = 0, end = 1;
    const int has_fog = (c->fog.density > 1E-8);
    const int has_bg = c->bgW > 0 && c->bg != NULL;
    const int screenI = pix / c->W, screenJ = pix % c->W;
    float att = 1.f;                                                     /* attenuationFactor (patch 7b) */
    vec color = V(0, 0, 0);
    ring[0] = mk_contrib(V(1.f, 1.f, 1.f), ro0, rd0, c->nb_bounces, 1, 0, 1);
    ring[0].rng = *e;
    while (start != end) {
        const contrib cur = ring[start];
        *e = cur.rng;
        vec ro = cur.o, rd = cur.d, w = cur.w;
        const int depth = cur.depth, show_lights = cur.show_lights, hadSS = cur.hadSS, show_envmap = cur.showenv;
        start++; if (start >= RING) start = 0;
        if (depth == 0) continue;                                       /* 240 */
        if (vnorm2(w) < 0.01f * 0.01f) continue;                        /* 241 */
        vec P = V(0, 0, 0); matvals mat = matvals_default(); int id = -1, tri = -1; float t = 0;
        int has = scene_hit(c, ro, rd, &P, &id, &t, &mat, &tri, counter);
        vec N = mat.shadingN;
        if (getenv("PTB_DBG")) fprintf(stderr, "P %d %d %d %.4f\n", pix, depth, has ? id : -1, has ? t : 0.f);
        if (has && depth == c->nb_bounces && normalValue) { *normalValue = N; *albedoValue = mat.Kd; }   /* 254-257 */
        if (depth == c->nb_bounces && has_bg && (!has || (has && id == 1))) {                           /* 260-268 */
            color = vadd(color, vmul(w, background_at(c, screenI, screenJ)));
            continue;
        }
        contrib fogc;
        if (has) {
            if (id == 1) {                                              /* 275-301 */
                if (!show_envmap) {
                    if (has_fog && fog_contribution(c, ro, rd, c->centerLight, t, w, depth, show_lights, hadSS, &fogc, &att, e, counter)) { fogc.rng = pcg_fork(e, 1); PUSH(fogc); }
                    continue;
                }
                if (has_fog) {
                    if (fog_contribution(c, ro, rd, c->centerLight, t, w, depth, show_lights, hadSS, &fogc, &att, e, counter)) { fogc.rng = pcg_fork(e, 1); PUSH(fogc); }
                    color = vadd(color, vmul(vscale(c->envmap_intensity, vscale(att, w)), mat.Ke));
                } else color = vadd(color, vmul(vscale(c->envmap_intensity, w), mat.Ke));
                continue;
            }
            if (id == 0) {                                              /* 303-316 */
                float lp = show_lights ? c->lightPower : 0.f;
                if (has_fog) {
                    if (fog_contribution(c, ro, rd, c->centerLight, t, w, depth, show_lights, hadSS, &fogc, &att, e, counter)) { fogc.rng = pcg_fork(e, 1); PUSH(fogc); }
                    color = vadd(color, vmul(vscale(att, w), V(lp, lp, lp)));
                } else color = vadd(color, vmul(w, V(lp, lp, lp)));
                continue;
            }
            const object* ob = c->objs[id];
            /* subsurface scattering (318-406): with probability 0.6 the path leaves the surface at a random nearby point of the same object */
            const int is_subsurface = vnorm2(mat.Ksub) > 1E-8;                                              /* 270 */
            const float subsProba = (hadSS || !is_subsurface) ? 0.f : 0.6f;
            const float inv1MSubsProba = 1.f / (1.f - subsProba);
            vec subsW = V(inv1MSubsProba, inv1MSubsProba, inv1MSubsProba);
            int sub_interaction = 0;
            const vec cur_d = rd;                                        /* currentRay.direction: what fogContribution keeps seeing */
            if (is_subsurface && pcg_unif(e) < subsProba) {
                sub_interaction = 1;
                const float invSubsProba = 1.f / subsProba;
                subsW = V(invSubsProba, invSubsProba, invSubsProba);
                const float sigmasub = 1.5f;
                const float diskR = sqrtf(12.46f) * sigmasub;
                float integ = 1.f - expf(-diskR * diskR / (2.f * sigmasub * sigmasub));
                float randR = sigmasub * sqrtf(-2.f * logf(1.f - pcg_unif(e) * integ));
                float randangle = pcg_unif(e) * 2.f * (float)M_PI;
                float g0 = randR * sinf(randangle), g1 = randR * cosf(randangle), g2 = randR;
                float gaussval = (float)((1. / (sigmasub * sigmasub * 2.f * (float)M_PI)) * expf(-(g2 * g2) / (2.f * sigmasub * sigmasub)));
                float pdfgauss = gaussval / integ;
                vec Tg = get_tangent(N), Tg2 = vcross(N, Tg);
                vec PtaboveP = vadd(vadd(vadd(P, vscale(g0, Tg)), vscale(g1, Tg2)), vscale(diskR, N));
                float r1 = pcg_unif(e);
                vec axis = vneg(N);
                float tmax, wAxis;
                float h = sqrtf(diskR * diskR - g2 * g2);
                vec subsOrigin = vadd(PtaboveP, vscale(diskR - h, vneg(N)));
                if (r1 < 0.5f) { wAxis = 0.5f; tmax = 2.f * h; }
                else {
                    wAxis = 0.25f; tmax = 2.f * g2;
                    axis = r1 < 0.75f ? Tg : Tg2;
                    float r2 = pcg_unif(e);
                    if (r2 < 0.5f) subsOrigin = vsub(subsOrigin, vscale(h, N));
                }
                matvals subsmat = matvals_default(); int substri = -1; float subst; vec localP2 = V(0, 0, 0);
                if (ob->type == T_MESH && scene_random_hit(c, subsOrigin, axis, &localP2, id, &subst, &subsmat, &substri, 0, tmax, e)) {
                    float chris = (float)exp(-vnorm2(vsub(P, localP2)) / (2. * sigmasub * sigmasub));
                    float a0 = vdot(subsmat.shadingN, N), a1 = vdot(subsmat.shadingN, Tg), a2 = vdot(subsmat.shadingN, Tg2);
                    float sumpdfs = (float)((0.5 * a0) * (0.5 * a0) + (0.25 * a1) * (0.25 * a1) + (0.25 * a2) * (0.25 * a2));
                    float pdfdisk = wAxis * fabsf(vdot(axis, subsmat.shadingN)) / sumpdfs;
                    subsW = vscale(pdfdisk / fmaxr(pdfgauss, 0.05f) * chris, subsW);
                    rd = vnormalize(vsub(localP2, P));                   /* rayDirection */
                    P = vadd(localP2, vscale(0.005f, subsmat.shadingN));
                    subsW = vscale(r1 < 0.5f ? 2.f : 4.f, subsW);
                    subsW = vmul(subsW, vdiv(mat.Ksub, (float)M_PI));
                    mat = subsmat;
                    N = mat.shadingN;
                }
            }
            color = vadd(color, vscale(c->envmap_intensity, vmul(w, mat.Ke)));                              /* 411 */
            if (ob->miroir) {                                            /* 413-436 */
                vec nd = vreflect(rd, N), no = vadd(P, vscale(0.001f, N));
                contrib k;
                if (has_fog) {
                    if (fog_contribution(c, ro, cur_d, c->centerLight, t, w, depth, show_lights, hadSS, &fogc, &att, e, counter)) { fogc.rng = pcg_fork(e, 1); PUSH(fogc); }
                    k = mk_contrib(vscale(att, w), no, nd, depth - 1, show_lights, hadSS, 1);
                } else k = mk_contrib(w, no, nd, depth - 1, show_lights, hadSS, 1);
                k.rng = *e; PUSH(k);
                continue;
            }
            if (mat.transp) {                                            /* 438-489 */
                float n1 = 1.f, n2 = mat.refr_index; vec Nt = N; int entering = 1;
                if (vdot(rd, N) > 0) { n1 = mat.refr_index; n2 = 1; Nt = vneg(N); entering = 0; }
                float c0 = vdot(Nt, rd);
                float radical = 1.f - (n1 / n2) * (n1 / n2) * (1.f - c0 * c0);
                vec no, nd;
                if (radical > 0) {
                    vec refr = vsub(vscale(n1 / n2, vsub(rd, vscale(vdot(rd, Nt), Nt))), vscale(sqrtf(radical), Nt));
                    float r0 = (n1 - n2) / (n1 + n2), R0 = r0 * r0, R;
                    if (entering) R = R0 + (1 - R0) * powf(1.f + vdot(rd, N), 5.f);
                    else R = R0 + (1 - R0) * powf(1.f - vdot(refr, N), 5.f);
                    if (pcg_unif(e) < R) { no = vadd(P, vscale(0.001f, Nt)); nd = vreflect(rd, N); }
                    else { no = vsub(P, vscale(0.001f, Nt)); nd = refr; }
                } else { no = vadd(P, vscale(0.001f, Nt)); nd = vreflect(rd, N); }
                contrib k;
                if (has_fog) {
                    if (fog_contribution(c, ro, cur_d, c->centerLight, t, w, depth, show_lights, hadSS, &fogc, &att, e, counter)) { fogc.rng = pcg_fork(e, 1); PUSH(fogc); }
                    k = mk_contrib(vscale(att, w), no, nd, depth - 1, show_lights, hadSS, 1);
                } else k = mk_contrib(w, no, nd, depth - 1, show_lights, hadSS, 1);
                k.rng = *e; PUSH(k);
                continue;
            }
            /* opaque: next-event estimation (494-566) */
            vec axeOP = vfast_normalize(vsub(P, c->centerLight));
            float l1 = pcg_unif(e), l2 = pcg_unif(e);
            vec dirl = random_cos(axeOP, l1, l2);
            vec xl = vadd(vscale(c->radiusLight, dirl), c->centerLight);
            vec wi = vfast_normalize(vsub(xl, P));
            float d2 = vnorm2(vsub(xl, P));
            int shadowed;
            if (vdot(mat.shadingN, wi) < 0) shadowed = 1;
            else shadowed = scene_shadow(c, vadd(P, vscale(0.01f, wi)), wi, sqrtf(d2) - 0.01f, counter);
            vec contribution = V(0, 0, 0);
            vec fog_o = ro, fog_d = cur_d;                               /* `currentRay` as fogContribution sees it below */
            if (!shadowed) {
                if (ob->ghost) {                                         /* 522-537: straight through, same depth */
                    vec offset = vdot(N, rd) > 0 ? N : vneg(N);
                    fog_o = vadd(vadd(P, vscale(0.001f, rd)), vscale(0.001f, offset)); fog_d = rd;
                    contrib k = mk_contrib(w, fog_o, rd, depth, show_lights, hadSS, show_envmap);
                    k.rng = pcg_fork(e, 2); PUSH(k);
                }
                vec fr;
                if (sub_interaction) fr = vdiv(mat.Ksub, (float)M_PI);
                else fr = ob->brdf == PTB_BRDF_MERL ? merl_eval(ob->merl, wi, vneg(rd), N) : phong_eval(&mat, wi, vneg(rd), N);
                float J = vdot(dirl, vneg(wi)) / d2;
                float proba = (float)(vdot(axeOP, dirl) / (M_PI * c->radiusLight * c->radiusLight));
                if (!ob->ghost && proba > 0.f) contribution = vadd(contribution, vmul(vscale(c->lightPower * fmaxr(0.f, vdot(N, wi)) * J / proba, subsW), fr));
            }
            if (has_fog) {                                               /* 556-566 */
                if (fog_contribution(c, fog_o, fog_d, xl, t, w, depth, show_lights, hadSS, &fogc, &att, e, counter)) { fogc.rng = pcg_fork(e, 1); PUSH(fogc); }
                color = vadd(color, vmul(vscale(att, w), contribution));
            } else color = vadd(color, vmul(w, contribution));
            /* continuation (570-632) */
            float tmp;
            float r1 = modff(c->randomPerPixel[pix].x + samples2d[sampleID].x, &tmp);
            float r2 = modff(c->randomPerPixel[pix].y + samples2d[sampleID].y, &tmp);
            float pdf; vec dir; int diffuse = 0;
            if (sub_interaction) { dir = random_cos(mat.shadingN, r1, r2); pdf = vdot(N, dir) / (float)M_PI; diffuse = 1; }   /* 598-601 */
            else if (ob->brdf == PTB_BRDF_MERL) { dir = random_cos(N, r1, r2); pdf = (float)(vdot(N, dir) / (M_PI)); }
            else dir = phong_sample(&mat, vneg(rd), N, &pdf, r1, r2, e, &diffuse);
            if (vdot(dir, N) < 0 || vdot(dir, vreflect(rd, N)) < 0 || pdf <= 0) continue;
            vec fi;
            if (sub_interaction) fi = vdiv(mat.Ksub, (float)M_PI);
            else fi = ob->brdf == PTB_BRDF_MERL ? merl_eval(ob->merl, dir, vneg(rd), N) : phong_eval(&mat, dir, vneg(rd), N);
            vec nw = vscale((vdot(N, dir) / pdf), vmul(vmul(w, subsW), fi));
            if (ob->ghost && has_bg) nw = vmul(nw, vdiv(background_at(c, screenI, screenJ), 196964.699f));  /* 614-621 */
            contrib k = mk_contrib(has_fog ? vscale(att, nw) : nw, vadd(P, vscale(0.01f, dir)), dir, depth - 1, 0, sub_interaction ? 1 : hadSS,
                                   (show_envmap && shadowed && diffuse) || !ob->ghost);
            k.rng = *e; PUSH(k);
        }
        if (c->fog.density == 0) continue;                               /* 654-655 */
        if (!has) break;                                                 /* 657 */
    }
    return color;
}
#undef PUSH

static float sat(const float* s, int w, int i0, int i1, int j0, int j1) { /* Raytracer.cpp:1276-1291 */
    float t1 = 0, t2 = 0, t3 = 0;
    if (i0 > 0) t1 = s[(i0 - 1) * w + j1];
    if (j0 > 0) t2 = s[i1 * w + j0 - 1];
    if (i0 > 0 && j0 > 0) t3 = s[(i0 - 1) * w + j0 - 1];
    return s[i1 * w + j1] - t1 - t2 + t3;
}

/* Raytracer::prepare_render (Raytracer.cpp:1321-1391) */
static void prepare_render(struct ptb_ctx* c) {
    if (c->rpp_n != c->W * c->H) {
        free(c->randomPerPixel);
        c->rpp_n = c->W * c->H;
        c->randomPerPixel = (vec*)malloc(sizeof(vec) * (size_t)c->rpp_n);
        pcg e0 = pcg_seed1(0);
        for (int i = 0; i < c->rpp_n; i++) { float a = pcg_unif(&e0); float b = pcg_unif(&e0); c->randomPerPixel[i] = V(a, b, 0); }
    }
    float sg = c->sigma_filter;
    c->filter_size = (int)ceilf(sg * 2);
    c->filter_total_width = 2 * c->filter_size + 1;
    int fs = c->filter_size, ftw = c->filter_total_width;
    for (int i = -fs; i <= fs; i++)
        for (int j = -fs; j <= fs; j++) {
            float integ = 0;
            for (int i2 = -fs; i2 <= i; i2++)
                for (int j2 = -fs; j2 <= j; j2++) { float w = (float)(fast_exp(-(i2 * i2 + j2 * j2) / (2. * sg * sg)) / (sg * sg * 2. * M_PI)); integ += w; }
            c->filter_integral[(i + fs) * ftw + (j + fs)] = integ;
        }
    for (int i = 0; i < c->n_objs; i++) build_matrix(c->objs[i], (float)c->current_frame);
    const object* L = c->objs[0];
    c->centerLight = xf_point(L->trans, L->O);
    c->radiusLight = L->scale_at * L->R;
    c->lightPower = c->intensite_lumiere / (L->scale_at * L->scale_at);
}

/* ---- ABI -------------------------------------------------------------------------------------------- */
const char* ptb_version(void) { return "ptb-oracle-port (plain C restatement)"; }
const char* ptb_last_error(const ptb_ctx* c) { return c ? c->err : g_err; }
int ptb_create(int device_id, ptb_ctx** out) {
    (void)device_id;
    if (!out) return PTB_ERR_INVALID;
    ptb_ctx* c = (ptb_ctx*)calloc(1, sizeof(ptb_ctx));
    c->envmap_intensity = 1; c->sigma_filter = 0.5f; c->gamma = 2.2f; c->nb_bounces = 5; c->W = c->H = 64; c->nrays = 1;
    *out = c;
    return PTB_OK;
}
static void free_object(object* o) {
    for (int s = 0; s < S_COUNT; s++) { for (int i = 0; i < o->slots[s].n; i++) free(o->slots[s].t[i].values); free(o->slots[s].t); }
    for (int k = 0; k < 3; k++) { free(o->kframe[k]); free(o->kval[k]); }
    free(o->vertices); free(o->normals); free(o->uvs); free(o->indices); free(o->soup); free(o->tangent_soup); free(o->permuted); free(o->nodes);
    free(o->pt_pos); free(o->pt_nrm); free(o->pt_col); free(o->pt_rad); free(o->pt_perm);
    free(o->yA); free(o->yB); free(o->yd); free(o->yR); free(o->ylen); free(o->y_perm);
    free(o);
}
static void prog_free(ptb_ctx* c);
void ptb_destroy(ptb_ctx* c) {
    if (c) prog_free(c);
    if (!c) return;
    for (int i = 0; i < c->n_objs; i++) free_object(c->objs[i]);
    free(c->objs);
    for (int i = 0; i < c->n_merl; i++) free(c->merl[i]);
    free(c->merl); free(c->env); free(c->bg); free(c->randomPerPixel); free(c);
}
static object* new_object(ptb_ctx* c, int type, const ptb_xform* xf, int flags, vec default_rc) {
    object* o = (object*)calloc(1, sizeof(object));
    o->type = type; o->miroir = (flags & PTB_OBJ_MIRROR) != 0; o->flip_normals = (flags & PTB_OBJ_FLIP_NORMALS) != 0;
    o->interp_normals = (flags & PTB_OBJ_FLAT_NORMALS) == 0; o->ghost = (flags & PTB_OBJ_GHOST) != 0;
    o->scale = 1; o->rot[0] = o->rot[4] = o->rot[8] = 1; o->rc = default_rc; o->tr = V(0, 0, 0);
    if (xf) {
        o->scale = xf->scale; memcpy(o->rot, xf->rotation, sizeof(o->rot)); o->tr = V(xf->translation[0], xf->translation[1], xf->translation[2]);
        if (!(xf->rotation_center[0] != xf->rotation_center[0])) o->rc = V(xf->rotation_center[0], xf->rotation_center[1], xf->rotation_center[2]);
    }
    c->objs = (object**)realloc(c->objs, sizeof(object*) * (size_t)(c->n_objs + 1));
    c->objs[c->n_objs++] = o;
    return o;
}
int ptb_add_sphere(ptb_ctx* c, const float O[3], float R, const ptb_xform* xf, int flags, int* out_id) {
    if (!c || !O) return PTB_ERR_INVALID;
    object* o = new_object(c, T_SPHERE, xf, flags, V(O[0], O[1], O[2]));
    o->O = V(O[0], O[1], O[2]); o->R = R; o->R2 = R * R;
    if (out_id) *out_id = c->n_objs - 1;
    return PTB_OK;
}
int ptb_add_pointset(ptb_ctx* c, const ptb_pointset* p, const ptb_xform* xf, int flags, int* out_id) {
    if (!c || !p || !p->points || !p->normals || !p->radii || p->n <= 0) return PTB_ERR_INVALID;
    int n = p->n;
    vec rc = V(0, 0, 0);                                                   /* init: rotation_center = mean of the points (PointSet.h:113-121) */
    for (int i = 0; i < n; i++) rc = vadd(rc, V(p->points[3 * i], p->points[3 * i + 1], p->points[3 * i + 2]));
    rc = vdiv(rc, (float)n);
    object* g = new_object(c, T_POINTSET, xf, flags, rc);
    g->display_edges = (flags & PTB_OBJ_DISPLAY_EDGES) != 0;
    g->np = n;
    g->pt_pos = (vec*)malloc(sizeof(vec) * (size_t)n); g->pt_nrm = (vec*)malloc(sizeof(vec) * (size_t)n);
    g->pt_col = p->colors ? (vec*)malloc(sizeof(vec) * (size_t)n) : NULL;
    g->pt_rad = (double*)malloc(sizeof(double) * (size_t)n); g->pt_perm = (int*)malloc(sizeof(int) * (size_t)n);
    for (int i = 0; i < n; i++) {
        g->pt_pos[i] = V(p->points[3 * i], p->points[3 * i + 1], p->points[3 * i + 2]);
        g->pt_nrm[i] = V(p->normals[3 * i], p->normals[3 * i + 1], p->normals[3 * i + 2]);
        if (g->pt_col) g->pt_col[i] = V(p->colors[3 * i], p->colors[3 * i + 1], p->colors[3 * i + 2]);
        g->pt_rad[i] = p->radii[i]; g->pt_perm[i] = i;
    }
    g->cap_nodes = 64; g->nodes = (bnode*)malloc(sizeof(bnode) * (size_t)g->cap_nodes); g->n_nodes = 0; g->bvh_depth = 0;
    g->bvh_bbox = pts_bbox(g, 0, n);                                       /* build_bvh, 28-32 */
    pts_bvh_recur(g, 0, 0, n, 0);
    if (out_id) *out_id = c->n_objs - 1;
    return PTB_OK;
}
/* `new Yarns(file)` (TriangleMesh.h:268-290) with the segments passed in memory: cyls[i] = Cylinder(A, B, R), then build_bvh */
int ptb_add_yarns(ptb_ctx* c, const ptb_yarns* y, const ptb_xform* xf, int flags, int* out_id) {
    if (!c || !y || !y->A || !y->B || !y->R || y->n <= 0) return PTB_ERR_INVALID;
    int n = y->n;
    object* g = new_object(c, T_YARNS, xf, flags, V(0, 0, 0));
    g->ny = n;
    g->yA = (vec*)malloc(sizeof(vec) * (size_t)n); g->yB = (vec*)malloc(sizeof(vec) * (size_t)n); g->yd = (vec*)malloc(sizeof(vec) * (size_t)n);
    g->yR = (float*)malloc(sizeof(float) * (size_t)n); g->ylen = (float*)malloc(sizeof(float) * (size_t)n); g->y_perm = (int*)malloc(sizeof(int) * (size_t)n);
    for (int i = 0; i < n; i++) {
        g->yA[i] = V(y->A[3 * i], y->A[3 * i + 1], y->A[3 * i + 2]); g->yB[i] = V(y->B[3 * i], y->B[3 * i + 1], y->B[3 * i + 2]); g->yR[i] = y->R[i];
        g->yd[i] = vnormalize(vsub(g->yB[i], g->yA[i]));                       /* Cylinder(A, B, R), Geometry.h:734-738 */
        g->ylen[i] = sqrtf(vnorm2(vsub(g->yB[i], g->yA[i])));
        g->y_perm[i] = i;
    }
    g->cap_nodes = 64; g->nodes = (bnode*)malloc(sizeof(bnode) * (size_t)g->cap_nodes); g->n_nodes = 0; g->bvh_depth = 0;
    g->bvh_bbox = yarn_bbox(g, 0, n);                                      /* build_bvh, 1550-1554 */
    yarn_bvh_recur(g, 0, 0, n, 0);
    if (out_id) *out_id = c->n_objs - 1;
    return PTB_OK;
}
int ptb_add_cylinder(ptb_ctx* c, const float A[3], const float B[3], float R, const ptb_xform* xf, int flags, int* out_id) {
    if (!c || !A || !B) return PTB_ERR_INVALID;
    object* o = new_object(c, T_CYLINDER, xf, flags, V(0, 0, 0));
    o->A = V(A[0], A[1], A[2]); o->cylB = V(B[0], B[1], B[2]); o->R = R;
    o->cyld = vnormalize(vsub(o->cylB, o->A));
    o->cyllen = sqrtf(vnorm2(vsub(o->cylB, o->A)));
    if (out_id) *out_id = c->n_objs - 1;
    return PTB_OK;
}
int ptb_add_plane(ptb_ctx* c, const float A[3], const float N[3], const ptb_xform* xf, int flags, int* out_id) {
    if (!c || !A || !N) return PTB_ERR_INVALID;
    object* o = new_object(c, T_PLANE, xf, flags, V(0, 0, 0));
    o->A = V(A[0], A[1], A[2]); o->vecN = V(N[0], N[1], N[2]);
    if (out_id) *out_id = c->n_objs - 1;
    return PTB_OK;
}
/* TriMesh::init (TriangleMesh.cpp:718-841), in-memory route */
int ptb_add_mesh(ptb_ctx* c, const ptb_mesh* m, const ptb_xform* xf, int flags, int* out_id) {
    if (!c || !m || !m->vertices || !m->tri || m->n_tri <= 0) return PTB_ERR_INVALID;
    struct timespec t0, t1; clock_gettime(CLOCK_MONOTONIC, &t0);
    object* g = new_object(c, T_MESH, NULL, flags, V(0, 0, 0));
    g->nv = m->n_vertices; g->nn = m->normals ? m->n_normals : 0; g->nuv = m->uvs ? m->n_uvs : 0; g->nt = m->n_tri;
    g->vertices = (vec*)malloc(sizeof(vec) * (size_t)g->nv);
    for (int i = 0; i < g->nv; i++) g->vertices[i] = V(-m->vertices[3 * i + 2], m->vertices[3 * i + 1], m->vertices[3 * i]);   /* 742-746 */
    g->normals = (vec*)malloc(sizeof(vec) * (size_t)(g->nn + 1));
    for (int i = 0; i < g->nn; i++) g->normals[i] = V(-m->normals[3 * i + 2], m->normals[3 * i + 1], m->normals[3 * i]);      /* 747-750 */
    g->uvs = (float*)malloc(sizeof(float) * 2 * (size_t)(g->nuv + 1));
    if (g->nuv) memcpy(g->uvs, m->uvs, sizeof(float) * 2 * (size_t)g->nuv);
    g->indices = (tindex*)malloc(sizeof(tindex) * (size_t)g->nt);
    g->permuted = (int*)malloc(sizeof(int) * (size_t)g->nt);
    for (int i = 0; i < g->nt; i++) {
        const int32_t* t = m->tri + 10 * (size_t)i;
        for (int k = 0; k < 3; k++) { g->indices[i].vtx[k] = t[k]; g->indices[i].uv[k] = t[3 + k]; g->indices[i].n[k] = t[6 + k]; }
        g->indices[i].group = t[9];
        g->permuted[i] = i;
    }
    box bb = {V(1E9f, 1E9f, 1E9f), V(-1E9f, -1E9f, -1E9f)};
    for (int i = 0; i < g->nv; i++) {
        bb.lo = V(fminr(bb.lo.x, g->vertices[i].x), fminr(bb.lo.y, g->vertices[i].y), fminr(bb.lo.z, g->vertices[i].z));
        bb.hi = V(fmaxr(bb.hi.x, g->vertices[i].x), fmaxr(bb.hi.y, g->vertices[i].y), fmaxr(bb.hi.z, g->vertices[i].z));
    }
    if (m->center) {                                                                                                          /* 760-770 */
        float s = fmaxr(bb.hi.x - bb.lo.x, fmaxr(bb.hi.y - bb.lo.y, bb.hi.z - bb.lo.z));
        vec cc = vscale(0.5f, vadd(bb.lo, bb.hi));
        for (int i = 0; i < g->nv; i++) {
            g->vertices[i].x = (g->vertices[i].x - cc.x) / s * m->scaling + m->offset[0];
            g->vertices[i].y = (g->vertices[i].y - cc.y) / s * m->scaling + m->offset[1];
            g->vertices[i].z = (g->vertices[i].z - cc.z) / s * m->scaling + m->offset[2];
        }
    }
    g->bvh_bbox = mesh_bbox(g, 0, g->nt);
    g->cap_nodes = 1024; g->nodes = (bnode*)malloc(sizeof(bnode) * (size_t)g->cap_nodes); g->n_nodes = 0; g->bvh_depth = 0;
    bvh_recur(g, 0, 0, g->nt, 0);                                                                                             /* 807-809 */
    box obb = mesh_bbox(g, 0, g->nt);
    g->soup = (tsoup*)malloc(sizeof(tsoup) * (size_t)g->nt);                                                                  /* 813-829 */
    for (int i = 0; i < g->nt; i++) {
        const tindex* t = &g->indices[i];
        g->soup[i] = soup_make(g->vertices[t->vtx[0]], g->vertices[t->vtx[1]], g->vertices[t->vtx[2]]);
        if (g->nn != 0) for (int k = 0; k < 3; k++) g->soup[i].normals[k] = g->normals[t->n[k]];
        if (g->nuv != 0) for (int k = 0; k < 3; k++) { g->soup[i].uvs[k][0] = g->uvs[2 * t->uv[k]]; g->soup[i].uvs[k][1] = g->uvs[2 * t->uv[k] + 1]; }
    }
    g->rc = vscale(0.5f, vadd(obb.lo, obb.hi));                                                                               /* 831-835 */
    setup_tangents(g);
    if (xf) {
        g->scale = xf->scale; memcpy(g->rot, xf->rotation, sizeof(g->rot)); g->tr = V(xf->translation[0], xf->translation[1], xf->translation[2]);
        if (!(xf->rotation_center[0] != xf->rotation_center[0])) g->rc = V(xf->rotation_center[0], xf->rotation_center[1], xf->rotation_center[2]);
    }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    c->ms_build += (t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6;
    c->n_tri += g->nt;
    if (out_id) *out_id = c->n_objs - 1;
    return PTB_OK;
}
static void put_slot(slotv* s, int group, const ptb_tex* t) {
    if (s->n <= group) {
        s->t = (tex*)realloc(s->t, sizeof(tex) * (size_t)(group + 1));
        for (int i = s->n; i <= group; i++) { tex d; d.mult[0] = d.mult[1] = d.mult[2] = 1; d.W = d.H = 0; d.values = NULL; s->t[i] = d; }  /* Texture() */
        s->n = group + 1;
    }
    tex* d = &s->t[group];
    free(d->values); d->values = NULL; d->W = d->H = 0;
    memcpy(d->mult, t->mult, sizeof(d->mult));
    if (t->texels && t->W > 0 && t->H > 0) {
        d->W = (size_t)t->W; d->H = (size_t)t->H;
        d->values = (float*)malloc(sizeof(float) * 3 * d->W * d->H);
        memcpy(d->values, t->texels, sizeof(float) * 3 * d->W * d->H);
    }
}
int ptb_set_group_material(ptb_ctx* c, int obj, int group, const ptb_material* m) {
    if (!c || !m || obj < 0 || obj >= c->n_objs || group < 0) return PTB_ERR_INVALID;
    object* o = c->objs[obj];
    if (m->present & PTB_SLOT_KD) put_slot(&o->slots[S_KD], group, &m->Kd);
    if (m->present & PTB_SLOT_KS) put_slot(&o->slots[S_KS], group, &m->Ks);
    if (m->present & PTB_SLOT_NE) put_slot(&o->slots[S_NE], group, &m->Ne);
    if (m->present & PTB_SLOT_TRANSP) put_slot(&o->slots[S_TRANSP], group, &m->transp);
    if (m->present & PTB_SLOT_REFR) put_slot(&o->slots[S_REFR], group, &m->refr);
    if (m->present & PTB_SLOT_NORMAL) put_slot(&o->slots[S_NORMAL], group, &m->normal);
    if (m->present & PTB_SLOT_ALPHA) put_slot(&o->slots[S_ALPHA], group, &m->alpha);
    if (m->present & PTB_SLOT_KSUB) {
        if (o->type != T_MESH && (m->Ksub.texels || m->Ksub.mult[0] * m->Ksub.mult[0] + m->Ksub.mult[1] * m->Ksub.mult[1] + m->Ksub.mult[2] * m->Ksub.mult[2] > 1E-8f)) {
            snprintf(c->err, sizeof(c->err), "subsurface scattering on a sphere / plane is undefined in the reference (Geometry.h:994-1012)"); return PTB_ERR_UNSUPPORTED;
        }
        put_slot(&o->slots[S_KSUB], group, &m->Ksub);
    }
    return PTB_OK;
}
int ptb_add_merl(ptb_ctx* c, const double* table, int* out_id) {
    if (!c || !table) return PTB_ERR_INVALID;
    size_t n = (size_t)3 * 90 * 90 * 180;
    c->merl = (double**)realloc(c->merl, sizeof(double*) * (size_t)(c->n_merl + 1));
    c->merl[c->n_merl] = (double*)malloc(n * sizeof(double));
    memcpy(c->merl[c->n_merl], table, n * sizeof(double));
    if (out_id) *out_id = c->n_merl;
    c->n_merl++;
    return PTB_OK;
}
int ptb_set_brdf(ptb_ctx* c, int obj, int kind, int merl_id) {
    if (!c || obj < 0 || obj >= c->n_objs) return PTB_ERR_INVALID;
    if (kind == PTB_BRDF_MERL) { if (merl_id < 0 || merl_id >= c->n_merl) return PTB_ERR_INVALID; c->objs[obj]->merl = c->merl[merl_id]; }
    else if (kind != PTB_BRDF_PHONG) return PTB_ERR_UNSUPPORTED;
    c->objs[obj]->brdf = kind;
    return PTB_OK;
}
int ptb_set_envmap(ptb_ctx* c, const uint8_t* rgb, int W, int H) {
    if (!c || c->n_objs < 2 || c->objs[1]->type != T_SPHERE) return PTB_ERR_STATE;
    free(c->env); c->env = NULL;
    object* dome = c->objs[1];
    if (!rgb || W <= 0 || H <= 0) { dome->has_envmap = 0; return PTB_OK; }
    c->env = (uint8_t*)malloc((size_t)W * H * 3);
    memcpy(c->env, rgb, (size_t)W * H * 3);
    dome->envtex = c->env; dome->envW = W; dome->envH = H; dome->has_envmap = 1;
    return PTB_OK;
}
int ptb_set_light(ptb_ctx* c, float il, float ei) { if (!c) return PTB_ERR_INVALID; c->intensite_lumiere = il; c->envmap_intensity = ei; return PTB_OK; }
int ptb_set_fog(ptb_ctx* c, const ptb_fog* f) { if (!c || !f) return PTB_ERR_INVALID; c->fog = *f; return PTB_OK; }
/* the std::map<float, ...> keyframe tracks: ascending frames, a later assignment to the same frame wins */
int ptb_set_keyframes(ptb_ctx* c, int obj, int kind, const float* frames, const float* values, int n) {
    static const int width[3] = {1, 3, 9};
    if (!c || obj < 0 || obj >= c->n_objs || kind < 0 || kind > 2 || n < 0) return PTB_ERR_INVALID;
    object* o = c->objs[obj]; int w = width[kind];
    free(o->kframe[kind]); free(o->kval[kind]); o->kframe[kind] = o->kval[kind] = NULL; o->nkey[kind] = 0;
    if (n == 0) return PTB_OK;
    o->kframe[kind] = (float*)malloc(n * sizeof(float)); o->kval[kind] = (float*)malloc((size_t)n * w * sizeof(float));
    int m = 0;
    for (int i = 0; i < n; i++) {                                       /* insertion into the sorted track */
        int pos = 0;
        while (pos < m && o->kframe[kind][pos] < frames[i]) pos++;
        if (pos < m && o->kframe[kind][pos] == frames[i]) { memcpy(o->kval[kind] + (size_t)pos * w, values + (size_t)i * w, w * sizeof(float)); continue; }
        memmove(o->kframe[kind] + pos + 1, o->kframe[kind] + pos, (m - pos) * sizeof(float));
        memmove(o->kval[kind] + (size_t)(pos + 1) * w, o->kval[kind] + (size_t)pos * w, (size_t)(m - pos) * w * sizeof(float));
        o->kframe[kind][pos] = frames[i]; memcpy(o->kval[kind] + (size_t)pos * w, values + (size_t)i * w, w * sizeof(float));
        m++;
    }
    o->nkey[kind] = m;
    return PTB_OK;
}
int ptb_set_frame(ptb_ctx* c, float frame) { if (!c) return PTB_ERR_INVALID; c->current_frame = (int)frame; return PTB_OK; }
int ptb_set_background(ptb_ctx* c, const float* rgb, int W, int H) {
    if (!c) return PTB_ERR_INVALID;
    free(c->bg); c->bg = NULL; c->bgW = c->bgH = 0;
    if (!rgb || W <= 0 || H <= 0) return PTB_OK;
    c->bg = (float*)malloc((size_t)W * H * 3 * sizeof(float));
    memcpy(c->bg, rgb, (size_t)W * H * 3 * sizeof(float));
    c->bgW = W; c->bgH = H;
    return PTB_OK;
}
int ptb_commit(ptb_ctx* c) {
    if (!c) return PTB_ERR_INVALID;
    if (c->n_objs < 2 || c->objs[0]->type != T_SPHERE || c->objs[1]->type != T_SPHERE) { snprintf(c->err, sizeof(c->err), "need light (id 0) and dome (id 1)"); return PTB_ERR_STATE; }
    if (c->fog.density > 1E-8 && c->n_objs < 3) { snprintf(c->err, sizeof(c->err), "fog needs object 2 (its translation is the ground level)"); return PTB_ERR_STATE; }
    c->committed = 1;
    return PTB_OK;
}
static int set_frame(ptb_ctx* c, const ptb_camera* cam, int W, int H) {
    c->cam_pos = V(cam->position[0], cam->position[1], cam->position[2]);
    c->cam_dir = V(cam->direction[0], cam->direction[1], cam->direction[2]);
    c->cam_up = V(cam->up[0], cam->up[1], cam->up[2]);
    c->fov = cam->fov; c->focus_distance = cam->focus_distance; c->aperture = cam->aperture;
    c->W = W; c->H = H;
    return PTB_OK;
}

/* Raytracer::render_image_nopreviz (Raytracer.cpp:1565-1708) with the per-(pixel,sample) streams of build_ref.py patch 5 */
int ptb_render(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, float* imagedouble, float* sample_count, uint8_t* image, ptb_stats* stats) {
    if (!c || !cam || !p || p->W <= 0 || p->H <= 0 || p->nrays <= 0) return PTB_ERR_INVALID;
    if (!c->committed) return PTB_ERR_STATE;
    if (p->shard_count > 1) return PTB_ERR_UNSUPPORTED;
    set_frame(c, cam, p->W, p->H);
    c->nrays = p->nrays; c->nb_bounces = p->nb_bounces; c->sigma_filter = p->sigma_filter; c->gamma = p->gamma; c->seed = p->seed;
    if ((int)ceilf(c->sigma_filter * 2) > 4) return PTB_ERR_UNSUPPORTED;
    int nt = c->threads > 0 ? c->threads : omp_get_num_procs();
    if (nt > 64) nt = 64;
    struct timespec t0, t1; clock_gettime(CLOCK_MONOTONIC, &t0);
    prepare_render(c);
    const int W = c->W, H = c->H, nrays = c->nrays, fs = c->filter_size, ftw = c->filter_total_width;
    vec* samples2d = (vec*)malloc(sizeof(vec) * (size_t)nrays);
    for (int i = 0; i < nrays; i++) { float x, y; lattice2d((uint32_t)i, &x, &y); samples2d[i] = V(x, y, 0); }
    float denom2 = 1.f / (2.f * c->sigma_filter * c->sigma_filter);
    const int bw = 4, bh = 4;
    const int nbx = (int)ceilf(W / (float)bw), nby = (int)ceilf(H / (float)bh);
    size_t npix = (size_t)W * H;
    float* img_t = (float*)calloc(npix * 3 * (size_t)nt, sizeof(float));
    float* cnt_t = (float*)calloc(npix * (size_t)nt, sizeof(float));
    unsigned long long counters[64][8];
    memset(counters, 0, sizeof(counters));
#pragma omp parallel num_threads(nt)
    {
        int th = omp_get_thread_num();
        float* img = img_t + (size_t)th * npix * 3;
        float* cnt = cnt_t + (size_t)th * npix;
#pragma omp for schedule(dynamic, 1)
        for (int batch = 0; batch < nbx * nby; batch++) {
            int bi = batch / nbx, bj = batch % nbx;
            int bW = (W < bj * bw + bw ? W : bj * bw + bw) - bj * bw, bH = (H < bi * bh + bh ? H : bi * bh + bh) - bi * bh;
            for (int id = 0; id < bW * bH; id++) {
                int i = bi * bh + id / bW, j = bj * bw + id % bW;
                int bmin_i = i - fs > 0 ? i - fs : 0, bmax_i = i + fs < H - 1 ? i + fs : H - 1;
                int bmin_j = j - fs > 0 ? j - fs : 0, bmax_j = j + fs < W - 1 ? j + fs : W - 1;
                float ratio = 1.f / sat(c->filter_integral, ftw, bmin_i - i + fs, bmax_i - i + fs, bmin_j - j + fs, bmax_j - j + fs);
                float denom1 = (float)(ratio / (c->sigma_filter * c->sigma_filter * 2. * M_PI));
                for (int k = 0; k < nrays; k++) {
                    pcg e = pcg_seed2((uint64_t)(i * W + j), (uint64_t)k ^ ((uint64_t)c->seed << 32));
                    float dx = pcg_unif(&e) - 0.5f, dy = pcg_unif(&e) - 0.5f;
                    float dxa = (pcg_unif(&e) - 0.5f) * c->aperture, dya = (pcg_unif(&e) - 0.5f) * c->aperture;
                    vec ro, rd;
                    camera_ray(c, 0.f, i, j, dx, dy, dxa, dya, W, H, &ro, &rd);
                    vec col = get_color(c, ro, rd, k, i * W + j, &e, counters[th], samples2d, NULL, NULL);
                    for (int i2 = bmin_i; i2 <= bmax_i; i2++)
                        for (int j2 = bmin_j; j2 <= bmax_j; j2++) {
                            size_t idx = ((size_t)(H - i2 - 1) * W + j2) * 3;
                            float a = (i2 - i - dy), b = (j2 - j - dx);
                            float w = (float)(fast_exp(-(a * a + b * b) * denom2) * denom1);
                            img[idx] += col.x * w; img[idx + 1] += col.y * w; img[idx + 2] += col.z * w;
                            cnt[(size_t)(H - i2 - 1) * W + j2] += w;
                        }
                }
            }
        }
    }
    float* acc = (float*)calloc(npix * 3, sizeof(float));
    float* sc = (float*)calloc(npix, sizeof(float));
    for (int th = 0; th < nt; th++)
        for (size_t i = 0; i < npix; i++) {
            acc[i * 3] += img_t[(size_t)th * npix * 3 + i * 3]; acc[i * 3 + 1] += img_t[(size_t)th * npix * 3 + i * 3 + 1];
            acc[i * 3 + 2] += img_t[(size_t)th * npix * 3 + i * 3 + 2]; sc[i] += cnt_t[(size_t)th * npix + i];
        }
    for (size_t i = 0; i < npix; i++) for (int q = 0; q < 3; q++) acc[i * 3 + q] /= sc[i];
    clock_gettime(CLOCK_MONOTONIC, &t1);
    if (imagedouble) memcpy(imagedouble, acc, npix * 3 * sizeof(float));
    if (sample_count) memcpy(sample_count, sc, npix * sizeof(float));
    if (image)
        for (size_t i = 0; i < npix * 3; i++) {
            double v = 255. * pow(acc[i] / 196964.7, 1 / c->gamma);
            v = v > 0. ? v : 0.; v = v < 255. ? v : 255.;
            image[i] = (uint8_t)v;
        }
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->samples = (uint64_t)npix * (uint64_t)nrays;
        for (int th = 0; th < 64; th++) { stats->rays_closest += counters[th][0]; stats->rays_shadow += counters[th][1]; }
        stats->ms_wall = (t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6;
    }
    free(acc); free(sc); free(img_t); free(cnt_t); free(samples2d);
    return PTB_OK;
}
/* render_image_nopreviz with has_denoiser == true (Raytracer.cpp:1631-1645 accumulation, 1669-1694 merge and normalisation) */
int ptb_render_denoiser_inputs(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, float* imagedouble, float* sample_count, float* albedoImage,
                               float* normalImage, float* first_hit_normal, ptb_stats* stats) {
    if (!c || !cam || !p || p->W <= 0 || p->H <= 0 || p->nrays <= 0) return PTB_ERR_INVALID;
    if (!c->committed) return PTB_ERR_STATE;
    if (p->shard_count > 1) return PTB_ERR_UNSUPPORTED;
    set_frame(c, cam, p->W, p->H);
    c->nrays = p->nrays; c->nb_bounces = p->nb_bounces; c->sigma_filter = p->sigma_filter; c->gamma = p->gamma; c->seed = p->seed;
    int nt = c->threads > 0 ? c->threads : omp_get_num_procs();
    if (nt > 64) nt = 64;
    prepare_render(c);
    const int W = c->W, H = c->H, nrays = c->nrays;
    vec* samples2d = (vec*)malloc(sizeof(vec) * (size_t)nrays);
    for (int i = 0; i < nrays; i++) { float x, y; lattice2d((uint32_t)i, &x, &y); samples2d[i] = V(x, y, 0); }
    const int bw = 4, bh = 4;
    const int nbx = (int)ceilf(W / (float)bw), nby = (int)ceilf(H / (float)bh);
    size_t npix = (size_t)W * H;
    float* img_t = (float*)calloc(npix * 3 * (size_t)nt, sizeof(float));
    float* cnt_t = (float*)calloc(npix * (size_t)nt, sizeof(float));
    float* alb_t = (float*)calloc(npix * 3 * (size_t)nt, sizeof(float));
    float* nrm_t = (float*)calloc(npix * 3 * (size_t)nt, sizeof(float));
    unsigned long long counters[64][8];
    memset(counters, 0, sizeof(counters));
#pragma omp parallel num_threads(nt)
    {
        int th = omp_get_thread_num();
        float* img = img_t + (size_t)th * npix * 3; float* cnt = cnt_t + (size_t)th * npix;
        float* alb = alb_t + (size_t)th * npix * 3; float* nrm = nrm_t + (size_t)th * npix * 3;
#pragma omp for schedule(dynamic, 1)
        for (int batch = 0; batch < nbx * nby; batch++) {
            int bi = batch / nbx, bj = batch % nbx;
            int bW = (W < bj * bw + bw ? W : bj * bw + bw) - bj * bw, bH = (H < bi * bh + bh ? H : bi * bh + bh) - bi * bh;
            for (int id = 0; id < bW * bH; id++) {
                int i = bi * bh + id / bW, j = bj * bw + id % bW;
                for (int k = 0; k < nrays; k++) {
                    pcg e = pcg_seed2((uint64_t)(i * W + j), (uint64_t)k ^ ((uint64_t)c->seed << 32));
                    float dx = pcg_unif(&e) - 0.5f, dy = pcg_unif(&e) - 0.5f;
                    float dxa = (pcg_unif(&e) - 0.5f) * c->aperture, dya = (pcg_unif(&e) - 0.5f) * c->aperture;
                    vec ro, rd, normal = V(0, 0, 0), albedo = V(0, 0, 0);          /* `Vector normal, albedo;` are zero-initialised (Vector.h:45) */
                    camera_ray(c, 0.f, i, j, dx, dy, dxa, dya, W, H, &ro, &rd);
                    vec col = get_color(c, ro, rd, k, i * W + j, &e, counters[th], samples2d, &normal, &albedo);
                    size_t idx = ((size_t)(H - i - 1) * W + j) * 3;
                    img[idx] += col.x; img[idx + 1] += col.y; img[idx + 2] += col.z;
                    cnt[(size_t)(H - i - 1) * W + j] += 1;
                    nrm[idx] += normal.x; nrm[idx + 1] += normal.y; nrm[idx + 2] += normal.z;
                    alb[idx] += albedo.x; alb[idx + 1] += albedo.y; alb[idx + 2] += albedo.z;
                }
            }
        }
    }
    float* acc = (float*)calloc(npix * 3, sizeof(float)); float* sc = (float*)calloc(npix, sizeof(float));
    float* al = (float*)calloc(npix * 3, sizeof(float)); float* nr = (float*)calloc(npix * 3, sizeof(float)); float* fh = (float*)calloc(npix * 3, sizeof(float));
    for (int th = 0; th < nt; th++)
        for (size_t i = 0; i < npix; i++) {
            sc[i] += cnt_t[(size_t)th * npix + i];
            for (int q = 0; q < 3; q++) {
                acc[i * 3 + q] += img_t[(size_t)th * npix * 3 + i * 3 + q];
                al[i * 3 + q] += alb_t[(size_t)th * npix * 3 + i * 3 + q];
                nr[i * 3 + q] += img_t[(size_t)th * npix * 3 + i * 3 + q];     /* 1680-1682: the reference adds imagedoublethreads here, not the normals */
                fh[i * 3 + q] += nrm_t[(size_t)th * npix * 3 + i * 3 + q];     /* what that line was meant to add */
            }
        }
    for (size_t i = 0; i < npix; i++) {                                         /* 1687-1694 */
        float nn = sqrtf(nr[i * 3] * nr[i * 3] + nr[i * 3 + 1] * nr[i * 3 + 1] + nr[i * 3 + 2] * nr[i * 3 + 2]);
        float nf = sqrtf(fh[i * 3] * fh[i * 3] + fh[i * 3 + 1] * fh[i * 3 + 1] + fh[i * 3 + 2] * fh[i * 3 + 2]);
        for (int q = 0; q < 3; q++) { acc[i * 3 + q] /= sc[i]; al[i * 3 + q] /= sc[i]; nr[i * 3 + q] /= nn; fh[i * 3 + q] /= nf; }
    }
    if (imagedouble) memcpy(imagedouble, acc, npix * 3 * sizeof(float));
    if (sample_count) memcpy(sample_count, sc, npix * sizeof(float));
    if (albedoImage) memcpy(albedoImage, al, npix * 3 * sizeof(float));
    if (normalImage) memcpy(normalImage, nr, npix * 3 * sizeof(float));
    if (first_hit_normal) memcpy(first_hit_normal, fh, npix * 3 * sizeof(float));
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->samples = (uint64_t)npix * (uint64_t)nrays;
        for (int th = 0; th < 64; th++) { stats->rays_closest += counters[th][0]; stats->rays_shadow += counters[th][1]; }
    }
    free(acc); free(sc); free(al); free(nr); free(fh); free(img_t); free(cnt_t); free(alb_t); free(nrm_t); free(samples2d);
    return PTB_OK;
}

/* Raytracer::render_image (Raytracer.cpp:1424-1563), a batch of passes per call; per-(pixel,sample) streams as in ptb_render */
static void prog_free(ptb_ctx* c) { free(c->prog_img); free(c->prog_cnt); free(c->prog_lowres); free(c->prog_samples2d); c->prog_img = c->prog_cnt = c->prog_lowres = NULL; c->prog_samples2d = NULL; c->prog_active = 0; }
int ptb_progressive_begin(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p) {
    if (!c || !cam || !p || p->W <= 0 || p->H <= 0 || p->nrays <= 0) return PTB_ERR_INVALID;
    if (!c->committed) return PTB_ERR_STATE;
    prog_free(c);
    set_frame(c, cam, p->W, p->H);
    c->nrays = p->nrays; c->nb_bounces = p->nb_bounces; c->sigma_filter = p->sigma_filter; c->gamma = p->gamma; c->seed = p->seed;
    if ((int)ceilf(c->sigma_filter * 2) > 4) return PTB_ERR_UNSUPPORTED;
    prepare_render(c);                                                          /* 1441: zeroes the buffers (1382-1389) */
    const size_t npix = (size_t)c->W * c->H;
    const int Wlr = (int)ceilf(c->W / 16.f), Hlr = (int)ceilf(c->H / 16.f);      /* 1329-1330 */
    c->prog_img = (float*)calloc(npix * 3, sizeof(float));
    c->prog_cnt = (float*)calloc(npix, sizeof(float));
    c->prog_lowres = (float*)calloc((size_t)Wlr * Hlr * 3, sizeof(float));
    c->prog_samples2d = (vec*)malloc(sizeof(vec) * (size_t)c->nrays);
    for (int i = 0; i < c->nrays; i++) { float x, y; lattice2d((uint32_t)i, &x, &y); c->prog_samples2d[i] = V(x, y, 0); }
    c->prog_iter = 0; c->prog_active = 1;
    return PTB_OK;
}
int ptb_progressive_pass(ptb_ctx* c, int n_spp, ptb_stats* stats) {
    if (!c) return PTB_ERR_INVALID;
    if (!c->prog_active) return PTB_ERR_STATE;
    const int W = c->W, H = c->H, fs = c->filter_size, ftw = c->filter_total_width;
    const int Wlr = (int)ceilf(W / 16.f), Hlr = (int)ceilf(H / 16.f);
    int n = n_spp < c->nrays - c->prog_iter ? n_spp : c->nrays - c->prog_iter;
    int nt = c->threads > 0 ? c->threads : omp_get_num_procs();
    if (nt > 64) nt = 64;
    float denom2 = (float)(1.f / (2. * c->sigma_filter * c->sigma_filter));      /* 1430: double arithmetic narrowed to float */
    memset(c->prog_counters, 0, sizeof(c->prog_counters));
    float* img = c->prog_img; float* cnt = c->prog_cnt; float* lr = c->prog_lowres;
    for (int k = c->prog_iter; k < c->prog_iter + (n > 0 ? n : 0); k++)
        for (int pib = 0; pib < 64; pib++) {                                     /* 1447-1449: 8x8 interleave */
            int i1 = pib % 8, j1 = pib / 8;
#pragma omp parallel for schedule(dynamic, 1) num_threads(nt)
            for (int i = i1; i < H; i += 8) {
                int th = omp_get_thread_num();
                for (int j = j1; j < W; j += 8) {
                    pcg e = pcg_seed2((uint64_t)(i * W + j), (uint64_t)k ^ ((uint64_t)c->seed << 32));
                    float dx = pcg_unif(&e) - 0.5f, dy = pcg_unif(&e) - 0.5f;
                    float dxa = (pcg_unif(&e) - 0.5f) * c->aperture, dya = (pcg_unif(&e) - 0.5f) * c->aperture;
                    vec ro, rd;
                    camera_ray(c, 0.f, i, j, dx, dy, dxa, dya, W, H, &ro, &rd);
                    vec col = get_color(c, ro, rd, k, i * W + j, &e, c->prog_counters[th], c->prog_samples2d, NULL, NULL);
                    int bmin_i = i - fs > 0 ? i - fs : 0, bmax_i = i + fs < H - 1 ? i + fs : H - 1;
                    int bmin_j = j - fs > 0 ? j - fs : 0, bmax_j = j + fs < W - 1 ? j + fs : W - 1;
                    float ratio = 1.f / sat(c->filter_integral, ftw, bmin_i - i + fs, bmax_i - i + fs, bmin_j - j + fs, bmax_j - j + fs);
                    float denom1 = (float)(ratio / (c->sigma_filter * c->sigma_filter * 2. * M_PI));
                    for (int i2 = bmin_i; i2 <= bmax_i; i2++)
                        for (int j2 = bmin_j; j2 <= bmax_j; j2++) {
                            size_t idx = ((size_t)(H - i2 - 1) * W + j2) * 3;
                            float a = (i2 - i - dy), b = (j2 - j - dx);
                            float w = (float)(fast_exp(-(a * a + b * b) * denom2) * denom1);
                            img[idx] += col.x * w; img[idx + 1] += col.y * w; img[idx + 2] += col.z * w;
                            cnt[(size_t)(H - i2 - 1) * W + j2] += w;
                        }
                    size_t li = ((size_t)(Hlr - i / 16 - 1) * Wlr + j / 16) * 3;   /* 1508-1510 (rows i and i+8 share a block: unordered adds when threaded) */
                    for (int q = 0; q < 3; q++) {
                        float add = (float)(vget(col, q) / 256.);
#pragma omp atomic
                        lr[li + q] += add;
                    }
                }
            }
        }
    if (n > 0) c->prog_iter += n;
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->samples = (uint64_t)W * H * (uint64_t)(n > 0 ? n : 0);
        for (int th = 0; th < 64; th++) { stats->rays_closest += c->prog_counters[th][0]; stats->rays_shadow += c->prog_counters[th][1]; }
    }
    return PTB_OK;
}
int ptb_progressive_read(ptb_ctx* c, float* imagedouble, float* sample_count, uint8_t* image, float* imagedouble_lowres, int32_t* current_nb_rays) {
    if (!c) return PTB_ERR_INVALID;
    if (!c->prog_active) return PTB_ERR_STATE;
    const size_t npix = (size_t)c->W * c->H;
    const int Wlr = (int)ceilf(c->W / 16.f), Hlr = (int)ceilf(c->H / 16.f);
    if (imagedouble) memcpy(imagedouble, c->prog_img, npix * 3 * sizeof(float));
    if (sample_count) memcpy(sample_count, c->prog_cnt, npix * sizeof(float));
    if (imagedouble_lowres) memcpy(imagedouble_lowres, c->prog_lowres, (size_t)Wlr * Hlr * 3 * sizeof(float));
    if (image)                                                                   /* 1540-1547 */
        for (size_t i = 0; i < npix; i++)
            for (int q = 0; q < 3; q++) {
                float d = c->prog_cnt[i] < 1.f ? 1.f : c->prog_cnt[i];           /* std::max(sample_count, 1.f) */
                double v = 255. * pow(c->prog_img[i * 3 + q] / 196964.7 / d, 1 / c->gamma);
                v = v > 0. ? v : 0.; v = v < 255. ? v : 255.;
                image[i * 3 + q] = (uint8_t)v;
            }
    if (current_nb_rays) *current_nb_rays = c->prog_iter;
    return PTB_OK;
}

int ptb_render_accum(ptb_ctx* c, const ptb_camera* a, const ptb_params* b, float* d, ptb_stats* s) { (void)c; (void)a; (void)b; (void)d; (void)s; return PTB_ERR_UNSUPPORTED; }
int ptb_resolve(ptb_ctx* c, const float* d, int W, int H, float g, float* a, float* b, uint8_t* e) { (void)c; (void)d; (void)W; (void)H; (void)g; (void)a; (void)b; (void)e; return PTB_ERR_UNSUPPORTED; }
int ptb_shard_pack_size(const ptb_params* p, int r, int64_t* o) { (void)p; (void)r; (void)o; return PTB_ERR_UNSUPPORTED; }
int ptb_shard_pack(ptb_ctx* c, const ptb_params* p, int r, const float* a, float* b) { (void)c; (void)p; (void)r; (void)a; (void)b; return PTB_ERR_UNSUPPORTED; }
int ptb_shard_unpack_add(ptb_ctx* c, const ptb_params* p, int r, const float* a, float* b) { (void)c; (void)p; (void)r; (void)a; (void)b; return PTB_ERR_UNSUPPORTED; }

/* the picking query (mainApp.h:686-692) */
int ptb_primary_ids(ptb_ctx* c, const ptb_camera* cam, int W, int H, int32_t* obj_id, int32_t* tri_id, float* tout) {
    if (!c || !cam || W <= 0 || H <= 0) return PTB_ERR_INVALID;
    if (!c->committed) return PTB_ERR_STATE;
    set_frame(c, cam, W, H);
    for (int i = 0; i < c->n_objs; i++) build_matrix(c->objs[i], (float)c->current_frame);
#pragma omp parallel for schedule(dynamic, 4)
    for (int i = 0; i < H; i++)
        for (int j = 0; j < W; j++) {
            vec ro, rd, P; matvals m = matvals_default(); int id = -1, tri = -1; float t;
            camera_ray(c, 0, i, j, 0, 0, 0, 0, W, H, &ro, &rd);
            int hit = scene_hit(c, ro, rd, &P, &id, &t, &m, &tri, NULL);
            int32_t oid = -1, tid = -1;
            if (hit) { oid = id; if (c->objs[id]->type == T_MESH && tri >= 0) tid = c->objs[id]->permuted[tri];
                       if (c->objs[id]->type == T_POINTSET && tri >= 0) tid = c->objs[id]->pt_perm[tri];
                       if (c->objs[id]->type == T_YARNS && tri >= 0) tid = c->objs[id]->y_perm[tri]; }
            if (obj_id) obj_id[(size_t)i * W + j] = oid;
            if (tri_id) tri_id[(size_t)i * W + j] = tid;
            if (tout) tout[(size_t)i * W + j] = hit ? t : -1.f;
        }
    return PTB_OK;
}
int ptb_set_option(ptb_ctx* c, int option, int64_t value) { if (!c) return PTB_ERR_INVALID; if (option == ORC_OPT_THREADS) c->threads = (int)value; return PTB_OK; }
int ptb_get_scene_info(const ptb_ctx* c, ptb_scene_info* info) {
    if (!c || !info) return PTB_ERR_INVALID;
    memset(info, 0, sizeof(*info));
    info->n_triangles = c->n_tri; info->n_objects = c->n_objs; info->ms_bvh_build = c->ms_build;
    for (int i = 0; i < c->n_objs; i++) if (c->objs[i]->type == T_MESH) { info->n_bvh_nodes += c->objs[i]->n_nodes; if (c->objs[i]->bvh_depth > info->bvh_depth) info->bvh_depth = c->objs[i]->bvh_depth; }
    info->bytes_nodes = info->n_bvh_nodes * (int64_t)sizeof(bnode); info->bytes_triangles = info->n_triangles * (int64_t)sizeof(tsoup);
    return PTB_OK;
}
int ptb_get_kernel_times(const ptb_ctx* c, ptb_kernel_times* t) { (void)c; (void)t; return PTB_ERR_UNSUPPORTED; }
/* PTB_KAT_RAY / PTB_KAT_RAY_WAVEFRONT on one float ray (the doubles narrowed, a zero keeps its sign): Scene::intersection restricted to
 * t < tmax -> object id, original triangle id (-1: not a triangle), t, b1, b2 (a miss: -1, -1, -1, 0, 0), or, any_hit != 0,
 * Scene::intersection_shadow(o, d, dist_light = tmax) -> occluded 0/1, 0, 0, 0, 0.  The reference's decisions near edges. */
static void kat_ray(const struct ptb_ctx* c, const double* a, double* out) {
    vec o = V((float)a[0], (float)a[1], (float)a[2]), d = V((float)a[3], (float)a[4], (float)a[5]);
    float tmax = (float)a[6];
    out[0] = -1; out[1] = -1; out[2] = -1; out[3] = 0; out[4] = 0;
    if (a[7] != 0) { out[0] = scene_shadow(c, o, d, tmax, NULL); out[1] = out[2] = 0; return; }
    vec P; matvals m = matvals_default(); int id = -1, tri = -1; float t;
    if (!scene_hit(c, o, d, &P, &id, &t, &m, &tri, NULL) || !(t < tmax)) return;
    const object* ob = c->objs[id];
    out[0] = id; out[2] = t;
    if (ob->type == T_MESH && tri >= 0) {
        vec dl = xf_dir(ob->inv, d), ol = xf_point(ob->inv, o), lp; float lt, al, be, ga;
        soup_hit(&ob->soup[tri], ol, dl, &lp, &lt, &al, &be, &ga);   /* the barycentrics mesh_hit found the hit with */
        out[1] = ob->permuted[tri]; out[3] = be; out[4] = ga;
    }
}

int ptb_kat(ptb_ctx* c, int which, const ptb_camera* cam, int W, int H, const double* in, int n, int is, double* out, int os) {
    if (!c || !in || !out) return PTB_ERR_INVALID;
    if (cam) set_frame(c, cam, W, H);
    if (which == PTB_KAT_RAY || which == PTB_KAT_RAY_WAVEFRONT) {
        if (!c->committed) return PTB_ERR_STATE;
        for (int i = 0; i < c->n_objs; i++) build_matrix(c->objs[i], (float)c->current_frame);
#pragma omp parallel for schedule(dynamic, 256)
        for (int k = 0; k < n; k++) kat_ray(c, in + (size_t)k * is, out + (size_t)k * os);
        return PTB_OK;
    }
    if (which == PTB_KAT_RANDOM_PER_PIXEL || which == PTB_KAT_FILTER_RATIO) {
        if (!c->committed) return PTB_ERR_STATE;
        c->W = W; c->H = H;
        if (which == PTB_KAT_FILTER_RATIO) c->sigma_filter = (float)in[2];
        prepare_render(c);
    }
    for (int k = 0; k < n; k++) {
        const double* a = in + (size_t)k * is; double* o = out + (size_t)k * os;
        switch (which) {
        case PTB_KAT_PCG32: { pcg e = pcg_seed2((uint64_t)a[0], (uint64_t)a[1]); for (int q = 0; q < 4; q++) o[q] = (double)pcg_next(&e); } break;
        case PTB_KAT_LATTICE: { float x, y; lattice2d((uint32_t)a[0], &x, &y); o[0] = x; o[1] = y; } break;
        case PTB_KAT_CAMERA: { vec ro, rd; camera_ray(c, 0, (int)a[0], (int)a[1], (float)a[2], (float)a[3], (float)a[4], (float)a[5], W, H, &ro, &rd);
            o[0] = ro.x; o[1] = ro.y; o[2] = ro.z; o[3] = rd.x; o[4] = rd.y; o[5] = rd.z; } break;
        case PTB_KAT_RANDOM_COS: { vec v = random_cos(V((float)a[0], (float)a[1], (float)a[2]), (float)a[3], (float)a[4]); o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
        case PTB_KAT_RANDOM_PHONG: { vec v = random_phong(V((float)a[0], (float)a[1], (float)a[2]), (float)a[3], (float)a[4], (float)a[5]); o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
        case PTB_KAT_PHONG_EVAL: { matvals m = matvals_default(); m.Kd = V((float)a[0], (float)a[1], (float)a[2]); m.Ks = V((float)a[3], (float)a[4], (float)a[5]); m.Ne = V((float)a[6], (float)a[7], (float)a[8]);
            vec v = phong_eval(&m, V((float)a[9], (float)a[10], (float)a[11]), V((float)a[12], (float)a[13], (float)a[14]), V((float)a[15], (float)a[16], (float)a[17])); o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
        case PTB_KAT_MERL_EVAL: { if (c->n_merl == 0) return PTB_ERR_STATE;
            vec v = merl_eval(c->merl[0], V((float)a[0], (float)a[1], (float)a[2]), V((float)a[3], (float)a[4], (float)a[5]), V((float)a[6], (float)a[7], (float)a[8])); o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
        case PTB_KAT_FAST_EXP: o[0] = fast_exp(a[0]); break;
        case PTB_KAT_FAST_NORMALIZE: { vec v = vfast_normalize(V((float)a[0], (float)a[1], (float)a[2])); o[0] = v.x; o[1] = v.y; o[2] = v.z; } break;
        case PTB_KAT_RANDOM_PER_PIXEL: { size_t p = (size_t)a[0]; o[0] = c->randomPerPixel[p].x; o[1] = c->randomPerPixel[p].y; } break;
        case PTB_KAT_FILTER_RATIO: { int i = (int)a[0], j = (int)a[1], fs = c->filter_size, ftw = c->filter_total_width;
            int bmin_i = i - fs > 0 ? i - fs : 0, bmax_i = i + fs < H - 1 ? i + fs : H - 1, bmin_j = j - fs > 0 ? j - fs : 0, bmax_j = j + fs < W - 1 ? j + fs : W - 1;
            o[0] = 1.f / sat(c->filter_integral, ftw, bmin_i - i + fs, bmax_i - i + fs, bmin_j - j + fs, bmax_j - j + fs); } break;
        default: return PTB_ERR_UNSUPPORTED;
        }
    }
    return PTB_OK;
}
