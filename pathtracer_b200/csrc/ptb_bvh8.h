// ptb_bvh8.h — compressed 8-wide BVH: node layout and ray traversal (closest hit and any hit).
//
// Replaces the reference's binary BVH (`BVHNodesT`, TriangleMesh.h:6-28; traversal
// TriangleMesh.cpp:1133-1319; slab tests Geometry.h:114-204; `Triangle::intersection`
// TriangleMesh.h:82-104).  Layout after Ylitie, Karras, Laine 2017 ("Efficient Incoherent Ray
// Traversal on GPUs Through Compressed Wide BVHs"): one 80-byte node = 5 x 16-byte loads holds 8
// child boxes quantised to 8 bits on a per-node power-of-two grid.
//
//   bytes  0-11  p        float3 grid origin (node box min)
//         12-14  e        int8 exponents: cell size 2^e per axis
//            15  imask    bit s set <=> slot s holds an internal node
//         16-19  child_base   index of the first internal child (children are contiguous, slot order)
//         20-23  tri_base     index of the node's first triangle (leaf children contiguous)
//         24-26  valid24  bit 3*s + k set <=> slot s is a leaf with more than k triangles (at most 3 per leaf); the node's
//                         triangles are stored compactly in this bit order: index = tri_base + popcount(valid24 below the bit)
//         27-31  reserved (0)
//         32-79  qlo_x[8] qlo_y[8] qlo_z[8] qhi_x[8] qhi_y[8] qhi_z[8]
//
// Triangles are stored in leaf order as 3 x float4 = 48 bytes {v0, e1 = v1-v0, e2 = v2-v0}; v0.w carries
// the flags, e1.w the barycentric distance from an edge below which the reference's own arithmetic
// decides the hit (PTB_EDGE_EPS, or +inf for alpha-tested triangles; tri_exact).  Semantics mirrored from the reference: two-sided, barycentrics >= 0 inclusive,
// t >= 0 accepted, strictly nearer than the current best wins (TriangleMesh.h:82-104,
// TriangleMesh.cpp:1196-1209); alpha-mapped hits are rejected inside traversal (1198-1205).
#pragma once
#include "ptb_core.h"
#if defined(__CUDACC__)
#include <cuda_fp16.h>
#endif

namespace ptb {

struct alignas(16) Node8 {
    float px, py, pz;
    uint8_t ex, ey, ez, imask;
    uint32_t child_base, tri_base;
    uint8_t valid24[3];   // see the layout above
    uint8_t reserved[5];  // bytes 27-31, 0
    uint8_t qlox[8], qloy[8], qloz[8], qhix[8], qhiy[8], qhiz[8];
};
static_assert(sizeof(Node8) == 80, "Node8 must be 80 bytes");

#define PTB_TRI_FLAG_ALPHA 1u  /* tri.w0 bit: this triangle's group has an alpha map that can reject */
#define PTB_TRI_FLAG_DISC 4u   /* tri.w0 bit: the triangle covers a disc of a point set (disc_cover_triangle, ptb_scene.h); tri_exact runs the disc test */
#define PTB_TRI_T_CUT (1.f - 1e-4f)   /* tri.w2 (e2.w) of an ordinary triangle: the fast test drops a hit when t * w2 >= t_best; 0 = never (volume covers, ptb_scene.h) */
#define PTB_TRI_FLAG_GHOST 2u  /* tri.w0 bit: the triangle belongs to a ghost object; shadow rays pass through it (Geometry.cpp:722) */

// what the quantisation adds to a node box next to the cell-relative part: a few ulps of the coordinates
PTB_HD float node_coord_slack(float lo, float hi) { return 4e-7f * fmaxf(fabsf(lo), fabsf(hi)); }

struct Hit {
    float t, b1, b2;   // distance, barycentric of v1 (beta), of v2 (gamma)
    int32_t prim;      // triangle index in leaf order, -1 none
};

PTB_HD uint32_t highest_bit(uint32_t v) {  // index of the highest set bit, v != 0
#if defined(__CUDA_ARCH__)
    return 31u - (uint32_t)__clz((int)v);
#else
    return 31u - (uint32_t)__builtin_clz(v);
#endif
}
PTB_HD uint32_t popcount32(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return (uint32_t)__popc(v);
#else
    return (uint32_t)__builtin_popcount(v);
#endif
}

#if defined(__CUDA_ARCH__)
#define PTB_LDG_F4(p) __ldg(reinterpret_cast<const float4*>(p))
#else
struct float4_host { float x, y, z, w; };
#define PTB_LDG_F4(p) (*reinterpret_cast<const ptb::float4_host*>(p))
#endif

// Per-ray constants of the slab test in quantised space.
struct RayPrep {
    V3 o, d, idir;
    uint32_t oct_inv4;  // byte 0: 7 - octant (octant bit set <=> direction component negative); bytes 1..3: the slot masks of
                        // pick_slot for that octant (the half, the pairs, the single slots visited first)
};
PTB_HD RayPrep ray_prep(V3 o, V3 d) {
    RayPrep r;
    r.o = o; r.d = d;
    const float eps = 1e-30f;
    // One sign per axis for the substitute of a tiny component, the octant and node_hitmask's entry plane: `d < 0`.  The sign bit
    // (copysignf) would call -0.0 negative where the slab test calls it positive, swap the entry and exit planes on that axis and
    // reject every node whose slab holds the origin (axis-aligned subsurface probes: -N0 of a face normal (0, 0, 1) is (-0, -0, -1)).
    const bool nx = d.x < 0, ny = d.y < 0, nz = d.z < 0;
    r.idir.x = 1.f / (fabsf(d.x) > eps ? d.x : (nx ? -eps : eps));
    r.idir.y = 1.f / (fabsf(d.y) > eps ? d.y : (ny ? -eps : eps));
    r.idir.z = 1.f / (fabsf(d.z) > eps ? d.z : (nz ? -eps : eps));
    const uint32_t oinv = (nx ? 0u : 4u) | (ny ? 0u : 2u) | (nz ? 0u : 1u);
    // children are visited in descending (slot ^ oinv): first the half of the slots whose bit 2 differs from oinv's, ...
    r.oct_inv4 = oinv | ((oinv & 4u) ? 0x0f00u : 0xf000u) | ((oinv & 2u) ? 0x330000u : 0xcc0000u) | ((oinv & 1u) ? 0x55000000u : 0xaa000000u);
    return r;
}

// Alpha callback data: uv + group + object of a triangle, and the material table (see ptb_scene.h).
struct AlphaCtx;
PTB_HD bool alpha_rejects(const AlphaCtx* ctx, int prim, float b1, float b2);
// Triangle::intersection (TriangleMesh.h:82-104) in the reference's own arithmetic: object-space ray, plane + Gram barycentrics, every
// operation rounded separately (ptb_scene.h).  Decides the hits the fast test below cannot call: rays within PTB_EDGE_EPS of an edge.
PTB_HD bool tri_exact_available(const AlphaCtx* ctx);
PTB_HD_NOINLINE bool tri_exact(const AlphaCtx* ctx, int prim, V3 o, V3 d, float tbest, float& t, float& b1, float& b2);   // out of line: the hot loop keeps its registers

// Tests the 8 children of `n` against the ray; returns the hit mask in SLOT order: bit 24 + s = the internal child in slot s,
// bits 3s..3s+2 = the triangles of the leaf in slot s (only bits that exist: valid24 / imask).
#if defined(__CUDA_ARCH__)
// Device form.  ncu on the straightforward form showed the XU pipe (48 I2F.U8 per node) as the busiest pipe, so the
// quantised planes are turned into floats without any conversion instruction (see planes4 below) and the bias is folded
// into the FFMA constant.
// Both the fma pipe (FFMA, HADD2, IMAD) and the alu pipe (PRMT, FMNMX, LOP3, SHF, SEL, ISETP) issue one warp instruction
// every 2 cycles per SM sub-partition; the node test is bound by the alu pipe (about 116 alu vs 96 fma instructions per node).
// One PRMT (alu) builds a half2 {1024+q0, 1024+q1} (0x6400 | q) for TWO planes and HADD2.F32 (fma pipe) widens each;
// the bias folds into the FFMA constant: t = (1024+q)*ad + (bo - 1024*ad), at most 2^-24 * 1024 = 6e-5 of a cell of rounding.
#define PTB_PLANE_BIAS 1024.f
__device__ __forceinline__ void planes4(uint32_t w, float ad, float bo, float& t0, float& t1, float& t2, float& t3) {
    const uint32_t h01 = __byte_perm(w, 0x64646464u, 0x4140), h23 = __byte_perm(w, 0x64646464u, 0x4342);
    const __half2 a = *reinterpret_cast<const __half2*>(&h01), b = *reinterpret_cast<const __half2*>(&h23);
    t0 = fmaf(__low2float(a), ad, bo); t1 = fmaf(__high2float(a), ad, bo);
    t2 = fmaf(__low2float(b), ad, bo); t3 = fmaf(__high2float(b), ad, bo);
}
__device__ __forceinline__ uint32_t node_hitmask(const F4& n0, const F4& n1, const F4& n2, const F4& n3, const F4& n4, const RayPrep& r, float tmax) {
    const uint32_t e_imask = f2u(n0.w);
    const float sx = u2f(((e_imask >> 0) & 0xffu) << 23), sy = u2f(((e_imask >> 8) & 0xffu) << 23), sz = u2f(((e_imask >> 16) & 0xffu) << 23);
    const float adx = sx * r.idir.x, ady = sy * r.idir.y, adz = sz * r.idir.z;
    const float box = fmaf(-PTB_PLANE_BIAS, adx, (n0.x - r.o.x) * r.idir.x), boy = fmaf(-PTB_PLANE_BIAS, ady, (n0.y - r.o.y) * r.idir.y),
                boz = fmaf(-PTB_PLANE_BIAS, adz, (n0.z - r.o.z) * r.idir.z);
    const bool negx = r.d.x < 0, negy = r.d.y < 0, negz = r.d.z < 0;
    // The mask is built in SLOT order with immediates (slot s: its three triangle bits and its internal-child bit) and cut down to
    // what exists with one AND; the octant order is applied when a child is picked (pick_slot).  The per-child byte extracts and
    // variable shifts of a traversal-ordered mask were a quarter of the node step's instructions.
    uint32_t hitmask = 0;
#pragma unroll
    for (int half = 0; half < 2; half++) {
        const uint32_t lox = f2u(half ? n2.y : n2.x), loy = f2u(half ? n2.w : n2.z), loz = f2u(half ? n3.y : n3.x);
        const uint32_t hix = f2u(half ? n3.w : n3.z), hiy = f2u(half ? n4.y : n4.x), hiz = f2u(half ? n4.w : n4.z);
        float tnx[4], tny[4], tnz[4], tfx[4], tfy[4], tfz[4];
        planes4(negx ? hix : lox, adx, box, tnx[0], tnx[1], tnx[2], tnx[3]);
        planes4(negx ? lox : hix, adx, box, tfx[0], tfx[1], tfx[2], tfx[3]);
        planes4(negy ? hiy : loy, ady, boy, tny[0], tny[1], tny[2], tny[3]);
        planes4(negy ? loy : hiy, ady, boy, tfy[0], tfy[1], tfy[2], tfy[3]);
        planes4(negz ? hiz : loz, adz, boz, tnz[0], tnz[1], tnz[2], tnz[3]);
        planes4(negz ? loz : hiz, adz, boz, tfz[0], tfz[1], tfz[2], tfz[3]);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const float tn = fmaxf(fmaxf(tnx[j], tny[j]), fmaxf(tnz[j], 0.f));
            const float tf = fminf(fminf(tfx[j], tfy[j]), fminf(tfz[j], tmax));
            const int s = 4 * half + j;
            if (tn <= tf) hitmask |= (7u << (3 * s)) | (1u << (24 + s));
        }
    }
    return hitmask & ((e_imask & 0xff000000u) | (f2u(n1.z) & 0x00ffffffu));
}
#else
inline uint32_t node_hitmask(const F4& n0, const F4& n1, const F4& n2, const F4& n3, const F4& n4, const RayPrep& r, float tmax) {
    const uint32_t e_imask = f2u(n0.w);
    const float sx = u2f(((e_imask >> 0) & 0xffu) << 23), sy = u2f(((e_imask >> 8) & 0xffu) << 23), sz = u2f(((e_imask >> 16) & 0xffu) << 23);
    const float adx = sx * r.idir.x, ady = sy * r.idir.y, adz = sz * r.idir.z;
    const float box = (n0.x - r.o.x) * r.idir.x, boy = (n0.y - r.o.y) * r.idir.y, boz = (n0.z - r.o.z) * r.idir.z;
    const uint32_t qlox_lo = f2u(n2.x), qlox_hi = f2u(n2.y), qloy_lo = f2u(n2.z), qloy_hi = f2u(n2.w);
    const uint32_t qloz_lo = f2u(n3.x), qloz_hi = f2u(n3.y), qhix_lo = f2u(n3.z), qhix_hi = f2u(n3.w);
    const uint32_t qhiy_lo = f2u(n4.x), qhiy_hi = f2u(n4.y), qhiz_lo = f2u(n4.z), qhiz_hi = f2u(n4.w);
    const bool negx = r.d.x < 0, negy = r.d.y < 0, negz = r.d.z < 0;
    uint32_t hitmask = 0;
    for (int half = 0; half < 2; half++) {
        const uint32_t lox = half ? qlox_hi : qlox_lo, loy = half ? qloy_hi : qloy_lo, loz = half ? qloz_hi : qloz_lo;
        const uint32_t hix = half ? qhix_hi : qhix_lo, hiy = half ? qhiy_hi : qhiy_lo, hiz = half ? qhiz_hi : qhiz_lo;
        // entry plane is lo for positive direction, hi for negative
        const uint32_t nx = negx ? hix : lox, fx = negx ? lox : hix;
        const uint32_t ny = negy ? hiy : loy, fy = negy ? loy : hiy;
        const uint32_t nz = negz ? hiz : loz, fz = negz ? loz : hiz;
        for (int j = 0; j < 4; j++) {
            const uint32_t sh = 8u * j;
            const float tnx = (float)((nx >> sh) & 0xffu) * adx + box;
            const float tny = (float)((ny >> sh) & 0xffu) * ady + boy;
            const float tnz = (float)((nz >> sh) & 0xffu) * adz + boz;
            const float tfx = (float)((fx >> sh) & 0xffu) * adx + box;
            const float tfy = (float)((fy >> sh) & 0xffu) * ady + boy;
            const float tfz = (float)((fz >> sh) & 0xffu) * adz + boz;
            const float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, 0.f));
            const float tf = fminf(fminf(tfx, tfy), fminf(tfz, tmax));
            const int s = 4 * half + j;
            if (tn <= tf) hitmask |= (7u << (3 * s)) | (1u << (24 + s));   // slot s: its triangle bits and its internal-child bit
        }
    }
    return hitmask & ((e_imask & 0xff000000u) | (f2u(n1.z) & 0x00ffffffu));   // what exists: imask, valid24
}
#endif


// Barycentric band around the triangle's edges inside which the fast test defers to tri_exact.  The fast test works on world-space
// float vertices, the reference on object-space ones: their barycentrics differ by up to a few 1e-5 (coordinates of magnitude 50
// against edges of 0.1), so a ray that close to an edge can land on either side.  A ray near a SHARED edge is near it in both
// triangles, so both get the reference's t and the reference's accept decision, and the nearer one wins as it does there.
#if !defined(PTB_EDGE_EPS)
#define PTB_EDGE_EPS 5e-4f
#endif

// Möller–Trumbore on {v0,e1,e2}, two-sided: the distance tt, the barycentrics u, v and m = min(u, v, 1-u-v).  False when the ray
// misses the triangle grown by PTB_EDGE_EPS, meets it behind the origin or clearly beyond the best hit (c.w = PTB_TRI_T_CUT: t of
// this formulation and of the reference's differs in the last bits; 0 on the covering triangles of a volume, whose own hit may be
// nearer than the face the ray crosses).  Written so that NaN (degenerate triangle, det == 0) fails every test.
PTB_HD bool tri_test_front(const F4& a, const F4& b, const F4& c, const RayPrep& r, float tbest, float& tt, float& u, float& v, float& m) {
    const V3 v0 = v3(a.x, a.y, a.z), e1 = v3(b.x, b.y, b.z), e2 = v3(c.x, c.y, c.z);
    const V3 pvec = cross(r.d, e2);
    const float det = dot(e1, pvec);
#if defined(__CUDA_ARCH__)
    // one MUFU.RCP instead of the IEEE division sequence (9 instructions + a slow path): the signs of u, v, t and hence every
    // accept test but the last ulp of `1-u-v >= 0` and `t < tbest` are unaffected; |det| below 1.2e-38 flushes to a miss.
    float inv;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(det));
#else
    const float inv = 1.f / det;
#endif
    const V3 tvec = r.o - v0;
    u = dot(tvec, pvec) * inv;
    const V3 qvec = cross(tvec, e1);
    v = dot(r.d, qvec) * inv;
    tt = dot(e2, qvec) * inv;
    m = fminf(fminf(u, v), 1.f - u - v);
    // same instruction count as a plain accept test for the common outcome (a miss): one min3 and three compares
    return m >= -PTB_EDGE_EPS && tt >= 0.f && tt * c.w < tbest;
}

// Accepts b1,b2 >= 0, b1+b2 <= 1, 0 <= t < tbest.  Near an edge, or on an alpha-tested triangle (b.w = PTB_EDGE_EPS, or +inf when
// the texel the uv lands on must be the reference's), the reference's arithmetic decides.
PTB_HD bool tri_test(const F4& a, const F4& b, const F4& c, const RayPrep& r, float tbest, float& t, float& b1, float& b2, const AlphaCtx* ex, int prim) {
    float tt, u, v, m;
    if (!tri_test_front(a, b, c, r, tbest, tt, u, v, m)) return false;
    if (m < b.w && tri_exact_available(ex)) return tri_exact(ex, prim, r.o, r.d, tbest, t, b1, b2);
    if (!(m >= 0.f) || !(tt < tbest)) return false;
    t = tt; b1 = u; b2 = v;
    return true;
}

// The same test for the persistent traversal kernel (k_trace), which must not carry tri_exact's registers through its hot loop:
// returns 0 miss, 1 hit (t, b1, b2 set), 2 "the reference's arithmetic has to decide" (a ray within PTB_EDGE_EPS of an edge, or an
// alpha-mapped triangle, whose texel must be the reference's).  k_trace pushes case 2 on the traversal stack as a deferred
// candidate and runs tri_exact when it pops it (a few node visits later: t_best is simply not shrunk in the meantime).
PTB_HD int tri_test_classify(const F4& a, const F4& b, const F4& c, const RayPrep& r, float tbest, float& t, float& b1, float& b2) {
    float tt, u, v, m;
    if (!tri_test_front(a, b, c, r, tbest, tt, u, v, m)) return 0;
    if (m < b.w) return 2;            // b.w = PTB_EDGE_EPS, or +inf on alpha-tested triangles
    if (!(tt < tbest)) return 0;
    t = tt; b1 = u; b2 = v;
    return 1;
}

// The hit internal child (bits 24..31 of a node group, slot order) that the ray meets first: the slot s with the largest s ^ oinv.
// Three narrowing steps: keep the preferred half / pairs / slots whenever one of them is hit.
PTB_HD uint32_t pick_slot(uint32_t hits8, uint32_t oct_inv4) {
    uint32_t x = hits8, t;
    t = x & (oct_inv4 >> 8) & 0xffu;  x = t ? t : x;
    t = x & (oct_inv4 >> 16) & 0xffu; x = t ? t : x;
    t = x & (oct_inv4 >> 24);         x = t ? t : x;
    return highest_bit(x);            // one bit is left
}

// Traversal stack entries per ray.  A node step pushes at most two entries (the node's other hit children and the triangle group it
// postpones), so a BVH8 of `depth` wide levels needs at most 2 * depth; ptb_commit refuses deeper trees (PTB_ERR_UNSUPPORTED) instead
// of dropping subtrees the way a full stack would (the reference's own 50-entry stack overflows silently, TriangleMesh.cpp:1158).
#if !defined(PTB_STACK)
#define PTB_STACK 64
#endif

struct TraverseCounters {
    uint32_t nodes, tris;
};

// Node `i` of the BVH (5 x LDG.128) and triangle `i` of the leaf-ordered triangle array (3 x LDG.128).
PTB_HD void load_node(const F4* __restrict__ nodes, uint32_t i, F4& n0, F4& n1, F4& n2, F4& n3, F4& n4) {
    const F4* np = nodes + (size_t)i * 5;
    const auto l0 = PTB_LDG_F4(np + 0), l1 = PTB_LDG_F4(np + 1), l2 = PTB_LDG_F4(np + 2), l3 = PTB_LDG_F4(np + 3), l4 = PTB_LDG_F4(np + 4);
    n0.x = l0.x; n0.y = l0.y; n0.z = l0.z; n0.w = l0.w; n1.x = l1.x; n1.y = l1.y; n1.z = l1.z; n1.w = l1.w;
    n2.x = l2.x; n2.y = l2.y; n2.z = l2.z; n2.w = l2.w; n3.x = l3.x; n3.y = l3.y; n3.z = l3.z; n3.w = l3.w;
    n4.x = l4.x; n4.y = l4.y; n4.z = l4.z; n4.w = l4.w;
}
PTB_HD void load_tri(const F4* __restrict__ tris, uint32_t i, F4& a, F4& b, F4& c) {
    const F4* tp = tris + (size_t)i * 3;
    const auto l0 = PTB_LDG_F4(tp + 0), l1 = PTB_LDG_F4(tp + 1), l2 = PTB_LDG_F4(tp + 2);
    a.x = l0.x; a.y = l0.y; a.z = l0.z; a.w = l0.w; b.x = l1.x; b.y = l1.y; b.z = l1.z; b.w = l1.w;
    c.x = l2.x; c.y = l2.y; c.z = l2.z; c.w = l2.w;
}

// What the walk does with an accepted triangle (alpha-mapped hits already rejected): keep the nearest, stop at the first one that is
// not a ghost's (Scene::intersection_shadow semantics: the caller passes tmax = 0.999*dist_light, TriangleMesh.cpp:1239-1319 +
// Geometry.cpp:735), or hand every one with 0 <= t < tmax to a visitor.
enum { WALK_CLOSEST, WALK_ANY, WALK_ALL };
template <int MODE, bool COUNT, class F>
PTB_HD bool walk(const F4* __restrict__ nodes, const F4* __restrict__ tris, const AlphaCtx* actx, V3 o, V3 d, float tmax,
                 Hit& hit, TraverseCounters* cnt, F& on_hit) {
    const RayPrep r = ray_prep(o, d);
    U2 stack[PTB_STACK];
    int sp = 0;
    U2 ngroup, tgroup;
    uint32_t tvalid = 0;
    // the root enters as a one-child group: bit 31 set, no imask bits -> relative index 0
    ngroup.x = 0; ngroup.y = 0x80000000u;
    bool found = false;
    float tbest = tmax;
    for (;;) {
        // invariant: ngroup has at least one pending internal child (a bit in 31..24)
        {
            const uint32_t hits_imask = ngroup.y;
            const uint32_t slot = pick_slot(hits_imask >> 24, r.oct_inv4);
            const uint32_t child_base = ngroup.x;
            ngroup.y &= ~(1u << (24u + slot));
            if (ngroup.y > 0x00ffffffu) {
                if (sp < PTB_STACK) stack[sp++] = ngroup;
            }
            const uint32_t rel = popcount32(hits_imask & ~(0xffffffffu << slot));
            F4 n0, n1, n2, n3, n4;
            load_node(nodes, child_base + rel, n0, n1, n2, n3, n4);
            if (COUNT) cnt->nodes++;
            const uint32_t hm = node_hitmask(n0, n1, n2, n3, n4, r, tbest);
            ngroup.x = f2u(n1.x);
            tgroup.x = f2u(n1.y);
            ngroup.y = (hm & 0xff000000u) | (f2u(n0.w) >> 24);
            tgroup.y = hm & 0x00ffffffu;
            tvalid = f2u(n1.z) & 0x00ffffffu;
        }
        while (tgroup.y != 0) {
            const uint32_t ti = highest_bit(tgroup.y);
            tgroup.y &= ~(1u << ti);
            const uint32_t prim = tgroup.x + popcount32(tvalid & ~(0xffffffffu << ti));
            F4 a, b, c;
            load_tri(tris, prim, a, b, c);
            if (COUNT) cnt->tris++;
            float t, b1, b2;
            if (tri_test(a, b, c, r, tbest, t, b1, b2, actx, (int)prim)) {
                if ((f2u(a.w) & PTB_TRI_FLAG_ALPHA) && alpha_rejects(actx, (int)prim, b1, b2)) continue;
                if (MODE == WALK_ALL) { on_hit((int32_t)prim, t, b1, b2); continue; }
                if (MODE == WALK_ANY && (f2u(a.w) & PTB_TRI_FLAG_GHOST)) continue;
                tbest = t;
                hit.t = t; hit.b1 = b1; hit.b2 = b2; hit.prim = (int32_t)prim;
                found = true;
                if (MODE == WALK_ANY) return true;
            }
        }
        if (ngroup.y <= 0x00ffffffu) {
            if (sp > 0) ngroup = stack[--sp];
            else break;
        }
    }
    return found;
}

struct NoVisitor {
    PTB_HD void operator()(int32_t, float, float, float) {}
};
// The closest hit with t < tmax, or (ANY_HIT) the first accepted triangle that is not a ghost's.
template <bool ANY_HIT, bool COUNT>
PTB_HD bool traverse(const F4* __restrict__ nodes, const F4* __restrict__ tris, const AlphaCtx* actx, V3 o, V3 d, float tmax,
                     Hit& hit, TraverseCounters* cnt) {
    NoVisitor none;
    return walk<ANY_HIT ? WALK_ANY : WALK_CLOSEST, COUNT>(nodes, tris, actx, o, d, tmax, hit, cnt, none);
}

// Every accepted triangle with 0 <= t < tmax, in traversal order: `on_hit(prim, t, b1, b2)`.  Used by the subsurface probe
// (TriMesh::reservoir_sampling_intersection, TriangleMesh.cpp:1321-1424), which is not a hot path.
template <class F>
PTB_HD void traverse_all(const F4* __restrict__ nodes, const F4* __restrict__ tris, const AlphaCtx* actx, V3 o, V3 d, float tmax, F& on_hit) {
    Hit unused;
    walk<WALK_ALL, false>(nodes, tris, actx, o, d, tmax, unused, nullptr, on_hit);
}

}  // namespace ptb
