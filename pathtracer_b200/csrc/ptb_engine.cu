// ptb_engine.cu — CUDA kernels (sm_100a) of the wavefront radiance loop, their launch schedule, and the
// C-ABI of include/ptb200.h.
//
// One render = passes over the shard's pixels; one pass keeps `pool` paths in flight in HBM (SoA, ptb_scene.h
// PoolDev) and runs, on one stream with no host synchronisation:
//     k_raygen -> [ k_trace<closest> -> k_exact -> k_shade -> k_trace<any-hit> -> k_exact ] x nb_bounces -> k_splat
// Queues are index lists compacted with warp ballots + one atomic per warp (k_shade); every kernel reads
// its element count from device memory, so the host never waits for a count.
// There is no CPU implementation behind this ABI: a missing device or a failed launch is an error code.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>
#include <omp.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "ptb_host.h"

using namespace ptb;

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            c->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                 \
            return PTB_ERR_CUDA;                                                                         \
        }                                                                                                \
    } while (0)

// counters layout (uint32), zeroed at the start of every pass:
//   [2*b] paths queued for bounce b          [2*b+1] shadow rays queued for the BVH at bounce b
//   [CUR + 2*b] / [CUR + 2*b+1]  work cursors of the persistent trace kernels (closest / any-hit) of bounce b
//   [SQ + b]  intersection_shadow-equivalent queries made at bounce b (ray statistics)
#define PTB_CNT_CUR (2 * (PTB_MAX_BOUNCES + 1))
#define PTB_CNT_SQ (4 * (PTB_MAX_BOUNCES + 1))
#define PTB_CNT_ALLOC (5 * (PTB_MAX_BOUNCES + 1))       // branching renders: side-branch slots handed out in this pass
#define PTB_CNT_DROPS (5 * (PTB_MAX_BOUNCES + 1) + 1)   // side branches that found the pool full
#define PTB_CNT_PROBE (5 * (PTB_MAX_BOUNCES + 1) + 2)   // subsurface probes emitted at the current level
#define PTB_CNT_DEFER (5 * (PTB_MAX_BOUNCES + 1) + 3)   // [+ 2*b] / [+ 2*b + 1]: rays of bounce b (closest / any-hit) that left candidates for k_exact
#define PTB_N_COUNTERS (7 * (PTB_MAX_BOUNCES + 1) + 3)
// 64-bit totals: 0 closest rays, 1 shadow rays, 2/3 node visits / triangle tests of the closest-hit trace, 4/5 of the any-hit trace
#define PTB_N_TOTALS 10   /* 0-1 rays, 2-5 node visits / triangle tests (closest, any hit), 6-9 triangle-phase warp iterations and their packed minimum (COUNT kernels) */

// ------------------------------------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(256) k_rpp(float* rpp, int n) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    float x, y;
    random_per_pixel((uint32_t)p, x, y);
    rpp[2 * p] = x;
    rpp[2 * p + 1] = y;
}

template <bool EXOTIC>
__global__ void __launch_bounds__(256) k_raygen(SceneDev sc, FrameDev f, PoolDev p, int n_paths) {
    const int path = blockIdx.x * blockDim.x + threadIdx.x;
    if (path >= n_paths) return;
    raygen_one<EXOTIC>(sc, f, p, path);
}

// ---- BVH8 traversal: persistent warps, dynamic ray fetch, postponed triangle tests -------------------------------------
// Replaces TriMesh::intersection / intersection_shadow (TriangleMesh.cpp:1133-1319).  One thread per ray diverges badly
// (ncu on the 2.5M-triangle scene: 7-10 of 32 lanes active per instruction), so the warp is kept busy instead:
//   * a lane whose ray has finished pulls the next queue entry (one atomic per warp) once fewer than `refill_below`
//     lanes are live (Aila & Laine 2009, persistent threads);
//   * every iteration of the warp loop is: [stack pop or finish] -> [ONE node step for lanes with node work] ->
//     [triangle steps while at least 1/tri_den of the live lanes take part]; triangles left over are postponed by pushing
//     the triangle group on the traversal stack (Ylitie et al. 2017, sec. 4).
// ANY_HIT = shadow rays (queue = shadow entries, first accepted triangle ends the ray; an unoccluded ray adds its deferred
// direct term to the path's radiance).  Closest-hit results overwrite the analytic hit record the ray's producer wrote.
template <bool ANY_HIT, bool COUNT, bool BRANCH = false>
__global__ void __launch_bounds__(128) k_trace(SceneDev sc, PoolDev p, const uint32_t* __restrict__ queue, const uint32_t* __restrict__ count,
                                               int n_static, uint32_t* cursor, unsigned long long* totals, int refill_below, int tri_den, int tri_min_pct,
                                               uint32_t* defer_count) {
    const uint32_t FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    // pick_slot as a table: slot = lut[7 - octant][hit internal children] (2 KB of shared memory, filled once per persistent block):
    // one LDS instead of thirteen ALU instructions per node visit (+1.2 % on C2 / C3, profiles/r01p_ab_pick_lut.txt)
    __shared__ uint8_t pick_lut[8 * 256];
    for (uint32_t i = threadIdx.x; i < 8u * 256u; i += blockDim.x) {
        const uint32_t oinv = i >> 8;
        const uint32_t packed = oinv | ((oinv & 4u) ? 0x0f00u : 0xf000u) | ((oinv & 2u) ? 0x330000u : 0xcc0000u) | ((oinv & 1u) ? 0x55000000u : 0xaa000000u);
        pick_lut[i] = (i & 0xffu) ? (uint8_t)pick_slot(i & 0xffu, packed) : (uint8_t)0;
    }
    __syncthreads();
    const uint32_t n = count ? *count : (uint32_t)n_static;
    const F4* __restrict__ nodes = sc.nodes;
    const F4* __restrict__ tris = sc.tris;
    bool live = false, exhausted = false;
    uint32_t item = 0, entry = 0;
    RayPrep r;
    float tbest = 0.f, hb1 = 0.f, hb2 = 0.f;
    int32_t hprim = -1;
    U2 ngroup, tgroup;
    U2 lstack[PTB_STACK];   // traversal stack (local memory)
    // candidates the ray has left for k_exact (tri_test_classify case 2) are counted in a register the variant has no other use for:
    // `entry` for closest-hit rays, `hprim` for any-hit rays
    uint32_t tvalid = 0;   // valid24 of the node the live triangle group came from (all ones for a group popped from the stack: compact bits)
    int sp = 0;
    ngroup.x = ngroup.y = tgroup.x = tgroup.y = 0;
    uint32_t cn = 0, ct = 0;
    uint32_t w_iters = 0, w_ideal = 0;   // COUNT: triangle-phase iterations of this warp, and how few would do if its tests were packed 32 to an iteration
    r.o = r.d = r.idir = v3(0, 0, 0); r.oct_inv4 = 0;
    for (;;) {
        // ---- refill idle lanes from the queue
        const uint32_t live_mask = __ballot_sync(FULL, live);
        if (!exhausted && __popc(live_mask) < refill_below) {
            const uint32_t idle = ~live_mask;
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(cursor, (uint32_t)__popc(idle));
            base = __shfl_sync(FULL, base, 0);
            if (!live) {
                const uint32_t qi = base + (uint32_t)__popc(idle & ((1u << lane) - 1u));
                if (qi < n) {
                    F4 o, d;
                    float tmax;
                    bool ok = true;
                    if (ANY_HIT) { entry = qi; o = p.sh_o[qi]; d = p.sh_d[qi]; tmax = o.w; }
                    else {
                        item = queue ? queue[qi] : qi;
                        ok = p.pixel[item] != 0xffffffffu;
                        o = p.ray_o[item]; d = p.ray_d[item]; tmax = p.hit[item].x;
                    }
                    if (ok) {
                        r = ray_prep(v3(o.x, o.y, o.z), v3(d.x, d.y, d.z));
                        tbest = tmax; hprim = ANY_HIT ? 0 : -1; sp = 0;
                        if (!ANY_HIT) entry = 0;
                        ngroup.x = 0; ngroup.y = 0x80000000u; tgroup.x = 0; tgroup.y = 0;
                        if (ANY_HIT) item = f2u(d.w);   // the path the shadow ray belongs to
                        live = true;
                    }
                }
            }
            if (base + (uint32_t)__popc(idle) >= n) exhausted = true;
        }
        if (__ballot_sync(FULL, live) == 0) {
            if (exhausted) break;
            continue;
        }
        // ---- pop / finish: lanes with neither node nor triangle work
        if (live && ngroup.y <= 0x00ffffffu && tgroup.y == 0) {
            if (sp > 0) {
                const U2 e = lstack[--sp];
                if (e.y > 0x00ffffffu) ngroup = e; else { tgroup = e; tvalid = 0x00ffffffu; }
            } else {
                // candidates left for k_exact: it finishes the ray (the nearest of them may beat the hit found here; a shadow ray is only
                // unoccluded if none of them blocks it)
                const uint32_t nd = ANY_HIT ? (uint32_t)hprim : entry;
                if (nd) {
                    const uint32_t qi = atomicAdd(defer_count, 1u);
                    U2 dr; dr.x = ANY_HIT ? entry : item; dr.y = nd;
                    p.defer_rays[qi] = dr;
                }
                if (!ANY_HIT) { if (hprim >= 0) p.hit[item] = hit_record(Hit{tbest, hb1, hb2, hprim}); }
                else if (!nd) {   // unoccluded (a ray that left candidates is delivered or settled by k_exact)
                    if (BRANCH) shadow_settle_branch(p, (int)entry, item, false);
                    else deliver_direct(p, entry, item);
                }
                live = false;
            }
        }
        // ---- node phase: ONE node step
        if (live && ngroup.y > 0x00ffffffu) {
            if (tgroup.y != 0) {   // postpone leftover triangles: stacked in compact form (bit = index relative to tri_base)
                uint32_t m = tgroup.y, cm = 0;
                do {
                    const uint32_t b = highest_bit(m);
                    m &= ~(1u << b);
                    cm |= 1u << popcount32(tvalid & ~(0xffffffffu << b));
                } while (m);
                tgroup.y = cm;
                lstack[sp++] = tgroup;   // never full: ptb_commit refuses trees deeper than PTB_STACK / 2
                tgroup.y = 0;
            }
            const uint32_t hits_imask = ngroup.y;
            const uint32_t slot = pick_lut[((r.oct_inv4 & 7u) << 8) | (hits_imask >> 24)];
            const uint32_t child_base = ngroup.x;
            ngroup.y &= ~(1u << (24u + slot));
            if (ngroup.y > 0x00ffffffu) lstack[sp++] = ngroup;
            const uint32_t rel = popcount32(hits_imask & ~(0xffffffffu << slot));
            F4 n0, n1, n2, n3, n4;
            load_node(nodes, child_base + rel, n0, n1, n2, n3, n4);
            if (COUNT) cn++;
            const uint32_t hm = node_hitmask(n0, n1, n2, n3, n4, r, tbest);
            ngroup.x = f2u(n1.x);
            tgroup.x = f2u(n1.y);
            ngroup.y = (hm & 0xff000000u) | (f2u(n0.w) >> 24);
            tgroup.y = hm & 0x00ffffffu;
            tvalid = f2u(n1.z) & 0x00ffffffu;
        }
        // ---- triangle phase: entered when tri_min_pct % of the live lanes hold triangle work (default 0: always; postponing
        //      further was measured to cost more node visits than it saves issue slots) or when nobody can do anything else;
        //      repeats while >= 1/tri_den of the live lanes take part.
        uint32_t tm = __ballot_sync(FULL, live && tgroup.y != 0);
        const int live_n = __popc(__ballot_sync(FULL, live));
        // (when no live lane can do anything else, every live lane holds triangles and the quorum is met: tri_min_pct <= 100)
        if (tm != 0 && __popc(tm) * 100 >= tri_min_pct * live_n) {
            uint32_t phase_tests = 0;
            do {
                if (COUNT) { w_iters++; phase_tests += (uint32_t)__popc(tm); }
                if (live && tgroup.y != 0) {
                    const uint32_t ti = highest_bit(tgroup.y);
                    tgroup.y &= ~(1u << ti);
                    const uint32_t prim = tgroup.x + popcount32(tvalid & ~(0xffffffffu << ti));
                    F4 a, b, c;
                    load_tri(tris, prim, a, b, c);
                    if (COUNT) ct++;
                    float t, b1, b2;
                    const int res = tri_test_classify(a, b, c, r, tbest, t, b1, b2);
                    if (res == 2) {            // near an edge / alpha-tested / a disc: left for k_exact (the reference's own arithmetic)
                        const uint32_t nd = ANY_HIT ? (uint32_t)hprim : entry;
                        if (nd < PTB_DEFER_K) p.defer_prims[(size_t)(ANY_HIT ? entry : item) * PTB_DEFER_K + nd] = prim | ((f2u(a.w) & 7u) << 28);
                        if (ANY_HIT) hprim++; else entry++;
                    } else if (res == 1) {
                        if (!(ANY_HIT && (f2u(a.w) & PTB_TRI_FLAG_GHOST))) {     // (alpha-tested triangles always take the deferred route)
                            if (ANY_HIT) { live = false; tgroup.y = 0; if (BRANCH) shadow_settle_branch(p, (int)entry, item, true); }   // occluded: nothing to deliver
                            else { tbest = t; hb1 = b1; hb2 = b2; hprim = (int32_t)prim; }
                        }
                    }
                }
                tm = __ballot_sync(FULL, live && tgroup.y != 0);
            } while (__popc(tm) * tri_den >= live_n && tm != 0);
            if (COUNT) w_ideal += (phase_tests + 31u) >> 5;
        }
    }
    if (COUNT) {
        for (int o = 16; o > 0; o >>= 1) { cn += __shfl_down_sync(FULL, cn, o); ct += __shfl_down_sync(FULL, ct, o); }
        if (lane == 0 && (cn | ct)) { atomicAdd(&totals[ANY_HIT ? 4 : 2], (unsigned long long)cn); atomicAdd(&totals[ANY_HIT ? 5 : 3], (unsigned long long)ct); }
        if (lane == 0 && w_iters) { atomicAdd(&totals[ANY_HIT ? 8 : 6], (unsigned long long)w_iters); atomicAdd(&totals[ANY_HIT ? 9 : 7], (unsigned long long)w_ideal); }
    }
}

// ---- k_exact: the candidates k_trace could not call (tri_test_classify case 2) ---------------------------------------------------------
// A ray within PTB_EDGE_EPS (barycentric) of a triangle edge, an alpha-tested triangle or a point-set disc is decided by the
// reference's own arithmetic (tri_exact, ptb_scene.h).  k_trace keeps that code out of its loop: it leaves up to PTB_DEFER_K candidates
// per ray in `defer_prims` and the ray in `defer_rays`; here one thread finishes one such ray: the nearest accepted candidate replaces
// the hit k_trace found if it is nearer (closest hit), or blocks the shadow ray, which otherwise delivers its direct term (any hit).
// About one ray in two hundred comes through here; a ray that left more than PTB_DEFER_K candidates is re-traced with the immediate test.
template <bool ANY_HIT, bool BRANCH>
__global__ void __launch_bounds__(128) k_exact(SceneDev sc, PoolDev p, const uint32_t* __restrict__ defer_count) {
    const uint32_t n = *defer_count;
    const AlphaCtx ac = alpha_ctx(sc);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const U2 e = p.defer_rays[i];
        const uint32_t ref = e.x, nd = e.y;
        uint32_t item;
        F4 o, d;
        float tbest;
        F4 best; best.x = best.y = best.z = best.w = 0;
        if (ANY_HIT) { o = p.sh_o[ref]; d = p.sh_d[ref]; tbest = o.w; item = f2u(d.w); }
        else { item = ref; o = p.ray_o[item]; d = p.ray_d[item]; best = p.hit[item]; tbest = best.x; }
        const V3 ro = v3(o.x, o.y, o.z), rd = v3(d.x, d.y, d.z);
        bool found = false;
        if (nd > PTB_DEFER_K) {
            Hit h;
            if (traverse<ANY_HIT, false>(sc.nodes, sc.tris, &ac, ro, rd, tbest, h, nullptr)) { found = true; best = hit_record(h); }
        } else {
            for (uint32_t k = 0; k < nd; k++) {
                const uint32_t w = p.defer_prims[(size_t)ref * PTB_DEFER_K + k], prim = w & 0x0fffffffu, fl = w >> 28;
                float t, b1, b2;
                if (!tri_exact(&ac, (int)prim, ro, rd, tbest, t, b1, b2)) continue;
                if ((fl & PTB_TRI_FLAG_ALPHA) && alpha_rejects(&ac, (int)prim, b1, b2)) continue;
                if (ANY_HIT && (fl & PTB_TRI_FLAG_GHOST)) continue;
                tbest = t; found = true;
                best = hit_record(Hit{t, b1, b2, (int32_t)prim});
                if (ANY_HIT) break;
            }
        }
        if (ANY_HIT) {
            if (BRANCH) shadow_settle_branch(p, (int)ref, item, found);
            else if (!found) deliver_direct(p, ref, item);   // unoccluded after all
        } else if (found) p.hit[item] = best;
    }
}

// warp-aggregated append: one atomic per warp, lanes take consecutive slots
__device__ __forceinline__ uint32_t warp_push(uint32_t* counter, bool want) {
    const uint32_t mask = __ballot_sync(0xffffffffu, want);
    if (mask == 0) return 0;
    const uint32_t lane = threadIdx.x & 31;
    const int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if ((int)lane == leader) base = atomicAdd(counter, __popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + __popc(mask & ((1u << lane) - 1u));
}

#define PTB_SHADE_BLOCK 256    /* threads per k_shade block: half as many blocks for a later bounce to launch only to see them return (r02w: k_shade -4 % on C2, -3 % on C4 against 128; 512 is no better) */
template <bool MERL, int MINB, bool AOV, bool EXOTIC = false>
__global__ void __launch_bounds__(PTB_SHADE_BLOCK, (MINB * 128) / PTB_SHADE_BLOCK) k_shade(SceneDev sc, FrameDev f, PoolDev p, const uint32_t* __restrict__ queue,
                                               const uint32_t* __restrict__ count, int n_static, uint32_t* __restrict__ next_queue,
                                               uint32_t* next_count, uint32_t* shadow_count, uint32_t* shadow_queries) {
    // one thread per pool slot; the queue length lives in device memory, so after the first bounce most blocks return at once.
    // A bounded grid striding over the live part of the queue was measured (profiles/r01m_ab_prefetch_shadegrid.txt): the loop
    // costs registers the 64-register kernel does not have (spills: +3 % on C2, +25 % with the MERL lookup) and saves nothing.
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = count ? (int)*count : n_static;
    ShadeOut out;
    out.cont = false; out.shadow = false; out.shadow_query = false;
    int path = 0;
    if (tid < n) {
        path = queue ? (int)queue[tid] : tid;
        shade_one<MERL, AOV, EXOTIC>(sc, f, p, path, out);
    }
    // both appends of the warp in one go: lane 0 issues the two returning atomics back to back, so their round trips to L2 overlap
    // (ncu r02t: 6.7 % of the kernel's stall samples sat on the first one's return before the second was even issued)
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t mc = __ballot_sync(0xffffffffu, out.cont), ms = __ballot_sync(0xffffffffu, out.shadow), sq = __ballot_sync(0xffffffffu, out.shadow_query);
    uint32_t bc = 0, bs = 0;
    if (lane == 0) {
        if (mc) bc = atomicAdd(next_count, (uint32_t)__popc(mc));
        if (ms) bs = atomicAdd(shadow_count, (uint32_t)__popc(ms));
        if (sq) atomicAdd(shadow_queries, (uint32_t)__popc(sq));
    }
    bc = __shfl_sync(0xffffffffu, bc, 0); bs = __shfl_sync(0xffffffffu, bs, 0);
    const uint32_t below = (1u << lane) - 1u;
    if (out.cont) next_queue[bc + __popc(mc & below)] = (uint32_t)path;
    if (out.shadow) { const uint32_t si = bs + __popc(ms & below); p.sh_o[si] = out.sh_o; p.sh_d[si] = out.sh_d; p.sh_c[si] = out.sh_c; }
}

// Branching renders (fog, ghost objects, background photograph): one getColor loop iteration per queue entry; side branches
// take fresh pool slots (one atomic per warp and kind) and join the next level's queue next to the continuations.
template <bool MERL>
__global__ void __launch_bounds__(128) k_shade_branch(SceneDev sc, FrameDev f, PoolDev p, const uint32_t* __restrict__ queue, const uint32_t* __restrict__ count,
                                                      int n_static, uint32_t* __restrict__ next_queue, uint32_t* next_count, uint32_t* shadow_count,
                                                      uint32_t* shadow_queries, uint32_t* alloc, uint32_t n_roots, uint32_t cap, uint32_t* drops,
                                                      uint32_t* probe_count, const F4* __restrict__ resume) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = count ? (int)*count : n_static;
    BranchOut out;
    out.base.cont = false; out.base.shadow = false; out.base.shadow_query = false;
    out.fog.want = false; out.ghost.want = false; out.ghost_pending = false; out.probe = false;
    int path = 0;
    uint32_t root = 0, pix = 0;
    if (tid < n) {
        // `resume`: second visit of the hits whose subsurface probe has been answered (the probe entries name the paths)
        path = resume ? (int)f2u(resume[tid].w) : (queue ? (int)queue[tid] : tid);
        root = p.root[path]; pix = p.pixel[path];
        if (pix != 0xffffffffu) shade_branch_one<MERL>(sc, f, p, path, out);
    }
    uint32_t ghost_slot = 0x7fffffffu;
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const ChildOut& ch = k == 0 ? out.fog : out.ghost;
        bool want = ch.want;
        const uint32_t slot = n_roots + warp_push(alloc, want);
        if (want && slot >= cap) { want = false; atomicAdd(drops, 1u); }
        if (want) { store_child(sc, p, slot, ch, root, pix); if (k == 1) ghost_slot = slot; }
        const uint32_t ci = warp_push(next_count, want);
        if (want) next_queue[ci] = slot;
    }
    const uint32_t qi = warp_push(next_count, out.base.cont);
    if (out.base.cont) next_queue[qi] = (uint32_t)path;
    const uint32_t si = warp_push(shadow_count, out.base.shadow);
    if (out.base.shadow) {
        F4 c = out.base.sh_c;
        if (out.ghost_pending) c.w = u2f(0x80000000u | ghost_slot);
        p.sh_o[si] = out.base.sh_o; p.sh_d[si] = out.base.sh_d; p.sh_c[si] = c;
    }
    const uint32_t sq = __ballot_sync(0xffffffffu, out.base.shadow_query);
    if ((threadIdx.x & 31) == 0 && sq) atomicAdd(shadow_queries, (uint32_t)__popc(sq));
    const uint32_t pi = warp_push(probe_count, out.probe);
    if (out.probe) { p.probe_o[pi] = out.probe_o; p.probe_d[pi] = out.probe_d; p.probe_x[pi] = out.probe_x; }
}

// Subsurface probes: one thread per probe, plain stack traversal collecting every hit of a short ray (not a hot path).
__global__ void __launch_bounds__(128) k_probe(SceneDev sc, PoolDev p, int n) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid < n) probe_one(sc, p, tid);
}

struct RedAddV4 {
    __device__ __forceinline__ void operator()(F4* addr, const F4& v) const {
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
    }
};

__global__ void __launch_bounds__(128) k_splat(FrameDev f, PoolDev p, F4* accum) {
    const int ps = blockIdx.x * blockDim.x + threadIdx.x;
    if (ps >= f.n_pixel_slots) return;
    splat_pixel(f, p, ps, accum, RedAddV4());
}

// ---- key-frame refit: a new frame of an animation without a rebuild -------------------------------------------------------------------
// Object::build_matrix(current_frame) moves whole objects rigidly (scale, rotation, translation keys, Geometry.h:322-360).  The BVH8
// keeps its topology; the world-space triangles are re-derived from the object-space corners that live on the device (tris_obj) with
// the roundings of the host's xf_point, and the node boxes are recomputed bottom-up, one launch per level (nodes are stored breadth
// first), with the builder's conservative quantisation (bvh8_build.cpp).  The reference re-poses by changing the matrices only (its BVH
// is in object space); here the re-pose costs one pass over the triangles and the nodes: well under a millisecond per million triangles.
// world-space corners of stored triangle `t` at the objects' current matrices: a mesh triangle's own corners, the covering triangle of a
// point-set disc (centre A, normal B.xyz, radius B.w) or one of the covering triangles of a yarn segment (A, B, radius B.w; which one in
// bits 28..30 of A.w)
__device__ __forceinline__ void refit_corners(const F4* __restrict__ tris_obj, const ObjectDev* __restrict__ objects, size_t t, V3& v0, V3& v1, V3& v2) {
    const F4 A = tris_obj[3 * t], B = tris_obj[3 * t + 1];
    const ObjectDev& ob = objects[f2u(A.w) & 0x0fffffffu];
    const float* m = ob.trans;
    if (ob.type == OBJ_POINTSET) {
        const float sc_ = sqrtf(m[0] * m[0] + m[4] * m[4] + m[8] * m[8]);
        disc_cover_triangle(xf_point_rn(m, v3(A.x, A.y, A.z)), xf_rot(ob.rot, v3(B.x, B.y, B.z)), B.w * sc_, v0, v1, v2);
    } else if (ob.type == OBJ_YARNS) {
        const float sc_ = sqrtf(m[0] * m[0] + m[4] * m[4] + m[8] * m[8]);
        yarn_cover_triangle(xf_point_rn(m, v3(A.x, A.y, A.z)), xf_point_rn(m, v3(B.x, B.y, B.z)), B.w * sc_, (int)(f2u(A.w) >> 28), v0, v1, v2);
    } else {
        const F4 C = tris_obj[3 * t + 2];
        v0 = xf_point_rn(m, v3(A.x, A.y, A.z)); v1 = xf_point_rn(m, v3(B.x, B.y, B.z)); v2 = xf_point_rn(m, v3(C.x, C.y, C.z));
    }
}
__global__ void __launch_bounds__(256) k_refit_tris(const F4* __restrict__ tris_obj, const ObjectDev* __restrict__ objects, F4* tris, size_t n_tri) {
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_tri) return;
    V3 v0, v1, v2;
    refit_corners(tris_obj, objects, k, v0, v1, v2);
    F4 q;
    q.x = v0.x; q.y = v0.y; q.z = v0.z; q.w = tris[3 * k].w; tris[3 * k] = q;                       // .w: the triangle's flags stay
    q.x = v1.x - v0.x; q.y = v1.y - v0.y; q.z = v1.z - v0.z; q.w = tris[3 * k + 1].w; tris[3 * k + 1] = q;   // .w: the edge threshold stays
    q.x = v2.x - v0.x; q.y = v2.y - v0.y; q.z = v2.z - v0.z; q.w = tris[3 * k + 2].w; tris[3 * k + 2] = q;   // .w: the t cut stays
}
__device__ __forceinline__ uint32_t refit_exponent_byte(float extent, float coord_slack, int e_lo) {   // bvh8_build.cpp exponent_byte
    int e = e_lo;
    const float x = (extent + 2.f * coord_slack) * (1.0001f / 255.f) * 1.000001f;       // the host evaluates this in double: stay on the safe side of its rounding
    if (x > 0.f) {
        const uint32_t b = f2u(x);
        const int k = (int)((b >> 23) & 0xffu) - 127;
        e = (b & 0x7fffffu) ? k + 1 : k;
        e = max(e_lo, min(100, e));
    }
    return (uint32_t)(e + 127);
}
__global__ void __launch_bounds__(128) k_refit_level(Node8* nodes, F4* node_box, const F4* __restrict__ tris_obj, const ObjectDev* __restrict__ objects,
                                                     uint32_t first, uint32_t count, int e_lo) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    Node8 nd = nodes[first + i];
    const uint32_t valid24 = (uint32_t)nd.valid24[0] | ((uint32_t)nd.valid24[1] << 8) | ((uint32_t)nd.valid24[2] << 16);
    float lo[8][3], hi[8][3];
    float nlo[3] = {INFINITY, INFINITY, INFINITY}, nhi[3] = {-INFINITY, -INFINITY, -INFINITY};
    uint32_t used = 0;
    for (int s = 0; s < 8; s++) {
        for (int k = 0; k < 3; k++) { lo[s][k] = INFINITY; hi[s][k] = -INFINITY; }
        if (nd.imask & (1u << s)) {
            const uint32_t ci = nd.child_base + __popc((uint32_t)nd.imask & ((1u << s) - 1u));
            const F4 a = node_box[2 * (size_t)ci], b = node_box[2 * (size_t)ci + 1];
            lo[s][0] = a.x; lo[s][1] = a.y; lo[s][2] = a.z; hi[s][0] = b.x; hi[s][1] = b.y; hi[s][2] = b.z;
            used |= 1u << s;
        } else if ((valid24 >> (3 * s)) & 7u) {
            const uint32_t cnt = __popc((valid24 >> (3 * s)) & 7u), t0 = nd.tri_base + __popc(valid24 & ((1u << (3 * s)) - 1u));
            for (uint32_t t = t0; t < t0 + cnt; t++) {
                const F4 A = tris_obj[3 * (size_t)t];
                const ObjectDev& ob = objects[f2u(A.w) & 0x0fffffffu];
                if (ob.type == OBJ_YARNS) {      // a covering triangle of a yarn segment: the tube's box (yarn_box), as at commit
                    const F4 Bq = tris_obj[3 * (size_t)t + 1];
                    const float* m = ob.trans;
                    float blo[3], bhi[3];
                    yarn_box(xf_point_rn(m, v3(A.x, A.y, A.z)), xf_point_rn(m, v3(Bq.x, Bq.y, Bq.z)), Bq.w * sqrtf(m[0] * m[0] + m[4] * m[4] + m[8] * m[8]), blo, bhi);
                    for (int k = 0; k < 3; k++) { lo[s][k] = fminf(lo[s][k], blo[k]); hi[s][k] = fmaxf(hi[s][k], bhi[k]); }
                    continue;
                }
                V3 q0, q1, q2;
                refit_corners(tris_obj, objects, (size_t)t, q0, q1, q2);
                const V3 qq[3] = {q0, q1, q2};
                for (int c = 0; c < 3; c++) {
                    lo[s][0] = fminf(lo[s][0], qq[c].x); lo[s][1] = fminf(lo[s][1], qq[c].y); lo[s][2] = fminf(lo[s][2], qq[c].z);
                    hi[s][0] = fmaxf(hi[s][0], qq[c].x); hi[s][1] = fmaxf(hi[s][1], qq[c].y); hi[s][2] = fmaxf(hi[s][2], qq[c].z);
                }
            }
            used |= 1u << s;
        }
        if (used & (1u << s)) for (int k = 0; k < 3; k++) { nlo[k] = fminf(nlo[k], lo[s][k]); nhi[k] = fmaxf(nhi[k], hi[s][k]); }
    }
    F4 q;
    q.x = nlo[0]; q.y = nlo[1]; q.z = nlo[2]; q.w = 0; node_box[2 * (size_t)(first + i)] = q;
    q.x = nhi[0]; q.y = nhi[1]; q.z = nhi[2]; node_box[2 * (size_t)(first + i) + 1] = q;
    const uint32_t eb[3] = {refit_exponent_byte(nhi[0] - nlo[0], node_coord_slack(nlo[0], nhi[0]), e_lo), refit_exponent_byte(nhi[1] - nlo[1], node_coord_slack(nlo[1], nhi[1]), e_lo),
                            refit_exponent_byte(nhi[2] - nlo[2], node_coord_slack(nlo[2], nhi[2]), e_lo)};
    nd.ex = (uint8_t)eb[0]; nd.ey = (uint8_t)eb[1]; nd.ez = (uint8_t)eb[2];
    float cell[3], eps[3], p[3];
    for (int k = 0; k < 3; k++) {
        cell[k] = u2f(eb[k] << 23);                                                       // 2^(e - 127 + 127 - 127)... the byte IS the float's exponent field
        eps[k] = cell[k] * 4e-3f + node_coord_slack(nlo[k], nhi[k]);                      // the builder's conservative slack
        p[k] = nlo[k] - eps[k];
    }
    nd.px = p[0]; nd.py = p[1]; nd.pz = p[2];
    uint8_t* ql[3] = {nd.qlox, nd.qloy, nd.qloz};
    uint8_t* qh[3] = {nd.qhix, nd.qhiy, nd.qhiz};
    for (int s = 0; s < 8; s++)
        for (int k = 0; k < 3; k++) {
            float a = 0.f, b = 0.f;
            if (used & (1u << s)) {
                a = fminf(fmaxf(floorf((lo[s][k] - eps[k] - p[k]) / cell[k]), 0.f), 255.f);
                b = fminf(fmaxf(ceilf((hi[s][k] + eps[k] - p[k]) / cell[k]), 0.f), 255.f);
            }
            ql[k][s] = (uint8_t)a; qh[k][s] = (uint8_t)b;
        }
    nodes[first + i] = nd;
}

__global__ void k_totals(const uint32_t* counters, int nb, unsigned long long valid_paths, unsigned long long* totals) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    unsigned long long closest = valid_paths, shadow = 0;
    for (int b = 0; b < nb; b++) { if (b > 0) closest += counters[2 * b]; shadow += counters[PTB_CNT_SQ + b]; }
    atomicAdd(&totals[0], closest);   // passes of different pipelines finish concurrently
    atomicAdd(&totals[1], shadow);
}

__global__ void __launch_bounds__(256) k_resolve(const F4* accum, size_t n, float gamma, float* imagedouble, float* sample_count, uint8_t* image) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    resolve_pixel(accum, idx, gamma, imagedouble, sample_count, image);
}

__global__ void __launch_bounds__(256) k_resolve_denoiser(const F4* accum, const F4* albedo, const F4* normal, size_t n, float* imagedouble, float* sample_count,
                                                          float* albedoImage, float* normalImage, float* first_hit_normal) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    resolve_denoiser_pixel(accum, albedo, normal, idx, imagedouble, sample_count, albedoImage, normalImage, first_hit_normal);
}

__global__ void __launch_bounds__(256) k_resolve_progressive(const F4* accum, size_t n, float gamma, float* imagedouble, float* sample_count, uint8_t* image) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    resolve_progressive_pixel(accum, idx, gamma, imagedouble, sample_count, image);
}

__global__ void __launch_bounds__(128) k_primary(SceneDev sc, CameraDev cam, int W, int H, int32_t* obj_id, int32_t* tri_id, float* tout) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= W * H) return;
    const int i = idx / W, j = idx - i * W;
    V3 o, d;
    camera_ray(cam, i, j, 0.f, 0.f, 0.f, 0.f, o, d);
    Hit h;
    int32_t id;
    extend_ray<false>(sc, o, d, h, id, nullptr);
    int32_t oid = -1, tid = -1;
    if (id >= 0) { oid = sc.tri_uv[id].object_has_uv & 0x7fffffff; tid = sc.tri_shade[id].orig; }
    else if (id != PTB_HIT_MISS) oid = -2 - id;
    if (obj_id) obj_id[idx] = oid;
    if (tri_id) tri_id[idx] = tid;
    if (tout) tout[idx] = (id == PTB_HIT_MISS) ? -1.f : h.t;
}

// tile pack / unpack-add with apron (multi-GPU gather).  One thread per packed texel.
__global__ void __launch_bounds__(256) k_shard_pack(const F4* rgbw, F4* packed, int W, int H, int tile, int apron, int tiles_x, int n_tiles_total, int shift,
                                                    int rank, int count, long long n_packed, int unpack) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_packed) return;
    shard_texel(const_cast<F4*>(rgbw), packed, idx, W, H, tile, apron, tiles_x, n_tiles_total, shift, rank, count, unpack, RedAddV4());
}

// The same gather over up to three float4 planes of the frame at once (denoiser inputs: colour, albedo and normal sums): plane k of
// the packed tiles lies at packed + k * n_packed, so that one message per rank carries them all.
#define PTB_MAX_PLANES 3
struct ShardPlanes { F4* p[PTB_MAX_PLANES]; int n; };
__global__ void __launch_bounds__(256) k_shard_pack_planes(ShardPlanes pl, F4* packed, int W, int H, int tile, int apron, int tiles_x, int n_tiles_total, int shift,
                                                           int rank, int count, long long n_packed, int unpack) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_packed) return;
    for (int k = 0; k < pl.n; k++)
        shard_texel(pl.p[k], packed + k * n_packed, idx, W, H, tile, apron, tiles_x, n_tiles_total, shift, rank, count, unpack, RedAddV4());
}

// dst[i] += src[i]: the progressive preview sums of one rank added into rank 0's copy
__global__ void __launch_bounds__(256) k_add(const float* __restrict__ src, float* dst, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += src[i];
}

__global__ void k_kat(int which, SceneDev sc, CameraDev cam, FilterDev filt, int W, int H, const double* in, int n, int is, double* out, int os) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    kat_one(which, sc, cam, filt, W, H, in + (size_t)k * is, out + (size_t)k * os);
}

// ------------------------------------------------------------------------------------------------ context
struct ptb_ctx {
    int device = 0;
    std::string err;
    HostScene host;
    FlatScene flat;
    bool committed = false;
    SceneDev sc;
    std::vector<void*> scene_allocs;
    double ms_upload = 0;
    int64_t bytes_nodes = 0, bytes_tris = 0, bytes_attr = 0, bytes_tex = 0;
    // path pool
    int64_t pool_paths = (int64_t)1 << 25, pool_cap = 0;   // measured: larger pools amortise the tails of the persistent kernels (tune4.log)
    PoolDev pool;
    uint32_t* d_queue[2] = {nullptr, nullptr};
    uint32_t* d_counters = nullptr;
    unsigned long long* d_totals = nullptr;
    float* d_rpp = nullptr;
    int64_t rpp_n = 0;
    F4* d_accum = nullptr;
    int64_t accum_n = 0;
    float* d_out_img = nullptr; float* d_out_cnt = nullptr; uint8_t* d_out_u8 = nullptr;
    int64_t out_n = 0;
    F4* d_aux = nullptr;                       // denoiser-input mode: albedo sums, normal sums (2 x W*H float4)
    int64_t aux_n = 0;
    float* d_out_aux = nullptr;                // 3 x (W*H*3) floats staged for the host: albedoImage, normalImage, first-hit normal
    int64_t out_aux_n = 0;
    // progressive session (Raytracer::render_image): persistent accumulator + low-resolution preview
    bool prog_active = false;
    bool prog_sharded = false;                 // begun with ptb_progressive_begin_sharded: read with ptb_progressive_read_sharded
    F4* d_prog_gather = nullptr;               // rank 0 of a sharded session: the gathered sums of a read (the accumulator stays this rank's own)
    int64_t prog_gather_n = 0;
    FrameDev prog_f;
    ptb_params prog_p;
    int prog_iter = 0;
    F4* d_prog_accum = nullptr;
    int64_t prog_n = 0;
    float* d_lowres = nullptr;
    int64_t lowres_n = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // pass pipelines (PTB_OPT_PIPES): consecutive passes of a linear render go round-robin to `n_pipes` streams, each with its own
    // slice of the path pool, queues and counters, so that the latency-bound k_shade of one pass shares the SMs with the issue-bound
    // k_trace of another and the tails of the persistent kernels are filled.  Pipe 0 is `stream`.
    int n_pipes = 2;                           // measured (profiles/r01m): 2 pipelines with 6 resident k_trace blocks per SM each: +3 % on C2 / C4, +1 % on C3
    int trace_blocks_piped = 148 * 6;          // persistent grid of k_trace per pipeline when more than one runs
    cudaStream_t pipe_stream[PTB_MAX_PIPES] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t pipe_done[PTB_MAX_PIPES] = {nullptr, nullptr, nullptr, nullptr};
    bool count_traversal = false;
    bool time_kernels = false;
    bool has_merl = false;
    int exact_blocks = 148 * 8;                // grid of k_exact: one thread per ray that left candidates for the usual counts (it strides beyond that); most threads exit at once
    int trace_blocks = 148 * 8;                // persistent grid of k_trace, set from the occupancy query in ptb_create
    int refill_below = 24;                     // a warp refills its idle lanes once fewer than this many are live
    int tri_min_pct = 25;                      // the triangle phase starts once this share of a warp's live lanes hold triangles
    int tri_den = 6;                           // triangle steps repeat while >= 1/tri_den of the live lanes take part (re-swept r01p: 6 is 0.3 % ahead of 4)
    // multi-GPU (ptb_multi.inl): this context's place in a tile-sharded render and its NCCL communicator
    void* comm = nullptr;                      // ncclComm_t
    int comm_n = 1, comm_rank = 0;
    bool comm_owned = false;
    F4* d_pack = nullptr;                      // packed tiles + aprons: what a rank sends, or everything rank 0 receives
    int64_t pack_n = 0;
    std::vector<std::pair<void*, int64_t>> pinned;   // host buffers page-locked through ptb_pin_host_buffer
    int64_t info_n_tri = -1, info_nodes = 0; int info_depth = 0;   // group followers: the leader's scene figures
    bool frame_dirty = false;                  // ptb_set_frame after the commit: the next device query re-poses the scene first (refit)
    F4* d_node_box = nullptr;                  // refit scratch: every node's own float box (2 x F4 per node)
    int64_t node_box_n = 0;
    double ms_refit = 0;                       // device time of the last refit
    int stack_limit = PTB_STACK;               // PTB_OPT_STACK_LIMIT (tests): refuse trees that need more traversal-stack entries than this
    int build_threads = 0;                     // PTB_OPT_BUILD_THREADS: OpenMP threads of the BVH build (0: the runtime's default)
    std::vector<cudaEvent_t> ev_pool;          // PTB_OPT_TIME_KERNELS: start/stop pairs, one per launch
    std::vector<int> ev_kind;
    ptb_kernel_times ktimes;
};

static std::string g_create_err;

static void free_scene(ptb_ctx* c) {
    for (void* p : c->scene_allocs) cudaFree(p);
    c->scene_allocs.clear();
}
static void free_pool(ptb_ctx* c) {
    for (const PoolArray& a : pool_arrays(c->pool, c->d_queue)) { if (*a.ptr) cudaFree(*a.ptr); *a.ptr = nullptr; }
    c->pool_cap = 0;
}

template <class T>
static int upload(ptb_ctx* c, const T* host, size_t n, const T** dev) {
    void* d = nullptr;
    const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
    CK(cudaMalloc(&d, bytes));
    c->scene_allocs.push_back(d);
    if (n) CK(cudaMemcpyAsync(d, host, n * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    *dev = (const T*)d;
    return PTB_OK;
}

static int ensure_pool(ptb_ctx* c, int64_t paths, bool aov = false, bool branch = false, bool sss = false) {
    if (paths <= c->pool_cap && (!aov || c->pool.aov_n) && (!branch || c->pool.root) && (!sss || c->pool.hit2)) return PTB_OK;
    paths = std::max(paths, c->pool_cap);
    aov = aov || c->pool.aov_n; branch = branch || c->pool.root; sss = sss || c->pool.hit2;
    free_pool(c);
    const bool need[] = {true, aov, branch, sss};   // by PoolArray::need
    for (const PoolArray& a : pool_arrays(c->pool, c->d_queue))
        if (need[a.need]) CK(cudaMalloc(a.ptr, (size_t)paths * a.bytes));
    c->pool_cap = paths;
    return PTB_OK;
}

static void camera_from_abi(CameraDev& cam, const ptb_camera* pc, int W, int H) {
    camera_setup(cam, pc->position, pc->direction, pc->up, pc->fov, pc->focus_distance, pc->aperture, W, H);
}

template <class T>
static int grow(ptb_ctx* c, T** buf, int64_t* have, int64_t want) {
    if (*have >= want) return PTB_OK;
    if (*buf) cudaFree(*buf);
    *buf = nullptr; *have = 0;
    CK(cudaMalloc((void**)buf, (size_t)want * sizeof(T)));
    *have = want;
    return PTB_OK;
}

// ------------------------------------------------------------------------------------------------ C-ABI
extern "C" int ptb_comm_destroy(ptb_ctx* c);

// A C++ exception (std::bad_alloc of a scene too large for the host, a reader's length_error) must not unwind through the C boundary
#define PTB_GUARD(c, body)                                                                               \
    try { body }                                                                                         \
    catch (const std::bad_alloc&) { if (c) (c)->err = "out of host memory"; return PTB_ERR_NOMEM; }      \
    catch (const std::exception& e_) { if (c) (c)->err = std::string("internal error: ") + e_.what(); return PTB_ERR_INVALID; }

// ptb_commit in three steps, so that a group of devices (ptb_multi.inl) flattens and builds once and uploads N times
static int commit_flatten(ptb_ctx* c) {
    if (c->build_threads > 0) omp_set_num_threads(c->build_threads);
    int rc = c->host.flatten(c->flat, c->err);
    if (rc) return rc;
    if (2 * c->flat.bvh.depth > c->stack_limit) {
        c->err = "commit: the BVH8 is " + std::to_string(c->flat.bvh.depth) + " levels deep; the traversal stack (" + std::to_string(c->stack_limit) +
                 " entries, two per level) cannot hold it";
        return PTB_ERR_UNSUPPORTED;
    }
    return PTB_OK;
}
static int commit_upload(ptb_ctx* c, FlatScene& f, const HostScene& host) {
    CK(cudaSetDevice(c->device));
    int rc;
    free_scene(c);
    auto t0 = std::chrono::steady_clock::now();
    SceneDev& sc = c->sc;
    memset(&sc, 0, sizeof(sc));
    scene_header(sc, f);        // before the upload: it tags objects that do not fit the inline table
    if ((rc = scene_modes(sc, host, c->err))) return rc;
    if (sc.bgW > 0 && (rc = upload(c, host.background.data(), host.background.size(), &sc.background))) return rc;
    c->has_merl = false;
    for (const ObjectDev& o : f.objects) if (o.brdf == 1) c->has_merl = true;
    const Node8* dn; const F4* dt; const uint8_t* de;
    if ((rc = upload(c, f.nodes.data(), f.nodes.size(), &dn))) return rc;
    if ((rc = upload(c, f.tris.data(), f.tris.size(), &dt))) return rc;
    if (!f.tris_obj.empty() && (rc = upload(c, f.tris_obj.data(), f.tris_obj.size(), &sc.tris_obj))) return rc;
    if ((rc = upload(c, f.tri_uv.data(), f.tri_uv.size(), &sc.tri_uv))) return rc;
    if ((rc = upload(c, f.tri_shade.data(), f.tri_shade.size(), &sc.tri_shade))) return rc;
    if ((rc = upload(c, f.objects.data(), f.objects.size(), &sc.objects))) return rc;
    if ((rc = upload(c, f.materials.data(), f.materials.size(), &sc.materials))) return rc;
    if ((rc = upload(c, f.texels.data(), f.texels.size(), &sc.texels))) return rc;
    if ((rc = upload(c, f.envmap.data(), f.envmap.size(), &de))) return rc;
    if ((rc = upload(c, f.merl.data(), f.merl.size(), &sc.merl))) return rc;
    sc.nodes = reinterpret_cast<const F4*>(dn);
    sc.tris = dt;
    sc.envmap = de;
    CK(cudaStreamSynchronize(c->stream));
    c->ms_upload = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    c->bytes_nodes = (int64_t)f.nodes.size() * sizeof(Node8);
    c->bytes_tris = (int64_t)f.tris.size() * sizeof(F4);     // what the traversal streams; the object-space corners count as attributes
    c->bytes_attr = (int64_t)f.tri_uv.size() * sizeof(TriUV) + (int64_t)f.tri_shade.size() * sizeof(TriShade) + (int64_t)f.tris_obj.size() * sizeof(F4);
    c->bytes_tex = (int64_t)f.texels.size() * 4 + (int64_t)f.envmap.size() + (int64_t)f.merl.size() * 4;
    c->committed = true;
    c->frame_dirty = false;
    return PTB_OK;
}
static void commit_release_host(ptb_ctx* c) {   // the host copies of the big arrays are no longer needed
    FlatScene& f = c->flat;
    std::vector<F4>().swap(f.tris); std::vector<F4>().swap(f.tris_obj); std::vector<TriUV>().swap(f.tri_uv); std::vector<TriShade>().swap(f.tri_shade);
    std::vector<float>().swap(f.texels); std::vector<float>().swap(f.merl);
}

// Re-pose a committed scene at HostScene::current_frame without rebuilding: host part (matrices, light, header) ...
static int refit_host(ptb_ctx* lead) {
    lead->host.replace_placements(lead->flat);
    return PTB_OK;
}
// ... and device part, from the (leader's) flattened scene: by-value header, object table, triangles, node boxes
static int refit_device(ptb_ctx* c, FlatScene& f, const HostScene& host) {
    CK(cudaSetDevice(c->device));
    SceneDev& sc = c->sc;
    const float* bg = sc.background;
    scene_header(sc, f);
    int rc = scene_modes(sc, host, c->err);
    sc.background = bg;
    if (rc) return rc;
    const size_t n_tri = (size_t)(c->bytes_tris / (3 * (int64_t)sizeof(F4)));
    const bool mesh = sc.has_mesh && n_tri > 0;
    if (mesh) {   // (the first re-pose of a context allocates the per-node boxes: not part of the measured device time)
        if (!sc.tris_obj) { c->err = "refit: the scene was committed without object-space triangles"; return PTB_ERR_STATE; }
        if ((rc = grow(c, &c->d_node_box, &c->node_box_n, 2 * (int64_t)f.bvh.n_nodes))) return rc;
    }
    CK(cudaEventRecord(c->ev0, c->stream));
    CK(cudaMemcpyAsync(const_cast<ObjectDev*>(sc.objects), f.objects.data(), f.objects.size() * sizeof(ObjectDev), cudaMemcpyHostToDevice, c->stream));
    if (mesh) {
        k_refit_tris<<<(unsigned)((n_tri + 255) / 256), 256, 0, c->stream>>>(sc.tris_obj, sc.objects, const_cast<F4*>(sc.tris), n_tri);
        const std::vector<uint32_t>& ls = f.bvh.level_start;
        for (int l = (int)ls.size() - 2; l >= 0; l--) {
            const uint32_t first = ls[l], count = ls[l + 1] - ls[l];
            if (count) k_refit_level<<<(count + 127) / 128, 128, 0, c->stream>>>(reinterpret_cast<Node8*>(const_cast<F4*>(sc.nodes)), c->d_node_box, sc.tris_obj, sc.objects, first, count, f.bvh.e_floor);
        }
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(c->ev1, c->stream));      // device time of the re-pose: upload of the object table, triangles, node boxes (no host round trip inside)
    CK(cudaStreamSynchronize(c->stream));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    c->ms_refit = ms;
    c->frame_dirty = false;
    return PTB_OK;
}
static int ensure_frame(ptb_ctx* c) {      // every device query of a single context starts here
    if (!c->frame_dirty) return PTB_OK;
    if (c->info_n_tri >= 0) { c->err = "a group member is re-posed by ptb_group_render"; return PTB_ERR_STATE; }
    int rc = refit_host(c);
    return rc ? rc : refit_device(c, c->flat, c->host);
}

extern "C" {

const char* ptb_version(void) { return "ptb200 0.1 (sm_100a wavefront, BVH8)"; }

const char* ptb_last_error(const ptb_ctx* c) { return c ? c->err.c_str() : g_create_err.c_str(); }

int ptb_create(int device_id, ptb_ctx** out) {
    if (!out) return PTB_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        g_create_err = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (this library has no CPU path)";
        return PTB_ERR_CUDA;
    }
    if (device_id < 0 || device_id >= n) { g_create_err = "device id out of range"; return PTB_ERR_INVALID; }
    ptb_ctx* c = new ptb_ctx();
    c->device = device_id;
    if (const char* e = getenv("PTB_PIPES")) c->n_pipes = std::max(1, std::min(atoi(e), PTB_MAX_PIPES));
    memset(&c->pool, 0, sizeof(c->pool));
    memset(&c->sc, 0, sizeof(c->sc));
    if (cudaSetDevice(device_id) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess ||
        cudaMalloc((void**)&c->d_counters, PTB_MAX_PIPES * PTB_N_COUNTERS * sizeof(uint32_t)) != cudaSuccess ||
        cudaMalloc((void**)&c->d_totals, PTB_N_TOTALS * sizeof(unsigned long long)) != cudaSuccess) {
        g_create_err = std::string("CUDA init failed: ") + cudaGetErrorString(cudaGetLastError());
        delete c;
        return PTB_ERR_CUDA;
    }
    {
        int sms = 148, per_sm = 8;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device_id);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_trace<false, false>, 128, 0) != cudaSuccess || per_sm < 1) per_sm = 8;
        c->trace_blocks = sms * per_sm;
        c->trace_blocks_piped = sms * std::max(1, (per_sm * 2 + 2) / 3);   // 6 of 9: two pipelines in their trace phase still fill the SM
    }
    *out = c;
    return PTB_OK;
}

void ptb_destroy(ptb_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    ptb_comm_destroy(c);
    for (auto& e : c->pinned) cudaHostUnregister(e.first);
    c->pinned.clear();
    free_scene(c);
    free_pool(c);
    void* ptrs[] = {c->d_counters, c->d_totals, c->d_rpp, c->d_accum, c->d_out_img, c->d_out_cnt, c->d_out_u8, c->d_aux, c->d_out_aux, c->d_prog_accum, c->d_prog_gather, c->d_lowres, c->d_pack, c->d_node_box};
    for (void* p : ptrs) if (p) cudaFree(p);
    cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1);
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    for (int i = 1; i < PTB_MAX_PIPES; i++) { if (c->pipe_stream[i]) cudaStreamDestroy(c->pipe_stream[i]); if (c->pipe_done[i]) cudaEventDestroy(c->pipe_done[i]); }
    cudaStreamDestroy(c->stream);
    delete c;
}

int ptb_add_sphere(ptb_ctx* c, const float O[3], float R, const ptb_xform* xf, int flags, int* out_id) {
    if (!c || !O) return PTB_ERR_INVALID;
    if (c->committed) { c->err = "scene already committed"; return PTB_ERR_STATE; }
    const int id = c->host.add_sphere(O, R, xf, flags);
    if (out_id) *out_id = id;
    return PTB_OK;
}
int ptb_add_plane(ptb_ctx* c, const float A[3], const float N[3], const ptb_xform* xf, int flags, int* out_id) {
    if (!c || !A || !N) return PTB_ERR_INVALID;
    if (c->committed) { c->err = "scene already committed"; return PTB_ERR_STATE; }
    const int id = c->host.add_plane(A, N, xf, flags);
    if (out_id) *out_id = id;
    return PTB_OK;
}
int ptb_add_cylinder(ptb_ctx* c, const float A[3], const float B[3], float R, const ptb_xform* xf, int flags, int* out_id) {
    if (!c || !A || !B) return PTB_ERR_INVALID;
    if (c->committed) { c->err = "scene already committed"; return PTB_ERR_STATE; }
    if (!(R > 0) || (A[0] == B[0] && A[1] == B[1] && A[2] == B[2])) { c->err = "add_cylinder: needs a radius > 0 and two distinct end points"; return PTB_ERR_INVALID; }
    const int id = c->host.add_cylinder(A, B, R, xf, flags);
    if (out_id) *out_id = id;
    return PTB_OK;
}
int ptb_add_pointset(ptb_ctx* c, const ptb_pointset* ps, const ptb_xform* xf, int flags, int* out_id) {
    if (!c) return PTB_ERR_INVALID;
    if (c->committed) { c->err = "scene already committed"; return PTB_ERR_STATE; }
    PTB_GUARD(c, {
        const int id = c->host.add_pointset(ps, xf, flags, c->err);
        if (id < 0) return id;
        if (out_id) *out_id = id;
        return PTB_OK;
    })
}
int ptb_add_yarns(ptb_ctx* c, const ptb_yarns* y, const ptb_xform* xf, int flags, int* out_id) {
    if (!c) return PTB_ERR_INVALID;
    if (c->committed) { c->err = "scene already committed"; return PTB_ERR_STATE; }
    PTB_GUARD(c, {
        const int id = c->host.add_yarns(y, xf, flags, c->err);
        if (id < 0) return id;
        if (out_id) *out_id = id;
        return PTB_OK;
    })
}
int ptb_add_mesh(ptb_ctx* c, const ptb_mesh* m, const ptb_xform* xf, int flags, int* out_id) {
    if (!c) return PTB_ERR_INVALID;
    if (c->committed) { c->err = "scene already committed"; return PTB_ERR_STATE; }
    PTB_GUARD(c, {
        const int id = c->host.add_mesh(m, xf, flags, c->err);
        if (id < 0) return id;
        if (out_id) *out_id = id;
        return PTB_OK;
    })
}
int ptb_set_group_material(ptb_ctx* c, int obj, int group, const ptb_material* m) {
    if (!c) return PTB_ERR_INVALID;
    if (c->committed) { c->err = "scene already committed"; return PTB_ERR_STATE; }
    return c->host.set_group_material(obj, group, m, c->err);
}
int ptb_set_brdf(ptb_ctx* c, int obj, int kind, int merl_id) {
    if (!c || obj < 0 || obj >= (int)c->host.objects.size()) return PTB_ERR_INVALID;
    if (kind == PTB_BRDF_MERL && (merl_id < 0 || merl_id >= (int)c->host.merl_tables.size())) { c->err = "set_brdf: unknown merl id"; return PTB_ERR_INVALID; }
    if (kind != PTB_BRDF_PHONG && kind != PTB_BRDF_MERL) return PTB_ERR_UNSUPPORTED;
    c->host.objects[obj].brdf = kind;
    c->host.objects[obj].merl = kind == PTB_BRDF_MERL ? merl_id : 0;
    return PTB_OK;
}
int ptb_add_merl(ptb_ctx* c, const double* table, int* out_merl_id) {
    if (!c || !table) return PTB_ERR_INVALID;
    c->host.merl_tables.emplace_back(table, table + 3 * (size_t)PTB_MERL_N);
    if (out_merl_id) *out_merl_id = (int)c->host.merl_tables.size() - 1;
    return PTB_OK;
}
int ptb_set_envmap(ptb_ctx* c, const uint8_t* rgb, int W, int H) {
    if (!c) return PTB_ERR_INVALID;
    if (c->committed) { c->err = "scene already committed"; return PTB_ERR_STATE; }
    if (!rgb || W <= 0 || H <= 0) { c->host.envmap.clear(); c->host.envW = c->host.envH = 0; return PTB_OK; }
    c->host.envmap.assign(rgb, rgb + (size_t)W * H * 3);
    c->host.envW = W; c->host.envH = H;
    return PTB_OK;
}
int ptb_set_light(ptb_ctx* c, float intensite_lumiere, float envmap_intensity) {
    if (!c) return PTB_ERR_INVALID;
    c->host.intensite_lumiere = intensite_lumiere;
    c->host.envmap_intensity = envmap_intensity;
    if (c->committed) {  // light constants live in the by-value scene header: cheap to refresh
        const float s = placement_at(c->host.objects[0], c->host.current_frame).scale;   // Object::get_scale at the frame, like flatten
        c->sc.lightPower = intensite_lumiere / (s * s);
        c->sc.envmap_intensity = envmap_intensity;
    }
    return PTB_OK;
}

int ptb_set_keyframes(ptb_ctx* c, int obj, int kind, const float* frames, const float* values, int n) {
    if (!c || obj < 0 || obj >= (int)c->host.objects.size() || kind < PTB_KEY_SCALE || kind > PTB_KEY_ROTATION || n < 0 || (n > 0 && (!frames || !values))) {
        if (c) c->err = "set_keyframes: bad object, kind or arrays";
        return PTB_ERR_INVALID;
    }
    static const int width[3] = {1, 3, 9};
    key_track_set(c->host.objects[obj].keys[kind], frames, values, n, width[kind]);
    return PTB_OK;
}

int ptb_set_frame(ptb_ctx* c, float frame) {
    if (!c) return PTB_ERR_INVALID;
    if (c->committed && frame != c->host.current_frame) c->frame_dirty = true;   // re-posed (refit, no rebuild) by the next render / picking query
    c->host.current_frame = frame;
    return PTB_OK;
}

int ptb_set_fog(ptb_ctx* c, const ptb_fog* fog) {
    if (!c || !fog) return PTB_ERR_INVALID;
    if (fog->type < 0 || fog->type > 1 || fog->phase_type < 0 || fog->phase_type > 2) { c->err = "set_fog: fog_type is 0..1, fog_phase_type 0..2"; return PTB_ERR_INVALID; }
    c->host.fog = *fog;
    return PTB_OK;
}

int ptb_set_background(ptb_ctx* c, const float* rgb, int W, int H) {
    if (!c) return PTB_ERR_INVALID;
    c->host.background.clear(); c->host.bgW = c->host.bgH = 0;
    if (!rgb || W <= 0 || H <= 0) return PTB_OK;
    c->host.background.assign(rgb, rgb + (size_t)W * H * 3);
    c->host.bgW = W; c->host.bgH = H;
    return PTB_OK;
}

int ptb_commit(ptb_ctx* c) {
    if (!c) return PTB_ERR_INVALID;
    PTB_GUARD(c, {
        int rc = commit_flatten(c);
        if (rc) return rc;
        if ((rc = commit_upload(c, c->flat, c->host))) return rc;
        commit_release_host(c);
        return PTB_OK;
    })
}

static int frame_setup(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, FrameDev& f) {
    const int rc = frame_geometry(cam, p, f, c->err);
    if (rc) return rc;
    // randomPerPixel (prepare_render): regenerated when the frame size changes
    const int64_t npix = (int64_t)p->W * p->H;
    if (c->rpp_n != npix) {
        if (c->d_rpp) cudaFree(c->d_rpp);
        c->d_rpp = nullptr; c->rpp_n = 0;
        CK(cudaMalloc((void**)&c->d_rpp, (size_t)npix * 2 * sizeof(float)));
        k_rpp<<<(unsigned)((npix + 255) / 256), 256, 0, c->stream>>>(c->d_rpp, (int)npix);
        CK(cudaGetLastError());
        c->rpp_n = npix;
    }
    f.rpp = c->d_rpp;
    return PTB_OK;
}

// PTB_OPT_TIME_KERNELS: a start/stop event pair around one launch, on the launching stream
struct LaunchTimer {
    ptb_ctx* c; size_t used = 0; cudaStream_t cur = nullptr;
    explicit LaunchTimer(ptb_ctx* ctx) : c(ctx) { c->ev_kind.clear(); }
    void begin(int kind, cudaStream_t st = nullptr) {
        if (!c->time_kernels) return;
        cur = st ? st : c->stream;
        if (used + 2 > c->ev_pool.size()) { cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b); c->ev_pool.push_back(a); c->ev_pool.push_back(b); }
        c->ev_kind.push_back(kind);
        cudaEventRecord(c->ev_pool[used], cur);
    }
    void end() {
        if (!c->time_kernels) return;
        cudaEventRecord(c->ev_pool[used + 1], cur);
        used += 2;
    }
};

// the slice of the path pool that starts at path `off` (one pipeline's share; queue entries are indices relative to it)
static PoolDev pool_slice(const PoolDev& p, size_t off) {
    if (off == 0) return p;
    PoolDev s = p;
    for (const PoolArray& a : pool_arrays(s))
        if (*a.ptr) *a.ptr = (char*)*a.ptr + off * a.bytes;
    return s;
}

}  // extern "C"

// One pass pipeline: its stream, pool slice, bounce queues and counters (pipe 0 is the context's own; branching renders only use it)
struct Pipe { cudaStream_t stream; PoolDev pool; uint32_t *queue[2], *counters; };
// What a render counts on the host: kernel launches, and the rays of the branching level loop
struct RenderTally { uint64_t launches = 0; unsigned long long branch_closest = 0, branch_shadow = 0; };

// One BVH query of a queue: k_trace (its COUNT instantiation with PTB_OPT_COUNT_TRAVERSAL), then k_exact for the candidates it left
template <bool ANY_HIT, bool BRANCH>
static void launch_trace(ptb_ctx* c, unsigned grid, cudaStream_t st, const PoolDev& p, const uint32_t* queue, const uint32_t* count, int n_static,
                         uint32_t* cursor, uint32_t* defer_count) {
    if (c->count_traversal) k_trace<ANY_HIT, true, BRANCH><<<grid, 128, 0, st>>>(c->sc, p, queue, count, n_static, cursor, c->d_totals, c->refill_below, c->tri_den, c->tri_min_pct, defer_count);
    else k_trace<ANY_HIT, false, BRANCH><<<grid, 128, 0, st>>>(c->sc, p, queue, count, n_static, cursor, c->d_totals, c->refill_below, c->tri_den, c->tri_min_pct, defer_count);
    k_exact<ANY_HIT, BRANCH><<<c->exact_blocks, 128, 0, st>>>(c->sc, p, defer_count);
}

// The queues and counters of one shade launch; `items` bounds the entries of its queue (one thread each)
struct ShadeIO {
    unsigned items;
    const uint32_t *queue, *count;
    int n_static;
    uint32_t *next_queue, *next_count, *shadow_count, *shadow_queries;
};
template <bool MERL, int MINB, bool AOV, bool EXOTIC>
static void shade_linear(ptb_ctx* c, const FrameDev& f, const PoolDev& p, cudaStream_t st, const ShadeIO& s) {
    k_shade<MERL, MINB, AOV, EXOTIC><<<(s.items + PTB_SHADE_BLOCK - 1) / PTB_SHADE_BLOCK, PTB_SHADE_BLOCK, 0, st>>>(c->sc, f, p, s.queue, s.count, s.n_static, s.next_queue,
                                                                                                               s.next_count, s.shadow_count, s.shadow_queries);
}
template <bool MERL>
static void shade_branch(ptb_ctx* c, const FrameDev& f, const ShadeIO& s, uint32_t n_roots, const F4* resume) {
    k_shade_branch<MERL><<<(s.items + 127) / 128, 128, 0, c->stream>>>(c->sc, f, c->pool, s.queue, s.count, s.n_static, s.next_queue, s.next_count, s.shadow_count,
                                                                        s.shadow_queries, c->d_counters + PTB_CNT_ALLOC, n_roots, (uint32_t)c->pool_cap,
                                                                        c->d_counters + PTB_CNT_DROPS, c->d_counters + PTB_CNT_PROBE, resume);
}
// The shade launch of a bounce (linear renders) or a level (branching renders, `n_roots` samples, `resume`: the answered subsurface
// probes to shade again, or null).  Scenes with Cylinder / PointSet / Yarns objects take the k_shade that carries their code (not
// register-squeezed); the AOV kernels shade the camera rays of a denoiser-input render.
static void launch_shade(ptb_ctx* c, const FrameDev& f, const PoolDev& p, cudaStream_t st, const ShadeIO& s, bool branch, bool aov_first,
                         uint32_t n_roots = 0, const F4* resume = nullptr) {
    const bool merl = c->has_merl;
    if (branch) merl ? shade_branch<true>(c, f, s, n_roots, resume) : shade_branch<false>(c, f, s, n_roots, resume);
    else if (c->sc.has_exotic && aov_first) merl ? shade_linear<true, 5, true, true>(c, f, p, st, s) : shade_linear<false, 6, true, true>(c, f, p, st, s);
    else if (c->sc.has_exotic) merl ? shade_linear<true, 5, false, true>(c, f, p, st, s) : shade_linear<false, 6, false, true>(c, f, p, st, s);
    else if (aov_first) merl ? shade_linear<true, 5, true, false>(c, f, p, st, s) : shade_linear<false, 6, true, false>(c, f, p, st, s);
    else merl ? shade_linear<true, 8, false, false>(c, f, p, st, s) : shade_linear<false, 8, false, false>(c, f, p, st, s);
}

// The linear schedule of one pass on its pipeline: per bounce, closest hits, shading, shadow rays.  Every kernel reads its item count
// from the pipeline's counters, so the host never waits.
static void run_bounces(ptb_ctx* c, const FrameDev& f, const Pipe& pp, int n_paths, int n_pipes, LaunchTimer& lt, RenderTally& tally) {
    const bool mesh = c->sc.has_mesh != 0, aov = f.accum_albedo != nullptr;
    uint32_t* const pc = pp.counters;
    // persistent grid: as many blocks as are resident at once, but no more than the queue can feed
    const unsigned gt = (unsigned)std::max(1, std::min<int>(n_pipes > 1 ? c->trace_blocks_piped : c->trace_blocks, (n_paths + 127) / 128));
    for (int b = 0; b < f.nb_bounces; b++) {
        const uint32_t* q = b == 0 ? nullptr : pp.queue[b & 1];
        const uint32_t* cnt = b == 0 ? nullptr : pc + 2 * b;
        if (mesh) {
            lt.begin(1 | (b << 8), pp.stream);
            launch_trace<false, false>(c, gt, pp.stream, pp.pool, q, cnt, n_paths, pc + PTB_CNT_CUR + 2 * b, pc + PTB_CNT_DEFER + 2 * b);
            lt.end();
            tally.launches += 2;
        }
        lt.begin(2 | (b << 8), pp.stream);
        launch_shade(c, f, pp.pool, pp.stream, {(unsigned)n_paths, q, cnt, n_paths, pp.queue[(b + 1) & 1], pc + 2 * (b + 1), pc + 2 * b + 1, pc + PTB_CNT_SQ + b}, false, aov && b == 0);
        lt.end();
        tally.launches++;
        if (mesh) {
            lt.begin(3 | (b << 8), pp.stream);
            launch_trace<true, false>(c, gt, pp.stream, pp.pool, nullptr, pc + 2 * b + 1, 0, pc + PTB_CNT_CUR + 2 * b + 1, pc + PTB_CNT_DEFER + 2 * b + 1);
            lt.end();
            tally.launches += 2;
        }
    }
}

// The branching schedule of one pass: a level-synchronous walk of the contribution tree on the context's stream, with the host reading
// each level's queue lengths (these are the reference's compositing / medium modes, not the benchmarked path).  Counter slots alternate
// with the level's parity.  A straight-through ray keeps its depth (Raytracer.cpp:529-531), and at grazing angles the shading-normal
// offset can put it back in front of the ghost triangle it just crossed: the reference then re-hits it for up to hundreds of iterations
// (its ring simply keeps turning).  Here such chains end after PTB_BRANCH_MAX_LEVELS.
static int run_branch_levels(ptb_ctx* c, const FrameDev& f, int n_paths, unsigned long long valid_here, LaunchTimer& lt, RenderTally& tally) {
    uint32_t n_level = (uint32_t)n_paths;
    const bool mesh = c->sc.has_mesh != 0;
    for (int b = 0; b < PTB_BRANCH_MAX_LEVELS && n_level > 0 && f.nb_bounces > 0; b++) {
        const int s = b & 1, ns = (b + 1) & 1, kind = std::min(b, 63) << 8;
        uint32_t* cnt_q = c->d_counters + 2 * s; uint32_t* cnt_sh = c->d_counters + 2 * s + 1; uint32_t* cnt_next = c->d_counters + 2 * ns;
        uint32_t* cur = c->d_counters + PTB_CNT_CUR + 2 * s; uint32_t* cnt_sq = c->d_counters + PTB_CNT_SQ + s;
        uint32_t* cnt_def = c->d_counters + PTB_CNT_DEFER + 2 * s;
        if (b >= 1) {
            CK(cudaMemsetAsync(cnt_next, 0, sizeof(uint32_t), c->stream));
            if (b >= 2) {
                CK(cudaMemsetAsync(cnt_sh, 0, sizeof(uint32_t), c->stream));
                CK(cudaMemsetAsync(cur, 0, 2 * sizeof(uint32_t), c->stream));
                CK(cudaMemsetAsync(cnt_sq, 0, sizeof(uint32_t), c->stream));
                CK(cudaMemsetAsync(cnt_def, 0, 2 * sizeof(uint32_t), c->stream));
            }
            CK(cudaMemsetAsync(c->d_counters + PTB_CNT_PROBE, 0, sizeof(uint32_t), c->stream));
        }
        const uint32_t* q = b == 0 ? nullptr : c->d_queue[s];
        const uint32_t* cnt = b == 0 ? nullptr : cnt_q;
        if (mesh) {
            const unsigned gt = (unsigned)std::max(1, std::min<int>(c->trace_blocks, (int)((n_level + 127) / 128)));
            lt.begin(1 | kind);
            launch_trace<false, false>(c, gt, c->stream, c->pool, q, cnt, n_paths, cur, cnt_def);
            lt.end();
            tally.launches += 2;
        }
        lt.begin(2 | kind);
        launch_shade(c, f, c->pool, c->stream, {n_level, q, cnt, n_paths, c->d_queue[ns], cnt_next, cnt_sh, cnt_sq}, true, false, (uint32_t)n_paths);
        lt.end();
        tally.launches++;
        if (c->sc.has_sss) {   // answer this level's subsurface probes, then shade those hits for good
            uint32_t h_probe = 0;
            CK(cudaMemcpyAsync(&h_probe, c->d_counters + PTB_CNT_PROBE, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            if (h_probe > 0) {
                k_probe<<<(h_probe + 127) / 128, 128, 0, c->stream>>>(c->sc, c->pool, (int)h_probe);
                lt.begin(2 | kind);
                launch_shade(c, f, c->pool, c->stream, {h_probe, nullptr, nullptr, (int)h_probe, c->d_queue[ns], cnt_next, cnt_sh, cnt_sq}, true, false, (uint32_t)n_paths,
                             c->pool.probe_d);
                lt.end();
                tally.launches += 2;
            }
        }
        uint32_t h_sh = 0, h_next = 0, h_sq = 0;
        CK(cudaMemcpyAsync(&h_sh, cnt_sh, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaMemcpyAsync(&h_next, cnt_next, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaMemcpyAsync(&h_sq, cnt_sq, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        if (mesh && h_sh > 0) {
            const unsigned ga = (unsigned)std::max(1, std::min<int>(c->trace_blocks, (int)((h_sh + 127) / 128)));
            lt.begin(3 | kind);
            launch_trace<true, true>(c, ga, c->stream, c->pool, nullptr, cnt_sh, 0, cur + 1, cnt_def + 1);
            lt.end();
            tally.launches += 2;
        }
        tally.branch_closest += b == 0 ? valid_here * (unsigned long long)f.spp_pass : (unsigned long long)n_level;
        tally.branch_shadow += h_sq;
        n_level = h_next;
    }
    uint32_t drops = 0;
    CK(cudaMemcpyAsync(&drops, c->d_counters + PTB_CNT_DROPS, sizeof(drops), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (drops > 0) {
        c->err = "branching render: contribution pool exhausted (" + std::to_string(drops) + " side branches dropped); raise PTB_OPT_POOL_PATHS";
        return PTB_ERR_NOMEM;
    }
    return PTB_OK;
}

// After a render's work has finished: the device totals and the host tally folded into ptb_kernel_times and `stats`, the launch
// timings of PTB_OPT_TIME_KERNELS, and the PTB_DEBUG_TRI / PTB_DEBUG_BOUNCES reports on stderr.
static int render_stats(ptb_ctx* c, int nb, unsigned long long samples, const RenderTally& tally, ptb_stats* stats, std::chrono::steady_clock::time_point w0) {
    unsigned long long t[PTB_N_TOTALS];
    CK(cudaMemcpy(t, c->d_totals, sizeof(t), cudaMemcpyDeviceToHost));
    t[0] += tally.branch_closest; t[1] += tally.branch_shadow;
    ptb_kernel_times& kt = c->ktimes;
    for (size_t i = 0; i < c->ev_kind.size(); i++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ev_pool[2 * i], c->ev_pool[2 * i + 1]);
        kt.ms[c->ev_kind[i] & 0xff] += ms;
        kt.launches[c->ev_kind[i] & 0xff]++;
    }
    if (getenv("PTB_DEBUG_TRI") && t[6]) {   // triangle phase of k_trace (COUNT kernels): warp iterations, lanes per iteration, packed minimum
        fprintf(stderr, "[ptb] triangle phase, closest: %llu tests in %llu warp iterations (%.1f lanes each), %llu if packed 32 to an iteration (%.1f %% fewer)\n", t[3], t[6],
                (double)t[3] / (double)t[6], t[7], 100.0 * (1.0 - (double)t[7] / (double)t[6]));
        if (t[8]) fprintf(stderr, "[ptb] triangle phase, any hit: %llu tests in %llu warp iterations (%.1f lanes each), %llu if packed (%.1f %% fewer)\n", t[5], t[8], (double)t[5] / (double)t[8], t[9],
                          100.0 * (1.0 - (double)t[9] / (double)t[8]));
    }
    if (getenv("PTB_DEBUG_BOUNCES")) {   // per-bounce launch times of the LAST pass + its queue lengths (diagnostics only)
        uint32_t cnt[PTB_N_COUNTERS];
        cudaMemcpy(cnt, c->d_counters, sizeof(cnt), cudaMemcpyDeviceToHost);
        const size_t per_pass = 2 + 3 * (size_t)nb;
        const size_t first = c->ev_kind.size() >= per_pass ? c->ev_kind.size() - per_pass : 0;
        for (size_t i = first; i < c->ev_kind.size(); i++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, c->ev_pool[2 * i], c->ev_pool[2 * i + 1]);
            const int kind = c->ev_kind[i] & 0xff, b = c->ev_kind[i] >> 8;
            const char* names[] = {"raygen", "closest", "shade", "anyhit", "splat"};
            const unsigned items = kind == 3 ? cnt[2 * b + 1] : ((kind == 1 || kind == 2) ? (b == 0 ? 0u : cnt[2 * b]) : 0u);
            fprintf(stderr, "[ptb] %-8s b=%d  %8.3f ms  items=%u\n", names[kind], b, ms, items);
        }
    }
    kt.items[0] = kt.items[4] = samples;
    kt.items[1] = kt.items[2] = t[0]; kt.items[3] = t[1];
    kt.node_visits[1] = t[2]; kt.tri_tests[1] = t[3]; kt.node_visits[3] = t[4]; kt.tri_tests[3] = t[5];
    if (stats) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
        memset(stats, 0, sizeof(*stats));
        stats->samples = samples;
        stats->rays_closest = t[0]; stats->rays_shadow = t[1]; stats->node_visits = t[2] + t[4]; stats->tri_tests = t[3] + t[5];
        stats->ms_device = ms;
        stats->ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count();
        stats->kernel_launches = tally.launches;
    }
    return PTB_OK;
}

// The pass loop: samples k_first .. k_first + nrays - 1 of every pixel of the shard, accumulated into d_rgbw (device, W*H float4).
// Every pass is raygen -> bounces (or levels of a branching render) -> splat -> k_totals on its pipeline; the pipelines join on the
// context's stream at the end.
static int render_passes(ptb_ctx* c, FrameDev f, int nrays, F4* d_rgbw, ptb_stats* stats, int k_first = 0) {
    const auto w0 = std::chrono::steady_clock::now();
    const int64_t pixel_slots = (int64_t)f.n_my_tiles * f.tile * f.tile;
    RenderTally tally;
    LaunchTimer lt(c);
    memset(&c->ktimes, 0, sizeof(c->ktimes));
    CK(cudaMemsetAsync(c->d_totals, 0, PTB_N_TOTALS * sizeof(unsigned long long), c->stream));
    CK(cudaEventRecord(c->ev0, c->stream));
    const unsigned long long valid_pixels = tile_range_pixels(f, 0, pixel_slots);
    if (pixel_slots > 0) {
        const PassPlan pl = plan_passes(c->sc, f.nb_bounces, f.tile, pixel_slots, nrays, c->pool_paths, c->n_pipes);
        if (pl.branch && f.accum_albedo) { c->err = "denoiser inputs are not available with fog, ghost objects, subsurface scattering or a background photograph"; return PTB_ERR_UNSUPPORTED; }
        int rc = ensure_pool(c, pl.pool_paths, f.accum_albedo != nullptr, pl.branch, c->sc.has_sss != 0);
        if (rc) return rc;
        for (int i = 1; i < pl.n_pipes; i++) {
            if (!c->pipe_stream[i]) { CK(cudaStreamCreateWithFlags(&c->pipe_stream[i], cudaStreamNonBlocking)); CK(cudaEventCreateWithFlags(&c->pipe_done[i], cudaEventDisableTiming)); }
            CK(cudaStreamWaitEvent(c->pipe_stream[i], c->ev0, 0));
        }
        int64_t pass_index = 0;
        for (int64_t s0 = 0; s0 < pixel_slots; s0 += pl.slots_pass) {
            const int64_t ns = std::min(pl.slots_pass, pixel_slots - s0);
            const unsigned long long valid_here = tile_range_pixels(f, s0, ns);   // for the ray statistics
            for (int k0 = 0; k0 < nrays; k0 += pl.spp_pass) {
                f.spp_pass = std::min(pl.spp_pass, nrays - k0);
                f.k0 = k_first + k0;
                f.slot0 = (int)s0;
                f.n_pixel_slots = (int)ns;
                const int n_paths = (int)(ns * f.spp_pass);
                const size_t pi = (size_t)(pass_index++ % pl.n_pipes);
                const Pipe pp = {pi ? c->pipe_stream[pi] : c->stream, pool_slice(c->pool, pi * (size_t)pl.stride),
                                 {c->d_queue[0] + pi * pl.stride, c->d_queue[1] + pi * pl.stride}, c->d_counters + pi * PTB_N_COUNTERS};
                CK(cudaMemsetAsync(pp.counters, 0, PTB_N_COUNTERS * sizeof(uint32_t), pp.stream));
                lt.begin(0, pp.stream);
                if (c->sc.has_exotic) k_raygen<true><<<(unsigned)((n_paths + 255) / 256), 256, 0, pp.stream>>>(c->sc, f, pp.pool, n_paths);
                else k_raygen<false><<<(unsigned)((n_paths + 255) / 256), 256, 0, pp.stream>>>(c->sc, f, pp.pool, n_paths);
                lt.end();
                tally.launches++;
                if (!pl.branch) run_bounces(c, f, pp, n_paths, pl.n_pipes, lt, tally);
                else if ((rc = run_branch_levels(c, f, n_paths, valid_here, lt, tally))) return rc;
                lt.begin(4, pp.stream);
                k_splat<<<(unsigned)((ns + 127) / 128), 128, 0, pp.stream>>>(f, pp.pool, d_rgbw);
                lt.end();
                // a branching render counted its rays on the host: k_totals adds nothing then
                k_totals<<<1, 32, 0, pp.stream>>>(pp.counters, pl.branch ? 0 : f.nb_bounces,
                                                  (f.nb_bounces > 0 && !pl.branch) ? valid_here * (unsigned long long)f.spp_pass : 0ull, c->d_totals);
                tally.launches += 2;
                CK(cudaGetLastError());
            }
        }
        for (int i = 1; i < pl.n_pipes; i++) {   // join the pipelines on the context's stream
            CK(cudaEventRecord(c->pipe_done[i], c->pipe_stream[i]));
            CK(cudaStreamWaitEvent(c->stream, c->pipe_done[i], 0));
        }
    }
    CK(cudaEventRecord(c->ev1, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return render_stats(c, f.nb_bounces, valid_pixels * (unsigned long long)nrays, tally, stats, w0);
}

extern "C" {

int ptb_render_accum(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, float* d_rgbw, ptb_stats* stats) {
    if (!c) return PTB_ERR_INVALID;
    if (!c->committed) { c->err = "render before commit"; return PTB_ERR_STATE; }
    { const int rf = ensure_frame(c); if (rf) return rf; }
    if (!d_rgbw) { c->err = "render_accum: null device buffer"; return PTB_ERR_INVALID; }
    CK(cudaSetDevice(c->device));
    FrameDev f;
    int rc = frame_setup(c, cam, p, f);
    if (rc) return rc;
    return render_passes(c, f, p->nrays, reinterpret_cast<F4*>(d_rgbw), stats);
}

// The staging buffers of a resolved n-pixel frame (imagedouble, sample_count, image), sized together
static int ensure_staging(ptb_ctx* c, int64_t n) {
    if (c->out_n >= n) return PTB_OK;
    void* ptrs[] = {c->d_out_img, c->d_out_cnt, c->d_out_u8};
    for (void* q : ptrs) if (q) cudaFree(q);
    c->d_out_img = nullptr; c->d_out_cnt = nullptr; c->d_out_u8 = nullptr; c->out_n = 0;
    CK(cudaMalloc((void**)&c->d_out_img, (size_t)n * 3 * sizeof(float)));
    CK(cudaMalloc((void**)&c->d_out_cnt, (size_t)n * sizeof(float)));
    CK(cudaMalloc((void**)&c->d_out_u8, (size_t)n * 3));
    c->out_n = n;
    return PTB_OK;
}

static int resolve_to_host(ptb_ctx* c, const F4* d_rgbw, int W, int H, float gamma, float* imagedouble, float* sample_count, uint8_t* image) {
    const int64_t n = (int64_t)W * H;
    const int rc = ensure_staging(c, n);
    if (rc) return rc;
    k_resolve<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(d_rgbw, (size_t)n, gamma, imagedouble ? c->d_out_img : nullptr,
                                                                 sample_count ? c->d_out_cnt : nullptr, image ? c->d_out_u8 : nullptr);
    CK(cudaGetLastError());
    if (imagedouble) CK(cudaMemcpyAsync(imagedouble, c->d_out_img, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (sample_count) CK(cudaMemcpyAsync(sample_count, c->d_out_cnt, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (image) CK(cudaMemcpyAsync(image, c->d_out_u8, (size_t)n * 3, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return PTB_OK;
}

int ptb_resolve(ptb_ctx* c, const float* d_rgbw, int W, int H, float gamma, float* imagedouble, float* sample_count, uint8_t* image) {
    if (!c || !d_rgbw || W <= 0 || H <= 0) return PTB_ERR_INVALID;
    CK(cudaSetDevice(c->device));
    return resolve_to_host(c, reinterpret_cast<const F4*>(d_rgbw), W, H, gamma, imagedouble, sample_count, image);
}

int ptb_render(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, float* imagedouble, float* sample_count, uint8_t* image, ptb_stats* stats) {
    if (!c) return PTB_ERR_INVALID;
    if (!c->committed) { c->err = "render before commit"; return PTB_ERR_STATE; }
    { const int rf = ensure_frame(c); if (rf) return rf; }
    CK(cudaSetDevice(c->device));
    auto w0 = std::chrono::steady_clock::now();
    FrameDev f;
    int rc = frame_setup(c, cam, p, f);
    if (rc) return rc;
    const int64_t n = (int64_t)p->W * p->H;
    if ((rc = grow(c, &c->d_accum, &c->accum_n, n))) return rc;
    CK(cudaMemsetAsync(c->d_accum, 0, (size_t)n * sizeof(F4), c->stream));
    rc = render_passes(c, f, p->nrays, c->d_accum, stats);
    if (rc) return rc;
    rc = resolve_to_host(c, c->d_accum, p->W, p->H, p->gamma, imagedouble, sample_count, image);
    if (rc) return rc;
    if (stats) stats->ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count();
    return PTB_OK;
}

// The has_denoiser accumulation of the shard `p` names (every tile for a whole frame): colour and count sums in d_accum, first-hit
// albedo sums in d_aux[0, n), first-hit normal sums in d_aux[n, 2n) (n = W*H; pixels outside the shard stay zero)
static int denoiser_render(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, ptb_stats* stats) {
    FrameDev f;
    int rc = frame_setup(c, cam, p, f);
    if (rc) return rc;
    const int64_t n = (int64_t)p->W * p->H;
    if ((rc = grow(c, &c->d_accum, &c->accum_n, n))) return rc;
    if ((rc = grow(c, &c->d_aux, &c->aux_n, 2 * n))) return rc;
    if ((rc = grow(c, &c->d_out_aux, &c->out_aux_n, 13 * n))) return rc;
    CK(cudaMemsetAsync(c->d_accum, 0, (size_t)n * sizeof(F4), c->stream));
    CK(cudaMemsetAsync(c->d_aux, 0, (size_t)n * 2 * sizeof(F4), c->stream));
    f.box_filter = 1;
    f.accum_albedo = c->d_aux;
    f.accum_normal = c->d_aux + n;
    return render_passes(c, f, p->nrays, c->d_accum, stats);
}
// ... and its resolve into host outputs (any may be NULL)
static int denoiser_resolve(ptb_ctx* c, int64_t n, float* imagedouble, float* sample_count, float* albedoImage, float* normalImage, float* first_hit_normal) {
    float* o = c->d_out_aux;   // staged back to back: imagedouble 3n | sample_count n | albedo 3n | normal 3n | first-hit normal 3n
    k_resolve_denoiser<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->d_accum, c->d_aux, c->d_aux + n, (size_t)n, o, o + 3 * n, o + 4 * n, o + 7 * n, o + 10 * n);
    CK(cudaGetLastError());
    struct { float* host; int64_t off, len; } out[] = {{imagedouble, 0, 3 * n}, {sample_count, 3 * n, n}, {albedoImage, 4 * n, 3 * n}, {normalImage, 7 * n, 3 * n}, {first_hit_normal, 10 * n, 3 * n}};
    for (auto& e : out) if (e.host) CK(cudaMemcpyAsync(e.host, o + e.off, (size_t)e.len * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return PTB_OK;
}

// render_image_nopreviz with has_denoiser == true (Raytracer.cpp:1631-1645, 1676-1693), up to the point where the reference
// hands the buffers to Open Image Denoise.  A shard (p->shard_count > 1) fills the full-frame outputs; its pixels outside its
// tiles have sample_count 0.
int ptb_render_denoiser_inputs(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, float* imagedouble, float* sample_count, float* albedoImage,
                               float* normalImage, float* first_hit_normal, ptb_stats* stats) {
    if (!c) return PTB_ERR_INVALID;
    if (!c->committed) { c->err = "render before commit"; return PTB_ERR_STATE; }
    { const int rf = ensure_frame(c); if (rf) return rf; }
    CK(cudaSetDevice(c->device));
    int rc = denoiser_render(c, cam, p, stats);
    if (rc) return rc;
    return denoiser_resolve(c, (int64_t)p->W * p->H, imagedouble, sample_count, albedoImage, normalImage, first_hit_normal);
}

// ---- progressive rendering: Raytracer::render_image (Raytracer.cpp:1424-1563) one batch of passes at a time ---------------------
// A session over the shard `p` names (every tile for a whole frame); `sharded`: begun by ptb_progressive_begin_sharded
static int progressive_begin(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p, bool sharded) {
    c->prog_active = false;
    int rc = frame_setup(c, cam, p, c->prog_f);
    if (rc) return rc;
    const int64_t n = (int64_t)p->W * p->H;
    const int Wlr = (int)ceilf(p->W / 16.f), Hlr = (int)ceilf(p->H / 16.f);     // Raytracer.cpp:1329-1330
    if ((rc = grow(c, &c->d_prog_accum, &c->prog_n, n))) return rc;
    if ((rc = grow(c, &c->d_lowres, &c->lowres_n, (int64_t)Wlr * Hlr * 3))) return rc;
    if ((rc = grow(c, &c->d_out_aux, &c->out_aux_n, (int64_t)Wlr * Hlr * 3))) return rc;
    CK(cudaMemsetAsync(c->d_prog_accum, 0, (size_t)n * sizeof(F4), c->stream));    // prepare_render: 1383-1385
    CK(cudaMemsetAsync(c->d_lowres, 0, (size_t)Wlr * Hlr * 3 * sizeof(float), c->stream));
    c->prog_f.lowres = c->d_lowres; c->prog_f.lowresW = Wlr; c->prog_f.lowresH = Hlr;
    c->prog_p = *p;
    c->prog_iter = 0;
    c->prog_sharded = sharded;
    c->prog_active = true;
    return PTB_OK;
}

// A shard (p->shard_count > 1) renders its tiles only: read gives full-frame outputs whose pixels outside them have sample_count 0.
int ptb_progressive_begin(ptb_ctx* c, const ptb_camera* cam, const ptb_params* p) {
    if (!c) return PTB_ERR_INVALID;
    if (!c->committed) { c->err = "render before commit"; return PTB_ERR_STATE; }
    { const int rf = ensure_frame(c); if (rf) return rf; }
    CK(cudaSetDevice(c->device));
    return progressive_begin(c, cam, p, false);
}

int ptb_progressive_pass(ptb_ctx* c, int n_spp, ptb_stats* stats) {
    if (!c) return PTB_ERR_INVALID;
    if (!c->prog_active) { c->err = "progressive_pass before progressive_begin"; return PTB_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    const int n = std::min(n_spp, c->prog_p.nrays - c->prog_iter);
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n <= 0) return PTB_OK;                                   // realtime_ray_iter reached nrays: the loop of 1444 has ended
    int rc = render_passes(c, c->prog_f, n, c->d_prog_accum, stats, c->prog_iter);
    if (rc) return rc;
    c->prog_iter += n;
    return PTB_OK;
}

// The outputs of a progressive read from the session's sums `accum` (W*H float4) and preview sums `lowres`
static int progressive_resolve(ptb_ctx* c, const F4* accum, const float* lowres, float* imagedouble, float* sample_count, uint8_t* image, float* imagedouble_lowres,
                               int32_t* current_nb_rays) {
    const ptb_params& p = c->prog_p;
    const int64_t n = (int64_t)p.W * p.H;
    const int rc = ensure_staging(c, n);
    if (rc) return rc;
    k_resolve_progressive<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(accum, (size_t)n, p.gamma, imagedouble ? c->d_out_img : nullptr,
                                                                             sample_count ? c->d_out_cnt : nullptr, image ? c->d_out_u8 : nullptr);
    CK(cudaGetLastError());
    if (imagedouble) CK(cudaMemcpyAsync(imagedouble, c->d_out_img, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (sample_count) CK(cudaMemcpyAsync(sample_count, c->d_out_cnt, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (image) CK(cudaMemcpyAsync(image, c->d_out_u8, (size_t)n * 3, cudaMemcpyDeviceToHost, c->stream));
    if (imagedouble_lowres) CK(cudaMemcpyAsync(imagedouble_lowres, lowres, (size_t)c->prog_f.lowresW * c->prog_f.lowresH * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (current_nb_rays) *current_nb_rays = c->prog_iter;
    return PTB_OK;
}

int ptb_progressive_read(ptb_ctx* c, float* imagedouble, float* sample_count, uint8_t* image, float* imagedouble_lowres, int32_t* current_nb_rays) {
    if (!c) return PTB_ERR_INVALID;
    if (!c->prog_active) { c->err = "progressive_read before progressive_begin"; return PTB_ERR_STATE; }
    if (c->prog_sharded) { c->err = "progressive_read: the session was begun with ptb_progressive_begin_sharded; read it with ptb_progressive_read_sharded"; return PTB_ERR_STATE; }
    CK(cudaSetDevice(c->device));
    return progressive_resolve(c, c->d_prog_accum, c->d_lowres, imagedouble, sample_count, image, imagedouble_lowres, current_nb_rays);
}

int ptb_shard_pack_size(const ptb_params* p, int shard_rank, int64_t* out_floats) {
    if (!p || !out_floats || p->W <= 0 || p->H <= 0) return PTB_ERR_INVALID;
    *out_floats = shard_geometry(p, shard_rank).texels() * 4;
    return PTB_OK;
}

static int shard_move(ptb_ctx* c, const ptb_params* p, int shard_rank, const float* d_rgbw, float* d_packed, int unpack) {
    if (!c || !p || !d_rgbw || !d_packed) return PTB_ERR_INVALID;
    CK(cudaSetDevice(c->device));
    const ShardGeometry g = shard_geometry(p, shard_rank);
    const long long n = g.texels();
    if (n == 0) return PTB_OK;
    k_shard_pack<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(reinterpret_cast<const F4*>(d_rgbw), reinterpret_cast<F4*>(d_packed), p->W, p->H, g.tile, g.apron,
                                                                    g.tiles_x, g.total, g.shift, shard_rank, g.count, n, unpack);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(c->stream));
    return PTB_OK;
}
int ptb_shard_pack(ptb_ctx* c, const ptb_params* p, int shard_rank, const float* d_rgbw, float* d_packed) { return shard_move(c, p, shard_rank, d_rgbw, d_packed, 0); }
int ptb_shard_unpack_add(ptb_ctx* c, const ptb_params* p, int shard_rank, const float* d_packed, float* d_rgbw) { return shard_move(c, p, shard_rank, d_rgbw, const_cast<float*>(d_packed), 1); }

int ptb_primary_ids(ptb_ctx* c, const ptb_camera* cam, int W, int H, int32_t* obj_id, int32_t* tri_id, float* t) {
    if (!c || !cam || W <= 0 || H <= 0) return PTB_ERR_INVALID;
    if (!c->committed) { c->err = "primary_ids before commit"; return PTB_ERR_STATE; }
    { const int rf = ensure_frame(c); if (rf) return rf; }
    CK(cudaSetDevice(c->device));
    CameraDev cd;
    camera_from_abi(cd, cam, W, H);
    const size_t n = (size_t)W * H;
    int32_t *d_o = nullptr, *d_t = nullptr; float* d_tt = nullptr;
    CK(cudaMalloc((void**)&d_o, n * 4)); CK(cudaMalloc((void**)&d_t, n * 4)); CK(cudaMalloc((void**)&d_tt, n * 4));
    k_primary<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(c->sc, cd, W, H, d_o, d_t, d_tt);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess && obj_id) e = cudaMemcpy(obj_id, d_o, n * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && tri_id) e = cudaMemcpy(tri_id, d_t, n * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && t) e = cudaMemcpy(t, d_tt, n * 4, cudaMemcpyDeviceToHost);
    cudaFree(d_o); cudaFree(d_t); cudaFree(d_tt);
    if (e != cudaSuccess) { c->err = std::string("primary_ids: ") + cudaGetErrorString(e); return PTB_ERR_CUDA; }
    return PTB_OK;
}

int ptb_set_option(ptb_ctx* c, int option, int64_t value) {
    if (!c) return PTB_ERR_INVALID;
    switch (option) {
    case PTB_OPT_COUNT_TRAVERSAL: c->count_traversal = value != 0; return PTB_OK;
    case PTB_OPT_POOL_PATHS: if (value < 1024) return PTB_ERR_INVALID; c->pool_paths = value; return PTB_OK;
    case PTB_OPT_TIME_KERNELS: c->time_kernels = value != 0; return PTB_OK;
    case PTB_OPT_REFILL_BELOW: if (value < 1 || value > 33) return PTB_ERR_INVALID; c->refill_below = (int)value; return PTB_OK;
    case PTB_OPT_TRI_FRACTION: if (value < 1 || value > 64) return PTB_ERR_INVALID; c->tri_den = (int)value; return PTB_OK;
    case PTB_OPT_TRI_MIN_PCT: if (value < 0 || value > 100) return PTB_ERR_INVALID; c->tri_min_pct = (int)value; return PTB_OK;
    case PTB_OPT_TRACE_BLOCKS: if (value < 1) return PTB_ERR_INVALID; c->trace_blocks = c->trace_blocks_piped = (int)value; return PTB_OK;
    case PTB_OPT_PIPES: if (value < 1 || value > PTB_MAX_PIPES) return PTB_ERR_INVALID; c->n_pipes = (int)value; return PTB_OK;
    case PTB_OPT_STACK_LIMIT: if (value < 2 || value > PTB_STACK) return PTB_ERR_INVALID; c->stack_limit = (int)value; return PTB_OK;
    case PTB_OPT_BUILD_THREADS: if (value < 0 || value > 4096) return PTB_ERR_INVALID; c->build_threads = (int)value; return PTB_OK;
    default: return PTB_OK;  // unknown options (e.g. the CPU checkers' thread count) are ignored
    }
}

int ptb_get_scene_info(const ptb_ctx* c, ptb_scene_info* info) {
    if (!c || !info) return PTB_ERR_INVALID;
    memset(info, 0, sizeof(*info));
    if (c->info_n_tri >= 0) {   // a group follower: the leader flattened the scene
        info->n_triangles = c->info_n_tri; info->n_bvh_nodes = c->info_nodes; info->bvh_depth = c->info_depth;
        info->bytes_nodes = c->bytes_nodes; info->bytes_triangles = c->bytes_tris; info->bytes_attributes = c->bytes_attr; info->bytes_textures = c->bytes_tex;
        info->ms_upload = c->ms_upload; info->ms_refit = c->ms_refit;
        return PTB_OK;
    }
    info->n_triangles = c->flat.n_tri_scene;   // as handed over; bytes_triangles counts those resident (alpha maps can rule triangles out, scene_host.cpp)
    info->n_bvh_nodes = c->flat.bvh.n_nodes;
    info->bytes_nodes = c->bytes_nodes; info->bytes_triangles = c->bytes_tris; info->bytes_attributes = c->bytes_attr; info->bytes_textures = c->bytes_tex;
    info->n_objects = (int32_t)c->host.objects.size();
    info->bvh_depth = c->flat.bvh.depth;
    info->ms_bvh_build = c->flat.ms_bvh; info->ms_upload = c->ms_upload; info->ms_refit = c->ms_refit;
    return PTB_OK;
}

int ptb_get_kernel_times(const ptb_ctx* c, ptb_kernel_times* out) {
    if (!c || !out) return PTB_ERR_INVALID;
    *out = c->ktimes;
    return PTB_OK;
}

int ptb_kat(ptb_ctx* c, int which, const ptb_camera* cam, int W, int H, const double* in, int n, int is, double* out, int os) {
    if (!c || !in || !out || n <= 0) return PTB_ERR_INVALID;
    CK(cudaSetDevice(c->device));
    if (which == PTB_KAT_MERL_EVAL && (!c->committed || c->host.merl_tables.empty())) { c->err = "kat: MERL needs a committed scene with a table"; return PTB_ERR_STATE; }
    CameraDev cd;
    memset(&cd, 0, sizeof(cd));
    if (cam) camera_from_abi(cd, cam, W, H);
    FilterDev fd;
    memset(&fd, 0, sizeof(fd));
    if (which == PTB_KAT_FILTER_RATIO) filter_setup(fd, (float)in[2]);
    double *d_in = nullptr, *d_out = nullptr;
    CK(cudaMalloc((void**)&d_in, (size_t)n * is * 8)); CK(cudaMalloc((void**)&d_out, (size_t)n * os * 8));
    cudaError_t e = cudaMemcpy(d_in, in, (size_t)n * is * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(d_out, 0, (size_t)n * os * 8);
    if (e == cudaSuccess) {
        k_kat<<<(n + 63) / 64, 64, 0, c->stream>>>(which, c->sc, cd, fd, W, H, d_in, n, is, d_out, os);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess) e = cudaMemcpy(out, d_out, (size_t)n * os * 8, cudaMemcpyDeviceToHost);
    cudaFree(d_in); cudaFree(d_out);
    if (e != cudaSuccess) { c->err = std::string("kat: ") + cudaGetErrorString(e); return PTB_ERR_CUDA; }
    return PTB_OK;
}

}  // extern "C"

#include "ptb_multi.inl"
