// bvh8_build.cpp — host builder of the compressed 8-wide BVH (ptb_bvh8.h) over world-space triangles.
//
// Replaces TriMesh::build_bvh / build_bvh_recur (reference TriangleMesh.cpp:878-885, 1029-1130: one
// binary BVH per mesh, 16 candidate planes on the longest centroid axis, <=4 triangles per leaf).
// Here: one BVH over ALL meshes' triangles baked to world space (scenes are static during a render,
// SURVEY §3.4), binned SAH on all three axes (16 bins) down to single triangles, then the cost-optimal
// collapse to 8-wide nodes with leaves of <=3 triangles, octant-ordered child slots and 8-bit quantised child boxes.
// The result is only an acceleration structure: which triangle a ray hits is decided by the triangle
// test, so parity with the reference does not depend on reproducing its tree.
#include "ptb_host.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>

namespace ptb {

namespace {

struct Box {
    float lo[3], hi[3];
    void reset() { for (int k = 0; k < 3; k++) { lo[k] = INFINITY; hi[k] = -INFINITY; } }
    void grow(const float* p) { for (int k = 0; k < 3; k++) { lo[k] = std::min(lo[k], p[k]); hi[k] = std::max(hi[k], p[k]); } }
    void grow(const Box& b) { for (int k = 0; k < 3; k++) { lo[k] = std::min(lo[k], b.lo[k]); hi[k] = std::max(hi[k], b.hi[k]); } }
    float area() const {
        float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        if (!(dx >= 0) || !(dy >= 0) || !(dz >= 0)) return 0.f;
        return 2.f * (dx * dy + dx * dz + dy * dz);
    }
};

struct BNode {   // binary node: leaf iff count > 0
    Box box;
    int32_t left, right;   // children (internal)
    int32_t first, count;  // range in the index array (leaf)
    int32_t sfirst, scount;  // range of the whole subtree in the index array (the in-place partition keeps it contiguous)
};

// Cost-optimal collapse (Ylitie, Karras, Laine 2017, sec. 3.1): for every binary node n and i = 1..7,
//   C(n,1) = min( leaf: A(n) * P(n) * c_prim  [P(n) <= 3],  wide node: A(n) * c_node + D(n,8) )
//   C(n,i) = min( D(n,i), C(n,i-1) )                      the subtree of n as a forest of at most i children of a wide node
//   D(n,j) = min over 0 < k < j of C(left,k) + C(right,j-k)
// A greedy collapse (open the child of largest area until 8) leaves the lowest wide nodes with 2-3 small leaves: 275k nodes of
// 2.8 children on average for the 1M-triangle mesh, hence one node visit per level of a deep tree; the optimal collapse decides
// leaf sizes and node shapes together.
struct Collapse {
    float c[7];            // C(n,1..7)
    uint8_t d[7];          // d[0]: 0 leaf / 1 wide node; d[i-1], i >= 2: 0 = "as C(n,i-1)", else k = children handed to the left subtree
    uint8_t k8;            // split of D(n,8), the children of the wide node rooted at n
};

struct Builder {
    const float* verts;            // 9 floats per triangle
    int64_t n;
    std::vector<Box> pbox;
    std::vector<float> pcen;       // 3 per prim
    std::vector<uint32_t> idx;
    std::vector<BNode> nodes;
    std::vector<Collapse> dp;
    std::atomic<int64_t> n_nodes{0};
    void solve(int64_t node);

    int64_t alloc2() { return n_nodes.fetch_add(2); }

    void build(int64_t node, int64_t b, int64_t e, int depth);
};

constexpr int64_t PAR_NODE = 1 << 18;      // nodes with at least this many primitives run their passes in chunks (tasks)
constexpr int NBINS = 16;                  // SAH bins per axis
constexpr float C_NODE = 1.f, C_PRIM = 0.5f;   // measured (profiles/r01m): 0.5 beats 0.3 and 0.15 on C2 and C3

void Builder::solve(int64_t node) {
    const BNode& nd = nodes[node];
    Collapse& q = dp[node];
    const float A = nd.box.area();
    if (nd.count > 0) {   // binary leaf (one triangle, or an unsplittable group)
        for (int i = 0; i < 7; i++) { q.c[i] = A * (float)nd.count * C_PRIM; q.d[i] = 0; }
        q.k8 = 0;
        return;
    }
    const Collapse& L = dp[nd.left];
    const Collapse& R = dp[nd.right];
    auto distribute = [&](int j, uint8_t& kbest) {
        float best = INFINITY; kbest = 1;
        for (int k = 1; k < j; k++) {
            if (k > 7 || j - k > 7) continue;
            const float v = L.c[k - 1] + R.c[j - k - 1];
            if (v < best) { best = v; kbest = (uint8_t)k; }
        }
        return best;
    };
    const float wide = A * C_NODE + distribute(8, q.k8);
    const float leaf = nd.scount <= 3 ? A * (float)nd.scount * C_PRIM : INFINITY;
    if (leaf <= wide) { q.c[0] = leaf; q.d[0] = 0; } else { q.c[0] = wide; q.d[0] = 1; }
    for (int i = 2; i <= 7; i++) {
        uint8_t k;
        const float dcost = distribute(i, k);
        if (dcost < q.c[i - 2]) { q.c[i - 1] = dcost; q.d[i - 1] = k; } else { q.c[i - 1] = q.c[i - 2]; q.d[i - 1] = 0; }
    }
}

void Builder::build(int64_t node, int64_t b, int64_t e, int depth) {
    BNode& nd = nodes[node];
    Box box, cb;
    box.reset(); cb.reset();
    const int64_t cnt = e - b;
    // The two passes over a node's primitives (bounds, SAH bins) of the few nodes at the top of the tree, which no sibling task can
    // overlap with, are cut into chunks that run as tasks; minima, maxima and counts merge exactly, so the tree is the serial one.
    const int n_chunks = cnt >= PAR_NODE ? (int)std::min<int64_t>(64, cnt / (PAR_NODE / 4)) : 1;
    if (n_chunks > 1) {
        std::vector<Box> cbx(2 * (size_t)n_chunks);
        for (int c = 0; c < n_chunks; c++) {
#pragma omp task default(shared) firstprivate(c)
            {
                const int64_t i0 = b + cnt * c / n_chunks, i1 = b + cnt * (c + 1) / n_chunks;
                Box x, y; x.reset(); y.reset();
                for (int64_t i = i0; i < i1; i++) { x.grow(pbox[idx[i]]); y.grow(&pcen[3 * (size_t)idx[i]]); }
                cbx[2 * (size_t)c] = x; cbx[2 * (size_t)c + 1] = y;
            }
        }
#pragma omp taskwait
        for (int c = 0; c < n_chunks; c++) { box.grow(cbx[2 * (size_t)c]); cb.grow(cbx[2 * (size_t)c + 1]); }
    } else
    for (int64_t i = b; i < e; i++) { box.grow(pbox[idx[i]]); cb.grow(&pcen[3 * (size_t)idx[i]]); }
    nd.box = box;
    nd.sfirst = (int32_t)b; nd.scount = (int32_t)cnt;
    if (cnt == 1) {   // the collapse forms the leaves itself, from single triangles
        nd.left = nd.right = -1; nd.first = (int32_t)b; nd.count = 1;
        solve(node);
        return;
    }

    // binned SAH over the three axes: ONE pass over the node's primitives fills the bins of all three (the boxes are reached through
    // the index array, a cache miss each: three passes were three misses per primitive)
    float best_cost = INFINITY;
    int best_axis = -1, best_bin = -1;
    struct Bins { Box bb[3][NBINS]; int64_t bc[3][NBINS]; };
    float lo3[3], scale3[3];
    bool use[3];
    for (int ax = 0; ax < 3; ax++) {
        const float ext = cb.hi[ax] - cb.lo[ax];
        use[ax] = ext > 0;
        lo3[ax] = cb.lo[ax]; scale3[ax] = use[ax] ? NBINS / ext : 0.f;
    }
    auto bin_range = [&](Bins& q, int64_t i0, int64_t i1) {
        for (int ax = 0; ax < 3; ax++) for (int k = 0; k < NBINS; k++) { q.bb[ax][k].reset(); q.bc[ax][k] = 0; }
        for (int64_t i = i0; i < i1; i++) {
            const uint32_t p = idx[i];
            const Box& pb = pbox[p];
            const float* pc = &pcen[3 * (size_t)p];
            for (int ax = 0; ax < 3; ax++) {
                if (!use[ax]) continue;
                int k = (int)((pc[ax] - lo3[ax]) * scale3[ax]);
                k = k < 0 ? 0 : (k >= NBINS ? NBINS - 1 : k);
                q.bb[ax][k].grow(pb); q.bc[ax][k]++;
            }
        }
    };
    Bins bins;      // 1.5 KB of stack per level of the recursion
    if (n_chunks > 1) {
        std::vector<Bins> part((size_t)n_chunks);
        for (int c = 0; c < n_chunks; c++) {
#pragma omp task default(shared) firstprivate(c)
            bin_range(part[(size_t)c], b + cnt * c / n_chunks, b + cnt * (c + 1) / n_chunks);
        }
#pragma omp taskwait
        for (int ax = 0; ax < 3; ax++) for (int k = 0; k < NBINS; k++) { bins.bb[ax][k].reset(); bins.bc[ax][k] = 0; }
        for (int c = 0; c < n_chunks; c++)
            for (int ax = 0; ax < 3; ax++) for (int k = 0; k < NBINS; k++) { if (part[(size_t)c].bc[ax][k]) bins.bb[ax][k].grow(part[(size_t)c].bb[ax][k]); bins.bc[ax][k] += part[(size_t)c].bc[ax][k]; }
    } else bin_range(bins, b, e);
    for (int ax = 0; ax < 3; ax++) {
        if (!use[ax]) continue;
        const Box* bb = bins.bb[ax]; const int64_t* bc = bins.bc[ax];
        float ra[NBINS]; int64_t rc[NBINS];
        Box acc; acc.reset(); int64_t c = 0;
        for (int k = NBINS - 1; k > 0; k--) { acc.grow(bb[k]); c += bc[k]; ra[k] = acc.area(); rc[k] = c; }
        acc.reset(); c = 0;
        for (int k = 0; k < NBINS - 1; k++) {
            acc.grow(bb[k]); c += bc[k];
            if (c == 0 || rc[k + 1] == 0) continue;
            const float cost = acc.area() * (float)c + ra[k + 1] * (float)rc[k + 1];
            if (cost < best_cost) { best_cost = cost; best_axis = ax; best_bin = k; }
        }
    }
    int64_t mid;
    if (best_axis < 0) {
        mid = b + cnt / 2;  // coincident centroids: split by index
    } else {
        const float lo = cb.lo[best_axis], scale = NBINS / (cb.hi[best_axis] - cb.lo[best_axis]);
        auto it = std::partition(idx.begin() + b, idx.begin() + e, [&](uint32_t p) {
            int k = (int)((pcen[3 * (size_t)p + best_axis] - lo) * scale);
            k = k < 0 ? 0 : (k >= NBINS ? NBINS - 1 : k);
            return k <= best_bin;
        });
        mid = it - idx.begin();
        if (mid == b || mid == e) mid = b + cnt / 2;
    }
    const int64_t c0 = alloc2();
    nd.left = (int32_t)c0; nd.right = (int32_t)(c0 + 1); nd.first = 0; nd.count = 0;
    if (cnt > 4096 && depth < 24) {
#pragma omp task default(shared) firstprivate(c0, b, mid, depth)
        build(c0, b, mid, depth + 1);
#pragma omp task default(shared) firstprivate(c0, mid, e, depth)
        build(c0 + 1, mid, e, depth + 1);
#pragma omp taskwait
    } else {
        build(c0, b, mid, depth + 1);
        build(c0 + 1, mid, e, depth + 1);
    }
    solve(node);
}

inline uint8_t exponent_byte(float extent, float coord_slack, int e_lo) {
    // smallest e with extent + 2 * slack <= 255 * 2^e, where slack = 4e-3 cells + coord_slack is what the quantisation adds on either
    // side (the 1.0001 pays for the cell-relative part: 255 / 1.0001 + 0.008 < 255).  Never below e_lo (Bvh8Stats::e_floor): a flat or
    // tiny box simply gets cells coarser than it needs.
    const double x = ((double)extent + 2.0 * (double)coord_slack) * 1.0001 / 255.0;
    int e = x > 0 ? (int)std::ceil(std::log2(x)) : e_lo;
    if (e < e_lo) e = e_lo;
    if (e > 100) e = 100;
    return (uint8_t)(e + 127);
}

}  // namespace

void build_bvh8(const float* verts9, int64_t n_tri, std::vector<Node8>& out_nodes, std::vector<uint32_t>& leaf_order, Bvh8Stats& stats, const float* boxes6) {
    out_nodes.clear(); leaf_order.clear();
    stats = Bvh8Stats();
    if (n_tri <= 0) return;
    Builder B;
    B.verts = verts9; B.n = n_tri;
    B.pbox.resize(n_tri); B.pcen.resize(3 * (size_t)n_tri); B.idx.resize(n_tri);
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n_tri; i++) {
        Box bx; bx.reset();
        const float* v = verts9 + 9 * (size_t)i;
        bx.grow(v); bx.grow(v + 3); bx.grow(v + 6);
        // a primitive that stands for a volume (the covering triangles of a yarn segment, ptb_scene.h) brings the volume's box: a ray
        // must reach its triangles whenever it can reach the volume, wherever the triangles themselves lie
        if (boxes6 && boxes6[6 * (size_t)i] <= boxes6[6 * (size_t)i + 3]) { bx.reset(); bx.grow(boxes6 + 6 * (size_t)i); bx.grow(boxes6 + 6 * (size_t)i + 3); }
        B.pbox[i] = bx;
        for (int k = 0; k < 3; k++) B.pcen[3 * (size_t)i + k] = 0.5f * (bx.lo[k] + bx.hi[k]);
        B.idx[i] = (uint32_t)i;
    }
    B.nodes.resize(2 * (size_t)n_tri + 2);
    B.dp.resize(B.nodes.size());
    B.n_nodes = 1;
#pragma omp parallel
    {
#pragma omp single
        B.build(0, 0, n_tri, 0);
    }

    // ---- collapse to 8-wide, breadth first so that a node's internal children are contiguous ----
    // Level by level (the emission order is breadth first, so the nodes of one level are consecutive): (A) every node of the level
    // picks its children, slots and counts, in parallel; (B) a serial prefix sum hands out the indices of the internal children and
    // the first triangle of each node, in the order a node-by-node loop would; (C) the nodes are quantised and written, in parallel.
    struct Item {
        int32_t bnode; uint32_t wide;
        int32_t ch[8]; bool ch_leaf[8]; int nc; int slot_child[8];
        Box nb;
        uint32_t n_internal, n_tris, child_base, tri_base;
    };
    std::vector<Item> level, next;
    out_nodes.assign(1, Node8());
    leaf_order.assign((size_t)n_tri, 0u);
    {
        Item root; memset(&root, 0, sizeof(root));
        root.bnode = 0; root.wide = 0;
        level.push_back(root);
    }
    {   // the finest cell: 2^-25 of the root's, whose cells are the largest of the tree
        const Box& rb = B.nodes[0].box;
        int e_root = -100;
        for (int k = 0; k < 3; k++)
            e_root = std::max(e_root, (int)exponent_byte(rb.hi[k] - rb.lo[k], node_coord_slack(rb.lo[k], rb.hi[k]), -100) - 127);
        stats.e_floor = e_root - 25;
    }
    const int e_lo = stats.e_floor;
    uint64_t tri_running = 0;
    int64_t leaves = 0;
    for (int depth = 1; !level.empty(); depth++) {
        stats.level_start.push_back(level[0].wide);     // breadth-first emission: the first node of this level
        stats.depth = depth;
        const int64_t n_items = (int64_t)level.size();
        // ---- (A) children, node box, slots
#pragma omp parallel for schedule(dynamic, 256)
        for (int64_t it_ = 0; it_ < n_items; it_++) {
            Item& w = level[(size_t)it_];
            int32_t* ch = w.ch; bool* ch_leaf = w.ch_leaf; int nc = 0;
            const BNode& root = B.nodes[w.bnode];
            // children of the wide node rooted at w.bnode: follow the recorded decisions
            struct It { int32_t n; int i; };
            It st[16]; int sp = 0;
            if (root.count > 0 || root.scount <= 3) { ch[nc] = w.bnode; ch_leaf[nc++] = true; }   // a tiny mesh: the root holds one leaf
            else {
                const int k = B.dp[w.bnode].k8;
                st[sp++] = {root.right, 8 - k}; st[sp++] = {root.left, k};
            }
            while (sp > 0) {
                const It it = st[--sp];
                const BNode& m = B.nodes[it.n];
                if (m.count > 0) { ch[nc] = it.n; ch_leaf[nc++] = true; continue; }
                if (it.i == 1) { ch[nc] = it.n; ch_leaf[nc++] = B.dp[it.n].d[0] == 0; continue; }
                const int k = B.dp[it.n].d[it.i - 1];
                if (k == 0) st[sp++] = {it.n, it.i - 1};
                else { st[sp++] = {m.right, it.i - k}; st[sp++] = {m.left, k}; }
            }
            w.nc = nc;
            Box nb; nb.reset();
            for (int i = 0; i < nc; i++) nb.grow(B.nodes[ch[i]].box);
            w.nb = nb;
            // slot s prefers the child lying towards corner s (bit2=+x, bit1=+y, bit0=+z)
            float ncx[3]; for (int k = 0; k < 3; k++) ncx[k] = 0.5f * (nb.lo[k] + nb.hi[k]);
            float cost[8][8];
            for (int i = 0; i < nc; i++) {
                const Box& cbx = B.nodes[ch[i]].box;
                float off[3]; for (int k = 0; k < 3; k++) off[k] = 0.5f * (cbx.lo[k] + cbx.hi[k]) - ncx[k];
                for (int s = 0; s < 8; s++)
                    cost[i][s] = ((s & 4) ? off[0] : -off[0]) + ((s & 2) ? off[1] : -off[1]) + ((s & 1) ? off[2] : -off[2]);
            }
            int* slot_child = w.slot_child; for (int s = 0; s < 8; s++) slot_child[s] = -1;
            bool child_done[8] = {false, false, false, false, false, false, false, false};
            for (int it = 0; it < nc; it++) {
                float bestc = -INFINITY; int bi = -1, bs = -1;
                for (int i = 0; i < nc; i++) {
                    if (child_done[i]) continue;
                    for (int s = 0; s < 8; s++) {
                        if (slot_child[s] >= 0) continue;
                        if (cost[i][s] > bestc) { bestc = cost[i][s]; bi = i; bs = s; }
                    }
                }
                slot_child[bs] = bi; child_done[bi] = true;
            }
            uint32_t ni = 0, nt = 0;
            for (int s = 0; s < 8; s++) {
                const int i = slot_child[s];
                if (i < 0) continue;
                if (ch_leaf[i]) nt += (uint32_t)B.nodes[ch[i]].scount; else ni++;
            }
            w.n_internal = ni; w.n_tris = nt;
        }
        // ---- (B) indices, in node order; the next level's nodes in slot order
        next.clear();
        uint64_t node_running = out_nodes.size();
        for (int64_t it_ = 0; it_ < n_items; it_++) {
            Item& w = level[(size_t)it_];
            w.child_base = (uint32_t)node_running; w.tri_base = (uint32_t)tri_running;
            for (int s = 0; s < 8; s++) {
                const int i = w.slot_child[s];
                if (i < 0 || w.ch_leaf[i]) continue;
                Item c; c.bnode = w.ch[i]; c.wide = (uint32_t)node_running++;
                next.push_back(c);
            }
            tri_running += w.n_tris;
        }
        out_nodes.resize((size_t)node_running);
        // ---- (C) quantise and write
#pragma omp parallel for schedule(dynamic, 256) reduction(+ : leaves)
        for (int64_t it_ = 0; it_ < n_items; it_++) {
            const Item& w = level[(size_t)it_];
            const int32_t* ch = w.ch; const bool* ch_leaf = w.ch_leaf; const int* slot_child = w.slot_child;
            const Box& nb = w.nb;
            Node8 nd;
            memset(&nd, 0, sizeof(nd));
            nd.ex = exponent_byte(nb.hi[0] - nb.lo[0], node_coord_slack(nb.lo[0], nb.hi[0]), e_lo);
            nd.ey = exponent_byte(nb.hi[1] - nb.lo[1], node_coord_slack(nb.lo[1], nb.hi[1]), e_lo);
            nd.ez = exponent_byte(nb.hi[2] - nb.lo[2], node_coord_slack(nb.lo[2], nb.hi[2]), e_lo);
            const float cell[3] = {std::ldexp(1.f, (int)nd.ex - 127), std::ldexp(1.f, (int)nd.ey - 127), std::ldexp(1.f, (int)nd.ez - 127)};
            // conservative slack: 4e-3 of a cell (covers the rounding of the traversal's folded plane bias, ptb_bvh8.h planes4) plus a
            // few ulps of the coordinate
            float eps[3], p[3];
            for (int k = 0; k < 3; k++) {
                eps[k] = cell[k] * 4e-3f + node_coord_slack(nb.lo[k], nb.hi[k]);
                p[k] = nb.lo[k] - eps[k];
            }
            nd.px = p[0]; nd.py = p[1]; nd.pz = p[2];
            nd.child_base = w.child_base;
            nd.tri_base = w.tri_base;
            uint32_t tri_off = 0, valid24 = 0;
            for (int s = 0; s < 8; s++) {
                const int i = slot_child[s];
                if (i < 0) continue;
                const BNode& c = B.nodes[ch[i]];
                uint8_t* ql[3] = {nd.qlox, nd.qloy, nd.qloz};
                uint8_t* qh[3] = {nd.qhix, nd.qhiy, nd.qhiz};
                for (int k = 0; k < 3; k++) {
                    float lo = std::floor((c.box.lo[k] - eps[k] - p[k]) / cell[k]);
                    float hi = std::ceil((c.box.hi[k] + eps[k] - p[k]) / cell[k]);
                    lo = std::min(std::max(lo, 0.f), 255.f);
                    hi = std::min(std::max(hi, 0.f), 255.f);
                    ql[k][s] = (uint8_t)lo; qh[k][s] = (uint8_t)hi;
                }
                if (ch_leaf[i]) {
                    const uint32_t unary = (c.scount == 1) ? 1u : (c.scount == 2 ? 3u : 7u);
                    valid24 |= unary << (3 * s);
                    for (int t = 0; t < c.scount; t++) leaf_order[(size_t)w.tri_base + tri_off + (uint32_t)t] = B.idx[c.sfirst + t];
                    tri_off += (uint32_t)c.scount;
                    leaves++;
                } else {
                    nd.imask |= (uint8_t)(1u << s);
                }
            }
            nd.valid24[0] = (uint8_t)(valid24 & 0xffu); nd.valid24[1] = (uint8_t)((valid24 >> 8) & 0xffu); nd.valid24[2] = (uint8_t)((valid24 >> 16) & 0xffu);
            out_nodes[w.wide] = nd;
        }
        level.swap(next);
    }
    stats.leaves = leaves;
    leaf_order.resize((size_t)tri_running);
    stats.n_nodes = (int64_t)out_nodes.size();
    stats.level_start.push_back((uint32_t)out_nodes.size());
    stats.n_binary_nodes = B.n_nodes.load();
}

}  // namespace ptb
