// Binned-SAH BVH2 builder emitting the 64-byte two-stream FlattenedBVH layout (see bvh_build.h, include/b200rt.h).
#include "bvh_build.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstring>
#include <limits>
#include <stdexcept>

#include <omp.h>

namespace b200rt {
namespace {

constexpr float kInf = std::numeric_limits<float>::infinity();

struct Box
{
    float lo[3] = { kInf, kInf, kInf };
    float hi[3] = { -kInf, -kInf, -kInf };
    void grow(const float* p) { for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], p[a]); hi[a] = std::max(hi[a], p[a]); } }
    void grow(const Box& b) { for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], b.lo[a]); hi[a] = std::max(hi[a], b.hi[a]); } }
    float half_area() const
    {
        float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        if (!(dx >= 0.0f) || !(dy >= 0.0f) || !(dz >= 0.0f)) return 0.0f;
        return dx * dy + dy * dz + dz * dx;
    }
};

struct Prim { Box box; float c[3]; };

struct BuildNode
{
    Box box;
    int left = -1, right = -1;   // children (build-node indices) or -1
    int first = 0, count = 0;    // range in the permuted index array (leaves)
};

struct Builder
{
    const std::vector<Prim>& prims;
    std::vector<int>& order;
    std::vector<BuildNode> nodes;
    std::atomic<int> n_nodes{ 0 };
    int max_leaf, bins;

    Builder(const std::vector<Prim>& p, std::vector<int>& o, int max_leaf_, int bins_)
        : prims(p), order(o), nodes(2 * p.size() + 2), max_leaf(max_leaf_), bins(bins_) {}

    int alloc() { return n_nodes.fetch_add(1); }

    void make_leaf(int me, int first, int count) { nodes[me].first = first; nodes[me].count = count; nodes[me].left = nodes[me].right = -1; }

    void build(int me, int first, int count, int depth)
    {
        Box box, cbox;
        for (int i = first; i < first + count; i++)
        {
            const Prim& p = prims[order[i]];
            box.grow(p.box);
            cbox.grow(p.c);
        }
        nodes[me].box = box;
        if (count <= 1) { make_leaf(me, first, count); return; }

        int split = -1;   // number of primitives going left
        const bool force_median = depth >= 28;   // keeps total depth < kMaxTraversalDepth for any input
        if (!force_median)
        {
            // binned SAH over all three axes
            float best_cost = kInf; int best_axis = -1, best_bin = -1;
            const int B = bins;
            for (int axis = 0; axis < 3; axis++)
            {
                float cmin = cbox.lo[axis], cmax = cbox.hi[axis];
                if (!(cmax > cmin)) continue;
                float scale = B / (cmax - cmin);
                Box bbox[32]; int bcount[32];
                for (int b = 0; b < B; b++) bcount[b] = 0;
                for (int i = first; i < first + count; i++)
                {
                    const Prim& p = prims[order[i]];
                    int b = std::min(B - 1, std::max(0, (int)((p.c[axis] - cmin) * scale)));
                    bbox[b].grow(p.box); bcount[b]++;
                }
                float right_area[32]; int right_cnt[32];
                Box acc; int cnt = 0;
                for (int b = B - 1; b > 0; b--) { acc.grow(bbox[b]); cnt += bcount[b]; right_area[b] = acc.half_area(); right_cnt[b] = cnt; }
                Box lacc; int lcnt = 0;
                for (int b = 0; b < B - 1; b++)
                {
                    lacc.grow(bbox[b]); lcnt += bcount[b];
                    if (lcnt == 0 || right_cnt[b + 1] == 0) continue;
                    float cost = lacc.half_area() * lcnt + right_area[b + 1] * right_cnt[b + 1];
                    if (cost < best_cost) { best_cost = cost; best_axis = axis; best_bin = b; }
                }
            }
            float parent_area = box.half_area();
            float leaf_cost = (float)count;
            float split_cost = parent_area > 0.0f ? 1.0f + best_cost / parent_area : kInf;
            if (best_axis >= 0 && (count > max_leaf || split_cost < leaf_cost))
            {
                float cmin = cbox.lo[best_axis], cmax = cbox.hi[best_axis];
                float scale = bins / (cmax - cmin);
                int* b = order.data() + first;
                int* mid = std::partition(b, b + count, [&](int id) {
                    int bin = std::min(bins - 1, std::max(0, (int)((prims[id].c[best_axis] - cmin) * scale)));
                    return bin <= best_bin;
                });
                split = (int)(mid - b);
            }
            else if (count <= max_leaf) { make_leaf(me, first, count); return; }
        }
        if (split <= 0 || split >= count)
        {
            // object median along the widest centroid axis (degenerate SAH, or the depth guard)
            int axis = 0;
            for (int a = 1; a < 3; a++) if (cbox.hi[a] - cbox.lo[a] > cbox.hi[axis] - cbox.lo[axis]) axis = a;
            if (count <= max_leaf && !(cbox.hi[axis] > cbox.lo[axis])) { make_leaf(me, first, count); return; }
            split = count / 2;
            int* b = order.data() + first;
            std::nth_element(b, b + split, b + count, [&](int x, int y) { return prims[x].c[axis] < prims[y].c[axis]; });
        }
        int l = alloc(), r = alloc();
        nodes[me].left = l; nodes[me].right = r;
        if (count > 20000)
        {
#pragma omp task default(shared) firstprivate(l, first, split, depth)
            build(l, first, split, depth + 1);
#pragma omp task default(shared) firstprivate(r, first, split, count, depth)
            build(r, first + split, count - split, depth + 1);
#pragma omp taskwait
        }
        else
        {
            build(l, first, split, depth + 1);
            build(r, first + split, count - split, depth + 1);
        }
    }
};

// leaf reference: ~((first << 4) | count), count in 0..15 — one int carries the whole triangle range
inline int leaf_ref(int first, int count) { return ~((first << 4) | count); }

struct Slabs
{
    float lo[3], hi[3], dnear[4], dfar[4];
    void reset()
    {
        for (int a = 0; a < 3; a++) { lo[a] = kInf; hi[a] = -kInf; }
        for (int k = 0; k < 4; k++) { dnear[k] = kInf; dfar[k] = -kInf; }
    }
    void grow_point(const float* p)
    {
        for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], p[a]); hi[a] = std::max(hi[a], p[a]); }
        for (int k = 0; k < 4; k++)
        {
            // exact in double (three floats sum without error in 53 bits for any sane exponent spread), rounded outward below
            double d = 0.0;
            switch (k)
            {
            case 0: d = (double)p[0] + (double)p[1] + (double)p[2]; break;
            case 1: d = -(double)p[0] + (double)p[1] + (double)p[2]; break;
            case 2: d = -(double)p[0] - (double)p[1] + (double)p[2]; break;
            default: d = (double)p[0] - (double)p[1] + (double)p[2]; break;
            }
            float f = (float)d;
            float fl = ((double)f > d) ? std::nextafter(f, -kInf) : f;
            float fh = ((double)f < d) ? std::nextafter(f, kInf) : f;
            dnear[k] = std::min(dnear[k], fl);
            dfar[k] = std::max(dfar[k], fh);
        }
    }
    void grow(const Slabs& s)
    {
        for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], s.lo[a]); hi[a] = std::max(hi[a], s.hi[a]); }
        for (int k = 0; k < 4; k++) { dnear[k] = std::min(dnear[k], s.dnear[k]); dfar[k] = std::max(dfar[k], s.dfar[k]); }
    }
};

LeafTriangle make_leaf_triangle(const float* tri9, int id)
{
    const float* p = tri9 + 9 * (size_t)id;
    LeafTriangle t;
    for (int a = 0; a < 3; a++)
    {
        t.a[a] = p[a];
        t.e1[a] = p[3 + a] - p[a];
        t.e2[a] = p[6 + a] - p[a];
    }
    t.prim = id; t.pad1 = 0.0f; t.pad2 = 0.0f;
    return t;
}

// the per-axis pad both layouts apply to a child box: the float slab tests must never reject a volume whose triangle the
// exact Moller-Trumbore test accepts
inline float box_pad(float lo, float hi, float abs_pad) { return 1e-5f * std::max(std::fabs(lo), std::fabs(hi)) + abs_pad; }

// One axis of a wide node: frame origin p, cell size 2^(e-127) and the 8 x 2 plane bytes from the (already padded) child boxes
// of the used slots. Cell size: 376 cells span the extent (the grid has 382; the rest absorbs the roundings below), and a
// cell is never finer than the float spacing of the coordinates. lo planes round down, hi planes up, on the grid
// v(q) = 128 + q (q < 128), 2q (q >= 128).
void quantise_slots(WideNode& w, int a, const float* klo, const float* khi, const bool* used, bool& overflow)
{
    float lo = kInf, hi = -kInf;
    for (int s = 0; s < 8; s++)
        if (used[s]) { lo = std::min(lo, klo[s]); hi = std::max(hi, khi[s]); }
    if (!(lo <= hi)) { lo = 0.0f; hi = 0.0f; }
    const double extent = (double)hi - (double)lo;
    int e = -100;
    if (extent > 0.0) { int ex; std::frexp(extent / 376.0, &ex); e = ex; }      // 2^ex > extent / 376
    const double amax = std::max(std::fabs((double)lo), std::fabs((double)hi));
    if (amax > 0.0) e = std::max(e, std::ilogb(amax) - 23);
    e = std::min(126, std::max(-100, e));
    const double cell = std::ldexp(1.0, e);
    const double pd = (double)lo - 128.0 * cell;
    float pf = (float)pd;
    if ((double)pf > pd) pf = std::nextafter(pf, -kInf);
    w.p[a] = pf;
    w.e[a] = (uint8_t)(e + 127);
    uint8_t* qlo = a == 0 ? w.lox : (a == 1 ? w.loy : w.loz);
    uint8_t* qhi = a == 0 ? w.hix : (a == 1 ? w.hiy : w.hiz);
    for (int s = 0; s < 8; s++)
    {
        qlo[s] = 255; qhi[s] = 0;                                                 // empty slots: inverted, never hit
        if (!used[s]) continue;
        long vl = (long)std::floor(((double)klo[s] - (double)pf) / cell);
        long vh = (long)std::ceil(((double)khi[s] - (double)pf) / cell);
        if (vl < 128 || vh > 510) overflow = true;
        vl = std::min(510L, std::max(128L, vl)); vh = std::min(510L, std::max(128L, vh));
        if (vl >= 256) vl &= ~1L;
        if (vh >= 256 && (vh & 1)) vh++;
        if (vh > 510) { overflow = true; vh = 510; }
        qlo[s] = (uint8_t)(vl < 256 ? vl - 128 : vl / 2);
        qhi[s] = (uint8_t)(vh < 256 ? vh - 128 : vh / 2);
    }
}

// Collapses the binary tree into the 8-ary quantised layout (WideNode) and fixes the order of the triangle stream:
// the triangles of a node's leaf children are contiguous, in slot order.
struct WideBuilder
{
    const Builder& b;
    const float* tri9;
    FlatBVH& out;
    float abs_pad;
    std::vector<int>& leaf_first;       // binary build node (leaf) -> first slot of its triangles
    int max_depth = 0;
    bool overflow = false;

    void emit_triangles(const BuildNode& n)
    {
        for (int i = 0; i < n.count; i++) out.tris.push_back(make_leaf_triangle(tri9, b.order[n.first + i]));
    }

    void quantise_axis(WideNode& w, int a, const int* kids, const int* slot_of, int nk)
    {
        float klo[8], khi[8]; bool used[8] = {};
        for (int k = 0; k < nk; k++)
        {
            const Box& bx = b.nodes[kids[k]].box;
            if (!(bx.lo[a] <= bx.hi[a])) continue;                                           // empty leaf
            const float pad = box_pad(bx.lo[a], bx.hi[a], abs_pad);
            klo[slot_of[k]] = bx.lo[a] - pad; khi[slot_of[k]] = bx.hi[a] + pad; used[slot_of[k]] = true;
        }
        quantise_slots(w, a, klo, khi, used, overflow);
    }

    // fills wide node `me` from binary inner node `bn`
    void emit(int bn, int me, int depth)
    {
        max_depth = std::max(max_depth, depth);
        // 1. greedy collapse: keep opening the inner child with the largest surface area until 8 children
        int kids[8]; int nk = 0;
        kids[nk++] = b.nodes[bn].left; kids[nk++] = b.nodes[bn].right;
        while (nk < 8)
        {
            int best = -1; float best_area = -1.0f;
            for (int k = 0; k < nk; k++)
            {
                const BuildNode& c = b.nodes[kids[k]];
                if (c.left < 0) continue;
                const float ar = c.box.half_area();
                if (ar > best_area) { best_area = ar; best = k; }
            }
            if (best < 0) break;
            const BuildNode& c = b.nodes[kids[best]];
            kids[best] = c.left; kids[nk++] = c.right;
        }
        // 2. slots: greedy assignment maximising sum of (child centre - node centre) . octant direction, so that
        //    slot ^ (7 - ray octant) visits the children front to back
        const Box& nb = b.nodes[bn].box;
        float nc[3];
        for (int a = 0; a < 3; a++) nc[a] = 0.5f * (nb.lo[a] + nb.hi[a]);
        float cost[8][8];
        for (int k = 0; k < nk; k++)
        {
            const Box& cb = b.nodes[kids[k]].box;
            float cc[3];
            for (int a = 0; a < 3; a++) cc[a] = (cb.lo[a] <= cb.hi[a]) ? 0.5f * (cb.lo[a] + cb.hi[a]) - nc[a] : 0.0f;
            for (int s = 0; s < 8; s++) cost[k][s] = ((s & 1) ? cc[0] : -cc[0]) + ((s & 2) ? cc[1] : -cc[1]) + ((s & 4) ? cc[2] : -cc[2]);
        }
        int slot_of[8]; bool slot_used[8] = {}; bool kid_done[8] = {};
        for (int round = 0; round < nk; round++)
        {
            int bk = -1, bs = -1; float bc = -kInf;
            for (int k = 0; k < nk; k++)
            {
                if (kid_done[k]) continue;
                for (int s = 0; s < 8; s++)
                    if (!slot_used[s] && cost[k][s] > bc) { bc = cost[k][s]; bk = k; bs = s; }
            }
            slot_of[bk] = bs; kid_done[bk] = true; slot_used[bs] = true;
        }
        // 3. the node
        WideNode w;
        std::memset(&w, 0, sizeof(w));
        int kid_in_slot[8];
        for (int s = 0; s < 8; s++) kid_in_slot[s] = -1;
        for (int k = 0; k < nk; k++) kid_in_slot[slot_of[k]] = k;
        int n_inner = 0;
        for (int s = 0; s < 8; s++)
            if (kid_in_slot[s] >= 0 && b.nodes[kids[kid_in_slot[s]]].left >= 0) { w.imask |= (uint8_t)(1u << s); n_inner++; }
        w.child_base = (uint32_t)out.wide.size();
        w.tri_base = (uint32_t)out.tris.size();
        out.wide.resize(out.wide.size() + (size_t)n_inner);
        for (int s = 0; s < 8; s++)
        {
            const int k = kid_in_slot[s];
            if (k < 0) continue;
            const BuildNode& c = b.nodes[kids[k]];
            if (c.left >= 0) continue;
            leaf_first[kids[k]] = (int)out.tris.size();
            emit_triangles(c);
            w.valid24 |= ((1u << c.count) - 1u) << (3 * s);
        }
        for (int a = 0; a < 3; a++) quantise_axis(w, a, kids, slot_of, nk);
        out.wide[(size_t)me] = w;
        int rank = 0;
        for (int s = 0; s < 8; s++)
            if (w.imask & (1u << s)) { emit(kids[kid_in_slot[s]], (int)w.child_base + rank, depth + 1); rank++; }
    }

    // whole tree; a root that is itself a leaf becomes the only child of the root node
    void run(int root)
    {
        out.wide.clear();
        out.wide.resize(1);
        const BuildNode& rn = b.nodes[root];
        if (rn.left >= 0) { emit(root, 0, 1); return; }
        WideNode w;
        std::memset(&w, 0, sizeof(w));
        w.child_base = 1; w.tri_base = (uint32_t)out.tris.size();
        leaf_first[root] = (int)out.tris.size();
        emit_triangles(rn);
        w.valid24 = (1u << rn.count) - 1u;
        int kids[1] = { root }, slot_of[1] = { 0 };
        for (int a = 0; a < 3; a++) quantise_axis(w, a, kids, slot_of, 1);
        out.wide[0] = w;
        max_depth = 1;
    }
};

struct Flattener
{
    const Builder& b;
    const float* tri9;
    FlatBVH& out;
    float abs_pad;
    const std::vector<int>* leaf_first = nullptr;     // set when the wide builder already fixed the triangle order
    int max_depth = 0, n_leaves = 0, max_leaf = 0;
    double sah = 0.0;

    // emits the triangles of a leaf (or finds them where the wide builder put them), returns its first slot
    int emit_leaf(int bn, Slabs& s)
    {
        const BuildNode& n = b.nodes[bn];
        int first = leaf_first ? (*leaf_first)[bn] : (int)out.tris.size();
        s.reset();
        for (int i = 0; i < n.count; i++)
        {
            int id = b.order[n.first + i];
            const float* p = tri9 + 9 * (size_t)id;
            if (!leaf_first) out.tris.push_back(make_leaf_triangle(tri9, id));
            s.grow_point(p); s.grow_point(p + 3); s.grow_point(p + 6);
        }
        n_leaves++;
        max_leaf = std::max(max_leaf, n.count);
        return first;
    }

    void store_child(AxisNode& an, DiagNode& dn, bool left, const Slabs& s, int ref, int count)
    {
        float* lo = left ? an.l_lo : an.r_lo;
        float* hi = left ? an.l_hi : an.r_hi;
        float* dnear = left ? dn.l_near : dn.r_near;
        float* dfar = left ? dn.l_far : dn.r_far;
        for (int a = 0; a < 3; a++)
        {
            // pad: the (float) slab test must never reject a volume whose triangle the exact test accepts
            float pad = box_pad(s.lo[a], s.hi[a], abs_pad);
            lo[a] = s.lo[a] - pad; hi[a] = s.hi[a] + pad;
        }
        for (int k = 0; k < 4; k++)
        {
            float pad = 1e-5f * std::max(std::fabs(s.dnear[k]), std::fabs(s.dfar[k])) + 2.0f * abs_pad;
            dnear[k] = s.dnear[k] - pad; dfar[k] = s.dfar[k] + pad;
        }
        if (left) { an.l_ref = ref; an.l_count = count; } else { an.r_ref = ref; an.r_count = count; }
    }

    // returns the child reference for build node `bn` and fills its slabs
    int flatten(int bn, int depth, Slabs& s, int& count_out)
    {
        const BuildNode& n = b.nodes[bn];
        max_depth = std::max(max_depth, depth);
        if (n.left < 0)
        {
            int first = emit_leaf(bn, s);
            count_out = n.count;
            return leaf_ref(first, n.count);
        }
        int me = (int)out.axis.size();
        out.axis.emplace_back();
        out.diag.emplace_back();
        Slabs ls, rs; int lc = 0, rc = 0;
        int lref = flatten(n.left, depth + 1, ls, lc);
        int rref = flatten(n.right, depth + 1, rs, rc);
        store_child(out.axis[me], out.diag[me], true, ls, lref, lc);
        store_child(out.axis[me], out.diag[me], false, rs, rref, rc);
        s = ls; s.grow(rs);
        count_out = 0;
        return me;
    }
};

} // namespace

void build_flat_bvh(const float* tri9, int n_tri, const b200rt_bvh_options& opts, FlatBVH& out)
{
    auto t0 = std::chrono::high_resolution_clock::now();
    out.wide.clear(); out.axis.clear(); out.diag.clear(); out.tris.clear();
    const int max_leaf = std::min(15, std::max(1, opts.max_leaf_size > 0 ? opts.max_leaf_size : kWideMaxLeaf));
    const int bins = std::min(32, std::max(4, opts.sah_bins > 0 ? opts.sah_bins : 16));

    std::vector<Prim> prims((size_t)n_tri);
    std::vector<int> order((size_t)n_tri);
    float scene_abs = 0.0f;
#pragma omp parallel for reduction(max : scene_abs) schedule(static)
    for (int i = 0; i < n_tri; i++)
    {
        const float* p = tri9 + 9 * (size_t)i;
        Prim& pr = prims[i];
        pr.box.grow(p); pr.box.grow(p + 3); pr.box.grow(p + 6);
        for (int a = 0; a < 3; a++)
        {
            pr.c[a] = 0.5f * (pr.box.lo[a] + pr.box.hi[a]);
            scene_abs = std::max(scene_abs, std::max(std::fabs(pr.box.lo[a]), std::fabs(pr.box.hi[a])));
        }
        order[i] = i;
    }
    if (!std::isfinite(scene_abs)) scene_abs = 1.0f;

    Builder builder(prims, order, max_leaf, bins);
    int root = builder.alloc();
    const int threads = opts.num_threads > 0 ? opts.num_threads : omp_get_num_procs();   // not omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1
    if (n_tri > 0)
    {
#pragma omp parallel num_threads(threads)
#pragma omp single
        builder.build(root, 0, n_tri, 0);
    }
    else builder.make_leaf(root, 0, 0);

    const float abs_pad = 2e-6f * scene_abs + 1e-30f;
    out.axis.reserve((size_t)std::max(1, n_tri / 2));
    out.tris.reserve((size_t)n_tri);
    // the 8-ary layout first (it fixes the triangle order), when the leaves are small enough for its unary counts
    std::vector<int> leaf_first;
    int wide_depth = 0;
    if (max_leaf <= kWideMaxLeaf)
    {
        leaf_first.assign((size_t)builder.n_nodes.load(), 0);
        out.wide.reserve((size_t)std::max(1, n_tri / 4));
        WideBuilder wb{ builder, tri9, out, abs_pad, leaf_first };
        wb.run(root);
        if (wb.overflow) throw std::runtime_error("wide BVH quantisation overflow");
        wide_depth = wb.max_depth;
    }
    Flattener fl{ builder, tri9, out, abs_pad };
    if (!leaf_first.empty()) fl.leaf_first = &leaf_first;
    Slabs s; int cnt = 0;
    const BuildNode& rn = builder.nodes[root];
    if (rn.left < 0)
    {
        // a single leaf (or an empty scene): wrap it in one inner record whose right child is an empty, unhittable leaf
        out.axis.emplace_back(); out.diag.emplace_back();
        Slabs ls; int first = fl.emit_leaf(root, ls);
        if (rn.count == 0) ls.reset();
        fl.store_child(out.axis[0], out.diag[0], true, ls, leaf_ref(first, rn.count), rn.count);
        Slabs empty; empty.reset();
        AxisNode& an = out.axis[0]; DiagNode& dn = out.diag[0];
        for (int a = 0; a < 3; a++) { an.r_lo[a] = kInf; an.r_hi[a] = -kInf; if (rn.count == 0) { an.l_lo[a] = kInf; an.l_hi[a] = -kInf; } }
        for (int k = 0; k < 4; k++) { dn.r_near[k] = kInf; dn.r_far[k] = -kInf; if (rn.count == 0) { dn.l_near[k] = kInf; dn.l_far[k] = -kInf; } }
        an.r_ref = leaf_ref((int)out.tris.size(), 0); an.r_count = 0;
        fl.max_depth = 1;
    }
    else fl.flatten(root, 0, s, cnt);

    // SAH cost of the final tree (diagnostic): sum over inner nodes of child areas / root area
    double root_area = std::max(1e-30f, builder.nodes[root].box.half_area());
    double sah = 0.0;
    for (int i = 0; i < builder.n_nodes.load(); i++)
    {
        const BuildNode& n = builder.nodes[i];
        double a = n.box.half_area() / root_area;
        sah += (n.left < 0) ? a * n.count : a;
    }

    auto t1 = std::chrono::high_resolution_clock::now();
    out.info.n_triangles = n_tri;
    out.info.n_inner_nodes = (int)out.axis.size();
    out.info.n_leaves = fl.n_leaves;
    out.info.max_leaf_size = fl.max_leaf;
    out.info.max_depth = fl.max_depth + 1;
    out.info.has_diag_slabs = opts.use_diag_slabs ? 1 : 0;
    out.info.build_seconds = std::chrono::duration<double>(t1 - t0).count();
    out.info.sah_cost = sah;
    out.info.n_wide_nodes = (int)out.wide.size();
    out.info.wide_max_depth = wide_depth;
}

// SAH cost of a flattened tree from its binary records (the same figure build_flat_bvh reports: sum over nodes of area / root area,
// leaves weighted by their triangle count), for trees that were not built here (the device builder's)
double sah_cost_of(const FlatBVH& bvh)
{
    if (bvh.axis.empty()) return 0.0;
    auto half_area = [](const float* lo, const float* hi) {
        const double dx = (double)hi[0] - lo[0], dy = (double)hi[1] - lo[1], dz = (double)hi[2] - lo[2];
        return (dx < 0 || dy < 0 || dz < 0) ? 0.0 : dx * dy + dy * dz + dz * dx;
    };
    const AxisNode& r = bvh.axis[0];
    float lo[3], hi[3];
    for (int a = 0; a < 3; a++) { lo[a] = std::min(r.l_lo[a], r.r_lo[a]); hi[a] = std::max(r.l_hi[a], r.r_hi[a]); }
    const double root_area = std::max(1e-30, half_area(lo, hi));
    double sah = 1.0;
    for (const AxisNode& n : bvh.axis)
    {
        const double al = half_area(n.l_lo, n.l_hi) / root_area, ar = half_area(n.r_lo, n.r_hi) / root_area;
        sah += n.l_ref >= 0 ? al : al * n.l_count;
        sah += n.r_ref >= 0 ? ar : ar * n.r_count;
    }
    return sah;
}

// The top level over triangles kept out of the tree (the device builder's outsized ones), in front of both layouts' roots: the old root
// record moves behind the existing records, record 0 becomes a top-level node whose one inner child is the old root (or the next
// top-level node) and whose other children are leaves holding the extra triangles (8-ary: 7 leaves x 3 triangles per node; binary: one
// leaf of up to 15 per record). Works from record 0 of each layout and the extra triangles' vertices alone, so a tree that lives on the
// device needs only those few records on the host.
void make_top_level(const WideNode& w0, const AxisNode& a0, size_t n_wide, size_t n_axis, size_t first_slot, const float* extra9, int n_extra,
                    float abs_pad, TopLevel& out, b200rt_bvh_info& info)
{
    out.wide.clear(); out.axis.clear();
    if (n_extra <= 0) return;
    std::vector<Box> tbox((size_t)n_extra);
    for (int i = 0; i < n_extra; i++)
    {
        const float* p = extra9 + 9 * (size_t)i;
        tbox[i].grow(p); tbox[i].grow(p + 3); tbox[i].grow(p + 6);
        for (int a = 0; a < 3; a++) { const float pad = box_pad(tbox[i].lo[a], tbox[i].hi[a], abs_pad); tbox[i].lo[a] -= pad; tbox[i].hi[a] += pad; }
    }
    // ---- 8-ary layout
    {
        Box root;                                                   // the old root's extent: union of its decoded child boxes
        const uint8_t* ql[3] = { w0.lox, w0.loy, w0.loz };
        const uint8_t* qh[3] = { w0.hix, w0.hiy, w0.hiz };
        for (int s = 0; s < 8; s++)
        {
            if (!((w0.imask >> s) & 1) && !((w0.valid24 >> (3 * s)) & 7u)) continue;
            float lo[3], hi[3];
            for (int a = 0; a < 3; a++)
            {
                const double cell = std::ldexp(1.0, (int)w0.e[a] - 127);
                const double dl = (double)w0.p[a] + cell * wide_grid_value(ql[a][s]), dh = (double)w0.p[a] + cell * wide_grid_value(qh[a][s]);
                lo[a] = (float)dl; if ((double)lo[a] > dl) lo[a] = std::nextafter(lo[a], -kInf);
                hi[a] = (float)dh; if ((double)hi[a] < dh) hi[a] = std::nextafter(hi[a], kInf);
            }
            root.grow(lo); root.grow(hi);
        }
        const int per_node = 7 * kWideMaxLeaf;
        const int n_top = top_level_wide(n_extra);
        const size_t moved = n_wide;
        out.wide.resize((size_t)n_top + 1);                         // [0]: record 0; [1 + j]: record moved + j (the old root, then top node j)
        out.wide[1] = w0;
        std::vector<Box> below((size_t)n_top + 1);                 // extent of everything under top node k's inner child
        below[(size_t)n_top] = root;
        for (int k = n_top - 1; k >= 0; k--)
        {
            below[(size_t)k] = below[(size_t)k + 1];
            for (int i = k * per_node; i < std::min(n_extra, (k + 1) * per_node); i++) below[(size_t)k].grow(tbox[i]);
        }
        bool overflow = false;
        for (int k = 0; k < n_top; k++)
        {
            WideNode w;
            std::memset(&w, 0, sizeof(w));
            float klo[3][8], khi[3][8]; bool used[8] = {};
            w.imask = 1;                                            // slot 0: the rest of the structure
            w.child_base = (uint32_t)(k + 1 < n_top ? moved + (size_t)k + 1 : moved);
            w.tri_base = (uint32_t)(first_slot + (size_t)k * per_node);
            used[0] = true;
            for (int a = 0; a < 3; a++) { klo[a][0] = below[(size_t)k + 1].lo[a]; khi[a][0] = below[(size_t)k + 1].hi[a]; }
            for (int s = 1; s < 8; s++)
            {
                const int i0 = k * per_node + (s - 1) * kWideMaxLeaf, cnt = std::min(kWideMaxLeaf, n_extra - i0);
                if (cnt <= 0) break;
                Box lb;
                for (int i = i0; i < i0 + cnt; i++) lb.grow(tbox[i]);
                used[s] = true;
                for (int a = 0; a < 3; a++) { klo[a][s] = lb.lo[a]; khi[a][s] = lb.hi[a]; }
                w.valid24 |= ((1u << cnt) - 1u) << (3 * s);
            }
            for (int a = 0; a < 3; a++) quantise_slots(w, a, klo[a], khi[a], used, overflow);
            out.wide[k == 0 ? 0 : 1 + (size_t)k] = w;
        }
        if (overflow) throw std::runtime_error("wide BVH quantisation overflow (top level)");
        info.n_wide_nodes = (int)(n_wide + (size_t)n_top);
        info.wide_max_depth += n_top;
    }
    // ---- binary layout
    {
        Box root;
        root.grow(a0.l_lo); root.grow(a0.l_hi);
        if (a0.r_lo[0] <= a0.r_hi[0]) { root.grow(a0.r_lo); root.grow(a0.r_hi); }
        const int per_rec = 15;
        const int n_top = top_level_axis(n_extra);
        const size_t moved = n_axis;
        out.axis.resize((size_t)n_top + 1);
        out.axis[1] = a0;
        std::vector<Box> below((size_t)n_top + 1);
        below[(size_t)n_top] = root;
        for (int k = n_top - 1; k >= 0; k--)
        {
            below[(size_t)k] = below[(size_t)k + 1];
            for (int i = k * per_rec; i < std::min(n_extra, (k + 1) * per_rec); i++) below[(size_t)k].grow(tbox[i]);
        }
        for (int k = 0; k < n_top; k++)
        {
            AxisNode an;
            const int i0 = k * per_rec, cnt = std::min(per_rec, n_extra - i0);
            Box lb;
            for (int i = i0; i < i0 + cnt; i++) lb.grow(tbox[i]);
            for (int a = 0; a < 3; a++)
            {
                an.l_lo[a] = below[(size_t)k + 1].lo[a]; an.l_hi[a] = below[(size_t)k + 1].hi[a];
                an.r_lo[a] = lb.lo[a]; an.r_hi[a] = lb.hi[a];
            }
            an.l_ref = (int)(k + 1 < n_top ? moved + (size_t)k + 1 : moved); an.l_count = 0;
            an.r_ref = leaf_ref((int)(first_slot + (size_t)i0), cnt); an.r_count = cnt;
            out.axis[k == 0 ? 0 : 1 + (size_t)k] = an;
        }
        info.n_inner_nodes = (int)(n_axis + (size_t)n_top);
        info.n_leaves += n_top;
        info.max_depth += n_top;
        info.max_leaf_size = std::max(info.max_leaf_size, std::min(per_rec, n_extra));
    }
}

// 8-ary layout: every triangle slot referenced exactly once, every decoded child box contains all vertices below it
// (decoded in double: plane = p + 2^e * v(q), exactly what the device evaluates up to its final roundings)
static int check_wide_bvh(const FlatBVH& bvh, const float* tri9, int n_tri)
{
    struct Bounds { double lo[3], hi[3]; };
    std::vector<char> seen((size_t)std::max(1, n_tri), 0);
    int covered = 0, err = 0;
    // recursive walk returning the exact vertex bounds of a subtree
    struct Walker
    {
        const FlatBVH& bvh; const float* tri9; int n_tri; std::vector<char>& seen; int& covered; int& err;
        void walk(size_t ni, int depth, Bounds& bd)
        {
            for (int a = 0; a < 3; a++) { bd.lo[a] = 1e300; bd.hi[a] = -1e300; }
            if (err) return;
            if (depth > kMaxTraversalDepth) { err = 25; return; }
            if (ni >= bvh.wide.size()) { err = 20; return; }
            const WideNode w = bvh.wide[ni];
            int rank = 0;
            for (int s = 0; s < 8 && !err; s++)
            {
                const unsigned m = (w.valid24 >> (3 * s)) & 7u;
                const bool inner = (w.imask >> s) & 1;
                if (inner && m) { err = 21; return; }
                if (!inner && !m) continue;
                Bounds cb;
                for (int a = 0; a < 3; a++) { cb.lo[a] = 1e300; cb.hi[a] = -1e300; }
                if (inner)
                {
                    walk((size_t)w.child_base + rank, depth + 1, cb);
                    rank++;
                }
                else
                {
                    const int count = m == 1 ? 1 : (m == 3 ? 2 : (m == 7 ? 3 : -1));
                    if (count < 0) { err = 22; return; }
                    unsigned below = 0;
                    for (int b2 = 0; b2 < 3 * s; b2++) below += (w.valid24 >> b2) & 1u;
                    for (int i = 0; i < count; i++)
                    {
                        const size_t slot = (size_t)w.tri_base + below + i;
                        if (slot >= bvh.tris.size()) { err = 23; return; }
                        if (seen[slot]++) { err = 23; return; }
                        covered++;
                        const float* p = tri9 + 9 * (size_t)bvh.tris[slot].prim;
                        for (int v = 0; v < 3; v++)
                            for (int a = 0; a < 3; a++) { cb.lo[a] = std::min(cb.lo[a], (double)p[3 * v + a]); cb.hi[a] = std::max(cb.hi[a], (double)p[3 * v + a]); }
                    }
                }
                if (err) return;
                const uint8_t* ql[3] = { w.lox, w.loy, w.loz };
                const uint8_t* qh[3] = { w.hix, w.hiy, w.hiz };
                for (int a = 0; a < 3; a++)
                {
                    const double cell = std::ldexp(1.0, (int)w.e[a] - 127);
                    const double lo = (double)w.p[a] + cell * wide_grid_value(ql[a][s]);
                    const double hi = (double)w.p[a] + cell * wide_grid_value(qh[a][s]);
                    if (cb.lo[a] < lo || cb.hi[a] > hi) { err = 24; return; }
                    bd.lo[a] = std::min(bd.lo[a], cb.lo[a]); bd.hi[a] = std::max(bd.hi[a], cb.hi[a]);
                }
            }
        }
    } wk{ bvh, tri9, n_tri, seen, covered, err };
    Bounds root;
    wk.walk(0, 1, root);
    if (err) return err;
    if (covered != n_tri) return 26;
    return 0;
}

int check_flat_bvh(const FlatBVH& bvh, const float* tri9, int n_tri)
{
    if ((int)bvh.tris.size() != n_tri) return 1;
    std::vector<int> seen((size_t)std::max(1, n_tri), 0);
    // every triangle exactly once, stored edges consistent
    for (const LeafTriangle& t : bvh.tris)
    {
        if (t.prim < 0 || t.prim >= n_tri) return 2;
        if (seen[t.prim]++) return 3;
        const float* p = tri9 + 9 * (size_t)t.prim;
        for (int a = 0; a < 3; a++)
            if (t.a[a] != p[a] || t.e1[a] != p[3 + a] - p[a] || t.e2[a] != p[6 + a] - p[a]) return 4;
    }
    // every child volume contains the vertices of every triangle below it (iterative walk carrying the volume chain
    // is O(n depth); instead check leaves against their own volume and inner volumes against their children's)
    struct Item { int node; int depth; };
    std::vector<Item> stack{ { 0, 1 } };
    int covered = 0;
    while (!stack.empty())
    {
        Item it = stack.back(); stack.pop_back();
        if (it.depth > kMaxTraversalDepth) return 5;
        if (it.node < 0 || it.node >= (int)bvh.axis.size()) return 6;
        const AxisNode& an = bvh.axis[it.node];
        static const DiagNode no_diag = { { -kInf, -kInf, -kInf, -kInf }, { kInf, kInf, kInf, kInf }, { -kInf, -kInf, -kInf, -kInf }, { kInf, kInf, kInf, kInf } };
        const DiagNode& dn = bvh.diag.empty() ? no_diag : bvh.diag[it.node];      // the device builder emits no diagonal slabs
        for (int side = 0; side < 2; side++)
        {
            const float* lo = side ? an.r_lo : an.l_lo; const float* hi = side ? an.r_hi : an.l_hi;
            const float* dnear = side ? dn.r_near : dn.l_near; const float* dfar = side ? dn.r_far : dn.l_far;
            int ref = side ? an.r_ref : an.l_ref; int count = side ? an.r_count : an.l_count;
            if (ref >= 0)
            {
                if (count != 0) return 7;
                // child's children must be inside this volume
                if (ref >= (int)bvh.axis.size()) return 6;
                const AxisNode& cn = bvh.axis[ref];
                const DiagNode& cd = bvh.diag.empty() ? no_diag : bvh.diag[ref];
                for (int cs = 0; cs < 2; cs++)
                {
                    const float* clo = cs ? cn.r_lo : cn.l_lo; const float* chi = cs ? cn.r_hi : cn.l_hi;
                    const float* cnear = cs ? cd.r_near : cd.l_near; const float* cfar = cs ? cd.r_far : cd.l_far;
                    if (!(clo[0] <= chi[0])) continue;   // empty child
                    for (int a = 0; a < 3; a++) if (clo[a] < lo[a] - 1e-3f * std::fabs(lo[a]) - 1e-6f || chi[a] > hi[a] + 1e-3f * std::fabs(hi[a]) + 1e-6f) return 8;
                    (void)cnear; (void)cfar;
                }
                stack.push_back({ ref, it.depth + 1 });
            }
            else
            {
                int first = (~ref) >> 4;
                if (((~ref) & 15) != count) return 13;
                if (first < 0 || first + count > n_tri) return 9;
                covered += count;
                for (int i = first; i < first + count; i++)
                {
                    const float* p = tri9 + 9 * (size_t)bvh.tris[i].prim;
                    for (int v = 0; v < 3; v++)
                    {
                        const float* q = p + 3 * v;
                        for (int a = 0; a < 3; a++) if (q[a] < lo[a] || q[a] > hi[a]) return 10;
                        for (int k = 0; k < 4; k++)
                        {
                            float d = diag_dist(k, q[0], q[1], q[2]);
                            if (d < dnear[k] || d > dfar[k]) return 11;
                        }
                    }
                }
            }
        }
    }
    if (covered != n_tri) return 12;
    if (!bvh.wide.empty())
    {
        const int r = check_wide_bvh(bvh, tri9, n_tri);
        if (r) return r;
    }
    return 0;
}

} // namespace b200rt
