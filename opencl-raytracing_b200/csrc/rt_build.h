// rt_build.h — device BVH builder: per-thread bodies of the build kernels.
//
// Replaces prepare_cpu_acceleration_structures (crates/raytracing-cpu/src/scene.rs:14-73),
// BVH2Builder::{add_tri,add_sphere,add_mesh} (crates/raytracing/src/accel/bvh2.rs:174-252) and Embree's
// rtcBuildBVH (crates/embree4/src/bvh.rs:204-254). Same primitive conventions — one build primitive per
// triangle of every root-aggregate child with (geomID = child index, primID = triangle index), world-space
// AABB of the transformed vertices; a sphere is one primitive whose box is the transformed object box
// (bvh2.rs:208-236) — but a different structure: a binary tree built on the device from the Morton order of
// the primitive centroids, then an SAH-area-guided collapse into 8-wide nodes with quantised child boxes
// (Ylitie et al. 2017 layout, 80 B).
//
// Binary tree, two builders over the same sorted Morton keys:
//   * PLOC (default; Meister & Bittner 2018, parallel locally-ordered clustering): clusters within
//     PLOC_RADIUS positions of each other in Morton order are merged bottom-up, always the mutually nearest
//     pairs by surface area of the union. A plain LBVH groups a wall-sized triangle with whatever small
//     triangles share its Morton neighbourhood and every ray then enters that fat subtree; clustering by
//     area keeps large primitives near the root. (This takes the place of the "LBVH + SAH treelet refit"
//     of the plan: same goal, one pass.)
//   * LBVH (Karras 2012) + bottom-up refit: kept for A/B comparison (RTCUDA_BUILDER=lbvh).
//
// Pipeline (one kernel each, see kernels.cu): prim_setup -> morton -> radix sort -> [ploc_init ->
// (ploc_nn -> scan -> ploc_merge)* | karras -> refit] -> collapse (one launch per wide level).
#pragma once
#include "rt_scene.h"

namespace rt {

constexpr uint32_t LEAF_MAX = 3;  // primitives per leaf child (unary count in 3 bits)

struct WorkItem { uint32_t bnode, wnode; };

struct BuildCtx {
    // inputs
    const Instance* instances;
    uint32_t instance_count;
    const float* vertices;
    const uint32_t* tris;
    uint32_t n;                 // build primitives
    // per-primitive (unsorted)
    Prim* prims_unsorted;
    float4* aabb_lo;            // xyz
    float4* aabb_hi;
    uint32_t* bounds_keys;      // 6 x u32 float_key: min xyz, max xyz
    uint64_t* keys;
    uint32_t* vals;
    // sorted order
    const uint64_t* keys_sorted;
    const uint32_t* vals_sorted;
    // binary tree: internal nodes [0, n-1), leaves [n-1, 2n-1)
    uint32_t* left;
    uint32_t* right;
    uint32_t* parent;           // 2n-1 (LBVH only)
    uint32_t* count;            // 2n-1: primitives below each node
    float4* node_lo;            // 2n-1
    float4* node_hi;
    uint32_t* visit;            // n-1 atomic counters
    // wide tree
    Node8* nodes;
    Prim* prims;
    const WorkItem* queue_in;
    WorkItem* queue_out;
    uint32_t* counters;         // [0] next-level size, [1] wide node count, [2] primitive slots handed out, [3] primitives placed
    uint32_t prim_capacity;     // slots allocated behind `prims` (writes beyond are dropped; the driver checks [2])
    // PLOC state
    const uint32_t* cl_in;      // current clusters (binary node ids) in Morton order
    uint32_t* cl_out;
    uint32_t m;                 // number of current clusters
    uint32_t* nn;               // nearest neighbour position of each cluster
    uint64_t* scan;             // per cluster: lo 32 = survives into the next round, hi 32 = leads a merge; exclusive-summed in place
    uint32_t next_node;         // internal node ids are handed out downwards from here, so the last merge creates node 0 (the root)
    uint32_t* ploc_out;         // [0] clusters after this round, [1] merges of this round
};

#ifndef RT_PLOC_RADIUS
#define RT_PLOC_RADIUS 16
#endif
constexpr int PLOC_RADIUS = RT_PLOC_RADIUS;

RT_HD uint32_t instance_of_prim(const BuildCtx& b, uint32_t i) {
    uint32_t lo = 0, hi = b.instance_count;  // last instance with prim_base <= i
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (b.instances[mid].prim_base <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// The 8 transformed corners of a sphere instance's object box (aabb.rs:81-95): its world box in the build and in the refit.
RT_HD void sphere_box(const Instance& inst, V3& lo, V3& hi) {
    V3 c = mk3(inst.center[0], inst.center[1], inst.center[2]);
    V3 r = mk3(inst.radius);
    V3 mn = c - r, mx = c + r;
    lo = mk3(RT_INF, RT_INF, RT_INF);
    hi = mk3(-RT_INF, -RT_INF, -RT_INF);
    for (int k = 0; k < 8; k++) {
        V3 q = apply_point(inst.o2w, mk3((k & 4) ? mx.x : mn.x, (k & 2) ? mx.y : mn.y, (k & 1) ? mx.z : mn.z));
        lo = vmin(lo, q);
        hi = vmax(hi, q);
    }
}

// Primitive `local` of instance g in world space and its world box: the one definition the build (prim_setup_body) and the
// refit (refit_prims_body) share, so a refit with unchanged transforms writes the bits a fresh build writes.
RT_HD void world_prim(const Instance& inst, uint32_t g, uint32_t local, const float* vertices, const uint32_t* tris, Prim& p, V3& lo, V3& hi) {
    if (inst.kind == 0) {
        const uint32_t* t = tris + 3 * (size_t)(inst.tri_offset + local);
        V3 v0 = apply_point(inst.o2w, load3(vertices, inst.vertex_offset + t[0]));
        V3 v1 = apply_point(inst.o2w, load3(vertices, inst.vertex_offset + t[1]));
        V3 v2 = apply_point(inst.o2w, load3(vertices, inst.vertex_offset + t[2]));
        lo = vmin(v0, vmin(v1, v2));
        hi = vmax(v0, vmax(v1, v2));
        p.a = make_float4(v0.x, v0.y, v0.z, u2f(g));
        p.b = make_float4(v1.x, v1.y, v1.z, u2f(local));
        p.c = make_float4(v2.x, v2.y, v2.z, u2f(0u));
    } else {
        sphere_box(inst, lo, hi);
        p.a = make_float4(inst.center[0], inst.center[1], inst.center[2], u2f(g));
        p.b = make_float4(inst.radius, 0.0f, 0.0f, u2f(0u));
        p.c = make_float4(0.0f, 0.0f, 0.0f, u2f(1u));
    }
}

RT_HD void prim_setup_body(uint32_t i, const BuildCtx& b) {
    uint32_t g = instance_of_prim(b, i);
    const Instance& inst = b.instances[g];
    V3 lo, hi;
    Prim p;
    world_prim(inst, g, i - inst.prim_base, b.vertices, b.tris, p, lo, hi);
    b.prims_unsorted[i] = p;
    b.aabb_lo[i] = make_float4(lo.x, lo.y, lo.z, 0.0f);
    b.aabb_hi[i] = make_float4(hi.x, hi.y, hi.z, 0.0f);
    atomic_min_u32(&b.bounds_keys[0], float_key(lo.x));
    atomic_min_u32(&b.bounds_keys[1], float_key(lo.y));
    atomic_min_u32(&b.bounds_keys[2], float_key(lo.z));
    atomic_max_u32(&b.bounds_keys[3], float_key(hi.x));
    atomic_max_u32(&b.bounds_keys[4], float_key(hi.y));
    atomic_max_u32(&b.bounds_keys[5], float_key(hi.z));
}

RT_HD uint64_t expand21(uint64_t v) {  // spread 21 bits to every third bit
    v &= 0x1fffffull;
    v = (v | v << 32) & 0x1f00000000ffffull;
    v = (v | v << 16) & 0x1f0000ff0000ffull;
    v = (v | v << 8) & 0x100f00f00f00f00full;
    v = (v | v << 4) & 0x10c30c30c30c30c3ull;
    v = (v | v << 2) & 0x1249249249249249ull;
    return v;
}

RT_HD void morton_body(uint32_t i, const BuildCtx& b) {
    V3 smin = mk3(key_float(b.bounds_keys[0]), key_float(b.bounds_keys[1]), key_float(b.bounds_keys[2]));
    V3 smax = mk3(key_float(b.bounds_keys[3]), key_float(b.bounds_keys[4]), key_float(b.bounds_keys[5]));
    V3 c = 0.5f * (xyz(b.aabb_lo[i]) + xyz(b.aabb_hi[i]));
    V3 ext = smax - smin;
    float fx = ext.x > 0.0f ? (c.x - smin.x) / ext.x : 0.0f;
    float fy = ext.y > 0.0f ? (c.y - smin.y) / ext.y : 0.0f;
    float fz = ext.z > 0.0f ? (c.z - smin.z) / ext.z : 0.0f;
    const float S = 2097151.0f;  // 2^21 - 1
    uint64_t x = (uint64_t)fminf(fmaxf(fx * S, 0.0f), S);
    uint64_t y = (uint64_t)fminf(fmaxf(fy * S, 0.0f), S);
    uint64_t z = (uint64_t)fminf(fmaxf(fz * S, 0.0f), S);
    b.keys[i] = (expand21(x) << 2) | (expand21(y) << 1) | expand21(z);
    b.vals[i] = i;
}

// Karras 2012: common-prefix length with index tie-break for duplicate keys.
RT_HD int delta_lbvh(const BuildCtx& b, int i, int j) {
    if (j < 0 || j >= (int)b.n) return -1;
    uint64_t x = b.keys_sorted[i] ^ b.keys_sorted[j];
    if (x == 0) return 64 + clz32((uint32_t)i ^ (uint32_t)j);
    return clz64(x);
}

RT_HD void karras_body(uint32_t idx, const BuildCtx& b) {
    const int i = (int)idx;
    const int n = (int)b.n;
    int d = (delta_lbvh(b, i, i + 1) - delta_lbvh(b, i, i - 1)) >= 0 ? 1 : -1;
    int dmin = delta_lbvh(b, i, i - d);
    int lmax = 2;
    while (delta_lbvh(b, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (delta_lbvh(b, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta_lbvh(b, i, j);
    int s = 0;
    int t = l;
    do {
        t = (t + 1) >> 1;
        if (delta_lbvh(b, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + (d < 0 ? d : 0);
    int lo = i < j ? i : j, hi = i < j ? j : i;
    uint32_t lc = (lo == gamma) ? (uint32_t)(n - 1 + gamma) : (uint32_t)gamma;
    uint32_t rc = (hi == gamma + 1) ? (uint32_t)(n - 1 + gamma + 1) : (uint32_t)(gamma + 1);
    b.left[i] = lc;
    b.right[i] = rc;
    b.parent[lc] = (uint32_t)i;
    b.parent[rc] = (uint32_t)i;
    b.count[i] = (uint32_t)(hi - lo + 1);
    if (i == 0) b.parent[0] = NONE;
}

RT_HD void refit_body(uint32_t k, const BuildCtx& b) {
    const uint32_t n = b.n;
    uint32_t node = n - 1 + k;
    uint32_t pi = b.vals_sorted[k];
    b.node_lo[node] = b.aabb_lo[pi];
    b.node_hi[node] = b.aabb_hi[pi];
    b.count[node] = 1u;
    if (n == 1) return;
    uint32_t cur = b.parent[node];
    while (cur != NONE) {
        mem_fence();
        if (atomic_add_u32(&b.visit[cur], 1u) == 0u) return;  // first child to arrive: the sibling finishes the job
        mem_fence();
        uint32_t l = b.left[cur], r = b.right[cur];
        // volatile-style reads: the sibling subtree was written by another thread
        const volatile float4* nlo = b.node_lo;
        const volatile float4* nhi = b.node_hi;
        V3 lo = vmin(mk3(nlo[l].x, nlo[l].y, nlo[l].z), mk3(nlo[r].x, nlo[r].y, nlo[r].z));
        V3 hi = vmax(mk3(nhi[l].x, nhi[l].y, nhi[l].z), mk3(nhi[r].x, nhi[r].y, nhi[r].z));
        b.node_lo[cur] = make_float4(lo.x, lo.y, lo.z, 0.0f);
        b.node_hi[cur] = make_float4(hi.x, hi.y, hi.z, 0.0f);
        cur = b.parent[cur];
    }
}

RT_HD float half_area(V3 lo, V3 hi) {
    V3 d = hi - lo;
    return d.x * d.y + d.y * d.z + d.z * d.x;
}

// ---- PLOC ------------------------------------------------------------------------------------------------
RT_HD void ploc_init_body(uint32_t k, const BuildCtx& b) {
    const uint32_t node = b.n - 1 + k;
    const uint32_t pi = b.vals_sorted[k];
    b.node_lo[node] = b.aabb_lo[pi];
    b.node_hi[node] = b.aabb_hi[pi];
    b.count[node] = 1u;
    b.cl_out[k] = node;
}

// nearest neighbour of cluster i among the clusters within PLOC_RADIUS positions: smallest union area, ties to the
// lower position (with this order the globally best pair is always mutual, so every round merges something)
RT_HD void ploc_nn_body(uint32_t i, const BuildCtx& b) {
    const uint32_t ci = b.cl_in[i];
    const V3 lo = xyz(b.node_lo[ci]), hi = xyz(b.node_hi[ci]);
    const uint32_t j0 = i > (uint32_t)PLOC_RADIUS ? i - PLOC_RADIUS : 0u;
    const uint32_t j1 = i + PLOC_RADIUS < b.m - 1 ? i + PLOC_RADIUS : b.m - 1;
    float best = RT_INF;
    uint32_t bj = NONE;
    for (uint32_t j = j0; j <= j1; j++) {
        if (j == i) continue;
        const uint32_t cj = b.cl_in[j];
        const float a = half_area(vmin(lo, xyz(b.node_lo[cj])), vmax(hi, xyz(b.node_hi[cj])));
        if (a < best || bj == NONE) { best = a; bj = j; }
    }
    b.nn[i] = bj;
}
// flags for the scan: lo word = the cluster (or the merged node that replaces it) is in the next round, hi word = merge leader
RT_HD void ploc_flag_body(uint32_t i, const BuildCtx& b) {
    const uint32_t j = b.nn[i];
    const bool mutual = j != NONE && b.nn[j] == i;
    const bool leader = mutual && i < j, absorbed = mutual && i > j;
    b.scan[i] = (absorbed ? 0ull : 1ull) | (leader ? (1ull << 32) : 0ull);
}
// after the exclusive sum of the flags: create the merged nodes and compact the cluster list, order preserved
RT_HD void ploc_merge_body(uint32_t i, const BuildCtx& b) {
    const uint32_t j = b.nn[i];
    const bool mutual = j != NONE && b.nn[j] == i;
    const uint64_t ex = b.scan[i];
    const uint32_t pos = (uint32_t)ex, rank = (uint32_t)(ex >> 32);
    if (mutual && i > j) {
        if (i == b.m - 1) { b.ploc_out[0] = pos; b.ploc_out[1] = rank; }
        return;
    }
    uint32_t id = b.cl_in[i];
    if (mutual) {
        const uint32_t l = id, r = b.cl_in[j];
        id = b.next_node - 1u - rank;
        b.left[id] = l;
        b.right[id] = r;
        const V3 lo = vmin(xyz(b.node_lo[l]), xyz(b.node_lo[r])), hi = vmax(xyz(b.node_hi[l]), xyz(b.node_hi[r]));
        b.node_lo[id] = make_float4(lo.x, lo.y, lo.z, 0.0f);
        b.node_hi[id] = make_float4(hi.x, hi.y, hi.z, 0.0f);
        b.count[id] = b.count[l] + b.count[r];
    }
    b.cl_out[pos] = id;
    if (i == b.m - 1) { b.ploc_out[0] = pos + 1u; b.ploc_out[1] = rank + (mutual ? 1u : 0u); }
}

// ---- quantised node planes (shared by the collapse and the refit) ------------------------------------------
// exponents: smallest power of two with lo + 255 * 2^e >= hi
RT_HD void node_exponents(V3 lo, V3 hi, uint32_t ebits[3]) {
    const float ext[3] = {hi.x - lo.x, hi.y - lo.y, hi.z - lo.z};
    const float lov[3] = {lo.x, lo.y, lo.z}, hiv[3] = {hi.x, hi.y, hi.z};
    for (int a = 0; a < 3; a++) {
        int e = 1;  // biased exponent
        if (ext[a] > 0.0f) {
            int ex;
            frexpf(ext[a] / 255.0f, &ex);  // ext/255 = m * 2^ex, m in [0.5, 1)
            e = ex + 127;
            if (e < 1) e = 1;
            if (e > 238) e = 238;  // rt_traverse.h folds 2^15 into the scale: e + 15 must stay a finite exponent
            while (e < 238 && lov[a] + 255.0f * u2f((uint32_t)e << 23) < hiv[a]) e++;
        }
        ebits[a] = (uint32_t)e;
    }
}

// the conservative 8-bit planes of child box [cl, ch] in slot s of a node with origin `lo`
RT_HD void quantize_child(const uint32_t ebits[3], V3 lo, V3 clo, V3 chi, int s, uint32_t q[6][8]) {
    const float lov[3] = {lo.x, lo.y, lo.z};
    const float cl[3] = {clo.x, clo.y, clo.z}, chh[3] = {chi.x, chi.y, chi.z};
    for (int a = 0; a < 3; a++) {
        const float scale = u2f(ebits[a] << 23);
        float ql = floorf((cl[a] - lov[a]) / scale);
        float qh = ceilf((chh[a] - lov[a]) / scale);
        ql = fminf(fmaxf(ql, 0.0f), 255.0f);
        qh = fminf(fmaxf(qh, 0.0f), 255.0f);
        while (ql > 0.0f && lov[a] + ql * scale > cl[a]) ql -= 1.0f;
        while (qh < 255.0f && lov[a] + qh * scale < chh[a]) qh += 1.0f;
        if (qh <= ql) { if (qh < 255.0f) qh = ql + 1.0f; else ql = qh - 1.0f; }  // never a zero-thickness slab
        q[a][s] = (uint32_t)ql;
        q[3 + a][s] = (uint32_t)qh;
    }
}

RT_HD uint32_t pack4(const uint32_t* v) { return v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24); }

// n0 and the plane words n2..n4 of a node (n1 is the caller's)
RT_HD void pack_node_planes(Node8& nd8, V3 lo, const uint32_t ebits[3], uint32_t imask, uint32_t q[6][8]) {
    nd8.n0 = make_float4(lo.x, lo.y, lo.z, u2f(ebits[0] | (ebits[1] << 8) | (ebits[2] << 16) | (imask << 24)));
    nd8.n2 = make_float4(u2f(pack4(q[0])), u2f(pack4(q[0] + 4)), u2f(pack4(q[1])), u2f(pack4(q[1] + 4)));
    nd8.n3 = make_float4(u2f(pack4(q[2])), u2f(pack4(q[2] + 4)), u2f(pack4(q[3])), u2f(pack4(q[3] + 4)));
    nd8.n4 = make_float4(u2f(pack4(q[4])), u2f(pack4(q[4] + 4)), u2f(pack4(q[5])), u2f(pack4(q[5] + 4)));
}

// One wide node per work item: gather up to 8 children by repeatedly opening the binary child with
// the largest surface area, order them into octant slots, quantise, emit child work items.
RT_HD void collapse_body(uint32_t item_idx, const BuildCtx& b) {
    const WorkItem it = b.queue_in[item_idx];
    const uint32_t n = b.n;
    const uint32_t first_leaf = n - 1;
    uint32_t ch[8];
    int nc = 0;
    if (n == 1) { ch[0] = first_leaf; nc = 1; }
    else { ch[0] = b.left[it.bnode]; ch[1] = b.right[it.bnode]; nc = 2; }

    for (int stage = 0; stage < 2; stage++) {
        while (nc < 8) {
            int best = -1;
            float best_area = -1.0f;
            for (int c = 0; c < nc; c++) {
                uint32_t nd = ch[c];
                if (nd >= first_leaf) continue;
                uint32_t cnt = b.count[nd];
                if (stage == 0 && cnt <= LEAF_MAX) continue;
                float a = half_area(xyz(b.node_lo[nd]), xyz(b.node_hi[nd]));
                if (a > best_area) { best_area = a; best = c; }
            }
            if (best < 0) break;
            uint32_t nd = ch[best];
            ch[best] = b.left[nd];
            ch[nc++] = b.right[nd];
        }
    }

    // node frame
    V3 lo = mk3(RT_INF, RT_INF, RT_INF), hi = mk3(-RT_INF, -RT_INF, -RT_INF);
    V3 clo[8], chi[8];
    for (int c = 0; c < nc; c++) {
        clo[c] = xyz(b.node_lo[ch[c]]);
        chi[c] = xyz(b.node_hi[ch[c]]);
        lo = vmin(lo, clo[c]);
        hi = vmax(hi, chi[c]);
    }
    const V3 center = 0.5f * (lo + hi);

    // greedy octant slot assignment: slot bit k set <=> child lies towards +axis k
    int slot_of[8];
    int child_in[8];
    for (int s = 0; s < 8; s++) child_in[s] = -1;
    for (int c = 0; c < nc; c++) slot_of[c] = -1;
#if RT_FIXED_SLOTS
    // Leaf children take the lowest slots (their primitives live at prim_base + 3 * slot: a contiguous run of 3 * n_leaves
    // primitive slots per node, see below); the octant order only matters for the children a ray descends into, and those
    // share the remaining slots by the greedy rule. Nodes with only inner children (the upper tree) are unaffected.
    int n_leaf_children = 0;
    for (int c = 0; c < nc; c++)
        if (ch[c] >= first_leaf || b.count[ch[c]] <= LEAF_MAX) {
            slot_of[c] = n_leaf_children;
            child_in[n_leaf_children++] = c;
        }
    const int n_greedy = nc - n_leaf_children;
#else
    const int n_greedy = nc;
#endif
    for (int round = 0; round < n_greedy; round++) {
        float best = -RT_INF;
        int bc = -1, bs = -1;
        for (int c = 0; c < nc; c++) {
            if (slot_of[c] >= 0) continue;
            V3 dv = 0.5f * (clo[c] + chi[c]) - center;
            for (int s = 0; s < 8; s++) {
                if (child_in[s] >= 0) continue;
                float cost = ((s & 1) ? dv.x : -dv.x) + ((s & 2) ? dv.y : -dv.y) + ((s & 4) ? dv.z : -dv.z);
                if (cost > best) { best = cost; bc = c; bs = s; }
            }
        }
        slot_of[bc] = bs;
        child_in[bs] = bc;
    }

    uint32_t ebits[3];
    node_exponents(lo, hi, ebits);

    uint32_t n_internal = 0, n_leaf_prims = 0;
    for (int s = 0; s < 8; s++) {
        int c = child_in[s];
        if (c < 0) continue;
        uint32_t nd = ch[c];
        uint32_t cnt = b.count[nd];
        if (cnt <= LEAF_MAX) n_leaf_prims += cnt; else n_internal++;
    }
    const uint32_t child_base = n_internal ? atomic_add_u32(&b.counters[1], n_internal) : 0u;
#if RT_FIXED_SLOTS
    // 3 primitive slots per leaf child, at prim_base + 3 * slot (leaf children are slots 0 .. n_leaves-1): a hit on child s
    // sets the fixed bits 3s..3s+2 of the ray's primitive mask and the node's `valid` word clears the slots a leaf does not
    // fill — no per-child decoding in the traversal (rt_traverse.h). Unfilled slots stay holes in the primitive array.
    const uint32_t prim_base = n_leaf_children ? atomic_add_u32(&b.counters[2], 3u * (uint32_t)n_leaf_children) : 0u;
    if (n_leaf_prims) atomic_add_u32(&b.counters[3], n_leaf_prims);
#else
    const uint32_t prim_base = n_leaf_prims ? atomic_add_u32(&b.counters[2], n_leaf_prims) : 0u;
    if (n_leaf_prims) atomic_add_u32(&b.counters[3], n_leaf_prims);
#endif
    const uint32_t q_base = n_internal ? atomic_add_u32(&b.counters[0], n_internal) : 0u;

    uint32_t meta[8], q[6][8];
    uint32_t imask = 0, k_internal = 0, k_prim = 0, valid = 0;
    for (int s = 0; s < 8; s++) {
        meta[s] = 0;
        (void)meta[s];
        for (int a = 0; a < 6; a++) q[a][s] = 0;
        int c = child_in[s];
        if (c < 0) continue;
        uint32_t nd = ch[c];
        uint32_t cnt = b.count[nd];
        quantize_child(ebits, lo, clo[c], chi[c], s, q);
        if (cnt <= LEAF_MAX) {
#if RT_FIXED_SLOTS
            k_prim = 3u * (uint32_t)s;
            valid |= ((1u << cnt) - 1u) << k_prim;
#else
            meta[s] = (((1u << cnt) - 1u) << 5) | k_prim;
#endif
            uint32_t walk[4];  // the <= LEAF_MAX leaves of this subtree, left to right
            int wsp = 0;
            walk[wsp++] = nd;
            while (wsp) {
                const uint32_t x = walk[--wsp];
                if (x >= first_leaf) {
                    if (prim_base + k_prim < b.prim_capacity) b.prims[prim_base + k_prim] = b.prims_unsorted[b.vals_sorted[x - first_leaf]];
                    k_prim++;
                }
                else { walk[wsp++] = b.right[x]; walk[wsp++] = b.left[x]; }
            }
        } else {
            meta[s] = (1u << 5) | (24u + (uint32_t)s);
            imask |= 1u << s;
            WorkItem w;
            w.bnode = nd;
            w.wnode = child_base + k_internal;
            b.queue_out[q_base + k_internal] = w;
            k_internal++;
        }
    }

    Node8 nd8;
#if RT_FIXED_SLOTS
    nd8.n1 = make_float4(u2f(child_base), u2f(prim_base), u2f(valid | (imask << 24)), u2f(0u));
#else
    nd8.n1 = make_float4(u2f(child_base), u2f(prim_base), u2f(pack4(meta)), u2f(pack4(meta + 4)));
#endif
    pack_node_planes(nd8, lo, ebits, imask, q);
    b.nodes[it.wnode] = nd8;
}

// ---- refit (rtcuda_scene_update) ------------------------------------------------------------------------------
// Moving instances keeps the tree: every filled primitive slot records its (geom, prim, kind), so it is recomputed in place
// from the updated Instance (refit_prims_body), and the wide nodes are re-fitted bottom-up, one launch per level, deepest
// first (refit_nodes_body). Child slots, child_base / prim_base / valid and the primitive order stay as they are; the node
// frame, exponents and planes are recomputed by the code the collapse uses. Traversal results do not depend on the tree
// (closest t, ties to the larger (geom, prim); conservative boxes, exact primitive tests), so a refitted tree renders the
// frame a fresh build of the same transforms renders.
struct RefitCtx {
    const Instance* instances;
    const float* vertices;
    const uint32_t* tris;
    Prim* prims;
    uint32_t prim_slots;
    uint32_t* bounds_keys;      // 6 x u32 float_key: min xyz, max xyz (initialised by the caller)
    Node8* nodes;
    // 2 per node: (lo.xyz | SAH term of the node's children), (hi.xyz | -): the float box the parent's refit reads
    float4* node_box;
    uint32_t write_nodes;       // 0: only node_box (the cost of the tree as it is, without touching a node)
};

// Recomputes slot i; false for a hole. lo / hi: the primitive's world box (for the bounds reduction).
RT_HD bool refit_prims_body(uint32_t i, const RefitCtx& r, V3& lo, V3& hi) {
    const Prim old = r.prims[i];
    if (f2u(old.c.w) == PRIM_HOLE) return false;
    const uint32_t g = f2u(old.a.w);
    Prim p;
    world_prim(r.instances[g], g, f2u(old.b.w), r.vertices, r.tris, p, lo, hi);
    r.prims[i] = p;
    return true;
}

// World box of a filled slot: the triangle's vertices as stored, or the sphere's transformed object box
RT_HD void prim_world_box(const Prim& p, const Instance* instances, V3& lo, V3& hi) {
    if (f2u(p.c.w) == 0u) {
        const V3 v0 = xyz(p.a), v1 = xyz(p.b), v2 = xyz(p.c);
        lo = vmin(v0, vmin(v1, v2));
        hi = vmax(v0, vmax(v1, v2));
    } else sphere_box(instances[f2u(p.a.w)], lo, hi);
}

// Node i of a level whose children (a deeper level) are refitted already.
RT_HD void refit_nodes_body(uint32_t i, const RefitCtx& r) {
    Node8 nd = r.nodes[i];
    const uint32_t child_base = f2u(nd.n1.x), prim_base = f2u(nd.n1.y), valid = f2u(nd.n1.z);
    const uint32_t imask = valid >> 24;
    V3 clo[8], chi[8];
    V3 lo = mk3(RT_INF, RT_INF, RT_INF), hi = mk3(-RT_INF, -RT_INF, -RT_INF);
    float sah = 0.0f;
    uint32_t k_internal = 0, present = 0;
#pragma unroll
    for (int s = 0; s < 8; s++) {
        if (imask & (1u << s)) {
            const uint32_t c = child_base + k_internal++;
            clo[s] = xyz(r.node_box[2 * (size_t)c]);
            chi[s] = xyz(r.node_box[2 * (size_t)c + 1]);
            sah += half_area(clo[s], chi[s]);
        } else {
            const uint32_t bits = (valid >> (3 * s)) & 7u;
            if (!bits) continue;
            clo[s] = mk3(RT_INF, RT_INF, RT_INF);
            chi[s] = mk3(-RT_INF, -RT_INF, -RT_INF);
            uint32_t cnt = 0;
#pragma unroll
            for (uint32_t k = 0; k < LEAF_MAX; k++) {
                if (!(bits & (1u << k))) continue;
                V3 plo, phi;
                prim_world_box(r.prims[prim_base + 3u * (uint32_t)s + k], r.instances, plo, phi);
                clo[s] = vmin(clo[s], plo);
                chi[s] = vmax(chi[s], phi);
                cnt++;
            }
            sah += half_area(clo[s], chi[s]) * (float)cnt;
        }
        present |= 1u << s;
        lo = vmin(lo, clo[s]);
        hi = vmax(hi, chi[s]);
    }
    r.node_box[2 * (size_t)i] = make_float4(lo.x, lo.y, lo.z, sah);
    r.node_box[2 * (size_t)i + 1] = make_float4(hi.x, hi.y, hi.z, 0.0f);
    if (!r.write_nodes) return;
    uint32_t ebits[3], q[6][8];
    node_exponents(lo, hi, ebits);
#pragma unroll
    for (int s = 0; s < 8; s++) {
        for (int a = 0; a < 6; a++) q[a][s] = 0;
        if (present & (1u << s)) quantize_child(ebits, lo, clo[s], chi[s], s, q);
    }
    pack_node_planes(nd, lo, ebits, imask, q);
    r.nodes[i] = nd;
}

// SAH cost of the wide tree from the node boxes (C_node = C_prim = 1, A = half the surface area, a factor that cancels):
// (A(root) + sum over inner children of A + sum over leaf children of A * primitives) / A(root).
// `partial`: per-node terms summed in a fixed order (kernels.cu k_sah_partial), so every GPU gets the same figure.
RT_HD double sah_cost(const float4* root_box, double children) {
    const double a = half_area(xyz(root_box[0]), xyz(root_box[1]));
    return a > 0.0 ? (a + children) / a : 0.0;
}

// Refit or rebuild: a refit whose SAH cost grew by more than this factor over the cost of the tree as last built is replaced
// by a fresh build from the resident geometry. B200 (profiles/r9_scene_update.json, DESIGN.md "Scene updates"): rigid motions of
// one instance by up to 50 % of the scene extent kept the refit within 0.5 % of the built cost on C3 and C5, while fresh builds
// of the same moved scenes differed from each other by up to 4 %; a rebuild costs 1.4 ms (C3) / 91 ms (C5) of device time against
// 7 ms for a C5 refit, and trace time follows the cost. 1.25 stays clear of build-to-build variation and rebuilds long before the
// extra trace time of one frame exceeds the price of the rebuild.
constexpr double REFIT_MAX_GROWTH = 1.25;
RT_HD bool refit_needs_rebuild(double sah_refit, double sah_built, double max_growth = REFIT_MAX_GROWTH) {
    return sah_refit > max_growth * sah_built;
}

}  // namespace rt
