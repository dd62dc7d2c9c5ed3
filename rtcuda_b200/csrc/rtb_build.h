// rtb_build.h — bodies of the GPU BVH builder kernels.
//
// Replaces Bvh::Bvh (bvh.cuh:30-219: single-threaded host full-sweep SAH over
// three std::sort'ed index arrays, ~260 ms for 69k triangles, minutes for
// 10M).  Pipeline, all on the device:
//   1. prim_setup     per-triangle record {p0,e1,e2,n}, bounds, scene bounds
//   2. morton         63-bit Morton code of the centroid, radix sort
//   3. PLOC           parallel locally-ordered clustering (Meister & Bittner
//                     2018): nearest neighbour within a window of the Morton
//                     order, merge mutual pairs, compact; repeat to one root
//   3'. binned SAH    (RTB_BUILDER_BINNED_SAH, instead of 2-3) top-down
//                     32-bin SAH splits down to single primitives: large
//                     ranges level by level, small ones one block each
//   3.5 treelets      (optional, RTB_BUILDER_TREELET_PASSES) passes of treelet
//                     restructuring (Karras & Aila 2013) over either tree:
//                     up to 7 subtrees under a node rewired into their
//                     cheapest binary topology, one launch per depth
//   4. collapse plan  (optional, RTB_COLLAPSE_SAH_OPTIMAL; default is the greedy
//                     "largest child first" of step 5)
//                     bottom-up dynamic programme over the binary tree (after
//                     Ylitie, Karras & Laine 2017): for every subtree, the
//                     cheapest way (SAH) to lay it out in 1..7 child slots of
//                     a wide node — one leaf child (<= 3 triangles), one inner
//                     child (its own wide node), or split between its two
//                     children; run round by round in PLOC merge order, which
//                     is a topological order
//   5. collapse       top-down, level-synchronous: expand each wide node's
//                     children as the plan says, slot assignment for
//                     octant-ordered traversal, 8-bit quantisation, triangles
//                     rewritten in leaf order
// Bodies are RTB_HD; see rtb_wavefront.h for why.
#pragma once
#include "rtb_shade.h"

namespace rtb {

struct B2Node {  // binary node, 32 bytes
    float lox, loy, loz; int32_t left;   // leaf: left = caller's triangle index
    float hix, hiy, hiz; int32_t right;  // leaf: right = -1
};

#if defined(__CUDA_ARCH__)
RTB_HD int atomic_add_i(int32_t *p, int v) { return atomicAdd(p, v); }
RTB_HD void atomic_min_i(int32_t *p, int v) { atomicMin(p, v); }
RTB_HD void atomic_max_i(int32_t *p, int v) { atomicMax(p, v); }
RTB_HD void atomic_add_f(float *p, float v) { atomicAdd(p, v); }
#else
RTB_HD int atomic_add_i(int32_t *p, int v) { int o = *p; *p += v; return o; }
RTB_HD void atomic_min_i(int32_t *p, int v) { if (v < *p) *p = v; }
RTB_HD void atomic_max_i(int32_t *p, int v) { if (v > *p) *p = v; }
RTB_HD void atomic_add_f(float *p, float v) { *p += v; }
#endif

// order-preserving float <-> int map for atomic min/max on floats
RTB_HD int32_t float_to_ordered(float f) { int32_t b = f2i(f); return b >= 0 ? b : b ^ 0x7fffffff; }
RTB_HD float ordered_to_float(int32_t b) { return i2f(b >= 0 ? b : b ^ 0x7fffffff); }

RTB_HD float half_area(float ex, float ey, float ez) { return ffma(fadd(ex, ey), ez, fmul(ex, ey)); }
RTB_HD float b2_half_area(const B2Node &n) {
    return half_area(fsub(n.hix, n.lox), fsub(n.hiy, n.loy), fsub(n.hiz, n.loz));
}
RTB_HD float union_half_area(const B2Node &a, const B2Node &b) {
    return half_area(fsub(fmaxf(a.hix, b.hix), fminf(a.lox, b.lox)), fsub(fmaxf(a.hiy, b.hiy), fminf(a.loy, b.loy)),
                     fsub(fmaxf(a.hiz, b.hiz), fminf(a.loz, b.loz)));
}

// ------------------------------------------------------------ 1. prim setup
struct PrimSetupArgs {
    const float *vertices;        // 9 per triangle, or null when tri_in is pre-filled
    Tri48 *tri_in;                // [n] caller order
    F4 *prim_lo, *prim_hi;        // [n] bounds (w unused)
    int32_t *scene_bounds;        // 6 ordered ints: min xyz, max xyz
    int32_t *bad;                 // raised when a vertex is not finite or beyond kMaxCoord
    int32_t n;
};
// Coordinates the builder accepts: finite and |x| <= 2^100.  (An infinite vertex gives a cluster whose merged area is
// never below any other, so PLOC could not pair it; beyond 2^100 box extents and areas overflow.  The reference has no
// such check: its host SAH sweep just produces a useless tree.)
constexpr float kMaxCoord = 1.2676506e30f;
// bounds of one triangle record, the vertex check and the scene bounds; t is triangle i's record (already stored)
RTB_HD void prim_setup_bounds(const PrimSetupArgs &a, int i, const Tri48 &t);
RTB_HD void prim_setup_box(const PrimSetupArgs &a, int i, const Tri48 &t, V3 &lo, V3 &hi);
RTB_HD bool tri_box(const Tri48 &t, V3 &lo, V3 &hi);
RTB_HD void prim_setup_body(const PrimSetupArgs &a, int i) {
    if (i >= a.n) return;
    Tri48 t;
    if (a.vertices) {
        const float *v = a.vertices + 9 * (size_t)i;
        t = tri_from_vertices(v3(v[0], v[1], v[2]), v3(v[3], v[4], v[5]), v3(v[6], v[7], v[8]));
        a.tri_in[i] = t;
    } else {
        t = a.tri_in[i];
    }
    prim_setup_bounds(a, i, t);
}
RTB_HD void prim_setup_bounds(const PrimSetupArgs &a, int i, const Tri48 &t) {
    V3 lo, hi;
    prim_setup_box(a, i, t, lo, hi);
#if defined(__CUDA_ARCH__)
    // one reduction per warp (redux.sync), then six atomics by one lane: 10 M triangles used to send 60 M atomics to six addresses
    const unsigned m = __activemask();
    const int lx = __reduce_min_sync(m, float_to_ordered(lo.x)), ly = __reduce_min_sync(m, float_to_ordered(lo.y)),
              lz = __reduce_min_sync(m, float_to_ordered(lo.z));
    const int hx = __reduce_max_sync(m, float_to_ordered(hi.x)), hy = __reduce_max_sync(m, float_to_ordered(hi.y)),
              hz = __reduce_max_sync(m, float_to_ordered(hi.z));
    if ((threadIdx.x & 31) == __ffs(m) - 1) {
        atomic_min_i(a.scene_bounds + 0, lx); atomic_min_i(a.scene_bounds + 1, ly); atomic_min_i(a.scene_bounds + 2, lz);
        atomic_max_i(a.scene_bounds + 3, hx); atomic_max_i(a.scene_bounds + 4, hy); atomic_max_i(a.scene_bounds + 5, hz);
    }
#else
    atomic_min_i(a.scene_bounds + 0, float_to_ordered(lo.x));
    atomic_min_i(a.scene_bounds + 1, float_to_ordered(lo.y));
    atomic_min_i(a.scene_bounds + 2, float_to_ordered(lo.z));
    atomic_max_i(a.scene_bounds + 3, float_to_ordered(hi.x));
    atomic_max_i(a.scene_bounds + 4, float_to_ordered(hi.y));
    atomic_max_i(a.scene_bounds + 5, float_to_ordered(hi.z));
#endif
}
RTB_HD void prim_setup_box(const PrimSetupArgs &a, int i, const Tri48 &t, V3 &lo, V3 &hi) {
    if (tri_box(t, lo, hi)) *a.bad = 1;
    F4 l; l.x = lo.x; l.y = lo.y; l.z = lo.z; l.w = 0.f;
    F4 h; h.x = hi.x; h.y = hi.y; h.z = hi.z; h.w = 0.f;
    a.prim_lo[i] = l; a.prim_hi[i] = h;
}
// box of one triangle record (the builder's and the refit's); true when a vertex is not finite or beyond kMaxCoord
RTB_HD bool tri_box(const Tri48 &t, V3 &lo, V3 &hi) {
    // Triangle::bounding_box, triangle.cuh:23-37 (p1 = p0 - e1, p2 = p0 + e2)
    V3 p0 = tri_p0(t), p1 = vsub(p0, tri_e1(t)), p2 = vadd(p0, tri_e2(t));
    lo = v3(fminf(p0.x, fminf(p1.x, p2.x)), fminf(p0.y, fminf(p1.y, p2.y)), fminf(p0.z, fminf(p1.z, p2.z)));
    hi = v3(fmaxf(p0.x, fmaxf(p1.x, p2.x)), fmaxf(p0.y, fmaxf(p1.y, p2.y)), fmaxf(p0.z, fmaxf(p1.z, p2.z)));
    // (fminf / fmaxf drop a NaN operand, so the vertices are looked at themselves)
    const float worst = fmaxf(fmaxf(fmaxf(fabsf(p0.x), fabsf(p0.y)), fmaxf(fabsf(p0.z), fabsf(p1.x))),
                              fmaxf(fmaxf(fabsf(p1.y), fabsf(p1.z)), fmaxf(fabsf(p2.x), fmaxf(fabsf(p2.y), fabsf(p2.z)))));
    const bool nan = p0.x != p0.x || p0.y != p0.y || p0.z != p0.z || p1.x != p1.x || p1.y != p1.y || p1.z != p1.z || p2.x != p2.x ||
                     p2.y != p2.y || p2.z != p2.z;
    return nan || !(worst <= kMaxCoord);
}

// ------------------------------------------------------------ 2. morton
RTB_HD uint64_t spread21(uint64_t x) {  // 21 bits -> every third bit
    x &= 0x1fffffull;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}
struct MortonArgs {
    const F4 *prim_lo, *prim_hi;
    const int32_t *scene_bounds;
    uint64_t *keys; int32_t *vals;
    int32_t n;
};
RTB_HD void morton_body(const MortonArgs &a, int i) {
    if (i >= a.n) return;
    float sx = ordered_to_float(a.scene_bounds[0]), sy = ordered_to_float(a.scene_bounds[1]), sz = ordered_to_float(a.scene_bounds[2]);
    float ex = fsub(ordered_to_float(a.scene_bounds[3]), sx), ey = fsub(ordered_to_float(a.scene_bounds[4]), sy),
          ez = fsub(ordered_to_float(a.scene_bounds[5]), sz);
    float e = fmaxf(ex, fmaxf(ey, ez));
    float inv = e > 0.f ? fdiv(2097151.f, e) : 0.f;  // same scale on all axes keeps cells cubic
    const F4 lo = a.prim_lo[i], hi = a.prim_hi[i];
    float cx = fmul(0.5f, fadd(lo.x, hi.x)), cy = fmul(0.5f, fadd(lo.y, hi.y)), cz = fmul(0.5f, fadd(lo.z, hi.z));
    float qx = fminf(fmaxf(fmul(fsub(cx, sx), inv), 0.f), 2097151.f);
    float qy = fminf(fmaxf(fmul(fsub(cy, sy), inv), 0.f), 2097151.f);
    float qz = fminf(fmaxf(fmul(fsub(cz, sz), inv), 0.f), 2097151.f);
    a.keys[i] = spread21((uint64_t)qx) | (spread21((uint64_t)qy) << 1) | (spread21((uint64_t)qz) << 2);
    a.vals[i] = i;
}

// ------------------------------------------------------------ 3. PLOC
struct PlocArgs {
    B2Node *nodes;        // [2n-1]; leaves 0..n-1 in Morton order
    int32_t *count;       // [2n-1] triangles below each node
    const int32_t *cin;   // clusters (node indices), Morton order kept
    int32_t *cout;        // after merge: node index or -1
    int32_t *nn;          // nearest neighbour position
    int32_t *node_counter;  // next free inner node, starts at n
    int32_t ncl;          // current cluster count — or, with ncl_dev set, an upper bound of it known to the host
    int32_t radius;
    // device-driven rounds (round 2): the count lives in device memory, the host enqueues several rounds without
    // reading it back (every PLOC round used to cost a device->host copy of the count and a stream synchronisation)
    const int32_t *ncl_dev;  // null: ncl is the count
    int32_t *log;            // [round] = cluster count at the start of that round (null: not kept)
    int32_t round;
};
RTB_HD int ploc_ncl(const PlocArgs &a) { return a.ncl_dev ? *a.ncl_dev : a.ncl; }
RTB_HD void ploc_leaf_body(const F4 *prim_lo, const F4 *prim_hi, const int32_t *sorted, B2Node *nodes,
                           int32_t *count, int32_t *clusters, int n, int i) {
    if (i >= n) return;
    const int p = sorted[i];
    const F4 lo = prim_lo[p], hi = prim_hi[p];
    B2Node b;
    b.lox = lo.x; b.loy = lo.y; b.loz = lo.z; b.left = p;
    b.hix = hi.x; b.hiy = hi.y; b.hiz = hi.z; b.right = -1;
    nodes[i] = b;
    count[i] = 1;
    clusters[i] = i;
}
// nearest neighbour by merged surface area within +-radius positions; ties go
// to the lowest position, which guarantees at least one mutual pair per round
RTB_HD void ploc_nn_body(const PlocArgs &a, int i) {
    const int ncl = ploc_ncl(a);
    if (i == 0 && a.log) a.log[a.round] = ncl;
    if (i >= ncl) return;
    const B2Node me = a.nodes[a.cin[i]];
    float best = FLT_MAX;
    int bj = -1;
    const int j0 = i - a.radius < 0 ? 0 : i - a.radius;
    const int j1 = i + a.radius > ncl - 1 ? ncl - 1 : i + a.radius;
    for (int j = j0; j <= j1; ++j) {
        if (j == i) continue;
        const float ar = union_half_area(me, a.nodes[a.cin[j]]);
        if (bj < 0 || ar < best) { best = ar; bj = j; }  // total: every cluster names a neighbour, whatever its area
    }
    a.nn[i] = bj;
}
RTB_HD void ploc_merge_body(const PlocArgs &a, int n_leaves, int i) {
    if (i >= ploc_ncl(a)) {
        if (i < a.ncl) a.cout[i] = -1;  // between the count and the host's bound: dropped by the compaction over the bound
        return;
    }
    const int j = a.nn[i];
    const int ci = a.cin[i];
    if (j >= 0 && a.nn[j] == i) {
        if (i < j) {
            const int cj = a.cin[j];
            const int id = atomic_add_i(a.node_counter, 1);
            const B2Node x = a.nodes[ci], y = a.nodes[cj];
            B2Node m;
            m.lox = fminf(x.lox, y.lox); m.loy = fminf(x.loy, y.loy); m.loz = fminf(x.loz, y.loz);
            m.hix = fmaxf(x.hix, y.hix); m.hiy = fmaxf(x.hiy, y.hiy); m.hiz = fmaxf(x.hiz, y.hiz);
            m.left = ci; m.right = cj;
            a.nodes[id] = m;
            a.count[id] = a.count[ci] + a.count[cj];
            a.cout[i] = id;
        } else {
            a.cout[i] = -1;
        }
    } else {
        a.cout[i] = ci;
    }
    (void)n_leaves;
}

// ------------------------------------------------------------ 3'. binned SAH (RTB_BUILDER_BINNED_SAH)
// Top-down, instead of steps 2-3: a node's primitives are a contiguous range [begin, end) of a primitive index array; its
// split is the cheapest of 31 planes per axis (cost A_L N_L + A_R N_R) between 32 bins over its centroid extent, and
// depends on nothing but its primitive set and centroid bounds (counts and boxes are accumulated as integers / ordered
// ints, so the order of accumulation is free).  A stable partition of the range then gives the two children.  Ranges go
// down to single primitives: a range of one primitive at position p is leaf node p (left = idx[p]); inner nodes take ids
// n .. 2n-2.  Large ranges are split level by level by the whole device, small ones (<= kSahSmall) by one block each.
constexpr int kSahBins = 32;
constexpr int kSahBinWords = 7;                              // count, box lo xyz, box hi xyz (ordered ints)
constexpr int kSahBinsWords = 3 * kSahBins * kSahBinWords;   // a node's bins, [axis][bin][word]
constexpr int kSahSmall = 1024;                              // ranges up to this size are finished in one block
constexpr int kSahChunk = 4096;                              // primitives per block of a level's kernels
// Binary depth beyond which the 8-wide tree cannot fit the traversal stack: the collapse turns at most 7 binary levels
// into one 8-wide level, and kStackSize 8-wide levels are already too deep.
constexpr int kSahMaxDepth = 7 * kStackSize;
struct SahRange { int32_t begin, end, id, depth; };
struct SahTask {          // a large range of one level
    SahRange r;
    int32_t bnd[12];      // ordered ints: box lo xyz, box hi xyz, centroid lo xyz, centroid hi xyz
    int32_t blk0;         // its first block in the level's block -> task map
    int32_t axis, plane, nl;  // the split: axis -1 = by position; nl = primitives going left
};
struct SahArgs {
    const F4 *prim_lo, *prim_hi;
    int32_t *idx, *idx2;          // [n] primitive at each position; scatter target
    int32_t *flags, *scan;        // [n] "goes left" and its exclusive scan (large ranges)
    B2Node *nodes; int32_t *count;
    int32_t *depth;               // [n-1] depth of inner node id, at [id - n]
    int32_t *node_counter;
    const SahTask *tin_c; SahTask *tin, *tout;  // this level's tasks (tin_c == tin), the next level's
    const int32_t *blk_in; int32_t *blk_out;    // block -> task
    const int32_t *n_tin, *n_blk_in;            // counts of this level (device memory)
    int32_t *n_tout, *n_blk_out;                // next level's counts
    int32_t *n_clear, *n_blk_clear;             // the counts of the level after the next, cleared by this level
    int32_t *bins;                // [task][kSahBinsWords], neutral between uses
    SahRange *small; int32_t *n_small;
    int32_t n;
};
RTB_HD V3 sah_centroid(const F4 &lo, const F4 &hi) {  // as morton_body
    return v3(fmul(0.5f, fadd(lo.x, hi.x)), fmul(0.5f, fadd(lo.y, hi.y)), fmul(0.5f, fadd(lo.z, hi.z)));
}
RTB_HD float v3_at(const V3 &v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : v.z); }
// bins per unit of centroid extent on axis k, 0 when the axis is unusable (no extent, or a scale that is not finite)
RTB_HD float sah_scale(const int32_t *bnd, int k) {
    const float e = fsub(ordered_to_float(bnd[9 + k]), ordered_to_float(bnd[6 + k]));
    const float s = e > 0.f ? fdiv((float)kSahBins, e) : 0.f;
    return s <= FLT_MAX ? s : 0.f;
}
RTB_HD int sah_bin(float c, float cmin, float scale) {
    const int b = (int)fmul(fsub(c, cmin), scale);
    return b < 0 ? 0 : (b >= kSahBins ? kSahBins - 1 : b);
}
RTB_HD void sah_bnd_init(int32_t *b) {
    for (int k = 0; k < 3; ++k) { b[k] = b[6 + k] = float_to_ordered(FLT_MAX); b[3 + k] = b[9 + k] = float_to_ordered(-FLT_MAX); }
}
RTB_HD void sah_bin_init(int32_t *w) {
    w[0] = 0;
    for (int k = 0; k < 3; ++k) { w[1 + k] = float_to_ordered(FLT_MAX); w[4 + k] = float_to_ordered(-FLT_MAX); }
}
// one primitive into the bins of the usable axes (atomics: shared memory on the device)
RTB_HD void sah_bin_add(int32_t *bins, const F4 &lo, const F4 &hi, const int32_t *bnd, const float *scale) {
    const V3 c = sah_centroid(lo, hi);
    const int32_t l[3] = {float_to_ordered(lo.x), float_to_ordered(lo.y), float_to_ordered(lo.z)};
    const int32_t h[3] = {float_to_ordered(hi.x), float_to_ordered(hi.y), float_to_ordered(hi.z)};
    for (int a = 0; a < 3; ++a) {
        if (scale[a] <= 0.f) continue;
        int32_t *w = bins + (a * kSahBins + sah_bin(v3_at(c, a), ordered_to_float(bnd[6 + a]), scale[a])) * kSahBinWords;
        atomic_add_i(w, 1);
        for (int k = 0; k < 3; ++k) { atomic_min_i(w + 1 + k, l[k]); atomic_max_i(w + 4 + k, h[k]); }
    }
}
RTB_HD void sah_bin_merge(int32_t *acc, const int32_t *w) {
    acc[0] += w[0];
    for (int k = 0; k < 3; ++k) { acc[1 + k] = acc[1 + k] < w[1 + k] ? acc[1 + k] : w[1 + k]; acc[4 + k] = acc[4 + k] > w[4 + k] ? acc[4 + k] : w[4 + k]; }
}
RTB_HD float sah_inf() { return i2f(0x7f800000); }
// cost of a plane with the bins l (left of it) and r (right of it) merged; +inf when a side is empty or the cost overflows
RTB_HD float sah_plane_cost(const int32_t *l, const int32_t *r) {
    if (l[0] <= 0 || r[0] <= 0) return sah_inf();
    const float al = half_area(fsub(ordered_to_float(l[4]), ordered_to_float(l[1])), fsub(ordered_to_float(l[5]), ordered_to_float(l[2])),
                               fsub(ordered_to_float(l[6]), ordered_to_float(l[3])));
    const float ar = half_area(fsub(ordered_to_float(r[4]), ordered_to_float(r[1])), fsub(ordered_to_float(r[5]), ordered_to_float(r[2])),
                               fsub(ordered_to_float(r[6]), ordered_to_float(r[3])));
    const float c = ffma(al, (float)l[0], fmul(ar, (float)r[0]));
    return c <= FLT_MAX ? c : sah_inf();
}
struct SahSplit { int32_t axis, plane, nl; };
// the split of a range of `size` primitives from its bins: lowest cost, ties to the lowest axis, then the lowest plane;
// without a usable plane, the range is halved by position
RTB_HD SahSplit sah_choose(const int32_t *bins, const float *scale, int size) {
    SahSplit s; s.axis = -1; s.plane = 0; s.nl = size / 2;
    float best = sah_inf();
    for (int a = 0; a < 3; ++a) {
        if (scale[a] <= 0.f) continue;
        const int32_t *b = bins + a * kSahBins * kSahBinWords;
        int32_t right[kSahBins][kSahBinWords];  // right[k]: bins k .. 31
        sah_bin_init(right[kSahBins - 1]);
        sah_bin_merge(right[kSahBins - 1], b + (kSahBins - 1) * kSahBinWords);
        for (int k = kSahBins - 2; k >= 0; --k) {
            for (int w = 0; w < kSahBinWords; ++w) right[k][w] = right[k + 1][w];
            sah_bin_merge(right[k], b + k * kSahBinWords);
        }
        int32_t left[kSahBinWords];
        sah_bin_init(left);
        for (int k = 0; k + 1 < kSahBins; ++k) {
            sah_bin_merge(left, b + k * kSahBinWords);
            const float c = sah_plane_cost(left, right[k + 1]);
            if (c < best) { best = c; s.axis = a; s.plane = k; s.nl = left[0]; }
        }
    }
    return s;
}
// does the primitive at offset `off` of its range (box lo / hi) go to the left child?
RTB_HD bool sah_goes_left(const SahSplit &s, int off, const F4 &lo, const F4 &hi, const int32_t *bnd) {
    if (s.axis < 0) return off < s.nl;
    const float c = v3_at(sah_centroid(lo, hi), s.axis);
    return sah_bin(c, ordered_to_float(bnd[6 + s.axis]), sah_scale(bnd, s.axis)) <= s.plane;
}
// box and centroid bounds of one primitive into b (plain min / max: the caller reduces)
RTB_HD void sah_bnd_add(int32_t *b, const F4 &lo, const F4 &hi) {
    const V3 c = sah_centroid(lo, hi);
    const int32_t v[12] = {float_to_ordered(lo.x), float_to_ordered(lo.y), float_to_ordered(lo.z), float_to_ordered(hi.x),
                           float_to_ordered(hi.y), float_to_ordered(hi.z), float_to_ordered(c.x), float_to_ordered(c.y),
                           float_to_ordered(c.z), float_to_ordered(c.x), float_to_ordered(c.y), float_to_ordered(c.z)};
    for (int k = 0; k < 3; ++k) {
        b[k] = b[k] < v[k] ? b[k] : v[k]; b[6 + k] = b[6 + k] < v[6 + k] ? b[6 + k] : v[6 + k];
        b[3 + k] = b[3 + k] > v[3 + k] ? b[3 + k] : v[3 + k]; b[9 + k] = b[9 + k] > v[9 + k] ? b[9 + k] : v[9 + k];
    }
}
// inner node r (box from bnd, split after nl primitives): writes the node, its count and depth, and its two children into
// ch; a child of one primitive is the leaf at its position, a larger one takes an id from *ids
RTB_HD void sah_make_node(const SahArgs &a, const SahRange &r, const int32_t *bnd, int nl, int32_t *ids, SahRange *ch) {
    ch[0].begin = r.begin; ch[0].end = r.begin + nl;
    ch[1].begin = r.begin + nl; ch[1].end = r.end;
    for (int k = 0; k < 2; ++k) {
        ch[k].depth = r.depth + 1;
        ch[k].id = ch[k].end - ch[k].begin == 1 ? ch[k].begin : atomic_add_i(ids, 1);
    }
    B2Node m;
    m.lox = ordered_to_float(bnd[0]); m.loy = ordered_to_float(bnd[1]); m.loz = ordered_to_float(bnd[2]); m.left = ch[0].id;
    m.hix = ordered_to_float(bnd[3]); m.hiy = ordered_to_float(bnd[4]); m.hiz = ordered_to_float(bnd[5]); m.right = ch[1].id;
    a.nodes[r.id] = m;
    a.count[r.id] = r.end - r.begin;
    a.depth[r.id - a.n] = r.depth;
}
// a child made by a level: to the next level (with its blocks), to the small ranges, or nothing (a leaf)
RTB_HD void sah_push_child(const SahArgs &a, const SahRange &c) {
    const int size = c.end - c.begin;
    if (size <= 1) return;
    if (size <= kSahSmall) { a.small[atomic_add_i(a.n_small, 1)] = c; return; }
    const int t = atomic_add_i(a.n_tout, 1), nb = (size + kSahChunk - 1) / kSahChunk;
    SahTask T;
    T.r = c; sah_bnd_init(T.bnd);
    T.blk0 = atomic_add_i(a.n_blk_out, nb);
    T.axis = -1; T.plane = 0; T.nl = 0;
    a.tout[t] = T;
    for (int k = 0; k < nb; ++k) a.blk_out[T.blk0 + k] = t;
}
// first block of the build: root range, counters
struct SahRootK {
    SahArgs a; int32_t *root;
    RTB_HD void operator()(int i) const {
        if (i != 0) return;
        *a.n_small = 0;
        if (a.n == 1) { *root = 0; return; }
        *root = a.n;
        *a.node_counter = a.n + 1;
        SahRange r; r.begin = 0; r.end = a.n; r.id = a.n; r.depth = 0;
        sah_push_child(a, r);  // (the "next level" of the root's push is level 0)
    }
};
struct SahIotaK { int32_t *p; int n; RTB_HD void operator()(int i) const { if (i < n) p[i] = i; } };
struct SahBinsInitK { int32_t *bins; int n; RTB_HD void operator()(int i) const { if (i < n) sah_bin_init(bins + (size_t)i * kSahBinWords); } };
// leaf node p = the primitive that ended at position p
struct SahLeafK {
    SahArgs a;
    RTB_HD void operator()(int p) const {
        if (p >= a.n) return;
        const int g = a.idx[p];
        const F4 lo = a.prim_lo[g], hi = a.prim_hi[g];
        B2Node b;
        b.lox = lo.x; b.loy = lo.y; b.loz = lo.z; b.left = g;
        b.hix = hi.x; b.hiy = hi.y; b.hiz = hi.z; b.right = -1;
        a.nodes[p] = b;
        a.count[p] = 1;
    }
};
// collapse plan order: inner nodes deepest first (sort key), and where each depth starts in that order
struct SahDepthKeyK {
    const int32_t *depth; uint64_t *keys; int32_t *vals; int n_inner, n;
    RTB_HD void operator()(int i) const {
        if (i >= n_inner) return;
        const int d = depth[i] < kSahMaxDepth + 1 ? depth[i] : kSahMaxDepth + 1;
        keys[i] = (uint64_t)(kSahMaxDepth + 1 - d);
        vals[i] = n + i;
    }
};
struct SahGroupK {
    const uint64_t *keys; int32_t *first; int n_inner;
    RTB_HD void operator()(int i) const {
        if (i >= n_inner) return;
        if (i == 0 || keys[i - 1] != keys[i]) first[keys[i]] = i;
    }
};

// ------------------------------------------------------------ 3.5 treelet restructuring (RTB_BUILDER_TREELET_PASSES)
// After either builder, on the binary tree in place (Karras & Aila 2013).  A pass visits the inner nodes deepest first,
// one launch per depth; a node whose subtree holds at least gamma triangles is the root of a treelet: starting from its
// two children, the treelet leaf with the largest area that is an inner node is opened (ties: the lower id) until 7
// leaves or only leaves remain.  A dynamic programme over the subsets of those leaves finds the binary topology over
// them with the lowest sum of inner node areas; when that sum is strictly lower than the present one, the treelet is
// rewired with its own inner ids.  The leaves (their subtrees) stay as they are, the root keeps its id, and nodes of one
// depth have disjoint subtrees, so a launch is free of races and its result does not depend on the schedule.  Costs
// use the explicitly rounded arithmetic of plan_body: the GPU and the host emulation pick the same topologies.
constexpr int kTloLeaves = 7;
constexpr int kTloSubsets = 1 << kTloLeaves;
constexpr int kTloMaxPasses = 8;  // RTB_BUILDER_TREELET_PASSES(k): k = 0..8
// Pass p (from 0) restructures the treelets of nodes with at least kTloGamma << p triangles: later passes leave the
// bottom of the tree, which the first pass already optimised, and cost a fraction of it.  (S1, 3 passes, both builders
// and both collapses: 7 doubling comes within 0.04 % of the SAH cost of restructuring every treelet in every pass,
// gamma 3; 14 doubling loses up to 0.1 % — DESIGN.md 4.1.)
constexpr int kTloGamma = 7;
struct TloArgs {
    B2Node *nodes; int32_t *count;
    int32_t *parent;          // [2n-1]: parent of every node, -1 at the root; kept up to date by the rewiring
    int32_t *depth;           // [n-1]: depth of inner node id at [id - n], at most kSahMaxDepth + 1
    const int32_t *root;      // the root's id (device memory)
    const int32_t *order;     // inner nodes deepest first; this launch: roots order[first .. first + num)
    int32_t first, num;
    int32_t gamma, n;
};
// parents from the inner nodes (ids n .. 2n-2, whichever builder made them)
struct TloParentK {
    TloArgs a;
    RTB_HD void operator()(int i) const {
        if (i >= a.n - 1) return;
        const B2Node x = a.nodes[a.n + i];
        a.parent[x.left] = a.n + i; a.parent[x.right] = a.n + i;
        if (i == 0) a.parent[*a.root] = -1;
    }
};
// depth of every inner node by walking up to the root; a walk longer than kSahMaxDepth stops there (too deep anyway)
struct TloDepthK {
    TloArgs a;
    RTB_HD void operator()(int i) const {
        if (i >= a.n - 1) return;
        int d = 0;
        for (int p = a.parent[a.n + i]; p >= 0 && d <= kSahMaxDepth; p = a.parent[p]) ++d;
        a.depth[i] = d;
    }
};
// one treelet under work (shared memory on the GPU, one per warp): subsets are bit masks over the leaf slots
struct TloWork {
    float area[kTloSubsets];      // half area of the union of a subset's leaves
    float cost[kTloSubsets];      // cheapest sum of inner areas over a subset (0 for one leaf)
    uint8_t part[kTloSubsets];    // that topology's left child: the lowest mask of the cheapest partition
    B2Node box[kTloLeaves];       // the leaves' nodes
    int32_t leaf[kTloLeaves];     // their ids
    int32_t lcount[kTloLeaves];   // and triangle counts
    int32_t inner[kTloLeaves - 1];  // the treelet's inner ids: [0] the root, then in opening order
    int32_t imask[kTloLeaves - 1]; float icost[kTloLeaves - 1];  // the present topology: leaves and cost of inner[j]
    int32_t qmask[kTloLeaves - 1], qid[kTloLeaves - 1];          // the rewiring's queue
    int32_t nl, ni;
};
RTB_HD void tlo_form(const TloArgs &a, TloWork &W, int root) {
    const B2Node r = a.nodes[root];
    W.inner[0] = root; W.ni = 1;
    W.leaf[0] = r.left; W.box[0] = a.nodes[r.left];
    W.leaf[1] = r.right; W.box[1] = a.nodes[r.right];
    W.nl = 2;
    const int32_t c0 = a.count[r.left], c1 = a.count[r.right];
    W.lcount[0] = c0; W.lcount[1] = c1;
    while (W.nl < kTloLeaves) {
        int best = -1; float ba = 0.f;
        for (int k = 0; k < W.nl; ++k) {
            if (W.box[k].right < 0) continue;
            const float ar = b2_half_area(W.box[k]);
            if (best < 0 || ar > ba || (ar == ba && W.leaf[k] < W.leaf[best])) { best = k; ba = ar; }
        }
        if (best < 0) break;
        const B2Node x = W.box[best];
        W.inner[W.ni++] = W.leaf[best];
        W.leaf[best] = x.left; W.box[best] = a.nodes[x.left]; W.lcount[best] = a.count[x.left];
        W.leaf[W.nl] = x.right; W.box[W.nl] = a.nodes[x.right]; W.lcount[W.nl] = a.count[x.right];
        ++W.nl;
    }
}
// box (exact: min / max) and triangle count of the union of subset m
RTB_HD B2Node tlo_union(const TloWork &W, int m, int &cnt) {
    B2Node u; cnt = 0;
    bool first = true;
    for (int k = 0; k < W.nl; ++k) {
        if (!(m >> k & 1)) continue;
        const B2Node &b = W.box[k];
        cnt += W.lcount[k];
        if (first) { u = b; first = false; continue; }
        u.lox = fminf(u.lox, b.lox); u.loy = fminf(u.loy, b.loy); u.loz = fminf(u.loz, b.loz);
        u.hix = fmaxf(u.hix, b.hix); u.hiy = fmaxf(u.hiy, b.hiy); u.hiz = fmaxf(u.hiz, b.hiz);
    }
    return u;
}
// cost of subset m from those of its proper subsets: the partition {p, m ^ p} where p lacks m's highest leaf, so p is
// the lower mask of the two; ties go to the lowest p
RTB_HD void tlo_dp(TloWork &W, int m) {
    int hb = m;
    while (hb & (hb - 1)) hb &= hb - 1;
    const int rest = m ^ hb;
    if (rest == 0) { W.cost[m] = 0.f; W.part[m] = 0; return; }
    float best = 0.f; int bp = -1;
    for (int p = rest; p > 0; p = (p - 1) & rest) {  // (descending: `<=` keeps the lowest mask among equal costs)
        const float v = fadd(W.cost[p], W.cost[m ^ p]);
        if (bp < 0 || v <= best) { best = v; bp = p; }
    }
    W.cost[m] = fadd(W.area[m], best); W.part[m] = (uint8_t)bp;
}
// a child of inner[j] in the present topology: its leaf mask and cost (a leaf slot, or an inner node opened after j)
RTB_HD void tlo_child(const TloWork &W, int id, int &mask, float &cost) {
    for (int k = 0; k < W.nl; ++k) if (W.leaf[k] == id) { mask = 1 << k; cost = 0.f; return; }
    for (int j = 1; j < W.ni; ++j) if (W.inner[j] == id) { mask = W.imask[j]; cost = W.icost[j]; return; }
    mask = 0; cost = 0.f;  // (unreachable: every child of a treelet inner node is in the treelet)
}
// sum of inner areas of the present topology, with the programme's arithmetic (so the programme's cost is never higher)
RTB_HD float tlo_present_cost(const TloArgs &a, TloWork &W) {
    for (int j = W.ni - 1; j >= 0; --j) {  // (children were opened after their parent)
        const B2Node x = a.nodes[W.inner[j]];
        int ml, mr; float cl, cr;
        tlo_child(W, x.left, ml, cl);
        tlo_child(W, x.right, mr, cr);
        W.imask[j] = ml | mr;
        W.icost[j] = fadd(W.area[ml | mr], fadd(cl, cr));
    }
    return W.icost[0];
}
// the cheapest topology written over the treelet's inner ids: the root keeps its id, the other ids, in ascending
// order, go to the new inner nodes in breadth-first order, left child first; boxes, counts and parents rewritten
RTB_HD void tlo_rewrite(const TloArgs &a, TloWork &W, int full) {
    for (int j = 2; j < W.ni; ++j)
        for (int k = j; k > 1 && W.inner[k - 1] > W.inner[k]; --k) { const int t = W.inner[k]; W.inner[k] = W.inner[k - 1]; W.inner[k - 1] = t; }
    int head = 0, tail = 0, next = 1;
    W.qmask[tail] = full; W.qid[tail] = W.inner[0]; ++tail;
    while (head < tail) {
        const int m = W.qmask[head], id = W.qid[head];
        ++head;
        int ch[2];
        for (int s = 0; s < 2; ++s) {
            const int q = s == 0 ? W.part[m] : m ^ W.part[m];
            if (q & (q - 1)) {
                ch[s] = W.inner[next++];
                W.qmask[tail] = q; W.qid[tail] = ch[s]; ++tail;
            } else {
                int k = 0;
                while (!(q >> k & 1)) ++k;
                ch[s] = W.leaf[k];
            }
        }
        int cnt;
        B2Node u = tlo_union(W, m, cnt);
        u.left = ch[0]; u.right = ch[1];
        a.nodes[id] = u;
        a.count[id] = cnt;
        a.parent[ch[0]] = id; a.parent[ch[1]] = id;
    }
}
#if defined(__CUDA_ARCH__)
#define RTB_TLO_SYNC() __syncwarp()
#else
#define RTB_TLO_SYNC()
#endif
// treelet of root order[first + tid], by `lanes` lanes (a warp on the GPU, 1 in the host emulation): lane 0 forms and
// rewires it, the subsets are shared out between the lanes
RTB_HD void tlo_treelet(const TloArgs &a, TloWork &W, int tid, int lane, int lanes) {
    const int root = a.order[a.first + tid];
    if (a.count[root] < a.gamma) return;
    if (lane == 0) tlo_form(a, W, root);
    RTB_TLO_SYNC();
    const int nl = W.nl;
    if (nl < 3) return;  // (two leaves: one topology)
    const int full = (1 << nl) - 1;
    for (int m = 1 + lane; m <= full; m += lanes) { int cnt; W.area[m] = b2_half_area(tlo_union(W, m, cnt)); }
    RTB_TLO_SYNC();
    for (int s = 1; s <= nl; ++s) {  // by subset size: a subset's partitions are smaller
        for (int m = 1 + lane; m <= full; m += lanes) if (popc((uint32_t)m) == s) tlo_dp(W, m);
        RTB_TLO_SYNC();
    }
    if (lane == 0 && W.cost[full] < tlo_present_cost(a, W)) tlo_rewrite(a, W, full);
}

// ------------------------------------------------------------ 4. collapse plan
// cost[n][i-1], i = 1..7: SAH cost of subtree n laid out in at most i child
// slots.  plan[n][i-1]: kPlanLeaf / kPlanInner (one slot), k = 1..6 (split:
// the left child gets k slots, the right one i-k), 0 (same as with i-1
// slots).  plan[n][7]: how a wide node rooted at n splits its 8 slots.
constexpr uint8_t kPlanLeaf = 100, kPlanInner = 101;
struct PlanArgs {
    const B2Node *nodes;
    const int32_t *count;
    float *cost;      // [num binary nodes][7]
    uint8_t *plan;    // [num binary nodes][8]
    int32_t first, n; // this launch covers binary nodes first .. first+n-1 (one PLOC round: children are older)
    int32_t max_leaf;
    const int32_t *order;  // null: the nodes are ids first ..; else order[first ..] (the binned-SAH tree: one depth per launch)
};
RTB_HD void plan_child_costs(const PlanArgs &a, int c, float *d) {
    const B2Node x = a.nodes[c];
    if (x.right < 0) {  // a single triangle: a leaf child whatever the slot budget
        const float v = fmul(b2_half_area(x), kSahTriCost);
        for (int i = 0; i < 7; ++i) d[i] = v;
    } else {
        for (int i = 0; i < 7; ++i) d[i] = a.cost[(size_t)c * 7 + i];
    }
}
RTB_HD void plan_body(const PlanArgs &a, int tid) {
    if (tid >= a.n) return;
    const int id = a.order ? a.order[a.first + tid] : a.first + tid;
    const B2Node self = a.nodes[id];
    if (self.right < 0) return;
    float dl[7], dr[7];
    plan_child_costs(a, self.left, dl);
    plan_child_costs(a, self.right, dr);
    // best split of i slots between the two children, i = 2..8
    float split[9]; uint8_t split_k[9];
    for (int i = 2; i <= 8; ++i) {
        float best = FLT_MAX; int bk = 1;
        for (int k = 1; k < i; ++k) {
            if (k > 7 || i - k > 7) continue;
            const float v = fadd(dl[k - 1], dr[i - k - 1]);
            if (v < best) { best = v; bk = k; }
        }
        split[i] = best; split_k[i] = (uint8_t)bk;
    }
    const float area = b2_half_area(self);
    const int cnt = a.count[id];
    const float as_inner = ffma(area, kSahNodeCost, split[8]);
    const float as_leaf = cnt <= a.max_leaf ? fmul(area, fmul(kSahTriCost, (float)cnt)) : FLT_MAX;
    float *cost = a.cost + (size_t)id * 7;
    uint8_t *plan = a.plan + (size_t)id * 8;
    float cur = as_leaf <= as_inner ? as_leaf : as_inner;
    cost[0] = cur; plan[0] = as_leaf <= as_inner ? kPlanLeaf : kPlanInner;
    for (int i = 2; i <= 7; ++i) {
        if (split[i] < cur) { cur = split[i]; plan[i - 1] = split_k[i]; }
        else plan[i - 1] = 0;
        cost[i - 1] = cur;
    }
    plan[7] = split_k[8];
}
// children of the wide node rooted at binary node `root`, as planned; returns their number (<= 8)
RTB_HD int plan_expand(const B2Node *nodes, const uint8_t *plan, int root, int *ch) {
    int nc = 0;
    int st_n[16], st_i[16]; int sp = 0;
    const B2Node r = nodes[root];
    const int k8 = plan[(size_t)root * 8 + 7];
    st_n[sp] = r.right; st_i[sp] = 8 - k8; ++sp;
    st_n[sp] = r.left; st_i[sp] = k8; ++sp;
    while (sp) {
        --sp;
        const int n = st_n[sp]; int i = st_i[sp];
        const B2Node x = nodes[n];
        if (x.right < 0) { ch[nc++] = n; continue; }
        if (i > 7) i = 7;
        const uint8_t *pl = plan + (size_t)n * 8;
        while (i > 1 && pl[i - 1] == 0) --i;
        const int d = pl[i - 1];
        if (i == 1 || d == kPlanLeaf || d == kPlanInner) { ch[nc++] = n; continue; }
        st_n[sp] = x.right; st_i[sp] = i - d; ++sp;
        st_n[sp] = x.left; st_i[sp] = d; ++sp;
    }
    return nc;
}

// ------------------------------------------------------------ 5. collapse
struct WorkItem {
    int32_t b2;    // binary node to expand
    int32_t wide;  // index of the 8-wide node to write
};
struct CollapseArgs {
    const B2Node *nodes;
    const int32_t *count;
    const uint8_t *plan;       // collapse plan, or null: open the largest child first (A/B)
    const Tri48 *tri_in;       // caller order
    const TriMeta *meta_in;    // caller order
    Q4 *nodes8;
    Tri48 *tris_out;           // leaf order
    TriMeta *meta_out;
    int32_t *prim_out;         // leaf order -> caller index
    int32_t *leaf_of_prim;     // caller index -> leaf order
    int32_t *node_counter;     // next free wide node (root = 0 pre-allocated)
    int32_t *tri_counter;
    const WorkItem *work_in; int32_t n_in;  // (n_in_dev set: n_in is unused)
    const int32_t *n_in_dev;                // work items of this level, in device memory: levels are enqueued without reading it back
    WorkItem *work_out; int32_t *n_out;
    float *sah;                // accumulated SAH cost (unnormalised)
    int32_t max_leaf;          // 1..3
    int32_t *gather;           // [n] leaf order: binary subtree whose triangles start at this slot, or -1 (gather_body)
    int32_t *level_nodes;      // null, or where this level records its number of work items = 8-wide nodes of its depth
                               // (the depth schedule of the refit: a level's nodes are one contiguous range of ids)
};
// triangles of the leaf children, in leaf order: slot d holds the binary subtree whose (<= 3) triangles go to d, d+1, ..
// (left to right) or -1; one thread per slot, after the collapse
RTB_HD void gather_body(const CollapseArgs &a, int n, int d) {
    if (d >= n) return;
    const int root = a.gather[d];
    if (root < 0) return;
    int st[4]; int sp = 0; st[sp++] = root;
    int dst = d;
    while (sp) {
        const int ni = st[--sp];
        const B2Node x = a.nodes[ni];
        if (x.right < 0) {
            if (a.tri_in) {  // (null: the tree over the instances of a two-level scene, whose leaves are boxes)
                a.tris_out[dst] = a.tri_in[x.left];
                a.meta_out[dst] = a.meta_in[x.left];
            }
            a.prim_out[dst] = x.left;
            a.leaf_of_prim[x.left] = dst;
            dst++;
        } else {
            st[sp++] = x.right; st[sp++] = x.left;
        }
    }
}

RTB_HD void collapse_body(const CollapseArgs &a, int tid) {
    const int n_in = a.n_in_dev ? *a.n_in_dev : a.n_in;
    if (tid >= n_in) return;
    if (tid == 0 && a.level_nodes) *a.level_nodes = n_in;
    const WorkItem item = a.work_in[tid];
    const B2Node self = a.nodes[item.b2];
    int ch[8];
    int nc;
    // boxes and triangle counts of the children chosen so far: every level of this loop costs one round trip to
    // memory (the two nodes a child is opened into), and nothing is read twice
    B2Node cb[8];
    int ccnt[8];
    if (a.count[item.b2] <= a.max_leaf) { ch[0] = item.b2; nc = 1; }  // tiny scene: root is one leaf
    else if (a.plan) { nc = plan_expand(a.nodes, a.plan, item.b2, ch); }
    else { ch[0] = self.left; ch[1] = self.right; nc = 2; }
    for (int k = 0; k < nc; ++k) { cb[k] = a.nodes[ch[k]]; ccnt[k] = a.count[ch[k]]; }
    // without a plan: open the largest child until 8 children or only leaves remain
    while (!a.plan && nc < 8) {
        int best = -1; float best_a = -1.f;
        for (int k = 0; k < nc; ++k) {
            if (ccnt[k] > a.max_leaf) {
                const float ar = b2_half_area(cb[k]);
                if (ar > best_a) { best_a = ar; best = k; }
            }
        }
        if (best < 0) break;
        const int l = cb[best].left, r = cb[best].right;
        ch[best] = l; ch[nc] = r;
        cb[best] = a.nodes[l]; cb[nc] = a.nodes[r];
        ccnt[best] = a.count[l]; ccnt[nc] = a.count[r];
        ++nc;
    }
    // slot assignment (greedy): slot s "looks" towards (s&1?+:-, s&2?+:-, s&4?+:-);
    // a child goes to the slot best aligned with its offset from the node
    // centre, so that `slot ^ octinv` orders children front to back
    const float pcx = fmul(0.5f, fadd(self.lox, self.hix)), pcy = fmul(0.5f, fadd(self.loy, self.hiy)),
                pcz = fmul(0.5f, fadd(self.loz, self.hiz));
    // (every index into cost / todo / free below is a compile-time constant once the loops are unrolled: the matrix stays
    // in registers; dynamically indexed it lived in local memory, and the 8 x 64 dependent compares of the greedy
    // assignment were a third of a level's critical path)
    float cost[8][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const B2Node &c = cb[k < nc ? k : 0];
        const float dx = fsub(fmul(0.5f, fadd(c.lox, c.hix)), pcx);
        const float dy = fsub(fmul(0.5f, fadd(c.loy, c.hiy)), pcy);
        const float dz = fsub(fmul(0.5f, fadd(c.loz, c.hiz)), pcz);
#pragma unroll
        for (int s = 0; s < 8; ++s)
            cost[k][s] = fadd(fadd((s & 1) ? dx : -dx, (s & 2) ? dy : -dy), (s & 4) ? dz : -dz);
    }
    int slot_child[8];
    for (int s = 0; s < 8; ++s) slot_child[s] = -1;
    uint32_t todo = (1u << nc) - 1u, free_slots = 0xffu;  // children not placed yet, slots not taken yet
    for (int round = 0; round < nc; ++round) {
        float bc = -FLT_MAX; int bk = -1, bs = -1;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (!(todo >> k & 1u)) continue;
#pragma unroll
            for (int s = 0; s < 8; ++s) {
                if (!(free_slots >> s & 1u)) continue;
                if (cost[k][s] > bc) { bc = cost[k][s]; bk = k; bs = s; }
            }
        }
        slot_child[bs] = bk;
        todo &= ~(1u << bk); free_slots &= ~(1u << bs);
    }
    // allocate children and triangles
    int n_inner = 0, n_tris = 0;
    for (int k = 0; k < nc; ++k) {
        const int cnt = ccnt[k];
        if (cnt > a.max_leaf) n_inner++; else n_tris += cnt;
    }
    const int child_base = n_inner ? atomic_add_i(a.node_counter, n_inner) : 0;
    const int tri_base = n_tris ? atomic_add_i(a.tri_counter, n_tris) : 0;
    const int work_base = n_inner ? atomic_add_i(a.n_out, n_inner) : 0;
    // quantisation frame
    const uint32_t ex = quant_exponent(fsub(self.hix, self.lox)), ey = quant_exponent(fsub(self.hiy, self.loy)),
                   ez = quant_exponent(fsub(self.hiz, self.loz));
    uint32_t meta[8], qlx[8], qly[8], qlz[8], qhx[8], qhy[8], qhz[8];
    uint32_t imask = 0;
    int inner_seen = 0, tri_off = 0;
    float sah = fmul(b2_half_area(self), kSahNodeCost);
    for (int s = 0; s < 8; ++s) {
        const int k = slot_child[s];
        if (k < 0) {
            meta[s] = 0; qlx[s] = qly[s] = qlz[s] = 255u; qhx[s] = qhy[s] = qhz[s] = 0u;
            continue;
        }
        const B2Node &c = cb[k];
        qlx[s] = quant_lo(c.lox, self.lox, ex); qhx[s] = quant_hi(c.hix, self.lox, ex);
        qly[s] = quant_lo(c.loy, self.loy, ey); qhy[s] = quant_hi(c.hiy, self.loy, ey);
        qlz[s] = quant_lo(c.loz, self.loz, ez); qhz[s] = quant_hi(c.hiz, self.loz, ez);
        const int cnt = ccnt[k];
        if (cnt > a.max_leaf) {
            meta[s] = 0x20u | (24u + (uint32_t)s);
            imask |= 1u << s;
            WorkItem w; w.b2 = ch[k]; w.wide = child_base + inner_seen;
            a.work_out[work_base + inner_seen] = w;
            inner_seen++;
        } else {
            meta[s] = (((1u << cnt) - 1u) << 5) | (uint32_t)tri_off;
            sah = ffma(b2_half_area(c), fmul(kSahTriCost, (float)cnt), sah);
            // the (<= 3) triangles of this subtree go to tri_base + tri_off ...: gathered by gather_body, one thread per
            // leaf child, after the last level (walking the subtree here put 8 x 3 dependent loads on every level's
            // critical path).  Every triangle slot is written once: the subtree at a leaf child's first slot, -1 behind it
            a.gather[tri_base + tri_off] = ch[k];
            for (int t = 1; t < cnt; ++t) a.gather[tri_base + tri_off + t] = -1;
            tri_off += cnt;
        }
    }
#if defined(__CUDA_ARCH__)
    {   // one float atomic per warp (a level of a 10 M-triangle build has a million nodes, and floating-point
        // reductions to one address are not aggregated by the compiler); the cost is a statistic, its summation order is free
        const unsigned m = __activemask();  // (whatever lanes arrive here together: the loops above diverge)
        float v = 0.f;
        for (unsigned r = m; r != 0u; r &= r - 1u) v += __shfl_sync(m, sah, __ffs(r) - 1);
        if ((threadIdx.x & 31) == __ffs(m) - 1) atomic_add_f(a.sah, v);
    }
#else
    atomic_add_f(a.sah, sah);
#endif
    Q4 w0, w1, w2, w3, w4;
    w0.x = f2u(self.lox); w0.y = f2u(self.loy); w0.z = f2u(self.loz);
    w0.w = ex | (ey << 8) | (ez << 16) | (imask << 24);
    w1.x = (uint32_t)child_base; w1.y = (uint32_t)tri_base;
    w1.z = meta[0] | (meta[1] << 8) | (meta[2] << 16) | (meta[3] << 24);
    w1.w = meta[4] | (meta[5] << 8) | (meta[6] << 16) | (meta[7] << 24);
#define RTB_PACK4(q, o) ((q)[o] | ((q)[o + 1] << 8) | ((q)[o + 2] << 16) | ((q)[o + 3] << 24))
    w2.x = RTB_PACK4(qlx, 0); w2.y = RTB_PACK4(qlx, 4); w2.z = RTB_PACK4(qly, 0); w2.w = RTB_PACK4(qly, 4);
    w3.x = RTB_PACK4(qlz, 0); w3.y = RTB_PACK4(qlz, 4); w3.z = RTB_PACK4(qhx, 0); w3.w = RTB_PACK4(qhx, 4);
    w4.x = RTB_PACK4(qhy, 0); w4.y = RTB_PACK4(qhy, 4); w4.z = RTB_PACK4(qhz, 0); w4.w = RTB_PACK4(qhz, 4);
#undef RTB_PACK4
    Q4 *dst = a.nodes8 + (size_t)item.wide * kNodeWords;
    dst[0] = w0; dst[1] = w1; dst[2] = w2; dst[3] = w3; dst[4] = w4;
}

// ------------------------------------------------------------ 6. refit (rtb_scene_refit)
// New vertices, same topology.  The record pass turns caller-order vertices into the records at leaf_of_prim[i], with the
// vertex check of prim_setup.  The refit pass then goes one depth at a time, deepest first, and recomputes each node
// from its own words: a leaf child's box is the union of its triangles' boxes (tri_box), an inner child's box is the
// exact box the deeper level left in `box`, and the node's origin, exponents and quantised planes are rewritten with the
// functions of collapse_body (child_base, tri_base, meta and imask stay).  The collapse's frame is its binary node's
// box, which is the union of the triangle boxes below it: with the original vertices the refit writes the same words.
struct RefitTrisArgs {
    const float *vertices;         // 9 per triangle, caller order
    const int32_t *leaf_of_prim;   // caller index -> leaf order
    F4 *tris;                      // [n] leaf order, 3 words per triangle (whole 16-byte stores: the writes scatter)
    int32_t *bad;                  // raised when a vertex is not finite or beyond kMaxCoord
    int32_t n;
};
RTB_HD void refit_tris_body(const RefitTrisArgs &a, int i) {
    if (i >= a.n) return;
    const float *v = a.vertices + 9 * (size_t)i;
    const Tri48 t = tri_from_vertices(v3(v[0], v[1], v[2]), v3(v[3], v[4], v[5]), v3(v[6], v[7], v[8]));
    V3 lo, hi;
    if (tri_box(t, lo, hi)) *a.bad = 1;
    F4 *d = a.tris + 3 * (size_t)a.leaf_of_prim[i];
    F4 w;
    w.x = t.p0x; w.y = t.p0y; w.z = t.p0z; w.w = t.e1x; d[0] = w;
    w.x = t.e1y; w.y = t.e1z; w.z = t.e2x; w.w = t.e2y; d[1] = w;
    w.x = t.e2z; w.y = t.nx; w.z = t.ny; w.w = t.nz; d[2] = w;
}
struct RefitArgs {
    Q4 *nodes8;
    const F4 *tris;           // leaf order, 3 words per triangle
    float *box;               // [nodes][6]: exact box (lo xyz, hi xyz) of every node refit so far
    const int32_t *order;     // null: this launch refits nodes first .. first + num - 1; else order[first .. first + num)
    int32_t first, num;
    float *sah;               // accumulated 8-wide SAH cost (unnormalised), as collapse_body sums it
};
// refits one node; returns its term of the SAH cost
RTB_HD float refit_body(const RefitArgs &a, int tid) {
    const int id = a.order ? a.order[a.first + tid] : a.first + tid;
    Q4 *nd = a.nodes8 + (size_t)id * kNodeWords;
    const Q4 w0 = nd[0], w1 = nd[1];
    const uint32_t imask = w0.w >> 24;
    V3 clo[8], chi[8];
    int cnt[8];  // triangles of a leaf child, 0: inner child or empty slot
    V3 lo = v3(FLT_MAX), hi = v3(-FLT_MAX);
#pragma unroll
    for (int s = 0; s < 8; ++s) {
        const uint32_t m = ((s < 4 ? w1.z : w1.w) >> (8 * (s & 3))) & 0xffu;
        cnt[s] = 0;
        clo[s] = v3(FLT_MAX); chi[s] = v3(-FLT_MAX);
        if (imask >> s & 1u) {
            const float *b = a.box + 6 * (size_t)(w1.x + (uint32_t)popc(imask & ((1u << s) - 1u)));
            clo[s] = v3(b[0], b[1], b[2]); chi[s] = v3(b[3], b[4], b[5]);
        } else if (m) {
            cnt[s] = popc(m >> 5);
            for (int t = 0; t < cnt[s]; ++t) {
                V3 l, h;
                tri_box(load_tri(a.tris, (int)(w1.y + (m & 31u)) + t), l, h);
                clo[s] = v3(fminf(clo[s].x, l.x), fminf(clo[s].y, l.y), fminf(clo[s].z, l.z));
                chi[s] = v3(fmaxf(chi[s].x, h.x), fmaxf(chi[s].y, h.y), fmaxf(chi[s].z, h.z));
            }
        } else {
            continue;
        }
        lo = v3(fminf(lo.x, clo[s].x), fminf(lo.y, clo[s].y), fminf(lo.z, clo[s].z));
        hi = v3(fmaxf(hi.x, chi[s].x), fmaxf(hi.y, chi[s].y), fmaxf(hi.z, chi[s].z));
    }
    const uint32_t ex = quant_exponent(fsub(hi.x, lo.x)), ey = quant_exponent(fsub(hi.y, lo.y)), ez = quant_exponent(fsub(hi.z, lo.z));
    uint32_t qlx[8], qly[8], qlz[8], qhx[8], qhy[8], qhz[8];
    float sah = fmul(half_area(fsub(hi.x, lo.x), fsub(hi.y, lo.y), fsub(hi.z, lo.z)), kSahNodeCost);
#pragma unroll
    for (int s = 0; s < 8; ++s) {
        const bool used = cnt[s] > 0 || (imask >> s & 1u);
        qlx[s] = used ? quant_lo(clo[s].x, lo.x, ex) : 255u; qhx[s] = used ? quant_hi(chi[s].x, lo.x, ex) : 0u;
        qly[s] = used ? quant_lo(clo[s].y, lo.y, ey) : 255u; qhy[s] = used ? quant_hi(chi[s].y, lo.y, ey) : 0u;
        qlz[s] = used ? quant_lo(clo[s].z, lo.z, ez) : 255u; qhz[s] = used ? quant_hi(chi[s].z, lo.z, ez) : 0u;
        if (cnt[s] > 0)
            sah = ffma(half_area(fsub(chi[s].x, clo[s].x), fsub(chi[s].y, clo[s].y), fsub(chi[s].z, clo[s].z)), fmul(kSahTriCost, (float)cnt[s]), sah);
    }
    float *b = a.box + 6 * (size_t)id;
    b[0] = lo.x; b[1] = lo.y; b[2] = lo.z; b[3] = hi.x; b[4] = hi.y; b[5] = hi.z;
    Q4 o0, w2, w3, w4;
    o0.x = f2u(lo.x); o0.y = f2u(lo.y); o0.z = f2u(lo.z);
    o0.w = ex | (ey << 8) | (ez << 16) | (imask << 24);
#define RTB_PACK4(q, o) ((q)[o] | ((q)[o + 1] << 8) | ((q)[o + 2] << 16) | ((q)[o + 3] << 24))
    w2.x = RTB_PACK4(qlx, 0); w2.y = RTB_PACK4(qlx, 4); w2.z = RTB_PACK4(qly, 0); w2.w = RTB_PACK4(qly, 4);
    w3.x = RTB_PACK4(qlz, 0); w3.y = RTB_PACK4(qlz, 4); w3.z = RTB_PACK4(qhx, 0); w3.w = RTB_PACK4(qhx, 4);
    w4.x = RTB_PACK4(qhy, 0); w4.y = RTB_PACK4(qhy, 4); w4.z = RTB_PACK4(qhz, 0); w4.w = RTB_PACK4(qhz, 4);
#undef RTB_PACK4
    nd[0] = o0; nd[2] = w2; nd[3] = w3; nd[4] = w4;
    return sah;
}

// ------------------------------------------------------------ two-level scenes
// bounds of pre-computed boxes (the instances' world boxes) instead of prim_setup
RTB_HD void box_bounds_body(const F4 *lo, const F4 *hi, int32_t *scene_bounds, int n, int i) {
    if (i >= n) return;
    const F4 l = lo[i], h = hi[i];
    atomic_min_i(scene_bounds + 0, float_to_ordered(l.x));
    atomic_min_i(scene_bounds + 1, float_to_ordered(l.y));
    atomic_min_i(scene_bounds + 2, float_to_ordered(l.z));
    atomic_max_i(scene_bounds + 3, float_to_ordered(h.x));
    atomic_max_i(scene_bounds + 4, float_to_ordered(h.y));
    atomic_max_i(scene_bounds + 5, float_to_ordered(h.z));
}
// world box of every instance from its mesh's transformed VERTICES (the box of the transformed mesh box is up to 40 %
// wider for a rotated mesh, and every box a ray crosses costs a visit of that mesh's root): one thread per
// (instance, run of kInstBoundsRun triangles)
constexpr int kInstBoundsRun = 64;
struct InstBoundsArgs {
    const Tri48 *tris;          // leaf order; mesh m = [first, first + count)
    const float *xforms;        // 12 floats per instance, object -> world
    const int32_t *first, *count;  // per instance: its mesh's range
    int32_t *bounds;            // 6 ordered ints per instance: min xyz, max xyz
    int32_t num_inst, runs;     // runs = ceil(largest mesh / kInstBoundsRun)
};
RTB_HD void inst_bounds_body(const InstBoundsArgs &a, int tid) {
    const int i = tid / a.runs, c = tid % a.runs;
    if (i >= a.num_inst) return;
    const int cnt = a.count[i], t0 = c * kInstBoundsRun;
    if (t0 >= cnt) return;
    const int t1 = t0 + kInstBoundsRun < cnt ? t0 + kInstBoundsRun : cnt;
    const float *m = a.xforms + 12 * (size_t)i;
    F4 r0, r1, r2;
    r0.x = m[0]; r0.y = m[1]; r0.z = m[2]; r0.w = m[3]; r1.x = m[4]; r1.y = m[5]; r1.z = m[6]; r1.w = m[7];
    r2.x = m[8]; r2.y = m[9]; r2.z = m[10]; r2.w = m[11];
    V3 lo = v3(FLT_MAX), hi = v3(-FLT_MAX);
    for (int t = t0; t < t1; ++t) {
        const Tri48 tr = a.tris[a.first[i] + t];
        const V3 p0 = tri_p0(tr);
        const V3 q[3] = {xform_point(r0, r1, r2, p0), xform_point(r0, r1, r2, vsub(p0, tri_e1(tr))), xform_point(r0, r1, r2, vadd(p0, tri_e2(tr)))};
        for (int k = 0; k < 3; ++k) {
            lo = v3(fminf(lo.x, q[k].x), fminf(lo.y, q[k].y), fminf(lo.z, q[k].z));
            hi = v3(fmaxf(hi.x, q[k].x), fmaxf(hi.y, q[k].y), fmaxf(hi.z, q[k].z));
        }
    }
    int32_t *b = a.bounds + 6 * (size_t)i;
    atomic_min_i(b + 0, float_to_ordered(lo.x)); atomic_min_i(b + 1, float_to_ordered(lo.y)); atomic_min_i(b + 2, float_to_ordered(lo.z));
    atomic_max_i(b + 3, float_to_ordered(hi.x)); atomic_max_i(b + 4, float_to_ordered(hi.y)); atomic_max_i(b + 5, float_to_ordered(hi.z));
}
// a mesh's tree is built with indices relative to itself; in the scene's arrays its nodes start at node_off and its
// triangles at tri_off
RTB_HD void rebase_node_body(const Q4 *src, Q4 *dst, uint32_t node_off, uint32_t tri_off, int n, int i) {
    if (i >= n) return;
    const Q4 *s = src + (size_t)i * kNodeWords;
    Q4 *d = dst + (size_t)i * kNodeWords;
    Q4 w1 = s[1];
    w1.x += node_off; w1.y += tri_off;
    d[0] = s[0]; d[1] = w1; d[2] = s[2]; d[3] = s[3]; d[4] = s[4];
}

// area lights refer to their triangle by leaf-order index after the build
RTB_HD void light_fix_body(LightDev *lights, const int64_t *light_tri, const int32_t *leaf_of_prim, int n, int i) {
    if (i >= n) return;
    if (lights[i].type == RTB_AREA_LIGHT) lights[i].tri = leaf_of_prim[light_tri[i]];
    else lights[i].tri = -1;
}

}  // namespace rtb
