// rtb_engine.h — host-side orchestration of the builder and of the wavefront
// loop, written once against a small backend interface.
//
// The product backend is CudaBackend (rtb_cuda.cu): device memory, named
// sm_100a kernels, CUB radix sort / select, CUDA events.  tests/emu has a
// HostBackend that runs the same kernel bodies in plain loops so the logic
// can be checked against the oracle on a machine without a GPU; the shipped
// library never contains it (no CPU fallback).
//
// Host loop being replaced: render(), render.cuh:366-457 (13 launches and 4
// blocking 4-byte device->host copies per iteration); here an iteration is 4
// launches (shade, generate, control, trace), and the host looks at one `done` word every few iterations.
#pragma once
#include <algorithm>
#include <cmath>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

#include "rtb_build.h"
#include "rtb_wavefront.h"

namespace rtb {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

// device temporary that is freed on every path out of its scope (an exception included)
template <class BE, class T>
struct DeviceBuf {
    BE &be; T *p;
    DeviceBuf(BE &b, size_t n) : be(b), p(n ? b.template alloc<T>(n) : nullptr) {}
    ~DeviceBuf() { be.free(p); }
    DeviceBuf(const DeviceBuf &) = delete;
    DeviceBuf &operator=(const DeviceBuf &) = delete;
    T *release() { T *q = p; p = nullptr; return q; }
};

// the device temporaries of one build: whatever is still held when the scope ends — normally or by an exception — is freed
template <class BE>
struct Temps {
    BE &be;
    std::vector<void *> held;
    explicit Temps(BE &b) : be(b) {}
    ~Temps() { for (void *p : held) be.free(p); }
    Temps(const Temps &) = delete;
    Temps &operator=(const Temps &) = delete;
    template <class T> T *alloc(size_t n) {
        held.push_back(nullptr);  // (the slot first: push_back may throw, an allocation must not be lost to it)
        T *p = be.template alloc<T>(n);
        held.back() = p;
        return p;
    }
    void free(void *p) {  // early release (peak memory): no longer held
        for (auto &h : held) if (h == p) { h = nullptr; break; }
        be.free(p);
    }
};

// ---- kernel functors (named types => readable kernel names in ncu) ----
struct PrimSetupK { PrimSetupArgs a; RTB_HD void operator()(int i) const { prim_setup_body(a, i); } };
struct MortonK { MortonArgs a; RTB_HD void operator()(int i) const { morton_body(a, i); } };
struct PlocLeafK {
    const F4 *lo, *hi; const int32_t *sorted; B2Node *nodes; int32_t *count, *clusters; int n;
    RTB_HD void operator()(int i) const { ploc_leaf_body(lo, hi, sorted, nodes, count, clusters, n, i); }
};
struct PlocNnK { PlocArgs a; RTB_HD void operator()(int i) const { ploc_nn_body(a, i); } };
struct PlocMergeK { PlocArgs a; int n_leaves; RTB_HD void operator()(int i) const { ploc_merge_body(a, n_leaves, i); } };
struct PlanK { PlanArgs a; RTB_HD void operator()(int i) const { plan_body(a, i); } };
struct CollapseK { CollapseArgs a; RTB_HD void operator()(int i) const { collapse_body(a, i); } };
struct GatherK { CollapseArgs a; int n; RTB_HD void operator()(int i) const { gather_body(a, n, i); } };
struct LightFixK {
    LightDev *lights; const int64_t *light_tri; const int32_t *leaf_of_prim; int n;
    RTB_HD void operator()(int i) const { light_fix_body(lights, light_tri, leaf_of_prim, n, i); }
};
// gather of reference-layout primitives (primitive.cuh:4-12 holding device pointers)
struct RefPrimitive { const void *tri, *mat, *light; };
struct IngestK {
    const RefPrimitive *prims; const char *tri_base, *mat_base, *light_base;
    const rtb_material *materials; Tri48 *tri_in; TriMeta *meta_in; int64_t *light_tri; const void **light_ptr; int32_t *bad;
    int n, num_mats, num_lights;
    RTB_HD void operator()(int i) const {
        if (i >= n) return;
        const RefPrimitive p = prims[i];
        const float *t = (const float *)p.tri;  // Triangle {p0,e1,e2,n}, 12 floats, triangle.cuh:20
        Tri48 r;
        r.p0x = t[0]; r.p0y = t[1]; r.p0z = t[2]; r.e1x = t[3]; r.e1y = t[4]; r.e1z = t[5];
        r.e2x = t[6]; r.e2y = t[7]; r.e2z = t[8]; r.nx = t[9]; r.ny = t[10]; r.nz = t[11];
        tri_in[i] = r;
        const long long mo = (const char *)p.mat - mat_base;
        TriMeta tm;
        tm.light = -1;
        if (mo < 0 || mo % 20 != 0 || mo / 20 >= num_mats) { *bad = 1; tm.material = 0; meta_in[i] = tm; return; }  // a pointer outside d_materials
        const int m = (int)(mo / 20);
        tm.material = m | (materials[m].type << 24);
        if (light_ptr) {  // lights follow later (attach_lights): remember the pointer
            light_ptr[i] = p.light;
        } else if (p.light) {
            const long long lo = (const char *)p.light - light_base;
            if (lo < 0 || lo % 40 != 0 || lo / 40 >= num_lights) { *bad = 2; meta_in[i] = tm; return; }
            tm.light = (int)(lo / 40);
            light_tri[tm.light] = i;
        }
        meta_in[i] = tm;
    }
};
// per-triangle material / light ids of a flat description -> TriMeta (material index | type << 24, light index)
struct MetaK {
    const int32_t *mat, *light; const rtb_material *materials; TriMeta *out; int32_t *bad; int n, num_mats, num_lights;
    RTB_HD void operator()(int i) const {
        if (i >= n) return;
        const int m = mat[i], l = light ? light[i] : -1;
        TriMeta t; t.material = 0; t.light = -1;
        if (m < 0 || m >= num_mats) atomic_max_i(bad, 2);  // (the material error outranks the light error when a description has both)
        else if (l >= num_lights) atomic_max_i(bad, 1);
        else { t.material = m | (materials[m].type << 24); t.light = l < 0 ? -1 : l; }
        out[i] = t;
    }
};
// Scene{bvh, num_lights, d_lights} filled in after Bvh::Bvh (scene.cuh:4-8, main.cu:151-156): resolve the primitives'
// light pointers against the light array now known
struct AttachLightsK {
    const void *const *light_ptr; const char *light_base; const int32_t *leaf_of_prim; TriMeta *meta; int32_t *bad; int n, num_lights;
    RTB_HD void operator()(int i) const {
        if (i >= n) return;
        int idx = -1;
        if (light_ptr[i]) {
            const long long lo = (const char *)light_ptr[i] - light_base;
            if (lo < 0 || lo % 40 != 0 || lo / 40 >= num_lights) *bad = 2; else idx = (int)(lo / 40);
        }
        meta[leaf_of_prim[i]].light = idx;
    }
};
struct GenerateK { WaveState W; RenderConsts rc; };
struct ShadeK { WaveState W; SceneView S; RenderConsts rc; int type; bool shadows; };
struct TonemapK {  // post_process_framebuffer, render.cuh:330-338
    const float *in; float *out; int64_t n; float inv_spp;
    RTB_HD void operator()(int i) const { if (i < n) out[i] = fsqrt(fmul(in[i], inv_spp)); }
};
// what a render leaves behind: SceneT::accum (one F4 per pixel) or, in deterministic mode, SceneT::accum_fx (three
// fixed-point sums per pixel); these fold it into the caller's buffers / tonemap it
struct FoldF32K {  // caller's float[3 * pixels] += sums
    const F4 *in; const unsigned long long *in_fx; float *out; int64_t pixels;
    RTB_HD void operator()(int i) const {
        if (i >= pixels) return;
        float *o = out + 3 * (size_t)i;
        if (in_fx) {
            const unsigned long long *f = in_fx + 3 * (size_t)i;
            o[0] = fadd(o[0], from_fixed((long long)f[0])); o[1] = fadd(o[1], from_fixed((long long)f[1])); o[2] = fadd(o[2], from_fixed((long long)f[2]));
        } else {
            const F4 a = in[i];
            o[0] = fadd(o[0], a.x); o[1] = fadd(o[1], a.y); o[2] = fadd(o[2], a.z);
        }
    }
};
struct FoldFixedK {  // caller's int64[3 * pixels] += fixed-point sums
    const unsigned long long *in_fx; long long *out; int64_t n;
    RTB_HD void operator()(int i) const { if (i < n) out[i] = (long long)((unsigned long long)out[i] + in_fx[i]); }
};
struct TonemapAccumK {  // post_process_framebuffer, render.cuh:330-338, straight from the sums
    const F4 *in; const unsigned long long *in_fx; float *out; int64_t pixels; float inv_spp;
    RTB_HD void operator()(int i) const {
        if (i >= pixels) return;
        float r, g, b;
        if (in_fx) {
            const unsigned long long *f = in_fx + 3 * (size_t)i;
            r = from_fixed((long long)f[0]); g = from_fixed((long long)f[1]); b = from_fixed((long long)f[2]);
        } else {
            const F4 a = in[i];
            r = a.x; g = a.y; b = a.z;
        }
        float *o = out + 3 * (size_t)i;
        o[0] = fsqrt(fmul(r, inv_spp)); o[1] = fsqrt(fmul(g, inv_spp)); o[2] = fsqrt(fmul(b, inv_spp));
    }
};
struct TonemapFixedK {  // the same from a caller's int64[n] buffer of fixed-point sums (after a reduction over GPUs)
    const long long *in; float *out; int64_t n; float inv_spp;
    RTB_HD void operator()(int i) const { if (i < n) out[i] = fsqrt(fmul(from_fixed(in[i]), inv_spp)); }
};
RTB_HD bool ray_is_finite(const rtb_ray &r) {
    return finite3(v3(r.origin[0], r.origin[1], r.origin[2])) && finite3(v3(r.dir[0], r.dir[1], r.dir[2]));
}
struct TraceClosestK {
    Bvh8View B; const rtb_ray *rays; rtb_hit *hits; int64_t n; unsigned long long *counts;
    RTB_HD void operator()(int i) const {
        if (i >= n) return;
        const rtb_ray r = rays[i];
        HitRec h;
        int32_t hi = -1;
        if (!ray_is_finite(r)) {  // can hit nothing, would walk the whole tree
            rtb_hit o; o.t = 0.f; o.u = 0.f; o.v = 0.f; o.prim = -1;
            hits[i] = o;
            return;
        }
        if (counts) {
            TraceCounters c; c.nodes = 0; c.tris = 0;
            scene_trace<false, true>(B, v3(r.origin[0], r.origin[1], r.origin[2]), v3(r.dir[0], r.dir[1], r.dir[2]), r.tmax, -1, -1, h, hi, &c);
#if defined(__CUDA_ARCH__)
            atomicAdd(counts, (unsigned long long)c.nodes); atomicAdd(counts + 1, (unsigned long long)c.tris);
#else
            counts[0] += c.nodes; counts[1] += c.tris;
#endif
        } else {
            scene_trace<false, false>(B, v3(r.origin[0], r.origin[1], r.origin[2]), v3(r.dir[0], r.dir[1], r.dir[2]), r.tmax, -1, -1, h, hi, nullptr);
        }
        rtb_hit o;
        o.t = h.t; o.u = h.u; o.v = h.v; o.prim = h.tri >= 0 ? hit_prim(B, h.tri, hi) : -1;
        hits[i] = o;
    }
};
struct TraceAnyK {
    Bvh8View B; const rtb_ray *rays; const int32_t *excluded; const int32_t *leaf_of_prim; uint8_t *occluded; int64_t n;
    RTB_HD void operator()(int i) const {
        if (i >= n) return;
        const rtb_ray r = rays[i];
        if (!ray_is_finite(r)) { occluded[i] = 0; return; }
        int ex = excluded ? excluded[i] : -1, ex_inst = -1;
        if (ex >= 0 && B.inst) {  // id in the flattened numbering -> (instance, triangle of its mesh)
            int lo = 0, hi = B.num_inst - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (inst_info(B.inst, mid).flat_first <= ex) lo = mid; else hi = mid - 1;
            }
            const InstInfo in = inst_info(B.inst, lo);
            ex_inst = lo;
            ex = ex - in.flat_first + in.mesh_first;
        }
        if (ex >= 0) ex = leaf_of_prim[ex];
        HitRec h;
        int32_t hi_ = -1;
        occluded[i] = scene_trace<true, false>(B, v3(r.origin[0], r.origin[1], r.origin[2]), v3(r.dir[0], r.dir[1], r.dir[2]), r.tmax, ex, ex_inst, h, hi_, nullptr) ? 1 : 0;
    }
};

// known-answer hooks (rtb_kat_eval): the device functions of the render path, one record per thread.  Record
// layouts (floats; integers travel as their bits) are given in include/rtb.h.
RTB_HD int kat_in_floats(int which) { return which == 1 ? 16 : which == 2 ? 6 : which == 3 ? 4 : which == 4 ? 16 : which == 5 ? 20 : which == 6 ? 16 : 0; }
RTB_HD int kat_out_floats(int which) { return which == 1 ? 4 : which == 2 ? 3 : which == 3 ? 4 : which == 4 ? 12 : which == 5 ? 1 : which == 6 ? 8 : 0; }
struct KatK {
    int32_t which; const float *in; float *out; int64_t n;
    RTB_HD void operator()(int i) const {
        if (i >= n) return;
        const float *a = in + (size_t)i * kat_in_floats(which);
        float *o = out + (size_t)i * kat_out_floats(which);
        if (which == RTB_KAT_TRI_INTERSECT) {  // Triangle(p0,p1,p2) + Triangle::intersect, triangle.cuh:4-58
            const Tri48 tr = tri_from_vertices(v3(a[0], a[1], a[2]), v3(a[3], a[4], a[5]), v3(a[6], a[7], a[8]));
            float t = 0.f, u = 0.f, v = 0.f;
            const bool hit = tri_intersect(tr, v3(a[9], a[10], a[11]), v3(a[12], a[13], a[14]), a[15], t, u, v);
            o[0] = hit ? 1.f : 0.f; o[1] = t; o[2] = u; o[3] = v;
        } else if (which == RTB_KAT_OFFSET_ORIGIN) {  // offset_ray_origin, utility.cuh:31-47
            const V3 r = offset_ray_origin(v3(a[0], a[1], a[2]), v3(a[3], a[4], a[5]));
            o[0] = r.x; o[1] = r.y; o[2] = r.z;
        } else if (which == RTB_KAT_RAND4) {  // the counter-based generator that replaces curand_uniform, render.cuh:68-73
            const Rand4 r = rand4(f2u(a[0]), f2u(a[1]), f2u(a[2]), f2u(a[3]));
            o[0] = r.a; o[1] = r.b; o[2] = r.c; o[3] = r.d;
        } else if (which == RTB_KAT_SAMPLE_F) {  // Material::sample_f, material.cuh:60-109
            rtb_material m;
            m.albedo[0] = a[0]; m.albedo[1] = a[1]; m.albedo[2] = a[2]; m.ior = a[3]; m.type = f2i(a[4]);
            const BsdfSample s = sample_f(m, v3(a[5], a[6], a[7]), v3(a[8], a[9], a[10]), a[11], a[12]);
            o[0] = s.f.x; o[1] = s.f.y; o[2] = s.f.z; o[3] = s.n.x; o[4] = s.n.y; o[5] = s.n.z;
            o[6] = s.wi.x; o[7] = s.wi.y; o[8] = s.wi.z; o[9] = s.pdf; o[10] = 0.f; o[11] = 0.f;
        } else if (which == RTB_KAT_SLAB) {  // one child box through the quantiser and the slab test of the 8-wide node
            const V3 plo = v3(a[0], a[1], a[2]), phi = v3(a[3], a[4], a[5]);
            const uint32_t ex = quant_exponent(fsub(phi.x, plo.x)), ey = quant_exponent(fsub(phi.y, plo.y)), ez = quant_exponent(fsub(phi.z, plo.z));
            const uint32_t e255 = 0xffffff00u, e0 = 0u;
            Q4 n0, n1, n2, n3, n4;
            n0.x = f2u(plo.x); n0.y = f2u(plo.y); n0.z = f2u(plo.z); n0.w = ex | (ey << 8) | (ez << 16);
            n1.x = 0u; n1.y = 0u; n1.z = (1u << 5); n1.w = 0u;  // slot 0: a leaf child with one triangle; the rest empty
            n2.x = quant_lo(a[6], plo.x, ex) | e255; n2.y = 0xffffffffu; n2.z = quant_lo(a[7], plo.y, ey) | e255; n2.w = 0xffffffffu;
            n3.x = quant_lo(a[8], plo.z, ez) | e255; n3.y = 0xffffffffu; n3.z = quant_hi(a[9], plo.x, ex) | e0; n3.w = 0u;
            n4.x = quant_hi(a[10], plo.y, ey) | e0; n4.y = 0u; n4.z = quant_hi(a[11], plo.z, ez) | e0; n4.w = 0u;
            const RaySetup r = ray_setup(v3(a[12], a[13], a[14]), v3(a[15], a[16], a[17]));
            o[0] = (node_hitmask(n0, n1, n2, n3, n4, r, a[18]) & 0x00ffffffu) ? 1.f : 0.f;
        } else if (which == RTB_KAT_SAMPLE_LI) {  // Light::sample_Li (area), light.cuh:38-46 with triangle.cuh:78-86
            const Tri48 tr = tri_from_vertices(v3(a[0], a[1], a[2]), v3(a[3], a[4], a[5]), v3(a[6], a[7], a[8]));
            LightDev l; l.type = RTB_AREA_LIGHT; l.px = l.py = l.pz = 0.f; l.tri = 0; l.Lx = l.Ly = l.Lz = 1.f;
            const LightSample s = sample_Li_area(l, tr, v3(a[9], a[10], a[11]), a[12], a[13]);
            o[0] = s.wi.x; o[1] = s.wi.y; o[2] = s.wi.z; o[3] = s.t; o[4] = s.pdf; o[5] = o[6] = o[7] = 0.f;
        }
    }
};

// primary-hit feature buffers (rtb_render_aovs)
struct AovK {
    SceneView S; rtb_camera cam; int32_t width, height;
    float *albedo, *normal, *depth; int32_t *prim;
    RTB_HD void operator()(int i) const {
        if (i >= width * height) return;
        V3 o, d;
        camera_ray(cam, fdiv(fadd((float)(i % width), 0.5f), (float)width), fdiv(fadd((float)(i / width), 0.5f), (float)height), o, d);
        HitRec h;
        int32_t hi = -1;
        scene_trace<false, false>(S.bvh, o, d, FLT_MAX, -1, -1, h, hi, nullptr);
        V3 al = v3(0.f), n = v3(0.f);
        if (h.tri >= 0) {
            const rtb_material m = S.materials[hit_material(S, h.tri, hi) & 0xffffff];
            al = v3(m.albedo[0], m.albedo[1], m.albedo[2]);
            n = vneg(vnormalize(tri_n(load_tri_world(S.bvh, h.tri, hi))));  // the shading normal of render.cuh:153
            if (vdot(n, d) > 0.f) n = vneg(n);
        }
        if (albedo) { albedo[3 * (size_t)i] = al.x; albedo[3 * (size_t)i + 1] = al.y; albedo[3 * (size_t)i + 2] = al.z; }
        if (normal) { normal[3 * (size_t)i] = n.x; normal[3 * (size_t)i + 1] = n.y; normal[3 * (size_t)i + 2] = n.z; }
        if (depth) depth[i] = h.tri >= 0 ? h.t : 0.f;
        if (prim) prim[i] = h.tri >= 0 ? hit_prim(S.bvh, h.tri, hi) : -1;
    }
};

// ---- scene ----
constexpr int kMaxPipelines = 4;
// The ray / hit queues of the last scene that was destroyed, kept by the context for the next scene that renders with the
// same shape (rtb_scene_create + rtb_render + rtb_scene_destroy per frame is the end-to-end step of bench.py).  Returning
// 19 GB of queues to the stream-ordered pool and asking for them again works only while nothing else carves the cached
// blocks up in between: the temporaries of a 10 M-triangle build do, and the next render then waited ~190 ms for fresh
// memory from the driver.
struct WaveCache {
    WaveState W[kMaxPipelines]{};
    int32_t pool = 0, pipes = 0;
    size_t nq = 0;
    bool inst = false;
};
template <class BE>
void wave_cache_release(BE &be, WaveCache &c) {
    for (int k = 0; k < c.pipes; ++k) {
        WaveState &w = c.W[k];
        be.free(w.ea); be.free(w.eb); be.free(w.ec); be.free(w.ma); be.free(w.mb); be.free(w.mc);
        be.free(w.sh_o); be.free(w.sh_d); be.free(w.sh_L); be.free(w.c); be.free(w.hit_inst);
        w = WaveState{};
    }
    c.pool = 0; c.pipes = 0; c.nq = 0; c.inst = false;
}
template <class BE>
struct SceneT {
    BE *be = nullptr;
    int64_t n = 0;       // triangles stored
    int64_t n_flat = 0;  // triangles of the flattened scene (= n unless the scene is instanced): range of the hit ids
    // two-level scenes (scene_from_instanced): instance records, leaf order of the top tree -> instance
    F4 *inst = nullptr; int32_t *top_inst = nullptr; int32_t num_inst = 0;
    Q4 *nodes8 = nullptr;
    F4 *tris = nullptr;
    TriMeta *meta = nullptr;
    int32_t *prim = nullptr, *leaf_of_prim = nullptr;
    rtb_material *materials = nullptr;
    LightDev *lights = nullptr;
    int32_t num_materials = 0, num_lights = 0, num_nodes = 0;
    uint32_t type_mask = 0;  // bit t set iff some material has type t
    // reference-pointer ingest with the lights still to come (rtb_scene_attach_lights): the primitives' light pointers
    // in caller order, and the base of the caller's triangle array (area lights name their triangle by pointer)
    const void **deferred_light_ptr = nullptr; const char *ref_tri_base = nullptr;
    rtb_bvh_stats stats{};
    // in-place updates (refit_scene, set_instances).  The collapse levels of every tree: one tree for a flat scene, one
    // per mesh for an instanced scene, whose mesh trees start at tree_first[m] after the top tree's nodes
    rtb_build_params bp{};
    std::vector<std::vector<int32_t>> tree_levels;
    std::vector<int32_t> tree_first;
    // instanced scenes: the description's meshes and instances, which meshes hold emitters, the material types
    std::vector<int64_t> mesh_first;
    std::vector<rtb_instance> instances;
    std::vector<uint8_t> mesh_emissive;
    std::vector<int32_t> material_type;
    int mesh_levels = 0;
    // render state kept between calls (the reference re-allocates ~293 MB per
    // render() and never frees it, render.cuh:374-391)
    WaveState W[kMaxPipelines]{};
    int32_t pool = 0, pipes = 0;  // pool = queue entries PER pipeline
    F4 *accum = nullptr; unsigned long long *accum_fx = nullptr; int64_t accum_pixels = 0;  // radiance sums of the last render
    float *own_out = nullptr; int64_t own_out_floats = 0;  // rtb_render's tonemapped image before its copy to the host
    void ensure_accum(int64_t pixels, bool fixed) {
        if (accum_pixels != pixels) { be->free(accum); be->free(accum_fx); accum = nullptr; accum_fx = nullptr; accum_pixels = pixels; }
        if (!fixed && !accum) accum = be->template alloc<F4>((size_t)pixels);
        if (fixed && !accum_fx) accum_fx = be->template alloc<unsigned long long>(3 * (size_t)pixels);
    }

    SceneView view() const {
        SceneView S;
        S.bvh.nodes = nodes8; S.bvh.tris = tris; S.bvh.prim = prim;
        S.bvh.num_nodes = num_nodes; S.bvh.num_tris = (int32_t)n;
        S.bvh.inst = inst; S.bvh.top_inst = top_inst; S.bvh.num_inst = num_inst;
        S.tri_meta = meta; S.materials = materials; S.lights = lights;
        S.num_lights = num_lights; S.num_materials = num_materials;
        return S;
    }
    // keep = true (the scene is being destroyed): the queues go to the context's cache for the next scene
    void free_wave(bool keep = false) {
        WaveCache &cache = be->wave_cache();
        if (keep && pipes > 0) {
            wave_cache_release(*be, cache);
            for (int k = 0; k < pipes; ++k) { be->free(W[k].mis); W[k].mis = nullptr; cache.W[k] = W[k]; W[k] = WaveState{}; }
            cache.pool = pool; cache.pipes = pipes; cache.nq = (size_t)num_present() * (size_t)pool; cache.inst = inst != nullptr;
            pool = 0; pipes = 0;
            return;
        }
        for (int k = 0; k < pipes; ++k) {
            WaveState &w = W[k];
            be->free(w.ea); be->free(w.eb); be->free(w.ec); be->free(w.ma); be->free(w.mb); be->free(w.mc);
            be->free(w.sh_o); be->free(w.sh_d); be->free(w.sh_L); be->free(w.c); be->free(w.mis); be->free(w.hit_inst);
            w.mis = nullptr; w.hit_inst = nullptr;
        }
        pool = 0; pipes = 0;
    }
    // hit queues exist for the material types the scene HAS (an all-matte scene used to carry three unused queues,
    // 4.8 GB at the default pool); type t's block starts at entry qbase[t] of ma / mb / mc / mis / hit_inst
    int num_present() const { int c = 0; for (int t = 0; t < kNumMaterialTypes; ++t) c += (type_mask >> t) & 1u; return c > 0 ? c : 1; }
    void fill_qbase(WaveState &w, int32_t p) const {
        int slot = 0;
        for (int t = 0; t < kNumMaterialTypes; ++t) {
            w.qbase[t] = ((type_mask >> t) & 1u) ? slot * p : 0;  // (a type that is absent is never pushed)
            slot += (type_mask >> t) & 1u;
        }
    }
    void ensure_wave(int32_t p, int np) {
        if (pool == p && pipes == np) return;
        free_wave();
        const size_t nq = (size_t)num_present() * (size_t)p;
        WaveCache &cache = be->wave_cache();
        if (cache.pipes == np && cache.pool == p && cache.nq == nq && cache.inst == (inst != nullptr)) {  // the last scene's queues fit
            for (int k = 0; k < np; ++k) {
                W[k] = cache.W[k]; cache.W[k] = WaveState{};
                W[k].pool = p; W[k].mis = nullptr;
                fill_qbase(W[k], p);
            }
            cache.pool = 0; cache.pipes = 0; cache.nq = 0;
            pool = p; pipes = np;
            return;
        }
        wave_cache_release(*be, cache);  // (another shape: its memory is needed now)
        for (int k = 0; k < np; ++k) {
            WaveState &w = W[k];
            w.ea = be->template alloc<F4>(p); w.eb = be->template alloc<F4>(p); w.ec = be->template alloc<F4>(p);
            w.ma = be->template alloc<F4>(nq); w.mb = be->template alloc<F4>(nq); w.mc = be->template alloc<F4>(nq);
            w.sh_o = be->template alloc<F4>(p); w.sh_d = be->template alloc<F4>(p); w.sh_L = be->template alloc<F4>(p);
            w.c = be->template alloc<Counters>(1);
            w.pool = p;
            fill_qbase(w, p);
            w.mis = nullptr;
            w.hit_inst = inst ? be->template alloc<int32_t>(nq) : nullptr;
        }
        pool = p; pipes = np;
    }
    ~SceneT() {
        if (!be) return;
        free_wave(true);
        be->free(accum); be->free(accum_fx); be->free(own_out);
        be->free(nodes8); be->free(tris); be->free(meta); be->free(prim); be->free(leaf_of_prim);
        be->free(materials); be->free(lights); be->free(inst); be->free(top_inst); be->free((void *)deferred_light_ptr);
    }
};

// ---- builder ----
// One 8-wide tree over n primitives.  Triangles: d_vertices (may be null when tri_in is already filled —
// reference-pointer ingest), tri_in / meta_in device arrays in caller order.  Boxes (box_lo != null: the tree over the
// instances of a two-level scene): tri_in / meta_in null.  Leaf-order outputs go to caller-allocated arrays of n entries
// (tris / meta unused for boxes); the nodes come back in an array of their own (indices relative to this tree).
struct BuiltTree {
    Q4 *nodes8 = nullptr;
    int32_t num_nodes = 0;
    int levels = 0, ploc_iterations = 0;
    std::vector<int32_t> level_nodes;  // nodes of each collapse level (depth): level L is ids [sum of the levels before, + count)
    float sah_cost = 0.f;
    float bounds[6] = {0, 0, 0, 0, 0, 0};  // xmin xmax ymin ymax zmin zmax
};
struct BoxBoundsK {
    const F4 *lo, *hi; int32_t *bounds; int n;
    RTB_HD void operator()(int i) const { box_bounds_body(lo, hi, bounds, n, i); }
};
struct RebaseK {
    const Q4 *src; Q4 *dst; uint32_t node_off, tri_off; int n;
    RTB_HD void operator()(int i) const { rebase_node_body(src, dst, node_off, tri_off, n, i); }
};
struct InstBoundsK { InstBoundsArgs a; RTB_HD void operator()(int i) const { inst_bounds_body(a, i); } };
struct AddK {
    int32_t *p; int32_t v; int n;
    RTB_HD void operator()(int i) const { if (i < n) p[i] += v; }
};
// Small constants for the build's counters, written by a kernel: an upload from a host temporary has to synchronise
// the stream before it returns (be.upload), and the build used to do five of them.
struct FillI32K {
    int32_t *p; int32_t v[24]; int n;
    RTB_HD void operator()(int i) const { if (i < n) p[i] = v[i]; }
};
struct RootItemK {  // the collapse starts from the root of the binary tree, which only the device knows
    const int32_t *root_src; WorkItem *dst;
    RTB_HD void operator()(int i) const { if (i == 0) { WorkItem r; r.b2 = *root_src; r.wide = 0; dst[0] = r; } }
};
// layout of the build's one block of counters (int32 unless noted): what the host reads back comes in ONE copy at the end
enum BuildCtr {
    kCtrB2 = 0, kCtrWide = 1, kCtrTri = 2, kCtrNcl = 4, kCtrLevels = 5, kCtrLvl0 = 6 /* 6,7,8: work items of a level, rotating */,
    kCtrSah = 9 /* float */, kCtrSahTasks = 10 /* 10,11,12: large ranges of a level, rotating */,
    kCtrSahBlocks = 13 /* 13,14,15: their blocks */, kCtrBounds = 16 /* 16..21 ordered floats, 22 = bad vertex */, kCtrTail = 24 /* 24: tail rounds, 25: root */,
    kCtrSahSmall = 26 /* small ranges */,
    kCtrLevelNodes = 32 /* 32 .. 32 + kStackSize - 1: 8-wide nodes of each collapse level */, kCtrCount = 32 + kStackSize
};
// rtb_build_params.builder: the builder in the low byte, RTB_BUILDER_TREELET_PASSES(k) in bits 8..11
inline int builder_kind(const rtb_build_params &bp) { return bp.builder & 0xff; }
inline int treelet_passes(const rtb_build_params &bp) { return bp.builder >> 8 & 0xf; }
inline void check_builder(const rtb_build_params &bp) {
    const int b = builder_kind(bp);
    if ((bp.builder & ~0xfff) != 0 || (b != RTB_BUILDER_PLOC && b != RTB_BUILDER_BINNED_SAH) || treelet_passes(bp) > kTloMaxPasses)
        throw Error(RTB_ERR_INVALID, "unknown BVH builder");
}
struct SetK {
    int32_t *p; int32_t v; int n;
    RTB_HD void operator()(int i) const { if (i < n) p[i] = v; }
};
// RTB_BUILDER_BINNED_SAH: the binary tree (b2, count) over n >= 1 primitive boxes, its root in ctr[kCtrTail + 1].  Large
// ranges are split level by level: the number of a level's ranges stays on the device (three rotating counters), the
// host enqueues levels in batches and reads it once per batch; the ranges of <= kSahSmall primitives are finished
// afterwards in one launch.  With `plan`, also the inner nodes deepest first (order) and where each depth starts in that
// order (first[kSahMaxDepth + 1 - depth], -1 = no node of that depth; first[0]: deeper than kSahMaxDepth).
// The binned-SAH steps as plain loops over the bodies of rtb_build.h, for a backend whose memory the host reads
// directly (the host emulation that checks the builder without a GPU).  A backend with kernels of its own provides
// sah_level / sah_small and is dispatched to them at compile time; rtb_cuda.cu asserts that CudaBackend does, so the
// shipped library never reaches these loops.
struct SahLoops {
    // the split of one range from its bounds and bins, and the range partitioned stably: the kernels' rule
    static SahSplit split(const SahArgs &a, const SahRange &r, int32_t *bnd) {
        sah_bnd_init(bnd);
        for (int p = r.begin; p < r.end; ++p) sah_bnd_add(bnd, a.prim_lo[a.idx[p]], a.prim_hi[a.idx[p]]);
        const float scale[3] = {sah_scale(bnd, 0), sah_scale(bnd, 1), sah_scale(bnd, 2)};
        std::vector<int32_t> bins(kSahBinsWords);
        for (int k = 0; k < 3 * kSahBins; ++k) sah_bin_init(&bins[(size_t)k * kSahBinWords]);
        for (int p = r.begin; p < r.end; ++p) sah_bin_add(bins.data(), a.prim_lo[a.idx[p]], a.prim_hi[a.idx[p]], bnd, scale);
        const SahSplit s = sah_choose(bins.data(), scale, r.end - r.begin);
        std::vector<int32_t> left, right;
        for (int p = r.begin; p < r.end; ++p)
            (sah_goes_left(s, p - r.begin, a.prim_lo[a.idx[p]], a.prim_hi[a.idx[p]], bnd) ? left : right).push_back(a.idx[p]);
        if ((int)left.size() != s.nl) throw Error(RTB_ERR_INVALID, "internal: binned SAH partition disagrees with its bins");
        std::copy(left.begin(), left.end(), a.idx + r.begin);
        std::copy(right.begin(), right.end(), a.idx + r.begin + s.nl);
        return s;
    }
    static void level(const SahArgs &a) {
        *a.n_clear = 0; *a.n_blk_clear = 0;
        for (int t = 0; t < *a.n_tin; ++t) {
            SahTask &T = a.tin[t];
            const SahSplit s = split(a, T.r, T.bnd);
            SahRange ch[2];
            sah_make_node(a, T.r, T.bnd, s.nl, a.node_counter, ch);
            sah_push_child(a, ch[0]); sah_push_child(a, ch[1]);
        }
    }
    static void subtree(const SahArgs &a, const SahRange &r) {
        int32_t bnd[12];
        const SahSplit s = split(a, r, bnd);
        SahRange ch[2];
        sah_make_node(a, r, bnd, s.nl, a.node_counter, ch);
        for (const SahRange &c : ch) if (c.end - c.begin > 1) subtree(a, c);
    }
};
template <class BE, class = void> struct HasSahKernels : std::false_type {};
template <class BE>
struct HasSahKernels<BE, std::void_t<decltype(std::declval<BE &>().sah_small(std::declval<const SahArgs &>(), 0))>> : std::true_type {};
template <class BE>
void sah_level(BE &be, const SahArgs &a, int block_bound, int task_bound) {
    if constexpr (HasSahKernels<BE>::value) be.sah_level(a, block_bound, task_bound);
    else SahLoops::level(a);
}
template <class BE>
void sah_small(BE &be, const SahArgs &a, int count) {
    if constexpr (HasSahKernels<BE>::value) be.sah_small(a, count);
    else for (int i = 0; i < count; ++i) SahLoops::subtree(a, a.small[i]);
}
struct SahOrder { const int32_t *order = nullptr, *first = nullptr; };
template <class BE>
SahOrder build_binned_sah(BE &be, Temps<BE> &tmp, int n, const F4 *prim_lo, const F4 *prim_hi, B2Node *b2, int32_t *count,
                          int32_t *ctr, bool plan) {
    SahArgs a{};
    a.prim_lo = prim_lo; a.prim_hi = prim_hi; a.n = n;
    a.nodes = b2; a.count = count; a.node_counter = ctr + kCtrB2; a.n_small = ctr + kCtrSahSmall;
    a.idx = tmp.template alloc<int32_t>(n); a.idx2 = tmp.template alloc<int32_t>(n);
    a.flags = tmp.template alloc<int32_t>(n); a.scan = tmp.template alloc<int32_t>(n);
    a.depth = tmp.template alloc<int32_t>(n > 1 ? n - 1 : 1);
    const int task_bound = n / (kSahSmall + 1) + 1, block_bound = n / kSahChunk + task_bound;
    SahTask *tasks[2] = {tmp.template alloc<SahTask>(task_bound), tmp.template alloc<SahTask>(task_bound)};
    int32_t *blocks[2] = {tmp.template alloc<int32_t>(block_bound), tmp.template alloc<int32_t>(block_bound)};
    a.bins = tmp.template alloc<int32_t>((size_t)task_bound * kSahBinsWords);
    a.small = tmp.template alloc<SahRange>(n / 2 + 1);
    { SahIotaK k; k.p = a.idx; k.n = n; be.launch(n, k); }
    be.zero(a.flags, (size_t)n);
    { SahBinsInitK k; k.bins = a.bins; k.n = task_bound * 3 * kSahBins; be.launch(k.n, k); }
    // level L reads tasks[L & 1] and the counters at L % 3, writes tasks[(L + 1) & 1] and the counters at (L + 1) % 3,
    // and clears those at (L + 2) % 3 for the level after the next
    auto level_args = [&](int L) {
        SahArgs l = a;
        l.tin = tasks[(L + 2) & 1]; l.tin_c = l.tin; l.tout = tasks[(L + 3) & 1];
        l.blk_in = blocks[(L + 2) & 1]; l.blk_out = blocks[(L + 3) & 1];
        l.n_tin = ctr + kCtrSahTasks + (L + 3) % 3; l.n_tout = ctr + kCtrSahTasks + (L + 4) % 3; l.n_clear = ctr + kCtrSahTasks + (L + 5) % 3;
        l.n_blk_in = ctr + kCtrSahBlocks + (L + 3) % 3; l.n_blk_out = ctr + kCtrSahBlocks + (L + 4) % 3;
        l.n_blk_clear = ctr + kCtrSahBlocks + (L + 5) % 3;
        return l;
    };
    { SahRootK r; r.a = level_args(-1); r.root = ctr + kCtrTail + 1; be.launch(1, r); }  // (the root is level 0's one range)
    int level = 0;
    int32_t pending = n > kSahSmall ? 1 : 0;
    while (pending > 0) {
        for (int b = 0; b < 4; ++b, ++level) sah_level(be, level_args(level), block_bound, task_bound);
        be.download(&pending, ctr + kCtrSahTasks + level % 3, 1);
        // (ranges of level L are at depth >= L: the loop ends, with a tree or with this error)
        if (pending > 0 && level > kSahMaxDepth) throw Error(RTB_ERR_INVALID, "BVH too deep for the traversal stack");
    }
    int32_t n_small = 0;
    be.download(&n_small, a.n_small, 1);
    sah_small(be, a, n_small);
    { SahLeafK k; k.a = a; be.launch(n, k); }
    tmp.free(a.idx); tmp.free(a.idx2); tmp.free(a.flags); tmp.free(a.scan); tmp.free(tasks[0]); tmp.free(tasks[1]);
    tmp.free(blocks[0]); tmp.free(blocks[1]); tmp.free(a.bins); tmp.free(a.small);
    SahOrder o;
    if (!plan || n < 2) return o;
    const int n_inner = n - 1;
    uint64_t *keys = tmp.template alloc<uint64_t>(n_inner);
    int32_t *order = tmp.template alloc<int32_t>(n_inner), *first = tmp.template alloc<int32_t>(kSahMaxDepth + 2);
    { SahDepthKeyK k; k.depth = a.depth; k.keys = keys; k.vals = order; k.n_inner = n_inner; k.n = n; be.launch(n_inner, k); }
    be.sort_pairs(keys, order, n_inner);
    { SetK k; k.p = first; k.v = -1; k.n = kSahMaxDepth + 2; be.launch(k.n, k); }
    { SahGroupK k; k.keys = keys; k.first = first; k.n_inner = n_inner; be.launch(n_inner, k); }
    tmp.free(keys);
    o.order = order; o.first = first;
    return o;
}
// RTB_BUILDER_TREELET_PASSES: the treelets of one depth as a plain loop (the host emulation), or as the backend's
// kernel; rtb_cuda.cu asserts that CudaBackend has one (k_tlo_treelet, one warp per treelet)
template <class BE, class = void> struct HasTreeletKernels : std::false_type {};
template <class BE>
struct HasTreeletKernels<BE, std::void_t<decltype(std::declval<BE &>().tlo_treelets(std::declval<const TloArgs &>()))>> : std::true_type {};
template <class BE>
void tlo_treelets(BE &be, const TloArgs &a) {
    if constexpr (HasTreeletKernels<BE>::value) {
        be.tlo_treelets(a);
    } else {
        TloWork w;
        for (int i = 0; i < a.num; ++i) tlo_treelet(a, w, i, 0, 1);
    }
}
// inner nodes deepest first (order) and the host's copy of where each depth starts in it (as SahOrder::first)
struct DepthOrder { const int32_t *order = nullptr; std::vector<int32_t> first; };
// `passes` treelet passes over the binary tree (b2, count, root in *root_src) of n >= 2 primitives; with `plan`, the
// depth order of the final tree for the collapse plan.  Per pass: depths, one sort, one read-back of the per-depth
// table, then one launch per depth.
template <class BE>
DepthOrder run_treelet_passes(BE &be, Temps<BE> &tmp, int n, B2Node *b2, int32_t *count, const int32_t *root_src, int passes, bool plan) {
    const int n_inner = n - 1;
    TloArgs a{};
    a.nodes = b2; a.count = count; a.root = root_src; a.n = n;
    a.parent = tmp.template alloc<int32_t>((size_t)2 * n - 1);
    a.depth = tmp.template alloc<int32_t>(n_inner);
    uint64_t *keys = tmp.template alloc<uint64_t>(n_inner);
    int32_t *order = tmp.template alloc<int32_t>(n_inner), *first = tmp.template alloc<int32_t>(kSahMaxDepth + 2);
    a.order = order;
    { TloParentK k; k.a = a; be.launch(n_inner, k); }
    DepthOrder o;
    o.first.resize(kSahMaxDepth + 2);
    auto sort_by_depth = [&]() {
        { TloDepthK k; k.a = a; be.launch(n_inner, k); }
        { SahDepthKeyK k; k.depth = a.depth; k.keys = keys; k.vals = order; k.n_inner = n_inner; k.n = n; be.launch(n_inner, k); }
        be.sort_pairs(keys, order, n_inner);
        { SetK k; k.p = first; k.v = -1; k.n = kSahMaxDepth + 2; be.launch(k.n, k); }
        { SahGroupK k; k.keys = keys; k.first = first; k.n_inner = n_inner; be.launch(n_inner, k); }
        be.download(o.first.data(), first, o.first.size());
        if (o.first[0] >= 0) throw Error(RTB_ERR_INVALID, "BVH too deep for the traversal stack");
    };
    for (int p = 0; p < passes; ++p) {
        sort_by_depth();
        a.gamma = kTloGamma << p;
        for (int k = 1; k <= kSahMaxDepth + 1; ++k) {  // deepest first
            if (o.first[(size_t)k] < 0) continue;
            int end = n_inner;
            for (int j = k + 1; j <= kSahMaxDepth + 1; ++j) if (o.first[(size_t)j] >= 0) { end = o.first[(size_t)j]; break; }
            a.first = o.first[(size_t)k]; a.num = end - a.first;
            tlo_treelets(be, a);
        }
    }
    if (plan) { sort_by_depth(); o.order = order; }
    tmp.free(a.parent); tmp.free(a.depth); tmp.free(keys); tmp.free(first);
    if (!plan) tmp.free(order);
    return o;
}
constexpr int kMaxPlocLog = 1 << 16;
template <class BE>
BuiltTree build_tree(BE &be, int n, const float *d_vertices, Tri48 *tri_in, TriMeta *meta_in, const F4 *box_lo, const F4 *box_hi,
                     const rtb_build_params &bp, int max_leaf, Tri48 *tris_out, TriMeta *meta_out, int32_t *prim_out,
                     int32_t *leaf_of_prim) {
    BuiltTree out;
    Temps<BE> tmp(be);
    // 1. per-triangle records, bounds
    F4 *prim_lo = tmp.template alloc<F4>(n), *prim_hi = tmp.template alloc<F4>(n);
    int32_t *ctr = tmp.template alloc<int32_t>(kCtrCount);
    int32_t *bounds = ctr + kCtrBounds;  // [6] = "a vertex is not finite / out of range"
    float *sah = (float *)(ctr + kCtrSah);
    {
        FillI32K f; f.p = ctr; f.n = kCtrCount;
        for (int k = 0; k < 24; ++k) f.v[k] = 0;
        f.n = 24;  // (the tail's words are written by its kernel)
        f.v[kCtrB2] = n; f.v[kCtrWide] = 1; f.v[kCtrNcl] = n; f.v[kCtrLvl0] = 1;
        for (int k = 0; k < 3; ++k) { f.v[kCtrBounds + k] = float_to_ordered(FLT_MAX); f.v[kCtrBounds + 3 + k] = float_to_ordered(-FLT_MAX); }
        be.launch(f.n, f);
        if (box_lo) {
            be.copy(prim_lo, box_lo, (size_t)n); be.copy(prim_hi, box_hi, (size_t)n);
            BoxBoundsK k; k.lo = box_lo; k.hi = box_hi; k.bounds = bounds; k.n = n;
            be.launch(n, k);
        } else {
            PrimSetupK k; k.a.vertices = d_vertices; k.a.tri_in = tri_in; k.a.prim_lo = prim_lo; k.a.prim_hi = prim_hi;
            k.a.scene_bounds = bounds; k.a.bad = bounds + 6; k.a.n = n;
            be.prim_setup(k.a);
            int32_t bad = 0;
            be.download(&bad, bounds + 6, 1);  // (kept: a scene with a non-finite vertex must not reach the sort and the PLOC rounds)
            if (bad) {
                throw Error(RTB_ERR_INVALID, "a triangle vertex is not finite or beyond 2^100: the scene cannot be built");
            }
        }
    }
    const int n_b2 = 2 * n - 1;
    B2Node *b2 = tmp.template alloc<B2Node>(n_b2);
    int32_t *count = tmp.template alloc<int32_t>(n_b2);
    const bool want_plan = bp.collapse == RTB_COLLAPSE_SAH_OPTIMAL && n > max_leaf;
    const int passes = n >= 2 ? treelet_passes(bp) : 0;
    float *plan_cost = nullptr; uint8_t *plan = nullptr;
    // 4. collapse plan, one launch per depth, deepest first (a node's children are deeper): first[] as SahOrder::first
    auto plan_by_depth = [&](const int32_t *order, const std::vector<int32_t> &first) {
        if (first[0] >= 0) throw Error(RTB_ERR_INVALID, "BVH too deep for the traversal stack");
        plan_cost = tmp.template alloc<float>((size_t)n_b2 * 7);
        plan = tmp.template alloc<uint8_t>((size_t)n_b2 * 8);
        for (int k = 1; k <= kSahMaxDepth + 1; ++k) {
            if (first[(size_t)k] < 0) continue;
            int end = n - 1;
            for (int j = k + 1; j <= kSahMaxDepth + 1; ++j) if (first[(size_t)j] >= 0) { end = first[(size_t)j]; break; }
            PlanK p; p.a.nodes = b2; p.a.count = count; p.a.cost = plan_cost; p.a.plan = plan;
            p.a.first = first[(size_t)k]; p.a.n = end - first[(size_t)k]; p.a.max_leaf = max_leaf; p.a.order = order;
            be.launch(p.a.n, p);
        }
    };
    const int32_t *root_src = ctr + kCtrTail + 1;
    int rounds = 0;
    bool tail = false;
    std::vector<int32_t> hlog, htail;
    int32_t *log = nullptr;
    auto read_logs = [&]() {
        const int logged = rounds < kMaxPlocLog ? rounds : kMaxPlocLog;
        hlog.resize((size_t)logged + 1);
        if (logged) be.download(hlog.data(), log, (size_t)logged);
        be.download(&hlog[(size_t)logged], ctr + kCtrNcl, 1);  // count after the last round of the batches
        if (tail) {
            int32_t h2[2];
            be.download(h2, ctr + kCtrTail, 2);
            if (h2[0] < 0) throw Error(RTB_ERR_INVALID, "internal: a PLOC round merged nothing");
            htail.resize((size_t)h2[0]);
            if (h2[0]) be.download(htail.data(), be.ploc_tail_counts(), (size_t)h2[0]);
        }
    };
    if (builder_kind(bp) == RTB_BUILDER_PLOC) {
        const int radius = bp.ploc_radius > 0 ? bp.ploc_radius : 16;
        // 2. Morton codes + sort
        uint64_t *keys = tmp.template alloc<uint64_t>(n);
        int32_t *sorted = tmp.template alloc<int32_t>(n);
        {
            MortonK k; k.a.prim_lo = prim_lo; k.a.prim_hi = prim_hi; k.a.scene_bounds = bounds; k.a.keys = keys; k.a.vals = sorted; k.a.n = n;
            be.launch(n, k);
            be.sort_pairs(keys, sorted, n);
        }
        // 3. PLOC.  The cluster count stays on the device (ctr[kCtrNcl]); the host enqueues a batch of rounds against an
        // upper bound of it and reads the count back once per batch (round 1: after every round).
        int32_t *ca = tmp.template alloc<int32_t>(n), *cb = tmp.template alloc<int32_t>(n), *nn = tmp.template alloc<int32_t>(n);
        log = tmp.template alloc<int32_t>(kMaxPlocLog);
        {
            PlocLeafK k; k.lo = prim_lo; k.hi = prim_hi; k.sorted = sorted; k.nodes = b2; k.count = count; k.clusters = ca; k.n = n;
            be.launch(n, k);
        }
        int bound = n;
        while (bound > 1) {
            PlocArgs a; a.nodes = b2; a.count = count; a.cin = ca; a.cout = cb; a.nn = nn; a.node_counter = ctr + kCtrB2; a.ncl = bound; a.radius = radius;
            a.ncl_dev = ctr + kCtrNcl; a.log = log; a.round = rounds;
            // the last rounds handle a few hundred clusters each and are pure launch latency (S1: 28 of 46 rounds): once
            // the clusters fit one thread block, one launch runs all the remaining rounds in shared memory
            if (be.ploc_tail(a, n, ctr + kCtrTail)) { tail = true; break; }
            // rounds of this batch: the count shrinks by about a fifth per round (S1 and S2 alike); go most of the way to
            // the tail's size, but not far on a large bound — every launch of the batch still covers the whole bound
            const double to_tail = std::log((double)bound / 1024.0) / 0.235;
            int batch = (int)(0.8 * to_tail);
            const int cap = bound > (1 << 21) ? 4 : (bound > (1 << 18) ? 8 : 16);
            if (batch > cap) batch = cap;
            if (batch < 1) batch = 1;
            for (int r = 0; r < batch; ++r) {
                // (a scene of identical triangles merges ONE pair per round: n - 1 rounds.  The per-round counts are a
                // statistic, and the SAH-optimal plan's launch schedule: beyond the log's size only the plan needs them)
                if (rounds >= kMaxPlocLog) {
                    if (want_plan) throw Error(RTB_ERR_INVALID, "RTB_COLLAPSE_SAH_OPTIMAL: too many PLOC rounds (degenerate scene)");
                    a.log = nullptr;
                }
                a.round = rounds;
                be.ploc_nn(a);
                PlocMergeK k2; k2.a = a; k2.n_leaves = n; be.launch(bound, k2);
                be.compact_nonneg(cb, ca, bound, ctr + kCtrNcl);
                ++rounds;
            }
            int32_t now = 0;
            be.download(&now, ctr + kCtrNcl, 1);
            if (now >= bound) throw Error(RTB_ERR_INVALID, "internal: a PLOC round merged nothing");  // (cannot happen with finite boxes: the lowest-area pair is mutual)
            bound = now;
        }
        if (!tail) root_src = ca;
        tmp.free(prim_lo); tmp.free(prim_hi); tmp.free(keys); tmp.free(sorted); tmp.free(nn);
        // 4. collapse plan: bottom-up over the binary tree, one launch per PLOC round (a round's nodes only have older
        // children; after treelet passes they need not be, and the plan goes by depth below)
        if (want_plan) read_logs();
        if (want_plan && !passes) {
            plan_cost = tmp.template alloc<float>((size_t)n_b2 * 7);
            plan = tmp.template alloc<uint8_t>((size_t)n_b2 * 8);
            int next_id = n;
            auto plan_round = [&](int made) {
                if (made > 0) {
                    PlanK k; k.a.nodes = b2; k.a.count = count; k.a.cost = plan_cost; k.a.plan = plan;
                    k.a.first = next_id; k.a.n = made; k.a.max_leaf = max_leaf; k.a.order = nullptr;
                    be.launch(made, k);
                }
                next_id += made;
            };
            for (size_t r = 0; r + 1 < hlog.size(); ++r) plan_round(hlog[r] - hlog[r + 1]);
            for (int32_t c : htail) plan_round(c);
        }
    } else {
        // 2'-3'. binned SAH, top down; the root goes to ctr[kCtrTail + 1]
        const SahOrder so = build_binned_sah(be, tmp, n, prim_lo, prim_hi, b2, count, ctr, want_plan && !passes);
        tmp.free(prim_lo); tmp.free(prim_hi);
        if (want_plan && !passes) {
            std::vector<int32_t> first(kSahMaxDepth + 2);
            be.download(first.data(), so.first, first.size());  // (the one read-back of the per-depth counts)
            plan_by_depth(so.order, first);
        }
    }
    // 3.5. treelet restructuring; the plan then goes by depth, whichever the builder
    if (passes) {
        const DepthOrder d = run_treelet_passes(be, tmp, n, b2, count, root_src, passes, want_plan);
        if (want_plan) plan_by_depth(d.order, d.first);
    }
    // 5. collapse to the 8-wide compressed tree, level by level; the number of work items of a level stays on the
    // device (three rotating counters: read, written, cleared), the host reads it once per batch of levels
    const int max_nodes = n > 1 ? n : 1;
    Q4 *nodes_tmp = tmp.template alloc<Q4>((size_t)max_nodes * kNodeWords);
    WorkItem *wa = tmp.template alloc<WorkItem>(max_nodes), *wb = tmp.template alloc<WorkItem>(max_nodes);
    int32_t *gather = tmp.template alloc<int32_t>(n);
    CollapseArgs ga{};
    {
        RootItemK r; r.root_src = root_src; r.dst = wa;
        be.launch(1, r);
    }
    int level = 0;
    while (true) {
        const int batch = level == 0 ? 8 : 4;
        for (int b = 0; b < batch; ++b, ++level) {
            CollapseK k;
            k.a.nodes = b2; k.a.count = count; k.a.plan = plan; k.a.tri_in = tri_in; k.a.meta_in = meta_in;
            k.a.nodes8 = nodes_tmp; k.a.tris_out = tris_out; k.a.meta_out = meta_out; k.a.prim_out = prim_out;
            k.a.leaf_of_prim = leaf_of_prim; k.a.node_counter = ctr + kCtrWide; k.a.tri_counter = ctr + kCtrTri;
            k.a.work_in = wa; k.a.n_in = 0; k.a.n_in_dev = ctr + kCtrLvl0 + level % 3; k.a.work_out = wb;
            k.a.n_out = ctr + kCtrLvl0 + (level + 1) % 3; k.a.sah = sah; k.a.max_leaf = max_leaf; k.a.gather = gather;
            k.a.level_nodes = level < kStackSize ? ctr + kCtrLevelNodes + level : nullptr;  // (deeper trees are rejected)
            ga = k.a;
            be.collapse_level(k, max_nodes, ctr + kCtrLvl0 + (level + 2) % 3, ctr + kCtrLevels);
            WorkItem *t = wa; wa = wb; wb = t;
        }
        int32_t pending = 0;
        be.download(&pending, ctr + kCtrLvl0 + level % 3, 1);
        if (pending == 0) break;
        if (level > 4 * kStackSize) throw Error(RTB_ERR_INVALID, "BVH too deep for the traversal stack");
    }
    { GatherK g; g.a = ga; g.n = n; be.launch(n, g); }  // triangles of the leaf children, one thread per leaf child
    int32_t c[kCtrCount];
    be.download(c, ctr, kCtrCount);
    out.num_nodes = c[kCtrWide];
    out.levels = c[kCtrLevels];
    out.level_nodes.assign(c + kCtrLevelNodes, c + kCtrLevelNodes + (out.levels < kStackSize ? out.levels : kStackSize));
    if (c[kCtrTri] != n) throw Error(RTB_ERR_INVALID, "internal: collapse lost triangles");
    out.nodes8 = be.template alloc<Q4>((size_t)out.num_nodes * kNodeWords);
    be.copy(out.nodes8, nodes_tmp, (size_t)out.num_nodes * kNodeWords);
    if (builder_kind(bp) == RTB_BUILDER_PLOC && !want_plan) read_logs();
    int iters = rounds > kMaxPlocLog ? rounds - kMaxPlocLog : 0;  // (rounds beyond the log are counted, not examined)
    for (size_t r = 0; r + 1 < hlog.size(); ++r) if (hlog[r] > hlog[r + 1]) ++iters;
    out.ploc_iterations = iters + (int)htail.size();
    float sah_h;
    memcpy(&sah_h, &c[kCtrSah], sizeof sah_h);
    float lo[3], hi[3];
    for (int k = 0; k < 3; ++k) { lo[k] = ordered_to_float(c[kCtrBounds + k]); hi[k] = ordered_to_float(c[kCtrBounds + 3 + k]); }
    const float root_area = half_area(hi[0] - lo[0], hi[1] - lo[1], hi[2] - lo[2]);
    out.sah_cost = root_area > 0.f ? sah_h / root_area : 0.f;
    for (int k = 0; k < 3; ++k) { out.bounds[2 * k] = lo[k]; out.bounds[2 * k + 1] = hi[k]; }
    return out;  // (Temps releases what is still held, on this path and on every throw)
}

// tri_in / meta_in / light_tri are device arrays in caller order; vertices may
// be null when tri_in is already filled (reference-pointer ingest).
template <class BE>
void build_bvh(BE &be, SceneT<BE> &sc, const float *d_vertices, Tri48 *tri_in, TriMeta *meta_in,
               const int64_t *d_light_tri, const rtb_build_params &bp) {
    const int64_t n64 = sc.n;
    if (n64 > 0x3fffffff) throw Error(RTB_ERR_INVALID, "too many triangles (max 2^30-1)");
    const int n = (int)n64;
    check_builder(bp);
    const int max_leaf = bp.max_leaf_tris >= 1 && bp.max_leaf_tris <= 3 ? bp.max_leaf_tris : 3;
    auto t0 = be.now();
    sc.stats = rtb_bvh_stats{};
    sc.stats.num_triangles = n;
    sc.n_flat = n;
    sc.tris = (F4 *)be.template alloc<Tri48>(n > 0 ? n : 1);
    sc.meta = be.template alloc<TriMeta>(n > 0 ? n : 1);
    sc.prim = be.template alloc<int32_t>(n > 0 ? n : 1);
    sc.leaf_of_prim = be.template alloc<int32_t>(n > 0 ? n : 1);
    if (n == 0) {  // empty scene: one node with eight empty slots
        std::vector<Q4> root(kNodeWords);
        memset(root.data(), 0, sizeof(Q4) * kNodeWords);
        root[2].x = root[2].y = root[2].z = root[2].w = 0xffffffffu;  // qlo = 255 > qhi = 0
        root[3].x = root[3].y = 0xffffffffu;
        root[0].w = 127u | (127u << 8) | (127u << 16);
        sc.nodes8 = be.template alloc<Q4>(kNodeWords);
        be.upload(sc.nodes8, root.data(), kNodeWords);
        sc.num_nodes = 1;
        sc.stats.num_nodes = 1;
        sc.stats.node_bytes = 80;
        return;
    }
    const BuiltTree bt = build_tree(be, n, d_vertices, tri_in, meta_in, nullptr, nullptr, bp, max_leaf, (Tri48 *)sc.tris, sc.meta, sc.prim,
                                    sc.leaf_of_prim);
    sc.nodes8 = bt.nodes8;
    sc.num_nodes = bt.num_nodes;
    if (bt.levels >= kStackSize) throw Error(RTB_ERR_INVALID, "BVH too deep for the traversal stack");
    sc.bp = bp;
    sc.tree_levels.assign(1, bt.level_nodes);
    sc.tree_first.assign(1, 0);
    if (sc.num_lights > 0) {
        LightFixK k; k.lights = sc.lights; k.light_tri = d_light_tri; k.leaf_of_prim = sc.leaf_of_prim; k.n = sc.num_lights;
        be.launch(sc.num_lights, k);
    }
    sc.stats.ploc_iterations = bt.ploc_iterations;
    sc.stats.num_bvh2_nodes = 2 * (int64_t)n - 1;
    sc.stats.sah_cost = bt.sah_cost;
    sc.stats.num_nodes = sc.num_nodes;
    sc.stats.node_bytes = (int64_t)sc.num_nodes * 80;
    sc.stats.triangle_bytes = (int64_t)n * 48;
    sc.stats.collapse_levels = bt.levels;
    for (int k = 0; k < 6; ++k) sc.stats.scene_bounds[k] = bt.bounds[k];
    sc.stats.build_ms = be.elapsed_ms(t0, be.now());
}

template <class BE>
SceneT<BE> *scene_from_desc(BE &be, const rtb_scene_desc &d, const rtb_build_params &bp) {
    if (d.num_triangles < 0 || (d.num_triangles > 0 && (!d.vertices || !d.material_ids)) || d.num_materials <= 0 || !d.materials)
        throw Error(RTB_ERR_INVALID, "rtb_scene_create: incomplete scene description");
    if (d.num_lights > 0 && !d.lights) throw Error(RTB_ERR_INVALID, "rtb_scene_create: lights missing");
    const int64_t n = d.num_triangles;
    for (int i = 0; i < d.num_materials; ++i)
        if (d.materials[i].type < 0 || d.materials[i].type >= kNumMaterialTypes) throw Error(RTB_ERR_INVALID, "unknown material type");
    if (n > 0x3fffffff) throw Error(RTB_ERR_INVALID, "too many triangles (max 2^30-1)");
    std::vector<LightDev> lights((size_t)d.num_lights);
    std::vector<int64_t> light_tri((size_t)d.num_lights);
    for (int i = 0; i < d.num_lights; ++i) {
        const rtb_light &l = d.lights[i];
        if (l.type == RTB_AREA_LIGHT && (l.triangle < 0 || l.triangle >= n)) throw Error(RTB_ERR_INVALID, "area light triangle out of range");
        LightDev &o = lights[(size_t)i];
        o.type = l.type; o.px = l.pos[0]; o.py = l.pos[1]; o.pz = l.pos[2]; o.tri = -1;
        o.Lx = l.L[0]; o.Ly = l.L[1]; o.Lz = l.L[2];
        light_tri[(size_t)i] = l.type == RTB_AREA_LIGHT ? l.triangle : 0;
    }
    SceneT<BE> *sc = new SceneT<BE>();
    try {
        sc->be = &be;
        sc->n = n;
        sc->num_materials = d.num_materials;
        sc->num_lights = d.num_lights;
        sc->materials = be.template alloc<rtb_material>(d.num_materials);
        be.upload(sc->materials, d.materials, d.num_materials);
        for (int i = 0; i < d.num_materials; ++i) sc->type_mask |= 1u << d.materials[i].type;
        sc->lights = be.template alloc<LightDev>(d.num_lights > 0 ? d.num_lights : 1);
        Temps<BE> tmp(be);
        int64_t *d_light_tri = tmp.template alloc<int64_t>(d.num_lights > 0 ? d.num_lights : 1);
        if (d.num_lights) { be.upload(sc->lights, lights.data(), d.num_lights); be.upload(d_light_tri, light_tri.data(), d.num_lights); }
        float *d_vertices = tmp.template alloc<float>(n > 0 ? 9 * (size_t)n : 1);
        Tri48 *tri_in = tmp.template alloc<Tri48>(n > 0 ? n : 1);
        TriMeta *meta_in = tmp.template alloc<TriMeta>(n > 0 ? n : 1);
        if (n) {
            // the per-triangle ids go up as they are and become TriMeta records on the device, where they are also range
            // checked (a 10 M-triangle description used to spend 30 ms of host time in that loop)
            int32_t *d_mat = tmp.template alloc<int32_t>((size_t)n), *d_light = d.light_ids ? tmp.template alloc<int32_t>((size_t)n) : nullptr;
            int32_t *bad = tmp.template alloc<int32_t>(1);
            be.zero(bad, 1);
            be.upload(d_vertices, d.vertices, 9 * (size_t)n);
            be.upload(d_mat, d.material_ids, (size_t)n);
            if (d_light) be.upload(d_light, d.light_ids, (size_t)n);
            MetaK k; k.mat = d_mat; k.light = d_light; k.materials = sc->materials; k.out = meta_in; k.bad = bad;
            k.n = (int)n; k.num_mats = d.num_materials; k.num_lights = d.num_lights;
            be.launch((int)n, k);
            int32_t b = 0;
            be.download(&b, bad, 1);
            if (b == 2) throw Error(RTB_ERR_INVALID, "material id out of range");
            if (b == 1) throw Error(RTB_ERR_INVALID, "light id out of range");
            tmp.free(d_mat); tmp.free(d_light); tmp.free(bad);
        }
        build_bvh(be, *sc, d_vertices, tri_in, meta_in, d_light_tri, bp);
    } catch (...) {
        delete sc;
        throw;
    }
    return sc;
}

// Bvh::Bvh(triangles, primitives) + Scene{bvh,num_lights,d_lights} through the
// reference's own device arrays (bvh.cuh:30, scene.cuh:4-8, main.cu:141-156)
// lights in the reference's layout (light.cuh:9-28: type@0 pos@4 d_triangle@16 L@24, 40 bytes) -> LightDev + the index
// of each area light's triangle in the caller's triangle array
template <class BE>
void ingest_ref_lights(BE &be, const void *d_lights, int num_lights, const void *d_tris, int64_t n, std::vector<LightDev> &lights,
                       std::vector<int64_t> &light_tri) {
    std::vector<char> hl(40 * (size_t)(num_lights > 0 ? num_lights : 1));
    if (num_lights) be.download(hl.data(), (const char *)d_lights, 40 * (size_t)num_lights);
    lights.assign((size_t)(num_lights > 0 ? num_lights : 1), LightDev{});
    light_tri.assign((size_t)(num_lights > 0 ? num_lights : 1), 0);
    for (int i = 0; i < num_lights; ++i) {
        const char *p = hl.data() + 40 * (size_t)i;
        LightDev &o = lights[(size_t)i];
        memcpy(&o.type, p, 4); memcpy(&o.px, p + 4, 12); memcpy(&o.Lx, p + 24, 12);
        o.tri = -1;
        if (o.type != RTB_POINT_LIGHT && o.type != RTB_AREA_LIGHT) throw Error(RTB_ERR_INVALID, "unknown light type");
        const void *tp; memcpy(&tp, p + 16, 8);
        if (o.type == RTB_AREA_LIGHT) {
            const long long off = (const char *)tp - (const char *)d_tris;
            if (off < 0 || off % 48 != 0 || off / 48 >= n) throw Error(RTB_ERR_INVALID, "area light: d_triangle does not point into the triangle array");
            light_tri[(size_t)i] = off / 48;
        }
    }
}
// Bvh::Bvh(triangles, primitives) + Scene{bvh,num_lights,d_lights} through the
// reference's own device arrays (bvh.cuh:30, scene.cuh:4-8, main.cu:141-156).
// num_lights < 0: the light array is not known yet (the reference fills `Scene` after constructing `Bvh`); the tree
// is built now and attach_lights() resolves the primitives' light pointers later.
template <class BE>
SceneT<BE> *scene_from_primitives(BE &be, const void *h_prims, int64_t n, const void *d_tris, const void *d_mats,
                                  int num_mats, const void *d_lights, int num_lights, const rtb_build_params &bp) {
    const bool deferred = num_lights < 0;
    if (deferred) num_lights = 0;
    if (n < 0 || n > 0x3fffffff || (n > 0 && (!h_prims || !d_tris)) || !d_mats || num_mats <= 0 || (num_lights > 0 && !d_lights))
        throw Error(RTB_ERR_INVALID, "rtb_scene_create_from_primitives: bad arguments");
    SceneT<BE> *sc = new SceneT<BE>();
    try {
        sc->be = &be;
        sc->n = n;
        sc->num_materials = num_mats;
        sc->num_lights = num_lights;
        sc->ref_tri_base = (const char *)d_tris;
        sc->materials = be.template alloc<rtb_material>(num_mats);
        be.copy((char *)sc->materials, (const char *)d_mats, 20 * (size_t)num_mats);  // same 20-byte layout
        {
            std::vector<rtb_material> hm((size_t)num_mats);
            be.download(hm.data(), sc->materials, (size_t)num_mats);
            for (int i = 0; i < num_mats; ++i) {
                if (hm[(size_t)i].type < 0 || hm[(size_t)i].type >= kNumMaterialTypes) throw Error(RTB_ERR_INVALID, "unknown material type");
                sc->type_mask |= 1u << hm[(size_t)i].type;
            }
        }
        std::vector<LightDev> lights;
        std::vector<int64_t> light_tri;
        ingest_ref_lights(be, d_lights, num_lights, d_tris, n, lights, light_tri);
        sc->lights = be.template alloc<LightDev>(lights.size());
        DeviceBuf<BE, int64_t> d_light_tri(be, light_tri.size());
        be.upload(sc->lights, lights.data(), lights.size());
        be.upload(d_light_tri.p, light_tri.data(), light_tri.size());
        DeviceBuf<BE, RefPrimitive> d_prims(be, (size_t)(n > 0 ? n : 1));
        DeviceBuf<BE, Tri48> tri_in(be, (size_t)(n > 0 ? n : 1));
        DeviceBuf<BE, TriMeta> meta_in(be, (size_t)(n > 0 ? n : 1));
        DeviceBuf<BE, int32_t> bad(be, 1);
        be.zero(bad.p, 1);
        if (deferred) sc->deferred_light_ptr = (const void **)be.template alloc<const void *>((size_t)(n > 0 ? n : 1));
        if (n) {
            be.upload(d_prims.p, (const RefPrimitive *)h_prims, (size_t)n);
            IngestK k; k.prims = d_prims.p; k.tri_base = (const char *)d_tris; k.mat_base = (const char *)d_mats;
            k.light_base = (const char *)d_lights; k.materials = sc->materials; k.tri_in = tri_in.p; k.meta_in = meta_in.p;
            k.light_tri = d_light_tri.p; k.light_ptr = sc->deferred_light_ptr; k.bad = bad.p; k.n = (int)n; k.num_mats = num_mats; k.num_lights = num_lights;
            be.launch((int)n, k);
            int32_t b = 0;
            be.download(&b, bad.p, 1);
            if (b == 1) throw Error(RTB_ERR_INVALID, "a Primitive's d_mat does not point into the material array");
            if (b == 2) throw Error(RTB_ERR_INVALID, "a Primitive's d_area_light does not point into the light array");
        }
        build_bvh(be, *sc, nullptr, tri_in.p, meta_in.p, d_light_tri.p, bp);
        be.sync();
    } catch (...) {
        delete sc;
        throw;
    }
    return sc;
}
template <class BE>
void attach_lights(BE &be, SceneT<BE> &sc, const void *d_lights, int num_lights) {
    if (!sc.deferred_light_ptr) throw Error(RTB_ERR_INVALID, "rtb_scene_attach_lights: the scene was not created with num_lights < 0");
    if (num_lights < 0 || (num_lights > 0 && !d_lights)) throw Error(RTB_ERR_INVALID, "rtb_scene_attach_lights: bad arguments");
    std::vector<LightDev> lights;
    std::vector<int64_t> light_tri;
    ingest_ref_lights(be, d_lights, num_lights, sc.ref_tri_base, sc.n, lights, light_tri);
    be.free(sc.lights);
    sc.lights = nullptr;
    sc.lights = be.template alloc<LightDev>(lights.size());
    sc.num_lights = num_lights;
    DeviceBuf<BE, int64_t> d_light_tri(be, light_tri.size());
    DeviceBuf<BE, int32_t> bad(be, 1);
    be.zero(bad.p, 1);
    be.upload(sc.lights, lights.data(), lights.size());
    be.upload(d_light_tri.p, light_tri.data(), light_tri.size());
    if (sc.n) {
        AttachLightsK k; k.light_ptr = sc.deferred_light_ptr; k.light_base = (const char *)d_lights; k.leaf_of_prim = sc.leaf_of_prim;
        k.meta = sc.meta; k.bad = bad.p; k.n = (int)sc.n; k.num_lights = num_lights;
        be.launch((int)sc.n, k);
        int32_t b = 0;
        be.download(&b, bad.p, 1);
        if (b) throw Error(RTB_ERR_INVALID, "a Primitive's d_area_light does not point into the light array");
    }
    if (num_lights > 0) {
        LightFixK k; k.lights = sc.lights; k.light_tri = d_light_tri.p; k.leaf_of_prim = sc.leaf_of_prim; k.n = num_lights;
        be.launch(num_lights, k);
    }
    be.sync();
}

// ---- a built scene copied to another GPU (rtb_multi_scene_replicate) ----
// SURVEY 7.3-6: "build once and broadcast, or build concurrently on all GPUs".  The copy moves the finished arrays
// (8-wide nodes, leaf-order triangles, meta, index maps, materials, lights, instance records) device to device; nothing
// is rebuilt, so every GPU traverses the very same tree.
template <class BE>
SceneT<BE> *clone_scene(BE &dst, BE &src_be, const SceneT<BE> &src) {
    SceneT<BE> *sc = new SceneT<BE>();
    try {
        sc->be = &dst;
        sc->n = src.n; sc->n_flat = src.n_flat; sc->num_inst = src.num_inst;
        sc->num_materials = src.num_materials; sc->num_lights = src.num_lights; sc->num_nodes = src.num_nodes;
        sc->type_mask = src.type_mask; sc->stats = src.stats;
        const size_t n = (size_t)(src.n > 0 ? src.n : 1);
        auto dup = [&](auto *&d, const auto *s_, size_t count) {
            using T = typename std::remove_cv<typename std::remove_pointer<decltype(s_)>::type>::type;
            d = dst.template alloc<T>(count);
            dst.copy_from(src_be, d, s_, count);
        };
        dup(sc->nodes8, src.nodes8, (size_t)src.num_nodes * kNodeWords);
        dup(sc->tris, src.tris, 3 * n);
        dup(sc->meta, src.meta, n);
        dup(sc->prim, src.prim, n);
        dup(sc->leaf_of_prim, src.leaf_of_prim, n);
        dup(sc->materials, src.materials, (size_t)src.num_materials);
        dup(sc->lights, src.lights, (size_t)(src.num_lights > 0 ? src.num_lights : 1));
        if (src.inst) {
            dup(sc->inst, src.inst, (size_t)src.num_inst * kInstWords);
            dup(sc->top_inst, src.top_inst, (size_t)src.num_inst);
        }
        dst.sync();
    } catch (...) {
        delete sc;
        throw;
    }
    return sc;
}

// contiguous, balanced split of `total` samples over `world` shards -> (first, count) of shard `rank`
inline void shard_samples(int total, int rank, int world, int &first, int &count) {
    const int base = total / world, rem = total % world;
    count = base + (rank < rem ? 1 : 0);
    first = rank * base + (rank < rem ? rank : rem);
}

// ---- two-level scenes (rtb_scene_create_instanced) ----
// One tree per mesh (object space), one over the instances' world boxes; all nodes in one array: the top tree first
// (traversal starts at node 0), then the meshes' trees with their indices rebased.  Triangles, meta, prim and
// leaf_of_prim keep mesh m in [mesh_first[m], mesh_first[m+1]) — leaf order permutes within a mesh only.
inline bool invert3x4(const float *m, double *inv) {  // rows of [A | b] -> rows of [A^-1 | -A^-1 b]
    const double a = m[0], b = m[1], c = m[2], d = m[4], e = m[5], f = m[6], g = m[8], h = m[9], i = m[10];
    const double det = a * (e * i - f * h) - b * (d * i - f * g) + c * (d * h - e * g);
    if (!(fabs(det) > 0.0) || !std::isfinite(det)) return false;
    const double r = 1.0 / det;
    const double A[9] = {(e * i - f * h) * r, (c * h - b * i) * r, (b * f - c * e) * r, (f * g - d * i) * r, (a * i - c * g) * r,
                         (c * d - a * f) * r, (d * h - e * g) * r, (b * g - a * h) * r, (a * e - b * d) * r};
    for (int k = 0; k < 3; ++k) {
        inv[4 * k] = A[3 * k]; inv[4 * k + 1] = A[3 * k + 1]; inv[4 * k + 2] = A[3 * k + 2];
        inv[4 * k + 3] = -(A[3 * k] * m[3] + A[3 * k + 1] * m[7] + A[3 * k + 2] * m[11]);
    }
    return true;
}
inline bool is_identity3x4(const float *m) {
    static const float id[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
    for (int k = 0; k < 12; ++k) if (m[k] != id[k]) return false;
    return true;
}
// mesh, material and transform of one instance; its world -> object matrix into inv
inline void check_instance(const rtb_instance &in, int num_meshes, int num_materials, double *inv) {
    if (in.mesh < 0 || in.mesh >= num_meshes) throw Error(RTB_ERR_INVALID, "instance: mesh out of range");
    if (in.material < -1 || in.material >= num_materials) throw Error(RTB_ERR_INVALID, "instance: material out of range");
    for (int k = 0; k < 12; ++k) if (!std::isfinite(in.xform[k])) throw Error(RTB_ERR_INVALID, "instance: transform not finite");
    if (!invert3x4(in.xform, inv)) throw Error(RTB_ERR_INVALID, "instance: transform not invertible");
}
// The tree over the instances and everything that depends on it, for the instances in sc.instances (checked, with their
// world -> object matrices in `inverse`): the instances' world boxes from the triangles `tris` (leaf order), the top
// tree, the stack-depth check, one node array (the top tree, then the mesh trees of `mesh_nodes`, whose indices are
// rebased to a top tree of `mesh_base` nodes, re-rebased to the new one) and the instance records.  Everything is built
// before anything of the scene is replaced; the scene's old arrays are freed after.  Scene creation and
// rtb_scene_set_instances both come here.
template <class BE>
void install_top(BE &be, SceneT<BE> &sc, const std::vector<double> &inverse, const Q4 *mesh_nodes, int32_t mesh_base,
                 int32_t num_mesh_nodes, const F4 *tris) {
    const int ni = (int)sc.instances.size();
    Temps<BE> tmp(be);
    // the instances' world boxes, from the transformed vertices of their meshes, padded by more than the rounding of
    // the ray transform can move a hit point (1e-5 of the coordinates' magnitude)
    std::vector<F4> blo((size_t)ni), bhi((size_t)ni);
    {
        std::vector<float> xf(12 * (size_t)ni);
        std::vector<int32_t> ifirst((size_t)ni), icount((size_t)ni), binit(6 * (size_t)ni), bout(6 * (size_t)ni);
        int largest = 1;
        for (int i = 0; i < ni; ++i) {
            const rtb_instance &in = sc.instances[(size_t)i];
            memcpy(&xf[12 * (size_t)i], in.xform, sizeof(float) * 12);
            ifirst[(size_t)i] = (int32_t)sc.mesh_first[(size_t)in.mesh];
            icount[(size_t)i] = (int32_t)(sc.mesh_first[(size_t)in.mesh + 1] - sc.mesh_first[(size_t)in.mesh]);
            if (icount[(size_t)i] > largest) largest = icount[(size_t)i];
            for (int k = 0; k < 3; ++k) { binit[6 * (size_t)i + k] = float_to_ordered(FLT_MAX); binit[6 * (size_t)i + 3 + k] = float_to_ordered(-FLT_MAX); }
        }
        InstBoundsK k;
        k.a.runs = (largest + kInstBoundsRun - 1) / kInstBoundsRun;
        if ((long long)k.a.runs * ni > 0x7fffffffll) throw Error(RTB_ERR_INVALID, "too many instances x triangles for the bounds pass");
        float *d_xf = tmp.template alloc<float>(xf.size());
        int32_t *d_first = tmp.template alloc<int32_t>(ni), *d_count = tmp.template alloc<int32_t>(ni), *d_b = tmp.template alloc<int32_t>(6 * (size_t)ni);
        be.upload(d_xf, xf.data(), xf.size()); be.upload(d_first, ifirst.data(), (size_t)ni); be.upload(d_count, icount.data(), (size_t)ni);
        be.upload(d_b, binit.data(), binit.size());
        k.a.tris = (const Tri48 *)tris; k.a.xforms = d_xf; k.a.first = d_first; k.a.count = d_count; k.a.bounds = d_b; k.a.num_inst = ni;
        be.launch(k.a.runs * ni, k);
        be.download(bout.data(), d_b, bout.size());
        tmp.free(d_xf); tmp.free(d_first); tmp.free(d_count); tmp.free(d_b);
        for (int i = 0; i < ni; ++i) {
            float lo[3], hi[3];
            double mag = 0.0;
            for (int k2 = 0; k2 < 3; ++k2) {
                lo[k2] = ordered_to_float(bout[6 * (size_t)i + k2]); hi[k2] = ordered_to_float(bout[6 * (size_t)i + 3 + k2]);
                mag = fmax(mag, fmax(fabs((double)lo[k2]), fabs((double)hi[k2])));
            }
            const double pad = 1e-5 * mag + 1e-30;
            F4 l, h;
            l.x = (float)(lo[0] - pad); l.y = (float)(lo[1] - pad); l.z = (float)(lo[2] - pad); l.w = 0.f;
            h.x = (float)(hi[0] + pad); h.y = (float)(hi[1] + pad); h.z = (float)(hi[2] + pad); h.w = 0.f;
            if (!(fabsf(l.x) <= FLT_MAX && fabsf(l.y) <= FLT_MAX && fabsf(l.z) <= FLT_MAX && fabsf(h.x) <= FLT_MAX && fabsf(h.y) <= FLT_MAX && fabsf(h.z) <= FLT_MAX))
                throw Error(RTB_ERR_INVALID, "instance: world box not finite");
            blo[(size_t)i] = l; bhi[(size_t)i] = h;
        }
    }
    F4 *d_blo = tmp.template alloc<F4>(ni), *d_bhi = tmp.template alloc<F4>(ni);
    be.upload(d_blo, blo.data(), (size_t)ni); be.upload(d_bhi, bhi.data(), (size_t)ni);
    DeviceBuf<BE, int32_t> top_inst(be, (size_t)ni);
    int32_t *top_leaf_of = tmp.template alloc<int32_t>(ni);
    // every instance gets a child box of its own in the top tree (leaf lists of one entry)
    // (the SAH-optimal collapse: its tie-breaking caveat concerns triangles, and it halves the top tree — S2: 57 -> 27
    // nodes, 3.55 -> 3.38 nodes per primary ray; leaf lists of 2 or 3 instances were measured worse)
    rtb_build_params tbp = sc.bp;
    tbp.collapse = RTB_COLLAPSE_SAH_OPTIMAL;
    const BuiltTree top = build_tree(be, ni, nullptr, nullptr, nullptr, d_blo, d_bhi, tbp, 1, nullptr, nullptr, top_inst.p, top_leaf_of);
    DeviceBuf<BE, Q4> top_nodes(be, 0);
    top_nodes.p = top.nodes8;
    tmp.free(d_blo); tmp.free(d_bhi); tmp.free(top_leaf_of);
    // stack: a node group per level of both trees, plus the rest of a leaf list per level of the top tree
    if (2 * top.levels + sc.mesh_levels >= kStackSize) throw Error(RTB_ERR_INVALID, "BVH too deep for the traversal stack");
    // one node array: the top tree, then the meshes' trees rebased by the change of the top tree's size
    const int32_t num_nodes = top.num_nodes + num_mesh_nodes;
    DeviceBuf<BE, Q4> nodes(be, (size_t)num_nodes * kNodeWords);
    be.copy(nodes.p, top.nodes8, (size_t)top.num_nodes * kNodeWords);
    {
        RebaseK k; k.src = mesh_nodes; k.dst = nodes.p + (size_t)top.num_nodes * kNodeWords;
        k.node_off = (uint32_t)(top.num_nodes - mesh_base); k.tri_off = 0u; k.n = num_mesh_nodes;  // (a smaller top tree: wraps, as intended)
        be.launch(k.n, k);
    }
    // instance records
    std::vector<F4> rec((size_t)ni * kInstWords);
    int64_t flat_first = 0;
    for (int i = 0; i < ni; ++i) {
        const rtb_instance &in = sc.instances[(size_t)i];
        const double *inv = &inverse[12 * (size_t)i];
        F4 *r = rec.data() + (size_t)i * kInstWords;
        for (int k = 0; k < 3; ++k) {
            r[k].x = (float)inv[4 * k]; r[k].y = (float)inv[4 * k + 1]; r[k].z = (float)inv[4 * k + 2]; r[k].w = (float)inv[4 * k + 3];
            r[3 + k].x = in.xform[4 * k]; r[3 + k].y = in.xform[4 * k + 1]; r[3 + k].z = in.xform[4 * k + 2]; r[3 + k].w = in.xform[4 * k + 3];
        }
        const int mat = in.material >= 0 ? (in.material | (sc.material_type[(size_t)in.material] << 24)) : -1;
        r[6].x = i2f(top.num_nodes + sc.tree_first[(size_t)in.mesh]); r[6].y = i2f(mat); r[6].z = i2f((int)flat_first);
        r[6].w = i2f((int)sc.mesh_first[(size_t)in.mesh]);
        r[7].x = r[7].y = r[7].z = r[7].w = 0.f;
        flat_first += sc.mesh_first[(size_t)in.mesh + 1] - sc.mesh_first[(size_t)in.mesh];
    }
    DeviceBuf<BE, F4> inst(be, (size_t)ni * kInstWords);
    be.upload(inst.p, rec.data(), rec.size());
    be.sync();
    // nothing below throws: the new arrays replace the old ones
    be.free(sc.nodes8); be.free(sc.inst); be.free(sc.top_inst);
    sc.nodes8 = nodes.release(); sc.inst = inst.release(); sc.top_inst = top_inst.release();
    sc.num_nodes = num_nodes;
    sc.num_inst = ni;
    sc.stats.num_nodes = num_nodes;
    sc.stats.node_bytes = (int64_t)num_nodes * 80;
    sc.stats.sah_cost = top.sah_cost;
    sc.stats.ploc_iterations = top.ploc_iterations;
    sc.stats.collapse_levels = top.levels + sc.mesh_levels;
    for (int k = 0; k < 6; ++k) sc.stats.scene_bounds[k] = top.bounds[k];
    sc.stats.num_top_nodes = top.num_nodes;
}
template <class BE>
SceneT<BE> *scene_from_instanced(BE &be, const rtb_instanced_scene_desc &D, const rtb_build_params &bp) {
    const rtb_scene_desc &d = D.geometry;
    if (d.num_triangles <= 0 || !d.vertices || !d.material_ids || d.num_materials <= 0 || !d.materials)
        throw Error(RTB_ERR_INVALID, "rtb_scene_create_instanced: incomplete geometry");
    if (d.num_lights > 0 && !d.lights) throw Error(RTB_ERR_INVALID, "rtb_scene_create_instanced: lights missing");
    if (D.num_meshes <= 0 || !D.mesh_first || D.num_instances <= 0 || !D.instances)
        throw Error(RTB_ERR_INVALID, "rtb_scene_create_instanced: meshes / instances missing");
    if (d.num_triangles > 0x3fffffff) throw Error(RTB_ERR_INVALID, "too many triangles (max 2^30-1)");
    const int n = (int)d.num_triangles, nm = D.num_meshes, ni = D.num_instances;
    if (D.mesh_first[0] != 0 || D.mesh_first[nm] != n) throw Error(RTB_ERR_INVALID, "mesh_first must run from 0 to num_triangles");
    for (int m = 0; m < nm; ++m)
        if (D.mesh_first[m + 1] <= D.mesh_first[m]) throw Error(RTB_ERR_INVALID, "mesh_first must ascend strictly (no empty meshes)");
    for (int i = 0; i < d.num_materials; ++i)
        if (d.materials[i].type < 0 || d.materials[i].type >= kNumMaterialTypes) throw Error(RTB_ERR_INVALID, "unknown material type");
    std::vector<int> uses((size_t)nm, 0), ident((size_t)nm, 1);
    std::vector<long long> flat_first((size_t)ni + 1, 0);
    std::vector<double> inverse(12 * (size_t)ni);  // world -> object, checked before any device work
    for (int i = 0; i < ni; ++i) {
        const rtb_instance &in = D.instances[i];
        check_instance(in, nm, d.num_materials, &inverse[12 * (size_t)i]);
        uses[(size_t)in.mesh]++;
        if (!is_identity3x4(in.xform)) ident[(size_t)in.mesh] = 0;
        flat_first[(size_t)i + 1] = flat_first[(size_t)i] + (D.mesh_first[in.mesh + 1] - D.mesh_first[in.mesh]);
    }
    if (flat_first[(size_t)ni] > 0x7fffffffll) throw Error(RTB_ERR_INVALID, "flattened scene beyond 2^31-1 triangles");
    std::vector<int> mesh_of((size_t)n);
    for (int m = 0; m < nm; ++m) for (long long t = D.mesh_first[m]; t < D.mesh_first[m + 1]; ++t) mesh_of[(size_t)t] = m;
    std::vector<TriMeta> meta((size_t)n);
    for (int i = 0; i < n; ++i) {
        const int m = d.material_ids[i];
        if (m < 0 || m >= d.num_materials) throw Error(RTB_ERR_INVALID, "material id out of range");
        const int l = d.light_ids ? d.light_ids[i] : -1;
        if (l >= d.num_lights) throw Error(RTB_ERR_INVALID, "light id out of range");
        if (l >= 0 && !(uses[(size_t)mesh_of[(size_t)i]] == 1 && ident[(size_t)mesh_of[(size_t)i]]))
            throw Error(RTB_ERR_INVALID, "an emissive triangle must belong to a mesh instanced exactly once with the identity transform");
        meta[(size_t)i].material = m | (d.materials[m].type << 24);
        meta[(size_t)i].light = l;
    }
    std::vector<LightDev> lights((size_t)d.num_lights);
    std::vector<int64_t> light_tri((size_t)d.num_lights);
    for (int i = 0; i < d.num_lights; ++i) {
        const rtb_light &l = d.lights[i];
        if (l.type == RTB_AREA_LIGHT) {
            if (l.triangle < 0 || l.triangle >= n) throw Error(RTB_ERR_INVALID, "area light triangle out of range");
            const int m = mesh_of[(size_t)l.triangle];
            if (!(uses[(size_t)m] == 1 && ident[(size_t)m]))
                throw Error(RTB_ERR_INVALID, "an area light's triangle must belong to a mesh instanced exactly once with the identity transform");
        }
        LightDev &o = lights[(size_t)i];
        o.type = l.type; o.px = l.pos[0]; o.py = l.pos[1]; o.pz = l.pos[2]; o.tri = -1;
        o.Lx = l.L[0]; o.Ly = l.L[1]; o.Lz = l.L[2];
        light_tri[(size_t)i] = l.type == RTB_AREA_LIGHT ? l.triangle : 0;
    }
    check_builder(bp);
    const int max_leaf = bp.max_leaf_tris >= 1 && bp.max_leaf_tris <= 3 ? bp.max_leaf_tris : 3;
    SceneT<BE> *sc = new SceneT<BE>();
    std::vector<BuiltTree> trees((size_t)nm);
    try {
        sc->be = &be;
        sc->n = n;
        sc->n_flat = flat_first[(size_t)ni];
        sc->num_materials = d.num_materials;
        sc->num_lights = d.num_lights;
        Temps<BE> tmp(be);
        auto t0 = be.now();
        sc->materials = be.template alloc<rtb_material>(d.num_materials);
        be.upload(sc->materials, d.materials, d.num_materials);
        for (int i = 0; i < d.num_materials; ++i) sc->type_mask |= 1u << d.materials[i].type;
        sc->lights = be.template alloc<LightDev>(d.num_lights > 0 ? d.num_lights : 1);
        int64_t *d_light_tri = tmp.template alloc<int64_t>(d.num_lights > 0 ? d.num_lights : 1);
        if (d.num_lights) { be.upload(sc->lights, lights.data(), d.num_lights); be.upload(d_light_tri, light_tri.data(), d.num_lights); }
        float *d_vertices = tmp.template alloc<float>(9 * (size_t)n);
        Tri48 *tri_in = tmp.template alloc<Tri48>(n);
        TriMeta *meta_in = tmp.template alloc<TriMeta>(n);
        be.upload(d_vertices, d.vertices, 9 * (size_t)n);
        be.upload(meta_in, meta.data(), (size_t)n);
        sc->tris = (F4 *)be.template alloc<Tri48>(n);
        sc->meta = be.template alloc<TriMeta>(n);
        sc->prim = be.template alloc<int32_t>(n);
        sc->leaf_of_prim = be.template alloc<int32_t>(n);
        // the meshes' trees, each with indices relative to itself
        int mesh_nodes = 0, mesh_levels = 0;
        for (int m = 0; m < nm; ++m) {
            const int first = (int)D.mesh_first[m], cnt = (int)(D.mesh_first[m + 1] - D.mesh_first[m]);
            trees[(size_t)m] = build_tree(be, cnt, d_vertices + 9 * (size_t)first, tri_in + first, meta_in + first, nullptr, nullptr, bp,
                                          max_leaf, (Tri48 *)sc->tris + first, sc->meta + first, sc->prim + first, sc->leaf_of_prim + first);
            if (first) {
                AddK k; k.p = sc->prim + first; k.v = first; k.n = cnt; be.launch(cnt, k);
                k.p = sc->leaf_of_prim + first; be.launch(cnt, k);
            }
            mesh_nodes += trees[(size_t)m].num_nodes;
            if (trees[(size_t)m].levels > mesh_levels) mesh_levels = trees[(size_t)m].levels;
        }
        tmp.free(d_vertices); tmp.free(tri_in); tmp.free(meta_in);
        // what updates of the scene need (refit_scene, set_instances)
        sc->bp = bp;
        sc->mesh_first.assign(D.mesh_first, D.mesh_first + nm + 1);
        sc->instances.assign(D.instances, D.instances + ni);
        sc->mesh_emissive.assign((size_t)nm, 0);
        for (int i = 0; i < n; ++i) if (meta[(size_t)i].light >= 0) sc->mesh_emissive[(size_t)mesh_of[(size_t)i]] = 1;
        for (int i = 0; i < d.num_lights; ++i)
            if (d.lights[i].type == RTB_AREA_LIGHT) sc->mesh_emissive[(size_t)mesh_of[(size_t)d.lights[i].triangle]] = 1;
        sc->material_type.resize((size_t)d.num_materials);
        for (int i = 0; i < d.num_materials; ++i) sc->material_type[(size_t)i] = d.materials[i].type;
        sc->mesh_levels = mesh_levels;
        // the meshes' trees in one array, rebased as if the top tree had no nodes (install_top moves them behind it)
        Q4 *mesh_nodes_d = tmp.template alloc<Q4>((size_t)mesh_nodes * kNodeWords);
        sc->tree_levels.resize((size_t)nm);
        sc->tree_first.resize((size_t)nm);
        {
            int off = 0;
            for (int m = 0; m < nm; ++m) {
                RebaseK k; k.src = trees[(size_t)m].nodes8; k.dst = mesh_nodes_d + (size_t)off * kNodeWords;
                k.node_off = (uint32_t)off; k.tri_off = (uint32_t)D.mesh_first[m]; k.n = trees[(size_t)m].num_nodes;
                be.launch(k.n, k);
                sc->tree_first[(size_t)m] = off;
                sc->tree_levels[(size_t)m] = trees[(size_t)m].level_nodes;
                off += trees[(size_t)m].num_nodes;
            }
        }
        be.sync();
        for (int m = 0; m < nm; ++m) { be.free(trees[(size_t)m].nodes8); trees[(size_t)m].nodes8 = nullptr; }
        sc->stats = rtb_bvh_stats{};
        install_top(be, *sc, inverse, mesh_nodes_d, 0, mesh_nodes, sc->tris);
        tmp.free(mesh_nodes_d);
        if (sc->num_lights > 0) {
            LightFixK k; k.lights = sc->lights; k.light_tri = d_light_tri; k.leaf_of_prim = sc->leaf_of_prim; k.n = sc->num_lights;
            be.launch(sc->num_lights, k);
        }
        be.sync();
        tmp.free(d_light_tri);
        sc->stats.num_triangles = n;
        sc->stats.num_bvh2_nodes = 2 * (int64_t)n - nm + 2 * (int64_t)ni - 1;
        sc->stats.triangle_bytes = (int64_t)n * 48;
        sc->stats.num_instances = ni;
        sc->stats.num_flat_triangles = sc->n_flat;
        sc->stats.build_ms = be.elapsed_ms(t0, be.now());
    } catch (...) {
        for (auto &t : trees) be.free(t.nodes8);
        delete sc;
        throw;
    }
    return sc;
}

// ---- in-place updates (rtb_scene_refit, rtb_scene_set_instances) ----
struct RefitTrisK { RefitTrisArgs a; RTB_HD void operator()(int i) const { refit_tris_body(a, i); } };
// The nodes of one depth: the backend's kernel (rtb_cuda.cu asserts that CudaBackend has one: k_refit_level, whose warps
// reduce the SAH terms over a full mask before one atomic), or a plain loop (the host emulation).
template <class BE, class = void> struct HasRefitKernels : std::false_type {};
template <class BE>
struct HasRefitKernels<BE, std::void_t<decltype(std::declval<BE &>().refit_level(std::declval<const RefitArgs &>()))>> : std::true_type {};
template <class BE>
void refit_level(BE &be, const RefitArgs &a) {
    if constexpr (HasRefitKernels<BE>::value) be.refit_level(a);
    else for (int i = 0; i < a.num; ++i) atomic_add_f(a.sah, refit_body(a, i));
}
// New vertex positions for every triangle (9 floats each, caller order; host or device memory), same topology.  Returns
// the GPU time of the update.  Every temporary is allocated first, and the scene is only touched once the vertices
// have passed the builder's check.  The records go to a new array that replaces the scene's (rather than a check-only
// pass over the vertices and an in-place write): an instanced scene needs the new records for the instance boxes before
// its top tree is rebuilt, and that rebuild may still fail (a world box beyond float, the stack depth), which must
// leave the scene as it was; reading the vertices once also keeps the large flat scenes at one pass over them.  The
// spare records cost the size of the triangle array while the call runs (S2: 480 MB of a B200's 180 GB).
template <class BE>
float refit_scene(BE &be, SceneT<BE> &sc, const float *h_vertices, const float *d_vertices) {
    const int n = (int)sc.n;
    if (n > 0 && !h_vertices && !d_vertices) throw Error(RTB_ERR_INVALID, "rtb_scene_refit: null vertices");
    if (n == 0) return 0.f;  // (the empty root has nothing to refit)
    const bool inst = sc.inst != nullptr;
    const int top_nodes = inst ? (int)sc.stats.num_top_nodes : 0;
    // depth schedule: the nodes of each depth, deepest first.  A flat scene's are one range per level; an instanced
    // scene's are the union of its mesh trees' ranges, as a list of ids
    int depths = 0;
    for (const auto &lv : sc.tree_levels) depths = (int)lv.size() > depths ? (int)lv.size() : depths;
    std::vector<int32_t> ids, dfirst((size_t)depths + 1, 0);
    {
        int64_t total = 0;
        for (size_t t = 0; t < sc.tree_levels.size(); ++t) for (int32_t c : sc.tree_levels[t]) total += c;
        if (total != (int64_t)sc.num_nodes - top_nodes) throw Error(RTB_ERR_INVALID, "internal: refit depth schedule does not cover the tree");
        // per depth (ascending) and tree: the range's first id
        std::vector<std::vector<int32_t>> first(sc.tree_levels.size());
        for (size_t t = 0; t < sc.tree_levels.size(); ++t) {
            int32_t f = top_nodes + sc.tree_first[t];
            for (int32_t c : sc.tree_levels[t]) { first[t].push_back(f); f += c; }
        }
        if (inst) {
            for (int d = depths - 1, k = 0; d >= 0; --d, ++k) {
                dfirst[(size_t)k] = (int32_t)ids.size();
                for (size_t t = 0; t < sc.tree_levels.size(); ++t)
                    if (d < (int)sc.tree_levels[t].size())
                        for (int32_t j = 0; j < sc.tree_levels[t][(size_t)d]; ++j) ids.push_back(first[t][(size_t)d] + j);
            }
            dfirst[(size_t)depths] = (int32_t)ids.size();
        } else {
            for (int d = depths - 1, k = 0; d >= 0; --d, ++k) dfirst[(size_t)k] = first[0][(size_t)d];
        }
    }
    Temps<BE> tmp(be);
    float *vup = h_vertices ? tmp.template alloc<float>(9 * (size_t)n) : nullptr;
    Tri48 *tris = tmp.template alloc<Tri48>(n);
    int32_t *ctr = tmp.template alloc<int32_t>(2);  // bad vertex, SAH sum (float)
    float *box = tmp.template alloc<float>(6 * (size_t)sc.num_nodes);
    Q4 *nodes = inst ? tmp.template alloc<Q4>((size_t)sc.num_nodes * kNodeWords) : sc.nodes8;  // (instanced: a copy, see above)
    int32_t *d_ids = inst ? tmp.template alloc<int32_t>(ids.size()) : nullptr;
    std::vector<double> inverse(12 * sc.instances.size());  // (instanced: the scene's instances, checked when they were set)
    for (size_t i = 0; i < sc.instances.size(); ++i) invert3x4(sc.instances[i].xform, &inverse[12 * i]);
    if (h_vertices) be.upload(vup, h_vertices, 9 * (size_t)n);
    if (inst) be.upload(d_ids, ids.data(), ids.size());
    auto t0 = be.now();
    try {
        be.zero(ctr, 2);
        {
            RefitTrisK k; k.a.vertices = h_vertices ? vup : d_vertices; k.a.leaf_of_prim = sc.leaf_of_prim; k.a.tris = (F4 *)tris; k.a.bad = ctr; k.a.n = n;
            be.launch(n, k);
        }
        int32_t bad = 0;
        be.download(&bad, ctr, 1);
        if (bad) throw Error(RTB_ERR_INVALID, "rtb_scene_refit: a triangle vertex is not finite or beyond 2^100; the scene is unchanged");
        if (inst) be.copy(nodes, sc.nodes8, (size_t)sc.num_nodes * kNodeWords);
        for (int k = 0; k < depths; ++k) {
            RefitArgs a; a.nodes8 = nodes; a.tris = (const F4 *)tris; a.box = box; a.sah = (float *)(ctr + 1);
            a.order = d_ids;
            if (inst) { a.first = dfirst[(size_t)k]; a.num = dfirst[(size_t)k + 1] - dfirst[(size_t)k]; }
            else { a.first = dfirst[(size_t)k]; a.num = sc.tree_levels[0][(size_t)(depths - 1 - k)]; }
            refit_level(be, a);
        }
        if (inst) {
            install_top(be, sc, inverse, nodes + (size_t)top_nodes * kNodeWords, top_nodes, sc.num_nodes - top_nodes, (const F4 *)tris);
        } else {
            float c[7];
            be.download(c, box, 6);
            be.download(c + 6, (const float *)(ctr + 1), 1);
            const float root_area = half_area(c[3] - c[0], c[4] - c[1], c[5] - c[2]);
            sc.stats.sah_cost = root_area > 0.f ? c[6] / root_area : 0.f;
            for (int k = 0; k < 3; ++k) { sc.stats.scene_bounds[2 * k] = c[k]; sc.stats.scene_bounds[2 * k + 1] = c[3 + k]; }
        }
    } catch (...) {
        be.release(t0);
        throw;
    }
    // the new records replace the old ones (flat scenes: the nodes were refit in place; instanced: install_top)
    for (auto &h : tmp.held) if (h == (void *)tris) h = (void *)sc.tris;  // (the old records are freed with the temporaries)
    sc.tris = (F4 *)tris;
    return be.elapsed_ms(t0, be.now());
}
// New instance records for an instanced scene: same count, every instance keeps its mesh (so the flattened hit ids keep
// their meaning), transforms and materials may change.  The mesh trees stay; the instance boxes, the top tree and the
// records are rebuilt (install_top).
template <class BE>
void set_instances(BE &be, SceneT<BE> &sc, const rtb_instance *h_instances, int32_t num_instances) {
    if (!sc.inst) throw Error(RTB_ERR_INVALID, "rtb_scene_set_instances: not an instanced scene");
    if (!h_instances) throw Error(RTB_ERR_INVALID, "rtb_scene_set_instances: null instances");
    if (num_instances != (int32_t)sc.instances.size()) throw Error(RTB_ERR_INVALID, "rtb_scene_set_instances: the instance count differs from the scene's");
    const int ni = num_instances, nm = (int)sc.mesh_first.size() - 1;
    std::vector<double> inverse(12 * (size_t)ni);
    for (int i = 0; i < ni; ++i) {
        const rtb_instance &in = h_instances[i];
        if (in.mesh != sc.instances[(size_t)i].mesh) throw Error(RTB_ERR_INVALID, "rtb_scene_set_instances: instance: mesh changed");
        check_instance(in, nm, sc.num_materials, &inverse[12 * (size_t)i]);
        if (sc.mesh_emissive[(size_t)in.mesh] && !is_identity3x4(in.xform))
            throw Error(RTB_ERR_INVALID, "rtb_scene_set_instances: an emissive triangle must belong to a mesh instanced exactly once with the identity transform");
    }
    const std::vector<rtb_instance> old = sc.instances;
    sc.instances.assign(h_instances, h_instances + ni);
    const int top_nodes = (int)sc.stats.num_top_nodes;
    try {
        install_top(be, sc, inverse, sc.nodes8 + (size_t)top_nodes * kNodeWords, top_nodes, sc.num_nodes - top_nodes, sc.tris);
    } catch (...) {
        sc.instances = old;
        throw;
    }
}

// ---- wavefront loop ----
// One iteration = shade (one launch per material type present) -> generate ->
// control -> trace (extend + shadow rays), in stream order.  The host never
// waits for an iteration: it keeps two batches of launches in flight and
// watches a `done` word that the control kernel raises in mapped host memory.
//
// Wavefronts.  The render is split into `np` independent wavefronts — the paths k mod np, each with its own queues and
// counters and an np-th of the pool — on their own streams; they only meet in the accumulation buffer (atomic adds).
// The CUDA backend launches each wavefront's trace kernel on an np-th of the SM (CudaBackend::trace_grid), so that one
// wavefront's issue-bound traversal runs beside another's DRAM-bound shading instead of after it: four wavefronts on
// scenes that fit L2 (C2 37.4 -> 35.0 ms, C4 37.6 -> 28.1 ms), two with full-size launches beyond (DESIGN.md 4.5).
// where the radiance sums of a render go once the wavefronts have finished (inside the timed region of the call)
struct RenderTarget {
    float *add_f32 = nullptr;        // float[3 * W * H] += sums                       (rtb_render_accumulate)
    long long *add_fixed = nullptr;  // int64[3 * W * H] += fixed-point sums           (rtb_render_accumulate_fixed)
    float *tonemap_to = nullptr;     // float[3 * W * H] = sqrt(sums / tonemap_spp)    (rtb_render)
    int32_t tonemap_spp = 0;
};
template <class BE>
void render_accumulate(BE &be, SceneT<BE> &sc, const rtb_camera &cam, const rtb_render_params &p, const RenderTarget &target,
                       rtb_render_stats *stats) {
    if (p.width <= 0 || p.height <= 0 || p.spp <= 0 || p.max_bounces < 0 || !(target.add_f32 || target.add_fixed || target.tonemap_to))
        throw Error(RTB_ERR_INVALID, "rtb_render: bad parameters");
    if (p.device_mask != 0 && be.device() >= 0 && !(p.device_mask >> be.device() & 1))
        throw Error(RTB_ERR_INVALID, "rtb_render: device_mask excludes the GPU of this scene's context (use rtb_multi_render to span GPUs)");
    if (p.max_bounces > kMaxBounces) throw Error(RTB_ERR_INVALID, "rtb_render: max_bounces > 255");
    if (p.first_sample < 0 || (long long)p.first_sample + p.spp > kMaxSampleIndex) throw Error(RTB_ERR_INVALID, "rtb_render: sample index >= 2^24");
    const unsigned long long total = (unsigned long long)p.width * (unsigned long long)p.height * (unsigned long long)p.spp;
    if ((unsigned long long)p.width * (unsigned long long)p.height > 0x7fffffffull) throw Error(RTB_ERR_INVALID, "image too large");
    const int mode = (p.flags & RTB_RENDER_COUNT_WORK) ? 2 : ((p.flags & RTB_RENDER_NONPERSISTENT) ? 1 : 0);
    // queue bytes of one path slot: two ray queues of 48 B and a 48-byte hit queue per material type present (+ side arrays)
    const size_t slot_bytes = 96 + (size_t)sc.num_present() * (48 + ((p.flags & RTB_RENDER_TRUE_MIS) ? 8 : 0) + (sc.inst ? 4 : 0));
    long long pool_all = p.pool_size > 0 ? p.pool_size : be.default_pool(slot_bytes);
    if ((unsigned long long)pool_all > total) pool_all = (long long)total;
    int np = be.pipelines(sc.view());
    if (np > kMaxPipelines) np = kMaxPipelines;
    if (np < 1 || mode != 0 || (p.flags & RTB_RENDER_SINGLE_PIPELINE) || pool_all < (1 << 16)) np = 1;
    const int pool = (int)(((pool_all + np - 1) / np + 31) & ~31ll);
    sc.ensure_wave(pool, np);
    const bool fixed = (p.flags & RTB_RENDER_DETERMINISTIC) != 0 || target.add_fixed != nullptr;
    const int64_t pixels = (int64_t)p.width * p.height;
    if (3 * pixels > 0x7fffff00ll) throw Error(RTB_ERR_INVALID, "image too large");
    sc.ensure_accum(pixels, fixed);
    const SceneView S = sc.view();
    const bool shadows = sc.num_lights > 0 && !(p.flags & RTB_RENDER_NO_SHADOW);
    WaveState W[kMaxPipelines];
    RenderConsts rc[kMaxPipelines];
    be.use_stream(0);  // (an error thrown out of an earlier call may have left another stream selected)
    be.begin_render(np);
    auto t0 = be.now();
    if (fixed) be.zero(sc.accum_fx, 3 * (size_t)pixels);  // init_framebuffer, render.cuh:61-66
    else be.zero(sc.accum, (size_t)pixels);
    for (int k = 0; k < np; ++k) {
        if ((p.flags & RTB_RENDER_TRUE_MIS) && !sc.W[k].mis) sc.W[k].mis = be.template alloc<float>(2 * (size_t)sc.num_present() * (size_t)pool);
        W[k] = sc.W[k];
        if (!(p.flags & RTB_RENDER_TRUE_MIS)) W[k].mis = nullptr;
        W[k].env[0] = p.env_L[0]; W[k].env[1] = p.env_L[1]; W[k].env[2] = p.env_L[2];
        W[k].has_env = (p.env_L[0] != 0.f || p.env_L[1] != 0.f || p.env_L[2] != 0.f) ? 1 : 0;
        W[k].accum = fixed ? nullptr : sc.accum;
        W[k].accum_fx = fixed ? sc.accum_fx : nullptr;
        W[k].host_done = be.done_flag_device(k);
        RenderConsts &r = rc[k];
        r.cam = cam; r.width = p.width; r.height = p.height; r.spp = p.spp; r.first_sample = p.first_sample;
        r.max_bounces = p.max_bounces; r.rr_start = p.rr_start; r.rr_threshold = p.rr_threshold; r.seed = p.seed; r.flags = p.flags;
        r.path_offset = k; r.path_stride = np;
        r.env[0] = p.env_L[0]; r.env[1] = p.env_L[1]; r.env[2] = p.env_L[2];
        Counters c0;
        memset(&c0, 0, sizeof c0);
        c0.total_paths = (total - (unsigned long long)k + (unsigned long long)np - 1ull) / (unsigned long long)np;
        be.reset_done(k);
        be.upload(W[k].c, &c0, 1);
    }
    for (int k = 1; k < np; ++k) be.fork(k);  // stream k starts after everything queued so far on the main stream
    unsigned long long launches = 0;
    const int batch = 4;
    const bool time_stages = stats != nullptr && np == 1;
    // per iteration: [0] before shade, [1] before the traversal kernels, [2] after extend (or after the
    // fused extend+shadow launch), [3] after shadow
    std::vector<typename BE::Time> stage_times, fences[kMaxPipelines];
    size_t fence_head[kMaxPipelines] = {0, 0};
    bool finished[kMaxPipelines] = {false, false};
    bool fused = false;
    int live = np;
    while (live > 0) {
        for (int k = 0; k < np; ++k) {
            if (finished[k]) continue;
            be.use_stream(k);
            for (int b = 0; b < batch; ++b) {
                if (time_stages) stage_times.push_back(be.now());
                for (int type = 0; type < kNumMaterialTypes; ++type) {
                    if (!(sc.type_mask >> type & 1u)) continue;
                    ShadeK ks; ks.W = W[k]; ks.S = S; ks.rc = rc[k]; ks.type = type; ks.shadows = shadows;
                    be.shade(ks);
                    ++launches;
                }
                { GenerateK kg; kg.W = W[k]; kg.rc = rc[k]; be.generate(kg); }
                be.control(W[k], shadows);
                if (time_stages) stage_times.push_back(be.now());
                if (be.trace_fused(W[k], S, mode)) {
                    fused = true;
                    if (time_stages) { stage_times.push_back(be.now()); stage_times.push_back(be.now()); }
                    launches += 3;
                } else {
                    be.extend(W[k], S, mode);
                    if (time_stages) stage_times.push_back(be.now());
                    be.shadow(W[k], S, mode);
                    if (time_stages) stage_times.push_back(be.now());
                    launches += 4;
                }
            }
            fences[k].push_back(be.now());
        }
        for (int k = 0; k < np; ++k) {
            if (finished[k]) continue;
            if (fences[k].size() - fence_head[k] > 2) be.wait(fences[k][fence_head[k]++]);
            if (be.done(k)) { finished[k] = true; --live; }
        }
    }
    be.use_stream(0);
    for (int k = 1; k < np; ++k) be.join(k);  // the main stream continues after stream k's work
    if (target.add_f32) {
        FoldF32K k; k.in = sc.accum; k.in_fx = fixed ? sc.accum_fx : nullptr; k.out = target.add_f32; k.pixels = pixels;
        be.launch((int)pixels, k);
    }
    if (target.add_fixed) { FoldFixedK k; k.in_fx = sc.accum_fx; k.out = target.add_fixed; k.n = 3 * pixels; be.launch((int)(3 * pixels), k); }
    if (target.tonemap_to) {  // post_process_framebuffer, render.cuh:330-338
        if (target.tonemap_spp <= 0) throw Error(RTB_ERR_INVALID, "rtb_render: bad total_spp");
        TonemapAccumK k; k.in = sc.accum; k.in_fx = fixed ? sc.accum_fx : nullptr; k.out = target.tonemap_to; k.pixels = pixels;
        k.inv_spp = 1.0f / (float)target.tonemap_spp;
        be.launch((int)pixels, k);
    }
    auto t1 = be.now();
    be.wait(t1);
    for (int k = 0; k < np; ++k) for (auto &e : fences[k]) be.release(e);
    float ms_extend = 0.f, ms_shadow = 0.f, ms_shade = 0.f;
    for (size_t i = 0; i + 3 < stage_times.size(); i += 4) {
        ms_shade += be.elapsed_keep(stage_times[i], stage_times[i + 1]);
        ms_extend += be.elapsed_keep(stage_times[i + 1], stage_times[i + 2]);
        ms_shadow += be.elapsed_keep(stage_times[i + 2], stage_times[i + 3]);
    }
    for (auto &e : stage_times) be.release(e);
    const float ms_total = be.elapsed_ms(t0, t1);
    if (stats) {
        memset(stats, 0, sizeof *stats);
        for (int k = 0; k < np; ++k) {
            Counters c;
            be.download(&c, W[k].c, 1);
            stats->paths += c.stat_paths;
            stats->extend_rays += c.stat_extend;
            stats->shadow_rays += c.stat_shadow;
            stats->iterations += c.stat_iters;
            stats->extend_nodes += c.work[0]; stats->extend_tris += c.work[1];
            stats->shadow_nodes += c.work[2]; stats->shadow_tris += c.work[3];
            stats->hits += c.stat_hits;
        }
        stats->kernel_launches = launches;
        stats->extend_launches = stats->iterations; stats->shadow_launches = stats->iterations;
        stats->ms_extend = ms_extend; stats->ms_shadow = ms_shadow;
        stats->ms_total = ms_total;
        stats->ms_other = ms_total - ms_extend - ms_shadow;
        stats->ms_shade = ms_shade;
        stats->fused_trace = fused ? 1 : 0;
        stats->pipelines = np;
        stats->pool = pool;
    }
}

// ---- the render path's traversal kernels on caller-supplied rays (rtb_trace_wavefront) ----
// rtb_trace_closest / rtb_trace_any run one thread per ray (Traversal::step).  The render path does not: its rays sit
// in the extend / shadow queues and are traversed by the persistent kernel (dynamic fetch, refill, stepped or pooled
// triangle tests, finish words staged by cp.async, hit records appended per material type).  This entry loads the
// caller's rays into those queues, runs ONE iteration's trace launch(es) exactly as render_accumulate does, and reads
// the results back from where the render path leaves them: hit records out of the per-type hit queues (the ray index
// travels in the pixel field, t in the `mis` side array), occlusion out of the accumulation buffer (an unoccluded
// shadow ray splats radiance (1,0,0) at "pixel" = ray index).  So the kernel compared with the reference's
// Bvh::traverse (bvh.cuh:251-357) by the parity tests is the one that renders.
struct RayLoadK {
    const rtb_ray *rays; WaveState W; int32_t first, n;
    RTB_HD void operator()(int i) const {
        if (i >= n) return;
        const rtb_ray r = rays[first + i];
        F4 a, b, c;
        a.x = r.origin[0]; a.y = r.origin[1]; a.z = r.origin[2]; a.w = u2f((uint32_t)i);
        b.x = r.dir[0]; b.y = r.dir[1]; b.z = r.dir[2]; b.w = u2f(0u);
        c.x = c.y = c.z = 1.f; c.w = 0.f;
        if (!ray_is_finite(r)) a.w = u2f(kHolePixel);  // retired before the queue in the render (shade_item): reported as a miss
        W.ea[i] = a; W.eb[i] = b; W.ec[i] = c;
    }
};
struct ShadowLoadK {
    const rtb_ray *rays; const int32_t *excluded; const int32_t *leaf_of_prim; Bvh8View B; WaveState W; int32_t first, n;
    RTB_HD void operator()(int i) const {
        if (i >= n) return;
        const rtb_ray r = rays[first + i];
        int ex = excluded ? excluded[first + i] : -1;
        if (ex >= 0) ex = leaf_of_prim[ex];
        F4 o, d, l;
        o.x = r.origin[0]; o.y = r.origin[1]; o.z = r.origin[2]; o.w = r.tmax;
        d.x = r.dir[0]; d.y = r.dir[1]; d.z = r.dir[2]; d.w = i2f(ex);
        l.x = 1.f; l.y = 0.f; l.z = 0.f; l.w = u2f((uint32_t)i);
        // a hole (tmax = 0) leaves the "pixel" at 0 = reads as occluded: a non-finite ray or tmax <= 0 is reported
        // unoccluded by TraceAnyK, so splat it here
        if (!ray_is_finite(r) || !(r.tmax > 0.f)) { o.w = 0.f; accum_add(W, (uint32_t)i, v3(1.f, 0.f, 0.f)); }
        W.sh_o[i] = o; W.sh_d[i] = d; W.sh_L[i] = l;
    }
};
struct HitGatherK {
    WaveState W; Bvh8View B; rtb_hit *hits; int32_t first, type, n;
    RTB_HD void operator()(int j) const {
        if (j >= n) return;
        const size_t q = (size_t)W.qbase[type] + (size_t)j;
        const F4 a = W.ma[q], c = W.mc[q];
        const int tri = f2i(c.w);
        rtb_hit h;
        h.t = W.mis[2 * q + 1]; h.u = c.y; h.v = c.z;
        h.prim = hit_prim(B, tri, W.hit_inst ? W.hit_inst[q] : -1);
        hits[first + (int)f2u(a.w)] = h;
    }
};
struct MissFillK {
    rtb_hit *hits; int64_t n;
    RTB_HD void operator()(int i) const {
        if (i >= n) return;
        rtb_hit h; h.t = 0.f; h.u = 0.f; h.v = 0.f; h.prim = -1;
        hits[i] = h;
    }
};
struct OccludedK {
    const F4 *accum; uint8_t *occ; int32_t first, n;
    RTB_HD void operator()(int i) const { if (i < n) occ[first + i] = accum[i].x == 0.f ? 1 : 0; }
};
template <class BE>
void trace_wavefront(BE &be, SceneT<BE> &sc, const rtb_ray *d_rays, int64_t n, rtb_hit *d_hits, const rtb_ray *d_srays,
                     const int32_t *d_excl, int64_t ns, uint8_t *d_occ, int32_t *launches_out) {
    if (sc.inst && d_excl) throw Error(RTB_ERR_INVALID, "rtb_trace_wavefront: excluded triangles are not supported on instanced scenes");
    const int64_t most = n > ns ? n : ns;
    const int32_t cap = (int32_t)(((most < (1 << 22) ? most : (1 << 22)) + 31) & ~31ll);
    if (cap == 0) return;
    be.use_stream(0);
    be.begin_render(1);
    WaveState W{};
    const SceneView S = sc.view();
    int launches = 0;
    try {
        W.ea = be.template alloc<F4>(cap); W.eb = be.template alloc<F4>(cap); W.ec = be.template alloc<F4>(cap);
        const size_t nq = (size_t)sc.num_present() * (size_t)cap;
        W.ma = be.template alloc<F4>(nq); W.mb = be.template alloc<F4>(nq); W.mc = be.template alloc<F4>(nq);
        W.sh_o = be.template alloc<F4>(cap); W.sh_d = be.template alloc<F4>(cap); W.sh_L = be.template alloc<F4>(cap);
        W.c = be.template alloc<Counters>(1);
        W.mis = be.template alloc<float>(2 * nq);
        W.hit_inst = sc.inst ? be.template alloc<int32_t>(nq) : nullptr;
        W.accum = be.template alloc<F4>((size_t)cap);
        W.pool = cap;
        sc.fill_qbase(W, cap);
        if (n > 0) { MissFillK k; k.hits = d_hits; k.n = n; be.launch((int)n, k); }
        for (int64_t first = 0; first < most; first += cap) {
            const int32_t ne = (int32_t)(first < n ? (n - first < cap ? n - first : cap) : 0);
            const int32_t nsh = (int32_t)(first < ns ? (ns - first < cap ? ns - first : cap) : 0);
            be.zero(W.accum, (size_t)cap);
            if (ne) { RayLoadK k; k.rays = d_rays; k.W = W; k.first = (int32_t)first; k.n = ne; be.launch(ne, k); }
            if (nsh) {
                ShadowLoadK k; k.rays = d_srays; k.excluded = d_excl; k.leaf_of_prim = sc.leaf_of_prim; k.B = S.bvh; k.W = W;
                k.first = (int32_t)first; k.n = nsh;
                be.launch(nsh, k);
            }
            Counters c0;
            memset(&c0, 0, sizeof c0);
            c0.n_extend = ne; c0.n_shadow = nsh;
            be.upload(W.c, &c0, 1);
            if (be.trace_fused(W, S, 0)) launches += 1;
            else { be.extend(W, S, 0); be.shadow(W, S, 0); launches += 2; }
            Counters c1;
            be.download(&c1, W.c, 1);
            for (int type = 0; type < kNumMaterialTypes; ++type) {
                if (c1.n_mat[type] <= 0) continue;
                HitGatherK k; k.W = W; k.B = S.bvh; k.hits = d_hits; k.first = (int32_t)first; k.type = type; k.n = c1.n_mat[type];
                be.launch(k.n, k);
            }
            if (nsh) { OccludedK k; k.accum = W.accum; k.occ = d_occ; k.first = (int32_t)first; k.n = nsh; be.launch(nsh, k); }
        }
        be.sync();
    } catch (...) {
        be.free(W.ea); be.free(W.eb); be.free(W.ec); be.free(W.ma); be.free(W.mb); be.free(W.mc); be.free(W.sh_o); be.free(W.sh_d);
        be.free(W.sh_L); be.free(W.c); be.free(W.mis); be.free(W.hit_inst); be.free(W.accum);
        throw;
    }
    be.free(W.ea); be.free(W.eb); be.free(W.ec); be.free(W.ma); be.free(W.mb); be.free(W.mc); be.free(W.sh_o); be.free(W.sh_d);
    be.free(W.sh_L); be.free(W.c); be.free(W.mis); be.free(W.hit_inst); be.free(W.accum);
    if (launches_out) *launches_out = launches;
}

template <class BE>
void tonemap(BE &be, const float *d_in, int64_t n, int total_spp, float *d_out) {
    if (n <= 0 || n > 0x7fffff00ll || total_spp <= 0) throw Error(RTB_ERR_INVALID, "rtb_tonemap: bad arguments");
    TonemapK k; k.in = d_in; k.out = d_out; k.n = n; k.inv_spp = 1.0f / (float)total_spp;
    be.launch((int)n, k);
}
template <class BE>
void tonemap_fixed(BE &be, const long long *d_in, int64_t n, int total_spp, float *d_out) {
    if (n <= 0 || n > 0x7fffff00ll || total_spp <= 0) throw Error(RTB_ERR_INVALID, "rtb_tonemap_fixed: bad arguments");
    TonemapFixedK k; k.in = d_in; k.out = d_out; k.n = n; k.inv_spp = 1.0f / (float)total_spp;
    be.launch((int)n, k);
}

}  // namespace rtb
