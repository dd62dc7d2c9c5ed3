// rtb_api_impl.h — the extern "C" entry points of include/rtb.h, written
// against `RTB_BACKEND` (a type defined by the including translation unit:
// CudaBackend in rtb_cuda.cu for the shipped library).  No entry point lets a
// C++ exception escape; errors become rtb_status codes + rtb_last_error().
#pragma once
#include <chrono>
#include <functional>
#include <map>
#include <memory>
#include <thread>

#include "host/host_util.h"
#include "rtb_engine.h"

struct rtb_context {
    RTB_BACKEND be;
    explicit rtb_context(int device) : be(device) {}
};
struct rtb_scene {
    rtb_context *ctx;
    rtb::SceneT<RTB_BACKEND> *impl;
};

namespace rtb {
template <class F>
int guarded(F f) {
    try {
        f();
        return RTB_OK;
    } catch (const Error &e) {
        return set_error(e.code, e.what());
    } catch (const std::bad_alloc &) {
        return set_error(RTB_ERR_OOM, "out of host memory");
    } catch (const std::exception &e) {
        return set_error(RTB_ERR_CUDA, e.what());
    }
}
inline rtb_build_params build_defaults() {
    rtb_build_params p;
    p.builder = RTB_BUILDER_PLOC; p.ploc_radius = 16; p.max_leaf_tris = 3; p.collapse = RTB_COLLAPSE_LARGEST_FIRST;
    return p;
}
}  // namespace rtb

extern "C" {

int rtb_context_create(int device, rtb_context **out) {
    if (!out) return rtb::set_error(RTB_ERR_INVALID, "rtb_context_create: null out");
    *out = nullptr;
    return rtb::guarded([&] { *out = new rtb_context(device); });
}
int rtb_context_destroy(rtb_context *ctx) {
    return rtb::guarded([&] { delete ctx; });
}
int rtb_context_device(const rtb_context *ctx) { return ctx ? ctx->be.device() : -1; }

int rtb_build_params_default(rtb_build_params *p) {
    if (!p) return rtb::set_error(RTB_ERR_INVALID, "null");
    *p = rtb::build_defaults();
    return RTB_OK;
}
int rtb_render_params_default(rtb_render_params *p) {
    if (!p) return rtb::set_error(RTB_ERR_INVALID, "null");
    memset(p, 0, sizeof *p);
    p->width = 600; p->height = 600; p->spp = 10; p->max_bounces = 10;  // main.cu:159-170
    p->rr_start = 4; p->rr_threshold = 1.f;                               // constant.hpp:9-10
    p->seed = 1;                                                          // render.cuh:417
    return RTB_OK;
}

int rtb_scene_create(rtb_context *ctx, const rtb_scene_desc *desc, const rtb_build_params *bp, rtb_scene **out) {
    if (!ctx || !desc || !out) return rtb::set_error(RTB_ERR_INVALID, "rtb_scene_create: null argument");
    *out = nullptr;
    return rtb::guarded([&] {
        ctx->be.make_current();
        rtb_build_params p = bp ? *bp : rtb::build_defaults();
        auto *impl = rtb::scene_from_desc(ctx->be, *desc, p);
        *out = new rtb_scene{ctx, impl};
    });
}
int rtb_scene_create_from_primitives(rtb_context *ctx, const void *h_primitives, int64_t n, const void *d_triangles,
                                     const void *d_materials, int32_t num_materials, const void *d_lights,
                                     int32_t num_lights, const rtb_build_params *bp, rtb_scene **out) {
    if (!ctx || !out) return rtb::set_error(RTB_ERR_INVALID, "rtb_scene_create_from_primitives: null argument");
    *out = nullptr;
    return rtb::guarded([&] {
        ctx->be.make_current();
        rtb_build_params p = bp ? *bp : rtb::build_defaults();
        auto *impl = rtb::scene_from_primitives(ctx->be, h_primitives, n, d_triangles, d_materials, num_materials,
                                                d_lights, num_lights, p);
        *out = new rtb_scene{ctx, impl};
    });
}
int rtb_scene_attach_lights(rtb_scene *s, const void *d_lights, int32_t num_lights) {
    if (!s) return rtb::set_error(RTB_ERR_INVALID, "rtb_scene_attach_lights: null scene");
    return rtb::guarded([&] {
        s->ctx->be.make_current();
        rtb::attach_lights(s->ctx->be, *s->impl, d_lights, num_lights);
    });
}
int rtb_scene_create_instanced(rtb_context *ctx, const rtb_instanced_scene_desc *desc, const rtb_build_params *bp, rtb_scene **out) {
    if (!ctx || !desc || !out) return rtb::set_error(RTB_ERR_INVALID, "rtb_scene_create_instanced: null argument");
    *out = nullptr;
    return rtb::guarded([&] {
        ctx->be.make_current();
        rtb_build_params p = bp ? *bp : rtb::build_defaults();
        auto *impl = rtb::scene_from_instanced(ctx->be, *desc, p);
        *out = new rtb_scene{ctx, impl};
    });
}
int rtb_scene_refit(rtb_scene *s, const float *h_vertices) {
    if (!s) return rtb::set_error(RTB_ERR_INVALID, "rtb_scene_refit: null scene");
    return rtb::guarded([&] {
        s->ctx->be.make_current();
        s->ctx->be.use_stream(0);
        rtb::refit_scene(s->ctx->be, *s->impl, h_vertices, nullptr);
    });
}
int rtb_scene_refit_device(rtb_scene *s, const float *d_vertices, float *ms) {
    if (!s) return rtb::set_error(RTB_ERR_INVALID, "rtb_scene_refit_device: null scene");
    return rtb::guarded([&] {
        s->ctx->be.make_current();
        s->ctx->be.use_stream(0);
        const float e = rtb::refit_scene(s->ctx->be, *s->impl, nullptr, d_vertices);
        if (ms) *ms = e;
    });
}
int rtb_scene_set_instances(rtb_scene *s, const rtb_instance *h_instances, int32_t num_instances) {
    if (!s) return rtb::set_error(RTB_ERR_INVALID, "rtb_scene_set_instances: null scene");
    return rtb::guarded([&] {
        s->ctx->be.make_current();
        s->ctx->be.use_stream(0);
        rtb::set_instances(s->ctx->be, *s->impl, h_instances, num_instances);
    });
}
int rtb_scene_destroy(rtb_scene *s) {
    return rtb::guarded([&] {
        if (!s) return;
        s->ctx->be.make_current();
        delete s->impl;
        delete s;
    });
}
int rtb_scene_stats(const rtb_scene *s, rtb_bvh_stats *out) {
    if (!s || !out) return rtb::set_error(RTB_ERR_INVALID, "rtb_scene_stats: null");
    *out = s->impl->stats;
    return RTB_OK;
}

int rtb_trace_closest_device(rtb_scene *s, const rtb_ray *d_rays, int64_t n, rtb_hit *d_hits, float *ms) {
    if (!s || n < 0 || (n && (!d_rays || !d_hits)) || n > 0x7fffffff) return rtb::set_error(RTB_ERR_INVALID, "rtb_trace_closest_device: bad arguments");
    return rtb::guarded([&] {
        RTB_BACKEND &be = s->ctx->be;
        be.make_current();
        rtb::TraceClosestK k; k.B = s->impl->view().bvh; k.rays = d_rays; k.hits = d_hits; k.n = n; k.counts = nullptr;
        auto t0 = be.now();
        if (n) be.launch_trace((int)n, k);
        const float e = be.elapsed_ms(t0, be.now());  // also waits for the launch
        if (ms) *ms = e;
    });
}
int rtb_trace_any_device(rtb_scene *s, const rtb_ray *d_rays, const int32_t *d_excluded, int64_t n, uint8_t *d_occ, float *ms) {
    if (!s || n < 0 || (n && (!d_rays || !d_occ)) || n > 0x7fffffff) return rtb::set_error(RTB_ERR_INVALID, "rtb_trace_any_device: bad arguments");
    return rtb::guarded([&] {
        RTB_BACKEND &be = s->ctx->be;
        be.make_current();
        rtb::TraceAnyK k; k.B = s->impl->view().bvh; k.rays = d_rays; k.excluded = d_excluded;
        k.leaf_of_prim = s->impl->leaf_of_prim; k.occluded = d_occ; k.n = n;
        auto t0 = be.now();
        if (n) be.launch_trace((int)n, k);
        const float e = be.elapsed_ms(t0, be.now());  // also waits for the launch
        if (ms) *ms = e;
    });
}
int rtb_trace_closest(rtb_scene *s, const rtb_ray *h_rays, int64_t n, rtb_hit *h_hits) {
    if (!s || n < 0 || (n && (!h_rays || !h_hits)) || n > 0x7fffffff) return rtb::set_error(RTB_ERR_INVALID, "rtb_trace_closest: bad arguments");
    if (n == 0) return RTB_OK;
    return rtb::guarded([&] {
        RTB_BACKEND &be = s->ctx->be;
        be.make_current();
        rtb_ray *dr = be.template alloc<rtb_ray>((size_t)n);
        rtb_hit *dh = be.template alloc<rtb_hit>((size_t)n);
        be.upload(dr, h_rays, (size_t)n);
        int rc = rtb_trace_closest_device(s, dr, n, dh, nullptr);
        if (rc == RTB_OK) be.download(h_hits, dh, (size_t)n);
        be.free(dr); be.free(dh);
        if (rc != RTB_OK) throw rtb::Error(rc, rtb_last_error());
    });
}
int rtb_trace_any(rtb_scene *s, const rtb_ray *h_rays, const int32_t *h_excluded, int64_t n, uint8_t *h_occ) {
    if (!s || n < 0 || (n && (!h_rays || !h_occ)) || n > 0x7fffffff) return rtb::set_error(RTB_ERR_INVALID, "rtb_trace_any: bad arguments");
    if (n == 0) return RTB_OK;
    return rtb::guarded([&] {
        RTB_BACKEND &be = s->ctx->be;
        be.make_current();
        rtb_ray *dr = be.template alloc<rtb_ray>((size_t)n);
        uint8_t *dout = be.template alloc<uint8_t>((size_t)n);
        int32_t *dex = nullptr;
        be.upload(dr, h_rays, (size_t)n);
        if (h_excluded) {
            for (int64_t i = 0; i < n; ++i)
                if (h_excluded[i] >= s->impl->n_flat) { be.free(dr); be.free(dout); throw rtb::Error(RTB_ERR_INVALID, "excluded triangle out of range"); }
            dex = be.template alloc<int32_t>((size_t)n);
            be.upload(dex, h_excluded, (size_t)n);
        }
        int rc = rtb_trace_any_device(s, dr, dex, n, dout, nullptr);
        if (rc == RTB_OK) be.download(h_occ, dout, (size_t)n);
        be.free(dr); be.free(dout); be.free(dex);
        if (rc != RTB_OK) throw rtb::Error(rc, rtb_last_error());
    });
}
int rtb_trace_wavefront(rtb_scene *s, const rtb_ray *h_rays, int64_t n, rtb_hit *h_hits, const rtb_ray *h_srays,
                        const int32_t *h_excluded, int64_t ns, uint8_t *h_occ, int32_t *launches) {
    if (!s || n < 0 || ns < 0 || (n && (!h_rays || !h_hits)) || (ns && (!h_srays || !h_occ)) || n > 0x7fffff00 || ns > 0x7fffff00)
        return rtb::set_error(RTB_ERR_INVALID, "rtb_trace_wavefront: bad arguments");
    if (launches) *launches = 0;
    if (n == 0 && ns == 0) return RTB_OK;
    if (h_excluded)
        for (int64_t i = 0; i < ns; ++i)
            if (h_excluded[i] >= s->impl->n_flat) return rtb::set_error(RTB_ERR_INVALID, "excluded triangle out of range");
    return rtb::guarded([&] {
        RTB_BACKEND &be = s->ctx->be;
        be.make_current();
        rtb::DeviceBuf<RTB_BACKEND, rtb_ray> dr(be, (size_t)n), ds(be, (size_t)ns);
        rtb::DeviceBuf<RTB_BACKEND, rtb_hit> dh(be, (size_t)n);
        rtb::DeviceBuf<RTB_BACKEND, uint8_t> docc(be, (size_t)ns);
        rtb::DeviceBuf<RTB_BACKEND, int32_t> dex(be, h_excluded ? (size_t)ns : 0);
        if (n) be.upload(dr.p, h_rays, (size_t)n);
        if (ns) be.upload(ds.p, h_srays, (size_t)ns);
        if (h_excluded && ns) be.upload(dex.p, h_excluded, (size_t)ns);
        rtb::trace_wavefront(be, *s->impl, dr.p, n, dh.p, ds.p, h_excluded ? dex.p : nullptr, ns, docc.p, launches);
        if (n) be.download(h_hits, dh.p, (size_t)n);
        if (ns) be.download(h_occ, docc.p, (size_t)ns);
    });
}
int rtb_kat_eval(rtb_context *ctx, int32_t which, const float *h_in, int64_t n, float *h_out) {
    if (!ctx || which < 1 || which > 6 || n < 0 || n > (1 << 26) || (n && (!h_in || !h_out))) return rtb::set_error(RTB_ERR_INVALID, "rtb_kat_eval: bad arguments");
    if (n == 0) return RTB_OK;
    return rtb::guarded([&] {
        RTB_BACKEND &be = ctx->be;
        be.make_current();
        const size_t ni = (size_t)n * rtb::kat_in_floats(which), no = (size_t)n * rtb::kat_out_floats(which);
        rtb::DeviceBuf<RTB_BACKEND, float> din(be, ni), dout(be, no);
        be.upload(din.p, h_in, ni);
        rtb::KatK k; k.which = which; k.in = din.p; k.out = dout.p; k.n = n;
        be.launch((int)n, k);
        be.download(h_out, dout.p, no);
    });
}
int rtb_context_set_option(rtb_context *ctx, const char *name, int64_t value) {
    if (!ctx || !name) return rtb::set_error(RTB_ERR_INVALID, "rtb_context_set_option: null argument");
    return rtb::guarded([&] {
        if (!ctx->be.set_option(name, (long long)value))
            throw rtb::Error(RTB_ERR_INVALID, std::string("rtb_context_set_option: unknown option or value out of range: ") + name);
    });
}
int rtb_context_get_option(const rtb_context *ctx, const char *name, int64_t *value) {
    if (!ctx || !name || !value) return rtb::set_error(RTB_ERR_INVALID, "rtb_context_get_option: null argument");
    long long v = 0;
    if (!ctx->be.get_option(name, v)) return rtb::set_error(RTB_ERR_INVALID, "rtb_context_get_option: unknown option");
    *value = v;
    return RTB_OK;
}
int rtb_trace_closest_counts(rtb_scene *s, const rtb_ray *h_rays, int64_t n, double *nodes_per_ray, double *tris_per_ray) {
    if (!s || n <= 0 || !h_rays || n > 0x7fffffff) return rtb::set_error(RTB_ERR_INVALID, "rtb_trace_closest_counts: bad arguments");
    return rtb::guarded([&] {
        RTB_BACKEND &be = s->ctx->be;
        be.make_current();
        rtb_ray *dr = be.template alloc<rtb_ray>((size_t)n);
        rtb_hit *dh = be.template alloc<rtb_hit>((size_t)n);
        unsigned long long *dc = be.template alloc<unsigned long long>(2);
        unsigned long long z[2] = {0, 0};
        be.upload(dr, h_rays, (size_t)n);
        be.upload(dc, z, 2);
        rtb::TraceClosestK k; k.B = s->impl->view().bvh; k.rays = dr; k.hits = dh; k.n = n; k.counts = dc;
        be.launch_trace((int)n, k);
        be.download(z, dc, 2);
        be.free(dr); be.free(dh); be.free(dc);
        if (nodes_per_ray) *nodes_per_ray = (double)z[0] / (double)n;
        if (tris_per_ray) *tris_per_ray = (double)z[1] / (double)n;
    });
}

int rtb_camera_primary_rays(const rtb_camera *cam, int32_t w, int32_t h, rtb_ray *rays) {
    if (!cam || !rays || w <= 0 || h <= 0) return rtb::set_error(RTB_ERR_INVALID, "rtb_camera_primary_rays: bad arguments");
    for (int j = 0; j < h; ++j)
        for (int i = 0; i < w; ++i) {
            rtb::V3 o, d;
            rtb::camera_ray(*cam, rtb::fdiv(rtb::fadd((float)i, 0.5f), (float)w), rtb::fdiv(rtb::fadd((float)j, 0.5f), (float)h), o, d);
            rtb_ray &r = rays[(size_t)j * w + i];
            r.origin[0] = o.x; r.origin[1] = o.y; r.origin[2] = o.z;
            r.dir[0] = d.x; r.dir[1] = d.y; r.dir[2] = d.z;
            r.tmax = FLT_MAX;
        }
    return RTB_OK;
}

int rtb_render_aovs(rtb_scene *s, const rtb_camera *cam, int32_t w, int32_t h, float *h_albedo, float *h_normal, float *h_depth,
                    int32_t *h_prim) {
    if (!s || !cam || w <= 0 || h <= 0 || (int64_t)w * h > 0x7fffffff) return rtb::set_error(RTB_ERR_INVALID, "rtb_render_aovs: bad arguments");
    return rtb::guarded([&] {
        RTB_BACKEND &be = s->ctx->be;
        be.make_current();
        const size_t n = (size_t)w * (size_t)h;
        rtb::AovK k;
        k.S = s->impl->view(); k.cam = *cam; k.width = w; k.height = h;
        k.albedo = h_albedo ? be.template alloc<float>(3 * n) : nullptr;
        k.normal = h_normal ? be.template alloc<float>(3 * n) : nullptr;
        k.depth = h_depth ? be.template alloc<float>(n) : nullptr;
        k.prim = h_prim ? be.template alloc<int32_t>(n) : nullptr;
        be.launch_trace((int)n, k);
        if (h_albedo) be.download(h_albedo, k.albedo, 3 * n);
        if (h_normal) be.download(h_normal, k.normal, 3 * n);
        if (h_depth) be.download(h_depth, k.depth, n);
        if (h_prim) be.download(h_prim, k.prim, n);
        be.sync();
        be.free(k.albedo); be.free(k.normal); be.free(k.depth); be.free(k.prim);
    });
}

int rtb_render_accumulate(rtb_scene *s, const rtb_camera *cam, const rtb_render_params *p, float *d_accum, rtb_render_stats *stats) {
    if (!s || !cam || !p || !d_accum) return rtb::set_error(RTB_ERR_INVALID, "rtb_render_accumulate: null argument");
    return rtb::guarded([&] {
        s->ctx->be.make_current();
        rtb::RenderTarget t; t.add_f32 = d_accum;
        rtb::render_accumulate(s->ctx->be, *s->impl, *cam, *p, t, stats);
    });
}
int rtb_render_accumulate_fixed(rtb_scene *s, const rtb_camera *cam, const rtb_render_params *p, int64_t *d_accum, rtb_render_stats *stats) {
    if (!s || !cam || !p || !d_accum) return rtb::set_error(RTB_ERR_INVALID, "rtb_render_accumulate_fixed: null argument");
    return rtb::guarded([&] {
        s->ctx->be.make_current();
        rtb::RenderTarget t; t.add_fixed = (long long *)d_accum;
        rtb::render_accumulate(s->ctx->be, *s->impl, *cam, *p, t, stats);
    });
}
int rtb_tonemap_device(rtb_context *ctx, const float *d_accum, int64_t n, int32_t total_spp, float *d_out) {
    if (!ctx || !d_accum || !d_out) return rtb::set_error(RTB_ERR_INVALID, "rtb_tonemap_device: null argument");
    return rtb::guarded([&] {
        ctx->be.make_current();
        rtb::tonemap(ctx->be, d_accum, n, total_spp, d_out);
        ctx->be.sync();
    });
}
int rtb_tonemap_fixed_device(rtb_context *ctx, const int64_t *d_accum, int64_t n, int32_t total_spp, float *d_out) {
    if (!ctx || !d_accum || !d_out) return rtb::set_error(RTB_ERR_INVALID, "rtb_tonemap_fixed_device: null argument");
    return rtb::guarded([&] {
        ctx->be.make_current();
        rtb::tonemap_fixed(ctx->be, (const long long *)d_accum, n, total_spp, d_out);
        ctx->be.sync();
    });
}
int rtb_render(rtb_scene *s, const rtb_camera *cam, const rtb_render_params *p, float *h_rgb, rtb_render_stats *stats) {
    if (!s || !cam || !p || !h_rgb) return rtb::set_error(RTB_ERR_INVALID, "rtb_render: null argument");
    return rtb::guarded([&] {
        RTB_BACKEND &be = s->ctx->be;
        be.make_current();
        auto &sc = *s->impl;
        const int64_t nf = 3 * (int64_t)p->width * (int64_t)p->height;
        if (p->width <= 0 || p->height <= 0 || nf > 0x7fffff00ll) throw rtb::Error(RTB_ERR_INVALID, "rtb_render: bad image size");
        if (sc.own_out_floats != nf) {
            be.free(sc.own_out);
            sc.own_out = nullptr; sc.own_out_floats = 0;
            sc.own_out = be.template alloc<float>((size_t)nf);
            sc.own_out_floats = nf;
        }
        rtb::RenderTarget t; t.tonemap_to = sc.own_out; t.tonemap_spp = p->total_spp > 0 ? p->total_spp : p->spp;
        rtb::render_accumulate(be, sc, *cam, *p, t, stats);
        be.download(h_rgb, sc.own_out, (size_t)nf);  // render.cuh:455-456
    });
}

}  // extern "C"

// ---------------------------------------------------------------- progressive rendering / checkpoints (rtb_accum)
struct rtb_accum {
    rtb_context *ctx = nullptr;
    int32_t width = 0, height = 0, samples = 0;
    bool fixed = false;
    float *sum_f32 = nullptr;      // float[3 * W * H]
    long long *sum_fixed = nullptr;  // int64[3 * W * H], units of 2^-28
    int64_t values() const { return 3 * (int64_t)width * height; }
};
namespace rtb {
struct AccumFileHeader {  // "RTBA", version 1
    uint32_t magic, version;
    int32_t width, height, samples, fixed;
};
inline rtb_accum *accum_new(rtb_context *ctx, int32_t w, int32_t h, bool fixed) {
    if (!ctx || w <= 0 || h <= 0 || 3 * (int64_t)w * h > 0x7fffff00ll) throw Error(RTB_ERR_INVALID, "rtb_accum: bad image size");
    std::unique_ptr<rtb_accum> a(new rtb_accum());
    a->ctx = ctx; a->width = w; a->height = h; a->fixed = fixed;
    RTB_BACKEND &be = ctx->be;
    be.make_current();
    be.use_stream(0);
    if (fixed) { a->sum_fixed = be.template alloc<long long>((size_t)a->values()); be.zero(a->sum_fixed, (size_t)a->values()); }
    else { a->sum_f32 = be.template alloc<float>((size_t)a->values()); be.zero(a->sum_f32, (size_t)a->values()); }
    be.sync();
    return a.release();
}
}  // namespace rtb

extern "C" {
int rtb_accum_create(rtb_context *ctx, int32_t w, int32_t h, int32_t deterministic, rtb_accum **out) {
    if (!out) return rtb::set_error(RTB_ERR_INVALID, "rtb_accum_create: null out");
    *out = nullptr;
    return rtb::guarded([&] { *out = rtb::accum_new(ctx, w, h, deterministic != 0); });
}
int rtb_accum_destroy(rtb_accum *a) {
    return rtb::guarded([&] {
        if (!a) return;
        a->ctx->be.make_current();
        a->ctx->be.free(a->sum_f32); a->ctx->be.free(a->sum_fixed);
        delete a;
    });
}
int rtb_accum_samples(const rtb_accum *a) { return a ? a->samples : 0; }
int rtb_accum_add_samples(rtb_accum *a, rtb_scene *s, const rtb_camera *cam, const rtb_render_params *p, rtb_render_stats *stats) {
    if (!a || !s || !cam || !p) return rtb::set_error(RTB_ERR_INVALID, "rtb_accum_add_samples: null argument");
    if (s->ctx != a->ctx) return rtb::set_error(RTB_ERR_INVALID, "rtb_accum_add_samples: scene and buffer belong to different contexts");
    if (p->width != a->width || p->height != a->height) return rtb::set_error(RTB_ERR_INVALID, "rtb_accum_add_samples: image size differs from the buffer's");
    return rtb::guarded([&] {
        RTB_BACKEND &be = a->ctx->be;
        be.make_current();
        rtb_render_params q = *p;
        q.first_sample = a->samples;
        q.total_spp = 0;
        if (a->fixed) q.flags |= RTB_RENDER_DETERMINISTIC;
        rtb::RenderTarget t;
        if (a->fixed) t.add_fixed = a->sum_fixed; else t.add_f32 = a->sum_f32;
        rtb::render_accumulate(be, *s->impl, *cam, q, t, stats);
        a->samples += p->spp;
    });
}
int rtb_accum_resolve(rtb_accum *a, float *h_rgb) {
    if (!a || !h_rgb) return rtb::set_error(RTB_ERR_INVALID, "rtb_accum_resolve: null argument");
    if (a->samples <= 0) return rtb::set_error(RTB_ERR_INVALID, "rtb_accum_resolve: no samples yet");
    return rtb::guarded([&] {
        RTB_BACKEND &be = a->ctx->be;
        be.make_current();
        be.use_stream(0);
        rtb::DeviceBuf<RTB_BACKEND, float> out(be, (size_t)a->values());
        if (a->fixed) rtb::tonemap_fixed(be, a->sum_fixed, a->values(), a->samples, out.p);
        else rtb::tonemap(be, a->sum_f32, a->values(), a->samples, out.p);
        be.download(h_rgb, out.p, (size_t)a->values());
    });
}
int rtb_accum_save(rtb_accum *a, const char *path) {
    if (!a || !path) return rtb::set_error(RTB_ERR_INVALID, "rtb_accum_save: null argument");
    return rtb::guarded([&] {
        RTB_BACKEND &be = a->ctx->be;
        be.make_current();
        be.use_stream(0);
        const size_t bytes = (size_t)a->values() * (a->fixed ? 8 : 4);
        std::vector<char> host(bytes);
        be.download(host.data(), a->fixed ? (const char *)a->sum_fixed : (const char *)a->sum_f32, bytes);
        rtb::AccumFileHeader h{0x41425452u, 1u, a->width, a->height, a->samples, a->fixed ? 1 : 0};
        FILE *f = fopen(path, "wb");
        if (!f) throw rtb::Error(RTB_ERR_IO, std::string("cannot write ") + path);
        const bool ok = fwrite(&h, sizeof h, 1, f) == 1 && fwrite(host.data(), 1, bytes, f) == bytes;
        if (fclose(f) != 0 || !ok) throw rtb::Error(RTB_ERR_IO, std::string("short write to ") + path);
    });
}
int rtb_accum_load(rtb_context *ctx, const char *path, rtb_accum **out) {
    if (!ctx || !path || !out) return rtb::set_error(RTB_ERR_INVALID, "rtb_accum_load: null argument");
    *out = nullptr;
    return rtb::guarded([&] {
        FILE *f = fopen(path, "rb");
        if (!f) throw rtb::Error(RTB_ERR_IO, std::string("cannot open ") + path);
        rtb::AccumFileHeader h;
        bool ok = fread(&h, sizeof h, 1, f) == 1 && h.magic == 0x41425452u && h.version == 1u && h.width > 0 && h.height > 0 && h.samples >= 0 &&
                  (h.fixed == 0 || h.fixed == 1) && 3 * (int64_t)h.width * h.height <= 0x7fffff00ll;
        std::vector<char> host;
        if (ok) {
            const size_t bytes = (size_t)(3 * (int64_t)h.width * h.height) * (h.fixed ? 8 : 4);
            long here = ftell(f);
            fseek(f, 0, SEEK_END);
            ok = (size_t)(ftell(f) - here) == bytes;  // the header must match the file before anything is sized from it
            fseek(f, here, SEEK_SET);
            if (ok) { host.resize(bytes); ok = fread(host.data(), 1, bytes, f) == bytes; }
        }
        fclose(f);
        if (!ok) throw rtb::Error(RTB_ERR_IO, std::string("not an accumulation checkpoint (or truncated): ") + path);
        std::unique_ptr<rtb_accum> a(rtb::accum_new(ctx, h.width, h.height, h.fixed != 0));
        a->samples = h.samples;
        RTB_BACKEND &be = ctx->be;
        be.upload(a->fixed ? (char *)a->sum_fixed : (char *)a->sum_f32, (const char *)host.data(), host.size());
        *out = a.release();
    });
}
}  // extern "C"

// ---------------------------------------------------------------- several GPUs, one process (rtb_multi)
struct rtb_multi {
    std::vector<rtb_context *> ctx;
    // communicators by device mask (bit i = member i): ncclCommInitAll over exactly the GPUs a render uses
    std::map<uint32_t, RTB_BACKEND::Group *> groups;
    RTB_BACKEND::Group *group_for(uint32_t mask, const std::vector<int> &sel) {
        auto it = groups.find(mask);
        if (it != groups.end()) return it->second;
        std::vector<RTB_BACKEND *> members;
        for (int i : sel) members.push_back(&ctx[(size_t)i]->be);
        RTB_BACKEND::Group *g = RTB_BACKEND::group_create(members);
        groups[mask] = g;
        return g;
    }
    ~rtb_multi() {
        for (auto &kv : groups) RTB_BACKEND::group_destroy(kv.second);
        for (rtb_context *c : ctx) delete c;
    }
};
struct rtb_multi_scene {
    rtb_multi *m = nullptr;
    std::vector<rtb_scene *> sc;     // one per member of m
    bool owns_first = true;          // false: sc[0] is the caller's (rtb_multi_scene_replicate)
    // per-GPU sums of the last render (float[3WH] or int64[3WH]) and the root's tonemapped image
    std::vector<float *> sum_f32; std::vector<long long *> sum_fixed; int64_t sum_values = 0; bool sum_is_fixed = false;
    float *root_out = nullptr; int64_t root_out_values = 0;
    void free_sums() {
        for (size_t i = 0; i < sum_f32.size(); ++i) { m->ctx[i]->be.make_current(); m->ctx[i]->be.free(sum_f32[i]); sum_f32[i] = nullptr; }
        for (size_t i = 0; i < sum_fixed.size(); ++i) { m->ctx[i]->be.make_current(); m->ctx[i]->be.free(sum_fixed[i]); sum_fixed[i] = nullptr; }
        sum_values = 0;
    }
    ~rtb_multi_scene() {
        if (!m) return;
        free_sums();
        if (root_out) { m->ctx[0]->be.make_current(); m->ctx[0]->be.free(root_out); }
        for (size_t i = 0; i < sc.size(); ++i) {
            if (!sc[i] || (i == 0 && !owns_first)) continue;
            m->ctx[i]->be.make_current();
            delete sc[i]->impl;
            delete sc[i];
        }
    }
};
struct rtb_comm {
    rtb_context *ctx;
    RTB_BACKEND::Comm *impl;
};

namespace rtb {
// run f(i) for i in [0, n) on n host threads (one per GPU); the first error, if any, is rethrown on the caller's thread
template <class F>
void for_each_gpu(int n, F f) {
    std::vector<std::thread> th;
    std::vector<int> code((size_t)n, 0);
    std::vector<std::string> msg((size_t)n);
    for (int i = 0; i < n; ++i)
        th.emplace_back([&, i] {
            try { f(i); }
            catch (const Error &e) { code[(size_t)i] = e.code; msg[(size_t)i] = e.what(); }
            catch (const std::bad_alloc &) { code[(size_t)i] = RTB_ERR_OOM; msg[(size_t)i] = "out of host memory"; }
            catch (const std::exception &e) { code[(size_t)i] = RTB_ERR_CUDA; msg[(size_t)i] = e.what(); }
        });
    for (auto &t : th) t.join();
    for (int i = 0; i < n; ++i)
        if (code[(size_t)i]) throw Error(code[(size_t)i], "GPU " + std::to_string(i) + " of the rtb_multi: " + msg[(size_t)i]);
}
inline void multi_render(rtb_multi_scene &ms, const rtb_camera &cam, const rtb_render_params &p, float *h_rgb, rtb_render_stats *stats) {
    rtb_multi &m = *ms.m;
    const int n = (int)m.ctx.size();
    if (p.width <= 0 || p.height <= 0 || p.spp <= 0) throw Error(RTB_ERR_INVALID, "rtb_multi_render: bad parameters");
    std::vector<int> sel;
    for (int i = 0; i < n; ++i) if (p.device_mask == 0 || (p.device_mask >> i & 1u)) sel.push_back(i);
    if (sel.empty() || (n < 32 && (p.device_mask >> n) != 0)) throw Error(RTB_ERR_INVALID, "rtb_multi_render: device_mask selects no GPU of this rtb_multi");
    uint32_t mask = 0;
    for (int i : sel) mask |= 1u << i;
    const int ns = (int)sel.size(), root = sel[0];
    const bool fixed = (p.flags & RTB_RENDER_DETERMINISTIC) != 0;
    const int64_t values = 3 * (int64_t)p.width * (int64_t)p.height;
    if (values > 0x7fffff00ll) throw Error(RTB_ERR_INVALID, "rtb_multi_render: image too large");
    if (ms.sum_values != values || ms.sum_is_fixed != fixed) {
        ms.free_sums();
        ms.sum_f32.assign((size_t)n, nullptr); ms.sum_fixed.assign((size_t)n, nullptr);
        ms.sum_values = values; ms.sum_is_fixed = fixed;
    }
    const int total_spp = p.total_spp > 0 ? p.total_spp : p.spp;
    std::vector<rtb_render_stats> st((size_t)ns);
    auto wall0 = std::chrono::steady_clock::now();
    for_each_gpu(ns, [&](int k) {
        const int i = sel[(size_t)k];
        RTB_BACKEND &be = m.ctx[(size_t)i]->be;
        be.make_current();
        be.use_stream(0);
        if (fixed) { if (!ms.sum_fixed[(size_t)i]) ms.sum_fixed[(size_t)i] = be.template alloc<long long>((size_t)values); be.zero(ms.sum_fixed[(size_t)i], (size_t)values); }
        else { if (!ms.sum_f32[(size_t)i]) ms.sum_f32[(size_t)i] = be.template alloc<float>((size_t)values); be.zero(ms.sum_f32[(size_t)i], (size_t)values); }
        int first = 0, count = 0;
        shard_samples(p.spp, k, ns, first, count);
        memset(&st[(size_t)k], 0, sizeof(rtb_render_stats));
        if (count > 0) {
            rtb_render_params q = p;
            q.spp = count; q.first_sample = p.first_sample + first; q.total_spp = total_spp; q.device_mask = 0;
            RenderTarget t;
            if (fixed) t.add_fixed = ms.sum_fixed[(size_t)i]; else t.add_f32 = ms.sum_f32[(size_t)i];
            render_accumulate(be, *ms.sc[(size_t)i]->impl, cam, q, t, &st[(size_t)k]);
        }
        be.sync();
    });
    // one sum-reduction to the first selected GPU (NVLink), then post_process_framebuffer there
    RTB_BACKEND &rb = m.ctx[(size_t)root]->be;
    rb.make_current();
    rb.use_stream(0);
    auto t0 = rb.now();
    if (ns > 1) {
        RTB_BACKEND::Group *g = m.group_for(mask, sel);
        std::vector<RTB_BACKEND *> members;
        for (int i : sel) members.push_back(&m.ctx[(size_t)i]->be);
        if (fixed) { std::vector<long long *> b; for (int i : sel) b.push_back(ms.sum_fixed[(size_t)i]); RTB_BACKEND::group_reduce(g, members, b, (size_t)values, 0); }
        else { std::vector<float *> b; for (int i : sel) b.push_back(ms.sum_f32[(size_t)i]); RTB_BACKEND::group_reduce(g, members, b, (size_t)values, 0); }
        rb.make_current();
    }
    if (ms.root_out && ms.root_out_values != values) {  // (kept between renders on GPU 0, the usual root)
        m.ctx[0]->be.make_current(); m.ctx[0]->be.free(ms.root_out); ms.root_out = nullptr; rb.make_current();
    }
    float *out = nullptr;
    DeviceBuf<RTB_BACKEND, float> tmp(rb, root != 0 ? (size_t)values : 0);
    if (root == 0) {
        if (!ms.root_out) { ms.root_out = rb.template alloc<float>((size_t)values); ms.root_out_values = values; }
        out = ms.root_out;
    } else out = tmp.p;
    if (fixed) tonemap_fixed(rb, ms.sum_fixed[(size_t)root], values, total_spp, out);
    else tonemap(rb, ms.sum_f32[(size_t)root], values, total_spp, out);
    rb.download(h_rgb, out, (size_t)values);
    const float ms_tail = rb.elapsed_ms(t0, rb.now());
    if (stats) {
        memset(stats, 0, sizeof *stats);
        float slowest = 0.f;
        for (const rtb_render_stats &s : st) {
            stats->paths += s.paths; stats->extend_rays += s.extend_rays; stats->shadow_rays += s.shadow_rays;
            stats->iterations += s.iterations; stats->kernel_launches += s.kernel_launches; stats->hits += s.hits;
            stats->extend_launches += s.extend_launches; stats->shadow_launches += s.shadow_launches;
            if (s.ms_total > slowest) slowest = s.ms_total;
            stats->fused_trace = s.fused_trace; stats->pipelines = s.pipelines;
        }
        stats->ms_total = slowest + ms_tail;
        stats->ms_other = ms_tail;  // reduce + tonemap + device->host copy
        (void)wall0;
    }
}
}  // namespace rtb

extern "C" {

int rtb_multi_create(const int32_t *devices, int32_t n, rtb_multi **out) {
    if (!out || !devices || n <= 0 || n > 32) return rtb::set_error(RTB_ERR_INVALID, "rtb_multi_create: bad arguments");
    *out = nullptr;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j] && devices[i] >= 0) return rtb::set_error(RTB_ERR_INVALID, "rtb_multi_create: a device is listed twice");
    return rtb::guarded([&] {
        std::unique_ptr<rtb_multi> m(new rtb_multi());
        for (int i = 0; i < n; ++i) m->ctx.push_back(new rtb_context(devices[i]));
        *out = m.release();
    });
}
int rtb_multi_destroy(rtb_multi *m) {
    return rtb::guarded([&] { delete m; });
}
int rtb_multi_size(const rtb_multi *m) { return m ? (int)m->ctx.size() : 0; }
int rtb_multi_context(rtb_multi *m, int32_t i, rtb_context **ctx) {
    if (!m || !ctx || i < 0 || i >= (int)m->ctx.size()) return rtb::set_error(RTB_ERR_INVALID, "rtb_multi_context: bad arguments");
    *ctx = m->ctx[(size_t)i];
    return RTB_OK;
}
static int multi_scene_build(rtb_multi *m, rtb_multi_scene **out, const std::function<rtb::SceneT<RTB_BACKEND> *(RTB_BACKEND &)> &make) {
    *out = nullptr;
    return rtb::guarded([&] {
        std::unique_ptr<rtb_multi_scene> ms(new rtb_multi_scene());
        ms->m = m;
        ms->sc.assign(m->ctx.size(), nullptr);
        rtb::for_each_gpu((int)m->ctx.size(), [&](int i) {
            RTB_BACKEND &be = m->ctx[(size_t)i]->be;
            be.make_current();
            be.use_stream(0);
            ms->sc[(size_t)i] = new rtb_scene{m->ctx[(size_t)i], make(be)};
        });
        *out = ms.release();
    });
}
int rtb_multi_scene_create(rtb_multi *m, const rtb_scene_desc *desc, const rtb_build_params *bp, rtb_multi_scene **out) {
    if (!m || !desc || !out) return rtb::set_error(RTB_ERR_INVALID, "rtb_multi_scene_create: null argument");
    const rtb_build_params p = bp ? *bp : rtb::build_defaults();
    return multi_scene_build(m, out, [&](RTB_BACKEND &be) { return rtb::scene_from_desc(be, *desc, p); });
}
int rtb_multi_scene_create_instanced(rtb_multi *m, const rtb_instanced_scene_desc *desc, const rtb_build_params *bp, rtb_multi_scene **out) {
    if (!m || !desc || !out) return rtb::set_error(RTB_ERR_INVALID, "rtb_multi_scene_create_instanced: null argument");
    const rtb_build_params p = bp ? *bp : rtb::build_defaults();
    return multi_scene_build(m, out, [&](RTB_BACKEND &be) { return rtb::scene_from_instanced(be, *desc, p); });
}
int rtb_multi_scene_replicate(rtb_multi *m, rtb_scene *primary, rtb_multi_scene **out) {
    if (!m || !primary || !out) return rtb::set_error(RTB_ERR_INVALID, "rtb_multi_scene_replicate: null argument");
    *out = nullptr;
    if (primary->ctx != m->ctx[0]) return rtb::set_error(RTB_ERR_INVALID, "rtb_multi_scene_replicate: the scene must belong to context 0 of the rtb_multi");
    return rtb::guarded([&] {
        std::unique_ptr<rtb_multi_scene> ms(new rtb_multi_scene());
        ms->m = m;
        ms->owns_first = false;
        ms->sc.assign(m->ctx.size(), nullptr);
        ms->sc[0] = primary;
        primary->ctx->be.make_current();
        primary->ctx->be.sync();
        rtb::for_each_gpu((int)m->ctx.size() - 1, [&](int k) {
            const int i = k + 1;
            RTB_BACKEND &be = m->ctx[(size_t)i]->be;
            be.make_current();
            be.use_stream(0);
            ms->sc[(size_t)i] = new rtb_scene{m->ctx[(size_t)i], rtb::clone_scene(be, primary->ctx->be, *primary->impl)};
        });
        *out = ms.release();
    });
}
int rtb_multi_scene_destroy(rtb_multi_scene *ms) {
    return rtb::guarded([&] { delete ms; });
}
int rtb_multi_render(rtb_multi_scene *ms, const rtb_camera *cam, const rtb_render_params *p, float *h_rgb, rtb_render_stats *stats) {
    if (!ms || !cam || !p || !h_rgb) return rtb::set_error(RTB_ERR_INVALID, "rtb_multi_render: null argument");
    return rtb::guarded([&] { rtb::multi_render(*ms, *cam, *p, h_rgb, stats); });
}
int rtb_render_multi(const int32_t *devices, int32_t n, const rtb_scene_desc *desc, const rtb_build_params *bp, const rtb_camera *cam,
                     const rtb_render_params *p, float *h_rgb, rtb_render_stats *stats) {
    rtb_multi *m = nullptr;
    rtb_multi_scene *ms = nullptr;
    int rc = rtb_multi_create(devices, n, &m);
    if (rc == RTB_OK) rc = rtb_multi_scene_create(m, desc, bp, &ms);
    if (rc == RTB_OK) rc = rtb_multi_render(ms, cam, p, h_rgb, stats);
    const std::string err = rc != RTB_OK ? rtb_last_error() : "";
    if (ms) rtb_multi_scene_destroy(ms);
    if (m) rtb_multi_destroy(m);
    return rc != RTB_OK ? rtb::set_error(rc, err) : RTB_OK;
}

int rtb_comm_unique_id(uint8_t *id_out) {
    if (!id_out) return rtb::set_error(RTB_ERR_INVALID, "rtb_comm_unique_id: null argument");
    return rtb::guarded([&] { RTB_BACKEND::comm_unique_id(id_out); });
}
int rtb_comm_create(rtb_context *ctx, const uint8_t *id, int32_t rank, int32_t world, rtb_comm **out) {
    if (!ctx || !id || !out || world <= 0 || rank < 0 || rank >= world) return rtb::set_error(RTB_ERR_INVALID, "rtb_comm_create: bad arguments");
    *out = nullptr;
    return rtb::guarded([&] { *out = new rtb_comm{ctx, ctx->be.comm_create(id, rank, world)}; });
}
int rtb_comm_destroy(rtb_comm *c) {
    return rtb::guarded([&] {
        if (!c) return;
        c->ctx->be.make_current();
        RTB_BACKEND::comm_destroy(c->impl);
        delete c;
    });
}
int rtb_comm_allreduce_f32(rtb_comm *c, float *d_buf, int64_t n) {
    if (!c || !d_buf || n <= 0) return rtb::set_error(RTB_ERR_INVALID, "rtb_comm_allreduce_f32: bad arguments");
    return rtb::guarded([&] { c->ctx->be.make_current(); c->ctx->be.comm_allreduce(c->impl, d_buf, (size_t)n); });
}
int rtb_comm_allreduce_i64(rtb_comm *c, int64_t *d_buf, int64_t n) {
    if (!c || !d_buf || n <= 0) return rtb::set_error(RTB_ERR_INVALID, "rtb_comm_allreduce_i64: bad arguments");
    return rtb::guarded([&] { c->ctx->be.make_current(); c->ctx->be.comm_allreduce(c->impl, (long long *)d_buf, (size_t)n); });
}

}  // extern "C"
