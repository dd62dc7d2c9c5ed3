/*
 * rtb.h — C ABI of the B200-native wavefront path tracer (rtcuda_b200).
 *
 * This is the drop-in boundary for the render path of lashhw/rtcuda.  Every
 * entry point cites the reference interface (file:line, relative to the
 * reference repo) that it replaces.  Signatures carry plain pointers and
 * sizes only; there are no C++ or torch types on this boundary.
 *
 * Conventions
 *   - every function returns RTB_OK (0) or a negative rtb_status; it never
 *     exits or throws across the boundary (the reference's CHECK_CUDA exits,
 *     utility.cuh:4-13).  rtb_last_error() returns a thread-local message.
 *   - "h_" pointers are host memory, "d_" pointers are device memory of the
 *     context's GPU.
 *   - struct layouts marked [ref layout] are byte-compatible with the
 *     reference structs so that reference-side host code can pass its own
 *     arrays without conversion.
 */
#ifndef RTB_H
#define RTB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTB_API __attribute__((visibility("default")))

typedef enum rtb_status {
    RTB_OK = 0,
    RTB_ERR_INVALID = -1,   /* bad argument */
    RTB_ERR_CUDA = -2,      /* CUDA runtime error, see rtb_last_error() */
    RTB_ERR_NO_DEVICE = -3, /* no usable sm_100 device: the library has NO CPU fallback */
    RTB_ERR_IO = -4,
    RTB_ERR_OOM = -5
} rtb_status;

/* material.cuh:4-8, plus RTB_GLOSSY which the reference does not have (SURVEY 8f-3 "a real glossy BSDF"): an
 * energy-normalised Phong lobe around the mirror direction, albedo = specular colour, `ior` = Phong exponent */
enum { RTB_MATTE = 0, RTB_MIRROR = 1, RTB_GLASS = 2, RTB_GLOSSY = 3 };
/* light.cuh:4-7 */
enum { RTB_POINT_LIGHT = 0, RTB_AREA_LIGHT = 1 };

/* [ref layout] Material, material.cuh:10-25 (20 B: albedo@0, ior@12, type@16) */
typedef struct rtb_material {
    float albedo[3];
    float ior;
    int32_t type;
} rtb_material;

/* Light, light.cuh:9-28.  Same 40-byte footprint; the reference's
 * `Triangle *d_triangle` (offset 16) is replaced by the triangle's index in
 * the scene's triangle list (the pointer form is accepted by
 * rtb_scene_create_from_primitives). */
typedef struct rtb_light {
    int32_t type;
    float pos[3];      /* point light position */
    int64_t triangle;  /* area light: index of its triangle */
    float L[3];        /* radiance (area) / intensity (point) */
    int32_t _pad;
} rtb_light;

/* [ref layout] Camera, camera.cuh:4-13 (48 B) */
typedef struct rtb_camera {
    float lookfrom[3];
    float upper_left[3];
    float horizontal[3];
    float vertical[3];
} rtb_camera;

/* [ref layout] Ray, ray.cuh:4-18 (28 B) */
typedef struct rtb_ray {
    float origin[3];
    float dir[3]; /* unit length */
    float tmax;
} rtb_ray;

/* Intersection (intersection.hpp:4-6) + hit primitive.  `prim` is the index
 * of the triangle in the caller's triangle list (== d_triangle - d_triangles
 * in the reference), or -1 for a miss (then t,u,v are 0). */
typedef struct rtb_hit {
    float t, u, v;
    int32_t prim;
} rtb_hit;

/* Flat scene description (host memory).  Triangles are given as vertices;
 * {p0, e1=p0-p1, e2=p2-p0, n=cross(e1,e2)} are derived without FMA
 * contraction exactly like the reference's host constructor
 * (triangle.cuh:6-7 run from main.cu:80). */
typedef struct rtb_scene_desc {
    int64_t num_triangles;
    const float *vertices;       /* 9 floats per triangle: p0 p1 p2 */
    const int32_t *material_ids; /* per triangle, index into materials */
    const int32_t *light_ids;    /* per triangle, index into lights or -1 (Primitive::d_area_light) */
    int32_t num_materials;
    const rtb_material *materials;
    int32_t num_lights;
    const rtb_light *lights;
} rtb_scene_desc;

/* ---- instanced scenes: a two-level BVH (SURVEY 8f-2 "instancing: two-level BVH instead of flattening").  The
 * reference has no instancing — main.cu:67-86 transforms every vertex on the host and Bvh::Bvh takes the flat list —
 * so this is a second INPUT FORMAT for the same path: `geometry` holds the triangles of all meshes in object space,
 * mesh m = triangles [mesh_first[m], mesh_first[m+1]), and every instance places one mesh with an affine transform.
 * One 8-wide BVH is built per mesh, one over the instances' world boxes; a ray is taken into object space when it
 * enters an instance (same parameter t, so hit distances compare directly).  A 10 M-triangle field of 144 bunnies is
 * then 4 MB of nodes + triangles (L2-resident) instead of 600 MB.
 * Results are those of the flattened scene (rtb_instanced_flatten) up to the rounding of the ray transform:
 * hit ids equal except on near-ties, t within 1e-5 relative (tests/test_instancing.py).
 * Hit ids (rtb_hit.prim, rtb_trace_any's excluded, AOV prim) number the triangles of the FLATTENED scene: instance
 * i owns [sum of the mesh sizes of instances 0..i-1, ... + its own mesh size).
 * Restriction: a triangle with light_ids >= 0 must belong to a mesh that is instanced exactly once, with the
 * identity transform (emitters live in the static part of the scene). */
typedef struct rtb_instance {
    int32_t mesh;      /* index into the mesh table */
    int32_t material;  /* material of every triangle of this instance, or -1: the triangles' own material_ids */
    float xform[12];   /* object -> world, row-major 3x4: world = xform[:, :3] * p + xform[:, 3]; must be invertible */
} rtb_instance;

typedef struct rtb_instanced_scene_desc {
    rtb_scene_desc geometry;    /* all meshes, object space; materials; lights (triangle = index into geometry) */
    int32_t num_meshes;
    const int64_t *mesh_first;  /* [num_meshes + 1], ascending, mesh_first[0] = 0, mesh_first[num_meshes] = num_triangles */
    int32_t num_instances;
    const rtb_instance *instances;
} rtb_instanced_scene_desc;

/* BVH builder selection (rtb_build_params.builder) */
enum {
    RTB_BUILDER_PLOC = 0,       /* parallel locally-ordered clustering over Morton order (default) */
    RTB_BUILDER_BINNED_SAH = 1  /* top-down binned SAH (32 bins per axis, split down to single primitives): a tree
                                   for faster traces at a longer build time; ploc_radius is ignored, ploc_iterations
                                   is 0.  Exact-t ties at shared edges can resolve differently from the reference, as
                                   with RTB_COLLAPSE_SAH_OPTIMAL (DESIGN.md 4.1) */
};
/* Treelet restructuring of the binary tree after the builder, k = 0..8 passes, or-ed into the builder value:
   bp.builder = RTB_BUILDER_PLOC | RTB_BUILDER_TREELET_PASSES(3).  One pass visits the inner nodes bottom-up; each node
   with enough triangles below it (7 in the first pass, doubling with every pass) is the root of a treelet of up to 7
   subtrees, which is rewired into the binary topology over them with the lowest total surface area (Karras & Aila
   2013).  Works with both builders and both collapse modes; k = 0 is the plain builder.  Costs build time and gives a
   lower SAH cost; exact-t ties at shared edges can resolve differently from the reference, as with
   RTB_COLLAPSE_SAH_OPTIMAL (DESIGN.md 4.1).  Other bits of rtb_build_params.builder must be zero. */
#define RTB_BUILDER_TREELET_PASSES(k) ((k) << 8)

/* how the binary tree is collapsed into 8-wide nodes (rtb_build_params.collapse) */
enum {
    RTB_COLLAPSE_LARGEST_FIRST = 0, /* greedy: open the child with the largest surface area until 8 children (default) */
    RTB_COLLAPSE_SAH_OPTIMAL = 1    /* dynamic programme: cheapest layout of every subtree in 1..7 child slots; a third
                                       fewer nodes, 0-3 % faster renders, but exact-t ties at shared edges then resolve
                                       differently from the reference on 48 rays of the golden fixture (DESIGN.md 4.1) */
};

typedef struct rtb_build_params {
    int32_t builder;      /* RTB_BUILDER_*, | RTB_BUILDER_TREELET_PASSES(k) */
    int32_t ploc_radius;  /* nearest-neighbour search radius, 0 = default (16) */
    int32_t max_leaf_tris;/* 1..3, 0 = default (3) */
    int32_t collapse;     /* RTB_COLLAPSE_* */
} rtb_build_params;

typedef struct rtb_bvh_stats {
    int64_t num_triangles;
    int64_t num_bvh2_nodes;
    int64_t num_nodes;        /* 80-byte 8-wide nodes */
    int64_t node_bytes;
    int64_t triangle_bytes;
    float sah_cost;           /* SAH cost of the 8-wide tree (Cn=1, Ct=0.3) */
    float build_ms;           /* GPU build time, CUDA events */
    int32_t ploc_iterations;
    int32_t collapse_levels;
    float scene_bounds[6];    /* xmin xmax ymin ymax zmin zmax */
    /* instanced scenes (0 otherwise): num_triangles / num_nodes above count what is STORED (all mesh trees + the
     * tree over the instances) */
    int64_t num_instances;
    int64_t num_flat_triangles; /* triangles of the flattened scene the description stands for */
    int64_t num_top_nodes;      /* 8-wide nodes of the tree over the instances (the first nodes of the array) */
} rtb_bvh_stats;

/* Runtime replacement of the reference's compile-time constants
 * (constant.hpp:4-10, render.cuh:413-417, main.cu:159-170). */
typedef struct rtb_render_params {
    int32_t width, height;
    int32_t spp;            /* samples rendered by THIS call */
    int32_t max_bounces;    /* MAX_BOUNCES, main.cu:170 */
    int32_t rr_start;       /* RR_START, constant.hpp:10 (default 4) */
    float rr_threshold;     /* RR_THRESHOLD, constant.hpp:9 (default 1) */
    uint32_t seed;          /* RAND_SEED, render.cuh:417 (default 1) */
    int32_t first_sample;   /* index of the first sample of this call (sample-pass sharding) */
    int32_t total_spp;      /* divisor used by the tonemap; 0 means spp */
    int32_t pool_size;      /* path slots (NUM_WORKING_PATHS, constant.hpp:8); 0 = the context's "pool" option */
    int32_t flags;          /* RTB_RENDER_* */
    uint32_t device_mask;   /* rtb_multi_render: bit i set = use GPU i of the rtb_multi; 0 = all of them.  rtb_render /
                               rtb_render_accumulate run on the one GPU of the scene's context and reject a mask without it */
    float env_L[3];         /* radiance of a constant environment seen by rays that leave the scene (the reference's
                               TODO at render.cuh:105,243,325); (0,0,0) = none, as in the reference */
    int32_t _reserved2;
} rtb_render_params;

enum {
    RTB_RENDER_DEFAULT = 0,
    RTB_RENDER_PIXEL_CENTRE = 1, /* no sub-pixel jitter: camera rays through pixel centres */
    RTB_RENDER_NO_SHADOW = 2,    /* skip next-event estimation (debug) */
    RTB_RENDER_NONPERSISTENT = 4, /* one-thread-per-ray traversal launch (A/B for the persistent kernel) */
    RTB_RENDER_COUNT_WORK = 8,    /* counting kernel variants: fill the *_nodes / *_tris statistics (slower) */
    RTB_RENDER_SINGLE_PIPELINE = 16, /* one wavefront on one stream (per-stage timing; default is four concurrent ones, two on scenes beyond L2) */
    /* ---- beyond the reference (SURVEY 8f-3): OFF by default, parity mode is untouched ---- */
    RTB_RENDER_TRUE_MIS = 32,     /* power_heuristic(float, float) for the light sample, and the path ray itself is the
                                     BSDF sample of the MIS pair: emitters met after a bounce add beta * L * w (the
                                     reference truncates the BSDF pdf to int and aims its MIS ray at the wrong triangle,
                                     utility.cuh:53, render.cuh:236; specular paths then never see a light) */
    RTB_RENDER_RR_TERMINATE = 64, /* a Russian-roulette kill ends the path (the reference only pauses it, render.cuh:112-126) */
    RTB_RENDER_DETERMINISTIC = 128 /* radiance sums in 64-bit fixed point (2^-28) instead of float atomics (vec3.cuh:149-153, whose
                                     result depends on the order of the splats): the image is bit-identical from run to run and for
                                     ANY split of the samples over wavefronts, calls and GPUs (rtb_multi_render reduces the integer
                                     sums).  Splats are clamped to +-2^24.  Slower splats (three 64-bit atomics instead of one
                                     128-bit vector reduction); off by default */
};

typedef struct rtb_render_stats {
    uint64_t paths;        /* camera paths started */
    uint64_t extend_rays;  /* closest-hit traversals */
    uint64_t shadow_rays;  /* any-hit traversals */
    uint64_t iterations;   /* wavefront iterations */
    uint64_t kernel_launches;
    uint64_t extend_nodes, extend_tris; /* 80-byte nodes fetched / triangles tested by extend rays */
    uint64_t shadow_nodes, shadow_tris; /* same for shadow rays (only with RTB_RENDER_COUNT_WORK) */
    uint64_t extend_launches, shadow_launches; /* launches of the two traversal kernels */
    uint64_t hits;         /* extend rays that hit something (= paths shaded) */
    float ms_total;        /* generate..accumulate, CUDA events on the render stream */
    float ms_extend;       /* summed duration of the extend launches (CUDA events) */
    float ms_shadow;       /* summed duration of the shadow launches */
    float ms_other;        /* ms_total - ms_extend - ms_shadow: shade, generate, control, host gaps */
    float ms_shade;        /* summed duration of shade + generate + control (part of ms_other) */
    int32_t fused_trace;   /* 1: extend and shadow rays ran in ONE launch per iteration; then ms_extend
                              is the duration of that launch and ms_shadow is 0 */
    int32_t pipelines;     /* independent wavefronts run on concurrent streams (1..4); the per-stage
                              times above are only measured with 1 (RTB_RENDER_SINGLE_PIPELINE) */
    int32_t pool;          /* path slots each wavefront ran with (rtb_render_params.pool_size, the "pool" option, or the
                              automatic size: see rtb_context_set_option) */
} rtb_render_stats;

typedef struct rtb_context rtb_context; /* one per GPU */
typedef struct rtb_scene rtb_scene;     /* device-resident scene + BVH */

/* ---- context / errors (replaces CHECK_CUDA, utility.cuh:4-13) ---- */
RTB_API const char *rtb_last_error(void);
RTB_API const char *rtb_version(void);
RTB_API int rtb_context_create(int device_ordinal, rtb_context **out);
RTB_API int rtb_context_destroy(rtb_context *ctx);
RTB_API int rtb_context_device(const rtb_context *ctx);
/* Schedule of the traversal / wavefront kernels (replaces compile-time choices such as BLOCK_SIZE, render.cuh:413, and
 * NUM_WORKING_PATHS, constant.hpp:8).  Every schedule gives bit-identical hits; the defaults are the measured best
 * (DESIGN.md 4).  Names: "refill" (1..32), "chunk" (>= 32), "prefetch" (0/1), "tri_step" (0..4), "pooled" (-1/0/1),
 * "fused" (0/1), "smem_stack" (0/1), "pipelines" (0 = by scene size, 1..4), "pool" (path slots, >= 1024; 0 = automatic, the default:
 * as many paths as fit an eighth of the device memory that was free when the context was created, at least 4 Mi, at most the
 * paths of the render — C2 on an empty B200: all 132.7 M paths, 19 GB of ray / hit queues; the queues of the last scene
 * that was destroyed stay with the context for the next scene that renders with the same shape, until
 * rtb_context_destroy),
 * "ploc_tail" (0/1), "nn_tiled" (0/1), "trace_blocks" (0 = auto, 1..8 resident blocks per SM).  Unknown names / values out of range:
 * RTB_ERR_INVALID.  Takes effect for scenes built and renders started afterwards. */
RTB_API int rtb_context_set_option(rtb_context *ctx, const char *name, int64_t value);
RTB_API int rtb_context_get_option(const rtb_context *ctx, const char *name, int64_t *value);

/* ---- scene + BVH build (replaces Bvh::Bvh, bvh.cuh:30-219, and the Scene
 *      aggregate scene.cuh:4-8; uploads that main.cu:46-138 does by hand) ---- */
RTB_API int rtb_build_params_default(rtb_build_params *p);
RTB_API int rtb_scene_create(rtb_context *ctx, const rtb_scene_desc *desc,
                             const rtb_build_params *bp, rtb_scene **out);
/* Reference-pointer ingest: `h_primitives` is the host vector of reference
 * Primitive structs (primitive.cuh:4-12; 24 B each, holding DEVICE pointers)
 * exactly as passed to Bvh::Bvh (bvh.cuh:17); d_triangles / d_materials /
 * d_lights are the device arrays those pointers point into (main.cu:49,120,135).
 * A device gather kernel dereferences the pointers into the SoA layout. */
RTB_API int rtb_scene_create_from_primitives(rtb_context *ctx, const void *h_primitives,
                                             int64_t num_primitives, const void *d_triangles,
                                             const void *d_materials, int32_t num_materials,
                                             const void *d_lights, int32_t num_lights,
                                             const rtb_build_params *bp, rtb_scene **out);
/* The reference constructs `Bvh` BEFORE the light array exists and fills `Scene{bvh, num_lights, d_lights}` afterwards
 * (main.cu:151-156): pass num_lights = -1 above to build the tree at once (stats are then available, as the
 * reference's Bvh::num_nodes / max_depth are after its constructor, bvh.cuh:23-27,203-204) and hand the lights over
 * here; may be called again when the light array changes.  A light pointer outside [d_lights, d_lights + num_lights):
 * RTB_ERR_INVALID. */
RTB_API int rtb_scene_attach_lights(rtb_scene *scene, const void *d_lights, int32_t num_lights);
/* two-level BVH over meshes + instances (see rtb_instanced_scene_desc); every query / render entry point below
 * works on the result like on a flat scene */
RTB_API int rtb_scene_create_instanced(rtb_context *ctx, const rtb_instanced_scene_desc *desc,
                                       const rtb_build_params *bp, rtb_scene **out);
RTB_API int rtb_scene_destroy(rtb_scene *scene);
RTB_API int rtb_scene_stats(const rtb_scene *scene, rtb_bvh_stats *out);

/* ---- updating a scene in place (animation) ---- */
/* New vertex positions for every triangle (9 floats per triangle, caller order, as many triangles as at creation);
 * topology, materials and lights unchanged.  The 8-wide tree keeps its topology and gets new boxes (refit), and the
 * triangle records are derived from these vertices (also for a scene of rtb_scene_create_from_primitives, as the
 * reference's host constructor derives them).  Instanced scenes: the geometry's object-space vertices; every mesh tree
 * is refit and the tree over the instances is rebuilt with the current transforms.  Area lights follow their moved
 * triangles.  A vertex that rtb_scene_create would reject (not finite, beyond 2^100), or a null pointer:
 * RTB_ERR_INVALID and the scene is unchanged.  Afterwards rtb_bvh_stats.sah_cost and scene_bounds describe the refit
 * tree; build_ms stays the time of the original build.
 * A refit tree keeps the topology that was built for the original geometry: the further the geometry moves from that
 * shape, the more nodes a ray visits and the slower traces and renders get (tools/refit_ab.py, DESIGN.md 4.9).
 * Rebuild the scene (rtb_scene_create*) when that happens.  The render state of the scene (queues, accumulation
 * buffer) is kept.  rtb_scene_refit_device reads the vertices from device memory on the scene's GPU, which must be
 * ready when it is called (it runs on the context's stream); *ms (may be NULL) gets the GPU time of the update. */
RTB_API int rtb_scene_refit(rtb_scene *scene, const float *h_vertices);
RTB_API int rtb_scene_refit_device(rtb_scene *scene, const float *d_vertices, float *ms);
/* Instanced scenes only: new instance records, as many as at creation; instance i keeps its mesh (so the flattened hit
 * ids keep their meaning), its transform and material may change.  The instance boxes and the tree over the instances
 * are rebuilt; the mesh trees are untouched.  The checks of rtb_scene_create_instanced apply (transform finite and
 * invertible, material in range, a mesh with emitters keeps its single identity placement, stack depth); on failure
 * RTB_ERR_INVALID and the scene is unchanged.  Afterwards rtb_bvh_stats.num_nodes, num_top_nodes, collapse_levels,
 * sah_cost and scene_bounds describe the new tree. */
RTB_API int rtb_scene_set_instances(rtb_scene *scene, const rtb_instance *h_instances, int32_t num_instances);

/* ---- ray queries (replace Bvh::traverse closest-hit bvh.cuh:251-303 with
 *      kernel ch render.cuh:297-328, and any-hit bvh.cuh:306-357 with kernel
 *      ah render.cuh:278-294) ---- */
RTB_API int rtb_trace_closest(rtb_scene *scene, const rtb_ray *h_rays, int64_t n, rtb_hit *h_hits);
/* h_excluded[i]: triangle index that may not occlude ray i (the light's own
 * triangle, render.cuh:197) or -1.  h_occluded[i] = 1 if any other triangle
 * is hit with 0 < t <= tmax. */
RTB_API int rtb_trace_any(rtb_scene *scene, const rtb_ray *h_rays, const int32_t *h_excluded,
                          int64_t n, uint8_t *h_occluded);
/* device-buffer variants, timed on the GPU; *ms may be NULL */
RTB_API int rtb_trace_closest_device(rtb_scene *scene, const rtb_ray *d_rays, int64_t n,
                                     rtb_hit *d_hits, float *ms);
RTB_API int rtb_trace_any_device(rtb_scene *scene, const rtb_ray *d_rays,
                                 const int32_t *d_excluded, int64_t n, uint8_t *d_occluded,
                                 float *ms);
/* The same two queries through the RENDER path's own traversal kernel (the persistent k_trace launch that
 * rtb_render runs once per wavefront iteration, in place of kernels ch / ah, render.cuh:278-328): the rays are
 * loaded into the extend / shadow queues, one iteration's trace launch(es) run with the context's schedule
 * (rtb_context_set_option), and the results are read back from the hit queues / the accumulation buffer.  The
 * parity tests compare THIS entry with the reference's Bvh::traverse (bvh.cuh:251-357), so the kernel that is pinned
 * is the kernel that renders.  Either ray set may be empty (n = 0, null pointers).  Closest-hit rays are unbounded
 * like the render's path rays (Ray::tmax = FLT_MAX, ray.cuh:10): their tmax field is ignored.  h_excluded as in
 * rtb_trace_any (not supported on instanced scenes).  *launches (may be NULL) = trace launches made. */
RTB_API int rtb_trace_wavefront(rtb_scene *scene, const rtb_ray *h_rays, int64_t n, rtb_hit *h_hits,
                                const rtb_ray *h_shadow_rays, const int32_t *h_excluded, int64_t n_shadow,
                                uint8_t *h_occluded, int32_t *launches);
/* traversal work counters for the roofline model: mean 80-byte nodes fetched
 * and triangles tested per ray (closest-hit), from a counting kernel variant */
RTB_API int rtb_trace_closest_counts(rtb_scene *scene, const rtb_ray *h_rays, int64_t n,
                                     double *nodes_per_ray, double *tris_per_ray);

/* ---- camera (replaces Camera::Camera, camera.cuh:15-29; host arithmetic) ---- */
RTB_API int rtb_camera_look_at(const float lookfrom[3], const float lookat[3], const float up[3],
                               float vfov_deg, float aspect, rtb_camera *out);
/* camera rays through pixel centres, Camera::get_ray((i+.5)/W,(j+.5)/H), camera.cuh:31-34 */
RTB_API int rtb_camera_primary_rays(const rtb_camera *cam, int32_t width, int32_t height,
                                    rtb_ray *h_rays);

/* ---- render (replaces render(), render.cuh:366-457) ---- */
RTB_API int rtb_render_params_default(rtb_render_params *p);
/* whole call with host output: fb is float[3*W*H], sqrt(sum/total_spp), row 0 = top
 * (render.cuh:330-338,455-456). */
RTB_API int rtb_render(rtb_scene *scene, const rtb_camera *cam, const rtb_render_params *p,
                       float *h_rgb_out, rtb_render_stats *stats);
/* adds the radiance SUM of this call's samples into d_accum (float[3*W*H],
 * device memory, not cleared) — the per-GPU accumulation of a sample-pass
 * shard; reduce across GPUs, then rtb_tonemap_device. */
RTB_API int rtb_render_accumulate(rtb_scene *scene, const rtb_camera *cam,
                                  const rtb_render_params *p, float *d_accum,
                                  rtb_render_stats *stats);
/* the same into a buffer of 64-bit fixed-point sums (int64_t[3*W*H], units of 2^-28, device memory, not cleared):
 * integer sums of sample-pass shards are exact, so the reduced image does not depend on the sharding
 * (implies RTB_RENDER_DETERMINISTIC) */
RTB_API int rtb_render_accumulate_fixed(rtb_scene *scene, const rtb_camera *cam, const rtb_render_params *p,
                                        int64_t *d_accum_fixed, rtb_render_stats *stats);
RTB_API int rtb_tonemap_fixed_device(rtb_context *ctx, const int64_t *d_accum_fixed, int64_t num_values,
                                     int32_t total_spp, float *d_out);
/* d_out[i] = sqrt(d_accum[i] / total_spp)  (post_process_framebuffer, render.cuh:330-338);
 * d_out may alias d_accum */
RTB_API int rtb_tonemap_device(rtb_context *ctx, const float *d_accum, int64_t num_floats,
                               int32_t total_spp, float *d_out);

/* ---- progressive rendering and checkpoints (SURVEY 5 "checkpoint / resume", 8f-4; the reference writes its image
 *      once at exit, main.cu:173-192, and its int sample counter caps one call at 258 spp in 4K, render.cuh:371) ----
 * An rtb_accum is the accumulation buffer of one image (device memory) plus the index of the next sample: sample
 * passes are added to it call by call (each pass renders samples [next, next + spp) of every pixel, so the passes of
 * one image never repeat a random stream), the image so far can be resolved after any pass, and the state can be
 * written to a file and picked up again — by another process or another day — exactly where it stopped. */
typedef struct rtb_accum rtb_accum;
/* deterministic != 0: 64-bit fixed-point sums (see RTB_RENDER_DETERMINISTIC): a resumed render is then bit-identical to
 * an uninterrupted one */
RTB_API int rtb_accum_create(rtb_context *ctx, int32_t width, int32_t height, int32_t deterministic, rtb_accum **out);
RTB_API int rtb_accum_destroy(rtb_accum *a);
/* adds p->spp samples; p->width / height must match, p->first_sample and p->total_spp are ignored (the buffer knows) */
RTB_API int rtb_accum_add_samples(rtb_accum *a, rtb_scene *scene, const rtb_camera *cam, const rtb_render_params *p,
                                  rtb_render_stats *stats);
RTB_API int rtb_accum_samples(const rtb_accum *a);  /* samples per pixel accumulated so far */
/* the image so far: sqrt(sum / samples), float[3*W*H], row 0 = top (as rtb_render) */
RTB_API int rtb_accum_resolve(rtb_accum *a, float *h_rgb_out);
RTB_API int rtb_accum_save(rtb_accum *a, const char *path);
RTB_API int rtb_accum_load(rtb_context *ctx, const char *path, rtb_accum **out);

/* ---- several GPUs of one box (SURVEY 5 / 8e; the reference has no cudaSetDevice, stream or collective anywhere and
 *      its render() is not re-entrant: globals at render.cuh:25-59) ----
 * Every (pixel, sample) path is independent under the counter-based RNG, so the GPUs split the SAMPLES of every pixel
 * (balanced, contiguous shares of p->spp), each accumulates into its own buffer, and one sum-reduction over NVLink
 * (NCCL ncclReduce: float sums, or the 64-bit fixed-point sums with RTB_RENDER_DETERMINISTIC, which makes the image
 * bit-identical for any number of GPUs) followed by the tonemap on the first GPU gives the image.  NCCL (libnccl.so.2)
 * is loaded on first use; a box without it gets RTB_ERR_NO_DEVICE from these entry points only.
 *
 * (1) ONE PROCESS, n GPUs — the drop-in for render() on a multi-GPU box: */
typedef struct rtb_multi rtb_multi;             /* n contexts + their communicator */
typedef struct rtb_multi_scene rtb_multi_scene; /* the scene, resident on every GPU of the rtb_multi */
RTB_API int rtb_multi_create(const int32_t *device_ordinals, int32_t n, rtb_multi **out);
RTB_API int rtb_multi_destroy(rtb_multi *m);
RTB_API int rtb_multi_size(const rtb_multi *m);
RTB_API int rtb_multi_context(rtb_multi *m, int32_t i, rtb_context **ctx); /* borrowed: do not destroy */
/* built concurrently, one host thread per GPU, each from the same host description */
RTB_API int rtb_multi_scene_create(rtb_multi *m, const rtb_scene_desc *desc, const rtb_build_params *bp, rtb_multi_scene **out);
RTB_API int rtb_multi_scene_create_instanced(rtb_multi *m, const rtb_instanced_scene_desc *desc, const rtb_build_params *bp,
                                             rtb_multi_scene **out);
/* built once: `primary` (a scene of context 0 of `m`, e.g. from rtb_scene_create_from_primitives, whose device
 * pointers live on that GPU only) is copied device to device to the other GPUs; `primary` stays owned by the caller
 * and must outlive the result */
RTB_API int rtb_multi_scene_replicate(rtb_multi *m, rtb_scene *primary, rtb_multi_scene **out);
RTB_API int rtb_multi_scene_destroy(rtb_multi_scene *ms);
/* replaces render(), render.cuh:366-367: p->spp samples per pixel in total, split over the GPUs that p->device_mask
 * selects (0 = all); h_rgb_out as in rtb_render.  stats: rays / paths summed over the GPUs, ms_total = the slowest GPU's
 * render + reduce + tonemap */
RTB_API int rtb_multi_render(rtb_multi_scene *ms, const rtb_camera *cam, const rtb_render_params *p, float *h_rgb_out,
                             rtb_render_stats *stats);
/* everything in one call (contexts, scene upload + build on every GPU, render, reduce, tonemap, teardown) */
RTB_API int rtb_render_multi(const int32_t *device_ordinals, int32_t n, const rtb_scene_desc *desc, const rtb_build_params *bp,
                             const rtb_camera *cam, const rtb_render_params *p, float *h_rgb_out, rtb_render_stats *stats);
/* (2) ONE PROCESS PER GPU (torchrun, MPI): rank 0 makes an id and hands its RTB_COMM_ID_BYTES bytes to the other ranks
 * through the launcher's own channel; every rank renders its shard with rtb_render_accumulate[_fixed] (first_sample /
 * spp / total_spp of its share) and the buffers are summed in place on every rank. */
#define RTB_COMM_ID_BYTES 128
typedef struct rtb_comm rtb_comm;
RTB_API int rtb_comm_unique_id(uint8_t *id_out);
RTB_API int rtb_comm_create(rtb_context *ctx, const uint8_t *id, int32_t rank, int32_t world, rtb_comm **out);
RTB_API int rtb_comm_destroy(rtb_comm *c);
RTB_API int rtb_comm_allreduce_f32(rtb_comm *c, float *d_buf, int64_t n);     /* ncclAllReduce(ncclFloat32, ncclSum), in place */
RTB_API int rtb_comm_allreduce_i64(rtb_comm *c, int64_t *d_buf, int64_t n);   /* fixed-point sums: exact */

/* Feature buffers of the primary hits, one camera ray through every pixel centre (what a denoiser wants next to the
 * radiance; SURVEY 8f-4 — the reference has nothing of the kind): albedo of the hit material (float[3*W*H]), geometric
 * unit normal turned towards the camera (float[3*W*H]), hit distance (float[W*H], 0 for a miss) and triangle index in
 * the caller's list (int32[W*H], -1 for a miss).  Any pointer may be NULL.  Row 0 = top, like rtb_render. */
RTB_API int rtb_render_aovs(rtb_scene *scene, const rtb_camera *cam, int32_t width, int32_t height,
                            float *h_albedo, float *h_normal, float *h_depth, int32_t *h_prim);

/* Known-answer hooks: evaluate ONE device function of the render path per record, on the GPU, so that unit tests
 * can compare it with the oracle (SURVEY 4: "unit KATs for ray/triangle, ray/box, offset_ray_origin, BSDF/light
 * sampling").  h_in / h_out hold n records of floats (integers travel as their bits):
 *   RTB_KAT_TRI_INTERSECT  in[16] p0 p1 p2 | ray origin, dir, tmax   out[4] hit (0/1), t, u, v      triangle.cuh:4-58
 *   RTB_KAT_OFFSET_ORIGIN  in[6]  p, n                               out[3] offset origin           utility.cuh:31-47
 *   RTB_KAT_RAND4          in[4]  seed, pixel, sample, block (u32)   out[4] four uniforms in (0,1]  replaces curand_uniform
 *   RTB_KAT_SAMPLE_F       in[16] albedo, ior, type (i32), wo, n, u1, u2, 3 pad   out[12] f, n, wi, pdf, 2 pad   material.cuh:60-109
 *   RTB_KAT_SLAB           in[20] parent box lo hi | child box lo hi | ray origin, dir, tmax, 1 pad   out[1] 1 if the quantised
 *                          child box passes the slab test of the 8-wide node (must hold whenever the exact box meets [0, tmax]:
 *                          aabb_intersector.cuh:14-36 restated conservatively)
 *   RTB_KAT_SAMPLE_LI      in[16] light triangle p0 p1 p2 | shading point, u1, u2, 2 pad   out[8] wi, t, pdf, 3 pad   light.cuh:38-46 */
enum { RTB_KAT_TRI_INTERSECT = 1, RTB_KAT_OFFSET_ORIGIN = 2, RTB_KAT_RAND4 = 3, RTB_KAT_SAMPLE_F = 4, RTB_KAT_SLAB = 5, RTB_KAT_SAMPLE_LI = 6 };
RTB_API int rtb_kat_eval(rtb_context *ctx, int32_t which, const float *h_in, int64_t n, float *h_out);

/* ---- host-side scene I/O and procedural scenes (host C++, no GPU work) ---- */
typedef struct rtb_host_scene rtb_host_scene; /* owns the arrays a rtb_scene_desc points to */
/* PLY, ASCII (what main.cu:60-62 reads through happly.h:1289,1451,1498) or binary_little_endian: vertex x y z first
 * (float32; float64 in a binary file), face index lists, polygons fanned into triangles */
RTB_API int rtb_mesh_load_ply(const char *path, float **verts_out, int64_t *num_verts,
                              int32_t **faces_out, int64_t *num_faces);
/* compact binary mesh fixture: "RTBM" u32 nv u32 nf, f32 verts[3nv], i32 faces[3nf] */
RTB_API int rtb_mesh_load_bin(const char *path, float **verts_out, int64_t *num_verts,
                              int32_t **faces_out, int64_t *num_faces);
RTB_API int rtb_mesh_save_bin(const char *path, const float *verts, int64_t num_verts,
                              const int32_t *faces, int64_t num_faces);
RTB_API void rtb_free(void *p);

enum {
    RTB_SCENE_S1 = 1,  /* main.cu:41-148 Cornell box + bunny, all matte (configs C1, C2) */
    RTB_SCENE_S1_MIXED = 2, /* same geometry, MATTE/MIRROR/GLASS round-robin by triangle index (C4) */
    RTB_SCENE_S2 = 3,  /* Cornell shell + grid x grid bunny instances, ~10M triangles at grid=12 (C3, C5) */
    RTB_SCENE_S1_GLOSSY = 4 /* S1 geometry, the bunny RTB_GLOSSY (exponent 50), the x = 1 wall RTB_GLOSSY (exponent 400) */
};
RTB_API int rtb_host_scene_build(int32_t kind, const float *mesh_verts, int64_t num_verts,
                                 const int32_t *mesh_faces, int64_t num_faces, int32_t grid,
                                 uint32_t seed, rtb_host_scene **out);
RTB_API int rtb_host_scene_desc(const rtb_host_scene *hs, rtb_scene_desc *out);
RTB_API int rtb_host_scene_camera(const rtb_host_scene *hs, float aspect, rtb_camera *out);
/* instanced form of a procedural scene (host C++, no GPU work).  RTB_SCENE_S2: mesh 0 = the bunny as loaded, placed
 * grid x grid times by the very transforms rtb_host_scene_build applies to its vertices, mesh 1 = the Cornell shell
 * with its two emitters (identity); flattening it gives the triangles of the flat RTB_SCENE_S2 in the same order. */
RTB_API int rtb_host_scene_build_instanced(int32_t kind, const float *mesh_verts, int64_t num_verts,
                                           const int32_t *mesh_faces, int64_t num_faces, int32_t grid,
                                           uint32_t seed, rtb_host_scene **out);
RTB_API int rtb_host_scene_instanced_desc(const rtb_host_scene *hs, rtb_instanced_scene_desc *out);
/* the flat scene an instanced description stands for: every instance's triangles transformed on the host
 * (Transform::apply, transform.hpp:26-33: double arithmetic on the float matrix), instance after instance */
RTB_API int rtb_instanced_flatten(const rtb_instanced_scene_desc *desc, rtb_host_scene **out);
RTB_API int rtb_host_scene_destroy(rtb_host_scene *hs);
/* scene file shared with the reference harness: see csrc/host/scene_io.cpp */
RTB_API int rtb_scene_desc_save(const char *path, const rtb_scene_desc *desc);
RTB_API int rtb_host_scene_load(const char *path, rtb_host_scene **out);
/* P3 PPM with clamp(int(256*c),0,255), main.cu:178-191 */
RTB_API int rtb_write_ppm(const char *path, const float *rgb, int32_t width, int32_t height);

#ifdef __cplusplus
}
#endif
#endif /* RTB_H */
