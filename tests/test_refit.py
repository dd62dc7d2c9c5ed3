"""In-place scene updates: rtb_scene_refit / rtb_scene_refit_device (new vertices, same tree topology, new boxes) and
rtb_scene_set_instances (new instance transforms and materials, the tree over the instances rebuilt).

A refit with the vertices the scene was built from reproduces the built tree exactly (the quantisation is a function of
the exact boxes, and the collapse's boxes are unions of the triangle boxes), so its hits and work counts are identical
byte for byte.  A refit to other vertices is checked against the oracle built from them.  Every test runs on the host
build of the kernel bodies (tests/emu) and, with -m gpu, on the shipped CUDA library (k_refit_level).
"""
import ctypes as C
import time

import numpy as np
import pytest

from rtcuda_b200 import capi
from conftest import make_desc, mean_rel_err, random_rays, small_scene_arrays, std_materials
from test_instancing import assert_hits_close, general_instanced_scene
from test_sah_builder import IMAGE_TOL, assert_hits_up_to_ties, shadow_rays_s1

RTB_ERR_INVALID = -1
VARIANTS = [(capi.RTB_BUILDER_PLOC, capi.RTB_COLLAPSE_LARGEST_FIRST, 0), (capi.RTB_BUILDER_PLOC, capi.RTB_COLLAPSE_SAH_OPTIMAL, 0),
            (capi.RTB_BUILDER_BINNED_SAH, capi.RTB_COLLAPSE_LARGEST_FIRST, 0), (capi.RTB_BUILDER_BINNED_SAH, capi.RTB_COLLAPSE_SAH_OPTIMAL, 0),
            (capi.RTB_BUILDER_PLOC, capi.RTB_COLLAPSE_LARGEST_FIRST, 3)]
VARIANT_IDS = ["ploc-greedy", "ploc-opt", "sah-greedy", "sah-opt", "ploc-treelet3"]


@pytest.fixture(scope="module", params=["emu", pytest.param("gpu", marks=pytest.mark.gpu)])
def L(request):
    return request.getfixturevalue(request.param)


@pytest.fixture(scope="module")
def ctx(L):
    return L.context(0)


@pytest.fixture(scope="module")
def s1(L, bunny):
    return L.host_scene(capi.RTB_SCENE_S1, *bunny)


def params(L, builder=capi.RTB_BUILDER_PLOC, collapse=capi.RTB_COLLAPSE_LARGEST_FIRST, passes=0):
    bp = capi.BuildParams()
    L.lib.rtb_build_params_default(C.byref(bp))
    bp.builder, bp.collapse = builder | capi.treelet_passes(passes), collapse
    return bp


def with_vertices(desc, verts):
    """a copy of a flat description with other vertices; returns (desc, keepalive)"""
    verts = np.ascontiguousarray(verts, np.float32)
    d = capi.SceneDesc.from_buffer_copy(desc)
    d.vertices = verts.ctypes.data_as(C.c_void_p).value
    return d, verts


def with_geometry(idesc, geometry):
    d = capi.InstancedSceneDesc.from_buffer_copy(idesc)
    d.geometry = geometry
    return d


def with_instances(idesc, instances):
    d = capi.InstancedSceneDesc.from_buffer_copy(idesc)
    d.instances = C.cast(instances, C.c_void_p).value
    return d


def vertices_of(desc):
    return np.ctypeslib.as_array(C.cast(desc.vertices, C.POINTER(C.c_float)), (desc.num_triangles, 9)).copy()


def instances_of(idesc):
    src = (capi.Instance * idesc.num_instances).from_address(idesc.instances)
    out = (capi.Instance * idesc.num_instances)()
    C.memmove(out, src, C.sizeof(out))
    return out


def smooth_displacement(verts, amp, freq=2.0):
    """a smooth field of amplitude `amp` applied to every vertex: vertices shared by triangles move together"""
    p = verts.reshape(-1, 3).astype(np.float64)
    w = 2 * np.pi * freq
    d = np.stack([np.sin(w * p[:, 1] + 0.3), np.sin(w * p[:, 2] + 1.1), np.sin(w * p[:, 0] + 2.0)], axis=1)
    return (p + amp * d).astype(np.float32).reshape(verts.shape)


def camera_rays(L, n_side=64):
    cam = L.camera_look_at((0.5, 0.5, 1.4), (0.5, 0.45, -0.5), (0, 1, 0), 40.0, 1.0)
    return L.primary_rays(cam, n_side, n_side)


def observe(sc, rays, srays, excl):
    """everything a refit must leave exactly as a build of the same tree gives it"""
    return (sc.trace_closest(rays).tobytes(), sc.trace_any(srays, excl).tobytes(), sc.trace_any(srays, None).tobytes(),
            sc.trace_counts(rays))


def assert_same_tree(a, b):
    sa, sb = a.stats(), b.stats()
    assert (sa.num_nodes, sa.collapse_levels, sa.num_triangles) == (sb.num_nodes, sb.collapse_levels, sb.num_triangles)
    assert list(sa.scene_bounds) == list(sb.scene_bounds)
    assert abs(sa.sah_cost - sb.sah_cost) <= 1e-5 * abs(sb.sah_cost), (sa.sah_cost, sb.sah_cost)


def small_case(n):
    verts, mat, _ = small_scene_arrays(seed=n, n=max(n, 1))
    verts, mat = verts[:n].copy(), mat[:n].copy()
    if n >= 9:
        verts[3, 3:6] = verts[3, 0:3]  # zero-area triangle
        verts[4] = verts[5]            # duplicate triangle
    return verts, mat


def small_rays(L, n):
    rays = np.concatenate([camera_rays(L, 48), random_rays(20000, seed=n + 1)])
    srays = random_rays(5000, seed=n + 2, tmax=np.float32(0.7))
    excl = np.random.default_rng(n).integers(-1, n, len(srays)).astype(np.int32) if n else np.full(len(srays), -1, np.int32)
    return rays, srays, excl


# ---------------------------------------------------------------- 1. identity
@pytest.mark.parametrize("n", [0, 1, 2, 3, 4, 9, 200, 5000])
@pytest.mark.parametrize("builder,collapse,passes", VARIANTS, ids=VARIANT_IDS)
def test_refit_with_the_original_vertices_is_the_identity(L, ctx, n, builder, collapse, passes):
    verts, mat = small_case(n)
    desc, keep = make_desc(verts, mat, np.full(n, -1, np.int32), std_materials(), [])
    built = ctx.scene(desc, params(L, builder, collapse, passes))
    refit = ctx.scene(desc, params(L, builder, collapse, passes))
    rays, srays, excl = small_rays(L, n)
    before = observe(refit, rays, srays, excl)
    refit.refit(verts)
    assert observe(refit, rays, srays, excl) == before == observe(built, rays, srays, excl)
    assert_same_tree(refit, built)
    built.close(); refit.close()


@pytest.mark.parametrize("builder,collapse,passes", VARIANTS, ids=VARIANT_IDS)
def test_refit_of_the_default_scene_is_the_identity(L, ctx, s1, builder, collapse, passes):
    sc = ctx.scene(s1.desc, params(L, builder, collapse, passes))
    st0 = sc.stats()
    rays = np.concatenate([L.primary_rays(s1.camera(1.0), 200, 200), random_rays(50000, seed=3)])
    srays, excl = shadow_rays_s1(s1.desc.num_triangles, 30000)
    before = observe(sc, rays, srays, excl)
    sc.refit(vertices_of(s1.desc))
    assert observe(sc, rays, srays, excl) == before
    st1 = sc.stats()
    assert (st1.num_nodes, st1.collapse_levels, list(st1.scene_bounds), st1.build_ms) == \
        (st0.num_nodes, st0.collapse_levels, list(st0.scene_bounds), st0.build_ms)
    assert abs(st1.sah_cost - st0.sah_cost) <= 1e-5 * st0.sah_cost
    sc.close()


# ---------------------------------------------------------------- 2. deformed geometry
def test_refit_to_deformed_geometry_matches_the_oracle(L, ctx, s1, oracle):
    """S1 under a smooth displacement of its vertices (emitters included): closest hits against the oracle built from
    the deformed vertices (t bit-exact, ids up to exact-t ties), any-hit with and without the excluded emitter
    identical; refit back to the original vertices: the fresh build's results exactly"""
    v0 = vertices_of(s1.desc)
    v1 = smooth_displacement(v0, 0.02)
    d1, keep = with_vertices(s1.desc, v1)
    sc = ctx.scene(s1.desc)
    sc.refit(v1)
    osc = oracle.scene(d1)
    rays = np.concatenate([L.primary_rays(s1.camera(1.0), 300, 300), random_rays(100000, seed=7)])
    assert_hits_up_to_ties(sc.trace_closest(rays), osc.trace_closest(rays, capi.HIT_DTYPE))
    srays, excl = shadow_rays_s1(s1.desc.num_triangles, 50000)
    ref = osc.trace_any(srays, excl)
    assert 0.02 < ref.mean() < 0.98
    assert (sc.trace_any(srays, excl) == ref).all()
    assert (sc.trace_any(srays, None) == osc.trace_any(srays, None)).all()
    fresh = ctx.scene(s1.desc)
    sc.refit(v0)
    assert observe(sc, rays, srays, excl) == observe(fresh, rays, srays, excl)
    assert_same_tree(sc, fresh)
    sc.close(); fresh.close()


@pytest.mark.parametrize("builder,collapse,passes", VARIANTS, ids=VARIANT_IDS)
def test_refit_of_a_soup_moved_at_random(L, ctx, oracle, builder, collapse, passes):
    """every triangle of a random soup moved by up to its own size, far from where the tree was built for"""
    verts, mat, lid = small_scene_arrays(seed=21, n=2000)
    desc, keep = make_desc(verts, mat, np.full(len(mat), -1, np.int32), std_materials(), [])
    moved = (verts + np.random.default_rng(4).normal(scale=0.15, size=verts.shape)).astype(np.float32)
    d1, keep1 = with_vertices(desc, moved)
    sc = ctx.scene(desc, params(L, builder, collapse, passes))
    sc.refit(moved)
    osc = oracle.scene(d1)
    rays, srays, excl = small_rays(L, 2000)
    hits, ref = sc.trace_closest(rays), osc.trace_closest(rays, capi.HIT_DTYPE)
    assert (ref["prim"] >= 0).mean() > 0.2
    assert_hits_up_to_ties(hits, ref)
    assert (sc.trace_any(srays, excl) == osc.trace_any(srays, excl)).all()
    assert (sc.trace_any(srays, None) == osc.trace_any(srays, None)).all()
    fresh = ctx.scene(desc, params(L, builder, collapse, passes))
    sc.refit(verts)
    assert observe(sc, rays, srays, excl) == observe(fresh, rays, srays, excl)
    assert_same_tree(sc, fresh)
    sc.close(); fresh.close()


# ---------------------------------------------------------------- 3. images, lights, render state
def moved_emitters(desc):
    """S1 deformed, with its two emitter triangles (the last two) moved a further step"""
    v = smooth_displacement(vertices_of(desc), 0.01)
    v[-2:] += np.float32([0.05, -0.03, 0.04] * 3)
    return v


@pytest.mark.gpu
def test_image_of_a_refit_scene_with_moved_emitters(gpu, oracle, bunny):
    """a small C2-shaped render (pixel jitter, depth 10) of refit S1 whose area lights moved: the oracle's image of
    the deformed scene (area lights read their triangle from the refit records)"""
    hs = gpu.host_scene(capi.RTB_SCENE_S1, *bunny)
    v1 = moved_emitters(hs.desc)
    d1, keep = with_vertices(hs.desc, v1)
    sc = gpu.context(0).scene(hs.desc)
    sc.refit(v1)
    cam = hs.camera(1.0)
    p = capi.render_params(gpu, width=160, height=160, spp=8, max_bounces=10)
    img, st = sc.render(cam, p)
    ref, _, ost = oracle.scene(d1).render(cam, p)
    assert st.paths == ost[0]
    assert mean_rel_err(img, ref) <= IMAGE_TOL
    sc.close()


def test_render_refit_render_keeps_the_render_state(L, ctx, s1, oracle):
    """the queues and the accumulation buffer of the first render serve the second; the second renders the new
    geometry"""
    sc = ctx.scene(s1.desc)
    cam = s1.camera(1.0)
    p = capi.render_params(L, width=48, height=48, spp=2, max_bounces=4)
    _, st0 = sc.render(cam, p)
    v1 = moved_emitters(s1.desc)
    sc.refit(v1)
    img, st1 = sc.render(cam, p)
    assert (st1.pool, st1.pipelines) == (st0.pool, st0.pipelines)
    d1, keep = with_vertices(s1.desc, v1)
    ref, _, _ = oracle.scene(d1).render(cam, p)
    assert mean_rel_err(img, ref) <= 1e-2  # (48 x 48 x 2 spp: a smoke-level bar; the image test above is the tight one)
    sc.close()


# ---------------------------------------------------------------- 4. the device entry, 5. GPU vs emulation
@pytest.mark.gpu
def test_refit_device_entry(gpu, bunny):
    import torch
    hs = gpu.host_scene(capi.RTB_SCENE_S1, *bunny)
    v1 = smooth_displacement(vertices_of(hs.desc), 0.02)
    ctx = gpu.context(0)
    a, b = ctx.scene(hs.desc), ctx.scene(hs.desc)
    a.refit(v1)
    dv = torch.from_numpy(v1).cuda()
    torch.cuda.synchronize()
    ms = b.refit_device(dv.data_ptr())
    assert ms > 0
    rays = np.concatenate([gpu.primary_rays(hs.camera(1.0), 200, 200), random_rays(50000, seed=5)])
    srays, excl = shadow_rays_s1(hs.desc.num_triangles, 20000)
    assert observe(a, rays, srays, excl) == observe(b, rays, srays, excl)
    a.close(); b.close()


@pytest.mark.gpu
def test_gpu_refit_and_its_host_emulation_agree(gpu, emu, bunny):
    v1 = None
    out = []
    for lib in (gpu, emu):
        hs = lib.host_scene(capi.RTB_SCENE_S1, *bunny)
        if v1 is None:
            v1 = smooth_displacement(vertices_of(hs.desc), 0.02)
        sc = lib.context(0).scene(hs.desc)
        sc.refit(v1)
        rays = np.concatenate([lib.primary_rays(hs.camera(1.0), 200, 200), random_rays(50000, seed=8)])
        out.append((sc.trace_closest(rays).tobytes(), sc.trace_counts(rays), sc.stats().num_nodes))
        sc.close()
    assert out[0] == out[1]


# ---------------------------------------------------------------- 6. moving instances
def emissive_meshes(idesc):
    g = idesc.geometry
    lid = np.ctypeslib.as_array(C.cast(g.light_ids, C.POINTER(C.c_int32)), (g.num_triangles,))
    mf = np.ctypeslib.as_array(C.cast(idesc.mesh_first, C.POINTER(C.c_int64)), (idesc.num_meshes + 1,))
    return {m for m in range(idesc.num_meshes) if (lid[mf[m]:mf[m + 1]] >= 0).any()}


def moved_instances(idesc, seed=0):
    """every instance of a mesh without emitters turned about its own y axis and shifted; one with a material override"""
    inst = instances_of(idesc)
    rng = np.random.default_rng(seed)
    emissive = emissive_meshes(idesc)
    first = True
    for k in range(len(inst)):
        if inst[k].mesh in emissive:
            continue
        x = np.array(inst[k].xform[:], np.float64).reshape(3, 4)
        a = rng.uniform(0.2, 1.0)
        ry = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
        x[:, :3] = x[:, :3] @ ry
        x[:, 3] += rng.uniform(-0.03, 0.03, 3)
        for j in range(12):
            inst[k].xform[j] = float(x.reshape(-1)[j])
        if first:
            inst[k].material = 1  # mirror
            first = False
    return inst


def check_set_instances(L, ctx, oracle, idesc, rays, tie_fraction):
    sc = ctx.scene(idesc)
    srays = random_rays(20000, seed=31, tmax=np.float32(0.6))
    before = (sc.trace_closest(rays).tobytes(), sc.trace_any(srays).tobytes(), sc.trace_counts(rays))
    inst = moved_instances(idesc)
    sc.set_instances(inst)
    d2 = with_instances(idesc, inst)
    fresh = ctx.scene(d2)
    assert (sc.trace_closest(rays).tobytes(), sc.trace_any(srays).tobytes(), sc.trace_counts(rays)) == \
        (fresh.trace_closest(rays).tobytes(), fresh.trace_any(srays).tobytes(), fresh.trace_counts(rays))
    sa, sb = sc.stats(), fresh.stats()
    assert (sa.num_nodes, sa.num_top_nodes, sa.collapse_levels, list(sa.scene_bounds)) == \
        (sb.num_nodes, sb.num_top_nodes, sb.collapse_levels, list(sb.scene_bounds))
    assert abs(sa.sah_cost - sb.sah_cost) <= 1e-5 * sb.sah_cost
    flat = L.flatten(d2)
    assert_hits_close(sc.trace_closest(rays), oracle.scene(flat.desc).trace_closest(rays, capi.HIT_DTYPE), tie_fraction)
    sc.set_instances(instances_of(idesc))
    assert (sc.trace_closest(rays).tobytes(), sc.trace_any(srays).tobytes(), sc.trace_counts(rays)) == before
    sc.close(); fresh.close()


def test_set_instances_on_the_instanced_field(L, ctx, oracle, bunny):
    hi = L.host_scene_instanced(capi.RTB_SCENE_S2, *bunny, grid=2)
    rays = np.concatenate([L.primary_rays(hi.camera(1.0), 200, 200), random_rays(50000, seed=17)])
    check_set_instances(L, ctx, oracle, hi.idesc, rays, 2e-4)


def test_set_instances_on_general_transforms(L, ctx, oracle):
    idesc, keep = general_instanced_scene()
    cam = L.camera_look_at((0.5, 0.5, 1.4), (0.5, 0.45, -0.5), (0, 1, 0), 40.0, 1.0)
    rays = np.concatenate([L.primary_rays(cam, 128, 128), random_rays(30000, seed=2)])
    check_set_instances(L, ctx, oracle, idesc, rays, 1e-3)


# ---------------------------------------------------------------- 7. instanced refit
def test_instanced_refit_matches_the_flattened_deformed_scene(L, ctx, oracle, bunny):
    hi = L.host_scene_instanced(capi.RTB_SCENE_S2, *bunny, grid=2)
    g = hi.idesc.geometry
    v0 = vertices_of(g)
    v1 = smooth_displacement(v0, 0.01, freq=3.0)
    g1, keep = with_vertices(g, v1)
    d1 = with_geometry(hi.idesc, g1)
    sc = ctx.scene(hi.idesc)
    sc.refit(v1)
    flat = L.flatten(d1)
    rays = np.concatenate([L.primary_rays(hi.camera(1.0), 200, 200), random_rays(50000, seed=19)])
    assert_hits_close(sc.trace_closest(rays), oracle.scene(flat.desc).trace_closest(rays, capi.HIT_DTYPE))
    srays = random_rays(20000, seed=23, tmax=np.float32(0.6))
    fresh = ctx.scene(d1)
    assert (sc.trace_any(srays) == fresh.trace_any(srays)).all()
    st, sf = sc.stats(), fresh.stats()
    assert (st.num_top_nodes, list(st.scene_bounds)) == (sf.num_top_nodes, list(sf.scene_bounds))
    sc.close(); fresh.close()


# ---------------------------------------------------------------- 8. rejections leave the scene unchanged
def rejected(L, rc, what):
    assert rc == RTB_ERR_INVALID, what
    assert L.lib.rtb_last_error(), what


def test_rejections_leave_the_scene_unchanged(L, ctx):
    verts, mat, lid = small_scene_arrays(seed=5, n=300)
    desc, keep = make_desc(verts, mat, np.full(len(mat), -1, np.int32), std_materials(), [])
    sc = ctx.scene(desc)
    rays, srays, excl = small_rays(L, 300)
    before = observe(sc, rays, srays, excl)
    for bad in (np.nan, np.float32(2.0 ** 101), -np.inf):
        v = verts.copy()
        v[7, 4] = bad
        rejected(L, L.lib.rtb_scene_refit(sc.h, v.ctypes.data_as(C.c_void_p)), f"vertex {bad}")
        assert observe(sc, rays, srays, excl) == before
    rejected(L, L.lib.rtb_scene_refit(sc.h, None), "null vertices")
    rejected(L, L.lib.rtb_scene_refit_device(sc.h, None, None), "null device vertices")
    rejected(L, L.lib.rtb_scene_refit(None, verts.ctypes.data_as(C.c_void_p)), "null scene")
    inst = (capi.Instance * 1)()
    rejected(L, L.lib.rtb_scene_set_instances(sc.h, inst, 1), "set_instances on a flat scene")
    assert observe(sc, rays, srays, excl) == before
    sc.close()

    idesc, keep2 = general_instanced_scene()
    si = ctx.scene(idesc)
    irays = np.concatenate([camera_rays(L, 64), random_rays(20000, seed=9)])
    israys = random_rays(5000, seed=10, tmax=np.float32(0.6))

    def seen():
        return si.trace_closest(irays).tobytes(), si.trace_any(israys).tobytes(), si.trace_counts(irays)
    base = seen()
    good = instances_of(idesc)

    def attempt(mutate, what, count=None):
        inst = instances_of(idesc)
        mutate(inst)
        rejected(L, L.lib.rtb_scene_set_instances(si.h, inst, len(inst) if count is None else count), what)
        assert seen() == base, what

    attempt(lambda i: None, "wrong count", count=len(good) - 1)
    attempt(lambda i: setattr(i[0], "mesh", 1), "changed mesh")

    def singular(i):
        i[0].xform[0] = i[0].xform[4] = i[0].xform[8] = 0.0
    attempt(singular, "singular transform")
    attempt(lambda i: i[2].xform.__setitem__(3, float("inf")), "non-finite transform")
    attempt(lambda i: setattr(i[1], "material", 9), "material out of range")
    attempt(lambda i: i[6].xform.__setitem__(3, 0.25), "emissive shell moved")
    rejected(L, L.lib.rtb_scene_set_instances(si.h, None, len(good)), "null instances")
    g = idesc.geometry
    v = vertices_of(g)
    v[3, 0] = np.nan
    rejected(L, L.lib.rtb_scene_refit(si.h, v.ctypes.data_as(C.c_void_p)), "instanced: NaN vertex")
    assert seen() == base
    si.set_instances(good)  # accepted: the same instances
    assert seen() == base
    si.close()


def test_python_wrapper_checks_the_vertex_count(L, ctx):
    verts, mat, lid = small_scene_arrays(seed=6, n=50)
    desc, keep = make_desc(verts, mat, np.full(len(mat), -1, np.int32), std_materials(), [])
    sc = ctx.scene(desc)
    with pytest.raises(capi.RtbError, match="9 per triangle"):
        sc.refit(verts[:-1])
    sc.close()


# ---------------------------------------------------------------- 9. scale
@pytest.mark.gpu
def test_s2_refit_against_the_reference_fixture(gpu, bunny):
    """10,000,956 triangles (C3 geometry), refit with its own vertices from device memory: the rays of
    tests/golden/s2_hits.npz / s2_any.npz through trace_wavefront and trace_closest / trace_any.  Id differences are
    exact-t ties only; any-hit bits identical"""
    import torch
    from test_wavefront_trace import golden, ray_checksum, s2_rays, s2_shadow_rays
    hs = gpu.host_scene(capi.RTB_SCENE_S2, *bunny, grid=12)
    sc = gpu.context(0).scene(hs.desc)
    st = sc.stats()
    dv = torch.from_numpy(vertices_of(hs.desc)).cuda()
    torch.cuda.synchronize()
    t0 = time.time()
    ms = sc.refit_device(dv.data_ptr())
    wall = 1e3 * (time.time() - t0)
    del dv
    g, a = golden("s2_hits.npz"), golden("s2_any.npz")
    rays = s2_rays(gpu, hs)
    srays, excl = s2_shadow_rays(len(a["occluded"]), hs.desc.num_triangles)
    assert ray_checksum(rays) == int(g["ray_checksum"]) and ray_checksum(srays) == int(a["ray_checksum"])
    for entry in ("wavefront", "per_ray"):
        if entry == "wavefront":
            hits, occ, _ = sc.trace_wavefront(rays, srays, excl)
        else:
            hits, occ = sc.trace_closest(rays), sc.trace_any(srays, excl)
        ties = assert_hits_up_to_ties(hits, g["hits"])
        print(f"S2 refit {entry}: refit {ms:.2f} ms GPU ({wall:.1f} ms call) against build {st.build_ms:.1f} ms, "
              f"{st.num_nodes} nodes, {ties} exact-t ties of {len(rays)} rays")
        assert (occ == a["occluded"]).all()
    sc.close()
