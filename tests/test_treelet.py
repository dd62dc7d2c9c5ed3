"""rtb_build_params.builder | RTB_BUILDER_TREELET_PASSES(k): treelet restructuring of the binary tree between the
builder and the collapse (rtb_build.h 3.5), for both builders and both collapse modes, against the oracle.

Every test runs on the host build of the kernel bodies (tests/emu) and, with -m gpu, on the shipped CUDA library
(k_tlo_treelet).  The restructured tree differs from the builder's, so exact-t ties (a ray through the shared edge of
two triangles) may resolve to the other triangle, as with RTB_COLLAPSE_SAH_OPTIMAL; t is bit-exact everywhere.
"""
import ctypes as C
import time

import numpy as np
import pytest

from rtcuda_b200 import capi
from conftest import make_desc, mean_rel_err, random_rays, small_scene_arrays, std_materials
from test_sah_builder import IMAGE_TOL, TIE_FRACTION, assert_hits_up_to_ties, shadow_rays_s1

BUILDERS = [capi.RTB_BUILDER_PLOC, capi.RTB_BUILDER_BINNED_SAH]
COLLAPSES = [capi.RTB_COLLAPSE_LARGEST_FIRST, capi.RTB_COLLAPSE_SAH_OPTIMAL]
VARIANTS = [(b, c) for b in BUILDERS for c in COLLAPSES]
VARIANT_IDS = [f"{'ploc' if b == capi.RTB_BUILDER_PLOC else 'sah'}-{'greedy' if c == capi.RTB_COLLAPSE_LARGEST_FIRST else 'opt'}"
               for b, c in VARIANTS]
PASSES = 3


@pytest.fixture(scope="module", params=["emu", pytest.param("gpu", marks=pytest.mark.gpu)])
def L(request):
    return request.getfixturevalue(request.param)


@pytest.fixture(scope="module")
def ctx(L):
    return L.context(0)


@pytest.fixture(scope="module")
def s1(L, bunny):
    return L.host_scene(capi.RTB_SCENE_S1, *bunny)


@pytest.fixture(scope="module")
def s1_orc(oracle, s1):
    return oracle.scene(s1.desc)


def params(L, builder=capi.RTB_BUILDER_PLOC, collapse=capi.RTB_COLLAPSE_LARGEST_FIRST, passes=PASSES):
    bp = capi.BuildParams()
    L.lib.rtb_build_params_default(C.byref(bp))
    bp.builder, bp.collapse = builder | capi.treelet_passes(passes), collapse
    return bp


def tree_stats(st):
    """what two builds of the same tree share exactly (sah_cost is summed by float atomics on the GPU, in any order:
    equal up to rounding, see same_cost)"""
    return (st.num_nodes, st.num_bvh2_nodes, st.collapse_levels, st.ploc_iterations, st.num_triangles)


def same_cost(a, b):
    return abs(a.sah_cost - b.sah_cost) <= 1e-5 * b.sah_cost


@pytest.mark.parametrize("builder,collapse", VARIANTS, ids=VARIANT_IDS)
def test_hits_default_scene(L, ctx, s1, s1_orc, builder, collapse):
    """pixel-centre rays at 600x600 and 200 k incoherent rays; any-hit with and without the excluded emitter identical"""
    sc = ctx.scene(s1.desc, params(L, builder, collapse))
    rays = np.concatenate([L.primary_rays(s1.camera(1.0), 600, 600), random_rays(200000, seed=7)])
    assert_hits_up_to_ties(sc.trace_closest(rays), s1_orc.trace_closest(rays, capi.HIT_DTYPE))
    srays, excl = shadow_rays_s1(s1.desc.num_triangles)
    occ, ref = sc.trace_any(srays, excl), s1_orc.trace_any(srays, excl)
    assert 0.05 < ref.mean() < 0.95
    assert (occ == ref).all()
    assert (sc.trace_any(srays, None) == s1_orc.trace_any(srays, None)).all()
    sc.close()


@pytest.mark.parametrize("n", [0, 1, 2, 3, 4, 7, 8, 9, 33, 200, 5000])
@pytest.mark.parametrize("builder,collapse", VARIANTS, ids=VARIANT_IDS)
def test_triangle_counts(L, ctx, oracle, n, builder, collapse):
    """no tree, no inner node, treelets of fewer than 7 leaves (or none above the first pass's 7 triangles) and full
    ones; zero-area and duplicated triangles included"""
    verts, mat, _ = small_scene_arrays(seed=n, n=max(n, 1))
    verts, mat = verts[:n].copy(), mat[:n].copy()
    if n >= 9:
        verts[3, 3:6] = verts[3, 0:3]  # zero-area triangle
        verts[4] = verts[5]            # duplicate triangle
    desc, keep = make_desc(verts, mat, np.full(n, -1, np.int32), std_materials(), [])
    sc = ctx.scene(desc, params(L, builder, collapse))
    st = sc.stats()
    assert st.num_triangles == n and st.num_nodes >= 1
    rays = random_rays(20000, seed=n + 1)
    hits = sc.trace_closest(rays)
    if n == 0:
        assert (hits["prim"] == -1).all()
        return
    assert st.num_bvh2_nodes == 2 * n - 1 and np.isfinite(st.sah_cost)
    osc = oracle.scene(desc)
    ref = osc.trace_closest(rays, capi.HIT_DTYPE)
    assert (hits["t"].view(np.uint32) == ref["t"].view(np.uint32)).all()
    diff = hits["prim"] != ref["prim"]
    if diff.any():  # ties: the duplicated pair, or a shared edge at exactly the same t
        assert diff.mean() <= TIE_FRACTION or (set(hits["prim"][diff]) | set(ref["prim"][diff])) <= {4, 5}
    assert (sc.trace_any(rays, None) == osc.trace_any(rays, None)).all()
    sc.close()


@pytest.mark.parametrize("builder,collapse", VARIANTS, ids=VARIANT_IDS)
def test_zero_passes_is_the_plain_builder(L, ctx, s1, builder, collapse):
    plain = ctx.scene(s1.desc, params(L, builder, collapse, passes=0))
    bp = params(L, builder, collapse, passes=0)
    bp.builder = builder | capi.treelet_passes(0)
    zero = ctx.scene(s1.desc, bp)
    assert tree_stats(plain.stats()) == tree_stats(zero.stats()) and same_cost(plain.stats(), zero.stats())
    rays = np.concatenate([L.primary_rays(s1.camera(1.0), 200, 200), random_rays(50000, seed=3)])
    assert plain.trace_closest(rays).tobytes() == zero.trace_closest(rays).tobytes()
    plain.close(); zero.close()


@pytest.mark.parametrize("builder,collapse", VARIANTS, ids=VARIANT_IDS)
def test_passes_lower_the_sah_cost(L, ctx, s1, builder, collapse):
    """three passes never raise the 8-wide SAH cost by more than 0.5 % (the collapse sees a different tree, so a lower
    binary cost need not give a lower 8-wide one); the binned-SAH tree with the greedy collapse improves strictly.
    Measured on S1 (host emulation and B200 alike): PLOC 2.937 -> 2.915 greedy, 2.888 -> 2.870 SAH-optimal; binned SAH
    3.200 -> 2.856 greedy, 3.161 -> 2.808 SAH-optimal (DESIGN.md 4.1)"""
    a = ctx.scene(s1.desc, params(L, builder, collapse, passes=0))
    b = ctx.scene(s1.desc, params(L, builder, collapse))
    sa, sb = a.stats(), b.stats()
    assert np.isfinite(sb.sah_cost) and 0 < sb.sah_cost <= 1.005 * sa.sah_cost, (sa.sah_cost, sb.sah_cost)
    if builder == capi.RTB_BUILDER_BINNED_SAH and collapse == capi.RTB_COLLAPSE_LARGEST_FIRST:
        assert sb.sah_cost < sa.sah_cost, (sa.sah_cost, sb.sah_cost)
    assert sb.ploc_iterations == sa.ploc_iterations and sb.num_bvh2_nodes == sa.num_bvh2_nodes
    a.close(); b.close()


@pytest.mark.gpu
def test_gpu_passes_and_their_host_emulation_build_the_same_tree(gpu, emu, bunny):
    """k_tlo_treelet (one warp per treelet) and the plain loop of the emulation pick the same topologies; two GPU
    builds give the same tree and the same hits"""
    for builder, collapse in VARIANTS:
        out = []
        for lib in (gpu, emu):
            hs = lib.host_scene(capi.RTB_SCENE_S1, *bunny)
            sc = lib.context(0).scene(hs.desc, params(lib, builder, collapse))
            st = sc.stats()
            out.append((st.num_nodes, st.collapse_levels, st.sah_cost))
            sc.close()
        assert out[0][:2] == out[1][:2], (builder, collapse, out)
        assert abs(out[0][2] - out[1][2]) <= 1e-5 * out[1][2], (builder, collapse, out)
        hs = gpu.host_scene(capi.RTB_SCENE_S1, *bunny)
        ctx = gpu.context(0)
        rays = np.concatenate([gpu.primary_rays(hs.camera(1.0), 300, 300), random_rays(100000, seed=9)])
        runs = []
        for _ in range(2):
            sc = ctx.scene(hs.desc, params(gpu, builder, collapse))
            runs.append((sc.stats(), sc.trace_closest(rays).tobytes()))
            sc.close()
        assert tree_stats(runs[0][0]) == tree_stats(runs[1][0]) and same_cost(runs[0][0], runs[1][0]), (builder, collapse)
        assert runs[0][1] == runs[1][1], (builder, collapse)


def test_identical_triangles(L, ctx, oracle):
    """2500 identical triangles: the binned-SAH tree is balanced, and a pass keeps it (every topology costs the same,
    and only a strictly cheaper one is written): it still fits the traversal stack"""
    n = 2500
    tri = np.array([0, 0, 0, 1, 0, 0, 0, 1, 0], np.float32)
    desc, keep = make_desc(np.tile(tri, (n, 1)), np.zeros(n, np.int32), np.full(n, -1, np.int32), std_materials(), [])
    for collapse in COLLAPSES:
        sc = ctx.scene(desc, params(L, capi.RTB_BUILDER_BINNED_SAH, collapse))
        st = sc.stats()
        assert st.num_triangles == n and st.collapse_levels <= (6 if collapse == capi.RTB_COLLAPSE_SAH_OPTIMAL else 8), st.collapse_levels
        rays = np.zeros(2, capi.RAY_DTYPE)
        rays["origin"] = [(0.2, 0.2, 1.0), (2.0, 2.0, 1.0)]
        rays["dir"] = [(0, 0, -1), (0, 0, -1)]
        rays["tmax"] = 1e30
        hits, ref = sc.trace_closest(rays), oracle.scene(desc).trace_closest(rays, capi.HIT_DTYPE)
        assert hits["prim"][0] >= 0 and hits["prim"][1] == -1
        assert (hits["t"].view(np.uint32) == ref["t"].view(np.uint32)).all()
        sc.close()


def test_instanced_scene(L, ctx, bunny):
    """mesh trees and the tree over the instance boxes (which takes the caller's builder bits) restructured: the hits
    of the plain PLOC build of the same instanced scene, except on exact-t ties"""
    hi = L.host_scene_instanced(capi.RTB_SCENE_S2, *bunny, grid=2)
    a = ctx.scene(hi.idesc, params(L))
    b = ctx.scene(hi.idesc, params(L, passes=0))
    assert a.stats().num_instances == b.stats().num_instances > 0
    rays = np.concatenate([L.primary_rays(hi.camera(1.0), 300, 300), random_rays(100000, seed=17)])
    assert_hits_up_to_ties(a.trace_closest(rays), b.trace_closest(rays))
    assert (a.trace_any(rays[:50000]) == b.trace_any(rays[:50000])).all()
    a.close(); b.close()


def test_multi_scene(L, s1):
    """rtb_multi_scene_create with the passes: the image of the single-context scene built the same way"""
    bp = params(L, capi.RTB_BUILDER_BINNED_SAH)
    cam = s1.camera(1.0)
    p = capi.render_params(L, width=64, height=48, spp=4, max_bounces=6)
    single, _ = L.context(0).scene(s1.desc, bp).render(cam, p)
    m = capi.Multi(L, [0])
    ms = m.scene(s1.desc, bp)
    img, _ = ms.render(cam, p)
    assert mean_rel_err(img, single) <= 1e-5
    ms.close(); m.close()


@pytest.mark.parametrize("builder", [capi.RTB_BUILDER_PLOC | capi.treelet_passes(9), capi.RTB_BUILDER_PLOC | 1 << 12,
                                     2 | capi.treelet_passes(3)], ids=["passes-9", "bit-12", "builder-2"])
def test_invalid_builder_bits_are_rejected(L, ctx, s1, builder):
    bp = params(L, passes=0)
    bp.builder = builder
    h = C.c_void_p()
    assert L.lib.rtb_scene_create(ctx.h, C.byref(s1.desc), C.byref(bp), C.byref(h)) == -1
    assert b"builder" in L.lib.rtb_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("builder", BUILDERS, ids=["ploc", "sah"])
def test_image_c2_shape(gpu, oracle, bunny, builder):
    """a small C2-shaped render (S1, pixel jitter, depth 10) on the restructured tree against the oracle"""
    hs = gpu.host_scene(capi.RTB_SCENE_S1, *bunny)
    sc = gpu.context(0).scene(hs.desc, params(gpu, builder))
    cam = hs.camera(1.0)
    p = capi.render_params(gpu, width=160, height=160, spp=8, max_bounces=10)
    img, st = sc.render(cam, p)
    ref, _, ost = oracle.scene(hs.desc).render(cam, p)
    assert st.paths == ost[0]
    assert mean_rel_err(img, ref) <= IMAGE_TOL
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("builder", BUILDERS, ids=["ploc", "sah"])
def test_s2_against_the_reference_fixture(gpu, bunny, builder):
    """10,000,956 triangles (C3 geometry): the rays of tests/golden/s2_hits.npz / s2_any.npz through trace_wavefront and
    trace_closest / trace_any on the restructured tree.  Id differences are exact-t ties only; any-hit bits identical"""
    from test_wavefront_trace import golden, ray_checksum, s2_rays, s2_shadow_rays
    hs = gpu.host_scene(capi.RTB_SCENE_S2, *bunny, grid=12)
    t0 = time.time()
    sc = gpu.context(0).scene(hs.desc, params(gpu, builder))
    st = sc.stats()
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
        print(f"S2 builder {builder} + {PASSES} treelet passes {entry}: build {st.build_ms:.1f} ms (scene call "
              f"{1e3 * (time.time() - t0):.0f} ms), {st.num_nodes} nodes, SAH {st.sah_cost:.2f}, {ties} exact-t ties of {len(rays)} rays")
        assert (occ == a["occluded"]).all()
    sc.close()
