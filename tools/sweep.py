"""Tuning sweep over the persistent-kernel knobs (RTB_REFILL / RTB_CHUNK / RTB_POOL / RTB_POOLED / RTB_FUSED / RTB_PREFETCH are read
when a context is created), one process, one scene build per setting.

    python tools/sweep.py --workload c2 --refill 8,16,24 --pooled 0,1 --fused 0,1 --chunk 128 --pool 8388608
"""
import argparse
import ctypes as C
import itertools
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rtcuda_b200 import capi  # noqa: E402

W = {"c1": (1, 0, 600, 600, 10, 10), "c2": (1, 0, 1920, 1080, 64, 8), "c2s": (1, 0, 1920, 1080, 8, 8),
     "c3s": (3, 12, 3840, 2160, 2, 8), "c3": (3, 12, 3840, 2160, 16, 8), "c4": (2, 0, 1920, 1080, 64, 16),
     "c4s": (2, 0, 1920, 1080, 8, 16)}
ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="c2")
ap.add_argument("--refill", default="24")
ap.add_argument("--chunk", default="128")
ap.add_argument("--pool", default="0")
ap.add_argument("--pooled", default="0")
ap.add_argument("--fused", default="1")
ap.add_argument("--prefetch", default="1")
ap.add_argument("--pipelines", default="2")
ap.add_argument("--first-sample", type=int, default=0)
ap.add_argument("--device", type=int, default=0)
ap.add_argument("--radius", type=int, default=0)
ap.add_argument("--leaf", type=int, default=0)
ap.add_argument("--collapse", type=int, default=-1)
ap.add_argument("--builder", type=int, default=-1, help="rtb_build_params.builder (0 PLOC, 1 binned SAH; + 256 * k for k treelet passes)")
ap.add_argument("--count", action="store_true", help="also print nodes / triangles per ray (counting kernels)")
ap.add_argument("--reps", type=int, default=2)
ap.add_argument("--flags", type=int, default=0)
a = ap.parse_args()
kind, grid, w, h, spp, depth = W[a.workload]
L = capi.Lib()
hs = L.host_scene(kind, *L.load_mesh(), grid=grid)
cam = hs.camera(w / h)
print(f"workload {a.workload}: {hs.desc.num_triangles} triangles, {w}x{h}x{spp}spp depth {depth}")
for refill, chunk, pool, pooled, fused, pf, pipes in itertools.product(a.refill.split(","), a.chunk.split(","), a.pool.split(","), a.pooled.split(","),
                                                                 a.fused.split(","), a.prefetch.split(","), a.pipelines.split(",")):
    os.environ.update(RTB_REFILL=refill, RTB_CHUNK=chunk, RTB_POOL=pool, RTB_POOLED=pooled, RTB_FUSED=fused, RTB_PREFETCH=pf, RTB_PIPELINES=pipes)
    ctx = L.context(a.device)
    bp = capi.BuildParams()
    L.lib.rtb_build_params_default(C.byref(bp))
    if a.radius: bp.ploc_radius = a.radius
    if a.leaf: bp.max_leaf_tris = a.leaf
    if a.collapse >= 0: bp.collapse = a.collapse
    if a.builder >= 0: bp.builder = a.builder
    sc = ctx.scene(hs.desc, bp)
    bs = sc.stats()
    p = capi.render_params(L, width=w, height=h, spp=spp, max_bounces=depth, flags=a.flags, first_sample=a.first_sample, total_spp=spp + a.first_sample)
    best = None
    for _ in range(a.reps):
        img, st = sc.render(cam, p)
        if best is None or st.ms_total < best.ms_total:
            best = st
    rays = best.extend_rays + best.shadow_rays
    print(f"pipes {best.pipelines} pooled {pooled} fused {best.fused_trace} pf {pf} refill {refill:>2} chunk {chunk:>4} pool {pool:>9}: {best.ms_total:8.2f} ms  trace/extend {best.ms_extend:7.2f} "
          f"shadow {best.ms_shadow:7.2f} shade {best.ms_shade:6.2f} other {best.ms_other:6.2f}  {rays / best.ms_total * 1e-3:8.1f} Mrays/s  "
          f"iters {best.iterations}  build {bs.build_ms:.1f} ms nodes {bs.num_nodes} sah {bs.sah_cost:.2f} mean {img.mean():.4f}", flush=True)
    if a.count:
        pc = capi.render_params(L, width=w, height=h, spp=1, max_bounces=depth, flags=capi.RTB_RENDER_COUNT_WORK)
        _, cs = sc.render(cam, pc)
        print(f"    per extend ray: {cs.extend_nodes / max(cs.extend_rays, 1):.2f} nodes {cs.extend_tris / max(cs.extend_rays, 1):.2f} tris; per shadow ray: "
              f"{cs.shadow_nodes / max(cs.shadow_rays, 1):.2f} nodes {cs.shadow_tris / max(cs.shadow_rays, 1):.2f} tris; hit fraction {cs.hits / max(cs.extend_rays, 1):.3f}", flush=True)
    sc.close()
    del sc, ctx
