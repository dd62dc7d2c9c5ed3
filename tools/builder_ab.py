"""A/B of the BVH builders: {PLOC, binned SAH} x {greedy, SAH-optimal collapse} x --optimize (treelet passes,
RTB_BUILDER_TREELET_PASSES) on the C2 shape (S1, 1920x1080, 64 spp, depth 8) and the C3 shape (S2 grid 12, 3840x2160,
16 spp, depth 8).  One JSON line per variant:

  build_ms        median of 3 builds after one warm-up build (rtb_bvh_stats.build_ms, CUDA events)
  num_nodes, sah_cost
  primary / incoherent: nodes and triangles per ray (rtb_trace_closest_counts) for the pixel-centre rays of the camera
                  and 500 k rays with origins in the scene box and uniform directions
  extend / shadow: nodes and triangles per ray of one RTB_RENDER_COUNT_WORK render (1 spp)
  ms_total        median of --steps renders, the variants of a workload alternated in one process

    python tools/builder_ab.py --steps 5 > profiles/r3/builder_ab.jsonl
    python tools/builder_ab.py --steps 5 --optimize 0,3    # every variant without and with 3 treelet passes
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rtcuda_b200 import capi  # noqa: E402

WORKLOADS = {"c2": (capi.RTB_SCENE_S1, 0, 1920, 1080, 64, 8), "c3": (capi.RTB_SCENE_S2, 12, 3840, 2160, 16, 8)}
BUILDERS = {"ploc": capi.RTB_BUILDER_PLOC, "binned_sah": capi.RTB_BUILDER_BINNED_SAH}
COLLAPSES = {"greedy": capi.RTB_COLLAPSE_LARGEST_FIRST, "sah_optimal": capi.RTB_COLLAPSE_SAH_OPTIMAL}


def incoherent_rays(n, seed=1):
    """origins in the unit scene box of S1 / S2 ([0,1] x [0,1] x [-1,0]), uniform directions"""
    rng = np.random.default_rng(seed)
    rays = np.zeros(n, dtype=capi.RAY_DTYPE)
    rays["origin"] = rng.random((n, 3)).astype(np.float32) * np.float32([1, 1, -1])
    d = rng.normal(size=(n, 3))
    rays["dir"] = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    rays["tmax"] = np.float32(3.0e38)
    return rays


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = out[0].split(",")
        return name.strip(), power.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--incoherent", type=int, default=500000)
    ap.add_argument("--optimize", default="0", help="comma-separated treelet pass counts (0..8) to run every variant with")
    a = ap.parse_args()
    assert a.steps >= 5, "the render time is the median of at least 5 steps"
    passes = [int(k) for k in a.optimize.split(",")]
    card, power = gpu_info()
    print(json.dumps({"card": card, "power_limit": power}), flush=True)
    L = capi.Lib()
    verts, faces = L.load_mesh()
    inc = incoherent_rays(a.incoherent)
    for wl in a.workloads.split(","):
        kind, grid, w, h, spp, depth = WORKLOADS[wl]
        hs = L.host_scene(kind, verts, faces, grid=grid)
        cam = hs.camera(w / h)
        ctx = L.context(0)
        prim = L.primary_rays(cam, w, h)
        variants = []
        for bname, b in BUILDERS.items():
            for cname, c, k in [(cn, c, k) for cn, c in COLLAPSES.items() for k in passes]:
                bp = capi.BuildParams()
                L.lib.rtb_build_params_default(C.byref(bp))
                bp.builder, bp.collapse = b | capi.treelet_passes(k), c
                ctx.scene(hs.desc, bp).close()  # warm-up build
                times = []
                for _ in range(3):
                    s = ctx.scene(hs.desc, bp)
                    times.append(s.stats().build_ms)
                    s.close()
                sc = ctx.scene(hs.desc, bp)
                st = sc.stats()
                pn, pt = sc.trace_counts(prim)
                inn, itr = sc.trace_counts(inc)
                _, cs = sc.render(cam, capi.render_params(L, width=w, height=h, spp=1, max_bounces=depth, flags=capi.RTB_RENDER_COUNT_WORK))
                rec = {"workload": wl, "builder": bname, "collapse": cname, "treelet_passes": k, "card": card, "power_limit": power,
                       "triangles": int(st.num_triangles), "build_ms": statistics.median(times), "build_ms_all": times,
                       "num_nodes": int(st.num_nodes), "collapse_levels": int(st.collapse_levels), "sah_cost": float(st.sah_cost),
                       "primary_nodes_per_ray": pn, "primary_tris_per_ray": pt, "incoherent_nodes_per_ray": inn, "incoherent_tris_per_ray": itr,
                       "extend_nodes_per_ray": cs.extend_nodes / max(cs.extend_rays, 1), "extend_tris_per_ray": cs.extend_tris / max(cs.extend_rays, 1),
                       "shadow_nodes_per_ray": cs.shadow_nodes / max(cs.shadow_rays, 1), "shadow_tris_per_ray": cs.shadow_tris / max(cs.shadow_rays, 1),
                       "ms_total": []}
                variants.append((sc, rec))
        p = capi.render_params(L, width=w, height=h, spp=spp, max_bounces=depth)
        for sc, _ in variants:  # warm-up render of every variant
            sc.render(cam, p)
        for _ in range(a.steps):  # variants alternated
            for sc, rec in variants:
                _, rs = sc.render(cam, p)
                rec["ms_total"].append(rs.ms_total)
        for sc, rec in variants:
            rec["ms_total_all"] = rec["ms_total"]
            rec["ms_total"] = statistics.median(rec["ms_total_all"])
            print(json.dumps(rec), flush=True)
            sc.close()
        del variants, ctx


if __name__ == "__main__":
    main()
