"""Scene updates against rebuilds: rtb_scene_refit / rtb_scene_set_instances on the C2 shape (S1, 1920x1080, 64 spp,
depth 8), the flat C3 shape (S2 grid 12, 3840x2160, 16 spp, depth 8) and the instanced C3i shape.  One JSON line per
case, after a first line with the card and its power limit:

  refit        (s1, s2) rtb_scene_refit_device with the scene's own vertices: GPU ms of the update (median of --runs,
               CUDA events), the host call with an upload of the vertices, and the PLOC build_ms of the same scene (median
               of 3 builds after a warm-up)
  deform       (s1, s2) at each amplitude of a smooth displacement field (fractions of the unit scene size): the refit
               tree against a fresh PLOC build of the deformed vertices — SAH cost, nodes / triangles per ray
               (rtb_trace_closest_counts) for the pixel-centre rays and for 500 k incoherent rays, and render ms (median
               of --steps renders of the C2 / C3 shape, the two trees alternated)
  instances    (c3i) rtb_scene_set_instances with every bunny turned and moved, against rtb_scene_create_instanced of
               the same description end to end (host wall clock of the calls); render ms before and after the move

    python tools/refit_ab.py > profiles/r3/refit_ab.jsonl
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from rtcuda_b200 import capi  # noqa: E402
from builder_ab import gpu_info, incoherent_rays  # noqa: E402

WORKLOADS = {"s1": (capi.RTB_SCENE_S1, 0, 1920, 1080, 64, 8), "s2": (capi.RTB_SCENE_S2, 12, 3840, 2160, 16, 8)}


def smooth_displacement(verts, amp, freq=2.0):
    """every vertex moved by amp * (sin(w y + .3), sin(w z + 1.1), sin(w x + 2)), w = 2 pi freq: shared vertices move
    together, so the deformed mesh stays closed"""
    p = verts.reshape(-1, 3)
    w = np.float32(2 * np.pi * freq)
    out = np.empty_like(p)
    out[:, 0] = p[:, 0] + np.float32(amp) * np.sin(w * p[:, 1] + np.float32(0.3))
    out[:, 1] = p[:, 1] + np.float32(amp) * np.sin(w * p[:, 2] + np.float32(1.1))
    out[:, 2] = p[:, 2] + np.float32(amp) * np.sin(w * p[:, 0] + np.float32(2.0))
    return out.reshape(verts.shape)


def vertices_of(desc):
    return np.ctypeslib.as_array(C.cast(desc.vertices, C.POINTER(C.c_float)), (desc.num_triangles, 9)).copy()


def median_build_ms(ctx, desc):
    ctx.scene(desc).close()
    times = []
    for _ in range(3):
        s = ctx.scene(desc)
        times.append(s.stats().build_ms)
        s.close()
    return statistics.median(times), times


def tree_record(L, sc, prim, inc):
    st = sc.stats()
    pn, pt = sc.trace_counts(prim)
    inn, itr = sc.trace_counts(inc)
    return {"num_nodes": int(st.num_nodes), "sah_cost": float(st.sah_cost), "primary_nodes_per_ray": pn, "primary_tris_per_ray": pt,
            "incoherent_nodes_per_ray": inn, "incoherent_tris_per_ray": itr}


def render_ms(scenes, cam, p, steps):
    for sc in scenes:  # warm-up
        sc.render(cam, p)
    out = [[] for _ in scenes]
    for _ in range(steps):
        for k, sc in enumerate(scenes):
            _, rs = sc.render(cam, p)
            out[k].append(rs.ms_total)
    return [statistics.median(o) for o in out], out


def flat_cases(L, torch, wl, verts, faces, a, card, power):
    kind, grid, w, h, spp, depth = WORKLOADS[wl]
    hs = L.host_scene(kind, verts, faces, grid=grid)
    ctx = L.context(0)
    cam = hs.camera(w / h)
    prim = L.primary_rays(cam, w, h)
    inc = incoherent_rays(a.incoherent)
    v0 = vertices_of(hs.desc)
    base = {"workload": wl, "card": card, "power_limit": power, "triangles": int(hs.desc.num_triangles)}
    # the refit with the scene's own vertices against the build
    build_ms, build_all = median_build_ms(ctx, hs.desc)
    sc = ctx.scene(hs.desc)
    dv = torch.from_numpy(v0).cuda()
    torch.cuda.synchronize()
    sc.refit_device(dv.data_ptr())  # warm-up
    gpu_ms = [sc.refit_device(dv.data_ptr()) for _ in range(a.runs)]
    host_ms = []
    for _ in range(3):
        t0 = time.perf_counter()
        sc.refit(v0)
        host_ms.append(1e3 * (time.perf_counter() - t0))
    rec = dict(base, case="refit", refit_gpu_ms=statistics.median(gpu_ms), refit_gpu_ms_all=gpu_ms,
               refit_host_call_ms=statistics.median(host_ms), build_ms=build_ms, build_ms_all=build_all,
               build_over_refit=build_ms / statistics.median(gpu_ms))
    print(json.dumps(rec), flush=True)
    sc.close()
    del dv
    # deformations: the refit tree against a fresh build of the deformed vertices
    p = capi.render_params(L, width=w, height=h, spp=spp, max_bounces=depth)
    for amp in [float(x) for x in a.amplitudes.split(",")]:
        v1 = smooth_displacement(v0, amp)
        d1 = capi.SceneDesc.from_buffer_copy(hs.desc)
        d1.vertices = v1.ctypes.data_as(C.c_void_p).value
        refit = ctx.scene(hs.desc)
        refit.refit(v1)
        fresh = ctx.scene(d1)
        ms, ms_all = render_ms([refit, fresh], cam, p, a.steps)
        rec = dict(base, case="deform", amplitude=amp, refit=dict(tree_record(L, refit, prim, inc), render_ms=ms[0], render_ms_all=ms_all[0]),
                   rebuild=dict(tree_record(L, fresh, prim, inc), render_ms=ms[1], render_ms_all=ms_all[1]))
        print(json.dumps(rec), flush=True)
        refit.close(); fresh.close()
        del v1


def instanced_case(L, verts, faces, a, card, power):
    _, grid, w, h, spp, depth = WORKLOADS["s2"]
    hi = L.host_scene_instanced(capi.RTB_SCENE_S2, verts, faces, grid=grid)
    ctx = L.context(0)
    cam = hi.camera(w / h)
    idesc = hi.idesc
    src = (capi.Instance * idesc.num_instances).from_address(idesc.instances)
    moved = (capi.Instance * idesc.num_instances)()
    C.memmove(moved, src, C.sizeof(moved))
    g = idesc.geometry
    lid = np.ctypeslib.as_array(C.cast(g.light_ids, C.POINTER(C.c_int32)), (g.num_triangles,))
    mf = np.ctypeslib.as_array(C.cast(idesc.mesh_first, C.POINTER(C.c_int64)), (idesc.num_meshes + 1,))
    emissive = {m for m in range(idesc.num_meshes) if (lid[mf[m]:mf[m + 1]] >= 0).any()}
    rng = np.random.default_rng(1)
    n_moved = 0
    for k in range(len(moved)):
        if moved[k].mesh in emissive:
            continue
        x = np.array(moved[k].xform[:], np.float64).reshape(3, 4)
        ang = rng.uniform(0.3, 2.5)
        ry = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]])
        x[:, :3] = x[:, :3] @ ry
        x[:, 3] += rng.uniform(-0.01, 0.01, 3) * np.array([1, 0, 1])
        for j in range(12):
            moved[k].xform[j] = float(x.reshape(-1)[j])
        n_moved += 1
    d2 = capi.InstancedSceneDesc.from_buffer_copy(idesc)
    d2.instances = C.cast(moved, C.c_void_p).value
    sc = ctx.scene(idesc)
    p = capi.render_params(L, width=w, height=h, spp=spp, max_bounces=depth)
    (before,), before_all = render_ms([sc], cam, p, a.steps)
    ctx.scene(d2).close()  # warm-up
    create_ms, create_build_ms = [], []
    for _ in range(a.runs):
        t0 = time.perf_counter()
        s = ctx.scene(d2)
        create_ms.append(1e3 * (time.perf_counter() - t0))
        create_build_ms.append(s.stats().build_ms)
        s.close()
    set_ms = []
    for _ in range(a.runs):  # alternately moved and back: every call changes every bunny
        for inst in (moved, src):
            t0 = time.perf_counter()
            sc.set_instances(inst)
            set_ms.append(1e3 * (time.perf_counter() - t0))
    sc.set_instances(moved)
    (after,), after_all = render_ms([sc], cam, p, a.steps)
    st = sc.stats()
    rec = {"workload": "c3i", "case": "instances", "card": card, "power_limit": power, "instances": int(idesc.num_instances),
           "instances_moved": n_moved, "set_instances_ms": statistics.median(set_ms), "set_instances_ms_all": set_ms,
           "create_instanced_call_ms": statistics.median(create_ms), "create_instanced_call_ms_all": create_ms,
           "create_instanced_build_ms": statistics.median(create_build_ms), "num_top_nodes": int(st.num_top_nodes),
           "render_ms_before": before, "render_ms_before_all": before_all[0], "render_ms_after": after, "render_ms_after_all": after_all[0]}
    print(json.dumps(rec), flush=True)
    sc.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="s1,s2,c3i")
    ap.add_argument("--amplitudes", default="0,0.01,0.05,0.2", help="displacement amplitudes, fractions of the unit scene size")
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--incoherent", type=int, default=500000)
    a = ap.parse_args()
    import torch
    card, power = gpu_info()
    print(json.dumps({"card": card, "power_limit": power}), flush=True)
    L = capi.Lib()
    verts, faces = L.load_mesh()
    for wl in a.workloads.split(","):
        if wl == "c3i":
            instanced_case(L, verts, faces, a, card, power)
        else:
            flat_cases(L, torch, wl, verts, faces, a, card, power)


if __name__ == "__main__":
    main()
