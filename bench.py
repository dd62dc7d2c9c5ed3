#!/usr/bin/env python
"""bench.py — the driver's benchmark contract for the render hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]

One "step" = one full render of the workload (generate .. extend/shadow .. shade
.. accumulate .. tonemap) on synthetic input: the reference's default scene
(Stanford bunny in a Cornell box, main.cu:41-166) at BASELINE.json configs[1]
"bunny 1920x1080, 64 spp, max depth 8, diffuse + area light, fixed RNG seed".
N > 1 (torchrun, one rank per GPU): weak scaling by sample pass — every rank
renders its own 64 samples of every pixel ([64r, 64r+64) of 64N), scene
replicated, per-GPU accumulation buffers summed inside the timed step with one
NCCL all-reduce issued by the LIBRARY (rtb_comm_allreduce_f32, include/rtb.h),
then tonemapped.  torch.distributed only carries the barrier, the NCCL id and
the timing exchange.

--dump-outputs DIR (rank 0) writes what the last timed step computed as DIR/<name>.npy, float32: image.npy (the
tonemapped frame) and accum.npy (the summed radiance it was tonemapped from), H x W x 3 each.  When the two exceed
64 MB (64,000,000 bytes) together, both hold the same fixed, seeded sample of pixels as rows, and pixel_index.npy
(float64) says which; a full-frame dump removes a pixel_index.npy an earlier dump left in DIR.
The scene, camera and sample seeds are fixed, so two builds run with the same arguments can be compared output for
output.

Prints ONE JSON line (rank 0).
  value      Mrays/s (extend + shadow rays actually traversed by all ranks) / device time
  e2e        the same metric through the public API from pinned HOST buffers, every step: scene upload +
             GPU BVH build + render + device->host framebuffer.  N = 1: rtb_scene_create + rtb_render.
             N > 1: per rank rtb_scene_create + rtb_render_accumulate + the library's all-reduce; rank 0 alone
             tonemaps and copies the image to the host.
  e2e_one_process  (N > 1) the same step through rtb_multi_scene_create + rtb_multi_render: ONE process (rank 0's)
             drives all N GPUs, the entry a reference-style C++ program calls; the other ranks idle on a host barrier
  roofline   the dominant kernel (k_trace), bound named by residency: "l2" for the L2-resident C2 scene,
             "hbm" for the 600 MB C3 scene; measured DRAM traffic, issue-slot and lane figures from the
             committed ncu capture (profiles/roofline_traffic.json)
  secondary  (default workload only) the same measurement on C3: the HBM-regime number
  strong     (default workload only) BASELINE.json configs[4] scaled to a bench step: the 10 M-triangle scene at
             3840x2160 with a FIXED total of 128 spp split over the N ranks + the 99.5 MB all-reduce

--impl reference times the reference itself: its own CUDA build
(oracle/_ref/ref_harness, compiled from /root/reference where it lies) on one
B200 — the reference is CUDA-only and has no CPU path (BASELINE.json) — and
falls back to the scalar host-C++ oracle port on the host cores when that
binary is absent.  That arm loads only the host-side library (librtb_host.so:
scene generator), never the product's GPU library.
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene kind, grid, width, height, spp per GPU, max depth, description)
    "c1": (1, 0, 600, 600, 10, 10, "C1 main.cu default: bunny+Cornell box 69,463 tris, 600x600, 10 spp, depth 10"),
    "c2": (1, 0, 1920, 1080, 64, 8, "C2 bunny+Cornell box 69,463 tris, 1920x1080, 64 spp, depth 8, matte + 2 area-light tris, seed 1"),
    "c3": (3, 12, 3840, 2160, 16, 8, "C3 144-bunny field 10,000,956 tris, 3840x2160, 16 spp, depth 8"),
    "c4": (2, 0, 1920, 1080, 64, 16, "C4 bunny+Cornell box, matte/mirror/glass round-robin, 1920x1080, 64 spp, depth 16 + RR"),
    # C5 is STRONG scaling: 1024 spp in total, split evenly over the ranks (the spp entry is the total)
    "c5": (3, 12, 3840, 2160, 1024, 8, "C5 144-bunny field 10,000,956 tris, 3840x2160, 1024 spp in total (sample passes split over the GPUs), depth 8"),
}
# the same scenes given as INSTANCES (rtb_scene_create_instanced, two-level BVH): identical flattened triangles,
# 4 MB of nodes + triangles instead of 600 MB; results equal the flat scene's up to the rounding of the ray transform
WORKLOADS["c3i"] = WORKLOADS["c3"][:6] + ("C3 as instances: 144 placements of one 69,451-triangle bunny + Cornell shell (two-level BVH; flattens to the 10,000,956 triangles of C3), 3840x2160, 16 spp, depth 8",)
WORKLOADS["c5i"] = WORKLOADS["c5"][:6] + ("C5 as instances (two-level BVH; flattens to the 10,000,956 triangles of C5), 3840x2160, 1024 spp in total, depth 8",)
INSTANCED = {"c3i", "c5i"}
STRONG = {"c5", "c5i"}
METRIC = "Mrays/s (extend+shadow)"
STRONG_TOTAL_SPP = 128  # the `strong` record: C5's scene and resolution, 128 spp in total (C5's 1024 spp = 8 such steps)


def config_block(workload, world, spp, total_spp, pool=None, strong=False):
    """the `config` object: the same keys on both arms (the reference arm fills what applies to it)"""
    return {"workload": WORKLOADS[workload][6], "spp_per_gpu": spp, "total_spp": total_spp,
            "sharding": ("sample passes split over the ranks (fixed total)" if strong else "sample pass per rank (64 spp each)") + ", scene replicated, NCCL all-reduce of the accumulation buffer" if world > 1 else "single GPU",
            "pool_size": pool,
            "l2": "256 MB device memset between timed steps (L2 flush)"}


def peaks():
    out = {"hbm": 6650.0, "hbm_source": "fallback (B200_PROFILING.md)", "l2": None, "l2_source": None}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            out["hbm"], out["hbm_source"] = float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        pass
    try:
        with open(os.path.join(ROOT, "profiles", "l2_bandwidth.json")) as f:
            out["l2"] = float(json.load(f)["l2_read_gbs"])
            out["l2_source"] = "builder-measured: tools/l2_bandwidth.cu, 128-bit ld.global.cg over a 64 MB buffer on this pool's B200 (profiles/l2_bandwidth.json); MEASURED_PEAKS.json has no L2 figure"
    except Exception:
        pass
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[4 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def load_scene(L, kind, grid, instanced=False):
    verts, faces = L.load_mesh()
    if instanced:
        return L.host_scene_instanced(kind, verts, faces, grid=grid)
    return L.host_scene(kind, verts, faces, grid=grid)


def plain_params(capi, **kw):
    """rtb_render_params with the defaults of rtb_render_params_default, filled without the GPU library"""
    p = capi.RenderParams()
    p.width, p.height, p.spp, p.max_bounces, p.rr_start, p.rr_threshold, p.seed = 600, 600, 10, 10, 4, 1.0, 1
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def cpu_baseline_port(hs, cam, params, budget_s=12.0, threads=None):
    """the oracle (scalar host-C++ restatement of the reference) on the host cores, bounded sample"""
    from oracle import binding
    threads = threads or os.cpu_count() or 1
    orc = binding.Oracle().scene(hs.desc)
    npix = params.width * params.height
    # sample = evenly spaced blocks of pixels (same spp / depth), sized from a calibration run
    calib = min(npix, 1024)
    start = (npix // 2) - calib // 2
    t0 = time.perf_counter()
    _, _, st = orc.render(cam, params, start, start + calib, threads=threads)
    dt = max(time.perf_counter() - t0, 1e-6)
    n = int(min(npix, max(calib, calib * budget_s / dt)))
    start = (npix - n) // 2
    t0 = time.perf_counter()
    _, _, st = orc.render(cam, params, start, start + n, threads=threads)
    dt = time.perf_counter() - t0
    rays = st[1] + st[2]
    return {"value": rays / dt * 1e-6, "unit": "Mrays/s", "cores": threads, "kind": "port",
            "sample": f"{n} of {npix} pixels (centre block) x {params.spp} spp, depth {params.max_bounces}: "
                      f"{rays} rays in {dt:.2f} s", "seconds": dt, "rays": int(rays)}


def run_reference(args, rank):
    if rank != 0:
        return 0
    from rtcuda_b200 import capi
    from oracle import binding
    kind, grid, W, H, spp, depth, desc_txt = WORKLOADS[args.workload]
    if args.workload in STRONG:
        # the reference's camera_ray_end_id is an int (render.cuh:371): 4K x 1024 spp overflows it; C5 is extrapolated
        # from the reference's ms/spp on C3 (BASELINE.md 3.1)
        print(json.dumps({"impl": "reference", "unavailable": "the reference cannot run 3840x2160x1024 spp in one call (int overflow, render.cuh:371); use --workload c3"}))
        return 0
    L = capi.Lib(capi.HOST_LIB)  # host-side scene generator only: the product's GPU library is not loaded on this arm
    hs = load_scene(L, kind, grid)
    cam = hs.camera(W / H)
    params = plain_params(capi, width=W, height=H, spp=spp, max_bounces=depth)
    line = {"impl": "reference", "metric": METRIC, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_block(args.workload, 1, spp, spp, pool=1 << 20),
            "reference_gpus_used": 1}
    line["config"]["sharding"] = "single GPU (the reference has no multi-GPU path: one GPU whatever --gpus says)"
    line["config"]["l2"] = "none (the reference streams ~293 MB of pools every iteration)"
    harness = binding.REF_HARNESS
    done = False
    if os.path.exists(harness) and not args.reference_cpu:
        try:
            with tempfile.TemporaryDirectory() as td:
                scene_file = os.path.join(td, "scene.rtbs")
                hs.save(scene_file)
                passes = args.warmup + args.steps

                def run(cmd):
                    out = subprocess.run([harness, scene_file] + [str(c) for c in cmd], capture_output=True, text=True, timeout=3000)
                    if out.returncode != 0:
                        raise RuntimeError(out.stderr[-500:])
                    return [json.loads(l[5:]) for l in out.stdout.splitlines() if l.startswith("JSON ")]
                js = run(["loop", W, H, spp, depth, passes, 1])
                scene_js, loop_js = js[0], js[-1]
                ms = loop_js["pass_ms"][args.warmup:]
                rays = loop_js["pass_rays"][args.warmup:]
                value = sum(rays) / sum(ms) * 1e-3
                js2 = run(["render", W, H, spp, depth, args.steps, args.warmup])
                render_js = js2[-1]
                e2e_ms = render_js["ms_per_call"] + js2[0]["bvh_build_ms"]
                line.update({"value": value, "ms_per_step": sum(ms) / len(ms),
                             "reference_kind": "reference CUDA build (unmodified kernels, nvcc -O3 sm_100a) on 1 B200; "
                                               "loop time excludes its cudaMallocs and RNG init",
                             "rays_per_step": rays[0], "ms_per_spp": sum(ms) / len(ms) / spp,
                             "reference_iterations": loop_js["iterations"] // passes,
                             "reference_bvh_build_ms_host": scene_js["bvh_build_ms"],
                             "e2e": {"value": rays[0] / e2e_ms * 1e-3, "unit": "Mrays/s", "h2d_bytes_per_step": 0,
                                     "d2h_bytes_per_step": 0,
                                     "note": "Bvh::Bvh host build + unmodified render() call incl. its mallocs and framebuffer copy"}})
                done = True
        except Exception as e:  # harness unusable on this box: fall through to the CPU port
            line["reference_harness_error"] = str(e)[-300:]
    cb = cpu_baseline_port(hs, cam, params, budget_s=15.0)
    line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if not done:
        line.update({"value": cb["value"], "ms_per_step": cb["seconds"] * 1e3,
                     "reference_kind": "oracle port (scalar host C++ restatement) on host cores",
                     "e2e": {"value": cb["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(line))
    return 0


class Rig:
    """per-rank plumbing: torch device + process group (barrier, NCCL id, timing exchange), the library's context and
    its own NCCL communicator"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        from rtcuda_b200 import capi
        self.torch, self.dist, self.capi = torch, dist, capi
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference --reference-cpu for the oracle)")
        torch.cuda.set_device(self.local_rank)
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        if self.world > 1:
            # (a rank that fails must not leave the others waiting for the default 10 minutes on a GPU lease)
            import datetime
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank), timeout=datetime.timedelta(seconds=240))
        self.L = capi.Lib()
        self.ctx = self.L.context(self.local_rank)
        self.comm = None
        if self.world > 1:  # the library's own communicator: rank 0's id travels over the launcher's process group
            idt = torch.zeros(capi.RTB_COMM_ID_BYTES, dtype=torch.uint8, device="cuda")
            if self.rank == 0:
                idt.copy_(torch.frombuffer(bytearray(capi.Comm.unique_id(self.L)), dtype=torch.uint8))
            dist.broadcast(idt, src=0)
            self.comm = capi.Comm(self.ctx, bytes(idt.cpu().numpy().tobytes()), self.rank, self.world)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce_max(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def reduce_sum(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.item()

    def gather(self, vals):
        if self.world == 1:
            return [vals]
        mine = self.torch.tensor(vals, dtype=self.torch.float64, device="cuda")
        allr = [self.torch.zeros_like(mine) for _ in range(self.world)]
        self.dist.all_gather(allr, mine)
        return [[float(v) for v in t] for t in allr]

    def close(self):
        if self.comm:
            self.comm.close()
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


class Job:
    """one workload resident on this rank's GPU: pinned host copy of the scene, device scene, accumulation buffers"""

    def __init__(self, rig, workload, spp, total_spp, first_sample, pool=0, flags=0, host_scene=None):
        torch, capi = rig.torch, rig.capi
        self.rig, self.workload = rig, workload
        kind, grid, self.W, self.H, _, self.depth, self.desc_txt = WORKLOADS[workload]
        self.instanced = workload in INSTANCED
        self.hs = host_scene or load_scene(rig.L, kind, grid, self.instanced)
        self.cam = self.hs.camera(self.W / self.H)
        self.spp, self.total_spp = spp, total_spp
        self.p = capi.render_params(rig.L, width=self.W, height=self.H, spp=spp, max_bounces=self.depth, first_sample=first_sample,
                                    total_spp=total_spp, pool_size=pool, flags=flags)
        # pinned host copies of the scene arrays: the e2e leg uploads from these every step
        arr = self.hs.arrays()
        self.pin = {k: torch.from_numpy(np.ascontiguousarray(arr[k])).pin_memory() for k in ("vertices", "material_ids", "light_ids")}
        pdesc = capi.SceneDesc()
        C.memmove(C.byref(pdesc), C.byref(self.hs.desc), C.sizeof(pdesc))
        pdesc.vertices = self.pin["vertices"].data_ptr(); pdesc.material_ids = self.pin["material_ids"].data_ptr(); pdesc.light_ids = self.pin["light_ids"].data_ptr()
        self.h2d = sum(t.numel() * t.element_size() for t in self.pin.values()) + self.hs.desc.num_materials * 20 + self.hs.desc.num_lights * 40
        if self.instanced:  # the same pinned geometry, placed by the instance table
            idesc = capi.InstancedSceneDesc()
            C.memmove(C.byref(idesc), C.byref(self.hs.idesc), C.sizeof(idesc))
            idesc.geometry = pdesc
            self.h2d += self.hs.idesc.num_instances * C.sizeof(capi.Instance) + (self.hs.idesc.num_meshes + 1) * 8
            pdesc = idesc
        self.pdesc = pdesc
        self.nfl = 3 * self.W * self.H
        self.scene = rig.ctx.scene(pdesc)
        self.bst = self.scene.stats()
        self.accum = torch.zeros(self.nfl, dtype=torch.float32, device="cuda")
        self.out = torch.empty_like(self.accum)
        self.seg = []  # (after render, after all-reduce) events of the timed steps

    def step(self, timed=False):
        torch, rig = self.rig.torch, self.rig
        self.accum.zero_()
        st = self.scene.render_accumulate(self.cam, self.p, self.accum.data_ptr())
        if rig.world > 1:
            if timed:
                e1 = torch.cuda.Event(enable_timing=True); e1.record()
            rig.comm.allreduce_f32(self.accum.data_ptr(), self.nfl)  # ncclAllReduce on the library's stream, inside the step
            if timed:
                e2 = torch.cuda.Event(enable_timing=True); e2.record()
                self.seg.append((e1, e2))
        rig.ctx.tonemap_device(self.accum.data_ptr(), self.nfl, self.total_spp, self.out.data_ptr())
        return st

    def timed(self, steps, warmup, sampler=None, spin=False):
        """W untimed steps, then K steps bracketed by barrier + synchronize, L2 flushed between steps; returns
        (ms per step as the max over ranks, Mrays/s of the whole job, per-step stats of this rank, clocks)"""
        torch, rig = self.rig.torch, self.rig
        for _ in range(warmup):
            self.step()
        rig.barrier()
        if sampler:
            sampler.start()
        # nvidia-smi needs ~0.1-0.3 s before its first sample and a timed region can be that short: keep the GPU
        # under the same load (untimed steps, EVERY rank alike: each step holds an all-reduce) until the sampler is running
        t_spin = time.perf_counter()
        self.step()
        torch.cuda.synchronize()
        n_extra = torch.tensor([max(0, min(32, int(0.6 / max(time.perf_counter() - t_spin, 1e-3)))) if spin else 0], device="cuda")
        if rig.world > 1:
            rig.dist.broadcast(n_extra, src=0)  # rank 0 decides how many
        for _ in range(int(n_extra.item())):
            self.step()
        rig.barrier()
        self.seg = []
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        stats = []
        for k in range(steps):
            rig.flush.zero_()  # evict L2 between timed steps
            torch.cuda.synchronize()
            ev[k][0].record()
            stats.append(self.step(timed=True))
            ev[k][1].record()
        rig.barrier()
        clocks = sampler.stop() if sampler else None
        ms_steps = [a.elapsed_time(b) for a, b in ev]
        allreduce_ms = sum(a.elapsed_time(b) for a, b in self.seg) / len(self.seg) if self.seg else 0.0
        render_ms = sum(ev[k][0].elapsed_time(self.seg[k][0]) for k in range(len(self.seg))) / len(self.seg) if self.seg else sum(ms_steps) / steps
        per = rig.gather([render_ms, allreduce_ms])
        t_total = rig.reduce_max(sum(ms_steps))
        rays_total = rig.reduce_sum(float(sum(s.extend_rays + s.shadow_rays for s in stats)))
        return {"ms_per_step": t_total / steps, "value": rays_total / t_total * 1e-3, "rays_per_step": rays_total / steps,
                "stats": stats, "clocks": clocks,
                "per_rank": {"render_ms": [round(p[0], 2) for p in per], "allreduce_ms": [round(p[1], 3) for p in per]} if rig.world > 1 else None}

    def roofline(self, steps):
        """the dominant kernel, measured live with ONE wavefront on one stream (the timed steps run four or two
        concurrent wavefronts whose kernels overlap), CUDA events inside rtb_render_accumulate on the render stream"""
        capi, rig = self.rig.capi, self.rig
        ps = capi.RenderParams()
        C.memmove(C.byref(ps), C.byref(self.p), C.sizeof(ps))
        ps.flags |= capi.RTB_RENDER_SINGLE_PIPELINE
        s0 = []
        for _ in range(max(1, min(steps, 3))):
            rig.flush.zero_()
            self.accum.zero_()
            s0.append(self.scene.render_accumulate(self.cam, ps, self.accum.data_ptr()))
        fused = all(s.fused_trace for s in s0)
        tr_ms = sum(s.ms_extend + s.ms_shadow for s in s0); sh_ms = sum(s.ms_shade for s in s0); tot_ms = sum(s.ms_total for s in s0)
        tr_launches = sum(s.extend_launches for s in s0)
        ext_rays = sum(s.extend_rays for s in s0); shd_rays = sum(s.shadow_rays for s in s0)
        pc = capi.render_params(rig.L, width=self.W, height=self.H, spp=max(1, min(2, self.spp)), max_bounces=self.depth,
                                first_sample=self.p.first_sample, total_spp=self.total_spp, flags=capi.RTB_RENDER_COUNT_WORK)
        self.accum.zero_()
        cst = self.scene.render_accumulate(self.cam, pc, self.accum.data_ptr())
        e_nodes = cst.extend_nodes / max(cst.extend_rays, 1); e_tris = cst.extend_tris / max(cst.extend_rays, 1)
        s_nodes = cst.shadow_nodes / max(cst.shadow_rays, 1); s_tris = cst.shadow_tris / max(cst.shadow_rays, 1)
        hit_frac = cst.hits / max(cst.extend_rays, 1)
        # algorithmic bytes (DESIGN.md 4.2): 80 B per node fetched, 48 B per triangle tested; an extend ray reads its
        # 32 B record (origin|pixel, dir|sample) and, when it hits, 16 B (beta) and writes the 48 B hit record; a
        # shadow ray reads 32 B (origin|tmax, dir|excluded) and, unoccluded, 16 B (radiance|pixel) + a 16 B splat
        bytes_extend = e_nodes * 80 + e_tris * 48 + 32 + 64 * hit_frac
        bytes_shadow = s_nodes * 80 + s_tris * 48 + 32 + 32
        rays_per_launch = (ext_rays + shd_rays) / max(tr_launches, 1)
        bytes_per_launch = (bytes_extend * ext_rays + bytes_shadow * shd_rays) / max(tr_launches, 1)
        avg_launch_ms = tr_ms / max(tr_launches, 1)
        achieved = bytes_per_launch / (avg_launch_ms * 1e-3) * 1e-9 if avg_launch_ms > 0 else 0.0
        pk = peaks()
        scene_bytes = self.bst.node_bytes + self.bst.triangle_bytes
        resident = scene_bytes < 100e6  # nodes + triangles stay in the 126 MB L2
        bound = "l2" if resident and pk["l2"] else "hbm"
        peak, peak_src = (pk["l2"], pk["l2_source"]) if bound == "l2" else (pk["hbm"], pk["hbm_source"])
        prof = {}
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                prof = json.load(f).get(self.workload.rstrip("i") if self.workload in ("c3i", "c5i") else {"c5": "c3", "c1": "c2"}.get(self.workload, self.workload), {})
        except Exception:
            pass
        per_ray = prof.get("k_trace_dram_bytes_per_ray")
        traffic = per_ray * rays_per_launch if per_ray is not None else None
        l2_per_ray = prof.get("k_trace_l2_bytes_per_ray")
        # SURVEY 8d floor model: one root-to-leaf descent of a BVH8 with <= 4 triangles per leaf, 80 B nodes, 48 B
        # triangles, 48 B of ray I/O: ceil(log8(n / 4)) * 80 + 4 * 48 + 48 bytes per ray, all of it from HBM
        n_flat = int(self.bst.num_flat_triangles) or int(self.bst.num_triangles)
        floor_bytes = math.ceil(math.log(max(n_flat / 4.0, 8.0), 8)) * 80 + 4 * 48 + 48
        rays_per_s = (ext_rays + shd_rays) / (tr_ms * 1e-3) if tr_ms > 0 else 0.0
        floor_rate = pk["hbm"] * 1e9 / floor_bytes
        return {"bound": bound,
                "kernel": "k_trace<3> (extend + shadow rays, one persistent launch per iteration)" if fused else "k_trace<1> + k_trace<2>",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "traffic": traffic,
                "dram_frac": (traffic / (avg_launch_ms * 1e-3) * 1e-9 / pk["hbm"]) if traffic is not None and avg_launch_ms > 0 else None,
                "hbm_peak": pk["hbm"], "hbm_peak_source": pk["hbm_source"],
                "frac_of_hbm_peak": achieved / pk["hbm"],
                "l2_traffic": l2_per_ray * rays_per_launch if l2_per_ray is not None else None,
                "l2_frac": (l2_per_ray * rays_per_launch / (avg_launch_ms * 1e-3) * 1e-9 / pk["l2"]) if l2_per_ray is not None and pk["l2"] and avg_launch_ms > 0 else None,
                "issue_slot_pct": prof.get("k_trace_issue_slot_pct"), "lanes_per_inst": prof.get("k_trace_lanes_per_inst"),
                "warps_active_pct": prof.get("k_trace_warps_active_pct"), "pipe_pct": prof.get("k_trace_pipe_pct"), "profile_source": prof.get("source"),
                "limiter": "no single unit: issue slots, the ALU pipe and the L1 data pipe each 55-70 % busy at 19-25 of 32 lanes with half the warps an SM "
                           "can hold (64 registers), a third of the stall samples on load latency; not memory bandwidth: "
                           + ("the scene is L2-resident, DRAM carries only the ray / hit queues" if resident else
                              "incoherent rays on a scene 5x the L2: DRAM traffic stays far below the HBM peak"),
                "algorithmic_bytes_per_extend_ray": bytes_extend, "algorithmic_bytes_per_shadow_ray": bytes_shadow,
                "extend_nodes_per_ray": e_nodes, "extend_tris_per_ray": e_tris, "shadow_nodes_per_ray": s_nodes,
                "shadow_tris_per_ray": s_tris, "hit_fraction": hit_frac, "rays_per_launch": rays_per_launch,
                "avg_launch_ms": avg_launch_ms, "launches": int(tr_launches), "timed_with": "single pipeline (kernel alone on one stream), %d steps" % len(s0),
                "single_pipeline_ms_per_step": tot_ms / len(s0),
                "kernel_share_of_step": tr_ms / tot_ms if tot_ms else None,
                "shade_share_of_step": sh_ms / tot_ms if tot_ms else None,
                "floor_model": {"bytes_per_ray": floor_bytes, "rays_per_s_at_hbm_peak": floor_rate, "kernel_rays_per_s": rays_per_s,
                                "frac": rays_per_s / floor_rate,
                                "note": "SURVEY 8d: rays per second of the trace kernel while it runs against the HBM peak divided by the floor-model bytes per ray; "
                                        "above 1 when the scene is served by L1 / L2"},
                "scene_mb": scene_bytes / 1e6}

    def close(self):
        self.scene.close()


DUMP_BYTES = 64_000_000  # --dump-outputs: the most it writes in all


def dump_outputs(outdir, job):
    """the last step's tonemapped image and accumulation buffer (see --dump-outputs in the module docstring)"""
    os.makedirs(outdir, exist_ok=True)
    npix = job.W * job.H
    out = {"image": job.out, "accum": job.accum}
    out = {k: v.view(npix, 3).cpu().numpy() for k, v in out.items()}
    per_pixel = sum(a.itemsize * 3 for a in out.values())
    if npix * per_pixel > DUMP_BYTES:
        keep = (DUMP_BYTES - 4096) // (per_pixel + 8)  # (4096: room for the .npy headers)
        idx = np.sort(np.random.default_rng(0).choice(npix, keep, replace=False))
        out = {k: a[idx] for k, a in out.items()}
        out["pixel_index"] = idx.astype(np.float64)
    else:
        out = {k: a.reshape(job.H, job.W, 3) for k, a in out.items()}
        stale = os.path.join(outdir, "pixel_index.npy")
        if os.path.exists(stale):
            os.remove(stale)
    for k, a in out.items():
        np.save(os.path.join(outdir, k + ".npy"), a)


def e2e_leg(rig, job, steps):
    """end to end through the public API from pinned host buffers, every step: upload + BVH build + render + D2H.
    N = 1: rtb_scene_create + rtb_render.  N > 1, one process per GPU as the driver launches them: every rank
    rtb_scene_create + rtb_render_accumulate, the library's ncclAllReduce (rtb_comm), tonemap + device->host on rank 0."""
    torch, capi, L = rig.torch, rig.capi, rig.L
    host_img = torch.empty(job.nfl, dtype=torch.float32).pin_memory()
    n_e2e = max(1, min(steps, 5))

    def once():
        sc2 = rig.ctx.scene(job.pdesc)  # rtb_scene_create: H2D of the triangle soup + GPU BVH build
        if rig.world == 1:
            st = capi.RenderStats()
            L.check(L.lib.rtb_render(sc2.h, C.byref(job.cam), C.byref(job.p), C.c_void_p(host_img.data_ptr()), C.byref(st)))
        else:
            job.accum.zero_()
            st = sc2.render_accumulate(job.cam, job.p, job.accum.data_ptr())
            rig.comm.allreduce_f32(job.accum.data_ptr(), job.nfl)
            if rig.rank == 0:  # one image leaves the box
                rig.ctx.tonemap_device(job.accum.data_ptr(), job.nfl, job.total_spp, job.out.data_ptr())
                host_img.copy_(job.out)
                torch.cuda.synchronize()
        sc2.close()
        return st
    once()
    rig.barrier()
    t0 = time.perf_counter()
    rays = 0
    for _ in range(n_e2e):
        s = once()
        rays += s.extend_rays + s.shadow_rays
    rig.barrier()
    dt = rig.reduce_max(time.perf_counter() - t0)
    rays = rig.reduce_sum(float(rays))
    return {"value": rays / dt * 1e-6, "unit": "Mrays/s", "h2d_bytes_per_step": int(job.h2d * rig.world), "d2h_bytes_per_step": int(job.nfl * 4),
            "steps": n_e2e, "ms_per_step": dt / n_e2e * 1e3,
            "api": "rtb_scene_create + rtb_render" if rig.world == 1 else
                   "per rank: rtb_scene_create + rtb_render_accumulate + rtb_comm_allreduce_f32; rank 0: rtb_tonemap_device + device->host",
            "note": "scene upload from pinned host memory + GPU BVH build + render + device->host framebuffer (rank 0 only), every step"}


def one_process_leg(rig, job, steps):
    """the same end-to-end step through the ONE-PROCESS entry a reference-style C++ program uses on a multi-GPU box:
    rtb_multi_scene_create + rtb_multi_render drive all N GPUs from rank 0's process (one host thread per GPU, NCCL
    reduce, tonemap and D2H on the first GPU).  The other ranks leave their GPUs idle meanwhile and wait on a HOST-side
    (gloo) barrier: no kernel of theirs may spin on a GPU that another process is rendering on."""
    torch, capi, L = rig.torch, rig.capi, rig.L
    if rig.world == 1:
        return None
    import datetime
    host_group = rig.dist.new_group(backend="gloo", timeout=datetime.timedelta(seconds=240))
    torch.cuda.synchronize()
    rig.dist.barrier(group=host_group)
    res = None
    if rig.rank == 0:
        try:
            host_img = torch.empty(job.nfl, dtype=torch.float32).pin_memory()
            n = max(1, min(steps, 5))
            multi = capi.Multi(L, list(range(rig.world)))
            pm = capi.RenderParams()
            C.memmove(C.byref(pm), C.byref(job.p), C.sizeof(pm))
            pm.spp, pm.first_sample, pm.total_spp = job.total_spp, 0, job.total_spp  # the whole job; the library shards it

            def once():
                ms = multi.scene(job.pdesc)  # H2D + BVH build on every GPU, one host thread each
                _, st = ms.render(job.cam, pm, out=host_img.data_ptr())
                ms.close()
                return st
            once()
            t0 = time.perf_counter()
            rays = 0
            for _ in range(n):
                s = once()
                rays += s.extend_rays + s.shadow_rays
            dt = time.perf_counter() - t0
            multi.close()
            res = {"value": rays / dt * 1e-6, "unit": "Mrays/s", "ms_per_step": dt / n * 1e3, "steps": n,
                   "h2d_bytes_per_step": int(job.h2d * rig.world), "d2h_bytes_per_step": int(job.nfl * 4),
                   "api": "rtb_multi_scene_create + rtb_multi_render (one process, one host thread per GPU, ncclReduce inside the library)"}
        except Exception as e:  # a reported extra: never a reason to lose the line
            res = {"error": str(e)[-300:]}
    rig.dist.barrier(group=host_group)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--pool", type=int, default=0)
    ap.add_argument("--reference-cpu", action="store_true", help="reference arm: force the CPU oracle port")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `secondary` (C3) and `strong` records of the default workload")
    ap.add_argument("--flags", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's image and accumulation buffer to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("bench.py: --steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        raise SystemExit("bench.py: --dump-outputs writes what --impl ours computes")
    # W >= 3 (timing contract); the multi-second C5 steps may run with fewer to fit a GPU lease
    args.warmup = max(args.warmup, 3) if args.impl == "ours" and args.workload not in STRONG else args.warmup
    if args.impl == "reference":
        return run_reference(args, int(os.environ.get("RANK", "0")))

    rig = Rig()
    capi, world, rank = rig.capi, rig.world, rig.rank
    kind, grid, W, H, spp, depth, desc_txt = WORKLOADS[args.workload]
    strong = args.workload in STRONG
    if strong:
        if spp % world:
            raise SystemExit(f"bench.py: {spp} spp do not split evenly over {world} ranks")
        total_spp, spp = spp, spp // world
    else:
        total_spp = spp * world
    job = Job(rig, args.workload, spp, total_spp, rank * spp, pool=args.pool, flags=args.flags)
    res = job.timed(args.steps, args.warmup, sampler=ClockSampler(rig.local_rank) if rank == 0 else None, spin=True)
    stats = res["stats"]
    if args.dump_outputs and rank == 0:  # before the legs below reuse the job's buffers
        dump_outputs(args.dump_outputs, job)
    launches = int(sum(s.kernel_launches for s in stats) + 2 * args.steps)  # + fold into the caller's buffer + tonemap per step
    e2e = e2e_leg(rig, job, args.steps)
    one_proc = one_process_leg(rig, job, args.steps)
    line = None
    if rank == 0:
        roofline = job.roofline(args.steps)
        pool_used = int(stats[0].pool) * int(stats[0].pipelines)  # path slots the render ran with (rtb_render_stats.pool, per wavefront)
        cfg = config_block(args.workload, world, spp, total_spp, pool=pool_used, strong=strong)
        n_types = {"c4": 3}.get(args.workload, 1)
        cfg["l2"] += "; the ray / hit queues (%.1f GB: pool %s) are streamed every iteration" % (
            pool_used * (96 + 48 * n_types) / 1e9, "as asked" if int(job.p.pool_size) else "automatic, an eighth of the free device memory at most")
        line = {"metric": METRIC, "value": res["value"], "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": cfg,
                "ms_per_spp": res["ms_per_step"] / total_spp * (1 if strong else world), "paths_per_step": int(stats[0].paths) * world,
                "rays_per_step": res["rays_per_step"],
                "iterations_per_step": int(stats[0].iterations), "pipelines": int(stats[0].pipelines),
                "per_rank": res["per_rank"], "collective": "ncclAllReduce issued by librtb.so (rtb_comm_allreduce_f32)" if world > 1 else None,
                "bvh_build_ms": job.bst.build_ms, "bvh_nodes": int(job.bst.num_nodes), "bvh_sah": job.bst.sah_cost,
                "e2e": e2e, "e2e_one_process": one_proc, "gpu_launches": launches, "clocks": res["clocks"], "roofline": roofline}
        if job.instanced:
            line["config"]["instances"] = int(job.bst.num_instances)
            line["config"]["stored_triangles"] = int(job.bst.num_triangles)
            line["config"]["flattened_triangles"] = int(job.bst.num_flat_triangles)
    host_scene_c2 = job.hs
    cam_c2, W2, H2, spp2, depth2 = job.cam, W, H, spp, depth
    job.close()
    del job

    # ---- the HBM regime and the north_star scaling config, in the same driver-run line (default workload only) ----
    if args.workload == "c2" and not args.no_extras:
        rig.torch.cuda.empty_cache()
        s_total = STRONG_TOTAL_SPP
        if s_total % world == 0:
            hs3 = load_scene(rig.L, 3, 12)
            if world == 1:  # `secondary`: C3 (16 spp) on one GPU
                j3 = Job(rig, "c3", 16, 16, 0, host_scene=hs3)
                r3 = j3.timed(3, 3)
                if rank == 0:
                    line["secondary"] = {"c3": {"workload": WORKLOADS["c3"][6], "value": r3["value"], "unit": "Mrays/s", "ms_per_step": r3["ms_per_step"],
                                                "ms_per_spp": r3["ms_per_step"] / 16, "steps": 3, "warmup": 3, "rays_per_step": r3["rays_per_step"],
                                                "bvh_build_ms": j3.bst.build_ms, "bvh_nodes": int(j3.bst.num_nodes),
                                                "roofline": j3.roofline(2)}}
                j3.close()
                del j3
            # `strong`: fixed total work, 128 spp of the 4K frame over the N ranks
            js = Job(rig, "c5", s_total // world, s_total, rank * (s_total // world), host_scene=hs3)
            rs = js.timed(2, 1)
            if rank == 0:
                line["strong"] = {"workload": "C5's scene and frame (144-bunny field 10,000,956 tris, 3840x2160, depth 8) with %d spp in TOTAL, split over the ranks" % s_total,
                                  "total_spp": s_total, "spp_per_gpu": s_total // world, "n_gpus": world, "steps": 2, "warmup": 1,
                                  "ms_per_step": rs["ms_per_step"], "value": rs["value"], "unit": "Mrays/s", "rays_per_step": rs["rays_per_step"],
                                  "per_rank": rs["per_rank"], "allreduce_bytes": js.nfl * 4,
                                  "note": "efficiency at N GPUs = ms_per_step(1) / (N * ms_per_step(N)); scene + BVH replicated (built once per rank, outside the step), "
                                          "the all-reduce of the 99.5 MB accumulation buffer is inside"}
            js.close()
            del js
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline and args.workload not in INSTANCED:  # (the oracle would need the 10 M flattened triangles)
            pcb = plain_params(capi, width=W2, height=H2, spp=spp2, max_bounces=depth2)
            cb = cpu_baseline_port(host_scene_c2, cam_c2, pcb)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
            try:  # SURVEY 8d: the same port on ONE host thread as well (smaller sample)
                c1 = cpu_baseline_port(host_scene_c2, cam_c2, pcb, budget_s=4.0, threads=1)
                line["cpu_baseline"]["one_thread"] = {"value": c1["value"], "unit": c1["unit"], "cores": 1, "sample": c1["sample"]}
            except Exception as e:  # (a reported extra, never a reason to lose the line)
                line["cpu_baseline"]["one_thread"] = {"error": str(e)}
        print(json.dumps(line))
    rig.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
