"""ctypes binding of the C ABI in include/rtb.h (plumbing only).

`load()` opens the CUDA library `librtb.so` next to this file and raises if
it is missing: there is no CPU fallback in the product path.  Tests may pass
an explicit path (tests/emu/librtb_emu.so is a host build of the same kernel
bodies used only to check logic without a GPU).
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.environ.get("RTB_LIB") or os.path.join(HERE, "librtb.so")  # RTB_LIB: A/B builds (tuning runs only)
HOST_LIB = os.path.join(HERE, "librtb_host.so")  # the host-side part alone: scene generators, mesh / scene / PPM I/O (no CUDA)
BUNNY_BIN = os.path.join(HERE, "data", "bunny.rtbm")

RTB_SCENE_S1, RTB_SCENE_S1_MIXED, RTB_SCENE_S2, RTB_SCENE_S1_GLOSSY = 1, 2, 3, 4
RTB_MATTE, RTB_MIRROR, RTB_GLASS, RTB_GLOSSY = 0, 1, 2, 3
RTB_RENDER_PIXEL_CENTRE, RTB_RENDER_NO_SHADOW, RTB_RENDER_NONPERSISTENT, RTB_RENDER_COUNT_WORK = 1, 2, 4, 8
RTB_RENDER_SINGLE_PIPELINE = 16
RTB_RENDER_TRUE_MIS, RTB_RENDER_RR_TERMINATE, RTB_RENDER_DETERMINISTIC = 32, 64, 128
RTB_BUILDER_PLOC, RTB_BUILDER_BINNED_SAH = 0, 1


def treelet_passes(k):
    """RTB_BUILDER_TREELET_PASSES(k), k = 0..8: or it into the builder, e.g. RTB_BUILDER_PLOC | treelet_passes(3)"""
    return k << 8


RTB_COLLAPSE_LARGEST_FIRST, RTB_COLLAPSE_SAH_OPTIMAL = 0, 1


class Material(C.Structure):
    _fields_ = [("albedo", C.c_float * 3), ("ior", C.c_float), ("type", C.c_int32)]


class Light(C.Structure):
    _fields_ = [("type", C.c_int32), ("pos", C.c_float * 3), ("triangle", C.c_int64),
                ("L", C.c_float * 3), ("_pad", C.c_int32)]


class Camera(C.Structure):
    _fields_ = [("lookfrom", C.c_float * 3), ("upper_left", C.c_float * 3),
                ("horizontal", C.c_float * 3), ("vertical", C.c_float * 3)]


class SceneDesc(C.Structure):
    _fields_ = [("num_triangles", C.c_int64), ("vertices", C.c_void_p), ("material_ids", C.c_void_p),
                ("light_ids", C.c_void_p), ("num_materials", C.c_int32), ("materials", C.c_void_p),
                ("num_lights", C.c_int32), ("lights", C.c_void_p)]


class Instance(C.Structure):
    _fields_ = [("mesh", C.c_int32), ("material", C.c_int32), ("xform", C.c_float * 12)]


class InstancedSceneDesc(C.Structure):
    _fields_ = [("geometry", SceneDesc), ("num_meshes", C.c_int32), ("mesh_first", C.c_void_p),
                ("num_instances", C.c_int32), ("instances", C.c_void_p)]


class BuildParams(C.Structure):
    _fields_ = [("builder", C.c_int32), ("ploc_radius", C.c_int32), ("max_leaf_tris", C.c_int32),
                ("collapse", C.c_int32)]


class BvhStats(C.Structure):
    _fields_ = [("num_triangles", C.c_int64), ("num_bvh2_nodes", C.c_int64), ("num_nodes", C.c_int64),
                ("node_bytes", C.c_int64), ("triangle_bytes", C.c_int64), ("sah_cost", C.c_float),
                ("build_ms", C.c_float), ("ploc_iterations", C.c_int32), ("collapse_levels", C.c_int32),
                ("scene_bounds", C.c_float * 6), ("num_instances", C.c_int64), ("num_flat_triangles", C.c_int64),
                ("num_top_nodes", C.c_int64)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("max_bounces", C.c_int32),
                ("rr_start", C.c_int32), ("rr_threshold", C.c_float), ("seed", C.c_uint32),
                ("first_sample", C.c_int32), ("total_spp", C.c_int32), ("pool_size", C.c_int32),
                ("flags", C.c_int32), ("device_mask", C.c_uint32), ("env_L", C.c_float * 3), ("_reserved2", C.c_int32)]


class RenderStats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("extend_rays", C.c_uint64), ("shadow_rays", C.c_uint64),
                ("iterations", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("extend_nodes", C.c_uint64), ("extend_tris", C.c_uint64), ("shadow_nodes", C.c_uint64),
                ("shadow_tris", C.c_uint64), ("extend_launches", C.c_uint64), ("shadow_launches", C.c_uint64), ("hits", C.c_uint64),
                ("ms_total", C.c_float), ("ms_extend", C.c_float), ("ms_shadow", C.c_float), ("ms_other", C.c_float),
                ("ms_shade", C.c_float), ("fused_trace", C.c_int32), ("pipelines", C.c_int32), ("pool", C.c_int32)]


RAY_DTYPE = np.dtype([("origin", np.float32, 3), ("dir", np.float32, 3), ("tmax", np.float32)])
HIT_DTYPE = np.dtype([("t", np.float32), ("u", np.float32), ("v", np.float32), ("prim", np.int32)])

# every symbol include/rtb.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    "rtb_last_error", "rtb_version", "rtb_context_create", "rtb_context_destroy", "rtb_context_device",
    "rtb_build_params_default", "rtb_scene_create", "rtb_scene_create_from_primitives", "rtb_scene_destroy",
    "rtb_scene_stats", "rtb_trace_closest", "rtb_trace_any", "rtb_trace_closest_device", "rtb_trace_any_device",
    "rtb_trace_closest_counts", "rtb_render_aovs", "rtb_camera_look_at", "rtb_camera_primary_rays", "rtb_render_params_default",
    "rtb_render", "rtb_render_accumulate", "rtb_tonemap_device", "rtb_mesh_load_ply", "rtb_mesh_load_bin",
    "rtb_mesh_save_bin", "rtb_free", "rtb_host_scene_build", "rtb_host_scene_desc", "rtb_host_scene_camera",
    "rtb_host_scene_destroy", "rtb_scene_desc_save", "rtb_host_scene_load", "rtb_write_ppm",
    "rtb_scene_create_instanced", "rtb_host_scene_build_instanced", "rtb_host_scene_instanced_desc", "rtb_instanced_flatten",
    "rtb_trace_wavefront", "rtb_kat_eval", "rtb_context_set_option", "rtb_context_get_option",
    "rtb_render_accumulate_fixed", "rtb_tonemap_fixed_device",
    "rtb_multi_create", "rtb_multi_destroy", "rtb_multi_size", "rtb_multi_context", "rtb_multi_scene_create",
    "rtb_multi_scene_create_instanced", "rtb_multi_scene_replicate", "rtb_multi_scene_destroy", "rtb_multi_render", "rtb_render_multi",
    "rtb_scene_attach_lights", "rtb_accum_create", "rtb_accum_destroy", "rtb_accum_add_samples", "rtb_accum_samples",
    "rtb_accum_resolve", "rtb_accum_save", "rtb_accum_load", "rtb_comm_unique_id", "rtb_comm_create", "rtb_comm_destroy", "rtb_comm_allreduce_f32", "rtb_comm_allreduce_i64",
    "rtb_scene_refit", "rtb_scene_refit_device", "rtb_scene_set_instances",
]
RTB_COMM_ID_BYTES = 128
RTB_KAT_TRI_INTERSECT, RTB_KAT_OFFSET_ORIGIN, RTB_KAT_RAND4, RTB_KAT_SAMPLE_F, RTB_KAT_SLAB, RTB_KAT_SAMPLE_LI = 1, 2, 3, 4, 5, 6
KAT_FLOATS = {1: (16, 4), 2: (6, 3), 3: (4, 4), 4: (16, 12), 5: (20, 1), 6: (16, 8)}  # floats per record: (in, out)


class RtbError(RuntimeError):
    pass


def load(path=None):
    path = path or DEFAULT_LIB
    if not os.path.exists(path):
        raise RtbError(f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(the CUDA library is required; there is no CPU fallback)")
    lib = C.CDLL(path)
    lib.rtb_last_error.restype = C.c_char_p
    lib.rtb_version.restype = C.c_char_p
    lib.rtb_free.restype = None
    return lib


class Lib:
    """Thin object wrapper; every call raises RtbError on a non-zero status."""

    def __init__(self, path=None):
        self.lib = load(path)

    def check(self, rc):
        if rc != 0:
            raise RtbError(f"rtb status {rc}: {self.lib.rtb_last_error().decode()}")

    # ---- host side ----
    def load_mesh(self, path=BUNNY_BIN):
        v, f = C.c_void_p(), C.c_void_p()
        nv, nf = C.c_int64(), C.c_int64()
        fn = self.lib.rtb_mesh_load_ply if path.endswith(".ply") else self.lib.rtb_mesh_load_bin
        self.check(fn(path.encode(), C.byref(v), C.byref(nv), C.byref(f), C.byref(nf)))
        verts = np.ctypeslib.as_array(C.cast(v, C.POINTER(C.c_float)), (nv.value, 3)).copy()
        faces = np.ctypeslib.as_array(C.cast(f, C.POINTER(C.c_int32)), (nf.value, 3)).copy()
        self.lib.rtb_free(v)
        self.lib.rtb_free(f)
        return verts, faces

    def host_scene(self, kind, verts, faces, grid=0, seed=1234):
        return HostScene(self, kind, verts, faces, grid, seed)

    def host_scene_instanced(self, kind, verts, faces, grid=0, seed=1234):
        """instanced form of a procedural scene: .idesc is the rtb_instanced_scene_desc"""
        return HostScene(self, kind, verts, faces, grid, seed, instanced=True)

    def flatten(self, idesc):
        """the flat HostScene an instanced description stands for"""
        h = C.c_void_p()
        self.check(self.lib.rtb_instanced_flatten(C.byref(idesc), C.byref(h)))
        return HostScene(self, handle=h)

    def camera_look_at(self, lookfrom, lookat, up, vfov, aspect):
        cam = Camera()
        a = (C.c_float * 3)(*lookfrom); b = (C.c_float * 3)(*lookat); c = (C.c_float * 3)(*up)
        self.check(self.lib.rtb_camera_look_at(a, b, c, C.c_float(vfov), C.c_float(aspect), C.byref(cam)))
        return cam

    def primary_rays(self, cam, w, h):
        rays = np.zeros(w * h, dtype=RAY_DTYPE)
        self.check(self.lib.rtb_camera_primary_rays(C.byref(cam), w, h, rays.ctypes.data_as(C.c_void_p)))
        return rays

    def write_ppm(self, path, rgb, w, h):
        rgb = np.ascontiguousarray(rgb, dtype=np.float32)
        self.check(self.lib.rtb_write_ppm(path.encode(), rgb.ctypes.data_as(C.c_void_p), w, h))

    # ---- device side ----
    def context(self, device=0):
        return Context(self, device)


class HostScene:
    def __init__(self, L, kind=None, verts=None, faces=None, grid=0, seed=1234, instanced=False, handle=None):
        self.L = L
        self.h = handle if handle is not None else C.c_void_p()
        if handle is None:
            verts = np.ascontiguousarray(verts, dtype=np.float32)
            faces = np.ascontiguousarray(faces, dtype=np.int32)
            fn = L.lib.rtb_host_scene_build_instanced if instanced else L.lib.rtb_host_scene_build
            L.check(fn(kind, verts.ctypes.data_as(C.c_void_p), C.c_int64(len(verts)), faces.ctypes.data_as(C.c_void_p),
                       C.c_int64(len(faces)), grid, C.c_uint32(seed), C.byref(self.h)))
        self.desc = SceneDesc()
        L.check(L.lib.rtb_host_scene_desc(self.h, C.byref(self.desc)))
        self.idesc = None
        if instanced:
            self.idesc = InstancedSceneDesc()
            L.check(L.lib.rtb_host_scene_instanced_desc(self.h, C.byref(self.idesc)))

    def arrays(self):
        """numpy views of the description (valid while this object lives)."""
        d = self.desc
        n = d.num_triangles
        return dict(
            vertices=np.ctypeslib.as_array(C.cast(d.vertices, C.POINTER(C.c_float)), (n, 9)),
            material_ids=np.ctypeslib.as_array(C.cast(d.material_ids, C.POINTER(C.c_int32)), (n,)),
            light_ids=np.ctypeslib.as_array(C.cast(d.light_ids, C.POINTER(C.c_int32)), (n,)),
            materials=np.ctypeslib.as_array(C.cast(d.materials, C.POINTER(Material)), (d.num_materials,)),
            lights=np.ctypeslib.as_array(C.cast(d.lights, C.POINTER(Light)), (d.num_lights,)) if d.num_lights else None,
        )

    def camera(self, aspect):
        cam = Camera()
        self.L.check(self.L.lib.rtb_host_scene_camera(self.h, C.c_float(aspect), C.byref(cam)))
        return cam

    def save(self, path):
        self.L.check(self.L.lib.rtb_scene_desc_save(path.encode(), C.byref(self.desc)))

    def __del__(self):
        try:
            if self.h:
                self.L.lib.rtb_host_scene_destroy(self.h)
        except Exception:
            pass


class Context:
    def __init__(self, L, device=0):
        self.L = L
        self.h = C.c_void_p()
        L.check(L.lib.rtb_context_create(device, C.byref(self.h)))

    def scene(self, desc, build_params=None):
        """desc: SceneDesc (flat) or InstancedSceneDesc (two-level BVH)"""
        return Scene(self, desc, build_params)

    def set_option(self, name, value):
        self.L.check(self.L.lib.rtb_context_set_option(self.h, name.encode(), C.c_int64(value)))

    def get_option(self, name):
        v = C.c_int64()
        self.L.check(self.L.lib.rtb_context_get_option(self.h, name.encode(), C.byref(v)))
        return v.value

    def kat(self, which, records):
        """evaluate one device function per record (rtb_kat_eval); records: float32 [n, KAT_FLOATS[which][0]]"""
        ni, no = KAT_FLOATS[which]
        a = np.ascontiguousarray(records, dtype=np.float32).reshape(-1, ni)
        out = np.zeros((len(a), no), np.float32)
        self.L.check(self.L.lib.rtb_kat_eval(self.h, which, a.ctypes.data_as(C.c_void_p), C.c_int64(len(a)), out.ctypes.data_as(C.c_void_p)))
        return out

    def tonemap_device(self, d_accum_ptr, num_floats, total_spp, d_out_ptr):
        self.L.check(self.L.lib.rtb_tonemap_device(self.h, C.c_void_p(d_accum_ptr), C.c_int64(num_floats),
                                                   total_spp, C.c_void_p(d_out_ptr)))

    def tonemap_fixed_device(self, d_accum_fixed_ptr, num_values, total_spp, d_out_ptr):
        self.L.check(self.L.lib.rtb_tonemap_fixed_device(self.h, C.c_void_p(d_accum_fixed_ptr), C.c_int64(num_values),
                                                         total_spp, C.c_void_p(d_out_ptr)))

    def __del__(self):
        try:
            if self.h:
                self.L.lib.rtb_context_destroy(self.h)
        except Exception:
            pass


def render_params(L, **kw):
    p = RenderParams()
    L.check(L.lib.rtb_render_params_default(C.byref(p)))
    for k, v in kw.items():
        if k == "env_L":
            p.env_L[0], p.env_L[1], p.env_L[2] = v
        else:
            setattr(p, k, v)
    return p


class Scene:
    def __init__(self, ctx, desc, build_params=None):
        self.ctx, self.L = ctx, ctx.L
        self.h = C.c_void_p()
        bp = C.byref(build_params) if build_params is not None else None
        create = self.L.lib.rtb_scene_create_instanced if isinstance(desc, InstancedSceneDesc) else self.L.lib.rtb_scene_create
        self.L.check(create(ctx.h, C.byref(desc), bp, C.byref(self.h)))

    def stats(self):
        s = BvhStats()
        self.L.check(self.L.lib.rtb_scene_stats(self.h, C.byref(s)))
        return s

    def trace_closest(self, rays):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.zeros(len(rays), dtype=HIT_DTYPE)
        self.L.check(self.L.lib.rtb_trace_closest(self.h, rays.ctypes.data_as(C.c_void_p), C.c_int64(len(rays)),
                                                  hits.ctypes.data_as(C.c_void_p)))
        return hits

    def trace_any(self, rays, excluded=None):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        occ = np.zeros(len(rays), dtype=np.uint8)
        ex = None
        if excluded is not None:
            excluded = np.ascontiguousarray(excluded, dtype=np.int32)
            ex = excluded.ctypes.data_as(C.c_void_p)
        self.L.check(self.L.lib.rtb_trace_any(self.h, rays.ctypes.data_as(C.c_void_p), ex, C.c_int64(len(rays)),
                                              occ.ctypes.data_as(C.c_void_p)))
        return occ

    def trace_wavefront(self, rays=None, shadow_rays=None, excluded=None):
        """closest hits / occlusion through the render path's persistent kernel (rtb_trace_wavefront);
        returns (hits or None, occluded or None, trace launches)"""
        n = ns = 0
        pr = ph = ps = pe = po = None
        hits = occ = None
        if rays is not None and len(rays):
            rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE); n = len(rays)
            hits = np.zeros(n, dtype=HIT_DTYPE)
            pr, ph = rays.ctypes.data_as(C.c_void_p), hits.ctypes.data_as(C.c_void_p)
        if shadow_rays is not None and len(shadow_rays):
            shadow_rays = np.ascontiguousarray(shadow_rays, dtype=RAY_DTYPE); ns = len(shadow_rays)
            occ = np.zeros(ns, dtype=np.uint8)
            ps, po = shadow_rays.ctypes.data_as(C.c_void_p), occ.ctypes.data_as(C.c_void_p)
            if excluded is not None:
                excluded = np.ascontiguousarray(excluded, dtype=np.int32)
                pe = excluded.ctypes.data_as(C.c_void_p)
        launches = C.c_int32()
        self.L.check(self.L.lib.rtb_trace_wavefront(self.h, pr, C.c_int64(n), ph, ps, pe, C.c_int64(ns), po, C.byref(launches)))
        return hits, occ, launches.value

    def trace_counts(self, rays):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        a, b = C.c_double(), C.c_double()
        self.L.check(self.L.lib.rtb_trace_closest_counts(self.h, rays.ctypes.data_as(C.c_void_p),
                                                         C.c_int64(len(rays)), C.byref(a), C.byref(b)))
        return a.value, b.value

    def refit(self, verts):
        """new vertex positions (float32 [num_triangles, 9], caller order; object space for an instanced scene): the tree
        keeps its topology and gets new boxes (rtb_scene_refit)"""
        verts = np.ascontiguousarray(verts, dtype=np.float32)
        if verts.size != 9 * self.stats().num_triangles:
            raise RtbError(f"refit: {verts.size} floats for {self.stats().num_triangles} triangles (9 per triangle)")
        self.L.check(self.L.lib.rtb_scene_refit(self.h, verts.ctypes.data_as(C.c_void_p)))

    def refit_device(self, d_vertices_ptr):
        """rtb_scene_refit_device from 9 floats per triangle in device memory (ready on the device); returns its GPU ms"""
        ms = C.c_float()
        self.L.check(self.L.lib.rtb_scene_refit_device(self.h, C.c_void_p(d_vertices_ptr), C.byref(ms)))
        return ms.value

    def set_instances(self, instances):
        """new transforms / materials for the instances of an instanced scene (a ctypes array of Instance, same count,
        same meshes): rtb_scene_set_instances"""
        self.L.check(self.L.lib.rtb_scene_set_instances(self.h, C.cast(instances, C.c_void_p), len(instances)))

    def render_aovs(self, cam, width, height):
        """primary-hit feature buffers: (albedo[h,w,3], normal[h,w,3], depth[h,w], prim[h,w])"""
        al = np.zeros((height, width, 3), np.float32); no = np.zeros((height, width, 3), np.float32)
        de = np.zeros((height, width), np.float32); pr = np.zeros((height, width), np.int32)
        self.L.check(self.L.lib.rtb_render_aovs(self.h, C.byref(cam), width, height, al.ctypes.data_as(C.c_void_p),
                                                no.ctypes.data_as(C.c_void_p), de.ctypes.data_as(C.c_void_p), pr.ctypes.data_as(C.c_void_p)))
        return al, no, de, pr

    def render(self, cam, params):
        out = np.zeros((params.height, params.width, 3), dtype=np.float32)
        st = RenderStats()
        self.L.check(self.L.lib.rtb_render(self.h, C.byref(cam), C.byref(params), out.ctypes.data_as(C.c_void_p),
                                           C.byref(st)))
        return out, st

    def render_accumulate(self, cam, params, d_accum_ptr):
        st = RenderStats()
        self.L.check(self.L.lib.rtb_render_accumulate(self.h, C.byref(cam), C.byref(params),
                                                      C.c_void_p(d_accum_ptr), C.byref(st)))
        return st

    def render_accumulate_fixed(self, cam, params, d_accum_fixed_ptr):
        """adds this call's fixed-point radiance sums into the int64[3*W*H] device buffer at d_accum_fixed_ptr"""
        st = RenderStats()
        self.L.check(self.L.lib.rtb_render_accumulate_fixed(self.h, C.byref(cam), C.byref(params),
                                                            C.c_void_p(d_accum_fixed_ptr), C.byref(st)))
        return st

    def close(self):
        if self.h:
            self.L.lib.rtb_scene_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Multi:
    """several GPUs driven from this process (rtb_multi): contexts + their NCCL communicator"""

    def __init__(self, L, devices):
        self.L = L
        self.h = C.c_void_p()
        arr = (C.c_int32 * len(devices))(*devices)
        L.check(L.lib.rtb_multi_create(arr, len(devices), C.byref(self.h)))
        self.n = len(devices)

    def context(self, i):
        """borrowed Context of member i (not destroyed by this wrapper)"""
        c = Context.__new__(Context)
        c.L, c.h = self.L, C.c_void_p()
        self.L.check(self.L.lib.rtb_multi_context(self.h, i, C.byref(c.h)))
        c.__class__ = BorrowedContext
        return c

    def scene(self, desc, build_params=None):
        return MultiScene(self, desc, build_params)

    def replicate(self, primary):
        return MultiScene(self, None, None, primary=primary)

    def close(self):
        if self.h:
            self.L.lib.rtb_multi_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BorrowedContext(Context):
    def __del__(self):
        pass


class MultiScene:
    def __init__(self, multi, desc, build_params=None, primary=None):
        self.multi, self.L = multi, multi.L
        self.h = C.c_void_p()
        self.primary = primary  # keep alive: the replica set borrows it
        bp = C.byref(build_params) if build_params is not None else None
        if primary is not None:
            self.L.check(self.L.lib.rtb_multi_scene_replicate(multi.h, primary.h, C.byref(self.h)))
        elif isinstance(desc, InstancedSceneDesc):
            self.L.check(self.L.lib.rtb_multi_scene_create_instanced(multi.h, C.byref(desc), bp, C.byref(self.h)))
        else:
            self.L.check(self.L.lib.rtb_multi_scene_create(multi.h, C.byref(desc), bp, C.byref(self.h)))

    def render(self, cam, params, out=None):
        """params.spp samples per pixel in TOTAL, split over the GPUs params.device_mask selects"""
        if out is None:
            out = np.zeros((params.height, params.width, 3), dtype=np.float32)
        st = RenderStats()
        ptr = out.ctypes.data_as(C.c_void_p) if isinstance(out, np.ndarray) else C.c_void_p(out)
        self.L.check(self.L.lib.rtb_multi_render(self.h, C.byref(cam), C.byref(params), ptr, C.byref(st)))
        return out, st

    def close(self):
        if self.h:
            self.L.lib.rtb_multi_scene_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Comm:
    """one process per GPU: NCCL communicator owned by the library (rtb_comm)"""

    def __init__(self, ctx, id_bytes, rank, world):
        self.ctx, self.L = ctx, ctx.L
        self.h = C.c_void_p()
        buf = (C.c_uint8 * RTB_COMM_ID_BYTES).from_buffer_copy(bytes(id_bytes))
        self.L.check(self.L.lib.rtb_comm_create(ctx.h, buf, rank, world, C.byref(self.h)))

    @staticmethod
    def unique_id(L):
        buf = (C.c_uint8 * RTB_COMM_ID_BYTES)()
        L.check(L.lib.rtb_comm_unique_id(buf))
        return bytes(buf)

    def allreduce_f32(self, d_ptr, n):
        self.L.check(self.L.lib.rtb_comm_allreduce_f32(self.h, C.c_void_p(d_ptr), C.c_int64(n)))

    def allreduce_i64(self, d_ptr, n):
        self.L.check(self.L.lib.rtb_comm_allreduce_i64(self.h, C.c_void_p(d_ptr), C.c_int64(n)))

    def close(self):
        if self.h:
            self.L.lib.rtb_comm_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Accum:
    """progressive accumulation buffer + sample counter (rtb_accum): add passes, resolve, save / load"""

    def __init__(self, ctx, width=0, height=0, deterministic=False, path=None):
        self.ctx, self.L = ctx, ctx.L
        self.h = C.c_void_p()
        if path is not None:
            self.L.check(self.L.lib.rtb_accum_load(ctx.h, path.encode(), C.byref(self.h)))
        else:
            self.L.check(self.L.lib.rtb_accum_create(ctx.h, width, height, 1 if deterministic else 0, C.byref(self.h)))
        self.width, self.height = width, height

    @property
    def samples(self):
        return self.L.lib.rtb_accum_samples(self.h)

    def add(self, scene, cam, params):
        st = RenderStats()
        self.L.check(self.L.lib.rtb_accum_add_samples(self.h, scene.h, C.byref(cam), C.byref(params), C.byref(st)))
        return st

    def resolve(self, width, height):
        out = np.zeros((height, width, 3), np.float32)
        self.L.check(self.L.lib.rtb_accum_resolve(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    def save(self, path):
        self.L.check(self.L.lib.rtb_accum_save(self.h, path.encode()))

    def close(self):
        if self.h:
            self.L.lib.rtb_accum_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
