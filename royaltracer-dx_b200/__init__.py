"""royaltracer-dx_b200 — B200-native wavefront path tracer behind the DXR seam of ML200/RoyalTracer-DX.

Python side: ctypes bindings of the C ABI (include/rtx_b200.h, librtx_b200.so: CUDA sm_100a) and of the C++ host
mirror of the reference's Renderer slices (host/Renderer.cpp, librtx_host.so).  There is no CPU fallback: if the CUDA
library is missing the import of `Context` fails loudly, and every compute entry point returns an error without a GPU.

The directory name has a hyphen (it is the reference's name); import it with
    import importlib; rtdx = importlib.import_module("royaltracer-dx_b200")
or through the repo-root shim `rtdx.py`.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RTX_B200_LIB") or os.path.join(HERE, "librtx_b200.so")   # the override is for A/B builds of the kernels
HOST_LIB_PATH = os.path.join(HERE, "librdx_prep.so")       # host-side data preparation (no engine inside; the C++ Renderer class lives in
HOST_FULL_LIB_PATH = os.path.join(HERE, "librtx_host.so")  # librtx_host.so, which links the engine)

# ---------------------------------------------------------------------------------------------- POD layouts (SURVEY §8a S-rows)
vertex_dt = np.dtype([("position", "<f4", 3), ("normal_material", "<f4", 4)])
material_dt = np.dtype([("Kd", "<f4", 4), ("Ks", "<f4", 3), ("Ni", "<f4"), ("Ke", "<f4", 3), ("pad0", "<f4"),
                        ("Pr_Pm_Ps_Pc", "<f4", 4), ("LUT", "<f4", 16)])
props_dt = np.dtype([("objectToWorld", "<f4", 16), ("objectToWorldInverse", "<f4", 16), ("prevObjectToWorld", "<f4", 16),
                     ("prevObjectToWorldInverse", "<f4", 16), ("objectToWorldNormal", "<f4", 16), ("prevObjectToWorldNormal", "<f4", 16)])
light_dt = np.dtype([("x", "<f4", 3), ("cdf", "<f4"), ("y", "<f4", 3), ("instanceID", "<u4"), ("z", "<f4", 3), ("weight", "<f4"),
                     ("emission", "<f4", 3), ("triCount", "<u4"), ("total_weight", "<f4"), ("pad0", "<f4", 3)])
camera_dt = np.dtype([("view", "<f4", 16), ("projection", "<f4", 16), ("viewI", "<f4", 16), ("projectionI", "<f4", 16),
                      ("prevView", "<f4", 16), ("prevProjection", "<f4", 16), ("time", "<f4"), ("pad", "<f4", 31)])
desc_dt = np.dtype([("transform", "<f4", (3, 4)), ("instance_id_mask", "<u4"), ("hit_group_flags", "<u4"), ("blas", "<u8")])
ray_dt = np.dtype([("origin", "<f4", 3), ("tmin", "<f4"), ("direction", "<f4", 3), ("tmax", "<f4")])
hit_dt = np.dtype([("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("prim", "<u4"), ("inst", "<u4")])
assert vertex_dt.itemsize == 28 and material_dt.itemsize == 128 and props_dt.itemsize == 384 and light_dt.itemsize == 80
assert camera_dt.itemsize == 512 and desc_dt.itemsize == 64 and ray_dt.itemsize == 32 and hit_dt.itemsize == 20

FLAG_JITTER, FLAG_LAMBERT_ONLY, FLAG_RESTIR, FLAG_LEGACY_RR, FLAG_FAST_MATH = 1, 2, 8, 16, 32
OPT_TRACE_STATS, OPT_STAGE_TIMING, OPT_PASS_PARTS, OPT_TLAS_REBUILD, OPT_TRACE_FETCH_TH, OPT_TRACE_SCHED, OPT_TRACE_WAVES, OPT_QUEUE_LPT, OPT_TRACE_CTAS, OPT_PASS_GRAPH, OPT_SHADOW_OVERLAP, OPT_PART_ROWS, OPT_PASS_PIPELINE, OPT_FRAME_PIPELINE = 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14
UPDATE_REFIT, UPDATE_REBUILD = 0, 1       # rtx_update_model* modes (include/rtx_b200.h)
MISS = 0xFFFFFFFF
STAGE_NAMES = ["generate", "closest", "any", "shade_primary", "di_finish", "gi_step", "scatter", "finalize", "accumulate"]


class RtxConfig(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("width", C.c_uint32), ("height", C.c_uint32),
                ("bounces", C.c_uint32), ("nee_samples", C.c_uint32), ("nee_samples_di", C.c_uint32), ("flags", C.c_uint32),
                ("samples_per_pass", C.c_uint32), ("stream", C.c_void_p)]


class RtxCounters(C.Structure):
    _fields_ = [("closest_rays", C.c_uint64), ("shadow_rays", C.c_uint64), ("paths", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("nodes_visited", C.c_uint64), ("tris_tested", C.c_uint64), ("instances_entered", C.c_uint64),
                ("shading_replays", C.c_uint64)]


class RtxBlasInfo(C.Structure):
    _fields_ = [("n_nodes", C.c_uint32), ("n_tris", C.c_uint32), ("bytes", C.c_uint64), ("sah_cost", C.c_float), ("build_ms", C.c_float)]


# every symbol include/rtx_b200.h declares (tests check the library exports all of them)
ABI_SYMBOLS = ["rtx_last_error", "rtx_create", "rtx_destroy", "rtx_upload_model", "rtx_update_model", "rtx_update_model_device",
               "rtx_blas_info_get", "rtx_set_material_ids",
               "rtx_set_materials", "rtx_set_instances", "rtx_set_emissive_triangles", "rtx_set_camera", "rtx_render_pass",
               "rtx_reset_accum", "rtx_synchronize", "rtx_read_accum", "rtx_read_output", "rtx_read_output_async", "rtx_wait_output", "rtx_set_resolve_source",
               "rtx_accum_device_ptr", "rtx_trace",
               "rtx_trace_device", "rtx_trace_stats", "rtx_get_counters", "rtx_reset_counters", "rtx_last_pass_ms", "rtx_last_pass_stage_ms", "rtx_set_option", "rtx_debug_pixel",
               "rtx_selftest_dmath", "rtx_render_frame", "rtx_reset_restir", "rtx_read_restir",
               "rtx_comm_unique_id", "rtx_comm_init", "rtx_reduce_accum", "rtx_read_reduced_accum", "rtx_comm_destroy"]
HOST_SYMBOLS = ["rdx_instance_properties", "rdx_collect_emissive_triangles", "rdx_camera_params", "rdx_generate_ess_lut",
                "rdx_obj_load", "rdx_obj_free", "rdx_obj_error", "rdx_obj_counts", "rdx_obj_copy"]

_lib = None
_host = None


class RtxError(RuntimeError):
    pass


def load_library():
    """Loads librtx_b200.so.  Fails loudly when it has not been built (python royaltracer-dx_b200/build.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RtxError("CUDA extension missing: %s (run `python royaltracer-dx_b200/build.py`); there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.rtx_last_error.restype = C.c_char_p
    vp, u32 = C.c_void_p, C.c_uint32
    lib.rtx_create.argtypes = [C.POINTER(RtxConfig), C.POINTER(vp)]
    lib.rtx_destroy.argtypes = [vp]
    lib.rtx_destroy.restype = None
    lib.rtx_upload_model.argtypes = [vp, vp, u32, vp, u32, u32, C.POINTER(u32)]
    lib.rtx_update_model.argtypes = [vp, u32, vp, u32, u32]
    lib.rtx_update_model_device.argtypes = [vp, u32, vp, u32, u32]
    lib.rtx_blas_info_get.argtypes = [vp, u32, C.POINTER(RtxBlasInfo)]
    lib.rtx_set_material_ids.argtypes = [vp, vp, u32]
    lib.rtx_set_materials.argtypes = [vp, vp, u32]
    lib.rtx_set_instances.argtypes = [vp, vp, vp, u32]
    lib.rtx_set_emissive_triangles.argtypes = [vp, vp, u32]
    lib.rtx_set_camera.argtypes = [vp, vp]
    lib.rtx_render_pass.argtypes = [vp, u32, u32]
    lib.rtx_reset_accum.argtypes = [vp]
    lib.rtx_synchronize.argtypes = [vp]
    lib.rtx_read_accum.argtypes = [vp, vp]
    lib.rtx_read_output.argtypes = [vp, vp]
    lib.rtx_read_output_async.argtypes = [vp, vp]
    lib.rtx_wait_output.argtypes = [vp]
    lib.rtx_set_resolve_source.argtypes = [vp, vp]
    lib.rtx_accum_device_ptr.argtypes = [vp, C.POINTER(vp)]
    lib.rtx_trace.argtypes = [vp, vp, u32, vp, C.c_int]
    lib.rtx_trace_device.argtypes = [vp, vp, u32, vp, C.c_int]
    lib.rtx_trace_stats.argtypes = [vp, vp, u32, vp, C.c_int]
    lib.rtx_get_counters.argtypes = [vp, C.POINTER(RtxCounters)]
    lib.rtx_reset_counters.argtypes = [vp]
    lib.rtx_last_pass_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.rtx_last_pass_stage_ms.argtypes = [vp, vp, u32, C.POINTER(C.c_float)]
    lib.rtx_debug_pixel.argtypes = [vp, u32, u32, vp]
    lib.rtx_set_option.argtypes = [vp, u32, u32]
    lib.rtx_selftest_dmath.argtypes = [vp, vp, u32]
    lib.rtx_render_frame.argtypes = [vp, u32]
    lib.rtx_reset_restir.argtypes = [vp]
    lib.rtx_read_restir.argtypes = [vp, vp]
    lib.rtx_comm_unique_id.argtypes = [vp]
    lib.rtx_comm_init.argtypes = [vp, vp, C.c_int, C.c_int]
    lib.rtx_reduce_accum.argtypes = [vp]
    lib.rtx_read_reduced_accum.argtypes = [vp, vp]
    lib.rtx_comm_destroy.argtypes = [vp]
    _lib = lib
    return lib


def load_host_library():
    global _host
    if _host is not None:
        return _host
    if not os.path.exists(HOST_LIB_PATH):
        raise RtxError("host library missing: %s (run `python royaltracer-dx_b200/build.py`)" % HOST_LIB_PATH)
    h = C.CDLL(HOST_LIB_PATH)
    vp, u32 = C.c_void_p, C.c_uint32
    h.rdx_instance_properties.argtypes = [vp, vp, u32, vp, vp]
    h.rdx_instance_properties.restype = None
    h.rdx_collect_emissive_triangles.argtypes = [u32, vp, u32, vp, vp, vp, vp, vp, vp, vp, u32]
    h.rdx_collect_emissive_triangles.restype = u32
    h.rdx_camera_params.argtypes = [vp, vp, vp, C.c_float, C.c_float, C.c_float, C.c_float, vp]
    h.rdx_camera_params.restype = None
    h.rdx_generate_ess_lut.argtypes = [vp, u32]
    h.rdx_obj_load.argtypes = [C.c_char_p, u32, C.c_char_p, u32]
    h.rdx_obj_load.restype = vp
    h.rdx_obj_free.argtypes = [vp]
    h.rdx_obj_error.argtypes = [vp]
    h.rdx_obj_error.restype = C.c_char_p
    h.rdx_obj_counts.argtypes = [vp, vp]
    h.rdx_obj_copy.argtypes = [vp, vp, vp, vp, vp]
    h.rdx_generate_ess_lut.restype = None
    _host = h
    return h


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


# ---------------------------------------------------------------------------------------------- host mirror (reference Renderer slices)
def xmmatrix_from_colvec(m4):
    """column-vector-convention 4x4 (translation in the last column) -> XMMATRIX memory (row-major, row-vector)."""
    return np.ascontiguousarray(np.asarray(m4, dtype=np.float32).T).reshape(16)


def instance_properties(xm_list, model_ids):
    """rdn/Renderer.cpp:2091-2121 + TopLevelASGenerator.cpp:181-199 -> (props[n], descs[n])."""
    h = load_host_library()
    n = len(xm_list)
    xm = np.ascontiguousarray(np.asarray(xm_list, dtype=np.float32).reshape(n, 16))
    mids = np.ascontiguousarray(np.asarray(model_ids, dtype=np.uint32))
    props = np.zeros(n, dtype=props_dt)
    descs = np.zeros(n, dtype=desc_dt)
    h.rdx_instance_properties(_ptr(xm), _ptr(mids), n, _ptr(props), _ptr(descs))
    return props, descs


def collect_emissive_triangles(scene):
    """rdn/Renderer.cpp:2123-2233,2241-2243 (F21)."""
    h = load_host_library()
    nm = len(scene.models)
    vp = (C.c_void_p * nm)(*[m["vertices"].ctypes.data for m in scene.models])
    ip = (C.c_void_p * nm)(*[m["indices"].ctypes.data for m in scene.models])
    ni = np.array([m["indices"].size for m in scene.models], dtype=np.uint32)
    off = np.array([m["material_id_offset"] for m in scene.models], dtype=np.uint32)
    inst_model = np.array([i[0] for i in scene.instances], dtype=np.uint32)
    args = (len(scene.instances), _ptr(inst_model), nm, C.cast(vp, C.c_void_p), C.cast(ip, C.c_void_p), _ptr(ni), _ptr(off),
            _ptr(scene.material_ids), _ptr(scene.materials))
    n = h.rdx_collect_emissive_triangles(*args, None, 0)
    out = np.zeros(max(n, 1), dtype=light_dt)
    h.rdx_collect_emissive_triangles(*args, _ptr(out), n)
    return out[:n]


def camera_params(eye, center, up, aspect, fovy_deg=60.0, zn=0.1, zf=1000.0):
    """rdn/Renderer.cpp:1722-1768 (S8)."""
    h = load_host_library()
    cam = np.zeros(1, dtype=camera_dt)
    e, c, u = (np.ascontiguousarray(np.asarray(v, dtype=np.float32)) for v in (eye, center, up))
    h.rdx_camera_params(_ptr(e), _ptr(c), _ptr(u), fovy_deg, aspect, zn, zf, _ptr(cam))
    return cam


def load_obj(path, material_offset=0, mtl_dir=None, lut_seed=12345):
    """src/Util/ObjLoader.h:393-495 (ObjLoader::loadObjFile): OBJ/MTL -> vertices (de-duplicated by position), indices, one global
    material id per face-vertex, and this model's material block [default, mtl...]."""
    h = load_host_library()
    hd = C.c_void_p(h.rdx_obj_load(os.fsencode(path), material_offset, os.fsencode(mtl_dir) if mtl_dir else None, lut_seed))
    try:
        err = h.rdx_obj_error(hd)
        if err:
            raise RtxError("load_obj: " + err.decode())
        cnt = np.zeros(4, dtype=np.uint32)
        h.rdx_obj_counts(hd, _ptr(cnt))
        v = np.zeros(int(cnt[0]), dtype=vertex_dt); idx = np.zeros(int(cnt[1]), dtype=np.uint32)
        mids = np.zeros(int(cnt[2]), dtype=np.uint32); mats = np.zeros(int(cnt[3]), dtype=material_dt)
        h.rdx_obj_copy(hd, _ptr(v), _ptr(idx), _ptr(mids), _ptr(mats))
    finally:
        h.rdx_obj_free(hd)
    return {"vertices": v, "indices": idx, "material_ids": mids, "materials": mats}


def generate_ess_lut(materials, seed=12345):
    """src/Util/ObjLoader.h:351-387 with a fixed seed (F23); fills LUT of every material in place."""
    h = load_host_library()
    for i in range(len(materials)):
        one = materials[i:i + 1]
        h.rdx_generate_ess_lut(_ptr(one), seed + i)
    return materials


# ---------------------------------------------------------------------------------------------- the engine context
class Context:
    """Thin object wrapper over rtx_ctx.  Mirrors the reference's call sequence: upload (OnInit), set_* (OnUpdate),
    render_pass (OnRender)."""

    def __init__(self, width, height, bounces=3, nee_samples=4, nee_samples_di=4, flags=0, samples_per_pass=1, device=0, stream=None):
        self.lib = load_library()
        cfg = RtxConfig(C.sizeof(RtxConfig), device, width, height, bounces, nee_samples, nee_samples_di, flags, samples_per_pass, stream)
        self.handle = C.c_void_p()
        self._check(self.lib.rtx_create(C.byref(cfg), C.byref(self.handle)))
        self.width, self.height = width, height

    def _check(self, st):
        if st != 0:
            raise RtxError("rtx error %d: %s" % (st, self.lib.rtx_last_error().decode()))

    def close(self):
        if self.handle:
            self.lib.rtx_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload_model(self, vertices, indices, material_id_offset):
        v = np.ascontiguousarray(vertices, dtype=vertex_dt)
        i = np.ascontiguousarray(indices, dtype=np.uint32)
        mid = C.c_uint32()
        self._check(self.lib.rtx_upload_model(self.handle, _ptr(v), v.size, _ptr(i), i.size, material_id_offset, C.byref(mid)))
        return mid.value

    def update_model(self, model_id, vertices, mode=UPDATE_REFIT):
        """New positions / normals for an uploaded model (same vertex count and indices): refit (default) or rebuild its BVH; instance
        boxes and the TLAS follow.  The accumulation is not reset and the light list is not touched."""
        v = np.ascontiguousarray(vertices, dtype=vertex_dt)
        self._check(self.lib.rtx_update_model(self.handle, model_id, _ptr(v), v.size, mode))

    def update_model_device(self, model_id, buf, n_vertices, mode=UPDATE_REFIT):
        """The same from device memory of n_vertices * 28 bytes: an int device pointer or anything with data_ptr() (a torch tensor),
        copied on the context stream; with UPDATE_REFIT the call neither waits nor allocates.  Work that wrote the buffer on another
        stream must be complete, or ordered before the context stream, when the call is made."""
        ptr = buf.data_ptr() if hasattr(buf, "data_ptr") else buf
        self._check(self.lib.rtx_update_model_device(self.handle, model_id, C.c_void_p(int(ptr) if ptr else None), n_vertices, mode))

    def blas_info(self, model_id):
        info = RtxBlasInfo()
        self._check(self.lib.rtx_blas_info_get(self.handle, model_id, C.byref(info)))
        return {"n_nodes": info.n_nodes, "n_tris": info.n_tris, "bytes": info.bytes, "build_ms": info.build_ms}

    def set_material_ids(self, ids):
        a = np.ascontiguousarray(ids, dtype=np.uint32)
        self._check(self.lib.rtx_set_material_ids(self.handle, _ptr(a), a.size))

    def set_materials(self, mats):
        a = np.ascontiguousarray(mats, dtype=material_dt)
        self._check(self.lib.rtx_set_materials(self.handle, _ptr(a), a.size))

    def set_instances(self, descs, props):
        d = np.ascontiguousarray(descs, dtype=desc_dt)
        p = np.ascontiguousarray(props, dtype=props_dt)
        assert d.size == p.size
        self._check(self.lib.rtx_set_instances(self.handle, _ptr(d), _ptr(p), d.size))

    def set_emissive_triangles(self, lights):
        a = np.ascontiguousarray(lights, dtype=light_dt)
        self._check(self.lib.rtx_set_emissive_triangles(self.handle, _ptr(a), a.size))

    def set_camera(self, cam):
        a = np.ascontiguousarray(cam, dtype=camera_dt)
        self._check(self.lib.rtx_set_camera(self.handle, _ptr(a)))

    def upload_scene(self, scene):
        """OnInit + OnUpdate for a scenes.SceneDesc: models, materials, instances, light list, camera."""
        ids = [self.upload_model(m["vertices"], m["indices"], m["material_id_offset"]) for m in scene.models]
        self.set_material_ids(scene.material_ids)
        self.set_materials(scene.materials)
        props, descs = instance_properties([i[1] for i in scene.instances], [ids[i[0]] for i in scene.instances])
        self.set_instances(descs, props)
        lights = collect_emissive_triangles(scene)
        self.set_emissive_triangles(lights)
        cam = camera_params(scene.eye, scene.center, scene.up, self.width / self.height)
        self.set_camera(cam)
        return {"props": props, "descs": descs, "lights": lights, "camera": cam, "model_ids": ids}

    def render_pass(self, first_sample, n_samples):
        self._check(self.lib.rtx_render_pass(self.handle, first_sample, n_samples))

    def render_frame(self, frame_index):
        """The reference's 3-pass frame (RayGen, RayGen2, RayGen3); the context needs FLAG_RESTIR."""
        self._check(self.lib.rtx_render_frame(self.handle, frame_index))

    def reset_restir(self):
        self._check(self.lib.rtx_reset_restir(self.handle))

    def read_restir(self):
        out = np.zeros((self.height, self.width, 40), dtype=np.float32)
        self._check(self.lib.rtx_read_restir(self.handle, _ptr(out)))
        return out

    def reset_accum(self):
        self._check(self.lib.rtx_reset_accum(self.handle))

    def synchronize(self):
        self._check(self.lib.rtx_synchronize(self.handle))

    def read_accum(self):
        out = np.zeros((self.height, self.width, 4), dtype=np.float32)
        self._check(self.lib.rtx_read_accum(self.handle, _ptr(out)))
        return out

    def read_output(self, out=None):
        """gOutput slice 0 as RGBA8; `out` may be a caller-owned (e.g. pinned) uint8 buffer of height*width*4 bytes."""
        if out is None:
            out = np.zeros((self.height, self.width, 4), dtype=np.uint8)
        assert out.dtype == np.uint8 and out.size == self.height * self.width * 4 and out.flags["C_CONTIGUOUS"]
        self._check(self.lib.rtx_read_output(self.handle, _ptr(out)))
        return out

    def read_output_async(self, out):
        """Enqueue resolve + read-back into the caller-owned (pinned) uint8 buffer `out`; wait_output() completes it."""
        assert out.dtype == np.uint8 and out.size == self.height * self.width * 4 and out.flags["C_CONTIGUOUS"]
        self._check(self.lib.rtx_read_output_async(self.handle, _ptr(out)))

    def set_resolve_source(self, device_ptr):
        """Resolve (read_output*) from an external device accumulation buffer, e.g. the reduced multi-GPU sum; None = the context's own."""
        self._check(self.lib.rtx_set_resolve_source(self.handle, C.c_void_p(int(device_ptr) if device_ptr else None)))

    def wait_output(self):
        self._check(self.lib.rtx_wait_output(self.handle))

    def accum_device_ptr(self):
        p = C.c_void_p()
        self._check(self.lib.rtx_accum_device_ptr(self.handle, C.byref(p)))
        return p.value

    # multi-GPU: the per-pass NCCL reduce of gPermanentData lives behind the C ABI (rtx_comm_init / rtx_reduce_accum)
    @staticmethod
    def _nccl_of_the_process():
        """The engine binds NCCL with dlopen("libnccl.so.2") at the first comm call and a process holds ONE library of that soname: in a
        Python process torch must load its bundled (newer) NCCL first, or a later `import torch` finds the system's older one in its place."""
        try:
            import torch  # noqa: F401
        except ImportError:
            pass

    def comm_unique_id(self):
        """128 bytes of ncclGetUniqueId (call on one rank, hand to the others)."""
        self._nccl_of_the_process()
        buf = (C.c_ubyte * 128)()
        self._check(self.lib.rtx_comm_unique_id(C.cast(buf, C.c_void_p)))
        return bytes(buf)

    def comm_init(self, unique_id, rank, world):
        assert len(unique_id) == 128
        self._nccl_of_the_process()
        buf = (C.c_ubyte * 128).from_buffer_copy(unique_id)
        self._check(self.lib.rtx_comm_init(self.handle, C.cast(buf, C.c_void_p), rank, world))

    def reduce_accum(self):
        self._check(self.lib.rtx_reduce_accum(self.handle))

    def read_reduced_accum(self):
        out = np.zeros((self.height, self.width, 4), dtype=np.float32)
        self._check(self.lib.rtx_read_reduced_accum(self.handle, _ptr(out)))
        return out

    def trace(self, rays, any_hit=False):
        r = np.ascontiguousarray(rays, dtype=ray_dt)
        out = np.zeros(r.size, dtype=hit_dt)
        self._check(self.lib.rtx_trace(self.handle, _ptr(r), r.size, _ptr(out), 1 if any_hit else 0))
        return out

    def trace_device(self, d_rays_ptr, n, d_hits_ptr, any_hit=False, stats=False):
        fn = self.lib.rtx_trace_stats if stats else self.lib.rtx_trace_device
        self._check(fn(self.handle, d_rays_ptr, n, d_hits_ptr, 1 if any_hit else 0))

    def counters(self):
        c = RtxCounters()
        self._check(self.lib.rtx_get_counters(self.handle, C.byref(c)))
        return {k: getattr(c, k) for k, _ in RtxCounters._fields_}

    def reset_counters(self):
        self._check(self.lib.rtx_reset_counters(self.handle))

    def last_pass_ms(self):
        a, b = C.c_float(), C.c_float()
        self._check(self.lib.rtx_last_pass_ms(self.handle, C.byref(a), C.byref(b)))
        return a.value, b.value

    def last_pass_stage_ms(self):
        """{stage name: ms} of the last pass (needs OPT_STAGE_TIMING) and the pass total."""
        k = np.zeros(len(STAGE_NAMES), dtype=np.float32)
        t = C.c_float()
        self._check(self.lib.rtx_last_pass_stage_ms(self.handle, _ptr(k), k.size, C.byref(t)))
        return {n: float(v) for n, v in zip(STAGE_NAMES, k)}, t.value

    def set_option(self, option, value):
        self._check(self.lib.rtx_set_option(self.handle, option, int(value)))

    def selftest_dmath(self):
        out = np.zeros(8, dtype=np.uint64)
        self._check(self.lib.rtx_selftest_dmath(self.handle, _ptr(out), 8))
        return {"rsqrt": int(out[0]), "div3": int(out[1])}

    def selftest_dmath_fast_paths(self):
        """Mismatch counts of the unguarded fast paths (csrc/dmath.cuh): a wrong result without the range flag, or a wrong flag."""
        out = np.zeros(8, dtype=np.uint64)
        self._check(self.lib.rtx_selftest_dmath(self.handle, _ptr(out), 8))
        return {k: int(out[i]) for i, k in enumerate(("sqrt", "rcp", "rsqrt", "div", "div_const"), start=2)}

    def debug_pixel(self, x, y):
        out = np.zeros(64, dtype=np.float32)
        self._check(self.lib.rtx_debug_pixel(self.handle, x, y, _ptr(out)))
        return out
