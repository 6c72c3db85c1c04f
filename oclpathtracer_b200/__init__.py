"""oclpathtracer_b200 -- ctypes view of libptb200.so (include/ptb200.h).

The product is the C-ABI library (hand-written sm_100a CUDA behind plain-C entry
points); this module only binds it for the parity tests and bench.py.  It never
touches the test oracle and has no CPU fallback: a missing library or a failing call
raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libptb200.so")

MODE_PRIMARY, MODE_AO, MODE_DIRECT, MODE_PATH = 0, 1, 2, 3
ACCUM_REFERENCE, ACCUM_LINEAR = 0, 1
OUTPUT_FLOAT4, OUTPUT_RGB8 = 0, 1
INTEGRATOR_AUTO, INTEGRATOR_MEGAKERNEL, INTEGRATOR_WAVEFRONT = 0, 1, 2
ACCEL_BVH, ACCEL_BRUTE = 0, 1
BUILDER_LBVH, BUILDER_SAH = 0, 1  # ptb_bvh_params.builder: the tree Device.scene(..., gpu_build=True) and scene_from_device build

TRIANGLE_DTYPE = np.dtype(
    [("p1", "<f4", 4), ("p2", "<f4", 4), ("p3", "<f4", 4), ("id", "<i4"), ("padding", "u1", 12)]
)
MATERIAL_DTYPE = np.dtype(
    [("albedo", "<f4", 4), ("emissive", "<f4", 4), ("roughness", "<f4"), ("type", "<i4"), ("padding", "u1", 24)]
)
NODE_DTYPE = np.dtype(  # binary node, 64 bytes (ptb_bvh_node)
    [
        ("c0", "<f4", 3), ("child0", "<i4"), ("e0", "<f4", 3), ("child1", "<i4"),
        ("c1", "<f4", 3), ("pad0", "<i4"), ("e1", "<f4", 3), ("pad1", "<i4"),
    ]
)
NODE4_DTYPE = np.dtype(  # 4-wide node, 128 bytes (ptb_bvh_node4)
    [
        ("c0", "<f4", 3), ("child0", "<i4"), ("e0", "<f4", 3), ("child1", "<i4"),
        ("c1", "<f4", 3), ("child2", "<i4"), ("e1", "<f4", 3), ("child3", "<i4"),
        ("c2", "<f4", 3), ("pad0", "<i4"), ("e2", "<f4", 3), ("pad1", "<i4"),
        ("c3", "<f4", 3), ("pad2", "<i4"), ("e3", "<f4", 3), ("pad3", "<i4"),
    ]
)
LEAFBOX_DTYPE = np.dtype(  # FLAT form, 32 bytes (ptb_bvh_leafbox)
    [("c", "<f4", 3), ("mask_lo", "<u4"), ("e", "<f4", 3), ("mask_hi", "<u4")]
)
STATS_DTYPE = np.dtype(
    [
        ("tri", "<i4"), ("quad", "<i4"), ("t_bits", "<u4"), ("visits_primary", "<u4"),
        ("visits_secondary", "<u4"), ("count", "<u4"), ("id_hash", "<u4"), ("tri_tests", "<u4"),
    ]
)
RAY_DTYPE = np.dtype(  # ptb_ray, 32 bytes (one 256-bit load); arrays must be 32-byte aligned
    [("o", "<f4", 3), ("tmax", "<f4"), ("d", "<f4", 3), ("reserved", "<i4")]
)
HIT_DTYPE = np.dtype([("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("tri", "<i4")])  # ptb_hit, 16 bytes; tri = -1: miss
SAMPLE_RAY_DTYPE = np.dtype(  # ptb_sample_ray, 32 bytes (one 256-bit load); seed = the sample's RNG state after the camera's draws
    [("o", "<f4", 3), ("seed", "<u4"), ("d", "<f4", 3), ("reserved", "<i4")]
)
QUERY_CLOSEST, QUERY_ANY = 0, 1


class RenderParams(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32),
        ("first_frame", C.c_int32), ("n_frames", C.c_int32),
        ("mode", C.c_int32), ("accum", C.c_int32), ("integrator", C.c_int32), ("accel", C.c_int32),
        ("max_depth", C.c_int32), ("ao_samples", C.c_int32), ("ao_max_dist", C.c_float),
        ("light_quad", C.c_int32),
        ("light_p1", C.c_float * 3), ("light_ea", C.c_float * 3), ("light_eb", C.c_float * 3),
        ("shard_index", C.c_int32), ("shard_count", C.c_int32), ("shard_block", C.c_int32),
        ("collect_stats", C.c_int32), ("frames_per_batch", C.c_int32), ("output", C.c_int32),
        ("reserved", C.c_int32 * 6),
    ]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rays_closest", "rays_any", "nodes", "tri_tests", "samples")] + [
        ("reserved", C.c_uint64 * 3)
    ]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n in ("rays_closest", "rays_any", "nodes", "tri_tests", "samples")}


class BvhParams(C.Structure):
    _fields_ = [("max_leaf", C.c_int32), ("pad_rel", C.c_float), ("n_bins", C.c_int32), ("smem_nodes", C.c_int32),
                ("traverse_cost", C.c_float), ("force_width", C.c_int32), ("builder", C.c_int32), ("reserved", C.c_int32 * 1)]


class Int4(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("z", C.c_int32), ("w", C.c_int32)]


class PtbError(RuntimeError):
    pass


_lib = None

# every symbol include/ptb200.h declares
EXPORTS = [
    "ptb_last_error", "ptb_version", "ptb_device_count", "ptb_device_create", "ptb_device_create_on_stream",
    "ptb_device_destroy", "ptb_device_sync", "ptb_device_name", "ptb_device_sm_count", "ptb_device_memory", "ptb_device_stream",
    "ptb_buffer_create", "ptb_buffer_wrap", "ptb_buffer_destroy", "ptb_buffer_write", "ptb_buffer_read",
    "ptb_buffer_map", "ptb_buffer_unmap", "ptb_buffer_clear", "ptb_buffer_device_ptr", "ptb_buffer_mark_dirty", "ptb_buffer_size",
    "ptb_kernel_get", "ptb_kernel_set_int", "ptb_launch1d", "ptb_launch_serialize", "ptb_launch_deserialize", "ptb_load_model", "ptb_tessellate",
    "ptb_light_from_quad", "ptb_free", "ptb_to_rgb8", "ptb_write_ppm", "ptb_bvh_params_default",
    "ptb_bvh_build_host", "ptb_scene_create", "ptb_scene_create_gpu", "ptb_scene_create_from_device", "ptb_scene_destroy", "ptb_scene_info", "ptb_scene_bvh_width", "ptb_scene_mode_width", "ptb_scene_copy_bvh", "ptb_scene_copy_bvh_quantized",
    "ptb_render_params_default", "ptb_render_local_pixels", "ptb_render", "ptb_render_host",
    "ptb_buffer_ipc_export", "ptb_buffer_ipc_import", "ptb_render_gather",
    "ptb_render_host_async", "ptb_job_wait", "ptb_host_alloc", "ptb_host_free", "ptb_trace", "ptb_scene_intersect", "ptb_scene_shade",
    "ptb_device_add_helper", "ptb_device_helper_count", "ptb_render_multi", "ptb_device_profile", "ptb_device_counters", "ptb_buffer_to_rgb8", "ptb_device_profile_read", "ptb_device_set_tuning", "ptb_test_sincos", "ptb_test_pow", "ptb_test_ieee", "ptb_test_rng", "ptb_test_camera",
]


def lib():
    """Load libptb200.so; fail loudly if the CUDA extension was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PtbError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(make -C oclpathtracer_b200/csrc).  There is no CPU fallback."
            )
        L = C.CDLL(LIB_PATH)
        L.ptb_last_error.restype = C.c_char_p
        L.ptb_buffer_device_ptr.restype = C.c_void_p
        L.ptb_buffer_size.restype = C.c_size_t
        L.ptb_device_stream.restype = C.c_void_p
        L.ptb_free.argtypes = [C.c_void_p]
        L.ptb_buffer_create.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        L.ptb_buffer_wrap.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.ptb_buffer_write.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
        L.ptb_buffer_read.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
        L.ptb_buffer_map.argtypes = [C.c_void_p, C.c_void_p]
        L.ptb_buffer_unmap.argtypes = [C.c_void_p, C.c_void_p]
        L.ptb_buffer_destroy.argtypes = [C.c_void_p]
        L.ptb_buffer_clear.argtypes = [C.c_void_p]
        L.ptb_buffer_device_ptr.argtypes = [C.c_void_p]
        L.ptb_buffer_mark_dirty.argtypes = [C.c_void_p]
        L.ptb_buffer_size.argtypes = [C.c_void_p]
        L.ptb_device_create.argtypes = [C.c_int, C.c_void_p]
        L.ptb_device_create_on_stream.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        for name in ("ptb_device_destroy", "ptb_device_sync", "ptb_scene_destroy"):
            getattr(L, name).argtypes = [C.c_void_p]
        L.ptb_device_name.argtypes = [C.c_void_p, C.c_char_p]
        L.ptb_device_sm_count.argtypes = [C.c_void_p, C.c_void_p]
        L.ptb_device_stream.argtypes = [C.c_void_p]
        L.ptb_device_memory.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.ptb_bvh_build_host.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 6
        L.ptb_scene_bvh_width.argtypes = [C.c_void_p]
        L.ptb_scene_mode_width.argtypes = [C.c_void_p, C.c_int]
        L.ptb_scene_copy_bvh_quantized.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ptb_device_counters.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.ptb_device_add_helper.argtypes = [C.c_void_p, C.c_void_p]
        L.ptb_device_helper_count.argtypes = [C.c_void_p]
        L.ptb_render_multi.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ptb_buffer_to_rgb8.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.ptb_scene_create.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.ptb_scene_create_gpu.argtypes = L.ptb_scene_create.argtypes
        L.ptb_scene_create_from_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.ptb_scene_info.argtypes = [C.c_void_p] + [C.c_void_p] * 4
        L.ptb_scene_copy_bvh.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.ptb_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ptb_render_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]
        L.ptb_render_host_async.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
        L.ptb_job_wait.argtypes = [C.c_void_p]
        L.ptb_host_alloc.argtypes = [C.c_size_t, C.c_void_p]
        L.ptb_host_free.argtypes = [C.c_void_p]
        L.ptb_kernel_get.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_void_p]
        L.ptb_kernel_set_int.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.ptb_launch1d.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int]
        L.ptb_launch_serialize.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int]
        L.ptb_launch_deserialize.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int] + [C.c_void_p] * 5
        L.ptb_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 9
        L.ptb_scene_intersect.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p]
        L.ptb_scene_shade.argtypes = [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 3
        L.ptb_device_profile.argtypes = [C.c_void_p, C.c_int]
        L.ptb_device_profile_read.argtypes = [C.c_void_p] * 5
        L.ptb_device_set_tuning.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.ptb_test_sincos.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.ptb_test_pow.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p]
        L.ptb_test_rng.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
        L.ptb_test_camera.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]
        L.ptb_load_model.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ptb_tessellate.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.ptb_light_from_quad.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ptb_to_rgb8.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.ptb_write_ppm.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int]
        L.ptb_render_local_pixels.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise PtbError(f"ptb error {rc}: {lib().ptb_last_error().decode()}")


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


# ---- host-side helpers (no GPU needed) -------------------------------------------------

def load_model(path):
    """RaytraceTest.cpp:87-198 loadModel -> (triangles, materials) structured arrays."""
    L = lib()
    tp, mp = C.c_void_p(), C.c_void_p()
    nt, nm = C.c_int(), C.c_int()
    _check(L.ptb_load_model(path.encode(), C.byref(tp), C.byref(nt), C.byref(mp), C.byref(nm)))
    try:
        tris = np.frombuffer(C.string_at(tp, nt.value * 64), TRIANGLE_DTYPE).copy()
        mats = np.frombuffer(C.string_at(mp, nm.value * 64), MATERIAL_DTYPE).copy()
    finally:
        L.ptb_free(tp)
        L.ptb_free(mp)
    return tris, mats


def tessellate(tris, k):
    L = lib()
    out, n = C.c_void_p(), C.c_int()
    tris = np.ascontiguousarray(tris)
    _check(L.ptb_tessellate(_p(tris), len(tris), k, C.byref(out), C.byref(n)))
    try:
        res = np.frombuffer(C.string_at(out, n.value * 64), TRIANGLE_DTYPE).copy()
    finally:
        L.ptb_free(out)
    return res


def light_from_quad(tris, quad):
    p1, ea, eb = (C.c_float * 3)(), (C.c_float * 3)(), (C.c_float * 3)()
    tris = np.ascontiguousarray(tris)
    _check(lib().ptb_light_from_quad(_p(tris), len(tris), quad, p1, ea, eb))
    return list(p1), list(ea), list(eb)


def to_rgb8(rgba):
    rgba = np.ascontiguousarray(rgba, np.float32).reshape(-1, 4)
    out = np.empty((rgba.shape[0], 3), np.uint8)
    _check(lib().ptb_to_rgb8(_p(rgba), rgba.shape[0], _p(out)))
    return out


def write_ppm(path, rgba, width, height):
    rgba = np.ascontiguousarray(rgba, np.float32)
    _check(lib().ptb_write_ppm(path.encode(), _p(rgba), width, height))


BVH_TRI_DTYPE = np.dtype(
    [("p1", "<f4", 3), ("index", "<i4"), ("e1", "<f4", 3), ("quad", "<i4"), ("e2", "<f4", 3), ("pad", "<i4")]
)


def build_bvh_host(tris, params=None, width=None):
    """Host-only BVH build (no GPU): dict(nodes, tri_order, ordered_tris, depth, smem_nodes, width).

    width 1 -> LEAFBOX_DTYPE records (the FLAT form of scenes with <= 32 leaves and <= 64 triangles), 4 -> NODE4_DTYPE
    records (what a shared-memory-resident scene uses), 2 -> NODE_DTYPE;
    None picks like ptb_scene_create does for the scenes of the tests (1 when <= 64 triangles, 4 when <= 256, else 2).
    """
    L = lib()
    tris = np.ascontiguousarray(tris)
    if width is None:
        width = 1 if len(tris) <= 64 else 4 if len(tris) <= 256 else 2
    nodes, order, otris = C.c_void_p(), C.c_void_p(), C.c_void_p()
    nn, depth, sn = C.c_int(), C.c_int(), C.c_int()
    _check(L.ptb_bvh_build_host(_p(tris), len(tris), C.byref(params) if params is not None else None, width,
                                C.byref(nodes), C.byref(nn), C.byref(order), C.byref(otris), C.byref(depth),
                                C.byref(sn)))
    dt = {1: LEAFBOX_DTYPE, 4: NODE4_DTYPE, 2: NODE_DTYPE}[width]
    try:
        res = {
            "width": width,
            "nodes": np.frombuffer(C.string_at(nodes, nn.value * dt.itemsize), dt).copy(),
            "tri_order": np.frombuffer(C.string_at(order, len(tris) * 4), np.int32).copy(),
            "ordered_tris": np.frombuffer(C.string_at(otris, len(tris) * 48), BVH_TRI_DTYPE).copy(),
            "depth": depth.value, "smem_nodes": sn.value,
        }
    finally:
        L.ptb_free(nodes)
        L.ptb_free(order)
        L.ptb_free(otris)
    return res


def default_params(**kw):
    p = RenderParams()
    lib().ptb_render_params_default(C.byref(p))
    for k, v in kw.items():
        if k in ("light_p1", "light_ea", "light_eb"):
            getattr(p, k)[:] = v
        else:
            if not hasattr(p, k):
                raise AttributeError(k)
            setattr(p, k, v)
    return p


def local_pixels(params):
    return lib().ptb_render_local_pixels(C.byref(params))


# ---- device objects ------------------------------------------------------------------------

class Device:
    """adl::DeviceUtils::allocate / deallocate (Adl/Adl.h:125-126) over ptb_device."""

    def __init__(self, index=0, stream=None):
        self._h = C.c_void_p()
        if stream is None:
            _check(lib().ptb_device_create(index, C.byref(self._h)))
        else:
            _check(lib().ptb_device_create_on_stream(index, C.c_void_p(stream), C.byref(self._h)))
        self._children = []

    @property
    def handle(self):
        return self._h

    def sync(self):
        _check(lib().ptb_device_sync(self._h))

    def name(self):
        b = C.create_string_buffer(128)
        _check(lib().ptb_device_name(self._h, b))
        return b.value.decode()

    def sm_count(self):
        n = C.c_int()
        _check(lib().ptb_device_sm_count(self._h, C.byref(n)))
        return n.value

    def stream(self):
        return lib().ptb_device_stream(self._h)

    def memory(self):
        """(free, total) bytes of device memory."""
        f, t = C.c_size_t(), C.c_size_t()
        _check(lib().ptb_device_memory(self._h, C.byref(f), C.byref(t)))
        return f.value, t.value

    def set_tuning(self, index, value):
        _check(lib().ptb_device_set_tuning(self._h, index, value))

    def profile(self, enable=True):
        _check(lib().ptb_device_profile(self._h, 1 if enable else 0))

    def profile_read(self):
        """Synchronises; totals since the previous read."""
        ti, tr, nb, nk = C.c_float(), C.c_float(), C.c_int(), C.c_uint64()
        _check(lib().ptb_device_profile_read(self._h, C.byref(ti), C.byref(tr), C.byref(nb), C.byref(nk)))
        return {"integrator_ms": ti.value, "resolve_ms": tr.value, "batches": nb.value, "kernel_launches": nk.value}

    def counters(self, cumulative=-1, read=True):
        """ptb_device_counters: switch the cumulative mode (1 | 0 | -1 = leave) and/or read + clear the totals."""
        ctr = Counters() if read else None
        _check(lib().ptb_device_counters(self._h, cumulative, C.byref(ctr) if ctr is not None else None))
        return ctr.as_dict() if ctr is not None else None

    def buffer(self, nbytes):
        return Buffer(self, nbytes)

    def wrap(self, device_ptr, nbytes):
        return Buffer(self, nbytes, device_ptr=device_ptr)

    def scene(self, tris, mats, bvh_params=None, gpu_build=False):
        return Scene(self, tris, mats, bvh_params, gpu_build)

    def scene_from_device(self, tris, mats, bvh_params=None):
        """ptb_scene_create_from_device: the scene Device.scene(..., gpu_build=True) builds, from records already on this device.

        tris is a Buffer of TRIANGLE_DTYPE records or a contiguous CUDA tensor of shape (n, 16) with 4-byte elements (float32
        records; the id is the int32 bits of column 12); mats is a Buffer, an (n_mats, 16) CUDA tensor or a numpy MATERIAL_DTYPE
        array (uploaded through a temporary Buffer).  With tensors the Device must have been created on torch's current stream,
        so that the build reads the records after the work that wrote them.  Synchronises; the scene keeps its own copies."""
        return Scene(self, tris, mats, bvh_params, from_device=True)

    def close(self):
        if self._h:
            for c in list(self._children):
                c.close()
            rc = lib().ptb_device_destroy(self._h)
            self._h = C.c_void_p()
            _check(rc)

    # ---- the hot path -------------------------------------------------------------------
    def render(self, scene, params, frame, stats=None, want_counters=False):
        ctr = Counters() if want_counters else None
        _check(lib().ptb_render(self._h, scene._h, C.byref(params), frame._h, stats._h if stats else None,
                                C.byref(ctr) if ctr is not None else None))
        return ctr.as_dict() if ctr is not None else None

    def ipc_import(self, handle, nbytes):
        return Buffer(self, nbytes, ipc_handle=handle)

    def render_gather(self, scene, params, full_frame, peer_frames=(), want_counters=False):
        """Render this rank's shard and store every pixel at its global position in full_frame and the peers' images."""
        ctr = Counters() if want_counters else None
        arr = (C.c_void_p * max(1, len(peer_frames)))(*[b._h for b in peer_frames])
        _check(lib().ptb_render_gather(self._h, scene._h, C.byref(params), full_frame._h, arr, len(peer_frames),
                                       C.byref(ctr) if ctr is not None else None))
        return ctr.as_dict() if ctr is not None else None

    def render_host(self, tris, mats, params, out=None, want_stats=False, want_counters=True):
        n = local_pixels(params)
        if out is None:
            out = np.zeros((n, 3), np.uint8) if params.output == OUTPUT_RGB8 else np.zeros((n, 4), np.float32)
        stats = np.zeros(n, STATS_DTYPE) if want_stats else None
        ctr = Counters() if want_counters else None
        tris = np.ascontiguousarray(tris)
        mats = np.ascontiguousarray(mats)
        _check(lib().ptb_render_host(self._h, _p(tris), len(tris), _p(mats), len(mats), C.byref(params), _p(out),
                                     _p(stats), C.byref(ctr) if ctr is not None else None))
        return out, stats, (ctr.as_dict() if ctr is not None else None)

    def add_helper(self, helper):
        """ptb_device_add_helper: `helper` (another Device) renders part of this device's work from now on"""
        _check(lib().ptb_device_add_helper(self._h, helper._h))

    def helper_count(self):
        return lib().ptb_device_helper_count(self._h)

    def render_multi(self, tris, mats, params, out=None, want_counters=True):
        """ptb_render_multi: ONE image sharded over this device and its helpers; host records in, host image out"""
        n = params.width * params.height
        if out is None:
            out = np.zeros((n, 3), np.uint8) if params.output == OUTPUT_RGB8 else np.zeros((n, 4), np.float32)
        ctr = Counters() if want_counters else None
        tris = np.ascontiguousarray(tris)
        mats = np.ascontiguousarray(mats)
        _check(lib().ptb_render_multi(self._h, _p(tris), len(tris), _p(mats), len(mats), C.byref(params), _p(out),
                                      C.byref(ctr) if ctr is not None else None))
        return out, (ctr.as_dict() if ctr is not None else None)

    def render_host_async(self, tris, mats, params, out, stats=None):
        """Returns a job handle; call job_wait(handle) before reading `out`.  At most two in flight."""
        job = C.c_void_p()
        _check(lib().ptb_render_host_async(self._h, _p(tris), len(tris), _p(mats), len(mats), C.byref(params), _p(out),
                                           _p(stats), C.byref(job)))
        return job

    def job_wait(self, job):
        _check(lib().ptb_job_wait(job))

    def kernel(self, file_name, func_name):
        k = C.c_void_p()
        _check(lib().ptb_kernel_get(self._h, file_name.encode(), func_name.encode(), C.byref(k)))
        return k

    def kernel_set_int(self, kernel, name, value):
        _check(lib().ptb_kernel_set_int(kernel, name.encode(), value))

    def launch1d(self, kernel, bufs, consts, n_threads, local_size=64):
        arr = (C.c_void_p * len(bufs))(*[b._h for b in bufs])
        _check(lib().ptb_launch1d(self._h, kernel, arr, len(bufs), C.byref(consts), C.sizeof(consts), n_threads,
                                  local_size))

    def launch_serialize(self, path, bufs, consts, n_threads, local_size=64):
        arr = (C.c_void_p * len(bufs))(*[b._h for b in bufs])
        _check(lib().ptb_launch_serialize(self._h, path.encode(), arr, len(bufs), C.byref(consts), C.sizeof(consts),
                                          n_threads, local_size))

    def launch_deserialize(self, path, cap=8):
        """-> (buffers, const block bytes, n_threads, local_size); the buffers belong to the caller."""
        handles = (C.c_void_p * cap)()
        nb, cb, nt, ls = C.c_int(), C.c_size_t(), C.c_int(), C.c_int()
        consts = C.create_string_buffer(64)
        _check(lib().ptb_launch_deserialize(self._h, path.encode(), handles, cap, C.byref(nb), consts, C.byref(cb),
                                            C.byref(nt), C.byref(ls)))
        bufs = []
        for i in range(nb.value):
            b = Buffer.__new__(Buffer)
            b.dev, b._h = self, C.c_void_p(handles[i])
            b.nbytes = lib().ptb_buffer_size(b._h)
            self._children.append(b)
            bufs.append(b)
        return bufs, consts.raw[: cb.value], nt.value, ls.value

    def trace(self, scene, o, d, tmax, accel=ACCEL_BVH, any_hit=False):
        n = len(o)
        o = np.ascontiguousarray(o, np.float32)
        d = np.ascontiguousarray(d, np.float32)
        tmax = np.ascontiguousarray(np.broadcast_to(np.asarray(tmax, np.float32), (n,)))
        out = {
            "tri": np.empty(n, np.int32), "t": np.empty(n, np.float32), "u": np.empty(n, np.float32),
            "v": np.empty(n, np.float32), "visits": np.empty(n, np.uint32), "tests": np.empty(n, np.uint32),
        }
        _check(lib().ptb_trace(self._h, scene._h, accel, 1 if any_hit else 0, n, _p(o), _p(d), _p(tmax),
                               _p(out["tri"]), _p(out["t"]), _p(out["u"]), _p(out["v"]), _p(out["visits"]),
                               _p(out["tests"])))
        return out

    def intersect(self, scene, rays, hits=None, any_hit=False, stats=None, want_counters=False):
        """ptb_scene_intersect: closest- (or any-) hit queries on rays that live on this device.

        rays, hits and stats are each a Buffer or a CUDA torch tensor: rays = RAY_DTYPE records (a float32 tensor of shape
        (n, 8): o.xyz, tmax, d.xyz, unused), hits = HIT_DTYPE records (a float32 (n, 4) tensor: t, u, v and the triangle
        index as the bits of an int32, read it with `.view(torch.int32)`), stats = NULL or 2 x uint32 per ray (nodes fetched,
        triangle tests; an int32 (n, 2) tensor).  hits=None allocates them (a tensor for tensor rays, else a Buffer).
        Tensors are wrapped for the duration of the call; the Device must have been created on torch's current stream, so
        that the query runs after the work that produced the rays.  Asynchronous unless want_counters.
        Returns hits, or (hits, counters) when want_counters."""
        args = _CallArgs(self, "Device.intersect", rays, hits, stats)
        if isinstance(rays, Buffer):
            n = rays.nbytes // RAY_DTYPE.itemsize
        else:
            import torch

            if rays.dim() != 2 or rays.shape[1] != 8 or rays.dtype != torch.float32:
                raise PtbError(f"Device.intersect: a ray tensor is float32 of shape (n, 8), got {tuple(rays.shape)} {rays.dtype}")
            n = rays.shape[0]
        if hits is None:
            hits = self.buffer(max(1, n) * HIT_DTYPE.itemsize) if isinstance(rays, Buffer) else \
                torch.empty((n, 4), dtype=torch.float32, device=rays.device)
        ctr = Counters() if want_counters else None
        with args:
            if not (n == 0 and args.tensors):  # an empty tensor has no storage to wrap; the call would be a no-op anyway
                _check(lib().ptb_scene_intersect(self._h, scene._h, QUERY_ANY if any_hit else QUERY_CLOSEST, args.handle(rays), n,
                                                 args.handle(hits), args.handle(stats), C.byref(ctr) if ctr is not None else None))
        return (hits, ctr.as_dict()) if want_counters else hits

    def shade(self, scene, params, rays, radiance=None, stats=None, want_counters=False):
        """ptb_scene_shade: render-mode samples (params.mode, max_depth, ao_samples, ao_max_dist, light) along rays that live on
        this device; sample i is what render() computes for one pixel-frame after its camera step, with ray i and its seed.

        rays, radiance and stats are each a Buffer or a contiguous CUDA torch tensor: rays = SAMPLE_RAY_DTYPE records (an (n, 8)
        tensor of any 4-byte dtype: o.xyz, the seed as the bits of a uint32, d.xyz, unused), radiance = float4 per ray (a
        float32 (n, 4) tensor: xyz, w = 1), stats = NULL or STATS_DTYPE per ray (an int32 (n, 8) tensor).  radiance=None
        allocates it (a tensor for tensor rays, else a Buffer).  The Device must have been created on torch's current stream
        when tensors are used.  Asynchronous unless want_counters.  Returns radiance, or (radiance, counters) when
        want_counters."""
        args = _CallArgs(self, "Device.shade", rays, radiance, stats)
        if isinstance(rays, Buffer):
            n = rays.nbytes // SAMPLE_RAY_DTYPE.itemsize
        else:
            import torch

            if rays.dim() != 2 or rays.shape[1] != 8:
                raise PtbError(f"Device.shade: a ray tensor has shape (n, 8), got {tuple(rays.shape)}")
            n = rays.shape[0]
            for x, name, dt, cols in ((radiance, "radiance", torch.float32, 4), (stats, "stats", torch.int32, 8)):
                if x is not None and not isinstance(x, Buffer) and (x.dtype != dt or x.dim() != 2 or tuple(x.shape) != (n, cols)):
                    raise PtbError(f"Device.shade: {name} is a {dt} tensor of shape ({n}, {cols}), got {tuple(x.shape)} {x.dtype}")
        if radiance is None:
            radiance = self.buffer(max(1, n) * 16) if isinstance(rays, Buffer) else \
                torch.empty((n, 4), dtype=torch.float32, device=rays.device)
        ctr = Counters() if want_counters else None
        with args:
            if not (n == 0 and args.tensors):  # an empty tensor has no storage to wrap; the call would be a no-op anyway
                _check(lib().ptb_scene_shade(self._h, scene._h, C.byref(params), args.handle(rays), n, args.handle(radiance),
                                             args.handle(stats), C.byref(ctr) if ctr is not None else None))
        return (radiance, ctr.as_dict()) if want_counters else radiance

    def test_sincos(self, x):
        x = np.ascontiguousarray(x, np.float32)
        s, c = np.empty_like(x), np.empty_like(x)
        _check(lib().ptb_test_sincos(self._h, _p(x), x.size, _p(s), _p(c)))
        return s, c

    def test_pow(self, x, y):
        x = np.ascontiguousarray(x, np.float32)
        o = np.empty_like(x)
        _check(lib().ptb_test_pow(self._h, _p(x), x.size, C.c_float(y), _p(o)))
        return o

    def test_ieee(self, x):
        """-> dict(rcp, sqrt, safe_rcp, nx, ny, nz) of the kernels' branch-reduced IEEE helpers applied to x."""
        x = np.ascontiguousarray(x, np.float32)
        o = np.empty(6 * x.size, np.float32)
        _check(lib().ptb_test_ieee(self._h, _p(x), x.size, _p(o)))
        o = o.reshape(6, x.size)
        return dict(rcp=o[0], sqrt=o[1], safe_rcp=o[2], nx=o[3], ny=o[4], nz=o[5])

    def test_rng(self, gid, frame, n):
        st, va = np.empty(n, np.uint32), np.empty(n, np.float32)
        _check(lib().ptb_test_rng(self._h, gid, frame, n, _p(st), _p(va)))
        return st, va

    def test_camera(self, width, height, frame, gids):
        gids = np.ascontiguousarray(gids, np.int32)
        n = gids.size
        o, d, s = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32), np.empty(n, np.uint32)
        _check(lib().ptb_test_camera(self._h, width, height, frame, n, _p(gids), _p(o), _p(d), _p(s)))
        return o, d, s



class _CallArgs:
    """Buffers or CUDA torch tensors as ptb_buffer handles for one call of `what` (Device.intersect, Device.shade,
    Device.scene_from_device).

    Tensors must be contiguous CUDA tensors of 4-byte elements, and the Device must have been created on torch's current
    stream: on another stream the call would race with the work that wrote its inputs.  Used as a context manager, the
    wrappers made by handle() are released when the call returns."""

    def __init__(self, dev, what, *xs):
        self.dev = dev
        self.tensors = [x for x in xs if x is not None and not isinstance(x, Buffer)]
        self.wrapped = []
        if self.tensors:
            import torch

            cur = torch.cuda.current_stream(self.tensors[0].device).cuda_stream
            if cur != (dev.stream() or 0):  # the legacy default stream is handle 0 (ctypes returns None for it)
                raise PtbError(f"{what}: tensors need a Device created on torch.cuda.current_stream() "
                               "(Device(index, stream=torch.cuda.current_stream().cuda_stream)); "
                               "on another stream the query would race with the work that wrote the rays")
            for x in self.tensors:
                if not x.is_cuda or not x.is_contiguous() or x.element_size() != 4:
                    raise PtbError(f"{what}: tensors must be contiguous CUDA tensors of 4-byte elements")

    def handle(self, x):
        if x is None:
            return None
        if isinstance(x, Buffer):
            return x._h
        b = Buffer(self.dev, x.numel() * x.element_size(), device_ptr=x.data_ptr())
        self.wrapped.append(b)
        return b._h

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        for b in self.wrapped:
            b.close()
        self.wrapped = []
        return False


class Buffer:
    """adl::Buffer<T> (Adl/Adl.h:203-265) over ptb_buffer."""

    def __init__(self, dev, nbytes, device_ptr=None, ipc_handle=None):
        self.dev = dev
        self.nbytes = nbytes
        self._h = C.c_void_p()
        if ipc_handle is not None:  # another process's buffer, mapped as peer memory
            _check(lib().ptb_buffer_ipc_import(dev._h, C.c_char_p(bytes(ipc_handle)), nbytes, C.byref(self._h)))
        elif device_ptr is None:
            _check(lib().ptb_buffer_create(dev._h, nbytes, C.byref(self._h)))
        else:
            _check(lib().ptb_buffer_wrap(dev._h, C.c_void_p(device_ptr), nbytes, C.byref(self._h)))
        dev._children.append(self)

    def write(self, arr, offset=0):
        arr = np.ascontiguousarray(arr)
        _check(lib().ptb_buffer_write(self._h, _p(arr), arr.nbytes, offset))
        self.dev.sync()  # the numpy temporary must outlive the async copy

    def read(self, dtype=np.float32, count=None, offset=0):
        dtype = np.dtype(dtype)
        if count is None:
            count = (self.nbytes - offset) // dtype.itemsize
        out = np.empty(count, dtype)
        _check(lib().ptb_buffer_read(self._h, _p(out), out.nbytes, offset))
        self.dev.sync()
        return out

    def write_async(self, arr, offset=0):
        """H2D on the device's stream without waiting; `arr` (page-locked for a truly asynchronous copy) must stay alive
        and unchanged until the device is synchronised."""
        _check(lib().ptb_buffer_write(self._h, _p(arr), arr.nbytes, offset))

    def read_async(self, out, offset=0):
        """D2H on the device's stream into `out` (a numpy array, page-locked for a truly asynchronous copy); valid after
        the device is synchronised."""
        _check(lib().ptb_buffer_read(self._h, _p(out), out.nbytes, offset))

    def to_rgb8(self, n_pixels, rgb):
        """the reference's output transform on the device: this float4 frame -> 3 bytes per pixel in `rgb` (a Buffer)"""
        _check(lib().ptb_buffer_to_rgb8(self._h, n_pixels, rgb._h))

    def clear(self):
        _check(lib().ptb_buffer_clear(self._h))

    def ipc_export(self):
        """64-byte CUDA IPC handle; another process maps the buffer with Device.ipc_import(handle, nbytes)."""
        h = C.create_string_buffer(64)
        _check(lib().ptb_buffer_ipc_export(self._h, h))
        return h.raw

    def device_ptr(self):
        return lib().ptb_buffer_device_ptr(self._h)

    def mark_dirty(self):
        """the contents were changed behind the API's back (a kernel writing through device_ptr()): ptb_launch1d must re-read them"""
        _check(lib().ptb_buffer_mark_dirty(self._h))

    def close(self):
        if self._h:
            lib().ptb_buffer_destroy(self._h)
            self._h = C.c_void_p()
            if self in self.dev._children:
                self.dev._children.remove(self)


class Scene:
    """Resident scene: relaid triangles + BVH (BUILD-DEFINED; the reference is brute force)."""

    def __init__(self, dev, tris, mats, bvh_params=None, gpu_build=False, from_device=False):
        self.dev = dev
        self._h = C.c_void_p()
        bp = C.byref(bvh_params) if bvh_params is not None else None
        if from_device:
            self._create_from_device(tris, mats, bp)
        else:
            tris = np.ascontiguousarray(tris)
            mats = np.ascontiguousarray(mats)
            create = lib().ptb_scene_create_gpu if gpu_build else lib().ptb_scene_create
            _check(create(dev._h, _p(tris), len(tris), _p(mats), len(mats), bp, C.byref(self._h)))
        dev._children.append(self)

    def _create_from_device(self, tris, mats, bp):
        def count(x, name):
            if isinstance(x, Buffer):
                return x.nbytes // 64
            if not hasattr(x, "is_cuda") or x.dim() != 2 or x.shape[1] != 16:
                raise PtbError(f"Device.scene_from_device: {name} is a Buffer or a CUDA tensor of shape (n, 16), got "
                               f"{type(x).__name__} {tuple(getattr(x, 'shape', ()))}")
            return x.shape[0]

        staged = None
        if isinstance(mats, np.ndarray):
            if mats.dtype != MATERIAL_DTYPE:
                raise PtbError(f"Device.scene_from_device: a numpy mats array has MATERIAL_DTYPE, got {mats.dtype}")
            staged = Buffer(self.dev, mats.nbytes)
            if len(mats):
                staged.write(mats)
            mats = staged
        try:
            n_tris, n_mats = count(tris, "tris"), count(mats, "mats")
            with _CallArgs(self.dev, "Device.scene_from_device", tris, mats) as args:
                _check(lib().ptb_scene_create_from_device(self.dev._h, args.handle(tris), n_tris, args.handle(mats), n_mats, bp,
                                                          C.byref(self._h)))
        finally:
            if staged is not None:
                staged.close()

    def info(self):
        a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        _check(lib().ptb_scene_info(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return {"n_nodes": a.value, "n_tris": b.value, "depth": c.value, "smem_nodes": d.value,
                "width": lib().ptb_scene_bvh_width(self._h)}

    def mode_width(self, mode):
        """form (1 FLAT, 4, 2) a render of `mode` walks"""
        return lib().ptb_scene_mode_width(self._h, mode)

    def bvh(self):
        inf = self.info()
        nodes = np.zeros(inf["n_nodes"], {1: LEAFBOX_DTYPE, 4: NODE4_DTYPE, 2: NODE_DTYPE}[inf["width"]])
        order = np.zeros(inf["n_tris"], np.int32)
        _check(lib().ptb_scene_copy_bvh(self._h, _p(nodes), _p(order)))
        return nodes, order

    def bvh_quantized(self):
        """width-2 scenes: (uint32[n_nodes, 8] quantised records the kernels traverse, grid lo[3], grid step[3])"""
        q = np.zeros((self.info()["n_nodes"], 8), np.uint32)
        lo, step = (C.c_float * 3)(), (C.c_float * 3)()
        _check(lib().ptb_scene_copy_bvh_quantized(self._h, _p(q), lo, step))
        return q, [float(x) for x in lo], [float(x) for x in step]

    def close(self):
        if self._h:
            lib().ptb_scene_destroy(self._h)
            self._h = C.c_void_p()
            if self in self.dev._children:
                self.dev._children.remove(self)


class PinnedArray:
    """numpy view of page-locked host memory (ptb_host_alloc); free() when done."""

    def __init__(self, shape, dtype):
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        self._p = C.c_void_p()
        _check(lib().ptb_host_alloc(n, C.byref(self._p)))
        buf = (C.c_uint8 * n).from_address(self._p.value)
        self.array = np.frombuffer(buf, dtype=dtype).reshape(shape)

    def free(self):
        if self._p:
            self.array = None
            lib().ptb_host_free(self._p)
            self._p = C.c_void_p()


def bvh_params(**kw):
    p = BvhParams()
    lib().ptb_bvh_params_default(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p
