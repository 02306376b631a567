"""cedecrt — Python host side of libcedecrt.so (the C ABI in include/cedecrt.h).

Mirrors the reference's host layer for the ReSTIR DI path: `TypedBuffer` (common/typedbuffer.hpp), the
per-kernel launches of `Shader::launch` (common/shader.hpp:179-199) and the frame loop of
examples/10_restir_di/10_restir_di.cpp:229-380 (`RestirDI`).  It is ctypes over the C ABI only — there is
no Python or CPU implementation of any kernel here: if the library or a CUDA device is missing, creating a
`Runtime` raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# CRT_LIB_VARIANT=<tag>: load libcedecrt_<tag>.so (a tuning build, csrc/Makefile VARIANT=<tag>) instead
_VARIANT = os.environ.get("CRT_LIB_VARIANT", "")
LIB_PATH = os.path.join(_HERE, "..", "libcedecrt%s.so" % ("_" + _VARIANT if _VARIANT else ""))

# ---- reference struct layouts as numpy dtypes (host-side views of device buffers)
_f3 = (np.float32, (3,))
TRIANGLE = np.dtype([("vertices", np.float32, (3, 3)), ("color", *_f3), ("emissive", *_f3)])  # core.hpp:38-43
VISIBILITY = np.dtype([("uv", np.float32, (2,)), ("index", np.int32), ("_pad", np.int32)])  # core.hpp:167-172
RESERVOIR = np.dtype(  # reservoir.hpp:5-38
    [("origin_position", *_f3), ("origin_normal", *_f3), ("hit_position", *_f3), ("hit_normal", *_f3),
     ("radiance", *_f3), ("visibility", np.uint8), ("_pad", np.uint8, (3,)), ("w_sum", np.float32),
     ("ucw", np.float32), ("M", np.int32)]
)
FLOAT4 = np.dtype((np.float32, (4,)))
assert TRIANGLE.itemsize == 60 and VISIBILITY.itemsize == 16 and RESERVOIR.itemsize == 76

MATH_LIBDEVICE, MATH_EXACT, MATH_FAST, MATH_REFERENCE = 0, 1, 2, 3  # include/cedecrt.h: CRT_MATH_*
LIGHTS_UNIFORM, LIGHTS_POWER = 0, 1  # include/cedecrt.h: CRT_LIGHTS_*
# (log2 T, log2 S) of RestirDI(light_tiles=True): 512 tiles of 1024 records, 32 MB, measured in DESIGN.md section 16
LIGHT_TILES_DEFAULT = (9, 10)
REUSE_REFERENCE, REUSE_UNBIASED = 0, 1  # include/cedecrt.h: CRT_REUSE_*


class Float3(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]


class RayGenerator(C.Structure):
    """common/camera.hpp:5-36"""

    _fields_ = [("m_origin", Float3), ("m_right", Float3), ("m_up", Float3)]


class Options(C.Structure):
    """common/options.hpp:4-23 with the reference defaults"""

    _fields_ = [
        ("accumulate", C.c_uint8), ("_p0", C.c_uint8 * 3),
        ("max_depth", C.c_int32),
        ("sky_color", Float3),
        ("ris_sample_count", C.c_int32),
        ("rejection_heuristics_threshold", C.c_float),
        ("use_temporal_resampling", C.c_uint8),
        ("use_spatial_resampling", C.c_uint8), ("_p1", C.c_uint8 * 2),
        ("spatial_resampling_sample_count", C.c_int32),
        ("spatial_resampling_radius", C.c_float),
        ("spatial_resampling_passes", C.c_int32),
        ("use_shadowed_target_function", C.c_uint8),
        ("use_visibility_reuse", C.c_uint8), ("_p2", C.c_uint8 * 2),
    ]

    def __init__(self, **kw):
        super().__init__()
        self.accumulate = 0
        self.max_depth = 6
        self.ris_sample_count = 32
        self.rejection_heuristics_threshold = 0.2
        self.spatial_resampling_sample_count = 5
        self.spatial_resampling_radius = 30.0
        self.spatial_resampling_passes = 3
        self.use_visibility_reuse = 1
        for k, v in kw.items():
            if k == "sky_color":
                self.sky_color = Float3(*v)
            else:
                setattr(self, k, v)

    @classmethod
    def from_numpy(cls, arr):
        """from a 48-byte numpy record laid out like the struct (e.g. oracle/orc.py OPTIONS)"""
        o = cls()
        C.memmove(C.byref(o), arr.tobytes(), 48)
        return o


class _Buffer(C.Structure):
    """device view of TypedBuffer<T>: {T* m_data; size_t m_size:63, m_isDevice:1} (typedbuffer.hpp:14-20)"""

    _fields_ = [("data", C.c_void_p), ("size_and_flag", C.c_uint64)]


class RestirBuffers(C.Structure):
    """crt_restir_buffers: the frame's six TypedBuffers (10_restir_di.cpp:96-122) for the fused frame calls"""

    _fields_ = [("pixels", _Buffer), ("accumulation", _Buffer), ("visibility", _Buffer), ("reservoir0", _Buffer),
                ("reservoir1", _Buffer), ("temporal", _Buffer)]


class SlabLinks(C.Structure):
    """crt_slab_links (include/cedecrt.h): peer pointers of the neighbouring row slabs"""

    _fields_ = [("up", C.c_void_p * 4), ("down", C.c_void_p * 4), ("up_flag", C.c_void_p), ("down_flag", C.c_void_p),
                ("my_flags", C.c_void_p)]


assert C.sizeof(Options) == 48 and C.sizeof(RayGenerator) == 36 and C.sizeof(_Buffer) == 16


class CrtError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise CrtError("libcedecrt.so is not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "or `make -C cedec-2024-rt_b200/csrc`. There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    B, G, P, I, F = _Buffer, C.c_void_p, C.c_void_p, C.c_int, C.c_float
    sigs = {
        "crt_init": [I, C.POINTER(C.c_void_p)],
        "crt_shutdown": [P],
        "crt_set_math_mode": [P, I],
        "crt_set_light_sampling": [P, I, I],
        "crt_light_sampling_table": [P, G, B, C.POINTER(C.c_void_p), C.POINTER(C.c_uint32)],
        "crt_lights_changed": [P, G],
        "crt_set_reuse_weights": [P, I],
        "crt_set_light_tiles": [P, I, I],
        "crt_light_tiles": [P, G, B, I, C.POINTER(C.c_void_p), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)],
        "crt_set_stream": [P, C.c_void_p],
        "crt_set_frame_overlap": [P, I],
        "crt_frame_join": [P],
        "crt_restir_prefetch_raycast": [P, I, I, G, RayGenerator],
        "crt_set_row_range": [P, I, I],
        "crt_malloc": [P, C.c_size_t, C.POINTER(C.c_void_p)],
        "crt_free": [P, C.c_void_p],
        "crt_memset": [P, C.c_void_p, I, C.c_size_t],
        "crt_memcpy_h2d": [P, C.c_void_p, C.c_void_p, C.c_size_t],
        "crt_memcpy_d2h": [P, C.c_void_p, C.c_void_p, C.c_size_t],
        "crt_memcpy_d2d": [P, C.c_void_p, C.c_void_p, C.c_size_t],
        "crt_memcpy_d2h_async": [P, C.c_void_p, C.c_void_p, C.c_size_t],
        "crt_sync": [P],
        "crt_timer_start": [P],
        "crt_timer_stop_ms": [P, C.POINTER(C.c_float)],
        "crt_profile_begin": [P],
        "crt_profile_end": [P, C.c_char_p, C.c_size_t, C.POINTER(C.c_float), I, C.POINTER(I)],
        "crt_build_geometry": [P, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)],
        "crt_destroy_geometry": [P, G],
        "crt_refit_geometry": [P, G],
        "crt_geometry_stats": [G, C.POINTER(C.c_double)],
        "crt_trace_closest": [P, G, C.c_size_t, C.c_void_p, C.c_void_p, F, F, C.c_void_p, C.c_void_p],
        "crt_trace_any": [P, G, C.c_size_t, C.c_void_p, C.c_void_p, F, F, C.c_void_p],
        "crt_trace_closest_brute": [P, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p, F, F, C.c_void_p,
                                    C.c_void_p],
        "crt_raycast": [P, I, I, G, B, RayGenerator, B],
        "crt_generate_candidate": [P, I, I, I, G, B, B, Float3, B, Options, B],
        "crt_temporal_resampling": [P, I, I, I, G, B, B, Float3, Options, B, B],
        "crt_temporal_resampling_reprojected": [P, I, I, I, G, B, B, Float3, Options, RayGenerator, B, B],
        "crt_temporal_resampling_reprojected_surfaces": [P, I, I, I, G, B, B, Float3, Options, RayGenerator, B, B, B],
        "crt_temporal_resampling_reprojected_motion": [P, I, I, I, G, B, B, Float3, Options, RayGenerator, B, B, B, B],
        "crt_save_temporal_reservoir": [P, I, I, B, B],
        "crt_spatial_resampling": [P, I, I, I, I, G, B, B, Float3, Options, B, B],
        "crt_resolve": [P, B, I, I, G, B, B, Float3, Options, B],
        "crt_clear": [P, B, I, I],
        "crt_tone_mapping": [P, B, B, I, I],
        "crt_path_trace_07": [P, I, I, I, G, B, RayGenerator, Options, B],
        "crt_path_trace_08": [P, I, I, I, G, B, B, RayGenerator, Options, B],
        "crt_path_trace_09": [P, I, I, I, G, B, B, RayGenerator, Options, B],
        "crt_ao_06": [P, B, RayGenerator, I, I, G, B, I],
        "crt_restir_di_frame": [P, I, I, I, G, B, RayGenerator, Float3, B, Options, C.POINTER(RestirBuffers)],
        "crt_restir_frame_begin": [P, I, I, I, G, B, RayGenerator, Float3, B, Options, C.POINTER(RestirBuffers)],
        "crt_restir_spatial_pass": [P, I, I, I, I, G, B, Float3, Options, C.POINTER(RestirBuffers)],
        "crt_restir_frame_end": [P, I, I, G, B, Float3, Options, C.POINTER(RestirBuffers)],
        "crt_restir_output_buffer": [Options, C.POINTER(RestirBuffers), C.POINTER(B)],
        "crt_restir_is_fused": [Options],
        "crt_restir_set_previous_camera": [P, C.POINTER(RayGenerator)],
        "crt_restir_set_previous_frame": [P, C.POINTER(RayGenerator), B],
        "crt_restir_set_previous_triangles": [P, B],
        "crt_restir_set_halo_surfaces": [P, I],
        "crt_restir_class_plane": [P, C.POINTER(C.c_void_p)],
        "crt_reservoir_export_aos": [P, I, I, B, B],
        "crt_reservoir_import_aos": [P, I, I, B, B],
        "crt_ipc_export": [P, C.c_void_p, C.c_char_p],
        "crt_ipc_open": [P, C.c_char_p, C.POINTER(C.c_void_p)],
        "crt_ipc_close": [P, C.c_void_p],
        "crt_restir_reserve": [P, I, I, C.POINTER(C.c_void_p)],
        "crt_slab_status": [P, C.POINTER(C.c_ulonglong)],
        "crt_slab_set_links": [P, C.POINTER(SlabLinks)],
        "crt_slab_exchange": [P, I, I, I, I, C.POINTER(RestirBuffers)],
        "crt_launch": [P, C.c_char_p, C.POINTER(C.c_void_p), C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_uint,
                       C.c_uint],
    }
    for name, args in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.crt_last_error.restype = C.c_char_p
    lib.crt_device_name.restype = C.c_char_p
    lib.crt_device_name.argtypes = [P]
    lib.crt_get_stream.restype = C.c_void_p
    lib.crt_get_stream.argtypes = [P]
    lib.crt_get_tail_stream.restype = C.c_void_p
    lib.crt_get_tail_stream.argtypes = [P]
    lib.crt_shadow_rays_traced.restype = C.c_int
    lib.crt_shadow_rays_traced.argtypes = [P, C.POINTER(C.c_ulonglong)]
    lib.crt_inline_rays_traced.restype = C.c_int
    lib.crt_inline_rays_traced.argtypes = [P, C.POINTER(C.c_ulonglong)]
    lib.crt_rays_decided_at_emission.restype = C.c_int
    lib.crt_rays_decided_at_emission.argtypes = [P, C.POINTER(C.c_ulonglong)]
    lib.crt_launch_count.restype = C.c_ulonglong
    lib.crt_launch_count.argtypes = [P]
    lib.crt_raygen_lookat.restype = None
    lib.crt_raygen_lookat.argtypes = [C.POINTER(RayGenerator), C.POINTER(C.c_float), C.POINTER(C.c_float),
                                      C.POINTER(C.c_float), F, I, I]
    return lib


_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        _LIB = _load()
    return _LIB


PI_F = np.float32(3.14159265358979323846)
FOVY_DEFAULT = float(np.float32(PI_F / np.float32(4.0)))  # PI / 4.0f (10_restir_di.cpp:243)


def lookat(eye, center, width, height, up=(0.0, 1.0, 0.0), fovy=FOVY_DEFAULT):
    """RayGenerator::lookat (common/camera.hpp:11-25); host arithmetic inside the library."""
    rg = RayGenerator()
    arr = lambda v: (C.c_float * 3)(*[float(x) for x in v])
    lib().crt_raygen_lookat(C.byref(rg), arr(eye), arr(center), arr(up), fovy, width, height)
    return rg


class TypedBuffer:
    """TypedBuffer<T>(TYPED_BUFFER_DEVICE) (common/typedbuffer.hpp): owns device memory, frees it on release."""

    def __init__(self, rt, dtype, n, ptr=None):
        self.rt, self.dtype, self.n = rt, np.dtype(dtype), int(n)
        self.owned = ptr is None
        if ptr is None:
            p = C.c_void_p()
            rt._check(rt.lib.crt_malloc(rt.ctx, self.nbytes, C.byref(p)))
            ptr = p.value
        self.ptr = ptr

    @property
    def nbytes(self):
        return self.n * self.dtype.itemsize

    def arg(self):
        return _Buffer(self.ptr, self.n | (1 << 63))

    def to_host(self):
        out = np.empty(self.n, self.dtype)
        if self.n:
            self.rt._check(self.rt.lib.crt_memcpy_d2h(self.rt.ctx, out.ctypes.data, self.ptr, self.nbytes))
        return out

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes == self.nbytes, (arr.nbytes, self.nbytes)
        if self.n:
            self.rt._check(self.rt.lib.crt_memcpy_h2d(self.rt.ctx, self.ptr, arr.ctypes.data, self.nbytes))
        return self

    def copy_from(self, other):
        """device-to-device copy of another buffer of the same size, on the context's stream"""
        assert other.nbytes == self.nbytes, (other.nbytes, self.nbytes)
        if self.n:
            self.rt._check(self.rt.lib.crt_memcpy_d2d(self.rt.ctx, self.ptr, other.ptr, self.nbytes))
        return self

    def zero(self):
        self.rt._check(self.rt.lib.crt_memset(self.rt.ctx, self.ptr, 0, self.nbytes))
        return self

    def free(self):
        if self.owned and self.ptr:
            self.rt.lib.crt_free(self.rt.ctx, self.ptr)
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Geometry:
    """the handle in hiprtGeometry's slot (common/loader.hpp:68-112)"""

    def __init__(self, rt, handle, triangles):
        self.rt, self.handle, self.triangles = rt, handle, triangles

    def stats(self):
        out = (C.c_double * 8)()
        self.rt._check(self.rt.lib.crt_geometry_stats(self.handle, out))
        keys = ("n_tris", "n_nodes", "max_depth", "build_ms", "node_bytes", "tri_bytes", "pad", "refit_ms")
        return dict(zip(keys, list(out)))

    def refit(self):
        """the vertices of `triangles` changed on the device (same count and order): update the tree in place"""
        self.rt._check(self.rt.lib.crt_refit_geometry(self.rt.ctx, self.handle))

    def destroy(self):
        if self.handle:
            self.rt.lib.crt_destroy_geometry(self.rt.ctx, self.handle)
            self.handle = None


class Runtime:
    """One context per GPU (crt_ctx): replaces the Orochi device/context/stream set-up of 10_restir_di.cpp:30-53."""

    def __init__(self, device=0, math_mode=MATH_REFERENCE):
        self.lib = lib()
        ctx = C.c_void_p()
        rc = self.lib.crt_init(device, C.byref(ctx))
        if rc != 0:
            raise CrtError("crt_init(%d) failed (%d): %s" % (device, rc, self.lib.crt_last_error().decode()))
        self.ctx = ctx
        self.device = device
        self.set_math_mode(math_mode)

    def _check(self, rc):
        if rc != 0:
            raise CrtError("libcedecrt error %d: %s" % (rc, self.lib.crt_last_error().decode()))

    def close(self):
        if self.ctx:
            self.lib.crt_shutdown(self.ctx)
            self.ctx = None

    def device_name(self):
        return self.lib.crt_device_name(self.ctx).decode()

    def set_math_mode(self, mode):
        self._check(self.lib.crt_set_math_mode(self.ctx, mode))
        self.math_mode = mode

    def set_light_sampling(self, mode, log2_slots=0):
        """LIGHTS_UNIFORM (the reference, default) or LIGHTS_POWER: select lights in proportion to their emitted power from
        a table of 2^log2_slots slots (0: the default size; include/cedecrt.h: crt_set_light_sampling)"""
        self._check(self.lib.crt_set_light_sampling(self.ctx, mode, log2_slots))
        self.light_mode, self.light_log2 = mode, log2_slots

    def light_sampling_table(self, geom, lights):
        """the light records the kernels read for `lights` (a TypedBuffer of uint32 triangle indices), copied to the host as
        a float32 array of shape (n_slots, 16)"""
        ptr, n = C.c_void_p(), C.c_uint32()
        self._check(self.lib.crt_light_sampling_table(self.ctx, geom.handle, lights.arg(), C.byref(ptr), C.byref(n)))
        out = np.zeros((n.value, 16), np.float32)
        if n.value:
            self._check(self.lib.crt_memcpy_d2h(self.ctx, out.ctypes.data, ptr, out.nbytes))
        return out

    def lights_changed(self, geom):
        """the host changed emission of triangles in place: rebuild the light records at their next use"""
        self._check(self.lib.crt_lights_changed(self.ctx, geom.handle))

    def set_light_tiles(self, log2_tiles, log2_tile_size):
        """presampled light tiles for the ReSTIR DI candidates: 2^log2_tiles tiles of 2^log2_tile_size records drawn once
        per frame from the light records; (0, 0) turns them off (include/cedecrt.h: crt_set_light_tiles)"""
        self._check(self.lib.crt_set_light_tiles(self.ctx, log2_tiles, log2_tile_size))

    def light_tiles(self, geom, lights, frame):
        """the tiles the candidates of `frame` read for `lights`, copied to the host as float32 (T, S, 16)"""
        ptr, t, s = C.c_void_p(), C.c_uint32(), C.c_uint32()
        self._check(self.lib.crt_light_tiles(self.ctx, geom.handle, lights.arg(), frame, C.byref(ptr), C.byref(t), C.byref(s)))
        out = np.zeros((t.value, s.value, 16), np.float32)
        self._check(self.lib.crt_memcpy_d2h(self.ctx, out.ctypes.data, ptr, out.nbytes))
        return out

    def set_reuse_weights(self, mode):
        """REUSE_REFERENCE (the reference's biased merge, default) or REUSE_UNBIASED: 1/Z weights in every temporal and
        spatial merge (include/cedecrt.h: crt_set_reuse_weights)"""
        self._check(self.lib.crt_set_reuse_weights(self.ctx, mode))
        self.reuse_mode = mode

    def set_row_range(self, y_begin=0, y_end=-1):
        """multi-GPU row slabs: kernels compute rows yi in [y_begin, y_end) only; indices stay global"""
        self._check(self.lib.crt_set_row_range(self.ctx, y_begin, y_end))

    def set_stream(self, cuda_stream_ptr):
        self._check(self.lib.crt_set_stream(self.ctx, cuda_stream_ptr))

    def stream(self):
        return self.lib.crt_get_stream(self.ctx)

    def set_frame_overlap(self, on=True):
        """the fused frame's tail (resolve rays + tone mapping) on a second stream beside the next frame's head"""
        self._check(self.lib.crt_set_frame_overlap(self.ctx, 1 if on else 0))

    def restir_prefetch_raycast(self, W, H, geom, raygen):
        """overlap mode: the next frame's primary rays now, on a third stream (no-op otherwise)"""
        self._check(self.lib.crt_restir_prefetch_raycast(self.ctx, W, H, geom.handle, raygen))

    def frame_join(self):
        self._check(self.lib.crt_frame_join(self.ctx))

    def tail_stream(self):
        return self.lib.crt_get_tail_stream(self.ctx)

    def launch_count(self):
        return int(self.lib.crt_launch_count(self.ctx))

    def shadow_rays_traced(self):
        """(visibility-reuse rays, resolve rays) traced through the wavefront queue since crt_init (synchronises)"""
        out = (C.c_ulonglong * 2)()
        self._check(self.lib.crt_shadow_rays_traced(self.ctx, out))
        return int(out[0]), int(out[1])

    def inline_rays_traced(self):
        """(closest-hit, shadow / AO) rays traced inside the single-kernel examples 06-09 since crt_init"""
        out = (C.c_ulonglong * 2)()
        self._check(self.lib.crt_inline_rays_traced(self.ctx, out))
        return int(out[0]), int(out[1])

    def rays_decided_at_emission(self):
        """(visibility-reuse rays of 10_restir_di, shadow rays of the wavefront 08_nee / 09_ris) that the emitting kernel's
        own-triangle pre-test settled as occluded since crt_init; traced + decided = the rays the reference traces"""
        out = (C.c_ulonglong * 2)()
        self._check(self.lib.crt_rays_decided_at_emission(self.ctx, out))
        return int(out[0]), int(out[1])

    def sync(self):
        self._check(self.lib.crt_sync(self.ctx))

    def timer_start(self):
        self._check(self.lib.crt_timer_start(self.ctx))

    def timer_stop_ms(self):
        ms = C.c_float()
        self._check(self.lib.crt_timer_stop_ms(self.ctx, C.byref(ms)))
        return ms.value

    def profile_begin(self):
        self._check(self.lib.crt_profile_begin(self.ctx))

    def profile_end(self, cap=4096):
        """[(kernel name, ms)] for every launch since profile_begin, in launch order"""
        names, ms, n = C.create_string_buffer(cap * 40), (C.c_float * cap)(), C.c_int()
        self._check(self.lib.crt_profile_end(self.ctx, names, len(names), ms, cap, C.byref(n)))
        return list(zip(names.value.decode().split("\n")[:n.value], list(ms)[:n.value]))

    # -- buffers
    def buffer(self, dtype, n):
        return TypedBuffer(self, dtype, n)

    def wrap(self, ptr, dtype, n):
        """view over device memory owned by someone else (e.g. a torch tensor's data_ptr())"""
        return TypedBuffer(self, dtype, n, ptr=ptr)

    def to_device(self, arr):
        arr = np.ascontiguousarray(arr)
        return TypedBuffer(self, arr.dtype, arr.size if arr.dtype.fields is None else len(arr)).upload(arr)

    # -- geometry
    def build_geometry(self, triangles):
        """triangles: TypedBuffer of TRIANGLE on the device (buildHiprtGeometry, loader.hpp:68-112)"""
        h = C.c_void_p()
        self._check(self.lib.crt_build_geometry(self.ctx, triangles.ptr, triangles.n, C.byref(h)))
        return Geometry(self, h, triangles)

    def trace_closest(self, geom, org, dirs, tmin=0.0, tmax=3.402823466e38, brute=False):
        org, dirs = np.ascontiguousarray(org, np.float32), np.ascontiguousarray(dirs, np.float32)
        n = len(org)
        d_o, d_d = self.to_device(org.reshape(-1)), self.to_device(dirs.reshape(-1))
        d_p, d_t = self.buffer(np.int32, n), self.buffer(np.float32, 3 * n)
        if brute:
            self._check(self.lib.crt_trace_closest_brute(self.ctx, geom.triangles.ptr, geom.triangles.n, n, d_o.ptr,
                                                         d_d.ptr, tmin, tmax, d_p.ptr, d_t.ptr))
        else:
            self._check(self.lib.crt_trace_closest(self.ctx, geom.handle, n, d_o.ptr, d_d.ptr, tmin, tmax, d_p.ptr,
                                                   d_t.ptr))
        return d_p.to_host(), d_t.to_host().reshape(n, 3)

    def trace_any(self, geom, org, dirs, tmin=0.0, tmax=3.402823466e38):
        org, dirs = np.ascontiguousarray(org, np.float32), np.ascontiguousarray(dirs, np.float32)
        n = len(org)
        d_o, d_d = self.to_device(org.reshape(-1)), self.to_device(dirs.reshape(-1))
        d_p = self.buffer(np.int32, n)
        self._check(self.lib.crt_trace_any(self.ctx, geom.handle, n, d_o.ptr, d_d.ptr, tmin, tmax, d_p.ptr))
        return d_p.to_host()

    # -- kernels: parameter lists of the reference KERNELs, verbatim
    def raycast(self, W, H, geom, triangles, raygen, visibility):
        self._check(self.lib.crt_raycast(self.ctx, W, H, geom.handle, triangles.arg(), raygen, visibility.arg()))

    def generate_candidate(self, W, H, frame, geom, triangles, visibility, eye, lights, options, reservoirs):
        self._check(self.lib.crt_generate_candidate(self.ctx, W, H, frame, geom.handle, triangles.arg(),
                                                    visibility.arg(), Float3(*eye), lights.arg(), options,
                                                    reservoirs.arg()))

    def temporal_resampling(self, W, H, frame, geom, triangles, visibility, eye, options, previous, reservoirs):
        self._check(self.lib.crt_temporal_resampling(self.ctx, W, H, frame, geom.handle, triangles.arg(),
                                                     visibility.arg(), Float3(*eye), options, previous.arg(),
                                                     reservoirs.arg()))

    def temporal_resampling_reprojected(self, W, H, frame, geom, triangles, visibility, eye, options, prev_raygen, previous,
                                        reservoirs):
        self._check(self.lib.crt_temporal_resampling_reprojected(self.ctx, W, H, frame, geom.handle, triangles.arg(),
                                                                 visibility.arg(), Float3(*eye), options, prev_raygen,
                                                                 previous.arg(), reservoirs.arg()))

    def temporal_resampling_reprojected_surfaces(self, W, H, frame, geom, triangles, visibility, eye, options, prev_raygen,
                                                 prev_visibility, previous, reservoirs):
        """temporal_resampling_reprojected that also reads the previous frame's Visibility buffer at the history pixel: the
        history's surface under REUSE_UNBIASED (include/cedecrt.h: crt_temporal_resampling_reprojected_surfaces)"""
        self._check(self.lib.crt_temporal_resampling_reprojected_surfaces(
            self.ctx, W, H, frame, geom.handle, triangles.arg(), visibility.arg(), Float3(*eye), options, prev_raygen,
            prev_visibility.arg(), previous.arg(), reservoirs.arg()))

    def temporal_resampling_reprojected_motion(self, W, H, frame, geom, triangles, visibility, eye, options, prev_raygen,
                                               prev_triangles, prev_visibility, previous, reservoirs):
        """temporal_resampling_reprojected_surfaces that follows moving geometry: prev_triangles is the previous frame's
        triangle array (include/cedecrt.h: crt_temporal_resampling_reprojected_motion); prev_visibility may be None under
        the reference's weights"""
        pv = prev_visibility.arg() if prev_visibility is not None else _Buffer()
        self._check(self.lib.crt_temporal_resampling_reprojected_motion(
            self.ctx, W, H, frame, geom.handle, triangles.arg(), visibility.arg(), Float3(*eye), options, prev_raygen,
            prev_triangles.arg(), pv, previous.arg(), reservoirs.arg()))

    def save_temporal_reservoir(self, W, H, src, dst):
        self._check(self.lib.crt_save_temporal_reservoir(self.ctx, W, H, src.arg(), dst.arg()))

    def spatial_resampling(self, W, H, frame, pas, geom, triangles, visibility, eye, options, rin, rout):
        self._check(self.lib.crt_spatial_resampling(self.ctx, W, H, frame, pas, geom.handle, triangles.arg(),
                                                    visibility.arg(), Float3(*eye), options, rin.arg(), rout.arg()))

    def resolve(self, accumulation, W, H, geom, triangles, visibility, eye, options, reservoirs):
        self._check(self.lib.crt_resolve(self.ctx, accumulation.arg(), W, H, geom.handle, triangles.arg(),
                                         visibility.arg(), Float3(*eye), options, reservoirs.arg()))

    def clear(self, buf, W, H):
        self._check(self.lib.crt_clear(self.ctx, buf.arg(), W, H))

    def tone_mapping(self, pixels, accumulation, W, H):
        self._check(self.lib.crt_tone_mapping(self.ctx, pixels.arg(), accumulation.arg(), W, H))

    def path_trace(self, example, W, H, frame, geom, triangles, lights, raygen, options, accumulation):
        if example == 7:
            rc = self.lib.crt_path_trace_07(self.ctx, W, H, frame, geom.handle, triangles.arg(), raygen, options,
                                            accumulation.arg())
        else:
            fn = self.lib.crt_path_trace_08 if example == 8 else self.lib.crt_path_trace_09
            rc = fn(self.ctx, W, H, frame, geom.handle, triangles.arg(), lights.arg(), raygen, options,
                    accumulation.arg())
        self._check(rc)

    def ao(self, pixels, raygen, W, H, geom, triangles, n_rays=64):
        self._check(self.lib.crt_ao_06(self.ctx, pixels.arg(), raygen, W, H, geom.handle, triangles.arg(), n_rays))

    # -- fused frame (include/cedecrt.h: crt_restir_di_frame and its staged form)
    @staticmethod
    def restir_buffers(pixels, accumulation, visibility, reservoir0, reservoir1, temporal):
        return RestirBuffers(pixels.arg(), accumulation.arg(), visibility.arg(), reservoir0.arg(), reservoir1.arg(),
                             temporal.arg())

    def restir_set_previous_camera(self, raygen):
        """temporal reprojection inside the fused frame: the previous frame's camera, or None for the reference's same-pixel history"""
        self._check(self.lib.crt_restir_set_previous_camera(self.ctx, C.byref(raygen) if raygen is not None else None))

    def restir_set_previous_frame(self, raygen, visibility):
        """restir_set_previous_camera plus the previous frame's Visibility buffer, kept by the host until the next frame has
        begun (include/cedecrt.h: crt_restir_set_previous_frame); raygen None clears both"""
        vis = visibility.arg() if raygen is not None else _Buffer()
        self._check(self.lib.crt_restir_set_previous_frame(self.ctx, C.byref(raygen) if raygen is not None else None, vis))

    def restir_set_previous_triangles(self, triangles):
        """the previous frame's triangle array for the fused frame's reprojection, kept by the host until the next frame has
        begun (include/cedecrt.h: crt_restir_set_previous_triangles); None clears it"""
        self._check(self.lib.crt_restir_set_previous_triangles(self.ctx, triangles.arg() if triangles is not None else _Buffer()))

    def restir_set_halo_surfaces(self, enable):
        """the fused frame with unbiased reuse weights on a row range or with slab links: restir_frame_begin also produces
        the G-buffer records of the halo rows its spatial passes read (include/cedecrt.h: crt_restir_set_halo_surfaces);
        nothing changes under the reference's weights"""
        self._check(self.lib.crt_restir_set_halo_surfaces(self.ctx, 1 if enable else 0))

    def restir_di_frame(self, W, H, frame, geom, triangles, raygen, eye, lights, options, bufs):
        self._check(self.lib.crt_restir_di_frame(self.ctx, W, H, frame, geom.handle, triangles.arg(), raygen,
                                                 Float3(*eye), lights.arg(), options, C.byref(bufs)))

    def restir_frame_begin(self, W, H, frame, geom, triangles, raygen, eye, lights, options, bufs):
        self._check(self.lib.crt_restir_frame_begin(self.ctx, W, H, frame, geom.handle, triangles.arg(), raygen,
                                                    Float3(*eye), lights.arg(), options, C.byref(bufs)))

    def restir_spatial_pass(self, W, H, frame, pas, geom, triangles, eye, options, bufs):
        self._check(self.lib.crt_restir_spatial_pass(self.ctx, W, H, frame, pas, geom.handle, triangles.arg(),
                                                     Float3(*eye), options, C.byref(bufs)))

    def restir_frame_end(self, W, H, geom, triangles, eye, options, bufs):
        self._check(self.lib.crt_restir_frame_end(self.ctx, W, H, geom.handle, triangles.arg(), Float3(*eye), options,
                                                  C.byref(bufs)))

    def restir_class_plane(self):
        p = C.c_void_p()
        self._check(self.lib.crt_restir_class_plane(self.ctx, C.byref(p)))
        return p.value

    def reservoir_export_aos(self, W, H, soa, aos_out):
        self._check(self.lib.crt_reservoir_export_aos(self.ctx, W, H, soa.arg(), aos_out.arg()))

    def reservoir_import_aos(self, W, H, aos_in, soa):
        self._check(self.lib.crt_reservoir_import_aos(self.ctx, W, H, aos_in.arg(), soa.arg()))

    # -- multi-GPU row slabs with direct peer stores (csrc/slab_p2p.cu)
    def ipc_export(self, ptr):
        h = C.create_string_buffer(64)
        self._check(self.lib.crt_ipc_export(self.ctx, ptr, h))
        return h.raw

    def ipc_open(self, handle):
        p = C.c_void_p()
        self._check(self.lib.crt_ipc_open(self.ctx, handle, C.byref(p)))
        return p.value

    def ipc_close(self, ptr):
        self._check(self.lib.crt_ipc_close(self.ctx, ptr))

    def restir_reserve(self, W, H):
        p = C.c_void_p()
        self._check(self.lib.crt_restir_reserve(self.ctx, W, H, C.byref(p)))
        return p.value

    def slab_set_links(self, links):
        self._check(self.lib.crt_slab_set_links(self.ctx, C.byref(links) if links is not None else None))

    def slab_status(self):
        """0, or the exchange count at which a wait for a neighbouring slab timed out"""
        out = C.c_ulonglong(0)
        self._check(self.lib.crt_slab_status(self.ctx, C.byref(out)))
        return int(out.value)

    def slab_exchange(self, W, H, which, bufs, push_rows=0):
        self._check(self.lib.crt_slab_exchange(self.ctx, W, H, which, push_rows, C.byref(bufs)))

    def launch(self, name, *args):
        """Shader::launch(name, ShaderArgument...) (shader.hpp:179-199): args are ctypes values / structures;
        TypedBuffer arguments are passed as their 16-byte device view, Geometry as its handle."""
        keep = []
        for a in args:
            if isinstance(a, TypedBuffer):
                a = a.arg()
            elif isinstance(a, Geometry):
                a = C.c_void_p(a.handle.value if isinstance(a.handle, C.c_void_p) else a.handle)
            elif isinstance(a, int):
                a = C.c_int(a)
            keep.append(a)
        arr = (C.c_void_p * len(keep))(*[C.cast(C.byref(a), C.c_void_p) for a in keep])
        self._check(self.lib.crt_launch(self.ctx, name.encode(), arr, 1, 1, 1, 256, 1, 1))


def light_indices(tris):
    """indices of emissive triangles, ascending (10_restir_di.cpp:196-206)"""
    e = tris["emissive"]
    return np.nonzero((e[:, 0] > 0) | (e[:, 1] > 0) | (e[:, 2] > 0))[0].astype(np.uint32)


class RestirDI:
    """The application loop of examples/10_restir_di/10_restir_di.cpp:96-122,184-226,229-380, headless:
    buffers live on the device, one `frame()` issues the reference's launch list on the context's stream."""

    def __init__(self, rt, width, height, triangles_host, eye, lookat_pt, options=None, fused=False, reproject=False,
                 light_tiles=None):
        """fused=False: the reference's launch list, one crt_* call per kernel, AoS reservoir buffers (drop-in mode);
        fused=True: one crt_restir_di_frame call per frame (SoA reservoirs inside the same buffers).
        reproject=True (extension): temporal resampling looks the previous reservoir up at the pixel the surface point had
        in the previous frame's camera (crt_temporal_resampling_reprojected; in fused mode crt_restir_set_previous_camera);
        set_camera() moves the camera and clears the accumulation like the reference's loop (10_restir_di.cpp:257-267).
        reproject="surfaces": the same look-up with the previous frame's surfaces, which unbiased reuse weights need with a
        moving camera: two Visibility buffers alternate and last frame's is passed on (the launch list's
        crt_temporal_resampling_reprojected_surfaces; in fused mode crt_restir_set_previous_frame).
        light_tiles (extension): None leaves the context's setting as it is; True sets LIGHT_TILES_DEFAULT, a pair
        (log2_tiles, log2_tile_size) sets those, (0, 0) turns tiles off (Runtime.set_light_tiles).
        set_triangles() moves the geometry; with reprojection the next frame follows it (DESIGN.md section 17)."""
        assert reproject in (False, True, "surfaces"), reproject
        if light_tiles is not None:
            rt.set_light_tiles(*(LIGHT_TILES_DEFAULT if light_tiles is True else light_tiles))
        self.rt, self.W, self.H, self.fused = rt, width, height, fused
        self.reproject, self.prev_raygen = reproject, None
        self.prefetch = False  # fused + crt_set_frame_overlap: trace the next frame's primary rays right after issuing a frame
        n = width * height
        self.options = options or Options()
        self.eye = tuple(float(np.float32(v)) for v in eye)
        self.raygen = lookat(eye, lookat_pt, width, height)
        self.triangles = rt.to_device(triangles_host)
        # set_triangles: last frame's triangle array (allocated on the first move), passed on while `moved` is set
        self.prev_triangles, self.moved = None, False
        self.lights = rt.to_device(light_indices(triangles_host))
        self.geom = rt.build_geometry(self.triangles)
        self.pixels = rt.buffer(np.uint8, 4 * n)
        self.accumulation = rt.buffer(FLOAT4, n)
        self.visibility = rt.buffer(VISIBILITY, n)
        # reproject="surfaces": last frame's Visibility, kept for one more frame (the two buffers swap at each frame)
        self.prev_visibility = rt.buffer(VISIBILITY, n) if reproject == "surfaces" else None
        self.reservoir0 = rt.buffer(RESERVOIR, n)
        self.reservoir1 = rt.buffer(RESERVOIR, n)
        # the reference leaves this uninitialised (10_restir_di.cpp:121-122); zero = "no history" (M = 0)
        self.temporal = rt.buffer(RESERVOIR, n).zero()
        self.output = self.reservoir1
        self.frame_index = 0
        rt.clear(self.accumulation, width, height)

    def set_camera(self, eye, lookat_pt):
        self.eye = tuple(float(np.float32(v)) for v in eye)
        self.raygen = lookat(eye, lookat_pt, self.W, self.H)
        self.rt.clear(self.accumulation, self.W, self.H)

    def set_triangles(self, triangles_host):
        """Moves the geometry: new vertices for the same triangles, in the same order, the same ones emitting.  The tree is
        refitted (Geometry.refit).  With reprojection the next frame follows the motion: its look-ups and, under unbiased
        weights, the history's surfaces read the outgoing array, which is kept in `prev_triangles`
        (crt_temporal_resampling_reprojected_motion; in fused mode crt_restir_set_previous_triangles).  Several calls
        between two frames keep the array of the last frame."""
        triangles_host = np.ascontiguousarray(triangles_host)
        if len(triangles_host) != self.triangles.n or triangles_host.dtype != self.triangles.dtype:
            raise ValueError("set_triangles takes the same number of triangles (%d), in the same layout" % self.triangles.n)
        if self.reproject and not self.moved:
            if self.prev_triangles is None:
                self.prev_triangles = self.rt.buffer(self.triangles.dtype, self.triangles.n)
            self.prev_triangles.copy_from(self.triangles)  # ordered before the upload on the context's stream
            self.moved = True
        self.triangles.upload(triangles_host)
        self.geom.refit()

    def output_reservoirs(self):
        """final reservoirs of the last frame in the reference's AoS layout (host numpy array)"""
        if not self.fused or not lib().crt_restir_is_fused(self.options):
            return self.output.to_host()
        bufs = self.rt.restir_buffers(self.pixels, self.accumulation, self.visibility, self.reservoir0,
                                      self.reservoir1, self.temporal)
        out = _Buffer()
        lib().crt_restir_output_buffer(self.options, C.byref(bufs), C.byref(out))
        src = next(b for b in (self.reservoir0, self.reservoir1, self.temporal) if b.ptr == out.data)
        return self.export_aos(src)

    def export_aos(self, buf):
        tmp = self.rt.buffer(RESERVOIR, self.W * self.H)
        self.rt.reservoir_export_aos(self.W, self.H, buf, tmp)
        return tmp.to_host()

    def frame(self):
        surfaces = self.reproject == "surfaces"
        if surfaces:  # this frame traces into the buffer two frames old; last frame's becomes the previous one
            self.visibility, self.prev_visibility = self.prev_visibility, self.visibility
        rt, W, H, o, g, t, v, eye = (self.rt, self.W, self.H, self.options, self.geom, self.triangles,
                                     self.visibility, self.eye)
        self.frame_index += 1
        f = self.frame_index
        # set_triangles since the last frame: the look-up follows the motion (no history to follow before the first frame)
        motion = self.moved and self.prev_raygen is not None
        self.moved = False
        if self.fused:
            bufs = rt.restir_buffers(self.pixels, self.accumulation, v, self.reservoir0, self.reservoir1, self.temporal)
            if surfaces:
                rt.restir_set_previous_frame(self.prev_raygen, self.prev_visibility)  # None before the first frame
            elif self.reproject:
                rt.restir_set_previous_camera(self.prev_raygen)  # None before the first frame: no history to look up
            if motion:
                rt.restir_set_previous_triangles(self.prev_triangles)
            rt.restir_di_frame(W, H, f, g, t, self.raygen, eye, self.lights, o, bufs)
            if self.reproject:
                self.prev_raygen = RayGenerator.from_buffer_copy(bytes(self.raygen))
                rt.restir_set_previous_camera(None)  # the context serves other hosts too: leave it as the reference behaves
                # (which clears the previous triangles too)
            if self.prefetch:
                rt.restir_prefetch_raycast(W, H, g, self.raygen)
            return
        rt.raycast(W, H, g, t, self.raygen, v)
        rt.generate_candidate(W, H, f, g, t, v, eye, self.lights, o, self.reservoir0)
        if motion:
            rt.temporal_resampling_reprojected_motion(W, H, f, g, t, v, eye, o, self.prev_raygen, self.prev_triangles,
                                                      self.prev_visibility, self.temporal, self.reservoir0)
        elif surfaces and self.prev_raygen is not None:
            rt.temporal_resampling_reprojected_surfaces(W, H, f, g, t, v, eye, o, self.prev_raygen, self.prev_visibility,
                                                        self.temporal, self.reservoir0)
        elif self.reproject and self.prev_raygen is not None:
            rt.temporal_resampling_reprojected(W, H, f, g, t, v, eye, o, self.prev_raygen, self.temporal, self.reservoir0)
        else:
            rt.temporal_resampling(W, H, f, g, t, v, eye, o, self.temporal, self.reservoir0)
        self.prev_raygen = RayGenerator.from_buffer_copy(bytes(self.raygen))
        rt.save_temporal_reservoir(W, H, self.reservoir0, self.temporal)
        bi, bo = self.reservoir0, self.reservoir1
        for k in range(o.spatial_resampling_passes):
            if k != 0:
                bi, bo = bo, bi
            rt.spatial_resampling(W, H, f, k, g, t, v, eye, o, bi, bo)
        self.output = bo
        rt.resolve(self.accumulation, W, H, g, t, v, eye, o, bo)
        rt.tone_mapping(self.pixels, self.accumulation, W, H)
