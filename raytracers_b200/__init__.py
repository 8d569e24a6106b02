"""raytracers_b200 — host-side mirror of the reference's Futhark entry points over libray_b200.so.

The reference's public surface for the render path is four Futhark entries (futhark/ray.fut:176,
223, 241, 246) reached through the generated C API that futhark/main.c calls (main.c:59-141).  This
module binds the same C ABI (include/ray.h, include/ray_b200.h) with ctypes and exposes the same
names with the same argument order and error behaviour:

    ctx = Context()
    scene = ctx.rgbbox()                      # entry rgbbox        (ray.fut:176)
    prepared = ctx.prepare_scene(h, w, scene) # entry prepare_scene (ray.fut:241)  note (h, w)
    img = ctx.render(h, w, prepared)          # entry render        (ray.fut:246)  -> Image [h][w] i32
    ctx.sync(); pixels = img.values()         # futhark_context_sync / futhark_values_i32_2d

All compute happens in hand-written sm_100a CUDA kernels inside the shared library.  There is no
Python or CPU fallback: if the library is missing or no B200 is visible, Context() raises.
This package never imports anything from oracle/.
"""
import ctypes as C
import os

import numpy as np

__all__ = ["Context", "RayError", "lib_path", "load_library", "KERNELS", "declared_symbols", "host_scene",
           "host_camera", "host_lbvh", "host_sample_offsets"]

_HERE = os.path.dirname(os.path.abspath(__file__))
KERNELS = {"auto": 0, "mega": 1, "persistent": 2, "wavefront": 3, "warpqueue": 4, "streamqueue": 5, "lanewalk": 6}
# The measured-slower alternative kernels are not part of the product library: they live in libray_b200_all.so (the
# same objects + render_alt_kernels.cu built with RAYB200_ALL_KERNELS), which Context() loads when one of them is named.
ALT_KERNELS = {2, 3, 5, 6}


class RayError(RuntimeError):
    pass


def lib_path(variant=""):
    # RAY_B200_LIB: load another build of the same library (development A/B runs only)
    if variant == "all":
        return os.path.join(_HERE, "libray_b200_all.so")
    return os.environ.get("RAY_B200_LIB") or os.path.join(_HERE, "libray_b200.so")


class BvhInfo(C.Structure):
    _fields_ = [("n_leaves", C.c_int64), ("n_inner", C.c_int64), ("max_depth", C.c_int32), ("refit_sweeps", C.c_int32),
                ("stale_nodes", C.c_int32), ("smem_nodes", C.c_int32), ("root_box", C.c_float * 6),
                ("camera", C.c_float * 12)]


class WorkCounters(C.Structure):
    _fields_ = [("segments", C.c_uint64), ("node_steps", C.c_uint64), ("box_tests", C.c_uint64),
                ("leaf_tests", C.c_uint64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class RenderJob(C.Structure):
    """struct ray_b200_render_job (include/ray_b200.h)."""
    _fields_ = [("prepared", C.c_void_p), ("h", C.c_int64), ("w", C.c_int64), ("spp", C.c_int32), ("shard_layout", C.c_int32),
                ("out_dev", C.c_void_p), ("out_rgb_dev", C.c_void_p), ("wait_flag", C.c_void_p), ("wait_value", C.c_uint32),
                ("reserved0", C.c_uint32), ("done_flag", C.c_void_p)]


_libs = {}


def load_library(variant=""):
    """Loads libray_b200.so (built by `make -C raytracers_b200/csrc` / __graft_entry__.build()); variant "all" =
    libray_b200_all.so, the build that also carries the alternative kernels K1 / K2 / K4."""
    if variant in _libs:
        return _libs[variant]
    path = lib_path(variant)
    if not os.path.exists(path):
        raise RayError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no fallback implementation)")
    L = C.CDLL(path)
    vp, i64, i32, u64 = C.c_void_p, C.c_int64, C.c_int32, C.c_uint64
    pp = C.POINTER(vp)
    sig = {
        "futhark_context_config_new": (vp, []),
        "futhark_context_config_free": (None, [vp]),
        "futhark_context_config_set_debugging": (None, [vp, C.c_int]),
        "futhark_context_config_set_profiling": (None, [vp, C.c_int]),
        "futhark_context_config_set_logging": (None, [vp, C.c_int]),
        "futhark_context_config_set_device": (None, [vp, C.c_char_p]),
        "futhark_context_config_set_tuning_param": (C.c_int, [vp, C.c_char_p, C.c_size_t]),
        "futhark_get_tuning_param_count": (C.c_int, []),
        "futhark_get_tuning_param_name": (C.c_char_p, [C.c_int]),
        "futhark_context_new": (vp, [vp]),
        "futhark_context_free": (None, [vp]),
        "futhark_context_sync": (C.c_int, [vp]),
        "futhark_context_get_error": (vp, [vp]),
        "futhark_context_report": (vp, [vp]),
        "futhark_context_clear_caches": (C.c_int, [vp]),
        "futhark_new_i32_2d": (vp, [vp, vp, i64, i64]),
        "futhark_new_raw_i32_2d": (vp, [vp, vp, i64, i64]),
        "futhark_free_i32_2d": (C.c_int, [vp, vp]),
        "futhark_values_i32_2d": (C.c_int, [vp, vp, vp]),
        "futhark_values_raw_i32_2d": (vp, [vp, vp]),
        "futhark_shape_i32_2d": (C.POINTER(i64), [vp, vp]),
        "futhark_free_opaque_scene": (C.c_int, [vp, vp]),
        "futhark_store_opaque_scene": (C.c_int, [vp, vp, pp, C.POINTER(C.c_size_t)]),
        "futhark_restore_opaque_scene": (vp, [vp, vp]),
        "futhark_free_opaque_prepared_scene": (C.c_int, [vp, vp]),
        "futhark_store_opaque_prepared_scene": (C.c_int, [vp, vp, pp, C.POINTER(C.c_size_t)]),
        "futhark_restore_opaque_prepared_scene": (vp, [vp, vp]),
        "futhark_entry_rgbbox": (C.c_int, [vp, pp]),
        "futhark_entry_irreg": (C.c_int, [vp, pp]),
        "futhark_entry_prepare_scene": (C.c_int, [vp, pp, i64, i64, vp]),
        "futhark_entry_render": (C.c_int, [vp, pp, i64, i64, vp]),
        "ray_b200_context_set_stream": (C.c_int, [vp, vp]),
        "ray_b200_context_set_spp": (C.c_int, [vp, i32]),
        "ray_b200_context_set_kernel": (C.c_int, [vp, i32]),
        "ray_b200_context_set_shard": (C.c_int, [vp, i32, i32]),
        "ray_b200_context_device": (C.c_int, [vp]),
        "ray_b200_context_last_render_ms": (C.c_int, [vp, C.POINTER(C.c_float)]),
        "ray_b200_render_batch": (C.c_int, [vp, C.POINTER(RenderJob), C.c_int32]),
        "ray_b200_render_job_size": (C.c_int64, []),
        "ray_b200_context_set_pipeline": (C.c_int, [vp, i32]),
        "ray_b200_pipeline_join": (C.c_int, [vp]),
        "ray_b200_context_trace_warps": (C.c_int, [vp, C.c_int32]),
        "ray_b200_context_warp_trace": (C.c_int, [vp, C.POINTER(C.c_float), C.c_int64, C.POINTER(C.c_int64)]),
        "ray_b200_context_launch_count": (i64, [vp]),
        "ray_b200_scene_from_arrays": (C.c_int, [vp, pp, vp, i64, vp]),
        "ray_b200_scene_random": (C.c_int, [vp, pp, i64, u64]),
        "ray_b200_scene_num_spheres": (i64, [vp, vp]),
        "ray_b200_scene_get_arrays": (C.c_int, [vp, vp, vp, vp]),
        "ray_b200_prepared_info": (C.c_int, [vp, vp, C.POINTER(BvhInfo)]),
        "ray_b200_prepared_dump": (C.c_int, [vp] * 8),
        "ray_b200_prepared_reupload": (C.c_int, [vp, vp]),
        "ray_b200_prepared_packed": (C.c_int, [vp, vp, vp, vp, vp, vp]),
        "ray_b200_prepared_upload_bytes": (i64, [vp, vp]),
        "ray_b200_prepared_device_bytes": (i64, [vp, vp]),
        "ray_b200_render_into": (C.c_int, [vp, vp, vp, i64, i64, i32, vp]),
        "ray_b200_render_host": (C.c_int, [vp, vp, vp, i64, i64, i32, vp]),
        "ray_b200_entry_render_spp": (C.c_int, [vp, pp, i64, i64, i32, vp]),
        "ray_b200_intersect_into": (C.c_int, [vp, vp, vp, i64, vp, vp, vp]),
        "ray_b200_trace_into": (C.c_int, [vp, vp, vp, i64, vp]),
        "ray_b200_intersect_host": (C.c_int, [vp, vp, vp, i64, vp, vp, vp]),
        "ray_b200_trace_host": (C.c_int, [vp, vp, vp, i64, vp]),
        "ray_b200_shard_tiles": (i64, [i64, i64, i32, i32]),
        "ray_b200_shard_tiles_padded": (i64, [i64, i64, i32]),
        "ray_b200_render_shard_into": (C.c_int, [vp, vp, i64, i64, i32, vp]),
        "ray_b200_detile": (C.c_int, [vp, vp, vp, i64, i64, i32]),
        "ray_b200_count_work": (C.c_int, [vp, i64, i64, i32, vp, C.POINTER(WorkCounters)]),
        "ray_b200_ipc_alloc": (C.c_int, [vp, i64, pp, vp]),
        "ray_b200_ipc_free": (C.c_int, [vp, vp]),
        "ray_b200_ipc_open": (C.c_int, [vp, vp, pp]),
        "ray_b200_ipc_close": (C.c_int, [vp, vp]),
        "ray_b200_flag_wait": (C.c_int, [vp, vp, vp, C.c_uint32, i32]),
        "ray_b200_flag_set": (C.c_int, [vp, vp, vp, C.c_uint32]),
        "ray_b200_flag_status": (C.c_int, [vp, C.POINTER(i64)]),
        "ray_b200_copy_to_host_async": (C.c_int, [vp, vp, vp, vp, i64]),
        "ray_b200_host_scene": (C.c_int, [C.c_char_p, i64, u64, vp, i64, vp, C.POINTER(i64)]),
        "ray_b200_host_camera": (C.c_int, [vp, i64, i64, vp]),
        "ray_b200_host_lbvh": (C.c_int, [vp, i64, vp, vp, vp, vp, vp, vp, vp]),
        "ray_b200_host_sample_offsets": (None, [i32, vp]),
        "ray_b200_version": (C.c_char_p, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError here = the library does not export what the headers declare
        fn.restype = res
        fn.argtypes = args
    L._declared = tuple(sig)
    _libs[variant] = L
    return L


def declared_symbols():
    """Names this binding expects the library to export (the test suite checks them against include/*.h)."""
    return load_library()._declared


_libc_free = None


def _free(ptr):
    global _libc_free
    if _libc_free is None:
        _libc_free = C.CDLL(None).free
        _libc_free.argtypes = [C.c_void_p]
    _libc_free(ptr)


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return C.c_void_p(int(a))  # raw device/host address (e.g. torch.Tensor.data_ptr())


# ---- host-only helpers (no GPU needed): the setup path's host logic, used by the CPU test suite -----------
def host_scene(name, n=0, seed=1):
    """(spheres[n][7], cam7) of a built-in scene generator (ray.fut:176-237 / the random extension)."""
    L = load_library()
    cnt = C.c_int64(0)
    if L.ray_b200_host_scene(name.encode(), int(n), int(seed), None, 0, None, C.byref(cnt)) != 0:
        raise RayError(f"unknown scene {name!r}")
    s = np.empty((cnt.value, 7), np.float32)
    c = np.empty(7, np.float32)
    if L.ray_b200_host_scene(name.encode(), int(n), int(seed), _ptr(s), cnt.value, _ptr(c), None) != 0:
        raise RayError("host_scene failed")
    return s, c


def host_camera(cam7, h, w):
    out = np.empty(12, np.float32)
    c = np.ascontiguousarray(cam7, np.float32)
    if load_library().ray_b200_host_camera(_ptr(c), int(h), int(w), _ptr(out)) != 0:
        raise RayError("host_camera failed")
    return out


def host_lbvh(spheres):
    """prepare_scene's LBVH (bvh.fut:30-59) in the reference's node order, built by the product's host code."""
    s = np.ascontiguousarray(spheres, np.float32).reshape(-1, 7)
    n = s.shape[0]
    m = max(n - 1, 0)
    out = dict(morton=np.empty(n, np.uint32), perm=np.empty(n, np.int32), left=np.empty(m, np.int32),
               right=np.empty(m, np.int32), parent=np.empty(m, np.int32), boxes=np.empty((m, 6), np.float32))
    info = np.zeros(4, np.int32)
    rc = load_library().ray_b200_host_lbvh(_ptr(s), n, _ptr(out["morton"]), _ptr(out["perm"]), _ptr(out["left"]),
                                           _ptr(out["right"]), _ptr(out["parent"]), _ptr(out["boxes"]), _ptr(info))
    if rc == 2:
        raise RayError("prepare_scene: a scene needs at least 2 spheres")
    if rc != 0:
        raise RayError("host_lbvh failed")
    out.update(refit_sweeps=int(info[0]), max_depth=int(info[1]), stale_nodes=int(info[2]))
    return out


def host_sample_offsets(spp):
    t = np.empty((spp, 2), np.float32)
    load_library().ray_b200_host_sample_offsets(int(spp), _ptr(t))
    return t


class _Handle:
    _free_fn = None

    def __init__(self, ctx, handle):
        self.ctx = ctx
        self.handle = handle

    def free(self):
        if self.handle and self.ctx.handle:
            getattr(self.ctx.lib, self._free_fn)(self.ctx.handle, self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Scene(_Handle):
    """`scene` (ray.fut:171-174), opaque as in the generated API."""
    _free_fn = "futhark_free_opaque_scene"

    @property
    def num_spheres(self):
        return int(self.ctx.lib.ray_b200_scene_num_spheres(self.ctx.handle, self.handle))

    def arrays(self):
        n = self.num_spheres
        s = np.empty((n, 7), np.float32)
        c = np.empty(7, np.float32)
        self.ctx._check(self.ctx.lib.ray_b200_scene_get_arrays(self.ctx.handle, self.handle, _ptr(s), _ptr(c)))
        return s, c

    def store(self):
        p = C.c_void_p(None)
        n = C.c_size_t(0)
        self.ctx._check(self.ctx.lib.futhark_store_opaque_scene(self.ctx.handle, self.handle, C.byref(p), C.byref(n)))
        blob = C.string_at(p, n.value)
        _free(p)
        return blob


class PreparedScene(_Handle):
    """`prepared_scene` (ray.fut:239): LBVH + camera, resident in HBM."""
    _free_fn = "futhark_free_opaque_prepared_scene"

    def info(self):
        bi = BvhInfo()
        self.ctx._check(self.ctx.lib.ray_b200_prepared_info(self.ctx.handle, self.handle, C.byref(bi)))
        return {"n_leaves": bi.n_leaves, "n_inner": bi.n_inner, "max_depth": bi.max_depth,
                "refit_sweeps": bi.refit_sweeps, "stale_nodes": bi.stale_nodes, "smem_nodes": bi.smem_nodes,
                "root_box": np.array(bi.root_box[:], np.float32), "camera": np.array(bi.camera[:], np.float32)}

    def dump(self):
        n = int(self.info()["n_leaves"])
        out = dict(morton=np.empty(n, np.uint32), perm=np.empty(n, np.int32), left=np.empty(n - 1, np.int32),
                   right=np.empty(n - 1, np.int32), parent=np.empty(n - 1, np.int32),
                   boxes=np.empty((n - 1, 6), np.float32))
        self.ctx._check(self.ctx.lib.ray_b200_prepared_dump(self.ctx.handle, self.handle, _ptr(out["morton"]),
                                                            _ptr(out["perm"]), _ptr(out["left"]), _ptr(out["right"]),
                                                            _ptr(out["parent"]), _ptr(out["boxes"])))
        return out

    def packed(self):
        """The packed BVH2C arrays as they sit in HBM (nodes, nodes_soa, geom, colour)."""
        n = int(self.info()["n_leaves"])
        out = dict(nodes=np.empty((n - 1, 16), np.float32), nodes_soa=np.empty((4, n - 1, 4), np.float32),
                   geom=np.empty((n, 4), np.float32), colour=np.empty((n, 4), np.float32))
        self.ctx._check(self.ctx.lib.ray_b200_prepared_packed(self.ctx.handle, self.handle, _ptr(out["nodes"]),
                                                              _ptr(out["nodes_soa"]), _ptr(out["geom"]), _ptr(out["colour"])))
        return out

    def upload_bytes(self):
        return int(self.ctx.lib.ray_b200_prepared_upload_bytes(self.ctx.handle, self.handle))

    def device_bytes(self):
        return int(self.ctx.lib.ray_b200_prepared_device_bytes(self.ctx.handle, self.handle))

    def reupload(self):
        """Host->device copy of the packed BVH + spheres again (the H2D leg of bench.py's e2e step)."""
        self.ctx._check(self.ctx.lib.ray_b200_prepared_reupload(self.ctx.handle, self.handle))

    def store(self):
        p = C.c_void_p(None)
        n = C.c_size_t(0)
        self.ctx._check(self.ctx.lib.futhark_store_opaque_prepared_scene(self.ctx.handle, self.handle, C.byref(p), C.byref(n)))
        blob = C.string_at(p, n.value)
        _free(p)
        return blob


class Image(_Handle):
    """`[h][w]i32` (ray.fut:164): packed 0x00RRGGBB, row 0 = top; lives on the device."""
    _free_fn = "futhark_free_i32_2d"

    @property
    def shape(self):
        s = self.ctx.lib.futhark_shape_i32_2d(self.ctx.handle, self.handle)
        return int(s[0]), int(s[1])

    def values(self, out=None):
        h, w = self.shape
        if out is None:
            out = np.empty((h, w), np.int32)
        self.ctx._check(self.ctx.lib.futhark_values_i32_2d(self.ctx.handle, self.handle, _ptr(out)))
        return out

    def device_ptr(self):
        return int(self.ctx.lib.futhark_values_raw_i32_2d(self.ctx.handle, self.handle) or 0)


class Context:
    """futhark_context + futhark_context_config (main.c:59-64)."""

    def __init__(self, device=None, kernel=None, spp=None, rank=None, world=None, **tuning):
        kid = KERNELS[kernel] if isinstance(kernel, str) else kernel
        self.lib = load_library("all" if kid in ALT_KERNELS else "")
        self.handle = None
        cfg = self.lib.futhark_context_config_new()
        if not cfg:
            raise RayError("futhark_context_config_new failed")
        try:
            if device is not None:
                self.lib.futhark_context_config_set_device(cfg, str(int(device)).encode())
            if kernel is not None:
                tuning["kernel"] = KERNELS[kernel] if isinstance(kernel, str) else int(kernel)
            if spp is not None:
                tuning["spp"] = int(spp)
            if rank is not None:
                tuning["rank"] = int(rank)
            if world is not None:
                tuning["world"] = int(world)
            for k, v in tuning.items():
                if self.lib.futhark_context_config_set_tuning_param(cfg, k.encode(), int(v)) != 0:
                    raise RayError(f"unknown tuning parameter {k!r}")
            h = self.lib.futhark_context_new(cfg)
        finally:
            self.lib.futhark_context_config_free(cfg)
        if not h:
            raise RayError("futhark_context_new returned NULL")
        self.handle = h
        err = self.get_error()
        if err is not None:  # main.c:64 asserts this is NULL
            self.lib.futhark_context_free(h)
            self.handle = None
            raise RayError(err)

    # -- errors --------------------------------------------------------------------------------
    def get_error(self):
        p = self.lib.futhark_context_get_error(self.handle)
        if not p:
            return None
        msg = C.string_at(p).decode(errors="replace")
        _free(p)
        return msg

    def _check(self, rc):
        if rc != 0:
            raise RayError(self.get_error() or f"ray_b200 call failed with code {rc}")

    def _out(self, cls, fn, *args):
        out = C.c_void_p(None)
        self._check(getattr(self.lib, fn)(self.handle, C.byref(out), *args))
        return cls(self, out.value)

    # -- the reference's entries ---------------------------------------------------------------
    def rgbbox(self):
        return self._out(Scene, "futhark_entry_rgbbox")

    def irreg(self):
        return self._out(Scene, "futhark_entry_irreg")

    def prepare_scene(self, h, w, scene):
        return self._out(PreparedScene, "futhark_entry_prepare_scene", int(h), int(w), scene.handle)

    def render(self, h, w, prepared, spp=None):
        if spp is None:
            return self._out(Image, "futhark_entry_render", int(h), int(w), prepared.handle)
        return self._out(Image, "ray_b200_entry_render_spp", int(h), int(w), int(spp), prepared.handle)

    def sync(self):
        self._check(self.lib.futhark_context_sync(self.handle))

    def report(self):
        p = self.lib.futhark_context_report(self.handle)
        msg = C.string_at(p).decode()
        _free(p)
        return msg

    # -- extensions ----------------------------------------------------------------------------
    def scene(self, name, n=None, seed=1):
        if name == "rgbbox":
            return self.rgbbox()
        if name == "irreg":
            return self.irreg()
        if name == "random":
            return self.scene_random(n, seed)
        raise ValueError(f"unknown scene {name!r}")

    def scene_random(self, n, seed=1):
        return self._out(Scene, "ray_b200_scene_random", int(n), int(seed))

    def scene_from_arrays(self, spheres, cam7):
        s = np.ascontiguousarray(spheres, np.float32).reshape(-1, 7)
        c = np.ascontiguousarray(cam7, np.float32).reshape(7)
        return self._out(Scene, "ray_b200_scene_from_arrays", _ptr(s), s.shape[0], _ptr(c))

    def restore_scene(self, blob):
        h = self.lib.futhark_restore_opaque_scene(self.handle, blob)
        if not h:
            raise RayError(self.get_error() or "restore failed")
        return Scene(self, h)

    def restore_prepared_scene(self, blob):
        h = self.lib.futhark_restore_opaque_prepared_scene(self.handle, blob)
        if not h:
            raise RayError(self.get_error() or "restore failed")
        return PreparedScene(self, h)

    def set_stream(self, cuda_stream):
        """cuda_stream: a cudaStream_t handle (torch.cuda.Stream.cuda_stream).  torch's default stream has
        handle 0, which the C API reads as "restore the context's own stream"; it is passed as
        cudaStreamLegacy (0x1) instead so the work really lands on the default stream.  None restores."""
        if cuda_stream is None:
            h = None
        else:
            h = int(cuda_stream) or 1
        self._check(self.lib.ray_b200_context_set_stream(self.handle, C.c_void_p(h)))

    def set_spp(self, spp):
        self._check(self.lib.ray_b200_context_set_spp(self.handle, int(spp)))

    def set_kernel(self, kernel):
        self._check(self.lib.ray_b200_context_set_kernel(self.handle, KERNELS[kernel] if isinstance(kernel, str) else int(kernel)))

    def set_shard(self, rank, world):
        self._check(self.lib.ray_b200_context_set_shard(self.handle, int(rank), int(world)))

    @property
    def device(self):
        return int(self.lib.ray_b200_context_device(self.handle))

    def last_render_ms(self):
        ms = C.c_float(0)
        self._check(self.lib.ray_b200_context_last_render_ms(self.handle, C.byref(ms)))
        return float(ms.value)

    def trace_warps(self, enable=True):
        """Diagnostic: record when each warp of the warp-queue kernel runs out of work (see warp_trace)."""
        self._check(self.lib.ray_b200_context_trace_warps(self.handle, 1 if enable else 0))

    def warp_trace(self):
        """float32[SMs * warps]: exit time of every warp of the last traced render, in us after the first CTA started."""
        n = C.c_int64(0)
        self._check(self.lib.ray_b200_context_warp_trace(self.handle, None, 0, C.byref(n)))
        out = np.empty(n.value, np.float32)
        self._check(self.lib.ray_b200_context_warp_trace(self.handle, out.ctypes.data_as(C.POINTER(C.c_float)), n.value, C.byref(n)))
        return out

    def launch_count(self):
        return int(self.lib.ray_b200_context_launch_count(self.handle))

    def render_into(self, out_pix_dev, h, w, prepared, spp=1, out_rgb_dev=None):
        self._check(self.lib.ray_b200_render_into(self.handle, _ptr(out_pix_dev), _ptr(out_rgb_dev), int(h), int(w), int(spp), prepared.handle))

    def render_host(self, h, w, prepared, spp=1, want_rgb=False, out=None):
        pix = out if out is not None else np.empty((h, w), np.int32)
        rgb = np.empty((h, w, 3), np.float32) if want_rgb else None
        self._check(self.lib.ray_b200_render_host(self.handle, _ptr(pix), _ptr(rgb), int(h), int(w), int(spp), prepared.handle))
        return (pix, rgb) if want_rgb else pix

    def intersect_into(self, rays_dev, n, prepared, index_dev, t_dev, pn_dev=None):
        """Closest hit of n device rays (float32[n][6]: origin, direction) into device int32[n] / float32[n] /
        optional float32[n][6]; asynchronous on the context's stream (include/ray_b200.h "ray queries")."""
        self._check(self.lib.ray_b200_intersect_into(self.handle, prepared.handle, _ptr(rays_dev), int(n), _ptr(index_dev),
                                                     _ptr(t_dev), _ptr(pn_dev)))

    def trace_into(self, rays_dev, n, prepared, colour_dev):
        """Path colour (ray_colour, 50 bounces) of n device rays into device float32[n][3]; asynchronous."""
        self._check(self.lib.ray_b200_trace_into(self.handle, prepared.handle, _ptr(rays_dev), int(n), _ptr(colour_dev)))

    @staticmethod
    def _rays(rays):
        if not isinstance(rays, np.ndarray) or rays.dtype != np.float32 or rays.ndim != 2 or rays.shape[1] != 6:
            raise RayError("rays must be a numpy float32 array of shape (n, 6): origin.xyz, direction.xyz")
        return np.ascontiguousarray(rays)

    def intersect(self, prepared, rays, want_pn=False):
        """Closest hit of each ray: (index int32[n] in the scene's sphere order or -1, t float32[n] or +inf), plus
        pn float32[n][6] (hit point, normal; 0 on a miss) when want_pn."""
        r = self._rays(rays)
        n = r.shape[0]
        index = np.empty(n, np.int32)
        t = np.empty(n, np.float32)
        pn = np.empty((n, 6), np.float32) if want_pn else None
        self._check(self.lib.ray_b200_intersect_host(self.handle, prepared.handle, _ptr(r), n, _ptr(index), _ptr(t), _ptr(pn)))
        return (index, t, pn) if want_pn else (index, t)

    def trace(self, prepared, rays):
        """Colour of each ray's path (ray_colour, 50 bounces, before quantisation): float32[n][3]."""
        r = self._rays(rays)
        colour = np.empty((r.shape[0], 3), np.float32)
        self._check(self.lib.ray_b200_trace_host(self.handle, prepared.handle, _ptr(r), r.shape[0], _ptr(colour)))
        return colour

    def shard_tiles(self, h, w, rank, world):
        return int(self.lib.ray_b200_shard_tiles(int(h), int(w), int(rank), int(world)))

    def shard_tiles_padded(self, h, w, world):
        return int(self.lib.ray_b200_shard_tiles_padded(int(h), int(w), int(world)))

    def render_shard_into(self, out_tiles_dev, h, w, prepared, spp=1):
        self._check(self.lib.ray_b200_render_shard_into(self.handle, _ptr(out_tiles_dev), int(h), int(w), int(spp), prepared.handle))

    def render_batch(self, jobs):
        """jobs: sequence of dicts(prepared=, h=, w=, out_dev=, spp=0, shard_layout=False, out_rgb_dev=None).  Enqueues all
        frames as one stream-ordered operation with up to two of them in flight (ray_b200_render_batch)."""
        arr = (RenderJob * len(jobs))()
        for a, j in zip(arr, jobs):
            a.prepared = j["prepared"].handle
            a.h, a.w = int(j["h"]), int(j["w"])
            a.spp = int(j.get("spp") or 0)
            a.shard_layout = 1 if j.get("shard_layout") else 0
            a.out_dev = int(j["out_dev"])
            a.out_rgb_dev = int(j["out_rgb_dev"]) if j.get("out_rgb_dev") is not None else None
            a.wait_flag = int(j["wait_flag"]) if j.get("wait_flag") else None   # peer-frame protocol (ray_b200.h)
            a.wait_value = int(j.get("wait_value") or 0)
            a.done_flag = int(j["done_flag"]) if j.get("done_flag") else None
        self._check(self.lib.ray_b200_render_batch(self.handle, arr, len(jobs)))

    def set_pipeline(self, on=True):
        """Pipelined submission: render_batch stops joining its second lane (frames of consecutive calls overlap)."""
        self._check(self.lib.ray_b200_context_set_pipeline(self.handle, 1 if on else 0))

    def pipeline_join(self):
        self._check(self.lib.ray_b200_pipeline_join(self.handle))

    # -- peer-memory frames (include/ray_b200.h): raw device addresses as ints ---------------------------------
    def ipc_alloc(self, nbytes):
        """cudaMalloc'ed, zeroed device memory + its 64-byte CUDA IPC handle: (address, handle bytes)."""
        ptr = C.c_void_p(None)
        handle = (C.c_ubyte * 64)()
        self._check(self.lib.ray_b200_ipc_alloc(self.handle, int(nbytes), C.byref(ptr), handle))
        return int(ptr.value), bytes(handle)

    def ipc_free(self, ptr):
        self._check(self.lib.ray_b200_ipc_free(self.handle, C.c_void_p(int(ptr))))

    def ipc_open(self, handle):
        """Maps another process's ipc_alloc allocation (a peer GPU's memory over NVLink); returns the local address."""
        ptr = C.c_void_p(None)
        buf = (C.c_ubyte * 64).from_buffer_copy(bytes(handle))
        self._check(self.lib.ray_b200_ipc_open(self.handle, buf, C.byref(ptr)))
        return int(ptr.value)

    def ipc_close(self, ptr):
        self._check(self.lib.ray_b200_ipc_close(self.handle, C.c_void_p(int(ptr))))

    def flag_wait(self, flag_ptr, value, stream=None, timeout_ms=5000):
        self._check(self.lib.ray_b200_flag_wait(self.handle, C.c_void_p(int(stream) if stream else None), C.c_void_p(int(flag_ptr)),
                                                int(value) & 0xffffffff, int(timeout_ms)))

    def flag_set(self, flag_ptr, value, stream=None):
        self._check(self.lib.ray_b200_flag_set(self.handle, C.c_void_p(int(stream) if stream else None), C.c_void_p(int(flag_ptr)),
                                               int(value) & 0xffffffff))

    def flag_timeouts(self):
        n = C.c_int64(0)
        self._check(self.lib.ray_b200_flag_status(self.handle, C.byref(n)))
        return int(n.value)

    def copy_to_host_async(self, host_ptr, dev_ptr, nbytes, stream=None):
        self._check(self.lib.ray_b200_copy_to_host_async(self.handle, C.c_void_p(int(stream) if stream else None), C.c_void_p(int(host_ptr)),
                                                         C.c_void_p(int(dev_ptr)), int(nbytes)))

    def detile(self, gathered_dev, out_pix_dev, h, w, world):
        self._check(self.lib.ray_b200_detile(self.handle, _ptr(gathered_dev), _ptr(out_pix_dev), int(h), int(w), int(world)))

    def count_work(self, h, w, prepared, spp=1):
        wc = WorkCounters()
        self._check(self.lib.ray_b200_count_work(self.handle, int(h), int(w), int(spp), prepared.handle, C.byref(wc)))
        return wc.as_dict()

    def close(self):
        if self.handle:
            self.lib.futhark_context_free(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
