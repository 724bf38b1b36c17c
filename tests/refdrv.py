"""Test-side ctypes wrapper around oracle/_ref/libtinsel_ref*.so (the reference's own code,
compiled by oracle/Makefile in the build container) and oracle/libtinsel_oracle.so (the CPU
restatement).  TEST INFRASTRUCTURE: only tests/, bench.py's cpu_baseline/reference arm and
__graft_entry__.smoke() may import this."""
import ctypes as C
import os

import numpy as np

from tinsel_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
REFERENCE_ROOT = "/root/reference"

_f32p = C.POINTER(C.c_float)


def _fp(a):
    return a.ctypes.data_as(_f32p)


def ref_lib_path(flavour):
    name = {"literal": "libtinsel_ref.so", "fast": "libtinsel_ref_fast.so"}.get(flavour, "libtinsel_ref_detmath.so")
    return os.path.join(REF_DIR, name)


def have_ref(flavour="detmath"):
    return os.path.exists(ref_lib_path(flavour))


def have_reference_tree():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "src"))


_libs = {}


def ref_gpu_lib_path():
    return os.path.join(REF_DIR, "libtinsel_ref_gpu.so")


def have_ref_gpu():
    return os.path.exists(ref_gpu_lib_path())


def load_ref_gpu():
    if "gpu" not in _libs:
        lib = C.CDLL(ref_gpu_lib_path())
        lib.refgpu_bench.restype = C.c_int
        lib.refgpu_bench.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, _f32p, C.POINTER(C.c_double)]
        _libs["gpu"] = lib
    return _libs["gpu"]


def load_ref(flavour="detmath"):
    if flavour in _libs:
        return _libs[flavour]
    lib = C.CDLL(ref_lib_path(flavour))
    lib.ref_load_tin.restype = C.c_void_p
    lib.ref_load_tin.argtypes = [C.c_char_p, C.c_int, C.c_int]
    lib.ref_from_snapshot.restype = C.c_void_p
    lib.ref_from_snapshot.argtypes = [C.c_char_p]
    lib.ref_scene.restype = C.POINTER(abi.Scene)
    lib.ref_scene.argtypes = [C.c_void_p]
    lib.ref_camera.restype = C.POINTER(abi.Camera)
    lib.ref_camera.argtypes = [C.c_void_p]
    lib.ref_options.restype = C.POINTER(abi.Options)
    lib.ref_options.argtypes = [C.c_void_p]
    for name in ("ref_native_scene", "ref_native_camera", "ref_native_options"):
        getattr(lib, name).restype = C.c_void_p
        getattr(lib, name).argtypes = [C.c_void_p]
    lib.ref_set_size.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.ref_set_mode.argtypes = [C.c_void_p, C.c_int]
    lib.ref_set_max_depth.argtypes = [C.c_void_p, C.c_int]
    lib.ref_save_snapshot.restype = C.c_int
    lib.ref_save_snapshot.argtypes = [C.c_void_p, C.c_char_p]
    lib.ref_render_literal.argtypes = [C.c_void_p, C.c_int, _f32p]
    lib.ref_render_seeded.argtypes = [C.c_void_p, C.c_int, C.c_int, _f32p, C.c_int]
    lib.ref_render_pool.argtypes = [C.c_void_p, C.c_int, C.c_int, _f32p, C.c_int]
    lib.ref_trace_frame.argtypes = [C.c_void_p, C.c_int, _f32p, _f32p, C.c_int]
    lib.ref_destroy.argtypes = [C.c_void_p]
    lib.ref_random_u32.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_uint32)]
    lib.ref_random_f32.argtypes = [C.c_int, C.c_int, _f32p]
    lib.ref_material_ior.restype = C.c_float
    lib.ref_material_ior.argtypes = [C.POINTER(abi.Material)]
    lib.ref_bsdf_eval.argtypes = [C.POINTER(abi.Material), C.c_float, C.c_float, _f32p, _f32p, _f32p, _f32p, _f32p]
    lib.ref_bsdf_sample.argtypes = [C.POINTER(abi.Material), C.c_float, C.c_float, _f32p, _f32p, C.c_int, _f32p, _f32p,
                                    C.POINTER(C.c_int), C.POINTER(C.c_uint32)]
    lib.ref_generate_ray.argtypes = [C.POINTER(abi.Camera), C.c_int, C.c_int, C.c_float, C.c_float, _f32p, _f32p]
    lib.ref_filter_eval.restype = C.c_float
    lib.ref_filter_eval.argtypes = [C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float]
    lib.ref_trace.restype = C.c_int
    lib.ref_trace.argtypes = [C.c_void_p, _f32p, _f32p, C.c_float, _f32p, _f32p]
    lib.ref_probe_sample.argtypes = [C.c_void_p, C.c_int, _f32p, _f32p, _f32p]
    lib.ref_sky_eval.argtypes = [C.c_void_p, _f32p, _f32p, _f32p]
    lib.ref_primitive_sample.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_int, _f32p, _f32p, _f32p]
    lib.ref_finish.argtypes = [_f32p, C.c_int, C.c_float, C.c_float, _f32p]
    lib.ref_write_png.argtypes = [_f32p, C.c_int, C.c_int, C.c_char_p]
    lib.ref_nlm.argtypes = [_f32p, _f32p, C.c_int, C.c_int, C.c_float, C.c_int]
    lib.ref_mesh_bin_export.restype = C.c_int
    lib.ref_mesh_bin_export.argtypes = [C.c_void_p, C.c_int, C.c_char_p]
    lib.ref_mesh_bin_import.restype = C.c_void_p
    lib.ref_mesh_bin_import.argtypes = [C.c_char_p]
    lib.ref_mesh_bin_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_float)]
    lib.ref_mesh_bin_copy.argtypes = [C.c_void_p, _f32p, _f32p, C.POINTER(C.c_int), C.c_void_p, _f32p]
    lib.ref_mesh_bin_free.argtypes = [C.c_void_p]
    _libs[flavour] = lib
    return lib


class RefScene:
    """A reference `Scene` + `Camera` + `Options`, from a .tin (build container) or a .tsnap."""

    def __init__(self, lib, handle):
        if not handle:
            raise RuntimeError("reference scene failed to load")
        self.lib = lib
        self.h = C.c_void_p(handle)

    @classmethod
    def from_tin(cls, path, width=0, height=0, flavour="detmath"):
        lib = load_ref(flavour)
        return cls(lib, lib.ref_load_tin(path.encode(), width, height))

    @classmethod
    def from_snapshot(cls, path, flavour="detmath"):
        lib = load_ref(flavour)
        return cls(lib, lib.ref_from_snapshot(path.encode()))

    @property
    def scene(self):
        return self.lib.ref_scene(self.h)

    @property
    def camera(self):
        return self.lib.ref_camera(self.h).contents

    @property
    def options(self):
        return self.lib.ref_options(self.h).contents

    def set_size(self, w, h):
        self.lib.ref_set_size(self.h, w, h)

    def set_mode(self, mode):
        self.lib.ref_set_mode(self.h, mode)

    def set_max_depth(self, d):
        self.lib.ref_set_max_depth(self.h, d)

    def save_snapshot(self, path):
        if self.lib.ref_save_snapshot(self.h, path.encode()) != 0:
            raise RuntimeError("snapshot save failed: " + path)

    def _shape(self):
        o = self.options
        return o.height, o.width

    def render_literal(self, spp):
        h, w = self._shape()
        out = np.zeros((h, w, 4), np.float32)
        self.lib.ref_render_literal(self.h, spp, _fp(out))
        return out

    def render_seeded(self, frame0, nframes, nthreads=1, out=None):
        h, w = self._shape()
        if out is None:
            out = np.zeros((h, w, 4), np.float32)
        self.lib.ref_render_seeded(self.h, frame0, nframes, _fp(out), nthreads)
        return out

    def render_pool(self, frame0, nframes, nthreads=1, out=None):
        """The benchmark's CPU arm: same samples as render_seeded, dynamic 4-row strips over nthreads."""
        h, w = self._shape()
        if out is None:
            out = np.zeros((h, w, 4), np.float32)
        self.lib.ref_render_pool(self.h, frame0, nframes, _fp(out), nthreads)
        return out

    def gpu_bench(self, warmup, calls):
        """The reference's own GPU renderer (src/render.cu RenderGpu, compiled for sm_100a with its Release
        flags) on this scene: (wall ms per Render() call, kernel ms per call).  Speed only, not parity."""
        lib = load_ref_gpu()
        out = (C.c_double * 2)()
        rc = lib.refgpu_bench(self.lib.ref_native_scene(self.h), self.lib.ref_native_camera(self.h),
                              self.lib.ref_native_options(self.h), warmup, calls, None, out)
        if rc != 0:
            raise RuntimeError("refgpu_bench failed: %d" % rc)
        return out[0], out[1]

    def trace_frame(self, frame, nthreads=1):
        h, w = self._shape()
        rad = np.zeros((h, w, 3), np.float32)
        ras = np.zeros((h, w, 2), np.float32)
        self.lib.ref_trace_frame(self.h, frame, _fp(rad), _fp(ras), nthreads)
        return rad, ras

    def trace(self, o, d, time=0.0):
        o = np.asarray(o, np.float32)
        d = np.asarray(d, np.float32)
        t = C.c_float()
        n = np.zeros(3, np.float32)
        prim = self.lib.ref_trace(self.h, _fp(o), _fp(d), time, C.byref(t), _fp(n))
        return prim, t.value, n

    def close(self):
        if self.h:
            self.lib.ref_destroy(self.h)
            self.h = None


# ---- the CPU restatement (oracle/libtinsel_oracle.so) ---------------------------------------------

# "detmath": the deterministic transcendentals the kernels use; "literal": the system libm's, as the
# reference ships (oracle/Makefile port)
PORT_PATHS = {"detmath": os.path.join(ROOT, "oracle", "libtinsel_oracle.so"),
              "literal": os.path.join(ROOT, "oracle", "libtinsel_oracle_libm.so")}
PORT_PATH = PORT_PATHS["detmath"]
_ports = {}


def have_port():
    return os.path.exists(PORT_PATH)


def load_port(flavour="detmath"):
    if flavour in _ports:
        return _ports[flavour]
    lib = C.CDLL(PORT_PATHS[flavour])
    lib.oracle_create.restype = C.c_void_p
    lib.oracle_create.argtypes = [C.POINTER(abi.Scene)]
    lib.oracle_destroy.argtypes = [C.c_void_p]
    lib.oracle_render_seeded.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.POINTER(abi.Options), C.c_int, C.c_int, _f32p, C.c_int]
    lib.oracle_trace_frame.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.POINTER(abi.Options), C.c_int, _f32p, _f32p, C.c_int]
    lib.oracle_render_normals.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.POINTER(abi.Options), _f32p]
    lib.oracle_random_u32.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_uint32)]
    lib.oracle_random_f32.argtypes = [C.c_int, C.c_int, _f32p]
    lib.oracle_material_ior.restype = C.c_float
    lib.oracle_material_ior.argtypes = [C.POINTER(abi.Material)]
    lib.oracle_bsdf_eval.argtypes = [C.POINTER(abi.Material), C.c_float, C.c_float, _f32p, _f32p, _f32p, _f32p, _f32p]
    lib.oracle_bsdf_sample.argtypes = [C.POINTER(abi.Material), C.c_float, C.c_float, _f32p, _f32p, C.c_int, _f32p, _f32p,
                                       C.POINTER(C.c_int), C.POINTER(C.c_uint32)]
    lib.oracle_generate_ray.argtypes = [C.POINTER(abi.Camera), C.c_int, C.c_int, C.c_float, C.c_float, _f32p, _f32p]
    lib.oracle_filter_eval.restype = C.c_float
    lib.oracle_filter_eval.argtypes = [C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float]
    lib.oracle_trace.restype = C.c_int
    lib.oracle_trace.argtypes = [C.c_void_p, _f32p, _f32p, C.c_float, _f32p, _f32p]
    lib.oracle_probe_sample.argtypes = [C.c_void_p, C.c_int, _f32p, _f32p, _f32p]
    lib.oracle_sky_eval.argtypes = [C.c_void_p, _f32p, _f32p, _f32p]
    lib.oracle_primitive_sample.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_int, _f32p, _f32p, _f32p]
    lib.oracle_finish.argtypes = [_f32p, C.c_int, C.c_float, C.c_float, _f32p]
    lib.oracle_quantize.argtypes = [_f32p, C.c_int, C.POINTER(C.c_ubyte)]
    lib.oracle_nlm.argtypes = [_f32p, _f32p, C.c_int, C.c_int, C.c_float, C.c_int]
    abi.declare_snapshot_api(lib)
    _ports[flavour] = lib
    return lib


class PortScene:
    """The CPU restatement over a tb200_scene (from a snapshot or any tb200_scene view)."""

    def __init__(self, scene_ptr, camera, options, keepalive=None, flavour="detmath"):
        self.lib = load_port(flavour)
        self.h = C.c_void_p(self.lib.oracle_create(scene_ptr))
        self.camera = abi.copy_struct(camera)
        self.options = abi.copy_struct(options)
        self._keep = keepalive

    @classmethod
    def from_snapshot(cls, path, flavour="detmath"):
        lib = load_port(flavour)
        h = lib.tb200_snapshot_load(path.encode())
        if not h:
            raise RuntimeError("cannot load " + path)
        scene = lib.tb200_snapshot_scene(h)
        return cls(scene, lib.tb200_snapshot_camera(h).contents, lib.tb200_snapshot_options(h).contents, keepalive=h,
                   flavour=flavour)

    def set_size(self, w, h):
        self.options.width, self.options.height = w, h

    def set_max_depth(self, d):
        self.options.maxDepth = d

    def render_seeded(self, frame0, nframes, nthreads=1, out=None):
        o = self.options
        if out is None:
            out = np.zeros((o.height, o.width, 4), np.float32)
        self.lib.oracle_render_seeded(self.h, C.byref(self.camera), C.byref(o), frame0, nframes, _fp(out), nthreads)
        return out

    render_pool = render_seeded   # RefScene.render_pool computes the same samples, only scheduled differently

    def trace_frame(self, frame, nthreads=1):
        o = self.options
        rad = np.zeros((o.height, o.width, 3), np.float32)
        ras = np.zeros((o.height, o.width, 2), np.float32)
        self.lib.oracle_trace_frame(self.h, C.byref(self.camera), C.byref(o), frame, _fp(rad), _fp(ras), nthreads)
        return rad, ras

    def trace(self, o, d, time=0.0):
        o = np.asarray(o, np.float32)
        d = np.asarray(d, np.float32)
        t = C.c_float()
        n = np.zeros(3, np.float32)
        prim = self.lib.oracle_trace(self.h, _fp(o), _fp(d), time, C.byref(t), _fp(n))
        return prim, t.value, n

    def render_normals(self):
        o = self.options
        out = np.zeros((o.height, o.width, 4), np.float32)
        self.lib.oracle_render_normals(self.h, C.byref(self.camera), C.byref(o), _fp(out))
        return out

    def close(self):
        if self.h:
            self.lib.oracle_destroy(self.h)
            self.h = None


# ---- display/finish step (src/main.cpp:262-271, src/png.cpp:329-343) -----------------------------
def ref_finish(pixels, exposure, limit=1.5, flavour="detmath"):
    """The reference's own ToneMap/LinearToSrgb over `pixels` (H,W,4 running sums)."""
    pixels = np.ascontiguousarray(pixels, np.float32)
    out = np.empty_like(pixels)
    load_ref(flavour).ref_finish(_fp(pixels), pixels.size // 4, exposure, limit, _fp(out))
    return out


def ref_png_bytes(filtered, path, flavour="detmath"):
    """Runs the reference's WritePng on `filtered` (H,W,4) and decodes the file: (H,W,3) uint8."""
    from PIL import Image
    filtered = np.ascontiguousarray(filtered, np.float32)
    h, w = filtered.shape[:2]
    load_ref(flavour).ref_write_png(_fp(filtered), w, h, str(path).encode())
    return np.asarray(Image.open(str(path)).convert("RGB"), dtype=np.uint8)


def port_finish(pixels, exposure, limit=1.5):
    pixels = np.ascontiguousarray(pixels, np.float32)
    out = np.empty_like(pixels)
    load_port().oracle_finish(_fp(pixels), pixels.size // 4, exposure, limit, _fp(out))
    return out


def port_quantize(filtered):
    filtered = np.ascontiguousarray(filtered, np.float32)
    h, w = filtered.shape[:2]
    out = np.empty((h, w, 3), np.uint8)
    load_port().oracle_quantize(_fp(filtered), h * w, out.ctypes.data_as(C.POINTER(C.c_ubyte)))
    return out


def ref_nlm(image, falloff, radius, flavour="detmath"):
    """The reference's NonLocalMeansFilter (src/nlm.cpp) over `image` (H,W,4)."""
    image = np.ascontiguousarray(image, np.float32)
    out = np.empty_like(image)
    load_ref(flavour).ref_nlm(_fp(image), _fp(out), image.shape[1], image.shape[0], falloff, radius)
    return out


def port_nlm(image, falloff, radius):
    image = np.ascontiguousarray(image, np.float32)
    out = np.empty_like(image)
    load_port().oracle_nlm(_fp(image), _fp(out), image.shape[1], image.shape[0], falloff, radius)
    return out
