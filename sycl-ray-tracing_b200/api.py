"""Host-side mirror of the reference's operator interface for the path-tracing hot path.

Same names, argument order and meaning as the reference's C++ classes, so tests read like the reference's own:

    RenderKernel(width, height, render_samples, max_bounces, image_buffer, triangle_buffer, materials_buffer,
                 emissive_triangle_indices, materials_indices, sphere_buffer, bvh, skysphere, env_map_cdf)
        .set_camera(camera) / .render()            include/render_kernel.h:24-57, source/main.cpp:95-113
    Camera(fov, transform) + presets                 include/camera.h:10-40, source/camera.cpp:3-8
    Image(w, h)                                      include/image.h:25-178
    SimpleMaterial                                   include/simple_material.h:6-13
    BVH(triangles).flatten() -> FlattenedBVH         include/bvh.h:263-280, include/flattened_bvh.h:12-48
    compute_env_map_cdf(image)                       source/utils.cpp:126-142

Everything that computes goes through the C ABI of include/b200rt.h to the CUDA kernels; nothing here has a CPU path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import binding as B


def _f32(x):
    return np.ascontiguousarray(x, dtype=np.float32)


# ---- Camera (camera.h:10-40) -----------------------------------------------------------------------------------------
def _hexrow(vals):
    return np.array([float.fromhex(v) for v in vals], dtype=np.float32)


# the reference's presets (camera.cpp:4-8), bit-exact as the compiled reference produces them (sinf/cosf/tan on the host)
_PRESETS = {
    "CORNELL_BOX_CAMERA": ['0x1p+0', '0x0p+0', '0x0p+0', '0x0p+0', '0x0p+0', '0x1p+0', '0x0p+0', '0x1p+0', '0x0p+0', '0x0p+0',
                           '-0x1p+0', '0x1.cp+1', '0x0p+0', '0x0p+0', '0x0p+0', '0x1p+0', '0x1.3504f2p+1'],
    "GANESHA_CAMERA": ['0x1p+0', '0x0p+0', '0x0p+0', '-0x1.4fdf3cp-6', '0x0p+0', '0x1.ee8dd4p-1', '-0x1.0907dcp-2', '0x1.cfddd6p-1',
                       '0x0p+0', '-0x1.0907dcp-2', '-0x1.ee8dd4p-1', '0x1.95c4ccp-1', '0x0p+0', '0x0p+0', '0x0p+0', '0x1p+0', '0x1.3504f2p+1'],
    "ITE_ORB_CAMERA": ['0x1p+0', '0x0p+0', '0x0p+0', '0x0p+0', '0x0p+0', '0x1.6a09e6p-1', '-0x1.6a09e6p-1', '0x1.2aae9p+0',
                       '0x0p+0', '-0x1.6a09e6p-1', '-0x1.6a09e6p-1', '0x1.e8c09p-1', '0x0p+0', '0x0p+0', '0x0p+0', '0x1p+0', '0x1.3504f2p+1'],
    "PBRT_DRAGON_CAMERA": ['0x1p+0', '0x0p+0', '0x0p+0', '0x0p+0', '0x0p+0', '0x1.6a09e6p-1', '-0x1.6a09e6p-1', '0x1.adebc2p+2',
                           '0x0p+0', '-0x1.6a09e6p-1', '-0x1.6a09e6p-1', '0x1.04371ep+3', '0x0p+0', '0x0p+0', '0x0p+0', '0x1p+0', '0x1.3504f2p+1'],
    "MIS_CAMERA": ['0x1p+0', '0x0p+0', '0x0p+0', '0x0p+0', '0x0p+0', '0x1.f838b8p-1', '-0x1.63a1a8p-3', '-0x1.2190e8p+0',
                   '0x0p+0', '-0x1.63a1a8p-3', '-0x1.f838b8p-1', '0x1.5b90ccp+3', '0x0p+0', '0x0p+0', '0x0p+0', '0x1p+0', '0x1.3504f2p+1'],
}


def Identity():
    return np.eye(4, dtype=np.float32)


def Translation(x, y, z):
    m = np.eye(4, dtype=np.float32)
    m[0, 3], m[1, 3], m[2, 3] = x, y, z
    return m


def _rot(angle_deg):
    a = np.float32(np.float32(np.pi) / np.float32(180.0)) * np.float32(angle_deg)     # radians(), mat.cpp:10-13
    return np.float32(np.sin(a)), np.float32(np.cos(a))


def RotationX(angle_deg):
    s, c = _rot(angle_deg)
    return np.array([[1, 0, 0, 0], [0, c, -s, 0], [0, s, c, 0], [0, 0, 0, 1]], dtype=np.float32)


def RotationY(angle_deg):
    s, c = _rot(angle_deg)
    return np.array([[c, 0, s, 0], [0, 1, 0, 0], [-s, 0, c, 0], [0, 0, 0, 1]], dtype=np.float32)


def compose_transform(a, b):
    """Transform * Transform in float32, term order of mat.cpp:365-373."""
    a, b = _f32(a), _f32(b)
    m = np.zeros((4, 4), np.float32)
    for i in range(4):
        for j in range(4):
            acc = np.float32(a[i, 0] * b[0, j])
            for k in range(1, 4):
                acc = np.float32(acc + np.float32(a[i, k] * b[k, j]))
            m[i, j] = acc
    return m


class Camera:
    """view_matrix = transformation * diag(1,1,-1); fov_dist = 1 / tan(fov/2) (camera.h:27-39)."""

    DEFAULT_COORDINATES_SYSTEM = np.diag([1.0, 1.0, -1.0, 1.0]).astype(np.float32)

    def __init__(self, full_fov: float = 45.0, transformation=None):
        t = Identity() if transformation is None else _f32(transformation)
        self.view_matrix = compose_transform(t, Camera.DEFAULT_COORDINATES_SYSTEM)
        self.fov = float(full_fov)
        rad = np.float32(np.float64(np.float32(full_fov) / np.float32(180.0)) * np.pi)   # fov / 180.0f * M_PI (double), to float
        self.fov_dist = np.float32(np.float32(1.0) / np.float32(np.tan(np.float32(rad / np.float32(2.0)))))

    @classmethod
    def from_array17(cls, a17):
        cam = cls.__new__(cls)
        a17 = _f32(a17)
        cam.view_matrix = a17[:16].reshape(4, 4).copy()
        cam.fov_dist = np.float32(a17[16])
        cam.fov = 45.0
        return cam

    def as_array17(self) -> np.ndarray:
        return np.concatenate([_f32(self.view_matrix).reshape(16), np.array([self.fov_dist], np.float32)])


for _name, _vals in _PRESETS.items():
    setattr(Camera, _name, Camera.from_array17(_hexrow(_vals)))


class _PinnedOwner:
    def __init__(self):
        self._pinned = None

    def __del__(self):
        try:
            if self._pinned:
                B.load_library().b200rt_host_free(self._pinned)
                self._pinned = None
        except Exception:
            pass


def pinned_array(shape, dtype=np.float32, owner=None) -> np.ndarray:
    """numpy array over page-locked host memory (b200rt_host_alloc). The memory lives as long as `owner` (default: an owner
    object attached to the returned array's base)."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    B.check(B.load_library().b200rt_host_alloc(max(n, 1), C.byref(p)))
    own = owner if owner is not None else _PinnedOwner()
    own._pinned = p
    buf = (C.c_ubyte * max(n, 1)).from_address(p.value)
    buf._owner = own                      # keeps the allocation alive with the array
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def rng_stream(x: int, y: int, spp: int, n: int = 16):
    """The RNG stream of pixel (x, y) as ray_trace_pixel seeds it (render_kernel.cpp:77-82), computed on the GPU:
    (state after the 10 warm-up draws, the next n floats)."""
    st = C.c_uint32()
    fl = np.zeros(n, np.float32)
    B.check(B.load_library().b200rt_rng_stream(x, y, spp, n, C.byref(st), B.fptr(fl)))
    return int(st.value), fl


def parse_obj(path: str) -> dict:
    """Utils::parse_obj (utils.cpp:16-98) through the library's own ingest (b200rt_obj_load): dict(tri9, mat_idx, mats10, emissive)."""
    L = B.load_library()
    h = C.c_void_p()
    B.check(L.b200rt_obj_load(str(path).encode(), C.byref(h)))
    try:
        FP, IP = C.POINTER(C.c_float), C.POINTER(C.c_int)
        tri, mi, mats, em = FP(), IP(), FP(), IP()
        nt, nm, ne = C.c_int(), C.c_int(), C.c_int()
        B.check(L.b200rt_obj_get(h, C.byref(tri), C.byref(nt), C.byref(mi), C.byref(mats), C.byref(nm), C.byref(em), C.byref(ne)))
        cp = lambda p, n, dt: (np.ctypeslib.as_array(p, shape=(n,)).astype(dt, copy=True) if n else np.zeros(0, dt))
        return dict(tri9=cp(tri, nt.value * 9, np.float32).reshape(-1, 9), mat_idx=cp(mi, nt.value, np.int32),
                    mats10=cp(mats, nm.value * 10, np.float32).reshape(-1, 10), emissive=cp(em, ne.value, np.int32))
    finally:
        L.b200rt_obj_destroy(h)


def read_image_float(path: str, flip_y: bool = True) -> np.ndarray:
    """Utils::read_image_float for Radiance .hdr files (utils.cpp:100-124) through b200rt_hdr_load: (h, w, 3) float32 RGB — pass it as
    a Scene's skysphere (the RGBA expansion, alpha 0, happens on the device)."""
    L = B.load_library()
    h = C.c_void_p()
    B.check(L.b200rt_hdr_load(str(path).encode(), 1 if flip_y else 0, C.byref(h)))
    try:
        p, w, ht = C.POINTER(C.c_float)(), C.c_int(), C.c_int()
        B.check(L.b200rt_hdr_get(h, C.byref(p), C.byref(w), C.byref(ht)))
        return np.ctypeslib.as_array(p, shape=(ht.value, w.value, 3)).astype(np.float32, copy=True)
    finally:
        L.b200rt_hdr_destroy(h)


# ---- Image (image.h:25-178) ----------------------------------------------------------------------------------------------
class Image:
    """RGBA float32, row-major, row 0 = bottom. Image(w, h) starts as Color::Black() = (0, 0, 0, 1)."""

    def __init__(self, w: int = 0, h: int = 0, color=(0.0, 0.0, 0.0, 1.0), data=None, pinned: bool = False):
        """pinned=True puts the pixels in page-locked memory (b200rt_host_alloc): renders then copy at the full PCIe rate."""
        self._pinned = None
        if data is not None:
            d = _f32(data)
            assert d.ndim == 3 and d.shape[2] == 4
            self.pixels = d
        else:
            self.pixels = pinned_array((h, w, 4), np.float32, self) if pinned else np.empty((h, w, 4), np.float32)
            self.pixels[...] = np.asarray(color, np.float32)

    def __del__(self):
        try:
            if getattr(self, "_pinned", None):
                B.load_library().b200rt_host_free(self._pinned)
                self._pinned = None
        except Exception:
            pass

    def width(self):
        return self.pixels.shape[1]

    def height(self):
        return self.pixels.shape[0]

    def data(self):
        return self.pixels

    def __getitem__(self, index):
        return self.pixels.reshape(-1, 4)[index]


@dataclass
class SimpleMaterial:
    """simple_material.h:6-13 (defaults included)."""
    emission: tuple = (0.0, 0.0, 0.0)
    diffuse: tuple = (1.0, 0.2, 0.7)
    metalness: float = 0.0
    roughness: float = 1.0

    def as_array10(self):
        e, d = tuple(self.emission)[:3], tuple(self.diffuse)[:3]
        return np.array([e[0], e[1], e[2], 1.0, d[0], d[1], d[2], 1.0, self.metalness, self.roughness], np.float32)


def materials_to_array(materials) -> np.ndarray:
    if isinstance(materials, np.ndarray):
        return _f32(materials).reshape(-1, 10)
    return np.stack([m.as_array10() for m in materials]).astype(np.float32)


def compute_env_map_cdf(skysphere: "Image | np.ndarray") -> np.ndarray:
    """Utils::compute_env_map_cdf (utils.cpp:126-142): serial float32 running sum of the per-texel luminance, whose
    weights are double constants (image.h:84)."""
    px = skysphere.pixels if isinstance(skysphere, Image) else _f32(skysphere)
    p = px.reshape(-1, 4).astype(np.float64)
    lum = (0.3086 * p[:, 0] + 0.6094 * p[:, 1] + 0.0820 * p[:, 2]).astype(np.float32)
    return np.cumsum(lum, dtype=np.float32)          # add.accumulate in float32 == the reference's serial loop


def env_alias_table(skysphere):
    """Alias table of an env map's luminance, built by the library on the host (b200rt_env_alias_table): (prob, alias, total)."""
    env = _f32(skysphere.pixels if isinstance(skysphere, Image) else skysphere)
    h, w = env.shape[:2]
    prob = np.empty(h * w, np.float32); alias = np.empty(h * w, np.int32); total = C.c_double()
    B.check(B.load_library().b200rt_env_alias_table(B.fptr(env), w, h, B.fptr(prob), alias.ctypes.data_as(C.POINTER(C.c_int)), C.byref(total)))
    return prob, alias, total.value


def OIDN_denoise(image, blend_factor: float = 1.0, iterations: int = 0, sigma: float = 0.0, albedo=None, normal=None) -> np.ndarray:
    """The denoise stage of main.cpp:118-120 (Utils::OIDN_denoise, utils.cpp:144-196) on the GPU: an edge-avoiding a-trous filter
    standing in for OIDN (whose binaries the reference does not ship), then blend * denoised + (1 - blend) * noisy. (h, w, 3|4).
    albedo / normal: OIDN's auxiliary images, (h, w, 3) each (Scene.render_aovs), used as edge-stopping guides when given."""
    img = _f32(image.pixels if isinstance(image, Image) else image)
    h, w, ch = img.shape
    guides = []
    for name, g in (("albedo", albedo), ("normal", normal)):
        if g is not None:
            g = _f32(g)
            if g.shape != (h, w, 3):
                raise ValueError(f"{name} guide has shape {g.shape}, the image needs {(h, w, 3)}")
        guides.append(g)
    out = np.empty_like(img)
    L = B.load_library()
    if albedo is None and normal is None:
        B.check(L.b200rt_denoise(B.fptr(img), ch, w, h, blend_factor, iterations, sigma, B.fptr(out)))
    else:
        B.check(L.b200rt_denoise_guided(B.fptr(img), ch, B.fptr(guides[0]), B.fptr(guides[1]), w, h, blend_factor, iterations, sigma,
                                        B.fptr(out)))
    return out


def quantise_rgba8(image, flip_y: bool = True) -> np.ndarray:
    """write_image_png's quantisation (image_io.cpp:165-182) on the GPU: (h, w, 4) float32 -> (h, w, 4) uint8."""
    img = _f32(image)
    h, w = img.shape[:2]
    out = np.empty((h, w, 4), np.uint8)
    B.check(B.load_library().b200rt_quantise_rgba8(B.fptr(img), w, h, 1 if flip_y else 0, out.ctypes.data_as(C.POINTER(C.c_ubyte))))
    return out


WIDE_NODE_DTYPE = np.dtype([("p", "<f4", 3), ("e", "u1", 3), ("imask", "u1"), ("child_base", "<u4"), ("tri_base", "<u4"), ("valid24", "<u4"),
                            ("spare", "<u4"), ("lox", "u1", 8), ("loy", "u1", 8), ("loz", "u1", 8), ("hix", "u1", 8), ("hiy", "u1", 8), ("hiz", "u1", 8)])
assert WIDE_NODE_DTYPE.itemsize == 80


# ---- BVH / FlattenedBVH ---------------------------------------------------------------------------------------------------
class BVH:
    """BVH(std::vector<Triangle>*) (bvh.cpp:19-37). Holds the host-side flattened tree built by the C library."""

    def __init__(self, triangles, max_leaf_size: int = 3, use_diag_slabs: bool = True, sah_bins: int = 16, num_threads: int = 0,
                 on_device: bool = False, device: int = -1):
        """on_device=True: linear BVH built by the GPU (b200rt_bvh_build_device) instead of the host's binned-SAH builder."""
        L = B.load_library()
        self.triangles = _f32(triangles).reshape(-1, 9)
        h = C.c_void_p()
        if on_device:
            B.check(L.b200rt_bvh_build_device(B.fptr(self.triangles), len(self.triangles), device, C.byref(h)))
        else:
            opts = B.BvhOptions(max_leaf_size, sah_bins, 1 if use_diag_slabs else 0, num_threads)
            B.check(L.b200rt_bvh_build(B.fptr(self.triangles), len(self.triangles), C.byref(opts), C.byref(h)))
        self._h = h

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                B.load_library().b200rt_bvh_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def info(self) -> dict:
        out = B.BvhInfo()
        B.check(B.load_library().b200rt_bvh_get_info(self._h, C.byref(out)))
        return out.as_dict()

    def check(self) -> None:
        B.check(B.load_library().b200rt_bvh_check(self._h, B.fptr(self.triangles), len(self.triangles)))

    def flatten(self) -> "FlattenedBVH":
        return FlattenedBVH(self)


class FlattenedBVH:
    """The re-laid-out FlattenedBVH (flattened_bvh.h:12-48): numpy views of the 64-byte axis / diag records and the
    leaf-ordered triangle stream. `intersect` runs the CUDA traversal (there is no host traversal)."""

    def __init__(self, bvh: BVH):
        self.bvh = bvh
        L = B.load_library()
        info = bvh.info()
        FP = C.POINTER(C.c_float)
        a, d, t = FP(), FP(), FP()
        B.check(L.b200rt_bvh_get_arrays(bvh._h, C.byref(a), C.byref(d), C.byref(t)))
        n = info["n_inner_nodes"]
        self.axis = np.ctypeslib.as_array(a, shape=(n, 16)) if (n and a) else np.zeros((0, 16), np.float32)
        # device-built trees carry no diagonal slabs (has_diag_slabs = 0): no diag records
        self.diag = np.ctypeslib.as_array(d, shape=(n, 16)) if (n and d and info["has_diag_slabs"]) else np.zeros((0, 16), np.float32)
        self.tris = np.ctypeslib.as_array(t, shape=(max(info["n_triangles"], 0), 12)) if info["n_triangles"] else np.zeros((0, 12), np.float32)
        # the 8-ary layout as a structured array (80-byte records, csrc/bvh_build.h WideNode)
        wp, wn = C.c_void_p(), C.c_int()
        B.check(L.b200rt_bvh_get_wide_nodes(bvh._h, C.byref(wp), C.byref(wn)))
        self.wide = (np.ctypeslib.as_array(C.cast(wp, C.POINTER(C.c_ubyte)), shape=(wn.value * 80,)).view(WIDE_NODE_DTYPE)
                     if wn.value else np.zeros(0, WIDE_NODE_DTYPE))

    def get_nodes(self):
        return self.axis, self.diag

    def intersect(self, rays6, triangles=None, any_hit: bool = False):
        """Batch version of FlattenedBVH::intersect(ray, hit_info, triangles): returns (prim, t, extra8)."""
        tri = self.bvh.triangles if triangles is None else _f32(triangles).reshape(-1, 9)
        scene = Scene(tri, np.zeros(len(tri), np.int32), materials_to_array([SimpleMaterial()]), np.zeros(0, np.int32),
                      bvh=self.bvh)
        return scene.trace_rays(rays6, any_hit=any_hit)


# ---- device-resident scene ---------------------------------------------------------------------------------------------------
_DIM_ENV = None


def constant_env(value: float = 1.0e-20, w: int = 4, h: int = 2) -> np.ndarray:
    """"No environment map" for the reference means a constant, negligibly dim one (an all-zero map makes its CDF
    sampling divide 0/0 — SURVEY §8c)."""
    e = np.full((h, w, 4), value, np.float32)
    e[..., 3] = 0.0
    return e


class Scene:
    def __init__(self, triangles, materials_indices, materials, emissive_triangle_indices, spheres=None, skysphere=None,
                 env_map_cdf=None, bvh: BVH | None = None, device: int = -1, devices=None):
        """devices: a list of CUDA device ids (or an int N = devices 0..N-1) replicates the scene on several GPUs of this
        process (b200rt_scene_create_multi); render() / render_rgba8() then partition every frame over them.
        skysphere may be (h, w, 3): stb's RGB triplets, expanded to RGBA on the device (multi-device entry point only)."""
        L = B.load_library()
        self.tri = _f32(triangles).reshape(-1, 9)
        self.mat_idx = np.ascontiguousarray(materials_indices, np.int32)
        self.mats = materials_to_array(materials)
        self.emissive = np.ascontiguousarray(emissive_triangle_indices, np.int32)
        sph = np.zeros(0, np.uint8)
        n_sph = 0
        if spheres is not None and len(spheres):
            rec = np.zeros(len(spheres), dtype=[("c", np.float32, 3), ("r", np.float32), ("prim", np.int32)])
            for i, s in enumerate(spheres):
                rec[i] = (tuple(s[0]), s[1], s[2])
            sph = rec.view(np.uint8)
            n_sph = len(spheres)
        env = constant_env() if skysphere is None else (skysphere.pixels if isinstance(skysphere, Image) else _f32(skysphere))
        assert env.ndim == 3 and env.shape[2] in (3, 4)
        self.env = np.ascontiguousarray(env)
        cdf = None if env_map_cdf is None else _f32(env_map_cdf)
        h = C.c_void_p()
        if devices is None and self.env.shape[2] == 4:
            B.check(L.b200rt_scene_create(
                B.fptr(self.tri), len(self.tri), B.iptr(self.mat_idx), len(self.mat_idx), B.fptr(self.mats), len(self.mats),
                B.iptr(self.emissive), len(self.emissive), sph.ctypes.data_as(C.c_void_p) if n_sph else None, n_sph,
                B.fptr(self.env), self.env.shape[1], self.env.shape[0], B.fptr(cdf), bvh._h if bvh is not None else None,
                device, C.byref(h)))
        else:
            if devices is None:
                devices = [device]
            devs = np.arange(devices, dtype=np.int32) if isinstance(devices, int) else np.ascontiguousarray(devices, np.int32)
            B.check(L.b200rt_scene_create_multi(
                B.fptr(self.tri), len(self.tri), B.iptr(self.mat_idx), len(self.mat_idx), B.fptr(self.mats), len(self.mats),
                B.iptr(self.emissive), len(self.emissive), sph.ctypes.data_as(C.c_void_p) if n_sph else None, n_sph,
                B.fptr(self.env), self.env.shape[2], self.env.shape[1], self.env.shape[0], B.fptr(cdf),
                bvh._h if bvh is not None else None, B.iptr(devs), len(devs), C.byref(h)))
        self._h = h

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                B.load_library().b200rt_scene_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def bvh_info(self) -> dict:
        out = B.BvhInfo()
        B.check(B.load_library().b200rt_scene_get_bvh_info(self._h, C.byref(out)))
        return out.as_dict()

    def device_bytes(self) -> int:
        return int(B.load_library().b200rt_scene_device_bytes(self._h))

    def device_count(self) -> int:
        return int(B.load_library().b200rt_scene_device_count(self._h))

    def env_alias(self):
        """The device-built alias table (b200rt_scene_get_env_alias): (prob, alias, total)."""
        n = self.env.shape[0] * self.env.shape[1]
        prob = np.empty(n, np.float32); alias = np.empty(n, np.int32); total = C.c_double()
        B.check(B.load_library().b200rt_scene_get_env_alias(self._h, B.fptr(prob), B.iptr(alias), C.byref(total)))
        return prob, alias, total.value

    def env_cdf(self) -> np.ndarray:
        """The CDF the integrator searches (device-computed when none was passed in)."""
        out = np.empty(self.env.shape[0] * self.env.shape[1], np.float32)
        B.check(B.load_library().b200rt_scene_get_env_cdf(self._h, B.fptr(out)))
        return out

    def env_cdf_search(self, values, use_guide: bool = True) -> np.ndarray:
        """env_map_cdf_search (render_kernel.cpp:532-567) for a batch of values on the device: (n, 2) int32 texels (x, y)."""
        v = _f32(values).reshape(-1)
        out = np.empty((len(v), 2), np.int32)
        B.check(B.load_library().b200rt_env_cdf_search(self._h, B.fptr(v), len(v), 1 if use_guide else 0, B.iptr(out)))
        return out

    def build_env_alias(self) -> None:
        """Alias table of the env map's luminance for FLAG_ENV_ALIAS renders (b200rt_scene_build_env_alias)."""
        B.check(B.load_library().b200rt_scene_build_env_alias(self._h))

    def set_materials(self, materials) -> None:
        self.mats = materials_to_array(materials)
        B.check(B.load_library().b200rt_scene_set_materials(self._h, B.fptr(self.mats), len(self.mats)))

    def update_triangles(self, triangles) -> dict:
        """New vertex positions for the scene's triangles (b200rt_scene_update_triangles): (n, 9) float32, n = the scene's triangle
        count, triangle i replacing triangle i. The BVH is refitted on the device; every result afterwards equals a fresh Scene's
        from these vertices bit for bit. Returns the stats (kernel_ms, total_ms, gpu_launches, h2d_bytes)."""
        tri = _f32(triangles)
        if tri.shape != self.tri.shape:
            raise ValueError(f"triangles have shape {tri.shape}; this scene takes {self.tri.shape} (an update keeps the topology)")
        st = B.Stats()
        B.check(B.load_library().b200rt_scene_update_triangles(self._h, B.fptr(tri), len(tri), C.byref(st)))
        self.tri = tri.copy() if tri is triangles else tri
        return st.as_dict()

    def update_triangles_device(self, dev_ptr: int, n: int, stream_ptr: int = 0) -> dict:
        """update_triangles from device memory of the scene's first device (b200rt_scene_update_triangles_device), e.g.
        tensor.data_ptr() of an (n, 9) float32 CUDA tensor, ordered after the work already queued on stream_ptr. self.tri is not
        updated (the vertices never reach the host). Returns the stats."""
        st = B.Stats()
        B.check(B.load_library().b200rt_scene_update_triangles_device(self._h, C.c_void_p(dev_ptr), n, C.c_void_p(stream_ptr), C.byref(st)))
        return st.as_dict()

    def bvh_arrays(self, replica: int = 0) -> dict:
        """The resident BVH of one replica, downloaded (b200rt_scene_get_bvh_arrays): wide (WIDE_NODE_DTYPE records), axis and diag
        ((n_inner_nodes, 16) float32; diag is empty without diagonal slabs) and tris ((n_triangles, 12) float32)."""
        info = self.bvh_info()
        wide = np.zeros(info["n_wide_nodes"], WIDE_NODE_DTYPE)
        axis = np.zeros((info["n_inner_nodes"], 16), np.float32)
        diag = np.zeros((info["n_inner_nodes"] if info["has_diag_slabs"] else 0, 16), np.float32)
        tris = np.zeros((info["n_triangles"], 12), np.float32)
        B.check(B.load_library().b200rt_scene_get_bvh_arrays(self._h, replica, wide.ctypes.data_as(C.c_void_p), B.fptr(axis),
                                                             B.fptr(diag) if len(diag) else None, B.fptr(tris)))
        return dict(wide=wide, axis=axis, diag=diag, tris=tris)

    @staticmethod
    def _opts(integrator=B.INTEGRATOR_WAVEFRONT, flags=0, rank=0, world=1):
        return B.RenderOptions(integrator, flags, rank, world)

    def render(self, camera: Camera, w: int, h: int, spp: int, max_bounces: int, framebuffer: np.ndarray | None = None,
               integrator: int = B.INTEGRATOR_WAVEFRONT, flags: int = 0, rank: int = 0, world: int = 1):
        """RenderKernel::render() on host buffers. Returns (framebuffer, stats)."""
        if framebuffer is None:
            framebuffer = Image(w, h).pixels
            flags |= B.FLAG_FB_IS_ZERO if world == 1 else 0
        assert framebuffer.dtype == np.float32 and framebuffer.shape == (h, w, 4) and framebuffer.flags["C_CONTIGUOUS"]
        st = B.Stats()
        o = self._opts(integrator, flags, rank, world)
        B.check(B.load_library().b200rt_render(self._h, B.fptr(camera.as_array17()), w, h, spp, max_bounces,
                                               B.fptr(framebuffer), C.byref(o), C.byref(st)))
        return framebuffer, st.as_dict()

    def render_rgba8(self, camera: Camera, w: int, h: int, spp: int, max_bounces: int, framebuffer: np.ndarray | None = None,
                     flip_y: bool = True, out: np.ndarray | None = None, integrator: int = B.INTEGRATOR_WAVEFRONT, flags: int = 0):
        """render() + write_image_png's quantisation on the device: returns ((h, w, 4) uint8, stats)."""
        if out is None:
            out = np.empty((h, w, 4), np.uint8)
        assert out.dtype == np.uint8 and out.shape == (h, w, 4) and out.flags["C_CONTIGUOUS"]
        if framebuffer is not None:
            assert framebuffer.dtype == np.float32 and framebuffer.shape == (h, w, 4) and framebuffer.flags["C_CONTIGUOUS"]
        st = B.Stats()
        o = self._opts(integrator, flags, 0, 1)
        B.check(B.load_library().b200rt_render_rgba8(self._h, B.fptr(camera.as_array17()), w, h, spp, max_bounces, B.fptr(framebuffer),
                                                     1 if flip_y else 0, out.ctypes.data_as(C.POINTER(C.c_ubyte)), C.byref(o), C.byref(st)))
        return out, st.as_dict()

    def render_region(self, camera: Camera, w: int, h: int, spp: int, max_bounces: int, x0: int, y0: int, x1: int, y1: int, flags: int = 0):
        """ray_trace_pixel(x, y) for every pixel of [x0, x1) x [y0, y1) of the w x h frame (b200rt_render_region)."""
        out = np.empty((y1 - y0, x1 - x0, 4), np.float32)
        st = B.Stats()
        o = self._opts(B.INTEGRATOR_MEGAKERNEL, flags, 0, 1)
        B.check(B.load_library().b200rt_render_region(self._h, B.fptr(camera.as_array17()), w, h, spp, max_bounces, x0, y0, x1, y1,
                                                      B.fptr(out), C.byref(o), C.byref(st)))
        return out, st.as_dict()

    def ray_trace_pixel(self, camera: Camera, w: int, h: int, spp: int, max_bounces: int, x: int, y: int):
        """RenderKernel::ray_trace_pixel(x, y) on a black framebuffer: the pixel's RGBA."""
        return self.render_region(camera, w, h, spp, max_bounces, x, y, x + 1, y + 1)[0][0, 0]

    def trace_primary(self, camera: Camera, w: int, h: int, sample: int = -1, spp_for_seed: int = 1, flags: int = 0,
                      rank: int = 0, world: int = 1):
        prim = np.zeros((h, w), np.int32)
        t = np.zeros((h, w), np.float32)
        st = B.Stats()
        o = self._opts(0, flags, rank, world)
        B.check(B.load_library().b200rt_trace_primary(self._h, B.fptr(camera.as_array17()), w, h, sample, spp_for_seed,
                                                      B.iptr(prim), B.fptr(t), C.byref(o), C.byref(st)))
        return prim, t, st.as_dict()

    def trace_primary_into(self, camera: Camera, w: int, h: int, prim: np.ndarray, t: np.ndarray, sample: int = -1, spp_for_seed: int = 1,
                           flags: int = 0):
        """trace_primary into caller-owned (e.g. page-locked) (h, w) int32 / float32 arrays; returns the stats."""
        assert prim.dtype == np.int32 and t.dtype == np.float32 and prim.shape == (h, w) and t.shape == (h, w)
        st = B.Stats()
        o = self._opts(0, flags, 0, 1)
        B.check(B.load_library().b200rt_trace_primary(self._h, B.fptr(camera.as_array17()), w, h, sample, spp_for_seed,
                                                      B.iptr(prim), B.fptr(t), C.byref(o), C.byref(st)))
        return st.as_dict()

    def render_aovs(self, camera: Camera, w: int, h: int, samples_per_axis: int = 2, flags: int = 0):
        """Feature buffers for a denoiser (b200rt_render_aovs): samples_per_axis^2 stratified camera rays per pixel; returns
        ((h, w, 3) mean albedo, (h, w, 3) mean geometric normal (not renormalised, 0 on misses), stats)."""
        albedo = np.empty((h, w, 3), np.float32)
        normal = np.empty((h, w, 3), np.float32)
        st = B.Stats()
        o = self._opts(0, flags, 0, 1)
        B.check(B.load_library().b200rt_render_aovs(self._h, B.fptr(camera.as_array17()), w, h, samples_per_axis, B.fptr(albedo),
                                                    B.fptr(normal), C.byref(o), C.byref(st)))
        return albedo, normal, st.as_dict()

    def trace_rays(self, rays6, any_hit: bool = False, flags: int = 0):
        rays6 = _f32(rays6).reshape(-1, 6)
        n = len(rays6)
        prim = np.zeros(n, np.int32)
        t = np.zeros(n, np.float32)
        extra = np.zeros((n, 8), np.float32)
        o = self._opts(0, flags)
        B.check(B.load_library().b200rt_trace_rays(self._h, B.fptr(rays6), n, 1 if any_hit else 0, B.iptr(prim), B.fptr(t),
                                                   B.fptr(extra), C.byref(o)))
        return prim, t, extra

    # device-pointer variants (pointers are plain ints, e.g. torch.Tensor.data_ptr())
    def render_tiles_device(self, camera: Camera, w, h, spp, max_bounces, dev_tiles_ptr: int, stream_ptr: int = 0,
                            integrator: int = B.INTEGRATOR_WAVEFRONT, flags: int = 0, rank: int = 0, world: int = 1, want_stats: bool = False):
        st = B.Stats()
        o = self._opts(integrator, flags, rank, world)
        B.check(B.load_library().b200rt_render_tiles_device(self._h, B.fptr(camera.as_array17()), w, h, spp, max_bounces,
                                                            C.c_void_p(dev_tiles_ptr), C.byref(o), C.c_void_p(stream_ptr),
                                                            C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def untile_accumulate_device(self, dev_gathered_ptr: int, tiles_per_rank_padded: int, world: int, w: int, h: int, dev_fb_inout_ptr: int,
                                 stream_ptr: int = 0):
        B.check(B.load_library().b200rt_untile_accumulate_device(self._h, C.c_void_p(dev_gathered_ptr), tiles_per_rank_padded, world, w, h,
                                                                 C.c_void_p(dev_fb_inout_ptr), C.c_void_p(stream_ptr)))

    def untile_device(self, dev_gathered_ptr: int, tiles_per_rank_padded: int, world: int, w: int, h: int, dev_image_ptr: int,
                      stream_ptr: int = 0):
        B.check(B.load_library().b200rt_untile_device(self._h, C.c_void_p(dev_gathered_ptr), tiles_per_rank_padded, world, w, h,
                                                      C.c_void_p(dev_image_ptr), C.c_void_p(stream_ptr)))

    def trace_rays_device(self, dev_rays6_ptr: int, n: int, dev_prim_ptr: int, dev_t_ptr: int, dev_extra8_ptr: int = 0,
                          any_hit: bool = False, stream_ptr: int = 0, flags: int = 0, want_stats: bool = False):
        st = B.Stats()
        o = self._opts(0, flags)
        B.check(B.load_library().b200rt_trace_rays_device(self._h, C.c_void_p(dev_rays6_ptr), n, 1 if any_hit else 0,
                                                          C.c_void_p(dev_prim_ptr), C.c_void_p(dev_t_ptr),
                                                          C.c_void_p(dev_extra8_ptr) if dev_extra8_ptr else None, C.byref(o),
                                                          C.c_void_p(stream_ptr), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def trace_primary_device(self, camera: Camera, w, h, dev_prim_ptr: int, dev_t_ptr: int, sample: int = -1,
                             spp_for_seed: int = 1, stream_ptr: int = 0, flags: int = 0, rank: int = 0, world: int = 1,
                             want_stats: bool = False):
        st = B.Stats()
        o = self._opts(0, flags, rank, world)
        B.check(B.load_library().b200rt_trace_primary_device(self._h, B.fptr(camera.as_array17()), w, h, sample, spp_for_seed,
                                                             C.c_void_p(dev_prim_ptr), C.c_void_p(dev_t_ptr), C.byref(o),
                                                             C.c_void_p(stream_ptr), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def render_aovs_device(self, camera: Camera, w, h, dev_albedo_ptr: int, dev_normal_ptr: int, samples_per_axis: int = 2,
                           stream_ptr: int = 0, flags: int = 0, rank: int = 0, world: int = 1, want_stats: bool = False):
        """render_aovs into device buffers of w*h*3 floats (either pointer may be 0, not both)."""
        st = B.Stats()
        o = self._opts(0, flags, rank, world)
        B.check(B.load_library().b200rt_render_aovs_device(self._h, B.fptr(camera.as_array17()), w, h, samples_per_axis,
                                                           C.c_void_p(dev_albedo_ptr) if dev_albedo_ptr else None,
                                                           C.c_void_p(dev_normal_ptr) if dev_normal_ptr else None, C.byref(o),
                                                           C.c_void_p(stream_ptr), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None


class Accumulator:
    """Progressive rendering (b200rt_accum_*): the samples of a frame streamed in chunks, each pixel's RNG stream continued across
    chunks; after spp_total samples resolve() equals Scene.render(spp_total) bit for bit. On a Scene(devices=...) every device keeps
    and renders the pixels of its own tiles, and a resolve gathers them on the first device."""

    def __init__(self, scene: Scene, camera: Camera, w: int, h: int, spp_total: int, max_bounces: int):
        self.scene, self.w, self.h = scene, w, h
        hnd = C.c_void_p()
        B.check(B.load_library().b200rt_accum_create(scene._h, B.fptr(camera.as_array17()), w, h, spp_total, max_bounces, C.byref(hnd)))
        self._h = hnd

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                B.load_library().b200rt_accum_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def add(self, n_samples: int, integrator: int = B.INTEGRATOR_WAVEFRONT, flags: int = 0) -> dict:
        st = B.Stats()
        o = B.RenderOptions(integrator, flags, 0, 1)
        B.check(B.load_library().b200rt_accum_add(self._h, n_samples, C.byref(o), C.byref(st)))
        return st.as_dict()

    def samples(self) -> int:
        return int(B.load_library().b200rt_accum_samples(self._h))

    def resolve(self, framebuffer_in: np.ndarray | None = None) -> np.ndarray:
        out = np.empty((self.h, self.w, 4), np.float32)
        B.check(B.load_library().b200rt_accum_resolve(self._h, B.fptr(framebuffer_in), B.fptr(out)))
        return out

    def resolve_rgba8(self, framebuffer_in: np.ndarray | None = None, flip_y: bool = True) -> np.ndarray:
        """resolve() quantised on the device as write_image_png would (b200rt_accum_resolve_rgba8): (h, w, 4) uint8, 4 B/pixel over
        PCIe instead of 16."""
        if framebuffer_in is not None:
            assert framebuffer_in.dtype == np.float32 and framebuffer_in.shape == (self.h, self.w, 4) and framebuffer_in.flags["C_CONTIGUOUS"]
        out = np.empty((self.h, self.w, 4), np.uint8)
        B.check(B.load_library().b200rt_accum_resolve_rgba8(self._h, B.fptr(framebuffer_in), 1 if flip_y else 0,
                                                            out.ctypes.data_as(C.POINTER(C.c_ubyte))))
        return out


# ---- RenderKernel (render_kernel.h:21-96) ----------------------------------------------------------------------------------------
class RenderKernel:
    """Same 13-argument constructor, set_camera() and render() as the reference's RenderKernel. Buffers are borrowed
    (the reference stores references, render_kernel.h:81-93); the device scene is created on the first render()."""

    def __init__(self, width, height, render_samples, max_bounces, image_buffer: Image, triangle_buffer, materials_buffer,
                 emissive_triangle_indices, materials_indices, analytic_spheres=None, bvh: BVH | None = None,
                 skysphere: Image | None = None, env_map_cdf=None, integrator: int = B.INTEGRATOR_WAVEFRONT, flags: int = 0, devices=None):
        self.m_width, self.m_height = int(width), int(height)
        self.m_render_samples, self.m_max_bounces = int(render_samples), int(max_bounces)
        self.m_frame_buffer = image_buffer
        self._args = (triangle_buffer, materials_indices, materials_buffer, emissive_triangle_indices, analytic_spheres, skysphere,
                      env_map_cdf, bvh)
        self.m_camera = Camera()
        self.integrator, self.flags, self.devices = integrator, flags, devices
        self._scene = None
        self.last_stats = None

    def set_camera(self, camera: Camera):
        self.m_camera = camera

    def scene(self) -> Scene:
        if self._scene is None:
            tri, mi, mats, em, sph, sky, cdf, bvh = self._args
            self._scene = Scene(tri, mi, mats, em, spheres=sph, skysphere=sky, env_map_cdf=cdf, bvh=bvh, devices=self.devices)
        return self._scene

    def ray_trace_pixel(self, x: int, y: int):
        """render_kernel.h:56 / the DEBUG_PIXEL mode (render_kernel.cpp:186-197): renders one pixel into the framebuffer in place."""
        px = self.scene().ray_trace_pixel(self.m_camera, self.m_width, self.m_height, self.m_render_samples, self.m_max_bounces, x, y)
        self.m_frame_buffer.pixels[y, x] = px
        return px

    def render(self):
        # the reference iterates the framebuffer's own size (render_kernel.cpp:199-201)
        fb = self.m_frame_buffer.pixels
        assert fb.shape == (self.m_height, self.m_width, 4), "framebuffer size must match width x height"
        _, self.last_stats = self.scene().render(self.m_camera, self.m_width, self.m_height, self.m_render_samples,
                                                 self.m_max_bounces, framebuffer=fb, integrator=self.integrator, flags=self.flags)
