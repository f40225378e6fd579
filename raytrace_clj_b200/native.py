"""Marshaller + ctypes binding of libraytrace_b200.so (the C ABI in include/raytrace_b200.h).

This is the Python stand-in for the JVM-side ``native.clj`` a maintainer would add to the
reference (INTEGRATION.md): walk ``world`` (bvh-node tree, hitable.clj:97-123) to its leaves,
de-duplicate by identity (a 1-element node stores the same object twice, hitable.clj:113-114),
and emit structure-of-arrays float32 buffers; any record outside the accelerated path is
rejected — there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

from . import camera as cam
from . import hitable as hit
from . import perlin
from . import shader as shad
from . import texture as tex

RT_SPHERE_UV, RT_SPHERE_MOVING = 1, 2
RT_MAT_LAMBERTIAN, RT_MAT_METAL, RT_MAT_DIELECTRIC, RT_MAT_DIFFUSE_LIGHT, RT_MAT_ISOTROPIC = 0, 1, 2, 3, 4
RT_TEX_CONSTANT, RT_TEX_UV_GRADIENT, RT_TEX_CHECKERBOARD = 0, 1, 2
RT_TEX_PERLIN_NOISE, RT_TEX_PERLIN_TURB, RT_TEX_MARBLE, RT_TEX_FLIP_U, RT_TEX_FLIP_V, RT_TEX_IMAGE_MAP = 3, 4, 5, 6, 7, 8
RT_PRIM_SPHERE, RT_PRIM_RECT_XY, RT_PRIM_RECT_XZ, RT_PRIM_RECT_YZ, RT_PRIM_TRIANGLE, RT_PRIM_MEDIUM = 0, 1, 2, 3, 4, 5
RT_XOP_NONE, RT_XOP_TRANSLATE, RT_XOP_ROTATE_Y, RT_XOP_FLIP = 0, 1, 2, 3
RT_XFORM_MAX_OPS = 4
RT_TIE_HITLIST, RT_TIE_BVH = 0, 1
RT_ACCEL_BRUTE_FORCE, RT_ACCEL_BVH = 0, 1
RT_CAM_PINHOLE, RT_CAM_THIN_LENS = 0, 1
RT_VARIANT_MEGAKERNEL, RT_VARIANT_WAVEFRONT = 0, 1
RT_TERM_LIGHT, RT_TERM_ABSORB, RT_TERM_DEPTH, RT_TERM_MISS = 1, 2, 3, 4
RT_CTR_COUNT = 24
COUNTER_NAMES = ["rays", "sphere_tests", "samples", "term_light", "term_absorb", "term_depth", "term_miss",
                 "kernel_ns", "candidates", "kernel_launches", "cull_ns", "refine_ns", "tiebreak_ns", "shade_ns",
                 "direct_tests", "bvh_node_tests", "reduce_ns", "common_origin_rays"]

# one logged bounce of rt_trace_paths (struct rt_path_bounce, 40 bytes)
PATH_BOUNCE_DTYPE = np.dtype([("o", np.float32, 3), ("time", np.float32), ("d", np.float32, 3), ("hit_id", np.int32),
                              ("t", np.float64)])
assert PATH_BOUNCE_DTYPE.itemsize == 40


class UnsupportedSceneError(ValueError):
    """A record type outside the accelerated hot path (RT_ERR_UNSUPPORTED on the JVM side)."""


class NativeError(RuntimeError):
    pass


@dataclass
class FlatScene:
    """The marshalled scene: exactly the buffers of ``rt_scene_desc`` (+ ``rt_scene_ext`` when anything beyond
    spheres / the three basic textures is present).  Per-primitive arrays hold the ``n_spheres`` world primitives
    in flatten order, then ``n_boundary`` boundary primitives of media."""
    center0_r: np.ndarray      # [n,4] f32
    center1: np.ndarray        # [n,4] f32
    t0t1: np.ndarray           # [n,2] f32
    sphere_flags: np.ndarray   # [n]   u32
    material_id: np.ndarray    # [n]   i32
    mat_type: np.ndarray       # [m]   i32
    mat_param: np.ndarray      # [m]   f32
    mat_tex: np.ndarray        # [m]   i32
    tex_type: np.ndarray       # [t]   i32
    tex_params: np.ndarray     # [t,12] f32
    tex_children: np.ndarray   # [t,2] i32
    # ---- rt_scene_ext (None / 0 => plain sphere scene, rt_set_scene) ----
    n_boundary: int = 0
    prim_type: np.ndarray | None = None      # [n]    i32 RT_PRIM_*
    prim_params: np.ndarray | None = None    # [n,12] f32
    prim_aux: np.ndarray | None = None       # [n,2]  i32
    prim_xform: np.ndarray | None = None     # [n]    i32
    xform_ops: np.ndarray | None = None      # [x,4]  i32
    xform_params: np.ndarray | None = None   # [x,4,4] f32
    tie_rule: int = RT_TIE_HITLIST
    perlin_vectors: np.ndarray | None = None  # [256,3] f32
    perlin_perm: np.ndarray | None = None     # [3,256] i32
    image_wh: np.ndarray | None = None        # [k,2] i32
    image_offset: np.ndarray | None = None    # [k]   i64
    image_rgb: np.ndarray | None = None       # bytes

    @property
    def n_spheres(self):
        """World primitives (the name is the C struct's field: spheres only in ABI v1)."""
        return int(self.center0_r.shape[0]) - int(self.n_boundary)

    @property
    def has_ext(self):
        return self.prim_type is not None or self.tie_rule != RT_TIE_HITLIST or self.perlin_vectors is not None \
            or self.image_wh is not None

    @property
    def generic(self):
        """Mirror of the library's `generic` flag (rt_set_scene_ex): some leaf is not a plain sphere, or a wrapper, an extended
        texture (Perlin / image / flip) or an Isotropic material is in use — such scenes run the GEN kernels and the FP32 cull."""
        g = self.perlin_vectors is not None
        if self.prim_type is not None:
            g = g or bool((np.asarray(self.prim_type)[: self.n_spheres] != RT_PRIM_SPHERE).any())
        if self.prim_xform is not None:
            g = g or bool((np.asarray(self.prim_xform) >= 0).any())
        g = g or bool((np.asarray(self.tex_type) > RT_TEX_CHECKERBOARD).any()) or bool((np.asarray(self.mat_type) == RT_MAT_ISOTROPIC).any())
        return g

    def copy(self):
        return FlatScene(**{k: (getattr(self, k).copy() if isinstance(getattr(self, k), np.ndarray) else getattr(self, k))
                            for k in self.__dataclass_fields__})

    def nbytes(self):
        return int(sum(getattr(self, k).nbytes for k in self.__dataclass_fields__ if isinstance(getattr(self, k), np.ndarray)))

    def sphere_tensors(self, device):
        """The five per-primitive arrays as torch CUDA tensors on `device`, in the dtypes and shapes
        ``Renderer.set_scene_device`` takes (sphere_flags as int32: the same bits)."""
        import torch
        c = np.ascontiguousarray
        return dict(center0_r=torch.from_numpy(c(self.center0_r, np.float32)).to(device),
                    center1=torch.from_numpy(c(self.center1, np.float32)).to(device),
                    t0t1=torch.from_numpy(c(self.t0t1, np.float32)).to(device),
                    sphere_flags=torch.from_numpy(c(self.sphere_flags, np.uint32).view(np.int32)).to(device),
                    material_id=torch.from_numpy(c(self.material_id, np.int32)).to(device))

    def tables(self):
        """The material and texture tables (host arrays), as ``Renderer.set_scene_device`` takes them."""
        return dict(mat_type=self.mat_type, mat_param=self.mat_param, mat_tex=self.mat_tex, tex_type=self.tex_type,
                    tex_params=self.tex_params, tex_children=self.tex_children)


_LEAF_TYPES = (hit.Sphere, hit.MovingSphere, hit.RectXY, hit.RectXZ, hit.RectYZ, hit.Triangle, hit.ConstantMedium)


def flatten_world(world, with_ops=False):
    """Leaves of the container tree, left to right.  A 1-element bvh-node stores the same object as both
    children (hitable.clj:113-114): it is visited once.  Wrappers (FlipNormals / Translate / RotateY,
    hitable.clj:375-486) are folded into a per-leaf op chain, outermost first; a Box (hitable.clj:491-511)
    contributes its six rectangles.  with_ops: return (leaf, ops) pairs instead of the bare leaves."""
    out, seen = [], set()

    def walk(h, ops):
        if isinstance(h, hit.BvhNode):
            walk(h.left, ops)
            if h.right is not h.left:
                walk(h.right, ops)
        elif isinstance(h, hit.Hitlist):
            for it in h.items:
                walk(it, ops)
        elif isinstance(h, hit.Box):
            walk(h.sides, ops)
        elif isinstance(h, hit.FlipNormals):
            walk(h.item, ops + ((RT_XOP_FLIP, (0.0, 0.0, 0.0, 0.0)),))
        elif isinstance(h, hit.Translate):
            o = h.offset
            walk(h.item, ops + ((RT_XOP_TRANSLATE, (float(o[0]), float(o[1]), float(o[2]), 0.0)),))
        elif isinstance(h, hit.RotateY):
            walk(h.obj, ops + ((RT_XOP_ROTATE_Y, (float(h.sin_theta), float(h.cos_theta), 0.0, 0.0)),))
        elif isinstance(h, _LEAF_TYPES):
            key = (id(h), ops)
            if key not in seen:
                seen.add(key)
                out.append((h, ops))
        else:
            raise UnsupportedSceneError(f"{type(h).__name__} is outside the accelerated path; no CPU fallback")

    # iterative-safe for deep trees
    import sys
    old = sys.getrecursionlimit()
    sys.setrecursionlimit(max(old, 10000))
    try:
        walk(world, ())
    finally:
        sys.setrecursionlimit(old)
    return out if with_ops else [h for h, _ in out]


def marshal_world(world, perlin_tables=None) -> FlatScene:
    leaves = flatten_world(world, with_ops=True)
    if len(leaves) == 0:
        raise UnsupportedSceneError("empty world")
    mats, mat_index = [], {}
    texs, tex_index = [], {}
    images = []
    xforms, xform_index = [], {}
    uses = {"perlin": False, "ext": False}

    def add_tex(t):
        if id(t) in tex_index:
            return tex_index[id(t)]
        p = np.zeros(12, np.float32)
        ch = [-1, -1]
        if isinstance(t, tex.Constant):
            ty = RT_TEX_CONSTANT
            p[0:3] = t.color
        elif isinstance(t, tex.UVGradient):
            ty = RT_TEX_UV_GRADIENT
            p[0:3], p[3:6], p[6:9], p[9:12] = t.co, t.cu, t.cv, t.cuv
        elif isinstance(t, tex.Checkerboard):
            ty = RT_TEX_CHECKERBOARD
            p[0] = t.scale
            ch = [add_tex(t.tex0), add_tex(t.tex1)]
        elif isinstance(t, tex.PerlinNoise):
            ty, p[0] = RT_TEX_PERLIN_NOISE, t.scale
            uses["perlin"] = True
        elif isinstance(t, tex.PerlinTurbulence):
            ty, p[0], p[1] = RT_TEX_PERLIN_TURB, t.scale, t.depth
            uses["perlin"] = True
        elif isinstance(t, tex.Marble):
            ty, p[0], p[1] = RT_TEX_MARBLE, t.scale, t.depth
            uses["perlin"] = True
        elif isinstance(t, (tex.FlipTextureU, tex.FlipTextureV)):
            ty = RT_TEX_FLIP_U if isinstance(t, tex.FlipTextureU) else RT_TEX_FLIP_V
            ch = [add_tex(t.tex), -1]
        elif isinstance(t, tex.ImageMap):
            ty, p[0] = RT_TEX_IMAGE_MAP, len(images)
            images.append(np.ascontiguousarray(t.image, np.uint8))
        else:
            raise UnsupportedSceneError(f"texture {type(t).__name__} is outside the accelerated path")
        if ty > RT_TEX_CHECKERBOARD:
            uses["ext"] = True
        tex_index[id(t)] = len(texs)
        texs.append((ty, p, ch))
        return tex_index[id(t)]

    def add_mat(m):
        if id(m) in mat_index:
            return mat_index[id(m)]
        if isinstance(m, shad.Lambertian):
            rec = (RT_MAT_LAMBERTIAN, 0.0, add_tex(m.albedo))
        elif isinstance(m, shad.Metal):
            rec = (RT_MAT_METAL, m.fuzz, add_tex(m.albedo))
        elif isinstance(m, shad.Dielectric):
            rec = (RT_MAT_DIELECTRIC, m.ri, -1)
        elif isinstance(m, shad.DiffuseLight):
            rec = (RT_MAT_DIFFUSE_LIGHT, 0.0, add_tex(m.tex))
        elif isinstance(m, shad.Isotropic):
            rec = (RT_MAT_ISOTROPIC, 0.0, add_tex(m.albedo))
            uses["ext"] = True
        else:
            raise UnsupportedSceneError(f"material {type(m).__name__} is outside the accelerated path")
        mat_index[id(m)] = len(mats)
        mats.append(rec)
        return mat_index[id(m)]

    def add_xform(ops):
        if not ops:
            return -1
        if len(ops) > RT_XFORM_MAX_OPS:
            raise UnsupportedSceneError(f"more than {RT_XFORM_MAX_OPS} nested wrappers around one leaf")
        if ops not in xform_index:
            xform_index[ops] = len(xforms)
            xforms.append(ops)
        uses["ext"] = True
        return xform_index[ops]

    rows = []          # world primitives
    boundary = []      # boundary primitives of media (appended after the world)

    def prim_row(s, ops, material=True):
        r = dict(c0r=np.zeros(4, np.float32), c1=np.zeros(4, np.float32), tt=np.array([0, 1], np.float32), flags=0,
                 type=RT_PRIM_SPHERE, q=np.zeros(12, np.float32), aux=[0, 0], xform=add_xform(ops),
                 mat=add_mat(s.material) if material else 0)
        if isinstance(s, hit.MovingSphere):
            r["c0r"][:3], r["c0r"][3] = s.center0, s.radius
            r["c1"][:3] = s.center1
            r["tt"][:] = (s.t0, s.t1)
            r["flags"] = RT_SPHERE_MOVING
        elif isinstance(s, hit.Sphere):
            r["c0r"][:3], r["c0r"][3] = s.center, s.radius
            r["c1"][:3] = s.center
            r["flags"] = RT_SPHERE_UV if isinstance(s, hit.UVSphere) else 0
        elif isinstance(s, hit.RectXY):
            r["type"], r["q"][:5] = RT_PRIM_RECT_XY, (s.x0, s.y0, s.x1, s.y1, s.k)
        elif isinstance(s, hit.RectXZ):
            r["type"], r["q"][:5] = RT_PRIM_RECT_XZ, (s.x0, s.z0, s.x1, s.z1, s.k)
        elif isinstance(s, hit.RectYZ):
            r["type"], r["q"][:5] = RT_PRIM_RECT_YZ, (s.y0, s.z0, s.y1, s.z1, s.k)
        elif isinstance(s, hit.Triangle):
            r["type"] = RT_PRIM_TRIANGLE
            r["q"][0:3], r["q"][3:6], r["q"][6:9] = s.v0, s.v1, s.v2
        else:
            raise UnsupportedSceneError(f"{type(s).__name__} cannot bound a medium / be a leaf here")
        if r["type"] != RT_PRIM_SPHERE:
            uses["ext"] = True
        return r

    pending_media = []
    for s, ops in leaves:
        if isinstance(s, hit.ConstantMedium):
            r = dict(c0r=np.zeros(4, np.float32), c1=np.zeros(4, np.float32), tt=np.array([0, 1], np.float32), flags=0,
                     type=RT_PRIM_MEDIUM, q=np.zeros(12, np.float32), aux=[0, 0], xform=add_xform(ops),
                     mat=add_mat(s.phase_fn))
            r["q"][0] = s.density
            uses["ext"] = True
            pending_media.append((r, s.boundary))
            rows.append(r)
        else:
            rows.append(prim_row(s, ops))
    n_world = len(rows)
    for r, bnd in pending_media:
        bl = flatten_world(bnd, with_ops=True)
        if any(isinstance(b, hit.ConstantMedium) for b, _ in bl):
            raise UnsupportedSceneError("a medium cannot bound a medium")
        r["aux"] = [n_world + len(boundary), len(bl)]
        boundary.extend(prim_row(b, bops, material=False) for b, bops in bl)
    allrows = rows + boundary
    tie = RT_TIE_BVH if isinstance(world, hit.BvhNode) else RT_TIE_HITLIST

    fs = FlatScene(
        np.stack([r["c0r"] for r in allrows]), np.stack([r["c1"] for r in allrows]), np.stack([r["tt"] for r in allrows]),
        np.array([r["flags"] for r in allrows], np.uint32), np.array([r["mat"] for r in allrows], np.int32),
        np.array([m[0] for m in mats], np.int32), np.array([m[1] for m in mats], np.float32),
        np.array([m[2] for m in mats], np.int32),
        np.array([t[0] for t in texs], np.int32).reshape(-1),
        np.array([t[1] for t in texs], np.float32).reshape(-1, 12),
        np.array([t[2] for t in texs], np.int32).reshape(-1, 2),
    )
    fs.tie_rule = tie
    if uses["ext"] or uses["perlin"] or images:
        fs.n_boundary = len(boundary)
        fs.prim_type = np.array([r["type"] for r in allrows], np.int32)
        fs.prim_params = np.stack([r["q"] for r in allrows]).astype(np.float32)
        fs.prim_aux = np.array([r["aux"] for r in allrows], np.int32).reshape(-1, 2)
        fs.prim_xform = np.array([r["xform"] for r in allrows], np.int32)
        xo = np.zeros((max(1, len(xforms)), RT_XFORM_MAX_OPS), np.int32)
        xp = np.zeros((max(1, len(xforms)), RT_XFORM_MAX_OPS, 4), np.float32)
        for i, ops in enumerate(xforms):
            for k, (ty, prm) in enumerate(ops):
                xo[i, k] = ty
                xp[i, k] = prm
        fs.xform_ops, fs.xform_params = xo[:len(xforms)], xp[:len(xforms)]
        if uses["perlin"]:
            tb = perlin_tables or perlin.TABLES
            fs.perlin_vectors = np.ascontiguousarray(tb.vectors, np.float32)
            fs.perlin_perm = np.ascontiguousarray(tb.perm, np.int32)
        if images:
            fs.image_wh = np.array([[im.shape[1], im.shape[0]] for im in images], np.int32)
            offs = np.cumsum([0] + [im.size for im in images])
            fs.image_offset = np.array(offs[:-1], np.int64)
            fs.image_rgb = np.concatenate([im.reshape(-1) for im in images]).astype(np.uint8)
    return fs


def marshal_camera(camera):
    """(cam_type, float32[24]) from a camera record (camera.clj:8,35)."""
    out = np.zeros(24, np.float32)
    if isinstance(camera, cam.ThinLensCamera):
        for k, v in enumerate([camera.origin, camera.lleft, camera.horiz, camera.vert, camera.u, camera.v, camera.w]):
            out[3 * k:3 * k + 3] = v
        out[21], out[22], out[23] = camera.aperture, camera.t0, camera.t1
        return RT_CAM_THIN_LENS, out
    if isinstance(camera, cam.PinholeCamera):
        for k, v in enumerate([camera.origin, camera.lleft, camera.horiz, camera.vert]):
            out[3 * k:3 * k + 3] = v
        return RT_CAM_PINHOLE, out
    raise UnsupportedSceneError(f"camera {type(camera).__name__} is not supported")


def marshal_views(cameras):
    """(cam_types int32[K], cams float32[K, 24]) for rt_render_views from a list of cameras: camera records
    (camera.clj:8,35) or ``marshal_camera`` results ``(cam_type, float[24])``.  Pure host code: it checks the list's
    shape and types and leaves the camera types themselves to the library, as ``rt_set_camera`` does."""
    if isinstance(cameras, (str, bytes)) or not hasattr(cameras, "__len__"):
        raise TypeError("cameras must be a list of cameras or of (cam_type, float[24]) pairs")
    if len(cameras) == 0:
        raise ValueError("cameras is empty: a batch renders at least one view")
    types = np.empty(len(cameras), np.int32)
    cams = np.empty((len(cameras), 24), np.float32)
    for v, c in enumerate(cameras):
        if isinstance(c, (cam.ThinLensCamera, cam.PinholeCamera)):
            c = marshal_camera(c)
        if not (isinstance(c, tuple) and len(c) == 2):
            raise TypeError(f"view {v}: expected a camera or a (cam_type, float[24]) pair, got {type(c).__name__}")
        t, f = c
        if isinstance(t, (bool, np.bool_)) or not isinstance(t, (int, np.integer)):
            raise TypeError(f"view {v}: the camera type must be an integer, got {type(t).__name__}")
        f = np.asarray(f)
        if f.shape != (24,):
            raise ValueError(f"view {v}: a camera record has 24 floats, got shape {f.shape}")
        if not np.issubdtype(f.dtype, np.floating):
            raise TypeError(f"view {v}: a camera record holds floats, got {f.dtype}")
        types[v] = t
        cams[v] = f
    return types, cams


# ---------------------------------------------------------------------------------------------
# ctypes binding
# ---------------------------------------------------------------------------------------------

_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int32)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)
_u8p = C.POINTER(C.c_uint8)


class _SceneDesc(C.Structure):
    _fields_ = [
        ("n_spheres", C.c_int32), ("center0_r", _f32p), ("center1", _f32p), ("t0t1", _f32p),
        ("sphere_flags", _u32p), ("material_id", _i32p),
        ("n_materials", C.c_int32), ("mat_type", _i32p), ("mat_param", _f32p), ("mat_tex", _i32p),
        ("n_textures", C.c_int32), ("tex_type", _i32p), ("tex_params", _f32p), ("tex_children", _i32p),
    ]


class _SceneExt(C.Structure):
    _fields_ = [
        ("struct_bytes", C.c_int32), ("n_boundary", C.c_int32),
        ("prim_type", _i32p), ("prim_params", _f32p), ("prim_aux", _i32p), ("prim_xform", _i32p),
        ("n_xforms", C.c_int32), ("xform_ops", _i32p), ("xform_params", _f32p),
        ("tie_rule", C.c_int32), ("perlin_vectors", _f32p), ("perlin_perm", _i32p),
        ("n_images", C.c_int32), ("image_wh", _i32p), ("image_offset", C.POINTER(C.c_int64)), ("image_rgb", _u8p),
    ]


LIB_NAME = "libraytrace_b200.so"
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

# every symbol include/raytrace_b200.h declares
ABI_SYMBOLS = [
    "rt_create", "rt_destroy", "rt_last_error", "rt_abi_version", "rt_set_scene", "rt_set_camera", "rt_render",
    "rt_render_accumulate_device", "rt_resolve_device", "rt_trace_primary", "rt_generate_rays", "rt_shade_batch",
    "rt_measure_fp32_peak", "rt_get_counters", "rt_reset_counters", "rt_set_profile", "rt_device_info", "rt_cull_check",
    "rt_set_scene_ex", "rt_trace_paths", "rt_set_accel", "rt_set_option", "rt_sample_device", "rt_host_alloc", "rt_host_free",
    "rt_get_bvh", "rt_set_scene_device", "rt_get_scene_blob", "rt_render_views", "rt_render_views_accumulate_device",
    "rt_resolve_views_device",
]

_lib = None


def load_library():
    """Load the CUDA library; fails loudly if it was not built (there is no fallback path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(f"{LIB_PATH} not built — run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a); the render path has no CPU fallback")
    L = C.CDLL(LIB_PATH)
    L.rt_last_error.restype = C.c_char_p
    L.rt_last_error.argtypes = [C.c_void_p]
    L.rt_create.argtypes = [C.POINTER(C.c_void_p), _i32p, C.c_int]
    L.rt_destroy.argtypes = [C.c_void_p]
    L.rt_destroy.restype = None
    L.rt_set_scene.argtypes = [C.c_void_p, C.POINTER(_SceneDesc)]
    L.rt_set_scene_ex.argtypes = [C.c_void_p, C.POINTER(_SceneDesc), C.POINTER(_SceneExt)]
    L.rt_set_accel.argtypes = [C.c_void_p, C.c_int]
    L.rt_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int64]
    L.rt_trace_paths.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _i32p, _i32p, C.c_int, C.c_uint64, C.c_int,
                                 _f32p, _i32p, _i32p, C.c_int, C.c_void_p]
    L.rt_sample_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint64, _f32p]
    L.rt_set_camera.argtypes = [C.c_void_p, C.c_int, _f32p]
    L.rt_render.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int, _f32p, _u8p]
    L.rt_render_accumulate_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                              C.c_int, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    L.rt_resolve_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int]
    L.rt_trace_primary.argtypes = [C.c_void_p, C.c_int, _f32p, _f32p, _f32p, C.c_double, C.c_double, _f64p, _i32p]
    L.rt_cull_check.argtypes = [C.c_void_p, C.c_int, _f32p, _f32p, _f32p, C.c_double, C.c_double, _u64p]
    L.rt_generate_rays.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _i32p, _i32p, C.c_uint64, _f32p, _f32p,
                                   _f32p, _f32p]
    L.rt_reset_counters.argtypes = [C.c_void_p]
    L.rt_set_profile.argtypes = [C.c_void_p, C.c_int]
    L.rt_shade_batch.argtypes = [C.c_void_p, C.c_int, _f32p, _f32p, _f32p, _i32p, _f64p, _f32p, _f32p, _f32p, _f32p,
                                 _f32p, _f32p, _i32p]
    L.rt_measure_fp32_peak.argtypes = [C.c_void_p, _f64p, _f64p]
    L.rt_get_counters.argtypes = [C.c_void_p, _u64p]
    L.rt_device_info.argtypes = [C.c_void_p, _i32p, _i32p, C.c_char_p]
    L.rt_host_alloc.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.rt_host_free.argtypes = [C.c_void_p, C.c_void_p]
    L.rt_get_bvh.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_int64, C.POINTER(C.c_int64)]
    L.rt_set_scene_device.argtypes = [C.c_void_p, C.POINTER(_SceneDesc), C.c_void_p]
    L.rt_get_scene_blob.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.rt_render_views.argtypes = [C.c_void_p, C.c_int, _i32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64,
                                  C.c_int, _f32p, _u8p]
    L.rt_render_views_accumulate_device.argtypes = [C.c_void_p, C.c_int, _i32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int,
                                                    C.c_int, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    L.rt_resolve_views_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_int]
    _lib = L
    return L


def _p(a, ty):
    return a.ctypes.data_as(ty) if a is not None else None


class Renderer:
    """One ``rt_ctx``: the object the front end holds in place of the claypoole pool (core.clj:100)."""

    def __init__(self, device_ids=None):
        self.L = load_library()
        self.h = C.c_void_p()
        ids = np.asarray(device_ids if device_ids is not None else [0], np.int32)
        self.device_ids = [int(i) for i in ids]
        rc = self.L.rt_create(C.byref(self.h), _p(ids, _i32p), C.c_int(len(ids)))
        if rc != 0:
            msg = self.L.rt_last_error(None)
            raise NativeError(f"rt_create failed ({rc}): {msg.decode() if msg else '?'}")
        self.flat = None

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.L.rt_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, what):
        if rc != 0:
            msg = self.L.rt_last_error(self.h)
            raise NativeError(f"{what} failed ({rc}): {msg.decode() if msg else '?'}")

    def host_empty(self, shape, dtype):
        """rt_host_alloc: a numpy array over page-locked host memory (rt_render has the device write such a buffer directly).
        The memory is returned by rt_host_free when the array (and every view of it) is gone."""
        import weakref
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dtype.itemsize
        ptr = C.c_void_p()
        self._check(self.L.rt_host_alloc(self.h, C.c_size_t(max(nbytes, 1)), C.byref(ptr)), "rt_host_alloc")
        buf = (C.c_uint8 * max(nbytes, 1)).from_address(ptr.value)
        weakref.finalize(buf, self.L.rt_host_free, None, C.c_void_p(ptr.value))
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def set_scene(self, flat: FlatScene):
        """rt_set_scene / rt_set_scene_ex with the scene's host arrays (the C side marshals and uploads them on EVERY call).
        The ctypes descriptors of a FlatScene whose arrays already have the ABI's dtypes and layout (no converted copies) are
        kept, so that calling this once per frame costs the C call, not eleven numpy conversions; the descriptors point at the
        caller's own arrays, so values changed in place are seen by the next call."""
        self.flat = flat
        names = ("center0_r", "center1", "t0t1", "sphere_flags", "material_id", "mat_type", "mat_param", "mat_tex", "tex_type",
                 "tex_params", "tex_children", "prim_type", "prim_params", "prim_aux", "prim_xform", "xform_ops", "xform_params",
                 "perlin_vectors", "perlin_perm", "image_wh", "image_offset", "image_rgb")
        sig = (tuple(id(getattr(flat, a)) for a in names), int(flat.n_boundary), int(flat.tie_rule))
        cached = getattr(self, "_scene_desc", None)
        if cached is not None and cached[0] is flat and cached[1] == sig:
            _, _, _keep, d, x = cached
        else:
            c = np.ascontiguousarray
            k = dict(
                c0=c(flat.center0_r, np.float32), c1=c(flat.center1, np.float32), tt=c(flat.t0t1, np.float32),
                fl=c(flat.sphere_flags, np.uint32), mi=c(flat.material_id, np.int32), mt=c(flat.mat_type, np.int32),
                mp=c(flat.mat_param, np.float32), mx=c(flat.mat_tex, np.int32), tt2=c(flat.tex_type, np.int32),
                tp=c(flat.tex_params, np.float32), tc=c(flat.tex_children, np.int32))
            d = _SceneDesc(flat.n_spheres, _p(k["c0"], _f32p), _p(k["c1"], _f32p), _p(k["tt"], _f32p), _p(k["fl"], _u32p),
                           _p(k["mi"], _i32p), len(k["mt"]), _p(k["mt"], _i32p), _p(k["mp"], _f32p), _p(k["mx"], _i32p),
                           len(k["tt2"]), _p(k["tt2"], _i32p), _p(k["tp"], _f32p), _p(k["tc"], _i32p))
            x, e = None, {}
            if flat.has_ext:
                e = dict(pt=None if flat.prim_type is None else c(flat.prim_type, np.int32),
                         pp=None if flat.prim_params is None else c(flat.prim_params, np.float32),
                         pa=None if flat.prim_aux is None else c(flat.prim_aux, np.int32),
                         px=None if flat.prim_xform is None else c(flat.prim_xform, np.int32),
                         xo=None if flat.xform_ops is None else c(flat.xform_ops, np.int32),
                         xp=None if flat.xform_params is None else c(flat.xform_params, np.float32),
                         pv=None if flat.perlin_vectors is None else c(flat.perlin_vectors, np.float32),
                         pm=None if flat.perlin_perm is None else c(flat.perlin_perm, np.int32),
                         iw=None if flat.image_wh is None else c(flat.image_wh, np.int32),
                         io=None if flat.image_offset is None else c(flat.image_offset, np.int64),
                         ir=None if flat.image_rgb is None else c(flat.image_rgb, np.uint8))
                x = _SceneExt(C.sizeof(_SceneExt), int(flat.n_boundary), _p(e["pt"], _i32p), _p(e["pp"], _f32p), _p(e["pa"], _i32p),
                              _p(e["px"], _i32p), 0 if e["xo"] is None else len(e["xo"]), _p(e["xo"], _i32p), _p(e["xp"], _f32p),
                              int(flat.tie_rule), _p(e["pv"], _f32p), _p(e["pm"], _i32p),
                              0 if e["iw"] is None else len(e["iw"]), _p(e["iw"], _i32p), _p(e["io"], C.POINTER(C.c_int64)),
                              _p(e["ir"], _u8p))
            src = {"c0": "center0_r", "c1": "center1", "tt": "t0t1", "fl": "sphere_flags", "mi": "material_id", "mt": "mat_type",
                   "mp": "mat_param", "mx": "mat_tex", "tt2": "tex_type", "tp": "tex_params", "tc": "tex_children", "pt": "prim_type",
                   "pp": "prim_params", "pa": "prim_aux", "px": "prim_xform", "xo": "xform_ops", "xp": "xform_params",
                   "pv": "perlin_vectors", "pm": "perlin_perm", "iw": "image_wh", "io": "image_offset", "ir": "image_rgb"}
            held = {**k, **e}
            no_copies = all(v is None or v is getattr(flat, src[key]) for key, v in held.items())
            self._scene_desc = (flat, sig, held, d, x) if no_copies else None
        if x is None:
            self._check(self.L.rt_set_scene(self.h, C.byref(d)), "rt_set_scene")
        else:
            self._check(self.L.rt_set_scene_ex(self.h, C.byref(d), C.byref(x)), "rt_set_scene_ex")

    def set_scene_device(self, center0_r, material_id, mat_type, mat_param, mat_tex, tex_type, tex_params, tex_children,
                         center1=None, t0t1=None, sphere_flags=None, stream=None):
        """rt_set_scene_device: the per-primitive arrays are torch CUDA tensors on the context's first device (center0_r /
        center1 [n,4] float32, t0t1 [n,2] float32, sphere_flags [n] int32 or uint32, material_id [n] int32, contiguous); the
        tables are host arrays.  The GPU builds the scene blob rt_set_scene would upload for the same values.  The library
        reads the tensors after the work already queued on `stream` (default: torch's current stream) and returns once the
        scene is built, so they may be changed right after.  Sphere scenes of rt_set_scene only (no rt_scene_ext): exact ties
        go to the first sphere in caller order (RT_TIE_HITLIST), also for arrays marshalled from a bvh-node world, whose
        FlatScene carries RT_TIE_BVH for rt_set_scene_ex."""
        import torch
        dev = torch.device("cuda", self.device_ids[0])
        n = center0_r.shape[0] if isinstance(center0_r, torch.Tensor) and center0_r.dim() == 2 else None

        def check(name, t, dtypes, cols):
            if t is None:
                return None
            if not isinstance(t, torch.Tensor) or t.device != dev:
                raise ValueError(f"{name} must be a torch tensor on {dev}")
            if t.dtype not in dtypes:
                raise ValueError(f"{name} must be {' or '.join(str(d) for d in dtypes)}, not {t.dtype}")
            shape = (n,) if cols is None else (n, cols)
            if tuple(t.shape) != shape:
                raise ValueError(f"{name} must have shape {shape}, not {tuple(t.shape)}")
            if not t.is_contiguous():
                raise ValueError(f"{name} must be contiguous")
            return C.c_void_p(t.data_ptr())

        if n is None or n == 0:
            raise ValueError("center0_r must be a [n,4] tensor with n >= 1")
        ptr = dict(c0=check("center0_r", center0_r, (torch.float32,), 4), c1=check("center1", center1, (torch.float32,), 4),
                   tt=check("t0t1", t0t1, (torch.float32,), 2),
                   fl=check("sphere_flags", sphere_flags, (torch.int32, getattr(torch, "uint32", torch.int32)), None),
                   mi=check("material_id", material_id, (torch.int32,), None))
        c = np.ascontiguousarray
        k = dict(mt=c(mat_type, np.int32), mp=c(mat_param, np.float32), mx=c(mat_tex, np.int32), tt2=c(tex_type, np.int32),
                 tp=c(tex_params, np.float32), tc=c(tex_children, np.int32))
        cast = lambda p, ty: C.cast(p, ty) if p is not None else None
        d = _SceneDesc(n, cast(ptr["c0"], _f32p), cast(ptr["c1"], _f32p), cast(ptr["tt"], _f32p), cast(ptr["fl"], _u32p),
                       cast(ptr["mi"], _i32p), len(k["mt"]), _p(k["mt"], _i32p), _p(k["mp"], _f32p), _p(k["mx"], _i32p),
                       len(k["tt2"]), _p(k["tt2"], _i32p), _p(k["tp"], _f32p), _p(k["tc"], _i32p))
        if stream is None:
            stream = torch.cuda.current_stream(dev).cuda_stream
        self.flat = None
        self._check(self.L.rt_set_scene_device(self.h, C.byref(d), C.c_void_p(int(stream) or None)), "rt_set_scene_device")

    def scene_blob(self, device_index=0):
        """rt_get_scene_blob: the scene blob one device of the context holds, as uint8 (diagnostic)."""
        nbytes = C.c_size_t(0)
        self._check(self.L.rt_get_scene_blob(self.h, int(device_index), None, 0, C.byref(nbytes)), "rt_get_scene_blob")
        out = np.zeros(nbytes.value, np.uint8)
        self._check(self.L.rt_get_scene_blob(self.h, int(device_index), out.ctypes.data_as(C.c_void_p), nbytes, C.byref(nbytes)),
                    "rt_get_scene_blob")
        return out

    def set_accel(self, accel):
        """RT_ACCEL_BRUTE_FORCE (the roofline path) or RT_ACCEL_BVH (flattened GPU BVH, hitable.clj:97-123's role)."""
        self._check(self.L.rt_set_accel(self.h, int(accel)), "rt_set_accel")

    def bvh(self, device_index=0):
        """rt_get_bvh: the RT_ACCEL_BVH tree of one device of the context (built first if it is out of date).  Returns
        (nodes [count, 16] f32 — words 12..15 hold int32 (left, right, 0, 0), a leaf child k as ~k — and
        {"nodes", "depth", "builder" ("host" | "device"), "build_ns"})."""
        info = np.zeros(4, np.int64)
        ip = info.ctypes.data_as(C.POINTER(C.c_int64))
        self._check(self.L.rt_get_bvh(self.h, int(device_index), None, 0, ip), "rt_get_bvh")
        nodes = np.zeros((int(info[0]), 16), np.float32)
        self._check(self.L.rt_get_bvh(self.h, int(device_index), _p(nodes, _f32p), int(info[0]), ip), "rt_get_bvh")
        return nodes, {"nodes": int(info[0]), "depth": int(info[1]), "builder": ("host", "device")[int(info[2])],
                       "build_ns": int(info[3])}

    def set_option(self, name, value):
        """Per-context tuning knob (the RT_* environment variables are only the defaults)."""
        self._check(self.L.rt_set_option(self.h, name.encode(), C.c_int64(int(value))), "rt_set_option")

    def trace_paths(self, nx, ny, pixel, sample, max_depth=50, seed=1, variant=RT_VARIANT_WAVEFRONT, log_bounces=0):
        """rt_trace_paths: the production render code run for chosen (pixel, sample) pairs.  Returns
        (radiance [n,3] f32, nrays [n] i32, term [n] i32, log [n, log_bounces] PATH_BOUNCE_DTYPE | None)."""
        pix = np.ascontiguousarray(pixel, np.int32)
        smp = np.ascontiguousarray(sample, np.int32)
        n = len(pix)
        rad = np.zeros((n, 3), np.float32)
        nr = np.zeros(n, np.int32)
        term = np.zeros(n, np.int32)
        log = np.zeros((n, log_bounces), PATH_BOUNCE_DTYPE) if log_bounces > 0 else None
        self._check(self.L.rt_trace_paths(self.h, nx, ny, n, _p(pix, _i32p), _p(smp, _i32p), max_depth, C.c_uint64(seed),
                                          variant, _p(rad, _f32p), _p(nr, _i32p), _p(term, _i32p), log_bounces,
                                          None if log is None else log.ctypes.data_as(C.c_void_p)), "rt_trace_paths")
        return rad, nr, term, log

    def sample_device(self, kind, n, seed=1):
        """rt_sample_device: n points of the device's rand-in-unit-sphere (kind 0, [n,3]) / rand-in-unit-disk (kind 1, [n,2])."""
        dim = 3 if kind == 0 else 2
        out = np.zeros((n, dim), np.float32)
        self._check(self.L.rt_sample_device(self.h, kind, n, C.c_uint64(seed), _p(out, _f32p)), "rt_sample_device")
        return out

    def set_camera(self, cam_type, camf):
        c = np.ascontiguousarray(camf, np.float32)
        assert c.shape == (24,)
        self._check(self.L.rt_set_camera(self.h, C.c_int(cam_type), _p(c, _f32p)), "rt_set_camera")

    def render(self, nx, ny, nsamples, max_depth=50, seed=1, variant=RT_VARIANT_WAVEFRONT, linear=True, rgb8=True,
               out_linear=None, out_rgb8=None):
        """rt_render with host buffers.  Returns (linear [ny,nx,3] f32 with j=0 bottom | None, rgb8 [ny,nx,3] | None)."""
        lin = (out_linear if out_linear is not None else np.empty((ny, nx, 3), np.float32)) if linear else None
        img = (out_rgb8 if out_rgb8 is not None else np.empty((ny, nx, 3), np.uint8)) if rgb8 else None
        self._check(self.L.rt_render(self.h, nx, ny, nsamples, max_depth, C.c_uint64(seed), variant, _p(lin, _f32p),
                                     _p(img, _u8p)), "rt_render")
        return lin, img

    def render_views(self, cameras, nx, ny, nsamples, max_depth=50, seed=1, variant=RT_VARIANT_WAVEFRONT, linear=True,
                     rgb8=True):
        """rt_render_views: K cameras (see ``marshal_views``) of the current scene in one call.  Returns (linear
        [K,ny,nx,3] f32 | None, rgb8 [K,ny,nx,3] | None), every view in ``render``'s convention (linear: j = 0 at the
        bottom; rgb8: row 0 at the top).  View v equals ``set_camera(camera v)`` + ``render`` up to the order of the
        sample sums.  The context's camera is neither needed nor changed."""
        types, cams = marshal_views(cameras)
        k = len(types)
        lin = np.empty((k, ny, nx, 3), np.float32) if linear else None
        img = np.empty((k, ny, nx, 3), np.uint8) if rgb8 else None
        self._check(self.L.rt_render_views(self.h, k, _p(types, _i32p), _p(cams, _f32p), nx, ny, nsamples, max_depth,
                                           C.c_uint64(seed), variant, _p(lin, _f32p), _p(img, _u8p)), "rt_render_views")
        return lin, img

    def render_views_accumulate_device(self, cameras, nx, ny, sample_begin, sample_count, d_sum_ptr, max_depth=50, seed=1,
                                       variant=RT_VARIANT_WAVEFRONT, stream=None, sync=True):
        """d_sum (K*ny*nx*3 float32 on device 0, view v at offset v*nx*ny*3) += the views' samples [sample_begin,
        sample_begin + sample_count)."""
        types, cams = marshal_views(cameras)
        self._check(self.L.rt_render_views_accumulate_device(
            self.h, len(types), _p(types, _i32p), _p(cams, _f32p), nx, ny, sample_begin, sample_count, max_depth,
            C.c_uint64(seed), variant, C.c_void_p(d_sum_ptr), C.c_void_p(stream or 0), 1 if sync else 0),
            "rt_render_views_accumulate_device")

    def resolve_views_device(self, n_views, nx, ny, nsamples_total, d_sum_ptr, d_rgb8_ptr, stream=None, sync=True):
        self._check(self.L.rt_resolve_views_device(self.h, n_views, nx, ny, nsamples_total, C.c_void_p(d_sum_ptr),
                                                   C.c_void_p(d_rgb8_ptr), C.c_void_p(stream or 0), 1 if sync else 0),
                    "rt_resolve_views_device")

    def render_accumulate_device(self, nx, ny, sample_begin, sample_count, d_sum_ptr, row_offset=0, row_stride=1,
                                 max_depth=50, seed=1, variant=RT_VARIANT_WAVEFRONT, stream=None, sync=True):
        self._check(self.L.rt_render_accumulate_device(
            self.h, nx, ny, sample_begin, sample_count, row_offset, row_stride, max_depth, C.c_uint64(seed), variant,
            C.c_void_p(d_sum_ptr), C.c_void_p(stream or 0), 1 if sync else 0), "rt_render_accumulate_device")

    def resolve_device(self, nx, ny, nsamples_total, d_sum_ptr, d_rgb8_ptr, stream=None, sync=True):
        self._check(self.L.rt_resolve_device(self.h, nx, ny, nsamples_total, C.c_void_p(d_sum_ptr),
                                             C.c_void_p(d_rgb8_ptr), C.c_void_p(stream or 0), 1 if sync else 0),
                    "rt_resolve_device")

    def trace_primary(self, origins, dirs, times=None, t_min=0.001, t_max=float(np.finfo(np.float32).max)):
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        n = o.shape[0]
        tm = None if times is None else np.ascontiguousarray(times, np.float32)
        t = np.empty(n, np.float64)
        ids = np.empty(n, np.int32)
        self._check(self.L.rt_trace_primary(self.h, n, _p(o, _f32p), _p(d, _f32p), _p(tm, _f32p), C.c_double(t_min),
                                            C.c_double(t_max), _p(t, _f64p), _p(ids, _i32p)), "rt_trace_primary")
        return t, ids

    def cull_check(self, origins, dirs, times=None, t_min=0.001, t_max=float(np.finfo(np.float32).max)):
        """(pairs the FP32 cull would lose — must be 0, cull survivors, exact candidates) over rays x listed spheres."""
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        tm = None if times is None else np.ascontiguousarray(times, np.float32)
        out = np.zeros(3, np.uint64)
        self._check(self.L.rt_cull_check(self.h, o.shape[0], _p(o, _f32p), _p(d, _f32p), _p(tm, _f32p), C.c_double(t_min),
                                         C.c_double(t_max), _p(out, _u64p)), "rt_cull_check")
        return int(out[0]), int(out[1]), int(out[2])

    def generate_rays(self, nx, ny, ij, s, seed=1):
        ij = np.ascontiguousarray(ij, np.int32).reshape(-1, 2)
        s = np.ascontiguousarray(s, np.int32)
        n = ij.shape[0]
        o = np.empty((n, 3), np.float32); d = np.empty((n, 3), np.float32); t = np.empty(n, np.float32)
        rnd = np.empty((n, 5), np.float32)
        self._check(self.L.rt_generate_rays(self.h, n, nx, ny, _p(ij, _i32p), _p(s, _i32p), C.c_uint64(seed),
                                            _p(o, _f32p), _p(d, _f32p), _p(t, _f32p), _p(rnd, _f32p)),
                    "rt_generate_rays")
        return o, d, t, rnd

    def shade_batch(self, origins, dirs, times, hit_id, hit_t, ball, u01):
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        n = o.shape[0]
        tm = np.ascontiguousarray(times, np.float32)
        hid = np.ascontiguousarray(hit_id, np.int32)
        ht = np.ascontiguousarray(hit_t, np.float64)
        b = np.ascontiguousarray(ball, np.float32).reshape(-1, 3)
        u = np.ascontiguousarray(u01, np.float32)
        oo = np.zeros((n, 3), np.float32); od = np.zeros((n, 3), np.float32)
        oa = np.zeros((n, 3), np.float32); oe = np.zeros((n, 3), np.float32)
        fl = np.zeros(n, np.int32)
        self._check(self.L.rt_shade_batch(self.h, n, _p(o, _f32p), _p(d, _f32p), _p(tm, _f32p), _p(hid, _i32p),
                                          _p(ht, _f64p), _p(b, _f32p), _p(u, _f32p), _p(oo, _f32p), _p(od, _f32p),
                                          _p(oa, _f32p), _p(oe, _f32p), _p(fl, _i32p)), "rt_shade_batch")
        return dict(origin=oo, dir=od, atten=oa, emitted=oe, flags=fl)

    def measure_fp32_peak(self):
        a = C.c_double(); b = C.c_double()
        self._check(self.L.rt_measure_fp32_peak(self.h, C.byref(a), C.byref(b)), "rt_measure_fp32_peak")
        return a.value, b.value

    def counters(self):
        out = np.zeros(RT_CTR_COUNT, np.uint64)
        self._check(self.L.rt_get_counters(self.h, _p(out, _u64p)), "rt_get_counters")
        return {k: int(v) for k, v in zip(COUNTER_NAMES, out)}

    def reset_counters(self):
        self._check(self.L.rt_reset_counters(self.h), "rt_reset_counters")

    def set_profile(self, on=True):
        self._check(self.L.rt_set_profile(self.h, 1 if on else 0), "rt_set_profile")

    def device_info(self):
        sm = C.c_int32(); clk = C.c_int32(); name = C.create_string_buffer(64)
        self._check(self.L.rt_device_info(self.h, C.byref(sm), C.byref(clk), name), "rt_device_info")
        return dict(sm_count=sm.value, clock_khz=clk.value, name=name.value.decode())
