"""ctypes host over include/drt.h.  No torch types cross the boundary: the ray queries (Scene.intersect / Scene.occluded) take CUDA tensors
and pass their device pointers; elsewhere torch is only used by callers that want device-resident outputs (multi-GPU tile gather)."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SCENES_DIR = os.path.join(ROOT, "scenes")
TEX_DIR = os.path.join(SCENES_DIR, "txtrs")

ACCEL_REFERENCE, ACCEL_REFERENCE_FAST, ACCEL_LBVH = 0, 1, 2


class DrtError(RuntimeError):
    pass


class _Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("cols", C.c_int32), ("rows", C.c_int32), ("counters", C.c_int32),
                ("seed", C.c_uint64), ("batch_rays", C.c_int64)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rays_primary", "rays_shadow", "rays_reflect", "rays_refract", "rays_photon",
                                           "box_tests", "prim_tests", "photons_stored", "kernel_launches", "box_tests_closest", "prim_tests_closest")] + \
               [(n, C.c_double) for n in ("ms_trace", "ms_shade", "ms_light", "ms_other", "ms_total")] + \
               [(n, C.c_uint64) for n in ("rays_deferred", "frame_retries", "host_syncs")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}

    @property
    def rays_total(self):
        return self.rays_primary + self.rays_shadow + self.rays_reflect + self.rays_refract + self.rays_photon


_LOADER = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_char_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.POINTER(C.c_int32)))

_lib = None


def lib_path():
    return os.environ.get("DRT_LIB") or os.path.join(HERE, "libdrt.so")     # DRT_LIB: tuning variants built by tools/, never a fallback


def load_library():
    """Load libdrt.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise DrtError("libdrt.so is not built (run `python -m distraytracer_old_b200.build` or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(p)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    sig = {
        "drt_create": (C.c_int, [C.POINTER(_Config), C.POINTER(vp)]),
        "drt_destroy": (None, [vp]),
        "drt_last_error": (C.c_char_p, [vp]),
        "drt_set_image_loader": (C.c_int, [vp, _LOADER, vp]),
        "drt_set_texture_dir": (C.c_int, [vp, C.c_char_p]),
        "drt_scene_reset": (C.c_int, [vp]),
        "drt_scene_command": (C.c_int, [vp, C.c_char_p]),
        "drt_scene_load_cli": (C.c_int, [vp, C.c_char_p, C.c_char_p]),
        "drt_scene_override": (C.c_int, [vp, i32, i64]),
        "drt_scene_finalize": (C.c_int, [vp, i32]),
        "drt_scene_reupload": (C.c_int, [vp]),
        "drt_scene_info": (C.c_int, [vp, C.POINTER(i32)]),
        "drt_accel_info": (C.c_int, [vp, C.POINTER(dbl)]),
        "drt_scene_counts": (C.c_int, [vp, C.POINTER(i64)]),
        "drt_build_info": (C.c_int, [vp, C.POINTER(dbl)]),
        "drt_bvh_order": (C.c_int, [vp, i32, vp, vp, i32]),
        "drt_scene_refine": (C.c_int, [vp]),
        "drt_refine_steps": (i32, [i32, i32, C.POINTER(i32)]),
        "drt_refine_pass": (C.c_int, [vp, i32, i32, i32, vp]),
        "drt_lbvh_probe": (i64, [vp, i32, i32, vp, vp, vp, vp, vp, i64]),
        "drt_emit_photons": (C.c_int, [vp, C.POINTER(Stats)]),
        "drt_render": (C.c_int, [vp, vp, C.POINTER(Stats)]),
        "drt_render_aov": (C.c_int, [vp, vp, vp, vp, vp, vp, C.POINTER(Stats)]),
        "drt_render_device": (C.c_int, [vp, i64, i64, vp, C.POINTER(Stats)]),
        "drt_render_device_chunks": (C.c_int, [vp, i32, i32, i32, vp, C.POINTER(Stats)]),
        "drt_save_png": (C.c_int, [C.c_char_p, vp, i32, i32]),
        "drt_trace_rays": (C.c_int, [vp, i64, vp, vp, vp, vp]),
        "drt_query_closest": (C.c_int, [vp, i64, vp, vp, vp, vp, vp, vp, vp, C.POINTER(Stats)]),
        "drt_query_occluded": (C.c_int, [vp, i64, vp, vp, vp, vp, C.POINTER(Stats)]),
        "drt_eval_texture": (C.c_int, [vp, i32, i64, vp, vp, vp]),
        "drt_dump_bvh": (i64, [vp, i32, vp, i64, vp]),
        "drt_obj_ctm": (C.c_int, [vp, i32, vp]),
        "drt_sample_u01": (dbl, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
        "drt_get_photons": (i64, [vp, vp, i64]),
        "drt_emit_photons_range": (C.c_int, [vp, i64, i64, C.POINTER(Stats)]),
        "drt_photons_export_device": (i64, [vp, vp, i64]),
        "drt_photons_build_device": (C.c_int, [vp, vp, i64, C.POINTER(Stats)]),
        "drt_photon_probe": (C.c_int, [vp, i64, vp, vp]),
        "drt_comm_unique_id": (C.c_int, [vp]),
        "drt_comm_init": (C.c_int, [vp, vp, i32, i32]),
        "drt_comm_destroy": (C.c_int, [vp]),
        "drt_render_distributed": (C.c_int, [vp, vp, vp, i32, i32, C.POINTER(Stats)]),
        "drt_dist_rank_pixels": (i64, [i32, i32, i32, i32, i32]),
        "drt_dist_abs_pixel": (i64, [i32, i32, i32, i32, i32, i64]),
        "drt_dist_photon_range": (C.c_int, [i64, i32, i32, C.POINTER(i64)]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args
    _lib = L
    return L


EXPORTS = ["drt_create", "drt_destroy", "drt_last_error", "drt_set_image_loader", "drt_set_texture_dir", "drt_scene_reset",
           "drt_scene_command", "drt_scene_load_cli", "drt_scene_override", "drt_scene_finalize", "drt_scene_reupload",
           "drt_scene_info", "drt_scene_counts", "drt_build_info", "drt_bvh_order", "drt_lbvh_probe", "drt_scene_refine", "drt_refine_steps", "drt_refine_pass", "drt_accel_info", "drt_emit_photons", "drt_render", "drt_render_aov", "drt_render_device", "drt_render_device_chunks", "drt_save_png",
           "drt_trace_rays", "drt_query_closest", "drt_query_occluded", "drt_eval_texture", "drt_dump_bvh", "drt_obj_ctm", "drt_sample_u01", "drt_get_photons",
           "drt_emit_photons_range", "drt_photons_export_device", "drt_photons_build_device", "drt_photon_probe",
           "drt_comm_unique_id", "drt_comm_init", "drt_comm_destroy", "drt_render_distributed",
           "drt_dist_rank_pixels", "drt_dist_abs_pixel", "drt_dist_photon_range"]


def decode_image_argb(path):
    """PApplet.loadImage(...).pixels: ARGB ints with alpha 0xFF."""
    from PIL import Image
    im = Image.open(path).convert("RGBA")
    a = np.asarray(im, dtype=np.uint32)
    argb = (np.uint32(0xFF) << 24) | (a[..., 0] << 16) | (a[..., 1] << 8) | a[..., 2]
    return im.width, im.height, np.ascontiguousarray(argb.astype(np.uint32).view(np.int32))


class Context:
    """One renderer context == one GPU (device=-1: host-only, interpreter + flattener, cannot render)."""

    def __init__(self, device=0, cols=300, rows=300, seed=0x5EED, counters=False, batch_rays=0, texture_dir=TEX_DIR):
        self.L = load_library()
        if cols <= 0 or rows <= 0:
            raise DrtError("frame size must be positive (got %d x %d): host buffers are sized from it" % (cols, rows))
        cfg = _Config(device, cols, rows, int(counters), seed, batch_rays)
        h = C.c_void_p()
        rc = self.L.drt_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise DrtError("drt_create failed (%d): no usable CUDA device and no CPU fallback exists" % rc)
        self.h = h
        self.cols, self.rows, self.device = cols, rows, device
        self._images = {}
        self._texture_dir = texture_dir
        self._cb = _LOADER(self._load_image)
        self._ck(self.L.drt_set_image_loader(self.h, self._cb, None))

    def _load_image(self, user, name, w, h, px):
        try:
            key = name.decode()
            if key not in self._images:
                self._images[key] = decode_image_argb(os.path.join(self._texture_dir, key))
            ww, hh, arr = self._images[key]
            w[0], h[0] = ww, hh
            px[0] = arr.ctypes.data_as(C.POINTER(C.c_int32))
            return 0
        except Exception:
            return 1

    def _ck(self, rc):
        if rc != 0:
            raise DrtError("drt error %d: %s" % (rc, (self.L.drt_last_error(self.h) or b"").decode()))

    # ---- multi-GPU inside the library (NCCL): rank 0 makes the id, the host ships it, every rank joins
    @staticmethod
    def comm_unique_id():
        buf = (C.c_uint8 * 128)()
        if load_library().drt_comm_unique_id(buf) != 0:
            raise DrtError("drt_comm_unique_id failed (NCCL not available?)")
        return bytes(buf)

    def comm_init(self, id128, world, rank):
        buf = (C.c_uint8 * 128).from_buffer_copy(id128) if id128 is not None else None
        self._ck(self.L.drt_comm_init(self.h, buf, world, rank))
        self.world, self.rank = world, rank

    def bvh_order(self, keys, on_device):
        """Parity probe: object order of the reference's median-split BVH for centroid keys [n, 3] (host recursion or device builder)."""
        k = np.ascontiguousarray(np.asarray(keys, dtype=np.float64).T)          # [3][n]
        n = k.shape[1]
        ord_ = np.empty(n, dtype=np.int32)
        self._ck(self.L.drt_bvh_order(self.h, n, k.ctypes.data, ord_.ctypes.data, 1 if on_device else 0))
        return ord_

    def close(self):
        if getattr(self, "h", None):
            self.L.drt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def refine_steps(cols, rows):
    """Step sequence of the reference's progressive refinement display for a cols x rows frame (myScene.setRefine)."""
    o = (C.c_int32 * 16)()
    n = load_library().drt_refine_steps(cols, rows, o)
    return [int(o[i]) for i in range(n)]


def refine_pass(argb_full, step):
    """Preview of one refinement step, made from the finished frame (rows x cols ARGB ints)."""
    a = np.ascontiguousarray(argb_full, dtype=np.int32)
    out = np.empty_like(a)
    if load_library().drt_refine_pass(a.ctypes.data, a.shape[1], a.shape[0], step, out.ctypes.data) != 0:
        raise DrtError("drt_refine_pass: bad arguments")
    return out


class Scene:
    """Mirror of the reference's myScene for the render path."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.L = ctx.L
        self.finalized = False
        ctx._ck(self.L.drt_scene_reset(ctx.h))

    @classmethod
    def from_cli(cls, ctx, file, data_dir=SCENES_DIR, spp=0, photons=-1, accel=ACCEL_REFERENCE, finalize=True):
        s = cls.__new__(cls)
        s.ctx, s.L, s.finalized = ctx, ctx.L, False
        ctx._ck(s.L.drt_scene_load_cli(ctx.h, file.encode(), data_dir.encode()))
        ctx._ck(s.L.drt_scene_override(ctx.h, spp, photons))
        if finalize:
            s.finalize(accel)
        return s

    def command(self, line):
        self.ctx._ck(self.L.drt_scene_command(self.ctx.h, line.encode()))

    def override(self, spp=0, photons=-1):
        self.ctx._ck(self.L.drt_scene_override(self.ctx.h, spp, photons))

    def finalize(self, accel=ACCEL_REFERENCE):
        self.ctx._ck(self.L.drt_scene_finalize(self.ctx.h, accel))
        self.finalized = True

    def reupload(self):
        self.ctx._ck(self.L.drt_scene_reupload(self.ctx.h))

    def info(self):
        o = (C.c_int32 * 16)()
        self.ctx._ck(self.L.drt_scene_info(self.ctx.h, o))
        k = ["cols", "rows", "spp", "top", "lights", "prims", "instances", "photon_kind", "shaders", "nodes", "xforms", "lists", "bvhs", "images", "warnings", "photons_cast"]
        return dict(zip(k, list(o)))

    def counts(self):
        o = (C.c_int64 * 8)()
        self.ctx._ck(self.L.drt_scene_counts(self.ctx.h, o))
        return {"tris_packed": o[0], "fast_bvhs": o[1], "top_tris_packed": o[2], "tris_in_fast_bvhs": o[3], "children": o[4], "pdata_doubles": o[5]}

    def refine_on(self):
        """`refine on` was set by the scene (myScene.setRefine)."""
        return self.L.drt_scene_refine(self.ctx.h) == 1

    def build_info(self):
        o = (C.c_double * 8)()
        self.ctx._ck(self.L.drt_build_info(self.ctx.h, o))
        return {"parse_ms": o[0], "bvh_order_ms": o[1], "bvh_order_device_ms": o[2], "bvh_shape_ms": o[3], "finalize_ms": o[4], "bvh_device_builds": int(o[5]), "bvh_objects": int(o[6]), "upload_ms": o[7]}

    def lbvh_probe(self, fast_index=0, resident=False):
        """Packed triangles of a fast BVH (host order, or as resident in HBM) + the GPU-built LBVH nodes (resident, DRT_ACCEL_LBVH mode)."""
        box = np.zeros(6)
        n = self.L.drt_lbvh_probe(self.ctx.h, fast_index, 1 if resident else 0, box.ctypes.data, None, None, None, None, 0)
        if n == -2:                          # DRT_ERR_BAD_ARG: no such fast BVH
            return None
        if n < 0:
            self.ctx._ck(int(n))
        nn = max(0, (n + 3) // 4 - 1)
        v, ser, links, boxes = np.zeros((n, 9)), np.zeros(n, dtype=np.int32), np.zeros((nn, 2), dtype=np.int32), np.zeros((nn, 12))
        r = self.L.drt_lbvh_probe(self.ctx.h, fast_index, 1 if resident else 0, box.ctypes.data, v.ctypes.data, ser.ctypes.data, links.ctypes.data, boxes.ctypes.data, n)
        if r < 0:
            self.ctx._ck(int(r))
        return {"box": box, "verts": v, "serial": ser, "links": links, "boxes": boxes}

    def accel_info(self):
        o = (C.c_double * 4)()
        self.ctx._ck(self.L.drt_accel_info(self.ctx.h, o))
        return {"lbvh_build_ms": o[0], "lbvh_tris": int(o[1]), "lbvh_nodes": int(o[2]), "scene_bytes": int(o[3])}

    # ---- rendering (myScene.draw)
    def draw(self, aov=False):
        n = self.ctx.cols * self.ctx.rows
        st = Stats()
        argb = np.zeros((self.ctx.rows, self.ctx.cols), dtype=np.int32)
        if not aov:
            self.ctx._ck(self.L.drt_render(self.ctx.h, argb.ctypes.data, C.byref(st)))
            return argb, st
        hp = np.zeros_like(argb)
        hi = np.zeros_like(argb)
        rgb = np.zeros((self.ctx.rows, self.ctx.cols, 3), dtype=np.float64)
        t = np.zeros((self.ctx.rows, self.ctx.cols), dtype=np.float64)
        self.ctx._ck(self.L.drt_render_aov(self.ctx.h, argb.ctypes.data, hp.ctypes.data, hi.ctypes.data, rgb.ctypes.data, t.ctypes.data, C.byref(st)))
        return {"argb": argb, "hit_prim": hp, "hit_inst": hi, "rgb": rgb, "t": t, "stats": st, "pixels": n}

    def draw_into(self, host_argb, stats=None):
        """Render into a caller-owned (e.g. pinned) int32 host buffer."""
        st = stats if stats is not None else Stats()
        self.ctx._ck(self.L.drt_render(self.ctx.h, host_argb, C.byref(st)))
        return st

    def draw_device(self, pix0, pix1, dev_ptr):
        st = Stats()
        self.ctx._ck(self.L.drt_render_device(self.ctx.h, pix0, pix1, dev_ptr, C.byref(st)))
        return st

    def draw_device_chunks(self, world, rank, chunk_rows, dev_ptr):
        st = Stats()
        self.ctx._ck(self.L.drt_render_device_chunks(self.ctx.h, world, rank, chunk_rows, dev_ptr, C.byref(st)))
        return st

    def draw_distributed(self, host_ptr=None, dev_ptr=None, chunk_rows=8, reemit_photons=False):
        """Collective: this rank's chunks + NCCL gather; rank 0 receives the frame in host_ptr and / or dev_ptr (see include/drt.h)."""
        st = Stats()
        self.ctx._ck(self.L.drt_render_distributed(self.ctx.h, host_ptr, dev_ptr, chunk_rows, int(reemit_photons), C.byref(st)))
        return st

    def emit_photons(self):
        st = Stats()
        self.ctx._ck(self.L.drt_emit_photons(self.ctx.h, C.byref(st)))
        return st

    def photons(self, cap=1 << 26):
        st = self.emit_photons()
        n = int(st.photons_stored)
        out = np.zeros((max(n, 1), 6), dtype=np.float64)
        m = self.L.drt_get_photons(self.ctx.h, out.ctypes.data, min(n, cap))
        return out[:max(m, 0)]

    def emit_photons_range(self, i0, i1):
        st = Stats()
        self.ctx._ck(self.L.drt_emit_photons_range(self.ctx.h, i0, i1, C.byref(st)))
        return st

    def photons_export_device(self, dev_ptr, cap):
        n = self.L.drt_photons_export_device(self.ctx.h, dev_ptr, cap)
        if n < 0:
            self.ctx._ck(int(n))
        return int(n)

    def photons_build_device(self, dev_ptr, n):
        st = Stats()
        self.ctx._ck(self.L.drt_photons_build_device(self.ctx.h, dev_ptr, n, C.byref(st)))
        return st

    def photon_probe(self, pts):
        """kNN radiance gather at world points: rows of {sum r, sum g, sum b, d2 of the farthest, gather tier taken (0 none, 1-4)}."""
        pts = np.ascontiguousarray(pts, dtype=np.float64)
        out = np.zeros((pts.shape[0], 5), dtype=np.float64)
        self.ctx._ck(self.L.drt_photon_probe(self.ctx.h, pts.shape[0], pts.ctypes.data, out.ctypes.data))
        return out

    def save(self, path, argb):
        a = np.ascontiguousarray(argb, dtype=np.int32)
        rc = self.L.drt_save_png(path.encode(), a.ctypes.data, a.shape[1], a.shape[0])
        if rc != 0:
            raise DrtError("drt_save_png failed")

    # ---- ray queries on CUDA tensors (drt_query_closest / drt_query_occluded)
    def _device_arrays(self, *specs):
        """specs: (tensor, name, cols).  Each must be a float64 torch tensor of shape (n, cols) (cols None: (n,)), contiguous, and on this
        context's CUDA device, with the same n: it is passed as is, never copied.  Form and device are checked in that order."""
        import torch
        for x, name, cols in specs:
            if not isinstance(x, torch.Tensor):
                raise ValueError("%s must be a torch.Tensor on cuda:%d, got %s" % (name, self.ctx.device, type(x).__name__))
            if x.dtype != torch.float64:
                raise ValueError("%s must be torch.float64, got %s" % (name, x.dtype))
            if (x.dim() != 2 or x.shape[1] != cols) if cols else x.dim() != 1:
                raise ValueError("%s must have shape %s, got %s" % (name, "(n, %d)" % cols if cols else "(n,)", tuple(x.shape)))
            if not x.is_contiguous():
                raise ValueError("%s must be contiguous" % name)
            if x.shape[0] != specs[0][0].shape[0]:
                raise ValueError("%s holds %d rows for %d rays" % (name, x.shape[0], specs[0][0].shape[0]))
        for x, name, _ in specs:
            if x.device.type != "cuda" or x.device.index != self.ctx.device:
                raise ValueError("%s must be on cuda:%d (the context's device), got %s" % (name, self.ctx.device, x.device))
        return specs[0][0].shape[0]

    def intersect(self, org, dirs, tmax=None, frame=False, stats=None):
        """Closest hit of n caller rays (CUDA float64 tensors (n, 3)): ids int32 (n, 2) = (primitive serial, instance serial), -1 on a miss,
        and t float64 (n,), 0 on a miss; a hit counts only when t < tmax (float64 (n,), None = +inf).  frame=True also returns the world hit
        point and unit normal the renderer shades with, (n, 3) each.  stats: a Stats to fill."""
        import torch
        n = self._device_arrays((org, "org", 3), (dirs, "dirs", 3), *([(tmax, "tmax", None)] if tmax is not None else []))
        ids = torch.empty((n, 2), dtype=torch.int32, device=org.device)
        t = torch.empty(n, dtype=torch.float64, device=org.device)
        pos = torch.empty((n, 3), dtype=torch.float64, device=org.device) if frame else None
        nrm = torch.empty((n, 3), dtype=torch.float64, device=org.device) if frame else None
        torch.cuda.current_stream(org.device).synchronize()        # the library's stream does not wait on torch's
        ptr = lambda a: a.data_ptr() if a is not None else None
        st = stats if stats is not None else Stats()
        self.ctx._ck(self.L.drt_query_closest(self.ctx.h, n, ptr(org), ptr(dirs), ptr(tmax), ptr(ids), ptr(t), ptr(pos), ptr(nrm), C.byref(st)))
        return (ids, t, pos, nrm) if frame else (ids, t)

    def occluded(self, org, dirs, dist, stats=None):
        """Shadow test of n caller rays (CUDA float64 tensors (n, 3)) against distances dist (float64 (n,), +inf allowed): torch.bool (n,),
        True when something is hit with dist - t > 1e-7 (the renderer's shadow rule).  stats: a Stats to fill."""
        import torch
        n = self._device_arrays((org, "org", 3), (dirs, "dirs", 3), (dist, "dist", None))
        occ = torch.empty(n, dtype=torch.bool, device=org.device)          # one byte per ray, written 0 / 1 by the library
        torch.cuda.current_stream(org.device).synchronize()
        st = stats if stats is not None else Stats()
        self.ctx._ck(self.L.drt_query_occluded(self.ctx.h, n, org.data_ptr(), dirs.data_ptr(), dist.data_ptr(), occ.data_ptr(), C.byref(st)))
        return occ

    # ---- parity probes
    def trace_rays(self, org, dirs):
        org = np.ascontiguousarray(org, dtype=np.float64)
        dirs = np.ascontiguousarray(dirs, dtype=np.float64)
        n = org.shape[0]
        ids = np.zeros((n, 2), dtype=np.int32)
        t = np.zeros(n, dtype=np.float64)
        self.ctx._ck(self.L.drt_trace_rays(self.ctx.h, n, org.ctypes.data, dirs.ctypes.data, ids.ctypes.data, t.ctypes.data))
        return ids, t

    def eval_texture(self, shader_serial, hit_loc, fwd_loc=None):
        hit_loc = np.ascontiguousarray(hit_loc, dtype=np.float64)
        fwd_loc = hit_loc if fwd_loc is None else np.ascontiguousarray(fwd_loc, dtype=np.float64)
        out = np.zeros_like(hit_loc)
        self.ctx._ck(self.L.drt_eval_texture(self.ctx.h, shader_serial, hit_loc.shape[0], hit_loc.ctypes.data, fwd_loc.ctypes.data, out.ctypes.data))
        return out

    def dump_bvh(self, top_index):
        box = np.zeros(6)
        n = self.L.drt_dump_bvh(self.ctx.h, top_index, None, 0, box.ctypes.data)
        if n < 0:
            return None, None
        out = np.zeros(n, dtype=np.int32)
        self.L.drt_dump_bvh(self.ctx.h, top_index, out.ctypes.data, n, box.ctypes.data)
        return out, box

    def obj_ctm(self, top_index):
        m = np.zeros(16)
        self.ctx._ck(self.L.drt_obj_ctm(self.ctx.h, top_index, m.ctypes.data))
        return m.reshape(4, 4)


class RTFileReader:
    """myRTFileReader: reads a .cli file line by line, forwards every line, renders on `write`."""

    def __init__(self, ctx, data_dir=SCENES_DIR, spp=0, photons=-1, accel=ACCEL_REFERENCE):
        self.ctx, self.data_dir, self.spp, self.photons, self.accel = ctx, data_dir, spp, photons, accel
        self.images = {}

    def readRTFile(self, file_name, scene=None, out_dir=None):
        main = scene is None
        if main:
            scene = Scene(self.ctx)
        with open(os.path.join(self.data_dir, file_name)) as f:
            for raw in f:
                line = raw.rstrip("\r\n")
                tok = [t for t in line.split(" ") if t]
                if not tok or tok[0].startswith("#"):
                    continue
                if tok[0] == "read":
                    self.readRTFile(tok[1], scene)
                    continue
                scene.command(line)
                if tok[0] == "write":      # the reference renders inside the parser (myRTFileReader.java:86-93)
                    scene.override(self.spp, self.photons)
                    scene.finalize(self.accel)
                    argb, st = scene.draw()
                    self.images[tok[1]] = (argb, st)
                    if out_dir:
                        scene.save(os.path.join(out_dir, os.path.splitext(tok[1])[0] + ".png"), argb)
        return scene


def dist_rank_pixels(cols, rows, world, rank, chunk_rows=8):
    return int(load_library().drt_dist_rank_pixels(cols, rows, world, rank, chunk_rows))


def dist_abs_pixels(cols, rows, world, rank, chunk_rows=8):
    """int64 array: absolute pixel of every compact slot of `rank` (-1 = padding), from the library's own mapping."""
    L = load_library()
    n = dist_rank_pixels(cols, rows, world, rank, chunk_rows)
    return np.array([L.drt_dist_abs_pixel(cols, rows, world, rank, chunk_rows, j) for j in range(n)], dtype=np.int64)


def dist_photon_range(n_cast, world, rank):
    o = (C.c_int64 * 2)()
    if load_library().drt_dist_photon_range(n_cast, world, rank, o) != 0:
        raise DrtError("bad photon partition")
    return int(o[0]), int(o[1])


def sample_u01(seed, stream, a, b, c, d):
    return load_library().drt_sample_u01(seed, stream, a, b, c, d)
