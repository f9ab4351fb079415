"""Ray queries on device buffers (drt_query_closest / drt_query_occluded, Scene.intersect / Scene.occluded).

The closest-hit query must return exactly what the generic-kernel probe (drt_trace_rays) returns, in every acceleration mode and kernel
variant, and both queries must agree with the CPU oracle bit for bit (ids, t, occlusion) or to FP64 rounding (hit point, normal).  The
argument checks and the Python wrapper's tensor checks also run without a GPU."""
import ctypes as C
import os
import re
import subprocess
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 1e-7          # DRT_EPS: the shadow rule is (dist - t) > EPS

PROBE_SCENES = ["p3_t09", "p3_t10", "p3_t11_sierp", "p3_t02_sierp", "old_t08", "cylinder1", "ext_torus_quadrics"]
ORACLE_SCENES = ["p3_t08", "p3_t02_sierp", "p3_t12", "old_t08", "cylinder1", "ext_torus_quadrics"]      # no moving spheres
SHAPES = (None, 0, 1, 7)          # None: the variant the scene chooses; else DRT_FORCE_SHAPE


def ray_set(rng, n):
    """Half aimed at the scene centre from all around, half from inside / on / outside the objects with random directions; a share of each
    exactly axis-parallel (components +0.0 / -0.0) or almost so (1e-17)."""
    h = n // 2
    org = np.empty((n, 3))
    org[:h] = rng.uniform(-6, 6, size=(h, 3)); org[:h, 2] = rng.uniform(-2, 6, size=h)
    d = np.empty((n, 3))
    d[:h] = rng.uniform(-1.5, 1.5, size=(h, 3)) + np.array([0, 0, -4.0]) - org[:h]
    org[h:] = rng.uniform(-3, 3, size=(n - h, 3)); org[h:, 2] -= 3
    d[h:] = rng.normal(size=(n - h, 3))
    for lo in (0, h):
        k = n // 16; rows = lo + np.arange(2 * k)
        zero = np.where(rng.random(size=(2 * k, 3)) < 0.5, 0.0, -0.0); ax = rng.integers(0, 3, size=2 * k)
        d[rows, ax] = zero[np.arange(2 * k), ax]
        d[rows[:k], (ax[:k] + 1) % 3] = zero[np.arange(k), (ax[:k] + 1) % 3]
        r3 = lo + 2 * k + np.arange(k)
        d[r3, rng.integers(0, 3, size=k)] = rng.choice([-1e-17, 1e-17], size=k) * rng.uniform(0.5, 2.0, size=k)
    return org, d


def light_positions(name):
    """Positions of the scene file's lights (first three numbers of every light line)."""
    src = open(os.path.join(ROOT, "scenes", name + ".cli")).read()
    pts = [[float(v) for v in m.split()[1:4]] for m in re.findall(r"^\s*(?:point_light|spotlight|disk_light)\s+[^\n]*", src, re.M)]
    return np.array(pts or [[0.0, 5.0, 0.0]])


def cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to("cuda:0")


def load(drt, make, name, accel, shape, monkeypatch):
    if shape is None:
        monkeypatch.delenv("DRT_FORCE_SHAPE", raising=False)
    else:
        monkeypatch.setenv("DRT_FORCE_SHAPE", str(shape))          # read when the scene is uploaded
    ctx = make()
    s = drt.Scene.from_cli(ctx, name + ".cli", accel=accel)
    monkeypatch.delenv("DRT_FORCE_SHAPE", raising=False)
    return ctx, s


def query(drt, s, org, d, **kw):
    st = drt.Stats()
    out = s.intersect(cuda(org), cuda(d), stats=st, **kw)
    return [x.cpu().numpy() for x in out], st


def occl(drt, s, org, d, dist):
    st = drt.Stats()
    return s.occluded(cuda(org), cuda(d), cuda(dist), stats=st).cpu().numpy(), st


class RayOracle:
    """tests/ray_query_oracle.cpp: the CPU oracle's closest hit (with its shading point and normal) and shadow test on explicit rays."""

    def __init__(self, lib_path):
        L = C.CDLL(lib_path)
        L.rq_load.restype = C.c_void_p
        L.rq_load.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int]
        L.rq_query_rays.argtypes = [C.c_void_p, C.c_longlong] + [C.c_void_p] * 6
        L.rq_shadow_rays.argtypes = [C.c_void_p, C.c_longlong] + [C.c_void_p] * 4
        self.L, self.scenes = L, {}

    def scene(self, name):
        if name not in self.scenes:
            err = C.create_string_buffer(512)
            h = self.L.rq_load((name + ".cli").encode(), os.path.join(ROOT, "scenes").encode(), os.path.join(ROOT, "scenes", "txtrs_argb").encode(), err, 512)
            if not h:
                raise RuntimeError("oracle: " + err.value.decode())
            self.scenes[name] = h          # kept for the session (the oracle's scenes are not freed)
        return self.scenes[name]

    def query_rays(self, name, org, dirs):
        org, dirs = np.ascontiguousarray(org, dtype=np.float64), np.ascontiguousarray(dirs, dtype=np.float64)
        n = org.shape[0]
        ids, t, pos, nrm = np.zeros((n, 2), dtype=np.int32), np.zeros(n), np.zeros((n, 3)), np.zeros((n, 3))
        if self.L.rq_query_rays(self.scene(name), n, org.ctypes.data, dirs.ctypes.data, ids.ctypes.data, t.ctypes.data, pos.ctypes.data, nrm.ctypes.data) != 0:
            raise RuntimeError("oracle: a winning hit carries no CTM")
        return ids, t, pos, nrm

    def shadow_rays(self, name, org, dirs, dist):
        org, dirs = np.ascontiguousarray(org, dtype=np.float64), np.ascontiguousarray(dirs, dtype=np.float64)
        dist = np.ascontiguousarray(dist, dtype=np.float64)
        occ = np.zeros(org.shape[0], dtype=np.uint8)
        self.L.rq_shadow_rays(self.scene(name), org.shape[0], org.ctypes.data, dirs.ctypes.data, dist.ctypes.data, occ.ctypes.data)
        return occ.astype(bool)


@pytest.fixture(scope="session")
def ray_oracle(orc, tmp_path_factory):
    """Builds tests/ray_query_oracle.cpp against the oracle's headers with oracle/Makefile's flags, into a temporary directory (the tree may
    be read-only).  Depends on `orc` for the decoded textures and the generated bun69k mesh."""
    out = str(tmp_path_factory.mktemp("ray_oracle") / "libray_query_oracle.so")
    subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-w", "-shared",
                           "-I", os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests", "ray_query_oracle.cpp"), "-o", out, "-lpthread"])
    return RayOracle(out)


def close_rel(a, b, tol=1e-12):
    return np.all(np.linalg.norm(a - b, axis=1) <= tol * np.maximum(np.linalg.norm(b, axis=1), 1.0))


# ---- without a GPU ------------------------------------------------------------------------------------------------------------------
def test_query_on_host_only_context_returns_no_device(drt):
    ctx = drt.Context(device=-1)
    drt.Scene.from_cli(ctx, "t01.cli")
    one = (C.c_double * 3)()
    for n in (0, 1):
        assert ctx.L.drt_query_closest(ctx.h, n, one, one, None, one, one, None, None, None) == -1          # DRT_ERR_NO_DEVICE
        assert ctx.L.drt_query_occluded(ctx.h, n, one, one, one, one, None) == -1
    assert b"no CPU fallback" in ctx.L.drt_last_error(ctx.h)
    assert ctx.L.drt_query_closest(None, 1, one, one, None, one, one, None, None, None) == -2             # no context: DRT_ERR_BAD_ARG
    ctx.close()


def test_wrapper_rejects_what_it_would_have_to_copy(drt):
    import torch
    ctx = drt.Context(device=-1)
    s = drt.Scene.from_cli(ctx, "t01.cli")
    good = torch.zeros((4, 3), dtype=torch.float64)
    bad = {"float64": good.float(), "contiguous": torch.zeros((3, 4), dtype=torch.float64).t(), "cuda": good,
           r"shape \(n, 3\)": torch.zeros((4, 2), dtype=torch.float64), "torch.Tensor": np.zeros((4, 3))}
    for msg, x in bad.items():
        with pytest.raises(ValueError, match=msg):
            s.intersect(x, good)
        with pytest.raises(ValueError, match=msg):
            s.intersect(good, x)
        with pytest.raises(ValueError, match=msg):
            s.occluded(x, good, torch.zeros(4, dtype=torch.float64))
    with pytest.raises(ValueError, match="float64"):
        s.occluded(good, good, torch.zeros(4, dtype=torch.float32))
    with pytest.raises(ValueError, match=r"shape \(n,\)"):
        s.intersect(good, good, tmax=torch.zeros((4, 1), dtype=torch.float64))
    ctx.close()


def test_ray_oracle_agrees_with_the_oracles_trace_probe(orc, ray_oracle):
    """The test-local oracle entry points trace what orc_trace_rays traces (same rays, same scene code); the shading point lies on the ray
    for an untransformed scene."""
    org, d = ray_set(np.random.default_rng(17), 4096)
    for name in ("p3_t08", "p3_t02_sierp", "cylinder1"):
        ti, tt = orc.OracleScene(name + ".cli").trace_rays(org, d)
        ids, t, pos, nrm = ray_oracle.query_rays(name, org, d)
        assert np.array_equal(ids, ti) and np.array_equal(t, tt), name
        hit = ids[:, 0] >= 0
        assert hit.sum() > 100 and np.allclose(np.linalg.norm(nrm[hit], axis=1), 1.0)
        occ = ray_oracle.shadow_rays(name, org, d, np.full(len(org), np.inf))
        assert occ[hit].all(), name          # whatever the closest-hit search hits also blocks an unbounded shadow ray


# ---- closest hit == the generic-kernel probe, bit for bit --------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("accel", [0, 1, 2])
@pytest.mark.parametrize("name", PROBE_SCENES)
def test_closest_equals_probe(drt, gpu_ctx_factory, monkeypatch, name, accel):
    org, d = ray_set(np.random.default_rng(11), 1 << 15)
    deferred = {}
    for shape in SHAPES:
        ctx, s = load(drt, gpu_ctx_factory, name, accel, shape, monkeypatch)
        pi, pt = s.trace_rays(org, d)
        (ids, t), st = query(drt, s, org, d)
        assert np.array_equal(ids, pi), (name, accel, shape)
        assert np.array_equal(t.view(np.int64), pt.view(np.int64)), (name, accel, shape)
        (ids2, t2, pos, nrm), _ = query(drt, s, org, d, frame=True)
        assert np.array_equal(ids2, ids) and np.array_equal(t2, t)
        assert np.all(pos[ids[:, 0] < 0] == 0) and np.all(np.abs(np.linalg.norm(nrm[ids[:, 0] >= 0], axis=1) - 1) < 1e-12)
        assert st.host_syncs == 1 and st.kernel_launches in (1, 2)
        deferred[shape] = st.rays_deferred
        ctx.close()
    assert (pi[:, 0] >= 0).sum() > 300, name
    assert deferred[7] == 0
    if accel > 0 and name in ("p3_t09", "p3_t11_sierp"):
        assert deferred[0] > 0, deferred          # the fix-up pass served part of these rays and the result is still the probe's


# ---- closest hit == oracle ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ORACLE_SCENES)
def test_closest_equals_oracle(drt, ray_oracle, gpu_ctx_factory, monkeypatch, name):
    org, d = ray_set(np.random.default_rng(12), 8192)
    oi, ot, opos, onrm = ray_oracle.query_rays(name, org, d)
    assert (oi[:, 0] >= 0).sum() > 100, name
    hit = oi[:, 0] >= 0
    for accel in (0, 1):
        ctx, s = load(drt, gpu_ctx_factory, name, accel, None, monkeypatch)
        (ids, t, pos, nrm), _ = query(drt, s, org, d, frame=True)
        assert np.array_equal(ids, oi), (name, accel, int((ids != oi).any(axis=1).sum()))
        assert np.array_equal(t.view(np.int64), ot.view(np.int64)), (name, accel)
        assert close_rel(pos[hit], opos[hit]) and close_rel(nrm[hit], onrm[hit]), (name, accel)
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["p3_t08", "p3_t02_sierp", "p3_t09"])
def test_tmax_reports_a_hit_exactly_when_t_is_below_it(drt, gpu_ctx_factory, monkeypatch, name):
    org, d = ray_set(np.random.default_rng(13), 1 << 14)
    for accel in (0, 1):
        ctx, s = load(drt, gpu_ctx_factory, name, accel, None, monkeypatch)
        (ids, t), _ = query(drt, s, org, d)
        hit = ids[:, 0] >= 0
        assert hit.sum() > 100
        tt = np.where(hit, t, 1.0)
        cases = {"t(1-2^-40)": tt * (1 - 2.0 ** -40), "t": tt, "nextafter": np.nextafter(tt, np.inf), "inf": np.full_like(tt, np.inf), "nan": np.full_like(tt, np.nan)}
        for label, tmax in cases.items():
            (bi, bt, bpos, _), _ = query(drt, s, org, d, tmax=cuda(tmax), frame=True)
            expect = hit & (t < tmax)
            assert np.array_equal(bi[expect], ids[expect]) and np.array_equal(bt[expect], t[expect]), label
            assert np.all(bi[~expect] == -1) and np.all(bt[~expect] == 0) and np.all(bpos[~expect] == 0), label
            assert expect.sum() == (hit.sum() if label in ("nextafter", "inf") else 0), label
        ctx.close()


# ---- occlusion == oracle --------------------------------------------------------------------------------------------------------------
def shadow_set(drt, s, name, rng, n):
    """Random rays with random distances, and shadow-shaped rays: from the hit points of a first query toward the scene's lights, with
    distances just around the closest blocker (relative 1e-9, DRT_EPS edge, twice as far, +inf)."""
    org, d = ray_set(rng, n)
    dist = rng.uniform(0, 12, size=n); dist[::7] = np.inf
    (ids, _, pos, _), _ = query(drt, s, org, d, frame=True)
    p = pos[ids[:, 0] >= 0][: n // 2]
    lights = light_positions(name)
    L = lights[rng.integers(0, len(lights), size=len(p))]
    sd = L - p
    (bi, bt), _ = query(drt, s, p, sd)
    blocked = bi[:, 0] >= 0
    choice = rng.integers(0, 6, size=len(p))
    tb = np.where(blocked, bt, np.linalg.norm(sd, axis=1))
    opts = np.stack([tb * (1 - 1e-9), tb * (1 + 1e-9), tb + EPS * (1 - 1e-6), tb + EPS * (1 + 1e-6), 2 * tb, np.full_like(tb, np.inf)], axis=1)
    sdist = opts[np.arange(len(p)), choice]
    return np.concatenate([org, p]), np.concatenate([d, sd]), np.concatenate([dist, sdist]), len(p), blocked


@pytest.mark.gpu
@pytest.mark.parametrize("name", ORACLE_SCENES + ["p3_t11_sierp"])
def test_occluded_equals_oracle(drt, ray_oracle, gpu_ctx_factory, monkeypatch, name):
    ctx, s = load(drt, gpu_ctx_factory, name, 0, None, monkeypatch)
    org, d, dist, ns, blocked = shadow_set(drt, s, name, np.random.default_rng(14), 8192)
    ctx.close()
    assert ns > 300 and blocked.sum() > 10, (ns, blocked.sum())
    ref = ray_oracle.shadow_rays(name, org, d, dist)
    assert 0 < ref.sum() < len(ref)
    for accel in (0, 1, 2):
        first = None
        for shape in SHAPES:
            ctx, s = load(drt, gpu_ctx_factory, name, accel, shape, monkeypatch)
            occ, st = occl(drt, s, org, d, dist)
            lbvh = accel == 2 and s.accel_info()["lbvh_tris"] > 0
            ctx.close()
            assert occ.dtype == bool and st.host_syncs == 1
            if lbvh:        # GPU-built mesh boxes: self-shadowing differs from the reference tree by construction (SURVEY Q1b)
                first = occ if first is None else first
                assert np.array_equal(occ, first), (name, accel, shape)
            else:
                assert np.array_equal(occ, ref), (name, accel, shape, int((occ != ref).sum()))


# ---- edges ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_edges_and_return_codes(drt, gpu_ctx_factory, monkeypatch):
    import torch
    ctx, s = load(drt, gpu_ctx_factory, "p3_t08", 1, None, monkeypatch)
    e = torch.zeros((0, 3), dtype=torch.float64, device="cuda:0")
    st = drt.Stats()
    ids, t = s.intersect(e, e, stats=st)
    assert ids.shape == (0, 2) and t.shape == (0,) and st.kernel_launches == 0 and st.host_syncs == 0
    assert s.occluded(e, e, torch.zeros(0, dtype=torch.float64, device="cuda:0")).shape == (0,)
    # rays that are not traced: non-finite origin or direction, zero-length direction (or one whose FP64 length under- / overflows)
    inf, nan = np.inf, np.nan
    org = np.array([[0, 0, 0], [nan, 0, 0], [0, inf, 0], [0, 0, 0], [0, 0, 0], [0, 0, 0], [0, 0, 0], [0, 0, 0], [0, 0, 0]], dtype=np.float64)
    d = np.array([[0, 0, -1], [0, 0, -1], [0, 0, -1], [0, 0, 0], [nan, 0, -1], [0, -inf, -1], [1e-300, 0, -1e-300], [1e300, 0, -1e300], [0, 0, -1]], dtype=np.float64)
    (ids, t, pos, nrm), _ = query(drt, s, org, d, frame=True)
    pi, pt = s.trace_rays(org, d)          # the probe follows the same rule: every ray, traced or not, gives the query's ids and t
    assert np.array_equal(ids, pi) and np.array_equal(t.view(np.int64), pt.view(np.int64))
    assert pi[0, 0] >= 0 and np.array_equal(ids[-1], pi[0]) and t[0] == pt[0] == t[-1]
    assert np.all(ids[1:-1] == -1) and np.all(t[1:-1] == 0) and np.all(pos[1:-1] == 0) and np.all(nrm[1:-1] == 0)
    dist = np.full(len(org), np.inf); dist[-1] = nan           # the last ray is a normal one, but a NaN distance is not occluded
    occ, _ = occl(drt, s, org, d, dist)
    assert occ[0] and not occ[1:].any(), occ
    # NULL optional outputs and tmax: the same ids and t
    org2, d2 = ray_set(np.random.default_rng(15), 4096)
    (a_ids, a_t), _ = query(drt, s, org2, d2)
    (b_ids, b_t, _, _), _ = query(drt, s, org2, d2, frame=True)
    assert np.array_equal(a_ids, b_ids) and np.array_equal(a_t, b_t)
    # return codes of the C entry points
    L, h = ctx.L, ctx.h
    o, dd, dist_t = cuda(org2), cuda(d2), cuda(np.ones(len(org2)))
    ids_t = torch.empty((len(org2), 2), dtype=torch.int32, device="cuda:0"); t_t = torch.empty(len(org2), dtype=torch.float64, device="cuda:0")
    occ_t = torch.empty(len(org2), dtype=torch.uint8, device="cuda:0")
    p = lambda x: x.data_ptr()
    assert L.drt_query_closest(h, -1, p(o), p(dd), None, p(ids_t), p(t_t), None, None, None) == -2
    for args in ((None, p(dd), p(ids_t), p(t_t)), (p(o), None, p(ids_t), p(t_t)), (p(o), p(dd), None, p(t_t)), (p(o), p(dd), p(ids_t), None)):
        assert L.drt_query_closest(h, 5, args[0], args[1], None, args[2], args[3], None, None, None) == -2, args
    assert L.drt_query_closest(h, 0, None, None, None, None, None, None, None, None) == 0
    assert L.drt_query_occluded(h, -1, p(o), p(dd), p(dist_t), p(occ_t), None) == -2
    for args in ((None, p(dd), p(dist_t), p(occ_t)), (p(o), None, p(dist_t), p(occ_t)), (p(o), p(dd), None, p(occ_t)), (p(o), p(dd), p(dist_t), None)):
        assert L.drt_query_occluded(h, 5, *args, None) == -2, args
    assert L.drt_query_occluded(h, 0, None, None, None, None, None) == 0
    assert L.drt_query_closest(h, len(org2), p(o), p(dd), None, p(ids_t), p(t_t), None, None, None) == 0      # stats NULL
    assert np.array_equal(ids_t.cpu().numpy(), a_ids)
    ctx.close()
    # before drt_scene_finalize: DRT_ERR_STATE
    ctx = gpu_ctx_factory()
    drt.Scene.from_cli(ctx, "p3_t08.cli", finalize=False)
    assert ctx.L.drt_query_closest(ctx.h, len(org2), p(o), p(dd), None, p(ids_t), p(t_t), None, None, None) == -5
    assert ctx.L.drt_query_occluded(ctx.h, len(org2), p(o), p(dd), p(dist_t), p(occ_t), None) == -5
    ctx.close()
    # a host tensor next to a device one is refused, not copied
    ctx, s = load(drt, gpu_ctx_factory, "t01", 0, None, monkeypatch)
    with pytest.raises(ValueError, match="cuda:0"):
        s.intersect(torch.zeros((4, 3), dtype=torch.float64), cuda(np.zeros((4, 3))))
    ctx.close()


# ---- queries leave rendering alone ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["p3_t09", "box_caustics"])
def test_queries_do_not_disturb_rendering(drt, gpu_ctx_factory, name):
    ctx = gpu_ctx_factory(200, 150)
    s = drt.Scene.from_cli(ctx, name + ".cli", accel=1)
    a = s.draw(aov=True)
    org, d = ray_set(np.random.default_rng(16), 1 << 16)
    (ids, t, pos, nrm), _ = query(drt, s, org, d, frame=True)
    occl(drt, s, pos, np.tile([0.3, 1.0, 0.2], (len(pos), 1)), np.full(len(pos), np.inf))
    b = s.draw(aov=True)
    assert zlib.crc32(a["argb"].tobytes()) == zlib.crc32(b["argb"].tobytes())
    for k in ("hit_prim", "hit_inst", "t", "rgb"):
        assert np.array_equal(a[k], b[k]), k
    assert a["stats"].host_syncs == 1 and b["stats"].host_syncs == 1 and b["stats"].frame_retries == 0
    assert b["stats"].kernel_launches <= a["stats"].kernel_launches
    ctx.close()
