"""GPU tests of the traversal modes (DESIGN.md §3): DRT_ACCEL_REFERENCE_FAST must reproduce DRT_ACCEL_REFERENCE bit for bit
(same tree, same box rule, same triangle arithmetic; only the visiting order and the pruning differ), and DRT_ACCEL_LBVH must keep
primary-ray hit IDs exact while its mesh self-shadowing differs by construction (SURVEY Q1b) -- that difference is measured here."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MESH_SCENES = ["p3_t08", "p3_t09", "p3_t10", "p3_t11", "p3_t11_sierp", "p4_t06", "plnts3ColsBunnies", "p3_t12", "p3_t05",
               "t03", "t06", "t07", "c2clear", "p2_t05", "box_caustics"]      # the last six: plain top-level triangles / quads (lean top-level path), no BVH


def render(drt, make, name, accel, cols, rows, spp=0, **kw):
    ctx = make(cols, rows, **kw)
    s = drt.Scene.from_cli(ctx, name + ".cli", spp=spp, accel=accel)
    g = s.draw(aov=True)
    info = s.info()
    ctx.close()
    return g, info


@pytest.mark.parametrize("name", MESH_SCENES)
def test_fast_mode_equals_reference_mode(drt, gpu_ctx_factory, name):
    spp = 2 if name == "plnts3ColsBunnies" else 0
    a, _ = render(drt, gpu_ctx_factory, name, drt.ACCEL_REFERENCE, 320, 240, spp)
    b, _ = render(drt, gpu_ctx_factory, name, drt.ACCEL_REFERENCE_FAST, 320, 240, spp)
    assert np.array_equal(a["hit_prim"], b["hit_prim"]) and np.array_equal(a["hit_inst"], b["hit_inst"])
    assert np.array_equal(a["t"], b["t"])
    assert np.array_equal(a["argb"], b["argb"])
    for k in ("rays_primary", "rays_shadow", "rays_reflect", "rays_refract"):
        assert getattr(a["stats"], k) == getattr(b["stats"], k)


def test_fast_mode_matches_oracle(drt, orc, gpu_ctx_factory):
    for name in ("p3_t09", "p3_t11_sierp"):
        g, _ = render(drt, gpu_ctx_factory, name, drt.ACCEL_REFERENCE_FAST, 160, 160)
        r = orc.OracleScene(name + ".cli", cols=160, rows=160).render(threads=os.cpu_count())
        assert (g["hit_prim"] != r["hit_prim"]).sum() <= 2 and (g["hit_inst"] != r["hit_inst"]).sum() <= 2
        d = np.abs(orc.argb_to_rgb8(g["argb"]).astype(int) - orc.argb_to_rgb8(r["argb"]).astype(int)).max(axis=-1)
        assert (d > 2).mean() <= 1e-3


def test_fast_mode_counters_do_less_work(drt, gpu_ctx_factory):
    a, _ = render(drt, gpu_ctx_factory, "p3_t09", drt.ACCEL_REFERENCE, 320, 240, counters=True)
    b, _ = render(drt, gpu_ctx_factory, "p3_t09", drt.ACCEL_REFERENCE_FAST, 320, 240, counters=True)
    assert b["stats"].prim_tests_closest <= a["stats"].prim_tests_closest
    assert np.array_equal(a["argb"], b["argb"])


def test_fast_mode_explicit_rays_from_everywhere(drt, gpu_ctx_factory):
    """Rays starting inside / on / outside the meshes' boxes, a share of them (almost) axis-parallel: closest-hit IDs and t must be identical
    in both modes."""
    rng = np.random.default_rng(3)
    for name in ("p3_t09", "p3_t10", "p3_t11_sierp"):
        n = 200000
        org = rng.uniform(-3, 3, size=(n, 3)); org[:, 2] -= 3
        d = rng.normal(size=(n, 3))
        # rows [0, 2k): exactly axis-parallel (one component +0.0 or -0.0, two in the first k); rows [2k, 3k): one component around 1e-17
        k = n // 8; rows = np.arange(2 * k)
        zero = np.where(rng.random(size=(2 * k, 3)) < 0.5, 0.0, -0.0); ax = rng.integers(0, 3, size=2 * k)
        d[rows, ax] = zero[rows, ax]
        d[rows[:k], (ax[:k] + 1) % 3] = zero[rows[:k], (ax[:k] + 1) % 3]
        d[np.arange(2 * k, 3 * k), rng.integers(0, 3, size=k)] = rng.choice([-1e-17, 1e-17], size=k) * rng.uniform(0.5, 2.0, size=k)
        res = []
        for accel in (drt.ACCEL_REFERENCE, drt.ACCEL_REFERENCE_FAST):
            ctx = gpu_ctx_factory()
            s = drt.Scene.from_cli(ctx, name + ".cli", accel=accel)
            res.append(s.trace_rays(org, d))
            ctx.close()
        assert np.array_equal(res[0][0], res[1][0]), name
        assert np.array_equal(res[0][1], res[1][1]), name
        assert (res[0][0][:, 0] >= 0).sum() > 1000 and (res[0][0][:2 * k, 0] >= 0).sum() > 1000


# ---- kernel variants and the sync-free wavefront loop (round 2) ------------------------------------------------------------------------
SHAPE_SCENES = [("p3_t09", 0), ("p3_t11_sierp", 0), ("p3_t12", 0), ("p3_t05", 0), ("planets3Ortho", 4), ("gen_ortho_bunny", 0), ("plnts3ColsBunnies", 2), ("p3_t10", 0), ("c5Fish", 0), ("box_caustics", 0)]


@pytest.mark.parametrize("name,spp", SHAPE_SCENES)
def test_kernel_variants_give_identical_frames(drt, gpu_ctx_factory, name, spp, monkeypatch):
    """The lean trace / light kernels (flat scenes: shape 0; instanced meshes: shape 1) defer what they cannot serve to the generic kernels
    (shape 7).  Whatever variant the scene runs with, every buffer must be identical -- including scenes where a variant defers EVERY ray
    (orthographic camera: axis-parallel rays; instance trees under the flat-scene kernel)."""
    if name == "gen_ortho_bunny":       # orthographic camera over a mesh: every primary ray is axis-parallel, so the lean descent defers all of them
        import tempfile
        d = tempfile.mkdtemp()
        src = open(os.path.join(drt.SCENES_DIR, "p3_t08.cli")).read().replace("fov 60", "orthographic 4 4")
        assert "orthographic" in src
        open(os.path.join(drt.SCENES_DIR, "gen_ortho_bunny.cli"), "w").write(src)
    res = {}
    for shape in (7, 0, 1):
        monkeypatch.setenv("DRT_FORCE_SHAPE", str(shape))
        res[shape], _ = render(drt, gpu_ctx_factory, name, drt.ACCEL_REFERENCE_FAST, 200, 150, spp)
    monkeypatch.delenv("DRT_FORCE_SHAPE")
    auto, _ = render(drt, gpu_ctx_factory, name, drt.ACCEL_REFERENCE_FAST, 200, 150, spp)
    for other in (res[0], res[1], auto):
        for k in ("argb", "hit_prim", "hit_inst", "t", "rgb"):
            assert np.array_equal(res[7][k], other[k]), (name, k)
        for k in ("rays_primary", "rays_shadow", "rays_reflect", "rays_refract"):
            assert getattr(res[7]["stats"], k) == getattr(other["stats"], k)
    assert res[7]["stats"].rays_deferred == 0
    if name == "gen_ortho_bunny":
        assert auto["stats"].rays_deferred > 1000        # every ray that reaches the mesh (the others miss its root box before any descent)
    if name == "p3_t11_sierp":          # the flat-scene kernel cannot enter an instance tree: every ray that reaches its root box is deferred
        assert res[0]["stats"].rays_deferred > 0


def test_frame_needs_one_host_sync_and_speculation_is_checked(drt, gpu_ctx_factory, monkeypatch):
    """No host round trip per bounce level: level sizes live on the device.  The two speculations of the loop -- queue capacity and the number of
    levels launched -- are verified by the device and a failed one re-renders the frame; the result never changes."""
    ctx = gpu_ctx_factory(256, 192)
    s = drt.Scene.from_cli(ctx, "planets3columns.cli", spp=2, accel=drt.ACCEL_REFERENCE_FAST)
    a, st = s.draw()
    assert st.host_syncs == 1 and st.frame_retries == 0 and st.rays_reflect + st.rays_refract > 0
    b, st2 = s.draw()                         # second frame of the same scene: launches only the depth the first one needed (+1)
    assert np.array_equal(a, b) and st2.frame_retries == 0 and st2.kernel_launches <= st.kernel_launches
    monkeypatch.setenv("DRT_DEPTH_HINT", "2")
    c, st3 = s.draw()
    assert np.array_equal(a, c) and st3.frame_retries >= 1
    monkeypatch.delenv("DRT_DEPTH_HINT")
    monkeypatch.setenv("DRT_QUEUE_FACTOR", "0.05")
    d, st4 = s.draw()
    assert np.array_equal(a, d) and st4.frame_retries >= 1
    for k in ("rays_primary", "rays_shadow", "rays_reflect", "rays_refract"):
        assert getattr(st, k) == getattr(st4, k) == getattr(st3, k)
    ctx.close()
