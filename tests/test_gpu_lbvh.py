"""GPU tests of DRT_ACCEL_LBVH (the GPU-built 30-bit-Morton LBVH, csrc/lbvh.cuh): primary-ray hit IDs and t must equal the
reference-topology modes bit for bit (same triangle set, same triangle arithmetic, same root gate); rays that start on a mesh
cannot match the reference (SURVEY Q1b) -- the image difference that causes is measured and written to gpurun_out/lbvh_parity.json."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MESH_SCENES = ["p3_t08", "p3_t09", "p3_t10", "p3_t11", "p4_t06", "p3_t11_sierp"]


def render(drt, make, name, accel, cols=320, rows=240, **kw):
    ctx = make(cols, rows, **kw)
    s = drt.Scene.from_cli(ctx, name + ".cli", accel=accel)
    g = s.draw(aov=True)
    ai = s.accel_info()
    ctx.close()
    return g, ai


@pytest.mark.parametrize("name", MESH_SCENES)
def test_lbvh_primary_hits_are_exact(drt, gpu_ctx_factory, name):
    a, _ = render(drt, gpu_ctx_factory, name, drt.ACCEL_REFERENCE)
    b, ai = render(drt, gpu_ctx_factory, name, drt.ACCEL_LBVH)
    assert ai["lbvh_tris"] > 0 and ai["lbvh_nodes"] == (ai["lbvh_tris"] + 3) // 4 - 1 or name == "p3_t10"
    assert np.array_equal(a["hit_prim"], b["hit_prim"]), (a["hit_prim"] != b["hit_prim"]).sum()
    assert np.array_equal(a["hit_inst"], b["hit_inst"])
    assert np.array_equal(a["t"], b["t"])
    assert a["stats"].rays_primary == b["stats"].rays_primary


def test_lbvh_explicit_rays_from_outside(drt, gpu_ctx_factory):
    rng = np.random.default_rng(9)
    n = 300000
    u = rng.normal(size=(n, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
    org = 9.0 * u + np.array([0, 0, -3.0])                      # outside every mesh box of the scenes below
    tgt = rng.uniform(-1.2, 1.2, size=(n, 3)) + np.array([0, 0, -3.0])
    # axis-parallel rays aimed at targets of the same region: one direction component +-1, the others +0.0 or -0.0
    m = 100000
    d2 = np.where(rng.random(size=(m, 3)) < 0.5, 0.0, -0.0)
    d2[np.arange(m), rng.integers(0, 3, size=m)] = rng.choice([-1.0, 1.0], size=m)
    tgt2 = rng.uniform(-1.2, 1.2, size=(m, 3)) + np.array([0, 0, -3.0])
    dirs = np.concatenate([tgt - org, d2])
    org = np.concatenate([org, tgt2 - 9.0 * d2])
    for name in ("p3_t09", "p3_t08"):
        res = []
        for accel in (drt.ACCEL_REFERENCE, drt.ACCEL_LBVH):
            ctx = gpu_ctx_factory()
            s = drt.Scene.from_cli(ctx, name + ".cli", accel=accel)
            res.append(s.trace_rays(org, dirs))
            ctx.close()
        assert (res[0][0][:n, 0] >= 0).sum() > 10000 and (res[0][0][n:, 0] >= 0).sum() > 1000
        assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1]), name


def test_lbvh_image_difference_is_measured(drt, orc, gpu_ctx_factory, tmp_path_factory):
    """Self-shadowing / self-reflection on a mesh depends on the reference's own tree (every box that contains the ray origin is
    skipped, myGeomBase.java:142-161,397-404); an LBVH with conventional boxes shadows correctly instead. Quantify, do not hide."""
    out = {}
    for name in ("p3_t08", "p3_t09", "p3_t11_sierp"):
        a, _ = render(drt, gpu_ctx_factory, name, drt.ACCEL_REFERENCE, 300, 300)
        b, ai = render(drt, gpu_ctx_factory, name, drt.ACCEL_LBVH, 300, 300)
        d = np.abs(orc.argb_to_rgb8(a["argb"]).astype(int) - orc.argb_to_rgb8(b["argb"]).astype(int)).max(axis=-1)
        on_mesh = a["hit_prim"] >= 0
        out[name] = {"px_gt2_frac": float((d > 2).mean()), "px_gt2_frac_of_hit_pixels": float((d[on_mesh] > 2).mean()), "max_diff": int(d.max()),
                     "lbvh_build_ms": ai["lbvh_build_ms"], "lbvh_tris": ai["lbvh_tris"], "lbvh_nodes": ai["lbvh_nodes"],
                     "shadow_rays_ref": int(a["stats"].rays_shadow), "shadow_rays_lbvh": int(b["stats"].rays_shadow)}
        assert (d > 2).mean() < 0.5
    # The shipped scenes all build their meshes under a translate/rotate, and the reference then shades at M.M.p (SURVEY Q6): shadow
    # rays start OFF the mesh, which is why the numbers above are zero.  A mesh under the identity CTM (vertices pre-translated in the
    # file) is the case where Q1b bites: the reference skips every box that contains the shadow-ray origin, the LBVH shadows correctly.
    tmp = tmp_path_factory.mktemp("lbvh")
    lines = open(os.path.join(ROOT, "scenes", "bun500.cli")).read().split("\n")
    moved = []
    for ln in lines:
        t = ln.split(" ")
        if t[0] == "vertex":
            ln = "vertex %r %r %r" % (float(t[1]), float(t[2]), float(t[3]) - 3.0)
        moved.append(ln)
    (tmp / "bunmoved.cli").write_text("\n".join(moved))
    (tmp / "ident.cli").write_text("fov 60\nbackground 0.2 0.2 1\npoint_light 3 4 0 .8 .8 .8\npoint_light -3 4 0 .2 .2 .2\ndiffuse .8 .8 .8 .2 .2 .2\n"
                                   "begin\nvertex -100 -1 -100\nvertex 100 -1 -100\nvertex 100 -1 100\nend\nbegin\nvertex 100 -1 100\nvertex -100 -1 100\nvertex -100 -1 -100\nend\n"
                                   "diffuse .9 .9 .9 0 0 0\nbegin_list\nread bunmoved.cli\nend_accel\nwrite x.png\n")
    imgs = []
    for accel in (drt.ACCEL_REFERENCE, drt.ACCEL_REFERENCE_FAST, drt.ACCEL_LBVH):
        ctx = gpu_ctx_factory(300, 300)
        imgs.append(drt.Scene.from_cli(ctx, "ident.cli", data_dir=str(tmp), accel=accel).draw(aov=True))
        ctx.close()
    assert np.array_equal(imgs[0]["argb"], imgs[1]["argb"])                      # fast mode: still the reference's answer
    assert np.array_equal(imgs[0]["hit_prim"], imgs[2]["hit_prim"])              # LBVH: primary hits exact ...
    d = np.abs(orc.argb_to_rgb8(imgs[0]["argb"]).astype(int) - orc.argb_to_rgb8(imgs[2]["argb"]).astype(int)).max(axis=-1)
    on_mesh = imgs[0]["hit_prim"] > 1
    out["bun500_identity_ctm"] = {"px_gt2_frac": float((d > 2).mean()), "px_gt2_frac_of_mesh_pixels": float((d[on_mesh] > 2).mean()), "max_diff": int(d.max())}
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "lbvh_parity.json"), "w"), indent=1)
    print(json.dumps(out))


def test_lbvh_is_deterministic(drt, gpu_ctx_factory):
    a, _ = render(drt, gpu_ctx_factory, "p3_t09", drt.ACCEL_LBVH, 200, 200)
    b, _ = render(drt, gpu_ctx_factory, "p3_t09", drt.ACCEL_LBVH, 200, 200)
    assert np.array_equal(a["argb"], b["argb"])


@pytest.mark.parametrize("kind,n", [("soup", 65536), ("grid", 4)])
def test_synthetic_scaling_scenes_sampled_rays_match_oracle(drt, orc, gpu_ctx_factory, kind, n):
    """SURVEY 8(d) synthetic scenes (tools/make_synth.py): 65 536 random triangles in one BVH, and a 4x4x4 grid of bunny instances inside an
    instance BVH.  Too slow for an oracle image at benchmark size, so parity is sampled: 20 000 random rays, closest-hit primitive /
    instance IDs and t bit-exact against the oracle, in every traversal mode (LBVH: rays start outside the mesh boxes, SURVEY Q1b)."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_synth
    name = "gen/" + os.path.basename(getattr(make_synth, kind)(n))
    rng = np.random.default_rng(17)
    m = 20000
    u = rng.normal(size=(m, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
    org = 9.0 * u + np.array([0, 0, -3.0])
    tgt = rng.uniform(-1.0, 1.0, size=(m, 3)) + np.array([0, 0, -3.0 if kind == "soup" else -3.5])
    oi, ot = orc.OracleScene(name).trace_rays(org, tgt - org)
    assert (oi[:, 0] >= 0).sum() > 2000
    for accel in (drt.ACCEL_REFERENCE, drt.ACCEL_REFERENCE_FAST, drt.ACCEL_LBVH):
        ctx = gpu_ctx_factory()
        gi, gt = drt.Scene.from_cli(ctx, name, accel=accel).trace_rays(org, tgt - org)
        ctx.close()
        assert (gi != oi).any(axis=1).sum() <= 2, (kind, accel, (gi != oi).any(axis=1).sum())
        same = (gi == oi).all(axis=1)
        assert np.array_equal(gt[same], ot[same]), (kind, accel)


@pytest.mark.parametrize("name", ["p3_t09", "gen/soup_65536"])
def test_lbvh_morton_order_and_tree_equal_the_cpu_restatement(drt, gpu_ctx_factory, name):
    """North star: "Morton/BVH ordering must be bit-exact".  The device build (k_lbvh_morton, radix sort, k_lbvh_hierarchy, k_lbvh_refit) against
    oracle/lbvh_oracle.py: resident triangle order, every child link and every node box."""
    from oracle import lbvh_oracle
    if name.startswith("gen/") and not os.path.exists(os.path.join(ROOT, "scenes", name + ".cli")):
        import subprocess, sys
        subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "make_synth.py"), "soup", "65536"])
    ctx = gpu_ctx_factory(64, 64)
    s = drt.Scene.from_cli(ctx, name + ".cli", accel=drt.ACCEL_LBVH)
    host, dev = s.lbvh_probe(0, resident=False), s.lbvh_probe(0, resident=True)
    assert len(host["verts"]) == len(dev["verts"]) > 1000 and len(dev["links"]) == (len(dev["verts"]) + 3) // 4 - 1
    order, links, boxes = lbvh_oracle.build(host["verts"], host["box"])
    assert np.array_equal(host["serial"][order], dev["serial"])                 # Morton order, ties in input order
    assert np.array_equal(host["verts"][order], dev["verts"])
    assert np.array_equal(links, dev["links"])                                  # Karras hierarchy
    assert np.array_equal(boxes, dev["boxes"])                                  # refit boxes, bit for bit
    ctx.close()


def test_lbvh_with_thousands_of_equal_morton_codes(drt, gpu_ctx_factory, tmp_path):
    """Traversal stacks are fixed-depth (32 entries in the lean kernels, 64 in the generic ones; overflow defers the ray / fails the call, never
    drops geometry silently).  The worst case for an LBVH is a mesh with many triangles in one Morton cell: the radix tree over (code, index)
    keys then splits on index bits and is as deep as 30 + log2(duplicates).  6 000 coincident small triangles + 3 000 spread ones: mode 2 must
    render, and its primary hits and t must equal the reference tree's."""
    rng = np.random.default_rng(21)
    lines = ["fov 60", "background 0 0 0", "point_light 2 4 3 1 1 1", "diffuse .8 .8 .8 .1 .1 .1", "begin_list"]
    def tri(c, e):
        a, b, d = c, c + np.array([e, 0, 0]), c + np.array([0, e, 0])
        return ["begin"] + ["vertex %.9g %.9g %.9g" % tuple(v) for v in (a, b, d)] + ["end"]
    for i in range(6000):
        lines += tri(np.array([0.1, 0.1, -4.0]) + rng.uniform(-1e-6, 1e-6, 3), 0.2)              # all in one Morton cell
    for i in range(3000):
        lines += tri(rng.uniform(-1.5, 1.5, 3) + np.array([0, 0, -4.0]), 0.15)
    lines += ["end_accel", "write x.png"]
    (tmp_path / "dup.cli").write_text("\n".join(lines) + "\n")
    res = []
    for accel in (drt.ACCEL_REFERENCE, drt.ACCEL_LBVH, drt.ACCEL_REFERENCE_FAST):
        ctx = gpu_ctx_factory(200, 150)
        g = drt.Scene.from_cli(ctx, "dup.cli", data_dir=str(tmp_path), accel=accel).draw(aov=True)      # a stack overflow would raise here
        ctx.close(); res.append(g)
    assert (res[0]["hit_prim"] >= 0).sum() > 2000
    for other in res[1:]:
        assert np.array_equal(res[0]["hit_prim"], other["hit_prim"]) and np.array_equal(res[0]["t"], other["t"])
    assert np.array_equal(res[0]["argb"], res[2]["argb"])
