"""CPU tests of the product's host side: the C ABI loads and exports what include/drt.h declares, the .cli
interpreter/flattener reproduces the oracle's scene graph (BVH order, boxes, CTMs), error behaviour, PNG output.
No compute entry point is called (no GPU here): a host-only context must refuse to render."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol(drt):
    hdr = open(os.path.join(ROOT, "include", "drt.h")).read()
    declared = set(re.findall(r"\b(drt_[a-z0-9_]+)\s*\(", hdr)) - {"drt_image_loader_fn"}
    assert len(declared) >= 20
    L = C.CDLL(drt.lib_path())
    for name in sorted(declared):
        assert hasattr(L, name), name
    from distraytracer_old_b200 import host
    assert declared == set(host.EXPORTS)


def test_no_cpu_fallback(drt):
    ctx = drt.Context(device=-1)
    s = drt.Scene.from_cli(ctx, "t01.cli")
    with pytest.raises(drt.DrtError, match="no CPU fallback"):
        s.draw()
    with pytest.raises(drt.DrtError):
        s.trace_rays(np.zeros((1, 3)), np.array([[0.0, 0.0, -1.0]]))
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(drt.DrtError):
            drt.Context(device=0)       # fails loudly instead of falling back


def test_product_does_not_import_oracle():
    for dp, _, files in os.walk(os.path.join(ROOT, "distraytracer_old_b200")):
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f), errors="ignore").read()
                for pat in ("import oracle", "from oracle", "oracle/", "liborc", "orc_", "orc."):
                    assert pat not in src, (f, pat)


SCENES = ["t01", "t03", "t05", "t11", "p3_t01", "p3_t02", "p3_t02_sierp", "p3_t03", "p3_t05", "p3_t06", "p3_t07", "p3_t08", "p3_t12",
          "p2_t06", "p4_st03", "p4_t03", "planets3Ortho", "c5Fish", "old_t07c", "trTrans", "cylinder1", "c3spotLight"]


@pytest.mark.parametrize("name", SCENES)
def test_flattener_matches_oracle_scene_graph(drt, orc, name):
    ctx = drt.Context(device=-1)
    s = drt.Scene.from_cli(ctx, name + ".cli")
    o = orc.OracleScene(name + ".cli")
    info = s.info()
    assert (info["top"], info["prims"], info["instances"], info["lights"], info["spp"], info["photon_kind"]) == (o.n_objs, o.n_prims, o.n_insts, o.n_lights, o.spp, o.photon_kind)
    for i in range(info["top"]):
        assert np.array_equal(s.obj_ctm(i), o.obj_ctm(i)), (name, i)      # bit-exact CTMs (matrix stack, rotations)
        a, abox = s.dump_bvh(i)
        b, bbox = o.dump_bvh(i)
        assert (a is None) == (b is None)
        if a is not None:
            assert np.array_equal(a, b), (name, i)                      # same topology, same leaf order, same dropped object
            assert np.array_equal(abox, bbox), (name, i)                # same (corner-only) boxes, bit for bit


def test_bun69k_standin_bvh(drt, orc):
    ctx = drt.Context(device=-1)
    s = drt.Scene.from_cli(ctx, "p3_t09.cli")
    o = orc.OracleScene("p3_t09.cli")
    a, abox = s.dump_bvh(2)
    b, bbox = o.dump_bvh(2)
    assert np.array_equal(a, b) and np.array_equal(abox, bbox)
    assert s.info()["prims"] == 61826


def test_line_by_line_interface_equals_file_loader(drt):
    ctx = drt.Context(device=-1)
    a = drt.Scene.from_cli(ctx, "p3_t12.cli")
    da, _ = a.dump_bvh(2)
    ia = a.info()
    rd = drt.RTFileReader(ctx)
    # forwarding every line through drt_scene_command builds the same scene (host-only: stop before `write` renders)
    sc = drt.Scene(ctx)
    for raw in open(os.path.join(drt.SCENES_DIR, "p3_t12.cli")):
        line = raw.rstrip("\r\n")
        tok = line.split()
        if not tok or tok[0].startswith("#"):
            continue
        if tok[0] == "read":
            for raw2 in open(os.path.join(drt.SCENES_DIR, tok[1])):
                sc.command(raw2.rstrip("\r\n"))
        else:
            sc.command(line)
    assert sc.info() == ia


def test_malformed_and_unknown_commands(drt):
    ctx = drt.Context(device=-1)
    sc = drt.Scene(ctx)
    sc.command("torus 1 2 3")             # unknown commands are ignored with a warning (myRTFileReader.java:343-345)
    assert sc.info()["warnings"] == 1
    with pytest.raises(drt.DrtError, match="malformed"):
        sc.command("sphere 1 0")          # Java: ArrayIndexOutOfBounds
    with pytest.raises(drt.DrtError):
        sc.command("instance nothing")
    with pytest.raises(drt.DrtError):
        drt.Scene.from_cli(ctx, "no_such_file.cli")
    # Q18: only 10 matrix-stack slots exist
    sc2 = drt.Scene(ctx)
    for _ in range(9):
        sc2.command("push")
    with pytest.raises(drt.DrtError):
        sc2.command("push")


def test_sampler_matches_oracle_bit_for_bit(drt, orc):
    from distraytracer_old_b200.host import sample_u01
    rng = np.random.default_rng(3)
    for _ in range(200):
        seed = int(rng.integers(0, 2 ** 63)); a, b, c, d = [int(x) for x in rng.integers(0, 2 ** 32, size=4)]
        stream = [0, 0x50484F54][int(rng.integers(0, 2))]
        assert sample_u01(seed, stream, a, b, c, d) == orc.u01(seed, stream, a, b, c, d)


def test_png_writer_roundtrip(drt, tmp_path):
    from PIL import Image
    rng = np.random.default_rng(0)
    rgb = rng.integers(0, 256, size=(37, 53, 3), dtype=np.uint32)
    argb = ((0xFF << 24) | (rgb[..., 0] << 16) | (rgb[..., 1] << 8) | rgb[..., 2]).astype(np.uint32).view(np.int32)
    ctx = drt.Context(device=-1)
    p = str(tmp_path / "x.png")
    drt.Scene(ctx).save(p, argb)
    back = np.asarray(Image.open(p).convert("RGB"))
    assert np.array_equal(back, rgb.astype(np.uint8))


def test_chunk_partition_covers_every_pixel_once():
    from distraytracer_old_b200 import dist as D
    for rows, cols, world in ((300, 300, 1), (2160, 3840, 8), (37, 11, 3), (8, 8, 4)):
        seen = np.zeros(rows * cols, dtype=np.int32)
        for r in range(world):
            for p0, p1 in D.chunk_table(rows, cols, world)[r]:
                seen[p0:p1] += 1
            idx = D.pack_index(rows, cols, world, r)
            assert len(idx) == D.packed_size(rows, cols, world)
        assert (seen == 1).all()
    lo = [D.photon_range(1000003, 8, r) for r in range(8)]
    assert lo[0][0] == 0 and lo[-1][1] == 1000003 and all(lo[i][1] == lo[i + 1][0] for i in range(7))


def test_fast_path_packing(drt):
    """Host flattener products the fast traversal modes rely on: every triangle of a pure-triangle BVH gets one packed record (the object the
    reference drops, SURVEY Q2, excepted), plain top-level triangles get one too, BVHs with mixed children / differing CTMs do not qualify."""
    ctx = drt.Context(device=-1)
    c = drt.Scene.from_cli(ctx, "p3_t08.cli", finalize=False).counts()          # bun500 (966 triangles) in a BVH + 2 floor triangles
    assert c["fast_bvhs"] == 1 and c["tris_in_fast_bvhs"] == 965 and c["top_tris_packed"] == 2 and c["tris_packed"] == 967
    c = drt.Scene.from_cli(ctx, "t01.cli", finalize=False).counts()             # spheres only
    assert c["tris_packed"] == 0 and c["fast_bvhs"] == 0
    c = drt.Scene.from_cli(ctx, "box_caustics.cli", finalize=False).counts()    # 12 box triangles in the top-level list
    assert c["top_tris_packed"] == 12 and c["fast_bvhs"] == 0
    c = drt.Scene.from_cli(ctx, "p3_t02_sierp.cli", finalize=False).counts()    # instance BVH over a sphere: nothing to pack
    assert c["fast_bvhs"] == 0
    ctx.close()


def test_unknown_accel_mode_is_rejected(drt):
    ctx = drt.Context(device=-1)
    s = drt.Scene.from_cli(ctx, "t01.cli", finalize=False)
    with pytest.raises(drt.DrtError):
        s.finalize(7)
    s.finalize(drt.ACCEL_LBVH)          # host-only context: flattening succeeds, nothing is uploaded
    ctx.close()


def test_finalize_rejects_unknown_accel_modes(drt):
    """drt_scene_finalize takes exactly DRT_ACCEL_REFERENCE (0), DRT_ACCEL_REFERENCE_FAST (1) and DRT_ACCEL_LBVH (2): no value outside
    them, flag bits included, is accepted."""
    ctx = drt.Context(device=-1)
    for m in (3, 4, -1, 256, 512, 257):
        with pytest.raises(drt.DrtError, match="unknown acceleration mode"):
            drt.Scene.from_cli(ctx, "t01.cli", accel=m)
    ctx.close()


def test_vertex_fast_path_keeps_the_token_rules(drt):
    """`vertex` lines are parsed in place (no token list); the rules must stay those of PApplet.splitTokens(line, " ") + Java number parsing as the
    general path applies them: any number of blanks, trailing tokens ignored, f / d suffixes accepted, a missing or malformed number is an error
    only when the vertex would be used (inside begin ... end, before the polygon is full)."""
    ctx = drt.Context(device=-1)

    def verts(lines):
        sc = drt.Scene(ctx)
        for l in ["diffuse .8 .8 .8 .1 .1 .1", "begin_list"] + (["begin"] + lines + ["end"]) * 8 + ["end_accel", "write x.png"]:
            sc.command(l)
        sc.finalize()
        p = sc.lbvh_probe(0)                      # packed triangles of the mesh (the reference's tree drops one of the eight, SURVEY Q2)
        assert sc.info()["prims"] == 8 and p is not None and len(p["verts"]) == 7
        return p["verts"]

    va = verts(["vertex 0 0.25 -5", "vertex 1.5 0 -5", "vertex 0 2 -5"])
    vb = verts(["   vertex   0   0.25f  -5d   trailing tokens", "vertex 1.5e0 +0 -5.0", "vertex 0 2 -.5e1", "vertex 9 9 9"])     # the fourth vertex of a triangle is ignored
    assert np.array_equal(va, vb) and np.array_equal(va[0], [0, 0.25, -5, 1.5, 0, -5, 0, 2, -5])
    c = drt.Scene(ctx)
    c.command("vertex nonsense here")             # outside begin ... end the reference never reads the numbers
    c.command("begin")
    with pytest.raises(drt.DrtError, match="malformed"):
        c.command("vertex 1 2")
    with pytest.raises(drt.DrtError, match="malformed"):
        c.command("vertex 1 2 3x")
    with pytest.raises(drt.DrtError, match="malformed"):
        c.command("vertex 1 two 3")
    ctx.close()


def test_build_probes_on_a_host_only_context(drt):
    """drt_build_info / drt_bvh_order / drt_lbvh_probe without a device: the host halves work, the device halves fail loudly (no CPU fallback)."""
    ctx = drt.Context(device=-1)
    s = drt.Scene.from_cli(ctx, "p3_t08.cli")
    b = s.build_info()
    assert b["bvh_objects"] == 966 and b["bvh_device_builds"] == 0 and b["parse_ms"] > 0 and b["upload_ms"] == 0
    p = s.lbvh_probe(0, resident=False)
    assert p is not None and len(p["verts"]) == 965 and len(p["links"]) == (965 + 3) // 4 - 1      # one object dropped at the root (Q2)
    assert s.lbvh_probe(5, resident=False) is None
    with pytest.raises(drt.DrtError):
        s.lbvh_probe(0, resident=True)
    keys = np.random.default_rng(1).normal(size=(100, 3))
    assert sorted(ctx.bvh_order(keys, on_device=False)) == list(range(100))
    assert len(ctx.bvh_order(np.zeros((0, 3)), on_device=False)) == 0
    with pytest.raises(drt.DrtError):
        ctx.bvh_order(keys, on_device=True)
    ctx.close()


def test_progressive_refinement_previews_match_the_reference_pass_loop(drt):
    """`refine on` (myScene.setRefine :796-803; draw() :1493-1526; writePxlSpan :1171-1177).  A literal Python restatement of the reference's
    pass loop -- every pass re-"traces" its pixels (here: looks them up in a finished frame, which is what a seeded sampler makes them), skips pixel
    (0, 0) on all passes but the first and paints step x step spans into the persistent image -- against drt_refine_steps / drt_refine_pass."""
    import math
    rng = np.random.default_rng(4)
    for cols, rows in ((300, 300), (317, 203), (64, 48), (3840, 2160)):
        ref_idx = int(math.log10(.5 * (cols + rows) / 16.0) / math.log10(2.0))
        want_steps = [2 ** i for i in range(ref_idx, -1, -1)]
        assert drt.refine_steps(cols, rows) == want_steps
        if cols > 1000:
            continue
        full = rng.integers(-2 ** 31, 2 ** 31 - 1, size=(rows, cols), dtype=np.int64).astype(np.int32)
        img = np.zeros((rows, cols), dtype=np.int32)                       # rndrdImg.pixels persists across the passes
        for k, step in enumerate(want_steps):
            skip = k != 0
            for row in range(0, rows, step):
                for col in range(0, cols, step):
                    if skip:
                        skip = False
                        continue
                    img[row:min(row + step, rows), col:min(col + step, cols)] = full[row, col]
            assert np.array_equal(drt.refine_pass(full, step), img), (cols, rows, step)
        assert np.array_equal(img, full)
    assert drt.refine_steps(8, 8) == []                                     # the reference's formula yields no pass (negative array size there)
    ctx = drt.Context(device=-1)
    sc = drt.Scene(ctx)
    assert not sc.refine_on()
    sc.command("refine on"); assert sc.refine_on()
    sc.command("refine off"); assert not sc.refine_on()
    ctx.close()
